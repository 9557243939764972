"""Launch plans: the raw-stream pass recorded once in Python, replayed from C through the C-ABI (include/avdf.h,
csrc/plan.cu).

`export_plan(model, path)` (also `model.export_plan(path)`) runs `run_staged` (interp/concat -> forward -> decode/NMS)
once per batch size with `ops._call_on_current` wrapped, and writes every launch to a file: the entry point, its scalars,
its host arrays by value, its args struct as bytes plus a relocation list, and every device pointer as (allocation,
byte offset). Each allocation is classified by where it comes from - the engine's packed weights and tables (constants,
whose bytes go into the file), its static buffers (scratch), this module's input staging (inputs), the result buffers
`run_staged` returns (outputs) and the `workspace` fields of args structs (workspace) - and a pointer into none of them
aborts the export. `engine.py` stays the only place that knows the launch sequence; the library only knows entry-point
signatures.

    python -m audio_visual_deepfake_detection_b200.libs.modeling.plan CFG CKPT OUT [--precision mixed|fp32] [--shards]
                                                                      [--batch-sizes 1 8 32] [--max-seconds 36]

`Plan` / `PlanSession` drive a plan file from Python through ctypes (tests, scripts/plan_bench.py);
`PlanSession.run_windows` runs sliding windows over long recordings (avdf_session_run_windows), like
`forward_streams(window=...)`.
"""
import argparse
import bisect
import ctypes
import os
import struct
from ctypes import c_float, c_int32, c_int64, c_void_p

import numpy as np
import torch

from ... import native as nv
from ... import ops
from ...native import AvdfError

MAGIC = b"AVDFPLAN"
FORMAT_VERSION = 1
KIND_CONST, KIND_SCRATCH, KIND_INPUT, KIND_OUTPUT, KIND_WORKSPACE = range(5)
(ROLE_NONE, ROLE_VIDEO, ROLE_BYOLA, ROLE_EMO, ROLE_OFFSETS, ROLE_META,
 ROLE_SEGS, ROLE_SCORES, ROLE_COUNTS, ROLE_VCLS) = range(10)
TAG_I32, TAG_I64, TAG_F32, TAG_PTR, TAG_HOST_I32, TAG_HOST_F32, TAG_STRUCT, TAG_STREAM = range(1, 9)
NULL, HOST_REF = 2 ** 64 - 1, 2 ** 64 - 2
ALIGN = 256

# the engine's A/B switches: read when an engine is built, recorded with the plan
SWITCHES = (("AVDF_FUSE_TAIL", "fuse_tail"), ("AVDF_FUSE_LN2", "fuse_ln2"), ("AVDF_FUSED_MLP", "fused_mlp"),
            ("AVDF_FUSED_MLP_MIN_ROWS", "fused_mlp_min_rows"), ("AVDF_HEAD_DOTS", "head_dots"))
# args struct of every entry point that takes one (sizes are checked against the C structs when a plan is opened)
STRUCTS = {"avdf_conv_gemm": nv.ConvGemmArgs, "avdf_mlp_fused": nv.MlpFusedArgs, "avdf_ln_dwconv_ln": nv.LnDwconvLnArgs,
           "avdf_postprocess": nv.PostprocessArgs}
# host-pointer fields of those structs: bytes the pointer covers (every other pointer field is a device pointer)
HOST_FIELDS = {(nv.ConvGemmArgs, "tap_rows"): lambda s: 4 * s.taps}


def _align(n):
    return (n + ALIGN - 1) // ALIGN * ALIGN


# ---------------------------------------------------------------------------- the file format (csrc/plan.cu)
def encode_plan(header, allocs, blob, lists):
    """header: dict(cc_major, cc_minor, sm_count, max_batch, max_seg_num, t_out, in_dtype, channels[3], stream_rows[3],
    description); allocs: [(kind, role, nbytes, data_offset)]; blob: bytes; lists: {batch: [(entry point, [(tag, value)])]}
    with value: int (I32 / I64), float (F32), (alloc | None, offset) (PTR), bytes (HOST_*), (bytes, [(field offset,
    alloc | HOST_REF, offset | host bytes)]) (STRUCT), None (STREAM)."""
    h = header
    out = [MAGIC, struct.pack("<II", FORMAT_VERSION, nv.lib().avdf_abi_version()),
           struct.pack("<7i", h["cc_major"], h["cc_minor"], h["sm_count"], h["max_batch"], h["max_seg_num"], h["t_out"],
                       h["in_dtype"]),
           struct.pack("<3i", *h["channels"]), struct.pack("<3q", *h["stream_rows"]),
           struct.pack("<Q", sum(1 << (b - 1) for b in lists))]
    desc = h["description"].encode()
    out += [struct.pack("<Q", len(desc)), desc, struct.pack("<Q", len(allocs))]
    out += [struct.pack("<IIQQ", k, r, n, o) for k, r, n, o in allocs]
    out += [struct.pack("<Q", len(blob)), blob, struct.pack("<Q", len(lists))]
    for b in sorted(lists):
        out.append(struct.pack("<QQ", b, len(lists[b])))
        for name, args in lists[b]:
            out += [struct.pack("<I", len(name)), name.encode(), struct.pack("<I", len(args))]
            for tag, v in args:
                out.append(struct.pack("<II", tag, 0))
                if tag in (TAG_I32, TAG_I64):
                    out.append(struct.pack("<q", v))
                elif tag == TAG_F32:
                    out.append(struct.pack("<fI", v, 0))
                elif tag == TAG_PTR:
                    out.append(struct.pack("<QQ", NULL if v[0] is None else v[0], v[1]))
                elif tag in (TAG_HOST_I32, TAG_HOST_F32):
                    out += [struct.pack("<Q", len(v) // 4), v]
                elif tag == TAG_STRUCT:
                    raw, relocs = v
                    out += [struct.pack("<Q", len(raw)), raw, struct.pack("<Q", len(relocs))]
                    for field, alloc, off in relocs:
                        if alloc == HOST_REF:
                            out += [struct.pack("<QQQ", field, HOST_REF, len(off)), off]
                        else:
                            out.append(struct.pack("<QQQ", field, alloc, off))
    return b"".join(out)


# ---------------------------------------------------------------------------- recording
class _Registry:
    """Every allocation a launch may point into, by origin: (start, end, kind, role, tensor) per torch storage."""

    def __init__(self):
        self.spans = {}

    def add(self, t, kind, role=ROLE_NONE):
        if isinstance(t, dict):
            for v in t.values():
                self.add(v, kind, role)
            return
        if isinstance(t, (list, tuple)):
            for v in t:
                self.add(v, kind, role)
            return
        if not torch.is_tensor(t):
            return
        st = t.untyped_storage()
        start = st.data_ptr()
        if start not in self.spans and st.nbytes():            # first origin wins: inputs / outputs before scratch
            self.spans[start] = (start, start + st.nbytes(), kind, role, t)

    def freeze(self):
        self.sorted = sorted(self.spans.values())
        self.starts = [s[0] for s in self.sorted]

    def find(self, p):
        i = bisect.bisect_right(self.starts, p) - 1
        if i >= 0 and p < self.sorted[i][1]:
            return self.sorted[i]
        return None


class _Recorder:
    def __init__(self, registry):
        self.reg = registry
        self.ids = {}                 # storage start -> allocation id, in first-reference order
        self.allocs = []              # span per id
        self.ws_id, self.ws_bytes = None, 0
        self.launches = None

    def alloc_id(self, span):
        if span[0] not in self.ids:
            self.ids[span[0]] = len(self.allocs)
            self.allocs.append(span)
        return self.ids[span[0]]

    def ptr(self, p, op, what):
        if not p:
            return (None, 0)
        span = self.reg.find(p)
        if span is None:
            raise AvdfError("export_plan: %s %s: device pointer %#x is outside every registered allocation" % (op, what, p))
        return (self.alloc_id(span), p - span[0])

    def workspace(self, nbytes):
        if self.ws_id is None:
            self.ws_id = len(self.allocs)
            self.allocs.append(None)
        self.ws_bytes = max(self.ws_bytes, int(nbytes))
        return self.ws_id

    def struct(self, op, s):
        cls = type(s)
        raw = bytearray(ctypes.string_at(ctypes.addressof(s), ctypes.sizeof(s)))
        relocs = []
        for fname, ftype in cls._fields_:
            off = getattr(cls, fname).offset
            if ftype is c_void_p:
                fields = [(fname, off, getattr(s, fname))]
            elif issubclass(ftype, ctypes.Array) and ftype._type_ is c_void_p:
                fields = [("%s[%d]" % (fname, i), off + 8 * i, v) for i, v in enumerate(getattr(s, fname))]
            elif issubclass(ftype, ctypes._Pointer):
                v = getattr(s, fname)
                raw[off:off + 8] = bytes(8)
                if v:
                    rule = HOST_FIELDS.get((cls, fname))
                    if rule is None:
                        raise AvdfError("export_plan: %s field %s: host pointer without a length rule" % (op, fname))
                    relocs.append((off, HOST_REF, ctypes.string_at(v, rule(s))))
                continue
            else:
                continue
            for name, o, v in fields:
                raw[o:o + 8] = bytes(8)
                if not v:
                    continue
                if fname == "workspace":                # session scratch of the recorded size
                    relocs.append((o, self.workspace(s.workspace_bytes), 0))
                else:
                    a, ao = self.ptr(v, op, "field " + name)
                    relocs.append((o, a, ao))
        return bytes(raw), relocs

    def record(self, name, fn, args):
        op = fn.__name__
        types = fn.argtypes
        if len(types) != len(args) or types[-1] is not c_void_p:
            raise AvdfError("export_plan: %s: unexpected signature" % op)
        out = []
        for k, (t, v) in enumerate(zip(types, args)):
            if k == len(args) - 1:
                out.append((TAG_STREAM, None))
            elif t is c_void_p:
                out.append((TAG_PTR, self.ptr(v.value if isinstance(v, c_void_p) else v, op, "argument %d" % k)))
            elif t is c_int32:
                out.append((TAG_I32, int(v.value if isinstance(v, ctypes._SimpleCData) else v)))
            elif t is c_int64:
                out.append((TAG_I64, int(v.value if isinstance(v, ctypes._SimpleCData) else v)))
            elif t is c_float:
                out.append((TAG_F32, float(v.value if isinstance(v, ctypes._SimpleCData) else v)))
            elif t in (ctypes.POINTER(c_int32), ctypes.POINTER(c_float)) and isinstance(v, ctypes.Array):
                out.append((TAG_HOST_I32 if t is ctypes.POINTER(c_int32) else TAG_HOST_F32, bytes(v)))
            elif op in STRUCTS and t is ctypes.POINTER(STRUCTS[op]):
                out.append((TAG_STRUCT, self.struct(op, v._obj)))
            else:
                raise AvdfError("export_plan: %s argument %d: cannot record a %s" % (op, k, t))
        self.launches.append((op, out))


# ---------------------------------------------------------------------------- export
STREAM_NAMES = ("video", "byola", "emo")


def _stream_dims(model_cfg):
    """(video, byola, emo) channels of the raw streams: audio_input_dim is BYOL-A (2048) + emotion2vec (768), or one of them."""
    audio = int(model_cfg["audio_input_dim"])
    split = {2816: (2048, 768), 2048: (2048, 0), 768: (0, 768), 0: (0, 0)}.get(audio)
    if split is None:
        raise AvdfError("export_plan: audio_input_dim %d is not BYOL-A / emotion2vec; pass `items` with the streams" % audio)
    return (int(model_cfg["video_input_dim"]),) + split


def _synthetic_items(dims, n, seed):
    from ..utils import synthetic as syn
    durs = syn.sample_durations(n, seed)
    return [{"video_id": "plan%d" % i, "duration": float(d),
             "streams": syn.synthetic_streams(float(d), seed + i, video_dim=dims[0], byola_dim=dims[1], emo_dim=dims[2])}
            for i, d in enumerate(durs)]


def _stage_streams(items, streams):
    """Raw-stream items -> the stream staging, recordings back to back; returns the row offsets [3, B + 1]."""
    from .streaming import _stream_array
    B = len(items)
    off = np.zeros((3, B + 1), np.int64)
    for s, name in enumerate(STREAM_NAMES):
        if streams[s] is None:
            continue
        arrs = [_stream_array(c["streams"][name]) for c in items]
        off[s, 1:] = np.cumsum([a.shape[0] for a in arrs])
        if off[s, B] > streams[s].shape[0]:
            raise AvdfError("%s: %d rows, the staging holds %d" % (name, off[s, B], streams[s].shape[0]))
        cat = np.concatenate(arrs, axis=0)
        host = torch.from_numpy(cat.view(np.int16)).view(torch.bfloat16) if cat.dtype == np.uint16 else torch.from_numpy(cat)
        if host.dtype != streams[s].dtype:
            raise AvdfError("%s: %s rows for %s staging" % (name, host.dtype, streams[s].dtype))
        streams[s][:int(off[s, B])].copy_(host, non_blocking=False)
    return off


def _stage_items(items, streams, offsets, meta, t_out):
    """Raw-stream items -> the staging tensors (recordings back to back, row prefixes, meta [4, B]); returns rows."""
    from .streaming import _stream_array, video_meta
    B = len(items)
    off = np.zeros((3, offsets.shape[1]), np.int32)
    off[:, :B + 1] = _stage_streams(items, streams)
    rows = [int(off[s, B]) for s in range(3)]
    m = np.empty((4, B), np.float32)
    for b, c in enumerate(items):
        first = c["streams"]["video"] if streams[0] is not None else c["streams"]["byola"]
        m[:, b] = video_meta(c, _stream_array(first).shape[0], t_out)
    offsets.copy_(torch.from_numpy(off))
    meta[:4 * B].copy_(torch.from_numpy(m.reshape(-1)))
    return rows


@torch.no_grad()
def record_plan(model, batch_sizes=None, shards=False, max_seconds=36.0, items=None, seed=0):
    """Record the raw-stream pass of `model` for every batch size; returns (header, allocs, blob, lists) for encode_plan.
    items: raw-stream items that fill the staging while recording (their streams fix which streams the plan takes;
    default: seeded synthetic recordings of the config's stream dims)."""
    from ..utils import synthetic as syn
    from .streaming import bf16_shard
    if model.test_nms_method not in ("hard", "soft"):
        raise AvdfError("export_plan: nms_method %r returns every decoded candidate; a plan needs hard or soft NMS"
                        % (model.test_nms_method,))
    eng = model.engine()
    mb = eng.max_batch
    batch_sizes = sorted(set(int(b) for b in (batch_sizes or range(1, mb + 1))))
    if not batch_sizes or batch_sizes[0] < 1 or batch_sizes[-1] > mb:
        raise AvdfError("export_plan: batch sizes must lie in 1 .. max_batch (%d)" % mb)
    if items is not None:
        for c in items:
            if "streams" not in c:
                raise AvdfError("export_plan: plans run the raw-stream path; 'feats' items (host-dependent masks) cannot be recorded")
        dims = [c.shape[1] if (c := items[0]["streams"].get(n)) is not None else 0 for n in STREAM_NAMES]
    else:
        dims = list(_stream_dims(model.model_cfg))
        items = _synthetic_items(dims, mb, seed)
    if shards:
        items = [dict(c, streams={n: (a if np.asarray(a).dtype == np.uint16 else bf16_shard(a)) for n, a in c["streams"].items()})
                 for c in items]
    if sum(dims) != eng.c_in:
        raise AvdfError("export_plan: streams carry %d channels, the model expects %d" % (sum(dims), eng.c_in))
    dev = eng.device
    in_dt = torch.bfloat16 if shards else torch.float32
    fps = (syn.VIDEO_FPS, syn.BYOLA_FPS, syn.EMO_FPS)
    # input staging: a full batch of max_seconds-long recordings at the dataset stream rates (as _Slot.ensure sizes it)
    rows_cap = [int(mb * max_seconds * fps[s] * 1.05) + 64 if dims[s] else 0 for s in range(3)]
    with torch.cuda.device(dev):
        streams = [torch.zeros((rows_cap[s], dims[s]), dtype=in_dt, device=dev) if dims[s] else None for s in range(3)]
        offsets = torch.zeros((3, mb + 1), dtype=torch.int32, device=dev)
        meta = torch.zeros(4 * mb, dtype=torch.float32, device=dev)

    def staged(B):
        batch = [items[i % len(items)] for i in range(B)]
        _stage_items(batch, streams, offsets, meta, eng.max_seq_len)
        return {"ids": [c["video_id"] for c in batch], "B": B, "meta": meta[:4 * B].view(4, B),
                "streams": streams, "offs": [offsets[s, :B + 1] if dims[s] else None for s in range(3)]}

    # warm-up: every lazily built constant (packed weights, folded MLP weights, mask / PE tables, FPN parameters) exists
    # before the recording; the mask cache is cleared so that no eviction can free a table a recorded launch points at
    eng._mask_cache.clear()
    res = None
    for B in batch_sizes:
        res = model.run_staged(staged(B))
    torch.cuda.synchronize(dev)
    reg = _Registry()
    for s, role in zip(range(3), (ROLE_VIDEO, ROLE_BYOLA, ROLE_EMO)):
        reg.add(streams[s], KIND_INPUT, role)
    reg.add(offsets, KIND_INPUT, ROLE_OFFSETS)
    reg.add(meta, KIND_INPUT, ROLE_META)
    for k, role in (("segs", ROLE_SEGS), ("scores", ROLE_SCORES), ("counts", ROLE_COUNTS), ("vcls", ROLE_VCLS)):
        reg.add(res[k], KIND_OUTPUT, role)
    reg.add(eng._bufs, KIND_SCRATCH)
    reg.add(eng._ws or {}, KIND_SCRATCH)
    reg.add(eng.w._cache, KIND_CONST)
    reg.add(eng._mask_cache, KIND_CONST)
    reg.add(eng._pe_cache, KIND_CONST)
    reg.add(getattr(eng, "_fpn_params", None), KIND_CONST)
    reg.freeze()
    rec = _Recorder(reg)
    # io allocations first, in role order: present whether or not a launch reads them
    for span in sorted((sp for sp in reg.sorted if sp[3] != ROLE_NONE), key=lambda sp: sp[3]):
        rec.alloc_id(span)
    lists = {}
    orig = ops._call_on_current

    def recording(name, fn, args, launches, work):
        rec.record(name, fn, args)
        return orig(name, fn, args, launches, work)

    ops._call_on_current = recording
    try:
        for B in batch_sizes:
            st = staged(B)
            rec.launches = []
            model.run_staged(st)
            lists[B] = rec.launches
    finally:
        ops._call_on_current = orig
    torch.cuda.synchronize(dev)

    # allocations: constants get their bytes in the blob (256-aligned), the rest are session memory
    allocs, blob = [], bytearray()
    for span in rec.allocs:
        if span is None:                  # the shared workspace
            allocs.append((KIND_WORKSPACE, ROLE_NONE, max(rec.ws_bytes, 1), 0))
            continue
        start, end, kind, role, t = span
        if kind == KIND_CONST:
            off = len(blob)
            raw = torch.empty(end - start, dtype=torch.uint8)
            raw.untyped_storage().copy_(t.untyped_storage())
            blob += raw.numpy().tobytes()
            blob += bytes(_align(len(blob)) - len(blob))
            allocs.append((KIND_CONST, ROLE_NONE, end - start, off))
        else:
            allocs.append((kind, role, end - start, 0))
    sms, ccma, ccmi = c_int32(), c_int32(), c_int32()
    with torch.cuda.device(dev):
        nv.check(nv.lib().avdf_device_info(ctypes.byref(sms), ctypes.byref(ccma), ctypes.byref(ccmi)), "avdf_device_info")
    switches = " ".join("%s=%d" % (env, int(getattr(eng, attr))) for env, attr in SWITCHES)
    desc = "model=%s precision=%s test_cfg=%s %s" % (model.MODEL_NAME, eng.precision,
                                                     dict(zip(model._TEST_ATTRS, model.test_key())), switches)
    header = dict(cc_major=ccma.value, cc_minor=ccmi.value, sm_count=sms.value, max_batch=mb,
                  max_seg_num=int(model.test_max_seg_num), t_out=eng.max_seq_len,
                  in_dtype=nv.DTYPE_BF16 if shards else nv.DTYPE_F32, channels=dims, stream_rows=rows_cap,
                  description=desc[:1023])
    return header, allocs, bytes(blob), lists


def export_plan(model, path, batch_sizes=None, shards=False, max_seconds=36.0, items=None):
    """Record `model`'s raw-stream pass for `batch_sizes` (default 1 .. max_batch) and write the plan file `path`
    (include/avdf.h, "the whole model"). shards: the plan takes bf16 streams (16-bit feature shards). Nothing is
    written when the recording fails."""
    data = encode_plan(*record_plan(model, batch_sizes, shards, max_seconds, items))
    tmp = path + ".tmp"
    with open(tmp, "wb") as f:
        f.write(data)
    os.replace(tmp, path)
    return path


# ---------------------------------------------------------------------------- replay through ctypes
class Plan:
    """An opened plan with its constants on `device`."""

    def __init__(self, path, device="cuda"):
        L = nv.lib()
        self.L, self.h = L, c_void_p()
        nv.check(L.avdf_plan_open(os.fsencode(path), ctypes.byref(self.h)), "avdf_plan_open")
        self.info = nv.PlanInfo()
        nv.check(L.avdf_plan_get_info(self.h, ctypes.byref(self.info)), "avdf_plan_get_info")
        self.device = torch.device(device)
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        with torch.cuda.device(self.device):
            self.consts = torch.empty(max(self.info.const_bytes, 1), dtype=torch.uint8, device=self.device)
            nv.check(L.avdf_plan_upload(self.h, self.consts.data_ptr(), self.info.const_bytes,
                                        c_void_p(torch.cuda.current_stream().cuda_stream)), "avdf_plan_upload")
            torch.cuda.current_stream().synchronize()
        self.sessions = []

    def session(self):
        s = PlanSession(self)
        self.sessions.append(s)
        return s

    def close(self):
        for s in self.sessions:
            s.close()
        if self.h:
            self.L.avdf_plan_close(self.h)
            self.h = c_void_p()


class PlanSession:
    """One buffer set of a plan: inputs / outputs as torch views of the session arena, and a stream of its own (graph
    capture needs a created stream)."""

    def __init__(self, plan):
        self.plan, info, L = plan, plan.info, plan.L
        self.h = c_void_p()
        with torch.cuda.device(plan.device):
            self.stream = torch.cuda.Stream()
            self.arena = torch.empty(max(info.session_bytes, 1), dtype=torch.uint8, device=plan.device)
            nv.check(L.avdf_session_create(plan.h, self.arena.data_ptr(), info.session_bytes, ctypes.byref(self.h)),
                     "avdf_session_create")
        io = nv.SessionIO()
        nv.check(L.avdf_session_get_io(self.h, ctypes.byref(io)), "avdf_session_get_io")
        mb, K = info.max_batch, info.max_seg_num
        in_dt = torch.float32 if info.in_dtype == nv.DTYPE_F32 else torch.bfloat16
        self.streams = [self._view(io.streams[s], (info.stream_rows[s], info.channels[s]), in_dt) if info.channels[s] else None
                        for s in range(3)]
        self.offsets = self._view(io.offsets, (3, mb + 1), torch.int32)
        self.meta = self._view(io.meta, (4 * mb,), torch.float32)
        self.segs = self._view(io.segs, (mb, K, 2), torch.float32)
        self.scores = self._view(io.scores, (mb, K), torch.float32)
        self.counts = self._view(io.counts, (mb,), torch.int32)
        self.vcls = self._view(io.video_cls, (mb,), torch.float32)
        self.win_block = None                 # device block of attach_windows

    def _view(self, p, shape, dtype):
        off = p - self.arena.data_ptr()
        n = int(np.prod(shape)) * torch.tensor([], dtype=dtype).element_size()
        return self.arena[off:off + n].view(dtype).view(shape)

    def stage(self, items):
        """Raw-stream items -> the session's inputs (copies on the session's stream); returns the rows per stream."""
        with torch.cuda.device(self.plan.device), torch.cuda.stream(self.stream):
            return _stage_items(items, self.streams, self.offsets, self.meta, self.plan.info.t_out)

    def launch(self, batch, rows, stream=None):
        """avdf_session_run on `stream` (default: the session's stream); asynchronous."""
        st = stream if stream is not None else self.stream
        r = (c_int64 * 3)(*[int(v) for v in rows])
        with torch.cuda.device(self.plan.device):
            rc = self.plan.L.avdf_session_run(self.h, int(batch), r, c_void_p(st.cuda_stream))
        nv.check(rc, "avdf_session_run")

    def results(self, ids):
        """The outputs of the last batch as the list of dicts forward_streams returns (synchronises)."""
        B = len(ids)
        torch.cuda.synchronize(self.plan.device)
        segs, scores, counts, vcls = (t[:B].cpu() for t in (self.segs, self.scores, self.counts, self.vcls))
        return [{"video_id": vid, "segments": segs[b, :int(counts[b])], "scores": scores[b, :int(counts[b])],
                 "labels": torch.zeros(int(counts[b]), dtype=torch.long), "video_cls": vcls[b:b + 1]}
                for b, vid in enumerate(ids)]

    def run(self, items, stream=None):
        rows = self.stage(items)
        self.launch(len(items), rows, stream)
        return self.results([c["video_id"] for c in items])

    def attach_windows(self, max_windows, max_windows_per_recording):
        """Give the session a window block (a torch device tensor) for run_windows calls with at most `max_windows`
        windows in all and `max_windows_per_recording` windows per recording."""
        L, mw, per = self.plan.L, int(max_windows), int(max_windows_per_recording)
        n = L.avdf_session_window_bytes(self.plan.h, mw, per)
        if n == 0:
            raise AvdfError("avdf_session_window_bytes failed: %s" % L.avdf_last_error().decode())
        with torch.cuda.device(self.plan.device):
            block = torch.empty(n, dtype=torch.uint8, device=self.plan.device)
            nv.check(L.avdf_session_attach_windows(self.h, block.data_ptr(), n, mw, per), "avdf_session_attach_windows")
        self.win_block = block
        return n

    def launch_windows(self, durations, rows, window, hop, outs, stream=None):
        """avdf_session_run_windows over recordings already staged (rows: [n_rec][3]) into outs = (segs [R, K, 2],
        scores [R, K], counts [R], video_cls [R]) on `stream` (default: the session's stream); asynchronous."""
        R = len(durations)
        a = nv.WindowRunArgs()
        dur = (ctypes.c_double * max(R, 1))(*[float(d) for d in durations])
        rws = (c_int64 * max(3 * R, 3))(*[int(v) for r in rows for v in r])
        a.n_rec, a.duration, a.rows, a.window, a.hop = R, dur, rws, float(window), float(hop)
        a.out_segs, a.out_scores, a.out_count, a.out_cls = (t.data_ptr() for t in outs)
        st = stream if stream is not None else self.stream
        with torch.cuda.device(self.plan.device):
            rc = self.plan.L.avdf_session_run_windows(self.h, ctypes.byref(a), c_void_p(st.cuda_stream))
        nv.check(rc, "avdf_session_run_windows")

    def run_windows(self, items, window, hop=None):
        """Sliding windows over raw-stream recordings of any length (hop defaults to window / 2): the same list of
        dicts as model.forward_streams(items, window=window, hop=hop). All recordings go into the stream staging at
        once, so their rows must fit it (export_plan's max_seconds); their windows may exceed max_batch."""
        W = float(window)
        H = W / 2.0 if hop is None else float(hop)
        R, K = len(items), self.plan.info.max_seg_num
        with torch.cuda.device(self.plan.device), torch.cuda.stream(self.stream):
            off = _stage_streams(items, self.streams)
        rows = (off[:, 1:] - off[:, :-1]).T.tolist()
        dev = self.plan.device
        outs = (torch.empty((R, K, 2), dtype=torch.float32, device=dev), torch.empty((R, K), dtype=torch.float32, device=dev),
                torch.empty((R,), dtype=torch.int32, device=dev), torch.empty((R,), dtype=torch.float32, device=dev))
        self.launch_windows([c["duration"] for c in items], rows, W, H, outs)
        torch.cuda.synchronize(dev)
        segs, scores, counts, vcls = (t.cpu() for t in outs)
        return [{"video_id": c["video_id"], "segments": segs[r, :int(counts[r])], "scores": scores[r, :int(counts[r])],
                 "labels": torch.zeros(int(counts[r]), dtype=torch.long), "video_cls": vcls[r:r + 1]}
                for r, c in enumerate(items)]

    def close(self):
        if self.h:
            self.plan.L.avdf_session_destroy(self.h)
            self.h = c_void_p()
        self.win_block = None


# ---------------------------------------------------------------------------- CLI
def main(argv=None):
    from ..core import load_config
    from . import make_meta_arch
    p = argparse.ArgumentParser(description="Export a launch plan of the raw-stream pass (replayed by libavdf_sm100.so's "
                                            "avdf_session_run)")
    p.add_argument("config", help="config file (the one inference.py takes)")
    p.add_argument("ckpt", help="checkpoint with a 'state_dict_ema' entry")
    p.add_argument("out", help="plan file to write")
    p.add_argument("--precision", default="mixed", choices=("mixed", "fp32"))
    p.add_argument("--shards", action="store_true", help="the plan takes bf16 streams (16-bit feature shards)")
    p.add_argument("--batch-sizes", type=int, nargs="+", default=None, help="default: 1 .. --max-batch")
    p.add_argument("--max-batch", type=int, default=32)
    p.add_argument("--max-seconds", type=float, default=36.0,
                   help="input staging: a full batch of recordings this long (sliding windows over long recordings "
                        "stage all of a call's recordings at once)")
    a = p.parse_args(argv)
    cfg = load_config(a.config)
    model = make_meta_arch(cfg["model_name"], **cfg["model"], precision=a.precision, max_batch=a.max_batch)
    ckpt = torch.load(a.ckpt, map_location="cpu")
    model.load_state_dict(ckpt["state_dict_ema"])
    del ckpt
    model.to(torch.device(cfg["devices"][0])).eval()
    export_plan(model, a.out, batch_sizes=a.batch_sizes, shards=a.shards, max_seconds=a.max_seconds)
    print("wrote %s (%d bytes)" % (a.out, os.path.getsize(a.out)))
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
