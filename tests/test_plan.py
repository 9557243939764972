"""CPU-side checks of launch plans (libs/modeling/plan.py, csrc/plan.cu): a plan serialised from a hand-built launch list
opens through avdf_plan_open without a GPU and reports what was written; every malformed file fails with its own message
and no crash; every entry point the raw-stream pass reaches has an adapter in the library, and every pointer field of
its args structs is relocated or has a length rule."""
import ctypes
import os
import re
import struct

import pytest
import torch

from audio_visual_deepfake_detection_b200 import native as nv
from audio_visual_deepfake_detection_b200.libs.modeling import plan as pl

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "audio_visual_deepfake_detection_b200")

MB, K = 2, 3
HEADER = dict(cc_major=10, cc_minor=0, sm_count=148, max_batch=MB, max_seg_num=K, t_out=16, in_dtype=nv.DTYPE_F32,
              channels=[0, 0, 4], stream_rows=[0, 0, 10], description="model=hand-built precision=fp32")
# io allocations (ids 0..7), one constant (8, 1 KB at blob offset 256), one scratch buffer (9)
ALLOCS = [(pl.KIND_INPUT, pl.ROLE_EMO, 10 * 4 * 4, 0), (pl.KIND_INPUT, pl.ROLE_OFFSETS, 3 * (MB + 1) * 4, 0),
          (pl.KIND_INPUT, pl.ROLE_META, 4 * MB * 4, 0), (pl.KIND_OUTPUT, pl.ROLE_SEGS, MB * K * 8, 0),
          (pl.KIND_OUTPUT, pl.ROLE_SCORES, MB * K * 4, 0), (pl.KIND_OUTPUT, pl.ROLE_COUNTS, MB * 4, 0),
          (pl.KIND_OUTPUT, pl.ROLE_VCLS, MB * 4, 0), (pl.KIND_CONST, pl.ROLE_NONE, 1024, 256),
          (pl.KIND_SCRATCH, pl.ROLE_NONE, 4096, 0)]
CONST, SCRATCH = 7, 8


def conv_gemm_struct(tap_rows=None):
    g = nv.ConvGemmArgs()
    g.batch, g.n_out, g.c_in, g.taps, g.stride, g.n_seg = 1, 4, 4, 3, 1, 1
    raw = bytes(ctypes.string_at(ctypes.addressof(g), ctypes.sizeof(g)))
    relocs = [(nv.ConvGemmArgs.a.offset, SCRATCH, 0), (nv.ConvGemmArgs.w.offset, CONST, 64),
              (nv.ConvGemmArgs.out_f32.offset, SCRATCH, 1024)]
    if tap_rows is not None:
        relocs.append((nv.ConvGemmArgs.tap_rows.offset, pl.HOST_REF, tap_rows))
    return raw, relocs


def ln_rows(x_off=0):
    return ("avdf_ln_rows", [(pl.TAG_PTR, (SCRATCH, x_off)), (pl.TAG_PTR, (CONST, 0)), (pl.TAG_PTR, (CONST, 16)),
                             (pl.TAG_PTR, (SCRATCH, 2048)), (pl.TAG_I32, nv.DTYPE_F32), (pl.TAG_I64, 4), (pl.TAG_I32, 4),
                             (pl.TAG_STREAM, None)])


def fpn_fuse(n_levels=2, level_len=(4, 2)):
    return ("avdf_fpn_fuse", [(pl.TAG_PTR, (SCRATCH, 0)), (pl.TAG_PTR, (SCRATCH, 512)), (pl.TAG_PTR, (CONST, 0)),
                              (pl.TAG_PTR, (CONST, 128)), (pl.TAG_PTR, (CONST, 256)), (pl.TAG_PTR, (SCRATCH, 1024)),
                              (pl.TAG_I32, nv.DTYPE_F32), (pl.TAG_I32, 1), (pl.TAG_I32, 4), (pl.TAG_I32, n_levels),
                              (pl.TAG_HOST_I32, struct.pack("<%di" % len(level_len), *level_len)), (pl.TAG_STREAM, None)])


def lists(**over):
    cg = ("avdf_conv_gemm", [(pl.TAG_STRUCT, over.get("struct", conv_gemm_struct())), (pl.TAG_STREAM, None)])
    return {1: [over.get("first", ln_rows()), cg], 2: [cg, over.get("fpn", fpn_fuse()), ln_rows()]}


def encode(header=None, allocs=None, **over):
    return pl.encode_plan(dict(HEADER, **(header or {})), allocs or ALLOCS, bytes(256) + bytes(range(256)) * 4, lists(**over))


def open_plan(data, tmp_path):
    path = tmp_path / "p.avdfplan"
    path.write_bytes(data)
    L = nv.lib()
    h = ctypes.c_void_p()
    rc = L.avdf_plan_open(os.fsencode(str(path)), ctypes.byref(h))
    msg = L.avdf_last_error().decode()
    if rc == 0:
        info = nv.PlanInfo()
        assert L.avdf_plan_get_info(h, ctypes.byref(info)) == 0
        L.avdf_plan_close(h)
        return rc, info
    assert not h.value
    return rc, msg


def test_hand_built_plan_opens_without_a_gpu(tmp_path):
    rc, info = open_plan(encode(struct=conv_gemm_struct(tap_rows=struct.pack("<3i", -1, 0, 1))), tmp_path)
    assert rc == 0
    assert (info.abi_version, info.cc_major, info.cc_minor, info.sm_count) == (3, 10, 0, 148)
    assert (info.max_batch, info.max_seg_num, info.t_out, info.in_dtype) == (MB, K, 16, nv.DTYPE_F32)
    assert list(info.channels) == [0, 0, 4] and list(info.stream_rows) == [0, 0, 10]
    assert info.batch_mask == 0b11
    assert info.const_bytes == 256 + 1024
    assert info.session_bytes == sum(pl._align(n) for k, _, n, _ in ALLOCS if k != pl.KIND_CONST)
    assert info.description == b"model=hand-built precision=fp32"


@pytest.mark.parametrize("case,data,message", [
    ("magic", lambda: b"AVDFPLAX" + encode()[8:], "bad magic"),
    ("version", lambda: encode()[:8] + struct.pack("<I", 2) + encode()[12:], "unsupported format version 2"),
    ("abi", lambda: encode()[:12] + struct.pack("<I", 2) + encode()[16:], "ABI version 2"),
    ("entry_point", lambda: encode(first=("avdf_ln_rowz", ln_rows()[1])), "unknown entry point 'avdf_ln_rowz'"),
    ("scalar_tag", lambda: encode(first=("avdf_ln_rows", ln_rows()[1][:4] + [(pl.TAG_F32, 1.0)] + ln_rows()[1][5:])),
     "avdf_ln_rows argument 4: type tag 3, expected 'I'"),
    ("pointer", lambda: encode(first=ln_rows(x_off=4096)), "relocation outside its allocation (offset 4096, allocation 8"),
    ("struct_reloc", lambda: encode(struct=(conv_gemm_struct()[0], [(nv.ConvGemmArgs.w.offset, CONST, 1024)])),
     "avdf_conv_gemm relocation 0: relocation outside its allocation"),
    ("alloc_id", lambda: encode(first=("avdf_ln_rows", [(pl.TAG_PTR, (10, 0))] + ln_rows()[1][1:])), "allocation 10 does not exist"),
    ("struct_size", lambda: encode(struct=(conv_gemm_struct()[0] + bytes(8), [])), "avdf_conv_gemm: struct size"),
    ("host_length", lambda: encode(struct=conv_gemm_struct(tap_rows=struct.pack("<2i", 0, 1))), "tap_rows: 8 bytes for 3 taps"),
    ("host_array", lambda: encode(fpn=fpn_fuse(n_levels=3)), "avdf_fpn_fuse argument 10: host array of 2 elements"),
    ("io", lambda: encode(allocs=ALLOCS[1:]), "io role 3: missing"),
    ("trailing", lambda: encode() + b"\0", "1 trailing bytes"),
])
def test_malformed_plans_fail_with_their_own_message(case, data, message, tmp_path):
    rc, msg = open_plan(data(), tmp_path)
    assert rc == -1, case
    assert message in msg, (case, msg)


def test_truncated_files_fail_and_never_crash(tmp_path):
    data = encode()
    for n in list(range(0, 200, 3)) + list(range(200, len(data), 37)) + [len(data) - 1]:
        rc, msg = open_plan(data[:n], tmp_path)
        assert rc == -1 and "truncated file" in msg, (n, msg)


def test_recorder_relocates_struct_pointers_and_names_unknown_ones():
    """The exporter's struct rule on host tensors: device pointer fields become (allocation, offset) relocations, the
    workspace becomes session scratch, the host tap table is stored by value, and a foreign pointer names op and field."""
    a, w, ws = torch.zeros(64), torch.zeros(32), torch.zeros(16)
    reg = pl._Registry()
    reg.add(a, pl.KIND_SCRATCH)
    reg.add({"w": w}, pl.KIND_CONST)
    reg.freeze()
    rec = pl._Recorder(reg)
    g = nv.ConvGemmArgs()
    g.taps = 3
    g.a, g.w, g.out_f32 = a.data_ptr() + 16, w.data_ptr(), a.data_ptr() + 128
    g.workspace, g.workspace_bytes = ws.data_ptr(), 64
    taps = (ctypes.c_int32 * 3)(-7, 0, 7)
    g.tap_rows = taps
    raw, relocs = rec.struct("avdf_conv_gemm", g)
    assert len(raw) == ctypes.sizeof(g) and raw[nv.ConvGemmArgs.a.offset:nv.ConvGemmArgs.a.offset + 8] == bytes(8)
    rel = {f: (al, o) for f, al, o in relocs}
    assert rel[nv.ConvGemmArgs.a.offset] == (0, 16) and rel[nv.ConvGemmArgs.w.offset] == (1, 0)
    assert rel[nv.ConvGemmArgs.out_f32.offset] == (0, 128)
    assert rel[nv.ConvGemmArgs.workspace.offset] == (2, 0) and rec.ws_bytes == 64 and rec.allocs[2] is None
    assert rel[nv.ConvGemmArgs.tap_rows.offset] == (pl.HOST_REF, struct.pack("<3i", -7, 0, 7))
    g.residual = torch.zeros(4).data_ptr()
    with pytest.raises(nv.AvdfError, match="avdf_conv_gemm field residual: device pointer"):
        rec.struct("avdf_conv_gemm", g)
    e = nv.EvalArgs()
    e.thresholds = (ctypes.c_double * 1)(0.5)
    with pytest.raises(nv.AvdfError, match="field thresholds: host pointer without a length rule"):
        rec.struct("avdf_eval_detection", e)


def _ops_calls(path, func=None):
    src = open(path).read()
    if func is not None:
        m = re.search(r"\n    def %s\(.*?(?=\n    (?:@|def ))" % func, src, flags=re.S)
        src = m.group(0)
    return set(re.findall(r"\bops\.([a-z_0-9]+)\(", src))


def test_every_entry_point_of_the_raw_stream_pass_has_an_adapter():
    engine = os.path.join(PKG, "libs", "modeling", "engine.py")
    reached = _ops_calls(engine) | _ops_calls(os.path.join(PKG, "libs", "modeling", "meta_archs.py"), "run_staged")
    reached -= {"interp_concat_ranges"}          # sliding windows: not part of a plan
    ops_src = open(os.path.join(PKG, "ops.py")).read()
    plan_src = open(os.path.join(PKG, "csrc", "plan.cu")).read()
    table = set(re.findall(r'\{"(avdf_[a-z0-9_]+)", "[A-Z]+"', plan_src))
    assert len(reached) >= 12
    for op in sorted(reached):
        body = re.search(r"\ndef %s\(.*?(?=\ndef )" % op, ops_src, flags=re.S).group(0)
        entry = re.findall(r"_call\(\"[a-z_0-9]+\", L\.(avdf_[a-z_0-9]+)", body)
        assert entry, op
        assert entry[0] in table, "ops.%s -> %s has no adapter in csrc/plan.cu" % (op, entry[0])
        assert "case OP_" in plan_src and entry[0] + "(" in plan_src, entry[0]
    # every pointer slot of every args struct a plan carries comes out as a relocation (device) or by value (host)
    buf = torch.zeros(4096, dtype=torch.uint8)
    reg = pl._Registry()
    reg.add(buf, pl.KIND_SCRATCH)
    reg.freeze()
    for name, cls in pl.STRUCTS.items():
        assert name in table
        s, slots, host = cls(), 0, ctypes.c_int32(0)
        for fname, ftype in cls._fields_:
            if ftype is ctypes.c_void_p:
                setattr(s, fname, buf.data_ptr() + 8 * slots)
                slots += 1
            elif issubclass(ftype, ctypes.Array) and ftype._type_ is ctypes.c_void_p:
                for i in range(len(getattr(s, fname))):
                    getattr(s, fname)[i] = buf.data_ptr() + 8 * slots
                    slots += 1
            elif issubclass(ftype, ctypes._Pointer):
                assert (cls, fname) in pl.HOST_FIELDS, "%s.%s: host pointer without a length rule" % (cls.__name__, fname)
                setattr(s, fname, ctypes.cast(ctypes.pointer(host), ftype))
                slots += 1
        if hasattr(s, "taps"):
            s.taps = 1
        _, relocs = pl._Recorder(reg).struct(name, s)
        assert len(relocs) == slots and len({f for f, _, _ in relocs}) == slots, name
