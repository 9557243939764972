"""Host <-> device pipeline of the raw-stream entry point (`model.forward_streams`, `model.stream`).

Per batch of <= max_batch videos:
  pack   (host threads)  (skipped when the caller's arrays are page-locked: `avdf_h2d_gather` then copies them to the
                         device where they are) every video's [T_s, C_s] fp32 arrays are gathered into ONE pinned buffer per stream by
                         `avdf_host_pack` (the library's own thread pool; row offsets + per-video metadata alongside)
  H2D    (copy engine)   pinned -> static device staging buffers, asynchronous on the compute stream
  GPU                    the whole pass (interp/concat -> model -> decode -> NMS) replayed as ONE CUDA graph
  D2H                    fixed-size results -> pinned host, then an event
n_slots (default 6, env AVDF_STREAM_SLOTS; round 2, one GPU: 4 / 6 / 10 slots = 17.7k / 19.5k / 19.1k videos/s end to end) staging slots rotate: one is being packed while up to n_slots-1 batches are in flight on the
GPU, each on its own stream and engine lane (buffer set), so copies and kernels of consecutive batches overlap. This replaces the
reference's DataLoader workers (which run F.interpolate on the CPU, libs/datasets/deepfake_video_audio.py:513-547)
plus the per-video `.to(device)` / `.cpu()` of libs/modeling/av_fd_no_recon.py:476-477, 841-846.
"""
import ctypes
import os
import queue
import threading

import numpy as np
import torch

from ... import native, ops

STREAMS = ("video", "byola", "emo")


def bf16_shard(a):
    """fp32 array -> the opt-in 16-bit feature-shard format: bf16 bit patterns (round to nearest even) in a uint16 array of
    the same shape. Arrays of this dtype are accepted wherever raw streams are (`model.stream`, `forward_streams`,
    `collate_pinned`): half the host -> device bytes per video; the GPU resampling reads bf16 and computes in fp32."""
    u = np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)
    r = ((u >> 16) & 1) + np.uint32(0x7FFF)
    return ((u + r) >> 16).astype(np.uint16)


def _stream_array(x):
    """numpy view of a raw-stream array: fp32, or uint16 holding bf16 bits (torch.bfloat16 tensors are viewed as such)."""
    if torch.is_tensor(x):
        x = x.view(torch.int16).numpy().view(np.uint16) if x.dtype == torch.bfloat16 else x.numpy()
    x = np.asarray(x)
    return x if x.dtype == np.uint16 else np.asarray(x, dtype=np.float32)


def collate_pinned(chunk):
    """A batch of raw-stream items ({video_id, duration, streams: {name: [T, C] fp32}}) re-homed in ONE page-locked block,
    laid out stream-major (every video's rows of stream 0, then stream 1, ...) - the layout the interp/concat kernel reads on
    the device. `StreamRunner` recognises page-locked sources and copies them where they are; with this layout a batch
    leaves as one host->device copy per stream (avdf_h2d_gather merges adjacent spans). This is the collate step of a
    loader that feeds `model.stream()` (the reference collates in DataLoader workers and pins per tensor,
    libs/datasets/datasets.py:27-43)."""
    names = [n for n in STREAMS if n in chunk[0]["streams"]]
    arrs = {n: [_stream_array(c["streams"][n]) for c in chunk] for n in names}
    dt = arrs[names[0]][0].dtype                   # float32, or uint16 = bf16 shards (bf16_shard)
    total = sum(a.size for n in names for a in arrs[n])
    block = torch.empty(total, dtype=torch.float32 if dt == np.float32 else torch.int16, pin_memory=torch.cuda.is_available()).numpy().view(dt)
    pos, views = 0, [dict() for _ in chunk]
    for n in names:
        for b, a in enumerate(arrs[n]):
            v = block[pos:pos + a.size].reshape(a.shape)
            v[...] = a
            views[b][n] = v
            pos += a.size
    return [{**c, "streams": views[b]} for b, c in enumerate(chunk)]


def video_meta(c, t_first, L, feat_stride=1, num_frames=1):
    """(feat_stride, 0.5 * feat_num_frames, fps, duration) of one raw-stream item as fp32, i.e. the scalars
    av_fd_no_recon.py:860-865 feeds into its fp32 tensor expression. An item that carries the dataset's own
    'feat_stride' / 'feat_num_frames' / 'fps' (libs/datasets/deepfake_video_audio.py:461, 495-500) is taken at its word;
    otherwise they are derived the way the dataset derives them under force_upsampling from the length of the first
    stream and the dataset-level feat_stride / num_frames."""
    fs = c.get("feat_stride")
    if fs is None:
        fs = float((t_first - 1) * feat_stride + num_frames) / L        # deepfake_video_audio.py:495-497
    nf = c.get("feat_num_frames", fs)
    fps = c.get("fps")
    if fps is None:
        fps = t_first / c["duration"]
    return (np.float32(fs), np.float32(0.5 * nf), np.float32(fps), np.float32(c["duration"]))


class _Slot:
    def __init__(self, runner, index):
        self.runner, self.index = runner, index
        self.cap = [0, 0, 0]              # rows
        self.host = [None, None, None]
        self.dev = [None, None, None]
        self.graphs = {}                  # (batch size, test-time config) -> GraphedPass
        self.done = torch.cuda.Event()
        self.stream = torch.cuda.Stream(device=runner.eng.device)     # slots run on their own streams: copies and kernels of consecutive batches overlap
        self.ids, self.B, self.busy = None, 0, False
        self.direct = None                    # (src, device dst, nbytes, n, keep-alive) of a batch whose arrays are pinned

    def ensure(self, rows, chans, max_batch, K, device, seconds, dtype=torch.float32):
        """Staging capacity. The captured graph holds the device staging pointers, so growing them forces a
        re-capture: size them once for a full batch of MAX_SECONDS-long videos at this stream's frame rate (the
        AV-Deepfake1M test split tops out at 33 s) and grow (x1.5) only if a batch still exceeds that."""
        MAX_SECONDS = 36.0
        grown = False
        for s in range(3):
            if chans[s] == 0:
                continue
            if self.host[s] is None or rows[s] > self.cap[s] or self.host[s].dtype != dtype:
                rate = rows[s] / max(seconds, 1e-3)                       # rows per second of video for this stream
                want = int(max_batch * MAX_SECONDS * rate * 1.05) + 64 if self.host[s] is None else 0
                self.cap[s] = max(want, int(rows[s] * 1.5) + 64)
                self.host[s] = torch.empty((self.cap[s], chans[s]), dtype=dtype, pin_memory=True)
                self.dev[s] = torch.empty((self.cap[s], chans[s]), dtype=dtype, device=device)
                grown = True
        if not hasattr(self, "h_off"):
            self.h_off = torch.zeros((3, max_batch + 1), dtype=torch.int32, pin_memory=True)
            self.d_off = torch.zeros((3, max_batch + 1), dtype=torch.int32, device=device)
            self.h_meta = torch.zeros((4, max_batch), dtype=torch.float32, pin_memory=True)
            self.d_meta = torch.zeros((4, max_batch), dtype=torch.float32, device=device)
            self.h_segs = torch.zeros((max_batch, K, 2), dtype=torch.float32, pin_memory=True)
            self.h_scores = torch.zeros((max_batch, K), dtype=torch.float32, pin_memory=True)
            self.h_counts = torch.zeros((max_batch,), dtype=torch.int32, pin_memory=True)
            self.h_vcls = torch.zeros((max_batch,), dtype=torch.float32, pin_memory=True)
            self.h_vidx = torch.zeros((max_batch,), dtype=torch.int32, pin_memory=True)
            self.d_vidx = torch.zeros((max_batch,), dtype=torch.int32, device=device)
        if grown:
            self.graphs.clear()           # captured kernels hold the old staging pointers


class StreamRunner:
    def __init__(self, model, n_slots=None, n_threads=None):
        n_slots = n_slots or int(os.environ.get("AVDF_STREAM_SLOTS", "6"))      # batches in flight (measured 4 / 6 / 8 / 10 / 14: 17.7k / 19.6k / 19.3k / 19.1k / 19.1k videos/s)
        self.model = model
        self.eng = model.engine()
        with torch.cuda.device(self.eng.device):
            self.slots = [_Slot(self, i) for i in range(n_slots)]
        self.next = 0
        # copy workers: the host cores are shared by the ranks of a node (torchrun exports LOCAL_WORLD_SIZE)
        local_world = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))
        self.n_threads = n_threads or int(os.environ.get("AVDF_PACK_THREADS", "0")) or max(2, min(16, (os.cpu_count() or 4) // local_world))
        self.h2d_bytes = 0
        self.d2h_bytes = 0
        self.n_direct = 0            # batches whose (pinned) arrays went to the device without a staging copy
        self.use_graph = True
        self.cuda_lock = threading.Lock()    # staging (pinned / device) allocation vs. graph capture on the launching thread
        self.zero_copy = os.environ.get("AVDF_ZERO_COPY", "1") != "0"    # pinned source arrays go to the copy engine directly
        self.n_packers = int(os.environ.get("AVDF_PACKERS", "1"))
        self.records = None          # (ring, counter): device-side result records (see enable_records)   # packer threads (measured 1 / 2 / 3: 15.56k / 15.45k / 15.39k videos/s: the gather itself is already parallel)

    def enable_records(self, capacity):
        """Every video of the following batches appends one fixed-size fp32 record ([item['index'], count, video_cls,
        scores[K], segs[K][2]]) to a device ring of `capacity` rows, written by the postprocess kernel: the unit the
        multi-GPU gather moves (libs/utils/sharding.py). Returns (ring, counter); None switches records off."""
        if capacity is None:
            self.records = None
            return None
        K = int(self.model.test_max_seg_num)
        with torch.cuda.device(self.eng.device):
            ring = torch.zeros((max(1, int(capacity)), 3 + 3 * K), dtype=torch.float32, device=self.eng.device)
            ring[:, 0] = -1.0
            counter = torch.zeros(1, dtype=torch.int32, device=self.eng.device)
        self.records = (ring, counter)
        return self.records

    # ---------------------------------------------------------------- stages
    def _pack(self, slot, chunk, feat_stride=1, num_frames=1):
        eng, L = self.eng, self.eng.max_seq_len
        B = len(chunk)
        present = [n in chunk[0]["streams"] for n in STREAMS]
        arrs = [[_stream_array(c["streams"][n]) for c in chunk] if p else None for n, p in zip(STREAMS, present)]
        np_dt = next(al[0].dtype for al in arrs if al)            # float32, or uint16 = bf16 feature shards
        item = np_dt.itemsize
        rows = [sum(a.shape[0] for a in al) if al else 0 for al in arrs]
        chans = [al[0].shape[1] if al else 0 for al in arrs]
        if sum(chans) != eng.c_in:
            raise ValueError("streams carry %d channels, the model expects %d" % (sum(chans), eng.c_in))
        K = int(eng.test_cfg["max_seg_num"])
        with self.cuda_lock:
            slot.ensure(rows, chans, eng.max_batch, K, eng.device, sum(float(c["duration"]) for c in chunk),
                        torch.float32 if item == 4 else torch.bfloat16)
        off = slot.h_off.numpy()
        src, dst, nbytes = [], [], []
        for s in range(3):
            if arrs[s] is None:
                continue
            off[s, 0] = 0
            off[s, 1:B + 1] = np.cumsum([a.shape[0] for a in arrs[s]])
            base, row_bytes = slot.host[s].data_ptr(), chans[s] * item
            for b, a in enumerate(arrs[s]):
                if a.dtype != np_dt:
                    raise ValueError("a batch mixes fp32 streams and 16-bit shards")
                if not a.flags.c_contiguous:                                   # the .npy files are row-major; anything else is converted
                    a = arrs[s][b] = np.ascontiguousarray(a)
                if a.shape[1] != chans[s]:
                    raise ValueError("stream %s: video %d has %d channels, the batch has %d" % (STREAMS[s], b, a.shape[1], chans[s]))
                src.append(a.ctypes.data); dst.append(base + int(off[s, b]) * row_bytes); nbytes.append(a.nbytes)
        n = len(src)
        lib_ = native.lib()
        c_src, c_n = (ctypes.c_void_p * n)(*src), (ctypes.c_size_t * n)(*nbytes)
        slot.direct = None
        if self.zero_copy and lib_.avdf_host_all_pinned(c_src, c_n, n) == 1:
            # the caller's arrays are page-locked (e.g. a loader that reads .npy files into a pinned pool): the copy engine
            # reads them where they are - no staging copy, no host core touches the features
            dev_dst, k = [], 0
            for s in range(3):
                if arrs[s] is None:
                    continue
                dbase, row_bytes = slot.dev[s].data_ptr(), chans[s] * item
                dev_dst += [dbase + int(off[s, b]) * row_bytes for b in range(B)]
            slot.direct = (c_src, (ctypes.c_void_p * n)(*dev_dst), c_n, n, arrs)      # arrs: keeps the sources alive
            self.n_direct += 1
        else:
            # the gather runs on the library's own thread pool (csrc/host_pack.cu: 256 KB pieces, non-temporal stores);
            # ctypes releases the GIL for the call
            native.check(lib_.avdf_host_pack(c_src, (ctypes.c_void_p * n)(*dst), c_n, n, self.n_threads), "avdf_host_pack")
        meta = slot.h_meta.numpy()
        for b, c in enumerate(chunk):
            first = c["streams"]["video"] if present[0] else c["streams"]["byola"]
            meta[:, b] = video_meta(c, first.shape[0], L, feat_stride, num_frames)
        vidx = slot.h_vidx.numpy()
        for b, c in enumerate(chunk):
            vidx[b] = int(c.get("index", b))
        slot.rows, slot.chans, slot.B, slot.ids, slot.item = rows, chans, B, [c["video_id"] for c in chunk], item

    def _launch(self, slot, dense=None):
        with torch.cuda.device(self.eng.device):      # the caller's thread may have another device selected
            slot.stream.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(slot.stream):
                self._launch_on_stream(slot, dense)

    def _launch_on_stream(self, slot, dense=None):
        eng, B = self.eng, slot.B
        nbytes = 0
        if slot.direct is not None:
            c_src, c_dst, c_n, n, _ = slot.direct
            native.check(native.lib().avdf_h2d_gather(c_src, c_dst, c_n, n, native.stream_ptr()), "avdf_h2d_gather")
        for s in range(3):
            if slot.chans[s]:
                if slot.direct is None:
                    slot.dev[s][:slot.rows[s]].copy_(slot.host[s][:slot.rows[s]], non_blocking=True)
                nbytes += slot.rows[s] * slot.chans[s] * slot.item
        slot.d_off.copy_(slot.h_off, non_blocking=True)
        slot.d_meta.copy_(slot.h_meta, non_blocking=True)
        if self.records is not None:
            slot.d_vidx.copy_(slot.h_vidx, non_blocking=True)
        self.h2d_bytes += nbytes + slot.h_off.numel() * 4 + slot.h_meta.numel() * 4
        staged = {"ids": slot.ids, "B": B, "meta": slot.d_meta[:, :B] if B == eng.max_batch else slot.d_meta[:, :B].contiguous(),
                  "streams": [slot.dev[s] if slot.chans[s] else None for s in range(3)],
                  "offs": [slot.d_off[s, :B + 1] if slot.chans[s] else None for s in range(3)]}
        if self.records is not None:
            staged["records"], staged["vidx"] = self.records, slot.d_vidx[:B]
        if self.use_graph and B == eng.max_batch:
            # the test-time config and the record ring are baked into the captured launches
            key = (B, self.model.test_key(), None if self.records is None else self.records[0].data_ptr(), slot.item)
            g = slot.graphs.get(key)
            if g is None:
                with self.cuda_lock:
                    g = self.model.capture(staged, lane=slot.index)
                slot.graphs[key] = g
            res = g.replay()
        else:
            res = self.model.run_staged(staged, lane=slot.index)
        if dense is not None:         # copies of what the pass's post-processing read, after the pass, on this stream
            logits, offsets = res["dense"]
            eng.keep_dense(dense, slot.ids, eng.max_seq_len, logits, offsets, res["vcls"], staged["meta"], [eng.max_seq_len] * B)
        if res["segs"].shape[1] != slot.h_segs.shape[1]:      # nms_method 'none': every decoded candidate comes back
            n_out = res["segs"].shape[1]
            slot.h_segs = torch.zeros((eng.max_batch, n_out, 2), dtype=torch.float32, pin_memory=True)
            slot.h_scores = torch.zeros((eng.max_batch, n_out), dtype=torch.float32, pin_memory=True)
        slot.h_segs[:B].copy_(res["segs"], non_blocking=True)
        slot.h_scores[:B].copy_(res["scores"], non_blocking=True)
        slot.h_counts[:B].copy_(res["counts"], non_blocking=True)
        slot.h_vcls[:B].copy_(res["vcls"], non_blocking=True)
        self.d2h_bytes += B * (slot.h_segs.shape[1] * 3 + 2) * 4
        slot.done.record()
        slot.busy = True

    def _collect(self, slot):
        slot.done.synchronize()
        slot.busy = False
        slot.direct = None                # the copy engine is done with the caller's arrays
        B = slot.B
        # one clone per result array (the pinned buffers are reused by the next batch), then cheap per-video views
        segs, scores, vcls = slot.h_segs[:B].clone(), slot.h_scores[:B].clone(), slot.h_vcls[:B].clone()
        counts = slot.h_counts[:B].tolist()
        empty_labels = torch.zeros(segs.shape[1], dtype=torch.long)
        return [{"video_id": vid, "segments": segs[b, :n], "scores": scores[b, :n], "labels": empty_labels[:n],
                 "video_cls": vcls[b:b + 1]} for b, (vid, n) in enumerate(zip(slot.ids, counts))]

    # ---------------------------------------------------------------- sliding windows (libs/modeling/windows.py)
    # A group of recordings is copied to the device ONCE (one pinned pack, one copy per stream); its windows - and its
    # recordings no longer than the window, as single windows - are packed in order into batches of max_batch that
    # read their rows through avdf_interp_concat_ranges, full batches by replaying a captured graph. Every window's
    # result is copied aside on the device, and avdf_window_merge turns them into one result (and optionally one
    # record) per recording. The only host synchronisation of a group is the final copy of its results.
    GROUP_BYTES = 1 << 30             # raw-stream bytes per group (at least one recording): bounds the pinned / device staging

    def run_windows(self, items, window, hop=None, feat_stride=1, num_frames=1):
        from ...native import AvdfError
        from .windows import check_window
        check_window(window, hop)
        if self.model.test_nms_method == "none":
            raise AvdfError("nms_method 'none' returns every decoded candidate: windows need hard or soft NMS to merge")
        for c in items:
            if "streams" not in c:
                raise AvdfError("sliding windows need raw streams; 'feats' items are already resampled to max_seq_len")
        out, group, nbytes = [], [], 0
        for c in items:
            b = sum(np.asarray(a).nbytes if not torch.is_tensor(a) else a.numel() * a.element_size() for a in c["streams"].values())
            if group and nbytes + b > self.GROUP_BYTES:
                out.extend(self._run_group(group, window, hop, feat_stride, num_frames))
                group, nbytes = [], 0
            group.append(c)
            nbytes += b
        if group:
            out.extend(self._run_group(group, window, hop, feat_stride, num_frames))
        return out

    def _win_stage(self, rows, chans, dtype, device):
        """Group staging, grown x1.5 when a group does not fit; growing drops the graphs that captured the old buffers."""
        if not hasattr(self, "win_cap"):
            self.win_cap, self.win_host, self.win_dev, self.win_graphs = [0, 0, 0], [None] * 3, [None] * 3, {}
        for s in range(3):
            if chans[s] == 0:
                continue
            t = self.win_host[s]
            if t is None or rows[s] > self.win_cap[s] or t.dtype != dtype or t.shape[1] != chans[s]:
                self.win_cap[s] = max(rows[s], int(self.win_cap[s] * 1.5)) + 64
                self.win_host[s] = torch.empty((self.win_cap[s], chans[s]), dtype=dtype, pin_memory=True)
                self.win_dev[s] = torch.empty((self.win_cap[s], chans[s]), dtype=dtype, device=device)
                self.win_graphs.clear()

    def _run_group(self, items, window, hop, feat_stride, num_frames):
        from .windows import window_meta, window_plan
        eng, L, MB = self.eng, self.eng.max_seq_len, self.eng.max_batch
        K = int(self.model.test_max_seg_num)
        present = [n in items[0]["streams"] for n in STREAMS]
        arrs = [[np.ascontiguousarray(_stream_array(c["streams"][n])) for c in items] if p else None for n, p in zip(STREAMS, present)]
        np_dt = next(al[0].dtype for al in arrs if al)
        item = np_dt.itemsize
        chans = [al[0].shape[1] if al else 0 for al in arrs]
        if sum(chans) != eng.c_in:
            raise ValueError("streams carry %d channels, the model expects %d" % (sum(chans), eng.c_in))
        for al in arrs:
            for a in al or ():
                if a.dtype != np_dt:
                    raise ValueError("a batch mixes fp32 streams and 16-bit shards")
        rows = [sum(a.shape[0] for a in al) if al else 0 for al in arrs]
        first = 0 if present[0] else 1
        # ---- plan: one unit per window (a recording no longer than the window is one unit with its own meta)
        rec_win, starts, counts, metas, s_k = [0], [], [], [], []
        base = [0, 0, 0]
        for r, c in enumerate(items):
            lens = [al[r].shape[0] if al else None for al in arrs]
            plan = window_plan(c["duration"], lens, window, hop)
            for s0, rng in plan:
                starts.append([base[s] + a for s, (a, _) in enumerate(rng)])
                counts.append([m for _, m in rng])
                metas.append(video_meta(c, lens[first], L, feat_stride, num_frames) if len(plan) == 1
                             else window_meta(rng[first][1], window, L, feat_stride, num_frames))
                s_k.append(np.float32(s0))
            rec_win.append(len(starts))
            base = [b + (l or 0) for b, l in zip(base, lens)]
        n_units, R = len(starts), len(items)
        slot = self.slots[0]                     # lane 0 and its stream: the window batches run one after the other
        with torch.cuda.device(eng.device):
            if slot.busy:
                self._collect(slot)
            with self.cuda_lock:
                self._win_stage(rows, chans, torch.float32 if item == 4 else torch.bfloat16, eng.device)
            # ---- pack the group's rows once (library thread pool), then one host -> device copy per stream
            src, dst, nb = [], [], []
            for s in range(3):
                if arrs[s] is None:
                    continue
                hb, row_bytes, off = self.win_host[s].data_ptr(), chans[s] * item, 0
                for a in arrs[s]:
                    if a.shape[1] != chans[s]:
                        raise ValueError("stream %s: recordings differ in channel count" % STREAMS[s])
                    src.append(a.ctypes.data); dst.append(hb + off * row_bytes); nb.append(a.nbytes)
                    off += a.shape[0]
            n = len(src)
            native.check(native.lib().avdf_host_pack((ctypes.c_void_p * n)(*src), (ctypes.c_void_p * n)(*dst),
                                                     (ctypes.c_size_t * n)(*nb), n, self.n_threads), "avdf_host_pack")
            # per-batch (start [3, b], count [3, b], meta [4, b]) blocks, one after the other, in one pinned buffer
            batches = [(u, min(MB, n_units - u)) for u in range(0, n_units, MB)]
            par = np.zeros(10 * n_units, np.float32)
            for u0, b in batches:
                blk = par[10 * u0: 10 * (u0 + b)]
                blk[:6 * b].view(np.int32)[:] = np.concatenate([np.asarray(starts[u0:u0 + b], np.int32).T,
                                                                np.asarray(counts[u0:u0 + b], np.int32).T]).reshape(-1)
                blk[6 * b:] = np.asarray(metas[u0:u0 + b], np.float32).T.reshape(-1)
            h_par = torch.from_numpy(par).pin_memory()
            h_idx = torch.tensor(rec_win + [int(c.get("index", r)) for r, c in enumerate(items)], dtype=torch.int32).pin_memory()
            h_start = torch.from_numpy(np.asarray(s_k, np.float32)).pin_memory()
            slot.stream.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(slot.stream):
                for s in range(3):
                    if chans[s]:
                        self.win_dev[s][:rows[s]].copy_(self.win_host[s][:rows[s]], non_blocking=True)
                d_par = h_par.to(eng.device, non_blocking=True)
                d_idx = h_idx.to(eng.device, non_blocking=True)
                d_start = h_start.to(eng.device, non_blocking=True)
                self.h2d_bytes += sum(rows[s] * chans[s] * item for s in range(3)) + 4 * (par.size + h_idx.numel() + n_units)
                w_segs = torch.empty((n_units, K, 2), dtype=torch.float32, device=eng.device)
                w_scores = torch.empty((n_units, K), dtype=torch.float32, device=eng.device)
                w_count = torch.empty((n_units,), dtype=torch.int32, device=eng.device)
                w_cls = torch.empty((n_units,), dtype=torch.float32, device=eng.device)
                streams = [self.win_dev[s] if chans[s] else None for s in range(3)]
                for u0, b in batches:
                    blk = d_par[10 * u0: 10 * (u0 + b)]
                    ranges = (blk[:6 * b].view(torch.int32)[:3 * b].view(3, b), blk[:6 * b].view(torch.int32)[3 * b:].view(3, b))
                    meta = blk[6 * b:].view(4, b)
                    if self.use_graph and b == MB:
                        key = (b, self.model.test_key(), item)
                        g = self.win_graphs.get(key)
                        if g is None:
                            fixed = {"start": torch.empty((3, b), dtype=torch.int32, device=eng.device),
                                     "count": torch.empty((3, b), dtype=torch.int32, device=eng.device),
                                     "meta": torch.empty((4, b), dtype=torch.float32, device=eng.device)}
                            fixed["start"].copy_(ranges[0]); fixed["count"].copy_(ranges[1]); fixed["meta"].copy_(meta)
                            staged = {"ids": [None] * b, "B": b, "meta": fixed["meta"], "streams": streams, "offs": None,
                                      "ranges": (fixed["start"], fixed["count"])}
                            with self.cuda_lock:
                                g = self.model.capture(staged, lane=slot.index)
                            self.win_graphs[key] = g
                        st = g.staged
                        st["ranges"][0].copy_(ranges[0], non_blocking=True)
                        st["ranges"][1].copy_(ranges[1], non_blocking=True)
                        st["meta"].copy_(meta, non_blocking=True)
                        res = g.replay()
                    else:
                        staged = {"ids": [None] * b, "B": b, "meta": meta, "streams": streams, "offs": None, "ranges": ranges}
                        res = self.model.run_staged(staged, lane=slot.index)
                    w_segs[u0:u0 + b].copy_(res["segs"], non_blocking=True)
                    w_scores[u0:u0 + b].copy_(res["scores"], non_blocking=True)
                    w_count[u0:u0 + b].copy_(res["counts"], non_blocking=True)
                    w_cls[u0:u0 + b].copy_(res["vcls"], non_blocking=True)
                # ---- merge: one result per recording
                cap = K * max(rec_win[r + 1] - rec_win[r] for r in range(R))
                o_segs = torch.empty((R, K, 2), dtype=torch.float32, device=eng.device)
                o_scores = torch.empty((R, K), dtype=torch.float32, device=eng.device)
                o_count = torch.empty((R,), dtype=torch.int32, device=eng.device)
                o_cls = torch.empty((R,), dtype=torch.float32, device=eng.device)
                m = self.model
                rec = None if self.records is None else (self.records[0], self.records[1], d_idx[R + 1:])
                ops.window_merge(d_idx[:R + 1], d_start, w_segs, w_scores, w_count, w_cls, cand_cap=cap,
                                 iou_threshold=m.test_iou_threshold, min_score=m.test_min_score, sigma=m.test_nms_sigma,
                                 voting_thresh=0.0 if m.test_multiclass_nms else m.test_voting_thresh,
                                 use_soft_nms=m.test_nms_method == "soft", out_segs=o_segs, out_scores=o_scores,
                                 out_count=o_count, out_cls=o_cls, records=rec)
                res = [t.to("cpu", non_blocking=True) for t in (o_segs, o_scores, o_count, o_cls)]
                self.d2h_bytes += R * (3 * K + 2) * 4
                done = torch.cuda.Event()
                done.record()
            done.synchronize()
        segs, scores, cnt, vcls = res
        empty_labels = torch.zeros(K, dtype=torch.long)
        return [{"video_id": c["video_id"], "segments": segs[r, :int(cnt[r])], "scores": scores[r, :int(cnt[r])],
                 "labels": empty_labels[:int(cnt[r])], "video_cls": vcls[r:r + 1]} for r, c in enumerate(items)]

    # ---------------------------------------------------------------- public
    def run(self, chunk, dense=None):
        """One batch, synchronously. dense: optional DenseStore that keeps the batch's dense outputs."""
        slot = self.slots[0]
        with torch.cuda.device(self.eng.device):
            if slot.busy:
                self._collect(slot)
            self._pack(slot, chunk)
            self._launch(slot, dense)
            return self._collect(slot)

    def stream(self, batches, dense=None):
        """Generator over an iterable of batches (each <= max_batch videos): yields every batch's results in order.
        A packer thread fills free staging slots (pinned memcpy on the worker pool, GIL released) while this thread
        launches slot i (H2D + graph + D2H on the slot's stream) and collects slot i - (n_slots - 1)."""
        free = queue.Queue()
        for slot in self.slots:
            if slot.busy:
                self._collect(slot)
            free.put(slot)
        err = []
        it = iter(batches)
        lock = threading.Lock()
        cond = threading.Condition()
        packed = {}                 # sequence number -> slot (None marks the end of the input)
        state = {"next": 0, "stop": False}

        def packer():
            try:
                # a fresh thread starts on device 0: pinned allocations and cudaPointerGetAttributes would create a context
                # there for every rank of a torchrun job
                torch.cuda.set_device(self.eng.device)
                while True:
                    slot = free.get()
                    if slot is None:
                        return
                    with lock:      # keep (sequence number, slot order) consistent with the input order
                        if state["stop"]:
                            free.put(slot)
                            return
                        try:
                            chunk = next(it)
                        except StopIteration:
                            state["stop"] = True
                            seq = state["next"]
                            with cond:
                                packed[seq] = None
                                cond.notify_all()
                            free.put(slot)
                            return
                        seq = state["next"]
                        state["next"] += 1
                    self._pack(slot, chunk)
                    with cond:
                        packed[seq] = slot
                        cond.notify_all()
            except BaseException as exc:      # surfaced in the consumer
                err.append(exc)
                with cond:
                    packed[-1] = None
                    cond.notify_all()

        threads = [threading.Thread(target=packer, daemon=True) for _ in range(self.n_packers)]
        for th in threads:
            th.start()

        class _Ready:
            seq = 0

            @staticmethod
            def get():
                with cond:
                    while _Ready.seq not in packed and -1 not in packed:
                        cond.wait()
                    if -1 in packed:
                        return None
                    slot_ = packed.pop(_Ready.seq)
                _Ready.seq += 1
                return slot_
        ready = _Ready
        inflight = []
        try:
            while True:
                slot = ready.get()
                if slot is None:
                    break
                self._launch(slot, dense)
                inflight.append(slot)
                if len(inflight) >= len(self.slots) - 1:
                    done = inflight.pop(0)
                    out = self._collect(done)
                    free.put(done)
                    yield out
            while inflight:
                done = inflight.pop(0)
                out = self._collect(done)
                free.put(done)
                yield out
        finally:
            with lock:
                state["stop"] = True
            for _ in threads:
                free.put(None)
            for th in threads:
                th.join(timeout=5)
        if err:
            raise err[0]
