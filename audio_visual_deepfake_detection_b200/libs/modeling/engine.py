"""Device-side execution plan of the localization-inference path.

`LocalizationEngine` owns the packed weights and the static activation buffers
(token-major [B, T, C], sized once for `max_batch`) and issues the kernel
sequence of one forward pass through `ops` (= the C-ABI). Nothing is computed
in PyTorch here: torch provides device memory and the stream, every arithmetic
step is a libavdf_sm100 kernel. Static buffers + a fixed launch sequence make
the whole pass CUDA-graph capturable.

Kernel sequence per batch (reference lines each step replaces):
  video-level branch  Contraction / Extract DownBlocks (blocks.py:1495-1516, 1544-1565, 1640-1661)
                      = conv_gemm(k3, stride 2|1, +bias, mask) -> instnorm_lrelu, x5; tail vcls_exp12 / vcls_exp13
  embedding           backbones.py:437-465 = 2 x conv_gemm(k3, mask, LN, ReLU [, +PE]); evaluated ONCE (the
                      reference runs it three times on identical inputs)
  18 blocks           blocks.py:783-876 / 1227-1317 = ln_dwconv_ln -> 3 x conv_gemm(1x1 q,k,v) -> attention ->
                      conv_gemm(proj, mask, residual, gamma) -> ln_rows -> conv_gemm(1x1, GELU) ->
                      conv_gemm(1x1, mask, residual, gamma); up/down-sampling between scales is an index map
                      inside ln_dwconv_ln (backbones.py:487,490); hh_branch[last] is dead and skipped
  neck                necks.py:62-93 = 6 x conv_gemm(1x1 lateral) into one pyramid buffer -> fpn_fuse
  heads               av_fd_no_recon.py:75-89,144-159 = 2 x 2 x conv_gemm(k3 over all 6 levels in one launch, LN, ReLU)
                      -> head_final
  postprocess         av_fd_no_recon.py:760-876 + libs/utils/nms.py = avdf_postprocess (one CTA per video)
"""
import math
import os

import numpy as np
import torch

from ... import ops
from ...native import AvdfError
from .spec import EXP5, EXP13, state_dict_spec


def sinusoid_table(n_pos, d):
    """blocks.py:116-127: fp64 table -> fp32, returned token-major [n_pos, d]."""
    pos = np.arange(n_pos, dtype=np.float64)[:, None]
    j = np.arange(d)[None, :]
    ang = pos / np.power(10000.0, 2.0 * (j // 2) / d)
    tab = np.empty_like(ang)
    tab[:, 0::2] = np.sin(ang[:, 0::2])
    tab[:, 1::2] = np.cos(ang[:, 1::2])
    return tab.astype(np.float32)


def up_weight(w_t):
    """ConvTranspose1d(k=3, stride=2, padding=1, output_padding=1) weight [c_in, c_out, 3] (blocks.py:1443-1468) -> the
    [2*c_out, 2*c_in] matrix of the equivalent forward-tap GEMM (avdf_conv_gemm tap_mode 1, taps at x[t], x[t+1]):
        out[2t]   = W[:, :, 1]^T x[t]                       (rows [0, c_out):        tap 0 = W1, tap 1 = 0)
        out[2t+1] = W[:, :, 2]^T x[t] + W[:, :, 0]^T x[t+1]   (rows [c_out, 2 c_out):  tap 0 = W2, tap 1 = W0)
    so that GEMM row t, viewed as [2, c_out], is the pair of output positions (2t, 2t+1); x[T] reads as zero."""
    w = w_t.detach().to(torch.float32)
    ci, co, k = w.shape
    assert k == 3
    even = torch.cat([w[:, :, 1].t(), torch.zeros(co, ci)], dim=1)
    odd = torch.cat([w[:, :, 2].t(), w[:, :, 0].t()], dim=1)
    return torch.cat([even, odd], dim=0).contiguous()


class PackedWeights:
    """Reference state_dict -> device tensors in the kernels' layouts.

    dense conv / linear [co, ci, k] -> [co, k*ci] (tap-major rows) in the dtype of the A operand;
    LN / AffineDropPath / bias vectors -> flat fp32; depthwise [C,1,3] -> [C,3] fp32.
    """

    def __init__(self, sd, device):
        self.sd = {(k[7:] if k.startswith("module.") else k): v for k, v in sd.items()}
        self.device = device
        self._cache = {}

    def has(self, key):
        return key in self.sd

    def vec(self, key):
        """flat fp32 vector (LN weight/bias [1,C,1], conv bias, scales)."""
        ck = ("v", key)
        if ck not in self._cache:
            self._cache[ck] = self.sd[key].detach().to(torch.float32).reshape(-1).contiguous().to(self.device)
        return self._cache[ck]

    def ln(self, prefix):
        return (self.vec(prefix + ".weight"), self.vec(prefix + ".bias"))

    def dense(self, key, dtype=torch.float32):
        """[co, ci, k] or [co, ci] -> [co, k*ci] in `dtype` (the dtype of the A operand it multiplies)."""
        ck = ("d", key, dtype)
        if ck not in self._cache:
            w = self.sd[key].detach().to(torch.float32)
            if w.dim() == 3:
                w = w.permute(0, 2, 1).reshape(w.shape[0], -1)
            self._cache[ck] = w.contiguous().to(self.device).to(dtype).contiguous()
        return self._cache[ck]

    def dense_t(self, key):
        """[co, ci(, 1)] -> transposed fp32 [ci, co] (thread-per-output-channel kernels read it coalesced)."""
        ck = ("t", key)
        if ck not in self._cache:
            w = self.sd[key].detach().to(torch.float32)
            w = w.reshape(w.shape[0], -1)
            self._cache[ck] = w.t().contiguous().to(self.device)
        return self._cache[ck]

    def stack_dense(self, keys, dtype):
        """Several [co, ci(, k)] weights stacked along co (one GEMM launch with per-segment weight blocks)."""
        ck = ("sd", tuple(keys), dtype)
        if ck not in self._cache:
            self._cache[ck] = torch.cat([self.dense(k, dtype) for k in keys], dim=0).contiguous()
        return self._cache[ck]

    def stack_vec(self, keys):
        ck = ("sv", tuple(keys))
        if ck not in self._cache:
            self._cache[ck] = torch.cat([self.vec(k) for k in keys]).contiguous()
        return self._cache[ck]

    def dw(self, key):
        ck = ("w", key)
        if ck not in self._cache:
            w = self.sd[key].detach().to(torch.float32)
            self._cache[ck] = w.reshape(w.shape[0], 3).contiguous().to(self.device)
        return self._cache[ck]


# Operand formats of the tensor-core GEMMs (accumulation is always fp32 in TMEM, the residual stream,
# LayerNorm statistics, softmax and the last head convolutions are always fp32):
#   "mixed" (default)  bf16 for GEMMs whose A operand is the raw feature tensor (unbounded range), fp16 for all others
#                      (normalised activations). Measured logit error <= 5.6e-3, offsets <= 1.2e-3 relative over 3 x 256
#                      videos at batch 32 (bar: 1e-2); same tensor-core rate and bytes as pure bf16.
#   "fp32"             CUDA-core fp32 parity mode (bar: 1e-4).
# Pure bf16 operands were measured at 1.2e-2 on the synthetic worst-case weights - over BASELINE.json's 1e-2 bar (the
# reference itself under torch.autocast(bfloat16) shows the same, SURVEY.md appendix B) - so that format is not offered.
PRECISIONS = ("mixed", "fp32")


class DenseStore:
    """Caller-owned device copy of what the in-graph post-processing reads, batch after batch: pyramid logits [P],
    offsets [P, 2], video_cls, the four seconds-conversion scalars (feat_stride, half frames, fps, duration) and the valid
    length of every video (the pyramid mask is rebuilt from it). Pass it as `dense=` to `forward_streams`, `stream` or
    `model(video_list)` (feats items); libs/utils/sweep.py then post-processes the kept outputs under many test_cfg
    settings without another forward pass. About 18 KB per video at max_seq_len 768.

    Videos are kept in the order they were added, in chunks of `chunk` videos that share one pyramid layout (feats items
    longer than max_seq_len are padded to other lengths)."""

    def __init__(self, chunk=4096):
        self.chunk = int(chunk)
        self.ids = []
        self.chunks = []              # dicts: L, level_len, level_stride, n, logits, offsets, vcls, meta, valid, pos (host)
        self._open = {}               # L -> chunk being filled

    def __len__(self):
        return len(self.ids)

    def nbytes(self):
        return sum(sum(c[k].numel() * c[k].element_size() for k in ("logits", "offsets", "vcls", "meta")) for c in self.chunks)

    def add(self, ids, L, level_len, level_stride, logits, offsets, vcls, meta, valid):
        """Device-to-device copies (on the current stream) of a batch: logits [B, P], offsets [B, P, 2], vcls [B],
        meta [4, B] fp32 (device); valid: host ints [B]."""
        B, P = logits.shape
        pos0 = len(self.ids)
        self.ids.extend(ids)
        done = 0
        while done < B:
            c = self._open.get(L)
            if c is None or c["n"] == self.chunk:
                dev = logits.device
                c = {"L": L, "level_len": list(level_len), "level_stride": list(level_stride), "n": 0,
                     "logits": torch.empty((self.chunk, P), dtype=torch.float32, device=dev),
                     "offsets": torch.empty((self.chunk, P, 2), dtype=torch.float32, device=dev),
                     "vcls": torch.empty((self.chunk,), dtype=torch.float32, device=dev),
                     "meta": torch.empty((4, self.chunk), dtype=torch.float32, device=dev),
                     "valid": np.zeros(self.chunk, np.int32), "pos": np.zeros(self.chunk, np.int32)}
                self.chunks.append(c)
                self._open[L] = c
            m = min(B - done, self.chunk - c["n"])
            dst, src = slice(c["n"], c["n"] + m), slice(done, done + m)
            c["logits"][dst].copy_(logits[src], non_blocking=True)
            c["offsets"][dst].copy_(offsets[src], non_blocking=True)
            c["vcls"][dst].copy_(vcls[src], non_blocking=True)
            c["meta"][:, dst].copy_(meta[:, src], non_blocking=True)
            c["valid"][dst] = np.asarray(valid[done:done + m], np.int32)
            c["pos"][dst] = np.arange(pos0 + done, pos0 + done + m, dtype=np.int32)
            c["n"] += m
            done += m


class LocalizationEngine:
    def __init__(self, model_cfg, model_name, state_dict, device, precision="mixed", max_batch=32):
        if not torch.cuda.is_available():
            raise AvdfError("LocalizationEngine needs a CUDA device: the path has no CPU fallback")
        if precision not in PRECISIONS:
            raise ValueError("precision must be one of %s" % (PRECISIONS,))
        c = model_cfg
        self.cfg = c
        self.name = model_name
        self.exp13 = model_name == EXP13
        self.recon = model_name == EXP5      # live Expansion: its output is embedded and becomes K of resselfattention
        self.device = torch.device(device)
        self.precision = precision
        # in_dt: format of the raw feature tensor (unbounded values -> bf16 range); adt: format of every
        # other GEMM operand (LayerNorm / InstanceNorm / softmax / GELU outputs: bounded -> fp16 mantissa)
        self.in_dt, self.adt = {"fp32": (torch.float32, torch.float32), "mixed": (torch.bfloat16, torch.float16)}[precision]
        self.max_batch = int(max_batch)
        # fused MLP kernel (csrc/mlp_fused.cu: one launch per block, the [rows, 1024] activations never leave the SM):
        # 51 vs 59 us per level-0 block next to the two GEMM launches, +4 % videos/s with 4 batches in flight, same
        # results to the last bits of fp32 accumulation order. AVDF_FUSED_MLP=0 switches back to the two launches;
        # AVDF_FUSED_MLP_MIN_ROWS sets the smallest level (rows = batch * t) that uses it.
        self.fused_mlp = os.environ.get("AVDF_FUSED_MLP", "1") != "0"
        self.fused_mlp_min_rows = int(os.environ.get("AVDF_FUSED_MLP_MIN_ROWS", "0"))
        self.fuse_ln2 = os.environ.get("AVDF_FUSE_LN2", "1") != "0"    # LN2 in the attention projection's epilogue (A/B switch)
        self.fuse_tail = os.environ.get("AVDF_FUSE_TAIL", "1") != "0"  # projection + LN2 + MLP as one launch (A/B switch)
        self.head_dots = os.environ.get("AVDF_HEAD_DOTS", "1") != "0"  # heads' final conv as dot products in the tower epilogue (A/B switch)
        self.C = c["embd_dim"]
        self.n_head = c["n_head"]
        self.c_in = c["video_input_dim"] + c["audio_input_dim"]
        self.arch = tuple(c["backbone_arch"])
        if c["backbone_type"] != "convHRLRFullResSelfAttTransformerRevised":
            raise AvdfError("only the convHRLRFullResSelfAttTransformerRevised backbone is on the accelerated path")
        if c["fpn_type"] != "fpn":
            raise AvdfError("only fpn_type 'fpn' is on the accelerated path")
        if self.C != 256 or c["fpn_dim"] != 256 or c["head_dim"] != 256 or self.n_head != 4:
            raise AvdfError("kernels are specialised for embd/fpn/head dim 256 with 4 heads")
        if c["scale_factor"] != 2 or c["embd_kernel_size"] != 3 or c["head_kernel_size"] != 3 or c["fpn_start_level"] != 0:
            raise AvdfError("unsupported scale_factor / kernel size / fpn_start_level")
        if c.get("use_rel_pe", False):
            raise AvdfError("use_rel_pe is not supported")
        nwin = c["n_mha_win_size"]
        self.win = [nwin] * (1 + self.arch[2]) if isinstance(nwin, int) else list(nwin)
        self.n_levels = self.arch[2] + 1
        self.max_seq_len = c["max_seq_len"]
        self.strides = [2 ** i for i in range(self.n_levels)]
        mdf = 1
        for s, w in zip(self.strides, self.win):       # av_fd_no_recon.py:217-224
            st = s * (w // 2) * 2 if w > 1 else s
            assert self.max_seq_len % st == 0, "max_seq_len must be divisible by fpn stride and window size"
            mdf = max(mdf, st)
        self.max_div_factor = mdf
        self.test_cfg = dict(c["test_cfg"])
        self.num_classes = c["num_classes"]
        if self.num_classes != 1:
            raise AvdfError("the fused postprocess handles num_classes == 1 (the shipped configs)")
        missing = [k for k in state_dict_spec(c, model_name) if (k not in state_dict and "module." + k not in state_dict)
                   and not (k.startswith("interpolator.expansion.") and not self.recon) and not k.startswith("segmentandCls.bn1")]
        if missing:
            raise KeyError("state_dict is missing %d tensors, e.g. %s" % (len(missing), missing[:3]))
        self.w = PackedWeights(state_dict, self.device)
        self._bufs = {}
        self.lane = 0                 # buffer set in use: independent batches in flight on different streams use different lanes
        self._mask_cache = {}
        self._pe_cache = {}
        self._ws = None
        # while a CUDA graph is being captured: every cached tensor the launches point at (mask tables, workspaces) is
        # appended here and kept alive by the GraphedPass - evicting the cache or growing a workspace must not free
        # memory a captured graph still reads
        self._capture_refs = None

    # ------------------------------------------------------------------ buffers
    def buf(self, name, shape, dtype):
        """Static buffer sized for max_batch; returns the [B, ...] prefix view."""
        B = shape[0]
        key = (self.lane, name, tuple(shape[1:]), dtype)
        t = self._bufs.get(key)
        if t is None:
            t = torch.empty((self.max_batch,) + tuple(shape[1:]), dtype=dtype, device=self.device)
            self._bufs[key] = t
        return t[:B]

    def workspace(self, nbytes):
        if self._ws is None:
            self._ws = {}
        ws = self._ws.get(self.lane)
        if ws is None or ws.numel() < nbytes:
            ws = torch.empty(int(nbytes), dtype=torch.uint8, device=self.device)
            self._ws[self.lane] = ws
        if self._capture_refs is not None:
            self._capture_refs.append(ws)
        return ws

    def padded_len(self, t):
        """av_fd_no_recon.py:458-466."""
        if t <= self.max_seq_len:
            return self.max_seq_len
        s = self.max_div_factor
        return (t + s - 1) // s * s

    def level_lens(self, L):
        return [L // s for s in self.strides]

    def masks(self, valid, L):
        """Per-level row masks [B, T_l] and the pyramid mask [B, P] (uint8) for valid lengths
        `valid` (host ints). mask_l[b, t] = (t * 2^l < valid[b]) (nearest down-sampling, blocks.py:51-55)."""
        key = (tuple(int(v) for v in valid), L)
        m = self._mask_cache.get(key)
        if m is None:
            lens = self.level_lens(L)
            v = np.asarray(key[0], dtype=np.int64)[:, None]
            lv = [((np.arange(n)[None, :] * s) < v).astype(np.uint8) for n, s in zip(lens, self.strides)]
            pyr = np.concatenate(lv, axis=1)
            # masks of the Expansion (UpBlock: nearest up-sampling of the coarsest Contraction mask, blocks.py:1480-1484):
            # up_l[b, t] = mask_last[b, t >> (last - l)]
            last = len(lens) - 1
            up = [lv[last][:, np.arange(n) >> (last - l)] for l, n in enumerate(lens)] if self.recon else []
            flat = np.concatenate([pyr.reshape(-1)] + [a.reshape(-1) for a in lv] + [np.ascontiguousarray(a).reshape(-1) for a in up])
            dev = torch.from_numpy(flat).to(self.device)
            B, P = len(valid), sum(lens)
            out = {"pyr": dev[: B * P].view(B, P)}
            off = B * P
            for l, n in enumerate(lens):
                out[l] = dev[off: off + B * n].view(B, n)
                off += B * n
            for l, n in enumerate(lens if self.recon else []):
                out["up%d" % l] = dev[off: off + B * n].view(B, n)
                off += B * n
            if len(self._mask_cache) > 64:
                self._mask_cache.clear()
            self._mask_cache[key] = out
            m = out
        if self._capture_refs is not None:
            self._capture_refs.append(m)
        return m

    def pe(self, L):
        """[L, C] fp32 table / sqrt(C) (backbones.py:336-338); for L > max_seq_len the reference
        linearly re-interpolates the constant table (backbones.py:456-461) - done once on the host."""
        t = self._pe_cache.get(L)
        if t is None:
            tab = torch.from_numpy(sinusoid_table(self.max_seq_len, self.C)) / math.sqrt(self.C)
            if L >= self.max_seq_len and L != self.max_seq_len:
                tab = torch.nn.functional.interpolate(tab.t().unsqueeze(0), L, mode="linear", align_corners=False)[0].t()
            t = tab[:L].contiguous().to(self.device)
            self._pe_cache[L] = t
        return t

    # ------------------------------------------------------------------ building blocks
    def _gemm(self, a, wkey, *, B, taps=1, stride=1, segs, a_rows, o_rows, bias=None, row_mask=None, ln=None,
              act=ops.ACT_NONE, pe=None, residual=None, gamma=None, out_f32=None, out_act=None, ln_after_residual=False,
              tap_mode=0, dots=None):
        w = self.w.dense(wkey, a.dtype) if isinstance(wkey, str) else self.w.stack_dense(wkey, a.dtype)
        n_out, k = w.shape
        if not isinstance(wkey, str):
            n_out //= len(wkey)
        c_in = k // taps
        out_h = None
        if out_act is not None:
            if out_act.dtype == torch.float32:
                assert out_f32 is None
                out_f32 = out_act
            else:
                out_h = out_act
        if ln_after_residual:
            assert out_h is not None and out_f32 is not None
        ws = None
        if a.dtype == torch.float32:
            ws = self.workspace(B * o_rows * n_out * 4)
        ops.conv_gemm(a, w, taps=taps, stride=stride, batch=B, c_in=c_in, n_out=n_out, segs=segs, a_rows=a_rows,
                      o_rows=o_rows, bias=bias, row_mask=row_mask, ln=ln, act=act, pe=pe, residual=residual, gamma=gamma,
                      out_f32=out_f32, out_h=out_h, workspace=ws, ln_after_residual=ln_after_residual, tap_mode=tap_mode, dots=dots)

    def _attn_and_mlp(self, pre, B, T, mask, skip, window, out_name, want_act_copy, pyr=None):
        """Shared tail of TransformerBlock / MutilModelTransformerBlock after the dwconv+LN stage:
        q,k,v 1x1 -> attention -> proj(+skip) -> LN2 -> MLP(+residual). Returns (out_f32, out_act|None)."""
        C, w = self.C, self.w
        seg = [(T, 0, 0)]
        # q, k, v projections as ONE launch: the dwconv+LN stage wrote a video's q/k/v rows stacked ([B, 3T, C]);
        # three segments with their own 256-row weight block each (blocks.py:1169-1171)
        qkvn = self.buf("qkvn", (B, 3 * T, C), self.adt)
        qkvp = self.buf("qkvp", (B, 3 * T, C), self.adt)
        names = ("query", "key", "value")
        self._gemm(qkvn, [f"{pre}.attn.{nm}.weight" for nm in names], B=B, segs=[(T, i * T, i * T, i * C) for i in range(3)],
                   a_rows=3 * T, o_rows=3 * T, bias=w.stack_vec([f"{pre}.attn.{nm}.bias" for nm in names]), out_act=qkvp)
        att = self.buf("att", (B, T, C), self.adt)
        ops.attention(None, None, None, mask, att, batch=B, t=T, n_head=self.n_head, window=window, qkv=qkvp)
        y = self.buf("y", (B, T, C), torch.float32)
        ga = w.vec(pre + ".drop_path_attn.scale") if w.has(pre + ".drop_path_attn.scale") else None
        gm = w.vec(pre + ".drop_path_mlp.scale") if w.has(pre + ".drop_path_mlp.scale") else None
        l2 = self.buf("ln2", (B, T, C), self.adt)
        # 16-bit path: LN2 (blocks.py:1311) runs in the projection's epilogue (ln_after_residual): y is normalised while it is
        # still in TMEM - one launch and one fp32 round trip of the residual stream less per block
        fuse_ln2 = self.fuse_ln2 and self.adt != torch.float32 and C == 256
        fused = self.fused_mlp and self.adt != torch.float32 and C == 256 and B * T >= self.fused_mlp_min_rows
        # block tail: projection + LN2 + MLP in ONE launch (csrc/mlp_fused.cu, PROJ variant): the LN2 output never leaves the SM
        fuse_tail = self.fuse_tail and fuse_ln2 and fused
        if fuse_tail:
            pass
        elif fuse_ln2:
            self._gemm(att, f"{pre}.attn.proj.weight", B=B, segs=seg, a_rows=T, o_rows=T, bias=w.vec(f"{pre}.attn.proj.bias"),
                       row_mask=mask, residual=skip, gamma=ga, out_f32=y, out_act=l2, ln=w.ln(pre + ".ln2"), ln_after_residual=True)
        else:
            self._gemm(att, f"{pre}.attn.proj.weight", B=B, segs=seg, a_rows=T, o_rows=T, bias=w.vec(f"{pre}.attn.proj.bias"),
                       row_mask=mask, residual=skip, gamma=ga, out_f32=y)
        out = self.buf(out_name, (B, T, C), torch.float32)
        out_act = None
        if want_act_copy and self.adt != torch.float32:
            # pyr = (pyramid buffer [B, P, C], first row of this level): the 16-bit copy goes straight into the operand of
            # the single FPN lateral launch (fused-MLP path only)
            out_act = pyr[0] if (pyr is not None and fused) else self.buf(out_name + "_act", (B, T, C), self.adt)
        if not fuse_ln2:
            ops.ln_rows(y, *w.ln(pre + ".ln2"), l2, B * T)
        if fused:
            # one launch: the [B*T, 4C] activations stay in shared memory / TMEM (csrc/mlp_fused.cu). (Folding LN2 into
            # the kernel was tried - two spare warps normalising the next 128-row tile straight into the operand
            # layout - and measured slower, 14.7k vs 15.9k videos/s: ~10 us per tile that cannot be hidden because the
            # x tile cannot be double-buffered in 227 KB. LN2 stays a separate 9 us launch.)
            proj = None
            w2, b2, g2 = w.dense(f"{pre}.mlp.3.weight", self.adt), w.vec(f"{pre}.mlp.3.bias"), gm
            if fuse_tail:
                # y stays in the accumulator and the second GEMM accumulates on top of it: the MLP's AffineDropPath scale
                # (blocks.py:1316) is folded into W2 / b2 once, in fp32, before the 16-bit rounding of the weights
                proj = (att, w.dense(f"{pre}.attn.proj.weight", self.adt), w.vec(f"{pre}.attn.proj.bias"), ga, w.ln(pre + ".ln2"), skip, None)
                if gm is not None:
                    ck = ("tail", pre, self.adt)
                    if ck not in w._cache:
                        w32 = w.sd[f"{pre}.mlp.3.weight"].detach().to(torch.float32).reshape(C, -1).to(self.device)
                        w._cache[ck] = ((w32 * gm[:, None]).to(self.adt).contiguous(), (b2 * gm).contiguous())
                    w2, b2 = w._cache[ck]
                    g2 = None
            ops.mlp_fused(None if fuse_tail else l2, w.dense(f"{pre}.mlp.0.weight", self.adt), w.vec(f"{pre}.mlp.0.bias"),
                          w2, b2, row_mask=mask, residual=y, gamma=g2, out=out, out_h=out_act, proj=proj,
                          out_h_level=(T, pyr[0].shape[1], pyr[1]) if (pyr is not None and out_act is not None) else None)
            return out, out_act
        h = self.buf("mlp_h", (B, T, 4 * C), self.adt)
        self._gemm(l2, f"{pre}.mlp.0.weight", B=B, segs=seg, a_rows=T, o_rows=T, bias=w.vec(f"{pre}.mlp.0.bias"),
                   act=ops.ACT_GELU, out_act=h)
        # the residual y is already zero on masked rows (blocks.py:1311-1313)
        w2 = self.w.dense(f"{pre}.mlp.3.weight", h.dtype)
        ws = self.workspace(B * T * C * 4) if self.adt == torch.float32 else None
        ops.conv_gemm(h, w2, taps=1, stride=1, batch=B, c_in=4 * C, n_out=C, segs=seg, a_rows=T, o_rows=T,
                      bias=w.vec(f"{pre}.mlp.3.bias"), row_mask=mask, residual=y, gamma=gm, out_f32=out, out_h=out_act,
                      workspace=ws)
        return out, (out if self.adt == torch.float32 else out_act)

    def transformer_block(self, pre, x, B, T, masks, level, stride, window, out_name, want_act_copy=False, pyr=None):
        """TransformerBlock.forward (blocks.py:1307-1317); x fp32 [B, T, C] at pyramid level `level`."""
        C, w = self.C, self.w
        To = T // stride
        lvl_out = level + (1 if stride == 2 else 0)
        mask = masks[lvl_out]
        qkvn = self.buf("qkvn", (B, 3 * To, C), self.adt)
        skip = self.buf("skip", (B, To, C), torch.float32) if stride == 2 else x
        ln1 = w.ln(pre + ".ln1")
        ops.ln_dwconv_ln(x, batch=B, t_src=T, t_virt=T, shift=0, stride=stride, mask_out=mask, ln_in=[ln1] * 3,
                         dw=[w.dw(f"{pre}.attn.{n}_conv.conv.weight") for n in ("query", "key", "value")],
                         ln_out=[w.ln(f"{pre}.attn.{n}_norm") for n in ("query", "key", "value")], outs=[qkvn] * 3,
                         out_rows=3 * To, out_row_offsets=[0, To, 2 * To], skip_out=skip if stride == 2 else None)
        return self._attn_and_mlp(pre, B, To, mask, skip, window, out_name, want_act_copy, pyr)

    def mm_block(self, pre, xq, kv, B, Tq, Tkv, masks, level, window, out_name, want_act_copy=False, pyr=None, xk=None):
        """MutilModelTransformerBlock.forward (blocks.py:866-876): q from xq [B,Tq,C]; k,v from kv [B,Tkv,C]
        nearest-resampled to Tq (backbones.py:487,490). xk (same length as xq): a separate source for the K stream - the
        embedded reconstruction of the exp5-style arch (backbones.py:469)."""
        C, w = self.C, self.w
        mask = masks[level]
        qkvn = self.buf("qkvn", (B, 3 * Tq, C), self.adt)
        names = ("query", "key", "value")
        dws = [w.dw(f"{pre}.attn.{n}_conv.conv.weight") for n in names]
        lno = [w.ln(f"{pre}.attn.{n}_norm") for n in names]
        lni = [w.ln(pre + ".lnq"), w.ln(pre + ".lnk"), w.ln(pre + ".lnv")]
        if xk is not None:
            assert kv is xq and Tkv == Tq
            for i, src in enumerate((xq, xk, xq)):
                ops.ln_dwconv_ln(src, batch=B, t_src=Tq, t_virt=Tq, shift=0, stride=1, mask_out=mask, ln_in=lni[i:i + 1],
                                 dw=dws[i:i + 1], ln_out=lno[i:i + 1], outs=[qkvn], out_rows=3 * Tq, out_row_offsets=[i * Tq])
        elif kv is xq:
            ops.ln_dwconv_ln(xq, batch=B, t_src=Tq, t_virt=Tq, shift=0, stride=1, mask_out=mask, ln_in=lni, dw=dws,
                             ln_out=lno, outs=[qkvn] * 3, out_rows=3 * Tq, out_row_offsets=[0, Tq, 2 * Tq])
        else:
            ops.ln_dwconv_ln(xq, batch=B, t_src=Tq, t_virt=Tq, shift=0, stride=1, mask_out=mask, ln_in=lni[:1],
                             dw=dws[:1], ln_out=lno[:1], outs=[qkvn], out_rows=3 * Tq, out_row_offsets=[0])
            if Tq >= Tkv:
                shift = int(round(math.log2(Tq // Tkv)))
            else:
                shift = -int(round(math.log2(Tkv // Tq)))
            ops.ln_dwconv_ln(kv, batch=B, t_src=Tkv, t_virt=Tq, shift=shift, stride=1, mask_out=mask, ln_in=lni[1:],
                             dw=dws[1:], ln_out=lno[1:], outs=[qkvn] * 2, out_rows=3 * Tq, out_row_offsets=[Tq, 2 * Tq])
        return self._attn_and_mlp(pre, B, Tq, mask, xq, window, out_name, want_act_copy, pyr)

    # ------------------------------------------------------------------ the pass
    def video_cls(self, x_act, B, L, masks):
        w, adt = self.w, self.adt
        vcls = self.buf("vcls", (B,), torch.float32)
        if self.exp13:
            pre, stride, dims = "segmentandCls", 1, [self.c_in, 1024, 512, 256, 128, 64]
        else:
            C = self.C
            pre, stride, dims = "interpolator", 2, [self.c_in, C, 2 * C, 4 * C, 8 * C, C]
        z, T, level = x_act, L, 0
        for i in range(5):
            To = T // stride
            level_o = level + (1 if stride == 2 else 0)
            raw = self.buf("vc_raw", (B, To * dims[i + 1]), torch.float32)
            self._gemm(z, f"{pre}.contraction.down_{i + 1}.conv_block.conv.weight", B=B, taps=3, stride=stride,
                       segs=[(To, 0, 0)], a_rows=T, o_rows=To,
                       bias=w.vec(f"{pre}.contraction.down_{i + 1}.conv_block.conv.bias"), row_mask=masks[level_o], out_f32=raw)
            z = self.buf("vc_z%d" % (i & 1), (B, To * dims[i + 1]), adt)
            ops.instnorm_lrelu(raw.view(B, To, dims[i + 1]), z.view(B, To, dims[i + 1]), batch=B, t=To, channels=dims[i + 1])
            z = z.view(B, To, dims[i + 1])
            T, level = To, level_o
        if self.exp13:
            ops.vcls_exp13(z, w.dense("segmentandCls.conv0.0.weight", torch.float32), w.vec("segmentandCls.seg_linear.weight"),
                           w.vec("segmentandCls.seg_linear.bias"), w.vec("segmentandCls.cls_linear1.weight"),
                           w.vec("segmentandCls.cls_linear1.bias"), vcls, batch=B, t=T)
        else:
            ops.vcls_exp12(z, w.dense_t("interpolator.conv0.0.weight"), w.dense_t("interpolator.conv1.weight"),
                           *w.ln("interpolator.bn1"), w.vec("interpolator.conv2.weight"), w.vec("interpolator.conv2.bias"),
                           vcls, batch=B, t=T)
        self._contracted = z          # [B, T_last, C]: the Expansion's input (exp5-style arch)
        return vcls

    def expansion(self, z, B, masks):
        """Expansion.forward (blocks.py:1568-1590): 5 x UpBlock = ConvTranspose1d(k3, s2, p1, output_padding 1) + bias ->
        * up-sampled mask -> InstanceNorm1d -> LeakyReLU(0.2) (blocks.py:1519-1541; `last` is False: DeepInterpolator builds
        Expansion(tanh=False)). A transposed conv with these parameters is the forward-tap GEMM of `up_weight`: row t of
        the [B, T, 2 c_out] result is the output pair (2t, 2t+1), i.e. the result IS [B, 2T, c_out]. Returns the
        reconstruction [B, L, c_in] in the raw-feature operand format (it goes through the same embedding weights)."""
        w = self.w
        last = self.n_levels - 1
        T = z.shape[1]
        for i in range(5):
            key = f"interpolator.expansion.up_{i + 1}.conv_transpose.conv"
            ck = ("up", key, z.dtype)
            if ck not in w._cache:
                w._cache[ck] = up_weight(w.sd[key + ".weight"]).to(self.device).to(z.dtype).contiguous()
                w._cache[("upb", key)] = torch.cat([w.vec(key + ".bias")] * 2).contiguous()
            wg, bias2 = w._cache[ck], w._cache[("upb", key)]
            co = wg.shape[0] // 2
            raw = self.buf("vc_raw", (B, T * 2 * co), torch.float32)
            ws = self.workspace(B * T * 2 * co * 4) if z.dtype == torch.float32 else None
            ops.conv_gemm(z, wg, taps=2, stride=1, batch=B, c_in=z.shape[2], n_out=2 * co, segs=[(T, 0, 0)], a_rows=T, o_rows=T,
                          bias=bias2, row_mask=masks["up%d" % (last - i)], out_f32=raw, workspace=ws, tap_mode=1)
            T *= 2
            out_dt = self.in_dt if i == 4 else self.adt
            z = self.buf("up_z%d" % (i & 1) if i < 4 else "reco", (B, T * co), out_dt)
            ops.instnorm_lrelu(raw.view(B, T, co), z.view(B, T, co), batch=B, t=T, channels=co)
            z = z.view(B, T, co)
        return z

    def forward_dense(self, x_act, valid):
        """x_act: [B, L, c_in] in `self.in_dt` (token-major), valid: host list of valid lengths.
        Returns (logits [B,P] f32, offsets [B,P,2] f32, vcls [B] f32, masks, level_lens)."""
        B, L, cin = x_act.shape
        assert cin == self.c_in and B <= self.max_batch and x_act.dtype == self.in_dt
        assert L % self.max_div_factor == 0 or L == self.max_seq_len
        C, w, adt = self.C, self.w, self.adt
        lens = self.level_lens(L)
        P = sum(lens)
        offs = [sum(lens[:l]) for l in range(self.n_levels)]
        masks = self.masks(valid, L)
        vcls = self.video_cls(x_act, B, L, masks)
        # ---- embedding (backbones.py:437-465), once
        n_embd = self.arch[0]

        def embed(h, out_name):
            x_ = None
            for i in range(n_embd):
                last = i == n_embd - 1
                ln = w.ln(f"backbone.embd_norm.{i}") if w.has(f"backbone.embd_norm.{i}.weight") else None
                bias = w.vec(f"backbone.embd.{i}.conv.bias") if w.has(f"backbone.embd.{i}.conv.bias") else None
                kw = dict(B=B, taps=3, segs=[(L, 0, 0)], a_rows=L, o_rows=L, bias=bias, row_mask=masks[0], ln=ln, act=ops.ACT_RELU)
                if last:
                    x_ = self.buf(out_name, (B, L, C), torch.float32)
                    self._gemm(h, f"backbone.embd.{i}.conv.weight", pe=self.pe(L) if self.cfg["use_abs_pe"] else None, out_f32=x_, **kw)
                else:
                    e = self.buf("embd%d" % i, (B, L, C), adt)
                    self._gemm(h, f"backbone.embd.{i}.conv.weight", out_act=e, **kw)
                    h = e
            return x_

        x = embed(x_act, "x_embd")
        # ---- backbone (backbones.py:467-495)
        w0 = self.win[0]
        if self.recon:
            # exp5-style: K of resselfattention = the embedded reconstruction (av_fd_meta_arch.py:346-348, backbones.py:469);
            # norm_x is identical to x (DeepInterpolator(norm=False)) and never used
            reco_e = embed(self.expansion(self._contracted, B, masks), "reco_embd")
            x, _ = self.mm_block("backbone.resselfattention", x, x, B, L, L, masks, 0, w0, "x_res", xk=reco_e)
        else:
            x, _ = self.mm_block("backbone.resselfattention", x, x, B, L, L, masks, 0, w0, "x_res")
        for i in range(self.arch[1]):
            x, _ = self.transformer_block(f"backbone.stem.{i}", x, B, L, masks, 0, 1, w0, "x_stem%d" % i)
        lh, lh_act = x, None
        feats_act = [None] * self.n_levels
        T = L
        nb = self.arch[2]
        # fused-MLP path: every level's 16-bit feature copy lands in ONE pyramid buffer, the FPN lateral convs become one
        # launch with six weight blocks (necks.py:62-75)
        one_lateral = self.fused_mlp and adt != torch.float32 and self.fused_mlp_min_rows == 0
        pyr_act = self.buf("pyr_act", (B, P, C), adt) if one_lateral else None
        for i in range(nb):
            x, x_act_copy = self.transformer_block(f"backbone.branch.{i}", x, B, T, masks, i, 2, self.win[1 + i],
                                                   "feat%d" % (i + 1), want_act_copy=True,
                                                   pyr=(pyr_act, offs[i + 1]) if one_lateral else None)
            T //= 2
            feats_act[i + 1] = x_act_copy
            lh, lh_act = self.mm_block(f"backbone.lh_branch.{i}", lh, x, B, L, T, masks, 0, w0, "lh%d" % (i & 1),
                                       want_act_copy=(i == nb - 1), pyr=(pyr_act, offs[0]) if one_lateral else None)
            if i + 1 < nb:            # hh_branch[last] is never consumed (backbones.py:485-495)
                x, _ = self.mm_block(f"backbone.hh_branch.{i}", x, lh, B, T, L, masks, i + 1, w0, "hh%d" % i)
        feats_act[0] = lh_act
        # ---- neck (necks.py:62-93)
        lat = self.buf("lat", (B, P, C), torch.float32)
        has_lat_bias = w.has("neck.lateral_convs.0.conv.bias")
        if one_lateral:
            keys = [f"neck.lateral_convs.{l}.conv.weight" for l in range(self.n_levels)]
            bias = w.stack_vec([f"neck.lateral_convs.{l}.conv.bias" for l in range(self.n_levels)]) if has_lat_bias else None
            self._gemm(pyr_act, keys, B=B, segs=[(lens[l], offs[l], offs[l], l * C) for l in range(self.n_levels)], a_rows=P,
                       o_rows=P, bias=bias, row_mask=masks["pyr"], out_f32=lat)
        else:
            for l in range(self.n_levels):
                bias = w.vec(f"neck.lateral_convs.{l}.conv.bias") if has_lat_bias else None
                self._gemm(feats_act[l], f"neck.lateral_convs.{l}.conv.weight", B=B, segs=[(lens[l], 0, offs[l])], a_rows=lens[l],
                           o_rows=P, bias=bias, row_mask=masks["pyr"], out_f32=lat)
        fpn = self.buf("fpn", (B, P, C), adt)
        if not hasattr(self, "_fpn_params"):
            dw = torch.stack([w.dw(f"neck.fpn_convs.{l}.conv.weight") for l in range(self.n_levels)]).contiguous()
            if w.has("neck.fpn_norms.0.weight"):
                lw = torch.stack([w.vec(f"neck.fpn_norms.{l}.weight") for l in range(self.n_levels)]).contiguous()
                lb = torch.stack([w.vec(f"neck.fpn_norms.{l}.bias") for l in range(self.n_levels)]).contiguous()
            else:
                raise AvdfError("fpn_with_ln=False is not on the accelerated path")
            self._fpn_params = (dw, lw, lb)
        ops.fpn_fuse(lat, masks["pyr"], *self._fpn_params, fpn, batch=B, level_len=lens)
        # ---- heads (av_fd_no_recon.py:75-89, 144-159): all levels in one launch per layer
        segs = [(lens[l], offs[l], offs[l]) for l in range(self.n_levels)]
        towers = {}
        nl = self.cfg["head_num_layers"] - 1
        # 16-bit path: the last tower layer does not write its 256-channel fp32 output at all - its epilogue emits, per row,
        # the dot products with the three taps of the heads' final convolution (fp32, like the convolution itself), and
        # head_combine adds the taps of neighbouring rows (av_fd_no_recon.py:82-89, 152-159)
        head_dots = self.head_dots and adt != torch.float32 and C == 256 and nl >= 1
        dots = {}
        for head in ("cls_head", "reg_head"):
            f = fpn
            for i in range(nl):
                ln = w.ln(f"{head}.norm.{i}") if w.has(f"{head}.norm.{i}.weight") else None
                bias = w.vec(f"{head}.head.{i}.conv.bias") if w.has(f"{head}.head.{i}.conv.bias") else None
                kw = dict(B=B, taps=3, segs=segs, a_rows=P, o_rows=P, bias=bias, row_mask=masks["pyr"], ln=ln, act=ops.ACT_RELU)
                if i == nl - 1 and head_dots and ln is not None:
                    last = "cls_head.cls_head" if head == "cls_head" else "reg_head.offset_head"
                    n_dot = 3 if head == "cls_head" else 6
                    dw = w.dense(last + ".conv.weight", torch.float32).view(n_dot, C)        # [o, 3 * C] -> rows (o, tap)
                    d = self.buf(head + "_dots", (B, P, n_dot), torch.float32)
                    self._gemm(f, f"{head}.head.{i}.conv.weight", dots=(dw, d), **kw)
                    dots[head] = d
                    continue
                if i == nl - 1:       # the last tower layer stays fp32: it feeds the fp32 logit / offset conv
                    o = self.buf(head + "_tower", (B, P, C), torch.float32)
                    self._gemm(f, f"{head}.head.{i}.conv.weight", out_f32=o, **kw)
                else:
                    o = self.buf("%s_t%d" % (head, i), (B, P, C), adt)
                    self._gemm(f, f"{head}.head.{i}.conv.weight", out_act=o, **kw)
                f = o
            towers[head] = f
        logits = self.buf("logits", (B, P), torch.float32)
        offsets = self.buf("offsets", (B, P, 2), torch.float32)
        if not hasattr(self, "_scales"):
            self._scales = [float(self.w.sd[f"reg_head.scale.{l}.scale"]) for l in range(self.n_levels)]
        if len(dots) == 2:
            ops.head_combine(dots["cls_head"], dots["reg_head"], masks["pyr"], w.vec("cls_head.cls_head.conv.bias"),
                             w.vec("reg_head.offset_head.conv.bias"), self._scales, logits, offsets, batch=B, level_len=lens)
            return logits, offsets, vcls, masks, lens
        ops.head_final(towers["cls_head"], towers["reg_head"], masks["pyr"], w.dense("cls_head.cls_head.conv.weight", torch.float32),
                       w.vec("cls_head.cls_head.conv.bias"), w.dense("reg_head.offset_head.conv.weight", torch.float32),
                       w.vec("reg_head.offset_head.conv.bias"), self._scales, logits, offsets, batch=B, level_len=lens)
        return logits, offsets, vcls, masks, lens

    def keep_dense(self, store, ids, L, logits, offsets, vcls, meta, valid):
        """Copy a batch's dense outputs at padded length L (what `postprocess` reads) into a DenseStore."""
        store.add(ids, L, self.level_lens(L), [float(s) for s in self.strides], logits, offsets, vcls, meta, valid)

    def postprocess(self, logits, offsets, masks, lens, meta, nms_method=None, records=None, vcls=None):
        """meta: device fp32 [4, B] rows = feat_stride, 0.5*feat_num_frames, fps, duration (or None).
        records: optional (ring [cap, 3 + 3K] f32, counter [1] i32, vid_index [B] i32 | None): every video appends its
        fixed-size result record to the ring (the unit the multi-GPU gather moves)."""
        tc = self.test_cfg
        B, P = logits.shape
        K = int(tc["max_seg_num"])
        method = nms_method or tc["nms_method"]
        if method not in ("hard", "soft", "none"):
            raise AvdfError("nms_method %r is not one of 'hard', 'soft', 'none'" % (method,))
        if tc["multiclass_nms"] and self.num_classes > 1:
            raise AvdfError("multiclass NMS with more than one class is not on the accelerated path")
        cs = self.buf("cand_segs", (B, P, 2), torch.float32)
        cc = self.buf("cand_scores", (B, P), torch.float32)
        cn = self.buf("cand_count", (B,), torch.int32)
        n_out = P if method == "none" else K        # 'none': every decoded candidate is returned (av_fd_no_recon.py:847)
        osg = self.buf("out_segs", (B, n_out, 2), torch.float32)
        osc = self.buf("out_scores", (B, n_out), torch.float32)
        ocn = self.buf("out_count", (B,), torch.int32)
        # multiclass with a single class == class-agnostic without voting (nms.py:123-156)
        voting = 0.0 if tc["multiclass_nms"] else tc["voting_thresh"]
        rec = None
        if records is not None and method != "none":
            rec = (records[0], records[1], records[2], vcls)
        ops.postprocess(B, logits=logits, offsets=offsets, mask=masks["pyr"], level_len=lens,
                        level_stride=[float(s) for s in self.strides], pre_nms_thresh=tc["pre_nms_thresh"],
                        pre_nms_topk=tc["pre_nms_topk"], duration_thresh=tc["duration_thresh"], cand_segs=cs, cand_scores=cc,
                        cand_count=cn, iou_threshold=tc["iou_threshold"], min_score=tc["min_score"], sigma=tc["nms_sigma"],
                        voting_thresh=voting, max_seg_num=K, use_soft_nms=(None if method == "none" else method == "soft"),
                        vid_meta=None if meta is None else [meta[0], meta[1], meta[2], meta[3]],
                        out_segs=osg, out_scores=osc, out_count=ocn, records=rec)
        return osg, osc, ocn
