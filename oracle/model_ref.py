"""CPU fp32 restatement of the reference's localization-inference forward path.

TEST INFRASTRUCTURE — the parity checker, never the product path. Only
`tests/`, `__graft_entry__.smoke()` and `bench.py`'s cpu_baseline /
`--impl reference` legs may import this module. The product package
(`audio_visual_deepfake_detection_b200`) never imports anything under oracle/.

Parity pin: `oracle/make_golden.py` runs the UNMODIFIED reference (imported
from /root/reference in the build container) on seeded weights/inputs and
stores its outputs under tests/golden/; `tests/test_oracle_golden.py` checks
this restatement against those fixtures (and against the live reference when
/root/reference is present). The reference itself ships no tests or golden
vectors (SURVEY.md §4), so that is the strongest pin available.

Everything is written as plain math on [B, C, T] fp32 tensors (torch on CPU is
used only as an array library: conv1d / matmul / softmax), in evaluation mode,
from the reference's state_dict. Each function cites the reference lines it
restates (paths relative to the reference root).
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn.functional as F

Tensor = torch.Tensor


# --------------------------------------------------------------------------
# primitives
# --------------------------------------------------------------------------
def masked_conv1d(x: Tensor, mask: Tensor, w: Tensor, b: Optional[Tensor],
                  stride: int = 1, groups: int = 1) -> Tuple[Tensor, Tensor]:
    """libs/modeling/blocks.py:41-63 (MaskedConv1D.forward).

    y = conv1d(x, pad=k//2, stride) * mask[::stride]; the strided mask is the
    nearest-neighbour resample, i.e. mask[:, :, s*i].
    """
    k = w.shape[-1]
    assert x.shape[-1] % stride == 0
    y = F.conv1d(x, w, b, stride=stride, padding=k // 2, groups=groups)
    m = mask[:, :, ::stride] if stride > 1 else mask
    return y * m.to(y.dtype), m


def channel_ln(x: Tensor, w: Tensor, b: Tensor, eps: float = 1e-5) -> Tensor:
    """libs/modeling/blocks.py:97-112: LayerNorm over C for each (b, t),
    biased variance, eps inside the sqrt, affine [1, C, 1]."""
    mu = x.mean(dim=1, keepdim=True)
    r = x - mu
    var = (r * r).mean(dim=1, keepdim=True)
    return r / torch.sqrt(var + eps) * w.view(1, -1, 1) + b.view(1, -1, 1)


def instance_norm_t(x: Tensor, eps: float = 1e-5) -> Tensor:
    """nn.InstanceNorm1d defaults (blocks.py:1508, 1601): per (b, c) over ALL T
    positions (masked zeros included), biased variance, no affine."""
    mu = x.mean(dim=2, keepdim=True)
    var = ((x - mu) ** 2).mean(dim=2, keepdim=True)
    return (x - mu) / torch.sqrt(var + eps)


def sinusoid_pe(n_pos: int, d: int) -> Tensor:
    """libs/modeling/blocks.py:116-127 (fp64 table -> fp32), shape [1, d, n_pos];
    the backbone divides it by sqrt(d) (backbones.py:337)."""
    pos = np.arange(n_pos, dtype=np.float64)[:, None]
    j = np.arange(d)[None, :]
    ang = pos / np.power(10000.0, 2.0 * (j // 2) / d)
    tab = np.empty_like(ang)
    tab[:, 0::2] = np.sin(ang[:, 0::2])
    tab[:, 1::2] = np.cos(ang[:, 1::2])
    return torch.from_numpy(tab.astype(np.float32)).t().unsqueeze(0).contiguous()


def gelu_erf(x: Tensor) -> Tensor:
    return 0.5 * x * (1.0 + torch.erf(x / math.sqrt(2.0)))


def max_pool_3_2_1(x: Tensor) -> Tensor:
    """nn.MaxPool1d(3, stride=2, padding=1) (blocks.py:1277-1281): out[t] =
    max(x[2t-1], x[2t], x[2t+1]) with out-of-range taps ignored (-inf)."""
    T = x.shape[-1]
    xp = F.pad(x, (1, 1), value=float("-inf"))
    idx = torch.arange(0, T, 2, device=x.device)
    return torch.maximum(torch.maximum(xp[..., idx], xp[..., idx + 1]), xp[..., idx + 2])


def nearest_resample(x: Tensor, t_out: int) -> Tensor:
    """F.interpolate(mode='nearest') with an integer up/down factor
    (backbones.py:487, 490; necks.py:78): out[t] = in[floor(t * T_in / T_out)]."""
    t_in = x.shape[-1]
    idx = (torch.arange(t_out, device=x.device) * t_in) // t_out
    return x[..., idx]


def banded_attention(q: Tensor, k: Tensor, v: Tensor, kv_mask: Tensor,
                     n_head: int, half_window: int) -> Tensor:
    """The sliding-chunk code of blocks.py:977-1150 / 535-708 restated as plain
    banded attention (SURVEY.md A.4).

    q,k,v: [B, C, T]; kv_mask [B, 1, T] bool. Score for |i-j| <= w inside
    [0, T): q_i.k_j / sqrt(d) + (-1e4 if key j is masked); outside the band or
    the sequence: -inf. Rows whose own position is masked are zeroed after the
    softmax (blocks.py:1208-1209).
    """
    B, C, T = q.shape
    d = C // n_head
    qh = q.view(B, n_head, d, T).transpose(2, 3) * (1.0 / math.sqrt(d))
    kh = k.view(B, n_head, d, T).transpose(2, 3)
    vh = v.view(B, n_head, d, T).transpose(2, 3)
    s = qh @ kh.transpose(-1, -2)                               # [B, H, T, T]
    i = torch.arange(T, device=q.device)
    band = (i[:, None] - i[None, :]).abs() <= half_window
    s = s + (~kv_mask).to(s.dtype).view(B, 1, 1, T) * (-1e4)
    s = s.masked_fill(~band.view(1, 1, T, T), float("-inf"))
    p = torch.softmax(s, dim=-1)
    p = p * kv_mask.to(p.dtype).view(B, 1, T, 1)
    o = p @ vh                                                  # [B, H, T, d]
    return o.transpose(2, 3).reshape(B, C, T)


def global_attention(q: Tensor, k: Tensor, v: Tensor, kv_mask: Tensor, n_head: int) -> Tensor:
    """blocks.py:291-309 (MaskedMHCA): full softmax attention, masked keys -inf,
    values multiplied by the key mask."""
    B, C, T = q.shape
    d = C // n_head
    qh = q.view(B, n_head, d, -1).transpose(2, 3) * (1.0 / math.sqrt(d))
    kh = k.view(B, n_head, d, -1).transpose(2, 3)
    vh = v.view(B, n_head, d, -1).transpose(2, 3)
    s = qh @ kh.transpose(-1, -2)
    s = s.masked_fill(~kv_mask.view(B, 1, 1, -1), float("-inf"))
    p = torch.softmax(s, dim=-1)
    o = p @ (vh * kv_mask.to(vh.dtype).view(B, 1, -1, 1))
    return o.transpose(2, 3).reshape(B, C, -1)


# --------------------------------------------------------------------------
# the model
# --------------------------------------------------------------------------
class OracleModel:
    """Functional restatement of AVPtTransformerRecovery (exp12,
    libs/modeling/av_fd_no_recon.py:162-876) and its `...NoreconTHE` sibling
    (exp13, libs/modeling/av_fd_no_recon2.py) in eval mode."""

    def __init__(self, model_cfg: dict, state_dict: Dict[str, Tensor], model_name: str):
        self.cfg = model_cfg
        self.name = model_name
        self.sd = {k[7:] if k.startswith("module.") else k: v.detach().to(torch.float32).cpu()
                   for k, v in state_dict.items()}
        self.exp13 = model_name.endswith("THE")
        # exp5-style arch (libs/modeling/av_fd_meta_arch.py:162): the Expansion's reconstruction is live
        self.recon = model_name == "AVLocPointTransformerRecoveryNoNorm"
        c = model_cfg
        self.n_head = c["n_head"]
        self.C = c["embd_dim"]
        self.arch = tuple(c["backbone_arch"])
        self.scale_factor = c["scale_factor"]
        nwin = c["n_mha_win_size"]
        self.win = [nwin] * (1 + self.arch[2]) if isinstance(nwin, int) else list(nwin)
        self.max_seq_len = c["max_seq_len"]
        self.fpn_strides = [self.scale_factor ** i for i in range(c["fpn_start_level"], self.arch[2] + 1)]
        self.reg_range = c["regression_range"]
        self.num_classes = c["num_classes"]
        self.test_cfg = c["test_cfg"]
        # av_fd_no_recon.py:217-224
        mdf = 1
        for s, w in zip(self.fpn_strides, self.win):
            st = s * (w // 2) * 2 if w > 1 else s
            assert self.max_seq_len % st == 0
            mdf = max(mdf, st)
        self.max_div_factor = mdf
        self.pe = sinusoid_pe(self.max_seq_len, self.C) / math.sqrt(self.C)

    # ---- helpers over the state dict -------------------------------------
    def p(self, key: str) -> Tensor:
        return self.sd[key]

    def has(self, key: str) -> bool:
        return key in self.sd

    def ln(self, x: Tensor, prefix: str) -> Tensor:
        return channel_ln(x, self.p(prefix + ".weight"), self.p(prefix + ".bias"))

    # ---- attention modules -----------------------------------------------
    def _attn(self, pre: str, xq: Tensor, mq: Tensor, xk: Tensor, mk: Tensor,
              xv: Tensor, mv: Tensor, stride: int, window: int) -> Tuple[Tensor, Tensor]:
        """LocalMaskedMHCA / LocalMaskedMMHCA / MaskedMHCA forward
        (blocks.py:1152-1224, 710-781, 274-313): depthwise conv k3 (stride s) ->
        channel LN -> 1x1 projection for each of q, k, v; attention; 1x1 proj."""
        q, qm = masked_conv1d(xq, mq, self.p(pre + ".query_conv.conv.weight"), None, stride, groups=xq.shape[1])
        q = self.ln(q, pre + ".query_norm")
        k, km = masked_conv1d(xk, mk, self.p(pre + ".key_conv.conv.weight"), None, stride, groups=xk.shape[1])
        k = self.ln(k, pre + ".key_norm")
        v, _ = masked_conv1d(xv, mv, self.p(pre + ".value_conv.conv.weight"), None, stride, groups=xv.shape[1])
        v = self.ln(v, pre + ".value_norm")
        q = F.conv1d(q, self.p(pre + ".query.weight"), self.p(pre + ".query.bias"))
        k = F.conv1d(k, self.p(pre + ".key.weight"), self.p(pre + ".key.bias"))
        v = F.conv1d(v, self.p(pre + ".value.weight"), self.p(pre + ".value.bias"))
        if window > 1:
            o = banded_attention(q, k, v, km, self.n_head, window // 2)
        else:
            o = global_attention(q, k, v, km, self.n_head)
        o = F.conv1d(o, self.p(pre + ".proj.weight"), self.p(pre + ".proj.bias")) * qm.to(o.dtype)
        return o, qm

    def _mlp_and_residual(self, pre: str, skip: Tensor, attn_out: Tensor, m: Tensor) -> Tensor:
        """blocks.py:1311-1313 / 870-872 with AffineDropPath in eval mode
        (blocks.py:1438-1439: per-channel scale, no drop)."""
        mf = m.to(skip.dtype)
        ga = self.p(pre + ".drop_path_attn.scale") if self.has(pre + ".drop_path_attn.scale") else 1.0
        gm = self.p(pre + ".drop_path_mlp.scale") if self.has(pre + ".drop_path_mlp.scale") else 1.0
        y = skip * mf + ga * attn_out
        h = F.conv1d(self.ln(y, pre + ".ln2"), self.p(pre + ".mlp.0.weight"), self.p(pre + ".mlp.0.bias"))
        h = gelu_erf(h)
        h = F.conv1d(h, self.p(pre + ".mlp.3.weight"), self.p(pre + ".mlp.3.bias"))
        return y + gm * (h * mf)

    def transformer_block(self, pre: str, x: Tensor, m: Tensor, stride: int, window: int):
        """TransformerBlock.forward, blocks.py:1307-1317."""
        u = self.ln(x, pre + ".ln1")
        a, om = self._attn(pre + ".attn", u, m, u, m, u, m, stride, window)
        skip = max_pool_3_2_1(x) if stride > 1 else x
        return self._mlp_and_residual(pre, skip, a, om), om

    def mm_block(self, pre: str, xq: Tensor, mq: Tensor, xk: Tensor, mk: Tensor, xv: Tensor, mv: Tensor, window: int):
        """MutilModelTransformerBlock.forward, blocks.py:866-876 (stride 1)."""
        a, om = self._attn(pre + ".attn", self.ln(xq, pre + ".lnq"), mq, self.ln(xk, pre + ".lnk"), mk,
                           self.ln(xv, pre + ".lnv"), mv, 1, window)
        return self._mlp_and_residual(pre, xq, a, om), om

    # ---- backbone -----------------------------------------------------------
    def _embed(self, x: Tensor, mask: Tensor) -> Tensor:
        """Embedding convs + LN + ReLU + absolute PE, backbones.py:437-465."""
        T = x.shape[-1]
        for i in range(self.arch[0]):
            x, _ = masked_conv1d(x, mask, self.p(f"backbone.embd.{i}.conv.weight"),
                                 self.sd.get(f"backbone.embd.{i}.conv.bias"))
            if self.has(f"backbone.embd_norm.{i}.weight"):
                x = self.ln(x, f"backbone.embd_norm.{i}")
            x = torch.relu(x)
        if self.cfg["use_abs_pe"]:
            pe = self.pe
            if T >= self.max_seq_len:
                pe = F.interpolate(pe, T, mode="linear", align_corners=False)
            x = x + pe[:, :, :T] * mask.to(x.dtype)
        return x

    def backbone(self, x: Tensor, mask: Tensor, taps: Optional[dict] = None, reco: Optional[Tensor] = None):
        """ConvHRLRFullResSelfAttTransformerBackboneRevised.forward,
        backbones.py:413-495. norm_x is dead; reco_x == x in the Norecon archs,
        so their embedding is evaluated once (identical values). In the exp5-style
        arch `reco` (the Expansion's output) is embedded with the same weights and is
        the K stream of resselfattention (backbones.py:469)."""
        reco_e = self._embed(reco, mask) if reco is not None else None
        x = self._embed(x, mask)
        if taps is not None:
            taps["embd"] = x
        w0 = self.win[0]
        xk = reco_e if reco_e is not None else x
        x, _ = self.mm_block("backbone.resselfattention", x, mask, xk, mask, x, mask, w0)
        if taps is not None:
            taps["res"] = x
        for i in range(self.arch[1]):
            x, mask = self.transformer_block(f"backbone.stem.{i}", x, mask, 1, w0)
        if taps is not None:
            taps["stem"] = x
        lh, lh_mask = x, mask
        feats, masks = [lh], [lh_mask]
        for i in range(self.arch[2]):
            x, mask = self.transformer_block(f"backbone.branch.{i}", x, mask, self.scale_factor, self.win[1 + i])
            up = nearest_resample(x, lh.shape[-1])
            lh, lh_mask = self.mm_block(f"backbone.lh_branch.{i}", lh, lh_mask, up, lh_mask, up, lh_mask, w0)
            feats.append(x)
            masks.append(mask)
            if i + 1 < self.arch[2]:      # hh_branch[last] output is never consumed (backbones.py:485-495)
                dn = nearest_resample(lh, x.shape[-1])
                x, mask = self.mm_block(f"backbone.hh_branch.{i}", x, mask, dn, mask, dn, mask, w0)
        feats[0], masks[0] = lh, lh_mask
        return feats, masks

    # ---- neck ----------------------------------------------------------------
    def neck(self, feats: Sequence[Tensor], masks: Sequence[Tensor]):
        """FPN1D.forward, necks.py:62-93."""
        lat = []
        for i, (f, m) in enumerate(zip(feats, masks)):
            y, _ = masked_conv1d(f, m, self.p(f"neck.lateral_convs.{i}.conv.weight"),
                                 self.sd.get(f"neck.lateral_convs.{i}.conv.bias"))
            lat.append(y)
        for i in range(len(lat) - 1, 0, -1):
            lat[i - 1] = lat[i - 1] + nearest_resample(lat[i], lat[i - 1].shape[-1])
        out = []
        for i, (y, m) in enumerate(zip(lat, masks)):
            z, _ = masked_conv1d(y, m, self.p(f"neck.fpn_convs.{i}.conv.weight"),
                                 self.sd.get(f"neck.fpn_convs.{i}.conv.bias"), groups=y.shape[1])
            if self.has(f"neck.fpn_norms.{i}.weight"):
                z = self.ln(z, f"neck.fpn_norms.{i}")
            out.append(z)
        return out, list(masks)

    # ---- heads ---------------------------------------------------------------
    def _tower(self, pre: str, f: Tensor, m: Tensor) -> Tensor:
        n = self.cfg["head_num_layers"] - 1
        for i in range(n):
            f, _ = masked_conv1d(f, m, self.p(f"{pre}.head.{i}.conv.weight"), self.sd.get(f"{pre}.head.{i}.conv.bias"))
            if self.has(f"{pre}.norm.{i}.weight"):
                f = self.ln(f, f"{pre}.norm.{i}")
            f = torch.relu(f)
        return f

    def heads(self, fpn: Sequence[Tensor], masks: Sequence[Tensor]):
        """PtTransformerClsHead / RegHead forward, av_fd_no_recon.py:75-89, 144-159."""
        logits, offsets = [], []
        for l, (f, m) in enumerate(zip(fpn, masks)):
            c = self._tower("cls_head", f, m)
            lg, _ = masked_conv1d(c, m, self.p("cls_head.cls_head.conv.weight"), self.p("cls_head.cls_head.conv.bias"))
            r = self._tower("reg_head", f, m)
            of, _ = masked_conv1d(r, m, self.p("reg_head.offset_head.conv.weight"), self.p("reg_head.offset_head.conv.bias"))
            of = torch.relu(of * self.p(f"reg_head.scale.{l}.scale"))
            logits.append(lg)
            offsets.append(of)
        return logits, offsets

    # ---- video-level branch --------------------------------------------------
    def _down_block(self, pre: str, x: Tensor, m: Tensor, stride: int):
        """DownBlock.forward, blocks.py:1512-1516."""
        y, m = masked_conv1d(x, m, self.p(pre + ".conv_block.conv.weight"), self.p(pre + ".conv_block.conv.bias"), stride)
        return F.leaky_relu(instance_norm_t(y), 0.2), m

    def expansion(self, z: Tensor, m: Tensor) -> Tensor:
        """Expansion.forward, blocks.py:1568-1590: 5 x UpBlock (blocks.py:1519-1541) =
        ConvTranspose1d(k3, stride 2, padding 1, output_padding 1) * nearest-upsampled
        mask (blocks.py:1472-1491) -> InstanceNorm1d -> LeakyReLU(0.2); `last` is
        False everywhere (DeepInterpolator passes tanh=False, blocks.py:1599)."""
        for i in range(1, 6):
            pre = f"interpolator.expansion.up_{i}.conv_transpose.conv"
            y = F.conv_transpose1d(z, self.p(pre + ".weight"), self.p(pre + ".bias"), stride=2, padding=1, output_padding=1)
            m = F.interpolate(m.to(y.dtype), size=y.shape[-1], mode="nearest")
            y = y * m
            m = m.bool()
            z = F.leaky_relu(instance_norm_t(y), 0.2)
        return z

    def video_cls_exp12(self, x: Tensor, mask: Tensor) -> Tensor:
        """DeepInterpolator.forward with norm=False, blocks.py:1627-1638; the
        Expansion output is discarded by the Norecon callers (av_fd_no_recon.py:346)
        and kept (self._reco) for the exp5-style arch (av_fd_meta_arch.py:346)."""
        z, m = x, mask
        for i in range(1, 6):
            z, m = self._down_block(f"interpolator.contraction.down_{i}", z, m, 2)
        self._reco = self.expansion(z, m) if self.recon else None
        g = F.conv1d(z, self.p("interpolator.conv0.0.weight"))
        g = F.leaky_relu(instance_norm_t(g), 0.2)
        pooled = torch.cat([g.max(dim=2).values, g.mean(dim=2)], dim=1)          # [B, 2C]
        h = pooled @ self.p("interpolator.conv1.weight").t()
        h = channel_ln(h.unsqueeze(-1), self.p("interpolator.bn1.weight"), self.p("interpolator.bn1.bias")).squeeze(-1)
        h = torch.relu(h)
        return h @ self.p("interpolator.conv2.weight").t() + self.p("interpolator.conv2.bias")

    def video_cls_exp13(self, x: Tensor, mask: Tensor) -> Tensor:
        """SegmentandCls.forward / segment, blocks.py:1682-1721 (norm=False)."""
        z, m = x, mask
        for i in range(1, 6):
            z, m = self._down_block(f"segmentandCls.contraction.down_{i}", z, m, 1)
        g = F.conv1d(z, self.p("segmentandCls.conv0.0.weight"))
        g = F.leaky_relu(instance_norm_t(g), 0.2)
        s = torch.einsum("bct,oc->bot", g, self.p("segmentandCls.seg_linear.weight")) \
            + self.p("segmentandCls.seg_linear.bias").view(1, -1, 1)                # [B, 1, T]
        pooled = torch.cat([s.max(dim=2).values, s.mean(dim=2)], dim=1)           # [B, 2]
        return pooled @ self.p("segmentandCls.cls_linear1.weight").t() + self.p("segmentandCls.cls_linear1.bias")

    # ---- dense forward ---------------------------------------------------------
    @torch.no_grad()
    def forward_dense(self, x: Tensor, mask: Tensor, taps: Optional[dict] = None):
        """x [B, C_in, T] fp32, mask [B, 1, T] bool -> (logits[l] [B,1,T_l],
        offsets[l] [B,2,T_l], masks[l] [B,1,T_l], video_cls [B,1])."""
        vcls = self.video_cls_exp13(x, mask) if self.exp13 else self.video_cls_exp12(x, mask)
        feats, masks = self.backbone(x, mask, taps, reco=self._reco if self.recon else None)
        if taps is not None:
            taps["feats"] = feats
        fpn, masks = self.neck(feats, masks)
        if taps is not None:
            taps["fpn"] = fpn
        logits, offsets = self.heads(fpn, masks)
        return logits, offsets, masks, vcls

    # ---- preprocessing / decode / postprocessing -------------------------------
    def preprocess(self, feats: Tensor) -> Tuple[Tensor, Tensor]:
        """av_fd_no_recon.py:431-479 (eval branch, one video)."""
        T = feats.shape[-1]
        if T <= self.max_seq_len:
            L = self.max_seq_len
        else:
            s = self.max_div_factor
            L = (T + s - 1) // s * s
        x = F.pad(feats, (0, L - T)).unsqueeze(0)
        mask = (torch.arange(L)[None, :] < T).unsqueeze(1)
        return x, mask

    def decode(self, logits: Sequence[Tensor], offsets: Sequence[Tensor], masks: Sequence[Tensor]):
        """inference_single_video, av_fd_no_recon.py:760-825, for ONE video:
        logits[l] [T_l, n_cls], offsets[l] [T_l, 2], masks[l] [T_l]."""
        tc = self.test_cfg
        segs_all, scores_all, labels_all = [], [], []
        for l, (lg, of, m) in enumerate(zip(logits, offsets, masks)):
            stride = float(self.fpn_strides[l])
            prob = (torch.sigmoid(lg) * m.unsqueeze(-1).to(lg.dtype)).flatten()
            keep = prob > tc["pre_nms_thresh"]
            idx = keep.nonzero(as_tuple=True)[0]
            prob = prob[keep]
            prob, order = prob.sort(descending=True, stable=True)
            k = min(tc["pre_nms_topk"], idx.numel())
            prob, idx = prob[:k], idx[order[:k]]
            pt = torch.div(idx, self.num_classes, rounding_mode="floor")
            cls = torch.fmod(idx, self.num_classes)
            t = pt.to(torch.float32) * stride
            left = t - of[pt, 0] * stride
            right = t + of[pt, 1] * stride
            ok = (right - left) > tc["duration_thresh"]
            segs_all.append(torch.stack([left, right], -1)[ok])
            scores_all.append(prob[ok])
            labels_all.append(cls[ok])
        return torch.cat(segs_all), torch.cat(scores_all), torch.cat(labels_all)

    def postprocess(self, segs, scores, labels, item: dict, nms_fn):
        """postprocessing, av_fd_no_recon.py:827-876. `nms_fn` is a
        batched_nms-compatible callable (oracle/nms_ref.py or the compiled
        reference)."""
        tc = self.test_cfg
        if tc["nms_method"] != "none":
            segs, scores, labels = nms_fn(
                segs, scores, labels, tc["iou_threshold"], tc["min_score"], tc["max_seg_num"],
                use_soft_nms=(tc["nms_method"] == "soft"), multiclass=tc["multiclass_nms"],
                sigma=tc["nms_sigma"], voting_thresh=tc["voting_thresh"])
        if segs.shape[0] > 0:
            segs = (segs * item["feat_stride"] + 0.5 * item["feat_num_frames"]) / item["fps"]
            segs = segs.clone()
            segs[segs <= 0.0] *= 0.0
            segs[segs >= item["duration"]] = segs[segs >= item["duration"]] * 0.0 + item["duration"]
        return segs, scores, labels

    @torch.no_grad()
    def __call__(self, video_list: List[dict], nms_fn, return_dense: bool = False):
        """Same contract as `model(video_list)` in eval mode
        (av_fd_no_recon.py:334-429), one video at a time (the reference
        asserts len == 1, :456; videos are independent, SURVEY.md §8)."""
        out = []
        for item in video_list:
            x, mask = self.preprocess(item["feats"].to(torch.float32))
            logits, offsets, masks, vcls = self.forward_dense(x, mask)
            lg = [a[0].permute(1, 0) for a in logits]
            of = [a[0].permute(1, 0) for a in offsets]
            ms = [a[0, 0] for a in masks]
            segs, scores, labels = self.decode(lg, of, ms)
            segs, scores, labels = self.postprocess(segs, scores, labels, item, nms_fn)
            r = {"video_id": item["video_id"], "segments": segs, "scores": scores,
                 "labels": labels, "video_cls": vcls[0]}
            if return_dense:
                r["dense_logits"] = torch.cat([a.flatten() for a in lg])
                r["dense_offsets"] = torch.cat(of, dim=0)
            out.append(r)
        return out
