"""float64 references of the `ops` entry points the localization forward pass launches, one per entry point, with the
entry point's own keyword arguments.

TEST INFRASTRUCTURE (see oracle/model_ref.py's header).

Each reference takes exactly the arguments of its `ops` function (tensors on any device; the reference computes on the
device of its operands) and returns a dict {output path: Out}. The path names the output argument: "out", "out_f32",
"dots.1" (element 1 of the `dots` tuple), "outs.2", "proj.6". Out holds, for the WHOLE tensor passed as that argument:
  ref      the expected values, float64
  written  bool mask of the elements the launch writes (every other element must keep its previous value)
  zero     bool mask of the elements that must be exactly 0.0 (masked rows, padding rows, ReLU-clamped values)
  mag      float64 magnitude of the terms the value was summed from, or None (= |ref|). Outputs that are a short
           contraction of long sums (head logits / offsets, row dots, the video-level scalar) are compared against it:
           their value can cancel to far below the size of the fp32 rounding of its terms.
Operands are what the kernel saw: 16-bit tensors convert exactly to float64. Intermediate roundings are modelled only
where the code documents them: the 16-bit hidden activations of mlp_fused (csrc/mlp_fused.cu: "-> 16-bit -> shared
memory") and the 16-bit LN2 operand of the block tail (mlp_fused proj=: "writes the 16-bit x tile").
"""
from collections import namedtuple

import numpy as np
import torch

import interp_ref
import model_ref

F64 = torch.float64
ACT_NONE, ACT_RELU, ACT_GELU = 0, 1, 2
Out = namedtuple("Out", "ref written zero mag")

# a ReLU output counts as a structural zero when its pre-activation is below -RELU_MARGIN x the row's largest magnitude:
# two orders of magnitude above the fp32 error of the values the kernels clamp
RELU_MARGIN = 1e-3


def _f(t):
    return None if t is None else t.to(F64)


def _ln(x, w, b):
    """LayerNorm over the last dim (blocks.py:97-112) through model_ref.channel_ln ([N, C, 1] view)."""
    C = x.shape[-1]
    return model_ref.channel_ln(x.reshape(-1, C, 1), _f(w).reshape(-1), _f(b).reshape(-1)).reshape(x.shape)


def _relu(x, zero):
    """ReLU; marks the clamped elements whose pre-activation is clearly negative as structural zeros."""
    row = x.abs().amax(dim=-1, keepdim=True)
    return torch.relu(x), zero | (x < -RELU_MARGIN * row)


def _round(x, dtype):
    """The kernel's rounding of an intermediate to a 16-bit format."""
    return x.to(dtype).to(F64)


def _full(t, fill=0.0):
    return torch.full(t.shape, fill, dtype=F64, device=t.device)


def _false(t):
    return torch.zeros(t.shape, dtype=torch.bool, device=t.device)


def _mask(m, shape, device):
    return torch.ones(shape, dtype=F64, device=device) if m is None else (m.reshape(shape) != 0).to(F64)


# --------------------------------------------------------------------------------------------------- K1 / preprocessing
def interp_concat(streams, offsets, t_out, out):
    """Linear resampling of every stream of every video to t_out rows + channel concat (oracle/interp_ref.py)."""
    batch = next(o for o in offsets if o is not None).numel() - 1
    ranges = []
    for s, o in zip(streams, offsets):
        if s is None:
            ranges.append(None)
            continue
        oc = o.cpu().tolist()
        ranges.append([(oc[b], oc[b + 1] - oc[b]) for b in range(batch)])
    return _interp(streams, ranges, batch, t_out, out)


def interp_concat_ranges(streams, start, count, t_out, out):
    st, ct = start.cpu().tolist(), count.cpu().tolist()
    batch = start.shape[1]
    ranges = [None if s is None else [(st[i][b], ct[i][b]) for b in range(batch)] for i, s in enumerate(streams)]
    return _interp(streams, ranges, batch, t_out, out)


def _interp(streams, ranges, batch, t_out, out):
    ref = torch.empty((batch, t_out, out.shape[-1]), dtype=F64)
    c0 = 0
    for s, rg in zip(streams, ranges):
        if s is None:
            continue
        host = s.float().cpu().numpy()
        for b, (r0, n) in enumerate(rg):
            ref[b, :, c0:c0 + s.shape[1]] = torch.from_numpy(interp_ref.linear_resize_tc(host[r0:r0 + n], t_out, np.float64))
        c0 += s.shape[1]
    ref = ref.to(out.device).reshape(out.shape)
    return {"out": Out(ref, ~_false(out), _false(out), None)}


def pack_feats(feats_ct, out):
    """feats [C, T] -> rows 0..T of out [L, C]; rows T..L are zero."""
    C, T = feats_ct.shape
    ref = _full(out)
    ref[:T] = _f(feats_ct).t()
    zero = _false(out)
    zero[T:] = True
    return {"out": Out(ref, ~_false(out), zero, None)}


# --------------------------------------------------------------------------------------------------- conv GEMM
def conv_gemm(a, w, *, taps, stride=1, batch, c_in, n_out, segs, a_rows, o_rows, bias=None, row_mask=None, ln=None,
              act=ACT_NONE, pe=None, residual=None, gamma=None, out_f32=None, out_h=None, workspace=None,
              ln_after_residual=False, tap_mode=0, dots=None, tap_rows=None):
    """MaskedConv1D as an implicit GEMM over row segments (csrc/gemm_simt.cu is the plain statement):
    segment (t_out, a_row, o_row[, w_row]), video b, output row t: tap j reads A row a_row + stride * t + off_j when
    0 <= stride * t + off_j < t_out * stride (off_j = j - taps // 2, j with tap_mode 1, tap_rows[j] when given), times
    weight rows w_row .. w_row + n_out (bias / ln / gamma advance with w_row); epilogue
        v = (acc + bias) * mask -> LN -> act -> + pe[t] * mask -> residual * mask + gamma * v
    with ln_after_residual: out_f32 = the residual result, out_h = its LayerNorm."""
    dev = a.device
    A = _f(a).reshape(batch, a_rows, c_in)
    W = _f(w)
    offs = list(tap_rows) if tap_rows is not None else [(j if tap_mode else j - taps // 2) for j in range(taps)]
    mask = _mask(row_mask, (batch, o_rows), dev)
    res = None if residual is None else _f(residual).reshape(batch, o_rows, n_out)
    ref = torch.zeros((batch, o_rows, n_out), dtype=F64, device=dev)
    ref_h = torch.zeros_like(ref) if ln_after_residual else None
    zero = torch.zeros(ref.shape, dtype=torch.bool, device=dev)
    written = torch.zeros((batch, o_rows), dtype=torch.bool, device=dev)
    for sg in segs:
        t_out, a_row, o_row = int(sg[0]), int(sg[1]), int(sg[2])
        wr = int(sg[3]) if len(sg) > 3 else 0
        Ws = W[wr:wr + n_out]
        t = torch.arange(t_out, device=dev)
        acc = torch.zeros((batch, t_out, n_out), dtype=F64, device=dev)
        for j, off in enumerate(offs):
            ti = stride * t + off
            ok = (ti >= 0) & (ti < t_out * stride)
            rows = A[:, a_row + ti.clamp(0, t_out * stride - 1)] * ok.to(F64)[None, :, None]
            acc = acc + rows @ Ws[:, j * c_in:(j + 1) * c_in].t()
        mk = mask[:, o_row:o_row + t_out, None]
        v = acc if bias is None else acc + _f(bias)[wr:wr + n_out]
        v = v * mk
        z = (mk == 0).expand(v.shape).clone()
        if ln is not None and not ln_after_residual:
            v = _ln(v, ln[0][wr:wr + n_out], ln[1][wr:wr + n_out])
            z = torch.zeros_like(z)
        if act == ACT_RELU:
            v, z = _relu(v, z)
        elif act == ACT_GELU:
            v = model_ref.gelu_erf(v)
        if pe is not None:
            v = v + _f(pe)[:t_out] * mk
            z = z & (mk == 0)
        if res is not None:
            g = 1.0 if gamma is None else _f(gamma)[wr:wr + n_out]
            v = res[:, o_row:o_row + t_out] * mk + g * v
            z = z & (mk == 0)
        ref[:, o_row:o_row + t_out] = v
        zero[:, o_row:o_row + t_out] = z
        written[:, o_row:o_row + t_out] = True
        if ln_after_residual:
            ref_h[:, o_row:o_row + t_out] = _ln(v, ln[0][wr:wr + n_out], ln[1][wr:wr + n_out])
    wr3 = written[..., None].expand(ref.shape)
    outs = {}
    if out_f32 is not None:
        outs["out_f32"] = Out(ref.reshape(out_f32.shape), wr3.reshape(out_f32.shape), zero.reshape(out_f32.shape), None)
    if out_h is not None:
        if ln_after_residual:
            outs["out_h"] = Out(ref_h.reshape(out_h.shape), wr3.reshape(out_h.shape), _false(out_h), None)
        else:
            outs["out_h"] = Out(ref.reshape(out_h.shape), wr3.reshape(out_h.shape), zero.reshape(out_h.shape), None)
    if dots is not None:
        dw, d = _f(dots[0]), dots[1]
        src = ref_h if ln_after_residual else ref
        dref = src @ dw.t()
        dmag = src.abs() @ dw.abs().t()
        dz = zero.all(dim=-1, keepdim=True).expand(dref.shape)
        dwr = written[..., None].expand(dref.shape)
        outs["dots.1"] = Out(dref.reshape(d.shape), dwr.reshape(d.shape), dz.reshape(d.shape), dmag.reshape(d.shape))
    return outs


# --------------------------------------------------------------------------------------------------- block kernels
def mlp_fused(x, w1, b1, w2, b2, *, row_mask, residual, gamma, out, out_h=None, out_h_level=None, proj=None):
    """out = residual * mask + gamma * ((round16(GELU(x w1^T + b1)) w2^T + b2) * mask); with proj = (att, w_o, b_o,
    gamma_attn, (ln2_w, ln2_b), skip, y): y = skip * mask + gamma_attn * ((att w_o^T + b_o) * mask),
    x = round16(LN2(y)), out = (y + round16(GELU(x w1^T + b1)) w2^T + b2) * mask (w2 / b2 carry the MLP's scale)."""
    dt = (proj[0] if x is None else x).dtype
    C = w1.shape[1]
    outs = {}
    if proj is not None:
        att, w_o, b_o, ga, ln2, skip, y = proj
        rows = att.numel() // C
        m = _mask(row_mask, (rows, 1), att.device)
        p = _f(att).reshape(rows, C) @ _f(w_o).t()
        if b_o is not None:
            p = p + _f(b_o)
        p = p * m
        yv = _f(skip).reshape(rows, C) * m + (1.0 if ga is None else _f(ga)) * p
        xin = _round(_ln(yv, ln2[0], ln2[1]), dt)
        if y is not None:
            z = (m == 0).expand(yv.shape)
            outs["proj.6"] = Out(yv.reshape(y.shape), ~_false(y), z.reshape(y.shape), None)
    else:
        rows = x.numel() // C
        m = _mask(row_mask, (rows, 1), x.device)
        xin = _f(x).reshape(rows, C)
    h = xin @ _f(w1).t()
    if b1 is not None:
        h = h + _f(b1)
    h = _round(model_ref.gelu_erf(h), dt)
    r = h @ _f(w2).t()
    if b2 is not None:
        r = r + _f(b2)
    if proj is not None:
        o = (yv + r) * m
    else:
        o = _f(residual).reshape(rows, C) * m + (1.0 if gamma is None else _f(gamma)) * (r * m)
    z = (m == 0).expand(o.shape)
    outs["out"] = Out(o.reshape(out.shape), ~_false(out), z.reshape(out.shape), None)
    if out_h is not None:
        if out_h_level is not None and int(out_h_level[0]) > 0:
            t, pitch, row0 = (int(v) for v in out_h_level)
            nb = rows // t
            ref = _full(out_h).reshape(nb, pitch, C)
            wr = torch.zeros(ref.shape, dtype=torch.bool, device=ref.device)
            zz = torch.zeros_like(wr)
            ref[:, row0:row0 + t] = o.reshape(nb, t, C)
            wr[:, row0:row0 + t] = True
            zz[:, row0:row0 + t] = z.reshape(nb, t, C)
            outs["out_h"] = Out(ref.reshape(out_h.shape), wr.reshape(out_h.shape), zz.reshape(out_h.shape), None)
        else:
            outs["out_h"] = Out(o.reshape(out_h.shape), ~_false(out_h), z.reshape(out_h.shape), None)
    return outs


def ln_dwconv_ln(src, *, batch, t_src, t_virt, shift, stride, mask_out, ln_in, dw, ln_out, outs, skip_out=None, out_rows=0,
                 out_row_offsets=None, tile_rows=0):
    """Per stream i: LN_in -> depthwise conv k3 (stride, zero padding) -> * mask -> LN_out over the source rows mapped
    by the nearest up / down-sampling index map (virtual row p reads source row p >> shift, or p << -shift); stream i
    lands in rows out_row_offsets[i] .. + t_virt / stride of every video's out_rows. skip_out: MaxPool1d(3, 2, 1) of
    the source rows (blocks.py:1277-1281)."""
    C = src.shape[-1]
    dev = src.device
    t_out = t_virt // stride
    rows_pv = out_rows if out_rows > 0 else t_out
    x = _f(src).reshape(batch, t_src, C)
    p = torch.arange(t_virt, device=dev)
    xv = x[:, (p >> shift) if shift >= 0 else (p << -shift)]
    m = _mask(mask_out, (batch, t_out, 1), dev)
    res = {}
    for i in range(len(outs)):
        u = _ln(xv, *ln_in[i])
        up = torch.nn.functional.pad(u, (0, 0, 1, 1))                  # zero rows at virtual positions -1 and t_virt
        k = _f(dw[i])                                                  # [C, 3]: tap j reads position stride * t + j - 1
        y = sum(k[:, j] * up[:, j:j + stride * (t_out - 1) + 1:stride] for j in range(3))
        o = _ln(y * m, *ln_out[i])
        off = out_row_offsets[i] if out_row_offsets else 0
        ref = torch.zeros((batch, rows_pv, C), dtype=F64, device=dev)
        wr = torch.zeros(ref.shape, dtype=torch.bool, device=dev)
        ref[:, off:off + t_out] = o
        wr[:, off:off + t_out] = True
        res["outs.%d" % i] = Out(ref.reshape(outs[i].shape), wr.reshape(outs[i].shape), _false(outs[i]), None)
    if skip_out is not None:
        sk = model_ref.max_pool_3_2_1(x.transpose(1, 2)).transpose(1, 2)
        res["skip_out"] = Out(sk.reshape(skip_out.shape), ~_false(skip_out), _false(skip_out), None)
    return res


def attention(q, k, v, kv_mask, out, *, batch, t, n_head, window, qkv=None):
    """window > 1: banded softmax attention, |i - j| <= window // 2, masked keys get the additive -1e4, masked query
    rows are exactly 0 (model_ref.banded_attention); window <= 1: MaskedMHCA's global attention, masked keys -inf,
    masked query rows are not zeroed (the projection's mask does it, blocks.py:291-309)."""
    if qkv is not None:
        Q, K, V = (_f(qkv).reshape(batch, 3 * t, -1)[:, i * t:(i + 1) * t] for i in range(3))
    else:
        Q, K, V = (_f(z).reshape(batch, t, -1) for z in (q, k, v))
    C = Q.shape[-1]
    dev = Q.device
    mk = torch.ones((batch, 1, t), dtype=torch.bool, device=dev) if kv_mask is None else (kv_mask.reshape(batch, 1, t) != 0)
    qc, kc, vc = (z.transpose(1, 2) for z in (Q, K, V))
    if window > 1:
        o = model_ref.banded_attention(qc, kc, vc, mk, n_head, window // 2)
        zero = (~mk).transpose(1, 2).expand(batch, t, C)
    else:
        o = model_ref.global_attention(qc, kc, vc, mk, n_head)
        zero = torch.zeros((batch, t, C), dtype=torch.bool, device=dev)
    o = o.transpose(1, 2)
    return {"out": Out(o.reshape(out.shape), ~_false(out), zero.reshape(out.shape), None)}


def ln_rows(x, w, b, out, rows):
    C = x.shape[-1]
    ref = _full(out).reshape(-1, C)
    wr = torch.zeros(ref.shape, dtype=torch.bool, device=ref.device)
    ref[:rows] = _ln(_f(x).reshape(-1, C)[:rows], w, b)
    wr[:rows] = True
    return {"out": Out(ref.reshape(out.shape), wr.reshape(out.shape), _false(out), None)}


def instnorm_lrelu(x, out, *, batch, t, channels, slope=0.2):
    """InstanceNorm1d over all t rows (biased variance, eps 1e-5, no affine) + LeakyReLU (blocks.py:1508-1515)."""
    xc = _f(x).reshape(batch, t, channels).transpose(1, 2)
    y = torch.nn.functional.leaky_relu(model_ref.instance_norm_t(xc), slope).transpose(1, 2)
    return {"out": Out(y.reshape(out.shape), ~_false(out), _false(out), None)}


def _levels(level_len):
    offs = [0]
    for n in level_len:
        offs.append(offs[-1] + int(n))
    return offs


def fpn_fuse(lat, mask, dw_w, ln_w, ln_b, out, *, batch, level_len):
    """FPN1D top-down path (lat[l-1] += nearest(lat[l])) -> depthwise conv k3 * mask -> LN per level (necks.py:62-93)."""
    offs = _levels(level_len)
    L = len(level_len)
    x = _f(lat)
    C = x.shape[-1]
    m = _mask(mask, (batch, offs[-1], 1), x.device)
    lv = [x[:, offs[l]:offs[l + 1]].transpose(1, 2) for l in range(L)]
    for l in range(L - 1, 0, -1):
        lv[l - 1] = lv[l - 1] + model_ref.nearest_resample(lv[l], int(level_len[l - 1]))
    ref = torch.empty((batch, offs[-1], C), dtype=F64, device=x.device)
    for l in range(L):
        y = torch.nn.functional.conv1d(lv[l], _f(dw_w)[l].reshape(C, 1, 3), None, padding=1, groups=C).transpose(1, 2)
        y = y * m[:, offs[l]:offs[l + 1]]
        ref[:, offs[l]:offs[l + 1]] = y if ln_w is None else _ln(y, ln_w[l], ln_b[l])
    return {"out": Out(ref.reshape(out.shape), ~_false(out), _false(out), None)}


def _head_out(acc_c, mag_c, acc_r, mag_r, mask, cls_b, reg_b, level_scale, level_len, batch, logits, offsets):
    offs = _levels(level_len)
    m = _mask(mask, (batch, offs[-1]), logits.device)
    lg = (acc_c + _f(cls_b)[0]) * m
    of = (acc_r + _f(reg_b)) * m[..., None]
    sc = torch.cat([torch.full((int(n),), float(s), dtype=F64) for n, s in zip(level_len, level_scale)]).to(logits.device)
    of = of * sc[None, :, None]
    omag = (mag_r + _f(reg_b).abs()) * sc[None, :, None]
    # ReLU-clamped offsets are structural zeros when clearly negative against the magnitude of their own terms
    oz = (m == 0)[..., None].expand(of.shape) | (of < -RELU_MARGIN * omag)
    of = torch.relu(of)
    return {"logits": Out(lg.reshape(logits.shape), ~_false(logits), (m == 0).reshape(logits.shape),
                          (mag_c + _f(cls_b).abs()[0]).reshape(logits.shape)),
            "offsets": Out(of.reshape(offsets.shape), ~_false(offsets), oz.reshape(offsets.shape), omag.reshape(offsets.shape))}


def _conv_k3_levels(x, wt, level_len):
    """Per-level k3 conv (zero padding inside each level) of token-major x [B, P, C] with w [o, 3 * C] (tap-major);
    returns (values, magnitudes) [B, P, o]."""
    offs = _levels(level_len)
    B, P, C = x.shape
    w = wt.reshape(wt.shape[0], 3, C)
    acc = torch.zeros((B, P, w.shape[0]), dtype=F64, device=x.device)
    mag = torch.zeros_like(acc)
    for l in range(len(level_len)):
        xl = torch.nn.functional.pad(x[:, offs[l]:offs[l + 1]], (0, 0, 1, 1))
        n = offs[l + 1] - offs[l]
        for j in range(3):
            acc[:, offs[l]:offs[l + 1]] += xl[:, j:j + n] @ w[:, j].t()
            mag[:, offs[l]:offs[l + 1]] += xl[:, j:j + n].abs() @ w[:, j].abs().t()
    return acc, mag


def head_final(cls_feat, reg_feat, mask, cls_w, cls_b, reg_w, reg_b, level_scale, logits, offsets, *, batch, level_len):
    """cls_head / offset_head k3 convs + mask, Scale, ReLU (av_fd_no_recon.py:82-89, 152-159)."""
    ac, mc = _conv_k3_levels(_f(cls_feat), _f(cls_w), level_len)
    ar, mr = _conv_k3_levels(_f(reg_feat), _f(reg_w), level_len)
    return _head_out(ac[..., 0], mc[..., 0], ar, mr, mask, cls_b, reg_b, level_scale, level_len, batch, logits, offsets)


def head_combine(cls_dots, reg_dots, mask, cls_b, reg_b, level_scale, logits, offsets, *, batch, level_len):
    """The same heads from per-tap partial sums: tap j of row t comes from row t + j - 1 of the same level."""
    offs = _levels(level_len)
    cd, rd = _f(cls_dots), _f(reg_dots)
    B, P = cd.shape[:2]
    taps = torch.cat([cd, rd], dim=-1).reshape(B, P, 3, 3)          # [.., output (cls, reg0, reg1), tap]
    acc = torch.zeros((B, P, 3), dtype=F64, device=cd.device)
    mag = torch.zeros_like(acc)
    for l in range(len(level_len)):
        n = offs[l + 1] - offs[l]
        tl = torch.nn.functional.pad(taps[:, offs[l]:offs[l + 1]], (0, 0, 0, 0, 1, 1))
        for j in range(3):
            acc[:, offs[l]:offs[l + 1]] += tl[:, j:j + n, :, j]
            mag[:, offs[l]:offs[l + 1]] += tl[:, j:j + n, :, j].abs()
    return _head_out(acc[..., 0], mag[..., 0], acc[..., 1:], mag[..., 1:], mask, cls_b, reg_b, level_scale, level_len, batch,
                     logits, offsets)


def _in_lrelu_tc(z):
    """InstanceNorm over t + LeakyReLU(0.2) of token-major [B, t, C]."""
    return torch.nn.functional.leaky_relu(model_ref.instance_norm_t(z.transpose(1, 2)), 0.2).transpose(1, 2)


def vcls_exp12(z, conv0_w, lin1_w, ln_w, ln_b, lin2_w, lin2_b, out, *, batch, t):
    """DeepInterpolator.classifier (blocks.py:1608-1626): conv0 (1x1, weight passed transposed [ci, co]) -> IN ->
    LeakyReLU -> [max_t, mean_t] -> linear (transposed [2C, C]) -> LN -> ReLU -> linear."""
    g = _in_lrelu_tc(_f(z).reshape(batch, t, -1) @ _f(conv0_w))
    pooled = torch.cat([g.amax(dim=1), g.mean(dim=1)], dim=1)
    h = torch.relu(_ln(pooled @ _f(lin1_w), ln_w, ln_b))
    o = h @ _f(lin2_w) + _f(lin2_b)[0]
    mag = h.abs() @ _f(lin2_w).abs() + _f(lin2_b).abs()[0]
    return {"out": Out(o.reshape(out.shape), ~_false(out), _false(out), mag.reshape(out.shape))}


def vcls_exp13(z, conv0_w, seg_w, seg_b, cls_w, cls_b, out, *, batch, t):
    """SegmentandCls.segment (blocks.py:1682-1700): conv0 (1x1, [co, ci]) -> IN -> LeakyReLU -> seg_linear -> [max_t,
    mean_t] -> cls_linear1."""
    g = _in_lrelu_tc(_f(z).reshape(batch, t, -1) @ _f(conv0_w).t())
    s = g @ _f(seg_w) + _f(seg_b)[0]                                   # [B, t]
    cw, cb = _f(cls_w), _f(cls_b)[0]
    o = cw[0] * s.amax(dim=1) + cw[1] * s.mean(dim=1) + cb
    sm = g.abs() @ _f(seg_w).abs() + _f(seg_b).abs()[0]
    mag = cw[0].abs() * sm.amax(dim=1) + cw[1].abs() * sm.mean(dim=1) + cb.abs()
    return {"out": Out(o.reshape(out.shape), ~_false(out), _false(out), mag.reshape(out.shape))}


REFERENCES = {f.__name__: f for f in (interp_concat, interp_concat_ranges, pack_feats, conv_gemm, mlp_fused, ln_dwconv_ln,
                                      attention, ln_rows, instnorm_lrelu, fpn_fuse, head_final, head_combine, vcls_exp12,
                                      vcls_exp13)}
# entry points the forward pass launches that have no reference here, and why
EXCLUDED = {"postprocess": "decode + NMS + seconds conversion: compared bit for bit with the C oracle (oracle/nms_ref.c) "
                           "in tests/test_gpu_kernels.py and tests/test_gpu_model.py"}


def ulp(x, dtype):
    """One ulp of the 16-bit `dtype` at |x| (float64)."""
    mant, emin = {torch.float16: (10, -14), torch.bfloat16: (7, -126)}[dtype]
    e = torch.floor(torch.log2(x.abs().clamp_min(2.0 ** emin)))
    return torch.pow(2.0, e - mant)


def check(got, o, width, bar, what=""):
    """Asserts a kernel output against its reference Out: structural zeros exactly 0, and the row-wise error
    max|got - ref| / max(|ref|, mag) over rows of `width` values within `bar` (16-bit outputs: beyond one ulp of their
    type at |ref|). Returns the worst row-wise error."""
    ref, written = o.ref.to(got.device), o.written.to(got.device)
    mag = ref.abs() if o.mag is None else o.mag.to(got.device)
    bad = o.zero.to(got.device) & written & (got != 0)
    if bool(bad.any()):
        i = tuple(int(v) for v in bad.nonzero()[0])
        raise AssertionError("%s: element %s must be exactly 0, got %r" % (what, i, float(got[i])))
    err = (got.to(F64) - ref).abs()
    if got.dtype in (torch.float16, torch.bfloat16):
        err = (err - ulp(ref, got.dtype)).clamp_min(0.0)
    err = torch.where(written, err, torch.zeros_like(err)).reshape(-1, width)
    denom = torch.maximum(ref.abs(), mag).reshape(-1, width).amax(dim=1, keepdim=True).clamp_min(1e-30)
    rel = torch.nan_to_num(err / denom, nan=float("inf"))
    worst = float(rel.max())
    if worst > bar:
        idx = tuple(int(v) for v in torch.unravel_index(rel.reshape(-1).argmax().cpu(), ref.shape))
        raise AssertionError("%s: row-wise error %.3g > bar %.1g at %s: got %r, float64 reference %r" %
                             (what, worst, bar, idx, float(got[idx]), float(ref[idx])))
    return worst


def get_path(kwargs, path):
    """The tensor an output path names in a call's keyword arguments ("dots.1" -> kwargs['dots'][1])."""
    parts = path.split(".")
    v = kwargs[parts[0]]
    for p in parts[1:]:
        v = v[int(p)]
    return v
