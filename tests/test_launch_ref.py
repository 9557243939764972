"""CPU checks of the float64 per-launch references (oracle/launch_ref.py) against independent torch formulations
(nn.Conv1d / ConvTranspose1d / Conv2d, nn.LayerNorm, nn.InstanceNorm1d, F.interpolate, a dense band-masked softmax),
their mask semantics, and a static check that every `ops` entry point the forward pass calls has a reference."""
import math
import os
import re

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import launch_ref as lr
from audio_visual_deepfake_detection_b200.libs.modeling.engine import up_weight

D = torch.float64
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def g(seed):
    return torch.Generator().manual_seed(seed)


def rn(gen, *shape, s=1.0):
    return torch.randn(*shape, generator=gen, dtype=D) * s


def close(a, b, tol=1e-10):
    assert a.shape == b.shape, (a.shape, b.shape)
    err = float((a - b).abs().max() / (b.abs().max() + 1e-300))
    assert err < tol, err


def layer_norm(x, w, b):
    return F.layer_norm(x, (x.shape[-1],), w, b, 1e-5)


# --------------------------------------------------------------------------------------------------- conv GEMM
@pytest.mark.parametrize("taps,stride,ln,act,pe,res", [(3, 1, True, lr.ACT_RELU, True, False), (3, 2, False, lr.ACT_NONE, False, True),
                                                       (1, 1, False, lr.ACT_GELU, False, False), (1, 1, False, lr.ACT_NONE, False, True)])
def test_conv_gemm_is_masked_conv1d(taps, stride, ln, act, pe, res):
    r = g(taps * 10 + stride)
    B, T, ci, co = 3, 12, 8, 16
    To = T // stride
    x = rn(r, B, T, ci)
    conv = torch.nn.Conv1d(ci, co, taps, stride=stride, padding=taps // 2).to(D)
    mask = torch.ones(B, To, dtype=torch.uint8)
    mask[1, 7:] = 0; mask[2, 3:] = 0
    lnw, lnb = rn(r, co) * 0.2 + 1, rn(r, co) * 0.2
    pet, rs, gm = rn(r, To, co), rn(r, B, To, co), rn(r, co)
    w = conv.weight.detach().permute(0, 2, 1).reshape(co, taps * ci)
    out = torch.empty(B, To, co)
    got = lr.conv_gemm(x, w, taps=taps, stride=stride, batch=B, c_in=ci, n_out=co, segs=[(To, 0, 0)], a_rows=T, o_rows=To,
                       bias=conv.bias.detach(), row_mask=mask, ln=(lnw, lnb) if ln else None, act=act, pe=pet if pe else None,
                       residual=rs if res else None, gamma=gm if res else None, out_f32=out)["out_f32"]
    m = mask.to(D)[..., None]
    y = conv(x.transpose(1, 2)).detach().transpose(1, 2) * m
    if ln:
        y = layer_norm(y, lnw, lnb)
    y = torch.relu(y) if act == lr.ACT_RELU else (F.gelu(y) if act == lr.ACT_GELU else y)
    if pe:
        y = y + pet * m
    if res:
        y = rs * m + gm * y
    close(got.ref, y)
    assert got.written.all()
    if not ln:                                  # masked rows are exactly zero unless a LayerNorm follows the mask
        assert bool((got.ref[mask == 0] == 0).all()) and bool(got.zero[mask == 0].all())


def test_conv_gemm_segments_weight_blocks_and_pyramid():
    """Per-segment weight blocks (seg[3]) with their own bias / LN / gamma rows, segments at row offsets of a bigger
    output: only the segment rows are written."""
    r = g(1)
    B, ci, co, lens = 2, 8, 4, [6, 3]
    P = sum(lens) + 2
    a = rn(r, B, P, ci)
    ws = [torch.nn.Conv1d(ci, co, 3, padding=1).to(D) for _ in lens]
    w = torch.cat([c.weight.detach().permute(0, 2, 1).reshape(co, 3 * ci) for c in ws])
    bias = torch.cat([c.bias.detach() for c in ws])
    lnw, lnb = rn(r, 2 * co) * 0.1 + 1, rn(r, 2 * co) * 0.1
    segs = [(6, 0, 1, 0), (3, 6, 7, co)]
    out = torch.empty(B, P, co)
    got = lr.conv_gemm(a, w, taps=3, batch=B, c_in=ci, n_out=co, segs=segs, a_rows=P, o_rows=P, bias=bias, ln=(lnw, lnb),
                       act=lr.ACT_RELU, out_f32=out)["out_f32"]
    assert got.written[:, [0, 10]].sum() == 0 and got.written[:, 1:10].all()
    for i, (n, ar, orow, wr) in enumerate(segs):
        y = ws[i](a[:, ar:ar + n].transpose(1, 2)).detach().transpose(1, 2)
        close(got.ref[:, orow:orow + n], torch.relu(layer_norm(y, lnw[wr:wr + co], lnb[wr:wr + co])))


def test_conv_gemm_forward_taps_is_conv_transpose_and_tap_rows_is_conv2d():
    r = g(2)
    B, T, ci, co = 2, 7, 6, 5
    x = rn(r, B, T, ci)
    wt, bias = rn(r, ci, co, 3).float().to(D), rn(r, co)         # (up_weight packs in fp32)
    got = lr.conv_gemm(x, up_weight(wt).to(D), taps=2, batch=B, c_in=ci, n_out=2 * co, segs=[(T, 0, 0)], a_rows=T, o_rows=T,
                       bias=torch.cat([bias, bias]), out_f32=torch.empty(B, T, 2 * co), tap_mode=1)["out_f32"]
    want = F.conv_transpose1d(x.transpose(1, 2), wt, bias, stride=2, padding=1, output_padding=1).transpose(1, 2)
    close(got.ref.reshape(B, 2 * T, co), want)
    # tap_rows: a 3x3 Conv2d over an (H + 2) x (W + 2) zero-padded grid flattened row-major, interior rows read back
    H, W = 4, 5
    img = rn(r, B, ci, H, W)
    k = rn(r, co, ci, 3, 3)
    grid = F.pad(img, (1, 1, 1, 1)).permute(0, 2, 3, 1).reshape(B, (H + 2) * (W + 2), ci)
    rows = (H + 2) * (W + 2)
    tr = [(dy - 1) * (W + 2) + (dx - 1) for dy in range(3) for dx in range(3)]
    wk = k.permute(0, 2, 3, 1).reshape(co, 9 * ci)
    got = lr.conv_gemm(grid, wk, taps=9, batch=B, c_in=ci, n_out=co, segs=[(rows, 0, 0)], a_rows=rows, o_rows=rows,
                       out_f32=torch.empty(B, rows, co), tap_rows=tr)["out_f32"]
    inner = got.ref.reshape(B, H + 2, W + 2, co)[:, 1:-1, 1:-1].permute(0, 3, 1, 2)
    close(inner, F.conv2d(img, k, padding=1))


def test_conv_gemm_ln_after_residual_and_dots():
    r = g(3)
    B, T, C = 2, 5, 8
    x, w, bias, res, gm = rn(r, B, T, C), rn(r, C, C), rn(r, C), rn(r, B, T, C), rn(r, C)
    lnw, lnb = rn(r, C) * 0.1 + 1, rn(r, C) * 0.1
    mask = torch.tensor([[1, 1, 1, 0, 0], [1, 1, 1, 1, 1]], dtype=torch.uint8)
    dw = rn(r, 3, C)
    o = lr.conv_gemm(x, w, taps=1, batch=B, c_in=C, n_out=C, segs=[(T, 0, 0)], a_rows=T, o_rows=T, bias=bias, row_mask=mask,
                     residual=res, gamma=gm, ln=(lnw, lnb), ln_after_residual=True, out_f32=torch.empty(B, T, C),
                     out_h=torch.empty(B, T, C, dtype=torch.float16))
    m = mask.to(D)[..., None]
    y = res * m + gm * ((x @ w.t() + bias) * m)
    close(o["out_f32"].ref, y)
    close(o["out_h"].ref, layer_norm(y, lnw, lnb))
    assert bool((o["out_h"].ref[0, 3:] == lnb).all())           # masked rows: LN of a zero row is the bias
    d = lr.conv_gemm(x, w, taps=1, batch=B, c_in=C, n_out=C, segs=[(T, 0, 0)], a_rows=T, o_rows=T, row_mask=mask,
                     dots=(dw, torch.empty(B, T, 3)))["dots.1"]
    close(d.ref, ((x @ w.t()) * m) @ dw.t())
    assert bool(d.zero[0, 3:].all()) and not bool(d.zero[1].any())


# --------------------------------------------------------------------------------------------------- block kernels
@pytest.mark.parametrize("stride,shift,T_src,T_virt", [(1, 0, 10, 10), (2, 0, 10, 10), (1, 1, 5, 10), (1, -2, 16, 4)])
def test_ln_dwconv_ln_is_layernorm_depthwise_conv_layernorm(stride, shift, T_src, T_virt):
    r = g(stride * 7 + shift + 20)
    B, C = 2, 8
    To = T_virt // stride
    x = rn(r, B, T_src, C)
    lni = [(rn(r, C) * 0.2 + 1, rn(r, C) * 0.2) for _ in range(2)]
    lno = [(rn(r, C) * 0.2 + 1, rn(r, C) * 0.2) for _ in range(2)]
    dws = [rn(r, C, 3) for _ in range(2)]
    mask = torch.ones(B, To, dtype=torch.uint8)
    mask[1, To // 2:] = 0
    out = torch.empty(B, 2 * To + 1, C)               # interleaved: stream i at rows 1 + i * To
    skip = torch.empty(B, To, C) if stride == 2 else None
    got = lr.ln_dwconv_ln(x, batch=B, t_src=T_src, t_virt=T_virt, shift=shift, stride=stride, mask_out=mask, ln_in=lni, dw=dws,
                          ln_out=lno, outs=[out, out], out_rows=2 * To + 1, out_row_offsets=[1, 1 + To], skip_out=skip)
    xv = F.interpolate(x.transpose(1, 2), size=T_virt, mode="nearest")            # backbones.py:487,490
    for i in range(2):
        conv = torch.nn.Conv1d(C, C, 3, stride=stride, padding=1, groups=C, bias=False).to(D)
        conv.weight.data = dws[i].reshape(C, 1, 3)
        u = layer_norm(xv.transpose(1, 2), *lni[i]).transpose(1, 2)
        y = conv(u).detach().transpose(1, 2) * mask.to(D)[..., None]
        close(got["outs.%d" % i].ref[:, 1 + i * To:1 + (i + 1) * To], layer_norm(y, *lno[i]))
        assert got["outs.%d" % i].written[:, 1 + i * To:1 + (i + 1) * To].all() and got["outs.%d" % i].written.sum() == B * To * C
    if skip is not None:
        close(got["skip_out"].ref, F.max_pool1d(x.transpose(1, 2), 3, 2, 1).transpose(1, 2))


def _dense_band_attention(q, k, v, kmask, H, window):
    """Every (query, key) score, the band and the key mask applied to the dense [T, T] matrix."""
    B, T, C = q.shape
    d = C // H
    qh, kh, vh = (z.reshape(B, T, H, d).transpose(1, 2) for z in (q, k, v))
    s = qh @ kh.transpose(-1, -2) / math.sqrt(d)
    if window > 1:
        i = torch.arange(T)
        s = s - 1e4 * (~kmask).to(D)[:, None, None, :]
        s = s.masked_fill((i[:, None] - i[None, :]).abs()[None, None] > window // 2, float("-inf"))
    else:
        s = s.masked_fill(~kmask[:, None, None, :], float("-inf"))
    o = (torch.softmax(s, -1) @ vh).transpose(1, 2).reshape(B, T, C)
    return o * kmask.to(D)[..., None] if window > 1 else o


@pytest.mark.parametrize("window", [7, 5, -1])
def test_attention_is_dense_band_masked_softmax(window):
    r = g(30 + window)
    B, T, C, H = 3, 17, 16, 4
    qkv = rn(r, B, 3 * T, C)
    valid = torch.tensor([T, 9, 1])
    kmask = torch.arange(T)[None] < valid[:, None]
    got = lr.attention(None, None, None, kmask.to(torch.uint8), torch.empty(B, T, C), batch=B, t=T, n_head=H, window=window, qkv=qkv)["out"]
    close(got.ref, _dense_band_attention(qkv[:, :T], qkv[:, T:2 * T], qkv[:, 2 * T:], kmask, H, window))
    if window > 1:                                 # masked query rows are exactly zero, and only those are structural zeros
        assert bool((got.ref[~kmask] == 0).all()) and bool(got.zero[~kmask].all()) and not bool(got.zero[kmask].any())
    none = lr.attention(qkv[:, :T], qkv[:, T:2 * T], qkv[:, 2 * T:], None, torch.empty(B, T, C), batch=B, t=T, n_head=H, window=window)["out"]
    close(none.ref, _dense_band_attention(qkv[:, :T], qkv[:, T:2 * T], qkv[:, 2 * T:], torch.ones(B, T, dtype=torch.bool), H, window))


def test_attention_masked_keys_are_minus_1e4_not_minus_inf():
    """A valid query whose valid keys score below -1e4 attends to the masked key next to it: the additive -1e4 of
    blocks.py:1194-1195 (attention_mma.cu), not a -inf mask."""
    B, T, C, H = 1, 4, 256, 4
    q = torch.full((B, T, C), 60.0, dtype=D)
    k = -q.clone()
    k[0, 1] = 0.0                                  # score 0 for key 1, -8 * 60^2 = -28800 for every valid key
    v = torch.zeros(B, T, C, dtype=D)
    v[0, 1] = 1.0
    mask = torch.tensor([[1, 0, 1, 1]], dtype=torch.uint8)
    o = lr.attention(q, k, v, mask, torch.empty(B, T, C), batch=B, t=T, n_head=H, window=7)["out"].ref
    assert torch.allclose(o[0, 0], torch.ones(C, dtype=D)) and bool((o[0, 1] == 0).all())


def test_ln_rows_and_instnorm():
    r = g(4)
    x, w, b = rn(r, 7, 32) * 3 + 1, rn(r, 32), rn(r, 32)
    got = lr.ln_rows(x, w, b, torch.empty(9, 32), 7)["out"]
    close(got.ref[:7], torch.nn.LayerNorm(32, eps=1e-5).to(D).requires_grad_(False).__call__(x) * w + b)
    assert got.written[:7].all() and not got.written[7:].any()
    B, T, C = 2, 9, 6
    x = rn(r, B, T, C) * 2 + 0.3
    got = lr.instnorm_lrelu(x, torch.empty(B, T, C), batch=B, t=T, channels=C, slope=0.2)["out"]
    close(got.ref, F.leaky_relu(torch.nn.InstanceNorm1d(C)(x.transpose(1, 2)), 0.2).transpose(1, 2))


def test_fpn_fuse():
    r = g(5)
    B, C, lens = 2, 8, [8, 4, 2]
    offs = np.cumsum([0] + lens)
    lat = rn(r, B, sum(lens), C)
    mask = (torch.rand(B, sum(lens), generator=r) > 0.3).to(torch.uint8)
    dw, lw, lb = rn(r, 3, C, 3), rn(r, 3, C) * 0.1 + 1, rn(r, 3, C) * 0.1
    got = lr.fpn_fuse(lat, mask, dw, lw, lb, torch.empty(B, sum(lens), C), batch=B, level_len=lens)["out"]
    lv = [lat[:, offs[l]:offs[l + 1]].transpose(1, 2) for l in range(3)]
    for l in (2, 1):
        lv[l - 1] = lv[l - 1] + F.interpolate(lv[l], size=lens[l - 1], mode="nearest")
    for l in range(3):
        z = F.conv1d(lv[l], dw[l].reshape(C, 1, 3), padding=1, groups=C).transpose(1, 2) * mask[:, offs[l]:offs[l + 1], None]
        close(got.ref[:, offs[l]:offs[l + 1]], layer_norm(z, lw[l], lb[l]))


def test_head_final_head_combine_and_zeros():
    r = g(6)
    B, C, lens = 2, 8, [6, 3]
    P = sum(lens)
    offs = [0, 6, 9]
    cf, rf = torch.relu(rn(r, B, P, C)), torch.relu(rn(r, B, P, C))
    cw, cb, rw, rb = rn(r, 1, C, 3), rn(r, 1), rn(r, 2, C, 3), rn(r, 2)
    mask = torch.ones(B, P, dtype=torch.uint8)
    mask[1, 4:6] = 0; mask[1, 8] = 0
    sc = [0.7, 1.3]
    lg, of = torch.empty(B, P), torch.empty(B, P, 2)
    got = lr.head_final(cf, rf, mask, cw.permute(0, 2, 1).reshape(1, 3 * C), cb, rw.permute(0, 2, 1).reshape(2, 3 * C), rb, sc,
                        lg, of, batch=B, level_len=lens)
    for l in range(2):
        m = mask[:, offs[l]:offs[l + 1]].to(D)
        close(got["logits"].ref[:, offs[l]:offs[l + 1]], F.conv1d(cf[:, offs[l]:offs[l + 1]].transpose(1, 2), cw, cb, padding=1)[:, 0] * m)
        want = torch.relu(F.conv1d(rf[:, offs[l]:offs[l + 1]].transpose(1, 2), rw, rb, padding=1) * m[:, None] * sc[l]).transpose(1, 2)
        close(got["offsets"].ref[:, offs[l]:offs[l + 1]], want)
    assert bool(got["logits"].zero[mask == 0].all()) and bool(got["offsets"].zero[mask == 0].all())
    clamped = got["offsets"].zero & (mask != 0)[..., None]
    assert bool((got["offsets"].ref[clamped] == 0).all())
    # the same heads from per-tap partial sums of the towers
    cd = torch.einsum("bpc,ocj->bpoj", cf, cw).reshape(B, P, 3)
    rd = torch.einsum("bpc,ocj->bpoj", rf, rw).reshape(B, P, 6)
    comb = lr.head_combine(cd, rd, mask, cb, rb, sc, lg, of, batch=B, level_len=lens)
    close(comb["logits"].ref, got["logits"].ref)
    close(comb["offsets"].ref, got["offsets"].ref)


def test_vcls_tails():
    r = g(7)
    B, T, C = 2, 5, 8
    z = rn(r, B, T, C)
    w0, w1 = rn(r, C, C), rn(r, C, 2 * C)
    lw, lb, w2, b2 = rn(r, C) * 0.1 + 1, rn(r, C) * 0.1, rn(r, C), rn(r, 1)
    got = lr.vcls_exp12(z, w0.t(), w1.t(), lw, lb, w2, b2, torch.empty(B), batch=B, t=T)["out"]
    conv0 = torch.nn.Conv1d(C, C, 1, bias=False).to(D)
    conv0.weight.data = w0[..., None]
    gg = F.leaky_relu(torch.nn.InstanceNorm1d(C)(conv0(z.transpose(1, 2))), 0.2).detach()
    h = torch.relu(layer_norm(torch.cat([gg.amax(2), gg.mean(2)], 1) @ w1.t(), lw, lb))
    close(got.ref, h @ w2 + b2)
    sw, sb, cw, cb = rn(r, C), rn(r, 1), rn(r, 2), rn(r, 1)
    got = lr.vcls_exp13(z, w0, sw, sb, cw, cb, torch.empty(B), batch=B, t=T)["out"]
    s = torch.einsum("bct,c->bt", gg, sw) + sb
    close(got.ref, cw[0] * s.amax(1) + cw[1] * s.mean(1) + cb)


@pytest.mark.parametrize("proj", [False, True])
def test_mlp_fused(proj):
    """Linear -> exact GELU -> 16-bit hidden -> Linear -> mask / gamma / residual; the block tail adds the projection and
    a 16-bit LN2 operand in front."""
    r = g(8 + proj)
    rows, C, H, dt = 6, 8, 32, torch.float16
    x = rn(r, rows, C).to(dt)
    w1, w2 = rn(r, H, C).to(dt), (rn(r, C, H) / 4).to(dt)
    b1, b2, gm, res = rn(r, H), rn(r, C), rn(r, C), rn(r, rows, C)
    mask = torch.tensor([1, 1, 0, 1, 0, 1], dtype=torch.uint8)
    m = mask.to(D)[:, None]
    lin1, lin2 = torch.nn.Linear(C, H).to(D), torch.nn.Linear(H, C).to(D)
    lin1.weight.data, lin1.bias.data, lin2.weight.data, lin2.bias.data = w1.to(D), b1, w2.to(D), b2
    if not proj:
        got = lr.mlp_fused(x, w1, b1, w2, b2, row_mask=mask, residual=res, gamma=gm, out=torch.empty(rows, C),
                           out_h=torch.empty(2, 5, C, dtype=dt), out_h_level=(3, 5, 1))
        want = res * m + gm * (lin2(F.gelu(lin1(x.to(D))).to(dt).to(D)).detach() * m)
        close(got["out"].ref, want)
        assert got["out_h"].written[:, 1:4].all() and got["out_h"].written.sum() == rows * C
        close(got["out_h"].ref[:, 1:4].reshape(rows, C), want)
    else:
        att, wo, bo, ga, skip = rn(r, rows, C).to(dt), rn(r, C, C).to(dt), rn(r, C), rn(r, C), rn(r, rows, C)
        lnw, lnb = rn(r, C) * 0.1 + 1, rn(r, C) * 0.1
        got = lr.mlp_fused(None, w1, b1, w2, b2, row_mask=mask, residual=None, gamma=None, out=torch.empty(rows, C),
                           proj=(att, wo, bo, ga, (lnw, lnb), skip, torch.empty(rows, C)))
        y = skip * m + ga * ((att.to(D) @ wo.to(D).t() + bo) * m)
        want = (y + lin2(F.gelu(lin1(layer_norm(y, lnw, lnb).to(dt).to(D))).to(dt).to(D)).detach()) * m
        close(got["proj.6"].ref, y)
        close(got["out"].ref, want)
    assert bool((got["out"].ref[mask == 0] == 0).all()) and bool(got["out"].zero[mask == 0].all())


def test_interp_concat_and_pack_feats():
    r = np.random.RandomState(9)
    a, b = r.standard_normal((5, 8)).astype(np.float32), r.standard_normal((12, 8)).astype(np.float32)
    e = r.standard_normal((16, 16)).astype(np.float32)
    s0 = torch.from_numpy(np.concatenate([a, b]))
    s2 = torch.from_numpy(np.concatenate([e, e[:9]]))
    o0, o2 = torch.tensor([0, 5, 17], dtype=torch.int32), torch.tensor([0, 16, 25], dtype=torch.int32)
    out = torch.empty(2, 16, 24)
    got = lr.interp_concat([s0, None, s2], [o0, None, o2], 16, out)["out"].ref
    for bi, (v, em) in enumerate(((a, e), (b, e[:9]))):
        want = torch.cat([F.interpolate(torch.from_numpy(z.T.copy()).to(D)[None], size=16, mode="linear", align_corners=False)[0].t()
                          for z in (v, em)], 1)
        close(got[bi], want, 1e-6)                  # the blend weights are the kernel's fp32 index math
    start = torch.tensor([[0, 5], [0, 0], [0, 16]], dtype=torch.int32)
    count = torch.tensor([[5, 12], [0, 0], [16, 9]], dtype=torch.int32)
    assert torch.equal(lr.interp_concat_ranges([s0, None, s2], start, count, 16, out)["out"].ref, got)
    f = torch.from_numpy(r.standard_normal((8, 5)).astype(np.float32))
    p = lr.pack_feats(f, torch.empty(7, 8))["out"]
    assert torch.equal(p.ref[:5], f.t().to(D)) and bool((p.ref[5:] == 0).all()) and bool(p.zero[5:].all()) and not p.zero[:5].any()


# --------------------------------------------------------------------------------------------------- coverage
def launched_entry_points():
    names = set()
    for rel in ("audio_visual_deepfake_detection_b200/libs/modeling/engine.py", "audio_visual_deepfake_detection_b200/libs/modeling/meta_archs.py"):
        with open(os.path.join(ROOT, rel)) as f:
            names |= set(re.findall(r"\bops\.(\w+)\(", f.read()))
    return names


def test_every_launched_entry_point_has_a_reference():
    from audio_visual_deepfake_detection_b200 import ops
    names = launched_entry_points()
    assert {"conv_gemm", "attention", "mlp_fused", "ln_dwconv_ln"} <= names
    missing = sorted(n for n in names if n not in lr.REFERENCES and n not in lr.EXCLUDED)
    assert not missing, "ops entry points launched by the forward pass without a float64 reference: %s" % missing
    assert set(lr.EXCLUDED) == {"postprocess"}
    import inspect
    for name, ref in lr.REFERENCES.items():           # the references take the entry points' own arguments
        assert list(inspect.signature(ref).parameters) == list(inspect.signature(getattr(ops, name)).parameters), name
