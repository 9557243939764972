"""GPU parity tests of every C-ABI kernel against the oracle (oracle/*.py, oracle/nms_ref.c) and the
golden fixtures written by the unmodified reference (tests/golden). Run on the B200 box:
    python -m pytest tests -m gpu -q
Integer / index results are compared bit-exactly; fp32 kernels within 1e-4 (BASELINE.json fp32 mode),
bf16 tensor-core GEMMs within 1e-2 relative.
"""
import json
import math
import os
import zlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import interp_ref
import launch_ref
import model_ref
import nms_ref
from make_golden import sweep_inputs
from audio_visual_deepfake_detection_b200 import native as nv
from audio_visual_deepfake_detection_b200 import ops
from audio_visual_deepfake_detection_b200.libs.utils import synthetic as syn

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
DEV = "cuda"


def dev(a, dtype=None):
    t = torch.as_tensor(a)
    if dtype is not None:
        t = t.to(dtype)
    return t.contiguous().to(DEV)


def rel_err(a, b):
    a, b = a.double(), b.double()
    return float((a - b).abs().max() / (b.abs().max() + 1e-12))


# --------------------------------------------------------------------------------------------- K1
def _pack_streams(stream_list, key):
    arrs = [s[key] for s in stream_list]
    off = np.zeros(len(arrs) + 1, np.int32)
    off[1:] = np.cumsum([a.shape[0] for a in arrs])
    return dev(np.concatenate(arrs, 0)), dev(off)


@pytest.mark.parametrize("use_video", [True, False])
def test_interp_concat_bit_exact(use_video):
    durs = [4.03, 7.42, 18.75, 33.02, 30.72]
    sl = [syn.synthetic_streams(d, 500 + i, video_dim=256 if use_video else 0) for i, d in enumerate(durs)]
    # one stream already at 768 rows exercises the identity branch
    sl[4]["emo"] = np.random.RandomState(1).standard_normal((768, 768)).astype(np.float32)
    names = ("video", "byola", "emo")
    streams, offs = [], []
    for n in names:
        if n in sl[0]:
            s, o = _pack_streams(sl, n)
            streams.append(s); offs.append(o)
        else:
            streams.append(None); offs.append(None)
    C = sum(s.shape[1] for s in streams if s is not None)
    out = torch.empty((len(durs), 768, C), dtype=torch.float32, device=DEV)
    ops.interp_concat(streams, offs, 768, out)
    ref = np.stack([np.concatenate([interp_ref.linear_resize_tc(s[n], 768) for n in names if n in s], 1) for s in sl])
    assert np.array_equal(out.cpu().numpy(), ref)
    out16 = torch.empty((len(durs), 768, C), dtype=torch.bfloat16, device=DEV)
    ops.interp_concat(streams, offs, 768, out16)
    assert torch.equal(out16.cpu(), torch.from_numpy(ref).to(torch.bfloat16))


def test_interp_golden():
    g = np.load(os.path.join(GOLD, "interp.npz"))
    for i, dur in enumerate(g["durations"]):
        st = syn.synthetic_streams(float(dur), 500 + i)
        for k, v in st.items():
            out = torch.empty((1, 768, v.shape[1]), dtype=torch.float32, device=DEV)
            s, o = dev(v), dev(np.array([0, v.shape[0]], np.int32))
            args = {"video": ([s, None, None], [o, None, None]), "byola": ([None, s, None], [None, o, None]),
                    "emo": ([None, None, s], [None, None, o])}[k]
            ops.interp_concat(args[0], args[1], 768, out)
            flat = out.cpu().numpy().reshape(-1)
            assert np.array_equal(flat[g[f"{i}_{k}_pos"]], g[f"{i}_{k}_val"]), (i, k)


def test_pack_feats():
    rng = np.random.RandomState(0)
    for C, T, L in ((3072, 768, 768), (2816, 500, 768), (96, 801, 864)):
        f = rng.standard_normal((C, T)).astype(np.float32)
        for dt in (torch.float32, torch.bfloat16):
            out = torch.full((L, C), 7.0, dtype=dt, device=DEV)
            ops.pack_feats(dev(f), out)
            ref = torch.zeros((L, C), dtype=torch.float32)
            ref[:T] = torch.from_numpy(f.T.copy())
            assert torch.equal(out.cpu(), ref.to(dt))


# --------------------------------------------------------------------------------------------- NMS
def test_nms_known_answers_gpu():
    kat = json.load(open(os.path.join(GOLD, "nms_kat.json")))
    for rec in kat:
        segs = np.array(rec["segs"], np.float32).reshape(-1, 2)
        sc = np.array(rec["scores"], np.float32)
        if len(sc) == 0:
            continue
        for thr in (0.1, 0.5):
            got = ops.nms_hard(dev(segs), dev(sc), thr).cpu().tolist()
            assert got == rec[f"nms_thr{thr}"], (rec["name"], thr)
        for m in (0, 1, 2):
            dets = torch.zeros((len(sc), 3), device=DEV)
            got = ops.nms_soft(dev(segs), dev(sc), dets, 0.1, 0.75, 0.2, m).cpu().tolist()
            assert got == rec[f"softnms_m{m}"]["inds"], (rec["name"], m)
            want = np.array(rec[f"softnms_m{m}"]["dets"], np.float32).reshape(-1, 3)
            assert np.array_equal(dets[:len(got)].cpu().numpy(), want), (rec["name"], m)


@pytest.mark.parametrize("n", [1000, 1512, 10000, 100000])
def test_nms_sweep_bit_exact_gpu(n):
    g = np.load(os.path.join(GOLD, "nms_sweep.npz"))
    segs, sc = sweep_inputs(n, 7000 + n)
    keep = sc > 0.2
    got = ops.nms_hard(dev(segs[keep]), dev(sc[keep]), 0.1).cpu().numpy()
    assert np.array_equal(got, g[f"hard_{n}"])
    # early stop after max_num picks returns the same prefix
    got100 = ops.nms_hard(dev(segs[keep]), dev(sc[keep]), 0.1, max_num=100).cpu().numpy()
    assert np.array_equal(got100, g[f"hard_{n}"][:100])
    dets = torch.zeros((n, 3), device=DEV)
    inds = ops.nms_soft(dev(segs), dev(sc), dets, 0.1, 0.75, 0.2, 2).cpu().numpy()
    assert np.array_equal(inds, g[f"soft_{n}_inds"])
    assert np.array_equal(dets[:len(inds), 2].cpu().numpy(), g[f"soft_{n}_scores"])


@pytest.mark.parametrize("method", [0, 1, 2])
def test_nms_soft_vs_oracle_random(method):
    rng = np.random.RandomState(5 + method)
    for n in (1, 2, 3, 17, 333, 2000, 7000):
        segs, sc = sweep_inputs(n, 40 + n)
        thr = float(rng.choice([0.1, 0.3, 0.5]))
        want_i, want_d = nms_ref.softnms(segs, sc, thr, 0.75, 0.2, method)
        dets = torch.zeros((n, 3), device=DEV)
        got = ops.nms_soft(dev(segs), dev(sc), dets, thr, 0.75, 0.2, method).cpu().numpy()
        assert np.array_equal(got, want_i), (n, method)
        assert np.array_equal(dets[:len(got)].cpu().numpy(), want_d), (n, method)
        assert np.array_equal(ops.nms_hard(dev(segs), dev(sc), thr).cpu().numpy(), nms_ref.nms(segs, sc, thr))


def _run_batched(cases, soft, voting=0.9, K=100):
    B = len(cases)
    cap = max(len(s) for _, s in cases)
    cs = torch.zeros((B, cap, 2), device=DEV); cc = torch.zeros((B, cap), device=DEV)
    cn = torch.zeros(B, dtype=torch.int32, device=DEV)
    for b, (segs, sc) in enumerate(cases):
        cs[b, :len(sc)] = dev(segs); cc[b, :len(sc)] = dev(sc); cn[b] = len(sc)
    osg = torch.zeros((B, K, 2), device=DEV); osc = torch.zeros((B, K), device=DEV)
    ocn = torch.zeros(B, dtype=torch.int32, device=DEV)
    ops.postprocess(B, cand_segs=cs, cand_scores=cc, cand_count=cn, iou_threshold=0.1, min_score=0.2, sigma=0.75,
                    voting_thresh=voting, max_seg_num=K, use_soft_nms=soft, out_segs=osg, out_scores=osc, out_count=ocn)
    return osg.cpu().numpy(), osc.cpu().numpy(), ocn.cpu().numpy()


@pytest.mark.parametrize("soft", [False, True])
def test_batched_nms_candidates(soft):
    g = np.load(os.path.join(GOLD, "nms_sweep.npz"))
    sizes = (1000, 1512, 10000)
    cases = [sweep_inputs(n, 7000 + n) for n in sizes]
    cases.append((np.zeros((0, 2), np.float32), np.zeros(0, np.float32)))          # a video without candidates
    cases.append((np.array([[0, 10], [1, 11], [20, 30]], np.float32), np.array([.19, .1, .05], np.float32)))
    segs, scores, counts = _run_batched(cases, soft)
    tag = "soft" if soft else "hard"
    for b, n in enumerate(sizes):
        gs, gp = g[f"batched_{tag}_{n}_segs"], g[f"batched_{tag}_{n}_scores"]
        assert counts[b] == len(gp)
        assert np.array_equal(scores[b, :counts[b]], gp)
        np.testing.assert_allclose(segs[b, :counts[b]], gs, atol=1e-4)
    assert counts[3] == 0
    assert counts[4] == (1 if soft else 0)       # SURVEY.md 8c: all below min_score -> hard empty, soft keeps the max


def test_batched_nms_100k_workspace_path():
    g = np.load(os.path.join(GOLD, "nms_sweep.npz"))
    case = sweep_inputs(100000, 7000 + 100000)
    for soft in (False, True):
        tag = "soft" if soft else "hard"
        segs, scores, counts = _run_batched([case], soft)
        gp = g[f"batched_{tag}_100000_scores"]
        assert counts[0] == len(gp)
        assert np.array_equal(scores[0, :counts[0]], gp)
        np.testing.assert_allclose(segs[0, :counts[0]], g[f"batched_{tag}_100000_segs"], atol=1e-4)


def test_decode_postprocess_vs_oracle():
    """decode (av_fd_no_recon.py:775-823) + batched_nms + seconds conversion, ragged masks."""
    rng = np.random.RandomState(11)
    B, lens = 5, [768, 384, 192, 96, 48, 24]
    P = sum(lens)
    strides = [2.0 ** l for l in range(6)]
    logits = rng.normal(-2.0, 2.5, (B, P)).astype(np.float32)
    offsets = np.abs(rng.normal(0, 6, (B, P, 2))).astype(np.float32)
    offsets[:, ::7] = 0.0                                    # zero-length segments -> duration filter
    valid = [768, 500, 640, 768, 97]
    mask = np.concatenate([(np.arange(n)[None] * s < np.array(valid)[:, None]) for n, s in zip(lens, strides)], 1).astype(np.uint8)
    durs = [4.03, 9.04, 26.37, 7.42, 12.0]
    meta = np.zeros((4, B), np.float32)
    items = []
    for b, d in enumerate(durs):
        t_v = int(round(25 * d)); fs = t_v / 768.0
        items.append({"feat_stride": fs, "feat_num_frames": fs, "fps": t_v / d, "duration": d})
        meta[:, b] = [np.float32(fs), np.float32(0.5 * fs), np.float32(t_v / d), np.float32(d)]
    cfg = {"pre_nms_thresh": 0.001, "pre_nms_topk": 200, "iou_threshold": 0.1, "min_score": 0.2, "max_seg_num": 100,
           "nms_sigma": 0.75, "duration_thresh": 0.001, "multiclass_nms": False, "voting_thresh": 0.9}

    class Stub(model_ref.OracleModel):
        def __init__(self):
            self.test_cfg = dict(cfg); self.fpn_strides = [1, 2, 4, 8, 16, 32]; self.num_classes = 1
    om = Stub()
    for method in ("hard", "soft"):
        om.test_cfg["nms_method"] = method
        cs = torch.zeros((B, P, 2), device=DEV); cc = torch.zeros((B, P), device=DEV)
        cn = torch.zeros(B, dtype=torch.int32, device=DEV)
        osg = torch.zeros((B, 100, 2), device=DEV); osc = torch.zeros((B, 100), device=DEV)
        ocn = torch.zeros(B, dtype=torch.int32, device=DEV)
        md = dev(meta)
        ops.postprocess(B, logits=dev(logits), offsets=dev(offsets), mask=dev(mask), level_len=lens, level_stride=strides,
                        pre_nms_thresh=0.001, pre_nms_topk=200, duration_thresh=0.001, cand_segs=cs, cand_scores=cc,
                        cand_count=cn, iou_threshold=0.1, min_score=0.2, sigma=0.75, voting_thresh=0.9, max_seg_num=100,
                        use_soft_nms=(method == "soft"), vid_meta=[md[0], md[1], md[2], md[3]], out_segs=osg,
                        out_scores=osc, out_count=ocn)
        for b in range(B):
            off = np.cumsum([0] + lens)
            lg = [torch.from_numpy(logits[b, off[l]:off[l + 1]]).unsqueeze(-1) for l in range(6)]
            of = [torch.from_numpy(offsets[b, off[l]:off[l + 1]]) for l in range(6)]
            ms = [torch.from_numpy(mask[b, off[l]:off[l + 1]].astype(bool)) for l in range(6)]
            segs, scores, labels = om.decode(lg, of, ms)
            n = int(cn[b])
            assert n == len(scores), (method, b)
            # sigmoid: the device expf differs from torch's by <= 2 ulp -> scores within 1e-6, same order
            np.testing.assert_allclose(cc[b, :n].cpu().numpy(), scores.numpy(), atol=2e-6, rtol=0)
            np.testing.assert_allclose(cs[b, :n].cpu().numpy(), segs.numpy(), atol=1e-5)
            fs, fp, fl = om.postprocess(segs, scores, labels, items[b], nms_ref.batched_nms)
            k = int(ocn[b])
            assert k == len(fp), (method, b)
            np.testing.assert_allclose(osc[b, :k].cpu().numpy(), fp.numpy(), atol=5e-6)
            np.testing.assert_allclose(osg[b, :k].cpu().numpy(), fs.numpy().reshape(-1, 2), atol=1e-3)


# --------------------------------------------------------------------------------------------- conv GEMM
def _conv_ref(x_btc, w, bias, taps, stride, mask_bt, ln, act, pe, residual, gamma):
    """plain torch fp32 reference: MaskedConv1D (+LN, act, PE, residual) on token-major input."""
    x = x_btc.permute(0, 2, 1)                                           # [B, C, T]
    y = F.conv1d(x, w, bias, stride=stride, padding=taps // 2)
    m = mask_bt[:, None, :].to(y.dtype)
    y = y * m
    if ln is not None:
        y = model_ref.channel_ln(y, ln[0], ln[1])
    if act == ops.ACT_RELU:
        y = torch.relu(y)
    elif act == ops.ACT_GELU:
        y = model_ref.gelu_erf(y)
    if pe is not None:
        y = y + pe.t()[None] * m
    if residual is not None:
        g = gamma.view(1, -1, 1) if gamma is not None else 1.0
        y = residual.permute(0, 2, 1) * m + g * y
    return y.permute(0, 2, 1).contiguous()


GEMM_CASES = [
    # name, B, T_in, c_in, n_out, taps, stride, bias, ln, act, pe, residual
    ("embd_k3_ln_relu_pe", 3, 96, 128, 256, 3, 1, False, True, ops.ACT_RELU, True, False),
    ("proj_1x1_res", 5, 64, 256, 256, 1, 1, True, False, ops.ACT_NONE, False, True),
    ("mlp_1x1_gelu", 2, 48, 256, 1024, 1, 1, True, False, ops.ACT_GELU, False, False),
    ("mlp2_1x1_res", 2, 48, 1024, 256, 1, 1, True, False, ops.ACT_NONE, False, True),
    ("down_k3_s2", 4, 192, 192, 512, 3, 2, True, False, ops.ACT_NONE, False, False),
    ("extract_k3_n64", 2, 256, 128, 64, 3, 1, True, False, ops.ACT_NONE, False, False),
    ("odd_batch_small_t", 33, 24, 64, 256, 3, 1, False, True, ops.ACT_RELU, False, False),
]


@pytest.mark.parametrize("case", GEMM_CASES, ids=[c[0] for c in GEMM_CASES])
@pytest.mark.parametrize("mode", ["fp32", "bf16", "fp16"])
def test_conv_gemm(case, mode):
    name, B, T, cin, nout, taps, stride, has_bias, has_ln, act, has_pe, has_res = case
    rng = np.random.RandomState(zlib.crc32(name.encode()) % 1000)
    To = T // stride
    x = torch.from_numpy(rng.standard_normal((B, T, cin)).astype(np.float32))
    w = torch.from_numpy((rng.standard_normal((nout, cin, taps)) / math.sqrt(cin * taps)).astype(np.float32))
    bias = torch.from_numpy(rng.normal(0, 0.3, nout).astype(np.float32)) if has_bias else None
    ln = (torch.from_numpy(rng.uniform(0.5, 1.5, nout).astype(np.float32)),
          torch.from_numpy(rng.normal(0, 0.2, nout).astype(np.float32))) if has_ln else None
    pe = torch.from_numpy(rng.normal(0, 0.1, (To, nout)).astype(np.float32)) if has_pe else None
    res = torch.from_numpy(rng.standard_normal((B, To, nout)).astype(np.float32)) if has_res else None
    gamma = torch.from_numpy(rng.uniform(0.5, 1.5, nout).astype(np.float32)) if has_res else None
    valid = rng.randint(To // 2, To + 1, B); valid[0] = To
    mask = (np.arange(To)[None] < valid[:, None])
    adt = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}[mode]
    xq, wq = x.to(adt).float(), w.to(adt).float()                       # what the kernel actually multiplies
    want = _conv_ref(xq, wq, bias, taps, stride, torch.from_numpy(mask), ln, act, pe, res, gamma)
    wp = w.permute(0, 2, 1).reshape(nout, taps * cin).contiguous()
    out32 = torch.zeros((B, To, nout), device=DEV)
    out16 = torch.zeros((B, To, nout), dtype=adt, device=DEV) if mode != "fp32" else None
    ops.conv_gemm(dev(x, adt), dev(wp, adt), taps=taps, stride=stride, batch=B, c_in=cin, n_out=nout, segs=[(To, 0, 0)],
                  a_rows=T, o_rows=To, bias=None if bias is None else dev(bias), row_mask=dev(mask.astype(np.uint8)),
                  ln=None if ln is None else (dev(ln[0]), dev(ln[1])), act=act, pe=None if pe is None else dev(pe),
                  residual=None if res is None else dev(res), gamma=None if gamma is None else dev(gamma),
                  out_f32=out32, out_h=out16)
    torch.cuda.synchronize()
    tol = 2e-5 if mode == "fp32" else 2e-4      # same operands, only the accumulation order differs
    err = rel_err(out32.cpu(), want)
    assert err < tol, (name, mode, err)
    if out16 is not None:
        assert rel_err(out16.float().cpu(), want) < 1e-2


@pytest.mark.parametrize("mode", ["fp32", "bf16", "fp16"])
def test_conv_gemm_pyramid_segments(mode):
    """k3 conv over a 6-level pyramid in ONE launch (head towers): levels must not bleed into each other."""
    rng = np.random.RandomState(3)
    B, C, lens = 3, 256, [96, 48, 24, 12]
    P = sum(lens)
    offs = np.cumsum([0] + lens)
    x = torch.from_numpy(rng.standard_normal((B, P, C)).astype(np.float32))
    w = torch.from_numpy((rng.standard_normal((C, C, 3)) / math.sqrt(3 * C)).astype(np.float32))
    ln = (torch.from_numpy(rng.uniform(0.5, 1.5, C).astype(np.float32)), torch.from_numpy(rng.normal(0, 0.2, C).astype(np.float32)))
    mask = rng.rand(B, P) > 0.2
    adt = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}[mode]
    xq, wq = x.to(adt).float(), w.to(adt).float()
    want = torch.cat([_conv_ref(xq[:, offs[l]:offs[l + 1]], wq, None, 3, 1, torch.from_numpy(mask[:, offs[l]:offs[l + 1]]), ln,
                                ops.ACT_RELU, None, None, None) for l in range(len(lens))], dim=1)
    out = torch.zeros((B, P, C), device=DEV)
    ops.conv_gemm(dev(x, adt), dev(w.permute(0, 2, 1).reshape(C, 3 * C), adt), taps=3, batch=B, c_in=C, n_out=C,
                  segs=[(lens[l], int(offs[l]), int(offs[l])) for l in range(len(lens))], a_rows=P, o_rows=P,
                  row_mask=dev(mask.astype(np.uint8)), ln=(dev(ln[0]), dev(ln[1])), act=ops.ACT_RELU, out_f32=out)
    assert rel_err(out.cpu(), want) < (2e-5 if mode == "fp32" else 2e-4)


# --------------------------------------------------------------------------------------------- block kernels
def _ln_params(rng, C=256):
    return (torch.from_numpy(rng.uniform(0.5, 1.5, C).astype(np.float32)), torch.from_numpy(rng.normal(0, 0.2, C).astype(np.float32)))


LDL_CASES = [pytest.param(*c, 3, torch.float32, id="%d-%d-%d-%d" % c)
             for c in [(1, 0, 96, 96), (2, 0, 96, 96), (1, 2, 24, 96), (1, -3, 192, 24), (1, 0, 20, 20)]]
LDL_CASES += [pytest.param(*c, id="%d-%d-%d-%d-%dstreams-%s" % (c[:5] + (str(c[5])[6:],)))
              for c in [(1, 2, 24, 96, 2, torch.float32), (1, -3, 192, 24, 2, torch.float16),      # the cross-modal K / V
                        (1, 1, 48, 96, 1, torch.float32), (1, -1, 192, 96, 1, torch.float16),
                        (2, 0, 96, 96, 2, torch.float32), (2, 0, 96, 96, 1, torch.float16),       # stride 2 without skip_out
                        (1, 0, 96, 96, 3, torch.float16), (2, 0, 96, 96, 3, torch.float16)]]


@pytest.mark.parametrize("tile_rows", [0, 2, 4, 8])
@pytest.mark.parametrize("stride,shift,T_src,T_virt,n_streams,out_dt", LDL_CASES)
def test_ln_dwconv_ln(stride, shift, T_src, T_virt, tile_rows, n_streams, out_dt):
    """tile_rows 0 is the automatic choice: two or three streams take the second-layout kernel (the K / V of every
    cross-modal block: two streams, shift != 0), one stream the first layout with automatic tile rows. Stride 2 with
    fewer than three streams runs without skip_out."""
    rng = np.random.RandomState(7)
    B, C = 3, 256
    To = T_virt // stride
    x = torch.from_numpy(rng.standard_normal((B, T_src, C)).astype(np.float32) * 2 + 0.5)
    lni = [_ln_params(rng) for _ in range(3)]
    lno = [_ln_params(rng) for _ in range(3)]
    dws = [torch.from_numpy(rng.normal(0, 0.6, (C, 3)).astype(np.float32)) for _ in range(3)]
    valid = np.array([To, To // 2, To - 1])
    mask = np.arange(To)[None] < valid[:, None]
    outs = [torch.full((B, To, C), float("nan"), dtype=out_dt, device=DEV) for _ in range(n_streams)]
    skip = torch.full((B, To, C), float("nan"), device=DEV) if (stride == 2 and n_streams == 3) else None
    kw = dict(batch=B, t_src=T_src, t_virt=T_virt, shift=shift, stride=stride, mask_out=dev(mask.astype(np.uint8)),
              ln_in=[(dev(a), dev(b)) for a, b in lni[:n_streams]], dw=[dev(d) for d in dws[:n_streams]],
              ln_out=[(dev(a), dev(b)) for a, b in lno[:n_streams]], outs=outs, skip_out=skip, tile_rows=tile_rows)
    ops.ln_dwconv_ln(dev(x), **kw)
    ref = launch_ref.ln_dwconv_ln(dev(x), **kw)
    for s in range(n_streams):
        launch_ref.check(outs[s], ref["outs.%d" % s], C, 5e-5, "stream %d" % s)
    xc = x.permute(0, 2, 1)
    idx = (torch.arange(T_virt) >> shift) if shift >= 0 else (torch.arange(T_virt) << -shift)
    xv = xc[..., idx]                                                  # nearest resample (backbones.py:487,490)
    for s in range(n_streams if out_dt == torch.float32 else 0):
        u = model_ref.channel_ln(xv, *lni[s])
        y = F.conv1d(u, dws[s].view(C, 1, 3), None, stride=stride, padding=1, groups=C) * torch.from_numpy(mask)[:, None, :].float()
        y = model_ref.channel_ln(y, *lno[s]).permute(0, 2, 1)
        assert rel_err(outs[s].cpu(), y) < 2e-5, s
    if skip is not None:
        want = model_ref.max_pool_3_2_1(xc).permute(0, 2, 1)
        assert torch.equal(skip.cpu(), want.contiguous())


ATT_CASES = [pytest.param(w, t, "plain", id="%d-%d" % (w, t)) for w, t in [(7, 96), (7, 5), (-1, 24), (-1, 48), (7, 17), (7, 33),
                                                                         (7, 100), (7, 768), (-1, 17), (-1, 100)]]
ATT_CASES += [pytest.param(w, t, v, id="%d-%d-%s" % (w, t, v)) for w, t, v in [(7, 96, "out16"), (-1, 48, "out16"), (7, 768, "out16"),
                                                                               (7, 96, "no_mask"), (-1, 24, "no_mask"),
                                                                               (7, 768, "sm_batch"), (7, 192, "sm_batch")]]


@pytest.mark.parametrize("window,T,variant", ATT_CASES)
@pytest.mark.parametrize("in_dt", [torch.float32, torch.bfloat16, torch.float16])
def test_attention(window, T, in_dt, variant):
    """plain: the fp32 output; out16: the 16-bit output the engine writes in mixed precision; no_mask: kv_mask=None;
    sm_batch: a batch that gives the tensor-core kernel its 64-row CTAs (as batch 32 does at T = 768). Video 1 ends
    after one row: its later query rows have their whole band masked."""
    if variant == "sm_batch" and (window != 7 or in_dt == torch.float32):
        pytest.skip("the 64-row CTAs belong to the 16-bit window-7 kernel")
    rng = np.random.RandomState(9)
    C, H = 256, 4
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    B = 3 if variant != "sm_batch" else max(3, -(-sms // -(-T // 64)))          # batch * ceil(T / 64) >= SM count
    q, k, v = (torch.from_numpy(rng.standard_normal((B, T, C)).astype(np.float32)).to(in_dt) for _ in range(3))
    valid = np.array([T, 1, T - 1] + [int(x) for x in rng.randint(1, T + 1, B - 3)])
    mask = torch.from_numpy(np.arange(T)[None] < valid[:, None])
    out_dt = torch.float16 if variant == "out16" else torch.float32
    out = torch.full((B, T, C), float("nan"), dtype=out_dt, device=DEV)
    km = None if variant == "no_mask" else dev(mask.to(torch.uint8))
    ops.attention(dev(q), dev(k), dev(v), km, out, batch=B, t=T, n_head=H, window=window)
    ref = launch_ref.attention(dev(q), dev(k), dev(v), km, out, batch=B, t=T, n_head=H, window=window)["out"]
    launch_ref.check(out, ref, C, 5e-5, "attention")
    if variant == "plain" and B == 3:
        qc, kc, vc = (t.float().permute(0, 2, 1).contiguous() for t in (q, k, v))
        if window > 1:
            want = model_ref.banded_attention(qc, kc, vc, mask[:, None, :], H, window // 2)
        else:
            want = model_ref.global_attention(qc, kc, vc, mask[:, None, :], H)
            want = want * mask[:, None, :].float()          # masked query rows are zeroed by the proj mask downstream
            out = out * dev(mask.float())[:, :, None]
        assert rel_err(out.cpu(), want.permute(0, 2, 1)) < 2e-5


@pytest.mark.parametrize("C", [256, 512, 1024])
def test_ln_rows(C):
    rng = np.random.RandomState(1)
    x = torch.from_numpy(rng.standard_normal((777, C)).astype(np.float32) * 3 + 1)
    w, b = _ln_params(rng, C)
    want = model_ref.channel_ln(x.t()[None], w, b)[0].t()
    for dt in (torch.float32, torch.bfloat16, torch.float16):
        out = torch.full((777, C), float("nan"), dtype=dt, device=DEV)
        ops.ln_rows(dev(x), dev(w), dev(b), out, 777)
        assert rel_err(out.float().cpu(), want) < (2e-6 if dt == torch.float32 else 5e-3)
        launch_ref.check(out, launch_ref.ln_rows(dev(x), dev(w), dev(b), out, 777)["out"], C, 5e-5, "ln_rows")


def test_instnorm_lrelu():
    """T / 16 rows per thread pick the register kernel (3, 6, 12, 24, 48 rows: T = 24 .. 768); T = 1000 runs the
    general kernel. 96 / 192 are exp12's contraction levels, 6 / 12 rows the exp5 expansion's. fp32 and the 16-bit
    outputs of mixed precision."""
    rng = np.random.RandomState(2)
    cases = ((3, 384, 256), (2, 24, 2048), (2, 768, 64), (2, 96, 512), (3, 192, 256), (2, 1000, 64), (2, 5, 32))
    for (B, T, C), out_dt in [(c, dt) for dt in (torch.float32, torch.float16, torch.bfloat16) for c in cases]:
        x = torch.from_numpy(rng.standard_normal((B, T, C)).astype(np.float32) * 2 + 0.3)
        want = F.leaky_relu(model_ref.instance_norm_t(x.permute(0, 2, 1)), 0.2).permute(0, 2, 1)
        out = torch.full((B, T, C), float("nan"), dtype=out_dt, device=DEV)
        ops.instnorm_lrelu(dev(x), out, batch=B, t=T, channels=C)
        if out_dt == torch.float32:
            assert rel_err(out.cpu(), want) < 5e-6
        ref = launch_ref.instnorm_lrelu(dev(x), out, batch=B, t=T, channels=C)["out"]
        launch_ref.check(out, ref, C, 5e-5, "instnorm T=%d" % T)


FPN_LENS = [[96, 48, 24, 12, 6, 3], [768, 384, 192, 96, 48, 24], [40, 20, 10, 5]]


@pytest.mark.parametrize("lens,out_dt", [pytest.param(l, torch.float32, id="lens%d" % i) for i, l in enumerate(FPN_LENS)] +
                         [pytest.param(l, torch.float16, id="lens%d-f16" % i) for i, l in enumerate(FPN_LENS)])
def test_fpn_fuse_and_head_final(lens, out_dt):
    """[96..3] / [768..24]: the column-blocked fpn kernel (level 0 divisible by 32); [40..5]: the row-per-warp kernel."""
    rng = np.random.RandomState(4)
    B, C = 2, 256
    P, L = sum(lens), len(lens)
    offs = np.cumsum([0] + lens)
    lat = torch.from_numpy(rng.standard_normal((B, P, C)).astype(np.float32))
    mask = rng.rand(B, P) > 0.15
    dw = torch.from_numpy(rng.normal(0, 0.6, (L, C, 3)).astype(np.float32))
    lw = torch.from_numpy(rng.uniform(0.5, 1.5, (L, C)).astype(np.float32)); lb = torch.from_numpy(rng.normal(0, 0.2, (L, C)).astype(np.float32))
    out = torch.full((B, P, C), float("nan"), dtype=out_dt, device=DEV)
    ops.fpn_fuse(dev(lat), dev(mask.astype(np.uint8)), dev(dw), dev(lw), dev(lb), out, batch=B, level_len=lens)
    ref = launch_ref.fpn_fuse(dev(lat), dev(mask.astype(np.uint8)), dev(dw), dev(lw), dev(lb), out, batch=B, level_len=lens)["out"]
    launch_ref.check(out, ref, C, 5e-5, "fpn_fuse")
    out = out.float()
    lats = [lat[:, offs[l]:offs[l + 1]].permute(0, 2, 1).clone() for l in range(L)]
    for l in range(L - 1, 0, -1):
        lats[l - 1] = lats[l - 1] + model_ref.nearest_resample(lats[l], lens[l - 1])
    fpn = []
    for l in range(L):
        m = torch.from_numpy(mask[:, offs[l]:offs[l + 1]])[:, None, :].float()
        z = F.conv1d(lats[l], dw[l].view(C, 1, 3), None, padding=1, groups=C) * m
        fpn.append(model_ref.channel_ln(z, lw[l], lb[l]))
        assert rel_err(out[:, offs[l]:offs[l + 1]].cpu(), fpn[l].permute(0, 2, 1)) < (2e-5 if out_dt == torch.float32 else 1e-3), l
    # head_final on top
    cw = torch.from_numpy((rng.standard_normal((1, C, 3)) / 10).astype(np.float32)); cb = torch.tensor([-1.0])
    rw = torch.from_numpy((rng.standard_normal((2, C, 3)) / 10).astype(np.float32)); rb = torch.tensor([0.3, -0.2])
    scales = [0.8, 0.9, 1.0, 1.1, 1.2, 1.3][:L]
    cf = torch.from_numpy(rng.standard_normal((B, P, C)).astype(np.float32)); rf = torch.from_numpy(rng.standard_normal((B, P, C)).astype(np.float32))
    logits = torch.full((B, P), float("nan"), device=DEV); offsets = torch.full((B, P, 2), float("nan"), device=DEV)
    ops.head_final(dev(cf), dev(rf), dev(mask.astype(np.uint8)), dev(cw.permute(0, 2, 1).reshape(1, -1)), dev(cb),
                   dev(rw.permute(0, 2, 1).reshape(2, -1)), dev(rb), scales, logits, offsets, batch=B, level_len=lens)
    for l in range(L):
        m = torch.from_numpy(mask[:, offs[l]:offs[l + 1]])[:, None, :].float()
        lg = F.conv1d(cf[:, offs[l]:offs[l + 1]].permute(0, 2, 1), cw, cb, padding=1) * m
        of = torch.relu(F.conv1d(rf[:, offs[l]:offs[l + 1]].permute(0, 2, 1), rw, rb, padding=1) * m * scales[l])
        assert rel_err(logits[:, offs[l]:offs[l + 1]].cpu(), lg[:, 0]) < 2e-5
        assert rel_err(offsets[:, offs[l]:offs[l + 1]].cpu(), of.permute(0, 2, 1)) < 2e-5


def test_vcls_tails():
    """exp12 / exp13 video-level tails, with the fp32 z and the 16-bit z the engine feeds them in mixed precision;
    exp13 with 64 and 32 channels."""
    for z_dt in (torch.float32, torch.float16, torch.bfloat16):
        _check_vcls_tails(z_dt)


def _check_vcls_tails(z_dt):
    rng = np.random.RandomState(6)
    B, T, C = 3, 24, 256
    z = torch.from_numpy(rng.standard_normal((B, T, C)).astype(np.float32)).to(z_dt)
    w0 = torch.from_numpy((rng.standard_normal((C, C)) / 16).astype(np.float32))
    w1 = torch.from_numpy((rng.standard_normal((C, 2 * C)) / 22).astype(np.float32))
    lw, lb = _ln_params(rng)
    w2 = torch.from_numpy((rng.standard_normal(C) / 16).astype(np.float32)); b2 = torch.tensor([0.1])
    g = F.leaky_relu(model_ref.instance_norm_t(torch.einsum("oc,btc->bot", w0, z.float())), 0.2)
    pooled = torch.cat([g.max(dim=2).values, g.mean(dim=2)], dim=1)
    h = torch.relu(model_ref.channel_ln((pooled @ w1.t()).unsqueeze(-1), lw, lb).squeeze(-1))
    want = h @ w2 + b2
    out = torch.full((B,), float("nan"), device=DEV)
    args = (dev(z), dev(w0.t().contiguous()), dev(w1.t().contiguous()), dev(lw), dev(lb), dev(w2), dev(b2), out)
    ops.vcls_exp12(*args, batch=B, t=T)
    assert rel_err(out.cpu(), want) < 2e-5
    launch_ref.check(out, launch_ref.vcls_exp12(*args, batch=B, t=T)["out"], 1, 5e-5, "vcls_exp12")
    for T, C in ((768, 64), (768, 32), (96, 32)):
        z = torch.from_numpy(rng.standard_normal((B, T, C)).astype(np.float32)).to(z_dt)
        w0 = torch.from_numpy((rng.standard_normal((C, C)) / 8).astype(np.float32))
        sw = torch.from_numpy((rng.standard_normal(C) / 8).astype(np.float32)); sb = torch.tensor([0.05])
        cw = torch.tensor([0.7, -0.4]); cb = torch.tensor([0.2])
        g = F.leaky_relu(model_ref.instance_norm_t(torch.einsum("oc,btc->bot", w0, z.float())), 0.2)
        s = torch.einsum("bct,c->bt", g, sw) + sb
        want = cw[0] * s.max(dim=1).values + cw[1] * s.mean(dim=1) + cb
        out = torch.full((B,), float("nan"), device=DEV)
        args = (dev(z), dev(w0), dev(sw), dev(sb), dev(cw), dev(cb), out)
        ops.vcls_exp13(*args, batch=B, t=T)
        assert rel_err(out.cpu(), want) < 2e-5, (T, C)
        launch_ref.check(out, launch_ref.vcls_exp13(*args, batch=B, t=T)["out"], 1, 5e-5, "vcls_exp13 T=%d C=%d" % (T, C))


@pytest.mark.parametrize("mode", ["fp32", "fp16"])
def test_conv_gemm_stacked_weight_blocks(mode):
    """q, k, v projections in one launch: three row segments per video, each with its own 256-row weight block."""
    rng = np.random.RandomState(8)
    B, T, C = 5, 48, 256
    adt = torch.float32 if mode == "fp32" else torch.float16
    a = torch.from_numpy(rng.standard_normal((B, 3 * T, C)).astype(np.float32))
    ws = [torch.from_numpy((rng.standard_normal((C, C)) / 16).astype(np.float32)) for _ in range(3)]
    bs = [torch.from_numpy(rng.normal(0, 0.3, C).astype(np.float32)) for _ in range(3)]
    out = torch.zeros((B, 3 * T, C), device=DEV)
    out_h = torch.zeros((B, 3 * T, C), dtype=torch.float16, device=DEV) if mode != "fp32" else None
    ops.conv_gemm(dev(a, adt), dev(torch.cat(ws), adt), taps=1, batch=B, c_in=C, n_out=C,
                  segs=[(T, i * T, i * T, i * C) for i in range(3)], a_rows=3 * T, o_rows=3 * T, bias=dev(torch.cat(bs)),
                  out_f32=out, out_h=out_h)
    aq = a.to(adt).float()
    for i in range(3):
        want = aq[:, i * T:(i + 1) * T] @ ws[i].to(adt).float().t() + bs[i]
        assert rel_err(out[:, i * T:(i + 1) * T].cpu(), want) < (2e-5 if mode == "fp32" else 2e-4), i
        if out_h is not None:
            assert rel_err(out_h[:, i * T:(i + 1) * T].float().cpu(), want) < 2e-3


WS_CASES = [
    # name, B, T, c_in, n_out, n_seg, bias, act, residual, out16_only
    ("qkv_stacked_16bit", 37, 96, 256, 256, 3, True, ops.ACT_NONE, False, True),       # <0,6,WS>: 3 groups, ragged last batch tile
    ("proj_res_fp32", 150, 128, 256, 256, 1, True, ops.ACT_NONE, True, False),         # <8,1,WS>: 150 tiles on <= 148 CTAs (2 tiles on some)
    ("lateral_fp32_small_t", 33, 24, 256, 256, 1, False, ops.ACT_NONE, False, False),  # <0,1,WS>: several videos per tile
    ("gelu_n1024_k128", 9, 64, 128, 1024, 1, True, ops.ACT_GELU, False, True),         # generic WS variant, 4 n-tile groups, 2 K blocks
]


@pytest.mark.parametrize("case", WS_CASES, ids=[c[0] for c in WS_CASES])
@pytest.mark.parametrize("adt", [torch.float16, torch.bfloat16], ids=["fp16", "bf16"])
def test_conv_gemm_weight_stationary(case, adt):
    """The weight-stationary configuration (W resident in shared memory, CTA pinned to a (segment, n-tile) group) forced
    on through the debug hook; the same launches in the streaming configuration must agree with it bit for bit."""
    name, B, T, cin, nout, n_seg, has_bias, act, has_res, out16_only = case
    rng = np.random.RandomState(zlib.crc32(name.encode()) % 1000)
    a = torch.from_numpy(rng.standard_normal((B, n_seg * T, cin)).astype(np.float32))
    ws = [torch.from_numpy((rng.standard_normal((nout, cin)) / math.sqrt(cin)).astype(np.float32)) for _ in range(n_seg)]
    bias = torch.from_numpy(rng.normal(0, 0.3, n_seg * nout).astype(np.float32)) if has_bias else None
    res = torch.from_numpy(rng.standard_normal((B, n_seg * T, nout)).astype(np.float32)) if has_res else None
    gamma = torch.from_numpy(rng.uniform(0.5, 1.5, nout).astype(np.float32)) if has_res else None
    valid = rng.randint(T // 2, T + 1, B); valid[0] = T
    mask = np.tile(np.arange(T)[None] < valid[:, None], (1, n_seg)).astype(np.uint8)
    L = nv.lib()
    outs = {}
    default_mode = L.avdf_debug_gemm_ws(0)
    try:
        for ws_mode in (1, 0):
            L.avdf_debug_gemm_ws(ws_mode)
            o32 = None if out16_only else torch.zeros((B, n_seg * T, nout), device=DEV)
            o16 = torch.zeros((B, n_seg * T, nout), dtype=adt, device=DEV) if out16_only else None
            ops.conv_gemm(dev(a, adt), dev(torch.cat(ws), adt), taps=1, batch=B, c_in=cin, n_out=nout,
                          segs=[(T, i * T, i * T, i * nout) for i in range(n_seg)], a_rows=n_seg * T, o_rows=n_seg * T,
                          bias=None if bias is None else dev(bias), row_mask=dev(mask) if not out16_only else None, act=act,
                          residual=None if res is None else dev(res), gamma=None if gamma is None else dev(gamma),
                          out_f32=o32, out_h=o16)
            torch.cuda.synchronize()
            outs[ws_mode] = (o16 if out16_only else o32).float().cpu()
    finally:
        L.avdf_debug_gemm_ws(default_mode)
    aq = a.to(adt).float()
    m = torch.from_numpy(mask).float()[..., None] if not out16_only else 1.0
    for i in range(n_seg):
        sl = slice(i * T, (i + 1) * T)
        y = aq[:, sl] @ ws[i].to(adt).float().t()
        if bias is not None:
            y = y + bias[i * nout:(i + 1) * nout]
        y = y * (m[:, sl] if not out16_only else 1.0)
        if act == ops.ACT_GELU:
            y = model_ref.gelu_erf(y)
        if res is not None:
            y = res[:, sl] * m[:, sl] + gamma * y
        assert rel_err(outs[1][:, sl], y) < (1e-2 if out16_only else 2e-4), (name, i)
    if act == ops.ACT_NONE:                 # (the GELU case runs the scalar formula in one configuration, the packed one in the other)
        assert torch.equal(outs[1], outs[0])


@pytest.mark.parametrize("case", ["ln_relu_16bit", "ln_relu_pe_fp32", "k1024_res_both"])
def test_conv_gemm_wide_tiles_eight_epilogue_warps(case):
    """256-wide tiles run with eight epilogue warps (two per row block, splitting the columns; LayerNorm statistics exchanged
    through shared memory). More tiles than SMs, ragged masks; checked against torch and against the four-warp configuration."""
    rng = np.random.RandomState({"ln_relu_16bit": 1, "ln_relu_pe_fp32": 2, "k1024_res_both": 3}[case])
    adt = torch.float16
    if case == "k1024_res_both":
        B, T, cin, nout, taps, has_ln, act, has_pe, has_res = 160, 128, 1024, 256, 1, False, ops.ACT_NONE, False, True
    else:
        B, T, cin, nout, taps, has_ln, act, has_pe, has_res = 170, 128, 256, 256, 3, True, ops.ACT_RELU, case == "ln_relu_pe_fp32", False
    x = torch.from_numpy(rng.standard_normal((B, T, cin)).astype(np.float32))
    w = torch.from_numpy((rng.standard_normal((nout, cin, taps)) / math.sqrt(cin * taps)).astype(np.float32))
    bias = torch.from_numpy(rng.normal(0, 0.3, nout).astype(np.float32)) if not has_ln else None
    ln = _ln_params(rng, nout) if has_ln else None
    pe = torch.from_numpy(rng.normal(0, 0.1, (T, nout)).astype(np.float32)) if has_pe else None
    res = torch.from_numpy(rng.standard_normal((B, T, nout)).astype(np.float32)) if has_res else None
    gamma = torch.from_numpy(rng.uniform(0.5, 1.5, nout).astype(np.float32)) if has_res else None
    valid = rng.randint(T // 2, T + 1, B); valid[0] = T
    mask = (np.arange(T)[None] < valid[:, None])
    want = _conv_ref(x.to(adt).float(), w.to(adt).float(), bias, taps, 1, torch.from_numpy(mask), ln, act, pe, res, gamma)
    wp = w.permute(0, 2, 1).reshape(nout, taps * cin).contiguous()
    L = nv.lib()
    outs = {}
    prev = L.avdf_debug_gemm_w8(1)
    try:
        for on in (1, 0):
            L.avdf_debug_gemm_w8(on)
            o32 = torch.zeros((B, T, nout), device=DEV) if case != "ln_relu_16bit" else None
            o16 = torch.zeros((B, T, nout), dtype=adt, device=DEV) if case != "ln_relu_pe_fp32" else None
            ops.conv_gemm(dev(x, adt), dev(wp, adt), taps=taps, stride=1, batch=B, c_in=cin, n_out=nout, segs=[(T, 0, 0)], a_rows=T, o_rows=T,
                          bias=None if bias is None else dev(bias), row_mask=dev(mask.astype(np.uint8)),
                          ln=None if ln is None else (dev(ln[0]), dev(ln[1])), act=act, pe=None if pe is None else dev(pe),
                          residual=None if res is None else dev(res), gamma=None if gamma is None else dev(gamma), out_f32=o32, out_h=o16)
            torch.cuda.synchronize()
            outs[on] = (None if o32 is None else o32.cpu(), None if o16 is None else o16.float().cpu())
    finally:
        L.avdf_debug_gemm_w8(prev)
    for on in (1, 0):
        if outs[on][0] is not None:
            assert rel_err(outs[on][0], want) < 2e-4, (case, on)
        if outs[on][1] is not None:
            assert rel_err(outs[on][1], want) < 1e-2, (case, on)
    if outs[1][0] is not None:                  # the two configurations differ only in the summation order of the LayerNorm statistics
        assert rel_err(outs[1][0], outs[0][0]) < 2e-6


@pytest.mark.parametrize("adt", [torch.float16, torch.bfloat16], ids=["fp16", "bf16"])
@pytest.mark.parametrize("B,T", [(3, 96), (170, 128), (5, 24)])
def test_conv_gemm_ln_after_residual(B, T, adt):
    """Attention projection + LN2 in one launch (ln_after_residual): out_f32 = the residual stream, bit-equal to the
    plain residual launch; out_h = LayerNorm of it (blocks.py:1309-1311), against torch and against avdf_ln_rows."""
    rng = np.random.RandomState(B * 7 + T)
    C = 256
    x = torch.from_numpy(rng.standard_normal((B, T, C)).astype(np.float32))
    w = torch.from_numpy((rng.standard_normal((C, C, 1)) / math.sqrt(C)).astype(np.float32))
    bias = torch.from_numpy(rng.normal(0, 0.3, C).astype(np.float32))
    ln = _ln_params(rng, C)
    res = torch.from_numpy(rng.standard_normal((B, T, C)).astype(np.float32) * 2 + 0.5)
    gamma = torch.from_numpy(rng.uniform(0.5, 1.5, C).astype(np.float32))
    valid = rng.randint(T // 2, T + 1, B); valid[0] = T
    mask = (np.arange(T)[None] < valid[:, None])
    y_want = _conv_ref(x.to(adt).float(), w.to(adt).float(), bias, 1, 1, torch.from_numpy(mask), None, ops.ACT_NONE, None, res, gamma)
    l_want = model_ref.channel_ln(y_want.permute(0, 2, 1), ln[0], ln[1]).permute(0, 2, 1)
    wp = w.reshape(C, C).contiguous()
    kw = dict(taps=1, stride=1, batch=B, c_in=C, n_out=C, segs=[(T, 0, 0)], a_rows=T, o_rows=T, bias=dev(bias),
              row_mask=dev(mask.astype(np.uint8)), residual=dev(res), gamma=dev(gamma))
    y_plain = torch.zeros((B, T, C), device=DEV)
    ops.conv_gemm(dev(x, adt), dev(wp, adt), out_f32=y_plain, **kw)
    y = torch.zeros((B, T, C), device=DEV)
    l2 = torch.zeros((B, T, C), dtype=adt, device=DEV)
    ops.conv_gemm(dev(x, adt), dev(wp, adt), out_f32=y, out_h=l2, ln=(dev(ln[0]), dev(ln[1])), ln_after_residual=True, **kw)
    l_rows = torch.zeros((B * T, C), dtype=adt, device=DEV)
    ops.ln_rows(y.view(B * T, C), dev(ln[0]), dev(ln[1]), l_rows, B * T)
    torch.cuda.synchronize()
    assert torch.equal(y, y_plain)
    assert rel_err(y.cpu(), y_want) < 2e-4
    assert rel_err(l2.float().cpu(), l_want) < (5e-3 if adt == torch.float16 else 1e-2)
    # against the separate LayerNorm kernel: only the summation order of the statistics and the last 16-bit ulp differ
    d = (l2.float() - l_rows.view(B, T, C).float()).abs().max().item()
    assert d <= (4e-3 if adt == torch.float16 else 4e-2), d


@pytest.mark.parametrize("mode", ["fp32", "fp16", "bf16"])
def test_conv_gemm_forward_taps_is_conv_transpose(mode):
    """tap_mode 1 (taps at offsets 0, +1): with the weight blocks of `engine.up_weight` one launch computes
    ConvTranspose1d(k=3, stride=2, padding=1, output_padding=1) (blocks.py:1443-1491): output row t of width 2*c_out
    holds the transposed conv's outputs 2t and 2t+1."""
    rng = np.random.RandomState(5)
    B, T, cin, cout = 3, 48, 128, 64
    x = torch.from_numpy(rng.standard_normal((B, T, cin)).astype(np.float32))
    wt = torch.from_numpy((rng.standard_normal((cin, cout, 3)) / math.sqrt(cin * 2)).astype(np.float32))   # ConvTranspose1d layout
    bias = torch.from_numpy(rng.normal(0, 0.3, cout).astype(np.float32))
    adt = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}[mode]
    want = F.conv_transpose1d(x.to(adt).float().permute(0, 2, 1), wt.to(adt).float(), bias, stride=2, padding=1, output_padding=1).permute(0, 2, 1)
    from audio_visual_deepfake_detection_b200.libs.modeling.engine import up_weight
    wg = up_weight(wt)                                                    # [2*cout, 2*cin]
    out = torch.zeros((B, T, 2 * cout), device=DEV)
    ops.conv_gemm(dev(x, adt), dev(wg, adt), taps=2, stride=1, batch=B, c_in=cin, n_out=2 * cout, segs=[(T, 0, 0)], a_rows=T, o_rows=T,
                  bias=dev(torch.cat([bias, bias])), out_f32=out, tap_mode=1)
    torch.cuda.synchronize()
    assert rel_err(out.view(B, 2 * T, cout).cpu(), want) < (2e-5 if mode == "fp32" else 2e-4)


def test_conv_gemm_row_dots_and_head_combine():
    """The last tower layer emits per-tap partial sums of the heads' final convolution instead of its 256-channel output
    (conv_gemm dots=...), avdf_head_combine adds the neighbouring rows' taps: against avdf_head_final on the stored tower
    outputs and against torch. Pyramid segments, ragged masks."""
    rng = np.random.RandomState(21)
    lens = [96, 48, 24, 12, 6, 3]
    B, C, P = 37, 256, sum(lens)
    offs = [sum(lens[:l]) for l in range(len(lens))]
    adt = torch.float16
    x = torch.from_numpy(rng.standard_normal((B, P, C)).astype(np.float32))
    valid = rng.randint(40, 97, B); valid[0] = 96
    mask = np.concatenate([(np.arange(n)[None] * (2 ** l)) < valid[:, None] for l, n in enumerate(lens)], axis=1).astype(np.uint8)
    towers, dots = {}, {}
    segs = [(lens[l], offs[l], offs[l]) for l in range(len(lens))]
    heads = {}
    for head, n_out in (("cls", 1), ("reg", 2)):
        w = torch.from_numpy((rng.standard_normal((C, C, 3)) / math.sqrt(3 * C)).astype(np.float32))
        ln = _ln_params(rng, C)
        hw = torch.from_numpy((rng.standard_normal((n_out, C, 3)) / math.sqrt(3 * C)).astype(np.float32))
        hb = torch.from_numpy(rng.normal(0, 0.3, n_out).astype(np.float32))
        wp = w.permute(0, 2, 1).reshape(C, 3 * C).contiguous()
        hwp = hw.permute(0, 2, 1).reshape(n_out, 3 * C).contiguous()              # [o, tap * C]
        kw = dict(taps=3, stride=1, batch=B, c_in=C, n_out=C, segs=segs, a_rows=P, o_rows=P, row_mask=dev(mask),
                  ln=(dev(ln[0]), dev(ln[1])), act=ops.ACT_RELU)
        t32 = torch.zeros((B, P, C), device=DEV)
        ops.conv_gemm(dev(x, adt), dev(wp, adt), out_f32=t32, **kw)
        d = torch.full((B, P, 3 * n_out), float("nan"), device=DEV)
        ops.conv_gemm(dev(x, adt), dev(wp, adt), dots=(dev(hwp).view(3 * n_out, C), d), **kw)
        towers[head], dots[head], heads[head] = t32, d, (dev(hwp), dev(hb))
        # the dot products themselves, against the stored tower output
        want = torch.einsum("bpc,jc->bpj", t32.cpu(), hwp.view(3 * n_out, C))
        assert rel_err(d.cpu(), want) < 1e-5
    scales = [float(v) for v in rng.uniform(0.8, 1.6, len(lens))]
    lg_a, of_a = torch.zeros((B, P), device=DEV), torch.zeros((B, P, 2), device=DEV)
    lg_b, of_b = torch.zeros((B, P), device=DEV), torch.zeros((B, P, 2), device=DEV)
    ops.head_final(towers["cls"], towers["reg"], dev(mask), heads["cls"][0], heads["cls"][1], heads["reg"][0], heads["reg"][1], scales,
                   lg_a, of_a, batch=B, level_len=lens)
    ops.head_combine(dots["cls"], dots["reg"], dev(mask), heads["cls"][1], heads["reg"][1], scales, lg_b, of_b, batch=B, level_len=lens)
    torch.cuda.synchronize()
    assert rel_err(lg_b.cpu(), lg_a.cpu()) < 1e-5 and rel_err(of_b.cpu(), of_a.cpu()) < 1e-5


def test_attention_stacked_qkv_and_interleaved_dwconv():
    rng = np.random.RandomState(10)
    B, T, C = 3, 80, 256
    qkv = torch.from_numpy(rng.standard_normal((B, 3 * T, C)).astype(np.float32)).to(torch.float16)
    mask = torch.from_numpy(np.arange(T)[None] < np.array([T, 50, T - 1])[:, None])
    out_a = torch.zeros((B, T, C), device=DEV); out_b = torch.zeros((B, T, C), device=DEV)
    ops.attention(None, None, None, dev(mask.to(torch.uint8)), out_a, batch=B, t=T, n_head=4, window=7, qkv=dev(qkv))
    q, k, v = (dev(qkv[:, i * T:(i + 1) * T].contiguous()) for i in range(3))
    ops.attention(q, k, v, dev(mask.to(torch.uint8)), out_b, batch=B, t=T, n_head=4, window=7)
    assert torch.equal(out_a, out_b)
    # ln_dwconv_ln writing three streams interleaved into one [B, 3T, C] buffer == three dense outputs
    x = torch.from_numpy(rng.standard_normal((B, T, C)).astype(np.float32))
    lni = [_ln_params(rng) for _ in range(3)]; lno = [_ln_params(rng) for _ in range(3)]
    dws = [torch.from_numpy(rng.normal(0, 0.6, (C, 3)).astype(np.float32)) for _ in range(3)]
    kw = dict(batch=B, t_src=T, t_virt=T, shift=0, stride=1, mask_out=dev(mask.to(torch.uint8)),
              ln_in=[(dev(a), dev(b)) for a, b in lni], dw=[dev(d) for d in dws], ln_out=[(dev(a), dev(b)) for a, b in lno])
    dense = [torch.zeros((B, T, C), device=DEV) for _ in range(3)]
    ops.ln_dwconv_ln(dev(x), outs=dense, **kw)
    inter = torch.zeros((B, 3 * T, C), device=DEV)
    ops.ln_dwconv_ln(dev(x), outs=[inter] * 3, out_rows=3 * T, out_row_offsets=[0, T, 2 * T], **kw)
    for i in range(3):
        assert torch.equal(inter[:, i * T:(i + 1) * T], dense[i])


# --------------------------------------------------------------------------------------------- fused MLP
@pytest.mark.parametrize("rows", [128, 100, 1000, 32 * 768])
@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
def test_mlp_fused(rows, dt):
    """avdf_mlp_fused == Linear(256,1024) -> exact GELU -> Linear(1024,256) -> mask, gamma, residual (blocks.py:1236-1243,
    1315-1316) computed in fp32 by torch from the same 16-bit operands; the hidden activations are rounded to the
    16-bit type once, like the kernel's on-chip tile (and the unfused path's intermediate tensor)."""
    rng = np.random.RandomState(rows + (1 if dt == torch.float16 else 2))
    C, H = 256, 1024
    x = torch.from_numpy(rng.standard_normal((rows, C)).astype(np.float32)).to(dt)
    w1 = torch.from_numpy((rng.standard_normal((H, C)) / 16).astype(np.float32)).to(dt)
    w2 = torch.from_numpy((rng.standard_normal((C, H)) / 32).astype(np.float32)).to(dt)
    b1 = torch.from_numpy(rng.normal(0, 0.3, H).astype(np.float32))
    b2 = torch.from_numpy(rng.normal(0, 0.3, C).astype(np.float32))
    gamma = torch.from_numpy(rng.uniform(0.5, 1.5, C).astype(np.float32))
    res = torch.from_numpy(rng.standard_normal((rows, C)).astype(np.float32))
    mask = torch.from_numpy((rng.rand(rows) > 0.15).astype(np.uint8))
    out = torch.full((rows, C), float("nan"), device=DEV)
    ops.mlp_fused(dev(x), dev(w1), dev(b1), dev(w2), dev(b2), row_mask=dev(mask), residual=dev(res), gamma=dev(gamma), out=out)
    h = F.gelu(x.float() @ w1.float().t() + b1).to(dt).float()
    m = mask.float()[:, None]
    want = res * m + gamma * ((h @ w2.float().t() + b2) * m)
    assert rel_err(out.cpu(), want) < (2e-4 if dt == torch.float16 else 1e-3)   # bf16: hidden activations at rounding ties
    # the same through the two-launch path
    hid = torch.empty((1, rows, H), device=DEV, dtype=dt)
    ops.conv_gemm(dev(x).view(1, rows, C), dev(w1), taps=1, batch=1, c_in=C, n_out=H, segs=[(rows, 0, 0)], a_rows=rows, o_rows=rows,
                  bias=dev(b1), act=ops.ACT_GELU, out_h=hid)
    out2 = torch.empty((1, rows, C), device=DEV)
    ops.conv_gemm(hid, dev(w2), taps=1, batch=1, c_in=H, n_out=C, segs=[(rows, 0, 0)], a_rows=rows, o_rows=rows, bias=dev(b2),
                  row_mask=dev(mask).view(1, rows), residual=dev(res).view(1, rows, C), gamma=dev(gamma), out_f32=out2)
    assert rel_err(out.cpu(), out2.view(rows, C).cpu()) < 2e-4


@pytest.mark.parametrize("rows", [128, 300, 32 * 96, 32 * 768])
@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
def test_block_tail_projection_ln2_mlp_in_one_launch(rows, dt):
    """avdf_mlp_fused with att != NULL (attention projection + LN2 + MLP of a block in one launch) against the two launches
    it replaces: conv_gemm(ln_after_residual) + mlp_fused. y is bit-equal; out differs only through last-bit differences of
    the 16-bit LN2 operand (the statistics are summed in another order)."""
    rng = np.random.RandomState(rows + (1 if dt == torch.float16 else 2))
    C, H = 256, 1024
    att = dev(torch.from_numpy(rng.standard_normal((rows, C)).astype(np.float32)), dt)
    wo = dev(torch.from_numpy((rng.standard_normal((C, C)) / math.sqrt(C)).astype(np.float32)), dt)
    bo = dev(torch.from_numpy(rng.normal(0, 0.3, C).astype(np.float32)))
    ga = dev(torch.from_numpy(rng.uniform(0.5, 1.5, C).astype(np.float32)))
    ln2 = tuple(dev(t) for t in _ln_params(rng, C))
    skip = dev(torch.from_numpy((rng.standard_normal((rows, C)) * 2 + 0.5).astype(np.float32)))
    w1 = dev(torch.from_numpy((rng.standard_normal((H, C)) / 16).astype(np.float32)), dt)
    w2 = dev(torch.from_numpy((rng.standard_normal((C, H)) / 32).astype(np.float32)), dt)
    b1 = dev(torch.from_numpy(rng.standard_normal(H).astype(np.float32)))
    b2 = dev(torch.from_numpy(rng.standard_normal(C).astype(np.float32)))
    gm = dev(torch.from_numpy(rng.uniform(0.5, 1.5, C).astype(np.float32)))
    mask_np = (rng.uniform(size=rows) > 0.15).astype(np.uint8); mask_np[:3] = 1
    mask = dev(torch.from_numpy(mask_np))
    # reference: two launches
    y_ref = torch.zeros((rows, C), device=DEV); l2 = torch.zeros((rows, C), dtype=dt, device=DEV); out_ref = torch.zeros((rows, C), device=DEV)
    ops.conv_gemm(att.view(1, rows, C), wo, taps=1, batch=1, c_in=C, n_out=C, segs=[(rows, 0, 0)], a_rows=rows, o_rows=rows, bias=bo,
                  row_mask=mask.view(1, rows), residual=skip.view(1, rows, C), gamma=ga, out_f32=y_ref.view(1, rows, C), out_h=l2.view(1, rows, C),
                  ln=ln2, ln_after_residual=True)
    ops.mlp_fused(l2, w1, b1, w2, b2, row_mask=mask, residual=y_ref, gamma=gm, out=out_ref)
    # one launch: y stays in the accumulator, so the MLP's scale is folded into W2 / b2 by the caller (fp32, before the rounding)
    w2f = dev((w2.float().cpu() * gm.cpu()[:, None]), dt)
    b2f = (b2 * gm).contiguous()
    y = torch.zeros((rows, C), device=DEV); out = torch.zeros((rows, C), device=DEV); out_noy = torch.zeros((rows, C), device=DEV)
    ops.mlp_fused(None, w1, b1, w2f, b2f, row_mask=mask, residual=None, gamma=None, out=out, proj=(att, wo, bo, ga, ln2, skip, y))
    ops.mlp_fused(None, w1, b1, w2f, b2f, row_mask=mask, residual=None, gamma=None, out=out_noy, proj=(att, wo, bo, ga, ln2, skip, None))
    torch.cuda.synchronize()
    assert torch.equal(y, y_ref)                 # the optional copy of the residual stream
    assert torch.equal(out, out_noy)             # storing it or not changes nothing
    assert rel_err(out.cpu(), out_ref.cpu()) < (2e-3 if dt == torch.float16 else 1.5e-2)
    with pytest.raises(AssertionError):          # an unfolded scale is refused
        ops.mlp_fused(None, w1, b1, w2, b2, row_mask=mask, residual=None, gamma=gm, out=out, proj=(att, wo, bo, ga, ln2, skip, None))
    # and against plain torch on the same 16-bit operands
    mk_t = torch.from_numpy(mask_np.astype(np.float32))[:, None]
    yt = skip.cpu() * mk_t + ga.cpu() * ((att.float().cpu() @ wo.float().cpu().t() + bo.cpu()) * mk_t)
    assert rel_err(y.cpu(), yt) < 2e-4


def test_mlp_fused_16bit_copy_into_pyramid_level():
    """out_h: the 16-bit copy of the fused MLP's result, dense or scattered into one level of a [batch, P, C] pyramid
    buffer (the operand of the single FPN lateral launch)."""
    rng = np.random.RandomState(77)
    C, H, B, T, P, row0 = 256, 1024, 3, 96, 200, 40
    rows = B * T
    dt = torch.float16
    x = torch.from_numpy(rng.standard_normal((rows, C)).astype(np.float32)).to(dt)
    w1 = torch.from_numpy((rng.standard_normal((H, C)) / 16).astype(np.float32)).to(dt)
    w2 = torch.from_numpy((rng.standard_normal((C, H)) / 32).astype(np.float32)).to(dt)
    b1 = torch.from_numpy(rng.normal(0, 0.3, H).astype(np.float32)); b2 = torch.from_numpy(rng.normal(0, 0.3, C).astype(np.float32))
    res = torch.from_numpy(rng.standard_normal((rows, C)).astype(np.float32))
    out = torch.empty((rows, C), device=DEV)
    dense = torch.zeros((rows, C), device=DEV, dtype=dt)
    ops.mlp_fused(dev(x), dev(w1), dev(b1), dev(w2), dev(b2), row_mask=None, residual=dev(res), gamma=None, out=out, out_h=dense)
    assert torch.equal(dense, out.to(dt))
    pyr = torch.full((B, P, C), 7.0, device=DEV, dtype=dt)
    out2 = torch.empty((rows, C), device=DEV)
    ops.mlp_fused(dev(x), dev(w1), dev(b1), dev(w2), dev(b2), row_mask=None, residual=dev(res), gamma=None, out=out2, out_h=pyr,
                  out_h_level=(T, P, row0))
    assert torch.equal(out2, out)
    assert torch.equal(pyr[:, row0:row0 + T].reshape(rows, C), dense)
    assert bool((pyr[:, :row0] == 7.0).all()) and bool((pyr[:, row0 + T:] == 7.0).all())


@pytest.mark.parametrize("case", ["towers_k768_ln", "embed_k2304_s1", "down_k1536_s2_n1024", "narrow_k512_n128", "dots_k768", "odd_tiles_fallback"])
def test_conv_gemm_weight_multicast(case):
    """CTA pairs on adjacent row tiles of one n-tile, two ways: `pair` = cta_group::2 MMAs (M = 256 over the two SMs, each CTA
    holds half of every weight tile; the default for K >= 512 in the wide configuration) and `mc` = independent MMAs with the
    weight tile fetched by TMA multicast (off by default): both bit-identical to the plain launch, and against torch. Many tiles per
    CTA (several trips around the stage ring), ragged masks, wide / narrow / strided / several n-tiles / row-dot epilogues."""
    rng = np.random.RandomState(zlib.crc32(case.encode()) & 0xffff)
    cfg = {"towers_k768_ln": dict(B=160, T=128, cin=256, taps=3, stride=1, nout=256, ln=True, act=ops.ACT_RELU),
           "embed_k2304_s1": dict(B=40, T=128, cin=768, taps=3, stride=1, nout=256, ln=True, act=ops.ACT_RELU),
           "down_k1536_s2_n1024": dict(B=12, T=128, cin=512, taps=3, stride=2, nout=1024, ln=False, act=ops.ACT_NONE),
           "narrow_k512_n128": dict(B=340, T=128, cin=512, taps=1, stride=1, nout=128, ln=False, act=ops.ACT_GELU),
           "dots_k768": dict(B=10, T=128, cin=256, taps=3, stride=1, nout=256, ln=True, act=ops.ACT_RELU, dots=True),
           "odd_tiles_fallback": dict(B=7, T=128, cin=256, taps=3, stride=1, nout=256, ln=True, act=ops.ACT_RELU)}[case]
    B, T, cin, taps, stride, nout = (cfg[k] for k in ("B", "T", "cin", "taps", "stride", "nout"))
    adt = torch.float16
    t_in = T * stride
    x = torch.from_numpy(rng.standard_normal((B, t_in, cin)).astype(np.float32))
    w = torch.from_numpy((rng.standard_normal((nout, cin, taps)) / math.sqrt(cin * taps)).astype(np.float32))
    bias = torch.from_numpy(rng.normal(0, 0.3, nout).astype(np.float32))
    ln = _ln_params(rng, nout) if cfg["ln"] else None
    valid = rng.randint(T // 2, T + 1, B); valid[0] = T
    mask = (np.arange(T)[None] < valid[:, None]).astype(np.uint8)
    wp = w.permute(0, 2, 1).reshape(nout, taps * cin).contiguous()
    dw = torch.from_numpy(rng.standard_normal((6, nout)).astype(np.float32) / 16) if cfg.get("dots") else None
    L = nv.lib()
    outs = {}
    prev = (L.avdf_debug_gemm_mc(0), L.avdf_debug_gemm_pair(0))
    try:
        for key, (mc, pair) in {"pair": (0, 512), 512: (512, 0), 0: (0, 0)}.items():
            L.avdf_debug_gemm_mc(mc); L.avdf_debug_gemm_pair(pair)
            o32 = torch.full((B, T, nout), float("nan"), device=DEV)
            o16 = torch.zeros((B, T, nout), dtype=adt, device=DEV)
            d = torch.full((B, T, 6), float("nan"), device=DEV) if dw is not None else None
            kw = dict(out_f32=o32, out_h=o16) if dw is None else dict(dots=(dev(dw), d))
            ops.conv_gemm(dev(x, adt), dev(wp, adt), taps=taps, stride=stride, batch=B, c_in=cin, n_out=nout, segs=[(T, 0, 0)], a_rows=t_in,
                          o_rows=T, bias=dev(bias), row_mask=dev(mask), ln=None if ln is None else (dev(ln[0]), dev(ln[1])), act=cfg["act"], **kw)
            torch.cuda.synchronize()
            outs[key] = (o32.cpu(), o16.float().cpu(), None if d is None else d.cpu())
    finally:
        L.avdf_debug_gemm_mc(prev[0]); L.avdf_debug_gemm_pair(prev[1])
    xq, wq = x.to(adt).float(), w.to(adt).float()
    y = F.conv1d(xq.transpose(1, 2), wq, bias, stride=stride, padding=taps // 2).transpose(1, 2) * torch.from_numpy(mask).float()[..., None]
    if ln is not None:
        y = F.layer_norm(y, (nout,), ln[0], ln[1], 1e-5)
    y = F.relu(y) if cfg["act"] == ops.ACT_RELU else (model_ref.gelu_erf(y) if cfg["act"] == ops.ACT_GELU else y)
    if dw is None:
        assert rel_err(outs[512][0], y) < 2e-4 and rel_err(outs[512][1], y) < 2e-3
        for key in (512, "pair"):
            assert torch.equal(outs[key][0], outs[0][0]) and torch.equal(outs[key][1], outs[0][1]), key
    else:
        assert rel_err(outs[512][2], torch.einsum("btn,jn->btj", y, dw)) < 2e-4
        assert torch.equal(outs[512][2], outs[0][2]) and torch.equal(outs["pair"][2], outs[0][2])
