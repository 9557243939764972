"""Every kernel launch of the BYOL-A extractor (libs/features/byola.py: `AudioNTT2020Task6.extract` and `forward`),
checked one by one against the float64 references of oracle/launch_ref.py with the overlap, replay, error and zeros
checks of tests/launch_check.py: avdf_logmel within its per-element fp32 FFT bound, avdf_byola_conv1_pool at 5e-5 row-wise
(+ one ulp for 16-bit outputs) with its row mask exact, avdf_byola_pool bit-exact (grid and fc rows), and the four
avdf_conv_gemm launches (the two 3x3 convolutions as nine-tap GEMMs, K = 576, and the fc layers, K = 512 and 2048) at
5e-5 row-wise + one ulp on the 16-bit operands the kernel saw. Weights: synthetic_byola_state_dict(0). Passes:
  bench    the benchmark's first batch (32 AV-Deepfake1M-length clips), fp32 / mixed / bf16
  edges    the shortest clips (1120 and 1279 samples: 8 frames, one output row), 9..24 frames (every residue mod 16, odd
           counts at every pooling level, varied sample residues mod 160), digital silence then a full-scale onset, and
           a 600 s recording (60,001 frames), fp32 / mixed / bf16
  no-pad   grids without a padding step at their end, and a batch with exactly 128 fc rows, mixed
  many     512 clips of 1-3 s (the clip search of the log-mel kernel over many clips), mixed
  module   `model(lms)` with a (2, 1, 64, 96) tensor and with a list of clips of different lengths, mixed / fp32"""
import collections
import time

import numpy as np
import pytest
import torch

import byola_ref
import launch_check
from audio_visual_deepfake_detection_b200.libs.features import AudioNTT2020Task6, BatchPlan
from audio_visual_deepfake_detection_b200.libs.utils import synthetic as syn

pytestmark = pytest.mark.gpu

OPS = ("logmel", "byola_conv1_pool", "byola_pool", "conv_gemm")
PER_BATCH = {"logmel": 1, "byola_conv1_pool": 1, "byola_pool": 2, "conv_gemm": 4}
GEMM_K = [576, 576, 512, 2048]            # conv 2, conv 3 (9 taps x 64 channels), fc 1, fc 2
STATS = collections.defaultdict(lambda: [0, 0.0])          # op -> [launches, worst error / bar] over the whole module
_CACHE = {}


@pytest.fixture
def recorder(monkeypatch):
    """Wraps the extractor's `ops` entry points; each call is checked as soon as it returns."""
    return launch_check.install(monkeypatch, OPS, launch_check.BYOLA_FILE)


def _wav(n, seed):
    if (n, seed) not in _CACHE:
        _CACHE[(n, seed)] = syn.synthetic_wav(n, seed)
    return _CACHE[(n, seed)]


def _plan(wavs):
    return BatchPlan([w.shape[0] for w in wavs], "cpu")


def _bench():
    durs = syn.sample_durations(256, seed=4321)[:32]                    # bench.py byola_extractor_bench, batch 0
    wavs = [_wav(int(16000 * d), 9000 + i) for i, d in enumerate(durs)]
    p = _plan(wavs)
    assert p.steps1 == 15552 and p.rows3 == 3968
    return [("wav", wavs)]


def _edges():
    shortest = [_wav(1120, 40)]
    mixed = [_wav(1279, 41)]
    mixed += [_wav(160 * (f - 1) + (37 * f) % 160, 40 + f) for f in range(9, 25)]       # f frames, residue mod 160 varied
    onset = np.zeros(16000 * 3, np.float32)
    onset[16000 * 2:] = np.clip(3.0 * _wav(16000, 60), -1.0, 1.0)                        # digital silence, full-scale onset
    mixed.append(onset)
    mixed.append(_wav(600 * 16000, 61))
    frames = [1 + w.shape[0] // 160 for w in shortest + mixed]
    assert frames[:2] == [8, 8] and frames[2:18] == list(range(9, 25)) and frames[-1] == 60001
    assert float(np.abs(onset).max()) == 1.0 and not onset[:16000 * 2].any()
    return [("wav", shortest), ("wav", mixed)]


def _no_pad():
    """One clip of 19,680 samples: 124 frames, 62 level-1 steps, a grid of exactly 1 + 62 + 1 = 64 steps. And 63 clips of
    8q + r frames (r in {0, 1}, sum q = 128): t1 = 4q, t2 = 2q, t3 = q, so the level-1 grid has 1 + 512 + 63 = 576 = 9 x 64
    steps, the level-2 grid 1 + 256 + 63 = 320 = 5 x 64, and the fc layers exactly 128 rows: no padding anywhere."""
    one = [_wav(19680, 70)]
    p = _plan(one)
    assert p.steps1 == 1 + p.t[1][0] + 1 == 64
    rng = np.random.RandomState(71)
    q = np.ones(63, np.int64)
    np.add.at(q, rng.randint(0, 63, 128 - 63), 1)
    frames = 8 * q + rng.randint(0, 2, 63)
    many = [_wav(int(160 * (f - 1) + rng.randint(0, 160)), 100 + i) for i, f in enumerate(frames)]
    p = _plan(many)
    assert p.steps1 == 1 + sum(t + 1 for t in p.t[1]) and p.steps2 == 1 + sum(t + 1 for t in p.t[2])
    assert sum(p.t[3]) == p.rows3 == 128
    return [("wav", one), ("wav", many)]


def _many():
    rng = np.random.RandomState(80)
    return [("wav", [_wav(int(16000 * d), 2000 + i) for i, d in enumerate(rng.uniform(1.0, 3.0, 512))])]


def _module():
    lms = [torch.from_numpy(byola_ref.log_mel(_wav(16000 * 2 + 77 * i, 90 + i))) for i in range(3)]      # [64, 201 + ...]
    return [("lms", torch.stack([lms[0][:, :96], lms[1][:, 100:196]])[:, None]),                       # (2, 1, 64, 96)
            ("lms", [lms[0][:, :96], lms[1][None, :, :131], lms[2][:, 3:11]])]                          # 96, 131, 8 frames


BATCHES = {"bench": _bench, "edges": _edges, "no-pad": _no_pad, "many": _many, "module": _module}
PASSES = [("bench", p) for p in ("fp32", "mixed", "bf16")] + [("edges", p) for p in ("fp32", "mixed", "bf16")]
PASSES += [("no-pad", "mixed"), ("many", "mixed"), ("module", "mixed"), ("module", "fp32")]


@pytest.mark.parametrize("case,precision", PASSES, ids=["%s-%s" % cp for cp in PASSES])
def test_every_extractor_launch(case, precision, recorder):
    m = AudioNTT2020Task6(n_mels=64, d=2048, precision=precision)
    m.load_state_dict(syn.synthetic_byola_state_dict(0))
    m = m.to("cuda").eval()
    batches = BATCHES[case]()
    t0 = time.time()
    for kind, batch in batches:
        before, n0 = collections.Counter(recorder.count), len(recorder.launches)
        outs = m.extract(batch) if kind == "wav" else m(batch)
        torch.cuda.synchronize()
        want = dict(PER_BATCH)
        if kind == "lms":
            del want["logmel"]                      # model(lms) starts from the spectrogram
            frames = [int(c.shape[-1]) for c in batch]
        else:
            frames = [1 + w.shape[0] // 160 for w in batch]
        assert dict(recorder.count - before) == want
        assert [kw["taps"] * kw["c_in"] for op, kw in recorder.launches[n0:] if op == "conv_gemm"] == GEMM_K
        assert [tuple(o.shape) for o in outs] == [(f // 8, 2048) for f in frames]
    n = sum(recorder.count.values())
    print("\nbyola launches %s-%s: %d launches in %d batches checked in %.1f s; %s; worst error / bar: %s" % (
        case, precision, n, len(batches), time.time() - t0, dict(recorder.count),
        {k: round(v, 3) for k, v in sorted(recorder.worst.items())}))
    for k, v in recorder.count.items():
        STATS[k][0] += v
        STATS[k][1] = max(STATS[k][1], recorder.worst.get(k, 0.0))


def teardown_module(module):
    launch_check.report("byola launches", STATS)
