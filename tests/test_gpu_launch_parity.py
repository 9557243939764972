"""Every kernel launch of real forward passes, checked one by one against the float64 references of
oracle/launch_ref.py. A fixture wraps the `ops` entry points the engine calls; each call's tensor arguments are cloned
before it runs and its outputs right after, and the launch is checked at once:
  (a) replay  the op runs again on the cloned inputs into fresh outputs (NaN where the launch writes, a sentinel
              elsewhere): the written region is bit-identical to the in-forward output, the sentinel survives elsewhere
  (b) error   row-wise  max|got - ref| / max|ref|  over each output row (one token's channels) within the op's bar;
              16-bit outputs may in addition differ by one ulp of their type at |ref|
  (c) zeros   every element the reference defines as zero (masked / padding rows, ReLU-clamped values) is exactly 0.0
A failure names the op, the engine call site and block, the shapes / dtypes and the worst element with both values.
Passes: every MODEL_CASES entry in fp32 and mixed at batch 3 and in mixed at batch 32 (the benchmark's batch: the only
passes that take the launch configurations that depend on the SM count), and exp12 mixed at batch 32 with each of the
engine's A/B switches AVDF_FUSE_TAIL, AVDF_FUSE_LN2, AVDF_FUSED_MLP turned off."""
import collections
import inspect
import os
import sys
import time

import pytest
import torch

import launch_ref
from make_golden import MODEL_CASES, VIDEO_CASES, make_item
from audio_visual_deepfake_detection_b200 import ops
from audio_visual_deepfake_detection_b200.libs.core import load_config_for
from audio_visual_deepfake_detection_b200.libs.modeling import make_meta_arch
from audio_visual_deepfake_detection_b200.libs.utils import synthetic as syn

pytestmark = pytest.mark.gpu

SENTINEL = 1024.0          # exact in fp32 / fp16 / bf16
BAR = 5e-5                 # results accumulated in fp32
# mlp_fused: the bars of test_mlp_fused / test_block_tail_projection_ln2_mlp_in_one_launch (fp16), per row: the 16-bit
# hidden activations (and the tail's 16-bit LN2 operand) round at ties the kernel's fp32 and the reference's fp64 values
# fall on different sides of
BAR_MLP, BAR_TAIL = 2e-4, 2e-3

ENGINE_FILE = os.path.join("libs", "modeling", "engine.py")
STATS = collections.defaultdict(lambda: [0, 0.0])          # op -> [launches, worst error / bar] over the whole module


def _tensors(v):
    if isinstance(v, torch.Tensor):
        yield v
    elif isinstance(v, (list, tuple)):
        for x in v:
            yield from _tensors(x)


def _clone_tree(v, memo):
    """Clone every tensor of an argument tree; a tensor passed twice (ln_dwconv_ln's interleaved outs) stays one tensor."""
    if isinstance(v, torch.Tensor):
        if id(v) not in memo:
            memo[id(v)] = v.clone()
        return memo[id(v)]
    if isinstance(v, (list, tuple)):
        return type(v)(_clone_tree(x, memo) for x in v)
    return v


def _span(t):
    s = t.data_ptr()
    return s, s + t.numel() * t.element_size()


def _call_site():
    f = sys._getframe(2)
    while f is not None and not f.f_code.co_filename.endswith(ENGINE_FILE):
        f = f.f_back
    if f is None:
        return "?"
    return "engine.py:%d %s %s" % (f.f_lineno, f.f_code.co_name, f.f_locals.get("pre", f.f_locals.get("head", "")))


def _bar(name, kw):
    if name == "mlp_fused":
        return BAR_TAIL if kw["proj"] is not None else BAR_MLP
    return BAR


def _describe(v):
    if isinstance(v, torch.Tensor):
        return "%s%s" % (str(v.dtype)[6:], list(v.shape))
    if isinstance(v, (list, tuple)):
        return "(%s)" % ", ".join(_describe(x) for x in v)
    if isinstance(v, dict):
        return ", ".join("%s=%s" % (k, _describe(x)) for k, x in v.items() if x is not None and k != "workspace")
    return repr(v)


def _row_width(name, path, kw, ref):
    """Values per output row (one token): the channels of the op's output, one head output per token."""
    if name == "conv_gemm":
        return ref.shape[-1] if path == "dots.1" else kw["n_out"]
    if name == "instnorm_lrelu":
        return kw["channels"]
    if name in ("head_final", "head_combine"):
        return 1 if path == "logits" else 2
    if name in ("vcls_exp12", "vcls_exp13"):
        return 1
    return ref.shape[-1]


class LaunchChecker:
    def __init__(self):
        self.count = collections.Counter()
        self.worst = {}

    def check(self, name, site, orig, kw_in, recorded):
        refs = launch_ref.REFERENCES[name](**kw_in)
        groups = {}                       # one entry per distinct output tensor: (tensor, [Out ...])
        for path, o in refs.items():
            t = launch_ref.get_path(kw_in, path)
            groups.setdefault(id(t), (t, path, []))[2].append(o)
        ctx = "%s at %s [%s]" % (name, site, _describe(kw_in))
        # (a) replay into fresh outputs
        memo = {}
        kw_re = {k: (None if k == "workspace" else _clone_tree(v, memo)) for k, v in kw_in.items()}
        merged = {}
        for key, (t, path, outs) in groups.items():
            written = outs[0].written.clone()
            ref, zero, mag = outs[0].ref.clone(), outs[0].zero.clone(), (outs[0].mag if outs[0].mag is not None else outs[0].ref.abs()).clone()
            for o in outs[1:]:
                written |= o.written
                ref = torch.where(o.written, o.ref, ref)
                zero = torch.where(o.written, o.zero, zero)
                mag = torch.where(o.written, o.mag if o.mag is not None else o.ref.abs(), mag)
            merged[key] = (path, written, ref, zero, mag)
            fresh = launch_ref.get_path(kw_re, path)
            fresh.fill_(SENTINEL)
            fresh[written] = float("nan")
        orig(**kw_re)
        torch.cuda.synchronize()
        bar = _bar(name, kw_in)
        for key, (path, written, ref, zero, mag) in merged.items():
            got = recorded[key]
            fresh = launch_ref.get_path(kw_re, path)
            assert torch.equal(fresh[written], got[written]), "%s: %s: replay differs from the in-forward output" % (ctx, path)
            assert bool((fresh[~written] == SENTINEL).all()), "%s: %s: replay wrote outside the region it owns" % (ctx, path)
            # (b) row-wise error against the float64 reference, (c) structural zeros
            worst = launch_ref.check(got, launch_ref.Out(ref, written, zero, mag), _row_width(name, path, kw_in, ref), bar,
                                     "%s: %s" % (ctx, path))
            self.worst[name] = max(self.worst.get(name, 0.0), worst / bar)
        self.count[name] += 1


@pytest.fixture
def recorder(monkeypatch):
    """Wraps every `ops` entry point that has a float64 reference; each call is checked as soon as it returns."""
    chk = LaunchChecker()
    for name in launch_ref.REFERENCES:
        orig = getattr(ops, name)
        sig = inspect.signature(orig)

        def wrapped(*args, __name=name, __orig=orig, __sig=sig, **kwargs):
            ba = __sig.bind(*args, **kwargs)
            ba.apply_defaults()
            kw = dict(ba.arguments)
            site = _call_site()
            outs = {id(launch_ref.get_path(kw, p)): launch_ref.get_path(kw, p) for p in _output_paths(__name, kw)}
            ins = [t for k, v in kw.items() if k != "workspace" for t in _tensors(v) if id(t) not in outs]
            for o in outs.values():
                for t in ins:
                    (a0, a1), (b0, b1) = _span(o), _span(t)
                    assert a1 <= b0 or b1 <= a0, "%s at %s: an input overlaps an output in memory" % (__name, site)
            memo = {}
            kw_in = {k: (None if k == "workspace" else _clone_tree(v, memo)) for k, v in kw.items()}
            r = __orig(**kw)
            recorded = {id(memo[k]): t.clone() for k, t in outs.items()}
            chk.check(__name, site, __orig, kw_in, recorded)
            return r
        monkeypatch.setattr(ops, name, wrapped)
    return chk


def _output_paths(name, kw):
    """The output argument paths of a call (the reference's keys, without running it)."""
    if name == "conv_gemm":
        return [p for p, on in (("out_f32", kw["out_f32"] is not None), ("out_h", kw["out_h"] is not None),
                                ("dots.1", kw["dots"] is not None)) if on]
    if name == "mlp_fused":
        return ["out"] + (["out_h"] if kw["out_h"] is not None else []) + \
               (["proj.6"] if kw["proj"] is not None and kw["proj"][6] is not None else [])
    if name == "ln_dwconv_ln":
        return ["outs.%d" % i for i in range(len(kw["outs"]))] + (["skip_out"] if kw["skip_out"] is not None else [])
    if name in ("head_final", "head_combine"):
        return ["logits", "offsets"]
    return ["out"]


_ITEMS = {}


def _items(use_video, batch):
    """batch items cycling through VIDEO_CASES' durations and the interp / ragged modes (ragged masks)."""
    if use_video not in _ITEMS:
        _ITEMS[use_video] = [make_item(d, s, m, use_video) for d, s, m in VIDEO_CASES]
    base = _ITEMS[use_video]
    return [base[i % len(base)] for i in range(batch)]


PASSES = [(case, prec, b, None) for case in MODEL_CASES for prec, b in (("fp32", 3), ("mixed", 3), ("mixed", 32))]
PASSES += [("exp12", "mixed", 32, env) for env in ("AVDF_FUSE_TAIL", "AVDF_FUSE_LN2", "AVDF_FUSED_MLP")]


@pytest.mark.parametrize("case,precision,batch,switch_off", PASSES,
                         ids=["%s-%s-b%d%s" % (c, p, b, "" if e is None else "-%s=0" % e) for c, p, b, e in PASSES])
def test_every_launch_of_a_forward_pass(case, precision, batch, switch_off, recorder, monkeypatch):
    if switch_off is not None:
        monkeypatch.setenv(switch_off, "0")          # read when the engine is built
    model_name, overrides, use_video, wseed = MODEL_CASES[case]
    cfg = load_config_for(model_name, dict(overrides))
    model = make_meta_arch(cfg["model_name"], **cfg["model"], precision=precision, max_batch=batch)
    model.load_state_dict(syn.synthetic_state_dict(cfg["model"], model_name, seed=wseed))
    model = model.to("cuda").eval()
    t0 = time.time()
    model.dense_outputs(_items(use_video, batch))
    torch.cuda.synchronize()
    n = sum(recorder.count.values())
    assert n > 0 and recorder.count["pack_feats"] == batch
    for op in ("conv_gemm", "attention", "ln_dwconv_ln"):
        assert recorder.count[op] > 0, op
    print("\nlaunch parity %s: %d launches checked in %.1f s; %s; worst error / bar: %s" % (
        "-".join(str(v) for v in (case, precision, batch, switch_off) if v is not None), n, time.time() - t0,
        dict(recorder.count), {k: round(v, 3) for k, v in sorted(recorder.worst.items())}))
    for k, v in recorder.count.items():
        STATS[k][0] += v
        STATS[k][1] = max(STATS[k][1], recorder.worst.get(k, 0.0))


def teardown_module(module):
    if STATS:
        print("\nlaunch parity, all passes: op: launches, worst error / bar")
        for k, (n, w) in sorted(STATS.items()):
            print("  %-16s %6d  %.3f" % (k, n, w))
