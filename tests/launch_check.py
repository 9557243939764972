"""Per-launch checking shared by the GPU launch-parity tests: `install` wraps `ops` entry points so that every call is
checked against its float64 reference of oracle/launch_ref.py as soon as it returns. Each call's tensor arguments are
cloned before it runs and its outputs right after; then
  (o) overlap no input tensor shares memory with an output tensor
  (a) replay  the op runs again on the cloned inputs into fresh outputs (NaN where the launch writes, a sentinel
              elsewhere; uint8 outputs: a sentinel byte everywhere): the written region is bit-identical to the
              in-pass output, the sentinel survives elsewhere
  (b) error   within the op's bar: row-wise  max|got - ref| / max|ref|  over each output row (one token's / one grid
              position's channels; 16-bit outputs may in addition differ by one ulp of their type at |ref|), or
              |got - ref| <= bar * tol element-wise where the reference gives a bound; uint8 outputs equal
  (c) zeros   every element the reference defines as zero (masked / padding rows, ReLU-clamped values) is exactly 0.0
A failure names the op, the product call site, the shapes / dtypes and the worst element with both values."""
import collections
import inspect
import os
import sys

import torch

import launch_ref
from audio_visual_deepfake_detection_b200 import ops

ENGINE_FILE = os.path.join("libs", "modeling", "engine.py")
BYOLA_FILE = os.path.join("libs", "features", "byola.py")

SENTINEL = 1024.0          # exact in fp32 / fp16 / bf16
SENTINEL_BYTE = 0xA5       # neither 0 nor 1, the values of a row mask
BAR = 5e-5                 # results accumulated in fp32
# mlp_fused: the bars of test_mlp_fused / test_block_tail_projection_ln2_mlp_in_one_launch (fp16), per row: the 16-bit
# hidden activations (and the tail's 16-bit LN2 operand) round at ties the kernel's fp32 and the reference's fp64 values
# fall on different sides of
BAR_MLP, BAR_TAIL = 2e-4, 2e-3
# logmel: the reference's per-element bound is the whole allowance; byola_pool: a max of stored values, exact
BAR_LOGMEL, BAR_POOL = 1.0, 0.0


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


def _call_site(product_file):
    """file:line, function and block (engine: `pre` / `head`; extractor: the conv layer `key`) of the product code that
    made the call."""
    f = sys._getframe(2)
    while f is not None and not f.f_code.co_filename.endswith(product_file):
        f = f.f_back
    if f is None:
        return "?"
    loc = f.f_locals
    return "%s:%d %s %s" % (os.path.basename(product_file), f.f_lineno, f.f_code.co_name,
                            loc.get("pre", loc.get("head", loc.get("key", ""))))


def _bar(name, kw):
    if name == "mlp_fused":
        return BAR_TAIL if kw["proj"] is not None else BAR_MLP
    if name == "logmel":
        return BAR_LOGMEL
    if name == "byola_pool":
        return BAR_POOL
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
    """Values per output row (one token, one grid position): the channels of the op's output, one head output per
    token, one mask byte per grid position."""
    if name == "conv_gemm":
        return ref.shape[-1] if path == "dots.1" else kw["n_out"]
    if name == "instnorm_lrelu":
        return kw["channels"]
    if name in ("head_final", "head_combine"):
        return 1 if path == "logits" else 2
    if name in ("vcls_exp12", "vcls_exp13"):
        return 1
    if name in ("byola_conv1_pool", "byola_pool"):
        return 1 if path == "mask_out" else 64
    return ref.shape[-1]


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
    if name == "logmel":
        return ["lms"]
    if name in ("byola_conv1_pool", "byola_pool"):
        return ["out"] + (["mask_out"] if kw["mask_out"] is not None else [])
    return ["out"]


class LaunchChecker:
    def __init__(self):
        self.count = collections.Counter()
        self.worst = {}
        self.launches = []                # (op, its scalar arguments) per checked launch, in call order

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
            tol = outs[0].tol
            for o in outs[1:]:
                written |= o.written
                ref = torch.where(o.written, o.ref, ref)
                zero = torch.where(o.written, o.zero, zero)
                mag = torch.where(o.written, o.mag if o.mag is not None else o.ref.abs(), mag)
                tol = None if tol is None else torch.where(o.written, o.tol, tol)
            merged[key] = (path, written, ref, zero, mag, tol)
            fresh = launch_ref.get_path(kw_re, path)
            if fresh.is_floating_point():
                fresh.fill_(SENTINEL)
                fresh[written] = float("nan")
            else:
                fresh.fill_(SENTINEL_BYTE)
        orig(**kw_re)
        torch.cuda.synchronize()
        bar = _bar(name, kw_in)
        for key, (path, written, ref, zero, mag, tol) in merged.items():
            got = recorded[key]
            fresh = launch_ref.get_path(kw_re, path)
            sentinel = SENTINEL if fresh.is_floating_point() else SENTINEL_BYTE
            assert torch.equal(fresh[written], got[written]), "%s: %s: replay differs from the in-pass output" % (ctx, path)
            assert bool((fresh[~written] == sentinel).all()), "%s: %s: replay wrote outside the region it owns" % (ctx, path)
            # (b) error against the float64 reference, (c) structural zeros
            worst = launch_ref.check(got, launch_ref.Out(ref, written, zero, mag, tol), _row_width(name, path, kw_in, ref), bar,
                                     "%s: %s" % (ctx, path))
            self.worst[name] = max(self.worst.get(name, 0.0), worst / bar if bar > 0 else worst)
        self.count[name] += 1
        self.launches.append((name, {k: v for k, v in kw_in.items() if isinstance(v, (int, float))}))


def install(monkeypatch, names, product_file):
    """Wraps the `ops` entry points `names` (each with a float64 reference); each call made from `product_file` or below
    it is checked as soon as it returns. Returns the LaunchChecker that counts them."""
    chk = LaunchChecker()
    for name in names:
        orig = getattr(ops, name)
        sig = inspect.signature(orig)

        def wrapped(*args, __name=name, __orig=orig, __sig=sig, **kwargs):
            ba = __sig.bind(*args, **kwargs)
            ba.apply_defaults()
            kw = dict(ba.arguments)
            site = _call_site(product_file)
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


def report(title, stats):
    """Prints a module's totals: op, launches, worst error / bar (byola_pool: worst error, bar 0)."""
    if stats:
        print("\n%s, all passes: op: launches, worst error / bar" % title)
        for k, (n, w) in sorted(stats.items()):
            print("  %-16s %6d  %.3f" % (k, n, w))
