"""GPU tier: the FP16 engine layer by layer against float64, with bit-exact epilogues.

Every conv is checked in isolation: its input (and residual) tensors are read back from the engine itself, so errors of
earlier layers do not compound and the bounds can be tight.  For each tensor-core conv L with K = cin * k * k:

* accumulators: ``A = conv_accumulators(L)`` (fp32) against ``ref = conv(x, w)`` in float64, elementwise
  ``|A - ref| <= acc_tol(K) * mag`` with ``mag = conv(|x|, |w|)``.  Products of two halves are exact in fp32, so the
  only error is the rounding of the fp32 partial sums: at most about ``K * 2^-24 * mag`` if they are rounded to
  nearest, ``K * 2^-23 * mag`` if they are truncated.  Blackwell's ``kind::f16`` MMA truncates: on a B200 (1000 W)
  84 % of the accumulators that differ from float64 lie closer to zero, and the mean of sign(ref) * (A - ref) / mag is
  negative in every layer.  The worst ``|A - ref| / mag`` measured over every layer of the cases below (370 layer
  launches, K = 57 ... 4608) was 16.4 * 2^-24 (K = 4140) and never more than 1.36 * log2(K) * 2^-24; ``acc_tol`` is
  2.8 * log2(K) * 2^-24, twice that and 5 to 40 times below the truncation bound;
* per output channel, the mean of ``(A - ref) / mag`` over the sampled pixels, at most ``mean_tol(K)``.  Truncation
  makes it non-zero (measured: at most 0.82 * log2(K) * 2^-24); ``mean_tol`` is 1.7 * log2(K) * 2^-24.  A dropped
  channel, tap or k-chunk that shifts a whole channel the same way shows here even where single elements stay inside
  ``acc_tol``;
* epilogue: ``fp16_rn(relu(fp32(A + bias) + float(residual)))`` recomputed with numpy float32 on the engine's own A
  equals the forward's output tensor exactly (conv_tc.cuh epilogue16_f16 / epilogue16_f16_pre, conv_dual.cuh; the
  CUDA-core cross-check conv_direct_f16_kernel uses the same order).  The output is read before the accumulator dump
  re-runs the launch, so this also proves that the dump launch computes the forward's accumulators;
* overflow: an output is +-inf exactly where the float64 value rounds past 65504 (outside the accumulation bound),
  never NaN or a clamped finite value.

Besides the convs: the CUDA-core stem (keep_tensors runs it instead of the fused front end) and the product front end
(``debug_frontend``) against float64 within the stem's accumulation bound plus half an fp16 ulp; the max-pool bitwise
against a 3x3/2/1 max over the engine's stem tensor; the head against the pooled mean rebuilt in the kernel's own fixed
summation order (head_f16_kernel) and a float64 fc, within one fp16 ulp plus the fp32 sum bound of the fc.  The engine
exposes the pooled half only to the calibration observers, so it is checked through the logits.

The float64 reference runs on the first, the middle and the last image of a batch: a conv computes each image on its
own, so those images check every tile position of the launch (the ragged last M tile included).
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from oracle import model_factory as mf  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WIDTHS = {"w57": mf.PRUNED_WIDTHS, "w60": mf.DEFAULT_CFG_WIDTHS, "w64": mf.UNPRUNED_WIDTHS}
OP_CONV, OP_MAXPOOL, OP_HEAD = 0, 1, 2

U32 = 2.0 ** -24              # unit roundoff of fp32
F16_OVERFLOW = 65520.0        # the smallest magnitude that rounds to inf in fp16 (round to nearest even)
ACC_TOL_LOG2K = 2.8           # acc_tol(K) / (log2(K) * 2^-24): twice the worst measured (module docstring)
MEAN_TOL_LOG2K = 1.7          # mean_tol(K) / (log2(K) * 2^-24)


def acc_tol(k):
    return ACC_TOL_LOG2K * np.log2(k) * U32


def mean_tol(k):
    return MEAN_TOL_LOG2K * np.log2(k) * U32


# ------------------------------------------------------------------------------------------ float64 references

def _conv64(x, w, stride, pad):
    return F.conv2d(torch.from_numpy(np.asarray(x, np.float64)), torch.from_numpy(np.asarray(w, np.float64)),
                    stride=stride, padding=pad).numpy()


def _ulp16(v):
    """Spacing of fp16 numbers at |v| (2^-24 in the subnormal range)."""
    a = np.maximum(np.abs(v), 2.0 ** -14)
    return 2.0 ** (np.floor(np.log2(a)) - 10)


def _epilogue_f16(acc, bias, res, relu):
    """The FP16 conv epilogue in numpy float32: acc + bias, + float(residual), fmaxf(., 0), round to nearest fp16."""
    f = acc.astype(np.float32) + bias.astype(np.float32)[None, :, None, None]
    if res is not None:
        f = f + res.astype(np.float32)
    if relu:
        f = np.fmax(f, np.float32(0.0))              # fmaxf: a NaN operand yields the other one
    return f.astype(np.float16)


def _maxpool(t):
    return F.max_pool2d(torch.from_numpy(np.asarray(t, np.float64)), 3, 2, 1).numpy()


def _check_rounded(got16, v64, acc_bound, what):
    """``got16`` is fp16 of a value within ``acc_bound`` of the float64 ``v64``: it is +-inf exactly where that value
    rounds past the fp16 range, never NaN, and otherwise within half an fp16 ulp plus ``acc_bound`` of ``v64``."""
    got = got16.astype(np.float64)
    assert not np.isnan(got).any(), f"{what}: NaN in the engine's output"
    must_inf = np.abs(v64) - acc_bound >= F16_OVERFLOW
    may_inf = np.abs(v64) + acc_bound >= F16_OVERFLOW
    inf = np.isinf(got)
    assert inf[must_inf].all(), f"{what}: {int((~inf[must_inf]).sum())} values past the fp16 range are finite"
    assert not inf[~may_inf].any(), f"{what}: {int(inf[~may_inf].sum())} values inside the fp16 range came out inf"
    assert (np.sign(got[inf]) == np.sign(v64[inf])).all(), f"{what}: an overflow has the wrong sign"
    fin = ~inf
    err = np.abs(got[fin] - v64[fin])
    bound = 0.5 * _ulp16(np.maximum(np.abs(got[fin]), np.abs(v64[fin]))) + acc_bound[fin]
    worst = int(np.argmax(err - bound))
    assert (err <= bound).all(), f"{what}: |engine - float64| = {err[worst]:.4g} > bound {bound[worst]:.4g}"
    return int(inf.sum()), int(((got != 0) & (np.abs(got) < 2.0 ** -14)).sum())


def _sample(n):
    return sorted({0, n // 2, n - 1})


def _head_pooled(t16, cpad):
    """head_f16_kernel's pooled half: per channel, pixel phases ph = 0..P-1 each summed in fp32 in pixel order ph, ph+P,
    ...; the phase sums added in phase order; times fp32(1/hw); rounded to fp16."""
    n, c, hh, ww = t16.shape
    hw = hh * ww
    groups = cpad // 8
    phases = 1 if groups >= 256 else 256 // groups              # head_phases() with kHeadThreads = 256
    if phases * cpad > 4096:                                    # kHeadSumWords
        phases = 4096 // cpad
    v = t16.reshape(n, c, hw).astype(np.float32)
    total = np.zeros((n, c), np.float32)
    for ph in range(phases):
        s = np.zeros((n, c), np.float32)
        for px in range(ph, hw, phases):
            s = s + v[:, :, px]
        total = total + s
    return (total * (np.float32(1.0) / np.float32(hw))).astype(np.float16)


# ------------------------------------------------------------------------------------------ one network, layer by layer

def _stem_bound(ref, mag, bias):
    """7x7x3 stem, which has no accumulator dump: the derived worst case of 147 truncated fp32 partial sums, then the
    fp32 bias add."""
    return 147 * 2 * U32 * mag + 2 * U32 * (np.abs(ref) + np.abs(bias)[None, :, None, None])


def check_layers(eng, ref_net, x16, logits, log):
    """All checks of the module docstring on an engine that has just run ``logits = eng(x16.cuda())`` with keep_tensors=1.
    Weights and biases of the reference come from ``ref_net``; every tensor comes from the engine.  Appends one line per
    conv to ``log``; returns (worst accumulator ratio, worst channel mean, overflows, subnormal outputs)."""
    layers = eng.net.layers
    n = x16.shape[0]
    s = _sample(n)
    worst_ratio = worst_mean = 0.0
    n_inf = n_sub = 0
    stem, pool = layers[0], layers[1]
    assert stem.op == OP_CONV and pool.op == OP_MAXPOOL and layers[-1].op == OP_HEAD
    # ---- stem (CUDA-core kernel under keep_tensors) and max-pool
    R = ref_net.layers[0]
    stem_out = eng.read_tensor(stem.out_tensor)
    xs = x16[s].astype(np.float64)
    ref = _conv64(xs, R.weight, R.stride, R.pad)
    mag = _conv64(np.abs(xs), np.abs(R.weight.astype(np.float64)), R.stride, R.pad)
    v64 = np.maximum(ref + R.bias.astype(np.float64)[None, :, None, None], 0.0)
    i, u = _check_rounded(stem_out[s], v64, _stem_bound(ref, mag, R.bias), "stem")
    n_inf, n_sub = n_inf + i, n_sub + u
    pooled = eng.read_tensor(pool.out_tensor)
    assert np.array_equal(pooled, _maxpool(stem_out).astype(np.float16)), "max-pool differs from a 3x3/2/1 max of the stem"
    # ---- every tensor-core conv
    for li, L in enumerate(layers):
        if L.op != OP_CONV or li == 0:
            continue
        R = ref_net.layers[li]
        out = eng.read_tensor(L.out_tensor)                   # the forward's output, before the dump launch rewrites it
        x = eng.read_tensor(L.in_tensor)
        res = eng.read_tensor(L.res_tensor) if L.res_tensor >= 0 else None
        acc = eng.conv_accumulators(L.name, n)
        assert np.array_equal(out, _epilogue_f16(acc, R.bias, res, R.relu), equal_nan=True), \
            f"{L.name}: output differs from fp16(relu(acc + bias (+ residual))) recomputed on the engine's accumulators " \
            f"({int((out != _epilogue_f16(acc, R.bias, res, R.relu)).sum())} elements)"
        xs = x[s].astype(np.float64)
        w = R.weight.astype(np.float64)
        ref = _conv64(xs, w, R.stride, R.pad)
        mag = _conv64(np.abs(xs), np.abs(w), R.stride, R.pad)
        a = acc[s].astype(np.float64)
        err = np.abs(a - ref)
        K = R.cin * R.ksize * R.ksize
        ok = err <= acc_tol(K) * mag
        ratio = float(np.max(np.where(mag > 0, err / np.where(mag > 0, mag, 1.0), np.where(err > 0, np.inf, 0.0))))
        rel = np.where(mag > 0, (a - ref) / np.where(mag > 0, mag, 1.0), 0.0)
        chan_mean = float(np.abs(rel.mean(axis=(0, 2, 3))).max())
        log.append(f"{L.name:24s} K={K:5d} worst |A-ref|/mag = {ratio:.3e} ({ratio / U32:6.2f} u, tol {acc_tol(K) / U32:6.2f} u)  "
                   f"worst |channel mean| = {chan_mean / U32:5.2f} u (tol {mean_tol(K) / U32:5.2f} u)")
        assert ok.all(), f"{L.name}: {int((~ok).sum())} accumulators off by more than {acc_tol(K):.2e} * mag (worst {ratio:.3e})"
        assert chan_mean <= mean_tol(K), f"{L.name}: a channel's mean (A - ref) / mag is {chan_mean:.3e} > {mean_tol(K):.2e}"
        worst_ratio, worst_mean = max(worst_ratio, ratio), max(worst_mean, chan_mean)
        r64 = res[s].astype(np.float64) if res is not None else 0.0
        v64 = ref + R.bias.astype(np.float64)[None, :, None, None] + r64
        if R.relu:
            v64 = np.maximum(v64, 0.0)
        bound = acc_tol(K) * mag + 2 * U32 * (np.abs(ref) + np.abs(R.bias)[None, :, None, None] + np.abs(r64))
        i, u = _check_rounded(out[s], v64, bound, L.name)
        n_inf, n_sub = n_inf + i, n_sub + u
    # ---- head: pooled mean in the kernel's order, fc in float64
    H = ref_net.layers[-1]
    t = eng.read_tensor(layers[-1].in_tensor)
    cpad = eng.tensor_shape(layers[-1].in_tensor)[4]
    y = logits.astype(np.float64)
    fin = np.isfinite(t.reshape(n, -1).astype(np.float32)).all(axis=1)    # an inf in the last tensor makes NaN logits
    mh = _head_pooled(t[fin], cpad).astype(np.float64)
    w = H.weight.astype(np.float64)
    b = H.bias.astype(np.float64)
    ref = mh @ w.T + b
    bound = _ulp16(ref) + (H.cin + 64) * U32 * (np.abs(mh) @ np.abs(w).T + np.abs(b))
    err = np.abs(y[fin] - ref)
    assert (err <= bound).all(), f"logits off by {float((err - bound).max()):.3g} beyond the bound"
    return worst_ratio, worst_mean, n_inf, n_sub


def check_front_end(eng, ref_net, x16):
    """The product front end (fused quantize-free FP16 stem + ReLU + max-pool, tensor cores) against float64."""
    pooled, _ = eng.debug_frontend(torch.from_numpy(x16).cuda(), want_acc=False)
    R = ref_net.layers[0]
    s = _sample(x16.shape[0])
    xs = x16[s].astype(np.float64)
    ref = _conv64(xs, R.weight, R.stride, R.pad)
    mag = _conv64(np.abs(xs), np.abs(R.weight.astype(np.float64)), R.stride, R.pad)
    v64 = np.maximum(ref + R.bias.astype(np.float64)[None, :, None, None], 0.0)
    # max is monotone and 1-Lipschitz: the pooled value is within the window's largest stem bound of the pooled float64
    _check_rounded(pooled[s], _maxpool(v64), _maxpool(_stem_bound(ref, mag, R.bias)), "front end (product)")


def run_case(ref_net, x16, eng_net=None, max_batch=None, dual=True, front_end=True):
    """Engine over ``eng_net`` (default: ``ref_net``), one forward with keep_tensors=1, all checks.  Returns the
    statistics of ``check_layers``."""
    import ievm_b200
    eng = ievm_b200.B200HalfResNet(eng_net if eng_net is not None else ref_net, max_batch=max_batch or x16.shape[0])
    try:
        eng.set_option("keep_tensors", 1)
        if not dual:
            eng.set_option("dual", 0)
        logits = eng(torch.from_numpy(x16).cuda()).cpu().numpy()
        log = []
        stats = check_layers(eng, ref_net, x16, logits, log)
        if front_end:                                  # last: it overwrites the kept max-pool tensor
            check_front_end(eng, ref_net, x16)
        print("\n".join(log))
        print(f"worst accumulator ratio {stats[0]:.3e}, worst channel mean {stats[1]:.3e}, "
              f"{stats[2]} overflows, {stats[3]} subnormal outputs")
        return stats
    finally:
        eng.close()


def student_spec(widths):
    import ievm_b200
    return ievm_b200.from_half_module(mf.cast_fp16(mf.make_student(widths)))


def images(n, seed):
    return mf.synthetic_images(n, seed=seed).half().numpy()


# ------------------------------------------------------------------------------------------ tests

# batch 3: every halo layer takes the single-accumulator ("tiny") path; 77: the accumulator ring, more than one sub-tile
# per SM and a ragged last M tile in every layer (77 * 28 * 28 = 471.6 tiles of 128 pixels).  max_batch 256 plans the
# tiles (widths, CTA pairs) as the product engine does.
@pytest.mark.parametrize("n", [3, 77])
@pytest.mark.parametrize("tag", ["w57", "w60", "w64"])
def test_fp16_student_every_conv_vs_float64(tag, n):
    run_case(student_spec(WIDTHS[tag]), images(n, seed=61 + n), max_batch=256 if n > 3 else 4)


@pytest.mark.parametrize("n", [3, 37])
def test_fp16_teacher_resnet50_every_conv_vs_float64(n):
    """Bottleneck shapes that exist only in FP16: 1x1 convs up to 2048 channels, the 3x3 stride-2 conv2, 1x1 stride-2
    downsamples and a 2048-wide head."""
    import ievm_b200
    spec = ievm_b200.from_half_module(mf.cast_fp16(mf.make_teacher()))
    run_case(spec, images(n, seed=67 + n), max_batch=256 if n > 3 else 4)


def test_fp16_student_without_dual_launch():
    """dual = 0: the 1x1 downsample convs run as launches of their own instead of as the second tile class."""
    run_case(student_spec(WIDTHS["w60"]), images(77, seed=71), max_batch=256, dual=False)


def test_fp16_edge_values_overflow_and_tiny_inputs():
    """Image 0 scaled by 1408: layer-4 tensors reach ~60000 and only the last conv overflows, so no conv reads an inf;
    image 1 filled with 1e-4 (stem products far below the fp16 normal range); image 2 plain.  Overflows must be inf
    exactly where the float64 value rounds to inf; the batch must really contain overflows and subnormal outputs."""
    x = images(3, seed=73)
    x[0] = (x[0].astype(np.float32) * 1408).astype(np.float16)
    x[1] = np.float16(1e-4)
    _, _, n_inf, n_sub = run_case(student_spec(WIDTHS["w57"]), x)
    assert n_inf > 0 and n_sub > 0, (n_inf, n_sub)


_VARIANT = r"""
import os, sys
sys.path.insert(0, sys.argv[1])
sys.path.insert(0, os.path.join(sys.argv[1], "tests"))
import test_gpu_fp16_layers as T
n = int(sys.argv[2])
T.run_case(T.student_spec(T.WIDTHS["w57"]), T.images(n, seed=79), max_batch=256 if n > 3 else 4, front_end=False)
print("variant ok")
"""


# batch 77 except for IEVM_TINY=0, which changes nothing there: batch 3 is where the single-accumulator form would run
@pytest.mark.parametrize("env,n", [
    ({"IEVM_HALO_STATIC": "0"}, 77),                       # run-time-shaped halo kernel (shape class 0)
    ({"IEVM_BAND_SUBS": "1"}, 77),                         # one sub-tile per TMA patch
    ({"IEVM_BAND_SUBS": "3", "IEVM_KB_GROUP": "1"}, 77),   # odd band size (partial last band), one k-block per barrier
    ({"IEVM_HALO": "0"}, 77),                              # every conv through per-tap im2col TMA
    ({"IEVM_DUAL": "0"}, 77),                              # the 1x1 downsample convs as launches of their own
    ({"IEVM_TINY": "0"}, 3),                               # small batches through the accumulator ring
], ids=["halo_dynamic", "band1", "band3_kb1", "no_halo", "no_dual", "no_tiny"])
def test_fp16_kernel_configuration_fallbacks_every_conv_vs_float64(env, n, tmp_path):
    script = tmp_path / "variant.py"
    script.write_text(_VARIANT)
    e = dict(os.environ)
    e.update(env)
    r = subprocess.run([sys.executable, str(script), ROOT, str(n)], env=e, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "variant ok" in r.stdout, (r.stdout[-3000:], r.stderr[-3000:])
