"""GPU tier, round 2: the parity gaps the round-1 review named (FP16 at full batch / ragged / per layer / other width
sets, INT8 accumulators for every width set), the pipelined host entry points, stream ordering on one handle, the
kernel-configuration fallbacks (run-time-shaped halo kernel, band sizes, k-block groups) and the measurement probes.
Everything goes through the C ABI (ctypes)."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from ievm_testutil import cached_quantized  # noqa: E402
from oracle import int8_forward as O  # noqa: E402
from oracle import model_factory as mf  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FP16_REL_TOL = 1e-2     # north_star: FP16 logits within 1e-2 relative (row-normalised, SURVEY 8c)
FP16_LAYER_TOL = 2e-2   # every FP16 tensor vs the fp32 forward of the same (fp16-stored) weights, relative to the tensor's max


def _row_rel(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return float((np.abs(a - b).max(axis=1) / np.maximum(np.abs(b).max(axis=1), 1.0)).max())


# ------------------------------------------------------------------------------------------ INT8: every width set

@pytest.mark.parametrize("widths", [mf.DEFAULT_CFG_WIDTHS, mf.UNPRUNED_WIDTHS], ids=["w60", "w64"])
def test_int8_tensors_and_accumulators_bit_exact_other_width_sets(widths):
    """Round 1 asserted accumulator exactness for [57,115,230,460] only; the other width sets pad differently
    (60 -> 64, 121 -> 128, 243 -> 256, 486 -> 2 x 256 / 64 ... 512 un-padded)."""
    import ievm_b200
    gm = cached_quantized(widths)
    net = O.extract_qnet(gm)
    eng = ievm_b200.B200QuantizedResNet.from_converted(gm, max_batch=4)
    eng.set_option("keep_tensors", 1)
    x = mf.synthetic_images(3, seed=23)
    y = eng(x.cuda()).cpu().numpy()
    yo = O.forward(net, x.numpy(), keep=True)
    assert np.array_equal(y, yo)
    checked = 0
    for tid, name in sorted(eng.net.tensor_names.items()):
        if name in net.trace:
            assert np.array_equal(eng.read_tensor(tid), net.trace[name]), f"tensor {name} differs"
            checked += 1
    assert checked == 22
    for L in eng.net.layers[2:-1]:
        if L.op == 0:
            assert np.array_equal(eng.conv_accumulators(L.name, 3), net.trace[L.name + ":acc"]), f"accumulators of {L.name}"
    eng.close()


# ------------------------------------------------------------------------------------------ FP16: the thin spots

def _fp16_engine_and_module(widths, max_batch):
    import ievm_b200
    m16 = mf.cast_fp16(mf.make_student(widths))
    return ievm_b200.B200HalfResNet.from_half_module(m16, max_batch=max_batch), m16


@pytest.mark.parametrize("widths", [mf.PRUNED_WIDTHS, mf.DEFAULT_CFG_WIDTHS, mf.UNPRUNED_WIDTHS], ids=["w57", "w60", "w64"])
def test_fp16_student_batch_256_vs_cudnn_half(widths):
    """BASELINE config 2 at its real batch (and config 5's un-pruned student): 256 images against the reference's own
    ``model.half()`` forward on this GPU (cuDNN), row-relative 1e-2 and identical arg-max."""
    eng, m16 = _fp16_engine_and_module(widths, 256)
    x = mf.synthetic_images(256, seed=41).half().cuda()
    y = eng(x).float().cpu().numpy()
    with torch.no_grad():
        ref = m16.cuda()(x).float().cpu().numpy()
    assert _row_rel(y, ref) < FP16_REL_TOL
    top2 = np.sort(ref, axis=1)[:, -2:]
    clear = (top2[:, 1] - top2[:, 0]) > 2e-2 * np.maximum(np.abs(ref).max(axis=1), 1.0)     # rows without a near tie
    assert (y.argmax(1) == ref.argmax(1))[clear].all() and clear.mean() > 0.9
    eng.close()


def test_fp16_ragged_batches_and_batch_invariance():
    """The FP16 twins of the INT8 ragged / invariance tests: an image's logits do not depend on the batch it rides in
    (bitwise: same kernels, same reduction order), ragged batches equal the reference within tolerance."""
    eng, m16 = _fp16_engine_and_module(mf.PRUNED_WIDTHS, 256)
    x = mf.synthetic_images(256, seed=43).half().cuda()
    full = eng(x).clone()
    m16 = m16.cuda()
    for n in (1, 5, 13, 64, 255):
        part = eng(x[:n])
        assert torch.equal(part, full[:n]), f"fp16 batch {n} differs from batch 256"
        with torch.no_grad():
            ref = m16(x[:n]).float().cpu().numpy()
        assert _row_rel(part.float().cpu().numpy(), ref) < FP16_REL_TOL
    parts = torch.cat([eng(x[i:i + 32]).clone() for i in range(0, 256, 32)])
    assert torch.equal(parts, full)
    eng.close()


def test_fp16_every_tensor_vs_fp32_forward():
    """Per-layer FP16 check: every tensor the engine produces against an fp32 torch forward of the same fp16-stored
    weights (BN applied in fp32, as the engine folds it), relative to the tensor's own magnitude."""
    import ievm_b200
    m16 = mf.cast_fp16(mf.make_student(mf.PRUNED_WIDTHS))
    eng = ievm_b200.B200HalfResNet.from_half_module(m16, max_batch=4)
    eng.set_option("keep_tensors", 1)
    x = mf.synthetic_images(3, seed=47).half()
    y = eng(x.cuda()).float().cpu().numpy()
    m32 = mf.cast_fp16(mf.make_student(mf.PRUNED_WIDTHS)).float().eval()
    ref = {}

    def hook(name):
        return lambda _m, _i, out: ref.__setitem__(name, out.detach().numpy())

    handles = [m32.maxpool.register_forward_hook(hook("maxpool"))]
    for li in (1, 2, 3, 4):
        for bi in (0, 1):
            blk = getattr(m32, f"layer{li}")[bi]
            handles.append(blk.register_forward_hook(hook(f"layer{li}.{bi}")))
    with torch.no_grad():
        y32 = m32(x.float()).numpy()
    for h in handles:
        h.remove()
    assert _row_rel(y, y32) < FP16_REL_TOL
    checked = 0
    names = {nm: tid for tid, nm in eng.net.tensor_names.items()}
    for name, want in ref.items():
        # the block's output tensor carries the name of its last conv (the add is fused into it)
        cands = [name, f"{name}.conv2", f"{name}.relu"]
        tid = next((names[c] for c in cands if c in names), None)
        if tid is None:
            continue
        got = eng.read_tensor(tid).astype(np.float32)
        assert got.shape == want.shape, (name, got.shape, want.shape)
        err = np.abs(got - want).max() / max(np.abs(want).max(), 1.0)
        assert err < FP16_LAYER_TOL, f"{name}: {err:.3e}"
        checked += 1
    assert checked >= 9, f"only {checked} FP16 tensors could be matched by name: {sorted(names)}"
    eng.close()


def test_fp16_teacher_resnet50_batch_64_vs_cudnn_half():
    import ievm_b200
    m16 = mf.cast_fp16(mf.make_teacher())
    eng = ievm_b200.B200HalfResNet.from_half_module(m16, max_batch=64)
    x = mf.synthetic_images(64, seed=49).half().cuda()
    y = eng(x).float().cpu().numpy()
    with torch.no_grad():
        ref = m16.cuda()(x).float().cpu().numpy()
    assert _row_rel(y, ref) < FP16_REL_TOL
    assert torch.equal(eng(x[:7]), eng(x)[:7])
    eng.close()


# ------------------------------------------------------------------------------------------ pipelined host path

def test_submit_wait_equals_the_synchronous_call():
    """ievm_submit_*_host / ievm_wait: five batches through two slots, results in order and bit-identical to the
    synchronous entry points, for f32, uint8 and FP16 inputs."""
    import ievm_b200
    gm = cached_quantized(mf.PRUNED_WIDTHS)
    eng = ievm_b200.B200QuantizedResNet.from_converted(gm, max_batch=16)
    xs = [mf.synthetic_images(n, seed=70 + i).pin_memory() for i, n in enumerate((16, 3, 16, 9, 1))]
    want = [eng(x.cuda()).cpu() for x in xs]
    pend = [eng.submit(x) for x in xs[:2]]
    got = []
    for x in xs[2:]:
        got.append(pend.pop(0).result())
        pend.append(eng.submit(x))
    got += [p.result() for p in pend]
    for g, w in zip(got, want):
        assert not g.is_cuda and torch.equal(g, w)
    # pageable (un-pinned) input works too
    assert torch.equal(eng.submit(mf.synthetic_images(5, seed=70)).result(), eng(mf.synthetic_images(5, seed=70).cuda()).cpu())
    # decoded 8-bit images, with and without the resize stage
    u8 = torch.randint(0, 256, (7, 224, 224, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(1)).pin_memory()
    assert torch.equal(eng.submit(u8).result(), eng.forward_u8(u8.cuda()).cpu())
    u200 = torch.randint(0, 256, (4, 200, 200, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(2)).pin_memory()
    assert torch.equal(eng.submit(u200).result(), eng.forward_u8(u200.cuda()).cpu())
    with pytest.raises(ValueError):
        eng.submit(xs[0].cuda())
    eng.close()
    e16, _ = _fp16_engine_and_module(mf.PRUNED_WIDTHS, 8)
    x16 = mf.synthetic_images(8, seed=75).half().pin_memory()
    assert torch.equal(e16.submit(x16).result(), e16(x16.cuda()).cpu())
    e16.close()


@pytest.mark.parametrize("kind", ["f32", "u8_resize", "fp16"])
def test_submit_results_read_out_of_order_are_not_overwritten(kind):
    """Three submits before any result: the third reuses the first call's pinned logits buffer.  Each result, read in
    the order 3, 2, 1, must still be its own batch's logits (the first call is settled before its buffer is reused)."""
    import ievm_b200
    sizes = (16, 3, 9)
    if kind == "fp16":
        eng, _ = _fp16_engine_and_module(mf.PRUNED_WIDTHS, 16)
        xs = [mf.synthetic_images(n, seed=110 + i).half().pin_memory() for i, n in enumerate(sizes)]
        want = [eng(x.cuda()).cpu() for x in xs]
    else:
        eng = ievm_b200.B200QuantizedResNet.from_converted(cached_quantized(mf.PRUNED_WIDTHS), max_batch=16)
        if kind == "f32":
            xs = [mf.synthetic_images(n, seed=110 + i).pin_memory() for i, n in enumerate(sizes)]
            want = [eng(x.cuda()).cpu() for x in xs]
        else:
            g = torch.Generator().manual_seed(110)
            xs = [torch.randint(0, 256, (n, 200, 200, 3), dtype=torch.uint8, generator=g).pin_memory() for n in sizes]
            want = [eng.forward_u8(x.cuda()).cpu() for x in xs]
    pend = [eng.submit(x) for x in xs]
    got = [None] * 3
    for i in (2, 1, 0):
        got[i] = pend[i].result()
    for i, (g_, w) in enumerate(zip(got, want)):
        assert g_.shape == w.shape and torch.equal(g_, w), \
            f"{kind}: result of submit {i + 1} (batch {sizes[i]}) is not its own batch's logits"
    eng.close()


def test_evaluate_accuracy_over_cpu_batches_is_pipelined_and_exact():
    """The reference's loop (engines.py:52-63) over CPU batches: same accuracy as the reference module on the CPU."""
    import ievm_b200
    gm = cached_quantized(mf.PRUNED_WIDTHS)
    torch.backends.quantized.engine = "fbgemm"
    eng = ievm_b200.B200QuantizedResNet.from_converted(gm, max_batch=32)
    g = torch.Generator().manual_seed(4)
    loader = [(mf.synthetic_images(n, seed=80 + i), torch.randint(0, 6, (n,), generator=g)) for i, n in enumerate((32, 32, 17))]
    correct = total = 0
    with torch.no_grad():
        for images, labels in loader:
            _, pred = torch.max(gm(images), 1)
            correct += int((pred == labels).sum())
            total += labels.shape[0]
    assert ievm_b200.evaluate_accuracy(eng, loader) == pytest.approx(100.0 * correct / total, abs=1e-9)
    eng.close()


def test_forwards_from_different_streams_are_ordered():
    """One handle, one activation workspace: a forward on a side stream followed by the host-buffer path (the engine's
    own stream), and forwards alternating between two torch streams, must not race (ADVICE r1)."""
    import ievm_b200
    gm = cached_quantized(mf.PRUNED_WIDTHS)
    eng = ievm_b200.B200QuantizedResNet.from_converted(gm, max_batch=64)
    xa = mf.synthetic_images(64, seed=90)
    xb = mf.synthetic_images(64, seed=91)
    xa_d, xb_d = xa.cuda(), xb.cuda()
    ya, yb = eng(xa_d).clone(), eng(xb_d).clone()
    torch.cuda.synchronize()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    for rep in range(10):
        with torch.cuda.stream(s1):
            y1 = eng(xa_d)
        y2 = eng(xb)                       # CPU tensor: H2D + forward on the engine's own stream + D2H
        with torch.cuda.stream(s2):
            y3 = eng(xb_d)
        with torch.cuda.stream(s1):
            y4 = eng(xa_d)
        torch.cuda.synchronize()
        assert torch.equal(y1, ya) and torch.equal(y2, yb.cpu()) and torch.equal(y3, yb) and torch.equal(y4, ya), rep
    assert torch.cuda.current_device() == eng.device_index
    eng.close()


def test_graph_cache_is_bounded_and_correct():
    import ievm_b200
    eng = ievm_b200.B200QuantizedResNet.from_converted(cached_quantized(mf.PRUNED_WIDTHS), max_batch=4)
    x = mf.synthetic_images(4, seed=95).cuda()
    want = eng(x).clone()
    eng.set_option("use_graph", 1)
    keep = []
    for i in range(40):                    # every call has fresh input / output pointers: 40 captures, 16 kept
        xi = x.clone()
        keep.append(xi)
        assert torch.equal(eng(xi), want), i
    eng.close()


# ------------------------------------------------------------------------------------------ loss / counter edge cases

def test_out_of_range_labels_do_not_read_out_of_bounds():
    import ievm_b200
    from ievm_b200 import _lib
    g = torch.Generator().manual_seed(5)
    s, t = torch.randn(64, 6, generator=g).cuda(), torch.randn(64, 6, generator=g).cuda()
    y = torch.randint(0, 6, (64,), generator=g)
    y[3], y[10] = -100, 6
    out = ievm_b200.kd_eval_loss(s, t, y.cuda()).cpu()
    assert torch.isnan(out[1]) and torch.isfinite(out[2])           # CE poisoned, KL untouched
    counters = torch.zeros(2, dtype=torch.int64, device="cuda")
    lib = _lib.load()
    _lib.check(lib.ievm_count_correct(s.data_ptr(), 0, y.cuda().data_ptr(), 64, 6, counters.data_ptr(), None), "count")
    ok = (s.cpu().argmax(1) == y)
    assert counters.cpu().tolist() == [int(ok.sum()), 64]
    with pytest.raises(ValueError):
        ievm_b200.kd_eval_loss(s, t[:32], y.cuda())
    with pytest.raises(ValueError):
        ievm_b200.kd_eval_loss(s, t, y)                              # labels on the CPU


def test_mma_peak_probe_is_plausible():
    """The roofline denominator bench.py measures: a B200 tensor core retires 8192 int8 / 4096 fp16 MACs per clock per
    SM; at 1.5-1.97 GHz on 148 SMs that is 3.6-4.8 / 1.8-2.4 peta-ops."""
    import ievm_b200
    i8 = ievm_b200.measure_mma_peak("i8", 0, iters=2000)
    f16 = ievm_b200.measure_mma_peak("f16", 0, iters=2000)
    assert 3000 < i8 < 5000, i8
    assert 1500 < f16 < 2500, f16
    assert 1.8 < i8 / f16 < 2.2


# ------------------------------------------------------------------------------------------ kernel-configuration fallbacks

_VARIANT = r"""
import os, sys
sys.path.insert(0, sys.argv[1])
sys.path.insert(0, os.path.join(sys.argv[1], "tests"))
import numpy as np, torch
import ievm_b200
from ievm_testutil import cached_quantized
from oracle import model_factory as mf
g = np.load(os.path.join(sys.argv[1], "tests", "golden", "int8_w57.npz"))
eng = ievm_b200.B200QuantizedResNet.from_converted(cached_quantized(mf.PRUNED_WIDTHS), max_batch=64)
y = eng(mf.synthetic_images(int(g["n_images"])).cuda()).cpu().numpy()
assert np.array_equal(y, g["logits"]), np.abs(y - g["logits"]).max()
x = mf.synthetic_images(64, seed=5).cuda()
y_tc = eng(x).clone()
eng.set_option("conv_impl", 1)
assert torch.equal(y_tc, eng(x))
m16 = mf.cast_fp16(mf.make_student(mf.PRUNED_WIDTHS))
e16 = ievm_b200.B200HalfResNet.from_half_module(m16, max_batch=8)
x16 = mf.synthetic_images(8, seed=6).half().cuda()
with torch.no_grad():
    r16 = m16.cuda()(x16).float()
y16 = e16(x16).float()
rel = float(((y16 - r16).abs().amax(1) / r16.abs().amax(1).clamp_min(1.0)).max())
assert rel < 1e-2, rel
print("variant ok")
"""


@pytest.mark.parametrize("env", [
    {"IEVM_HALO_STATIC": "0"},                       # run-time-shaped halo kernel (shape class 0)
    {"IEVM_BAND_SUBS": "1"},                         # one sub-tile per TMA patch
    {"IEVM_BAND_SUBS": "3", "IEVM_KB_GROUP": "1"},   # odd band size (partial last band), one k-block per barrier
    {"IEVM_HALO": "0"},                              # every conv through per-tap im2col TMA
    {"IEVM_DUAL": "0"},                              # the 1x1 downsample convs as launches of their own
    {"IEVM_S2": "0"},                                # stride-2 dual launch as pixel pairs instead of phase patches (conv_s2.cuh off)
    {"IEVM_S2": "0", "IEVM_WIDE": "0"},              # ... and without the pixel-pair form (nine 64-byte-row taps)
    {"IEVM_TINY": "0"},                              # small batches through the accumulator ring (no single-accumulator form)
], ids=["halo_dynamic", "band1", "band3_kb1", "no_halo", "no_dual", "no_phase_patches", "no_pixel_pairs", "no_tiny"])
def test_kernel_configuration_fallbacks_stay_bit_exact(env, tmp_path):
    script = tmp_path / "variant.py"
    script.write_text(_VARIANT)
    e = dict(os.environ)
    e.update(env)
    r = subprocess.run([sys.executable, str(script), ROOT], env=e, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "variant ok" in r.stdout, (r.stdout[-2000:], r.stderr[-3000:])


# ------------------------------------------------------------------------------------------ non-zero input zero points

def test_tensor_core_convs_with_nonzero_input_zero_points():
    """SURVEY section 7: a tensor-core layer whose input zero point is not 0 gets the border-aware -zp * sum(w)
    correction instead of being refused.  The converted ResNet never has one (every conv input is post-ReLU), so the
    test moves the zero points of block outputs and of the ConvReLU2d outputs away from 0 in the converted module
    (tests/ievm_testutil.py: with_nonzero_zero_points), so the oracle and the engine's flattened description both read
    them, and demands bit-exact tensors and accumulators again -- through the halo kernel (layers 1-2), the im2col
    kernels (stride 2, 1x1, layers 3-4), the CTA-pair kernels and the head."""
    import ievm_b200
    from ievm_testutil import with_nonzero_zero_points
    gm = with_nonzero_zero_points(cached_quantized(mf.PRUNED_WIDTHS))
    onet = O.extract_qnet(gm)
    spec = ievm_b200.from_converted(gm)
    assert sum(1 for L in spec.layers if L.op == 0 and L.in_zp != 0 and L.in_tensor != 0) >= 15
    assert [b.add_zp for b in onet.blocks] == [5 + 3 * i for i in range(8)]
    eng = ievm_b200.B200QuantizedResNet(spec, max_batch=8)
    eng.set_option("keep_tensors", 1)
    x = mf.synthetic_images(5, seed=33)
    y = eng(x.cuda()).cpu().numpy()
    yo = O.forward(onet, x.numpy(), keep=True)
    for tid, name in sorted(eng.net.tensor_names.items()):
        if name in onet.trace:
            assert np.array_equal(eng.read_tensor(tid), onet.trace[name]), f"tensor {name} differs"
    for L in eng.net.layers[2:-1]:
        if L.op == 0:
            assert np.array_equal(eng.conv_accumulators(L.name, 5), onet.trace[L.name + ":acc"]), f"accumulators of {L.name}"
    assert np.array_equal(y, yo)
    eng.set_option("keep_tensors", 0)              # product configuration (fused front end, shared workspace)
    assert np.array_equal(eng(x.cuda()).cpu().numpy(), yo)
    eng.set_option("conv_impl", 1)                 # CUDA-core cross-check
    assert np.array_equal(eng(x.cuda()).cpu().numpy(), yo)
    eng.close()
