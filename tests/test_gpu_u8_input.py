"""GPU tier: the decoded-image input path of the INT8 engine -- the u8 front end (``frontend2_kernel<I8, 1, ...>``: a 3 x
256 lookup table in place of ToTensor + Normalize + quantize_per_tensor) and the GPU Pillow resize -- bit for bit against
the reference transform, tensor by tensor, at the bench plan (max_batch 256) and batch sizes.

The reference of every image is the transform the reference's dataset runs, built from PIL and torchvision ops:
``T.Resize((224, 224))`` when the source is another size, ``ToTensor``, ``Normalize(IMAGENET_MEAN, IMAGENET_STD)``, then
the converted graph's own ``torch.quantize_per_tensor``.  From that quantised input, with every parameter read from the
converted module (``O.extract_qnet``), never from the engine's flattened description:

* stem accumulators: ``O.conv_acc`` in float64 over chunks of 32 images; stem output: ``O.requant``; pooled tensor:
  ``O.maxpool3x3s2``.  The front end is run alone through ``debug_frontend`` on the u8 images: the debug instantiation
  with the accumulator dump, and the product instantiation the forward would launch.  A failure names the first bad
  element (image, channel, y, x), the fraction that differs, and whether the accumulators or only the pooled bytes are
  wrong; for a wrong input it also names the input channel(s) whose lookup is wrong (``_input_channel_probe``);
* logits: the live fbgemm module ``gm(x)``.

Edge images (all 0 / all 255, pure R, G and B, a 0/255 checkerboard, a 255 frame two pixels wide and its inverse, and two
ramps that together hold every level of every channel) sit at the first, a middle and the last position of every batch of
9 or more.  The frames show whether out-of-image records hold the input zero point rather than ``LUT[c][0]``.
"""
import copy
import os
import re
import subprocess
import sys
import time

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from ievm_testutil import cached_quantized  # noqa: E402
from oracle import int8_forward as O  # noqa: E402
from oracle import model_factory as mf  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WIDTHS = {"w57": mf.PRUNED_WIDTHS, "w60": mf.DEFAULT_CFG_WIDTHS, "w64": mf.UNPRUNED_WIDTHS}
MEAN, STD = [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]
CHUNK = 32                   # images per float64 oracle stem
BENCH_PLAN = 256
CHANNEL_NAMES = "RGB"


# ------------------------------------------------------------------------------------------ inputs

def edge_images(h=224, w=224):
    z = np.zeros((h, w, 3), np.uint8)
    out = [z, z + 255]
    for c in range(3):
        im = z.copy()
        im[..., c] = 255
        out.append(im)
    yy, xx = np.mgrid[0:h, 0:w]
    out.append(np.repeat((((yy + xx) % 2) * 255).astype(np.uint8)[..., None], 3, axis=2))
    frame = np.zeros((h, w), np.uint8)
    frame[:2], frame[-2:], frame[:, :2], frame[:, -2:] = 255, 255, 255, 255
    out += [np.repeat(frame[..., None], 3, axis=2), np.repeat((255 - frame)[..., None], 3, axis=2)]
    off = np.array([0, 85, 170])
    out.append(((xx[..., None] + off) % 256).astype(np.uint8))           # levels off .. off + w - 1
    out.append(((yy[..., None] + w + off) % 256).astype(np.uint8))       # levels off + w .. off + w + h - 1
    return np.stack(out)


def edge_starts(n, k):
    return (0, n // 2 - k // 2, n - k) if n >= 9 else ()


def images(n, seed, h=224, w=224):
    """Seeded uniform u8 images; batches of 9 or more carry the edge images (as many as fit three times) at the first,
    a middle and the last position."""
    x = np.random.default_rng(seed).integers(0, 256, (n, h, w, 3), dtype=np.uint8)
    e = edge_images(h, w)
    k = min(len(e), n // 3)
    for s in edge_starts(n, k):
        x[s:s + k] = e[:k]
    return x


def reference_input(imgs):
    """f32 NCHW: the reference transform of every image, through PIL and torchvision."""
    from PIL import Image
    from torchvision import transforms as T
    ops = ([T.Resize((224, 224))] if imgs.shape[1:3] != (224, 224) else []) + [T.ToTensor(), T.Normalize(MEAN, STD)]
    tf = T.Compose(ops)
    return torch.stack([tf(Image.fromarray(im)) for im in imgs])


def reference_logits(gm, x):
    torch.backends.quantized.engine = "fbgemm"
    with torch.no_grad():
        return torch.cat([gm(x[s:s + 64]) for s in range(0, x.shape[0], 64)])


def quantised_input(qnet, x):
    """The converted graph's own op; O.quantize_input must agree with it."""
    xq = torch.quantize_per_tensor(x, qnet.in_scale, qnet.in_zp, torch.quint8).int_repr().numpy()
    oq = O.quantize_input(x.numpy(), qnet.in_scale, qnet.in_zp)
    assert np.array_equal(oq, xq), f"O.quantize_input differs from quantize_per_tensor on {int((oq != xq).sum())} values"
    return xq


def stem_reference(qnet, xq):
    """Generator of (start, accumulators, stem output, pooled) over chunks of CHUNK images."""
    s_ = qnet.stem
    for s in range(0, xq.shape[0], CHUNK):
        acc = O.conv_acc(xq[s:s + CHUNK], qnet.in_zp, s_.w, s_.stride, s_.pad)
        out = O.requant(acc, qnet.in_scale, s_.w_scale, s_.bias, s_.out_scale, s_.out_zp, s_.relu)
        yield s, acc, out, O.maxpool3x3s2(out)


# ------------------------------------------------------------------------------------------ the checker

class _Diff:
    """First differing element and the count of differing elements over a whole batch, chunk by chunk."""

    def __init__(self, name):
        self.name, self.bad, self.total, self.first = name, 0, 0, None

    def add(self, got, want, s):
        self.total += want.size
        bad = got != want
        cnt = int(bad.sum())
        if cnt and self.first is None:
            i, c, y, x = (int(v) for v in np.argwhere(bad)[0])
            self.first = (i + s, c, y, x, got[i, c, y, x], want[i, c, y, x])
        self.bad += cnt

    def text(self):
        i, c, y, x, g, w = self.first
        return (f"{self.name}: {self.bad} of {self.total} ({self.bad / self.total:.4%}) differ; first at image {i}, "
                f"channel {c}, y {y}, x {x}: engine {g} vs reference {w}")


def _input_channel_probe(eng, qnet, img):
    """Input channels whose lookup is wrong, from one failing image: for each channel c, the image with channel c kept
    and the other two set to a constant k, for k = 0 and k = 255.  A wrong entry (c*, v) fails both probes of c*, and a
    probe of another channel only when k = v in c*, which cannot hold for both k."""
    bad = []
    for c in range(3):
        fails = 0
        for k in (0, 255):
            p = np.full_like(img, k)
            p[..., c] = img[..., c]
            pooled, acc = eng.debug_frontend(torch.from_numpy(p[None]).cuda())
            _, ra, _, rp = next(stem_reference(qnet, quantised_input(qnet, reference_input(p[None]))))
            fails += int(not (np.array_equal(acc, ra) and np.array_equal(pooled, rp)))
        if fails == 2:
            bad.append(c)
    return bad


def check_front_end(eng, qnet, imgs, label="", cross_f32=True):
    """The u8 front end on ``imgs`` (u8 [n, 224, 224, 3]) against the reference, per tensor; raises AssertionError."""
    t0 = time.time()
    n = imgs.shape[0]
    x = reference_input(imgs)
    xq = quantised_input(qnet, x)
    dev = torch.from_numpy(imgs).cuda()
    pooled, acc = eng.debug_frontend(dev)                     # <I8, 1, false, true>: accumulators written out
    product, _ = eng.debug_frontend(dev, want_acc=False)      # the instantiation enqueue_forward launches
    d_acc, d_pool, d_prod = _Diff("stem accumulators"), _Diff("pooled tensor"), _Diff("pooled tensor (product kernel)")
    ref_pool = np.empty_like(pooled)
    for s, ra, _, rp in stem_reference(qnet, xq):
        e = s + ra.shape[0]
        d_acc.add(acc[s:e], ra, s)
        d_pool.add(pooled[s:e], rp, s)
        d_prod.add(product[s:e], rp, s)
        ref_pool[s:e] = rp
    del acc
    msgs = []
    if d_acc.bad:
        msgs.append("accumulators differ (input records: lookup table, TMA rows, zero-point borders, or the MMA): " +
                    d_acc.text())
    if d_pool.bad:
        msgs.append(("pooled bytes differ" + ("" if d_acc.bad else " with matching accumulators (epilogue, pool or "
                                                                    "store)")) + ": " + d_pool.text())
    if d_prod.bad:
        msgs.append(d_prod.text())
    if msgs:
        first = (d_acc.first or d_pool.first or d_prod.first)[0]
        chans = _input_channel_probe(eng, qnet, imgs[first])
        if chans:
            msgs.append("wrong lookup in input channel(s) " + ", ".join(f"{c} ({CHANNEL_NAMES[c]})" for c in chans))
        raise AssertionError(f"{label} n={n}: " + "; ".join(msgs))
    if cross_f32:        # the f32 product front end on the transformed batch writes the same bytes
        f32, _ = eng.debug_frontend(x.cuda(), want_acc=False)
        assert np.array_equal(f32, pooled), f"{label} n={n}: f32 and u8 front ends differ on {int((f32 != pooled).sum())} bytes"
    print(f"\n{label} n={n}: stem accumulators and pooled tensor bit-exact ({time.time() - t0:.1f} s)")
    return x, ref_pool


def _engine(gm, max_batch=BENCH_PLAN):
    import ievm_b200
    eng = ievm_b200.B200QuantizedResNet.from_converted(gm, max_batch=max_batch)
    eng.set_input_transform()
    return eng


# ------------------------------------------------------------------------------------------ front end, per tensor

@pytest.fixture(scope="module")
def bench_engine_w57():
    eng = _engine(cached_quantized(mf.PRUNED_WIDTHS))
    yield eng
    eng.close()


@pytest.mark.parametrize("n", [1, 2, 3, 5, 148, 251, 256])
def test_u8_front_end_bit_exact_on_the_bench_plan(n, bench_engine_w57):
    """n = 1, 2: every CTA's range of pooled rows inside one image (grid = min(56 n, SMs)); from 3 the ranges cross image
    boundaries; 251 is ragged, 256 the bench batch."""
    check_front_end(bench_engine_w57, O.extract_qnet(cached_quantized(mf.PRUNED_WIDTHS)), images(n, seed=300 + n), "w57")


@pytest.mark.parametrize("tpu", [1, 5, 56])
def test_u8_front_end_work_unit_sizes(tpu, monkeypatch):
    monkeypatch.setenv("IEVM_FRONT_TPU", str(tpu))
    gm = cached_quantized(mf.PRUNED_WIDTHS)
    eng = _engine(gm)
    try:
        check_front_end(eng, O.extract_qnet(gm), images(5, seed=320 + tpu), f"w57 tpu={tpu}")
    finally:
        eng.close()


@pytest.mark.parametrize("tag", ["w60", "w64"])
def test_u8_front_end_other_width_sets(tag):
    """w57 at 251 images is a case of the bench-plan test."""
    gm = cached_quantized(WIDTHS[tag])
    eng = _engine(gm)
    try:
        check_front_end(eng, O.extract_qnet(gm), images(251, seed=340), tag)
    finally:
        eng.close()


def test_edge_images_cover_every_level():
    e = edge_images()
    for c in range(3):
        assert len(np.unique(e[-2:, ..., c])) == 256
    assert (images(37, seed=0)[[0, 13, 27]] == e[[0, 0, 0]]).all()


# ------------------------------------------------------------------------------------------ qparam variants

_MINMAX = {}


def _minmax():
    if "m" not in _MINMAX:
        _MINMAX["m"] = mf.static_quantize_minmax(mf.make_student(mf.PRUNED_WIDTHS))
    return _MINMAX["m"]


def _set_attr(g, name, value):
    old = getattr(g, name)
    setattr(g, name, torch.tensor(value, dtype=old.dtype) if isinstance(old, torch.Tensor) else value)


def saturating_input(gm):
    """Input scale divided by 4, zero point 112 (R reaches 255 from 111 on, B reaches 0 up to 115): the lookup table
    clamps at both ends in every channel."""
    g = copy.deepcopy(gm)
    _set_attr(g, "conv1_input_scale_0", float(g.conv1_input_scale_0) / 4)
    _set_attr(g, "conv1_input_zero_point_0", 112)
    return g


def stem_zero_point_7(gm):
    """Stem output zero point 7: its ReLU clamps at 7, so the front end runs the general rounding instantiation."""
    g = copy.deepcopy(gm)
    dict(g.named_modules())["conv1"].zero_point = 7
    return g


@pytest.mark.parametrize("variant", ["minmax", "saturating", "stem_zp7"])
def test_u8_front_end_qparam_variants(variant):
    """The converted module itself is edited, so the lookup table, the oracle, the engine and fbgemm read the same
    definition.  Per tensor, then the logits against the live module."""
    import ievm_b200
    gm = {"minmax": _minmax, "saturating": lambda: saturating_input(cached_quantized(mf.PRUNED_WIDTHS)),
          "stem_zp7": lambda: stem_zero_point_7(cached_quantized(mf.PRUNED_WIDTHS))}[variant]()
    qnet = O.extract_qnet(gm)
    eng = ievm_b200.B200QuantizedResNet.from_converted(gm, max_batch=BENCH_PLAN)
    try:
        lut = eng.set_input_transform()
        if variant == "minmax":
            assert qnet.in_zp >= 100, qnet.in_zp          # full-range input observer: large input zero point
        if variant == "saturating":
            assert (lut.min(axis=1) == 0).all() and (lut.max(axis=1) == 255).all(), (lut.min(axis=1), lut.max(axis=1))
        if variant == "stem_zp7":
            assert eng.net.layers[0].out_zp == 7 and qnet.stem.out_zp == 7
        imgs = images(37, seed=360)
        x, _ = check_front_end(eng, qnet, imgs, variant)
        assert torch.equal(eng.forward_u8(torch.from_numpy(imgs).cuda()).cpu(), reference_logits(gm, x)), \
            f"{variant}: logits differ from the live module"
    finally:
        eng.close()


# ------------------------------------------------------------------------------------------ configurations (subprocesses)

def run_config(which):
    """Body of a configuration subprocess (knobs in its environment)."""
    gm = cached_quantized(mf.PRUNED_WIDTHS)
    eng = _engine(gm)
    try:
        imgs = images(64, seed=380)
        if which == "no_fast_round":
            x, _ = check_front_end(eng, O.extract_qnet(gm), imgs, "IEVM_FAST_ROUND=0")
            assert torch.equal(eng.forward_u8(torch.from_numpy(imgs).cuda()).cpu(), reference_logits(gm, x))
        else:
            with pytest.raises(RuntimeError, match="needs the fused front end"):
                eng.forward_u8(torch.from_numpy(imgs).cuda())
    finally:
        eng.close()


_CONFIG = r"""
import os, sys
sys.path.insert(0, sys.argv[1])
sys.path.insert(0, os.path.join(sys.argv[1], "tests"))
import test_gpu_u8_input as T
T.run_config(sys.argv[2])
print("config ok")
"""


@pytest.mark.parametrize("which,env", [("no_fast_round", {"IEVM_FAST_ROUND": "0"}),
                                       ("separate_front", {"IEVM_FUSED_FRONT": "0"})])
def test_u8_input_under_kernel_configurations(which, env, tmp_path):
    """IEVM_FAST_ROUND=0: the general rounding instantiation <I8, 1, false> on the default qconfig, bit-exact.
    IEVM_FUSED_FRONT=0: forward_u8 must refuse (the u8 input exists only in the fused front end), never return logits."""
    script = tmp_path / "config.py"
    script.write_text(_CONFIG)
    e = dict(os.environ)
    e.update(env)
    e["IEVM_VERBOSE"] = "1"
    r = subprocess.run([sys.executable, str(script), ROOT, which], env=e, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "config ok" in r.stdout, (r.stdout[-3000:], r.stderr[-3000:])
    if which == "no_fast_round":       # the knob is applied to every conv's plan, the stem's included
        flags = re.findall(r"fast_round=(\d)", r.stderr)
        assert flags and set(flags) == {"0"}, r.stderr[-2000:]


def test_u8_input_refused_with_keep_tensors(bench_engine_w57):
    eng = bench_engine_w57
    imgs = torch.from_numpy(images(2, seed=390))
    eng.set_option("keep_tensors", 1)
    try:
        for src in (imgs.cuda(), imgs):
            with pytest.raises(RuntimeError, match="needs the fused front end"):
                eng.forward_u8(src)
    finally:
        eng.set_option("keep_tensors", 0)


# ------------------------------------------------------------------------------------------ the checker's sensitivity

def _upload_lut(eng, lut):
    from ievm_b200 import _lib
    lut = np.ascontiguousarray(lut, dtype=np.uint8)
    _lib.check(eng._lib.ievm_set_input_lut(eng._handle, lut.ctypes.data), "ievm_set_input_lut")


@pytest.mark.parametrize("mutation", ["one_level", "r_b_swapped"])
def test_checker_catches_a_wrong_lookup_table(mutation):
    gm = cached_quantized(mf.PRUNED_WIDTHS)
    qnet = O.extract_qnet(gm)
    eng = _engine(gm, max_batch=8)
    try:
        lut = eng.set_input_transform().copy()
        if mutation == "one_level":
            lut[1, 128] += 1 if lut[1, 128] < 255 else -1
            pattern = r"input channel\(s\) 1 \(G\)$"
        else:
            lut = lut[[2, 1, 0]]
            pattern = r"accumulators differ"
        _upload_lut(eng, lut)
        with pytest.raises(AssertionError, match=pattern):
            check_front_end(eng, qnet, images(5, seed=400), mutation, cross_f32=False)
    finally:
        eng.close()


# ------------------------------------------------------------------------------------------ whole forward, production shapes

@pytest.mark.parametrize("src", [224, 200])
def test_whole_forward_at_the_bench_batch(src, bench_engine_w57):
    """256 images from device buffers (use_graph 0 and 1), 251 from host buffers (chunked copies), and evaluate_accuracy
    over a loader of pinned batches built as the bench builds it: logits identical to fbgemm on the reference transform,
    accuracy identical to the reference loop on the module."""
    import ievm_b200
    gm = cached_quantized(mf.PRUNED_WIDTHS)
    eng = bench_engine_w57
    imgs = images(256, seed=420 + src, h=src, w=src)
    ref = reference_logits(gm, reference_input(imgs))
    dev = torch.from_numpy(imgs).cuda()
    try:
        for g in (0, 1):
            eng.set_option("use_graph", g)
            for rep in range(2):                  # with graphs: capture, then replay
                assert torch.equal(eng.forward_u8(dev).cpu(), ref), f"{src}x{src} device buffers, use_graph={g}, call {rep}"
        eng.set_option("use_graph", 0)
        assert torch.equal(eng.forward_u8(torch.from_numpy(imgs[:251])), ref[:251]), f"{src}x{src} host buffers, n=251"
        labels = torch.randint(0, mf.NUM_CLASSES, (256,), generator=torch.Generator().manual_seed(src))
        loader = [(torch.from_numpy(imgs).pin_memory(), labels)] * 3
        want = 100.0 * int((torch.max(ref, 1)[1] == labels).sum()) / 256      # engines.py:61, every batch alike
        assert ievm_b200.evaluate_accuracy(eng, loader) == pytest.approx(want, abs=1e-9)
        if src == 224:                            # more images than max_batch: split into 256 + 44
            extra = np.ascontiguousarray(imgs[:44, :, ::-1])
            ref300 = torch.cat([ref, reference_logits(gm, reference_input(extra))])
            assert torch.equal(eng.forward_u8(torch.from_numpy(np.concatenate([imgs, extra])).cuda()).cpu(), ref300)
    finally:
        eng.set_option("use_graph", 0)


SIZE_SEQUENCE = [(200, 200), (300, 260), (200, 200), (224, 224), (200, 200)]


def test_source_size_changes_under_graphs_and_submit(bench_engine_w57):
    """One engine with use_graph = 1 fed a sequence of source sizes: every ievm_set_resize drops the graph cache, and a
    graph captured for one size must never replay for another.  Then submit() with the same sizes (the staging buffers
    grow), results read in reverse order."""
    gm = cached_quantized(mf.PRUNED_WIDTHS)
    eng = bench_engine_w57
    batches = [images(6, seed=440 + i, h=h, w=w) for i, (h, w) in enumerate(SIZE_SEQUENCE)]
    refs = [reference_logits(gm, reference_input(b)) for b in batches]
    eng.set_option("use_graph", 1)
    try:
        for (h, w), b, r in zip(SIZE_SEQUENCE, batches, refs):
            assert torch.equal(eng.forward_u8(torch.from_numpy(b).cuda()).cpu(), r), f"{h}x{w} under graphs"
    finally:
        eng.set_option("use_graph", 0)
    pend = [eng.submit(torch.from_numpy(b).pin_memory()) for b in batches]
    for i in reversed(range(len(pend))):
        assert torch.equal(pend[i].result(), refs[i]), f"submit {i} ({SIZE_SEQUENCE[i]})"
