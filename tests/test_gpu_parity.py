"""GPU tier (-m gpu): the CUDA engine, called through the C ABI, against the CPU oracle, the golden
fixtures recorded from the reference's own engine, and size-independent properties at full batch.

Bars (BASELINE.json north_star): int32 accumulators bit-exact; requantised activations within +-1 LSB
(we assert bit-exact); INT8 logits identical => top-1 agreement 100 % (lowest index on ties);
FP16 logits within 1e-2 row-relative of the reference's ``.half()`` path.
"""
import ctypes
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from ievm_testutil import RESIZE_SOURCES, cached_quantized  # noqa: E402
from oracle import int8_forward as O  # noqa: E402
from oracle import model_factory as mf  # noqa: E402

WIDTHS = {"w57": mf.PRUNED_WIDTHS, "w60": mf.DEFAULT_CFG_WIDTHS, "w64": mf.UNPRUNED_WIDTHS}
FP16_REL_TOL = 1e-2     # north_star: "FP16 logits within 1e-2 relative" (row-normalised, SURVEY 8c)


def _engine(widths, **kw):
    import ievm_b200
    return ievm_b200.B200QuantizedResNet.from_converted(cached_quantized(widths), **kw)


def _row_rel(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return (np.abs(a - b).max(axis=1) / np.maximum(np.abs(b).max(axis=1), 1.0)).max()


# ------------------------------------------------------------------------------------------ TMA probe

def _swizzle(tile, kc):
    """[128, kc] row-major bytes -> the raw shared-memory image TMA writes (16-byte chunk XOR)."""
    rows, chunks = tile.shape[0], kc // 16
    t = tile.reshape(rows, chunks, 16)
    out = np.empty_like(t)
    for r in range(rows):
        x = (r % 8) if kc == 128 else ((r // 2) % 4)
        for j in range(chunks):
            out[r, j ^ x] = t[r, j]
    return out.reshape(rows, kc)


def _swizzle_rows(rows, kc):
    """Same XOR pattern for an arbitrary number of rows (swizzle follows the row's address bits)."""
    n, chunks = rows.shape[0], kc // 16
    t = rows.reshape(n, chunks, 16)
    out = np.empty_like(t)
    for r in range(n):
        x = (r % 8) if kc == 128 else ((r // 2) % 4)
        for j in range(chunks):
            out[r, j ^ x] = t[r, j]
    return out.reshape(n, kc)


def _expected_im2col(x, ksize, stride, pad, kc, m0, tx, ty, c0):
    n, h, w, cp = x.shape
    ho, wo = (h + 2 * pad - ksize) // stride + 1, (w + 2 * pad - ksize) // stride + 1
    tile = np.zeros((128, kc), np.uint8)
    for r in range(128):
        m = m0 + r
        if m >= n * ho * wo:
            continue
        img, rem = divmod(m, ho * wo)
        oy, ox = divmod(rem, wo)
        iy, ix = oy * stride - pad + ty, ox * stride - pad + tx
        if 0 <= iy < h and 0 <= ix < w:
            seg = x[img, iy, ix, c0:c0 + kc]
            tile[r, :len(seg)] = seg
    return tile


@pytest.mark.parametrize("case", [
    dict(n=2, h=56, w=56, cp=64, k=3, s=1, p=1, kc=64, m0=0, tx=0, ty=0, c0=0),
    dict(n=2, h=56, w=56, cp=64, k=3, s=1, p=1, kc=64, m0=3072, tx=2, ty=2, c0=0),       # crosses an image boundary
    dict(n=2, h=28, w=28, cp=128, k=3, s=1, p=1, kc=128, m0=128, tx=1, ty=0, c0=0),
    dict(n=2, h=56, w=56, cp=64, k=3, s=2, p=1, kc=64, m0=640, tx=0, ty=1, c0=0),        # stride 2
    dict(n=2, h=28, w=28, cp=128, k=1, s=2, p=0, kc=128, m0=256, tx=0, ty=0, c0=0),      # 1x1 downsample, ragged end
    dict(n=3, h=7, w=7, cp=480, k=3, s=1, p=1, kc=128, m0=128, tx=2, ty=1, c0=384),      # partial channel chunk + past the last image
])
def test_tma_im2col_semantics(case):
    from ievm_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(0)
    x = rng.integers(1, 255, size=(case["n"], case["h"], case["w"], case["cp"]), dtype=np.uint8)
    xd = torch.from_numpy(x).cuda()
    out = torch.zeros(128 * case["kc"], dtype=torch.uint8, device="cuda")
    _lib.check(lib.ievm_probe_im2col(xd.data_ptr(), case["n"], case["h"], case["w"], case["cp"], case["k"], case["s"],
                                     case["p"], case["kc"], case["m0"], case["tx"], case["ty"], case["c0"],
                                     out.data_ptr()), "probe")
    got = out.cpu().numpy().reshape(128, case["kc"])
    exp = _expected_im2col(x, case["k"], case["s"], case["p"], case["kc"], case["m0"], case["tx"], case["ty"], case["c0"])
    raw = _swizzle(exp, case["kc"])
    if not np.array_equal(got, raw):
        same_rows = np.array_equal(np.sort(got, axis=1), np.sort(raw, axis=1))
        pytest.fail(f"im2col tile mismatch (rows match up to chunk order: {same_rows}); "
                    f"first bad row {int(np.argmax((got != raw).any(axis=1)))}")


# ------------------------------------------------------------------------------------------ INT8 parity

@pytest.mark.parametrize("tag", ["w57", "w60", "w64"])
def test_int8_logits_match_reference_golden(tag, golden_dir):
    g = np.load(os.path.join(golden_dir, f"int8_{tag}.npz"))
    eng = _engine(WIDTHS[tag], max_batch=8)
    x = mf.synthetic_images(int(g["n_images"])).cuda()
    y = eng(x).cpu().numpy()
    assert np.array_equal(y, g["logits"]), f"max |diff| = {np.abs(y - g['logits']).max()}"
    eng.close()


def test_int8_every_tensor_and_accumulator_bit_exact():
    gm = cached_quantized(mf.PRUNED_WIDTHS)
    net = O.extract_qnet(gm)
    eng = _engine(mf.PRUNED_WIDTHS, max_batch=4)
    eng.set_option("keep_tensors", 1)
    x = mf.synthetic_images(3, seed=21)
    y = eng(x.cuda()).cpu().numpy()
    yo = O.forward(net, x.numpy(), keep=True)
    checked = 0
    for tid, name in sorted(eng.net.tensor_names.items()):
        if name in net.trace:
            got = eng.read_tensor(tid)
            assert np.array_equal(got, net.trace[name]), f"tensor {name}: {(got != net.trace[name]).mean():.3%} bytes differ"
            checked += 1
    assert checked == 22
    for L in eng.net.layers[2:-1]:
        if L.op == 0:
            acc = eng.conv_accumulators(L.name, 3)
            assert np.array_equal(acc, net.trace[L.name + ":acc"]), f"accumulators of {L.name} differ"
    assert np.array_equal(y, yo)
    eng.close()


@pytest.mark.parametrize("n,tpu", [(3, 0), (2, 5), (1, 56), (5, 1)])
def test_int8_fused_front_end_accumulators_and_pooled_tensor(n, tpu, monkeypatch):
    """frontend_v2.cuh alone (quantize + record build + stacked-row tcgen05 stem + pool in registers): stem
    accumulators and the pooled tensor bit-identical to the oracle, for several work-unit sizes (tpu = pooled
    rows per unit: exercises the warm-up tile, ragged last units and whole-image units)."""
    if tpu:
        monkeypatch.setenv("IEVM_FRONT_TPU", str(tpu))
    gm = cached_quantized(mf.PRUNED_WIDTHS)
    net = O.extract_qnet(gm)
    eng = _engine(mf.PRUNED_WIDTHS, max_batch=8)
    x = mf.synthetic_images(n, seed=40 + n)
    x[0, :, :5, :7] = 1e4       # saturating inputs in a corner
    x[-1, :, -3:, -9:] = -1e4
    pooled, acc = eng.debug_frontend(x.cuda())
    O.forward(net, x.numpy(), keep=True)
    assert np.array_equal(acc, net.trace["conv1:acc"]), \
        f"stem accumulators: {(acc != net.trace['conv1:acc']).mean():.3%} differ"
    assert np.array_equal(pooled, net.trace["maxpool"]), \
        f"pooled tensor: {(pooled != net.trace['maxpool']).mean():.3%} bytes differ"
    # without the accumulator dump the PRODUCT instantiation runs (magic-number rounding, no debug code in its loop)
    pooled_product, _ = eng.debug_frontend(x.cuda(), want_acc=False)
    assert np.array_equal(pooled_product, net.trace["maxpool"])
    eng.close()


@pytest.mark.parametrize("n", [1, 6])
def test_int8_u8_image_input_is_bit_identical_to_the_f32_pipeline(n):
    """SURVEY 8(f)-1: decoded u8 HWC images through the fused ToTensor+Normalize+quantize front end == the
    reference's transform (quantization/dataset.py:14-19) followed by the converted module on the CPU."""
    from PIL import Image
    from torchvision import transforms as T
    gm = cached_quantized(mf.PRUNED_WIDTHS)
    torch.backends.quantized.engine = "fbgemm"
    eng = _engine(mf.PRUNED_WIDTHS, max_batch=8)
    rng = np.random.default_rng(50 + n)
    imgs = rng.integers(0, 256, (n, 224, 224, 3), dtype=np.uint8)
    imgs[0, :3] = 255
    imgs[-1, -2:, -5:] = 0
    tf = T.Compose([T.ToTensor(), T.Normalize(mean=[0.485, 0.456, 0.406], std=[0.229, 0.224, 0.225])])
    x = torch.stack([tf(Image.fromarray(im)) for im in imgs])
    with torch.no_grad():
        ref = gm(x)
    u8 = torch.from_numpy(imgs)
    assert torch.equal(eng.forward_u8(u8.cuda()).cpu(), ref)          # device buffers
    assert torch.equal(eng.forward_u8(u8), ref)                       # host buffers (H2D of a quarter of the bytes)
    assert torch.equal(eng(x.cuda()).cpu(), ref)
    eng.close()


@pytest.mark.parametrize("hw", RESIZE_SOURCES)
def test_int8_resize_stage_and_full_transform_are_bit_identical(hw):
    """SURVEY 8(f)-1 complete: Resize (Pillow bilinear) + ToTensor + Normalize + quantize on the GPU == the reference's
    transform (quantization/dataset.py:14-19) on PIL images followed by the converted module on the CPU."""
    from PIL import Image
    from torchvision import transforms as T
    from oracle.pil_resize import resize_bilinear_u8
    gm = cached_quantized(mf.PRUNED_WIDTHS)
    torch.backends.quantized.engine = "fbgemm"
    eng = _engine(mf.PRUNED_WIDTHS, max_batch=8)
    rng = np.random.default_rng(hw[0])
    imgs = rng.integers(0, 256, (2 if hw[0] * hw[1] > 1000000 else 3,) + hw + (3,), dtype=np.uint8)
    u8 = torch.from_numpy(imgs)
    resized = eng.debug_resize(u8.cuda())
    pil = np.stack([np.asarray(Image.fromarray(im).resize((224, 224), Image.BILINEAR)) for im in imgs])
    assert np.array_equal(resized, pil), f"{(resized != pil).mean():.3%} bytes differ from PIL"
    assert np.array_equal(resized, resize_bilinear_u8(imgs, 224, 224))
    tf = T.Compose([T.Resize((224, 224)), T.ToTensor(), T.Normalize(mean=[0.485, 0.456, 0.406], std=[0.229, 0.224, 0.225])])
    x = torch.stack([tf(Image.fromarray(im)) for im in imgs])
    with torch.no_grad():
        ref = gm(x)
    assert torch.equal(eng.forward_u8(u8.cuda()).cpu(), ref)
    assert torch.equal(eng.forward_u8(u8), ref)                       # host buffers
    eng.close()


def test_engines_from_on_disk_artifacts_and_eval_drop_ins(tmp_path):
    """SURVEY 8(f)-2/3: engines built from the files the reference writes; evaluate_accuracy / measure_latency
    drop-ins agree with the reference's own helpers run on the CPU module."""
    import ievm_b200
    gm = cached_quantized(mf.PRUNED_WIDTHS)
    torch.save(gm.state_dict(), tmp_path / "model_static_int8.pth")                   # quantization/main.py:306-308
    student = mf.make_student(mf.PRUNED_WIDTHS)
    torch.save(student, tmp_path / "pruned_model.pth")                                # pruning/main.py:164-165
    torch.save(mf.cast_fp16(student).state_dict(), tmp_path / "model_fp16.pth")
    e8 = ievm_b200.load_engine(str(tmp_path / "model_static_int8.pth"), max_batch=16)
    e16a = ievm_b200.load_engine(str(tmp_path / "pruned_model.pth"), max_batch=16)
    e16b = ievm_b200.load_engine(str(tmp_path / "model_fp16.pth"), max_batch=16)
    assert isinstance(e8, ievm_b200.B200QuantizedResNet) and isinstance(e16a, ievm_b200.B200HalfResNet)
    x = mf.synthetic_images(16, seed=3)
    torch.backends.quantized.engine = "fbgemm"
    with torch.no_grad():
        ref = gm(x)
    assert torch.equal(e8(x.cuda()).cpu(), ref)
    assert torch.equal(e16a(x.half().cuda()), e16b(x.half().cuda()))
    # evaluate_accuracy: same number as the reference's loop (engines.py:37-65) on the CPU module
    labels = torch.randint(0, 6, (48,), generator=torch.Generator().manual_seed(4))
    xs = mf.synthetic_images(48, seed=8)
    loader = [(xs[i:i + 16], labels[i:i + 16]) for i in range(0, 48, 16)]
    with torch.no_grad():
        pred = torch.cat([torch.max(gm(b), 1)[1] for b, _ in loader])
    ref_acc = 100 * int((pred == labels).sum()) / 48
    assert ievm_b200.evaluate_accuracy(e8, loader) == pytest.approx(ref_acc)
    acc16 = ievm_b200.evaluate_accuracy(e16a, loader)
    assert 0.0 <= acc16 <= 100.0
    ms = ievm_b200.measure_latency(e8, xs[:1], num_runs=20)
    assert 0.0 < ms < 50.0
    for e in (e8, e16a, e16b):
        e.close()


@pytest.mark.parametrize("n", [1, 2, 5, 13])
def test_int8_ragged_batches(n):
    gm = cached_quantized(mf.PRUNED_WIDTHS)
    eng = _engine(mf.PRUNED_WIDTHS, max_batch=16)
    x = mf.synthetic_images(n, seed=30 + n)
    y = eng(x.cuda()).cpu().numpy()
    assert np.array_equal(y, O.forward(O.extract_qnet(gm), x.numpy()))
    eng.close()


def test_int8_edge_batches_and_argument_errors():
    """Empty batch, a batch larger than max_batch (split by the wrapper), and the loud failures of the boundary:
    wrong dtype / shape raise, the C entry points return an error status instead of touching memory."""
    from ievm_b200 import _lib
    gm = cached_quantized(mf.PRUNED_WIDTHS)
    torch.backends.quantized.engine = "fbgemm"
    eng = _engine(mf.PRUNED_WIDTHS, max_batch=4)
    x = mf.synthetic_images(11, seed=60)
    assert tuple(eng(x[:0].cuda()).shape) == (0, 6) and tuple(eng(x[:0]).shape) == (0, 6)
    with torch.no_grad():
        ref = gm(x)
    assert torch.equal(eng(x.cuda()).cpu(), ref)                # 11 > max_batch = 4: 4 + 4 + 3
    assert torch.equal(eng(x), ref)
    with pytest.raises(TypeError):
        eng(x.half().cuda())
    with pytest.raises(ValueError):
        eng(x[:, :, :200].cuda())
    with pytest.raises(ValueError):
        eng.forward_u8(torch.zeros(2, 3, 224, 224, dtype=torch.uint8))
    lib = _lib.load()
    out = torch.empty(5, 6, device="cuda")
    assert lib.ievm_forward_i8(eng._handle, x.cuda().data_ptr(), 5, out.data_ptr(), None) < 0      # 5 > max_batch
    assert b"outside" in lib.ievm_last_error()
    assert lib.ievm_forward_f16(eng._handle, x.cuda().data_ptr(), 1, out.data_ptr(), None) < 0     # wrong entry point
    eng.close()


def test_int8_tensor_core_equals_direct_conv_at_batch_64():
    eng = _engine(mf.PRUNED_WIDTHS, max_batch=64)
    x = mf.synthetic_images(64, seed=5).cuda()
    y_tc = eng(x).clone()
    eng.set_option("conv_impl", 1)
    y_ref = eng(x)
    assert torch.equal(y_tc, y_ref)
    eng.close()


def test_int8_host_path_graph_path_and_state_dict_path_agree():
    import ievm_b200
    gm = cached_quantized(mf.PRUNED_WIDTHS)
    eng = _engine(mf.PRUNED_WIDTHS, max_batch=8)
    x = mf.synthetic_images(8, seed=9)
    y_dev = eng(x.cuda()).cpu()
    y_host = eng(x)                       # CPU tensor in -> H2D/D2H inside the C call
    assert not y_host.is_cuda and torch.equal(y_dev, y_host)
    eng.set_option("use_graph", 1)
    xd = x.cuda()
    y_g1 = eng(xd).cpu()
    y_g2 = eng(xd).cpu()
    assert torch.equal(y_dev, y_g1) and torch.equal(y_dev, y_g2)
    eng2 = ievm_b200.B200QuantizedResNet.from_quantized_state_dict(gm.state_dict(), max_batch=8)
    assert torch.equal(y_dev, eng2(x.cuda()).cpu())
    # nn.Module protocol the reference's callers rely on (engines.py:19-20,41-47; utils.py:124)
    assert eng.eval() is eng and next(eng.parameters()).dtype == torch.float32
    assert set(eng.state_dict().keys()) == set(gm.state_dict().keys())
    eng.close()
    eng2.close()


def test_int8_top1_agreement_4096_images_vs_cpu_fbgemm():
    gm = cached_quantized(mf.PRUNED_WIDTHS)
    torch.backends.quantized.engine = "fbgemm"
    eng = _engine(mf.PRUNED_WIDTHS, max_batch=256)
    agree = total = exact = 0
    for chunk in range(16):
        x = mf.synthetic_images(256, seed=1000 + chunk)
        with torch.no_grad():
            ref = gm(x)
        got = eng(x.cuda()).cpu()
        exact += int(torch.equal(ref, got))
        agree += int((torch.max(ref, 1)[1] == torch.max(got, 1)[1]).sum())    # lowest index on ties, both sides
        total += 256
    assert agree / total >= 0.999, f"top-1 agreement {agree}/{total}"
    assert exact == 16, f"only {exact}/16 chunks had bit-identical logits"
    eng.close()


def test_batch_sharding_is_bitwise_invariant():
    """Data-parallel property: logits of a batch do not depend on how it is split across ranks."""
    eng = _engine(mf.PRUNED_WIDTHS, max_batch=32)
    x = mf.synthetic_images(32, seed=77).cuda()
    whole = eng(x).clone()
    parts = torch.cat([eng(x[i:i + 8]).clone() for i in range(0, 32, 8)])
    assert torch.equal(whole, parts)
    eng.close()


def test_int8_batch_size_invariance_up_to_1024():
    """Size-independent property at full batch sizes: an image's logits do not depend on the batch it rides in
    (ragged M tiles, tile-width heuristic, fused front-end strips, halo tiles all change with N)."""
    eng = _engine(mf.PRUNED_WIDTHS, max_batch=1024)
    x = mf.synthetic_images(1024, seed=99).cuda()
    full = eng(x).clone()
    for n in (1, 3, 64, 255, 256, 777):
        assert torch.equal(eng(x[:n]), full[:n]), f"batch {n} differs from batch 1024"
    # and against the CPU fbgemm module on a slice
    gm = cached_quantized(mf.PRUNED_WIDTHS)
    torch.backends.quantized.engine = "fbgemm"
    with torch.no_grad():
        ref = gm(x[1000:1024].cpu())
    assert torch.equal(full[1000:1024].cpu(), ref)
    eng.close()


@pytest.mark.parametrize("case", [
    dict(h=56, w=56, cp=64, rb=64, bw=58, bh=6, w0=-1, h0=-1),
    dict(h=28, w=28, cp=128, rb=128, bw=30, bh=8, w0=-1, h0=3),
    dict(h=56, w=56, cp=64, rb=128, bw=58, bh=6, w0=-1, h0=53),      # channel over-read + past the bottom edge
])
def test_tma_halo_patch_layout(case):
    """The halo-mode convolution relies on a tiled 4-D TMA box landing as a swizzled *linear* run of pixels with
    zero-filled borders (ievm_probe_patch)."""
    from ievm_b200 import _lib
    lib = _lib.load()
    rng = np.random.default_rng(1)
    h, w, cp, rb, bw, bh, w0, h0 = (case[k] for k in ("h", "w", "cp", "rb", "bw", "bh", "w0", "h0"))
    x = rng.integers(1, 255, size=(2, h, w, cp), dtype=np.uint8)
    xd = torch.from_numpy(x).cuda()
    out = torch.zeros(bw * bh * rb, dtype=torch.uint8, device="cuda")
    _lib.check(lib.ievm_probe_patch(xd.data_ptr(), 2, h, w, cp, rb, 1, w0, h0, bw, bh, out.data_ptr()), "probe_patch")
    got = out.cpu().numpy().reshape(bh * bw, rb)
    exp = np.zeros((bh, bw, rb), np.uint8)
    for r in range(bh):
        for c in range(bw):
            iy, ix = h0 + r, w0 + c
            if 0 <= iy < h and 0 <= ix < w:
                exp[r, c, :min(cp, rb)] = x[1, iy, ix, :rb]
    assert np.array_equal(got, _swizzle_rows(exp.reshape(bh * bw, rb), rb))


# ------------------------------------------------------------------------------------------ FP16 parity

def test_fp16_student_matches_reference_half_path(golden_dir):
    import ievm_b200
    g = np.load(os.path.join(golden_dir, "fp16_w57.npz"))
    m16 = mf.cast_fp16(mf.make_student(mf.PRUNED_WIDTHS))
    eng = ievm_b200.B200HalfResNet.from_half_module(m16, max_batch=8)
    x = mf.synthetic_images(int(g["n_images"])).half()
    y = eng(x.cuda()).float().cpu().numpy()
    assert _row_rel(y, g["logits_fp16"]) < FP16_REL_TOL      # reference .half() on CPU (fixture)
    assert _row_rel(y, g["logits_fp32"]) < FP16_REL_TOL
    with torch.no_grad():                                      # reference .half() on this GPU (cuDNN)
        y_cudnn = m16.cuda()(x.cuda()).float().cpu().numpy()
    assert _row_rel(y, y_cudnn) < FP16_REL_TOL
    assert (y.argmax(1) == y_cudnn.argmax(1)).all()
    assert next(eng.parameters()).dtype == torch.float16
    eng.set_option("conv_impl", 1)
    y_direct = eng(x.cuda()).float().cpu().numpy()
    assert _row_rel(y, y_direct) < 2e-3
    eng.close()


def test_fp16_fused_front_end_matches_torch():
    """frontend_v2.cuh, FP16 flavour: conv1 + folded bn1 + ReLU + maxpool against the same modules in fp32."""
    import ievm_b200
    m16 = mf.cast_fp16(mf.make_student(mf.PRUNED_WIDTHS))
    eng = ievm_b200.B200HalfResNet.from_half_module(m16, max_batch=4)
    x = mf.synthetic_images(3, seed=11).half()
    pooled, _ = eng.debug_frontend(x.cuda(), want_acc=False)
    m32 = mf.cast_fp16(mf.make_student(mf.PRUNED_WIDTHS)).float()
    with torch.no_grad():
        ref = m32.maxpool(m32.relu(m32.bn1(m32.conv1(x.float())))).numpy()
    err = np.abs(pooled.astype(np.float32) - ref).max() / max(np.abs(ref).max(), 1.0)
    assert err < 5e-3, f"fp16 front end off by {err}"
    eng.close()


def test_fp16_teacher_resnet50_matches_reference_half_path(golden_dir):
    import ievm_b200
    g = np.load(os.path.join(golden_dir, "fp16_teacher_r50.npz"))
    m16 = mf.cast_fp16(mf.make_teacher())
    eng = ievm_b200.B200HalfResNet.from_half_module(m16, max_batch=4)
    x = mf.synthetic_images(int(g["n_images"])).half()
    y = eng(x.cuda()).float().cpu().numpy()
    assert _row_rel(y, g["logits_fp16"]) < FP16_REL_TOL
    with torch.no_grad():
        y_cudnn = m16.cuda()(x.cuda()).float().cpu().numpy()
    assert _row_rel(y, y_cudnn) < FP16_REL_TOL
    eng.close()


def test_kd_eval_loss_matches_torch():
    import ievm_b200
    g = torch.Generator().manual_seed(3)
    s = torch.randn(512, 6, generator=g) * 3
    t = torch.randn(512, 6, generator=g) * 3
    y = torch.randint(0, 6, (512,), generator=g)
    out = ievm_b200.kd_eval_loss(s.cuda(), t.cuda(), y.cuda(), alpha=0.5, temperature=4.0).cpu()
    T = 4.0   # knowledge_distillation/train.py:47-57
    ce = torch.nn.functional.cross_entropy(s, y)
    kd = torch.nn.KLDivLoss(reduction="batchmean")(torch.log_softmax(s / T, 1), torch.softmax(t / T, 1)) * T * T
    assert abs(out[1] - ce) < 1e-4 and abs(out[2] - kd) < 1e-4
    assert abs(out[0] - (0.5 * ce + 0.5 * kd)) < 1e-4
    assert int(out[3]) == int((s.argmax(1) == y).sum())
