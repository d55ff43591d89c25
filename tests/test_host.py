"""CPU tier: host-side logic, the C-ABI surface, and the sharding helpers (gloo, world size 2)."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

import ievm_b200
from ievm_b200 import _lib
from oracle import model_factory as mf
from ievm_testutil import RESIZE_SOURCES, ROOT, cached_quantized


def test_library_builds_and_exports_every_declared_symbol():
    path = _lib.build()
    lib = ctypes.CDLL(path)
    header = open(os.path.join(ROOT, "include", "ievm.h")).read()
    declared = set(re.findall(r"\b(ievm_[a-z0-9_]+)\s*\(", header))
    assert declared >= {"ievm_create", "ievm_forward_i8", "ievm_forward_f16", "ievm_destroy", "ievm_last_error"}
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/ievm.h but not exported"
    assert set(_lib.EXPORTS) == declared
    info = _lib.load().ievm_build_info().decode()
    assert "sm_100a" in info


def test_sass_contains_blackwell_instructions():
    out = subprocess.run(["cuobjdump", "-sass", _lib.build()], capture_output=True, text=True).stdout
    for mnemonic in ("UTCIMMA", "UTCHMMA", "UTMALDG.4D.IM2COL", "LDTM"):
        assert mnemonic in out, f"{mnemonic} missing from SASS"


def test_hot_kernels_do_not_spill():
    """The tensor-core kernels run at their register caps (96 for the conv kernels, 128 for the fused front end): a
    spill (STACK / LOCAL bytes in cuobjdump -res-usage) in any of them is a silent performance regression."""
    out = subprocess.run(["cuobjdump", "-res-usage", _lib.build()], capture_output=True, text=True).stdout
    found = 0
    lines = out.splitlines()
    for i, line in enumerate(lines):
        m = re.search(r"Function (\S+):", line)
        if not m or i + 1 >= len(lines):
            continue
        name, usage = m.group(1), lines[i + 1]
        if any(k in name for k in ("conv_tc_kernel", "frontend2_kernel", "head_i8_kernel", "head_f16_kernel")):
            found += 1
            # a handful of kernel-entry values (schedule bounds, ring pointers) may be parked on the stack of the shape-
            # specialised kernels -- reloaded once per warp role, never inside a tile loop; anything bigger is a real spill
            stack = int(re.search(r"STACK:(\d+)", usage).group(1))
            assert stack <= 48 and "LOCAL:0 " in usage, f"{name}: {usage.strip()}"
            regs = int(re.search(r"REG:(\d+)", usage).group(1))
            assert regs <= (128 if "frontend2" in name else 96), f"{name}: {regs} registers"
    assert found >= 23          # 18 conv_tc instantiations, 3 front ends, 2 heads


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_fallback():
    net = ievm_b200.from_converted(cached_quantized(mf.PRUNED_WIDTHS))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ievm_b200.B200QuantizedResNet(net)
    # and the C entry point itself refuses rather than degrading
    from ievm_b200.engine import _marshal
    nd, keep = _marshal(net)
    h = ctypes.c_void_p()
    rc = _lib.load().ievm_create(ctypes.byref(nd), 0, 8, ctypes.byref(h))
    assert rc == -3 and not h.value
    assert b"no CPU fallback" in _lib.load().ievm_last_error()


def test_flatten_converted_and_state_dict_agree():
    gm = cached_quantized(mf.PRUNED_WIDTHS)
    a = ievm_b200.from_converted(gm)
    b = ievm_b200.from_quantized_state_dict(gm.state_dict())
    assert a.tensor_names == b.tensor_names and len(a.layers) == len(b.layers) == 22
    for la, lb in zip(a.layers, b.layers):
        for f in la.__dataclass_fields__:
            va, vb = getattr(la, f), getattr(lb, f)
            if isinstance(va, np.ndarray):
                assert np.array_equal(va, vb), (la.name, f)
            else:
                assert va == vb, (la.name, f)
    assert a.conv_macs_per_image() == 1466823640          # SURVEY section 8(d): 1.4668 GMAC
    assert [L.cout for L in a.layers if L.op == 0][:2] == [57, 57]
    # every tensor-core layer's input zero point is 0 (TMA zero fill == real zero)
    assert all(L.in_zp == 0 for L in a.layers[1:] if L.op == 0)


def test_flatten_half_modules():
    s = ievm_b200.from_half_module(mf.cast_fp16(mf.make_student()))
    assert len(s.layers) == 22 and s.conv_macs_per_image() == 1466823640
    t = ievm_b200.from_half_module(mf.cast_fp16(mf.make_teacher()))
    assert sum(L.op == 0 for L in t.layers) == 53 and t.conv_macs_per_image() == 4087148544
    # BN folding is exact algebra: conv(x, w') + b' == bn(conv(x, w)) in fp32
    m = mf.make_student((16, 24, 32, 40))
    spec = ievm_b200.from_half_module(m)       # fp32 module: fold in fp32, weights rounded to fp16
    x = torch.randn(2, 3, 32, 32)
    ref = torch.relu(m.bn1(m.conv1(x)))
    got = torch.relu(torch.nn.functional.conv2d(x, torch.from_numpy(spec.layers[0].weight).float(), None, 2, 3)
                     + torch.from_numpy(spec.layers[0].bias).view(1, -1, 1, 1))
    assert torch.allclose(ref, got, atol=5e-3)


def test_input_lut_equals_the_reference_transform_pipeline():
    """SURVEY 8(f)-1: lut[c][v] must equal quantize_per_tensor(Normalize(ToTensor(v))) from the reference's own
    transform (quantization/dataset.py:14-19) for every level, so the fused u8 path is exact by construction."""
    from PIL import Image
    from torchvision import transforms as T
    gm = cached_quantized(mf.PRUNED_WIDTHS)
    scale, zp = float(gm.conv1_input_scale_0), int(gm.conv1_input_zero_point_0)
    lut = ievm_b200.input_lut(scale, zp)
    assert lut.shape == (3, 256) and lut.dtype == np.uint8
    img = np.random.default_rng(0).integers(0, 256, (224, 224, 3), dtype=np.uint8)
    img[0, :256 % 224] = 0
    img[1, :, :] = np.arange(224, dtype=np.uint8)[:, None]
    t = T.Compose([T.ToTensor(), T.Normalize(mean=[0.485, 0.456, 0.406], std=[0.229, 0.224, 0.225])])(Image.fromarray(img))
    q = torch.quantize_per_tensor(t, scale, zp, torch.quint8).int_repr().numpy()
    assert np.array_equal(q, np.stack([lut[c][img[..., c]] for c in range(3)]))


def test_resize_tables_equal_the_oracle_restatement():
    """The product's Pillow coefficient tables (host side of ievm_set_resize) against the oracle's restatement."""
    from oracle.pil_resize import precompute_coeffs
    sizes = {200, 224, 300, 97, 31, 500} | {v for hw in RESIZE_SOURCES for v in hw}
    for src in sorted(sizes):
        b, k = ievm_b200.pil_bilinear_coeffs(src, 224)
        bo, ko = precompute_coeffs(src, 224)
        assert np.array_equal(b, bo) and np.array_equal(k, ko), src


def test_on_disk_formats_are_recognised(tmp_path):
    """SURVEY 8(f)-2: widths and block kind recovered from tensor shapes; the rebuilt module reproduces the saved one."""
    from ievm_b200 import pipeline
    m = mf.make_student((24, 40, 56, 72))
    sd = {k: v.half() if v.is_floating_point() else v for k, v in m.state_dict().items()}      # model_fp16.pth layout
    assert pipeline._widths_from_float_state_dict(sd) == ("basic", [24, 40, 56, 72], 6)
    rebuilt = pipeline._module_from_float_state_dict(sd)
    x = torch.randn(2, 3, 64, 64)
    with torch.no_grad():
        assert torch.allclose(rebuilt(x), m.half().float()(x), atol=1e-5)
    assert pipeline._widths_from_float_state_dict(mf.make_teacher().state_dict())[0] == "bottleneck"
    with pytest.raises(ValueError):
        pipeline.load_engine({"foo": torch.zeros(1)})
    with pytest.raises(TypeError):
        pipeline.load_engine(3.14)


def test_engine_blob_round_trips_exactly(tmp_path):
    """SURVEY 8(f)-2 export: NetSpec -> .npz -> NetSpec is the identity (every scalar, every array and its dtype), for
    the INT8 and the FP16 network; load_engine dispatches a .npz path to the engine constructor."""
    from ievm_b200 import pipeline
    specs = [ievm_b200.from_converted(cached_quantized(mf.PRUNED_WIDTHS)),
             ievm_b200.from_half_module(mf.cast_fp16(mf.make_student((24, 40, 56, 72))))]
    for i, a in enumerate(specs):
        path = tmp_path / f"net{i}.npz"
        pipeline.save_engine(a, path)
        b = ievm_b200.NetSpec.load(path)
        assert (a.dtype, a.in_c, a.in_h, a.in_w, a.num_classes, a.in_scale, a.in_zp, a.tensor_names) == \
               (b.dtype, b.in_c, b.in_h, b.in_w, b.num_classes, b.in_scale, b.in_zp, b.tensor_names)
        assert len(a.layers) == len(b.layers)
        for la, lb in zip(a.layers, b.layers):
            for f in la.__dataclass_fields__:
                va, vb = getattr(la, f), getattr(lb, f)
                if isinstance(va, np.ndarray):
                    assert va.dtype == vb.dtype and np.array_equal(va, vb), (la.name, f)
                else:
                    assert va == vb and type(va) is type(vb), (la.name, f)
        if not torch.cuda.is_available():
            with pytest.raises(RuntimeError, match="no CPU fallback"):     # reached the engine constructor
                pipeline.load_engine(str(path))
    bad = tmp_path / "bad.npz"
    np.savez(bad, header=np.frombuffer(b'{"format": "other"}', dtype=np.uint8))
    with pytest.raises(ValueError, match="not an ievm NetSpec blob"):
        ievm_b200.NetSpec.load(bad)


def test_unsupported_graphs_fail_loudly():
    net = ievm_b200.from_converted(cached_quantized(mf.PRUNED_WIDTHS))
    import copy
    bad = copy.deepcopy(net)
    bad.layers[2].in_tensor = 17            # consumes a tensor produced later
    from ievm_b200.netdesc import _check_order
    with pytest.raises(ValueError):
        _check_order(bad)


_WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
import bench
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:%s" % sys.argv[2], rank=int(sys.argv[3]), world_size=2)
rank = dist.get_rank()
lo, hi = bench.shard_bounds(10, rank, 2)
full = torch.arange(60, dtype=torch.float32).view(10, 6)
gathered = bench.gather_logits(full[lo:hi], 10, rank, 2)
ms = bench.max_over_ranks(float(rank + 1), torch.device("cpu"))
if rank == 0:
    assert torch.equal(gathered, full), gathered
assert ms == 2.0
dist.barrier()
dist.destroy_process_group()
print("ok", rank)
'''


def test_sharding_helpers_world_size_2_gloo(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    port = str(29500 + os.getpid() % 1000)
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, port, str(r)], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=180)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o


def test_bench_work_model_matches_the_survey():
    """bench.py's per-launch work table (the roofline's numerator) reproduces SURVEY 8(d): 1.4668 GMAC and -- with the
    fused front end as ONE row -- 4.80 MB of compulsory HBM traffic per image for the pruned INT8 net; the network
    roofline is the sum of per-launch max(compute, HBM) times: 273 us at batch 256 with 2 x burst bf16 and the
    measured copy bandwidth."""
    import bench
    net = ievm_b200.from_converted(cached_quantized(mf.PRUNED_WIDTHS))
    rows = bench.layer_table(net, 1)
    names = [r[0] for r in rows]
    assert names[0] == "conv1" and names[-1] == "fc" and len(rows) == 21      # one row per launch of the product engine
    assert sum(m for _, m, _ in rows) == 1466823640                 # SURVEY 8(d): 20 convs + the 460 x 6 fc
    unfused = bench.layer_table(net, 1, fused_front=False)
    assert [r[0] for r in unfused][:3] == ["quantize_input", "conv1", "maxpool"] and len(unfused) == 23
    rows256 = bench.layer_table(net, 256)
    per_image = sum(b for _, _, b in rows256) / 256
    assert 4.78e6 < per_image < 4.90e6, per_image                   # 4.80 MB/img + 9.0 MB of weights per batch
    ms = bench.network_roofline_ms(rows256, 2 * 1677.3, 6545.3)
    expect = 1e3 * sum(max(2 * m / (2 * 1677.3e12), b / 6545.3e9) for _, m, b in rows256)
    assert ms == pytest.approx(expect)
    assert 0.265 < ms < 0.285, ms                                   # SURVEY 8(d): 273 us
    lo, hi = bench.shard_bounds(1024, 3, 8)
    assert (lo, hi) == (384, 512)
