"""GPU tier: the INT8 engine layer by layer against the integer oracle (oracle/int8_forward.py), bit for bit, at the
production tile plan (max_batch 256, the bench plan) and batch sizes, and under every kernel configuration.

The logits alone are a weak check: each is a requantised fc over a 7x7 average of the last tensor, so a wrong tile in an
early layer can be averaged and rounded away.  Here every tensor of every image is compared:

* stem: the quantised input, the tensor-core stem's accumulators (``conv_accumulators("conv1")``) and u8 output, the
  max-pool, and the product front end (``debug_frontend``: accumulators, pooled tensor, and the instantiation without
  the accumulator dump);
* every conv: the forward's output tensor against the oracle's (for a block's conv2 that is ``add_relu(requant(acc),
  residual)``), read before any accumulator dump re-runs the launch (a dual launch rewrites both of its outputs, so
  both are read first), then ``conv_accumulators`` against ``O.conv_acc``.  Matching accumulators with a wrong output
  put the fault in the epilogue or the store; wrong accumulators put it in the operand path.  The first bad element is
  named as (image, channel, y, x) with its M tile, ``m // 128``: scheduling bugs show up as tiles;
* head: the logits of the keep_tensors forward against avgpool + fc + requant + dequant on the engine's last tensor,
  the product configuration (keep_tensors = 0: fused front end, shared workspace) identical, and the live fbgemm module.

The reference walks the oracle chain one conv at a time over chunks of images: ``O.forward(keep=True)`` holds about
12 MB per image.  Its parameters come from ``O.extract_qnet`` of the converted module, matched by layer name, never
from the engine's flattened description, so a flattening bug cannot cancel itself out.

Kernel configurations (environment knobs, read when an engine is created) run in subprocesses and compare SHA-256
digests of every image of every tensor with those of one reference walk per session; the first mismatch is localised by
recomputing that one layer from the engine's own input.
"""
import copy
import hashlib
import json
import os
import pickle
import re
import subprocess
import sys
import tempfile
import time

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from ievm_testutil import cached_quantized, with_nonzero_zero_points  # noqa: E402
from oracle import int8_forward as O  # noqa: E402
from oracle import model_factory as mf  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
WIDTHS = {"w57": mf.PRUNED_WIDTHS, "w60": mf.DEFAULT_CFG_WIDTHS, "w64": mf.UNPRUNED_WIDTHS}
TILE_M = 128
CHUNK = 32                   # images per float64 oracle conv
GAIN = 40.0                  # edge images: x * GAIN saturates quantize_per_tensor on most pixels
SEED = 101


def num_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ------------------------------------------------------------------------------------------ inputs

def edge_starts(n):
    """First index of each edge triplet (gain, all-zero, negative gain): first, middle and last images of the batch."""
    return (0, n // 2 - 1, n - 3) if n >= 9 else ()


def images(n, seed=SEED):
    """Seeded images; batches of 9 or more carry three edge triplets, so they land in the first, a middle and the
    last (ragged) M tile of every layer."""
    x = mf.synthetic_images(n, seed=seed).numpy()
    for s in edge_starts(n):
        x[s] *= GAIN                 # saturates quantize: pushes deep layers to 255
        x[s + 1] = 0.0               # constant quantised input: only the zero-point borders differ
        x[s + 2] *= -GAIN
    return x


# ------------------------------------------------------------------------------------------ qparam variants

def _conv_jobs(qnet):
    """The convs after the stem in the engine's launch order, with what each reads:
    (QConv, input name, input scale, input zp, residual) -- residual = (name, scale, zp, add scale, add zp) or None.
    Tensors are named after the conv producing them ("maxpool" for the pool); a block's output carries its conv2's."""
    jobs = []
    cur, cs, cz = "maxpool", qnet.stem.out_scale, qnet.stem.out_zp
    for blk in qnet.blocks:
        jobs.append((blk.conv1, cur, cs, cz, None))
        if blk.down is not None:
            jobs.append((blk.down, cur, cs, cz, None))
            res = (blk.down.name, blk.down.out_scale, blk.down.out_zp)
        else:
            res = (cur, cs, cz)
        jobs.append((blk.conv2, blk.conv1.name, blk.conv1.out_scale, blk.conv1.out_zp, res + (blk.add_scale, blk.add_zp)))
        cur, cs, cz = blk.conv2.name, blk.add_scale, blk.add_zp
    return jobs


def _set_conv(mod, w_scale=None, zero_bias=False):
    w, b = mod.weight(), mod.bias()
    if w_scale is not None:
        w = torch._make_per_channel_quantized_tensor(w.int_repr(), torch.from_numpy(w_scale.astype(np.float64)),
                                                     w.q_per_channel_zero_points(), w.q_per_channel_axis())
    if zero_bias:
        b = torch.zeros(w.shape[0], dtype=torch.float32)
    mod.set_weight_bias(w, b)


TIE_LAYERS = ("layer1.0.conv1", "layer3.1.conv1", "layer1.1.conv2")   # two-CTA halo, CTA pair, residual (fused add_relu)


def with_ties(gm):
    """Bias 0 on TIE_LAYERS, their output scale moved to in_s * 2^j and every weight scale to a power of two (each within
    a factor sqrt(2) of the calibrated value): fl(in_s * w_s[c]) and the requantisation multiplier fl(fl(in_s * w_s[c]) /
    out_s) are then exact, the multiplier is a power of two 2^-k, acc * 2^-k is exact, and every acc that is an odd
    multiple of 2^(k-1) requantises to an exact .5 tie."""
    g = copy.deepcopy(gm)
    mods = dict(g.named_modules())
    in_scale = {c.name: s for c, _, s, _, _ in _conv_jobs(O.extract_qnet(g))}
    pow2 = lambda v: np.float32(2.0) ** np.round(np.log2(v.astype(np.float64))).astype(np.float32)   # noqa: E731
    for name in TIE_LAYERS:
        mod = mods[name]
        i32 = np.float32(in_scale[name])
        o32 = np.float32(i32 * pow2(np.array([mod.scale / i32]))[0])
        ws = pow2(mod.weight().q_per_channel_scales().numpy())
        mult = ((i32 * ws).astype(np.float32) / o32).astype(np.float32)
        assert (mult == pow2(mult)).all() and (mult < 1).all(), name
        mod.scale = float(o32)
        _set_conv(mod, w_scale=ws, zero_bias=True)
    return g


SAT_LAYERS = ("layer1.0.conv1", "layer3.1.conv1")


def rounding_bound(c):
    """The host's bound on |value before rounding| (ievm.cu upload_conv_operands) for QConv ``c``, given its input scale."""
    def bound(in_s):
        atw = (np.float32(in_s) * c.w_scale.astype(np.float32)).astype(np.float32)
        ep0 = np.abs((c.bias.astype(np.float32) / atw).astype(np.float32)).astype(np.float64)
        ep1 = np.abs((atw / np.float32(c.out_scale)).astype(np.float32)).astype(np.float64)
        sw = np.abs(c.w.astype(np.float64)).reshape(c.w.shape[0], -1).sum(1)
        return float(((255.0 * sw + ep0) * ep1).max())
    return bound


def with_saturation(gm):
    """SAT_LAYERS' output scales divided until the host's rounding bound passes 4 * 2^21: those layers run the general
    rounding epilogue (fast_round = 0) with most outputs clamped at 255."""
    g = copy.deepcopy(gm)
    mods = dict(g.named_modules())
    jobs = {c.name: (c, s) for c, _, s, _, _ in _conv_jobs(O.extract_qnet(g))}
    for name in SAT_LAYERS:
        c, in_s = jobs[name]
        f = float(2 ** np.ceil(np.log2(4 * 2.0 ** 21 / rounding_bound(c)(in_s))))
        mods[name].scale = float(np.float32(c.out_scale / f))
    return g


VARIANTS = {"ties": with_ties, "saturation": with_saturation, "zero_points": with_nonzero_zero_points}


# ------------------------------------------------------------------------------------------ engine + plan

_PLAN_LINE = re.compile(r"\[ievm\] layer\s+(\d+) (\d)x\d s(\d)\s+(\d+)->\s*(\d+) @(\d+)x(\d+) (.*)")


def parse_plan(text):
    """IEVM_VERBOSE lines -> {layer index: {field: value}} (ints where the value is an integer)."""
    plan = {}
    for m in _PLAN_LINE.finditer(text):
        f = {k: (int(v) if re.fullmatch(r"-?\d+", v) else v) for k, v in re.findall(r"(\w+)=(\S+)", m.group(8))}
        f.update(k=int(m.group(2)), stride=int(m.group(3)), cin=int(m.group(4)), cout=int(m.group(5)), ho=int(m.group(6)))
        plan[int(m.group(1))] = f
    return plan


def create_engine(spec, max_batch):
    """Engine over ``spec`` and its tile plan, read from the IEVM_VERBOSE lines ievm_create writes to stderr."""
    import ievm_b200
    had = os.environ.get("IEVM_VERBOSE")
    os.environ["IEVM_VERBOSE"] = "1"
    with tempfile.TemporaryFile() as f:
        saved = os.dup(2)
        os.dup2(f.fileno(), 2)
        try:
            eng = ievm_b200.B200QuantizedResNet(spec, max_batch=max_batch)
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            if had is None:
                del os.environ["IEVM_VERBOSE"]
        f.seek(0)
        text = f.read().decode(errors="replace")
    return eng, parse_plan(text)


def form(eng, plan, li, n):
    """The kernel form a conv runs in at batch n: tiny (one accumulator) vs ring is decided per call from n * sub-tiles
    against the SM count (ievm.cu launch_conv)."""
    p = plan.get(li)
    if p is None:
        return "?"
    if p["dual"] != "none":
        return f"dual-{p['dual']} cl={p['cluster']}"
    if p["mode"] == "halo":
        if n * p["subs"] <= num_sms():
            return "halo-tiny" + ("-zc" if p["zcorr"] else "")
        return ("halo-2cta-ring" if p["two_cta"] and not p["zcorr"] else "halo-ring") + ("-zc" if p["zcorr"] else "")
    return f"im2col cl={p['cluster']} bn={p['bn']}x{p['n_tiles']}" + (" zc" if p["zcorr"] else "")


# ------------------------------------------------------------------------------------------ comparison helpers

def _digests(a):
    return [hashlib.sha256(np.ascontiguousarray(a[i]).tobytes()).hexdigest() for i in range(a.shape[0])]


def _first_bad(got, want, i0=0):
    """(image, channel, y, x) of the first differing element and how many differ."""
    bad = got != want
    idx = np.argwhere(bad)[0]
    return (int(idx[0]) + i0, int(idx[1]), int(idx[2]), int(idx[3])), int(bad.sum())


def _where(name, pos, count, ho, wo, got, want):
    i, c, y, x = pos
    m = (i * ho + y) * wo + x
    return (f"{name}: {count} elements differ; first at image {i}, channel {c}, y {y}, x {x} (M tile {m // TILE_M}): "
            f"engine {got} vs oracle {want}")


def _ref_conv(c, xq, x_scale, x_zp, res):
    """Oracle conv over one chunk of images: (int32 accumulators, u8 output)."""
    acc = O.conv_acc(xq, x_zp, c.w, c.stride, c.pad)
    out = O.requant(acc, x_scale, c.w_scale, c.bias, c.out_scale, c.out_zp, c.relu)
    if res is not None:
        r, rs, rz, a_s, a_z = res
        out = O.add_relu(out, c.out_scale, c.out_zp, r, rs, rz, a_s, a_z)
    return acc, out


def _ties(acc, x_scale, c):
    """Requantisations of ``acc`` that are exact .5 ties with both neighbours inside the u8 output range."""
    atw = (np.float32(x_scale) * c.w_scale.astype(np.float32)).astype(np.float32)
    bdiv = (c.bias.astype(np.float32) / atw).astype(np.float32)[None, :, None, None]
    mult = (atw / np.float32(c.out_scale)).astype(np.float32)[None, :, None, None]
    v = ((acc.astype(np.float32) + bdiv).astype(np.float32) * mult).astype(np.float32)
    fl = np.floor(v)
    lo = c.out_zp if c.relu else 0
    return int(((v - fl == 0.5) & (fl + c.out_zp >= lo) & (fl + 1 + c.out_zp <= 255)).sum())


def _head_logits(qnet, last, zp, scale):
    pooled = O.avgpool(last)
    acc = ((pooled.astype(np.int64) - zp) @ qnet.fc_w.astype(np.int64).T).astype(np.int32)
    q = O.requant(acc, scale, qnet.fc_w_scale, qnet.fc_bias, qnet.fc_scale, qnet.fc_zp, False, ch_axis=1)
    return ((q.astype(np.float32) - np.float32(qnet.fc_zp)) * np.float32(qnet.fc_scale)).astype(np.float32)


def _layer_index(eng):
    return {L.name: i for i, L in enumerate(eng.net.layers)}


# ------------------------------------------------------------------------------------------ the checker

def check_layers_i8(eng, qnet, x, logits, plan=None):
    """Every check of the module docstring on an engine that has just run ``logits = eng(x)`` with keep_tensors=1.
    Returns (rows of the per-layer table, per-image digests of every reference tensor)."""
    n = x.shape[0]
    idx = _layer_index(eng)
    layers = eng.net.layers
    digests, rows = {}, []
    # ---- input, stem, max-pool
    xq = O.quantize_input(x, qnet.in_scale, qnet.in_zp)
    got = eng.read_tensor(0)
    if not np.array_equal(got, xq):
        pos, cnt = _first_bad(got, xq)
        raise AssertionError("quantized input: " + _where("quantize", pos, cnt, 224, 224, got[pos], xq[pos]))
    S = qnet.stem
    Ls = layers[idx[S.name]]
    stem_out = eng.read_tensor(Ls.out_tensor)
    pool_out = eng.read_tensor(layers[1].out_tensor)
    stem_acc = eng.conv_accumulators(S.name, n)
    ho, wo = stem_out.shape[2:]
    ref_pool = np.empty_like(pool_out)
    digests[S.name + ":acc"], digests[S.name] = [], []
    for s in range(0, n, CHUNK):
        ra, ro = _ref_conv(S, xq[s:s + CHUNK], qnet.in_scale, qnet.in_zp, None)
        if not np.array_equal(stem_acc[s:s + CHUNK], ra):
            pos, cnt = _first_bad(stem_acc[s:s + CHUNK], ra, s)
            raise AssertionError("accumulators differ (operand path): " +
                                 _where(S.name, pos, cnt, ho, wo, stem_acc[pos], ra[(pos[0] - s,) + pos[1:]]))
        if not np.array_equal(stem_out[s:s + CHUNK], ro):
            pos, cnt = _first_bad(stem_out[s:s + CHUNK], ro, s)
            raise AssertionError("output differs with matching accumulators (epilogue or store): " +
                                 _where(S.name, pos, cnt, ho, wo, stem_out[pos], ro[(pos[0] - s,) + pos[1:]]))
        ref_pool[s:s + CHUNK] = O.maxpool3x3s2(ro)
        digests[S.name + ":acc"] += _digests(ra)
        digests[S.name] += _digests(ro)
    del stem_acc
    if not np.array_equal(pool_out, ref_pool):
        pos, cnt = _first_bad(pool_out, ref_pool)
        raise AssertionError(_where("maxpool", pos, cnt, *pool_out.shape[2:], pool_out[pos], ref_pool[pos]))
    digests["maxpool"] = _digests(ref_pool)
    ref = {"maxpool": ref_pool}
    rows.append((S.name, "stem_tc", stem_out.size, int((stem_out == 255).sum()),
                 int((stem_out == (S.out_zp if S.relu else 0)).sum()), -1))
    del stem_out
    # ---- every conv, in launch order; a block's conv1 and downsample (a dual launch) are both read before either dump
    fwd = {}
    for c, src, x_scale, x_zp, res in _conv_jobs(qnet):
        li = idx[c.name]
        L = layers[li]
        if c.name not in fwd:
            fwd[c.name] = eng.read_tensor(L.out_tensor)
            mate = [d for d, s2, _, _, r2 in _conv_jobs(qnet) if s2 == src and r2 is None and d.name != c.name]
            if res is None and mate:
                fwd[mate[0].name] = eng.read_tensor(layers[idx[mate[0].name]].out_tensor)
        out = fwd.pop(c.name)
        acc = eng.conv_accumulators(c.name, n)
        ho, wo = out.shape[2:]
        xin = ref[src]
        rres = None if res is None else (ref[res[0]],) + res[1:]
        ref_out = np.empty_like(out)
        ties = 0
        digests[c.name + ":acc"], digests[c.name] = [], []
        for s in range(0, n, CHUNK):
            sl = slice(s, s + CHUNK)
            ra, ro = _ref_conv(c, xin[sl], x_scale, x_zp, None if rres is None else (rres[0][sl],) + rres[1:])
            if not np.array_equal(acc[sl], ra):
                pos, cnt = _first_bad(acc[sl], ra, s)
                raise AssertionError("accumulators differ (operand path: A/B loads, im2col / halo addressing, MMA): " +
                                     _where(c.name, pos, cnt, ho, wo, acc[pos], ra[(pos[0] - s,) + pos[1:]]))
            if not np.array_equal(out[sl], ro):
                pos, cnt = _first_bad(out[sl], ro, s)
                raise AssertionError("output differs with matching accumulators (epilogue or store, or the forward's "
                                     "launch read an unfinished input): " +
                                     _where(c.name, pos, cnt, ho, wo, out[pos], ro[(pos[0] - s,) + pos[1:]]))
            ties += _ties(ra, x_scale, c)
            ref_out[sl] = ro
            digests[c.name + ":acc"] += _digests(ra)
            digests[c.name] += _digests(ro)
        ref[c.name] = ref_out
        lo = res[4] if res is not None else (c.out_zp if c.relu else 0)
        rows.append((c.name, form(eng, plan or {}, li, n), out.size, int((out == 255).sum()), int((out == lo).sum()), ties))
        del acc
    # ---- head
    last = qnet.blocks[-1].conv2.name
    want = _head_logits(qnet, ref[last], qnet.blocks[-1].add_zp, qnet.blocks[-1].add_scale)
    if not np.array_equal(logits, want):
        i = int(np.argwhere((logits != want).any(1))[0][0])
        raise AssertionError(f"head: logits of image {i} differ: engine {logits[i]} vs oracle {want[i]}")
    digests["logits"] = _digests(want)
    # ---- product front end at the same batch (last: it overwrites the kept max-pool tensor)
    pooled, facc = eng.debug_frontend(torch.from_numpy(x).cuda())
    bad = [i for i, d in enumerate(_digests(facc)) if d != digests[S.name + ":acc"][i]]
    assert not bad, f"front end: stem accumulators of {len(bad)} images differ, first image {bad[0]}"
    del facc
    assert np.array_equal(pooled, ref_pool), f"front end: pooled tensor differs ({int((pooled != ref_pool).sum())} bytes)"
    pooled_product, _ = eng.debug_frontend(torch.from_numpy(x).cuda(), want_acc=False)
    assert np.array_equal(pooled_product, ref_pool), "front end (product instantiation): pooled tensor differs"
    return rows, digests


def print_table(rows, label, t0):
    print(f"\n{label}: {'layer':24s} {'form':24s} {'elements':>11s} {'=255':>10s} {'=lo':>10s} {'ties':>9s}")
    for name, fm, el, hi, lo, ties in rows:
        print(f"{'':{len(label)}s}  {name:24s} {fm:24s} {el:11d} {hi:10d} {lo:10d} {ties if ties >= 0 else '-':>9}")
    print(f"{label}: {time.time() - t0:.1f} s")


def run_case(gm, x, max_batch=256, spec=None, qnet=None, live=True, label=""):
    """Engine over ``spec`` (default: the flattened ``gm``), one keep_tensors forward of ``x`` checked layer by layer
    against the oracle of ``qnet`` (default: ``gm``'s), then the product configuration and the live fbgemm module.
    Returns (rows, digests, logits)."""
    import ievm_b200
    t0 = time.time()
    qnet = qnet or O.extract_qnet(gm)
    eng, plan = create_engine(spec or ievm_b200.from_converted(gm), max_batch)
    try:
        eng.set_option("keep_tensors", 1)
        logits = eng(torch.from_numpy(x).cuda()).cpu().numpy()
        rows, digests = check_layers_i8(eng, qnet, x, logits, plan)
        eng.set_option("keep_tensors", 0)
        assert np.array_equal(eng(torch.from_numpy(x).cuda()).cpu().numpy(), logits), "product configuration's logits differ"
    finally:
        eng.close()
    if live:
        torch.backends.quantized.engine = "fbgemm"
        with torch.no_grad():
            assert np.array_equal(gm(torch.from_numpy(x)).numpy(), logits), "logits differ from the live fbgemm module"
    print_table(rows, label or f"n={x.shape[0]}", t0)
    return rows, digests, logits


def assert_clamps(rows):
    """Every conv output of an edge batch reaches its lower clamp, and every one except the 1x1 downsamples reaches 255
    (no ReLU and zero points near 70: in the reference, layer3.0's reaches 255 on none of the 251 images)."""
    for name, _, _, hi, lo, _ in rows:
        assert lo > 0 and (hi > 0 or "downsample" in name), \
            f"{name}: the batch does not reach both clamps ({hi} at 255, {lo} at the lower clamp)"


# ------------------------------------------------------------------------------------------ cases

def test_int8_w57_n251_every_tensor_bit_exact_with_edge_images(reference_w57):
    """Layers 3 and 4 end on an odd, partial M tile (385 and 97 tiles of 128 pixels) after more than one round of CTA
    pairs over the persistent grid; edge images in the first, a middle and the last tile."""
    rows = reference_w57["rows"]
    assert_clamps(rows)


@pytest.mark.parametrize("tag,n", [("w57", 256), ("w60", 251), ("w64", 251)])
def test_int8_every_tensor_bit_exact_at_the_bench_plan(tag, n):
    rows, _, _ = run_case(cached_quantized(WIDTHS[tag]), images(n), label=f"{tag} n={n}")
    assert_clamps(rows)


@pytest.mark.parametrize("n", [1, 5, 6, 21, 22])
def test_int8_small_batches_on_the_bench_plan(n):
    """bs 1 (one half-empty CTA pair) and both sides of the single-accumulator / ring threshold of the layer-1 (28
    sub-tiles per image) and layer-2 (7) halo convs on a 148-SM part; test_plan_covers_the_intended_forms checks that
    these batches straddle the thresholds of the SM count at hand."""
    run_case(cached_quantized(WIDTHS["w57"]), images(n, seed=SEED + n), label=f"w57 n={n}")


def test_int8_batch_263_on_the_1024_plan():
    """The plan of test_int8_batch_size_invariance_up_to_1024 (tile widths and CTA pairs chosen for 1024 images); 263
    images give odd, ragged M-tile counts in layers 3 (403) and 4 (101)."""
    rows, _, _ = run_case(cached_quantized(WIDTHS["w57"]), images(263, seed=SEED + 1), max_batch=1024, label="w57 n=263 @1024")
    assert_clamps(rows)


@pytest.mark.parametrize("variant", sorted(VARIANTS))
def test_int8_qparam_variants_bit_exact(variant):
    """ties: exact .5 ties at a known rate on TIE_LAYERS; saturation: the general rounding epilogue (fast_round = 0) with
    most outputs clamped on SAT_LAYERS; zero_points: every conv after the stem reads a non-zero zero point (the zcorr
    kernels at CTA pairs and over several rounds)."""
    gm = VARIANTS[variant](cached_quantized(WIDTHS["w57"]))
    rows, _, _ = run_case(gm, images(251), label=f"w57 n=251 {variant}")
    by = {r[0]: r for r in rows}
    if variant == "ties":
        for name in TIE_LAYERS:
            assert by[name][5] >= 1000, f"{name}: only {by[name][5]} ties inside the u8 range"
    if variant == "saturation":
        for name in SAT_LAYERS:
            _, _, el, hi, lo, _ = by[name]
            assert hi + lo >= 0.9 * el and hi > 0, f"{name}: only {hi} + {lo} of {el} outputs clamp"


# ------------------------------------------------------------------------------------------ sensitivity

def _mutated(mutate):
    import ievm_b200
    gm = cached_quantized(WIDTHS["w57"])
    spec = copy.deepcopy(ievm_b200.from_converted(gm))
    mutate({L.name: L for L in spec.layers})
    return gm, spec


def _flip(w, pos):
    w[pos] = w[pos] - 1 if w[pos] > -127 else w[pos] + 1


def _last_tap(L):
    L.weight = L.weight.copy()
    _flip(L.weight, (L.cout - 1, 0, 1, 1))


def _bias(L):
    L.bias = L.bias.copy()
    L.bias[7] += 3 * L.out_scale


def _down(L):
    L.weight = L.weight.copy()
    _flip(L.weight, (11, 5, 0, 0))


@pytest.mark.parametrize("mutate,pattern", [
    (("layer4.1.conv1", _last_tap), r"accumulators differ.*layer4\.1\.conv1:.*channel 459,"),
    (("layer1.1.conv2", _bias), r"output differs with matching accumulators.*layer1\.1\.conv2:"),
    (("layer3.0.downsample.0", _down), r"accumulators differ.*layer3\.0\.downsample\.0:.*channel 11,"),
], ids=["weight_tap_cta_pair", "bias_two_cta_halo_add_relu", "dual_second_class"])
def test_checker_catches_injected_bugs_at_their_layer(mutate, pattern):
    """The engine runs a mutated flattened description; the oracle runs the module.  The checker must fail at the
    mutated layer, with the kind of failure and the channel the mutation implies."""
    name, fn = mutate
    gm, spec = _mutated(lambda by: fn(by[name]))
    with pytest.raises(AssertionError, match=pattern) as e:
        run_case(gm, images(6, seed=SEED + 6), spec=spec, live=False, label=f"mutated {name}")
    print(f"\ncaught: {str(e.value)[:300]}")


# ------------------------------------------------------------------------------------------ reference digests and configurations

@pytest.fixture(scope="session")
def reference_w57(tmp_path_factory):
    """One full reference walk of w57 at n = 251 on the bench plan; writes the flattened network, the oracle's QNet,
    the per-image SHA-256 digests of every reference tensor and the logits for the configuration subprocesses."""
    import ievm_b200
    gm = cached_quantized(WIDTHS["w57"])
    x = images(251)
    rows, digests, logits = run_case(gm, x, label="w57 n=251")
    d = tmp_path_factory.mktemp("int8_reference")
    ievm_b200.from_converted(gm).save(str(d / "spec.npz"))
    with open(d / "qnet.pkl", "wb") as f:
        pickle.dump(O.extract_qnet(gm), f)
    (d / "digests.json").write_text(json.dumps(digests))
    np.save(d / "logits.npy", logits)
    return {"dir": str(d), "rows": rows}


def check_digests(eng, qnet, x, logits, digests):
    """check_layers_i8 for a configuration subprocess: per-image digests of the forward's tensors and of the dumped
    accumulators against the reference walk's; the first mismatching layer is recomputed from the engine's own input."""
    n = x.shape[0]
    idx = _layer_index(eng)
    layers = eng.net.layers

    def compare(name, arr, kind, recompute):
        bad = [i for i, d in enumerate(_digests(arr)) if d != digests[name + kind][i]]
        if bad:
            i = bad[0]
            ra, ro = recompute(i)
            want = ra if kind == ":acc" else ro
            pos, cnt = _first_bad(arr[i:i + 1], want, i)
            what = "accumulators differ (operand path)" if kind == ":acc" else "output differs (epilogue or store)"
            raise AssertionError(f"{what} in {len(bad)} images: " +
                                 _where(name, pos, cnt, *arr.shape[2:], arr[pos], want[(0,) + pos[1:]]))

    S = qnet.stem
    xq = eng.read_tensor(0)
    stem_re = lambda i: _ref_conv(S, xq[i:i + 1], qnet.in_scale, qnet.in_zp, None)   # noqa: E731
    compare(S.name, eng.read_tensor(layers[idx[S.name]].out_tensor), "", stem_re)
    pool = eng.read_tensor(layers[1].out_tensor)
    compare("maxpool", pool, "", lambda i: (None, O.maxpool3x3s2(stem_re(i)[1])))
    compare(S.name, eng.conv_accumulators(S.name, n), ":acc", stem_re)
    fwd = {}
    jobs = _conv_jobs(qnet)
    for c, src, x_scale, x_zp, res in jobs:
        L = layers[idx[c.name]]
        if c.name not in fwd:
            fwd[c.name] = eng.read_tensor(L.out_tensor)
            mate = [d for d, s2, _, _, r2 in jobs if s2 == src and r2 is None and d.name != c.name]
            if res is None and mate:
                fwd[mate[0].name] = eng.read_tensor(layers[idx[mate[0].name]].out_tensor)
        xin = eng.read_tensor(L.in_tensor)
        rin = eng.read_tensor(L.res_tensor) if res is not None else None

        def recompute(i, c=c, xin=xin, rin=rin, x_scale=x_scale, x_zp=x_zp, res=res):
            return _ref_conv(c, xin[i:i + 1], x_scale, x_zp, None if res is None else (rin[i:i + 1],) + res[1:])
        compare(c.name, fwd.pop(c.name), "", recompute)
        compare(c.name, eng.conv_accumulators(c.name, n), ":acc", recompute)
    assert _digests(logits) == digests["logits"][:n], "logits differ from the reference walk's"


def run_variant(ref_dir, n):
    """Body of a configuration subprocess (knobs in its environment): the reference batch's first n images."""
    import ievm_b200
    spec = ievm_b200.NetSpec.load(os.path.join(ref_dir, "spec.npz"))
    with open(os.path.join(ref_dir, "qnet.pkl"), "rb") as f:
        qnet = pickle.load(f)
    with open(os.path.join(ref_dir, "digests.json")) as f:
        digests = json.load(f)
    want = np.load(os.path.join(ref_dir, "logits.npy"))[:n]
    x = images(251)[:n]
    eng = ievm_b200.B200QuantizedResNet(spec, max_batch=256)
    try:
        eng.set_option("keep_tensors", 1)
        logits = eng(torch.from_numpy(x).cuda()).cpu().numpy()
        assert np.array_equal(logits, want), "keep_tensors logits differ from the verified ones"
        check_digests(eng, qnet, x, logits, digests)
        eng.set_option("keep_tensors", 0)              # product configuration: fused / chunked / separate front end
        assert np.array_equal(eng(torch.from_numpy(x).cuda()).cpu().numpy(), want), "product-configuration logits differ"
    finally:
        eng.close()


_VARIANT = r"""
import os, sys
sys.path.insert(0, sys.argv[1])
sys.path.insert(0, os.path.join(sys.argv[1], "tests"))
import test_gpu_int8_layers as T
T.run_variant(sys.argv[2], int(sys.argv[3]))
print("variant ok")
"""

CONFIGS = {
    "halo_dynamic": ({"IEVM_HALO_STATIC": "0"}, 251),                   # run-time-shaped halo kernel (shape class 0)
    "band1": ({"IEVM_BAND_SUBS": "1"}, 251),                             # one sub-tile per TMA patch
    "band3_kb1": ({"IEVM_BAND_SUBS": "3", "IEVM_KB_GROUP": "1"}, 251),   # odd band size, one k-block per barrier
    "no_halo": ({"IEVM_HALO": "0"}, 251),                                # every conv through per-tap im2col TMA
    "no_dual": ({"IEVM_DUAL": "0"}, 251),                                # the 1x1 downsample convs as launches of their own
    "no_phase_patches": ({"IEVM_S2": "0"}, 251),                         # stride-2 dual launch as pixel pairs
    "no_pixel_pairs": ({"IEVM_S2": "0", "IEVM_WIDE": "0"}, 251),         # ... and as nine 64-byte-row taps
    "no_tiny": ({"IEVM_TINY": "0"}, 5),                                  # small batches through the accumulator ring
    "no_two_cta": ({"IEVM_TWO_CTA": "0"}, 251),                          # one CTA per SM for the 64-channel halo convs
    "no_cluster": ({"IEVM_CLUSTER": "0"}, 251),                          # no CTA pairs / weight multicast
    "fixed_bn": ({"IEVM_FIXED_BN": "1"}, 251),                           # one N tile per <= 256 channels
    "no_fast_round": ({"IEVM_FAST_ROUND": "0"}, 251),                    # the general rounding epilogues everywhere
    "no_pdl": ({"IEVM_PDL": "0"}, 251),                                  # no programmatic dependent launch
    "separate_front": ({"IEVM_FUSED_FRONT": "0"}, 251),                  # quantize / stem / max-pool kernels
    "chunked_front": ({"IEVM_FUSED_FRONT": "0", "IEVM_FRONT_CHUNK": "64"}, 251),   # ... in chunks of 64 images
}


def _plan_check(cfg, plan):
    """What each knob must change in the plan (the IEVM_VERBOSE lines of the subprocess)."""
    convs = [p for p in plan.values()]
    im2col3 = [p for p in convs if p["mode"] == "im2col" and p["k"] == 3]
    if cfg == "no_halo":
        assert all(p["mode"] == "im2col" for p in convs)
    if cfg == "no_two_cta":
        assert not any(p["two_cta"] for p in convs)
    if cfg == "no_cluster":
        assert all(p["cluster"] == 1 for p in convs)
    if cfg == "fixed_bn":
        assert all(p["n_tiles"] == -(-p["cout"] // 256) for p in im2col3)
    if cfg == "no_fast_round":
        assert all(p["fast_round"] == 0 for p in convs)
    if cfg == "no_phase_patches":
        assert not any(p["dual"] == "s2" for p in convs) and any(p["dual"] == "wide" for p in convs)
    if cfg == "no_pixel_pairs":
        assert all(p["dual"] in ("none", "plain") for p in convs)


@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_int8_kernel_configurations_every_tensor_bit_exact(cfg, reference_w57, tmp_path):
    """Each knob in a subprocess of its own (read when the engine is created): every tensor and accumulator of the
    forward against the reference digests, and the product configuration's logits against the verified logits (the
    keep_tensors forward bypasses the fused and chunked front ends).  A missing PDL dependency wait corrupts only the
    forward's tensors, never a dump launch: outputs are read from the forward."""
    env, n = CONFIGS[cfg]
    script = tmp_path / "variant.py"
    script.write_text(_VARIANT)
    e = dict(os.environ)
    e.update(env)
    e["IEVM_VERBOSE"] = "1"
    t0 = time.time()
    r = subprocess.run([sys.executable, str(script), ROOT, reference_w57["dir"], str(n)], env=e, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0 and "variant ok" in r.stdout, (r.stdout[-3000:], r.stderr[-3000:])
    plan = parse_plan(r.stderr)
    assert plan, r.stderr[-2000:]
    _plan_check(cfg, plan)
    print(f"\n{cfg} n={n}: every tensor and accumulator bit-exact ({time.time() - t0:.1f} s)")


# ------------------------------------------------------------------------------------------ the forms each case runs

def test_plan_covers_the_intended_forms():
    """Creation only: the plan each case's engine gets, and the per-call tiny / ring choice of its halo convs."""
    import ievm_b200
    sms = num_sms()

    def plan_of(gm, max_batch):
        eng, plan = create_engine(ievm_b200.from_converted(gm), max_batch)
        names = {i: L.name for i, L in enumerate(eng.net.layers)}
        eng.close()
        return {names[i]: p for i, p in plan.items()}

    gm = cached_quantized(WIDTHS["w57"])
    for max_batch in (256, 1024):
        p = plan_of(gm, max_batch)
        for name, f in p.items():
            print(f"@{max_batch} {name:24s} " + " ".join(f"{k}={v}" for k, v in f.items()))
        for b in ("layer1.0", "layer1.1"):
            for cv in ("conv1", "conv2"):
                assert p[f"{b}.{cv}"]["mode"] == "halo" and p[f"{b}.{cv}"]["two_cta"] == 1
        for b in ("layer2.0.conv2", "layer2.1.conv1", "layer2.1.conv2"):
            assert p[b]["mode"] == "halo" and p[b]["two_cta"] == 0
        assert not any(f["zcorr"] for f in p.values())
        if max_batch == 256:
            for b in ("layer3.0.conv1", "layer3.0.conv2", "layer3.1.conv1", "layer3.1.conv2",
                      "layer4.0.conv1", "layer4.0.conv2", "layer4.1.conv1", "layer4.1.conv2"):
                assert p[b]["cluster"] == 2, (b, p[b])
            assert p["layer2.0.conv1"]["dual"] == "s2" and p["layer3.0.conv1"]["dual"] == "plain"
            assert p["layer3.0.downsample.0"]["dual"] == "plain" and p["layer4.0.downsample.0"]["dual"] == "plain"
            assert p["layer3.0.downsample.0"]["cluster"] == 1                      # resident weights
            assert p["layer4.1.conv1"]["n_tiles"] == 3 and p["layer4.1.conv1"]["bn"] == 160
            spi1, spi2 = p["layer1.0.conv1"]["subs"], p["layer2.1.conv1"]["subs"]
            # the small-batch cases straddle both tiny / ring thresholds (28 and 7 sub-tiles per image on 148 SMs)
            t1, t2 = sms // spi1, sms // spi2
            print(f"{sms} SMs: layer-1 halo convs tiny up to n = {t1}, layer-2 up to n = {t2}")
            assert {t1, t1 + 1} <= {1, 5, 6, 21, 22} and {t2, t2 + 1} <= {1, 5, 6, 21, 22}, (t1, t2)
    for tag in ("w60", "w64"):
        p = plan_of(cached_quantized(WIDTHS[tag]), 256)
        assert p["layer1.0.conv1"]["mode"] == "halo" and p["layer4.1.conv1"]["cluster"] == 2, tag
    p = plan_of(VARIANTS["saturation"](gm), 256)
    for name in SAT_LAYERS:
        assert p[name]["fast_round"] == 0, name
    assert sum(f["fast_round"] == 0 for f in p.values()) == len(SAT_LAYERS)
    p = plan_of(VARIANTS["zero_points"](gm), 256)
    assert sum(f["zcorr"] for f in p.values()) >= 15 and p["layer3.1.conv1"]["zcorr"] == 1
    assert p["layer3.1.conv1"]["cluster"] == 2 and all(f["dual"] == "none" for f in p.values())
