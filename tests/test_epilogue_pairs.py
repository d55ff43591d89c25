"""The INT8 conv epilogues on paired FP32 instructions (FADD2 / FMUL2 / FFMA2, csrc/conv_tc.cuh).

ptxas contracts a paired multiply followed by a paired add into one FFMA2, even when both carry an explicit .rn.  The
epilogues round with a magic-number add (x + 1.5 * 2^23), and fl(x * mu + M) differs from fl(fl(x * mu) + M) whenever
the exact product lies within half an ulp of a .5 point, so a contracted epilogue is not bit-exact with ATen.
  * CPU: no FFMA / FFMA2 in an INT8 conv kernel adds the magic constant, and the paired forms are really there.
  * GPU: the production device functions, run through a small test kernel, on operands chosen so that a contracted
    multiply-add WOULD round differently, equal the scalar op-by-op definition (tests/test_epilogue_math.py shows that
    definition equals the oracle's)."""
import ctypes as C
import re
import shutil
import subprocess

import numpy as np
import pytest

from ievm_b200 import _lib

MAGIC = np.float32(12582912.0)          # 1.5 * 2^23
INT8_KERNELS = re.compile(r"conv_tc_kernelILi0E|conv_s2_kernel|conv_dual_kernelILi0E")
MAGIC_IMM = ("12582912", "0x4b400000")


def _sass_by_kernel(lib):
    out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    kernels, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            cur = kernels.setdefault(m.group(1), [])
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4}\*/\s+(.*?)\s*;", line)
        if m and cur is not None:
            cur.append(re.sub(r"^@!?U?P\w+\s+", "", m.group(1)))
    return kernels


def _magic_in_addend(ins, magic_regs):
    addend = ins.split(",")[-1].strip().lstrip("-|")
    reg = re.match(r"(U?R\d+)", addend)
    return addend.split()[0] in MAGIC_IMM or (reg is not None and reg.group(1) in magic_regs)


def test_no_magic_number_add_is_contracted_into_an_fma():
    kernels = {k: v for k, v in _sass_by_kernel(_lib.build()).items() if INT8_KERNELS.search(k)}
    assert len(kernels) >= 20
    paired = 0
    for name, code in kernels.items():
        magic_regs = set()      # registers that ever hold the magic constant: not a legal FFMA addend either
        for ins in code:
            op = ins.split()[0]
            dst = re.match(r"\S+\s+(U?R\d+)", ins)
            if dst and any(re.search(rf"(?<![\w.]){imm}\b", ins) for imm in MAGIC_IMM) and \
                    op.split(".")[0] in ("MOV", "UMOV", "IMAD", "MOV32I"):
                magic_regs.add(dst.group(1))
        for ins in code:
            op = ins.split()[0].split(".")[0]
            if op in ("FFMA", "FFMA2"):
                assert not _magic_in_addend(ins, magic_regs), f"{name}: contracted magic-number rounding: {ins}"
        ops = {ins.split()[0].split(".")[0] for ins in code}
        assert {"FADD2", "FMUL2", "FFMA2"} <= ops, f"{name}: the epilogue is not on paired instructions"
        paired += 1
    assert paired == len(kernels)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the device functions themselves on adversarial operands

_KERNEL_SRC = r"""
#include <cuda_runtime.h>
#include "conv_tc.cuh"
using namespace ievm;

template <bool kFast>
__global__ void requant16(const int* acc, const float* bd, const float* mu, int zp, int lo, uint4* out, int n) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  uint32_t v[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = static_cast<uint32_t>(acc[16 * t + i]);
  out[t] = epilogue16_i8<kFast>(v, bd + 16 * t, mu + 16 * t, zp, lo);
}

// per-thread constants: f = {a_scale, r_scale, inv_scale}, z = {out_zp, res_zp, add_zp, out_lo}; built as the conv kernels do
template <bool kFast, bool kResI2F>
__global__ void add_relu16(const int* acc, const uint4* res, const float* bd, const float* mu, const float* f, const int* z,
                           uint4* out, int n) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const int out_zp = z[4 * t], res_zp = z[4 * t + 1], add_zp = z[4 * t + 2], out_lo = z[4 * t + 3];
  AddReluConst k;
  k.lo_f = static_cast<float>(out_lo - out_zp);
  k.hi_f = static_cast<float>(255 - out_zp);
  k.a_scale = f[3 * t];
  k.r_scale = f[3 * t + 1];
  k.inv_scale = f[3 * t + 2];
  k.pa = __fmul_rn(k.a_scale, -static_cast<float>(out_zp));
  k.pb = __fmul_rn(k.r_scale, -static_cast<float>(res_zp));
  k.lo_q = static_cast<float>(out_lo);
  k.zp_f = static_cast<float>(out_zp);
  k.add_zp = add_zp;
  k.c1_add = -kRoundMagicBits - (out_lo - out_zp);
  k.c1_max = 255 - out_lo;
  k.c2_add = -kRoundMagicBits;
  k.c2_max = 255 - add_zp;
  k.zp4 = static_cast<uint32_t>(add_zp) * 0x01010101u;
  uint32_t v[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = static_cast<uint32_t>(acc[16 * t + i]);
  out[t] = epilogue16_i8_res<kFast, kResI2F>(v, res[t], bd + 16 * t, mu + 16 * t, k);
}

template <typename T>
static T* dev(const void* h, size_t bytes) {
  T* d = nullptr;
  cudaMalloc(&d, bytes);
  if (h) cudaMemcpy(d, h, bytes, cudaMemcpyHostToDevice);
  return d;
}

// form: 0 general, 1 fast; res: 0 requant, 1 add_relu with PRMT + FADD bytes, 2 add_relu with I2F.U8 bytes
extern "C" int run(int res, int form, int n, const int* acc, const unsigned char* r, const float* bd, const float* mu,
                   const float* f, const int* z, int zp, int lo, unsigned char* out) {
  const size_t n16 = static_cast<size_t>(n) * 16;
  int* d_acc = dev<int>(acc, n16 * 4);
  float* d_bd = dev<float>(bd, n16 * 4);
  float* d_mu = dev<float>(mu, n16 * 4);
  uint4* d_out = dev<uint4>(nullptr, n16);
  uint4* d_r = dev<uint4>(r, n16);
  float* d_f = dev<float>(f, static_cast<size_t>(n) * 12);
  int* d_z = dev<int>(z, static_cast<size_t>(n) * 16);
  const int b = 128, g = (n + b - 1) / b;
  if (res == 0) {
    if (form) requant16<true><<<g, b>>>(d_acc, d_bd, d_mu, zp, lo, d_out, n);
    else requant16<false><<<g, b>>>(d_acc, d_bd, d_mu, zp, lo, d_out, n);
  } else if (res == 1) {
    if (form) add_relu16<true, false><<<g, b>>>(d_acc, d_r, d_bd, d_mu, d_f, d_z, d_out, n);
    else add_relu16<false, false><<<g, b>>>(d_acc, d_r, d_bd, d_mu, d_f, d_z, d_out, n);
  } else {
    if (form) add_relu16<true, true><<<g, b>>>(d_acc, d_r, d_bd, d_mu, d_f, d_z, d_out, n);
    else add_relu16<false, true><<<g, b>>>(d_acc, d_r, d_bd, d_mu, d_f, d_z, d_out, n);
  }
  int err = static_cast<int>(cudaGetLastError());
  const int sync = static_cast<int>(cudaMemcpy(out, d_out, n16, cudaMemcpyDeviceToHost));
  if (!err) err = sync;
  cudaFree(d_acc); cudaFree(d_bd); cudaFree(d_mu); cudaFree(d_out); cudaFree(d_r); cudaFree(d_f); cudaFree(d_z);
  return err;
}
"""


@pytest.fixture(scope="module")
def epi_lib(tmp_path_factory):
    d = tmp_path_factory.mktemp("epi")
    src = d / "epi_test.cu"
    src.write_text(_KERNEL_SRC)
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    out = d / "epi_test.so"
    res = subprocess.run([nvcc] + _lib.NVCC_FLAGS + ["-I", _lib.CSRC, "-o", str(out), str(src)],
                         capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    lib = C.CDLL(str(out))
    lib.run.argtypes = [C.c_int] * 3 + [C.c_void_p] * 6 + [C.c_int, C.c_int, C.c_void_p]
    lib.run.restype = C.c_int
    return lib


def _f32(x):
    return np.asarray(x, np.float32)


def _fma(a, b, c):       # one rounding: float64 holds these products and sums exactly
    return (np.asarray(a, np.float64) * np.asarray(b, np.float64) + np.asarray(c, np.float64)).astype(np.float32)


def _near_ties(rng, t, lo_k, hi_k):
    """mu > 0 with t * mu within a few ulps of k + 0.5 for a k in [lo_k, hi_k] of t's sign."""
    k = rng.integers(lo_k, hi_k + 1, t.shape)
    k = np.where(t < 0, -np.abs(k) - 1, np.abs(k))            # k + 0.5 has t's sign
    mu = _f32((k + 0.5) / t.astype(np.float64))
    for _ in range(3):
        mu = np.where(rng.random(t.shape) < 0.5, np.nextafter(mu, np.float32(np.inf)), np.nextafter(mu, np.float32(0)))
    return mu


def _contracted_differs(t, mu):
    """rint(fl(t * mu)) != rint(t * mu): the elements where an FFMA with the magic addend changes the result."""
    p = t.astype(np.float64) * mu.astype(np.float64)
    return np.rint(p.astype(np.float32)) != np.rint(p)


def _requant_operands(rng, n, zp, lo):
    m = n * 16
    acc = rng.integers(-60_000, 60_000, m).astype(np.int32)
    acc[acc == 0] = 1
    bd = _f32(rng.standard_normal(m) * 40)
    t = _f32(acc.astype(np.float32) + bd)
    mu = _near_ties(rng, t, lo - zp - 2, 255 - zp + 2)
    kind = rng.random(m)
    tie = kind < 0.1                                           # exact .5 ties: odd acc, zero bias, mu = 1/2
    acc[tie] = (rng.integers(lo - zp - 2, 257 - zp, tie.sum()) * 2 + 1).astype(np.int32)
    bd[tie], mu[tie] = 0, 0.5
    big = (kind >= 0.1) & (kind < 0.15)                        # both clamps, far outside the u8 range
    mu[big] = _f32(rng.random(big.sum()) * 0.05 + 0.01)
    return acc, bd, mu


def _requant_ref(acc, bd, mu, zp, lo, fused=False):
    t = _f32(acc.astype(np.float32) + bd)
    v = np.rint(t.astype(np.float64) * mu) if fused else np.rint(_f32(t * mu))
    assert np.abs(v).max() < 2 ** 21
    return np.clip(np.maximum(v.astype(np.int64) + zp, lo), 0, 255).astype(np.uint8)


@pytest.mark.gpu
@pytest.mark.parametrize("zp,lo", [(61, 0), (61, 61), (0, 0)])
@pytest.mark.parametrize("form", [1, 0])
def test_requant_on_near_ties_is_the_scalar_definition(epi_lib, form, zp, lo):
    rng = np.random.default_rng(11 + zp + lo)
    n = 8192
    acc, bd, mu = _requant_operands(rng, n, zp, lo)
    want = _requant_ref(acc, bd, mu, zp, lo)
    assert (want != _requant_ref(acc, bd, mu, zp, lo, fused=True)).sum() > 1000          # adversarial for contraction
    assert (want == lo).any() and (want == 255).any()
    got = np.empty(n * 16, np.uint8)
    assert epi_lib.run(0, form, n, acc.ctypes.data, None, bd.ctypes.data, mu.ctypes.data, None, None, zp, lo,
                       got.ctypes.data) == 0
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, f"{bad.size} bytes differ, first at {bad[0]}: got {got[bad[0]]} want {want[bad[0]]}"


FLAVOURS = {   # (a_scale, r_scale, add_scale, out_zp, res_zp, add_zp): tests/test_epilogue_math.py's two qconfigs
    "fbgemm_reduce_range": (0.0391, 0.0208, 0.0311, 67, 58, 0),
    "main_py_full_range": (0.0197, 0.0101, 0.0159, 133, 117, 0),
}


def _add_relu_ref(acc, r, bd, mu, f, z, fused1=False, fused2=False):
    """Scalar definition of epilogue16_i8_res (general form; the fast form equals it for out_lo == 0), per element."""
    a_s, r_s, inv = (np.repeat(f[:, i], 16) for i in range(3))
    out_zp, res_zp, add_zp, out_lo = (np.repeat(z[:, i], 16) for i in range(4))
    t = _f32(acc.astype(np.float32) + bd)
    t = np.rint(t.astype(np.float64) * mu) if fused1 else np.rint(_f32(t * mu))
    q2 = np.clip(t + out_zp, out_lo, 255)
    a = _fma(a_s, _f32(q2), _f32(a_s * _f32(-out_zp)))
    rb = _fma(r_s, _f32(r), _f32(r_s * _f32(-res_zp)))
    s = np.maximum(_f32(a + rb), np.float32(0))
    u = np.rint(s.astype(np.float64) * inv) if fused2 else np.rint(_f32(s * inv))
    return np.clip(u + add_zp, 0, 255).astype(np.uint8)


def _add_relu_operands(rng, n, flavour):
    a_s0, r_s0, add_s0, out_zp, res_zp, add_zp = FLAVOURS[flavour]
    jit = lambda x: _f32(x * (1 + 0.2 * (rng.random(n) - 0.5)))
    f = np.stack([jit(a_s0), jit(r_s0), _f32(1) / jit(add_s0)], 1)
    z = np.tile(np.array([out_zp, res_zp, add_zp, 0], np.int32), (n, 1))
    m = n * 16
    acc = rng.integers(-60_000, 60_000, m).astype(np.int32)
    acc[acc == 0] = 1
    bd = _f32(rng.standard_normal(m) * 40)
    t = _f32(acc.astype(np.float32) + bd)
    mu = _near_ties(rng, t, -out_zp - 2, 255 - out_zp + 2)    # even slots: the conv's own requantisation near ties
    r = rng.integers(0, 256, m).astype(np.uint8)
    # odd slots: an exact conv value q2 and a residual byte, with a per-thread 1/add_scale that puts the sum's scaled
    # value within a few ulps of a .5 point (the add's magic-number rounding)
    q2 = rng.integers(0, 256, n)
    rb = rng.integers(0, 256, n)
    s = _f32(_fma(f[:, 0], _f32(q2), _f32(f[:, 0] * _f32(-out_zp))) + _fma(f[:, 1], _f32(rb), _f32(f[:, 1] * _f32(-res_zp))))
    ok = s > 0                                                 # a closed ReLU is covered by the even slots
    f[ok, 2] = _near_ties(rng, s[ok], 0, 255 - add_zp)
    odd = np.zeros(m, bool)
    odd[1::2] = True
    sel = odd & np.repeat(ok, 16)
    acc[sel] = np.repeat(q2 - out_zp, 16)[sel]
    bd[sel], mu[sel] = 0, 1
    r[sel] = np.repeat(rb, 16)[sel]
    return acc, r, bd, mu, f, z


@pytest.mark.gpu
@pytest.mark.parametrize("flavour", list(FLAVOURS))
@pytest.mark.parametrize("res_form", [1, 2])
@pytest.mark.parametrize("form", [1, 0])
def test_add_relu_on_near_ties_is_the_scalar_definition(epi_lib, form, res_form, flavour):
    rng = np.random.default_rng(5 + res_form + 7 * len(flavour))
    n = 8192
    acc, r, bd, mu, f, z = _add_relu_operands(rng, n, flavour)
    want = _add_relu_ref(acc, r, bd, mu, f, z)
    assert (want != _add_relu_ref(acc, r, bd, mu, f, z, fused1=True)).sum() > 500
    assert (want != _add_relu_ref(acc, r, bd, mu, f, z, fused2=True)).sum() > 500
    assert (want == 0).any() and (want == 255).any()
    got = np.empty(n * 16, np.uint8)
    assert epi_lib.run(res_form, form, n, acc.ctypes.data, r.ctypes.data, bd.ctypes.data, mu.ctypes.data, f.ctypes.data,
                       z.ctypes.data, 0, 0, got.ctypes.data) == 0
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, f"{bad.size} bytes differ, first at {bad[0]}: got {got[bad[0]]} want {want[bad[0]]}"
