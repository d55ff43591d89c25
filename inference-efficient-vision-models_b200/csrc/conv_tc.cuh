// Implicit-GEMM convolution on tcgen05 tensor cores (sm_100a).
//
//   D[pixel, cout] = sum_{tap, cin} A[pixel, (tap, cin)] * W[cout, (tap, cin)]
//
// * A tiles (128 consecutive output pixels in (n, oy, ox) order x one channel chunk of one filter tap)
//   are gathered straight from the NHWC activation tensor by TMA in im2col mode; spatial padding and
//   the ragged last tile are zero-filled by the TMA unit (zero == the real value 0 because every
//   tensor-core layer's input zero-point is 0, checked at engine creation).
// * W tiles come from a pre-packed K-major [cout_pad][taps * cin_chunks * kc] matrix by tiled TMA;
//   when the whole matrix fits in shared memory it is loaded once per CTA and stays resident.
// * Both land in shared memory in the 64B/128B-swizzled K-major layout tcgen05.mma reads directly.
// * Accumulators (int32 for kind::i8, fp32 for kind::f16) live in TMEM, double buffered so that the
//   epilogue of tile i overlaps the MMAs of tile i+1; the kernel is persistent (grid <= #SMs).
// * The epilogue is fused: INT8 requantisation (+ReLU clamp) and, for a block's last conv, the whole
//   quantized::add_relu with the residual; FP16 bias (+residual) (+ReLU).
//
// Warp roles (576 threads): warp 0 = TMA producer, warp 1 = TMEM owner + MMA issuer,
// warps 2..17 = epilogue, organised as FOUR GROUPS of four warps (one per TMEM lane quadrant, = warp % 4).
// A group owns whole tiles (tile sequence number % 4 == group) and walks all of the tile's 16-column chunks;
// accumulators sit in a ring of up to eight TMEM buffers.  The groups therefore run out of phase with one
// another and with the MMA warp: the conversion / float / integer pipes see a steady mix instead of sixteen
// warps hitting the same pipe at the same moment, a group's TMEM-load and residual-fetch latency hides behind
// the other groups' arithmetic, and the per-tile bookkeeping is paid once per 128 x bn outputs per warp.
#pragma once
#include <cuda_fp16.h>

#include <type_traits>

#include "ptx.cuh"

namespace ievm {

constexpr int kTileM = 128;
#ifndef IEVM_EPI_WARPS
#define IEVM_EPI_WARPS 16      // multiple of 4 whose quarter is a power of two: 8 or 16 (A/B builds)
#endif
constexpr int kEpiWarps = IEVM_EPI_WARPS;
constexpr int kEpiSub = kEpiWarps / 4;     // epilogue warps per TMEM lane quadrant (stem_tc.cuh: they interleave chunks)
constexpr int kEpiGroups = kEpiWarps / 4;  // conv_tc_kernel: groups of four warps, each owning every 4th tile
constexpr int kMaxAcc = 8;                 // accumulator buffers in TMEM (512 columns / 64)
constexpr int kConvThreads = 64 + 32 * kEpiWarps;

enum : int { kDtypeI8 = 0, kDtypeF16 = 1 };
// A-operand feeding modes.
//  kModeIm2col: one im2col TMA per (filter tap, channel chunk) -- any 1x1/3x3, stride 1|2.
//  kModeHalo  : 3x3 stride-1 pad-1 convs whose pixel fits one smem row (<= 128 B).  The image is cut into BANDS of
//               S sub-tiles; a sub-tile is R = floor(128 / (W+2)) whole output rows = R*(W+2) consecutive positions
//               of the halo-extended row-major space (<= 128 MMA rows, the remainder are junk lanes).  ONE tiled
//               TMA box brings the band's (S*R+2) x (W+2) input patch with zero-filled borders; every sub-tile's
//               nine taps are nine row-shifted views of that patch (descriptor start + (sub*R*(W+2) + ky*(W+2)+kx)
//               rows), all with compile-time-like constant offsets because sub-tiles are row aligned.
//               Why bands: a tcgen05.mma queue is only ~1-2 instructions deep and every mbarrier test by the issuing
//               thread costs ~150 clk of idle tensor pipe (profiles/r02_mma_convlike.txt); with S sub-tiles per
//               patch the issuer pays one batched barrier test per S*9*ksteps instructions, the patch is re-read
//               (S*R+2)/(S*R) times instead of 2.7x, and one TMA replaces S.
enum : int { kModeIm2col = 0, kModeHalo = 1 };
constexpr int kMaxBandSubs = 4;
constexpr int kEpConst = 128;
// Halo-mode shape classes.  For the shapes the networks of this path actually have, (W+2, row bytes, N) are template
// constants, so that every descriptor offset of a sub-tile's 18 / 36 instructions is an immediate added to ONE uniform
// base register.  With run-time offsets ptxas keeps the nine tap offsets in vector registers and pays ~20 R2UR moves
// (~200 cycles of idle tensor pipe) per sub-tile.  Class 0 is the generic run-time fallback.
//   1: 56x56 x 64-byte pixels, N = 64 (INT8 layer 1)     2: 28x28 x 128-byte pixels, N = 128 (INT8 layer 2)
//   3: 56x56 x 128-byte pixels, N = 64 (FP16 layer 1)
constexpr int kHaloShapes = 4;
__host__ __device__ constexpr int halo_shape_wp(int s) { return s == 1 ? 58 : s == 2 ? 30 : s == 3 ? 58 : 0; }
__host__ __device__ constexpr int halo_shape_rb(int s) { return s == 1 ? 64 : s == 2 ? 128 : s == 3 ? 128 : 0; }
__host__ __device__ constexpr int halo_shape_bn(int s) { return s == 1 ? 64 : s == 2 ? 128 : s == 3 ? 64 : 0; }
inline int halo_shape_class(int wp, int rb, int bn) {
  for (int s = 1; s < kHaloShapes; ++s)
    if (halo_shape_wp(s) == wp && halo_shape_rb(s) == rb && halo_shape_bn(s) == bn) return s;
  return 0;
}

struct ConvTcParams {
  // implicit-GEMM geometry
  int m_total;         // n * ho * wo
  int ho, wo;
  int stride, pad, ksize;
  int phase_bytes;           // conv_s2.cuh: bytes of one phase buffer of a patch stage
  int kw, stride_w, pad_w;   // conv_dual.cuh, pixel-pair form: taps / stride / padding along W when they differ from H (kw == 0: same)
  int kchunks;         // channel chunks per filter tap
  int kc_bytes;        // bytes per smem row == bytes per channel chunk (64 or 128)
  int kc_elems;
  int bn;              // UMMA N (multiple of 16, <= 256)
  int n_tiles, m_tiles;
  int stages;
  int resident_b;      // 1: all weight k-blocks stay in shared memory (n_tiles == 1)
  int a_stage_bytes;   // distance between A stages in shared memory
  int a_tx_bytes;      // bytes one A-operand TMA delivers
  int kb_group;        // im2col mode: k-blocks per pipeline stage (one full/empty barrier pair per group)
  // halo (band) mode
  int h_in, w_in, wp;  // input height / width, wp = w_in + 2
  int sub_rows;        // R: output rows per sub-tile
  int sub_pos;         // R * wp: MMA rows of a sub-tile that are real positions
  int subs_per_img;    // T = ceil(h_in / R)
  int band_subs;       // S: sub-tiles per band (<= kMaxBandSubs, <= nacc)
  int total_subs;      // n * T
  uint32_t spi_magic, wp_magic, hw_magic, wo_magic;   // ceil(2^32 / d), or 0 = divide normally: see fast_div
  int tmem_cols;       // power of two >= 32 covering the accumulator ring
  int acc_stride;      // column distance between accumulator buffers (power of two >= bn)
  int nacc;            // accumulator buffers in the ring (2 .. kMaxAcc)
  int fast_round;      // i8: |requantised value| < 2^21 for every possible input (checked at engine creation), so
                       // round-to-nearest-even may use the 1.5*2^23 magic add instead of F2I (8 cycles/warp on B200)
  int cout_pad;        // n_tiles * bn
  uint32_t idesc;
  // epilogue
  void* out;
  int out_pitch;       // elements per output pixel row (== padded cout)
  const void* res;     // residual tensor (same pixel indexing), or nullptr
  int res_pitch;
  const float* ep0;    // i8: bias / (x_scale * w_scale[c]);  f16: folded bias
  const float* ep1;    // i8: (x_scale * w_scale[c]) / out_scale
  int out_zp, out_lo;  // i8: zero point of the conv's own output and its lower clamp (zp if ReLU else 0)
  float a_scale;       // i8 residual path: scale of the conv's own output
  float res_scale;
  int res_zp;
  float inv_add_scale; // 1 / scale of quantized::add_relu's output
  int add_zp;
  int relu;            // f16: apply ReLU at the end
  // Input zero point != 0 (never the case for the post-ReLU tensors of a ResNet, but any qconfig the reference's
  // quantization/main.py:187-222 style can produce with a non-ReLU conv input): TMA fills padding with the integer 0, so
  // the tensor core computes sum_{in-bounds taps} x * w; the true accumulator is sum (x - zp) * w over the same taps.
  // zcorr[cls][cout_pad] = zp * sum_{taps of class cls} sum_ci w, cls = (row-tap mask << ksize) | column-tap mask.
  const int32_t* zcorr;
  int32_t* dump_acc;   // debug: raw accumulators [m_total][dump_pitch] (bit pattern for f16)
  int dump_pitch;
  unsigned int* stuck_flag;   // mapped host word; written before a bounded wait gives up
  // The same per-channel tables as ep0 / ep1 inside the kernel-parameter block (filled when cout_pad <= kEpConst): the
  // statically shaped halo kernels unroll their chunk loop, so every table entry becomes a constant-bank operand of the
  // FADD / FMUL that uses it -- no shared-memory loads (and no short-scoreboard stalls behind them) in the epilogue.
  float epc0[128];
  float epc1[128];
#ifdef IEVM_EXP_TIMING
  int timing_slot;     // A/B instrumentation: where this launch's per-CTA role timers go (g_exp_timing)
#endif
};

// n / d.  magic = ceil(2^32 / d) is exact while n * d < 2^32; the host passes magic = 0 (plain division) when
// the largest n of the launch could violate that, or when d == 1.
__device__ __forceinline__ int fast_div(int n, int d, uint32_t magic) {
  return magic ? static_cast<int>(__umulhi(static_cast<uint32_t>(n), magic)) : n / d;
}

__device__ __forceinline__ void wait_or_die(uint64_t* bar, uint32_t parity, uint32_t code, unsigned int* flag) {
  if (mbar_try_wait(bar, parity)) return;
  const uint64_t t0 = globaltimer_ns();
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 0x3ff) == 0 && globaltimer_ns() - t0 > IEVM_WAIT_LIMIT_NS) {
      if (flag) {
        *reinterpret_cast<volatile unsigned int*>(flag) = code;
        __threadfence_system();
      }
      __trap();
    }
  }
}
// The same with the bounded spin OUT OF LINE: a wait site is one try_wait (which already parks the warp for up to the
// suspend hint), a branch and a rarely taken call instead of thirty instructions of slow path inside a pipeline loop --
// instruction fetch is a first-order cost in these kernels.  For kernels with registers to spare only (the fused front
// end: 81.5 -> 79.5 us): at the 96-register cap of the conv kernels the call's register saves spill (56 -> 61 us).
__device__ __noinline__ void wait_or_die_slow(uint64_t* bar, uint32_t parity, uint32_t code, unsigned int* flag) {
  const uint64_t t0 = globaltimer_ns();
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 0x3ff) == 0 && globaltimer_ns() - t0 > IEVM_WAIT_LIMIT_NS) {
      if (flag) {
        *reinterpret_cast<volatile unsigned int*>(flag) = code;
        __threadfence_system();
      }
      __trap();
    }
  }
}
__device__ __forceinline__ void wait_or_die_ool(uint64_t* bar, uint32_t parity, uint32_t code, unsigned int* flag) {
  if (mbar_try_wait(bar, parity)) return;
  wait_or_die_slow(bar, parity, code, flag);
}

#ifdef IEVM_EXP_TIMING
// [slot][cta][16]: 0 mma loop clk, 1 mma wait tempty, 2 mma wait full, 3 mma loop ns, 4 producer loop clk, 5 producer wait empty,
// 6 epilogue(warp 2) loop clk, 7 epilogue wait tfull, 8 tiles of this CTA, 9 whole-kernel clk (warp 1), 10 whole-kernel ns
constexpr int kExpSlots = 32, kExpCtas = 160, kExpWords = 16;
__device__ unsigned long long g_exp_timing[kExpSlots * kExpCtas * kExpWords];
#define IEVM_TIMED_WAIT(acc, ...)                 \
  do {                                            \
    const long long t__ = clock64();              \
    wait_or_die(__VA_ARGS__);                     \
    acc += clock64() - t__;                       \
  } while (0)
#else
#define IEVM_TIMED_WAIT(acc, ...) wait_or_die(__VA_ARGS__)
#endif

// ---- INT8 epilogue arithmetic: float32, no FMA contraction, round-half-even (== fbgemm/ATen) ----
// Scalar forms (used by the CUDA-core kernels and as the definition the fast forms must equal).
__device__ __forceinline__ int requant_i8(int acc, float bdiv, float mult, int zp, int lo) {
  const float v = __fmul_rn(__fadd_rn(__int2float_rn(acc), bdiv), mult);
  const int q = __float2int_rn(v) + zp;
  return min(max(q, lo), 255);
}
__device__ __forceinline__ int add_relu_i8(int aq, int a_zp, float a_scale, int rq, int r_zp, float r_scale,
                                           float inv_scale, int zp) {
  // ATen's vectorised qadd dequantises with ONE fused multiply-add against a pre-rounded product,
  // fma(scale, float(q), fl(scale * -zp)) (Vectorized<quint8>::dequantize), not (q - zp) * scale: the two differ by an
  // ulp often enough to move ~1e-5 of the outputs by one LSB when both zero points are large (oracle/int8_forward.py).
  const float a = __fmaf_rn(a_scale, __int2float_rn(aq), __fmul_rn(a_scale, -__int2float_rn(a_zp)));
  const float b = __fmaf_rn(r_scale, __int2float_rn(rq), __fmul_rn(r_scale, -__int2float_rn(r_zp)));
  const float s = fmaxf(__fadd_rn(a, b), 0.0f);
  const int q = __float2int_rn(__fmul_rn(s, inv_scale)) + zp;
  return min(max(q, 0), 255);
}

// (sat_u8(a) << 8 | sat_u8(b)) | c << 16 : two saturating int32 -> u8 conversions per instruction.
__device__ __forceinline__ uint32_t pack_sat_u8(int a_hi, int b_lo, uint32_t c_upper) {
  uint32_t d;
  asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a_hi), "r"(b_lo), "r"(c_upper));
  return d;
}
__device__ __forceinline__ uint32_t pack4_sat_u8(int q0, int q1, int q2, int q3) {
  return pack_sat_u8(q1, q0, pack_sat_u8(q3, q2, 0u));
}

constexpr float kRoundMagic = 12582912.0f;   // 1.5 * 2^23: (x + M) - M == rint(x) for |x| < 2^22

// Per-thread constants of the fused add_relu epilogue.
struct AddReluConst {
  float lo_f, hi_f;        // clamp of the conv's own requantised value, relative to its zero point
  float a_scale, r_scale, inv_scale;
  float pa, pb;            // fl(a_scale * -out_zp), fl(r_scale * -res_zp): addends of ATen's fused dequantisation
  float lo_q, zp_f;        // float(out_lo), float(out_zp)
  int add_zp;
  // fast form (magic-number rounding allowed): integer clamps done by one VIADDMNMX.RELU each
  int c1_add, c1_max;      // clamp(rne(v), lo, hi) - lo == max(min(bits(v + M) + c1_add, c1_max), 0)
  int c2_add, c2_max;      // q - add_zp          == max(min(bits(u + M) + c2_add, c2_max), 0)
  uint32_t zp4;            // add_zp in every byte
};

// rne(x) + zp as an integer.  kFast: (x + 1.5*2^23) rounds to an integer with ties to even (the magic constant is
// even), and its bit pattern minus the constant's is that integer -- one FADD + one IADD instead of F2I.
constexpr int kRoundMagicBits = 0x4B400000;
template <bool kFast>
__device__ __forceinline__ int round_add(float x, int zp) {
  if (kFast) return __float_as_int(__fadd_rn(x, 12582912.0f)) + (zp - kRoundMagicBits);
  return __float2int_rn(x) + zp;
}
// max(rne(x) + zp, lo): with the magic add the integer add and the lower clamp are ONE instruction (VIADDMNMX).
template <bool kFast>
__device__ __forceinline__ int round_add_max(float x, int zp, int lo) {
  if (kFast) return __viaddmax_s32(__float_as_int(__fadd_rn(x, 12582912.0f)), zp - kRoundMagicBits, lo);
  return max(__float2int_rn(x) + zp, lo);
}

#ifndef IEVM_EXP_SCALAR_EPI
// Paired forms (default): values 2j and 2j + 1 of a chunk go through one FADD2 / FMUL2 / FFMA2 (add/mul/fma.rn.f32x2),
// each lane rounded exactly like the scalar op, so the arithmetic is the scalar definition's, op for op.
//
// Contraction fence: ptxas contracts mul.rn.f32x2 followed by add.rn.f32x2 into one FFMA2 although both carry .rn (it
// never does this to scalar mul.rn / add.rn), also under -fmad=false.  fl(x * mu + M) differs from fl(fl(x * mu) + M)
// whenever the exact product lies within half an ulp of a .5 point, so every multiply whose result feeds the
// magic-number add is written as fma(x, mu, -0) instead: equal to fl(x * mu) for every input (+-0 + -0 keeps the sign of
// a zero product, every other sum is the product), and an FFMA2 has nothing left to contract.  The -0 comes from the
// constant bank, so ptxas cannot fold the fma back into a multiply; it is an FFMA2 operand (uniform register), and the
// fence costs no instruction.
__constant__ float2 g_neg_zero2 = {-0.0f, -0.0f};
__device__ __forceinline__ float2 fmul2_fenced(float2 a, float2 b) { return __ffma2_rn(a, b, g_neg_zero2); }
__device__ __forceinline__ float2 splat2(float a) { return make_float2(a, a); }
__device__ __forceinline__ float2 i2f2(uint32_t a, uint32_t b) {
  return make_float2(__int2float_rn(static_cast<int>(a)), __int2float_rn(static_cast<int>(b)));
}

// 16 accumulators -> 16 requantised bytes (no residual).
template <bool kFast>
__device__ __forceinline__ uint4 epilogue16_i8(const uint32_t (&v)[16], const float* s_bd, const float* s_mu, int zp,
                                               int lo) {
  int q[16];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float4 b4 = *reinterpret_cast<const float4*>(s_bd + 4 * j);
    const float4 m4 = *reinterpret_cast<const float4*>(s_mu + 4 * j);
    const float2 bd[2] = {make_float2(b4.x, b4.y), make_float2(b4.z, b4.w)};
    const float2 mu[2] = {make_float2(m4.x, m4.y), make_float2(m4.z, m4.w)};
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int i = 4 * j + 2 * h;
      const float2 t = __fadd2_rn(i2f2(v[i], v[i + 1]), bd[h]);
      if (kFast) {
        const float2 u = __fadd2_rn(fmul2_fenced(t, mu[h]), splat2(kRoundMagic));
        q[i] = __viaddmax_s32(__float_as_int(u.x), zp - kRoundMagicBits, lo);
        q[i + 1] = __viaddmax_s32(__float_as_int(u.y), zp - kRoundMagicBits, lo);
      } else {
        const float2 u = __fmul2_rn(t, mu[h]);
        q[i] = max(__float2int_rn(u.x) + zp, lo);
        q[i + 1] = max(__float2int_rn(u.y) + zp, lo);
      }
    }
  }
  return make_uint4(pack4_sat_u8(q[0], q[1], q[2], q[3]), pack4_sat_u8(q[4], q[5], q[6], q[7]),
                    pack4_sat_u8(q[8], q[9], q[10], q[11]), pack4_sat_u8(q[12], q[13], q[14], q[15]));
}

// 16 accumulators + 16 residual bytes -> 16 bytes of quantized::add_relu(requant(acc), residual).
// All float steps reproduce the scalar definition exactly: clamping before rounding commutes with
// RNE because the clamp bounds are integers, and (x + M) - M is RNE for |x| <= 256.
template <bool kFast, bool kResI2F = false>
__device__ __forceinline__ uint4 epilogue16_i8_res(const uint32_t (&v)[16], const uint4 r4, const float* s_bd,
                                                   const float* s_mu, const AddReluConst& k) {
  const uint32_t rw[4] = {r4.x, r4.y, r4.z, r4.w};
  int q[16];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float4 b4 = *reinterpret_cast<const float4*>(s_bd + 4 * j);
    const float4 m4 = *reinterpret_cast<const float4*>(s_mu + 4 * j);
    const float2 bd[2] = {make_float2(b4.x, b4.y), make_float2(b4.z, b4.w)};
    const float2 mu[2] = {make_float2(m4.x, m4.y), make_float2(m4.z, m4.w)};
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int i = 4 * j + 2 * h;
      float2 t = __fadd2_rn(i2f2(v[i], v[i + 1]), bd[h]);
      // dequantised residual bytes 2h, 2h + 1 of the word (the two forms of float(byte): see the scalar form below)
      const float2 rbyte =
          kResI2F ? make_float2(static_cast<float>((rw[j] >> (16 * h)) & 0xffu), static_cast<float>((rw[j] >> (16 * h + 8)) & 0xffu))
                  : __fadd2_rn(make_float2(__uint_as_float(__byte_perm(rw[j], 0x4B400000u, 0x7650 + 2 * h)),
                                           __uint_as_float(__byte_perm(rw[j], 0x4B400000u, 0x7651 + 2 * h))),
                               splat2(-kRoundMagic));
      const float2 rb = __ffma2_rn(splat2(k.r_scale), rbyte, splat2(k.pb));
      if (kFast) {
        t = __fadd2_rn(fmul2_fenced(t, mu[h]), splat2(kRoundMagic));
        const int tq0 = __viaddmin_s32_relu(__float_as_int(t.x), k.c1_add, k.c1_max);   // q2 - lo (lo == 0 here)
        const int tq1 = __viaddmin_s32_relu(__float_as_int(t.y), k.c1_add, k.c1_max);
        const float2 a = __ffma2_rn(splat2(k.a_scale), make_float2(__int2float_rn(tq0), __int2float_rn(tq1)), splat2(k.pa));
        const float2 u = __fadd2_rn(fmul2_fenced(__fadd2_rn(a, rb), splat2(k.inv_scale)), splat2(kRoundMagic));
        q[i] = __viaddmin_s32_relu(__float_as_int(u.x), k.c2_add, k.c2_max);                  // q - add_zp
        q[i + 1] = __viaddmin_s32_relu(__float_as_int(u.y), k.c2_add, k.c2_max);
      } else {
        // the clamps (FMNMX) stand between the multiply and the magic-number adds: nothing here can be contracted
        t = __fmul2_rn(t, mu[h]);
        t = make_float2(fminf(fmaxf(t.x, k.lo_f), k.hi_f), fminf(fmaxf(t.y, k.lo_f), k.hi_f));
        t = __fadd2_rn(__fadd2_rn(t, splat2(kRoundMagic)), splat2(-kRoundMagic));   // == float(q2 - zp2)
        const float2 a = __ffma2_rn(splat2(k.a_scale), __fadd2_rn(t, splat2(k.zp_f)), splat2(k.pa));
        const float2 s = __fadd2_rn(a, rb);
        const float2 u = __fmul2_rn(make_float2(fmaxf(s.x, 0.0f), fmaxf(s.y, 0.0f)), splat2(k.inv_scale));
        q[i] = __float2int_rn(u.x) + k.add_zp;
        q[i + 1] = __float2int_rn(u.y) + k.add_zp;
      }
    }
  }
  uint4 o = make_uint4(pack4_sat_u8(q[0], q[1], q[2], q[3]), pack4_sat_u8(q[4], q[5], q[6], q[7]),
                       pack4_sat_u8(q[8], q[9], q[10], q[11]), pack4_sat_u8(q[12], q[13], q[14], q[15]));
  if (kFast) {     // bytes hold q - add_zp <= 255 - add_zp: the per-byte add cannot carry
    o.x += k.zp4;
    o.y += k.zp4;
    o.z += k.zp4;
    o.w += k.zp4;
  }
  return o;
}

#else   // IEVM_EXP_SCALAR_EPI: the scalar forms, one FADD / FMUL / FFMA per value (A/B build, scripts/build_ab.py)

// 16 accumulators -> 16 requantised bytes (no residual).
template <bool kFast>
__device__ __forceinline__ uint4 epilogue16_i8(const uint32_t (&v)[16], const float* s_bd, const float* s_mu, int zp,
                                               int lo) {
  int q[16];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float4 b4 = *reinterpret_cast<const float4*>(s_bd + 4 * j);
    const float4 m4 = *reinterpret_cast<const float4*>(s_mu + 4 * j);
    q[4 * j + 0] = round_add_max<kFast>(__fmul_rn(__fadd_rn(__int2float_rn(static_cast<int>(v[4 * j + 0])), b4.x), m4.x), zp, lo);
    q[4 * j + 1] = round_add_max<kFast>(__fmul_rn(__fadd_rn(__int2float_rn(static_cast<int>(v[4 * j + 1])), b4.y), m4.y), zp, lo);
    q[4 * j + 2] = round_add_max<kFast>(__fmul_rn(__fadd_rn(__int2float_rn(static_cast<int>(v[4 * j + 2])), b4.z), m4.z), zp, lo);
    q[4 * j + 3] = round_add_max<kFast>(__fmul_rn(__fadd_rn(__int2float_rn(static_cast<int>(v[4 * j + 3])), b4.w), m4.w), zp, lo);
  }
  return make_uint4(pack4_sat_u8(q[0], q[1], q[2], q[3]), pack4_sat_u8(q[4], q[5], q[6], q[7]),
                    pack4_sat_u8(q[8], q[9], q[10], q[11]), pack4_sat_u8(q[12], q[13], q[14], q[15]));
}

// 16 accumulators + 16 residual bytes -> 16 bytes of quantized::add_relu(requant(acc), residual).
// All float steps reproduce the scalar definition exactly: clamping before rounding commutes with
// RNE because the clamp bounds are integers, and (x + M) - M is RNE for |x| <= 256.
template <bool kFast, bool kResI2F = false>
__device__ __forceinline__ uint4 epilogue16_i8_res(const uint32_t (&v)[16], const uint4 r4, const float* s_bd,
                                                   const float* s_mu, const AddReluConst& k) {
  const uint32_t rw[4] = {r4.x, r4.y, r4.z, r4.w};
  int q[16];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float4 b4 = *reinterpret_cast<const float4*>(s_bd + 4 * j);
    const float4 m4 = *reinterpret_cast<const float4*>(s_mu + 4 * j);
    const float bd[4] = {b4.x, b4.y, b4.z, b4.w};
    const float mu[4] = {m4.x, m4.y, m4.z, m4.w};
#pragma unroll
    for (int b = 0; b < 4; ++b) {
      const int i = 4 * j + b;
      float t = __fmul_rn(__fadd_rn(__int2float_rn(static_cast<int>(v[i])), bd[b]), mu[b]);
      // dequantised residual: (magic | byte) - magic == float(byte), then fma(s_r, byte, fl(s_r * -zp_r)) as ATen does
      // float(byte): (magic | byte) - magic is PRMT + FADD, two issue slots on the ALU and FMA pipes; I2F.U8 with a byte
      // selector is one slot on the 4-cycle conversion pipe, which the two I2Fs of the requantisation already load.
      // Measured: the unrolled 64-channel kernels are faster with the first form (58 vs 60 us), the 128-channel loop
      // kernels with the second (39 vs 41 us) -- kResI2F picks per instantiation.  Both are exact.
      const float rbyte = kResI2F ? static_cast<float>((rw[j] >> (8 * b)) & 0xffu)
                                  : __fadd_rn(__uint_as_float(__byte_perm(rw[j], 0x4B400000u, 0x7650 + b)), -kRoundMagic);
      const float rb = __fmaf_rn(k.r_scale, rbyte, k.pb);
      if (kFast) {
        // Integer clamps after the magic-number rounding: rne commutes with clamping to integer bounds, and
        // max(s, 0) before the final scaling equals clamping the rounded value at 0 (the scale is positive), so
        // each clamp pair is ONE add-min-relu instruction instead of two FMNMX (the ALU pipe issues at half rate).
        const int tq = __viaddmin_s32_relu(__float_as_int(__fadd_rn(t, kRoundMagic)), k.c1_add, k.c1_max);   // q2 - lo
        // the fast form is only enabled for a conv without its own ReLU (lower clamp 0: every residual conv of a ResNet),
        // so q2 == tq and the float(lo) addend is gone
        const float a = __fmaf_rn(k.a_scale, __int2float_rn(tq), k.pa);                                      // fma(s2, q2, fl(s2 * -zp2))
        const float u = __fmul_rn(__fadd_rn(a, rb), k.inv_scale);
        q[i] = __viaddmin_s32_relu(__float_as_int(__fadd_rn(u, kRoundMagic)), k.c2_add, k.c2_max);          // q - add_zp
      } else {
        t = fminf(fmaxf(t, k.lo_f), k.hi_f);
        t = __fadd_rn(__fadd_rn(t, kRoundMagic), -kRoundMagic);          // == float(q2 - zp2)
        const float a = __fmaf_rn(k.a_scale, __fadd_rn(t, k.zp_f), k.pa);
        const float s = fmaxf(__fadd_rn(a, rb), 0.0f);
        q[i] = __float2int_rn(__fmul_rn(s, k.inv_scale)) + k.add_zp;
      }
    }
  }
  uint4 o = make_uint4(pack4_sat_u8(q[0], q[1], q[2], q[3]), pack4_sat_u8(q[4], q[5], q[6], q[7]),
                       pack4_sat_u8(q[8], q[9], q[10], q[11]), pack4_sat_u8(q[12], q[13], q[14], q[15]));
  if (kFast) {     // bytes hold q - add_zp <= 255 - add_zp: the per-byte add cannot carry
    o.x += k.zp4;
    o.y += k.zp4;
    o.z += k.zp4;
    o.w += k.zp4;
  }
  return o;
}
#endif   // IEVM_EXP_SCALAR_EPI

template <bool kHasRes, bool kRelu>
__device__ __forceinline__ void epilogue16_f16(const uint32_t (&v)[16], const float* s_bias, const __half* rp,
                                               __half* op, bool valid) {
  float f[16];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float4 b4 = *reinterpret_cast<const float4*>(s_bias + 4 * j);
    f[4 * j] = __uint_as_float(v[4 * j]) + b4.x;
    f[4 * j + 1] = __uint_as_float(v[4 * j + 1]) + b4.y;
    f[4 * j + 2] = __uint_as_float(v[4 * j + 2]) + b4.z;
    f[4 * j + 3] = __uint_as_float(v[4 * j + 3]) + b4.w;
  }
  if (kHasRes && valid) {
    const uint4 r0 = *reinterpret_cast<const uint4*>(rp);
    const uint4 r1 = *reinterpret_cast<const uint4*>(rp + 8);
    const uint32_t rw[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float2 r2 = __half22float2(*reinterpret_cast<const __half2*>(&rw[j]));
      f[2 * j] += r2.x;
      f[2 * j + 1] += r2.y;
    }
  }
  uint32_t hw2[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    float x = f[2 * j], y = f[2 * j + 1];
    if (kRelu) {
      x = fmaxf(x, 0.0f);
      y = fmaxf(y, 0.0f);
    }
    const __half2 h = __floats2half2_rn(x, y);
    hw2[j] = *reinterpret_cast<const uint32_t*>(&h);
  }
  if (valid) {
    *reinterpret_cast<uint4*>(op) = make_uint4(hw2[0], hw2[1], hw2[2], hw2[3]);
    *reinterpret_cast<uint4*>(op + 8) = make_uint4(hw2[4], hw2[5], hw2[6], hw2[7]);
  }
}

// The same with the residual's 16 halves already in registers (fetched a chunk ahead, like the INT8 residual bytes: the
// in-place loads above expose an L2 round trip per chunk -- 98 vs 66 us for the FP16 layer-1 convs with / without residual).
template <bool kRelu>
__device__ __forceinline__ void epilogue16_f16_pre(const uint32_t (&v)[16], const float* s_bias, const uint4 r0, const uint4 r1,
                                                   __half* op, bool valid) {
  float f[16];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float4 b4 = *reinterpret_cast<const float4*>(s_bias + 4 * j);
    f[4 * j] = __uint_as_float(v[4 * j]) + b4.x;
    f[4 * j + 1] = __uint_as_float(v[4 * j + 1]) + b4.y;
    f[4 * j + 2] = __uint_as_float(v[4 * j + 2]) + b4.z;
    f[4 * j + 3] = __uint_as_float(v[4 * j + 3]) + b4.w;
  }
  const uint32_t rw[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float2 r2 = __half22float2(*reinterpret_cast<const __half2*>(&rw[j]));
    f[2 * j] += r2.x;
    f[2 * j + 1] += r2.y;
  }
  uint32_t hw2[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    float x = f[2 * j], y = f[2 * j + 1];
    if (kRelu) {
      x = fmaxf(x, 0.0f);
      y = fmaxf(y, 0.0f);
    }
    const __half2 h = __floats2half2_rn(x, y);
    hw2[j] = *reinterpret_cast<const uint32_t*>(&h);
  }
  if (valid) {
    *reinterpret_cast<uint4*>(op) = make_uint4(hw2[0], hw2[1], hw2[2], hw2[3]);
    *reinterpret_cast<uint4*>(op + 8) = make_uint4(hw2[4], hw2[5], hw2[6], hw2[7]);
  }
}

// One 16-column chunk of the epilogue for pixel row `m`.
// Residual bytes for one 16-channel chunk of pixel row m (INT8), fetched ahead of the TMEM load so
// that the L2 latency is hidden behind the wait for the accumulator.
__device__ __forceinline__ uint4 load_res16_i8(const ConvTcParams& p, int m, bool valid, int ch) {
  if (!valid) return make_uint4(0u, 0u, 0u, 0u);
  return __ldg(reinterpret_cast<const uint4*>(static_cast<const uint8_t*>(p.res) + static_cast<size_t>(m) * p.res_pitch + ch));
}

// FP16: the residual's 16 halves of one chunk (two 16-byte words; zeros for a row that does not exist).
__device__ __forceinline__ void load_res16_f16(const ConvTcParams& p, int m, bool valid, int ch, uint4& a, uint4& b) {
  a = b = make_uint4(0u, 0u, 0u, 0u);
  if (!valid) return;
  const uint4* rp = reinterpret_cast<const uint4*>(static_cast<const __half*>(p.res) + static_cast<size_t>(m) * p.res_pitch + ch);
  a = __ldg(rp);
  b = __ldg(rp + 1);
}

// kFastSel: -1 = ConvTcParams::fast_round decides per call (both forms compiled into the caller's loop), 0 / 1 = the caller
// has already branched, once per tile, so the hot loop is straight-line code (40 % of the stall samples of the residual
// kernels were `no_instructions`: instruction fetch behind taken branches and a footprint twice the size it needs to be).
template <int kDtype, bool kHasRes, bool kResI2F = false, int kFastSel = -1>
__device__ __forceinline__ void epilogue_chunk(const ConvTcParams& p, const uint32_t (&v)[16], const uint4 r4, int m,
                                               bool valid, int ch, const float* s_ep0, const float* s_ep1,
                                               const AddReluConst& k, const uint4 r4b = make_uint4(0u, 0u, 0u, 0u)) {
  if (valid && p.dump_acc != nullptr) {
    int4* d = reinterpret_cast<int4*>(p.dump_acc + static_cast<size_t>(m) * p.dump_pitch + ch);
#pragma unroll
    for (int j = 0; j < 4; ++j)
      d[j] = make_int4(static_cast<int>(v[4 * j]), static_cast<int>(v[4 * j + 1]), static_cast<int>(v[4 * j + 2]),
                       static_cast<int>(v[4 * j + 3]));
  }
  if (kDtype == kDtypeI8) {
    uint8_t* op = static_cast<uint8_t*>(p.out) + static_cast<size_t>(m) * p.out_pitch + ch;
    uint4 o;
    if (kFastSel >= 0) {
      if (kHasRes) o = epilogue16_i8_res<kFastSel == 1, kResI2F>(v, r4, s_ep0 + ch, s_ep1 + ch, k);
      else o = epilogue16_i8<kFastSel == 1>(v, s_ep0 + ch, s_ep1 + ch, p.out_zp, p.out_lo);
    } else if (kHasRes) {
      o = p.fast_round ? epilogue16_i8_res<true, kResI2F>(v, r4, s_ep0 + ch, s_ep1 + ch, k)
                       : epilogue16_i8_res<false, kResI2F>(v, r4, s_ep0 + ch, s_ep1 + ch, k);
    } else {
      o = p.fast_round ? epilogue16_i8<true>(v, s_ep0 + ch, s_ep1 + ch, p.out_zp, p.out_lo)
                       : epilogue16_i8<false>(v, s_ep0 + ch, s_ep1 + ch, p.out_zp, p.out_lo);
    }
    if (valid) *reinterpret_cast<uint4*>(op) = o;
  } else {
    __half* op = static_cast<__half*>(p.out) + static_cast<size_t>(m) * p.out_pitch + ch;
    if (kHasRes) {               // (r4, r4b): the residual halves, prefetched by the caller
      if (p.relu) epilogue16_f16_pre<true>(v, s_ep0 + ch, r4, r4b, op, valid);
      else epilogue16_f16_pre<false>(v, s_ep0 + ch, r4, r4b, op, valid);
    } else {
      if (p.relu) epilogue16_f16<false, true>(v, s_ep0 + ch, op, op, valid);
      else epilogue16_f16<false, false>(v, s_ep0 + ch, op, op, valid);
    }
  }
}

// kCluster == 2 (im2col mode, streamed weights): a CTA PAIR runs one tcgen05.mma.cta_group::2 per k-step over
// M = 256 (two consecutive M tiles) x N = bn.  Each CTA loads its own 128 A rows and only HALF of the weight
// k-block (bn/2 rows) into its own shared memory; the tensor cores of both SMs read both halves.  The layers with
// deep K (layers 3-4) are bound by how fast an SM can ingest operands (~40 B/clk), and the pair ingests
// (128 + bn/2) instead of (128 + bn) rows per k-block for the same MMA work.  Only the leader (even) CTA issues
// MMAs; full barriers live in the leader, empty / tmem-full barriers are signalled in both CTAs by the commit.
// kEpiW = 16 (576 threads, one CTA per SM) or 8 (320 threads, TWO CTAs per SM: layers whose operands fit in half of the
// shared memory and half of TMEM run two independent producer -> MMA -> epilogue pipelines per SM, so that the stalls of
// one -- the issuer's barrier tests, an epilogue group waiting for its accumulator -- are filled by the other).
// kZc: the layer's input zero point is not 0 (ConvTcParams::zcorr); a separate instantiation so that the
// register-starved default kernels carry none of it.
template <int kDtype, bool kHasRes, int kMode, int kCluster, int kShape = 0, int kEpiW = kEpiWarps, bool kZc = false>
__global__ void __launch_bounds__(64 + 32 * kEpiW, kEpiW == 8 ? 2 : 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
               const __grid_constant__ ConvTcParams p) {
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment (required by the 128B swizzle atoms) in the shared address space.
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);

  const int num_kb = p.ksize * p.ksize * p.kchunks;
  const int a_bytes = p.a_stage_bytes;
  const int b_bytes = (p.bn / kCluster) * p.kc_bytes;      // a pair CTA holds half of the weight k-block
  const int slots = p.stages * p.kb_group;                  // im2col: kb_group k-blocks share one barrier pair
  const int b_slots = p.resident_b ? num_kb : slots;
  uint8_t* sA = smem;
  uint8_t* sB = smem + slots * a_bytes;
  float* s_ep0 = reinterpret_cast<float*>(sB + b_slots * b_bytes);
  float* s_ep1 = s_ep0 + p.cout_pad;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(s_ep1 + p.cout_pad);
  uint64_t* empty_bar = full_bar + p.stages;
  uint64_t* tfull_bar = empty_bar + p.stages;
  uint64_t* tempty_bar = tfull_bar + kMaxAcc;
  uint64_t* bres_bar = tempty_bar + kMaxAcc;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bres_bar + 1);

  const int warp = threadIdx.x >> 5;       // warp-uniform
  const int lane = threadIdx.x & 31;

  constexpr int kThreads = 64 + 32 * kEpiW;
  constexpr int kGroupsMax = kEpiW / 4;
  for (int i = threadIdx.x; i < p.cout_pad; i += kThreads) {
    s_ep0[i] = p.ep0[i];
    s_ep1[i] = p.ep1[i];
  }
  const uint32_t crank = kCluster > 1 ? cluster_ctarank() : 0u;
  const bool leader = crank == 0;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
    for (int i = 0; i < p.stages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < p.nacc; ++i) {
      mbar_init(&tfull_bar[i], 1);
      // one arrival per warp of the owning group (of both CTAs of a pair); groups = min(4, nacc), see the epilogue
      mbar_init(&tempty_bar[i], kCluster * kEpiW / (p.nacc < kGroupsMax ? p.nacc : kGroupsMax));
    }
    mbar_init(bres_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    if (kCluster > 1) {
      tmem_alloc_pair(tmem_slot, static_cast<uint32_t>(p.tmem_cols));
      tmem_relinquish_pair();
    } else {
      tmem_alloc(tmem_slot, static_cast<uint32_t>(p.tmem_cols));
      tmem_relinquish();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (kCluster > 1) cluster_sync_all();     // the peer's barriers are initialised before anyone signals them
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
  griddep_launch_dependents();          // the next kernel may begin its prologue as SMs free up

  // Work schedule.
  //   im2col : work item `tile` of stride `tile_step` starting at `tile_first`:
  //              single CTA : tile -> (m_tile = tile / n_tiles, n_tile = tile % n_tiles)
  //              cluster    : tile is a cluster tile -> (m_tile = (tile / n_tiles) * kCluster + rank, n_tile = tile % n_tiles)
  //   halo   : the sub-tiles (img, s) = (t / T, t % T) are numbered t = 0 .. n*T-1; CTA b owns the CONTIGUOUS range
  //            [t_begin, t_end) (sizes differ by at most one sub-tile) and walks it in bands of up to S sub-tiles of the
  //            same image.  All three roles derive the same band sequence from (t_begin, t_end).
  const int total_tiles = kCluster > 1 ? ((p.m_tiles + kCluster - 1) / kCluster) * p.n_tiles : p.m_tiles * p.n_tiles;
  const int tile_first = kCluster > 1 ? static_cast<int>(blockIdx.x) / kCluster : static_cast<int>(blockIdx.x);
  const int tile_step = kCluster > 1 ? static_cast<int>(gridDim.x) / kCluster : static_cast<int>(gridDim.x);
  const int hw = p.ho * p.wo;
  int t_begin = 0, t_end = 0;
  if (kMode == kModeHalo) {
    const int q = p.total_subs / static_cast<int>(gridDim.x), r = p.total_subs - q * static_cast<int>(gridDim.x);
    const int b = static_cast<int>(blockIdx.x);
    t_begin = b * q + (b < r ? b : r);
    t_end = t_begin + q + (b < r ? 1 : 0);
  }
#ifdef IEVM_EXP_TIMING
  long long tm_wait_a = 0, tm_wait_b = 0;
  const long long tm_t0 = clock64();
  const unsigned long long tm_ns0 = globaltimer_ns();
  unsigned long long* tm_out = g_exp_timing + (static_cast<size_t>(p.timing_slot) * kExpCtas + blockIdx.x) * kExpWords;
  int tm_tiles = 0;
#endif

  if (warp == 0) {
    // ================================ TMA producer ================================
    // The whole warp walks the schedule (so coordinates stay in uniform registers); one elected lane
    // arms the barrier and issues the copies.
    if (p.resident_b && elect_one()) {
      mbar_expect_tx(bres_bar, static_cast<uint32_t>(num_kb * b_bytes));
      for (int kb = 0; kb < num_kb; ++kb) tma_load_2d(sB + kb * b_bytes, &tmap_b, bres_bar, kb * p.kc_elems, 0);
    }
    __syncwarp();
    griddep_wait_conv();                     // weights were loadable early; activations need the previous kernel done
    const uint32_t tx_bytes = static_cast<uint32_t>(p.resident_b ? p.a_tx_bytes : p.a_tx_bytes + b_bytes);
    int stage = 0;
    uint32_t phase = 0;
    if (kMode == kModeHalo) {
      int img = fast_div(t_begin, p.subs_per_img, p.spi_magic);
      int s0 = t_begin - img * p.subs_per_img;
      for (int t = t_begin; t < t_end;) {
        const int ns = min(p.band_subs, min(p.subs_per_img - s0, t_end - t));
        IEVM_TIMED_WAIT(tm_wait_a, &empty_bar[stage], phase ^ 1u, 0x100u | stage, p.stuck_flag);
        if (elect_one()) {
          mbar_expect_tx(&full_bar[stage], tx_bytes);
          tma_load_4d(sA + stage * a_bytes, &tmap_a, &full_bar[stage], 0, -1, s0 * p.sub_rows - 1, img);
        }
        __syncwarp();
        if (++stage == p.stages) {
          stage = 0;
          phase ^= 1u;
        }
        t += ns;
        s0 += ns;
        if (s0 == p.subs_per_img) {
          s0 = 0;
          ++img;
        }
      }
    } else {
      const int G = p.kb_group;
      for (int tile = tile_first; tile < total_tiles; tile += tile_step) {
        const int m_group = tile / p.n_tiles;
        const int n_tile = tile - m_group * p.n_tiles;
        const int m_tile = kCluster > 1 ? m_group * kCluster + static_cast<int>(crank) : m_group;
        const int m0 = m_tile * kTileM;
        const int img = fast_div(m0, hw, p.hw_magic);
        const int rem = m0 - img * hw;
        const int oy = fast_div(rem, p.wo, p.wo_magic);
        const int ox = rem - oy * p.wo;
        const int base_w = ox * p.stride - p.pad;
        const int base_h = oy * p.stride - p.pad;
        int kb = 0, g = 0;
        for (int ty = 0; ty < p.ksize; ++ty) {
          for (int tx = 0; tx < p.ksize; ++tx) {
            for (int ch = 0; ch < p.kchunks; ++ch, ++kb) {
              if (g == 0) IEVM_TIMED_WAIT(tm_wait_a, &empty_bar[stage], phase ^ 1u, 0x100u | stage, p.stuck_flag);
              const int slot = stage * G + g;
              if (elect_one()) {
                if (kCluster > 1) {
                  // both CTAs fill their own stage and complete bytes on the leader's barrier; the leader arms it
                  // for the pair's total
                  if (leader && g == 0) mbar_expect_tx(&full_bar[stage], 2u * tx_bytes * static_cast<uint32_t>(G));
                  tma_load_im2col_4d_pair(sA + slot * a_bytes, &tmap_a, &full_bar[stage], ch * p.kc_elems, base_w, base_h,
                                          img, static_cast<uint16_t>(tx), static_cast<uint16_t>(ty));
                  tma_load_2d_pair(sB + slot * b_bytes, &tmap_b, &full_bar[stage], kb * p.kc_elems,
                                   n_tile * p.bn + static_cast<int>(crank) * (p.bn / kCluster));
                } else {
                  if (g == 0) mbar_expect_tx(&full_bar[stage], tx_bytes * static_cast<uint32_t>(G));
                  tma_load_im2col_4d(sA + slot * a_bytes, &tmap_a, &full_bar[stage], ch * p.kc_elems, base_w, base_h, img,
                                     static_cast<uint16_t>(tx), static_cast<uint16_t>(ty));
                  if (!p.resident_b)
                    tma_load_2d(sB + slot * b_bytes, &tmap_b, &full_bar[stage], kb * p.kc_elems, n_tile * p.bn);
                }
              }
              __syncwarp();
              if (++g == G) {
                g = 0;
                if (++stage == p.stages) {
                  stage = 0;
                  phase ^= 1u;
                }
              }
            }
          }
        }
      }
    }
#ifdef IEVM_EXP_TIMING
    if (lane == 0 && blockIdx.x < kExpCtas) {
      tm_out[4] = clock64() - tm_t0;
      tm_out[5] = tm_wait_a;
    }
#endif
  } else if (warp == 1) {
    // ================================ MMA issuer ================================
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    // One tcgen05.mma consumes 32 bytes of K per row: 2 (64-byte rows) or 4 (128-byte rows) per k-block.
    // Everything the issuing thread needs per instruction is reduced to one add on a precomputed descriptor low
    // word, and barrier tests are batched: the tensor unit's instruction queue is only one or two instructions
    // deep, so whatever the issuing thread does between two instructions beyond ~50 cycles is idle tensor time
    // (one mbarrier test is ~150).
    const bool wide = p.kc_bytes == 128;
    const uint32_t hi = smem_desc_hi(static_cast<uint32_t>(p.kc_bytes));
    const uint32_t a_lo0 = smem_desc_lo(smem_u32(sA));
    const uint32_t b_lo0 = smem_desc_lo(smem_u32(sB));
    const uint32_t a_step = static_cast<uint32_t>(a_bytes) >> 4;
    const uint32_t b_step = static_cast<uint32_t>(b_bytes) >> 4;
    const uint32_t row16 = static_cast<uint32_t>(p.kc_bytes) >> 4;      // one pixel row in 16-byte units
    const uint32_t idesc = p.idesc;
    auto mma = [&](uint32_t d, uint32_t a_lo, uint32_t b_lo, uint32_t accum) {
      if (kCluster > 1) {
        if (kDtype == kDtypeI8) umma_i8_lohi_pair(d, a_lo, b_lo, hi, idesc, accum);
        else umma_f16_lohi_pair(d, a_lo, b_lo, hi, idesc, accum);
      } else {
        if (kDtype == kDtypeI8) umma_i8_lohi(d, a_lo, b_lo, hi, idesc, accum);
        else umma_f16_lohi(d, a_lo, b_lo, hi, idesc, accum);
      }
    };
    auto mma_kblock = [&](uint32_t d, uint32_t a_lo, uint32_t b_lo, uint32_t first_accum) {
      mma(d, a_lo, b_lo, first_accum);
      mma(d, a_lo + 2, b_lo + 2, 1u);
      if (wide) {
        mma(d, a_lo + 4, b_lo + 4, 1u);
        mma(d, a_lo + 6, b_lo + 6, 1u);
      }
    };
    if (p.resident_b) wait_or_die(bres_bar, 0, 0x500u, p.stuck_flag);
    if (kMode == kModeHalo) {
      constexpr bool kStatic = kShape != 0;
      const uint32_t row16v = kStatic ? static_cast<uint32_t>(halo_shape_rb(kShape) / 16) : row16;
      const uint32_t wp16 = kStatic ? static_cast<uint32_t>(halo_shape_wp(kShape) * (halo_shape_rb(kShape) / 16))
                                    : static_cast<uint32_t>(p.wp) * row16;
      const uint32_t bstep = kStatic ? static_cast<uint32_t>(halo_shape_bn(kShape) * halo_shape_rb(kShape) / 16) : b_step;
      const bool widev = kStatic ? halo_shape_rb(kShape) == 128 : wide;
      const uint32_t sub_step = static_cast<uint32_t>(p.sub_pos) * row16;
      int s0 = t_begin - fast_div(t_begin, p.subs_per_img, p.spi_magic) * p.subs_per_img;
      for (int t = t_begin; t < t_end;) {
        const int ns = min(p.band_subs, min(p.subs_per_img - s0, t_end - t));
        // ONE batched test of the band's barriers (patch landed, its ns accumulators drained): the tests are issued back
        // to back, so the batch costs one round trip instead of ns + 1
        {
          uint64_t* bars[kMaxBandSubs + 1];
          uint32_t par[kMaxBandSubs + 1];
          bars[0] = &full_bar[stage];
          par[0] = phase;
          int a = acc;
          uint32_t ph = acc_phase;
#pragma unroll
          for (int j = 0; j < kMaxBandSubs; ++j) {
            if (j < ns) {
              bars[j + 1] = &tempty_bar[a];
              par[j + 1] = ph ^ 1u;
              if (++a == p.nacc) {
                a = 0;
                ph ^= 1u;
              }
            } else {
              bars[j + 1] = bars[j];
              par[j + 1] = par[j];
            }
          }
#ifdef IEVM_EXP_TIMING
          const long long tw0 = clock64();
#endif
          if (!mbar_try_wait5(bars[0], par[0], bars[1], par[1], bars[2], par[2], bars[3], par[3], bars[4], par[4])) {
            // not there yet: repeat the batched test (one round trip per attempt) instead of five blocking waits in a row
            const uint64_t t0 = globaltimer_ns();
            uint32_t spins = 0;
            while (!mbar_try_wait5(bars[0], par[0], bars[1], par[1], bars[2], par[2], bars[3], par[3], bars[4], par[4])) {
              if ((++spins & 0x3ff) == 0 && globaltimer_ns() - t0 > IEVM_WAIT_LIMIT_NS) {
                wait_or_die(bars[0], par[0], 0x300u | stage, p.stuck_flag);      // names the barrier that is stuck, then traps
#pragma unroll
                for (int j = 1; j <= kMaxBandSubs; ++j) wait_or_die(bars[j], par[j], 0x200u | j, p.stuck_flag);
              }
            }
          }
#ifdef IEVM_EXP_TIMING
          tm_wait_b += clock64() - tw0;
#endif
        }
        tc_fence_after();
        const uint32_t a_band = a_lo0 + static_cast<uint32_t>(stage) * a_step;
        if (elect_one()) {
          int a2 = acc;
#ifdef IEVM_EXP_TIMING
          const long long ti0 = clock64();
#endif
#pragma unroll 1
          for (int j = 0; j < ns; ++j) {
            const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(a2 * p.acc_stride);
            const uint32_t a_lo = a_band + static_cast<uint32_t>(j) * sub_step;
            // opaque to the optimiser: the 18 / 36 weight descriptors are then base + immediate (one uniform add each)
            // instead of loop-invariant values parked in vector registers and moved back with R2UR before every use
            uint32_t b_base = b_lo0;
            asm volatile("" : "+r"(b_base));
#pragma unroll
            for (int tap = 0; tap < 9; ++tap) {
              const uint32_t ao = a_lo + static_cast<uint32_t>(tap / 3) * wp16 + static_cast<uint32_t>(tap % 3) * row16v;
              const uint32_t bo = b_base + static_cast<uint32_t>(tap) * bstep;
              mma(d_tmem, ao, bo, tap != 0 ? 1u : 0u);
              mma(d_tmem, ao + 2, bo + 2, 1u);
              if (widev) {
                mma(d_tmem, ao + 4, bo + 4, 1u);
                mma(d_tmem, ao + 6, bo + 6, 1u);
              }
            }
            umma_commit(&tfull_bar[a2]);
            if (++a2 == p.nacc) a2 = 0;
          }
          umma_commit(&empty_bar[stage]);
#ifdef IEVM_EXP_TIMING
          tm_wait_a += clock64() - ti0;      // halo mode: slot 1 = cycles inside the issue region (tempty waits are in slot 2)
#endif
        }
        __syncwarp();
        {
          const int adv = acc + ns;
          acc_phase ^= (adv >= p.nacc) ? 1u : 0u;
          acc = adv >= p.nacc ? adv - p.nacc : adv;
        }
        if (++stage == p.stages) {
          stage = 0;
          phase ^= 1u;
        }
        t += ns;
        s0 += ns;
        if (s0 == p.subs_per_img) s0 = 0;
      }
    } else {
      const int G = p.kb_group;
      const int groups_per_tile = num_kb / G;
      for (int tile = tile_first; leader && tile < total_tiles; tile += tile_step) {   // the peer CTA issues no MMAs
        IEVM_TIMED_WAIT(tm_wait_a, &tempty_bar[acc], acc_phase ^ 1u, 0x200u | acc, p.stuck_flag);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * p.acc_stride);
        for (int kg = 0; kg < groups_per_tile; ++kg) {
          IEVM_TIMED_WAIT(tm_wait_b, &full_bar[stage], phase, 0x300u | stage, p.stuck_flag);
          tc_fence_after();
          if (elect_one()) {
            for (int g = 0; g < G; ++g) {
              const int kb = kg * G + g;
              const uint32_t a_lo = a_lo0 + static_cast<uint32_t>(stage * G + g) * a_step;
              const uint32_t b_lo = b_lo0 + static_cast<uint32_t>(p.resident_b ? kb : stage * G + g) * b_step;
              mma_kblock(d_tmem, a_lo, b_lo, kb != 0 ? 1u : 0u);
            }
            if (kCluster > 1) {
              umma_commit_pair(&empty_bar[stage]);          // frees the stage in both CTAs
              if (kg == groups_per_tile - 1) umma_commit_pair(&tfull_bar[acc]);
            } else {
              umma_commit(&empty_bar[stage]);               // smem slots reusable once these MMAs retire
              if (kg == groups_per_tile - 1) umma_commit(&tfull_bar[acc]);   // accumulator complete
            }
          }
          __syncwarp();
          if (++stage == p.stages) {
            stage = 0;
            phase ^= 1u;
          }
        }
        if (++acc == p.nacc) {
          acc = 0;
          acc_phase ^= 1u;
        }
      }
    }
#ifdef IEVM_EXP_TIMING
    for (int o = 16; o > 0; o >>= 1) {      // the issue-region timer lives in the elected lane
      const long long other = __shfl_xor_sync(0xffffffffu, tm_wait_a, o);
      tm_wait_a = other > tm_wait_a ? other : tm_wait_a;
    }
    if (lane == 0 && blockIdx.x < kExpCtas) {
      tm_out[0] = clock64() - tm_t0;
      tm_out[1] = tm_wait_a;
      tm_out[2] = tm_wait_b;
      tm_out[3] = globaltimer_ns() - tm_ns0;
    }
#endif
  } else {
    // ================================ epilogue ================================
    const int quad = warp & 3;
    // groups = min(4, nacc) so that a TMEM buffer is always drained by the same group: a waiter can tell only
    // adjacent mbarrier phases apart, so it has to see every phase of the barriers it waits on.  With two
    // buffers (bn > 128) there are two groups of eight warps, two per quadrant, which interleave chunks.
    const int groups = p.nacc < kGroupsMax ? p.nacc : kGroupsMax;      // 2 or 4
    const int group = ((warp - 2) >> 2) & (groups - 1);
    const int sub = ((warp - 2) >> 2) / groups;                        // which of the group's warps of this quadrant
    const int csub = kGroupsMax / groups;                              // warps per quadrant in a group
    const int row = quad * 32 + lane;
    const int nchunks = p.bn >> 4;
    griddep_wait_conv();                     // before the first residual read / output store
    AddReluConst k;
    k.lo_f = static_cast<float>(p.out_lo - p.out_zp);
    k.hi_f = static_cast<float>(255 - p.out_zp);
    k.a_scale = p.a_scale;
    k.r_scale = p.res_scale;
    k.inv_scale = p.inv_add_scale;
    k.pa = __fmul_rn(p.a_scale, -static_cast<float>(p.out_zp));
    k.pb = __fmul_rn(p.res_scale, -static_cast<float>(p.res_zp));
    k.lo_q = static_cast<float>(p.out_lo);
    k.zp_f = static_cast<float>(p.out_zp);
    k.add_zp = p.add_zp;
    k.c1_add = -kRoundMagicBits - (p.out_lo - p.out_zp);
    k.c1_max = 255 - p.out_lo;
    k.c2_add = -kRoundMagicBits;
    k.c2_max = 255 - p.add_zp;
    k.zp4 = static_cast<uint32_t>(p.add_zp) * 0x01010101u;
    // this thread's place inside a halo sub-tile (fixed: sub-tiles are row aligned)
    const int sub_row = kMode == kModeHalo ? fast_div(row, p.wp, p.wp_magic) : 0;
    const int sub_x = row - sub_row * p.wp;
    const bool sub_ok = kMode == kModeHalo && row < p.sub_pos && sub_x < p.w_in;
    constexpr bool kResI8 = kHasRes && kDtype == kDtypeI8;
    constexpr bool kResF16 = kHasRes && kDtype == kDtypeF16;
    // One tile (accumulator buffer `acc`) of output rows starting at pixel index m (valid = this thread's row exists).
    // Border class of output pixel (oy, ox) for the zero-point correction: which filter taps read inside the image.
    auto zcorr_row = [&](int oy, int ox) -> const int32_t* {
      int my = 0, mx = 0;
      for (int t = 0; t < p.ksize; ++t) {
        const int iy = oy * p.stride - p.pad + t, ix = ox * p.stride - p.pad + t;
        my |= (iy >= 0 && iy < p.h_in) ? (1 << t) : 0;
        mx |= (ix >= 0 && ix < p.w_in) ? (1 << t) : 0;
      }
      return p.zcorr + static_cast<size_t>((my << p.ksize) | mx) * p.cout_pad;
    };
    auto drain = [&](int acc, uint32_t acc_phase, int m, bool valid, int n0, const int32_t* zc = nullptr) {
      uint4 ra = make_uint4(0u, 0u, 0u, 0u), rb = ra;
      uint4 sa = ra, sb = ra;                    // FP16: second half of a chunk's residual
      int c = sub;
      if (kResI8 && c < nchunks) ra = load_res16_i8(p, m, valid, n0 + c * 16);   // does not depend on the MMA
      if (kResF16 && c < nchunks) load_res16_f16(p, m, valid, n0 + c * 16, ra, sa);
      IEVM_TIMED_WAIT(tm_wait_a, &tfull_bar[acc], acc_phase, 0x400u | acc, p.stuck_flag);
      tc_fence_after();
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) +
                             static_cast<uint32_t>(acc * p.acc_stride);
      // two register buffers: the TMEM load (and residual fetch) of the next chunk is in flight while this
      // one is processed
      uint32_t va[16], vb[16];
      if (c < nchunks) tmem_ld_32x32b_x16(t_row + static_cast<uint32_t>(c * 16), va);
      while (c < nchunks) {
        tmem_ld_wait();
        if (kZc && zc != nullptr) {
#pragma unroll
          for (int j = 0; j < 16; ++j) va[j] -= static_cast<uint32_t>(__ldg(zc + n0 + c * 16 + j));
        }
        if (c + csub < nchunks) {
          tmem_ld_32x32b_x16(t_row + static_cast<uint32_t>((c + csub) * 16), vb);
          if (kResI8) rb = load_res16_i8(p, m, valid, n0 + (c + csub) * 16);
          if (kResF16) load_res16_f16(p, m, valid, n0 + (c + csub) * 16, rb, sb);
        }
        epilogue_chunk<kDtype, kHasRes>(p, va, ra, m, valid, n0 + c * 16, s_ep0, s_ep1, k, sa);
        c += csub;
        if (c >= nchunks) break;
        tmem_ld_wait();
        if (kZc && zc != nullptr) {
#pragma unroll
          for (int j = 0; j < 16; ++j) vb[j] -= static_cast<uint32_t>(__ldg(zc + n0 + c * 16 + j));
        }
        if (c + csub < nchunks) {
          tmem_ld_32x32b_x16(t_row + static_cast<uint32_t>((c + csub) * 16), va);
          if (kResI8) ra = load_res16_i8(p, m, valid, n0 + (c + csub) * 16);
          if (kResF16) load_res16_f16(p, m, valid, n0 + (c + csub) * 16, ra, sa);
        }
        epilogue_chunk<kDtype, kHasRes>(p, vb, rb, m, valid, n0 + c * 16, s_ep0, s_ep1, k, sb);
        c += csub;
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (kCluster > 1 && !leader) mbar_arrive_remote(&tempty_bar[acc], 0u);   // the leader's MMA warp waits for both
        else mbar_arrive(&tempty_bar[acc]);
      }
    };
    // The same for a statically shaped halo layer: one warp per quadrant owns the tile (four groups), the chunk loop is
    // unrolled and the per-channel tables are constant-bank operands (ConvTcParams::epc0 / epc1).
    auto drain_static = [&](auto fast_sel, int acc, uint32_t acc_phase, int m, bool valid) {
      constexpr int kFs = kDtype == kDtypeI8 ? decltype(fast_sel)::value : -1;
      constexpr int kNch = kShape != 0 ? halo_shape_bn(kShape) / 16 : 1;
      uint4 rr[2];
      rr[0] = rr[1] = make_uint4(0u, 0u, 0u, 0u);
      uint4 rq[2];                                // FP16: second half of a chunk's residual
      rq[0] = rq[1] = rr[0];
      // INT8, at most four chunks: every residual chunk of the row is loaded before the accumulator wait (loading one
      // chunk ahead leaves an L2 round trip exposed behind each chunk's arithmetic: 53 vs 49 us per layer-1 residual conv)
      constexpr bool kResAll = kResI8 && kNch <= 4;
      uint4 ra[kResAll ? kNch : 1];
      if (kResAll) {
#pragma unroll
        for (int c = 0; c < (kResAll ? kNch : 1); ++c) ra[c] = load_res16_i8(p, m, valid, c * 16);
      }
      if (kResI8 && !kResAll) rr[0] = load_res16_i8(p, m, valid, 0);
      if (kResF16) load_res16_f16(p, m, valid, 0, rr[0], rq[0]);
      IEVM_TIMED_WAIT(tm_wait_a, &tfull_bar[acc], acc_phase, 0x400u | acc, p.stuck_flag);
      tc_fence_after();
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) +
                             static_cast<uint32_t>(acc * p.acc_stride);
      uint32_t vv[2][16];
      tmem_ld_32x32b_x16(t_row, vv[0]);
      if (kNch <= 4) {
#pragma unroll
        for (int c = 0; c < kNch; ++c) {
          tmem_ld_wait();
          if (c + 1 < kNch) {
            tmem_ld_32x32b_x16(t_row + static_cast<uint32_t>((c + 1) * 16), vv[(c + 1) & 1]);
            if (kResI8 && !kResAll) rr[(c + 1) & 1] = load_res16_i8(p, m, valid, (c + 1) * 16);
            if (kResF16) load_res16_f16(p, m, valid, (c + 1) * 16, rr[(c + 1) & 1], rq[(c + 1) & 1]);
          }
          epilogue_chunk<kDtype, kHasRes, false, kFs>(p, vv[c & 1], kResAll ? ra[c < (kResAll ? kNch : 1) ? c : 0] : rr[c & 1],
                                                     m, valid, c * 16, p.epc0, p.epc1, k, rq[c & 1]);
        }
      } else {
        // wide layers: the chunk loop stays a loop over chunk PAIRS (register budget); the tables are still read from
        // the constant bank, through a uniform index
#pragma unroll 1
        for (int c = 0; c < kNch; c += 2) {
          tmem_ld_wait();
          tmem_ld_32x32b_x16(t_row + static_cast<uint32_t>((c + 1) * 16), vv[1]);
          if (kResI8) rr[1] = load_res16_i8(p, m, valid, (c + 1) * 16);
          if (kResF16) load_res16_f16(p, m, valid, (c + 1) * 16, rr[1], rq[1]);
          epilogue_chunk<kDtype, kHasRes, true, kFs>(p, vv[0], rr[0], m, valid, c * 16, p.epc0, p.epc1, k, rq[0]);
          tmem_ld_wait();
          if (c + 2 < kNch) {
            tmem_ld_32x32b_x16(t_row + static_cast<uint32_t>((c + 2) * 16), vv[0]);
            if (kResI8) rr[0] = load_res16_i8(p, m, valid, (c + 2) * 16);
            if (kResF16) load_res16_f16(p, m, valid, (c + 2) * 16, rr[0], rq[0]);
          }
          epilogue_chunk<kDtype, kHasRes, true, kFs>(p, vv[1], rr[1], m, valid, (c + 1) * 16, p.epc0, p.epc1, k, rq[1]);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[acc]);
    };
    if (kMode == kModeHalo) {
      // group g owns the CTA's tiles g, g + groups, ... ; the accumulator ring position follows from the tile's sequence
      // number (nacc is a power of two)
      const int nacc_shift = 31 - __clz(p.nacc);
      for (int t = t_begin + group; t < t_end; t += groups) {
        const int seq = t - t_begin;
        const int acc = seq & (p.nacc - 1);
        const uint32_t acc_phase = static_cast<uint32_t>(seq >> nacc_shift) & 1u;
#ifdef IEVM_EXP_TIMING
        ++tm_tiles;
#endif
        const int img = fast_div(t, p.subs_per_img, p.spi_magic);
        const int oy = (t - img * p.subs_per_img) * p.sub_rows + sub_row;
        const bool valid = sub_ok && oy < p.h_in;
        const int m = (img * p.h_in + oy) * p.w_in + sub_x;
        if (kShape != 0) {
          if (p.fast_round) drain_static(std::integral_constant<int, 1>{}, acc, acc_phase, m, valid);
          else drain_static(std::integral_constant<int, 0>{}, acc, acc_phase, m, valid);
        } else drain(acc, acc_phase, m, valid, 0, kZc ? zcorr_row(oy, sub_x) : nullptr);
      }
    } else {
      int acc_next = 0, seq = 0;
      uint32_t acc_phase_next = 0;
      for (int tile = tile_first; tile < total_tiles; tile += tile_step, ++seq) {
        const int acc = acc_next;
        const uint32_t acc_phase = acc_phase_next;
        if (++acc_next == p.nacc) {
          acc_next = 0;
          acc_phase_next ^= 1u;
        }
        if ((seq & (groups - 1)) != group) continue;
#ifdef IEVM_EXP_TIMING
        ++tm_tiles;
#endif
        const int m_group = tile / p.n_tiles;
        const int n_tile = tile - m_group * p.n_tiles;
        const int m_tile = kCluster > 1 ? m_group * kCluster + static_cast<int>(crank) : m_group;
        const int m = m_tile * kTileM + row;
        const int32_t* zc = nullptr;
        if (kZc) {
          const int rem = m - (m / hw) * hw;
          zc = zcorr_row(rem / p.wo, rem - (rem / p.wo) * p.wo);
        }
        drain(acc, acc_phase, m, m < p.m_total, n_tile * p.bn, zc);
      }
    }
  }

#ifdef IEVM_EXP_TIMING
  if (warp == 2 && lane == 0 && blockIdx.x < kExpCtas) {
    tm_out[6] = clock64() - tm_t0;
    tm_out[7] = tm_wait_a;
    tm_out[8] = tm_tiles;
  }
#endif
  tc_fence_before();
  __syncthreads();
#ifdef IEVM_EXP_TIMING
  if (warp == 1 && lane == 0 && blockIdx.x < kExpCtas) {
    tm_out[9] = clock64() - tm_t0;
    tm_out[10] = globaltimer_ns() - tm_ns0;
  }
#endif
  if (kCluster > 1) cluster_sync_all();     // no CTA leaves while its peer may still signal its barriers
  if (warp == 1) {
    tc_fence_after();
    if (kCluster > 1) tmem_dealloc_pair(tmem_base, static_cast<uint32_t>(p.tmem_cols));
    else tmem_dealloc(tmem_base, static_cast<uint32_t>(p.tmem_cols));
  }
}

}  // namespace ievm
