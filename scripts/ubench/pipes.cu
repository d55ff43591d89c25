// Micro-benchmark: per-SM issue rate of the instructions the requantisation epilogues are made of.
// One CTA per SM, W warps, each warp runs N iterations of 16 independent chains of one op.
// Prints cycles per warp-instruction per SMSP (lower = faster).   nvcc -arch=sm_100a -O3 pipes.cu -o pipes
// The paired rows (FADD2 / FMUL2 / FFMA2) run chains of float2: one instruction does two lanes' work, so a paired op at the
// scalar op's cycles per instruction halves the issue cost per value.
#include <cstdio>
#include <cstdint>
#include <cuda_runtime.h>

enum Op { I2F, F2I, FADD, FMUL, FFMA, FADD2, FMUL2, FFMA2, IADD, IMNMX, PRMT, I2IP, FMNMX, MIX_CUR, MIX_MAGIC, MIX_H1, ADDRELU_CUR, ADDRELU_NEW, NOPS };
static const char* kNames[] = {"I2F", "F2I", "FADD", "FMUL", "FFMA", "FADD2", "FMUL2", "FFMA2", "IADD", "VIMNMX", "PRMT", "I2IP(cvt.pack)", "FMNMX",
                               "requant_current(6/val)", "requant_magic(8.75/val)", "requant_H1(I2F+magic round)",
                               "add_relu_current", "add_relu_new(magic final round)"};

template <int kOp>
__global__ void bench(int iters, float fa, int ia, unsigned long long* out_cycles, int* sink) {
  int x[16];
  float f[16];
  float2 g[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    x[i] = threadIdx.x * 17 + i * ia;
    f[i] = fa * (threadIdx.x + i);
    g[i] = make_float2(f[i], fa * (threadIdx.x + 2 * i));
  }
  const float2 fa2 = make_float2(fa, fa * fa);
  __syncthreads();
  const unsigned long long t0 = clock64();
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      if (kOp == I2F) { f[i] = __int2float_rn(x[i]); x[i] = __float_as_int(f[i]) ^ ia; }          // I2F + LOP
      else if (kOp == F2I) { x[i] = __float2int_rn(f[i]); f[i] = __int_as_float(x[i] | 0x3f800000); }
      else if (kOp == FADD) f[i] = __fadd_rn(f[i], fa);
      else if (kOp == FMUL) f[i] = __fmul_rn(f[i], fa);
      else if (kOp == FFMA) f[i] = __fmaf_rn(f[i], fa, fa);
      else if (kOp == FADD2) g[i] = __fadd2_rn(g[i], fa2);
      else if (kOp == FMUL2) g[i] = __fmul2_rn(g[i], fa2);
      else if (kOp == FFMA2) g[i] = __ffma2_rn(g[i], fa2, fa2);
      else if (kOp == IADD) x[i] = x[i] + ia;
      else if (kOp == IMNMX) x[i] = max(x[i], ia + i) ;
      else if (kOp == PRMT) x[i] = __byte_perm(x[i], ia, 0x4321);
      else if (kOp == I2IP) { unsigned d; asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(x[i]), "r"(ia), "r"(0)); x[i] = d; }
      else if (kOp == FMNMX) f[i] = fmaxf(f[i], fa);
      else if (kOp == MIX_CUR) {
        const float v = __fmul_rn(__fadd_rn(__int2float_rn(x[i]), fa), 0.37f);
        x[i] = max(__float2int_rn(v) + ia, 3);
      } else if (kOp == MIX_H1) {
        const float v = __fmul_rn(__fadd_rn(__int2float_rn(x[i]), fa), 0.37f);
        x[i] = max(__float_as_int(__fadd_rn(v, 12582912.0f)) + (ia - 0x4B400000), 3);
      } else if (kOp == ADDRELU_CUR || kOp == ADDRELU_NEW) {
        float t = __fmul_rn(__fadd_rn(__int2float_rn(x[i]), fa), 0.37f);
        t = fminf(fmaxf(t, -60.f), 195.f);
        t = __fadd_rn(__fadd_rn(t, 12582912.0f), -12582912.0f);
        const float a = __fmul_rn(t, 0.051f);
        const float rb = __fadd_rn(__uint_as_float(__byte_perm(x[(i + 1) & 15], 0x4B400000u, 0x7650 + (i & 3))), -12582912.0f);
        const float s2 = fmaxf(__fadd_rn(a, __fmul_rn(rb, 0.043f)), 0.0f);
        if (kOp == ADDRELU_CUR) x[i] = __float2int_rn(__fmul_rn(s2, 13.7f)) + ia;
        else x[i] = __float_as_int(__fadd_rn(__fmul_rn(s2, 13.7f), 12582912.0f)) + (ia - 0x4B400000);
      } else if (kOp == MIX_MAGIC) {
        float v = __fadd_rn(__int_as_float(x[i] + 0x4B400000), -12582912.0f);
        v = __fmul_rn(__fadd_rn(v, fa), 0.37f);
        v = fminf(fmaxf(v, -60.f), 195.f);
        x[i] = __float_as_int(__fadd_rn(v, 12582912.0f)) + ia;
      }
    }
  }
  const unsigned long long t1 = clock64();
  int s = 0;
#pragma unroll
  for (int i = 0; i < 16; ++i) s += x[i] + __float_as_int(f[i]) + __float_as_int(g[i].x) + __float_as_int(g[i].y);
  if (s == 0x12345) *sink = s;
  if (threadIdx.x == 0 && blockIdx.x == 0) *out_cycles = t1 - t0;
}

template <int kOp>
void run(int warps, unsigned long long* d_cyc, int* d_sink) {
  const int iters = 2000;
  bench<kOp><<<148, warps * 32>>>(iters, 1.0001f, 3, d_cyc, d_sink);
  cudaDeviceSynchronize();
  bench<kOp><<<148, warps * 32>>>(iters, 1.0001f, 3, d_cyc, d_sink);
  cudaDeviceSynchronize();
  unsigned long long c = 0;
  cudaMemcpy(&c, d_cyc, sizeof(c), cudaMemcpyDeviceToHost);
  const double warp_insts_per_smsp = static_cast<double>(iters) * 16 * warps / 4.0;
  printf("%-26s warps/SM=%2d  cycles per 'op' per SMSP = %.2f\n", kNames[kOp], warps, c / warp_insts_per_smsp);
}

int main() {
  unsigned long long* d_cyc;
  int* d_sink;
  cudaMalloc(&d_cyc, 8);
  cudaMalloc(&d_sink, 4);
  for (int warps : {4, 8, 16}) {
    run<I2F>(warps, d_cyc, d_sink);
    run<F2I>(warps, d_cyc, d_sink);
    run<FADD>(warps, d_cyc, d_sink);
    run<FMUL>(warps, d_cyc, d_sink);
    run<FFMA>(warps, d_cyc, d_sink);
    run<FADD2>(warps, d_cyc, d_sink);
    run<FMUL2>(warps, d_cyc, d_sink);
    run<FFMA2>(warps, d_cyc, d_sink);
    run<IADD>(warps, d_cyc, d_sink);
    run<IMNMX>(warps, d_cyc, d_sink);
    run<PRMT>(warps, d_cyc, d_sink);
    run<I2IP>(warps, d_cyc, d_sink);
    run<FMNMX>(warps, d_cyc, d_sink);
    run<MIX_CUR>(warps, d_cyc, d_sink);
    run<MIX_MAGIC>(warps, d_cyc, d_sink);
    run<MIX_H1>(warps, d_cyc, d_sink);
    run<ADDRELU_CUR>(warps, d_cyc, d_sink);
    run<ADDRELU_NEW>(warps, d_cyc, d_sink);
  }
  return 0;
}
