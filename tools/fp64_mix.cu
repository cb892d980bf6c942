// What does a non-MMA FP64 instruction cost on the FP64 pipe it shares with DMMA, as a function of what surrounds it?
// k_fwd3 pays ~4.2 clk per activation instruction, tools/dmma_chain.cu (pure register DFMA chains) measured 2.7.
// Per iteration a warp issues NA m16n8k8 MMAs (independent accumulators) and one "activation group" of NCH elements:
//   MODE 0  NCH chains x 12 dependent DFMA (register operands)               -- the dmma_chain baseline
//   MODE 1  the same 12 ops as DFMA / DADD / DMUL with immediate constants (the mix of the swish chain)
//   MODE 2  MODE 0 + NI independent integer instructions per FP64 instruction (issue-slot pressure only)
//   MODE 3  MODE 0 with an integer select on the high word between FP64 ops (ALU -> FP64 dependencies)
//   MODE 4  the kernel's swish (bnn_act: clamp + NaN fix-up + table + MUFU seed), table in shared memory
//   MODE 5  the kernel's vote-guarded fast swish (bnn_act_fast)
//   MODE 6  MODE 0 + one random shared-memory table read per chain (LDS with bank conflicts)
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o tools/fp64_mix tools/fp64_mix.cu
#include <cstdio>
#include <cuda_runtime.h>
#include "../npbnn_b200/csrc/bnn_common.cuh"

template <int MODE, int NI>
__device__ __forceinline__ double act_model(double v, double x, double y, const double* tab, int& isink) {
  if (MODE == 0 || MODE == 2 || MODE == 6) {
    double f = v;
    if (MODE == 6) f = tab[__double2loint(f) & (BNN_EXP_TAB_SIZE - 1)] * f;    // 1 DMUL + random LDS
#pragma unroll
    for (int s = 0; s < (MODE == 6 ? 11 : 12); ++s) {
      f = fma(f, x, y);
      if (MODE == 2) {
#pragma unroll
        for (int i = 0; i < NI; ++i) isink = (isink ^ (isink >> 3)) + 0x9e3779b9;   // 2 int ops per i... LOP3 + IADD
      }
    }
    return f;
  }
  if (MODE == 1) {
    double f = v;
    double t = fma(f, -2954.639443740597, 6755399441055744.0);
    double kd = t - 6755399441055744.0;
    double rs = fma(kd, 0.0003384507717577858, f);
    double q = fma(rs, -1.66666666666666657e-01, 0.5);
    double r2 = rs * rs;
    double p = fma(r2, q, -rs);
    double res = fma(x, p, x);
    double d = res + 1.0;
    double e = fma(-d, y, 1.0);
    e = fma(e, e, e);
    double yy = fma(y, e, y);
    return f * yy;
  }
  if (MODE == 3) {
    double f = v;
#pragma unroll
    for (int s = 0; s < 12; ++s) {
      f = fma(f, x, y);
      if (s % 3 == 0) {
        const int hi = __double2hiint(f);
        const bool big = (hi & 0x7fffffff) >= 0x40862000;
        f = big ? __hiloint2double((hi & 0x80000000) | 0x40862000, 0) : f;
      }
    }
    return f;
  }
  if (MODE == 4) return bnn_act<BNN_ACT_SWISH>(v, 0.0, tab);
  return bnn_act_fast<BNN_ACT_SWISH>(v, 0.0, tab);
}

template <int NW, int NA, int NCH, int MODE, int NI>
__global__ void __launch_bounds__(NW * 32, 1) k_mix(double* out, int iters, double x, double y, const double* gtab) {
  __shared__ double tab[BNN_EXP_TAB_SIZE];
  for (int i = threadIdx.x; i < BNN_EXP_TAB_SIZE; i += blockDim.x) tab[i] = gtab[i];
  __syncthreads();
  double c[NA > 0 ? NA : 1][4];
#pragma unroll
  for (int i = 0; i < (NA > 0 ? NA : 1); ++i) c[i][0] = c[i][1] = c[i][2] = c[i][3] = 0.0;
  double a[4], b[2], f[NCH > 0 ? NCH : 1];
  f[0] = 0.0;
#pragma unroll
  for (int i = 0; i < 4; ++i) a[i] = x + threadIdx.x * 1e-6 + i * 1e-3;
  b[0] = y + threadIdx.x * 1e-6; b[1] = y * 0.5;
#pragma unroll
  for (int i = 0; i < NCH; ++i) f[i] = 0.3 * i + threadIdx.x * 1e-3;
  int isink = threadIdx.x;
  const double off = 0.25 + (threadIdx.x & 31) * 0.37;     // per-lane fixed points => scattered table reads
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < NA; ++i) dmma16x8x8(c[i], a[0], a[1], a[2], a[3], b[0], b[1]);
#pragma unroll
    for (int q = 0; q < NCH; ++q) f[q] = act_model<MODE, NI>(f[q], x, y, tab, isink) + ((MODE >= 4) ? off : 0.0);
  }
  double s = isink;
#pragma unroll
  for (int i = 0; i < (NA > 0 ? NA : 1); ++i) s += c[i][0] + c[i][1] + c[i][2] + c[i][3];
#pragma unroll
  for (int i = 0; i < NCH; ++i) s += f[i];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

template <int NW, int NA, int NCH, int MODE, int NI>
void run(int sms, double* out, const double* tab, const char* what) {
  const int iters = 4096 / (NA > 0 ? NA : 4);
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  k_mix<NW, NA, NCH, MODE, NI><<<sms, NW * 32>>>(out, iters, 1.0000001, 1e-9, tab);
  cudaEventRecord(e0);
  for (int r = 0; r < 5; ++r) k_mix<NW, NA, NCH, MODE, NI><<<sms, NW * 32>>>(out, iters, 1.0000001, 1e-9, tab);
  cudaEventRecord(e1);
  cudaEventSynchronize(e1);
  float ms;
  cudaEventElapsedTime(&ms, e0, e1);
  ms /= 5;
  const double clk = ms * 1e-3 * 1.965e9;
  const double wps = NW / 4.0;                                   // warps per sub-partition
  const double per_smsp_mma = (double)iters * NA * wps;
  const int fp_per_el = (MODE >= 4) ? 13 : 12;                   // swish: 12 + the "+ 0.25" that keeps the chain alive
  const double per_smsp_fp = (double)iters * NCH * fp_per_el * wps;
  printf("%-34s warps=%2d mma/it=%d act/it=%2d  %.3f ms  clk/mma(all-in) %.1f  clk per FP64 instr beyond 64.4/mma: %.2f  err=%s\n",
         what, NW, NA, NCH, ms, NA ? clk / per_smsp_mma : 0.0, NCH ? (clk - 64.4 * per_smsp_mma) / per_smsp_fp : 0.0,
         cudaGetErrorString(cudaGetLastError()));
}

int main() {
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, 0);
  const int sms = prop.multiProcessorCount;
  double *out, *tab;
  cudaMalloc(&out, sizeof(double) * sms * 1024);
  cudaMalloc(&tab, sizeof(double) * BNN_EXP_TAB_SIZE);
  double h[BNN_EXP_TAB_SIZE];
  for (int i = 0; i < BNN_EXP_TAB_SIZE; ++i) h[i] = exp2((double)i / BNN_EXP_TAB_SIZE);
  cudaMemcpy(tab, h, sizeof(h), cudaMemcpyHostToDevice);
  printf("%s, %d SMs\n", prop.name, sms);
  run<12, 8, 0, 0, 0>(sms, out, tab, "mma only");
  run<12, 4, 4, 0, 0>(sms, out, tab, "12 dfma chain");
  run<12, 4, 4, 1, 0>(sms, out, tab, "dfma/dadd/dmul + immediates");
  run<12, 4, 4, 2, 1>(sms, out, tab, "dfma + 2 int per fp64");
  run<12, 4, 4, 2, 2>(sms, out, tab, "dfma + 4 int per fp64");
  run<12, 4, 4, 3, 0>(sms, out, tab, "dfma + int select on hi word");
  run<12, 4, 4, 6, 0>(sms, out, tab, "dfma + random LDS");
  run<12, 4, 4, 4, 0>(sms, out, tab, "kernel swish (bnn_act)");
  run<12, 4, 4, 5, 0>(sms, out, tab, "kernel swish fast path");
  run<12, 4, 8, 4, 0>(sms, out, tab, "kernel swish (bnn_act) x8");
  run<12, 4, 8, 5, 0>(sms, out, tab, "kernel swish fast path x8");
  run<12, 8, 4, 4, 0>(sms, out, tab, "kernel swish, 8 mma per 4 act");
  run<12, 8, 4, 5, 0>(sms, out, tab, "fast swish, 8 mma per 4 act");
  run<16, 4, 4, 0, 0>(sms, out, tab, "12 dfma chain");
  run<16, 4, 4, 4, 0>(sms, out, tab, "kernel swish (bnn_act)");
  run<16, 4, 4, 5, 0>(sms, out, tab, "kernel swish fast path");
  run<8, 4, 4, 4, 0>(sms, out, tab, "kernel swish (bnn_act)");
  run<8, 4, 4, 5, 0>(sms, out, tab, "kernel swish fast path");
  run<24, 4, 4, 4, 0>(sms, out, tab, "kernel swish (bnn_act)");
  run<24, 4, 4, 5, 0>(sms, out, tab, "kernel swish fast path");
  run<12, 0, 8, 4, 0>(sms, out, tab, "kernel swish alone (no mma)");
  run<12, 0, 8, 5, 0>(sms, out, tab, "fast swish alone (no mma)");
  run<12, 0, 8, 0, 0>(sms, out, tab, "dfma chains alone (no mma)");
  return 0;
}
