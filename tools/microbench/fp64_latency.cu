// Dependent-issue latency of the fp64 operations the sampler's sequential paths are made of (one warp, one SM),
// and of rc_log / rc_exp / Philox as compiled for the kernels (-fmad=false).
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -fmad=false -o fp64_latency fp64_latency.cu
#include <cstdio>
#include <cuda_runtime.h>
#include "../../redclust.jl_b200/csrc/rc_math.h"
#include "../../redclust.jl_b200/csrc/rc_rng.h"
template <int OP>
__global__ void k(double* out, long long* cyc, double a, double b, int iters) {
  double x = a + threadIdx.x * 1e-9;
  long long t0 = clock64();
  for (int i = 0; i < iters; ++i) {
    if (OP == 0) x = x + b;
    if (OP == 1) x = x * b;
    if (OP == 2) x = fma(x, b, a);
    if (OP == 3) x = rc_log(x) + 3.0;
    if (OP == 4) x = rc_exp(x * 1e-3) + 1.0;
    if (OP == 5) { rc_draw d = rc_draw2(12345ull, (uint32_t)i, 10, 0, (uint32_t)__double2int_rn(x), 3); x = d.u0 + 1.0; }
    if (OP == 6) x = rc_dequant((long long)(x * 1e6), 20) + 1.5;
    if (OP == 7) x = -rc_log(-rc_log(x * 1e-3 + 0.2)) + 2.0;
  }
  long long t1 = clock64();
  out[threadIdx.x] = x;
  if (threadIdx.x == 0) *cyc = t1 - t0;
}
int main() {
  double* out; long long* cyc;
  cudaMalloc(&out, 8 * 1024); cudaMalloc(&cyc, 8);
  const char* names[] = {"DADD", "DMUL", "DFMA", "rc_log(+add)", "rc_exp(+mul,add)", "philox draw2 (+cvt)", "rc_dequant(+cvt)", "gumbel -log(-log u)"};
  const int iters = 2000;
  for (int warps = 1; warps <= 16; warps *= 4)
  for (int op = 0; op < 8; ++op) {
    long long h = 0;
    for (int rep = 0; rep < 2; ++rep) {
      switch (op) {
        case 0: k<0><<<1, 32 * warps>>>(out, cyc, 1.5, 1.000001, iters); break;
        case 1: k<1><<<1, 32 * warps>>>(out, cyc, 1.5, 1.000001, iters); break;
        case 2: k<2><<<1, 32 * warps>>>(out, cyc, 1.5, 0.999, iters); break;
        case 3: k<3><<<1, 32 * warps>>>(out, cyc, 1.5, 1.0, iters); break;
        case 4: k<4><<<1, 32 * warps>>>(out, cyc, 1.5, 1.0, iters); break;
        case 5: k<5><<<1, 32 * warps>>>(out, cyc, 1.5, 1.0, iters); break;
        case 6: k<6><<<1, 32 * warps>>>(out, cyc, 1.5, 1.0, iters); break;
        case 7: k<7><<<1, 32 * warps>>>(out, cyc, 1.5, 1.0, iters); break;
      }
      cudaDeviceSynchronize();
      cudaMemcpy(&h, cyc, 8, cudaMemcpyDeviceToHost);
    }
    printf("warps=%2d %-22s %8.1f cycles per dependent op\n", warps, names[op], (double)h / iters);
  }
  return 0;
}
