// Butterfly-rate microbenchmark on sm_100a: the NTT butterflies of sdk_b200/csrc/ntt_core.cuh on register-resident values
// (no shared memory, no barriers), i.e. the arithmetic bound of the transforms.  Prints warp-butterflies per clock per SM and the
// equivalent clocks per 2048-point transform (11 264 butterflies = 352 warp-butterflies).
// Kinds 4..7 take the Shoup quotient floor(y W / q) (or one less) on the FP64 pipe instead of mul.hi.u32, with wd = M 2^-53,
// M = floor(W 2^53 / q):  "dadd"  yd = (2^52 + y) - 2^52, quot = lo(fma.rm(yd, wd, 2^52));
//                          "1fma"  quot = lo(fma.rm(2^52 + y, wd, c)) with the per-twiddle constant c = 2^52 (1 - wd).
// They measured no faster than kinds 1 and 3 (DESIGN.md section 4.2), so the transforms keep the integer quotient.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -I ../../sdk_b200/csrc -o bfly bfly.cu
#include <cstdio>
#include <cstdint>
#include <cuda_runtime.h>
#include "ntt_core.cuh"

using namespace b200pir;
constexpr int ITER = 512;

struct TwF { uint32_t w; double wd, c; };
template <bool ONE_FMA>
__device__ __forceinline__ uint32_t quot_f64(uint32_t y, const TwF& t) {
  const double yb = __hiloint2double(0x43300000, (int)y);              // 2^52 + y, exact
  if (ONE_FMA) return (uint32_t)__double2loint(__fma_rd(yb, t.wd, t.c));
  return (uint32_t)__double2loint(__fma_rd(yb - 0x1p52, t.wd, 0x1p52));
}
template <bool ONE_FMA>
__device__ __forceinline__ void bfly_fwd_lz_f(uint32_t& x, uint32_t& y, const TwF& tw, uint32_t q, uint32_t two_q) {
  const uint32_t t = tw.w * y - quot_f64<ONE_FMA>(y, tw) * q;
  y = x + two_q - t;
  x = x + t;
}
template <bool ONE_FMA>
__device__ __forceinline__ void bfly_inv_nh_f(uint32_t& x, uint32_t& y, const TwF& tw, uint32_t q, uint32_t off, uint32_t eight_q) {
  const uint32_t tt = x - y + off;
  const uint32_t s = ntt_c8(x + y, eight_q);
  x = s;
  y = tw.w * tt - quot_f64<ONE_FMA>(tt, tw) * q;
}

template <int KIND>
__global__ void __launch_bounds__(256) k_bfly(uint32_t* out, uint32_t seed, uint32_t q) {
  uint32_t x[8];
  Twiddle tw[4];
#pragma unroll
  for (int j = 0; j < 8; j++) x[j] = (seed + j * 7777u + threadIdx.x * 31u) % q;
#pragma unroll
  for (int j = 0; j < 4; j++) { tw[j].w = (seed * (j + 3) + threadIdx.x) % q; tw[j].wp = (uint32_t)(((uint64_t)tw[j].w << 32) / q); }
  TwF tf[4];
#pragma unroll
  for (int j = 0; j < 4; j++) {                                       // M = floor(w 2^53 / q) by long division
    const uint64_t hi = ((uint64_t)tw[j].w << 32) / q, rem = ((uint64_t)tw[j].w << 32) % q;
    const uint64_t m = (hi << 21) | ((rem << 21) / q);
    tf[j].w = tw[j].w; tf[j].wd = (double)m * 0x1p-53; tf[j].c = 0x1p52 - (double)m * 0x1p-1;
  }
  const uint32_t two_q = 2 * q;
  for (int it = 0; it < ITER; it++) {
    // 12 butterflies per trip: the three stages of a radix-8 pass
    if (KIND == 0) {
#pragma unroll
      for (int a = 0; a < 4; a++) bfly_fwd(x[a], x[a + 4], tw[0], q, two_q);
#pragma unroll
      for (int h = 0; h < 2; h++) { bfly_fwd(x[4 * h], x[4 * h + 2], tw[1 + h], q, two_q); bfly_fwd(x[4 * h + 1], x[4 * h + 3], tw[1 + h], q, two_q); }
#pragma unroll
      for (int h = 0; h < 4; h++) bfly_fwd(x[2 * h], x[2 * h + 1], tw[h], q, two_q);
    } else if (KIND == 1) {
#pragma unroll
      for (int a = 0; a < 4; a++) bfly_fwd_lz(x[a], x[a + 4], tw[0], q, two_q);
#pragma unroll
      for (int a = 0; a < 8; a++) x[a] = ntt_c8(x[a], 4 * two_q);      // keeps the endless loop in range (1 per 12 butterflies, as in pass C)
#pragma unroll
      for (int h = 0; h < 2; h++) { bfly_fwd_lz(x[4 * h], x[4 * h + 2], tw[1 + h], q, two_q); bfly_fwd_lz(x[4 * h + 1], x[4 * h + 3], tw[1 + h], q, two_q); }
#pragma unroll
      for (int h = 0; h < 4; h++) bfly_fwd_lz(x[2 * h], x[2 * h + 1], tw[h], q, two_q);
#pragma unroll
      for (int a = 0; a < 8; a++) x[a] = ntt_c8(x[a], 4 * two_q);
    } else if (KIND == 2) {
#pragma unroll
      for (int a = 0; a < 4; a++) bfly_inv(x[a], x[a + 4], tw[0], q, two_q);
#pragma unroll
      for (int h = 0; h < 2; h++) { bfly_inv(x[4 * h], x[4 * h + 2], tw[1 + h], q, two_q); bfly_inv(x[4 * h + 1], x[4 * h + 3], tw[1 + h], q, two_q); }
#pragma unroll
      for (int h = 0; h < 4; h++) bfly_inv(x[2 * h], x[2 * h + 1], tw[h], q, two_q);
    } else if (KIND == 4 || KIND == 6) {
      constexpr bool F1 = KIND == 6;
#pragma unroll
      for (int a = 0; a < 4; a++) bfly_fwd_lz_f<F1>(x[a], x[a + 4], tf[0], q, two_q);
#pragma unroll
      for (int a = 0; a < 8; a++) x[a] = ntt_c8(x[a], 4 * two_q);
#pragma unroll
      for (int h = 0; h < 2; h++) { bfly_fwd_lz_f<F1>(x[4 * h], x[4 * h + 2], tf[1 + h], q, two_q); bfly_fwd_lz_f<F1>(x[4 * h + 1], x[4 * h + 3], tf[1 + h], q, two_q); }
#pragma unroll
      for (int h = 0; h < 4; h++) bfly_fwd_lz_f<F1>(x[2 * h], x[2 * h + 1], tf[h], q, two_q);
#pragma unroll
      for (int a = 0; a < 8; a++) x[a] = ntt_c8(x[a], 4 * two_q);
    } else if (KIND == 5 || KIND == 7) {
      constexpr bool F1 = KIND == 7;
#pragma unroll
      for (int a = 0; a < 4; a++) bfly_inv_nh_f<F1>(x[a], x[a + 4], tf[0], q, 4 * two_q, 4 * two_q);
#pragma unroll
      for (int h = 0; h < 2; h++) { bfly_inv_nh_f<F1>(x[4 * h], x[4 * h + 2], tf[1 + h], q, 4 * two_q, 4 * two_q); bfly_inv_nh_f<F1>(x[4 * h + 1], x[4 * h + 3], tf[1 + h], q, 4 * two_q, 4 * two_q); }
#pragma unroll
      for (int h = 0; h < 4; h++) bfly_inv_nh_f<F1>(x[2 * h], x[2 * h + 1], tf[h], q, 4 * two_q, 4 * two_q);
    } else {
#pragma unroll
      for (int a = 0; a < 4; a++) bfly_inv_nh<true>(x[a], x[a + 4], tw[0], q, 4 * two_q, 4 * two_q);
#pragma unroll
      for (int h = 0; h < 2; h++) { bfly_inv_nh<true>(x[4 * h], x[4 * h + 2], tw[1 + h], q, 4 * two_q, 4 * two_q); bfly_inv_nh<true>(x[4 * h + 1], x[4 * h + 3], tw[1 + h], q, 4 * two_q, 4 * two_q); }
#pragma unroll
      for (int h = 0; h < 4; h++) bfly_inv_nh<true>(x[2 * h], x[2 * h + 1], tw[h], q, 4 * two_q, 4 * two_q);
    }
  }
  uint32_t s = 0;
#pragma unroll
  for (int j = 0; j < 8; j++) s ^= x[j];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

int main() {
  cudaDeviceProp p; cudaGetDeviceProperties(&p, 0);
  const int sms = p.multiProcessorCount;
  const double clk = 1.965e9;
  uint32_t* buf; cudaMalloc(&buf, (size_t)sms * 8 * 256 * 4);
  const char* names[8] = {"forward, corrected per butterfly (round 1)", "forward, relaxed range (lz)", "inverse, halving per stage (round 1)",
                          "inverse, no halving (nh)", "forward lz, FP64 quotient (dadd)", "inverse nh, FP64 quotient (dadd)",
                          "forward lz, FP64 quotient (1fma)", "inverse nh, FP64 quotient (1fma)"};
  printf("device %s, %d SMs, assuming %.3f GHz\n", p.name, sms, clk / 1e9);
  for (int ctas_per_sm : {2, 3, 4, 8}) {
    printf("-- %d CTAs of 256 threads per SM\n", ctas_per_sm);
    for (int kind = 0; kind < 8; kind++) {
      auto launch = [&] {
        const int ctas = sms * ctas_per_sm;
        if (kind == 0) k_bfly<0><<<ctas, 256>>>(buf, 3, 268369921u);
        if (kind == 1) k_bfly<1><<<ctas, 256>>>(buf, 3, 268369921u);
        if (kind == 2) k_bfly<2><<<ctas, 256>>>(buf, 3, 268369921u);
        if (kind == 3) k_bfly<3><<<ctas, 256>>>(buf, 3, 268369921u);
        if (kind == 4) k_bfly<4><<<ctas, 256>>>(buf, 3, 268369921u);
        if (kind == 5) k_bfly<5><<<ctas, 256>>>(buf, 3, 268369921u);
        if (kind == 6) k_bfly<6><<<ctas, 256>>>(buf, 3, 268369921u);
        if (kind == 7) k_bfly<7><<<ctas, 256>>>(buf, 3, 268369921u);
      };
      launch(); cudaDeviceSynchronize();
      cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
      cudaEventRecord(a);
      for (int i = 0; i < 5; i++) launch();
      cudaEventRecord(b); cudaEventSynchronize(b);
      float ms; cudaEventElapsedTime(&ms, a, b); ms /= 5;
      const double wb = (double)sms * ctas_per_sm * 8 * ITER * 12;       // warp-butterflies
      const double per_clk_sm = wb / (ms * 1e-3 * clk) / sms;
      printf("%-46s %7.3f ms  %6.3f warp-butterflies/clk/SM  = %6.0f clk per 2048-point transform per SM\n", names[kind], ms, per_clk_sm, 352.0 / per_clk_sm);
    }
  }
  return cudaGetLastError() != cudaSuccess;
}
