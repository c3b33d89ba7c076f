// Pipe-rate microbenchmarks on sm_100a: legacy mma.sync variants, the integer ops used by the NTT butterflies and the FP64 ops
// of a Shoup quotient taken on the FP64 pipe (bfly.cu kinds 4..7), alone and interleaved with mad.lo to show whether the two
// pipes issue concurrently.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o pipes pipes.cu ; prints per-SM per-clock rates.
#include <cstdio>
#include <cstdint>
#include <cuda_runtime.h>
#include <cuda_fp16.h>

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %d\n", cudaGetErrorString(e), __LINE__); return 1; } } while (0)

constexpr int ITER = 2048;
constexpr int NACC = 8;

__global__ void k_imma_u8(int* out, int seed) {
  int acc[NACC][4] = {};
  unsigned a[4] = {(unsigned)seed, (unsigned)seed + 1, (unsigned)seed + 2, (unsigned)seed + 3}, b[2] = {(unsigned)seed * 3, (unsigned)seed * 5};
  for (int it = 0; it < ITER; it++) {
#pragma unroll
    for (int j = 0; j < NACC; j++)
      asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.u8.u8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                   : "+r"(acc[j][0]), "+r"(acc[j][1]), "+r"(acc[j][2]), "+r"(acc[j][3])
                   : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
  }
  int s = 0;
  for (int j = 0; j < NACC; j++) for (int k = 0; k < 4; k++) s += acc[j][k];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
__global__ void k_hmma_f16(float* out, int seed) {
  float acc[NACC][4] = {};
  unsigned a[4] = {(unsigned)seed, (unsigned)seed + 1, (unsigned)seed + 2, (unsigned)seed + 3}, b[2] = {(unsigned)seed * 3, (unsigned)seed * 5};
  for (int it = 0; it < ITER; it++) {
#pragma unroll
    for (int j = 0; j < NACC; j++)
      asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                   : "+f"(acc[j][0]), "+f"(acc[j][1]), "+f"(acc[j][2]), "+f"(acc[j][3])
                   : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
  }
  float s = 0;
  for (int j = 0; j < NACC; j++) for (int k = 0; k < 4; k++) s += acc[j][k];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
__global__ void k_hmma_bf16(float* out, int seed) {
  float acc[NACC][4] = {};
  unsigned a[4] = {(unsigned)seed, (unsigned)seed + 1, (unsigned)seed + 2, (unsigned)seed + 3}, b[2] = {(unsigned)seed * 3, (unsigned)seed * 5};
  for (int it = 0; it < ITER; it++) {
#pragma unroll
    for (int j = 0; j < NACC; j++)
      asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                   : "+f"(acc[j][0]), "+f"(acc[j][1]), "+f"(acc[j][2]), "+f"(acc[j][3])
                   : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
  }
  float s = 0;
  for (int j = 0; j < NACC; j++) for (int k = 0; k < 4; k++) s += acc[j][k];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
__global__ void k_hmma_f16acc(unsigned* out, int seed) {      // f16 accumulate
  unsigned acc[NACC][2] = {};
  unsigned a[4] = {(unsigned)seed, (unsigned)seed + 1, (unsigned)seed + 2, (unsigned)seed + 3}, b[2] = {(unsigned)seed * 3, (unsigned)seed * 5};
  for (int it = 0; it < ITER; it++) {
#pragma unroll
    for (int j = 0; j < NACC; j++)
      asm volatile("mma.sync.aligned.m16n8k16.row.col.f16.f16.f16.f16 {%0,%1}, {%2,%3,%4,%5}, {%6,%7}, {%0,%1};"
                   : "+r"(acc[j][0]), "+r"(acc[j][1])
                   : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
  }
  unsigned s = 0;
  for (int j = 0; j < NACC; j++) for (int k = 0; k < 2; k++) s += acc[j][k];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
__global__ void k_imma_s4like_k64(int* out, int seed) {        // u8 m8n8k16 small shape for comparison
  int acc[NACC][2] = {};
  unsigned a = seed, b = seed * 3;
  for (int it = 0; it < ITER; it++) {
#pragma unroll
    for (int j = 0; j < NACC; j++)
      asm volatile("mma.sync.aligned.m8n8k16.row.col.s32.u8.u8.s32 {%0,%1}, {%2}, {%3}, {%0,%1};"
                   : "+r"(acc[j][0]), "+r"(acc[j][1]) : "r"(a), "r"(b));
  }
  int s = 0;
  for (int j = 0; j < NACC; j++) for (int k = 0; k < 2; k++) s += acc[j][k];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

// integer ops: 8 independent chains per thread
template <int OP>
__global__ void k_int(unsigned* out, unsigned seed, unsigned m) {
  unsigned x[8];
#pragma unroll
  for (int j = 0; j < 8; j++) x[j] = seed + j * 77u + threadIdx.x;
  for (int it = 0; it < ITER; it++) {
#pragma unroll
    for (int j = 0; j < 8; j++) {
      if (OP == 0) asm volatile("mul.hi.u32 %0, %0, %1;" : "+r"(x[j]) : "r"(m));
      if (OP == 1) asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(x[j]) : "r"(m), "r"(seed));
      if (OP == 2) asm volatile("add.u32 %0, %0, %1;" : "+r"(x[j]) : "r"(m));
      if (OP == 3) asm volatile("min.u32 %0, %0, %1;" : "+r"(x[j]) : "r"(m + it));
      if (OP == 4) { unsigned long long w; asm volatile("mul.wide.u32 %0, %1, %2;" : "=l"(w) : "r"(x[j]), "r"(m)); x[j] = (unsigned)(w >> 32) ^ (unsigned)w; }
      if (OP == 5) { asm volatile("mul.hi.u32 %0, %0, %1;" : "+r"(x[j]) : "r"(m)); asm volatile("add.u32 %0, %0, %1;" : "+r"(x[j]) : "r"(seed)); asm volatile("min.u32 %0, %0, %1;" : "+r"(x[j]) : "r"(m + it)); }
      if (OP == 6) { asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(x[j]) : "r"(m), "r"(seed)); asm volatile("add.u32 %0, %0, %1;" : "+r"(x[j]) : "r"(m)); }
    }
  }
  unsigned s = 0;
#pragma unroll
  for (int j = 0; j < 8; j++) s ^= x[j];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

// FP64 ops: 8 independent chains per thread.  OP 3 interleaves one mad.lo.u32 chain step with one fma.rm.f64 chain step.
template <int OP>
__global__ void k_f64(unsigned* out, unsigned seed, double m) {
  double x[8];
  unsigned u[8];
#pragma unroll
  for (int j = 0; j < 8; j++) { x[j] = 1.0 + (seed + j * 77u + threadIdx.x) * 0x1p-40; u[j] = seed + j * 77u + threadIdx.x; }
  for (int it = 0; it < ITER; it++) {
#pragma unroll
    for (int j = 0; j < 8; j++) {
      if (OP == 0) asm volatile("fma.rn.f64 %0, %0, %1, %2;" : "+d"(x[j]) : "d"(m), "d"(-m));
      if (OP == 1) asm volatile("fma.rm.f64 %0, %0, %1, %2;" : "+d"(x[j]) : "d"(m), "d"(-m));
      if (OP == 2) asm volatile("add.f64 %0, %0, %1;" : "+d"(x[j]) : "d"(m));
      if (OP == 3) {
        asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(u[j]) : "r"(seed), "r"(seed));
        asm volatile("fma.rm.f64 %0, %0, %1, %2;" : "+d"(x[j]) : "d"(m), "d"(-m));
      }
    }
  }
  unsigned s = 0;
#pragma unroll
  for (int j = 0; j < 8; j++) s ^= (unsigned)__double2loint(x[j]) ^ u[j];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

template <typename F>
float time_ms(F launch) {
  cudaEvent_t a, b;
  cudaEventCreate(&a); cudaEventCreate(&b);
  launch(); launch();
  cudaDeviceSynchronize();
  cudaEventRecord(a);
  for (int i = 0; i < 5; i++) launch();
  cudaEventRecord(b);
  cudaEventSynchronize(b);
  float ms; cudaEventElapsedTime(&ms, a, b);
  return ms / 5;
}

int main() {
  cudaDeviceProp p; CK(cudaGetDeviceProperties(&p, 0));
  int sms = p.multiProcessorCount; int khz; CK(cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, 0));
  const double clk = 1.965e9;   // boost clock under load on this pool (bench.py's clock sampler)
  printf("device %s, %d SMs, attr clock %d kHz, assuming %.3f GHz\n", p.name, sms, khz, clk / 1e9);
  const int ctas = sms * 4, thr = 256;
  void* buf; CK(cudaMalloc(&buf, (size_t)ctas * thr * 8));
  const double warps = (double)ctas * thr / 32;
  auto rep = [&](const char* name, float ms, double macs_per_warp_instr, double instrs_per_iter) {
    double winst = warps * ITER * instrs_per_iter;
    double per_clk_sm = winst / (ms * 1e-3 * clk) / sms;
    printf("%-28s %8.3f ms  %7.3f warp-instr/clk/SM  %9.1f MAC/clk/SM\n", name, ms, per_clk_sm, per_clk_sm * macs_per_warp_instr);
  };
  rep("imma m16n8k32 u8", time_ms([&] { k_imma_u8<<<ctas, thr>>>((int*)buf, 3); }), 16 * 8 * 32, NACC);
  rep("imma m8n8k16 u8", time_ms([&] { k_imma_s4like_k64<<<ctas, thr>>>((int*)buf, 3); }), 8 * 8 * 16, NACC);
  rep("hmma m16n8k16 f16->f32", time_ms([&] { k_hmma_f16<<<ctas, thr>>>((float*)buf, 3); }), 16 * 8 * 16, NACC);
  rep("hmma m16n8k16 bf16->f32", time_ms([&] { k_hmma_bf16<<<ctas, thr>>>((float*)buf, 3); }), 16 * 8 * 16, NACC);
  rep("hmma m16n8k16 f16->f16", time_ms([&] { k_hmma_f16acc<<<ctas, thr>>>((unsigned*)buf, 3); }), 16 * 8 * 16, NACC);
  rep("mul.hi.u32", time_ms([&] { k_int<0><<<ctas, thr>>>((unsigned*)buf, 3, 12345677u); }), 32, 8);
  rep("mad.lo.u32", time_ms([&] { k_int<1><<<ctas, thr>>>((unsigned*)buf, 3, 12345677u); }), 32, 8);
  rep("add.u32", time_ms([&] { k_int<2><<<ctas, thr>>>((unsigned*)buf, 3, 12345677u); }), 32, 8);
  rep("min.u32", time_ms([&] { k_int<3><<<ctas, thr>>>((unsigned*)buf, 3, 12345677u); }), 32, 8);
  rep("mul.wide.u32 (+xor)", time_ms([&] { k_int<4><<<ctas, thr>>>((unsigned*)buf, 3, 12345677u); }), 32, 8);
  rep("mulhi+add+min (3 instr)", time_ms([&] { k_int<5><<<ctas, thr>>>((unsigned*)buf, 3, 12345677u); }), 32, 24);
  rep("mad+add (2 instr)", time_ms([&] { k_int<6><<<ctas, thr>>>((unsigned*)buf, 3, 12345677u); }), 32, 16);
  rep("fma.rn.f64", time_ms([&] { k_f64<0><<<ctas, thr>>>((unsigned*)buf, 3, 1.0000001); }), 32, 8);
  rep("fma.rm.f64", time_ms([&] { k_f64<1><<<ctas, thr>>>((unsigned*)buf, 3, 1.0000001); }), 32, 8);
  rep("add.f64", time_ms([&] { k_f64<2><<<ctas, thr>>>((unsigned*)buf, 3, 1.0000001); }), 32, 8);
  rep("mad.lo.u32 + fma.rm.f64 (2)", time_ms([&] { k_f64<3><<<ctas, thr>>>((unsigned*)buf, 3, 1.0000001); }), 32, 16);
  CK(cudaDeviceSynchronize());
  CK(cudaGetLastError());
  return 0;
}
