// Shared device/host definitions for the B200 PIR kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <stdexcept>
#include "ntt_core.cuh"

namespace b200pir {

typedef unsigned __int128 u128;

// Constants every kernel needs; passed by value (lives in the kernel parameter constant bank).
struct DevParams {
  uint32_t q[2];               // CRT moduli (lib/spiral-rs/src/util.rs:246-247)
  uint64_t cr1[2];             // floor(2^64 / q_n)            (arith.rs:122-134 Barrett ratio, high word)
  uint64_t modulus;            // q = q0*q1
  uint64_t cr1_mod;            // floor(2^64 / q)
  uint32_t q1_inv_mod_q0;      // Garner constant for the CRT lift
  const Twiddle* fwd[2];       // [n] -> 2048 (W, W') forward, bit-reversed table order (ntt.rs:39-65)
  const Twiddle* inv[2];       // inverse (pre-halved) tables
  const Twiddle* inv_lz[2];    // inverse tables of the relaxed-range transform (un-halved, 1/N in the last stage; ntt_tables.hpp)
  uint32_t mu58[2];            // floor(2^58 / q_n): 32-bit Barrett for values < 2^57 (barrett57)
};

// x mod q for any 64-bit x  (== arith.rs:122-134 barrett_raw_u64)
__device__ __forceinline__ uint32_t barrett64(uint64_t x, uint64_t cr1, uint32_t q) {
  uint64_t t = __umul64hi(x, cr1);
  uint64_t r = x - t * (uint64_t)q;
  uint32_t r32 = (uint32_t)r;                 // r < 2q < 2^32
  return ntt_min(r32, r32 - q);
}
// x mod q for x < 2^57 (2^27 < q < 2^28) with 32-bit operations: the quotient estimate floor((x >> 26) mu / 2^32), mu =
// floor(2^58 / q), is the true quotient or one less (x / 2^58 + 2^26 / q < 1), so the remainder estimate lies in [0, 2q)
// and its low 32 bits suffice.  One IMAD.HI + one IMAD instead of a 64 x 64 -> high multiply.
__device__ __forceinline__ uint32_t barrett57(uint64_t x, uint32_t mu, uint32_t q) {
  const uint32_t qh = __umulhi((uint32_t)(x >> 26), mu);
  const uint32_t r = (uint32_t)x - qh * q;
  return ntt_min(r, r - q);
}
// x mod q (56-bit q) for any 64-bit x
__device__ __forceinline__ uint64_t barrett64_big(uint64_t x, uint64_t cr1, uint64_t q) {
  uint64_t t = __umul64hi(x, cr1);
  uint64_t r = x - t * q;
  return r >= q ? r - q : r;
}
// (a + b) mod q for canonical a, b
__device__ __forceinline__ uint32_t addmod(uint32_t a, uint32_t b, uint32_t q) {
  uint32_t s = a + b;
  return ntt_min(s, s - q);
}
// CRT lift of (x mod q0, y mod q1) to [0, q): equals params.rs:207-214 crt_compose_2 (the unique
// representative), computed with Garner's formula instead of the 128-bit Barrett.
__device__ __forceinline__ uint64_t crt_compose(uint32_t x, uint32_t y, const DevParams& P) {
  uint32_t d = x >= y ? x - y : x + P.q[0] - y;          // y < q1 < q0
  uint32_t m = barrett57((uint64_t)d * P.q1_inv_mod_q0, P.mu58[0], P.q[0]);       // d, q1^-1 < q0 < 2^28: product < 2^56
  return (uint64_t)y + (uint64_t)P.q[1] * m;
}
// gadget digit k of a raw coefficient (gadget.rs:34-60)
// bits <= 32 for every parameter set (bits_per of t >= 2 is at most 29), so a digit is the low word of v >> sh: two
// clamped funnel shifts (the second one is a no-op until sh >= 32 and yields 0 from sh >= 64) and one AND.
__device__ __forceinline__ uint32_t gadget_digit(uint64_t v, int k, int bits, uint64_t mask) {
  const int sh = k * bits;
  const uint32_t lo = (uint32_t)v, hi = (uint32_t)(v >> 32);
  const uint32_t w = __funnelshift_rc(__funnelshift_rc(lo, hi, sh), 0u, sh > 32 ? sh - 32 : 0);
  return w & (uint32_t)mask;
}
// Number of leading gadget digits that can be non-zero for values v <= bound: digit k of every such v is zero once
// bound < 2^(k bits).  With modulus_log2 = 56 and t = 8 (bits = 8), digit 7 covers bits 56..63 and is always zero because
// q0 q1 < 2^56.  Its forward transform is then zero mod q, so callers that reduce their accumulators mod q may skip it.
__device__ __forceinline__ int gadget_live_digits(int t, int bits, uint64_t bound) {
  int k = 0;
  while (k < t && k * bits < 64 && (bound >> (k * bits)) != 0) k++;
  return k;
}

__device__ __forceinline__ uint4 ld_stream_v4(const uint4* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}

// ---- host-side error plumbing
struct Error : std::runtime_error {
  int code;
  Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};
#define B200_CUDA(expr)                                                                              \
  do {                                                                                               \
    cudaError_t _e = (expr);                                                                         \
    if (_e != cudaSuccess)                                                                           \
      throw ::b200pir::Error(-3, std::string(#expr) + ": " + cudaGetErrorString(_e));               \
  } while (0)

}  // namespace b200pir
