// Ring-arithmetic kernels for the Spiral second dimension, query expansion and packing (sm_100a).
//
// Every kernel here runs CTAs of 512 threads = two groups of 256; group g works modulo q_g, so the
// two CRT halves of a polynomial are transformed side by side and can be CRT-lifted inside the CTA.
// A "digit external product" (gadget-decompose a raw polynomial, forward-NTT each digit polynomial,
// multiply-accumulate with the columns of an NTT-domain key matrix) is the common inner loop of
// fold_ciphertexts (server.rs:388-427), coefficient_expansion (:19-121), regev_to_gsw (:123-151)
// and pack (:429-468): it is written once (digits_mac) and fused with the surrounding inverse
// transforms, automorphisms and CRT lifts so intermediates never leave the SM.
#include "kernels.h"
#include "ntt_core4096.cuh"

namespace b200pir {

namespace {

constexpr int CTA = 512;
constexpr int HI_TW = NTT_N - 64;       // twiddle table entries 64..2047 (passes C, D)

// Table entries 0..63 (passes A and B) of every (modulus, direction) live in the constant bank: the
// index is thread-uniform (pass A) or warp-uniform (pass B), so they cost no load/store-unit traffic.
__constant__ Twiddle c_tw_lo[2][3][64];     // [n][0 = forward, 1 = inverse][index]

struct TwConst {
  int n, dir;
  __device__ __forceinline__ Twiddle operator()(int i) const { return c_tw_lo[n][dir][i]; }
  __device__ __forceinline__ void load2(int i, Twiddle (&t)[2]) const { t[0] = (*this)(i); t[1] = (*this)(i + 1); }
  __device__ __forceinline__ void load4(int i, Twiddle (&t)[4]) const {
    t[0] = (*this)(i); t[1] = (*this)(i + 1); t[2] = (*this)(i + 2); t[3] = (*this)(i + 3);
  }
};
struct TwShared {            // shared-memory copy of entries 64..2047
  const Twiddle* p;
  __device__ __forceinline__ Twiddle operator()(int i) const { return p[i - 64]; }
  __device__ __forceinline__ void load2(int i, Twiddle (&t)[2]) const {
    uint4 v = *reinterpret_cast<const uint4*>(p + (i - 64));
    t[0] = Twiddle{v.x, v.y}; t[1] = Twiddle{v.z, v.w};
  }
  __device__ __forceinline__ void load4(int i, Twiddle (&t)[4]) const {
    uint4 v = *reinterpret_cast<const uint4*>(p + (i - 64)), w = *(reinterpret_cast<const uint4*>(p + (i - 64)) + 1);
    t[0] = Twiddle{v.x, v.y}; t[1] = Twiddle{v.z, v.w}; t[2] = Twiddle{w.x, w.y}; t[3] = Twiddle{w.z, w.w};
  }
};
struct TwGlobal {            // straight from global memory through L1 (rarely used transforms)
  const Twiddle* p;
  __device__ __forceinline__ Twiddle operator()(int i) const {
    uint2 v = __ldg(reinterpret_cast<const uint2*>(p + i));
    return Twiddle{v.x, v.y};
  }
  __device__ __forceinline__ void load2(int i, Twiddle (&t)[2]) const {
    uint4 v = __ldg(reinterpret_cast<const uint4*>(p + i));
    t[0] = Twiddle{v.x, v.y}; t[1] = Twiddle{v.z, v.w};
  }
  __device__ __forceinline__ void load4(int i, Twiddle (&t)[4]) const {
    uint4 v = __ldg(reinterpret_cast<const uint4*>(p + i)), w = __ldg(reinterpret_cast<const uint4*>(p + i) + 1);
    t[0] = Twiddle{v.x, v.y}; t[1] = Twiddle{v.z, v.w}; t[2] = Twiddle{w.x, w.y}; t[3] = Twiddle{w.z, w.w};
  }
};

struct Grp {
  int tid;              // 0..255 inside the group
  int n;                // modulus index handled by this group
  uint32_t q;
  uint64_t cr1;
  const Twiddle* fwd;   // global tables
  const Twiddle* inv;
  const Twiddle* inv_lz; // relaxed-range inverse table (ntt_core.cuh "lz")
  uint32_t* smem;       // this group's NTT exchange buffer (NTT_SMEM_WORDS)
  uint32_t* smem2;      // second buffer for paired transforms (null when the kernel has none)
  const Twiddle* fwd_hi_sm;   // shared copy of fwd[64..], or null
};
struct CtaSync {
  __device__ __forceinline__ void operator()() const { __syncthreads(); }
};

// group g of a 512-thread CTA (threads 256g..256g+255) works modulo q_g
__device__ __forceinline__ Grp make_grp(const DevParams& P, uint32_t* ntt_smem) {
  Grp g;
  g.n = threadIdx.x >> 8;
  g.tid = threadIdx.x & 255;
  g.q = g.n ? P.q[1] : P.q[0];
  g.cr1 = g.n ? P.cr1[1] : P.cr1[0];
  g.fwd = g.n ? P.fwd[1] : P.fwd[0];
  g.inv = g.n ? P.inv[1] : P.inv[0];
  g.inv_lz = g.n ? P.inv_lz[1] : P.inv_lz[0];
  g.smem = ntt_smem + g.n * NTT_SMEM_WORDS;
  g.smem2 = nullptr;
  g.fwd_hi_sm = nullptr;
  return g;
}
// one 256-thread CTA per modulus (blockIdx.y = n)
__device__ __forceinline__ Grp make_grp_single(const DevParams& P, uint32_t* ntt_smem, int n) {
  Grp g;
  g.n = n;
  g.tid = threadIdx.x;
  g.q = n ? P.q[1] : P.q[0];
  g.cr1 = n ? P.cr1[1] : P.cr1[0];
  g.fwd = n ? P.fwd[1] : P.fwd[0];
  g.inv = n ? P.inv[1] : P.inv[0];
  g.inv_lz = n ? P.inv_lz[1] : P.inv_lz[0];
  g.smem = ntt_smem;
  g.smem2 = nullptr;
  g.fwd_hi_sm = nullptr;
  return g;
}
// copy this group's forward table entries 64..2047 into shared memory (visible after the next barrier)
__device__ __forceinline__ void stage_fwd_twiddles(Grp& g, Twiddle* dst) {
  for (int i = g.tid; i < HI_TW; i += 256) {
    uint2 v = __ldg(reinterpret_cast<const uint2*>(g.fwd + 64 + i));
    dst[i] = Twiddle{v.x, v.y};
  }
  g.fwd_hi_sm = dst;
}
// SM = true: the kernel staged the forward hi-table with stage_fwd_twiddles()
// canonical forward transform of inputs < 4q (the old per-butterfly-corrected transform's input contract, which
// to_ntt_no_reduce's callers rely on), canonical inverse transform of inputs < 2q: relaxed-range versions (ntt_core.cuh "lz")
template <bool SM>
__device__ __forceinline__ void grp_ntt_fwd(const Grp& g, uint32_t (&x)[8]) {
  if (SM) ntt_forward_group_lz<NTT_OUT_CANON, true>(g.tid, x, g.smem, TwConst{g.n, 0}, TwShared{g.fwd_hi_sm}, g.q, CtaSync());
  else ntt_forward_group_lz<NTT_OUT_CANON, true>(g.tid, x, g.smem, TwConst{g.n, 0}, TwGlobal{g.fwd}, g.q, CtaSync());
}
__device__ __forceinline__ void grp_ntt_inv(const Grp& g, uint32_t (&x)[8]) {
  ntt_inverse_group_nh(g.tid, x, g.smem, TwConst{g.n, 2}, TwGlobal{g.inv_lz}, g.q, CtaSync());
}

// contiguous-layout load/store of 8 ntt32 words (two 16-byte accesses)
__device__ __forceinline__ void ld8(uint32_t (&x)[8], const uint32_t* p) {
  uint4 a = *reinterpret_cast<const uint4*>(p), b = *reinterpret_cast<const uint4*>(p + 4);
  x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; x[4] = b.x; x[5] = b.y; x[6] = b.z; x[7] = b.w;
}
__device__ __forceinline__ void ld8_ro(uint32_t (&x)[8], const uint32_t* p) {
  uint4 a = __ldg(reinterpret_cast<const uint4*>(p)), b = __ldg(reinterpret_cast<const uint4*>(p + 4));
  x[0] = a.x; x[1] = a.y; x[2] = a.z; x[3] = a.w; x[4] = b.x; x[5] = b.y; x[6] = b.z; x[7] = b.w;
}
__device__ __forceinline__ void st8(uint32_t* p, const uint32_t (&x)[8]) {
  *reinterpret_cast<uint4*>(p) = make_uint4(x[0], x[1], x[2], x[3]);
  *reinterpret_cast<uint4*>(p + 4) = make_uint4(x[4], x[5], x[6], x[7]);
}

template <int ROWS>
__device__ __forceinline__ void acc_reduce(uint64_t (&acc)[ROWS][8], const Grp& g) {
#pragma unroll
  for (int r = 0; r < ROWS; r++)
#pragma unroll
    for (int k = 0; k < 8; k++) acc[r][k] = barrett64(acc[r][k], g.cr1, g.q);
}

// digit k of a raw coefficient; bits == 8 (the common t = 8): digit k is byte k, and since the values are <= q < 2^56 byte 7
// is a zero byte to fill the upper three bytes with — one PRMT instead of two funnel shifts and a mask
template <bool BYTE>
__device__ __forceinline__ uint32_t gadget_digit_fast(uint64_t v, int k, int bits, uint64_t mask) {
  if (BYTE) return __byte_perm((uint32_t)v, (uint32_t)(v >> 32), 0x7770u | (uint32_t)k);
  return gadget_digit(v, k, bits, mask);
}

// acc[r][.] += sum_k  C[r][col0 + k*col_step] (.) NTT(digit_k(v))     (pointwise, this group's modulus)
// v[a] = raw coefficient at index a*256 + tid (strided layout).  c0 points at element (row 0, first
// column) of this group's modulus, offset by tid*8.  `cnt` counts products held per accumulator.
// Relaxed-range forward transforms (ntt_core.cuh "lz"): digits are < 2^19 < 2q (gadget dimensions >= 3), the outputs
// (< 16q < 2^32) go straight into the 64-bit accumulators: products < 2^60, at most 16 per accumulator between reductions.
template <int ROWS, bool SM, bool BYTE>
__device__ __forceinline__ void digits_mac_impl(uint64_t (&acc)[ROWS][8], int& cnt, const uint64_t (&v)[8], int ndig,
                                                int bits, const uint32_t* c0, size_t col_step, size_t row_step,
                                                const Grp& g) {
  const uint64_t mask = (1ull << bits) - 1;
  int k = 0;
  if (SM) {
    // two digit polynomials per trip: twice the instruction-level parallelism, half the barriers
    // (kernels that stage twiddles also provide the second exchange buffer g.smem2)
#pragma unroll 1
    for (; k + 1 < ndig; k += 2) {
      uint32_t x0[8], x1[8];
#pragma unroll
      for (int a = 0; a < 8; a++) {
        x0[a] = gadget_digit_fast<BYTE>(v[a], k, bits, mask);
        x1[a] = gadget_digit_fast<BYTE>(v[a], k + 1, bits, mask);
      }
      ntt_forward_group2_lz<NTT_OUT_LAZY16>(g.tid, x0, x1, g.smem, g.smem2, TwConst{g.n, 0}, TwShared{g.fwd_hi_sm}, g.q, CtaSync());
      if (cnt + 2 > 16) { acc_reduce<ROWS>(acc, g); cnt = 1; }
      cnt += 2;
      const uint32_t* c = c0 + (size_t)k * col_step;
#pragma unroll
      for (int r = 0; r < ROWS; r++) {
        uint32_t cv[8];
        ld8_ro(cv, c + (size_t)r * row_step);
#pragma unroll
        for (int e = 0; e < 8; e++) acc[r][e] += (uint64_t)x0[e] * cv[e];
        ld8_ro(cv, c + col_step + (size_t)r * row_step);
#pragma unroll
        for (int e = 0; e < 8; e++) acc[r][e] += (uint64_t)x1[e] * cv[e];
      }
    }
  }
#pragma unroll 1
  for (; k < ndig; k++) {
    uint32_t x[8];
#pragma unroll
    for (int a = 0; a < 8; a++) x[a] = gadget_digit_fast<BYTE>(v[a], k, bits, mask);
    if (SM) ntt_forward_group_lz<NTT_OUT_LAZY16>(g.tid, x, g.smem, TwConst{g.n, 0}, TwShared{g.fwd_hi_sm}, g.q, CtaSync());
    else ntt_forward_group_lz<NTT_OUT_LAZY16>(g.tid, x, g.smem, TwConst{g.n, 0}, TwGlobal{g.fwd}, g.q, CtaSync());
    if (cnt + 1 > 16) { acc_reduce<ROWS>(acc, g); cnt = 1; }
    cnt += 1;
    const uint32_t* c = c0 + (size_t)k * col_step;
#pragma unroll
    for (int r = 0; r < ROWS; r++) {
      uint32_t cv[8];
      ld8_ro(cv, c + (size_t)r * row_step);
#pragma unroll
      for (int e = 0; e < 8; e++) acc[r][e] += (uint64_t)x[e] * cv[e];
    }
  }
}

// one warp-uniform branch per call (not per digit): the byte-permute and the funnel-shift digit extraction as two loop bodies.
// The expansion passes ndig = gadget_live_digits(t, bits, q0 q1): its values are <= q0 q1, so the digits it leaves out are
// zero and would add only multiples of q to the accumulators, which are reduced mod q.
template <int ROWS, bool SM>
__device__ __forceinline__ void digits_mac(uint64_t (&acc)[ROWS][8], int& cnt, const uint64_t (&v)[8], int ndig,
                                           int bits, const uint32_t* c0, size_t col_step, size_t row_step,
                                           const Grp& g) {
  if (bits == 8) digits_mac_impl<ROWS, SM, true>(acc, cnt, v, ndig, bits, c0, col_step, row_step, g);
  else digits_mac_impl<ROWS, SM, false>(acc, cnt, v, ndig, bits, c0, col_step, row_step, g);
}

// CRT-lift one polynomial whose two residue vectors sit in the two groups' registers (strided layout,
// canonical) and hand the 4 coefficients this thread is responsible for to `sink(z, value)`.
// res: 2*2048-word exchange buffer.  Thread (g,tid) lifts z = a*256 + tid for a in [4g, 4g+4).
template <typename Sink>
__device__ __forceinline__ void crt_lift(const uint32_t (&x)[8], uint32_t* res, const Grp& g, const DevParams& P,
                                         Sink sink) {
  __syncthreads();                       // previous users of `res` are done
#pragma unroll
  for (int a = 0; a < 8; a++) res[g.n * POLY + a * 256 + g.tid] = x[a];
  __syncthreads();
#pragma unroll
  for (int a4 = 0; a4 < 4; a4++) {
    int z = (g.n * 4 + a4) * 256 + g.tid;
    sink(z, crt_compose(res[z], res[POLY + z], P));
  }
}

// ------------------------------------------------------------------ plain transforms
// grid = (polys, 2 moduli), 256 threads: one CTA per single-modulus transform.
__global__ void __launch_bounds__(256) k_ntt32(DevParams P, uint32_t* polys, int inverse) {
  __shared__ __align__(16) uint32_t ntt_smem[NTT_SMEM_WORDS];
  Grp g = make_grp_single(P, ntt_smem, blockIdx.y);
  uint32_t* p = polys + ((size_t)blockIdx.x * 2 + g.n) * POLY;
  uint32_t x[8];
  if (!inverse) {
#pragma unroll
    for (int a = 0; a < 8; a++) x[a] = p[a * 256 + g.tid];
    grp_ntt_fwd<false>(g, x);
    st8(p + g.tid * 8, x);
  } else {
    ld8(x, p + g.tid * 8);
    grp_ntt_inv(g, x);
#pragma unroll
    for (int a = 0; a < 8; a++) p[a * 256 + g.tid] = x[a];
  }
}
// BASELINE config #5, poly_len = 4096: one 512-thread CTA per single-modulus transform, all twiddles through L1
// (tables of 4096 (W, W') pairs per modulus and direction, built like the 2048 ones).  ntt32 layout [poly][n][4096].
__global__ void __launch_bounds__(NTT4K_THREADS)
k_ntt32_4k(uint32_t q0, uint32_t q1, const Twiddle* __restrict__ tw /* fwd0, inv0, fwd1, inv1 */, uint32_t* polys, int inverse) {
  __shared__ __align__(16) uint32_t sm[NTT4K_SMEM_WORDS];
  const int n = blockIdx.y, tid = threadIdx.x;
  const uint32_t q = n ? q1 : q0;
  uint32_t* p = polys + ((size_t)blockIdx.x * 2 + n) * NTT4K_N;
  const TwGlobal tab{tw + (size_t)(2 * n + (inverse ? 1 : 0)) * NTT4K_N};
  uint32_t x[8];
  if (!inverse) {
#pragma unroll
    for (int a = 0; a < 8; a++) x[a] = p[a * NTT4K_THREADS + tid];
    ntt4k_forward_group(tid, x, sm, tab, q, CtaSync());
    st8(p + tid * 8, x);
  } else {
    ld8(x, p + tid * 8);
    ntt4k_inverse_group(tid, x, sm, tab, q, CtaSync());
#pragma unroll
    for (int a = 0; a < 8; a++) p[a * NTT4K_THREADS + tid] = x[a];
  }
}
// u64 ABI words (ntt.rs:68 / :213 operate on &mut [u64]); values are truncated to 32 bits exactly as
// the reference's forward butterfly does (`as u32`, ntt.rs:93-94).
__global__ void __launch_bounds__(256) k_ntt_u64(DevParams P, uint64_t* polys, int inverse) {
  __shared__ __align__(16) uint32_t ntt_smem[NTT_SMEM_WORDS];
  Grp g = make_grp_single(P, ntt_smem, blockIdx.y);
  uint64_t* p = polys + ((size_t)blockIdx.x * 2 + g.n) * POLY;
  uint32_t x[8];
  if (!inverse) {
#pragma unroll
    for (int a = 0; a < 8; a++) x[a] = (uint32_t)p[a * 256 + g.tid];
    grp_ntt_fwd<false>(g, x);
#pragma unroll
    for (int k = 0; k < 8; k++) p[g.tid * 8 + k] = x[k];
  } else {
#pragma unroll
    for (int k = 0; k < 8; k++) x[k] = (uint32_t)p[g.tid * 8 + k];
    grp_ntt_inv(g, x);
#pragma unroll
    for (int a = 0; a < 8; a++) p[a * 256 + g.tid] = x[a];
  }
}
// blockIdx.z selects one of several equally shaped batches (out_stride / raw_stride words apart)
__global__ void __launch_bounds__(256) k_to_ntt(DevParams P, uint32_t* out, const uint64_t* raw, size_t out_stride,
                                                size_t raw_stride) {
  __shared__ __align__(16) uint32_t ntt_smem[NTT_SMEM_WORDS];
  Grp g = make_grp_single(P, ntt_smem, blockIdx.y);
  out += (size_t)blockIdx.z * out_stride;
  raw += (size_t)blockIdx.z * raw_stride;
  const uint64_t* src = raw + (size_t)blockIdx.x * POLY;
  uint32_t x[8];
#pragma unroll
  for (int a = 0; a < 8; a++) x[a] = barrett64(src[a * 256 + g.tid], g.cr1, g.q);
  grp_ntt_fwd<false>(g, x);
  st8(out + ((size_t)blockIdx.x * 2 + g.n) * POLY + g.tid * 8, x);
}
// raw u64 coefficients -> residue form u32 [poly][n][z] (coefficient domain), and back (CRT lift)
__global__ void k_raw_to_res(DevParams P, uint32_t* out, const uint64_t* raw, size_t polys) {
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;     // over polys * 2048
  if (idx >= polys * POLY) return;
  size_t poly = idx / POLY;
  int z = (int)(idx % POLY);
  uint64_t v = raw[idx];
  out[(poly * 2 + 0) * POLY + z] = barrett64(v, P.cr1[0], P.q[0]);
  out[(poly * 2 + 1) * POLY + z] = barrett64(v, P.cr1[1], P.q[1]);
}
__global__ void k_res_to_raw(DevParams P, uint64_t* out, const uint32_t* res, size_t polys) {
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= polys * POLY) return;
  size_t poly = idx / POLY;
  int z = (int)(idx % POLY);
  out[idx] = crt_compose(res[(poly * 2 + 0) * POLY + z], res[(poly * 2 + 1) * POLY + z], P);
}
__global__ void __launch_bounds__(CTA) k_from_ntt(DevParams P, uint64_t* out, const uint32_t* in) {
  __shared__ __align__(16) uint32_t ntt_smem[2 * NTT_SMEM_WORDS];
  __shared__ uint32_t res[2 * POLY];
  Grp g = make_grp(P, ntt_smem);
  uint32_t x[8];
  ld8(x, in + ((size_t)blockIdx.x * 2 + g.n) * POLY + g.tid * 8);
  grp_ntt_inv(g, x);
  uint64_t* dst = out + (size_t)blockIdx.x * POLY;
  crt_lift(x, res, g, P, [&](int z, uint64_t v) { dst[z] = v; });
}
__global__ void k_widen(uint64_t* out, const uint32_t* in, size_t words) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < words) out[i] = in[i];
}
__global__ void k_narrow(uint32_t* out, const uint64_t* in, size_t words) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < words) out[i] = (uint32_t)in[i];
}

// ------------------------------------------------------------------ fold (one round)
// server.rs:405-425.  CTA = one (batch entry, i) step.
__global__ void __launch_bounds__(CTA, 1)
k_fold_round(DevParams P, uint64_t* cts, size_t batch_stride, int half, const uint32_t* c_pos, const uint32_t* c_neg,
             size_t c_batch_stride, int slices_per_query, int t_gsw, int bits) {
  __shared__ __align__(16) uint32_t ntt_smem[2 * NTT_SMEM_WORDS];
  __shared__ uint32_t res[2 * POLY];
  Grp g = make_grp(P, ntt_smem);
  const int b = blockIdx.x / half, i = blockIdx.x % half;
  uint64_t* base = cts + (size_t)b * batch_stride;
  const size_t qoff = (size_t)(b / slices_per_query) * c_batch_stride;
  const int cols = 2 * t_gsw;
  const size_t col_step = (size_t)2 * 2 * POLY;          // column index advances by rdim = 2 per digit
  const size_t row_step = (size_t)cols * 2 * POLY;

  uint64_t acc[2][8];
#pragma unroll
  for (int r = 0; r < 2; r++)
#pragma unroll
    for (int e = 0; e < 8; e++) acc[r][e] = 0;
  int cnt = 0;
#pragma unroll 1
  for (int src = 0; src < 2; src++) {
    const uint64_t* ct = base + (size_t)(src == 0 ? i : half + i) * 2 * POLY;
    const uint32_t* C = (src == 0 ? c_neg : c_pos) + qoff;
#pragma unroll 1
    for (int rho = 0; rho < 2; rho++) {
      uint64_t v[8];
#pragma unroll
      for (int a = 0; a < 8; a++) v[a] = ct[rho * POLY + a * 256 + g.tid];
      // G^-1 row index = rho + 2k  -> key-matrix column rho + 2k
      const uint32_t* c0 = C + ((size_t)rho * 2 + g.n) * POLY + g.tid * 8;
      digits_mac<2, false>(acc, cnt, v, t_gsw, bits, c0, col_step, row_step, g);
    }
  }
  uint64_t* dst = base + (size_t)i * 2 * POLY;
#pragma unroll 1
  for (int r = 0; r < 2; r++) {
    uint32_t x[8];
#pragma unroll
    for (int e = 0; e < 8; e++) x[e] = barrett64(acc[r][e], g.cr1, g.q);
    grp_ntt_inv(g, x);
    uint64_t* d = dst + r * POLY;
    crt_lift(x, res, g, P, [&](int z, uint64_t val) { d[z] = val; });
  }
}

// ------------------------------------------------------------------ fold, fast path (residue form)
// Ciphertexts are kept in "residue form": u32 [ct][row][n][z] = coefficient z of the row modulo q_n
// (what the inverse NTT of each CRT half produces, before the CRT lift).  One step computes
//     out[i] = ct[i] + INTT( C_k . NTT( G^-1(ct[half+i]) - G^-1(ct[i]) ) )            (mod q_n, per modulus)
// which is the same canonical value as server.rs:405-425's
//     from_ntt( (G - C_k) . NTT(G^-1(ct[i])) + C_k . NTT(G^-1(ct[half+i])) )
// because v_folding_neg[k] = G - C_k (server.rs:505-523), G . G^-1(x) = x and the NTT is linear over
// Z_{q_n}; canonical representatives are unique, so the bytes agree.  It needs half the forward
// transforms, no CRT lift on the way out, and no v_folding_neg at all.
// grid = (batch*half, 2 moduli), 256 threads.  in/out are distinct buffers (ping-pong): the CTA of
// modulus n reads BOTH residues of its inputs (for the gadget digits) while the other CTA writes.
// Digit k of vh minus digit k of vi, offset by q: in (q - 2^bits, q + 2^bits), a subset of [0, 2q) for bits <= 27 (the
// context rejects gadget dimensions below 3, so bits <= 19) — the relaxed-range forward transform needs no more.
// BYTE: bits == 8, where digit k is simply byte k; the values are < 2^56, so byte 7 serves as the zero filler.
template <bool BYTE>
__device__ __forceinline__ uint32_t digit_diff(uint64_t vh, uint64_t vi, int k, int bits, uint64_t mask, uint32_t q) {
  if (BYTE) {
    const uint32_t sel = 0x7770u | (uint32_t)k;
    return __byte_perm((uint32_t)vh, (uint32_t)(vh >> 32), sel) - __byte_perm((uint32_t)vi, (uint32_t)(vi >> 32), sel) + q;
  }
  return gadget_digit(vh, k, bits, mask) - gadget_digit(vi, k, bits, mask) + q;
}

// Same step as k_fold_res on the relaxed-range transforms (ntt_core.cuh "lz"): no per-butterfly range correction in the
// forward transforms (outputs < 16q feed the 64-bit multiply-accumulate directly: 16 products of < 2^32 x < 2^28 fit),
// no halving in the inverse transform, byte-permute digit extraction when bits_per = 8, 32-bit Barrett in the CRT lift.
// Digits that are zero for every value < q0 q1 (digit 7 of the t = 8, 8-bit gadget) are skipped: fold stage 3.53 -> 3.26 ms
// (S8, 16 queries, B200).  Tried before that and measured without gain (fold stage 3.53 ms): pass C / D twiddles held in registers at
// 2 CTAs per SM (3.60 ms: 35 % less shared-memory traffic, so that is not the limit), key columns prefetched into L1 before the
// pair's transforms (3.60 ms: the L2 latency ncu attributes to the multiply-accumulate is covered by the other CTAs).  The
// kernel runs at ~80 % of its integer-multiply-pipe bound (DESIGN.md 4.3).
template <int MINB, bool BYTE>
__global__ void __launch_bounds__(256, MINB)
k_fold_res_lz(DevParams P, const uint32_t* __restrict__ in, uint32_t* __restrict__ out, size_t batch_stride, int half,
              const uint32_t* __restrict__ c_pos, size_t c_batch_stride, int slices_per_query, int t_gsw, int bits,
              const uint32_t* __restrict__ zero_flags /* null, or [batch][2*half]: 1 = ciphertext is all zero */) {
  if (zero_flags) {            // lib/server/src/compute/fold.rs:37-43, see k_fold_res
    const int bz = blockIdx.x / half, iz = blockIdx.x % half;
    const uint32_t fa = zero_flags[(size_t)bz * 2 * half + iz], fb = zero_flags[(size_t)bz * 2 * half + half + iz];
    if (fa | fb) {
      const uint32_t* src = in + (size_t)bz * batch_stride + (size_t)((fa ? half : 0) + iz) * 4 * POLY;
      uint32_t* dst = out + (size_t)bz * batch_stride + (size_t)iz * 4 * POLY;
#pragma unroll
      for (int rho = 0; rho < 2; rho++) {
        uint32_t x[8];
        ld8_ro(x, src + ((size_t)rho * 2 + blockIdx.y) * POLY + threadIdx.x * 8);
        st8(dst + ((size_t)rho * 2 + blockIdx.y) * POLY + threadIdx.x * 8, x);
      }
      return;
    }
  }
  extern __shared__ __align__(16) uint8_t dyn_smem[];
  uint32_t* sm0 = reinterpret_cast<uint32_t*>(dyn_smem);
  uint32_t* sm1 = sm0 + NTT_SMEM_WORDS;
  Twiddle* tw = reinterpret_cast<Twiddle*>(sm1 + NTT_SMEM_WORDS);
  Grp g = make_grp_single(P, sm0, blockIdx.y);
  stage_fwd_twiddles(g, tw);
  const TwConst lo{g.n, 0};
  const TwShared hi{tw};
  const int b = blockIdx.x / half, i = blockIdx.x % half;
  const uint32_t* ci = in + (size_t)b * batch_stride + (size_t)i * 4 * POLY;
  const uint32_t* ch = in + (size_t)b * batch_stride + (size_t)(half + i) * 4 * POLY;
  const uint32_t* C = c_pos + (size_t)(b / slices_per_query) * c_batch_stride;
  const int cols = 2 * t_gsw;
  const size_t row_step = (size_t)cols * 2 * POLY;
  const uint64_t mask = (1ull << bits) - 1;
  const uint32_t q = g.q;
  // the CRT-lifted coefficients are < q0 q1: digits from ndig on are zero in both ciphertexts, so their differences (q) transform
  // to multiples of q and add nothing mod q to the accumulators
  const int ndig = gadget_live_digits(t_gsw, bits, P.modulus);

  uint64_t acc[2][8];
#pragma unroll
  for (int r = 0; r < 2; r++)
#pragma unroll
    for (int e = 0; e < 8; e++) acc[r][e] = 0;
  int cnt = 0;                                   // products (< 2^60 each) held by every accumulator: at most 16
#pragma unroll 1
  for (int rho = 0; rho < 2; rho++) {
    uint64_t vi[8], vh[8];
#pragma unroll
    for (int a = 0; a < 8; a++) {
      const int z = a * 256 + g.tid;
      vi[a] = crt_compose(__ldg(ci + (rho * 2 + 0) * POLY + z), __ldg(ci + (rho * 2 + 1) * POLY + z), P);
      vh[a] = crt_compose(__ldg(ch + (rho * 2 + 0) * POLY + z), __ldg(ch + (rho * 2 + 1) * POLY + z), P);
    }
    const uint32_t* c0 = C + ((size_t)rho * 2 + g.n) * POLY + g.tid * 8;       // key-matrix column of digit k: rho + 2k
    int k = 0;
#pragma unroll 1
    for (; k + 1 < ndig; k += 2) {
      uint32_t x0[8], x1[8];
#pragma unroll
      for (int a = 0; a < 8; a++) {
        x0[a] = digit_diff<BYTE>(vh[a], vi[a], k, bits, mask, q);
        x1[a] = digit_diff<BYTE>(vh[a], vi[a], k + 1, bits, mask, q);
      }
      ntt_forward_group2_lz<NTT_OUT_LAZY16>(g.tid, x0, x1, sm0, sm1, lo, hi, q, CtaSync());
      if (cnt + 2 > 16) { acc_reduce<2>(acc, g); cnt = 1; }
      cnt += 2;
#pragma unroll
      for (int r = 0; r < 2; r++) {
        uint32_t cv[8];
        ld8_ro(cv, c0 + (size_t)r * row_step + (size_t)k * 4 * POLY);
#pragma unroll
        for (int e = 0; e < 8; e++) acc[r][e] += (uint64_t)x0[e] * cv[e];
        ld8_ro(cv, c0 + (size_t)r * row_step + (size_t)(k + 1) * 4 * POLY);
#pragma unroll
        for (int e = 0; e < 8; e++) acc[r][e] += (uint64_t)x1[e] * cv[e];
      }
    }
    if (k < ndig) {                             // odd digit count: last digit alone
      uint32_t x0[8];
#pragma unroll
      for (int a = 0; a < 8; a++) x0[a] = digit_diff<BYTE>(vh[a], vi[a], k, bits, mask, q);
      ntt_forward_group_lz<NTT_OUT_LAZY16>(g.tid, x0, sm0, lo, hi, q, CtaSync());
      if (cnt + 1 > 16) { acc_reduce<2>(acc, g); cnt = 1; }
      cnt += 1;
#pragma unroll
      for (int r = 0; r < 2; r++) {
        uint32_t cv[8];
        ld8_ro(cv, c0 + (size_t)r * row_step + (size_t)k * 4 * POLY);
#pragma unroll
        for (int e = 0; e < 8; e++) acc[r][e] += (uint64_t)x0[e] * cv[e];
      }
    }
  }
  uint32_t y0[8], y1[8];
#pragma unroll
  for (int e = 0; e < 8; e++) {
    y0[e] = barrett64(acc[0][e], g.cr1, q);
    y1[e] = barrett64(acc[1][e], g.cr1, q);
  }
  ntt_inverse_group2_nh(g.tid, y0, y1, sm0, sm1, TwConst{g.n, 2}, TwGlobal{g.inv_lz}, q, CtaSync());
  uint32_t* co = out + (size_t)b * batch_stride + (size_t)i * 4 * POLY;
#pragma unroll
  for (int a = 0; a < 8; a++) {
    const int z = a * 256 + g.tid;
    co[(0 * 2 + g.n) * POLY + z] = addmod(y0[a], __ldg(ci + (0 * 2 + g.n) * POLY + z), q);
    co[(1 * 2 + g.n) * POLY + z] = addmod(y1[a], __ldg(ci + (1 * 2 + g.n) * POLY + z), q);
  }
}

// flags[b][idx] = 1 iff ciphertext idx of batch b (residue form, 4 x 2048 words) is all zero  (fold.rs:6-13 is_all_zeros:
// the CRT-lifted polynomial is zero exactly when every residue is)
__global__ void __launch_bounds__(256)
k_ct_zero_flags(const uint32_t* __restrict__ cts, size_t batch_stride, int per_batch, uint32_t* __restrict__ flags) {
  const int b = blockIdx.x / per_batch, idx = blockIdx.x % per_batch;
  const uint4* p = reinterpret_cast<const uint4*>(cts + (size_t)b * batch_stride + (size_t)idx * 4 * POLY);
  uint32_t acc = 0;
#pragma unroll
  for (int k = 0; k < 8; k++) {
    const uint4 v = __ldg(p + k * 256 + threadIdx.x);
    acc |= v.x | v.y | v.z | v.w;
  }
  const int any = __syncthreads_or(acc != 0);
  if (threadIdx.x == 0) flags[blockIdx.x] = any ? 0u : 1u;
}

// neg[k][r][c] = (q_n - C[k][r][c]) + G[r][c]   with G[i][i + 2j] = 2^{bits*j}  (gadget.rs:11-32)
__global__ void k_folding_neg(DevParams P, uint32_t* out, const uint32_t* vf, size_t total, int t_gsw, int bits) {
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  int n = (int)((idx / POLY) & 1);
  size_t poly = idx / (2 * POLY);            // ((k*2 + r)*cols + c)
  int cols = 2 * t_gsw;
  int c = (int)(poly % cols);
  int r = (int)((poly / cols) & 1);
  uint32_t q = P.q[n];
  uint32_t v = vf[idx];
  uint32_t neg = v == 0 ? 0u : q - v;
  uint32_t gval = 0;
  if ((c & 1) == r) {
    int j = c >> 1;
    if (bits * j < 64) gval = barrett64(1ull << (bits * j), P.cr1[n], q);
  }
  out[idx] = addmod(neg, gval, q);
}

// ------------------------------------------------------------------ query expansion
// server.rs:105-110: v[num_in + i] = v[i] (.) neg1
__global__ void k_expand_scalar(DevParams P, uint32_t* v, size_t v_stride, int num_in, const uint32_t* neg1) {
  v += (size_t)blockIdx.y * v_stride;
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;     // over num_in * 2 rows * 2 mod * 2048
  size_t total = (size_t)num_in * 4 * POLY;
  if (idx >= total) return;
  int z = (int)(idx % POLY);
  int n = (int)((idx / POLY) & 1);
  uint32_t a = v[idx], b = neg1[n * POLY + z];
  v[total + idx] = barrett64((uint64_t)a * b, P.cr1[n], P.q[n]);
}

// server.rs:39-103 action_expand for ciphertext index blockIdx.x of round R.r (in place on v).
__global__ void __launch_bounds__(CTA, 1) k_expand_round(DevParams P, uint32_t* v, size_t v_stride, ExpandRound R) {
  v += (size_t)blockIdx.y * v_stride;
  extern __shared__ __align__(16) uint8_t dyn_smem[];
  uint32_t* ntt_smem = reinterpret_cast<uint32_t*>(dyn_smem);
  uint32_t* res = ntt_smem + 4 * NTT_SMEM_WORDS;
  uint64_t* autom = reinterpret_cast<uint64_t*>(res + 2 * POLY);      // [2][2048]
  Twiddle* tw = reinterpret_cast<Twiddle*>(autom + 2 * POLY);         // [2][HI_TW]
  Grp g = make_grp(P, ntt_smem);
  g.smem2 = ntt_smem + (2 + g.n) * NTT_SMEM_WORDS;

  const int i = blockIdx.x;
  const int ih = i < R.num_in ? i : i - R.num_in;       // index within its half (server.rs:112-119)
  if ((R.stop_round > 0 && R.r > R.stop_round && (ih & 1)) ||
      (R.stop_round > 0 && R.r == R.stop_round && (ih & 1) && (ih / 2) >= R.max_bits_to_gen_right))
    return;
  const bool left = (R.r != 0) && ((ih & 1) == 0);
  const uint32_t* W = left ? R.tab_left[blockIdx.y] + R.off_left : R.tab_right[blockIdx.y] + R.off_right;
  const int t_exp = left ? R.t_left : R.t_right;
  const int bits = left ? R.bits_left : R.bits_right;

  stage_fwd_twiddles(g, tw + g.n * HI_TW);
  uint32_t* vi = v + (size_t)i * 4 * POLY;
  uint32_t keep[2][8];
  // row 0: from_ntt + automorph (poly.rs:393-405), scattered into shared memory for the gadget digits
  {
    uint32_t x[8];
    ld8(x, vi + (size_t)g.n * POLY + g.tid * 8);
#pragma unroll
    for (int e = 0; e < 8; e++) keep[0][e] = x[e];
    grp_ntt_inv(g, x);
    const int t_auto = R.t_auto;
    const uint64_t Q = P.modulus;
    crt_lift(x, res, g, P, [&](int z, uint64_t val) {
      unsigned prod = (unsigned)z * (unsigned)t_auto;
      unsigned num = prod >> NTT_LOG_N, rem = prod & (POLY - 1);
      autom[rem] = (num & 1u) ? Q - val : val;           // zero maps to q, as in the reference
    });
  }
  // row 1: the reference computes to_ntt(automorph(from_ntt(row 1))) (server.rs:80-88).  X -> X^t permutes the
  // roots of X^N + 1, so in the NTT domain the automorphism is a pure permutation of the evaluation slots:
  // slot s holds the value at psi^(2 br(s) + 1), and tau_t(a) there equals a at psi^((2 br(s) + 1) t).  The
  // values are canonical residues either way, so the gathered vector is bit-identical to the reference's.
  uint32_t y[8];
  {
    const uint32_t* row1 = vi + ((size_t)2 + g.n) * POLY;
    ld8(keep[1], row1 + g.tid * 8);
#pragma unroll
    for (int k = 0; k < 8; k++) {
      const unsigned sidx = (unsigned)(g.tid * 8 + k);
      const unsigned e = 2u * (__brev(sidx) >> (32 - NTT_LOG_N)) + 1u;
      const unsigned e2 = (e * (unsigned)R.t_auto) & (2u * POLY - 1u);
      const unsigned src = __brev((e2 - 1u) >> 1) >> (32 - NTT_LOG_N);
      y[k] = row1[src];
    }
  }
  __syncthreads();
  uint64_t acc[2][8];
#pragma unroll
  for (int r = 0; r < 2; r++)
#pragma unroll
    for (int e = 0; e < 8; e++) acc[r][e] = 0;
  int cnt = 0;
  {
    uint64_t vv[8];
#pragma unroll
    for (int a = 0; a < 8; a++) vv[a] = autom[a * 256 + g.tid];
    // gadget_invert_rdim(.., rdim = 1): digit k -> key column k  (server.rs:82-89)
    const uint32_t* c0 = W + (size_t)g.n * POLY + g.tid * 8;
    digits_mac<2, true>(acc, cnt, vv, gadget_live_digits(t_exp, bits, P.modulus), bits, c0, (size_t)2 * POLY, (size_t)t_exp * 2 * POLY, g);
  }
#pragma unroll
  for (int rho = 0; rho < 2; rho++) {
    uint32_t o[8];
#pragma unroll
    for (int e = 0; e < 8; e++) {
      uint32_t s = addmod(keep[rho][e], barrett64(acc[rho][e], g.cr1, g.q), g.q);
      o[e] = rho ? addmod(s, y[e], g.q) : s;
    }
    st8(vi + ((size_t)rho * 2 + g.n) * POLY + g.tid * 8, o);
  }
}

// Paired variant for the wide rounds: CTA i produces BOTH outputs that derive from v[i], i.e. index i and index
// i + num_in (= action_expand on v[i] (.) neg1[r], server.rs:105-110).  neg1[r] is the NTT of -X^(N - 2^r) = X^(-2^r), so
//   * from_ntt(v[i] (.) neg1) is the negacyclic shift of from_ntt(v[i]) by 2^r places: coefficient k is residue k + 2^r
//     of the first output, negated mod q_n (0 stays 0, the canonical residue the reference's inverse NTT returns) when
//     k + 2^r wraps past N.  One inverse transform serves both outputs and the separate scalar-multiply pass
//     (k_expand_scalar: 64 KiB of HBM traffic per ciphertext) disappears;
//   * the NTT-domain rows of the second output are pointwise products with neg1, formed in registers.
// Only CTA i touches v[i] and v[i + num_in], so the round stays in place.  Used when the round has enough active
// ciphertexts to fill the GPU; narrow rounds keep one CTA per output (half the latency).
__global__ void __launch_bounds__(CTA, 1)
k_expand_round_pair(DevParams P, uint32_t* v, size_t v_stride, ExpandRound R, const uint32_t* __restrict__ neg1) {
  v += (size_t)blockIdx.y * v_stride;
  extern __shared__ __align__(16) uint8_t dyn_smem[];
  uint32_t* ntt_smem = reinterpret_cast<uint32_t*>(dyn_smem);
  uint32_t* res = ntt_smem + 4 * NTT_SMEM_WORDS;
  uint64_t* autom = reinterpret_cast<uint64_t*>(res + 2 * POLY);
  Twiddle* tw = reinterpret_cast<Twiddle*>(autom + 2 * POLY);
  Grp g = make_grp(P, ntt_smem);
  g.smem2 = ntt_smem + (2 + g.n) * NTT_SMEM_WORDS;

  const int i = blockIdx.x;                               // index within the half == i for both outputs
  if ((R.stop_round > 0 && R.r > R.stop_round && (i & 1)) ||
      (R.stop_round > 0 && R.r == R.stop_round && (i & 1) && (i / 2) >= R.max_bits_to_gen_right)) {
    // never read again by the query path; the reference still leaves v[i + num_in] = v[i] (.) neg1 there
    // (server.rs:105-110 runs before the skip test), which the stage-level entry point reproduces
    if (R.fill_skipped) {
      const int n = threadIdx.x >> 8, tid = threadIdx.x & 255;
      const uint32_t qn = n ? P.q[1] : P.q[0];
      const uint64_t cr1 = n ? P.cr1[1] : P.cr1[0];
      uint32_t nn[8];
      ld8_ro(nn, neg1 + (size_t)n * POLY + tid * 8);
#pragma unroll
      for (int rho = 0; rho < 2; rho++) {
        uint32_t x[8];
        ld8(x, v + ((size_t)i * 4 + rho * 2 + n) * POLY + tid * 8);
#pragma unroll
        for (int e = 0; e < 8; e++) x[e] = barrett64((uint64_t)x[e] * nn[e], cr1, qn);
        st8(v + ((size_t)(i + R.num_in) * 4 + rho * 2 + n) * POLY + tid * 8, x);
      }
    }
    return;
  }
  const bool left = (R.r != 0) && ((i & 1) == 0);
  const uint32_t* W = left ? R.tab_left[blockIdx.y] + R.off_left : R.tab_right[blockIdx.y] + R.off_right;
  const int t_exp = left ? R.t_left : R.t_right;
  const int bits = left ? R.bits_left : R.bits_right;

  stage_fwd_twiddles(g, tw + g.n * HI_TW);
  uint32_t* vi = v + (size_t)i * 4 * POLY;
  uint32_t* vo = v + (size_t)(i + R.num_in) * 4 * POLY;
  const uint32_t* ng = neg1 + (size_t)g.n * POLY;
  uint32_t keep[2][8], y[8];
  {
    uint32_t x[8];
    ld8(x, vi + (size_t)g.n * POLY + g.tid * 8);
#pragma unroll
    for (int e = 0; e < 8; e++) keep[0][e] = x[e];
    grp_ntt_inv(g, x);
    __syncthreads();
#pragma unroll
    for (int a = 0; a < 8; a++) res[g.n * POLY + a * 256 + g.tid] = x[a];      // canonical residues, coefficient order
  }
  const uint32_t* row1 = vi + ((size_t)2 + g.n) * POLY;
  ld8(keep[1], row1 + g.tid * 8);
#pragma unroll
  for (int k = 0; k < 8; k++) {
    const unsigned sidx = (unsigned)(g.tid * 8 + k);
    const unsigned e = 2u * (__brev(sidx) >> (32 - NTT_LOG_N)) + 1u;
    const unsigned e2 = (e * (unsigned)R.t_auto) & (2u * POLY - 1u);
    const unsigned src = __brev((e2 - 1u) >> 1) >> (32 - NTT_LOG_N);
    y[k] = row1[src];
  }
  __syncthreads();
  const uint64_t Q = P.modulus;
  const uint32_t q0 = P.q[0], q1 = P.q[1];
#pragma unroll 1
  for (int half = 1; half >= 0; half--) {
    const int shift = half ? R.num_in : 0;                // 2^r
#pragma unroll
    for (int a4 = 0; a4 < 4; a4++) {
      const int k = (g.n * 4 + a4) * 256 + g.tid;
      const int zs = (k + shift) & (POLY - 1);
      uint32_t a0 = res[zs], a1 = res[POLY + zs];
      if (k + shift >= POLY) {
        a0 = a0 ? q0 - a0 : 0u;
        a1 = a1 ? q1 - a1 : 0u;
      }
      const uint64_t val = crt_compose(a0, a1, P);
      const unsigned prod = (unsigned)k * (unsigned)R.t_auto;
      const unsigned num = prod >> NTT_LOG_N, rem = prod & (POLY - 1);
      autom[rem] = (num & 1u) ? Q - val : val;            // zero maps to q, as in the reference
    }
    __syncthreads();
    uint64_t acc[2][8];
#pragma unroll
    for (int r = 0; r < 2; r++)
#pragma unroll
      for (int e = 0; e < 8; e++) acc[r][e] = 0;
    int cnt = 0;
    {
      uint64_t vv[8];
#pragma unroll
      for (int a = 0; a < 8; a++) vv[a] = autom[a * 256 + g.tid];
      const uint32_t* c0 = W + (size_t)g.n * POLY + g.tid * 8;
      digits_mac<2, true>(acc, cnt, vv, gadget_live_digits(t_exp, bits, P.modulus), bits, c0, (size_t)2 * POLY, (size_t)t_exp * 2 * POLY, g);
    }
    uint32_t* dst = half ? vo : vi;
#pragma unroll
    for (int rho = 0; rho < 2; rho++) {
      uint32_t o[8], nn[8];
      if (half) ld8_ro(nn, ng + g.tid * 8);
#pragma unroll
      for (int e = 0; e < 8; e++) {
        uint32_t base = keep[rho][e];
        if (half) base = barrett64((uint64_t)base * nn[e], g.cr1, g.q);
        uint32_t s = addmod(base, barrett64(acc[rho][e], g.cr1, g.q), g.q);
        if (rho) {
          uint32_t yy = y[e];
          if (half) {
            const unsigned sidx = (unsigned)(g.tid * 8 + e);
            const unsigned ee = 2u * (__brev(sidx) >> (32 - NTT_LOG_N)) + 1u;
            const unsigned e2 = (ee * (unsigned)R.t_auto) & (2u * POLY - 1u);
            const unsigned src = __brev((e2 - 1u) >> 1) >> (32 - NTT_LOG_N);
            yy = barrett64((uint64_t)yy * __ldg(ng + src), g.cr1, g.q);
          }
          s = addmod(s, yy, g.q);
        }
        o[e] = s;
      }
      st8(dst + ((size_t)rho * 2 + g.n) * POLY + g.tid * 8, o);
    }
    __syncthreads();
  }
}

// ---- paired rounds, residue pipeline: the same arithmetic as k_expand_round_pair split the way k_fold_res is, so that
// the transforms run in 256-thread single-modulus CTAs at 3 CTAs per SM instead of one 512-thread CTA per SM.
//   k_expand_intt:       inverse transform of row 0 of every processed v[i], residues in coefficient order -> xr
//   k_expand_round_res:  CTA (i, n): CRT lift (+ negacyclic shift for the second output) + automorphism + gadget digits
//                        + forward transforms and key products modulo q_n; writes rows (., n) of v[i] and v[i + num_in].
// xr: [query][i][n][2048] u32.
__global__ void __launch_bounds__(256)
k_expand_intt(DevParams P, const uint32_t* __restrict__ v, size_t v_stride, uint32_t* __restrict__ xr, size_t xr_stride,
              ExpandRound R) {
  __shared__ __align__(16) uint32_t ntt_smem[NTT_SMEM_WORDS];
  const int i = blockIdx.x;
  if ((R.stop_round > 0 && R.r > R.stop_round && (i & 1)) ||
      (R.stop_round > 0 && R.r == R.stop_round && (i & 1) && (i / 2) >= R.max_bits_to_gen_right))
    return;
  Grp g = make_grp_single(P, ntt_smem, blockIdx.y);
  const uint32_t* src = v + (size_t)blockIdx.z * v_stride + ((size_t)i * 4 + g.n) * POLY;
  uint32_t x[8];
  ld8_ro(x, src + g.tid * 8);
  grp_ntt_inv(g, x);
  uint32_t* dst = xr + (size_t)blockIdx.z * xr_stride + ((size_t)i * 2 + g.n) * POLY;
#pragma unroll
  for (int a = 0; a < 8; a++) dst[a * 256 + g.tid] = x[a];
}

template <int MINB>
__global__ void __launch_bounds__(256, MINB)
k_expand_round_res(DevParams P, uint32_t* v, size_t v_stride, const uint32_t* __restrict__ xr, size_t xr_stride,
                   ExpandRound R, const uint32_t* __restrict__ neg1) {
  v += (size_t)blockIdx.z * v_stride;
  xr += (size_t)blockIdx.z * xr_stride;
  extern __shared__ __align__(16) uint8_t dyn_smem[];
  uint32_t* sm0 = reinterpret_cast<uint32_t*>(dyn_smem);
  uint32_t* sm1 = sm0 + NTT_SMEM_WORDS;
  uint64_t* autom = reinterpret_cast<uint64_t*>(sm1 + NTT_SMEM_WORDS);     // [2048]
  Twiddle* tw = reinterpret_cast<Twiddle*>(autom + POLY);                   // [HI_TW]
  Grp g = make_grp_single(P, sm0, blockIdx.y);
  g.smem2 = sm1;
  const int i = blockIdx.x;
  const uint32_t* ng = neg1 + (size_t)g.n * POLY;
  uint32_t* vi = v + (size_t)i * 4 * POLY;
  uint32_t* vo = v + (size_t)(i + R.num_in) * 4 * POLY;
  if ((R.stop_round > 0 && R.r > R.stop_round && (i & 1)) ||
      (R.stop_round > 0 && R.r == R.stop_round && (i & 1) && (i / 2) >= R.max_bits_to_gen_right)) {
    if (R.fill_skipped) {                                  // see k_expand_round_pair
      uint32_t nn[8];
      ld8_ro(nn, ng + g.tid * 8);
#pragma unroll
      for (int rho = 0; rho < 2; rho++) {
        uint32_t x[8];
        ld8(x, vi + ((size_t)rho * 2 + g.n) * POLY + g.tid * 8);
#pragma unroll
        for (int e = 0; e < 8; e++) x[e] = barrett64((uint64_t)x[e] * nn[e], g.cr1, g.q);
        st8(vo + ((size_t)rho * 2 + g.n) * POLY + g.tid * 8, x);
      }
    }
    return;
  }
  const bool left = (R.r != 0) && ((i & 1) == 0);
  const uint32_t* W = left ? R.tab_left[blockIdx.z] + R.off_left : R.tab_right[blockIdx.z] + R.off_right;
  const int t_exp = left ? R.t_left : R.t_right;
  const int bits = left ? R.bits_left : R.bits_right;
  stage_fwd_twiddles(g, tw);
  const uint32_t* x0r = xr + (size_t)i * 2 * POLY;         // residues mod q_0 / q_1 of from_ntt(row 0 of v[i])
  const uint32_t* x1r = x0r + POLY;
  const uint32_t* row1 = vi + ((size_t)2 + g.n) * POLY;
  const uint64_t Q = P.modulus;
  const uint32_t q0 = P.q[0], q1 = P.q[1];
#pragma unroll 1
  for (int half = 1; half >= 0; half--) {
    const int shift = half ? R.num_in : 0;                 // 2^r
#pragma unroll
    for (int a = 0; a < 8; a++) {
      const int k = a * 256 + g.tid;
      const int zs = (k + shift) & (POLY - 1);
      uint32_t a0 = __ldg(x0r + zs), a1 = __ldg(x1r + zs);
      if (k + shift >= POLY) {
        a0 = a0 ? q0 - a0 : 0u;
        a1 = a1 ? q1 - a1 : 0u;
      }
      const uint64_t val = crt_compose(a0, a1, P);
      const unsigned prod = (unsigned)k * (unsigned)R.t_auto;
      const unsigned num = prod >> NTT_LOG_N, rem = prod & (POLY - 1);
      autom[rem] = (num & 1u) ? Q - val : val;             // zero maps to q, as in the reference
    }
    __syncthreads();                                       // autom complete (and the staged twiddles visible)
    uint64_t acc[2][8];
#pragma unroll
    for (int r = 0; r < 2; r++)
#pragma unroll
      for (int e = 0; e < 8; e++) acc[r][e] = 0;
    int cnt = 0;
    {
      uint64_t vv[8];
#pragma unroll
      for (int a = 0; a < 8; a++) vv[a] = autom[a * 256 + g.tid];
      const uint32_t* c0 = W + (size_t)g.n * POLY + g.tid * 8;
      digits_mac<2, true>(acc, cnt, vv, gadget_live_digits(t_exp, bits, P.modulus), bits, c0, (size_t)2 * POLY, (size_t)t_exp * 2 * POLY, g);
    }
    // row 1 automorphism = slot permutation (see k_expand_round); gather before any thread overwrites v[i]
    uint32_t yy[8];
#pragma unroll
    for (int e = 0; e < 8; e++) {
      const unsigned sidx = (unsigned)(g.tid * 8 + e);
      const unsigned ee = 2u * (__brev(sidx) >> (32 - NTT_LOG_N)) + 1u;
      const unsigned e2 = (ee * (unsigned)R.t_auto) & (2u * POLY - 1u);
      const unsigned src = __brev((e2 - 1u) >> 1) >> (32 - NTT_LOG_N);
      uint32_t t = row1[src];
      if (half) t = barrett64((uint64_t)t * __ldg(ng + src), g.cr1, g.q);
      yy[e] = t;
    }
    __syncthreads();
    uint32_t* dst = half ? vo : vi;
    uint32_t nn[8];
    if (half) ld8_ro(nn, ng + g.tid * 8);
#pragma unroll
    for (int rho = 0; rho < 2; rho++) {
      uint32_t o[8];
      ld8(o, vi + ((size_t)rho * 2 + g.n) * POLY + g.tid * 8);
#pragma unroll
      for (int e = 0; e < 8; e++) {
        uint32_t base = o[e];
        if (half) base = barrett64((uint64_t)base * nn[e], g.cr1, g.q);
        uint32_t s = addmod(base, barrett64(acc[rho][e], g.cr1, g.q), g.q);
        o[e] = rho ? addmod(s, yy[e], g.q) : s;
      }
      st8(dst + ((size_t)rho * 2 + g.n) * POLY + g.tid * 8, o);
    }
  }
}

// util.rs:323-355
__global__ void k_reorient(MulGeom G, uint4* q_dev, size_t q_stride, const uint32_t* v, size_t v_stride, int idx_factor) {
  q_dev += (size_t)blockIdx.y * q_stride;
  v += (size_t)blockIdx.y * v_stride;
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;     // over dim0 * 2048
  if (idx >= (size_t)G.dim0 * POLY) return;
  int z = (int)(idx % POLY), j = (int)(idx / POLY);
  const uint32_t* ct = v + (size_t)idx_factor * j * 4 * POLY;
  uint4 o = make_uint4(ct[z], ct[POLY + z], ct[2 * POLY + z], ct[3 * POLY + z]);
  q_dev[((size_t)(j >> 1) * 2 + (j & 1)) * POLY + z] = o;
}

// server.rs:134-150.  CTA = (gsw index i, digit j).
__global__ void __launch_bounds__(CTA, 1)
k_regev_to_gsw(DevParams P, uint32_t* v_gsw, size_t gsw_stride, const uint32_t* v, size_t v_stride, int idx_factor,
               int idx_offset, const uint32_t* const* tab_conv, int t_gsw, int t_conv, int bits_conv) {
  const uint32_t* v_conv = tab_conv[blockIdx.y];
  v_gsw += (size_t)blockIdx.y * gsw_stride;
  v += (size_t)blockIdx.y * v_stride;
  extern __shared__ __align__(16) uint8_t dyn_smem[];
  uint32_t* ntt_smem = reinterpret_cast<uint32_t*>(dyn_smem);
  uint32_t* res = ntt_smem + 4 * NTT_SMEM_WORDS;
  uint64_t* raw = reinterpret_cast<uint64_t*>(res + 2 * POLY);        // [2][2048]
  Twiddle* tw = reinterpret_cast<Twiddle*>(raw + 2 * POLY);           // [2][HI_TW]
  Grp g = make_grp(P, ntt_smem);
  g.smem2 = ntt_smem + (2 + g.n) * NTT_SMEM_WORDS;
  stage_fwd_twiddles(g, tw + g.n * HI_TW);
  const int i = blockIdx.x / t_gsw, j = blockIdx.x % t_gsw;
  const int idx_inp = idx_factor * (i * t_gsw + j) + idx_offset;
  const uint32_t* inp = v + (size_t)idx_inp * 4 * POLY;
  const int cols = 2 * t_gsw;
  uint32_t* out = v_gsw + (size_t)i * 2 * cols * 2 * POLY;
#pragma unroll 1
  for (int rho = 0; rho < 2; rho++) {
    uint32_t x[8];
    ld8(x, inp + ((size_t)rho * 2 + g.n) * POLY + g.tid * 8);
    st8(out + (((size_t)rho * cols + 2 * j + 1) * 2 + g.n) * POLY + g.tid * 8, x);      // ct.copy_into(.., 0, 2j+1)
    grp_ntt_inv(g, x);
    uint64_t* d = raw + rho * POLY;
    crt_lift(x, res, g, P, [&](int z, uint64_t val) { d[z] = val; });
  }
  __syncthreads();
  uint64_t acc[2][8];
#pragma unroll
  for (int r = 0; r < 2; r++)
#pragma unroll
    for (int e = 0; e < 8; e++) acc[r][e] = 0;
  int cnt = 0;
  const int ccols = 2 * t_conv;
#pragma unroll 1
  for (int rho = 0; rho < 2; rho++) {
    uint64_t vv[8];
#pragma unroll
    for (int a = 0; a < 8; a++) vv[a] = raw[rho * POLY + a * 256 + g.tid];
    const uint32_t* c0 = v_conv + ((size_t)rho * 2 + g.n) * POLY + g.tid * 8;
    digits_mac<2, true>(acc, cnt, vv, t_conv, bits_conv, c0, (size_t)2 * 2 * POLY, (size_t)ccols * 2 * POLY, g);
  }
#pragma unroll
  for (int r = 0; r < 2; r++) {
    uint32_t o[8];
#pragma unroll
    for (int e = 0; e < 8; e++) o[e] = barrett64(acc[r][e], g.cr1, g.q);
    st8(out + (((size_t)r * cols + 2 * j) * 2 + g.n) * POLY + g.tid * 8, o);
  }
}

// ------------------------------------------------------------------ pack (v0: server.rs:429-468; v1: lib/server pack.rs:45-98)
template <int ROWS>
__global__ void __launch_bounds__(CTA, 1)
k_pack(DevParams P, uint64_t* out_raw, size_t out_q_stride, const uint32_t* folded, size_t ct_stride, size_t in_q_stride,
       const uint32_t* const* tab_pack, int t_conv, int bits, int version) {
  const uint32_t* v_packing = tab_pack[blockIdx.y];
  out_raw += (size_t)blockIdx.y * out_q_stride;
  folded += (size_t)blockIdx.y * in_q_stride;
  extern __shared__ __align__(16) uint8_t dyn_smem[];
  uint32_t* ntt_smem = reinterpret_cast<uint32_t*>(dyn_smem);
  uint32_t* res = ntt_smem + 4 * NTT_SMEM_WORDS;
  uint64_t* rawbuf = reinterpret_cast<uint64_t*>(res + 2 * POLY);     // [2048] (+ [2048] unused)
  Twiddle* tw = reinterpret_cast<Twiddle*>(rawbuf + 2 * POLY);        // [2][HI_TW]
  Grp g = make_grp(P, ntt_smem);
  g.smem2 = ntt_smem + (2 + g.n) * NTT_SMEM_WORDS;
  stage_fwd_twiddles(g, tw + g.n * HI_TW);
  constexpr int n = ROWS - 1;
  const int inst = blockIdx.x / n, c = blockIdx.x % n;
  const size_t mat_words = (size_t)ROWS * t_conv * 2 * POLY;
  const size_t row_step = (size_t)t_conv * 2 * POLY, col_step = (size_t)2 * POLY;

  uint32_t vint[ROWS][8];
#pragma unroll
  for (int m = 0; m < ROWS; m++)
#pragma unroll
    for (int e = 0; e < 8; e++) vint[m][e] = 0;

#pragma unroll 1
  for (int r = 0; r < n; r++) {
    // residue form: u32 [row][n][z]
    const uint32_t* ct = folded + ((size_t)inst * n * n + (size_t)r * n + c) * ct_stride;
    const uint32_t* W = v_packing + (version == 0 ? (size_t)r * mat_words : 0);
    uint64_t acc[ROWS][8];
#pragma unroll
    for (int m = 0; m < ROWS; m++)
#pragma unroll
      for (int e = 0; e < 8; e++) acc[m][e] = 0;
    int cnt = 0;
    {
      uint64_t vv[8];
#pragma unroll
      for (int a = 0; a < 8; a++) vv[a] = crt_compose(__ldg(ct + a * 256 + g.tid), __ldg(ct + POLY + a * 256 + g.tid), P);
      digits_mac<ROWS, true>(acc, cnt, vv, t_conv, bits, W + (size_t)g.n * POLY + g.tid * 8, col_step, row_step, g);
    }
    uint32_t y[8];
#pragma unroll
    for (int a = 0; a < 8; a++) y[a] = __ldg(ct + (2 + g.n) * POLY + a * 256 + g.tid);   // row 1 mod q_n
    grp_ntt_fwd<true>(g, y);
    uint32_t prod[ROWS][8];
#pragma unroll
    for (int m = 0; m < ROWS; m++)
#pragma unroll
      for (int e = 0; e < 8; e++) prod[m][e] = barrett64(acc[m][e], g.cr1, g.q);
    if (version == 0) {
      // add_into_at(v_int, ct_2_ntt, 1 + r, 0); add_into(v_int, prod)
#pragma unroll
      for (int m = 0; m < ROWS; m++)
#pragma unroll
        for (int e = 0; e < 8; e++) {
          uint32_t s = addmod(vint[m][e], prod[m][e], g.q);
          vint[m][e] = (m == 1 + r) ? addmod(s, y[e], g.q) : s;
        }
    } else {
      // add_into_at(prod, ct_2_ntt, 1, 0); then r row shifts through w_shift (= v_packing[1])
#pragma unroll
      for (int e = 0; e < 8; e++) prod[1][e] = addmod(prod[1][e], y[e], g.q);
      const uint32_t* Wshift = v_packing + mat_words;
#pragma unroll 1
      for (int sft = 0; sft < r; sft++) {
        uint32_t x[8];
#pragma unroll
        for (int e = 0; e < 8; e++) x[e] = prod[0][e];
        grp_ntt_inv(g, x);
        crt_lift(x, res, g, P, [&](int z, uint64_t val) { rawbuf[z] = val; });
        __syncthreads();
        uint64_t vv[8];
#pragma unroll
        for (int a = 0; a < 8; a++) vv[a] = rawbuf[a * 256 + g.tid];
#pragma unroll
        for (int m = 0; m < ROWS; m++)
#pragma unroll
          for (int e = 0; e < 8; e++) acc[m][e] = 0;
        cnt = 0;
        digits_mac<ROWS, true>(acc, cnt, vv, t_conv, bits, Wshift + (size_t)g.n * POLY + g.tid * 8, col_step, row_step, g);
        uint32_t np[ROWS][8];
#pragma unroll
        for (int m = 0; m < ROWS; m++)
#pragma unroll
          for (int e = 0; e < 8; e++) {
            uint32_t p1 = barrett64(acc[m][e], g.cr1, g.q);
            // shifted rest rows: new[1] = old[n]; new[1+k] = old[k] (k = 1..n-1); new[0] gets nothing
            uint32_t p2 = (m == 0) ? 0u : (m == 1 ? prod[n][e] : prod[m - 1][e]);
            np[m][e] = addmod(p1, p2, g.q);
          }
#pragma unroll
        for (int m = 0; m < ROWS; m++)
#pragma unroll
          for (int e = 0; e < 8; e++) prod[m][e] = np[m][e];
      }
#pragma unroll
      for (int m = 0; m < ROWS; m++)
#pragma unroll
        for (int e = 0; e < 8; e++) vint[m][e] = addmod(vint[m][e], prod[m][e], g.q);
    }
  }
  // result.copy_into(v_int, 0, c); packed_ct.raw()   (server.rs:464, :736)
#pragma unroll 1
  for (int m = 0; m < ROWS; m++) {
    uint32_t x[8];
#pragma unroll
    for (int e = 0; e < 8; e++) x[e] = vint[m][e];
    grp_ntt_inv(g, x);
    uint64_t* d = out_raw + (((size_t)inst * ROWS + m) * n + c) * POLY;
    crt_lift(x, res, g, P, [&](int z, uint64_t val) { d[z] = val; });
  }
}

// ------------------------------------------------------------------ encode (server.rs:470-503)
// arith.rs:429-444
__device__ __forceinline__ uint64_t rescale_dev(uint64_t a, uint64_t inp_mod, uint64_t out_mod) {
  typedef __int128 i128;
  long long inp_mod_i = (long long)inp_mod;
  long long inp_val = (long long)(a % inp_mod);
  if (inp_val >= inp_mod_i / 2) inp_val -= inp_mod_i;
  long long sign = inp_val >= 0 ? 1 : -1;
  i128 val = (i128)inp_val * (i128)out_mod;
  i128 result = (val + (i128)(sign * (inp_mod_i / 2))) / (i128)inp_mod;
  i128 om = (i128)out_mod;
  result = (result + (i128)((inp_mod / out_mod) * out_mod) + 2 * om) % om;
  return (uint64_t)((result + om) % om);
}
// One thread per output 64-bit word.  Stream = per instance: n*2048 values of q2_bits (row 0 of the
// packed matrix), then n*n*2048 values of q1_bits (rows 1..n), LSB-first (util.rs:303-321).
__global__ void k_encode(DevParams P, uint64_t* out, size_t out_words, const uint64_t* packed, size_t packed_q_stride, int n,
                         int instances, uint64_t q2, int q2_bits, uint64_t q1, int q1_bits) {
  size_t w = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= out_words) return;
  out += (size_t)blockIdx.y * out_words;
  packed += (size_t)blockIdx.y * packed_q_stride;
  const uint64_t first_cnt = (uint64_t)n * POLY, rest_cnt = (uint64_t)n * n * POLY;
  const uint64_t inst_bits = first_cnt * q2_bits + rest_cnt * q1_bits;
  uint64_t lo_bit = (uint64_t)w * 64, hi_bit = lo_bit + 64;
  uint64_t word = 0;
  uint64_t bit = lo_bit;
  while (bit < hi_bit) {
    uint64_t inst = bit / inst_bits;
    if (inst >= (uint64_t)instances) break;
    uint64_t off = bit - inst * inst_bits;
    const uint64_t* pk = packed + inst * (uint64_t)(n + 1) * n * POLY;
    uint64_t vstart, val;
    int vb;
    if (off < first_cnt * q2_bits) {
      uint64_t vi = off / q2_bits;
      vstart = inst * inst_bits + vi * q2_bits;
      vb = q2_bits;
      val = rescale_dev(pk[vi], P.modulus, q2);
    } else {
      uint64_t o2 = off - first_cnt * q2_bits;
      uint64_t vi = o2 / q1_bits;
      vstart = inst * inst_bits + first_cnt * q2_bits + vi * q1_bits;
      vb = q1_bits;
      val = rescale_dev(pk[first_cnt + vi], P.modulus, q1);
    }
    val &= (vb >= 64) ? ~0ull : ((1ull << vb) - 1);
    // bits [vstart, vstart+vb) of the stream hold val; copy the part overlapping this word
    if (vstart >= lo_bit) word |= val << (vstart - lo_bit);
    else word |= val >> (lo_bit - vstart);
    bit = vstart + vb;
  }
  out[w] = word;
}

inline unsigned grid1d(size_t total, int block) { return (unsigned)((total + block - 1) / block); }
const size_t kDynSmemBig = (size_t)(4 * NTT_SMEM_WORDS + 2 * POLY) * 4 + (size_t)2 * POLY * 8 + (size_t)2 * HI_TW * 8;
const size_t kDynSmemFold = (size_t)(2 * NTT_SMEM_WORDS) * 4 + (size_t)HI_TW * 8;

}  // namespace

void upload_poly_constants(const Twiddle* lo /* [2][3][64]: forward, inverse, relaxed-range inverse */) {
  B200_CUDA(cudaMemcpyToSymbol(c_tw_lo, lo, sizeof(Twiddle) * 2 * 3 * 64));
}
void launch_ntt_u64(const DevParams& P, uint64_t* polys, size_t count, bool inverse, cudaStream_t s) {
  if (count) ++g_kernel_launches, k_ntt_u64<<<dim3((unsigned)count, 2), 256, 0, s>>>(P, polys, inverse ? 1 : 0);
}
void launch_ntt32(const DevParams& P, uint32_t* polys, size_t count, bool inverse, cudaStream_t s) {
  if (count) ++g_kernel_launches, k_ntt32<<<dim3((unsigned)count, 2), 256, 0, s>>>(P, polys, inverse ? 1 : 0);
}
void launch_ntt32_4k(uint32_t q0, uint32_t q1, const Twiddle* tw, uint32_t* polys, size_t count, bool inverse, cudaStream_t s) {
  if (count) ++g_kernel_launches, k_ntt32_4k<<<dim3((unsigned)count, 2), NTT4K_THREADS, 0, s>>>(q0, q1, tw, polys, inverse ? 1 : 0);
}
void launch_to_ntt(const DevParams& P, uint32_t* out, const uint64_t* raw, size_t count, cudaStream_t s) {
  if (count) ++g_kernel_launches, k_to_ntt<<<dim3((unsigned)count, 2), 256, 0, s>>>(P, out, raw, 0, 0);
}
void launch_to_ntt_strided(const DevParams& P, uint32_t* out, size_t out_stride, const uint64_t* raw, size_t raw_stride,
                           size_t count, int batches, cudaStream_t s) {
  if (count && batches)
    ++g_kernel_launches, k_to_ntt<<<dim3((unsigned)count, 2, (unsigned)batches), 256, 0, s>>>(P, out, raw, out_stride, raw_stride);
}
void launch_raw_to_res(const DevParams& P, uint32_t* out, const uint64_t* raw, size_t polys, cudaStream_t s) {
  if (polys) ++g_kernel_launches, k_raw_to_res<<<grid1d(polys * POLY, 256), 256, 0, s>>>(P, out, raw, polys);
}
void launch_res_to_raw(const DevParams& P, uint64_t* out, const uint32_t* res, size_t polys, cudaStream_t s) {
  if (polys) ++g_kernel_launches, k_res_to_raw<<<grid1d(polys * POLY, 256), 256, 0, s>>>(P, out, res, polys);
}
void launch_fold_res(const DevParams& P, const uint32_t* in, uint32_t* out, size_t batch, size_t batch_stride, int half,
                     const uint32_t* c_pos, size_t c_batch_stride, int slices_per_query, int t_gsw, int bits,
                     int variant, uint32_t* zero_flags, cudaStream_t s) {
  if (batch == 0 || half == 0) return;
  if (zero_flags) {            // scratch of batch * 2 * half words: recomputed every round, as the reference re-tests every step
    ++g_kernel_launches;
    k_ct_zero_flags<<<(unsigned)(batch * 2 * half), 256, 0, s>>>(in, batch_stride, 2 * half, zero_flags);
  }
  ++g_kernel_launches;
  // variant 3: 2 CTAs per SM (128 registers); anything else: 3 CTAs per SM (80 registers) — same speed on S8, kept for A/B runs
  const dim3 grid((unsigned)(batch * half), 2);
#define FOLD_LZ(MINB, BYTE)                                                                                             \
  do {                                                                                                                  \
    opt_in_smem(k_fold_res_lz<MINB, BYTE>, (int)kDynSmemFold);                                                          \
    k_fold_res_lz<MINB, BYTE><<<grid, 256, kDynSmemFold, s>>>(P, in, out, batch_stride, half, c_pos, c_batch_stride,    \
                                                             slices_per_query, t_gsw, bits, zero_flags);               \
  } while (0)
  if (variant == 3) { if (bits == 8) FOLD_LZ(2, true); else FOLD_LZ(2, false); }
  else { if (bits == 8) FOLD_LZ(3, true); else FOLD_LZ(3, false); }
#undef FOLD_LZ
}
void launch_from_ntt(const DevParams& P, uint64_t* out_raw, const uint32_t* in, size_t count, cudaStream_t s) {
  if (count) ++g_kernel_launches, k_from_ntt<<<(unsigned)count, CTA, 0, s>>>(P, out_raw, in);
}
void launch_widen(uint64_t* out, const uint32_t* in, size_t words, cudaStream_t s) {
  if (words) ++g_kernel_launches, k_widen<<<grid1d(words, 256), 256, 0, s>>>(out, in, words);
}
void launch_narrow(uint32_t* out, const uint64_t* in, size_t words, cudaStream_t s) {
  if (words) ++g_kernel_launches, k_narrow<<<grid1d(words, 256), 256, 0, s>>>(out, in, words);
}
void launch_fold_round(const DevParams& P, uint64_t* cts, size_t batch, size_t batch_stride, int half,
                       const uint32_t* c_pos, const uint32_t* c_neg, size_t c_batch_stride, int slices_per_query,
                       int t_gsw, int bits, cudaStream_t s) {
  if (batch == 0 || half == 0) return;
  ++g_kernel_launches;
  k_fold_round<<<(unsigned)(batch * half), CTA, 0, s>>>(P, cts, batch_stride, half, c_pos, c_neg, c_batch_stride,
                                                        slices_per_query, t_gsw, bits);
}
void launch_folding_neg(const DevParams& P, uint32_t* out, const uint32_t* v_folding, int count, int t_gsw, int bits,
                        cudaStream_t s) {
  size_t total = (size_t)count * 2 * 2 * t_gsw * 2 * POLY;
  if (total) ++g_kernel_launches, k_folding_neg<<<grid1d(total, 256), 256, 0, s>>>(P, out, v_folding, total, t_gsw, bits);
}
void launch_expand_scalar(const DevParams& P, uint32_t* v, size_t v_stride, int nq, int num_in, const uint32_t* neg1_r,
                          cudaStream_t s) {
  size_t total = (size_t)num_in * 4 * POLY;
  ++g_kernel_launches;
  k_expand_scalar<<<dim3(grid1d(total, 256), nq), 256, 0, s>>>(P, v, v_stride, num_in, neg1_r);
}
void launch_expand_round(const DevParams& P, uint32_t* v, size_t v_stride, int nq, const ExpandRound& R, cudaStream_t s) {
  opt_in_smem(k_expand_round, (int)kDynSmemBig);
  ++g_kernel_launches;
  k_expand_round<<<dim3((unsigned)(2 * R.num_in), nq), CTA, kDynSmemBig, s>>>(P, v, v_stride, R);
}
void launch_expand_round_pair(const DevParams& P, uint32_t* v, size_t v_stride, int nq, const ExpandRound& R,
                              const uint32_t* neg1_r, cudaStream_t s) {
  opt_in_smem(k_expand_round_pair, (int)kDynSmemBig);
  ++g_kernel_launches;
  k_expand_round_pair<<<dim3((unsigned)R.num_in, nq), CTA, kDynSmemBig, s>>>(P, v, v_stride, R, neg1_r);
}
void launch_expand_round_res(const DevParams& P, uint32_t* v, size_t v_stride, uint32_t* xr, size_t xr_stride, int nq,
                             const ExpandRound& R, const uint32_t* neg1_r, cudaStream_t s) {
  const size_t smem = (size_t)2 * NTT_SMEM_WORDS * 4 + (size_t)POLY * 8 + (size_t)HI_TW * 8;
  opt_in_smem(k_expand_round_res<3>, (int)smem);
  g_kernel_launches += 2;
  k_expand_intt<<<dim3((unsigned)R.num_in, 2, nq), 256, 0, s>>>(P, v, v_stride, xr, xr_stride, R);
  k_expand_round_res<3><<<dim3((unsigned)R.num_in, 2, nq), 256, smem, s>>>(P, v, v_stride, xr, xr_stride, R, neg1_r);
}
void launch_reorient(const MulGeom& G, uint4* q_dev, size_t q_stride, const uint32_t* v, size_t v_stride, int nq,
                     int idx_factor, cudaStream_t s) {
  size_t total = (size_t)G.dim0 * POLY;
  ++g_kernel_launches;
  k_reorient<<<dim3(grid1d(total, 256), nq), 256, 0, s>>>(G, q_dev, q_stride, v, v_stride, idx_factor);
}
void launch_regev_to_gsw(const DevParams& P, uint32_t* v_gsw, size_t gsw_stride, const uint32_t* v, size_t v_stride,
                         int nq, int count, int idx_factor, int idx_offset, const uint32_t* const* tab_conv, int t_gsw,
                         int t_conv, int bits_conv, cudaStream_t s) {
  if (count == 0) return;
  opt_in_smem(k_regev_to_gsw, (int)kDynSmemBig);
  ++g_kernel_launches;
  k_regev_to_gsw<<<dim3((unsigned)(count * t_gsw), nq), CTA, kDynSmemBig, s>>>(P, v_gsw, gsw_stride, v, v_stride,
                                                                               idx_factor, idx_offset, tab_conv, t_gsw,
                                                                               t_conv, bits_conv);
}
template <int ROWS>
static void launch_pack_t(const DevParams& P, uint64_t* out_raw, size_t out_q_stride, const uint32_t* folded,
                          size_t ct_stride, size_t in_q_stride, int nq, const uint32_t* const* tab_pack, int instances,
                          int t_conv, int bits_conv, int version, cudaStream_t s) {
  opt_in_smem(k_pack<ROWS>, (int)kDynSmemBig);
  ++g_kernel_launches;
  k_pack<ROWS><<<dim3((unsigned)(instances * (ROWS - 1)), nq), CTA, kDynSmemBig, s>>>(
      P, out_raw, out_q_stride, folded, ct_stride, in_q_stride, tab_pack, t_conv, bits_conv, version);
}
void launch_pack(const DevParams& P, uint64_t* out_raw, size_t out_q_stride, const uint32_t* folded, size_t ct_stride,
                 size_t in_q_stride, int nq, const uint32_t* const* tab_pack, int n, int instances, int t_conv, int bits_conv,
                 int version, cudaStream_t s) {
  switch (n) {
    case 1: launch_pack_t<2>(P, out_raw, out_q_stride, folded, ct_stride, in_q_stride, nq, tab_pack, instances, t_conv, bits_conv, version, s); break;
    case 2: launch_pack_t<3>(P, out_raw, out_q_stride, folded, ct_stride, in_q_stride, nq, tab_pack, instances, t_conv, bits_conv, version, s); break;
    case 3: launch_pack_t<4>(P, out_raw, out_q_stride, folded, ct_stride, in_q_stride, nq, tab_pack, instances, t_conv, bits_conv, version, s); break;
    case 4: launch_pack_t<5>(P, out_raw, out_q_stride, folded, ct_stride, in_q_stride, nq, tab_pack, instances, t_conv, bits_conv, version, s); break;
    default: throw Error(-2, "pack: n must be 1..4");
  }
}
void launch_encode(const DevParams& P, uint8_t* out, size_t out_bytes, const uint64_t* packed_raw, size_t packed_q_stride,
                   int nq, int n, int instances, uint64_t q2, int q2_bits, uint64_t q1, int q1_bits, cudaStream_t s) {
  size_t words = out_bytes / 8;
  ++g_kernel_launches;
  k_encode<<<dim3(grid1d(words, 128), nq), 128, 0, s>>>(P, reinterpret_cast<uint64_t*>(out), words, packed_raw,
                                                        packed_q_stride, n, instances, q2, q2_bits, q1, q1_bits);
}

}  // namespace b200pir
