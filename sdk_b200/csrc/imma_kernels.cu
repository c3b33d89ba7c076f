// First dimension on the INT8 tensor-core path (batched queries).
//
// multiply_reg_by_database (lib/spiral-rs/src/server.rs:155-221) is, for every NTT coordinate z and CRT
// modulus n, a small integer GEMM  C[ii][(query,row)] = sum_j A[ii][j] * B[j][(query,row)]  mod q_n  with
// M = num_per, K = dim0, N = 2 * (number of queries).  With one query the database stream (8 B per word) is the
// bound and the IMAD kernel in mul_kernels.cu already runs at the HBM roofline; with several queries per
// database pass the 32x32->64-bit IMADs become the bound.  Here the 28-bit residues are split into four 7-bit
// limbs and the products are formed by u8 x u8 -> s32 tensor-core MMAs (mma.sync m16n8k32, SASS IMMA.16832.U8.U8):
//
//     a * b = sum_{l,m < 4} a_l b_m 2^{7(l+m)}          a_l, b_m < 2^7
//
// Every limb product is < 2^14, a K = dim0 <= 1024 accumulation < 2^24, and the (at most 4) limb pairs with the
// same shift l+m share one s32 accumulator (< 2^26): all integer arithmetic is EXACT.  The seven shift groups
// are recombined as  sum_s acc_s * (2^{7s} mod q_n)  (< 2^57) and reduced with one Barrett step, which yields the
// same canonical residue as the reference's u128 accumulate + `%`.  Parity is asserted bit-for-bit against the
// oracle in tests/test_gpu_parity.py before this path is used by anything.
//
// The database is re-tiled once into MMA *fragment order*, so a lane's A operand is one coalesced 16-byte load
// straight from HBM (no shared memory, no ldmatrix):
//     dbF[slice][n][z][mt][ks][limb l][lane] = uint4{a0,a1,a2,a3}     (mt: 16 rows, ks: 32 values of j)
// One CTA = one (slice, n, z): its 8 warps share the query operand B (<= 32 KiB, shared memory) and each streams
// the fragments of two row tiles.
#include "kernels.h"
#include "item_write.cuh"

namespace b200pir {

namespace {

__device__ __forceinline__ void mma_u8(int (&c)[4], const uint4& a, const uint2& b) {
  asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.u8.u8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3])
               : "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w), "r"(b.x), "r"(b.y));
}
__device__ __forceinline__ uint32_t limb4(uint32_t x0, uint32_t x1, uint32_t x2, uint32_t x3, int l) {
  const int sh = 7 * l;
  return ((x0 >> sh) & 127u) | (((x1 >> sh) & 127u) << 8) | (((x2 >> sh) & 127u) << 16) | (((x3 >> sh) & 127u) << 24);
}

// format 0 (mul_kernels.cu: uint4 [row][jp][z]) of one slice  ->  fragment order.  One warp per (z, mt, ks).
__global__ void __launch_bounds__(256)
k_db_to_frag(ImmaGeom F, const uint4* __restrict__ db0_slice, uint4* __restrict__ dbf, int slice) {
  const int lane = threadIdx.x & 31;
  const size_t warp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const size_t total = (size_t)POLY * F.mt * F.ks;
  if (warp >= total) return;
  const int ks = (int)(warp % F.ks);
  const int mt = (int)((warp / F.ks) % F.mt);
  const int z = (int)(warp / ((size_t)F.ks * F.mt));
  const int g = lane >> 2, t = lane & 3;
  const int half = F.dim0 >> 1;
  uint32_t res[2][2][2][4];        // [n][row half (g, g+8)][k half (0, +16)][i]
#pragma unroll
  for (int rh = 0; rh < 2; rh++) {
    const int ii = mt * 16 + g + 8 * rh;
#pragma unroll
    for (int kh = 0; kh < 2; kh++) {
      const int j0 = ks * 32 + 16 * kh + 4 * t;       // j0 .. j0+3
#pragma unroll
      for (int p = 0; p < 2; p++) {                   // two uint4 cells: (j0, j0+1), (j0+2, j0+3)
        const int jp = (j0 >> 1) + p;
        uint4 w = make_uint4(0, 0, 0, 0);
        if (ii < F.rows && jp < half) w = db0_slice[((size_t)ii * half + jp) * POLY + z];
        res[0][rh][kh][2 * p] = w.x; res[1][rh][kh][2 * p] = w.y;
        res[0][rh][kh][2 * p + 1] = w.z; res[1][rh][kh][2 * p + 1] = w.w;
      }
    }
  }
#pragma unroll
  for (int n = 0; n < 2; n++) {
    uint4* dst = dbf + (((((size_t)slice * 2 + n) * POLY + z) * F.mt + mt) * F.ks + ks) * 4 * 32 + lane;
#pragma unroll
    for (int l = 0; l < 4; l++) {
      uint4 o;
      o.x = limb4(res[n][0][0][0], res[n][0][0][1], res[n][0][0][2], res[n][0][0][3], l);   // a0: row g,   k 4t..
      o.y = limb4(res[n][1][0][0], res[n][1][0][1], res[n][1][0][2], res[n][1][0][3], l);   // a1: row g+8
      o.z = limb4(res[n][0][1][0], res[n][0][1][1], res[n][0][1][2], res[n][0][1][3], l);   // a2: row g,   k 16+4t..
      o.w = limb4(res[n][1][1][0], res[n][1][1][1], res[n][1][1][2], res[n][1][1][3], l);   // a3: row g+8
      dst[(size_t)l * 32] = o;
    }
  }
}

// where word z of item (slice, local row il, j) lives in fragment order (byte writes); w = lo | hi << 32
struct FragStore {
  ImmaGeom F;
  uint4* dbf;
  __device__ __forceinline__ void operator()(int slice, int il, int j, int z, uint64_t w) const {
    const int mt = il >> 4, row = il & 15, ks = j >> 5, k = j & 31;
    const int g = row & 7, rh = row >> 3, kh = k >> 4, t = (k & 15) >> 2, i = k & 3;
    const int lane = g * 4 + t, reg = rh + 2 * kh;     // a0..a3 = (row g,k lo), (row g+8,k lo), (row g,k hi), (row g+8,k hi)
#pragma unroll
    for (int n = 0; n < 2; n++) {
      uint32_t r = n ? (uint32_t)(w >> 32) : (uint32_t)w;
      uint8_t* base = reinterpret_cast<uint8_t*>(dbf + (((((size_t)slice * 2 + n) * POLY + z) * F.mt + mt) * F.ks + ks) * 4 * 32);
#pragma unroll
      for (int l = 0; l < 4; l++) base[((size_t)l * 32 + lane) * 16 + reg * 4 + i] = (uint8_t)((r >> (7 * l)) & 127u);
    }
  }
};

// one item polynomial (2048 packed words lo|hi<<32) into the fragment-order database
__global__ void k_db_upsert_frag(FragStore st, int slice, int il, int j, const uint64_t* poly) {
  int z = blockIdx.x * blockDim.x + threadIdx.x;
  if (z >= POLY) return;
  st(slice, il, j, z, poly[z]);
}

// expanded queries (format of mul_kernels.cu: uint4 [jp][jb][z]) -> B fragments
//   qf[n][z][nt][ks][limb m][lane] = uint2{b0, b1};  column (nt*8 + g) = 2*query + ciphertext row
__global__ void __launch_bounds__(256)
k_query_to_frag(ImmaGeom F, const uint4* __restrict__ q_dev, size_t q_stride, int nq, int ntiles, uint2* __restrict__ qf) {
  const int lane = threadIdx.x & 31;
  const size_t warp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const size_t total = (size_t)POLY * ntiles * F.ks;
  if (warp >= total) return;
  const int ks = (int)(warp % F.ks);
  const int nt = (int)((warp / F.ks) % ntiles);
  const int z = (int)(warp / ((size_t)F.ks * ntiles));
  const int g = lane >> 2, t = lane & 3;
  const int q = nt * 4 + (g >> 1), r = g & 1;
  uint32_t res[2][2][4];      // [n][k half][i]
#pragma unroll
  for (int kh = 0; kh < 2; kh++)
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const int j = ks * 32 + 16 * kh + 4 * t + i;
      uint4 w = make_uint4(0, 0, 0, 0);
      if (q < nq && j < F.dim0) w = q_dev[(size_t)q * q_stride + ((size_t)(j >> 1) * 2 + (j & 1)) * POLY + z];
      res[0][kh][i] = r ? w.z : w.x;
      res[1][kh][i] = r ? w.w : w.y;
    }
#pragma unroll
  for (int n = 0; n < 2; n++)
#pragma unroll
    for (int m = 0; m < 4; m++) {
      uint2 o;
      o.x = limb4(res[n][0][0], res[n][0][1], res[n][0][2], res[n][0][3], m);
      o.y = limb4(res[n][1][0], res[n][1][1], res[n][1][2], res[n][1][3], m);
      qf[(((((size_t)n * POLY + z) * ntiles + nt) * F.ks + ks) * 4 + m) * 32 + lane] = o;
    }
}

// out_zm[query][slice][n][z][row][ct_row] (u32): the product for up to 4*NT queries in one database pass.
// NT = 1: each warp iteration covers 2 row tiles x 1 column tile; NT = 2: 1 row tile x 2 column tiles.
template <int NT>
__global__ void __launch_bounds__(256, 2)
k_multiply_imma(DevParams P, ImmaGeom F, const uint4* __restrict__ dbf, const uint2* __restrict__ qf,
                uint32_t* __restrict__ out_zm, size_t out_stride, int nq, int slice_begin, int slice_count) {
  extern __shared__ __align__(16) uint2 bsm[];            // [nt][ks][m][lane]
  constexpr int RT = NT == 1 ? 2 : 1;                     // row tiles per warp iteration
  // CTA = one (n, z): the B operand is staged once and shared by every slice; the work items (slice, row tiles) are
  // spread over the 8 warps, so small row shards (multi-GPU) still keep all warps busy
  const int z = blockIdx.x, n = blockIdx.y;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  {
    const uint2* src = qf + ((size_t)n * POLY + z) * NT * F.ks * 4 * 32;
    for (int i = threadIdx.x; i < NT * F.ks * 128; i += blockDim.x) bsm[i] = __ldg(src + i);
  }
  __syncthreads();
  const uint32_t q = n ? P.q[1] : P.q[0];
  const uint64_t cr1 = n ? P.cr1[1] : P.cr1[0];
  uint32_t p7[7];                                          // 2^{7s} mod q_n
#pragma unroll
  for (int s = 0; s < 7; s++) p7[s] = (uint32_t)((1ull << (7 * s)) % q);
  const int g = lane >> 2, t = lane & 3;
  const int nwarps = blockDim.x >> 5;
  const int groups = (F.mt + RT - 1) / RT;                 // row-tile groups per slice
  for (int item = warp; item < slice_count * groups; item += nwarps) {
    const int slice = slice_begin + item / groups;
    const int mt0 = (item % groups) * RT;
    const uint4* base = dbf + (((size_t)slice * 2 + n) * POLY + z) * F.mt * F.ks * 4 * 32 + lane;
    const bool two = RT == 2 && (mt0 + 1) < F.mt;
    int acc[2][7][4];                                      // [row tile (NT=1) or column tile (NT=2)][shift][c]
#pragma unroll
    for (int a = 0; a < 2; a++)
#pragma unroll
      for (int s = 0; s < 7; s++)
#pragma unroll
        for (int i = 0; i < 4; i++) acc[a][s][i] = 0;
    const uint4* a0p = base + (size_t)mt0 * F.ks * 4 * 32;
    const uint4* a1p = a0p + (size_t)(two ? 1 : 0) * F.ks * 4 * 32;
#pragma unroll 1
    for (int ks = 0; ks < F.ks; ks++) {
      uint4 A0[4], A1[4];
#pragma unroll
      for (int l = 0; l < 4; l++) {
        A0[l] = ld_stream_v4(a0p + ((size_t)ks * 4 + l) * 32);
        if (RT == 2) A1[l] = ld_stream_v4(a1p + ((size_t)ks * 4 + l) * 32);
      }
      uint2 B0[4], B1[4];
#pragma unroll
      for (int m = 0; m < 4; m++) {
        B0[m] = bsm[(ks * 4 + m) * 32 + lane];
        if (NT == 2) B1[m] = bsm[((F.ks + ks) * 4 + m) * 32 + lane];
      }
#pragma unroll
      for (int l = 0; l < 4; l++)
#pragma unroll
        for (int m = 0; m < 4; m++) {
          mma_u8(acc[0][l + m], A0[l], B0[m]);
          if (RT == 2) mma_u8(acc[1][l + m], A1[l], B0[m]);
          if (NT == 2) mma_u8(acc[1][l + m], A0[l], B1[m]);
        }
    }
    // recombine the shift groups, reduce, store:  c0,c1 -> row g, columns 2t, 2t+1 ; c2,c3 -> row g+8
#pragma unroll
    for (int a = 0; a < 2; a++) {
      const int mt = RT == 2 ? mt0 + a : mt0;
      const int qi = (NT == 2 ? a * 4 : 0) + t;            // column pair (2t, 2t+1) of column tile = query, ct rows 0/1
      if (RT == 2 && a == 1 && !two) break;
      if (qi >= nq) continue;
#pragma unroll
      for (int rh = 0; rh < 2; rh++) {
        const int ii = mt * 16 + g + 8 * rh;
        if (ii < F.rows) {
          uint64_t v0 = 0, v1 = 0;
#pragma unroll
          for (int s = 0; s < 7; s++) {
            v0 += (uint64_t)(uint32_t)acc[a][s][2 * rh] * p7[s];
            v1 += (uint64_t)(uint32_t)acc[a][s][2 * rh + 1] * p7[s];
          }
          uint2 o = make_uint2(barrett64(v0, cr1, q), barrett64(v1, cr1, q));
          uint32_t* dst = out_zm + (size_t)qi * out_stride + ((((size_t)slice * 2 + n) * POLY + z) * F.rows + ii) * 2;
          *reinterpret_cast<uint2*>(dst) = o;
        }
      }
    }
  }
}


// ---- 5..8 queries per database pass, software-pipelined --------------------------------------------------------------
// Same arithmetic as k_multiply_imma<2> (one row tile x two column tiles per warp step).  With eight queries per pass the
// kernel sits between the HBM and the IMMA roofs, so it has to keep far more bytes in flight than a load-then-use loop
// does: every warp runs its own IMMA_STAGES-deep cp.async ring (2 KiB = one k-step of A fragments per stage, each lane
// copies and later reads only its own 16-byte chunks, so no barrier is involved), flattened over all of its (slice, row
// tile) work items so that the ring never drains at an item boundary.
constexpr int IMMA_STAGES = 4;          // NT = 2: two CTAs per SM
constexpr int IMMA_STAGES16 = 8;        // NT = 4 (9..16 queries per pass): one CTA per SM, 112 accumulator registers

__device__ __forceinline__ void cp_async16(uint32_t smem_addr, const void* gptr) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_addr), "l"(gptr) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <int NT, int STAGES>
__global__ void __launch_bounds__(256, NT == 2 ? 2 : 1)
k_multiply_imma8(DevParams P, ImmaGeom F, const uint4* __restrict__ dbf, const uint2* __restrict__ qf,
                 uint32_t* __restrict__ out_zm, size_t out_stride, int nq, int slice_begin, int slice_count) {
  extern __shared__ __align__(16) uint2 bsm[];            // [nt][ks][m][lane], then the per-warp A rings
  const int z = blockIdx.x, n = blockIdx.y;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nwarps = blockDim.x >> 5;
  uint4* ring = reinterpret_cast<uint4*>(bsm + (size_t)NT * F.ks * 128) + (size_t)warp * STAGES * 128;
  const uint32_t ring_s = (uint32_t)__cvta_generic_to_shared(ring);
  const int total_items = slice_count * F.mt;
  const int my_items = warp < total_items ? (total_items - warp + nwarps - 1) / nwarps : 0;
  const int T = my_items * F.ks;
  const uint4* zbase = dbf + ((size_t)n * POLY + z) * F.mt * F.ks * 128 + lane;
  const size_t slice_words = (size_t)2 * POLY * F.mt * F.ks * 128;
  auto issue = [&](int it) {                              // stage `it`: A fragments of (item it / ks, k-step it % ks)
    if (it < T) {
      const int item = warp + (it / F.ks) * nwarps, ks = it % F.ks;
      const int slice = slice_begin + item / F.mt, mt = item % F.mt;
      const uint4* src = zbase + (size_t)slice * slice_words + ((size_t)mt * F.ks + ks) * 128;
      const uint32_t dst = ring_s + (uint32_t)(((it % STAGES) * 128 + lane) * 16);
#pragma unroll
      for (int l = 0; l < 4; l++) cp_async16(dst + l * 32 * 16, src + l * 32);
    }
    cp_async_commit();
  };
#pragma unroll
  for (int s = 0; s < STAGES - 1; s++) issue(s);
  {
    const uint2* src = qf + ((size_t)n * POLY + z) * NT * F.ks * 128;
    for (int i = threadIdx.x; i < NT * F.ks * 128; i += blockDim.x) bsm[i] = __ldg(src + i);
  }
  __syncthreads();
  const uint32_t q = n ? P.q[1] : P.q[0];
  const uint64_t cr1 = n ? P.cr1[1] : P.cr1[0];
  uint32_t p7[7];
#pragma unroll
  for (int s = 0; s < 7; s++) p7[s] = (uint32_t)((1ull << (7 * s)) % q);
  const int g = lane >> 2, t = lane & 3;
  int acc[NT][7][4];
#pragma unroll
  for (int a = 0; a < NT; a++)
#pragma unroll
    for (int s = 0; s < 7; s++)
#pragma unroll
      for (int i = 0; i < 4; i++) acc[a][s][i] = 0;
  int ks = 0, item = warp;
#pragma unroll 1
  for (int it = 0; it < T; it++) {
    cp_async_wait<STAGES - 2>();                          // stage `it` has landed (this lane's own chunks)
    issue(it + STAGES - 1);                               // refill the slot consumed in the previous iteration
    const uint4* st = ring + (it % STAGES) * 128 + lane;
    uint4 A[4];
#pragma unroll
    for (int l = 0; l < 4; l++) A[l] = st[l * 32];
#pragma unroll
    for (int m = 0; m < 4; m++) {
      uint2 b[NT];
#pragma unroll
      for (int c = 0; c < NT; c++) b[c] = bsm[((c * F.ks + ks) * 4 + m) * 32 + lane];
#pragma unroll
      for (int l = 0; l < 4; l++)
#pragma unroll
        for (int c = 0; c < NT; c++) mma_u8(acc[c][l + m], A[l], b[c]);
    }
    if (++ks == F.ks) {
      // recombine the shift groups, reduce, store:  c0,c1 -> row g, columns 2t, 2t+1 ; c2,c3 -> row g+8
      const int slice = slice_begin + item / F.mt, mt = item % F.mt;
#pragma unroll
      for (int a = 0; a < NT; a++) {
        const int qi = a * 4 + t;
#pragma unroll
        for (int rh = 0; rh < 2; rh++) {
          const int ii = mt * 16 + g + 8 * rh;
          if (qi < nq && ii < F.rows) {
            uint64_t v0 = 0, v1 = 0;
#pragma unroll
            for (int s = 0; s < 7; s++) {
              v0 += (uint64_t)(uint32_t)acc[a][s][2 * rh] * p7[s];
              v1 += (uint64_t)(uint32_t)acc[a][s][2 * rh + 1] * p7[s];
            }
            uint2 o = make_uint2(barrett64(v0, cr1, q), barrett64(v1, cr1, q));
            uint32_t* dst = out_zm + (size_t)qi * out_stride + ((((size_t)slice * 2 + n) * POLY + z) * F.rows + ii) * 2;
            *reinterpret_cast<uint2*>(dst) = o;
          }
        }
#pragma unroll
        for (int s = 0; s < 7; s++)
#pragma unroll
          for (int i = 0; i < 4; i++) acc[a][s][i] = 0;
      }
      ks = 0;
      item += nwarps;
    }
  }
  cp_async_wait<0>();
}

__constant__ Twiddle c_tw_lo_imma[2][3][64];
struct TwConstI {
  int n, dir;
  __device__ __forceinline__ Twiddle operator()(int i) const { return c_tw_lo_imma[n][dir][i]; }
  __device__ __forceinline__ void load2(int i, Twiddle (&t)[2]) const { t[0] = (*this)(i); t[1] = (*this)(i + 1); }
  __device__ __forceinline__ void load4(int i, Twiddle (&t)[4]) const {
    t[0] = (*this)(i); t[1] = (*this)(i + 1); t[2] = (*this)(i + 2); t[3] = (*this)(i + 3);
  }
};
struct TwGlobalI {
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
struct SyncI {
  __device__ __forceinline__ void operator()() const { __syncthreads(); }
};

// inverse NTT of every (ciphertext row, modulus) of the z-major product -> residue-form ciphertexts
//   out[((query*slices + slice)*rows + ii)][ct_row][n][z]     (server.rs:707-709 without the CRT lift)
// grid = (rows*2 polys, 2 moduli, nq*slices), 256 threads
__global__ void __launch_bounds__(256)
k_intt_from_zmajor(DevParams P, ImmaGeom F, const uint32_t* __restrict__ in_zm, size_t in_stride, uint32_t* __restrict__ out,
                   int slices) {
  __shared__ __align__(16) uint32_t sm[NTT_SMEM_WORDS];
  const int tid = threadIdx.x, n = blockIdx.y;
  const int ii = blockIdx.x >> 1, r = blockIdx.x & 1;
  const int qs = blockIdx.z, qi = qs / slices, slice = qs % slices;
  const uint32_t q = n ? P.q[1] : P.q[0];
  const uint32_t* src = in_zm + (size_t)qi * in_stride + (((size_t)slice * 2 + n) * POLY) * F.rows * 2 + (size_t)ii * 2 + r;
  uint32_t x[8];
#pragma unroll
  for (int k = 0; k < 8; k++) x[k] = __ldg(src + (size_t)(tid * 8 + k) * F.rows * 2);
  ntt_inverse_group_nh(tid, x, sm, TwConstI{n, 2}, TwGlobalI{n ? P.inv_lz[1] : P.inv_lz[0]}, q, SyncI());
  uint32_t* dst = out + ((((size_t)qs * F.rows + ii) * 2 + r) * 2 + n) * POLY;
#pragma unroll
  for (int a = 0; a < 8; a++) dst[a * 256 + tid] = x[a];
}

// Tiled variant: one CTA handles PP (= 2, 4 or 8) polynomials that are adjacent in the z-major product, so every
// 32-byte sector it fetches is fully used (the simple kernel above uses 4 of every 32 bytes).  The PP polynomials are
// transposed through shared memory, then inverse-transformed two at a time.
// grid = (rows*2 / PP, 2 moduli, nq*slices), 256 threads, dynamic smem = PP*2048*4 + 2*NTT_SMEM_WORDS*4
template <int PP>
__global__ void __launch_bounds__(256)
k_intt_from_zmajor_tiled(DevParams P, ImmaGeom F, const uint32_t* __restrict__ in_zm, size_t in_stride,
                         uint32_t* __restrict__ out, int slices) {
  extern __shared__ __align__(16) uint32_t tsm[];
  uint32_t* polybuf = tsm;                               // [PP][2048]
  uint32_t* sm0 = tsm + PP * POLY;
  uint32_t* sm1 = sm0 + NTT_SMEM_WORDS;
  const int tid = threadIdx.x, n = blockIdx.y;
  const int p0 = blockIdx.x * PP;                        // index into the flattened [row][ct_row] axis
  const int qs = blockIdx.z, qi = qs / slices, slice = qs % slices;
  const uint32_t q = n ? P.q[1] : P.q[0];
  const size_t zstride = (size_t)F.rows * 2;
  const uint32_t* src = in_zm + (size_t)qi * in_stride + (((size_t)slice * 2 + n) * POLY) * zstride + p0;
  for (int z = tid; z < POLY; z += 256) {
    uint32_t v[PP];
    const uint32_t* s = src + (size_t)z * zstride;
    if (PP == 8) {
      uint4 a = __ldg(reinterpret_cast<const uint4*>(s)), b = __ldg(reinterpret_cast<const uint4*>(s) + 1);
      v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4 % PP] = b.x; v[5 % PP] = b.y; v[6 % PP] = b.z; v[7 % PP] = b.w;
    } else if (PP == 4) {
      uint4 a = __ldg(reinterpret_cast<const uint4*>(s));
      v[0] = a.x; v[1] = a.y; v[2 % PP] = a.z; v[3 % PP] = a.w;
    } else {
      uint2 a = __ldg(reinterpret_cast<const uint2*>(s));
      v[0] = a.x; v[1] = a.y;
    }
#pragma unroll
    for (int p = 0; p < PP; p++) polybuf[p * POLY + z] = v[p];
  }
  __syncthreads();
  const TwConstI lo{n, 2};                               // relaxed-range inverse (ntt_core.cuh "lz"): inputs are canonical residues
  const TwGlobalI hi{n ? P.inv_lz[1] : P.inv_lz[0]};
#pragma unroll 1
  for (int p = 0; p < PP; p += 2) {
    uint32_t x0[8], x1[8];
#pragma unroll
    for (int k = 0; k < 8; k++) {
      x0[k] = polybuf[p * POLY + tid * 8 + k];
      x1[k] = polybuf[(p + 1) * POLY + tid * 8 + k];
    }
    ntt_inverse_group2_nh(tid, x0, x1, sm0, sm1, lo, hi, q, SyncI());
    const int f0 = p0 + p, f1 = p0 + p + 1;               // flattened (row, ct_row)
    uint32_t* d0 = out + ((((size_t)qs * F.rows + (f0 >> 1)) * 2 + (f0 & 1)) * 2 + n) * POLY;
    uint32_t* d1 = out + ((((size_t)qs * F.rows + (f1 >> 1)) * 2 + (f1 & 1)) * 2 + n) * POLY;
#pragma unroll
    for (int a = 0; a < 8; a++) {
      d0[a * 256 + tid] = x0[a];
      d1[a * 256 + tid] = x1[a];
    }
  }
}

// z-major product -> the ABI's [ii][r][n][z] NTT-form layout (stage-level entry point only)
__global__ void k_zmajor_to_ntt32(ImmaGeom F, const uint32_t* __restrict__ in_zm, uint32_t* __restrict__ out, int slice) {
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;      // over rows*4*2048, z fastest
  if (idx >= (size_t)F.rows * 4 * POLY) return;
  int z = (int)(idx % POLY);
  int n = (int)((idx / POLY) & 1), r = (int)((idx / (2 * POLY)) & 1);
  int ii = (int)(idx / (4 * POLY));
  out[idx] = in_zm[((((size_t)slice * 2 + n) * POLY + z) * F.rows + ii) * 2 + r];
}

inline unsigned grid1d(size_t total, int block) { return (unsigned)((total + block - 1) / block); }

}  // namespace

void upload_imma_constants(const Twiddle* lo) {
  B200_CUDA(cudaMemcpyToSymbol(c_tw_lo_imma, lo, sizeof(Twiddle) * 2 * 3 * 64));
}
size_t imma_db_cells(const ImmaGeom& F, int slices) {
  return (size_t)slices * 2 * POLY * F.mt * F.ks * 4 * 32;
}
size_t imma_query_cells(const ImmaGeom& F) { return (size_t)2 * POLY * 4 * F.ks * 4 * 32; }   // up to 4 column tiles
// 16 queries per pass need the B operand (4 tiles) plus the A rings in one CTA's shared memory
bool imma_supports_16(const ImmaGeom& F) {
  return (size_t)4 * F.ks * 128 * sizeof(uint2) + (size_t)8 * IMMA_STAGES16 * 128 * sizeof(uint4) <= 224 * 1024;
}

void launch_db_to_frag(const ImmaGeom& F, const uint4* db0_slice, uint4* dbf, int slice, cudaStream_t s) {
  size_t warps = (size_t)POLY * F.mt * F.ks;
  ++g_kernel_launches;
  k_db_to_frag<<<grid1d(warps * 32, 256), 256, 0, s>>>(F, db0_slice, dbf, slice);
}
void launch_db_upsert_frag(const ImmaGeom& F, uint4* dbf, int slice, int il, int j, const uint64_t* poly, cudaStream_t s) {
  ++g_kernel_launches;
  k_db_upsert_frag<<<POLY / 256, 256, 0, s>>>(FragStore{F, dbf}, slice, il, j, poly);
}
void launch_write_items(const DevParams& P, const ImmaGeom& F, uint4* dbf, int slices, const ItemWrite* items, int count,
                        const uint8_t* data, int bpc, uint64_t pt_modulus, cudaStream_t s) {
  item_write::launch(P, FragStore{F, dbf}, items, count, slices, data, bpc, pt_modulus, s);
}
void launch_query_to_frag(const ImmaGeom& F, const uint4* q_dev, size_t q_stride, int nq, uint2* qf, cudaStream_t s) {
  const int ntiles = imma_query_tiles(nq);
  size_t warps = (size_t)POLY * ntiles * F.ks;
  ++g_kernel_launches;
  k_query_to_frag<<<grid1d(warps * 32, 256), 256, 0, s>>>(F, q_dev, q_stride, nq, ntiles, qf);
}
void launch_multiply_imma(const DevParams& P, const ImmaGeom& F, const uint4* dbf, const uint2* qf, uint32_t* out_zm,
                          size_t out_stride, int nq, int slice_begin, int slice_count, int variant, cudaStream_t s) {
  if (nq < 1 || nq > 16) throw Error(-2, "imma multiply: 1..16 queries per pass");
  const int ntiles = imma_query_tiles(nq);
  const size_t smem = (size_t)ntiles * F.ks * 128 * sizeof(uint2);
  const size_t smem8 = smem + (size_t)8 * IMMA_STAGES * 128 * sizeof(uint4);
  const size_t smem16 = smem + (size_t)8 * IMMA_STAGES16 * 128 * sizeof(uint4);
  opt_in_smem(k_multiply_imma<1>, 96 * 1024);
  opt_in_smem(k_multiply_imma<2>, 96 * 1024);
  opt_in_smem((k_multiply_imma8<2, IMMA_STAGES>), 112 * 1024);
  opt_in_smem((k_multiply_imma8<4, IMMA_STAGES16>), 224 * 1024);
  ++g_kernel_launches;
  if (ntiles == 4) {
    if (smem16 > 224 * 1024) throw Error(-2, "imma multiply: dim0 too large for 16 queries per pass");
    k_multiply_imma8<4, IMMA_STAGES16><<<dim3(POLY, 2), 256, smem16, s>>>(P, F, dbf, qf, out_zm, out_stride, nq, slice_begin,
                                                                        slice_count);
    return;
  }
  if (smem > 96 * 1024) throw Error(-2, "imma multiply: dim0 too large");
  if (ntiles == 2 && variant == 0 && smem8 <= 112 * 1024)
    k_multiply_imma8<2, IMMA_STAGES><<<dim3(POLY, 2), 256, smem8, s>>>(P, F, dbf, qf, out_zm, out_stride, nq, slice_begin,
                                                                       slice_count);
  else if (ntiles == 1)
    k_multiply_imma<1><<<dim3(POLY, 2), 256, smem, s>>>(P, F, dbf, qf, out_zm, out_stride, nq, slice_begin, slice_count);
  else
    k_multiply_imma<2><<<dim3(POLY, 2), 256, smem, s>>>(P, F, dbf, qf, out_zm, out_stride, nq, slice_begin, slice_count);
}
template <int PP>
static void launch_intt_tiled(const DevParams& P, const ImmaGeom& F, const uint32_t* in_zm, size_t in_stride, uint32_t* out,
                              int nq, int slices, cudaStream_t s) {
  const size_t smem = (size_t)(PP * POLY + 2 * NTT_SMEM_WORDS) * 4;
  opt_in_smem(k_intt_from_zmajor_tiled<PP>, (int)smem);
  k_intt_from_zmajor_tiled<PP><<<dim3(F.rows * 2 / PP, 2, nq * slices), 256, smem, s>>>(P, F, in_zm, in_stride, out, slices);
}
void launch_intt_from_zmajor(const DevParams& P, const ImmaGeom& F, const uint32_t* in_zm, size_t in_stride, uint32_t* out,
                             int nq, int slices, int variant, cudaStream_t s) {
  ++g_kernel_launches;
  const int polys = F.rows * 2;
  if (variant == 1)
    k_intt_from_zmajor<<<dim3(F.rows * 2, 2, nq * slices), 256, 0, s>>>(P, F, in_zm, in_stride, out, slices);
  else if (polys % 8 == 0) launch_intt_tiled<8>(P, F, in_zm, in_stride, out, nq, slices, s);
  else if (polys % 4 == 0) launch_intt_tiled<4>(P, F, in_zm, in_stride, out, nq, slices, s);
  else launch_intt_tiled<2>(P, F, in_zm, in_stride, out, nq, slices, s);
}
void launch_zmajor_to_ntt32(const ImmaGeom& F, const uint32_t* in_zm, uint32_t* out, int slice, cudaStream_t s) {
  size_t total = (size_t)F.rows * 4 * POLY;
  ++g_kernel_launches;
  k_zmajor_to_ntt32<<<grid1d(total, 256), 256, 0, s>>>(F, in_zm, out, slice);
}

}  // namespace b200pir
