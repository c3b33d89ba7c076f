// First-dimension kernels: multiply_reg_by_database (lib/spiral-rs/src/server.rs:155-221) over an
// HBM-resident database, the database loaders that produce its device layout, and DoublePIR's packed
// matvec (lib/doublepir/src/matrix/kernels.rs:14-178).  All of these are pure streams of the
// database: 8 bytes read -> 4 (u32 x u32 -> u64) multiply-adds, so the design goal is coalesced
// 16-byte loads, many of them in flight per SM, and no shared-memory or shuffle traffic at all.
//
// Device layout of one slice (re-tiled at upload; the C ABI accepts the reference layout
// [z][ii][j], server.rs:263-266):
//     db_dev[ii][jp][z] = uint4{ w(j=2jp).lo, w(2jp).hi, w(2jp+1).lo, w(2jp+1).hi }      (lo = mod q0, hi = mod q1)
// so thread z of a warp reads 16 contiguous bytes and the warp 512 contiguous bytes.  The NTT
// coordinate z is the one fully independent axis of the product, so it is the thread axis: each
// thread owns one z, R database rows and all j, and keeps its 4R (x NQ queries) 64-bit partial sums
// in registers.  Products are < 2^56, so the sums are reduced mod q_n every 256 terms (the reference
// accumulates in u128 and reduces once; both give the canonical residue).
#include "kernels.h"
#include "item_write.cuh"
#include <algorithm>

namespace b200pir {

namespace {

__constant__ Twiddle c_tw_lo_mul[2][3][64];
struct TwConstM {
  int n, dir;
  __device__ __forceinline__ Twiddle operator()(int i) const { return c_tw_lo_mul[n][dir][i]; }
  __device__ __forceinline__ void load2(int i, Twiddle (&t)[2]) const { t[0] = (*this)(i); t[1] = (*this)(i + 1); }
  __device__ __forceinline__ void load4(int i, Twiddle (&t)[4]) const {
    t[0] = (*this)(i); t[1] = (*this)(i + 1); t[2] = (*this)(i + 2); t[3] = (*this)(i + 3);
  }
};
struct TwGlobalM {
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

template <int R, int NQ, int UNROLL>
__global__ void __launch_bounds__(512)
k_multiply(DevParams P, MulGeom G, const uint4* __restrict__ db, const uint4* __restrict__ qv, uint32_t* __restrict__ out,
           int slice_begin, size_t q_stride, size_t out_stride) {
  const int z = blockIdx.x * blockDim.x + threadIdx.x;
  const int rowgroup = blockIdx.y * blockDim.y + threadIdx.y;
  const int ii0 = rowgroup * R;
  const int slice = slice_begin + blockIdx.z;
  if (ii0 >= G.num_per) return;
  const int half = G.dim0 >> 1;
  const size_t row_stride = (size_t)half * POLY;
  const uint4* dbp = db + ((size_t)slice * G.num_per + ii0) * row_stride + z;
  const uint4* qp = qv + z;

  uint64_t acc[NQ][R][4];
#pragma unroll
  for (int a = 0; a < NQ; a++)
#pragma unroll
    for (int r = 0; r < R; r++)
#pragma unroll
      for (int c = 0; c < 4; c++) acc[a][r][c] = 0;

  for (int jp0 = 0; jp0 < half; jp0 += 128) {
    const int jend = min(jp0 + 128, half);
#pragma unroll UNROLL
    for (int jp = jp0; jp < jend; jp++) {
      uint4 d[R];
#pragma unroll
      for (int r = 0; r < R; r++) d[r] = ld_stream_v4(dbp + (size_t)r * row_stride + (size_t)jp * POLY);
#pragma unroll
      for (int a = 0; a < NQ; a++) {
        const uint4 qa = __ldg(qp + (size_t)a * q_stride + (size_t)(2 * jp) * POLY);
        const uint4 qb = __ldg(qp + (size_t)a * q_stride + (size_t)(2 * jp + 1) * POLY);
#pragma unroll
        for (int r = 0; r < R; r++) {
          acc[a][r][0] += (uint64_t)d[r].x * qa.x;     // n0, row 0 of the ciphertext
          acc[a][r][1] += (uint64_t)d[r].x * qa.z;     // n0, row 1
          acc[a][r][2] += (uint64_t)d[r].y * qa.y;     // n1, row 0
          acc[a][r][3] += (uint64_t)d[r].y * qa.w;     // n1, row 1
          acc[a][r][0] += (uint64_t)d[r].z * qb.x;
          acc[a][r][1] += (uint64_t)d[r].z * qb.z;
          acc[a][r][2] += (uint64_t)d[r].w * qb.y;
          acc[a][r][3] += (uint64_t)d[r].w * qb.w;
        }
      }
    }
    if (jend < half) {       // 256 products per accumulator so far: fold back below 2^28
#pragma unroll
      for (int a = 0; a < NQ; a++)
#pragma unroll
        for (int r = 0; r < R; r++) {
          acc[a][r][0] = barrett64(acc[a][r][0], P.cr1[0], P.q[0]);
          acc[a][r][1] = barrett64(acc[a][r][1], P.cr1[0], P.q[0]);
          acc[a][r][2] = barrett64(acc[a][r][2], P.cr1[1], P.q[1]);
          acc[a][r][3] = barrett64(acc[a][r][3], P.cr1[1], P.q[1]);
        }
    }
  }
  // out[ii].data[r*2N + n*N + z]   (server.rs:204-217)
#pragma unroll
  for (int a = 0; a < NQ; a++)
#pragma unroll
    for (int r = 0; r < R; r++) {
      uint32_t* o = out + (size_t)a * out_stride + ((size_t)slice * G.num_per + ii0 + r) * 4 * POLY + z;
      o[0 * POLY] = barrett64(acc[a][r][0], P.cr1[0], P.q[0]);      // row 0, n0
      o[1 * POLY] = barrett64(acc[a][r][2], P.cr1[1], P.q[1]);      // row 0, n1
      o[2 * POLY] = barrett64(acc[a][r][1], P.cr1[0], P.q[0]);      // row 1, n0
      o[3 * POLY] = barrett64(acc[a][r][3], P.cr1[1], P.q[1]);      // row 1, n1
    }
}

template <int R, int NQ, int UNROLL>
void launch_mul_t(const DevParams& P, const MulGeom& G, const uint4* db, const uint4* q, uint32_t* out, int slice_begin,
                  int slice_count, size_t q_stride, size_t out_stride, int groups, cudaStream_t s) {
  int rowgroups = G.num_per / R;
  if (rowgroups * R != G.num_per) throw Error(-2, "multiply: num_per must be a multiple of the row tile");
  if (groups > rowgroups) groups = rowgroups;
  while (rowgroups % groups) groups--;
  dim3 block(128, groups);
  dim3 grid(POLY / 128, rowgroups / groups, slice_count);
  ++g_kernel_launches;
  k_multiply<R, NQ, UNROLL><<<grid, block, 0, s>>>(P, G, db, q, out, slice_begin, q_stride, out_stride);
}

__global__ void k_query_to_dev(MulGeom G, uint4* q_dev, const uint64_t* v) {
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;     // over dim0 * 2048, z fastest
  if (idx >= (size_t)G.dim0 * POLY) return;
  int z = (int)(idx % POLY), j = (int)(idx / POLY);
  const uint64_t* src = v + ((size_t)z * G.dim0 + j) * 2;
  uint64_t a0 = src[0], a1 = src[1];
  q_dev[((size_t)(j >> 1) * 2 + (j & 1)) * POLY + z] =
      make_uint4((uint32_t)a0, (uint32_t)(a0 >> 32), (uint32_t)a1, (uint32_t)(a1 >> 32));
}

// ref: u64 [zc][num_per_global][dim0] for z in [z0, z0+zc)  ->  db_dev slice [il][jp][z], ii = il*count + index
__global__ void k_db_retile(MulGeom G, Shard sh, uint4* db_slice, const uint64_t* ref, int z0, int zc) {
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;     // over num_per * half * zc, z fastest
  const int half = G.dim0 >> 1;
  size_t total = (size_t)G.num_per * half * zc;
  if (idx >= total) return;
  int zl = (int)(idx % zc);
  size_t rest = idx / zc;
  int jp = (int)(rest % half), ii = (int)(rest / half);
  const size_t ii_global = (size_t)ii * sh.count + sh.index;
  const uint64_t* src = ref + ((size_t)zl * G.num_per * sh.count + ii_global) * G.dim0 + 2 * jp;
  uint64_t w0 = src[0], w1 = src[1];
  db_slice[((size_t)ii * half + jp) * POLY + z0 + zl] =
      make_uint4((uint32_t)w0, (uint32_t)(w0 >> 32), (uint32_t)w1, (uint32_t)(w1 >> 32));
}

// where word z of item (slice, local row il, j) lives in the IMAD layout; w = lo | hi << 32
struct ImadStore {
  MulGeom G;
  uint4* db;
  __device__ __forceinline__ void operator()(int slice, int il, int j, int z, uint64_t w) const {
    const int half = G.dim0 >> 1;
    uint2* cell = reinterpret_cast<uint2*>(db + (((size_t)slice * G.num_per + il) * half + (j >> 1)) * POLY + z) + (j & 1);
    *cell = make_uint2((uint32_t)w, (uint32_t)(w >> 32));
  }
};

__global__ void k_db_upsert(ImadStore st, int slice, int il, int j, const uint64_t* poly) {
  int z = blockIdx.x * blockDim.x + threadIdx.x;
  if (z >= POLY) return;
  st(slice, il, j, z, poly[z]);
}

__device__ __forceinline__ uint64_t splitmix64_at(uint64_t seed, uint64_t index) {
  uint64_t z = seed + (index + 1) * 0x9E3779B97F4A7C15ULL;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
  return z ^ (z >> 31);
}

// CTA (512 threads) = one (slice, ii, jp) cell pair: builds the two items j = 2jp, 2jp+1 from their
// plaintext (server.rs:245-270: uniform mod p, recenter_mod, NTT, pack) and writes 2048 uint4.
__global__ void __launch_bounds__(512, 1)
k_db_synth(DevParams P, MulGeom G, Shard sh, uint4* db, uint64_t seed, uint64_t pt, int slice_begin) {
  extern __shared__ __align__(16) uint32_t synth_smem[];
  uint32_t* ntt_smem = synth_smem;                       // 2 * NTT_SMEM_WORDS
  uint32_t* cell = synth_smem + 2 * NTT_SMEM_WORDS;      // POLY * 4
  const int n = threadIdx.x >> 8, tid = threadIdx.x & 255;
  const int half = G.dim0 >> 1;
  const int jp = blockIdx.x % half;
  const int ii = (blockIdx.x / half) % G.num_per;                 // local row
  const int slice = slice_begin + blockIdx.x / (half * G.num_per);
  const uint32_t q = n ? P.q[1] : P.q[0];
  const uint64_t num_per_global = (uint64_t)G.num_per * sh.count;
  const uint64_t num_items = (uint64_t)G.dim0 * num_per_global;
  struct S { __device__ __forceinline__ void operator()() const { __syncthreads(); } };
#pragma unroll 1
  for (int jb = 0; jb < 2; jb++) {
    const uint64_t item = (uint64_t)(2 * jp + jb) * num_per_global + ((uint64_t)ii * sh.count + sh.index);
    const uint64_t base = ((uint64_t)slice * num_items + item) * POLY;
    uint32_t x[8];
#pragma unroll
    for (int a = 0; a < 8; a++) {
      uint64_t v = splitmix64_at(seed, base + a * 256 + tid) % pt;
      x[a] = (v > pt / 2) ? (uint32_t)(q - (uint32_t)(pt - v)) : (uint32_t)v;     // recenter_mod, then mod q_n
    }
    ntt_forward_group_lz<NTT_OUT_CANON>(tid, x, ntt_smem + n * NTT_SMEM_WORDS, TwConstM{n, 0}, TwGlobalM{n ? P.fwd[1] : P.fwd[0]}, q, S());   // inputs canonical
#pragma unroll
    for (int k = 0; k < 8; k++) cell[(tid * 8 + k) * 4 + jb * 2 + n] = x[k];
  }
  __syncthreads();
  uint4* dst = db + (((size_t)slice * G.num_per + ii) * half + jp) * POLY;
  const uint4* c4 = reinterpret_cast<const uint4*>(cell);
  for (int z = threadIdx.x; z < POLY; z += 512) dst[z] = c4[z];
}

// ------------------------------------------------------------------ DoublePIR
// out[i] = sum_k sum_{m<3} ((a[i][k] >> 10m) & 1023) * b[3k+m]   (wrapping u32; kernels.rs:52-93)
// One warp per ROWS rows; lanes stride over k.  b is staged in shared memory as three planes
// bm[m][k] so that a lane's two consecutive k read one conflict-free 8-byte word per plane.
template <int ROWS>
__global__ void __launch_bounds__(256)
k_dpir_matvec(uint32_t* __restrict__ out, const uint32_t* __restrict__ a, const uint32_t* __restrict__ b, size_t rows,
              size_t cols, size_t cols_pad) {
  extern __shared__ __align__(16) uint32_t bsm[];          // [3][cols_pad]
  for (size_t k = threadIdx.x; k < cols; k += blockDim.x) {
    bsm[k] = b[3 * k];
    bsm[cols_pad + k] = b[3 * k + 1];
    bsm[2 * cols_pad + k] = b[3 * k + 2];
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const bool vec2 = (cols & 1) == 0;
  for (size_t row0 = ((size_t)blockIdx.x * nwarps + warp) * ROWS; row0 < rows; row0 += (size_t)gridDim.x * nwarps * ROWS) {
    uint32_t acc[ROWS];
#pragma unroll
    for (int r = 0; r < ROWS; r++) acc[r] = 0;
    if (vec2) {
      for (size_t k = 2 * (size_t)lane; k < cols; k += 64) {
        uint2 b0 = *reinterpret_cast<const uint2*>(bsm + k);
        uint2 b1 = *reinterpret_cast<const uint2*>(bsm + cols_pad + k);
        uint2 b2 = *reinterpret_cast<const uint2*>(bsm + 2 * cols_pad + k);
#pragma unroll
        for (int r = 0; r < ROWS; r++) {
          if (row0 + r < rows) {
            uint2 d;
            asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];"
                         : "=r"(d.x), "=r"(d.y) : "l"(a + (row0 + r) * cols + k));
            acc[r] += (d.x & 1023u) * b0.x + ((d.x >> 10) & 1023u) * b1.x + ((d.x >> 20) & 1023u) * b2.x;
            acc[r] += (d.y & 1023u) * b0.y + ((d.y >> 10) & 1023u) * b1.y + ((d.y >> 20) & 1023u) * b2.y;
          }
        }
      }
    } else {
      for (size_t k = lane; k < cols; k += 32) {
        uint32_t b0 = bsm[k], b1 = bsm[cols_pad + k], b2 = bsm[2 * cols_pad + k];
#pragma unroll
        for (int r = 0; r < ROWS; r++) {
          if (row0 + r < rows) {
            uint32_t d = __ldg(a + (row0 + r) * cols + k);
            acc[r] += (d & 1023u) * b0 + ((d >> 10) & 1023u) * b1 + ((d >> 20) & 1023u) * b2;
          }
        }
      }
    }
#pragma unroll
    for (int r = 0; r < ROWS; r++) {
      uint32_t v = acc[r];
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
      if (lane == 0 && row0 + r < rows) out[row0 + r] = v;
    }
  }
}

// One row per warp; every lane keeps U independent 8-byte streaming loads in flight before it consumes them.
template <int U>
__global__ void __launch_bounds__(256)
k_dpir_matvec_row(uint32_t* __restrict__ out, const uint32_t* __restrict__ a, const uint32_t* __restrict__ b, size_t rows,
                  size_t cols, size_t cols_pad) {
  extern __shared__ __align__(16) uint32_t bsm[];          // [3][cols_pad]
  for (size_t k = threadIdx.x; k < cols_pad; k += blockDim.x) {
    bool in = k < cols;
    bsm[k] = in ? b[3 * k] : 0u;
    bsm[cols_pad + k] = in ? b[3 * k + 1] : 0u;
    bsm[2 * cols_pad + k] = in ? b[3 * k + 2] : 0u;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const size_t pairs = cols >> 1;                           // cols is even on this path
  for (size_t row = (size_t)blockIdx.x * nwarps + warp; row < rows; row += (size_t)gridDim.x * nwarps) {
    const uint2* ar = reinterpret_cast<const uint2*>(a + row * cols);
    uint32_t acc = 0;
    for (size_t p0 = 0; p0 < pairs; p0 += 32 * U) {
      uint2 d[U];
#pragma unroll
      for (int u = 0; u < U; u++) {
        size_t p = p0 + (size_t)u * 32 + lane;
        d[u] = make_uint2(0u, 0u);
        if (p < pairs)
          asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(d[u].x), "=r"(d[u].y) : "l"(ar + p));
      }
#pragma unroll
      for (int u = 0; u < U; u++) {
        size_t p = p0 + (size_t)u * 32 + lane;
        if (p < pairs) {
          uint2 b0 = *reinterpret_cast<const uint2*>(bsm + 2 * p);
          uint2 b1 = *reinterpret_cast<const uint2*>(bsm + cols_pad + 2 * p);
          uint2 b2 = *reinterpret_cast<const uint2*>(bsm + 2 * cols_pad + 2 * p);
          acc += (d[u].x & 1023u) * b0.x + ((d[u].x >> 10) & 1023u) * b1.x + ((d[u].x >> 20) & 1023u) * b2.x;
          acc += (d[u].y & 1023u) * b0.y + ((d[u].y >> 10) & 1023u) * b1.y + ((d[u].y >> 20) & 1023u) * b2.y;
        }
      }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if (lane == 0) out[row] = acc;
  }
}

// Rows too wide for `b` to fit in shared memory (3 * cols words > 200 KiB; the reference's short-and-wide databases, e.g.
// l = 29, m = 65536 for 2^24 one-bit entries, doublepir.rs:471-483): one CTA per row, `b` read through L2.
__global__ void __launch_bounds__(256)
k_dpir_matvec_wide(uint32_t* __restrict__ out, const uint32_t* __restrict__ a, const uint32_t* __restrict__ b, size_t rows,
                   size_t cols) {
  __shared__ uint32_t part[8];
  const size_t row = blockIdx.x;
  if (row >= rows) return;
  const uint32_t* ar = a + row * cols;
  uint32_t acc = 0;
  for (size_t k = threadIdx.x; k < cols; k += blockDim.x) {
    const uint32_t d = __ldg(ar + k);
    const uint32_t* bp = b + 3 * k;
    acc += (d & 1023u) * __ldg(bp) + ((d >> 10) & 1023u) * __ldg(bp + 1) + ((d >> 20) & 1023u) * __ldg(bp + 2);
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t t = 0;
    for (int w = 0; w < 8; w++) t += part[w];
    out[row] = t;
  }
}

// kernels.rs:180-278: out[i][j] = sum_k sum_m ((a[i][k] >> 10m) & 1023) * b[j][3k+m]   (one warp per output)
__global__ void k_dpir_mul_transposed(uint32_t* __restrict__ out, const uint32_t* __restrict__ a, const uint32_t* __restrict__ b,
                                      size_t a_rows, size_t a_cols, size_t b_rows, size_t b_cols) {
  const size_t warp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= a_rows * b_rows) return;
  const size_t i = warp / b_rows, j = warp % b_rows;
  uint32_t acc = 0;
  for (size_t k = lane; k < a_cols; k += 32) {
    uint32_t d = __ldg(a + i * a_cols + k);
    const uint32_t* bp = b + j * b_cols + 3 * k;
    acc += (d & 1023u) * __ldg(bp) + ((d >> 10) & 1023u) * __ldg(bp + 1) + ((d >> 20) & 1023u) * __ldg(bp + 2);
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
  if (lane == 0) out[i * b_rows + j] = acc;
}
// matrix/indexing.rs:117-143 (basis 10, d 3): one thread per output word
__global__ void k_dpir_transpose_expand(uint32_t* __restrict__ out, const uint32_t* __restrict__ a, size_t rows, size_t cols,
                                        uint64_t modulus, size_t delta, size_t concat, size_t out_rows, size_t out_cols) {
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= out_rows * out_cols) return;
  const size_t r = idx / out_cols, cd = idx % out_cols;
  const size_t jmod = r / (cols * delta), rem = r % (cols * delta), i = rem / delta, f = rem % delta;
  uint32_t acc = 0;
  for (size_t cc = 0; cc < 3; cc++) {
    const size_t c = cd * 3 + cc, j = c * concat + jmod;
    if (j < rows) {
      uint64_t val = a[i + j * cols];
      for (size_t t = 0; t < f; t++) val /= modulus;
      acc += (uint32_t)((val % modulus) << (10 * cc));
    }
  }
  out[idx] = acc;
}

inline unsigned grid1d(size_t total, int block) { return (unsigned)((total + block - 1) / block); }

}  // namespace

void launch_dpir_mul_transposed(uint32_t* out, const uint32_t* a, const uint32_t* b, size_t a_rows, size_t a_cols,
                                size_t b_rows, size_t b_cols, cudaStream_t s) {
  ++g_kernel_launches;
  k_dpir_mul_transposed<<<grid1d(a_rows * b_rows * 32, 256), 256, 0, s>>>(out, a, b, a_rows, a_cols, b_rows, b_cols);
}
void launch_dpir_transpose_expand(uint32_t* out, const uint32_t* a, size_t rows, size_t cols, uint64_t modulus, size_t delta,
                                  size_t concat, size_t out_rows, size_t out_cols, cudaStream_t s) {
  ++g_kernel_launches;
  k_dpir_transpose_expand<<<grid1d(out_rows * out_cols, 256), 256, 0, s>>>(out, a, rows, cols, modulus, delta, concat,
                                                                           out_rows, out_cols);
}
void upload_mul_constants(const Twiddle* lo) {
  B200_CUDA(cudaMemcpyToSymbol(c_tw_lo_mul, lo, sizeof(Twiddle) * 2 * 3 * 64));
}
void launch_multiply(const DevParams& P, const MulGeom& G, const uint4* db_dev, const uint4* q_dev, uint32_t* out,
                     int slice_begin, int slice_count, int nq, size_t q_stride, size_t out_stride, int variant,
                     cudaStream_t s) {
  if (G.dim0 < 2 || (G.dim0 & 1)) throw Error(-2, "multiply: dim0 must be even");
  // row tile: the largest of {8,4,2,1} dividing num_per (num_per is a power of two)
  int R = G.num_per >= 8 ? 8 : G.num_per;
  if (variant == 1 && R == 8) R = 4;
#define MUL_CASE(RR, QQ, UU, GG)                                                                                     \
  launch_mul_t<RR, QQ, UU>(P, G, db_dev, q_dev, out, slice_begin, slice_count, q_stride, out_stride, GG, s)
  if (nq == 1) {
    if (R == 8) { if (variant == 2) MUL_CASE(8, 1, 1, 1); else MUL_CASE(8, 1, 1, 2); }
    else if (R == 4) { if (variant == 3) MUL_CASE(4, 1, 2, 2); else MUL_CASE(4, 1, 2, 4); }
    else if (R == 2) MUL_CASE(2, 1, 2, 2);
    else MUL_CASE(1, 1, 2, 1);
  } else if (nq == 2) {
    if (R >= 4) { if (G.num_per % 4) throw Error(-2, "multiply: bad num_per"); MUL_CASE(4, 2, 1, 2); }
    else if (R == 2) MUL_CASE(2, 2, 1, 2);
    else MUL_CASE(1, 2, 1, 1);
  } else if (nq == 4) {
    if (R >= 2) MUL_CASE(2, 4, 1, 2);
    else MUL_CASE(1, 4, 1, 1);
  } else {
    throw Error(-2, "multiply: nq must be 1, 2 or 4");
  }
#undef MUL_CASE
}
void launch_query_to_dev(const MulGeom& G, uint4* q_dev, const uint64_t* v_firstdim, cudaStream_t s) {
  size_t total = (size_t)G.dim0 * POLY;
  ++g_kernel_launches;
  k_query_to_dev<<<grid1d(total, 256), 256, 0, s>>>(G, q_dev, v_firstdim);
}
void launch_db_retile_chunk(const MulGeom& G, Shard sh, uint4* db_dev_slice, const uint64_t* ref_chunk, int z0, int zc,
                            cudaStream_t s) {
  size_t total = (size_t)G.num_per * (G.dim0 >> 1) * zc;
  ++g_kernel_launches;
  k_db_retile<<<grid1d(total, 256), 256, 0, s>>>(G, sh, db_dev_slice, ref_chunk, z0, zc);
}
void launch_db_upsert(const MulGeom& G, uint4* db_dev, int slice, int il, int j, const uint64_t* poly, cudaStream_t s) {
  ++g_kernel_launches;
  k_db_upsert<<<POLY / 256, 256, 0, s>>>(ImadStore{G, db_dev}, slice, il, j, poly);
}
void launch_write_items(const DevParams& P, const MulGeom& G, uint4* db_dev, int slices, const ItemWrite* items, int count,
                        const uint8_t* data, int bpc, uint64_t pt_modulus, cudaStream_t s) {
  item_write::launch(P, ImadStore{G, db_dev}, items, count, slices, data, bpc, pt_modulus, s);
}
void launch_db_synth(const DevParams& P, const MulGeom& G, Shard sh, uint4* db_dev, uint64_t seed, uint64_t pt_modulus,
                     int slice_begin, int slice_count, cudaStream_t s) {
  size_t ctas = (size_t)slice_count * G.num_per * (G.dim0 >> 1);
  if (ctas == 0) return;
  if (ctas > 0x7fffffffULL) throw Error(-2, "db_synth: grid too large");
  const size_t smem = (size_t)(2 * NTT_SMEM_WORDS + 4 * POLY) * 4;
  opt_in_smem(k_db_synth, (int)smem);
  ++g_kernel_launches;
  k_db_synth<<<(unsigned)ctas, 512, smem, s>>>(P, G, sh, db_dev, seed, pt_modulus, slice_begin);
}
void launch_dpir_matvec(uint32_t* out, const uint32_t* a, const uint32_t* b, size_t rows, size_t cols, int variant,
                        cudaStream_t s) {
  size_t cols_pad = (cols + 3) & ~(size_t)3;
  size_t smem = 3 * cols_pad * 4;
  if (rows == 0) return;
  if (smem > 200 * 1024) {
    if (rows > 0x7FFFFFFFull) throw Error(-2, "dpir: too many rows for the wide-row kernel");
    ++g_kernel_launches;
    k_dpir_matvec_wide<<<(unsigned)rows, 256, 0, s>>>(out, a, b, rows, cols);
    return;
  }
  if ((cols & 1) == 0 && variant != 1 && variant != 4) {
    // default: one row per warp, 8 loads in flight per lane (variant 2: 4 loads)
    unsigned g = (unsigned)std::min<size_t>((rows + 7) / 8, (size_t)148 * 8);
    ++g_kernel_launches;
    if (variant == 2) {
      cudaFuncSetAttribute(k_dpir_matvec_row<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      k_dpir_matvec_row<4><<<g, 256, smem, s>>>(out, a, b, rows, cols, cols_pad);
    } else {
      cudaFuncSetAttribute(k_dpir_matvec_row<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      k_dpir_matvec_row<8><<<g, 256, smem, s>>>(out, a, b, rows, cols, cols_pad);
    }
    return;
  }
  const int rows_per_warp = variant == 1 ? 2 : 4;
  size_t warps_needed = (rows + rows_per_warp - 1) / rows_per_warp;
  unsigned grid = (unsigned)std::min<size_t>((warps_needed + 7) / 8, (size_t)148 * 8);
  if (grid == 0) return;
  if (rows_per_warp == 2) {
    cudaFuncSetAttribute(k_dpir_matvec<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    ++g_kernel_launches;
    k_dpir_matvec<2><<<grid, 256, smem, s>>>(out, a, b, rows, cols, cols_pad);
  } else {
    cudaFuncSetAttribute(k_dpir_matvec<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    ++g_kernel_launches;
    k_dpir_matvec<4><<<grid, 256, smem, s>>>(out, a, b, rows, cols, cols_pad);
  }
}

}  // namespace b200pir
