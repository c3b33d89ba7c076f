// First dimension on the 5th-generation tensor cores (tcgen05.mma kind::i8, accumulators in TMEM) — database format 2.
//
// STATUS: validated on a B200 (raw accumulators match the assumed TMEM layout, parity tests bit-exact against the oracle,
// tests/test_gpu_tcgen05.py); the default database format wherever the geometry is supported.  The arithmetic is the one
// of the mma.sync path (imma_kernels.cu): 28-bit residues as four 7-bit limbs, exact s32 accumulation, recombination with
// powers of 2^7 and one Barrett reduction per output word.
//
// multiply_reg_by_database (lib/spiral-rs/src/server.rs:155-221) for one NTT coordinate z and modulus n is the integer
// GEMM  C[ii][(query,row)] = sum_j A[ii][j] * B[j][(query,row)] mod q_n.  Here both operands carry their limb index as
// part of the GEMM's M / N index, so one UMMA tile produces all 16 limb-pair products separately:
//
//     M index = 4 * row_local + l      (32 database rows x 4 limbs  = 128 = UMMA_M)
//     N index = 4 * col       + m      (32 columns = 16 queries x 2 ciphertext rows, x 4 limbs = 128 = UMMA_N)
//     K       = 32 values of j per instruction (kind::i8), dim0 / 32 instructions per tile
//     D[M][N] = sum_j a_l(ii, j) * b_m(j, col)  < dim0 * 2^14 <= 2^24        (exact in s32)
//
// The epilogue (tc5_layout.cuh) reads a row of D from TMEM (lane = M index), folds the four m-limbs of every column with shifts,
// weights the 47-bit sum with 2^{7l} mod q in two wide multiply-adds, reduce-scatters over the four l-limb lanes of a row
// (two shuffle rounds) and finishes with one 32-bit Barrett per stored word.
//
// Operand images.  Both operands are stored in global memory as exact images of the shared-memory tiles the MMA reads
// (canonical K-major, no swizzle: 8-row x 16-byte core matrices, LBO = 128 B between the two K halves, SBO = 256 B
// between 8-row groups; byte (midx, k) of a tile lives at (midx>>3)*256 + (k>>4)*128 + (midx&7)*16 + (k&15)), so a tile
// moves with ONE 1-D bulk copy (cp.async.bulk ... mbarrier::complete_tx::bytes) and needs no tensor map:
//     dbT[slice][n][z][mt][ks][4096 B]      (mt: 32 rows, ks: 32 values of j)     == 8 bytes per database word, as before
//     qT [n][z][ks][4096 B]                 (16 queries)
// One persistent CTA per SM walks the (n, z) pairs; warp 0 = bulk-copy producer, warp 1 = MMA issuer (one thread),
// warps 2..9 = epilogue (two per TMEM lane quadrant, 64 accumulator columns each: two warps per scheduler hide the latency
// of the TMEM loads, shuffles and wide multiplies).  Pipelines: A ring (full/empty mbarriers), double-buffered B operand
// (bfull/bempty), double-buffered accumulator in TMEM (tfull/tempty).
#include "kernels.h"
#include "item_write.cuh"
#include "tc5_ptx.cuh"
#include <cstdio>
#include <cstdlib>
#include <vector>

namespace b200pir {

namespace {

constexpr int TC5_SMEM_BUDGET = 227 * 1024 - 1024;      // dynamic shared memory of the CTA minus barriers / alignment slack
constexpr int TC5_EPI_WARPS = 8;
constexpr int TC5_THREADS = 64 + 32 * TC5_EPI_WARPS;    // producer warp, MMA warp, epilogue warps
constexpr int TC5_DBG_TILES = 4;

using namespace tc5;

// ---- operand images ---------------------------------------------------------------------------------------------------
// format 0 slice (uint4 [row][jp][z]) -> tile images.  CTA = (z, mt, ks); thread = (row_local, group of 4 values of j).
__global__ void __launch_bounds__(256)
k_db_to_tc5(Tc5Geom T, const uint4* __restrict__ db0_slice, uint8_t* __restrict__ dbt, int slice) {
  const int z = blockIdx.x, mt = blockIdx.y, ks = blockIdx.z;
  const Tc5DbThread t = tc5_db_thread(threadIdx.x, mt, ks);
  const int half = T.dim0 >> 1;
  uint32_t res[2][4];
#pragma unroll
  for (int p = 0; p < 2; p++) {
    const int jp = t.jp0 + p;
    uint4 w = make_uint4(0, 0, 0, 0);
    if (t.ii < T.rows && jp < half) w = db0_slice[((size_t)t.ii * half + jp) * POLY + z];
    res[0][2 * p] = w.x; res[1][2 * p] = w.y; res[0][2 * p + 1] = w.z; res[1][2 * p + 1] = w.w;
  }
#pragma unroll
  for (int n = 0; n < 2; n++) tc5_db_store(dbt + tc5_db_tile(T, slice, n, z, mt, ks) * TC5_TILE, t, res[n]);
}

// where word z of item (slice, local row il, j) lives in the tile images (byte writes); w = lo | hi << 32
struct Tc5Store {
  Tc5Geom T;
  uint8_t* dbt;
  __device__ __forceinline__ void operator()(int slice, int il, int j, int z, uint64_t w) const {
    const int mt = il >> 5, row_local = il & 31, ks = j >> 5, k = j & 31;
#pragma unroll
    for (int n = 0; n < 2; n++) {
      const uint32_t r = n ? (uint32_t)(w >> 32) : (uint32_t)w;
      uint8_t* tile = dbt + tc5_db_tile(T, slice, n, z, mt, ks) * TC5_TILE;
#pragma unroll
      for (int l = 0; l < 4; l++) tile[tc5_tile_off(tc5_m_index(row_local, l), k)] = (uint8_t)((r >> (7 * l)) & 127u);
    }
  }
};

// one item polynomial (2048 packed words lo|hi<<32) into the tile images
__global__ void k_db_upsert_tc5(Tc5Store st, int slice, int il, int j, const uint64_t* poly) {
  const int z = blockIdx.x * blockDim.x + threadIdx.x;
  if (z >= POLY) return;
  st(slice, il, j, z, poly[z]);
}

// expanded queries (uint4 [j][z] per query, q_stride apart) -> qT.  CTA = (pair of z, ks): every 32-byte sector it reads is
// fully used; the four 4 KiB tiles (2 z x 2 n) are assembled in shared memory and written out contiguously.
__global__ void __launch_bounds__(256)
k_query_to_tc5(Tc5Geom T, const uint4* __restrict__ q_dev, size_t q_stride, int nq, uint8_t* __restrict__ qt) {
  __shared__ __align__(16) uint8_t img[2][2][TC5_TILE];          // [z parity][n]
  const int z0 = blockIdx.x * 2, ks = blockIdx.y;
  for (int i = threadIdx.x; i < 2 * 2 * TC5_TILE / 16; i += blockDim.x) reinterpret_cast<uint4*>(&img[0][0][0])[i] = make_uint4(0, 0, 0, 0);
  __syncthreads();
  // 16 queries x 32 values of j x 2 z = 1024 cells, 4 per thread; consecutive threads take consecutive z, then j, then query
  for (int cell = threadIdx.x; cell < 16 * 32 * 2; cell += blockDim.x) {
    const Tc5QueryCell qc = tc5_query_cell(cell);
    const int j = ks * 32 + qc.k;
    if (qc.q < nq && j < T.dim0) {
      const uint4 w = q_dev[(size_t)qc.q * q_stride + (size_t)j * POLY + z0 + qc.zp];
#pragma unroll
      for (int r = 0; r < 2; r++)
#pragma unroll
        for (int n = 0; n < 2; n++) tc5_query_store(img[qc.zp][n], qc.q, r, qc.k, r ? (n ? w.w : w.z) : (n ? w.y : w.x));
    }
  }
  __syncthreads();
#pragma unroll
  for (int zp = 0; zp < 2; zp++)
#pragma unroll
    for (int n = 0; n < 2; n++) {
      uint4* dst = reinterpret_cast<uint4*>(qt + tc5_q_tile(T, n, z0 + zp, ks) * TC5_TILE);
      dst[threadIdx.x] = reinterpret_cast<const uint4*>(&img[zp][n][0])[threadIdx.x];
    }
}

// The same images straight from the expansion workspace (reorient_reg_ciphertexts, util.rs:323-355, fused with the re-tiling):
// v = ntt32 [query][slot][ct row][n][z] (v_stride words per query), first-dimension ciphertext j = slot idx_factor * j.
// CTA = (8 consecutive z, ks): 2048 polynomial segments of 8 words (one 32-byte sector each), 8 per thread; the sixteen 4 KiB
// tiles (8 z x 2 n) are assembled in shared memory and written out contiguously.
__global__ void __launch_bounds__(256)
k_reorient_to_tc5(Tc5Geom T, const uint32_t* __restrict__ v, size_t v_stride, int idx_factor, int nq, uint8_t* __restrict__ qt) {
  extern __shared__ __align__(16) uint8_t rimg[];                    // [8 z][2 n][TC5_TILE]
  const int z0 = blockIdx.x * 8, ks = blockIdx.y;
  for (int i = threadIdx.x; i < 16 * TC5_TILE / 16; i += 256) reinterpret_cast<uint4*>(rimg)[i] = make_uint4(0, 0, 0, 0);
  __syncthreads();
  for (int seg = threadIdx.x; seg < 16 * 32 * 4; seg += 256) {
    const int n = seg & 1, r = (seg >> 1) & 1, k = (seg >> 2) & 31, q = seg >> 7;
    const int j = ks * 32 + k;
    if (q >= nq || j >= T.dim0) continue;
    const uint32_t* src = v + (size_t)q * v_stride + ((size_t)idx_factor * j * 4 + r * 2 + n) * 2048 + z0;
    const uint4 a = __ldg(reinterpret_cast<const uint4*>(src)), b = __ldg(reinterpret_cast<const uint4*>(src) + 1);
    const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
    for (int zz = 0; zz < 8; zz++) tc5_query_store(rimg + ((size_t)zz * 2 + n) * TC5_TILE, q, r, k, w[zz]);
  }
  __syncthreads();
#pragma unroll
  for (int zz = 0; zz < 8; zz++)
#pragma unroll
    for (int n = 0; n < 2; n++) {
      uint4* dst = reinterpret_cast<uint4*>(qt + tc5_q_tile(T, n, z0 + zz, ks) * TC5_TILE);
      dst[threadIdx.x] = reinterpret_cast<const uint4*>(rimg + ((size_t)zz * 2 + n) * TC5_TILE)[threadIdx.x];
    }
}

// ---- the multiply -----------------------------------------------------------------------------------------------------
constexpr int TC5_MAX_STAGES = 24;
struct Tc5Smem {
  uint64_t full[TC5_MAX_STAGES], empty[TC5_MAX_STAGES];
  uint64_t bfull[2], bempty[2];
  uint64_t tfull[4], tempty[4];
  uint32_t tmem_base;
};
// ring stages that fit beside the query operand: the bytes in flight per SM bound the HBM bandwidth the kernel can pull
// (latency x bandwidth = about 90 KiB per SM at 6.5 TB/s and 2 us), and a stage is out of flight while its MMAs run
__host__ __device__ inline int tc5_ring_stages(int ks, int ksps, int bbufs) {
  const int n = (TC5_SMEM_BUDGET - bbufs * ks * TC5_TILE) / (ksps * TC5_TILE);
  return n > TC5_MAX_STAGES ? TC5_MAX_STAGES : n;
}

// out_zm[query][slice][n][z][row][ct_row] (u32), the format of k_multiply_imma
// KSPS = k-steps (4 KiB tiles) per ring stage.  dbg_mode (bring-up / bottleneck analysis only, B200PIR_TC5_DBG): bit 0 = the MMA
// thread releases every stage without issuing MMAs, bit 1 = the epilogue warps release the accumulators without reading them.
// BBUFS: buffers of the query operand (2 = the next (n, z) pair's operand loads under the current pair's MMAs; 1 = its 64 KiB go
// to the database ring instead, at the price of a reload bubble per pair).  ABUFS: accumulator buffers in TMEM (128 columns each).
template <int KSPS, int BBUFS, int ABUFS>
__global__ void __launch_bounds__(TC5_THREADS, 1)
k_multiply_tc5(DevParams P, Tc5Geom T, const uint8_t* __restrict__ dbt, const uint8_t* __restrict__ qt,
               uint32_t* __restrict__ out_zm, size_t out_stride, int nq, int slice_begin, int slice_count,
               uint32_t* __restrict__ dbg /* bring-up aid: raw accumulators of CTA 0's first TC5_DBG_TILES tiles, or null */,
               int dbg_mode, const uint32_t* __restrict__ tile_mask /* [slice][mt]: bit ks = the 32-row x 32-j tile holds a present item */) {
  const bool hinted = (dbg_mode & 4) != 0;
#define mbar_wait(bar, par) do { if (hinted) mbar_wait_hinted(bar, par); else (mbar_wait)(bar, par); } while (0)
  constexpr int TC5_KS_PER_STAGE = KSPS;
  constexpr int TC5_STAGE_BYTES = KSPS * TC5_TILE;
  constexpr int TC5_TMEM_COLS = ABUFS * TC5_N;
  const int TC5_STAGES = tc5_ring_stages(T.ks, KSPS, BBUFS);
  extern __shared__ __align__(1024) uint8_t tc5_smem[];
  uint8_t* smem_b = tc5_smem;                                         // [BBUFS][ks][4096]
  uint8_t* smem_a = smem_b + (size_t)BBUFS * T.ks * TC5_TILE;         // [STAGES][KSPS x 4 KiB]
  Tc5Smem* S = reinterpret_cast<Tc5Smem*>(smem_a + (size_t)TC5_STAGES * TC5_STAGE_BYTES);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int stages_per_tile = (T.ks + TC5_KS_PER_STAGE - 1) / TC5_KS_PER_STAGE;
  const int tiles_per_item = slice_count * T.mt;
  const int n_items = 2 * POLY;
  const uint32_t b_bytes = (uint32_t)T.ks * TC5_TILE;

  if (threadIdx.x == 0) {
    for (int s = 0; s < TC5_STAGES; s++) { mbar_init(&S->full[s], 1); mbar_init(&S->empty[s], 1); }
    for (int b = 0; b < 2; b++) { mbar_init(&S->bfull[b], 1); mbar_init(&S->bempty[b], 1); }
    for (int b = 0; b < 4; b++) { mbar_init(&S->tfull[b], 1); mbar_init(&S->tempty[b], TC5_EPI_WARPS); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {                                                    // TMEM allocation is owned by the MMA warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&S->tmem_base)),
                 "n"(TC5_TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = S->tmem_base;

  // The producer and MMA warps run their loops CONVERGED (all 32 lanes, warp-uniform values); only the asynchronous
  // instructions themselves are issued by one elected lane.  (Issuing from inside an `if (lane == 0)` region makes every
  // operand of UBLKCP / UTCIMMA / UTCBAR a per-thread value: ptxas then wraps each of them in an ELECT / R2UR serialisation
  // loop, and the single MMA thread needs ~140 clocks per 64-clock MMA — measured, profiles/ncu_tc5_r02a_source.md.)
  if (warp == 0) {
    // ===== producer =====
    int stage = 0; uint32_t sphase = 0;
    int it = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, it++) {
      const int n = item & 1, z = item >> 1, bb = it % BBUFS;
      mbar_wait(&S->bempty[bb], ((it / BBUFS) & 1) ^ 1);
      if (elect_one()) {
        mbar_expect_tx(&S->bfull[bb], b_bytes);
        bulk_g2s(smem_b + (size_t)bb * b_bytes, qt + tc5_q_tile(T, n, z, 0) * TC5_TILE, b_bytes, &S->bfull[bb]);
      }
      __syncwarp();
      for (int sl = 0; sl < slice_count; sl++)
        for (int mt = 0; mt < T.mt; mt++) {
          const uint8_t* src = dbt + tc5_db_tile(T, slice_begin + sl, n, z, mt, 0) * TC5_TILE;
          // lib/server's sparse database (db/sparse_db.rs, compute/dot_product.rs:35): tiles without a present item are neither
          // fetched nor multiplied (they are zero: the sums are unchanged); a stage without any such tile takes no ring slot
          const uint32_t mask = __ldg(tile_mask + (size_t)(slice_begin + sl) * T.mt + mt);
          for (int st = 0; st < stages_per_tile; st++) {
            const int ks_here = min(TC5_KS_PER_STAGE, T.ks - st * TC5_KS_PER_STAGE);
            const uint32_t full_m = ks_here == 32 ? 0xffffffffu : ((1u << ks_here) - 1u);
            const uint32_t km = (mask >> (st * TC5_KS_PER_STAGE)) & full_m;
            if (km == 0) continue;
            mbar_wait(&S->empty[stage], sphase ^ 1);
            if (elect_one()) {
              uint8_t* dst = smem_a + (size_t)stage * TC5_STAGE_BYTES;
              const uint8_t* from = src + (size_t)st * TC5_STAGE_BYTES;
              mbar_expect_tx(&S->full[stage], (uint32_t)__popc(km) * TC5_TILE);
              if (km == full_m) bulk_g2s(dst, from, (uint32_t)ks_here * TC5_TILE, &S->full[stage]);
              else
                for (int kk = 0; kk < ks_here; kk++)
                  if ((km >> kk) & 1u) bulk_g2s(dst + (size_t)kk * TC5_TILE, from + (size_t)kk * TC5_TILE, TC5_TILE, &S->full[stage]);
            }
            __syncwarp();
            if (++stage == TC5_STAGES) { stage = 0; sphase ^= 1; }
          }
        }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    int stage = 0; uint32_t sphase = 0;
    int it = 0, tile_no = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, it++) {
      const int bb = it % BBUFS;
      mbar_wait(&S->bfull[bb], (it / BBUFS) & 1);
      const uint32_t b_addr = smem_u32(smem_b + (size_t)bb * b_bytes);
      for (int t = 0, sl = 0, mt = 0; t < tiles_per_item; t++, tile_no++, mt++) {
        if (mt == T.mt) { mt = 0; sl++; }
        const uint32_t mask = __ldg(tile_mask + (size_t)(slice_begin + sl) * T.mt + mt);
        uint32_t issued = 0;                                          // the first MMA of a tile overwrites the accumulator
        const int ab = tile_no % ABUFS;
        mbar_wait(&S->tempty[ab], ((tile_no / ABUFS) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d_addr = tmem_base + (uint32_t)ab * TC5_N;
        for (int st = 0; st < stages_per_tile; st++) {
          const int ks_here = min(TC5_KS_PER_STAGE, T.ks - st * TC5_KS_PER_STAGE);
          const uint32_t km = (mask >> (st * TC5_KS_PER_STAGE)) & (ks_here == 32 ? 0xffffffffu : ((1u << ks_here) - 1u));
          if (km == 0) continue;                                      // nothing fetched for this stage (see the producer)
          mbar_wait(&S->full[stage], sphase);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(smem_a + (size_t)stage * TC5_STAGE_BYTES);
          if (elect_one()) {
            if (dbg_mode & 1) mbar_arrive(&S->empty[stage]);
            else {
#pragma unroll
              for (int kk = 0; kk < TC5_KS_PER_STAGE; kk++) {
                if ((km >> kk) & 1u) {
                  const int ks = st * TC5_KS_PER_STAGE + kk;
                  tc_mma_i8(d_addr, tc5_smem_desc(a_addr + kk * TC5_TILE), tc5_smem_desc(b_addr + ks * TC5_TILE), issued);
                  issued = 1u;
                }
              }
              tc_commit(&S->empty[stage]);                            // frees the A stage when these MMAs have completed
            }
          }
          issued = 1u;                                                // warp-uniform copy of the elected lane's flag (km != 0)
          __syncwarp();
          if (++stage == TC5_STAGES) { stage = 0; sphase ^= 1; }
        }
        if (elect_one()) {
          if (dbg_mode & 1) mbar_arrive(&S->tfull[ab]);
          else tc_commit(&S->tfull[ab]);                              // accumulator ready for the epilogue
        }
        __syncwarp();
      }
      if (elect_one()) {
        if (dbg_mode & 1) mbar_arrive(&S->bempty[bb]);
        else tc_commit(&S->bempty[bb]);                               // every MMA reading this B buffer has completed
      }
      __syncwarp();
    }
  } else {
    // ===== epilogue: warps 2..9, TMEM lane quadrant = warp % 4 (hardware rule), column half = (warp - 2) / 4 =====
    const int quad = warp & 3, colhalf = (warp - 2) >> 2;
    const int l = tc5_lane_limb(lane);                                // database limb held by this lane
    int it = 0, tile_no = 0;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x, it++) {
      const int n = item & 1, z = item >> 1;
      const uint32_t q = n ? P.q[1] : P.q[0];
      const Tc5Weights W = tc5_lane_weights(l, q);
      for (int t = 0, slice = slice_begin, mt = 0; t < tiles_per_item; t++, tile_no++, mt++) {
        if (mt == T.mt) { mt = 0; slice++; }
        const int ab = tile_no % ABUFS;
        mbar_wait(&S->tfull[ab], (tile_no / ABUFS) & 1);
        tc_fence_after();
        const int ii = mt * 32 + tc5_lane_row(quad, lane);
        const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)ab * TC5_N;
        const bool empty_tile = __ldg(tile_mask + (size_t)slice * T.mt + mt) == 0;   // no MMA touched the accumulator: the product is zero
        // both 32-column chunks of this warp go to registers first, so the accumulator buffer is released after the TMEM
        // load latency, not after the arithmetic: the MMA of a later tile never waits for epilogue math
        uint32_t v[2][32];
        if (!(dbg_mode & 2) && !empty_tile) {
          tc_ld32(taddr + (colhalf * 2 + 0) * 32, v[0]);
          tc_ld32(taddr + (colhalf * 2 + 1) * 32, v[1]);
          tc_wait_ld();
        }
        if (empty_tile) {
#pragma unroll
          for (int c = 0; c < 32; c++) { v[0][c] = 0; v[1][c] = 0; }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&S->tempty[ab]);                   // this warp has drained its part of the accumulator
#pragma unroll
        for (int ch = 0; ch < ((dbg_mode & 2) ? 0 : 2); ch++) {       // 32 TMEM columns = 8 GEMM columns = 4 queries
          const int chunk = colhalf * 2 + ch;
          if (dbg && blockIdx.x == 0 && tile_no < TC5_DBG_TILES) {
#pragma unroll
            for (int c = 0; c < 32; c++) dbg[((size_t)tile_no * TC5_M + quad * 32 + lane) * TC5_N + chunk * 32 + c] = v[ch][c];
          }
          uint64_t part[8], send4[4], keep4[4], send2[2], keep2[2];
#pragma unroll
          for (int c = 0; c < 8; c++) part[c] = tc5_lane_partial(v[ch] + 4 * c, W.w, W.wp);   // < 2^53
          tc5_rs_select_a(l, part, send4, keep4);
#pragma unroll
          for (int i = 0; i < 4; i++) keep4[i] += shfl_xor_u64(send4[i], 2);
          tc5_rs_select_b(l, keep4, send2, keep2);
#pragma unroll
          for (int i = 0; i < 2; i++) keep2[i] += shfl_xor_u64(send2[i], 1);              // columns 2l, 2l+1 over all four limbs, < 2^55
          // lane l stores query 4*chunk + l (both ciphertext rows = GEMM columns 2l, 2l+1 of this chunk)
          const int qi = tc5_lane_query(chunk, lane);
          if (qi < nq && ii < T.rows) {
            uint2 r = make_uint2(tc5_barrett57(keep2[0], W.mu, q), tc5_barrett57(keep2[1], W.mu, q));
            uint32_t* dst = out_zm + (size_t)qi * out_stride + ((((size_t)slice * 2 + n) * POLY + z) * T.rows + ii) * 2;
            *reinterpret_cast<uint2*>(dst) = r;
          }
        }
      }
    }
  }

#undef mbar_wait
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(TC5_TMEM_COLS) : "memory");
  }
}

}  // namespace

size_t tc5_db_bytes(const Tc5Geom& T, int slices) { return (size_t)slices * 2 * POLY * T.mt * T.ks * TC5_TILE; }
size_t tc5_query_bytes(const Tc5Geom& T) { return (size_t)2 * POLY * T.ks * TC5_TILE; }
static size_t tc5_smem_bytes(const Tc5Geom& T, int ksps, int bbufs) {
  return (size_t)bbufs * T.ks * TC5_TILE + (size_t)tc5_ring_stages(T.ks, ksps, bbufs) * ksps * TC5_TILE + sizeof(Tc5Smem) + 16;
}
// at least two ring stages beside a single-buffered query operand
bool tc5_supported(const Tc5Geom& T) { return T.dim0 % 2 == 0 && tc5_ring_stages(T.ks, 4, 1) >= 2; }

void launch_db_to_tc5(const Tc5Geom& T, const uint4* db0_slice, uint8_t* dbt, int slice, cudaStream_t s) {
  ++g_kernel_launches;
  k_db_to_tc5<<<dim3(POLY, T.mt, T.ks), 256, 0, s>>>(T, db0_slice, dbt, slice);
}
void launch_db_upsert_tc5(const Tc5Geom& T, uint8_t* dbt, int slice, int il, int j, const uint64_t* poly, cudaStream_t s) {
  ++g_kernel_launches;
  k_db_upsert_tc5<<<POLY / 256, 256, 0, s>>>(Tc5Store{T, dbt}, slice, il, j, poly);
}
void launch_write_items(const DevParams& P, const Tc5Geom& T, uint8_t* dbt, int slices, const ItemWrite* items, int count,
                        const uint8_t* data, int bpc, uint64_t pt_modulus, cudaStream_t s) {
  item_write::launch(P, Tc5Store{T, dbt}, items, count, slices, data, bpc, pt_modulus, s);
}
void launch_query_to_tc5(const Tc5Geom& T, const uint4* q_dev, size_t q_stride, int nq, uint8_t* qt, cudaStream_t s) {
  if (nq < 1 || nq > 16) throw Error(-2, "tcgen05 multiply: 1..16 queries per pass");
  ++g_kernel_launches;
  k_query_to_tc5<<<dim3(POLY / 2, T.ks), 256, 0, s>>>(T, q_dev, q_stride, nq, qt);
}
void launch_reorient_to_tc5(const Tc5Geom& T, const uint32_t* v, size_t v_stride, int idx_factor, int nq, uint8_t* qt, cudaStream_t s) {
  if (nq < 1 || nq > 16) throw Error(-2, "tcgen05 multiply: 1..16 queries per pass");
  ++g_kernel_launches;
  opt_in_smem(k_reorient_to_tc5, 16 * TC5_TILE);
  k_reorient_to_tc5<<<dim3(POLY / 8, T.ks), 256, 16 * TC5_TILE, s>>>(T, v, v_stride, idx_factor, nq, qt);
}
void launch_multiply_tc5(const DevParams& P, const Tc5Geom& T, const uint8_t* dbt, const uint32_t* tile_mask, const uint8_t* qt,
                         uint32_t* out_zm, size_t out_stride, int nq, int slice_begin, int slice_count, int sm_count, cudaStream_t s) {
  if (nq < 1 || nq > 16) throw Error(-2, "tcgen05 multiply: 1..16 queries per pass");
  if (!tc5_supported(T)) throw Error(-2, "tcgen05 multiply: dim0 too large for one CTA's shared memory");
  ++g_kernel_launches;
  const int grid = sm_count > 0 ? (sm_count < 2 * POLY ? sm_count : 2 * POLY) : 148;
  // bring-up aid (scripts/tc5_probe.py): B200PIR_TC5_DUMP=<file> receives the raw s32 accumulators D[M][N] of the first
  // tiles CTA 0 computes (item n = 0, z = 0), so a mismatch can be traced to the operand layout / TMEM mapping assumption
  const char* dump = getenv("B200PIR_TC5_DUMP");
  uint32_t* dbg = nullptr;
  const size_t dbg_words = (size_t)TC5_DBG_TILES * TC5_M * TC5_N;
  if (dump) {
    B200_CUDA(cudaMalloc(&dbg, dbg_words * 4));
    B200_CUDA(cudaMemsetAsync(dbg, 0xFF, dbg_words * 4, s));
  }
  static const int dbg_mode = getenv("B200PIR_TC5_DBG") ? atoi(getenv("B200PIR_TC5_DBG")) : 0;     // analysis only: wrong results
  static const int ksps_env = getenv("B200PIR_TC5_KSPS") ? atoi(getenv("B200PIR_TC5_KSPS")) : 8;
  static const int bbufs_env = getenv("B200PIR_TC5_BBUFS") ? atoi(getenv("B200PIR_TC5_BBUFS")) : 2;
  static const int abufs = getenv("B200PIR_TC5_ABUFS") ? atoi(getenv("B200PIR_TC5_ABUFS")) : 4;
  int ksps = ksps_env == 4 ? 4 : 8, bbufs = bbufs_env == 2 ? 2 : 1;
  if (tc5_ring_stages(T.ks, ksps, bbufs) < 2) ksps = 4;                  // large dim0: smaller stages,
  if (tc5_ring_stages(T.ks, ksps, bbufs) < 2) bbufs = 1;                 // single-buffered operand
  const size_t smem = tc5_smem_bytes(T, ksps, bbufs);
#define TC5_LAUNCH(K, B, A)                                                                                                    \
  do {                                                                                                                         \
    opt_in_smem(k_multiply_tc5<K, B, A>, 227 * 1024);                                                                          \
    k_multiply_tc5<K, B, A><<<grid, TC5_THREADS, smem, s>>>(P, T, dbt, qt, out_zm, out_stride, nq, slice_begin, slice_count,   \
                                                            dbg, dbg_mode, tile_mask);                                         \
  } while (0)
#define TC5_PICK_A(K, B) do { if (abufs == 2) TC5_LAUNCH(K, B, 2); else TC5_LAUNCH(K, B, 4); } while (0)
  if (ksps == 4) { if (bbufs == 2) TC5_PICK_A(4, 2); else TC5_PICK_A(4, 1); }
  else { if (bbufs == 2) TC5_PICK_A(8, 2); else TC5_PICK_A(8, 1); }
#undef TC5_PICK_A
#undef TC5_LAUNCH
  if (dump) {
    std::vector<uint32_t> host(dbg_words);
    B200_CUDA(cudaStreamSynchronize(s));
    B200_CUDA(cudaMemcpy(host.data(), dbg, dbg_words * 4, cudaMemcpyDeviceToHost));
    cudaFree(dbg);
    if (FILE* f = fopen(dump, "wb")) { fwrite(host.data(), 4, dbg_words, f); fclose(f); }
  }
}

}  // namespace b200pir
