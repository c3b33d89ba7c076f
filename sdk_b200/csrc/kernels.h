// Launch wrappers (host side) for the sm_100a kernels.  All pointers are DEVICE pointers unless
// noted; every launch goes to the given stream and returns immediately.
//
// Device formats
//   ntt32 poly : uint32_t [n(2)][z(2048)]  residues mod q_n in the reference's (bit-reversed) NTT order
//   raw poly   : uint64_t [z(2048)]        coefficients in [0, q]  (q itself can occur: reference quirk,
//                                           lib/spiral-rs/src/poly.rs:387-405, SURVEY A.6)
//   matrices   : row-major [row][col] of polys, as PolyMatrixRaw / PolyMatrixNTT (poly.rs:59-71)
#pragma once
#include "common.cuh"
#include "tc5_layout.cuh"

namespace b200pir {

static const int POLY = 2048;

// number of kernels this library has launched from the calling thread (bench.py reports it)
extern thread_local unsigned long long g_kernel_launches;

// Opt a kernel in to more than 48 KiB of dynamic shared memory.  cudaFuncSetAttribute applies to the CURRENT device only, so
// the opt-in is remembered per (kernel, device): one process may drive several GPUs (one context per GPU) from several host
// threads.  Thread-safe.
void opt_in_smem_impl(const void* kernel, int bytes);
template <typename K>
inline void opt_in_smem(K* kernel, int bytes) { opt_in_smem_impl(reinterpret_cast<const void*>(kernel), bytes); }

// ---- generic transforms (K3/K4 of SURVEY §2.3)
// u64 ABI format [poly][n][z]  <->  in place forward / inverse NTT (ntt.rs:67-113 / :212-258)
void launch_ntt_u64(const DevParams& P, uint64_t* polys, size_t count, bool inverse, cudaStream_t s);
// ntt32 in place
void launch_ntt32(const DevParams& P, uint32_t* polys, size_t count, bool inverse, cudaStream_t s);
// poly.rs:613-638 to_ntt: raw u64 -> ntt32 (reduce mod q_n, forward NTT)
// poly_len = 4096 (config #5 only): polys ntt32 [count][2][4096]; tw = {fwd0, inv0, fwd1, inv1} x 4096 entries
void launch_ntt32_4k(uint32_t q0, uint32_t q1, const Twiddle* tw, uint32_t* polys, size_t count, bool inverse, cudaStream_t s);
void launch_to_ntt(const DevParams& P, uint32_t* out, const uint64_t* raw, size_t count, cudaStream_t s);
// `batches` groups of `count` polynomials, groups out_stride (u32) / raw_stride (u64) words apart, in one launch
void launch_to_ntt_strided(const DevParams& P, uint32_t* out, size_t out_stride, const uint64_t* raw, size_t raw_stride,
                           size_t count, int batches, cudaStream_t s);
// client.rs:47-80: first rows of n_mats raw matrices = q - (ChaCha20 keystream u64 % q), keystream u64 index word0 onwards
void launch_chacha_first_rows(uint64_t* raw, const uint8_t seed[32], uint64_t word0, uint32_t n_mats, uint32_t row_words,
                              uint64_t mat_words, uint64_t modulus, cudaStream_t s);
// client.rs:316-327: regenerated row-0 transforms (ntt32 [j][n][z]) + uploaded words ([z][j]) -> q_dev (format of launch_query_to_dev)
void launch_direct_query_to_dev(uint4* q_dev, const uint32_t* sig_ntt, const uint64_t* wire_words, int dim0, cudaStream_t s);
// poly.rs:646-663 from_ntt: ntt32 -> raw u64 (inverse NTT both moduli + CRT lift)
void launch_from_ntt(const DevParams& P, uint64_t* out_raw, const uint32_t* in, size_t count, cudaStream_t s);
// raw u64 coefficients <-> residue form u32 [poly][n][z] (coefficient domain; the CRT lift is poly.rs:658)
void launch_raw_to_res(const DevParams& P, uint32_t* out, const uint64_t* raw, size_t polys, cudaStream_t s);
void launch_res_to_raw(const DevParams& P, uint64_t* out, const uint32_t* res, size_t polys, cudaStream_t s);
// twiddle entries 0..63 of every (modulus, direction) -> constant bank of the poly kernels' module
void upload_poly_constants(const Twiddle* lo /* [2][3][64]: forward, inverse, relaxed-range inverse */);
void upload_mul_constants(const Twiddle* lo /* [2][3][64]: forward, inverse, relaxed-range inverse */);
// format converters for the C ABI (u64 [n][z] words < 2^32  <->  ntt32)
void launch_widen(uint64_t* out, const uint32_t* in, size_t words, cudaStream_t s);
void launch_narrow(uint32_t* out, const uint64_t* in, size_t words, cudaStream_t s);

// ---- first dimension (K1): server.rs:155-221
struct MulGeom { int dim0, num_per, slices; };
// db_dev : uint4 [slice][ii][jp = j/2][z] = {w(2jp).lo, w(2jp).hi, w(2jp+1).lo, w(2jp+1).hi}
// q_dev  : uint4 [jp][jb][z] = {a[j][r0].lo, a[j][r0].hi, a[j][r1].lo, a[j][r1].hi},  j = 2jp+jb
// out    : ntt32 [slice][ii][r][n][z]
// `nq` queries are processed per DB pass (q_dev / out strided by q_stride / out_stride uint4 / u32).
void launch_multiply(const DevParams& P, const MulGeom& G, const uint4* db_dev, const uint4* q_dev, uint32_t* out,
                     int slice_begin, int slice_count, int nq, size_t q_stride, size_t out_stride, int variant,
                     cudaStream_t s);
// reference layout v_firstdim u64 [z][j][r]  ->  q_dev
void launch_query_to_dev(const MulGeom& G, uint4* q_dev, const uint64_t* v_firstdim, cudaStream_t s);
// Row sharding of the second-dimension index: this GPU holds global rows ii = il*count + index
// (il = local row, G.num_per local rows).  index=0,count=1 is the whole database.
struct Shard { int index, count; };
// reference layout u64 [zc][num_per_global][dim0] (z in [z0,z0+zc))  ->  db_dev slice (local rows)
void launch_db_retile_chunk(const MulGeom& G, Shard sh, uint4* db_dev_slice, const uint64_t* ref_chunk, int z0, int zc,
                            cudaStream_t s);
// one item poly (2048 packed words, lo|hi<<32) -> its place in db_dev   (lib/server db/loading.rs:317-359)
void launch_db_upsert(const MulGeom& G, uint4* db_dev, int slice, int il, int j, const uint64_t* poly, cudaStream_t s);
// One item of a bulk write (item_write.cuh): its raw bytes are data[off, off + len), zero padded to slices * bpc; it goes to
// local row il, column j of every slice.
struct ItemWrite { uint32_t off, len, il, j; };
// lib/server db/loading.rs:317-359 update_item_raw for `count` distinct items in one launch (raw bytes -> recenter, NTT, pack
// -> the database layout); one overload per layout
void launch_write_items(const DevParams& P, const MulGeom& G, uint4* db_dev, int slices, const ItemWrite* items, int count,
                        const uint8_t* data, int bpc, uint64_t pt_modulus, cudaStream_t s);
// synthetic DB: plaintext coeff = splitmix64(seed, ((slice*items + item)*2048 + z)) % p, recentred, NTT'd, packed
// (server.rs:223-275 with a counter PRNG; item = j*num_per_global + ii)
void launch_db_synth(const DevParams& P, const MulGeom& G, Shard sh, uint4* db_dev, uint64_t seed, uint64_t pt_modulus,
                     int slice_begin, int slice_count, cudaStream_t s);

// ---- first dimension on INT8 tensor cores (imma_kernels.cu): database in MMA fragment order
struct ImmaGeom { int dim0, rows, mt /* ceil(rows/16) */, ks /* ceil(dim0/32) */; };
inline ImmaGeom make_imma_geom(int dim0, int rows) { return ImmaGeom{dim0, rows, (rows + 15) / 16, (dim0 + 31) / 32}; }
size_t imma_db_cells(const ImmaGeom& F, int slices);      // uint4 cells of the whole database
size_t imma_query_cells(const ImmaGeom& F);               // uint2 cells of the B operand (up to 16 queries)
bool imma_supports_16(const ImmaGeom& F);                 // 16 queries per database pass fit one CTA's shared memory
inline int imma_query_tiles(int nq) { return nq > 8 ? 4 : (nq > 4 ? 2 : 1); }   // column tiles of 4 queries
void upload_imma_constants(const Twiddle* lo);
// one slice in the IMAD layout (uint4 [row][jp][z]) -> fragment order
void launch_db_to_frag(const ImmaGeom& F, const uint4* db0_slice, uint4* dbf, int slice, cudaStream_t s);
void launch_db_upsert_frag(const ImmaGeom& F, uint4* dbf, int slice, int il, int j, const uint64_t* poly, cudaStream_t s);
void launch_write_items(const DevParams& P, const ImmaGeom& F, uint4* dbf, int slices, const ItemWrite* items, int count,
                        const uint8_t* data, int bpc, uint64_t pt_modulus, cudaStream_t s);
void launch_query_to_frag(const ImmaGeom& F, const uint4* q_dev, size_t q_stride, int nq, uint2* qf, cudaStream_t s);
// out_zm: u32 [query][slice][n][z][row][ct_row]  (queries out_stride words apart)
void launch_multiply_imma(const DevParams& P, const ImmaGeom& F, const uint4* dbf, const uint2* qf, uint32_t* out_zm,
                          size_t out_stride, int nq, int slice_begin, int slice_count, int variant, cudaStream_t s);
// inverse NTT of the z-major product -> residue-form ciphertexts [query*slices + slice][row][ct_row][n][z]
// variant 0: tiled (sector-efficient) kernel, 1: simple gather kernel
void launch_intt_from_zmajor(const DevParams& P, const ImmaGeom& F, const uint32_t* in_zm, size_t in_stride, uint32_t* out,
                             int nq, int slices, int variant, cudaStream_t s);
// z-major product of one slice -> ntt32 [row][ct_row][n][z]
void launch_zmajor_to_ntt32(const ImmaGeom& F, const uint32_t* in_zm, uint32_t* out, int slice, cudaStream_t s);

// ---- first dimension on tcgen05 (tc5_kernels.cu): operands stored as shared-memory tile images (database format 2)
size_t tc5_db_bytes(const Tc5Geom& T, int slices);
size_t tc5_query_bytes(const Tc5Geom& T);                 // 16 queries
bool tc5_supported(const Tc5Geom& T);
void launch_db_to_tc5(const Tc5Geom& T, const uint4* db0_slice, uint8_t* dbt, int slice, cudaStream_t s);
void launch_db_upsert_tc5(const Tc5Geom& T, uint8_t* dbt, int slice, int il, int j, const uint64_t* poly, cudaStream_t s);
void launch_write_items(const DevParams& P, const Tc5Geom& T, uint8_t* dbt, int slices, const ItemWrite* items, int count,
                        const uint8_t* data, int bpc, uint64_t pt_modulus, cudaStream_t s);
void launch_query_to_tc5(const Tc5Geom& T, const uint4* q_dev, size_t q_stride, int nq, uint8_t* qt, cudaStream_t s);
// out_zm as launch_multiply_imma; up to 16 queries per pass; one persistent CTA per SM
// reorient_reg_ciphertexts (util.rs:323-355) fused with the re-tiling: expansion workspace v (ntt32 [query][slot][row][n][z]) ->
// tile images of up to 16 queries (the B operand of launch_multiply_tc5)
void launch_reorient_to_tc5(const Tc5Geom& T, const uint32_t* v, size_t v_stride, int idx_factor, int nq, uint8_t* qt, cudaStream_t s);
// tile_mask: u32 [slice][mt], bit ks set = the tile (32 rows x 32 values of j) holds at least one present item; clear bits are
// neither fetched nor multiplied (lib/server's sparse database: absent items cost nothing, db/sparse_db.rs, dot_product.rs:35)
void launch_multiply_tc5(const DevParams& P, const Tc5Geom& T, const uint8_t* dbt, const uint32_t* tile_mask, const uint8_t* qt,
                         uint32_t* out_zm, size_t out_stride, int nq, int slice_begin, int slice_count, int sm_count, cudaStream_t s);

// ---- second dimension
// mult output ntt32 [cnt][r][n][z] -> raw ciphertexts u64 [cnt][r][z]   (server.rs:707-709)
// (== launch_from_ntt with 2*cnt polys)
// fold (server.rs:388-427): one launch per round.  cts: raw [batch][num][2][2048] (in place);
// step (b,i) : ct[i] <- from_ntt(Cneg * G^-1(ct[i]) + C * G^-1(ct[half+i]))
void launch_fold_round(const DevParams& P, uint64_t* cts, size_t batch, size_t batch_stride /*u64 words*/, int half,
                       const uint32_t* c_pos, const uint32_t* c_neg, size_t c_batch_stride /*u32 words, per query*/,
                       int slices_per_query, int t_gsw, int bits, cudaStream_t s);
// Fast path on residue-form ciphertexts u32 [batch][num][row][n][z] (see k_fold_res): out[i] (i < half) from
// in[i], in[half+i]; in != out.  Needs only v_folding (c_pos).
void launch_fold_res(const DevParams& P, const uint32_t* in, uint32_t* out, size_t batch, size_t batch_stride /*u32*/,
                     int half, const uint32_t* c_pos, size_t c_batch_stride, int slices_per_query, int t_gsw, int bits,
                     int variant, uint32_t* zero_flags /* null = dense semantics (spiral-rs); else scratch of batch*2*half words: lib/server fold.rs:37-43 */, cudaStream_t s);
// server.rs:505-523 get_v_folding_neg, computed pointwise: neg = (q_n - C) + G  (NTT is linear and the
// gadget matrix is constant-coefficient, so this is the same canonical value)
void launch_folding_neg(const DevParams& P, uint32_t* out, const uint32_t* v_folding, int count, int t_gsw, int bits,
                        cudaStream_t s);

// ---- query expansion (server.rs:19-151, 525-591)
// v: ntt32 [nq][2^g][2][n][z] (queries v_stride words apart).  One round = scalar-multiply launch + expand
// launch, each covering all nq queries (grid.y).
void launch_expand_scalar(const DevParams& P, uint32_t* v, size_t v_stride, int nq, int num_in, const uint32_t* neg1_r,
                          cudaStream_t s);
// Public parameters are per QUERY: device arrays of base pointers (the ntt32 matrices of the client that sent query i), so one
// launch serves concurrent queries of different clients — lib/server looks the parameters up per request (bin/server.rs:113-117).
struct PpTable { const uint32_t* const* pack; const uint32_t* const* left; const uint32_t* const* right; const uint32_t* const* conv; };
struct ExpandRound {
  int r, num_in, stop_round, max_bits_to_gen_right, t_auto;
  const uint32_t* const* tab_left;    // [query] -> v_expansion_left of that query's client; this round's matrix (ntt32 [2][t_exp_left])
  const uint32_t* const* tab_right;   // starts off_left / off_right words further
  size_t off_left, off_right;
  int t_left, t_right, bits_left, bits_right;
  int fill_skipped;         // paired kernel: also write v[i + num_in] = v[i] (.) neg1 for skipped i (stage-level parity)
};
void launch_expand_round(const DevParams& P, uint32_t* v, size_t v_stride, int nq, const ExpandRound& R, cudaStream_t s);
// both outputs of every input ciphertext in one CTA; replaces launch_expand_scalar + launch_expand_round for that round
void launch_expand_round_pair(const DevParams& P, uint32_t* v, size_t v_stride, int nq, const ExpandRound& R,
                              const uint32_t* neg1_r, cudaStream_t s);
// the paired round split into an inverse-transform kernel (residues -> xr) and single-modulus CTAs at 3 per SM
void launch_expand_round_res(const DevParams& P, uint32_t* v, size_t v_stride, uint32_t* xr, size_t xr_stride, int nq,
                             const ExpandRound& R, const uint32_t* neg1_r, cudaStream_t s);
// util.rs:323-355 reorient: v[idx_factor*j] -> q_dev   (per query: q_stride uint4 apart)
void launch_reorient(const MulGeom& G, uint4* q_dev, size_t q_stride, const uint32_t* v, size_t v_stride, int nq,
                     int idx_factor, cudaStream_t s);
// server.rs:123-151: v_gsw[i] (ntt32 [2][2 t_gsw]) from v_inp[idx_factor*(i t_gsw + j) + idx_offset]
void launch_regev_to_gsw(const DevParams& P, uint32_t* v_gsw, size_t gsw_stride, const uint32_t* v, size_t v_stride,
                         int nq, int count, int idx_factor, int idx_offset, const uint32_t* const* tab_conv, int t_gsw,
                         int t_conv, int bits_conv, cudaStream_t s);

// ---- packing + encoding (server.rs:429-503; lib/server compute/pack.rs)
// folded: residue-form ciphertexts, ct (inst, t) at folded + (inst*n*n + t)*ct_stride (u32 words);
// w: ntt32 packing matrices; out: raw [inst][n+1][n][2048]
// nq queries per launch: query k reads folded + k*in_q_stride and writes out_raw + k*out_q_stride
void launch_pack(const DevParams& P, uint64_t* out_raw, size_t out_q_stride, const uint32_t* folded, size_t ct_stride,
                 size_t in_q_stride, int nq, const uint32_t* const* tab_pack, int n, int instances, int t_conv, int bits_conv,
                 int version, cudaStream_t s);
// out: nq x out_bytes; packed_raw: nq matrices packed_q_stride words apart
void launch_encode(const DevParams& P, uint8_t* out, size_t out_bytes, const uint64_t* packed_raw, size_t packed_q_stride,
                   int nq, int n, int instances, uint64_t q2, int q2_bits, uint64_t q1, int q1_bits, cudaStream_t s);

// ---- DoublePIR packed matvec (K6): lib/doublepir/src/matrix/kernels.rs:14-178
void launch_dpir_matvec(uint32_t* out, const uint32_t* a, const uint32_t* b, size_t rows, size_t cols, int variant,
                        cudaStream_t s);

// lib/doublepir/src/matrix/kernels.rs:180-278 and matrix/indexing.rs:117-143 (the small tail of answer())
void launch_dpir_mul_transposed(uint32_t* out, const uint32_t* a, const uint32_t* b, size_t a_rows, size_t a_cols,
                                size_t b_rows, size_t b_cols, cudaStream_t s);
void launch_dpir_transpose_expand(uint32_t* out, const uint32_t* a, size_t rows, size_t cols, uint64_t modulus, size_t delta,
                                  size_t concat, size_t out_rows, size_t out_cols, cudaStream_t s);

// ---- DoublePIR offline setup (dpir_gemm.cu): doublepir.rs:76-108
// c (rows x n_cols) = a (rows x k_dim, entries in [-2^15, 2^15) as wrapping u32) * b (k_dim x n_cols) mod 2^32; device pointers;
// 8-bit limb products on the tcgen05 tensor cores (exact); synchronises the stream
void launch_dpir_gemm(uint32_t* c, const uint32_t* a, const uint32_t* b, size_t rows, size_t k_dim, size_t n_cols, cudaStream_t s);
// transpose + expand (contract.rs:62-78) + concat_cols (indexing.rs:82-101): h (l x n) -> out ((n delta x) x (l / x)), centred digits
void launch_dpir_transpose_expand_concat(uint32_t* out, const uint32_t* h, size_t l, size_t n, uint32_t p, int delta, size_t x,
                                         cudaStream_t s);
// squish(m + add), three 10-bit values per word (squish.rs:52-70)
void launch_dpir_add_squish(uint32_t* out, const uint32_t* m, size_t rows, size_t cols, uint32_t add, cudaStream_t s);
// rows padded with zeros to rows3, then transposed (doublepir.rs:96-100)
void launch_dpir_pad_transpose(uint32_t* out, const uint32_t* a, size_t rows, size_t cols, size_t rows3, cudaStream_t s);

}  // namespace b200pir
