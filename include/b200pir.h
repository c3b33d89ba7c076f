/* b200pir — C ABI of the B200-native server-side PIR query path.
 *
 * This is the drop-in boundary: every entry point replaces one Rust function of blyssprivacy/sdk
 * (reference @ fdb7206); the Rust host code keeps its own signature and forwards here through a thin
 * `extern "C"` shim (see INTEGRATION.md).  The reference has no FFI of its own, so the ABI flattens
 * the reference's argument types to plain pointers + sizes:
 *
 *   PolyMatrixRaw   rows x cols polys, each 2048 u64 coefficients            (lib/spiral-rs/src/poly.rs:59-64)
 *   PolyMatrixNTT   rows x cols polys, each [crt(2)][2048] u64 residues     (poly.rs:66-71, :263-265)
 *   db: &[u64]      [instance][trial][z][ii][j] words = q0-residue | q1-residue << 32   (server.rs:263-269)
 *   v_firstdim      [z][j][r] words, same packing                            (util.rs:343-350)
 *
 * All buffers are HOST memory owned by the caller unless the name says `_dev`.  Outputs are caller
 * allocated.  Nothing unwinds across the boundary: every function returns 0 on success or a negative
 * code (B200PIR_E_*), and b200pir_last_error() returns the message for the calling thread.
 * Concurrent calls on one context are serialised internally (one CUDA stream per context); use one
 * context per host thread / GPU for concurrency.
 */
#ifndef B200PIR_H
#define B200PIR_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200PIR_E_BADARG (-1)
#define B200PIR_E_SHAPE (-2)
#define B200PIR_E_CUDA (-3)
#define B200PIR_E_UNSUPPORTED (-4)

typedef struct b200pir_ctx b200pir_ctx;  /* params + tables + workspace on one GPU */
typedef struct b200pir_db b200pir_db;    /* HBM-resident database                   */
typedef struct b200pir_pp b200pir_pp;    /* HBM-resident PublicParameters of a client */
typedef struct b200pir_dpir b200pir_dpir; /* HBM-resident DoublePIR packed matrix    */

/* The scalar fields of spiral_rs::params::Params that params_from_json_obj reads
 * (lib/spiral-rs/src/util.rs:224-263); poly_len = 2048 and the two CRT moduli are fixed there (:246-247). */
typedef struct {
  uint64_t n, nu_1, nu_2, p, q2_bits, t_gsw, t_conv, t_exp_left, t_exp_right, instances, db_item_size, version;
  int32_t expand_queries; /* 0 = direct_upload */
} b200pir_params;

const char* b200pir_last_error(void);
int b200pir_device_count(void);

/* Params::init (params.rs:224-296): builds NTT tables, Barrett constants, v_neg1 on `device`. */
int b200pir_ctx_create(const b200pir_params* params, int device, b200pir_ctx** out);
void b200pir_ctx_destroy(b200pir_ctx* ctx);
/* Use an externally owned cudaStream_t (e.g. torch's current stream) for all work of this context. */
int b200pir_ctx_set_stream(b200pir_ctx* ctx, void* cuda_stream);
int b200pir_ctx_synchronize(b200pir_ctx* ctx);
/* knobs: "mul_variant" (kernel tiling), "batch" (max queries per database pass: 1, 2, 4, 8 or 16;
 * the IMAD layout uses at most 4), "db_format" (layout of databases created afterwards: -1 = automatic (default): 2 wherever the
 * tcgen05 kernel supports the geometry, else 1; 0 = IMAD, 1 = mma.sync INT8 fragments, 2 = tcgen05 tile images, tc5_kernels.cu), "profile" (0 off, 1 per call,
 * 2 accumulate over calls until set again); A/B switches for kernel variants: "fold_variant", "intt_variant", "imma_variant",
 * "expand_variant" (0 = default everywhere); "coalesce" (1 = default: concurrent single-query callers
 * share database passes, see b200pir_coalesce_stats), "coalesce_window_us" (default 200: how long a batch that directly
 * follows a multi-query batch is held open for the callers of that batch to return; 0 = never), "sparse_fold" (1 = fold like lib/server's sparse server,
 * compute/fold.rs:15-65: an all-zero ciphertext short-cuts the external product; 0 = spiral-rs's dense fold, default); "expand_pair_min_ctas" (expansion rounds with at least this many active
 * ciphertexts use the paired kernel, default 592);
 * unknown keys -> B200PIR_E_BADARG */
int b200pir_ctx_set_option(b200pir_ctx* ctx, const char* key, int64_t value);
/* Size the context's workspace once, up front, for `queries` concurrent queries against a database with `rows_local`
 * second-dimension rows (num_per for an unsharded database): afterwards no entry point allocates device memory for batches up
 * to that size (the workspace otherwise grows on first use; coalesced single-query calls size it for 32 queries).
 * B200PIR_E_CUDA when the device cannot hold it. */
int b200pir_ctx_reserve(b200pir_ctx* ctx, size_t queries, size_t rows_local);
/* params.setup_bytes / query_bytes / response length (params.rs:146-182, server.rs:476-481) */
int b200pir_ctx_sizes(b200pir_ctx* ctx, uint64_t* setup_bytes, uint64_t* query_bytes, uint64_t* response_bytes);

/* ---- database: replaces the `db: &[u64]` argument of process_query (server.rs:650-655) ---------- */
/* Allocates slices*dim0*num_per*2048 words in HBM (zero = every item empty).
 * Multi-GPU row sharding (DESIGN.md): with shard_count = G (a power of two dividing num_per) this GPU holds
 * the second-dimension rows ii = shard_index (mod G); pass 0,1 for the whole database. */
int b200pir_db_create(b200pir_ctx* ctx, uint64_t shard_index, uint64_t shard_count, b200pir_db** out);
void b200pir_db_destroy(b200pir_db* db);
/* Upload one (instance,trial) slice in the reference layout [z][ii][j] (server.rs:263-266). */
int b200pir_db_upload_slice(b200pir_ctx* ctx, b200pir_db* db, uint64_t slice, const uint64_t* words, size_t n_words);
/* Whole db: &[u64] of instances*n^2 slices. */
int b200pir_db_upload(b200pir_ctx* ctx, b200pir_db* db, const uint64_t* words, size_t n_words);
/* load_preprocessed_db_from_file (server.rs:373-386; lib/server/src/db/loading.rs:263-276): `path` holds the native-endian
 * u64 stream of the whole database (slices*dim0*num_per*2048 words, the layout b200pir_db_upload takes); it is streamed
 * to the GPU through a staging buffer. */
int b200pir_db_load_file(b200pir_ctx* ctx, b200pir_db* db, const char* path);
/* load_db_from_seek (server.rs:277-357; lib/server/src/db/loading.rs:192-247): `path` is the RAW database, item i at byte
 * i*db_item_size; chunk c of an item = bytes_per_chunk bytes from i*db_item_size + c*bytes_per_chunk, clipped at the end of
 * the file; conversion (recenter, NTT, pack) on the GPU.  logp == 8 only. */
int b200pir_db_load_raw_file(b200pir_ctx* ctx, b200pir_db* db, const char* path);
/* One preprocessed item polynomial: 2048 packed words (lib/server/src/db/loading.rs:34-41 pack_ntt_poly,
 * :317-359 update_item_raw -> db.upsert(inst_trial*num_items + db_idx)); item_idx = j*num_per + ii. */
int b200pir_db_upsert_item(b200pir_ctx* ctx, b200pir_db* db, uint64_t slice, uint64_t item_idx, const uint64_t* poly);
/* lib/server/src/db/loading.rs:317-359 update_item_raw (the /write and /update-row path): `data` = the raw bucket bytes
 * of item db_idx (at most instances*n^2*bytes_per_chunk, zero padded); chunk c becomes the item polynomial of slice c
 * (convert_pt_to_poly :278-299: coefficient i = byte i, recenter_mod, NTT; pack_ntt_poly :34-41), all on the GPU. */
int b200pir_db_update_item_raw(b200pir_ctx* ctx, b200pir_db* db, uint64_t db_idx, const uint8_t* data, size_t len);
/* lib/server/src/db/loading.rs:361-377 update_many_items (the /update-row body): entries [u32 BE chunk_len][u32 BE db_idx]
 * [chunk_len - 4 raw bytes], back to back; each entry is update_item (:301-315) -> update_item_raw (:317-359).
 * largest_update (may be NULL) receives the longest entry's chunk_len, as the handler reports it.
 * Entries are checked in body order with the codes and messages of b200pir_db_update_item_raw: a truncated length prefix, a
 * chunk_len below 4 or past the end of the body, a chunk_len above 4 + instances*n^2*bytes_per_chunk and a db_idx >= num_items
 * each give B200PIR_E_SHAPE, with every entry before the bad one written and none after it (the reference's serial loop).  The
 * last entry of an item wins.  On a sharded database entries of other GPUs' rows are checked but not written.  The whole body
 * is applied under the context lock and finished before the call returns, so concurrent queries see the database as it was
 * before the call or as the call leaves it, never halfway.
 * Entries are converted and placed in groups of at most 4096 items or 32 MiB of raw bytes (one fused kernel launch each),
 * staged through two pinned buffers owned by the context: they grow on first use, later calls allocate nothing. */
int b200pir_db_update_many_items(b200pir_ctx* ctx, b200pir_db* db, const uint8_t* body, size_t len, uint64_t* largest_update);
/* Synthetic database generated on the GPU: plaintext coefficient = splitmix64(seed, ((slice*items+item)*2048+z)) % p,
 * then recenter_mod / NTT / pack as generate_random_db_and_get_item does (server.rs:223-275). */
int b200pir_db_fill_synthetic(b200pir_ctx* ctx, b200pir_db* db, uint64_t seed);
/* What `db` is: its layout (the "db_format" it was created with, resolved when that was -1), the second-dimension rows
 * this GPU holds, and its size in HBM.  Any out pointer may be NULL. */
int b200pir_db_info(b200pir_db* db, int* format, uint64_t* local_rows, uint64_t* hbm_bytes);
/* lib/server's SparseDb (db/sparse_db.rs:5-47): an item exists once it has been written (upsert / update_item_raw; bulk uploads,
 * file loads and the synthetic fill write every item).  `items` = present items on this GPU, `capacity` = slices x local rows x
 * dim0.  Absent items are zero polynomials in HBM, so results equal the sparse server's sums; on the tcgen05 layout every
 * 32-row x 32-j tile without a present item is neither fetched nor multiplied (multiply_reg_by_sparse_database skips absent
 * items, compute/dot_product.rs:35). */
int b200pir_db_present_items(b200pir_db* db, uint64_t* items, uint64_t* capacity);

/* ---- public parameters: replaces &PublicParameters (client.rs:146-152), all matrices in NTT form ---- */
/* v_packing: num_packing x (n+1) x t_conv ; v_expansion_left: g x 2 x t_exp_left ;
 * v_expansion_right: (stop_round+1) x 2 x t_exp_right or NULL (-> left, server.rs:549) ; v_conversion: 2 x 2 t_conv.
 * Expansion / conversion may be NULL when expand_queries == 0. */
int b200pir_pp_create(b200pir_ctx* ctx, const uint64_t* v_packing, const uint64_t* v_expansion_left,
                      const uint64_t* v_expansion_right, const uint64_t* v_conversion, b200pir_pp** out);
/* PublicParameters::deserialize (client.rs:212-259): data = 32-byte seed || rows 1.. of every matrix (raw u64, native
 * endian) in the order v_packing, v_expansion_left, v_expansion_right (if present), v_conversion; len == setup_bytes.
 * The first rows are regenerated on the GPU from ChaCha20Rng::from_seed(seed) (rand_chacha 0.3.1 keystream order). */
int b200pir_pp_create_from_bytes(b200pir_ctx* ctx, const uint8_t* data, size_t len, b200pir_pp** out);
void b200pir_pp_destroy(b200pir_pp* pp);

/* ---- stage-level entry points (each == one reference function, host buffers) ----------------------- */
/* ntt.rs:67-113 ntt_forward / :212-258 ntt_inverse over `count` polys of [2][2048] u64, in place. */
int b200pir_ntt_forward(b200pir_ctx* ctx, uint64_t* polys, size_t count);
int b200pir_ntt_inverse(b200pir_ctx* ctx, uint64_t* polys, size_t count);
/* Device-resident batch (BASELINE config #5): `count` polys of u32 [2][2048] residues, in place, stream-ordered. */
int b200pir_ntt32_dev(b200pir_ctx* ctx, uint32_t* polys_dev, size_t count, int inverse);
/* BASELINE config #5, poly_len = 4096 (not a size the reference's parameterisation uses, util.rs:246): the same transform
 * definition (ntt.rs:67-113, :212-258) and table construction (ntt.rs:39-65) over the same two moduli.
 * _dev: polys_dev = count x [2][4096] u32 on the device, in place; host variant: count x [2][4096] u64. */
int b200pir_ntt4096_dev(b200pir_ctx* ctx, uint32_t* polys_dev, size_t count, int inverse);
int b200pir_ntt4096(b200pir_ctx* ctx, uint64_t* polys, size_t count, int inverse);
/* poly.rs:613-623 to_ntt / :646-663 from_ntt over `count` polys. */
int b200pir_to_ntt(b200pir_ctx* ctx, uint64_t* out_ntt, const uint64_t* raw, size_t count);
int b200pir_from_ntt(b200pir_ctx* ctx, uint64_t* out_raw, const uint64_t* ntt, size_t count);
/* server.rs:155-221 multiply_reg_by_database on slice `slice`: out = num_per x PolyMatrixNTT(2,1). */
int b200pir_multiply_reg_by_database(b200pir_ctx* ctx, b200pir_db* db, uint64_t slice, const uint64_t* v_firstdim,
                                     uint64_t* out);
/* server.rs:388-427 fold_ciphertexts: v_cts = num x PolyMatrixRaw(2,1) in place (result in v_cts[0]);
 * v_folding / v_folding_neg = log2(num) x PolyMatrixNTT(2, 2 t_gsw).  v_folding_neg may be NULL, meaning
 * get_v_folding_neg(v_folding) as process_query always passes (server.rs:680): the library then uses its
 * fast path, which never materialises the negated matrices (same bytes). */
int b200pir_fold_ciphertexts(b200pir_ctx* ctx, uint64_t* v_cts, size_t num, const uint64_t* v_folding,
                             const uint64_t* v_folding_neg);
/* server.rs:505-523 get_v_folding_neg */
int b200pir_get_v_folding_neg(b200pir_ctx* ctx, uint64_t* out, const uint64_t* v_folding);
/* server.rs:19-121 coefficient_expansion over v = 2^g x PolyMatrixNTT(2,1), in place */
int b200pir_coefficient_expansion(b200pir_ctx* ctx, b200pir_pp* pp, uint64_t* v);
/* server.rs:525-591 expand_query: query ct (PolyMatrixRaw 2x1) -> v_firstdim [z][j][r], v_folding nu_2 x (2 x 2 t_gsw) */
int b200pir_expand_query(b200pir_ctx* ctx, b200pir_pp* pp, const uint64_t* query_ct, uint64_t* out_v_firstdim,
                         uint64_t* out_v_folding);
/* server.rs:429-468 pack (version 0) / lib/server/src/compute/pack.rs:45-98 (version 1):
 * v_ct = n*n x PolyMatrixRaw(2,1) of one instance -> PolyMatrixNTT(n+1, n) */
int b200pir_pack(b200pir_ctx* ctx, b200pir_pp* pp, const uint64_t* v_ct, uint64_t* out_ntt);
/* server.rs:470-503 encode: instances x PolyMatrixRaw(n+1, n) -> response bytes */
int b200pir_encode(b200pir_ctx* ctx, const uint64_t* v_packed_raw, uint8_t* out, size_t* out_len);

/* ---- the drop-in: spiral_rs::server::process_query (server.rs:650-741) ------------------------------- */
/* expand_queries != 0: query_ct = Query.ct (PolyMatrixRaw 2x1), v_buf = v_ct = NULL.
 * expand_queries == 0: query_ct = NULL, v_buf = Query.v_buf ([z][j][r]), v_ct = nu_2 x PolyMatrixRaw(2, 2 t_gsw).
 * out: response_bytes bytes. */
int b200pir_process_query(b200pir_ctx* ctx, b200pir_db* db, b200pir_pp* pp, const uint64_t* query_ct,
                          const uint64_t* v_buf, const uint64_t* v_ct, uint8_t* out, size_t* out_len);
/* Query::deserialize (client.rs:303-315, expand_queries only): data = seed || row 1 of ct; query_ct: PolyMatrixRaw(2,1). */
int b200pir_query_from_bytes(b200pir_ctx* ctx, const uint8_t* data, size_t len, uint64_t* query_ct);
/* process_query on `count` serialized queries (count x query_bytes, back to back); out: count x response_bytes.
 * Replaces Query::deserialize + process_query as lib/server's /private-read handler chains them (bin/server.rs:99-141).
 * Both branches of Query::deserialize (client.rs:303-329): expand_queries != 0 -> seed || row 1 of ct;
 * expand_queries == 0 (direct upload) -> seed || the odd-indexed words of v_buf || rows 1 of the nu_2 v_ct matrices, the
 * seed-derived halves being regenerated on the GPU.  (In direct-upload mode the handler's body is setup || query: pass the
 * first setup_bytes to b200pir_pp_create_from_bytes and the rest here.) */
int b200pir_process_query_bytes(b200pir_ctx* ctx, b200pir_db* db, b200pir_pp* pp, const uint8_t* queries, size_t len,
                                size_t count, uint8_t* out, size_t* out_len_each);
/* `count` queries of DIFFERENT clients in one database pass: pps[i] = the public parameters of the client that sent query_cts[i]
 * (host PolyMatrixRaw(2,1) each; expand_queries only); outs[i] receives response_bytes bytes.  lib/server looks the parameters up
 * per request (bin/server.rs:113-117); the kernels take them per query. */
int b200pir_process_queries(b200pir_ctx* ctx, b200pir_db* db, b200pir_pp* const* pps, const uint64_t* const* query_cts,
                            size_t count, uint8_t* const* outs);
/* Concurrent callers: b200pir_process_query and single-query b200pir_process_query_bytes calls on one context are coalesced —
 * requests that arrive while a batch is running are served together (up to 32) in one database pass by the next caller to
 * find the GPU free; a lone caller is served at once.  Option "coalesce" = 0 restores strictly serial calls.  Counters: */
int b200pir_coalesce_stats(b200pir_ctx* ctx, uint64_t* batches, uint64_t* queries);
/* `count` queries of one client in one call; the database is streamed once per group of up to 4 (IMAD layout)
 * or 16 (INT8 tensor-core layout) queries.
 * queries: count x PolyMatrixRaw(2,1); out: count x response_bytes. */
int b200pir_process_query_batch(b200pir_ctx* ctx, b200pir_db* db, b200pir_pp* pp, const uint64_t* query_cts,
                                size_t count, uint8_t* out, size_t* out_len_each);
/* Device-resident variants for measurement and multi-GPU composition: inputs/outputs are DEVICE pointers
 * and nothing is synchronised (stream-ordered).  query_dev: count x PolyMatrixRaw(2,1) (u64);
 * out_dev: count x response_bytes. */
int b200pir_process_query_batch_dev(b200pir_ctx* ctx, b200pir_db* db, b200pir_pp* pp, const uint64_t* query_cts_dev,
                                    size_t count, uint8_t* out_dev);
/* Multi-GPU row sharding (DESIGN.md "multi-GPU"): stage A = expansion + first dimension + local fold rounds
 * on this GPU's rows; writes this rank's surviving ciphertexts to `partial_dev` as count x slices ciphertexts
 * in residue form (u32 [row(2)][crt(2)][2048] = coefficients mod q0 / q1, 32 KiB each).  Stage B = remaining
 * log2(world) fold rounds + pack + encode over the all-gathered `gathered_dev` ([world][count][slices][2][2][2048]). */
int b200pir_query_stage_a_dev(b200pir_ctx* ctx, b200pir_db* db, b200pir_pp* pp, const uint64_t* query_cts_dev,
                              size_t count, uint32_t* partial_dev);
int b200pir_query_stage_b_dev(b200pir_ctx* ctx, b200pir_pp* pp, const uint32_t* gathered_dev, size_t world,
                              size_t count, uint8_t* out_dev);

/* The same three phases with caller-owned device buffers in between (so a collective can sit between them):
 *   expand:  count queries -> q_expanded_dev (count x dim0 x 2048 x 16 B, the first-dimension operand) and
 *            v_folding_dev (count x nu_2 x 2 x 2 t_gsw x 2 x 2048 u32, NTT form)
 *   first_dim_fold: any `count` expanded queries against this GPU's rows -> partial_dev (count x slices residue-form cts)
 *   finish:  queries [first, first+count) of gathered_dev ([world][total_count][slices][ct]) -> responses; v_folding_dev holds
 *            the folding matrices of exactly those `count` queries. */
int b200pir_expand_queries_dev(b200pir_ctx* ctx, b200pir_pp* pp, const uint64_t* query_cts_dev, size_t count,
                               void* q_expanded_dev, uint32_t* v_folding_dev);
int b200pir_first_dim_fold_dev(b200pir_ctx* ctx, b200pir_db* db, const void* q_expanded_dev, const uint32_t* v_folding_dev,
                               size_t count, uint32_t* partial_dev);
/* The first two phases with the first-dimension operand exchanged as UMMA tile images (tcgen05-layout databases): the rank that
 * expands a group of <= 16 queries also re-tiles it, once (fused with reorient_reg_ciphertexts, util.rs:323-355); the receivers
 * multiply straight from the images.  image_dev: b200pir_query_image_bytes(ctx) bytes per group; partial_dev as above with
 * query index = group * per_group + i. */
size_t b200pir_query_image_bytes(b200pir_ctx* ctx);
int b200pir_expand_queries_images_dev(b200pir_ctx* ctx, b200pir_pp* pp, const uint64_t* query_cts_dev, size_t count, void* image_dev,
                                      uint32_t* v_folding_dev);
int b200pir_first_dim_fold_images_dev(b200pir_ctx* ctx, b200pir_db* db, const void* images_dev, size_t groups, size_t per_group,
                                      const uint32_t* v_folding_dev, uint32_t* partial_dev);
int b200pir_finish_queries_dev(b200pir_ctx* ctx, b200pir_pp* pp, const uint32_t* gathered_dev, size_t world,
                               size_t total_count, size_t first, size_t count, const uint32_t* v_folding_dev,
                               uint8_t* out_dev);

/* Per-stage device time of the last profiled call, in milliseconds, measured with CUDA events on the
 * context's stream.  Enable with b200pir_ctx_set_option(ctx, "profile", 1).
 * out[0..8] = expand, first-dim multiply kernel, from_ntt, fold, pack, encode, total, multiply launches, re-tiling of the query
 * operand for the tensor-core first dimension (k_query_to_tc5 / k_query_to_frag) */
int b200pir_last_stage_ms(b200pir_ctx* ctx, double* out9);
/* ---- peer memory for the multi-GPU exchange (one process per GPU, NVLink) ------------------------------------------------
 * The expanded queries every rank needs (24 MiB per query) are PUSHED into the peers' gather buffers by the copy engines
 * (cudaMemcpyAsync over CUDA-IPC mappings), not all-gathered by SM-resident collective kernels that compete with the
 * compute kernels for SMs.  b200pir_peer_alloc: device buffer + the 64-byte IPC handle to hand to the other ranks (any
 * transport); b200pir_peer_open: map a peer's buffer (handle from ANOTHER process) for access from `device`;
 * b200pir_peer_copy_async: stream-ordered copy between any two device pointers (local or mapped). */
int b200pir_peer_alloc(int device, size_t bytes, void** out_ptr, uint8_t out_handle[64]);
int b200pir_peer_open(int device, const uint8_t handle[64], void** out_ptr);
int b200pir_peer_close(int device, void* mapped_ptr);
int b200pir_peer_free(int device, void* ptr);
int b200pir_peer_copy_async(void* dst, const void* src, size_t bytes, void* cuda_stream);
/* Number of CUDA kernels this library has launched from the calling host thread since load. */
unsigned long long b200pir_kernel_launches(void);

/* ---- DoublePIR: matrix_mul_vec_packed(a, b, basis=10, compression=3) (lib/doublepir/src/matrix/kernels.rs:118-178) */
int b200pir_dpir_create(int device, const uint32_t* a, uint64_t rows, uint64_t cols, b200pir_dpir** out);
/* synthetic a: word(i,k) = low 30 bits of splitmix64(seed, i*cols+k) */
int b200pir_dpir_create_synthetic(int device, uint64_t rows, uint64_t cols, uint64_t seed, b200pir_dpir** out);
/* Offline setup (lib/doublepir/src/doublepir/doublepir.rs:76-108): h_1 = db.data * a_1 and h_2 = h_1' * a_2 as exact 8-bit limb
 * products on the tcgen05 tensor cores (small signed left operand x 32-bit right operand, modulo 2^32), transpose / expand /
 * concat_cols / squish as small kernels.  Host pointers.  db: l x m, entries centred in [-p/2, p/2) as wrapping u32, p <= 2^10;
 * a1: m x n; a2: (l/x) x n; delta = params.delta(), x = db.info.x.  Outputs: db_squished l x ceil(m/3); h1_squished
 * (n delta x) x ceil((l/x)/3); a2_t n x ((l/x) rounded up to a multiple of 3); h2 (n delta x) x n. */
int b200pir_dpir_setup(int device, const uint32_t* db, uint64_t l, uint64_t m, const uint32_t* a1, uint64_t n, const uint32_t* a2,
                       uint32_t p, uint64_t delta, uint64_t x, uint32_t* db_squished, uint32_t* h1_squished, uint32_t* a2_t,
                       uint32_t* h2);
/* `&Matrix * &Matrix` (matrix/ops.rs:169-191) on the same kernel: out (a_rows x b_cols) = a * b mod 2^32, entries of a in [-2^15, 2^15). */
int b200pir_dpir_matmul(int device, const uint32_t* a, uint64_t a_rows, uint64_t a_cols, const uint32_t* b, uint64_t b_cols,
                        uint32_t* out);
void b200pir_dpir_destroy(b200pir_dpir* m);
int b200pir_dpir_set_stream(b200pir_dpir* m, void* cuda_stream);
/* b: 3*cols u32 ; out: rows u32 */
int b200pir_dpir_matvec_packed(b200pir_dpir* m, const uint32_t* b, uint32_t* out);
int b200pir_dpir_matvec_packed_dev(b200pir_dpir* m, const uint32_t* b_dev, uint32_t* out_dev, int variant);
/* same over the row range [row_begin, row_begin+row_count): answer()'s `db.rows(start, batch)` (doublepir.rs:301) */
int b200pir_dpir_matvec_packed_rows(b200pir_dpir* m, uint64_t row_begin, uint64_t row_count, const uint32_t* b, uint32_t* out);
/* The small tail of answer() (doublepir.rs:317-349), host buffers:
 * matrix_mul_transposed_packed (kernels.rs:180-278): out (a_rows x b_rows); b_cols must be 3*a_cols.
 * transpose_expand_concat_cols_squish (matrix/indexing.rs:117-143, basis 10, d 3): out (cols*delta*concat) x ceil((rows/concat)/3). */
int b200pir_dpir_matrix_mul_transposed_packed(int device, const uint32_t* a, uint64_t a_rows, uint64_t a_cols, const uint32_t* b,
                                              uint64_t b_rows, uint64_t b_cols, uint32_t* out);
int b200pir_dpir_transpose_expand_concat_cols_squish(int device, const uint32_t* a, uint64_t rows, uint64_t cols, uint64_t modulus,
                                                     uint64_t delta, uint64_t concat, uint32_t* out, uint64_t* out_rows,
                                                     uint64_t* out_cols);

#ifdef __cplusplus
}
#endif
#endif
