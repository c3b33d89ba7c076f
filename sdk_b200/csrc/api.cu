// C-ABI implementation (include/b200pir.h): contexts, HBM-resident handles and the host-side
// orchestration of spiral_rs::server::process_query (lib/spiral-rs/src/server.rs:650-741) as a
// stream of sm_100a kernel launches.  No CPU fallback exists anywhere on this path: every entry
// point either runs on the GPU or returns an error.
#include "../../include/b200pir.h"
#include "kernels.h"
#include "ntt_tables.hpp"
#include <cstdio>
#include <algorithm>
#include <cmath>
#include <memory>
#include <cstdint>
#include <cstring>
#include <condition_variable>
#include <chrono>
#include <deque>
#include <mutex>
#include <set>
#include <string>
#include <unordered_set>
#include <utility>
#include <vector>

using namespace b200pir;

namespace b200pir {
thread_local unsigned long long g_kernel_launches = 0;

void opt_in_smem_impl(const void* kernel, int bytes) {
  static std::mutex mu;
  static std::set<std::pair<const void*, int>> done;      // (kernel, device) pairs already opted in
  int dev = 0;
  B200_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lk(mu);
  if (done.count({kernel, dev})) return;
  B200_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  done.insert({kernel, dev});
}
}  // namespace b200pir

namespace {

thread_local std::string g_last_error;

using b200pir::tables::build_tables;
using b200pir::tables::invmod;
uint64_t log2_ceil_u64(uint64_t a) { return (uint64_t)std::ceil(std::log2((double)a)); }
int bits_per(int t) {                        // gadget.rs:3-9 with modulus_log2 = 56
  if (t == 56) return 1;
  return 56 / t + 1;
}
const uint64_t kQ2Values[37] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 12289ULL, 12289ULL, 61441ULL, 65537ULL,
                                65537ULL, 520193ULL, 786433ULL, 786433ULL, 3604481ULL, 7340033ULL, 16515073ULL,
                                33292289ULL, 67043329ULL, 132120577ULL, 268369921ULL, 469762049ULL, 1073479681ULL,
                                2013265921ULL, 4293918721ULL, 8588886017ULL, 17175674881ULL, 34359214081ULL,
                                68718428161ULL};   // params.rs:8-46

template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  DevBuf() {}
  explicit DevBuf(size_t count) { alloc(count); }
  void alloc(size_t count) {
    release();
    n = count;
    if (count) B200_CUDA(cudaMalloc(&p, count * sizeof(T)));
  }
  void ensure(size_t count) { if (count > n) alloc(count); }
  void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
  ~DevBuf() { release(); }
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
};

// Bulk writes (update_many_items, update_item_raw, load_raw_file) go through the fused kernel of item_write.cuh in groups of at
// most kWriteGroupItems items, closed once their raw bytes reach kWriteGroupBytes (b200pir.h).
constexpr size_t kWriteGroupItems = 4096;
constexpr size_t kWriteGroupBytes = (size_t)32 << 20;

// One staging buffer of the write path: [ItemWrite x count][raw bytes], pinned on the host and mirrored on the device.  A
// context owns two and alternates, so that the host fills one while the kernel of the previous group reads the other.
struct WriteStage {
  uint8_t* host = nullptr;
  size_t cap = 0;
  DevBuf<uint8_t> dev;
  cudaEvent_t copied = nullptr;     // the last copy out of `host` has finished: it may be refilled
  void ensure(size_t bytes) {
    if (!copied) B200_CUDA(cudaEventCreateWithFlags(&copied, cudaEventDisableTiming));
    B200_CUDA(cudaEventSynchronize(copied));
    if (bytes <= cap) return;
    bytes = std::max(bytes, (size_t)64 << 10);
    if (host) cudaFreeHost(host);
    host = nullptr;
    cap = 0;
    B200_CUDA(cudaHostAlloc(&host, bytes, cudaHostAllocDefault));
    cap = bytes;
    dev.alloc(bytes);
  }
  ~WriteStage() {
    if (host) cudaFreeHost(host);
    if (copied) cudaEventDestroy(copied);
  }
};

enum Stage { ST_EXPAND = 0, ST_MUL, ST_FROMNTT, ST_FOLD, ST_PACK, ST_ENCODE, ST_QIMG /* query operand re-tiling */, ST_COUNT };

}  // namespace

struct b200pir_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = true;
  std::recursive_mutex mu;
  b200pir_params hp;
  // derived (params.rs:116-200)
  int dim0, num_per, slices, trials, g, stop_round, num_packing;
  int bits_gsw, bits_conv, bits_left, bits_right;
  bool has_right;
  uint64_t q2, q1, setup_bytes, query_bytes, response_bytes;
  int q1_bits;
  DevParams dp;
  DevBuf<Twiddle> d_tw;      // fwd0, inv0, fwd1, inv1, inv_lz0, inv_lz1
  DevBuf<Twiddle> d_tw4k;    // same for poly_len 4096 (config #5 sweep), built on first use
  DevBuf<uint32_t> d_neg1;   // [11][2][2048] ntt32 (params.rs:98-107)
  // options
  int mul_variant = 0, max_group = 16, profile = 0;  // max_group: queries per database pass (IMAD path: <= 4)
  int fold_variant = 2;          // k_fold_res_lz at 3 CTAs per SM (default); 3: 2 CTAs per SM (A/B switch)
  int intt_variant = 0;
  int expand_variant = 0;        // wide rounds: 0 paired + residue pipeline (3 CTAs/SM), 2 paired single kernel; 1: never paired
  long pair_min_ctas = 592;      // 4 x 148 SMs
  int sparse_fold = 0;           // 1: lib/server's fold (all-zero ciphertext shortcut, compute/fold.rs:37-43); 0: spiral-rs dense fold
  int imma_variant = 0;          // 0: cp.async-pipelined kernel for 5..8 queries per pass, 1: load-then-use kernel
  int db_format = -1;            // format given to databases created from now on: -1 = automatic (2 where the tcgen05 kernel
                                 // supports the geometry, else 1), 0 = IMAD layout, 1 = mma.sync fragments, 2 = tcgen05 tile images
  DevBuf<uint2> w_qf;            // B operand of the IMMA path (one group of <= 16 queries)
  DevBuf<uint8_t> w_qt;          // B operand of the tcgen05 path (tile images, 16 queries)
  int sm_count = 0;
  // workspace, sized for `ws_queries` queries
  size_t ws_queries = 0, ws_rows = 0;
  DevBuf<uint64_t> w_query;      // [Q][2][2048] raw
  DevBuf<uint32_t> w_v;          // [Q][2^g][2][2][2048]
  DevBuf<uint32_t> w_zflags;     // all-zero flags of the current fold round's ciphertexts ("sparse_fold")
  DevBuf<uint32_t> w_xr;         // [Q][num_in][2][2048] residues of row 0 (paired expansion rounds)
  DevBuf<uint4> w_qdev;          // [Q][dim0][2048]
  DevBuf<uint32_t> w_vfold, w_vfold_neg;   // [Q][nu_2][2][2t][2][2048]
  DevBuf<uint32_t> w_mult;       // [Q][slices][rows][2][2][2048]  NTT form, then residue form in place
  DevBuf<uint32_t> w_cts;        // ping-pong partner of w_mult for the fold rounds (same size)
  const uint32_t* folded = nullptr;   // where the last fold left its survivors
  size_t folded_stride = 0;           // u32 words between consecutive (query, slice) survivors
  DevBuf<uint64_t> w_packed;     // [Q][inst][n+1][n][2048]
  DevBuf<uint8_t> w_resp;        // [Q][response_bytes]
  WriteStage wstage[2];          // staging of the write path, used alternately
  int wnext = 0;
  // Coalescing of concurrent callers ("coalesce", default on): lib/server takes a READ lock around process_query
  // (bin/server.rs:102), so actix workers call it concurrently.  Requests arriving while a batch runs queue up here; the
  // thread that finds no batch in flight becomes the leader and serves everything queued (up to kCoalesceMax) in ONE
  // database pass.  A lone caller is served immediately.  Two refinements for sustained load: a batch larger than one
  // database pass (16 queries) is trimmed to whole passes, the remainder joining the next batch (it would have finished no
  // earlier inside this one); and a leader that follows a multi-query batch by less than 1 ms gives the callers of that batch
  // up to "coalesce_window_us" (default 200) to come back before it starts, so closed-loop clients do not alternate between
  // full and near-empty passes.
  struct Pending {
    b200pir_db* db; b200pir_pp* pp; const uint64_t* query_ct; const uint8_t* query_bytes; uint8_t* out;
    int rc = 0; std::string err; bool done = false;
  };
  static constexpr size_t kCoalesceMax = 32;
  static constexpr size_t kPassQueries = 16;
  int coalesce = 1;
  int coalesce_window_us = 200;
  size_t last_batch = 0;
  std::chrono::steady_clock::time_point last_batch_end{};
  std::mutex qmu;
  std::condition_variable qcv;
  std::deque<Pending*> pending;
  bool leader_active = false;
  unsigned long long coalesced_batches = 0, coalesced_queries = 0;
  // per-query public parameters (PpTable, kernels.h): device arrays [4][pptab_cap] of base pointers; `multi_pps` (host array, one
  // handle per query of the call in flight) is set by the multi-client entry points, otherwise one handle serves every query
  DevBuf<const uint32_t*> d_pptab;
  size_t pptab_cap = 0;
  std::vector<const uint32_t*> h_pptab;          // what d_pptab holds (skip the upload when unchanged)
  b200pir_pp* const* multi_pps = nullptr;
  PpTable pp_table(b200pir_pp* pp, size_t count);
  // profiling
  struct Span { int stage; cudaEvent_t a, b; };
  std::vector<Span> spans;
  std::vector<cudaEvent_t> event_pool;
  size_t event_next = 0;
  int mul_launches = 0;
  double last_ms[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};   // expand, multiply, from_ntt, fold, pack, encode, total, multiply launches, query image

  size_t v_words() const { return ((size_t)1 << g) * 4 * POLY; }
  size_t fold_words() const { return (size_t)hp.nu_2 * 2 * 2 * hp.t_gsw * 2 * POLY; }
  MulGeom geom(int rows) const { return MulGeom{dim0, rows, slices}; }

  cudaEvent_t get_event() {
    if (event_next == event_pool.size()) {
      cudaEvent_t e;
      B200_CUDA(cudaEventCreate(&e));
      event_pool.push_back(e);
    }
    return event_pool[event_next++];
  }
  struct Scope {
    b200pir_ctx* c; int stage; cudaEvent_t a = nullptr;
    Scope(b200pir_ctx* ctx, int st) : c(ctx), stage(st) {
      if (c->profile) { a = c->get_event(); cudaEventRecord(a, c->stream); }
    }
    ~Scope() {
      if (c->profile) { cudaEvent_t b = c->get_event(); cudaEventRecord(b, c->stream); c->spans.push_back({stage, a, b}); }
    }
  };
  // profile == 1: per call; profile == 2: accumulate over calls until the option is set again
  void prof_reset() { if (profile == 2) return; spans.clear(); event_next = 0; mul_launches = 0; }
  void prof_collect() {
    if (!profile) return;
    B200_CUDA(cudaStreamSynchronize(stream));
    for (int i = 0; i < 9; i++) last_ms[i] = 0;
    for (auto& s : spans) {
      float ms = 0;
      cudaEventElapsedTime(&ms, s.a, s.b);
      last_ms[s.stage == ST_QIMG ? 8 : s.stage] += ms;
      last_ms[6] += ms;
    }
    last_ms[7] = mul_launches;
  }
  // buffers of the first dimension / fold / pack only (queries expanded elsewhere)
  void ensure_workspace_lite(size_t queries, size_t rows) {
    w_mult.ensure(queries * slices * rows * 4 * POLY);
    w_cts.ensure(queries * slices * rows * 4 * POLY);
    w_packed.ensure(queries * hp.instances * (hp.n + 1) * hp.n * POLY);
  }
  void ensure_workspace(size_t queries, size_t rows) {
    if (queries <= ws_queries && rows <= ws_rows) return;
    queries = std::max(queries, ws_queries);
    rows = std::max(rows, ws_rows);
    w_query.ensure(queries * 2 * POLY);
    if (hp.expand_queries) w_v.ensure(queries * v_words());
    w_qdev.ensure(queries * (size_t)dim0 * POLY);
    w_vfold.ensure(queries * std::max<size_t>(fold_words(), 1));
    w_vfold_neg.ensure(queries * std::max<size_t>(fold_words(), 1));
    w_mult.ensure(queries * slices * rows * 4 * POLY);
    w_cts.ensure(queries * slices * rows * 4 * POLY);
    w_packed.ensure(queries * hp.instances * (hp.n + 1) * hp.n * POLY);
    w_resp.ensure(queries * response_bytes);
    ws_queries = queries;
    ws_rows = rows;
  }
};

struct b200pir_db {
  b200pir_ctx* ctx;
  Shard shard;
  int rows;                 // local second-dimension rows
  int format = 0;           // 0: d (IMAD layout)  1: f (INT8 MMA fragment order)  2: t (tcgen05 tile images)
  DevBuf<uint4> d;          // [slice][row][dim0/2][2048]
  DevBuf<uint4> f;          // [slice][n][z][mt][ks][limb][lane]
  DevBuf<uint8_t> t;        // format 2: [slice][n][z][mt][ks][4096 B] tile images (tc5_kernels.cu)
  Tc5Geom T;
  ImmaGeom F;
  size_t slice_cells() const { return (size_t)rows * (ctx->dim0 / 2) * POLY; }
  // Presence (lib/server's SparseDb, db/sparse_db.rs:5-47: an item exists once it has been written).  Storage stays dense in HBM
  // (absent = zero polynomial, so every sum is unchanged); what the map buys is COST: on the tcgen05 path whole 32-row x 32-j
  // tiles without a present item are neither fetched nor multiplied (tile_mask, one bit per tile, kept on the device).
  std::vector<uint64_t> present;          // bit ((slice * rows + il) * dim0 + j)
  uint64_t present_count = 0;
  std::vector<uint32_t> h_tile_mask;      // [slice][mt], bit ks
  DevBuf<uint32_t> tile_mask;
  uint64_t capacity() const { return (uint64_t)ctx->slices * rows * ctx->dim0; }
  void presence_init() {
    present.assign((capacity() + 63) / 64, 0);
    present_count = 0;
    h_tile_mask.assign((size_t)ctx->slices * T.mt, 0u);
    tile_mask.alloc(h_tile_mask.size());
    B200_CUDA(cudaMemset(tile_mask.p, 0, h_tile_mask.size() * 4));
  }
  // one item written (stream-ordered update of the device mask word)
  void mark(int slice, int il, int j, cudaStream_t s) {
    const uint64_t bit = ((uint64_t)slice * rows + il) * ctx->dim0 + j;
    if (!((present[bit >> 6] >> (bit & 63)) & 1)) { present[bit >> 6] |= 1ull << (bit & 63); present_count++; }
    const size_t w = (size_t)slice * T.mt + (il >> 5);
    const uint32_t nv = h_tile_mask[w] | (1u << (j >> 5));
    if (nv != h_tile_mask[w]) {
      h_tile_mask[w] = nv;
      B200_CUDA(cudaMemcpyAsync(tile_mask.p + w, &h_tile_mask[w], 4, cudaMemcpyHostToDevice, s));
    }
  }
  // a group of items written into every slice: host bits first, then one copy of the changed tile-mask range per slice
  void mark_many(const ItemWrite* items, size_t count, cudaStream_t s) {
    for (int slice = 0; slice < ctx->slices; slice++) {
      size_t lo = SIZE_MAX, hi = 0;
      for (size_t k = 0; k < count; k++) {
        const uint64_t bit = ((uint64_t)slice * rows + items[k].il) * ctx->dim0 + items[k].j;
        if (!((present[bit >> 6] >> (bit & 63)) & 1)) { present[bit >> 6] |= 1ull << (bit & 63); present_count++; }
        const size_t w = (size_t)slice * T.mt + (items[k].il >> 5);
        const uint32_t nv = h_tile_mask[w] | (1u << (items[k].j >> 5));
        if (nv != h_tile_mask[w]) { h_tile_mask[w] = nv; lo = std::min(lo, w); hi = std::max(hi, w); }
      }
      if (lo <= hi)
        B200_CUDA(cudaMemcpyAsync(tile_mask.p + lo, &h_tile_mask[lo], (hi - lo + 1) * 4, cudaMemcpyHostToDevice, s));
    }
  }
  // a whole slice written at once (bulk upload, file load, synthetic fill): every item of it exists from now on
  void mark_slice(int slice, cudaStream_t s) {
    const uint64_t lo = (uint64_t)slice * rows * ctx->dim0, hi = lo + (uint64_t)rows * ctx->dim0;
    for (uint64_t b = lo; b < hi; b++)
      if (!((present[b >> 6] >> (b & 63)) & 1)) { present[b >> 6] |= 1ull << (b & 63); present_count++; }
    const uint32_t full = T.ks >= 32 ? 0xffffffffu : ((1u << T.ks) - 1u);
    for (int m = 0; m < T.mt; m++) h_tile_mask[(size_t)slice * T.mt + m] = full;
    B200_CUDA(cudaMemcpyAsync(tile_mask.p + (size_t)slice * T.mt, &h_tile_mask[(size_t)slice * T.mt], (size_t)T.mt * 4,
                              cudaMemcpyHostToDevice, s));
  }
};

struct b200pir_pp {
  b200pir_ctx* ctx;
  DevBuf<uint32_t> pack, left, right, conv;    // ntt32
};

PpTable b200pir_ctx::pp_table(b200pir_pp* pp, size_t count) {
  if (count > pptab_cap) {
    pptab_cap = std::max<size_t>(count, 16);
    d_pptab.alloc(4 * pptab_cap);
    h_pptab.clear();
  }
  std::vector<const uint32_t*> h(4 * pptab_cap, nullptr);
  for (size_t i = 0; i < count; i++) {
    const b200pir_pp* p = multi_pps ? multi_pps[i] : pp;
    h[0 * pptab_cap + i] = p->pack.p;
    h[1 * pptab_cap + i] = p->left.p;
    h[2 * pptab_cap + i] = p->right.p ? p->right.p : p->left.p;     // unwrap_or(v_w_left), server.rs:549
    h[3 * pptab_cap + i] = p->conv.p;
  }
  if (h != h_pptab) {
    B200_CUDA(cudaMemcpyAsync(d_pptab.p, h.data(), h.size() * sizeof(const uint32_t*), cudaMemcpyHostToDevice, stream));
    h_pptab = h;
  }
  return PpTable{d_pptab.p, d_pptab.p + pptab_cap, d_pptab.p + 2 * pptab_cap, d_pptab.p + 3 * pptab_cap};
}

struct b200pir_dpir {
  int device;
  std::mutex mu;            // calls on one handle stage through its b / out buffers: serialised
  cudaStream_t stream = nullptr;
  bool own_stream = true;
  uint64_t rows, cols;
  DevBuf<uint32_t> a;
  DevBuf<uint32_t> b, out;
};

namespace {

int fail(const std::exception& e) {
  cudaGetLastError();        // a failed runtime call leaves its code as the "last error": clear it, or the next entry point's check reports it
  g_last_error = e.what();
  const Error* pe = dynamic_cast<const Error*>(&e);
  return pe ? pe->code : B200PIR_E_CUDA;
}
#define API_BEGIN try {
#define API_END                                     \
  }                                                 \
  catch (const std::exception& e) { return fail(e); } \
  return 0;

struct Guard {
  std::lock_guard<std::recursive_mutex> lk;
  explicit Guard(b200pir_ctx* c) : lk(c->mu) { cudaSetDevice(c->device); }
};

// upload u64 NTT-form matrices (words < 2^32) as ntt32
void upload_ntt32(b200pir_ctx* c, DevBuf<uint32_t>& dst, const uint64_t* host, size_t words) {
  dst.alloc(words);
  DevBuf<uint64_t> tmp(words);
  B200_CUDA(cudaMemcpyAsync(tmp.p, host, words * 8, cudaMemcpyHostToDevice, c->stream));
  launch_narrow(dst.p, tmp.p, words, c->stream);
  B200_CUDA(cudaStreamSynchronize(c->stream));
}

// ---- pipeline pieces (all stream-ordered, device pointers)

// server.rs:19-121 over `nq` queries at once (v: [nq][2^g][4][2048], v_stride words apart)
void run_coefficient_expansion(b200pir_ctx* c, b200pir_pp* pp, uint32_t* v, size_t v_stride, int nq, bool all_slots) {
  const auto& hp = c->hp;
  cudaStream_t s = c->stream;
  const int g = c->g;
  const int stop_round = hp.nu_2 > 0 ? c->stop_round : 0;
  const int max_right = hp.nu_2 > 0 ? (int)(hp.t_gsw * hp.nu_2) : 0;
  const PpTable T = c->pp_table(pp, (size_t)nq);
  for (int r = 0; r < g; r++) {
    const int num_in = 1 << r;
    // wide rounds: one CTA per input ciphertext produces both outputs (no scalar-multiply pass, one inverse transform);
    // narrow rounds keep one CTA per output, which halves their latency
    const long active = (long)((stop_round > 0 && r > stop_round) ? num_in / 2 : num_in) * nq;
    const bool pair = c->expand_variant != 1 && active >= c->pair_min_ctas;
    if (!pair) launch_expand_scalar(c->dp, v, v_stride, nq, num_in, c->d_neg1.p + (size_t)r * 2 * POLY, s);
    ExpandRound R;
    R.r = r; R.num_in = num_in; R.stop_round = stop_round; R.max_bits_to_gen_right = max_right;
    R.fill_skipped = all_slots ? 1 : 0;
    R.t_auto = (POLY >> r) + 1;
    R.t_left = (int)hp.t_exp_left; R.bits_left = c->bits_left;
    R.tab_left = T.left; R.off_left = (size_t)r * 2 * hp.t_exp_left * 2 * POLY;
    if (hp.nu_2 > 0 && c->has_right) {
      // v_w_right has stop_round+1 matrices; rounds beyond that never take the right branch for a
      // processed (even) index except r == 0 (server.rs:60-73), so clamp the pointer for safety.
      int rr = r <= c->stop_round ? r : c->stop_round;
      R.t_right = (int)hp.t_exp_right; R.bits_right = c->bits_right;
      R.tab_right = T.right; R.off_right = (size_t)rr * 2 * hp.t_exp_right * 2 * POLY;
    } else {
      R.t_right = R.t_left; R.bits_right = R.bits_left; R.tab_right = T.left; R.off_right = R.off_left;   // unwrap_or(v_w_left), server.rs:549
    }
    if (pair && c->expand_variant == 0) {
      const size_t xr_stride = (size_t)num_in * 2 * POLY;
      c->w_xr.ensure((size_t)nq * xr_stride);
      launch_expand_round_res(c->dp, v, v_stride, c->w_xr.p, xr_stride, nq, R, c->d_neg1.p + (size_t)r * 2 * POLY, s);
    } else if (pair) launch_expand_round_pair(c->dp, v, v_stride, nq, R, c->d_neg1.p + (size_t)r * 2 * POLY, s);
    else launch_expand_round(c->dp, v, v_stride, nq, R, s);
  }
}

// server.rs:525-591 for `nq` queries.  v: [nq][2^g][4][2048]; writes v_fold of every query and the first-dimension operand:
// q_dev (uint4 [query][dim0][2048], reorient_reg_ciphertexts util.rs:323-355) or, when `images` is given (tcgen05 databases),
// the UMMA tile images of groups of 16 queries directly (image g = queries 16g .., tc5_query_bytes apart): no intermediate.
void run_expand_query(b200pir_ctx* c, b200pir_pp* pp, const uint64_t* query_raw, uint32_t* v, uint4* q_dev,
                      uint32_t* v_fold, int nq, uint8_t* images = nullptr) {
  const auto& hp = c->hp;
  cudaStream_t s = c->stream;
  // no clear of v: every slot the query path reads (even slots < 2 dim0, odd slots < 2 t_gsw nu_2) is written by the rounds
  launch_to_ntt_strided(c->dp, v, c->v_words(), query_raw, (size_t)2 * POLY, 2, nq, s);   // v[0] = query.ct.ntt()
  run_coefficient_expansion(c, pp, v, c->v_words(), nq, false);
  const int factor = hp.nu_2 > 0 ? 2 : 1;
  if (images) {
    const Tc5Geom T = make_tc5_geom(c->dim0, 32);
    for (int q0 = 0; q0 < nq; q0 += 16)
      launch_reorient_to_tc5(T, v + (size_t)q0 * c->v_words(), c->v_words(), factor, std::min(16, nq - q0),
                             images + (size_t)(q0 / 16) * tc5_query_bytes(T), s);
  } else {
    launch_reorient(c->geom(c->num_per), q_dev, (size_t)c->dim0 * POLY, v, c->v_words(), nq, factor, s);
  }
  if (hp.nu_2 > 0)
    launch_regev_to_gsw(c->dp, v_fold, c->fold_words(), v, c->v_words(), nq, (int)hp.nu_2, 2, 1, c->pp_table(pp, (size_t)nq).conv,
                        (int)hp.t_gsw, (int)hp.t_conv, c->bits_conv, s);
}

// fold `num` ciphertexts per batch entry with matrices k = k0, k0-1, ...
void run_fold(b200pir_ctx* c, uint64_t* cts, size_t batch, size_t batch_stride, size_t num, int k0,
              const uint32_t* vfold, const uint32_t* vfold_neg, int slices_per_query) {
  const size_t mat = (size_t)2 * 2 * c->hp.t_gsw * 2 * POLY;
  int k = k0;
  for (size_t half = num / 2; half >= 1; half /= 2, k--) {
    launch_fold_round(c->dp, cts, batch, batch_stride, (int)half, vfold + (size_t)k * mat, vfold_neg + (size_t)k * mat,
                      c->fold_words(), slices_per_query, (int)c->hp.t_gsw, c->bits_gsw, c->stream);
  }
}

// Fast path on residue-form ciphertexts: ping-pong between `a` (input of the first round) and `b`.
// Returns the buffer holding the survivors (entry 0 of each batch element).
const uint32_t* run_fold_res(b200pir_ctx* c, uint32_t* a, uint32_t* b, size_t batch, size_t batch_stride, size_t num,
                             int k0, const uint32_t* vfold, int slices_per_query) {
  const size_t mat = (size_t)2 * 2 * c->hp.t_gsw * 2 * POLY;
  int k = k0;
  uint32_t* src = a;
  uint32_t* dst = b;
  uint32_t* zero_flags = nullptr;                      // lib/server's fold shortcut (fold.rs:37-43) when "sparse_fold" is set
  if (c->sparse_fold) {
    c->w_zflags.ensure(batch * num);
    zero_flags = c->w_zflags.p;
  }
  for (size_t half = num / 2; half >= 1; half /= 2, k--) {
    launch_fold_res(c->dp, src, dst, batch, batch_stride, (int)half, vfold + (size_t)k * mat, c->fold_words(),
                    slices_per_query, (int)c->hp.t_gsw, c->bits_gsw, c->fold_variant, zero_flags, c->stream);
    std::swap(src, dst);
  }
  return src;
}

// expansion (or direct upload) for `count` queries already in w_query / w_qdev,w_vfold
void run_prepare(b200pir_ctx* c, b200pir_pp* pp, size_t count, bool images = false) {
  b200pir_ctx::Scope sc(c, ST_EXPAND);
  if (images) c->w_qt.ensure((count + 15) / 16 * tc5_query_bytes(make_tc5_geom(c->dim0, 32)));
  if (c->hp.expand_queries)
    run_expand_query(c, pp, c->w_query.p, c->w_v.p, c->w_qdev.p, c->w_vfold.p, (int)count, images ? c->w_qt.p : nullptr);
  // v_folding_neg (server.rs:680) is not materialised: the fold fast path uses G - C_k implicitly.
}

// first dimension + from_ntt + local fold.  Leaves survivors at w_cts[(qi*slices + slice)*rows*2*POLY].
// `images`: the first-dimension operand already sits as tile images (groups of `per_group` <= 16 queries, one image each)
void run_first_dim_and_fold(b200pir_ctx* c, b200pir_db* db, size_t count, const uint4* qdev = nullptr,
                            const uint32_t* vfold = nullptr, const uint8_t* images = nullptr, size_t per_group = 16) {
  if (!qdev) qdev = c->w_qdev.p;
  if (!vfold) vfold = c->w_vfold.p;
  const int rows = db->rows;
  MulGeom G = c->geom(rows);
  const size_t q_stride = (size_t)c->dim0 * POLY;
  const size_t out_stride = (size_t)c->slices * rows * 4 * POLY;
  if (db->format == 0) {
    {
      b200pir_ctx::Scope sc(c, ST_MUL);
      size_t qi = 0;
      while (qi < count) {
        int nq = 1;
        if (count - qi >= 4 && c->max_group >= 4) nq = 4;
        else if (count - qi >= 2 && c->max_group >= 2) nq = 2;
        launch_multiply(c->dp, G, db->d.p, qdev + qi * q_stride, c->w_mult.p + qi * out_stride, 0, c->slices, nq,
                        q_stride, out_stride, c->mul_variant, c->stream);
        c->mul_launches++;
        qi += nq;
      }
    }
    {
      // server.rs:707-709 from_ntt, minus the CRT lift: inverse NTT of every CRT half in place -> residue form
      b200pir_ctx::Scope sc(c, ST_FROMNTT);
      launch_ntt32(c->dp, c->w_mult.p, count * c->slices * rows * 2, true, c->stream);
    }
  } else if (db->format == 2) {
    // tcgen05 path: same z-major product as the mma.sync path, 16 queries per database pass
    if (!images) c->w_qt.ensure(tc5_query_bytes(db->T));
    const size_t step = images ? per_group : 16;
    for (size_t qi = 0, g = 0; qi < count; qi += step, g++) {
      const int nq = (int)std::min<size_t>(step, count - qi);
      const uint8_t* qt = images ? images + g * tc5_query_bytes(db->T) : c->w_qt.p;
      if (!images) {
        b200pir_ctx::Scope sq(c, ST_QIMG);
        launch_query_to_tc5(db->T, qdev + qi * q_stride, q_stride, nq, c->w_qt.p, c->stream);
      }
      b200pir_ctx::Scope sc(c, ST_MUL);
      launch_multiply_tc5(c->dp, db->T, db->t.p, db->tile_mask.p, qt, c->w_cts.p + qi * out_stride, out_stride, nq, 0, c->slices,
                          c->sm_count, c->stream);
      c->mul_launches++;
    }
    {
      b200pir_ctx::Scope sc(c, ST_FROMNTT);
      launch_intt_from_zmajor(c->dp, db->F, c->w_cts.p, out_stride, c->w_mult.p, (int)count, c->slices, c->intt_variant, c->stream);
    }
  } else {
    // INT8 tensor-core path: z-major product in w_cts (free until the fold starts), then inverse NTT into w_mult
    c->w_qf.ensure(imma_query_cells(db->F));
    const size_t per_pass = (c->max_group >= 16 && imma_supports_16(db->F)) ? 16 : (c->max_group >= 8 ? 8 : 4);
    for (size_t qi = 0; qi < count; qi += per_pass) {
      const int nq = (int)std::min<size_t>(per_pass, count - qi);
      {
        b200pir_ctx::Scope sq(c, ST_QIMG);
        launch_query_to_frag(db->F, qdev + qi * q_stride, q_stride, nq, c->w_qf.p, c->stream);
      }
      {
        b200pir_ctx::Scope sc(c, ST_MUL);
        launch_multiply_imma(c->dp, db->F, db->f.p, c->w_qf.p, c->w_cts.p + qi * out_stride, out_stride, nq, 0, c->slices,
                             c->imma_variant, c->stream);
        c->mul_launches++;
      }
    }
    {
      b200pir_ctx::Scope sc(c, ST_FROMNTT);
      launch_intt_from_zmajor(c->dp, db->F, c->w_cts.p, out_stride, c->w_mult.p, (int)count, c->slices, c->intt_variant, c->stream);
    }
  }
  {
    b200pir_ctx::Scope sc(c, ST_FOLD);
    c->folded = c->w_mult.p;
    c->folded_stride = (size_t)rows * 4 * POLY;
    if (rows > 1)
      c->folded = run_fold_res(c, c->w_mult.p, c->w_cts.p, count * c->slices, (size_t)rows * 4 * POLY, rows,
                               (int)c->hp.nu_2 - 1, vfold, c->slices);
  }
}

// pack + encode for `count` queries whose folded ciphertexts sit at folded + ((qi*slices)+t)*ct_stride
void run_pack_encode(b200pir_ctx* c, b200pir_pp* pp, const uint32_t* folded, size_t ct_stride, size_t count,
                     uint8_t* out_dev) {
  const auto& hp = c->hp;
  const size_t packed_words = (size_t)hp.instances * (hp.n + 1) * hp.n * POLY;
  {
    b200pir_ctx::Scope sc(c, ST_PACK);
    launch_pack(c->dp, c->w_packed.p, packed_words, folded, ct_stride, (size_t)c->slices * ct_stride, (int)count, c->pp_table(pp, count).pack,
                (int)hp.n, (int)hp.instances, (int)hp.t_conv, c->bits_conv, (int)hp.version, c->stream);
  }
  {
    b200pir_ctx::Scope sc(c, ST_ENCODE);
    launch_encode(c->dp, out_dev, c->response_bytes, c->w_packed.p, packed_words, (int)count, (int)hp.n, (int)hp.instances,
                  c->q2, (int)hp.q2_bits, c->q1, c->q1_bits, c->stream);
  }
}

// handles may be used from any context with identical parameters on the same device (one context per host
// thread / CUDA stream sharing one HBM-resident database)
bool same_params(const b200pir_ctx* a, const b200pir_ctx* b) {
  return a == b || (a->device == b->device && std::memcmp(&a->hp, &b->hp, sizeof(b200pir_params)) == 0);
}
void check_db(b200pir_ctx* c, b200pir_db* db) {
  if (!db || !same_params(db->ctx, c)) throw Error(B200PIR_E_BADARG, "db handle was created for different parameters / device");
}
void check_pp(b200pir_ctx* c, b200pir_pp* pp) {
  if (!pp || !same_params(pp->ctx, c)) throw Error(B200PIR_E_BADARG, "pp handle was created for different parameters / device");
}

}  // namespace

extern "C" {

const char* b200pir_last_error(void) { return g_last_error.c_str(); }
int b200pir_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

int b200pir_ctx_create(const b200pir_params* params, int device, b200pir_ctx** out) {
  API_BEGIN
  if (!params || !out) throw Error(B200PIR_E_BADARG, "null argument");
  int ndev = 0;
  B200_CUDA(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) throw Error(B200PIR_E_BADARG, "no such CUDA device (this library has no CPU path)");
  B200_CUDA(cudaSetDevice(device));
  std::unique_ptr<b200pir_ctx> c(new b200pir_ctx());
  c->device = device;
  B200_CUDA(cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device));
  c->hp = *params;
  auto& hp = c->hp;
  if (hp.q2_bits < 14) hp.q2_bits = 14;                       // util.rs:230, params.rs:7
  if (hp.q2_bits > 36) throw Error(B200PIR_E_BADARG, "q2_bits out of range");
  if (hp.instances == 0) hp.instances = 1;
  if (hp.n < 1 || hp.n > 4) throw Error(B200PIR_E_UNSUPPORTED, "n must be 1..4");
  if (hp.nu_1 < 1 || hp.nu_1 > 16 || hp.nu_2 > 16) throw Error(B200PIR_E_BADARG, "nu_1/nu_2 out of range");
  if (hp.version > 1) throw Error(B200PIR_E_BADARG, "unknown version");
  if (hp.p < 2 || (hp.p & (hp.p - 1)) || hp.p > (1u << 20)) throw Error(B200PIR_E_BADARG, "p must be a power of two <= 2^20");
  for (uint64_t t : {hp.t_gsw, hp.t_conv, hp.t_exp_left, hp.t_exp_right})
    if (t < 3 || t > 56)   // t = 2 would mean 29-bit digits: above q, outside the transforms' input range (and no parameter
      throw Error(B200PIR_E_UNSUPPORTED, "gadget dimensions must be in 3..56");   // set of the reference uses it)
  if (hp.db_item_size == 0) hp.db_item_size = hp.instances * hp.n * hp.n * 2048 * log2_ceil_u64(hp.p) / 8;
  c->dim0 = 1 << hp.nu_1;
  c->num_per = 1 << hp.nu_2;
  c->trials = (int)(hp.n * hp.n);
  c->slices = (int)(hp.instances * c->trials);
  c->g = (int)log2_ceil_u64(hp.t_gsw * hp.nu_2 + c->dim0);
  c->stop_round = hp.nu_2 ? (int)log2_ceil_u64(hp.t_gsw * hp.nu_2) : 0;
  if (c->g > 11) throw Error(B200PIR_E_UNSUPPORTED, "expansion needs more than 2048 slots");
  c->num_packing = hp.version == 0 ? (int)hp.n : 2;
  c->has_right = hp.expand_queries && (hp.version == 0 || hp.t_exp_right != hp.t_exp_left);
  c->bits_gsw = bits_per((int)hp.t_gsw);
  c->bits_conv = bits_per((int)hp.t_conv);
  c->bits_left = bits_per((int)hp.t_exp_left);
  c->bits_right = bits_per((int)hp.t_exp_right);
  c->q2 = kQ2Values[hp.q2_bits];
  c->q1 = 4 * hp.p;
  c->q1_bits = (int)log2_ceil_u64(c->q1);
  {
    uint64_t bits = hp.instances * (hp.q2_bits * hp.n * 2048 + (uint64_t)c->q1_bits * hp.n * hp.n * 2048);
    c->response_bytes = ((bits + 63) / 64) * 8;
    uint64_t sz = (uint64_t)c->num_packing * hp.n * hp.t_conv;
    if (hp.expand_queries) {
      uint64_t right = (uint64_t)(c->stop_round + 1) * hp.t_exp_right;
      if (hp.version > 0 && hp.t_exp_left == hp.t_exp_right) right = 0;
      sz += (uint64_t)c->g * hp.t_exp_left + right + 2 * hp.t_conv;
    }
    c->setup_bytes = 32 + sz * 2048 * 8;
    uint64_t qp = hp.expand_queries ? 1 : (uint64_t)c->dim0 + hp.nu_2 * 2 * hp.t_gsw;
    c->query_bytes = 32 + qp * 2048 * 8;
  }
  B200_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  // tables
  const uint64_t q0 = 268369921ULL, q1m = 249561089ULL;            // util.rs:246-247
  std::vector<Twiddle> f0, i0, f1, i1;
  build_tables(q0, f0, i0);
  build_tables(q1m, f1, i1);
  std::vector<Twiddle> l0, l1;                                     // relaxed-range inverse tables (ntt_core.cuh "lz")
  b200pir::tables::build_inverse_table_lz(q0, l0);
  b200pir::tables::build_inverse_table_lz(q1m, l1);
  c->d_tw.alloc(6 * POLY);
  B200_CUDA(cudaMemcpy(c->d_tw.p + 4 * POLY, l0.data(), POLY * sizeof(Twiddle), cudaMemcpyHostToDevice));
  B200_CUDA(cudaMemcpy(c->d_tw.p + 5 * POLY, l1.data(), POLY * sizeof(Twiddle), cudaMemcpyHostToDevice));
  B200_CUDA(cudaMemcpy(c->d_tw.p, f0.data(), POLY * sizeof(Twiddle), cudaMemcpyHostToDevice));
  B200_CUDA(cudaMemcpy(c->d_tw.p + POLY, i0.data(), POLY * sizeof(Twiddle), cudaMemcpyHostToDevice));
  B200_CUDA(cudaMemcpy(c->d_tw.p + 2 * POLY, f1.data(), POLY * sizeof(Twiddle), cudaMemcpyHostToDevice));
  B200_CUDA(cudaMemcpy(c->d_tw.p + 3 * POLY, i1.data(), POLY * sizeof(Twiddle), cudaMemcpyHostToDevice));
  {
    std::vector<Twiddle> lo(2 * 3 * 64);                           // [n][forward, inverse, relaxed-range inverse][64]
    for (int i = 0; i < 64; i++) { lo[(0 * 3 + 0) * 64 + i] = f0[i]; lo[(0 * 3 + 1) * 64 + i] = i0[i]; lo[(0 * 3 + 2) * 64 + i] = l0[i];
                                   lo[(1 * 3 + 0) * 64 + i] = f1[i]; lo[(1 * 3 + 1) * 64 + i] = i1[i]; lo[(1 * 3 + 2) * 64 + i] = l1[i]; }
    upload_poly_constants(lo.data());
    upload_mul_constants(lo.data());
    upload_imma_constants(lo.data());
  }
  DevParams& dp = c->dp;
  dp.q[0] = (uint32_t)q0; dp.q[1] = (uint32_t)q1m;
  dp.cr1[0] = (uint64_t)(((u128)1 << 64) / q0);
  dp.cr1[1] = (uint64_t)(((u128)1 << 64) / q1m);
  dp.modulus = q0 * q1m;
  dp.cr1_mod = (uint64_t)(((u128)1 << 64) / dp.modulus);
  dp.q1_inv_mod_q0 = (uint32_t)invmod(q1m % q0, q0);
  dp.fwd[0] = c->d_tw.p; dp.inv[0] = c->d_tw.p + POLY; dp.fwd[1] = c->d_tw.p + 2 * POLY; dp.inv[1] = c->d_tw.p + 3 * POLY;
  dp.inv_lz[0] = c->d_tw.p + 4 * POLY; dp.inv_lz[1] = c->d_tw.p + 5 * POLY;
  dp.mu58[0] = (uint32_t)(((uint64_t)1 << 58) / q0); dp.mu58[1] = (uint32_t)(((uint64_t)1 << 58) / q1m);
  // v_neg1 (params.rs:98-107): NTT of -(X^{N - 2^i})
  {
    std::vector<uint32_t> h((size_t)NTT_LOG_N * 2 * POLY, 0);
    for (int i = 0; i < NTT_LOG_N; i++) {
      int idx = POLY - (1 << i);
      h[((size_t)i * 2 + 0) * POLY + idx] = (uint32_t)(q0 - 1);
      h[((size_t)i * 2 + 1) * POLY + idx] = (uint32_t)(q1m - 1);
    }
    c->d_neg1.alloc(h.size());
    B200_CUDA(cudaMemcpy(c->d_neg1.p, h.data(), h.size() * 4, cudaMemcpyHostToDevice));
    launch_ntt32(dp, c->d_neg1.p, NTT_LOG_N, false, c->stream);
    B200_CUDA(cudaStreamSynchronize(c->stream));
  }
  B200_CUDA(cudaGetLastError());
  *out = c.release();
  API_END
}

void b200pir_ctx_destroy(b200pir_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  for (auto e : c->event_pool) cudaEventDestroy(e);
  if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
  delete c;
}
int b200pir_ctx_set_stream(b200pir_ctx* c, void* cuda_stream) {
  API_BEGIN
  if (!c) throw Error(B200PIR_E_BADARG, "null ctx");
  Guard gd(c);
  B200_CUDA(cudaStreamSynchronize(c->stream));
  if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
  c->stream = (cudaStream_t)cuda_stream;
  c->own_stream = false;
  API_END
}
int b200pir_ctx_synchronize(b200pir_ctx* c) {
  API_BEGIN
  if (!c) throw Error(B200PIR_E_BADARG, "null ctx");
  Guard gd(c);
  B200_CUDA(cudaStreamSynchronize(c->stream));
  B200_CUDA(cudaGetLastError());
  API_END
}
int b200pir_ctx_reserve(b200pir_ctx* c, size_t queries, size_t rows_local) {
  API_BEGIN
  if (!c) throw Error(B200PIR_E_BADARG, "null ctx");
  if (queries == 0 || queries > 4096 || rows_local == 0 || rows_local > ((size_t)1 << c->hp.nu_2))
    throw Error(B200PIR_E_BADARG, "reserve: 1..4096 queries, 1..num_per rows");
  Guard gd(c);
  B200_CUDA(cudaStreamSynchronize(c->stream));          // buffers may be replaced: nothing in flight may still use them
  c->ensure_workspace(queries, rows_local);
  B200_CUDA(cudaGetLastError());
  API_END
}
int b200pir_ctx_set_option(b200pir_ctx* c, const char* key, int64_t value) {
  API_BEGIN
  if (!c || !key) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  std::string k(key);
  if (k == "mul_variant") c->mul_variant = (int)value;
  else if (k == "batch") { if (value != 1 && value != 2 && value != 4 && value != 8 && value != 16) throw Error(B200PIR_E_BADARG, "batch must be 1, 2, 4, 8 or 16"); c->max_group = (int)value; }
  else if (k == "fold_variant") c->fold_variant = (int)value;
  else if (k == "intt_variant") c->intt_variant = (int)value;
  else if (k == "imma_variant") c->imma_variant = (int)value;
  else if (k == "sparse_fold") c->sparse_fold = value != 0;
  else if (k == "coalesce") c->coalesce = value != 0;
  else if (k == "coalesce_window_us") { if (value < 0 || value > 100000) throw Error(B200PIR_E_BADARG, "coalesce_window_us must be 0..100000"); c->coalesce_window_us = (int)value; }
  else if (k == "expand_variant") c->expand_variant = (int)value;
  else if (k == "expand_pair_min_ctas") c->pair_min_ctas = (long)value;
  else if (k == "db_format") { if (value < -1 || value > 2) throw Error(B200PIR_E_BADARG, "db_format must be -1 (automatic), 0, 1 or 2"); c->db_format = (int)value; }
  else if (k == "profile") {
    if (value < 0 || value > 2) throw Error(B200PIR_E_BADARG, "profile must be 0, 1 or 2");
    c->profile = (int)value;
    c->spans.clear(); c->event_next = 0; c->mul_launches = 0;
  }
  else throw Error(B200PIR_E_BADARG, "unknown option " + k);
  API_END
}
int b200pir_ctx_sizes(b200pir_ctx* c, uint64_t* setup_bytes, uint64_t* query_bytes, uint64_t* response_bytes) {
  API_BEGIN
  if (!c) throw Error(B200PIR_E_BADARG, "null ctx");
  if (setup_bytes) *setup_bytes = c->setup_bytes;
  if (query_bytes) *query_bytes = c->query_bytes;
  if (response_bytes) *response_bytes = c->response_bytes;
  API_END
}

// ---------------------------------------------------------------- database
int b200pir_db_create(b200pir_ctx* c, uint64_t shard_index, uint64_t shard_count, b200pir_db** out) {
  API_BEGIN
  if (!c || !out) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  if (shard_count == 0) { shard_count = 1; shard_index = 0; }
  if (shard_index >= shard_count || (shard_count & (shard_count - 1)) || (uint64_t)c->num_per % shard_count)
    throw Error(B200PIR_E_BADARG, "shard_count must be a power of two dividing num_per");
  std::unique_ptr<b200pir_db> db(new b200pir_db());
  db->ctx = c;
  db->shard = Shard{(int)shard_index, (int)shard_count};
  db->rows = c->num_per / (int)shard_count;
  db->F = make_imma_geom(c->dim0, db->rows);
  db->T = make_tc5_geom(c->dim0, db->rows);
  db->format = c->db_format >= 0 ? c->db_format : (tc5_supported(db->T) ? 2 : 1);
  db->presence_init();
  if (db->format == 0) {
    size_t cells = (size_t)c->slices * db->slice_cells();
    db->d.alloc(cells);
    B200_CUDA(cudaMemsetAsync(db->d.p, 0, cells * sizeof(uint4), c->stream));
  } else if (db->format == 2) {
    if (!tc5_supported(db->T)) throw Error(B200PIR_E_UNSUPPORTED, "db_format 2: dim0 too large for the tcgen05 kernel");
    size_t bytes = tc5_db_bytes(db->T, c->slices);
    db->t.alloc(bytes);
    B200_CUDA(cudaMemsetAsync(db->t.p, 0, bytes, c->stream));
  } else {
    size_t cells = imma_db_cells(db->F, c->slices);
    db->f.alloc(cells);
    B200_CUDA(cudaMemsetAsync(db->f.p, 0, cells * sizeof(uint4), c->stream));
  }
  B200_CUDA(cudaStreamSynchronize(c->stream));
  *out = db.release();
  API_END
}
void b200pir_db_destroy(b200pir_db* db) {
  if (!db) return;
  cudaSetDevice(db->ctx->device);
  delete db;
}
extern "C++" {
namespace {
// One slice in the reference's z-major layout, delivered chunk by chunk: fetch(word_offset, n_words) returns a host pointer
// to that range of the slice (valid until the next call).
template <typename Fetch>
void upload_slice_impl(b200pir_ctx* c, b200pir_db* db, uint64_t slice, Fetch fetch) {
  // reference layout is z-major: stage a range of z at a time (<= 64 MiB)
  const size_t per_z = (size_t)c->dim0 * c->num_per;
  int zc = (int)std::max<size_t>(1, std::min<size_t>(POLY, ((size_t)64 << 20) / (per_z * 8)));
  DevBuf<uint64_t> stage(per_z * zc);
  MulGeom G = c->geom(db->rows);
  DevBuf<uint4> tmp;
  uint4* dst;
  if (db->format == 0) dst = db->d.p + (size_t)slice * db->slice_cells();
  else { tmp.alloc(db->slice_cells()); dst = tmp.p; }
  for (int z0 = 0; z0 < POLY; z0 += zc) {
    int cur = std::min(zc, POLY - z0);
    const uint64_t* src = fetch((size_t)z0 * per_z, per_z * cur);
    B200_CUDA(cudaMemcpyAsync(stage.p, src, per_z * cur * 8, cudaMemcpyHostToDevice, c->stream));
    launch_db_retile_chunk(G, db->shard, dst, stage.p, z0, cur, c->stream);
    B200_CUDA(cudaStreamSynchronize(c->stream));
  }
  if (db->format == 1) {
    launch_db_to_frag(db->F, tmp.p, db->f.p, (int)slice, c->stream);
    B200_CUDA(cudaStreamSynchronize(c->stream));
  } else if (db->format == 2) {
    launch_db_to_tc5(db->T, tmp.p, db->t.p, (int)slice, c->stream);
    B200_CUDA(cudaStreamSynchronize(c->stream));
  }
  db->mark_slice((int)slice, c->stream);
  B200_CUDA(cudaStreamSynchronize(c->stream));
  B200_CUDA(cudaGetLastError());
}
}  // namespace
}  // extern "C++"

int b200pir_db_upload_slice(b200pir_ctx* c, b200pir_db* db, uint64_t slice, const uint64_t* words, size_t n_words) {
  API_BEGIN
  if (!c || !words) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  check_db(c, db);
  const size_t slice_words = (size_t)c->dim0 * c->num_per * POLY;
  if (slice >= (uint64_t)c->slices) throw Error(B200PIR_E_SHAPE, "slice out of range");
  if (n_words != slice_words) throw Error(B200PIR_E_SHAPE, "slice must hold dim0*num_per*2048 words");
  upload_slice_impl(c, db, slice, [&](size_t off, size_t) { return words + off; });
  API_END
}
// load_preprocessed_db_from_file (lib/spiral-rs/src/server.rs:373-386, lib/server/src/db/loading.rs:263-276): the file is the
// native-endian u64 stream of the whole `db: &[u64]`; it is streamed through a 64 MiB staging buffer, never held in RAM.
int b200pir_db_load_file(b200pir_ctx* c, b200pir_db* db, const char* path) {
  API_BEGIN
  if (!c || !path) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  check_db(c, db);
  const size_t slice_words = (size_t)c->dim0 * c->num_per * POLY;
  struct Closer { FILE* f; ~Closer() { if (f) fclose(f); } } file{fopen(path, "rb")};
  if (!file.f) throw Error(B200PIR_E_BADARG, std::string("cannot open ") + path);
  if (fseeko(file.f, 0, SEEK_END)) throw Error(B200PIR_E_BADARG, "cannot seek in the database file");
  const off_t bytes = ftello(file.f);
  if (bytes < 0 || (uint64_t)bytes != (uint64_t)slice_words * c->slices * 8)
    throw Error(B200PIR_E_SHAPE, "database file must hold slices*dim0*num_per*2048 u64 words");
  std::vector<uint64_t> buf;
  for (int s = 0; s < c->slices; s++) {
    upload_slice_impl(c, db, (uint64_t)s, [&](size_t off, size_t n) -> const uint64_t* {
      buf.resize(n);
      if (fseeko(file.f, (off_t)(((size_t)s * slice_words + off) * 8), SEEK_SET) || fread(buf.data(), 8, n, file.f) != n)
        throw Error(B200PIR_E_SHAPE, "short read from the database file");
      return buf.data();
    });
  }
  API_END
}
int b200pir_db_upload(b200pir_ctx* c, b200pir_db* db, const uint64_t* words, size_t n_words) {
  if (!c) { g_last_error = "null ctx"; return B200PIR_E_BADARG; }
  const size_t slice_words = (size_t)c->dim0 * c->num_per * POLY;
  if (n_words != slice_words * c->slices) { g_last_error = "db must hold slices*dim0*num_per*2048 words"; return B200PIR_E_SHAPE; }
  for (int s = 0; s < c->slices; s++) {
    int rc = b200pir_db_upload_slice(c, db, s, words + (size_t)s * slice_words, slice_words);
    if (rc) return rc;
  }
  return 0;
}
int b200pir_db_upsert_item(b200pir_ctx* c, b200pir_db* db, uint64_t slice, uint64_t item_idx, const uint64_t* poly) {
  API_BEGIN
  if (!c || !poly) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  check_db(c, db);
  if (slice >= (uint64_t)c->slices || item_idx >= (uint64_t)c->dim0 * c->num_per) throw Error(B200PIR_E_SHAPE, "index out of range");
  int ii = (int)(item_idx % c->num_per), j = (int)(item_idx / c->num_per);
  if (ii % db->shard.count != db->shard.index) return 0;           // row lives on another GPU
  DevBuf<uint64_t> tmp(POLY);
  B200_CUDA(cudaMemcpyAsync(tmp.p, poly, POLY * 8, cudaMemcpyHostToDevice, c->stream));
  if (db->format == 0) launch_db_upsert(c->geom(db->rows), db->d.p, (int)slice, ii / db->shard.count, j, tmp.p, c->stream);
  else if (db->format == 2) launch_db_upsert_tc5(db->T, db->t.p, (int)slice, ii / db->shard.count, j, tmp.p, c->stream);
  else launch_db_upsert_frag(db->F, db->f.p, (int)slice, ii / db->shard.count, j, tmp.p, c->stream);
  db->mark((int)slice, ii / db->shard.count, j, c->stream);
  // the host RwLock gives upserts exclusive access (bin/server.rs:35,49): finish before returning
  B200_CUDA(cudaStreamSynchronize(c->stream));
  API_END
}
extern "C++" {
namespace {
// bytes_per_chunk of the raw write paths (convert_pt_to_poly asserts logp == 8, loading.rs:291; chunks fit a polynomial)
size_t write_chunk_bytes(b200pir_ctx* c) {
  if (c->hp.p != 256) throw Error(B200PIR_E_UNSUPPORTED, "convert_pt_to_poly asserts logp == 8 (loading.rs:291)");
  const size_t chunks = (size_t)c->slices;
  const size_t bpc = (c->hp.db_item_size + chunks - 1) / chunks;            // params.bytes_per_chunk()
  if (bpc > (size_t)POLY) throw Error(B200PIR_E_SHAPE, "bytes_per_chunk exceeds poly_len");           // server.rs:292
  return bpc;
}
// One group of distinct items (their raw bytes: `data_bytes` filled by fill(dst); items[k].off relative to dst) converted and
// placed by one launch of the fused kernel, staged through the context's next pinned / device buffer pair.  Stream-ordered:
// the caller synchronises.
template <typename Fill>
void write_group(b200pir_ctx* c, b200pir_db* db, const std::vector<ItemWrite>& items, size_t data_bytes, Fill fill) {
  if (items.empty()) return;
  WriteStage& st = c->wstage[c->wnext];
  c->wnext ^= 1;
  const size_t head = (items.size() * sizeof(ItemWrite) + 15) & ~(size_t)15;
  st.ensure(head + data_bytes);
  std::memcpy(st.host, items.data(), items.size() * sizeof(ItemWrite));
  fill(st.host + head);
  B200_CUDA(cudaMemcpyAsync(st.dev.p, st.host, head + data_bytes, cudaMemcpyHostToDevice, c->stream));
  B200_CUDA(cudaEventRecord(st.copied, c->stream));
  const ItemWrite* d_items = reinterpret_cast<const ItemWrite*>(st.dev.p);
  const uint8_t* d_data = st.dev.p + head;
  const int bpc = (int)write_chunk_bytes(c), count = (int)items.size();
  if (db->format == 0) launch_write_items(c->dp, c->geom(db->rows), db->d.p, c->slices, d_items, count, d_data, bpc, c->hp.p, c->stream);
  else if (db->format == 2) launch_write_items(c->dp, db->T, db->t.p, c->slices, d_items, count, d_data, bpc, c->hp.p, c->stream);
  else launch_write_items(c->dp, db->F, db->f.p, c->slices, d_items, count, d_data, bpc, c->hp.p, c->stream);
  B200_CUDA(cudaGetLastError());
}
uint32_t load_be32(const uint8_t* p) { return ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | p[3]; }
}  // namespace
}  // extern "C++"

// lib/server/src/db/loading.rs:361-377 update_many_items: the entries are checked and applied in body order; on a malformed
// entry everything before it stays written.  Entries are gathered into groups (kWriteGroupItems / kWriteGroupBytes); within a
// group only the last entry of an item is converted (the reference's serial loop leaves exactly that one), groups run in
// order on one stream, so the last entry of an item wins across groups too.
int b200pir_db_update_many_items(b200pir_ctx* c, b200pir_db* db, const uint8_t* body, size_t len, uint64_t* largest_update) {
  API_BEGIN
  if (!c || (!body && len)) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  check_db(c, db);
  const size_t bpc = write_chunk_bytes(c);
  const size_t max_data = (size_t)c->slices * bpc;
  const uint64_t num_items = (uint64_t)c->dim0 * c->num_per;
  struct Entry { size_t off; uint32_t len, idx; };
  std::vector<Entry> group;
  size_t group_bytes = 0;
  std::vector<ItemWrite> items;
  std::vector<size_t> src;                                                  // body offset of items[k]'s bytes
  std::unordered_set<uint32_t> seen;
  auto flush = [&]() {
    items.clear();
    src.clear();
    seen.clear();
    size_t bytes = 0;
    for (size_t k = group.size(); k-- > 0;) {                               // last occurrence first
      const Entry& e = group[k];
      if (!seen.insert(e.idx).second) continue;
      const int ii = (int)(e.idx % c->num_per), j = (int)(e.idx / c->num_per);
      items.push_back(ItemWrite{(uint32_t)bytes, e.len, (uint32_t)(ii / db->shard.count), (uint32_t)j});
      src.push_back(e.off);
      bytes += e.len;
    }
    write_group(c, db, items, bytes, [&](uint8_t* dst) {
      for (size_t k = 0; k < items.size(); k++) std::memcpy(dst + items[k].off, body + src[k], items[k].len);
    });
    db->mark_many(items.data(), items.size(), c->stream);
    group.clear();
    group_bytes = 0;
  };
  std::string err;
  uint64_t largest = 0;
  size_t offs = 0;
  while (offs < len) {
    if (len - offs < 4) { err = "truncated entry length"; break; }
    const uint32_t chunk_len = load_be32(body + offs);
    if (chunk_len > len - offs - 4) { err = "entry runs past the end of the body"; break; }
    largest = std::max<uint64_t>(largest, chunk_len);
    if (chunk_len > 4 + max_data) { err = "update longer than instances*n^2*bytes_per_chunk"; break; }   // loading.rs:308-310
    if (chunk_len < 4) { err = "entry shorter than its db_idx"; break; }
    const uint32_t idx = load_be32(body + offs + 4);
    if (idx >= num_items) { err = "bad db idx"; break; }                                               // loading.rs:333-340
    if ((idx % c->num_per) % db->shard.count == (uint64_t)db->shard.index) {   // else the row lives on another GPU
      group.push_back(Entry{offs + 8, chunk_len - 4, idx});
      group_bytes += chunk_len - 4;
      if (group.size() == kWriteGroupItems || group_bytes >= kWriteGroupBytes) flush();
    }
    offs += 4 + (size_t)chunk_len;
  }
  flush();
  // the host RwLock gives writers exclusive access (bin/server.rs:31-43): readers see the body applied up to `err`, never less
  B200_CUDA(cudaStreamSynchronize(c->stream));
  if (!err.empty()) throw Error(B200PIR_E_SHAPE, err);
  if (largest_update) *largest_update = largest;
  API_END
}

int b200pir_db_update_item_raw(b200pir_ctx* c, b200pir_db* db, uint64_t db_idx, const uint8_t* data, size_t len) {
  API_BEGIN
  if (!c || (!data && len)) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  check_db(c, db);
  const size_t bpc = write_chunk_bytes(c);
  if (len > (size_t)c->slices * bpc) throw Error(B200PIR_E_SHAPE, "update longer than instances*n^2*bytes_per_chunk");   // loading.rs:308-310
  if (db_idx >= (uint64_t)c->dim0 * c->num_per) throw Error(B200PIR_E_SHAPE, "bad db idx");                      // loading.rs:333-340
  const int ii = (int)(db_idx % c->num_per), j = (int)(db_idx / c->num_per);
  if (ii % db->shard.count != db->shard.index) return 0;                      // row lives on another GPU
  const std::vector<ItemWrite> items{ItemWrite{0, (uint32_t)len, (uint32_t)(ii / db->shard.count), (uint32_t)j}};
  write_group(c, db, items, len, [&](uint8_t* dst) { if (len) std::memcpy(dst, data, len); });
  db->mark_many(items.data(), 1, c->stream);
  B200_CUDA(cudaStreamSynchronize(c->stream));                                // writers hold the host write lock
  API_END
}

// load_db_from_seek (lib/spiral-rs/src/server.rs:277-357; lib/server/src/db/loading.rs:192-247): `path` is the raw database,
// item i at byte i * db_item_size.  Chunk c of item i is the bytes_per_chunk bytes at i * db_item_size + c * bytes_per_chunk,
// clipped at the end of the FILE (as the reference's read does), each byte one plaintext coefficient; items past the end
// of the file are zero polynomials.  So item i is the update_item_raw of the file's bytes [i * db_item_size, + chunks *
// bytes_per_chunk), clipped at its end: one read per group of items, whose ranges may overlap, converted and placed by the
// fused kernel.
int b200pir_db_load_raw_file(b200pir_ctx* c, b200pir_db* db, const char* path) {
  API_BEGIN
  if (!c || !path) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  check_db(c, db);
  const size_t bpc = write_chunk_bytes(c);
  const size_t span = (size_t)c->slices * bpc, isz = c->hp.db_item_size;
  struct Closer { FILE* f; ~Closer() { if (f) fclose(f); } } file{fopen(path, "rb")};
  if (!file.f) throw Error(B200PIR_E_BADARG, std::string("cannot open ") + path);
  if (fseeko(file.f, 0, SEEK_END)) throw Error(B200PIR_E_BADARG, "cannot seek in the database file");
  const off_t fbytes = ftello(file.f);
  if (fbytes < 0) throw Error(B200PIR_E_BADARG, "cannot size the database file");
  const size_t flen = (size_t)fbytes;
  const size_t num_items = (size_t)c->dim0 * c->num_per;
  const size_t group = std::max<size_t>(1, std::min(kWriteGroupItems, (kWriteGroupBytes - std::min(span, kWriteGroupBytes)) / std::max<size_t>(isz, 1) + 1));
  std::vector<ItemWrite> items;
  for (size_t i0 = 0; i0 < num_items; i0 += group) {
    const size_t cnt = std::min(group, num_items - i0);
    const size_t lo = std::min(i0 * isz, flen), hi = std::min((i0 + cnt - 1) * isz + span, flen);
    items.clear();
    for (size_t k = 0; k < cnt; k++) {
      const size_t idx = i0 + k, pos = idx * isz;
      const int ii = (int)(idx % c->num_per), j = (int)(idx / c->num_per);
      if (ii % db->shard.count != db->shard.index) continue;                  // row lives on another GPU
      const size_t have = pos < flen ? std::min(span, flen - pos) : 0;
      items.push_back(ItemWrite{(uint32_t)(have ? pos - lo : 0), (uint32_t)have, (uint32_t)(ii / db->shard.count), (uint32_t)j});
    }
    write_group(c, db, items, hi - lo, [&](uint8_t* dst) {
      if (hi > lo && (fseeko(file.f, (off_t)lo, SEEK_SET) || fread(dst, 1, hi - lo, file.f) != hi - lo))
        throw Error(B200PIR_E_SHAPE, "short read from the database file");
    });
  }
  for (int s = 0; s < c->slices; s++) db->mark_slice(s, c->stream);            // load_db_from_seek builds a dense database
  B200_CUDA(cudaStreamSynchronize(c->stream));
  B200_CUDA(cudaGetLastError());
  API_END
}

int b200pir_db_present_items(b200pir_db* db, uint64_t* items, uint64_t* capacity) {
  API_BEGIN
  if (!db) throw Error(B200PIR_E_BADARG, "null db");
  if (items) *items = db->present_count;
  if (capacity) *capacity = db->capacity();
  API_END
}
int b200pir_db_info(b200pir_db* db, int* format, uint64_t* local_rows, uint64_t* hbm_bytes) {
  API_BEGIN
  if (!db) throw Error(B200PIR_E_BADARG, "null db");
  if (format) *format = db->format;
  if (local_rows) *local_rows = (uint64_t)db->rows;
  if (hbm_bytes) *hbm_bytes = (uint64_t)(db->d.n * sizeof(uint4) + db->f.n * sizeof(uint4) + db->t.n);
  API_END
}
int b200pir_db_fill_synthetic(b200pir_ctx* c, b200pir_db* db, uint64_t seed) {
  API_BEGIN
  if (!c) throw Error(B200PIR_E_BADARG, "null ctx");
  Guard gd(c);
  check_db(c, db);
  MulGeom G = c->geom(db->rows);
  // keep each launch's grid below 2^31 CTAs
  size_t per_slice = (size_t)db->rows * (c->dim0 / 2);
  int step = (int)std::max<size_t>(1, std::min<size_t>(c->slices, ((size_t)1 << 30) / per_slice));
  if (db->format == 0) {
    for (int s0 = 0; s0 < c->slices; s0 += step)
      launch_db_synth(c->dp, G, db->shard, db->d.p, seed, c->hp.p, s0, std::min(step, c->slices - s0), c->stream);
  } else {
    // build each slice in the IMAD layout in a scratch buffer, then re-tile it into fragment order
    DevBuf<uint4> tmp(db->slice_cells());
    for (int s0 = 0; s0 < c->slices; s0++) {
      launch_db_synth(c->dp, G, db->shard, tmp.p - (size_t)s0 * db->slice_cells(), seed, c->hp.p, s0, 1, c->stream);
      if (db->format == 2) launch_db_to_tc5(db->T, tmp.p, db->t.p, s0, c->stream);
      else launch_db_to_frag(db->F, tmp.p, db->f.p, s0, c->stream);
    }
  }
  for (int s0 = 0; s0 < c->slices; s0++) db->mark_slice(s0, c->stream);
  B200_CUDA(cudaStreamSynchronize(c->stream));
  B200_CUDA(cudaGetLastError());
  API_END
}

// ---------------------------------------------------------------- public parameters
int b200pir_pp_create(b200pir_ctx* c, const uint64_t* v_packing, const uint64_t* left, const uint64_t* right,
                      const uint64_t* conv, b200pir_pp** out) {
  API_BEGIN
  if (!c || !out || !v_packing) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  const auto& hp = c->hp;
  std::unique_ptr<b200pir_pp> pp(new b200pir_pp());
  pp->ctx = c;
  const size_t W = 2 * POLY;
  upload_ntt32(c, pp->pack, v_packing, (size_t)c->num_packing * (hp.n + 1) * hp.t_conv * W);
  if (hp.expand_queries) {
    if (!left || !conv) throw Error(B200PIR_E_BADARG, "expansion parameters missing");
    upload_ntt32(c, pp->left, left, (size_t)c->g * 2 * hp.t_exp_left * W);
    if (c->has_right) {
      if (!right) throw Error(B200PIR_E_BADARG, "v_expansion_right missing");
      upload_ntt32(c, pp->right, right, (size_t)(c->stop_round + 1) * 2 * hp.t_exp_right * W);
    }
    upload_ntt32(c, pp->conv, conv, (size_t)2 * 2 * hp.t_conv * W);
  }
  *out = pp.release();
  API_END
}

namespace {
// One group of serialized matrices (client.rs:55-80): `count` raw matrices rows x cols; row 0 regenerated from the seed's
// keystream (u64 position `word`), rows 1.. copied from the byte stream.  Result: NTT form, ntt32 layout, in `dst`.
void deserialize_group(b200pir_ctx* c, DevBuf<uint32_t>& dst, const uint8_t* seed, const uint8_t*& data, uint64_t& word,
                       size_t count, size_t rows, size_t cols) {
  const size_t row_words = cols * POLY, mat_words = rows * row_words, rest = (rows - 1) * row_words;
  DevBuf<uint64_t> raw(count * mat_words);
  launch_chacha_first_rows(raw.p, seed, word, (uint32_t)count, (uint32_t)row_words, mat_words, c->dp.modulus, c->stream);
  word += count * row_words;
  for (size_t i = 0; i < count; i++) {
    B200_CUDA(cudaMemcpyAsync(raw.p + i * mat_words + row_words, data, rest * 8, cudaMemcpyHostToDevice, c->stream));
    data += rest * 8;
  }
  dst.alloc(count * mat_words * 2);
  launch_to_ntt(c->dp, dst.p, raw.p, count * rows * cols, c->stream);
  B200_CUDA(cudaStreamSynchronize(c->stream));
}
}  // namespace

// PublicParameters::deserialize (client.rs:212-259)
int b200pir_pp_create_from_bytes(b200pir_ctx* c, const uint8_t* data, size_t len, b200pir_pp** out) {
  API_BEGIN
  if (!c || !out || !data) throw Error(B200PIR_E_BADARG, "null argument");
  if (len != c->setup_bytes) throw Error(B200PIR_E_SHAPE, "setup data: expected " + std::to_string(c->setup_bytes) + " bytes");
  Guard gd(c);
  const auto& hp = c->hp;
  std::unique_ptr<b200pir_pp> pp(new b200pir_pp());
  pp->ctx = c;
  const uint8_t* seed = data;
  const uint8_t* cur = data + 32;
  uint64_t word = 0;
  deserialize_group(c, pp->pack, seed, cur, word, (size_t)c->num_packing, hp.n + 1, hp.t_conv);
  if (hp.expand_queries) {
    deserialize_group(c, pp->left, seed, cur, word, (size_t)c->g, 2, hp.t_exp_left);
    if (c->has_right) deserialize_group(c, pp->right, seed, cur, word, (size_t)c->stop_round + 1, 2, hp.t_exp_right);
    deserialize_group(c, pp->conv, seed, cur, word, 1, 2, 2 * hp.t_conv);
  }
  if ((size_t)(cur - data) != len) throw Error(B200PIR_E_SHAPE, "setup data: trailing bytes");
  *out = pp.release();
  API_END
}

namespace {
// Query::deserialize, expand_queries branch (client.rs:303-315): `count` serialized queries -> [count] PolyMatrixRaw(2,1) on device
void deserialize_queries(b200pir_ctx* c, const uint8_t* data, size_t count, uint64_t* dst_dev) {
  for (size_t i = 0; i < count; i++) {
    const uint8_t* q = data + i * c->query_bytes;
    launch_chacha_first_rows(dst_dev + i * 2 * POLY, q, 0, 1, POLY, 2 * POLY, c->dp.modulus, c->stream);
    B200_CUDA(cudaMemcpyAsync(dst_dev + i * 2 * POLY + POLY, q + 32, POLY * 8, cudaMemcpyHostToDevice, c->stream));
  }
}
// Query::deserialize, direct-upload branch (client.rs:316-327): one serialized query -> the device-format first-dimension
// operand (q_dev) and the NTT-form folding matrices (v_fold) of workspace slot `slot`.
// Keystream order (interleave_rng_data :107-131, deserialize_vec_polymatrix_rng :81-93): 2048 words per first-dimension
// ciphertext (its row 0), then the first rows (2 t_gsw polynomials) of the nu_2 GSW matrices.
void deserialize_query_direct(b200pir_ctx* c, const uint8_t* q, size_t slot) {
  const size_t dim0 = (size_t)c->dim0, t2 = 2 * c->hp.t_gsw, nu2 = c->hp.nu_2;
  cudaStream_t s = c->stream;
  // row 0 of every first-dimension ciphertext: a raw 1 x 1 "matrix" per ciphertext (row 1 of sigma stays zero and is never used)
  DevBuf<uint64_t> sig_raw(dim0 * POLY);
  DevBuf<uint32_t> sig_ntt(dim0 * 2 * POLY);
  launch_chacha_first_rows(sig_raw.p, q, 0, (uint32_t)dim0, POLY, POLY, c->dp.modulus, s);
  launch_to_ntt(c->dp, sig_ntt.p, sig_raw.p, dim0, s);
  DevBuf<uint64_t> wire(dim0 * POLY);
  B200_CUDA(cudaMemcpyAsync(wire.p, q + 32, dim0 * POLY * 8, cudaMemcpyHostToDevice, s));
  launch_direct_query_to_dev(c->w_qdev.p + slot * dim0 * POLY, sig_ntt.p, wire.p, (int)dim0, s);
  if (nu2) {
    DevBuf<uint64_t> raw(nu2 * 2 * t2 * POLY);
    launch_chacha_first_rows(raw.p, q, dim0 * POLY, (uint32_t)nu2, (uint32_t)(t2 * POLY), 2 * t2 * POLY, c->dp.modulus, s);
    const uint8_t* rest = q + 32 + dim0 * POLY * 8;
    for (size_t i = 0; i < nu2; i++)
      B200_CUDA(cudaMemcpyAsync(raw.p + (i * 2 + 1) * t2 * POLY, rest + i * t2 * POLY * 8, t2 * POLY * 8, cudaMemcpyHostToDevice, s));
    launch_to_ntt(c->dp, c->w_vfold.p + slot * c->fold_words(), raw.p, nu2 * 2 * t2, s);
  }
  B200_CUDA(cudaStreamSynchronize(s));        // the staging buffers above are freed on return
}
}  // namespace

int b200pir_query_from_bytes(b200pir_ctx* c, const uint8_t* data, size_t len, uint64_t* query_ct) {
  API_BEGIN
  if (!c || !data || !query_ct) throw Error(B200PIR_E_BADARG, "null argument");
  if (!c->hp.expand_queries) throw Error(B200PIR_E_UNSUPPORTED, "serialized direct-upload queries are not supported");
  if (len != c->query_bytes) throw Error(B200PIR_E_SHAPE, "query: expected " + std::to_string(c->query_bytes) + " bytes");
  Guard gd(c);
  DevBuf<uint64_t> ct(2 * POLY);
  deserialize_queries(c, data, 1, ct.p);
  B200_CUDA(cudaMemcpyAsync(query_ct, ct.p, 2 * POLY * 8, cudaMemcpyDeviceToHost, c->stream));
  B200_CUDA(cudaStreamSynchronize(c->stream));
  API_END
}

void b200pir_pp_destroy(b200pir_pp* pp) {
  if (!pp) return;
  cudaSetDevice(pp->ctx->device);
  delete pp;
}

// ---------------------------------------------------------------- stage-level entry points
static int ntt_host(b200pir_ctx* c, uint64_t* polys, size_t count, bool inverse) {
  API_BEGIN
  if (!c || (!polys && count)) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  if (count == 0) return 0;
  DevBuf<uint64_t> d(count * 2 * POLY);
  B200_CUDA(cudaMemcpyAsync(d.p, polys, d.n * 8, cudaMemcpyHostToDevice, c->stream));
  launch_ntt_u64(c->dp, d.p, count, inverse, c->stream);
  B200_CUDA(cudaMemcpyAsync(polys, d.p, d.n * 8, cudaMemcpyDeviceToHost, c->stream));
  B200_CUDA(cudaStreamSynchronize(c->stream));
  B200_CUDA(cudaGetLastError());
  API_END
}
int b200pir_ntt_forward(b200pir_ctx* c, uint64_t* polys, size_t count) { return ntt_host(c, polys, count, false); }
int b200pir_ntt_inverse(b200pir_ctx* c, uint64_t* polys, size_t count) { return ntt_host(c, polys, count, true); }

int b200pir_ntt32_dev(b200pir_ctx* c, uint32_t* polys_dev, size_t count, int inverse) {
  API_BEGIN
  if (!c || !polys_dev) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  launch_ntt32(c->dp, polys_dev, count, inverse != 0, c->stream);
  B200_CUDA(cudaGetLastError());
  API_END
}

// ---- poly_len = 4096 transforms (BASELINE config #5; not part of the reference's parameterisation, util.rs:246)
namespace {
const Twiddle* tables_4k(b200pir_ctx* c) {
  if (!c->d_tw4k.p) {
    const int N = 4096, LG = 12;
    std::vector<Twiddle> all;
    for (int n = 0; n < 2; n++) {
      std::vector<Twiddle> f, i;
      build_tables(c->dp.q[n], f, i, N, LG);
      all.insert(all.end(), f.begin(), f.end());
      all.insert(all.end(), i.begin(), i.end());
    }
    c->d_tw4k.alloc(all.size());
    B200_CUDA(cudaMemcpy(c->d_tw4k.p, all.data(), all.size() * sizeof(Twiddle), cudaMemcpyHostToDevice));
  }
  return c->d_tw4k.p;
}
}  // namespace
int b200pir_ntt4096_dev(b200pir_ctx* c, uint32_t* polys_dev, size_t count, int inverse) {
  API_BEGIN
  if (!c || !polys_dev) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  launch_ntt32_4k(c->dp.q[0], c->dp.q[1], tables_4k(c), polys_dev, count, inverse != 0, c->stream);
  B200_CUDA(cudaGetLastError());
  API_END
}
int b200pir_ntt4096(b200pir_ctx* c, uint64_t* polys, size_t count, int inverse) {
  API_BEGIN
  if (!c || (!polys && count)) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  if (count == 0) return 0;
  const size_t words = count * 2 * 4096;
  DevBuf<uint64_t> wide(words);
  DevBuf<uint32_t> nar(words);
  B200_CUDA(cudaMemcpyAsync(wide.p, polys, words * 8, cudaMemcpyHostToDevice, c->stream));
  launch_narrow(nar.p, wide.p, words, c->stream);
  launch_ntt32_4k(c->dp.q[0], c->dp.q[1], tables_4k(c), nar.p, count, inverse != 0, c->stream);
  launch_widen(wide.p, nar.p, words, c->stream);
  B200_CUDA(cudaMemcpyAsync(polys, wide.p, words * 8, cudaMemcpyDeviceToHost, c->stream));
  B200_CUDA(cudaStreamSynchronize(c->stream));
  B200_CUDA(cudaGetLastError());
  API_END
}

int b200pir_to_ntt(b200pir_ctx* c, uint64_t* out_ntt, const uint64_t* raw, size_t count) {
  API_BEGIN
  if (!c || !out_ntt || !raw) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  DevBuf<uint64_t> in(count * POLY), wide(count * 2 * POLY);
  DevBuf<uint32_t> o(count * 2 * POLY);
  B200_CUDA(cudaMemcpyAsync(in.p, raw, in.n * 8, cudaMemcpyHostToDevice, c->stream));
  launch_to_ntt(c->dp, o.p, in.p, count, c->stream);
  launch_widen(wide.p, o.p, o.n, c->stream);
  B200_CUDA(cudaMemcpyAsync(out_ntt, wide.p, wide.n * 8, cudaMemcpyDeviceToHost, c->stream));
  B200_CUDA(cudaStreamSynchronize(c->stream));
  B200_CUDA(cudaGetLastError());
  API_END
}
int b200pir_from_ntt(b200pir_ctx* c, uint64_t* out_raw, const uint64_t* ntt, size_t count) {
  API_BEGIN
  if (!c || !out_raw || !ntt) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  DevBuf<uint64_t> wide(count * 2 * POLY), o(count * POLY);
  DevBuf<uint32_t> in(count * 2 * POLY);
  B200_CUDA(cudaMemcpyAsync(wide.p, ntt, wide.n * 8, cudaMemcpyHostToDevice, c->stream));
  launch_narrow(in.p, wide.p, in.n, c->stream);
  launch_from_ntt(c->dp, o.p, in.p, count, c->stream);
  B200_CUDA(cudaMemcpyAsync(out_raw, o.p, o.n * 8, cudaMemcpyDeviceToHost, c->stream));
  B200_CUDA(cudaStreamSynchronize(c->stream));
  B200_CUDA(cudaGetLastError());
  API_END
}

int b200pir_multiply_reg_by_database(b200pir_ctx* c, b200pir_db* db, uint64_t slice, const uint64_t* v_firstdim,
                                     uint64_t* out) {
  API_BEGIN
  if (!c || !v_firstdim || !out) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  check_db(c, db);
  if (slice >= (uint64_t)c->slices) throw Error(B200PIR_E_SHAPE, "slice out of range");
  const int rows = db->rows;
  MulGeom G = c->geom(rows);
  DevBuf<uint64_t> vq((size_t)c->dim0 * 2 * POLY);
  DevBuf<uint4> qd((size_t)c->dim0 * POLY);
  DevBuf<uint32_t> o((size_t)c->slices * rows * 4 * POLY);
  DevBuf<uint64_t> wide((size_t)rows * 4 * POLY);
  B200_CUDA(cudaMemcpyAsync(vq.p, v_firstdim, vq.n * 8, cudaMemcpyHostToDevice, c->stream));
  launch_query_to_dev(G, qd.p, vq.p, c->stream);
  if (db->format == 0) {
    launch_multiply(c->dp, G, db->d.p, qd.p, o.p, (int)slice, 1, 1, 0, 0, c->mul_variant, c->stream);
  } else if (db->format == 2) {
    DevBuf<uint8_t> qt(tc5_query_bytes(db->T));
    DevBuf<uint32_t> zm((size_t)c->slices * rows * 4 * POLY);
    launch_query_to_tc5(db->T, qd.p, 0, 1, qt.p, c->stream);
    launch_multiply_tc5(c->dp, db->T, db->t.p, db->tile_mask.p, qt.p, zm.p, 0, 1, (int)slice, 1, c->sm_count, c->stream);
    launch_zmajor_to_ntt32(db->F, zm.p, o.p + (size_t)slice * rows * 4 * POLY, (int)slice, c->stream);
    B200_CUDA(cudaStreamSynchronize(c->stream));
  } else {
    DevBuf<uint2> qf(imma_query_cells(db->F));
    DevBuf<uint32_t> zm((size_t)c->slices * rows * 4 * POLY);
    launch_query_to_frag(db->F, qd.p, 0, 1, qf.p, c->stream);
    launch_multiply_imma(c->dp, db->F, db->f.p, qf.p, zm.p, 0, 1, (int)slice, 1, c->imma_variant, c->stream);
    launch_zmajor_to_ntt32(db->F, zm.p, o.p + (size_t)slice * rows * 4 * POLY, (int)slice, c->stream);
    B200_CUDA(cudaStreamSynchronize(c->stream));
  }
  launch_widen(wide.p, o.p + (size_t)slice * rows * 4 * POLY, wide.n, c->stream);
  B200_CUDA(cudaMemcpyAsync(out, wide.p, wide.n * 8, cudaMemcpyDeviceToHost, c->stream));
  B200_CUDA(cudaStreamSynchronize(c->stream));
  B200_CUDA(cudaGetLastError());
  API_END
}

int b200pir_fold_ciphertexts(b200pir_ctx* c, uint64_t* v_cts, size_t num, const uint64_t* v_folding,
                             const uint64_t* v_folding_neg) {
  API_BEGIN
  if (!c || !v_cts) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  if (num == 0 || (num & (num - 1))) throw Error(B200PIR_E_SHAPE, "number of ciphertexts must be a power of two");
  if (num == 1) return 0;                                          // server.rs:394-396
  if (!v_folding) throw Error(B200PIR_E_BADARG, "null argument");
  int dims = 0;
  while (((size_t)1 << dims) < num) dims++;
  if (dims > (int)c->hp.nu_2) throw Error(B200PIR_E_SHAPE, "more ciphertexts than 2^nu_2");
  const size_t mat = (size_t)2 * 2 * c->hp.t_gsw * 2 * POLY;
  DevBuf<uint64_t> cts(num * 2 * POLY), wide(dims * mat);
  DevBuf<uint32_t> vf(c->fold_words());
  B200_CUDA(cudaMemcpyAsync(cts.p, v_cts, cts.n * 8, cudaMemcpyHostToDevice, c->stream));
  B200_CUDA(cudaMemcpyAsync(wide.p, v_folding, wide.n * 8, cudaMemcpyHostToDevice, c->stream));
  launch_narrow(vf.p, wide.p, wide.n, c->stream);
  if (v_folding_neg && !c->sparse_fold) {
    // general path: honours an arbitrary v_folding_neg exactly as server.rs:405-425 does
    DevBuf<uint32_t> vfn(c->fold_words());
    B200_CUDA(cudaMemcpyAsync(wide.p, v_folding_neg, wide.n * 8, cudaMemcpyHostToDevice, c->stream));
    launch_narrow(vfn.p, wide.p, wide.n, c->stream);
    run_fold(c, cts.p, 1, num * 2 * POLY, num, dims - 1, vf.p, vfn.p, 1);
  } else {
    // fast path (what process_query uses): v_folding_neg = get_v_folding_neg(v_folding) implied.
    // Round results are copied back so every slot ends up as the reference's in-place loop leaves it.
    // With "sparse_fold" set this is lib/server's fold (compute/fold.rs:15-65): v_folding_neg is then taken to be
    // get_v_folding_neg(v_folding), which is what that server passes (lib/server/src/server.rs).
    DevBuf<uint32_t> a(num * 4 * POLY), b(num * 4 * POLY);
    DevBuf<uint32_t> zflags;
    if (c->sparse_fold) zflags.alloc(num);
    launch_raw_to_res(c->dp, a.p, cts.p, num * 2, c->stream);
    int k = dims - 1;
    for (size_t half = num / 2; half >= 1; half /= 2, k--) {
      launch_fold_res(c->dp, a.p, b.p, 1, num * 4 * POLY, (int)half, vf.p + (size_t)k * mat, c->fold_words(), 1,
                      (int)c->hp.t_gsw, c->bits_gsw, c->fold_variant, zflags.p, c->stream);
      B200_CUDA(cudaMemcpyAsync(a.p, b.p, half * 4 * POLY * 4, cudaMemcpyDeviceToDevice, c->stream));
    }
    launch_res_to_raw(c->dp, cts.p, a.p, num * 2, c->stream);
  }
  B200_CUDA(cudaMemcpyAsync(v_cts, cts.p, cts.n * 8, cudaMemcpyDeviceToHost, c->stream));
  B200_CUDA(cudaStreamSynchronize(c->stream));
  B200_CUDA(cudaGetLastError());
  API_END
}

int b200pir_get_v_folding_neg(b200pir_ctx* c, uint64_t* out, const uint64_t* v_folding) {
  API_BEGIN
  if (!c || !out || !v_folding) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  const size_t words = c->fold_words();
  if (!words) return 0;
  DevBuf<uint64_t> wide(words);
  DevBuf<uint32_t> in(words), o(words);
  B200_CUDA(cudaMemcpyAsync(wide.p, v_folding, words * 8, cudaMemcpyHostToDevice, c->stream));
  launch_narrow(in.p, wide.p, words, c->stream);
  launch_folding_neg(c->dp, o.p, in.p, (int)c->hp.nu_2, (int)c->hp.t_gsw, c->bits_gsw, c->stream);
  launch_widen(wide.p, o.p, words, c->stream);
  B200_CUDA(cudaMemcpyAsync(out, wide.p, words * 8, cudaMemcpyDeviceToHost, c->stream));
  B200_CUDA(cudaStreamSynchronize(c->stream));
  B200_CUDA(cudaGetLastError());
  API_END
}

int b200pir_coefficient_expansion(b200pir_ctx* c, b200pir_pp* pp, uint64_t* v) {
  API_BEGIN
  if (!c || !v) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  check_pp(c, pp);
  if (!c->hp.expand_queries) throw Error(B200PIR_E_BADARG, "context was created with expand_queries = 0");
  const size_t words = c->v_words();
  DevBuf<uint64_t> wide(words);
  DevBuf<uint32_t> dv(words);
  B200_CUDA(cudaMemcpyAsync(wide.p, v, words * 8, cudaMemcpyHostToDevice, c->stream));
  launch_narrow(dv.p, wide.p, words, c->stream);
  run_coefficient_expansion(c, pp, dv.p, words, 1, true);
  launch_widen(wide.p, dv.p, words, c->stream);
  B200_CUDA(cudaMemcpyAsync(v, wide.p, words * 8, cudaMemcpyDeviceToHost, c->stream));
  B200_CUDA(cudaStreamSynchronize(c->stream));
  B200_CUDA(cudaGetLastError());
  API_END
}

int b200pir_expand_query(b200pir_ctx* c, b200pir_pp* pp, const uint64_t* query_ct, uint64_t* out_v_firstdim,
                         uint64_t* out_v_folding) {
  API_BEGIN
  if (!c || !query_ct || !out_v_firstdim) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  check_pp(c, pp);
  if (!c->hp.expand_queries) throw Error(B200PIR_E_BADARG, "context was created with expand_queries = 0");
  c->ensure_workspace(1, 1);
  B200_CUDA(cudaMemcpyAsync(c->w_query.p, query_ct, 2 * POLY * 8, cudaMemcpyHostToDevice, c->stream));
  run_expand_query(c, pp, c->w_query.p, c->w_v.p, c->w_qdev.p, c->w_vfold.p, 1);
  // q_dev -> reference layout [z][j][r]
  const size_t qwords = (size_t)c->dim0 * 2 * POLY;
  std::vector<uint32_t> hq(qwords * 2);
  B200_CUDA(cudaMemcpyAsync(hq.data(), c->w_qdev.p, hq.size() * 4, cudaMemcpyDeviceToHost, c->stream));
  B200_CUDA(cudaStreamSynchronize(c->stream));
  for (int j = 0; j < c->dim0; j++)
    for (int z = 0; z < POLY; z++) {
      const uint32_t* cell = hq.data() + (((size_t)(j >> 1) * 2 + (j & 1)) * POLY + z) * 4;
      out_v_firstdim[((size_t)z * c->dim0 + j) * 2 + 0] = (uint64_t)cell[0] | ((uint64_t)cell[1] << 32);
      out_v_firstdim[((size_t)z * c->dim0 + j) * 2 + 1] = (uint64_t)cell[2] | ((uint64_t)cell[3] << 32);
    }
  if (out_v_folding && c->fold_words()) {
    DevBuf<uint64_t> wide(c->fold_words());
    launch_widen(wide.p, c->w_vfold.p, c->fold_words(), c->stream);
    B200_CUDA(cudaMemcpyAsync(out_v_folding, wide.p, wide.n * 8, cudaMemcpyDeviceToHost, c->stream));
    B200_CUDA(cudaStreamSynchronize(c->stream));
  }
  B200_CUDA(cudaGetLastError());
  API_END
}

int b200pir_pack(b200pir_ctx* c, b200pir_pp* pp, const uint64_t* v_ct, uint64_t* out_ntt) {
  API_BEGIN
  if (!c || !v_ct || !out_ntt) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  check_pp(c, pp);
  const auto& hp = c->hp;
  const size_t nn = hp.n * hp.n, outp = (hp.n + 1) * hp.n;
  DevBuf<uint64_t> cts(nn * 2 * POLY), raw(outp * POLY), wide(outp * 2 * POLY);
  DevBuf<uint32_t> o(outp * 2 * POLY), res(nn * 4 * POLY);
  B200_CUDA(cudaMemcpyAsync(cts.p, v_ct, cts.n * 8, cudaMemcpyHostToDevice, c->stream));
  launch_raw_to_res(c->dp, res.p, cts.p, nn * 2, c->stream);
  launch_pack(c->dp, raw.p, 0, res.p, 4 * POLY, 0, 1, c->pp_table(pp, 1).pack, (int)hp.n, 1, (int)hp.t_conv, c->bits_conv, (int)hp.version, c->stream);
  // the reference's pack returns the NTT-form matrix (server.rs:467); the kernel already applied .raw()
  launch_to_ntt(c->dp, o.p, raw.p, outp, c->stream);
  launch_widen(wide.p, o.p, o.n, c->stream);
  B200_CUDA(cudaMemcpyAsync(out_ntt, wide.p, wide.n * 8, cudaMemcpyDeviceToHost, c->stream));
  B200_CUDA(cudaStreamSynchronize(c->stream));
  B200_CUDA(cudaGetLastError());
  API_END
}

int b200pir_encode(b200pir_ctx* c, const uint64_t* v_packed_raw, uint8_t* out, size_t* out_len) {
  API_BEGIN
  if (!c || !v_packed_raw || !out) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  const auto& hp = c->hp;
  const size_t words = (size_t)hp.instances * (hp.n + 1) * hp.n * POLY;
  DevBuf<uint64_t> in(words);
  DevBuf<uint8_t> o(c->response_bytes);
  B200_CUDA(cudaMemcpyAsync(in.p, v_packed_raw, words * 8, cudaMemcpyHostToDevice, c->stream));
  launch_encode(c->dp, o.p, c->response_bytes, in.p, 0, 1, (int)hp.n, (int)hp.instances, c->q2, (int)hp.q2_bits, c->q1, c->q1_bits, c->stream);
  B200_CUDA(cudaMemcpyAsync(out, o.p, c->response_bytes, cudaMemcpyDeviceToHost, c->stream));
  B200_CUDA(cudaStreamSynchronize(c->stream));
  if (out_len) *out_len = c->response_bytes;
  B200_CUDA(cudaGetLastError());
  API_END
}

// ---------------------------------------------------------------- process_query
static void run_query_batch_resident(b200pir_ctx* c, b200pir_db* db, b200pir_pp* pp, size_t count, uint8_t* out_dev) {
  // queries are already in c->w_query; tcgen05 databases get their operand as tile images straight from the expansion
  const bool images = db->format == 2 && c->hp.expand_queries;
  run_prepare(c, pp, count, images);
  run_first_dim_and_fold(c, db, count, nullptr, nullptr, images ? c->w_qt.p : nullptr, 16);
  run_pack_encode(c, pp, c->folded, c->folded_stride, count, out_dev);
}

int b200pir_process_query_batch_dev(b200pir_ctx* c, b200pir_db* db, b200pir_pp* pp, const uint64_t* query_cts_dev,
                                    size_t count, uint8_t* out_dev) {
  API_BEGIN
  if (!c || !out_dev || !query_cts_dev) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  check_db(c, db);
  check_pp(c, pp);
  if (db->shard.count != 1) throw Error(B200PIR_E_BADARG, "sharded database: use the stage_a / stage_b entry points");
  if (!c->hp.expand_queries) throw Error(B200PIR_E_BADARG, "batch entry point needs expand_queries");
  if (count == 0) return 0;
  c->ensure_workspace(count, db->rows);
  c->prof_reset();
  B200_CUDA(cudaMemcpyAsync(c->w_query.p, query_cts_dev, count * 2 * POLY * 8, cudaMemcpyDeviceToDevice, c->stream));
  run_query_batch_resident(c, db, pp, count, out_dev);
  B200_CUDA(cudaGetLastError());
  API_END
}

int b200pir_process_query_batch(b200pir_ctx* c, b200pir_db* db, b200pir_pp* pp, const uint64_t* query_cts, size_t count,
                                uint8_t* out, size_t* out_len_each) {
  API_BEGIN
  if (!c || !out || !query_cts) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  check_db(c, db);
  check_pp(c, pp);
  if (db->shard.count != 1) throw Error(B200PIR_E_BADARG, "sharded database: use the stage_a / stage_b entry points");
  if (!c->hp.expand_queries) throw Error(B200PIR_E_BADARG, "batch entry point needs expand_queries");
  if (count == 0) return 0;
  c->ensure_workspace(count, db->rows);
  c->prof_reset();
  B200_CUDA(cudaMemcpyAsync(c->w_query.p, query_cts, count * 2 * POLY * 8, cudaMemcpyHostToDevice, c->stream));
  run_query_batch_resident(c, db, pp, count, c->w_resp.p);
  B200_CUDA(cudaMemcpyAsync(out, c->w_resp.p, count * c->response_bytes, cudaMemcpyDeviceToHost, c->stream));
  B200_CUDA(cudaStreamSynchronize(c->stream));
  if (c->profile == 1) c->prof_collect();
  if (out_len_each) *out_len_each = c->response_bytes;
  B200_CUDA(cudaGetLastError());
  API_END
}

namespace {
// `count` queries of possibly different clients in one database pass.  cts[i]: host PolyMatrixRaw(2,1), or bytes[i]: the
// serialized query (exactly one of the two non-null per entry); outs[i]: response_bytes.  Caller holds no lock.
void process_multi(b200pir_ctx* c, b200pir_db* db, b200pir_pp* const* pps, const uint64_t* const* cts,
                   const uint8_t* const* bytes, size_t count, uint8_t* const* outs) {
  Guard gd(c);
  check_db(c, db);
  for (size_t i = 0; i < count; i++) check_pp(c, pps[i]);
  if (db->shard.count != 1) throw Error(B200PIR_E_BADARG, "sharded database: use the stage_a / stage_b entry points");
  if (!c->hp.expand_queries) throw Error(B200PIR_E_BADARG, "multi-client batches need expand_queries");
  // workspace sized once for a full coalesced batch: batch sizes vary from call to call, the buffers do not
  c->ensure_workspace(std::max(count, c->coalesce ? b200pir_ctx::kCoalesceMax : count), db->rows);
  c->prof_reset();
  for (size_t i = 0; i < count; i++) {
    if (bytes && bytes[i]) deserialize_queries(c, bytes[i], 1, c->w_query.p + i * 2 * POLY);
    else B200_CUDA(cudaMemcpyAsync(c->w_query.p + i * 2 * POLY, cts[i], 2 * POLY * 8, cudaMemcpyHostToDevice, c->stream));
  }
  c->multi_pps = pps;
  try {
    run_query_batch_resident(c, db, pps[0], count, c->w_resp.p);
  } catch (...) { c->multi_pps = nullptr; throw; }
  c->multi_pps = nullptr;
  for (size_t i = 0; i < count; i++)
    B200_CUDA(cudaMemcpyAsync(outs[i], c->w_resp.p + i * c->response_bytes, c->response_bytes, cudaMemcpyDeviceToHost, c->stream));
  B200_CUDA(cudaStreamSynchronize(c->stream));
  if (c->profile == 1) c->prof_collect();
  B200_CUDA(cudaGetLastError());
}

// one query through the combiner (see b200pir_ctx::Pending)
int coalesced_query(b200pir_ctx* c, b200pir_db* db, b200pir_pp* pp, const uint64_t* query_ct, const uint8_t* query_bytes,
                    uint8_t* out) {
  b200pir_ctx::Pending me;
  me.db = db; me.pp = pp; me.query_ct = query_ct; me.query_bytes = query_bytes; me.out = out;
  std::unique_lock<std::mutex> lk(c->qmu);
  c->pending.push_back(&me);
  c->qcv.notify_all();                       // a leader may be holding its batch open for us
  while (!me.done) {
    if (c->leader_active) { c->qcv.wait(lk); continue; }
    // become the leader: take the queued requests for the database at the head of the queue
    c->leader_active = true;
    if (c->coalesce_window_us > 0 && c->last_batch > 1 && c->pending.size() < std::min(c->last_batch, b200pir_ctx::kPassQueries)) {
      const auto now = std::chrono::steady_clock::now();
      if (now - c->last_batch_end < std::chrono::milliseconds(1)) {
        const size_t want = std::min(c->last_batch, b200pir_ctx::kPassQueries);
        c->qcv.wait_until(lk, now + std::chrono::microseconds(c->coalesce_window_us), [&] { return c->pending.size() >= want; });
      }
    }
    std::vector<b200pir_ctx::Pending*> batch;
    b200pir_db* bdb = c->pending.front()->db;
    size_t avail = 0;
    for (auto* p : c->pending) avail += p->db == bdb;
    size_t take = std::min(avail, b200pir_ctx::kCoalesceMax);
    if (take > b200pir_ctx::kPassQueries) take -= take % b200pir_ctx::kPassQueries;
    for (auto it = c->pending.begin(); it != c->pending.end() && batch.size() < take;) {
      if ((*it)->db == bdb) { batch.push_back(*it); it = c->pending.erase(it); } else ++it;
    }
    lk.unlock();
    int rc = 0;
    std::string err;
    try {
      std::vector<b200pir_pp*> pps; std::vector<const uint64_t*> cts; std::vector<const uint8_t*> bys; std::vector<uint8_t*> outs;
      for (auto* p : batch) { pps.push_back(p->pp); cts.push_back(p->query_ct); bys.push_back(p->query_bytes); outs.push_back(p->out); }
      process_multi(c, bdb, pps.data(), cts.data(), bys.data(), batch.size(), outs.data());
    } catch (const std::exception& e) { rc = fail(e); err = e.what(); }
    lk.lock();
    c->coalesced_batches++; c->coalesced_queries += batch.size();
    c->last_batch = batch.size();
    c->last_batch_end = std::chrono::steady_clock::now();
    for (auto* p : batch) { p->rc = rc; p->err = err; p->done = true; }
    c->leader_active = false;
    c->qcv.notify_all();
  }
  if (me.rc) g_last_error = me.err;
  return me.rc;
}
}  // namespace

int b200pir_process_queries(b200pir_ctx* c, b200pir_db* db, b200pir_pp* const* pps, const uint64_t* const* query_cts, size_t count,
                            uint8_t* const* outs) {
  API_BEGIN
  if (!c || !pps || !query_cts || !outs) throw Error(B200PIR_E_BADARG, "null argument");
  for (size_t i = 0; i < count; i++)
    if (!pps[i] || !query_cts[i] || !outs[i]) throw Error(B200PIR_E_BADARG, "null entry");
  if (count == 0) return 0;
  process_multi(c, db, pps, query_cts, nullptr, count, outs);
  API_END
}
int b200pir_coalesce_stats(b200pir_ctx* c, uint64_t* batches, uint64_t* queries) {
  API_BEGIN
  if (!c) throw Error(B200PIR_E_BADARG, "null ctx");
  std::lock_guard<std::mutex> lk(c->qmu);
  if (batches) *batches = c->coalesced_batches;
  if (queries) *queries = c->coalesced_queries;
  API_END
}

// process_query over the wire format: `count` serialized queries (Query::serialize, client.rs:279-301) back to back
int b200pir_process_query_bytes(b200pir_ctx* c, b200pir_db* db, b200pir_pp* pp, const uint8_t* queries, size_t len,
                                size_t count, uint8_t* out, size_t* out_len_each) {
  API_BEGIN
  if (!c || !out || !queries) throw Error(B200PIR_E_BADARG, "null argument");
  if (len != count * c->query_bytes) throw Error(B200PIR_E_SHAPE, "queries: expected " + std::to_string(count * c->query_bytes) + " bytes");
  if (count == 1 && c->coalesce && c->hp.expand_queries && db && pp) {          // the /private-read handler's call: one query per request
    const int rc = coalesced_query(c, db, pp, nullptr, queries, out);
    if (rc == 0 && out_len_each) *out_len_each = c->response_bytes;
    return rc;
  }
  Guard gd(c);
  check_db(c, db);
  check_pp(c, pp);
  if (db->shard.count != 1) throw Error(B200PIR_E_BADARG, "sharded database: use the stage_a / stage_b entry points");
  if (count == 0) return 0;
  c->ensure_workspace(count, db->rows);
  c->prof_reset();
  if (c->hp.expand_queries) {
    deserialize_queries(c, queries, count, c->w_query.p);
    run_query_batch_resident(c, db, pp, count, c->w_resp.p);
  } else {
    // direct upload (client.rs:316-327; the body lib/server's handler parses at bin/server.rs:122-137 is setup || query):
    // every query arrives expanded; nothing to prepare beyond the deserialization
    for (size_t i = 0; i < count; i++) deserialize_query_direct(c, queries + i * c->query_bytes, i);
    run_first_dim_and_fold(c, db, count);
    run_pack_encode(c, pp, c->folded, c->folded_stride, count, c->w_resp.p);
  }
  B200_CUDA(cudaMemcpyAsync(out, c->w_resp.p, count * c->response_bytes, cudaMemcpyDeviceToHost, c->stream));
  B200_CUDA(cudaStreamSynchronize(c->stream));
  if (c->profile == 1) c->prof_collect();
  if (out_len_each) *out_len_each = c->response_bytes;
  B200_CUDA(cudaGetLastError());
  API_END
}

int b200pir_process_query(b200pir_ctx* c, b200pir_db* db, b200pir_pp* pp, const uint64_t* query_ct, const uint64_t* v_buf,
                          const uint64_t* v_ct, uint8_t* out, size_t* out_len) {
  if (!c) { g_last_error = "null ctx"; return B200PIR_E_BADARG; }
  if (c->hp.expand_queries) {
    if (!query_ct || !out || !db || !pp) { g_last_error = "null argument"; return B200PIR_E_BADARG; }
    if (!c->coalesce) return b200pir_process_query_batch(c, db, pp, query_ct, 1, out, out_len);
    const int rc = coalesced_query(c, db, pp, query_ct, nullptr, out);
    if (rc == 0 && out_len) *out_len = c->response_bytes;
    return rc;
  }
  API_BEGIN
  if (!v_buf || (!v_ct && c->hp.nu_2) || !out) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  check_db(c, db);
  check_pp(c, pp);
  if (db->shard.count != 1) throw Error(B200PIR_E_BADARG, "sharded database: use the stage_a / stage_b entry points");
  c->ensure_workspace(1, db->rows);
  c->prof_reset();
  // server.rs:666-678: v_reg_reoriented = query.v_buf ; v_folding = v_ct.map(ntt)
  DevBuf<uint64_t> vq((size_t)c->dim0 * 2 * POLY);
  B200_CUDA(cudaMemcpyAsync(vq.p, v_buf, vq.n * 8, cudaMemcpyHostToDevice, c->stream));
  launch_query_to_dev(c->geom(db->rows), c->w_qdev.p, vq.p, c->stream);
  const size_t npolys = (size_t)c->hp.nu_2 * 2 * 2 * c->hp.t_gsw;
  DevBuf<uint64_t> raw(std::max<size_t>(npolys, 1) * POLY);
  if (npolys) {
    B200_CUDA(cudaMemcpyAsync(raw.p, v_ct, npolys * POLY * 8, cudaMemcpyHostToDevice, c->stream));
    launch_to_ntt(c->dp, c->w_vfold.p, raw.p, npolys, c->stream);
  }
  run_prepare(c, pp, 1);
  run_first_dim_and_fold(c, db, 1);
  run_pack_encode(c, pp, c->folded, c->folded_stride, 1, c->w_resp.p);
  B200_CUDA(cudaMemcpyAsync(out, c->w_resp.p, c->response_bytes, cudaMemcpyDeviceToHost, c->stream));
  B200_CUDA(cudaStreamSynchronize(c->stream));
  if (c->profile == 1) c->prof_collect();
  if (out_len) *out_len = c->response_bytes;
  B200_CUDA(cudaGetLastError());
  API_END
}

// ---- multi-GPU building blocks: the three phases with caller-owned device buffers in between, so the host can put a
// collective between them (bench.py: queries are expanded by the rank that received them, everything is all-gathered)
int b200pir_expand_queries_dev(b200pir_ctx* c, b200pir_pp* pp, const uint64_t* query_cts_dev, size_t count,
                               void* q_expanded_dev, uint32_t* v_folding_dev) {
  API_BEGIN
  if (!c || !query_cts_dev || !q_expanded_dev || (!v_folding_dev && c->hp.nu_2)) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  check_pp(c, pp);
  if (!c->hp.expand_queries) throw Error(B200PIR_E_BADARG, "needs expand_queries");
  if (count == 0) return 0;
  c->w_v.ensure(count * c->v_words());
  c->prof_reset();
  {
    b200pir_ctx::Scope sc(c, ST_EXPAND);
    run_expand_query(c, pp, query_cts_dev, c->w_v.p, (uint4*)q_expanded_dev, v_folding_dev, (int)count);
  }
  B200_CUDA(cudaGetLastError());
  API_END
}
int b200pir_first_dim_fold_dev(b200pir_ctx* c, b200pir_db* db, const void* q_expanded_dev, const uint32_t* v_folding_dev,
                               size_t count, uint32_t* partial_dev) {
  API_BEGIN
  if (!c || !q_expanded_dev || !partial_dev || (!v_folding_dev && c->hp.nu_2)) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  check_db(c, db);
  if (count == 0) return 0;
  c->ensure_workspace_lite(count, db->rows);
  run_first_dim_and_fold(c, db, count, (const uint4*)q_expanded_dev, v_folding_dev);
  B200_CUDA(cudaMemcpy2DAsync(partial_dev, 4 * POLY * 4, c->folded, c->folded_stride * 4, 4 * POLY * 4, count * c->slices,
                              cudaMemcpyDeviceToDevice, c->stream));
  B200_CUDA(cudaGetLastError());
  API_END
}
// The same two phases with the first-dimension operand exchanged as UMMA tile images (tcgen05 databases): the rank that expands a
// group of <= 16 queries also re-tiles it, once; the receivers multiply straight from the image.
size_t b200pir_query_image_bytes(b200pir_ctx* c) { return c ? tc5_query_bytes(make_tc5_geom(c->dim0, 32)) : 0; }
int b200pir_expand_queries_images_dev(b200pir_ctx* c, b200pir_pp* pp, const uint64_t* query_cts_dev, size_t count, void* image_dev,
                                      uint32_t* v_folding_dev) {
  API_BEGIN
  if (!c || !query_cts_dev || !image_dev || (!v_folding_dev && c->hp.nu_2)) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  check_pp(c, pp);
  if (!c->hp.expand_queries) throw Error(B200PIR_E_BADARG, "needs expand_queries");
  if (count == 0 || count > 16) throw Error(B200PIR_E_SHAPE, "one image holds 1..16 queries");
  if (!tc5_supported(make_tc5_geom(c->dim0, 32))) throw Error(B200PIR_E_UNSUPPORTED, "dim0 too large for the tcgen05 kernel");
  c->w_v.ensure(count * c->v_words());
  c->prof_reset();
  {
    b200pir_ctx::Scope sc(c, ST_EXPAND);
    run_expand_query(c, pp, query_cts_dev, c->w_v.p, nullptr, v_folding_dev, (int)count, (uint8_t*)image_dev);
  }
  B200_CUDA(cudaGetLastError());
  API_END
}
int b200pir_first_dim_fold_images_dev(b200pir_ctx* c, b200pir_db* db, const void* images_dev, size_t groups, size_t per_group,
                                      const uint32_t* v_folding_dev, uint32_t* partial_dev) {
  API_BEGIN
  if (!c || !images_dev || !partial_dev || (!v_folding_dev && c->hp.nu_2)) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  check_db(c, db);
  if (db->format != 2) throw Error(B200PIR_E_BADARG, "tile images need a tcgen05-layout database (db_format 2)");
  if (per_group == 0 || per_group > 16) throw Error(B200PIR_E_SHAPE, "one image holds 1..16 queries");
  const size_t count = groups * per_group;
  if (count == 0) return 0;
  c->ensure_workspace_lite(count, db->rows);
  run_first_dim_and_fold(c, db, count, nullptr, v_folding_dev, (const uint8_t*)images_dev, per_group);
  B200_CUDA(cudaMemcpy2DAsync(partial_dev, 4 * POLY * 4, c->folded, c->folded_stride * 4, 4 * POLY * 4, count * c->slices,
                              cudaMemcpyDeviceToDevice, c->stream));
  B200_CUDA(cudaGetLastError());
  API_END
}
int b200pir_finish_queries_dev(b200pir_ctx* c, b200pir_pp* pp, const uint32_t* gathered_dev, size_t world, size_t total_count,
                               size_t first, size_t count, const uint32_t* v_folding_dev, uint8_t* out_dev) {
  API_BEGIN
  if (!c || !gathered_dev || !out_dev || (!v_folding_dev && world > 1)) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  check_pp(c, pp);
  if (world == 0 || (world & (world - 1)) || world > (size_t)c->num_per) throw Error(B200PIR_E_SHAPE, "bad world size");
  if (first + count > total_count) throw Error(B200PIR_E_SHAPE, "query range out of bounds");
  if (count == 0) return 0;
  c->ensure_workspace_lite(count, world);
  const size_t ct = 4 * POLY;
  for (size_t w = 0; w < world; w++)
    B200_CUDA(cudaMemcpy2DAsync(c->w_mult.p + w * ct, world * ct * 4, gathered_dev + (w * total_count + first) * c->slices * ct,
                                ct * 4, ct * 4, count * c->slices, cudaMemcpyDeviceToDevice, c->stream));
  int dims = 0;
  while (((size_t)1 << dims) < world) dims++;
  {
    b200pir_ctx::Scope sc(c, ST_FOLD);
    c->folded = c->w_mult.p;
    c->folded_stride = world * ct;
    if (world > 1)
      c->folded = run_fold_res(c, c->w_mult.p, c->w_cts.p, count * c->slices, world * ct, world, dims - 1, v_folding_dev,
                               c->slices);
  }
  run_pack_encode(c, pp, c->folded, c->folded_stride, count, out_dev);
  B200_CUDA(cudaGetLastError());
  API_END
}

int b200pir_query_stage_a_dev(b200pir_ctx* c, b200pir_db* db, b200pir_pp* pp, const uint64_t* query_cts_dev, size_t count,
                              uint32_t* partial_dev) {
  API_BEGIN
  if (!c || !query_cts_dev || !partial_dev) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  check_db(c, db);
  check_pp(c, pp);
  if (!c->hp.expand_queries) throw Error(B200PIR_E_BADARG, "needs expand_queries");
  c->ensure_workspace(count, db->rows);
  c->prof_reset();
  B200_CUDA(cudaMemcpyAsync(c->w_query.p, query_cts_dev, count * 2 * POLY * 8, cudaMemcpyDeviceToDevice, c->stream));
  run_prepare(c, pp, count);
  run_first_dim_and_fold(c, db, count);
  // gather the survivors [count][slices] into a dense buffer of residue-form ciphertexts
  B200_CUDA(cudaMemcpy2DAsync(partial_dev, 4 * POLY * 4, c->folded, c->folded_stride * 4, 4 * POLY * 4, count * c->slices,
                              cudaMemcpyDeviceToDevice, c->stream));
  B200_CUDA(cudaGetLastError());
  API_END
}

int b200pir_query_stage_b_dev(b200pir_ctx* c, b200pir_pp* pp, const uint32_t* gathered_dev, size_t world, size_t count,
                              uint8_t* out_dev) {
  API_BEGIN
  if (!c || !gathered_dev || !out_dev) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  check_pp(c, pp);
  if (world == 0 || (world & (world - 1)) || world > (size_t)c->num_per) throw Error(B200PIR_E_SHAPE, "bad world size");
  c->ensure_workspace(count, world);
  // gathered: [world][count][slices][ct]  ->  w_mult as [count][slices][world][ct]   (ct = 4*2048 u32)
  const size_t ct = 4 * POLY;
  for (size_t w = 0; w < world; w++)
    B200_CUDA(cudaMemcpy2DAsync(c->w_mult.p + w * ct, world * ct * 4, gathered_dev + w * count * c->slices * ct, ct * 4,
                                ct * 4, count * c->slices, cudaMemcpyDeviceToDevice, c->stream));
  int dims = 0;
  while (((size_t)1 << dims) < world) dims++;
  {
    b200pir_ctx::Scope sc(c, ST_FOLD);
    c->folded = c->w_mult.p;
    c->folded_stride = world * ct;
    if (world > 1)
      c->folded = run_fold_res(c, c->w_mult.p, c->w_cts.p, count * c->slices, world * ct, world, dims - 1, c->w_vfold.p,
                               c->slices);
  }
  run_pack_encode(c, pp, c->folded, c->folded_stride, count, out_dev);
  B200_CUDA(cudaGetLastError());
  API_END
}

unsigned long long b200pir_kernel_launches(void) { return g_kernel_launches; }

// ---- peer memory (CUDA IPC) for the copy-engine exchange of the multi-GPU flow
int b200pir_peer_alloc(int device, size_t bytes, void** out_ptr, uint8_t out_handle[64]) {
  API_BEGIN
  if (!out_ptr || !out_handle || !bytes) throw Error(B200PIR_E_BADARG, "null or empty argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  B200_CUDA(cudaSetDevice(device));
  void* p = nullptr;
  B200_CUDA(cudaMalloc(&p, bytes));
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) { cudaFree(p); throw Error(B200PIR_E_CUDA, std::string("cudaIpcGetMemHandle: ") + cudaGetErrorString(e)); }
  std::memcpy(out_handle, &h, 64);
  *out_ptr = p;
  API_END
}
int b200pir_peer_open(int device, const uint8_t handle[64], void** out_ptr) {
  API_BEGIN
  if (!handle || !out_ptr) throw Error(B200PIR_E_BADARG, "null argument");
  B200_CUDA(cudaSetDevice(device));
  cudaIpcMemHandle_t h;
  std::memcpy(&h, handle, 64);
  B200_CUDA(cudaIpcOpenMemHandle(out_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  API_END
}
int b200pir_peer_close(int device, void* mapped_ptr) {
  API_BEGIN
  B200_CUDA(cudaSetDevice(device));
  if (mapped_ptr) B200_CUDA(cudaIpcCloseMemHandle(mapped_ptr));
  API_END
}
int b200pir_peer_free(int device, void* ptr) {
  API_BEGIN
  B200_CUDA(cudaSetDevice(device));
  if (ptr) B200_CUDA(cudaFree(ptr));
  API_END
}
int b200pir_peer_copy_async(void* dst, const void* src, size_t bytes, void* cuda_stream) {
  API_BEGIN
  if (!dst || !src) throw Error(B200PIR_E_BADARG, "null argument");
  if (bytes) B200_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, (cudaStream_t)cuda_stream));
  API_END
}

int b200pir_last_stage_ms(b200pir_ctx* c, double* out9) {
  API_BEGIN
  if (!c || !out9) throw Error(B200PIR_E_BADARG, "null argument");
  Guard gd(c);
  c->prof_collect();
  for (int i = 0; i < 9; i++) out9[i] = c->last_ms[i];
  API_END
}

// ---------------------------------------------------------------- DoublePIR
namespace {
__global__ void k_dpir_synth(uint32_t* a, size_t words, uint64_t seed, size_t index0) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= words) return;
  uint64_t z = seed + (index0 + i + 1) * 0x9E3779B97F4A7C15ULL;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
  z ^= z >> 31;
  a[i] = (uint32_t)z & 0x3FFFFFFFu;
}
b200pir_dpir* dpir_new(int device, uint64_t rows, uint64_t cols) {
  int ndev = 0;
  B200_CUDA(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) throw Error(B200PIR_E_BADARG, "no such CUDA device (this library has no CPU path)");
  if (rows == 0 || cols == 0) throw Error(B200PIR_E_SHAPE, "empty matrix");
  B200_CUDA(cudaSetDevice(device));
  std::unique_ptr<b200pir_dpir> m(new b200pir_dpir());
  m->device = device; m->rows = rows; m->cols = cols;
  B200_CUDA(cudaStreamCreateWithFlags(&m->stream, cudaStreamNonBlocking));
  m->a.alloc(rows * cols);
  m->b.alloc(3 * cols);
  m->out.alloc(rows);
  return m.release();
}
}  // namespace

int b200pir_dpir_create(int device, const uint32_t* a, uint64_t rows, uint64_t cols, b200pir_dpir** out) {
  API_BEGIN
  if (!a || !out) throw Error(B200PIR_E_BADARG, "null argument");
  b200pir_dpir* m = dpir_new(device, rows, cols);
  cudaError_t e = cudaMemcpy(m->a.p, a, rows * cols * 4, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) { b200pir_dpir_destroy(m); throw Error(B200PIR_E_CUDA, cudaGetErrorString(e)); }
  *out = m;
  API_END
}
int b200pir_dpir_create_synthetic(int device, uint64_t rows, uint64_t cols, uint64_t seed, b200pir_dpir** out) {
  API_BEGIN
  if (!out) throw Error(B200PIR_E_BADARG, "null argument");
  b200pir_dpir* m = dpir_new(device, rows, cols);
  size_t words = rows * cols;
  const size_t chunk = (size_t)1 << 30;
  for (size_t off = 0; off < words; off += chunk) {
    size_t cur = std::min(chunk, words - off);
    k_dpir_synth<<<(unsigned)((cur + 255) / 256), 256, 0, m->stream>>>(m->a.p + off, cur, seed, off);
  }
  cudaError_t e = cudaStreamSynchronize(m->stream);
  if (e != cudaSuccess) { b200pir_dpir_destroy(m); throw Error(B200PIR_E_CUDA, cudaGetErrorString(e)); }
  *out = m;
  API_END
}
// doublepir.rs:76-108 setup(): both matrix products on the tensor cores (dpir_gemm.cu), the rest as small kernels.  Host pointers.
int b200pir_dpir_setup(int device, const uint32_t* db, uint64_t l, uint64_t m, const uint32_t* a1, uint64_t n, const uint32_t* a2,
                       uint32_t p, uint64_t delta, uint64_t x, uint32_t* db_squished, uint32_t* h1_squished, uint32_t* a2_t,
                       uint32_t* h2) {
  API_BEGIN
  if (!db || !a1 || !a2 || !db_squished || !h1_squished || !a2_t || !h2) throw Error(B200PIR_E_BADARG, "null argument");
  if (!l || !m || !n || !x || !delta || l % x) throw Error(B200PIR_E_SHAPE, "setup: l must be a positive multiple of x");
  if (p < 2 || p > 1024) throw Error(B200PIR_E_UNSUPPORTED, "setup: p must be at most 2^10 (squish basis, database.rs:274)");
  int ndev = 0;
  B200_CUDA(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) throw Error(B200PIR_E_BADARG, "no such CUDA device (this library has no CPU path)");
  B200_CUDA(cudaSetDevice(device));
  cudaStream_t s = nullptr;
  B200_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
  try {
    const size_t lx = l / x, rows1 = n * delta * x, lx3 = lx + (3 - lx % 3) % 3;
    DevBuf<uint32_t> d_db(l * m), d_a1(m * n), d_a2(lx * n), d_h(l * n), d_hc(rows1 * lx), d_h2(rows1 * n);
    DevBuf<uint32_t> d_dbsq(l * ((m + 2) / 3)), d_h1sq(rows1 * ((lx + 2) / 3)), d_a2t(n * lx3);
    B200_CUDA(cudaMemcpyAsync(d_db.p, db, l * m * 4, cudaMemcpyHostToDevice, s));
    B200_CUDA(cudaMemcpyAsync(d_a1.p, a1, m * n * 4, cudaMemcpyHostToDevice, s));
    B200_CUDA(cudaMemcpyAsync(d_a2.p, a2, lx * n * 4, cudaMemcpyHostToDevice, s));
    launch_dpir_gemm(d_h.p, d_db.p, d_a1.p, l, m, n, s);                                   // h_1 = db.data * a_1
    launch_dpir_transpose_expand_concat(d_hc.p, d_h.p, l, n, p, (int)delta, x, s);        // transpose, expand, concat_cols
    launch_dpir_gemm(d_h2.p, d_hc.p, d_a2.p, rows1, lx, n, s);                             // h_2 = h_1 * a_2
    launch_dpir_add_squish(d_dbsq.p, d_db.p, l, m, p / 2, s);                              // db.data += p/2; db.squish()
    launch_dpir_add_squish(d_h1sq.p, d_hc.p, rows1, lx, p / 2, s);                         // h_1 += p/2; squish
    launch_dpir_pad_transpose(d_a2t.p, d_a2.p, lx, n, lx3, s);                             // a_2_copy
    B200_CUDA(cudaMemcpyAsync(db_squished, d_dbsq.p, d_dbsq.n * 4, cudaMemcpyDeviceToHost, s));
    B200_CUDA(cudaMemcpyAsync(h1_squished, d_h1sq.p, d_h1sq.n * 4, cudaMemcpyDeviceToHost, s));
    B200_CUDA(cudaMemcpyAsync(a2_t, d_a2t.p, d_a2t.n * 4, cudaMemcpyDeviceToHost, s));
    B200_CUDA(cudaMemcpyAsync(h2, d_h2.p, d_h2.n * 4, cudaMemcpyDeviceToHost, s));
    B200_CUDA(cudaStreamSynchronize(s));
    B200_CUDA(cudaGetLastError());
  } catch (...) { cudaStreamDestroy(s); throw; }
  cudaStreamDestroy(s);
  API_END
}
// &Matrix * &Matrix (matrix/ops.rs:169-191) for a left operand with small signed entries (|a| < 2^15): out = a * b mod 2^32
int b200pir_dpir_matmul(int device, const uint32_t* a, uint64_t a_rows, uint64_t a_cols, const uint32_t* b, uint64_t b_cols,
                        uint32_t* out) {
  API_BEGIN
  if (!a || !b || !out || !a_rows || !a_cols || !b_cols) throw Error(B200PIR_E_BADARG, "null or empty argument");
  int ndev = 0;
  B200_CUDA(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) throw Error(B200PIR_E_BADARG, "no such CUDA device (this library has no CPU path)");
  B200_CUDA(cudaSetDevice(device));
  for (size_t i = 0; i < (size_t)a_rows * a_cols; i++)
    if ((int32_t)a[i] < -32768 || (int32_t)a[i] > 32767) throw Error(B200PIR_E_UNSUPPORTED, "matmul: left operand entries must lie in [-2^15, 2^15)");
  DevBuf<uint32_t> da(a_rows * a_cols), dbm(a_cols * b_cols), dc(a_rows * b_cols);
  B200_CUDA(cudaMemcpy(da.p, a, da.n * 4, cudaMemcpyHostToDevice));
  B200_CUDA(cudaMemcpy(dbm.p, b, dbm.n * 4, cudaMemcpyHostToDevice));
  launch_dpir_gemm(dc.p, da.p, dbm.p, a_rows, a_cols, b_cols, nullptr);
  B200_CUDA(cudaMemcpy(out, dc.p, dc.n * 4, cudaMemcpyDeviceToHost));
  API_END
}
void b200pir_dpir_destroy(b200pir_dpir* m) {
  if (!m) return;
  cudaSetDevice(m->device);
  cudaDeviceSynchronize();
  if (m->own_stream && m->stream) cudaStreamDestroy(m->stream);
  delete m;
}
int b200pir_dpir_set_stream(b200pir_dpir* m, void* cuda_stream) {
  API_BEGIN
  if (!m) throw Error(B200PIR_E_BADARG, "null handle");
  std::lock_guard<std::mutex> lk(m->mu);
  cudaSetDevice(m->device);
  B200_CUDA(cudaStreamSynchronize(m->stream));                     // pending work on the old stream first
  if (m->own_stream && m->stream) cudaStreamDestroy(m->stream);
  m->stream = (cudaStream_t)cuda_stream;
  m->own_stream = false;
  API_END
}
int b200pir_dpir_matvec_packed_dev(b200pir_dpir* m, const uint32_t* b_dev, uint32_t* out_dev, int variant) {
  API_BEGIN
  if (!m || !b_dev || !out_dev) throw Error(B200PIR_E_BADARG, "null argument");
  std::lock_guard<std::mutex> lk(m->mu);
  cudaSetDevice(m->device);
  launch_dpir_matvec(out_dev, m->a.p, b_dev, m->rows, m->cols, variant, m->stream);
  B200_CUDA(cudaGetLastError());
  API_END
}
// matrix_mul_vec_packed over the row range [row_begin, row_begin + row_count)  (answer(): db.rows(start, batch), doublepir.rs:301)
int b200pir_dpir_matvec_packed_rows(b200pir_dpir* m, uint64_t row_begin, uint64_t row_count, const uint32_t* b, uint32_t* out) {
  API_BEGIN
  if (!m || !b || !out) throw Error(B200PIR_E_BADARG, "null argument");
  if (row_begin + row_count > m->rows) throw Error(B200PIR_E_SHAPE, "row range out of bounds");
  if (row_count == 0) return 0;
  std::lock_guard<std::mutex> lk(m->mu);
  cudaSetDevice(m->device);
  B200_CUDA(cudaMemcpyAsync(m->b.p, b, 3 * m->cols * 4, cudaMemcpyHostToDevice, m->stream));
  launch_dpir_matvec(m->out.p, m->a.p + row_begin * m->cols, m->b.p, row_count, m->cols, 0, m->stream);
  B200_CUDA(cudaMemcpyAsync(out, m->out.p, row_count * 4, cudaMemcpyDeviceToHost, m->stream));
  B200_CUDA(cudaStreamSynchronize(m->stream));
  B200_CUDA(cudaGetLastError());
  API_END
}
int b200pir_dpir_matrix_mul_transposed_packed(int device, const uint32_t* a, uint64_t a_rows, uint64_t a_cols, const uint32_t* b,
                                              uint64_t b_rows, uint64_t b_cols, uint32_t* out) {
  API_BEGIN
  if (!a || !b || !out) throw Error(B200PIR_E_BADARG, "null argument");
  if (b_cols != 3 * a_cols) throw Error(B200PIR_E_SHAPE, "b.cols must equal 3 * a.cols");
  B200_CUDA(cudaSetDevice(device));
  DevBuf<uint32_t> da(a_rows * a_cols), db_(b_rows * b_cols), dout(a_rows * b_rows);
  B200_CUDA(cudaMemcpy(da.p, a, da.n * 4, cudaMemcpyHostToDevice));
  B200_CUDA(cudaMemcpy(db_.p, b, db_.n * 4, cudaMemcpyHostToDevice));
  launch_dpir_mul_transposed(dout.p, da.p, db_.p, a_rows, a_cols, b_rows, b_cols, 0);
  B200_CUDA(cudaMemcpy(out, dout.p, dout.n * 4, cudaMemcpyDeviceToHost));
  B200_CUDA(cudaGetLastError());
  API_END
}
int b200pir_dpir_transpose_expand_concat_cols_squish(int device, const uint32_t* a, uint64_t rows, uint64_t cols, uint64_t modulus,
                                                     uint64_t delta, uint64_t concat, uint32_t* out, uint64_t* out_rows,
                                                     uint64_t* out_cols) {
  API_BEGIN
  if (!a || !out) throw Error(B200PIR_E_BADARG, "null argument");
  if (modulus < 2 || modulus > 1024 || delta == 0 || concat == 0) throw Error(B200PIR_E_BADARG, "bad modulus / delta / concat");
  if (rows % concat) throw Error(B200PIR_E_SHAPE, "rows must be a multiple of concat");
  B200_CUDA(cudaSetDevice(device));
  const uint64_t orows = cols * delta * concat, ocols = (rows / concat + 2) / 3;
  DevBuf<uint32_t> da(rows * cols), dout(orows * ocols);
  B200_CUDA(cudaMemcpy(da.p, a, da.n * 4, cudaMemcpyHostToDevice));
  launch_dpir_transpose_expand(dout.p, da.p, rows, cols, modulus, delta, concat, orows, ocols, 0);
  B200_CUDA(cudaMemcpy(out, dout.p, dout.n * 4, cudaMemcpyDeviceToHost));
  if (out_rows) *out_rows = orows;
  if (out_cols) *out_cols = ocols;
  B200_CUDA(cudaGetLastError());
  API_END
}

int b200pir_dpir_matvec_packed(b200pir_dpir* m, const uint32_t* b, uint32_t* out) {
  API_BEGIN
  if (!m || !b || !out) throw Error(B200PIR_E_BADARG, "null argument");
  std::lock_guard<std::mutex> lk(m->mu);
  cudaSetDevice(m->device);
  B200_CUDA(cudaMemcpyAsync(m->b.p, b, 3 * m->cols * 4, cudaMemcpyHostToDevice, m->stream));
  launch_dpir_matvec(m->out.p, m->a.p, m->b.p, m->rows, m->cols, 0, m->stream);
  B200_CUDA(cudaMemcpyAsync(out, m->out.p, m->rows * 4, cudaMemcpyDeviceToHost, m->stream));
  B200_CUDA(cudaStreamSynchronize(m->stream));
  B200_CUDA(cudaGetLastError());
  API_END
}

}  // extern "C"
