// C++ host-side mirror of the reference's Spiral server interface over the C ABI (b200pir.h).
// Same names, argument meaning and failure behaviour as lib/spiral-rs/src/{server,poly,ntt}.rs:
// shape violations that `assert!`/panic in the reference throw std::runtime_error here.
// Header-only; link with libb200pir.so.
#pragma once
#include "b200pir.h"
#include <cstdint>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

namespace spiral_rs {

inline void check(int rc) {
  if (rc != 0) throw std::runtime_error(std::string("b200pir: ") + b200pir_last_error());
}

// spiral_rs::params::Params (params.rs:49-82) + the GPU context built from it
struct Params {
  b200pir_params p{};
  b200pir_ctx* ctx = nullptr;
  size_t poly_len = 2048, crt_count = 2;
  uint64_t setup_bytes = 0, query_bytes = 0, response_bytes = 0;
  Params(const b200pir_params& params, int device = 0) : p(params) {
    check(b200pir_ctx_create(&p, device, &ctx));
    check(b200pir_ctx_sizes(ctx, &setup_bytes, &query_bytes, &response_bytes));
  }
  ~Params() { b200pir_ctx_destroy(ctx); }
  Params(const Params&) = delete;
  Params& operator=(const Params&) = delete;
  // workspace for `queries` concurrent queries allocated now instead of on first use
  void reserve(size_t queries) { check(b200pir_ctx_reserve(ctx, queries, (size_t)1 << p.nu_2)); }
  size_t dim0() const { return (size_t)1 << p.nu_1; }
  size_t num_per() const { return (size_t)1 << p.nu_2; }
  size_t slices() const { return p.instances * p.n * p.n; }
};

// poly.rs:59-71
struct PolyMatrixRaw {
  size_t rows, cols;
  std::vector<uint64_t> data;          // rows*cols*2048
  PolyMatrixRaw(size_t r, size_t c) : rows(r), cols(c), data(r * c * 2048, 0) {}
};
struct PolyMatrixNTT {
  size_t rows, cols;
  std::vector<uint64_t> data;          // rows*cols*2*2048
  PolyMatrixNTT(size_t r, size_t c) : rows(r), cols(c), data(r * c * 2 * 2048, 0) {}
};

// client.rs:146-152, resident in HBM
struct PublicParameters {
  b200pir_pp* h = nullptr;
  PublicParameters(const Params& params, const std::vector<uint64_t>& v_packing,
                   const std::vector<uint64_t>* v_expansion_left, const std::vector<uint64_t>* v_expansion_right,
                   const std::vector<uint64_t>* v_conversion) {
    check(b200pir_pp_create(params.ctx, v_packing.data(), v_expansion_left ? v_expansion_left->data() : nullptr,
                            v_expansion_right ? v_expansion_right->data() : nullptr,
                            v_conversion ? v_conversion->data() : nullptr, &h));
  }
  // PublicParameters::deserialize (client.rs:212-259): seed || rows 1.. of every matrix
  PublicParameters(const Params& params, const uint8_t* data, size_t len) {
    check(b200pir_pp_create_from_bytes(params.ctx, data, len, &h));
  }
  ~PublicParameters() { b200pir_pp_destroy(h); }
  PublicParameters(const PublicParameters&) = delete;
};

// client.rs:262-267 after deserialisation
struct Query {
  std::vector<uint64_t> ct;      // expand_queries: PolyMatrixRaw(2,1)
  std::vector<uint64_t> v_buf;   // direct upload
  std::vector<uint64_t> v_ct;
};

// The `db: &[u64]` argument, resident in HBM
struct Database {
  b200pir_db* h = nullptr;
  const Params& params;
  explicit Database(const Params& p, uint64_t shard_index = 0, uint64_t shard_count = 1) : params(p) {
    check(b200pir_db_create(p.ctx, shard_index, shard_count, &h));
  }
  Database(const Params& p, const uint64_t* words, size_t n_words) : Database(p) {
    check(b200pir_db_upload(p.ctx, h, words, n_words));
  }
  ~Database() { b200pir_db_destroy(h); }
  Database(const Database&) = delete;
  void upsert_item(uint64_t slice, uint64_t item_idx, const uint64_t* poly) {
    check(b200pir_db_upsert_item(params.ctx, h, slice, item_idx, poly));
  }
  // lib/server/src/db/loading.rs:361-377 update_many_items: returns largest_update
  uint64_t update_many_items(const uint8_t* body, size_t len) {
    uint64_t largest = 0;
    check(b200pir_db_update_many_items(params.ctx, h, body, len, &largest));
    return largest;
  }
};

namespace ntt {
inline void ntt_forward(const Params& params, uint64_t* operand_overall, size_t polys = 1) {   // ntt.rs:68
  check(b200pir_ntt_forward(params.ctx, operand_overall, polys));
}
inline void ntt_inverse(const Params& params, uint64_t* operand_overall, size_t polys = 1) {   // ntt.rs:213
  check(b200pir_ntt_inverse(params.ctx, operand_overall, polys));
}
}  // namespace ntt

namespace server {
// server.rs:155-162
inline void multiply_reg_by_database(std::vector<PolyMatrixNTT>& out, const Database& db, uint64_t slice,
                                     const uint64_t* v_firstdim, const Params& params) {
  std::vector<uint64_t> flat(params.num_per() * 4 * 2048);
  check(b200pir_multiply_reg_by_database(params.ctx, db.h, slice, v_firstdim, flat.data()));
  out.assign(params.num_per(), PolyMatrixNTT(2, 1));
  for (size_t i = 0; i < out.size(); i++) std::copy(flat.begin() + i * 8192, flat.begin() + (i + 1) * 8192, out[i].data.begin());
}
// server.rs:388-393
inline void fold_ciphertexts(const Params& params, std::vector<PolyMatrixRaw>& v_cts, const std::vector<PolyMatrixNTT>& v_folding,
                             const std::vector<PolyMatrixNTT>& v_folding_neg) {
  std::vector<uint64_t> cts, vf, vfn;
  for (auto& m : v_cts) cts.insert(cts.end(), m.data.begin(), m.data.end());
  for (auto& m : v_folding) vf.insert(vf.end(), m.data.begin(), m.data.end());
  for (auto& m : v_folding_neg) vfn.insert(vfn.end(), m.data.begin(), m.data.end());
  check(b200pir_fold_ciphertexts(params.ctx, cts.data(), v_cts.size(), vf.data(), vfn.empty() ? nullptr : vfn.data()));
  for (size_t i = 0; i < v_cts.size(); i++) std::copy(cts.begin() + i * 4096, cts.begin() + (i + 1) * 4096, v_cts[i].data.begin());
}
// server.rs:650-655
inline std::vector<uint8_t> process_query(const Params& params, const PublicParameters& public_params, const Query& query,
                                          const Database& db) {
  std::vector<uint8_t> out(params.response_bytes);
  size_t n = 0;
  check(b200pir_process_query(params.ctx, db.h, public_params.h, query.ct.empty() ? nullptr : query.ct.data(),
                              query.v_buf.empty() ? nullptr : query.v_buf.data(),
                              query.v_ct.empty() ? nullptr : query.v_ct.data(), out.data(), &n));
  out.resize(n);
  return out;
}
// Query::deserialize + process_query on `count` serialized queries back to back (bin/server.rs:99-141); both query modes
inline std::vector<uint8_t> process_query_bytes(const Params& params, const PublicParameters& public_params, const uint8_t* queries,
                                                size_t len, size_t count, const Database& db) {
  std::vector<uint8_t> out(count * params.response_bytes);
  size_t each = 0;
  check(b200pir_process_query_bytes(params.ctx, db.h, public_params.h, queries, len, count, out.data(), &each));
  return out;
}
// concurrent queries of different clients in one database pass: public_params[i] belongs to the sender of queries[i]
inline std::vector<std::vector<uint8_t>> process_queries(const Params& params, const std::vector<const PublicParameters*>& public_params,
                                                         const std::vector<const Query*>& queries, const Database& db) {
  if (public_params.size() != queries.size()) throw std::runtime_error("b200pir: one PublicParameters per query");
  std::vector<std::vector<uint8_t>> out(queries.size(), std::vector<uint8_t>(params.response_bytes));
  std::vector<b200pir_pp*> pps;
  std::vector<const uint64_t*> cts;
  std::vector<uint8_t*> outs;
  for (size_t i = 0; i < queries.size(); i++) {
    pps.push_back(public_params[i]->h);
    cts.push_back(queries[i]->ct.data());
    outs.push_back(out[i].data());
  }
  check(b200pir_process_queries(params.ctx, db.h, pps.data(), cts.data(), queries.size(), outs.data()));
  return out;
}
}  // namespace server
}  // namespace spiral_rs
