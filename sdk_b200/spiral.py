"""Host-side mirror of the reference's Spiral server interface over the C ABI.

Names, argument meaning and error behaviour follow lib/spiral-rs/src/{server,ntt,poly}.rs: the same
functions exist (process_query, multiply_reg_by_database, fold_ciphertexts, ntt_forward, ...),
they take the same data in the same layouts (numpy uint64 arrays standing in for &[u64] /
AlignedMemory64), and shape violations raise (the reference panics).  All arithmetic happens in the
CUDA library; this module never computes."""
import ctypes as C

import numpy as np

from ._lib import LIB, CParams, check, B200PirError  # noqa: F401

POLY_LEN = 2048          # lib/spiral-rs/src/util.rs:246
CRT_COUNT = 2
MODULI = (268369921, 249561089)   # util.rs:247


def _ptr(a, dtype=np.uint64):
    if a is None:
        return None
    if not isinstance(a, np.ndarray) or a.dtype != dtype or not a.flags["C_CONTIGUOUS"]:
        raise TypeError("expected a C-contiguous numpy array of dtype %s" % np.dtype(dtype).name)
    return a.ctypes.data


def _need(a, words, what):
    """The C ABI takes no lengths for these buffers (as the Rust functions take slices whose lengths they assert): check here,
    so a short array is a ValueError and not an out-of-bounds read inside cudaMemcpy."""
    if a is not None and a.size != words:
        raise ValueError("%s must hold %d words, got %d" % (what, words, a.size))


class Params:
    """spiral_rs::params::Params (params.rs:49-82) + the GPU context built from it."""

    FIELDS = ("n", "nu_1", "nu_2", "p", "q2_bits", "t_gsw", "t_conv", "t_exp_left", "t_exp_right", "instances",
              "db_item_size", "version")

    def __init__(self, device=0, expand_queries=True, **kw):
        cp = CParams()
        for k in self.FIELDS:
            v = int(kw.get(k, 1 if k == "instances" else 0))
            setattr(cp, k, v)
            setattr(self, k, v)
        cp.expand_queries = 1 if expand_queries else 0
        self.expand_queries = bool(expand_queries)
        h = C.c_void_p()
        check(LIB.b200pir_ctx_create(C.byref(cp), int(device), C.byref(h)))
        self._h = h
        self.device = device
        self.poly_len = POLY_LEN
        self.crt_count = CRT_COUNT
        self.dim0 = 1 << self.nu_1
        self.num_per = 1 << self.nu_2
        self.slices = self.instances * self.n * self.n
        sb, qb, rb = C.c_uint64(), C.c_uint64(), C.c_uint64()
        check(LIB.b200pir_ctx_sizes(self._h, C.byref(sb), C.byref(qb), C.byref(rb)))
        self.setup_bytes, self.query_bytes, self.response_bytes = sb.value, qb.value, rb.value
        import math
        W = POLY_LEN * CRT_COUNT
        self.g = int(math.ceil(math.log2(self.t_gsw * self.nu_2 + self.dim0)))
        self.stop_round = int(math.ceil(math.log2(self.t_gsw * self.nu_2))) if self.nu_2 else 0
        self.num_packing = self.n if self.version == 0 else 2
        self.has_right = self.expand_queries and (self.version == 0 or self.t_exp_right != self.t_exp_left)
        # word counts of the matrices of PublicParameters (client.rs:146-152) and of the stage-level operands
        self.words = dict(pack=self.num_packing * (self.n + 1) * self.t_conv * W, left=self.g * 2 * self.t_exp_left * W,
                          right=(self.stop_round + 1) * 2 * self.t_exp_right * W, conv=2 * 2 * self.t_conv * W,
                          v_folding=self.nu_2 * 2 * 2 * self.t_gsw * W, v_buf=self.dim0 * 2 * POLY_LEN,
                          v_ct=self.nu_2 * 2 * 2 * self.t_gsw * POLY_LEN, ct=2 * POLY_LEN, v=(1 << self.g) * 2 * W)

    @classmethod
    def from_json(cls, obj, device=0):
        """params_from_json_obj (util.rs:224-263)."""
        kw = dict(n=obj["n"], nu_1=obj["nu_1"], nu_2=obj["nu_2"], p=obj["p"], q2_bits=obj["q2_bits"],
                  t_gsw=obj["t_gsw"], t_conv=obj["t_conv"], t_exp_left=obj["t_exp_left"],
                  t_exp_right=obj["t_exp_right"], instances=obj.get("instances", 1),
                  db_item_size=obj.get("db_item_size", 0), version=obj.get("version", 0))
        return cls(device=device, expand_queries="direct_upload" not in obj, **kw)

    def close(self):
        if getattr(self, "_h", None):
            LIB.b200pir_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_option(self, key, value):
        check(LIB.b200pir_ctx_set_option(self._h, key.encode(), int(value)))

    def reserve(self, queries, rows_local=None):
        """Allocate the workspace for `queries` concurrent queries now instead of on first use."""
        check(LIB.b200pir_ctx_reserve(self._h, int(queries), int(rows_local if rows_local is not None else self.num_per)))

    def set_stream(self, cuda_stream):
        check(LIB.b200pir_ctx_set_stream(self._h, C.c_void_p(int(cuda_stream))))

    def synchronize(self):
        check(LIB.b200pir_ctx_synchronize(self._h))

    def last_stage_ms(self):
        out = (C.c_double * 9)()
        check(LIB.b200pir_last_stage_ms(self._h, out))
        keys = ("expand", "multiply", "from_ntt", "fold", "pack", "encode", "total", "multiply_launches", "query_image")
        return dict(zip(keys, list(out)))


class Database:
    """The `db: &[u64]` argument of process_query, resident in HBM."""

    def __init__(self, params, shard_index=0, shard_count=1, fmt=None):
        """fmt: 0 = IMAD layout (CUDA-core kernel, at most 4 queries per pass), 1 = mma.sync fragment order,
        2 = tcgen05 tile images (16 queries per pass); None = the context's "db_format" option (default -1 = automatic:
        2 wherever the tcgen05 kernel supports the geometry, else 1).  An explicit fmt applies to this database only."""
        self.params = params
        h = C.c_void_p()
        if fmt is not None:
            params.set_option("db_format", fmt)
        try:
            check(LIB.b200pir_db_create(params._h, shard_index, shard_count, C.byref(h)))
        finally:
            if fmt is not None:
                params.set_option("db_format", -1)
        self._h = h
        self.shard_index, self.shard_count = shard_index, shard_count

    @classmethod
    def from_words(cls, params, db, fmt=None):
        """db: the reference's dense layout [instance][trial][z][ii][j] (server.rs:263-266)."""
        self = cls(params, fmt=fmt)
        check(LIB.b200pir_db_upload(params._h, self._h, _ptr(db), db.size))
        return self

    @classmethod
    def from_file(cls, params, path, fmt=None, shard_index=0, shard_count=1):
        """load_preprocessed_db_from_file (server.rs:373-386): native-endian u64 stream of the whole database."""
        self = cls(params, shard_index=shard_index, shard_count=shard_count, fmt=fmt)
        check(LIB.b200pir_db_load_file(params._h, self._h, str(path).encode()))
        return self

    @classmethod
    def from_raw_file(cls, params, path, fmt=None, shard_index=0, shard_count=1):
        """load_db_from_seek (server.rs:320-357): raw item bytes, item i at byte i * db_item_size."""
        self = cls(params, shard_index=shard_index, shard_count=shard_count, fmt=fmt)
        check(LIB.b200pir_db_load_raw_file(params._h, self._h, str(path).encode()))
        return self

    def upload_slice(self, slice_idx, words):
        check(LIB.b200pir_db_upload_slice(self.params._h, self._h, slice_idx, _ptr(words), words.size))

    def upsert_item(self, slice_idx, item_idx, poly):
        if poly.size != POLY_LEN:
            raise ValueError("item polynomial must have 2048 packed words")
        check(LIB.b200pir_db_upsert_item(self.params._h, self._h, slice_idx, item_idx, _ptr(poly)))

    def update_item_raw(self, db_idx, data):
        """lib/server/src/db/loading.rs:317-359: write the raw bucket bytes of item db_idx."""
        data = np.ascontiguousarray(data, dtype=np.uint8)
        check(LIB.b200pir_db_update_item_raw(self.params._h, self._h, db_idx, data.ctypes.data, data.size))

    def update_many_items(self, body):
        """lib/server/src/db/loading.rs:361-377 (the /update-row body): entries [u32 BE chunk_len][u32 BE db_idx][data]
        applied in order, the last entry of an item winning; returns largest_update (the longest chunk_len).  body: bytes or
        a uint8 array.  A malformed entry raises B200PirError with the entries before it written."""
        body = np.frombuffer(body, dtype=np.uint8) if isinstance(body, (bytes, bytearray, memoryview)) else \
            np.ascontiguousarray(body, dtype=np.uint8)
        largest = C.c_uint64(0)
        check(LIB.b200pir_db_update_many_items(self.params._h, self._h, body.ctypes.data, body.size, C.byref(largest)))
        return largest.value

    def fill_synthetic(self, seed):
        check(LIB.b200pir_db_fill_synthetic(self.params._h, self._h, seed))

    def info(self):
        """{"format": resolved layout (0, 1 or 2), "local_rows": second-dimension rows on this GPU, "hbm_bytes": size}"""
        f, r, b = C.c_int(0), C.c_uint64(0), C.c_uint64(0)
        check(LIB.b200pir_db_info(self._h, C.byref(f), C.byref(r), C.byref(b)))
        it, cap = C.c_uint64(0), C.c_uint64(0)
        check(LIB.b200pir_db_present_items(self._h, C.byref(it), C.byref(cap)))
        return {"format": f.value, "local_rows": r.value, "hbm_bytes": b.value, "present_items": it.value, "capacity": cap.value}

    def close(self):
        if getattr(self, "_h", None):
            LIB.b200pir_db_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class PublicParameters:
    """spiral_rs::client::PublicParameters (client.rs:146-152), NTT form, resident in HBM."""

    def __init__(self, params, v_packing, v_expansion_left=None, v_expansion_right=None, v_conversion=None):
        self.params = params
        _need(v_packing, params.words["pack"], "v_packing")
        if params.expand_queries:
            _need(v_expansion_left, params.words["left"], "v_expansion_left")
            _need(v_expansion_right, params.words["right"], "v_expansion_right")
            _need(v_conversion, params.words["conv"], "v_conversion")
        h = C.c_void_p()
        check(LIB.b200pir_pp_create(params._h, _ptr(v_packing), _ptr(v_expansion_left), _ptr(v_expansion_right),
                                    _ptr(v_conversion), C.byref(h)))
        self._h = h

    @classmethod
    def deserialize(cls, params, data):
        """PublicParameters::deserialize (client.rs:212-259): seed || rows 1.. of every matrix."""
        data = np.ascontiguousarray(np.frombuffer(data, dtype=np.uint8) if isinstance(data, (bytes, bytearray)) else data,
                                    dtype=np.uint8)
        self = cls.__new__(cls)
        self.params = params
        h = C.c_void_p()
        check(LIB.b200pir_pp_create_from_bytes(params._h, _ptr(data, np.uint8), data.size, C.byref(h)))
        self._h = h
        return self

    def close(self):
        if getattr(self, "_h", None):
            LIB.b200pir_pp_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Query:
    """spiral_rs::client::Query (client.rs:262-267) after deserialisation."""

    def __init__(self, ct=None, v_buf=None, v_ct=None):
        self.ct, self.v_buf, self.v_ct = ct, v_buf, v_ct

    @classmethod
    def deserialize(cls, params, data):
        """Query::deserialize (client.rs:303-315), expand_queries parameter sets."""
        data = np.ascontiguousarray(np.frombuffer(data, dtype=np.uint8) if isinstance(data, (bytes, bytearray)) else data,
                                    dtype=np.uint8)
        ct = np.zeros(2 * POLY_LEN, dtype=np.uint64)
        check(LIB.b200pir_query_from_bytes(params._h, _ptr(data, np.uint8), data.size, _ptr(ct)))
        return cls(ct=ct)


# ---- lib/spiral-rs/src/ntt.rs
def ntt_forward(params, operand_overall):
    """ntt.rs:67-113.  In place over one or more [crt][2048] u64 polynomials."""
    if operand_overall.size % (CRT_COUNT * POLY_LEN):
        raise ValueError("operand must hold whole [2][2048] polynomials")
    check(LIB.b200pir_ntt_forward(params._h, _ptr(operand_overall), operand_overall.size // (CRT_COUNT * POLY_LEN)))


def ntt_inverse(params, operand_overall):
    """ntt.rs:212-258."""
    if operand_overall.size % (CRT_COUNT * POLY_LEN):
        raise ValueError("operand must hold whole [2][2048] polynomials")
    check(LIB.b200pir_ntt_inverse(params._h, _ptr(operand_overall), operand_overall.size // (CRT_COUNT * POLY_LEN)))


def ntt4096(params, operand_overall, inverse=False):
    """BASELINE config #5: the transforms of ntt.rs at poly_len = 4096, in place over [2][4096] u64 polynomials."""
    if operand_overall.size % (CRT_COUNT * 4096):
        raise ValueError("operand must hold whole [2][4096] polynomials")
    check(LIB.b200pir_ntt4096(params._h, _ptr(operand_overall), operand_overall.size // (CRT_COUNT * 4096), 1 if inverse else 0))


# ---- lib/spiral-rs/src/poly.rs
def to_ntt(params, raw):
    """poly.rs:613-623 (PolyMatrixRaw -> PolyMatrixNTT, any shape flattened)."""
    count = raw.size // POLY_LEN
    out = np.zeros(count * CRT_COUNT * POLY_LEN, dtype=np.uint64)
    check(LIB.b200pir_to_ntt(params._h, _ptr(out), _ptr(raw), count))
    return out


def from_ntt(params, ntt):
    """poly.rs:646-663."""
    count = ntt.size // (CRT_COUNT * POLY_LEN)
    out = np.zeros(count * POLY_LEN, dtype=np.uint64)
    check(LIB.b200pir_from_ntt(params._h, _ptr(out), _ptr(ntt), count))
    return out


# ---- lib/spiral-rs/src/server.rs
def multiply_reg_by_database(params, db, slice_idx, v_firstdim):
    """server.rs:155-221 on one (instance, trial) slice; returns num_per x PolyMatrixNTT(2,1)."""
    if v_firstdim.size != params.dim0 * 2 * POLY_LEN:
        raise ValueError("v_firstdim must hold dim0*2*poly_len words")
    rows = params.num_per // db.shard_count
    out = np.zeros(rows * 4 * POLY_LEN, dtype=np.uint64)
    check(LIB.b200pir_multiply_reg_by_database(params._h, db._h, slice_idx, _ptr(v_firstdim), _ptr(out)))
    return out


def fold_ciphertexts(params, v_cts, v_folding, v_folding_neg=None):
    """server.rs:388-427.  v_cts (num x 2 x 2048) is folded in place; result in v_cts[0].
    v_folding_neg=None means get_v_folding_neg(v_folding) (what process_query passes) and selects the
    library's fast path."""
    num = v_cts.size // (2 * POLY_LEN)
    if v_cts.size != num * 2 * POLY_LEN or num == 0 or num & (num - 1) or num > params.num_per:
        raise ValueError("v_cts must hold a power of two (<= num_per) of 2 x poly_len ciphertexts")
    _need(v_folding, params.words["v_folding"], "v_folding")
    _need(v_folding_neg, params.words["v_folding"], "v_folding_neg")
    check(LIB.b200pir_fold_ciphertexts(params._h, _ptr(v_cts), num, _ptr(v_folding), _ptr(v_folding_neg)))


def get_v_folding_neg(params, v_folding):
    """server.rs:505-523."""
    _need(v_folding, params.words["v_folding"], "v_folding")
    out = np.zeros_like(v_folding)
    check(LIB.b200pir_get_v_folding_neg(params._h, _ptr(out), _ptr(v_folding)))
    return out


def coefficient_expansion(params, public_params, v):
    """server.rs:19-121, in place over v = 2^g x PolyMatrixNTT(2,1)."""
    _need(v, params.words["v"], "v")
    check(LIB.b200pir_coefficient_expansion(params._h, public_params._h, _ptr(v)))


def expand_query(params, public_params, query):
    """server.rs:525-591 -> (v_reg_reoriented, v_folding)."""
    _need(query.ct, params.words["ct"], "query.ct")
    v_reg = np.zeros(params.dim0 * 2 * POLY_LEN, dtype=np.uint64)
    v_fold = np.zeros(max(1, params.nu_2 * 2 * 2 * params.t_gsw * CRT_COUNT * POLY_LEN), dtype=np.uint64)
    check(LIB.b200pir_expand_query(params._h, public_params._h, _ptr(query.ct), _ptr(v_reg), _ptr(v_fold)))
    return v_reg, v_fold


def pack(params, public_params, v_ct):
    """server.rs:429-468 / lib/server/src/compute/pack.rs (by params.version)."""
    _need(v_ct, params.n * params.n * 2 * POLY_LEN, "v_ct")
    out = np.zeros((params.n + 1) * params.n * CRT_COUNT * POLY_LEN, dtype=np.uint64)
    check(LIB.b200pir_pack(params._h, public_params._h, _ptr(v_ct), _ptr(out)))
    return out


def encode(params, v_packed_ct):
    """server.rs:470-503."""
    _need(v_packed_ct, params.instances * (params.n + 1) * params.n * POLY_LEN, "v_packed_ct")
    out = np.zeros(params.response_bytes, dtype=np.uint8)
    n = C.c_size_t(0)
    check(LIB.b200pir_encode(params._h, _ptr(v_packed_ct), _ptr(out, np.uint8), C.byref(n)))
    return out[: n.value]


def process_query(params, public_params, query, db):
    """spiral_rs::server::process_query (server.rs:650-741) -> response bytes."""
    if params.expand_queries:
        _need(query.ct, params.words["ct"], "query.ct")
    else:
        _need(query.v_buf, params.words["v_buf"], "query.v_buf")
        _need(query.v_ct, params.words["v_ct"], "query.v_ct")
    out = np.zeros(params.response_bytes, dtype=np.uint8)
    n = C.c_size_t(0)
    check(LIB.b200pir_process_query(params._h, db._h, public_params._h, _ptr(query.ct), _ptr(query.v_buf),
                                    _ptr(query.v_ct), _ptr(out, np.uint8), C.byref(n)))
    return out[: n.value]


def process_query_bytes(params, public_params, queries, db):
    """Query::deserialize + process_query on serialized queries (count x query_bytes back to back), the chain
    lib/server's private-read handler runs; returns count x response_bytes."""
    queries = np.ascontiguousarray(np.frombuffer(queries, dtype=np.uint8) if isinstance(queries, (bytes, bytearray))
                                   else queries, dtype=np.uint8)
    if queries.size % params.query_bytes:
        raise ValueError("queries must hold whole serialized queries")
    count = queries.size // params.query_bytes
    out = np.zeros(count * params.response_bytes, dtype=np.uint8)
    n = C.c_size_t(0)
    check(LIB.b200pir_process_query_bytes(params._h, db._h, public_params._h, _ptr(queries, np.uint8), queries.size, count,
                                          _ptr(out, np.uint8), C.byref(n)))
    return out.reshape(count, params.response_bytes)


def process_queries(params, public_params_list, query_cts, db):
    """Concurrent queries of DIFFERENT clients in one database pass: public_params_list[i] belongs to the client that sent
    query_cts[i] (each a PolyMatrixRaw(2,1) as u64 array).  Returns [count][response_bytes]."""
    count = len(query_cts)
    if len(public_params_list) != count:
        raise ValueError("one PublicParameters per query")
    cts = [np.ascontiguousarray(q, dtype=np.uint64) for q in query_cts]
    for q in cts:
        if q.size != 2 * POLY_LEN:
            raise ValueError("query ct must hold 2 x 2048 words")
    out = np.zeros((count, params.response_bytes), dtype=np.uint8)
    vp = C.c_void_p * count
    pps = vp(*[pp._h for pp in public_params_list])
    qs = vp(*[q.ctypes.data for q in cts])
    outs = vp(*[out[i].ctypes.data for i in range(count)])
    check(LIB.b200pir_process_queries(params._h, db._h, pps, qs, count, outs))
    return out


def coalesce_stats(params):
    """(batches, queries) served through the concurrent-caller combiner of this context so far."""
    b, q = C.c_uint64(0), C.c_uint64(0)
    check(LIB.b200pir_coalesce_stats(params._h, C.byref(b), C.byref(q)))
    return b.value, q.value


def process_query_batch(params, public_params, query_cts, db):
    """`count` expanded-mode queries of one client; the database is streamed once per group."""
    count = query_cts.size // (2 * POLY_LEN)
    _need(query_cts, count * 2 * POLY_LEN, "query_cts")
    out = np.zeros(count * params.response_bytes, dtype=np.uint8)
    n = C.c_size_t(0)
    check(LIB.b200pir_process_query_batch(params._h, db._h, public_params._h, _ptr(query_cts), count,
                                          _ptr(out, np.uint8), C.byref(n)))
    return out.reshape(count, params.response_bytes)
