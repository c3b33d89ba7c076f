"""/update-row on the GPU: b200pir_db_update_many_items (lib/server/src/db/loading.rs:361-377) against the serial
restatement in update_bodies.py (built on the CPU oracle's update_item_raw), against per-item update_item_raw calls, with
malformed entries, on a sharded database, at the bench size, without steady-state allocation, and under concurrent
readers."""
import threading

import numpy as np
import pytest

import oracle_lib as O
import update_bodies as U
from test_gpu_parity import _gpu, setup_case, Q0, Q1

pytestmark = [pytest.mark.gpu]


def _empty(P):
    return np.zeros(P.slices * P.N * P.num_per * P.dim0, dtype=np.uint64)


def _firstdim(P, seed):
    rng = np.random.default_rng(seed)
    return (rng.integers(0, Q0, P.dim0 * 2 * P.N, dtype=np.uint64)
            | (rng.integers(0, Q1, P.dim0 * 2 * P.N, dtype=np.uint64) << np.uint64(32)))


def _assert_db_equals_image(S, P, G, gdb, img, v):
    view = img.reshape(P.slices, -1)
    for s in range(P.slices):
        assert np.array_equal(S.multiply_reg_by_database(G, gdb, s, v), P.multiply_reg_by_database(view[s], v)), s


def _decoded_bytes(P, cl, resp):
    dec = cl.decode_response(resp).reshape(P.slices, P.N)        # slice order == bucket chunk order
    return dec[:, :P.bytes_per_chunk].astype(np.uint8).reshape(-1)


def _padded(P, data):
    out = np.zeros(P.slices * P.bytes_per_chunk, dtype=np.uint8)
    out[: len(data)] = data
    return out


@pytest.mark.parametrize("fmt", [0, 1, 2])
def test_update_many_items_matches_oracle(fmt):
    S, P, cl, pp, db, G, gdb, gpp = setup_case("T")
    rng = np.random.default_rng(40 + fmt)
    entries = U.random_entries(rng, P, 300)                      # 256 items: many duplicates
    body = U.body(entries)
    img = _empty(P)
    ref_largest = U.update_many_items(P, body, img)
    wdb = S.Database(G, fmt=fmt)
    assert wdb.update_many_items(body) == ref_largest == max(4 + len(d) for _, d in entries)
    _assert_db_equals_image(S, P, G, wdb, img, _firstdim(P, 3))
    assert wdb.info()["present_items"] == P.slices * len({i for i, _ in entries})
    wdb.close()


def test_update_many_items_equals_per_item_calls_across_groups():
    """A body of more than three groups (4096 entries each): the same index recurs inside a group and across groups."""
    S, P, cl, pp, db, G, gdb, gpp = setup_case("T")
    rng = np.random.default_rng(50)
    full = P.slices * P.bytes_per_chunk
    entries = U.random_entries(rng, P, 3 * 4096 + 700, lengths=[0, 1, 100, full - 5, full])
    bulk, serial = S.Database(G), S.Database(G)
    bulk.update_many_items(U.body(entries))
    for idx, data in entries:
        serial.update_item_raw(idx, data)
    assert bulk.info()["present_items"] == serial.info()["present_items"]
    idxs = [entries[-1][0], entries[0][0]] + [int(i) for i in rng.integers(0, P.dim0 * P.num_per, 14)]
    qs = np.concatenate([cl.generate_query(i)["ct"] for i in idxs])
    a = S.process_query_batch(G, gpp, qs, bulk)
    b = S.process_query_batch(G, gpp, qs, serial)
    assert np.array_equal(a, b)
    last = {}
    for idx, data in entries:
        last[idx] = data
    for k, i in enumerate(idxs):
        exp = _padded(P, last[i]) if i in last else np.zeros(full, dtype=np.uint8)
        assert np.array_equal(_decoded_bytes(P, cl, a[k]), exp), i
    bulk.close()
    serial.close()


@pytest.mark.parametrize("case", ["truncated_prefix", "chunk_len_below_4", "past_the_end", "too_long", "bad_index"])
def test_malformed_entry_keeps_the_valid_prefix(case):
    S, P, cl, pp, db, G, gdb, gpp = setup_case("T")
    name, bad, tail = {m[0]: m for m in U.malformed(P)}[case]
    rng = np.random.default_rng(60)
    before = [e for e in U.random_entries(rng, P, 20) if e[0] != 200]
    after = [(200, rng.integers(0, 256, 64, dtype=np.uint8))] if tail else []
    body = U.body(before) + bad + U.body(after)
    img = _empty(P)
    with pytest.raises(RuntimeError):
        U.update_many_items(P, body, img)
    wdb = S.Database(G)
    with pytest.raises(S.B200PirError):
        wdb.update_many_items(body)
    _assert_db_equals_image(S, P, G, wdb, img, _firstdim(P, 4))
    assert wdb.info()["present_items"] == P.slices * len({i for i, _ in before})
    wdb.close()


def test_sharded_update_many_items_equals_unsharded():
    import torch
    from sdk_b200._lib import LIB, check
    S, P, cl, pp, db, G, gdb, gpp = setup_case("T")
    rng = np.random.default_rng(70)
    body = U.body(U.random_entries(rng, P, 200))
    whole = S.Database(G)
    whole.update_many_items(body)
    world = 2
    shards = [S.Database(G, shard_index=s, shard_count=world) for s in range(world)]
    for sh in shards:
        sh.update_many_items(body)
    assert sum(sh.info()["present_items"] for sh in shards) == whole.info()["present_items"]
    idxs = [1, 2, 77, P.dim0 * P.num_per - 1]
    qs = np.concatenate([cl.generate_query(i)["ct"] for i in idxs])
    count = len(idxs)
    d_q = torch.from_numpy(qs.view(np.int64)).cuda()
    ct_words = 4 * P.N
    gathered = torch.zeros(world * count * P.slices * ct_words, dtype=torch.int32, device="cuda")
    for s, sh in enumerate(shards):
        part = gathered[s * count * P.slices * ct_words:(s + 1) * count * P.slices * ct_words]
        check(LIB.b200pir_query_stage_a_dev(G._h, sh._h, gpp._h, d_q.data_ptr(), count, part.data_ptr()))
    out = torch.zeros(count * G.response_bytes, dtype=torch.uint8, device="cuda")
    check(LIB.b200pir_query_stage_b_dev(G._h, gpp._h, gathered.data_ptr(), world, count, out.data_ptr()))
    G.synchronize()
    got = out.cpu().numpy().reshape(count, G.response_bytes)
    for k in range(count):
        ref = S.process_query(G, gpp, S.Query(ct=qs[k * 2 * P.N:(k + 1) * 2 * P.N]), whole)
        assert np.array_equal(got[k], ref), k
    for h in shards + [whole]:
        h.close()


def test_s8_bulk_write_into_empty_database_decodes():
    """The bench configuration: 4096 full-size items bulk-written into an empty tcgen05 database (sparse: tile skipping)."""
    S = _gpu()
    P = O.Params.named("S8")
    cl = O.Client(P, 9)
    pp = cl.generate_keys()
    G = S.Params(**P.kw)
    gpp = S.PublicParameters(G, pp["pack"], pp.get("left"), pp.get("right"), pp.get("conv"))
    gdb = S.Database(G)
    assert gdb.info()["format"] == 2
    rng = np.random.default_rng(80)
    n_items = P.dim0 * P.num_per
    idxs = rng.choice(n_items, 4096 + 1, replace=False)
    full = P.slices * P.bytes_per_chunk
    data = {int(i): rng.integers(0, 256, full, dtype=np.uint8) for i in idxs[:-1]}
    assert gdb.update_many_items(U.body(data.items())) == 4 + full
    assert gdb.info()["present_items"] == P.slices * 4096
    ask = [int(i) for i in idxs[:15]] + [int(idxs[-1])]                 # the last one was never written
    out = S.process_query_batch(G, gpp, np.concatenate([cl.generate_query(i)["ct"] for i in ask]), gdb)
    for k, i in enumerate(ask):
        exp = data.get(i, np.zeros(full, dtype=np.uint8))
        assert np.array_equal(_decoded_bytes(P, cl, out[k]), exp), (k, i)
    for h in (gdb, gpp, G):
        h.close()


def test_repeated_update_many_items_allocates_nothing():
    import torch
    S, P, cl, pp, db, G, gdb, gpp = setup_case("T")
    rng = np.random.default_rng(90)
    body = U.body(U.random_entries(rng, P, 5000))
    wdb = S.Database(G)
    wdb.update_many_items(body)
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    wdb.update_many_items(body)
    torch.cuda.synchronize()
    assert torch.cuda.mem_get_info()[0] == free0
    wdb.close()


def test_concurrent_readers_see_whole_items():
    """Readers loop process_query (coalesced) on the items a writer keeps rewriting from content A to B and back: every
    decoded item is entirely A or entirely B."""
    S, P, cl, pp, db, G, gdb, gpp = setup_case("T")
    rng = np.random.default_rng(100)
    full = P.slices * P.bytes_per_chunk
    items = [int(i) for i in rng.choice(P.dim0 * P.num_per, 48, replace=False)]
    A = {i: rng.integers(0, 256, full, dtype=np.uint8) for i in items}
    B = {i: rng.integers(0, 256, full, dtype=np.uint8) for i in items}
    body_a, body_b = U.body(A.items()), U.body(B.items())
    wdb = S.Database(G)
    wdb.update_many_items(body_a)
    queries = {i: cl.generate_query(i)["ct"] for i in items[:8]}
    stop = threading.Event()
    bad, seen = [], {"A": 0, "B": 0}

    def reader(k):
        n = 0
        while not stop.is_set() or n < 4:
            i = items[(k + n) % 8]
            got = _decoded_bytes(P, cl, S.process_query(G, gpp, S.Query(ct=queries[i]), wdb))
            if np.array_equal(got, A[i]):
                seen["A"] += 1
            elif np.array_equal(got, B[i]):
                seen["B"] += 1
            else:
                bad.append(i)
            n += 1

    threads = [threading.Thread(target=reader, args=(k,)) for k in range(4)]
    for t in threads:
        t.start()
    for r in range(20):
        wdb.update_many_items(body_b if r % 2 == 0 else body_a)
    stop.set()
    for t in threads:
        t.join()
    assert not bad and seen["A"] + seen["B"] >= 16
    wdb.close()
