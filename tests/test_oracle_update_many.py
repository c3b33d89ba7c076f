"""The restatement of update_many_items (lib/server/src/db/loading.rs:361-377) in update_bodies.py, the definition the GPU
bulk-write tests compare against: equal to the oracle's update_item_raw applied entry by entry onto the dense
[slice][z][ii][j] image, last entry wins, and a malformed entry leaves exactly the valid prefix applied."""
import numpy as np
import pytest

import oracle_lib as O
import update_bodies as U


@pytest.fixture(scope="module")
def P():
    return O.Params.named("T")


def _empty(P):
    return np.zeros(P.slices * P.N * P.num_per * P.dim0, dtype=np.uint64)


def _serial(P, entries, img=None):
    """entry by entry with the existing oracle update_item_raw"""
    img = _empty(P) if img is None else img
    view = img.reshape(P.slices, P.N, P.num_per, P.dim0)
    for idx, data in entries:
        view[:, :, idx % P.num_per, idx // P.num_per] = P.update_item_raw(np.asarray(data, dtype=np.uint8)).reshape(P.slices, P.N)
    return img


def test_update_many_equals_update_item_raw_per_entry(P):
    rng = np.random.default_rng(5)
    entries = U.random_entries(rng, P, 40)
    img = _empty(P)
    largest = U.update_many_items(P, U.body(entries), img)
    assert np.array_equal(img, _serial(P, entries))
    assert largest == max(4 + len(d) for _, d in entries)
    assert U.update_many_items(P, b"", img) == 0


def test_duplicates_resolve_to_last_occurrence(P):
    rng = np.random.default_rng(6)
    a, b, c = (rng.integers(0, 256, n, dtype=np.uint8) for n in (P.db_item_size, 17, 0))
    img = _empty(P)
    U.update_many_items(P, U.body([(9, a), (3, a), (9, b), (3, c)]), img)
    assert np.array_equal(img, _serial(P, [(9, b), (3, c)]))


@pytest.mark.parametrize("case", range(5))
def test_malformed_entry_raises_with_valid_prefix(P, case):
    name, bad, tail = U.malformed(P)[case]
    rng = np.random.default_rng(7)
    before = U.random_entries(rng, P, 6)
    after = [(200, rng.integers(0, 256, 64, dtype=np.uint8))] if tail else []
    img = _empty(P)
    with pytest.raises(RuntimeError):
        U.update_many_items(P, U.body(before) + bad + U.body(after), img)
    assert np.array_equal(img, _serial(P, before)), name
