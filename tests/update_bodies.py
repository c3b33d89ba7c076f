"""/update-row bodies (lib/server/src/db/loading.rs:361-377): entries [u32 BE chunk_len][u32 BE db_idx][data] back to back,
and the serial restatement of update_many_items that the GPU bulk-write tests compare against."""
import struct

import numpy as np


def entry(idx, data):
    data = bytes(np.asarray(data, dtype=np.uint8))
    return struct.pack(">II", 4 + len(data), idx) + data


def body(entries):
    """entries: [(db_idx, data bytes / uint8 array)]"""
    return b"".join(entry(i, d) for i, d in entries)


def random_entries(rng, P, count, lengths=None):
    """`count` entries with random indices (duplicates likely when count is large against num_items) and data lengths
    drawn from `lengths` (default: 0, 1, a last chunk shorter than bytes_per_chunk, and the maximum)."""
    full = P.slices * P.bytes_per_chunk
    lengths = lengths or [0, 1, full - P.bytes_per_chunk // 2 - 3, full]
    out = []
    for _ in range(count):
        n = int(lengths[rng.integers(len(lengths))])
        out.append((int(rng.integers(P.dim0 * P.num_per)), rng.integers(0, 256, n, dtype=np.uint8)))
    return out


def update_many_items(P, body, db):
    """Restatement of update_many_items (loading.rs:361-377) -> update_item (:301-315) -> update_item_raw (:317-359), serial,
    onto the dense image `db` [slice][z][ii][j] (packed lo | hi << 32) in place; the item polynomials come from the CPU
    oracle's update_item_raw.  Returns largest_update (the longest chunk_len).  A malformed entry raises RuntimeError with
    every entry before it applied, as the reference leaves the database: `?` on InvalidLength or a bad index, a slice panic
    on a truncated length prefix, a chunk_len below 4 or one running past the end of the body."""
    body = bytes(body)
    view = db.reshape(P.slices, P.N, P.num_per, P.dim0)
    max_len = 4 + P.slices * P.bytes_per_chunk
    offs, largest = 0, 0
    while offs < len(body):
        if len(body) - offs < 4:
            raise RuntimeError("truncated entry length")
        (chunk_len,) = struct.unpack_from(">I", body, offs)
        if chunk_len > len(body) - offs - 4:
            raise RuntimeError("entry runs past the end of the body")
        largest = max(largest, chunk_len)
        if chunk_len > max_len:
            raise RuntimeError("update too long")                      # InvalidLength
        if chunk_len < 4:
            raise RuntimeError("entry shorter than its db_idx")
        (idx,) = struct.unpack_from(">I", body, offs + 4)
        if idx >= P.dim0 * P.num_per:
            raise RuntimeError("bad db idx")
        data = np.frombuffer(body, dtype=np.uint8, count=chunk_len - 4, offset=offs + 8)
        view[:, :, idx % P.num_per, idx // P.num_per] = P.update_item_raw(data).reshape(P.slices, P.N)
        offs += 4 + chunk_len
    return largest


# each way an entry can be malformed: (name, raw bytes of the bad entry, whether entries may follow it).  A truncated length
# prefix is necessarily the end of the body; an entry running past the end swallows whatever follows it.
def malformed(P):
    full = P.slices * P.bytes_per_chunk
    return [
        ("truncated_prefix", b"\x00\x00", False),
        ("chunk_len_below_4", struct.pack(">I", 3) + b"\x00\x00\x00", True),
        ("past_the_end", struct.pack(">II", 0x7FFFFFFF, 1) + b"\x07" * 50, True),
        ("too_long", struct.pack(">II", 4 + full + 1, 1) + b"\x07" * (full + 1), True),
        ("bad_index", struct.pack(">II", 4 + 8, P.dim0 * P.num_per) + b"\x07" * 8, True),
    ]
