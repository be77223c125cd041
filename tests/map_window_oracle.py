"""CPU restatement of gm_map_evict and gm_map_merge (include/gm_capi.h), TEST INFRASTRUCTURE ONLY.

A map is restated as its GMM1 file: leaf, and the voxels in key order with their counts and 2^-20 m fixed-point sums.
The window keeps a voxel iff its cell is within half_cells of the centre cell in every axis (integers); the centre cell
is float32 floor(x * inv_leaf) with inv_leaf = float32(1 / float32(leaf)), as gm_map_create and gm_map_insert compute it.
A merge adds counts and sums key by key, which is exact.
"""
from __future__ import annotations

import struct

import numpy as np

MAGIC, VERSION = 0x314D4D47, 1
_OFF = 1 << 20
_M21 = (1 << 21) - 1


def inv_leaf(leaf):
    return np.float32(1.0) / np.float32(leaf)


def center_cell(center3, leaf):
    """-> int64[3] centre cell, or None where gm_map_evict gives GM_ERR_INVALID_ARG (non-finite, out of the key range)."""
    c = np.asarray(center3, np.float32).reshape(3)
    with np.errstate(invalid="ignore", over="ignore"):
        f = np.floor(c * inv_leaf(leaf)).astype(np.float32)
    if not (np.abs(f) < np.float32(2.0e6)).all():
        return None
    cell = f.astype(np.int64)
    if ((cell < -_OFF) | (cell >= _OFF)).any():
        return None
    return cell


def unpack(keys):
    k = np.asarray(keys, np.uint64)
    return np.stack([(k & _M21).astype(np.int64) - _OFF, ((k >> 21) & _M21).astype(np.int64) - _OFF,
                     ((k >> 42) & _M21).astype(np.int64) - _OFF], axis=1)


def pack(ijk):
    a = np.asarray(ijk, np.int64) + _OFF
    return (a[:, 0] | (a[:, 1] << 21) | (a[:, 2] << 42)).astype(np.uint64)


def keep(ijk, cell, half_cells):
    """The window's predicate on integer cells (n x 3): max_a |ijk_a - cell_a| <= half_cells, in int64."""
    d = np.abs(np.asarray(ijk, np.int64).reshape(-1, 3) - np.asarray(cell, np.int64).reshape(1, 3))
    return d.max(axis=1) <= np.int64(half_cells)


def make(leaf, keys, counts, sums):
    """A map dict in key order (sorts and checks uniqueness)."""
    keys = np.asarray(keys, np.uint64)
    o = np.argsort(keys, kind="stable")
    keys = keys[o]
    assert (np.diff(keys.astype(np.uint64)) > 0).all(), "keys must be unique"
    return {"leaf": float(leaf), "keys": keys, "counts": np.asarray(counts, np.int32)[o],
            "sums": np.asarray(sums, np.int64).reshape(-1, 3)[o]}


def read_gmm1(path_or_bytes):
    b = path_or_bytes if isinstance(path_or_bytes, (bytes, bytearray)) else open(path_or_bytes, "rb").read()
    magic, version, leaf, V = struct.unpack_from("<IIdQ", b, 0)
    assert magic == MAGIC and version == VERSION and len(b) == 24 + 36 * V, (magic, version, V, len(b))
    o = 24
    keys = np.frombuffer(b, "<u8", V, o).astype(np.uint64)
    counts = np.frombuffer(b, "<i4", V, o + 8 * V).astype(np.int32)
    sums = np.frombuffer(b, "<i8", 3 * V, o + 12 * V).astype(np.int64).reshape(V, 3)
    return {"leaf": leaf, "keys": keys, "counts": counts, "sums": sums}


def write_gmm1(m) -> bytes:
    V = m["keys"].shape[0]
    return (struct.pack("<IIdQ", MAGIC, VERSION, m["leaf"], V) + m["keys"].astype("<u8").tobytes() +
            m["counts"].astype("<i4").tobytes() + m["sums"].astype("<i8").tobytes())


def subset(m, mask):
    return {"leaf": m["leaf"], "keys": m["keys"][mask], "counts": m["counts"][mask], "sums": m["sums"][mask]}


def evict(m, center3, half_cells):
    """-> (kept, evicted) maps of gm_map_evict(m, ..., center3, half_cells)."""
    cell = center_cell(center3, m["leaf"])
    assert cell is not None and half_cells >= 0
    k = keep(unpack(m["keys"]), cell, half_cells)
    return subset(m, k), subset(m, ~k)


def merge(a, b):
    """Key-wise sum of two maps of the same leaf (gm_map_merge, or two GMM1 segment files)."""
    assert np.float64(a["leaf"]).tobytes() == np.float64(b["leaf"]).tobytes()
    keys = np.concatenate([a["keys"], b["keys"]])
    u, inv = np.unique(keys, return_inverse=True)
    counts = np.zeros(u.shape[0], np.int64)
    sums = np.zeros((u.shape[0], 3), np.int64)
    np.add.at(counts, inv, np.concatenate([a["counts"], b["counts"]]).astype(np.int64))
    np.add.at(sums, inv, np.concatenate([a["sums"], b["sums"]]))
    return {"leaf": a["leaf"], "keys": u.astype(np.uint64), "counts": counts.astype(np.int32), "sums": sums}


def centroids(m):
    """float32 (V x 3) as gm_map_download: float((double)sum / 2^20 / count)."""
    return (m["sums"].astype(np.float64) / 1048576.0 / m["counts"].astype(np.float64)[:, None]).astype(np.float32)


def equal(a, b):
    return (a["keys"].shape == b["keys"].shape and np.array_equal(a["keys"], b["keys"]) and
            np.array_equal(a["counts"], b["counts"]) and np.array_equal(a["sums"], b["sums"]))
