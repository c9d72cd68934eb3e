"""CPU reference of inside-range mode (cub_set_inside_range), built on the CPU oracle (oracle/oracle_py.py).

TEST INFRASTRUCTURE.  In range mode a voxel is inside when !(v < lower) && !(upper < v) in the pixel type; everything
after that predicate (faces, vertex order, ids, positions, the triangle split) is the oracle's iso-mode algorithm on the
resulting mask.  So the reference mesh is the oracle's mesh of a volume that has the same mask at iso 1: the inside
voxels carry 1 + their linear index, the outside ones 0.  The oracle's cell data of that volume is 1 + the index of
the generating voxel (txx:279-332), which gives the original pixel value of the voxel for every cell."""
from __future__ import annotations

import numpy as np

from util import oracle

LITERAL, CLOSED_FORM = 0, 1


def inside_range(vol: np.ndarray, lower, upper) -> np.ndarray:
    """the range predicate, per voxel, in the pixel type (a NaN pixel is inside)"""
    with np.errstate(invalid="ignore"):
        return ~(vol < np.array(lower).astype(vol.dtype)) & ~(np.array(upper).astype(vol.dtype) < vol)


def classify_range(vol: np.ndarray, lower, upper, words_per_row: int | None = None) -> np.ndarray:
    """the inside bitmask in the layout of oracle_py.classify: shape (z, y, words_per_row) uint32, padding bits zero"""
    wpr = words_per_row or (vol.shape[2] + 31) // 32
    bits = np.zeros(vol.shape[:2] + (wpr * 32,), np.uint8)
    bits[..., :vol.shape[2]] = inside_range(vol, lower, upper)
    return np.packbits(bits, axis=-1, bitorder="little").view("<u4").astype(np.uint32)


def index_volume(vol: np.ndarray, lower, upper) -> np.ndarray:
    """1 + linear index on the inside voxels, 0 elsewhere: the same mask as the range at iso 1"""
    assert vol.size < 2**32 - 1
    idx = np.arange(1, vol.size + 1, dtype=np.uint32).reshape(vol.shape)
    return np.ascontiguousarray(np.where(inside_range(vol, lower, upper), idx, np.uint32(0)))


def cuberille_range(vol: np.ndarray, lower, upper, *, cell_data=False, project=False, **kw):
    """the oracle's mesh of the voxels in [lower, upper] (no projection: a range has no iso-surface); cell data is the
    generating voxel's pixel, raw bits included"""
    assert not project, "range mode has no iso-surface to project onto"
    ref = oracle().cuberille(index_volume(vol, lower, upper), 1, cell_data=True, project=False, **kw)
    ref.cell_data = vol.reshape(-1)[ref.cell_data.astype(np.int64) - 1] if cell_data else None
    return ref
