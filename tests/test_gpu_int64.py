"""int64 and uint64 pixels on the device: every classification route, the meshes and projections of 64-bit volumes, the
label-map calls on 64-bit label maps, and the C++ adapter on itk::Image<unsigned long> / <long long>.

Bitmasks are compared with numpy's predicate in the pixel type, meshes with the CPU oracle's 64-bit instantiation
(tests/oracle64.py), bit for bit.  The volumes hold the values where 64-bit compares and conversions go wrong when they
are done in fewer bits: the type's extremes, +-2^53 and +-(2^53 + 2) where doubles start to skip integers, labels that
agree in their low 32 bits, and 2^60 + 2^36 + 1, whose float conversion differs from its conversion through double.

The tests marked gpu need a CUDA device; the others check the premises of the GPU tests and run anywhere."""
import os
import subprocess

import numpy as np
import pytest

import oracle64 as O64
import range_oracle as R
from test_gpu_pixel_edges import _count_params, _gpu_mesh, assert_same_mesh, set_borrowed_volume, unpack_bitmask
from util import ROOT, oracle, pkg, smooth_volume

gpu = pytest.mark.gpu

I64_TYPES = [np.int64, np.uint64]
I64_IDS = ["int64", "uint64"]
SPLIT = 2**60 + 2**36 + 1   # (float)v = 2^60 + 2^37, (float)(double)v = 2^60


# ---- values --------------------------------------------------------------------------------------------------------------
def top_double(dt):
    """the largest double below the type's maximum + 1: 2^63 - 1024 for int64, 2^64 - 2048 for uint64"""
    return 2**63 - 1024 if np.dtype(dt) == np.int64 else 2**64 - 2048


def value_pool64(dt):
    info = np.iinfo(dt)
    cand = {info.min, info.min + 1, -(2**53) - 2, -(2**53), -(2**53) + 1, -(2**32) - 5, -5, -1, 0, 1, 5, 2**32 + 5,
            2**53 - 1, 2**53, 2**53 + 1, 2**53 + 2, SPLIT, -SPLIT, 2**60, top_double(dt), info.max - 1, info.max}
    return np.array(sorted(v for v in cand if info.min <= v <= info.max), dtype=dt)


def iso_pool64(dt):
    """the pool values a double holds exactly: the isos and range bounds of the tests"""
    return [v for v in (int(x) for x in value_pool64(dt)) if int(float(v)) == v]


def pool_volume64(dt, shape, seed):
    rng = np.random.default_rng(seed)
    pool = value_pool64(dt)
    n = int(np.prod(shape))
    assert n >= pool.size
    raw = np.concatenate([pool, pool[rng.integers(0, pool.size, n - pool.size)]])
    return np.ascontiguousarray(raw[rng.permutation(n)].reshape(shape))


def inside_iso(vol, iso):
    return ~(vol < np.array(int(iso), vol.dtype))


def inside_range(vol, lo, hi):
    return ~(vol < np.array(int(lo), vol.dtype)) & ~(np.array(int(hi), vol.dtype) < vol)


def split_field(dt, shape, seed):
    """a smooth field 2^40 x [0, 120] on an offset (2^60 for uint64, -2^61 for int64) whose float and double conversions
    both round, with one voxel in five moved to the nearest value whose two conversion chains to float differ; the iso
    at the middle of the field"""
    f, _ = smooth_volume(shape, np.float64, seed=seed)
    rng = np.random.default_rng(seed + 1)
    mag = (np.rint(f * 2**40).astype(np.int64) + (2**60 if dt is np.uint64 else 2**60 + 2**47)).astype(np.uint64)
    split = rng.random(shape) < 0.2
    mag = np.where(split, (mag >> np.uint64(38) << np.uint64(38)) + np.uint64(2**36 + 1), mag)
    if dt is np.uint64:
        return np.ascontiguousarray(mag), 2**60 + 60 * 2**40
    return np.ascontiguousarray(-(mag.astype(np.int64))), -(2**60 + 2**47 + 60 * 2**40)


def test_value_premises():
    for dt in I64_TYPES:
        pool = value_pool64(dt)
        assert pool.dtype == np.dtype(dt) and SPLIT in pool.tolist() and np.iinfo(dt).max in pool.tolist()
        isos = iso_pool64(dt)
        assert top_double(dt) in isos and 2**53 + 2 in isos and 2**53 + 1 not in isos and SPLIT not in isos
        assert float(top_double(dt)) < 2.0 ** (63 if dt is np.int64 else 64)
        vol, iso = split_field(dt, (6, 7, 8), seed=3)
        v = [int(x) for x in vol.reshape(-1)]
        assert int(float(iso)) == iso and min(v) < iso < max(v)
        # the seeded voxels: float(double(v)) and the one-step float differ
        from test_int64_oracle import round_to_float32
        assert sum(round_to_float32(x) != float(np.float32(float(x))) for x in v) > len(v) // 10


# ---- classification routes -----------------------------------------------------------------------------------------------
# row length, borrowed pointer one pixel past a 16-byte boundary, fused kernel expected
ROUTES64 = {"fused": (36, False, True), "full_rows_unaligned": (512, True, False), "ragged33": (33, False, False),
            "ragged70_unaligned": (70, True, False)}


def _check(h, vol, fused, what, ranges):
    for lo, hi in ranges:
        if hi is None:
            h.clear_inside_range()
            h.count(_count_params(lo))
            want = inside_iso(vol, lo)
        else:
            h.set_inside_range(lo, hi)
            h.count(_count_params(0))
            want = inside_range(vol, lo, hi)
        assert h.count_was_fused() == fused, f"{what}: fused={h.count_was_fused()}"
        got = unpack_bitmask(h.bitmask(), vol.shape[2])
        bad = np.argwhere(got != want)
        assert bad.size == 0, f"{what} {lo, hi}: {len(bad)} voxels differ, first {bad[0]} = {vol[tuple(bad[0])]!r}"


def _ranges(dt):
    isos = iso_pool64(dt)
    pairs = [(isos[i], isos[j]) for i in range(0, len(isos), 2) for j in range(i, len(isos), 3)]
    return [(v, None) for v in isos] + pairs


@gpu
@pytest.mark.parametrize("route", sorted(ROUTES64))
@pytest.mark.parametrize("dt", I64_TYPES, ids=I64_IDS)
def test_classification_routes(dt, route):
    nx, misaligned, fused = ROUTES64[route]
    vol = pool_volume64(dt, (5, 9, nx), seed=nx)
    h = pkg().capi.Handle(0)
    buf = set_borrowed_volume(h, vol, 8) if misaligned else h.set_volume(vol)
    _check(h, vol, fused, f"{np.dtype(dt).name} {route}", _ranges(dt))
    h.close()
    del buf


@gpu
@pytest.mark.parametrize("dt", I64_TYPES, ids=I64_IDS)
def test_padded_route_meshes(dt):
    """image_border_faces (k_classify_padded) in iso and range mode against the oracle's mesh of the padded image"""
    O, P = oracle(), pkg()
    vol = pool_volume64(dt, (6, 7, 11), seed=4)
    h = P.capi.Handle(0)
    isos = iso_pool64(dt)
    for iso in isos[1::3]:
        h.set_volume(vol)
        got = _gpu_mesh(h, _count_params(iso, image_border_faces=1, save_pixel_as_cell_data=1))
        assert not h.count_was_fused()
        ref = O64.cuberille(vol, iso, triangles=False, project=False, cell_data=True, border_faces=True, mode=O.CLOSED_FORM)
        assert_same_mesh(got, ref, f"padded iso {iso}")
    for lo, hi in [(isos[1], isos[-2]), (2**53, 2**53 + 2), (0, 0)]:
        h.set_volume(vol)
        h.set_inside_range(lo, hi)
        got = _gpu_mesh(h, _count_params(0, image_border_faces=1, save_pixel_as_cell_data=1))
        ref = R.cuberille_range(vol, lo, hi, triangles=False, cell_data=True, border_faces=True, mode=O.CLOSED_FORM)
        assert_same_mesh(got, ref, f"padded range {lo, hi}")
    h.close()


# ---- which doubles are pixel values ----------------------------------------------------------------------------------------
REPRESENTABLE = {
    np.int64: ([-(2**63), 2**63 - 1024, 0.0, 2**53 + 2, -(2**53) - 2],
               [2.0**63, 2.0**64, -(2.0**63) - 2048, 0.5, float("nan"), float("inf")]),
    np.uint64: ([0.0, 2**64 - 2048, 2**63, 2**53 + 2],
                [2.0**64, -1.0, 0.5, float("nan"), -float("inf")]),
}


@gpu
@pytest.mark.parametrize("dt", I64_TYPES, ids=I64_IDS)
def test_iso_range_bounds_and_labels_must_be_pixel_values(dt):
    P = pkg()
    ok, bad = REPRESENTABLE[dt]
    h = P.capi.Handle(0)
    h.set_volume(np.zeros((2, 2, 4), dt))
    with pytest.raises(P.capi.CuberilleError, match="not representable"):
        h.set_inside_range(2**53 + 2, 2.0**64)

    for v in ok:
        h.count(_count_params(v))
        h.set_inside_range(v, v)
        h.clear_inside_range()
    for v in bad:
        p = _count_params(0)
        p.iso_value = v
        with pytest.raises(P.capi.CuberilleError, match="not representable"):
            h.count(p)
        for lo, hi in [(v, v), (0.0, v), (v, 2**53)]:
            with pytest.raises(P.capi.CuberilleError, match="not representable|NaN"):
                h.set_inside_range(lo, hi)
    # labels: the rule of the bounds, and (uint64) at most 2^63 - 1, the windows of cub_label_bounds
    for v in ok:
        if v <= 2**63 - 1024:
            h.run_labels(_count_params(0), [v])
    for v in bad + ([2.0**63, 2**64 - 2048] if dt is np.uint64 else []):
        with pytest.raises(P.capi.CuberilleError, match="not representable|largest label"):
            h.run_labels(_count_params(0), [v])
    with pytest.raises(ValueError, match="not exactly representable"):
        h.run_labels(_count_params(0), [2**53 + 1])
    with pytest.raises(P.capi.CuberilleError, match="given twice"):
        h.run_labels(_count_params(0), [2**53 + 2, 5, 2**53 + 2])
    h.close()


# ---- meshes ---------------------------------------------------------------------------------------------------------------
_C30, _S30 = float(np.cos(np.pi / 6)), float(np.sin(np.pi / 6))
ROT_X_30 = (1.0, 0.0, 0.0, 0.0, _C30, -_S30, 0.0, _S30, _C30)
MESH_MODES = {
    "quads": dict(triangles=False, project=False),
    "quads_cd_ids64": dict(triangles=False, project=False, cell_data=True, id_bytes=8),
    "tris_proj_cd": dict(triangles=True, project=True, cell_data=True),
    "tris_proj_oriented": dict(triangles=True, project=True, direction=ROT_X_30, spacing=(0.8, 1.0, 1.3)),
    "tris_proj_region_index": dict(triangles=True, project=True, region_index=(3, -7, 11), origin=(1.5, -2.0, 0.25)),
    "advanced": dict(triangles=True, project=True, method=1),
    "linesearch": dict(triangles=False, project=True, method=2),
}


def gpu_run(h, vol, iso, triangles, project, cell_data=False, id_bytes=4, direction=None, spacing=(1.0, 1.0, 1.0),
            origin=(0.0, 0.0, 0.0), region_index=(0, 0, 0), method=0):
    h.set_volume(vol, spacing, origin, direction)
    h.set_region_index(region_index)
    p = _count_params(iso, generate_triangles=int(triangles), project_vertices=int(project),
                      save_pixel_as_cell_data=int(cell_data), projection_method=method)
    return _gpu_mesh(h, p, id_bytes)


def oracle_run(vol, iso, id_bytes=4, **kw):
    return O64.cuberille(vol, iso, mode=oracle().CLOSED_FORM, **kw)


@gpu
@pytest.mark.parametrize("mode", sorted(MESH_MODES))
@pytest.mark.parametrize("dt", I64_TYPES, ids=I64_IDS)
def test_meshes_of_a_field_beyond_2_53(dt, mode):
    kw = MESH_MODES[mode]
    vol, iso = split_field(dt, (18, 20, 23), seed=21)
    h = pkg().capi.Handle(0)
    got = gpu_run(h, vol, iso, **kw)
    ref = oracle_run(vol, iso, **kw)
    assert ref.cells.shape[0] > 200
    assert_same_mesh(got, ref, f"{np.dtype(dt).name} {mode}")
    if kw.get("id_bytes") == 8:
        assert got[1].dtype == np.uint64
    h.close()


@gpu
@pytest.mark.parametrize("dt", I64_TYPES, ids=I64_IDS)
def test_projection_of_points_reads_both_conversions(dt):
    """cub_debug_project_points on the lattice points of the field against the oracle, every method"""
    P = pkg()
    vol, iso = split_field(dt, (12, 13, 14), seed=8)
    pts = O64.cuberille(vol, iso, triangles=False, project=False).points
    h = P.capi.Handle(0)
    h.set_volume(vol)
    for method in (0, 1, 2):
        p = _count_params(iso, project_vertices=1, projection_method=method)
        got = h.project_points(p, pts)
        ref = O64.project_points(vol, iso, pts, method=method)
        assert np.array_equal(got.view(np.uint32), ref.view(np.uint32)), method
    h.close()


@gpu
@pytest.mark.parametrize("dt", I64_TYPES, ids=I64_IDS)
def test_slabs_at_the_exact_projection_halo(dt):
    """three z-slabs whose buffers hold exactly the halo of cub_projection_halo_oriented: the concatenation is the
    whole-volume run bit for bit"""
    P = pkg()
    p0 = _count_params(0, generate_triangles=1, project_vertices=1, save_pixel_as_cell_data=1)
    below, above = P.capi.projection_halo(p0, (1.0, 1.0, 1.0))
    a = below + 4
    b = a + 6
    nz = b + above + 4
    vol, iso = split_field(dt, (nz, 10, 12), seed=33)
    p = _count_params(iso, generate_triangles=1, project_vertices=1, save_pixel_as_cell_data=1)
    h = P.capi.Handle(0)
    h.set_volume(vol)
    whole = _gpu_mesh(h, p)
    assert_same_mesh(whole, oracle_run(vol, iso, triangles=True, project=True, cell_data=True), "whole")
    pts, cells, cds, pb, cb = [], [], [], 0, 0
    for z0, z1 in [(0, a), (a, b), (b, nz)]:
        lo, hi = max(0, z0 - below), min(nz, z1 + above)
        h.set_volume(vol[lo:hi])
        h.set_slab(nz, lo, z0, z1)
        n_pts, n_quads = h.count(p)
        h.set_id_base(pb, cb)
        h.emit(4)
        x, y, c = h.fetch(want_cell_data=True)
        pts.append(x), cells.append(y), cds.append(c)
        pb, cb = pb + n_pts, cb + 2 * n_quads
    for x, y, name in zip(whole, (np.concatenate(pts), np.concatenate(cells), np.concatenate(cds)), ("points", "cells", "cd")):
        assert x.shape == y.shape and np.array_equal(x.view(np.uint8), y.view(np.uint8)), name
    h.close()


@gpu
@pytest.mark.parametrize("dt", I64_TYPES, ids=I64_IDS)
@pytest.mark.parametrize("box", ["in_place", "gathered"])
def test_regions_of_interest(dt, box):
    """a box of whole rows and slices (in place) and one that is copied (k_gather_box), projected, against the oracle
    on a copy of the box"""
    P = pkg()
    vol, iso = split_field(dt, (16, 18, 21), seed=12)
    lo, size = ((0, 0, 3), (21, 18, 10)) if box == "in_place" else ((2, 3, 4), (15, 13, 10))
    h = P.capi.Handle(0)
    h.set_volume(vol)
    h.set_region_of_interest(lo, size)
    p = _count_params(iso, generate_triangles=1, project_vertices=1, save_pixel_as_cell_data=1)
    got = _gpu_mesh(h, p)
    crop = np.ascontiguousarray(vol[lo[2]:lo[2] + size[2], lo[1]:lo[1] + size[1], lo[0]:lo[0] + size[0]])
    ref = oracle_run(crop, iso, triangles=True, project=True, cell_data=True, region_index=lo)
    assert ref.cells.shape[0] > 50
    assert_same_mesh(got, ref, box)
    h.close()


@gpu
@pytest.mark.parametrize("dt", I64_TYPES, ids=I64_IDS)
def test_async_pipeline_and_re_emit(dt):
    """cub_count_async / cub_emit_async / cub_finish with buffers sized by a smaller first run, then a second emission
    of the same count with 64-bit ids"""
    P = pkg()
    h = P.capi.Handle(0)
    for shape, seed in [((8, 9, 10), 1), ((20, 22, 26), 2)]:
        vol, iso = split_field(dt, shape, seed=seed)
        ref = oracle_run(vol, iso, triangles=True, project=True, cell_data=True)
        h.set_volume(vol)
        h.count_async(_count_params(iso, generate_triangles=1, project_vertices=1, save_pixel_as_cell_data=1))
        h.emit_async(4)
        assert h.finish() == (ref.points.shape[0], ref.cells.shape[0])
        assert_same_mesh(h.fetch(want_cell_data=True), ref, f"async {shape}")
        h.emit(8)
        got = h.fetch(want_cell_data=True)
        assert got[1].dtype == np.uint64
        assert_same_mesh(got, ref, f"re-emit {shape}")
    h.close()


@gpu
@pytest.mark.parametrize("dt", I64_TYPES, ids=I64_IDS)
def test_filter_mirror_threshold_clamp_and_run(dt):
    """filter.py clamps the threshold at the type's maximum (np.iinfo) and runs a 64-bit image end to end"""
    P = pkg()
    vol, iso = split_field(dt, (10, 11, 12), seed=5)
    f = P.CuberilleImageToMeshFilter.New()
    f.SetInput(P.Image(vol))
    f.SetProjectVertexSurfaceDistanceThreshold(1e300)
    assert f.GetProjectVertexSurfaceDistanceThreshold() == float(np.iinfo(dt).max)
    f.SetProjectVertexSurfaceDistanceThreshold(0.5)
    f.SetIsoSurfaceValue(iso)
    f.Update()
    m = f.GetOutput()
    ref = oracle_run(vol, iso, triangles=True, project=True)
    assert np.array_equal(m.cells.astype(np.uint64), ref.cells)
    assert np.array_equal(m.points.view(np.uint32), ref.points.view(np.uint32))
    f2 = P.CuberilleImageToMeshFilter.New()
    f2.SetInput(P.Image(vol))
    f2.SetIsoSurfaceValue(SPLIT)
    with pytest.raises(ValueError, match="not exactly representable"):
        f2.Update()


# ---- label maps -------------------------------------------------------------------------------------------------------------
def bounds64(vol, first, n):
    """{count, box} of labels first .. first + n - 1 compared in the pixel type"""
    out = np.zeros((n, 8), np.uint64)
    for i in range(n):
        k = first + i
        if not np.iinfo(vol.dtype).min <= k <= np.iinfo(vol.dtype).max:
            continue
        z, y, x = np.nonzero(vol == np.array(k, vol.dtype))
        if z.size:
            out[i] = [z.size, x.min(), y.min(), z.min(), x.max(), y.max(), z.max(), 0]
    return out


def label_volume(dt, values, shape=(9, 10, 37), seed=3):
    rng = np.random.default_rng(seed)
    vol = np.array(values, dt)[rng.integers(0, len(values), shape)]
    return np.ascontiguousarray(vol)


@gpu
@pytest.mark.parametrize("dt", I64_TYPES, ids=I64_IDS)
def test_label_bounds_compare_64_bit_keys(dt):
    """labels 5 and 2^32 + 5 (and 2^53 + 5) share low bits and are counted apart; negative int64 labels; on aligned and
    borrowed unaligned buffers"""
    P = pkg()
    values = [0, 5, 6, 2**32 + 5, 2**32 + 6, 2**53 + 5] + ([-5, -1, -(2**32) + 5, -(2**62)] if dt is np.int64 else [2**63 + 5])
    h = P.capi.Handle(0)
    for nx in (37, 64):
        vol = label_volume(dt, values, (9, 10, nx))
        for off in (0, 8, 24):
            buf = set_borrowed_volume(h, vol, off) if off else h.set_volume(vol)
            windows = [(0, 7), (5, 1), (2**32 + 4, 3), (2**53 + 5, 1)] + ([(-7, 10), (-(2**32), 8), (-(2**62), 2)]
                                                                          if dt is np.int64 else [])
            for first, n in windows:
                got = h.label_bounds(first, n)
                assert np.array_equal(got, bounds64(vol, first, n)), (nx, off, first, n)
            del buf
    h.close()


@gpu
@pytest.mark.parametrize("dt", I64_TYPES, ids=I64_IDS)
def test_label_windows_at_the_type_edges(dt):
    P = pkg()
    info = np.iinfo(dt)
    values = [info.min, info.min + 1, info.max - 1, info.max, 0, 2**63 - 1, 2**63 - 2] + ([2**63] if dt is np.uint64 else [])
    vol = label_volume(dt, values)
    h = P.capi.Handle(0)
    h.set_volume(vol)
    top = 2**63 - 1   # the last label a window reaches, in either type
    for first, n in [(int(info.min), 3), (top - 2, 3), (top, 1), (int(info.min), 65536)]:
        assert np.array_equal(h.label_bounds(first, n), bounds64(vol, first, n)), (first, n)
    for first, n in [(top - 1, 3), (top, 2)] + ([(-1, 2), (-(2**63), 1)] if dt is np.uint64 else []):
        with pytest.raises(P.capi.CuberilleError, match="not inside the pixel type's range"):
            h.label_bounds(first, n)
    h.close()


def label_map64(dt, labels, shape=(22, 24, 26), seed=7):
    """the ball map of test_gpu_labels with label i + 1 replaced by labels[i] and the background by 0"""
    from test_gpu_labels import blob_labels
    idx = blob_labels(shape, len(labels), np.uint8, seed)
    return np.ascontiguousarray(np.array([0] + list(labels), dt)[idx])


LABELS64 = {np.int64: [2**60, -5, 7, 2**32 + 7, -(2**62), 2**53 + 2, 2**63 - 1024],
            np.uint64: [2**60, 7, 2**32 + 7, 2**53 + 2, 2**63 - 1024, 5]}


@gpu
@pytest.mark.parametrize("dt", I64_TYPES, ids=I64_IDS)
@pytest.mark.parametrize("mode", ["quads", "triangles_cd", "quads_ids64_border"])
def test_run_labels_parts_equal_the_whole_volume_runs(dt, mode):
    P = pkg()
    kw = {"quads": dict(generate_triangles=0), "triangles_cd": dict(generate_triangles=1, save_pixel_as_cell_data=1),
          "quads_ids64_border": dict(generate_triangles=0, image_border_faces=1)}[mode]
    id_bytes = 8 if "ids64" in mode else 4
    labels = LABELS64[dt] + [0, 99]   # the background, and a label without voxels
    vol = label_map64(dt, LABELS64[dt])
    p = _count_params(0, **kw)
    cd = bool(p.save_pixel_as_cell_data)
    h = P.capi.Handle(0)
    h.set_volume(vol)
    po, co = h.run_labels(p, labels, id_bytes)
    mesh = h.fetch(want_cell_data=cd)
    assert po[-2] == po[-1] and co[-2] == co[-1]
    for i, k in enumerate(labels):
        h.set_volume(vol)
        h.set_inside_range(k, k)
        h.count(p)
        h.set_id_base(int(po[i]), int(co[i]))
        h.emit(id_bytes)
        one = h.fetch(want_cell_data=cd)
        p0, p1, c0, c1 = (int(v) for v in (po[i], po[i + 1], co[i], co[i + 1]))
        part = (mesh[0][p0:p1], mesh[1][c0:c1], None if mesh[2] is None else mesh[2][c0:c1])
        for x, y, name in zip(part, one, ("points", "cells", "cell data")):
            assert (x is None) == (y is None)
            if x is not None:
                assert x.shape == y.shape and np.array_equal(x.view(np.uint8), y.view(np.uint8)), f"label {k}: {name}"
        if cd and c1 > c0:
            assert np.all(mesh[2][c0:c1] == np.array(k, dt))
    assert sum(int(co[i + 1]) > int(co[i]) for i in range(len(labels))) >= len(labels) - 2
    h.close()


# ---- the C++ adapter ---------------------------------------------------------------------------------------------------------
def build_labels64_driver(out_dir):
    """tests/cpp/labels64_test01.cxx against the ITK stand-in and the library (the flags of tests/cpp/Makefile)"""
    pkg().build()
    exe = os.path.join(str(out_dir), "labels64_test01")
    lib = os.path.dirname(pkg().capi.lib_path())
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-Wall", "-Wextra", "-Wno-unused-parameter", "-Wno-unused-local-typedefs",
                           "-I", os.path.join(ROOT, "include"), "-I", os.path.join(ROOT, "tests", "itk_shim"),
                           os.path.join(ROOT, "tests", "cpp", "labels64_test01.cxx"), "-o", exe,
                           "-L", lib, "-lcuberille_cuda", "-Wl,-rpath," + lib])
    return exe


@gpu
def test_cpp_filter_on_64bit_images(tmp_path):
    """itk::Image<unsigned long, 3>: SetLabelValues parts equal the SetLabelValue runs; itk::Image<long long, 3>: an iso
    run with projection equals the oracle"""
    labels = LABELS64[np.uint64]
    vol = label_map64(np.uint64, labels)
    raw = str(tmp_path / "labels.raw")
    vol.tofile(raw)
    exe = build_labels64_driver(tmp_path)
    dims = [str(d) for d in vol.shape[::-1]]
    r = subprocess.run([exe, "Labels", raw, *dims, *[str(k) for k in labels + [0]]], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert f"Mesh of {len(labels) + 1} labels" in r.stdout
    # an unrepresentable label is refused by the adapter before the C-ABI rounds it
    r = subprocess.run([exe, "Labels", raw, *dims, str(2**53 + 1)], capture_output=True, text=True)
    assert r.returncode != 0 and "not exactly representable" in r.stderr
    vol, iso = split_field(np.int64, (14, 15, 16), seed=2)
    vol.tofile(raw)
    out = str(tmp_path / "iso.bin")
    r = subprocess.run([exe, "Iso", raw, *[str(d) for d in vol.shape[::-1]], str(iso), out], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    ref = oracle_run(vol, iso, triangles=True, project=True)
    n = ref.points.shape[0]
    data = np.fromfile(out, np.uint8)
    pts = data[:12 * n].view(np.float32).reshape(n, 3)
    cells = data[12 * n:].view(np.uint64).reshape(-1, 3)
    assert np.array_equal(cells, ref.cells) and np.array_equal(pts.view(np.uint32), ref.points.view(np.uint32))
