"""Label maps: per-label bounds (cub_label_bounds), a region of interest (cub_set_region_of_interest), and every label
meshed in its own box in one call (cub_run_labels).

A label's mesh depends only on the voxels of that label and their neighbours, so meshing it on its bounding box grown
by one voxel and clipped to the image, with the box's first voxel as region index, gives the mesh of range mode on the
whole image bit for bit.  The CPU tests check that premise on the oracle alone; the GPU tests check the bounds against
numpy, the box against a numpy copy of it, and every part of cub_run_labels against the oracle and against the
whole-volume range run it replaces.

The tests marked gpu need a CUDA device; the others run anywhere."""
import os
import subprocess

import numpy as np
import pytest

import range_oracle as R
from test_gpu_inside_range import ORACLE_MODES, label_map
from test_gpu_pixel_edges import _count_params, _gpu_mesh, assert_same_mesh
from util import ROOT, oracle, pkg, smooth_volume

gpu = pytest.mark.gpu

INT_TYPES = [np.uint8, np.int8, np.uint16, np.int16, np.uint32, np.int32]
INT_IDS = [np.dtype(d).name for d in INT_TYPES]


# ---- references -------------------------------------------------------------------------------------------------------
def np_label_bounds(vol, first, n):
    """{count, xmin, ymin, zmin, xmax, ymax, zmax, 0} of labels first .. first + n - 1 by bincount and nonzero extremes"""
    out = np.zeros((n, 8), np.uint64)
    k = vol.astype(np.int64) - int(first)
    inside = (k >= 0) & (k < n)
    idx = k[inside]
    out[:, 0] = np.bincount(idx, minlength=n)
    zyx = np.nonzero(inside)
    for a, c in enumerate((zyx[2], zyx[1], zyx[0])):
        lo = np.full(n, np.iinfo(np.int64).max, np.int64)
        hi = np.full(n, -1, np.int64)
        np.minimum.at(lo, idx, c)
        np.maximum.at(hi, idx, c)
        present = out[:, 0] > 0
        out[present, 1 + a] = lo[present]
        out[present, 4 + a] = hi[present]
    return out


def grown_box(vol, k):
    """the bounding box of label k grown by one voxel and clipped to the image: (lo, size) in (x, y, z)"""
    z, y, x = np.nonzero(vol == k)
    dims = vol.shape[::-1]
    lo = [max(int(c.min()) - 1, 0) for c in (x, y, z)]
    hi = [min(int(c.max()) + 1, d - 1) for c, d in zip((x, y, z), dims)]
    return lo, [h - l + 1 for l, h in zip(lo, hi)]


def crop(vol, lo, size):
    return np.ascontiguousarray(vol[lo[2]:lo[2] + size[2], lo[1]:lo[1] + size[1], lo[0]:lo[0] + size[0]])


def blob_labels(shape, n, dtype, seed, full_xy_label=None):
    """a seeded label map: n balls of varied radius on background 0, labels 1..n in draw order (later balls cover
    earlier ones); full_xy_label adds a slab of that label across the whole x/y extent"""
    rng = np.random.default_rng(seed)
    vol = np.zeros(shape, dtype)
    nz, ny, nx = shape
    for lab in range(1, n + 1):
        r = int(rng.integers(2, max(3, min(shape) // 6)))
        c = [int(rng.integers(0, s)) for s in shape]
        sl = tuple(slice(max(ci - r, 0), min(ci + r + 1, s)) for ci, s in zip(c, shape))
        zz, yy, xx = np.ogrid[sl]
        ball = (zz - c[0]) ** 2 + (yy - c[1]) ** 2 + (xx - c[2]) ** 2 <= r * r
        vol[sl][ball] = lab
    if full_xy_label is not None:
        vol[nz // 2:nz // 2 + 3] = full_xy_label
    return np.ascontiguousarray(vol)


def same_bytes(a, b, what):
    for x, y, name in zip(a, b, ("points", "cells", "cell data")):
        assert (x is None) == (y is None), f"{what}: {name}"
        if x is not None:
            assert x.dtype == y.dtype and x.shape == y.shape, f"{what}: {name} {x.dtype}{x.shape} vs {y.dtype}{y.shape}"
            assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), f"{what}: {name} differ"


def part(mesh, po, co, i):
    """label i's part of a cub_run_labels mesh, point ids shifted back to 0"""
    pts, cells, cd = mesh
    p0, p1, c0, c1 = int(po[i]), int(po[i + 1]), int(co[i]), int(co[i + 1])
    return pts[p0:p1], cells[c0:c1] - cells.dtype.type(p0), None if cd is None else cd[c0:c1]


# ---- the equivalence premise, on the oracle alone -----------------------------------------------------------------------
@pytest.mark.parametrize("fixture", ["neghip", "fuel"])
def test_grown_box_mesh_is_the_whole_volume_mesh_in_the_oracle(fixture):
    """for every label (0 is the background and touches every image face), the oracle's range mesh of the grown,
    clipped box with region_index = lo equals its range mesh of the whole volume, cell data included"""
    O = oracle()
    vol = label_map(fixture, np.uint16)
    faces = 0
    for k in np.unique(vol):
        lo, size = grown_box(vol, k)
        faces += sum(l == 0 for l in lo) + sum(l + s == d for l, s, d in zip(lo, size, vol.shape[::-1]))
        for kw in (dict(triangles=False), dict(triangles=True), dict(triangles=False, border_faces=True)):
            whole = R.cuberille_range(vol, k, k, cell_data=True, mode=O.CLOSED_FORM, **kw)
            box = R.cuberille_range(crop(vol, lo, size), k, k, cell_data=True, mode=O.CLOSED_FORM, region_index=lo, **kw)
            assert whole.cells.shape[0] > 0
            for a, b, what in ((box.points, whole.points, "points"), (box.cells, whole.cells, "cells"),
                               (box.cell_data, whole.cell_data, "cell data")):
                assert a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8)), f"{fixture} {k} {kw}: {what}"
    assert faces >= 6


def test_np_label_bounds_reference():
    vol = np.array([[[3, 3, 0], [1, 0, 3]]], np.uint8)   # z=0, two rows
    b = np_label_bounds(vol, 0, 5)
    assert b[3].tolist() == [3, 0, 0, 0, 2, 1, 0, 0]
    assert b[1].tolist() == [1, 0, 1, 0, 0, 1, 0, 0]
    assert b[2].tolist() == [0] * 8 and b[4].tolist() == [0] * 8


def test_label_symbols_are_declared():
    P = pkg()
    for name in ("cub_label_bounds", "cub_set_region_of_interest", "cub_run_labels"):
        assert name in P.capi.SYMBOLS
        assert name + "(" in open(os.path.join(ROOT, "include", "cuberille_c.h")).read()


# ---- cub_label_bounds against numpy -------------------------------------------------------------------------------------
def check_bounds(h, vol, first, n, what):
    got = h.label_bounds(first, n)
    want = np_label_bounds(vol, first, n)
    if not np.array_equal(got, want):
        i = np.nonzero((got != want).any(axis=1))[0][0]
        raise AssertionError(f"{what}: label {first + i}: {got[i].tolist()} vs {want[i].tolist()}")


def windows(dt):
    info = np.iinfo(dt)
    w = [(info.min, 256), (info.max - 255, 256), (-3 if info.min < 0 else 0, 9), (1, 1)]
    if info.bits == 8:
        w.append((info.min, 256))
    else:
        w.append((info.min, 65536))
        w.append((info.max - 65535, 65536))
    return w


@gpu
@pytest.mark.parametrize("dtype", INT_TYPES, ids=INT_IDS)
def test_label_bounds_on_ragged_rows(dtype):
    """row lengths 1..67, seeded labels with values outside the window and the type's extremes"""
    P = pkg()
    dt = np.dtype(dtype)
    info = np.iinfo(dt)
    rng = np.random.default_rng(7)
    h = P.capi.Handle(0)
    for nx in range(1, 68):
        vol = rng.integers(-2, 10, size=(5, 3, nx)).astype(dt)
        vol.reshape(-1)[rng.integers(0, vol.size, 3)] = [info.min, info.max, info.max - 1]
        h.set_volume(vol)
        for first, n in [(0, 8), (-1 if info.min < 0 else 0, 12), (info.min, 4), (info.max - 3, 4)]:
            check_bounds(h, vol, first, n, f"{dt.name} nx={nx} [{first}, +{n})")
    h.close()


@gpu
@pytest.mark.parametrize("dtype", INT_TYPES, ids=INT_IDS)
def test_label_bounds_on_label_maps(dtype):
    """coherent maps (the fixtures, blobs), iid-random labels, one label everywhere, labels only in the eight corners,
    windows at the type's minimum and maximum"""
    P = pkg()
    dt = np.dtype(dtype)
    info = np.iinfo(dt)
    rng = np.random.default_rng(3)
    maps = {
        "neghip": label_map("neghip", dt),
        "fuel": label_map("fuel", dt),
        "blobs": blob_labels((40, 52, 70), 30, dt, seed=1, full_xy_label=31),
        "iid": rng.integers(max(info.min, -300), min(info.max, 300), size=(17, 33, 129)).astype(dt),
        "one": np.full((9, 10, 200), 5, dt),
        "extremes": rng.choice(np.array([info.min, info.min + 1, info.max - 1, info.max, 0, 1], dt), size=(7, 11, 93)),
    }
    corners = np.zeros((12, 13, 77), dt)
    for i, (z, y, x) in enumerate([(z, y, x) for z in (0, -1) for y in (0, -1) for x in (0, -1)]):
        corners[z, y, x] = i + 1
    maps["corners"] = corners
    h = P.capi.Handle(0)
    for name, vol in maps.items():
        h.set_volume(vol)
        for first, n in windows(dt):
            check_bounds(h, vol, first, n, f"{dt.name} {name} [{first}, +{n})")
    h.close()


@gpu
@pytest.mark.parametrize("dtype", INT_TYPES, ids=INT_IDS)
def test_label_bounds_of_borrowed_pointers_at_every_alignment(dtype):
    """a device volume at every pixel-aligned offset: the 16-byte loads give way to narrow ones at the row ends"""
    import torch
    P = pkg()
    dt = np.dtype(dtype)
    h = P.capi.Handle(0)
    for nx in (13, 64, 203):
        vol = blob_labels((11, 9, nx), 12, dt, seed=nx)
        vol[::3, ::2, ::5] = 7
        raw = torch.from_numpy(vol.reshape(-1).view(np.uint8).copy())
        buf = torch.zeros(raw.numel() + 64, dtype=torch.uint8, device="cuda")
        for off in range(0, 32, dt.itemsize):
            buf[off:off + raw.numel()].copy_(raw)
            torch.cuda.synchronize()
            h.set_volume_ptr(buf.data_ptr() + off, dt, vol.shape[::-1], P.capi.MEM_DEVICE)
            check_bounds(h, vol, 0, 16, f"{dt.name} nx={nx} offset {off}")
        del buf
    h.close()


@gpu
def test_label_bounds_refusals():
    P = pkg()
    h = P.capi.Handle(0)

    def refused(code, text, call, *args):
        with pytest.raises(P.capi.CuberilleError) as e:
            call(*args)
        assert e.value.code == code and text in str(e.value), str(e.value)

    refused(1, "before cub_set_volume", h.label_bounds, 0, 4)
    for dt in (np.float32, np.float64):
        h.set_volume(np.zeros((2, 3, 4), dt))
        refused(5, "integer", h.label_bounds, 0, 4)
    h.set_volume(np.zeros((4, 3, 4), np.uint8))
    refused(1, "n_labels", h.label_bounds, 0, 0)
    refused(1, "n_labels", h.label_bounds, 0, 65537)
    refused(1, "window", h.label_bounds, -1, 4)
    refused(1, "window", h.label_bounds, 250, 7)
    h.label_bounds(250, 6)
    h.set_volume(np.zeros((4, 3, 4), np.int16))
    refused(1, "window", h.label_bounds, -32769, 2)
    h.label_bounds(-32768, 65536)
    h.set_region_of_interest((0, 0, 1), (4, 3, 2))
    refused(1, "region of interest", h.label_bounds, 0, 4)
    h.clear_region_of_interest()
    h.label_bounds(0, 4)
    h.set_slab(4, 0, 0, 2)
    refused(1, "z-slab", h.label_bounds, 0, 4)
    h.close()


# ---- region of interest --------------------------------------------------------------------------------------------------
DIRECTION = (0.0, 1.0, 0.0, 0.0, 0.0, 1.0, 1.0, 0.0, 0.0)
ROI_MODES = {
    "project_default": (dict(generate_triangles=1, project_vertices=1), {}),
    "project_advanced": (dict(generate_triangles=1, project_vertices=1, projection_method=1), {}),
    "project_linesearch": (dict(generate_triangles=1, project_vertices=1, projection_method=2), {}),
    "triangles": (dict(generate_triangles=1), {}),
    "quads_u64_cell_data": (dict(save_pixel_as_cell_data=1), dict(id_bytes=8)),
    "raster": (dict(vertex_order=1, save_pixel_as_cell_data=1), {}),
    "border_faces": (dict(image_border_faces=1, generate_triangles=1), {}),
    "oriented_projected": (dict(generate_triangles=1, project_vertices=1), dict(direction=DIRECTION)),
}
GEO = dict(spacing=(0.7, 1.1, 1.3), origin=(1.5, -2.0, 0.25))


def boxes(shape):
    """(lo, size) in (x, y, z): every face touched, a 1-voxel box, whole rows and slices (used in place), gathered"""
    X, Y, Z = shape[::-1]
    return [([0, 0, 0], [X, Y, Z]), ([0, 0, 3], [X, Y, Z - 5]), ([0, 0, Z - 4], [X, Y, 4]),
            ([0, 2, 1], [X - 3, Y - 2, Z - 1]), ([3, 0, 0], [X - 3, 7, 5]), ([5, 4, 2], [9, 6, 7]),
            ([X - 6, Y - 5, Z - 4], [6, 5, 4]), ([7, 5, 3], [1, 1, 1])]


def box_and_copy(h, vol, lo, size, params, id_bytes=4, direction=None, inside_range=None, region_index=(2, -3, 5)):
    h.set_volume(vol, GEO["spacing"], GEO["origin"], direction)
    h.set_region_index(region_index)
    if inside_range:
        h.set_inside_range(*inside_range)
    h.set_region_of_interest(lo, size)
    a = _gpu_mesh(h, params, id_bytes)
    h.set_volume(crop(vol, lo, size), GEO["spacing"], GEO["origin"], direction)
    h.set_region_index([r + l for r, l in zip(region_index, lo)])
    if inside_range:
        h.set_inside_range(*inside_range)
    b = _gpu_mesh(h, params, id_bytes)
    return a, b


@gpu
@pytest.mark.parametrize("mode", sorted(ROI_MODES))
def test_region_of_interest_is_the_mesh_of_the_copied_box(mode):
    P = pkg()
    p_kw, kw = ROI_MODES[mode]
    vol, iso = smooth_volume((18, 21, 26), np.float32, seed=4)
    h = P.capi.Handle(0)
    for lo, size in boxes(vol.shape):
        a, b = box_and_copy(h, vol, lo, size, _count_params(iso, **p_kw), kw.get("id_bytes", 4), kw.get("direction"))
        same_bytes(a, b, f"{mode} box {lo}+{size}")
    h.close()


@gpu
@pytest.mark.parametrize("dtype", [np.uint8, np.int16, np.uint32], ids=lambda d: np.dtype(d).name)
def test_region_of_interest_in_range_mode(dtype):
    P = pkg()
    vol = blob_labels((17, 20, 37), 9, dtype, seed=5)
    h = P.capi.Handle(0)
    for lo, size in boxes(vol.shape):
        for p_kw in (dict(), dict(generate_triangles=1, save_pixel_as_cell_data=1), dict(vertex_order=1, image_border_faces=1)):
            a, b = box_and_copy(h, vol, lo, size, _count_params(0, **p_kw), inside_range=(2, 4))
            same_bytes(a, b, f"{np.dtype(dtype).name} box {lo}+{size} {p_kw}")
    h.close()


@gpu
def test_region_of_interest_sees_the_box_and_the_whole_box_is_no_box():
    P = pkg()
    vol, iso = smooth_volume((14, 15, 40), np.int16, seed=8)
    h = P.capi.Handle(0)
    h.set_volume(vol)
    p = _count_params(iso, generate_triangles=1, project_vertices=1)
    none = _gpu_mesh(h, p)
    h.set_region_of_interest((0, 0, 0), vol.shape[::-1])
    same_bytes(_gpu_mesh(h, p), none, "whole-volume box")
    for lo, size in boxes(vol.shape):
        h.set_region_of_interest(lo, size)
        assert np.array_equal(h.download_volume(), crop(vol, lo, size))
        h.count(_count_params(iso))
        bits = h.bitmask()
        h2 = P.capi.Handle(0)
        h2.set_volume(crop(vol, lo, size))
        h2.count(_count_params(iso))
        assert np.array_equal(bits, h2.bitmask()), f"bitmask of {lo}+{size}"
        h2.close()
    h.clear_region_of_interest()
    same_bytes(_gpu_mesh(h, p), none, "after clear")
    h.close()


@gpu
def test_region_of_interest_in_the_async_pipeline():
    P = pkg()
    vol, iso = smooth_volume((20, 24, 33), np.float32, seed=2)
    h = P.capi.Handle(0)
    h.set_volume(vol)
    for lo, size in boxes(vol.shape)[::-1]:
        p = _count_params(iso, generate_triangles=1, project_vertices=1, save_pixel_as_cell_data=1)
        h.set_region_of_interest(lo, size)
        h.count_async(p)
        h.emit_async(4)
        h.finish()
        a = h.fetch(want_cell_data=True)
        h2 = P.capi.Handle(0)
        h2.set_volume(crop(vol, lo, size))
        h2.set_region_index(lo)
        same_bytes(a, _gpu_mesh(h2, p), f"async box {lo}+{size}")
        h2.close()
    h.close()


@gpu
@pytest.mark.parametrize("fixture,iso", [("neghip", 55), ("fuel", 15)])
def test_region_of_interest_against_the_oracle(fixture, iso):
    O, P = oracle(), pkg()
    from util import read_fixture
    vol = read_fixture(fixture).data
    h = P.capi.Handle(0)
    for lo, size in boxes(vol.shape):
        for tri, proj in ((False, False), (True, True)):
            ref = O.cuberille(crop(vol, lo, size), iso, triangles=tri, project=proj, mode=O.CLOSED_FORM, region_index=lo)
            h.set_volume(vol)
            h.set_region_of_interest(lo, size)
            got = _gpu_mesh(h, _count_params(iso, generate_triangles=int(tri), project_vertices=int(proj)))
            assert_same_mesh(got, ref, f"{fixture} box {lo}+{size} tri={tri} proj={proj}")
    h.close()


@gpu
def test_region_of_interest_refusals():
    P = pkg()
    h = P.capi.Handle(0)

    def refused(code, text, call, *args):
        with pytest.raises(P.capi.CuberilleError) as e:
            call(*args)
        assert e.value.code == code and text in str(e.value), str(e.value)

    refused(1, "before cub_set_volume", h.set_region_of_interest, (0, 0, 0), (1, 1, 1))
    vol = np.zeros((6, 5, 4), np.uint8)
    h.set_volume(vol)
    for lo, size in [((0, 0, 0), (0, 1, 1)), ((0, 0, 0), (5, 5, 6)), ((4, 0, 0), (1, 1, 1)), ((1, 1, 1), (4, 4, 4)),
                     ((0, 0, 2**63), (1, 1, 1))]:
        refused(1, "region of interest", h.set_region_of_interest, lo, size)
    h.set_slab(6, 0, 0, 3)
    refused(5, "z-slab", h.set_region_of_interest, (0, 0, 0), (4, 5, 6))
    h.set_volume(vol)   # clears the slab
    h.set_region_of_interest((0, 0, 0), (4, 5, 6))
    refused(5, "region of interest", h.set_slab, 6, 0, 0, 3)
    h.set_volume(vol)   # clears the box
    assert h.download_volume().shape == vol.shape
    h.generate(P.capi.GEN_GYROID, (8, 8, 4), (8, 8, 12), z_offset=4)
    refused(5, "z-slab", h.set_region_of_interest, (0, 0, 0), (8, 8, 4))
    h.close()


@gpu
def test_region_index_and_the_box_add():
    P = pkg()
    vol, iso = smooth_volume((12, 13, 14), np.float32, seed=6)
    h = P.capi.Handle(0)
    h.set_volume(vol)
    h.set_region_of_interest((2, 3, 4), (8, 7, 6))
    h.set_region_index((10, 20, 30))       # after the box: still the index of the whole buffer
    a = _gpu_mesh(h, _count_params(iso))
    h.set_volume(vol)
    h.set_region_index((10, 20, 30))
    h.set_region_of_interest((2, 3, 4), (8, 7, 6))
    same_bytes(a, _gpu_mesh(h, _count_params(iso)), "region index before / after the box")
    h.close()


# ---- cub_run_labels --------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dtype", [np.uint8, np.uint16, np.uint32], ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize("fixture", ["neghip", "fuel"])
def test_run_labels_against_the_oracle(fixture, dtype):
    O, P = oracle(), pkg()
    vol = label_map(fixture, dtype)
    labels = [2, 0, 3, 1]
    h = P.capi.Handle(0)
    h.set_volume(vol)
    for mode, m in ORACLE_MODES.items():
        m = dict(m)
        id_bytes = m.pop("id_bytes", 4)
        cd = m.get("cell_data", False)
        p = _count_params(0, generate_triangles=int(m["triangles"]), save_pixel_as_cell_data=int(cd),
                          image_border_faces=int(m.get("border_faces", False)))
        po, co = h.run_labels(p, labels, id_bytes)
        mesh = h.fetch(want_cell_data=cd)
        assert mesh[0].shape[0] == po[-1] and mesh[1].shape[0] == co[-1]
        for i, k in enumerate(labels):
            ref = R.cuberille_range(vol, k, k, project=False, mode=O.CLOSED_FORM, **m)
            assert_same_mesh(part(mesh, po, co, i), ref, f"{fixture} {np.dtype(dtype).name} label {k} {mode}")
            if cd:
                assert (mesh[2][co[i]:co[i + 1]] == k).all()
    h.close()


RUN_MODES = {
    "quads": (dict(), {}),
    "triangles_u64_cell_data": (dict(generate_triangles=1, save_pixel_as_cell_data=1), dict(id_bytes=8)),
    "raster": (dict(vertex_order=1), {}),
    "border_faces": (dict(image_border_faces=1, generate_triangles=1), {}),
    "oriented": (dict(generate_triangles=1, save_pixel_as_cell_data=1), dict(direction=DIRECTION)),
}


@gpu
@pytest.mark.parametrize("mode", sorted(RUN_MODES))
def test_run_labels_equals_the_whole_volume_range_runs(mode):
    """256^3 uint16 with 50 blobs and one label across the whole x/y extent: every part equals inside range [k, k] +
    count + id base + emit on the whole volume, byte for byte"""
    P = pkg()
    p_kw, kw = RUN_MODES[mode]
    id_bytes, direction = kw.get("id_bytes", 4), kw.get("direction")
    vol = blob_labels((256, 256, 256), 50, np.uint16, seed=11, full_xy_label=51)
    labels = list(range(51, -1, -1)) + [60000]   # descending, the background, an absent label
    p = _count_params(0, **p_kw)
    cd = bool(p.save_pixel_as_cell_data)
    h = P.capi.Handle(0)
    h.set_volume(vol, GEO["spacing"], GEO["origin"], direction)
    h.set_region_index((3, -2, 7))
    po, co = h.run_labels(p, labels, id_bytes)
    got = h.fetch(want_cell_data=cd)
    assert po[-2] == po[-1] and co[-2] == co[-1]   # the absent label has an empty part
    ref = P.capi.Handle(0)
    ref.set_volume(vol, GEO["spacing"], GEO["origin"], direction)
    ref.set_region_index((3, -2, 7))
    for i, k in enumerate(labels[:-1]):
        ref.set_inside_range(k, k)
        ref.count(p)
        ref.set_id_base(int(po[i]), int(co[i]))
        ref.emit(id_bytes)
        want = ref.fetch(want_cell_data=cd)
        pts, cells, cdata = got
        a = (pts[po[i]:po[i + 1]], cells[co[i]:co[i + 1]], None if cdata is None else cdata[co[i]:co[i + 1]])
        same_bytes(a, want, f"{mode} label {k}")
    ref.close()
    h.close()


@gpu
def test_run_labels_leaves_the_handle_as_it_was():
    """the inside-range setting is kept, and later iso- and range-mode runs equal those of a fresh handle"""
    P = pkg()
    vol = blob_labels((30, 31, 45), 8, np.int16, seed=9)
    p = _count_params(2)
    fresh = P.capi.Handle(0)
    fresh.set_volume(vol)
    iso = _gpu_mesh(fresh, p)
    fresh.set_inside_range(3, 5)
    rng = _gpu_mesh(fresh, p)
    fresh.close()
    h = P.capi.Handle(0)
    h.set_volume(vol)
    h.run_labels(p, [1, 2, 8])
    same_bytes(_gpu_mesh(h, p), iso, "iso mode after run_labels")
    h.set_inside_range(3, 5)
    h.run_labels(_count_params(0, generate_triangles=1), [4, 7])
    same_bytes(_gpu_mesh(h, p), rng, "range mode after run_labels")
    h.close()


@gpu
def test_run_labels_refusals():
    P = pkg()
    h = P.capi.Handle(0)
    p = _count_params(0)

    def refused(code, text, *args):
        with pytest.raises(P.capi.CuberilleError) as e:
            h.run_labels(*args)
        assert e.value.code == code and text in str(e.value), str(e.value)

    refused(1, "before cub_set_volume", p, [1])
    for dt in (np.float32, np.float64):
        h.set_volume(np.zeros((3, 3, 3), dt))
        refused(5, "integer", p, [1])
    vol = blob_labels((10, 11, 12), 4, np.uint8, seed=1)
    h.set_volume(vol)
    refused(1, "twice", p, [1, 2, 1])
    refused(1, "not representable", p, [1, 256])
    refused(1, "not representable", p, [0.5])
    refused(1, "not representable", p, [-1])
    refused(1, "project_vertices", _count_params(0, project_vertices=1), [1])
    h.set_region_of_interest((0, 0, 0), (12, 11, 5))
    refused(1, "region of interest", p, [1])
    h.set_volume(vol)
    h.set_slab(10, 0, 0, 5)
    refused(1, "z-slab", p, [1])
    h.set_volume(vol)
    po, co = h.run_labels(p, [])
    assert po.tolist() == [0] and co.tolist() == [0]
    h.close()


@gpu
def test_run_labels_names_the_label_with_an_empty_interior_slice():
    P = pkg()
    vol = np.zeros((9, 5, 5), np.uint8)
    vol[2, 2, 2] = vol[4, 2, 2] = 3
    vol[3, 2, 2] = 1
    h = P.capi.Handle(0)
    h.set_volume(vol)
    h.run_labels(_count_params(0), [1, 3])
    w = h.last_warning()
    assert "empty voxel slice" in w and "(label 3)" in w
    h.run_labels(_count_params(0), [1])
    assert h.last_warning() == ""
    h.close()


# ---- filter mirror and C++ adapter --------------------------------------------------------------------------------------
@gpu
def test_filter_mirror_label_values():
    O, P = oracle(), pkg()
    vol = label_map("fuel", np.uint8)
    f = P.CuberilleImageToMeshFilter.New()
    f.SetInput(P.Image(vol, (1.0, 1.0, 1.0), (0.0, 0.0, 0.0)))
    f.SetLabelValues([3, 1])
    assert f.GetLabelValues() == [3, 1]
    with pytest.raises(RuntimeError, match="ProjectVerticesToIsoSurface"):
        f.Update()
    f.ProjectVerticesToIsoSurfaceOff()
    f.SetLabelValue(2)
    with pytest.raises(RuntimeError, match="inside range"):
        f.Update()
    f.InsideRangeOff()
    f.SavePixelAsCellDataOn()
    f.Update()
    out = f.GetOutput()
    assert out.label_point_offsets.tolist()[0] == 0 and out.label_cell_offsets[-1] == out.GetNumberOfCells()
    for i, k in enumerate([3, 1]):
        ref = R.cuberille_range(vol, k, k, triangles=True, project=False, cell_data=True, mode=O.CLOSED_FORM)
        assert_same_mesh(part((out.points, out.cells, out.cell_data), out.label_point_offsets, out.label_cell_offsets, i),
                         ref, f"filter label {k}")
    f.SetLabelValues(None)
    assert f.GetLabelValues() is None
    f.SetInput(P.Image(vol.astype(np.float32), (1.0, 1.0, 1.0), (0.0, 0.0, 0.0)))
    f.SetLabelValues([1])
    with pytest.raises(RuntimeError, match="integer"):
        f.Update()


def build_labels_driver(out_dir):
    """tests/cpp/labels_test01.cxx against the ITK stand-in and the library (the flags of tests/cpp/Makefile)"""
    pkg().build()
    exe = os.path.join(str(out_dir), "labels_test01")
    lib = os.path.dirname(pkg().capi.lib_path())
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-Wall", "-Wextra", "-Wno-unused-parameter", "-Wno-unused-local-typedefs",
                           "-I", os.path.join(ROOT, "include"), "-I", os.path.join(ROOT, "tests", "itk_shim"),
                           os.path.join(ROOT, "tests", "cpp", "labels_test01.cxx"), "-o", exe,
                           "-L", lib, "-lcuberille_cuda", "-Wl,-rpath," + lib])
    return exe


def test_adapter_label_setters_for_every_pixel_type(tmp_path):
    """compile + run without a device: SetLabelValues / ClearLabelValues and the getters"""
    exe = build_labels_driver(tmp_path)
    r = subprocess.run([exe, "Instantiate"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr


@gpu
def test_cpp_filter_labels_test(tmp_path):
    """labels_test01 LabelsTest01: each part of the label run equals the SetLabelValue(k) run of the same filter"""
    P = pkg()
    vol = label_map("neghip", np.uint8)
    path = str(tmp_path / "labels.mha")
    P.mha.write_mha(path, P.Image(vol, (1.0, 1.0, 1.0), (0.0, 0.0, 0.0)), compress=False)
    exe = build_labels_driver(tmp_path)
    r = subprocess.run([exe, "LabelsTest01", path, "3", "0", "2", "7"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "Mesh of 4 labels" in r.stdout and "LabelValues: 3 0 2 7" in r.stdout
