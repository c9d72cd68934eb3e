"""Inside-range mode (cub_set_inside_range): a voxel is inside when !(v < lower) && !(upper < v) in the pixel type.

Classification through every K1 route (packed, fused, full-row, ragged, the padded lattice of image_border_faces and
borrowed device pointers at every pixel-aligned offset) is compared with numpy over the full value range of each pixel
type.  A range [iso, type maximum or +inf] must reproduce iso mode bit for bit, and a range mesh must equal the iso-1 mesh
of the binarised volume.  Label maps made from the shipped fixtures are compared with the CPU oracle in every emit
mode, through the asynchronous pipeline, streamed z-slabs and the C++ filter.

The tests marked gpu need a CUDA device; the others check the oracle's range mode and run anywhere."""
import math
import os
import subprocess

import numpy as np
import pytest

import range_oracle as R
from test_gpu_pixel_edges import (DTYPES, DT_IDS, ROUTES, _count_params, _gpu_mesh, _handle, _int_specials,
                                  _special_floats, assert_same_mesh, pool_volume, route_shape, unpack_bitmask)
from util import ROOT, assert_mesh_equal, assert_mesh_equal_up_to_vertex_order, oracle, pkg, read_fixture, smooth_volume

gpu = pytest.mark.gpu


# ---- bounds --------------------------------------------------------------------------------------------------------------
def type_max(dt):
    dt = np.dtype(dt)
    return math.inf if dt.kind == "f" else float(np.iinfo(dt).max)


def range_bounds(dt, seed=13):
    """(lower, upper) pairs with lower <= upper.  8-bit: every lower with upper in {lower, lower + 1, max, 8 seeded},
    and every upper with lower in {min, upper - 1}.  Wider integers: every pair of the edge values (0, +-1, the sign and
    top-bit edges, the extremes, around 2^24 and 2^31 for 32 bits) plus 32 seeded pairs.  Floats: every pair of the
    special values (infinities, both zeros, subnormals, extremes)."""
    dt = np.dtype(dt)
    rng = np.random.default_rng(seed)
    if dt.kind == "f":
        vals = _special_floats(dt)
        return sorted({(a, b) for a in vals for b in vals if a <= b})
    info = np.iinfo(dt)
    pairs = set()
    if info.bits == 8:
        for v in range(info.min, info.max + 1):
            for u in {v, min(v + 1, info.max), info.max} | set(int(x) for x in rng.integers(v, info.max, 8, endpoint=True)):
                pairs.add((v, u))
            for lo in {info.min, max(v - 1, info.min)}:
                pairs.add((lo, v))
    else:
        edges = _int_specials(dt)
        pairs |= {(a, b) for a in edges for b in edges if a <= b}
        for _ in range(32):
            a, b = sorted(int(x) for x in rng.integers(info.min, info.max, 2, endpoint=True))
            pairs.add((a, b))
    return sorted((float(a), float(b)) for a, b in pairs)


reference_inside_range = R.inside_range   # `~(vol < lo) & ~(hi < vol)` evaluated by numpy in the pixel type


def check_range_bitmasks(h, vol, bounds, fused, what):
    for lo, hi in bounds:
        h.set_inside_range(lo, hi)
        h.count(_count_params(0))
        assert h.count_was_fused() == fused, f"{what}: fused={h.count_was_fused()}"
        got = unpack_bitmask(h.bitmask(), vol.shape[2])
        bad = np.argwhere(got != reference_inside_range(vol, lo, hi))
        if bad.size:
            z, y, x = bad[0]
            raise AssertionError(f"{what} [{lo!r}, {hi!r}]: {len(bad)} voxels differ, first (x={x}, y={y}, z={z}) = "
                                 f"{vol[z, y, x]!r} classified {int(got[z, y, x])}")


def _subset(seq, n):
    return seq if len(seq) <= n else seq[::len(seq) // n]


# ---- every route x dtype -------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dtype,route", [(d, r) for d in DTYPES for r in sorted(ROUTES) if np.dtype(d).itemsize in ROUTES[r][1]],
                         ids=lambda v: v if isinstance(v, str) else np.dtype(v).name)
def test_range_classification_over_the_full_value_range(dtype, route):
    env, xs, fused = ROUTES[route]
    vol = pool_volume(dtype, route_shape(dtype, xs[np.dtype(dtype).itemsize]), seed=11)
    h = _handle(**env)
    h.set_volume(vol)
    check_range_bitmasks(h, vol, range_bounds(dtype), fused, f"{np.dtype(dtype).name} {route} {vol.shape}")
    h.close()


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_range_on_the_padded_lattice(dtype):
    """image_border_faces classifies into the padded lattice (k_classify_padded): meshes against the oracle"""
    O, P = oracle(), pkg()
    vol = pool_volume(dtype, route_shape(dtype, ROUTES["fused"][1][np.dtype(dtype).itemsize]), seed=5)
    h = P.capi.Handle(0)
    h.set_volume(vol)
    for lo, hi in _subset(range_bounds(dtype), 48):
        h.set_inside_range(lo, hi)
        ref = R.cuberille_range(vol, lo, hi, triangles=False, project=False, mode=O.CLOSED_FORM, border_faces=True)
        assert_same_mesh(_gpu_mesh(h, _count_params(0, image_border_faces=1)), ref,
                         f"{np.dtype(dtype).name} border faces [{lo!r}, {hi!r}]")
    h.close()


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_range_classification_of_borrowed_pointers_at_every_alignment(dtype):
    """a device volume at an offset that is a multiple of the pixel size but not of 16 (or 4): the fused and packed
    kernels must not run, the others must classify it as they do an aligned one"""
    import torch
    P = pkg()
    size = np.dtype(dtype).itemsize
    offsets = sorted({o for o in (size, 4, 8, 12, 16, 24) if o % size == 0})
    xs = sorted({ROUTES["fused"][1][size]} | ({ROUTES["packed"][1][size]} if size <= 2 else set()))
    bounds = _subset(range_bounds(dtype), 48)
    h = P.capi.Handle(0)
    for nx in xs:
        vol = pool_volume(dtype, route_shape(dtype, nx), seed=nx)
        raw = torch.from_numpy(vol.reshape(-1).view(np.uint8).copy())
        buf = torch.zeros(raw.numel() + 64, dtype=torch.uint8, device="cuda")
        for off in offsets:
            buf[off:off + raw.numel()].copy_(raw)
            torch.cuda.synchronize()  # (the handle's stream does not wait for torch's)
            h.set_volume_ptr(buf.data_ptr() + off, dtype, vol.shape[::-1], P.capi.MEM_DEVICE)
            h.set_inside_range(*bounds[0])
            h.count(_count_params(0))
            if off % 16:
                assert not h.count_was_fused(), f"fused kernel on a buffer at offset {off}"
            check_range_bitmasks(h, vol, bounds, h.count_was_fused(), f"{np.dtype(dtype).name} nx={nx} offset {off}")
    h.close()
    del buf


# ---- identities ------------------------------------------------------------------------------------------------------------
EMIT_MODES = {
    "quads": dict(),
    "triangles": dict(generate_triangles=1),
    "quads_u64": dict(id_bytes=8),
    "cell_data": dict(generate_triangles=1, save_pixel_as_cell_data=1),
    "raster": dict(vertex_order=1, save_pixel_as_cell_data=1),
    "oriented": dict(generate_triangles=1, direction=(0.0, 1.0, 0.0, 0.0, 0.0, 1.0, 1.0, 0.0, 0.0)),
    "border_faces": dict(image_border_faces=1),
}


def _emit(h, vol, mode, lo_hi=None, iso=0.0):
    m = dict(EMIT_MODES[mode])
    id_bytes = m.pop("id_bytes", 4)
    direction = m.pop("direction", None)
    h.set_volume(vol, (1.0, 1.0, 1.0), (0.0, 0.0, 0.0), direction)
    if lo_hi is not None:
        h.set_inside_range(*lo_hi)
    return _gpu_mesh(h, _count_params(iso, **m), id_bytes)


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_range_up_to_the_type_maximum_is_iso_mode(dtype):
    """[iso, max] (or [iso, +inf]) gives the iso-mode bitmask, and a byte-identical mesh in every emit mode"""
    P = pkg()
    dt = np.dtype(dtype)
    size = dt.itemsize
    h = P.capi.Handle(0)
    for nx in sorted({ROUTES["fused"][1][size]} | ({ROUTES["packed"][1][size]} if size <= 2 else set())):
        vol = pool_volume(dtype, route_shape(dtype, nx), seed=21 + nx)
        isos = [lo for lo, _ in _subset(range_bounds(dtype), 24)]
        for iso in isos:
            h.set_volume(vol)
            h.count(_count_params(iso))
            want = h.bitmask()
            h.set_inside_range(iso, type_max(dt))
            h.count(_count_params(iso))
            assert np.array_equal(h.bitmask(), want), f"{dt.name} nx={nx} iso={iso!r}: bitmask"
        for iso in isos[::6]:
            for mode in EMIT_MODES:
                a = _emit(h, vol, mode, iso=iso)
                b = _emit(h, vol, mode, (iso, type_max(dt)))
                for x, y, what in zip(a, b, ("points", "cells", "cell data")):
                    assert (x is None) == (y is None)
                    if x is not None:
                        assert x.dtype == y.dtype and np.array_equal(x.view(np.uint8), y.view(np.uint8)), \
                            f"{dt.name} iso={iso!r} {mode}: {what} differ"
    h.close()


@gpu
@pytest.mark.parametrize("dtype", [np.uint8, np.int16, np.uint32, np.float32, np.float64], ids=lambda d: np.dtype(d).name)
def test_range_mesh_is_the_mesh_of_the_binarised_volume(dtype):
    """what a user gets today by binarising first: the iso-1 mesh of inside(vol) as uint8, points and cells bit for bit"""
    P = pkg()
    vol = pool_volume(dtype, route_shape(dtype, 40), seed=3)
    h = P.capi.Handle(0)
    for lo, hi in _subset([b for b in range_bounds(dtype) if b[0] != b[1]], 12) + [range_bounds(dtype)[len(range_bounds(dtype)) // 2]]:
        binary = np.ascontiguousarray(reference_inside_range(vol, lo, hi).astype(np.uint8))
        for mode in ("quads", "triangles", "raster", "oriented", "border_faces"):
            a = _emit(h, vol, mode, (lo, hi))
            b = _emit(h, binary, mode, iso=1.0)
            assert np.array_equal(a[0].view(np.uint32), b[0].view(np.uint32)), f"[{lo!r}, {hi!r}] {mode}: points"
            assert np.array_equal(a[1], b[1]), f"[{lo!r}, {hi!r}] {mode}: cells"
    h.close()


# ---- label maps from the fixtures against the oracle -------------------------------------------------------------------
def label_map(name, dtype):
    """the fixture cut into 4 labels 0..3: 0 below the first quartile of its non-zero voxels, 1..3 from there up"""
    data = read_fixture(name).data
    edges = np.quantile(data[data > 0], [0.25, 0.5, 0.75])
    return np.ascontiguousarray(np.digitize(data, edges).astype(dtype))


LABEL_RANGES = [(1, 1), (2, 2), (3, 3), (1, 3), (0, 1)]
ORACLE_MODES = {
    "quads": dict(triangles=False),
    "triangles": dict(triangles=True),
    "quads_u64_cell_data": dict(triangles=False, cell_data=True, id_bytes=8),
    "triangles_cell_data": dict(triangles=True, cell_data=True),
    "border_faces": dict(triangles=False, border_faces=True),
}


@gpu
@pytest.mark.parametrize("dtype", [np.uint8, np.uint16, np.uint32], ids=lambda d: np.dtype(d).name)
@pytest.mark.parametrize("fixture", ["neghip", "fuel"])
def test_label_maps_against_the_oracle(fixture, dtype):
    O, P = oracle(), pkg()
    vol = label_map(fixture, dtype)
    h = P.capi.Handle(0)
    h.set_volume(vol)
    for lo, hi in LABEL_RANGES:
        for mode, m in ORACLE_MODES.items():
            m = dict(m)
            id_bytes = m.pop("id_bytes", 4)
            ref = R.cuberille_range(vol, lo, hi, project=False, mode=O.CLOSED_FORM, **m)
            assert ref.cells.shape[0] > 0
            h.set_inside_range(lo, hi)
            p = _count_params(0, generate_triangles=int(m["triangles"]), save_pixel_as_cell_data=int(m.get("cell_data", False)),
                              image_border_faces=int(m.get("border_faces", False)))
            got = _gpu_mesh(h, p, id_bytes)
            assert_same_mesh(got, ref, f"{fixture} {np.dtype(dtype).name} [{lo}, {hi}] {mode}")
            if m.get("cell_data"):
                # every cell carries the label of the voxel that generated it
                assert got[2].dtype == vol.dtype and ((got[2] >= lo) & (got[2] <= hi)).all()
    h.close()


@gpu
def test_raster_order_on_a_label_map():
    O, P = oracle(), pkg()
    vol = label_map("neghip", np.uint16)
    h = P.capi.Handle(0)
    h.set_volume(vol)
    h.set_inside_range(2, 3)
    ref = R.cuberille_range(vol, 2, 3, triangles=False, project=False, cell_data=True, mode=O.CLOSED_FORM)
    pts, cells, cd = _gpu_mesh(h, _count_params(0, vertex_order=1, save_pixel_as_cell_data=1))
    mesh = P.Mesh(pts, cells, cd)
    assert_mesh_equal_up_to_vertex_order(mesh, ref, mesh, ref, "raster label map")
    h.close()


@gpu
def test_empty_interior_slice_warning_in_range_mode():
    """label 3 on slices 2 and 4, label 1 on slice 3: for [1, 3] the slices are contiguous, for [3, 3] slice 3 is empty"""
    P = pkg()
    vol = np.zeros((9, 5, 5), np.uint8)
    vol[2, 2, 2] = vol[4, 2, 2] = 3
    vol[3, 2, 2] = 1
    h = P.capi.Handle(0)
    h.set_volume(vol)
    h.set_inside_range(1, 3)
    h.run(_count_params(0))
    assert h.last_warning() == ""
    h.set_inside_range(3, 3)
    assert h.run(_count_params(0)) == (16, 12)
    assert "empty voxel slice" in h.last_warning()
    h.close()


# ---- pipelines ---------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("mode", ["quads", "triangles", "triangles_cell_data"])
def test_async_pipeline_in_range_mode(mode):
    """cub_count_async / cub_emit_async / cub_finish in range mode: buffers sized by a small first run, a larger second
    run overflows them on the device, cub_finish redoes the emission"""
    O, P = oracle(), pkg()
    tri, cd = mode.startswith("triangles"), mode.endswith("cell_data")
    h = P.capi.Handle(0)
    for shape, seed in [((10, 12, 33), 1), ((30, 40, 70), 2), ((30, 40, 70), 3), ((12, 9, 20), 4)]:
        vol, _ = smooth_volume(shape, np.int16, seed=seed)
        lo, hi = 45, 75
        h.set_volume(vol)
        h.set_inside_range(lo, hi)
        h.count_async(_count_params(0, generate_triangles=int(tri), save_pixel_as_cell_data=int(cd)))
        h.emit_async(4)
        n_pts, n_cells = h.finish()
        ref = R.cuberille_range(vol, lo, hi, triangles=tri, project=False, cell_data=cd, mode=O.CLOSED_FORM)
        assert (n_pts, n_cells) == (ref.points.shape[0], ref.cells.shape[0])
        a, b, c = h.fetch(want_cell_data=cd)
        assert_mesh_equal(P.Mesh(a, b, c), ref, f"async range {mode} {shape}")
    h.close()


@gpu
@pytest.mark.parametrize("n_slabs", [2, 3, 5])
def test_streamed_slabs_in_range_mode(n_slabs):
    """slabs.run_streamed with inside_range equals the mesh of one handle"""
    import torch
    O, P = oracle(), pkg()
    vol = label_map("fuel", np.uint16)
    lo, hi = 1, 2
    h = P.capi.Handle(0)
    h.set_volume(vol)
    h.set_inside_range(lo, hi)
    one = _gpu_mesh(h, _count_params(0, generate_triangles=1))
    h.close()
    ref = R.cuberille_range(vol, lo, hi, triangles=True, project=False, mode=O.CLOSED_FORM)
    assert_same_mesh(one, ref, "single handle")
    vt = torch.from_numpy(vol).pin_memory()
    pts = torch.zeros((ref.points.shape[0] + 8, 3), dtype=torch.float32).pin_memory()
    cells = torch.zeros((ref.cells.shape[0] + 8, 3), dtype=torch.int32).pin_memory()
    handles = [P.capi.Handle(0) for _ in range(2)]
    n_pts, n_cells = P.slabs.run_streamed(handles, vt.data_ptr(), np.uint16, vol.shape[::-1], _count_params(0, generate_triangles=1),
                                          n_slabs, pts.data_ptr(), cells.data_ptr(), inside_range=(lo, hi))
    assert (n_pts, n_cells) == (one[0].shape[0], one[1].shape[0])
    assert np.array_equal(pts.numpy()[:n_pts].view(np.uint32), one[0].view(np.uint32))
    assert np.array_equal(cells.numpy()[:n_cells].view(np.uint32), one[1])
    for h in handles:
        h.close()


def build_range_driver(out_dir):
    """tests/cpp/range_test01.cxx against the ITK stand-in and the library (the flags of tests/cpp/Makefile)"""
    pkg().build()
    exe = os.path.join(str(out_dir), "range_test01")
    lib = os.path.dirname(pkg().capi.lib_path())
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-Wall", "-Wextra", "-Wno-unused-parameter", "-Wno-unused-local-typedefs",
                           "-I", os.path.join(ROOT, "include"), "-I", os.path.join(ROOT, "tests", "itk_shim"),
                           os.path.join(ROOT, "tests", "cpp", "range_test01.cxx"), "-o", exe,
                           "-L", lib, "-lcuberille_cuda", "-Wl,-rpath," + lib])
    return exe


def test_adapter_range_setters_for_every_pixel_type(tmp_path):
    """compile + run without a device: SetInsideRange / SetLabelValue / InsideRangeOff and the getters"""
    exe = build_range_driver(tmp_path)
    assert subprocess.run([exe, "Instantiate"]).returncode == 0


@gpu
@pytest.mark.parametrize("lo,hi,tri", [(2, 2, 1), (1, 3, 0)])
def test_cpp_filter_range_test(lo, hi, tri, tmp_path):
    """range_test01 RangeTest01 on a label map of neghip: refused with the default projection, then the reference
    counts"""
    P = pkg()
    vol = label_map("neghip", np.uint8)
    path = str(tmp_path / "labels.mha")
    P.mha.write_mha(path, P.Image(vol, (1.0, 1.0, 1.0), (0.0, 0.0, 0.0)), compress=False)
    ref = R.cuberille_range(vol, lo, hi, triangles=bool(tri), mode=R.CLOSED_FORM)
    exe = build_range_driver(tmp_path)
    r = subprocess.run([exe, "RangeTest01", path, str(lo), str(hi), str(ref.points.shape[0]), str(ref.cells.shape[0]), str(tri)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert f"Mesh has {ref.points.shape[0]} vertices and {ref.cells.shape[0]} cells" in r.stdout
    assert f"InsideRange: 1 [{lo}, {hi}]" in r.stdout


@gpu
def test_filter_mirror_label_value():
    O, P = oracle(), pkg()
    vol = label_map("fuel", np.uint8)
    f = P.CuberilleImageToMeshFilter.New()
    f.SetInput(P.Image(vol, (1.0, 1.0, 1.0), (0.0, 0.0, 0.0)))
    f.SetLabelValue(2)
    assert f.GetInsideRange() == (2, 2) and f.GetInsideRangeLower() == 2 and f.GetInsideRangeUpper() == 2
    with pytest.raises(P.capi.CuberilleError) as e:
        f.Update()   # projection is on by default
    assert "project_vertices off" in str(e.value)
    f.ProjectVerticesToIsoSurfaceOff()
    f.GenerateTriangleFacesOff()
    f.SavePixelAsCellDataOn()
    f.Update()
    ref = R.cuberille_range(vol, 2, 2, triangles=False, project=False, cell_data=True, mode=O.CLOSED_FORM)
    assert_mesh_equal(f.GetOutput(), ref, "filter label 2")
    f.InsideRangeOff()
    f.Update()
    ref = O.cuberille(vol, 1, triangles=False, project=False, cell_data=True, mode=O.CLOSED_FORM)
    assert_mesh_equal(f.GetOutput(), ref, "filter iso mode again")


# ---- refusals ------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_range_refusals(dtype):
    P = pkg()
    dt = np.dtype(dtype)
    h = P.capi.Handle(0)
    vol = pool_volume(dtype, route_shape(dtype, 36), seed=2)

    def refused(lo, hi, text):
        with pytest.raises(P.capi.CuberilleError) as e:
            h.set_inside_range(lo, hi)
        assert e.value.code == 1 and text in str(e.value), (lo, hi, str(e.value))

    with pytest.raises(P.capi.CuberilleError):
        h.set_inside_range(0, 1)   # no volume yet
    h.set_volume(vol)
    if dt.kind in "iu":
        info = np.iinfo(dt)
        for lo, hi in [(0.5, 1.0), (0.0, 1.5), (float(info.min) - 1.0, 0.0), (0.0, float(info.max) + 1.0), (-math.inf, 0.0),
                       (0.0, math.inf), (1e300, 1e300)]:
            refused(lo, hi, "not representable")
        h.set_inside_range(float(info.min), float(info.max))
    else:
        if dt == np.float32:
            refused(0.1, 1.0, "not representable")
            refused(0.0, 1e39, "not representable")
        h.set_inside_range(-math.inf, math.inf)
        h.set_inside_range(0.0, -0.0)
    refused(math.nan, 1.0, "NaN")
    refused(0.0, math.nan, "NaN")
    refused(2.0, 1.0, "lower exceeds upper")
    # projection needs an iso-surface: refused by cub_count, cub_count_async and cub_debug_project_points
    h.set_inside_range(0.0, 1.0)
    for call in (h.count, h.count_async):
        with pytest.raises(P.capi.CuberilleError) as e:
            call(_count_params(1, project_vertices=1))
        assert e.value.code == 1 and "project_vertices off" in str(e.value)
    with pytest.raises(P.capi.CuberilleError) as e:
        h.project_points(_count_params(1, project_vertices=1), np.zeros((4, 3), np.float32))
    assert e.value.code == 1 and "iso-surface" in str(e.value)
    # the iso value is not validated in range mode
    h.count(_count_params(math.nan))
    assert np.array_equal(unpack_bitmask(h.bitmask(), vol.shape[2]), reference_inside_range(vol, 0.0, 1.0))
    # enable = 0 returns to iso mode, and so does cub_set_volume
    h.clear_inside_range()
    h.count(_count_params(1))
    iso_bits = h.bitmask()
    with np.errstate(invalid="ignore"):
        assert np.array_equal(unpack_bitmask(iso_bits, vol.shape[2]), ~(vol < np.array(1).astype(dt)))
    h.set_inside_range(0.0, 1.0)
    h.set_volume(vol)
    h.count(_count_params(1))
    assert np.array_equal(h.bitmask(), iso_bits)
    h.close()


# ---- the range reference (no device) ----------------------------------------------------------------------------------------
def test_range_reference_bitmask_layout_matches_the_oracle():
    """classify_range packs like oracle_py.classify: [lo, max] is the oracle's iso-lo bitmask, NaN pixels are inside"""
    O = oracle()
    for dtype in (np.uint8, np.int16, np.float32):
        vol = pool_volume(dtype, route_shape(dtype, 70), seed=1)
        for lo, _ in _subset(range_bounds(dtype), 24):
            assert np.array_equal(R.classify_range(vol, lo, type_max(dtype)), O.classify(vol, lo)), (dtype, lo)
    vol = pool_volume(np.float32, (6, 7, 70), seed=1)
    assert unpack_bitmask(R.classify_range(vol, 0.0, 0.0), vol.shape[2])[np.isnan(vol)].all()


@pytest.mark.parametrize("fixture,iso", [("neghip", 55), ("fuel", 15), ("silicium", 85)])
@pytest.mark.parametrize("mode", ["literal", "closed_form"])
def test_range_reference_up_to_the_maximum_is_the_iso_oracle(fixture, iso, mode):
    """the index-volume construction of range_oracle reproduces the oracle's iso mesh, cell data included"""
    O = oracle()
    vol = read_fixture(fixture).data
    m = O.LITERAL if mode == "literal" else O.CLOSED_FORM
    for kw in (dict(triangles=False), dict(triangles=True, cell_data=True), dict(triangles=False, border_faces=True)):
        a = O.cuberille(vol, iso, project=False, mode=m, **kw)
        b = R.cuberille_range(vol, iso, 255, mode=m, **kw)
        assert_mesh_equal(b, a, f"{fixture} {mode} {kw}")
    f = np.ascontiguousarray(vol.astype(np.float32))
    assert_mesh_equal(R.cuberille_range(f, iso, math.inf, mode=m, cell_data=True),
                      O.cuberille(f, iso, project=False, mode=m, cell_data=True), f"{fixture} float32")


def test_range_reference_cell_data_is_the_generating_voxel():
    vol = label_map("neghip", np.uint16)
    for lo, hi in LABEL_RANGES:
        ref = R.cuberille_range(vol, lo, hi, triangles=False, cell_data=True)
        assert ref.cell_data.dtype == vol.dtype and ((ref.cell_data >= lo) & (ref.cell_data <= hi)).all()
