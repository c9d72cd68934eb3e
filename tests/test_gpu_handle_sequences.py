"""Long-lived handles through every mode, and z-slabs cut at the exact projection halo, against the CPU oracle.

Callers keep one handle for many runs, and what a run computes must not depend on the runs before it: the scratch is
grow-only with conditional clears, the result buffers are swapped by cub_run_labels, a region of interest moves the
volume pointer, the asynchronous path emits into buffers an earlier run sized.  make_plan turns (seed, n_steps) into a
list of fully described steps (volume, geometry, mode, emission, call path) drawn so that layouts coincide and change
between consecutive runs; every step is compared with the oracle, independently of the handle.  A failing step is
rerun on a fresh handle, which tells a state bug from a kernel bug.

The second half cuts tall volumes into z-slabs whose buffers hold exactly the halo cub_projection_halo_oriented
reports, over a grid of projection parameters and image geometries: the slabs must give the whole-image mesh bit for
bit, and one slice less on either side must be refused.

The tests marked gpu need a CUDA device; the others run anywhere."""
import ctypes
import itertools
import math
from types import SimpleNamespace

import numpy as np
import pytest

import range_oracle as R
from test_gpu_inside_range import label_map
from test_gpu_labels import blob_labels, crop, part
from test_gpu_pixel_edges import _count_params, _gpu_mesh, assert_same_mesh, set_route_volume
from util import (assert_mesh_equal, assert_mesh_equal_up_to_vertex_order, oracle, pkg, random_volume,
                  smooth_volume)

gpu = pytest.mark.gpu

DTYPES = [np.uint8, np.int8, np.uint16, np.int16, np.uint32, np.int32, np.float32, np.float64]
INT_TYPES = DTYPES[:6]
_C30, _S30 = math.cos(math.pi / 6), math.sin(math.pi / 6)
_C40, _S40 = math.cos(0.7), math.sin(0.7)
DIRECTIONS = {  # rotations that mix z with x or y: the z row of M^-1 is not (0, 0, 1 / spacing_z)
    "rot_x_30": (1.0, 0.0, 0.0, 0.0, _C30, -_S30, 0.0, _S30, _C30),
    "rot_y_40": (_C40, 0.0, _S40, 0.0, 1.0, 0.0, -_S40, 0.0, _C40),
    "oblique": tuple(float(v) for v in np.linalg.qr(np.random.default_rng(5).normal(size=(3, 3)))[0].reshape(9)),
}
SPACINGS = [(1.0, 1.0, 1.0), (0.7, 1.1, 1.3), (1.0, 1.0, 0.5), (0.5, 1.25, 2.0)]
ORIGINS = [(0.0, 0.0, 0.0), (1.5, -2.0, 0.25), (3.0, -2.0, 7.0)]

# ---- shapes (z, y, x) that make the lattices of consecutive runs coincide and change ------------------------------------
# the K1 route each row length takes (cuberille_capi.cu: choose_count_route), with the pixel types it applies to;
# "full" needs a buffer that is not 16-byte aligned (else rows of whole tasks fuse)
ROUTE_SHAPES = {
    "packed": [((5, 6, 128), [np.uint8, np.int8]), ((5, 6, 64), [np.uint16, np.int16])],
    "fused": [((6, 7, 48), DTYPES)],
    "full": [((3, 3, 512), DTYPES)],
    "ragged": [((7, 9, 33), DTYPES), ((8, 5, 70), DTYPES)],
}
GROW, SHRINK = (14, 26, 70), (4, 5, 9)
SLAB_Z = 26   # slab steps take the drawn rows on this many slices: room for a cut with a projection halo


def k1_route(shape, dtype, border, misaligned):
    """the K1 route of a count on a (z, y, x) buffer: choose_count_route restated"""
    x, pb = shape[2], np.dtype(dtype).itemsize
    if border:
        return "padded"
    if pb <= 2 and x % (32 * 4 // pb) == 0 and not misaligned % 4:
        return "packed"
    if (x * pb) % 16 == 0 and not misaligned % 16:
        return "fused"
    if x % 512 == 0:
        return "full"
    return "ragged"


# ---- the plan -----------------------------------------------------------------------------------------------------------
MODES = ["iso", "range", "roi", "labels", "slab"]
PATHS = ["run", "count_emit", "async", "reemit"]


def _pick(rng, seq):
    return seq[int(rng.integers(len(seq)))]


def _draw_shape(rng, prev, mode):
    """(shape, dtype, border faces, move) relative to the previous step of the handle"""
    moves = ["route", "route", "grow", "shrink"]
    if prev is not None and prev["shape"] is not None:
        moves += ["same_xyz_other_type", "border_twin", "border_twin"]
    move = _pick(rng, moves)
    dtypes = INT_TYPES if mode == "labels" else DTYPES
    border = bool(rng.random() < 0.2) and mode != "slab"
    dtype = _pick(rng, dtypes)
    if move == "same_xyz_other_type":
        shape = prev["shape"]
        dtype = _pick(rng, [d for d in dtypes if np.dtype(d) != np.dtype(prev["dtype"])])
        border = prev["border"] and mode != "slab"
    elif move == "border_twin":   # (Z, Y, X) with border faces has the lattice of (Z+2, Y+2, X+2) without
        z, y, x = prev["shape"]
        if prev["border"] or mode == "slab" or min(z, y, x) < 4:
            shape, border = (z + 2, y + 2, x + 2), False
        else:
            shape, border = (z - 2, y - 2, x - 2), True
    elif move == "grow":
        shape = GROW
    elif move == "shrink":
        shape = SHRINK
    else:
        route = _pick(rng, sorted(ROUTE_SHAPES))
        shape, types = _pick(rng, ROUTE_SHAPES[route])
        types = [d for d in types if d in dtypes] or types
        dtype = _pick(rng, types if mode != "labels" else [d for d in types if d in INT_TYPES] or INT_TYPES)
    if mode == "slab":
        shape = (SLAB_Z,) + tuple(shape[1:])
    return tuple(shape), dtype, border, move


def _draw_step(rng, prev, index):
    mode = _pick(rng, MODES)
    shape, dtype, border, move = _draw_shape(rng, prev, mode)
    s = dict(index=index, mode=mode, shape=shape, dtype=np.dtype(dtype).name, border=border, move=move,
             seed=int(rng.integers(1 << 30)))
    s["field"] = "labels" if mode == "labels" else _pick(rng, ["noise", "smooth"])
    s["fill"] = float(_pick(rng, [0.1, 0.5, 0.9]))
    if mode == "labels" and rng.random() < 0.15:
        s["field"], s["shape"] = "fixture", None   # a reference fixture cut into 4 labels (label_map)
    s["spacing"] = _pick(rng, SPACINGS)
    s["origin"] = _pick(rng, ORIGINS)
    # rows of 512 voxels come as a borrowed device pointer one pixel past a 16-byte boundary, the "full" route
    # (cub_set_volume takes a direction only with a host upload through the binding)
    s["misaligned"] = s["shape"] is not None and s["shape"][2] == 512 and mode in ("iso", "range", "roi")
    s["direction"] = _pick(rng, sorted(DIRECTIONS)) if rng.random() < 0.25 and not s["misaligned"] else None
    s["region_index"] = tuple(int(v) for v in rng.integers(-5, 6, 3)) if rng.random() < 0.4 else (0, 0, 0)
    # emission
    s["triangles"] = bool(rng.random() < 0.5)
    s["cell_data"] = bool(rng.random() < 0.4)
    s["id_bytes"] = 8 if rng.random() < 0.3 else 4
    s["project"] = mode in ("iso", "roi", "slab") and s["field"] == "smooth" and rng.random() < 0.6
    # (raster order is checked up to vertex order, which sorts the unprojected points of a non-oriented image)
    s["raster"] = not s["project"] and mode != "slab" and s["direction"] is None and rng.random() < 0.25
    s["method"] = int(rng.integers(3)) if s["project"] else 0
    s["thr"] = float(_pick(rng, [0.02, 0.2]))
    s["step"] = float(_pick(rng, [-1.0, 0.3]))
    s["relax"] = float(_pick(rng, [0.5, 0.95]))
    s["max_steps"] = int(_pick(rng, [0, 3, 20]))
    s["range"] = mode in ("range", "labels") or (mode in ("roi", "slab") and not s["project"] and rng.random() < 0.4)
    s["nan"] = s["range"] and mode != "labels" and np.dtype(dtype).kind == "f" and not s["raster"] and rng.random() < 0.7
    s["path"] = "labels" if mode == "labels" else _pick(rng, PATHS if mode != "slab" else PATHS[1:])
    if mode == "roi":
        s["roi"] = _pick(rng, ["in_place", "gathered", "gathered", "cleared"])
        s["roi_twice"] = bool(rng.random() < 0.3)          # another box first: the second replaces it
        s["index_after_box"] = bool(rng.random() < 0.5)    # cub_set_region_index after the box (still the buffer's)
    if mode == "labels":
        s["n_labels"] = int(rng.integers(3, 9))
        s["before"] = _pick(rng, ["iso", "range"])          # the handle's own mode, which cub_run_labels must keep
    if mode == "slab":
        s["n_slabs"] = int(rng.integers(2, 5))
        s["slab"] = int(rng.integers(s["n_slabs"]))
    return s


def make_plan(seed, n_steps):
    """n_steps fully described runs for one handle; the same (seed, n_steps) gives the same plan everywhere"""
    rng = np.random.default_rng(seed)
    plan = []
    for i in range(n_steps):
        plan.append(_draw_step(rng, plan[-1] if plan else None, i))
    return plan


def lattice(s):
    """(X, Y, Zl) of the count lattice a step's first count runs on (None: a label map, one box per label)"""
    if s["mode"] == "labels":
        return None
    z, y, x = s["shape"]
    if s["mode"] == "roi" and s["roi"] != "cleared":
        (x, y, z) = roi_box(s)[1]
    if s["mode"] == "slab":
        z = slab_cut(s)[1] - slab_cut(s)[0]
    p = 2 if s["border"] else 0
    return (x + p, y + p, z + p)


def route_of(s):
    if s["mode"] == "labels":
        return None
    z, y, x = s["shape"]
    off = np.dtype(s["dtype"]).itemsize if s["misaligned"] else 0
    if s["mode"] == "roi" and s["roi"] != "cleared":
        (lx, ly, lz), (sx, sy, sz) = roi_box(s)
        if (lx, ly, sx, sy) == (0, 0, x, y):   # whole rows and slices: in place, the pointer moves by lz slices
            off += lz * x * y * np.dtype(s["dtype"]).itemsize
        else:
            off = 0                             # gathered into the handle's own buffer
        z, y, x = sz, sy, sx
    return k1_route((z, y, x), s["dtype"], s["border"], off)


def transitions(plan):
    """every per-step property and every transition between consecutive runs of one handle the plan contains"""
    tags = set()
    for i, s in enumerate(plan):
        tags |= {f"mode:{s['mode']}", f"path:{s['path']}", f"ids:{s['id_bytes']}"}
        tags.add("emit:triangles" if s["triangles"] else "emit:quads")
        tags |= {t for t, on in (("emit:cell_data", s["cell_data"]), ("emit:raster", s["raster"]),
                                 ("geo:direction", s["direction"]), ("geo:region_index", any(s["region_index"])),
                                 ("range:nan", s["nan"]), ("border_faces", s["border"])) if on}
        if s["project"]:
            tags.add(f"project:{s['method']}")
        if s["mode"] == "roi":
            tags.add(f"roi:{roi_kind(s)}")
        if s["mode"] == "labels":
            tags.add(f"labels:cell_data_{'on' if s['cell_data'] else 'off'}")
        if s["mode"] == "slab" and s["direction"] and s["project"]:
            tags.add("slab:oriented_projected")
        if route_of(s):
            tags.add(f"route:{route_of(s)}")
        if i == 0:
            continue
        p = plan[i - 1]
        if s["move"] == "same_xyz_other_type" and s["shape"] == p["shape"] and s["dtype"] != p["dtype"]:
            tags.add("same_xyz_other_type")
        a, b = lattice(p), lattice(s)
        if a and b and a == b and p["border"] != s["border"]:
            tags.add("border_lattice_shared")
        if route_of(p) and route_of(s) and route_of(p) != route_of(s):
            tags.add(f"route_into:{route_of(s)}")
        if i >= 2 and a and b and lattice(plan[i - 2]):
            if np.prod(a) > np.prod(lattice(plan[i - 2])) and np.prod(b) < np.prod(a):
                tags.add("shrink_after_grow")
        if s["path"] == "async" and a and b:
            tags.add("async_after_larger" if np.prod(a) > np.prod(b) else "async_after_smaller" if np.prod(a) < np.prod(b) else "async_after_same")
    return tags


REQUIRED = ({f"mode:{m}" for m in MODES} | {f"path:{p}" for p in PATHS + ["labels"]} | {"ids:4", "ids:8"}
            | {"emit:quads", "emit:triangles", "emit:cell_data", "emit:raster", "project:0", "project:1", "project:2"}
            | {"geo:direction", "geo:region_index", "range:nan", "border_faces", "slab:oriented_projected"}
            | {"roi:in_place", "roi:gathered", "roi:cleared", "labels:cell_data_on", "labels:cell_data_off"}
            | {f"route:{r}" for r in ("fused", "packed", "full", "ragged", "padded")}
            | {f"route_into:{r}" for r in ("fused", "packed", "full", "ragged", "padded")}
            | {"same_xyz_other_type", "border_lattice_shared", "shrink_after_grow", "async_after_larger",
               "async_after_smaller"})

SEEDS, N_STEPS = list(range(6)), 40


# ---- the boxes and cuts a step describes ------------------------------------------------------------------------------
def roi_box(s):
    """(lo, size) in (x, y, z) of a region-of-interest step: whole rows and slices, or any box"""
    z, y, x = s["shape"]
    rng = np.random.default_rng(s["seed"] + 1)
    lz = int(rng.integers(0, z))
    sz = int(rng.integers(1, z - lz + 1))
    if s["roi"] == "in_place":
        return (0, 0, lz), (x, y, sz)
    lx, ly = int(rng.integers(0, x)), int(rng.integers(0, y))
    return (lx, ly, lz), (int(rng.integers(1, x - lx + 1)), int(rng.integers(1, y - ly + 1)), sz)


def roi_kind(s):
    if s["roi"] == "cleared":
        return "cleared"
    (lx, ly, _), (sx, sy, _) = roi_box(s)
    z, y, x = s["shape"]
    return "in_place" if (lx, ly, sx, sy) == (0, 0, x, y) else "gathered"


def slab_cut(s):
    """(local_z0, local_z1, own_z0, own_z1) of a slab step: slab s['slab'] of s['n_slabs'] plus the halo"""
    P = pkg()
    nz = s["shape"][0]
    z0, z1 = nz * s["slab"] // s["n_slabs"], nz * (s["slab"] + 1) // s["n_slabs"]
    below, above = P.capi.projection_halo(params(s), s["spacing"], DIRECTIONS.get(s["direction"]))
    return max(0, z0 - below), min(nz, z1 + above), z0, z1


def params(s):
    p = _count_params(0, generate_triangles=int(s["triangles"]), project_vertices=int(s["project"]),
                      save_pixel_as_cell_data=int(s["cell_data"]), vertex_order=int(s["raster"]),
                      image_border_faces=int(s["border"]), projection_method=s["method"],
                      surface_distance_threshold=s["thr"], step_length=s["step"], step_relaxation=s["relax"],
                      max_steps=s["max_steps"])
    return p


# ---- volumes and references -------------------------------------------------------------------------------------------
def volume(s):
    """(volume, iso, inside range or None) of a step"""
    dt = np.dtype(s["dtype"])
    if s["field"] == "fixture":
        vol = label_map(_pick(np.random.default_rng(s["seed"]), ["neghip", "fuel"]), dt)
        return vol, 1, None
    if s["field"] == "labels":
        vol = blob_labels(s["shape"], s["n_labels"], dt, s["seed"])
        iso = 1
    elif s["field"] == "noise":
        vol, iso = random_volume(s["shape"], dt, s["seed"], fill=s["fill"])
    else:
        vol, iso = smooth_volume(s["shape"], dt, s["seed"])
    rng = np.random.default_rng(s["seed"] + 2)
    if s["nan"]:
        vol = vol.copy()
        vol[rng.random(vol.shape) < 0.1] = np.nan
    rg = None
    if s["range"] and s["mode"] != "labels":
        vals = np.unique(vol[~np.isnan(vol)] if dt.kind == "f" else vol)
        a, b = sorted(rng.choice(vals, 2))
        rg = (a.item(), b.item())
    return np.ascontiguousarray(vol), iso, rg


def oracle_kw(s, with_projection=True):
    kw = dict(mode=oracle().CLOSED_FORM, triangles=s["triangles"], spacing=s["spacing"], origin=s["origin"],
              border_faces=s["border"], direction=DIRECTIONS.get(s["direction"]))
    if with_projection:
        kw.update(project=s["project"], thr=s["thr"], step=s["step"], relax=s["relax"], max_steps=s["max_steps"],
                  method=s["method"])
    return kw


def reference(vol, iso, rg, s, region_index):
    if rg is not None:
        return R.cuberille_range(vol, *rg, cell_data=s["cell_data"], region_index=region_index,
                                 **oracle_kw(s, with_projection=False))
    return oracle().cuberille(vol, iso, cell_data=s["cell_data"], region_index=region_index, **oracle_kw(s))


def labels_of(vol, s):
    rng = np.random.default_rng(s["seed"] + 3)
    present = [int(v) for v in np.unique(vol)]
    labels = [int(v) for v in rng.permutation(present)][: max(2, len(present) - 1)]
    absent = max(present) + 1
    if absent <= np.iinfo(vol.dtype).max:
        labels.insert(int(rng.integers(len(labels) + 1)), absent)   # an empty part
    return labels


# ---- comparison -----------------------------------------------------------------------------------------------------------
def check(got, ref, s, what, shift=0):
    """one emission of a step against its reference, point ids shifted by `shift`"""
    pts, cells, cd = got
    want = np.uint64 if s["id_bytes"] == 8 else np.uint32
    assert cells.dtype == want, f"{what}: ids {cells.dtype}, want {np.dtype(want).name}"
    local = (cells.astype(np.int64) - shift).astype(np.uint64)
    if s["raster"]:
        mesh = SimpleNamespace(points=pts, cells=local, cell_data=cd)
        assert_mesh_equal_up_to_vertex_order(mesh, ref, mesh, ref, what)
    else:
        assert_same_mesh((pts, local, cd), ref, what)


def emit_and_check(h, s, p, ref, what, base=(0, 0), ref_base=0):
    """the step's call path, every emission it makes compared with ref, whose point ids start at ref_base (the
    emissions' at base[0])"""
    cd, ib = s["cell_data"], s["id_bytes"]
    path = s["path"]
    if path == "run":
        assert base == (0, 0)
        n = h.run(p, ib)
        assert n == (ref.points.shape[0], ref.cells.shape[0]), f"{what}: run returned {n}"
    elif path == "async":
        h.count_async(p)
        if base != (0, 0):
            h.set_id_base(*base)
        h.emit_async(ib)
        n = h.finish()
        assert n == (ref.points.shape[0], ref.cells.shape[0]), f"{what}: finish returned {n}"
    else:
        n_pts, n_quads = h.count(p)
        assert n_pts == ref.points.shape[0] and n_quads * (2 if s["triangles"] else 1) == ref.cells.shape[0], \
            f"{what}: count returned {(n_pts, n_quads)}"
        h.set_id_base(*base)
        if path == "reemit":   # a first emission with the other id width, then new bases on the same count
            h.emit(12 - ib)
            first = h.fetch(want_cell_data=cd)
            other = dict(s, id_bytes=12 - ib)
            check(first, ref, other, f"{what} (first emit, {12 - ib}-byte ids)", base[0] - ref_base)
            base = (base[0] + 1000, base[1] + 77)
            h.set_id_base(*base)
        h.emit(ib)
    check(h.fetch(want_cell_data=cd), ref, s, what, base[0] - ref_base)


def check_route(h, s, what):
    r = route_of(s)
    if r is not None:
        assert h.count_was_fused() == (r == "fused"), f"{what}: count_was_fused() = {h.count_was_fused()}, route {r}"


# ---- one step on a handle ------------------------------------------------------------------------------------------------
def set_volume(h, vol, s, keep):
    geo = dict(spacing=s["spacing"], origin=s["origin"])
    if s["misaligned"]:   # the buffer set_route_volume fills, again with the step's geometry
        keep["buf"] = set_route_volume(h, vol, True)
        h.set_volume_ptr(keep["buf"].data_ptr() + vol.dtype.itemsize, vol.dtype, vol.shape[::-1], pkg().capi.MEM_DEVICE,
                         **geo)
    else:
        keep["buf"] = None
        h.set_volume(vol, direction=DIRECTIONS.get(s["direction"]), **geo)


def run_step(h, s, keep):
    """execute step s on handle h and compare every result with the oracle; AssertionError on a mismatch"""
    what = f"step {s['index']} ({describe(s)})"
    vol, iso, rg = volume(s)
    p = params(s)
    p.iso_value = float(iso)
    mode, ri = s["mode"], s["region_index"]
    if mode in ("iso", "range"):
        set_volume(h, vol, s, keep)
        if any(ri):
            h.set_region_index(ri)
        if rg:
            h.set_inside_range(*rg)
        emit_and_check(h, s, p, reference(vol, iso, rg, s, ri), what)
        check_route(h, s, what)
    elif mode == "roi":
        set_volume(h, vol, s, keep)
        if not s["index_after_box"] and any(ri):
            h.set_region_index(ri)
        if rg:
            h.set_inside_range(*rg)
        lo, size = roi_box(s)
        if s["roi_twice"]:
            h.set_region_of_interest((0, 0, 0), (1, 1, 1))
        h.set_region_of_interest(lo, size)
        if s["index_after_box"] and any(ri):
            h.set_region_index(ri)
        if s["roi"] == "cleared":
            h.clear_region_of_interest()
            ref = reference(vol, iso, rg, s, ri)
        else:
            ref = reference(crop(vol, lo, size), iso, rg, s, tuple(r + l for r, l in zip(ri, lo)))
        emit_and_check(h, s, p, ref, f"{what} box {lo}+{size}")
        check_route(h, s, what)
    elif mode == "slab":
        lz0, lz1, z0, z1 = slab_cut(s)
        nz = vol.shape[0]
        h.set_volume(vol[lz0:lz1], s["spacing"], s["origin"], DIRECTIONS.get(s["direction"]))
        keep["buf"] = None
        if any(ri):
            h.set_region_index(ri)
        if rg:
            h.set_inside_range(*rg)
        h.set_slab(nz, lz0, z0, z1)
        whole = reference(vol, iso, rg, s, ri)
        pb, cb = whole.points_before_slice, whole.cells_before_slice
        sec = SimpleNamespace(points=whole.points[int(pb[z0]):int(pb[z1])], cells=whole.cells[int(cb[z0]):int(cb[z1])],
                              cell_data=None if whole.cell_data is None else whole.cell_data[int(cb[z0]):int(cb[z1])])
        emit_and_check(h, s, p, sec, f"{what} slab [{z0},{z1}) in [{lz0},{lz1})", (int(pb[z0]), int(cb[z0])),
                       int(pb[z0]))
        check_route(h, s, what)
    else:
        run_labels_step(h, s, vol, p, keep, what)


def run_labels_step(h, s, vol, p, keep, what):
    ri = s["region_index"]
    h.set_volume(vol, s["spacing"], s["origin"], DIRECTIONS.get(s["direction"]))
    keep["buf"] = None
    if any(ri):
        h.set_region_index(ri)
    # the handle's own mode before the call, which it must find again afterwards
    present = np.unique(vol)
    k0 = int(present[len(present) // 2])
    before = (k0, k0) if s["before"] == "range" else None
    if before:
        h.set_inside_range(*before)
    labels = labels_of(vol, s)
    po, co = h.run_labels(p, labels, s["id_bytes"])
    got = h.fetch(want_cell_data=s["cell_data"])
    assert got[0].shape[0] == po[-1] and got[1].shape[0] == co[-1], f"{what}: totals"
    for i, k in enumerate(labels):
        ref = R.cuberille_range(vol, k, k, cell_data=s["cell_data"], region_index=ri, **oracle_kw(s, False))
        assert (po[i + 1] - po[i], co[i + 1] - co[i]) == ref.points.shape[:1] + ref.cells.shape[:1], \
            f"{what}: label {k} part has {po[i + 1] - po[i]} points / {co[i + 1] - co[i]} cells, want " \
            f"{ref.points.shape[0]} / {ref.cells.shape[0]}"
        check(part(got, po, co, i), ref, s, f"{what} label {k}")
    # the handle is back to the whole volume in its own mode
    iso_p = _count_params(float(k0), vertex_order=int(s["raster"]), image_border_faces=int(s["border"]))
    after = _gpu_mesh(h, iso_p)
    if before:
        ref = R.cuberille_range(vol, *before, region_index=ri, **dict(oracle_kw(s, False), triangles=False))
    else:
        ref = oracle().cuberille(vol, k0, project=False, region_index=ri, **dict(oracle_kw(s, False), triangles=False))
    check(after, ref, dict(s, id_bytes=4), f"{what}: the handle's own {'range' if before else 'iso'} mode after run_labels")


def describe(s):
    bits = [s["mode"], s["dtype"], "fixture" if s["shape"] is None else "x".join(map(str, s["shape"][::-1])), s["field"],
            s["path"], "tri" if s["triangles"] else "quads", f"ids{s['id_bytes']}"]
    bits += [t for t, on in (("cell_data", s["cell_data"]), ("raster", s["raster"]), ("border", s["border"]),
                             ("nan", s["nan"]), ("misaligned", s["misaligned"])) if on]
    if s["project"]:
        bits.append(f"project(method {s['method']}, thr {s['thr']}, step {s['step']}, relax {s['relax']}, "
                    f"max_steps {s['max_steps']})")
    if s["direction"]:
        bits.append(s["direction"])
    if s["mode"] == "roi":
        bits.append(f"roi {s['roi']}{' twice' if s['roi_twice'] else ''}")
    if s["mode"] == "slab":
        bits.append(f"slab {s['slab']}/{s['n_slabs']}")
    return ", ".join(bits)


# ---- a handle that records its calls ---------------------------------------------------------------------------------------
def _short(v):
    if isinstance(v, np.ndarray):
        return f"<{v.dtype} {'x'.join(map(str, v.shape))}>"
    if isinstance(v, pkg().capi.Params):
        return "params(" + ", ".join(f"{n}={getattr(v, n)}" for n, _ in v._fields_ if n != "reserved") + ")"
    if isinstance(v, (list, tuple)) and len(v) > 6:
        return f"[{len(v)} values]"
    return repr(v)


class Recorded:
    """a capi.Handle that logs every call made on it, per step"""

    def __init__(self, h):
        self.h, self.log = h, []

    def __getattr__(self, name):
        f = getattr(self.h, name)
        if not callable(f):
            return f

        def call(*args, **kw):
            self.log[-1][1].append(f"{name}({', '.join([_short(a) for a in args] + [f'{k}={_short(v)}' for k, v in kw.items()])})")
            return f(*args, **kw)
        return call


def run_plan_steps(handles, plans, seeds):
    """the steps of the plans round-robin, plan k on handles[k]; a failure names the seed, the step and the calls"""
    keeps = [dict() for _ in handles]
    recs = [Recorded(h) for h in handles]
    for i in range(max(len(p) for p in plans)):
        for k, (rec, plan) in enumerate(zip(recs, plans)):
            if i >= len(plan):
                continue
            s = plan[i]
            rec.log.append((i, []))
            try:
                run_step(rec, s, keeps[k])
            except (AssertionError, pkg().capi.CuberilleError) as e:
                raise AssertionError(failure_report(seeds[k], s, rec, plan, e)) from e


def failure_report(seed, s, rec, plan, err):
    P = pkg()
    fresh = P.capi.Handle(0)
    try:
        run_step(fresh, s, {})
        verdict = "passes on a fresh handle: the state left by the earlier steps is the cause"
    except (AssertionError, P.capi.CuberilleError) as e2:
        verdict = f"fails on a fresh handle too ({str(e2).splitlines()[0]}): not a state bug"
    finally:
        fresh.close()
    lines = [f"seed {seed}, step {s['index']}: {err}", f"  {verdict}", "  calls on this handle:"]
    for i, calls in rec.log:
        lines.append(f"    step {i} [{describe(plan[i])}]: " + "; ".join(calls))
    return "\n".join(lines)


# ---- the plans ---------------------------------------------------------------------------------------------------------------
def test_plans_are_reproducible():
    assert make_plan(3, 40) == make_plan(3, 40)
    assert make_plan(3, 40) != make_plan(4, 40)


def test_plans_contain_every_transition():
    """the plans the GPU tests run hold every mode, emission, path, route and layout transition at least once,
    and asynchronous runs after both a larger and a smaller run on the same handle (the redo and the fitting path)"""
    tags = set().union(*(transitions(make_plan(seed, N_STEPS)) for seed in SEEDS))
    assert not REQUIRED - tags, f"missing from the plans: {sorted(REQUIRED - tags)}"


def test_k1_route_restatement_matches_the_route_table_of_the_classification_tests():
    from test_gpu_pixel_edges import ROUTES
    for name, (xs, misaligned, fused) in ROUTES.items():
        for pb, x in xs.items():
            dt = {1: np.uint8, 2: np.uint16, 4: np.float32, 8: np.float64}[pb]
            r = k1_route((4, 4, x), dt, False, pb if misaligned else 0)
            assert (r == "fused") == fused, (name, pb, r)
            if name.startswith("packed"):
                assert r == "packed"


@gpu
@pytest.mark.parametrize("seed", SEEDS)
def test_one_handle_runs_a_seeded_plan(seed):
    P = pkg()
    h = P.capi.Handle(0)
    try:
        run_plan_steps([h], [make_plan(seed, N_STEPS)], [seed])
    finally:
        h.close()


@gpu
@pytest.mark.parametrize("seeds", [(0, 1), (2, 5)])
def test_two_handles_on_two_streams_run_interleaved_plans(seeds):
    import torch
    P = pkg()
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    hs = [P.capi.Handle(0, stream=st.cuda_stream) for st in streams]
    try:
        run_plan_steps(hs, [make_plan(sd, N_STEPS) for sd in seeds], list(seeds))
    finally:
        for h in hs:
            h.close()


# ---- z-slabs at the exact projection halo ---------------------------------------------------------------------------------
RELAX = [0.0, 0.5, 0.95, 1.0]
MAX_STEPS = [0, 1, 60]
STEPS = ["auto", "tiny", "small", "large"]   # -1, 1e-12 and 1e-3 x the largest spacing, 2 x the largest spacing


def _step_length(kind, spacing):
    return {"auto": -1.0, "tiny": 1e-12 * max(spacing), "small": 1e-3 * max(spacing), "large": 2.0 * max(spacing)}[kind]


def halo_cases():
    """every (relaxation, max_steps, step) with the threshold, z spacing and method cycled through, then rotations
    that mix z with x or y on anisotropic voxels"""
    cases = []
    for i, (r, n, st) in enumerate(itertools.product(RELAX, MAX_STEPS, STEPS)):
        zs = (0.5, 1.0, 2.0)[i % 3]
        cases.append(dict(relax=r, max_steps=n, step=st, thr=(0.0, 0.02)[(i // 3) % 2], method=(i // 2) % 3,
                          spacing=(1.0, 1.0, zs), direction=None))
    for i, d in enumerate(sorted(DIRECTIONS)):
        for sp in [(0.7, 1.1, 1.6), (1.3, 0.9, 0.6)]:
            cases.append(dict(relax=0.95, max_steps=20, step="auto", thr=0.02, method=i % 3, spacing=sp, direction=d))
    return cases


def _case_id(c):
    return (f"r{c['relax']}-n{c['max_steps']}-{c['step']}-thr{c['thr']}-m{c['method']}-sz{c['spacing'][2]}"
            + (f"-{c['direction']}" if c["direction"] else ""))


HALO_CASES = halo_cases()


def halo_params(c, iso):
    return _count_params(iso, generate_triangles=1, project_vertices=1, projection_method=c["method"],
                         surface_distance_threshold=c["thr"], step_length=_step_length(c["step"], c["spacing"]),
                         step_relaxation=c["relax"], max_steps=c["max_steps"])


def expected_halo(c):
    """the reach of a vertex in slices, from the geometric sum of its <= max_steps + 2 moves, in exact rationals as
    far as the inputs allow: below = reach + 3, above = reach + 2 (no projection: 2 / 1)"""
    sp = c["spacing"]
    step = _step_length(c["step"], sp)
    step = 0.25 * max(sp) if step < 0 else step
    r, n = c["relax"], c["max_steps"] + 2
    travel = step * n if r >= 1.0 else step * (1.0 - r ** n) / (1.0 - r)
    if c["direction"]:
        D = np.array(DIRECTIONS[c["direction"]]).reshape(3, 3)
        zpu = float(np.abs(np.linalg.inv(D * np.array(sp))[2]).sum())
    else:
        zpu = 1.0 / sp[2]
    ct = math.ceil(travel / (1.0 / zpu) - 1e-9)
    return ct + 3, ct + 2


def test_projection_halo_is_the_reach_plus_the_footprints():
    """cub_projection_halo_oriented over the whole grid (a CPU call): the asymmetric +3 / +2, the r >= 1 branch, max_steps 0, a
    reach of zero slices, and the z row of M^-1 for rotated images"""
    P = pkg()
    seen = set()
    for c in HALO_CASES:
        got = P.capi.projection_halo(halo_params(c, 0.0), c["spacing"], DIRECTIONS.get(c["direction"]))
        assert got == expected_halo(c), (_case_id(c), got, expected_halo(c))
        seen.add(got[0] - 3)
    assert 0 in seen and max(seen) > 100
    # cub_projection_halo is the same halo of a non-oriented image
    L, lo, hi = P.capi.load(), ctypes.c_uint64(), ctypes.c_uint64()
    for c in HALO_CASES:
        if not c["direction"]:
            assert L.cub_projection_halo(ctypes.byref(halo_params(c, 0.0)), (ctypes.c_double * 3)(*c["spacing"]),
                                         ctypes.byref(lo), ctypes.byref(hi)) == 0
            assert (lo.value, hi.value) == expected_halo(c), _case_id(c)
    p = halo_params(HALO_CASES[0], 0.0)
    p.project_vertices = 0
    assert P.capi.projection_halo(p, (1.0, 1.0, 0.5), DIRECTIONS["oblique"]) == (2, 1)
    # a rotation that mixes z needs more slices than the same spacing without it
    c = dict(relax=0.95, max_steps=20, step="auto", thr=0.02, method=0, spacing=(1.0, 1.0, 1.0), direction=None)
    plain = P.capi.projection_halo(halo_params(c, 0.0), c["spacing"])
    rotated = P.capi.projection_halo(halo_params(c, 0.0), c["spacing"], DIRECTIONS["rot_x_30"])
    assert rotated[0] > plain[0] and rotated[1] > plain[1]


def test_projection_halo_refuses_a_bad_geometry():
    P = pkg()
    p = halo_params(HALO_CASES[0], 0.0)
    for sp, d in [((1.0, 0.0, 1.0), None), ((1.0, float("nan"), 1.0), None), ((1.0, 1.0, 1.0), (0.0,) * 9),
                  ((1.0, 1.0, 1.0), (1.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, float("inf")))]:
        with pytest.raises(P.capi.CuberilleError):
            P.capi.projection_halo(p, sp, d)


@gpu
@pytest.mark.parametrize("c", HALO_CASES, ids=_case_id)
def test_slabs_at_the_exact_projection_halo(c):
    """three slabs whose buffers hold exactly (below, above) of cub_projection_halo_oriented: the concatenation is the whole
    run and the oracle's mesh bit for bit, and the middle slab with one slice less below or above is refused"""
    O, P = oracle(), pkg()
    D = DIRECTIONS.get(c["direction"])
    probe = halo_params(c, 60.0)
    below, above = P.capi.projection_halo(probe, c["spacing"], D)
    a = below + 4            # own ranges [0, a), [a, b), [b, nz): every cut has its whole halo inside the image
    b = a + 6
    nz = b + above + 4
    vol, iso = smooth_volume((nz, 10, 12), np.float32, seed=int(sum(map(ord, _case_id(c)))))
    p = halo_params(c, iso)
    cuts = [(0, a), (a, b), (b, nz)]
    kw = dict(triangles=True, project=True, thr=c["thr"], step=p.step_length, relax=c["relax"], max_steps=c["max_steps"],
              method=c["method"], spacing=c["spacing"], direction=D)
    ref = O.cuberille(vol, iso, mode=O.CLOSED_FORM, **kw)
    h = P.capi.Handle(0)
    h.set_volume(vol, c["spacing"], (0.0, 0.0, 0.0), D)
    whole = _gpu_mesh(h, p)
    assert_same_mesh(whole, ref, "whole image")
    pts, cells, pb, cb = [], [], 0, 0
    for z0, z1 in cuts:
        lo, hi = max(0, z0 - below), min(nz, z1 + above)
        # a true slab: the halo on each cut side lies inside the image, so nothing is clipped there
        assert (z0 == 0 or z0 - below > 0) and (z1 == nz or z1 + above < nz), (z0, z1, below, above, nz)
        h.set_volume(vol[lo:hi], c["spacing"], (0.0, 0.0, 0.0), D)
        h.set_slab(nz, lo, z0, z1)
        n_pts, n_quads = h.count(p)
        h.set_id_base(pb, cb)
        h.emit(4)
        x, y, _ = h.fetch()
        pts.append(x)
        cells.append(y)
        pb, cb = pb + n_pts, cb + 2 * n_quads
    got = P.Mesh(np.concatenate(pts), np.concatenate(cells))
    assert_mesh_equal(got, ref, f"slabs {cuts} with halo ({below}, {above})")
    # the contract is exact: one slice less on either side of the middle slab is refused by cub_count
    for lo, hi, side in [(a - below + 1, b + above, "below"), (a - below, b + above - 1, "above")]:
        h.set_volume(vol[lo:hi], c["spacing"], (0.0, 0.0, 0.0), D)
        h.set_slab(nz, lo, a, b)
        with pytest.raises(P.capi.CuberilleError) as e:
            h.count(p)
        assert e.value.code == 1 and "halo" in str(e.value), f"one slice less {side}: {e.value}"
    h.close()
