"""Every classification route and the projection across the full value range of each pixel type.

Classification (K1 in its packed, fused, full-row, ragged and padded forms, and on borrowed device pointers at every
pixel-aligned offset) is compared with numpy's `~(vol < iso)` in the pixel type: every value of the 8- and 16-bit
types, the extremes of the 32-bit ones around 2^24 and 2^31, and the special floats (infinities, signed zeros,
subnormals, NaNs with several payloads).  Meshes, cell data and projections are compared with the CPU oracle, bit for
bit; a NaN coordinate only has to be NaN on both sides (DESIGN.md section 2).  The normalisation of the projection is
driven directly with gradients whose normalised components lie within two double ulps of a float rounding midpoint,
where the kernel's rsqrt fast path must hand over to the exact division.

The tests marked gpu need a CUDA device; the others check the premises of the GPU tests and run anywhere."""
import math
import os

import numpy as np
import pytest

from util import oracle, pkg, smooth_volume

gpu = pytest.mark.gpu

DTYPES = [np.uint8, np.int8, np.uint16, np.int16, np.uint32, np.int32, np.float32, np.float64]
DT_IDS = [np.dtype(d).name for d in DTYPES]


class _env:
    """the tuning knobs are read once, in cub_create: a handle per setting"""

    def __init__(self, **kv):
        self.kv = {k: str(v) for k, v in kv.items()}

    def __enter__(self):
        self.old = {k: os.environ.get(k) for k in self.kv}
        os.environ.update(self.kv)

    def __exit__(self, *a):
        for k, v in self.old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _handle(**env):
    with _env(**env):
        return pkg().capi.Handle(0)


# ---- values ----------------------------------------------------------------------------------------------------------
_UINT = {4: np.uint32, 8: np.uint64}
_NAN_BITS = {  # quiet / signalling, both signs, with and without payload
    4: [0x7FC00000, 0xFFC00000, 0x7F800001, 0xFF800001, 0x7FC12345, 0x7FA00000],
    8: [0x7FF8000000000000, 0xFFF8000000000000, 0x7FF0000000000001, 0xFFF0000000000001, 0x7FF800000000ABCD,
        0x7FF4000000000000],
}


def _special_floats(dt):
    """-inf, -max, -1, -min normal, -min subnormal, -0, +0, subnormals, min normal, 1, max, +inf"""
    fi = np.finfo(dt)
    sub = fi.smallest_subnormal
    return [-math.inf, -float(fi.max), -1.0, -float(fi.tiny), -float(sub), -0.0, 0.0, float(sub), float(3 * sub),
            float(fi.tiny - sub), float(fi.tiny), 1.0, float(fi.max), math.inf]


def _int_specials(dt):
    info = np.iinfo(dt)
    cand = {info.min, info.min + 1, -1, 0, 1, 0x7F, 0x80, 0xFF, 0x100, 0x7FFE, 0x7FFF, 0x8000, 0x8001, info.max - 1,
            info.max}
    if info.bits == 32:  # where an fp32 conversion starts to round, and the top bit of uint32
        cand |= {2**24 - 1, 2**24, 2**24 + 1, -(2**24) - 1, -(2**24), -(2**24) + 1, 2**31 - 1, 2**31, 2**31 + 1, 2**32 - 1}
    return sorted(v for v in cand if info.min <= v <= info.max)


def value_pool(dt):
    """the values every test volume of `dt` contains: all of them for 8/16-bit, the edge values otherwise"""
    dt = np.dtype(dt)
    if dt.kind in "iu":
        info = np.iinfo(dt)
        if info.bits <= 16:
            return np.arange(info.min, info.max + 1, dtype=np.int64).astype(dt)
        return np.array(_int_specials(dt), np.int64).astype(dt)
    finite = np.array(_special_floats(dt), dt)
    nans = np.array(_NAN_BITS[dt.itemsize], _UINT[dt.itemsize]).view(dt)
    return np.concatenate([finite.view(_UINT[dt.itemsize]), nans.view(_UINT[dt.itemsize])]).view(dt)


def pool_volume(dt, shape, seed):
    """the value pool once each, in a seeded order, the rest of the shape seeded draws (full-range integers for the
    32-bit types, pool values otherwise); built on the raw bits so that signalling NaNs stay as they are"""
    dt = np.dtype(dt)
    rng = np.random.default_rng(seed)
    pool = value_pool(dt)
    n = int(np.prod(shape))
    assert n >= pool.size
    if dt.kind in "iu" and dt.itemsize == 4:
        info = np.iinfo(dt)
        extra = rng.integers(info.min, info.max, n - pool.size, dtype=np.int64, endpoint=True).astype(dt)
    else:
        extra = pool[rng.integers(0, pool.size, n - pool.size)]
    raw = np.concatenate([pool.view(f"u{dt.itemsize}"), extra.view(f"u{dt.itemsize}")])
    return np.ascontiguousarray(raw[rng.permutation(n)].reshape(shape)).view(dt)


def iso_values(dt, seed=7):
    """8-bit: every value; 16-bit: the boundary set and 32 seeded ones; 32-bit: the edge values and 8 seeded ones;
    floats: every finite special value and both infinities"""
    dt = np.dtype(dt)
    if dt.kind == "f":
        return _special_floats(dt)
    info = np.iinfo(dt)
    if info.bits == 8:
        return [float(v) for v in range(info.min, info.max + 1)]
    rng = np.random.default_rng(seed)
    extra = rng.integers(info.min, info.max, 32 if info.bits == 16 else 8, dtype=np.int64, endpoint=True)
    return [float(v) for v in sorted(set(_int_specials(dt)) | set(int(v) for v in extra))]


def reference_inside(vol, iso):
    """`~(vol < iso)` evaluated by numpy in the pixel type"""
    with np.errstate(invalid="ignore"):
        return ~(vol < np.array(iso).astype(vol.dtype))


def unpack_bitmask(bits, nx):
    """the library's bitmask (bit x % 32 of word x // 32 of a row) as one bool per voxel"""
    return np.unpackbits(bits.astype("<u4").view(np.uint8), axis=-1, bitorder="little")[..., :nx].astype(bool)


def _pixel_bytes(dt):
    return np.dtype(dt).itemsize


# ---- classification routes (cuberille_capi.cu: launch_fused, launch_classify, ClassifyPacked) --------------------------
# row length per pixel size, environment, and whether the fused classification + sweep kernel must have run
ROUTES = {
    "packed": (dict(), {1: 128, 2: 64}, False),                         # 4 bytes per lane: whole warp loads per row
    "fused": (dict(), {1: 48, 2: 40, 4: 36, 8: 36}, True),              # rows of whole 16-byte groups
    "fused_unpacked": (dict(CUB_K1_PACKED=0), {1: 128, 2: 64}, True),
    "full_rows": (dict(CUB_FUSE=0, CUB_K1_PACKED=0), {1: 512, 2: 512, 4: 512, 8: 512}, False),
    "ragged33": (dict(CUB_FUSE=0), {1: 33, 2: 33, 4: 33, 8: 33}, False),
    "ragged70": (dict(CUB_FUSE=0), {1: 70, 2: 70, 4: 70, 8: 70}, False),
}


def route_shape(dt, nx):
    rows = max(48, -(-value_pool(dt).size // nx))
    ny = min(rows, 16)
    return (-(-rows // ny), ny, nx)


def _count_params(iso, **kw):
    p = pkg().capi.default_params()
    p.iso_value, p.generate_triangles, p.project_vertices = float(iso), 0, 0
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def check_bitmasks(h, vol, isos, fused, what):
    for iso in isos:
        h.count(_count_params(iso))
        assert h.count_was_fused() == fused, f"{what}: fused={h.count_was_fused()}"
        got = unpack_bitmask(h.bitmask(), vol.shape[2])
        bad = np.argwhere(got != reference_inside(vol, iso))
        if bad.size:
            z, y, x = bad[0]
            raise AssertionError(f"{what} iso={iso!r}: {len(bad)} voxels differ, first (x={x}, y={y}, z={z}) = "
                                 f"{vol[z, y, x]!r} classified {int(got[z, y, x])}")


@gpu
@pytest.mark.parametrize("dtype,route", [(d, r) for d in DTYPES for r in sorted(ROUTES) if _pixel_bytes(d) in ROUTES[r][1]],
                         ids=lambda v: v if isinstance(v, str) else np.dtype(v).name)
def test_classification_over_the_full_value_range(dtype, route):
    env, xs, fused = ROUTES[route]
    vol = pool_volume(dtype, route_shape(dtype, xs[_pixel_bytes(dtype)]), seed=11)
    h = _handle(**env)
    h.set_volume(vol)
    check_bitmasks(h, vol, iso_values(dtype), fused, f"{np.dtype(dtype).name} {route} {vol.shape}")
    h.close()


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_classification_of_borrowed_pointers_at_every_alignment(dtype):
    """a device volume at an offset that is a multiple of the pixel size but not of 16 (or 4): the fused and packed
    kernels must not run, the others must classify it as they do an aligned one"""
    import torch
    P = pkg()
    size = _pixel_bytes(dtype)
    offsets = sorted({o for o in (size, 4, 8, 12, 16, 24) if o % size == 0})
    xs = sorted({ROUTES["fused"][1][size]} | ({ROUTES["packed"][1][size]} if size <= 2 else set()))
    isos = iso_values(dtype)
    if len(isos) > 48:
        isos = isos[::len(isos) // 48]
    h = P.capi.Handle(0)
    for nx in xs:
        vol = pool_volume(dtype, route_shape(dtype, nx), seed=nx)
        raw = torch.from_numpy(vol.reshape(-1).view(np.uint8).copy())
        buf = torch.zeros(raw.numel() + 64, dtype=torch.uint8, device="cuda")
        for off in offsets:
            buf[off:off + raw.numel()].copy_(raw)
            torch.cuda.synchronize()  # (the handle's stream does not wait for torch's)
            h.set_volume_ptr(buf.data_ptr() + off, dtype, vol.shape[::-1], P.capi.MEM_DEVICE)
            h.count(_count_params(isos[0]))
            if off % 16:
                assert not h.count_was_fused(), f"fused kernel on a buffer at offset {off}"
            check_bitmasks(h, vol, isos, h.count_was_fused(), f"{np.dtype(dtype).name} nx={nx} offset {off}")
    h.close()
    del buf


@gpu
def test_device_pointer_not_aligned_to_the_pixel_is_refused():
    import torch
    P = pkg()
    buf = torch.zeros(256, dtype=torch.uint8, device="cuda")
    h = P.capi.Handle(0)
    for dtype in DTYPES:
        size = _pixel_bytes(dtype)
        for off in range(1, size):
            with pytest.raises(P.capi.CuberilleError) as e:
                h.set_volume_ptr(buf.data_ptr() + off, dtype, (4, 2, 2), P.capi.MEM_DEVICE)
            assert e.value.code == 1 and "aligned" in str(e.value)
        h.set_volume_ptr(buf.data_ptr() + size, dtype, (4, 2, 2), P.capi.MEM_DEVICE)  # accepted (nothing launched)
    h.close()


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_iso_must_be_a_pixel_value(dtype):
    """integer types: min and max are isos, one beyond them, fractions and NaN are not; float types: the infinities and
    -0 are isos, NaN is not"""
    P = pkg()
    dt = np.dtype(dtype)
    h = P.capi.Handle(0)
    h.set_volume(np.zeros((2, 2, 4), dt))
    if dt.kind in "iu":
        info = np.iinfo(dt)
        ok = [float(info.min), float(info.max), 0.0, -0.0]
        bad = [float(info.max) + 1.0, float(info.min) - 1.0, 0.5, float(info.max) - 0.5, math.nan, math.inf, -math.inf,
               1e300, -1e300]
    else:
        fi = np.finfo(dt)
        ok = [math.inf, -math.inf, -0.0, float(fi.max), float(fi.smallest_subnormal)]
        bad = [math.nan] + ([0.1, 1e39, float(fi.smallest_subnormal) / 2] if dt == np.float32 else [])
    for iso in ok:
        h.count(_count_params(iso))
    for iso in bad:
        with pytest.raises(P.capi.CuberilleError) as e:
            h.count(_count_params(iso))
        assert e.value.code == 1 and "not representable" in str(e.value), iso
    h.close()


# ---- meshes over the full value range -----------------------------------------------------------------------------------
TOP_BIT_ISO = {np.uint8: 200, np.int8: -56, np.uint16: 0xC000, np.int16: -0x4000, np.uint32: 0xC0000000,
               np.int32: -(2**30), np.float32: -1.0, np.float64: -1.0}


def _gpu_mesh(h, p, id_bytes=4):
    h.count(p)
    h.emit(id_bytes)
    return h.fetch(want_cell_data=bool(p.save_pixel_as_cell_data))


def assert_same_mesh(got, ref, what):
    """connectivity and cell data (as bytes) exactly; points bit for bit, except that a NaN coordinate only has to be
    NaN on both sides (the device's NaN is 0x7fffffff, the host's a default NaN or a propagated payload)"""
    pts, cells, cd = got
    assert pts.shape == ref.points.shape, f"{what}: #points {pts.shape} vs {ref.points.shape}"
    assert np.array_equal(cells.astype(np.uint64).reshape(ref.cells.shape), ref.cells), f"{what}: connectivity differs"
    assert_same_points(pts, ref.points, what)
    if ref.cell_data is not None:
        assert cd.dtype == ref.cell_data.dtype
        assert np.array_equal(cd.view(np.uint8), ref.cell_data.view(np.uint8)), f"{what}: cell data bytes differ"


def assert_same_points(got, ref, what):
    gn, rn = np.isnan(got), np.isnan(ref)
    if not np.array_equal(gn, rn):
        i = np.nonzero((gn != rn).any(axis=1))[0]
        raise AssertionError(f"{what}: {i.size} points are NaN on one side only, first {i[0]}: {got[i[0]]} vs {ref[i[0]]}")
    a, b = np.where(gn, 0, got.view(np.uint32)), np.where(rn, 0, ref.view(np.uint32))
    if not np.array_equal(a, b):
        i = np.nonzero((a != b).any(axis=1))[0]
        raise AssertionError(f"{what}: {i.size} points differ, first {i[0]}: {got[i[0]]!r} vs {ref[i[0]]!r}")


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=DT_IDS)
def test_full_range_meshes_and_cell_data(dtype):
    """quads and fixed-split triangles at an iso with the top bit set, with the raw pixel as cell data (negative values,
    top-bit values and NaN payloads come back byte for byte); the padded lattice (image_border_faces) at the route isos"""
    O, P = oracle(), pkg()
    size = _pixel_bytes(dtype)
    vol = pool_volume(dtype, route_shape(dtype, ROUTES["fused"][1][size]), seed=5)
    h = P.capi.Handle(0)
    h.set_volume(vol)
    iso = TOP_BIT_ISO[dtype]
    for tri in (False, True):
        p = _count_params(iso, generate_triangles=int(tri), save_pixel_as_cell_data=1)
        ref = O.cuberille(vol, iso, triangles=tri, project=False, cell_data=True, mode=O.CLOSED_FORM)
        assert ref.cells.shape[0] > 0
        assert_same_mesh(_gpu_mesh(h, p), ref, f"{np.dtype(dtype).name} tri={tri}")
    isos = iso_values(dtype)
    for iso in (isos if len(isos) <= 64 else isos[::len(isos) // 64]):
        p = _count_params(iso, image_border_faces=1)
        ref = O.cuberille(vol, iso, triangles=False, project=False, mode=O.CLOSED_FORM, border_faces=True)
        assert_same_mesh(_gpu_mesh(h, p), ref, f"{np.dtype(dtype).name} border faces iso={iso!r}")
    h.close()


# ---- projection at value edges ------------------------------------------------------------------------------------------
FLT_MAX = float(np.finfo(np.float32).max)


def mapped_volume(shape, dtype, lo, hi, seed):
    """a band-limited random field mapped onto [lo, hi]"""
    f, _ = smooth_volume(shape, np.float64, seed, scale=0.5)  # in [0, 1]
    v = np.clip(lo + f * (hi - lo), lo, hi)
    dt = np.dtype(dtype)
    return np.ascontiguousarray(np.rint(v).astype(dt) if dt.kind in "iu" else v.astype(dt))


def nonfinite_volume(shape, seed):
    """a smooth float32 field with +-inf and NaNs (several payloads) on voxels next to the surface, some of them on the
    image border"""
    vol, iso = smooth_volume(shape, np.float32, seed)
    rng = np.random.default_rng(seed)
    inside = vol >= iso
    near = np.zeros_like(inside)
    for ax in range(3):
        for s in (1, -1):
            near |= inside != np.roll(inside, s, axis=ax)
    cand = np.argwhere(near)
    border = cand[(cand == 0).any(axis=1) | (cand == np.array(shape) - 1).any(axis=1)]
    pick = np.concatenate([cand[rng.choice(len(cand), 40, replace=False)], border[rng.choice(len(border), 8, replace=False)]])
    special = np.array([0x7F800000, 0xFF800000] + _NAN_BITS[4], np.uint32).view(np.float32)
    raw = vol.view(np.uint32)
    for i, (z, y, x) in enumerate(pick):
        raw[z, y, x] = special.view(np.uint32)[i % special.size]
    return vol, iso


# name: (volume, iso, spacing, thr)
def projection_case(name):
    shape = (20, 18, 26)
    if name in ("int32", "uint32", "int16", "uint16"):
        dt = np.dtype(name)
        info = np.iinfo(dt)
        lo, hi = (2**31 + 3, 2**32 - 1) if name == "uint32" else (info.min, info.max)
        vol = mapped_volume(shape, dt, lo, hi, seed=41)
        return vol, (lo + hi) // 2, (1.0, 1.0, 1.0), (hi - lo) * 2e-3
    if name == "f32_near_max":  # spacing < 1: the central differences of opposite-signed neighbours overflow to inf
        return mapped_volume(shape, np.float32, -FLT_MAX, FLT_MAX, seed=42), 0.0, (0.5, 0.75, 0.25), 1e35
    if name == "f64_beyond_max":  # pixels that become +-inf in the fp32 gradient
        return mapped_volume(shape, np.float64, -4 * FLT_MAX, 4 * FLT_MAX, seed=43), 0.0, (1.0, 1.0, 1.0), 1e36
    if name == "f32_subnormal":
        return mapped_volume(shape, np.float32, -1e-39, 1e-39, seed=44), 0.0, (1.0, 1.0, 1.0), 1e-42
    if name == "f32_nonfinite":
        vol, iso = nonfinite_volume(shape, seed=45)
        return vol, iso, (1.0, 1.0, 1.0), 0.05
    raise KeyError(name)


PROJECTION_CASES = ["int32", "uint32", "int16", "uint16", "f32_near_max", "f64_beyond_max", "f32_subnormal", "f32_nonfinite"]


@gpu
@pytest.mark.parametrize("method", [0, 1, 2], ids=["default", "advanced", "linesearch"])
@pytest.mark.parametrize("name", PROJECTION_CASES)
def test_projection_at_value_edges(name, method):
    """triangles with projection (vertices in the interior take the cached-cell path, those on the image border the
    clamped one), and the projection kernel alone on points in and around the image"""
    O, P = oracle(), pkg()
    vol, iso, sp, thr = projection_case(name)
    kw = dict(thr=thr, step=0.3, relax=0.9, max_steps=30, method=method)
    ref = O.cuberille(vol, iso, triangles=True, project=True, spacing=sp, **kw)
    assert ref.points.shape[0] > 500
    h = P.capi.Handle(0)
    h.set_volume(vol, sp)
    p = _count_params(iso, generate_triangles=1, project_vertices=1, surface_distance_threshold=thr, step_length=0.3,
                      step_relaxation=0.9, max_steps=30, projection_method=method)
    assert_same_mesh(_gpu_mesh(h, p), ref, f"{name} method {method}")
    rng = np.random.default_rng(3)
    ext = np.array(vol.shape[::-1]) * np.array(sp)
    pts = (rng.random((4000, 3)) * (ext + 4) - 2 - 0.5 * np.array(sp)).astype(np.float32)
    got = h.project_points(p, pts)
    refp = O.project_points(vol, iso, pts, spacing=sp, **kw)
    assert_same_points(got, refp, f"{name} method {method}: project_points")
    if name.startswith("f") and name != "f32_subnormal" and method == 0:
        assert np.isnan(ref.points).any() or np.isnan(refp).any(), "no non-finite arithmetic was exercised"
    h.close()


# ---- the normalisation fast path (k_project.cuh: rsqrt, and the exact division near float rounding midpoints) ----------
def _near_midpoint(q, ulps=2):
    """float64 values within `ulps` double ulps of a float rounding midpoint (low 29 mantissa bits near 2^28)"""
    low = np.ascontiguousarray(q, np.float64).view(np.uint64) & np.uint64((1 << 29) - 1)
    return np.abs(low.astype(np.int64) - (1 << 28)) <= ulps


def exact_normal(g):
    """the oracle's normalisation of a float gradient: fp64 norm of the float components, fp64 quotients"""
    g = np.asarray(g, np.float32).astype(np.float64)
    sq = ((0.0 + g[0] * g[0]) + g[1] * g[1]) + g[2] * g[2]
    return g / np.sqrt(sq)


def sweep_for_midpoints(x0, gy, gz, n):
    """g_x over n consecutive floats from x0 at fixed g_y, g_z: the triples with a normalised component near a
    float rounding midpoint (about one in 10^7 candidates)"""
    gx = (np.float32(x0).view(np.int32) + np.arange(n, dtype=np.int32)).view(np.float32).astype(np.float64)
    gy, gz = float(np.float32(gy)), float(np.float32(gz))
    nrm = np.sqrt((gx * gx + gy * gy) + gz * gz)
    hit = _near_midpoint(gx / nrm) | _near_midpoint(gy / nrm) | _near_midpoint(gz / nrm)
    return [(float(np.float32(x)), gy, gz) for x in gx[hit]]


# found by sweep_for_midpoints over 5 x 10^7 to 8 x 10^7 candidates for each (g_y, g_z) pair
MIDPOINT_GRADIENTS = [
    (2.960162878036499, 0.75, -0.30000001192092896),
    (12.896516799926758, 0.75, -0.30000001192092896),
    (26.28196907043457, 0.75, -0.30000001192092896),
    (1772131.375, -170000.0, 22000.0),
    (-0.033652130514383316, 0.0024999999441206455, 0.0010999999940395355),
    (55266812887040.0, 299999985664.0, 799999983616.0),
    (-7.025059700012207, -2.0, 9.0),
    (-173.4060821533203, -2.0, 9.0),
    # here g_x times the correctly rounded 1 / sqrt(sq) rounds to the other float than g_x / sqrt(sq)
    (39588.0078125, 77.0, -250.0),
]
# a component that normalises below the smallest normal float, and subnormal inputs
SUBNORMAL_GRADIENTS = [(1e30, 1e-9, 0.0), (-1e30, 0.0, 3e-9), (1e-40, -3e-40, 2e-41)]
PLANTED = MIDPOINT_GRADIENTS + SUBNORMAL_GRADIENTS
PERMUTE = (0.0, 1.0, 0.0, 0.0, 0.0, 1.0, 1.0, 0.0, 0.0)  # an axis permutation: an exact rotation of the gradient
PLANT_ARGS = dict(iso=1.0, thr=0.5, step=1.0, relax=0.0, max_steps=0)


def planted_volume(g):
    """3x3x3 float32 volume, spacing 1, origin -1: the centre node sits at physical (0, 0, 0), its value 0 is far from
    the iso (1), and its -1 / +1 neighbours are 0 / 2 g_k, so that its fp32 central difference is exactly g_k"""
    g = np.asarray(g, np.float32)
    vol = np.zeros((3, 3, 3), np.float32)
    vol[1, 1, 2], vol[1, 2, 1], vol[2, 1, 1] = 2 * g[0], 2 * g[1], 2 * g[2]
    return vol


def oracle_gradient_at_centre(vol):
    """numpy float32 restatement of the oracle's gradient_at: 0 + (-c) I[-1] + 0 I[0] + c I[+1]"""
    c = np.float32(0.5 * (1.0 / 1.0))
    mid = vol[1, 1, 1]
    out = []
    for lo, hi in ((vol[1, 1, 0], vol[1, 1, 2]), (vol[1, 0, 1], vol[1, 2, 1]), (vol[0, 1, 1], vol[2, 1, 1])):
        s = np.float32(0.0)
        s = np.float32(s + np.float32(-c) * lo)
        s = np.float32(s + np.float32(0.0) * mid)
        s = np.float32(s + c * hi)
        out.append(s)
    return np.array(out, np.float32)


def _project_planted(project, g, direction=None):
    """the vertex starts on the centre node: the first move puts it at +normal (value 0 < iso), relaxation 0 keeps it
    there.  With a direction the planted gradient is g rotated back, so that the rotated one is g again."""
    if direction is not None:
        g = np.array(direction).reshape(3, 3).T @ np.asarray(g, np.float64)
    return project(planted_volume(g), np.zeros((1, 3), np.float32), direction)[0]


def _oracle_project(vol, pts, direction):
    a = dict(PLANT_ARGS)
    return oracle().project_points(vol, a.pop("iso"), pts, spacing=(1.0, 1.0, 1.0), origin=(-1.0, -1.0, -1.0),
                                   direction=direction, **a)


def test_planted_components_lie_within_two_ulps_of_a_rounding_midpoint():
    for g in MIDPOINT_GRADIENTS:
        assert np.array_equal(np.asarray(g, np.float32).astype(np.float64), np.asarray(g)), g  # floats as written
        assert _near_midpoint(exact_normal(g)).any(), g
    for g in SUBNORMAL_GRADIENTS:
        n = np.abs(exact_normal(g))
        assert ((n > 0) & (n < np.finfo(np.float32).tiny)).any() or (np.abs(np.float32(g)) < np.finfo(np.float32).tiny).all()


def test_the_midpoint_search_finds_the_planted_gradients():
    x, gy, gz = MIDPOINT_GRADIENTS[0]
    start = (np.float32(x).view(np.int32) - 5000).view(np.float32)
    assert (x, gy, gz) in sweep_for_midpoints(float(start), gy, gz, 10000)


@pytest.mark.parametrize("g", PLANTED)
def test_the_planted_node_gradient_is_exactly_g(g):
    got = oracle_gradient_at_centre(planted_volume(g))
    assert np.array_equal(got.view(np.uint32), np.asarray(g, np.float32).view(np.uint32))


@pytest.mark.parametrize("g", PLANTED)
def test_the_oracle_moves_the_planted_vertex_to_the_normal(g):
    normal = exact_normal(g).astype(np.float32)
    got = _project_planted(_oracle_project, g)
    assert np.array_equal(got.view(np.uint32), normal.view(np.uint32)), (got, normal)
    got = _project_planted(_oracle_project, g, PERMUTE)
    assert np.array_equal(got.view(np.uint32), normal.view(np.uint32)), (got, normal)


@gpu
@pytest.mark.parametrize("centre", [math.inf, -math.inf, math.nan], ids=["inf", "-inf", "nan"])
def test_non_finite_node_under_a_vertex_on_it(centre):
    """a vertex exactly on a node weighs that node alone, so only the node's `0 * I[0]` term (NaN for a non-finite
    I[0]) makes its gradient NaN: the planted volume with its centre replaced, finite neighbours"""
    P = pkg()
    vol = planted_volume((1.0, 2.0, 3.0))
    vol[1, 1, 1] = centre
    pts = np.zeros((1, 3), np.float32)
    ref = _oracle_project(vol, pts, None)
    assert np.isnan(ref).all()
    h = P.capi.Handle(0)
    h.set_volume(vol, (1.0, 1.0, 1.0), (-1.0, -1.0, -1.0))
    p = _count_params(PLANT_ARGS["iso"], project_vertices=1, surface_distance_threshold=PLANT_ARGS["thr"],
                      step_length=PLANT_ARGS["step"], step_relaxation=PLANT_ARGS["relax"], max_steps=PLANT_ARGS["max_steps"])
    assert_same_points(h.project_points(p, pts), ref, f"centre {centre}")
    h.close()


@gpu
@pytest.mark.parametrize("oriented", [False, True])
def test_normalisation_near_rounding_midpoints(oriented):
    """K4 alone on the planted gradients: a one-ulp error of the normal would survive in the vertex"""
    P = pkg()
    direction = PERMUTE if oriented else None
    h = P.capi.Handle(0)
    p = _count_params(PLANT_ARGS["iso"], project_vertices=1, surface_distance_threshold=PLANT_ARGS["thr"],
                      step_length=PLANT_ARGS["step"], step_relaxation=PLANT_ARGS["relax"], max_steps=PLANT_ARGS["max_steps"])

    def gpu_project(vol, pts, direction):
        h.set_volume(vol, (1.0, 1.0, 1.0), (-1.0, -1.0, -1.0), direction)
        return h.project_points(p, pts)

    bad = []
    for g in PLANTED:
        got = _project_planted(gpu_project, g, direction)
        ref = _project_planted(_oracle_project, g, direction)
        if not np.array_equal(got.view(np.uint32), ref.view(np.uint32)):
            bad.append((g, got, ref))
    assert not bad, f"{len(bad)} of {len(PLANTED)} planted normals differ, first: {bad[0]}"
    h.close()
