"""int64 and uint64 pixels without a device: the oracle's 64-bit instantiations (tests/oracle64.cpp), the conversion
rule of the projection, MetaImage IO, the C++ adapter's pixel codes, and the Python guard on pixel values.

The oracle is one template over the pixel type.  On values an int32 holds, its int64 and uint64 meshes must be its int32
meshes; on values beyond 2^53 the projection must convert a pixel to float and to double in one rounding each, as the
kernels do (DESIGN.md section 2)."""
import os
import subprocess

import numpy as np
import pytest

import oracle64 as O64
import range_oracle as R
from util import ROOT, oracle, pkg, smooth_volume

I64_TYPES = [np.int64, np.uint64]
I64_IDS = ["int64", "uint64"]
CPP = os.path.join(ROOT, "tests", "cpp")


def round_to_float32(n: int) -> float:
    """the float32 nearest to the integer n, ties to even, computed on the integer itself (one rounding)"""
    m = abs(n)
    shift = max(m.bit_length() - 24, 0)
    q, r = divmod(m, 1 << shift)
    half = (1 << shift) >> 1
    if shift and (r > half or (r == half and q & 1)):
        q += 1
    v = float(q << shift)   # at most 25 significant bits: exact in a double and in a float
    assert float(np.float32(v)) == v
    return -v if n < 0 else v


def test_round_to_float32_reference():
    v = 2**60 + 2**36 + 1
    assert round_to_float32(v) == float(2**60 + 2**37)
    assert float(np.float32(float(v))) == float(2**60)   # through double: the double is a tie and rounds to even
    assert round_to_float32(2**24 + 1) == float(2**24) and round_to_float32(2**24 + 3) == float(2**24 + 4)
    assert round_to_float32(-(2**60 + 2**36 + 1)) == -float(2**60 + 2**37)


# ---- the oracle on values an int32 holds ---------------------------------------------------------------------------------
@pytest.mark.parametrize("dt", I64_TYPES, ids=I64_IDS)
@pytest.mark.parametrize("kw", [dict(triangles=False, project=False), dict(triangles=True, project=True),
                                dict(triangles=True, project=True, method=1), dict(triangles=False, project=True, method=2),
                                dict(triangles=True, project=False, border_faces=True)],
                         ids=["quads", "tris_proj", "advanced", "linesearch", "border"])
@pytest.mark.parametrize("cell_data", [False, True], ids=["nocd", "cd"])
def test_oracle_64bit_iso_meshes_equal_the_int32_meshes(dt, kw, cell_data):
    v32, iso = smooth_volume((14, 17, 19), np.int32, seed=5)
    if dt is np.int64:
        v32, iso = v32 - 60, iso - 60   # negative values too
    ref = O64.cuberille(v32, iso, cell_data=cell_data, **kw)
    got = O64.cuberille(v32.astype(dt), iso, cell_data=cell_data, **kw)
    assert ref.cells.shape[0] > 100
    assert np.array_equal(got.cells, ref.cells)
    assert np.array_equal(got.points.view(np.uint32), ref.points.view(np.uint32))
    if cell_data:
        assert got.cell_data.dtype == np.dtype(dt) and np.array_equal(got.cell_data.astype(np.int64), ref.cell_data)
    else:
        assert got.cell_data is None


@pytest.mark.parametrize("dt", I64_TYPES, ids=I64_IDS)
@pytest.mark.parametrize("cell_data", [False, True], ids=["nocd", "cd"])
def test_range_meshes_of_64bit_maps_equal_the_int32_ones(dt, cell_data):
    v32, _ = smooth_volume((12, 13, 15), np.int32, seed=9)
    lo, hi = 50, 70
    ref = R.cuberille_range(v32, lo, hi, cell_data=cell_data, triangles=True)
    got = R.cuberille_range(v32.astype(dt), lo, hi, cell_data=cell_data, triangles=True)
    assert ref.cells.shape[0] > 50
    assert np.array_equal(got.cells, ref.cells) and np.array_equal(got.points.view(np.uint32), ref.points.view(np.uint32))
    if cell_data:
        assert got.cell_data.dtype == np.dtype(dt) and np.array_equal(got.cell_data.astype(np.int64), ref.cell_data)


@pytest.mark.parametrize("dt", I64_TYPES, ids=I64_IDS)
def test_oracle_classify_compares_in_64_bits(dt):
    info = np.iinfo(dt)
    vals = np.array(sorted({info.min, info.min + 1, 0, 1, 2**53, 2**53 + 1, 2**53 + 2, 2**60 + 2**36 + 1, info.max - 1,
                            info.max} | ({-(2**53) - 2, -1} if info.min < 0 else set())), dt)
    vol = np.ascontiguousarray(np.resize(vals, (2, 3, 40)))
    for iso in (2**53, 2**53 + 2, float(2**60), float(info.min)):
        bits = O64.classify(vol, iso)
        want = ~(vol < np.array(int(iso)).astype(dt))
        got = np.unpackbits(bits.view(np.uint8), axis=-1, bitorder="little")[..., :vol.shape[2]].astype(bool)
        assert np.array_equal(got, want), iso


# ---- the conversion rule of the projection --------------------------------------------------------------------------------
@pytest.mark.parametrize("dt", I64_TYPES, ids=I64_IDS)
def test_gradient_converts_a_pixel_to_float_directly(dt):
    """the gradient at node 1 of the row [0, 0, v] is 0.5f * (float)v; v = 2^60 + 2^36 + 1 tells the one-step conversion
    (2^60 + 2^37) from int64 -> double -> float (2^60); interpolation reads (double)v"""
    v = 2**60 + 2**36 + 1
    vol = np.zeros((1, 1, 3), dt)
    vol[0, 0, 2] = v
    val, grad = O64.sample(vol, np.array([[1.0, 0.0, 0.0], [2.0, 0.0, 0.0]]))
    assert grad[0, 0] == 0.5 * round_to_float32(v) != 0.5 * float(2**60)
    assert val[1] == float(v) == float(2**60 + 2**36)
    if dt is np.int64:
        vol[0, 0, 2] = -v
        val, grad = O64.sample(vol, np.array([[1.0, 0.0, 0.0], [2.0, 0.0, 0.0]]))
        assert grad[0, 0] == -0.5 * round_to_float32(v) and val[1] == -float(v)


# ---- MetaImage --------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dt", I64_TYPES, ids=I64_IDS)
@pytest.mark.parametrize("compress", [False, True])
def test_mha_round_trip(dt, compress, tmp_path):
    P = pkg()
    info = np.iinfo(dt)
    data = np.array([info.min, info.max, 0, 2**60 + 2**36 + 1, 2**53 + 1, 7], dt).reshape(1, 2, 3)
    path = str(tmp_path / "v.mha")
    P.write_mha(path, P.Image(data, (1.0, 2.0, 3.0), (0.5, 0.0, -1.0)), compress=compress)
    head = open(path, "rb").read(400)
    assert (b"MET_LONG_LONG" if dt is np.int64 else b"MET_ULONG_LONG") in head
    img = P.read_mha(path)
    assert img.data.dtype == np.dtype(dt) and np.array_equal(img.data, data)
    assert img.spacing == (1.0, 2.0, 3.0) and img.origin == (0.5, 0.0, -1.0)


# ---- bindings ---------------------------------------------------------------------------------------------------------------
def test_dtype_codes():
    capi = pkg().capi
    assert capi.DTYPE_CODES[np.dtype(np.int64)] == capi.I64 == 8
    assert capi.DTYPE_CODES[np.dtype(np.uint64)] == capi.U64 == 9
    assert capi.CODE_DTYPES[8] == np.dtype(np.int64) and capi.CODE_DTYPES[9] == np.dtype(np.uint64)
    assert [capi.DTYPE_CODES[np.dtype(d)] for d in (np.uint8, np.int8, np.uint16, np.int16, np.uint32, np.int32,
                                                    np.float32, np.float64)] == list(range(8))


def test_pixel_values_that_a_double_does_not_hold_are_refused_before_the_c_abi():
    capi = pkg().capi
    for v in (2**53 + 1, 2**60 + 2**36 + 1, np.int64(2**62 + 1), np.uint64(2**64 - 1), 2**63 - 1):
        with pytest.raises(ValueError, match="not exactly representable"):
            capi.pixel_value(v)
    for v in (2**53, 2**60, -(2**63), 2**64 - 2048, np.uint64(2**63), np.int64(-5), 0.5, 1e300, True, np.float32(2.5)):
        assert capi.pixel_value(v) == float(v)


# ---- the C++ adapter ------------------------------------------------------------------------------------------------------
def test_adapter_maps_the_64bit_integer_types_and_instantiates_for_them(tmp_path):
    """compile + link + run (no GPU needed: nothing calls Update()) of tests/cpp/adapter_instantiations64.cxx"""
    pkg().build()
    exe = str(tmp_path / "inst64")
    subprocess.check_call(["g++", "-O0", "-std=c++17", "-Wall", "-Wextra", "-Wno-unused-parameter", "-Wno-unused-local-typedefs",
                           "-I", os.path.join(ROOT, "include"), "-I", os.path.join(ROOT, "tests", "itk_shim"),
                           os.path.join(CPP, "adapter_instantiations64.cxx"), "-o", exe,
                           "-L", os.path.dirname(pkg().capi.lib_path()), "-lcuberille_cuda",
                           "-Wl,-rpath," + os.path.dirname(pkg().capi.lib_path())])
    assert subprocess.run([exe]).returncode == 0
