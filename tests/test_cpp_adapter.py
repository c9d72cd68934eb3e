"""The C++ drop-in: include/itkCuberilleImageToMeshFilter.h compiled against the minimal ITK stand-in and
driven by tests/cpp/cuberille_test01.cxx with the reference's own command lines (Testing/CMakeLists.txt)."""
import os
import subprocess

import numpy as np
import pytest

from util import DATA, KAT, ROOT, oracle, pkg, read_fixture

CPP = os.path.join(ROOT, "tests", "cpp")
EXE = os.path.join(CPP, "CuberilleTest01")


def build_driver():
    pkg().build()
    subprocess.check_call(["make", "-C", CPP, "-s"])
    return EXE


def kat_args(row, out):
    name, fixture, iso, exp_points, exp_cells, tri, proj, max_steps = row
    return [EXE, "Test01", os.path.join(DATA, fixture + ".mha"), out, str(iso), str(exp_points), str(exp_cells),
            str(tri), str(proj), "0.2", "0.24", "0.95", str(max_steps)]


def test_driver_compiles_and_fails_loudly_without_a_gpu(tmp_path):
    build_driver()
    # CUDA_VISIBLE_DEVICES hides a device that is present
    r = subprocess.run(kat_args(KAT[0], str(tmp_path / "o.vtk")), capture_output=True, text=True,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode != 0
    assert "ExceptionObject caught" in r.stderr and "no usable CUDA device" in r.stderr


def test_adapter_instantiates_for_every_pixel_type_and_exports_the_reference_typedefs(tmp_path):
    """compile + link + run (no GPU needed: nothing calls Update()) of tests/cpp/adapter_instantiations.cxx"""
    pkg().build()
    exe = str(tmp_path / "inst")
    subprocess.check_call(["g++", "-O0", "-std=c++17", "-Wall", "-Wextra", "-Wno-unused-parameter", "-Wno-unused-local-typedefs",
                           "-I", os.path.join(ROOT, "include"), "-I", os.path.join(ROOT, "tests", "itk_shim"),
                           os.path.join(CPP, "adapter_instantiations.cxx"), "-o", exe,
                           "-L", os.path.dirname(pkg().capi.lib_path()), "-lcuberille_cuda",
                           "-Wl,-rpath," + os.path.dirname(pkg().capi.lib_path())])
    assert subprocess.run([exe]).returncode == 0


def test_driver_usage_message(tmp_path):
    build_driver()
    r = subprocess.run([EXE], capture_output=True, text=True)
    assert r.returncode != 0 and "USAGE" in r.stdout


def read_vtk(path):
    lines = open(path).read().split("\n")
    i = next(k for k, l in enumerate(lines) if l.startswith("POINTS"))
    n = int(lines[i].split()[1])
    pts = np.array([[float(v) for v in lines[i + 1 + k].split()] for k in range(n)], np.float32).reshape(n, 3)
    j = next(k for k, l in enumerate(lines) if l.startswith("POLYGONS"))
    m = int(lines[j].split()[1])
    cells = np.array([[int(v) for v in lines[j + 1 + k].split()[1:]] for k in range(m)], np.uint64)
    return pts, cells


@pytest.mark.gpu
@pytest.mark.parametrize("row", KAT, ids=[r[0] for r in KAT])
def test_reference_ctest_rows_through_the_cpp_filter(row, tmp_path):
    build_driver()
    out = str(tmp_path / "mesh.vtk")
    r = subprocess.run(kat_args(row, out), capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert f"Mesh has {row[3]} vertices and {row[4]} cells" in r.stdout
    name, fixture, iso, _, _, tri, proj, max_steps = row
    ref = oracle().cuberille(read_fixture(fixture).data, iso, triangles=tri, project=proj, thr=0.2, step=0.24,
                             relax=0.95, max_steps=max_steps)
    pts, cells = read_vtk(out)
    assert np.array_equal(cells.reshape(ref.cells.shape), ref.cells)
    assert np.array_equal(pts.view(np.uint32), ref.points.view(np.uint32))  # %.9g round-trips float32
