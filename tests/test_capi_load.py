"""CPU: the C-ABI library builds, loads, and exports every symbol include/cuberille_c.h declares.
No compute call is made (there is no GPU here); creating a handle without a device must fail loudly."""
import os
import re

import pytest

from util import ROOT, pkg


def test_library_builds_and_exports_every_declared_symbol():
    P = pkg()
    P.build()
    L = P.capi.load()
    header = open(os.path.join(ROOT, "include", "cuberille_c.h")).read()
    declared = set(re.findall(r"\b(cub_[a-z_0-9]+)\s*\(", header))
    declared -= {"cub_handle_s"}
    assert declared == set(P.capi.SYMBOLS), declared ^ set(P.capi.SYMBOLS)
    for s in declared:
        assert hasattr(L, s), f"{s} not exported"
    assert L.cub_abi_version() == 3


def test_default_params_are_the_reference_constructor_defaults():
    p = pkg().capi.default_params()  # txx:31-41
    assert (p.iso_value, p.generate_triangles, p.project_vertices, p.save_pixel_as_cell_data) == (1.0, 1, 1, 0)
    assert (p.surface_distance_threshold, p.step_length, p.step_relaxation, p.max_steps) == (0.5, -1.0, 0.95, 50)


def test_no_cpu_fallback():
    # in a child process that sees no device (CUDA_VISIBLE_DEVICES hides one that is present)
    import subprocess
    import sys
    code = ("import importlib, sys\n"
            "P = importlib.import_module('midas-journal-740_b200')\n"
            "try:\n"
            "    P.capi.Handle(0)\n"
            "except P.capi.CuberilleError:\n"
            "    sys.exit(0)\n"
            "sys.exit('a handle was created without a device')\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr


def test_product_does_not_import_the_oracle():
    pk = os.path.join(ROOT, "midas-journal-740_b200")
    for dirpath, _, files in os.walk(pk):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                text = open(os.path.join(dirpath, f)).read()
                # comments may cite the oracle; nothing may import, load or include it
                assert "oracle_py" not in text and "liboracle" not in text, f
                assert not re.search(r'#include\s*[<"][^>"]*oracle', text), f
    for f in os.listdir(os.path.join(ROOT, "include")):
        text = open(os.path.join(ROOT, "include", f)).read()
        assert "liboracle" not in text and not re.search(r'#include\s*[<"][^>"]*oracle', text), f


def test_filter_mirror_defaults_and_clamps():
    # constructing the mirror needs a device; only the static parts are checked here
    P = pkg()
    F = P.CuberilleImageToMeshFilter
    f = F.__new__(F)
    f._image = None
    f._modified = False
    for name, val in dict(_iso=1, _triangles=True, _project=True, _cell_data=False, _thr=0.5, _step=-1.0, _relax=0.95,
                          _max_steps=50).items():
        setattr(f, name, val)
    f.SetProjectVertexStepLengthRelaxationFactor(1.5)   # itkSetClampMacro h:223
    assert f.GetProjectVertexStepLengthRelaxationFactor() == 1.0
    f.SetProjectVertexStepLength(-3.0)                  # h:216: the -1 "auto" sentinel cannot be restored
    assert f.GetProjectVertexStepLength() == 0.0
    f.SetProjectVertexSurfaceDistanceThreshold(-1.0)    # h:210
    assert f.GetProjectVertexSurfaceDistanceThreshold() == 0.0
    f.GenerateTriangleFacesOff()
    assert f.GetGenerateTriangleFaces() is False and f._modified
    # h:187-188: only the default (trilinear) interpolator exists on the GPU path
    f.SetInterpolator(P.LinearInterpolateImageFunction())
    assert isinstance(f.GetInterpolator(), P.LinearInterpolateImageFunction)
    with pytest.raises(TypeError):
        f.SetInterpolator(object())


def test_params_struct_layout_matches_the_header(tmp_path):
    """the ctypes mirror of cub_params (capi.Params) has the layout the C compiler gives the header's struct"""
    import ctypes as C
    import os
    import subprocess
    P = pkg()
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "layout.c"
    fields = [name for name, _ in P.capi.Params._fields_]
    body = "\n".join(f'  printf("{f} %zu\\n", offsetof(cub_params, {f}));' for f in fields)
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "cuberille_c.h"\nint main(void) {\n'
                   '  printf("sizeof %zu\\n", sizeof(cub_params));\n' + body + "\n  return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-I", os.path.join(root, "include"), "-o", str(exe), str(src)])
    out = dict(line.split() for line in subprocess.check_output([str(exe)], text=True).splitlines())
    assert int(out["sizeof"]) == C.sizeof(P.capi.Params)
    for f in fields:
        assert int(out[f]) == getattr(P.capi.Params, f).offset, f
