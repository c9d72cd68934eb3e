"""Python mirror of itk::CuberilleImageToMeshFilter's public interface (h:110-228).

The product host side is C++ (include/itkCuberilleImageToMeshFilter.h); this mirror exists so
that the parity tests and the bench can drive the C-ABI with the reference's own vocabulary:
same method names, argument meaning, defaults (txx:31-41), clamps (h:210,216,223) and the sticky
auto step length (txx:82-85).  It holds no algorithm: every Update() goes through
libcuberille_cuda.so.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from . import capi
from .mha import Image


@dataclass
class Mesh:
    """What an itk::Mesh<TPixel,3> receives: points (float32), cells (ids), optional cell data."""
    points: np.ndarray
    cells: np.ndarray
    cell_data: np.ndarray | None = None

    def GetNumberOfPoints(self) -> int:
        return int(self.points.shape[0])

    def GetNumberOfCells(self) -> int:
        return int(self.cells.shape[0])


def _clamp(v, lo, hi):
    return lo if v < lo else (hi if v > hi else v)


class LinearInterpolateImageFunction:
    """Marker for the default TInterpolator (h:110): trilinear, what k_project implements."""


class CuberilleImageToMeshFilter:
    def __init__(self, device: int = 0, stream: int | None = None, id_bytes: int = 4):
        self._handle = capi.Handle(device, stream)
        self._image: Image | None = None
        self._output: Mesh | None = None
        self._modified = True
        self._id_bytes = id_bytes
        # constructor defaults, txx:31-41
        self._iso = 1
        self._triangles = True
        self._project = True
        self._cell_data = False
        self._raster_order = False
        self._border_faces = False
        self._projection_method = capi.PROJECT_DEFAULT
        self._inside_range = None   # (lower, upper): range mode instead of the iso value
        self._thr = 0.5
        self._step = -1.0
        self._relax = 0.95
        self._max_steps = 50
        self._interpolator = LinearInterpolateImageFunction()

    @classmethod
    def New(cls, **kw):
        return cls(**kw)

    # -- setters / getters (itkSetMacro / itkGetMacro / itkBooleanMacro, h:180-228) ------------
    def _set(self, name, value):
        if getattr(self, name) != value:
            setattr(self, name, value)
            self._modified = True

    def SetInput(self, image: Image):
        self._image = image
        self._modified = True

    def SetInterpolator(self, interpolator):
        """h:187-188.  The GPU path implements the default trilinear interpolation only
        (LinearInterpolateImageFunction, txx:87-91): anything else is rejected, as in the C++ adapter."""
        if interpolator is not None and not isinstance(interpolator, LinearInterpolateImageFunction):
            raise TypeError("only LinearInterpolateImageFunction is supported by the B200 path")
        self._interpolator = interpolator or LinearInterpolateImageFunction()
        self._modified = True

    def GetInterpolator(self):
        return self._interpolator

    def SetIsoSurfaceValue(self, v): self._set("_iso", v)
    def GetIsoSurfaceValue(self): return self._iso
    def SetGenerateTriangleFaces(self, b): self._set("_triangles", bool(b))
    def GetGenerateTriangleFaces(self): return self._triangles
    def GenerateTriangleFacesOn(self): self.SetGenerateTriangleFaces(True)
    def GenerateTriangleFacesOff(self): self.SetGenerateTriangleFaces(False)
    def SetProjectVerticesToIsoSurface(self, b): self._set("_project", bool(b))
    def GetProjectVerticesToIsoSurface(self): return self._project
    def ProjectVerticesToIsoSurfaceOn(self): self.SetProjectVerticesToIsoSurface(True)
    def ProjectVerticesToIsoSurfaceOff(self): self.SetProjectVerticesToIsoSurface(False)
    def SetSavePixelAsCellData(self, b): self._set("_cell_data", bool(b))
    def GetSavePixelAsCellData(self): return self._cell_data
    def SavePixelAsCellDataOn(self): self.SetSavePixelAsCellData(True)
    def SavePixelAsCellDataOff(self): self.SetSavePixelAsCellData(False)
    # extension: number the vertices in lattice-corner raster order instead of the reference's creation order
    def SetImageBorderFaces(self, b): self._set("_border_faces", bool(b))   # opt-in closed mesh (txx:133 TODO)
    def GetImageBorderFaces(self): return self._border_faces
    # the reference's compile-time alternates USE_ADVANCED_PROJECTION / USE_LINESEARCH_PROJECTION (h:22-23), at run time
    def SetProjectionMethod(self, m): self._set("_projection_method", int(m))
    def GetProjectionMethod(self): return self._projection_method
    def SetRasterVertexOrder(self, b): self._set("_raster_order", bool(b))
    def GetRasterVertexOrder(self): return self._raster_order

    # extension: inside range instead of the iso value (cub_set_inside_range); a label k is the range [k, k].  The
    # projection needs an iso-surface: Update() raises while a range is set and ProjectVerticesToIsoSurface is on.
    def SetInsideRange(self, lower, upper): self._set("_inside_range", (lower, upper))
    def SetLabelValue(self, k): self.SetInsideRange(k, k)
    def InsideRangeOff(self): self._set("_inside_range", None)
    def GetInsideRange(self): return self._inside_range
    def GetInsideRangeLower(self): return None if self._inside_range is None else self._inside_range[0]
    def GetInsideRangeUpper(self): return None if self._inside_range is None else self._inside_range[1]

    def SetProjectVertexSurfaceDistanceThreshold(self, v):
        # itkSetClampMacro(.., 0.0, NumericTraits<InputPixelType>::max())  h:210
        hi = float("inf")
        if self._image is not None:
            dt = self._image.data.dtype
            hi = float(np.iinfo(dt).max) if np.issubdtype(dt, np.integer) else float(np.finfo(dt).max)
        self._set("_thr", _clamp(float(v), 0.0, hi))

    def GetProjectVertexSurfaceDistanceThreshold(self): return self._thr
    def SetProjectVertexStepLength(self, v): self._set("_step", _clamp(float(v), 0.0, 100000.0))  # h:216
    def GetProjectVertexStepLength(self): return self._step
    def SetProjectVertexStepLengthRelaxationFactor(self, v): self._set("_relax", _clamp(float(v), 0.0, 1.0))  # h:223
    def GetProjectVertexStepLengthRelaxationFactor(self): return self._relax
    def SetProjectVertexMaximumNumberOfSteps(self, v): self._set("_max_steps", int(v))
    def GetProjectVertexMaximumNumberOfSteps(self): return self._max_steps

    # -- pipeline ------------------------------------------------------------------------------
    def params(self) -> capi.Params:
        p = capi.default_params()
        p.iso_value = float(self._iso)
        p.generate_triangles = int(self._triangles)
        p.project_vertices = int(self._project)
        p.save_pixel_as_cell_data = int(self._cell_data)
        p.vertex_order = capi.ORDER_RASTER if self._raster_order else capi.ORDER_REFERENCE
        p.image_border_faces = int(self._border_faces)
        p.surface_distance_threshold = self._thr
        p.step_length = self._step
        p.step_relaxation = self._relax
        p.max_steps = self._max_steps
        p.projection_method = self._projection_method
        return p

    def Update(self):
        if not self._modified and self._output is not None:
            return
        if self._image is None:
            raise RuntimeError("Input is not set")  # SetNumberOfRequiredInputs(1), txx:33
        img = self._image
        if self._step < 0.0:
            self._step = max(img.spacing) * 0.25  # sticky, txx:82-85
        self._handle.set_volume(img.data, img.spacing, img.origin, img.direction)
        self._handle.set_region_index(getattr(img, "region_index", (0, 0, 0)))
        if self._inside_range is not None:
            self._handle.set_inside_range(*self._inside_range)
        self._handle.run(self.params(), self._id_bytes)
        pts, cells, cd = self._handle.fetch(self._cell_data)
        self._output = Mesh(pts, cells, cd)
        self._modified = False

    def GetOutput(self) -> Mesh:
        return self._output

    def __str__(self):  # PrintSelf, txx:501-520
        return (f"IsoSurfaceValue: {self._iso}\nGenerateTriangleFaces: {int(self._triangles)}\n"
                f"ProjectVerticesToIsoSurface: {int(self._project)}\n"
                + (f"InsideRange: [{self._inside_range[0]}, {self._inside_range[1]}]\n" if self._inside_range is not None else ""))
