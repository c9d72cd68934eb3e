"""ctypes binding of include/cuberille_c.h (libcuberille_cuda.so).

There is no fallback: if the shared library is missing or no CUDA device is usable the
calls raise.  Nothing in this package imports oracle/.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _build

U8, I8, U16, I16, U32, I32, F32, F64, I64, U64 = range(10)
MEM_HOST, MEM_DEVICE = 0, 1
GEN_GYROID, GEN_MARSCHNER_LOBB, GEN_BLOBS = 0, 1, 2
ORDER_REFERENCE, ORDER_RASTER = 0, 1
PROJECT_DEFAULT, PROJECT_ADVANCED, PROJECT_LINESEARCH = 0, 1, 2

DTYPE_CODES = {
    np.dtype(np.uint8): U8, np.dtype(np.int8): I8, np.dtype(np.uint16): U16, np.dtype(np.int16): I16,
    np.dtype(np.uint32): U32, np.dtype(np.int32): I32, np.dtype(np.float32): F32, np.dtype(np.float64): F64,
    np.dtype(np.int64): I64, np.dtype(np.uint64): U64,
}
CODE_DTYPES = {v: k for k, v in DTYPE_CODES.items()}

# every symbol include/cuberille_c.h declares (tests check that the library exports all of them)
SYMBOLS = [
    "cub_abi_version", "cub_default_params", "cub_create", "cub_destroy", "cub_last_error", "cub_set_volume",
    "cub_set_region_index", "cub_set_inside_range", "cub_set_slab", "cub_label_bounds", "cub_set_region_of_interest",
    "cub_run_labels", "cub_count", "cub_set_id_base", "cub_emit_vertices", "cub_emit", "cub_run", "cub_fetch", "cub_fetch_async",
    "cub_synchronize", "cub_device_buffers",
    "cub_debug_bitmask", "cub_debug_project_points", "cub_generate_volume", "cub_download_volume",
    "cub_enable_timing", "cub_get_timings", "cub_launch_count", "cub_count_was_fused",
    "cub_projection_halo", "cub_projection_halo_oriented", "cub_count_async", "cub_device_counts", "cub_emit_async", "cub_finish", "cub_last_warning",
    "cub_comm_unique_id", "cub_comm_create", "cub_comm_destroy", "cub_comm_exchange_counts", "cub_comm_counts",
    "cub_comm_gather_mesh", "cub_device_alloc", "cub_device_free", "cub_device_copy",
    "cub_host_register", "cub_host_unregister", "cub_host_alloc", "cub_host_free",
]


class Params(C.Structure):
    _fields_ = [
        ("iso_value", C.c_double),
        ("generate_triangles", C.c_int32),
        ("project_vertices", C.c_int32),
        ("save_pixel_as_cell_data", C.c_int32),
        ("vertex_order", C.c_int32),
        ("surface_distance_threshold", C.c_double),
        ("step_length", C.c_double),
        ("step_relaxation", C.c_double),
        ("max_steps", C.c_uint32),
        ("image_border_faces", C.c_uint32),
        ("projection_method", C.c_int32),
        ("reserved", C.c_int32),
    ]


def pixel_value(v) -> float:
    """A pixel value (iso value, range bound, label) as the double the C-ABI takes.  Python and numpy integers beyond
    2^53 may have no such double; rounding would silently put a neighbouring value in their place, so they raise."""
    if isinstance(v, (int, np.integer)) and not isinstance(v, bool):
        d = float(int(v))
        if int(d) != int(v):
            raise ValueError(f"pixel value {int(v)} is not exactly representable as a double")
        return d
    return float(v)


class CuberilleError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"cuberille C-ABI error {code}: {msg}")
        self.code = code


_lib = None


def lib_path() -> str:
    return _build.LIB


def load() -> C.CDLL:
    """Load libcuberille_cuda.so (must have been built: __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_build.LIB):
        raise FileNotFoundError(f"{_build.LIB} is missing: run `python -c 'import __graft_entry__ as g; g.build()'`")
    L = C.CDLL(_build.LIB)
    vp, u64, i = C.c_void_p, C.c_uint64, C.c_int
    pu64, pd = C.POINTER(C.c_uint64), C.POINTER(C.c_double)
    L.cub_abi_version.restype = i
    L.cub_default_params.restype = None
    L.cub_default_params.argtypes = [C.POINTER(Params)]
    L.cub_create.restype = i
    L.cub_create.argtypes = [i, vp, C.POINTER(vp)]
    L.cub_destroy.restype = i
    L.cub_destroy.argtypes = [vp]
    L.cub_last_error.restype = C.c_char_p
    L.cub_last_error.argtypes = [vp]
    L.cub_set_volume.restype = i
    L.cub_set_volume.argtypes = [vp, vp, i, pu64, pd, pd, pd, i]
    L.cub_set_region_index.restype = i
    L.cub_set_region_index.argtypes = [vp, C.POINTER(C.c_int64)]
    L.cub_set_inside_range.restype = i
    L.cub_set_inside_range.argtypes = [vp, i, C.c_double, C.c_double]
    L.cub_set_slab.restype = i
    L.cub_set_slab.argtypes = [vp, u64, u64, u64, u64]
    L.cub_label_bounds.restype = i
    L.cub_label_bounds.argtypes = [vp, C.c_int64, C.c_uint32, pu64]
    L.cub_set_region_of_interest.restype = i
    L.cub_set_region_of_interest.argtypes = [vp, pu64, pu64]
    L.cub_run_labels.restype = i
    L.cub_run_labels.argtypes = [vp, C.POINTER(Params), pd, u64, i, pu64, pu64]
    L.cub_count.restype = i
    L.cub_count.argtypes = [vp, C.POINTER(Params), pu64, pu64]
    L.cub_set_id_base.restype = i
    L.cub_set_id_base.argtypes = [vp, u64, u64]
    L.cub_emit.restype = i
    L.cub_emit_vertices.restype = i
    L.cub_emit_vertices.argtypes = [vp]
    L.cub_emit.argtypes = [vp, i]
    L.cub_run.restype = i
    L.cub_run.argtypes = [vp, C.POINTER(Params), i, pu64, pu64]
    L.cub_fetch.restype = i
    L.cub_fetch.argtypes = [vp, vp, vp, vp, i]
    L.cub_fetch_async.restype = i
    L.cub_fetch_async.argtypes = [vp, vp, vp, vp, i]
    L.cub_synchronize.restype = i
    L.cub_synchronize.argtypes = [vp]
    L.cub_device_buffers.restype = i
    L.cub_device_buffers.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), pu64, pu64, C.POINTER(i), C.POINTER(i)]
    L.cub_debug_bitmask.restype = i
    L.cub_debug_bitmask.argtypes = [vp, vp, pu64]
    L.cub_debug_project_points.restype = i
    L.cub_debug_project_points.argtypes = [vp, C.POINTER(Params), vp, u64]
    L.cub_generate_volume.restype = i
    L.cub_generate_volume.argtypes = [vp, i, pu64, pu64, u64, C.c_double, C.c_double, u64]
    L.cub_download_volume.restype = i
    L.cub_download_volume.argtypes = [vp, vp, u64]
    L.cub_enable_timing.restype = i
    L.cub_enable_timing.argtypes = [vp, i]
    L.cub_get_timings.restype = i
    L.cub_get_timings.argtypes = [vp, C.POINTER(C.c_float)]
    L.cub_launch_count.restype = u64
    L.cub_launch_count.argtypes = [vp]
    L.cub_count_was_fused.restype = i
    L.cub_count_was_fused.argtypes = [vp]
    L.cub_projection_halo.restype = i
    L.cub_projection_halo.argtypes = [C.POINTER(Params), pd, pu64, pu64]
    L.cub_projection_halo_oriented.restype = i
    L.cub_projection_halo_oriented.argtypes = [C.POINTER(Params), pd, pd, pu64, pu64]
    L.cub_count_async.restype = i
    L.cub_count_async.argtypes = [vp, C.POINTER(Params)]
    L.cub_device_counts.restype = i
    L.cub_device_counts.argtypes = [vp, C.POINTER(vp)]
    L.cub_emit_async.restype = i
    L.cub_emit_async.argtypes = [vp, i]
    L.cub_finish.restype = i
    L.cub_finish.argtypes = [vp, pu64, pu64]
    L.cub_last_warning.restype = C.c_char_p
    L.cub_last_warning.argtypes = [vp]
    L.cub_device_alloc.restype = i
    L.cub_device_alloc.argtypes = [vp, u64, C.POINTER(vp)]
    L.cub_device_free.restype = i
    L.cub_device_free.argtypes = [vp, vp]
    L.cub_device_copy.restype = i
    L.cub_device_copy.argtypes = [vp, vp, vp, u64, i, i]
    L.cub_host_register.restype = i
    L.cub_host_register.argtypes = [vp, vp, u64]
    L.cub_host_unregister.restype = i
    L.cub_host_unregister.argtypes = [vp, vp]
    L.cub_host_alloc.restype = i
    L.cub_host_alloc.argtypes = [vp, u64, C.POINTER(vp)]
    L.cub_host_free.restype = i
    L.cub_host_free.argtypes = [vp, vp]
    L.cub_comm_unique_id.restype = i
    L.cub_comm_unique_id.argtypes = [vp]
    L.cub_comm_create.restype = i
    L.cub_comm_create.argtypes = [vp, vp, i, i, C.POINTER(vp)]
    L.cub_comm_destroy.restype = i
    L.cub_comm_destroy.argtypes = [vp]
    L.cub_comm_exchange_counts.restype = i
    L.cub_comm_exchange_counts.argtypes = [vp]
    L.cub_comm_counts.restype = i
    L.cub_comm_counts.argtypes = [vp, pu64]
    L.cub_comm_gather_mesh.restype = i
    L.cub_comm_gather_mesh.argtypes = [vp, vp, vp, vp]
    _lib = L
    return L


def projection_halo(params: Params, spacing=(1.0, 1.0, 1.0), direction=None) -> tuple[int, int]:
    """Halo slices (below, above) a z-slab of an image with this spacing and direction needs for these parameters
    (cub_projection_halo_oriented)."""
    lo, hi = C.c_uint64(), C.c_uint64()
    dr = (C.c_double * 9)(*direction) if direction is not None else None
    rc = load().cub_projection_halo_oriented(C.byref(params), (C.c_double * 3)(*spacing), dr, C.byref(lo), C.byref(hi))
    if rc != 0:
        raise CuberilleError(rc, "cub_projection_halo_oriented: bad spacing or direction")
    return lo.value, hi.value


def default_params() -> Params:
    p = Params()
    load().cub_default_params(C.byref(p))
    return p


class Handle:
    """One cub_handle: a device, a stream, the scratch and result buffers."""

    def __init__(self, device: int = 0, stream: int | None = None):
        self._L = load()
        self._h = C.c_void_p()
        rc = self._L.cub_create(int(device), C.c_void_p(stream) if stream else None, C.byref(self._h))
        if rc != 0:
            raise CuberilleError(rc, "cub_create failed (no usable CUDA device?)")
        self._keep = None
        self.dtype = None
        self.dims = None
        self._whole_dims = None   # the volume's dims while a region of interest is set (self.dims: the box)

    def close(self):
        if self._h:
            self._L.cub_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != 0:
            raise CuberilleError(rc, self._L.cub_last_error(self._h).decode())

    # -- input -------------------------------------------------------------------------------
    def set_volume(self, vol: np.ndarray, spacing=(1.0, 1.0, 1.0), origin=(0.0, 0.0, 0.0), direction=None):
        """Host volume indexed [z, y, x]; copied to the device."""
        assert vol.ndim == 3
        vol = np.ascontiguousarray(vol)
        self._keep = vol
        dims = (C.c_uint64 * 3)(vol.shape[2], vol.shape[1], vol.shape[0])
        sp = (C.c_double * 3)(*spacing)
        og = (C.c_double * 3)(*origin)
        dr = (C.c_double * 9)(*direction) if direction is not None else None
        self._check(self._L.cub_set_volume(self._h, vol.ctypes.data, DTYPE_CODES[vol.dtype], dims, sp, og, dr, MEM_HOST))
        self.dtype, self.dims, self._whole_dims = vol.dtype, (vol.shape[2], vol.shape[1], vol.shape[0]), None

    def set_volume_ptr(self, ptr: int, dtype, dims_xyz, mem_kind, spacing=(1.0, 1.0, 1.0), origin=(0.0, 0.0, 0.0)):
        """Raw pointer (host pinned or device) with dims (x, y, z)."""
        dims = (C.c_uint64 * 3)(*dims_xyz)
        sp = (C.c_double * 3)(*spacing)
        og = (C.c_double * 3)(*origin)
        self._check(self._L.cub_set_volume(self._h, C.c_void_p(ptr), DTYPE_CODES[np.dtype(dtype)], dims, sp, og, None, mem_kind))
        self.dtype, self.dims, self._whole_dims = np.dtype(dtype), tuple(dims_xyz), None

    def set_region_index(self, index_xyz):
        """Image index of the buffer's first voxel (after set_volume, which resets it to 0)."""
        self._check(self._L.cub_set_region_index(self._h, (C.c_int64 * 3)(*[int(v) for v in index_xyz])))

    def set_inside_range(self, lower, upper):
        """Range mode: a voxel is inside when lower <= v <= upper in the pixel type (NaN pixels too), instead of
        v >= iso.  Both bounds must be pixel values of the volume's type; a label k is (k, k).  Projection is refused
        while the mode is on.  After set_volume, which turns the mode off."""
        self._check(self._L.cub_set_inside_range(self._h, 1, pixel_value(lower), pixel_value(upper)))

    def clear_inside_range(self):
        """Back to iso mode."""
        self._check(self._L.cub_set_inside_range(self._h, 0, 0.0, 0.0))

    def label_bounds(self, first: int, n: int) -> np.ndarray:
        """(n, 8) uint64: {count, xmin, ymin, zmin, xmax, ymax, zmax, 0} of the labels first .. first + n - 1 of the
        current integer volume (buffer indices, inclusive maxima; all zero for an absent label)."""
        out = np.zeros((int(n), 8), np.uint64)
        self._check(self._L.cub_label_bounds(self._h, int(first), int(n), out.ctypes.data_as(C.POINTER(C.c_uint64))))
        return out

    def set_region_of_interest(self, lo_xyz, size_xyz):
        """Count on the box [lo, lo + size) of the current volume, as on a copy of it with the region index moved by lo."""
        self._check(self._L.cub_set_region_of_interest(self._h, (C.c_uint64 * 3)(*[int(v) for v in lo_xyz]),
                                                       (C.c_uint64 * 3)(*[int(v) for v in size_xyz])))
        self._whole_dims = self._whole_dims or self.dims
        self.dims = tuple(int(v) for v in size_xyz)

    def clear_region_of_interest(self):
        self._check(self._L.cub_set_region_of_interest(self._h, None, None))
        self.dims, self._whole_dims = self._whole_dims or self.dims, None

    def run_labels(self, params: Params, labels, id_bytes: int = 4):
        """Mesh every label as the range [k, k], concatenated in the given order; returns (point_offsets, cell_offsets),
        n_labels + 1 entries each.  Read the mesh with fetch() / device_buffers()."""
        lab = np.array([pixel_value(k) for k in np.asarray(labels).reshape(-1).tolist()], np.float64)
        po = np.zeros(lab.size + 1, np.uint64)
        co = np.zeros(lab.size + 1, np.uint64)
        self._check(self._L.cub_run_labels(self._h, C.byref(params), lab.ctypes.data_as(C.POINTER(C.c_double)), lab.size,
                                           id_bytes, po.ctypes.data_as(C.POINTER(C.c_uint64)),
                                           co.ctypes.data_as(C.POINTER(C.c_uint64))))
        return po, co

    def set_slab(self, image_nz: int, local_z0: int, own_z0: int, own_z1: int):
        self._check(self._L.cub_set_slab(self._h, image_nz, local_z0, own_z0, own_z1))

    def generate(self, kind: int, dims_xyz, image_dims_xyz=None, z_offset: int = 0, p0: float = 128.0, p1: float = 1.0,
                 seed: int = 1234):
        image_dims_xyz = image_dims_xyz or dims_xyz
        d = (C.c_uint64 * 3)(*dims_xyz)
        im = (C.c_uint64 * 3)(*image_dims_xyz)
        self._check(self._L.cub_generate_volume(self._h, kind, d, im, z_offset, p0, p1, seed))
        self.dtype, self.dims, self._whole_dims = np.dtype(np.float32), tuple(dims_xyz), None

    def download_volume(self) -> np.ndarray:
        x, y, z = self.dims
        out = np.empty((z, y, x), self.dtype)
        self._check(self._L.cub_download_volume(self._h, out.ctypes.data, out.nbytes))
        return out

    # -- run ---------------------------------------------------------------------------------
    def count(self, params: Params):
        npts, nq = C.c_uint64(), C.c_uint64()
        self._check(self._L.cub_count(self._h, C.byref(params), C.byref(npts), C.byref(nq)))
        return npts.value, nq.value

    def count_async(self, params: Params):
        """Queue phase 1 without waiting for the counts (they stay on the device)."""
        self._check(self._L.cub_count_async(self._h, C.byref(params)))

    def emit_async(self, id_bytes: int = 4):
        self._check(self._L.cub_emit_async(self._h, id_bytes))

    def finish(self):
        """Synchronise; returns (n_points, n_cells) of the queued run."""
        npts, nc = C.c_uint64(), C.c_uint64()
        self._check(self._L.cub_finish(self._h, C.byref(npts), C.byref(nc)))
        return npts.value, nc.value

    def device_counts_ptr(self) -> int:
        p = C.c_void_p()
        self._check(self._L.cub_device_counts(self._h, C.byref(p)))
        return p.value

    def last_warning(self) -> str:
        return self._L.cub_last_warning(self._h).decode()

    def set_id_base(self, point_base: int, cell_base: int):
        self._check(self._L.cub_set_id_base(self._h, point_base, cell_base))

    def emit_vertices(self):
        """Queue the vertex stage now (before the id base is known); emit() then only emits the cells."""
        self._check(self._L.cub_emit_vertices(self._h))

    def emit(self, id_bytes: int = 4):
        self._check(self._L.cub_emit(self._h, id_bytes))

    def run(self, params: Params, id_bytes: int = 4):
        npts, nc = C.c_uint64(), C.c_uint64()
        self._check(self._L.cub_run(self._h, C.byref(params), id_bytes, C.byref(npts), C.byref(nc)))
        return npts.value, nc.value

    def device_buffers(self):
        p, c, d = C.c_void_p(), C.c_void_p(), C.c_void_p()
        npts, nc, k, ib = C.c_uint64(), C.c_uint64(), C.c_int(), C.c_int()
        self._check(self._L.cub_device_buffers(self._h, C.byref(p), C.byref(c), C.byref(d), C.byref(npts), C.byref(nc),
                                               C.byref(k), C.byref(ib)))
        return dict(points=p.value, cells=c.value, cell_data=d.value, n_points=npts.value, n_cells=nc.value,
                    verts_per_cell=k.value, id_bytes=ib.value)

    def fetch(self, want_cell_data: bool = False):
        info = self.device_buffers()
        n, m, k, ib = info["n_points"], info["n_cells"], info["verts_per_cell"], info["id_bytes"]
        pts = np.empty((n, 3), np.float32)
        cells = np.empty((m, k), np.uint32 if ib == 4 else np.uint64)
        cd = np.empty(m, self.dtype) if want_cell_data else None
        self._check(self._L.cub_fetch(self._h, pts.ctypes.data, cells.ctypes.data,
                                      cd.ctypes.data if cd is not None else None, MEM_HOST))
        return pts, cells, cd

    def synchronize(self):
        self._check(self._L.cub_synchronize(self._h))

    def fetch_into(self, points_ptr: int, cells_ptr: int, cell_data_ptr: int = 0, mem_kind: int = MEM_HOST, sync: bool = True):
        fn = self._L.cub_fetch if sync else self._L.cub_fetch_async
        self._check(fn(self._h, C.c_void_p(points_ptr) if points_ptr else None,
                                      C.c_void_p(cells_ptr) if cells_ptr else None,
                                      C.c_void_p(cell_data_ptr) if cell_data_ptr else None, mem_kind))

    # -- diagnostics -------------------------------------------------------------------------
    def bitmask(self) -> np.ndarray:
        wpr = C.c_uint64()
        self._check(self._L.cub_debug_bitmask(self._h, None, C.byref(wpr)))
        x, y, z = self.dims
        out = np.empty((z, y, wpr.value), np.uint32)
        self._check(self._L.cub_debug_bitmask(self._h, out.ctypes.data, C.byref(wpr)))
        return out

    def project_points(self, params: Params, pts: np.ndarray) -> np.ndarray:
        out = np.ascontiguousarray(pts, np.float32).copy()
        self._check(self._L.cub_debug_project_points(self._h, C.byref(params), out.ctypes.data, out.shape[0]))
        return out

    def enable_timing(self, on: bool = True):
        self._check(self._L.cub_enable_timing(self._h, int(on)))

    def timings(self) -> dict:
        ms = (C.c_float * 8)()
        self._check(self._L.cub_get_timings(self._h, ms))
        names = ["classify", "count_scan", "emit", "project", "split", "count_phase", "emit_phase", "scan_only"]
        return {n: float(v) for n, v in zip(names, ms)}

    def launch_count(self) -> int:
        return int(self._L.cub_launch_count(self._h))

    def count_was_fused(self) -> bool:
        """True if the last count ran classification + sweep as the one fused kernel (k_fused.cuh)."""
        return bool(self._L.cub_count_was_fused(self._h))


def comm_unique_id() -> bytes:
    """ncclGetUniqueId through the C-ABI (rank 0 calls it, the host distributes the 128 bytes)."""
    buf = (C.c_ubyte * 128)()
    rc = load().cub_comm_unique_id(buf)
    if rc != 0:
        raise CuberilleError(rc, "cub_comm_unique_id failed (is libnccl.so.2 loadable?)")
    return bytes(buf)


class Comm:
    """One cub_comm: binds a Handle to its rank of an NCCL communicator created by the library."""

    def __init__(self, handle: Handle, unique_id: bytes, world: int, rank: int):
        self._L, self._handle = handle._L, handle
        self._c = C.c_void_p()
        self.world, self.rank = world, rank
        buf = (C.c_ubyte * 128).from_buffer_copy(unique_id)
        handle._check(self._L.cub_comm_create(handle._h, buf, world, rank, C.byref(self._c)))

    def close(self):
        if self._c:
            self._L.cub_comm_destroy(self._c)
            self._c = C.c_void_p()

    def exchange_counts(self):
        """Queue the all-gather of the counts + the device-side prefix that becomes the id bases."""
        self._handle._check(self._L.cub_comm_exchange_counts(self._c))

    def counts(self) -> list[tuple[int, int]]:
        out = (C.c_uint64 * (2 * self.world))()
        self._handle._check(self._L.cub_comm_counts(self._c, out))
        return [(int(out[2 * r]), int(out[2 * r + 1])) for r in range(self.world)]

    def gather_mesh(self, points_ptr: int, cells_ptr: int, cell_data_ptr: int = 0):
        self._handle._check(self._L.cub_comm_gather_mesh(self._c, C.c_void_p(points_ptr) if points_ptr else None,
                                                         C.c_void_p(cells_ptr) if cells_ptr else None,
                                                         C.c_void_p(cell_data_ptr) if cell_data_ptr else None))
