"""z-slab decomposition of the hot path across ranks (SURVEY §8e).

The reference's GenerateData is one raster loop (txx:136-206); concatenating contiguous z-slabs keeps
its cell order and its first-touch vertex order.  Each rank runs the same kernels on its slab (with a
halo) and the ONLY exchange of the data path is an all-gather of two integers per rank: the exclusive
scan of (points, cells) counts gives the global id bases.  Host logic only - works with any
torch.distributed backend (nccl on GPUs, gloo in the CPU tests).
"""
from __future__ import annotations

from dataclasses import dataclass


@dataclass(frozen=True)
class Slab:
    rank: int
    image_nz: int
    own_z0: int      # global half-open range of slices whose voxels this rank emits
    own_z1: int
    local_z0: int    # global half-open range of slices the rank holds (own range + halo, clipped to the image)
    local_z1: int


def plan_slabs(image_nz: int, world: int, halo: int = 2, z_range: tuple[int, int] | None = None) -> list[Slab]:
    """Contiguous, near-equal z-slabs of the image (or of its slices `z_range`, e.g. a rank's own range cut once
    more); `halo` >= 2 (classification + first-touch ownership of the shared corner plane); when vertices are
    projected use capi.projection_halo(params, spacing, direction) (8 for the default parameters and isotropic voxels:
    cub_count refuses a shorter one)."""
    if halo < 2:
        raise ValueError("the halo must be at least 2 slices")
    a, b = z_range if z_range is not None else (0, image_nz)
    if world < 1 or b - a < world:
        raise ValueError("need at least one slice per rank")
    out = []
    for r in range(world):
        z0, z1 = a + ((b - a) * r) // world, a + ((b - a) * (r + 1)) // world
        out.append(Slab(r, image_nz, z0, z1, max(0, z0 - halo), min(image_nz, z1 + halo)))
    return out


def exclusive_bases(counts: list[tuple[int, int]], rank: int) -> tuple[int, int]:
    """(point id base, cell id base) of `rank` from every rank's (points, cells)."""
    return sum(c[0] for c in counts[:rank]), sum(c[1] for c in counts[:rank])


def all_gather_counts(n_points: int, n_cells: int, device=None, stream=None) -> list[tuple[int, int]]:
    """All-gather of the per-rank (points, cells) counts: NCCL has no exclusive scan, so every rank gathers
    the 2 x world integers and sums its prefix locally.  Single process: no communication.
    `stream`: a side torch stream for the exchange, so that it does not queue behind kernels the caller has
    already launched on the current stream (Handle.emit_vertices runs meanwhile)."""
    import contextlib
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return [(int(n_points), int(n_cells))]
    world = dist.get_world_size()
    ctx = torch.cuda.stream(stream) if stream is not None else contextlib.nullcontext()
    with ctx:
        mine = torch.tensor([n_points, n_cells], dtype=torch.int64, device=device)
        out = torch.empty(2 * world, dtype=torch.int64, device=device)
        dist.all_gather_into_tensor(out, mine)
        flat = out.cpu().tolist()
    return [(flat[2 * r], flat[2 * r + 1]) for r in range(world)]


def create_comm(handle, device=None):
    """A capi.Comm for `handle` over all ranks of the initialised torch.distributed group: rank 0 asks the
    library for an NCCL unique id (cub_comm_unique_id), torch.distributed only carries the 128 bytes, and the
    library creates its own communicator (cub_comm_create).  Returns None in a single-process run."""
    import torch
    import torch.distributed as dist
    from . import capi
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return None
    world, rank = dist.get_world_size(), dist.get_rank()
    on_gpu = dist.get_backend() == "nccl"
    t = torch.zeros(128, dtype=torch.uint8, device=device if on_gpu else None)
    if rank == 0:
        t.copy_(torch.frombuffer(bytearray(capi.comm_unique_id()), dtype=torch.uint8))
    dist.broadcast(t, 0)
    return capi.Comm(handle, bytes(t.cpu().tolist()), world, rank)


def step_async(handle, comm, params, id_bytes: int = 4):
    """One pass of the hot path on this rank's slab with no host round trip: count -> [count exchange over
    NCCL, device to device, beside the vertex stage] -> emit.  The counts stay on the device; read them with
    handle.finish()."""
    handle.count_async(params)
    if comm is not None:
        comm.exchange_counts()
    handle.emit_async(id_bytes)


def gather_mesh(handle, comm, want_cell_data: bool = False):
    """The whole mesh on every rank ("allgatherv" over NVLink, cub_comm_gather_mesh): device tensors
    (points [n, 3] float32, cells [m, k] int32 / int64, cell data or None) whose rows are exactly the
    single-GPU mesh.  Single process: this rank's mesh."""
    import numpy as np
    import torch
    from . import capi
    n_pts, n_cells = handle.finish()
    info = handle.device_buffers()
    k, ib = info["verts_per_cell"], info["id_bytes"]
    dev = torch.device("cuda", torch.cuda.current_device())
    if comm is None:
        tot_p, tot_c = n_pts, n_cells
    else:
        counts = comm.counts()
        cpq = 2 if k == 3 else 1
        tot_p, tot_c = sum(c[0] for c in counts), sum(c[1] for c in counts) * cpq
    pts = torch.empty((max(tot_p, 1), 3), dtype=torch.float32, device=dev)
    cells = torch.empty((max(tot_c, 1), k), dtype=torch.int32 if ib == 4 else torch.int64, device=dev)
    cd = None
    if want_cell_data:
        item = np.dtype(handle.dtype).itemsize
        cd = torch.empty(max(tot_c, 1) * item, dtype=torch.uint8, device=dev)
    if comm is None:
        handle.fetch_into(pts.data_ptr(), cells.data_ptr(), cd.data_ptr() if cd is not None else 0, capi.MEM_DEVICE)
    else:
        comm.gather_mesh(pts.data_ptr(), cells.data_ptr(), cd.data_ptr() if cd is not None else 0)
        handle.synchronize()
    return pts[:tot_p], cells[:tot_c], (cd[:tot_c * np.dtype(handle.dtype).itemsize] if cd is not None else None)


def run_streamed_rank(handles, streams, vol_ptr: int, dtype, dims_xyz, image_nz: int, local_z0: int, own: tuple[int, int],
                      params, out_points_ptr: int, out_cells_ptr: int, device_volume, exchange, id_bytes: int = 4,
                      halo: int = 2, spacing=(1.0, 1.0, 1.0), origin=(0.0, 0.0, 0.0), inside_range=None):
    """One rank of a multi-GPU run, host volume in, host mesh out.  The rank's buffer (pinned, slices
    [local_z0, local_z0 + nz) of the image, its own range `own` plus halo) is copied once, in len(handles)
    consecutive pieces on a copy stream, into `device_volume`; sub-slab c is counted on handles[c] as soon as its
    piece has landed.  The ids of a rank start where the lower ranks end, which is only known when EVERY rank has
    counted, so the run has two phases: (1) upload + count all sub-slabs, exchange(points, quads) -> this rank's
    (point base, quad base) [an all-gather of two integers], (2) emit + copy out sub-slab by sub-slab.
    Outputs: this rank's part of the mesh at the start of its (pinned) output buffers.
    `inside_range`: (lower, upper) meshes that range instead of the iso value (Handle.set_inside_range).
    Returns (n_points, n_cells, point_base, cell_base) of the rank."""
    import ctypes
    import numpy as np
    import torch
    from . import capi
    nx, ny, nz = dims_xyz
    item = np.dtype(dtype).itemsize
    slice_bytes = ny * nx * item
    n_sub = len(handles)
    subs = plan_slabs(image_nz, n_sub, halo, z_range=own)
    verts_per_cell = 3 if params.generate_triangles else 4
    cells_per_quad = 2 if params.generate_triangles else 1
    dev = device_volume.view(torch.uint8).reshape(-1)
    host = torch.from_numpy(np.ctypeslib.as_array((ctypes.c_uint8 * (nz * slice_bytes)).from_address(vol_ptr)))
    copy_stream = _copy_stream(dev.device)
    for st in streams:
        copy_stream.wait_stream(st)
    events, done = [], 0
    with torch.cuda.stream(copy_stream):
        for s in subs:  # piece c ends where sub-slab c's window ends (clipped to the rank's buffer)
            end = min(s.local_z1, local_z0 + nz) - local_z0
            a, b = done * slice_bytes, end * slice_bytes
            if b > a:
                dev[a:b].copy_(host[a:b], non_blocking=True)
            done = max(done, end)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
            events.append(ev)
    # ---- phase 1: count every sub-slab as its piece lands
    for c, (s, h) in enumerate(zip(subs, handles)):
        lo, hi = max(s.local_z0, local_z0), min(s.local_z1, local_z0 + nz)
        streams[c].wait_event(events[c])
        h.set_volume_ptr(device_volume.data_ptr() + (lo - local_z0) * slice_bytes, dtype, (nx, ny, hi - lo), capi.MEM_DEVICE,
                         spacing, origin)
        if inside_range is not None:
            h.set_inside_range(*inside_range)
        h.set_slab(image_nz, lo, s.own_z0, s.own_z1)
        h.count_async(params)
    counts = []
    for h in handles:
        n_pts, n_cells = h.finish()
        counts.append((n_pts, n_cells // cells_per_quad))
    tot_p, tot_q = sum(c[0] for c in counts), sum(c[1] for c in counts)
    pbase0, qbase0 = exchange(tot_p, tot_q)
    # ---- phase 2: emit + copy out
    pb, qb = pbase0, qbase0
    for h, (n_pts, n_quads) in zip(handles, counts):
        h.set_id_base(pb, qb * cells_per_quad)
        h.emit(id_bytes)
        h.fetch_into(out_points_ptr + (pb - pbase0) * 12, out_cells_ptr + (qb - qbase0) * cells_per_quad * verts_per_cell * id_bytes,
                     0, capi.MEM_HOST, sync=False)
        pb += n_pts
        qb += n_quads
    for h in handles:
        h.synchronize()
    return tot_p, tot_q * cells_per_quad, pbase0, qbase0 * cells_per_quad


def run_streamed(handles, vol_ptr: int, dtype, dims_xyz, params, n_slabs: int, out_points_ptr: int, out_cells_ptr: int,
                 id_bytes: int = 4, halo: int = 2, spacing=(1.0, 1.0, 1.0), origin=(0.0, 0.0, 0.0),
                 device_volume=None, streams=None, inside_range=None):
    """One GPU, host volume in, host mesh out, streamed: the image is cut into `n_slabs` z-slabs that travel
    through `handles` (>= 2 capi.Handle objects, each on its own stream) round-robin, so the host->device copy
    of slab c+1, the kernels of slab c and the device->host copy of slab c-1 overlap.  Ids are global: the id
    base of a slab is the running sum of the counts of the slabs before it (the same exclusive scan the
    multi-GPU path gets from its all-gather).  `vol_ptr` / `out_*_ptr`: pinned host memory; the outputs must
    be large enough for the whole mesh.  Returns (n_points, n_cells).

    Two ways for the volume to travel:
    * default: every handle copies its slab *with* its halo slices into its own buffer (cub_set_volume with
      CUB_MEM_HOST); works for volumes larger than the device memory, re-sends 2 * halo slices per cut;
    * `device_volume` (a torch uint8 CUDA tensor of the volume's size) + `streams` (the torch streams the
      handles were created on): the volume is copied once, in n_slabs consecutive pieces on a copy stream, into
      that buffer and the handles borrow windows of it (CUB_MEM_DEVICE); nothing is sent twice.

    `inside_range`: (lower, upper) meshes that range instead of the iso value (Handle.set_inside_range)."""
    import numpy as np
    from . import capi
    nx, ny, nz = dims_xyz
    item = np.dtype(dtype).itemsize
    slice_bytes = ny * nx * item
    slabs = plan_slabs(nz, n_slabs, halo)
    verts_per_cell = 3 if params.generate_triangles else 4
    cells_per_quad = 2 if params.generate_triangles else 1
    pbase = cbase = 0
    resident = device_volume is not None
    events = []
    if resident:
        import ctypes
        import torch
        assert streams is not None and len(streams) == len(handles), "resident mode needs the handles' torch streams"
        assert device_volume.is_cuda and device_volume.numel() * device_volume.element_size() >= nz * slice_bytes
        dev = device_volume.view(torch.uint8).reshape(-1)
        host = torch.from_numpy(np.ctypeslib.as_array((ctypes.c_uint8 * (nz * slice_bytes)).from_address(vol_ptr)))
        copy_stream = _copy_stream(dev.device)
        for st in streams:
            copy_stream.wait_stream(st)  # earlier work on the handles may still read the buffer
        done = 0
        with torch.cuda.stream(copy_stream):
            for s in slabs:  # piece c ends where slab c's window ends: after it, slab c has all it reads
                a, b = done * slice_bytes, s.local_z1 * slice_bytes
                if b > a:
                    dev[a:b].copy_(host[a:b], non_blocking=True)
                done = max(done, s.local_z1)
                ev = torch.cuda.Event()
                ev.record(copy_stream)
                events.append(ev)

    def upload(c):
        s, h = slabs[c], handles[c % len(handles)]
        if resident:
            streams[c % len(handles)].wait_event(events[c])
            h.set_volume_ptr(device_volume.data_ptr() + s.local_z0 * slice_bytes, dtype, (nx, ny, s.local_z1 - s.local_z0),
                             capi.MEM_DEVICE, spacing, origin)
        else:
            h.set_volume_ptr(vol_ptr + s.local_z0 * slice_bytes, dtype, (nx, ny, s.local_z1 - s.local_z0), capi.MEM_HOST,
                             spacing, origin)
        if inside_range is not None:
            h.set_inside_range(*inside_range)
        h.set_slab(nz, s.local_z0, s.own_z0, s.own_z1)

    upload(0)
    for c in range(n_slabs):
        h = handles[c % len(handles)]
        if c + 1 < n_slabs:
            upload(c + 1)             # queued on the next handle's stream before this slab's count blocks the host
        n_pts, n_quads = h.count(params)
        h.set_id_base(pbase, cbase)
        h.emit(id_bytes)
        h.fetch_into(out_points_ptr + pbase * 12, out_cells_ptr + cbase * verts_per_cell * id_bytes, 0, capi.MEM_HOST,
                     sync=False)
        pbase += n_pts
        cbase += n_quads * cells_per_quad
    for h in handles:
        h.synchronize()
    return pbase, cbase


_COPY_STREAMS = {}


def _copy_stream(device):
    import torch
    key = (device.type, device.index)
    if key not in _COPY_STREAMS:
        _COPY_STREAMS[key] = torch.cuda.Stream(device=device)
    return _COPY_STREAMS[key]
