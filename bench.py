#!/usr/bin/env python
"""bench.py — headline benchmark of the cuberille hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--size S] [--period P] [--dump-outputs DIR]

One "step" = one pass of the hot path through the C-ABI (cub_count_async -> [count exchange] ->
cub_emit_async: classify -> ownership sweep -> segment scan -> vertices -> faces) over a synthetic
float32 gyroid that is already resident in HBM; the counts stay on the device, so a step has no host
round trip.  N > 1 (launched by torchrun, one rank per GPU): BASELINE.json's configuration, the ONE
1024^3 gyroid split into z-slabs with a 2-slice halo (strong scaling); every rank runs the same kernels
on its slab and the only exchange of the data path is an NCCL all-gather of the per-rank (points,
quads) counts, device to device, whose prefix gives the global ids (cub_comm_exchange_counts).  The
mesh all-gather over NVLink (cub_comm_gather_mesh) and the weak-scaling run (1024^3 per GPU) are timed
separately (`gather`, `extras.weak`).  Rank 0 prints ONE JSON line.

`--impl reference` times the CPU restatement of the reference filter (oracle/, single-threaded like
GenerateData itself) on a bounded sample of the same workload.

`--dump-outputs DIR` writes the mesh of the last timed step to DIR/*.npy (see dump_outputs); the
volume is generated on the device from the arguments alone, so two builds can be compared file for file.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True  # the tree this runs from may be read-only: nothing is written there
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--size", type=int, default=1024, help="voxels per axis per GPU")
    ap.add_argument("--period", type=float, default=128.0, help="gyroid period in voxels")
    ap.add_argument("--field", default="gyroid", choices=["gyroid", "marschner_lobb", "blobs"])
    ap.add_argument("--scaling", default="strong", choices=["weak", "strong"])
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target CPU time of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-gather", action="store_true", help="skip the all-gather of the meshes (N > 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the mesh of the last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 0:
        ap.error("--warmup must not be negative")
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs applies to --impl cuda (the reference's sample size depends on the host's speed)")
    return args


FIELD_KIND = {"gyroid": 0, "marschner_lobb": 1, "blobs": 2}
FIELD_ISO = {"gyroid": 0.0, "marschner_lobb": 0.5, "blobs": 0.5}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        busy = [s for s in sm if s > 0.5 * max(mx or [1])] or sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def oracle_sample_rate(vol, iso, triangles, project, params):
    import oracle_py as O
    t = time.perf_counter()
    m = O.cuberille(vol, iso, triangles=triangles, project=project, mode=O.LITERAL, **params)
    dt = time.perf_counter() - t
    return dt, m


def cpu_baseline_from_volume(get_slab, nx, ny, nz_max, iso, seconds):
    """time the oracle on a bounded z-sample of the workload: calibrate on 8 slices, then size the
    sample for about `seconds` of CPU work."""
    vol = get_slab(8)
    dt, _ = oracle_sample_rate(vol, iso, False, False, {})
    rate = vol.size / max(dt, 1e-6)
    nz = int(min(nz_max, max(8, seconds * rate / (nx * ny))))
    vol = get_slab(nz)
    dt, m = oracle_sample_rate(vol, iso, False, False, {})
    return {"value": vol.size / dt / 1e9, "unit": "Gvoxels/s", "cores": 1, "kind": "port",
            "sample": f"{nx}x{ny}x{nz} z-sub-slab of the same volume (same bytes, downloaded from the GPU), "
                      f"quads, no projection, {dt:.2f} s, {m.cells.shape[0]} quads",
            "mfaces_per_s": m.cells.shape[0] / dt / 1e6, "seconds": dt,
            "host_cores_available": os.cpu_count()}


def run_reference(args):
    """the reference's own CPU implementation of the path (the oracle port: ITK is not installable here,
    DESIGN.md §6), single-threaded like GenerateData (txx:136-206), on a bounded sample."""
    import numpy as np
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle_py as O
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    S = args.size
    # same field as the CUDA arm, generated on the host (numpy float32); the sample is a z-sub-slab
    k = np.float32(2.0 * np.pi / args.period)

    def slab(nz):
        z, y, x = np.meshgrid(np.arange(nz, dtype=np.float32), np.arange(S, dtype=np.float32), np.arange(S, dtype=np.float32),
                              indexing="ij")
        g = (np.sin(k * x) * np.cos(k * y) + np.sin(k * y) * np.cos(k * z) + np.sin(k * z) * np.cos(k * x)).astype(np.float32)
        g[0] = -2; g[-1] = -2; g[:, 0] = -2; g[:, -1] = -2; g[:, :, 0] = -2; g[:, :, -1] = -2
        return np.ascontiguousarray(g)

    cal = slab(8)
    dt, _ = oracle_sample_rate(cal, 0.0, False, False, {})
    rate = cal.size / max(dt, 1e-6)
    per_step = max(2.0, min(20.0, 120.0 / max(1, args.steps + args.warmup)))
    nz = int(min(S, max(8, per_step * rate / (S * S))))
    vol = slab(nz)
    times, faces = [], 0
    for i in range(args.warmup + args.steps):
        dt, m = oracle_sample_rate(vol, 0.0, False, False, {})
        faces = m.cells.shape[0]
        if i >= args.warmup:
            times.append(dt)
    t = sum(times) / len(times)
    v = vol.size / t / 1e9
    # Beside it, not instead of it: what every host core gives when each runs its own single-threaded instance on a
    # z-sub-slab (something the reference does not do: GenerateData is one sequential loop, txx:136-206).  The
    # oracle is a C++ library behind ctypes, which drops the GIL for the call.
    all_cores = None
    try:
        from concurrent.futures import ThreadPoolExecutor
        cores = len(os.sched_getaffinity(0))
        sub = vol[:max(8, nz // 4)]
        t0 = time.perf_counter()
        with ThreadPoolExecutor(cores) as ex:
            list(ex.map(lambda _: oracle_sample_rate(sub, 0.0, False, False, {})[0], range(cores)))
        wall = time.perf_counter() - t0
        all_cores = {"value": cores * sub.size / wall / 1e9, "unit": "Gvoxels/s", "cores": cores,
                     "note": f"{cores} independent single-threaded instances at once, each on a {S}x{S}x{sub.shape[0]} sub-slab"}
    except Exception as e:
        all_cores = {"unavailable": str(e)[:120]}
    line = {
        "impl": "reference", "metric": "Gvoxels/s", "value": v, "unit": "Gvoxels/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, args.gpus),
        "mfaces_per_s": faces / t / 1e6,
        "cpu_baseline": {"value": v, "unit": "Gvoxels/s", "cores": 1, "kind": "port",
                         "sample": f"{S}x{S}x{nz} z-sub-slab of the gyroid per step (CPU restatement of txx:59-498, "
                                   f"single-threaded like the reference; ITK itself is not installable offline)",
                         "host_cores_available": os.cpu_count(), "all_cores": all_cores},
        "e2e": {"value": v, "unit": "Gvoxels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def workload_config(args, n, scaling=None):
    S = args.size
    scaling = scaling or args.scaling
    nz = S * n if scaling == "weak" else S
    return {"workload": f"synthetic {args.field} {S}x{S}x{nz} float32"
                        + (f" period {args.period:g} voxels" if args.field == "gyroid" else "")
                        + f", iso {FIELD_ISO[args.field]}, quads, no projection, uint32 ids"
                        + (f", z-slabs over {n} GPUs (2-slice halo)" if n > 1 else ""),
            "voxels": S * S * nz, "l2_policy": "inputs larger than L2 (4.3 GB volume vs 126 MB L2), no flush needed"
            if S * S * (nz // n) * 4 > 4 * 126e6 else "per-GPU slab comparable to L2: the volume buffer is re-generated (overwritten) between "
            "timed regions only; every step still reads its slab from HBM after the previous step's 2+ GB of scratch and mesh traffic"}


# rows of the points and of the cells that --dump-outputs writes, over all ranks: at most 12 + 4 * 8 bytes a row
# (a float32 point, a quad's ids as float64), 46 MB in all
DUMP_ROWS = 1 << 20


def dump_outputs(out_dir, capi, h, dev, rank, n_ranks):
    """Write the mesh the last step left in the handle, as a caller fetches it, to out_dir: `points` [n, 3] float32,
    `cells` [m, k] vertex ids (float64, exact below 2**53) and `counts` (n, m).  A mesh of more than
    DUMP_ROWS / n_ranks rows is sampled: the rows are seeded and sorted, so the same counts give the same rows.
    With several ranks every rank writes its own part (ids global), with a `_rank<r>` suffix."""
    import numpy as np
    import torch
    info = h.device_buffers()
    n, m, k = info["n_points"], info["n_cells"], info["verts_per_cell"]
    pts = torch.empty((max(n, 1), 3), dtype=torch.float32, device=dev)
    cells = torch.empty((max(m, 1), k), dtype=torch.int32 if info["id_bytes"] == 4 else torch.int64, device=dev)
    h.fetch_into(pts.data_ptr(), cells.data_ptr(), 0, capi.MEM_DEVICE)
    rows = DUMP_ROWS // n_ranks

    def sample(t, total, seed):
        if total <= rows:
            return t[:total].cpu().numpy()
        idx = np.sort(np.random.default_rng(seed).choice(total, rows, replace=False))
        return t.index_select(0, torch.from_numpy(idx).to(dev)).cpu().numpy()

    suffix = f"_rank{rank}" if n_ranks > 1 else ""
    cell_ids = sample(cells, m, 2)
    if cell_ids.dtype == np.int32:
        cell_ids = cell_ids.view(np.uint32)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, f"points{suffix}.npy"), sample(pts, n, 1))
    np.save(os.path.join(out_dir, f"cells{suffix}.npy"), cell_ids.astype(np.float64))
    np.save(os.path.join(out_dir, f"counts{suffix}.npy"), np.array([n, m], np.float64))
    del pts, cells
    torch.cuda.empty_cache()


def bind_to_gpu_numa_node(local_rank):
    """Run this rank (and allocate its pinned buffers: first touch) on the NUMA node its GPU hangs off."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id
        dom = torch.cuda.get_device_properties(local_rank).pci_domain_id
        devn = torch.cuda.get_device_properties(local_rank).pci_device_id
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{devn:02x}.0/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.extend(range(int(a), int(b or a) + 1))
        allowed = sorted(set(cpus) & os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
        return node
    except Exception:
        return None


class Rank:
    """One rank's state for one workload: handle, slab, communicator."""

    def __init__(self, P, args, dev, local_rank, stream, N, rank, scaling, field=None, size=None, halo=2):
        capi = P.capi
        self.P, self.N, self.rank, self.dev = P, N, rank, dev
        self.h = capi.Handle(local_rank, stream.cuda_stream)
        S = size or args.size
        field = field or args.field
        self.S, self.field = S, field
        self.image_nz = S * N if scaling == "weak" else S
        slab = P.slabs.plan_slabs(self.image_nz, N, halo=halo)[rank]
        self.own0, self.own1, self.lo, self.hi = slab.own_z0, slab.own_z1, slab.local_z0, slab.local_z1
        kind = FIELD_KIND[field]
        p0, p1 = (args.period, 1.0) if field == "gyroid" else ((48.0, 1.0) if field == "blobs" else (0.0, 0.0))
        self.h.generate(kind, (S, S, self.hi - self.lo), (S, S, self.image_nz), self.lo, p0, p1)
        if N > 1:
            self.h.set_slab(self.image_nz, self.lo, self.own0, self.own1)
        self.iso = FIELD_ISO[field]
        self.comm = P.slabs.create_comm(self.h, dev) if N > 1 else None

    def params(self, triangles=0, project=0, raster=False, thr=None):
        prm = self.P.capi.default_params()
        prm.iso_value, prm.generate_triangles, prm.project_vertices = self.iso, triangles, project
        if raster:
            prm.vertex_order = self.P.capi.ORDER_RASTER
        if thr is not None:
            prm.surface_distance_threshold = thr
        return prm

    def step(self, prm, handle=None):
        self.P.slabs.step_async(handle or self.h, self.comm if handle is None else None, prm, 4)

    def totals(self):
        """(own points, own quads, total points, total quads) of the last step (synchronises)."""
        n_pts, n_cells = self.h.finish()
        n_quads = n_cells // (2 if self.h.device_buffers()["verts_per_cell"] == 3 else 1)
        if self.comm is None:
            return n_pts, n_quads, n_pts, n_quads
        counts = self.comm.counts()
        return n_pts, n_quads, sum(c[0] for c in counts), sum(c[1] for c in counts)

    def close(self):
        if self.comm is not None:
            self.comm.close()
        self.h.close()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the hot path has no CPU fallback)")
    numa_node = bind_to_gpu_numa_node(local_rank)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    N = world

    P = importlib.import_module("midas-journal-740_b200")
    capi = P.capi
    # a real (non-default) stream: torch's default stream has handle 0, which the C-ABI reads as "create your
    # own stream" - and then torch events would not bracket the library's work
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0

    def barrier():
        if N > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, handle=None):
        for _ in range(warmup):
            fn()
        barrier()
        l0 = handle.launch_count() if handle else 0
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if N > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) / steps, (handle.launch_count() - l0) if handle else 0

    def sum_ranks(v):
        t = torch.tensor([v], dtype=torch.int64, device=dev)
        if N > 1:
            dist.all_reduce(t)
        return int(t.item())

    S = args.size
    R = Rank(P, args, dev, local_rank, stream, N, rank, args.scaling)
    h = R.h
    prm = R.params()
    own0, own1, lo, hi = R.own0, R.own1, R.lo, R.hi

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_step, launches = timed(lambda: R.step(prm), args.steps, args.warmup, h)
    clocks = sampler.stop() if rank == 0 else None
    n_pts, n_quads, tot_p, tot_q = R.totals()
    tot = (tot_p, tot_q)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, capi, h, dev, rank, N)

    voxels_total = sum_ranks(S * S * (own1 - own0))
    gvox = voxels_total / (ms_step * 1e-3) / 1e9
    mfaces = tot[1] / (ms_step * 1e-3) / 1e6

    peak, peak_src = measured_peaks()

    # ---- per-kernel device times (CUDA events inside the library, separate passes) ---------------
    h.enable_timing(True)
    kt = {"classify": [], "count_scan": [], "scan_only": [], "emit": []}
    for _ in range(max(3, min(args.steps, 10))):
        h.count(prm)
        if R.comm is not None:
            R.comm.exchange_counts()
        h.emit(4)
        t = h.timings()
        for k in kt:
            kt[k].append(t[k])
    h.enable_timing(False)
    kavg = {k: sum(v) / len(v) for k, v in kt.items()}
    own_vox = S * S * (own1 - own0)
    local_vox = S * S * (hi - lo)
    alg_k1 = local_vox * 4  # K1 reads every voxel of the local buffer once
    fused = h.count_was_fused()  # K1 + K2a ran as one kernel: "classify" is that kernel, "count_scan" the scan alone
    k1_gbs = alg_k1 / (max(kavg["classify"], 1e-6) * 1e-3) / 1e9
    alg_pipe = own_vox * 4 + n_pts * 12 + n_quads * 16
    cc_ms = kavg["classify"] + kavg["count_scan"]
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            traffic = json.load(f).get("k_classify_sweep_dram_bytes_per_launch" if fused else "k_classify_dram_bytes_per_launch")
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": "k_classify_sweep<float> (classification + ownership sweep, fused)" if fused else "k_classify<float>",
                "achieved": k1_gbs, "peak": peak, "unit": "GB/s",
                "frac": k1_gbs / peak, "traffic": traffic if N == 1 and S == 1024 else None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_k1, "avg_launch_ms": kavg["classify"],
                # the same launch against the bytes it actually moves (ncu dram__bytes of one launch, profiles/traffic.json):
                # the fused kernel also writes the sweep's intermediates, which the algorithmic figure does not count
                "traffic_frac": (traffic / (kavg["classify"] * 1e-3) / 1e9 / peak) if (traffic and N == 1 and S == 1024 and kavg["classify"] > 0) else None,
                "kernel_ms": kavg,
                "classify_plus_compact": {"ms": cc_ms, "achieved": alg_k1 / (cc_ms * 1e-3) / 1e9,
                                          "frac_input_only": alg_k1 / (cc_ms * 1e-3) / 1e9 / peak,
                                          "note": "K1 + K2a + K2b (classification + compaction) against the input bytes: north_star target >= 0.60"},
                "pipeline": {"algorithmic_bytes_per_step": alg_pipe, "achieved": alg_pipe / (ms_step * 1e-3) / 1e9,
                             "frac": alg_pipe / (ms_step * 1e-3) / 1e9 / peak,
                             "input_only_frac": own_vox * 4 / (ms_step * 1e-3) / 1e9 / peak}}

    # ---- extras -------------------------------------------------------------------------------------
    extras = {}
    if not args.no_extras:
        prm1 = R.params(raster=True)
        ms1, _ = timed(lambda: R.step(prm1), max(3, args.steps // 2), 2)
        _, _, _, q1 = R.totals()
        extras["raster_vertex_order"] = {"ms_per_step": ms1, "gvoxels_per_s": voxels_total / (ms1 * 1e-3) / 1e9,
                                         "mfaces_per_s": q1 / (ms1 * 1e-3) / 1e6,
                                         "note": "CUB_ORDER_RASTER: same mesh up to vertex renumbering (canonical ordering)"}
        # the old step with its host round trip between count and emit (cub_count + cub_emit), for comparison
        def sync_step():
            a, b = h.count(prm)
            if R.comm is not None:
                R.comm.exchange_counts()
            h.emit(4)
        ms_sync, _ = timed(sync_step, max(3, args.steps // 2), 2)
        extras["synchronous_api"] = {"ms_per_step": ms_sync, "note": "cub_count (returns the counts to the host) + cub_emit"}

    # the full default filter (triangles + projection) needs the projection halo: its own slabs
    if not args.no_extras:
        prm2 = R.params(triangles=1, project=1, thr=0.01 if args.field == "gyroid" else 0.005)
        halo2 = max(capi.projection_halo(prm2))
        R2 = R if N == 1 else None
        if N > 1:
            R.close()
            R = None
            R2 = Rank(P, args, dev, local_rank, stream, N, rank, args.scaling, halo=halo2)
        ms2, _ = timed(lambda: R2.step(prm2), max(2, args.steps // 3), 1)
        np2, nq2, tp2, tq2 = R2.totals()
        R2.h.enable_timing(True)
        R2.h.count(prm2)
        if R2.comm is not None:
            R2.comm.exchange_counts()
        R2.h.emit(4)
        t2 = R2.h.timings()
        R2.h.enable_timing(False)
        extras["triangles_projection"] = {"ms_per_step": ms2, "gvoxels_per_s": voxels_total / (ms2 * 1e-3) / 1e9,
                                          "mtriangles_per_s": 2 * tq2 / (ms2 * 1e-3) / 1e6,
                                          "mvertices_per_s_project_kernel": np2 / (t2["project"] * 1e-3) / 1e6 if t2["project"] else None,
                                          "kernel_ms": t2, "threshold": prm2.surface_distance_threshold, "halo": halo2}
        if N > 1:
            R2.close()
            R = Rank(P, args, dev, local_rank, stream, N, rank, args.scaling)
        h = R.h

    # ---- the mesh all-gather over NVLink (reported separately, SURVEY section 8e) --------------------------
    gather = None
    if N > 1 and not args.no_gather:
        R.step(prm)
        R.totals()
        pts_all, cells_all, _ = P.slabs.gather_mesh(h, R.comm)   # allocates + first gather (warm-up)

        def gstep():
            R.comm.gather_mesh(pts_all.data_ptr(), cells_all.data_ptr(), 0)
        ms_g, _ = timed(gstep, 5, 1)
        gbytes = int(pts_all.numel() * 4 + cells_all.numel() * 4)
        gather = {"ms": ms_g, "mesh_bytes": gbytes, "recv_gb_per_s_per_gpu": gbytes * (N - 1) / N / (ms_g * 1e-3) / 1e9,
                  "collective": "cub_comm_gather_mesh: grouped ncclSend/ncclRecv with the true counts, every part lands at its id base",
                  "n_points": int(pts_all.shape[0]), "n_cells": int(cells_all.shape[0])}
        del pts_all, cells_all

    # ---- e2e: host volume in, host mesh out, through the public call sequence ----------------------
    e2e = None
    if not args.no_e2e:
        vol_host = torch.empty((hi - lo, S, S), dtype=torch.float32, pin_memory=True)
        h._check(h._L.cub_download_volume(h._h, vol_host.data_ptr(), vol_host.numel() * 4))
        R.step(prm)
        n_pts, n_quads, _, _ = R.totals()
        pts_host = torch.empty((max(n_pts, 1) + 1024, 3), dtype=torch.float32, pin_memory=True)
        cells_host = torch.empty((max(n_quads, 1) + 1024, 4), dtype=torch.int32, pin_memory=True)
        n_sub = max(2, 16 // N)
        sts = [torch.cuda.Stream() for _ in range(min(3, n_sub) if N == 1 else n_sub)]
        hs = [capi.Handle(local_rank, st.cuda_stream) for st in sts]
        vol_dev = torch.empty(vol_host.numel() * 4, dtype=torch.uint8, device=dev)
        # achieved host -> device bandwidth with all ranks copying at once (the ceiling of the e2e number)
        def h2d_only():
            vol_dev.copy_(vol_host.view(torch.uint8).reshape(-1), non_blocking=True)
        ms_h2d, _ = timed(h2d_only, 3, 1)
        h2d_gbs = vol_host.numel() * 4 / (ms_h2d * 1e-3) / 1e9

        if N == 1:
            # streamed: the volume travels through 3 handles (3 streams) as 16 z-slabs, so the PCIe copies in both
            # directions and the kernels overlap (slabs.run_streamed: the same public calls, ids stay global).
            # The volume fits in HBM beside its mesh, so it is copied once (16 consecutive pieces on a copy stream)
            # into a device buffer and the handles borrow windows of it: no halo slice crosses PCIe twice.
            def e2e_streamed():
                a, b = P.slabs.run_streamed(hs, vol_host.data_ptr(), np.float32, (S, S, hi - lo), prm, 16,
                                            pts_host.data_ptr(), cells_host.data_ptr(), device_volume=vol_dev, streams=sts)
                assert (a, b) == (n_pts, n_quads)
            mode = "streamed: volume copied once in 16 pieces, 16 z-slabs through 3 handles / streams borrow windows of it"
        else:
            gl = torch.zeros(2 * N, dtype=torch.int64, device=dev)

            def exchange(tp, tq):
                mine = torch.tensor([tp, tq], dtype=torch.int64, device=dev)
                dist.all_gather_into_tensor(gl, mine)
                flat = gl.cpu().tolist()
                return sum(flat[0:2 * rank:2]), sum(flat[1:2 * rank:2])

            def e2e_streamed():
                a, b, _, _ = P.slabs.run_streamed_rank(hs, sts, vol_host.data_ptr(), np.float32, (S, S, hi - lo), R.image_nz, lo,
                                                       (own0, own1), prm, pts_host.data_ptr(), cells_host.data_ptr(), vol_dev, exchange)
                assert (a, b) == (n_pts, n_quads), (a, b, n_pts, n_quads)
            mode = (f"per rank: slab copied once in {n_sub} pieces, {n_sub} sub-slabs counted as they land, one all-gather of the rank "
                    f"totals, then emit + copy out (slabs.run_streamed_rank)")
        ms_s, _ = timed(e2e_streamed, max(2, min(args.steps, 5)), 1)
        h2d_total = sum_ranks(int(vol_host.numel() * 4))
        d2h_total = sum_ranks(int(n_pts * 12 + n_quads * 16))
        e2e = {"value": voxels_total / (ms_s * 1e-3) / 1e9, "unit": "Gvoxels/s", "ms_per_step": ms_s,
               "h2d_bytes_per_step": h2d_total, "d2h_bytes_per_step": d2h_total, "mfaces_per_s": tot[1] / (ms_s * 1e-3) / 1e6,
               "mode": mode, "h2d_gb_per_s_per_rank_all_ranks_copying": h2d_gbs,
               "h2d_gb_per_s_aggregate": h2d_gbs * N, "pcie_floor_ms": ms_h2d, "numa_node": numa_node}
        for x in hs:
            x.close()
        del vol_dev, vol_host

    # ---- cpu baseline (rank 0, N == 1 only) ---------------------------------------------------------
    cpu = None
    if rank == 0 and N == 1 and not args.no_cpu_baseline:
        full = None

        def get_slab(nz):
            nonlocal full
            if full is None:
                full = h.download_volume()
            z0 = (full.shape[0] - nz) // 2
            v = np.ascontiguousarray(full[z0:z0 + nz])
            return v
        cpu = cpu_baseline_from_volume(get_slab, S, S, hi - lo, R.iso, args.cpu_seconds)
    R.close()

    # ---- the drop-in itself: Update() of the C++ adapter (tests/cpp/cuberille_test01.cxx DropInBench) ---
    if rank == 0 and N == 1 and not args.no_extras:
        exe = os.path.join(ROOT, "tests", "cpp", "CuberilleTest01")
        try:
            if not os.path.exists(exe):
                subprocess.check_call(["make", "-C", os.path.dirname(exe), "-s", "CuberilleTest01"])
            runs = []
            for a in (("512", "0", "0", "0"), ("512", "1", "1", "0")):
                out = subprocess.run([exe, "DropInBench", *a], capture_output=True, text=True, timeout=300)
                runs.append(json.loads(out.stdout.strip().splitlines()[-1]))
            extras["cpp_adapter"] = {"runs": runs, "note": "itk::CuberilleImageToMeshFilter::Update() of include/itkCuberilleImageToMeshFilter.h on a "
                                     "512^3 uint8 volume (pageable itk::Image buffer in, itk::Mesh out; tests/itk_shim stands in for ITK): host -> device "
                                     "copy, kernels, device -> host copy into page-locked staging, itk::Mesh fill (one heap cell per face, txx:310-329)"}
        except Exception as e:  # the C++ driver is optional for the bench line
            extras["cpp_adapter"] = {"unavailable": str(e)[:200]}

    # ---- other workloads of BASELINE.json, where the driver can see them ------------------------------
    if not args.no_extras:
        if N == 1 and args.field == "gyroid" and S >= 512:
            # config 3: Marschner-Lobb 512^3, single B200
            Rm = Rank(P, args, dev, local_rank, stream, 1, 0, "strong", field="marschner_lobb", size=512)
            pm = Rm.params()
            msm, _ = timed(lambda: Rm.step(pm), max(5, args.steps), 3)
            _, _, pp, qq = Rm.totals()
            extras["marschner_lobb_512"] = {"ms_per_step": msm, "gvoxels_per_s": 512 ** 3 / (msm * 1e-3) / 1e9,
                                            "mfaces_per_s": qq / (msm * 1e-3) / 1e6, "n_points": pp, "n_quads": qq}
            Rm.close()
        if N > 1 and args.scaling == "strong":
            # weak scaling: S^3 voxels per GPU, image S x S x (S*N)
            Rw = Rank(P, args, dev, local_rank, stream, N, rank, "weak")
            pw = Rw.params()
            msw, _ = timed(lambda: Rw.step(pw), max(3, args.steps // 2), 2)
            _, _, pp, qq = Rw.totals()
            extras["weak"] = {"ms_per_step": msw, "gvoxels_per_s": S * S * S * N / (msw * 1e-3) / 1e9, "mfaces_per_s": qq / (msw * 1e-3) / 1e6,
                              "config": workload_config(args, N, "weak"), "n_points": pp, "n_quads": qq}
            Rw.close()
            # config 5: sphere blobs with triangles + projection (halo from cub_projection_halo), 1024^3 per GPU
            prb = capi.default_params()
            prb.iso_value, prb.generate_triangles, prb.project_vertices, prb.surface_distance_threshold = 0.5, 1, 1, 0.005
            Rb = Rank(P, args, dev, local_rank, stream, N, rank, "weak", field="blobs", halo=max(capi.projection_halo(prb)))
            msb, _ = timed(lambda: Rb.step(prb), 3, 1)
            _, _, pp, qq = Rb.totals()
            extras["blobs_projection"] = {"ms_per_step": msb, "gvoxels_per_s": S * S * S * N / (msb * 1e-3) / 1e9,
                                          "mtriangles_per_s": 2 * qq / (msb * 1e-3) / 1e6, "n_points": pp, "n_triangles": 2 * qq,
                                          "workload": f"sphere blobs {S}x{S}x{S * N} float32, triangles + projection, halo {max(capi.projection_halo(prb))}"}
            Rb.close()

    if rank == 0:
        line = {
            "metric": "Gvoxels/s", "value": gvox, "unit": "Gvoxels/s", "n_gpus": N, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args, N),
            "mfaces_per_s": mfaces, "n_points": tot[0], "n_quads": tot[1],
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches),
            "clocks": clocks, "extras": extras,
        }
        if gather:
            line["gather"] = gather
        print(json.dumps(line), flush=True)
    if N > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    # stdout carries exactly ONE line, the JSON result: anything a library prints there meanwhile (NCCL's version
    # banner, for one) is sent to stderr instead
    sys.stdout.flush()
    _stdout_fd = os.dup(1)
    os.dup2(2, 1)
    _result = sys.stdout = os.fdopen(_stdout_fd, "w")
    try:
        main()
    finally:
        _result.flush()
