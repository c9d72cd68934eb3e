"""Label maps on one GPU: the per-label bounds pass (k_label_bounds) and every label meshed in its box (cub_run_labels)
against the loop of whole-volume range-mode runs it replaces.

Volumes, built on the device with torch from a seed: a 1024^3 label map of 100 balls of radius 4..100 on background 0
(labels 1..100, later balls cover earlier ones), the same map with one more label (101) across the whole x/y extent
(slices 500..507), and an iid-random map (labels 0..100 at every voxel: a run break at nearly every voxel, the
adversarial case of the bounds pass).  Each is benchmarked as uint8 and as uint16 (the same labels).  1 GB and more, so
the passes read HBM, not L2.

  * k_label_bounds: host clock around cub_label_bounds (one memset, the kernel, a 64 * n-byte copy back and a
    synchronise), median of --steps calls, as bytes read per second, against a device-to-device copy of the same bytes
    timed with CUDA events in the same run (reported as bytes read per second; the copy also writes them).
  * cub_run_labels for labels 1..N against the loop inside_range(k, k) + count + set_id_base + emit on the whole
    volume (host clock, each ends in a synchronise); the outputs are compared byte for byte.
  * the fixed cost of a label: cub_run_labels of 100 one-voxel labels, less one bounds pass, per label.
  * sum of the grown, clipped box volumes over the volume.

Prints the card name and power limit with the numbers, and one JSON line.
Usage: python tools/labels_bench.py [--size 1024] [--steps 5] [--warmup 1] [--out FILE]"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.dont_write_bytecode = True
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
P = importlib.import_module("midas-journal-740_b200")


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        q = "unavailable"
    return name, q


def blob_map(n, n_blobs, seed, full_xy=False):
    """int16 label map on the device: n_blobs balls, labels 1..n_blobs in draw order"""
    g = np.random.default_rng(seed)
    vol = torch.zeros((n, n, n), dtype=torch.int16, device="cuda")
    for lab in range(1, n_blobs + 1):
        r = int(g.integers(4, max(5, n * 100 // 1024)))
        c = [int(g.integers(0, n)) for _ in range(3)]
        sl = [slice(max(ci - r, 0), min(ci + r + 1, n)) for ci in c]
        ax = [torch.arange(s.start, s.stop, device="cuda") - ci for s, ci in zip(sl, c)]
        ball = ax[0][:, None, None] ** 2 + ax[1][None, :, None] ** 2 + ax[2][None, None, :] ** 2 <= r * r
        sub = vol[sl[0], sl[1], sl[2]]
        sub[ball] = lab
    if full_xy:
        vol[n // 2 - 12:n // 2 - 4] = n_blobs + 1
    return vol


def timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts))


def copy_ms(src, steps):
    dst = torch.empty_like(src)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    dst.copy_(src)
    ts = []
    for _ in range(steps):
        ev[0].record()
        dst.copy_(src)
        ev[1].record()
        ev[1].synchronize()
        ts.append(ev[0].elapsed_time(ev[1]))
    del dst
    return float(np.median(ts))


def as_dtype(vol16, dtype):
    return vol16.to(torch.uint8) if dtype == np.uint8 else vol16


def set_device_volume(h, t, dtype):
    torch.cuda.synchronize()   # (the handle's stream does not wait for torch's)
    h.set_volume_ptr(t.data_ptr(), dtype, tuple(t.shape[::-1]), P.capi.MEM_DEVICE)


def box_fraction(b, dims):
    present = b[:, 0] > 0
    lo = np.maximum(b[present, 1:4].astype(np.int64) - 1, 0)
    hi = np.minimum(b[present, 4:7].astype(np.int64) + 1, np.array(dims) - 1)
    return float(np.prod(hi - lo + 1, axis=1).sum() / np.prod(dims))


def loop_runs(h, prm, labels):
    """the whole-volume range run of every label with the running id bases"""
    pts, cells = 0, 0
    for k in labels:
        h.set_inside_range(k, k)
        npt, nq = h.count(prm)
        h.set_id_base(pts, cells)
        h.emit(4)
        pts += npt
        cells += 2 * nq if prm.generate_triangles else nq
    h.synchronize()


def loop_mesh(h, prm, labels):
    parts, pts, cells = [], 0, 0
    for k in labels:
        h.set_inside_range(k, k)
        h.count(prm)
        h.set_id_base(pts, cells)
        h.emit(4)
        a, b, c = h.fetch(want_cell_data=bool(prm.save_pixel_as_cell_data))
        parts.append((a, b, c))
        pts += a.shape[0]
        cells += b.shape[0]
    h.clear_inside_range()
    return [np.concatenate([p[i] for p in parts]) for i in range(3 if prm.save_pixel_as_cell_data else 2)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--blobs", type=int, default=100)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("labels_bench needs a CUDA device")
    P.build()
    name, limits = card()
    print(f"card: {name}; power.limit, clocks.max.sm: {limits}", flush=True)
    n, nb = a.size, a.blobs
    voxels = n ** 3
    h = P.capi.Handle(0)
    res = dict(card=name, power_limit_and_max_sm_clock=limits, size=n, blobs=nb, results={})
    maps = {
        "blobs": lambda: blob_map(n, nb, seed=1),
        "blobs_full_xy": lambda: blob_map(n, nb, seed=1, full_xy=True),
        "iid": lambda: torch.randint(0, nb + 1, (n, n, n), dtype=torch.int16, device="cuda",
                                     generator=torch.Generator(device="cuda").manual_seed(7)),
    }
    prm = P.capi.default_params()
    prm.project_vertices, prm.generate_triangles, prm.save_pixel_as_cell_data = 0, 1, 1
    for mname, make in maps.items():
        vol16 = make()
        for dtype in (np.uint8, np.uint16):
            t = as_dtype(vol16, dtype)
            set_device_volume(h, t, dtype)
            n_labels = int(t.max().item()) + 1
            bounds = h.label_bounds(0, n_labels)
            ms = timed(lambda: h.label_bounds(0, n_labels), a.steps, a.warmup)
            cms = copy_ms(t, a.steps)
            nbytes = voxels * np.dtype(dtype).itemsize
            r = dict(bounds_ms=ms, bounds_read_GBps=nbytes / ms / 1e6, copy_ms=cms, copy_read_GBps=nbytes / cms / 1e6,
                     labels=n_labels, box_voxels_over_volume=box_fraction(bounds[1:], (n, n, n)))
            print(f"{mname} {np.dtype(dtype).name}: k_label_bounds {ms:.3f} ms ({r['bounds_read_GBps']:.0f} GB/s read), "
                  f"copy {cms:.3f} ms ({r['copy_read_GBps']:.0f} GB/s read), sum of boxes / volume "
                  f"{r['box_voxels_over_volume']:.4f}", flush=True)
            if mname != "iid":
                labels = list(range(1, n_labels))
                po, co = h.run_labels(prm, labels, 4)
                got = h.fetch(want_cell_data=True)
                want = loop_mesh(h, prm, labels)
                same = all(x.shape == y.shape and np.array_equal(x.view(np.uint8), y.view(np.uint8)) for x, y in zip(got, want))
                t_labels = timed(lambda: h.run_labels(prm, labels, 4), a.steps, a.warmup)
                t_loop = timed(lambda: loop_runs(h, prm, labels), max(1, a.steps // 2), a.warmup)
                r.update(run_labels_ms=t_labels, loop_ms=t_loop, speedup=t_loop / t_labels, identical=bool(same),
                         points=int(po[-1]), cells=int(co[-1]))
                print(f"  run_labels {len(labels)} labels: {t_labels:.1f} ms, loop of whole-volume runs {t_loop:.1f} ms "
                      f"(x{t_loop / t_labels:.1f}), {int(po[-1])} points, {int(co[-1])} cells, identical={same}", flush=True)
                if not same:
                    raise SystemExit("cub_run_labels differs from the whole-volume runs")
            res["results"][f"{mname}_{np.dtype(dtype).name}"] = r
            del t
        del vol16
        torch.cuda.empty_cache()
    # the fixed cost of a label: one-voxel labels spread over the volume
    g = np.random.default_rng(3)
    tiny = torch.zeros((n, n, n), dtype=torch.uint8, device="cuda")
    for k in range(1, nb + 1):
        z, y, x = (int(v) for v in g.integers(0, n, 3))
        tiny[z, y, x] = k
    set_device_volume(h, tiny, np.uint8)
    labels = list(range(1, nb + 1))
    t_tiny = timed(lambda: h.run_labels(prm, labels, 4), a.steps, a.warmup)
    t_b = timed(lambda: h.label_bounds(0, nb + 1), a.steps, a.warmup)
    per_label = (t_tiny - t_b) / nb
    res["fixed_cost"] = dict(run_labels_ms=t_tiny, bounds_ms=t_b, per_label_ms=per_label, labels=nb)
    print(f"fixed cost: run_labels of {nb} one-voxel labels {t_tiny:.2f} ms, bounds pass {t_b:.3f} ms, "
          f"{per_label * 1e3:.0f} us per label", flush=True)
    h.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
