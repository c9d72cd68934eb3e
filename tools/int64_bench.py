"""int64 volumes and label maps on one GPU, against what a caller would otherwise do.

  * the fused classification + sweep kernel (k_fused.cuh) on a 1024^3 int64 gyroid (the float field x 1000, rounded)
    against the same field as float64, the same 8.6 GB: CUDA-event time of the count's first kernel (cub_enable_timing,
    "classify"), median of --steps counts, and the bytes it reads per second.
  * k_label_bounds on the 1024^3 map of 100 balls (tools/labels_bench.py, seed 1) as int64: host clock around
    cub_label_bounds, median of --steps, against a device-to-device copy of the same bytes (CUDA events).
  * cub_run_labels of labels 1..100 on that int64 map against the path a caller without 64-bit support takes: a torch
    cast to int32, then the int32 run (host clock around both, each ending in a synchronise).  Points and cells must be
    byte-identical and the cell data equal as values.

Prints the card name and power limit with the numbers, and one JSON line.
Usage: python tools/int64_bench.py [--size 1024] [--steps 5] [--warmup 1] [--out FILE]"""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.dont_write_bytecode = True
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from labels_bench import P, blob_map, card, copy_ms, set_device_volume, timed  # noqa: E402


def classify_ms(h, prm, steps, warmup):
    h.enable_timing(True)
    for _ in range(warmup):
        h.count(prm)
    ts = []
    for _ in range(steps):
        h.count(prm)
        ts.append(h.timings()["classify"])
    h.enable_timing(False)
    return float(np.median(ts)), h.count_was_fused()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--blobs", type=int, default=100)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("int64_bench needs a CUDA device")
    P.build()
    name, limits = card()
    print(f"card: {name}; power.limit, clocks.max.sm: {limits}", flush=True)
    n = a.size
    voxels = n ** 3
    res = dict(card=name, power_limit_and_max_sm_clock=limits, size=n, blobs=a.blobs)
    h = P.capi.Handle(0)

    # the fused kernel: int64 against float64 of the same size
    z = torch.arange(n, device="cuda", dtype=torch.float32)
    k = 2.0 * np.pi / 128.0
    s, c = torch.sin(k * z), torch.cos(k * z)
    field = (s[None, None, :] * c[None, :, None] + s[None, :, None] * c[:, None, None] + s[:, None, None] * c[None, None, :])
    fused = {}
    for dtype, t in (("int64", torch.round(field * 1000).to(torch.int64)), ("float64", (field * 1000).to(torch.float64))):
        set_device_volume(h, t, np.dtype(dtype))
        prm = P.capi.default_params()
        prm.iso_value, prm.project_vertices = 0.0, 0
        ms, was_fused = classify_ms(h, prm, a.steps, a.warmup)
        fused[dtype] = dict(ms=ms, read_GBps=voxels * 8 / ms / 1e6, fused=was_fused)
        print(f"fused kernel, {dtype} {n}^3: {ms:.3f} ms ({voxels * 8 / ms / 1e6:.0f} GB/s read), fused={was_fused}", flush=True)
        del t
    del field
    torch.cuda.empty_cache()
    res["fused"] = fused

    # the ball map as int64
    t64 = blob_map(n, a.blobs, seed=1).to(torch.int64)
    torch.cuda.empty_cache()
    set_device_volume(h, t64, np.int64)
    n_labels = int(t64.max().item()) + 1
    ms = timed(lambda: h.label_bounds(0, n_labels), a.steps, a.warmup)
    cms = copy_ms(t64, a.steps)
    res["label_bounds"] = dict(ms=ms, read_GBps=voxels * 8 / ms / 1e6, copy_ms=cms, copy_read_GBps=voxels * 8 / cms / 1e6)
    print(f"k_label_bounds int64: {ms:.3f} ms ({voxels * 8 / ms / 1e6:.0f} GB/s read), device copy {cms:.3f} ms "
          f"({voxels * 8 / cms / 1e6:.0f} GB/s read)", flush=True)

    prm = P.capi.default_params()
    prm.project_vertices, prm.generate_triangles, prm.save_pixel_as_cell_data = 0, 1, 1
    labels = list(range(1, n_labels))
    h.run_labels(prm, labels, 4)
    got = h.fetch(want_cell_data=True)
    t_64 = timed(lambda: h.run_labels(prm, labels, 4), a.steps, a.warmup)

    def cast_and_run():
        t32 = t64.to(torch.int32)
        set_device_volume(h, t32, np.int32)
        h.run_labels(prm, labels, 4)
        h.synchronize()
        return t32

    t32 = cast_and_run()
    want = h.fetch(want_cell_data=True)
    del t32
    t_32 = timed(cast_and_run, a.steps, a.warmup)
    same = all(x.shape == y.shape and np.array_equal(x.view(np.uint8), y.view(np.uint8)) for x, y in zip(got[:2], want[:2]))
    same = same and np.array_equal(got[2].astype(np.int64), want[2].astype(np.int64))
    res["run_labels"] = dict(int64_ms=t_64, cast_int32_ms=t_32, speedup=t_32 / t_64, identical=bool(same),
                             labels=len(labels), points=int(got[0].shape[0]), cells=int(got[1].shape[0]))
    print(f"run_labels {len(labels)} labels: int64 {t_64:.1f} ms, torch cast to int32 + int32 run {t_32:.1f} ms "
          f"(x{t_32 / t_64:.2f}), identical={same}", flush=True)
    h.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    if not same:
        raise SystemExit("the int64 label run differs from the int32 run")


if __name__ == "__main__":
    main()
