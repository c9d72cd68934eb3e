"""Inside-range mode against iso mode on one GPU: what the second compare costs in the classification kernel, and what a
range saves over binarising the volume first.

Volumes: the 1024^3 float32 gyroid of cub_generate_volume (values in about [-1.5, 1.5], border -2) and a uint8 cast of
it made on the device (60 * v + 128).  K1 is the fused classification + sweep kernel for float32 and the packed
classification kernel for uint8; its time is slot [0] of cub_get_timings (CUDA events around the kernel).

  * K1, iso mode against range mode with the same mask: iso v against [v, type max].  The mesh, and so everything
    the fused kernel's sweep does, is the same, so the difference is the second compare.  A narrow band (two surfaces)
    is reported too.
  * The whole step (count + emit, quads, host clock around work that ends in a synchronise) of range mode on the uint8
    volume against a torch compare that writes a binarised uint8 copy followed by iso mode at 1 on that copy.

Iso and range runs alternate in one process, three runs of --steps timed steps each.  Prints the card name and power
limit with the numbers, and one JSON line.
Usage: python tools/range_bench.py [--size 1024] [--steps 20] [--warmup 3] [--out FILE]"""
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


def k1_ms(h, prm, rng, steps, warmup):
    """mean slot-[0] time over `steps` counts (after `warmup`), with the handle in iso mode (rng None) or range mode"""
    if rng is None:
        h.clear_inside_range()
    else:
        h.set_inside_range(*rng)
    h.enable_timing(True)
    ts = []
    for i in range(warmup + steps):
        h.count(prm)
        if i >= warmup:
            ts.append(h.timings()["classify"])
    h.enable_timing(False)
    return float(np.mean(ts)), h.count(prm)


def step_ms(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    out = []
    for _ in range(steps):
        t0 = time.perf_counter()
        fn()
        out.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=1024)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    S = a.size
    torch.cuda.set_device(0)
    st = torch.cuda.Stream()
    torch.cuda.set_stream(st)
    name, power = card()
    print(f"card: {name}; power limit, max SM clock: {power}")
    gen = P.capi.Handle(0, st.cuda_stream)
    gen.generate(P.capi.GEN_GYROID, (S, S, S), p0=128.0)
    f = torch.from_numpy(gen.download_volume()).cuda()
    gen.close()
    u8 = (f * 60.0 + 128.0).to(torch.uint8)
    torch.cuda.synchronize()
    h = P.capi.Handle(0, st.cuda_stream)
    prm = P.capi.default_params()
    prm.generate_triangles, prm.project_vertices = 0, 0
    res = {"card": name, "power_limit_max_sm_clock": power, "size": S, "k1": {}, "step": {}}

    cases = [
        ("float32", f, np.float32, 0.0, (0.0, float("inf")), (-0.25, 0.25)),
        ("uint8", u8, np.uint8, 128.0, (128.0, 255.0), (113.0, 143.0)),
    ]
    for dname, vol, ndt, iso, same, band in cases:
        h.set_volume_ptr(vol.data_ptr(), ndt, (S, S, S), P.capi.MEM_DEVICE)
        prm.iso_value = iso
        runs = {"iso": [], "range_same_mask": [], "range_band": []}
        for _ in range(a.runs):
            t, n_iso = k1_ms(h, prm, None, a.steps, a.warmup)
            runs["iso"].append(t)
            t, n_same = k1_ms(h, prm, same, a.steps, a.warmup)
            runs["range_same_mask"].append(t)
            assert n_same == n_iso, (dname, n_same, n_iso)
            t, n_band = k1_ms(h, prm, band, a.steps, a.warmup)
            runs["range_band"].append(t)
        fused = h.count_was_fused()
        h.clear_inside_range()
        res["k1"][dname] = {"kernel": "fused classify+sweep" if fused else "classify", "iso": iso, "same_mask_range": same,
                            "band": band, "ms": runs, "quads_iso": n_iso[1], "quads_band": n_band[1]}
        print(f"{dname:8s} K1 ({res['k1'][dname]['kernel']}) ms, runs alternating:  iso {iso:g}: "
              + " ".join(f"{v:.4f}" for v in runs["iso"]) + f" | range {same}: " + " ".join(f"{v:.4f}" for v in runs["range_same_mask"])
              + f" | band {band}: " + " ".join(f"{v:.4f}" for v in runs["range_band"]))

    # whole step on the uint8 volume: range mode against torch binarise + iso 1 on the copy
    lo, hi = 113, 143
    binary = torch.empty_like(u8)

    def range_step():
        h.set_volume_ptr(u8.data_ptr(), np.uint8, (S, S, S), P.capi.MEM_DEVICE)
        h.set_inside_range(lo, hi)
        h.count(prm)
        h.emit(4)
        h.synchronize()

    def binarise_step():
        torch.logical_and(u8 >= lo, u8 <= hi, out=binary.view(torch.bool))
        torch.cuda.synchronize()   # (the handle's stream is torch's current stream; this keeps the two legs alike)
        h.set_volume_ptr(binary.data_ptr(), np.uint8, (S, S, S), P.capi.MEM_DEVICE)
        h.count(prm)
        h.emit(4)
        h.synchronize()

    prm.iso_value = 1.0
    steps = {"range": [], "binarise_then_iso": []}
    for _ in range(a.runs):
        steps["range"].append(step_ms(range_step, a.steps, a.warmup))
        steps["binarise_then_iso"].append(step_ms(binarise_step, a.steps, a.warmup))
    h.set_volume_ptr(u8.data_ptr(), np.uint8, (S, S, S), P.capi.MEM_DEVICE)
    h.set_inside_range(lo, hi)
    h.count(prm)
    h.emit(4)
    pr, cr, _ = h.fetch()
    h.set_volume_ptr(binary.data_ptr(), np.uint8, (S, S, S), P.capi.MEM_DEVICE)
    h.count(prm)
    h.emit(4)
    pb, cb, _ = h.fetch()
    same_mesh = bool(np.array_equal(pr.view(np.uint32), pb.view(np.uint32)) and np.array_equal(cr, cb))
    res["step"] = {"band": [lo, hi], "quads": int(cr.shape[0]), "median_ms": steps, "same_mesh": same_mesh}
    print(f"uint8 step (count + emit quads), medians of runs, alternating: range [{lo}, {hi}]: "
          + " ".join(f"{v:.3f}" for v in steps["range"]) + " | binarise + iso 1: "
          + " ".join(f"{v:.3f}" for v in steps["binarise_then_iso"]) + f" ms; same mesh: {same_mesh}")
    h.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
