"""Throughput of `evaluate-segmentation` on the device: DeviceChunk.evaluate (contingency table in one pass over both label
volumes, reduction to exact sums, scores) on three workloads that bound it from different sides, each with uint32 and uint64
labels:

    realistic      connected components of a smooth thresholded field at two thresholds, one as seg and one as gt
    one_label      one label everywhere: every voxel updates the same table entry (worst contention)
    random         a random label per voxel on both sides: one table entry per voxel (worst table size)

Per call: ms (host clock around a synchronised call, after a warm-up call), table entries, and the label-read bound --
n * (bytes_seg + bytes_gt) over the HBM bandwidth measured in the same run with a device-to-device copy -- with the
fraction of it the call reaches.  The volumes (>= 1 GB) exceed the 126 MB L2.  One JSON line.

    python tools/bench_evaluate.py [--size 512] [--reps 5] [--cpu]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from chunkflow_b200.chunk.device import DeviceChunk  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = (v.strip() for v in out.split(","))
        return name, power
    except Exception:
        return torch.cuda.get_device_name(0), "unknown"


def hbm_copy_gbs(reps=10):
    """Best device-to-device copy rate of a 4 GiB buffer: bytes read + written per second."""
    a = torch.empty(1 << 32, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    best = float("inf")
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        b.copy_(a)
        torch.cuda.synchronize()
        best = min(best, time.perf_counter() - t0)
    del a, b
    return 2 * (1 << 32) / best / 1e9


def blobs(n, threshold, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    f = torch.randn((1, 1, n, n, n), device="cuda", generator=g)
    k = torch.ones((1, 1, 5, 5, 5), device="cuda") / 125
    for _ in range(3):
        f = torch.nn.functional.conv3d(f, k, padding=2)
    f = (f[0, 0] / f.std()).contiguous()
    return DeviceChunk(f).connected_component(threshold=threshold).tensor.view(torch.int32)


def workloads(n, wide):
    dt = torch.int64 if wide else torch.int32
    seg, gt = blobs(n, 0.2, 1), blobs(n, 0.6, 2)
    yield "realistic", seg.to(dt), gt.to(dt)
    del seg, gt
    ones = torch.ones((n, n, n), dtype=dt, device="cuda")
    yield "one_label", ones, ones
    del ones
    g = torch.Generator(device="cuda").manual_seed(3)
    hi = 2 ** 62 if wide else 2 ** 31 - 1
    yield "random", torch.randint(0, hi, (n, n, n), dtype=dt, device="cuda", generator=g), \
        torch.randint(0, hi, (n, n, n), dtype=dt, device="cuda", generator=g)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--cpu", action="store_true", help="also time the numpy oracle on the same inputs")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_evaluate: no CUDA device")
    n = args.size
    name, power = card()
    peak = hbm_copy_gbs()
    result = {"operator": "evaluate-segmentation", "volume": f"{n}^3", "device": name, "power_limit": power,
              "hbm_copy_gbs_measured": round(peak, 1),
              "timing": "host wall clock around synchronised DeviceChunk.evaluate calls, after one warm-up call",
              "workloads": []}
    for wide in (False, True):
        for label, s, g in workloads(n, wide):
            seg, gt = DeviceChunk(s, layer_type="segmentation"), DeviceChunk(g, layer_type="segmentation")
            seg.evaluate(gt)
            torch.cuda.synchronize()
            times = []
            for _ in range(args.reps):
                t0 = time.perf_counter()
                scores = seg.evaluate(gt)
                torch.cuda.synchronize()
                times.append((time.perf_counter() - t0) * 1e3)
            work, _, entries, voxels = seg._contingency(gt)
            del work
            ms = float(np.median(times))
            nbytes = voxels * (s.element_size() + g.element_size())
            bound_ms = nbytes / (peak * 1e9) * 1e3
            row = {"workload": label, "labels": "uint64" if wide else "uint32", "ms": round(ms, 3), "ms_min": round(min(times), 3),
                   "table_entries": int(entries), "label_bytes": int(nbytes), "label_read_bound_ms": round(bound_ms, 3),
                   "fraction_of_bound": round(bound_ms / ms, 3),
                   "scores": {k: (list(map(float, v)) if isinstance(v, tuple) else float(v)) for k, v in scores.items()}}
            if args.cpu:
                from oracle import evaluation_oracle as O
                a = s.cpu().numpy().view(np.uint64 if wide else np.uint32)
                b = g.cpu().numpy().view(np.uint64 if wide else np.uint32)
                t0 = time.perf_counter()
                O.evaluate(a, b)
                row["oracle_cpu_ms"] = round((time.perf_counter() - t0) * 1e3, 1)
            result["workloads"].append(row)
            del seg, gt, s, g
            torch.cuda.empty_cache()
    print(json.dumps(result))


if __name__ == "__main__":
    main()
