#!/usr/bin/env python
"""Benchmark of the `inference` hot path (BASELINE.json metric: Mvoxels/s for the 3-channel
affinity U-Net on a 1024^3 uint8 chunk at 1/2/4/8 B200).

    python bench.py --gpus N --steps K --warmup W          # this repo's CUDA path
    python bench.py --impl reference --gpus N ...           # the reference algorithm on the host CPUs

A "step" is one pass of the hot path over one synthetic chunk per GPU (weak scaling: one
independent chunk per rank, no data-path collective).  Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
MODEL_FILE = os.path.join(ROOT, "chunkflow_b200", "convnet", "unet3l.py")

WORKLOADS = {
    # name: (chunk zyx, patch, overlap)   -- BASELINE.json configs #3/#4 and #2
    "1024": ((1024, 1024, 1024), (32, 256, 256), (8, 64, 64)),
    "512": ((512, 512, 512), (20, 256, 256), (4, 64, 64)),
    "256": ((256, 512, 512), (32, 256, 256), (8, 64, 64)),   # quick functional check, not a bench line
}
FLOP_PER_PATCH_VOXEL = 141248  # SURVEY.md section 7.2
CONV3_FLOP = {  # per full-resolution patch voxel, 3x3x3 layers only (by kernel class name)
    "enc0.0": 864, "enc0.2": 13824, "enc1.0": 27648 / 4, "enc1.2": 55296 / 4, "enc2.0": 110592 / 16,
    "enc2.2": 221184 / 16, "dec1.0": 110592 / 4, "dec1.2": 55296 / 4, "dec0.0": 27648, "dec0.2": 13824,
    "dec0.2+head+blend": 13824 + 96,  # last conv with the fused 1x1x1 head + sigmoid + mask + blend epilogue
}


DUMP_SEED = 20260922
DUMP_VOXELS = 1 << 21   # spatial positions sampled for --dump-outputs: C x 2^21 float32 (24 MB for 3 channels)


def dump_outputs(directory, out):
    """Writes the affinity map a caller of the timed path receives, as float32 .npy files under `directory`:
    affinity_voxels.npy  (C, 2^21): every channel at a fixed, seeded, sorted set of flat zyx positions (drawn with
                         replacement from np.random.default_rng(DUMP_SEED), so it depends only on the output shape)
    affinity_plane.npy   (C, Y, X): the whole z plane in the middle of the chunk (every patch seam in y and x).
    `out` is a (C, Z, Y, X) float32 torch tensor (on the GPU: only the sample leaves the device) or numpy array."""
    os.makedirs(directory, exist_ok=True)
    c, z = out.shape[0], out.shape[1]
    idx = np.sort(np.random.default_rng(DUMP_SEED).integers(0, int(np.prod(out.shape[1:])), DUMP_VOXELS))
    if isinstance(out, np.ndarray):
        voxels, plane = out.reshape(c, -1)[:, idx], out[:, z // 2]
    else:
        import torch
        voxels = out.reshape(c, -1)[:, torch.from_numpy(idx).to(out.device)].cpu().numpy()
        plane = out[:, z // 2].cpu().numpy()
    np.save(os.path.join(directory, "affinity_voxels.npy"), np.ascontiguousarray(voxels, dtype=np.float32))
    np.save(os.path.join(directory, "affinity_plane.npy"), np.ascontiguousarray(plane, dtype=np.float32))


def patch_count(chunk, patch, overlap):
    n = 1
    for c, p, o in zip(chunk, patch, overlap):
        n *= len(range(0, c - o, p - o))
    return n


def synthetic_chunk(shape, seed, pinned=True):
    """uint8 chunk from np.random.default_rng(20260922 + k) (SURVEY.md section 8d)."""
    import torch
    rng = np.random.default_rng(seed)
    if pinned and torch.cuda.is_available():
        t = torch.empty(shape, dtype=torch.uint8, pin_memory=True)
        a = t.numpy()
    else:
        t, a = None, np.empty(shape, np.uint8)
    for z in range(0, shape[0], 64):  # slab-wise to bound temporary memory
        a[z:z + 64] = rng.integers(0, 256, size=a[z:z + 64].shape, dtype=np.uint8)
    return t, a


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()

    def run(self):
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=5)
        sm, smax, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); smax = max(smax, float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def host_threads():
    """Physical cores this process may use (SMT siblings oversubscribe the torch-CPU convolutions: the round-1 number
    swung 3x between two identical boxes with os.cpu_count() threads)."""
    n = os.cpu_count() or 1
    try:
        import psutil
        n = psutil.cpu_count(logical=False) or n
    except Exception:
        n = max(1, n // 2)
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    return max(1, n)


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.lower().startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


class CpuReference:
    """The reference algorithm on the host cores (oracle port: torch-CPU network + numpy extract / blend / normalise,
    bit-identical to the reference's `-f pytorch` CPU path, tests/test_oracle_vs_reference.py) on a sub-chunk that holds
    `n_patches` whole patches of the workload's geometry.

    Outside the timed region, as SURVEY.md section 8d / BASELINE.md section 3 define the metric: model load, patch mask
    and output-chunk mask (built once per process / chunk shape by the reference, inferencer.py:300-312), the synthetic
    input, one warm-up patch.  Inside: `/255` of the sub-chunk, per patch cutout + network + crop/mask + blend, the final
    `*= 1/W` and the `< 1.0001` scan."""

    def __init__(self, patch, overlap, threads):
        import torch
        from chunkflow_b200.lib import load_source
        from oracle import inferencer_oracle as O
        self.O, self.patch, self.overlap, self.threads = O, patch, overlap, threads
        torch.set_num_threads(threads)
        self.model = load_source(MODEL_FILE).load_model(None)
        self.pmask = O.make_patch_mask(patch, overlap)
        self.masks = {}
        self.warm = False

    def sub_chunk(self, chunk_shape, n_patches):
        nx = min(n_patches, 2)
        nz = (n_patches + nx - 1) // nx
        sub = (self.patch[0] + (nz - 1) * (self.patch[0] - self.overlap[0]), self.patch[1],
               self.patch[2] + (nx - 1) * (self.patch[2] - self.overlap[2]))
        return tuple(min(a, c) for a, c in zip(sub, chunk_shape))

    def run(self, chunk_shape, n_patches, seed):
        """-> dict(seconds, patches, sub, per-part seconds, output, image)"""
        O = self.O
        sub = self.sub_chunk(chunk_shape, n_patches)
        img = np.random.default_rng(seed).integers(0, 256, size=sub, dtype=np.uint8)
        kw = dict(input_patch_size=self.patch, output_patch_overlap=self.overlap, num_output_channels=3, framework="pytorch",
                  model=self.model)
        if sub not in self.masks:
            geom = O.Geometry(self.patch, None, self.overlap)
            slices = O.patch_slices_list(geom, sub)
            self.masks[sub] = (self.pmask, O.output_chunk_mask(geom, slices, sub, (0, 0, 0), self.pmask), len(slices))
        if not self.warm:   # one warm-up patch (thread pool, oneDNN primitive cache)
            O.infer_chunk(img[:self.patch[0], :self.patch[1], :self.patch[2]], patch_limit=1, precomputed=None, **kw)
            self.warm = True
        timers = {}
        t0 = time.perf_counter()
        out, _ = O.infer_chunk(img, precomputed=self.masks[sub][:2], timers=timers, **kw)
        dt = time.perf_counter() - t0
        return dict(seconds=dt, patches=self.masks[sub][2], sub=sub, parts=timers, output=out, image=img)


def extrapolate_cpu(run, chunk_shape, P):
    """Seconds for the whole chunk from a sample: per-patch parts scale with the patch count, per-voxel parts (the /255
    of the input, the final normalise + range scan) with the chunk volume."""
    nvox, svox = float(np.prod(chunk_shape)), float(np.prod(run["sub"]))
    t = run["parts"]
    per_patch = (t["network"] + t["extract_blend"]) / run["patches"]
    per_voxel = (t["normalize_input"] + t["finalize"]) / svox
    other = max(0.0, run["seconds"] - sum(t.values())) / run["patches"]   # python glue between the timers
    return (per_patch + other) * P + per_voxel * nvox, per_patch, t["network"] / run["patches"]


SPLIT_CHUNK = (512, 2048, 2048)   # BASELINE config #5 (zyx), 2541 patches of 32x256x256


def split_chunk_block(inf, Chunk, patch, overlap, rank, world, local_rank, args, barrier, max_over_ranks):
    """One oversized chunk over all ranks (chunkflow_b200.distributed.infer_chunk_split): z-slabs of patch rows, partial sums
    of the overlapping planes sent to their owner over NCCL, added by cfb_halo_add_device, normalised by the owner.  Timed
    with host buffers in (each rank uploads its sub-chunk inside the timed region) and the result left on the GPUs; then the
    parts are gathered on rank 0 and compared with the single-GPU result of the same chunk."""
    import torch
    import torch.distributed as dist
    from chunkflow_b200 import distributed as D
    shape = SPLIT_CHUNK
    img = np.empty(shape, np.uint8)
    for z in range(0, shape[0], 64):   # same data on every rank
        img[z:z + 64] = np.random.default_rng(20260922 + 1000 + z).integers(0, 256, size=img[z:z + 64].shape, dtype=np.uint8)
    chunk = Chunk(img)
    slabs = D.plan_z_slabs(shape[0], patch[0], overlap[0], world)
    tm = {}
    part = D.infer_chunk_split(inf, chunk, to_host=False, timing=tm)   # warm-up (autotune for this rank's batch shapes)
    del part
    n_steps = min(args.steps, 3)
    times, tms = [], []
    for _ in range(n_steps):
        barrier()
        t0 = time.perf_counter()
        tm = {}
        part = D.infer_chunk_split(inf, chunk, to_host=False, timing=tm)
        torch.cuda.synchronize()
        times.append(max_over_ranks(time.perf_counter() - t0))
        tms.append(tm)
        if _ < n_steps - 1:
            del part
    exch = max_over_ranks(float(np.mean([t.get("exchange_ms", 0.0) for t in tms])))
    # the rank that arrives last at the exchange waits for nobody: its time is the transfer + add itself
    exch_min = -max_over_ranks(-float(np.mean([t.get("exchange_ms", 0.0) for t in tms])))
    comp = max_over_ranks(float(np.mean([t.get("compute_ms", 0.0) for t in tms])))
    sent = torch.tensor([float(tms[-1].get("halo_bytes_sent", 0))], dtype=torch.float64, device="cuda")
    dist.all_reduce(sent)
    # ---- gather on rank 0 and compare with the single-GPU result of the same chunk
    C = 3
    max_abs = None
    me = slabs[rank]
    if rank == 0:
        full = torch.empty((C,) + shape, dtype=torch.float32, device="cuda")
        if part is not None:
            full[:, me.own_z0:me.own_z1] = part.tensor
        for s in slabs[1:]:
            if s.empty or s.own_z1 <= s.own_z0:
                continue
            for c in range(C):
                dist.recv(full[c, s.own_z0:s.own_z1], src=s.rank)
        del part
        single = torch.empty((C,) + shape, dtype=torch.float32, device="cuda")
        d_in = torch.from_numpy(img).cuda()
        inf.engine.infer_chunk_device(d_in.data_ptr(), np.uint8, shape, single.data_ptr(), torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        max_abs = 0.0
        for c in range(C):
            for z in range(0, shape[0], 64):
                max_abs = max(max_abs, float((full[c, z:z + 64] - single[c, z:z + 64]).abs().max().item()))
        del full, single, d_in
    else:
        if part is not None:
            t = part.tensor
            for c in range(C):
                dist.send(t[c].contiguous(), dst=0)
        del part
    torch.cuda.empty_cache()
    barrier()
    sec = float(np.mean(times))
    nv = float(np.prod(shape))
    return {"workload": f"ONE {'x'.join(map(str, shape))} uint8 chunk split into z-slabs of patch rows over {world} GPUs, "
                        f"patch {'x'.join(map(str, patch))} overlap {'x'.join(map(str, overlap))}, host chunk in (H2D inside), result left on the GPUs",
            "seconds": sec, "value": nv / sec / 1e6, "unit": "Mvoxels/s", "steps": n_steps, "ranks": world,
            "rows_per_rank": [s.row_end - s.row_begin for s in slabs],
            "halo_bytes_total": float(sent.item()), "exchange_ms_max_over_ranks": exch, "exchange_ms_min_over_ranks": exch_min,
            "compute_ms_max_over_ranks": comp,
            "exchange_share_of_step": exch_min / (sec * 1e3) if sec > 0 else None,
            "exchange_note": "max over ranks includes waiting for the slowest rank's slab (row imbalance); min over ranks = NCCL transfer + add",
            "exchange": "NCCL send/recv of the overlapping planes to their owner + cfb_halo_add_device; weight volume computed locally",
            "max_abs_vs_single_gpu": max_abs, "tolerance": 2e-6}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=os.environ.get("CFB_BENCH_WORKLOAD", "1024"), choices=sorted(WORKLOADS))
    ap.add_argument("--batch-size", type=int, default=int(os.environ.get("CFB_BENCH_BATCH", 12)))
    ap.add_argument("--precision", default=os.environ.get("CHUNKFLOW_B200_PRECISION"))
    ap.add_argument("--cpu-sample-patches", type=int, default=0, help="patches per CPU sample (0 = 12 for the cpu_baseline leg; the "
                    "reference arm spreads >= 26 patches over its timed steps)")
    ap.add_argument("--no-split-chunk", action="store_true", help="N > 1: skip the config-#5 block (one chunk split over the ranks)")
    ap.add_argument("--no-pageable", action="store_true")
    ap.add_argument("--no-alt-precision", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write a fixed sample of what the last timed step "
                    "computed to DIR/*.npy (rank 0; see dump_outputs), to compare two builds output for output")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    chunk_shape, patch, overlap = WORKLOADS[args.workload]
    nvox = int(np.prod(chunk_shape))
    P = patch_count(chunk_shape, patch, overlap)
    threads = host_threads()
    config = {"workload": f"{'x'.join(map(str, chunk_shape))} uint8 chunk per GPU, 3-ch affinity UNet3L(16,32,64), "
                          f"patch {'x'.join(map(str, patch))} overlap {'x'.join(map(str, overlap))}, mask_output_chunk",
              "patches_per_chunk": P, "batch_size": args.batch_size, "chunks": world,
              "l2_policy": "inputs and outputs (1 GB + 12.9 GB per step) are far larger than the 126 MB L2",
              "parallelism": f"{world} independent chunk(s), one per GPU, no collective"}

    if args.impl == "reference":
        # The reference's own CPU algorithm on the host cores (oracle port; /root/reference does not travel).
        if rank != 0:
            return
        ref = CpuReference(patch, overlap, threads)
        per_step = args.cpu_sample_patches or int(min(14, max(2, -(-26 // max(1, args.steps)))))
        runs = []
        for i in range(args.warmup + args.steps):
            timed = i >= args.warmup
            r = ref.run(chunk_shape, per_step if timed else 1, 20260922 + i)   # a warm-up step is one patch
            if timed:
                runs.append(r)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, runs[-1]["output"])
        agg = dict(seconds=sum(r["seconds"] for r in runs), patches=sum(r["patches"] for r in runs), sub=runs[0]["sub"],
                   parts={k: sum(r["parts"][k] for r in runs) for k in runs[0]["parts"]})
        agg["sub"] = (runs[0]["sub"][0] * len(runs),) + tuple(runs[0]["sub"][1:])   # voxels of all timed sub-chunks
        total_s, per_patch, net_per_patch = extrapolate_cpu(agg, chunk_shape, P)
        value = nvox / total_s / 1e6
        sample = (f"{agg['patches']} patches of {'x'.join(map(str, patch))} timed over {len(runs)} steps (sub-chunk "
                  f"{'x'.join(map(str, runs[0]['sub']))} per step): {per_patch:.3f} s/patch ({net_per_patch:.3f} s torch-CPU network + "
                  f"{per_patch - net_per_patch:.3f} s numpy cutout/blend), per-voxel /255 + normalise + range scan scaled by volume; "
                  f"extrapolated to {P} patches; excluded: model load, patch-mask and output-chunk-mask construction, one warm-up patch")
        print(json.dumps({
            "impl": "reference", "metric": "Mvoxels/s", "value": value, "unit": "Mvoxels/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": agg["seconds"] / len(runs) * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
            "cpu_baseline": {"value": value, "unit": "Mvoxels/s", "cores": threads, "kind": "port", "sample": sample,
                             "cpu": cpu_model(), "s_per_patch": per_patch, "s_per_patch_network": net_per_patch},
            "e2e": {"value": value, "unit": "Mvoxels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    import torch
    import torch.distributed as dist
    from chunkflow_b200 import Chunk, Inferencer

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    pin_t, host_in = synthetic_chunk(chunk_shape, 20260922 + rank)
    inf = Inferencer(MODEL_FILE, None, patch, output_patch_overlap=overlap, num_output_channels=3, framework="b200",
                     batch_size=args.batch_size, mask_output_chunk=True, device=local_rank, precision=args.precision)
    eng = inf.engine
    out_shape = eng.output_shape(chunk_shape)
    d_in = torch.from_numpy(host_in).cuda(non_blocking=False) if pin_t is None else pin_t.cuda()
    d_out = torch.empty(out_shape, dtype=torch.float32, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream

    def step_device():
        eng.infer_chunk_device(d_in.data_ptr(), np.uint8, chunk_shape, d_out.data_ptr(), stream)

    for _ in range(args.warmup):
        step_device()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    barrier()
    if sampler:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ncu_range = bool(os.environ.get("CFB_NCU_RANGE"))  # `ncu --profile-from-start off`: capture the timed region only
    if ncu_range:
        torch.cuda.cudart().cudaProfilerStart()
    e0.record()
    for _ in range(args.steps):
        step_device()
    e1.record()
    torch.cuda.synchronize()
    if ncu_range:
        torch.cuda.cudart().cudaProfilerStop()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:   # before the profiled step below overwrites d_out
        dump_outputs(args.dump_outputs, d_out)
    launches = eng.last_timing()["launches"]
    value = nvox * world * args.steps / (ms / 1e3) / 1e6

    # ---- per-kernel-class roofline: one extra profiled step (CUDA events around every launch, same stream)
    eng.set_profiling(True)
    step_device()
    torch.cuda.synchronize()
    layers = eng.layer_timing()
    eng.set_profiling(False)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    conv_ms = sum(layers[k][0] for k in CONV3_FLOP if k in layers)
    conv_launches = sum(layers[k][1] for k in CONV3_FLOP if k in layers)
    pvox = int(np.prod(patch))
    conv_flop = sum(v for k, v in CONV3_FLOP.items() if k in layers) * P * pvox
    tf_peak = peaks.get("bf16_tflops_sustained", 1400.0)
    # dominant kernel = the 3x3x3 layer with the largest share of the step (dec0.0 / dec1.0, the concat layers)
    dom = max((k for k in CONV3_FLOP if k in layers), key=lambda k: layers[k][0])
    dom_ms, dom_launches = layers[dom]
    dom_flop_per_launch = CONV3_FLOP[dom] * P * pvox / dom_launches
    achieved = dom_flop_per_launch / (dom_ms / dom_launches / 1e3) / 1e12 if dom_ms > 0 else 0.0
    traffic, pipe_note = None, ""
    try:  # DRAM bytes per launch from the committed ncu --set full capture (profiles/r01_ncu_traffic.json), scaled to this batch
        prof = "r02_ncu_traffic.json" if eng.params.precision == 3 else "r01_ncu_traffic.json"   # --set full capture of the same precision mode
        tl = json.load(open(os.path.join(ROOT, "profiles", prof)))["layers"]
        t = tl.get(dom)
        if t and t.get("dram_bytes_per_patch"):
            traffic = t["dram_bytes_per_patch"] * P / dom_launches
        pipes = [v["tensor_pipe_active_pct"] for k, v in tl.items() if k in CONV3_FLOP and "conv3" in v.get("kernel", "")]
        if pipes:
            pipe_note = "; ncu tensor-pipe active %.0f-%.0f %% over the 3x3x3 layers, %.0f %% on this one" % (
                min(pipes), max(pipes), (t or {}).get("tensor_pipe_active_pct", float("nan")))
    except Exception:
        pass
    roofline = {"bound": "tensor", "kernel": f"{dom}: tcgen05 3x3x3 convolution (conv3_ts_umma_kernel: z-stacked, A operand in tensor memory)",
                "achieved": achieved, "peak": tf_peak, "unit": "TFLOP/s", "frac": achieved / tf_peak,
                "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "fallback (B200_PROFILING.md)",
                "traffic": traffic, "launches": dom_launches, "ms_per_launch": dom_ms / max(dom_launches, 1),
                "algorithmic_flop_per_launch": dom_flop_per_launch,
                "note": ("the f16f8 mode executes 2x these algorithmic FLOPs on the tensor pipe (one fp16 + one e4m3 K=32 product per multiply)"
                         if eng.params.precision == 3 else "the fp16 hi/lo split (f16x3) executes 3x these algorithmic FLOPs on the tensor pipe") + pipe_note +
                        " (profiles/r02_ncu_full_summary.md / r01_ncu_full_summary.md)",
                "conv_stack": {"achieved": conv_flop / (conv_ms / 1e3) / 1e12 if conv_ms > 0 else 0.0, "unit": "TFLOP/s",
                               "ms_per_chunk": conv_ms, "launches": conv_launches, "algorithmic_flop_per_chunk": conv_flop}}
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    pv = P * int(np.prod(patch))
    mem = {}
    parts = {0: 0, 1: 2, 2: 1, 3: 2}[eng.params.precision]
    # fused head+blend reads the last CP8 activation (16 ch x 2 B x parts) and read-modify-writes 3 fp32 channels
    for name, bytes_per in (("extract", 5 * pv), ("blend", 36 * pv), ("head+blend", (32 * parts + 24) * pv)):
        if name in layers and layers[name][0] > 0:
            gbs = bytes_per / (layers[name][0] / 1e3) / 1e9
            mem[name] = {"ms_per_chunk": layers[name][0], "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / hbm_peak}
    step_ms = {k: round(v[0], 3) for k, v in layers.items()}

    # ---- end to end through the public API: host uint8 chunk in -> host float32 affinity map out
    e2e = None
    if not args.no_e2e:
        need = int(np.prod(out_shape)) * 4
        pin = True
        try:  # page-locking 12.9 GB per rank: only when the host clearly has the room (all local ranks do the same)
            import psutil
            pin = psutil.virtual_memory().available > 3 * need * max(1, int(os.environ.get("LOCAL_WORLD_SIZE", world)))
        except Exception:
            pass
        pin_out = torch.empty(out_shape, dtype=torch.float32, pin_memory=pin)
        host_out = pin_out.numpy()
        chunk = Chunk(host_in)
        inf(chunk, output_buffer=host_out)  # warm-up (allocates the staging buffers)
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            inf(chunk, output_buffer=host_out)
        torch.cuda.synchronize()
        dt = max_over_ranks(time.perf_counter() - t0)
        barrier()
        e2e = {"value": nvox * world * args.steps / dt / 1e6, "unit": "Mvoxels/s", "h2d_bytes_per_step": int(host_in.nbytes),
               "d2h_bytes_per_step": int(host_out.nbytes), "ms_per_step": dt / args.steps * 1e3,
               "host_buffers": "pinned" if pin else "pageable (not enough free host memory to page-lock the output)",
               "timing_of_last_step_ms": {k: round(v, 3) for k, v in inf.timing.items()}}
        del pin_out

    # ---- the contract a drop-in caller gets: plain (pageable) numpy chunk in, `inf(chunk)` allocates its own result
    e2e_pageable = None
    if not args.no_e2e and not args.no_pageable:
        plain = np.array(host_in, copy=True)   # ordinary pageable memory
        chunk = Chunk(plain)
        res = inf(chunk)                       # warm-up (creates the engine's pinned staging ring)
        del res
        barrier()
        n_steps = min(args.steps, 3)
        t0 = time.perf_counter()
        free_s = 0.0
        for _ in range(n_steps):
            res = inf(chunk)                   # a fresh 12.9 GB result array per call, like the reference (inferencer.py:360,479)
            checksum = float(res.array[0, -1, -1, -1])
            t1 = time.perf_counter()
            del res                            # the caller's free of the previous result is part of the steady state
            free_s += time.perf_counter() - t1
        dt = max_over_ranks(time.perf_counter() - t0)
        barrier()
        e2e_pageable = {"value": nvox * world * n_steps / dt / 1e6, "unit": "Mvoxels/s", "ms_per_step": dt / n_steps * 1e3,
                        "free_of_result_ms_per_step": free_s / n_steps * 1e3,
                        "steps": n_steps, "host_buffers": "pageable numpy in; the result array is allocated by the call (np.empty; the "
                        "Inferencer hands the previous result array out again once the caller has dropped every reference to it) and "
                        "filled through the engine's pinned staging ring by host threads; the timed loop includes dropping the previous "
                        "result", "last_value": checksum}
        del plain, chunk

    # ---- CPU baseline (rank 0, N = 1) and parity of the GPU path on the SAME sub-chunk at the benchmarked geometry
    cpu, parity, cpu_sample = None, None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        ref = CpuReference(patch, overlap, threads)
        r = ref.run(chunk_shape, args.cpu_sample_patches or 12, 20260922)
        total_s, per_patch, net_per_patch = extrapolate_cpu(r, chunk_shape, P)
        cpu = {"value": nvox / total_s / 1e6, "unit": "Mvoxels/s", "cores": threads, "kind": "port", "cpu": cpu_model(),
               "s_per_patch": per_patch, "s_per_patch_network": net_per_patch,
               "sample": f"{r['patches']} patches of {'x'.join(map(str, patch))} (sub-chunk {'x'.join(map(str, r['sub']))}): {per_patch:.3f} s/patch "
                         f"({net_per_patch:.3f} s torch-CPU network + {per_patch - net_per_patch:.3f} s numpy cutout/blend), per-voxel /255 + normalise + "
                         f"range scan scaled by volume; extrapolated to {P} patches; excluded: model load, patch-mask and output-chunk-mask "
                         "construction, one warm-up patch"}
        got = inf(Chunk(r["image"])).array     # same Inferencer (batch, precision, autotuned tilings) as the timed steps
        parity = {"max_abs": float(np.abs(got - r["output"]).max()), "tolerance": 1e-3,
                  "config": f"sub-chunk {'x'.join(map(str, r['sub']))} = {r['patches']} patches of the benchmarked geometry, batch "
                            f"{args.batch_size}, GPU result vs the CPU reference port (bit-identical to the reference's -f pytorch path)"}
        del got
        cpu_sample = r

    # ---- the other fp32-parity mode of the convolution stack, device-resident, for the record (rank 0, N = 1)
    alt = None
    if rank == 0 and world == 1 and not args.no_alt_precision and eng.params.precision in (1, 3):
        other = "f16x3" if eng.params.precision == 3 else "f16f8"
        inf2 = Inferencer(MODEL_FILE, None, patch, output_patch_overlap=overlap, num_output_channels=3, framework="b200",
                          batch_size=args.batch_size, mask_output_chunk=True, device=local_rank, precision=other)
        d_out2 = torch.empty_like(d_out)
        for _ in range(2):
            inf2.engine.infer_chunk_device(d_in.data_ptr(), np.uint8, chunk_shape, d_out2.data_ptr(), stream)
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(min(args.steps, 3)):
            inf2.engine.infer_chunk_device(d_in.data_ptr(), np.uint8, chunk_shape, d_out2.data_ptr(), stream)
        a1.record()
        torch.cuda.synchronize()
        alt_ms = a0.elapsed_time(a1) / min(args.steps, 3)
        alt = {"precision": other, "ms_per_step": alt_ms, "value": nvox / (alt_ms / 1e3) / 1e6, "unit": "Mvoxels/s"}
        # size-independent check at the FULL benchmark size: the two fp32-parity modes (different number formats, different kernels for
        # the first layer / transposed convolutions / pooling) agree over the whole volume -- all 1075 patches, clamped last patches,
        # every tile boundary.  d_out still holds the default mode's result of the last device-resident step.
        full = 0.0
        for c in range(d_out.shape[0]):
            for z in range(0, d_out.shape[1], 64):
                full = max(full, float((d_out[c, z:z + 64] - d_out2[c, z:z + 64]).abs().max().item()))
        alt["full_volume_max_abs_vs_default_mode"] = full
        alt["full_volume_check"] = ("max |default - %s| over the whole %s output volume; each mode is within its own tolerance of the CPU "
                                    "reference on the 12-patch sub-chunk (parity / alt_precision.parity_max_abs)" % (other, "x".join(map(str, out_shape))))
        del d_out2
        if cpu_sample is not None:   # parity of this mode on the same sub-chunk as the main parity block
            got2 = inf2(Chunk(cpu_sample["image"])).array
            alt["parity_max_abs"] = float(np.abs(got2 - cpu_sample["output"]).max())
            del got2
        del inf2
    cpu_sample = None

    # ---- BASELINE config #5: ONE 512x2048x2048 chunk split over the N ranks, halo planes exchanged over NCCL
    split = None
    if world > 1 and not args.no_split_chunk:
        inf._last_result = None   # the recycled 12.9 GB host result of the pageable block
        del d_out
        torch.cuda.empty_cache()
        split = split_chunk_block(inf, Chunk, patch, overlap, rank, world, local_rank, args, barrier, max_over_ranks)

    if rank == 0:
        precision = {0: "f32 (FFMA, CUDA cores)", 1: "f16x3 hi/lo split on tcgen05, f32 accumulate",
                     2: "f16 on tcgen05, f32 accumulate",
                     3: "f16f8: fp16 main product + one e4m3 (K=32) product carrying both hi/lo correction terms on tcgen05, f32 accumulate"}[eng.params.precision]
        print(json.dumps({
            "metric": "Mvoxels/s", "value": value, "unit": "Mvoxels/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": {0: "f32", 1: "f16x3", 2: "f16", 3: "f16f8"}[eng.params.precision], "precision_mode": precision,
            "data": "synthetic", "config": config, "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches) * args.steps,
            "e2e_pageable": e2e_pageable, "parity": parity, "split_chunk": split, "alt_precision": alt,
            "roofline": roofline, "memory_kernels": mem, "kernel_ms_per_chunk": step_ms, "cpu_baseline": cpu}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
