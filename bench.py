#!/usr/bin/env python
"""Benchmark of the per-frame YOLO11-seg hot path (BASELINE.json: "YOLO11-seg 640x640 frames/s").

  python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torchrun, one rank per GPU)
  python bench.py --impl reference ...                      (the CPU oracle standing in for the reference's Inference
                                                             Engine CPU backend, which cannot run outside Unity)

Workload (BASELINE.json configs[1]): YOLO11n-seg, 640x640, batch 64 synthetic uint8 frames, random-init weights.
A step = one pass of the whole path (preprocess -> backbone/neck/head -> decode -> NMS -> gather -> masks) over one
batch of 64 frames per GPU.  Frames are sharded over ranks with no collective (weak scaling: 64 frames per GPU).

  value        : frames/s with the frames already resident in HBM (xrseg_schedule_device), CUDA events on the runners'
                 streams; consecutive steps alternate over --value-streams runners so that the sparse tail of one step
                 overlaps the head of the next (every step is still a full pass over its own 64 frames)
  value_serial : the same with ONE runner / one stream: strictly serial batch-64 steps
  e2e          : through the reference-facing call with HOST buffers: H2D of the frames from pinned memory and D2H of
                 boxes + labels + bit-packed masks inside the timed region, every step (--e2e-depth runners round-robin)
  e2e_contract : the same with the reference's own readback contract instead of the compact one: all four graph outputs,
                 output_3 as f32 [N,160,160] (IEExecutor.cs:446-449), 102 400 B per detection
  latency      : batch-1 1280x960 frame -> letterbox -> detections on the host, p50 / p99 of 1000 samples after 100 warm-up
                 (BASELINE.json configs[3])
  roofline / cpu_baseline : see DESIGN.md section 5

  --config 2 : BASELINE.json configs[2] (YOLO11s-seg, batch 512 split over the GPUs; 64 frames on one GPU)
  --config 4 : BASELINE.json configs[4] (post-processing stress: 8400 x 80 logits, 300 detections, 640x640 masks)

  --dump-outputs DIR : after the timed steps of `value`, write what its last step returned to a caller (rank 0's frames)
                       as DIR/<name>.npy, float32; the inputs are seeded, so two builds can be compared output for output
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH = 64
SEED_FRAMES, SEED_WEIGHTS = 0, 1
CLS_BIAS = None   # frozen per-scale default of weights.random_weights
METRIC = "YOLO11-seg 640x640 frames/s"
WORKLOAD = "YOLO11n-seg 640x640, batch 64 synthetic uint8 frames per GPU, random-init weights (seed 1)"
SCALE = "n"       # --scale s: BASELINE.json configs[2] shapes (YOLO11s-seg); not the default bench line


def synthetic_frames(n, seed):
    rng = np.random.default_rng(seed)
    return rng.integers(0, 256, (n, 640, 640, 3), dtype=np.uint8)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d["hbm_gbs"], d["bf16_tflops"], d.get("bf16_tflops_sustained", d["bf16_tflops"]), "measured"
    return 6650.0, 1590.0, 1400.0, "fallback"


class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = []
        for line in open(self.f.name):
            parts = [x.strip() for x in line.split(",")]
            if len(parts) >= 7:
                try:
                    rows.append((float(parts[0]), float(parts[1]), float(parts[2]), parts[3:7]))
                except ValueError:
                    pass
        os.unlink(self.f.name)
        if rows:
            busy = [r for r in rows if r[2] > 250.0] or rows        # samples under load (power above idle)
            out["sm_mhz"] = float(np.median([r[0] for r in busy]))
            out["sm_max_mhz"] = rows[0][1]
            out["power_w_max"] = max(r[2] for r in rows)
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            out["reasons"] = [n for i, n in enumerate(names) if any(r[3][i].lower().startswith("active") for r in rows)]
            out["samples"] = len(rows)
        return out


DUMP_BYTES = 60 << 20     # --dump-outputs stays under 64 MB (decimal) with the .npy headers


def dump_outputs(path, r):
    """The arrays a caller of the finished run of Runner `r` receives (xrseg_counts, xrseg_keep_indices, xrseg_readback
    0-3), as float32 .npy files of at most DUMP_BYTES in all: the 160x160 mask probabilities are subsampled on a fixed
    pixel grid (every 2nd, 4th, ... row and column) when all of them would not fit."""
    os.makedirs(path, exist_ok=True)
    keep, scores = r.keep_indices()
    outs = {"counts": r.counts(), "keep": keep, "scores": scores, "boxes": r.readback(0), "labels": r.readback(1),
            "coefs": r.readback(2)}
    probs = r.readback(3)
    step = 1
    while 4 * (sum(a.size for a in outs.values()) + probs[:, ::step, ::step].size) > DUMP_BYTES:
        step *= 2
    outs["mask_probs"] = probs[:, ::step, ::step]                    # [N, 160 / step, 160 / step]
    for name, a in outs.items():
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(a, np.float32))


def cpu_oracle_fps(ws, frames, threads, budget_s=12.0, chunk=4, max_frames=64):
    """The oracle (CPU restatement of the reference path) on a bounded sample of the same workload."""
    import torch

    from oracle import preprocess as pre
    from oracle import yolo11seg as Y
    torch.set_num_threads(threads)
    x = torch.from_numpy(np.concatenate([pre.to_tensor(f) for f in frames[:chunk]]))
    Y.run_model(ws, x[:1], SCALE)                                       # warm-up
    done, t0 = 0, time.perf_counter()
    while True:
        i = done % len(frames)
        x = torch.from_numpy(np.concatenate([pre.to_tensor(f) for f in frames[i:i + chunk]]))
        Y.run_model(ws, x, SCALE)
        done += x.shape[0]
        dt = time.perf_counter() - t0
        if dt >= budget_s or done >= max_frames:
            return done / dt, done, dt


def run_reference(args, rank, world):
    """--impl reference: the reference's own path on the host cores (oracle port; Unity cannot run here)."""
    if rank != 0:
        return
    import torch

    # nothing of the product is imported on this arm (no libxrseg.so in the process): the oracle has its own weight
    # generator, proven equal to the product-side one by tests/test_abi.py
    from oracle import preprocess as pre
    from oracle import yolo11seg as Y
    ws = Y.random_weights(SCALE, SEED_WEIGHTS, CLS_BIAS)
    frames = synthetic_frames(8, SEED_FRAMES)
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    sample = 8
    x = torch.from_numpy(np.concatenate([pre.to_tensor(f) for f in frames]))
    for _ in range(max(1, min(args.warmup, 2))):
        Y.run_model(ws, x[:2], SCALE)
    times = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        Y.run_model(ws, x, SCALE)
        times.append(time.perf_counter() - t0)
    t = float(np.sum(times))
    fps = sample * args.steps / t
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD + "; reference arm: each step = a bounded SAMPLE of 8 of the 64 frames on the host cores",
                   "frames_per_step": sample},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port",
                         "sample": f"{sample} frames per step x {args.steps} steps, torch CPU fp32 oracle"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def run_post_stress(args, device):
    """--config 4 (BASELINE.json configs[4]): the post-processing kernels of the product on the stress tensors -- 8400
    anchors x 80 classes, 300 planted objects x 3 overlapping anchors per frame (854 candidates -> 300 kept), 32 x 160 x 160
    prototypes, fp16 like the network's own head tensors -- plus the fused 640x640 mask kernel.  The tensors enter through
    libxrseg_debug.so's xrseg_debug_post_f16 (the product has no entry point that takes head tensors); every launch is timed
    with CUDA events on the runner's stream (XRSEG_DBG_TIME)."""
    os.environ["XRSEG_DBG_TIME"] = "1"
    from xr_image_segmentation_b200 import _lib, inference as I, weights as W
    B = args.batch
    layers, ws = W.random_weights("n", SEED_WEIGHTS, None)
    r = I.Runner(I.Model(W.write_pack("n", layers, ws), "n"), device=device, max_batch=B, max_det=300, debug=True)
    rng = np.random.default_rng(5)
    A = 8400
    box = rng.standard_normal((B, A, 64)).astype(np.float32)
    box.reshape(B, A, 4, 16)[..., 1] += 6.0
    cls = (rng.standard_normal((B, A, 80)) - 6).astype(np.float32)
    for f in range(B):
        for a in rng.choice(6400, 300, replace=False):
            for d in (0, 1, 80):
                if a + d < 6400:
                    cls[f, a + d, rng.integers(0, 80)] = 2.0 + rng.standard_normal()
    coef = rng.standard_normal((B, A, 32)).astype(np.float32)
    proto = rng.standard_normal((B, 32, 25600)).astype(np.float32)
    hbm, _, _, how = measured_peaks()
    sampler = ClockSampler(device)
    acc = {}
    for it in range(args.warmup + args.steps):
        r.debug_post(box, cls, coef, proto, f16=True)
        r.wait(strict=False)                               # more than 300 boxes would be kept: the cap is part of the workload
        if it >= args.warmup:
            for name, ms, by in r.debug_post_timings():
                a_ = acc.setdefault(name, [0.0, by])
                a_[0] += ms / args.steps
    n_det = int(r.counts().sum())
    # fused 640x640 masks (coef x proto -> bilinear x4 -> crop -> threshold) into device scratch: kernel time only
    r.masks(_lib.MASK_UPSAMPLE_640, to_host=False)
    r.event_record(0)
    for _ in range(args.steps):
        r.masks(_lib.MASK_UPSAMPLE_640, to_host=False)
    r.event_record(1)
    r.sync()
    ms640 = r.event_elapsed_ms(0, 1) / args.steps
    bytes640 = n_det * 640 * 640 + B * 32 * 25600 * 2      # u8 masks written + fp16 prototypes read once per frame
    acc["mask640_kernel"] = [ms640, bytes640]
    clocks = sampler.stop()
    total_ms = sum(v[0] for v in acc.values())
    kernels = {k: {"ms": v[0], "mbytes": v[1] / 1e6, "gbs": (v[1] / (v[0] * 1e-3) / 1e9) if v[1] else None,
                   "frac_of_hbm_peak": (v[1] / (v[0] * 1e-3) / 1e9 / hbm) if v[1] else None} for k, v in acc.items()}
    top = max((k for k in acc if acc[k][1]), key=lambda k: acc[k][0])
    print(json.dumps({
        "metric": "post-process stress frames/s (decode + NMS + gather + 160x160 mask assembly + 640x640 masks)",
        "value": B / (total_ms * 1e-3), "unit": "frames/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": total_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
        "config": {"workload": f"BASELINE.json configs[4]: batch {B}, 8400 anchors x 80 classes, 854 candidates -> 300 detections per "
                               "frame, 32x160x160 prototypes, 160x160 f32 probabilities + 640x640 u8 masks",
                   "detections": n_det, "timing": "sum of per-launch CUDA-event times on the runner's stream (launches run back to back)"},
        "roofline": {"kernel": top, "bound": "hbm", "achieved": kernels[top]["gbs"], "peak": hbm, "unit": "GB/s",
                     "frac": kernels[top]["frac_of_hbm_peak"], "traffic": None, "peak_source": how + " (copy bandwidth)"},
        "kernels": kernels, "gpu_launches": (len(acc) - 1 + 1) * args.steps, "clocks": clocks,
    }))
    r.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--scale", default="n", choices=["n", "s"], help="n = BASELINE configs[1] (default); s = configs[2] shapes")
    ap.add_argument("--e2e-micro-batch", type=int, default=0, help="frames per network pass of the e2e leg (0 = whole batch)")
    ap.add_argument("--latency-iters", type=int, default=1000, help="batch-1 latency samples after 100 warm-up frames (0 = skip)")
    ap.add_argument("--config", type=int, default=1, choices=[1, 2, 4],
                    help="BASELINE.json configs[]: 1 = YOLO11n-seg batch 64 (default, the metric's configuration); 2 = YOLO11s-seg, "
                         "batch 512 split over the GPUs; 4 = post-processing stress")
    ap.add_argument("--e2e-depth", type=int, default=4, help="runners of the end-to-end leg (submissions in flight + 1)")
    ap.add_argument("--value-streams", type=int, default=4, help="runners (streams) the device-resident leg alternates over")
    ap.add_argument("--profile-ops", type=int, default=5, help="iterations for the per-launch timing pass (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.config == 4):
        ap.error("--dump-outputs writes the outputs of the product's network path: not with --impl reference or --config 4")
    global SCALE, WORKLOAD, SEED_WEIGHTS
    world_env = int(os.environ.get("WORLD_SIZE", 1))
    if args.config == 2:
        args.scale = "s"
        args.batch = 512 // world_env if world_env in (2, 4, 8) else 64
        if args.batch > 64:                                   # 128 / 256-frame YOLO11s arenas: keep the runner count down
            args.value_streams = min(args.value_streams, 2)
            args.e2e_depth = min(args.e2e_depth, 2)
    if args.scale == "s":
        SCALE, SEED_WEIGHTS = "s", 3
        WORKLOAD = (f"YOLO11s-seg 640x640, batch {args.batch} synthetic uint8 frames per GPU, random-init weights (seed 3); "
                    "BASELINE.json configs[2] per-GPU share")
    elif args.batch != BATCH:
        WORKLOAD = WORKLOAD.replace("batch 64", f"batch {args.batch}")
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    args.warmup = max(args.warmup, 3)
    if args.config == 4:
        if rank == 0:
            run_post_stress(args, local_rank)
        return

    # bind this rank to the CPUs (and therefore the host memory) next to its GPU before anything allocates pinned
    # buffers: eight ranks streaming frames from one NUMA node would share that node's memory and PCIe root
    try:
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local_rank))
    except Exception:
        pass

    import torch
    import torch.distributed as dist

    from xr_image_segmentation_b200 import _lib, inference as I, weights as W

    if world > 1:
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lib = _lib.load_library()
    if lib.xrseg_device_count() == 0:
        raise SystemExit("bench.py: no B200 visible and there is no CPU fallback (use --impl reference for the CPU oracle)")

    B = args.batch
    layers, ws = W.random_weights(SCALE, SEED_WEIGHTS, CLS_BIAS)
    model = I.Model(W.write_pack(SCALE, layers, ws), SCALE)
    # the random-init YOLO11s-seg network produces ~150 overlapping detections per frame: run it with the reference's
    # unlimited NMS (caps at the anchor count) instead of the 2048-candidate / 300-detection defaults, which would
    # (correctly) report XRSEG_ERR_CAPACITY
    caps = dict(max_candidates=8400, max_det=1000) if SCALE == "s" else {}
    runner = I.Runner(model, device=local_rank, max_batch=B, **caps)
    # end-to-end leg: runners used round-robin (inference.PipelinedRunner): the host->device copies and the network passes
    # of the next steps overlap the readback of step i; every step still copies its frames from pinned host memory and
    # reads its detections back
    pipe = I.PipelinedRunner(model, device=local_rank, max_batch=B, depth=args.e2e_depth, micro_batch=args.e2e_micro_batch, **caps)
    runner_e2e = pipe.runners[0]
    # 4 distinct frame sets (4 x 78.6 MB > 126 MB L2) so no step finds its input in L2; every rank has its own frames
    NSETS = 4
    nbytes = B * 640 * 640 * 3
    host = [lib.xrseg_host_alloc(nbytes) for _ in range(NSETS)]
    assert all(host), "pinned allocation failed"
    import ctypes as C
    dev = torch.empty((NSETS, nbytes), dtype=torch.uint8, device=f"cuda:{local_rank}")
    for s in range(NSETS):
        fr = synthetic_frames(B, SEED_FRAMES + 1000 * rank + s)
        C.memmove(host[s], fr.ctypes.data, nbytes)
        dev[s].copy_(torch.from_numpy(fr.reshape(-1)))
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        runner.sync()

    # ---------------- device-resident leg: `value` ----------------
    for i in range(args.warmup):
        runner.schedule_device(dev[i % NSETS].data_ptr(), B, 640, 640, 3)
    runner.wait()
    counts = runner.counts()
    dets_per_frame = float(counts.mean())
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    # Consecutive steps alternate between two runners (own stream, own activation arena each), so the sparse tail of
    # step i (NMS / gather / masks keep few SMs busy) overlaps the head of step i+1.  --value-streams 1 serialises them.
    vr = [runner] if args.value_streams <= 1 else pipe.runners[:min(args.value_streams, len(pipe.runners))]
    for r_ in vr:
        r_.schedule_device(dev[0].data_ptr(), B, 640, 640, 3)      # graph capture / warm-up of every runner used
        r_.sync()
    barrier()
    vr[0].event_record(0)
    for i in range(args.steps):
        vr[i % len(vr)].schedule_device(dev[i % NSETS].data_ptr(), B, 640, 640, 3)
    for r_ in vr:
        r_.sync()
    vr[0].event_record(1)               # recorded after every stream has drained
    vr[0].sync()
    ms_dev = vr[0].event_elapsed_ms(0, 1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, vr[(args.steps - 1) % len(vr)])
    barrier()
    # the same steps strictly serial: one runner, one stream, step i+1 starts when step i has finished on the device
    runner.event_record(4)
    for i in range(args.steps):
        runner.schedule_device(dev[i % NSETS].data_ptr(), B, 640, 640, 3)
    runner.event_record(5)
    runner.sync()
    ms_serial = runner.event_elapsed_ms(4, 5)
    barrier()

    # ---------------- end-to-end leg: host frames in, detections out, every step ----------------
    d2h = 0

    def collect():
        nonlocal d2h
        counts, boxes, labels, bits = pipe.collect(_lib.MASK_BITS_160)
        d2h = boxes.nbytes + labels.nbytes + bits.nbytes + 4 * B
        return counts

    for i in range(min(args.warmup, 4)):
        pipe.submit_ptr(host[i % NSETS], B, 640, 640, 3)
        collect()
    barrier()
    for r_ in pipe.runners:
        r_.sync()
    runner_e2e.event_record(2)
    ahead = args.e2e_depth - 1                         # submissions in flight while the oldest one is collected
    for i in range(min(ahead, args.steps)):
        pipe.submit_ptr(host[i % NSETS], B, 640, 640, 3)
    for i in range(args.steps):
        if i + ahead < args.steps:
            pipe.submit_ptr(host[(i + ahead) % NSETS], B, 640, 640, 3)
        collect()
    for r_ in pipe.runners:
        r_.sync()
    runner_e2e.event_record(3)          # everything of both runners has completed before this record
    runner_e2e.sync()
    ms_e2e = runner_e2e.event_elapsed_ms(2, 3)
    barrier()

    # ---------------- the same with the reference's readback contract: all four outputs, output_3 f32 [N,160,160] -------
    d2h_contract = 0

    # caller-owned result buffers, allocated once (pinned, like the frame buffers): sized for 4x the detections seen
    cap_det = max(64, int(4 * dets_per_frame * B))
    row_bytes = [16, 4, 128, 160 * 160 * 4]
    pinned = [(lib.xrseg_host_alloc(cap_det * rb), cap_det * rb) for rb in row_bytes]
    assert all(p_[0] for p_ in pinned), "pinned allocation failed"

    def collect_contract():
        nonlocal d2h_contract
        out = pipe.collect(contract=True, pinned=pinned)
        d2h_contract = sum(int(np.prod(shp)) * 4 for shp in out[1:]) + 4 * B

    pipe.submit_ptr(host[0], B, 640, 640, 3)
    collect_contract()
    barrier()
    runner_e2e.event_record(6)
    for i in range(min(ahead, args.steps)):
        pipe.submit_ptr(host[i % NSETS], B, 640, 640, 3)
    for i in range(args.steps):
        if i + ahead < args.steps:
            pipe.submit_ptr(host[(i + ahead) % NSETS], B, 640, 640, 3)
        collect_contract()
    for r_ in pipe.runners:
        r_.sync()
    runner_e2e.event_record(7)
    runner_e2e.sync()
    ms_contract = runner_e2e.event_elapsed_ms(6, 7)
    barrier()

    # ---------------- batch-1 streaming latency (BASELINE.json configs[3]): 1280x960 -> letterbox -> detections on the host
    lat = None
    if rank == 0 and args.latency_iters > 0:
        r1 = I.Runner(model, device=local_rank, max_batch=1, resize_mode=_lib.RESIZE_LETTERBOX, **caps)
        fb = 960 * 1280 * 3
        hf = lib.xrseg_host_alloc(fb)
        C.memmove(hf, np.random.default_rng(4).integers(0, 256, fb, dtype=np.uint8).ctypes.data, fb)
        ts = []
        LAT_WARM = 100
        for i in range(args.latency_iters + LAT_WARM):
            t0 = time.perf_counter()
            r1.schedule_ptr(hf, 1, 960, 1280, 3)
            r1.collect(_lib.MASK_BITS_160)                   # waits, then boxes + labels + bit masks in one call / one sync
            ts.append(time.perf_counter() - t0)
        ts = np.array(ts[LAT_WARM:]) * 1e3
        lat = {"p50_ms": float(np.percentile(ts, 50)), "p99_ms": float(np.percentile(ts, 99)), "iters": int(len(ts)),
               "warmup_iters": LAT_WARM,
               "config": f"YOLO11{SCALE}-seg batch 1, 1280x960 RGB host frame -> letterbox 640 -> boxes+labels+bit masks on the host"}
        lib.xrseg_host_free(hf)
        r1.close()
    clocks = sampler.stop() if sampler else None

    t = torch.tensor([ms_dev, ms_e2e, ms_serial, ms_contract], dtype=torch.float64, device=f"cuda:{local_rank}")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_dev, ms_e2e, ms_serial, ms_contract = (float(v) for v in t)
    launches = runner.launch_count()
    launches_e2e = runner_e2e.launch_count()

    if rank == 0:
        hbm, tf_burst, tf_sust, how = measured_peaks()
        value = world * B * args.steps / (ms_dev * 1e-3)
        e2e = world * B * args.steps / (ms_e2e * 1e-3)
        out = {
            "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "value_serial": world * B * args.steps / (ms_serial * 1e-3), "ms_per_step_serial": ms_serial / args.steps,
            "config": {"workload": WORKLOAD, "frames_per_gpu_per_step": B, "dets_per_frame": dets_per_frame,
                       "l2": "inputs rotate over 4 distinct 78.6 MB frame sets (> 126 MB L2); each step streams ~3 GB of activations",
                       "parallelism": f"frame-parallel x{world}, no collective",
                       "streams_per_gpu": len(vr)},
            "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_step": nbytes, "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": ms_e2e / args.steps, "pipeline": f"{args.e2e_depth} runners round-robin, one run in flight each",
                    "readback": "compact: output_0 boxes + output_1 labels + bit-packed 160x160 masks (NOT the reference's four-output "
                                "readback; that one is e2e_contract)"},
            "e2e_contract": {"value": world * B * args.steps / (ms_contract * 1e-3), "unit": "frames/s", "steps": args.steps,
                             "h2d_bytes_per_step": nbytes, "d2h_bytes_per_step": int(d2h_contract),
                             "ms_per_step": ms_contract / args.steps,
                             "readback": "the reference's contract (IEExecutor.cs:446-449): output_0 f32 [N,4], output_1 i32 [N], "
                                         "output_2 f32 [N,32], output_3 f32 [N,160,160] into caller-owned pinned buffers"},
            "gpu_launches": (2 * launches + launches_e2e + 1) * args.steps + (launches_e2e + 1) * (args.steps + 1),
            "clocks": clocks,
        }
        if lat:
            out["latency"] = lat
        # ---------------- roofline of the dominant kernel, timed live per launch ----------------
        if args.profile_ops > 0:
            runner.schedule_device(dev[0].data_ptr(), B, 640, 640, 3)
            runner.wait()
            ops = runner.profile_ops(args.profile_ops)
            tot = sum(o[1] for o in ops)
            # every launch of this pass is event-timed ALONE on an otherwise idle GPU (full clocks, no sustained power cap):
            # the burst cuBLAS figure is the honest tensor denominator (the sustained one was taken at a 1.2 GHz median)
            tf_peak = tf_burst
            ridge = tf_peak * 1e12 / (hbm * 1e9)                      # FLOP/B above which a kernel is tensor-bound
            traffic_tab = {}
            tpath = os.path.join(ROOT, "profiles", "traffic.json")
            if os.path.exists(tpath) and SCALE == "n" and B == BATCH:
                traffic_tab = json.load(open(tpath)).get("launches", {})

            def roof(o):
                name, ms, fl, by = o
                tensor = fl > 0 and by > 0 and fl / by > ridge
                ach = fl / (ms * 1e-3) / 1e12 if tensor else by / (ms * 1e-3) / 1e9
                peak = tf_peak if tensor else hbm
                t = traffic_tab.get(name, {}).get("dram_bytes")
                return {"kernel": name, "bound": "tensor" if tensor else "hbm", "achieved": ach, "peak": peak,
                        "unit": "TFLOP/s" if tensor else "GB/s", "frac": ach / peak, "traffic": t,
                        "ms_per_launch": ms, "share_of_step": ms / tot, "flop_per_byte": fl / by if by else None}

            conv = [o for o in ops if o[2] > 0 and not o[0].startswith("post.")]
            top = max(ops, key=lambda o: o[1])
            conv_ms, conv_fl = sum(o[1] for o in conv), sum(o[2] for o in conv)
            post = [o for o in ops if o[0] in ("post.decode", "post.decode_exact", "post.mask_prob")]
            out["roofline"] = roof(top)
            if "+cv3" in top[0]:
                out["roofline"]["note"] = ("proto.cv2 (3x3, 64->64) and proto.cv3 (1x1, 64->32) run as ONE launch: the 1x1 is a second set of "
                                           "tcgen05.mma (A operand from tensor memory) on the epilogue's packed fp16 tile; FLOPs and bytes are those of "
                                           "both layers without the 64-channel intermediate.  As two launches (XRSEG_FUSE_TAIL=0) the pair takes "
                                           "133 + 58 us (proto.cv2 alone: 0.55-0.58 of the burst peak, the pair 0.40)")
            out["roofline"].update({
                "peak_source": how + (" (burst bf16 cuBLAS: the launch is timed alone)" if out["roofline"]["bound"] == "tensor" else " (copy bandwidth)"),
                "algorithmic": "flops = 2*M*Cout*Cin*k*k, bytes = (in + out (+res) + weights) * 2 B, real channel counts (DESIGN.md 4)",
                "top5": [roof(o) for o in sorted(ops, key=lambda o: -o[1])[:5]],
                "conv_stack": {"tflops": conv_fl / (conv_ms * 1e-3) / 1e12, "frac_of_tensor_peak": conv_fl / (conv_ms * 1e-3) / 1e12 / tf_peak,
                               "frac_of_sustained_tensor_peak": conv_fl / (conv_ms * 1e-3) / 1e12 / tf_sust,
                               "gbs": sum(o[3] for o in conv) / (conv_ms * 1e-3) / 1e9,
                               "frac_of_hbm_peak": sum(o[3] for o in conv) / (conv_ms * 1e-3) / 1e9 / hbm, "ms": conv_ms},
                # per launch: timed here with CUDA events around the single launch (a ~20 us kernel carries the ~4 us of an isolated
                # launch in that figure) and, beside it, the duration of the same launch in the committed ncu capture
                # (profiles/traffic.json: gpu__time_duration of tools/gpu_round.sh, cold caches, the kernel alone)
                "post": {o[0]: dict({"ms": o[1], "gbs": o[3] / (o[1] * 1e-3) / 1e9, "frac_of_hbm_peak": o[3] / (o[1] * 1e-3) / 1e9 / hbm},
                                    **({"ncu_us": traffic_tab[o[0]]["us_under_ncu"],
                                        "ncu_gbs": o[3] / (traffic_tab[o[0]]["us_under_ncu"] * 1e-6) / 1e9,
                                        "ncu_frac_of_hbm_peak": o[3] / (traffic_tab[o[0]]["us_under_ncu"] * 1e-6) / 1e9 / hbm}
                                       if traffic_tab.get(o[0], {}).get("us_under_ncu") else {})) for o in post},
                "sum_launch_ms": tot,
                # the whole step against the same peaks: all algorithmic FLOPs / bytes of one pass over the TIMED step (`value`:
                # four runners overlapped, sustained clocks) -- the per-launch figures above time every launch ALONE with its
                # product grid, and the small launches deliberately use half the SMs (DESIGN.md 4 "Scheduling")
                "whole_step": {"tflops": sum(o[2] for o in ops) / (out["ms_per_step"] * 1e-3) / 1e12,
                               "frac_of_sustained_tensor_peak": sum(o[2] for o in ops) / (out["ms_per_step"] * 1e-3) / 1e12 / tf_sust,
                               "gbs": sum(o[3] for o in ops) / (out["ms_per_step"] * 1e-3) / 1e9,
                               "frac_of_hbm_peak": sum(o[3] for o in ops) / (out["ms_per_step"] * 1e-3) / 1e9 / hbm,
                               "ms": out["ms_per_step"]},
            })
        if not args.no_cpu_baseline and world == 1:
            threads = os.cpu_count() or 1
            fps, n, dt = cpu_oracle_fps(ws, synthetic_frames(8, SEED_FRAMES), threads)
            out["cpu_baseline"] = {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port",
                                   "sample": f"{n} frames of the same workload in {dt:.1f} s (torch CPU fp32 oracle, chunks of 4)"}
        print(json.dumps(out))
    for h in host:
        lib.xrseg_host_free(h)
    for p_ in pinned:
        lib.xrseg_host_free(p_[0])
    runner.close()
    pipe.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
