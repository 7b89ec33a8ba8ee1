"""Throughput and decode cost against the class count: BASELINE.json configs[1] shapes (YOLO11n-seg, 640x640, batch 64,
synthetic frames and weights of bench.py's seeds) for models of 1, 80, 365 and 1024 classes.  One JSON line per class count:
frames/s (four runners round-robin on device-resident frames, like bench.py's `value`), the streaming decode filter's time,
bytes (B * A * class pitch * 2) and share of the HBM data-sheet peak, the class convolutions' launch times, and the card's
name and power limit read in the same run.

    python tools/bench_classes.py [--steps 60] [--warmup 10] [--classes 1,80,365,1024]

For nc != 80 the final class bias is set on four frames so that ~1.5 % of the anchors pass the score filter (the frozen
80-class bias of weights.INIT_CLS_BIAS does that for 80 classes)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_PEAK = 7.7e12          # B/s, NVIDIA HGX B200 data sheet, one GPU
SCORE_THR = 0.301


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().split(", ")
    return {"gpu": q[0], "power_limit": q[1] if len(q) > 1 else "unknown"}


def tuned_bias(I, W, frames, nc):
    layers, ws = W.random_weights("n", 1, cls_bias=0.0, nc=nc)
    r = I.Runner(I.Model(W.write_pack("n", layers, ws), "n", nc), max_batch=len(frames), debug=True)
    r.schedule(frames)
    r.wait(strict=False)
    m = np.concatenate([r.fetch(f"cls_logits.{i}").reshape(len(frames), nc, -1).max(axis=1) for i in range(3)], axis=1)
    r.close()
    return float(np.log(SCORE_THR / (1 - SCORE_THR)) - np.quantile(m, 1 - 0.015))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--classes", default="1,80,365,1024")
    args = ap.parse_args()
    import torch

    from bench import SEED_FRAMES, SEED_WEIGHTS, synthetic_frames
    from xr_image_segmentation_b200 import inference as I, weights as W

    B, NSETS = 64, 4
    dev = torch.empty((NSETS, B * 640 * 640 * 3), dtype=torch.uint8, device="cuda:0")
    for s in range(NSETS):
        dev[s].copy_(torch.from_numpy(synthetic_frames(B, SEED_FRAMES + s).reshape(-1)))
    torch.cuda.synchronize()
    info = card()
    for nc in [int(c) for c in args.classes.split(",")]:
        bias = None if nc == 80 else tuned_bias(I, W, synthetic_frames(4, SEED_FRAMES), nc)
        layers, ws = W.random_weights("n", SEED_WEIGHTS, bias, nc=nc)
        model = I.Model(W.write_pack("n", layers, ws), "n", nc)
        runners = [I.Runner(model, max_batch=B, max_candidates=8400, max_det=1000) for _ in range(4)]
        for i in range(args.warmup):
            runners[i % 4].schedule_device(dev[i % NSETS].data_ptr(), B, 640, 640, 3)
        for r in runners:
            r.sync()
        runners[0].event_record(0)
        for i in range(args.steps):
            runners[i % 4].schedule_device(dev[i % NSETS].data_ptr(), B, 640, 640, 3)
        for r in runners:
            r.sync()
        runners[0].event_record(1)
        runners[0].sync()
        ms = runners[0].event_elapsed_ms(0, 1)
        r = runners[0]
        r.schedule_device(dev[0].data_ptr(), B, 640, 640, 3)
        r.wait(strict=False)
        dets = float(r.counts().mean())
        ops = r.profile_ops(20)
        dec = [o for o in ops if o[0] == "post.decode"][0]
        out = {
            "num_classes": nc,
            "cls_bias": bias,
            "frames_per_s": round(args.steps * B / (ms * 1e-3), 1),
            "detections_per_frame": round(dets, 2),
            "post_decode": {"us": round(dec[1] * 1e3, 2), "bytes": dec[3],
                            "hbm_share": round(dec[3] / (dec[1] * 1e-3) / HBM_PEAK, 3)},
            "post_decode_exact_us": round(sum(o[1] for o in ops if o[0] == "post.decode_exact") * 1e3, 2),
            "class_conv_us": {o[0]: round(o[1] * 1e3, 2) for o in ops if o[0].endswith(".cls.2")},
            "config": {"scale": "n", "batch": B, "runners": 4, "steps": args.steps, "hbm_peak_Bps": HBM_PEAK},
            **info,
        }
        print(json.dumps(out), flush=True)
        for r in runners:
            r.close()


if __name__ == "__main__":
    main()
