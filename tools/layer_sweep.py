#!/usr/bin/env python
"""Per-layer error sweep (VERDICT r1 item 2): every named intermediate of the network (xrseg_debug_fetch through
libxrseg_debug.so) against the oracle's fp32 tensor of the same layer, on the committed golden frames.

  python tools/layer_sweep.py [--out gpurun_out/layer_sweep.md] [--frames coco139,coco632,bus]

Per layer: relative L2 error ||gpu - ref|| / ||ref|| and max abs error over the sampled frames, plus the error of the
layer's INPUT (so one can see whether a layer adds error or only passes it on).  Layers whose tensor does not exist in the
fused pipeline (the middle of a fused Bottleneck) or is updated in place later (C2PSA residuals) are marked.
"""
import argparse
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import preprocess as pre  # noqa: E402
from oracle import yolo11seg as Y  # noqa: E402
from xr_image_segmentation_b200 import inference as I, weights as W  # noqa: E402

IN_PLACE = {"b10.attn.proj", "b10.ffn.1"}       # written into the C2PSA `b` slice, which later layers update again
# second convolution of every Bottleneck: its launch adds the Bottleneck input (fused residual)
RESIDUAL = {f"{b}.m0.cv2" for b in ("b2", "b4", "n13", "n16", "n19")} | \
           {f"{b}.m0.{m}.cv2" for b in ("b6", "b8", "n22") for m in ("m0", "m1")}
FUSED_AWAY = {"b2.m0.cv1", "b4.m0.cv1", "n16.m0.cv1"}   # intermediate of the fused Bottleneck lives in shared memory only


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "gpurun_out", "layer_sweep.md"))
    ap.add_argument("--frames", default="coco139,coco632,bus")
    args = ap.parse_args()
    g = os.path.join(ROOT, "tests", "golden")
    model = I.ModelLoader.Load(os.path.join(g, "yolo11n_seg.xrsw"))
    _, layers = W.read_pack(model.pack)
    weights = [(w, b) for _, w, b in layers]
    names = [n for n, _, _ in layers]
    inputs = np.load(os.path.join(g, "inputs.npz"))
    os.environ.setdefault("XRSEG_FUSE_UP", "0")     # proto.up / proto.cv2 as their own launches: the merged launch has no such maps
    r = I.Runner(model, max_batch=1, debug=True)
    acc = {n: [0.0, 0.0, 0.0] for n in names}          # sum sq err, sum sq ref, max abs
    head = {k: [0.0, 0.0, 0.0] for k in ("box_logits", "cls_logits", "coefs", "protos")}
    for fname in args.frames.split(","):
        img = inputs[fname]
        trace = {}
        raw = Y.run_raw(weights, torch.from_numpy(pre.to_tensor(img)), "n", trace=trace)
        r.schedule(img[None])
        r.wait()
        for n in names:
            if n in FUSED_AWAY:
                continue
            if n == "b10.attn.pe":
                continue                                   # the kernel writes pe + attention output (fused residual)
            got = r.fetch(n)[0]
            ref = trace[n][0].numpy()
            if n in RESIDUAL:
                ref = ref + trace["in:" + n[:-1] + "1"][0].numpy()      # Bottleneck: the launch writes x + cv2(cv1(x))
            elif n == "b10.cv1":
                got, ref = got[:got.shape[0] // 2], ref[:ref.shape[0] // 2]   # the second half is the in-place residual target
            d = got - ref
            a = acc[n]
            a[0] += float((d.astype(np.float64) ** 2).sum())
            a[1] += float((ref.astype(np.float64) ** 2).sum())
            a[2] = max(a[2], float(np.abs(d).max()))
        for key, ch in (("box_logits", 64), ("cls_logits", 80), ("coefs", 32)):
            got = np.concatenate([r.fetch(f"{key}.{i}").reshape(ch, -1) for i in range(3)], axis=1).T
            ref = raw[key][0].numpy()
            d = got - ref
            h = head[key]
            h[0] += float((d.astype(np.float64) ** 2).sum()); h[1] += float((ref.astype(np.float64) ** 2).sum())
            h[2] = max(h[2], float(np.abs(d).max()))
        got = r.fetch("protos").reshape(32, -1)
        ref = raw["protos"][0].reshape(32, -1).numpy()
        d = got - ref
        h = head["protos"]
        h[0] += float((d.astype(np.float64) ** 2).sum()); h[1] += float((ref.astype(np.float64) ** 2).sum())
        h[2] = max(h[2], float(np.abs(d).max()))
    r.close()
    lines = [f"# Per-layer error of the GPU network vs the fp32 oracle (product build; frames: {args.frames})", "",
             "relative L2 = ||gpu - oracle|| / ||oracle|| over the whole tensor, fp16 storage on the GPU side.", "",
             "| layer | rel L2 | max abs | note |", "|---|---|---|---|"]
    worst = 0.0
    for n in names:
        a = acc[n]
        if n in FUSED_AWAY:
            lines.append(f"| {n} | - | - | lives in shared memory only (fused Bottleneck) |")
            continue
        if n == "b10.attn.pe":
            lines.append(f"| {n} | - | - | kernel output is pe + attention (fused residual) |")
            continue
        rel = (a[0] / a[1]) ** 0.5 if a[1] > 0 else 0.0
        note = "in-place residual target: holds the block's final value" if n in IN_PLACE else ""
        if n not in IN_PLACE:
            worst = max(worst, rel)
        lines.append(f"| {n} | {rel:.2e} | {a[2]:.3g} | {note} |")
    lines += ["", "| head tensor | rel L2 | max abs |", "|---|---|---|"]
    for k, h in head.items():
        lines.append(f"| {k} | {(h[0] / h[1]) ** 0.5:.2e} | {h[2]:.3g} |")
    lines += ["", f"worst per-layer relative L2 (excluding in-place targets): {worst:.2e}"]
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    open(args.out, "w").write("\n".join(lines) + "\n")
    print("\n".join(lines[-8:]))


if __name__ == "__main__":
    main()
