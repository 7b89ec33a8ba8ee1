"""Developer probe for the GPU box (not a pytest file): runs one named step and prints diagnostics.

  python tests/gpu_probe.py conv_direct | conv_umma [variant] | pipeline direct|umma | bench ...
"""
import os
import sys
import time

import numpy as np
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, ".."))

from xr_image_segmentation_b200 import _lib, inference as I, weights as W  # noqa: E402

CASES = [
    # B, cin, cout, h, w, k, s, act, transposed, residual
    (1, 16, 16, 8, 8, 1, 1, 0, False, False),
    (1, 64, 64, 16, 16, 1, 1, 1, False, False),
    (2, 48, 64, 9, 7, 1, 1, 1, False, True),
    (1, 384, 128, 20, 20, 1, 1, 1, False, False),
    (1, 256, 512, 6, 6, 1, 1, 1, False, False),
    (1, 16, 32, 13, 11, 3, 2, 1, False, False),
    (2, 64, 64, 20, 20, 3, 2, 1, False, False),
    (1, 64, 64, 5, 6, 2, 2, 0, True, False),
    (1, 16, 16, 8, 8, 3, 1, 0, False, False),
    (2, 16, 8, 12, 10, 3, 1, 1, False, True),
    (1, 64, 64, 40, 40, 3, 1, 1, False, False),
    (1, 64, 64, 20, 160, 3, 1, 1, False, False),
    (3, 128, 32, 20, 20, 3, 1, 1, False, True),
    (1, 256, 64, 20, 20, 3, 1, 1, False, False),
    (1, 80, 80, 7, 7, 1, 1, 0, False, False),
]


def torch_conv(x, w, b, k, s, act, tr, res):
    xt = torch.from_numpy(x)
    # the kernels see fp16 inputs / weights: quantize the reference inputs the same way
    xt = xt.half().float()
    wt = torch.from_numpy(w).half().float()
    if tr:
        y = F.conv_transpose2d(xt, wt, torch.from_numpy(b), stride=2)
    else:
        y = F.conv2d(xt, wt, torch.from_numpy(b), stride=s, padding=k // 2)
    if act:
        y = y * torch.sigmoid(y)
    if res is not None:
        y = y + torch.from_numpy(res).half().float()
    return y.numpy()


def step_conv(impl, variant):
    rng = np.random.default_rng(0)
    worst = 0.0
    for (B, cin, cout, h, wd, k, s, act, tr, useres) in CASES:
        x = rng.standard_normal((B, cin, h, wd), dtype=np.float32)
        w = rng.standard_normal((cin, cout, k, k) if tr else (cout, cin, k, k), dtype=np.float32) * np.float32(1.0 / np.sqrt(cin * k * k))
        b = rng.standard_normal(cout, dtype=np.float32)
        ho = h * 2 if tr else (h + 2 * (k // 2) - k) // s + 1
        wo = wd * 2 if tr else (wd + 2 * (k // 2) - k) // s + 1
        res = rng.standard_normal((B, cout, ho, wo), dtype=np.float32) if useres else None
        ref = torch_conv(x, w, b, k, s, act, tr, res)
        t = time.time()
        y = I.debug_conv(x, w, b, k, s, act, tr, res, impl=impl, variant=variant)
        err = float(np.abs(y - ref).max())
        rel = err / (float(np.abs(ref).max()) + 1e-9)
        worst = max(worst, rel)
        print(f"impl={impl} var={variant} case={(B, cin, cout, h, wd, k, s, act, tr, useres)} maxabs={err:.4g} rel={rel:.3g} "
              f"{'OK' if rel < 5e-3 else 'BAD'} ({time.time() - t:.2f}s)", flush=True)
    print("WORST_REL", worst)


def load_golden():
    g = os.path.join(HERE, "..", "tests", "golden")
    model = I.ModelLoader.Load(os.path.join(g, "yolo11n_seg.xrsw"))
    inputs = np.load(os.path.join(g, "inputs.npz"))
    exp = np.load(os.path.join(g, "expected.npz"))
    return model, inputs, exp


def step_pipeline(impl_name):
    impl = _lib.CONV_DIRECT if impl_name == "direct" else _lib.CONV_UMMA
    model, inputs, exp = load_golden()
    r = I.Runner(model, max_batch=1, conv_impl=impl, use_cuda_graph=False)
    for name in inputs.files:
        img = inputs[name]
        t = time.time()
        r.schedule(img[None])
        r.wait()
        dt = time.time() - t
        keep, sc = r.keep_indices()
        boxes = r.readback(0)
        labels = r.readback(1)
        print(name, "n", len(keep), "keep", keep.tolist(), "labels", labels.tolist(), f"{dt * 1e3:.1f} ms", flush=True)
        print("   expected keep", exp[f"{name}.keep"].tolist(), "labels", exp[f"{name}.labels"].tolist())
        if len(keep) == len(exp[f"{name}.keep"]):
            print("   box maxdiff", float(np.abs(boxes - exp[f"{name}.boxes"]).max()))
        inp = r.fetch("input")
        print("   input sample diff", float(np.abs(inp[0, :3, ::16, ::16] - exp[f"{name}.input_sample"]).max()))
        for i in range(3):
            pass
        bl = np.concatenate([r.fetch(f"box_logits.{i}").reshape(1, 64, -1) for i in range(3)], axis=2)[0]
        cl = np.concatenate([r.fetch(f"cls_logits.{i}").reshape(1, 80, -1) for i in range(3)], axis=2)[0]
        head = np.concatenate([bl, cl], axis=0)
        d = np.abs(head[:, ::25] - exp[f"{name}.head_sample"])
        print("   head logits: max abs diff", float(d.max()), "mean", float(d.mean()))
        pr = r.fetch("protos").reshape(32, -1)
        d = np.abs(pr[:, ::64] - exp[f"{name}.proto_sample"])
        print("   protos: max abs diff", float(d.max()), "mean", float(d.mean()))
    r.close()


def step_layers():
    """Per-layer comparison UMMA vs DIRECT runner on one golden frame."""
    model, inputs, exp = load_golden()
    img = inputs["coco139"]
    os.environ.setdefault("XRSEG_FUSE_UP", "0")     # fetch proto.up / proto.cv2 by name: keep them as their own launches
    ra = I.Runner(model, max_batch=1, conv_impl=_lib.CONV_DIRECT, use_cuda_graph=False)
    rb = I.Runner(model, max_batch=1, conv_impl=_lib.CONV_UMMA, use_cuda_graph=False)
    ra.schedule(img[None]); ra.wait()
    rb.schedule(img[None]); rb.wait()
    for l in W.layer_table("n"):
        a = ra.fetch(l.name)
        b = rb.fetch(l.name)
        err = float(np.abs(a - b).max())
        print(f"{l.name:18s} k{l.k} s{l.stride} {l.cin}->{l.cout} @{l.h_in}: maxdiff {err:.4g} ref absmax {float(np.abs(a).max()):.4g}",
              "BAD" if err > 0.05 * (float(np.abs(a).max()) + 1e-3) else "", flush=True)


if __name__ == "__main__":
    step = sys.argv[1]
    if step == "conv_direct":
        step_conv(_lib.CONV_DIRECT, 0)
    elif step == "conv_umma":
        step_conv(_lib.CONV_UMMA, int(sys.argv[2]) if len(sys.argv) > 2 else 0)
    elif step == "pipeline":
        step_pipeline(sys.argv[2])
    elif step == "layers":
        step_layers()
