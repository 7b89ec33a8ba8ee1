"""The kernels before and after the network, element by element, against float64 references fed exactly the operands each
kernel multiplies: the input resample (preprocess_kernel), the decode scores and boxes, the fp16 mask product
(mask_prob_mma_kernel) and the 640-px masks (mask640_kernel); plus the frame-entry paths (pitched rows through each fused stem,
device frames, raw host pointers, micro-batches, graph replays over alternating buffers).

Bounds (u = 2^-24 is the fp32 unit roundoff; U, A_OUT, SUB, ACC and SILU are test_layer_local's constants):

Resample.  Reference: bilinear interpolation in float64 at fx = (x + 0.5) sx - 0.5 with the kernel's fp32 scale sx = w / 640
(letterbox: w / nw), edge clamp, / 255.
  - fp16 output rounding: A_OUT |ref| + SUB.
  - the sample position: fl(fl((x + 0.5) sx) - 0.5) (or one FFMA) is off by <= u (|(x + 0.5) sx| + |fx|); interpolation is
    continuous, so a floor that flips costs nothing extra, and the value moves by at most that times the largest step between
    neighbouring pixels (the interval's and its two neighbours', both rows) / 255.  Same in y.
  - fp32 roundings of the three lerps (the two products, the sum and 1 - t of each) and of the division: <= 8 u M / 255, M the
    largest of the four pixels.
  Exact: letterbox padding is fp16(fl(114 / 255)) bit for bit; the whole tensor also equals oracle/preprocess, rounded to fp16,
  bit for bit (the kernel evaluates the same fp32 operations in the same order).
Mask probabilities (product path).  Reference: sigmoid(z), z = sum_k c16_k p16_k in float64 with the coefficients and the
prototypes rounded to fp16 as the kernel rounds them.  The kernel accumulates on mma.sync in fp32 (ACC (K + 1) S, S = sum |c p|,
K = 32) and evaluates 0.5 tanh.approx(0.5 z) + 0.5: sigmoid' <= 1/4, tanh.approx is off by <= TANH = 2 SILU (2^-10.987, PTX ISA),
0.5 z is exact, the final fmaf rounds once (u):
    |gpu - ref| <= ACC (K + 1) S / 4 + TANH / 2 + 2 u.
640-px masks.  Logits in float64 from the fp32 coefficients and the fp16 prototypes; bilinear at (X + 0.5) 0.25 - 0.5 (exact in
fp32), edge clamp.  E = 1.01 (max over the four source pixels of 32 u S) (the 32-term fp32 FMA chain) + 1.01 * 4 u M (the three
interpolation roundings: two products and a sum per lerp, M the largest |logit| of the four).  A pixel's bit must match wherever
|ref - logit_thr| > E (+ 2 ulp of logf for thresholds other than 0.5); the box crop is fp32 with __f*_rn in a fixed order and is
reproduced in numpy fp32, so outside the box every bit must be 0.  The pixels within E of the threshold are counted and reported.
Scores.  Reference 1 / (1 + exp(-l16)) in float64.  expf is off by <= 2 ulp (CUDA programming guide) = 4 u relative, the sum and
the division round once each; through d s / s = -(1 - s) d e / e:  |gpu - ref| <= 1.01 s (4 u (1 - s) + 2 u).
Boxes.  Reference: the DFL expectation and the anchor decode in float64 on the fp16 box logits.  Per bin, e = expf(l - m) is off by
4 u + u |l - m| (the subtraction may round) relative; the 16-term sum by max(that) + 16 u; each probability by both + u; the
expectation d by sum k p (that + u) + 16 u d; x1 = a - d, x2 = a + d, cx = (x1 + x2) 0.5 s, w = (x2 - x1) s add one rounding each
(0.5 and the stride are powers of two).

Every check prints its largest |err| / bound and where it occurs; a failure names the frame, the detection and the element.
"""
from __future__ import annotations

import math
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
if HERE not in sys.path:
    sys.path.insert(0, HERE)

from oracle import postprocess as pp  # noqa: E402
from oracle import preprocess as pre  # noqa: E402
from xr_image_segmentation_b200 import _lib, inference as I, weights as W  # noqa: E402

from test_gpu_parity import NAMES  # noqa: E402
from test_layer_local import ACC, A_OUT, GOLDEN, SILU, SUB, U, _gpu_name  # noqa: E402

u = 2.0 ** -24            # fp32 unit roundoff
TANH = 2 * SILU           # tanh.approx.f32: max abs error 2^-10.987 (PTX ISA), 1 % slack (test_layer_local's SILU = TANH / 2)
EXPF = 4 * u              # expf: 2 ulp, relative
f32 = np.float32
A = 8400
SIZES = [(80, 80), (40, 40), (20, 20)]
PAD16 = float(np.float16(f32(114) / f32(255)))


# ---- checking and reporting ---------------------------------------------------------------------------------------------
def check(name, gpu, ref, bound, where):
    """Element-wise |gpu - ref| <= bound.  where(index tuple) -> text naming the frame / detection / element."""
    gpu, ref = np.asarray(gpu, np.float64), np.asarray(ref, np.float64)
    assert gpu.shape == ref.shape, (name, gpu.shape, ref.shape)
    bound = np.broadcast_to(np.asarray(bound, np.float64), ref.shape)
    if gpu.size == 0:
        return dict(name=name, ratio=0.0, where="(empty)", n=0, fail=None)
    with np.errstate(invalid="ignore"):
        ratio = np.where(np.isfinite(gpu), np.abs(gpu - ref) / bound, np.inf)
    worst = np.unravel_index(int(np.argmax(ratio)), ratio.shape)
    res = dict(name=name, ratio=float(ratio[worst]), where=where(worst), n=ratio.size, fail=None)
    bad = ~(ratio <= 1.0)
    if bad.any():
        i = tuple(int(v) for v in np.argwhere(bad)[0])
        res["fail"] = (f"{name}: first offending element {where(i)}: gpu {gpu[i]:.9g} ref {ref[i]:.9g} bound {bound[i]:.3g} "
                       f"({int(bad.sum())} of {bad.size} elements out of bound)")
    return res


def settle(results, extra=()):
    for r in results:
        print(f"{r['name']:44s} max|err|/bound {r['ratio']:8.3g} at {r['where']} ({r['n']} elements)")
    for line in extra:
        print(line)
    fails = [r["fail"] for r in results if r["fail"]]
    assert not fails, "\n".join(fails)


def r16(a):
    return np.asarray(a, np.float32).astype(np.float16).astype(np.float64)


# ---- resample reference ----------------------------------------------------------------------------------------------
def placement(h, w, letterbox):
    """(nh, nw, top, left, scale_y, scale_x) as the host computes them (xrseg_api.cu preprocess)."""
    if not letterbox:
        return 640, 640, 0, 0, f32(h) / f32(640), f32(w) / f32(640)
    rr = min(640.0 / h, 640.0 / w)
    nh, nw = int(round(h * rr)), int(round(w * rr))          # half to even, like nearbyint
    return nh, nw, (640 - nh) // 2, (640 - nw) // 2, f32(h) / f32(nh), f32(w) / f32(nw)


def _axis(n_in, scale, offset):
    o = np.arange(640, dtype=np.float64) - offset
    p = (o + 0.5) * float(scale)                              # exact in float64
    f = p - 0.5
    i0f = np.floor(f)
    t = f - i0f
    clip = lambda v: np.clip(v, 0, n_in - 1).astype(np.int64)  # noqa: E731
    steps = [(clip(i0f + j), clip(i0f + j + 1)) for j in (-1, 0, 1)]   # the interval and its two neighbours
    return clip(i0f), clip(i0f + 1), t, u * (np.abs(p) + np.abs(f)), steps


def resample_ref(img, letterbox):
    """img uint8 [H,W,C] (top row first) -> (ref [3,640,640], bound [3,640,640]) in float64; padding exact."""
    h, w = img.shape[:2]
    nh, nw, top, left, sy, sx = placement(h, w, letterbox)
    I3 = img[..., :3].astype(np.float64)
    y0, y1, ty, dy, ysteps = _axis(h, sy, top)
    x0, x1, tx, dx, xsteps = _axis(w, sx, left)
    g = lambda ys, xs: I3[ys[:, None], xs[None, :]]           # noqa: E731  [640,640,3]
    a, b, c, d = g(y0, x0), g(y0, x1), g(y1, x0), g(y1, x1)
    txx, tyy = tx[None, :, None], ty[:, None, None]
    ref = ((a * (1 - txx) + b * txx) * (1 - tyy) + (c * (1 - txx) + d * txx) * tyy) / 255.0
    Dx = np.max([np.abs(g(r, s1) - g(r, s0)) for r in (y0, y1) for s0, s1 in xsteps], axis=0)
    Dy = np.max([np.abs(g(s1, q) - g(s0, q)) for q in (x0, x1) for s0, s1 in ysteps], axis=0)
    M = np.maximum(np.maximum(a, b), np.maximum(c, d))
    bound = A_OUT * np.abs(ref) + 1.01 * (dx[None, :, None] * Dx + dy[:, None, None] * Dy + 8 * u * M) / 255.0 + SUB
    inside = np.zeros((640, 640), bool)
    inside[top:top + nh, left:left + nw] = True
    ref[~inside] = PAD16                                      # padding: exact
    bound[~inside] = 2.0 ** -80
    return ref.transpose(2, 0, 1), bound.transpose(2, 0, 1)


def oracle_input(img, letterbox):
    return r16(pre.letterbox(img) if letterbox else pre.to_tensor(img))[0]


def check_resample(label, got, refs):
    """got [B,3,640,640] (fetch("input")) against the float64 references; returns the check results."""
    res = []
    for f, (ref, bound) in enumerate(refs):
        res.append(check(f"{label} frame {f}", got[f], ref, bound, lambda i, f=f: f"frame {f} channel {i[0]} y {i[1]} x {i[2]}"))
    return res


# ---- post-processing references ---------------------------------------------------------------------------------------
def anchor(scale, gx, gy):
    return (0, 6400, 8000)[scale] + gy * (80, 40, 20)[scale] + gx


def anchor_geometry(a):
    """(anchor centre x, y in grid units, stride) of anchor a."""
    for (h, w), off, s in zip(SIZES, (0, 6400, 8000), (8, 16, 32)):
        if a < off + h * w:
            gy, gx = divmod(a - off, w)
            return gx + 0.5, gy + 0.5, s
    raise IndexError(a)


def dfl_ref(bl16, anchors):
    """float64 boxes (cx, cy, w, h) of the listed anchors and their bounds, from fp16-rounded box logits [n,64]."""
    n = len(anchors)
    l = bl16.reshape(n, 4, 16)
    m = l.max(2, keepdims=True)
    e = np.exp(l - m)
    p = e / e.sum(2, keepdims=True)
    k = np.arange(16.0)
    d = (p * k).sum(2)                                        # [n,4]: left, top, right, bottom
    rel_e = EXPF + u * np.abs(l - m)
    rel_p = rel_e + (rel_e.max(2, keepdims=True) + 16 * u) + u
    ed = 1.01 * ((p * k * (rel_p + u)).sum(2) + 16 * u * d)
    geo = np.array([anchor_geometry(int(a)) for a in anchors], np.float64).reshape(n, 3)
    ax, ay, st = geo[:, 0], geo[:, 1], geo[:, 2]
    x1, y1, x2, y2 = ax - d[:, 0], ay - d[:, 1], ax + d[:, 2], ay + d[:, 3]
    ex1, ey1 = ed[:, 0] + u * np.abs(x1), ed[:, 1] + u * np.abs(y1)
    ex2, ey2 = ed[:, 2] + u * np.abs(x2), ed[:, 3] + u * np.abs(y2)
    box = np.stack([(x1 + x2) * 0.5 * st, (y1 + y2) * 0.5 * st, (x2 - x1) * st, (y2 - y1) * st], 1)
    bound = 1.01 * np.stack([0.5 * st * (ex1 + ex2 + u * np.abs(x1 + x2)), 0.5 * st * (ey1 + ey2 + u * np.abs(y1 + y2)),
                             st * (ex1 + ex2 + u * np.abs(x2 - x1)), st * (ey1 + ey2 + u * np.abs(y2 - y1))], 1)
    return box, bound


def score_ref(l16):
    s = 1.0 / (1.0 + np.exp(-l16))
    return s, 1.01 * s * (EXPF * (1.0 - s) + 2 * u)


def prob_ref(c16, p16):
    """c16 [n,32], p16 [32,P] float64 -> (sigmoid(z), bound) [n,P]."""
    z = c16 @ p16
    S = np.abs(c16) @ np.abs(p16)
    return 1.0 / (1.0 + np.exp(-z)), ACC * (32 + 1) * S / 4 + TANH / 2 + 2 * u


_X = np.arange(640)
_F = np.maximum((_X + 0.5) * 0.25 - 0.5, 0.0)
_I0 = np.minimum(np.floor(_F).astype(np.int64), 159)
_I1 = np.minimum(_I0 + 1, 159)
_WT = _F - _I0


def up640_ref(c, p16):
    """c [32] fp32 coefficients, p16 [32,25600] -> (bilinear logits [640,640], E [640,640]) in float64."""
    L = (c.astype(np.float64) @ p16).reshape(160, 160)
    Ec = 1.01 * 32 * u * (np.abs(c.astype(np.float64)) @ np.abs(p16)).reshape(160, 160)
    q = lambda T, ys, xs: T[ys][:, xs]                        # noqa: E731
    a, b, cc, d = q(L, _I0, _I0), q(L, _I0, _I1), q(L, _I1, _I0), q(L, _I1, _I1)
    wx, wy = _WT[None, :], _WT[:, None]
    val = (a * (1 - wx) + b * wx) * (1 - wy) + (cc * (1 - wx) + d * wx) * wy
    E4 = np.maximum(np.maximum(q(Ec, _I0, _I0), q(Ec, _I0, _I1)), np.maximum(q(Ec, _I1, _I0), q(Ec, _I1, _I1)))
    M = np.maximum(np.maximum(np.abs(a), np.abs(b)), np.maximum(np.abs(cc), np.abs(d)))
    return val, E4 + 1.01 * 4 * u * M


def box_inside(raw):
    """mask640_kernel's crop predicate in numpy fp32 (same operations, same order): bool [640,640]."""
    cx, cy, w, h = (f32(v) for v in raw)
    x1, x2 = f32(cx - f32(w * f32(0.5))), f32(cx + f32(w * f32(0.5)))
    y1, y2 = f32(cy - f32(h * f32(0.5))), f32(cy + f32(h * f32(0.5)))
    xs = np.arange(640, dtype=f32)
    return ((xs >= y1) & (xs < y2))[:, None] & ((xs >= x1) & (xs < x2))[None, :]


def logit_threshold(thr):
    """(float64 logit the kernel compares with, its uncertainty): thr <= 0 -> everything inside the box."""
    if thr < 0:
        return -3.0e38, 0.0
    t = f32(thr)
    if t == f32(0.5):
        return 0.0, 0.0
    lg = math.log(float(t / f32(f32(1) - t)))                # the host's fp32 quotient, then logf (<= 2 ulp here)
    return lg, 2 * 2.0 ** -23 * abs(lg) + 2.0 ** -149


def check_bits(name, got, val, E, inside, thr, where):
    """got uint8 [640,640] against the reference logits: exact outside the box, exact inside wherever decidable."""
    lt, margin = logit_threshold(thr)
    decid = np.abs(val - lt) > E + margin
    want = inside & (val > lt)
    bad = (got > 1) | (~inside & (got != 0)) | (inside & decid & (got != want))
    und = int((inside & ~decid).sum())
    res = dict(name=name, n_inside=int(inside.sum()), undecidable=und, fail=None)
    if bad.any():
        y, x = (int(v) for v in np.argwhere(bad)[0])
        res["fail"] = (f"{name}: first offending pixel {where} y {y} x {x}: gpu bit {int(got[y, x])}, inside box {bool(inside[y, x])}, "
                       f"ref logit {val[y, x]:.6g} threshold {lt:.6g} E {E[y, x]:.3g} ({int(bad.sum())} pixels wrong)")
    return res


# ---- designed post-processing tensors ---------------------------------------------------------------------------------
POST_COUNTS = [0, 1, 0, 15, 16, 17, 0, 63, 64, 65, 129, 0, 300]   # kept detections per frame; a geometry frame follows
# (scale, gx, gy, (left, top, right, bottom) in grid units, what the 640-px mask exercises)
GEOMETRY = [
    (0, 7, 15, (1.0, 1.0, 1.0, 1.0), "straddles x = 64 and y = 128"),
    (1, 11, 3, (0.75, 0.5, 0.6, 0.75), "straddles x = 192 and y = 64"),
    (0, 20, 20, (0.5, 0.5, 0.5, 0.5), "inside one 64-px tile"),
    (0, 50, 60, (0.03, 0.5, 0.03, 0.5), "narrower than 1 px"),
    (0, 70, 5, (0.02, 0.02, 0.02, 0.02), "narrower and lower than 1 px"),
    (2, 19, 0, (3.0, 3.0, 3.0, 3.0), "partly outside the frame"),
    (2, 9, 9, (14.5, 14.5, 14.5, 14.5), "the full frame"),
]


def _side_logits(d):
    row = np.full(16, -12.0)
    k0 = min(int(math.floor(d)), 15)
    fr = d - k0
    row[k0] = math.log(1 - fr) if fr < 1 else -12.0
    if fr > 0 and k0 < 15:
        row[k0 + 1] = math.log(fr)
    return row


def designed_post(nc, seed=0):
    """Head tensors whose result is known in advance.  Planted objects are boxes of < 4 px on distinct anchors (anchor centres
    of different anchors lie >= 4 px apart, so no two boxes overlap: NMS keeps all of them), plus the GEOMETRY frame, whose
    boxes overlap by IoU < 0.05 at most; every other class logit sits near -8.  Mask coefficients scale by 0.02 .. 3 per anchor
    over N(0, 1) prototypes: mask logits from ~0 to saturation, all far inside the fp16 range."""
    rng = np.random.default_rng(seed)
    B = len(POST_COUNTS) + 1
    box = rng.normal(0.0, 0.3, (B, A, 64)).astype(f32)
    box.reshape(B, A, 4, 16)[..., 0] += f32(9.0)              # d ~ 0.02 grid units: boxes of < 4 px
    cls = np.minimum(rng.normal(-8.0, 0.5, (B, A, nc)), -5.0).astype(f32)
    planted = []
    for f, n in enumerate(POST_COUNTS):
        a = rng.choice(A, n, replace=False)
        cls[f, a, rng.integers(0, nc, n)] = rng.uniform(0.0, 4.0, n)
        planted.append(n)
    g = B - 1
    for s, gx, gy, sides, _ in GEOMETRY:
        a = anchor(s, gx, gy)
        box[g, a] = np.concatenate([_side_logits(d) for d in sides]).astype(f32)
        cls[g, a, rng.integers(0, nc)] = 3.0 + rng.uniform(0.0, 1.0)
    planted.append(len(GEOMETRY))
    coefs = (rng.standard_normal((B, A, 32)) * np.exp(rng.uniform(np.log(0.02), np.log(3.0), (B, A, 1)))).astype(f32)
    protos = rng.standard_normal((B, 32, 160 * 160)).astype(f32)
    return box, cls, coefs, protos, planted


def oracle_keep(box16, cls16):
    """Keep indices, labels, fp32 scores and boxes of the oracle's decode + NMS on one frame (no masks)."""
    ax, ay, st = pp.make_anchors(SIZES)
    boxes = pp.dfl_decode(box16.astype(f32), ax, ay, st)
    score, label = pp.class_scores(cls16.astype(f32))
    keep = pp.nms_onnx(pp.cxcywh_to_corners(boxes), score, 0.43, 0.301, 300)
    return keep, label[keep], score[keep], boxes[keep]


def post_runner(nc, batch):
    layers, ws = W.random_weights("n", 1, cls_bias=-5.0, nc=nc)
    return I.Runner(I.Model(W.write_pack("n", layers, ws), "n", nc), max_batch=batch, debug=True)


def run_post(r, box, cls, coefs, protos):
    r.debug_post(box, cls, coefs, protos, f16=True)
    r.wait()
    keep, scores = r.keep_indices()
    return dict(counts=r.counts().copy(), keep=keep, scores=scores, boxes=r.readback(0), labels=r.readback(1),
                coefs=r.readback(2), probs=r.readback(3))


def check_post(out, box, cls, coefs, protos, planted, label):
    """Exact and bounded checks of one debug_post_f16 run; returns (results, report lines)."""
    counts = out["counts"]
    offs = np.concatenate([[0], np.cumsum(counts)])
    results, lines, exact = [], [], []
    bit_equal = total = 0
    for f in range(len(counts)):
        b16, c16 = r16(box[f]), r16(cls[f])
        keep, labels, oscores, _ = oracle_keep(b16, c16)
        n = int(counts[f])
        sl = slice(offs[f], offs[f + 1])
        assert n == len(keep) == planted[f], f"{label}: frame {f} kept {n}, oracle {len(keep)}, planted {planted[f]}"
        assert out["keep"][sl].tolist() == keep.tolist(), f"{label}: frame {f} keep indices differ"
        assert out["labels"][sl].tolist() == labels.tolist(), f"{label}: frame {f} labels differ"
        assert np.array_equal(out["coefs"][sl], coefs[f][keep].astype(np.float16).astype(f32)), f"{label}: frame {f} coefficients"
        if n == 0:
            continue
        name = lambda i, f=f: f"frame {f} detection {i[0]}" + (f" element {i[1]}" if len(i) > 1 else "")   # noqa: E731
        s_ref, s_bound = score_ref(c16[keep, labels])
        results.append(check(f"{label} scores f{f}", out["scores"][sl], s_ref, s_bound, name))
        bit_equal += int(np.sum(out["scores"][sl] == oscores))
        total += n
        b_ref, b_bound = dfl_ref(b16[keep], keep)
        results.append(check(f"{label} boxes f{f}", out["boxes"][sl], b_ref, b_bound, name))
        p_ref, p_bound = prob_ref(r16(coefs[f][keep]), r16(protos[f]))
        results.append(check(f"{label} mask probs f{f}", out["probs"][sl].reshape(n, -1), p_ref, p_bound,
                             lambda i, f=f: f"frame {f} detection {i[0]} y {i[1] // 160} x {i[1] % 160}"))
        exact.append(f)
    lines.append(f"{label}: counts {counts.tolist()} exact (keep, labels, coefficients) on every frame; scores bit-equal to the "
                 f"oracle's fp32 all_scores on {bit_equal} of {total} detections")
    return results, lines


def mask640_ranges(counts):
    """(first, count) ranges of output rows: the whole geometry frame, two detections of frames 5 (17 kept) and 10 (129),
    and the last detection of frame 12 (300)."""
    offs = np.concatenate([[0], np.cumsum(counts)])
    g = len(counts) - 1
    return [(int(offs[g]), int(counts[g])), (int(offs[5]), 2), (int(offs[10]) + 64, 2), (int(offs[13]) - 1, 1)]


# ---- CPU: the checkers against simulated kernels -------------------------------------------------------------------------
@pytest.mark.parametrize("hw,letterbox", [((5, 7), False), ((5, 7), True), ((23, 37), True), ((1, 1), False), ((640, 9), True)])
def test_resample_checker_passes_faithful_outputs_and_names_a_moved_element(hw, letterbox):
    rng = np.random.default_rng(sum(hw))
    img = rng.integers(0, 256, hw + (3,), dtype=np.uint8)
    ref, bound = resample_ref(img, letterbox)
    for sim in (r16(ref), oracle_input(img, letterbox)):     # the reference as the kernel stores it; the fp32 oracle, in fp16
        assert not check("resample", sim, ref, bound, str)["fail"]
    idx = (1, 320, 320)
    moved = r16(ref)
    moved[idx] += 2 * bound[idx]
    res = check("resample", moved[None], ref[None], bound[None], lambda i: f"frame {i[0]} channel {i[1]} y {i[2]} x {i[3]}")
    assert res["fail"] and "frame 0 channel 1 y 320 x 320:" in res["fail"], res["fail"]
    if letterbox:                                            # padding is exact: one fp16 step off fails
        nh, nw, top, left, _, _ = placement(*hw, True)
        py, px = (top - 1, 10) if top > 0 else (10, left - 1)
        moved = r16(ref)
        moved[0, py, px] = float(np.nextafter(np.float16(PAD16), np.float16(1)))
        assert check("pad", moved, ref, bound, str)["fail"]


def test_post_checkers_pass_faithful_outputs_and_name_a_moved_element():
    rng = np.random.default_rng(3)
    n = 5
    c16 = r16(rng.standard_normal((n, 32)) * np.exp(rng.uniform(-4, 1, (n, 1))))
    p16 = r16(rng.standard_normal((32, 25600)))
    p_ref, p_bound = prob_ref(c16, p16)
    where = lambda i: f"frame 2 detection {i[0]} y {i[1] // 160} x {i[1] % 160}"     # noqa: E731
    assert not check("probs", p_ref.astype(f32), p_ref, p_bound, where)["fail"]
    assert not check("probs", pp.mask_probs(c16, p16).reshape(n, -1), p_ref, p_bound, where)["fail"]   # the fp32 oracle
    moved = p_ref.astype(f32).astype(np.float64)
    moved[3, 161 * 7] += 2 * p_bound[3, 161 * 7]
    assert "frame 2 detection 3 y 7 x 7:" in check("probs", moved, p_ref, p_bound, where)["fail"]
    l16 = r16(rng.uniform(-0.8, 9, 40))
    s_ref, s_bound = score_ref(l16)
    score32, _ = pp.class_scores(l16.astype(f32)[:, None])
    assert not check("scores", s_ref.astype(f32), s_ref, s_bound, str)["fail"]
    assert not check("scores", score32, s_ref, s_bound, str)["fail"]
    moved = s_ref.astype(f32).astype(np.float64)
    moved[17] -= 2 * s_bound[17]
    assert "(17,)" in check("scores", moved, s_ref, s_bound, str)["fail"]
    anchors = np.array([0, 6399, 6400, 8399, 4321])
    b16 = r16(rng.normal(0, 2, (5, 64)))
    b_ref, b_bound = dfl_ref(b16, anchors)
    ax, ay, st = pp.make_anchors(SIZES)
    ob = pp.dfl_decode(b16.astype(f32), ax[anchors], ay[anchors], st[anchors])
    assert not check("boxes", ob, b_ref, b_bound, str)["fail"]
    moved = ob.astype(np.float64)
    moved[2, 3] += 2 * b_bound[2, 3]
    assert "(2, 3)" in check("boxes", moved, b_ref, b_bound, str)["fail"]


def test_mask640_checker_passes_faithful_bits_and_names_a_flipped_pixel():
    rng = np.random.default_rng(4)
    c = r16(rng.standard_normal(32)).astype(f32)
    p16 = r16(rng.standard_normal((32, 25600)))
    raw = np.array([300.5, 200.25, 130.0, 97.0], f32)
    val, E = up640_ref(c, p16)
    inside = box_inside(raw)
    oracle = pp.upsample_mask_640(pp.mask_logits(c[None], p16)[0].reshape(160, 160), raw)   # a faithful fp32 kernel
    res = check_bits("m640", oracle, val, E, inside, 0.5, "frame 0 detection 0")
    assert not res["fail"] and res["undecidable"] < 0.01 * res["n_inside"], res
    for thr in (0.3, 0.7, -1.0):
        lt, _ = logit_threshold(thr)
        assert not check_bits("m640", (inside & (val > lt)).astype(np.uint8), val, E, inside, thr, "f0")["fail"]
    y, x = np.argwhere(inside & (np.abs(val) > 10 * E))[0]
    flipped = oracle.copy()
    flipped[y, x] ^= 1
    assert f"y {y} x {x}:" in check_bits("m640", flipped, val, E, inside, 0.5, "frame 0 detection 0")["fail"]
    flipped = oracle.copy()
    flipped[5, 5] = 1                                        # outside the box
    assert "y 5 x 5:" in check_bits("m640", flipped, val, E, inside, 0.5, "frame 0 detection 0")["fail"]


@pytest.mark.parametrize("nc", [80, 3, 365])
def test_designed_tensors_give_the_planned_detections(nc):
    """The oracle keeps every planted object on the designed tensors, and the geometry frame's boxes land where planned."""
    box, cls, _, _, planted = designed_post(nc)
    for f in range(len(planted)):
        keep, _, _, boxes = oracle_keep(r16(box[f]), r16(cls[f]))
        assert len(keep) == planted[f], (f, len(keep), planted[f])
    keep, _, _, b = oracle_keep(r16(box[-1]), r16(cls[-1]))
    geo = {anchor(s, gx, gy): what for s, gx, gy, _, what in GEOMETRY}
    x1, x2 = b[:, 0] - b[:, 2] / 2, b[:, 0] + b[:, 2] / 2
    y1, y2 = b[:, 1] - b[:, 3] / 2, b[:, 1] + b[:, 3] / 2
    for i, a in enumerate(keep):
        what = geo[int(a)]
        if what.startswith("straddles"):
            assert np.floor(x1[i] / 64) != np.floor(x2[i] / 64) and np.floor(y1[i] / 64) != np.floor(y2[i] / 64), what
        elif what == "inside one 64-px tile":
            assert np.floor(x1[i] / 64) == np.floor(x2[i] / 64) and np.floor(y1[i] / 64) == np.floor(y2[i] / 64)
        elif what.startswith("narrower"):
            assert b[i, 2] < 1
        elif what == "partly outside the frame":
            assert x2[i] > 640 and y1[i] < 0 and x1[i] > 0
        else:
            assert x1[i] < 0 and y1[i] < 0 and x2[i] > 640 and y2[i] > 640


# ---- GPU: post side ----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def post80(lib):
    box, cls, coefs, protos, planted = designed_post(80)
    r = post_runner(80, len(planted))
    out = run_post(r, box, cls, coefs, protos)
    yield r, out, (box, cls, coefs, protos, planted)
    r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("nc", [80, 3, 365])
def test_post_on_designed_tensors_exact_and_within_bounds(post80, nc):
    """debug_post_f16 on tensors whose result is known: counts 0 / 1 / 15 / 16 / 17 / 63 / 64 / 65 / 129 / 300 (the MMA tile
    edge, the 64-detection staging edge, frame offsets, exactly max_det) with empty frames between; 80, 3 and 365 classes run the
    specialised, the nc and the wide decode filter."""
    if nc == 80:
        _, out, (box, cls, coefs, protos, planted) = post80
    else:
        box, cls, coefs, protos, planted = designed_post(nc)
        r = post_runner(nc, len(planted))
        out = run_post(r, box, cls, coefs, protos)
        r.close()
    print(_gpu_name())
    results, lines = check_post(out, box, cls, coefs, protos, planted, f"nc {nc}")
    settle(results, lines)


@pytest.mark.gpu
def test_640_masks_on_debug_post_f16_tensors(post80):
    """XRSEG_MASK_UPSAMPLE_640 after debug_post_f16 reads the caller's prototypes (it once read the network arena's), at
    thresholds 0.5, 0.3, 0.7 and negative (exactly 0), on boxes that straddle tile edges, sit inside one tile, are narrower than
    a pixel, leave the frame or cover it, and on detections of other frames."""
    r, out, (box, cls, coefs, protos, planted) = post80
    counts = out["counts"]
    frame_of = np.repeat(np.arange(len(counts)), counts)
    offs = np.concatenate([[0], np.cumsum(counts)])
    refs = {}
    fails, lines = [], [_gpu_name()]
    for thr in (0.5, 0.3, 0.7, -1.0):
        n_in = n_und = 0
        for first, count in mask640_ranges(counts):
            got = r.masks(_lib.MASK_UPSAMPLE_640, first=first, count=count, threshold=thr)
            for j in range(count):
                o = first + j
                f = int(frame_of[o])
                if o not in refs:
                    refs[o] = up640_ref(out["coefs"][o], r16(protos[f]))
                val, E = refs[o]
                res = check_bits(f"640 mask thr {thr}", got[j], val, E, box_inside(out["boxes"][o]), thr,
                                 f"frame {f} detection {o - offs[f]}")
                n_in, n_und = n_in + res["n_inside"], n_und + res["undecidable"]
                if res["fail"]:
                    fails.append(res["fail"])
        lines.append(f"640 masks, threshold {thr}: {n_in} pixels inside the boxes of {len(refs)} detections, {n_und} within E of "
                     f"the threshold (undecidable), {len(fails)} failures so far")
        assert n_und <= 1e-3 * n_in, lines[-1]
    print("\n".join(lines))
    assert not fails, "\n".join(fails[:10])


@pytest.mark.gpu
def test_640_masks_after_fp32_debug_post_are_refused(lib):
    """The fp32 debug path keeps its prototypes planar in fp32, which the 640-px kernel cannot read: the call says so."""
    box, cls, coefs, protos, _ = designed_post(80)
    r = post_runner(80, 1)
    r.debug_post(box[-1:], cls[-1:], coefs[-1:], protos[-1:])
    r.wait()
    assert r.counts()[0] == len(GEOMETRY)
    with pytest.raises(I.XrsegError) as e:
        r.masks(_lib.MASK_UPSAMPLE_640)
    assert e.value.code == _lib.ERR_STATE and "debug_post_f16" in str(e.value)
    r.close()


# ---- GPU: input side ---------------------------------------------------------------------------------------------------
RESAMPLE_SIZES = [(1, 1), (7, 5), (64, 64), (639, 640), (640, 639), (641, 641), (1280, 720), (1920, 1080), (3840, 2160),
                  (4000, 120), (120, 4000), (973, 733)]   # W x H


def place(frames, pitch, offset=0, seed=99):
    """frames [B,H,W,C] copied into a fresh buffer with rows `pitch` bytes apart (random bytes in the padding), starting
    `offset` bytes past a 16-byte boundary; returns the [B,H,W,C] view."""
    B, H, Wd, C = frames.shape
    raw = np.random.default_rng(seed).integers(0, 256, B * H * pitch + 64, dtype=np.uint8)
    base = (-raw.ctypes.data) % 16 + offset
    buf = raw[base:base + B * H * pitch].reshape(B, H, pitch)
    buf[:, :, :Wd * C] = frames.reshape(B, H, Wd * C)
    view = np.lib.stride_tricks.as_strided(buf, shape=frames.shape, strides=(H * pitch, pitch, C, 1))
    assert view.ctypes.data % 16 == offset % 16
    return view


@pytest.mark.gpu
@pytest.mark.parametrize("letterbox", [False, True], ids=["stretch", "letterbox"])
def test_resample_matrix_within_bounds_and_equal_to_the_oracle(golden, letterbox):
    """preprocess_kernel at upscales from 1x1 / 7x5, extreme aspect ratios (nh or nw ~ 19 px), sizes one pixel off 640 and
    camera sizes; RGB and RGBA, top-down and bottom-up, packed and with padded rows (random bytes in the padding)."""
    mode = _lib.RESIZE_LETTERBOX if letterbox else _lib.RESIZE_STRETCH
    r = I.Runner(golden["model"], max_batch=2, resize_mode=mode, debug=True)
    results, lines = [], [_gpu_name()]
    rng = np.random.default_rng(7)
    for (w, h) in RESAMPLE_SIZES:
        pics = rng.integers(0, 256, (2, h, w, 3), dtype=np.uint8)
        refs = [resample_ref(p, letterbox) for p in pics]
        oracle = [oracle_input(p, letterbox) for p in pics]
        worst = 0.0
        for c in (3, 4):
            frames = pics if c == 3 else np.concatenate([pics, rng.integers(0, 256, (2, h, w, 1), dtype=np.uint8)], 3)
            for bottom_up in (False, True):
                mem = frames[:, ::-1] if bottom_up else frames
                for pitch in (w * c, w * c + 7):
                    view = place(np.ascontiguousarray(mem), pitch)
                    r.schedule(view, bottom_up=bottom_up, stride_bytes=pitch)
                    r.wait(strict=False)
                    got = r.fetch("input")
                    label = f"{w}x{h} {'RGBA' if c == 4 else 'RGB'} {'bottom-up' if bottom_up else 'top-down'} pitch {pitch}"
                    res = check_resample(label, got, refs)
                    results += [x for x in res if x["fail"]]
                    worst = max([worst] + [x["ratio"] for x in res])
                    for f in range(2):
                        nd = int(np.sum(got[f] != oracle[f]))
                        assert nd == 0, f"{label}: frame {f}: {nd} elements differ from oracle/preprocess in fp16"
        nh, nw, *_ = placement(h, w, letterbox)
        lines.append(f"resample {'letterbox' if letterbox else 'stretch'} {w}x{h} (placed {nw}x{nh}): worst |err|/bound over 8 "
                     f"variants {worst:.3g}; bit-equal to the oracle")
    settle(results, lines)
    r.close()


def stem_kernel(addr, pitch, c):
    """The fused stem a 640x640 frame selects (xrseg_api.cu OP_STEM)."""
    if addr % 16 == 0 and pitch % 16 == 0 and c == 3:
        return "stem_rows"
    if addr % 4 == 0 and pitch % 4 == 0:
        return "stem_mma"
    return "stem_u8"


def golden_640(n):
    """n 640x640 uint8 frames with real content: the sample frames stretched on the host, then mirrored."""
    g = np.load(os.path.join(GOLDEN, "inputs.npz"))
    out = []
    for i in range(n):
        x = pre.to_tensor(g[NAMES[i % len(NAMES)]])[0].transpose(1, 2, 0)
        u8 = np.rint(x * 255.0).astype(np.uint8)
        out.append(u8[:, ::-1] if i >= len(NAMES) else u8)
    return np.ascontiguousarray(np.stack(out))


def outputs(r, fetch_b0=False):
    keep, scores = r.keep_indices()
    o = dict(counts=r.counts().copy(), keep=keep, scores=scores, boxes=r.readback(0), labels=r.readback(1), coefs=r.readback(2),
             probs=r.readback(3), bits=r.masks(_lib.MASK_BITS_160))
    if fetch_b0:
        o["b0"] = r.fetch("b0")
    return o


def assert_same(a, b, what):
    for k in a:
        assert np.array_equal(a[k], b[k]), f"{what}: {k} differs"


STEM_CASES = [   # (kernel, channels, pitch of the padded frame, buffer offset of the packed twin)
    ("stem_rows", 3, 1936, 0), ("stem_mma", 3, 1924, 4), ("stem_mma", 4, 2564, 0), ("stem_u8", 3, 1921, 1)]


def dev_place(frames, pitch, offset):
    """frames [B,H,W,C] in GPU memory with rows `pitch` bytes apart, starting `offset` bytes past a 16-byte boundary (host
    frames go through the runner's own staging buffer, whose alignment is the allocator's): (device address, owning tensor)."""
    import torch
    B, H, Wd, C = frames.shape
    t = torch.randint(0, 256, (B * H * pitch + 64,), dtype=torch.uint8, device="cuda")
    base = (-t.data_ptr()) % 16 + offset
    t[base:base + B * H * pitch].view(B, H, pitch)[:, :, :Wd * C] = torch.from_numpy(frames.reshape(B, H, Wd * C)).cuda()
    return t.data_ptr() + base, t


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,c,pitch,twin_offset", STEM_CASES, ids=[f"{k}_c{c}_{p}" for k, c, p, _ in STEM_CASES])
def test_pitched_640_frames_equal_their_packed_twin(golden, kernel, c, pitch, twin_offset):
    """Padded rows through each fused stem: the stem output and every result bit-identical to a packed frame that selects the
    same kernel.  The frames sit in device memory, where the kernel choice reads the address."""
    frames = golden_640(2)
    if c == 4:
        frames = np.concatenate([frames, np.random.default_rng(5).integers(0, 256, (2, 640, 640, 1), dtype=np.uint8)], 3)
    twin, keep_twin = dev_place(frames, 640 * c, twin_offset)
    padded, keep_padded = dev_place(frames, pitch, 0)
    assert stem_kernel(twin, 640 * c, c) == kernel == stem_kernel(padded, pitch, c)
    r = I.Runner(golden["model"], max_batch=2, debug=True)
    r.schedule_device(twin, 2, 640, 640, c)
    r.wait()
    want = outputs(r, fetch_b0=True)
    r.schedule_device(padded, 2, 640, 640, c, stride_bytes=pitch)
    r.wait()
    got = outputs(r, fetch_b0=True)
    assert int(want["counts"].sum()) > 0
    assert_same(want, got, f"{kernel}, pitch {pitch}")
    r.schedule(place(frames, pitch), stride_bytes=pitch)      # host frames: the staging copy is aligned, the pitch decides
    r.wait()
    assert_same(want, outputs(r, fetch_b0=True), f"{kernel}, pitch {pitch}, from host memory")
    print(f"{kernel} RGB{'A' if c == 4 else ''}: pitch {pitch} bit-identical to the packed twin (offset {twin_offset}), "
          f"{int(want['counts'].sum())} detections")
    r.close()


@pytest.mark.gpu
def test_device_and_pointer_entry_points_equal_host_frames(golden):
    """schedule_device (the benchmark's path) and schedule from a raw host pointer give exactly what schedule() gives on a host
    copy, for 640x640 frames (fused stem) and 1280x720 frames (resample); a graph-capturing runner fed two device buffers in
    turn reproduces each buffer's own result every time (the stem sits outside the graph and reads a pointer that changes)."""
    import torch
    r = I.Runner(golden["model"], max_batch=3)
    for frames in (golden_640(6)[:3], np.ascontiguousarray(np.repeat(np.repeat(golden_640(3), 2, 1), 2, 2)[:, :720, :1280])):
        b, h, w, c = frames.shape
        r.schedule(frames)
        r.wait()
        want = outputs(r)
        dev = torch.from_numpy(frames).cuda()
        r.schedule_device(dev.data_ptr(), b, h, w, c)
        r.wait()
        assert_same(want, outputs(r), f"schedule_device {w}x{h}")
        r.schedule_ptr(frames.ctypes.data, b, h, w, c)
        r.wait()
        assert_same(want, outputs(r), f"schedule_ptr {w}x{h}")
    sets = [golden_640(6)[:3], golden_640(6)[3:]]
    refs = []
    for s in sets:
        r.schedule(s)
        r.wait()
        refs.append(outputs(r))
    devs = [torch.from_numpy(s).cuda() for s in sets]
    for k in range(4):
        r.schedule_device(devs[k % 2].data_ptr(), 3, 640, 640, 3)
        r.wait()
        assert_same(refs[k % 2], outputs(r), f"alternating device buffers, call {k}")
    assert refs[0]["counts"].sum() > 0 and not np.array_equal(refs[0]["boxes"], refs[1]["boxes"])
    print("schedule_device / schedule_ptr / alternating buffers: bit-identical to host schedule()")
    r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("pitch", [1920, 1924], ids=["packed", "pitched"])
def test_device_micro_batches_equal_separate_chunk_runs(golden, pitch):
    """10 device frames in micro-batches of 4 (chunk k reads d_src + b0 * frame_bytes) equal three runs of a max_batch = 4
    runner on the same chunks."""
    import torch
    frames = golden_640(10)
    dev = torch.zeros((10, 640, pitch), dtype=torch.uint8, device="cuda")
    dev[:, :, :1920] = torch.from_numpy(frames.reshape(10, 640, 1920)).cuda()
    mb = I.Runner(golden["model"], max_batch=10, micro_batch=4)
    mb.schedule_device(dev.data_ptr(), 10, 640, 640, 3, stride_bytes=pitch)
    mb.wait()
    keep, scores = mb.keep_indices()
    got = dict(counts=mb.counts().copy(), keep=keep, scores=scores, boxes=mb.readback(0), labels=mb.readback(1),
               coefs=mb.readback(2), probs=mb.readback(3), bits=mb.masks(_lib.MASK_BITS_160))
    with pytest.raises(I.XrsegError):
        mb.masks(_lib.MASK_UPSAMPLE_640)                         # only the last chunk's prototypes are resident
    mb.close()
    ch = I.Runner(golden["model"], max_batch=4)
    parts = []
    for b0 in (0, 4, 8):
        nb = min(4, 10 - b0)
        ch.schedule_device(dev.data_ptr() + b0 * 640 * pitch, nb, 640, 640, 3, stride_bytes=pitch)
        ch.wait()
        parts.append(outputs(ch))
    ch.close()
    want = {k: np.concatenate([p[k] for p in parts]) for k in parts[0]}
    assert int(want["counts"].sum()) > 0
    assert_same(want, got, f"micro-batches of 4, pitch {pitch}")
    print(f"10 device frames, micro-batches of 4, pitch {pitch}: bit-identical to three chunk runs ({int(want['counts'].sum())} "
          f"detections)")
