"""Layer-local parity: every launch of the product network, element by element, against a float64 reference fed the GPU's
own inputs.

`LocalCheck` runs the oracle's topology (oracle/yolo11seg.py `forward_raw`) in float64.  For every convolution it computes
ref = act(conv(x, w, b)) and S = conv(|x|, |w|) + |b| from whatever input the oracle hands it, compares ref with the GPU's
tensor of that layer (`Runner(debug=True).fetch`), and hands the GPU's tensor on.  Every later layer's input is therefore
built from GPU activations (the oracle's own concat / split / upsample / max-pool / residual / attention code does the
building), so each launch is judged on its own arithmetic only and error cannot pile up from layer to layer.

The operands are what each kernel multiplies, so operand rounding is not part of the tolerance: weights rounded to fp16
(round to nearest) for the tcgen05, fused-Bottleneck, direct and mma.sync-stem paths and inside the depthwise kernel, fp32
weights for the fp32 stems (stem_conv_kernel, stem_u8_kernel), the fused positional encoding and the merged proto.up+cv2
launch (whose fp16 weights are formed from the fp32 ones, see below), and fp32 biases everywhere.

Per element the bound is

    |gpu - ref| <= A_OUT |ref| + SILU |z| + ACC (K + 1) S + SUB   (+ the kernel-specific terms listed with the constants)

with z the pre-activation, K the products per output and S the |x|.|w| sum above.  There is no per-layer constant.
A failure names the launch and its first offending element (frame, channel, y, x); every run prints, per launch, the
largest |err| / bound and where it occurs.
"""
from __future__ import annotations

import dataclasses
import json
import os
import subprocess
import sys
import time

import numpy as np
import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
for p in (ROOT, os.path.dirname(os.path.abspath(__file__))):
    if p not in sys.path:
        sys.path.insert(0, p)

from oracle import yolo11seg as Y  # noqa: E402

from test_abi import plan_dump  # noqa: E402,F401  (fixture: tools/plan_dump.cu compiled for the host)

GOLDEN = os.path.join(ROOT, "tests", "golden")

# ---- the bound's constants -------------------------------------------------------------------------------------------
U = 2.0 ** -11            # fp16 unit roundoff (round to nearest)
A_OUT = 1.01 * U          # the output's rounding to fp16; 1 % covers |gpu| > |ref| by at most the bound itself
SILU = 1.01 * 2.0 ** -12  # silu(z) = h tanh(h) + h, h = z / 2, with tanh.approx.f32 (max abs error 2^-10.987, PTX ISA): |err| <= 2^-12 |z|
ACC = 1.1 * 2.0 ** -23    # fp32 accumulation, per product: at most one fp32 ulp per addition (tensor-core adders truncate), times
                          # max silu'(z) = 1.0998 for the layers with SiLU
SUB = 2.0 ** -24          # fp16 subnormal spacing: the absolute floor of the output rounding
DW_HALF = 3 * U           # depthwise kernel: each kernel row is HMUL2 + 2 HFMA2 in fp16, three roundings of partial sums <= the
                          # row's |x|.|w| sum; S summed over the three rows bounds them all
DW_HALF_SUB = 9 * 2.0 ** -25   # ... and their fp16 subnormal floor, one half-spacing per half-precision operation
# Hidden fp16 intermediates (the fused Bottleneck's cv1 output in shared memory, proto.cv2's output in the fused cv3 tail): the
# reference rounds them as the kernel does, but the two roundings can land one fp16 step apart, so the consumer's bound carries
# 1.1 * conv(E, |w|) with E = the producer's bound + U |t| (1.1 = max silu' of the consumer).
# The merged proto.up+cv2 launch multiplies fp16 weights Wm formed in fp64 from the fp32 weights of both layers and rounded once;
# the reference forms and rounds them the same way (merged_weights), so that rounding is in the operands, as for every other layer.
# Attention (b10.attn.pe holds attention(v) + pe(v)): Q is scaled and rounded to fp16 (U plus the fp16 rounding of the scale),
# QK^T accumulates 32 products in fp32, so each logit is off by at most eps_i = c_s * max_j scale |q_i|.|k_j|; that moves every
# softmax weight by a factor within exp(+-2 eps_i), and P is rounded to fp16 (U) against an fp32 denominator (U): the output's
# error is <= (expm1(2 eps_i) + 2 U + N ACC) * sum_j p_ij |v_j|.

RESIDUAL = {f"{b}.m0.cv2" for b in ("b2", "b4", "n13", "n16", "n19")} | \
           {f"{b}.m0.{m}.cv2" for b in ("b6", "b8", "n22") for m in ("m0", "m1")}


def r16(t: torch.Tensor) -> torch.Tensor:
    """float64 -> nearest fp16 value (through fp32: both roundings are exact for values already representable)."""
    return t.float().half().double()


def spec_for(scale: str, nc: int) -> Y.Spec:
    sp = Y.make_spec(scale)
    return dataclasses.replace(sp, nc=nc, cls_mid=max(sp.ch[2], min(nc, 100)))


@dataclasses.dataclass
class Fusion:
    """How the runner's launch list computes the layers (derived from tools/plan_dump's op list)."""
    bneck_cv1: frozenset = frozenset()   # cv1 layers of fused Bottlenecks (their output lives in shared memory)
    tail: bool = False                   # proto.cv3 runs inside proto.cv2's launch
    merged: bool = False                 # proto.up runs inside that launch too
    pe_fused: bool = False               # b10.attn.pe rides in the attention kernel (fp32 weights)
    stem_f32: bool = True                # stem_conv_kernel / stem_u8_kernel (fp32 weights) rather than the mma.sync stems

    @staticmethod
    def from_ops(lines: list[str], stem_f32: bool) -> "Fusion":
        ops = parse_ops(lines)
        return Fusion(bneck_cv1=frozenset(o["name"] for o in ops if o["kind"] == "bneck"),
                      tail=any(o["tail"] for o in ops), merged=any(o["merged"] for o in ops),
                      pe_fused=any(o["kind"] == "attn" and o["name"] == "b10.attn.pe" for o in ops), stem_f32=stem_f32)


def parse_ops(lines: list[str]) -> list[dict]:
    ops = []
    for l in lines:
        t = l.split()
        if l.startswith("op "):
            ops.append(dict(kind=t[1], name=t[2], tail=None, merged=None))
        elif "(merged:" in l:
            ops[-1]["merged"] = t[1]
        elif "(tail:" in l:
            ops[-1]["tail"] = t[1]
    return ops


class LocalCheck(Y._ConvFeed):
    """Teacher-forced float64 reference.  provider(name) -> float64 tensor [F,C,H,W] of the sampled frames (the GPU's tensor);
    provider None simulates a GPU that stores every checked value rounded to fp16 (`synth` keeps those tensors)."""

    def __init__(self, weights, provider, fusion: Fusion, heads: int, targets: set[str] | None = None):
        super().__init__(weights=weights)
        self.provider = provider
        self.targets = targets                          # None: check every tensor; else only these (see __call__)
        self.fu = fusion
        self.heads = heads
        self.results: dict[str, dict] = {}
        self.synth: dict[str, torch.Tensor] = {}
        self.bounds: dict[str, torch.Tensor] = {}
        self.last_in: dict[str, torch.Tensor] = {}
        self.pending: dict[str, torch.Tensor] = {}      # consumer name -> error of its (hidden) input
        self.st: dict[str, torch.Tensor] = {}           # C2PSA / proto chain state

    # ---- GPU tensors ----
    def fetch(self, name, expected):
        if self.provider is None:
            t = r16(expected)
            self.synth[name] = t
            return t
        t = self.provider(name)
        assert tuple(t.shape) == tuple(expected.shape), (name, tuple(t.shape), tuple(expected.shape))
        return t

    def check(self, name, kind, gpu, ref, bound):
        self.bounds[name] = bound
        err = (gpu - ref).abs()
        ratio = err / bound
        bad = ratio > 1.0
        worst = int(torch.argmax(ratio))
        res = dict(kind=kind, ratio=float(ratio.reshape(-1)[worst]), where=np.unravel_index(worst, ratio.shape),
                   n=int(ratio.numel()), fail=None)
        if bool(bad.any()) or not bool(torch.isfinite(gpu).all()):
            idx = torch.nonzero(bad | ~torch.isfinite(gpu))[0].tolist()
            res["fail"] = (f"{name} ({kind}): first offending element frame {idx[0]} channel {idx[1]} y {idx[2]} x {idx[3]}: "
                           f"gpu {float(gpu[tuple(idx)]):.6g} ref {float(ref[tuple(idx)]):.6g} bound {float(bound[tuple(idx)]):.3g} "
                           f"({int(bad.sum())} of {ratio.numel()} elements out of bound)")
        self.results[name] = res

    def _stored(self, name):
        """The GPU stores this layer's own output under its name, unchanged by a later launch: targets mode may take it as
        is.  Not so for a fused Bottleneck's cv1 (shared memory), the C2PSA block's in-place chain and attention, and the
        prototype launches whose intermediates never leave the SM."""
        return name not in self.fu.bneck_cv1 and not name.startswith("b10.") and not name.startswith("proto.")

    # ---- arithmetic ----
    def _w(self, name, w):
        w = torch.as_tensor(w)
        fp32 = (name == "b0" and self.fu.stem_f32) or (name == "b10.attn.pe" and self.fu.pe_fused) or \
               (self.fu.merged and name in ("proto.up", "proto.cv2"))
        return w.double() if fp32 else w.half().double()

    @staticmethod
    def _conv(x, w, b, s, k, groups, transposed):
        if transposed:
            return F.conv_transpose2d(x, w, b, stride=s)
        return F.conv2d(x, w, b, stride=s, padding=k // 2, groups=groups)

    def __call__(self, x, cout, k=1, s=1, act=True, groups=1, transposed=False, name=""):
        if self.weights is None or self.record is not None:
            return super().__call__(x, cout, k, s, act, groups, transposed, name)
        w, b = self.weights[self.i]
        self.i += 1
        self.last_in[name] = x
        if self.targets is not None and name not in self.targets and self._stored(name):
            self.pending.pop(name, None)
            gpu = self.provider(name)
            return gpu - self.last_in[name[:-1] + "1"] if name in RESIDUAL else gpu
        w, b = self._w(name, w), torch.as_tensor(b).double()
        conv = lambda xx, ww, bb: self._conv(xx, ww, bb, s, k, groups, transposed)   # noqa: E731
        K = (x.shape[1] // groups) * (1 if transposed else k * k)
        z = conv(x, w, b)
        S = conv(x.abs(), w.abs(), b.abs())
        ref = Y.silu(z) if act else z
        bound = A_OUT * ref.abs() + ACC * (K + 1) * S + SUB
        if act:
            bound = bound + SILU * z.abs()
        if name in self.pending:                         # error of a hidden fp16 input, propagated through |w|
            e = conv(self.pending.pop(name), w.abs(), None)
            bound = bound + (1.1 if act else 1.0) * e
        kind = "stem" if name == "b0" else "convT" if transposed else "dw3x3" if groups > 1 else f"conv{k}x{k}" + ("/s2" if s == 2 else "")

        if name in self.fu.bneck_cv1:                    # fused Bottleneck: cv1's output never leaves shared memory
            self.pending[name[:-1] + "2"] = bound + U * ref.abs()
            return r16(ref)
        if name in RESIDUAL:                             # the launch adds the Bottleneck input: gpu = x + cv2(...)
            res = self.last_in[name[:-1] + "1"]
            kind = "bneck" if name[:-1] + "1" in self.fu.bneck_cv1 else kind + "+res"
            exp = res + ref
            gpu = self.fetch(name, exp)
            self.check(name, kind, gpu, exp, bound + U * exp.abs())
            return gpu - res
        if groups > 1 and name != "b10.attn.pe":         # depthwise kernel: fp16 row sums
            bound = bound + DW_HALF * S + DW_HALF_SUB
        if name == "b10.cv1":                            # second half (b) is updated in place by attn.proj / ffn.1
            c = cout // 2
            gpu = self.fetch(name, ref)
            self.check(name, kind, gpu[:, :c], ref[:, :c], bound[:, :c])
            b0 = r16(ref[:, c:])
            self.st["b0_err"] = bound[:, c:] + U * ref[:, c:].abs()
            self.pending["b10.attn.qkv"] = self.st["b0_err"]
            return torch.cat([gpu[:, :c], b0], 1)
        if name == "b10.attn.pe":
            return self._attn_pe(x, z, S, w, bound)
        if name == "b10.attn.proj":                      # b += proj(...): checked with ffn.1 against the final b
            self.st["proj_bound"] = bound
            self.st["proj"] = ref
            return ref
        if name == "b10.ffn.0":                          # input b1 = b0 + proj: not resident any more, its error rides along
            b1 = x
            e_b1 = self.st["b0_err"] + self.st["proj_bound"] + U * b1.abs() + SUB
            self.st["b1"], self.st["b1_err"] = b1, e_b1
            bound = bound + 1.1 * conv(e_b1, w.abs(), None)
        if name == "b10.ffn.1":                          # final b = b1 + ffn(f), in place
            b1 = self.st["b1"]
            exp = b1 + ref
            gpu = self.fetch(name, exp)
            self.check(name, "1x1+proj chain", gpu, exp, self.st["b1_err"] + bound + U * exp.abs())
            return gpu - b1
        if name == "proto.up" and self.fu.merged:        # merged launch: the upsampled map never exists
            self.st["up_x"], self.st["up_w"], self.st["up_b"] = x, w, b
            return ref
        if name == "proto.cv2" and (self.fu.merged or self.fu.tail):
            if self.fu.merged:                           # the launch multiplies fp16 Wm (4 taps x 64 channels) with the 80x80 map
                xu, up_b = self.st["up_x"], self.st["up_b"]
                wms = merged_weights(self.st["up_w"], w)
                # merged bias: the up bias through cv2 over the zero-padded upsampled map (border pixels see fewer taps), + cv2's bias
                bias = conv(up_b.reshape(1, -1, 1, 1).expand(1, -1, *z.shape[2:]), w, b)
                z = parity_conv(xu, wms) + bias
                S = parity_conv(xu.abs(), {k: v.abs() for k, v in wms.items()}) + bias.abs()
                ref = Y.silu(z)
                bound = A_OUT * ref.abs() + SILU * z.abs() + ACC * (4 * 64 + 1) * S + SUB
            self.pending["proto.cv3"] = bound + U * ref.abs()
            return r16(ref)
        if name == "proto.cv3" and self.fu.tail:
            kind = "up+cv2+cv3 merged" if self.fu.merged else "cv2+cv3 tail"
        gpu = self.fetch(name, ref)
        self.check(name, kind, gpu, ref, bound)
        return gpu

    def _attn_pe(self, v, z_pe, S_pe, w, bound_pe):
        """b10.attn.pe holds attention(q, k, v) + pe(v): attention computed in float64 exactly as the oracle does (its sum
        with the returned tensor reproduces the GPU's value), bounded as described with the constants."""
        B, c, H, Wd = v.shape
        N, heads = H * Wd, self.heads
        kd, hd = 32, c // heads
        qkv = self.st["qkv"].reshape(B, heads, 2 * kd + hd, N)
        q, k, vv = qkv[:, :, :kd], qkv[:, :, kd:2 * kd], qkv[:, :, 2 * kd:]
        scale = float(np.float32(kd ** -0.5))
        attn = torch.softmax(torch.matmul(q.transpose(-2, -1), k) * scale, dim=-1)         # [B, h, Nq, Nk]
        att = torch.matmul(vv, attn.transpose(-2, -1)).reshape(B, c, H, Wd)
        sc16 = float(np.float16(np.float32(kd ** -0.5)))
        c_s = abs(sc16 / scale - 1) + U + (kd + 1) * 2.0 ** -23
        eps = c_s * scale * torch.matmul(q.abs().transpose(-2, -1), k.abs()).amax(-1)     # [B, h, Nq]
        pv = torch.matmul(vv.abs(), attn.transpose(-2, -1))                               # [B, h, hd, Nq]
        b_att = ((torch.expm1(2 * eps) + 2 * U + N * ACC)[:, :, None, :] * pv).reshape(B, c, H, Wd)
        exp = att + z_pe
        bound = bound_pe - A_OUT * z_pe.abs() + A_OUT * exp.abs() + b_att
        if not self.fu.pe_fused:                         # depthwise launch, then its fp16 sum with the attention output
            bound = bound + DW_HALF * S_pe + DW_HALF_SUB + U * (z_pe.abs() + att.abs())
        gpu = self.fetch("b10.attn.pe", exp)
        self.check("b10.attn.pe", "attention+pe" if self.fu.pe_fused else "attention + dw3x3", gpu, exp, bound)
        return gpu - att


def merged_weights(wu, w2):
    """The fp16 weights of the merged proto.up+cv2 launch, as the host forms them (conv_tma.cuh merge_upconv_weights /
    pack_upmerge_weights_sw): for output parity (dy, dx), cv2's tap (ky, kx) reads the upsampled map at input offset
    (dy + ky - 1) // 2 through ConvTranspose tap (dy + ky - 1) % 2, so Wm[dy, dx][co, ci, offset] = sum over the taps landing on
    that offset of sum_k w2[co, k, ky, kx] wu[ci, k, tap], summed in fp64 from the fp32 weights and rounded to fp16 once."""
    w2, wu = w2.numpy(), wu.numpy()
    out = {}
    for dy in (0, 1):
        for dx in (0, 1):
            wm = np.zeros((w2.shape[0], wu.shape[0], 2, 2))
            for ky in range(3):
                for kx in range(3):
                    sy, sx = dy + ky - 1, dx + kx - 1
                    wm[:, :, sy // 2 + (1 - dy), sx // 2 + (1 - dx)] += w2[:, :, ky, kx] @ wu[:, :, sy % 2, sx % 2].T
            out[dy, dx] = torch.from_numpy(wm.astype(np.float16).astype(np.float64))   # float64 -> fp16 rounds once, to nearest
    return out


def parity_conv(x, wms):
    """The merged launch's arithmetic without its bias: output pixel (2y + dy, 2x + dx) is a 2x2 convolution of x with
    wms[dy, dx]; parity 0 reads input offsets {-1, 0}, parity 1 reads {0, +1}."""
    B, _, H, W = x.shape
    out = x.new_zeros(B, wms[0, 0].shape[0], 2 * H, 2 * W)
    for (dy, dx), wm in wms.items():
        out[:, :, dy::2, dx::2] = F.conv2d(F.pad(x, (1 - dx, dx, 1 - dy, dy)), wm)
    return out


def run_reference(weights, sp: Y.Spec, fusion: Fusion, provider, x, targets: set[str] | None = None):
    """One teacher-forced pass plus the bit-exact checks of the copy / max kernels.  Returns the LocalCheck.  targets: check
    only these tensors (LocalCheck targets mode)."""
    chk = LocalCheck(weights, provider, fusion, sp.heads, targets)
    feed = _Hook(chk)
    with torch.no_grad():
        Y.forward_raw(x, feed, sp, taps=feed.taps)
    assert chk.i == len(weights)
    return chk


class _Hook:
    """Wraps a LocalCheck so that the qkv tensor, the SPPF pools and the two upsamples are seen on their way through."""

    def __init__(self, chk: LocalCheck):
        self.chk = chk
        self.taps = {}

    def __call__(self, x, cout, k=1, s=1, act=True, groups=1, transposed=False, name=""):
        chk = self.chk
        if name == "b9.cv2":                             # x = [y0 | pool(y0) | pool^2 | pool^3], pooled by the oracle
            c_ = x.shape[1] // 4
            exp = x[:, c_:]
            gpu = chk.fetch("b9.pool", exp)
            chk.check("b9.pool", "sppf max-pool (bit-exact)", gpu, exp, torch.zeros_like(exp) + 2.0 ** -80)
            x = torch.cat([x[:, :c_], gpu], 1)
        if name in ("n13.cv1", "n16.cv1"):               # x = [up2(f) | skip]: the upsample half is the GPU's copy
            tag = "up." + name[1:3]
            c_up = x.shape[1] - chk.st[tag + ".skip"]
            exp = x[:, :c_up]
            gpu = chk.fetch(tag, exp)
            chk.check(tag, "upsample2x (bit-exact)", gpu, exp, torch.zeros_like(exp) + 2.0 ** -80)
            x = torch.cat([gpu, x[:, c_up:]], 1)
        y = chk(x, cout, k, s, act, groups, transposed, name)
        if name == "b10.attn.qkv":
            chk.st["qkv"] = y
        if name == "b6.cv2":
            chk.st["up.13.skip"] = y.shape[1]
        if name == "b4.cv2":
            chk.st["up.16.skip"] = y.shape[1]
        return y


def report(chk: LocalCheck, label: str) -> list[str]:
    lines = []
    for name, r in chk.results.items():
        f, c, y, x = (int(v) for v in r["where"])
        lines.append(f"{label:28s} {name:18s} {r['kind']:26s} max|err|/bound {r['ratio']:8.3g} at frame {f} c {c} y {y} x {x}")
    return lines


def failures(chk: LocalCheck) -> list[str]:
    return [r["fail"] for r in chk.results.values() if r["fail"]]


# ---- launch-list coverage ---------------------------------------------------------------------------------------------
def launch_tensors(o: dict, ups: int) -> tuple[list[str], set[str]] | None:
    """(layers computed by launch o, tensors the checker compares for it); ups = nearest-upsample launches before it.
    None for an unknown launch kind."""
    kind, name = o["kind"], o["name"]
    if kind in ("stem", "conv", "dw"):
        layers = name.split("+")                         # sibling fusion: "b6.m0.cv1+b6.m0.cv2"
        if o["tail"]:
            layers.append(o["tail"])
        if o["merged"]:
            layers.append(o["merged"])
        # hidden and in-place outputs are checked through the tensor that carries them
        keys = {"b10.attn.proj": "b10.ffn.1"}
        if o["tail"]:
            keys.update({"proto.up": "proto.cv3", "proto.cv2": "proto.cv3"})
        return layers, {keys.get(l, l) for l in layers}
    if kind == "bneck":
        return [name, name[:-1] + "2"], {name[:-1] + "2"}
    if kind == "attn":
        return ([name] if name != "-" else []), {"b10.attn.pe"}   # attention alone (pe unfused): through pe's residual
    if kind == "sppf":
        return [], {"b9.pool"}
    if kind == "up":
        return [], {("up.13", "up.16")[ups]}
    return None


def launch_coverage(ops: list[dict], checked: set[str], layer_names: list[str]) -> list[str]:
    """Every launch of the op list maps to at least one checked tensor, and every layer is computed by a checked launch.
    Returns the problems (empty: covered)."""
    problems, covered = [], set()
    ups = 0
    for o in ops:
        kind, name = o["kind"], o["name"]
        lt = launch_tensors(o, ups)
        ups += kind == "up"
        if lt is None:
            problems.append(f"unknown launch kind {kind} ({name})")
            continue
        layers, tensors = lt
        missing = tensors - checked
        if not tensors or missing:
            problems.append(f"launch {kind} {name}: no checked tensor ({sorted(missing)})")
        covered.update(layers)
    lost = [n for n in layer_names if n not in covered]
    if lost:
        problems.append(f"layers computed by no launch of the list: {lost}")
    return problems


def plan_ops(exe: str, scale: str, nc: int, env: dict | None = None) -> list[str]:
    e = dict(os.environ)
    e.update(env or {})
    out = subprocess.run([exe, "8", scale, "ops", "up", str(nc)], capture_output=True, text=True, check=True, env=e).stdout
    return out.splitlines()


# ---- weights ----------------------------------------------------------------------------------------------------------
def random_weights(scale: str, nc: int, seed: int):
    from xr_image_segmentation_b200 import weights as W
    layers, ws = W.random_weights(scale, seed, cls_bias=None if nc == 80 else -5.15, nc=nc)
    return layers, ws


# ---- CPU: the checker against a simulated GPU, and the coverage guard ------------------------------------------------
def _small_input(seed=0, hw=96, frames=1):
    rng = np.random.default_rng(seed)
    return torch.from_numpy(rng.integers(0, 256, (frames, 3, hw, hw)).astype(np.float64) / 255.0)


@pytest.mark.parametrize("scale,nc,fusion", [
    ("n", 80, Fusion(bneck_cv1=frozenset({"b2.m0.cv1", "b4.m0.cv1", "n16.m0.cv1"}), tail=True, merged=True, pe_fused=True)),
    ("n", 365, Fusion(tail=True, pe_fused=False, stem_f32=False)),
    ("s", 80, Fusion(bneck_cv1=frozenset({"b2.m0.cv1"}), pe_fused=True)),
])
def test_checker_passes_a_faithful_gpu_and_names_a_moved_element(scale, nc, fusion):
    """Fed the float64 reference's own values rounded to fp16 (a GPU that stores every tensor exactly rounded), the checker
    passes; with one element moved by twice its bound, it fails and names that launch and that element."""
    _, ws = random_weights(scale, nc, seed=5)
    weights = [(w, b) for w, b in ws]
    sp = spec_for(scale, nc)
    x = _small_input()
    sim = run_reference(weights, sp, fusion, None, x)
    assert not failures(sim)
    provider = lambda n: sim.synth[n]                     # noqa: E731
    again = run_reference(weights, sp, fusion, provider, x)
    assert not failures(again)
    assert set(again.results) == set(sim.results)
    for victim in ("h5.cls.2", "proto.cv3", "b10.attn.pe", "n19.cv2"):
        t = sim.synth[victim].clone()
        idx = (0, min(3, t.shape[1] - 1), t.shape[2] // 2, t.shape[3] - 1)
        t[idx] += 2 * float(sim.bounds[victim][idx])
        moved = dict(sim.synth)
        moved[victim] = t
        chk = run_reference(weights, sp, fusion, lambda n: moved[n], x)
        fails = {r: v["fail"] for r, v in chk.results.items() if v["fail"]}
        assert victim in fails, (victim, sorted(fails))
        assert f"frame 0 channel {idx[1]} y {idx[2]} x {idx[3]}:" in fails[victim], fails[victim]
        upstream = [n for n in fails if list(chk.results).index(n) < list(chk.results).index(victim)]
        assert not upstream, upstream


@pytest.mark.parametrize("scale,nc", [("n", 80), ("n", 365), ("n", 1024), ("s", 80), ("s", 365), ("s", 1024)])
@pytest.mark.parametrize("merge", [True, False])
def test_every_launch_maps_to_a_checked_tensor(plan_dump, scale, nc, merge):
    """Coverage guard: every op of the runner's launch list (tools/plan_dump `ops up`, with XRSEG_FUSE_UP=0 for the
    three-launch prototype path) maps to at least one tensor the checker compares, and every layer runs in a checked launch.
    An unknown launch kind fails, so a new fusion pass cannot add a launch the checker does not see."""
    env = {} if merge else {"XRSEG_FUSE_UP": "0"}
    lines = plan_ops(plan_dump, scale, nc, env)
    fusion = Fusion.from_ops(lines, stem_f32=True)
    assert fusion.merged == (merge and scale == "n")
    layers, ws = random_weights(scale, nc, seed=1)
    chk = run_reference([(w, b) for w, b in ws], spec_for(scale, nc), fusion, None, _small_input(hw=64))
    problems = launch_coverage(parse_ops(lines), set(chk.results), [l.name for l in layers])
    assert not problems, problems


def test_coverage_guard_rejects_an_unknown_launch(plan_dump):
    lines = plan_ops(plan_dump, "n", 80) + ["op fancy  n19.cv2+h4.box.0  in  40x40  c128 out c64  res 0 branch 0"]
    layers, ws = random_weights("n", 80, seed=1)
    chk = run_reference([(w, b) for w, b in ws], spec_for("n", 80), Fusion.from_ops(lines, True), None, _small_input(hw=64))
    problems = launch_coverage(parse_ops(lines), set(chk.results), [l.name for l in layers])
    assert problems == ["unknown launch kind fancy (n19.cv2+h4.box.0)"]


# ---- GPU: the real runner ---------------------------------------------------------------------------------------------
def _frames(cfg, rng):
    if cfg.get("frames") == "golden":
        g = np.load(os.path.join(GOLDEN, "inputs.npz"))
        return np.stack([g[n] for n in ("coco139", "coco7108")])   # both 426 x 640: the resample path
    return rng.integers(0, 256, (cfg["batch"], 640, 640, 3), dtype=np.uint8)


def run_config(cfg: dict, plan_exe: str) -> tuple[list[str], list[str]]:
    """Runs one configuration on the GPU and checks its sampled frames.  Returns (report lines, failures)."""
    from xr_image_segmentation_b200 import _lib, inference as I, weights as W
    scale, nc = cfg.get("scale", "n"), cfg.get("nc", 80)
    if cfg.get("weights") == "golden":
        model = I.ModelLoader.Load(os.path.join(GOLDEN, "yolo11n_seg.xrsw"))
        _, pl = W.read_pack(model.pack)
        weights = [(w, b) for _, w, b in pl]
    else:
        layers, ws = random_weights(scale, nc, cfg.get("seed", 0))
        weights = [(w, b) for w, b in ws]
        gpu_ws = weights
        if "perturb" in cfg:                              # the GPU runs a pack with one weight moved; the reference keeps the original
            name, co, log2_move = cfg["perturb"]
            li = [l.name for l in layers].index(name)
            w = weights[li][0].copy()
            flat = np.abs(w[co] if co is not None else w)
            j = np.unravel_index(int(np.argmax(flat)), flat.shape)
            j = ((co,) + j) if co is not None else j
            w[j] += np.float32(2.0 ** log2_move * np.abs(w).max())
            gpu_ws = list(weights)
            gpu_ws[li] = (w, weights[li][1])
        model = I.Model(W.write_pack(scale, layers, gpu_ws), scale, nc)
    impl = _lib.CONV_DIRECT if cfg.get("impl") == "direct" else _lib.CONV_UMMA
    env = dict(cfg.get("env", {}))
    if impl == _lib.CONV_DIRECT:
        env["XRSEG_FUSE"] = "0"                           # xrseg_create: the direct engine runs the unfused layer list
    fusion = Fusion.from_ops(plan_ops(plan_exe, scale, nc, env),
                             stem_f32=cfg.get("frames") == "golden" or impl == _lib.CONV_DIRECT)
    rng = np.random.default_rng(cfg.get("seed", 0) + 100)
    frames = _frames(cfg, rng)
    batch = frames.shape[0]
    mb = cfg.get("max_batch", batch)
    r = I.Runner(model, max_batch=mb, micro_batch=cfg.get("micro_batch", 0), conv_impl=impl, debug=True)
    r.schedule(np.ascontiguousarray(frames))
    r.wait(strict=False)                                  # random class logits may overflow the NMS caps: the network's tensors are whole
    chunk = min(cfg.get("micro_batch", 0) or mb, mb)
    b0 = (-(-batch // chunk) - 1) * chunk                # first frame of the resident (last) chunk
    sample = cfg.get("sample", list(range(b0, batch)))
    local = [s - b0 for s in sample]
    assert min(local) >= 0, "sampled frames must lie in the last micro-batch"
    probe = r.fetch("b10.cv2")
    assert probe.shape[0] == batch - b0, (probe.shape, batch, b0)
    cache = {}

    def provider(name):
        if name not in cache:
            cache.clear()                                 # one layer at a time: only the tensor being compared is kept
            cache[name] = torch.from_numpy(r.fetch(name)[local]).double()
        return cache[name]

    if fusion.stem_f32 and cfg.get("frames") == "golden":
        x = provider("input")                             # the resample path writes the fp16 image
    else:
        x = torch.from_numpy(frames[sample].transpose(0, 3, 1, 2).astype(np.float64) / 255.0)
    t0 = time.time()
    chk = run_reference(weights, spec_for(scale, nc), fusion, provider, x)
    r.close()
    label = cfg["label"]
    lines = report(chk, label) + [f"{label}: {len(chk.results)} tensors, {len(sample)} frames checked in {time.time() - t0:.1f} s"]
    return lines, failures(chk)


def _gpu_name():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 and out.stdout.strip() else "unknown GPU"


def _summarise(lines):
    print("\n".join(lines))


MATRIX = [
    dict(label="n golden, resample", weights="golden", frames="golden", seed=0),
    dict(label="n golden, fused stem", weights="golden", batch=2, seed=1),
    dict(label="n random, max_batch 1", batch=1, seed=2),
    dict(label="n random, mb 8 / 3 frames", max_batch=8, batch=3, seed=3),
    dict(label="n random, batch 72", batch=72, sample=[0, 63, 64, 71], seed=4),
    dict(label="n random, mb 10 / micro 4", max_batch=10, micro_batch=4, batch=10, seed=5),
    dict(label="s random, batch 2", scale="s", batch=2, seed=6),
    dict(label="n nc 1", nc=1, batch=1, seed=7),
    dict(label="n nc 365", nc=365, batch=1, seed=8),
    dict(label="n nc 1024", nc=1024, batch=1, seed=9),
    dict(label="n CONV_DIRECT", impl="direct", batch=1, seed=10),
]
SWITCHES = ["XRSEG_FUSE", "XRSEG_FUSE_BNECK", "XRSEG_FUSE_PE", "XRSEG_FUSE_TAIL", "XRSEG_FUSE_UP", "XRSEG_TINY_GRID",
            "XRSEG_FLAT_TMA", "XRSEG_S2_TMA", "XRSEG_SPLIT_SMALL", "XRSEG_HALO_SPLIT_N", "XRSEG_S2_PAIR", "XRSEG_PDL+XRSEG_BRANCHES"]


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", MATRIX, ids=[c["label"] for c in MATRIX])
def test_every_launch_is_within_its_bound(lib, dlib, plan_dump, cfg):
    lines, fails = run_config(cfg, plan_dump)
    _summarise([_gpu_name()] + lines)
    assert not fails, "\n".join(fails)


@pytest.mark.gpu
@pytest.mark.parametrize("switch", SWITCHES)
def test_every_launch_is_within_its_bound_with_a_switch_off(lib, dlib, plan_dump, switch):
    """Each "off" switch of tools/README.md that changes arithmetic or plans, in a fresh process (several are read once
    into function-local statics)."""
    env = {k: "0" for k in switch.split("+")}
    cfg = dict(label=f"n random, {switch}=0", batch=2, seed=11, env=env)
    e = dict(os.environ)
    e.update(env)
    p = subprocess.run([sys.executable, os.path.abspath(__file__), json.dumps(cfg), plan_dump], capture_output=True, text=True,
                       env=e, cwd=ROOT)
    print(p.stdout[-20000:])
    assert p.returncode == 0, p.stdout[-4000:] + p.stderr[-4000:]


# (layer, output channel or None, classes, log2 of the move relative to max |w|).  The fused Bottleneck's cv2 and the merged
# proto launch are checked through a hidden fp16 intermediate (cv1's output in shared memory, proto.cv2's output in the cv3
# tail), whose bound carries two fp16 roundings and the SiLU approximation of every one of its channels into the consumer;
# there one weight moved by 2^-6 stays inside that allowance (simulated: 0.38 of the bound for proto.up), 2^-3 reaches ~2.7x.
SENSITIVITY = [("b0", None, 80, -6), ("h3.box.1", None, 80, -6), ("b2.m0.cv2", None, 80, -3), ("b3", None, 80, -6),
               ("b4.cv2", None, 80, -6), ("h3.cls.1dw", None, 80, -6), ("b10.attn.pe", None, 80, -6), ("proto.up", None, 80, -3),
               ("h4.cls.2", 300, 365, -6)]
FLAGGED_AS = {"proto.up": "proto.cv3"}                   # proto.up runs inside the merged launch that writes the prototypes


@pytest.mark.gpu
@pytest.mark.parametrize("layer,co,nc,log2_move", SENSITIVITY, ids=[s[0] for s in SENSITIVITY])
def test_a_moved_weight_is_flagged_in_its_own_launch_only(lib, dlib, plan_dump, layer, co, nc, log2_move):
    """The GPU runs a pack in which one weight moved by 2^-6 (or 2^-3, see SENSITIVITY) of its layer's max |w| (for h4.cls.2 at 365 classes: a weight of
    output channel 300, which only the second N tile computes); the reference keeps the original weights.  The checker
    must flag that launch and no other."""
    cfg = dict(label=f"moved weight in {layer}", nc=nc, batch=1, seed=12, perturb=(layer, co, log2_move))
    lines, fails = run_config(cfg, plan_dump)
    flagged = sorted({f.split(" ")[0] for f in fails})
    print("\n".join(lines[-1:] + fails))
    assert flagged == [FLAGGED_AS.get(layer, layer)], flagged


if __name__ == "__main__":                               # one configuration in a fresh process (the switch tests)
    lines, fails = run_config(json.loads(sys.argv[1]), sys.argv[2])
    _summarise([_gpu_name()] + lines)
    if fails:
        print("\n".join(fails))
        sys.exit(1)
