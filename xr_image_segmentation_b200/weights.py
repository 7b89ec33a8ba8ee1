"""XRSW weight packs: the on-disk / in-memory weight format libxrseg.so consumes (csrc/model.cuh).

↔ the constants of the reference's model asset, Assets/Resources/Model/yolo11n-seg-sentis.sentis: 100 convolutions
(the DFL 1x1 conv is structural), each weight / bias tensor per-tensor affine uint8 (SURVEY.md fact 6).  A pack keeps
those uint8 tensors with their (scale, zero point) so that the library dequantizes exactly like the graph's
`DequantizeUint8` layers, or carries plain float32 tensors (random-init networks of BASELINE.json configs 2/3).

Layout (little endian): 32-byte header | n_layers x 96-byte records | payload.  Layers are in the canonical order =
the asset's chain order = the order `xrseg_layer_info_get` reports.
"""
from __future__ import annotations

import ctypes as C
import struct
from dataclasses import dataclass

import numpy as np

from . import _lib

HEADER = struct.Struct("<4sIIIQ8s")
RECORD = struct.Struct("<32sIIIIIIIIfifiQQ")
assert HEADER.size == 32 and RECORD.size == 96

CLS_FINAL = ("h3.cls.2", "h4.cls.2", "h5.cls.2")


@dataclass
class Layer:
    name: str
    cin: int
    cout: int
    k: int
    stride: int
    groups: int
    act: int
    transposed: int
    h_in: int
    w_in: int

    @property
    def weight_shape(self):
        if self.transposed:
            return (self.cin, self.cout, self.k, self.k)
        return (self.cout, self.cin // self.groups, self.k, self.k)


def layer_table(scale: str, nc: int = 80) -> list[Layer]:
    """The topology's convolution list for a model of `nc` classes, straight from the C library (single source of truth)."""
    lib = _lib.load_library()
    n = _lib.check(lib.xrseg_layer_count_nc(ord(scale), nc))
    out = []
    for i in range(n):
        info = _lib.LayerInfo()
        _lib.check(lib.xrseg_layer_info_get_nc(ord(scale), nc, i, C.byref(info)))
        out.append(Layer(info.name.decode(), info.cin, info.cout, info.k, info.stride, info.groups, info.act,
                         info.transposed, info.h_in, info.w_in))
    return out


@dataclass
class Tensor8:
    """Per-tensor affine uint8 tensor: value = (q - zp) * scale."""
    q: np.ndarray
    scale: float
    zp: int

    def dequant(self) -> np.ndarray:
        return ((self.q.astype(np.float32) - np.float32(self.zp)) * np.float32(self.scale)).astype(np.float32)


def write_pack(scale: str, layers: list[Layer], tensors: list[tuple]) -> bytes:
    """tensors[i] = (w, b) with each either a float32 ndarray or a Tensor8."""
    assert len(layers) == len(tensors)
    payload = bytearray()
    recs = []
    for l, (w, b) in zip(layers, tensors):
        quant = isinstance(w, Tensor8)
        assert quant == isinstance(b, Tensor8)
        wa = w.q if quant else np.ascontiguousarray(w, np.float32)
        ba = b.q if quant else np.ascontiguousarray(b, np.float32)
        assert tuple(wa.shape) == l.weight_shape, (l.name, wa.shape, l.weight_shape)
        assert ba.shape == (l.cout,)
        while len(payload) % 16:
            payload.append(0)
        w_off = len(payload)
        payload += wa.tobytes()
        while len(payload) % 16:
            payload.append(0)
        b_off = len(payload)
        payload += ba.tobytes()
        recs.append(RECORD.pack(l.name.encode()[:31], l.cout, l.cin // l.groups, l.k, l.stride, l.groups, l.act,
                                l.transposed, 3 if quant else 0,
                                float(w.scale) if quant else 1.0, int(w.zp) if quant else 0,
                                float(b.scale) if quant else 1.0, int(b.zp) if quant else 0, w_off, b_off))
    payload_offset = HEADER.size + RECORD.size * len(layers)
    head = HEADER.pack(b"XRSW", 1, len(layers), ord(scale), payload_offset, b"\0" * 8)
    return head + b"".join(recs) + bytes(payload)


def read_pack(data: bytes):
    """-> (scale, [(name, w float32, b float32)]) with uint8 tensors dequantized as (q - zp) * scale."""
    magic, version, n, scale, payload_offset, _ = HEADER.unpack_from(data, 0)
    assert magic == b"XRSW" and version == 1
    out = []
    for i in range(n):
        (name, cout, cin_g, k, stride, groups, act, transposed, dtype, ws, wz, bs, bz, w_off, b_off) = \
            RECORD.unpack_from(data, HEADER.size + i * RECORD.size)
        name = name.split(b"\0")[0].decode()
        # transposed records keep torch's ConvTranspose layout [cin, cout, k, k] with cin_g = cin
        shape = (cin_g, cout, k, k) if transposed else (cout, cin_g, k, k)
        nw = int(np.prod(shape))
        if dtype == 0:
            w = np.frombuffer(data, np.float32, nw, payload_offset + w_off).reshape(shape).copy()
            b = np.frombuffer(data, np.float32, cout, payload_offset + b_off).copy()
        else:
            w = Tensor8(np.frombuffer(data, np.uint8, nw, payload_offset + w_off).reshape(shape), ws, wz).dequant()
            b = Tensor8(np.frombuffer(data, np.uint8, cout, payload_offset + b_off), bs, bz).dequant()
        out.append((name, w, b))
    return chr(scale), out


# Frozen random-init recipe (SURVEY.md §8d config 2).  The survey proposed gain 1.85 / bias std 0.85 (medians of the
# trained asset); measured here, that init diverges through the ~30 sequential SiLU layers (head logits ~1e6, fp16
# overflow), so the generator uses a variance-preserving gain instead.  The three final class convolutions get their
# bias shifted so that ~1.5 % of the 8400 anchors pass the 0.301 score filter on uniform-noise frames (a trained net
# on a real image: 43 / 8400); the shift was tuned once per scale on frames of seed 0 and is frozen.
INIT_GAIN = 1.5
INIT_BIAS_STD = 0.2
# ("s" re-tuned in round 2 for the weights of seed 3 that bench.py --config 2 and the s-scale parity test use: with the old -4.87
# 7 700 of the 8 400 anchors passed the filter -- a post-processing stress test, not a detector; -12.4 gives ~126 = 1.5 %)
INIT_CLS_BIAS = {"n": -5.15, "s": -12.4}


def random_weights(scale: str, seed: int, cls_bias: float | None = None, nc: int = 80):
    """Random-init network of BASELINE.json configs 2/3: w ~ N(0, (1.5/sqrt(fan_in))^2), b ~ N(0, 0.2^2), final class
    conv biases N(cls_bias, 0.05^2).  Returns (layers, [(w, b)]).  INIT_CLS_BIAS was tuned for 80 classes: a network of
    another class count needs its own cls_bias."""
    if cls_bias is None:
        if nc != 80:
            raise ValueError(f"random_weights: pass cls_bias for a {nc}-class network (INIT_CLS_BIAS is tuned for 80 classes)")
        cls_bias = INIT_CLS_BIAS[scale]
    rng = np.random.default_rng(seed)
    layers = layer_table(scale, nc)
    out = []
    for l in layers:
        fan_in = l.cin if l.transposed else (l.cin // l.groups) * l.k * l.k
        w = (rng.standard_normal(l.weight_shape, dtype=np.float32) * np.float32(INIT_GAIN / np.sqrt(fan_in))).astype(np.float32)
        b = (rng.standard_normal(l.cout, dtype=np.float32) * np.float32(INIT_BIAS_STD)).astype(np.float32)
        if l.name in CLS_FINAL:
            b = (b * np.float32(0.25) + np.float32(cls_bias)).astype(np.float32)
        out.append((w, b))
    return layers, out
