"""ORACLE (test infrastructure, not product): reader for the `.sentis` model container.

The reference ships its network as one Unity Inference Engine asset
(/root/reference/Assets/Resources/Model/yolo11n-seg-sentis.sentis, loaded at
Assets/Scripts/InferenceEngine/IEExecutor.cs:382 via `ModelLoader.Load`).  The package
that defines the format (`com.unity.ai.inference` 2.2.1, Packages/manifest.json:4) is
NOT vendored in the reference, so the layout below is restated from the file itself
(SURVEY.md Appendix C): a u32 size + FlatBuffer "Program", then u32 size + FlatBuffer
"Buffer" chunks holding the weight blob.

Only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s cpu_baseline / `--impl reference`
legs may import anything under `oracle/`.
"""
from __future__ import annotations

import struct
from dataclasses import dataclass, field
from typing import Any

import numpy as np


class _FB:
    """Minimal read-only FlatBuffer accessor (tables, vectors, strings, scalars)."""

    def __init__(self, buf: bytes, base: int = 0):
        self.b = buf
        self.base = base

    def root(self) -> int:
        return self.base + struct.unpack_from("<I", self.b, self.base)[0]

    def _field(self, table: int, idx: int) -> int:
        """Absolute offset of field `idx` inside `table`, or 0 when absent."""
        vt = table - struct.unpack_from("<i", self.b, table)[0]
        vt_size = struct.unpack_from("<H", self.b, vt)[0]
        slot = 4 + 2 * idx
        if slot >= vt_size:
            return 0
        off = struct.unpack_from("<H", self.b, vt + slot)[0]
        return table + off if off else 0

    def scalar(self, table: int, idx: int, fmt: str, default=0):
        p = self._field(table, idx)
        return struct.unpack_from("<" + fmt, self.b, p)[0] if p else default

    def indirect(self, table: int, idx: int) -> int:
        p = self._field(table, idx)
        return p + struct.unpack_from("<I", self.b, p)[0] if p else 0

    def string(self, table: int, idx: int) -> str | None:
        p = self.indirect(table, idx)
        if not p:
            return None
        n = struct.unpack_from("<I", self.b, p)[0]
        return self.b[p + 4:p + 4 + n].decode("utf-8")

    def vec_len(self, table: int, idx: int) -> int:
        p = self.indirect(table, idx)
        return struct.unpack_from("<I", self.b, p)[0] if p else 0

    def vec_scalars(self, table: int, idx: int, fmt: str) -> list:
        p = self.indirect(table, idx)
        if not p:
            return []
        n = struct.unpack_from("<I", self.b, p)[0]
        return list(struct.unpack_from("<%d%s" % (n, fmt), self.b, p + 4))

    def vec_tables(self, table: int, idx: int) -> list[int]:
        p = self.indirect(table, idx)
        if not p:
            return []
        n = struct.unpack_from("<I", self.b, p)[0]
        out = []
        for i in range(n):
            e = p + 4 + 4 * i
            out.append(e + struct.unpack_from("<I", self.b, e)[0])
        return out

    def vec_strings(self, table: int, idx: int) -> list[str]:
        out = []
        for t in self.vec_tables(table, idx):
            n = struct.unpack_from("<I", self.b, t)[0]
            out.append(self.b[t + 4:t + 4 + n].decode("utf-8"))
        return out

    def vec_bytes_span(self, table: int, idx: int) -> tuple[int, int]:
        p = self.indirect(table, idx)
        n = struct.unpack_from("<I", self.b, p)[0]
        return p + 4, n


_DTYPES = {0: np.float32, 1: np.int32, 2: np.int16, 3: np.uint8}


@dataclass
class TensorValue:
    dtype: Any
    length_byte: int
    shape: list[int]
    is_const: bool
    storage_offset: int
    dynamic: bool
    data: np.ndarray | None = None  # filled for constants


@dataclass
class Chain:
    index: int
    op: str
    inputs: list[int]      # value ids (-1 = omitted optional tensor input)
    outputs: list[int]
    args: list[int]        # value ids of attribute EValues


@dataclass
class SentisModel:
    version: int
    values: list[Any]                   # TensorValue | int | float | bool | list | None
    chains: list[Chain]
    inputs: list[int]
    input_names: list[str]
    outputs: list[int]
    output_names: list[str]
    operators: list[str]
    blob: bytes = field(repr=False, default=b"")


def load_sentis(path_or_bytes) -> SentisModel:
    """Parse a `.sentis` file (SURVEY.md Appendix C; ↔ `ModelLoader.Load`, IEExecutor.cs:382)."""
    raw = path_or_bytes if isinstance(path_or_bytes, (bytes, bytearray)) else open(path_or_bytes, "rb").read()
    prog_size = struct.unpack_from("<I", raw, 0)[0]
    fb = _FB(raw, 4)
    prog = fb.root()
    version = fb.scalar(prog, 0, "I")
    plan = fb.indirect(prog, 1)

    # weight chunks follow the program
    blobs = []
    pos = 4 + prog_size
    while pos + 4 <= len(raw):
        csize = struct.unpack_from("<I", raw, pos)[0]
        cfb = _FB(raw, pos + 4)
        start, n = cfb.vec_bytes_span(cfb.root(), 0)
        blobs.append(raw[start:start + n])
        pos += 4 + csize
    blob = b"".join(blobs)

    operators = [fb.string(t, 0) for t in fb.vec_tables(plan, 7)]

    values: list[Any] = []
    for ev in fb.vec_tables(plan, 1):
        vt = fb.scalar(ev, 0, "B")
        v = fb.indirect(ev, 1)
        if vt in (0, 1):
            values.append(None)
        elif vt == 2:
            values.append(int(fb.scalar(v, 0, "i")))
        elif vt == 3:
            values.append(float(fb.scalar(v, 0, "f", 0.0)))
        elif vt == 4:
            values.append(bool(fb.scalar(v, 0, "B")))
        elif vt == 6:
            st = fb.scalar(v, 0, "B")
            t = TensorValue(
                dtype=_DTYPES[st],
                length_byte=fb.scalar(v, 1, "i"),
                shape=fb.vec_scalars(v, 2, "i"),
                is_const=bool(fb.scalar(v, 3, "I")),
                storage_offset=fb.scalar(v, 4, "i"),
                dynamic=bool(fb.scalar(v, 5, "B")),
            )
            if t.is_const:
                n = int(np.prod(t.shape)) if t.shape else 1
                nbytes = n * np.dtype(t.dtype).itemsize
                t.data = np.frombuffer(blob, dtype=t.dtype, count=n, offset=t.storage_offset).reshape(t.shape).copy() \
                    if nbytes else np.zeros(t.shape, t.dtype)
            values.append(t)
        elif vt == 8:
            values.append([int(x) for x in fb.vec_scalars(v, 0, "i")])
        elif vt == 9:
            values.append([float(x) for x in fb.vec_scalars(v, 0, "f")])
        else:
            raise ValueError(f"unknown EValue type {vt}")

    chains = []
    for i, c in enumerate(fb.vec_tables(plan, 6)):
        ins = fb.vec_scalars(c, 0, "i")
        outs = fb.vec_scalars(c, 1, "i")
        instrs = fb.vec_tables(c, 2)
        assert len(instrs) == 1, "one kernel call per chain expected"
        kc = fb.indirect(instrs[0], 1)
        op_index = fb.scalar(kc, 0, "i")
        args = fb.vec_scalars(kc, 1, "i")
        chains.append(Chain(i, operators[op_index], ins, outs, args))

    return SentisModel(
        version=version,
        values=values,
        chains=chains,
        inputs=fb.vec_scalars(plan, 2, "i"),
        input_names=fb.vec_strings(plan, 3),
        outputs=fb.vec_scalars(plan, 4, "i"),
        output_names=fb.vec_strings(plan, 5),
        operators=operators,
        blob=blob,
    )


class _FBWriter:
    """Minimal FlatBuffer builder for the layout _FB reads: objects are prepended (children before the tables that point
    at them, so every offset points forward); positions are counted from the end of the buffer."""

    def __init__(self):
        self.parts, self.size = [], 0

    def _prepend(self, data: bytes) -> int:
        self.parts.append(bytes(data))
        self.size += len(data)
        return self.size

    def scalars(self, fmt: str, items) -> int:
        items = list(items)
        return self._prepend(struct.pack("<I%d%s" % (len(items), fmt), len(items), *items))

    def bytes_(self, data: bytes) -> int:
        return self._prepend(struct.pack("<I", len(data)) + bytes(data))

    def string(self, s: str) -> int:
        return self.bytes_(s.encode("utf-8"))

    def offsets(self, targets) -> int:
        targets = list(targets)
        pos = self.size + 4 + 4 * len(targets)
        return self._prepend(struct.pack("<I%dI" % len(targets), len(targets),
                                         *(pos - 4 - 4 * i - q for i, q in enumerate(targets))))

    def table(self, fields) -> int:
        """fields[i]: None (absent), (struct format, value), or the position of an object written earlier."""
        body, slots, refs = bytearray(), [], []
        for f in fields:
            if f is None:
                slots.append(0)
                continue
            slots.append(4 + len(body))
            if isinstance(f, tuple):
                body += struct.pack("<" + f[0], f[1])
            else:
                refs.append((4 + len(body), f))
                body += bytes(4)
        pos = self.size + 4 + len(body)
        for off, q in refs:
            struct.pack_into("<I", body, off - 4, pos - off - q)
        vt = struct.pack("<HH%dH" % len(slots), 4 + 2 * len(slots), 4 + len(body), *slots)
        self._prepend(vt + struct.pack("<i", len(vt)) + bytes(body))
        return pos

    def finish(self, root: int) -> bytes:
        self._prepend(struct.pack("<I", self.size + 4 - root))
        return b"".join(reversed(self.parts))


def write_sentis(convs, iou_threshold: float, score_threshold: float, chunk_bytes: int = 1 << 20) -> bytes:
    """A `.sentis` container in the layout load_sentis reads, holding what the loaders take from the reference's asset:
    per convolution a DequantizeUint8 chain for the weights and one for the bias feeding a Conv / ConvTranspose chain,
    the bias-free DFL convolution (weights 0..15), and a NonMaxSuppression chain whose iou / score thresholds are 0-d
    f32 constants.  convs[i] = (w_q uint8, w_scale, w_zp, b_q uint8, b_scale, b_zp, transposed).  The weight blob is
    split into chunks of `chunk_bytes`."""
    fb, blob = _FBWriter(), bytearray()
    operators = ["DequantizeUint8", "Conv", "ConvTranspose", "NonMaxSuppression"]
    values, chains = [], []

    def tensor(dtype, shape, data=None):           # -> value id; data: bytes of a constant
        if data is not None:
            off = len(blob)
            blob.extend(data)
        body = fb.table([("B", dtype), ("i", len(data) if data is not None else 0), fb.scalars("i", shape),
                         ("I", int(data is not None)), ("i", off if data is not None else 0), ("B", 0)])
        values.append(fb.table([("B", 6), body]))
        return len(values) - 1

    def number(v):
        values.append(fb.table([("B", 3), fb.table([("f", v)])]) if isinstance(v, float) else
                      fb.table([("B", 2), fb.table([("i", v)])]))
        return len(values) - 1

    def chain(op, ins, outs, args=()):
        call = fb.table([("i", operators.index(op)), fb.scalars("i", args)])
        chains.append(fb.table([fb.scalars("i", ins), fb.scalars("i", outs), fb.offsets([fb.table([None, call])])]))

    def dequant(q, scale, zp):
        q = np.ascontiguousarray(q, np.uint8)
        out = tensor(0, q.shape)
        chain("DequantizeUint8", [tensor(3, q.shape, q.tobytes())], [out], [number(float(scale)), number(int(zp))])
        return out

    x = tensor(0, [1, 3, 640, 640])
    for i, (wq, ws, wz, bq, bs, bz, transposed) in enumerate(convs):
        w, b = dequant(wq, ws, wz), dequant(bq, bs, bz)
        chain("ConvTranspose" if transposed else "Conv", [x, w, b], [tensor(0, [])])
        if i == len(convs) - 1:
            chain("Conv", [x, dequant(np.arange(16, dtype=np.uint8).reshape(1, 16, 1, 1), 1.0, 0)], [tensor(0, [])])
    thr = [tensor(0, [], np.float32(t).tobytes()) for t in (iou_threshold, score_threshold)]
    chain("NonMaxSuppression", [x, x, -1] + thr, [tensor(1, [])])

    ops = [fb.table([fb.string(op)]) for op in operators]
    plan = fb.table([None, fb.offsets(values), fb.scalars("i", [x]), fb.offsets([fb.string("images")]), fb.scalars("i", []),
                     fb.offsets([]), fb.offsets(chains), fb.offsets(ops)])
    program = fb.finish(fb.table([("I", 1), plan]))
    out = [struct.pack("<I", len(program)), program]
    for start in range(0, len(blob), chunk_bytes):
        cw = _FBWriter()
        chunk = cw.finish(cw.table([cw.bytes_(blob[start:start + chunk_bytes])]))
        out += [struct.pack("<I", len(chunk)), chunk]
    return b"".join(out)
