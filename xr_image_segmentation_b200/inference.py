"""Host-side mirror of the Unity Inference Engine surface the reference's hot path calls, on top of libxrseg.so.

Reference call sites (Assets/Scripts/InferenceEngine/IEExecutor.cs, "IEE"):
  ModelLoader.Load(asset) IEE:382 | new Worker(model, backend) IEE:383 | Worker.Schedule(t) IEE:385 |
  TextureConverter.ToTensor(tex, 640, 640, 3) IEE:370 | Worker.ScheduleIterable(t) IEE:371 |
  Worker.PeekOutput(i) IEE:426 | Tensor.dataOnBackend / ReadbackRequest() IEE:427 |
  Tensor.IsReadbackRequestDone() IEE:439 | Tensor.ReadbackAndClone() IEE:446-449 | indexers + shape | Dispose().

Same names, argument meaning and ownership rules (peeked tensors are borrowed until the next schedule, clones are
caller-owned).  All arithmetic runs in the CUDA library; this file only moves bytes and tracks state.  `Runner` is the
thin pythonic wrapper of the C ABI used by tests and bench.py (batch > 1, debug entry points).
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _lib
from ._lib import XrsegError


class BackendType:
    GPUCompute = 256   # XRScene.unity:1221
    CPU = 512          # TestScene.unity:747 -- not available here: there is no CPU path in this build


class Model:
    """↔ Unity.InferenceEngine.Model: an XRSW weight pack (or .sentis asset) + the topology scale and class count."""

    def __init__(self, pack: bytes, scale: str = "n", nc: int = 80):
        self.pack = pack
        self.scale = scale
        self.nc = nc


class ModelLoader:
    @staticmethod
    def Load(asset) -> Model:
        """↔ ModelLoader.Load(ModelAsset) IEE:382.  `asset`: path to / bytes of an XRSW pack or a .sentis asset (parsed
        inside libxrseg.so); the scale and class count are read from the weights (xrseg_weights_info)."""
        data = asset if isinstance(asset, (bytes, bytearray)) else open(os.fspath(asset), "rb").read()
        lib = _lib.load_library()
        buf = C.create_string_buffer(bytes(data), len(data))
        scale, nc = C.c_int32(), C.c_int32()
        rc = lib.xrseg_weights_info(C.cast(buf, C.c_void_p), len(data), C.byref(scale), C.byref(nc))
        if rc < 0:
            raise XrsegError(_lib.ERR_WEIGHTS, "not a usable XRSW weight pack or .sentis asset: " + lib.xrseg_last_error(None).decode())
        return Model(bytes(data), chr(scale.value), nc.value)


class Runner:
    """One libxrseg runner (one GPU).  Thin wrapper of the C ABI."""

    def __init__(self, model: Model, device: int = 0, max_batch: int = 1, iou=0.0, score=0.0, mask_thr=0.0,
                 max_det=0, max_candidates=0, resize_mode=_lib.RESIZE_STRETCH, conv_impl=_lib.CONV_UMMA,
                 use_cuda_graph=True, micro_batch=0, debug=False, num_classes=0):
        # debug=True: the runner lives in libxrseg_debug.so (same sources + the parity hooks of include/xrseg_debug.h:
        # fetch / debug_post / debug_nms / debug_mask_threshold); the product library exports none of them
        self.debug = debug
        self.lib = _lib.load_library(debug)
        self._pack = C.create_string_buffer(model.pack, len(model.pack))
        cfg = _lib.Config()
        cfg.struct_size = C.sizeof(_lib.Config)
        cfg.device = device
        cfg.max_batch = max_batch
        cfg.model_scale = ord(model.scale)
        cfg.weights = C.cast(self._pack, C.c_void_p)
        cfg.weights_bytes = len(model.pack)
        cfg.iou_threshold, cfg.score_threshold, cfg.mask_threshold = iou, score, mask_thr
        cfg.max_det, cfg.max_candidates = max_det, max_candidates
        cfg.resize_mode, cfg.conv_impl = resize_mode, conv_impl
        cfg.use_cuda_graph = 1 if use_cuda_graph else 0
        cfg.micro_batch = micro_batch
        cfg.num_classes = num_classes
        self.h = C.c_void_p()
        _lib.check(self.lib.xrseg_create(C.byref(cfg), C.byref(self.h)), None, self.lib)
        self.max_batch = max_batch
        self.batch = 0
        self._max_det = max_det if max_det > 0 else 300          # the library's default cap per frame (xrseg_config.max_det)
        self._collect_buf = None

    @property
    def num_classes(self) -> int:
        """Classes of the runner's model (labels are 0 .. num_classes - 1)."""
        return self._ck(self.lib.xrseg_num_classes(self.h))

    def close(self):
        if getattr(self, "h", None) and self.h.value:
            self.lib.xrseg_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        return _lib.check(rc, self.h, self.lib)

    def _need_debug(self):
        if not self.debug:
            raise XrsegError(_lib.ERR_STATE, "parity hook: create the Runner with debug=True (libxrseg_debug.so)")

    # ---- per-frame path ----
    def schedule(self, frames: np.ndarray, fmt=None, bottom_up=False, stride_bytes=None):
        """frames uint8 [B,H,W,3|4] (host).  Asynchronous.  bottom_up: memory row 0 is the BOTTOM of the picture (Unity's
        GetPixels32 order, XRSEG_FMT_BOTTOM_UP).  stride_bytes: row pitch of padded rows (default w * c); frames is then a
        view whose rows lie stride_bytes apart and whose frames lie h * stride_bytes apart."""
        assert frames.dtype == np.uint8 and frames.ndim == 4
        b, h, w, c = frames.shape
        stride_bytes = w * c if stride_bytes is None else stride_bytes
        want = (h * stride_bytes, stride_bytes, c, 1)
        assert all(n == 1 or s == t for n, s, t in zip(frames.shape, frames.strides, want)), (frames.strides, stride_bytes)
        fmt = (_lib.FMT_RGBA8 if c == 4 else _lib.FMT_RGB8) if fmt is None else fmt
        if bottom_up:
            fmt |= _lib.FMT_BOTTOM_UP
        self._keep = frames
        self.batch = b
        self._ck(self.lib.xrseg_schedule(self.h, frames.ctypes.data, w, h, stride_bytes, fmt, b))

    def schedule_ptr(self, host_ptr: int, b, h, w, c):
        self.batch = b
        self._ck(self.lib.xrseg_schedule(self.h, host_ptr, w, h, w * c, _lib.FMT_RGBA8 if c == 4 else _lib.FMT_RGB8, b))

    def schedule_device(self, dev_ptr: int, b, h, w, c, stride_bytes=None):
        """dev_ptr: frames already on the runner's GPU, rows stride_bytes apart (default w * c), frames h * stride_bytes apart."""
        self.batch = b
        stride_bytes = w * c if stride_bytes is None else stride_bytes
        self._ck(self.lib.xrseg_schedule_device(self.h, dev_ptr, w, h, stride_bytes, _lib.FMT_RGBA8 if c == 4 else _lib.FMT_RGB8, b))

    def poll(self) -> int:
        return self._ck(self.lib.xrseg_poll(self.h))

    def wait(self, strict=True):
        """Blocks until the run is complete.  A run that hit max_candidates / max_det raises XrsegError(ERR_CAPACITY) once
        (strict=False: returns the overflow bits instead; the truncated results stay readable either way)."""
        rc = self.lib.xrseg_wait(self.h)
        if rc == _lib.ERR_CAPACITY and not strict:
            return self.overflow()
        self._ck(rc)
        return 0

    def overflow(self) -> int:
        """Capacity flags of the finished run (bit 0: candidates > max_candidates, bit 1: kept > max_det)."""
        return self._ck(self.lib.xrseg_overflow(self.h))

    def counts(self) -> np.ndarray:
        out = np.zeros(self.max_batch, np.int32)
        n = self._ck(self.lib.xrseg_counts(self.h, out.ctypes.data_as(C.POINTER(C.c_int32)), self.max_batch))
        return out[:n]

    def peek(self, idx: int) -> _lib.TensorView:
        v = _lib.TensorView()
        self._ck(self.lib.xrseg_peek_output(self.h, idx, C.byref(v)))
        return v

    _DT = {0: np.float32, 1: np.int32}

    def readback(self, idx: int) -> np.ndarray:
        v = self.peek(idx)
        shape = [int(v.shape[i]) for i in range(v.rank)]
        out = np.empty(shape, self._DT[v.dtype])
        shp = (C.c_int64 * 4)()
        rank = C.c_int()
        self._ck(self.lib.xrseg_readback(self.h, idx, out.ctypes.data, out.nbytes, shp, C.byref(rank)))
        return out

    def readback_into(self, idx: int, host_ptr: int, cap_bytes: int):
        """↔ ReadbackAndClone into caller memory (e.g. pinned memory of xrseg_host_alloc): returns the tensor's shape."""
        shp = (C.c_int64 * 4)()
        rank = C.c_int()
        self._ck(self.lib.xrseg_readback(self.h, idx, host_ptr, cap_bytes, shp, C.byref(rank)))
        return tuple(int(shp[i]) for i in range(rank.value))

    def keep_indices(self):
        n = int(self.peek(0).shape[0])
        idx = np.zeros(max(n, 1), np.int32)
        sc = np.zeros(max(n, 1), np.float32)
        self._ck(self.lib.xrseg_keep_indices(self.h, idx.ctypes.data_as(C.POINTER(C.c_int32)),
                                             sc.ctypes.data_as(C.POINTER(C.c_float)), max(n, 1)))
        return idx[:n], sc[:n]

    def decode(self, screen_w: float, screen_h: float, convention: int):
        cap = max(1, int(self.peek(0).shape[0]))
        arr = (_lib.Box * cap)()
        n = C.c_int()
        self._ck(self.lib.xrseg_decode(self.h, screen_w, screen_h, convention, arr, cap, C.byref(n)))
        out = np.zeros((n.value, 4), np.float32)
        lab = np.zeros(n.value, np.int32)
        frm = np.zeros(n.value, np.int32)
        for i in range(n.value):
            out[i] = (arr[i].center_x, arr[i].center_y, arr[i].width, arr[i].height)
            lab[i] = arr[i].label_id
            frm[i] = arr[i].frame
        return out, lab, frm

    def masks(self, mode: int, box_convention=_lib.BOX_DRAWBOXES, screen_w=640.0, screen_h=640.0, image_w=640,
              image_h=640, first=0, count=0, threshold=0.0, to_host=True) -> np.ndarray:
        total = int(self.peek(0).shape[0])
        n = count if count > 0 else total - first
        shape = {_lib.MASK_REFERENCE_160: (n, 160, 160), _lib.MASK_CROP_160: (n, 160, 160),
                 _lib.MASK_UPSAMPLE_640: (n, 640, 640), _lib.MASK_BITS_160: (n, 160, 20)}[mode]
        out = np.zeros(shape, np.uint8) if to_host else None
        if n == 0:
            return out
        p = _lib.MaskParams(C.sizeof(_lib.MaskParams), mode, box_convention, screen_w, screen_h, image_w, image_h, first, n,
                            threshold)
        if not to_host:                                   # masks stay in the runner's device scratch (kernel timing)
            self._ck(self.lib.xrseg_masks(self.h, C.byref(p), None, 0))
            return None
        self._ck(self.lib.xrseg_masks(self.h, C.byref(p), out.ctypes.data, out.nbytes))
        return out.view(np.uint32).reshape(n, 160, 5) if mode == _lib.MASK_BITS_160 else out

    def collect(self, mask_mode: int = _lib.MASK_BITS_160, box_convention=_lib.BOX_DRAWBOXES, screen_w=640.0, screen_h=640.0,
                image_w=640, image_h=640, threshold=0.0):
        """xrseg_collect: waits for the run and returns (counts, boxes f32 [N,4], labels i32 [N], masks) with ONE call and ONE
        synchronisation (what a frame loop reads back; the four raw tensors stay available through readback()).  mask_mode None:
        no masks.  max_det bounds the buffers, so nothing is peeked first."""
        cap = self.max_batch * self._max_det
        if self._collect_buf is None or self._collect_buf[0].shape[0] < cap:
            per = {_lib.MASK_BITS_160: 160 * 20, _lib.MASK_REFERENCE_160: 160 * 160, _lib.MASK_CROP_160: 160 * 160}
            self._collect_buf = (np.empty((cap, 4), np.float32), np.empty(cap, np.int32), {m: None for m in per}, per)
        boxes, labels, mbufs, per = self._collect_buf
        mp = None
        masks = None
        if mask_mode is not None:
            if mask_mode not in per:
                raise XrsegError(_lib.ERR_INVALID, "collect(): mask mode not supported here (use masks())")
            if mbufs[mask_mode] is None:
                mbufs[mask_mode] = np.empty(cap * per[mask_mode], np.uint8)
            masks = mbufs[mask_mode]
            mp = _lib.MaskParams(C.sizeof(_lib.MaskParams), mask_mode, box_convention, screen_w, screen_h, image_w, image_h, 0, 0,
                                 threshold)
        n = self.lib.xrseg_collect(self.h, boxes.ctypes.data, labels.ctypes.data, cap, C.byref(mp) if mp is not None else None,
                                   masks.ctypes.data if masks is not None else None, masks.nbytes if masks is not None else 0)
        if n == _lib.ERR_CAPACITY and self.overflow():          # a truncated run: same contract as wait()
            self._ck(n)
        n = self._ck(n)
        m = None
        if masks is not None:
            m = masks[:n * per[mask_mode]]
            m = m.view(np.uint32).reshape(n, 160, 5) if mask_mode == _lib.MASK_BITS_160 else m.reshape(n, 160, 160)
        return self.counts(), boxes[:n], labels[:n], m

    def extract_points(self, detection: int, depth_half: np.ndarray, screen_w: float, screen_h: float, camera_position,
                       camera_rotation, focal_length, principal_point, sensor_resolution, sampling_step=5, max_points=8000,
                       confidence_threshold=0.0) -> np.ndarray:
        """↔ IEExecutor.ExtractDepthData (IEE:561-667).  depth_half: uint16 [H,W] half floats.  Returns f32 [n,4] x,y,z,depth."""
        d = np.ascontiguousarray(depth_half, np.uint16)
        p = _lib.DepthParams()
        p.struct_size = C.sizeof(_lib.DepthParams)
        p.detection, p.depth_h, p.depth_w = detection, d.shape[0], d.shape[1]
        p.sampling_step, p.max_points, p.confidence_threshold = sampling_step, max_points, confidence_threshold
        p.screen_w, p.screen_h = screen_w, screen_h
        p.camera_position[:] = [float(v) for v in camera_position]
        p.camera_rotation[:] = [float(v) for v in camera_rotation]
        p.focal_length[:] = [float(v) for v in focal_length]
        p.principal_point[:] = [float(v) for v in principal_point]
        p.sensor_resolution[:] = [float(v) for v in sensor_resolution]
        out = np.zeros((max_points, 4), np.float32)
        n = C.c_int()
        self._ck(self.lib.xrseg_extract_points(self.h, C.byref(p), d.ctypes.data, out.ctypes.data, max_points, C.byref(n)))
        return out[:n.value]

    def associate(self, frame: int, locked_cx: float, locked_cy: float, locked_label: int, screen_w: float, screen_h: float,
                  max_dist: float = 300.0):
        """↔ the locked-target search of ProcessInferenceResult (IEE:488-507): (index inside the frame or -1, min distance)."""
        idx, dist = C.c_int(), C.c_float()
        self._ck(self.lib.xrseg_associate(self.h, frame, locked_cx, locked_cy, locked_label, screen_w, screen_h, max_dist,
                                          C.byref(idx), C.byref(dist)))
        return idx.value, dist.value

    def timings(self):
        ms = (C.c_float * 5)()
        self._ck(self.lib.xrseg_last_timings(self.h, ms, 5))
        return list(ms)

    def launch_count(self) -> int:
        return self.lib.xrseg_launch_count(self.h)

    def event_record(self, slot: int):
        self._ck(self.lib.xrseg_event_record(self.h, slot))

    def event_elapsed_ms(self, a: int, b: int) -> float:
        ms = C.c_float()
        self._ck(self.lib.xrseg_event_elapsed_ms(self.h, a, b, C.byref(ms)))
        return ms.value

    def sync(self):
        self._ck(self.lib.xrseg_sync(self.h))

    def profile_ops(self, iters: int = 5):
        """Per-launch device time of the last scheduled input: list of (name, ms, flops, bytes)."""
        cap = 512
        ms = (C.c_float * cap)()
        names = C.create_string_buffer(cap * 32)
        fl = (C.c_double * cap)()
        by = (C.c_double * cap)()
        n = self._ck(self.lib.xrseg_profile_ops(self.h, iters, ms, names, fl, by, cap))
        return [(names.raw[i * 32:(i + 1) * 32].split(b"\0")[0].decode(), ms[i], fl[i], by[i]) for i in range(n)]

    # ---- parity / debug ----
    def fetch(self, name: str, first: int = 0, count: int = -1) -> np.ndarray:
        """A named activation of the last run, frames [first, first + count) of the resident chunk (count -1: all)."""
        self._need_debug()
        shp = (C.c_int64 * 4)()
        probe = np.empty(1, np.float32)                  # a zero-capacity call reports the shape (class logits grow with nc)
        rc = self.lib.xrseg_debug_fetch_frames(self.h, name.encode(), first, count, probe.ctypes.data, 0, shp)
        if rc != _lib.ERR_CAPACITY:
            self._ck(rc)
        shape = [int(s) for s in shp]
        n = int(np.prod(shape))
        buf = np.empty(max(n, 1), np.float32)
        self._ck(self.lib.xrseg_debug_fetch_frames(self.h, name.encode(), first, count, buf.ctypes.data, n, shp))
        return buf[:n].reshape(shape)

    def launches(self) -> list[tuple[str, int, int, int]]:
        """The last run's launch list (resident chunk): (name, grid CTAs, work items, conv mode or -1) per launch."""
        self._need_debug()
        cap = 512
        g, it, md = (C.c_int * cap)(), (C.c_int * cap)(), (C.c_int * cap)()
        names = C.create_string_buffer(cap * 32)
        n = self._ck(self.lib.xrseg_debug_launches(self.h, g, it, md, names, cap))
        return [(names.raw[i * 32:(i + 1) * 32].split(b"\0")[0].decode(), g[i], it[i], md[i]) for i in range(n)]

    def debug_post(self, box_logits, cls_logits, coefs, protos, f16=False):
        """Post-processing alone on caller tensors: fp32 bit-exact kernels, or (f16) the product's fp16 kernels."""
        self._need_debug()
        arrs = [np.ascontiguousarray(a, np.float32) for a in (box_logits, cls_logits, coefs, protos)]
        if arrs[1].shape[-1] != self.num_classes:
            raise ValueError(f"cls_logits have {arrs[1].shape[-1]} classes, the runner's model {self.num_classes}")
        b = arrs[0].shape[0]
        self.batch = b
        fn = self.lib.xrseg_debug_post_f16 if f16 else self.lib.xrseg_debug_post
        self._ck(fn(self.h, *(a.ctypes.data for a in arrs), b))

    def debug_post_timings(self):
        """(name, ms, algorithmic bytes) per launch of the last debug_post call made with XRSEG_DBG_TIME=1."""
        self._need_debug()
        cap = 64
        ms, by, names = (C.c_float * cap)(), (C.c_double * cap)(), C.create_string_buffer(cap * 32)
        n = self._ck(self.lib.xrseg_debug_post_timings(self.h, ms, by, names, cap))
        return [(names.raw[i * 32:(i + 1) * 32].split(b"\0")[0].decode(), ms[i], by[i]) for i in range(n)]

    def debug_nms(self, corners, scores):
        self._need_debug()
        c = np.ascontiguousarray(corners, np.float32)
        s = np.ascontiguousarray(scores, np.float32)
        self.batch = c.shape[0]
        self._ck(self.lib.xrseg_debug_nms(self.h, c.ctypes.data, s.ctypes.data, c.shape[0], c.shape[1]))

    def debug_mask_threshold(self, probs, boxes, image_w, image_h, thr=0.5):
        self._need_debug()
        p = np.ascontiguousarray(probs, np.float32)
        bx = np.ascontiguousarray(boxes, np.float32)
        out = np.zeros(p.shape, np.uint8)
        self._ck(self.lib.xrseg_debug_mask_threshold(self.h, p.ctypes.data, bx.ctypes.data, p.shape[0], image_w, image_h,
                                                     thr, out.ctypes.data))
        return out


class PipelinedRunner:
    """`depth` runners on one GPU used round-robin: the host->device copy and the network pass of submission i+1
    overlap the readback of submission i (each runner still has exactly one run in flight, like the reference's
    `_started` gate, IEE:365).  Throughput-oriented callers use this instead of a single Runner."""

    def __init__(self, model: Model, device: int = 0, max_batch: int = 1, depth: int = 2, **runner_kw):
        self.runners = [Runner(model, device=device, max_batch=max_batch, **runner_kw) for _ in range(depth)]
        self._head = 0          # next runner to submit to
        self._inflight = []     # runner indices in submission order

    def submit_ptr(self, host_ptr: int, b, h, w, c):
        if len(self._inflight) == len(self.runners):
            raise XrsegError(_lib.ERR_STATE, "pipeline full: collect() first")
        self.runners[self._head].schedule_ptr(host_ptr, b, h, w, c)
        self._inflight.append(self._head)
        self._head = (self._head + 1) % len(self.runners)

    def submit(self, frames: np.ndarray):
        if len(self._inflight) == len(self.runners):
            raise XrsegError(_lib.ERR_STATE, "pipeline full: collect() first")
        self.runners[self._head].schedule(frames)
        self._inflight.append(self._head)
        self._head = (self._head + 1) % len(self.runners)

    def collect(self, mask_mode=_lib.MASK_BITS_160, contract=False, pinned=None):
        """Results of the oldest submission: (counts, boxes [N,4], labels [N], masks).  contract=True: the reference's own
        readback instead -- all four graph outputs as ReadbackAndClone would return them (IEE:446-449): (counts, output_0
        f32 [N,4], output_1 i32 [N], output_2 f32 [N,32], output_3 f32 [N,160,160])."""
        if not self._inflight:
            raise XrsegError(_lib.ERR_STATE, "nothing in flight")
        r = self.runners[self._inflight.pop(0)]
        r.wait()
        if contract and pinned is not None:           # pinned = [(host_ptr, cap_bytes)] * 4: returns the four shapes
            return (r.counts(),) + tuple(r.readback_into(i, *pinned[i]) for i in range(4))
        if contract:
            return (r.counts(),) + tuple(r.readback(i) for i in range(4))
        if mask_mode in (_lib.MASK_BITS_160, _lib.MASK_REFERENCE_160, _lib.MASK_CROP_160):
            c, b, l, m = r.collect(mask_mode)                 # one call, one synchronisation
            return c, b.copy(), l.copy(), m.copy()
        return r.counts(), r.readback(0), r.readback(1), r.masks(mask_mode)

    def close(self):
        for r in self.runners:
            r.close()


def debug_conv(x, w, b, k, stride, act, transposed=False, residual=None, impl=_lib.CONV_UMMA, variant=0, device=0):
    """One convolution through the CUDA library (parity tests; libxrseg_debug.so)."""
    lib = _lib.load_library(True)
    x = np.ascontiguousarray(x, np.float32)
    w = np.ascontiguousarray(w, np.float32)
    B, cin, h, wd = x.shape
    cout = w.shape[1] if transposed else w.shape[0]
    ho = h * 2 if transposed else (h + 2 * (k // 2) - k) // stride + 1
    wo = wd * 2 if transposed else (wd + 2 * (k // 2) - k) // stride + 1
    y = np.zeros((B, cout, ho, wo), np.float32)
    bb = None if b is None else np.ascontiguousarray(b, np.float32)
    rr = None if residual is None else np.ascontiguousarray(residual, np.float32)
    _lib.check(lib.xrseg_debug_conv(device, impl, x.ctypes.data, B, cin, h, wd, w.ctypes.data,
                                    bb.ctypes.data if bb is not None else None, cout, k, stride, 1, int(act),
                                    int(transposed), rr.ctypes.data if rr is not None else None, y.ctypes.data, variant), None, lib)
    return y


def debug_bottleneck(x, w1, b1, w2, b2, residual=True, device=0):
    """The fused Bottleneck kernel (Conv3x3+SiLU -> Conv3x3+SiLU (+ x)) on caller tensors (parity tests)."""
    lib = _lib.load_library(True)
    x, w1, b1, w2, b2 = (np.ascontiguousarray(a, np.float32) for a in (x, w1, b1, w2, b2))
    B, c1, h, wd = x.shape
    cm, c2 = w1.shape[0], w2.shape[0]
    y = np.zeros((B, c2, h, wd), np.float32)
    _lib.check(lib.xrseg_debug_bottleneck(device, x.ctypes.data, B, c1, h, wd, w1.ctypes.data, b1.ctypes.data, cm,
                                          w2.ctypes.data, b2.ctypes.data, c2, int(residual), y.ctypes.data), None, lib)
    return y


def debug_attention(qkv, heads, device=0, pe_w=None, pe_b=None, map_w=0):
    """The C2PSA attention kernel alone: qkv f32 [B,N,heads*128] (per head 32 q | 32 k | 64 v) -> [B,N,heads*64].
    pe_w [heads*64,3,3] / pe_b [heads*64] / map_w: the fused positional encoding (depthwise 3x3 on the V map) is added."""
    lib = _lib.load_library(True)
    q = np.ascontiguousarray(qkv, np.float32)
    B, N, _ = q.shape
    y = np.zeros((B, N, heads * 64), np.float32)
    w = np.ascontiguousarray(pe_w, np.float32) if pe_w is not None else None
    bb = np.ascontiguousarray(pe_b, np.float32) if pe_b is not None else None
    _lib.check(lib.xrseg_debug_attention(device, q.ctypes.data, B, N, heads, y.ctypes.data, w.ctypes.data if w is not None else None,
                                         bb.ctypes.data if bb is not None else None, map_w), None, lib)
    return y


# --------------------------------------------------------------------------------------------------
# Inference Engine mirror
# --------------------------------------------------------------------------------------------------
class Tensor:
    """↔ Tensor<float> / Tensor<int>.  Either a host tensor (owns `array`) or a worker-owned backend tensor."""

    def __init__(self, array: np.ndarray | None = None, worker: "Worker | None" = None, index: int = -1):
        self._array = array
        self._worker = worker
        self._index = index
        self._requested = False
        self.disposed = False

    @property
    def dataOnBackend(self):
        """Non-None when the tensor has device data (IEE:427)."""
        if self._worker is None:
            return None
        return self._worker._runner.peek(self._index).device_ptr or None

    @property
    def shape(self):
        if self._array is not None:
            return tuple(self._array.shape)
        v = self._worker._runner.peek(self._index)
        return tuple(int(v.shape[i]) for i in range(v.rank))

    def ReadbackRequest(self):
        self._requested = True

    def IsReadbackRequestDone(self) -> bool:
        return self._worker._runner.poll() == 1

    def ReadbackAndClone(self) -> "Tensor":
        return Tensor(array=self._worker._runner.readback(self._index))

    def __getitem__(self, idx):
        if self._array is None:
            raise XrsegError(_lib.ERR_STATE, "backend tensor: ReadbackAndClone() first")
        return self._array[idx]

    def numpy(self) -> np.ndarray:
        return self._array

    def Dispose(self):
        self.disposed = True
        self._array = None


class InputTensor(Tensor):
    """Result of TextureConverter.ToTensor: the frame bytes; the resample to 640x640 runs on the GPU at schedule time."""

    def __init__(self, frame_u8: np.ndarray, width: int, height: int, channels: int):
        super().__init__(array=np.ascontiguousarray(frame_u8))
        self.target = (width, height, channels)


class TextureConverter:
    @staticmethod
    def ToTensor(texture: np.ndarray, width: int = 640, height: int = 640, channels: int = 3) -> InputTensor:
        """↔ TextureConverter.ToTensor(tex, 640, 640, 3) IEE:370.  texture: uint8 [H,W,3|4], top row first."""
        if (width, height, channels) != (640, 640, 3):
            raise XrsegError(_lib.ERR_INVALID, "the network input is 640x640x3")
        t = np.asarray(texture)
        if t.dtype != np.uint8 or t.ndim != 3 or t.shape[2] not in (3, 4):
            raise XrsegError(_lib.ERR_INVALID, "texture must be uint8 [H,W,3|4]")
        return InputTensor(t, width, height, channels)


class _Schedule:
    """↔ the IEnumerator returned by Worker.ScheduleIterable: MoveNext() is True while the run is in flight."""

    def __init__(self, worker: "Worker"):
        self._w = worker
        self._started = False

    def MoveNext(self) -> bool:
        if not self._started:
            self._w._enqueue()
            self._started = True
            return True
        return self._w._runner.poll() != 1

    def __iter__(self):
        return self

    def __next__(self):
        if not self.MoveNext():
            raise StopIteration
        return None


class Worker:
    """↔ Unity.InferenceEngine.Worker for this model (IEE:383-385, 371, 426, 303)."""

    def __init__(self, model: Model, backend: int = BackendType.GPUCompute, device: int = 0, **runner_kw):
        if backend != BackendType.GPUCompute:
            raise XrsegError(_lib.ERR_NO_DEVICE, "only BackendType.GPUCompute exists in this build (no CPU fallback)")
        self._runner = Runner(model, device=device, max_batch=1, **runner_kw)
        self._input = None

    def _enqueue(self):
        f = self._input.numpy()
        self._runner.schedule(f[None])

    def Schedule(self, input: InputTensor):
        """↔ Worker.Schedule(tensor) IEE:385: enqueue the whole run."""
        self._input = input
        self._enqueue()

    def ScheduleIterable(self, input: InputTensor) -> _Schedule:
        """↔ Worker.ScheduleIterable(tensor) IEE:371."""
        self._input = input
        return _Schedule(self)

    def PeekOutput(self, index: int) -> Tensor:
        """↔ Worker.PeekOutput(i) IEE:426: borrowed, valid until the next schedule."""
        if not 0 <= index <= 3:
            raise XrsegError(_lib.ERR_INVALID, "the model has outputs 0..3")
        return Tensor(worker=self, index=index)

    def Dispose(self):
        self._runner.close()
