"""CPU tests of the drop-in boundary: libxrseg.so loads, exports every symbol include/xrseg.h declares, reports the
same topology as the oracle, fails loudly without a GPU, and its conv index math (host emulation of the tcgen05
kernel's data movement) reproduces torch convolutions."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import yolo11seg as Y
from xr_image_segmentation_b200 import _lib, inference as I, sharding as S, weights as W

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def _declared(header):
    hdr = open(os.path.join(ROOT, "include", header)).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)                  # declarations only, not names mentioned in comments
    return set(re.findall(r"\b(xrseg_[a-z0-9_]+)\s*\(", hdr))


def test_exports_every_declared_symbol(lib, dlib):
    product, debug = _declared("xrseg.h"), _declared("xrseg_debug.h")
    assert len(product) >= 28 and len(debug) >= 11 and not (product & debug)
    assert product == set(_lib.PRODUCT_SIGNATURES) and debug == set(_lib.DEBUG_SIGNATURES)
    for name in sorted(product):
        assert hasattr(lib, name), f"{name} declared in include/xrseg.h but not exported by libxrseg.so"
        assert hasattr(dlib, name), f"{name} missing from libxrseg_debug.so"
    for name in sorted(debug):
        assert hasattr(dlib, name), f"{name} declared in include/xrseg_debug.h but not exported by libxrseg_debug.so"
        assert not hasattr(lib, name), f"the product library exports the debug hook {name}"
    assert lib.xrseg_abi_version() == dlib.xrseg_abi_version() == _lib.ABI_VERSION == 2
    assert C.sizeof(_lib.Config) == 104 and C.sizeof(_lib.MaskParams) == 40


@pytest.mark.parametrize("scale", ["n", "s"])
def test_layer_table_matches_oracle(lib, scale):
    a, b = W.layer_table(scale), Y.layer_table(scale)
    assert len(a) == len(b) == 100
    for x, y in zip(a, b):
        assert (x.name, x.cin, x.cout, x.k, x.stride, x.groups, x.act, x.transposed, x.h_in, x.w_in) == \
               (y["name"], y["cin"], y["cout"], y["k"], y["s"], y["groups"], int(y["act"]), int(y["transposed"]), y["h_in"], y["w_in"])
        assert x.weight_shape == Y.weight_shape(y)
    assert lib.xrseg_layer_count(ord("x")) < 0


def test_no_gpu_means_loud_failure(lib, golden):
    if lib.xrseg_device_count() > 0:
        pytest.skip("a B200 is present")
    with pytest.raises(I.XrsegError) as e:
        I.Runner(golden["model"])
    assert e.value.code == _lib.ERR_NO_DEVICE and "no CPU fallback" in str(e.value)
    with pytest.raises(I.XrsegError):
        I.Worker(golden["model"], I.BackendType.CPU)
    with pytest.raises(I.XrsegError):
        I.ModelLoader.Load(b"not a pack")
    with pytest.raises(I.XrsegError):
        I.TextureConverter.ToTensor(np.zeros((4, 4, 3), np.uint8), 320, 320, 3)


def test_weight_pack_roundtrip_and_validation(lib):
    layers, ws = W.random_weights("n", seed=1)
    pack = W.write_pack("n", layers, ws)
    scale, back = W.read_pack(pack)
    assert scale == "n" and len(back) == 100
    for (w, b), (_, w2, b2) in zip(ws, back):
        assert np.array_equal(w, w2) and np.array_equal(b, b2)
    # same seed -> same weights as the oracle-side generator (the two must agree for parity tests)
    ow = Y.random_weights("n", 1)
    for (w, b), (w2, b2) in zip(ws, ow):
        assert np.array_equal(w, w2) and np.array_equal(b, b2)
    q = W.Tensor8(np.array([0, 85, 255], np.uint8), 0.0058823530562222, 85)
    np.testing.assert_allclose(q.dequant(), [-0.5, 0.0, 1.0], atol=1e-6)


CASES = [
    (2, 16, 8, 12, 10, 3, 1, 1, False, True, 0), (2, 16, 8, 12, 10, 3, 1, 1, False, True, 1),
    (1, 32, 16, 20, 20, 3, 1, 0, False, False, 0), (2, 48, 64, 9, 7, 1, 1, 1, False, True, 0),
    (1, 16, 32, 13, 11, 3, 2, 1, False, False, 0), (2, 8, 16, 6, 5, 3, 1, 1, False, False, 0),
    (1, 64, 64, 5, 6, 2, 2, 0, True, False, 0), (1, 80, 80, 7, 7, 1, 1, 0, False, False, 0),
    (3, 128, 32, 4, 4, 3, 1, 1, False, True, 0), (1, 16, 8, 3, 170, 3, 1, 1, False, False, 0),
    (1, 256, 512, 3, 3, 1, 1, 1, False, False, 0), (1, 128, 128, 3, 3, 2, 2, 0, True, False, 0),
    (1, 256, 64, 5, 4, 3, 1, 1, False, False, 0),
    # stride-2 3x3 on even maps -> parity-plane TMA mode (variant 0); flat 1x1 with a partial last K-block / 2 N tiles
    (1, 16, 32, 12, 10, 3, 2, 1, False, False, 0), (2, 64, 64, 8, 8, 3, 2, 1, False, False, 0),
    (1, 128, 256, 6, 4, 3, 2, 0, False, False, 0), (1, 32, 16, 40, 6, 3, 2, 1, False, False, 0),
    (2, 144, 32, 5, 5, 1, 1, 1, False, False, 0), (1, 512, 256, 4, 4, 1, 1, 1, False, True, 0),
]


@pytest.mark.parametrize("case", CASES)
def test_umma_conv_index_math_emulation(dlib, case):
    """Host emulation (fp32) of the tcgen05 kernel's packing / slot mapping / tap shifts / epilogue scatter."""
    B, cin, cout, h, wd, k, s, act, tr, useres, variant = case
    rng = np.random.default_rng(hash(case) % 2**32)
    x = rng.standard_normal((B, cin, h, wd), dtype=np.float32)
    w = rng.standard_normal((cin, cout, k, k) if tr else (cout, cin, k, k), dtype=np.float32) * np.float32(0.1)
    b = rng.standard_normal(cout, dtype=np.float32)
    if tr:
        ref = F.conv_transpose2d(torch.from_numpy(x), torch.from_numpy(w), torch.from_numpy(b), stride=2)
    else:
        ref = F.conv2d(torch.from_numpy(x), torch.from_numpy(w), torch.from_numpy(b), stride=s, padding=k // 2)
    if act:
        ref = ref * torch.sigmoid(ref)
    res = None
    if useres:
        res = rng.standard_normal(tuple(ref.shape), dtype=np.float32)
        ref = ref + torch.from_numpy(res)
    y = np.zeros(tuple(ref.shape), np.float32)
    rc = dlib.xrseg_debug_emulate_conv(x.ctypes.data, B, cin, h, wd, w.ctypes.data, b.ctypes.data, cout, k, s, act, int(tr),
                                      res.ctypes.data if res is not None else None, y.ctypes.data, variant)
    assert rc == 0, lib.xrseg_last_error(None)
    np.testing.assert_allclose(y, ref.numpy(), atol=2e-5, rtol=1e-5)


def test_shard_range_and_merge():
    for total in (0, 1, 7, 64, 512):
        for world in (1, 2, 3, 4, 8):
            spans = [S.shard_range(total, world, r) for r in range(world)]
            assert spans[0][0] == 0 and sum(c for _, c in spans) == total
            for (s0, c0), (s1, _) in zip(spans, spans[1:]):
                assert s0 + c0 == s1
            assert max(c for _, c in spans) - min(c for _, c in spans) <= 1
    with pytest.raises(ValueError):
        S.shard_range(8, 2, 2)
    a = S.Detections(0, np.array([1, 0]), np.ones((1, 4), np.float32), np.array([3]), np.array([0.9], np.float32))
    b = S.Detections(2, np.array([2]), np.zeros((2, 4), np.float32), np.array([1, 2]), np.array([0.8, 0.7], np.float32))
    m = S.merge_detections([b, a])
    assert m.counts.tolist() == [1, 0, 2] and m.labels.tolist() == [3, 1, 2] and m.boxes.shape == (3, 4)
    with pytest.raises(ValueError):
        S.merge_detections([a, S.Detections(3, np.array([0]), np.zeros((0, 4), np.float32), np.zeros(0, np.int64))])


# ---- .sentis loader inside the library (SURVEY.md §8f N2) ------------------------------------------------------------
def test_sentis_loader_matches_oracle_reader_and_golden_pack(lib, golden, golden_sentis):
    """The C++ FlatBuffer walk + uint8 dequantization (csrc/sentis.cuh) against the oracle's Python reader and the committed
    XRSW pack the container was written from: every convolution, bit for bit; thresholds as decoded in SURVEY.md fact 3."""
    import ctypes as C

    from oracle.sentis import load_sentis
    from xr_image_segmentation_b200 import weights as W
    data = golden_sentis
    buf = C.create_string_buffer(data, len(data))
    ptr = C.cast(buf, C.c_void_p)
    n, iou, sc = C.c_int32(), C.c_float(), C.c_float()
    assert lib.xrseg_sentis_info(ptr, len(data), C.byref(n), C.byref(iou), C.byref(sc)) == 0
    assert n.value == 100 and abs(iou.value - 0.43) < 1e-6 and abs(sc.value - 0.301) < 1e-6
    # oracle reader: DequantizeUint8 chains feeding Conv / ConvTranspose chains in file order
    m = load_sentis(data)
    deq, ref = {}, []
    for c in m.chains:
        if c.op == "DequantizeUint8":
            deq[c.outputs[0]] = W.Tensor8(m.values[c.inputs[0]].data, m.values[c.args[0]], m.values[c.args[1]]).dequant()
        elif c.op in ("Conv", "ConvTranspose") and len(c.inputs) >= 3 and c.inputs[2] >= 0:
            ref.append((deq[c.inputs[1]], deq[c.inputs[2]], c.op == "ConvTranspose"))
    _, packed = W.read_pack(golden["model"].pack)
    assert len(ref) == 100 == len(packed)
    for i, (w, b, tr) in enumerate(ref):
        wb, bb = np.zeros(w.size, np.float32), np.zeros(b.size, np.float32)
        shp, t = (C.c_int32 * 4)(), C.c_int32()
        rc = lib.xrseg_sentis_layer(ptr, len(data), i, wb.ctypes.data, wb.size, bb.ctypes.data, bb.size, shp, C.byref(t))
        assert rc == w.size and list(shp) == list(w.shape) and bool(t.value) == tr
        assert np.array_equal(wb.reshape(w.shape), w) and np.array_equal(bb, b)
        assert np.array_equal(w, packed[i][1]) and np.array_equal(b, packed[i][2])
    # ModelLoader.Load accepts the asset bytes unchanged (IEE:382)
    from xr_image_segmentation_b200 import inference as I
    assert I.ModelLoader.Load(data).scale == "n"


def test_sentis_loader_rejects_corrupt_input(lib, golden_sentis):
    import ctypes as C
    data = bytearray(golden_sentis)
    n = C.c_int32()

    def info(b):
        buf = C.create_string_buffer(bytes(b), len(b))
        return lib.xrseg_sentis_info(C.cast(buf, C.c_void_p), len(b), C.byref(n), None, None)

    assert info(data[:1000]) < 0                      # truncated program
    assert info(data[:len(data) // 2]) < 0            # truncated weight blob
    assert info(b"XRSW" + bytes(60)) < 0              # not a sentis container
    rng = np.random.default_rng(0)
    for _ in range(20):                               # random corruption of the program: an error code, never a crash
        d = bytearray(data)
        for p in rng.integers(8, 100000, 16):
            d[p] = int(rng.integers(0, 256))
        assert info(d) <= 0


# ---- launch planner invariants (host-only: tools/plan_dump.cu compiles the planners without a GPU) --------------------
@pytest.fixture(scope="module")
def plan_dump(tmp_path_factory):
    import shutil
    import subprocess
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    exe = str(tmp_path_factory.mktemp("plan") / "plan_dump")
    r = subprocess.run([nvcc, "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "--expt-relaxed-constexpr", "-o", exe,
                        os.path.join(ROOT, "tools", "plan_dump.cu"), "-lcuda"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    return exe


@pytest.mark.parametrize("batch,scale", [(1, "n"), (3, "n"), (64, "n"), (64, "s"), (5, "s"), (72, "n"), (256, "n"), (512, "n"),
                                         (96, "s"), (256, "s")])
def test_every_conv_plan_respects_the_hardware_limits(plan_dump, batch, scale):
    """Every convolution of the network gets a TMA plan (no thread-gather fallback at 640x640) that fits the SM:
    <= 227 KB shared memory, <= 512 TMEM columns, >= 2 pipeline stages, <= 4 sub-tiles, and covers all its work."""
    import subprocess
    out = subprocess.run([plan_dump, str(batch), scale], capture_output=True, text=True, check=True).stdout
    rows = [l for l in out.splitlines() if " smem " in l]
    # 100 layers - stem - 7 depthwise - 6 fused siblings (- proto.cv3 on the n scale: it runs inside proto.cv2's launch)
    assert len(rows) == (85 if scale == "n" else 86)
    for l in rows:
        tok = l.split()
        f = {tok[i]: tok[i + 1] for i in range(len(tok) - 1)}
        mode = tok[5]
        assert mode in ("halo_tma", "flat_tma", "s2_tma"), l
        assert int(f["smem"]) <= 232448 and int(f["tmem"]) <= 512 and int(f["S"]) >= 2, l
        assert 1 <= int(f["nsub"]) <= 4 and int(f["items"]) >= 1, l
        if mode != "flat_tma":
            assert int(f["R"]) >= 1, l
        else:
            assert int(f["nsub"]) in (1, 2, 4), l   # an item is whole TMA boxes of <= 256 rows (batch > 64 once picked 3)
    # N tiles: two for the s scale's wide 128-channel proto.cv2 at every batch; two / four for >= 128 / 256-channel layers whose
    # work items keep at most half / a quarter of the SMs busy (batch-1 streaming); one everywhere else at the bench batch
    nt = {l.split()[0]: int(l.split()[l.split().index("ntiles") + 1]) for l in rows}
    if batch == 64 and scale == "n":
        assert all(v == 1 for v in nt.values()), nt
    if batch == 64 and scale == "s":
        assert nt["proto.cv2"] == 2 and nt["proto.cv1"] == 1 and nt["b7"] == 2, nt      # (512-channel layers are two tiles of 256 anyway)
    if batch == 1 and scale == "n":
        assert nt["b8.cv2"] == 4 and nt["b9.cv2"] == 4 and nt["b6.cv1"] == 2 and nt["b2.cv2"] == 1 and nt["proto.cv2"] == 1, nt
    # pixel-pair operand rows (conv_tma.cuh plan_conv_s2_tma_impl): only where a K-block is the whole pixel -- the n scale's b1
    paired = [l.split()[0] for l in rows if "pixel-pair rows" in l]
    assert paired == (["b1"] if scale == "n" else []), paired


@pytest.mark.parametrize("scale,expect", [
    ("n", {"stem": 1, "conv": 79, "dw": 6, "sppf": 1, "up": 2, "attn": 1, "bneck": 3}),
    ("s", {"stem": 1, "conv": 84, "dw": 6, "sppf": 1, "up": 2, "attn": 1, "bneck": 1}),
])
def test_fusion_passes_produce_the_expected_launch_list(plan_dump, scale, expect):
    """model.cuh: fuse_siblings / fuse_bottlenecks / fuse_attention_pe / fuse_tail_1x1.  n scale: 100 layers -> 93 network
    launches (six sibling pairs, the Bottlenecks of b2 / b4 / n16, the C2PSA positional encoding inside the attention kernel,
    proto.cv3 inside proto.cv2's launch); the s scale has one supported Bottleneck (b2: 32-16-32).  Every fused Bottleneck
    keeps its residual and stays on the main stream."""
    import subprocess
    out = subprocess.run([plan_dump, "64", scale, "ops"], capture_output=True, text=True, check=True).stdout
    rows = [l.split() for l in out.splitlines() if l.startswith("op ")]
    kinds = {}
    for r in rows:
        kinds[r[1]] = kinds.get(r[1], 0) + 1
    assert kinds == expect
    for r in rows:
        if r[1] == "bneck":
            assert r[2].endswith(".m0.cv1") and r[r.index("res") + 1] == "1" and r[r.index("branch") + 1] == "0", r
    assert sum(1 for r in rows if r[1] == "conv" and "+" in r[2]) == 6
    attn = [r for r in rows if r[1] == "attn"][0]
    assert attn[2] == "b10.attn.pe"                         # the attention launch carries the depthwise layer's weights


# ---- fused Bottleneck kernel: weight fragment order (host-only) ------------------------------------------------------
@pytest.mark.parametrize("cin,cout,C,N,taps", [(16, 8, 16, 8, 9), (8, 16, 8, 16, 9), (32, 16, 32, 16, 9), (16, 32, 16, 32, 9),
                                               (32, 32, 32, 32, 1), (48, 64, 48, 64, 1), (12, 5, 16, 8, 9)])
def test_bottleneck_weight_fragments(cin, cout, C, N, taps):
    """pack_bneck_weights (bottleneck.cuh) against the mma.sync m16n8k16 B-fragment definition: word 0 of lane (g, t) of
    (k-step s, n-tile nt) holds W[16 s + 2 t][8 nt + g] (low half) and W[16 s + 2 t + 1][..]; word 1 the rows + 8;
    W[k][n] = w[n][c][tap] with k = tap * C + c, zero beyond the real channels and beyond K = taps * C."""
    import ctypes as C_
    from xr_image_segmentation_b200 import _lib
    lib = _lib.load_library(True)
    rng = np.random.default_rng(cin * 131 + cout)
    w = rng.standard_normal((cout, cin, taps)).astype(np.float32)
    K = taps * C
    KS, NT = (K + 15) // 16, N // 8
    out = np.zeros(KS * NT * 64, np.uint32)
    n = lib.xrseg_debug_pack_bneck(w.ctypes.data, cin, cout, C, N, taps, out.ctypes.data, out.size)
    assert n == out.size
    Wm = np.zeros((KS * 16, N), np.float16)
    for tap in range(taps):
        Wm[tap * C:tap * C + cin, :cout] = w[:, :, tap].T.astype(np.float16)
    halves = out.view(np.float16).reshape(KS, NT, 32, 2, 2)          # [s][nt][lane][word][low/high]
    for lane in range(32):
        g, t = lane >> 2, lane & 3
        for word in range(2):
            for h in range(2):
                k = 2 * t + 8 * word + h
                got = halves[:, :, lane, word, h]                     # [KS, NT]
                exp = Wm.reshape(KS, 16, NT, 8)[:, k, :, g]
                assert np.array_equal(got, exp), (lane, word, h)
