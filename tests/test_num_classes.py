"""Models trained on any number of classes (1..1024): topology, weight introspection, launch plans (CPU) and the decode /
end-to-end parity against the oracle (GPU, -m gpu).

The oracle's forward pass already takes a Spec carrying the class count; the helpers below build that Spec with the
Ultralytics rule cls_mid = max(ch[2], min(nc, 100)) and otherwise call oracle/ unchanged."""
import ctypes as C
import dataclasses
import subprocess

import numpy as np
import pytest
import torch

from oracle import preprocess as pre
from oracle import yolo11seg as Y
from oracle.sentis import write_sentis
from xr_image_segmentation_b200 import _lib, inference as I, weights as W

from test_abi import plan_dump  # noqa: F401  (fixture: tools/plan_dump.cu compiled for the host)
from test_gpu_parity import SCORE_THR, assert_batch_parity, gpu_frames, iou_cxcywh, oracle_frames, NAMES

NC_TABLES = [1, 3, 20, 80, 96, 120, 365, 601, 1024]
SIZES = [(80, 80), (40, 40), (20, 20)]


# ---- oracle side ---------------------------------------------------------------------------------------------------
def spec(scale, nc):
    s = Y.make_spec(scale)
    return dataclasses.replace(s, nc=nc, cls_mid=max(s.ch[2], min(nc, 100)))


def oracle_layer_table(scale, nc):
    rec = []
    with torch.no_grad():
        Y.forward_raw(torch.empty(1, 3, 640, 640, device="meta"), Y._ConvFeed(record=rec), spec(scale, nc))
    return rec


def oracle_random_weights(scale, seed, cls_bias, nc):
    """Y.random_weights' frozen recipe over the nc-class topology."""
    rng = np.random.default_rng(seed)
    out = []
    for l in oracle_layer_table(scale, nc):
        shp = Y.weight_shape(l)
        fan_in = (l["cin"] // l["groups"]) * l["k"] * l["k"] if not l["transposed"] else l["cin"]
        w = (rng.standard_normal(shp, dtype=np.float32) * np.float32(1.5 / np.sqrt(fan_in))).astype(np.float32)
        b = (rng.standard_normal(l["cout"], dtype=np.float32) * np.float32(0.2)).astype(np.float32)
        if l["name"] in Y.CLS_FINAL:
            b = (b * np.float32(0.25) + np.float32(cls_bias)).astype(np.float32)
        out.append((w, b))
    return out


@torch.no_grad()
def oracle_raw(weights, x, scale):
    nc = int(np.asarray(weights[[l["name"] for l in oracle_layer_table(scale, 80)].index("h3.cls.2")][1]).shape[0])
    feed = Y._ConvFeed(weights=weights)
    out = Y.forward_raw(x.float(), feed, spec(scale, nc))
    assert feed.i == len(weights)
    return out


def oracle_frames_of(raw):
    res = []
    for i in range(raw["box_logits"].shape[0]):
        protos = raw["protos"][i].reshape(raw["protos"].shape[1], -1).numpy()
        res.append(Y.postprocess_frame(raw["box_logits"][i].numpy(), raw["cls_logits"][i].numpy(), raw["coefs"][i].numpy(), protos,
                                       raw["sizes"]))
    return res


def info(lib, data):
    buf = C.create_string_buffer(bytes(data), len(data))
    s, n = C.c_int32(), C.c_int32()
    rc = lib.xrseg_weights_info(C.cast(buf, C.c_void_p), len(data), C.byref(s), C.byref(n))
    return rc, (chr(s.value) if rc == 0 else None), n.value


def quantize(a, rng):
    """Random uint8 tensor of a's shape with a per-tensor scale / zero point (weights_info reads shapes only)."""
    return rng.integers(0, 256, a, dtype=np.uint8), 0.01, 128


def sentis_of(layers, rng):
    convs = []
    for l in layers:
        wq, ws, wz = quantize(l.weight_shape, rng)
        bq, bs, bz = quantize((l.cout,), rng)
        convs.append((wq, ws, wz, bq, bs, bz, bool(l.transposed)))
    return write_sentis(convs, 0.43, 0.301)


# ---- CPU -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("scale", ["n", "s"])
@pytest.mark.parametrize("nc", NC_TABLES)
def test_layer_table_matches_oracle(lib, scale, nc):
    a, b = W.layer_table(scale, nc), oracle_layer_table(scale, nc)
    assert len(a) == len(b) == 100
    for x, y in zip(a, b):
        assert (x.name, x.cin, x.cout, x.k, x.stride, x.groups, x.act, x.transposed, x.h_in, x.w_in) == \
               (y["name"], y["cin"], y["cout"], y["k"], y["s"], y["groups"], int(y["act"]), int(y["transposed"]), y["h_in"], y["w_in"])
    cls = {x.name: x for x in a}
    assert cls["h3.cls.2"].cout == cls["h5.cls.2"].cout == nc
    assert cls["h4.cls.0pw"].cout == max(64 if scale == "n" else 128, min(nc, 100))
    if nc == 80:
        assert a == W.layer_table(scale)
        assert [tuple(sorted(d.items())) for d in b] == [tuple(sorted(d.items())) for d in Y.layer_table(scale)]
    assert lib.xrseg_layer_count_nc(ord(scale), 0) < 0 and lib.xrseg_layer_count_nc(ord(scale), 1025) < 0


@pytest.mark.parametrize("scale,nc", [("n", 3), ("n", 365), ("s", 20), ("s", 1024)])
def test_random_generator_matches_oracle(lib, scale, nc):
    _, ws = W.random_weights(scale, seed=4, cls_bias=-6.0, nc=nc)
    ow = oracle_random_weights(scale, 4, -6.0, nc)
    for (w, b), (w2, b2) in zip(ws, ow):
        assert np.array_equal(w, w2) and np.array_equal(b, b2)
    with pytest.raises(ValueError):
        W.random_weights(scale, seed=4, nc=nc)                     # INIT_CLS_BIAS is tuned for 80 classes only


def test_weights_info_on_packs_and_sentis_assets(lib, golden, golden_sentis):
    assert info(lib, golden["model"].pack)[0:3] == (0, "n", 80)
    assert info(lib, golden_sentis) == (0, "n", 80)
    rng = np.random.default_rng(0)
    for scale, nc in (("n", 1), ("s", 20), ("s", 80), ("n", 1024)):
        layers = W.layer_table(scale, nc)
        assert info(lib, sentis_of(layers, rng)) == (0, scale, nc)
        _, ws = W.random_weights(scale, 1, cls_bias=-5.0, nc=nc)
        pack = W.write_pack(scale, layers, ws)
        assert info(lib, pack) == (0, scale, nc)
        m = I.ModelLoader.Load(pack)
        assert (m.scale, m.nc) == (scale, nc)
    m = I.ModelLoader.Load(golden_sentis)
    assert (m.scale, m.nc) == ("n", 80)
    m = I.ModelLoader.Load(sentis_of(W.layer_table("s", 365), rng))        # an s-scale asset is no longer taken for 'n'
    assert (m.scale, m.nc) == ("s", 365)


def test_weights_info_rejects_bad_class_convolutions(lib):
    rng = np.random.default_rng(1)
    base = W.layer_table("n", 20)

    def with_cls(couts):
        ls = [dataclasses.replace(l, cout=couts[W.CLS_FINAL.index(l.name)]) if l.name in W.CLS_FINAL else l for l in base]
        return ls, [(np.zeros(l.weight_shape, np.float32), np.zeros(l.cout, np.float32)) for l in ls]

    for couts in ((20, 21, 20), (0, 0, 0), (1025, 1025, 1025)):
        ls, ws = with_cls(couts)
        assert info(lib, W.write_pack("n", ls, ws))[0] == _lib.ERR_WEIGHTS, couts
        assert info(lib, sentis_of(ls, rng))[0] == _lib.ERR_WEIGHTS, couts
    assert "supported are 1..1024" in lib.xrseg_last_error(None).decode()
    ls, ws = with_cls((20, 21, 20))
    info(lib, W.write_pack("n", ls, ws))
    assert "disagree" in lib.xrseg_last_error(None).decode()
    with pytest.raises(I.XrsegError):
        I.ModelLoader.Load(W.write_pack("n", *with_cls((1025, 1025, 1025))))


@pytest.mark.parametrize("scale", ["n", "s"])
@pytest.mark.parametrize("batch", [1, 64])
@pytest.mark.parametrize("nc", [1, 3, 365, 601, 1024])
def test_every_conv_plan_respects_the_hardware_limits(plan_dump, scale, batch, nc):
    """The checks of test_abi's planner test for other class counts: every convolution, the class convolutions included,
    gets a TMA plan within the SM's limits; a class convolution wider than 256 channels runs as 2 / 4 N tiles."""
    out = subprocess.run([plan_dump, str(batch), scale, str(nc)], capture_output=True, text=True, check=True).stdout
    rows = [l for l in out.splitlines() if " smem " in l]
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
            assert int(f["nsub"]) in (1, 2, 4), l
    cls = [l.split() for l in rows if ".cls.2" in l.split()[0]]
    assert len(cls) == 3
    for t in cls:
        assert t[5] == "flat_tma" and t[2].endswith(f"->{nc}"), t
        nt = int(t[t.index("ntiles") + 1])
        assert nt in ((1, 2, 4) if nc <= 256 else (2, 4)), t


# ---- GPU -----------------------------------------------------------------------------------------------------------
def tuned_network(scale, nc, frames, seed=1, target=0.015):
    """Random-init network of nc classes whose class bias is chosen on the oracle so that `target` of the anchors of these
    frames pass the 0.301 score filter: the class logits move one for one with the bias."""
    x = torch.from_numpy(np.concatenate([pre.to_tensor(f) for f in frames]))
    _, ws0 = W.random_weights(scale, seed, cls_bias=0.0, nc=nc)
    m = oracle_raw(ws0, x, scale)["cls_logits"].numpy().max(axis=2).ravel()
    bias = float(np.log(SCORE_THR / (1 - SCORE_THR)) - np.quantile(m, 1 - target))
    layers, ws = W.random_weights(scale, seed, cls_bias=bias, nc=nc)
    raw = oracle_raw(ws, x, scale)
    return layers, ws, raw, x


def own_logit_frames(r, n_frames, nc):
    """The oracle's post-processing on the GPU network's own head tensors."""
    cat = lambda nm, c: np.concatenate([r.fetch(f"{nm}.{i}").reshape(n_frames, c, -1) for i in range(3)], axis=2).transpose(0, 2, 1)
    bl, cl, cf = cat("box_logits", 64), cat("cls_logits", nc), cat("coefs", 32)
    pr = r.fetch("protos").reshape(n_frames, 32, -1)
    return cl, [Y.postprocess_frame(np.ascontiguousarray(bl[f]), np.ascontiguousarray(cl[f]), np.ascontiguousarray(cf[f]), pr[f], SIZES)
                for f in range(n_frames)]


@pytest.mark.gpu
@pytest.mark.parametrize("scale,nc", [("n", 1), ("n", 3), ("n", 20), ("n", 365), ("n", 1024), ("s", 1), ("s", 365)])
def test_random_init_parity_vs_oracle(lib, scale, nc):
    frames = np.random.default_rng(nc).integers(0, 256, (2, 640, 640, 3), dtype=np.uint8)
    layers, ws, raw, x = tuned_network(scale, nc, frames)
    ref = oracle_frames_of(raw)
    passing = float(np.mean(np.concatenate([r["all_scores"] for r in ref]) > SCORE_THR))
    assert 0.005 <= passing <= 0.03, passing
    r = I.Runner(I.Model(W.write_pack(scale, layers, ws), scale, nc), max_batch=2, max_det=1000, max_candidates=8400, debug=True)
    assert r.num_classes == nc
    r.schedule(frames)
    r.wait()
    cl, hyb = own_logit_frames(r, 2, nc)
    rl = raw["cls_logits"].numpy()
    assert np.abs(cl - rl).mean() <= 0.02 * max(1.0, float(np.abs(rl).mean()))
    got = gpu_frames(r, 2)
    for f in range(2):                                               # decode / NMS exact on the network's own logits
        assert got[f]["keep"].tolist() == hyb[f]["keep"].tolist(), f
        assert got[f]["labels"].tolist() == hyb[f]["labels"].tolist()
        assert (got[f]["labels"] < nc).all()
    pairs, unpaired = assert_batch_parity(got, oracle_frames(ref), min_pairs=5, max_unpaired=0.3, max_mask_diff=2e-3)
    print(f"{scale} nc={nc}: {passing:.2%} of anchors pass, {pairs} pairs, {unpaired} borderline")
    r.close()


def widened_golden(golden, nc):
    """The golden network's uint8 tensors widened to nc classes: new class-branch channels dequantize to exactly 0 (q = zp),
    new class rows are copies of classes 0 .. nc - 81.  -> [(w Tensor8, b Tensor8, transposed)] in canonical order."""
    pack = golden["model"].pack
    _, _, n, _, payload, _ = W.HEADER.unpack_from(pack, 0)
    mid = max(64, min(nc, 100))
    out = []
    for i in range(n):
        (name, cout, cin_g, k, _, _, _, tr, dtype, ws, wz, bs, bz, w_off, b_off) = W.RECORD.unpack_from(pack, W.HEADER.size + i * W.RECORD.size)
        name = name.split(b"\0")[0].decode()
        shape = (cin_g, cout, k, k) if tr else (cout, cin_g, k, k)
        wq = np.frombuffer(pack, np.uint8, int(np.prod(shape)), payload + w_off).reshape(shape)
        bq = np.frombuffer(pack, np.uint8, cout, payload + b_off)
        assert dtype == 3 and 0 <= wz <= 255 and 0 <= bz <= 255

        def pad(a, axis, size, zp):
            w = [(0, 0)] * a.ndim
            w[axis] = (0, size - a.shape[axis])
            return np.pad(a, w, constant_values=zp)
        if name.endswith((".cls.0pw", ".cls.1dw", ".cls.1pw")):
            wq, bq = pad(wq, 0, mid, wz), pad(bq, 0, mid, bz)
            if name.endswith(".cls.1pw"):
                wq = pad(wq, 1, mid, wz)
        elif name.endswith(".cls.2"):
            wq = pad(wq, 1, mid, wz)
            wq, bq = np.concatenate([wq, wq[:nc - 80]]), np.concatenate([bq, bq[:nc - 80]])
        out.append((W.Tensor8(np.ascontiguousarray(wq), ws, wz), W.Tensor8(np.ascontiguousarray(bq), bs, bz), bool(tr)))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("nc", [96, 120])
def test_trained_weights_widened_to_more_classes(golden, nc):
    """The golden network with 16 / 40 duplicated classes: the copies tie exactly with their originals and the first-max rule
    keeps every label below 80, so the six reference frames give the golden outputs and the labels of the 80-class runner."""
    t = widened_golden(golden, nc)
    model = I.Model(W.write_pack("n", W.layer_table("n", nc), [(w, b) for w, b, _ in t]), "n", nc)
    base, wide = I.Runner(golden["model"]), I.Runner(model)           # the sample frames differ in size: one at a time
    assert wide.num_classes == nc
    res = [[], []]
    for name in NAMES:
        for k, r in enumerate((base, wide)):
            r.schedule(golden["inputs"][name][None])
            r.wait()
            res[k] += gpu_frames(r, 1)
    exp = golden["expected"]
    for f, name in enumerate(NAMES):
        g, b0 = res[1][f], res[0][f]
        assert g["keep"].tolist() == exp[f"{name}.keep"].tolist() == b0["keep"].tolist()
        assert g["labels"].tolist() == exp[f"{name}.labels"].tolist() == b0["labels"].tolist()
        assert np.abs(g["boxes"] - exp[f"{name}.boxes"]).max(initial=0) <= 0.5
        assert len(g["boxes"]) == 0 or iou_cxcywh(g["boxes"], exp[f"{name}.boxes"]).min() >= 0.99
        bits = np.packbits(g["masks"], axis=-1)
        assert np.mean(np.unpackbits(bits ^ exp[f"{name}.mask_bits"])) <= 1e-3
    base.close()
    wide.close()


@pytest.mark.gpu
@pytest.mark.parametrize("nc", [1, 3, 365])
def test_post_kernels_bit_exact_on_oracle_tensors(lib, nc):
    """debug_post with nc-class logits (planted objects among low logits): keep indices and labels exactly the oracle's."""
    _, ws = W.random_weights("n", 1, cls_bias=-5.0, nc=nc)
    r = I.Runner(I.Model(W.write_pack("n", W.layer_table("n", nc), ws), "n", nc), max_batch=2, max_det=1000, max_candidates=8400,
                 debug=True)
    rng = np.random.default_rng(nc)
    A = 8400
    box = rng.standard_normal((2, A, 64)).astype(np.float32)
    box.reshape(2, A, 4, 16)[..., 1] += 6.0
    cls = (rng.standard_normal((2, A, nc)) - 6).astype(np.float32)
    for f in range(2):
        for a in rng.choice(A, 150, replace=False):
            cls[f, a, rng.integers(0, nc)] = 1.0 + rng.standard_normal()
    if nc > 1:
        cls[0, :40, 1] = cls[0, :40, 0] = 2.5                    # exact ties: the first index wins
    coefs = rng.standard_normal((2, A, 32)).astype(np.float32)
    protos = rng.standard_normal((2, 32, 25600)).astype(np.float32)
    r.debug_post(box, cls, coefs, protos)
    r.wait()
    counts, (keep, _), labels = r.counts(), r.keep_indices(), r.readback(1)
    off = 0
    for f in range(2):
        ref = Y.postprocess_frame(box[f], cls[f], coefs[f], protos[f], SIZES)
        assert len(ref["keep"]) >= 20
        assert keep[off:off + counts[f]].tolist() == ref["keep"].tolist()
        assert labels[off:off + counts[f]].tolist() == ref["labels"].tolist()
        off += counts[f]
    with pytest.raises(ValueError):
        r.debug_post(box, cls[..., :1] if nc > 1 else np.zeros((2, A, 2), np.float32), coefs, protos)
    r.close()


@pytest.mark.gpu
def test_padding_channels_never_count(lib):
    """nc = 1: the class tensor's 15 padding channels hold logit 0 (probability 0.5 > 0.301).  With a class bias of -20 no
    anchor may pass -- and none may reach the candidate cap of 2048 either."""
    layers, ws = W.random_weights("n", 1, cls_bias=-20.0, nc=1)
    r = I.Runner(I.Model(W.write_pack("n", layers, ws), "n", 1), max_batch=2)
    r.schedule(np.random.default_rng(0).integers(0, 256, (2, 640, 640, 3), dtype=np.uint8))
    r.wait()
    assert r.counts().tolist() == [0, 0] and r.overflow() == 0
    r.close()


@pytest.mark.gpu
def test_custom_class_sentis_equals_pack_and_num_classes_config(golden):
    t = widened_golden(golden, 96)
    pack = W.write_pack("n", W.layer_table("n", 96), [(w, b) for w, b, _ in t])
    sentis = write_sentis([(w.q, w.scale, w.zp, b.q, b.scale, b.zp, tr) for w, b, tr in t], 0.43, 0.301)
    outs = []
    for data in (pack, sentis):
        m = I.ModelLoader.Load(data)
        assert (m.scale, m.nc) == ("n", 96)
        r = I.Runner(m)                                              # num_classes = 0: taken from the weights
        assert r.num_classes == 96
        outs.append([])
        for name in NAMES[:3]:
            r.schedule(golden["inputs"][name][None])
            r.wait()
            outs[-1] += [r.readback(i) for i in range(4)]
        r.close()
    for a, b in zip(*outs):
        assert np.array_equal(a, b)
    assert I.Runner(I.ModelLoader.Load(sentis), num_classes=96).num_classes == 96
    for wrong in (80, 95):
        with pytest.raises(I.XrsegError) as e:
            I.Runner(I.ModelLoader.Load(sentis), num_classes=wrong)
        assert e.value.code == _lib.ERR_WEIGHTS and "96" in str(e.value) and str(wrong) in str(e.value)


@pytest.mark.gpu
def test_365_classes_batch_72_equals_batch_8(lib):
    frames = np.random.default_rng(0).integers(0, 256, (8, 640, 640, 3), dtype=np.uint8)
    layers, ws = W.random_weights("n", 1, cls_bias=-5.0, nc=365)
    model = I.Model(W.write_pack("n", layers, ws), "n", 365)
    out = {}
    for b in (8, 72):
        r = I.Runner(model, max_batch=b, debug=True)
        r.schedule(np.ascontiguousarray(np.tile(frames, (b // 8, 1, 1, 1))))
        r.wait(strict=False)
        cl = np.concatenate([r.fetch(f"cls_logits.{i}").reshape(b, 365, -1) for i in range(3)], axis=2)
        out[b] = (r.counts().copy(), cl[-8:])
        r.close()
    assert np.abs(out[72][1] - out[8][1]).max() <= 0.1 and np.abs(out[72][1] - out[8][1]).mean() <= 5e-3
    assert np.abs(out[72][0][-8:].astype(int) - out[8][0].astype(int)).max() <= 3
    assert np.array_equal(out[72][0][:8], out[72][0][-8:])
    w = I.Worker(model, I.BackendType.GPUCompute)
    w.Schedule(I.TextureConverter.ToTensor(frames[0], 640, 640, 3))
    shapes = [tuple(w.PeekOutput(i).shape) for i in range(4)]
    k = shapes[0][0]
    assert shapes == [(k, 4), (k,), (k, 32), (k, 160, 160)]
    w.Dispose()
