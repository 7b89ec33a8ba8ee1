"""CPU tests pinning the ORACLE: (1) against the committed golden vectors, which were produced by the interpreter
over the reference asset's own 499-chain graph (tests/golden/make_golden.py); (2) its .sentis reader against the golden
weight pack; (3) properties / hand-computed cases of the restated C#."""
import numpy as np
import pytest
import torch

from oracle import postprocess as pp
from oracle import preprocess as pre
from oracle import yolo11seg as Y

NAMES = ["coco139", "coco632", "coco2006", "coco4495", "coco7108", "bus"]   # all six sample frames of the reference


@pytest.fixture(scope="module")
def oracle_runs(golden, golden_weights):
    out = {}
    for name in NAMES:
        x = torch.from_numpy(pre.to_tensor(golden["inputs"][name]))
        res, raw = Y.run_model(golden_weights, x, "n")
        out[name] = (res[0], raw, x)
    return out


@pytest.mark.parametrize("name", NAMES)
def test_generic_oracle_matches_golden(golden, oracle_runs, name):
    exp = golden["expected"]
    r, raw, x = oracle_runs[name]
    assert r["keep"].tolist() == exp[f"{name}.keep"].tolist()          # NMS keep indices: exact
    assert r["labels"].tolist() == exp[f"{name}.labels"].tolist()
    np.testing.assert_allclose(r["boxes"], exp[f"{name}.boxes"], atol=1e-3)
    np.testing.assert_allclose(r["coefs"], exp[f"{name}.coefs"], atol=1e-4)
    bits = np.packbits(r["masks"] > np.float32(0.5), axis=-1)
    assert np.mean(np.unpackbits(bits ^ exp[f"{name}.mask_bits"])) <= 1e-4
    np.testing.assert_allclose(r["masks"][:, ::8, ::8], exp[f"{name}.mask_prob_sample"], atol=1e-4)
    head = torch.cat([raw["box_logits"][0], raw["cls_logits"][0]], 1).numpy().T     # [144,8400]
    np.testing.assert_allclose(head[:, ::25], exp[f"{name}.head_sample"], atol=2e-4)
    np.testing.assert_allclose(r["protos"][:, ::64], exp[f"{name}.proto_sample"], atol=2e-4)
    np.testing.assert_allclose(x[0, :, ::16, ::16].numpy(), exp[f"{name}.input_sample"], atol=0)


@pytest.mark.parametrize("name", NAMES)
def test_csharp_postprocess_matches_golden(golden, oracle_runs, name):
    exp = golden["expected"]
    boxes, labels = exp[f"{name}.boxes"], exp[f"{name}.labels"]
    pb, _ = pp.parse_boxes(boxes, labels, 1920.0, 1080.0)
    db, _ = pp.draw_boxes(boxes, labels, 1920.0, 1080.0)
    assert np.array_equal(pb, exp[f"{name}.parse_boxes"])
    assert np.array_equal(db, exp[f"{name}.draw_boxes"])
    masks = oracle_runs[name][0]["masks"]
    dm = np.stack([pp.draw_mask_bits(masks[i], db[i], 1920, 1080) for i in range(len(db))])
    assert np.mean(np.unpackbits(np.packbits(dm.astype(bool), axis=-1) ^ exp[f"{name}.draw_mask_bits"])) <= 1e-4


def test_xrsw_pack_roundtrip_matches_reference_dequant(golden_sentis, golden_weights):
    """The pack keeps the asset's uint8 tensors: put back into a .sentis container, the oracle's own dequantization of
    them gives the pack's weights."""
    from oracle.sentis import load_sentis
    ref = Y.weights_from_sentis(load_sentis(golden_sentis))
    assert len(ref) == len(golden_weights) == 100
    for (w0, b0), (w1, b1) in zip(ref, golden_weights):
        assert np.array_equal(w0, w1) and np.array_equal(b0, b1)
    assert sum(w.size + b.size for w, b in golden_weights) == 2868648


# ---- NMS -------------------------------------------------------------------------------------------------------
def _rand_boxes(rng, n, size=640.0):
    c = rng.uniform(0, size, (n, 2)).astype(np.float32)
    wh = rng.uniform(4, 200, (n, 2)).astype(np.float32)
    return np.concatenate([c - wh / 2, c + wh / 2], 1).astype(np.float32)


def test_nms_properties():
    rng = np.random.default_rng(0)
    for trial in range(20):
        n = int(rng.integers(1, 400))
        boxes = _rand_boxes(rng, n)
        scores = rng.uniform(0, 1, n).astype(np.float32)
        if trial % 3 == 0:
            scores = np.round(scores, 1)           # many ties
        keep = pp.nms_onnx(boxes, scores, 0.43, 0.301)
        assert np.all(scores[keep] > np.float32(0.301))
        assert np.all(np.diff(scores[keep]) <= 0)                        # score-descending
        ties = np.diff(scores[keep]) == 0
        assert np.all(np.diff(keep)[ties] > 0)                           # index ascending on ties
        for a in range(len(keep)):                                       # kept boxes do not suppress each other
            if a:
                assert not np.any(pp.iou_f32(boxes[keep[a]], boxes[keep[:a]]) > np.float32(0.43))
        sub = pp.nms_onnx(boxes[keep], scores[keep], 0.43, 0.301)        # idempotence
        assert sub.tolist() == list(range(len(keep)))
        dropped = np.setdiff1d(np.nonzero(scores > np.float32(0.301))[0], keep)
        for d in dropped:                                                # every dropped candidate has a reason
            better = keep[(scores[keep] > scores[d]) | ((scores[keep] == scores[d]) & (keep < d))]
            assert np.any(pp.iou_f32(boxes[d], boxes[better]) > np.float32(0.43))


def test_nms_edge_cases():
    assert pp.nms_onnx(np.zeros((0, 4), np.float32), np.zeros(0, np.float32), 0.43, 0.301).tolist() == []
    b = np.array([[0, 0, 10, 10]] * 5, np.float32)
    s = np.array([0.9, 0.9, 0.9, 0.2, 0.95], np.float32)
    assert pp.nms_onnx(b, s, 0.43, 0.301).tolist() == [4]               # identical boxes: only the best survives
    assert pp.nms_onnx(b, np.full(5, 0.301, np.float32), 0.43, 0.301).tolist() == []   # strict score threshold
    z = np.array([[5, 5, 5, 5], [5, 5, 5, 5]], np.float32)               # zero-area boxes: IoU = 0/0 = nan, not > thr
    assert pp.nms_onnx(z, np.array([0.9, 0.8], np.float32), 0.43, 0.301).tolist() == [0, 1]
    far = np.array([[0, 0, 10, 10], [100, 100, 110, 110]], np.float32)
    assert pp.nms_onnx(far, np.array([0.5, 0.6], np.float32), 0.43, 0.301).tolist() == [1, 0]
    assert pp.nms_onnx(far, np.array([0.5, 0.6], np.float32), 0.43, 0.301, max_out=1).tolist() == [1]


def test_decode_hand_case():
    # uniform logits -> every side's expectation is 7.5 bins: box centred on the anchor, 15 bins wide
    ax, ay, st = pp.make_anchors()
    assert ax.shape == (8400,) and ax[0] == 0.5 and ay[80] == 1.5 and st[6400] == 16 and st[8399] == 32
    boxes = pp.dfl_decode(np.zeros((8400, 64), np.float32), ax, ay, st)
    np.testing.assert_allclose(boxes[0], [4.0, 4.0, 120.0, 120.0], rtol=1e-6)
    np.testing.assert_allclose(boxes[8399], [19.5 * 32, 19.5 * 32, 480.0, 480.0], rtol=1e-6)
    logits = np.full((1, 80), -5.0, np.float32)
    logits[0, 17] = 2.0
    logits[0, 40] = 2.0                                                   # tie: first maximum wins (chain 471)
    s, l = pp.class_scores(logits)
    assert l[0] == 17 and abs(s[0] - 1 / (1 + np.exp(-2.0))) < 1e-6


def test_csharp_boxes_hand_case():
    boxes = np.array([[320, 320, 64, 32], [0, 640, 10, 10]], np.float32)
    pb, _ = pp.parse_boxes(boxes, np.array([0, 1]), 1280.0, 640.0)
    assert pb.tolist() == [[0.0, 0.0, 128.0, 32.0], [-640.0, -320.0, 20.0, 10.0]]        # centred, Y-up
    db, _ = pp.draw_boxes(boxes, np.array([0, 1]), 1280.0, 640.0)
    assert db.tolist() == [[0.0, 0.0, 128.0, 32.0], [-640.0, 320.0, 20.0, 10.0]]         # centred, Y-down
    many = np.tile(boxes[:1], (300, 1))
    assert len(pp.parse_boxes(many, np.zeros(300, np.int32), 640, 640)[0]) == 50          # IEE:534
    assert len(pp.draw_boxes(many, np.zeros(300, np.int32), 640, 640)[0]) == 200          # IEB:50
    labels = pp.load_labels("person\r\ntraffic light\n\n")
    assert labels == ["person", "traffic light"]
    assert pp.get_class_name(labels, 1) == "traffic_light" and pp.get_class_name(labels, 7) == "unknown"


def test_pixel_in_bounding_box_hand_case():
    # DrawBoxes box of a 64x32 box centred at (320,320) with image == 640: mask centre (80, 80), half sizes (8, 4)
    box = (0.0, 0.0, 64.0, 32.0)
    xs, ys = np.meshgrid(np.arange(160), np.arange(160))
    inside = pp.pixel_in_bounding_box(box, xs, ys, 640, 640)
    assert inside.sum() == 17 * 9 and inside[80, 80] and inside[76, 72] and not inside[75, 72] and inside[84, 88]
    m = np.ones((160, 160), np.float32)
    out = pp.draw_mask_bits(m, box, 640, 640)
    assert out.sum() == 17 * 9 and out[80, 80] == 1
    m[:] = 0.5                                                            # strict > threshold (IEM:105)
    assert pp.draw_mask_bits(m, box, 640, 640).sum() == 0


def test_preprocess_identity_and_letterbox():
    rng = np.random.default_rng(1)
    img = rng.integers(0, 256, (640, 640, 3), dtype=np.uint8)
    t = pre.to_tensor(img)
    assert t.shape == (1, 3, 640, 640)
    assert np.array_equal(t[0].transpose(1, 2, 0), (img.astype(np.float32) / np.float32(255)))
    rgba = np.concatenate([img, np.full((640, 640, 1), 9, np.uint8)], -1)
    assert np.array_equal(pre.to_tensor(rgba), t)                         # alpha dropped
    lb = pre.letterbox(rng.integers(0, 256, (960, 1280, 3), dtype=np.uint8))
    assert np.allclose(lb[0, :, :80, :], 114 / 255) and np.allclose(lb[0, :, 560:, :], 114 / 255)
    assert not np.allclose(lb[0, :, 80:560, :], 114 / 255)


def test_mask_upsample_constant():
    L = np.full((160, 160), 1.0, np.float32)
    up = pp.upsample_mask_640(L, np.array([320, 320, 100, 50], np.float32))
    assert up.sum() == 100 * 50 and up[320, 320] == 1 and up[294, 320] == 0 and up[295, 320] == 1
