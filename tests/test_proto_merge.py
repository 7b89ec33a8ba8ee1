"""proto.up (ConvTranspose 2x2 / stride 2) merged into proto.cv2 (3x3) as four parity convolutions on the 80x80 map
(model.cuh fuse_up_conv, conv_tma.cuh merge_upconv_weights / plan_conv_upmerge_tma).

Host part: tools/merge_check.cu evaluates the merged weights and border biases against cv2(convT(x)) in fp64 on random
80x80 maps, every border class included.  GPU part: the merged launch against the three-launch path (XRSEG_FUSE_UP=0) on
the same frames, the golden frames against the oracle, and batch 1 / 72 against batch 8."""
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

from oracle import preprocess as pre
from oracle import yolo11seg as Y
from xr_image_segmentation_b200 import inference as I, weights as W

from test_abi import plan_dump  # noqa: F401  (fixture: tools/plan_dump.cu compiled for the host)

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
GOLDEN_PACK = os.path.join(ROOT, "tests", "golden", "yolo11n_seg.xrsw")


@pytest.fixture(scope="module")
def merge_check(tmp_path_factory):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    exe = str(tmp_path_factory.mktemp("merge") / "merge_check")
    r = subprocess.run([nvcc, "-std=c++17", "-O2", "-gencode", "arch=compute_100a,code=sm_100a", "--expt-relaxed-constexpr", "-o", exe,
                        os.path.join(ROOT, "tools", "merge_check.cu"), "-lcuda"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    return exe


def _run_check(exe, pack_path, seed):
    out = subprocess.run([exe, pack_path, str(seed)], capture_output=True, text=True, check=True).stdout.split()
    return {out[i]: float(out[i + 1]) for i in range(0, len(out) - 1, 2)}


@pytest.mark.parametrize("which,seed", [("random", 0), ("random", 7), ("golden", 3)])
def test_merged_weights_and_border_biases_are_exact(merge_check, tmp_path, which, seed):
    """fp64 merge against the fp64 two-layer reference: <= 1e-9 of the largest output everywhere and in each of the nine
    border classes (interior, four edges, four corners of the 160x160 map).  Prints max |Wm| and the error of rounding Wm to
    fp16 once, for the random-init network and the golden pack."""
    if which == "random":
        layers, ws = W.random_weights("n", seed=seed + 1)
        path = str(tmp_path / "rand.xrsw")
        with open(path, "wb") as f:
            f.write(W.write_pack("n", layers, ws))
    else:
        path = GOLDEN_PACK
    r = _run_check(merge_check, path, seed)
    print(f"{which}: max |Wm| = {r['wm_max']:.4g}, fp16 rounding of Wm = {r['wm_f16_rel_err']:.3e} of max |Wm|, "
          f"merge error = {r['rel_err']:.3e} of max |out| = {r['out_max']:.4g}")
    assert r["rel_err"] <= 1e-9, r
    for c in range(9):
        assert r[f"n{c}"] >= 1 and r[f"cls{c}"] <= 1e-9, (c, r)
    assert [r[f"n{c}"] for c in range(9)] == [158 * 158, 158, 158, 158, 1, 1, 158, 1, 1]
    assert r["wm_f16_rel_err"] <= 2 ** -11                        # one rounding: half an fp16 ulp of the largest weight


@pytest.mark.parametrize("batch", [1, 3, 64, 72, 512])
def test_merged_plan_respects_the_hardware_limits(plan_dump, batch):
    """The runner's n-scale launch list (plan_dump "up"): proto.up has no launch of its own, every convolution still gets a TMA
    plan within the SM's limits, and the merged launch is a halo plan of three 80x80 rows x two sub-tiles x two column
    parities (4 virtual sub-tiles of 64 columns, 512 TMEM columns, two stages), with room left for the tail's 4 KB of W2."""
    out = subprocess.run([plan_dump, str(batch), "n", "up"], capture_output=True, text=True, check=True).stdout
    rows = [l for l in out.splitlines() if " smem " in l]
    assert len(rows) == 84 and not any(l.split()[0] == "proto.up" for l in rows)
    for l in rows:
        tok = l.split()
        f = {tok[i]: tok[i + 1] for i in range(len(tok) - 1)}
        assert tok[5] in ("halo_tma", "flat_tma", "s2_tma"), l
        assert int(f["smem"]) <= 232448 and int(f["tmem"]) <= 512 and int(f["S"]) >= 2 and 1 <= int(f["nsub"]) <= 4, l
    m = [l for l in rows if "merged proto.up" in l]
    assert len(m) == 1 and m[0].split()[0] == "proto.cv2"
    tok = m[0].split()
    f = {tok[i]: tok[i + 1] for i in range(len(tok) - 1)}
    assert tok[5] == "halo_tma" and f["R"] == "3" and f["nsub"] == "4" and f["tmem"] == "512" and f["cb"] == "64"
    assert f["ntiles"] == "1" and f["bres"] == "1"
    assert int(f["smem"]) + 1024 + 32 * 64 * 2 <= 232448
    ops = [l.split() for l in subprocess.run([plan_dump, str(batch), "n", "ops", "up"], capture_output=True, text=True,
                                              check=True).stdout.splitlines() if l.startswith("op ")]
    assert sum(1 for r in ops if r[1] == "conv") == 78 and not any(r[2] == "proto.up" for r in ops)


# ---- GPU ---------------------------------------------------------------------------------------------------------------
def _run(model, frames, **kw):
    r = I.Runner(model, max_batch=len(frames), debug=True, **kw)
    r.schedule(np.ascontiguousarray(frames))
    r.wait()
    keep, _ = r.keep_indices()
    out = dict(counts=r.counts().copy(), keep=keep.copy(), boxes=r.readback(0).copy(), probs=r.readback(3).copy(),
               protos=r.fetch("protos").copy())
    r.close()
    return out


@pytest.mark.gpu
def test_merged_protos_match_the_three_launch_path(golden, monkeypatch):
    """Same frames, same weights: prototypes of the merged launch within fp16 tolerance of proto.up -> proto.cv2 -> proto.cv3
    as separate launches; detections identical (the prototypes do not feed them), masks within the fp16 noise."""
    im = golden["inputs"]["coco139"]
    frames = np.stack([im, im[:, ::-1], im[::-1]])
    merged = _run(golden["model"], frames)
    monkeypatch.setenv("XRSEG_FUSE_UP", "0")
    ref = _run(golden["model"], frames)
    d = np.abs(merged["protos"] - ref["protos"])
    print(f"protos: max |diff| {d.max():.3e}, mean {d.mean():.3e}, max |ref| {np.abs(ref['protos']).max():.3g}")
    assert d.max() <= 5e-2 and d.mean() <= 2e-3, (float(d.max()), float(d.mean()))
    assert merged["counts"].tolist() == ref["counts"].tolist() and merged["keep"].tolist() == ref["keep"].tolist()
    assert np.array_equal(merged["boxes"], ref["boxes"])
    bits = lambda p: np.packbits(p > np.float32(0.5), axis=-1)
    assert np.mean(np.unpackbits(bits(merged["probs"]) ^ bits(ref["probs"]))) <= 1e-3


@pytest.mark.gpu
def test_golden_frames_vs_oracle_with_the_merged_launch(golden, golden_weights):
    """DESIGN.md section 2 rules on every golden frame: same detections and labels, boxes within 0.5 px, <= 0.1 % of mask
    pixels flipped against the committed expectations, prototypes within 5e-2 of the oracle run live."""
    exp = golden["expected"]
    for name in sorted(golden["inputs"]):
        img = golden["inputs"][name]
        r = I.Runner(golden["model"], max_batch=1, debug=True)
        r.schedule(img[None])
        r.wait()
        keep, _ = r.keep_indices()
        boxes, labels, probs = r.readback(0), r.readback(1), r.readback(3)
        assert keep.tolist() == exp[f"{name}.keep"].tolist(), name
        assert labels.tolist() == exp[f"{name}.labels"].tolist(), name
        assert np.abs(boxes - exp[f"{name}.boxes"]).max() <= 0.5, name
        bits = np.packbits(probs > np.float32(0.5), axis=-1)
        assert np.mean(np.unpackbits(bits ^ exp[f"{name}.mask_bits"])) <= 1e-3, name
        res, _ = Y.run_model(golden_weights, torch.from_numpy(pre.to_tensor(img)), "n")
        assert np.abs(r.fetch("protos").reshape(32, -1) - res[0]["protos"]).max() <= 5e-2, name
        r.close()


@pytest.mark.gpu
def test_batch_1_and_72_match_batch_8(lib):
    """The merged plan changes with the batch (grid, last partial wave, an even grid for the row parities): prototypes of
    batch 1 and batch 72 within fp16 rounding of a batch-8 run of the same frames (the tolerance of test_gpu_parity's batch
    test: the other layers' plans change with the batch too)."""
    layers, ws = W.random_weights("n", seed=1)
    model = I.Model(W.write_pack("n", layers, ws), "n")
    fr = np.random.default_rng(0).integers(0, 256, (8, 640, 640, 3), dtype=np.uint8)
    ref = _run(model, fr)["protos"].reshape(8, 32, -1)
    one = _run(model, fr[3:4])["protos"].reshape(1, 32, -1)
    assert np.abs(one[0] - ref[3]).max() <= 0.1
    big = _run(model, np.tile(fr, (9, 1, 1, 1)))["protos"].reshape(72, 32, -1)
    assert np.abs(big[-8:] - ref).max() <= 0.1
    assert np.abs(big[:8] - ref).max() <= 0.1
