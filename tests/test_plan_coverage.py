"""Plan coverage: every convolution plan the planner can emit runs through the layer-local float64 check.

The planner picks each launch's mode, K-blocks, rows per item, sub-tiles, stages and N split from the micro-batch and the
class count, and the runner then shrinks the plan for a partial last chunk and caps the grid of small launches.  Those
choices decide how many rounds each CTA runs through the item loop, whether the last round is ragged and whether the last
item is a partial tile -- the bookkeeping where a kernel goes wrong at one batch size and not at another.

`tools/plan_dump sig` prints, per launch of the runner's list, the signature of the code path it runs (see its header)
with exactly the parameters the runner derives (model.cuh plan_conv_op / conv_launch_params).  The sweep enumerates the
signatures over

    scale n and s, micro-batch 1 .. 512 at 80 classes, each with the full chunk and partial chunks of 1, 2, 3 and mb - 1
    frames; and every class count of NC_EDGES at micro-batch 1,

and COVER lists the runner configurations (scale, max_batch, batch, micro_batch, classes) that reach every (launch,
signature) pair of it.  On the CPU the guard fails, naming each pair and a configuration that reaches it, as soon as a
planner change adds a plan COVER does not run.  `python tests/test_plan_coverage.py <plan_dump>` prints a fresh table:
greedy, the configuration that reaches the most uncovered pairs first, smaller batches first among equals.

On the GPU each COVER entry runs the runner and checks, with test_layer_local's LocalCheck in targets mode, the launches
whose pair that entry is the first of the table to reach, on the frames the sig line names for them (those holding item
0, the first item of the second round and the last item).  The bound is LocalCheck's, unchanged.  It also asserts that
the runner's launch list is the sig list: the same launches in the same order, each with the sig line's grid, work items
and mode.
"""
from __future__ import annotations

import functools
import os
import re
import subprocess
import sys
import time

import numpy as np
import pytest
import torch

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
for p in (ROOT, os.path.dirname(os.path.abspath(__file__))):
    if p not in sys.path:
        sys.path.insert(0, p)

from test_abi import plan_dump  # noqa: E402,F401  (fixture: tools/plan_dump.cu compiled for the host)
from test_layer_local import (Fusion, _gpu_name, failures, launch_tensors, plan_ops, random_weights, run_reference,  # noqa: E402
                              spec_for)

SMS = 148                 # the planner's inputs include the SM count: the table holds for a 148-SM B200 only
# Class counts at the ends of each range over which the decode variant (80-class, segment table, wide) and the N split of
# every class launch stay the same at micro-batch 1 (test_class_count_edges_come_from_the_sweep derives them).
NC_EDGES = [1, 79, 80, 81, 112, 113, 128, 129, 144, 145, 160, 161, 176, 177, 192, 193, 208, 209, 224, 225, 240, 241, 256, 257, 512,
            513, 1024]
SWEEP = [("ns", "1-512", "mb,1,2,3,mb-1", "80"), ("ns", "1", "mb", ",".join(map(str, NC_EDGES)))]

# (scale, max_batch, batch, micro_batch, classes): batch < max_batch runs a partial chunk planned for max_batch frames
COVER = [
    ('n', 1, 1, 0, 1), ('n', 1, 1, 0, 79), ('n', 1, 1, 0, 81), ('n', 1, 1, 0, 112), ('n', 1, 1, 0, 113),
    ('n', 1, 1, 0, 129), ('n', 1, 1, 0, 145), ('n', 1, 1, 0, 161), ('n', 1, 1, 0, 177), ('n', 1, 1, 0, 193),
    ('n', 1, 1, 0, 209), ('n', 1, 1, 0, 225), ('n', 1, 1, 0, 241), ('n', 1, 1, 0, 257), ('n', 1, 1, 0, 512),
    ('n', 1, 1, 0, 513), ('n', 1, 1, 0, 1024), ('n', 2, 1, 0, 80), ('n', 2, 2, 0, 80), ('n', 3, 2, 0, 80),
    ('n', 3, 3, 0, 80), ('n', 4, 4, 0, 80), ('n', 5, 1, 0, 80), ('n', 6, 1, 0, 80), ('n', 6, 2, 0, 80), ('n', 6, 5, 0, 80),
    ('n', 8, 8, 0, 80), ('n', 9, 1, 0, 80), ('n', 9, 2, 0, 80), ('n', 11, 11, 0, 80), ('n', 12, 1, 0, 80),
    ('n', 12, 2, 0, 80), ('n', 12, 12, 0, 80), ('n', 15, 1, 0, 80), ('n', 15, 2, 0, 80), ('n', 15, 3, 0, 80),
    ('n', 16, 16, 0, 80), ('n', 18, 1, 0, 80), ('n', 18, 2, 0, 80), ('n', 19, 19, 0, 80), ('n', 22, 21, 0, 80),
    ('n', 24, 1, 0, 80), ('n', 24, 2, 0, 80), ('n', 24, 24, 0, 80), ('n', 30, 1, 0, 80), ('n', 30, 29, 0, 80),
    ('n', 32, 31, 0, 80), ('n', 36, 2, 0, 80), ('n', 37, 37, 0, 80), ('n', 38, 38, 0, 80), ('n', 43, 1, 0, 80),
    ('n', 48, 2, 0, 80), ('n', 48, 3, 0, 80), ('n', 48, 47, 0, 80), ('n', 48, 48, 0, 80), ('n', 60, 1, 0, 80),
    ('n', 60, 2, 0, 80), ('n', 60, 59, 0, 80), ('n', 60, 60, 0, 80), ('n', 71, 71, 0, 80), ('n', 72, 1, 0, 80),
    ('n', 72, 2, 0, 80), ('n', 72, 71, 0, 80), ('n', 73, 73, 0, 80), ('n', 74, 74, 0, 80), ('n', 75, 74, 0, 80),
    ('n', 83, 83, 0, 80), ('n', 89, 88, 0, 80), ('n', 95, 2, 0, 80), ('n', 95, 94, 0, 80), ('n', 112, 112, 0, 80),
    ('n', 142, 142, 0, 80), ('n', 143, 1, 0, 80), ('n', 143, 142, 0, 80), ('n', 144, 144, 0, 80), ('n', 148, 148, 0, 80),
    ('n', 149, 148, 0, 80), ('n', 190, 1, 0, 80), ('n', 192, 192, 0, 80), ('n', 213, 213, 0, 80), ('n', 223, 223, 0, 80),
    ('n', 237, 1, 0, 80), ('n', 237, 236, 0, 80), ('n', 240, 240, 0, 80), ('n', 284, 284, 0, 80), ('n', 285, 1, 0, 80),
    ('n', 285, 284, 0, 80), ('n', 285, 285, 0, 80), ('n', 296, 296, 0, 80), ('n', 297, 296, 0, 80), ('n', 367, 367, 0, 80),
    ('n', 379, 1, 0, 80), ('n', 384, 384, 0, 80), ('n', 426, 426, 0, 80), ('n', 445, 1, 0, 80), ('n', 445, 444, 0, 80),
    ('n', 445, 445, 0, 80), ('s', 1, 1, 0, 1), ('s', 1, 1, 0, 79), ('s', 1, 1, 0, 81), ('s', 1, 1, 0, 112),
    ('s', 1, 1, 0, 113), ('s', 1, 1, 0, 129), ('s', 1, 1, 0, 145), ('s', 1, 1, 0, 161), ('s', 1, 1, 0, 177),
    ('s', 1, 1, 0, 193), ('s', 1, 1, 0, 209), ('s', 1, 1, 0, 225), ('s', 1, 1, 0, 241), ('s', 1, 1, 0, 257),
    ('s', 1, 1, 0, 512), ('s', 1, 1, 0, 513), ('s', 1, 1, 0, 1024), ('s', 2, 1, 0, 80), ('s', 2, 2, 0, 80),
    ('s', 3, 1, 0, 80), ('s', 3, 2, 0, 80), ('s', 3, 3, 0, 80), ('s', 4, 1, 0, 80), ('s', 4, 4, 0, 80), ('s', 5, 1, 0, 80),
    ('s', 6, 1, 0, 80), ('s', 6, 2, 0, 80), ('s', 7, 7, 0, 80), ('s', 8, 8, 0, 80), ('s', 9, 2, 0, 80), ('s', 9, 3, 0, 80),
    ('s', 11, 1, 0, 80), ('s', 12, 1, 0, 80), ('s', 12, 2, 0, 80), ('s', 12, 11, 0, 80), ('s', 13, 13, 0, 80),
    ('s', 15, 1, 0, 80), ('s', 15, 2, 0, 80), ('s', 15, 3, 0, 80), ('s', 16, 16, 0, 80), ('s', 18, 1, 0, 80),
    ('s', 18, 2, 0, 80), ('s', 19, 19, 0, 80), ('s', 21, 2, 0, 80), ('s', 22, 1, 0, 80), ('s', 22, 21, 0, 80),
    ('s', 24, 2, 0, 80), ('s', 24, 24, 0, 80), ('s', 30, 1, 0, 80), ('s', 30, 29, 0, 80), ('s', 36, 1, 0, 80),
    ('s', 36, 2, 0, 80), ('s', 37, 37, 0, 80), ('s', 38, 38, 0, 80), ('s', 48, 2, 0, 80), ('s', 48, 3, 0, 80),
    ('s', 48, 47, 0, 80), ('s', 48, 48, 0, 80), ('s', 60, 1, 0, 80), ('s', 60, 2, 0, 80), ('s', 60, 59, 0, 80),
    ('s', 60, 60, 0, 80), ('s', 71, 71, 0, 80), ('s', 72, 1, 0, 80), ('s', 72, 2, 0, 80), ('s', 72, 71, 0, 80),
    ('s', 73, 73, 0, 80), ('s', 74, 74, 0, 80), ('s', 75, 74, 0, 80), ('s', 95, 2, 0, 80), ('s', 96, 96, 0, 80),
    ('s', 112, 1, 0, 80), ('s', 112, 111, 0, 80), ('s', 142, 142, 0, 80), ('s', 143, 1, 0, 80), ('s', 143, 142, 0, 80),
    ('s', 144, 144, 0, 80), ('s', 148, 148, 0, 80), ('s', 149, 148, 0, 80), ('s', 190, 1, 0, 80), ('s', 190, 189, 0, 80),
    ('s', 192, 192, 0, 80), ('s', 213, 213, 0, 80), ('s', 237, 1, 0, 80), ('s', 237, 236, 0, 80), ('s', 240, 240, 0, 80),
    ('s', 284, 284, 0, 80), ('s', 285, 1, 0, 80), ('s', 285, 284, 0, 80), ('s', 285, 285, 0, 80), ('s', 296, 296, 0, 80),
    ('s', 297, 296, 0, 80), ('s', 367, 367, 0, 80), ('s', 379, 1, 0, 80), ('s', 384, 384, 0, 80), ('s', 426, 426, 0, 80),
    ('s', 445, 1, 0, 80), ('s', 445, 444, 0, 80), ('s', 445, 445, 0, 80),
]


# ---- signatures ---------------------------------------------------------------------------------------------------------
def parse_sig(out: str):
    """plan_dump sig lines -> dicts: cfg (scale, mb, nb, nc), kind, launch, pair (scale, launch, signature), geo."""
    for line in out.splitlines():
        head, sig, geo = line.split(" | ")
        t = head.split()
        g = geo.split()
        yield dict(cfg=(t[1], int(t[2]), int(t[3]), int(t[4])), kind=t[5], launch=t[6], pair=(t[1], t[6], sig), sig=sig,
                   geo=dict(zip(g[0::2], g[1::2])), frames=g[g.index("frames") + 1:] if "frames" in g else [])


def run_sig(exe: str, *args: str) -> list[dict]:
    out = subprocess.run([exe, "sig", *args], capture_output=True, text=True, check=True).stdout
    return list(parse_sig(out))


def sweep_pairs(exe: str) -> dict:
    """(scale, launch, signature) -> the first sweep configuration (scale, mb, nb, nc) that reaches it."""
    first = {}
    for args in SWEEP:
        for l in run_sig(exe, *args, "uniq"):
            first.setdefault(l["pair"], l["cfg"])
    return first


def entry_lines(exe: str, entry) -> list[dict]:
    scale, mb, batch, micro, nc = entry
    assert micro == 0, "COVER runs one chunk: batch <= max_batch"
    return run_sig(exe, scale, str(mb), str(batch), str(nc))


def reached(exe: str, cover) -> dict:
    """(scale, launch, signature) -> index of the first COVER entry that reaches it."""
    first = {}
    for i, e in enumerate(cover):
        for l in entry_lines(exe, e):
            first.setdefault(l["pair"], i)
    return first


def uncovered(all_pairs: dict, reach: dict) -> list[str]:
    return [f"{s} {launch}: [{sig}] -- reached by (scale {c[0]}, max_batch {c[1]}, batch {c[2]}, micro_batch 0, nc {c[3]})"
            for (s, launch, sig), c in sorted(all_pairs.items()) if (s, launch, sig) not in reach]


def greedy_cover(exe: str) -> list[tuple]:
    first = sweep_pairs(exe)
    cands = sorted(set(first.values()), key=lambda c: (c[1], c[2], c[0], c[3]))
    sets = {c: {l["pair"] for l in run_sig(exe, c[0], str(c[1]), str(c[2]), str(c[3]))} for c in cands}
    left, chosen = set(first), []
    while left:
        c = max(cands, key=lambda c: (len(sets[c] & left), -c[1], -c[2]))
        chosen.append(c)
        left -= sets[c]
    return [(c[0], c[1], c[2], 0, c[3]) for c in sorted(chosen)]


# ---- CPU --------------------------------------------------------------------------------------------------------------
def test_cover_reaches_every_plan_of_the_sweep(plan_dump):
    all_pairs = sweep_pairs(plan_dump)
    missing = uncovered(all_pairs, reached(plan_dump, COVER))
    for s in "ns":
        print(f"scale {s}: {sum(p[0] == s for p in all_pairs)} (launch, signature) pairs, "
              f"{sum(e[0] == s for e in COVER)} COVER entries")
    assert not missing, f"{len(missing)} plans no COVER entry runs:\n" + "\n".join(missing[:200])


def test_dropping_a_cover_entry_names_the_pairs_only_it_reaches(plan_dump):
    all_pairs = sweep_pairs(plan_dump)
    for drop in (0, len(COVER) // 2, len(COVER) - 1):
        rest = COVER[:drop] + COVER[drop + 1:]
        own = {l["pair"] for l in entry_lines(plan_dump, COVER[drop])} - set(reached(plan_dump, rest))
        missing = uncovered(all_pairs, reached(plan_dump, rest))
        assert own, f"COVER entry {COVER[drop]} reaches nothing the others do not"
        assert len(missing) == len(own)
        for (s, launch, sig) in own:
            assert any(m.startswith(f"{s} {launch}: [{sig}]") for m in missing), (launch, sig)


def test_class_count_edges_come_from_the_sweep(plan_dump):
    """At micro-batch 1, every range of class counts over which the decode variant and the N split of every class launch
    stay the same starts and ends at a count of NC_EDGES."""
    for s in "ns":
        key = {}
        for l in run_sig(plan_dump, s, "1", "mb", "1-1024"):
            nc = l["cfg"][3]
            if l["kind"] == "post":
                key.setdefault(nc, []).append(l["sig"].split()[1])
            elif ".cls." in l["launch"] and l["kind"] == "conv":
                t = l["sig"].split()
                key.setdefault(nc, []).append(t[t.index("n_tiles") + 1])
        edges = {1, 1024}
        for nc in range(2, 1025):
            if key[nc] != key[nc - 1]:
                edges |= {nc - 1, nc}
        assert edges <= set(NC_EDGES), (s, sorted(edges - set(NC_EDGES)))


# ---- GPU --------------------------------------------------------------------------------------------------------------
MODES = {"gather": 0, "halo": 1, "halo_tma": 2, "flat_tma": 3, "s2_tma": 4}


@functools.lru_cache(maxsize=None)
def _targets_of(exe: str) -> dict:
    return reached(exe, COVER)


@functools.lru_cache(maxsize=4)
def _model(scale: str, nc: int):
    from xr_image_segmentation_b200 import inference as I, weights as W
    layers, ws = random_weights(scale, nc, seed=21)
    return I.Model(W.write_pack(scale, layers, ws), scale, nc), [(w, b) for w, b in ws]


def runner_name(l: dict) -> str:
    """The name xrseg_api.cu add_network_launches gives the launch of sig line l."""
    kind, name = l["kind"], l["launch"]
    sig = l["sig"].split()
    if kind == "bneck":
        return name[:-len(".cv1")]                       # "b2.m0.cv1" -> "b2.m0"
    if kind == "attn":
        return "c2psa.attention" if name == "attn" else "c2psa.attention+pe"
    if kind in ("sppf", "up"):
        return {"sppf": "sppf.pool", "up": "upsample2x"}[kind]
    if kind == "conv" and "+" in name:                  # siblings: "b6.m0.cv1+m0.cv2", at most 31 characters
        a, b = name.split("+")
        return (a + "+" + b[b.index(".") + 1:])[:31]
    if kind == "conv" and sig[sig.index("tail") + 1] == "1":
        n = name + "+cv3"                                 # the fused proto.cv3 tail
        return "proto.up+" + n[n.index(".") + 1:] if sig[sig.index("upm") + 1] == "1" else n
    return name


def _frames_of(lines: list[dict]) -> list[int]:
    out = set()
    for l in lines:
        for r in l["frames"]:
            if r != "-":
                a, b = (int(v) for v in r.split(":"))
                out.update(range(a, b + 1))
    return sorted(out)


def run_entry(exe: str, idx: int) -> tuple[str, list[str]]:
    from xr_image_segmentation_b200 import _lib, inference as I
    entry = COVER[idx]
    scale, mb, batch, micro, nc = entry
    t0 = time.time()
    lines = entry_lines(exe, entry)
    first = _targets_of(exe)
    target_lines = [l for l in lines if first[l["pair"]] == idx and l["kind"] != "post"]
    ups, targets = 0, set()
    for l in lines:
        if l["kind"] == "post":
            continue
        sig = l["sig"].split()
        o = dict(kind=l["kind"], name="-" if l["kind"] == "up" else l["launch"],
                 tail="proto.cv3" if "tail" in sig and sig[sig.index("tail") + 1] == "1" else None,
                 merged="proto.up" if "upm" in sig and sig[sig.index("upm") + 1] == "1" else None)
        if l in target_lines:
            targets |= launch_tensors(o, ups)[1]
        ups += l["kind"] == "up"
    sample = _frames_of(target_lines)
    if not sample:
        return f"{entry}: no network launch to check (post side only)", []
    model, weights = _model(scale, nc)
    rng = np.random.default_rng(idx)
    frames = rng.integers(0, 256, (batch, 640, 640, 3), dtype=np.uint8)
    r = I.Runner(model, max_batch=mb, micro_batch=micro, conv_impl=_lib.CONV_UMMA, debug=True)
    try:
        r.schedule(frames)
        r.wait(strict=False)                              # random class logits may overflow the NMS caps
        # the runner's launch geometry is the sig line's
        net = [l for l in lines if l["kind"] != "post"]
        got = r.launches()
        assert len(got) > len(net) and got[len(net)][0].startswith("post.") and \
            not got[len(net) - 1][0].startswith("post."), (len(net), [g[0] for g in got])
        bad = []
        for l, (name, grid, items, mode) in zip(net, got):
            if name != runner_name(l):
                bad.append(f"{l['launch']}: the runner launches {name} here, the sig list {runner_name(l)}")
            if l["kind"] == "stem":
                continue
            g = l["geo"]
            want = (int(g["grid"]), int(g["items"]), MODES[l["sig"].split()[1]] if l["kind"] == "conv" else -1)
            if (grid, items, mode) != want:
                bad.append(f"{l['launch']} ({name}): runner grid/items/mode {(grid, items, mode)}, sig {want}")
        assert not bad, "\n".join(bad)
        cache = {}

        def provider(name):
            if name not in cache:
                cache.clear()
                cache[name] = torch.from_numpy(np.concatenate([r.fetch(name, f, 1) for f in sample])).double()
            return cache[name]

        fusion = Fusion.from_ops(plan_ops(exe, scale, nc), stem_f32=False)   # 640x640 host frames: the fp16 mma stems
        x = torch.from_numpy(frames[sample].transpose(0, 3, 1, 2).astype(np.float64) / 255.0)
        chk = run_reference(weights, spec_for(scale, nc), fusion, provider, x, targets)
    finally:
        r.close()
    assert targets <= set(chk.results), sorted(targets - set(chk.results))
    name, res = max(((n, v) for n, v in chk.results.items() if n in targets), key=lambda kv: kv[1]["ratio"])
    f, c, y, xx = (int(v) for v in res["where"])
    line = (f"{entry}: {len(target_lines)} target launches, frames {sample}: worst |err|/bound {res['ratio']:.3g} at {name} "
            f"frame {sample[f]} c {c} y {y} x {xx}; {time.time() - t0:.1f} s")
    # a failure names the frame within the chunk, not its index among the sampled frames
    fails = [re.sub(r"frame (\d+) ", lambda m: f"frame {sample[int(m.group(1))]} ", f, count=1) for f in failures(chk)]
    return line, fails


@pytest.mark.gpu
@pytest.mark.parametrize("idx", range(len(COVER)), ids=[f"{e[0]}-mb{e[1]}-b{e[2]}-nc{e[4]}" for e in COVER])
def test_every_plan_is_within_its_bound(lib, dlib, plan_dump, idx):
    assert torch.cuda.get_device_properties(0).multi_processor_count == SMS, "COVER was computed for 148 SMs"
    line, fails = run_entry(plan_dump, idx)
    print(_gpu_name() + ": " + line)
    assert not fails, "\n".join(fails)


@pytest.mark.gpu
@pytest.mark.parametrize("nc", NC_EDGES)
def test_post_side_of_every_class_range(lib, plan_dump, nc):
    """test_pipeline_ends' designed post-processing tensors at every class count of NC_EDGES: each decode variant (80-class,
    segment table, wide) and class pitch at the ends of its range."""
    import test_pipeline_ends as PE
    post = [l for l in run_sig(plan_dump, "n", "1", "mb", str(nc)) if l["kind"] == "post"]
    assert len(post) == 1, post
    box, cls, coefs, protos, planted = PE.designed_post(nc)
    r = PE.post_runner(nc, len(planted))
    try:
        out = PE.run_post(r, box, cls, coefs, protos)
    finally:
        r.close()
    results, lines = PE.check_post(out, box, cls, coefs, protos, planted, f"nc {nc} ({post[0]['sig']})")
    print(_gpu_name())
    PE.settle(results, lines)


if __name__ == "__main__":                               # print a fresh COVER table
    for e in greedy_cover(sys.argv[1]):
        print(f"    {e!r},")
