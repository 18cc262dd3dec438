"""Cost of the lens instantiation of the geometry kernels (CameraRecord.from_colmap cameras), beside pinhole cameras.

Bench shape: the bench.py workload (185 views, 46 reference views, RoMa fast 512x512, 4 neighbours, M = 10 000, all filters)
with three camera sets - pinhole, OPENCV, OPENCV_FISHEYE - kept 3 launches in flight on a DensifyRing, the variants
alternating in one process, timed with CUDA events.  Also: per-kernel times of one profiled launch per variant, and the
config-3 shape (RoMa precise: 1280x1280 maps, 800x800 matching, OPENCV) run once.

    python scratch/lens_bench.py [--steps 200] [--rounds 5] [--out results.json]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from lichtfeld_densification_plugin_b200 import synth  # noqa: E402
from lichtfeld_densification_plugin_b200.engine import DensifyEngine, DensifyRing, PathConfig  # noqa: E402

VARIANTS = {"pinhole": None, "OPENCV": ("OPENCV", [-0.12, 0.03, 4e-4, -3e-4]),
            "OPENCV_FISHEYE": ("OPENCV_FISHEYE", [0.05, -0.01, 0.003, -0.0005])}


def batch_for(eng, scene, inputs):
    b = eng.new_batch(scene.H, scene.W, scene.w_match, scene.h_match)
    cams = scene.cameras
    for inp in inputs:
        nn = len(inp["nbr_indices"])
        b.add([inp["cert"][k] for k in range(nn)], [inp["warp"][k] for k in range(nn)], inp["image"], cams[inp["ref_index"]],
              [cams[j] for j in inp["nbr_indices"]], rng_stream=inp["ref_index"])
    return b


def kernel_times(eng, batch, cfg, reps: int = 10):
    """us per kernel, averaged over `reps` profiled launches (CUDA events around each kernel, one launch at a time)."""
    lib = eng.lib
    lib.ldp_profile_enable(1)
    buf = (C.c_float * 64)()
    acc = {}
    for _ in range(reps):
        eng.densify(batch, cfg)
        n = lib.ldp_profile_read(buf, 64)
        for k in range(n):          # names are valid until profiling is switched off
            name = lib.ldp_profile_name(k).decode()
            acc[name] = acc.get(name, 0.0) + float(buf[k]) * 1e3 / reps
    lib.ldp_profile_enable(0)
    return {k: round(v, 2) for k, v in acc.items()}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the results as JSON here")
    args = ap.parse_args()
    dev = torch.device("cuda", torch.cuda.current_device())
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    print("card:", card)
    cfg = PathConfig(matches_per_ref=10000)
    ring = DensifyRing(dev, depth=3)
    prepared = {}
    for name, lens in VARIANTS.items():
        scene = synth.make_scene(185, "fast", 0.25, 4, lens=lens)
        inputs = [synth.synth_ref_inputs(scene, rp, device=dev, cert_family="R", seed=0) for rp in range(scene.n_refs)]
        prepared[name] = [e.prepare(batch_for(e, scene, inputs), cfg) for e in ring.engines]
        assert prepared[name][0].params.lens == (0 if lens is None else 1)
    torch.cuda.synchronize()

    def run(name, steps):
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        evs[0].record()
        for s in range(steps):
            j = s % ring.depth
            st = ring.streams[j]
            st.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(st):
                prepared[name][j].launch()
        for st in ring.streams:            # join the ring once, after the last launch: the launches overlap
            torch.cuda.current_stream().wait_stream(st)
        evs[1].record()
        torch.cuda.synchronize()
        return evs[0].elapsed_time(evs[1]) / steps

    for name in VARIANTS:
        run(name, 20)
    ms = {name: [] for name in VARIANTS}
    for _ in range(args.rounds):
        for name in VARIANTS:
            ms[name].append(run(name, args.steps))
    result = {"card": card, "shape": "185 views, 46 refs, fast 512x512, 4 nn, M=10000, all filters, 3 in flight", "variants": {}}
    for name in VARIANTS:
        pl = prepared[name][0]
        pts = pl.outputs.total_points()
        kt = kernel_times(ring.engines[0], pl.outputs._keep[2], cfg)
        med = float(np.median(ms[name]))
        step_total = sum(kt.values())
        geo = sum(v for k, v in kt.items() if k in ("ldp_geometry_kernel", "ldp_fix_kernel"))
        result["variants"][name] = dict(ms_per_step_median=round(med, 4), ms_per_step_rounds=[round(x, 4) for x in ms[name]],
                                        points_per_step=pts, points_per_s=round(pts / (med * 1e-3)),
                                        kernel_us=kt, geometry_share=round(geo / step_total, 3))
        print(name, json.dumps(result["variants"][name]))
    # config 3: RoMa precise, OPENCV, run once (after one warm-up launch)
    scene = synth.make_scene(40, "precise", 0.2, 4, lens=VARIANTS["OPENCV"])
    inputs = [synth.synth_ref_inputs(scene, rp, device=dev, cert_family="R", seed=0) for rp in range(scene.n_refs)]
    eng = DensifyEngine(dev)
    b = batch_for(eng, scene, inputs)
    eng.densify(b, cfg)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    o = eng.densify(b, cfg)
    e1.record()
    torch.cuda.synchronize()
    result["config3_opencv"] = dict(refs=len(inputs), ms=round(e0.elapsed_time(e1), 3), points=o.total_points(),
                                    kernel_us=kernel_times(eng, b, cfg))
    print("config3", json.dumps(result["config3_opencv"]))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
