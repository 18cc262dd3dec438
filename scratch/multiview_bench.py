"""Cost of the multi-view refinement (PathConfig.multiview): the geometry and fix-up kernels' MV instantiations.

Bench shape: the bench.py workload (185 views, 46 reference views, RoMa fast 512x512, M = 10 000, all filters) at 4 and at 8
neighbours, multiview off and on, kept 3 launches in flight on a DensifyRing, the variants alternating in one process, timed
with CUDA events.  Also: per-kernel times (ldp_profile_*) of profiled launches, one at a time, per variant.

    python scratch/multiview_bench.py [--steps 200] [--rounds 5] [--out results.json]
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
from lichtfeld_densification_plugin_b200.engine import DensifyRing, PathConfig  # noqa: E402

VARIANTS = {"nn4_off": (4, False), "nn4_on": (4, True), "nn8_off": (8, False), "nn8_on": (8, True)}


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
    cfgs = {name: PathConfig(matches_per_ref=10000, multiview=mv) for name, (nn, mv) in VARIANTS.items()}
    rings = {name: DensifyRing(dev, depth=3) for name in VARIANTS}      # one per variant: each keeps its own workspaces
    prepared = {}
    for nn in (4, 8):
        scene = synth.make_scene(185, "fast", 0.25, nn)
        inputs = [synth.synth_ref_inputs(scene, rp, device=dev, cert_family="R", seed=0) for rp in range(scene.n_refs)]
        for name, (vnn, mv) in VARIANTS.items():
            if vnn == nn:
                prepared[name] = [e.prepare(batch_for(e, scene, inputs), cfgs[name]) for e in rings[name].engines]
    torch.cuda.synchronize()

    def run(name, steps):
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        evs[0].record()
        ring = rings[name]
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
    result = {"card": card, "shape": "185 views, 46 refs, fast 512x512, M=10000, all filters, 3 in flight", "variants": {}}
    for name in VARIANTS:
        pl = prepared[name][0]
        pts = pl.outputs.total_points()
        kt = kernel_times(rings[name].engines[0], pl.outputs._keep[2], cfgs[name])
        med = float(np.median(ms[name]))
        result["variants"][name] = dict(ms_per_step_median=round(med, 4), ms_per_step_rounds=[round(x, 4) for x in ms[name]],
                                        points_per_step=pts, points_per_s=round(pts / (med * 1e-3)), kernel_us=kt)
        if VARIANTS[name][1]:
            n = pl.outputs.total_points()
            vm = pl.outputs.view_mask[:n].cpu().numpy().view(np.uint32)
            result["variants"][name]["cameras_per_point"] = np.bincount(np.bitwise_count(vm) + 1).tolist()
        print(name, json.dumps(result["variants"][name]))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
