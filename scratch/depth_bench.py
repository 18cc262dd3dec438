"""Cost of the dense depth maps (ldp_depth_maps) at the bench shape (46 views, 512^2 maps, nn = 4, all filters) and at
config 5's 640^2 maps (32 views per launch), multi-view refinement off and on.

Per case: the depth kernel's and the fix-up's time from ldp_profile_* (CUDA events around each kernel; median of --reps
calls after a warm-up call), pixels per second, the bytes the kernel has to move (certainty words of every neighbour at
every pixel, the winner's 16-byte warp row at every candidate, the 4-byte depth) against a device-to-device copy's measured
rate in the same process, and the fix-up's entry count.  Certainty planes are the synthetic "R" family with its floor at
0.2, min_certainty 0.5.

    python scratch/depth_bench.py [--reps 5] [--out results.json]
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
from lichtfeld_densification_plugin_b200.engine import DensifyEngine, PathConfig  # noqa: E402


def copy_rate(dev) -> float:
    """bytes/s of a 2 GB device-to-device copy (read + write counted), median of 5"""
    a = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
    b = torch.empty_like(a)
    b.copy_(a)
    ts = []
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); b.copy_(a); e1.record(); e1.synchronize()
        ts.append(e0.elapsed_time(e1) / 1e3)
    return 2 * a.numel() / float(np.median(ts))


def run_case(eng, setting, n_refs, nn, multiview, reps, min_cert=0.5):
    scene = synth.make_scene(max(n_refs, 8), setting, ref_fraction=1.0, nn=nn)
    dev = eng.device
    inputs = [synth.synth_ref_inputs(scene, rp, device=dev, cert_family="R", seed=rp) for rp in range(n_refs)]
    b = eng.new_batch(scene.H, scene.W, scene.w_match, scene.h_match)
    for inp in inputs:
        k = len(inp["nbr_indices"])
        b.add([inp["cert"][q] for q in range(k)], [inp["warp"][q] for q in range(k)], inp["image"], scene.cameras[inp["ref_index"]],
              [scene.cameras[j] for j in inp["nbr_indices"]])
    cfg = PathConfig(multiview=multiview)
    lib = eng.lib
    eng.depth_maps(b, cfg, min_cert)
    torch.cuda.synchronize()
    lib.ldp_profile_enable(1)
    kd, kf = [], []
    buf = (C.c_float * 8)()
    for _ in range(reps):
        out = eng.depth_maps(b, cfg, min_cert, want_flags=True)
        n = lib.ldp_profile_read(buf, 8)
        names = [lib.ldp_profile_name(i).decode() for i in range(n)]
        kd.append(buf[names.index("ldp_depth_kernel")])
        kf.append(buf[names.index("ldp_depth_fix_kernel")])
    lib.ldp_profile_enable(0)
    torch.cuda.synchronize()
    flags = out.flags.cpu().numpy()
    cand = int((flags & 1).sum())
    kept = int(out.kept.sum().item())
    fix = int(eng.depth_fixups(n_refs).sum())
    px = n_refs * scene.H * scene.W
    bytes_moved = px * (4 * nn + 4) + cand * 16
    t = float(np.median(kd)) / 1e3
    return dict(setting=setting, H=scene.H, W=scene.W, n_refs=n_refs, nn=nn, multiview=multiview, pixels=px, candidates=cand,
                kept=kept, fixup_entries=fix, depth_kernel_ms=float(np.median(kd)), fix_kernel_ms=float(np.median(kf)),
                pixels_per_s=px / t, bytes=bytes_moved, bytes_per_s=bytes_moved / t)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    eng = DensifyEngine()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    peak = copy_rate(eng.device)
    res = dict(gpu=gpu, copy_bytes_per_s=peak, cases=[])
    print(f"GPU: {gpu}; device copy {peak / 1e12:.2f} TB/s")
    for setting, R in (("fast", 46), ("base", 32)):
        for mv in (False, True):
            c = run_case(eng, setting, R, 4, mv, a.reps)
            c["share_of_copy_rate"] = c["bytes_per_s"] / peak
            res["cases"].append(c)
            print(f"{c['H']}^2 x {R} views, multiview={mv}: depth kernel {c['depth_kernel_ms']:.3f} ms, fix-up "
                  f"{c['fix_kernel_ms']:.3f} ms ({c['fixup_entries']} entries); {c['pixels_per_s'] / 1e9:.2f} G px/s; "
                  f"{c['bytes'] / 1e6:.0f} MB = {c['bytes_per_s'] / 1e12:.2f} TB/s ({100 * c['share_of_copy_rate']:.1f} % of the copy); "
                  f"candidates {c['candidates']}, kept {c['kept']}")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        json.dump(res, open(a.out, "w"), indent=1)


if __name__ == "__main__":
    main()
