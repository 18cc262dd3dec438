"""Cost of the normal maps (ldp_depth_normals) and of the oriented fusion (ldp_fuse_depth_maps_oriented) on the analytic
sphere maps of scratch/fusion_bench.py, at 46 views x 512^2 and 250 views x 640^2.

Normal maps: the check and normal kernels' times from ldp_profile_* (CUDA events around each kernel), median of --reps calls
after a warm-up call, at radius 1, 2 and 3 (rel_tol 0.05), as ms and pixels/s over all pixels of the maps.  Beside them, a
device-to-device copy of the xyz maps timed with CUDA events in the same process: the bandwidth the kernel's reads could
reach.  Fusion: ldp_fuse_depth_maps and, on the same maps with radius-2 normal maps, the oriented entry point at 10 degrees,
per kernel.  The card's name and power limit are read in the same run.

    python scratch/depth_normals_bench.py [--reps 5] [--out results.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from lichtfeld_densification_plugin_b200 import _native as N  # noqa: E402
from lichtfeld_densification_plugin_b200.engine import DepthViews  # noqa: E402
from lichtfeld_densification_plugin_b200.output import estimate_depth_normals, fuse_depth_maps  # noqa: E402
from scratch.fusion_bench import profiled, sphere_views  # noqa: E402


def copy_rate(views, reps):
    """bytes/s of a device-to-device copy of every view's xyz map (read + write), median of reps"""
    src = torch.stack(views.xyz)
    dst = torch.empty_like(src)
    dst.copy_(src)
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        dst.copy_(src)
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    return 2 * src.numel() * 4 / (float(np.median(ts)) / 1e3)


def case(lib, V, S, reps, dev):
    views = sphere_views(V, S, dev)
    px = V * S * S
    finite = int(sum(int(torch.isfinite(m).sum()) for m in views.maps))
    out = dict(V=V, H=S, W=S, pixels=px, finite_pixels=finite, copy_GBps=copy_rate(views, reps) / 1e9, normals=[])
    for r in (1, 2, 3):
        k = profiled(lib, lambda: estimate_depth_normals(views, radius=r), reps)
        t = k["ldp_depth_normals_kernel"]
        res = estimate_depth_normals(views, radius=r)
        # bytes the kernel must move at least: depth + xyz read, normals + curvature written, 28 bytes per pixel
        out["normals"].append(dict(radius=r, kernel_ms=t, check_ms=k.get("ldp_depth_normals_check_kernel", float("nan")),
                                   pixels_per_s=px / (t / 1e3), min_bytes_GBps=28 * px / (t / 1e3) / 1e9,
                                   undefined=res.undefined))
    nrm = estimate_depth_normals(views, radius=2).normals
    oriented = DepthViews(S, S, S, S, dev)
    for v in range(V):
        oriented.add(views.maps[v], views.cameras[v], xyz=views.xyz[v], rgb=views.rgb[v], err=views.err[v], normals=nrm[v])
    plain_k = profiled(lib, lambda: fuse_depth_maps(views), reps)
    orient_k = profiled(lib, lambda: fuse_depth_maps(oriented, max_normal_angle=10.0), reps)
    p, o = fuse_depth_maps(views), fuse_depth_maps(oriented, max_normal_angle=10.0)
    names = ("ldp_fusion_verdict_kernel", "ldp_fusion_emit_kernel", "ldp_fusion_sum_kernel")
    out["fusion"] = dict(plain={n: plain_k[n] for n in names}, oriented={n: orient_k[n] for n in names},
                         plain_emitted=int(p.source.numel()), oriented_emitted=int(o.source.numel()),
                         plain_mean_views=float(p.n_views.float().mean()), oriented_mean_views=float(o.n_views.float().mean()))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    lib = N.load()
    dev = torch.device("cuda", torch.cuda.current_device())
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print(f"GPU: {gpu}")
    res = dict(gpu=gpu, cases=[])
    for V, S in ((46, 512), (250, 640)):
        c = case(lib, V, S, a.reps, dev)
        res["cases"].append(c)
        print(f"{V} x {S}^2 ({c['pixels'] / 1e6:.1f} M pixels, {c['finite_pixels'] / 1e6:.1f} M with depth); "
              f"xyz copy {c['copy_GBps']:.0f} GB/s")
        for n in c["normals"]:
            print(f"  normal maps r={n['radius']}: {n['kernel_ms']:.3f} ms (check {n['check_ms']:.3f} ms), "
                  f"{n['pixels_per_s'] / 1e9:.2f} G px/s, {n['min_bytes_GBps']:.0f} GB/s of the 28 B/px floor; "
                  f"undefined {n['undefined']}")
        f = c["fusion"]
        fmt = lambda d: " + ".join(f"{d[k]:.2f}" for k in d)      # noqa: E731
        print(f"  fusion plain {fmt(f['plain'])} ms -> {f['plain_emitted']} points ({f['plain_mean_views']:.2f} views); "
              f"oriented 10 deg {fmt(f['oriented'])} ms -> {f['oriented_emitted']} points ({f['oriented_mean_views']:.2f} views)")
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        json.dump(res, open(a.out, "w"), indent=1)


if __name__ == "__main__":
    main()
