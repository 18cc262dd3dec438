"""Cost of the cross-view depth consistency check (ldp_depth_consistency) at three sizes:

* one bench step's kept cloud (~416 k points) against its 46 maps at 512^2;
* 2.3 M points against 250 maps at 640^2 (config 5's reference views);
* 10 M points against 250 maps at 640^2.

The maps are the analytic depth of the sphere of synth.SPHERE_RADIUS seen by orbit cameras (pinhole), 2 % NaN holes.  The
cloud comes in emission order like the pipeline's: view by view, each view's points at ascending map pixels (the world
point of every k-th finite pixel of its map, moved radially by up to 1 %), owner = that view.  Per size: the kernel's time
(ldp_profile_*, CUDA events around it; median of --reps calls after a warm-up call), the whole call's time (host clock
around check_depth_consistency, which ends in a synchronising read), point-view tests per second, and the bytes the kernel
moves at most (12 + 4 B in and 12 B out per point, one 4-byte map read per test) against a device-to-device copy's
measured rate.  With --oracle, the numpy restatement on the host at the first size, for context.

    python scratch/consistency_bench.py [--reps 5] [--oracle] [--out results.json]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from lichtfeld_densification_plugin_b200 import _native as N  # noqa: E402
from lichtfeld_densification_plugin_b200 import synth  # noqa: E402
from lichtfeld_densification_plugin_b200.engine import DepthViews, depth_map_scales  # noqa: E402
from lichtfeld_densification_plugin_b200.output import check_depth_consistency  # noqa: E402


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


def scene(V, side, n_points, seed=0):
    """(cameras, maps f32 [V, side, side], xyz f32 [n, 3] in emission order, owner int32 [n])"""
    cams = synth.make_orbit_cameras(V)
    rs = np.random.RandomState(seed)
    wm = side
    maps, pts, own = [], [], []
    per_view = -(-n_points // V)
    for v, c in enumerate(cams):
        xs = (np.arange(side) + 0.5) / side * (wm - 1) * (c.width / wm)
        ys = (np.arange(side) + 0.5) / side * (wm - 1) * (c.height / wm)
        u, w = np.meshgrid(xs, ys)
        K = np.asarray(c.K, np.float64)
        ray = np.stack([(u - K[0, 2]) / K[0, 0], (w - K[1, 2]) / K[1, 1], np.ones_like(u)], -1).reshape(-1, 3)
        d = ray @ np.asarray(c.R, np.float64)
        Cc = np.asarray(c.C, np.float64).reshape(3)
        a, b, cc = (d * d).sum(-1), d @ Cc, Cc @ Cc - synth.SPHERE_RADIUS ** 2
        disc = b * b - a * cc
        with np.errstate(invalid="ignore"):
            t = np.where(disc >= 0, (-b - np.sqrt(disc)) / a, np.nan)
        m = t.astype(np.float32)
        m[rs.random_sample(m.shape) < 0.02] = np.nan
        maps.append(m.reshape(side, side))
        fin = np.nonzero(np.isfinite(t))[0]
        sel = fin[np.linspace(0, fin.size - 1, min(per_view, fin.size)).astype(np.int64)]
        X = (Cc + t[sel, None] * d[sel]) * rs.uniform(0.99, 1.01, size=(sel.size, 1))
        pts.append(X.astype(np.float32))
        own.append(np.full(sel.size, v, np.int32))
    return cams, np.stack(maps), np.concatenate(pts)[:n_points], np.concatenate(own)[:n_points]


def run(dev, V, side, n, reps, oracle):
    cams, maps, xyz, owner = scene(V, side, n)
    views = DepthViews(side, side, side, side, dev)
    for m, c in zip(maps, cams):
        views.add(m, c)
    x = torch.from_numpy(xyz).to(dev)
    o = torch.from_numpy(owner).to(dev)
    lib = N.load()
    res = check_depth_consistency(x, views, owner=o)                   # warm-up
    torch.cuda.synchronize()
    buf = (C.c_float * 8)()
    kt, ct = [], []
    for _ in range(reps):
        lib.ldp_profile_enable(1)
        t0 = time.perf_counter()
        res = check_depth_consistency(x, views, owner=o)
        ct.append(time.perf_counter() - t0)
        k = lib.ldp_profile_read(buf, 8)
        names = [lib.ldp_profile_name(i).decode() for i in range(k)]
        kt.append(buf[names.index("ldp_consistency_kernel")])
        lib.ldp_profile_enable(0)
    nc = res.n_consistent.cpu().numpy()
    nv = res.n_violations.cpu().numpy()
    tests = n * (V - 1)
    t = float(np.median(kt)) / 1e3
    nbytes = n * 28 + 4 * tests
    out = dict(V=V, side=side, n=n, kernel_ms=float(np.median(kt)), call_ms=1e3 * float(np.median(ct)), tests=tests,
               tests_per_s=tests / t, bytes_at_most=nbytes, bytes_per_s=nbytes / t, kept=int(res.kept_idx.numel()),
               mean_consistent=float(nc.mean()), share_violated=float((nv > 0).mean()))
    if oracle:
        from tests import consistency_oracle as CO
        P = np.stack([np.asarray(c.P, np.float32).reshape(12) for c in cams])
        S = np.array([depth_map_scales(c.width, c.height, side, side, side, side) for c in cams])
        t0 = time.perf_counter()
        ores = CO.check(xyz, maps, P, S, owner=owner)
        out["oracle_s"] = time.perf_counter() - t0
        out["oracle_equal"] = bool(np.array_equal(ores.n_consistent, nc) and np.array_equal(ores.n_violations, nv))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--oracle", action="store_true")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    dev = torch.device("cuda")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    peak = copy_rate(dev)
    res = dict(gpu=gpu, copy_bytes_per_s=peak, host_cores=os.cpu_count(), cases=[])
    print(f"GPU: {gpu}; device copy {peak / 1e12:.2f} TB/s; host cores {os.cpu_count()}")
    for i, (V, side, n) in enumerate(((46, 512, 416000), (250, 640, 2300000), (250, 640, 10000000))):
        c = run(dev, V, side, n, a.reps, a.oracle and i == 0)
        c["share_of_copy_rate"] = c["bytes_per_s"] / peak
        res["cases"].append(c)
        extra = f"; numpy oracle {c['oracle_s']:.2f} s (equal {c['oracle_equal']})" if "oracle_s" in c else ""
        print(f"{n} points x {V} maps at {side}^2: kernel {c['kernel_ms']:.3f} ms, call {c['call_ms']:.3f} ms; "
              f"{c['tests_per_s'] / 1e9:.1f} G tests/s; <= {c['bytes_at_most'] / 1e9:.2f} GB = {c['bytes_per_s'] / 1e12:.2f} TB/s "
              f"({100 * c['share_of_copy_rate']:.1f} % of the copy); kept {c['kept']}, mean support {c['mean_consistent']:.2f}, "
              f"violated {100 * c['share_violated']:.2f} %{extra}")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        json.dump(res, open(a.out, "w"), indent=1)


if __name__ == "__main__":
    main()
