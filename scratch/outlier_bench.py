"""Cost of statistical outlier removal (ldp_statistical_outliers) on the device, against scipy's cKDTree on the host.

Clouds: a noisy unit sphere plus 1 % floaters at 418 k (one bench step's cloud), 2.3 M (the config-5 cloud) and 10 M points,
and, when given, the kept points of a bench.py run (`bench.py --dump-outputs DIR` writes DIR/xyz.npy).  k = 20 and 64,
std_ratio = 2.  Reported per case: the call time from CUDA events (median of --reps calls after a warm-up call; the call
includes its one host synchronisation), the per-phase split from ldp_profile_*, the share of points whose search left the
finest grid, and cKDTree(workers=-1) build + query in the same process.

    python scratch/outlier_bench.py [--reps 5] [--bench-xyz DIR/xyz.npy] [--out results.json]
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
from lichtfeld_densification_plugin_b200 import build  # noqa: E402
from tests import outlier_oracle as OO  # noqa: E402


def call(lib, xyz, k, bufs):
    ws, kept, m, stats, status = bufs
    st = torch.cuda.current_stream()
    N.check(lib.ldp_statistical_outliers(C.c_void_p(xyz.data_ptr()), int(xyz.shape[0]), k, C.c_double(2.0), C.c_void_p(kept.data_ptr()),
                                         C.c_void_p(m.data_ptr()), C.c_void_p(stats.data_ptr()), C.c_void_p(status.data_ptr()),
                                         C.c_void_p(ws.data_ptr()), C.c_size_t(ws.numel()), C.c_void_p(st.cuda_stream)),
            "ldp_statistical_outliers")


def run_case(lib, name, xyz_np, k, reps):
    n = xyz_np.shape[0]
    xyz = torch.from_numpy(xyz_np).cuda()
    need = C.c_size_t(0)
    N.check(lib.ldp_outlier_workspace_bytes(n, k, C.byref(need)), "ws")
    bufs = (torch.empty((need.value,), dtype=torch.uint8, device="cuda"), torch.empty((n,), dtype=torch.int64, device="cuda"),
            torch.empty((n,), dtype=torch.float64, device="cuda"), torch.empty((3,), dtype=torch.float64, device="cuda"),
            torch.empty((3,), dtype=torch.int32, device="cuda"))
    call(lib, xyz, k, bufs)                                            # warm-up
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        call(lib, xyz, k, bufs)
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    lib.ldp_profile_enable(1)
    call(lib, xyz, k, bufs)
    ms = (C.c_float * 64)()
    cnt = lib.ldp_profile_read(ms, 64)
    split = {lib.ldp_profile_name(i).decode(): round(ms[i], 3) for i in range(cnt)}
    lib.ldp_profile_enable(0)
    status = bufs[4].cpu().numpy()
    t0 = time.perf_counter()
    from scipy.spatial import cKDTree
    tree = cKDTree(xyz_np.astype(np.float64))
    tree.query(xyz_np.astype(np.float64), k=k, workers=-1)
    cpu_s = time.perf_counter() - t0
    r = dict(cloud=name, n=n, k=k, gpu_ms_median=round(float(np.median(times)), 3), gpu_ms_all=[round(t, 3) for t in times],
             split_ms=split, kept=int(status[1]), escalated=int(status[2]), escalated_share=round(float(status[2]) / n, 5),
             ckdtree_s=round(cpu_s, 3), workspace_gb=round(need.value / 1e9, 3))
    print(json.dumps(r), flush=True)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--bench-xyz", default=None)
    ap.add_argument("--sizes", default="418000,2300000,10000000")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    build.build()
    lib = N.load()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print(json.dumps({"gpu": smi, "host_cpus": os.cpu_count()}), flush=True)
    results = []
    clouds = [(f"sphere+1%floaters", OO.sphere_with_floaters(int(s), seed=0)[0]) for s in args.sizes.split(",")]
    if args.bench_xyz and os.path.isfile(args.bench_xyz):
        clouds.append(("bench.py kept points", np.ascontiguousarray(np.load(args.bench_xyz), dtype=np.float32)))
    for name, xyz in clouds:
        for k in (20, 64):
            results.append(run_case(lib, name, xyz, k, args.reps))
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"gpu": smi, "results": results}, f, indent=1)


if __name__ == "__main__":
    main()
