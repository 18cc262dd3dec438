"""Cost of oriented normals (ldp_estimate_normals) on the device, beside ldp_statistical_outliers at the same k (the same
k-NN search without neighbour indices) and scipy's cKDTree + batched numpy.linalg.eigh on the host.

Clouds: the shapes of DESIGN §4.5, a noisy unit sphere plus 1 % floaters at 418 k, 2.3 M and 10 M points, and, when
given, the kept points of a bench.py run (`bench.py --dump-outputs DIR` writes DIR/xyz.npy).  k = 8, 20 and 64.
Reported per case: the call time from CUDA events (median of --reps calls after a warm-up call; the call includes its one
host synchronisation), the per-phase split from ldp_profile_* (the k-NN + normal kernel's own time), the outlier call's
time and split in the same process, and cKDTree(workers=-1) build + query + covariance + eigh on the host.

    python scratch/normals_bench.py [--reps 5] [--bench-xyz DIR/xyz.npy] [--out results.json] [--no-host]
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


def timed(lib, fn, reps):
    fn()                                                               # warm-up
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    lib.ldp_profile_enable(1)
    fn()
    ms = (C.c_float * 64)()
    cnt = lib.ldp_profile_read(ms, 64)
    split = {lib.ldp_profile_name(i).decode(): round(ms[i], 3) for i in range(cnt)}
    lib.ldp_profile_enable(0)
    return float(np.median(times)), [round(t, 3) for t in times], split


def host_normals(x: np.ndarray, k: int) -> float:
    """cKDTree(workers=-1) build + query, then f64 covariances and batched eigh, in chunks: seconds."""
    from scipy.spatial import cKDTree
    t0 = time.perf_counter()
    xd = x.astype(np.float64)
    _, idx = cKDTree(xd).query(xd, k=k, workers=-1)
    for a in range(0, xd.shape[0], 1 << 18):
        p = xd[idx[a:a + (1 << 18)]]
        d = p - p.mean(axis=1, keepdims=True)
        np.linalg.eigh(np.einsum("nki,nkj->nij", d, d) / k)
    return time.perf_counter() - t0


def run_case(lib, name, xyz_np, k, reps, host):
    n = xyz_np.shape[0]
    xyz = torch.from_numpy(xyz_np).cuda()
    st = torch.cuda.current_stream()
    need = C.c_size_t(0)
    N.check(lib.ldp_normals_workspace_bytes(n, k, C.byref(need)), "ws")
    ws = torch.empty((need.value,), dtype=torch.uint8, device="cuda")
    nrm = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    curv = torch.empty((n,), dtype=torch.float32, device="cuda")
    status = torch.empty((3,), dtype=torch.int32, device="cuda")

    def normals():
        N.check(lib.ldp_estimate_normals(C.c_void_p(xyz.data_ptr()), n, k, C.c_void_p(0), 0, C.c_void_p(0),
                                         C.c_void_p(nrm.data_ptr()), C.c_void_p(curv.data_ptr()), C.c_void_p(0),
                                         C.c_void_p(status.data_ptr()), C.c_void_p(ws.data_ptr()), C.c_size_t(ws.numel()),
                                         C.c_void_p(st.cuda_stream)), "ldp_estimate_normals")
    med, all_ms, split = timed(lib, normals, reps)
    s = status.cpu().numpy()
    del ws
    N.check(lib.ldp_outlier_workspace_bytes(n, k, C.byref(need)), "ws")
    ows = torch.empty((need.value,), dtype=torch.uint8, device="cuda")
    kept = torch.empty((n,), dtype=torch.int64, device="cuda")
    ostatus = torch.empty((3,), dtype=torch.int32, device="cuda")

    def outliers():
        N.check(lib.ldp_statistical_outliers(C.c_void_p(xyz.data_ptr()), n, k, C.c_double(2.0), C.c_void_p(kept.data_ptr()),
                                             C.c_void_p(0), C.c_void_p(0), C.c_void_p(ostatus.data_ptr()),
                                             C.c_void_p(ows.data_ptr()), C.c_size_t(ows.numel()), C.c_void_p(st.cuda_stream)),
                "ldp_statistical_outliers")
    omed, oall, osplit = timed(lib, outliers, reps)
    del ows
    r = dict(cloud=name, n=n, k=k, normals_ms_median=round(med, 3), normals_ms_all=all_ms, normals_split_ms=split,
             undefined=int(s[1]), escalated_share=round(float(s[2]) / n, 5),
             outliers_ms_median=round(omed, 3), outliers_split_ms=osplit,
             host_ckdtree_eigh_s=round(host_normals(xyz_np, k), 3) if host else None)
    print(json.dumps(r), flush=True)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--bench-xyz", default=None)
    ap.add_argument("--sizes", default="418000,2300000,10000000")
    ap.add_argument("--ks", default="8,20,64")
    ap.add_argument("--no-host", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    build.build()
    lib = N.load()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print(json.dumps({"gpu": smi, "host_cpus": os.cpu_count()}), flush=True)
    results = []
    clouds = [("sphere+1%floaters", OO.sphere_with_floaters(int(s), seed=0)[0]) for s in args.sizes.split(",")]
    if args.bench_xyz and os.path.isfile(args.bench_xyz):
        clouds.append(("bench.py kept points", np.ascontiguousarray(np.load(args.bench_xyz), dtype=np.float32)))
    for name, xyz in clouds:
        for k in (int(v) for v in args.ks.split(",")):
            results.append(run_case(lib, name, xyz, k, args.reps, not args.no_host))
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"gpu": smi, "results": results}, f, indent=1)


if __name__ == "__main__":
    main()
