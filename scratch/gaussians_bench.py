"""Cost of the 3DGS initialisation (output.init_gaussians / ldp_gaussian_init) and of its PLY records
(ldp_pack_gaussian_ply_records) on the device, beside scipy's cKDTree(k + 1) + the numpy formulas on the host.

Clouds: a noisy unit sphere plus 1 % floaters at 418 k, 2.3 M and 10 M points, and, when given, the kept points of a
bench.py run (`bench.py --dump-outputs DIR` writes DIR/xyz.npy and DIR/rgb.npy).  k = 3 (3DGS's).
Reported per case: the init_gaussians call time from CUDA events (median of --reps calls after a warm-up call; the call
includes its two host synchronisations), the per-phase split from ldp_profile_*, the records kernel's time (CUDA events
around --rec-reps launches, sh_degree 3) and its achieved GB/s (bytes written over kernel time), and cKDTree(k + 1,
workers=-1) build + query plus the numpy formulas on the host.

    python scratch/gaussians_bench.py [--reps 5] [--bench-dir DIR] [--out results.json] [--no-host]
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
from lichtfeld_densification_plugin_b200 import build, output  # noqa: E402
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


def host_init(x: np.ndarray, rgb: np.ndarray, k: int) -> float:
    """cKDTree(k + 1, workers=-1) build + query, then dist2, scales, rotations, SH DC and opacity in numpy: seconds."""
    from scipy.spatial import cKDTree
    t0 = time.perf_counter()
    d, _ = cKDTree(x).query(x, k=k + 1, workers=-1)
    dist2 = np.maximum((d[:, 1:] ** 2).mean(axis=1).astype(np.float32), np.float32(1e-7))
    s = np.log(np.sqrt(dist2))
    np.repeat(s[:, None], 3, axis=1)
    rot = np.zeros((x.shape[0], 4), np.float32)
    rot[:, 0] = 1
    (rgb - np.float32(0.5)) / np.float32(0.28209479177387814)
    np.full(x.shape[0], np.log(0.1 / 0.9), np.float32)
    return time.perf_counter() - t0


def run_case(lib, name, xyz_np, rgb_np, k, reps, rec_reps, host):
    n = xyz_np.shape[0]
    xyz, rgb = torch.from_numpy(xyz_np).cuda(), torch.from_numpy(rgb_np).cuda()
    box = {}

    def init():
        box["g"] = output.init_gaussians(xyz, rgb, nb_neighbors=k)
    med, all_ms, split = timed(lib, init, reps)
    g = box["g"]
    st = torch.cuda.current_stream()
    size = output.gaussian_record_bytes(3)
    rec = torch.empty((n * size,), dtype=torch.uint8, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr())          # noqa: E731

    def records():
        N.check(lib.ldp_pack_gaussian_ply_records(p(xyz), C.c_void_p(0), p(g.sh_dc), p(g.opacity), p(g.scales), p(g.rotations),
                                                  n, C.c_void_p(0), 3, p(rec), C.c_void_p(st.cuda_stream)),
                "ldp_pack_gaussian_ply_records")
    records()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(rec_reps):
        records()
    b.record()
    b.synchronize()
    rec_ms = a.elapsed_time(b) / rec_reps
    r = dict(cloud=name, n=n, k=k, init_ms_median=round(med, 3), init_ms_all=all_ms, init_split_ms=split,
             records_ms=round(rec_ms, 4), records_bytes=n * size, records_gb_s=round(n * size / (rec_ms * 1e-3) / 1e9, 1),
             host_ckdtree_numpy_s=round(host_init(xyz_np, rgb_np, k), 3) if host else None)
    print(json.dumps(r), flush=True)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--rec-reps", type=int, default=20)
    ap.add_argument("--bench-dir", default=None)
    ap.add_argument("--sizes", default="418000,2300000,10000000")
    ap.add_argument("--k", type=int, default=3)
    ap.add_argument("--no-host", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    build.build()
    lib = N.load()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print(json.dumps({"gpu": smi, "host_cpus": os.cpu_count()}), flush=True)
    rng = np.random.default_rng(0)
    clouds = []
    for s in args.sizes.split(","):
        x = OO.sphere_with_floaters(int(s), seed=0)[0]
        clouds.append(("sphere+1%floaters", x, rng.random(x.shape).astype(np.float32)))
    if args.bench_dir and os.path.isfile(os.path.join(args.bench_dir, "xyz.npy")):
        x = np.ascontiguousarray(np.load(os.path.join(args.bench_dir, "xyz.npy")), dtype=np.float32).reshape(-1, 3)
        rp = os.path.join(args.bench_dir, "rgb.npy")
        c = np.ascontiguousarray(np.load(rp), dtype=np.float32).reshape(-1, 3) if os.path.isfile(rp) else rng.random(x.shape)
        clouds.append(("bench.py kept points", x, np.ascontiguousarray(c, dtype=np.float32)))
    results = [run_case(lib, name, x, c, args.k, args.reps, args.rec_reps, not args.no_host) for name, x, c in clouds]
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"gpu": smi, "results": results}, f, indent=1)


if __name__ == "__main__":
    main()
