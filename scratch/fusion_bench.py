"""Cost of depth-map fusion: the colour maps (ldp_depth_colors) at the bench shape (46 views, 512^2 maps, nn = 4), and
ldp_fuse_depth_maps on analytic sphere maps at 46 views x 512^2 and at 250 views x 640^2.

Per case: each kernel's time from ldp_profile_* (CUDA events around each kernel), median of --reps calls after a warm-up
call, and the whole call (CUDA events around fuse_depth_maps' enqueue, without its read-back).  Pass 1 (verdict kernel) runs
one point-view test per finite pixel and other view; pass 2 (emit kernel over the views below a pixel, sum kernel over the
views above an emitted one) stops early, so its rate is stated against the same nominal count.  The sphere maps are the
ray-cast depth of synth.SPHERE_RADIUS seen from orbit cameras 4 units out, with 0.1 % depth noise.  The card's name and
power limit are read in the same run.

    python scratch/fusion_bench.py [--reps 5] [--out results.json]
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
from lichtfeld_densification_plugin_b200 import _native as N  # noqa: E402
from lichtfeld_densification_plugin_b200 import synth  # noqa: E402
from lichtfeld_densification_plugin_b200.engine import DensifyEngine, DepthViews, PathConfig  # noqa: E402


def profiled(lib, fn, reps):
    """median ms per kernel name over reps profiled calls of fn (one C call each), after a warm-up call"""
    fn()
    torch.cuda.synchronize()
    buf = (C.c_float * 16)()
    times = {}
    lib.ldp_profile_enable(1)
    for _ in range(reps):
        fn()
        n = lib.ldp_profile_read(buf, 16)
        for i in range(n):
            times.setdefault(lib.ldp_profile_name(i).decode(), []).append(buf[i])
    lib.ldp_profile_enable(0)
    return {k: float(np.median(v)) for k, v in times.items()}


def colour_case(eng, reps):
    scene = synth.make_scene(46, "fast", ref_fraction=1.0, nn=4)
    dev = eng.device
    inputs = [synth.synth_ref_inputs(scene, rp, device=dev, cert_family="R", seed=rp) for rp in range(46)]
    b = eng.new_batch(scene.H, scene.W, scene.w_match, scene.h_match)
    for inp in inputs:
        k = len(inp["nbr_indices"])
        b.add([inp["cert"][q] for q in range(k)], [inp["warp"][q] for q in range(k)], inp["image"], scene.cameras[inp["ref_index"]],
              [scene.cameras[j] for j in inp["nbr_indices"]])
    cfg = PathConfig()
    dm = eng.depth_maps(b, cfg, 0.5, want_flags=True, want_rgb=True)
    params = eng._params(b, cfg, False, N.LDP_RNG_PHILOX, 0)
    descs = eng.upload_descs(b)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    call = lambda: N.check(eng.lib.ldp_depth_colors(C.byref(params), C.c_void_p(descs.data_ptr()), C.c_void_p(dm.flags.data_ptr()),  # noqa: E731
                                                    C.c_void_p(dm.rgb.data_ptr()), st), "ldp_depth_colors")
    t = profiled(eng.lib, call, reps)["ldp_depth_color_kernel"]
    px = 46 * scene.H * scene.W
    return dict(H=scene.H, W=scene.W, n_refs=46, pixels=px, kept=int(dm.kept.sum()), colour_kernel_ms=t, pixels_per_s=px / (t / 1e3))


def sphere_views(V, S, dev, noise=1e-3, seed=0):
    cams = synth.make_orbit_cameras(V)
    g = torch.Generator(device=dev).manual_seed(seed)
    views = DepthViews(S, S, S, S, dev)
    for c in cams:
        xs = (torch.arange(S, device=dev, dtype=torch.float64) + 0.5) / S * (S - 1) * (c.width / S)
        ys = (torch.arange(S, device=dev, dtype=torch.float64) + 0.5) / S * (S - 1) * (c.height / S)
        v, u = torch.meshgrid(ys, xs, indexing="ij")
        K = torch.as_tensor(np.asarray(c.K, np.float64), device=dev)
        R = torch.as_tensor(np.asarray(c.R, np.float64), device=dev)
        Cc = torch.as_tensor(np.asarray(c.C, np.float64).reshape(3), device=dev)
        t = torch.as_tensor(np.asarray(c.t, np.float64).reshape(3), device=dev)
        ray = torch.stack([(u - K[0, 2]) / K[0, 0], (v - K[1, 2]) / K[1, 1], torch.ones_like(u)], -1)
        d = ray @ R
        a, bb, cc = (d * d).sum(-1), d @ Cc, Cc @ Cc - synth.SPHERE_RADIUS ** 2
        disc = bb * bb - a * cc
        z = (-bb - torch.sqrt(disc)) / a
        z = z * (1 + noise * torch.randn(z.shape, generator=g, device=dev, dtype=torch.float64))
        z = torch.where(disc >= 0, z, torch.full_like(z, float("nan")))
        world = ((ray * z[..., None]) - t) @ R
        rgb = torch.rand((S, S, 3), generator=g, device=dev)
        views.add(z.float(), c, xyz=world.float(), rgb=rgb, err=torch.rand((S, S), generator=g, device=dev))
    return views


def fusion_case(lib, V, S, reps, dev):
    from lichtfeld_densification_plugin_b200.output import fuse_depth_maps
    views = sphere_views(V, S, dev)
    finite = int(sum(int(torch.isfinite(m).sum()) for m in views.maps))
    k = profiled(lib, lambda: fuse_depth_maps(views), reps)
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        f = fuse_depth_maps(views)
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    tests = finite * (V - 1)
    p1 = k["ldp_fusion_verdict_kernel"]
    p2 = k["ldp_fusion_emit_kernel"] + k["ldp_fusion_sum_kernel"]
    return dict(V=V, H=S, W=S, finite_pixels=finite, emitted=int(f.source.numel()), mean_views=float(f.n_views.float().mean()),
                verdict_ms=p1, emit_ms=k["ldp_fusion_emit_kernel"], sum_ms=k["ldp_fusion_sum_kernel"], call_ms=float(np.median(ts)),
                pass1_tests_per_s=tests / (p1 / 1e3), pass2_nominal_tests_per_s=tests / (p2 / 1e3))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    eng = DensifyEngine()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print(f"GPU: {gpu}")
    res = dict(gpu=gpu, colour=colour_case(eng, a.reps), fusion=[])
    c = res["colour"]
    print(f"colour maps {c['H']}^2 x {c['n_refs']} views: {c['colour_kernel_ms']:.3f} ms, {c['pixels_per_s'] / 1e9:.1f} G px/s "
          f"({c['kept']} kept)")
    for V, S in ((46, 512), (250, 640)):
        f = fusion_case(eng.lib, V, S, a.reps, eng.device)
        res["fusion"].append(f)
        print(f"fusion {V} x {S}^2: pass 1 {f['verdict_ms']:.2f} ms ({f['pass1_tests_per_s'] / 1e9:.0f} G tests/s), pass 2 emit "
              f"{f['emit_ms']:.2f} + sum {f['sum_ms']:.2f} ms ({f['pass2_nominal_tests_per_s'] / 1e9:.0f} G nominal tests/s), "
              f"call {f['call_ms']:.2f} ms; {f['finite_pixels']} pixels -> {f['emitted']} points, {f['mean_views']:.2f} views each")
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        json.dump(res, open(a.out, "w"), indent=1)


if __name__ == "__main__":
    main()
