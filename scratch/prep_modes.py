"""Dev tool: the shapes whose prep kernel column mode is not CONST/QUAD on the vector path, run through one tree.

    python scratch/prep_modes.py TREE OUT.npz      every output and tap of each shape (Philox and explicit uniforms) to
                                                   OUT.npz, and the prep kernel's time (ldp_profile_read) per shape
    python scratch/prep_modes.py --compare A.npz B.npz     byte-for-byte comparison of two such files

Run the first form once per tree (each in its own process: the package is imported from TREE) and compare."""
import json
import os
import sys
import time

import numpy as np

SHAPES = [(50, 61), (40, 36), (64, 8448), (1001, 1001), (1281, 1279), (8, 327680), (512, 512)]   # 512^2: CONST, unchanged
FIELDS = ("sel_idx", "flags", "xyzerr", "xyz", "rgb", "err", "status", "uniforms_used", "rounds", "weight_sum",
          "group_order", "group_count")


def run(tree: str, out_path: str) -> None:
    sys.path.insert(0, os.path.abspath(tree))
    import ctypes as C
    import torch
    from lichtfeld_densification_plugin_b200 import synth
    from lichtfeld_densification_plugin_b200.engine import DensifyEngine
    from tests import gpu_harness as G
    dev = torch.device("cuda", 0)
    eng = DensifyEngine(dev)
    saved = {}
    for H, W in SHAPES:
        R = 8 if H * W < 2_000_000 else 4
        scene = synth.make_scene(3 * R, "turbo", ref_fraction=1 / 3, nn=4)
        scene.H, scene.W = H, W
        M = min(10000, H * W // 3)
        c = dict(M=M, no_filter=False, wm=scene.w_match, hm=scene.h_match)
        inputs = [synth.synth_ref_inputs(scene, rp, device=dev, cert_family="R", seed=500 + rp) for rp in range(scene.n_refs)]
        U = np.stack([np.random.RandomState(70 + r).random_sample(3 * M + 64) for r in range(len(inputs))])
        for mode, u in (("philox", None), ("explicit", U)):
            g = G.run_gpu(eng, scene, inputs, G.path_cfg(c, seed=3), uniforms=u)
            for f in FIELDS:
                v = getattr(g, f)
                for r, a in enumerate(v if isinstance(v, list) else [v]):
                    saved[f"{H}x{W}/{mode}/{f}/{r}"] = np.ascontiguousarray(a)
        # prep kernel time: CUDA events around each kernel of a launch (ldp_profile_read), mean over 50 launches
        batch = eng.new_batch(H, W, scene.w_match, scene.h_match)
        cams = scene.cameras
        for inp in inputs:
            nn = len(inp["nbr_indices"])
            batch.add([inp["cert"][k] for k in range(nn)], [inp["warp"][k] for k in range(nn)], inp["image"].to(dev),
                      cams[inp["ref_index"]], [cams[j] for j in inp["nbr_indices"]], rng_stream=inp["ref_index"])
        cfg = G.path_cfg(c, seed=3)
        pl = eng.prepare(batch, cfg)
        for _ in range(5):
            pl.launch()
        torch.cuda.synchronize()
        eng.lib.ldp_profile_enable(1)
        buf = (C.c_float * 64)()
        t = {}
        n_prof = 50
        for _ in range(n_prof):
            pl.launch()
            n = eng.lib.ldp_profile_read(buf, 64)
            for k in range(n):
                name = eng.lib.ldp_profile_name(k).decode()
                t[name] = t.get(name, 0.0) + 1e3 * float(buf[k]) / n_prof
        eng.lib.ldp_profile_enable(0)
        print(json.dumps({"tree": tree, "shape": f"{H}x{W}", "views": R, "M": M,
                          "prep_us": round(t["ldp_prep_kernel"], 2), "stream_us": round(t["ldp_stream_kernel"], 2)}), flush=True)
        del inputs, batch, pl
        torch.cuda.empty_cache()
    np.savez(out_path, **saved)


def compare(a_path: str, b_path: str) -> int:
    a, b = np.load(a_path), np.load(b_path)
    bad = sorted(set(a.files) ^ set(b.files))
    bad += [k for k in sorted(set(a.files) & set(b.files)) if a[k].dtype != b[k].dtype or a[k].shape != b[k].shape
            or a[k].tobytes() != b[k].tobytes()]
    shapes = sorted({k.split("/")[0] for k in a.files})
    print(json.dumps({"arrays": len(a.files), "shapes": shapes, "differ": bad[:20], "identical": not bad}))
    return 1 if bad else 0


if __name__ == "__main__":
    if sys.argv[1] == "--compare":
        sys.exit(compare(sys.argv[2], sys.argv[3]))
    t0 = time.time()
    run(sys.argv[1], sys.argv[2])
    print(f"{sys.argv[1]}: {time.time() - t0:.0f} s", file=sys.stderr)
