"""The fixed list of launches that tests/test_gpu_reach.py runs once per kernel switch (DESIGN §5.1).

The switches are environment variables read once per process, so each setting runs in a child process of its own:

    python -m tests.reach_child OUT.npz

runs every case of ``CASES`` at whatever switches the environment holds and writes every output array, bit for bit, to
OUT.npz, with the launch count, the fix-up worklist and the last cluster size of each case under ``meta``.  The parent
runs the same ``run_cases`` in its own process at the defaults and compares.  Not collected by pytest (no test_ prefix).
"""
from __future__ import annotations

import ctypes as C
import json
import sys
from typing import Dict, Tuple

import numpy as np
import torch

from lichtfeld_densification_plugin_b200 import _native as N
from lichtfeld_densification_plugin_b200 import synth
from tests import gpu_harness as G
from tests.helpers import load_golden

OPENCV = ("OPENCV", [-0.12, 0.03, 4e-4, -3e-4])
FISHEYE = ("OPENCV_FISHEYE", [0.05, -0.01, 0.003, -0.0005])

# case -> does the fused front kernel (LDP_FRONT=1) apply to it?  It needs W % 4 == 0, tiles wider than a pixel,
# nn_max <= 8, no warped neighbour masks, the filters on, and at most 3 tiles of 2048 pixels per resident CTA
# (ldp_api.cu:make_plan).
CASES = {
    "golden": True,           # small_T_all_bins: 96^2, nn 3, explicit uniforms and weight sum
    "override": True,         # the same with a weight sum 1e-4 above the stored one: the override, not the device sum, normalises
    "lens": True,             # OPENCV + fisheye + pinhole views, 320^2, nn 4
    "raw": False,             # raw planes, reference and warped neighbour masks, nn 5
    "raw_nowarp": True,       # raw planes, reference masks only, nn 3: ldp_front_kernel<true>
    "debug": True,            # collect_debug, nn 4
    "no_filter": False,
    "ragged": False,          # nn 1, 7, 9 and 16 in one launch
    "big": False,             # 1536^2: chunk_shift 8, prep kernel <0, *>, atomic chunk sums
    "multiview": True,        # every 7th two-view and every 5th multi-view solve sent to the fix-up worklist
    "ring": True,             # DensifyRing, depth 3, four launches in flight
}


def _scene(nn, setting="turbo", n_views=24, ref_fraction=0.125, **kw):
    return synth.make_scene(n_views, setting, ref_fraction=ref_fraction, nn=nn, **kw)


def _inputs(scene, fam="T", seed=41, **kw):
    return [synth.synth_ref_inputs(scene, rp, cert_family=fam, seed=seed, **kw) for rp in range(scene.n_refs)]


def _trim(inp, k):
    """The same view with only its first k neighbours."""
    return dict(inp, cert=inp["cert"][:k], warp=inp["warp"][:k], nbr_indices=list(inp["nbr_indices"][:k]))


def _batch(engine, scene, inputs):
    dev = engine.device
    b = engine.new_batch(scene.H, scene.W, scene.w_match, scene.h_match)
    to_dev = lambda m: None if m is None else torch.as_tensor(np.ascontiguousarray(m), dtype=torch.uint8).to(dev)
    for inp in inputs:
        nb = inp["nbr_indices"]
        cert, warp = inp["cert"].to(dev), inp["warp"].to(dev)
        b.add([cert[k] for k in range(len(nb))], [warp[k] for k in range(len(nb))], inp["image"].to(dev),
              scene.cameras[inp["ref_index"]], [scene.cameras[j] for j in nb], rng_stream=inp["ref_index"],
              weight_sum_override=float(inp.get("wsum", 0.0)), mask_a=to_dev(inp.get("mask_a")),
              masks_b=[to_dev(m) for m in inp["masks_b"]] if inp.get("masks_b") is not None else None)
    return b


def _arrays(out, R) -> Dict[str, np.ndarray]:
    """Every output of a launch, as host arrays."""
    torch.cuda.synchronize()
    k = int(out.ref_offset[-1].item())
    d = dict(ref_offset=out.ref_offset, status=out.status, n_samples=out.n_samples, group_count=out.group_count,
             group_order=out.group_order, uniforms_used=out.uniforms_used, rounds=out.rounds, weight_sum=out.weight_sum,
             xyz=out.xyz[:k], rgb=out.rgb[:k], err=out.err[:k])
    for name in ("sel_idx", "sample_flags", "sample_xyzerr", "view_mask"):
        if getattr(out, name) is not None:
            d[name] = getattr(out, name)
    if out.dbg_matches is not None:
        d["dbg_matches"], d["dbg_cert"] = out.dbg_matches[:k], out.dbg_cert[:k]
    if "view_mask" in d:
        d["view_mask"] = d["view_mask"][:k]
    return {n: t.cpu().numpy() for n, t in d.items()}


def _launch(engine, scene, inputs, cfg, uniforms=None, collect_debug=False) -> Tuple[Dict[str, np.ndarray], dict]:
    u = torch.from_numpy(np.ascontiguousarray(uniforms)).to(engine.device) if uniforms is not None else None
    pl = engine.prepare(_batch(engine, scene, inputs), cfg, uniforms=u, collect_debug=collect_debug, taps=True)
    out = pl.launch()
    arrays = _arrays(out, len(inputs))
    fx = (C.c_int32 * 2)()
    N.check(engine.lib.ldp_debug_read_fixups(C.byref(pl.params), C.c_void_p(pl.workspace.data_ptr()), fx), "ldp_debug_read_fixups")
    meta = dict(launches=int(out.launches), fixups=[int(fx[0]), int(fx[1])], cluster=int(engine.lib.ldp_debug_last_cluster()))
    return arrays, meta


def run_case(engine, name: str) -> Tuple[Dict[str, np.ndarray], dict]:
    if name in ("golden", "override"):
        c, scene, inp, z = load_golden("small_T_all_bins")
        U = np.random.RandomState(int(z["mt_seed"])).random_sample(3 * c["M"] + 64)[None, :]
        wsum = float(z["weight_sum"]) * (1.0 if name == "golden" else 1.0 + 1e-4)
        return _launch(engine, scene, [dict(inp, wsum=wsum)], G.path_cfg(c), U, collect_debug=True)
    if name == "lens":
        scene = _scene(4, lens=[[OPENCV, None, FISHEYE][v % 3] for v in range(24)])
        return _launch(engine, scene, _inputs(scene), G.path_cfg(dict(M=6000, no_filter=False), seed=2))
    if name in ("raw", "raw_nowarp"):
        nn = 5 if name == "raw" else 3
        scene = _scene(nn)
        inputs = _inputs(scene, fam="R", seed=43)
        rs = np.random.RandomState(8)
        hm, wm = scene.h_match, scene.w_match
        for i, inp in enumerate(inputs):
            inp["cert"] = inp["cert"] - 0.1 * torch.rand(inp["cert"].shape, generator=torch.Generator().manual_seed(i))
            inp["mask_a"] = (rs.random_sample((hm, wm)) > 0.15).astype(np.uint8)
            inp["masks_b"] = ([(rs.random_sample((hm, wm)) > 0.2).astype(np.uint8) if k % 2 else None for k in range(nn)]
                              if name == "raw" else None)
        cfg = G.path_cfg(dict(M=6000, no_filter=False), seed=3)
        cfg.certainty_floor = 0.25
        return _launch(engine, scene, inputs, cfg, collect_debug=True)
    if name == "debug":
        scene = _scene(4)
        return _launch(engine, scene, _inputs(scene, fam="R"), G.path_cfg(dict(M=6000, no_filter=False), seed=4), collect_debug=True)
    if name == "no_filter":
        scene = _scene(4)
        return _launch(engine, scene, _inputs(scene), G.path_cfg(dict(M=6000, no_filter=True)), collect_debug=True)
    if name == "ragged":
        scene = _scene(16, n_views=20, ref_fraction=0.2)
        inputs = [_trim(inp, k) for inp, k in zip(_inputs(scene, fam="R"), (1, 7, 9, 16))]
        return _launch(engine, scene, inputs, G.path_cfg(dict(M=6000, no_filter=False), seed=5), collect_debug=True)
    if name == "big":
        scene = _scene(2, n_views=10, ref_fraction=0.1)
        scene.H = scene.W = 1536
        return _launch(engine, scene, _inputs(scene, fam="R"), G.path_cfg(dict(M=10000, no_filter=False), seed=6))
    if name == "multiview":
        scene = _scene(4)
        cfg = G.path_cfg(dict(M=6000, no_filter=False), seed=7)
        cfg.multiview = True
        engine.lib.ldp_debug_force_fixup(7, 5)
        try:
            return _launch(engine, scene, _inputs(scene), cfg)
        finally:
            engine.lib.ldp_debug_force_fixup(0, 0)
    if name == "ring":
        from lichtfeld_densification_plugin_b200.engine import DensifyRing
        scene = _scene(4, n_views=40, ref_fraction=0.2)
        inputs = _inputs(scene, fam="R")
        cfg = G.path_cfg(dict(M=6000, no_filter=False), seed=8)
        ring = DensifyRing(engine.device, depth=3)
        cuts = [(0, 3), (3, 8), (0, 8), (2, 6)]
        outs = [ring.submit(_batch(ring.engines[ring.slot()], scene, inputs[lo:hi]), cfg, taps=True) for lo, hi in cuts]
        for o in outs:
            ring.wait(o)
        arrays = {}
        for i, ((lo, hi), o) in enumerate(zip(cuts, outs)):
            arrays.update({f"{i}.{n}": a for n, a in _arrays(o, hi - lo).items()})
        return arrays, dict(launches=int(outs[-1].launches), fixups=[0, 0], cluster=int(engine.lib.ldp_debug_last_cluster()))
    raise KeyError(name)


def run_cases(engine):
    """{case: (arrays, meta)} for every case of CASES, in order."""
    return {name: run_case(engine, name) for name in CASES}


def main(path: str) -> None:
    from lichtfeld_densification_plugin_b200.engine import DensifyEngine
    engine = DensifyEngine(torch.device("cuda", 0))
    results = run_cases(engine)
    flat = {f"{name}/{k}": a for name, (arrays, _) in results.items() for k, a in arrays.items()}
    flat["meta"] = np.array(json.dumps({name: meta for name, (_, meta) in results.items()}))
    np.savez(path, **flat)


if __name__ == "__main__":
    main(sys.argv[1])
