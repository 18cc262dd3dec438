"""GPU: dense depth maps (ldp_depth_maps, DensifyEngine.depth_maps) against the sampled path of the same batch, against their
numpy restatement (tests/depth_oracle.py), through the fix-up, a ring, launch cuts and the pipeline."""
import ctypes as C
import json
import os

import numpy as np
import pytest
import torch

from lichtfeld_densification_plugin_b200 import _native as N
from lichtfeld_densification_plugin_b200 import synth
from lichtfeld_densification_plugin_b200.engine import PathConfig
from tests import depth_oracle as D
from tests import gpu_harness as G
from tests.helpers import oracle_cam

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    from lichtfeld_densification_plugin_b200.engine import DensifyEngine
    return DensifyEngine()


def _batch(engine, scene, inputs, W=None, H=None):
    """``W`` / ``H``: the maps cut to their first columns / rows."""
    dev = engine.device
    W, H = W or scene.W, H or scene.H
    b = engine.new_batch(H, W, scene.w_match, scene.h_match)
    to_dev = lambda m: None if m is None else torch.as_tensor(np.ascontiguousarray(m), dtype=torch.uint8).to(dev)
    for inp in inputs:
        nb = inp["nbr_indices"]
        cert = inp["cert"][:, :H, :W].contiguous().to(dev)
        warp = inp["warp"][:, :H, :W, :].contiguous().to(dev)
        b.add([cert[k] for k in range(len(nb))], [warp[k] for k in range(len(nb))], inp["image"].to(dev),
              scene.cameras[inp["ref_index"]], [scene.cameras[j] for j in nb], rng_stream=inp["ref_index"],
              mask_a=to_dev(inp.get("mask_a")),
              masks_b=[to_dev(m) for m in inp["masks_b"]] if inp.get("masks_b") is not None else None)
    return b


def _cfg(no_filter=False, sampson=5.0, multiview=False, floor=None, M=6000) -> PathConfig:
    p = PathConfig(matches_per_ref=M, no_filter=no_filter, sampson_thresh=sampson, multiview=multiview)
    p.certainty_floor = floor
    return p


def _host(dm):
    return {k: (getattr(dm, k).cpu().numpy() if getattr(dm, k) is not None else None) for k in ("depth", "err", "xyz", "flags", "kept")}


def _z_ref(P1, X):
    """row 3 of P1 on (X, 1) with the kernels' FMA order, emulated in f64 (within an ulp of the f32 FMA chain)."""
    acc = (X[:, 0].astype(np.float64) * np.float64(P1[2, 0])).astype(np.float32)
    for j in (1, 2):
        acc = (X[:, j].astype(np.float64) * np.float64(P1[2, j]) + acc).astype(np.float32)
    return (np.float64(P1[2, 3]) + acc).astype(np.float32)


def _cross_path(engine, scene, inputs, cfg, W=None, H=None, min_cert=0.2, tag=""):
    b = _batch(engine, scene, inputs, W, H)
    out = engine.prepare(b, cfg, taps=True).launch()
    dm = _host(engine.depth_maps(b, cfg, min_cert, want_err=True, want_xyz=True, want_flags=True))
    torch.cuda.synchronize()
    off = out.ref_offset.cpu().numpy()
    S = out.n_samples.cpu().numpy()
    assert (out.status.cpu().numpy() == 0).all(), tag
    n_cmp = n_kept = z_exact = 0
    for r, inp in enumerate(inputs):
        sel = out.sel_idx[r, :S[r]].cpu().numpy().astype(np.int64)
        sf = out.sample_flags[r, :S[r]].cpu().numpy().astype(np.int64)
        taps = out.sample_xyzerr[r, :S[r]].cpu().numpy()
        f = dm["flags"][r].reshape(-1)[sel].astype(np.int64)
        cand = (f & 1) == 1
        assert S[r] > 0 and cand.mean() > 0.5, (tag, r)
        assert np.array_equal((f[cand] >> 4), sf[cand] >> 2), (tag, r)           # winner (no repeated neighbour here)
        assert np.array_equal((f[cand] >> 1) & 1, (sf[cand] >> 1) & 1), (tag, r)
        assert np.array_equal((f[cand] >> 2) & 1, sf[cand] & 1), (tag, r)
        err = dm["err"][r].reshape(-1)[sel]
        xyz = dm["xyz"][r].reshape(-1, 3)[sel]
        depth = dm["depth"][r].reshape(-1)[sel]
        good = cand & (((sf >> 1) & 1) == 1)
        kept = cand & ((sf & 1) == 1)
        ref_xyz, ref_err = taps[:, :3].copy(), taps[:, 3].copy()
        if cfg.multiview:                         # kept points: the packed cloud's (refined) values, in pack order
            order = G.expected_pack_order(sf)
            ref_xyz[order] = out.xyz[off[r]:off[r + 1]].cpu().numpy()
            ref_err[order] = out.err[off[r]:off[r + 1]].cpu().numpy()
        assert err[good].tobytes() == ref_err[good].tobytes(), (tag, r)
        assert np.isnan(err[cand & ~good]).all()
        assert xyz[kept].tobytes() == ref_xyz[kept].tobytes(), (tag, r)
        assert np.isnan(depth[cand & ~kept]).all() and np.isnan(xyz[cand & ~kept]).all()
        P1 = scene.cameras[inp["ref_index"]].P.astype(np.float32)
        z = _z_ref(P1, xyz[kept])
        dz = np.abs(depth[kept].view(np.int32).astype(np.int64) - z.view(np.int32).astype(np.int64))
        assert (dz <= 1).all(), (tag, r)
        z_exact += int((dz == 0).sum())
        assert int(dm["kept"][r]) == int(((dm["flags"][r] >> 2) & 1).sum())
        n_cmp += int(cand.sum())
        n_kept += int(kept.sum())
    print(f"[cross-path] {tag}: {n_cmp} sampled candidates, {n_kept} kept, depths bit-equal to the f64 emulation {z_exact}")
    return dm


CASES = ["pinhole", "lens", "raw_masks", "no_sampson", "no_filter", "mv_nn2", "mv_nn4", "mv_nn8", "narrow"]


@pytest.mark.parametrize("case", CASES)
def test_cross_path_identity(engine, case):
    nn = {"mv_nn2": 2, "mv_nn8": 8}.get(case, 4)
    lens = None
    if case == "lens":
        OPENCV = ("OPENCV", [-0.12, 0.03, 4e-4, -3e-4])
        FISHEYE = ("OPENCV_FISHEYE", [0.05, -0.01, 0.003, -0.0005])
        lens = [[OPENCV, None, FISHEYE][v % 3] for v in range(24)]
    scene = synth.make_scene(24, "fast", ref_fraction=0.125, nn=nn, lens=lens)
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family="R", seed=21) for rp in range(scene.n_refs)]
    # narrow: a 40 x 64 map (coverage tiles one pixel wide; the sampler takes at most 4096 of them).  Its 2560 pixels, less
    # the zero-weight border, hold fewer than int(0.85 * 6000) positive weights, which the reference rejects (status
    # LDP_REF_FEWER_NONZERO, no samples): M = 1000 draws 850 of them
    cfg = _cfg(no_filter=case == "no_filter", sampson=0.0 if case == "no_sampson" else 5.0, multiview=case.startswith("mv"),
               M=1000 if case == "narrow" else 6000)
    if case == "raw_masks":
        cfg.certainty_floor = 0.3
        rs = np.random.RandomState(9)
        for inp in inputs:
            inp["mask_a"] = (rs.random_sample((64, 64)) > 0.1).astype(np.uint8)
            inp["masks_b"] = [(rs.random_sample((64, 64)) > 0.2).astype(np.uint8) if k % 2 else None for k in range(nn)]
    _cross_path(engine, scene, inputs, cfg, W=40 if case == "narrow" else None, H=64 if case == "narrow" else None,
                min_cert=0.3 if case == "raw_masks" else 0.2, tag=case)


def test_maps_vs_oracle(engine):
    scene = synth.make_scene(12, "turbo", ref_fraction=0.17, nn=3)
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family="R", seed=5) for rp in range(scene.n_refs)]
    cfg = _cfg()
    ocfg = G.oracle_cfg(dict(M=6000, no_filter=False, wm=scene.w_match, hm=scene.h_match))
    dm = _host(engine.depth_maps(_batch(engine, scene, inputs), cfg, 0.3, want_err=True, want_flags=True))
    total = flips = 0
    rels = []
    for r, inp in enumerate(inputs):
        nb = inp["nbr_indices"]
        o = D.depth_maps([inp["cert"][k] for k in range(len(nb))], [inp["warp"][k] for k in range(len(nb))],
                         oracle_cam(scene.cameras[inp["ref_index"]]), [oracle_cam(scene.cameras[j]) for j in nb], ocfg, 0.3)
        f = dm["flags"][r].reshape(-1).astype(np.int64)
        assert np.array_equal((f & 1) == 1, o.cand), r
        assert np.array_equal(f[o.cand] >> 4, o.winner[o.cand]), r
        keep = ((f >> 2) & 1) == 1
        bad = keep != o.keep
        near = bad & (o.margin < 1e-5)                  # admitted: a quantity within 1e-5 (relative) of its threshold
        for i in np.nonzero(bad)[0][:10]:
            print(f"   flip ref{r} pixel {int(i)}: gpu keep {int(keep[i])}, oracle {int(o.keep[i])}, margin {o.margin[i]:.2e}")
        assert not (bad & ~near).any(), (r, int((bad & ~near).sum()))
        both = keep & o.keep
        d = dm["depth"][r].reshape(-1)[both].astype(np.float64)
        rels.append(np.abs(d - o.depth[both]) / np.abs(o.depth[both]))
        flips += int(bad.sum())
        total += int(both.sum())
    rel = np.concatenate(rels)
    print(f"[oracle] kept by both {total}, admitted flips {flips}; depth relative difference median {np.median(rel):.2e}, "
          f"share within 2e-7 {np.mean(rel <= 2e-7):.5f}, max {rel.max():.2e}")
    assert flips <= max(3, total // 10000)
    assert np.mean(rel <= 2e-7) > 0.999 and rel.max() < 1e-4


@pytest.mark.parametrize("multiview", [False, True])
def test_forced_fixup(engine, multiview):
    """ldp_debug_force_fixup sends every 7th pixel (and every 5th kept pixel's multi-view solve) to the fix-up, which redoes it
    with Jacobi: every other pixel is bit-identical to the same call without it, and the forced ones keep their verdicts
    (except within 1e-5 of a threshold) and their depths to within the two solvers' difference."""
    scene = synth.make_scene(24, "fast", ref_fraction=0.125, nn=4)
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family="R", seed=31) for rp in range(scene.n_refs)]
    cfg = _cfg(multiview=multiview)
    b = _batch(engine, scene, inputs)
    plain = _host(engine.depth_maps(b, cfg, 0.2, want_err=True, want_xyz=True, want_flags=True))
    n_plain = engine.depth_fixups(len(inputs)).sum()
    engine.lib.ldp_debug_force_fixup(7, 5)
    try:
        forced = _host(engine.depth_maps(b, cfg, 0.2, want_err=True, want_xyz=True, want_flags=True))
        n_forced = engine.depth_fixups(len(inputs))
    finally:
        engine.lib.ldp_debug_force_fixup(0, 0)
    HW = scene.H * scene.W
    idx = np.arange(HW)
    kept_plain = ((plain["flags"] >> 2) & 1).reshape(len(inputs), -1)
    touched = (idx % 7 == 0)[None, :] | ((idx % 5 == 0)[None, :] & (kept_plain == 1) & multiview)
    for key in ("depth", "err", "flags"):
        a, c = plain[key].reshape(len(inputs), HW, -1), forced[key].reshape(len(inputs), HW, -1)
        assert a[~touched].tobytes() == c[~touched].tobytes(), key
    same = plain["flags"].reshape(len(inputs), -1)[touched] == forced["flags"].reshape(len(inputs), -1)[touched]
    assert same.mean() > 0.999
    both = ((plain["flags"] & forced["flags"]) >> 2 & 1).reshape(len(inputs), -1).astype(bool) & touched
    da, dc = plain["depth"].reshape(len(inputs), -1)[both], forced["depth"].reshape(len(inputs), -1)[both]
    rel = np.abs(da.astype(np.float64) - dc) / np.abs(da)
    print(f"[fix-up] multiview={multiview}: entries without forcing {int(n_plain)}, forced {int(n_forced.sum())} "
          f"(per view {n_forced.tolist()}); forced pixels with the same flags {same.mean():.5f}, depth rel diff max {rel.max():.2e}")
    assert int(n_forced.sum()) >= (idx % 7 == 0).sum() * 0.5 * len(inputs)
    assert rel.max() < 1e-4
    assert np.array_equal(plain["kept"], ((plain["flags"] >> 2) & 1).reshape(len(inputs), -1).sum(1))
    assert np.array_equal(forced["kept"], ((forced["flags"] >> 2) & 1).reshape(len(inputs), -1).sum(1))


def test_ring_and_cuts_are_byte_identical(engine):
    from lichtfeld_densification_plugin_b200.engine import DensifyRing
    scene = synth.make_scene(24, "fast", ref_fraction=0.5, nn=4)
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family="R", seed=12) for rp in range(scene.n_refs)]
    cfg = _cfg(multiview=True)
    whole = _host(engine.depth_maps(_batch(engine, scene, inputs), cfg, 0.4, want_err=True, want_flags=True))
    ring = DensifyRing(engine.device, depth=3)
    for cut in (1, 5):
        groups = [list(range(a, min(a + cut, len(inputs)))) for a in range(0, len(inputs), cut)]
        outs = [ring.submit_depth_maps(_batch(ring.engines[ring.slot()], scene, [inputs[i] for i in g]), cfg, 0.4,
                                       want_err=True, want_flags=True) for g in groups]
        ring.synchronize()
        for g, o in zip(groups, outs):
            h = _host(o)
            for key in ("depth", "err", "flags", "kept"):
                assert h[key].tobytes() == whole[key][g].tobytes(), (cut, key)


def test_pipeline_writes_the_maps(engine, tmp_path):
    from lichtfeld_densification_plugin_b200.core import pipeline as P
    from lichtfeld_densification_plugin_b200.core.config import DensePipelineConfig
    scene = synth.make_scene(24, "turbo", ref_fraction=0.5, nn=4)
    cams = scene.cameras
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family="R", seed=12) for rp in range(scene.n_refs)]

    def match_source(rp):
        inp = inputs[rp]
        ri, nb = inp["ref_index"], inp["nbr_indices"]
        packed = P._PackedReferenceBatch(ref_id=cams[ri].uid, ref_path="", imA_np=inp["image"].numpy(), maskA_np=None,
                                         wA_cam=cams[ri].width, hA_cam=cams[ri].height, nn_ids=[cams[j].uid for j in nb],
                                         nn_masks=[None] * len(nb), nn_arrays=[None] * len(nb))
        return P._MatchedReference(packed=packed, warp_list_cpu=[inp["warp"][k] for k in range(len(nb))],
                                   cert_list_cpu=[inp["cert"][k] for k in range(len(nb))], pair_index_by_nbr={}, image_by_nbr={})
    refs = list(range(scene.n_refs))
    ddir = tmp_path / "depth"
    kw = dict(output_path=str(tmp_path / "dense.ply"), matches_per_ref=4000, refs_per_launch=4)
    res = P.run_dense_pipeline(cams, refs, None, DensePipelineConfig(depth_dir=str(ddir), depth_min_certainty=0.4, **kw),
                               match_source=match_source, w_match=scene.w_match, h_match=scene.h_match)
    assert res.depth_paths is not None and len(res.depth_paths) == scene.n_refs
    index = json.load(open(ddir / "depth_maps.json"))
    assert len(index["maps"]) == scene.n_refs
    dm = _host(engine.depth_maps(_batch(engine, scene, inputs), _cfg(), 0.4))
    for e in index["maps"]:
        r = [inp["ref_index"] for inp in inputs].index([c.uid for c in cams].index(e["camera_uid"]))
        a = np.load(ddir / e["file"])
        assert (e["H"], e["W"], e["w_match"], e["h_match"]) == (scene.H, scene.W, scene.w_match, scene.h_match)
        assert (e["width"], e["height"]) == (cams[inputs[r]["ref_index"]].width, cams[inputs[r]["ref_index"]].height)
        assert a.dtype == np.float32 and a.tobytes() == dm["depth"][r].tobytes(), e["file"]
        assert res.depth_paths[e["camera_uid"]] == str(ddir / e["file"])
    before = sorted(str(p) for p in tmp_path.rglob("*.npy")) + sorted(str(p) for p in tmp_path.rglob("*.json"))
    off = P.run_dense_pipeline(cams, refs, None, DensePipelineConfig(**kw), match_source=match_source,
                               w_match=scene.w_match, h_match=scene.h_match)
    assert off.depth_paths is None
    assert sorted(str(p) for p in tmp_path.rglob("*.npy")) + sorted(str(p) for p in tmp_path.rglob("*.json")) == before
    assert off.xyz.tobytes() == res.xyz.tobytes()


def test_edge_cases(engine):
    scene = synth.make_scene(12, "turbo", ref_fraction=0.17, nn=2)
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family="R", seed=2) for rp in range(scene.n_refs)]
    b = _batch(engine, scene, inputs)
    for bad in (0.0, -1.0, 1.01, float("nan")):
        with pytest.raises(ValueError):
            engine.depth_maps(b, _cfg(), bad)
    # the C entry point's own checks: min_certainty, a workspace one byte short
    params = engine._params(b, _cfg(), False, N.LDP_RNG_PHILOX, 0)
    need = C.c_size_t(0)
    N.check(engine.lib.ldp_depth_workspace_bytes(C.byref(params), C.byref(need)), "ldp_depth_workspace_bytes")
    descs = engine.upload_descs(b)
    R, HW = len(inputs), scene.H * scene.W
    depth = torch.empty((R, HW), dtype=torch.float32, device=engine.device)
    kept = torch.empty((R,), dtype=torch.int64, device=engine.device)
    ws = torch.empty((int(need.value),), dtype=torch.uint8, device=engine.device)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    call = lambda mc, n: engine.lib.ldp_depth_maps(C.byref(params), C.c_void_p(descs.data_ptr()), mc, C.c_void_p(depth.data_ptr()),
                                                   None, None, None, C.c_void_p(kept.data_ptr()), C.c_void_p(ws.data_ptr()),
                                                   C.c_size_t(n), st)
    assert call(0.0, ws.numel()) == -1 and call(1.5, ws.numel()) == -1
    assert call(0.5, int(need.value) - 257) == -3                  # LDP_ERR_WORKSPACE (the 256 slack is for alignment)
    assert call(0.5, ws.numel()) == 0
    torch.cuda.synchronize()
    # an empty batch; a view without neighbours; NaN warps
    e = engine.depth_maps(engine.new_batch(scene.H, scene.W, scene.w_match, scene.h_match), _cfg(), 0.5)
    assert e.depth.shape == (0, scene.H, scene.W)
    nan_in = [dict(inp) for inp in inputs]
    w = nan_in[0]["warp"].clone()
    w[:, :40] = float("nan")
    nan_in[0]["warp"] = w
    nan_in.append(dict(inputs[0], nbr_indices=[], cert=inputs[0]["cert"][:0], warp=inputs[0]["warp"][:0]))
    h = _host(engine.depth_maps(_batch(engine, scene, nan_in), _cfg(), 0.2, want_err=True, want_flags=True))
    f0 = h["flags"][0][:40]
    assert ((f0 & 1) == 1).all() and ((f0 >> 2) & 1 == 0).all() and np.isnan(h["depth"][0][:40]).all()
    assert (h["flags"][-1] == 0).all() and np.isnan(h["depth"][-1]).all() and h["kept"][-1] == 0
    assert h["kept"][0] > 0
