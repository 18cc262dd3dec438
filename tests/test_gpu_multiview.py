"""GPU: the multi-view refinement (ldp_params.multiview, PathConfig.multiview) against the same launches without it, against
its numpy restatement (tests/multiview_oracle.py) and against the synthetic scenes' ground truth."""
import ctypes as C

import numpy as np
import pytest
import torch

from lichtfeld_densification_plugin_b200 import _native as N
from lichtfeld_densification_plugin_b200 import synth
from lichtfeld_densification_plugin_b200.engine import PathConfig
from oracle import densify_oracle as O
from tests import gpu_harness as G
from tests import lens_oracle as LO
from tests import multiview_oracle as MV
from tests.helpers import oracle_cam

pytestmark = pytest.mark.gpu

MASK_NEAR_PX = 1e-3          # a mask may differ from the oracle's only where a trimming / acceptance error is this close to
                             # reproj_thresh (float32 projections in a different order)


@pytest.fixture(scope="module")
def engine():
    from lichtfeld_densification_plugin_b200.engine import DensifyEngine
    return DensifyEngine()


def _cfg(c: dict, multiview: bool, min_cert: float = 0.5, seed: int = 0) -> PathConfig:
    p = G.path_cfg(c, seed=seed)
    p.multiview, p.multiview_min_certainty = multiview, min_cert
    if "floor" in c:
        p.certainty_floor = c["floor"]
    return p


def _batch(engine, scene, inputs, cams=None):
    cams = cams or scene.cameras
    dev = engine.device
    b = engine.new_batch(scene.H, scene.W, scene.w_match, scene.h_match)
    to_dev = lambda m: None if m is None else torch.as_tensor(np.ascontiguousarray(m), dtype=torch.uint8).to(dev)
    for inp in inputs:
        nb = inp["nbr_indices"]
        cert, warp = inp["cert"].to(dev), inp["warp"].to(dev)
        b.add([cert[k] for k in range(len(nb))], [warp[k] for k in range(len(nb))], inp["image"].to(dev), cams[inp["ref_index"]],
              [cams[j] for j in nb], rng_stream=inp["ref_index"], weight_sum_override=float(inp.get("wsum", 0.0)),
              mask_a=to_dev(inp.get("mask_a")),
              masks_b=[to_dev(m) for m in inp["masks_b"]] if inp.get("masks_b") is not None else None)
    return b


def _run(engine, scene, inputs, cfg, uniforms=None, collect_debug=False, cams=None):
    """One launch; every output as host arrays, per view."""
    u = torch.from_numpy(np.ascontiguousarray(uniforms)).to(engine.device) if uniforms is not None else None
    pl = engine.prepare(_batch(engine, scene, inputs, cams), cfg, uniforms=u, collect_debug=collect_debug, taps=True)
    out = pl.launch()
    torch.cuda.synchronize()
    off = out.ref_offset.cpu().numpy()
    S = out.n_samples.cpu().numpy()
    R = len(inputs)
    per = lambda t: [t[off[r]:off[r + 1]].cpu().numpy() for r in range(R)]
    d = dict(ref_offset=off, status=out.status.cpu().numpy(), group_order=out.group_order.cpu().numpy(),
             group_count=out.group_count.cpu().numpy(),
             sel=[out.sel_idx[r, :S[r]].cpu().numpy() for r in range(R)],
             flags=[out.sample_flags[r, :S[r]].cpu().numpy() for r in range(R)],
             taps=[out.sample_xyzerr[r, :S[r]].cpu().numpy() for r in range(R)],
             xyz=per(out.xyz), rgb=per(out.rgb), err=per(out.err))
    if collect_debug:
        d["dbg_matches"], d["dbg_cert"] = per(out.dbg_matches), per(out.dbg_cert)
    if cfg.multiview:
        d["view_mask"] = per(out.view_mask)
        fx = (C.c_int32 * 2)()           # the launch's fix-up worklist: entries, of which multi-view solves only
        N.check(engine.lib.ldp_debug_read_fixups(C.byref(pl.params), C.c_void_p(pl.workspace.data_ptr()), fx),
                "ldp_debug_read_fixups")
        d["fixups"] = (int(fx[0]), int(fx[1]))
    return d


SAME = ("ref_offset", "status", "group_order", "group_count", "sel", "flags", "taps", "rgb")


def _assert_same_but_points(on, off, R):
    for f in SAME + tuple(f for f in ("dbg_matches", "dbg_cert") if f in off):
        a, b = on[f], off[f]
        if isinstance(a, list):
            for r in range(R):
                assert a[r].tobytes() == b[r].tobytes(), (f, r)
        else:
            assert a.tobytes() == b.tobytes(), f
    moved = 0
    for r in range(R):
        vm = on["view_mask"][r]
        winner = (on["flags"][r][G.expected_pack_order(on["flags"][r])] >> 2).astype(np.int64)
        assert ((vm >> winner) & 1).all()                 # the winner's bit is always set
        single = np.array([bin(int(m)).count("1") == 1 for m in vm], dtype=bool)
        # winner-only points: bit-identical xyz and err
        assert on["xyz"][r][single].tobytes() == off["xyz"][r][single].tobytes(), r
        assert on["err"][r][single].tobytes() == off["err"][r][single].tobytes(), r
        assert (on["err"][r] <= np.float32(0.8)).all()
        moved += int((~single).sum())
    return moved


# ---- 1. on vs off: everything but the points is the same launch ------------------------------------------------------------
@pytest.mark.parametrize("rng,fam,raw", [("philox", "R", False), ("explicit", "T", False), ("philox", "R", True),
                                         ("explicit", "R", True)])
def test_multiview_changes_only_the_points(engine, rng, fam, raw):
    scene = synth.make_scene(24, "fast", ref_fraction=0.25, nn=4)
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family=fam, seed=3) for rp in range(scene.n_refs)]
    c = dict(M=10000, no_filter=False)
    if raw:          # raw matcher planes: the floor and a reference / neighbour mask applied in the kernels
        c["floor"] = 0.3
        rs = np.random.RandomState(9)
        for inp in inputs:
            inp["mask_a"] = (rs.random_sample((64, 64)) > 0.1).astype(np.uint8)
            inp["masks_b"] = [(rs.random_sample((64, 64)) > 0.2).astype(np.uint8) if k % 2 else None for k in range(4)]
    U = None
    if rng == "explicit":
        U = np.stack([np.random.RandomState(50 + r).random_sample(3 * c["M"] + 64) for r in range(len(inputs))])
    off = _run(engine, scene, inputs, _cfg(c, False), U, collect_debug=True)
    on = _run(engine, scene, inputs, _cfg(c, True), U, collect_debug=True)
    moved = _assert_same_but_points(on, off, len(inputs))
    print(f"[on/off] {rng}/{fam}/raw={raw}: {moved} of {sum(x.shape[0] for x in on['xyz'])} points refined")
    assert moved > 0


# ---- 2./3. kernel vs oracle -------------------------------------------------------------------------------------------------
def _vs_oracle(engine, scene, inputs, c, tag, min_cert=0.5, force=None):
    R = len(inputs)
    U = np.stack([np.random.RandomState(700 + r).random_sample(3 * c["M"] + 64) for r in range(R)])
    cams = scene.cameras
    ocfg = G.oracle_cfg(c)
    refs = []
    for r, inp in enumerate(inputs):
        nb = inp["nbr_indices"]
        certs, warps = [inp["cert"][k] for k in range(len(nb))], [inp["warp"][k] for k in range(len(nb))]
        ref_o, nbr_o = oracle_cam(cams[inp["ref_index"]]), [oracle_cam(cams[j]) for j in nb]
        lref, lnb = LO.lens_of(cams[inp["ref_index"]]), [LO.lens_of(cams[j]) for j in nb]
        res = LO.triangulate_ref_lens(certs, warps, inp["image"].numpy(), ref_o, nbr_o, ocfg, lref, lnb, uniforms=U[r])
        mv = MV.refine(res, [x.numpy() for x in certs], [w.numpy() for w in warps], ref_o, nbr_o, ocfg,
                       MV.groups_of([cams[j].uid for j in nb]), min_cert, lref, lnb)
        inp["wsum"] = res.taps.get("s", 0.0)
        refs.append((res, mv))
    g = _run(engine, scene, inputs, _cfg(c, True, min_cert), U)
    if force is not None:
        engine.lib.ldp_debug_force_fixup(*force)
        try:
            g = _run(engine, scene, inputs, _cfg(c, True, min_cert), U)
        finally:
            engine.lib.ldp_debug_force_fixup(0, 0)
    near_total, kept_total, multi = 0, 0, 0
    for r, (res, mv) in enumerate(refs):
        assert np.array_equal(g["sel"][r], res.sel_idx), (tag, r)
        order = G.expected_pack_order(g["flags"][r])
        both = mv.keep[order]                      # kept by the kernel and by the oracle's two-view verdict
        vm, xyz, err = g["view_mask"][r][both], g["xyz"][r][both], g["err"][r][both]
        pos = order[both]
        bad = vm != mv.mask[pos]
        near = bad & (mv.margin[pos] < MASK_NEAR_PX)
        far = bad & ~near
        for i in np.nonzero(bad)[0][:5]:
            print(f"   mask {tag}/ref{r} sample {int(pos[i])}: gpu {int(vm[i]):#x} oracle {int(mv.mask[pos[i]]):#x} "
                  f"margin {mv.margin[pos[i]]:.2e}")
        assert not far.any(), (tag, r, int(far.sum()))
        same = ~bad
        X = mv.xyz[pos[same]].astype(np.float64)
        dx = np.abs(xyz[same].astype(np.float64) - X)
        assert (dx <= G.XYZ_ATOL + G.XYZ_RTOL * np.abs(X)).all(), (tag, r, float(dx.max()))
        de = np.abs(err[same].astype(np.float64) - mv.err[pos[same]])
        assert (de <= G.ERR_ATOL).all(), (tag, r, float(de.max()))
        near_total += int(near.sum())
        kept_total += int(both.sum())
        multi += int(np.array([bin(int(m)).count("1") > 1 for m in vm]).sum())
    print(f"[vs oracle] {tag}: kept {kept_total}, refined {multi}, masks within {MASK_NEAR_PX} px of the threshold {near_total}, "
          f"fix-up entries {g['fixups'][0]} (multi-view solves {g['fixups'][1]})")
    assert near_total <= max(3, kept_total // 500), tag
    assert multi > 0.1 * kept_total, tag
    return g


@pytest.mark.parametrize("case", ["nn2", "nn4", "nn8", "no_sampson", "outliers"])
def test_multiview_vs_oracle(engine, case):
    nn = {"nn2": 2, "nn8": 8}.get(case, 4)
    scene = synth.make_scene(24, "fast", ref_fraction=0.125, nn=nn)
    c = dict(M=10000, no_filter=False, wm=scene.w_match, hm=scene.h_match)
    if case == "no_sampson":
        c["sampson"] = 0.0
    kw = dict(outlier_frac=0.3, noise_sigma=3e-3) if case == "outliers" else {}
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family="T", seed=31, **kw) for rp in range(scene.n_refs)]
    _vs_oracle(engine, scene, inputs, c, case)


def test_multiview_lens_vs_oracle(engine):
    OPENCV = ("OPENCV", [-0.12, 0.03, 4e-4, -3e-4])
    FISHEYE = ("OPENCV_FISHEYE", [0.05, -0.01, 0.003, -0.0005])
    lens = [[OPENCV, None, FISHEYE][v % 3] for v in range(24)]
    scene = synth.make_scene(24, "fast", ref_fraction=0.125, nn=4, lens=lens)
    c = dict(M=10000, no_filter=False, wm=scene.w_match, hm=scene.h_match)
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family="T", seed=31) for rp in range(scene.n_refs)]
    _vs_oracle(engine, scene, inputs, c, "lens")


def test_multiview_fixup_vs_oracle(engine):
    """The fix-up worklist with both kinds of entry, held to the oracle like any other launch: every 7th sample's two-view
    solve and every 5th kept sample's multi-view solve are sent to the fix-up (ldp_debug_force_fixup), which solves them with
    Jacobi - kept two-view fix-ups are refined there, multi-view-only entries redo the refinement from their record."""
    scene = synth.make_scene(24, "fast", ref_fraction=0.125, nn=4)
    c = dict(M=10000, no_filter=False, wm=scene.w_match, hm=scene.h_match)
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family="T", seed=31) for rp in range(scene.n_refs)]
    g = _vs_oracle(engine, scene, inputs, c, "forced fix-up", force=(7, 5))
    n, n_mv = g["fixups"]
    kept_two = sum(int((f[::7] & 1).sum()) for f in g["flags"])      # samples i % 7 == 0: all went through the fix-up
    print(f"[fix-up] entries {n}: multi-view only {n_mv}, two-view {n - n_mv} of which kept {kept_two}")
    assert n - n_mv >= sum(f[::7].size for f in g["flags"])
    assert kept_two > 100 and n_mv > 100
    # against the same launch without forcing: kept set and masks agree except where a Jacobi and an inverse-iteration
    # solve of the same matrix put an error on the other side of a threshold (two-view verdicts of the forced samples)
    plain = _run(engine, scene, inputs, _cfg(c, True), np.stack([np.random.RandomState(700 + r).random_sample(3 * c["M"] + 64)
                                                                  for r in range(len(inputs))]))
    for r in range(len(inputs)):
        same = (g["flags"][r] & 1) == (plain["flags"][r] & 1)
        assert same.mean() > 0.999, r


def test_natural_fixups_are_counted(engine):
    """Without forcing: the worklist of a launch with many gross outliers (reported, not asserted: its size is the data's)."""
    scene = synth.make_scene(24, "fast", ref_fraction=0.25, nn=4)
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family="R", seed=6, outlier_frac=0.3, noise_sigma=3e-3)
              for rp in range(scene.n_refs)]
    g = _run(engine, scene, inputs, _cfg(dict(M=10000, no_filter=False), True))
    print(f"[fix-up] natural, 30 % outliers: entries {g['fixups'][0]}, multi-view only {g['fixups'][1]}")
    assert g["fixups"][0] >= g["fixups"][1] >= 0


# ---- 4. edge cases ----------------------------------------------------------------------------------------------------------
def _scene_inputs(nn, seed=4, n_refs=3, **kw):
    scene = synth.make_scene(24, "fast", ref_fraction=0.125, nn=nn)
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family="R", seed=seed, **kw) for rp in range(n_refs)]
    return scene, inputs


def test_duplicate_low_certainty_and_single_neighbours(engine):
    c = dict(M=10000, no_filter=False)
    scene, inputs = _scene_inputs(4)
    # slot 3 repeats slot 1's neighbour: it may never appear beside slot 1 (one uid counts once)
    dup = [dict(inp, nbr_indices=inp["nbr_indices"][:3] + [inp["nbr_indices"][1]],
                cert=torch.cat([inp["cert"][:3], inp["cert"][1:2]]), warp=torch.cat([inp["warp"][:3], inp["warp"][1:2]]))
           for inp in inputs]
    g = _run(engine, scene, dup, _cfg(c, True))
    for vm in g["view_mask"]:
        assert not ((vm & 0b1010) == 0b1010).any()
        assert ((vm & 0b0010) != 0).any()
    # slot 0 below the threshold everywhere: never in a mask unless it is the winner
    low = []
    for inp in inputs:
        cert = inp["cert"].clone()
        cert[0] = 0.3
        low.append(dict(inp, cert=cert))
    g = _run(engine, scene, low, _cfg(c, True, min_cert=0.5))
    for r in range(len(low)):
        vm = g["view_mask"][r]
        winner = g["flags"][r][G.expected_pack_order(g["flags"][r])] >> 2
        assert not ((vm & 1) != 0)[winner != 0].any()
    # one neighbour: the winner's bit alone, and the plain launch's points
    scene1, inputs1 = _scene_inputs(1)
    on, off = _run(engine, scene1, inputs1, _cfg(c, True)), _run(engine, scene1, inputs1, _cfg(c, False))
    for r in range(len(inputs1)):
        assert (on["view_mask"][r] == 1).all()
        assert on["xyz"][r].tobytes() == off["xyz"][r].tobytes()


def test_random_neighbour_rarely_joins_and_does_not_hurt(engine):
    c = dict(M=10000, no_filter=False)
    scene, inputs = _scene_inputs(4, return_points=True)
    g0 = torch.Generator().manual_seed(77)
    bad = []
    for inp in inputs:
        warp = inp["warp"].clone()
        warp[3, ..., 2:] = torch.rand(warp.shape[1:3] + (2,), generator=g0) * 2 - 1
        cert = inp["cert"].clone()
        cert[3] = 0.6                                    # confident enough to join, and wrong
        bad.append(dict(inp, warp=warp, cert=cert))
    on, off = _run(engine, scene, bad, _cfg(c, True)), _run(engine, scene, bad, _cfg(c, False))
    joined, total, d_on, d_off = 0, 0, [], []
    for r, inp in enumerate(bad):
        vm = on["view_mask"][r]
        order = G.expected_pack_order(on["flags"][r])
        winner = on["flags"][r][order] >> 2
        joined += int((((vm & 0b1000) != 0) & (winner != 3)).sum())
        total += vm.size
        truth = inp["points"].reshape(-1, 3).numpy()[on["sel"][r][order]]
        d_on.append(np.linalg.norm(on["xyz"][r].astype(np.float64) - truth, axis=1))
        d_off.append(np.linalg.norm(off["xyz"][r].astype(np.float64) - truth, axis=1))
    print(f"[random neighbour] in {joined} of {total} masks; median GT error {np.median(np.concatenate(d_on)):.3e} "
          f"(two-view {np.median(np.concatenate(d_off)):.3e})")
    assert joined < 0.01 * total
    assert np.median(np.concatenate(d_on)) <= np.median(np.concatenate(d_off))


def test_view_mask_without_multiview_is_invalid(engine):
    scene, inputs = _scene_inputs(2, n_refs=1)
    pl = engine.prepare(_batch(engine, scene, inputs), _cfg(dict(M=2000, no_filter=False), False))
    vm = torch.zeros(pl.outputs.err.shape[0], dtype=torch.int32, device=engine.device)
    pl.c_outputs.view_mask = vm.data_ptr()
    rc = engine.lib.ldp_densify_refs(*pl._args, C.c_void_p(torch.cuda.current_stream(engine.device).cuda_stream))
    assert rc == -1                                  # LDP_ERR_INVALID
    with pytest.raises(ValueError):
        engine.prepare(_batch(engine, scene, inputs), _cfg(dict(M=2000, no_filter=True), True))


# ---- 5. ground truth on the device path -------------------------------------------------------------------------------------
@pytest.mark.parametrize("nn,ratio", [(4, 0.8), (8, 0.7)])
def test_ground_truth_accuracy(engine, nn, ratio):
    scene = synth.make_scene(40, "turbo", nn=nn)
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family="R", return_points=True) for rp in range(3)]
    c = dict(M=4000, no_filter=False)
    on, off = _run(engine, scene, inputs, _cfg(c, True)), _run(engine, scene, inputs, _cfg(c, False))
    d_on, d_off = [], []
    for r, inp in enumerate(inputs):
        order = G.expected_pack_order(on["flags"][r])
        truth = inp["points"].reshape(-1, 3).numpy()[on["sel"][r][order]]
        d_on.append(np.linalg.norm(on["xyz"][r].astype(np.float64) - truth, axis=1))
        d_off.append(np.linalg.norm(off["xyz"][r].astype(np.float64) - truth, axis=1))
    m_on, m_off = np.median(np.concatenate(d_on)), np.median(np.concatenate(d_off))
    print(f"[ground truth] nn={nn}: median two-view {m_off:.3e}, multi-view {m_on:.3e}, ratio {m_on / m_off:.3f}")
    assert m_on <= ratio * m_off


# ---- 6. stage entry point and ring ------------------------------------------------------------------------------------------
def test_triangulate_samples_and_ring(engine):
    from lichtfeld_densification_plugin_b200.engine import DensifyRing
    scene = synth.make_scene(24, "fast", ref_fraction=0.5, nn=4)
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family="R", seed=12) for rp in range(scene.n_refs)]
    cfg = _cfg(dict(M=6000, no_filter=False), True)
    full = _run(engine, scene, inputs, cfg)
    # ldp_triangulate_samples on the full path's samples
    pl = engine.prepare(_batch(engine, scene, inputs), cfg, taps=True)
    dev = engine.device
    for r, s in enumerate(full["sel"]):
        pl.outputs.sel_idx[r, :s.size] = torch.from_numpy(s.astype(np.int32)).to(dev)
    pl.outputs.n_samples.copy_(torch.tensor([s.size for s in full["sel"]], dtype=torch.int32, device=dev))
    rc = engine.lib.ldp_triangulate_samples(C.byref(pl.params), C.c_void_p(pl.descs_dev.data_ptr()), C.byref(pl.c_outputs),
                                            C.c_void_p(pl.workspace.data_ptr()), C.c_size_t(pl.workspace.numel()),
                                            C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
    N.check(rc, "ldp_triangulate_samples")
    torch.cuda.synchronize()
    o = pl.outputs
    off = o.ref_offset.cpu().numpy()
    for r in range(len(inputs)):
        assert np.array_equal(o.xyz[off[r]:off[r + 1]].cpu().numpy(), full["xyz"][r]), r
        assert np.array_equal(o.view_mask[off[r]:off[r + 1]].cpu().numpy(), full["view_mask"][r]), r
    # three launches in flight on a ring == one at a time
    groups = [list(range(q, len(inputs), 3)) for q in range(3)]
    one = []
    for views in groups:
        x = engine.densify(_batch(engine, scene, [inputs[i] for i in views]), cfg)
        torch.cuda.synchronize()
        n = x.total_points()
        one.append((x.xyz[:n].cpu().numpy(), x.view_mask[:n].cpu().numpy()))
    ring = DensifyRing(dev, depth=3)
    outs = [ring.submit(_batch(ring.engines[ring.slot()], scene, [inputs[i] for i in views]), cfg) for views in groups]
    ring.synchronize()
    for (xyz, vm), x in zip(one, outs):
        n = x.total_points()
        assert n > 0 and xyz.tobytes() == x.xyz[:n].cpu().numpy().tobytes() and vm.tobytes() == x.view_mask[:n].cpu().numpy().tobytes()


# ---- 7. run_dense_pipeline --------------------------------------------------------------------------------------------------
def test_run_dense_pipeline_n_views(tmp_path):
    from lichtfeld_densification_plugin_b200.core import pipeline as P
    from lichtfeld_densification_plugin_b200.core.config import DensePipelineConfig
    nn = 4
    scene = synth.make_scene(24, "turbo", ref_fraction=0.5, nn=nn)
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
    kw = dict(output_path=str(tmp_path / "dense.ply"), matches_per_ref=4000, refs_per_launch=4)
    on = P.run_dense_pipeline(cams, refs, None, DensePipelineConfig(multiview=True, **kw), match_source=match_source,
                              w_match=scene.w_match, h_match=scene.h_match)
    off = P.run_dense_pipeline(cams, refs, None, DensePipelineConfig(**kw), match_source=match_source,
                               w_match=scene.w_match, h_match=scene.h_match)
    assert off.n_views is None
    assert on.n_views.dtype == np.uint8 and on.n_views.shape[0] == on.xyz.shape[0] == off.xyz.shape[0]
    assert on.n_views.min() >= 2 and on.n_views.max() <= 1 + nn and (on.n_views > 2).any()
    assert on.rgb.tobytes() == off.rgb.tobytes()
