"""GPU: size-independent properties at full BASELINE sizes, edge cases, determinism, the drop-in API."""
import numpy as np
import pytest
import torch

from tests import gpu_harness as G

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    from lichtfeld_densification_plugin_b200.engine import DensifyEngine
    return DensifyEngine()


@pytest.fixture(scope="module")
def fast_scene():
    from lichtfeld_densification_plugin_b200 import synth
    scene = synth.make_scene(40, "fast", ref_fraction=0.2, nn=4)
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family="R", seed=5) for rp in range(scene.n_refs)]
    return scene, inputs


def test_philox_properties_full_size(engine, fast_scene):
    scene, inputs = fast_scene
    c = dict(M=10000, no_filter=False, wm=scene.w_match, hm=scene.h_match)
    g = G.run_gpu(engine, scene, inputs, G.path_cfg(c, seed=7))
    H, W = scene.H, scene.W
    for r, inp in enumerate(inputs):
        assert g.status[r] & 0xFF == 0
        sel = g.sel_idx[r]
        assert np.all(np.diff(sel) > 0), "sel_idx must be strictly ascending (np.unique)"
        x, y = sel % W, sel // W
        assert x.min() >= 2 and x.max() <= W - 3 and y.min() >= 2 and y.max() <= H - 3, "border pixels are never sampled"
        assert 8500 <= sel.size <= 8500 + 625
        assert g.uniforms_used[r] >= 8500 and g.rounds[r] >= 1
        # every tile's best pixel is among the samples (coverage)
        best = inp["cert"].max(dim=0).values.numpy()
        wts = np.minimum(best, np.float32(0.9))
        wts[:2] = 0; wts[-2:] = 0; wts[:, :2] = 0; wts[:, -2:] = 0
        tile = max(1, W // 24)
        selset = set(sel.tolist())
        for ty in range(0, H, tile):
            for tx in range(0, W, tile):
                blk = wts[ty:ty + tile, tx:tx + tile]
                if blk.max() > 0:
                    ys, xs = np.nonzero(blk == blk.max())
                    assert any(((ty + a) * W + (tx + b)) in selset for a, b in zip(ys, xs))
        # kept points satisfy the filters when recomputed independently in f64
        keep = (g.flags[r] & 1).astype(bool)
        order = G.expected_pack_order(g.flags[r])
        assert np.array_equal(g.xyz[r], g.xyzerr[r][order, :3])
        assert g.err[r].size == keep.sum() and np.all(g.err[r] <= np.float32(0.8))
        cams = scene.cameras
        P1 = cams[inp["ref_index"]].P.astype(np.float64)
        Xh = np.concatenate([g.xyz[r].astype(np.float64), np.ones((g.xyz[r].shape[0], 1))], axis=1)
        assert np.all((Xh @ P1.T)[:, 2] > 0)
        assert np.all((g.rgb[r] >= 0) & (g.rgb[r] <= 1))


def test_deterministic_and_batch_independent(engine, fast_scene):
    scene, inputs = fast_scene
    c = dict(M=10000, no_filter=False, wm=scene.w_match, hm=scene.h_match)
    a = G.run_gpu(engine, scene, inputs, G.path_cfg(c, seed=11))
    b = G.run_gpu(engine, scene, inputs, G.path_cfg(c, seed=11))
    solo = G.run_gpu(engine, scene, inputs[2:3], G.path_cfg(c, seed=11))
    other = G.run_gpu(engine, scene, inputs[2:3], G.path_cfg(c, seed=12))
    for r in range(len(inputs)):
        assert np.array_equal(a.sel_idx[r], b.sel_idx[r]) and np.array_equal(a.xyz[r], b.xyz[r])
        assert np.array_equal(a.rgb[r], b.rgb[r]) and np.array_equal(a.err[r], b.err[r])
    # a view's result depends on (seed, rng_stream) only, not on what else is in the launch (sharding invariance)
    assert np.array_equal(a.sel_idx[2], solo.sel_idx[0]) and np.array_equal(a.xyz[2], solo.xyz[0])
    assert not np.array_equal(a.sel_idx[2], other.sel_idx[0])


def test_no_filter_full_size(engine, fast_scene):
    scene, inputs = fast_scene
    c = dict(M=10000, no_filter=True, wm=scene.w_match, hm=scene.h_match)
    g = G.run_gpu(engine, scene, inputs[:3], G.path_cfg(c))
    for r in range(3):
        res = G.run_oracle_ref(scene, inputs[r], c)
        sel = g.sel_idx[r]
        assert sel.size == 10000 and np.unique(sel).size == 10000
        capped = np.minimum(inputs[r]["cert"].max(dim=0).values.numpy().reshape(-1), np.float32(0.9))
        v = capped[sel]
        assert np.all(np.diff(v) <= 0), "descending certainty"
        assert np.array_equal(np.sort(v), np.sort(capped[res.sel_idx])), "same multiset of certainties as argsort(-cert)[:M]"
        assert v.min() >= np.sort(capped)[-10000]
        keep = (g.flags[r] & 1).astype(bool)
        assert keep.sum() == np.isfinite(g.xyzerr[r]).all(axis=1).sum()


def _mk_single(scene_hw, nn, cert_fn, M):
    from lichtfeld_densification_plugin_b200 import synth
    H, W = scene_hw
    scene = synth.make_scene(8, "turbo", ref_fraction=0.13, nn=nn)
    scene.H, scene.W, scene.h_match, scene.w_match = H, W, H, W
    inp = synth.synth_ref_inputs(scene, 0, cert_family="T", seed=9)
    inp["cert"] = cert_fn(inp["cert"])
    return scene, inp, dict(M=M, no_filter=False, wm=W, hm=H)


def test_edge_all_zero_weights(engine):
    scene, inp, c = _mk_single((64, 64), 2, lambda x: torch.zeros_like(x), 500)
    g = G.run_gpu(engine, scene, [inp], G.path_cfg(c))
    assert g.status[0] & 0xFF == 1 and g.sel_idx[0].size == 0 and g.xyz[0].shape[0] == 0     # LDP_REF_EMPTY


def test_edge_fewer_nonzero_than_size(engine):
    def sparse(x):
        y = torch.zeros_like(x)
        y[:, 10:20, 10:20] = x[:, 10:20, 10:20]
        return y
    scene, inp, c = _mk_single((64, 64), 2, sparse, 500)
    g = G.run_gpu(engine, scene, [inp], G.path_cfg(c))
    assert g.status[0] & 0xFF == 2                                                            # LDP_REF_FEWER_NONZERO
    with pytest.raises(ValueError, match="Fewer non-zero"):
        G.run_oracle_ref(scene, inp, c, uniforms=np.zeros(4000))


def test_edge_nan_and_ragged_neighbours(engine):
    def nanify(x):
        y = x.clone()
        y[0, 30, 30] = float("nan")
        return y
    scene, inp, c = _mk_single((64, 64), 2, nanify, 500)
    g = G.run_gpu(engine, scene, [inp], G.path_cfg(c))
    assert g.status[0] & 0xFF == 3                                                            # LDP_REF_BAD_WEIGHTS
    # ragged: views with 1 and 3 neighbours in the same launch
    from lichtfeld_densification_plugin_b200 import synth
    scene = synth.make_scene(10, "turbo", ref_fraction=0.2, nn=3)
    scene.H = scene.W = scene.h_match = scene.w_match = 96
    a = synth.synth_ref_inputs(scene, 0, cert_family="T", seed=1)
    b = synth.synth_ref_inputs(scene, 1, cert_family="T", seed=1)
    b = dict(b, cert=b["cert"][:1], warp=b["warp"][:1], nbr_indices=b["nbr_indices"][:1])
    c = dict(M=2000, no_filter=False, wm=96, hm=96)
    U = np.stack([np.random.RandomState(r).random_sample(6000) for r in range(2)])
    ress = [G.run_oracle_ref(scene, x, c, uniforms=U[i]) for i, x in enumerate((a, b))]
    g = G.run_gpu(engine, scene, [a, b], G.path_cfg(c), uniforms=U, weight_sums=[r.taps["s"] for r in ress])
    for i in range(2):
        rep = G.compare_ref(g, i, ress[i], c, scene)
        assert rep.ok(), rep


def test_edge_non_multiple_of_four_width_and_tiny_m(engine):
    from lichtfeld_densification_plugin_b200 import synth
    scene = synth.make_scene(8, "turbo", ref_fraction=0.13, nn=2)
    scene.H, scene.W, scene.h_match, scene.w_match = 50, 61, 50, 61
    inp = synth.synth_ref_inputs(scene, 0, cert_family="T", seed=4)
    for M in (1, 7, 700):
        c = dict(M=M, no_filter=False, wm=61, hm=50)
        U = np.random.RandomState(M).random_sample(3 * M + 16)
        res = G.run_oracle_ref(scene, inp, c, uniforms=U)
        g = G.run_gpu(engine, scene, [inp], G.path_cfg(c), uniforms=U[None, :],
                      weight_sums=[res.taps["s"]] if res is not None else None)
        if res is None:
            assert g.xyz[0].shape[0] == 0
            continue
        rep = G.compare_ref(g, 0, res, c, scene)
        assert rep.ok(), (M, rep)


def test_drop_in_triangulate_ref_numpy_global_stream(engine):
    """core.pipeline._triangulate_ref with rng_mode='numpy' consumes np.random's global stream like the reference."""
    from lichtfeld_densification_plugin_b200 import synth
    from lichtfeld_densification_plugin_b200.core import pipeline as P
    from lichtfeld_densification_plugin_b200.core.config import DensePipelineConfig
    scene = synth.make_scene(10, "turbo", ref_fraction=0.2, nn=3)
    cams = scene.cameras
    cfg = DensePipelineConfig(output_path="/tmp/x.ply", rng_mode="numpy")
    ctx = P._TriangulationContext(cameras=P._build_camera_lookup(cams), config=cfg, matcher_sample_cap=0.9,
                                  w_match=scene.w_match, h_match=scene.h_match)
    c = dict(M=10000, no_filter=False, wm=scene.w_match, hm=scene.h_match)
    np.random.seed(123)
    outs = []
    for rp in range(2):
        inp = synth.synth_ref_inputs(scene, rp, cert_family="T", seed=2)
        ri, nb = inp["ref_index"], inp["nbr_indices"]
        packed = P._PackedReferenceBatch(ref_id=cams[ri].uid, ref_path="", imA_np=inp["image"].numpy(), maskA_np=None,
                                         wA_cam=cams[ri].width, hA_cam=cams[ri].height, nn_ids=[cams[j].uid for j in nb],
                                         nn_masks=[None] * len(nb), nn_arrays=[None] * len(nb))
        mr = P._MatchedReference(packed=packed, warp_list_cpu=[inp["warp"][k] for k in range(len(nb))],
                                 cert_list_cpu=[inp["cert"][k] for k in range(len(nb))], pair_index_by_nbr={}, image_by_nbr={})
        outs.append((inp, P._triangulate_ref(mr, ctx, collect_debug_matches=True)))
    after = np.random.random_sample()
    # oracle: same global stream, sequentially (the reference's production behaviour)
    rs = np.random.RandomState(123)
    for inp, tri in outs:
        res = G.run_oracle_ref(scene, inp, c, rng=rs, collect_debug=True)
        assert tri is not None and abs(tri.xyz.shape[0] - res.xyz.shape[0]) <= 3
        if tri.xyz.shape == res.xyz.shape:
            np.testing.assert_allclose(tri.xyz, res.xyz, rtol=G.XYZ_RTOL, atol=G.XYZ_ATOL)
            np.testing.assert_allclose(tri.rgb, res.rgb, rtol=G.XYZ_RTOL, atol=G.XYZ_ATOL)
            assert list(tri.debug_matches_by_nbr.keys()) == list(res.debug_matches_by_nbr.keys())
    assert after == rs.random_sample(), "global MT19937 stream position must match the reference's"


def test_cluster_size_does_not_change_results(engine, fast_scene):
    """The draw kernel runs as a thread-block cluster per view; any cluster size gives identical samples."""
    scene, inputs = fast_scene
    c = dict(M=10000, no_filter=False, wm=scene.w_match, hm=scene.h_match)
    lib = engine.lib
    base = None
    used = []
    try:
        for cs in (1, 2, 3, 4, 5, 8):
            assert lib.ldp_debug_set_cluster(cs) == 0
            g = G.run_gpu(engine, scene, inputs[:3], G.path_cfg(c, seed=3))
            used.append(lib.ldp_debug_last_cluster())
            if base is None:
                base = g
                continue
            for r in range(3):
                assert np.array_equal(base.sel_idx[r], g.sel_idx[r]), (cs, r)
                assert np.array_equal(base.xyz[r], g.xyz[r]) and base.uniforms_used[r] == g.uniforms_used[r]
    finally:
        lib.ldp_debug_set_cluster(0)
    print("cluster sizes actually launched:", used)
    assert used[0] == 1 and max(used) >= 2


def test_select_samples_with_coverage_drop_in(engine):
    """core.sampling.select_samples_with_coverage: reference signature, reference RNG stream semantics."""
    from lichtfeld_densification_plugin_b200.core.sampling import select_samples_with_coverage
    from oracle import densify_oracle as O
    rs = np.random.RandomState(3)
    vals = (0.2 + 0.7 * (rs.permutation(120 * 90) + 0.5) / (120 * 90)).astype(np.float32).reshape(90, 120)
    cert = torch.from_numpy(vals)
    np.random.seed(77)
    got = select_samples_with_coverage(cert, 3000)
    after = np.random.random_sample()
    ref_rng = np.random.RandomState(77)
    taps = {}
    want = O.select_samples(cert, 3000, rng=ref_rng, taps=taps)
    # the oracle's s comes from torch-CPU; ours from an exact f64 sum: compare through the oracle fed with our s
    if not np.array_equal(got, want):
        s_exact = np.float32(taps["weights"].astype(np.float64).sum())
        want = O.select_samples(cert, 3000, rng=np.random.RandomState(77), s_override=s_exact)
        ref_rng = np.random.RandomState(77)
        O.select_samples(cert, 3000, rng=ref_rng, s_override=s_exact)
    assert np.array_equal(got, want)
    assert after == ref_rng.random_sample()
    top = select_samples_with_coverage(cert, 500, no_filter=True)
    assert np.array_equal(top, O.select_samples(cert, 500, no_filter=True))


def _colliding_weight_map(H=90, W=120, seed=11):
    """f32 map, distinct values, in which 49 tiles hold an adjacent-float pair (smaller weight at the lower index) whose
    quotients by s = f32(sum of the border-masked weights) round to the same f32."""
    tile = max(1, W // 24)
    rs = np.random.RandomState(seed)
    vals = (0.2 + 0.6 * (rs.permutation(H * W) + 0.5) / (H * W)).astype(np.float32).reshape(H, W)      # < 0.8, distinct
    inside = np.zeros((H, W), bool)
    inside[2:H - 2, 2:W - 2] = True
    wsum = lambda: np.where(inside, vals, 0).astype(np.float64).sum()
    s = np.float32(wsum())                                # the normaliser is pinned first ...
    tiles = [(ty, tx) for ty in range(2, 16, 2) for tx in range(2, 22, 3)]
    cands = np.arange(0.85, 0.899, 1e-4, dtype=np.float32)
    ok = [a for a in cands if np.float32(a / s) == np.float32(np.nextafter(a, np.float32(1)) / s)]
    assert len(ok) >= len(tiles)
    for (ty, tx), a in zip(tiles, ok):
        y, x = ty * tile + 1, tx * tile + 1
        vals[y, x] = a                                    # lower index, smaller weight
        vals[y + 2, x + 2] = np.nextafter(a, np.float32(1))
    # ... and the mass the pairs added is taken back from pixels of the last tile row, which stay far from any tile maximum
    by, bx = np.nonzero(inside & (np.arange(H)[:, None] >= 17 * tile) & (vals > 0.5) & (vals < 0.75))
    for _ in range(8):
        d = wsum() - float(s)
        if np.float32(wsum()) == s and abs(d) < 1e-4:
            break
        vals[by, bx] = (vals[by, bx].astype(np.float64) - d / by.size).astype(np.float32)
    assert np.float32(wsum()) == s and vals[by, bx].min() > 0.2
    pairs = [((ty * tile + 1) * W + tx * tile + 1, (ty * tile + 3) * W + tx * tile + 3) for ty, tx in tiles]
    flat = vals.reshape(-1)
    assert all(np.float32(flat[i] / s) == np.float32(flat[j] / s) and flat[i] < flat[j] for i, j in pairs)
    return vals, s, pairs


def test_coverage_walk_is_on_normalised_p(engine):
    """core/sampling.py:29 rebinds `weights` to p = weights / s BEFORE the coverage walk (:38): two adjacent f32
    weights whose quotients round to the same p are a TIE for np.argsort (unstable), not an ordered pair.  The kernel
    must therefore agree with the reference everywhere except inside such tied pairs, where either pixel is valid."""
    from lichtfeld_densification_plugin_b200.core.sampling import select_samples_with_coverage
    from oracle import densify_oracle as O
    vals, s, pairs = _colliding_weight_map()
    cert = torch.from_numpy(vals)
    M = 3000
    np.random.seed(5)
    got = set(select_samples_with_coverage(cert, M).tolist())
    want = set(O.select_samples(cert, M, rng=np.random.RandomState(5), s_override=s).tolist())
    decided = [(i, j) for i, j in pairs if (i in want) != (j in want)]
    assert len(decided) >= 10, "test construction: the main draw took too many of the pairs"
    partner = {i: j for i, j in pairs}
    partner.update({j: i for i, j in pairs})
    for only_a, b in ((got - want, want), (want - got, got)):
        for i in only_a:
            assert i in partner and partner[i] in b, f"pixel {i} differs outside a tied pair"


def test_more_views_than_sms(engine):
    """A launch with more reference views than the device has SMs (the draw kernels then run one CTA per view in
    several waves): every view's result equals its result in a launch of its own."""
    from lichtfeld_densification_plugin_b200 import synth
    scene = synth.make_scene(340, "turbo", ref_fraction=0.5, nn=2)
    scene.H = scene.W = scene.h_match = scene.w_match = 64
    R = scene.n_refs
    assert R > 160
    c = dict(M=600, no_filter=False, wm=64, hm=64)
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family="T", seed=3) for rp in range(R)]
    streams = list(range(R))
    whole = G.run_gpu(engine, scene, inputs, G.path_cfg(c, seed=5), rng_streams=streams)
    assert (whole.status & 0xFF == 0).all()
    for rp in (0, 1, 77, 159, R - 1):
        single = G.run_gpu(engine, scene, [inputs[rp]], G.path_cfg(c, seed=5), rng_streams=[streams[rp]])
        assert np.array_equal(single.sel_idx[0], whole.sel_idx[rp]), rp
        assert np.array_equal(single.xyz[0], whole.xyz[rp]) and np.array_equal(single.rgb[0], whole.rgb[rp])
        assert single.uniforms_used[0] == whole.uniforms_used[rp]
    res = G.run_oracle_ref(scene, inputs[77], c, uniforms=np.random.RandomState(1).random_sample(3000))
    g1 = G.run_gpu(engine, scene, [inputs[77]], G.path_cfg(c), uniforms=np.random.RandomState(1).random_sample(3000)[None, :],
                   weight_sums=[res.taps["s"]])
    rep = G.compare_ref(g1, 0, res, c, scene)
    assert rep.ok(), rep


def test_no_filter_cluster_sizes_and_tie_rule(engine, fast_scene):
    """no_filter top-M: one cluster of 1/2/4/8 CTAs per view gives the same, fully determined order
    (descending capped certainty, ascending pixel index among equal certainties = a stable argsort)."""
    scene, inputs = fast_scene
    lib = engine.lib
    used = []
    try:
        for M in (10000, 777, 3):
            c = dict(M=M, no_filter=True, wm=scene.w_match, hm=scene.h_match)
            for cs in (1, 2, 4, 8):
                assert lib.ldp_debug_set_cluster(cs) == 0
                g = G.run_gpu(engine, scene, inputs[:3], G.path_cfg(c))
                used.append(lib.ldp_debug_last_cluster())
                for r in range(3):
                    capped = np.minimum(inputs[r]["cert"].max(dim=0).values.numpy().reshape(-1), np.float32(0.9))
                    want = np.argsort(-capped, kind="stable")[:M]
                    assert np.array_equal(g.sel_idx[r], want), (M, cs, r)
    finally:
        lib.ldp_debug_set_cluster(0)
    print("top-M cluster sizes launched:", used)
    assert max(used) >= 2


def test_no_filter_ties_cut_inside_a_plateau(engine):
    """More pixels tie at the M-th certainty than are needed: the lowest pixel indices win, whichever CTA holds them."""
    H = W = 96
    rs = np.random.RandomState(5)

    def cert_fn(cert):
        v = rs.choice(np.array([0.3, 0.5, 0.7, 0.95, 0.99], np.float32), size=cert.shape).astype(np.float32)
        return torch.from_numpy(v)
    for M in (50, 4000, 9000):
        scene, inp, c = _mk_single((H, W), 2, cert_fn, M)
        c = dict(c, no_filter=True)
        capped = np.minimum(inp["cert"].max(dim=0).values.numpy().reshape(-1), np.float32(0.9))
        want = np.argsort(-capped, kind="stable")[:min(M, H * W)]
        try:
            for cs in (1, 2, 4, 8):
                engine.lib.ldp_debug_set_cluster(cs)
                g = G.run_gpu(engine, scene, [inp], G.path_cfg(c))
                assert np.array_equal(g.sel_idx[0], want), (M, cs)
        finally:
            engine.lib.ldp_debug_set_cluster(0)


def test_no_filter_distinct_certainties_cluster_sizes(engine):
    """Tie-free certainties (nothing saturated): the generic path - radix select, gather, cluster-wide bitonic sort."""
    from lichtfeld_densification_plugin_b200 import synth
    scene = synth.make_scene(40, "fast", ref_fraction=0.2, nn=4)
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family="T", seed=6) for rp in range(2)]
    try:
        for M in (10000, 16384, 130, 1):
            c = dict(M=M, no_filter=True, wm=scene.w_match, hm=scene.h_match)
            for cs in (1, 2, 4, 8):
                engine.lib.ldp_debug_set_cluster(cs)
                g = G.run_gpu(engine, scene, inputs, G.path_cfg(c))
                for r in range(2):
                    capped = np.minimum(inputs[r]["cert"].max(dim=0).values.numpy().reshape(-1), np.float32(0.9))
                    assert np.array_equal(g.sel_idx[r], np.argsort(-capped, kind="stable")[:M]), (M, cs, r)
    finally:
        engine.lib.ldp_debug_set_cluster(0)


def test_no_filter_more_matches_than_the_shared_memory_sort_holds(engine, fast_scene):
    """M > 16384: the one-CTA kernel that sorts in global memory (same order rule)."""
    scene, inputs = fast_scene
    M = 20000
    c = dict(M=M, no_filter=True, wm=scene.w_match, hm=scene.h_match)
    g = G.run_gpu(engine, scene, inputs[:2], G.path_cfg(c))
    for r in range(2):
        capped = np.minimum(inputs[r]["cert"].max(dim=0).values.numpy().reshape(-1), np.float32(0.9))
        assert np.array_equal(g.sel_idx[r], np.argsort(-capped, kind="stable")[:M])


def test_ring_of_launches_gives_the_same_results(engine, fast_scene):
    """DensifyRing: launches in flight on several streams / workspaces produce exactly what one engine produces."""
    from lichtfeld_densification_plugin_b200.engine import DensifyRing, PathConfig
    scene, inputs = fast_scene
    dev = engine.device
    cfg = PathConfig(matches_per_ref=10000, seed=11)

    def batch_for(eng, lo, hi):
        b = eng.new_batch(scene.H, scene.W, scene.w_match, scene.h_match)
        for rp in range(lo, hi):
            inp = inputs[rp]
            k = len(inp["nbr_indices"])
            b.add([inp["cert"][q].to(dev) for q in range(k)], [inp["warp"][q].to(dev) for q in range(k)], inp["image"].to(dev),
                  scene.cameras[inp["ref_index"]], [scene.cameras[j] for j in inp["nbr_indices"]], rng_stream=rp)
        return b
    n = len(inputs)
    cuts = [(0, n // 3), (n // 3, 2 * n // 3), (2 * n // 3, n), (0, n)]
    want = []
    for lo, hi in cuts:
        o = engine.densify(batch_for(engine, lo, hi), cfg)
        k = o.total_points()
        want.append((o.xyz[:k].clone(), o.rgb[:k].clone(), o.ref_offset.clone()))
    ring = DensifyRing(dev, depth=3)
    outs = [ring.submit(batch_for(ring.engines[0], lo, hi), cfg) for _ in range(2) for lo, hi in cuts]     # 8 launches, 3 in flight
    for o in outs:
        ring.wait(o)
    torch.cuda.synchronize()
    for idx, o in enumerate(outs):
        xyz, rgb, off = want[idx % len(cuts)]
        k = int(off[-1])
        assert torch.equal(o.ref_offset, off) and torch.equal(o.xyz[:k], xyz) and torch.equal(o.rgb[:k], rgb), idx


def test_launches_in_flight_with_late_starting_draw_ctas(engine):
    """Regression: the first draw round of a view runs on several independent CTAs that build their search tables from the
    view's chunk sums whenever they happen to start; with three launches in flight and more draw CTAs than SMs some start
    after their siblings have found pixels.  The chunk sums must still read as the prep kernel left them (round-1 finds are
    accounted in a side table).  BASELINE config-5 shapes (640^2, 42 views per launch: 126 one-CTA-per-SM draw CTAs per
    launch), four passes of six launches back to back on the ring, against one engine running the launches one by one."""
    from lichtfeld_densification_plugin_b200 import synth
    from lichtfeld_densification_plugin_b200.engine import DensifyRing, PathConfig
    dev = engine.device
    scene = synth.make_scene(1000, "base", 0.25, 4)
    R, per = scene.n_refs, 42
    cfg = PathConfig(matches_per_ref=10000, seed=5)
    inputs = [synth.synth_ref_inputs(scene, rp, device=dev, cert_family="R", seed=500) for rp in range(R)]

    def batch_for(eng, lo, hi):
        b = eng.new_batch(scene.H, scene.W, scene.w_match, scene.h_match)
        for rp in range(lo, hi):
            inp = inputs[rp]
            k = len(inp["nbr_indices"])
            b.add([inp["cert"][q] for q in range(k)], [inp["warp"][q] for q in range(k)], inp["image"],
                  scene.cameras[inp["ref_index"]], [scene.cameras[j] for j in inp["nbr_indices"]], rng_stream=rp)
        return b
    chunks = [(a, min(a + per, R)) for a in range(0, R, per)]
    sel_cap = engine.sel_capacity(cfg.matches_per_ref)
    want = []
    for lo, hi in chunks:
        o = engine.densify(batch_for(engine, lo, hi), cfg)
        torch.cuda.synchronize()
        k = o.total_points()
        want.append((o.n_samples.clone(), o.uniforms_used.clone(), o.ref_offset.clone(), o.xyz[:k].clone()))
    ring = DensifyRing(dev, depth=3)
    outs = [engine.alloc_outputs(hi - lo, sel_cap) for lo, hi in chunks]
    prepared = []
    for c, (lo, hi) in enumerate(chunks):
        e = ring.engines[c % 3]
        b = batch_for(e, lo, hi)
        prepared.append((c % 3, e.prepare(b, cfg, descs_dev=e.upload_descs(b), outputs=outs[c])))
    main = torch.cuda.current_stream(dev)
    for _ in range(4):                                   # no host synchronisation between the passes
        for st in ring.streams:
            st.wait_stream(main)
        for j, p in prepared:
            with torch.cuda.stream(ring.streams[j]):
                p.launch()
        for st in ring.streams:
            main.wait_stream(st)
    torch.cuda.synchronize()
    for c, o in enumerate(outs):
        ns, uu, off, xyz = want[c]
        assert torch.equal(o.n_samples, ns) and torch.equal(o.uniforms_used, uu), (c, (o.uniforms_used != uu).nonzero().flatten().tolist())
        assert torch.equal(o.ref_offset, off) and torch.equal(o.xyz[:int(off[-1])], xyz), c


@pytest.mark.parametrize("no_filter, kernels", [
    (False, ["ldp_stream_kernel", "ldp_prep_kernel", "ldp_draw_kernel", "ldp_resume_kernel", "ldp_geometry_kernel", "ldp_fix_kernel",
             "ldp_pack_kernel"]),
    (True, ["ldp_stream_kernel", "ldp_topm_kernel", "ldp_geometry_kernel", "ldp_fix_kernel", "ldp_pack_kernel"]),
])
def test_profile_names_and_launch_count(engine, fast_scene, no_filter, kernels):
    """One call's profile lists its kernels in launch order under the names bench.py's per-kernel report keys on, and
    ldp_last_launch_count (bench.py's gpu_launches) counts exactly those launches."""
    import ctypes as C
    from lichtfeld_densification_plugin_b200.engine import PathConfig
    scene, inputs = fast_scene
    dev = engine.device
    b = engine.new_batch(scene.H, scene.W, scene.w_match, scene.h_match)
    for rp in range(2):
        inp = inputs[rp]
        k = len(inp["nbr_indices"])
        b.add([inp["cert"][q].to(dev) for q in range(k)], [inp["warp"][q].to(dev) for q in range(k)], inp["image"].to(dev),
              scene.cameras[inp["ref_index"]], [scene.cameras[j] for j in inp["nbr_indices"]], rng_stream=rp)
    lib = engine.lib
    assert lib.ldp_profile_enable(1) == 0
    try:
        engine.densify(b, PathConfig(matches_per_ref=10000, no_filter=no_filter, seed=3))
        assert lib.ldp_last_launch_count() == len(kernels)
        ms = (C.c_float * 64)()
        assert lib.ldp_profile_read(ms, 64) == len(kernels)
        assert [lib.ldp_profile_name(i).decode() for i in range(len(kernels))] == kernels
    finally:
        lib.ldp_profile_enable(0)
