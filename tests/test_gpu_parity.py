"""GPU parity: the CUDA path (through the C ABI) vs the oracle on identical inputs, uniforms and weight sum."""
import json

import numpy as np
import pytest
import torch

from tests.helpers import GOLDEN_CASES, load_golden
from tests import gpu_harness as G

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    from lichtfeld_densification_plugin_b200.engine import DensifyEngine
    return DensifyEngine()


def _report(name, rep):
    print(f"[parity] {name}: S={rep.n_samples} sel_exact={rep.sel_exact} tie_swaps={rep.sel_tie_swaps} "
          f"kept gpu/ref={rep.n_kept_gpu}/{rep.n_kept_ref} flips={len(rep.keep_flips)} far={rep.keep_flips_far} "
          f"max_xyz_rel={rep.max_xyz_rel:.3e} max_err_abs={rep.max_err_abs:.3e} max_rgb_abs={rep.max_rgb_abs:.3e}")
    for f in rep.keep_flips[:10]:
        print("   flip:", json.dumps(f))


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_golden_case_vs_oracle_and_reference_golden(engine, name):
    c, scene, inp, z = load_golden(name)
    U = np.random.RandomState(int(z["mt_seed"])).random_sample(3 * c["M"] + 64)
    s = z["weight_sum"]
    res = G.run_oracle_ref(scene, inp, c, uniforms=None if c["no_filter"] else U, s_override=s, collect_debug=True)
    g = G.run_gpu(engine, scene, [inp], G.path_cfg(c), uniforms=U[None, :], weight_sums=[s], collect_debug=True)
    assert g.status[0] & 0xFF == 0
    rep = G.compare_ref(g, 0, res, c, scene)
    _report(name, rep)
    assert rep.ok(), rep
    assert len(rep.keep_flips) == 0, rep.keep_flips        # goldens: keep masks are bit-exact, no point is even near a flip
    if not c["no_filter"]:
        assert g.uniforms_used[0] == res.taps["uniforms_used"] and g.rounds[0] == res.taps["rounds"]
        # the frozen output of the LIVE reference (made in the build container)
        assert np.array_equal(g.sel_idx[0], z["sel_idx"]) or rep.sel_tie_swaps > 0
    # packed output is exactly the kept per-sample values in the reference's emission order
    order = G.expected_pack_order(g.flags[0])
    assert np.array_equal(g.xyz[0], g.xyzerr[0][order, :3])
    assert np.array_equal(g.err[0], g.xyzerr[0][order, 3])
    if not rep.keep_flips and rep.sel_exact:
        assert g.xyz[0].shape == z["xyz"].shape
        np.testing.assert_allclose(g.xyz[0], z["xyz"], rtol=G.XYZ_RTOL, atol=G.XYZ_ATOL)
        np.testing.assert_allclose(g.rgb[0], z["rgb"], rtol=G.XYZ_RTOL, atol=G.XYZ_ATOL)
        np.testing.assert_allclose(g.err[0], z["err"], rtol=G.XYZ_RTOL, atol=G.ERR_ATOL)
        # debug outputs, split per neighbour like the reference's dicts
        pos = 0
        uids = [scene.cameras[j].uid for j in inp["nbr_indices"]]
        seen = []
        for gid in g.group_order[0]:
            if gid < 0:
                break
            cnt = int(g.group_count[0][gid])
            if cnt:
                uid = uids[gid]
                seen.append(uid)
                np.testing.assert_allclose(g.dbg_matches[0][pos:pos + cnt], z[f"dbg_matches_{uid}"], rtol=0, atol=1e-4)
                np.testing.assert_allclose(g.dbg_cert[0][pos:pos + cnt], z[f"dbg_cert_{uid}"], rtol=0, atol=1e-6)
            pos += cnt
        assert seen == [int(u) for u in z["dbg_uids"]]


@pytest.mark.parametrize("setting,nn,fam", [("fast", 4, "T"), ("fast", 4, "R"), ("base", 3, "T")])
def test_preset_sizes_vs_oracle(engine, setting, nn, fam):
    from lichtfeld_densification_plugin_b200 import synth
    scene = synth.make_scene(24, setting, ref_fraction=0.125, nn=nn)
    c = dict(M=10000, no_filter=False, wm=scene.w_match, hm=scene.h_match)
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family=fam, seed=21) for rp in range(scene.n_refs)]
    R = len(inputs)
    U = np.stack([np.random.RandomState(500 + r).random_sample(3 * c["M"]) for r in range(R)])
    ress, sums = [], []
    for r, inp in enumerate(inputs):
        res = G.run_oracle_ref(scene, inp, c, uniforms=U[r])
        ress.append(res)
        sums.append(res.taps["s"])
    g = G.run_gpu(engine, scene, inputs, G.path_cfg(c), uniforms=U, weight_sums=sums)
    for r in range(R):
        rep = G.compare_ref(g, r, ress[r], c, scene)
        _report(f"{setting}/{nn}nn/{fam}/ref{r}", rep)
        assert rep.ok(), rep
        assert g.uniforms_used[r] == ress[r].taps["uniforms_used"]
        if fam == "T":
            assert rep.sel_exact or rep.sel_tie_swaps > 0
        order = G.expected_pack_order(g.flags[r])
        assert np.array_equal(g.xyz[r], g.xyzerr[r][order, :3])


def test_bench_batch_philox_mode_vs_oracle(engine):
    """The PRODUCTION configuration at the bench size: the 46-view batch bench.py times (BASELINE config 2: 185 views,
    fast 512x512, 4 neighbours, M = 10 000, all filters), Philox mode, computed normaliser.  The oracle is fed the host
    restatement of the same Philox stream (oracle.philox_uniforms, pinned by Random123's known answers in
    tests/test_oracle_philox.py) and the f32 normaliser the launch reports; sampled indices, uniforms consumed,
    rejection rounds and keep masks must then agree exactly (coverage picks up to equal-weight ties inside a tile: the
    realistic certainty family saturates at the cap; keep flips only where gpu_harness._explain_flip shows the GPU holds
    the exact verdict and the reference's f32 SVD noise crossed the threshold, each listed), xyz / rgb / err within tolerance."""
    from lichtfeld_densification_plugin_b200 import synth
    scene = synth.make_scene(185, "fast", ref_fraction=0.25, nn=4)
    assert scene.n_refs == 46
    c = dict(M=10000, no_filter=False, wm=scene.w_match, hm=scene.h_match)
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family="R", seed=100) for rp in range(scene.n_refs)]
    seed = 0xB200
    streams = [1000 + rp for rp in range(scene.n_refs)]
    g = G.run_gpu(engine, scene, inputs, G.path_cfg(c, seed=seed), rng_streams=streams)
    assert g.launches > 0
    n_flips = 0
    for r, inp in enumerate(inputs):
        assert g.status[r] & 0xFF == 0
        U = O_philox(seed, streams[r], int(g.uniforms_used[r]) + 64)
        res = G.run_oracle_ref(scene, inp, c, uniforms=U, s_override=np.float32(g.weight_sum[r]))
        rep = G.compare_ref(g, r, res, c, scene)
        if r < 4 or not rep.ok() or rep.keep_flips:
            _report(f"bench-batch/philox/ref{r}", rep)
        assert rep.ok(), rep
        assert rep.sel_exact or rep.sel_tie_swaps > 0
        assert np.array_equal(np.setdiff1d(res.taps["idx_main"], g.sel_idx[r]), np.zeros(0, dtype=np.int64))   # every weighted draw
        assert g.uniforms_used[r] == res.taps["uniforms_used"] and g.rounds[r] == res.taps["rounds"]
        n_flips += len(rep.keep_flips)
    print(f"[parity] bench batch, philox mode: 46 views, {sum(x.size for x in g.sel_idx)} samples, keep flips {n_flips} "
          "(each listed above: the GPU's verdict is the exact one, the reference's f32 SVD crossed the threshold)")
    assert n_flips <= 4          # 1 in 418 000 samples measured; anything more is a regression


def O_philox(seed, stream, n):
    from oracle import densify_oracle as O
    return O.philox_uniforms(seed, stream, n)


def test_computed_weight_sum_is_correctly_rounded(engine):
    """Without an override, s is the f64 sum of the f32 weights rounded once to f32."""
    from lichtfeld_densification_plugin_b200 import synth
    scene = synth.make_scene(12, "turbo", ref_fraction=0.1, nn=2)
    c = dict(M=4000, no_filter=False, wm=scene.w_match, hm=scene.h_match)
    inp = synth.synth_ref_inputs(scene, 0, cert_family="R", seed=3)
    U = np.random.RandomState(1).random_sample(3 * c["M"])
    res = G.run_oracle_ref(scene, inp, c, uniforms=U)
    g = G.run_gpu(engine, scene, [inp], G.path_cfg(c), uniforms=U[None, :])
    want = np.float32(res.taps["weights"].astype(np.float64).sum())
    assert g.weight_sum[0] == want
    # and feeding that s to the oracle reproduces the GPU's samples exactly
    res2 = G.run_oracle_ref(scene, inp, c, uniforms=U, s_override=want)
    rep = G.compare_ref(g, 0, res2, c, scene)
    _report("computed-s", rep)
    assert rep.ok() and (rep.sel_exact or rep.sel_tie_swaps > 0)


def test_config3_precise_1280_maps_800_match(engine):
    """BASELINE config 3 shape: 'precise' preset -> 1280x1280 maps, 800x800 match resolution, 4 neighbours, all filters on.
    (Distortion parameters of OPENCV cameras are ignored by the reference, SURVEY F2; bidirectional warps never reach
    the path, F3.)  Exercises the 128-pixel chunk table."""
    from lichtfeld_densification_plugin_b200 import synth
    scene = synth.make_scene(16, "precise", ref_fraction=0.07, nn=4)
    assert (scene.H, scene.W, scene.h_match, scene.w_match) == (1280, 1280, 800, 800)
    c = dict(M=10000, no_filter=False, wm=800, hm=800)
    inp = synth.synth_ref_inputs(scene, 0, cert_family="T", seed=31)
    U = np.random.RandomState(900).random_sample(3 * c["M"])
    res = G.run_oracle_ref(scene, inp, c, uniforms=U)
    g = G.run_gpu(engine, scene, [inp], G.path_cfg(c), uniforms=U[None, :], weight_sums=[res.taps["s"]])
    rep = G.compare_ref(g, 0, res, c, scene)
    _report("precise/1280/4nn/T", rep)
    assert rep.ok(), rep
    assert rep.sel_exact or rep.sel_tie_swaps > 0
    assert g.uniforms_used[0] == res.taps["uniforms_used"] and g.rounds[0] == res.taps["rounds"]


def test_config4_roi_8_neighbours_no_filter(engine):
    """BASELINE config 4 shape: 8 neighbours per reference, 'No Filter' raw output path (top-M by certainty, finite-only keep)."""
    from lichtfeld_densification_plugin_b200 import synth
    scene = synth.make_scene(40, "fast", ref_fraction=0.05, nn=8)
    c = dict(M=10000, no_filter=True, wm=scene.w_match, hm=scene.h_match)
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family="T", seed=33) for rp in range(scene.n_refs)]
    g = G.run_gpu(engine, scene, inputs, G.path_cfg(c))
    for r, inp in enumerate(inputs):
        assert len(inp["nbr_indices"]) == 8
        res = G.run_oracle_ref(scene, inp, c)
        rep = G.compare_ref(g, r, res, c, scene)
        _report(f"roi/8nn/no_filter/ref{r}", rep)
        assert rep.ok(), rep
        assert np.array_equal(g.sel_idx[r], res.sel_idx)          # tie-free certainties: even the order is pinned
        order = G.expected_pack_order(g.flags[r])
        assert np.array_equal(g.xyz[r], g.xyzerr[r][order, :3])


def test_config5_base_640_sharding_invariance(engine):
    """BASELINE config 5 shape ('base' 640x640, 4 neighbours): a view's result does not depend on which views share
    its launch, so sharding the reference list over ranks and concatenating in rank order equals the single-GPU run."""
    from lichtfeld_densification_plugin_b200 import synth
    from lichtfeld_densification_plugin_b200 import distributed as D
    scene = synth.make_scene(48, "base", ref_fraction=0.125, nn=4)
    c = dict(M=10000, no_filter=False, wm=scene.w_match, hm=scene.h_match)
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family="R", seed=35) for rp in range(scene.n_refs)]
    streams = list(range(scene.n_refs))
    whole = G.run_gpu(engine, scene, inputs, G.path_cfg(c, seed=9), rng_streams=streams)
    for world in (2, 3):
        xyz = []
        for rank in range(world):
            lo, hi = D.shard_bounds(len(inputs), rank, world)
            part = G.run_gpu(engine, scene, inputs[lo:hi], G.path_cfg(c, seed=9), rng_streams=streams[lo:hi])
            xyz += part.xyz
        assert len(xyz) == len(whole.xyz)
        for a, b in zip(xyz, whole.xyz):
            assert np.array_equal(a, b)


@pytest.mark.parametrize("case", list(range(24)) + [34, 38, 44])      # 34 / 38 / 44: maps 36 px wide, coverage tiles of ONE pixel
def test_randomised_shapes(engine, case):
    """Seeded random shapes through every kernel variant (vector / scalar rows, every column mode of the prep kernel,
    ragged neighbour counts, map != match resolution, small and binding coverage budgets) against the oracle."""
    from lichtfeld_densification_plugin_b200 import synth
    rs = np.random.RandomState(1000 + case)
    H = int(rs.choice([40, 57, 64, 96, 128, 150, 33, 200]))
    W = int(rs.choice([48, 61, 64, 100, 128, 256, 52, 36]))
    hm = int(rs.choice([H, max(16, H // 2), H + 7]))
    wm = int(rs.choice([W, max(16, W // 2), W + 5]))
    nn = int(rs.randint(1, 9)) if case >= 10 else int(rs.randint(1, 6))
    M = int(rs.choice([50, 400, 1500, min(4000, H * W // 3)])) if case < 10 else int(rs.choice([8, 123, 900, 2500, H * W // 2]))
    fam = "T" if case % 3 else "R"
    no_filter = bool(case in (7, 15, 21))
    scene = synth.make_scene(10, "turbo", ref_fraction=0.2, nn=nn)
    scene.H, scene.W, scene.h_match, scene.w_match = H, W, hm, wm
    c = dict(M=M, no_filter=no_filter, wm=wm, hm=hm, sampson=float(rs.choice([5.0, 0.0])), parallax=float(rs.choice([0.5, 0.0])))
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family=fam, seed=200 + case) for rp in range(scene.n_refs)]
    tile = max(1, W // 24)
    if -(-W // tile) * -(-H // tile) > 4096 and not no_filter:
        # documented limit of the C ABI (LDP_MAX_BINS coverage tiles; tile = max(1, W // 24), so only maps narrower than
        # 48 px with thousands of rows get there): refused loudly, never computed wrongly
        from lichtfeld_densification_plugin_b200._native import NativeLibraryError
        with pytest.raises(NativeLibraryError, match="too many coverage tiles"):
            G.run_gpu(engine, scene, inputs, G.path_cfg(c))
        return
    U = np.stack([np.random.RandomState(case * 10 + r).random_sample(3 * M + 64) for r in range(len(inputs))])
    ress = [G.run_oracle_ref(scene, inp, c, uniforms=U[r]) for r, inp in enumerate(inputs)]
    g = G.run_gpu(engine, scene, inputs, G.path_cfg(c), uniforms=None if no_filter else U,
                  weight_sums=None if no_filter else [res.taps["s"] if res is not None else 0.0 for res in ress])
    for r, res in enumerate(ress):
        if res is None:
            assert g.xyz[r].shape[0] == 0
            continue
        rep = G.compare_ref(g, r, res, c, scene)
        _report(f"random{case}/{H}x{W}/m{hm}x{wm}/nn{nn}/M{M}/{fam}/ref{r}", rep)
        assert rep.ok(), (case, H, W, hm, wm, nn, M, fam, rep)
        if not no_filter:
            assert g.uniforms_used[r] == res.taps["uniforms_used"] and g.rounds[r] == res.taps["rounds"]


def test_neighbours_with_their_own_camera_sizes(engine):
    """SURVEY 8g: the pixel scales of a neighbour use ITS camera's (width, height) (core/pipeline.py:697-699); here every
    third camera is a different sensor (other size, other intrinsics), as neighbour and as reference view."""
    from lichtfeld_densification_plugin_b200 import synth
    from lichtfeld_densification_plugin_b200.core.camera_models import CameraRecord
    scene = synth.make_scene(16, "turbo", ref_fraction=0.25, nn=3)
    for i, cam in enumerate(scene.cameras):
        if i % 3 == 1:
            w2, h2 = 973, 1111
            K2 = np.array([[0.9 * w2, 0.0, w2 / 2.0 + 3.0], [0.0, 0.85 * w2, h2 / 2.0 - 2.0], [0.0, 0.0, 1.0]], dtype=np.float32)
            scene.cameras[i] = CameraRecord.from_KRt(cam.uid, w2, h2, K2, cam.R, cam.t, image_path=cam.image_path)
    c = dict(M=6000, no_filter=False, wm=scene.w_match, hm=scene.h_match)
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family="T", seed=33) for rp in range(scene.n_refs)]
    sizes = {(scene.cameras[j].width, scene.cameras[j].height) for inp in inputs for j in list(inp["nbr_indices"]) + [inp["ref_index"]]}
    assert len(sizes) == 2
    U = np.stack([np.random.RandomState(900 + r).random_sample(3 * c["M"]) for r in range(len(inputs))])
    ress = [G.run_oracle_ref(scene, inp, c, uniforms=U[r], collect_debug=True) for r, inp in enumerate(inputs)]
    g = G.run_gpu(engine, scene, inputs, G.path_cfg(c), uniforms=U, weight_sums=[res.taps["s"] for res in ress], collect_debug=True)
    for r in range(len(inputs)):
        rep = G.compare_ref(g, r, ress[r], c, scene)
        _report(f"mixed-sensors/ref{r}", rep)
        assert rep.ok(), rep
        assert rep.n_kept_ref > 1000
