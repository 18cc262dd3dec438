"""GPU: the kernel instantiations and launch branches that users can reach but the shapes of the other suites do not.

A. Neighbour counts 5-16: ldp_stream_kernel<0, *> (the generic neighbour count, and raw planes at nn >= 5), the 16-slot
   group tables of the geometry, fix and pack kernels, multiview masks above bit 7, the last lens-table entries.
B. Maps above 2^19 pixels: chunk_shift 6 and 7, chunk_shift >= 8 (ldp_prep_kernel<0, *>, chunk sums accumulated with f64
   atomics), each in every column mode of the prep kernel.

Every test holds the kernels to the oracle with the bars of tests/gpu_harness.py: samples, uniforms consumed and rounds
exact; keep masks exact up to the solver-noise flips compare_ref admits; xyz / rgb within the harness tolerances; group
order and counts and the pack order exact.
"""
import dataclasses
import json
import time

import numpy as np
import pytest
import torch

from lichtfeld_densification_plugin_b200 import synth
from oracle import densify_oracle as O
from tests import gpu_harness as G
from tests.test_gpu_lens import _compare as lens_compare, _oracle as lens_oracle_ref
from tests.test_gpu_multiview import _vs_oracle as multiview_vs_oracle

pytestmark = pytest.mark.gpu

MAX_NN = 16                      # LDP_MAX_NN (include/ldp_b200.h)
OPENCV = ("OPENCV", [-0.12, 0.03, 4e-4, -3e-4])
FISHEYE = ("OPENCV_FISHEYE", [0.05, -0.01, 0.003, -0.0005])


@pytest.fixture(scope="module")
def engine():
    from lichtfeld_densification_plugin_b200.engine import DensifyEngine
    return DensifyEngine(torch.device("cuda", 0))


# ---- host rules restated ----------------------------------------------------------------------------------------------------
def chunk_shift(H: int, W: int, tiles: int = 24) -> int:
    """make_plan's chunk size, log2 (ldp_api.cu:181-201): the smallest shift >= 5 whose draw-kernel prefix table fits the
    200 KB shared-memory budget.  The kernels switch to atomic chunk sums (and ldp_prep_kernel<0, *>) above 7."""
    N = H * W
    cs = 5
    while True:
        nchunk = (N + (1 << cs) - 1) >> cs
        ept = 8 * ((nchunk + 8 * 1024 - 1) // (8 * 1024))          # KD_THREADS = 1024
        pre_cap = ept * 1024 // 8 * 10 + 16
        ng = 1
        while ng * 2 <= nchunk // 2:
            ng *= 2
        if pre_cap * 8 + (ng + 2) * 4 + 16 <= 200 * 1024:
            return cs
        cs += 1


def prep_cols(H: int, W: int, tiles: int = 24) -> str:
    """launch_sample's column mode of ldp_prep_kernel: QUAD when every quad lies in one row and in at most two tiles whose
    columns umulhi(x, t_magic32) finds exactly; CONST when W also divides the 1024-pixel pass stride; PIXEL otherwise."""
    tile = max(1, W // tiles)
    if W % 4 or tile == 1 or (W - 1) * tile >= 1 << 32:
        return "PIXEL"
    return "CONST" if 1024 % W == 0 else "QUAD"


def topm_generic(H: int, W: int, M: int) -> bool:
    """launch_sample's no-filter choice (ldp_api.cu:363-370): the one-CTA sort buffer over the 200 KB budget takes
    ldp_topm_generic_kernel."""
    N = H * W
    n2 = 1
    while n2 < min(M, N):
        n2 <<= 1
    n4 = ((N + 255) // 256 * 256) // 4
    return max(n2, min(n2, 1024)) * 8 + (((n4 + 31) & ~31) // 32) * 4 > 200 * 1024


def test_host_rules_restated():
    assert chunk_shift(1280, 1280) == 7 and chunk_shift(512, 512) == 5       # the largest / the bench map of the other suites
    assert chunk_shift(1536, 1536) == 8 and chunk_shift(2048, 2048) == 8 and chunk_shift(2560, 2560) == 9
    assert prep_cols(512, 512) == "CONST"
    assert prep_cols(640, 640) == "QUAD" and prep_cols(64, 8448) == "QUAD"
    assert all(prep_cols(H, W) == "PIXEL" for H, W in ((50, 61), (40, 36), (1001, 1001), (1281, 1279), (8, 327680)))
    assert prep_cols(64, 2, tiles=1) == "PIXEL"           # W divides the stride, but a quad spans two rows


# ---- comparison against the oracle --------------------------------------------------------------------------------------------
def _uniforms(R, M, seed):
    return np.stack([np.random.RandomState(seed + r).random_sample(3 * M + 64) for r in range(R)])


def _check_groups(g: G.GpuRun, r: int, res, rep: G.ParityReport, scene, inp, tag):
    """Pack order against the taps, and group order and counts against the oracle's first-appearance groups."""
    order = G.expected_pack_order(g.flags[r])
    assert np.array_equal(g.xyz[r], g.xyzerr[r][order, :3]), tag
    assert np.array_equal(g.err[r], g.xyzerr[r][order, 3]), tag
    counts = g.group_count.reshape(-1, MAX_NN)[r]
    gorder = [int(x) for x in g.group_order.reshape(-1, MAX_NN)[r] if x >= 0]
    grp = (g.flags[r] >> 2).astype(np.int64)
    keep = (g.flags[r] & 1).astype(bool)
    for k in range(MAX_NN):                     # counts agree with the per-sample flags
        assert counts[k] == int((keep & (grp == k)).sum()), (tag, k)
    if rep.keep_flips or not rep.sel_exact:
        return
    uids = [scene.cameras[j].uid for j in inp["nbr_indices"]]
    want_order, want_count = [], np.zeros(MAX_NN, dtype=np.int64)
    for gt in res.taps["groups"]:
        k = uids.index(gt["uid"])
        n = int(gt["keep"].sum()) if "pos" in gt else 0
        want_count[k] = n
        if n:
            want_order.append(k)
    assert [k for k in gorder if counts[k] > 0] == want_order, tag
    assert np.array_equal(counts.astype(np.int64), want_count), tag


def _check_debug(g: G.GpuRun, r: int, res, scene, inp, tag):
    """collect_debug: the kernel's matches and certainties, split by group, equal the oracle's per-neighbour arrays."""
    uids = [scene.cameras[j].uid for j in inp["nbr_indices"]]
    counts = g.group_count.reshape(-1, MAX_NN)[r]
    pos, seen = 0, []
    for gid in g.group_order.reshape(-1, MAX_NN)[r]:
        if gid < 0:
            break
        cnt = int(counts[gid])
        if cnt:
            uid = uids[gid]
            seen.append(uid)
            dm, dc = g.dbg_matches[r][pos:pos + cnt], g.dbg_cert[r][pos:pos + cnt]
            assert np.array_equal(dm, res.debug_matches_by_nbr[uid]), (tag, uid, float(np.abs(dm - res.debug_matches_by_nbr[uid]).max()))
            assert np.array_equal(dc, res.debug_cert_by_nbr[uid]), (tag, uid)
        pos += cnt
    assert seen == list(res.debug_matches_by_nbr.keys()), tag
    assert seen and max(uids.index(u) for u in seen) >= 8 or len(uids) <= 8, tag      # groups above 8 reached


def _vs_oracle(engine, scene, inputs, c, tag, cfg=None, collect_debug=False, seed=900):
    """Oracle on every view (its CPU seconds reported), one GPU launch, every bar of the harness."""
    R = len(inputs)
    nf = c["no_filter"]
    U = None if nf else _uniforms(R, c["M"], seed)
    t0 = time.process_time()
    ress = [G.run_oracle_ref(scene, inp, c, uniforms=None if nf else U[r], collect_debug=collect_debug) for r, inp in enumerate(inputs)]
    cpu = time.process_time() - t0
    g = G.run_gpu(engine, scene, inputs, cfg or G.path_cfg(c), uniforms=U, collect_debug=collect_debug,
                  weight_sums=None if nf else [res.taps["s"] if res is not None else 0.0 for res in ress])
    flips = 0
    for r, res in enumerate(ress):
        if res is None:
            assert g.xyz[r].shape[0] == 0, tag
            continue
        rep = G.compare_ref(g, r, res, c, scene)
        flips += len(rep.keep_flips)
        print(f"[reach] {tag}/ref{r} nn={len(inputs[r]['nbr_indices'])}: S={rep.n_samples} sel_exact={rep.sel_exact} "
              f"kept gpu/ref={rep.n_kept_gpu}/{rep.n_kept_ref} flips={len(rep.keep_flips)} max_xyz_rel={rep.max_xyz_rel:.2e}")
        for f in rep.keep_flips[:5]:
            print("   flip:", json.dumps(f))
        assert rep.ok(), (tag, r, rep)
        assert rep.n_kept_gpu > 0, (tag, r)
        if not nf:
            assert g.uniforms_used[r] == res.taps["uniforms_used"] and g.rounds[r] == res.taps["rounds"], (tag, r)
        _check_groups(g, r, res, rep, scene, inputs[r], tag)
        if collect_debug and not rep.keep_flips:
            _check_debug(g, r, res, scene, inputs[r], tag)
    print(f"[reach] {tag}: oracle {cpu:.1f} CPU s, admitted flips {flips}, fix-up entries {g.fixups}")
    return g, ress


def _scene(nn, n_views=24, ref_fraction=0.1, setting="turbo", **kw):
    return synth.make_scene(n_views, setting, ref_fraction=ref_fraction, nn=nn, **kw)


def _inputs(scene, fam="T", seed=41, **kw):
    return [synth.synth_ref_inputs(scene, rp, cert_family=fam, seed=seed, **kw) for rp in range(scene.n_refs)]


def _trim(inp, k):
    """The same view with only its first k neighbours."""
    return dict(inp, cert=inp["cert"][:k], warp=inp["warp"][:k], nbr_indices=list(inp["nbr_indices"][:k]))


# ---- A. neighbour counts 5-16 -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("filters", ["on", "off"])
@pytest.mark.parametrize("fam", ["R", "T"])
@pytest.mark.parametrize("nn", [9, 10, 12, 16])
def test_neighbour_counts_vs_oracle(engine, nn, fam, filters):
    """ldp_stream_kernel<0, 0> and the 16-slot group tables, with the Sampson gate and parallax test on and off."""
    scene = _scene(nn)
    assert scene.nn == nn
    f = 1.0 if filters == "on" else 0.0
    c = dict(M=6000, no_filter=False, wm=scene.w_match, hm=scene.h_match, sampson=5.0 * f, parallax=0.5 * f)
    inputs = _inputs(scene, fam=fam, seed=60 + nn)
    g, _ = _vs_oracle(engine, scene, inputs, c, f"nn{nn}/{fam}/filters-{filters}")
    # neighbour slots 8.. win samples and keep points
    assert any(((f_ >> 2) >= 8).any() for f_ in g.flags), "no sample was won by a neighbour above slot 7"


def test_ragged_neighbour_lists_in_one_launch(engine):
    """Views with 1, 7, 9 and 16 neighbours in one launch (nn_max = 16)."""
    scene = _scene(16, n_views=20, ref_fraction=0.2)
    inputs = [_trim(inp, k) for inp, k in zip(_inputs(scene, fam="R", seed=71), (1, 7, 9, 16))]
    assert [len(i["nbr_indices"]) for i in inputs] == [1, 7, 9, 16]
    c = dict(M=6000, no_filter=False, wm=scene.w_match, hm=scene.h_match)
    _vs_oracle(engine, scene, inputs, c, "ragged")


def test_collect_debug_at_16_neighbours(engine):
    scene = _scene(16)
    c = dict(M=6000, no_filter=False, wm=scene.w_match, hm=scene.h_match)
    _vs_oracle(engine, scene, _inputs(scene, fam="T", seed=72), c, "debug/nn16", collect_debug=True)


def test_no_filter_at_16_neighbours(engine):
    """Also the plain path's fix-up (ldp_fix_kernel<*, false>) with a non-empty worklist: ldp_debug_force_fixup acts on
    multiview launches only, but no_filter keeps grossly inconsistent matches, and some of their two-view solves do not
    converge."""
    scene = _scene(16)
    c = dict(M=6000, no_filter=True, wm=scene.w_match, hm=scene.h_match)
    g, _ = _vs_oracle(engine, scene, _inputs(scene, fam="T", seed=73), c, "no_filter/nn16")
    assert g.fixups > 0


@pytest.mark.parametrize("warped", [True, False], ids=["warped-masks", "reference-mask-only"])
@pytest.mark.parametrize("nn", [5, 8, 9, 16])
def test_raw_planes_vs_stage_and_oracle(engine, nn, warped):
    """Raw matcher planes at nn >= 5 (ldp_stream_kernel<0, 1> / <0, 2>): the fused path equals the certainty stage plus
    the plain path on every output; the stage equals the oracle's certainty_prologue; the plain path equals the oracle."""
    scene = _scene(nn)
    hm, wm = scene.h_match, scene.w_match
    floor = 0.25
    rs = np.random.RandomState(80 + nn)
    inputs = _inputs(scene, fam="R", seed=74)
    for i, inp in enumerate(inputs):
        inp["cert"] = inp["cert"] - 0.1 * torch.rand(inp["cert"].shape, generator=torch.Generator().manual_seed(10 * nn + i))
        inp["mask_a"] = (rs.random_sample((hm, wm)) > 0.15).astype(np.uint8)
        inp["masks_b"] = [(rs.random_sample((hm, wm)) > 0.2).astype(np.uint8) if k % 3 != 1 else None for k in range(nn)] if warped else None
    c = dict(M=6000, no_filter=False, wm=wm, hm=hm)
    dev = engine.device
    batch = engine.new_batch(scene.H, scene.W, wm, hm)
    to_dev = lambda m: None if m is None else torch.from_numpy(np.ascontiguousarray(m)).to(dev)
    for inp in inputs:
        cert, warp = inp["cert"].to(dev), inp["warp"].to(dev)
        batch.add([cert[k] for k in range(nn)], [warp[k] for k in range(nn)], inp["image"].to(dev), scene.cameras[inp["ref_index"]],
                  [scene.cameras[j] for j in inp["nbr_indices"]], mask_a=to_dev(inp["mask_a"]),
                  masks_b=[to_dev(m) for m in inp["masks_b"]] if warped else None)
    assert batch.has_warped_masks == warped
    post_planes = engine.postprocess_certainty(batch, floor).cpu()
    for i, inp in enumerate(inputs):
        mbs = inp["masks_b"] if warped else [None] * nn
        for k in range(nn):
            want = O.certainty_prologue(inp["cert"][k].numpy(), inp["warp"][k].numpy(), inp["mask_a"], mbs[k], floor)
            assert np.array_equal(post_planes[i, k].numpy(), want, equal_nan=True), (nn, warped, i, k)
    post = [dict(inp, cert=post_planes[i, :nn], mask_a=None, masks_b=None) for i, inp in enumerate(inputs)]
    plain, ress = _vs_oracle(engine, scene, post, c, f"raw/nn{nn}/warped={warped}")
    U = _uniforms(len(inputs), c["M"], 900)
    s = [res.taps["s"] for res in ress]
    fused = G.run_gpu(engine, scene, inputs, dataclasses.replace(G.path_cfg(c), certainty_floor=floor), uniforms=U, weight_sums=s)
    for r in range(len(inputs)):
        for name in ("sel_idx", "flags", "xyzerr", "xyz", "rgb", "err"):
            assert getattr(fused, name)[r].tobytes() == getattr(plain, name)[r].tobytes(), (nn, warped, r, name)
    for name in ("uniforms_used", "rounds", "weight_sum", "group_order", "group_count", "status"):
        assert getattr(fused, name).tobytes() == getattr(plain, name).tobytes(), (nn, warped, name)


@pytest.mark.parametrize("nn", [10, 16])
def test_multiview_masks_above_bit_7(engine, nn):
    """Multi-view refinement against tests/multiview_oracle.py: view masks exact (up to the solve's own threshold
    margin, as in test_gpu_multiview), including the bits of neighbour slots 8 and up."""
    scene = _scene(nn, ref_fraction=0.125)
    c = dict(M=6000, no_filter=False, wm=scene.w_match, hm=scene.h_match)
    inputs = _inputs(scene, fam="T", seed=75)
    g = multiview_vs_oracle(engine, scene, inputs, c, f"multiview/nn{nn}")
    vm = np.concatenate(g["view_mask"]).astype(np.int64)
    high = int(((vm >> 8) != 0).sum())
    n_views = max(bin(int(m)).count("1") for m in vm) + 1              # the reference view counts
    print(f"[reach] multiview/nn{nn}: points with a view above slot 7: {high}, most cameras on one point: {n_views}")
    if nn == 16:
        assert high > 0


def test_lens_cameras_at_16_neighbours(engine):
    """OPENCV and fisheye cameras mixed with pinhole ones at nn = 16 (every lens-table slot) against the lens oracle."""
    lens = [[OPENCV, None, FISHEYE][v % 3] for v in range(24)]
    scene = _scene(16, lens=lens)
    c = dict(M=6000, no_filter=False, wm=scene.w_match, hm=scene.h_match)
    inputs = _inputs(scene, fam="T", seed=76)
    U = _uniforms(len(inputs), c["M"], 700)
    t0 = time.process_time()
    ress = [lens_oracle_ref(scene, inp, c, U[r]) for r, inp in enumerate(inputs)]
    cpu = time.process_time() - t0
    g = G.run_gpu(engine, scene, inputs, G.path_cfg(c), uniforms=U, weight_sums=[res.taps["s"] for res in ress])
    for r in range(len(inputs)):
        lens_compare(g, r, ress[r], c, scene, f"lens/nn16/ref{r}")
        assert ((g.flags[r] >> 2) >= 8).any()
    print(f"[reach] lens/nn16: oracle {cpu:.1f} CPU s")


# ---- B. large maps ----------------------------------------------------------------------------------------------------------
LARGE = [(1536, 1536, 8, "QUAD"), (2048, 2048, 8, "QUAD"), (2560, 2560, 9, "QUAD"), (64, 8448, 6, "QUAD"),
         (1024, 1024, 6, "CONST"), (1536, 1024, 7, "CONST"), (2304, 1024, 8, "CONST"),
         (1001, 1001, 6, "PIXEL"), (1281, 1279, 7, "PIXEL"), (8, 327680, 8, "PIXEL")]


@pytest.mark.parametrize("H,W,cs,cols", LARGE, ids=[f"{h}x{w}" for h, w, _, _ in LARGE])
def test_large_maps_vs_oracle(engine, H, W, cs, cols):
    """chunk_shift >= 8 (ldp_prep_kernel<0, *>, atomic chunk sums, wide in-chunk scans), and every column mode of
    ldp_prep_kernel at chunk_shift 6, 7 and >= 8, which the maps of the other suites do not reach.  64x8448 is QUAD above
    8192 columns; 8x327680 is PIXEL because (W - 1) * tile passes 2^32 there."""
    assert chunk_shift(H, W) == cs and prep_cols(H, W) == cols
    scene = _scene(4, n_views=10)
    scene.H, scene.W = H, W
    c = dict(M=10000, no_filter=False, wm=scene.w_match, hm=scene.h_match)
    inputs = _inputs(scene, fam="R", seed=77)
    _vs_oracle(engine, scene, inputs, c, f"large/{H}x{W}/cs{cs}")


def test_large_map_no_filter(engine):
    H = W = 2048
    assert chunk_shift(H, W) == 8 and topm_generic(H, W, 10000)          # ldp_topm_generic_kernel, by the size alone
    scene = _scene(4, n_views=10)
    scene.H, scene.W = H, W
    c = dict(M=10000, no_filter=True, wm=scene.w_match, hm=scene.h_match)
    _vs_oracle(engine, scene, _inputs(scene, fam="T", seed=78), c, "large/no_filter/2048")
