"""GPU: cameras with a lens model (CameraRecord.lens_model, include/ldp_b200.h: ldp_lens) through the device path, against the
lens oracle (tests/lens_oracle.py), against ground truth, and beside pinhole cameras in the same launch."""
import json

import numpy as np
import pytest
import torch

from lichtfeld_densification_plugin_b200 import synth
from lichtfeld_densification_plugin_b200.core.camera_models import CameraRecord
from tests import gpu_harness as G
from tests import lens_oracle as LO
from tests.golden import make_lens_golden as LG
from tests.helpers import oracle_cam

pytestmark = pytest.mark.gpu

OPENCV = ("OPENCV", [-0.12, 0.03, 4e-4, -3e-4])
FULL_OPENCV = ("FULL_OPENCV", [0.2, -0.05, 4e-4, -3e-4, 0.01, 0.25, -0.03, 0.01])
FISHEYE = ("OPENCV_FISHEYE", [0.05, -0.01, 0.003, -0.0005])
RADIAL = ("SIMPLE_RADIAL", [-0.12])


@pytest.fixture(scope="module")
def engine():
    from lichtfeld_densification_plugin_b200.engine import DensifyEngine
    return DensifyEngine()


def _strip(cam: CameraRecord) -> CameraRecord:
    """The same camera without its lens (what the reference would triangulate)."""
    return CameraRecord.from_KRt(cam.uid, cam.width, cam.height, cam.K, cam.R, cam.t, image_path=cam.image_path)


# ---- 1. lens and pinhole views in one launch --------------------------------------------------------------------------------
def test_pinhole_views_bit_identical_in_a_lens_launch(engine):
    lens = [OPENCV, FISHEYE, FULL_OPENCV, RADIAL] + [None] * 8
    scene = synth.make_scene(12, "fast", ref_fraction=1.0, nn=2, lens=lens)
    pin = [i for i in range(scene.n_refs)
           if all(scene.cameras[j].lens_model is None for j in [scene.refs_local[i], *scene.nn_table[scene.refs_local[i]][:2]])]
    assert len(pin) >= 4
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family="R", seed=5) for rp in range(scene.n_refs)]
    cfg = G.path_cfg(dict(M=6000, no_filter=False))
    mixed = G.run_gpu(engine, scene, inputs, cfg)
    alone = G.run_gpu(engine, scene, [inputs[i] for i in pin], cfg)
    for j, i in enumerate(pin):
        for f in ("sel_idx", "flags", "xyzerr", "xyz", "rgb", "err"):
            a, b = getattr(mixed, f)[i], getattr(alone, f)[j]
            assert a.tobytes() == b.tobytes(), (i, f)
        assert mixed.group_order[i].tolist() == alone.group_order[j].tolist()
        assert mixed.group_count[i].tolist() == alone.group_count[j].tolist()
    lensed = [i for i in range(scene.n_refs) if i not in pin]
    assert sum(mixed.xyz[i].shape[0] for i in lensed) > 1000


# ---- 2. ldp_undistort_points vs the oracle ----------------------------------------------------------------------------------
def _f32_ulps(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    ia = a.view(np.int32).astype(np.int64)
    ib = b.view(np.int32).astype(np.int64)
    ia = np.where(ia < 0, -(ia & 0x7FFFFFFF), ia)
    ib = np.where(ib < 0, -(ib & 0x7FFFFFFF), ib)
    return np.abs(ia - ib)


@pytest.mark.parametrize("name", list(LG.CASES) + ["FOLD", "WIDE_FISHEYE"])
def test_undistort_entry_point_vs_oracle(engine, name):
    if name == "FOLD":       # strong barrel distortion: the outer image lies past the fold (NaN)
        rec = CameraRecord.from_colmap(0, "RADIAL", [LG.FOCAL, LG.WIDTH / 2, LG.HEIGHT / 2, -0.9, 0.05], LG.WIDTH, LG.HEIGHT,
                                       np.eye(3), np.zeros(3))
    elif name == "WIDE_FISHEYE":   # short focal length: distorted radii up to ~2.3, past pi/2 and past theta_d(pi/2) = 1.71
        rec = CameraRecord.from_colmap(0, "OPENCV_FISHEYE", [350.0, 350.0, LG.WIDTH / 2, LG.HEIGHT / 2] + LG.CASES["OPENCV_FISHEYE"],
                                       LG.WIDTH, LG.HEIGHT, np.eye(3), np.zeros(3))
    else:
        rec = LG.record(name)
    rng = np.random.default_rng(11)
    n = 1 << 20
    uv = rng.uniform([-0.25 * LG.WIDTH, -0.25 * LG.HEIGHT], [1.25 * LG.WIDTH, 1.25 * LG.HEIGHT], size=(n, 2)).astype(np.float32)
    got = engine.undistort_pixels(torch.from_numpy(uv).to(engine.device), rec).cpu().numpy()
    want = LO.undistort_px(LO.lens_of(rec), uv)
    nan_g, nan_w = np.isnan(got).any(axis=1), np.isnan(want).any(axis=1)
    assert np.array_equal(nan_g, nan_w), (name, int((nan_g != nan_w).sum()))
    fin = ~nan_w
    ulps = _f32_ulps(got[fin], want[fin])
    at1 = np.nonzero(ulps.max(axis=1) == 1)[0]
    print(f"[undistort] {name}: n={n} NaN={int(nan_w.sum())} at 1 ulp={at1.size} max ulp={int(ulps.max()) if ulps.size else 0}")
    for i in at1[:5]:
        print("   1 ulp:", uv[fin][i].tolist(), got[fin][i].tolist(), want[fin][i].tolist())
    assert ulps.max() <= 1
    if name == "FOLD":
        assert nan_w.sum() > 1000
    if name == "WIDE_FISHEYE":   # beyond 90 degrees: NaN; between pi/2 and theta_d(pi/2): a valid ray
        rd = np.hypot((uv[:, 0].astype(np.float64) - LG.WIDTH / 2) / 350.0, (uv[:, 1].astype(np.float64) - LG.HEIGHT / 2) / 350.0)
        band = (rd > 1.58) & (rd < 1.70)
        assert band.sum() > 1000 and not nan_g[band].any() and nan_g[rd > 1.72].all()
    # a pinhole record is passed through
    pin = _strip(rec)
    assert np.array_equal(engine.undistort_pixels(torch.from_numpy(uv[:1000]).to(engine.device), pin).cpu().numpy(), uv[:1000])


# ---- 3. parity with the lens oracle --------------------------------------------------------------------------------------
def _oracle(scene, inp, c, uniforms):
    cams = scene.cameras
    nb = inp["nbr_indices"]
    return LO.triangulate_ref_lens([inp["cert"][k] for k in range(len(nb))], [inp["warp"][k] for k in range(len(nb))],
                                   inp["image"].numpy(), oracle_cam(cams[inp["ref_index"]]), [oracle_cam(cams[j]) for j in nb],
                                   G.oracle_cfg(c), LO.lens_of(cams[inp["ref_index"]]), [LO.lens_of(cams[j]) for j in nb],
                                   uniforms=uniforms)


def _explain(gt, j, c, ref_C, nbr_C):
    """The exactly solved point (f64 SVD of the f32 DLT matrix, rounded once to f32) under the oracle's filter code: how far
    it lies from the reprojection and parallax thresholds."""
    P1, P2 = gt["P1"], gt["P2"]
    uvA, uvB = gt["uvA"][j], gt["uvB"][j]
    A = np.stack([uvA[0] * P1[2] - P1[0], uvA[1] * P1[2] - P1[1], uvB[0] * P2[2] - P2[0], uvB[1] * P2[2] - P2[1]]).astype(np.float32)
    v = np.linalg.svd(A.astype(np.float64))[2][-1]
    X = np.repeat(np.concatenate([(v[:3] / v[3]).astype(np.float32), np.ones(1, np.float32)])[None], 256, axis=0)
    e = float(np.maximum(LO.reprojection_error(P1, X, np.repeat(gt["uvA_obs"][j:j + 1], 256, 0), gt.get("ref_lens")),
                         LO.reprojection_error(P2, X, np.repeat(gt["uvB_obs"][j:j + 1], 256, 0), gt["lensB"]))[0])
    thr = float(np.float32(c.get("reproj", 0.8)))
    out = {"err_exact": e, "dist_reproj": abs(e - thr)}
    near = abs(e - thr) < G.NEAR_REPROJ
    if c.get("parallax", 0.5) > 0:
        a, b = X[0, :3].astype(np.float64) - ref_C, X[0, :3].astype(np.float64) - nbr_C
        ang = float(np.degrees(np.arccos(np.clip(a @ b / (np.linalg.norm(a) * np.linalg.norm(b)), -1, 1))))
        out["dist_parallax_deg"] = abs(ang - c.get("parallax", 0.5))
        near = near or out["dist_parallax_deg"] < G.NEAR_PARALLAX
    out["near"] = bool(near)
    return out


def _compare(g, r, res, c, scene, tag):
    sel = g.sel_idx[r]
    assert np.array_equal(sel, res.sel_idx), tag
    S = sel.size
    keep_r = np.zeros(S, dtype=bool)
    X_r = np.full((S, 3), np.nan)
    e_r = np.full(S, np.nan)
    loc = {}
    for gt in res.taps["groups"]:
        if "pos" in gt:
            gt["ref_lens"] = res.taps["ref_lens"]
            keep_r[gt["pos"]] = gt["keep"]
            X_r[gt["pos"]] = gt["X"][:, :3]
            e_r[gt["pos"]] = gt["err"]
            for j, p in enumerate(gt["pos"]):
                loc[int(p)] = (gt, j)
    keep_g = (g.flags[r] & 1).astype(bool)
    xe = g.xyzerr[r].astype(np.float64)
    cams = {cam.uid: cam for cam in scene.cameras}
    flips = []
    for i in np.nonzero(keep_g != keep_r)[0]:
        if int(i) not in loc:          # the oracle's Sampson gate dropped it
            flips.append(dict(sample=int(i), keep_gpu=bool(keep_g[i]), sampson_side=True, near=False))
            continue
        gt, j = loc[int(i)]
        info = _explain(gt, j, c, cams[res.taps["ref_uid"]].C.astype(np.float64), cams[gt["uid"]].C.astype(np.float64))
        info.update(sample=int(i), keep_gpu=bool(keep_g[i]), err_gpu=float(xe[i, 3]), err_ref=float(e_r[i]))
        flips.append(info)
    judge = (keep_r | keep_g) & np.isfinite(X_r).all(axis=1) & np.isfinite(xe[:, :3]).all(axis=1)
    # the oracle's f32 LAPACK point must itself be within half the tolerance of the f64 answer (else: listed, not judged)
    stable = np.zeros(S, dtype=bool)
    for i in np.nonzero(judge)[0]:
        gt, j = loc[int(i)]
        P1, P2, uvA, uvB = gt["P1"], gt["P2"], gt["uvA"][j], gt["uvB"][j]
        A = np.stack([uvA[0] * P1[2] - P1[0], uvA[1] * P1[2] - P1[1], uvB[0] * P2[2] - P2[0], uvB[1] * P2[2] - P2[1]]).astype(np.float32)
        v = np.linalg.svd(A.astype(np.float64))[2][-1]
        X64 = v[:3] / v[3]
        stable[i] = bool((np.abs(X_r[i] - X64) <= 0.5 * (G.XYZ_ATOL + G.XYZ_RTOL * np.abs(X64))).all())
    unstable = int((judge & ~stable).sum())
    judge &= stable
    dx = np.abs(xe[judge, :3] - X_r[judge])
    xyz_viol = int((dx > G.XYZ_ATOL + G.XYZ_RTOL * np.abs(X_r[judge])).any(axis=1).sum())
    de = np.abs(xe[judge, 3] - e_r[judge])
    err_viol = int((de > 1e-3 + 1e-4 * np.abs(e_r[judge])).sum())
    far = [f for f in flips if not f["near"]]
    print(f"[lens parity] {tag}: S={S} kept gpu/ref={int(keep_g.sum())}/{int(keep_r.sum())} flips={len(flips)} far={len(far)} "
          f"unstable_ref={unstable} max_dx={dx.max() if dx.size else 0:.3e} max_derr={de.max() if de.size else 0:.3e}")
    for f in flips[:10]:
        print("   flip:", json.dumps(f))
    assert not far and xyz_viol == 0 and err_viol == 0, tag
    assert int(keep_g.sum()) > 0.2 * S, tag
    order = G.expected_pack_order(g.flags[r])
    assert np.array_equal(g.xyz[r], g.xyzerr[r][order, :3]), tag


def _triangulate_samples(engine, scene, inputs, cfg, sel_idx, n_samples):
    """ldp_triangulate_samples on given sample indices, through the same batch the densify call used."""
    import ctypes as C
    from lichtfeld_densification_plugin_b200 import _native as N
    batch = engine.new_batch(scene.H, scene.W, scene.w_match, scene.h_match)
    dev = engine.device
    for inp in inputs:
        nn = len(inp["nbr_indices"])
        cert, warp = inp["cert"].to(dev), inp["warp"].to(dev)
        batch.add([cert[k] for k in range(nn)], [warp[k] for k in range(nn)], inp["image"].to(dev),
                  scene.cameras[inp["ref_index"]], [scene.cameras[j] for j in inp["nbr_indices"]])
    assert batch.has_lens
    pl = engine.prepare(batch, cfg, taps=True)
    for r, s in enumerate(sel_idx):
        pl.outputs.sel_idx[r, :s.size] = torch.from_numpy(s.astype(np.int32)).to(dev)
    pl.outputs.n_samples.copy_(torch.tensor(n_samples, dtype=torch.int32, device=dev))
    rc = engine.lib.ldp_triangulate_samples(C.byref(pl.params), C.c_void_p(pl.descs_dev.data_ptr()), C.byref(pl.c_outputs),
                                            C.c_void_p(pl.workspace.data_ptr()), C.c_size_t(pl.workspace.numel()),
                                            C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
    N.check(rc, "ldp_triangulate_samples")
    torch.cuda.synchronize()
    out = pl.outputs
    return [(out.sample_flags[r, :n_samples[r]].cpu().numpy(), out.sample_xyzerr[r, :n_samples[r]].cpu().numpy())
            for r in range(len(inputs))]


@pytest.mark.parametrize("case", ["OPENCV", "FULL_OPENCV", "OPENCV_FISHEYE", "mixed", "mixed_nofilter", "mixed_no_sampson"])
def test_parity_with_lens_oracle(engine, case):
    spec = {"OPENCV": OPENCV, "FULL_OPENCV": FULL_OPENCV, "OPENCV_FISHEYE": FISHEYE}.get(case)
    lens = spec if spec is not None else [[OPENCV, None, FISHEYE, RADIAL, FULL_OPENCV, None][v % 6] for v in range(24)]
    scene = synth.make_scene(24, "fast", ref_fraction=0.125, nn=4, lens=lens)
    c = dict(M=10000, no_filter=case == "mixed_nofilter", wm=scene.w_match, hm=scene.h_match)
    if case == "mixed_no_sampson":
        c["sampson"] = 0.0
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family="T", seed=31) for rp in range(scene.n_refs)]
    R = len(inputs)
    U = np.stack([np.random.RandomState(700 + r).random_sample(3 * c["M"] + 64) for r in range(R)])
    ress = [_oracle(scene, inp, c, None if c["no_filter"] else U[r]) for r, inp in enumerate(inputs)]
    sums = [res.taps.get("s", 0.0) for res in ress]
    g = G.run_gpu(engine, scene, inputs, G.path_cfg(c), uniforms=None if c["no_filter"] else U,
                  weight_sums=None if c["no_filter"] else sums)
    for r in range(R):
        _compare(g, r, ress[r], c, scene, f"{case}/ref{r}")
    # the triangulation stage alone on the same samples: the same per-sample results
    stage = _triangulate_samples(engine, scene, inputs, G.path_cfg(c), g.sel_idx, [s.size for s in g.sel_idx])
    for r, (flags, xyzerr) in enumerate(stage):
        assert np.array_equal(flags & 3, g.flags[r] & 3), (case, r)
        fin = np.isfinite(g.xyzerr[r]).all(axis=1) & ((g.flags[r] & 2) > 0)
        assert np.array_equal(xyzerr[fin], g.xyzerr[r][fin]), (case, r)


# ---- 4. ground truth ------------------------------------------------------------------------------------------------------
def _median_dist(engine, scene, inputs, cams):
    sc = synth.SynthScene(cameras=cams, refs_local=scene.refs_local, nn_table=scene.nn_table, H=scene.H, W=scene.W,
                          h_match=scene.h_match, w_match=scene.w_match, nn=scene.nn)
    g = G.run_gpu(engine, sc, inputs, G.path_cfg(dict(M=10000, no_filter=False)))
    d, kept = [], 0
    for r, inp in enumerate(inputs):
        keep = (g.flags[r] & 1).astype(bool)
        truth = inp["points"].reshape(-1, 3).numpy()[g.sel_idx[r][keep]]
        d.append(np.linalg.norm(g.xyzerr[r][keep, :3].astype(np.float64) - truth, axis=1))
        kept += int(keep.sum())
    d = np.concatenate(d)
    return (float(np.median(d)) if d.size else float("inf")), kept


def test_ground_truth_surface(engine):
    """Noise-free scene, k1 = -0.12 on a 1297 x 840 camera (the image corners move by ~60 px).  The factors asserted here
    (lens within 2x of the pinhole twin scene, stripped coefficients at least 10x worse) came from a back-of-envelope
    estimate and hold with a wide margin; measured on a B200: median 3.8e-7 with the lens, 3.5e-7 for the pinhole twin,
    2.5e-2 with the coefficients stripped, where the reprojection filter still kept 28 855 points (36 398 with the lens)."""
    lensed = synth.make_scene(16, "fast", ref_fraction=0.25, nn=3, lens=RADIAL)
    twin = synth.make_scene(16, "fast", ref_fraction=0.25, nn=3)
    kw = dict(cert_family="R", seed=8, noise_sigma=0.0, outlier_frac=0.0, return_points=True)
    inp_l = [synth.synth_ref_inputs(lensed, rp, **kw) for rp in range(lensed.n_refs)]
    inp_t = [synth.synth_ref_inputs(twin, rp, **kw) for rp in range(twin.n_refs)]
    m_lens, k_lens = _median_dist(engine, lensed, inp_l, lensed.cameras)
    m_twin, k_twin = _median_dist(engine, twin, inp_t, twin.cameras)
    m_strip, k_strip = _median_dist(engine, lensed, inp_l, [_strip(cam) for cam in lensed.cameras])
    print(f"[ground truth] median |X - X_true|: lens {m_lens:.3e} ({k_lens} kept), pinhole twin {m_twin:.3e} ({k_twin}), "
          f"coefficients stripped {m_strip:.3e} ({k_strip})")
    assert k_lens > 0.5 * k_twin
    assert m_lens <= 2.0 * max(m_twin, 1e-6)
    assert k_strip == 0 or m_strip >= 10.0 * m_lens


# ---- 5. ring and pipeline -------------------------------------------------------------------------------------------------
def test_ring_and_pipeline_with_lens_records(engine, tmp_path):
    from lichtfeld_densification_plugin_b200.core import pipeline as P
    from lichtfeld_densification_plugin_b200.core.config import DensePipelineConfig
    from lichtfeld_densification_plugin_b200.engine import DensifyRing, PathConfig
    lens = [[OPENCV, FISHEYE, None, RADIAL][v % 4] for v in range(24)]
    scene = synth.make_scene(24, "turbo", ref_fraction=0.5, nn=3, lens=lens)
    cams = scene.cameras
    inputs = [synth.synth_ref_inputs(scene, rp, cert_family="R", seed=12) for rp in range(scene.n_refs)]
    dev = engine.device
    cfg = PathConfig(matches_per_ref=4000)

    def batch_of(eng, views):
        b = eng.new_batch(scene.H, scene.W, scene.w_match, scene.h_match)
        for i in views:
            inp = inputs[i]
            nn = len(inp["nbr_indices"])
            b.add([inp["cert"][k].to(dev) for k in range(nn)], [inp["warp"][k].to(dev) for k in range(nn)], inp["image"].to(dev),
                  cams[inp["ref_index"]], [cams[j] for j in inp["nbr_indices"]], rng_stream=inp["ref_index"])
        return b
    groups = [list(range(q, scene.n_refs, 4)) for q in range(4)]
    one = []
    for views in groups:
        o = engine.densify(batch_of(engine, views), cfg)
        torch.cuda.synchronize()
        one.append((o.xyz[:o.total_points()].cpu().numpy(), o.err[:o.total_points()].cpu().numpy()))
    ring = DensifyRing(dev, depth=3)
    outs = [ring.submit(batch_of(ring.engines[ring.slot()], views), cfg) for views in groups]
    ring.synchronize()
    for (xyz, err), o in zip(one, outs):
        n = o.total_points()
        assert n > 0 and np.array_equal(o.xyz[:n].cpu().numpy(), xyz) and np.array_equal(o.err[:n].cpu().numpy(), err)

    def match_source(rp):
        inp = inputs[rp]
        ri, nb = inp["ref_index"], inp["nbr_indices"]
        packed = P._PackedReferenceBatch(ref_id=cams[ri].uid, ref_path="", imA_np=inp["image"].numpy(), maskA_np=None,
                                         wA_cam=cams[ri].width, hA_cam=cams[ri].height, nn_ids=[cams[j].uid for j in nb],
                                         nn_masks=[None] * len(nb), nn_arrays=[None] * len(nb))
        return P._MatchedReference(packed=packed, warp_list_cpu=[inp["warp"][k] for k in range(len(nb))],
                                   cert_list_cpu=[inp["cert"][k] for k in range(len(nb))], pair_index_by_nbr={}, image_by_nbr={})
    refs = list(range(scene.n_refs))
    pc = DensePipelineConfig(output_path=str(tmp_path / "dense.ply"), matches_per_ref=4000, refs_per_launch=4)
    res = P.run_dense_pipeline(cams, refs, None, pc, match_source=match_source, w_match=scene.w_match, h_match=scene.h_match)
    assert res.pairs_processed == len(refs) and res.xyz.shape[0] > 1000
    # the lens reached the kernels: the same run with the coefficients stripped triangulates other points
    plain = P.run_dense_pipeline([_strip(c) for c in cams], refs, None, pc, match_source=match_source, w_match=scene.w_match,
                                 h_match=scene.h_match)
    assert res.xyz.shape != plain.xyz.shape or not np.array_equal(res.xyz, plain.xyz)
