"""GPU: oriented normals (ldp_estimate_normals / output.estimate_normals) against the numpy oracle of
tests/normals_oracle.py: neighbour lists bit for bit, normals within f32 rounding plus eigenvector conditioning."""
import ctypes as C

import numpy as np
import pytest
import torch

from lichtfeld_densification_plugin_b200 import _native as N
from lichtfeld_densification_plugin_b200 import build, output, synth
from lichtfeld_densification_plugin_b200.core import writers
from tests import normals_oracle as NO
from tests import outlier_oracle as OO
from tests.test_oracle_normals import SPHERE_BOUND_DEG, SPHERE_N, SPHERE_SEED

pytestmark = pytest.mark.gpu

KS = (3, 8, 20, 64)
# normal angle bound: f32 output rounding plus COND * lambda2 / (lambda1 - lambda0), the eigenvector's conditioning in f64.
# Calibration: the host restatement of the kernel's Jacobi solver differs from eigh by at most 6.2e-16 * lambda2 / gap on
# the clouds below, so 1e-13 leaves two orders of magnitude.  On the first B200 run every judged normal passed, and the
# largest angle * gap / lambda2 was 4.0e-8: the f32 rounding of well-conditioned normals, inside the 2e-7 term.
COND = 1e-13
GRAZING = 1e-6


@pytest.fixture(scope="module")
def lib():
    build.build()
    return N.load()


def _raw(lib, xyz: torch.Tensor, k: int, centers=None, center_idx=None, stream=None):
    """The C entry point: (normals, curvature, neighbours, status) on the host."""
    dev, n = xyz.device, int(xyz.shape[0])
    ke = min(k, n)
    need = C.c_size_t(0)
    N.check(lib.ldp_normals_workspace_bytes(n, k, C.byref(need)), "ldp_normals_workspace_bytes")
    ws = torch.empty((max(1, need.value),), dtype=torch.uint8, device=dev)
    nrm = torch.full((n, 3), -7.0, dtype=torch.float32, device=dev)
    curv = torch.full((n,), -7.0, dtype=torch.float32, device=dev)
    idx = torch.full((n, ke), -1, dtype=torch.int32, device=dev)
    status = torch.full((3,), -1, dtype=torch.int32, device=dev)
    st = stream if stream is not None else torch.cuda.current_stream(dev)
    ptr = lambda t: C.c_void_p(t.data_ptr() if t is not None else 0)          # noqa: E731
    with torch.cuda.stream(st):
        rc = lib.ldp_estimate_normals(ptr(xyz), n, k, ptr(centers), int(centers.shape[0]) if centers is not None else 0,
                                      ptr(center_idx), ptr(nrm), ptr(curv), ptr(idx), ptr(status), ptr(ws),
                                      C.c_size_t(need.value), C.c_void_p(st.cuda_stream))
    N.check(rc, "ldp_estimate_normals")
    st.synchronize()
    return nrm.cpu().numpy(), curv.cpu().numpy(), idx.cpu().numpy(), status.cpu().numpy()


def _judge(x, k, got, centers=None, center_idx=None, ref_idx=None, tag=""):
    """Neighbours bit-identical, undefined sets equal (ratios l1/l2 in [1e-13, 1e-11] listed, not judged), angles and
    curvature within the bounds of the module docstring.  Returns the largest angle / (lambda2 / gap)."""
    nrm, curv, idx, status = got
    if ref_idx is None:
        ref_idx = NO.knn_lex_exact(x, k)
    assert np.array_equal(idx, ref_idx), (tag, int(np.sum(np.any(idx != ref_idx, axis=1))))
    rn, rc, ru, lam = NO.normals_from_neighbors(x, ref_idx, centers, center_idx)
    gu = ~np.any(nrm != 0, axis=1)
    with np.errstate(invalid="ignore", divide="ignore"):
        ratio = lam[:, 1] / lam[:, 2]
    listed = (ratio >= 1e-13) & (ratio <= 1e-11)
    if listed.any():
        print(f"{tag}: {int(listed.sum())} points with l1/l2 in [1e-13, 1e-11] not judged: {np.nonzero(listed)[0][:20].tolist()}")
    assert np.array_equal(gu[~listed], ru[~listed]), (tag, int(np.sum(gu[~listed] != ru[~listed])))
    assert int(status[1]) == int(gu.sum()) and int(status[0]) == 0
    assert np.isnan(curv[gu]).all()
    d = ~gu & ~ru
    with np.errstate(divide="ignore"):
        tol = 2e-7 + COND * lam[d, 2] / (lam[d, 1] - lam[d, 0])
    ang = NO.angle(nrm[d], rn[d])
    # where the sign is a near tie the solvers may choose differently: the canonical sign when the two largest magnitudes
    # of the normal are within the angle bound, the orientation when the centre is within GRAZING of the tangent plane
    s = np.sort(np.abs(rn[d]), axis=1)
    amb = (s[:, 2] - s[:, 1]) <= 2 * tol
    if centers is not None:
        cen = np.asarray(centers, np.float64)[np.zeros(len(x), np.int64) if center_idx is None else np.asarray(center_idx)][d]
        dc = cen - x[d].astype(np.float64)
        dot = np.abs(np.sum(rn[d] * dc, axis=1)) / np.maximum(np.linalg.norm(dc, axis=1), 1e-300)
        amb = np.where(dot > np.maximum(GRAZING, 2 * tol), False, True)
    ang = np.where(amb, np.minimum(ang, np.pi - ang), ang)
    bad = ang > tol
    assert not bad.any(), (tag, int(bad.sum()), ang[bad][:5], tol[bad][:5])
    cerr = np.abs(curv[d].astype(np.float64) - rc[d])
    assert np.all(cerr <= np.maximum(1e-6 * np.abs(rc[d]), 1e-12)), (tag, cerr.max())
    gap = lam[d, 1] - lam[d, 0]
    return float(np.max(ang * gap / lam[d, 2])) if d.any() else 0.0


@pytest.mark.parametrize("kind", OO.CLOUDS)
@pytest.mark.parametrize("n", [1, 2, 3, 17, 1000, 50_000])
def test_kernel_vs_oracle(lib, kind, n):
    x = OO.make_cloud(kind, n, seed=n)
    dev = torch.from_numpy(x).cuda()
    ref64 = NO.knn_lex_exact(x, max(KS))            # the (d^2, index) list for k is the first k_eff entries of this one
    worst = 0.0
    for k in KS:
        got = _raw(lib, dev, k)
        worst = max(worst, _judge(x, k, got, ref_idx=ref64[:, :min(k, n)], tag=f"{kind} n={n} k={k}"))
        if n == 50_000:
            print(f"{kind} n={n} k={k}: undefined {got[3][1]}, left the finest grid {got[3][2]}")
    print(f"{kind} n={n}: largest angle * gap / lambda2 = {worst:.2e}")


def test_orientation(lib):
    x = NO.noisy_sphere(50_000, seed=5)
    dev = torch.from_numpy(x).cuda()
    cen = torch.from_numpy(3 * x).cuda()
    ci = torch.arange(x.shape[0], dtype=torch.int32, device="cuda")
    for k in (8, 20):
        nrm, _, idx, status = _raw(lib, dev, k, cen, ci)
        _judge(x, k, (nrm, _, idx, status), centers=3 * x, center_idx=np.arange(x.shape[0]), tag=f"sphere k={k}")
        dc = 2.0 * x.astype(np.float64)
        dot = np.sum(nrm * dc, axis=1) / np.linalg.norm(dc, axis=1)
        assert np.all((dot >= 0) | (np.abs(dot) < GRAZING))
        one = np.array([[0.3, -0.2, 4.0]], np.float32)
        nrm1, _, _, status1 = _raw(lib, dev, k, torch.from_numpy(one).cuda())
        assert status1[0] == 0
        dc1 = one.astype(np.float64) - x
        dot1 = np.sum(nrm1 * dc1, axis=1) / np.linalg.norm(dc1, axis=1)
        assert np.all((dot1 >= 0) | (np.abs(dot1) < GRAZING))


@pytest.mark.parametrize("k", [8, 20])
def test_sphere_bound_on_the_device(k):
    """The oracle's measured angle bound (tests/test_oracle_normals.py) holds for the kernel's normals."""
    x = NO.noisy_sphere(SPHERE_N, seed=SPHERE_SEED)
    r = output.estimate_normals(torch.from_numpy(x).cuda(), nb_neighbors=k, centers=torch.from_numpy(3 * x).cuda(),
                                center_idx=torch.arange(SPHERE_N, device="cuda"))
    assert r.undefined == 0
    radial = x / np.linalg.norm(x, axis=1, keepdims=True)
    ang = np.degrees(NO.angle(r.normals.cpu().numpy(), radial))
    print(f"device sphere k={k}: median {np.median(ang):.3f} deg, p99 {np.percentile(ang, 99):.3f} deg")
    assert np.median(ang) <= SPHERE_BOUND_DEG[k][0] and np.percentile(ang, 99) <= SPHERE_BOUND_DEG[k][1]


@pytest.mark.parametrize("kind", ["sphere_floaters", "duplicates", "two_clusters", "lattice"])
def test_shells_do_not_change_results(lib, kind):
    xyz = torch.from_numpy(OO.make_cloud(kind, 20_000, seed=7)).cuda()
    try:
        N.check(lib.ldp_debug_outlier_max_shells(1), "max_shells")
        a = _raw(lib, xyz, 20)
        N.check(lib.ldp_debug_outlier_max_shells(0), "max_shells")
        b = _raw(lib, xyz, 20)
    finally:
        lib.ldp_debug_outlier_max_shells(0)
    assert a[3][2] >= b[3][2]
    for u, v in zip(a, b):
        if u.dtype == np.int32 and u.ndim == 1:
            continue                                   # status: the escalation count depends on the shells
        assert u.tobytes() == v.tobytes()
    assert a[3][:2].tolist() == b[3][:2].tolist()


def test_large_sphere_vs_kdtree(lib):
    """2.3 M points, sphere + 1 % floaters: neighbours from cKDTree candidates, normals from eigh."""
    xyz, _ = OO.sphere_with_floaters(2_300_000, seed=1)
    got = _raw(lib, torch.from_numpy(xyz).cuda(), 20)
    worst = _judge(xyz, 20, got, tag="2.3M k=20")
    print(f"2.3M: undefined {got[3][1]}, left the finest grid {got[3][2]} ({got[3][2] / xyz.shape[0]:.2%}), "
          f"largest angle * gap / lambda2 = {worst:.2e}")


def test_rejections(lib):
    xyz = torch.from_numpy(OO.make_cloud("cube", 1000)).cuda()
    for k in (0, 2, 65):
        with pytest.raises(ValueError):
            output.estimate_normals(xyz, nb_neighbors=k)
        need = C.c_size_t(0)
        assert lib.ldp_normals_workspace_bytes(10, k, C.byref(need)) == -1
    for bad in (float("nan"), float("inf"), -float("inf")):
        x = xyz.clone()
        x[17, 2] = bad
        with pytest.raises(ValueError):
            output.estimate_normals(x, nb_neighbors=8)
        assert _raw(lib, x, 8)[3][0] == 1
    cen = torch.zeros((2, 3), device="cuda")
    ci = torch.zeros((1000,), dtype=torch.int32, device="cuda")
    ci[5] = 2
    with pytest.raises(ValueError):
        output.estimate_normals(xyz, nb_neighbors=8, centers=cen, center_idx=ci)
    assert _raw(lib, xyz, 8, cen, ci)[3][0] == 2
    ci[5] = -1
    assert _raw(lib, xyz, 8, cen, ci)[3][0] == 2
    with pytest.raises(ValueError):
        output.estimate_normals(xyz, nb_neighbors=8, center_idx=ci)
    ws = torch.empty((1 << 20,), dtype=torch.uint8, device="cuda")
    out = torch.empty((1000, 3), device="cuda")
    status = torch.zeros((3,), dtype=torch.int32, device="cuda")
    rc = lib.ldp_estimate_normals(C.c_void_p(xyz.data_ptr()), 1000, 8, C.c_void_p(0), 0, C.c_void_p(ci.data_ptr()),
                                  C.c_void_p(out.data_ptr()), C.c_void_p(0), C.c_void_p(0), C.c_void_p(status.data_ptr()),
                                  C.c_void_p(ws.data_ptr()), C.c_size_t(ws.numel()), C.c_void_p(0))
    assert rc == -1


def test_streams_inputs_and_empty(lib):
    x = OO.make_cloud("sphere_floaters", 100_000, seed=9)
    xyz = torch.from_numpy(x).cuda()
    a = _raw(lib, xyz, 20)
    b = _raw(lib, xyz, 20, stream=torch.cuda.Stream())
    assert all(u.tobytes() == v.tobytes() for u, v in zip(a, b))
    r = output.estimate_normals(xyz, nb_neighbors=20, return_neighbors=True)
    torch.cuda.synchronize()
    assert xyz.cpu().numpy().tobytes() == x.tobytes()
    assert r.normals.cpu().numpy().tobytes() == a[0].tobytes() and r.curvature.cpu().numpy().tobytes() == a[1].tobytes()
    assert np.array_equal(r.neighbors.cpu().numpy(), a[2]) and r.undefined == int(a[3][1])
    assert output.estimate_normals(xyz, nb_neighbors=20).neighbors is None
    e = output.estimate_normals(xyz[:0], nb_neighbors=20)
    assert e.normals.shape == (0, 3) and e.undefined == 0


@pytest.mark.parametrize("n", [1, 255, 1000])
def test_write_ply_with_normals_matches_host_writer(tmp_path, n):
    rng = np.random.default_rng(n)
    xyz = rng.normal(size=(n, 3)).astype(np.float32)
    rgb = rng.random(size=(n, 3)).astype(np.float32)
    nrm = output.estimate_normals(torch.from_numpy(xyz).cuda(), nb_neighbors=8).normals
    output.write_ply(str(tmp_path / "d.ply"), torch.from_numpy(xyz).cuda(), torch.from_numpy(rgb).cuda(), normals=nrm)
    writers.write_ply(str(tmp_path / "h.ply"), xyz, writers.to_uint8_rgb(rgb), normals=nrm.cpu().numpy())
    assert (tmp_path / "d.ply").read_bytes() == (tmp_path / "h.ply").read_bytes()
    output.write_ply(str(tmp_path / "d0.ply"), torch.from_numpy(xyz).cuda(), torch.from_numpy(rgb).cuda())
    writers.write_ply(str(tmp_path / "h0.ply"), xyz, writers.to_uint8_rgb(rgb))
    assert (tmp_path / "d0.ply").read_bytes() == (tmp_path / "h0.ply").read_bytes()


@pytest.mark.parametrize("outliers", [0, 20])
def test_run_dense_pipeline_normals(tmp_path, outliers):
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
    kw = dict(output_path=str(tmp_path / "dense.ply"), matches_per_ref=4000, refs_per_launch=4, multiview=True,
              outlier_neighbors=outliers)
    run = lambda cfg, refs_=refs, cb=None: P.run_dense_pipeline(cams, refs_, None, cfg, match_source=match_source,   # noqa: E731
                                                                w_match=scene.w_match, h_match=scene.h_match, progress_callback=cb)
    steps = []
    on = run(DensePipelineConfig(normal_neighbors=20, **kw), cb=lambda p, s: steps.append(s))
    off = run(DensePipelineConfig(**kw))
    assert "Estimating normals..." in steps and off.normals is None
    assert on.xyz.tobytes() == off.xyz.tobytes() and on.rgb.tobytes() == off.rgb.tobytes()
    assert on.err.tobytes() == off.err.tobytes() and on.n_views.tobytes() == off.n_views.tobytes()
    # each point's reference view: views triangulate independently (Philox keyed by view), so the unfiltered cloud is the
    # concatenation of one-view runs
    kw1 = dict(kw, outlier_neighbors=0)
    parts = [run(DensePipelineConfig(**kw1), refs_=[r]) for r in refs]
    full = run(DensePipelineConfig(**kw1))
    assert np.concatenate([p.xyz for p in parts]).tobytes() == full.xyz.tobytes()
    uid = np.concatenate([np.full(p.xyz.shape[0], cams[inputs[r]["ref_index"]].uid) for r, p in zip(refs, parts)])
    if outliers:
        keep = output.remove_statistical_outliers(torch.from_numpy(full.xyz).cuda(), torch.from_numpy(full.xyz).cuda(),
                                                  nb_neighbors=outliers, std_ratio=2.0).kept_idx.cpu().numpy()
        assert 0 < keep.size < full.xyz.shape[0]
        uid = uid[keep]
    assert uid.shape[0] == on.xyz.shape[0]
    by_uid = {c.uid: c for c in cams}
    uids, ci = np.unique(uid, return_inverse=True)
    centers = np.stack([np.asarray(by_uid[int(u)].C, np.float64).reshape(3) for u in uids]).astype(np.float32)
    ref = output.estimate_normals(torch.from_numpy(on.xyz).cuda(), nb_neighbors=20, centers=torch.from_numpy(centers).cuda(),
                                  center_idx=torch.from_numpy(ci.astype(np.int32)).cuda())
    assert on.normals.dtype == np.float32 and on.normals.tobytes() == ref.normals.cpu().numpy().tobytes()
    defined = np.any(on.normals != 0, axis=1)
    dc = centers[ci].astype(np.float64) - on.xyz
    dot = np.sum(on.normals * dc, axis=1) / np.linalg.norm(dc, axis=1)
    assert defined.mean() > 0.99
    assert np.all((dot[defined] >= 0) | (np.abs(dot[defined]) < GRAZING))
