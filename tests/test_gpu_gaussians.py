"""GPU: 3DGS initialisation (ldp_gaussian_init / output.init_gaussians) against the numpy oracle of tests/gaussian_oracle.py
(dist2, sh_dc and opacity bit for bit, scales within 1 f32 ulp, rotations taking e_z to the normal), and the 3DGS PLY records
against the host writer byte for byte."""
import ctypes as C

import numpy as np
import pytest
import torch

from lichtfeld_densification_plugin_b200 import _native as N
from lichtfeld_densification_plugin_b200 import build, output, synth
from lichtfeld_densification_plugin_b200.core import writers
from tests import gaussian_oracle as GO
from tests import outlier_oracle as OO
from tests.test_oracle_gaussians import _ulps, _unit

pytestmark = pytest.mark.gpu

KS = (1, 3, 8, 63)


@pytest.fixture(scope="module")
def lib():
    build.build()
    return N.load()


def _raw(lib, xyz: torch.Tensor, rgb: torch.Tensor, k: int, normals=None, opacity=0.1, flatten=1.0, stream=None):
    """The C entry point: dict of host arrays and the status."""
    dev, n = xyz.device, int(xyz.shape[0])
    need = C.c_size_t(0)
    N.check(lib.ldp_gaussian_workspace_bytes(n, k, C.byref(need)), "ldp_gaussian_workspace_bytes")
    ws = torch.empty((max(1, need.value),), dtype=torch.uint8, device=dev)
    out = {name: torch.full(shape, -7.0, dtype=torch.float32, device=dev)
           for name, shape in (("sh_dc", (n, 3)), ("opacity", (n,)), ("scales", (n, 3)), ("rotations", (n, 4)), ("dist2", (n,)))}
    status = torch.full((3,), -1, dtype=torch.int32, device=dev)
    st = stream if stream is not None else torch.cuda.current_stream(dev)
    ptr = lambda t: C.c_void_p(t.data_ptr() if t is not None else 0)          # noqa: E731
    with torch.cuda.stream(st):
        rc = lib.ldp_gaussian_init(ptr(xyz), ptr(rgb), ptr(normals), n, k, opacity, flatten, ptr(out["sh_dc"]), ptr(out["opacity"]),
                                   ptr(out["scales"]), ptr(out["rotations"]), ptr(out["dist2"]), ptr(status), ptr(ws),
                                   C.c_size_t(need.value), C.c_void_p(st.cuda_stream))
    N.check(rc, "ldp_gaussian_init")
    st.synchronize()
    got = {name: t.cpu().numpy() for name, t in out.items()}
    got["status"] = status.cpu().numpy()
    return got


def _judge(x, rgb, nrm, k, got, flatten=1.0, tag=""):
    ref = GO.init_gaussians(x, rgb, normals=nrm, k=k, flatten=flatten)
    assert got["status"][0] == 0, tag
    assert got["dist2"].tobytes() == ref["dist2"].tobytes(), (tag, int(np.sum(got["dist2"] != ref["dist2"])))
    assert got["sh_dc"].tobytes() == ref["sh_dc"].tobytes(), tag
    assert got["opacity"].tobytes() == ref["opacity"].tobytes(), tag
    assert _ulps(got["scales"], ref["scales"]).max(initial=0) <= 1, tag
    q = got["rotations"]
    assert np.all(np.abs(np.linalg.norm(q.astype(np.float64), axis=1) - 1) <= 1e-6), tag
    _, defined = GO.rotations(nrm, x.shape[0])
    assert int(got["status"][1]) == int((~defined).sum()) == ref["undefined"], tag
    assert np.all(q[~defined] == np.array([1, 0, 0, 0], np.float32)), tag
    if defined.any():
        ez = GO.build_rotation(q[defined])[:, :, 2]
        err = np.abs(ez - _unit(np.asarray(nrm, np.float64)[defined])).max()
        assert err <= 1e-6, (tag, err)
    return ref


def _cloud(kind: str, n: int, seed: int) -> np.ndarray:
    if kind == "dup_clusters":                 # clusters of 100 exact duplicates (more than k + 1 for every k) and a few strays
        rng = np.random.default_rng(seed)
        c = rng.uniform(-1, 1, size=(max(1, n // 100), 3))
        x = np.repeat(c, 100, axis=0)[:n]
        x[::37] += 0.01 * rng.normal(size=x[::37].shape)
        return x.astype(np.float32)
    return OO.make_cloud(kind, n, seed=seed)


@pytest.mark.parametrize("kind,n", [("sphere_floaters", 30_000), ("lattice", 8000), ("dup_clusters", 6000),
                                    ("sphere_floaters", 1), ("sphere_floaters", 2), ("lattice", 3), ("dup_clusters", 4)])
def test_kernel_vs_oracle(lib, kind, n):
    x = _cloud(kind, n, seed=n)
    rng = np.random.default_rng(n)
    rgb = rng.random((n, 3)).astype(np.float32)
    nrm = _unit(rng.normal(size=(n, 3))).astype(np.float32)
    nrm[::5] = 0.0                                          # undefined: zero normals
    if n >= 3:
        nrm[1] = (0, 0, -1)
        nrm[2] = (1e-7, 0, -1)
    xd, rd, nd = (torch.from_numpy(a).cuda() for a in (x, rgb, nrm))
    for k in KS:
        got = _raw(lib, xd, rd, k)
        _judge(x, rgb, None, k, got, tag=f"{kind} n={n} k={k}")
        got = _raw(lib, xd, rd, k, normals=nd, flatten=0.1)
        _judge(x, rgb, nrm, k, got, flatten=0.1, tag=f"{kind} n={n} k={k} normals")
        if n >= 1000:
            print(f"{kind} n={n} k={k}: left the finest grid {got['status'][2]}, at the floor {int(np.sum(got['dist2'] == GO.FLOOR))}")


@pytest.mark.parametrize("kind", ["sphere_floaters", "lattice", "dup_clusters"])
def test_shells_do_not_change_results(lib, kind):
    x = _cloud(kind, 20_000, seed=7)
    rgb = np.random.default_rng(7).random((20_000, 3)).astype(np.float32)
    xd, rd = torch.from_numpy(x).cuda(), torch.from_numpy(rgb).cuda()
    ref = GO.dist2(x, 8)
    try:
        for shells in (1, 2, 6):
            N.check(lib.ldp_debug_outlier_max_shells(shells), "max_shells")
            got = _raw(lib, xd, rd, 8)
            assert got["dist2"].tobytes() == ref.tobytes(), (kind, shells)
    finally:
        lib.ldp_debug_outlier_max_shells(0)


@pytest.mark.parametrize("d", [0, 1, 2, 3])
@pytest.mark.parametrize("with_normals", [False, True])
def test_records_match_host_writer(lib, tmp_path, d, with_normals):
    n = 1000
    rng = np.random.default_rng(d)
    x = rng.normal(size=(n, 3)).astype(np.float32)
    rgb = rng.random((n, 3)).astype(np.float32)
    xd, rd = torch.from_numpy(x).cuda(), torch.from_numpy(rgb).cuda()
    nd = output.estimate_normals(xd, nb_neighbors=8).normals if with_normals else None
    g = output.init_gaussians(xd, rd, normals=nd, flatten=0.5 if with_normals else 1.0)
    h = lambda t: None if t is None else t.cpu().numpy()          # noqa: E731
    output.write_gaussian_ply(str(tmp_path / "d.ply"), xd, g, normals=nd, sh_degree=d)
    writers.write_gaussian_ply(str(tmp_path / "h.ply"), x, h(g.sh_dc), h(g.opacity), h(g.scales), h(g.rotations),
                               normals=h(nd), sh_degree=d)
    assert (tmp_path / "d.ply").read_bytes() == (tmp_path / "h.ply").read_bytes()
    size = output.gaussian_record_bytes(d)
    host = writers.gaussian_ply_vertices(x, h(g.sh_dc), h(g.opacity), h(g.scales), h(g.rotations), h(nd), d)
    # n_dev truncation: only min(n, *n_dev) records are written, the rest of the buffer is untouched
    for m in (0, 1, 417, n, n + 5):
        n_dev = torch.tensor([m], dtype=torch.int64, device="cuda")
        rec = output.gaussian_ply_records(xd, g, nd, d, n_dev=n_dev)
        w = min(m, n)
        assert rec[:w * size].cpu().numpy().tobytes() == host[:w].astype("<f4").tobytes(), (d, m)


def test_rejections_and_non_finite(lib):
    x = OO.make_cloud("cube", 1000)
    xd = torch.from_numpy(x).cuda()
    rd = torch.rand((1000, 3), device="cuda")
    nd = torch.zeros((1000, 3), device="cuda")
    for kw in (dict(nb_neighbors=0), dict(nb_neighbors=64), dict(opacity=0.0), dict(opacity=1.0), dict(flatten=0.0),
               dict(flatten=1.5), dict(flatten=0.5)):
        with pytest.raises(ValueError):
            output.init_gaussians(xd, rd, **kw)
    need = C.c_size_t(0)
    for k in (0, 64):
        assert lib.ldp_gaussian_workspace_bytes(10, k, C.byref(need)) == -1
    ws = torch.empty((1 << 24,), dtype=torch.uint8, device="cuda")
    outs = [torch.empty((1000, 4), device="cuda") for _ in range(5)]
    status = torch.zeros((3,), dtype=torch.int32, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr() if t is not None else 0)          # noqa: E731

    def call(k=3, opacity=0.1, flatten=1.0, normals=None):
        return lib.ldp_gaussian_init(p(xd), p(rd), p(normals), 1000, k, opacity, flatten, *(p(t) for t in outs), p(status), p(ws),
                                     C.c_size_t(ws.numel()), C.c_void_p(0))
    for kw in (dict(k=0), dict(k=64), dict(opacity=0.0), dict(opacity=1.0), dict(opacity=float("nan")), dict(flatten=0.0),
               dict(flatten=1.01), dict(flatten=float("nan")), dict(flatten=0.5)):
        assert call(**kw) == -1, kw
    assert call(flatten=0.5, normals=nd) == 0
    torch.cuda.synchronize()
    assert lib.ldp_pack_gaussian_ply_records(p(xd), p(None), *(p(t) for t in outs[:4]), 1000, p(None), 4, p(ws), C.c_void_p(0)) == -1
    assert lib.ldp_pack_gaussian_ply_records(p(xd), p(None), *(p(t) for t in outs[:4]), 1000, p(None), 0, C.c_void_p(ws.data_ptr() + 2),
                                             C.c_void_p(0)) == -1
    for bad in (float("nan"), float("inf"), -float("inf")):
        xb = xd.clone()
        xb[17, 2] = bad
        with pytest.raises(ValueError):
            output.init_gaussians(xb, rd)
        assert _raw(lib, xb, rd, 3)["status"][0] == 1


def test_streams_inputs_and_empty(lib):
    x = OO.make_cloud("sphere_floaters", 100_000, seed=9)
    rgb = np.random.default_rng(9).random((100_000, 3)).astype(np.float32)
    xd, rd = torch.from_numpy(x).cuda(), torch.from_numpy(rgb).cuda()
    nd = output.estimate_normals(xd, nb_neighbors=20).normals
    a = _raw(lib, xd, rd, 3, normals=nd, flatten=0.2)
    b = _raw(lib, xd, rd, 3, normals=nd, flatten=0.2, stream=torch.cuda.Stream())
    assert all(a[key].tobytes() == b[key].tobytes() for key in a)
    g = output.init_gaussians(xd, rd, normals=nd, nb_neighbors=3, flatten=0.2)
    torch.cuda.synchronize()
    assert xd.cpu().numpy().tobytes() == x.tobytes()
    for key in ("sh_dc", "opacity", "scales", "rotations", "dist2"):
        assert getattr(g, key).cpu().numpy().tobytes() == a[key].tobytes(), key
    assert g.undefined == int(a["status"][1])
    e = output.init_gaussians(xd[:0], rd[:0])
    assert e.scales.shape == (0, 3) and e.rotations.shape == (0, 4) and e.undefined == 0


@pytest.mark.parametrize("outliers", [0, 20])
def test_run_dense_pipeline_gaussians(tmp_path, outliers):
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
    kw = dict(output_path=str(tmp_path / "dense.ply"), matches_per_ref=4000, refs_per_launch=4, multiview=True,
              outlier_neighbors=outliers, normal_neighbors=20)
    run = lambda cfg, cb=None: P.run_dense_pipeline(cams, list(range(scene.n_refs)), None, cfg, match_source=match_source,  # noqa: E731
                                                    w_match=scene.w_match, h_match=scene.h_match, progress_callback=cb)
    steps = []
    on = run(DensePipelineConfig(gaussian_neighbors=3, gaussian_flatten=0.1, **kw), cb=lambda p, s: steps.append(s))
    off = run(DensePipelineConfig(**kw))
    assert "Initialising Gaussians..." in steps and off.gaussians is None
    for key in ("xyz", "rgb", "err", "normals", "n_views"):
        assert getattr(on, key).tobytes() == getattr(off, key).tobytes(), key
    ref = output.init_gaussians(torch.from_numpy(on.xyz).cuda(), torch.from_numpy(on.rgb).cuda(),
                                normals=torch.from_numpy(on.normals).cuda(), nb_neighbors=3, flatten=0.1)
    assert sorted(on.gaussians) == ["opacity", "rotations", "scales", "sh_dc"]
    for key, v in on.gaussians.items():
        assert v.dtype == np.float32 and v.tobytes() == getattr(ref, key).cpu().numpy().tobytes(), key
    assert on.gaussians["scales"].shape == (on.xyz.shape[0], 3)
