"""CPU: the lens oracle (tests/lens_oracle.py) against OpenCV, and the lens fields of the camera records.

OpenCV is compared live where cv2 is installed, and through tests/golden/lens/cv2_lens.npz (written by
tests/golden/make_lens_golden.py from cv2) everywhere.
"""
import os
import re

import numpy as np
import pytest
import torch

from lichtfeld_densification_plugin_b200.core.camera_models import COLMAP_MODELS, CameraRecord
from lichtfeld_densification_plugin_b200.core.pipeline import _build_camera_lookup, _record_for
from lichtfeld_densification_plugin_b200.engine import RefBatch
from tests import lens_oracle as LO
from tests.golden import make_lens_golden as G

try:
    import cv2
except ImportError:          # the stored vectors still run
    cv2 = None

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LENS_CASES = list(G.CASES)


def _golden():
    return np.load(G.GOLDEN)


def _cv2_sources():
    z = _golden()
    yield "golden", z["ideal"], z["obs"], {n: (z[f"fwd_{n}"], z[f"und_{n}"]) for n in LENS_CASES}
    if cv2 is not None:
        live = {n: G.cv2_results(cv2, G.record(n))[2:] for n in LENS_CASES}
        yield "live", G.pixel_grid(), G.pixel_grid().astype(np.float32).astype(np.float64), live


def test_constants_shared_with_the_kernel():
    src = open(os.path.join(ROOT, "lichtfeld_densification_plugin_b200", "csrc", "ldp_geometry.cu")).read()
    assert int(re.search(r"constexpr int LENS_MAX_ITERS = (\d+);", src).group(1)) == LO.LENS_MAX_ITERS
    assert float(re.search(r"constexpr double LENS_STEP_TOL = ([0-9.e+-]+);", src).group(1)) == LO.LENS_STEP_TOL
    assert "constexpr double LENS_FISHEYE_THETA0_MAX = 1.5707963267948966 - 1e-6;" in src
    assert LO.FISHEYE_THETA0_MAX == 1.5707963267948966 - 1e-6


@pytest.mark.parametrize("name", LENS_CASES)
def test_forward_model_matches_opencv(name):
    L = LO.lens_of(G.record(name))
    for src, ideal, _, res in _cv2_sources():
        d = np.abs(LO.distort_px(L, ideal) - res[name][0]).max()
        assert d <= 1e-9, (src, name, d)


@pytest.mark.parametrize("name", LENS_CASES)
def test_undistortion_matches_opencv(name):
    L = LO.lens_of(G.record(name))
    for src, _, obs, res in _cv2_sources():
        x, y = LO.undistort(L, (obs[:, 0] - L.cx) / L.fx, (obs[:, 1] - L.cy) / L.fy)
        ours = np.stack([L.fx * x + L.cx, L.fy * y + L.cy], axis=1)
        theirs = res[name][1]
        # where both converge: ours is finite, cv2's result distorts back onto the observation
        both = np.isfinite(ours).all(axis=1) & (np.abs(LO.distort_px(L, theirs) - obs).max(axis=1) < 1e-6)
        assert both.mean() > 0.99, (src, name, both.mean())
        d = np.abs(ours[both] - theirs[both]).max()
        assert d <= 1e-6, (src, name, d)


@pytest.mark.parametrize("name", LENS_CASES)
def test_round_trip(name):
    L = LO.lens_of(G.record(name))
    rng = np.random.default_rng(7)
    obs = rng.uniform([0.0, 0.0], [G.WIDTH, G.HEIGHT], size=(20000, 2))
    x, y = LO.undistort(L, (obs[:, 0] - L.cx) / L.fx, (obs[:, 1] - L.cy) / L.fy)
    assert np.isfinite(x).all() and np.isfinite(y).all()
    back = LO.distort_px(L, np.stack([L.fx * x + L.cx, L.fy * y + L.cy], axis=1))
    assert np.abs(back - obs).max() <= 1e-9


def test_invalid_regions_are_nan():
    fish = LO.Lens("fisheye", np.array([0.02, 0.0, 0.0, 0.0, 0, 0, 0, 0], dtype=np.float64), 500.0, 500.0, 0.0, 0.0)
    # theta_d(pi/2) = 1.62: a distorted radius beyond it has no ray in front of the camera
    x, y = LO.undistort(fish, np.array([0.5, 1.7, 3.0]), np.array([0.0, 0.0, 0.0]))
    assert np.isfinite(x[0]) and np.isnan(x[1:]).all() and np.isnan(y[1:]).all()
    # a strong positive k1 puts theta_d(pi/2) above pi/2: distorted radii in [pi/2, theta_d(pi/2)) still have a ray in front
    # of the camera (the iteration starts inside [0, pi/2), like cv2.fisheye)
    wide = LO.lens_of(G.record("OPENCV_FISHEYE"))
    t = LO.HALF_PI
    top = t * (1 + wide.k[0] * t ** 2 + wide.k[1] * t ** 4 + wide.k[2] * t ** 6 + wide.k[3] * t ** 8)
    assert top > 1.7
    rd = np.array([1.58, 1.6, 1.65, 0.999 * top, 1.001 * top])
    x, y = LO.undistort(wide, rd, np.zeros(5))
    assert np.isfinite(x[:4]).all() and np.isnan(x[4])
    xd, _ = LO.distort(wide, x[:4], np.zeros(4))
    assert np.abs(xd - rd[:4]).max() < 1e-12
    # OpenCV k1 = -0.5: r (1 - 0.5 r^2) folds at r^2 = 2/3 (distorted radius 0.544); beyond it there is no valid inverse
    barrel = LO.Lens("opencv", np.array([-0.5, 0, 0, 0, 0, 0, 0, 0], dtype=np.float64), 500.0, 500.0, 0.0, 0.0)
    x, y = LO.undistort(barrel, np.array([0.3, 0.54, 0.6, 0.9]), np.zeros(4))
    assert np.isfinite(x[:2]).all() and np.isnan(x[2:]).all()
    xd, _ = LO.distort(barrel, x[:2], np.zeros(2))
    assert np.abs(xd - [0.3, 0.54]).max() < 1e-12


# ---- records -------------------------------------------------------------------------------------------------------------
R0 = np.array([[0.0, 0.0, 1.0], [0.0, 1.0, 0.0], [-1.0, 0.0, 0.0]])
T0 = np.array([0.1, -0.2, 3.0])


@pytest.mark.parametrize("name", list(COLMAP_MODELS))
def test_from_colmap(name):
    family, n_focal, slots = COLMAP_MODELS[name]
    dist = [0.01 * (i + 1) * (-1) ** i for i in range(len(slots))]
    focal = [800.5, 810.25][:n_focal]
    rec = CameraRecord.from_colmap(3, name, focal + [640.5, 400.25] + dist, 1297, 840, R0, T0, image_path="a.png")
    ref = CameraRecord.from_KRt(3, 1297, 840, [[800.5, 0, 640.5], [0, focal[-1], 400.25], [0, 0, 1]], R0, T0, image_path="a.png")
    for f in ("K", "R", "t", "P", "C"):
        assert np.array_equal(getattr(rec, f), getattr(ref, f)) and getattr(rec, f).dtype == np.float32, f
    if family is None:
        assert rec.lens_model is None and rec.lens_coeffs is None
    else:
        assert rec.lens_model == family
        expect = np.zeros(8)
        expect[list(slots)] = dist
        assert rec.lens_coeffs.dtype == np.float64 and np.array_equal(rec.lens_coeffs, expect)
    # all-zero coefficients: no lens
    zero = CameraRecord.from_colmap(3, name, focal + [640.5, 400.25] + [0.0] * len(slots), 1297, 840, R0, T0)
    assert zero.lens_model is None


def test_from_colmap_refuses():
    with pytest.raises(ValueError):
        CameraRecord.from_colmap(0, "THIN_PRISM_FISHEYE", [1.0] * 16, 10, 10, R0, T0)
    with pytest.raises(ValueError):
        CameraRecord.from_colmap(0, "FOV", [1.0] * 5, 10, 10, R0, T0)
    with pytest.raises(ValueError):
        CameraRecord.from_colmap(0, "OPENCV", [1.0] * 5, 10, 10, R0, T0)         # wrong parameter count
    rec = CameraRecord.from_colmap(0, "OPENCV", [800.0, 800.0, 5.0, 5.0, -0.1, 0, 0, 0], 10, 10, R0, T0)
    K = rec.K.copy()
    K[0, 1] = 0.5
    with pytest.raises(ValueError):
        CameraRecord(0, "", 10, 10, K, rec.R, rec.t, rec.P, rec.C, None, rec.lens_model, rec.lens_coeffs)
    # positional construction with the reference's fields still works
    CameraRecord(0, "", 10, 10, K, rec.R, rec.t, rec.P, rec.C)


def _template_bytes(ref, nbrs):
    b = RefBatch(8, 8, 8, 8, torch.device("cpu"))
    cert = torch.zeros((8, 8), dtype=torch.float32)
    warp = torch.zeros((8, 8, 4), dtype=torch.float32)
    b.add([cert] * len(nbrs), [warp] * len(nbrs), torch.zeros((8, 8, 3), dtype=torch.uint8), ref, nbrs)
    desc = b.desc_array().copy()
    for f in ("cert", "warp", "image", "mask_a", "mask_b"):     # tensor addresses: not part of the camera template
        desc[f] = 0
    return desc.tobytes(), b.has_lens


@pytest.mark.parametrize("name", ["PINHOLE", "SIMPLE_PINHOLE"])
def test_pinhole_records_carry_no_lens(name):
    focal = [800.0, 800.0][:COLMAP_MODELS[name][1]]
    recs = [CameraRecord.from_colmap(i, name, focal + [640.0, 400.0], 1280, 800, R0, T0 + i) for i in range(3)]
    krt = [CameraRecord.from_KRt(i, 1280, 800, [[800.0, 0, 640.0], [0, 800.0, 400.0], [0, 0, 1]], R0, T0 + i) for i in range(3)]
    a, lens_a = _template_bytes(recs[0], recs[1:])
    b, lens_b = _template_bytes(krt[0], krt[1:])
    assert a == b and not lens_a and not lens_b


def test_lens_descriptor_fields():
    cams = [G.record("OPENCV"), G.record("OPENCV_FISHEYE"), CameraRecord.from_KRt(2, 1297, 840, np.eye(3), R0, T0)]
    desc, has_lens = _template_bytes(cams[0], cams[1:])
    assert has_lens
    from lichtfeld_densification_plugin_b200 import _native as N
    row = np.frombuffer(desc, dtype=N.REF_DESC_DTYPE)[0]
    assert row["lens_a"]["model"] == N.LDP_LENS_OPENCV and row["lens_b"][0]["model"] == N.LDP_LENS_FISHEYE
    assert row["lens_b"][1]["model"] == N.LDP_LENS_PINHOLE
    assert np.array_equal(row["lens_a"]["k"], cams[0].lens_coeffs)
    assert row["lens_a"]["fx"] == cams[0].K[0, 0] and row["lens_a"]["cy"] == cams[0].K[1, 2]


def test_record_for_resized_copy_keeps_the_lens():
    rec = G.record("FULL_OPENCV")
    lookup = _build_camera_lookup([rec])
    sized = _record_for(lookup, rec.uid, size=(640, 415))
    assert (sized.width, sized.height) == (640, 415)
    assert sized.lens_model == rec.lens_model and np.array_equal(sized.lens_coeffs, rec.lens_coeffs)
    assert _record_for(lookup, rec.uid, size=(640, 415)) is sized
