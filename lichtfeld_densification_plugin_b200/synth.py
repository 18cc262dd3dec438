"""Synthetic scenes shaped like the matcher's outputs (SURVEY.md section 8d).

The RoMa network is out of scope, so its outputs are synthesised: pinhole cameras on orbit rings
looking at the origin, an analytic depth field per reference view back-projected and re-projected
into each neighbour to give the ``warp_AB`` channels in RoMa's normalised coordinates, plus noise
and gross outliers so every filter rejects a realistic fraction; certainty maps in two families:

* ``"T"`` tie-free: all values distinct f32 in [0.2, 0.9) -- bit-exact sampler parity is
  well-defined on these (SURVEY F5);
* ``"R"`` realistic: ``sigmoid`` of a smooth field + noise, floor-clamped at ``certainty_thresh``
  like reference core/pipeline.py:407, with a large saturated area above the 0.9 cap (ties).

Cameras may carry a COLMAP lens model (``lens=``): the warp then maps each matcher pixel of the reference view, an
observed (distorted) pixel, through the inverse lens to its ray, through the depth field to a world point, into the
neighbour's pinhole projection and through the neighbour's forward lens.  The lens arithmetic here is a torch f64
statement of its own (fixed-point inversion for OpenCV, Newton on theta for the fisheye); without a lens nothing of it runs.

Everything is generated with torch on the requested device (CPU for tests, GPU for the bench).
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from .core.camera_models import COLMAP_MODELS, CameraRecord
from .core.config import ROMA_PRESETS


@dataclass
class SynthScene:
    cameras: List[CameraRecord]
    refs_local: List[int]          # indices into ``cameras``
    nn_table: np.ndarray           # [V, nn] int64 neighbour indices (self excluded)
    H: int                         # map resolution
    W: int
    h_match: int                   # match resolution (H_lr, W_lr)
    w_match: int
    nn: int

    @property
    def n_refs(self) -> int:
        return len(self.refs_local)

    @property
    def n_pairs(self) -> int:
        return self.n_refs * self.nn


LensSpec = Optional[Tuple[str, Sequence[float]]]        # (COLMAP model name, its distortion parameters)


def make_orbit_cameras(n_views: int, width: int = 1297, height: int = 840, radius: float = 4.0,
                       focal_frac: float = 0.74, lens: Union[LensSpec, Sequence[LensSpec]] = None) -> List[CameraRecord]:
    """Pinhole cameras on stacked orbit rings, all looking at the origin.  Rings hold at most 200
    views so that nearest neighbours keep a ~2 degree baseline at any ``n_views``.

    ``lens``: one ``(model_name, distortion params)`` for every view, or a list of one per view (None = pinhole); the
    records are built by ``CameraRecord.from_colmap`` with the same K."""
    if lens is None or isinstance(lens[0], str):
        lens = [lens] * n_views
    if len(lens) != n_views:
        raise ValueError("lens: one spec, or one per view")
    n_rings = max(1, math.ceil(n_views / 200))
    per_ring = math.ceil(n_views / n_rings)
    fx = focal_frac * width
    K = np.array([[fx, 0.0, width / 2.0], [0.0, fx, height / 2.0], [0.0, 0.0, 1.0]], dtype=np.float32)
    cams: List[CameraRecord] = []
    for v in range(n_views):
        ring, slot = divmod(v, per_ring)
        theta = 2.0 * math.pi * (slot + 0.37 * ring) / per_ring
        elev = 0.35 * (ring - 0.5 * (n_rings - 1)) + 0.08 * math.sin(3.0 * theta)
        centre = np.array([radius * math.cos(theta), elev, radius * math.sin(theta)], dtype=np.float64)
        fwd = -centre / np.linalg.norm(centre)
        right = np.cross(np.array([0.0, 1.0, 0.0]), fwd)
        right /= np.linalg.norm(right)
        down = np.cross(fwd, right)
        R = np.stack([right, down, fwd], axis=0)                 # world -> camera
        t = -R @ centre
        if lens[v] is None:
            cams.append(CameraRecord.from_KRt(v, width, height, K, R, t, image_path=f"synthetic/{v:05d}.png"))
        else:
            name, dist = lens[v]
            focal = [fx] * COLMAP_MODELS[name.upper()][1]
            cams.append(CameraRecord.from_colmap(v, name, focal + [width / 2.0, height / 2.0] + list(dist), width, height, R, t,
                                                 image_path=f"synthetic/{v:05d}.png"))
    return cams


def make_scene(n_views: int, setting: str = "fast", ref_fraction: float = 0.25, nn: int = 4,
               width: int = 1297, height: int = 840, lens: Union[LensSpec, Sequence[LensSpec]] = None) -> SynthScene:
    h_lr, h_map = ROMA_PRESETS[setting]
    cams = make_orbit_cameras(n_views, width, height, lens=lens)
    centres = torch.from_numpy(np.stack([c.C for c in cams]).astype(np.float32))
    if n_views > 1:
        dist = torch.cdist(centres, centres)
        dist.fill_diagonal_(float("inf"))
        k = max(1, min(nn, n_views - 1))
        nn_table = torch.topk(dist, k, largest=False, dim=1).indices.numpy()
    else:
        nn_table = np.zeros((n_views, 0), dtype=np.int64)
    n_refs = max(1, min(n_views, int(round(n_views * ref_fraction))))
    refs = sorted(set(int(round(x)) for x in np.linspace(0, n_views - 1, n_refs)))
    return SynthScene(cameras=cams, refs_local=refs, nn_table=nn_table, H=h_map, W=h_map,
                      h_match=h_lr, w_match=h_lr, nn=nn_table.shape[1])


def _gen(device, seed: int) -> torch.Generator:
    g = torch.Generator(device=device)
    g.manual_seed(int(seed))
    return g


def _lens_t(cam: CameraRecord):
    if cam.lens_model is None:
        return None
    K = cam.K.astype(np.float64)
    return (cam.lens_model, [float(c) for c in cam.lens_coeffs], K[0, 0], K[1, 1], K[0, 2], K[1, 2])


def _distort_t(lens, x: torch.Tensor, y: torch.Tensor):
    model, k = lens[0], lens[1]
    r2 = x * x + y * y
    if model == "fisheye":
        r = torch.sqrt(r2)
        th = torch.atan(r)
        thd = th * (1 + k[0] * th ** 2 + k[1] * th ** 4 + k[2] * th ** 6 + k[3] * th ** 8)
        s = torch.where(r > 0, thd / torch.where(r > 0, r, torch.ones_like(r)), torch.ones_like(r))
        return x * s, y * s
    radial = (1 + k[0] * r2 + k[1] * r2 ** 2 + k[4] * r2 ** 3) / (1 + k[5] * r2 + k[6] * r2 ** 2 + k[7] * r2 ** 3)
    return (x * radial + 2 * k[2] * x * y + k[3] * (r2 + 2 * x * x),
            y * radial + k[2] * (r2 + 2 * y * y) + 2 * k[3] * x * y)


def _undistort_t(lens, xd: torch.Tensor, yd: torch.Tensor):
    """Inverse lens: fixed-point iteration (OpenCV) / Newton on theta (fisheye), run to convergence; NaN where the
    result does not reproduce the distorted point."""
    model, k = lens[0], lens[1]
    if model == "fisheye":
        rd = torch.sqrt(xd * xd + yd * yd)
        th = rd.clone()
        for _ in range(50):
            f = th * (1 + k[0] * th ** 2 + k[1] * th ** 4 + k[2] * th ** 6 + k[3] * th ** 8) - rd
            d = 1 + 3 * k[0] * th ** 2 + 5 * k[1] * th ** 4 + 7 * k[2] * th ** 6 + 9 * k[3] * th ** 8
            th = th - f / d
        s = torch.where(rd > 0, torch.tan(th) / torch.where(rd > 0, rd, torch.ones_like(rd)), torch.ones_like(rd))
        x, y = xd * s, yd * s
        x = torch.where((th >= 0) & (th < math.pi / 2), x, torch.full_like(x, float("nan")))
    else:
        x, y = xd.clone(), yd.clone()
        for _ in range(200):
            r2 = x * x + y * y
            radial = (1 + k[0] * r2 + k[1] * r2 ** 2 + k[4] * r2 ** 3) / (1 + k[5] * r2 + k[6] * r2 ** 2 + k[7] * r2 ** 3)
            dx = 2 * k[2] * x * y + k[3] * (r2 + 2 * x * x)
            dy = k[2] * (r2 + 2 * y * y) + 2 * k[3] * x * y
            x, y = (xd - dx) / radial, (yd - dy) / radial
    bx, by = _distort_t(lens, x, y)
    bad = ~((bx - xd).abs() < 1e-10) | ~((by - yd).abs() < 1e-10)
    nan = torch.full_like(x, float("nan"))
    return torch.where(bad, nan, x), torch.where(bad, nan, y)


def synth_ref_inputs(scene: SynthScene, ref_pos: int, device="cpu", cert_family: str = "R",
                     seed: int = 0, noise_sigma: float = 1e-3, outlier_frac: float = 0.10,
                     certainty_thresh: float = 0.20, return_points: bool = False) -> Dict[str, object]:
    """Matcher-shaped inputs for the ``ref_pos``-th reference view of ``scene``.

    Returns dict(cert f32 [nn,H,W], warp f32 [nn,H,W,4], image u8 [h_match,w_match,3],
    ref_index, nbr_indices); with ``return_points`` also ``points`` f64 [H,W,3], the world point of every map pixel.
    """
    dev = torch.device(device)
    H, W, hm, wm = scene.H, scene.W, scene.h_match, scene.w_match
    ref_i = scene.refs_local[ref_pos]
    nbrs = [int(j) for j in scene.nn_table[ref_i][: scene.nn]]
    camA = scene.cameras[ref_i]
    g = _gen(dev, seed * 1000003 + ref_i)

    # the matcher's reference grid (reference core/matcher.py:131-135)
    ys = torch.linspace(-1 + 1 / H, 1 - 1 / H, H, device=dev)
    xs = torch.linspace(-1 + 1 / W, 1 - 1 / W, W, device=dev)
    gy, gx = torch.meshgrid(ys, xs, indexing="ij")

    # pixel coords the path will decode (reference core/pipeline.py:655-656,681-683), in f64
    xA = (gx.double() + 1.0) * 0.5 * (wm - 1) * (camA.width / float(wm))
    yA = (gy.double() + 1.0) * 0.5 * (hm - 1) * (camA.height / float(hm))
    depth = 3.6 + 0.5 * torch.sin(2.1 * gx.double() + 0.3 * ref_i) * torch.cos(1.7 * gy.double())
    Kinv = torch.from_numpy(np.linalg.inv(camA.K.astype(np.float64))).to(dev)
    RA = torch.from_numpy(camA.R.astype(np.float64)).to(dev)
    tA = torch.from_numpy(camA.t.astype(np.float64)).to(dev).reshape(3)
    lensA = _lens_t(camA)
    if lensA is None:
        pix = torch.stack([xA, yA, torch.ones_like(xA)], dim=-1)                # [H,W,3]
        Xc = (pix @ Kinv.T) * depth.unsqueeze(-1)
    else:                  # the matcher pixel is an observed (distorted) pixel: its ray is that of the undistorted one
        K64 = camA.K.astype(np.float64)
        xu, yu = _undistort_t(lensA, (xA - K64[0, 2]) / K64[0, 0], (yA - K64[1, 2]) / K64[1, 1])
        Xc = torch.stack([xu, yu, torch.ones_like(xu)], dim=-1) * depth.unsqueeze(-1)
    Xw = (Xc - tA) @ RA                                                       # R^T (Xc - t)

    warp = torch.empty((len(nbrs), H, W, 4), dtype=torch.float32, device=dev)
    cert = torch.empty((len(nbrs), H, W), dtype=torch.float32, device=dev)
    smooth_lo = 8
    for k, j in enumerate(nbrs):
        camB = scene.cameras[j]
        PB = torch.from_numpy(camB.P.astype(np.float64)).to(dev)
        q = Xw @ PB[:, :3].T + PB[:, 3]
        uB = q[..., 0] / q[..., 2]
        vB = q[..., 1] / q[..., 2]
        lensB = _lens_t(camB)
        if lensB is not None:
            KB = camB.K.astype(np.float64)
            xd, yd = _distort_t(lensB, (uB - KB[0, 2]) / KB[0, 0], (vB - KB[1, 2]) / KB[1, 1])
            uB, vB = KB[0, 0] * xd + KB[0, 2], KB[1, 1] * yd + KB[1, 2]
        xBn = uB / (camB.width / float(wm)) / (0.5 * (wm - 1)) - 1.0
        yBn = vB / (camB.height / float(hm)) / (0.5 * (hm - 1)) - 1.0
        xBn = xBn + noise_sigma * torch.randn((H, W), generator=g, device=dev, dtype=torch.float64)
        yBn = yBn + noise_sigma * torch.randn((H, W), generator=g, device=dev, dtype=torch.float64)
        bad = torch.rand((H, W), generator=g, device=dev) < outlier_frac
        rx = torch.rand((H, W), generator=g, device=dev, dtype=torch.float64) * 2 - 1
        ry = torch.rand((H, W), generator=g, device=dev, dtype=torch.float64) * 2 - 1
        if lensA is not None or lensB is not None:      # no valid inverse at this pixel: an outlier like the others
            bad = bad | ~torch.isfinite(xBn) | ~torch.isfinite(yBn)
        xBn = torch.where(bad, rx, xBn)
        yBn = torch.where(bad, ry, yBn)
        warp[k, ..., 0] = gx
        warp[k, ..., 1] = gy
        warp[k, ..., 2] = xBn.float()
        warp[k, ..., 3] = yBn.float()
        if cert_family == "R":
            lo = torch.randn((1, 1, smooth_lo, smooth_lo), generator=g, device=dev)
            field = torch.nn.functional.interpolate(lo, size=(H, W), mode="bicubic", align_corners=False)[0, 0]
            logit = 3.0 * field + 1.0 + 0.7 * torch.randn((H, W), generator=g, device=dev)
            c = torch.sigmoid(logit)
            c = torch.where(bad, c * 0.5, c)
            cert[k] = torch.clamp(c, min=certainty_thresh)
    if cert_family == "T":
        n = cert.numel()
        perm = torch.randperm(n, generator=g, device=dev)
        vals = 0.2 + 0.7 * (perm.double() + 0.5) / n
        cert = vals.float().reshape(cert.shape)
    elif cert_family != "R":
        raise ValueError("cert_family must be 'T' or 'R'")
    image = torch.randint(0, 256, (hm, wm, 3), generator=g, device=dev, dtype=torch.uint8)
    out = {"cert": cert, "warp": warp, "image": image, "ref_index": ref_i, "nbr_indices": nbrs}
    if return_points:
        out["points"] = Xw
    return out
