"""Device-resident batched engine above the C ABI.

``RefBatch`` describes n reference views whose matcher outputs (certainty / warp planes, resized
reference image) already live on one CUDA device -- by pointer, nothing is stacked or copied -- plus
their camera constants.  ``DensifyEngine.densify`` runs the whole path for the batch in one call of
``ldp_densify_refs`` on the current torch stream and returns device tensors.

PyTorch is used for device memory and streams only; all compute is in csrc/.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _native as N
from .core.camera_models import CameraRecord, check_lens
from .core.geometry import fundamental_from_world2cam

# 64-bit word offsets of the pointer fields inside an ldp_ref_desc (patched per call without numpy field lookups)
_CERT_WORD = N.REF_DESC_DTYPE.fields["cert"][1] // 8
_WARP_WORD = N.REF_DESC_DTYPE.fields["warp"][1] // 8
_IMAGE_WORD = N.REF_DESC_DTYPE.fields["image"][1] // 8
assert N.REF_DESC_DTYPE.itemsize % 8 == 0

_LENS_MODELS = {None: N.LDP_LENS_PINHOLE, "opencv": N.LDP_LENS_OPENCV, "fisheye": N.LDP_LENS_FISHEYE}


def lens_of(cam: CameraRecord) -> N.LdpLens:
    """The ldp_lens of a record: its lens model and coefficients, and the f32 K entries that built its P and F."""
    check_lens(cam)
    model = getattr(cam, "lens_model", None)
    L = N.LdpLens()
    L.model = _LENS_MODELS[model]
    K = np.asarray(cam.K, dtype=np.float32)
    L.fx, L.fy, L.cx, L.cy = float(K[0, 0]), float(K[1, 1]), float(K[0, 2]), float(K[1, 2])
    if model is not None:
        for i, c in enumerate(np.asarray(cam.lens_coeffs, dtype=np.float64)):
            L.k[i] = float(c)
    return L


def _fill_lens(field, cam: CameraRecord) -> None:
    L = lens_of(cam)
    field["model"] = L.model
    field["fx"], field["fy"], field["cx"], field["cy"] = L.fx, L.fy, L.cx, L.cy
    field["k"] = np.frombuffer(bytes(L.k), dtype=np.float64)


SAMPLE_CAP_DEFAULT = 0.9     # matcher.sample_thresh, reference core/matcher.py:92
BORDER_DEFAULT = 2           # reference core/pipeline.py:646
TILES_DEFAULT = 24           # reference core/pipeline.py:647


@dataclass
class PathConfig:
    """Scalars of the path (subset of DensePipelineConfig + _TriangulationContext)."""
    matches_per_ref: int = 10000
    reproj_thresh: float = 0.8
    sampson_thresh: float = 5.0
    min_parallax_deg: float = 0.5
    no_filter: bool = False
    sample_cap: float = SAMPLE_CAP_DEFAULT
    border: int = BORDER_DEFAULT
    tiles: int = TILES_DEFAULT
    seed: int = 0
    # None: certainty planes are already post-processed (what the reference's _triangulate_ref receives).
    # A float: the planes are RAW matcher outputs and the kernels apply clamp(min=certainty_floor) and the masks
    # registered with RefBatch.add on the fly (reference core/pipeline.py:405-430, config.certainty_thresh).
    certainty_floor: Optional[float] = None
    # Multi-view refinement (include/ldp_b200.h): a kept point is re-triangulated from every other neighbour whose certainty at
    # the pixel is >= multiview_min_certainty and whose match agrees; which points are kept does not change.
    multiview: bool = False
    multiview_min_certainty: float = 0.5

    @classmethod
    def from_pipeline_config(cls, cfg, sample_cap: float = SAMPLE_CAP_DEFAULT) -> "PathConfig":
        return cls(matches_per_ref=int(cfg.matches_per_ref), reproj_thresh=float(cfg.reproj_thresh),
                   sampson_thresh=float(cfg.sampson_thresh), min_parallax_deg=float(cfg.min_parallax_deg),
                   no_filter=bool(cfg.no_filter), sample_cap=float(sample_cap), seed=int(getattr(cfg, "seed", 0)),
                   multiview=bool(getattr(cfg, "multiview", False)),
                   multiview_min_certainty=float(getattr(cfg, "multiview_min_certainty", 0.5)))

    def check_multiview(self) -> None:
        if not self.multiview:
            return
        if self.no_filter:
            raise ValueError("multiview needs the filters: it cannot be combined with no_filter")
        if not 0.0 < float(self.multiview_min_certainty) <= 1.0:
            raise ValueError("multiview_min_certainty must lie in (0, 1]")


class PairConstantCache:
    """Per (reference, neighbour) camera constants, computed once on the host with the reference's
    float32 numpy arithmetic (reference core/geometry.py:122-130), and whole descriptor rows with every camera constant of a
    (reference view, neighbour list) filled in.  Keys are object identities (the records are pinned so an id cannot be
    recycled): two scenes may reuse camera uids with other poses."""
    MAX_ROWS = 8192

    def __init__(self) -> None:
        self._F: Dict[Tuple[int, int], tuple] = {}
        self._rows: Dict[tuple, tuple] = {}

    def row_template(self, key: tuple, pins: tuple, make):
        hit = self._rows.get(key)
        if hit is None:
            if len(self._rows) >= self.MAX_ROWS:
                self._rows.clear()
            hit = (make(), pins)
            self._rows[key] = hit
        return hit[0]

    def fundamental(self, a: CameraRecord, b: CameraRecord) -> np.ndarray:
        key = (id(a), id(b))
        hit = self._F.get(key)
        if hit is None:
            F = np.ascontiguousarray(fundamental_from_world2cam(a.K, a.R, a.t, b.K, b.R, b.t), dtype=np.float32)
            hit = (F, a, b)            # pin the records so their ids cannot be recycled
            self._F[key] = hit
        return hit[0]


class RefBatch:
    """n reference views resident on one CUDA device, described by pointer."""

    def __init__(self, H: int, W: int, w_match: int, h_match: int, device: torch.device,
                 pair_cache: Optional[PairConstantCache] = None) -> None:
        self.H, self.W, self.w_match, self.h_match = int(H), int(W), int(w_match), int(h_match)
        self.device = torch.device(device)
        self._arr = np.zeros((16,), dtype=N.REF_DESC_DTYPE)       # descriptor rows, grown by doubling
        self._n = 0
        self._keep_alive: List[object] = []
        self.nbr_uids: List[List[int]] = []
        self.ref_uids: List[int] = []
        self.force_scalar_loads = False
        self.has_warped_masks = False        # some neighbour mask (mask_b) was registered: the warp planes are read per pixel
        self.has_lens = False                # some camera carries a lens model: the geometry kernels' lens instantiation runs
        self.pairs = pair_cache or PairConstantCache()

    def __len__(self) -> int:
        return self._n

    def _new_row(self, template: Optional[np.ndarray] = None):
        """Next descriptor row (a view into the batch's array), initialised from ``template`` or zeroed; also returns the
        row as uint64 words for pointer patching without numpy field lookups."""
        if self._n == self._arr.shape[0]:
            grown = np.zeros((2 * self._n,), dtype=N.REF_DESC_DTYPE)
            grown[:self._n] = self._arr
            self._arr = grown
        i = self._n
        self._n += 1
        if template is not None:
            self._arr[i] = template
        else:
            self._arr[i] = np.zeros((), dtype=N.REF_DESC_DTYPE)
        words = self._arr.view(np.uint64).reshape(self._arr.shape[0], -1)[i]
        return self._arr[i:i + 1], words

    def _check_plane(self, t: torch.Tensor, shape, what: str, allow_pinned_host: bool = False) -> torch.Tensor:
        if not isinstance(t, torch.Tensor):
            raise ValueError(f"{what} must be a tensor")
        if t.device != self.device:
            # Warp planes are read only at the ~9k sampled pixels of a view, and certainty planes exactly once, front
            # to back: both may stay in pinned (page-locked, UVA-mapped) host memory and be read over PCIe by the
            # kernels instead of being uploaded first.
            if not (allow_pinned_host and t.device.type == "cpu" and t.is_pinned()):
                raise ValueError(f"{what} must be a tensor on {self.device}"
                                 + (" or in pinned host memory" if allow_pinned_host else ""))
        if t.dtype != torch.float32 or tuple(t.shape) != tuple(shape):
            raise ValueError(f"{what} must be float32 {tuple(shape)}, got {t.dtype} {tuple(t.shape)}")
        if not t.is_contiguous():
            t = t.contiguous()
        return t

    def add(self, cert_planes: Sequence[torch.Tensor], warp_planes: Sequence[torch.Tensor], image: torch.Tensor,
            ref_cam: CameraRecord, nbr_cams: Sequence[CameraRecord], rng_stream: int = 0,
            weight_sum_override: float = 0.0, mask_a: Optional[torch.Tensor] = None,
            masks_b: Optional[Sequence[Optional[torch.Tensor]]] = None) -> None:
        """``mask_a`` / ``masks_b[k]``: uint8 [mask_h, mask_w] device tensors (``packed.maskA_np`` / ``packed.nn_masks``),
        read only when ``PathConfig.certainty_floor`` is set (raw certainty planes)."""
        nn = len(cert_planes)
        if nn != len(warp_planes) or nn != len(nbr_cams):
            raise ValueError("cert_planes, warp_planes and nbr_cams must have the same length")
        if nn > N.LDP_MAX_NN:
            raise ValueError(f"at most {N.LDP_MAX_NN} neighbours per reference view")
        if image.device != self.device or image.dtype != torch.uint8 or image.dim() != 3 or image.shape[2] != 3:
            raise ValueError("image must be a uint8 [h, w, 3] tensor on the batch device")
        image = image.contiguous()
        ih, iw = int(image.shape[0]), int(image.shape[1])
        uids = [int(c.uid) for c in nbr_cams]

        def make_template():
            """every camera constant of this (reference view, neighbour list): computed once, copied per call"""
            t = np.zeros((), dtype=N.REF_DESC_DTYPE)
            wm, hm = float(self.w_match), float(self.h_match)
            t["nn"] = nn
            t["img_w"], t["img_h"] = iw, ih
            # python-float scale factors rounded to f32 at the multiply (NEP 50), reference core/pipeline.py:662-663,681-682
            t["sxA"], t["syA"] = np.float32(ref_cam.width / wm), np.float32(ref_cam.height / hm)
            t["sx_img"], t["sy_img"] = np.float32(iw / wm), np.float32(ih / hm)
            t["P1"] = np.asarray(ref_cam.P, dtype=np.float32).reshape(12)
            t["C1"] = np.asarray(ref_cam.C, dtype=np.float32).reshape(3)
            for k, cam in enumerate(nbr_cams):
                t["P2"][k] = np.asarray(cam.P, dtype=np.float32).reshape(12)
                t["C2"][k] = np.asarray(cam.C, dtype=np.float32).reshape(3)
                t["F"][k] = self.pairs.fundamental(ref_cam, cam).reshape(9)
                t["sxB"][k], t["syB"][k] = np.float32(cam.width / wm), np.float32(cam.height / hm)
                t["group"][k] = uids.index(uids[k])          # the reference groups by neighbour uid
            if any(getattr(c, "lens_model", None) is not None for c in (ref_cam, *nbr_cams)):
                _fill_lens(t["lens_a"], ref_cam)
                for k, cam in enumerate(nbr_cams):
                    _fill_lens(t["lens_b"][k], cam)
            return t

        key = (id(ref_cam), tuple(id(c) for c in nbr_cams), self.w_match, self.h_match, iw, ih)
        row1, words = self._new_row(self.pairs.row_template(key, (ref_cam, tuple(nbr_cams)), make_template))
        if any(getattr(c, "lens_model", None) is not None for c in (ref_cam, *nbr_cams)):
            self.has_lens = True
        for k in range(nn):
            c = self._check_plane(cert_planes[k], (self.H, self.W), "certainty plane", allow_pinned_host=True)
            w = self._check_plane(warp_planes[k], (self.H, self.W, 4), "warp plane", allow_pinned_host=True)
            cp, wp = c.data_ptr(), w.data_ptr()
            if cp % 16 != 0:
                self.force_scalar_loads = True
            if wp % 16 != 0:
                raise ValueError("warp planes must be 16-byte aligned")
            words[_CERT_WORD + k] = cp
            words[_WARP_WORD + k] = wp
            self._keep_alive += [c, w]
        self._keep_alive.append(image)
        words[_IMAGE_WORD] = image.data_ptr()
        row1["rng_stream"] = np.uint32(int(rng_stream) & 0xFFFFFFFF)
        if weight_sum_override:
            row1["weight_sum_override"] = np.float32(weight_sum_override)
        self._add_masks(row1, nn, mask_a, masks_b)
        self.nbr_uids.append(uids)
        self.ref_uids.append(int(ref_cam.uid))

    def _add_masks(self, row, nn: int, mask_a, masks_b) -> None:
        if mask_a is None and masks_b is None:
            return
        masks = [mask_a] + list(masks_b if masks_b is not None else [])
        if len(masks) - 1 not in (0, nn):
            raise ValueError("masks_b must have one entry (tensor or None) per neighbour")
        shape = None
        for j, m in enumerate(masks):
            if m is None:
                continue
            if not isinstance(m, torch.Tensor) or m.device != self.device or m.dtype != torch.uint8 or m.dim() != 2:
                raise ValueError("masks must be uint8 [h, w] tensors on the batch device")
            m = m.contiguous()
            if shape is None:
                shape = tuple(m.shape)
            elif tuple(m.shape) != shape:
                raise ValueError("all masks of a reference view must share one resolution")
            self._keep_alive.append(m)
            if j == 0:
                row["mask_a"][0] = m.data_ptr()
            else:
                row["mask_b"][0, j - 1] = m.data_ptr()
                self.has_warped_masks = True
        if shape is not None:
            mh, mw = shape
            row["mask_w"][0], row["mask_h"][0] = mw, mh
            # F.interpolate(mode="nearest") scale: f32(in) / f32(out) (reference core/pipeline.py:373-378)
            row["mask_sx"][0] = np.float32(mw) / np.float32(self.W)
            row["mask_sy"][0] = np.float32(mh) / np.float32(self.H)

    def add_cert_only(self, cert_planes: Sequence[torch.Tensor], rng_stream: int = 0,
                      weight_sum_override: float = 0.0) -> None:
        """A view described by its certainty planes only -- enough for the sampling stage (``ldp_sample_refs``)."""
        nn = len(cert_planes)
        if nn > N.LDP_MAX_NN:
            raise ValueError(f"at most {N.LDP_MAX_NN} neighbours per reference view")
        row1, words = self._new_row()
        for k in range(nn):
            c = self._check_plane(cert_planes[k], (self.H, self.W), "certainty plane", allow_pinned_host=True)
            if c.data_ptr() % 16 != 0:
                self.force_scalar_loads = True
            words[_CERT_WORD + k] = c.data_ptr()
            self._keep_alive.append(c)
        row1["nn"] = nn
        row1["rng_stream"] = np.uint32(int(rng_stream) & 0xFFFFFFFF)
        row1["weight_sum_override"] = np.float32(weight_sum_override)
        self.nbr_uids.append(list(range(nn)))
        self.ref_uids.append(self._n - 1)

    def desc_array(self) -> np.ndarray:
        return self._arr[:self._n]


@dataclass
class DensifyOutputs:
    """Device tensors written by one launch (see include/ldp_b200.h:ldp_outputs)."""
    n_refs: int
    sel_cap: int
    xyz: torch.Tensor
    rgb: torch.Tensor
    err: torch.Tensor
    ref_offset: torch.Tensor
    status: torch.Tensor
    n_samples: torch.Tensor
    group_count: torch.Tensor
    group_order: torch.Tensor
    uniforms_used: torch.Tensor
    rounds: torch.Tensor
    weight_sum: torch.Tensor
    dbg_matches: Optional[torch.Tensor] = None
    dbg_cert: Optional[torch.Tensor] = None
    view_mask: Optional[torch.Tensor] = None   # int32 [capacity], multiview launches: neighbour slots behind each point
    sel_idx: Optional[torch.Tensor] = None
    sample_flags: Optional[torch.Tensor] = None
    sample_xyzerr: Optional[torch.Tensor] = None
    launches: int = 0
    packed: Optional[torch.Tensor] = None      # the u8 allocation behind ref_offset | status words | xyz | rgb | err [| debug]
    layout: Optional[dict] = None              # name -> (byte offset, bytes) inside ``packed``
    ready: Optional[torch.cuda.Event] = None   # DensifyRing: recorded on the ring stream after the launch sequence

    def total_points(self) -> int:
        """Synchronises."""
        return int(self.ref_offset[-1].item()) if self.n_refs else 0


class DensifyEngine:
    """Owns the scratch workspace and enqueues launches on the current torch CUDA stream."""

    def __init__(self, device=None) -> None:
        if not torch.cuda.is_available():
            raise N.NativeLibraryError("DensifyEngine needs a CUDA device (there is no CPU fallback)")
        self.lib = N.load()
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self._workspace: Optional[torch.Tensor] = None
        self.sm_reserve = -1         # SMs the first draw kernel leaves to other launches in flight (-1: process default, 0: none)
        self.pairs = PairConstantCache()

    def new_batch(self, H: int, W: int, w_match: int, h_match: int) -> RefBatch:
        return RefBatch(H, W, w_match, h_match, self.device, self.pairs)

    def _params(self, batch: RefBatch, cfg: PathConfig, collect_debug: bool, rng_mode: int,
                uniforms_per_ref: int) -> N.LdpParams:
        p = N.LdpParams()
        p.n_refs = len(batch)
        p.H, p.W, p.w_match, p.h_match = batch.H, batch.W, batch.w_match, batch.h_match
        p.matches_per_ref = int(cfg.matches_per_ref)
        p.border, p.tiles = int(cfg.border), int(cfg.tiles)
        p.sample_cap = float(np.float32(cfg.sample_cap))
        p.reproj_thresh = float(np.float32(cfg.reproj_thresh))
        p.min_parallax_deg = float(np.float32(cfg.min_parallax_deg))
        p.sampson_thresh = float(cfg.sampson_thresh)
        p.no_filter = 1 if cfg.no_filter else 0
        p.collect_debug = 1 if collect_debug else 0
        p.rng_mode = int(rng_mode)
        p.scalar_loads = 1 if batch.force_scalar_loads else 0
        p.nn_max = max((len(u) for u in batch.nbr_uids), default=0)
        p.prologue = 0 if cfg.certainty_floor is None else 1
        p.certainty_floor = float(np.float32(cfg.certainty_floor if cfg.certainty_floor is not None else 0.0))
        p.no_warped_masks = 0 if batch.has_warped_masks else 1
        p.lens = 1 if batch.has_lens else 0
        cfg.check_multiview()
        p.multiview = 1 if cfg.multiview else 0
        p.multiview_min_cert = float(np.float32(cfg.multiview_min_certainty))
        p.sm_reserve = int(self.sm_reserve)
        p.seed = int(cfg.seed) & 0xFFFFFFFFFFFFFFFF
        p.uniforms_per_ref = int(uniforms_per_ref)
        return p

    def _ensure_workspace(self, params: N.LdpParams) -> torch.Tensor:
        need = C.c_size_t(0)
        N.check(self.lib.ldp_workspace_bytes(C.byref(params), C.byref(need)), "ldp_workspace_bytes")
        if self._workspace is None or self._workspace.numel() < need.value:
            self._workspace = None
            self._workspace = torch.empty(int(need.value), dtype=torch.uint8, device=self.device)
        return self._workspace

    def sel_capacity(self, matches_per_ref: int) -> int:
        return int(self.lib.ldp_sel_capacity(int(matches_per_ref)))

    def upload_descs(self, batch: RefBatch) -> torch.Tensor:
        arr = batch.desc_array()
        host = torch.from_numpy(arr.view(np.uint8).reshape(-1))
        return host.to(self.device, non_blocking=False)

    def prepare(self, batch: RefBatch, cfg: PathConfig, uniforms: Optional[torch.Tensor] = None,
                collect_debug: bool = False, taps: bool = False, descs_dev: Optional[torch.Tensor] = None,
                outputs: Optional[DensifyOutputs] = None) -> "PreparedLaunch":
        """Everything ``densify`` does on the host except the call itself: parameter block, workspace, descriptor upload,
        output allocation.  ``PreparedLaunch.launch()`` can then be repeated (same batch, same outputs) at the cost of one
        C call - for callers that re-run a batch or keep several launches in flight."""
        R = len(batch)
        dev = self.device
        rng_mode = N.LDP_RNG_PHILOX
        upr = 0
        if uniforms is not None:
            if uniforms.dtype != torch.float64 or uniforms.device != dev or uniforms.dim() != 2 or uniforms.shape[0] != R:
                raise ValueError("uniforms must be a float64 [n_refs, U] tensor on the engine device")
            uniforms = uniforms.contiguous()
            rng_mode = N.LDP_RNG_EXPLICIT
            upr = int(uniforms.shape[1])
        params = self._params(batch, cfg, collect_debug, rng_mode, upr)
        ws = self._ensure_workspace(params)
        sel_cap = self.sel_capacity(cfg.matches_per_ref)
        out = outputs if outputs is not None else self.alloc_outputs(R, sel_cap, collect_debug, taps, multiview=cfg.multiview)
        if cfg.multiview and out.view_mask is None:
            raise ValueError("a multiview launch needs outputs allocated with multiview=True")
        if descs_dev is None:
            descs_dev = self.upload_descs(batch)
        o = N.LdpOutputs()
        o.xyz, o.rgb, o.err = out.xyz.data_ptr(), out.rgb.data_ptr(), out.err.data_ptr()
        o.capacity = int(out.err.shape[0])
        o.ref_offset, o.status, o.n_samples = out.ref_offset.data_ptr(), out.status.data_ptr(), out.n_samples.data_ptr()
        o.group_count, o.group_order = out.group_count.data_ptr(), out.group_order.data_ptr()
        o.uniforms_used, o.rounds, o.weight_sum = out.uniforms_used.data_ptr(), out.rounds.data_ptr(), out.weight_sum.data_ptr()
        if out.dbg_matches is not None:
            o.dbg_matches, o.dbg_cert = out.dbg_matches.data_ptr(), out.dbg_cert.data_ptr()
        if cfg.multiview:
            o.view_mask = out.view_mask.data_ptr()
        if out.sel_idx is not None:
            o.sel_idx = out.sel_idx.data_ptr()
        if out.sample_flags is not None:
            o.sample_flags, o.sample_xyzerr = out.sample_flags.data_ptr(), out.sample_xyzerr.data_ptr()
        out._keep = (descs_dev, uniforms, batch)      # keep inputs alive until the stream is done with them
        return PreparedLaunch(self, params, o, out, descs_dev, uniforms, ws)

    def densify(self, batch: RefBatch, cfg: PathConfig, uniforms: Optional[torch.Tensor] = None,
                collect_debug: bool = False, taps: bool = False, descs_dev: Optional[torch.Tensor] = None,
                outputs: Optional[DensifyOutputs] = None) -> DensifyOutputs:
        """Run the whole path for ``batch``.  ``uniforms``: f64 [n_refs, U] device tensor selects the
        explicit (parity) RNG mode; otherwise Philox keyed by (cfg.seed, rng_stream)."""
        return self.prepare(batch, cfg, uniforms, collect_debug, taps, descs_dev, outputs).launch()

    def postprocess_certainty(self, batch: RefBatch, certainty_floor: float) -> torch.Tensor:
        """``ldp_postprocess_certainty``: the reference's certainty post-processing alone (core/pipeline.py:405-430).
        Returns f32 [n_refs, nn_max, H, W] (planes beyond a view's neighbour count are zero)."""
        R = len(batch)
        nn_max = max((len(u) for u in batch.nbr_uids), default=0)
        out = torch.zeros((R, max(nn_max, 1), batch.H, batch.W), dtype=torch.float32, device=self.device)
        if R == 0 or nn_max == 0:
            return out
        params = self._params(batch, PathConfig(certainty_floor=float(certainty_floor)), False, N.LDP_RNG_PHILOX, 0)
        descs = self.upload_descs(batch)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        rc = self.lib.ldp_postprocess_certainty(C.byref(params), C.c_void_p(descs.data_ptr()), C.c_void_p(out.data_ptr()),
                                                C.c_size_t(out.stride(0)), C.c_size_t(out.stride(1)), C.c_void_p(stream))
        N.check(rc, "ldp_postprocess_certainty")
        out._keep = (descs, batch)
        return out

    def sample(self, batch: RefBatch, cfg: PathConfig, uniforms: Optional[torch.Tensor] = None):
        """Sampling stage only (``ldp_sample_refs``): returns (sel_idx [R, sel_cap] i32, n_samples, status, uniforms_used)."""
        R = len(batch)
        dev = self.device
        rng_mode, upr = N.LDP_RNG_PHILOX, 0
        if uniforms is not None:
            uniforms = uniforms.contiguous()
            rng_mode, upr = N.LDP_RNG_EXPLICIT, int(uniforms.shape[1])
        params = self._params(batch, cfg, False, rng_mode, upr)
        ws = self._ensure_workspace(params)
        sel_cap = self.sel_capacity(cfg.matches_per_ref)
        sel = torch.zeros((R, sel_cap), dtype=torch.int32, device=dev)
        n_samples = torch.zeros((R,), dtype=torch.int32, device=dev)
        status = torch.zeros((R,), dtype=torch.int32, device=dev)
        used = torch.zeros((R,), dtype=torch.int32, device=dev)
        rounds = torch.zeros((R,), dtype=torch.int32, device=dev)
        wsum = torch.zeros((R,), dtype=torch.float32, device=dev)
        descs = self.upload_descs(batch)
        o = N.LdpOutputs()
        o.status, o.n_samples, o.sel_idx = status.data_ptr(), n_samples.data_ptr(), sel.data_ptr()
        o.uniforms_used, o.rounds, o.weight_sum = used.data_ptr(), rounds.data_ptr(), wsum.data_ptr()
        stream = torch.cuda.current_stream(dev).cuda_stream
        rc = self.lib.ldp_sample_refs(C.byref(params), C.c_void_p(descs.data_ptr()),
                                      C.c_void_p(uniforms.data_ptr() if uniforms is not None else 0), C.byref(o),
                                      C.c_void_p(ws.data_ptr()), C.c_size_t(ws.numel()), C.c_void_p(stream))
        N.check(rc, "ldp_sample_refs")
        torch.cuda.current_stream(dev).synchronize()
        return sel, n_samples, status, used

    def undistort_pixels(self, uv: torch.Tensor, record: CameraRecord) -> torch.Tensor:
        """``ldp_undistort_points``: the ideal pinhole pixels of the observed pixels ``uv`` (f32 [n, 2] on the engine device)
        of camera ``record``, NaN where its lens has no valid inverse - the inversion the geometry kernels apply.  Enqueued
        on the current stream; a record without a lens returns a copy."""
        if not isinstance(uv, torch.Tensor) or uv.device != self.device or uv.dtype != torch.float32 or uv.dim() != 2 \
                or uv.shape[1] != 2:
            raise ValueError(f"uv must be a float32 [n, 2] tensor on {self.device}")
        uv = uv.contiguous()
        out = torch.empty_like(uv)
        L = lens_of(record)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        rc = self.lib.ldp_undistort_points(C.byref(L), int(uv.shape[0]), C.c_void_p(uv.data_ptr()), C.c_void_p(out.data_ptr()),
                                           C.c_void_p(stream))
        N.check(rc, "ldp_undistort_points")
        return out

    def alloc_outputs(self, R: int, sel_cap: int, collect_debug: bool = False, taps: bool = False,
                      multiview: bool = False) -> DensifyOutputs:
        """Everything a caller reads back lives in ONE allocation (``packed``): ref_offset | per-view status words | xyz | rgb |
        err [| debug matches | debug certainties] [| view masks] - a rank hands its whole result to a single collective
        (``distributed`` / bench.py) and the drop-in path reads it back with a single device->host copy."""
        dev = self.device
        cap = max(1, R * sel_cap)
        i32 = dict(dtype=torch.int32, device=dev)
        NN = N.LDP_MAX_NN
        sizes = [("ref_offset", 8 * (R + 1)), ("status", 4 * R), ("n_samples", 4 * R), ("uniforms_used", 4 * R), ("rounds", 4 * R),
                 ("weight_sum", 4 * R), ("group_count", 4 * R * NN), ("group_order", 4 * R * NN),
                 ("xyz", 12 * cap), ("rgb", 12 * cap), ("err", 4 * cap)]
        if collect_debug:
            sizes += [("dbg_matches", 16 * cap), ("dbg_cert", 4 * cap)]
        if multiview:
            sizes += [("view_mask", 4 * cap)]
        off, layout = 0, {}
        for name, nbytes in sizes:
            off = (off + 15) // 16 * 16
            layout[name] = (off, nbytes)
            off += nbytes
        packed = torch.zeros((off,), dtype=torch.uint8, device=dev)

        def view(name, dtype, shape):
            a, n = layout[name]
            return packed[a:a + n].view(dtype).view(*shape)

        out = DensifyOutputs(
            n_refs=R, sel_cap=sel_cap,
            xyz=view("xyz", torch.float32, (cap, 3)), rgb=view("rgb", torch.float32, (cap, 3)), err=view("err", torch.float32, (cap,)),
            ref_offset=view("ref_offset", torch.int64, (R + 1,)),
            status=view("status", torch.int32, (R,)), n_samples=view("n_samples", torch.int32, (R,)),
            group_count=view("group_count", torch.int32, (R, NN)), group_order=view("group_order", torch.int32, (R, NN)),
            uniforms_used=view("uniforms_used", torch.int32, (R,)), rounds=view("rounds", torch.int32, (R,)),
            weight_sum=view("weight_sum", torch.float32, (R,)),
        )
        out.group_order.fill_(-1)
        out.packed = packed
        out.layout = layout
        if collect_debug:
            out.dbg_matches = view("dbg_matches", torch.float32, (cap, 4))
            out.dbg_cert = view("dbg_cert", torch.float32, (cap,))
        if multiview:
            out.view_mask = view("view_mask", torch.int32, (cap,))
        if taps:
            out.sel_idx = torch.zeros((R, sel_cap), **i32)
            out.sample_flags = torch.zeros((R, sel_cap), dtype=torch.uint8, device=dev)
            out.sample_xyzerr = torch.zeros((R, sel_cap, 4), dtype=torch.float32, device=dev)
        return out


class PreparedLaunch:
    """A launch of the path with its host-side arguments frozen (``DensifyEngine.prepare``)."""

    def __init__(self, engine: "DensifyEngine", params, c_outputs, outputs: DensifyOutputs, descs_dev, uniforms, workspace) -> None:
        self.engine, self.params, self.c_outputs, self.outputs = engine, params, c_outputs, outputs
        self.descs_dev, self.uniforms, self.workspace = descs_dev, uniforms, workspace
        self._args = (C.byref(params), C.c_void_p(descs_dev.data_ptr()),
                      C.c_void_p(uniforms.data_ptr() if uniforms is not None else 0), C.byref(c_outputs),
                      C.c_void_p(workspace.data_ptr()), C.c_size_t(workspace.numel()))

    def launch(self) -> DensifyOutputs:
        """Enqueue the launch sequence on the current torch CUDA stream."""
        eng = self.engine
        if eng._workspace is not self.workspace:
            raise RuntimeError("the engine's workspace was re-allocated for a larger launch: prepare() again")
        stream = torch.cuda.current_stream(eng.device).cuda_stream
        rc = eng.lib.ldp_densify_refs(*self._args, C.c_void_p(stream))
        N.check(rc, "ldp_densify_refs")
        self.outputs.launches = int(eng.lib.ldp_last_launch_count())
        return self.outputs


class DensifyRing:
    """Several launches in flight: a caller with more than one batch of views (a large scene cut into launches, or one
    scene after another) submits them round-robin to ``depth`` engines, each with its own workspace and CUDA stream.
    The kernels of a launch sequence are bound by different things - the first streams HBM, the draw and geometry
    kernels are latency / issue bound and leave most of the memory system idle - so consecutive launches overlap:
    measured 175 -> 152 -> 145 us per 46-view launch at depth 1 / 2 / 3 (``scratch/two_streams.py``).  Results are
    those of ``DensifyEngine.densify`` (same kernels, same RNG streams); only the scheduling differs."""

    def __init__(self, device=None, depth: int = 3, sm_reserve: int = 16) -> None:
        if depth < 1:
            raise ValueError("depth must be >= 1")
        self.engines = [DensifyEngine(device) for _ in range(depth)]
        for e in self.engines:       # per engine (passed with every call): the first draw kernel leaves SMs to the other launches in flight
            e.sm_reserve = int(sm_reserve) if depth > 1 else 0
        self.device = self.engines[0].device
        self.streams = [torch.cuda.Stream(self.device) for _ in range(depth)]
        self.depth = depth
        self._n = 0

    def slot(self) -> int:
        """Index of the engine / stream the next ``submit`` uses."""
        return self._n % self.depth

    def submit(self, batch: RefBatch, cfg: PathConfig, **kw) -> DensifyOutputs:
        """Enqueue ``DensifyEngine.densify(batch, cfg, **kw)`` on the next ring stream, ordered after the work already on
        the caller's current stream (which produced the inputs).  ``outputs.ready`` is recorded behind it."""
        j = self._n % self.depth
        self._n += 1
        st = self.streams[j]
        st.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(st):
            out = self.engines[j].densify(batch, cfg, **kw)
            out.ready = torch.cuda.Event()
            out.ready.record(st)
        return out

    def wait(self, out: DensifyOutputs) -> None:
        """Order the caller's current stream after ``out``."""
        if out.ready is not None:
            torch.cuda.current_stream(self.device).wait_event(out.ready)

    def synchronize(self) -> None:
        for st in self.streams:
            st.synchronize()
