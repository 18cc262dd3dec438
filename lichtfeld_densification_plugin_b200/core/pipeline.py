"""Drop-in host interface of the densification path.

Keeps the reference's names, argument meaning and error behaviour for this path
(reference core/pipeline.py):

* ``PipelineResult``                          :37-43
* ``_PackedReferenceBatch`` / ``_CameraLookup`` / ``_MatchedReference`` / ``_TriangulationContext`` /
  ``_TriangulatedReference``                  :53-114
* ``_build_camera_lookup``                    :270-281
* ``_triangulate_ref(matched_ref, tri_ctx, collect_debug_matches)``  :602-780  (one view, host or device tensors)
* ``run_dense_pipeline(...) -> PipelineResult``                      :783-928  (the matcher is supplied by the caller:
  the RoMa network is out of scope)

plus the batched form the B200 path is built for: ``triangulate_refs`` processes every reference view
of a rank in ONE launch sequence.  All compute happens in the CUDA library; without it these functions
raise (no CPU fallback).
"""
from __future__ import annotations

import json
import os
import time
from dataclasses import dataclass, field
from typing import Callable, Dict, Iterable, List, Optional, Sequence, Tuple

import numpy as np
import torch

from .. import _native as N
from ..engine import DensifyEngine, DensifyOutputs, DepthMaps, PathConfig, RefBatch
from .camera_models import CameraRecord
from .config import RNG_EXPLICIT, RNG_NUMPY_GLOBAL, RNG_PHILOX, DensePipelineConfig


@dataclass
class PipelineResult:
    xyz: np.ndarray
    rgb: np.ndarray
    err: np.ndarray
    elapsed_seconds: float
    pairs_processed: int
    n_views: Optional[np.ndarray] = None          # extra, config.multiview: uint8 cameras per point, the reference view included
    normals: Optional[np.ndarray] = None          # extra, config.normal_neighbors: f32 [n,3] unit normals facing each point's
                                                  # reference camera; (0, 0, 0) where undefined.  Without normal_neighbors,
                                                  # config.depth_fusion_max_normal_angle: the fused normals (unit, each facing
                                                  # its source camera)
    gaussians: Optional[Dict[str, np.ndarray]] = None   # extra, config.gaussian_neighbors: 3DGS's initial splats, f32
                                                  # sh_dc [n,3], opacity [n], scales [n,3] (log), rotations [n,4] (w, x, y, z)
    depth_paths: Optional[Dict[int, str]] = None  # extra, config.depth_dir: reference camera uid -> its depth map file
    consistent_views: Optional[np.ndarray] = None  # extra, config.depth_consistency / depth_fusion: int32 per point, the other
                                                  # reference views whose depth maps agree with it
    fused_views: Optional[np.ndarray] = None      # extra, config.depth_fusion: int32 per point, the views averaged into it


class PipelineCancelled(RuntimeError):
    """Raised when a running dense pipeline is cancelled."""


_DEBUG_PREVIEW_INTERVAL = 3          # reference core/pipeline.py:34
_PREVIEW_MAX_MATCHES = 10000         # reference core/pipeline.py:50


@dataclass
class MatchPreview:
    """reference core/debug_viz.py:13-26 (what ``MatchDebugState.submit_preview`` receives)."""
    ref_id: int
    nbr_id: int
    ref_label: str
    nbr_label: str
    left_image: np.ndarray
    right_image: np.ndarray
    matches: np.ndarray
    cert_norm: np.ndarray
    match_count: int
    pair_index: int
    total_pairs: int


@dataclass
class _PackedReferenceBatch:
    ref_id: int
    ref_path: str
    imA_np: np.ndarray
    maskA_np: Optional[np.ndarray]
    wA_cam: int
    hA_cam: int
    nn_ids: List[int]
    nn_masks: List[Optional[np.ndarray]]
    nn_arrays: List[np.ndarray]


@dataclass(frozen=True)
class _CameraLookup:
    img_ids: List[int]
    path_by: Dict[int, str]
    mask_by: Dict[int, Optional[str]]
    size_by: Dict[int, Tuple[int, int]]
    K_by: Dict[int, np.ndarray]
    R_by: Dict[int, np.ndarray]
    t_by: Dict[int, np.ndarray]
    P_by: Dict[int, np.ndarray]
    C_by: Dict[int, np.ndarray]
    record_by: Dict[int, CameraRecord] = field(default_factory=dict)     # extra: uid -> record


@dataclass
class _MatchedReference:
    packed: _PackedReferenceBatch
    warp_list_cpu: List[torch.Tensor]       # host OR device tensors (device tensors skip the H2D copy)
    cert_list_cpu: List[torch.Tensor]
    pair_index_by_nbr: Dict[int, int]
    image_by_nbr: Dict[int, np.ndarray]
    # extra: True when cert_list_cpu holds RAW matcher certainties (made by this package's _collect_reference_matches):
    # the floor clamp and the masks of ``packed`` are then applied inside the kernels (reference core/pipeline.py:405-430)
    raw_certainty: bool = False


@dataclass(frozen=True)
class _TriangulationContext:
    cameras: _CameraLookup
    config: DensePipelineConfig
    matcher_sample_cap: float
    w_match: int
    h_match: int


@dataclass
class _TriangulatedReference:
    xyz: np.ndarray
    rgb: np.ndarray
    err: np.ndarray
    debug_matches_by_nbr: Dict[int, np.ndarray]
    debug_cert_by_nbr: Dict[int, np.ndarray]
    ply_records: Optional[np.ndarray] = None      # extra: this view's 15-byte PLY vertex records, packed on the device
    n_views: Optional[np.ndarray] = None          # extra, config.multiview: uint8 cameras per point, the reference view included


def _build_camera_lookup(camera_records: Sequence[CameraRecord]) -> _CameraLookup:
    recs = list(camera_records)
    return _CameraLookup(
        img_ids=[c.uid for c in recs],
        path_by={c.uid: c.image_path for c in recs},
        mask_by={c.uid: getattr(c, "mask_path", None) for c in recs},
        size_by={c.uid: (c.width, c.height) for c in recs},
        K_by={c.uid: c.K for c in recs},
        R_by={c.uid: c.R for c in recs},
        t_by={c.uid: c.t for c in recs},
        P_by={c.uid: c.P for c in recs},
        C_by={c.uid: c.C for c in recs},
        record_by={c.uid: c for c in recs},
    )


_side_tables: Dict[int, tuple] = {}      # lookups built by the reference's own helper carry no record_by: (pinned lookup, table)


def _record_for(cameras, uid: int, size: Optional[Tuple[int, int]] = None) -> CameraRecord:
    """The ``CameraRecord`` of ``uid`` - always the SAME object for the same (lookup, uid, size), so that the engine's
    per-pair constant cache (keyed by record identity) hits.  ``size``: the (width, height) a packed reference view carries
    when it differs from the camera's own (``packed.wA_cam`` / ``hA_cam``, reference core/pipeline.py:681-682)."""
    table = getattr(cameras, "record_by", None)
    if table is None:
        table = _side_tables.setdefault(id(cameras), (cameras, {}))[1]
    rec = table.get(uid)
    if rec is None:
        w, h = cameras.size_by[uid]
        rec = CameraRecord(uid=uid, image_path=cameras.path_by.get(uid, ""), width=w, height=h, K=cameras.K_by[uid],
                           R=cameras.R_by[uid], t=cameras.t_by[uid], P=cameras.P_by[uid], C=cameras.C_by[uid])
        table[uid] = rec
    if size is not None and (rec.width, rec.height) != (int(size[0]), int(size[1])):
        key = (uid, int(size[0]), int(size[1]))
        sized = table.get(key)
        if sized is None:
            sized = CameraRecord(uid=rec.uid, image_path=rec.image_path, width=int(size[0]), height=int(size[1]),
                                 K=rec.K, R=rec.R, t=rec.t, P=rec.P, C=rec.C,
                                 lens_model=getattr(rec, "lens_model", None), lens_coeffs=getattr(rec, "lens_coeffs", None))
            table[key] = sized
        rec = sized
    return rec


# ------------------------------------------------------------------------------------------------
_engines: Dict[int, DensifyEngine] = {}


def get_engine(device: Optional[torch.device] = None) -> DensifyEngine:
    if not torch.cuda.is_available():
        raise N.NativeLibraryError("the densification path needs a CUDA device (there is no CPU fallback)")
    idx = torch.cuda.current_device() if device is None else (torch.device(device).index or 0)
    eng = _engines.get(idx)
    if eng is None:
        eng = DensifyEngine(torch.device("cuda", idx))
        _engines[idx] = eng
    return eng


_rings: Dict[int, "DensifyRing"] = {}


def get_ring(device: Optional[torch.device] = None, depth: int = 3):
    """Per-device ring of engines for callers that keep several launches in flight (run_dense_pipeline with
    ``config.refs_per_launch``)."""
    from ..engine import DensifyRing
    if not torch.cuda.is_available():
        raise N.NativeLibraryError("the densification path needs a CUDA device (there is no CPU fallback)")
    idx = torch.cuda.current_device() if device is None else (torch.device(device).index or 0)
    ring = _rings.get(idx)
    if ring is None or ring.depth != depth:
        ring = DensifyRing(torch.device("cuda", idx), depth)
        _rings[idx] = ring
    return ring


def _to_device(t, device, dtype) -> torch.Tensor:
    if isinstance(t, np.ndarray):
        t = torch.from_numpy(t)
    if t.dtype != dtype:
        t = t.to(dtype)
    if t.device != device:
        t = t.to(device, non_blocking=True)
    return t.contiguous()


def _raise_for_status(code: int) -> None:
    """Same exceptions the reference path raises for a view (np.random.choice ValueErrors)."""
    code &= N.LDP_REF_CODE_MASK
    if code in (N.LDP_REF_FEWER_NONZERO, N.LDP_REF_BAD_WEIGHTS, N.LDP_REF_PSUM):
        raise ValueError(N.REF_STATUS_MESSAGES[code])
    if code in (N.LDP_REF_UNIFORMS_EXHAUSTED, N.LDP_REF_ROUNDS_EXCEEDED):
        raise RuntimeError(N.REF_STATUS_MESSAGES[code])


def _split_reference(out: DensifyOutputs, host: dict, r: int, nbr_uids: List[int],
                     collect_debug: bool) -> Optional[_TriangulatedReference]:
    a, b = int(host["ref_offset"][r]), int(host["ref_offset"][r + 1])
    if b <= a:
        return None
    dbg_m: Dict[int, np.ndarray] = {}
    dbg_c: Dict[int, np.ndarray] = {}
    if collect_debug:
        pos = a
        for g in host["group_order"][r]:
            if g < 0:
                break
            cnt = int(host["group_count"][r][g])
            if cnt > 0:
                dbg_m[nbr_uids[g]] = host["dbg_matches"][pos:pos + cnt]
                dbg_c[nbr_uids[g]] = host["dbg_cert"][pos:pos + cnt]
            pos += cnt
    rec = host["ply"][15 * a:15 * b] if "ply" in host else None
    n_views = None
    if "view_mask" in host:
        n_views = (np.bitwise_count(host["view_mask"][a:b].view(np.uint32)) + 1).astype(np.uint8)
    return _TriangulatedReference(xyz=host["xyz"][a:b], rgb=host["rgb"][a:b], err=host["err"][a:b],
                                  debug_matches_by_nbr=dbg_m, debug_cert_by_nbr=dbg_c, ply_records=rec, n_views=n_views)


def _download(out: DensifyOutputs, collect_debug: bool, ply_records: bool = False) -> dict:
    """ONE device->host copy of the launch's packed result (offsets, per-view status words, xyz, rgb, err and, when asked
    for, the debug rows: ``DensifyOutputs.packed``) into page-locked memory, one synchronisation; every array of the
    returned dict is a view of that host block.  The block is the CALLER'S: it comes from torch's caching page-locked
    allocator for this call alone and goes back to the pool when the last array that views it is dropped, so the results
    are handed out without a second copy (a memcpy of the 13 MB of a 46-view launch costs three times its PCIe transfer)."""
    rec = None
    if ply_records and out.n_refs:      # packed before the first host read: the point count is taken on the device
        from .. import output as _output
        rec = _output.ply_records(out.xyz, out.rgb, n=int(out.err.shape[0]), n_dev=out.ref_offset[-1:])
    host_t = torch.empty((int(out.packed.numel()),), dtype=torch.uint8, pin_memory=True)
    host_t.copy_(out.packed, non_blocking=True)
    torch.cuda.current_stream(out.packed.device).synchronize()
    host = host_t.numpy()
    R, NN = out.n_refs, N.LDP_MAX_NN
    L = out.layout

    def arr(name, dtype, shape):
        a, n = L[name]
        return host[a:a + n].view(dtype).reshape(shape)

    meta = {"ref_offset": arr("ref_offset", np.int64, (R + 1,))}
    total = int(meta["ref_offset"][-1]) if R else 0
    cap = int(out.err.shape[0])
    meta["status"] = arr("status", np.int32, (R,))
    meta["uniforms_used"] = arr("uniforms_used", np.int32, (R,))
    meta["group_order"] = arr("group_order", np.int32, (R, NN))
    meta["group_count"] = arr("group_count", np.int32, (R, NN))
    meta["xyz"] = arr("xyz", np.float32, (cap, 3))[:total]
    meta["rgb"] = arr("rgb", np.float32, (cap, 3))[:total]
    meta["err"] = arr("err", np.float32, (cap,))[:total]
    if collect_debug:
        meta["dbg_matches"] = arr("dbg_matches", np.float32, (cap, 4))[:total]
        meta["dbg_cert"] = arr("dbg_cert", np.float32, (cap,))[:total]
    if "view_mask" in L:
        meta["view_mask"] = arr("view_mask", np.int32, (cap,))[:total]
    if rec is not None:
        meta["ply"] = rec[:15 * total].cpu().numpy()
    return meta


def _mt_stream_from_global(n: int) -> np.ndarray:
    """The next n doubles the process-global MT19937 stream would produce, without consuming them."""
    rs = np.random.RandomState()
    rs.set_state(np.random.get_state())
    return rs.random_sample(n)


@dataclass
class _PendingLaunch:
    """A submitted launch of ``triangulate_refs`` whose results have not been read back yet."""
    out: DensifyOutputs
    batch: RefBatch
    n: int
    collect_debug: bool
    ply_records: bool
    depth: Optional[DepthMaps] = None            # config.depth_dir / depth_consistency: the launch's depth maps, written
                                                 # or kept when it is collected
    ref_cams: Optional[List[CameraRecord]] = None   # the reference camera of every view, as the launch used it


def submit_refs(matched_refs: Sequence[_MatchedReference], tri_ctx: _TriangulationContext,
                collect_debug_matches: bool = False, *, rng_streams: Optional[Sequence[int]] = None,
                uniforms: Optional[np.ndarray] = None, weight_sums: Optional[Sequence[float]] = None,
                ply_records: bool = False, ring=None) -> _PendingLaunch:
    """First half of ``triangulate_refs``: upload what is not on the device yet and enqueue the launch sequence - on the
    next stream of ``ring`` (a ``DensifyRing``: several launches in flight) or on the current stream."""
    n = len(matched_refs)
    eng = get_engine() if ring is None else ring.engines[ring.slot()]
    dev = eng.device
    cfg = tri_ctx.config
    pcfg = PathConfig.from_pipeline_config(cfg, sample_cap=tri_ctx.matcher_sample_cap)
    raw = [bool(getattr(mr, "raw_certainty", False)) for mr in matched_refs]
    if any(raw) and not all(raw):
        raise ValueError("a launch takes either raw or post-processed certainty planes, not a mix")
    if raw[0]:
        pcfg.certainty_floor = float(cfg.certainty_thresh)
    first = matched_refs[0].cert_list_cpu[0]
    H, W = int(first.shape[0]), int(first.shape[1])
    batch = eng.new_batch(H, W, tri_ctx.w_match, tri_ctx.h_match)
    ref_cams: List[CameraRecord] = []
    for i, mr in enumerate(matched_refs):
        packed = mr.packed
        certs = [_to_device(c, dev, torch.float32) for c in mr.cert_list_cpu]
        warps = [_to_device(w, dev, torch.float32) for w in mr.warp_list_cpu]
        image = _to_device(packed.imA_np, dev, torch.uint8)
        ref_cam = _record_for(tri_ctx.cameras, packed.ref_id, size=(packed.wA_cam, packed.hA_cam))
        nbrs = [_record_for(tri_ctx.cameras, uid) for uid in packed.nn_ids]
        ref_cams.append(ref_cam)
        mask_a = masks_b = None
        if raw[i]:
            mask_a = None if packed.maskA_np is None else _to_device(packed.maskA_np, dev, torch.uint8)
            masks_b = [None if m is None else _to_device(m, dev, torch.uint8) for m in packed.nn_masks]
        batch.add(certs, warps, image, ref_cam, nbrs,
                  rng_stream=(rng_streams[i] if rng_streams is not None else i),
                  weight_sum_override=(float(weight_sums[i]) if weight_sums is not None else 0.0),
                  mask_a=mask_a, masks_b=masks_b)
    u_dev = None
    if uniforms is not None:
        u_dev = torch.from_numpy(np.ascontiguousarray(uniforms, dtype=np.float64)).to(dev)
        batch._keep_alive.append(u_dev)      # read by kernels on a ring stream: alive until the launch is collected, like the planes
    depth = None
    fusion = bool(getattr(cfg, "depth_fusion", False))
    want_depth = bool(getattr(cfg, "depth_dir", "")) or bool(getattr(cfg, "depth_consistency", False)) or fusion
    maps = dict(want_err=True, want_xyz=True, want_rgb=True) if fusion else (dict(want_xyz=True) if _normal_radius(cfg) else {})
    if ring is None:
        out = eng.densify(batch, pcfg, uniforms=u_dev, collect_debug=collect_debug_matches)
        if want_depth:
            depth = eng.depth_maps(batch, pcfg, float(cfg.depth_min_certainty), **maps)
    else:
        out = ring.submit(batch, pcfg, uniforms=u_dev, collect_debug=collect_debug_matches)
        if want_depth:
            depth = ring.submit_depth_maps(batch, pcfg, float(cfg.depth_min_certainty), **maps)
    return _PendingLaunch(out=out, batch=batch, n=n, collect_debug=collect_debug_matches, ply_records=ply_records, depth=depth,
                          ref_cams=ref_cams)


def _fused_normals(cfg) -> bool:
    """Depth fusion with the normal test (config.depth_fusion_max_normal_angle): the fused cloud has normals."""
    return (bool(getattr(cfg, "depth_fusion", False)) and int(getattr(cfg, "depth_normal_radius", 0)) > 0
            and float(getattr(cfg, "depth_fusion_max_normal_angle", 0.0)) > 0.0)


def _normal_radius(cfg) -> int:
    """Window radius of the launches' normal maps; 0 when no consumer (depth_dir files, the fusion's normal test) wants them."""
    r = int(getattr(cfg, "depth_normal_radius", 0))
    return r if (r > 0 and (getattr(cfg, "depth_dir", "") or _fused_normals(cfg))) else 0


def _launch_normal_maps(pending: "_PendingLaunch", tri_ctx: _TriangulationContext, ok: List[bool]) -> Dict[int, torch.Tensor]:
    """``output.estimate_depth_normals`` of the launch's maps, on the current stream: {view index: f32 [H, W, 3]} for every view
    whose sampling succeeded."""
    from ..engine import DepthViews
    from ..output import estimate_depth_normals
    cfg, dm = tri_ctx.config, pending.depth
    rs = [r for r in range(pending.n) if ok[r]]
    if not rs:
        return {}
    views = DepthViews(int(dm.depth.shape[1]), int(dm.depth.shape[2]), tri_ctx.w_match, tri_ctx.h_match, dm.depth.device)
    for r in rs:
        views.add(dm.depth[r], pending.ref_cams[r], xyz=dm.xyz[r])
    res = estimate_depth_normals(views, radius=int(cfg.depth_normal_radius), rel_tol=float(cfg.depth_normal_rel_tol))
    return {r: res.normals[i] for i, r in enumerate(rs)}


def depth_map_name(cameras, uid: int) -> str:
    """File name of reference view ``uid``'s depth map: the stem of its image path (its uid when it has none) + ``.npy``."""
    path = cameras.path_by.get(int(uid), "") if hasattr(cameras, "path_by") else ""
    stem = os.path.splitext(os.path.basename(path))[0] if path else ""
    return (stem or str(int(uid))) + ".npy"


def _write_depth_maps(pending: _PendingLaunch, tri_ctx: _TriangulationContext, ok: List[bool], ring,
                      depth_paths: Optional[Dict[int, str]], normal_maps: Optional[Dict[int, torch.Tensor]] = None) -> None:
    """The launch's depth maps, one file per view whose sampling succeeded (the views the cloud has too); with
    ``normal_maps`` also each view's normal map, f32 [H, W, 3], under the same name in ``normals/``."""
    from ..output import write_depth_map
    if ring is not None:
        ring.wait(pending.depth)
    maps = pending.depth.depth.cpu().numpy()              # only these maps travel to the host, one launch at a time
    out_dir = tri_ctx.config.depth_dir
    os.makedirs(out_dir, exist_ok=True)
    if normal_maps is not None:
        os.makedirs(os.path.join(out_dir, "normals"), exist_ok=True)
    for r in range(pending.n):
        if not ok[r]:
            continue
        uid = int(pending.batch.ref_uids[r])
        path = os.path.join(out_dir, depth_map_name(tri_ctx.cameras, uid))
        write_depth_map(path, maps[r])
        if normal_maps is not None:
            np.save(os.path.join(out_dir, "normals", depth_map_name(tri_ctx.cameras, uid)),
                    np.ascontiguousarray(normal_maps[r].cpu().numpy(), dtype=np.float32), allow_pickle=False)
        if depth_paths is not None:
            depth_paths[uid] = path


def collect_refs(pending: _PendingLaunch, errors: Optional[list] = None, ring=None, tri_ctx: Optional[_TriangulationContext] = None,
                 depth_paths: Optional[Dict[int, str]] = None, depth_kept: Optional[list] = None,
                 normals_kept: Optional[list] = None) -> List[Optional[_TriangulatedReference]]:
    """Second half: one synchronising read of the launch's results, split per view.  A launch with depth maps writes them
    under ``tri_ctx.config.depth_dir`` and records each file in ``depth_paths`` (reference camera uid -> path); with
    ``depth_kept`` it appends (uid, device map [H, W], reference camera, xyz, rgb, err maps or None) for every view whose
    sampling succeeded, and with ``normals_kept`` each such view's normal map [H, W, 3] (config.depth_normal_radius)."""
    out, batch = pending.out, pending.batch
    if ring is not None:
        ring.wait(out)                                 # the current stream (which does the read-back) follows the ring stream
    host = _download(out, pending.collect_debug, pending.ply_records)
    triangulate_refs.last_uniforms_used = host["uniforms_used"].copy()
    # the per-view results are slices of the launch's own host block (see _download): nothing is copied again
    results: List[Optional[_TriangulatedReference]] = []
    ok: List[bool] = []
    for r in range(pending.n):
        try:
            _raise_for_status(int(host["status"][r]))
            ok.append(True)
            results.append(_split_reference(out, host, r, batch.nbr_uids[r], pending.collect_debug))
        except Exception as exc:      # the reference's caller logs and skips (core/pipeline.py:874-879)
            if errors is not None:
                errors.append((r, exc))
            ok.append(False)
            results.append(None)
    if pending.depth is not None:
        if tri_ctx is None:
            raise ValueError("a launch with depth maps is collected with its tri_ctx")
        normal_maps = None
        if _normal_radius(tri_ctx.config):
            if ring is not None:
                ring.wait(pending.depth)           # computed on the current stream, which reads the maps
            normal_maps = _launch_normal_maps(pending, tri_ctx, ok)
        if getattr(tri_ctx.config, "depth_dir", ""):
            _write_depth_maps(pending, tri_ctx, ok, ring, depth_paths, normal_maps)
        if depth_kept is not None:
            if ring is not None:
                ring.wait(pending.depth)           # the maps are read later on the current stream
            for r in range(pending.n):
                if ok[r]:
                    dm = pending.depth
                    depth_kept.append((int(pending.batch.ref_uids[r]), dm.depth[r], pending.ref_cams[r],
                                       *(None if t is None else t[r] for t in (dm.xyz, dm.rgb, dm.err))))
                    if normals_kept is not None:
                        normals_kept.append(normal_maps[r])
    triangulate_refs.last_launches = out.launches
    return results


def triangulate_refs(matched_refs: Sequence[_MatchedReference], tri_ctx: _TriangulationContext,
                     collect_debug_matches: bool = False, *, rng_streams: Optional[Sequence[int]] = None,
                     uniforms: Optional[np.ndarray] = None,
                     weight_sums: Optional[Sequence[float]] = None,
                     errors: Optional[list] = None, ply_records: bool = False,
                     depth_paths: Optional[Dict[int, str]] = None,
                     depth_kept: Optional[list] = None, normals_kept: Optional[list] = None) -> List[Optional[_TriangulatedReference]]:
    """Batched ``_triangulate_ref``: every view of ``matched_refs`` in one launch sequence.

    RNG: ``uniforms`` (f64 [n, U], explicit parity stream per view) or Philox keyed by
    (config.seed, rng_streams[i]).  Views the reference would skip (None return / exception) come back as
    None; the exception a per-view call would raise is appended to ``errors`` as (index, exc).
    ``ply_records``: also return every view's PLY vertex records (built on the device, 15 bytes per point).
    ``config.depth_dir``: also write every view's depth map there (``depth_paths``: see ``collect_refs``);
    ``depth_kept`` / ``normals_kept``: keep the maps on the device (see ``collect_refs``).
    """
    if len(matched_refs) == 0:
        return []
    pending = submit_refs(matched_refs, tri_ctx, collect_debug_matches, rng_streams=rng_streams, uniforms=uniforms,
                          weight_sums=weight_sums, ply_records=ply_records)
    return collect_refs(pending, errors, tri_ctx=tri_ctx, depth_paths=depth_paths, depth_kept=depth_kept, normals_kept=normals_kept)


def _triangulate_ref(matched_ref: _MatchedReference, tri_ctx: _TriangulationContext,
                     collect_debug_matches: bool = False, *,
                     depth_paths: Optional[Dict[int, str]] = None,
                     depth_kept: Optional[list] = None, normals_kept: Optional[list] = None) -> Optional[_TriangulatedReference]:
    """Triangulate matches for a single reference view (reference core/pipeline.py:602-780).

    ``config.rng_mode``: "numpy" consumes the process-global MT19937 stream like the reference's ``np.random.choice``:
    the same uniforms, in the same order, and the same stream position afterwards.  The sampled INDICES are the
    reference's bit for bit only given the same float32 normaliser ``s``: the reference takes ``weights.sum()`` from a
    torch-CPU float32 reduction whose last bit depends on the thread count (SURVEY F5-ii), the kernels take the float64 sum
    rounded once.  When the two differ by an ulp, ``p = w / s`` and with it a handful of inverse-CDF hits move to a
    neighbouring pixel (tests/test_gpu_properties.py::test_drop_in_triangulate_ref_numpy_global_stream bounds it: kept
    points within 3 of the reference's, stream position identical); the parity tests pin ``s`` (``weight_sums=``) and are
    exact.  "philox" (default) uses the counter-based generator keyed by (config.seed, packed.ref_id): reproducible from
    run to run and across sharding, pinned value for value against the oracle
    (tests/test_gpu_parity.py::test_bench_batch_philox_mode_vs_oracle), but not the reference's ``np.random.seed`` stream.
    """
    cfg = tri_ctx.config
    mode = getattr(cfg, "rng_mode", RNG_PHILOX)
    errs: list = []
    if mode == RNG_NUMPY_GLOBAL and not cfg.no_filter:
        size = int(cfg.matches_per_ref * 0.85)
        n_uni = 2 * size + 64
        while True:
            U = _mt_stream_from_global(n_uni)
            kept_here: Optional[list] = [] if depth_kept is not None else None
            normals_here: Optional[list] = [] if normals_kept is not None else None
            res = triangulate_refs([matched_ref], tri_ctx, collect_debug_matches, uniforms=U[None, :], errors=errs,
                                   depth_paths=depth_paths, depth_kept=kept_here, normals_kept=normals_here)
            if errs and "exhausted" in str(errs[0][1]):
                errs.clear()
                n_uni *= 2
                continue
            if depth_kept is not None:
                depth_kept += kept_here
            if normals_kept is not None:
                normals_kept += normals_here
            break
        used = int(triangulate_refs.last_uniforms_used[0])
        if used > 0:
            np.random.random_sample(used)          # advance the global stream like np.random.choice did
    else:
        res = triangulate_refs([matched_ref], tri_ctx, collect_debug_matches,
                               rng_streams=[int(matched_ref.packed.ref_id)], errors=errs, depth_paths=depth_paths,
                               depth_kept=depth_kept, normals_kept=normals_kept)
    if errs:
        raise errs[0][1]
    return res[0]


def _collect_reference_matches(packed: _PackedReferenceBatch, matcher, config: DensePipelineConfig, pair_counter: int,
                               cancel_requested: Optional[Callable[[], bool]] = None
                               ) -> Tuple[Optional[_MatchedReference], int]:
    """Reference signature (core/pipeline.py:385-391).  ``matcher.match_grids_batch(imA, nn_images)`` yields one
    (warp_hw, cert_hw) pair per neighbour, as ``RomaMatcher`` does (core/matcher.py:141-196).

    Unlike the reference, nothing is post-processed or copied to the host here: the matcher's tensors are handed on
    as they are (``raw_certainty=True``) and the floor clamp / mask products of core/pipeline.py:405-430 happen inside
    the kernels that read them.  The ``.to("cpu")`` + ``cuda.synchronize()`` of :432-442 disappears."""
    imA, nn_images = packed.imA_np, list(packed.nn_arrays)
    try:                                   # the reference hands PIL images to the matcher (:392-393)
        from PIL import Image
        imA = Image.fromarray(np.ascontiguousarray(packed.imA_np))
        nn_images = [Image.fromarray(np.ascontiguousarray(a)) for a in packed.nn_arrays]
    except ImportError:
        pass
    results = matcher.match_grids_batch(imA, nn_images)
    if _is_cancelled(cancel_requested):
        raise PipelineCancelled("Cancelled")
    warps: List[torch.Tensor] = []
    certs: List[torch.Tensor] = []
    pair_index_by_nbr: Dict[int, int] = {}
    image_by_nbr: Dict[int, np.ndarray] = {}
    for (warp_hw, cert_hw), nbr_id, imB_np in zip(results, packed.nn_ids, packed.nn_arrays):
        warps.append(warp_hw.detach())
        certs.append(cert_hw.detach())
        pair_counter += 1
        pair_index_by_nbr[nbr_id] = pair_counter
        image_by_nbr[nbr_id] = imB_np
    if not certs:
        return None, pair_counter
    return _MatchedReference(packed=packed, warp_list_cpu=warps, cert_list_cpu=certs, pair_index_by_nbr=pair_index_by_nbr,
                             image_by_nbr=image_by_nbr, raw_certainty=True), pair_counter


def _build_filtered_match_preview(imA_np, imB_np, matches, cert_norm, ref_id: int, nbr_id: int, ref_label: str, nbr_label: str,
                                  pair_index: int, total_pairs: int, match_count: int,
                                  max_matches: int = _PREVIEW_MAX_MATCHES) -> Optional[MatchPreview]:
    """reference core/pipeline.py:551-599: at most ``max_matches`` of the kept matches, drawn with the pair's own seed."""
    if matches is None or cert_norm is None or matches.size == 0 or cert_norm.size == 0:
        return None
    matches = np.asarray(matches, dtype=np.float32)
    cert_norm = np.asarray(cert_norm, dtype=np.float32)
    total = int(match_count if match_count > 0 else matches.shape[0])
    if matches.shape[0] > max_matches > 0:
        from ..output import preview_seed
        sel = np.random.default_rng(preview_seed(ref_id, nbr_id)).choice(matches.shape[0], size=max_matches, replace=False)
        matches, cert_norm = matches[sel], cert_norm[sel]
    return MatchPreview(ref_id=ref_id, nbr_id=nbr_id, ref_label=ref_label, nbr_label=nbr_label, left_image=imA_np,
                        right_image=imB_np, matches=matches, cert_norm=cert_norm.astype(np.float32, copy=False),
                        match_count=total, pair_index=int(pair_index), total_pairs=int(total_pairs))


def _emit_debug_previews(matched_ref: _MatchedReference, tri_ref: _TriangulatedReference, debug_state, cameras: _CameraLookup,
                         total_pairs_est: int, pair_counter: int, cancel_requested: Optional[Callable[[], bool]]) -> None:
    """reference core/pipeline.py:458-505: one preview per neighbour of the view (every third pair when auto-stepping)."""
    if debug_state is None:
        return
    packed = matched_ref.packed
    total_pairs_val = total_pairs_est if total_pairs_est > 0 else max(pair_counter, 1)
    for nbr_id, matches in tri_ref.debug_matches_by_nbr.items():
        if _is_cancelled(cancel_requested):
            raise PipelineCancelled("Cancelled")
        imB_np = matched_ref.image_by_nbr.get(nbr_id)
        pair_idx = matched_ref.pair_index_by_nbr.get(nbr_id)
        cert_norm = tri_ref.debug_cert_by_nbr.get(nbr_id)
        if imB_np is None or pair_idx is None or cert_norm is None:
            continue
        auto = debug_state.is_auto_step() if hasattr(debug_state, "is_auto_step") else True
        if auto and _DEBUG_PREVIEW_INTERVAL > 0 and pair_idx % _DEBUG_PREVIEW_INTERVAL != 1:
            continue
        try:
            preview = _build_filtered_match_preview(packed.imA_np, imB_np, matches, cert_norm, packed.ref_id, nbr_id,
                                                    os.path.basename(packed.ref_path), os.path.basename(cameras.path_by.get(nbr_id, "")),
                                                    pair_idx, total_pairs_val, match_count=int(matches.shape[0]))
            if preview:
                debug_state.submit_preview(preview)
        except Exception:                                      # the reference logs and carries on (:503-504)
            pass


# ------------------------------------------------------------------------------------------------
MatchSource = Callable[[int], Optional[_MatchedReference]]


def _prepare_intermediate_ply_base(output_path: str, viz_interval: int,
                                   on_sequential_viz: Optional[Callable[[str], None]]) -> Optional[str]:
    """reference core/pipeline.py:296-306"""
    if not on_sequential_viz or viz_interval <= 0:
        return None
    output_dir = os.path.dirname(output_path)
    base_no_ext = os.path.splitext(os.path.basename(output_path))[0]
    os.makedirs(output_dir, exist_ok=True)
    return os.path.join(output_dir, f"{base_no_ext}_intermediate")


def _ply_records_host(xyz: np.ndarray, rgb: np.ndarray) -> np.ndarray:
    from . import writers as _w
    rec = np.empty(int(xyz.shape[0]), dtype=_w._PLY_VERTEX)
    rec["x"], rec["y"], rec["z"] = xyz[:, 0], xyz[:, 1], xyz[:, 2]
    u8 = _w.to_uint8_rgb(rgb)
    rec["r"], rec["g"], rec["b"] = u8[:, 0], u8[:, 1], u8[:, 2]
    return rec.view(np.uint8)


def _emit_intermediate_ply(path: str, n_points: int, parts: List[np.ndarray],
                           on_sequential_viz: Callable[[str], None]) -> None:
    """reference core/pipeline.py:523-530: same file bytes as write_ply(path, concat(xyz), to_uint8_rgb(concat(rgb)))."""
    from . import writers as _w
    try:
        with open(path, "wb") as f:
            f.write(_w.ply_header(n_points))
            for p in parts:
                p.tofile(f)
        on_sequential_viz(path)
    except Exception:                                          # the reference logs and carries on (:531-532)
        pass


def _is_cancelled(cancel_requested: Optional[Callable[[], bool]]) -> bool:
    if cancel_requested is None:
        return False
    try:
        return bool(cancel_requested())
    except Exception:
        return False


def run_dense_pipeline(
    camera_records: List[CameraRecord],
    refs_local: List[int],
    nn_table: np.ndarray,
    config: DensePipelineConfig,
    progress_callback: Optional[Callable[[float, str], None]] = None,
    on_sequential_viz: Optional[Callable[[str], None]] = None,
    debug_state=None,
    cancel_requested: Optional[Callable[[], bool]] = None,
    *,
    match_source: Optional[MatchSource] = None,
    w_match: Optional[int] = None,
    h_match: Optional[int] = None,
    sample_cap: float = 0.9,
) -> PipelineResult:
    """Reference signature (core/pipeline.py:783-792) + ``match_source``: a callable
    ``ref_local -> _MatchedReference | None`` standing in for pack loader + RoMa matcher (out of scope here;
    an integrator wraps ``RomaMatcher.match_grids_batch`` and may keep its outputs on the GPU).

    Views are processed ``config.refs_per_launch`` at a time (default 32; 0 = all in one launch): ``match_source`` is
    asked for one launch worth of views, the launch is enqueued on a ring of engines, and the oldest launch in flight is
    read back - so device memory holds the matcher outputs of at most ring-depth launches, ``cancel_requested`` is polled
    before every launch and ``progress_callback`` fires after every collected launch.
    ``debug_state`` (reference ``MatchDebugState``: ``is_enabled``, ``set_total_pairs``, ``is_auto_step``,
    ``submit_preview``, ``release_waiters``): when enabled, the launches collect the kept matches per neighbour and a
    ``MatchPreview`` per pair is submitted exactly as the reference does (core/pipeline.py:866-893)."""
    if match_source is None:
        raise RuntimeError("run_dense_pipeline needs a match_source: the RoMa matcher is not part of this package")
    from .config import ROMA_PRESETS
    from .selection import _estimate_total_pairs
    if w_match is None or h_match is None:
        h_lr, _ = ROMA_PRESETS[config.roma_setting]
        w_match = h_match = h_lr
    if getattr(config, "rng_mode", RNG_PHILOX) == RNG_NUMPY_GLOBAL:
        np.random.seed(config.seed)                                    # core/pipeline.py:793
    cameras = _build_camera_lookup(camera_records)
    total_pairs_est = 0
    if debug_state is not None and nn_table is not None:
        try:
            total_pairs_est = int(_estimate_total_pairs(refs_local, nn_table, cameras.img_ids, config.nns_per_ref))
        except Exception:
            total_pairs_est = 0
        debug_state.set_total_pairs(total_pairs_est)                   # core/pipeline.py:796-798
    tri_ctx = _TriangulationContext(cameras=cameras, config=config, matcher_sample_cap=sample_cap,
                                    w_match=int(w_match), h_match=int(h_match))
    t0 = time.time()
    step = int(getattr(config, "refs_per_launch", 32)) or max(1, len(refs_local))
    parts_xyz, parts_rgb, parts_err, parts_nv, parts_ref = [], [], [], [], []
    pairs = 0
    pair_counter = 0
    # live update (core/pipeline.py:296-306,508-532): every viz_interval views the reference re-concatenates and re-packs
    # all points so far; here every view's PLY records are packed once, on the device, and an emission is a bulk write
    viz_interval = int(getattr(config, "viz_interval", 0))
    ply_base = _prepare_intermediate_ply_base(config.output_path, viz_interval, on_sequential_viz)
    every_emission = bool(getattr(config, "viz_every_emission", False))
    ply_parts: List[np.ndarray] = []
    ply_points = 0
    total = len(refs_local)
    n_chunks = (total + step - 1) // step
    ring = get_ring() if (n_chunks > 1 and getattr(config, "rng_mode", RNG_PHILOX) != RNG_NUMPY_GLOBAL) else None
    in_flight: List[tuple] = []      # (views done when this launch is collected, launch, its matched references)
    depth_paths: Optional[Dict[int, str]] = {} if getattr(config, "depth_dir", "") else None
    fusion = bool(getattr(config, "depth_fusion", False))
    depth_kept: Optional[list] = [] if (getattr(config, "depth_consistency", False) or fusion) else None
    normals_kept: Optional[list] = [] if _fused_normals(config) else None      # beside depth_kept, entry for entry

    def consume(outs, done: int, matched_refs) -> None:
        nonlocal pairs, ply_points, pair_counter
        latest = None                 # (file name, points, parts) of the newest due emission of this launch
        for tri, mr in zip(outs, matched_refs):
            pair_counter = max([pair_counter] + list(mr.pair_index_by_nbr.values()))
            if tri is None:
                continue
            parts_xyz.append(tri.xyz)
            parts_rgb.append(tri.rgb)
            parts_err.append(tri.err)
            parts_ref.append(np.full((int(tri.xyz.shape[0]),), int(mr.packed.ref_id), np.int64))   # each point's reference view
            if tri.n_views is not None:
                parts_nv.append(tri.n_views)
            pairs += 1
            if tri.debug_matches_by_nbr and debug_state is not None:
                _emit_debug_previews(mr, tri, debug_state, cameras, total_pairs_est, pair_counter, cancel_requested)
            if ply_base is not None:
                rec = tri.ply_records
                if rec is None:                               # numpy-RNG mode goes through _triangulate_ref: pack on the host
                    rec = _ply_records_host(tri.xyz, tri.rgb)
                ply_parts.append(rec)
                ply_points += int(tri.xyz.shape[0])
                if pairs % viz_interval == 0:
                    if every_emission:
                        _emit_intermediate_ply(f"{ply_base}_{pairs}.ply", ply_points, ply_parts, on_sequential_viz)
                    else:
                        latest = (f"{ply_base}_{pairs}.ply", ply_points, len(ply_parts))
        if latest is not None:
            _emit_intermediate_ply(latest[0], latest[1], ply_parts[:latest[2]], on_sequential_viz)
        if progress_callback:
            progress_callback(10.0 + 80.0 * done / max(1, total), f"Matching {done}/{total} references")

    try:
        for lo in range(0, total, step):
            if _is_cancelled(cancel_requested):
                raise PipelineCancelled("Cancelled")
            chunk = refs_local[lo:lo + step]
            done = min(total, lo + step)
            matched = [(r, match_source(r)) for r in chunk]
            matched = [(r, m) for r, m in matched if m is not None]
            if not matched:
                continue
            mrs = [m for _, m in matched]
            collect_debug = debug_state is not None and bool(debug_state.is_enabled())      # core/pipeline.py:866
            if getattr(config, "rng_mode", RNG_PHILOX) == RNG_NUMPY_GLOBAL:
                outs = []
                for m in mrs:
                    try:
                        outs.append(_triangulate_ref(m, tri_ctx, collect_debug, depth_paths=depth_paths, depth_kept=depth_kept,
                                                     normals_kept=normals_kept))
                    except Exception:
                        outs.append(None)
                consume(outs, done, mrs)
            elif ring is None:
                consume(triangulate_refs(mrs, tri_ctx, collect_debug, rng_streams=[int(r) for r, _ in matched],
                                         ply_records=ply_base is not None, depth_paths=depth_paths, depth_kept=depth_kept,
                                         normals_kept=normals_kept),
                        done, mrs)
            else:
                # several launches in flight: the next chunk is uploaded and enqueued before the oldest one is read back
                in_flight.append((done, submit_refs(mrs, tri_ctx, collect_debug, rng_streams=[int(r) for r, _ in matched],
                                                    ply_records=ply_base is not None, ring=ring), mrs))
                if len(in_flight) >= ring.depth:
                    d, pend, pm = in_flight.pop(0)
                    consume(collect_refs(pend, ring=ring, tri_ctx=tri_ctx, depth_paths=depth_paths, depth_kept=depth_kept,
                                 normals_kept=normals_kept), d, pm)
        for d, pend, pm in in_flight:
            if _is_cancelled(cancel_requested):
                raise PipelineCancelled("Cancelled")
            consume(collect_refs(pend, ring=ring, tri_ctx=tri_ctx, depth_paths=depth_paths, depth_kept=depth_kept,
                                 normals_kept=normals_kept), d, pm)
    finally:
        if debug_state is not None and hasattr(debug_state, "release_waiters"):
            debug_state.release_waiters()                              # core/pipeline.py:547-548
    if _is_cancelled(cancel_requested):
        raise PipelineCancelled("Cancelled")
    if progress_callback:
        progress_callback(90.0, "Finalizing triangulation...")
    if depth_paths is not None:
        _write_depth_index(config, tri_ctx, depth_paths)
    if not parts_xyz:
        raise RuntimeError("No points triangulated. Try adjusting parameters.")
    xyz, rgb, err = np.concatenate(parts_xyz, axis=0), np.concatenate(parts_rgb, axis=0), np.concatenate(parts_err, axis=0)
    n_views = np.concatenate(parts_nv, axis=0) if getattr(config, "multiview", False) else None
    ref_uid = np.concatenate(parts_ref, axis=0)
    consistent = fused_views = fused_normals = None
    if fusion:
        # the fused maps replace the sampled cloud (its test includes depth_consistency's); the intermediate PLYs above stay
        # those of the sampled path
        if progress_callback:
            progress_callback(93.0, "Fusing depth maps...")
        if normals_kept is None:
            xyz, rgb, err, ref_uid, fused_views, consistent = _fuse_depth_maps(depth_kept, tri_ctx)
        else:                                  # with the normal test: one normal per fused point
            xyz, rgb, err, ref_uid, fused_views, consistent, fused_normals = _fuse_depth_maps(depth_kept, tri_ctx, normals=normals_kept)
        depth_kept = normals_kept = None
        n_views = None                         # the multiview counts belong to the sampled points
    elif depth_kept is not None:
        # visibility test against the other reference views' maps, before the outlier filter, normals and Gaussians; the
        # intermediate PLYs above stay unfiltered
        if progress_callback:
            progress_callback(93.0, "Checking depth consistency...")
        consistent, keep = _check_consistency(xyz, ref_uid, depth_kept, tri_ctx)
        depth_kept = None                      # the maps are not needed any more
        xyz, rgb, err, ref_uid = xyz[keep], rgb[keep], err[keep], ref_uid[keep]
        if n_views is not None:
            n_views = n_views[keep]
    k_out = int(getattr(config, "outlier_neighbors", 0))
    k_nrm = int(getattr(config, "normal_neighbors", 0))
    k_gs = int(getattr(config, "gaussian_neighbors", 0))
    normals = gaussians = nrm_dev = None
    if k_out > 0 or k_nrm > 0 or k_gs > 0:
        dev = torch.device("cuda", torch.cuda.current_device())
        xyz_dev = torch.from_numpy(np.ascontiguousarray(xyz, dtype=np.float32)).to(dev)
    if k_out > 0:
        # floaters: the whole cloud at once (neighbours cross views); the intermediate PLYs above stay unfiltered
        if progress_callback:
            progress_callback(95.0, "Removing outliers...")
        from ..output import remove_statistical_outliers
        # xyz stands in for rgb: only kept_idx is used, and it is applied to every per-point array on the host
        res = remove_statistical_outliers(xyz_dev, xyz_dev, nb_neighbors=k_out, std_ratio=float(config.outlier_std_ratio))
        keep = res.kept_idx.cpu().numpy()
        xyz, rgb, err, ref_uid = xyz[keep], rgb[keep], err[keep], ref_uid[keep]
        xyz_dev = res.xyz
        if n_views is not None:
            n_views = n_views[keep]
        if consistent is not None:
            consistent = consistent[keep]
        if fused_views is not None:
            fused_views = fused_views[keep]
        if fused_normals is not None:
            fused_normals = fused_normals[keep]
    if k_nrm > 0:
        # every point faces the camera it was triangulated from (its reference view, a contributing view in every mode)
        if progress_callback:
            progress_callback(97.0, "Estimating normals...")
        from ..output import estimate_normals
        uids, center_idx = np.unique(ref_uid, return_inverse=True)
        centers = np.stack([np.asarray(cameras.C_by[int(u)], np.float64).reshape(3) for u in uids]).astype(np.float32)
        nres = estimate_normals(xyz_dev, nb_neighbors=k_nrm, centers=torch.from_numpy(centers).to(dev),
                                center_idx=torch.from_numpy(center_idx.astype(np.int32)).to(dev))
        normals, nrm_dev = nres.normals.cpu().numpy(), nres.normals
    elif fused_normals is not None:
        # the fused normals (averaged over each point's members, facing its source camera) in place of a k-NN search
        normals = fused_normals
        if k_gs > 0:
            nrm_dev = torch.from_numpy(np.ascontiguousarray(normals)).to(dev)
    if k_gs > 0:
        # the final cloud, after the outlier filter; discs along the normals above when there are any
        if progress_callback:
            progress_callback(98.0, "Initialising Gaussians...")
        from ..output import init_gaussians
        rgb_dev = torch.from_numpy(np.ascontiguousarray(rgb, dtype=np.float32)).to(dev)
        g = init_gaussians(xyz_dev, rgb_dev, normals=nrm_dev, nb_neighbors=k_gs,
                           opacity=float(config.gaussian_opacity), flatten=float(config.gaussian_flatten))
        gaussians = {name: getattr(g, name).cpu().numpy() for name in ("sh_dc", "opacity", "scales", "rotations")}
    return PipelineResult(xyz=xyz, rgb=rgb, err=err, elapsed_seconds=time.time() - t0, pairs_processed=pairs, n_views=n_views,
                          normals=normals, gaussians=gaussians, depth_paths=depth_paths, consistent_views=consistent,
                          fused_views=fused_views)


def _fuse_depth_maps(depth_kept: list, tri_ctx: _TriangulationContext, normals: Optional[list] = None):
    """``output.fuse_depth_maps`` of the kept maps (``collect_refs``), views in collection order.  Returns host arrays
    (xyz, rgb, err, reference camera uid of each point's source view, n_views, n_consistent); with ``normals`` (each kept
    view's normal map, ``collect_refs``' ``normals_kept``) the fusion takes the normal test and the fused normals follow."""
    from ..engine import DepthViews
    from ..output import fuse_depth_maps
    cfg = tri_ctx.config
    m0 = depth_kept[0][1]
    views = DepthViews(int(m0.shape[0]), int(m0.shape[1]), tri_ctx.w_match, tri_ctx.h_match, m0.device)
    for v, (uid, depth, cam, xyz, rgb, err) in enumerate(depth_kept):
        views.add(depth, cam, xyz=xyz, rgb=rgb, err=err, normals=None if normals is None else normals[v])
    f = fuse_depth_maps(views, rel_tol=float(cfg.consistency_rel_tol), min_views=int(cfg.consistency_min_views),
                        max_violations=int(cfg.consistency_max_violations),
                        max_normal_angle=None if normals is None else float(cfg.depth_fusion_max_normal_angle))
    uids = np.array([e[0] for e in depth_kept], np.int64)
    src_view = (f.source // (views.H * views.W)).cpu().numpy()
    out = (f.xyz.cpu().numpy(), f.rgb.cpu().numpy(), f.err.cpu().numpy(), uids[src_view], f.n_views.cpu().numpy(),
           f.n_consistent.cpu().numpy())
    return out if normals is None else out + (f.normals.cpu().numpy(),)


def _check_consistency(xyz: np.ndarray, ref_uid: np.ndarray, depth_kept: list, tri_ctx: _TriangulationContext):
    """``output.check_depth_consistency`` of the cloud against the kept maps (``collect_refs``), each point owned by the map of
    its reference view.  Returns (n_consistent of the kept points, kept indices), host arrays."""
    from ..engine import DepthViews
    from ..output import check_depth_consistency
    cfg = tri_ctx.config
    m0 = depth_kept[0][1]
    views = DepthViews(int(m0.shape[0]), int(m0.shape[1]), tri_ctx.w_match, tri_ctx.h_match, m0.device)
    index: Dict[int, int] = {}
    for uid, depth, cam, *_ in depth_kept:
        index[uid] = views.add(depth, cam)
    uids, inv = np.unique(ref_uid, return_inverse=True)
    owner = np.array([index.get(int(u), -1) for u in uids], dtype=np.int32)[inv.reshape(-1)]
    xyz_dev = torch.from_numpy(np.ascontiguousarray(xyz, dtype=np.float32)).to(m0.device)
    res = check_depth_consistency(xyz_dev, views, owner=torch.from_numpy(owner), rel_tol=float(cfg.consistency_rel_tol),
                                  min_views=int(cfg.consistency_min_views), max_violations=int(cfg.consistency_max_violations))
    keep = res.kept_idx.cpu().numpy()
    return res.n_consistent.cpu().numpy()[keep], keep


def _write_depth_index(config: DensePipelineConfig, tri_ctx: _TriangulationContext, depth_paths: Dict[int, str]) -> None:
    """``<depth_dir>/depth_maps.json``: what a reader needs to place each map (see output.write_depth_map)."""
    os.makedirs(config.depth_dir, exist_ok=True)
    maps = []
    for uid, path in depth_paths.items():
        H, W = np.load(path, mmap_mode="r").shape
        width, height = tri_ctx.cameras.size_by[uid]
        entry = dict(file=os.path.basename(path), camera_uid=int(uid), H=int(H), W=int(W), w_match=int(tri_ctx.w_match),
                     h_match=int(tri_ctx.h_match), width=int(width), height=int(height))
        if _normal_radius(config):
            entry["normals_file"] = "normals/" + os.path.basename(path)         # f32 [H, W, 3], NaN = no normal
        maps.append(entry)
    index = dict(min_certainty=float(config.depth_min_certainty), nan="no depth", maps=maps)
    with open(os.path.join(config.depth_dir, "depth_maps.json"), "w") as f:
        json.dump(index, f, indent=1)
