"""Pipeline configuration for the B200 densification path.

Field-for-field superset of the reference's ``DensePipelineConfig`` (reference core/config.py:7-26)
so that a config object built for the reference drives this path unchanged; the extra fields at
the bottom are opt-in and default to reference behaviour.
"""
from __future__ import annotations

import dataclasses
from dataclasses import dataclass
from typing import Any

# RoMa preset -> (H_lr=W_lr match resolution, H=W map resolution).  The maps are produced at the
# high-resolution stage when a preset has one (SURVEY F3; reference RoMaV2/src/romav2/romav2.py:118-160,
# plugin override for "high" at core/matcher.py:82-87).
ROMA_PRESETS = {
    "turbo": (320, 320),
    "fast": (512, 512),
    "base": (640, 640),
    "high": (640, 960),
    "precise": (800, 1280),
}

# RNG modes of the sampler.
RNG_PHILOX = "philox"            # production: counter-based Philox4x32-10 keyed by (seed, ref id)
RNG_NUMPY_GLOBAL = "numpy"       # drop-in: consume the process-global MT19937 stream like np.random.choice
RNG_EXPLICIT = "explicit"        # parity: caller supplies the f64 uniform stream


@dataclass
class DensePipelineConfig:
    # --- reference fields (same names, order, defaults) ---
    output_path: str
    roma_setting: str = "fast"
    roi_only_selected: bool = False
    num_refs: float = 0.8
    nns_per_ref: int = 3
    matches_per_ref: int = 10000
    certainty_thresh: float = 0.20
    reproj_thresh: float = 0.8
    sampson_thresh: float = 5.0
    min_parallax_deg: float = 0.5
    max_points: int = 0
    no_filter: bool = False
    use_masks: bool = True
    voxel_size: float = 0.0
    seed: int = 0
    viz_interval: int = 3
    prefetch_packages: int = 8
    pack_workers: int = 4
    # --- B200 path, opt-in ---
    rng_mode: str = RNG_PHILOX
    refs_per_launch: int = 32        # reference views per launch sequence (launches are kept in flight on a ring of engines, so
                                     # memory, cancellation latency and progress granularity are bounded by this); 0 = all in one launch
    viz_every_emission: bool = False # live update: True writes every intermediate PLY the reference would (one per viz_interval
                                     # views, each a rewrite of all points so far); False only the latest one per collected launch
    multiview: bool = False          # re-triangulate every kept point from all of its confident, consistent neighbours (the
                                     # reference uses the best neighbour alone); which points are kept does not change
    multiview_min_certainty: float = 0.5   # multiview: certainty a neighbour's match needs at the pixel to join
    outlier_neighbors: int = 0       # > 0: drop statistical outliers (floaters) from the final cloud, Open3D's
                                     # remove_statistical_outlier(nb_neighbors = this, std_ratio); 0 = off
    outlier_std_ratio: float = 2.0
    normal_neighbors: int = 0        # > 0: PipelineResult.normals, PCA over this many nearest points, each normal facing
                                     # the camera that triangulated its point; 0 = off
    gaussian_neighbors: int = 0      # > 0: PipelineResult.gaussians, 3DGS's initial splats (create_from_pcd), scales from
                                     # this many nearest other points (3DGS: 3); 0 = off
    gaussian_opacity: float = 0.1    # initial opacity of every splat (3DGS: 0.1)
    gaussian_flatten: float = 1.0    # < 1: splats become discs along the normals (needs normal_neighbors); 1 = isotropic
    depth_dir: str = ""              # non-empty: one float32 depth map <depth_dir>/<image stem>.npy per reference view (every
                                     # pixel whose best certainty is >= depth_min_certainty, triangulated and filtered like a
                                     # sample) plus depth_maps.json; "" = off
    depth_min_certainty: float = 0.5 # depth maps: certainty a pixel's best match needs to be evaluated, in (0, 1]
    depth_consistency: bool = False  # keep a point only where the other reference views' depth maps agree with it (MVS
                                     # fusion's visibility test, include/ldp_b200.h: ldp_depth_consistency); the maps of every
                                     # view stay on the device until the end: R * H * W * 4 bytes (46 views at 512^2: 48 MB,
                                     # 250 views at 640^2: 410 MB)
    consistency_rel_tol: float = 0.01    # relative depth difference that still agrees (COLMAP fusion's default), in (0, 1)
    consistency_min_views: int = 1   # other views that must agree with a point
    consistency_max_violations: int = 0  # other views that may look through a point (see it in front of their surface)
    depth_fusion: bool = False       # replace the sampled cloud by the fused depth maps of every reference view (MVS fusion,
                                     # include/ldp_b200.h: ldp_fuse_depth_maps): each surface point once, averaged over the
                                     # views that agree with it; the rule takes the three consistency_* values above (and
                                     # includes depth_consistency's test).  The depth, xyz, rgb and err maps of every view
                                     # stay on the device until the end: about 32 bytes per pixel (46 views at 512^2: 386 MB,
                                     # 250 views at 640^2: 3.3 GB)
    depth_normal_radius: int = 0     # 1..3: oriented normal maps of the reference views, PCA over each pixel's
                                     # (2r + 1)^2 map window (include/ldp_b200.h: ldp_depth_normals), written to
                                     # <depth_dir>/normals/ and used by depth_fusion; needs depth_dir or depth_fusion.  With
                                     # depth_fusion the maps stay on the device beside the others: 12 bytes more per pixel
                                     # (46 views at 512^2: 145 MB, 250 views at 640^2: 1.2 GB).  0 = off
    depth_normal_rel_tol: float = 0.05   # normal maps: relative depth difference of a window pixel that still counts as the
                                     # same surface, in (0, 1); a slanted surface changes depth across the window by more
                                     # than consistency_rel_tol does
    depth_fusion_max_normal_angle: float = 0.0   # (0, 90) degrees: depth_fusion also requires agreeing normals (COLMAP
                                     # fusion's test; its default is 10) and PipelineResult.normals become the fused normals
                                     # unless normal_neighbors is set; needs depth_fusion and depth_normal_radius.  0 = off

    def validate(self) -> "DensePipelineConfig":
        if self.matches_per_ref < 0:
            raise ValueError("matches_per_ref must be >= 0")
        if self.multiview and self.no_filter:
            raise ValueError("multiview needs the filters: it cannot be combined with no_filter")
        if not 0.0 < float(self.multiview_min_certainty) <= 1.0:
            raise ValueError("multiview_min_certainty must lie in (0, 1]")
        if not 0 <= int(self.outlier_neighbors) <= 64:
            raise ValueError("outlier_neighbors must lie in [0, 64] (0 = off)")
        if not float(self.outlier_std_ratio) > 0.0:
            raise ValueError("outlier_std_ratio must be positive")
        if not (int(self.normal_neighbors) == 0 or 3 <= int(self.normal_neighbors) <= 64):
            raise ValueError("normal_neighbors must be 0 (off) or lie in [3, 64]")
        if not 0 <= int(self.gaussian_neighbors) <= 63:
            raise ValueError("gaussian_neighbors must lie in [0, 63] (0 = off)")
        if not 0.0 < float(self.gaussian_opacity) < 1.0:
            raise ValueError("gaussian_opacity must lie in (0, 1)")
        if not 0.0 < float(self.gaussian_flatten) <= 1.0:
            raise ValueError("gaussian_flatten must lie in (0, 1]")
        if float(self.gaussian_flatten) < 1.0 and int(self.normal_neighbors) == 0 and not self.fused_normals():
            raise ValueError("gaussian_flatten < 1 needs normal_neighbors (or depth_fusion_max_normal_angle)")
        if not isinstance(self.depth_dir, str):
            raise ValueError("depth_dir must be a string (\"\" = off)")
        if not 0.0 < float(self.depth_min_certainty) <= 1.0:
            raise ValueError("depth_min_certainty must lie in (0, 1]")
        if not 0.0 < float(self.consistency_rel_tol) < 1.0:
            raise ValueError("consistency_rel_tol must lie in (0, 1)")
        if int(self.consistency_min_views) < 0:
            raise ValueError("consistency_min_views must be >= 0")
        if int(self.consistency_max_violations) < 0:
            raise ValueError("consistency_max_violations must be >= 0")
        if not 0 <= int(self.depth_normal_radius) <= 3:
            raise ValueError("depth_normal_radius must lie in [0, 3] (0 = off)")
        if int(self.depth_normal_radius) > 0 and not (self.depth_dir or self.depth_fusion):
            raise ValueError("depth_normal_radius needs depth_dir or depth_fusion")
        if not 0.0 < float(self.depth_normal_rel_tol) < 1.0:
            raise ValueError("depth_normal_rel_tol must lie in (0, 1)")
        if not 0.0 <= float(self.depth_fusion_max_normal_angle) < 90.0:
            raise ValueError("depth_fusion_max_normal_angle must lie in [0, 90) degrees (0 = off)")
        if float(self.depth_fusion_max_normal_angle) > 0.0 and not (self.depth_fusion and int(self.depth_normal_radius) > 0):
            raise ValueError("depth_fusion_max_normal_angle needs depth_fusion and depth_normal_radius")
        if self.rng_mode not in (RNG_PHILOX, RNG_NUMPY_GLOBAL, RNG_EXPLICIT):
            raise ValueError(f"unknown rng_mode {self.rng_mode!r}")
        return self

    def fused_normals(self) -> bool:
        """Whether depth fusion runs with the normal test and so yields a normal per fused point."""
        return bool(self.depth_fusion) and int(self.depth_normal_radius) > 0 and float(self.depth_fusion_max_normal_angle) > 0.0

    @classmethod
    def from_reference(cls, cfg: Any, **overrides) -> "DensePipelineConfig":
        """Adopt a reference ``DensePipelineConfig`` (or any object with the same attributes)."""
        names = [f.name for f in dataclasses.fields(cls)]
        kw = {n: getattr(cfg, n) for n in names if hasattr(cfg, n)}
        kw.update(overrides)
        return cls(**kw).validate()
