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
        if self.rng_mode not in (RNG_PHILOX, RNG_NUMPY_GLOBAL, RNG_EXPLICIT):
            raise ValueError(f"unknown rng_mode {self.rng_mode!r}")
        return self

    @classmethod
    def from_reference(cls, cfg: Any, **overrides) -> "DensePipelineConfig":
        """Adopt a reference ``DensePipelineConfig`` (or any object with the same attributes)."""
        names = [f.name for f in dataclasses.fields(cls)]
        kw = {n: getattr(cfg, n) for n in names if hasattr(cfg, n)}
        kw.update(overrides)
        return cls(**kw).validate()
