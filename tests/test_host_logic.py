"""CPU: host-side mirrors of the reference's configuration and seeds (no device work)."""
import dataclasses
import json
import types

import numpy as np
import pytest

from lichtfeld_densification_plugin_b200.core.config import DensePipelineConfig, ROMA_PRESETS
from oracle import ref_import


def reference_config_fields():
    """(name, default or None) of the reference's DensePipelineConfig: live where the reference is installed, otherwise
    the stored record (tests/golden/make_reference_golden.py)."""
    if ref_import.reference_available():
        ref = ref_import.import_reference(full_pipeline=False)
        return [(f.name, None if f.default is dataclasses.MISSING else f.default)
                for f in dataclasses.fields(ref.config.DensePipelineConfig)]
    from tests.helpers import load_reference_golden
    return [tuple(f) for f in json.loads(str(load_reference_golden().z["config/fields"]))]


def test_config_is_a_field_for_field_superset_of_the_reference():
    ref_fields = reference_config_fields()
    ours = {f.name: f for f in dataclasses.fields(DensePipelineConfig)}
    names = [f.name for f in dataclasses.fields(DensePipelineConfig)]
    assert names[:len(ref_fields)] == [name for name, _ in ref_fields]             # same names, same order
    for name, default in ref_fields:
        if default is not None:
            assert ours[name].default == default, name                             # same defaults
    ref_cfg = types.SimpleNamespace(**{name: default for name, default in ref_fields})
    ref_cfg.output_path, ref_cfg.matches_per_ref, ref_cfg.no_filter = "a.ply", 123, True
    cfg = DensePipelineConfig.from_reference(ref_cfg)
    assert cfg.matches_per_ref == 123 and cfg.no_filter and cfg.rng_mode == "philox"
    with pytest.raises(ValueError):
        DensePipelineConfig(output_path="x", rng_mode="nope").validate()


def test_path_config_takes_the_pipeline_scalars():
    from lichtfeld_densification_plugin_b200.engine import PathConfig
    cfg = DensePipelineConfig(output_path="x", matches_per_ref=777, reproj_thresh=1.5, sampson_thresh=0.0, min_parallax_deg=0.0, seed=9)
    p = PathConfig.from_pipeline_config(cfg, sample_cap=0.8)
    assert (p.matches_per_ref, p.reproj_thresh, p.sampson_thresh, p.min_parallax_deg, p.seed, p.sample_cap) == (777, 1.5, 0.0, 0.0, 9, 0.8)
    assert p.border == 2 and p.tiles == 24 and p.certainty_floor is None           # core/sampling.py:8 defaults, core/pipeline.py:647
    assert ROMA_PRESETS["precise"] == (800, 1280) and ROMA_PRESETS["fast"] == (512, 512)


def test_preview_seed_formula():
    """core/pipeline.py:574-575: ids are masked to 32 bits before and after the mix."""
    from lichtfeld_densification_plugin_b200.output import preview_seed
    rs = np.random.RandomState(0)
    for _ in range(200):
        a, b = int(rs.randint(0, 2 ** 62)), int(rs.randint(0, 2 ** 62))
        want = (((a & 0xFFFFFFFF) * 73856093) ^ ((b & 0xFFFFFFFF) * 19349663)) & 0xFFFFFFFF
        assert preview_seed(a, b) == want
    assert preview_seed(5, 9) == ((5 * 73856093) ^ (9 * 19349663)) & 0xFFFFFFFF


def test_estimate_total_pairs_matches_reference():
    from lichtfeld_densification_plugin_b200.core.selection import _estimate_total_pairs
    rs = np.random.RandomState(1)
    nn = rs.randint(0, 20, size=(20, 5))
    ids = [int(v) for v in rs.randint(0, 12, size=20)]                                # duplicate image ids: self-pairs are skipped
    refs = [0, 3, 7, 19]
    if ref_import.reference_available():
        ref = ref_import.import_reference(full_pipeline=True)
        want = [ref.pipeline._estimate_total_pairs(refs, nn, ids, k) for k in (1, 3, 5)]
    else:
        from tests.helpers import load_reference_golden
        want = [int(v) for v in load_reference_golden().z["pairs/estimate"]]
    assert [_estimate_total_pairs(refs, nn, ids, k) for k in (1, 3, 5)] == want


def test_packed_cloud_layout_is_one_allocation():
    """output.PackedCloud: header (int64 count) | xyz | rgb | err alias ONE buffer, every block 16-byte aligned, so that a
    rank's cloud goes into a single collective / is read by a peer as one mapping (distributed.PeerClouds)."""
    import torch
    from lichtfeld_densification_plugin_b200.output import PackedCloud
    c = PackedCloud(10, "cpu")
    assert c.capacity == 12 and c.packed.numel() == PackedCloud.nbytes(10) == 16 + 28 * 12
    c.xyz.fill_(1.0); c.rgb.fill_(2.0); c.err.fill_(3.0); c.count.fill_(7)
    raw = c.packed.numpy()
    assert int(raw[:8].view("<i8")[0]) == 7
    f = raw[16:].view("<f4")
    assert (f[:36] == 1.0).all() and (f[36:72] == 2.0).all() and (f[72:84] == 3.0).all()
    again = PackedCloud(10, "cpu", storage=c.packed)
    assert again.total_points() == 7 and torch.equal(again.err, c.err)
    for cap in (1, 2, 3, 5, 4097):
        assert PackedCloud.nbytes(cap) % 16 == 0
