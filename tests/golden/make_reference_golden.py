"""Stored vectors for the tests that compare with the unmodified reference plugin (tests/test_oracle_vs_reference.py,
tests/test_host_logic.py, tests/test_oracle_prologue.py), so that those comparisons also run where the reference is not
installed: tests/golden/reference/oracle_vs_reference.npz.

Where the reference is installed, those tests compare the oracle (and the host code) with it bit for bit on exactly these
seeded inputs; they did so up to commit 49486be. The values here were recorded from the oracle and the host code at that
state of the project, so they are the reference's. Large outputs are kept as a fixed seeded sample of rows plus float64
column sums, which keeps the file small.

    python tests/golden/make_reference_golden.py
"""
from __future__ import annotations

import dataclasses
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from lichtfeld_densification_plugin_b200 import synth  # noqa: E402
from lichtfeld_densification_plugin_b200.core.config import DensePipelineConfig  # noqa: E402
from lichtfeld_densification_plugin_b200.core.selection import _estimate_total_pairs  # noqa: E402
from oracle import densify_oracle as O  # noqa: E402

PATH = os.path.join(HERE, "reference", "oracle_vs_reference.npz")
N_REFERENCE_FIELDS = 18          # core/config.py: the block of fields the reference's DensePipelineConfig has
SAMPLE_ROWS = 64                 # arrays longer than this are stored as a seeded sample of rows + column sums


def sample_rows(n: int) -> np.ndarray:
    """The rows of an n-row output that are stored (the same rule in the tests)."""
    if n <= SAMPLE_ROWS:
        return np.arange(n)
    return np.sort(np.random.RandomState(n).choice(n, SAMPLE_ROWS, replace=False))


def column_stats(a: np.ndarray) -> np.ndarray:
    """[row count, float64 column sums, float64 column sums of |a| (NaN skipped)] of a float array; [row count] otherwise."""
    head = [np.float64(a.shape[0])]
    if a.dtype.kind != "f":
        return np.asarray(head)
    a64 = a.astype(np.float64)
    return np.concatenate([head, np.ravel(a64.sum(axis=0)), np.ravel(np.nansum(np.abs(a64), axis=0))])


def put(out: dict, key: str, a) -> None:
    a = np.asarray(a)
    out[f"{key}.rows"] = a[sample_rows(a.shape[0])]
    out[f"{key}.stats"] = column_stats(a)


def triangulate_cases(out: dict) -> None:
    from tests.helpers import oracle_cam
    from tests.test_oracle_vs_reference import TRIANGULATE_CASES
    for fam, no_filter, nn in TRIANGULATE_CASES:
        scene = synth.make_scene(10, "turbo", ref_fraction=0.2, nn=nn)
        scene.H = scene.W = 128
        scene.h_match = scene.w_match = 96
        cams = scene.cameras
        for rp in range(scene.n_refs):
            inp = synth.synth_ref_inputs(scene, rp, cert_family=fam, seed=3)
            nb = inp["nbr_indices"]
            ocfg = O.OracleConfig(matches_per_ref=5000, no_filter=no_filter, w_match=scene.w_match, h_match=scene.h_match)
            got = O.triangulate_ref([inp["cert"][k] for k in range(len(nb))], [inp["warp"][k] for k in range(len(nb))],
                                    inp["image"].numpy(), oracle_cam(cams[inp["ref_index"]]), [oracle_cam(cams[j]) for j in nb],
                                    ocfg, rng=np.random.RandomState(40 + rp), collect_debug=True)
            key = f"tri/{fam}/{int(no_filter)}/{nn}/{rp}"
            for name in ("xyz", "rgb", "err"):
                put(out, f"{key}/{name}", getattr(got, name))
            out[f"{key}/dbg_uids"] = np.asarray(list(got.debug_matches_by_nbr.keys()), dtype=np.int64)
            for uid in got.debug_matches_by_nbr:
                put(out, f"{key}/dbg_matches/{uid}", got.debug_matches_by_nbr[uid])
                put(out, f"{key}/dbg_cert/{uid}", got.debug_cert_by_nbr[uid])


def sampler_and_geometry(out: dict) -> None:
    rs = np.random.RandomState(0)
    cert = torch.from_numpy(rs.random_sample((90, 120)).astype(np.float32))
    put(out, "fn/select_samples", O.select_samples(cert, 2000, rng=np.random.RandomState(5)))
    a, b = synth.make_orbit_cameras(5)[:2]
    F = O.fundamental_matrix(a.K, a.R, a.t, b.K, b.R, b.t)
    out["fn/F"] = F
    uv1 = (rs.random_sample((500, 2)) * 800).astype(np.float32)
    uv2 = (uv1 + rs.standard_normal((500, 2)) * 5).astype(np.float32)
    X = O.dlt_points(a.P, b.P, uv1, uv2)
    put(out, "fn/sampson", O.sampson_distance(F, uv1, uv2))
    put(out, "fn/dlt", X)
    put(out, "fn/dlt1", O.dlt_points(a.P, b.P, uv1[:1], uv2[:1]))
    put(out, "fn/reproj", O.reprojection_error(a.P, X, uv1))
    put(out, "fn/cheirality", O.in_front(b.P, X))
    put(out, "fn/parallax", O.parallax_ok(a.C, b.C, X, 0.5))


def random_configurations(out: dict) -> None:
    from tests import gpu_harness as G
    from tests.golden.make_golden import build_scene
    from tests.test_oracle_vs_reference import random_configuration
    for seed in range(12):
        c = random_configuration(seed)
        scene = build_scene(c)
        inp = synth.synth_ref_inputs(scene, 0, cert_family=c["fam"], seed=c["seed"])
        np.random.seed(c["seed"])
        key = f"rand/{seed}"
        try:
            got, err = G.run_oracle_ref(scene, inp, c), ""
        except Exception as exc:
            got, err = None, f"{type(exc).__name__}: {exc}"
        out[f"{key}/error"] = np.str_(err)
        if got is not None:
            for name in ("xyz", "rgb", "err"):
                put(out, f"{key}/{name}", getattr(got, name))


def host_logic(out: dict) -> None:
    fields = dataclasses.fields(DensePipelineConfig)[:N_REFERENCE_FIELDS]
    out["config/fields"] = np.str_(json.dumps([[f.name, None if f.default is dataclasses.MISSING else f.default] for f in fields]))
    rs = np.random.RandomState(1)
    nn = rs.randint(0, 20, size=(20, 5))
    ids = [int(v) for v in rs.randint(0, 12, size=20)]
    out["pairs/estimate"] = np.asarray([_estimate_total_pairs([0, 3, 7, 19], nn, ids, k) for k in (1, 3, 5)], dtype=np.int64)


def collect_reference_matches(out: dict) -> None:
    from tests.test_oracle_prologue import collect_case
    raw, warp, mA, mBs = collect_case()
    for k in range(raw.shape[0]):
        put(out, f"collect/cert/{k}", O.certainty_prologue(raw[k], warp[k], mA, mBs[k], 0.35).ravel())


def main() -> None:
    torch.set_num_threads(1)
    out = {"meta": np.str_(json.dumps({"numpy": np.__version__, "torch": torch.__version__, "sample_rows": SAMPLE_ROWS}))}
    triangulate_cases(out)
    sampler_and_geometry(out)
    random_configurations(out)
    host_logic(out)
    collect_reference_matches(out)
    os.makedirs(os.path.dirname(PATH), exist_ok=True)
    np.savez_compressed(PATH, **out)
    print(f"{PATH}: {len(out)} arrays, {os.path.getsize(PATH) / 1024:.0f} KiB")


if __name__ == "__main__":
    main()
