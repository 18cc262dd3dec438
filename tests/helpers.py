"""Shared test helpers: golden-case loading and oracle plumbing (test infrastructure)."""
from __future__ import annotations

import glob
import hashlib
import json
import os

import numpy as np
import torch

from lichtfeld_densification_plugin_b200 import synth
from oracle import densify_oracle as O

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GOLDEN_CASES = sorted(os.path.splitext(os.path.basename(p))[0]
                      for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz")) if not p.endswith(("writers.npz", "output_reducers.npz", "selection.npz")))


def golden_scene(c) -> synth.SynthScene:
    """Same construction as tests/golden/make_golden.py:build_scene."""
    cams = synth.make_orbit_cameras(9)
    centres = torch.from_numpy(np.stack([cam.C for cam in cams]))
    d = torch.cdist(centres, centres)
    d.fill_diagonal_(float("inf"))
    nn_table = torch.topk(d, c["nn"], largest=False, dim=1).indices.numpy()
    return synth.SynthScene(cameras=cams, refs_local=[4], nn_table=nn_table, H=c["H"], W=c["W"],
                            h_match=c["hm"], w_match=c["wm"], nn=c["nn"])


def load_golden(name: str):
    z = np.load(os.path.join(GOLDEN_DIR, f"{name}.npz"), allow_pickle=False)
    c = json.loads(str(z["case"]))
    scene = golden_scene(c)
    if "cert" in z.files:
        inp = {"cert": torch.from_numpy(z["cert"]), "warp": torch.from_numpy(z["warp"]),
               "image": torch.from_numpy(z["image"])}
    else:
        inp = synth.synth_ref_inputs(scene, 0, cert_family=c["fam"], seed=c["seed"])
        h = hashlib.sha256()
        for k in ("cert", "warp", "image"):
            h.update(np.ascontiguousarray(inp[k].numpy()).tobytes())
        if h.hexdigest() != str(z["input_sha256"]):
            raise RuntimeError(f"{name}: regenerated synthetic inputs differ from the ones the golden was made on "
                               "(torch RNG stream changed?)")
    inp["ref_index"] = int(z["ref_index"])
    inp["nbr_indices"] = [int(x) for x in z["nbr_indices"]]
    return c, scene, inp, z


class ReferenceGolden:
    """tests/golden/reference/oracle_vs_reference.npz (tests/golden/make_reference_golden.py): what the tests that compare
    with the unmodified reference compare against where it is not installed."""

    def __init__(self, path: str) -> None:
        self.z = np.load(path, allow_pickle=False)

    def check(self, key: str, got, rtol: float = 0.0, atol: float = 0.0) -> None:
        """Row count, the stored sample of rows and the column sums of ``got`` against the record ``key``; floats within
        rtol / atol per element (LAPACK / BLAS may differ in the last bits between CPUs), everything else exactly."""
        from tests.golden.make_reference_golden import column_stats, sample_rows
        got = np.asarray(got)
        stats = self.z[f"{key}.stats"]
        n = int(stats[0])
        assert got.shape[0] == n, (key, got.shape, n)
        rows, want = got[sample_rows(n)], self.z[f"{key}.rows"]
        assert rows.dtype == want.dtype and rows.shape == want.shape, (key, rows.dtype, rows.shape, want.dtype, want.shape)
        if want.dtype.kind != "f":
            assert np.array_equal(rows, want), key
            return
        np.testing.assert_allclose(rows, want, rtol=rtol, atol=atol, equal_nan=True, err_msg=key)
        mine = column_stats(got)
        c = (len(stats) - 1) // 2
        s, w = mine[1:1 + c], stats[1:1 + c]
        tol = n * atol + rtol * stats[1 + c:]
        assert np.array_equal(np.isnan(s), np.isnan(w)) and np.all(np.nan_to_num(np.abs(s - w)) <= tol), (key, s, w)


def load_reference_golden() -> ReferenceGolden:
    return ReferenceGolden(os.path.join(GOLDEN_DIR, "reference", "oracle_vs_reference.npz"))


def oracle_cam(c) -> O.OracleCamera:
    return O.OracleCamera(c.uid, c.width, c.height, c.K, c.R, c.t, c.P, c.C)


def oracle_cfg(c) -> O.OracleConfig:
    return O.OracleConfig(matches_per_ref=c["M"], no_filter=c["no_filter"], sampson_thresh=c.get("sampson", 5.0),
                          min_parallax_deg=c.get("parallax", 0.5), w_match=c["wm"], h_match=c["hm"])


def run_oracle(c, scene, inp, **kw):
    cams = scene.cameras
    nn = len(inp["nbr_indices"])
    return O.triangulate_ref([inp["cert"][k] for k in range(nn)], [inp["warp"][k] for k in range(nn)],
                             inp["image"].numpy(), oracle_cam(cams[inp["ref_index"]]),
                             [oracle_cam(cams[j]) for j in inp["nbr_indices"]], oracle_cfg(c), **kw)
