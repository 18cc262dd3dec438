"""CPU: the oracle's certainty post-processing (SURVEY 8f row 1, reference core/pipeline.py:405-430) against the golden
vectors frozen from the live reference, and its explicit index arithmetic against the torch calls the reference makes."""
import glob
import json
import os

import numpy as np
import pytest
import torch

from oracle import densify_oracle as O
from oracle import ref_import

PRO_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "prologue")
PRO_CASES = sorted(os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(PRO_DIR, "*.npz")))


def load_prologue_golden(name):
    z = np.load(os.path.join(PRO_DIR, f"{name}.npz"), allow_pickle=False)
    c = json.loads(str(z["case"]))
    mA = z["maskA"] if int(z["has_maskA"]) else None
    mBs = [z[f"maskB_{k}"] if on else None for k, on in enumerate(z["has_maskB"])]
    return c, z, mA, mBs


@pytest.mark.parametrize("name", PRO_CASES)
def test_prologue_matches_live_reference_golden(name):
    c, z, mA, mBs = load_prologue_golden(name)
    for k in range(c["nn"]):
        got = O.certainty_prologue(z["raw_cert"][k], z["warp"][k], mA, mBs[k], c["certainty_thresh"])
        assert np.array_equal(got, z["cert_post"][k], equal_nan=True), (name, k)
        via_torch = O.certainty_prologue_torch(torch.from_numpy(z["raw_cert"][k]), torch.from_numpy(z["warp"][k]), mA, mBs[k],
                                               c["certainty_thresh"]).numpy()
        assert np.array_equal(via_torch, z["cert_post"][k], equal_nan=True), (name, k)


@pytest.mark.parametrize("shape", [(64, 64, 64, 64), (128, 128, 80, 80), (96, 120, 60, 75), (50, 61, 50, 61), (64, 64, 32, 32),
                                   (40, 40, 37, 53), (160, 160, 100, 100)])
def test_explicit_index_arithmetic_equals_aten(shape):
    """nearest resize + nearest grid_sample restated with explicit indices == F.interpolate / F.grid_sample, including
    coordinates exactly between two pixels, outside the image, NaN and inf."""
    H, W, hm, wm = shape
    rs = np.random.RandomState(H * 7 + wm)
    cert = rs.rand(H, W).astype(np.float32)
    cert[3, 3], cert[4, 4] = np.nan, np.inf
    warp = rs.rand(H, W, 4).astype(np.float32) * 2.4 - 1.2
    for ch, size in ((2, W), (3, H)):
        k = rs.randint(-1, size + 1, size=(H, W)).astype(np.float64) + 0.5
        adv = ((k + 0.5) / (size / 2) - 1).astype(np.float32)
        rows = slice(ch - 2, None, 3)
        warp[rows, :, ch] = adv[rows]
    warp[1, 1, 2], warp[2, 2, 3], warp[5, 5, 2] = np.nan, np.inf, -np.inf
    mA = (rs.rand(hm, wm) > 0.3).astype(np.uint8)
    mB = (rs.rand(hm, wm) > 0.3).astype(np.uint8)
    for a, b in ((None, None), (mA, None), (None, mB), (mA, mB)):
        e = O.certainty_prologue(cert, warp, a, b, 0.2)
        t = O.certainty_prologue_torch(torch.from_numpy(cert), torch.from_numpy(warp), a, b, 0.2).numpy()
        assert np.array_equal(e, t, equal_nan=True)


def collect_case():
    """Raw certainty, warp and masks of three neighbours (80^2 maps, 50^2 masks, the second neighbour without a mask)."""
    rs = np.random.RandomState(77)
    H = W = 80
    hm = wm = 50
    nn = 3
    raw = rs.rand(nn, H, W).astype(np.float32)
    warp = rs.rand(nn, H, W, 4).astype(np.float32) * 2.2 - 1.1
    mA = (rs.rand(hm, wm) > 0.2).astype(np.uint8)
    mBs = [(rs.rand(hm, wm) > 0.4).astype(np.uint8), None, (rs.rand(hm, wm) > 0.1).astype(np.uint8)]
    return raw, warp, mA, mBs


def test_prologue_vs_live_collect_reference_matches():
    """Fresh inputs through the unmodified ``_collect_reference_matches`` with a stub matcher where the reference is
    installed; elsewhere against its stored output (tests/golden/make_reference_golden.py)."""
    raw, warp, mA, mBs = collect_case()
    nn, (hm, wm) = raw.shape[0], mA.shape
    if not ref_import.reference_available():
        from tests.helpers import load_reference_golden
        stored = load_reference_golden()
        for k in range(nn):
            stored.check(f"collect/cert/{k}", O.certainty_prologue(raw[k], warp[k], mA, mBs[k], 0.35).ravel())
        return
    ref = ref_import.import_reference(full_pipeline=True)
    P = ref.pipeline

    class Stub:
        def match_grids_batch(self, imA, nn_images):
            return [(torch.from_numpy(warp[k]), torch.from_numpy(raw[k])) for k in range(nn)]

    cfg = ref.config.DensePipelineConfig(output_path="/tmp/x.ply", certainty_thresh=0.35)
    packed = P._PackedReferenceBatch(ref_id=0, ref_path="", imA_np=np.zeros((hm, wm, 3), np.uint8), maskA_np=mA, wA_cam=100,
                                     hA_cam=100, nn_ids=[1, 2, 3], nn_masks=mBs,
                                     nn_arrays=[np.zeros((hm, wm, 3), np.uint8)] * nn)
    mr, cnt = P._collect_reference_matches(packed, Stub(), cfg, 0, None)
    assert cnt == nn
    for k in range(nn):
        got = O.certainty_prologue(raw[k], warp[k], mA, mBs[k], 0.35)
        assert np.array_equal(got, mr.cert_list_cpu[k].numpy(), equal_nan=True)
        assert torch.equal(mr.warp_list_cpu[k], torch.from_numpy(warp[k]))
