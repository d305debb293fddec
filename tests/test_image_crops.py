"""The reference's own tests for this path (tests/test_image_crops.py:6-57) re-hosted against
moondream_b200.image_crops, plus the golden crop hashes produced by the reference implementation."""
import hashlib
import json
import os

import numpy as np
import torch

from moondream_b200.image_crops import overlap_crop_image, reconstruct_from_crops, select_tiling

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def test_overlap_crop_basic():
    test_image = np.zeros((800, 600, 3), dtype=np.uint8)
    test_image[300:500, 200:400] = 255
    result = overlap_crop_image(test_image, overlap_margin=4, max_crops=12)
    assert result["crops"][0].shape == (378, 378, 3)
    assert len(result["crops"]) > 1
    assert all(crop.shape == (378, 378, 3) for crop in result["crops"])
    assert len(result["tiling"]) == 2


def test_overlap_crop_small_image():
    test_image = np.zeros((300, 200, 3), dtype=np.uint8)
    result = overlap_crop_image(test_image, overlap_margin=4, max_crops=12)
    assert result["crops"][0].shape == (378, 378, 3)
    assert len(result["crops"]) == 2
    assert result["tiling"] == (1, 1)


def test_reconstruction():
    test_image = np.zeros((800, 600, 3), dtype=np.uint8)
    test_image[300:500, 200:400] = 255
    result = overlap_crop_image(test_image, overlap_margin=4, max_crops=12)
    crops_tensor = [torch.from_numpy(crop) for crop in result["crops"][1:]]
    reconstructed = reconstruct_from_crops(crops_tensor, result["tiling"], overlap_margin=4)
    rec = reconstructed.numpy()
    center = rec[rec.shape[0] // 2 - 100: rec.shape[0] // 2 + 100,
                 rec.shape[1] // 2 - 100: rec.shape[1] // 2 + 100].mean()
    assert center > rec[:100, :100].mean() + 100


def test_golden_crops_from_reference():
    from moondream_b200 import synth
    from oracle.moondream_oracle import overlap_crops

    gold = json.load(open(os.path.join(GOLDEN, "crops.json")))
    for c in gold["cases"]:
        img = synth.synthetic_image(c["image_index"], c["height"], c["width"])
        out = overlap_crop_image(img, overlap_margin=4, max_crops=12)
        assert list(out["tiling"]) == c["tiling"] and out["crops"].shape[0] == c["n_crops"]
        assert hashlib.sha256(out["crops"].tobytes()).hexdigest()[:16] == c["sha256"], c
        mine, tiling = overlap_crops(img, 4, 12)            # the oracle's restatement as well
        assert list(tiling) == c["tiling"] and np.array_equal(mine, out["crops"])


def test_select_tiling_properties():
    for (h, w, expect) in [(266, 266, (1, 1)), (267, 267, (3, 3)), (656, 912, (3, 4)), (912, 656, (4, 3)),
                           (968, 1808, (2, 4)), (688, 488, (4, 2))]:
        assert select_tiling(h, w, 266, 12) == expect, (h, w)
    rng = np.random.default_rng(0)
    for _ in range(500):
        h, w = int(rng.integers(1, 4000)), int(rng.integers(1, 4000))
        th, tw = select_tiling(h, w, 266, 12)
        assert th >= 1 and tw >= 1 and th * tw <= 12


def test_random_sizes_against_the_oracle_and_the_reference():
    """Ragged sizes, extreme aspect ratios and every max_crops: product == oracle restatement bit for bit == the
    unmodified reference (`image_crops.py:58-167`, PIL-Lanczos branch; tests/golden/reference_bitwise.json); margins
    other than the default too.  Reconstruction of per-crop index maps must tile the stitched grid without holes."""
    from moondream_b200 import synth
    from neartie import reference_bitwise
    from oracle.make_golden_bitwise import crop_cases
    from oracle.reference_shim import tensor_sha256
    from oracle.moondream_oracle import overlap_crops

    gold = reference_bitwise()["crops"]
    cases = crop_cases()
    assert len(cases) == len(gold) == 21
    for (idx, h, w, max_crops, margin), theirs in zip(cases, gold):
        img = synth.synthetic_image(idx, h, w)
        out = overlap_crop_image(img, overlap_margin=margin, max_crops=max_crops)
        th, tw = out["tiling"]
        assert out["crops"].dtype == np.uint8 and out["crops"].shape == (1 + th * tw, 378, 378, 3) and th * tw <= max_crops
        mine, tiling = overlap_crops(img, margin, max_crops)
        assert tuple(tiling) == (th, tw) and np.array_equal(mine, out["crops"]), (h, w, max_crops, margin)
        assert theirs["tiling"] == [th, tw] and theirs["sha256"] == tensor_sha256(torch.from_numpy(out["crops"])), (h, w)
        # stitching per-crop constant maps: every output cell is owned by exactly one crop (no holes, no NaNs)
        grid = 27
        feats = [torch.full((grid, grid, 1), float(i)) for i in range(th * tw)]
        rec = reconstruct_from_crops(feats, (th, tw), patch_size=1, overlap_margin=margin)
        assert rec.shape[:2] == (th * (grid - 2 * margin) + 2 * margin, tw * (grid - 2 * margin) + 2 * margin)
        assert set(rec.unique().tolist()) == set(float(i) for i in range(th * tw))
