"""Recognition crop preprocessing (SURVEY §8 f2), CPU side: the numpy restatement of OpenCV's float32 Lanczos4 / cubic resize is pinned
against cv2 itself (the reference's dependency), the whole per-crop chain against the product's cv2-based host mirror (itself pinned to
the reference processor in test_host_cpu.py::test_tiling_and_prompt_match_oracle), and the host plan of the device path is checked."""
from pathlib import Path

import numpy as np
import pytest
import torch

cv2 = pytest.importorskip("cv2")

from oracle import preproc_oracle as P
from surya_b200.config import tiny_rec
from surya_b200.recognition import build_preprocess_plan, scale_to_fit, tile_image

GOLDEN = Path(__file__).resolve().parent / "golden"
TOL_255 = 5e-4          # on the 0..255 scale: float32 summation-order noise of a 64-tap sum of values up to 255 (measured ~1e-4)


@pytest.mark.parametrize("h,w,dh,dw", [(48, 512, 52, 549), (52, 549, 56, 560), (40, 300, 56, 308), (64, 900, 84, 924),
                                       (300, 2000, 202, 1297), (20, 60, 97, 291), (33, 47, 28, 56)])
def test_resize_restatement_pinned_to_cv2(h, w, dh, dw):
    rng = np.random.default_rng(h * w)
    img = rng.integers(0, 256, (h, w, 3)).astype(np.float32)
    for mode, flag in (("lanczos", cv2.INTER_LANCZOS4), ("cubic", cv2.INTER_CUBIC)):
        ref = cv2.resize(img, (dw, dh), interpolation=flag)
        err = np.abs(ref - P.resize(img, dw, dh, mode)).max()
        assert err <= TOL_255, f"{mode} {h}x{w}->{dh}x{dw}: {err}"


@pytest.mark.parametrize("h,w", [(48, 512), (40, 300), (64, 900), (300, 2000), (20, 60), (168, 168), (56, 560), (250, 1100)])
def test_crop_chain_matches_the_cv2_host_mirror(h, w):
    rng = np.random.default_rng(h + w)
    crop = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    tiles, grid = P.process_crop(crop)
    ref_tiles, ref_grid = tile_image(scale_to_fit(np.asarray(crop, dtype=np.float32), (1024, 256)))
    assert grid == ref_grid and tiles.shape == ref_tiles.shape
    # normalised scale: 1 / (255 * std) per unit of the 0..255 scale; the cubic stage amplifies the first stage's noise by < 2
    assert np.abs(tiles - ref_tiles).max() <= 2 * TOL_255 / 255 / 0.224


def test_preprocess_plan():
    cfg = tiny_rec()
    rng = np.random.default_rng(1)
    sizes = [(48, 512), (40, 300), (300, 2000), (56, 560), (168, 168)]
    crops = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in sizes]
    plan = build_preprocess_plan(crops, cfg)
    desc = plan["desc"].reshape(len(crops), -1)
    row = 0
    for i, (h, w) in enumerate(sizes):
        nh, nw = P.fit_size(h, w)
        hb, wb = -(-nh // 28) * 28, -(-nw // 28) * 28
        assert desc[i, 1:7].tolist() == [h, w, nh, nw, hb, wb]
        assert desc[i, 8] == row and plan["grids"][i] == (1, hb // 14, wb // 14)
        assert desc[i, 0] % 16 == 0
        assert np.array_equal(plan["packed"][desc[i, 0]: desc[i, 0] + h * w * 3].reshape(h, w, 3), crops[i])
        row += (hb // 14) * (wb // 14)
    assert plan["n_rows"] == row and plan["any_stage1"] == 1
    assert plan["max"] == (max(d[3] for d in desc), max(d[4] for d in desc), max(d[5] for d in desc), max(d[6] for d in desc))
    with pytest.raises(Exception):
        build_preprocess_plan([np.zeros((0, 5, 3), np.uint8)], cfg)


def test_crop_chain_pinned_to_the_reference_processor():
    """The restatement against what the reference's OWN SuryaOCRProcessor (scale_to_fit + _process_and_tile, unmodified) returned
    for the same seeded crops (tests/golden/reference_host.pt, written by oracle/make_golden.py): same grids, tiles equal to float32
    rounding of the OpenCV resizes — a seeded sample of tile rows element by element, every row through its sum and sum of squares."""
    from oracle.make_golden import preproc_crops

    cfg = tiny_rec()
    golden = torch.load(GOLDEN / "reference_host.pt")["crop_chain"]
    crops = preproc_crops()
    assert len(crops) == len(golden)
    tol = 2 * TOL_255 / 255 / 0.224
    for crop, ref in zip(crops, golden):
        tiles, grid = P.process_crop(crop, cfg.vision_encoder.patch_size, cfg.merge_size)
        assert crop.shape == ref["shape"] and tuple(grid) == ref["grid"], crop.shape
        assert tiles.shape[0] == ref["row_sums"].numel()
        assert np.abs(tiles[ref["rows"].numpy()] - ref["tile_rows"].numpy()).max() <= tol, crop.shape
        assert np.abs(tiles.astype(np.float64).sum(1) - ref["row_sums"].numpy()).max() <= tol * tiles.shape[1], crop.shape
        sq_tol = tol * (2 * np.abs(tiles.astype(np.float64)).sum(1) + tol * tiles.shape[1])     # |a^2 - b^2| <= |a - b| (2|a| + |a - b|)
        assert (np.abs((tiles.astype(np.float64) ** 2).sum(1) - ref["row_sq"].numpy()) <= sq_tol).all(), crop.shape
