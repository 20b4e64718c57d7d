"""CPU: pins oracle/io_oracle.py (the checker of csrc/io.cu) against the reference's own functions, through their outputs
stored in tests/golden/io_reference.npz (oracle/make_golden.py runs the unmodified source): DataLoadPreprocess.random_crop /
train_preprocess / augment_image / ToTensor (pytorch/bts_dataloader.py) and compute_errors (pytorch/bts_main.py:144-165)."""
import random

import numpy as np
import pytest

import io_oracle as IO


def test_compute_errors_matches_reference_function(golden):
    want = golden("io_reference")["compute_errors"]
    rng = np.random.RandomState(0)
    gt = rng.uniform(0.5, 70, 5000).astype(np.float32)
    pred = (gt * rng.uniform(0.6, 1.6, 5000)).astype(np.float32)
    got = IO.compute_errors(gt, pred)
    np.testing.assert_allclose(np.array(got, dtype=np.float64), want, rtol=1e-6)


@pytest.mark.parametrize("dataset", ["nyu", "kitti"])
def test_input_prep_matches_reference_loader_transform(golden, dataset):
    g = golden("io_reference")
    rng = np.random.RandomState(1)
    img_u8 = rng.randint(0, 256, (40, 56, 3)).astype(np.uint8)
    dep_u16 = rng.randint(0, 60000, (40, 56)).astype(np.uint16)
    div = 1000.0 if dataset == "nyu" else 256.0
    H, W = 32, 32
    assert len(g[dataset + "_image"]) == 6
    for seed in range(6):
        # replay the reference's own random draws: random_crop (x then y), flip, do_augment, gamma, brightness, np colours
        random.seed(seed)
        np.random.seed(seed)
        x0 = random.randint(0, img_u8.shape[1] - W)
        y0 = random.randint(0, img_u8.shape[0] - H)
        do_flip = random.random()
        do_aug = random.random()
        gamma = brightness = 1.0
        colors = np.ones(3)
        if do_aug > 0.5:
            gamma = random.uniform(0.9, 1.1)
            brightness = random.uniform(0.75, 1.25) if dataset == "nyu" else random.uniform(0.9, 1.1)
            colors = np.random.uniform(0.9, 1.1, size=3)
        want_i, want_d = g[dataset + "_image"][seed], g[dataset + "_depth"][seed]
        got_i, got_d = IO.input_prep(img_u8, dep_u16, div, y0, x0, H, W, do_flip > 0.5, do_aug > 0.5, gamma, brightness, colors)
        np.testing.assert_allclose(got_i, want_i, rtol=1e-6, atol=1e-6)
        np.testing.assert_array_equal(got_d, want_d)


def test_eval_errors_masks_and_clamps():
    rng = np.random.RandomState(2)
    gt = rng.uniform(0, 90, (20, 30)).astype(np.float32)
    pred = rng.uniform(-1, 100, (20, 30)).astype(np.float32)
    pred[0, 0], pred[1, 1] = np.inf, np.nan
    m, n = IO.eval_errors(pred, gt, 1e-3, 80.0, crop=(2, 18, 3, 27))
    assert n == int(((gt > 1e-3) & (gt < 80))[2:18, 3:27].sum()) and all(np.isfinite(m))
    assert IO.depth_to_u16(np.array([1.9996, 0.0, 65.0], dtype=np.float32), 1000.0).tolist() == [1999, 0, 65000]
