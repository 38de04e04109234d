"""CPU checks of oracle/init_loss_oracle.py, the yardstick of the fused expert-initialisation loss (init_expert.py:112-132).

* In float64 its autograd gradient equals central finite differences away from the kinks (d = cut, d = 0).
* In float32 it returns what the reference's own lines return: tests/golden/init_loss/literal_f32.npz holds the loss and
  gradient of those lines (util.assert_size + init_expert.py:114-130, run by tests/golden/make_init_loss_golden.py) on the
  cases below.
* The edge cases the kernel has to reproduce are pinned: an image without a valid cell, a NaN target cell, d == 0,
  d == cut exactly, and the +-1 crop in each direction, including mixed signs.
"""
import math
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle.init_loss_oracle import distances, init_loss, init_loss_and_grad, valid_count

GOLDEN = Path(__file__).resolve().parent / "golden" / "init_loss" / "literal_f32.npz"
CUT = 100.0   # init_expert.py:38


def make_case(seed, ph, pw, gh, gw, sparse=0.0, spread=150.0):
    """prediction [1,3,ph,pw], target [1,3,gh,gw] float32; `sparse` = share of target cells set to zero; errors spread
    around the cut so both branches of the robust loss are taken."""
    rng = np.random.default_rng(seed)
    gt = rng.normal(0.0, 20.0, (1, 3, gh, gw)).astype(np.float32)
    gt[:, :, rng.random((gh, gw)) < sparse] = 0.0
    pred = rng.normal(0.0, 20.0, (1, 3, ph, pw)).astype(np.float32)
    h, w = min(ph, gh), min(pw, gw)
    dirs = rng.normal(size=(3, h, w))
    dirs /= np.linalg.norm(dirs, axis=0, keepdims=True)
    pred[0, :, :h, :w] = gt[0, :, :h, :w] + (dirs * rng.uniform(0.0, spread, (h, w))).astype(np.float32)
    return pred, gt


def golden_cases():
    """name -> (prediction, target, cut): the inputs the golden file records the reference lines on."""
    cases = {
        "dense": make_case(1, 6, 8, 6, 8),
        "sparse": make_case(2, 9, 12, 9, 12, sparse=0.95),
        "crop_pred_taller": make_case(3, 7, 8, 6, 8),
        "crop_gt_wider": make_case(4, 6, 8, 6, 9),
        "crop_mixed_h+_w-": make_case(5, 7, 8, 6, 9),
        "crop_mixed_h-_w+": make_case(6, 6, 9, 7, 8),
        "all_invalid": (make_case(7, 4, 5, 4, 5)[0], np.zeros((1, 3, 4, 5), np.float32)),
    }
    p, g = make_case(8, 5, 6, 5, 6)
    g[0, :, 1, 2] = [np.nan, 0.0, 0.0]          # NaN target cell: valid, counted, not summed, NaN gradient
    p[0, :, 2, 3] = g[0, :, 2, 3]               # d == 0
    g[0, :, 3, 4] = [0.0, 0.0, 0.0]             # invalid
    g[0, :, 4, 0] = [1.0, 2.0, 3.0]
    p[0, :, 4, 0] = [61.0, 82.0, 3.0]          # d == cut exactly (60-80-100 triangle, exact in float32)
    cases["edges"] = (p, g)
    return {k: (v[0], v[1], CUT) for k, v in cases.items()}


def test_oracle_gradient_matches_finite_differences():
    pred, gt = make_case(11, 5, 7, 5, 7, sparse=0.3)
    p64, g64 = pred.astype(np.float64), gt.astype(np.float64)
    _, grad = init_loss_and_grad(p64, g64, CUT, dtype=torch.float64)
    d = distances(p64, g64).numpy()
    eps = 1e-6
    for c in range(3):
        for y in range(5):
            for x in range(7):
                if abs(d[y, x] - CUT) < 1e-3 or d[y, x] < 1e-3:
                    continue
                q = p64.copy()
                q[0, c, y, x] += eps
                lp = float(init_loss(torch.from_numpy(q), torch.from_numpy(g64), CUT, torch.float64))
                q[0, c, y, x] -= 2 * eps
                lm = float(init_loss(torch.from_numpy(q), torch.from_numpy(g64), CUT, torch.float64))
                fd = (lp - lm) / (2 * eps)
                assert abs(fd - float(grad[c, y, x])) < 1e-7 * max(1.0, abs(fd)), (c, y, x, fd, float(grad[c, y, x]))


@pytest.mark.parametrize("name", sorted(golden_cases()))
def test_oracle_float32_equals_reference_lines(name):
    pred, gt, cut = golden_cases()[name]
    z = np.load(GOLDEN)
    np.testing.assert_array_equal(z[name + "/pred"], pred)     # the case generator has not drifted
    np.testing.assert_array_equal(z[name + "/gt"], gt)
    loss, grad = init_loss_and_grad(pred, gt, cut)
    ref_loss, ref_grad = float(z[name + "/loss"]), z[name + "/grad"]
    if math.isnan(ref_loss):
        assert math.isnan(loss)
    else:
        assert abs(loss - ref_loss) <= 1e-6 * max(1.0, abs(ref_loss)), (loss, ref_loss)
    np.testing.assert_allclose(grad.numpy(), ref_grad, rtol=1e-6, atol=1e-9, equal_nan=True)


def test_edge_cases():
    cases = golden_cases()
    # no valid cell: loss NaN (0 / 0.0), gradient all zero
    pred, gt, cut = cases["all_invalid"]
    loss, grad = init_loss_and_grad(pred, gt, cut)
    assert math.isnan(loss) and (grad == 0).all()
    # NaN target cell: counted but not summed -> finite loss, NaN gradient in that cell only; d == 0 -> zero gradient;
    # invalid cell -> zero gradient; d == cut exactly -> the L1 branch, (p - g)/d / count
    pred, gt, cut = cases["edges"]
    loss, grad = init_loss_and_grad(pred, gt, cut)
    assert math.isfinite(loss)
    n = valid_count(gt, 5, 6)
    assert n == 29
    g = grad.numpy()
    assert np.isnan(g[:, 1, 2]).all() and np.isfinite(np.delete(g.reshape(3, -1), 1 * 6 + 2, axis=1)).all()
    assert (g[:, 2, 3] == 0).all() and (g[:, 3, 4] == 0).all()
    dvec = (pred[0, :, 4, 0].astype(np.float64) - gt[0, :, 4, 0])
    assert np.linalg.norm(dvec) == cut
    np.testing.assert_allclose(g[:, 4, 0], dvec / cut / n, rtol=1e-6)
    # the loss leaves the NaN cell out of the sums but in the count
    d = distances(pred, gt).numpy()
    keep = np.isfinite(d) & (np.abs(gt[0]).sum(0) != 0)
    s = np.where(d <= cut, d, np.sqrt(cut * d))[keep].sum()
    assert abs(loss - s / n) < 1e-5 * max(1.0, s / n)


@pytest.mark.parametrize("ph,pw,gh,gw", [(7, 8, 6, 8), (6, 8, 7, 8), (6, 9, 6, 8), (6, 8, 6, 9), (7, 8, 6, 9), (6, 9, 7, 8),
                                         (7, 9, 6, 8), (6, 8, 7, 9)])
def test_crop_is_top_left_and_cropped_cells_get_zero(ph, pw, gh, gw):
    pred, gt = make_case(20 + ph * 10 + pw, ph, pw, gh, gw)
    h, w = min(ph, gh), min(pw, gw)
    loss, grad = init_loss_and_grad(pred, gt, CUT, dtype=torch.float64)
    ref, ref_grad = init_loss_and_grad(pred[:, :, :h, :w], gt[:, :, :h, :w], CUT, dtype=torch.float64)
    assert loss == ref
    assert tuple(grad.shape) == (3, ph, pw)
    assert (grad[:, h:, :] == 0).all() and (grad[:, :, w:] == 0).all()
    assert torch.equal(grad[:, :h, :w], ref_grad)


def test_size_mismatch_of_two_is_an_error():
    pred, gt = make_case(30, 8, 8, 6, 8)
    with pytest.raises(RuntimeError, match="size mismatch"):
        init_loss(torch.from_numpy(pred), torch.from_numpy(gt), CUT)
    pred, gt = make_case(31, 6, 8, 6, 10)
    with pytest.raises(RuntimeError, match="size mismatch"):
        init_loss(torch.from_numpy(pred), torch.from_numpy(gt), CUT)
