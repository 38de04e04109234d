"""GPU parity of the fused expert-initialisation loss (init_expert.py:112-132) against the torch restatement (run with
`-m gpu`).

The bar is the one tests/test_gpu_reproj.py states: the yardstick is the float64 evaluation of the original op sequence,
and the kernel must be at least as accurate as torch's own float32 evaluation -- RMS deviation of the gradient from
float64 within 1.5x of torch-float32's, worst cell within 4x of torch-float32's worst cell, loss within 1e-5 relative,
valid-cell counts exact.  At d = cut the gradient halves, and a cell whose distance lies within float32 rounding of the
cut may land on either side in ANY float32 evaluation; cells within 1e-4 of the cut (relative, by the float64 evaluation)
are left out of the gradient comparison and counted (they must stay a handful).
"""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

CUT = 100.0


def _case(B, ph, pw, gh, gw, sparse, seed):
    from test_init_loss_oracle import make_case
    pairs = [make_case(seed + b, ph, pw, gh, gw, sparse=sparse) for b in range(B)]
    return np.concatenate([p for p, _ in pairs]), np.concatenate([g for _, g in pairs])


@pytest.mark.parametrize("B,ph,pw,gh,gw,sparse", [
    (1, 60, 80, 60, 80, 0.0),
    (3, 60, 80, 60, 80, 0.0),
    (3, 60, 80, 60, 80, 0.95),     # SfM-style targets: most cells invalid
    (2, 33, 47, 33, 47, 0.1),      # odd size: scalar path
    (2, 61, 80, 60, 80, 0.0),      # prediction one row taller: vector path with a dead row
    (2, 60, 80, 61, 79, 0.3),      # mixed-sign crop: scalar path
    (1, 480, 640, 480, 640, 0.0),
    (1, 480, 640, 480, 640, 0.95),
])
@pytest.mark.parametrize("kind", ["cpu", "cuda"])
def test_init_loss_and_gradient_match_torch(B, ph, pw, gh, gw, sparse, kind):
    import torch
    import esac_b200.api as api
    from oracle.init_loss_oracle import distances, init_loss_and_grad, valid_count
    pred, gt = _case(B, ph, pw, gh, gw, sparse, 400 + ph + pw)
    dev = "cuda" if kind == "cuda" else "cpu"
    tp, tt = torch.from_numpy(pred).to(dev), torch.from_numpy(gt).to(dev)
    tg = torch.full(pred.shape, 7.0, device=dev)      # overwritten, not accumulated; cropped cells -> 0
    res = api.init_loss(tp, tt, CUT, outGradients=tg)
    g = tg.cpu().numpy().astype(np.float64)
    h, w = min(ph, gh), min(pw, gw)
    for b in range(B):
        loss, count = res[b]
        assert count == valid_count(gt[b], h, w)
        l32, g32 = init_loss_and_grad(pred[b:b + 1], gt[b:b + 1], CUT)
        l64, g64 = init_loss_and_grad(pred[b:b + 1], gt[b:b + 1], CUT, dtype=torch.float64)
        assert abs(loss - l64) <= 1e-5 * max(1.0, abs(l64)), (loss, l32, l64)
        gk = g[b] / count                              # the kernel writes the gradient of the image's sum
        assert (gk[:, h:, :] == 0).all() and (gk[:, :, w:] == 0).all()
        d64 = np.zeros((ph, pw))
        d64[:h, :w] = distances(pred[b], gt[b]).numpy()
        kink = np.abs(d64 - CUT) < 1e-4 * CUT
        assert kink.sum() <= 2e-4 * ph * pw + 2
        keep = ~kink[None]
        d32 = (g32.double() - g64).numpy() * keep
        dk = (gk - g64.numpy()) * keep
        scale = g64.abs().max().item()
        rms_k, rms_t = np.sqrt((dk ** 2).mean()), np.sqrt((d32 ** 2).mean())
        assert rms_k <= 1.5 * rms_t + 1e-7 * scale, (rms_k, rms_t)
        assert np.abs(dk).max() <= 4 * np.abs(d32).max() + 1e-6 * scale, (np.abs(dk).max(), np.abs(d32).max(), scale)
    # repeat: bit-identical; loss-only call: the same numbers, no gradient needed
    tg2 = torch.empty_like(tg)
    assert api.init_loss(tp, tt, CUT, outGradients=tg2) == res
    assert torch.equal(tg2, tg)
    assert api.init_loss(tp, tt, CUT) == res


def test_init_loss_edge_cases():
    """No valid cell -> NaN loss, count 0, zero gradient; NaN target cell -> counted, not summed, NaN gradient; d == 0
    and invalid cells -> zero gradient; d == cut -> the L1 branch."""
    import torch
    import esac_b200.api as api
    from oracle.init_loss_oracle import init_loss_and_grad
    from test_init_loss_oracle import golden_cases
    cases = golden_cases()
    p, g, _ = cases["edges"]
    pz, gz, _ = cases["all_invalid"]
    for pred, gt in ((p, g), (pz, gz)):
        tg = torch.full(pred.shape, 7.0, device="cuda")
        (loss, count), = api.init_loss(torch.from_numpy(pred).cuda(), torch.from_numpy(gt).cuda(), CUT, outGradients=tg)
        l64, g64 = init_loss_and_grad(pred, gt, CUT, dtype=torch.float64)
        gk = tg[0].cpu().double()
        if count == 0:
            assert math.isnan(loss) and math.isnan(l64) and (gk == 0).all()
            continue
        assert count == 29 and abs(loss - l64) <= 1e-5 * abs(l64)
        assert torch.isnan(gk[:, 1, 2]).all() and torch.isnan(g64[:, 1, 2]).all()
        assert (gk[:, 2, 3] == 0).all() and (gk[:, 3, 4] == 0).all()
        fin = ~torch.isnan(g64)
        assert torch.isfinite(gk[fin]).all()
        np.testing.assert_allclose((gk / count)[fin].numpy(), g64[fin].numpy(), rtol=1e-5, atol=1e-9)
        np.testing.assert_allclose(gk[:, 4, 0].numpy(), np.array([60.0, 80.0, 0.0]) / CUT, rtol=1e-6)


def test_init_loss_autograd_node_trains_like_the_original():
    import torch
    from esac_b200.autograd import init_loss
    from oracle.init_loss_oracle import init_loss as ref_loss
    pred, gt = _case(3, 24, 32, 24, 32, 0.5, 900)
    gt[1] = 0.0                                        # an image without a valid cell: NaN loss, zero gradient
    p = torch.from_numpy(pred).cuda().requires_grad_(True)
    loss = init_loss(p, torch.from_numpy(gt).cuda(), CUT)
    (loss * 3.0).backward()
    assert math.isnan(loss.item())
    assert (p.grad[1] == 0).all()
    # the other two images against the float64 original, with the mean over B = 3 in the scale
    q = torch.from_numpy(pred).double().requires_grad_(True)
    ref = sum(ref_loss(q[b], torch.from_numpy(gt[b]), CUT, dtype=torch.float64) for b in (0, 2)) / 3
    (ref * 3.0).backward()
    gk = p.grad.cpu().double()
    assert (gk - q.grad).abs().max().item() < 1e-5 * q.grad.abs().max().item()
    # B = 1 drop-in with [3,h,w] tensors: the loss block of init_expert.py followed by .backward()
    p1 = torch.from_numpy(pred[0]).cuda().requires_grad_(True)
    l1 = init_loss(p1, torch.from_numpy(gt[0]).cuda(), CUT)
    l1.backward()
    q1 = torch.from_numpy(pred[0]).double().requires_grad_(True)
    r1 = ref_loss(q1, torch.from_numpy(gt[0]), CUT, dtype=torch.float64)
    r1.backward()
    assert abs(l1.item() - r1.item()) < 1e-5 * abs(r1.item())
    assert (p1.grad.cpu().double() - q1.grad).abs().max().item() < 1e-5 * q1.grad.abs().max().item()


def test_init_loss_rejects_bad_input():
    import torch
    import esac_b200.api as api
    with pytest.raises(RuntimeError, match="size mismatch"):
        api.init_loss(torch.zeros(1, 3, 10, 8), torch.ones(1, 3, 8, 8), CUT)
    with pytest.raises(RuntimeError, match="size mismatch"):
        api.init_loss(torch.zeros(1, 3, 8, 8).cuda(), torch.ones(1, 3, 8, 6).cuda(), CUT)
    with pytest.raises(RuntimeError, match="Float"):
        api.init_loss(torch.zeros(1, 3, 8, 8, dtype=torch.float64), torch.ones(1, 3, 8, 8), CUT)
    with pytest.raises(RuntimeError, match="batch"):
        api.init_loss(torch.zeros(2, 3, 8, 8), torch.ones(1, 3, 8, 8), CUT)
    with pytest.raises(RuntimeError):
        api.init_loss(torch.zeros(1, 3, 8, 8), torch.ones(1, 3, 8, 8), CUT, outGradients=torch.zeros(1, 3, 8, 7))
