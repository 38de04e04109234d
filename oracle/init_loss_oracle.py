"""Oracle for the expert-initialisation scene-coordinate loss.  TEST INFRASTRUCTURE ONLY.

A restatement of util.py:18-35 (assert_size) and init_expert.py:114-130 (crop, mask of valid target cells, distance,
robust loss) built from the same torch ops in the same order, so that torch's own autograd provides the reference
gradient.  It runs on the CPU in float32 (what the original computes in, on its GPU) or, with dtype=torch.float64, as the
higher-precision yardstick that the fp32 comparison is judged by.  One deliberate difference: where assert_size prints an
error and calls exit(), this raises RuntimeError, as esac_b200.api.init_loss does.

Only tests/ and examples/ may import this module; the product path (esac_b200/csrc/initloss.cu) never does.
"""
from __future__ import annotations

import torch


def clamp_tensor(coords1: torch.Tensor, coords2: torch.Tensor) -> torch.Tensor:
    """util.py:13-16: crop coords1 to the height and width of coords2."""
    return coords1[:, :, 0:coords2.size(2), 0:coords2.size(3)]


def assert_size(coords1: torch.Tensor, coords2: torch.Tensor):
    """util.py:18-35: equal height and width up to 1 px, then both cropped to the common top-left region."""
    delta_h = coords1.size(2) - coords2.size(2)
    delta_w = coords1.size(3) - coords2.size(3)
    if abs(delta_h) > 1 or abs(delta_w) > 1:
        raise RuntimeError(f"Tensor size mismatch! {tuple(coords1.size())} {tuple(coords2.size())}")
    if delta_h > 0 or delta_w > 0:
        coords1 = clamp_tensor(coords1, coords2)
    if delta_h < 0 or delta_w < 0:
        coords2 = clamp_tensor(coords2, coords1)
    return coords1, coords2


def init_loss(prediction: torch.Tensor, gt_coords: torch.Tensor, cutloss: float, dtype=torch.float32) -> torch.Tensor:
    """The robust loss of init_expert.py:114-130 for one image.  prediction / gt_coords [1,3,h,w] or [3,h,w]
    (prediction may require grad)."""
    if prediction.dim() == 3:
        prediction = prediction.unsqueeze(0)
    if gt_coords.dim() == 3:
        gt_coords = gt_coords.unsqueeze(0)
    prediction = prediction.to(dtype)
    gt_coords = gt_coords.to(dtype)
    prediction, gt_coords = assert_size(prediction, gt_coords)       # :114
    prediction = prediction.squeeze().contiguous().view(3, -1)       # :115
    gt_coords = gt_coords.squeeze().contiguous().view(3, -1)         # :116
    coords_mask = gt_coords.abs().sum(0) != 0                        # :119
    prediction = prediction[:, coords_mask]                          # :120
    gt_coords = gt_coords[:, coords_mask]                            # :121
    loss = torch.norm(prediction - gt_coords, dim=0)                 # :123
    loss_l1 = loss[loss <= cutloss]                                  # :126
    loss_sqrt = loss[loss > cutloss]                                 # :127
    loss_sqrt = torch.sqrt(cutloss * loss_sqrt)                      # :128
    return (loss_l1.sum() + loss_sqrt.sum()) / float(loss.size(0))   # :130


def valid_count(gt_coords: torch.Tensor, h: int, w: int) -> int:
    """Number of valid target cells in the top-left h x w region (the denominator of the loss)."""
    g = torch.as_tensor(gt_coords)
    g = g.reshape(3, g.shape[-2], g.shape[-1])[:, :h, :w]
    return int((g.abs().sum(0) != 0).sum())


def init_loss_and_grad(prediction, gt_coords, cutloss, dtype=torch.float32):
    """(loss, d loss / d prediction [3,H,W] of the UNcropped prediction) through torch autograd, as
    `robust_loss.backward()` (init_expert.py:132)."""
    p = torch.as_tensor(prediction).detach().clone().to(dtype).requires_grad_(True)
    loss = init_loss(p, torch.as_tensor(gt_coords), cutloss, dtype)
    loss.backward()
    g = p.grad
    return float(loss.detach()), (g[0] if g.dim() == 4 else g)


def distances(prediction, gt_coords, dtype=torch.float64):
    """Per-cell ||prediction - gt|| over the common top-left region, [h,w] (for locating cells near the kink)."""
    p = torch.as_tensor(prediction).to(dtype)
    g = torch.as_tensor(gt_coords).to(dtype)
    p = p.reshape(3, p.shape[-2], p.shape[-1])
    g = g.reshape(3, g.shape[-2], g.shape[-1])
    h, w = min(p.shape[1], g.shape[1]), min(p.shape[2], g.shape[2])
    return torch.norm(p[:, :h, :w] - g[:, :h, :w], dim=0)
