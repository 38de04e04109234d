"""torch.autograd wrapper around esac.backward (SURVEY.md section 8f, rank 1).

The reference's trainer calls the extension, then builds the gating gradient by hand and feeds both gradients to
torch.autograd.backward (train_esac.py:151-180).  EsacLoss packages exactly that: its forward returns the expected
pose loss, its backward hands d loss / d sceneCoordinates (from the extension) and the REINFORCE-style gating
gradient to autograd -- loss * histogram(e_hyps) in the default mode (train_esac.py:174-176), or, in the trainer's
`expertselection` mode (one expert drawn and expanded to all hypotheses, train_esac.py:133-135), `loss` at the drawn
expert only (train_esac.py:171-173).  CUDA tensors stay on the device."""
from __future__ import annotations

import torch

from . import api


class EsacLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, scene_coordinates, gating_log_probs, hyp_assignment, gt_pose, w_rot, w_trans, loss_cut, shift_x,
                shift_y, focal_length, ppoint_x, ppoint_y, inlier_threshold, inlier_alpha, inlier_beta, max_reproj,
                sub_sampling, expert_selection=None):
        grads = torch.zeros_like(scene_coordinates)
        loss = api.backward(scene_coordinates.detach(), grads, hyp_assignment, gt_pose, w_rot, w_trans, loss_cut, shift_x,
                            shift_y, focal_length, ppoint_x, ppoint_y, inlier_threshold, inlier_alpha, inlier_beta,
                            max_reproj, sub_sampling)
        E = scene_coordinates.shape[0]
        if expert_selection is None:
            # expert.expand(M) (train_esac.py:135-136) is a stride-0 view: that is the expertselection branch
            expert_selection = hyp_assignment.dim() == 1 and hyp_assignment.shape[0] > 1 and hyp_assignment.stride(0) == 0
        if expert_selection:
            g_gating = torch.zeros(E)
            g_gating[int(hyp_assignment[0])] = loss                                      # train_esac.py:171-173
        else:
            hist = torch.histc(hyp_assignment.float().cpu(), bins=E, min=0, max=E - 1)   # train_esac.py:140
            g_gating = loss * hist                                                        # train_esac.py:174-176
        ctx.save_for_backward(grads, g_gating.to(gating_log_probs.device).reshape(gating_log_probs.shape))
        return scene_coordinates.new_tensor(loss)

    @staticmethod
    def backward(ctx, grad_out):
        g_coords, g_gating = ctx.saved_tensors
        return (g_coords * grad_out, g_gating * grad_out) + (None,) * 16


def esac_loss(scene_coordinates, gating_log_probs, hyp_assignment, gt_pose, *params, expert_selection=None):
    """params: wLossRot, wLossTrans, lossCut, shiftX, shiftY, focalLength, ppointX, ppointY, inlierThreshold,
    inlierAlpha, inlierBeta, maxReproj, subSampling -- the positional tail of esac.backward.
    expert_selection: True = the trainer's `expertselection` gating gradient (loss at the drawn expert), False = loss *
    histogram, None = decide from the assignment tensor (a stride-0 `expert.expand(M)` view means expert selection)."""
    return EsacLoss.apply(scene_coordinates, gating_log_probs, hyp_assignment, gt_pose, *params, expert_selection)


class ReprojLoss(torch.autograd.Function):
    """ref_expert.py:103-150 as one autograd node: forward = the robust reprojection loss of a batch of predictions
    (mean over the batch of the per-image losses; the reference has one image per step), backward = its gradient, both
    from the single fused kernel behind api.reproj_loss."""

    @staticmethod
    def forward(ctx, prediction, gt_poses, focal_length, pad_x, pad_y, cut_loss, sub_sampling, ppoint_x, ppoint_y):
        grads = torch.empty_like(prediction)
        losses = api.reproj_loss(prediction.detach(), gt_poses, focal_length, pad_x, pad_y, cut_loss, sub_sampling, ppoint_x,
                                 ppoint_y, outGradients=grads)
        ctx.save_for_backward(grads)
        ctx.batch = len(losses)
        return prediction.new_tensor(sum(losses) / len(losses))

    @staticmethod
    def backward(ctx, grad_out):
        (grads,) = ctx.saved_tensors
        return (grads * (grad_out / ctx.batch),) + (None,) * 8


def reproj_loss(prediction, gt_poses, focal_length, pad_x, pad_y, cut_loss, sub_sampling=8, ppoint_x=None, ppoint_y=None):
    """Drop-in for the loss block of ref_expert.py: `robust_loss = reproj_loss(prediction, gt_pose, f, padX, padY,
    opt.cutloss)` followed by `robust_loss.backward()`.  prediction [B,3,H,W] (CUDA), gt_poses [B,4,4] camera->world."""
    return ReprojLoss.apply(prediction, gt_poses, focal_length, pad_x, pad_y, cut_loss, sub_sampling, ppoint_x, ppoint_y)


class InitLoss(torch.autograd.Function):
    """init_expert.py:112-132 as one autograd node: forward = mean over the batch of the per-image scene-coordinate
    losses, backward = their gradient, both from the single fused kernel behind api.init_loss.  The kernel returns the
    gradient of each image's SUM; the 1/(B*count_b) of the two means is folded into the multiply by grad_out, with a scale
    of 0 for an image without a valid cell (its loss is NaN, its gradient zero, as autograd gives the original)."""

    @staticmethod
    def forward(ctx, prediction, gt_coords, cut_loss):
        grads = torch.empty_like(prediction)
        res = api.init_loss(prediction.detach(), gt_coords, cut_loss, outGradients=grads)
        B = len(res)
        scale = torch.tensor([1.0 / (B * c) if c else 0.0 for _, c in res], dtype=prediction.dtype)
        shape = (B, 1, 1, 1) if prediction.dim() == 4 else (1, 1, 1)
        ctx.save_for_backward(grads, scale.view(shape).to(prediction.device))
        return prediction.new_tensor(sum(l for l, _ in res) / B)

    @staticmethod
    def backward(ctx, grad_out):
        grads, scale = ctx.saved_tensors
        return grads * (scale * grad_out), None, None


def init_loss(prediction, gt_coords, cut_loss):
    """Drop-in for the loss block of init_expert.py: `robust_loss = init_loss(prediction, gt_coords, opt.cutloss)`
    followed by `robust_loss.backward()`, in place of util.assert_size through the division (:114-130).  prediction and
    gt_coords [B,3,h,w] or [3,h,w] (sizes may differ by one pixel); returns the mean of the B per-image losses."""
    return InitLoss.apply(prediction, gt_coords, cut_loss)
