"""The expert-initialisation training step (code/init_expert.py:102-139) with its loss block replaced by the fused kernel.

init_expert.py builds its scene-coordinate loss from about ten torch ops per step, two of them boolean-mask gathers that
each stall the host until the device reports how many cells survived; `esac_b200.autograd.init_loss` is the same loss and
gradient as ONE kernel (esac_b200/csrc/initloss.cu) and one read-back.  Dataset and network are stand-ins
(esac_b200.compat, a 1x1-conv "expert" started away from the identity so that there is something to learn); the loop
itself is the reference's.  Target cells without ground truth are zero, as in the reference's datasets: a few percent
(missing depth) by default, ~95 % with --sparse (SfM-initialised environments).  With --check every step is also
evaluated with the original op sequence (oracle/init_loss_oracle.py), loss and gradient.

    python examples/init_expert_step_synthetic.py --iterations 5 --check [--sparse]
"""
from __future__ import annotations

import argparse
import sys
import time
from pathlib import Path

import numpy as np
import torch
import torch.nn as nn

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from esac_b200.autograd import init_loss  # noqa: E402
from esac_b200.compat import OUTPUT_SUBSAMPLE, SyntheticRoomDataset, random_shift  # noqa: E402


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--iterations", type=int, default=5)
    ap.add_argument("--learningrate", "-lr", type=float, default=0.0001)   # init_expert.py:22
    ap.add_argument("--cutloss", "-cl", type=float, default=100)           # :38
    ap.add_argument("--sparse", action="store_true", help="zero ~95%% of the target cells (SfM-style ground truth)")
    ap.add_argument("--check", action="store_true")
    opt = ap.parse_args(argv)
    dev = torch.device("cuda")
    trainset = SyntheticRoomDataset(num_experts=1, length=max(opt.iterations, 1), seed=13, noise=0.05)
    trainset_loader = torch.utils.data.DataLoader(trainset, shuffle=False, num_workers=0)
    model = nn.Conv2d(3, 3, 1).to(dev)                                      # stand-in for Expert
    with torch.no_grad():
        model.weight.copy_((0.9 * torch.eye(3)).view(3, 3, 1, 1))
        model.bias.fill_(0.5)
    optimizer = torch.optim.Adam(model.parameters(), lr=opt.learningrate)   # :86
    missing = 0.95 if opt.sparse else 0.03
    out = []
    for iteration, (idx, image, focallength, gt_pose, gt_coords, gt_expert) in enumerate(trainset_loader):   # :102
        start_time = time.time()
        # cells without ground truth are all-zero targets (deterministic per image)
        rng = np.random.default_rng(1000 + int(idx))
        gt_coords[:, :, torch.from_numpy(rng.random(gt_coords.shape[2:]) < missing)] = 0.0
        gt_coords = gt_coords.to(dev)                                       # :106
        image = image.to(dev)
        padX, padY, image = random_shift(image, OUTPUT_SUBSAMPLE / 2)       # :110
        prediction = model(trainset.prediction_for(int(idx)).to(dev))       # :112 (the stand-in expert sees its prior)
        robust_loss = init_loss(prediction, gt_coords, opt.cutloss)         # :114-130 in one call
        robust_loss.backward()                                              # :132
        loss_value = robust_loss.item()
        if opt.check:
            from oracle.init_loss_oracle import init_loss as original
            p = prediction.detach().cpu().requires_grad_(True)
            ref = original(p, gt_coords.cpu(), opt.cutloss)
            ref.backward()
            assert abs(float(ref) - loss_value) < 1e-5 * max(1.0, abs(float(ref))), (float(ref), loss_value)
            # d loss / d prediction, what autograd hands on to the expert, against the original ops' gradient
            mine = torch.autograd.grad(init_loss(prediction, gt_coords, opt.cutloss), prediction)[0].cpu()
            err = (mine - p.grad).abs().max().item()
            assert err <= 1e-5 * p.grad.abs().max().item(), (err, p.grad.abs().max().item())
        optimizer.step()                                                    # :133
        optimizer.zero_grad()                                               # :135
        print("Iteration: %6d, Loss: %.1f, Time: %.2fs" % (iteration, loss_value, time.time() - start_time), flush=True)  # :137
        out.append(loss_value)
    return out


if __name__ == "__main__":
    main()
