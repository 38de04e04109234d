"""HBM roofline of the fused expert-initialisation loss kernel (esac_b200/csrc/initloss.cu): 24 B read + 12 B written per
cell.  For B in {1, 8, 64, 256} maps of 60x80 and 480x640, dense (3 % of the target cells empty) and sparse (95 % empty),
prints the kernel time (CUDA events around the launch, the library's own stage timer, median of warm calls), the
achieved bytes/s at 36 B per cell against the project's measured HBM peak, the time of the whole call, and the time of
the original torch op sequence + autograd (init_expert.py:114-132, one image at a time as the reference trains,
including the host synchronisations of its two boolean-mask gathers) on the same inputs.

Every timed call reads inputs that are not in L2: where one batch is smaller than ~3x the 126 MB L2, the calls rotate
over enough copies of it that the rotation exceeds that.  The GPU name and power limit are read in the same run.

    python tools/initloss_bandwidth.py [--reps 30]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import esac_b200.api as api  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BYTES_PER_CELL = 36
CUT = 100.0
L2_BYTES = 126 * 2 ** 20
HBM_PEAK_DESIGN = 6569.3   # GB/s, MEASURED_PEAKS.json of the B200 boxes the project measures on (DESIGN.md section 4)


def torch_ref(pred, gt, cut):
    """init_expert.py:114-132 on CUDA tensors, one image (sizes already equal)."""
    p = pred.detach().clone().requires_grad_(True)
    prediction = p.squeeze().contiguous().view(3, -1)
    gt_coords = gt.squeeze().contiguous().view(3, -1)
    coords_mask = gt_coords.abs().sum(0) != 0
    prediction = prediction[:, coords_mask]
    gt_coords = gt_coords[:, coords_mask]
    loss = torch.norm(prediction - gt_coords, dim=0)
    loss_l1 = loss[loss <= cut]
    loss_sqrt = loss[loss > cut]
    loss_sqrt = torch.sqrt(cut * loss_sqrt)
    robust_loss = (loss_l1.sum() + loss_sqrt.sum()) / float(loss.size(0))
    robust_loss.backward()
    return robust_loss, p.grad


def make_batch(B, H, W, missing, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    gt = torch.randn((B, 3, H, W), device="cuda", generator=g) * 20.0
    gt[(torch.rand((B, 1, H, W), device="cuda", generator=g) < missing).expand(B, 3, H, W)] = 0.0
    pred = gt + torch.randn((B, 3, H, W), device="cuda", generator=g) * 40.0
    return pred, gt


def gpu_facts():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        smi = r.stdout.strip().splitlines()[torch.cuda.current_device()] if r.returncode == 0 else r.stderr.strip()
    except Exception as e:  # noqa: BLE001
        smi = f"nvidia-smi unavailable ({e})"
    return torch.cuda.get_device_name(), smi


def copy_bandwidth():
    """Device-to-device copy of 2 GiB (read + write), GB/s: what plain streaming reaches on this card right now."""
    a = torch.empty(2 ** 29, device="cuda")
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    return 2 * a.numel() * 4 * 10 / (e0.elapsed_time(e1) * 1e-3) / 1e9


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    opt = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    name, smi = gpu_facts()
    peak, src = HBM_PEAK_DESIGN, "DESIGN.md section 4"
    try:
        peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
        src = "MEASURED_PEAKS.json"
    except Exception:  # noqa: BLE001
        pass
    print(f"GPU: {name}; nvidia-smi name, power.limit, clocks.max.sm: {smi}")
    print(f"HBM peak used: {peak:.1f} GB/s ({src}); torch device-to-device copy in this run: {copy_bandwidth():.1f} GB/s")
    print(f"bytes per cell: {BYTES_PER_CELL} (24 read + 12 written); cut = {CUT}")
    ctx = api.context()
    for (H, W) in [(60, 80), (480, 640)]:
        for B in [1, 8, 64, 256]:
            for kind, missing in [("dense", 0.03), ("sparse", 0.95)]:
                ws = B * H * W * BYTES_PER_CELL
                copies = max(1, -(-3 * L2_BYTES // ws))
                if copies <= 64:
                    sets = [make_batch(B, H, W, missing, 17 + i) for i in range(copies)]
                else:   # many small batches: slices of one pool
                    pool_p, pool_g = make_batch(B * copies, H, W, missing, 17)
                    sets = [(pool_p[i * B:(i + 1) * B], pool_g[i * B:(i + 1) * B]) for i in range(copies)]
                grads = [torch.empty_like(p) for p, _ in sets]
                ms, wall = [], []
                for it in range(opt.reps + 5):
                    p, g = sets[it % len(sets)]
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    api.init_loss(p, g, CUT, outGradients=grads[it % len(sets)])
                    wall.append((time.perf_counter() - t0) * 1e3)
                    ms.append(ctx.stats()["ms_score"])
                ms = sorted(ms[5:])[len(ms[5:]) // 2]
                wl = sorted(wall[5:])[len(wall[5:]) // 2]
                nbytes = B * H * W * BYTES_PER_CELL
                line = (f"{H}x{W} B={B:4d} {kind:6s}: kernel {ms * 1e3:8.1f} us  {nbytes / ms / 1e6:8.1f} GB/s "
                        f"({nbytes / ms / 1e6 / peak:.2f} of peak)  call {wl * 1e3:8.1f} us  "
                        f"[{len(sets)} input sets rotated, {len(sets) * ws / 2 ** 20:.0f} MB]")
                # the torch op sequence on the same inputs, one image after another (up to 16 per timing)
                p, g = sets[0]
                nimg = min(B, 16)
                for b in range(min(nimg, 3)):
                    torch_ref(p[b:b + 1], g[b:b + 1], CUT)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for b in range(nimg):
                    rl, _ = torch_ref(p[b:b + 1], g[b:b + 1], CUT)
                torch.cuda.synchronize()
                tt = (time.perf_counter() - t0) / nimg * 1e3
                mine = api.init_loss(p[nimg - 1:nimg], g[nimg - 1:nimg], CUT)[0][0]
                assert abs(rl.item() - mine) < 1e-4 * abs(rl.item()), (rl.item(), mine)
                line += f"  | torch ops + autograd: {tt * 1e3:8.1f} us per image ({B * tt * 1e3:10.1f} us for B images)"
                print(line, flush=True)
                del sets, grads, p, g


if __name__ == "__main__":
    main()
