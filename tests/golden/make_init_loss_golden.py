"""Writes tests/golden/init_loss/literal_f32.npz: the loss and gradient that the reference's OWN loss block of
init_expert.py (util.assert_size through the division, read from the reference sources and executed as they stand, with
the reference's util module) returns in float32 on the cases of tests/test_init_loss_oracle.golden_cases().
tests/test_init_loss_oracle.py compares oracle/init_loss_oracle.py against it.

Needs the reference sources.  Run:  python tests/golden/make_init_loss_golden.py [reference code directory]
"""
import sys
from pathlib import Path
from types import SimpleNamespace

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
import test_init_loss_oracle as T  # noqa: E402


def loss_block(code_dir: Path) -> str:
    """The lines of init_expert.py from `util.assert_size` up to the robust loss, dedented."""
    lines = (code_dir / "init_expert.py").read_text().splitlines()
    start = next(i for i, l in enumerate(lines) if "util.assert_size(prediction, gt_coords)" in l)
    end = next(i for i, l in enumerate(lines) if l.strip().startswith("robust_loss ="))
    block = [l.strip() for l in lines[start:end + 1]]
    return "\n".join(l for l in block if l and not l.startswith("#"))


def main():
    code_dir = Path(sys.argv[1] if len(sys.argv) > 1 else "/root/reference/code")
    sys.path.insert(0, str(code_dir))
    import util  # the reference's util.py
    src = loss_block(code_dir)
    print(src)
    out = {}
    for name, (pred, gt, cut) in T.golden_cases().items():
        p = torch.from_numpy(pred.copy()).requires_grad_(True)
        ns = {"util": util, "torch": torch, "opt": SimpleNamespace(cutloss=cut), "prediction": p,
              "gt_coords": torch.from_numpy(gt.copy())}
        exec(src, ns)
        ns["robust_loss"].backward()
        out[name + "/pred"] = pred
        out[name + "/gt"] = gt
        out[name + "/loss"] = np.float32(ns["robust_loss"].item())
        out[name + "/grad"] = p.grad[0].numpy().copy()
        print(f"{name}: loss {out[name + '/loss']}")
    dst = ROOT / "tests" / "golden" / "init_loss" / "literal_f32.npz"
    dst.parent.mkdir(exist_ok=True)
    np.savez_compressed(dst, **out)
    print(dst, dst.stat().st_size, "bytes")


if __name__ == "__main__":
    main()
