"""Writes tests/golden/ref_pin/compiled_reference.npz: what the reference's OWN compiled code (oracle/_ref/esac_ref, built by
oracle/build_ref.py from the unmodified reference sources on the real OpenCV of the cv2 wheel) returns for every call
tests/test_ref_pin.py compares the oracle with.  The scenes are regenerated from the test's make_scene() arguments; the
fixture stores a checksum of each so that a drift of make_scene is caught instead of compared against.

Needs the reference sources to build oracle/_ref.  Run:  python tests/golden/make_ref_pin_golden.py
"""
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
from esac_b200.synth import make_scene  # noqa: E402
from oracle.build_ref import load_ref  # noqa: E402
import test_ref_pin as T  # noqa: E402


def forward(R, sc, seed=1305):
    R.force_init(seed)
    out = torch.zeros(4, 4)
    e = R.forward(torch.from_numpy(sc.coords), torch.from_numpy(sc.assign), out, *sc.params)
    return e, out.numpy().copy()


def backward(R, sc, gt, loss_args, start, seed=1305):
    R.force_init(seed)
    g = torch.full(sc.coords.shape, float(start))
    loss = R.backward(torch.from_numpy(sc.coords), g, torch.from_numpy(sc.assign), torch.from_numpy(gt), *loss_args, *sc.params)
    return loss, g.numpy().copy()


def record(R) -> dict:
    z = {}

    def scene(key, kw):
        sc = make_scene(**kw)
        z[f"{key}/coords_sum"] = sc.coords.astype(np.float64).sum()
        return sc

    # thread_rand.cpp:34-43,68-71: generator 0 after force_init
    R.force_init(T.STREAM_SEED)
    z["stream/draws"] = np.array([[R.irand(0, m, 0) for _ in range(T.STREAM_DRAWS)] for m in T.STREAM_EXC_MAX], np.int64)
    R.force_init(T.STREAM_SEED_2)
    z["stream/draws_3_11"] = np.array([R.irand(3, 11, 0) for _ in range(T.STREAM_DRAWS_2)], np.int64)

    for name, kw in T.CASES.items():
        sc = scene(name, kw)
        z[f"{name}/expert"], z[f"{name}/pose"] = forward(R, sc)
        z[f"{name}/loss"], z[f"{name}/grads"] = backward(R, sc, sc.gt_pose, T.LOSS_ARGS, T.GRAD_START)

    sc = scene("loss_cut", T.LOSS_CUT_SCENE)
    gt = T.wrong_ground_truth(sc)
    for i, loss_args in enumerate(T.LOSS_CUT_ARGS):
        z[f"loss_cut/{i}/loss"], z[f"loss_cut/{i}/grads"] = backward(R, sc, gt, loss_args, 0.0)

    sc = scene("persist", T.PERSIST_SCENE)
    R.force_init(1305)
    for i in range(2):  # no force_init in between: the second call continues the stream
        out = torch.zeros(4, 4)
        z[f"persist/{i}/expert"] = R.forward(torch.from_numpy(sc.coords), torch.from_numpy(sc.assign), out, *sc.params)
        z[f"persist/{i}/pose"] = out.numpy().copy()

    sc = scene("native", T.NATIVE_SCENE)
    for native in (False, True):
        R.set_native_project(native)
        z[f"native/{int(native)}/expert"], z[f"native/{int(native)}/pose"] = forward(R, sc)
    R.set_native_project(False)

    sc = scene("openmp", T.OPENMP_SCENE)
    R.set_num_threads(T.OPENMP_THREADS)
    try:
        z["openmp/expert"], z["openmp/pose"] = forward(R, sc)
    finally:
        R.set_num_threads(1)
    return z


if __name__ == "__main__":
    R = load_ref()
    assert R is not None, "oracle/_ref is not built and the reference sources are absent"
    R.set_num_threads(1)
    R.set_native_project(False)
    z = record(R)
    path = Path(__file__).resolve().parent / "ref_pin" / "compiled_reference.npz"
    np.savez_compressed(path, **{k: np.asarray(v) for k, v in z.items()})
    print(f"{path.name}: {len(z)} arrays, {path.stat().st_size} bytes")
