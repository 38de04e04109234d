"""Pins the oracle to the reference's OWN compiled code.

tests/golden/ref_pin/compiled_reference.npz holds what oracle/_ref/esac_ref -- the unmodified reference esac.cpp and
thread_rand.cpp (+ its headers) compiled against oracle/ref_shim/opencv2/opencv.hpp, whose solvePnP / projectPoints /
Rodrigues / Mat::inv are executed by the real OpenCV inside the cv2 wheel (oracle/build_ref.py) -- returned for the calls
below (tests/golden/make_ref_pin_golden.py).  With one OpenMP thread the reference consumes one std::mt19937 stream in a
fixed order; oracle.esac_oracle.ThreadRandStream reproduces that stream, so both see identical minimal sets and every
output of esac_forward / esac_backward can be compared.
"""
from pathlib import Path

import numpy as np
import pytest

from esac_b200.synth import make_scene, pose_error
from oracle import esac_oracle as O

GOLD = Path(__file__).resolve().parent / "golden" / "ref_pin" / "compiled_reference.npz"

STREAM_SEED, STREAM_EXC_MAX, STREAM_DRAWS = 1305, (79, 59, 639, 479, 2, 3_000_000_000 // 2, 7), 300
STREAM_SEED_2, STREAM_DRAWS_2 = 77, 50
CASES = {
    "c1_60x80": dict(E=1, H=60, W=80, M=64, sub=8, seed=3),
    "ensemble3_shift": dict(E=3, H=30, W=40, M=32, sub=8, seed=3, shiftX=3, shiftY=-2),
    "world_scale": dict(E=2, H=24, W=32, M=24, sub=8, seed=3, outdoor=True, world_offset=700.0),
    "portrait_odd": dict(E=2, H=40, W=27, M=24, sub=8, seed=4),
}
LOSS_ARGS = (1.0, 100.0, 100.0)
GRAD_START = 0.25  # esac_backward accumulates into the caller's tensor: start from a non-zero one
LOSS_CUT_SCENE = dict(E=2, H=24, W=32, M=24, sub=8, seed=9)
LOSS_CUT_ARGS = ((1.0, 100.0, 5.0), (0.5, 10.0, 1000.0))
PERSIST_SCENE = dict(E=1, H=24, W=32, M=16, sub=8, seed=11)
NATIVE_SCENE = dict(E=2, H=30, W=40, M=32, sub=8, seed=5, outdoor=True, world_offset=300.0)
OPENMP_SCENE = dict(E=2, H=30, W=40, M=32, sub=8, seed=6, noise=0.0, outlier_frac=0.2)
OPENMP_THREADS = 4


def wrong_ground_truth(sc):
    gt = sc.gt_pose.copy()
    gt[:3, 3] += np.array([3.0, -2.0, 1.0], np.float32)
    return gt


@pytest.fixture(scope="module")
def ref():
    return np.load(GOLD)


def scene(ref, key, kw):
    """The scene the fixture was recorded on (checksum of the maps: make_scene must still regenerate it)."""
    sc = make_scene(**kw)
    want = float(ref[f"{key}/coords_sum"])
    assert abs(sc.coords.astype(np.float64).sum() - want) <= 1e-9 * abs(want), "make_scene no longer regenerates " + key
    return sc


def test_thread_rand_stream_is_the_references(ref):
    """thread_rand.cpp:34-43,68-71 on generator 0 == ThreadRandStream (mt19937 + libstdc++ uniform_int_distribution)."""
    mt = O.ThreadRandStream(STREAM_SEED)
    for exc_max, a in zip(STREAM_EXC_MAX, ref["stream/draws"].tolist()):
        b = [mt.irand(0, exc_max) for _ in range(STREAM_DRAWS)]
        assert a == b
        assert max(a) <= exc_max - 1 and min(a) >= 0
    mt = O.ThreadRandStream(STREAM_SEED_2)
    assert ref["stream/draws_3_11"].tolist() == [mt.irand(3, 11) for _ in range(STREAM_DRAWS_2)]


@pytest.mark.parametrize("name", list(CASES))
def test_forward_and_backward_equal_the_compiled_reference(ref, name):
    sc = scene(ref, name, CASES[name])
    # forward: esac.cpp:64-190
    mine = np.zeros((4, 4), np.float32)
    e_or = O.forward(sc.coords, sc.assign, mine, *sc.params, mt=O.ThreadRandStream(1305))
    assert int(ref[f"{name}/expert"]) == e_or
    assert np.abs(ref[f"{name}/pose"] - mine).max() <= 1e-6  # observed: bit-identical
    # backward: esac.cpp:213-511
    l_ref, g_ref = float(ref[f"{name}/loss"]), ref[f"{name}/grads"]
    g_or = np.full(sc.coords.shape, GRAD_START, np.float32)
    l_or = O.backward(sc.coords, g_or, sc.assign, sc.gt_pose, *LOSS_ARGS, *sc.params, mt=O.ThreadRandStream(1305))
    assert abs(l_ref - l_or) <= 1e-9 * max(1.0, abs(l_ref))
    scale = np.abs(g_or - GRAD_START).max()
    assert scale > 0
    assert np.abs(g_ref - g_or).max() <= 1e-6 * scale  # observed: <= 3e-9


def test_loss_cut_and_weights_equal_the_compiled_reference(ref):
    """The cut branch (esac_loss.h:78-80 vs :133-137,202-203 -- the sqrt(cut*loss) / 0.5/sqrt(loss) mismatch) and
    non-default weights, on a scene whose poses are far from a deliberately wrong ground truth."""
    sc = scene(ref, "loss_cut", LOSS_CUT_SCENE)
    gt = wrong_ground_truth(sc)
    for i, (w_rot, w_trans, cut) in enumerate(LOSS_CUT_ARGS):
        l_ref, g_ref = float(ref[f"loss_cut/{i}/loss"]), ref[f"loss_cut/{i}/grads"]
        g_or = np.zeros_like(sc.coords)
        l_or = O.backward(sc.coords, g_or, sc.assign, gt, w_rot, w_trans, cut, *sc.params, mt=O.ThreadRandStream(1305))
        assert abs(l_ref - l_or) <= 1e-9 * max(1.0, abs(l_ref))
        assert np.abs(g_ref - g_or).max() <= 1e-6 * max(np.abs(g_or).max(), 1e-30)


def test_stream_state_persists_across_calls(ref):
    """thread_rand.cpp:4-5: static generators -- a second call continues the stream; so does the oracle's object."""
    sc = scene(ref, "persist", PERSIST_SCENE)
    mt = O.ThreadRandStream(1305)
    for i in range(2):
        mine = np.zeros((4, 4), np.float32)
        e = O.forward(sc.coords, sc.assign, mine, *sc.params, mt=mt)
        assert e == int(ref[f"persist/{i}/expert"])
        assert np.abs(ref[f"persist/{i}/pose"] - mine).max() <= 1e-6


def test_native_projection_of_the_shim_is_bit_identical(ref):
    """The timing-only fast path of the shim (projectPoints without Jacobian as a native loop) changes nothing; both
    runs of the reference equal the oracle."""
    sc = scene(ref, "native", NATIVE_SCENE)
    outs = [(int(ref[f"native/{n}/expert"]), ref[f"native/{n}/pose"]) for n in (0, 1)]
    assert outs[0][0] == outs[1][0] and np.array_equal(outs[0][1], outs[1][1])
    mine = np.zeros((4, 4), np.float32)
    e = O.forward(sc.coords, sc.assign, mine, *sc.params, mt=O.ThreadRandStream(1305))
    assert e == outs[0][0] and np.abs(outs[0][1] - mine).max() <= 1e-6


def test_openmp_threads_do_not_deadlock_and_find_the_pose(ref):
    """More than one OpenMP thread: the sample stream is schedule-dependent (not comparable), the estimate is not: the
    reference found the pose, and the oracle finds the same expert and a pose as close to it."""
    sc = scene(ref, "openmp", OPENMP_SCENE)
    e, pose = int(ref["openmp/expert"]), ref["openmp/pose"]
    rot, trans = pose_error(pose, sc.gt_pose)
    assert e == sc.gt_expert and rot < 0.05 and trans < 0.01
    mine = np.zeros((4, 4), np.float32)
    assert O.forward(sc.coords, sc.assign, mine, *sc.params, mt=O.ThreadRandStream(1305)) == e
    rot, trans = pose_error(mine, pose)
    assert rot < 0.05 and trans < 0.01
