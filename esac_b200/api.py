"""Host-side mirror of the reference's `esac` extension module on top of libesac_b200.so.

`forward` / `backward` keep the positional signatures of esac_forward / esac_backward
(/root/reference/code/esac/esac.cpp:64-77, 213-230; bound at esac.cpp:513-516) so
train_esac.py:151-168 and test_esac.py:192-205 run unchanged with `import esac` resolving to the
top-level `esac.py` shim of this repository.  Tensors may be CPU tensors (what the reference's
callers pass) or CUDA tensors (no host round trip), or numpy arrays.

There is no CPU implementation behind this module: if libesac_b200.so is missing or no CUDA device is
visible, calls raise RuntimeError.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "libesac_b200.so"


class Stats(C.Structure):
    _fields_ = [("M", C.c_int), ("winner", C.c_int), ("n_contrib", C.c_int), ("refine_rounds", C.c_int),
                ("entropy", C.c_double), ("expected_loss", C.c_double),
                ("ms_h2d", C.c_float), ("ms_prep", C.c_float), ("ms_sample", C.c_float), ("ms_score", C.c_float),
                ("ms_select", C.c_float), ("ms_refine", C.c_float), ("ms_backward", C.c_float), ("ms_total", C.c_float),
                ("score_launches", C.c_int), ("kernel_launches", C.c_int),
                ("score_ppt", C.c_int), ("score_grid", C.c_int), ("refine_group", C.c_int)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


_lib = None
PACK_TAIL = 21  # doubles behind the M_pad scores of a shard's record (include/esac_b200.h)
EXCHANGE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_double), C.c_int)


def load_library() -> C.CDLL:
    """dlopen libesac_b200.so and declare the prototypes of include/esac_b200.h."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise RuntimeError(f"{LIB_PATH} is not built: run `python -m esac_b200.build` "
                           "(or __graft_entry__.build()); there is no CPU fallback")
    lib = C.CDLL(str(LIB_PATH))
    vp, i32, i64, f32, f64 = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_double
    lib.esacb200_create.argtypes = [i32, C.POINTER(vp)]
    lib.esacb200_create.restype = i32
    lib.esacb200_destroy.argtypes = [vp]
    lib.esacb200_destroy.restype = None
    lib.esacb200_last_error.argtypes = [vp]
    lib.esacb200_last_error.restype = C.c_char_p
    lib.esacb200_set_stream.argtypes = [vp, vp]
    lib.esacb200_set_seed.argtypes = [vp, C.c_uint64]
    lib.esacb200_set_option.argtypes = [vp, C.c_char_p, f64]
    lib.esacb200_inject_cells.argtypes = [vp, vp, i32, i32]
    cam = [i32, i32, f32, f32, f32, f32, f32, f32, f32, i32]  # shiftX .. subSampling
    lib.esacb200_forward.argtypes = [vp, vp, i32, i32, i32, vp, i64, i32, vp] + cam + [C.POINTER(i32)]
    lib.esacb200_backward.argtypes = [vp, vp, vp, i32, i32, i32, vp, i64, i32, vp, f32, f32, f32] + cam + [C.POINTER(f64)]
    lib.esacb200_forward_batch.argtypes = [vp, i32, vp, i32, i32, i32, vp, i64, i32, vp] + cam + [vp]
    lib.esacb200_forward_batch.restype = i32
    lib.esacb200_forward_pack.argtypes = [vp, vp, i32, i32, i32, vp, i64, i32, i32] + cam + [i32, vp]
    lib.esacb200_forward_pack.restype = i32
    lib.esacb200_nccl_unique_id.argtypes = [vp]
    lib.esacb200_nccl_unique_id.restype = i32
    lib.esacb200_comm_init.argtypes = [vp, i32, i32, vp]
    lib.esacb200_comm_init.restype = i32
    lib.esacb200_comm_destroy.argtypes = [vp]
    lib.esacb200_comm_destroy.restype = i32
    lib.esacb200_forward_sharded.argtypes = [vp, vp, i32, i32, i32, vp, i64, i32, i32, vp] + cam + [i32, C.POINTER(i32)]
    lib.esacb200_forward_sharded.restype = i32
    lib.esacb200_backward_sharded_nccl.argtypes = [vp, vp, vp, i32, i32, i32, vp, i64, i32, vp, f32, f32, f32] + cam + [i32, C.POINTER(f64)]
    lib.esacb200_backward_sharded_nccl.restype = i32
    lib.esacb200_backward_batch.argtypes = ([vp, i32, vp, vp, i32, i32, i32, vp, i64, i32, vp, f32, f32, f32, vp, vp] + cam[2:] +
                                             [vp])
    lib.esacb200_backward_batch.restype = i32
    lib.esacb200_assign_hypotheses.argtypes = [vp, i32, i32, i32, vp, i32, i32, C.c_uint64, vp, vp]
    lib.esacb200_assign_hypotheses.restype = i32
    lib.esacb200_reproj_loss.argtypes = [vp, i32, vp, vp, i32, i32, vp, vp, vp, f32, f32, f32, i32, f32, f32, f32, vp]
    lib.esacb200_reproj_loss.restype = i32
    lib.esacb200_init_loss.argtypes = [vp, i32, vp, i32, i32, vp, i32, i32, vp, f32, vp, vp]
    lib.esacb200_init_loss.restype = i32
    lib.esacb200_backward_sharded.argtypes = ([vp, vp, vp, i32, i32, i32, vp, i64, i32, vp, f32, f32, f32] + cam +
                                               [EXCHANGE_FN, vp, C.POINTER(f64)])
    lib.esacb200_backward_sharded.restype = i32
    lib.esacb200_score_poses.argtypes = [vp, vp, i32, i32, i32, vp, i64, i32, vp] + cam + [vp]
    lib.esacb200_refine_poses.argtypes = [vp, vp, i32, i32, i32, vp, i64, i32, vp, i32, i32, f32, f32, f32, f32, f32, i32, vp, vp]
    lib.esacb200_get_refine_profile.argtypes = [vp, vp]
    lib.esacb200_get_refine_profile.restype = i32
    lib.esacb200_get_sample_trace.argtypes = [vp, vp]
    lib.esacb200_get_sample_trace.restype = i32
    lib.esacb200_get_sample_profile.argtypes = [vp, vp]
    lib.esacb200_get_sample_profile.restype = i32
    lib.esacb200_get_stats.argtypes = [vp, C.POINTER(Stats)]
    lib.esacb200_get_hypotheses.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    lib.esacb200_device_info.argtypes = [vp, C.POINTER(i32), C.c_char_p, i32]
    lib.esacb200_copy_last_scores.argtypes = [vp, vp, i32]
    lib.esacb200_copy_last_scores.restype = i32
    for name in ("set_stream", "set_seed", "set_option", "inject_cells", "forward", "backward", "score_poses",
                 "refine_poses", "get_stats", "get_hypotheses", "device_info"):
        getattr(lib, "esacb200_" + name).restype = i32
    # host test hooks (include/esac_b200_testhooks.h)
    lib.esacb200_host_rodrigues.argtypes = [vp, vp, vp]
    lib.esacb200_host_rodrigues.restype = None
    lib.esacb200_host_rodrigues_inv.argtypes = [vp, vp]
    lib.esacb200_host_rodrigues_inv.restype = None
    lib.esacb200_host_p3p_all.argtypes = [vp, vp, vp, vp]
    lib.esacb200_host_p3p_all.restype = i32
    lib.esacb200_host_p3p_pose.argtypes = [vp, vp, f32, f32, f32, f32, vp, C.POINTER(i32)]
    lib.esacb200_host_p3p_pose.restype = i32
    lib.esacb200_host_try.argtypes = [vp, vp, f32, f32, f32, f32, f32, C.POINTER(i32), C.POINTER(i32)]
    lib.esacb200_host_try.restype = None
    lib.esacb200_host_try_verdict.argtypes = [vp, vp, f32, f32, f32, f32, C.POINTER(i32), vp]
    lib.esacb200_host_try_verdict.restype = None
    lib.esacb200_host_project.argtypes = [vp, f32, f32, f32, vp, vp, vp, vp]
    lib.esacb200_host_project.restype = None
    lib.esacb200_host_loss.argtypes = [vp, vp, f64, f64, f64]
    lib.esacb200_host_loss.restype = f64
    lib.esacb200_host_dloss.argtypes = [vp, vp, f64, f64, f64, vp]
    lib.esacb200_host_dloss.restype = None
    lib.esacb200_host_pose2trans.argtypes = [vp, vp]
    lib.esacb200_host_pose2trans.restype = None
    lib.esacb200_host_trans2pose.argtypes = [vp, vp]
    lib.esacb200_host_trans2pose.restype = None
    lib.esacb200_host_dprojectdobj.argtypes = [vp, vp, vp, f32, f32, f32, f32, vp]
    lib.esacb200_host_dprojectdobj.restype = None
    lib.esacb200_host_pinv6.argtypes = [vp, vp]
    lib.esacb200_host_pinv6.restype = None
    lib.esacb200_host_draw_cells.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, i32, i32, vp]
    lib.esacb200_host_draw_cells.restype = None
    _lib = lib
    return lib


# ------------------------------------------------------------------------------------------------
# contexts (one per device) -- the analogue of the reference's static ThreadRand state
# ------------------------------------------------------------------------------------------------
class Context:
    def __init__(self, device: int = 0):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.esacb200_create(int(device), C.byref(h))
        if rc != 0:
            raise RuntimeError(f"esac_b200: cannot create a context on CUDA device {device} (status {rc}); "
                               "this implementation has no CPU path")
        self.handle = h
        self.device = int(device)
        self.comm_world, self.comm_rank = 1, 0

    def close(self):
        if getattr(self, "handle", None):
            self.lib.esacb200_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc: int):
        if rc != 0:
            msg = self.lib.esacb200_last_error(self.handle)
            raise RuntimeError(f"esac_b200 (status {rc}): {msg.decode() if msg else ''}")

    # additive API ------------------------------------------------------------------------------
    def set_seed(self, seed: int):
        self.check(self.lib.esacb200_set_seed(self.handle, C.c_uint64(seed & ((1 << 64) - 1))))

    def set_option(self, key: str, value: float):
        self.check(self.lib.esacb200_set_option(self.handle, key.encode(), float(value)))

    def set_stream(self, stream_ptr: int):
        self.check(self.lib.esacb200_set_stream(self.handle, C.c_void_p(stream_ptr or None)))

    def inject_cells(self, cells):
        if cells is None:
            self.check(self.lib.esacb200_inject_cells(self.handle, None, 0, 0))
            return
        cells = np.ascontiguousarray(cells, np.int32)
        assert cells.ndim == 4 and cells.shape[2:] == (4, 2), "cells must be [M, T, 4, 2] (x, y)"
        self.check(self.lib.esacb200_inject_cells(self.handle, cells.ctypes.data, cells.shape[0], cells.shape[1]))

    def stats(self) -> dict:
        s = Stats()
        self.check(self.lib.esacb200_get_stats(self.handle, C.byref(s)))
        return s.as_dict()

    def comm_init(self, world: int, rank: int, unique_id: bytes):
        """ncclCommInitRank inside the library (collective over all ranks); unique_id from nccl_unique_id() of rank 0."""
        buf = C.create_string_buffer(bytes(unique_id), 128)
        self.check(self.lib.esacb200_comm_init(self.handle, int(world), int(rank), buf))
        self.comm_world, self.comm_rank = int(world), int(rank)

    def comm_destroy(self):
        self.check(self.lib.esacb200_comm_destroy(self.handle))
        self.comm_world, self.comm_rank = 1, 0

    def refine_profile(self) -> np.ndarray:
        """Phase cycle counters of the last refinement (option "refine_profile" = 1), see include/esac_b200.h."""
        out = np.zeros(16, np.int64)
        self.check(self.lib.esacb200_get_refine_profile(self.handle, out.ctypes.data))
        return out

    def sample_profile(self) -> dict:
        out = np.zeros(8, np.int64)
        self.check(self.lib.esacb200_get_sample_profile(self.handle, out.ctypes.data))
        d = {"tries_prefiltered": int(out[0]), "survivors_judged": int(out[1]), "waves": int(out[2]),
             "left_to_tail": int(out[3]), "accepted_staged": int(out[4]), "lanes": int(out[5])}
        return d

    def sample_trace(self) -> np.ndarray:
        """[lane, wave, kernel (0 prefilter, 1 exact), (start, end)] in ns relative to the first stamp; -1 where nothing ran."""
        raw = np.zeros(512, np.uint64)
        self.check(self.lib.esacb200_get_sample_trace(self.handle, raw.ctypes.data))
        t = raw.reshape(4, 32, 2, 2)
        ran = t[..., 0] != np.uint64(0xFFFFFFFFFFFFFFFF)
        t0 = t[..., 0][ran].min() if ran.any() else np.uint64(0)
        out = np.full(t.shape, -1, np.int64)
        out[ran] = (t[ran] - t0).astype(np.int64)
        return out

    def copy_last_scores(self, dst):
        """dst: float64 torch tensor (CUDA or CPU) or numpy array of M elements; stream-ordered copy."""
        n = int(dst.numel()) if _is_torch(dst) else int(np.asarray(dst).size)
        ptr = dst.data_ptr() if _is_torch(dst) else np.asarray(dst).ctypes.data
        self.check(self.lib.esacb200_copy_last_scores(self.handle, ptr, n))

    def device_info(self) -> dict:
        n = C.c_int()
        buf = C.create_string_buffer(128)
        self.check(self.lib.esacb200_device_info(self.handle, C.byref(n), buf, 128))
        return {"sm_count": n.value, "name": buf.value.decode()}

    def hypotheses(self, losses: bool = False) -> dict:
        M = self.stats()["M"]
        out = {"poses": np.zeros((M, 6)), "cells": np.zeros((M, 4, 2), np.int32), "tries": np.zeros(M, np.int32),
               "scores": np.zeros(M), "probs": np.zeros(M), "refined": np.zeros((M, 6))}
        lo = np.zeros(M) if losses else None
        self.check(self.lib.esacb200_get_hypotheses(self.handle, out["poses"].ctypes.data, out["cells"].ctypes.data,
                                                    out["tries"].ctypes.data, out["scores"].ctypes.data,
                                                    out["probs"].ctypes.data, out["refined"].ctypes.data,
                                                    lo.ctypes.data if losses else None))
        if losses:
            out["losses"] = lo
        return out


_contexts: dict[int, Context] = {}


def context(device: int | None = None) -> Context:
    if device is None:
        device = 0
        try:
            import torch
            if torch.cuda.is_available():
                device = torch.cuda.current_device()
        except Exception:
            pass
    if device not in _contexts:
        _contexts[device] = Context(device)
    return _contexts[device]


# ------------------------------------------------------------------------------------------------
# tensor plumbing
# ------------------------------------------------------------------------------------------------
_TORCH_NAMES = {"torch.float32": "Float", "torch.float64": "Double", "torch.float16": "Half", "torch.int64": "Long",
                "torch.int32": "Int", "torch.bfloat16": "BFloat16", "torch.uint8": "Byte", "torch.int16": "Short",
                "torch.int8": "Char", "torch.bool": "Bool"}
_NP_NAMES = {"float32": "Float", "float64": "Double", "float16": "Half", "int64": "Long", "int32": "Int"}


def _is_torch(t) -> bool:
    return type(t).__module__.startswith("torch")


def _dtype_name(t) -> str:
    if _is_torch(t):
        return _TORCH_NAMES.get(str(t.dtype), str(t.dtype))
    return _NP_NAMES.get(str(np.asarray(t).dtype), str(np.asarray(t).dtype))


def _check(t, want: str, rank: int, what: str):
    """Same failure mode as at::Tensor::accessor<T, N>() in the reference (esac.cpp:80-84): RuntimeError."""
    have = _dtype_name(t)
    if have != want:
        raise RuntimeError(f"expected scalar type {want} but found {have} ({what})")
    nd = t.dim() if _is_torch(t) else np.asarray(t).ndim
    if nd != rank:
        raise RuntimeError(f"expected {rank} dims but tensor has {nd} ({what})")


class _Arg:
    """Pointer view of a tensor argument; keeps temporaries alive and writes results back."""

    def __init__(self, t, writable=False, need_contig=True):
        self.orig = t
        self.writable = writable
        self.tmp = None
        if _is_torch(t):
            self.is_cuda = t.is_cuda
            self.device = t.device.index if t.is_cuda else None
            v = t
            if need_contig and not t.is_contiguous():
                v = t.contiguous()
                self.tmp = v
            self.view = v
            self.ptr = v.data_ptr()
        else:
            a = np.asarray(t)
            self.is_cuda = False
            self.device = None
            v = a
            if need_contig and not a.flags["C_CONTIGUOUS"]:
                v = np.ascontiguousarray(a)
                self.tmp = v
            self.view = v
            self.ptr = v.ctypes.data

    def finish(self):
        if self.writable and self.tmp is not None:
            if _is_torch(self.orig):
                self.orig.copy_(self.tmp)
            else:
                np.copyto(np.asarray(self.orig), self.tmp)


def _assign_arg(t):
    """hypAssignment: int64 [M], any stride (stride 0 for expert.expand(), test_esac.py:173)."""
    if _is_torch(t):
        M = int(t.shape[0])
        stride = int(t.stride(0)) if M > 0 else 1
        return t.data_ptr(), stride, M, (t.device.index if t.is_cuda else None), t
    a = np.asarray(t)
    M = int(a.shape[0])
    stride = int(a.strides[0] // a.itemsize) if M > 0 else 1
    return a.ctypes.data, stride, M, None, a


_CUDA_STREAM_LEGACY = 0x1


def _pick_ctx(*devices) -> Context:
    devs = {d for d in devices if d is not None}
    if len(devs) > 1:
        raise RuntimeError(f"esac_b200: tensors live on different CUDA devices {sorted(devs)}")
    ctx = context(next(iter(devs)) if devs else None)
    stream = 0
    if devs:
        # CUDA tensors: run on torch's current stream so that the call is ordered after whatever produced them.  torch
        # reports its default stream as handle 0, which the C ABI reads as "use the context's own stream"; the legacy
        # default stream has the explicit handle cudaStreamLegacy = 0x1.
        import torch
        stream = torch.cuda.current_stream(ctx.device).cuda_stream or _CUDA_STREAM_LEGACY
    ctx.set_stream(stream)
    return ctx


def _pick_ctx_host(device: int | None) -> Context:
    """Context for host-only arguments on an explicit device (sharded entry points: one process per GPU)."""
    ctx = context(device)
    ctx.set_stream(0)
    return ctx


# ------------------------------------------------------------------------------------------------
# the reference's two entry points
# ------------------------------------------------------------------------------------------------
def forward(sceneCoordinates, hypAssignment, outPose, shiftX, shiftY, focalLength, ppointX, ppointY,
            inlierThreshold, inlierAlpha, inlierBeta, maxReproj, subSampling) -> int:
    """esac.forward (esac.cpp:64-190): writes the estimated camera pose into outPose (4x4, in place) and
    returns the index of the winning expert."""
    _check(sceneCoordinates, "Float", 4, "sceneCoordinates")
    _check(hypAssignment, "Long", 1, "hypAssignment")
    _check(outPose, "Float", 2, "outPose")
    if tuple(sceneCoordinates.shape)[1] != 3:
        raise RuntimeError("sceneCoordinates must be [E, 3, H, W]")
    if tuple(outPose.shape) != (4, 4):
        raise RuntimeError("outPose must be [4, 4]")
    co = _Arg(sceneCoordinates)
    op = _Arg(outPose, writable=True)
    aptr, astride, M, adev, _keep = _assign_arg(hypAssignment)
    ctx = _pick_ctx(co.device, op.device, adev)
    E, _, H, W = (int(s) for s in sceneCoordinates.shape)
    expert = C.c_int(-1)
    ctx.check(ctx.lib.esacb200_forward(ctx.handle, co.ptr, E, H, W, aptr, astride, M, op.ptr, int(shiftX), int(shiftY),
                                       float(focalLength), float(ppointX), float(ppointY), float(inlierThreshold),
                                       float(inlierAlpha), float(inlierBeta), float(maxReproj), int(subSampling),
                                       C.byref(expert)))
    op.finish()
    return int(expert.value)


def backward(sceneCoordinates, outGradients, hypAssignment, gtPose, wLossRot, wLossTrans, lossCut, shiftX, shiftY,
             focalLength, ppointX, ppointY, inlierThreshold, inlierAlpha, inlierBeta, maxReproj, subSampling) -> float:
    """esac.backward (esac.cpp:213-511): accumulates d(expected pose loss)/d(sceneCoordinates) into
    outGradients (in place, +=) and returns the expected loss."""
    _check(sceneCoordinates, "Float", 4, "sceneCoordinates")
    _check(outGradients, "Float", 4, "outGradients")
    _check(hypAssignment, "Long", 1, "hypAssignment")
    _check(gtPose, "Float", 2, "gtPose")
    if tuple(sceneCoordinates.shape)[1] != 3 or tuple(outGradients.shape) != tuple(sceneCoordinates.shape):
        raise RuntimeError("sceneCoordinates / outGradients must both be [E, 3, H, W]")
    if tuple(gtPose.shape) != (4, 4):
        raise RuntimeError("gtPose must be [4, 4]")
    co = _Arg(sceneCoordinates)
    gr = _Arg(outGradients, writable=True)
    gt = _Arg(gtPose)
    aptr, astride, M, adev, _keep = _assign_arg(hypAssignment)
    ctx = _pick_ctx(co.device, gr.device, gt.device, adev)
    E, _, H, W = (int(s) for s in sceneCoordinates.shape)
    loss = C.c_double(0.0)
    ctx.check(ctx.lib.esacb200_backward(ctx.handle, co.ptr, gr.ptr, E, H, W, aptr, astride, M, gt.ptr, float(wLossRot),
                                        float(wLossTrans), float(lossCut), int(shiftX), int(shiftY), float(focalLength),
                                        float(ppointX), float(ppointY), float(inlierThreshold), float(inlierAlpha),
                                        float(inlierBeta), float(maxReproj), int(subSampling), C.byref(loss)))
    gr.finish()
    return float(loss.value)


def backward_sharded(sceneCoordinates, outGradients, hypAssignment, gtPose, wLossRot, wLossTrans, lossCut, shiftX, shiftY,
                     focalLength, ppointX, ppointY, inlierThreshold, inlierAlpha, inlierBeta, maxReproj, subSampling,
                     exchange, hyp_offset=0) -> float:
    """esac.backward on this rank's shard of the experts / hypotheses.  `exchange(phase, values) -> list` performs the two
    cross-rank reductions (see include/esac_b200.h); returns the GLOBAL expected loss."""
    _check(sceneCoordinates, "Float", 4, "sceneCoordinates")
    _check(outGradients, "Float", 4, "outGradients")
    _check(hypAssignment, "Long", 1, "hypAssignment")
    _check(gtPose, "Float", 2, "gtPose")
    co = _Arg(sceneCoordinates)
    gr = _Arg(outGradients, writable=True)
    gt = _Arg(gtPose)
    aptr, astride, M, adev, _keep = _assign_arg(hypAssignment)
    ctx = _pick_ctx(co.device, gr.device, gt.device, adev)
    E, _, H, W = (int(s) for s in sceneCoordinates.shape)
    err = []

    def _cb(user, phase, values, n):
        try:
            out = exchange(int(phase), [values[i] for i in range(n)])
            for i in range(n):
                values[i] = float(out[i])
            return 0
        except Exception as e:  # never let an exception cross the C boundary
            err.append(e)
            return 1

    cb = EXCHANGE_FN(_cb)
    loss = C.c_double(0.0)
    ctx.set_option("hyp_offset", hyp_offset)
    try:
        rc = ctx.lib.esacb200_backward_sharded(ctx.handle, co.ptr, gr.ptr, E, H, W, aptr, astride, M, gt.ptr, float(wLossRot),
                                               float(wLossTrans), float(lossCut), int(shiftX), int(shiftY), float(focalLength),
                                               float(ppointX), float(ppointY), float(inlierThreshold), float(inlierAlpha),
                                               float(inlierBeta), float(maxReproj), int(subSampling), cb, None, C.byref(loss))
    finally:
        ctx.set_option("hyp_offset", 0)
    if err:
        raise err[0]
    ctx.check(rc)
    gr.finish()
    return float(loss.value)


# ------------------------------------------------------------------------------------------------
# additive entry points
# ------------------------------------------------------------------------------------------------
def forward_batch(sceneCoordinates, hypAssignment, outPoses, shiftX, shiftY, focalLength, ppointX, ppointY,
                  inlierThreshold, inlierAlpha, inlierBeta, maxReproj, subSampling) -> list:
    """esac.forward over a batch: sceneCoordinates [B,E,3,H,W] float32, hypAssignment [B,M] int64 (contiguous rows),
    outPoses [B,4,4] float32 written in place.  Returns the winning expert of every image.  One host synchronisation
    for the whole batch; host tensors (pinned) are copied on a second stream while the previous image computes."""
    _check(sceneCoordinates, "Float", 5, "sceneCoordinates")
    _check(hypAssignment, "Long", 2, "hypAssignment")
    _check(outPoses, "Float", 3, "outPoses")
    B, E, C3, H, W = (int(v) for v in sceneCoordinates.shape)
    if C3 != 3 or tuple(outPoses.shape) != (B, 4, 4) or int(hypAssignment.shape[0]) != B:
        raise RuntimeError("shapes must be [B,E,3,H,W], [B,M], [B,4,4]")
    co = _Arg(sceneCoordinates)
    op = _Arg(outPoses, writable=True)
    ha = _Arg(hypAssignment)
    M = int(hypAssignment.shape[1])
    ctx = _pick_ctx(co.device, op.device, ha.device)
    experts = (C.c_int * B)()
    ctx.check(ctx.lib.esacb200_forward_batch(ctx.handle, B, co.ptr, E, H, W, ha.ptr, 1, M, op.ptr, int(shiftX), int(shiftY),
                                             float(focalLength), float(ppointX), float(ppointY), float(inlierThreshold),
                                             float(inlierAlpha), float(inlierBeta), float(maxReproj), int(subSampling),
                                             experts))
    op.finish()
    return [int(e) for e in experts]


def backward_batch(sceneCoordinates, outGradients, hypAssignment, gtPoses, wLossRot, wLossTrans, lossCut, shiftX, shiftY,
                   focalLength, ppointX, ppointY, inlierThreshold, inlierAlpha, inlierBeta, maxReproj, subSampling) -> list:
    """esac.backward over a batch: sceneCoordinates / outGradients [B,E,3,H,W] float32 (gradients accumulated in place),
    hypAssignment [B,M] int64, gtPoses [B,4,4] float32 (camera->world), shiftX / shiftY an int or a sequence of B ints
    (train_esac.py:125 draws one shift per image).  Returns the expected loss of every image; equal, image by image, to B
    consecutive esac.backward calls on the same context."""
    _check(sceneCoordinates, "Float", 5, "sceneCoordinates")
    _check(outGradients, "Float", 5, "outGradients")
    _check(hypAssignment, "Long", 2, "hypAssignment")
    _check(gtPoses, "Float", 3, "gtPoses")
    B, E, C3, H, W = (int(v) for v in sceneCoordinates.shape)
    if (C3 != 3 or tuple(outGradients.shape) != tuple(sceneCoordinates.shape) or tuple(gtPoses.shape) != (B, 4, 4)
            or int(hypAssignment.shape[0]) != B):
        raise RuntimeError("shapes must be [B,E,3,H,W], [B,E,3,H,W], [B,M], [B,4,4]")
    co = _Arg(sceneCoordinates)
    og = _Arg(outGradients, writable=True)
    ha = _Arg(hypAssignment)
    gt = _Arg(gtPoses)
    M = int(hypAssignment.shape[1])

    def shifts(v):
        if isinstance(v, (int, float)):
            v = [int(v)] * B
        a = np.ascontiguousarray(np.asarray(v, dtype=np.int32).reshape(-1))
        if a.shape[0] != B:
            raise RuntimeError(f"shift must be an int or {B} ints")
        return a

    sx, sy = shifts(shiftX), shifts(shiftY)
    ctx = _pick_ctx(co.device, og.device, ha.device, gt.device)
    losses = np.zeros(B, np.float64)
    ctx.check(ctx.lib.esacb200_backward_batch(ctx.handle, B, co.ptr, og.ptr, E, H, W, ha.ptr, 1, M, gt.ptr, float(wLossRot),
                                              float(wLossTrans), float(lossCut), sx.ctypes.data, sy.ctypes.data,
                                              float(focalLength), float(ppointX), float(ppointY), float(inlierThreshold),
                                              float(inlierAlpha), float(inlierBeta), float(maxReproj), int(subSampling),
                                              losses.ctypes.data))
    og.finish()
    return [float(v) for v in losses]


def assign_hypotheses(gatingProbs, hypotheses: int, seed: int, maxExperts: int = -1, expertSelection: bool = False):
    """The callers' hypothesis assignment (util.clamp_probs + torch.multinomial(replacement=True) + torch.histc,
    train_esac.py:130-140, test_esac.py:169-177) for a batch of gating outputs, on the device.  gatingProbs [B,E] float32
    (CPU, CUDA or numpy; need not be normalised).  Returns (e_hyps int64 [B,M], e_hyps_hist float32 [B,E]) of the same
    kind as the input.  A pure function of (seed, image, hypothesis); see oracle.esac_oracle.assign_hypotheses."""
    _check(gatingProbs, "Float", 2, "gatingProbs")
    B, E = (int(v) for v in gatingProbs.shape)
    M = int(hypotheses)
    gp = _Arg(gatingProbs)
    if _is_torch(gatingProbs):
        import torch
        assign = torch.empty((B, M), dtype=torch.int64, device=gatingProbs.device)
        hist = torch.empty((B, E), dtype=torch.float32, device=gatingProbs.device)
        ap, hp = assign.data_ptr(), hist.data_ptr()
    else:
        assign = np.empty((B, M), np.int64)
        hist = np.empty((B, E), np.float32)
        ap, hp = assign.ctypes.data, hist.ctypes.data
    ctx = _pick_ctx(gp.device)
    ctx.check(ctx.lib.esacb200_assign_hypotheses(ctx.handle, B, E, M, gp.ptr, int(maxExperts), int(bool(expertSelection)),
                                                 int(seed) & 0xFFFFFFFFFFFFFFFF, ap, hp))
    return assign, hist


def reproj_loss(prediction, gtPoses, focalLength, padX, padY, cutLoss, subSampling=8, ppointX=None, ppointY=None,
                outGradients=None, maxReproj=100.0, minDepth=0.1):
    """The robust reprojection loss of ref_expert.py:103-148 and, when outGradients is given, d loss / d prediction in the
    same pass (what `robust_loss.backward()` hands to the expert, ref_expert.py:150).  prediction [B,3,H,W] float32 (the
    reference has B = 1), gtPoses [B,4,4] float32 camera->world, padX / padY an int or B ints (the random shift),
    outGradients [B,3,H,W] float32 written in place (overwritten) or None.  The principal point defaults to the centre of
    the sub*W x sub*H image (ref_expert.py:118-119).  Returns the B losses."""
    _check(prediction, "Float", 4, "prediction")
    _check(gtPoses, "Float", 3, "gtPoses")
    B, C3, H, W = (int(v) for v in prediction.shape)
    if C3 != 3 or tuple(gtPoses.shape) != (B, 4, 4):
        raise RuntimeError("shapes must be [B,3,H,W] and [B,4,4]")
    pr = _Arg(prediction)
    gt = _Arg(gtPoses)
    og = None
    if outGradients is not None:
        _check(outGradients, "Float", 4, "outGradients")
        if tuple(outGradients.shape) != tuple(prediction.shape):
            raise RuntimeError("outGradients must have the shape of prediction")
        og = _Arg(outGradients, writable=True)

    def shifts(v):
        if isinstance(v, (int, float)):
            v = [int(v)] * B
        a = np.ascontiguousarray(np.asarray(v, dtype=np.int32).reshape(-1))
        if a.shape[0] != B:
            raise RuntimeError(f"pad must be an int or {B} ints")
        return a

    sx, sy = shifts(padX), shifts(padY)
    ppx = float(W * subSampling / 2 if ppointX is None else ppointX)
    ppy = float(H * subSampling / 2 if ppointY is None else ppointY)
    ctx = _pick_ctx(pr.device, gt.device, og.device if og else None)
    losses = np.zeros(B, np.float64)
    ctx.check(ctx.lib.esacb200_reproj_loss(ctx.handle, B, pr.ptr, og.ptr if og else None, H, W, gt.ptr, sx.ctypes.data,
                                           sy.ctypes.data, float(focalLength), ppx, ppy, int(subSampling), float(cutLoss),
                                           float(maxReproj), float(minDepth), losses.ctypes.data))
    if og:
        og.finish()
    return [float(v) for v in losses]


def init_loss(prediction, gtCoords, cutLoss, outGradients=None):
    """The scene-coordinate loss of init_expert.py:112-130 for a batch of images.  prediction [B,3,h,w] or [3,h,w] float32,
    gtCoords float32 of the same rank and batch; heights and widths may differ by one (both are cropped to the common
    top-left region, util.assert_size), by more is a RuntimeError.  Target cells whose three components are all zero do not
    count.  Returns [(loss, count)] per image: loss = robust sum / count (NaN for an image without a valid cell, as in the
    reference), count = number of valid cells.  outGradients (prediction's shape, float32) or None receives, overwritten,
    d(robust sum of image b) / d prediction -- the gradient of the per-image SUM; multiply image b by 1/count_b for the
    gradient of its loss (autograd.init_loss does).  CPU, CUDA tensors or numpy arrays; CUDA work runs on torch's current
    stream."""
    for t, what in ((prediction, "prediction"), (gtCoords, "gtCoords")):
        have = _dtype_name(t)
        if have != "Float":
            raise RuntimeError(f"expected scalar type Float but found {have} ({what})")
    ps, gs = tuple(int(v) for v in prediction.shape), tuple(int(v) for v in gtCoords.shape)
    if len(ps) not in (3, 4) or len(gs) != len(ps):
        raise RuntimeError(f"prediction and gtCoords must both be [3,h,w] or [B,3,h,w] (got {list(ps)} and {list(gs)})")
    if len(ps) == 3:
        ps, gs = (1,) + ps, (1,) + gs
    if ps[1] != 3 or gs[1] != 3:
        raise RuntimeError(f"prediction and gtCoords need 3 channels (got {ps[1]} and {gs[1]})")
    if ps[0] != gs[0]:
        raise RuntimeError(f"batch sizes differ: prediction {ps[0]}, gtCoords {gs[0]}")
    B = ps[0]
    pr = _Arg(prediction)
    gt = _Arg(gtCoords)
    og = None
    if outGradients is not None:
        if _dtype_name(outGradients) != "Float" or tuple(outGradients.shape) != tuple(prediction.shape):
            raise RuntimeError("outGradients must be float32 of prediction's shape")
        og = _Arg(outGradients, writable=True)
    ctx = _pick_ctx(pr.device, gt.device, og.device if og else None)
    sums = np.zeros(B, np.float64)
    counts = np.zeros(B, np.int64)
    ctx.check(ctx.lib.esacb200_init_loss(ctx.handle, B, pr.ptr, ps[2], ps[3], gt.ptr, gs[2], gs[3], og.ptr if og else None,
                                         float(cutLoss), sums.ctypes.data, counts.ctypes.data))
    if og:
        og.finish()
    return [(float(s) / int(c) if c else float("nan"), int(c)) for s, c in zip(sums, counts)]


def nccl_unique_id() -> bytes:
    """128-byte ncclUniqueId (call on one rank, distribute to the others, then Context.comm_init on every rank)."""
    buf = C.create_string_buffer(128)
    rc = load_library().esacb200_nccl_unique_id(buf)
    if rc != 0:
        raise RuntimeError(f"esac_b200: ncclGetUniqueId failed (status {rc}); is libnccl.so.2 loadable?")
    return buf.raw


def forward_pack(sceneCoordinates, hypAssignment, params, expert_offset: int, pack_out, M_pad: int | None = None):
    """The local half of a sharded forward, enqueued on the current CUDA stream without a host synchronisation
    (esacb200_forward_pack).  sceneCoordinates [E,3,H,W] / hypAssignment [M] are CUDA tensors, params the positional tail of
    esac.forward (shiftX .. subSampling), pack_out a CUDA float64 tensor of M_pad + 21 elements (see include/esac_b200.h);
    M_pad (default M) = the largest M of any shard."""
    _check(sceneCoordinates, "Float", 4, "sceneCoordinates")
    _check(hypAssignment, "Long", 1, "hypAssignment")
    if not (_is_torch(sceneCoordinates) and sceneCoordinates.is_cuda and hypAssignment.is_cuda and pack_out.is_cuda):
        raise RuntimeError("forward_pack takes CUDA tensors")
    co = _Arg(sceneCoordinates)
    aptr, astride, M, adev, _keep = _assign_arg(hypAssignment)
    M_pad = M if M_pad is None else int(M_pad)
    if pack_out.dtype != __import__("torch").float64 or pack_out.numel() != M_pad + PACK_TAIL or not pack_out.is_contiguous():
        raise RuntimeError(f"pack_out must be a contiguous float64 tensor of M_pad + {PACK_TAIL} elements")
    ctx = _pick_ctx(co.device, adev, pack_out.device.index)
    E, _, H, W = (int(v) for v in sceneCoordinates.shape)
    shiftX, shiftY, f, ppx, ppy, tau, alpha, beta, maxReproj, sub = params
    ctx.check(ctx.lib.esacb200_forward_pack(ctx.handle, co.ptr, E, H, W, aptr, astride, M, M_pad, int(shiftX), int(shiftY), float(f),
                                            float(ppx), float(ppy), float(tau), float(alpha), float(beta), float(maxReproj),
                                            int(sub), int(expert_offset), pack_out.data_ptr()))


def forward_sharded(sceneCoordinates, hypAssignment, outPose, shiftX, shiftY, focalLength, ppointX, ppointY, inlierThreshold,
                    inlierAlpha, inlierBeta, maxReproj, subSampling, expert_offset: int = 0, M_pad: int | None = None,
                    hyp_offset: int = 0, device: int | None = None, hyp_stride: int = 1) -> int:
    """esac.forward over experts / hypotheses sharded across the ranks of the library's communicator (Context.comm_init):
    this rank's shard in, the GLOBAL winner's pose (outPose, in place) and expert index out, on every rank.  One
    ncclAllGather on the library's stream, no torch collective.  hypAssignment may be empty (M = 0)."""
    _check(sceneCoordinates, "Float", 4, "sceneCoordinates")
    _check(hypAssignment, "Long", 1, "hypAssignment")
    _check(outPose, "Float", 2, "outPose")
    co = _Arg(sceneCoordinates)
    op = _Arg(outPose, writable=True)
    aptr, astride, M, adev, _keep = _assign_arg(hypAssignment)
    M_pad = max(M, 1) if M_pad is None else int(M_pad)
    devs = [d for d in (co.device, op.device, adev) if d is not None]
    ctx = _pick_ctx(*devs) if devs else _pick_ctx_host(device)
    E, _, H, W = (int(s) for s in sceneCoordinates.shape)
    expert = C.c_int(-1)
    ctx.set_option("hyp_offset", hyp_offset)
    ctx.set_option("hyp_stride", hyp_stride)
    try:
        rc = ctx.lib.esacb200_forward_sharded(ctx.handle, co.ptr, E, H, W, aptr, astride, M, M_pad, op.ptr, int(shiftX), int(shiftY),
                                              float(focalLength), float(ppointX), float(ppointY), float(inlierThreshold),
                                              float(inlierAlpha), float(inlierBeta), float(maxReproj), int(subSampling),
                                              int(expert_offset), C.byref(expert))
    finally:
        ctx.set_option("hyp_offset", 0)
        ctx.set_option("hyp_stride", 1)
    ctx.check(rc)
    op.finish()
    return int(expert.value)


def backward_sharded_nccl(sceneCoordinates, outGradients, hypAssignment, gtPose, wLossRot, wLossTrans, lossCut, shiftX, shiftY,
                          focalLength, ppointX, ppointY, inlierThreshold, inlierAlpha, inlierBeta, maxReproj, subSampling,
                          hyp_offset: int = 0, device: int | None = None, reduce_grads: bool = False, hyp_stride: int = 1) -> float:
    """esac.backward on this rank's shard; the two exchanges run as NCCL collectives inside the library.  Returns the GLOBAL
    expected loss; outGradients receives this shard's gradient slices, or -- reduce_grads, hypothesis-major sharding with all
    planes on every rank -- the gradient summed over all ranks.  hypAssignment may be empty."""
    _check(sceneCoordinates, "Float", 4, "sceneCoordinates")
    _check(outGradients, "Float", 4, "outGradients")
    _check(hypAssignment, "Long", 1, "hypAssignment")
    _check(gtPose, "Float", 2, "gtPose")
    co = _Arg(sceneCoordinates)
    gr = _Arg(outGradients, writable=True)
    gt = _Arg(gtPose)
    aptr, astride, M, adev, _keep = _assign_arg(hypAssignment)
    devs = [d for d in (co.device, gr.device, gt.device, adev) if d is not None]
    ctx = _pick_ctx(*devs) if devs else _pick_ctx_host(device)
    E, _, H, W = (int(s) for s in sceneCoordinates.shape)
    loss = C.c_double(0.0)
    ctx.set_option("hyp_offset", hyp_offset)
    ctx.set_option("hyp_stride", hyp_stride)
    try:
        rc = ctx.lib.esacb200_backward_sharded_nccl(ctx.handle, co.ptr, gr.ptr, E, H, W, aptr, astride, M, gt.ptr, float(wLossRot),
                                                    float(wLossTrans), float(lossCut), int(shiftX), int(shiftY), float(focalLength),
                                                    float(ppointX), float(ppointY), float(inlierThreshold), float(inlierAlpha),
                                                    float(inlierBeta), float(maxReproj), int(subSampling), int(bool(reduce_grads)),
                                                    C.byref(loss))
    finally:
        ctx.set_option("hyp_offset", 0)
        ctx.set_option("hyp_stride", 1)
    ctx.check(rc)
    gr.finish()
    return float(loss.value)


def score_poses(sceneCoordinates, hypAssignment, poses6, shiftX, shiftY, focalLength, ppointX, ppointY,
                inlierThreshold, inlierAlpha, inlierBeta, maxReproj, subSampling) -> np.ndarray:
    """Soft-inlier scores (getReproErrs + getHypScores) of given scene poses [M, 6] = (rvec, tvec)."""
    _check(sceneCoordinates, "Float", 4, "sceneCoordinates")
    _check(hypAssignment, "Long", 1, "hypAssignment")
    co = _Arg(sceneCoordinates)
    aptr, astride, M, adev, _keep = _assign_arg(hypAssignment)
    poses6 = np.ascontiguousarray(poses6, np.float64)
    assert poses6.shape == (M, 6)
    ctx = _pick_ctx(co.device, adev)
    E, _, H, W = (int(s) for s in sceneCoordinates.shape)
    out = np.zeros(M)
    ctx.check(ctx.lib.esacb200_score_poses(ctx.handle, co.ptr, E, H, W, aptr, astride, M, poses6.ctypes.data, int(shiftX),
                                           int(shiftY), float(focalLength), float(ppointX), float(ppointY),
                                           float(inlierThreshold), float(inlierAlpha), float(inlierBeta), float(maxReproj),
                                           int(subSampling), out.ctypes.data))
    return out


def refine_poses(sceneCoordinates, hypAssignment, poses6, shiftX, shiftY, focalLength, ppointX, ppointY,
                 inlierThreshold, maxReproj, subSampling):
    """refineHyp for every given pose.  Returns (refined [M, 6], accepted rounds [M], final inlier counts [M])."""
    _check(sceneCoordinates, "Float", 4, "sceneCoordinates")
    _check(hypAssignment, "Long", 1, "hypAssignment")
    co = _Arg(sceneCoordinates)
    aptr, astride, M, adev, _keep = _assign_arg(hypAssignment)
    poses6 = np.array(poses6, np.float64, order="C", copy=True)
    assert poses6.shape == (M, 6)
    ctx = _pick_ctx(co.device, adev)
    E, _, H, W = (int(s) for s in sceneCoordinates.shape)
    rounds = np.zeros(M, np.int32)
    inl = np.zeros(M, np.int32)
    ctx.check(ctx.lib.esacb200_refine_poses(ctx.handle, co.ptr, E, H, W, aptr, astride, M, poses6.ctypes.data, int(shiftX),
                                            int(shiftY), float(focalLength), float(ppointX), float(ppointY),
                                            float(inlierThreshold), float(maxReproj), int(subSampling),
                                            rounds.ctypes.data, inl.ctypes.data))
    return poses6, rounds, inl


def set_seed(seed: int, device: int | None = None):
    context(device).set_seed(seed)


def set_option(key: str, value: float, device: int | None = None):
    context(device).set_option(key, value)


def inject_cells(cells, device: int | None = None):
    context(device).inject_cells(cells)


def last_stats(device: int | None = None) -> dict:
    return context(device).stats()


def last_hypotheses(device: int | None = None, losses: bool = False) -> dict:
    return context(device).hypotheses(losses)
