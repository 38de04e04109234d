#!/usr/bin/env python
"""Benchmark of the ESAC hot path (esac.forward) on B200s.

Metric (BASELINE.json): pose hypotheses scored per second at 640x480, 256 hypotheses x E experts.
A step = one batch of IMAGES_PER_STEP synthetic images, each through one esac.forward call (sample -> score -> select ->
refine), exactly as the reference's callers loop over a test set with batch size 1 (test_esac.py:137-205).

  python bench.py [--gpus N] [--steps K] [--warmup W]          this repository's CUDA path
  python bench.py ... --dump-outputs DIR                       also write what the timed path returned for the images of
                                                               its last step: DIR/poses.npy [32, 4, 4] float32 (outPose) and
                                                               DIR/experts.npy [32] float64 (the returned expert index)
  python bench.py --impl reference ...                         the reference's CPU path on the host cores: oracle/_ref (the
                                                               reference's own esac.cpp compiled against the cv2-backed OpenCV
                                                               stand-in), or the cv2 oracle port where _ref is not built
For N > 1 launch under torchrun (one rank per GPU); experts are sharded expert-major across the ranks, every rank runs the
full local pipeline on its shard and ONE ncclAllGather of the per-shard records -- issued by the library on its own stream --
picks the global winner (SURVEY.md section 8e).

One JSON line on stdout (rank 0): value = device-resident whole-job hypotheses/s; e2e = the same through esac.forward with
pinned HOST tensors (H2D copy of the coordinate maps and D2H of the pose inside the timed region), e2e_pageable with ordinary
host tensors (what `prediction.cpu()` hands the reference, test_esac.py:187); roofline = the scoring kernel's algorithmic
bytes (12*N per hypothesis) / its CUDA-event time / the measured HBM peak; cpu_baseline = the reference's CPU path on this
box's host cores on a bounded sample; configs = BASELINE.json's configs[2..4] at this GPU count.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "pose hypotheses scored/sec (640x480, 256 hyp x E experts)"
UNIT = "hypotheses/s"
E_PER_GPU, HYPS_PER_EXPERT, H, W, SUB = 7, 256, 480, 640, 1
N_SCENES = 6          # rotating inputs: 6 x 25.8 MB > 126 MB L2, so no forward finds its planes in L2
IMAGES_PER_STEP = 32  # one step = 32 images: long enough (~45 ms) for the clock sampler to see every step


def workload_config(n_gpus: int) -> dict:
    return {"workload": f"BASELINE configs[1]: 7Scenes-style ensemble, {E_PER_GPU} experts/GPU x {HYPS_PER_EXPERT} "
                        f"hypotheses each ({E_PER_GPU * HYPS_PER_EXPERT * n_gpus} per image), {W}x{H} scene-coordinate maps "
                        f"(subSampling=1), f=525, tau=10 alpha=100 beta=0.5 maxReproj=100, 40% outliers; one step = "
                        f"{IMAGES_PER_STEP} images, one esac.forward each",
            "experts_per_gpu": E_PER_GPU, "hyps_per_expert": HYPS_PER_EXPERT, "map": [H, W],
            "hyps_per_image": E_PER_GPU * HYPS_PER_EXPERT * n_gpus, "images_per_step": IMAGES_PER_STEP,
            "hyps_per_step": E_PER_GPU * HYPS_PER_EXPERT * n_gpus * IMAGES_PER_STEP,
            "parallelism": "single GPU" if n_gpus == 1 else f"expert-major shard over {n_gpus} GPUs + 1 ncclAllGather of scores",
            "l2_policy": f"inputs larger than L2: {N_SCENES} distinct scenes ({N_SCENES * E_PER_GPU * 3 * H * W * 4 / 1e6:.0f} MB) used round-robin"}


def make_inputs(rank: int, n: int = N_SCENES):
    from esac_b200.synth import make_scene
    return [make_scene(E=E_PER_GPU, H=H, W=W, M=HYPS_PER_EXPERT, sub=SUB, seed=100 * rank + i, per_expert=True,
                       active_only=False) for i in range(n)]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.lines, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); mx = float(p[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# -------------------------------------------------------------------------------------------------
# the reference's CPU path
# -------------------------------------------------------------------------------------------------
def cpu_sample(scene, take: int, seed: int):
    """One bounded sample of the workload on the host cores: `take` of the image's hypotheses, spread over all experts,
    through a full esac.forward of the reference's CPU implementation.  Returns (hyps/s, seconds, workers, kind, how)."""
    idx = np.linspace(0, len(scene.assign) - 1, take).astype(int)
    from oracle import ref_parallel
    if ref_parallel.available():
        n, secs, workers = ref_parallel.forward_ref_parallel(scene, idx, seed=seed)
        return n / secs, secs, workers, "reference", ("oracle/_ref = the reference's unmodified esac.cpp + thread_rand.cpp compiled against "
                                                      "the cv2-backed OpenCV stand-in; one single-threaded esac.forward per slice of <= 4 "
                                                      "hypotheses on a fork pool (the shim's GIL would serialise OpenMP threads)")
    from copy import copy
    from oracle.parallel import forward_parallel, scene_dict
    sc2 = copy(scene)
    sc2.assign = scene.assign[idx]
    e, T, secs, workers = forward_parallel(scene_dict(sc2, take), seed=seed)
    return take / secs, secs, workers, "port", "cv2 oracle port (oracle/esac_oracle.py), fork pool over hypotheses"


def run_reference(args, rank: int, world: int):
    """--impl reference: the reference's own CPU implementation on a bounded sample per step."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    from esac_b200.synth import make_scene
    sc = make_scene(E=E_PER_GPU, H=H, W=W, M=HYPS_PER_EXPERT, sub=SUB, seed=0, per_expert=True, active_only=False)
    take = min(max(4 * cores, 64), E_PER_GPU * HYPS_PER_EXPERT)
    warm_run, steps_run = args.warmup, args.steps
    for _ in range(warm_run):
        cpu_sample(sc, take, 1)
    t0 = time.perf_counter()
    kind = how = None
    workers = cores
    for k in range(steps_run):
        _, _, workers, kind, how = cpu_sample(sc, take, 2 + k)
    dt = time.perf_counter() - t0
    val = take * steps_run / dt
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "steps_run": steps_run, "warmup_run": warm_run, "ms_per_step": 1e3 * dt / steps_run,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64/f32 mix (OpenCV)", "data": "synthetic",
            "config": workload_config(args.gpus),
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": workers, "kind": kind,
                             "sample": f"{take} of {E_PER_GPU * HYPS_PER_EXPERT} hypotheses of one image per step (every "
                                       f"{E_PER_GPU * HYPS_PER_EXPERT // take}-th, all experts), full esac.forward "
                                       f"(sample+score+select+refine); {how}"},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# -------------------------------------------------------------------------------------------------
# BASELINE.json configs[2..4] at this GPU count
# -------------------------------------------------------------------------------------------------
def split_experts(E: int, world: int):
    base, extra = divmod(E, world)
    sizes = [base + (1 if r < extra else 0) for r in range(world)]
    return [sum(sizes[:r]) for r in range(world)], sizes


def run_configs(rank: int, world: int, dev, api, sharded, dist, reps: int = 4):
    """c3: 19 experts, 256 hypotheses per image, batch of 8 images -- images dealt to the ranks (no communication);
    c4: 10 experts x 512 hypotheses each, ONE image -- strong scaling, experts dealt expert-major (unequal shards);
    c5: 20 experts, 1024 hypotheses, forward + backward (the esac_loss of train_esac.py:105-183) -- hypotheses dealt to the ranks,
        all planes everywhere; the two backward exchanges and the gradient sum as NCCL collectives inside the library.
    Every entry: whole-job hypotheses/s = hypotheses of the job / max-over-ranks device time."""
    import torch
    from esac_b200.synth import make_scene
    out = {}

    def timed(fn, n):
        fn(); fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def rank_stages():
        """The library's CUDA-event stage timers of this rank's LAST call, as lists over the ranks (ms)."""
        keys = ["ms_sample", "ms_score", "ms_select", "ms_refine", "ms_backward", "ms_total"]
        st = api.context(dev.index).stats()
        t = torch.tensor([st[k] for k in keys], device=dev, dtype=torch.float64)
        if world > 1:
            g = torch.empty(world * len(keys), device=dev, dtype=torch.float64)
            dist.all_gather_into_tensor(g, t)
            g = g.view(world, len(keys)).cpu().numpy()
        else:
            g = t.view(1, -1).cpu().numpy()
        return {k: [round(float(v), 4) for v in g[:, i]] for i, k in enumerate(keys)}

    # ---- c3 ----
    B = 8
    if B % world == 0:
        Bl = B // world
        scs = [make_scene(E=19, H=H, W=W, M=256, sub=SUB, seed=300 + b) for b in range(rank * Bl, rank * Bl + min(Bl, 2))]
        coords = torch.stack([torch.from_numpy(scs[b % len(scs)].coords) for b in range(Bl)]).to(dev)
        assign = torch.stack([torch.from_numpy(scs[b % len(scs)].assign) for b in range(Bl)]).to(dev)
        poses = torch.zeros(Bl, 4, 4, device=dev)
        ms = timed(lambda: api.forward_batch(coords, assign, poses, *scs[0].params), reps)
        out["c3_19experts_256hyp_batch8"] = {"value": B * 256 / (ms * 1e-3), "unit": UNIT, "ms_per_batch": ms, "images": B,
                                             "images_per_gpu": Bl, "hyps_per_image": 256, "scaling": "strong",
                                             "parallelism": f"8 images dealt to {world} GPU(s), esac_b200.api.forward_batch per rank, no collective"}
        del coords, assign, poses
    # ---- c4 ----
    E4, M4 = 10, 512
    sc = make_scene(E=E4, H=H, W=W, M=M4, sub=SUB, seed=400, per_expert=True, active_only=False)
    starts, sizes = split_experts(E4, world)
    e0, El = starts[rank], sizes[rank]
    c_l = torch.from_numpy(sc.coords[e0:e0 + El]).to(dev) if El else torch.zeros(1, 3, H, W, device=dev)
    a_l = torch.from_numpy(sc.assign[e0 * M4:(e0 + El) * M4] - e0).to(dev)
    pose = torch.zeros(4, 4, device=dev)
    M_pad = max(max(sizes) * M4, 1)
    if world == 1:
        fn = lambda: api.forward(c_l, a_l, pose, *sc.params)
    else:
        fn = lambda: sharded.forward_sharded(c_l, a_l, pose, sc.params, expert_offset=e0, hyp_offset=e0 * M4, M_pad=M_pad)
    ms = timed(fn, reps)
    out["c4_10experts_512hyp_each_one_image"] = {"value": E4 * M4 / (ms * 1e-3), "unit": UNIT, "ms_per_image": ms, "hyps_per_image": E4 * M4,
                                                 "experts_per_rank": sizes, "scaling": "strong", "stages_ms_by_rank": rank_stages(),
                                                 "parallelism": "single GPU" if world == 1 else "expert-major shard, 1 ncclAllGather"}
    del c_l, a_l
    # ---- c5 ----
    E5, M5 = 20, 1024
    sc = make_scene(E=E5, H=H, W=W, M=M5, sub=SUB, seed=500, active_only=False)   # 1024 hypotheses drawn from the gating (60% on the true expert)
    order = np.argsort(sc.assign, kind="stable")                                    # hypotheses grouped expert-major
    assign_sorted = sc.assign[order]
    # hypothesis-major: every rank holds all 20 planes (74 MB) and every N-th of the expert-sorted hypotheses, so the
    # contributing hypotheses -- all on the true expert -- spread over the ranks; their gradient slices overlap and are summed
    # with one ncclAllReduce (esacb200_backward_sharded_nccl, reduce_grads)
    counts = [len(range(r, M5, world)) for r in range(world)]   # dealt round-robin: hypothesis h of the sorted list goes to rank h % N
    M_pad = max(max(counts), 1)
    c_l = torch.from_numpy(sc.coords).to(dev)
    a_l = torch.from_numpy(np.ascontiguousarray(assign_sorted[rank::world])).to(dev)
    g_l = torch.zeros_like(c_l)
    gt = torch.from_numpy(sc.gt_pose)
    if world == 1:
        f_fwd = lambda: api.forward(c_l, a_l, pose, *sc.params)
        f_bwd = lambda: api.backward(c_l, g_l, a_l, gt, 1.0, 100.0, 100.0, *sc.params)
    else:
        f_fwd = lambda: sharded.forward_sharded(c_l, a_l, pose, sc.params, expert_offset=0, hyp_offset=rank, hyp_stride=world, M_pad=M_pad)
        f_bwd = lambda: sharded.backward_sharded(c_l, g_l, a_l, gt, 1.0, 100.0, 100.0, sc.params, hyp_offset=rank, hyp_stride=world,
                                                 reduce_grads=True)
    ms_f = timed(f_fwd, reps)
    st_f = rank_stages()
    ms_b = timed(f_bwd, reps)
    st_b = rank_stages()
    st = api.context(dev.index).stats()
    out["c5_20experts_1024hyp_forward_backward"] = {
        "value": M5 / ((ms_f + ms_b) * 1e-3), "unit": UNIT, "ms_forward": ms_f, "ms_backward": ms_b, "hyps_per_image": M5,
        "hyps_per_rank": counts, "contributing_hypotheses_rank0": st["n_contrib"], "scaling": "strong",
        "stages_ms_by_rank_forward": st_f, "stages_ms_by_rank_backward": st_b,
        "parallelism": "single GPU" if world == 1 else "hypothesis-major shard (all planes on every rank, hypotheses dealt round-robin); forward: "
                       "1 ncclAllGather; backward: ncclAllGather of (max, sum exp) + ncclAllReduce of the expectation + "
                       "ncclAllReduce of the gradient planes that received contributions on some rank (3.7 of 74 MB here)",
        "note": "the gating puts 60% of the hypotheses and every contributing one on the true expert: dealing experts to ranks "
                "would leave the refine-all stage on one GPU, dealing hypotheses spreads it"}
    return out


# -------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the poses and expert indices of the last timed step's images to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs applies to the CUDA path (--impl ours)")
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: this implementation has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    import esac
    import esac_b200.api as api
    from esac_b200 import sharded
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")  # the driver's own setting (it greps NCCL's communicator lines) wins
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        sharded.init_comm(device=local_rank)         # the library's own communicator: collectives on its stream

    ctx = api.context(local_rank)
    scenes = make_inputs(rank)
    M_local = len(scenes[0].assign)
    M_total = M_local * world
    N = H * W
    d_coords = [torch.from_numpy(s.coords).to(dev) for s in scenes]
    d_assign = [torch.from_numpy(s.assign).to(dev) for s in scenes]
    h_coords = [torch.from_numpy(s.coords).pin_memory() for s in scenes]
    h_assign = [torch.from_numpy(s.assign).pin_memory() for s in scenes]
    p_coords = [torch.from_numpy(s.coords) for s in scenes]     # ordinary (pageable) host tensors
    p_assign = [torch.from_numpy(s.assign) for s in scenes]
    d_out = torch.zeros(4, 4, device=dev)
    # device-resident timed path: image p of a step writes its own 4x4 view, so the last step's poses can be dumped
    d_poses = torch.zeros(IMAGES_PER_STEP, 4, 4, device=dev)
    d_pose_views = list(d_poses.unbind(0))
    h_out = torch.zeros(4, 4).pin_memory()
    p_out = torch.zeros(4, 4)
    # input preparation, not a step: the first transfers out of freshly pinned pages run at a fraction of the steady PCIe rate
    # (measured: ~22 GB/s over the first 20 copies, >50 GB/s afterwards), so every pinned buffer is pushed through a few times
    scratch = torch.empty_like(d_coords[0])
    for _ in range(8):
        for hcrd in h_coords:
            scratch.copy_(hcrd, non_blocking=True)
    torch.cuda.synchronize()
    del scratch
    params = scenes[0].params
    api.set_seed(1305 + rank, local_rank)
    STAGES = ("ms_h2d", "ms_prep", "ms_sample", "ms_score", "ms_select", "ms_refine", "ms_total")

    def forward_once(i, mode: str):
        j = i % N_SCENES
        co, asg, outs = {"device": (d_coords, d_assign, d_pose_views), "pinned": (h_coords, h_assign, [h_out]),
                         "pageable": (p_coords, p_assign, [p_out])}[mode]
        out = outs[i % len(outs)]
        if world == 1:
            return esac.forward(co[j], asg[j], out, *params)
        return sharded.forward_sharded(co[j], asg[j], out, params, expert_offset=rank * E_PER_GPU, hyp_offset=rank * M_local,
                                       M_pad=M_local, device=local_rank)

    def timed(mode: str, steps: int, warmup: int):
        k = 0
        for _ in range(warmup * IMAGES_PER_STEP):
            forward_once(k, mode); k += 1
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        acc = {s: 0.0 for s in STAGES}
        launches = score_launches = 0
        experts = [None] * IMAGES_PER_STEP  # k starts at a multiple of IMAGES_PER_STEP: slot p = image p of a step
        e0.record()
        for _ in range(steps * IMAGES_PER_STEP):
            experts[k % IMAGES_PER_STEP] = forward_once(k, mode); k += 1
            st = ctx.stats()
            for s in STAGES:
                acc[s] += st[s]
            launches += st["kernel_launches"]
            score_launches += st["score_launches"]
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        n = steps * IMAGES_PER_STEP
        return ms, {s: acc[s] / n for s in STAGES}, launches, score_launches, ctx.stats(), experts

    sampler = ClockSampler(local_rank)
    sampler.start()
    ms, stages, launches, score_launches, last, last_experts = timed("device", args.steps, args.warmup)
    clocks = sampler.stop()
    last_poses = d_poses.cpu().numpy()
    ms_e2e, stages_e2e, _, _, _, _ = timed("pinned", args.steps, args.warmup)
    steps_pg = max(1, args.steps // 4)
    ms_pg, _, _, _, _, _ = timed("pageable", steps_pg, 1)

    # per-rank stage timers (CUDA events inside the library, read after each call's single synchronisation): max / mean over ranks
    stage_table = None
    if world > 1:
        t = torch.tensor([stages[s] for s in STAGES], device=dev, dtype=torch.float64)
        g = torch.empty(world * len(STAGES), device=dev, dtype=torch.float64)
        dist.all_gather_into_tensor(g, t)
        g = g.view(world, len(STAGES)).cpu().numpy()
        stage_table = {s: {"max": float(g[:, i].max()), "mean": float(g[:, i].mean())} for i, s in enumerate(STAGES)}

    # informative: the batched entry point (8 images per call, pinned host tensors, copy of image b+1 overlapping image b)
    batched = None
    if world == 1:
        Bsz = 8
        hb_coords = torch.stack([h_coords[i % N_SCENES] for i in range(Bsz)]).pin_memory()
        hb_assign = torch.stack([h_assign[i % N_SCENES] for i in range(Bsz)])
        hb_out = torch.zeros(Bsz, 4, 4).pin_memory()
        reps = max(2, args.steps // 4)
        api.forward_batch(hb_coords, hb_assign, hb_out, *params)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            api.forward_batch(hb_coords, hb_assign, hb_out, *params)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        batched = {"value": M_local * Bsz * reps / dt, "unit": UNIT, "images_per_call": Bsz, "ms_per_image": 1e3 * dt / (reps * Bsz),
                   "note": "esac_b200.api.forward_batch, pinned host maps, H2D overlapped with compute, one sync per call (host wall clock)"}
        del hb_coords

    # informative: esac.backward on the same workload (SURVEY 8d item 3), device-resident tensors
    bwd = None
    if world == 1:
        g = torch.zeros_like(d_coords[0])
        reps = 5
        esac.backward(d_coords[0], g, d_assign[0], torch.from_numpy(scenes[0].gt_pose), 1.0, 100.0, 100.0, *params)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        contrib, ms_ref = 0, 0.0
        for i in range(reps):
            j = i % N_SCENES
            esac.backward(d_coords[j], g, d_assign[j], torch.from_numpy(scenes[j].gt_pose), 1.0, 100.0, 100.0, *params)
            st = ctx.stats()
            contrib += st["n_contrib"]; ms_ref += st["ms_refine"]
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        bwd = {"ms_per_call": 1e3 * dt / reps, "value": M_local * reps / dt, "unit": UNIT, "ms_refine_all": ms_ref / reps,
               "contributing_hypotheses_per_call": contrib / reps,
               "note": "esac.backward (sample+score+refine every hypothesis with p>=1e-3 + gradients), CUDA tensors, host wall clock"}
        del g

    configs = None
    if not args.no_configs:
        del d_coords[2:], h_coords[2:], p_coords[2:]   # room for the 19 / 20-expert maps
        torch.cuda.empty_cache()
        try:
            configs = run_configs(rank, world, dev, api, sharded, dist)
        except Exception as exc:  # never let the extra block break the headline line
            configs = {"error": f"{type(exc).__name__}: {exc}"[:300]}

    if rank == 0:
        n_fwd = args.steps * IMAGES_PER_STEP
        value = M_total * n_fwd / (ms * 1e-3)
        e2e = M_total * n_fwd / (ms_e2e * 1e-3)
        e2e_pg = M_total * steps_pg * IMAGES_PER_STEP / (ms_pg * 1e-3)
        peak, peak_src = measured_peak()
        alg_bytes = M_local * 12.0 * N  # per scoring launch on this rank
        t_score = stages["ms_score"] * 1e-3
        achieved = alg_bytes / t_score / 1e9 if t_score > 0 else 0.0
        # the resource that actually binds the kernel: 3 MUFU ops per cell-hypothesis at 16 lanes/clk/SM (profiles/r01_pipes.txt)
        sm_count = ctx.device_info()["sm_count"]
        mhz = (clocks or {}).get("sm_mhz") or 1965.0
        mufu_peak = sm_count * (16.0 / 3.0) * mhz * 1e6 / N  # hypotheses/s
        on_chip = {"pipe": "MUFU (rsqrt, ex2, rcp per cell-hypothesis; 16 lanes/clk/SM measured)", "peak_hyps_per_s": mufu_peak,
                   "achieved_hyps_per_s": M_local / t_score if t_score > 0 else None,
                   "frac": (M_local / t_score) / mufu_peak if t_score > 0 else None}
        traffic = None
        tp = ROOT / "profiles" / "score_kernel_traffic.json"
        if tp.exists():
            try:
                traffic = json.loads(tp.read_text()).get("dram_bytes_per_launch")
            except Exception:
                traffic = None
        h2d = int(scenes[0].coords.nbytes + scenes[0].assign.nbytes) * IMAGES_PER_STEP
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "ms_per_forward": ms / n_fwd, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32 (scoring, f32x2 FFMA2) / f64 (P3P, refinement)", "data": "synthetic",
                "config": workload_config(world), "clocks": clocks,
                "e2e": {"value": e2e, "unit": UNIT, "ms_per_step": ms_e2e / args.steps, "ms_per_forward": ms_e2e / n_fwd,
                        "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": (132 if world == 1 else 80) * IMAGES_PER_STEP, "host_memory": "pinned"},
                "e2e_pageable": {"value": e2e_pg, "unit": UNIT, "ms_per_forward": ms_pg / (steps_pg * IMAGES_PER_STEP),
                                 "steps": steps_pg, "host_memory": "pageable (what prediction.cpu() hands the reference, test_esac.py:187)"},
                "gpu_launches": int(launches), "gpu_launches_per_forward": launches / n_fwd,
                "batched_e2e": batched, "backward": bwd,
                "roofline": {"kernel": "esacb200::score_kernel_tma<8>", "bound": "hbm", "achieved": achieved, "peak": peak,
                             "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": alg_bytes, "ms_per_launch": t_score * 1e3,
                             "launches_timed": int(score_launches),
                             "hyps_per_s_kernel_only": M_local / t_score if t_score > 0 else None,
                             "note": "achieved = hypotheses x 12 B x 307200 cells / mean CUDA-event time of the scoring launch over the "
                                     "timed region; each plane is read once per 64-hypothesis chunk, so frac > 1 is expected",
                             "on_chip_ceiling": on_chip},
                "stages_ms_per_forward": stages, "stages_ms_per_forward_e2e": stages_e2e, "stages_over_ranks": stage_table,
                "score_launch": {"ppt": last["score_ppt"], "grid": last["score_grid"], "refine_group": last["refine_group"]},
                "configs": configs}
        if args.dump_outputs:
            d = Path(args.dump_outputs)
            d.mkdir(parents=True, exist_ok=True)
            np.save(d / "poses.npy", last_poses.astype(np.float32))
            np.save(d / "experts.npy", np.array(last_experts, np.float64))
        if world == 1 and not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            take = min(max(4 * cores, 64), M_local)
            try:
                v, secs, workers, kind, how = cpu_sample(scenes[0], take, 1)
                line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": workers, "kind": kind,
                                        "sample": f"{take} of {M_local} hypotheses of one image, one full esac.forward "
                                                  f"(sample+score+select+refine), {secs:.1f} s; {how}"}
            except Exception as exc:
                line["cpu_baseline"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
            # informative: the scoring stage alone in compiled C/OpenMP (oracle/esac_oracle_c.c, no OpenCV, no Python in the
            # loop) -- an upper bound on what a compiled CPU forward could reach on this host
            try:
                from oracle.build import c_score
                sc = scenes[0]
                esac.forward(d_coords[0], d_assign[0], d_out, *params)
                poses = ctx.hypotheses()["poses"]
                n_c = min(M_local, max(256, 4 * cores))
                idx_c = np.linspace(0, M_local - 1, n_c).astype(int)
                c_score(sc.coords, sc.assign[idx_c[:cores]], poses[idx_c[:cores]], *params)      # warm-up, builds the library
                t0 = time.perf_counter()
                _, used = c_score(sc.coords, sc.assign[idx_c], poses[idx_c], *params)
                dtc = time.perf_counter() - t0
                line.setdefault("cpu_baseline", {})["compiled_scoring_only"] = {
                    "value": n_c / dtc, "unit": UNIT, "cores": int(used),
                    "sample": f"{n_c} of {M_local} hypotheses, getReproErrs+getHypScores restated in C/OpenMP, {dtc:.1f} s"}
            except Exception as exc:  # never let the informative leg break the bench line
                line.setdefault("cpu_baseline", {})["compiled_scoring_only"] = {"error": str(exc)[:200]}
        print(json.dumps(line), flush=True)
    if world > 1:
        sharded.destroy_comm(local_rank)
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
