"""Two-GPU identity tests (skipped on a single-GPU box): experts sharded expert-major over 2 ranks must reproduce the
single-GPU result -- same winner / pose in forward (one all-gather of scores), same expected loss and the same gradient
slices in backward (two KB-sized exchanges)."""
import os
import socket

import numpy as np
import pytest
import torch

from esac_b200.synth import make_scene

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _split(E, world):
    """Experts dealt expert-major, as evenly as possible (E need not be divisible by the number of ranks)."""
    base, extra = divmod(E, world)
    sizes = [base + (1 if r < extra else 0) for r in range(world)]
    starts = [sum(sizes[:r]) for r in range(world)]
    return starts, sizes


def _worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    import esac_b200.api as api
    from esac_b200 import sharded
    E, Mper = 5, 24                      # 5 experts over 2 ranks: 3 + 2 -> shards of 72 and 48 hypotheses
    sc = make_scene(E=E, H=30, W=40, M=Mper, sub=8, seed=77, per_expert=True, active_only=False)
    starts, sizes = _split(E, world)
    e0, Eloc = starts[rank], sizes[rank]
    hsel = slice(e0 * Mper, (e0 + Eloc) * Mper)
    M_pad = max(sizes) * Mper
    dev = torch.device("cuda", rank)
    coords_l = torch.from_numpy(sc.coords[e0:e0 + Eloc]).to(dev)
    assign_l = torch.from_numpy(sc.assign[hsel] - e0).to(dev)
    ctx = api.context(rank)
    ctx.set_option("fixed_seed", 1)
    res = {"rank": rank}
    # ---- transport 1: torch.distributed around forward_pack / the exchange callback ----
    ctx.set_seed(5)
    out = torch.zeros(4, 4, device=dev)
    res["expert_t"] = sharded.forward_sharded(coords_l, assign_l, out, sc.params, expert_offset=e0, hyp_offset=e0 * Mper, M_pad=M_pad)
    res["pose_t"] = out.cpu().numpy()
    ctx.set_seed(5)
    grads_l = torch.zeros_like(coords_l)
    res["loss_t"] = sharded.backward_sharded(coords_l, grads_l, assign_l, torch.from_numpy(sc.gt_pose), 1.0, 100.0, 100.0, sc.params,
                                             hyp_offset=e0 * Mper)
    res["grads_t"] = grads_l.cpu().numpy()
    # ---- transport 2: the library's own NCCL communicator ----
    sharded.init_comm(device=rank)
    ctx.set_seed(5)
    out2 = torch.zeros(4, 4, device=dev)
    res["expert"] = sharded.forward_sharded(coords_l, assign_l, out2, sc.params, expert_offset=e0, hyp_offset=e0 * Mper, M_pad=M_pad)
    res["pose"] = out2.cpu().numpy()
    # host tensors through the same entry (what the reference's callers hold)
    ctx.set_seed(5)
    out3 = torch.zeros(4, 4)
    res["expert_h"] = sharded.forward_sharded(coords_l.cpu(), assign_l.cpu(), out3, sc.params, expert_offset=e0,
                                              hyp_offset=e0 * Mper, M_pad=M_pad, device=rank)
    res["pose_h"] = out3.numpy()
    ctx.set_seed(5)
    grads2 = torch.zeros_like(coords_l)
    res["loss"] = sharded.backward_sharded(coords_l, grads2, assign_l, torch.from_numpy(sc.gt_pose), 1.0, 100.0, 100.0, sc.params,
                                           hyp_offset=e0 * Mper)
    res["grads"] = grads2.cpu().numpy()
    # ---- a rank WITHOUT hypotheses (rank 1 hands everything to rank 0's experts): must still take part ----
    ctx.set_seed(5)
    if rank == 0:
        c_e, a_e = torch.from_numpy(sc.coords).to(dev), torch.from_numpy(sc.assign).to(dev)
    else:
        c_e, a_e = torch.zeros(1, 3, 30, 40, device=dev), torch.zeros(0, dtype=torch.int64, device=dev)
    out4 = torch.zeros(4, 4, device=dev)
    res["expert_e"] = sharded.forward_sharded(c_e, a_e, out4, sc.params, expert_offset=0, hyp_offset=0, M_pad=E * Mper)
    res["pose_e"] = out4.cpu().numpy()
    ctx.set_seed(5)
    g_e = torch.zeros_like(c_e)
    res["loss_e"] = sharded.backward_sharded(c_e, g_e, a_e, torch.from_numpy(sc.gt_pose), 1.0, 100.0, 100.0, sc.params, hyp_offset=0)
    # ---- hypothesis-major: every rank holds ALL planes and a contiguous slice of the hypotheses; gradients all-reduced ----
    Mh = E * Mper
    cut = (Mh * 3) // 5                      # 72 / 48: the slices cut through an expert
    lo, hi = (0, cut) if rank == 0 else (cut, Mh)
    c_all = torch.from_numpy(sc.coords).to(dev)
    a_h = torch.from_numpy(sc.assign[lo:hi]).to(dev)
    ctx.set_seed(5)
    out5 = torch.zeros(4, 4, device=dev)
    res["expert_hm"] = sharded.forward_sharded(c_all, a_h, out5, sc.params, expert_offset=0, hyp_offset=lo, M_pad=max(cut, Mh - cut))
    res["pose_hm"] = out5.cpu().numpy()
    ctx.set_seed(5)
    g_hm = torch.full_like(c_all, 0.5)       # += semantics survive the reduction
    res["loss_hm"] = sharded.backward_sharded(c_all, g_hm, a_h, torch.from_numpy(sc.gt_pose), 1.0, 100.0, 100.0, sc.params,
                                              hyp_offset=lo, reduce_grads=True)
    res["grads_hm"] = g_hm.cpu().numpy() - 0.5
    # ---- the same dealt round-robin (hypothesis h -> rank h % 2): hyp_offset = rank, hyp_stride = 2 ----
    a_s = torch.from_numpy(np.ascontiguousarray(sc.assign[rank::2])).to(dev)
    ctx.set_seed(5)
    out6 = torch.zeros(4, 4, device=dev)
    res["expert_hs"] = sharded.forward_sharded(c_all, a_s, out6, sc.params, expert_offset=0, hyp_offset=rank, hyp_stride=2, M_pad=(Mh + 1) // 2)
    res["pose_hs"] = out6.cpu().numpy()
    ctx.set_seed(5)
    g_hs = torch.zeros_like(c_all)
    res["loss_hs"] = sharded.backward_sharded(c_all, g_hs, a_s, torch.from_numpy(sc.gt_pose), 1.0, 100.0, 100.0, sc.params,
                                              hyp_offset=rank, hyp_stride=2, reduce_grads=True)
    res["grads_hs"] = g_hs.cpu().numpy()
    sharded.destroy_comm(rank)
    if rank == 0:  # the unsharded problem on one GPU
        ctx.set_seed(5)
        ref_out = np.zeros((4, 4), np.float32)
        ref_e = api.forward(sc.coords, sc.assign, ref_out, *sc.params)
        ctx.set_seed(5)
        g = np.zeros_like(sc.coords)
        ref_loss = api.backward(sc.coords, g, sc.assign, sc.gt_pose, 1.0, 100.0, 100.0, *sc.params)
        res.update(ref_expert=ref_e, ref_pose=ref_out, ref_loss=ref_loss, ref_grads=g, starts=starts, sizes=sizes)
    q.put(res)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpu_sharding_reproduces_single_gpu():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    ps = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in ps:
        p.start()
    res = {}
    for _ in range(2):
        r = q.get(timeout=300)
        res[r["rank"]] = r
    for p in ps:
        p.join(timeout=120)
        assert p.exitcode == 0
    ref = res[0]
    scale = max(np.abs(ref["ref_grads"]).max(), 1e-12)
    for r in (0, 1):
        sl = slice(ref["starts"][r], ref["starts"][r] + ref["sizes"][r])
        for tag in ("_t", "", "_h", "_e", "_hm", "_hs"):   # torch transport, library NCCL, host tensors, empty shard, hypothesis-major
            assert res[r]["expert" + tag] == ref["ref_expert"], tag
            assert np.allclose(res[r]["pose" + tag], ref["ref_pose"], atol=1e-6), tag
        for tag in ("_t", "", "_e", "_hm", "_hs"):
            assert abs(res[r]["loss" + tag] - ref["ref_loss"]) < 1e-9 * max(1.0, abs(ref["ref_loss"])), tag
        for tag in ("_t", ""):
            assert np.abs(res[r]["grads" + tag] - ref["ref_grads"][sl]).max() / scale < 1e-6, tag
        # hypothesis-major: the rank-summed gradient of the whole tensor on every rank (float sums in a different order)
        assert np.abs(res[r]["grads_hm"] - ref["ref_grads"]).max() / scale < 1e-5
        assert np.abs(res[r]["grads_hs"] - ref["ref_grads"]).max() / scale < 1e-5
    assert np.abs(ref["ref_grads"]).max() > 0


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_one_process_two_devices_full_resolution_and_current_device_kept():
    """One process, contexts on cuda:0 and cuda:1: the scoring kernel's >48 KB shared-memory opt-in is a per-device
    attribute (it used to be set once per process), and no entry point may leave the caller's current device switched."""
    import esac_b200.api as api
    sc = make_scene(E=2, H=480, W=640, M=32, sub=1, seed=3)
    outs = []
    torch.cuda.set_device(0)
    for d in (0, 1):
        ctx = api.context(d)
        ctx.set_option("fixed_seed", 1)
        ctx.set_seed(9)
        out = torch.zeros(4, 4, device=f"cuda:{d}")
        e = api.forward(torch.from_numpy(sc.coords).to(f"cuda:{d}"), torch.from_numpy(sc.assign).to(f"cuda:{d}"), out, *sc.params)
        assert torch.cuda.current_device() == 0          # tensors on cuda:1 did not move the caller's device
        g = torch.zeros(sc.coords.shape, device=f"cuda:{d}")
        ctx.set_seed(9)
        api.backward(torch.from_numpy(sc.coords).to(f"cuda:{d}"), g, torch.from_numpy(sc.assign).to(f"cuda:{d}"),
                     torch.from_numpy(sc.gt_pose), 1.0, 100.0, 100.0, *sc.params)
        assert torch.cuda.current_device() == 0
        outs.append((e, out.cpu().numpy(), g.cpu().numpy()))
    assert outs[0][0] == outs[1][0]
    assert np.array_equal(outs[0][1], outs[1][1]) and np.array_equal(outs[0][2], outs[1][2])
