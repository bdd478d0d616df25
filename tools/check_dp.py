"""Multi-GPU check (run with torchrun on >= 2 GPUs): data-parallel training over G ranks with a global batch of 1024
reproduces the single-GPU run of the same global batch (same permutation, global loss divisor, summed gradients, global
GradScaler decision), and image-sharded registration returns the same poses as one rank."""
import os
import sys
from types import SimpleNamespace

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from acezero_b200.head import HeadEngine  # noqa: E402
from acezero_b200.trainer import TrainLoop  # noqa: E402
from acezero_b200 import dsac, parallel  # noqa: E402
from oracle import ace_ref, dsacstar_ref as D  # noqa: E402  (deterministic inputs only)
import bench  # noqa: E402


def run(world, rank, dev, iters=40):
    o = bench.options(1024, iterations=1000)
    peers = dist.group.WORLD if (world > 1 and os.environ.get("ACEZ_DP_PEERS", "1") != "0") else None
    head = HeadEngine(1, True, (0, 0, 0), max_rows=1024 // world, training=True, device=dev, peer_group=peers)
    head.load_state(ace_ref.make_head_state(200, 1, True))
    buf = bench.synth_buffer(65536, dev, 7)
    loop = TrainLoop(head, o, buf, rank=rank, world_size=world, use_graph=False)
    perm = torch.randperm(65536, generator=loop.training_generator)
    losses = []
    for i in range(iters):
        loop.train_iteration(perm[i * 1024:(i + 1) * 1024], want_stats=True)
        losses.append(float(loop.last_stats[0]))
    head.gather_params_from_shards()
    if rank == 0 and world > 1:
        print(f"[dp{world}] gradient exchange: {'NVLink peer memory (adamw_dp.cu)' if loop._dp_peers else 'NCCL all-reduce'}"
              f"{', NVLink SHARP multicast (multimem.ld_reduce / multimem.st)' if getattr(head, 'dp_multicast', None) is not None else ''}")
    return losses, head.params.clone(), float(head.scaler_state[0])


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    l_dp, p_dp, s_dp = run(world, rank, dev)
    ok = True
    if rank == 0:
        l_1, p_1, s_1 = run(1, 0, dev)
        rel = max(abs(a - b) / abs(b) for a, b in zip(l_dp, l_1))
        upd = (p_dp - p_1).norm() / (p_1 - HeadEngine(1, True, (0, 0, 0), max_rows=128, device=dev).params).norm()
        print(f"[dp{world}] loss trajectory max rel diff vs 1 GPU: {rel:.3e}; scale {s_dp} vs {s_1}; "
              f"param diff / param norm {float((p_dp - p_1).norm() / p_1.norm()):.3e}")
        ok &= rel < 2e-2 and s_dp == s_1
    # all ranks hold identical parameters after training
    ref = p_dp.clone()
    dist.broadcast(ref, 0)
    same = torch.equal(ref, p_dp)
    t = torch.tensor([int(same)], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    if rank == 0:
        print(f"[dp{world}] parameters bit-identical across ranks: {bool(t.item())}")
        ok &= bool(t.item())
    # registration: sharded == single
    maps = np.concatenate([D.synth_scene(300 + i)[0] for i in range(8)], 0)
    mine = [i for i in range(8) if parallel.image_owner(i, world) == rank]
    res = []
    for i in mine:
        p, n = dsac.forward_rgb_batch(torch.from_numpy(maps[i:i + 1]).to(dev), 525.0, 320.0, 240.0, 64, seed=5, max_tries=16,
                                      image_index_base=i)
        res.append({"index": i, "pose": p[0].cpu().numpy(), "inliers": int(n[0]), "file": str(i), "focal": 525.0})
    # ---- timing of the data-parallel optimiser step alone (10 steps per CUDA graph replay; all ranks in lockstep) ----
    if world > 1 and os.environ.get("ACEZ_DP_PEERS", "1") != "0":
        o = bench.options(5120 * world, iterations=1000)
        head = HeadEngine(1, True, (0, 0, 0), max_rows=5120, training=True, device=dev, peer_group=dist.group.WORLD)
        head.load_state(ace_ref.make_head_state(200, 1, True))
        buf = bench.synth_buffer(3 * 5120 * world, dev, 7)
        loop = TrainLoop(head, o, buf, rank=rank, world_size=world, use_graph=False)
        perm = torch.randperm(3 * 5120 * world, generator=loop.training_generator)
        for i in range(3):
            loop.train_iteration(perm[i * 5120 * world:(i + 1) * 5120 * world])
        torch.cuda.synchronize()
        dist.barrier()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(10):
                head.adamw_step_peers()
        g.replay()
        torch.cuda.synchronize()
        dist.barrier()
        e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
        e0.record()
        for _ in range(10):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 10.0   # ms / 100 steps -> us per step
        st = head.peer["reduced"][:16].view(torch.int64).cpu().numpy()
        if rank == 0 and st[0] > 0:
            d = [(int(st[i]) - int(st[0])) / 1000.0 for i in range(8)]
            print(f"[dp{world}] phases of the last fused optimiser kernel (us after its start, %globaltimer): gradients of all ranks ready {d[1]:.1f}, "
                  f"reduced + checked {d[2]:.1f}, global verdict {d[3]:.1f}, stored {d[4]:.1f}, block-0 fence {d[5]:.1f}, "
                  f"last block signalled {d[6]:.1f}, all ranks' weights landed {d[7]:.1f}")
        if rank == 0:
            print(f"[dp{world}] optimiser step over peer memory alone (reduce + apply, in-kernel signals): "
                  f"{us:.1f} us per step (single-GPU AdamW kernel: ~16.5 us)")
        del loop, head
    merged = parallel.gather_registration(res, world)
    if rank == 0:
        p, n = dsac.forward_rgb_batch(torch.from_numpy(maps).to(dev), 525.0, 320.0, 240.0, 64, seed=5, max_tries=16)
        same = all(np.array_equal(m["pose"], p[m["index"]].cpu().numpy()) and m["inliers"] == int(n[m["index"]]) for m in merged)
        print(f"[dp{world}] sharded registration == single batch: {same}")
        ok &= same
        print("RESULT", "PASS" if ok else "FAIL")
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
