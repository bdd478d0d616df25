#!/usr/bin/env python
"""Benchmark of the ACE Zero hot path on B200 (BASELINE.json metric: ACE training iters/s + dsacstar poses/s).

    python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a path
    python bench.py --impl reference --steps K --warmup W    # the reference's algorithm on the host cores (oracle port)
    python bench.py --steps K --warmup W --dump-outputs DIR  # also write what the timed steps computed, DIR/<name>.npy

The sm_100a path loads the libacez.so that `python -m acezero_b200.build` left in the tree and writes nothing there.

One JSON line on stdout (rank 0). A "step" is one ACE training iteration over a 5120-patch batch (head forward, fused
reprojection loss, backward, GradScaler + AdamW; reference ace_trainer.py:499-640); the DSAC* pose solve
(dsacstar.forward_rgb, 64 hypotheses, 60x80 scene-coordinate maps) is timed in the same run and reported under "dsac".

Workload = BASELINE.json configs[1] ("7-Scenes 'chess' synthetic: ACE head training + register_mapping on 1 B200"):
synthetic patch buffer of 1 024 000 rows x 1230 B (1.26 GB, larger than L2; rows are drawn through the epoch
permutation, so every batch gathers fresh rows from HBM), head with num_head_blocks=1, homogeneous output, dyntanh
loss, one-cycle lr, fp16 autocast semantics + GradScaler. Multi-GPU: weak scaling — every rank trains on its own
5120-patch shard of a 5120*N global batch (the loss divisor is the global batch, gradients are all-reduced over NCCL);
DSAC* images are sharded across ranks with no collective.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
from types import SimpleNamespace

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

B = 5120
BUFFER_ROWS = 1_024_000
FLOP_PER_ITER = 61.80e9          # SURVEY §8d: 12.07 MFLOP / patch x 5120
FLOP_FWD_GEMM = 2 * 5120 * 512 * 512   # one hidden-layer GEMM launch
DSAC_HYPS = 64
DSAC_H, DSAC_W = 60, 80
ENC_BATCH = 8
# encoder MACs per 480x640 image (ace_network.py:14-59): conv1..4 + res1 + res2, 2 FLOP per MAC
ENC_FLOP_PER_IMAGE = 2.0 * (9 * 32 * 480 * 640 + 9 * 32 * 64 * 240 * 320 + 9 * 64 * 128 * 120 * 160 + 4800 * (
    9 * 128 * 256 + 9 * 256 * 256 + 256 * 256 + 9 * 256 * 256 + 9 * 256 * 512 + 512 * 512 + 9 * 512 * 512 + 256 * 512))
DSAC_BATCH = 1024                # images per batched solver call


def options(b_global, iterations=5000):
    return SimpleNamespace(
        batch_size=b_global, base_seed=2089, use_half=True, iterations=iterations, iterations_output=10 ** 9,
        learning_rate_schedule="circle", learning_rate_min=0.0005, learning_rate_max=0.005,
        learning_rate_warmup_iterations=1000, learning_rate_warmup_learning_rate=0.0005,
        learning_rate_cooldown_iterations=5000, learning_rate_cooldown_trigger_percent_threshold=0.7,
        learning_rate_cooldown_trigger_px_threshold=10, repro_loss_type="dyntanh", repro_loss_schedule="circle",
        repro_loss_soft_clamp=50, repro_loss_soft_clamp_min=1, repro_loss_hard_clamp=1000, depth_min=0.1,
        depth_max=1000.0, depth_target=10.0)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "hbm_gbs": d["hbm_gbs"], "source": "MEASURED_PEAKS.json (measured)"}
    return {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i] == "Active" for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------------------
# synthetic data
# ----------------------------------------------------------------------------------------------------------------
def synth_buffer(rows, device, seed):
    """Patch buffer with the reference's layout (ace_trainer.py:330-340), generated on the device."""
    g = torch.Generator(device=device).manual_seed(seed)
    n_img = 1000
    ang = torch.rand((n_img, 3), device=device, generator=g) - 0.5
    cx, sx = torch.cos(ang[:, 0]), torch.sin(ang[:, 0])
    cy, sy = torch.cos(ang[:, 1]), torch.sin(ang[:, 1])
    cz, sz = torch.cos(ang[:, 2]), torch.sin(ang[:, 2])
    R = torch.stack([cz * cy, cz * sy * sx - sz * cx, cz * sy * cx + sz * sx,
                     sz * cy, sz * sy * sx + cz * cx, sz * sy * cx - cz * sx,
                     -sy, cy * sx, cy * cx], 1).view(n_img, 3, 3)
    T = torch.eye(4, device=device).repeat(n_img, 1, 1)
    T[:, :3, :3] = R
    T[:, :3, 3] = torch.rand((n_img, 3), device=device, generator=g) - 0.5
    T[:, 2, 3] = 2 + 2 * torch.rand(n_img, device=device, generator=g)
    img = torch.randint(0, n_img, (rows,), device=device, generator=g)
    a = (torch.rand(rows, device=device, generator=g) - 0.5) * 0.52
    aug = torch.zeros((rows, 3, 4), device=device)
    aug[:, 0, 0], aug[:, 0, 1], aug[:, 1, 0], aug[:, 1, 1], aug[:, 2, 2] = torch.cos(a), -torch.sin(a), torch.sin(a), torch.cos(a), 1.0
    sc = 2 / 3 + torch.rand(rows, device=device, generator=g) * (3 / 2 - 2 / 3)
    K = torch.zeros((rows, 3, 3), device=device)
    K[:, 0, 0] = K[:, 1, 1] = 525.0 * sc
    K[:, 0, 2], K[:, 1, 2], K[:, 2, 2] = 320.0 * sc, 240.0 * sc, 1.0
    Kinv = torch.zeros_like(K)
    Kinv[:, 0, 0] = Kinv[:, 1, 1] = 1.0 / K[:, 0, 0]
    Kinv[:, 0, 2], Kinv[:, 1, 2], Kinv[:, 2, 2] = -K[:, 0, 2] / K[:, 0, 0], -K[:, 1, 2] / K[:, 0, 0], 1.0
    px = torch.stack([8 * (torch.randint(0, 80, (rows,), device=device, generator=g) + 0.5),
                      8 * (torch.randint(0, 60, (rows,), device=device, generator=g) + 0.5)], 1).float()
    return {
        "features": (torch.randn((rows, 512), device=device, generator=g) * 0.5).half(),
        "target_px": px, "aug_poses_inv": aug, "poses_inv": T[img].contiguous(), "intrinsics": K,
        "intrinsics_inv": Kinv, "target_crds": torch.zeros((rows, 3), device=device),
        "pose_idx": img.to(torch.int16).view(-1, 1),
    }


def synth_scene_maps(n, seed):
    """n scene-coordinate maps [n,3,60,80] with known poses (SURVEY §8d config 5 generator, via the oracle module's
    numpy code path; a data generator, not a checker)."""
    from oracle import dsacstar_ref as D
    base = [D.synth_scene(seed + i)[0] for i in range(16)]
    sc = np.concatenate(base, 0)
    reps = (n + 15) // 16
    return np.tile(sc, (reps, 1, 1, 1))[:n]


# ----------------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline (oracle port on the host cores)
# ----------------------------------------------------------------------------------------------------------------
CPU_ROWS = B     # rows per reference step: the FULL 5120-patch batch (same config as the GPU arm; ~0.2-0.5 s per step)


def _best_thread_count():
    """The reference's PyTorch CPU path is fastest well below the core count of a 100+-core host: pick the thread
    count that maximises throughput on a short probe (all the host threads it can *use*)."""
    from oracle import ace_ref
    cores = os.cpu_count() or 1
    sd = ace_ref.make_head_state(200, 1, True)
    bt = ace_ref.synth_batch(600, CPU_ROWS)
    best, best_t = 1, 1e9
    for n in sorted({min(8, cores), 16, 32, 64, cores}):
        if n > cores:
            continue
        torch.set_num_threads(n)
        tr = ace_ref.TrainerRef(sd, 1, True, ace_ref.LossOptions(iterations=5000), lambda i: 1e-3, emulate_half=False)
        args = (bt["features"].float(), bt["target_px"], bt["aug_poses_inv"], bt["poses_inv"], bt["intrinsics"],
                bt["intrinsics_inv"], bt["target_crds"])
        tr.step(*args)
        t0 = time.perf_counter()
        tr.step(*args); tr.step(*args)
        dt = (time.perf_counter() - t0) / 2
        if dt < best_t:
            best, best_t = n, dt
    return best


def cpu_train_iters_per_s(steps, warmup, threads=None, min_seconds=0.0, max_steps=400):
    """Reference trainer port on the host cores. One step = one full training iteration over 5120 patches (forward, loss,
    backward, AdamW over the 2.1 M head parameters): iterations/s."""
    from oracle import ace_ref
    threads = threads or _best_thread_count()
    torch.set_num_threads(threads)
    sd = ace_ref.make_head_state(200, 1, True)
    o = ace_ref.LossOptions(iterations=5000)
    tr = ace_ref.TrainerRef(sd, 1, True, o, ace_ref.one_cycle_lr(0.005, 5000), emulate_half=False)
    bts = [ace_ref.synth_batch(600 + i, CPU_ROWS) for i in range(4)]

    def one(i):
        bt = bts[i % 4]
        tr.step(bt["features"].float(), bt["target_px"], bt["aug_poses_inv"], bt["poses_inv"], bt["intrinsics"],
                bt["intrinsics_inv"], bt["target_crds"])
    for i in range(warmup):
        one(i)
    t0 = time.perf_counter()
    done = 0
    while done < steps or (time.perf_counter() - t0 < min_seconds and done < max_steps):
        one(done)
        done += 1
    dt = time.perf_counter() - t0
    cpu_train_iters_per_s.last_steps = done
    return done / dt * CPU_ROWS / B, dt, threads


def cpu_dsac_poses_per_s(n_poses):
    from oracle import dsacstar_ref as D
    import cv2
    cv2.setNumThreads(os.cpu_count())
    scenes = [D.synth_scene(100 + i) for i in range(min(n_poses, 8))]
    D.forward_rgb(scenes[0][0], DSAC_HYPS, 10.0, 525.0, 320.0, 240.0, 100.0, 100.0, 8, 1, 16)
    t0 = time.perf_counter()
    for i in range(n_poses):
        sc, _, f, px, py = scenes[i % len(scenes)]
        D.forward_rgb(sc, DSAC_HYPS, 10.0, f, px, py, 100.0, 100.0, 8, 1 + i, 16)
    dt = time.perf_counter() - t0
    return n_poses / dt, dt


def torch_gpu_train_iters_per_s(dev, buf, steps, warmup):
    """SURVEY section 8(d)(iii): the reference's OWN execution path on the same B200 — eager PyTorch, cuDNN 1x1 convolutions
    on the (b/512, 512, 16, 32) view under fp16 autocast, autograd, torch.amp.GradScaler, torch.optim.AdamW, OneCycleLR
    (ace_trainer.py:499-640, ace_network.py:120-149, ace_schedule.py:106-126), batch rows gathered from the GPU-resident
    buffer with CPU index tensors as ace_trainer.py:485-494 does. The loss is the restated ace_trainer.py:521-613 of the
    oracle module (same tensor ops, same host syncs). This is the on-box bar for the hand-written kernels; it runs none of
    them. Returns (iterations/s, ms per iteration)."""
    from oracle import ace_ref
    import torch.nn as nn
    import torch.nn.functional as F

    class HeadTorch(nn.Module):
        def __init__(self, sd):
            super().__init__()
            names = ace_ref.head_layer_names(1)
            self.convs = nn.ModuleList([nn.Conv2d(512, 512, 1) for _ in names])
            self.fc3 = nn.Conv2d(512, 4, 1)
            with torch.no_grad():
                for c, n in zip(self.convs, names):
                    c.weight.copy_(sd[n + ".weight"]); c.bias.copy_(sd[n + ".bias"])
                self.fc3.weight.copy_(sd["fc3.weight"]); self.fc3.bias.copy_(sd["fc3.bias"])
            self.h_beta, self.max_inv, self.min_inv = float(sd["h_beta"]), float(sd["max_inv_scale"]), float(sd["min_inv_scale"])

        def forward(self, res):                                   # ace_network.py:120-149
            c = self.convs
            x = F.relu(c[0](res)); x = F.relu(c[1](x)); x = F.relu(c[2](x)); res = res + x
            x = F.relu(c[3](res)); x = F.relu(c[4](x)); x = F.relu(c[5](x)); res = res + x
            sc = F.relu(c[6](res)); sc = F.relu(c[7](sc)); sc = self.fc3(sc)
            h = F.softplus(sc[:, 3:4], beta=self.h_beta) + self.max_inv
            h = torch.clamp(h, max=self.min_inv)
            return sc[:, :3] / h

    torch.backends.cudnn.benchmark = False                        # ace_trainer.py:295 leaves it off
    net = HeadTorch(ace_ref.make_head_state(200, 1, True)).to(dev)
    n_total = steps + warmup + 8
    opt = torch.optim.AdamW(net.parameters(), lr=0.0005)
    sched = torch.optim.lr_scheduler.OneCycleLR(opt, max_lr=0.005, total_steps=max(5000, n_total + 1), cycle_momentum=False)
    scaler = torch.amp.GradScaler("cuda")
    o = ace_ref.LossOptions(iterations=5000)
    gen = torch.Generator().manual_seed(2089 + 8191)
    rows = buf["features"].shape[0]
    perm = torch.randperm(rows, generator=gen)

    def one(i):
        idx = perm[(i * B) % (rows - B):(i * B) % (rows - B) + B]                              # CPU indices (:469-477)
        feats = buf["features"][idx].contiguous()                                              # :485-494
        tpx = buf["target_px"][idx].contiguous(); aug = buf["aug_poses_inv"][idx].contiguous()
        pinv = buf["poses_inv"][idx].contiguous(); K = buf["intrinsics"][idx].contiguous()
        Kinv = buf["intrinsics_inv"][idx].contiguous(); crds = buf["target_crds"][idx].contiguous()
        with torch.autocast("cuda", dtype=torch.float16):
            x = feats[None, None, ...].view(-1, 16, 32, 512).permute(0, 3, 1, 2)                # :516
            pred = net(x)
        pred = pred.permute(0, 2, 3, 1).flatten(0, 2).float()                                  # :521
        loss, inl, nv = ace_ref.training_loss(o, pred, tpx, aug, pinv, K, Kinv, crds, i)
        opt.zero_grad(set_to_none=True)
        scaler.scale(loss).backward()
        scaler.step(opt)
        scaler.update()
        sched.step()
        return float(loss)                                                                     # :615 (the reference's sync)

    for i in range(warmup):
        one(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        one(warmup + i)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return 1000.0 / ms, ms


def dsac_roofline(score_ms, n_img, clk):
    """Sampling + scoring kernel of DSAC* (refinement off): algorithmic work per (hypothesis, cell) = 45 FLOP + 4 MUFU
    (rcp, rsqrt, ex2, rcp) against the CUDA-core peaks of the chip at the clock the run saw (no tensor cores, not HBM)."""
    mhz = (clk or {}).get("sm_mhz") or 1965.0
    pairs = n_img * DSAC_HYPS * DSAC_H * DSAC_W
    t = score_ms * 1e-3
    fma_peak = 148 * 128 * 2 * mhz * 1e6          # FP32 FLOP/s
    mufu_peak = 148 * 16 * mhz * 1e6              # MUFU ops/s
    flops, mufu = 45.0 * pairs / t, 4.0 * pairs / t
    return {"bound": "fp32 issue (FFMA + MUFU), CUDA cores", "kernel": "dsac_sample_score_kernel (max_refine_steps = 0)",
            "ms_per_call": score_ms, "achieved_gflops": flops / 1e9, "peak_gflops": fma_peak / 1e9,
            "achieved_gmufu": mufu / 1e9, "peak_gmufu": mufu_peak / 1e9,
            "frac": max(flops / fma_peak, mufu / mufu_peak), "sm_mhz": mhz}


def run_pipeline(dev, H=480, W=640, focal=525.0, iterations=5000):
    """Mapping + registration of a 64-frame procedural scene through the product classes the CLIs use."""
    import tempfile
    from pathlib import Path
    from torch.utils.data import DataLoader
    import train_ace
    from ace_network import Regressor
    from ace_trainer import TrainerACE
    from acezero_b200.registration import register
    from acezero_b200.synthetic import CachedDataset, SyntheticDataset, trajectory
    from acezero_b200.weights import random_encoder_state
    logging_off()
    n = 64
    # the reference's shipped encoder weights when they are on the box (the path the CLIs default to, else the copy
    # __graft_entry__.build() stages for the parity tests); random weights otherwise
    esd, enc_kind = None, "RANDOM weights (no checkpoint on the box), which limits the angular accuracy of the learned map"
    for cand in (os.path.join(ROOT, "ace_encoder_pretrained.pt"), os.path.join(ROOT, "oracle", "_ref", "ace_encoder_pretrained.pt")):
        if os.path.exists(cand):
            try:
                esd = torch.load(cand, map_location="cpu")
                enc_kind = "the reference's pretrained weights (ace_encoder_pretrained.pt)"
                break
            except Exception:  # noqa: BLE001
                esd = None
    if esd is None:
        esd = random_encoder_state(77)
    train = CachedDataset(SyntheticDataset(n, H=H, W=W, focal=focal, device=str(dev)))
    with tempfile.TemporaryDirectory() as tmp:
        o = train_ace.build_parser().parse_args(["synthetic", str(Path(tmp) / "map.pt"), "--iterations", str(iterations),
                                                  "--use_external_focal_length", str(focal), "--iterations_output", "1000"])
        o.encoder_state_dict = esd
        o.num_data_workers = 0
        tr = TrainerACE(o, dataset=train)
        tr.train()
        timing = tr.timing
        log_last = [float(x) for x in (Path(tmp) / "map.txt").read_text().strip().splitlines()[-1].split()]
        head_sd = torch.load(Path(tmp) / "map.pt", map_location="cpu")
    net = Regressor.create_from_split_state_dict(esd, head_sd).to(dev).eval()
    test = SyntheticDataset(n, H=H, W=W, focal=focal, device=str(dev), s_offset=0.5)   # views between the mapping frames
    test.gt_poses = trajectory(n, s_offset=0.5)
    test.poses = [p.clone() for p in test.gt_poses]
    test = CachedDataset(test, keep_base=False)   # no CUDA state: the loader forks worker processes
    from acezero_b200.registration import collate_same_size
    gen = torch.Generator().manual_seed(1305)

    # what register_mapping.py builds: shuffled, batches of 8 collated by worker processes and pinned (the reference runs 12
    # workers, register_mapping.py:8,147); the workers persist across the timed passes
    ld = DataLoader(test, shuffle=True, num_workers=12, persistent_workers=True, generator=gen, batch_size=8,
                    collate_fn=collate_same_size, pin_memory=True)
    register(net, ld, hypotheses=64, max_tries=16, device=dev)   # warm-up (starts the workers)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    reps = 4
    for _ in range(reps):
        res, _ = register(net, ld, hypotheses=64, max_tries=16, device=dev)
    dt = (time.perf_counter() - t0) / reps
    rot, tra = [], []
    for r in res:
        T, G = r["pose"].astype(np.float64), test.gt_poses[r["index"]].numpy().astype(np.float64)
        dR = T[:3, :3].T @ G[:3, :3]
        rot.append(float(np.rad2deg(np.arccos(np.clip((np.trace(dR) - 1) / 2, -1, 1)))))
        tra.append(float(np.linalg.norm(T[:3, 3] - G[:3, 3])))
    ok = float(np.mean([(a < 5.0) and (b < 0.05) for a, b in zip(rot, tra)]))
    del ld
    return {
        "what": f"64 rendered {H}x{W} frames (f = {focal}): TrainerACE.train (buffer fill + {iterations} iterations) then "
                "registration.register on 64 held-out views through a shuffled DataLoader with 12 workers (host images in, host "
                f"poses out); the encoder has {enc_kind}",
        "buffer_fill_images_per_s": timing["images_encoded"] / timing["buffer_s"],
        "buffer_fill_s": timing["buffer_s"], "images_encoded": timing["images_encoded"],
        "train_iters_per_s": timing["iterations"] / timing["train_s"], "train_s": timing["train_s"],
        "final_loss": log_last[2], "final_batch_inliers": log_last[3],
        "register_poses_per_s": n / dt, "register_ms_per_image": dt / n * 1e3,
        "median_rot_deg": float(np.median(rot)), "median_trans_m": float(np.median(tra)), "acc_5cm_5deg": ok,
        "median_inliers": float(np.median([r["inliers"] for r in res])),
    }


def logging_off():
    import logging
    logging.disable(logging.INFO)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count()
    ips, dt, threads = cpu_train_iters_per_s(args.steps, args.warmup)
    pps, dt2 = cpu_dsac_poses_per_s(max(4, min(40, args.steps)))
    line = {
        "impl": "reference", "metric": "ace_train_iters_per_s", "value": ips, "unit": "iters/s (5120-patch iterations)",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 / ips,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[1] 'chess'-shaped: ACE head training (b=5120, 1 head block, homogeneous, dyntanh, "
                               "one-cycle lr) + register_mapping's DSAC* (64 hyps, 60x80 maps)", "global_batch": B,
                   "parallelism": "cpu", "arithmetic": "fp32 on the host cores (autocast / GradScaler disable themselves without CUDA)"},
        "cpu_baseline": {"value": ips, "unit": "iters/s", "cores": threads, "kind": "port",
                         "sample": f"{args.steps} full 5120-patch iterations, oracle/ace_ref.py TrainerRef = restated reference "
                                   f"trainer, torch CPU fp32, {threads} of {cores} threads (best of a thread-count probe), {dt:.1f} s"},
        "e2e": {"value": ips, "unit": "iters/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "dsac": {"poses_per_s": pps, "unit": "poses/s", "hyps": DSAC_HYPS,
                 "cpu_baseline": {"value": pps, "unit": "poses/s", "cores": cores, "kind": "port",
                                  "sample": f"cv2 restatement (oracle/dsacstar_ref.py), {dt2:.1f} s"},
                 "e2e": {"value": pps, "unit": "poses/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------
# this repo's arm
# ----------------------------------------------------------------------------------------------------------------
def dump_outputs(out_dir, arrays):
    """Write each array as out_dir/<name>.npy (float32 or float64, 64 MB at most in all), so that two builds run with the
    same arguments can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        a = a.astype(np.float64 if a.dtype.kind in "iu" or a.dtype == np.float64 else np.float32)
        total += a.nbytes
        np.save(os.path.join(out_dir, name + ".npy"), a)
    assert total <= 64 << 20, total


def run_ours(args):
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        dist.barrier()
    from acezero_b200.head import HeadEngine
    from acezero_b200.trainer import TrainLoop, BUFFER_KEYS
    from acezero_b200 import dsac
    from oracle import ace_ref  # only for the deterministic head-state generator (numpy) and the cpu_baseline leg

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    # ---------------- training ----------------
    o = options(B * world, max(5000, 2 * (args.steps + args.warmup + 400)))
    peers = dist.group.WORLD if (world > 1 and os.environ.get("ACEZ_DP_PEERS", "1") != "0") else None
    head = HeadEngine(1, True, (0.0, 0.0, 0.0), max_rows=B, training=True, device=dev, peer_group=peers)
    head.load_state(ace_ref.make_head_state(200, 1, True))
    buf = synth_buffer(BUFFER_ROWS, dev, 2089)   # identical on every rank (same seed), as the replicated buffer is
    loop = TrainLoop(head, o, buf, rank=rank, world_size=world, use_graph=True)
    perm = torch.randperm(BUFFER_ROWS, generator=loop.training_generator)
    bg = B * world
    n_batches = BUFFER_ROWS // bg
    it = [0]

    def step():
        s = (it[0] % n_batches) * bg
        assert loop.train_iteration(perm[s:s + bg]), "the schedule ended inside the benchmark"
        it[0] += 1

    for _ in range(max(args.warmup, 3) + 2):   # +2: the CUDA graph is captured on the third call
        step()
    barrier()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    ms_per_step = ms_total / args.steps
    iters_per_s = world * 1000.0 / ms_per_step      # 5120-patch iterations per second, whole job
    loss_final = float(head.stats[0])
    # what the last timed training step leaves its caller (the sections below train further on the same head): the fp32
    # head parameters and this rank's [loss sum, inlier count, valid count, non-finite flag]
    outputs = {"train_head_params": head.params.clone(), "train_stats": head.stats.clone()}

    # ---------------- strong scaling: the SAME global batch of 5120 split over the ranks (what train_ace.py semantics mean:
    # --batch_size is the global batch; ace_trainer.py:613 divides by it) ----------------
    strong = None
    if world > 1 and B % world == 0:
        o_s = options(B, max(5000, 2 * (args.steps + args.warmup + 400)))
        head_s = HeadEngine(1, True, (0.0, 0.0, 0.0), max_rows=B // world, training=True, device=dev, peer_group=peers)
        head_s.load_state(ace_ref.make_head_state(200, 1, True))
        loop_s = TrainLoop(head_s, o_s, buf, rank=rank, world_size=world, use_graph=True)
        n_b = BUFFER_ROWS // B
        its = [0]

        def step_s():
            st = (its[0] % n_b) * B
            loop_s.train_iteration(perm[st:st + B])
            its[0] += 1
        for _ in range(max(args.warmup, 3) + 2):
            step_s()
        barrier()
        e0.record()
        for _ in range(args.steps):
            step_s()
        e1.record()
        barrier()
        ms_s = max_over_ranks(e0.elapsed_time(e1)) / args.steps
        strong = {"scaling": "strong", "global_batch": B, "rows_per_rank": B // world, "ms_per_step": ms_s,
                  "value": 1000.0 / ms_s, "unit": "iters/s (5120-patch iterations, global batch fixed)"}
        del loop_s, head_s

    # ---------------- end-to-end (host buffers in, loss out) ----------------
    host_batches = []
    for i in range(4):
        idx = perm[i * B:(i + 1) * B].to(dev)
        hb = loop.new_host_batch()             # pinned, packed: one host->device copy per step
        for k in BUFFER_KEYS:
            hb[k].copy_(buf[k][idx])
        host_batches.append(hb)
    torch.cuda.synchronize()
    h2d = sum(host_batches[0][k].numel() * host_batches[0][k].element_size() for k in BUFFER_KEYS)
    for i in range(4):
        loop.train_step_from_host(host_batches[i % 4])
    barrier()
    n_e2e = max(10, min(args.steps, 200))
    # every step: H2D copy of ITS batch from pinned host memory (issued one step ahead on a copy stream so that it
    # overlaps the previous step's compute), the training step, and a D2H read of the loss statistics: the host reads
    # step i-1's loss while step i runs (lag 1; the last one is drained inside the timed region), so no step's result
    # is skipped and the device never waits for the host
    loop.prefetch_host_batch(host_batches[0])
    for i in range(4):
        loop.prefetch_host_batch(host_batches[(i + 1) % 4])
        loop.train_step_prefetched(lag=1)
    loop.drain_prefetched()
    barrier()
    t0 = time.perf_counter()
    n_read = 0
    for i in range(n_e2e):
        loop.prefetch_host_batch(host_batches[(i + 1) % 4])
        n_read += loop.train_step_prefetched(lag=1) is not None
    n_read += loop.drain_prefetched() is not None
    torch.cuda.synchronize()
    assert n_read == n_e2e or world > 1, (n_read, n_e2e)
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1000.0 / n_e2e)
    e2e_ips = world * 1000.0 / e2e_ms

    # ---------------- roofline of the dominant kernel: the hidden-layer forward GEMM (tcgen05) ----------------
    g = torch.cuda.CUDAGraph()
    reps = 10
    feats = host_batches[0]["features"].to(dev)
    head.input_buffer(B).copy_(feats)
    lib = head.lib
    from acezero_b200 import _lib
    for _ in range(2):
        _lib.check(lib.acez_head_forward(head.plan, None, B, None, _lib.stream_ptr()))
    torch.cuda.synchronize()
    with torch.cuda.graph(g):
        for _ in range(reps):
            _lib.check(lib.acez_head_forward(head.plan, None, B, None, _lib.stream_ptr()))
    g.replay()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(5):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    pk = peaks()
    chain = head.fused_chain
    if chain:
        # one launch = all 8 hidden layers of the forward pass (head_chain.cu)
        gemm_us = e0.elapsed_time(e1) * 1000.0 / (5 * reps)
        achieved_tf = head.L * FLOP_FWD_GEMM / (gemm_us * 1e-6) / 1e12
        roof_kernel = (f"{head.chain_kernel_symbol()}: {head.L} fused layers of 5120x512x512 in one launch (cluster of 4 CTAs = two 128-row "
                       "tiles x two channel halves, tcgen05 cta_group::2)")
        launches = {"gather": 1, "fwd_chain": 1, "tail": 1, "fc3_reduce": 1,
                    "dgrad_chain": 1, "wgrad_gemm": 1, "adamw": 1}
    else:
        gemm_us = e0.elapsed_time(e1) * 1000.0 / (5 * reps * head.L)
        achieved_tf = FLOP_FWD_GEMM / (gemm_us * 1e-6) / 1e12
        roof_kernel = "gemm_tcgen05_kernel<256,K,K,FWD> 5120x512x512"
        launches = {"gather": 1, "fwd_gemm": 8, "tail": 1, "fc3_reduce": 1,
                    "dgrad_gemm": 7, "wgrad_gemm": 1, "adamw": 1}
    clk = clocks.stop() if rank == 0 else None
    # DRAM traffic of the roofline kernel from the committed `ncu --set full` capture (profiles/), per launch
    traffic = None
    try:
        # only a capture of the kernel that is timed here counts (round 1 read a stale constant): the file names the kernel symbol
        tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic_r02.json")))
        if chain and tj.get("kernel_symbol") == head.chain_kernel_symbol():
            traffic = int(tj["dram_bytes_per_launch"])   # bytes; algorithmic: 9 tiles x 5.24 MB + 4.19 MB of fp16 weights
    except Exception:
        traffic = None

    # ---------------- DSAC* ----------------
    n_img = DSAC_BATCH
    maps_host = torch.from_numpy(synth_scene_maps(n_img, 1000 + rank * n_img)).pin_memory()
    maps = maps_host.to(dev)
    kw = dict(hyps=DSAC_HYPS, inlier_threshold=10.0, inlier_alpha=100.0, max_reproj=100.0, subsample=8, seed=2089,
              max_tries=16, image_index_base=rank * n_img)
    for _ in range(3):
        dsac.forward_rgb_batch(maps, 525.0, 320.0, 240.0, **kw)
    barrier()
    e0.record()
    d_steps = max(3, min(args.steps, 20))
    for _ in range(d_steps):
        d_poses, d_inliers = dsac.forward_rgb_batch(maps, 525.0, 320.0, 240.0, **kw)
    e1.record()
    barrier()
    dsac_ms = max_over_ranks(e0.elapsed_time(e1) / d_steps)
    outputs.update(dsac_poses=d_poses, dsac_inliers=d_inliers)
    poses_per_s = world * n_img * 1000.0 / dsac_ms
    # end to end: host scene coordinates in, host poses out
    t0 = time.perf_counter()
    for _ in range(d_steps):
        p, n = dsac.forward_rgb_batch(maps_host.to(dev, non_blocking=True), 525.0, 320.0, 240.0, **kw)
        p_h, n_h = p.cpu(), n.cpu()
    dsac_e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1000.0 / d_steps)

    # ---------------- encoder + head inference (the buffer-fill / registration front end, SURVEY.md §8 "next") ----------
    from acezero_b200.encoder import EncoderEngine
    from acezero_b200.weights import random_encoder_state
    n_enc = ENC_BATCH
    enc = EncoderEngine(random_encoder_state(7), max_n=n_enc, max_h=480, max_w=640, device=dev)
    inf_head = HeadEngine(1, True, (0.0, 0.0, 0.0), max_rows=n_enc * 4800, training=False, device=dev)
    inf_head.load_state(ace_ref.make_head_state(200, 1, True))
    img_host = (torch.rand((4, n_enc, 1, 480, 640), generator=torch.Generator().manual_seed(3)) - 0.4).half().pin_memory()
    img_dev = img_host.to(dev)
    f_enc = torch.empty((n_enc, 60, 80, 512), device=dev, dtype=torch.float16)
    sc_enc = torch.empty((n_enc * 4800, 3), device=dev, dtype=torch.float32)

    def enc_step(img):
        enc.forward_nhwc(img, out=f_enc)
        inf_head.forward(f_enc.view(-1, 512), out=sc_enc)

    for i in range(3):
        enc_step(img_dev[i % 4])
    barrier()
    e_steps = max(5, min(args.steps, 40))
    e0.record()
    for i in range(e_steps):
        enc_step(img_dev[i % 4])
    e1.record()
    barrier()
    enc_ms = max_over_ranks(e0.elapsed_time(e1) / e_steps)
    outputs["encoder_head_scene_coords"] = sc_enc.clone()
    e0.record()
    for i in range(e_steps):
        enc.forward_nhwc(img_dev[i % 4], out=f_enc)
    e1.record()
    barrier()
    enc_only_ms = max_over_ranks(e0.elapsed_time(e1) / e_steps)
    sc_host = torch.empty((n_enc * 4800, 3), dtype=torch.float32).pin_memory()
    t0 = time.perf_counter()
    for i in range(e_steps):
        enc_step(img_host[i % 4].to(dev, non_blocking=True))
        sc_host.copy_(sc_enc, non_blocking=True)
        torch.cuda.current_stream().synchronize()
    enc_e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1000.0 / e_steps)

    # ---------------- DSAC*: scoring-only time (roofline of the warp-per-hypothesis kernel) and the hypothesis sweep ----------
    def time_dsac(m, hyps, refine_steps, reps):
        kw2 = dict(kw); kw2["hyps"] = hyps
        for _ in range(2):
            dsac.forward_rgb_batch(m, 525.0, 320.0, 240.0, max_refine_steps=refine_steps, **kw2)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            dsac.forward_rgb_batch(m, 525.0, 320.0, 240.0, max_refine_steps=refine_steps, **kw2)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps
    score_ms = time_dsac(maps, DSAC_HYPS, 0, 5)          # sampling + scoring (+ argmax): no refinement rounds
    sweep = {}
    n_sw = 256
    for hy in (64, 256, 1024, 4096):
        sweep[str(hy)] = world * n_sw * 1000.0 / max_over_ranks(time_dsac(maps[:n_sw], hy, 100, 2))

    # ---------------- configs[1] in miniature THROUGH THE PRODUCT ENTRY POINTS: TrainerACE.train (buffer fill + training loop)
    # and registration.register (shuffled loader -> encoder + head + DSAC*), pose accuracy against ground truth -------------
    pipe = None
    if world == 1 and not args.no_pipeline:
        pipe = {"480x640": run_pipeline(dev, 480, 640, 525.0), "240x320": run_pipeline(dev, 240, 320, 262.5)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    # ---------------- the reference's PyTorch path on this same GPU (rank 0, N = 1 only; SURVEY 8(d)(iii)) ----------------
    torch_gpu = None
    if world == 1 and not args.no_torch_baseline:
        try:
            t_ips, t_ms = torch_gpu_train_iters_per_s(dev, buf, 40, 8)
            torch_gpu = {"value": t_ips, "unit": "iters/s", "ms_per_step": t_ms, "kind": "port",
                         "what": "eager PyTorch restatement of ace_trainer.py:499-640 on this GPU: nn.Conv2d 1x1 head (cuDNN/cuBLAS) "
                                 "under fp16 autocast, autograd, torch.amp.GradScaler, AdamW, OneCycleLR, batch gathered from the "
                                 "GPU-resident buffer with CPU indices; same 5120-patch batches, same buffer; none of this repo's kernels",
                         "ours_over_torch": iters_per_s / t_ips}
        except Exception as e:  # noqa: BLE001  (the baseline leg must never take the measurement down)
            torch_gpu = {"unavailable": f"{type(e).__name__}: {e}"[:300]}
    # ---------------- cpu baseline (bounded sample, rank 0, N = 1 only) ----------------
    cpu = cpu_d = None
    if world == 1 and not args.no_cpu_baseline:
        ips_c, dt_c, threads = cpu_train_iters_per_s(12, 2, min_seconds=10.0)   # about 10 s of CPU work, at least 12 iterations
        n_cpu = cpu_train_iters_per_s.last_steps
        pps_c, dt_d = cpu_dsac_poses_per_s(48)
        cores = os.cpu_count()
        cpu = {"value": ips_c, "unit": "iters/s", "cores": threads, "kind": "port",
               "sample": f"{n_cpu} full 5120-patch iterations, oracle/ace_ref.py (restated reference trainer, torch CPU fp32, "
                         f"{threads} of {cores} threads = best of a thread-count probe), {dt_c:.1f} s"}
        cpu_d = {"value": pps_c, "unit": "poses/s", "cores": cores, "kind": "port",
                 "sample": f"48 poses, 64 hyps, cv2 restatement oracle/dsacstar_ref.py, {dt_d:.1f} s"}
    line = {
        "metric": "ace_train_iters_per_s", "value": iters_per_s, "unit": "iters/s (5120-patch iterations)",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16 operands / f32 accumulate",
        "data": "synthetic",
        "config": {"workload": "configs[1] 'chess'-shaped: ACE head training (b=5120/GPU, 1 head block, homogeneous, dyntanh, "
                               "one-cycle lr, GradScaler) + register_mapping's DSAC* (64 hyps, 60x80 maps)",
                   "global_batch": B * world, "buffer_rows": BUFFER_ROWS, "parallelism": f"dp{world}",
                   "gradient_exchange": ("none" if world == 1 else ((
                       "NVLink peer memory, ONE kernel per step (csrc/adamw_dp.cu): reduce-scatter"
                       + (" in the NVSwitch (multimem.ld_reduce)" if getattr(head, "dp_multicast", None) is not None else " by peer loads")
                       + " + global GradScaler verdict + AdamW on the shard + fp16 weights to all ranks"
                       + (" (multimem.st)" if getattr(head, "dp_multicast", None) is not None else "")
                       + ", cross-GPU synchronisation by in-kernel epoch signals, whole iteration one CUDA graph")
                       if loop._dp_peers else "NCCL all-reduce")),
                   "l2": "inputs larger than L2 (1.26 GB patch buffer, fresh random rows gathered every step)"},
        "roofline": {"bound": "tensor", "kernel": roof_kernel,
                     "achieved": achieved_tf, "peak": pk["bf16_tflops"], "unit": "TFLOP/s",
                     "frac": achieved_tf / pk["bf16_tflops"], "traffic": traffic, "us_per_launch": gemm_us,
                     "peak_source": pk["source"] + " burst bf16 (kernel timed alone)",
                     "step_frac_of_sustained": FLOP_PER_ITER / (ms_per_step * 1e-3) / 1e12 / pk["bf16_tflops_sustained"]},
        "cpu_baseline": cpu,
        "torch_gpu_baseline": torch_gpu,
        "strong": strong,
        "e2e": {"value": e2e_ips, "unit": "iters/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 16,
                "ms_per_step": e2e_ms},
        "gpu_launches": args.steps * sum(launches.values()),
        "launches_per_step": launches,
        "loss_final": loss_final,
        "dsac": {"poses_per_s": poses_per_s, "unit": "poses/s", "hyps": DSAC_HYPS, "images_per_call": n_img,
                 "ms_per_call": dsac_ms, "gpu_launches_per_call": 2,
                 "e2e": {"value": world * n_img * 1000.0 / dsac_e2e_ms, "unit": "poses/s",
                         "h2d_bytes_per_step": n_img * 3 * DSAC_H * DSAC_W * 4, "d2h_bytes_per_step": n_img * 68},
                 "cpu_baseline": cpu_d,
                 "work": "13.8 MFLOP + 307 k exp per pose (scoring) + refinement; FP32 FMA / MUFU issue bound, 57.6 KB in / 68 B out",
                 "roofline": dsac_roofline(score_ms, n_img, clk),
                 "hyps_sweep_poses_per_s": sweep, "hyps_sweep_images_per_call": n_sw},
        "pipeline": pipe,
        "encoder": {"images_per_s": world * n_enc * 1000.0 / enc_ms, "unit": "480x640 images/s (encoder + head -> scene coordinates)",
                    "images_per_call": n_enc, "ms_per_call": enc_ms, "encoder_only_ms_per_call": enc_only_ms,
                    "encoder_tflops": ENC_FLOP_PER_IMAGE * n_enc / (enc_only_ms * 1e-3) / 1e12,
                    "encoder_frac_of_bf16_peak": ENC_FLOP_PER_IMAGE * n_enc / (enc_only_ms * 1e-3) / 1e12 / pk["bf16_tflops"],
                    "e2e": {"value": world * n_enc * 1000.0 / enc_e2e_ms, "unit": "images/s",
                            "h2d_bytes_per_step": n_enc * 480 * 640 * 2, "d2h_bytes_per_step": n_enc * 4800 * 12},
                    "gpu_launches_per_call": 11 + 9},
        "clocks": clk,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", type=str, default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-torch-baseline", action="store_true")
    ap.add_argument("--no-pipeline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed steps computed in their last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the sm_100a path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
