"""Generate tests/golden/*.npz by running the UNMODIFIED reference (from /root/reference) on CPU.

Run in the build container only (`python oracle/make_golden.py`); /root/reference does not exist on the GPU box, the
committed fixtures travel instead. What is executed is the reference's own code:
  - `ace_network.Regressor` / `Head.forward`            (ace_network.py:120-149)
  - `ace_trainer.TrainerACE.training_step`              (ace_trainer.py:499-640), called unbound on a stand-in `self`
    that carries the reference's `ScheduleACE`, `ReproLoss`, `Regressor` objects (the modules ace_trainer imports
    but that cannot be imported here — roma, skimage, pyrender via refine_poses / dataset / ace_visualizer — are
    stubbed; none of them is touched by training_step with pose refinement 'none' and no calibration refinement)
  - `ace_loss.ReproLoss.compute`                        (ace_loss.py:39-90)
On a CPU-only torch, `autocast(enabled=True)` and `GradScaler(enabled=True)` disable themselves, so the reference
computes in fp32: that is what these vectors pin (oracle mode emulate_half=False).
Inputs come from numpy RandomState generators (oracle.ace_ref.make_head_state / synth_batch), so the fixture only
needs to store the reference's outputs.
"""
import os
import sys
import types
from pathlib import Path

import numpy as np
import torch

REPO = Path(__file__).resolve().parent.parent
REF = Path("/root/reference")
sys.path.insert(0, str(REPO))

from oracle import ace_ref  # noqa: E402


def import_reference_trainer():
    sys.path.insert(0, str(REF))
    for name, attrs in {
        "refine_poses": ["PoseRefiner"],
        "dataset": ["CamLocDataset"],
        "ace_visualizer": ["ACEVisualizer"],
    }.items():
        m = types.ModuleType(name)
        for a in attrs:
            setattr(m, a, type(a, (), {}))
        sys.modules[name] = m
    import ace_trainer  # noqa: E402  (the reference's file)
    import ace_network  # noqa: E402
    import ace_loss  # noqa: E402
    import ace_schedule  # noqa: E402
    return ace_trainer, ace_network, ace_loss, ace_schedule


class _NoPoseRefiner:
    """pose_refinement == 'none' behaviour of refine_poses.PoseRefiner (refine_poses.py:212-219): poses pass through."""

    def get_current_poses(self, inv_poses_b44, idx):
        return inv_poses_b44

    def zero_grad(self, set_to_none=False):
        pass

    def step(self):
        pass


def main():
    torch.manual_seed(0)
    torch.set_num_threads(8)
    ace_trainer, ace_network, ace_loss, ace_schedule = import_reference_trainer()
    out = {}
    out["meta_torch_version"] = np.array(torch.__version__)

    # ---------------------------------------------------------------- 1. Head forward (fp32, CPU)
    for homog in (True, False):
        for nb in (1, 2):
            sd = ace_ref.make_head_state(100 + nb, nb, homog, mean=(0.3, -0.2, 1.5))
            reg = ace_network.Regressor(torch.tensor([0.3, -0.2, 1.5]), nb, homog, 512)
            reg.heads.load_state_dict(sd)
            reg.eval()
            feats = ace_ref.synth_batch(7, 512)["features"].float()
            with torch.no_grad():
                x = feats[None, None, ...].view(-1, 16, 32, 512).permute(0, 3, 1, 2)  # ace_trainer.py:516
                sc = reg.get_scene_coordinates(x).permute(0, 2, 3, 1).flatten(0, 2)   # ace_trainer.py:521
            out[f"head_sc_h{int(homog)}_b{nb}"] = sc.numpy()

    # ---------------------------------------------------------------- 1b. Encoder forward (fp32, CPU)
    for tag, (h, w) in {"96x128": (96, 128), "75x101": (75, 101)}.items():
        esd = ace_ref.make_encoder_state(77)
        enc = ace_network.Encoder(out_channels=512)
        enc.load_state_dict(esd)
        enc.eval()
        with torch.no_grad():
            f = enc(ace_ref.synth_image(5, h, w))
        out[f"encoder_{tag}_shape"] = np.array(f.shape)
        out[f"encoder_{tag}_sample"] = f.reshape(-1)[::53].numpy().copy()

    # ---------------------------------------------------------------- 2. training_step x N (fp32, CPU)
    for tag, loss_type, use_depth, sched in (("dyntanh", "dyntanh", False, "circle"), ("l1sqrt_depth", "l1+sqrt", True, "constant"),
                                              ("tanh", "tanh", False, "circle"), ("l1", "l1", False, "circle"),
                                              ("l1log", "l1+log", False, "circle")):
        nb, homog, b, iters = 1, True, 512, 4
        sd = ace_ref.make_head_state(200, nb, homog, mean=(0.0, 0.0, 0.0))
        reg = ace_network.Regressor(torch.zeros(3), nb, homog, 512)
        reg.heads.load_state_dict(sd)
        reg.train()
        opts = types.SimpleNamespace(
            learning_rate_min=0.0005, learning_rate_max=0.005, learning_rate_schedule=sched, iterations=1000,
            use_half=True, depth_min=0.1, depth_max=1000.0, depth_target=10.0, repro_loss_hard_clamp=1000,
            learning_rate_cooldown_trigger_px_threshold=10, pose_refinement_wait=0, iterations_output=10 ** 9)
        fake = types.SimpleNamespace()
        fake.options = opts
        fake.iteration = 1  # 0 would take the logging branch (ace_trainer.py:642) that needs the full trainer
        fake.regressor = reg
        fake.training_scheduler = ace_schedule.ScheduleACE(reg, opts)
        fake.pose_refiner = _NoPoseRefiner()
        fake.K_optimizer = None
        fake.use_depth = use_depth
        fake.repro_loss = ace_loss.ReproLoss(total_iterations=1000, soft_clamp=50, soft_clamp_min=1, type=loss_type,
                                             circle_schedule=True)
        fake.iterations_output = 10 ** 9
        fake.ace_visualizer = None
        losses, inliers = [], []
        orig_backward = fake.training_scheduler.backward
        orig_step = fake.training_scheduler.step

        def backward(loss, _o=orig_backward):
            losses.append(float(loss))
            _o(loss)

        def step(batch_inliers, _o=orig_step):
            inliers.append(float(batch_inliers))
            _o(batch_inliers)

        fake.training_scheduler.backward = backward
        fake.training_scheduler.step = step
        lrs = []
        for it in range(iters):
            bt = ace_ref.synth_batch(300 + it, b, with_depth=use_depth)
            lrs.append(fake.training_scheduler.optimizer.param_groups[0]["lr"])
            ace_trainer.TrainerACE.training_step(
                fake, bt["features"].float(), bt["target_px"], bt["aug_poses_inv"], bt["poses_inv"],
                bt["intrinsics"], bt["intrinsics_inv"], bt["target_crds"], bt["pose_idx"])
            fake.iteration += 1  # ace_trainer.py:495
        out[f"train_{tag}_loss"] = np.array(losses)
        out[f"train_{tag}_inliers"] = np.array(inliers)
        out[f"train_{tag}_lr"] = np.array(lrs)
        hs = reg.heads.state_dict()
        # a strided sample of every parameter after `iters` updates
        for k in ("res3_conv1.weight", "0c1.weight", "fc2.bias", "fc3.weight", "fc3.bias"):
            out[f"train_{tag}_{k}"] = hs[k].detach().reshape(-1)[::97].numpy().copy()

    # ---------------------------------------------------------------- 3. ReproLoss.compute across the schedule
    errs = torch.from_numpy(np.random.RandomState(5).uniform(0, 200, 4096).astype(np.float32))
    for t in ("tanh", "dyntanh", "l1", "l1+sqrt", "l1+log"):
        rl = ace_loss.ReproLoss(total_iterations=1000, soft_clamp=50, soft_clamp_min=1, type=t, circle_schedule=True)
        out[f"reproloss_{t}"] = np.array([float(rl.compute(errs, it)) for it in (0, 250, 999)])

    dst = REPO / "tests" / "golden" / "ace_train_golden.npz"
    dst.parent.mkdir(parents=True, exist_ok=True)
    np.savez_compressed(dst, **out)
    print("wrote", dst, os.path.getsize(dst), "bytes;", len(out), "arrays")


def pretrained_encoder_golden():
    """The reference's own `Encoder` (ace_network.py:14-59) with the weights it ships (`ace_encoder_pretrained.pt`) on two
    image sizes: pins oracle.ace_ref.encoder_forward on the real weight distribution, not only on random weights. The
    22 MB weight file is not committed: `__graft_entry__.build()` stages it into the git-ignored `oracle/_ref/`."""
    sys.path.insert(0, str(REF))
    import ace_network  # noqa: E402  (the reference's file)
    torch.set_num_threads(8)
    esd = torch.load(REF / "ace_encoder_pretrained.pt", map_location="cpu")
    enc = ace_network.Encoder(out_channels=512)
    enc.load_state_dict(esd)
    enc.eval()
    out = {"meta_torch_version": np.array(torch.__version__),
           "weights_checksum": np.array(sum(float(v.double().abs().sum()) for v in esd.values()))}
    for tag, (h, w) in {"96x128": (96, 128), "120x168": (120, 168)}.items():
        with torch.no_grad():
            f = enc(ace_ref.synth_image(11, h, w))
        out[f"encoder_{tag}_shape"] = np.array(f.shape)
        out[f"encoder_{tag}_sample"] = f.reshape(-1)[::29].numpy().copy()
        out[f"encoder_{tag}_absmax"] = np.array(float(f.abs().max()))
    dst = REPO / "tests" / "golden" / "encoder_pretrained_golden.npz"
    np.savez_compressed(dst, **out)
    print("wrote", dst, os.path.getsize(dst), "bytes")


def refine_golden():
    """The reference's `refine_poses.PoseRefiner` (refine_poses.py:85-250) in its three modes on the 7-pose dataset and the
    index batch of tests/test_refine_cpu.py: poses it returns for the batch and for the whole dataset, before and after one
    optimiser step on a fixed objective. Its `roma` dependency is stubbed with acezero_b200.refine's Gram-Schmidt /
    Procrustes, so those two functions are pinned by their own tests, not by this fixture."""
    from acezero_b200 import refine
    sys.path.insert(0, str(REF))
    roma = types.ModuleType("roma")
    roma.special_gramschmidt = refine.special_gramschmidt
    roma.special_procrustes = refine.special_procrustes
    sys.modules["roma"] = roma
    import refine_poses  # noqa: E402  (the reference's file)
    torch.set_num_threads(8)
    g = torch.Generator().manual_seed(1)
    poses = []
    for _ in range(7):
        T = torch.eye(4)
        T[:3, :3] = refine.special_procrustes(torch.randn(3, 3, generator=g))
        T[:3, 3] = torch.randn(3, generator=g)
        poses.append(T)
    ds = type("DS", (), {"poses": poses, "__len__": lambda self: len(self.poses),
                         "get_focal_length": lambda self, i: 525.0})()
    idx = torch.tensor([[3], [0], [6], [3]], dtype=torch.int32)
    orig = torch.stack([poses[i].inverse() for i in idx.view(-1).tolist()])
    out = {"meta_torch_version": np.array(torch.__version__), "dataset_poses": torch.stack(poses).numpy()}
    for mode in ("none", "naive", "mlp"):
        opts = types.SimpleNamespace(pose_refinement=mode, pose_refinement_lr=0.001, pose_refinement_weight=0.1,
                                     refinement_ortho="gram-schmidt")
        torch.manual_seed(5)
        r = refine_poses.PoseRefiner(ds, torch.device("cpu"), opts)
        r.create_pose_buffer()
        cur = r.get_current_poses(orig, idx)
        out[f"pose_{mode}_current"] = cur.detach().numpy().copy()
        out[f"pose_{mode}_all"] = r.get_all_current_poses().detach().cpu().numpy().copy()
        if mode != "none":
            r.zero_grad(set_to_none=True)
            (cur[:, :3] * torch.arange(12.).view(1, 3, 4)).sum().backward()
            r.step()
            out[f"pose_{mode}_all_after_step"] = r.get_all_current_poses().detach().cpu().numpy().copy()
    dst = REPO / "tests" / "golden" / "refine_golden.npz"
    np.savez_compressed(dst, **out)
    print("wrote", dst, os.path.getsize(dst), "bytes")


if __name__ == "__main__":
    if "--pretrained-encoder" in sys.argv:
        pretrained_encoder_golden()
    elif "--refine" in sys.argv:
        refine_golden()
    else:
        main()
        pretrained_encoder_golden()
        refine_golden()
