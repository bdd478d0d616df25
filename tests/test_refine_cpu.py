"""CPU checks of the pose / calibration refiners (acezero_b200/refine.py) — including a comparison with what the
reference's own refine_poses.PoseRefiner returns on the same inputs (tests/golden/refine_golden.npz, written by
oracle/make_golden.py; its `roma` dependency was stubbed with the restated Gram-Schmidt / Procrustes, so that part is
compared against itself)."""
import types
from pathlib import Path

import numpy as np
import pytest
import torch

from acezero_b200 import refine

GOLDEN = Path(__file__).resolve().parent / "golden" / "refine_golden.npz"


def test_special_gramschmidt_and_procrustes_are_rotations():
    g = torch.Generator().manual_seed(0)
    M = torch.randn(16, 3, 3, generator=g)
    for fn in (refine.special_gramschmidt, refine.special_procrustes):
        R = fn(M)
        assert torch.allclose(R @ R.transpose(1, 2), torch.eye(3).expand(16, 3, 3), atol=1e-5)
        assert torch.allclose(torch.det(R), torch.ones(16), atol=1e-5)
    # a rotation is a fixed point
    R0 = refine.special_procrustes(M)
    assert torch.allclose(refine.special_gramschmidt(R0), R0, atol=1e-5)
    # Gram-Schmidt keeps the direction of the first column
    x = torch.nn.functional.normalize(M[:, :, 0], dim=-1)
    assert torch.allclose(refine.special_gramschmidt(M)[:, :, 0], x, atol=1e-6)


class _DS:
    def __init__(self, n=7):
        g = torch.Generator().manual_seed(1)
        self.poses = []
        for _ in range(n):
            T = torch.eye(4)
            T[:3, :3] = refine.special_procrustes(torch.randn(3, 3, generator=g))
            T[:3, 3] = torch.randn(3, generator=g)
            self.poses.append(T)

    def __len__(self):
        return len(self.poses)

    def get_focal_length(self, i):
        return 525.0


def _opts(mode):
    return types.SimpleNamespace(pose_refinement=mode, pose_refinement_lr=0.001, pose_refinement_weight=0.1,
                                 refinement_ortho="gram-schmidt")


@pytest.mark.parametrize("mode", ["none", "naive", "mlp"])
def test_pose_refiner_against_reference(mode):
    golden = np.load(GOLDEN)
    ds = _DS()
    np.testing.assert_allclose(torch.stack(ds.poses).numpy(), golden["dataset_poses"], atol=1e-6)
    torch.manual_seed(5)
    ours = refine.PoseRefiner(ds, torch.device("cpu"), _opts(mode))
    ours.create_pose_buffer()
    idx = torch.tensor([[3], [0], [6], [3]], dtype=torch.int32)
    orig = torch.stack([ds.poses[i].inverse() for i in idx.view(-1).tolist()])
    a = ours.get_current_poses(orig, idx)
    assert torch.allclose(a, torch.from_numpy(golden[f"pose_{mode}_current"]), atol=1e-6)
    assert torch.allclose(ours.get_all_current_poses(), torch.from_numpy(golden[f"pose_{mode}_all"]), atol=1e-6)
    if mode != "none":
        # one optimisation step on the same objective moves both identically
        ours.zero_grad(set_to_none=True)
        (a[:, :3] * torch.arange(12.).view(1, 3, 4)).sum().backward()
        ours.step()
        assert torch.allclose(ours.get_all_current_poses(), torch.from_numpy(golden[f"pose_{mode}_all_after_step"]),
                              atol=1e-6)


def test_calibration_refiner_against_reference():
    ds = _DS()
    ours = refine.CalibrationRefiner(ds, 0.001, torch.device("cpu"))
    K = torch.eye(3).repeat(5, 1, 1)
    K[:, 0, 0] = K[:, 1, 1] = torch.tensor([525.0, 350.0, 787.5, 525.0, 600.0])
    K[:, 0, 2], K[:, 1, 2] = 320.0, 240.0
    with torch.no_grad():
        ours.global_f += 0.05
    out = ours.get_refined_calibration_matrices(K)
    # refine_calibration.py:40-51 (the reference hard-codes .cuda() there, so it is restated here)
    expect = K.clone()
    expect[:, 0, 0] = expect[:, 1, 1] = 1.05 * 525.0 * (K[:, 0, 0] / 525.0)
    expect[:, 0, 1] = expect[:, 1, 0] = 0
    assert torch.allclose(out, expect, atol=1e-4)
    out.sum().backward()
    assert ours.global_f.grad is not None and float(ours.global_f.grad) > 0
    assert abs(float(ours.get_focal_length()) - 551.25) < 1e-3
