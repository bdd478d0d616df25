"""The CPU oracle (oracle/ace_ref.py) against golden vectors produced by the reference's own code
(oracle/make_golden.py ran ace_network.Regressor, ace_trainer.TrainerACE.training_step, ace_loss.ReproLoss)."""
import numpy as np
import pytest
import torch

from oracle import ace_ref


@pytest.mark.parametrize("homog", [True, False])
@pytest.mark.parametrize("nb", [1, 2])
def test_head_forward_matches_reference(golden, homog, nb):
    sd = ace_ref.make_head_state(100 + nb, nb, homog, mean=(0.3, -0.2, 1.5))
    feats = ace_ref.synth_batch(7, 512)["features"].float()
    with torch.no_grad():
        sc = ace_ref.head_forward(sd, feats, nb, homog, emulate_half=False).numpy()
    ref = golden[f"head_sc_h{int(homog)}_b{nb}"]
    assert sc.shape == ref.shape == (512, 3)
    np.testing.assert_allclose(sc, ref, rtol=2e-5, atol=2e-5)


CASES = [("dyntanh", "dyntanh", False, "circle"), ("l1sqrt_depth", "l1+sqrt", True, "constant"),
         ("tanh", "tanh", False, "circle"), ("l1", "l1", False, "circle"), ("l1log", "l1+log", False, "circle")]


@pytest.mark.parametrize("tag,loss_type,use_depth,sched", CASES)
def test_training_step_matches_reference(golden, tag, loss_type, use_depth, sched):
    """4 iterations of the restated training step reproduce the reference's losses, inlier fractions and weights."""
    sd = ace_ref.make_head_state(200, 1, True, mean=(0.0, 0.0, 0.0))
    opts = ace_ref.LossOptions(repro_loss_type=loss_type, use_depth=use_depth, iterations=1000)
    lrs = golden[f"train_{tag}_lr"]
    if sched == "circle":
        fn = ace_ref.one_cycle_lr(0.005, 1000)
        np.testing.assert_allclose([fn(i) for i in range(len(lrs))], lrs, rtol=1e-9)
        lr_fn = lambda it: fn(it - 1)  # the golden run starts at iteration 1 with a fresh scheduler
    else:
        assert np.allclose(lrs, 0.0005)
        lr_fn = lambda it: 0.0005
    tr = ace_ref.TrainerRef(sd, 1, True, opts, lr_fn, emulate_half=False)
    tr.iteration = 1
    losses, inl = [], []
    for it in range(4):
        bt = ace_ref.synth_batch(300 + it, 512, with_depth=use_depth)
        l, i, _, _ = tr.step(bt["features"].float(), bt["target_px"], bt["aug_poses_inv"], bt["poses_inv"],
                             bt["intrinsics"], bt["intrinsics_inv"], bt["target_crds"])
        losses.append(l)
        inl.append(i)
    np.testing.assert_allclose(losses, golden[f"train_{tag}_loss"], rtol=2e-4)
    np.testing.assert_allclose(inl, golden[f"train_{tag}_inliers"], atol=1e-9)
    for k in ("res3_conv1.weight", "0c1.weight", "fc2.bias", "fc3.weight", "fc3.bias"):
        got = tr.sd[k].detach().reshape(-1)[::97].numpy()
        np.testing.assert_allclose(got, golden[f"train_{tag}_{k}"], rtol=1e-3, atol=2e-5, err_msg=k)


@pytest.mark.parametrize("t", ["tanh", "dyntanh", "l1", "l1+sqrt", "l1+log"])
def test_repro_loss_compute(golden, t):
    errs = torch.from_numpy(np.random.RandomState(5).uniform(0, 200, 4096).astype(np.float32))
    o = ace_ref.LossOptions(repro_loss_type=t, iterations=1000)
    got = [float(ace_ref.repro_loss_compute(o, errs, it)) for it in (0, 250, 999)]
    np.testing.assert_allclose(got, golden[f"reproloss_{t}"], rtol=1e-6)


def test_synth_batch_has_valid_and_invalid_rows():
    bt = ace_ref.synth_batch(300, 512)
    sd = ace_ref.make_head_state(200, 1, True)
    with torch.no_grad():
        sc = ace_ref.head_forward(sd, bt["features"].float(), 1, True)
        _, inl, n_valid = ace_ref.training_loss(ace_ref.LossOptions(), sc, bt["target_px"], bt["aug_poses_inv"],
                                                bt["poses_inv"], bt["intrinsics"], bt["intrinsics_inv"],
                                                bt["target_crds"], 10)
    assert 50 < n_valid < 500


@pytest.mark.parametrize("tag,h,w", [("96x128", 96, 128), ("75x101", 75, 101)])
def test_encoder_forward_matches_reference(golden, tag, h, w):
    esd = ace_ref.make_encoder_state(77)
    with torch.no_grad():
        f = ace_ref.encoder_forward(esd, ace_ref.synth_image(5, h, w), emulate_half=False)
    assert list(f.shape) == list(golden[f"encoder_{tag}_shape"])
    ref = golden[f"encoder_{tag}_sample"]
    got = f.reshape(-1)[::53].numpy()
    np.testing.assert_allclose(got, ref, rtol=1e-4, atol=1e-4 * np.abs(ref).max())


def _pretrained_encoder_state():
    """The reference's shipped encoder weights (22 MB, too large for the repository): the git-ignored copy
    `__graft_entry__.build()` stages under oracle/_ref/ when the reference checkout is available to it."""
    import os
    here = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    p = os.path.join(here, "oracle", "_ref", "ace_encoder_pretrained.pt")
    return torch.load(p, map_location="cpu") if os.path.exists(p) else None


@pytest.mark.parametrize("tag,h,w", [("96x128", 96, 128), ("120x168", 120, 168)])
def test_encoder_forward_with_pretrained_weights_matches_reference(tag, h, w):
    """oracle.ace_ref.encoder_forward on the weights the reference ships vs the reference's own Encoder
    (fixture: oracle/make_golden.py::pretrained_encoder_golden)."""
    import os
    esd = _pretrained_encoder_state()
    if esd is None:
        pytest.skip("ace_encoder_pretrained.pt not staged under oracle/_ref/")
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "encoder_pretrained_golden.npz"))
    chk = sum(float(v.double().abs().sum()) for v in esd.values())
    assert abs(chk - float(g["weights_checksum"])) <= 1e-9 * abs(chk), "not the weight file the fixture was made with"
    with torch.no_grad():
        f = ace_ref.encoder_forward(esd, ace_ref.synth_image(11, h, w), emulate_half=False)
    assert list(f.shape) == list(g[f"encoder_{tag}_shape"])
    ref = g[f"encoder_{tag}_sample"]
    np.testing.assert_allclose(f.reshape(-1)[::29].numpy(), ref, rtol=1e-4, atol=1e-4 * np.abs(ref).max())
