"""GPU parity of the encoder kernels (conv1 direct + tcgen05 implicit-GEMM convolutions) against the CPU oracle in its
autocast-emulating mode (fp16 operands, fp32 accumulation, fp16 activations)."""
import numpy as np
import pytest
import torch

from oracle import ace_ref

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("n,h,w", [(1, 96, 128), (2, 75, 101), (1, 480, 640), (3, 64, 72)])
def test_encoder_matches_oracle(n, h, w):
    from acezero_b200.encoder import EncoderEngine, out_hw
    esd = ace_ref.make_encoder_state(77)
    eng = EncoderEngine(esd, max_n=n, max_h=h, max_w=w)
    img = torch.cat([ace_ref.synth_image(5 + i, h, w) for i in range(n)], 0)
    f = eng.forward_nhwc(img.cuda()).float().cpu()
    h8, w8 = out_hw(h, w)
    assert tuple(f.shape) == (n, h8, w8, 512)
    with torch.no_grad():
        ref = ace_ref.encoder_forward(esd, img, emulate_half=True).permute(0, 2, 3, 1)
    err = (f - ref).abs()
    scale = ref.abs().max()
    # 11 layers of fp16 activations: a handful of 1-ulp flips propagate; 1 % of the activation range at worst
    assert err.max() < 1e-2 * scale, f"max err {err.max():.4f} vs scale {scale:.3f}"
    assert err.mean() < 1e-3 * scale


def test_encoder_fp16_input_and_plan_regrow():
    from acezero_b200.encoder import EncoderEngine
    esd = ace_ref.make_encoder_state(78)
    eng = EncoderEngine(esd, max_n=1, max_h=64, max_w=64)
    img = ace_ref.synth_image(9, 120, 88)
    a = eng.forward_nhwc(img.cuda())                 # grows the plan
    b = eng.forward_nhwc(img.half().cuda())          # conv1 rounds its input to fp16 in both cases
    assert torch.equal(a, b)
    c = eng.forward_nhwc(ace_ref.synth_image(9, 64, 64).cuda())
    assert tuple(c.shape) == (1, 8, 8, 512) and torch.isfinite(c.float()).all()


@pytest.mark.parametrize("h,w", [(96, 128), (120, 168), (480, 640)])
def test_encoder_with_pretrained_weights_matches_oracle(h, w):
    """The same comparison on the weights the reference ships (`ace_encoder_pretrained.pt`, staged by
    `__graft_entry__.build()` into the git-ignored oracle/_ref/): real weight statistics, not random ones. The oracle is
    pinned to the reference's own Encoder on these weights by tests/test_oracle_golden.py."""
    import os
    from acezero_b200.encoder import EncoderEngine, out_hw
    here = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    path = os.path.join(here, "oracle", "_ref", "ace_encoder_pretrained.pt")
    if not os.path.exists(path):
        pytest.skip("ace_encoder_pretrained.pt not staged under oracle/_ref/ (too large for the repository)")
    esd = torch.load(path, map_location="cpu")
    eng = EncoderEngine(esd, max_n=1, max_h=h, max_w=w)
    img = ace_ref.synth_image(11, h, w)
    f = eng.forward_nhwc(img.cuda()).float().cpu()
    assert tuple(f.shape) == (1, *out_hw(h, w), 512)
    with torch.no_grad():
        ref = ace_ref.encoder_forward(esd, img, emulate_half=True).permute(0, 2, 3, 1)
    err = (f - ref).abs()
    scale = ref.abs().max()
    assert err.max() < 1e-2 * scale, f"max err {err.max():.4f} vs scale {scale:.3f}"
    assert err.mean() < 1e-3 * scale
