"""GPU checks of the augmented-image kernels (csrc/imageprep.cu): prepared fp16 images and mask cells equal the CPU
oracle (oracle/image_ref.py) bit for bit on written JPEG / PNG frames, and buffer creation through GpuImageDataset
builds the same buffer as through the oracle's dataset on the trainer's CPU-mask path."""
import random

import numpy as np
import pytest
import torch
import torchvision.transforms.functional as TF

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def frames(tmp_path_factory):
    """BoxRoom renders tinted to RGB: 480x640 JPEG and PNG (one of them gray) and 1920x1080 JPEG."""
    from acezero_b200.synthetic import write_frames
    d = tmp_path_factory.mktemp("frames")
    a, pa = write_frames(d / "a", 4, H=480, W=640, focal=525.0, ext="jpg", device="cuda")
    b, pb = write_frames(d / "b", 2, H=480, W=640, focal=525.0, ext="png", gray=(1,), device="cuda")
    c, pc = write_frames(d / "c", 2, H=1080, W=1920, focal=1400.0, ext="jpg", device="cuda")
    return a + b + c, pa + pb + pc


def _base(frames, **kw):
    from acezero_b200.synthetic import FrameDataset
    files, poses = frames
    return FrameDataset(files, poses, focal=525.0, **kw)


def _items(ds_gpu, ds_ref, seed):
    """(wrapper item, oracle tuple) per image under the same python / torch seeds."""
    out = []
    for i in range(len(ds_gpu)):
        random.seed(seed + i)
        torch.manual_seed(seed + i)
        g = ds_gpu[[i]]
        random.seed(seed + i)
        torch.manual_seed(seed + i)
        out.append((g, ds_ref[[i]]))
    return out


def _check_mask(prep, g, ref_mask):
    from acezero_b200.encoder import out_hw
    h8, w8 = out_hw(*g["size"])
    cells = prep.mask_cells(g, h8, w8).view(h8, w8).cpu()
    expect = TF.resize(ref_mask[0], [h8, w8], interpolation=TF.InterpolationMode.NEAREST).bool()[0].float()
    assert torch.equal(cells, expect)


def test_prepared_images_and_mask_cells_equal_oracle(frames):
    from acezero_b200.imageprep import GpuImageDataset, ImagePrep
    from oracle.image_ref import ImageRefDataset
    prep = ImagePrep(torch.device("cuda"))
    # random scale: every image its own size (1 image per call), 1920x1080 sources included
    base = _base(frames)
    n_checked = 0
    for seed in (11, 907):
        for g, ref in _items(GpuImageDataset(base), ImageRefDataset(base), seed):
            h, w = g["size"]
            out = torch.empty((1, 1, h, w), dtype=torch.float16, device="cuda")
            prep.prepare([g], out)
            got, expect = out.cpu(), ref[0]
            diff = (got.view(torch.int16) != expect.view(torch.int16)).sum().item()
            assert diff == 0, f"{g['idx']}: {diff} of {h * w} fp16 values differ"
            _check_mask(prep, g, ref[1])
            n_checked += 1
    assert n_checked == 16
    # fixed scale: the 480x640 frames (JPEG, RGB PNG, gray PNG) share the output size -> one batched call
    base = _base((frames[0][:6], frames[1][:6]), aug_scale_min=1.0, aug_scale_max=1.0)
    pairs = _items(GpuImageDataset(base), ImageRefDataset(base), 31)
    out = torch.empty((6, 1, 480, 640), dtype=torch.float16, device="cuda")
    prep.prepare([g for g, _ in pairs], out)
    expect = torch.cat([ref[0] for _, ref in pairs])
    assert torch.equal(out.cpu().view(torch.int16), expect.view(torch.int16))


def _options(tmp_path, **kw):
    import train_ace
    o = train_ace.build_parser().parse_args(["synthetic", str(tmp_path / "map.pt")])
    o.encoder_state_dict = None
    for k, v in kw.items():
        setattr(o, k, v)
    return o


@pytest.mark.parametrize("workers", [0, 2])
def test_training_buffer_gpu_images_equals_oracle_path(frames, tmp_path, workers):
    """use_aug=True: same sample_log and bit-identical buffer arrays through GpuImageDataset (device masks, prep
    kernels) and through the oracle dataset (CPU masks, the trainer's existing path)."""
    from ace_trainer import TrainerACE
    from acezero_b200.imageprep import GpuImageDataset
    from acezero_b200.weights import random_encoder_state
    from oracle.image_ref import ImageRefDataset
    base = _base(frames)
    bufs, logs = [], []
    for ds in (ImageRefDataset(base), GpuImageDataset(base)):
        o = _options(tmp_path, samples_per_image=256, max_dataset_passes=2, keep_sample_log=True, batch_size=512,
                     num_data_workers=workers, use_aug=True)
        o.encoder_state_dict = random_encoder_state(77)
        tr = TrainerACE(o, dataset=ds)
        assert tr.gpu_images == isinstance(ds, GpuImageDataset)
        tr.create_training_buffer()
        torch.cuda.synchronize()
        bufs.append({k: v.clone() for k, v in tr.training_buffer.items()})
        logs.append(tr.sample_log)
        del tr
    assert len(logs[0]) == 2 * len(frames[0])
    assert [i for i, _ in logs[0]] == [i for i, _ in logs[1]]
    assert all(torch.equal(a, b) for (_, a), (_, b) in zip(logs[0], logs[1]))
    for k in bufs[0]:
        assert torch.equal(bufs[0][k], bufs[1][k]), k


def test_oracle_rotation_matches_scikit_image():
    """The oracle's numpy restatement against scikit-image itself, where it is installed."""
    skimage_transform = pytest.importorskip("skimage.transform")
    from oracle import image_ref
    rs = np.random.RandomState(0)
    for rows, cols, angle in ((480, 640, 13.37), (333, 591, -14.2), (64, 48, 7.0)):
        img = rs.standard_normal((rows, cols, 1)).astype(np.float32)
        ref = skimage_transform.rotate(img, angle, order=1, mode="reflect")
        got = image_ref.rotate(img[..., 0], angle, "reflect")
        assert np.array_equal(torch.from_numpy(ref[..., 0]).float().half(), torch.from_numpy(got).float().half())
        ones = np.ones((rows, cols, 1), np.float32)
        ref_m = skimage_transform.rotate(ones, angle, order=1, mode="constant")[..., 0] > 0
        assert np.array_equal(ref_m, image_ref.rotate(ones[..., 0], angle, "constant") > 0)
