"""CPU checks of the GPU image path (csrc/imageprep.cu, acezero_b200/imageprep.py): the coefficient tables and the
fixed-point resize against Pillow, L and the jitter against torchvision, the exported per-pixel device functions
(`acez_host_*`) against numpy and the oracle, the draw order of GpuImageDataset against oracle.image_ref, and the
no-device error of the new entries."""
import ctypes as C
import random

import numpy as np
import pytest
import torch
import torchvision.transforms.functional as TF
from PIL import Image

from acezero_b200 import imageprep as IP
from oracle import image_ref


def np_resize(a, h, w):
    """The kernels' resize in numpy: horizontal pass (uint8 intermediate), then vertical; a pass is skipped when that
    dimension is unchanged."""
    x = a.astype(np.int64)

    def one_pass(x, axis, n_out):
        n_in = x.shape[axis]
        if n_in == n_out:
            return x
        t = IP.resize_coeffs(n_in, n_out).astype(np.int64)
        k = t[:, 2:]
        idx = np.minimum(t[:, :1] + np.arange(k.shape[1])[None, :], n_in - 1)
        xs = np.moveaxis(x, axis, 0)[idx]                    # [n_out, taps, ...]
        kk = k.reshape(k.shape + (1,) * (xs.ndim - 2))
        acc = (1 << 21) + (xs * kk).sum(axis=1)
        return np.moveaxis(np.clip(acc >> 22, 0, 255), 0, axis)

    return one_pass(one_pass(x, 1, w), 0, h).astype(np.uint8)


def np_luma(rgb):
    r, g, b = (rgb[..., i].astype(np.int64) for i in range(3))
    return ((19595 * r + 38470 * g + 7471 * b + 0x8000) >> 16).astype(np.uint8)


def np_blend(d, v, f):
    t = np.float32(d) + np.float32(f) * (v.astype(np.int32) - d).astype(np.float32)
    return np.clip(np.where(t <= 0, 0, np.where(t >= 255, 255, t)), 0, 255).astype(np.float32).astype(np.int64)


def np_contrast_mean(v):
    return int(float(v.astype(np.int64).sum()) / v.size + 0.5)


def np_jitter(L, contrast_first, fb, fc):
    if contrast_first:
        return np_blend(0, np_blend(np_contrast_mean(L), L, fc), fb)
    b = np_blend(0, L, fb)
    return np_blend(np_contrast_mean(b), b, fc)


def np_normalize(v):
    return (v.astype(np.float32) / np.float32(255) - np.float32(0.4)) / np.float32(0.25)


@pytest.mark.parametrize("h0,w0,short", [(480, 640, 480), (480, 640, 320), (480, 640, 719), (1080, 1920, 480),
                                         (131, 97, 45), (200, 300, 333)])
def test_resize_matches_pillow(h0, w0, short):
    rs = np.random.RandomState(h0 * 7 + short)
    a = rs.randint(0, 256, (h0, w0, 3), dtype=np.uint8)
    ref = np.asarray(TF.resize(TF.to_pil_image(a), short))
    h, w = IP.resized_size(h0, w0, short)
    assert ref.shape == (h, w, 3)
    assert np.array_equal(np_resize(a, h, w), ref)


def test_luma_and_jitter_match_torchvision():
    rs = np.random.RandomState(3)
    a = rs.randint(0, 256, (61, 83, 3), dtype=np.uint8)
    pil = Image.fromarray(a)
    L = np.asarray(TF.rgb_to_grayscale(pil))
    assert np.array_equal(np_luma(a), L)
    gray = Image.fromarray(L)
    for f in (0.9, 0.93731, 1.0, 1.04127, 1.1, 1.7):
        assert np.array_equal(np_blend(0, L, f), np.asarray(TF.adjust_brightness(gray, f))), f
        assert np.array_equal(np_blend(np_contrast_mean(L), L, f), np.asarray(TF.adjust_contrast(gray, f))), f
    # the whole Grayscale -> ColorJitter -> ToTensor -> Normalize chain, both randperm orders
    for seed in range(6):
        torch.manual_seed(seed)
        order, fb, fc, _, _ = TF_get_params()
        torch.manual_seed(seed)
        from torchvision import transforms
        t = transforms.Compose([transforms.Grayscale(), transforms.ColorJitter(brightness=0.1, contrast=0.1),
                                transforms.ToTensor(), transforms.Normalize(mean=[0.4], std=[0.25])])
        ref = t(pil)[0].numpy()
        cf = int([int(i) for i in order if int(i) in (0, 1)][0] == 1)
        assert np.array_equal(np_normalize(np_jitter(L, cf, fb, fc)), ref)


def TF_get_params():
    from torchvision import transforms
    cj = transforms.ColorJitter(brightness=0.1, contrast=0.1)
    return transforms.ColorJitter.get_params(cj.brightness, cj.contrast, None, None)


def test_host_pixel_functions(lib):
    rs = np.random.RandomState(5)
    # fixed-point resize sample: every output of a downscale and an upscale table
    for n_in, n_out in ((640, 213), (97, 131), (1920, 853)):
        t = IP.resize_coeffs(n_in, n_out)
        row = rs.randint(0, 256, n_in + 8, dtype=np.uint8)
        ref = np_resize(row[None, :n_in, None], 1, n_out)[0, :, 0]
        for o in range(n_out):
            k = np.ascontiguousarray(t[o, 2:])
            p = row[t[o, 0]:].ctypes.data_as(C.c_void_p)
            assert lib.acez_host_resize_sample(p, 1, k.ctypes.data_as(C.c_void_p), int(t[o, 1])) == ref[o]
    # L
    px = rs.randint(0, 256, (500, 3))
    assert [lib.acez_host_luma(*map(int, p)) for p in px] == list(np_luma(px[None].astype(np.uint8))[0])
    # jitter + normalise over every value, both orders, factors below and above 1
    v = np.arange(256)
    for cf in (0, 1):
        for fb, fc in ((0.9, 1.1), (1.07, 0.93), (1.1, 1.1)):
            mean = 117
            ref = np_blend(0, np_blend(mean, v, fc), fb) if cf else np_blend(mean, np_blend(0, v, fb), fc)
            got = [lib.acez_host_jitter(int(x), cf, fb, fc, mean) for x in v]
            assert got == list(ref)
    assert [lib.acez_host_normalize(int(x)) for x in v] == list(np_normalize(v).astype(np.float64))
    # rotation tap (unclipped) against the oracle's warp, reflect mode
    for rows, cols, angle in ((37, 53, 13.7), (48, 31, -14.99), (20, 20, 0.5)):
        img = rs.standard_normal((rows, cols)).astype(np.float32)
        M = image_ref.rotate_matrix(rows, cols, angle)
        ref = image_ref.warp_bilinear(img, M, "reflect")
        m6 = (C.c_double * 6)(*IP.rotation_matrix(rows, cols, angle)[:2].ravel())
        ip = img.ctypes.data_as(C.c_void_p)
        got = np.array([[lib.acez_host_rotate_sample(m6, ip, rows, cols, r, c) for c in range(cols)] for r in range(rows)])
        assert np.array_equal(got, ref)
    # mask cells against the oracle's rotated ones + the trainer's NEAREST resize
    from acezero_b200.encoder import out_hw
    for rows, cols, angle in ((480, 640, 14.3), (320, 427, -15.0), (719, 958, 7.1), (16, 21, 15.0)):
        h8, w8 = out_hw(rows, cols)
        mask = torch.from_numpy(image_ref.rotate(np.ones((rows, cols), np.float32), angle, "constant")).float()[None] > 0
        ref = TF.resize(mask, [h8, w8], interpolation=TF.InterpolationMode.NEAREST).bool()[0].numpy()
        m6 = (C.c_double * 6)(*IP.rotation_matrix(rows, cols, angle)[:2].ravel())
        got = np.array([[lib.acez_host_mask_cell(m6, rows, cols, h8, w8, i, j) for j in range(w8)] for i in range(h8)])
        assert np.array_equal(got.astype(bool), ref)
        assert got.any()


@pytest.fixture(scope="module")
def frames(tmp_path_factory):
    from acezero_b200.synthetic import write_frames
    d = tmp_path_factory.mktemp("frames")
    jpg, poses = write_frames(d / "jpg", 3, H=96, W=128, focal=105.0, ext="jpg")
    png, _ = write_frames(d / "png", 2, H=128, W=96, focal=105.0, ext="png", gray=(1,))
    return jpg + png, poses + poses[:2]


def test_wrapper_draws_and_pixels_match_oracle(frames):
    """Same seeds: GpuImageDataset makes the oracle's draws (generator states agree after every item), its matrices
    equal the oracle's, and its parameters drive a numpy restatement of the kernels to the oracle's image bit for bit."""
    from acezero_b200.synthetic import FrameDataset
    files, poses = frames
    base = FrameDataset(files, poses, focal=105.0, image_short_size=96)
    gpu, ref = IP.GpuImageDataset(base), image_ref.ImageRefDataset(base)
    for i in range(len(files)):
        random.seed(100 + i)
        torch.manual_seed(200 + i)
        item = gpu[[i]]
        st_gpu = (random.getstate(), torch.get_rng_state())
        random.seed(100 + i)
        torch.manual_seed(200 + i)
        image, mask, pose_inv, aug_inv, K, Kinv, _, _, idx = ref[[i]]
        assert random.getstate() == st_gpu[0] and torch.equal(torch.get_rng_state(), st_gpu[1])
        assert int(idx) == item["idx"] == i
        assert tuple(image.shape[2:]) == item["size"]
        mats = np.concatenate([aug_inv.numpy()[0, :3].ravel(), pose_inv.numpy()[0].ravel(), K.numpy()[0].ravel(),
                               Kinv.numpy()[0].ravel()]).astype(np.float32)
        assert np.array_equal(mats, item["mats"])
        # pixels: numpy restatement of the kernels from the wrapper's raw pixels and parameters
        h, w = item["size"]
        a = item["pixels"].numpy()
        r = np_resize(a, h, w)
        L = np_luma(r) if a.shape[2] == 3 else r[..., 0]
        x = np_normalize(np_jitter(L, item["contrast_first"], item["brightness"], item["contrast"]))
        rot = image_ref.rotate(x, item["angle"], "reflect")
        assert np.array_equal(torch.from_numpy(rot).float().half().numpy(), image[0, 0].numpy())


def test_new_entries_fail_without_device(lib):
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from acezero_b200 import _lib
    d = (_lib.ImagePrepDesc * 1)()
    d[0].src, d[0].h_in, d[0].w_in, d[0].channels = 16, 8, 8, 1
    ws = lib.acez_image_prep_workspace_bytes(d, 1, 8, 8)
    assert ws > 0
    assert lib.acez_image_prep(d, 1, 8, 8, C.c_void_p(16), ws, C.c_void_p(16), None) == 4
    m6 = (C.c_double * 6)(1, 0, 0, 0, 1, 0)
    assert lib.acez_image_mask_cells(m6, 16, 16, 2, 2, C.c_void_p(16), None) == 4
    # argument validation still comes first
    assert lib.acez_image_prep(d, 1, 8, 4, C.c_void_p(16), ws, C.c_void_p(16), None) == 1
