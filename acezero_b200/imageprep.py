"""Augmented training images prepared on the GPU (csrc/imageprep.cu).

The reference's loader (dataset.py `CamLocDataset._get_single_item`) does, per image on the CPU workers: decode, PIL
bilinear resize to a random short side, grayscale, ColorJitter(brightness, contrast), ToTensor + Normalize and a
scikit-image order-1 rotation of the image and of an all-ones mask. `GpuImageDataset` keeps the decode and every random
draw on the workers, in the reference's order and on the reference's generators, and returns the raw uint8 pixels with
the drawn parameters. `ImagePrep` then runs the pixel arithmetic in the sm_100a kernels, bit for bit, straight into the
encoder's batch slot, and evaluates the rotated mask only at the cells the sampler reads.

Draw order per loader item (dataset.py `__getitem__`, then `_get_single_item`):
  1. random.uniform(aug_scale_min, aug_scale_max)                      (python `random`)
  2. ColorJitter.get_params: randperm(4), brightness, contrast          (torch CPU generator)
  3. random.uniform(-aug_rotation, aug_rotation)                        (python `random`)
"""
import ctypes
import math
import random

import numpy as np
import torch
from PIL import Image
from torch.utils.data import Dataset
from torchvision import transforms

from acezero_b200 import _lib

# A rotation about the centre keeps every pixel within min(h, w) / 2 of the centre inside the image; with a short side
# of at least 16 px some cell the NEAREST mask resize picks lies within that distance, so the mask is never empty and
# the reference's empty-mask `continue` cannot happen.
MIN_SHORT_SIDE = 16
_EXIF_ORIENTATION = 0x0112


def decode(path):
    """uint8 [h, w, 1 | 3] as skimage.io.imread (imageio's PIL plugin) returns it, before `color.gray2rgb`.

    JPEG frames are turned upright by their EXIF orientation the way imageio's legacy PIL reader does (`exifrotate`);
    that this matches the imageio version of the reference's environment is not verified."""
    with Image.open(path) as im:
        fmt = im.format
        orientation = im.getexif().get(_EXIF_ORIENTATION) if fmt == "JPEG" else None
        if im.mode == "L":
            a = np.array(im)[:, :, None]
        elif im.mode == "RGB":
            a = np.array(im)
        else:
            raise ValueError(f"{path}: image mode {im.mode} is not supported by the GPU image path (L or RGB)")
    if orientation in (3, 4):
        a = np.rot90(a, 2)
    if orientation in (5, 6):
        a = np.rot90(a, 3)
    if orientation in (7, 8):
        a = np.rot90(a)
    if orientation in (2, 4, 5, 7):
        a = np.fliplr(a)
    return np.ascontiguousarray(a)


def resized_size(h, w, short):
    """torchvision `resize(img, short)`: the short side becomes `short`, the long side int(short * long / short_in)."""
    if w <= h:
        return int(short * h / w), short
    return short, int(short * w / h)


def resize_coeffs(in_size, out_size):
    """PIL's bilinear coefficients (Resample.c precompute_coeffs + normalize_coeffs_8bpc) as int32 [out, 2 + k]:
    first source index, tap count, k weights in Q22. The weights are normalised by their sequentially accumulated sum."""
    scale = in_size / out_size
    fs = max(scale, 1.0)
    support = 1.0 * fs
    ksize = int(math.ceil(support)) * 2 + 1
    xx = np.arange(out_size, dtype=np.float64)
    center = 0.0 + (xx + 0.5) * scale
    ss = 1.0 / fs
    xmin = np.maximum(np.trunc(center - support + 0.5), 0).astype(np.int64)
    xmax = np.minimum(np.trunc(center + support + 0.5), in_size).astype(np.int64) - xmin
    x = np.arange(ksize, dtype=np.int64)[None, :]
    t = np.abs(((x + xmin[:, None]) - center[:, None] + 0.5) * ss)
    w = np.where((x < xmax[:, None]) & (t < 1.0), 1.0 - t, 0.0)
    ww = np.cumsum(w, axis=1)[:, -1:]          # trailing zeros leave the sequential sum unchanged
    k = np.where(ww != 0.0, w / np.where(ww != 0.0, ww, 1.0), w)
    kq = np.where(k < 0, np.trunc(-0.5 + k * (1 << 22)), np.trunc(0.5 + k * (1 << 22))).astype(np.int32)
    return np.ascontiguousarray(np.concatenate([xmin[:, None], xmax[:, None], kq], axis=1).astype(np.int32))


def rotation_matrix(h, w, angle):
    """skimage.transform.rotate's inverse map, composed as skimage does: T(c) @ (R(deg2rad(angle)) @ T(-c)),
    c = (w / 2 - 0.5, h / 2 - 0.5). float64 [3, 3]; (col, row) of the output -> (col, row) of the input."""
    center = np.array((w, h)) / 2. - 0.5
    rot = np.deg2rad(angle)
    t1, t2, t3 = np.eye(3), np.eye(3), np.eye(3)
    t1[0:2, 2] = center
    t2[0:2, 0:2] = [[math.cos(rot), -math.sin(rot)], [math.sin(rot), math.cos(rot)]]
    t3[0:2, 2] = -center
    return t1 @ (t2 @ t3)


class GpuImageDataset(Dataset):
    """Wraps a CamLocDataset-like `base` (without depth): same items, same draws, pixel work left to `ImagePrep`.

    `base` provides rgb_files, valid_file_indices, poses, get_focal_length, augment, aug_rotation, aug_scale_min/max,
    aug_black_white and image_short_size. An item (the loader passes `[i]`) is a dict of the raw uint8 pixels
    [h0, w0, C], the drawn parameters, the 46 matrix floats (aug_pose_inv 3x4 | pose_inv | K | K^-1) and the image index.
    """

    def __init__(self, base):
        self.base = base
        self.augment = bool(base.augment)
        self.jitter = transforms.ColorJitter(brightness=base.aug_black_white, contrast=base.aug_black_white)

    def __len__(self):
        return len(self.base.valid_file_indices)

    def __getattr__(self, name):   # rgb_files, poses, mean_cam_center, get_focal_length, set_external_focal_length ...
        if name == "base":
            raise AttributeError(name)
        return getattr(self.base, name)

    def __getitem__(self, idx):
        b = self.base
        scale = random.uniform(b.aug_scale_min, b.aug_scale_max) if self.augment else 1
        short = int(b.image_short_size * scale)
        if isinstance(idx, list):
            assert len(idx) == 1, "the GPU image path serves one image per loader item"
            idx = idx[0]
        return self._single(int(idx), short)

    def _single(self, idx, short):
        b = self.base
        idx = int(b.valid_file_indices[idx])
        pixels = decode(b.rgb_files[idx])
        h0, w0 = pixels.shape[:2]
        focal = b.get_focal_length(idx) * (short / min(h0, w0))
        h, w = resized_size(h0, w0, short)
        if self.augment:
            order, fb, fc, _, _ = transforms.ColorJitter.get_params(self.jitter.brightness, self.jitter.contrast,
                                                                    None, None)
            contrast_first = int([int(i) for i in order if int(i) in (0, 1)][0] == 1)
            angle = random.uniform(-b.aug_rotation, b.aug_rotation)
        else:
            contrast_first, fb, fc, angle = 0, 1.0, 1.0, 0.0
        if self.augment and min(h, w) < MIN_SHORT_SIDE:
            raise ValueError(f"image {idx}: {h}x{w} after scaling; the GPU image path needs a short side of at least "
                             f"{MIN_SHORT_SIDE} px (the rotated mask is then never empty)")
        pose = b.poses[idx].clone()
        pose_rot = torch.eye(4)
        if self.augment:
            a = angle * math.pi / 180.
            pose_rot[0, 0] = math.cos(a)
            pose_rot[0, 1] = -math.sin(a)
            pose_rot[1, 0] = math.sin(a)
            pose_rot[1, 1] = math.cos(a)
        pose_inv, pose_rot_inv = pose.inverse(), pose_rot.inverse()
        if not (torch.isfinite(pose_inv).all() and torch.isfinite(pose_rot_inv).all()):
            raise ValueError(f"Pose at index {idx} is invalid.")
        K = torch.eye(3)
        K[0, 0] = focal
        K[1, 1] = focal
        K[0, 2] = w / 2
        K[1, 2] = h / 2
        Kinv = K.inverse()
        mats = np.concatenate([pose_rot_inv.numpy()[:3].ravel(), pose_inv.numpy().ravel(), K.numpy().ravel(),
                               Kinv.numpy().ravel()]).astype(np.float32)
        affine = rotation_matrix(h, w, angle)[:2].ravel() if self.augment else np.zeros(6)
        return {"pixels": torch.from_numpy(pixels), "size": (h, w), "contrast_first": contrast_first,
                "brightness": float(fb), "contrast": float(fc), "angle": float(angle), "rotate": int(self.augment),
                "affine": affine, "mats": mats, "idx": idx}


class ImagePrep:
    """Device side: coefficient tables cached per (in, out) pair, the mask cells of one image, the prepared images of
    one group. Everything is enqueued on the current stream; nothing synchronises the host."""

    def __init__(self, device):
        self.lib = _lib.load()
        self.device = device
        self.tables = {}

    def table(self, n_in, n_out):
        if n_in == n_out:
            return None, 0
        t = self.tables.get((n_in, n_out))
        if t is None:
            t = self.tables[(n_in, n_out)] = torch.from_numpy(resize_coeffs(n_in, n_out)).to(self.device)
        return t, t.shape[1] - 2

    def mask_cells(self, item, h8, w8):
        """float32 [h8 * w8] on the device: the reference's rotated mask after TF.resize(NEAREST) to (h8, w8)."""
        h, w = item["size"]
        cells = torch.empty(h8 * w8, dtype=torch.float32, device=self.device)
        aff = (ctypes.c_double * 6)(*[float(v) for v in np.asarray(item["affine"]).ravel()])
        _lib.check(self.lib.acez_image_mask_cells(aff, h, w, h8, w8, _lib.ptr(cells), _lib.stream_ptr()),
                   "acez_image_mask_cells")
        return cells

    def prepare(self, items, out):
        """Prepare the images of `items` (one output size) into fp16 `out` [n, 1, h, w]. The pinned pixel tensors go
        to the device asynchronously. The uploads are held until the kernels are enqueued: released earlier, the caching
        allocator would hand an upload's block to the next image's copy, which runs before the kernels read it."""
        n = len(items)
        h, w = items[0]["size"]
        descs = (_lib.ImagePrepDesc * n)()
        srcs = []
        for k, it in enumerate(items):
            assert tuple(it["size"]) == (h, w)
            src = it["pixels"].to(self.device, non_blocking=True)
            srcs.append(src)
            d = descs[k]
            d.src = src.data_ptr()
            d.h_in, d.w_in, d.channels = src.shape
            tx, d.kx = self.table(d.w_in, w)
            ty, d.ky = self.table(d.h_in, h)
            d.coef_x = tx.data_ptr() if tx is not None else None
            d.coef_y = ty.data_ptr() if ty is not None else None
            d.contrast_first, d.brightness, d.contrast = int(it["contrast_first"]), it["brightness"], it["contrast"]
            d.rotate = int(it["rotate"])
            d.affine[:] = [float(v) for v in np.asarray(it["affine"]).ravel()]
        nbytes = self.lib.acez_image_prep_workspace_bytes(descs, n, h, w)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        _lib.check(self.lib.acez_image_prep(descs, n, h, w, _lib.ptr(ws), nbytes, _lib.ptr(out), _lib.stream_ptr()),
                   "acez_image_prep")
