"""CPU oracle of the reference's augmented loader item (dataset.py `CamLocDataset._get_single_item`, no depth).

PIL decode; torchvision's own `TF.resize`, `Grayscale`, `ColorJitter`, `ToTensor` and `Normalize`; a numpy restatement
of scikit-image 0.19's `transform.rotate(img, angle, order=1, mode=..., clip=True)` for the image ('reflect') and the
all-ones mask ('constant', cval 0). `ImageRefDataset(base)` yields the reference's 9-tuple, so it drives the trainer's
CPU-mask path exactly as the reference's dataset would.

The rotation evaluates coordinates, taps and weights in float64. Whether scikit-image's `_warp_fast` keeps float32
intermediates for float32 input is not verified (scikit-image is not a dependency); a difference would show as rare
1-ulp fp16 differences of the image and, at worst, a mask pixel within float32 rounding of the border.
"""
import math
import random

import numpy as np
import torch
import torchvision.transforms.functional as TF
from PIL import Image
from torch.utils.data import Dataset
from torch.utils.data.dataloader import default_collate
from torchvision import transforms


def imread(path):
    """skimage.io.imread through imageio's PIL plugin, JPEG EXIF orientation applied as imageio's `exifrotate`."""
    with Image.open(path) as im:
        orientation = im.getexif().get(0x0112) if im.format == "JPEG" else None
        image = np.array(im)
    if orientation in (3, 4):
        image = np.rot90(image, 2)
    if orientation in (5, 6):
        image = np.rot90(image, 3)
    if orientation in (7, 8):
        image = np.rot90(image)
    if orientation in (2, 4, 5, 7):
        image = np.fliplr(image)
    return np.ascontiguousarray(image)


def rotate_matrix(rows, cols, angle):
    """skimage.transform.rotate: tform3 + tform2 + tform1 (translate by -centre, rotate, translate back)."""
    center = np.array((cols, rows)) / 2. - 0.5
    tform1, tform2, tform3 = np.eye(3), np.eye(3), np.eye(3)
    tform1[0:2, 2] = center
    rotation = np.deg2rad(angle)
    tform2[0:2, 0:2] = [[math.cos(rotation), -math.sin(rotation)], [math.sin(rotation), math.cos(rotation)]]
    tform3[0:2, 2] = -center
    return tform1 @ (tform2 @ tform3)


def _reflect(dim, coord):
    """skimage coord_map, mode 'R' (mirror, edge pixel not repeated)."""
    cmax = dim - 1
    if cmax == 0:
        return np.zeros_like(coord)
    out = coord.copy()
    neg, pos = coord < 0, coord > cmax
    a = -coord[neg]
    out[neg] = np.where((a // cmax) % 2 != 0, cmax - a % cmax, a % cmax)
    b = coord[pos]
    out[pos] = np.where((b // cmax) % 2 != 0, cmax - b % cmax, b % cmax)
    return out


def warp_bilinear(image, M, mode, cval=0.0):
    """Unclipped order-1 samples of a 2-D image at every output pixel under the inverse map M (float64)."""
    rows, cols = image.shape
    img = image.astype(np.float64)
    yy, xx = np.mgrid[0:rows, 0:cols].astype(np.float64)
    c = M[0, 0] * xx + M[0, 1] * yy + M[0, 2]
    r = M[1, 0] * xx + M[1, 1] * yy + M[1, 2]
    minr, minc = np.floor(r).astype(np.int64), np.floor(c).astype(np.int64)
    maxr, maxc = np.ceil(r).astype(np.int64), np.ceil(c).astype(np.int64)
    dr, dc = r - minr, c - minc

    def get(rr, cc):
        if mode == "reflect":
            return img[_reflect(rows, rr), _reflect(cols, cc)]
        inside = (rr >= 0) & (rr < rows) & (cc >= 0) & (cc < cols)
        return np.where(inside, img[np.clip(rr, 0, rows - 1), np.clip(cc, 0, cols - 1)], cval)

    top = (1 - dc) * get(minr, minc) + dc * get(minr, maxc)
    bottom = (1 - dc) * get(maxr, minc) + dc * get(maxr, maxc)
    return (1 - dr) * top + dr * bottom


def rotate(image, angle, mode):
    """skimage.transform.rotate(image, angle, order=1, mode=mode, cval=0, clip=True) of a 2-D float32 image."""
    rows, cols = image.shape
    out = warp_bilinear(image, rotate_matrix(rows, cols, angle), mode)
    lo, hi = image.min(), image.max()
    preserve_cval = mode == "constant" and not lo <= 0.0 <= hi
    cval_mask = out == 0.0 if preserve_cval else None
    np.clip(out, lo, hi, out=out)
    if preserve_cval:
        out[cval_mask] = 0.0
    return out


class ImageRefDataset(Dataset):
    """The reference's item for a CamLocDataset-like `base` (same accessors as acezero_b200.imageprep.GpuImageDataset)."""

    def __init__(self, base, use_half=True):
        self.base = base
        self.use_half = use_half
        if base.augment:
            self.image_transform = transforms.Compose([
                transforms.Grayscale(),
                transforms.ColorJitter(brightness=base.aug_black_white, contrast=base.aug_black_white),
                transforms.ToTensor(),
                transforms.Normalize(mean=[0.4], std=[0.25]),
            ])
        else:
            self.image_transform = transforms.Compose([
                transforms.Grayscale(), transforms.ToTensor(), transforms.Normalize(mean=[0.4], std=[0.25])])

    def __len__(self):
        return len(self.base.valid_file_indices)

    def __getattr__(self, name):
        if name == "base":
            raise AttributeError(name)
        return getattr(self.base, name)

    def _single(self, idx, image_short_size):
        b = self.base
        idx = b.valid_file_indices[idx]
        image = imread(b.rgb_files[idx])
        if image.ndim < 3:
            image = np.stack([image] * 3, axis=-1)            # skimage.color.gray2rgb
        focal_length = b.get_focal_length(idx)
        focal_length *= image_short_size / min(image.shape[0], image.shape[1])
        image = TF.resize(TF.to_pil_image(image), image_short_size)
        image_mask = torch.ones((1, image.size[1], image.size[0]))
        coords = torch.zeros((3, math.ceil(image.size[0] / 8), math.ceil(image.size[1] / 8)))
        image = self.image_transform(image)
        pose = b.poses[idx].clone()
        if b.augment:
            angle = random.uniform(-b.aug_rotation, b.aug_rotation)
            image = torch.from_numpy(rotate(image[0].numpy(), angle, "reflect")).float()[None]
            image_mask = torch.from_numpy(rotate(image_mask[0].numpy(), angle, "constant")).float()[None]
            angle = angle * math.pi / 180.
            pose_rot = torch.eye(4)
            pose_rot[0, 0] = math.cos(angle)
            pose_rot[0, 1] = -math.sin(angle)
            pose_rot[1, 0] = math.sin(angle)
            pose_rot[1, 1] = math.cos(angle)
        else:
            pose_rot = torch.eye(4)
        if self.use_half:
            image = image.half()
        image_mask = image_mask > 0
        pose_inv = pose.inverse()
        pose_rot_inv = pose_rot.inverse()
        intrinsics = torch.eye(3)
        intrinsics[0, 0] = focal_length
        intrinsics[1, 1] = focal_length
        intrinsics[0, 2] = image.shape[2] / 2
        intrinsics[1, 2] = image.shape[1] / 2
        intrinsics_inv = intrinsics.inverse()
        return image, image_mask, pose_inv, pose_rot_inv, intrinsics, intrinsics_inv, coords, str(b.rgb_files[idx]), idx

    def __getitem__(self, idx):
        scale_factor = random.uniform(self.base.aug_scale_min, self.base.aug_scale_max) if self.base.augment else 1
        image_short_size = int(self.base.image_short_size * scale_factor)
        if isinstance(idx, list):
            return default_collate([self._single(i, image_short_size) for i in idx])
        return self._single(idx, image_short_size)
