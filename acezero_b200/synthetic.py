"""Procedural scenes for the benchmark configs and end-to-end tests (SURVEY.md §8d): a textured box room rendered by
ray–plane intersection, with ground-truth camera poses on a smooth trajectory. Yields the 9-tuple the reference's
`CamLocDataset.__getitem__` returns (reference dataset.py:278-417) so that the trainer / registration code paths are the
same as with real data. (The reference's dataset.py needs skimage and real image files; it is out of scope, SURVEY §2.)
"""
import math

import numpy as np
import torch
from torch.utils.data import Dataset
from torch.utils.data.dataloader import default_collate


class BoxRoom:
    """Axis-aligned room [-hx,hx] x [-hy,hy] x [-hz,hz] with a smooth multi-scale texture f(x,y,z) in [0,1]."""

    def __init__(self, seed=2089, half=(3.0, 2.0, 2.5), n_waves=48, octave_shift=0.0):
        rs = np.random.RandomState(seed)
        self.half = torch.tensor(half, dtype=torch.float32)
        # random plane waves over several octaves; view-consistent, high-entropy. `octave_shift` moves the band with the image
        # resolution (one octave per doubling of the focal length) so that the 81-pixel receptive field of the encoder sees the
        # same amount of texture at 480x640 / f = 525 as at 240x320 / f = 262.5
        freq = rs.standard_normal((n_waves, 3)).astype(np.float32)
        freq /= np.linalg.norm(freq, axis=1, keepdims=True)
        octave = (2.0 ** (rs.uniform(0.5, 4.5, n_waves) + octave_shift)).astype(np.float32)
        self.freq = torch.from_numpy(freq * octave[:, None])
        self.phase = torch.from_numpy(rs.uniform(0, 2 * math.pi, n_waves).astype(np.float32))
        self.amp = torch.from_numpy((1.0 / np.sqrt(octave)).astype(np.float32))

    def to(self, device):
        for k in ("half", "freq", "phase", "amp"):
            setattr(self, k, getattr(self, k).to(device))
        return self

    def texture(self, p):
        v = torch.sin(p @ self.freq.t() + self.phase) * self.amp
        v = v.sum(-1) / self.amp.sum() * 2.5
        return (0.5 + 0.5 * torch.tanh(v)).clamp(0, 1)

    def render(self, c2w, f, H, W, cx=None, cy=None, subsample=1, offset=0.5):
        """Grayscale image [H/sub, W/sub] and hit points [.., 3] for camera-to-world pose c2w (4x4)."""
        dev = self.half.device
        cx = W / 2 if cx is None else cx
        cy = H / 2 if cy is None else cy
        ys = (torch.arange(0, H // subsample, device=dev, dtype=torch.float32) + offset) * subsample
        xs = (torch.arange(0, W // subsample, device=dev, dtype=torch.float32) + offset) * subsample
        if subsample == 1:
            ys, xs = ys, xs
        yy, xx = torch.meshgrid(ys, xs, indexing="ij")
        d = torch.stack([(xx - cx) / f, (yy - cy) / f, torch.ones_like(xx)], -1)
        R, t = c2w[:3, :3].to(dev), c2w[:3, 3].to(dev)
        dw = d @ R.t()
        tt = (torch.sign(dw) * self.half - t) / torch.where(dw.abs() < 1e-9, torch.full_like(dw, 1e-9), dw)
        tt = torch.where(tt > 0, tt, torch.full_like(tt, 1e9))
        thit = tt.min(-1).values
        p = t + dw * thit.unsqueeze(-1)
        return self.texture(p), p


def trajectory(n, seed=2089, half=(3.0, 2.0, 2.5), s_offset=0.0):
    """n camera-to-world poses on a smooth closed path inside the room, looking around; `s_offset` (in frames) shifts
    the sampling along the path (held-out views between the training frames)."""
    rs = np.random.RandomState(seed + 17)
    ph = rs.uniform(0, 2 * math.pi, 6)
    poses = []
    for i in range(n):
        s = 2 * math.pi * (i + s_offset) / max(n, 1)
        c = np.array([0.45 * half[0] * math.sin(s + ph[0]), 0.35 * half[1] * math.sin(2 * s + ph[1]),
                      0.45 * half[2] * math.cos(s + ph[2])])
        yaw = s * 1.0 + 0.6 * math.sin(3 * s + ph[3])
        pitch = 0.3 * math.sin(2 * s + ph[4])
        roll = 0.1 * math.sin(5 * s + ph[5])
        Ry = np.array([[math.cos(yaw), 0, math.sin(yaw)], [0, 1, 0], [-math.sin(yaw), 0, math.cos(yaw)]])
        Rx = np.array([[1, 0, 0], [0, math.cos(pitch), -math.sin(pitch)], [0, math.sin(pitch), math.cos(pitch)]])
        Rz = np.array([[math.cos(roll), -math.sin(roll), 0], [math.sin(roll), math.cos(roll), 0], [0, 0, 1]])
        T = np.eye(4)
        T[:3, :3] = Ry @ Rx @ Rz
        T[:3, 3] = c
        poses.append(torch.from_numpy(T).float())
    return poses


class SyntheticDataset(Dataset):
    """CamLocDataset look-alike over a BoxRoom (no augmentation): items are
    (image 1xHxW normalised, mask 1xHxW bool, pose_inv 4x4, aug_pose_inv 4x4 = I, K 3x3, K^-1, gt coords 3xhxw, name, idx)."""

    def __init__(self, n_images=64, H=480, W=640, focal=525.0, seed=2089, with_coords=False, device="cpu",
                 pose_noise=0.0, indices=None, s_offset=0.0):
        self.room = BoxRoom(seed, octave_shift=math.log2(max(float(focal), 1.0) / 262.5)).to(device)
        self.device = device
        self.H, self.W, self.focal = H, W, float(focal)
        all_poses = trajectory(n_images if indices is None else max(indices) + 1, seed, s_offset=s_offset)
        self.indices = list(range(n_images)) if indices is None else list(indices)
        self.gt_poses = [all_poses[i] for i in self.indices]
        self.poses = [p.clone() for p in self.gt_poses]            # camera-to-world, like CamLocDataset.poses
        if pose_noise > 0:
            rs = np.random.RandomState(seed + 5)
            for p in self.poses:
                p[:3, 3] += torch.from_numpy(rs.normal(scale=pose_noise, size=3)).float()
        self.rgb_files = [f"synthetic/frame-{i:06d}.color.png" for i in self.indices]
        self.with_coords = with_coords
        self.external_focal = None
        self.mean_cam_center = torch.stack([p[:3, 3] for p in self.poses]).mean(0)

    def __len__(self):
        return len(self.poses)

    def set_external_focal_length(self, f):
        self.external_focal = float(f)

    def get_focal_length(self, idx):
        return self.external_focal if self.external_focal is not None else self.focal

    def _single(self, idx):
        img, _ = self.room.render(self.gt_poses[idx], self.focal, self.H, self.W)
        image = ((img - 0.4) / 0.25).unsqueeze(0).cpu()                     # dataset.py:150-153 normalisation
        mask = torch.ones((1, self.H, self.W), dtype=torch.bool)
        pose_inv = self.poses[idx].inverse()
        f = self.get_focal_length(idx)
        K = torch.eye(3)
        K[0, 0] = K[1, 1] = f
        K[0, 2], K[1, 2] = self.W / 2, self.H / 2
        h8, w8 = math.ceil(self.H / 8), math.ceil(self.W / 8)
        if self.with_coords:
            _, p = self.room.render(self.gt_poses[idx], self.focal, self.H, self.W, subsample=8)
            coords = p.permute(2, 0, 1).cpu().contiguous()
        else:
            coords = torch.zeros((3, h8, w8))
        return image, mask, pose_inv, torch.eye(4), K, K.inverse(), coords, self.rgb_files[idx], idx

    def __getitem__(self, idx):
        if isinstance(idx, list):
            return default_collate([self._single(i) for i in idx])
        return self._single(idx)


class CachedDataset(Dataset):
    """The items of another dataset rendered ONCE and served from host memory (benchmarks: the procedural renderer of
    SyntheticDataset costs more than the encoder; real datasets decode on DataLoader workers). Same 9-tuples, same
    accessor surface as CamLocDataset / SyntheticDataset. keep_base=False drops the reference to the source dataset (and
    with it any CUDA state), so that the object can be handed to forked DataLoader workers."""

    def __init__(self, base, keep_base=True):
        self.items = [base[i] for i in range(len(base))]
        self.rgb_files = base.rgb_files
        self.poses = base.poses
        self.gt_poses = getattr(base, "gt_poses", base.poses)
        self.mean_cam_center = base.mean_cam_center
        self._focals = [base.get_focal_length(i) for i in range(len(base))]
        self.base = base if keep_base else None

    def __len__(self):
        return len(self.items)

    def set_external_focal_length(self, f):
        if self.base is None:
            raise RuntimeError("CachedDataset(keep_base=False) cannot re-render for another focal length")
        self.base.set_external_focal_length(f)
        self.items = [self.base[i] for i in range(len(self.base))]
        self._focals = [self.base.get_focal_length(i) for i in range(len(self.base))]

    def get_focal_length(self, idx):
        return self._focals[idx]

    def __getitem__(self, idx):
        if isinstance(idx, list):
            return default_collate([self.items[i] for i in idx])
        return self.items[idx]


def write_frames(out_dir, n_images, H=480, W=640, focal=525.0, seed=2089, ext="jpg", gray=(), device="cpu"):
    """Render n BoxRoom frames to image files (`ext` "jpg" or "png"), tinted to RGB so that the three channels differ;
    the frames whose index is in `gray` are written as single-channel PNGs. Returns (paths, camera-to-world poses)."""
    from pathlib import Path
    from PIL import Image
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    room = BoxRoom(seed, octave_shift=math.log2(max(float(focal), 1.0) / 262.5)).to(device)
    poses = trajectory(n_images, seed)
    tint = torch.tensor([1.0, 0.85, 0.6], device=device)
    paths = []
    for i, c2w in enumerate(poses):
        img, _ = room.render(c2w, focal, H, W)
        if i in gray:
            path = out_dir / f"frame-{i:06d}.gray.png"
            Image.fromarray((img * 255).round().byte().cpu().numpy(), mode="L").save(path)
        else:
            x = torch.stack([img * tint[0], img * tint[1] + 0.1 * (1 - img), img * tint[2] + 0.3 * img * img], -1)
            path = out_dir / f"frame-{i:06d}.color.{ext}"
            a = (x.clamp(0, 1) * 255).round().byte().cpu().numpy()
            Image.fromarray(a, mode="RGB").save(path, **({"quality": 90} if ext == "jpg" else {}))
        paths.append(str(path))
    return paths, poses


class FrameDataset(Dataset):
    """A minimal file-backed CamLocDataset look-alike: the attributes the reference's `_get_single_item` reads
    (augmentation settings, image files, poses, focal length). Items come from a wrapper (acezero_b200.imageprep
    .GpuImageDataset or oracle.image_ref.ImageRefDataset), not from this class."""

    def __init__(self, rgb_files, poses, focal=525.0, augment=True, aug_rotation=15, aug_scale_min=2 / 3,
                 aug_scale_max=3 / 2, aug_black_white=0.1, image_short_size=480):
        self.rgb_files = list(rgb_files)
        self.poses = [p.clone() for p in poses]
        self.focal = float(focal)
        self.external_focal = None
        self.augment, self.aug_rotation = augment, aug_rotation
        self.aug_scale_min, self.aug_scale_max = aug_scale_min, aug_scale_max
        self.aug_black_white, self.image_short_size = aug_black_white, image_short_size
        self.valid_file_indices = np.arange(len(self.rgb_files))
        self.mean_cam_center = torch.stack([p[:3, 3] for p in self.poses]).mean(0)

    def __len__(self):
        return len(self.rgb_files)

    def set_external_focal_length(self, f):
        self.external_focal = float(f)

    def get_focal_length(self, idx):
        return self.external_focal if self.external_focal is not None else self.focal
