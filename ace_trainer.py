"""Drop-in for the reference's `ace_trainer.TrainerACE` (reference ace_trainer.py:45-728) on the sm_100a kernels.

Same options object (train_ace.py flags), same seeds / generators / call order for everything that is part of the
integer contract (image order, patch indices, epoch permutations), same output files (fp16 head state dict, log file,
`poses_<map>_preliminary.txt`). What changes is how the work is executed:

  create_training_buffer : encoder = tcgen05 implicit-GEMM plan, NHWC rows; `torch.multinomial` with the reference's CUDA
                           generator (bit-exact indices); one fused fill kernel per image instead of ~12 small kernels;
                           the mask test runs on the CPU copy of the mask (no GPU sync per image). With G ranks
                           (torchrun, see acezero_b200/launch.py) rank r encodes every G-th image of the reference's loader
                           order, every rank replays the sampling generator for all images (indices stay bit-exact) and
                           the rows are all-gathered into the same replicated buffer a single GPU would build
  run_epoch/training_step: `acezero_b200.trainer.TrainLoop` — one CUDA graph per iteration, no host sync; with
                           `--pose_refinement naive|mlp` / `--refine_calibration` the refiners stay PyTorch-autograd
                           models fed by the kernel's dL/dP, dL/dK (eager launches)
"""
import logging
import os
import random
import time

import numpy as np
import torch
import torchvision.transforms.functional as TF
from torch.utils.data import DataLoader, sampler

from ace_network import Regressor
from acezero_b200 import _lib
from acezero_b200 import posefile
from acezero_b200.encoder import out_hw as encoder_out_hw
from acezero_b200.imageprep import GpuImageDataset, ImagePrep
from acezero_b200.parallel import rows_capacity_per_rank
from acezero_b200.trainer import TrainLoop, BUFFER_KEYS

_logger = logging.getLogger(__name__)


def _permute_rows_gpu(src, index, out):
    """out[i, :] = src[index[i], :] for 2-D byte views on the GPU (one launch of the library's row-gather kernel)."""
    lib = _lib.load()
    rc = lib.acez_gather_rows(_lib.ptr(src), _lib.ptr(index), int(index.numel()), int(src.shape[1]), _lib.ptr(out),
                              _lib.stream_ptr())
    _lib.check(rc, "acez_gather_rows")


def set_seed(seed):
    """reference ace_trainer.py:36-42"""
    torch.manual_seed(seed)
    np.random.seed(seed)
    random.seed(seed)


class TrainerACE:
    def __init__(self, options, dataset=None, rank=0, world_size=1):
        self.log_file = None
        self.options = options
        # one process per GPU: the launcher (acezero_b200.launch.select_device) has selected this rank's device
        self.rank, self.world = int(rank), int(world_size)
        self.device = torch.device('cuda', torch.cuda.current_device())
        if not options.use_half:
            _logger.warning("--use_half False: the sm_100a head computes with fp16 operands / fp32 accumulation in either "
                            "mode; dynamic loss scaling with the overflow check stays on (an unscaled fp16 backward "
                            "underflows and has no skip-on-inf)")
        if getattr(options, "training_buffer_cpu", False):
            _logger.warning("--training_buffer_cpu is ignored: the patch buffer stays in HBM (<= 9.8 GB of 180 GB)")
        if getattr(options, "render_visualization", False):
            raise NotImplementedError("the visualiser is out of scope (SURVEY §2.1 row 13)")

        # Seeds and generators exactly as the reference (ace_trainer.py:61-80).
        self.base_seed = options.base_seed
        set_seed(self.base_seed)
        self.batch_generator = torch.Generator()
        self.batch_generator.manual_seed(self.base_seed + 1023)
        self.loader_generator = torch.Generator()
        self.loader_generator.manual_seed(self.base_seed + 511)
        self.sampling_generator = torch.Generator(device=self.device)
        self.sampling_generator.manual_seed(self.base_seed + 4095)

        self.iteration = 0
        self.epoch = 0
        self.training_start = None
        self.num_data_loader_workers = options.num_data_workers
        self.use_depth = (options.use_pose_seed >= 0) or (options.depth_files is not None)
        if self.use_depth and options.depth_files is None:
            self.num_data_loader_workers = 0

        if dataset is None:
            # the reference's CamLocDataset (dataset.py) when this runs inside an ACE0 checkout
            try:
                from dataset import CamLocDataset
            except ImportError as e:
                raise RuntimeError("no dataset object was passed and the reference's dataset.CamLocDataset cannot be "
                                   f"imported ({e}); dataset I/O is outside the hot path (SURVEY §2.1 row 9)") from e
            dataset = CamLocDataset(
                rgb_files=options.rgb_files, pose_files=options.pose_files, ace_pose_file=options.use_ace_pose_file,
                ace_pose_file_conf_threshold=options.ace_pose_file_conf_threshold, pose_seed=options.use_pose_seed,
                depth_files=options.depth_files, use_depth=self.use_depth, augment=options.use_aug,
                aug_rotation=options.aug_rotation, aug_scale_max=options.aug_scale, aug_scale_min=1 / options.aug_scale,
                image_short_size=options.image_resolution, use_half=options.use_half,
                use_heuristic_focal_length=options.use_heuristic_focal_length)
            if os.environ.get("ACEZ_GPU_IMAGES", "0") == "1" and not self.use_depth:
                dataset = GpuImageDataset(dataset)
        self.dataset = dataset
        # decode and random draws on the loader workers, pixel arithmetic in csrc/imageprep.cu (acezero_b200/imageprep.py)
        self.gpu_images = isinstance(dataset, GpuImageDataset)
        if self.gpu_images and (self.use_depth or not options.use_half):
            raise NotImplementedError("the GPU image path prepares fp16 images without depth (use_half, no depth files "
                                      "or pose seed)")
        if options.use_external_focal_length is not None:
            self.dataset.set_external_focal_length(options.use_external_focal_length)
        _logger.info("Loaded training scan from: {} -- {} images, mean: {:.2f} {:.2f} {:.2f}".format(
            options.rgb_files, len(self.dataset), *[float(v) for v in self.dataset.mean_cam_center]))

        # Network (reference :127-148). Head weights are initialised by nn.Conv2d under the global seed, in the
        # reference's construction order.
        encoder_state_dict = options.encoder_state_dict if getattr(options, "encoder_state_dict", None) is not None \
            else torch.load(options.encoder_path, map_location="cpu")
        if options.load_weights is None:
            self.regressor = Regressor.create_from_encoder(encoder_state_dict, mean=self.dataset.mean_cam_center,
                                                           num_head_blocks=options.num_head_blocks,
                                                           use_homogeneous=options.use_homogeneous)
        else:
            head_state_dict = torch.load(options.load_weights, map_location="cpu")
            self.regressor = Regressor.create_from_split_state_dict(encoder_state_dict, head_state_dict)
        self.regressor = self.regressor.to(self.device)
        self.regressor.train()

        # Pose / calibration refinement (reference :173-184): PyTorch-autograd models fed by the kernel's dL/dP, dL/dK.
        from acezero_b200.refine import PoseRefiner, CalibrationRefiner
        self.pose_refiner = PoseRefiner(dataset=self.dataset, device=self.device, options=options)
        self.K_optimizer = CalibrationRefiner(dataset=self.dataset, learning_rate=options.refine_calibration_lr,
                                              device=self.device) if options.refine_calibration else None

        self.iterations_output = options.iterations_output
        self.training_buffer = None
        self.training_buffer_size = options.max_training_buffer_size
        self.loop = None

    # ------------------------------------------------------------------------------------------------------------
    def train(self):
        creating_buffer_time = 0.
        self.training_start = time.time()
        t0 = time.time()
        self.create_training_buffer()
        torch.cuda.synchronize()
        creating_buffer_time += time.time() - t0
        _logger.info(f"Filled training buffer in {creating_buffer_time:.1f}s.")

        base_file_name, _ = os.path.splitext(self.options.output_map_file)
        # rank 0 owns the output files; every rank still reads the statistics (the read is a collective)
        self.log_file = open(base_file_name + '.txt', 'w') if self.rank == 0 else None

        self.pose_refiner.create_pose_buffer()            # reference :231 (after the buffer: same RNG order)
        head = self._training_engine()
        self.loop = TrainLoop(head, self.options, self.training_buffer, use_depth=self.use_depth,
                              pose_refiner=self.pose_refiner, K_optimizer=self.K_optimizer, rank=self.rank,
                              world_size=self.world)
        t0 = time.time()
        while self.loop.run_epoch(on_iteration=self._log_iteration):
            pass
        self.loop.finish()            # device schedule -> host: the final iteration count (cool-down may have shortened it)
        head.gather_params_from_shards()   # peer-memory data parallel: fp32 master weights live on their owner rank
        torch.cuda.synchronize()
        training_time = time.time() - t0
        self.iteration, self.epoch = self.loop.iteration, self.loop.epoch
        self.regressor.heads.export_engine_weights()

        if self.rank == 0:
            self.save_model()
            self.save_poses()
            self.log_file.close()
        self.timing = {"buffer_s": creating_buffer_time, "train_s": training_time, "images_encoded": self.images_encoded,
                       "iterations": self.iteration}
        _logger.info(f'Done without errors. Creating buffer time: {creating_buffer_time:.1f} seconds. '
                     f'Training time: {training_time:.1f} seconds. '
                     f'Total time: {time.time() - self.training_start:.1f} seconds.')

    def _training_engine(self):
        """The head engine of this rank. Data parallel: parameters / gradient / workspace in symmetric memory, so that the
        optimiser step runs over NVLink peer memory (csrc/adamw_dp.cu); ACEZ_DP_PEERS=0 or a failing rendezvous (no peer access
        between the GPUs) selects the NCCL all-reduce path."""
        heads = self.regressor.heads
        refining = self.pose_refiner.active or self.K_optimizer is not None
        if self.world > 1 and not refining and os.environ.get("ACEZ_DP_PEERS", "1") != "0":
            import torch.distributed as dist
            try:
                head = heads.engine(training=True, max_rows=self.options.batch_size, peer_group=dist.group.WORLD)
                head.setup_peers()
                return head
            except Exception as e:  # noqa: BLE001
                _logger.warning(f"peer-memory data parallel unavailable ({type(e).__name__}: {e}); using the NCCL all-reduce path")
                heads._engine = None
        return heads.engine(training=True, max_rows=self.options.batch_size)

    def _log_iteration(self, loop):
        """reference ace_trainer.py:642-673 (pose statistics are zero without pose refinement)."""
        st = loop.last_stats
        loss, inl = float(st[0]), float(st[1]) / loop.b_global
        if float(st[3]) != 0 or not np.isfinite(loss):
            # st[3] is latched on the device: a non-finite loss of ANY iteration since the last read (reference :615-617
            # checks every step; here the check costs no per-step host sync and still cannot miss one)
            _logger.error("Aborting because of NaN loss")
            raise SystemExit(1)
        if self.rank != 0:
            return
        t = time.time() - self.training_start
        it = loop.iteration - 1   # the iteration these statistics belong to (the reference logs before incrementing, :642-651)
        _logger.info(f'Iteration: {it:6d}|{loop.schedule.max_iterations:6d} / Epoch {loop.epoch:03d}, '
                     f'Loss: {loss:.1f}, Batch inliers ({self.options.learning_rate_cooldown_trigger_px_threshold}px): '
                     f'{inl * 100:.1f}%, Time: {t:.0f}s')
        orig, cur = self.pose_refiner.get_all_original_poses(), self.pose_refiner.get_all_current_poses()
        dist = torch.linalg.norm(cur[:, :, 3] - orig[:, :, 3], dim=1)
        _logger.info(f'Poses moved by: Avg={dist.mean() * 100:.1f}cm, Min={dist.min() * 100:.1f}cm, '
                     f'Max={dist.max() * 100:.1f}cm')
        line = f"{it} {t} {loss} {inl} {dist.mean()} {dist.min()} {dist.max()}"
        if self.K_optimizer is not None:
            focal = float(self.K_optimizer.get_focal_length())
            _logger.info(f"Current Focal Length: {focal:.1f}")
            line += f" {focal}"
        self.log_file.write(line + "\n")

    # ------------------------------------------------------------------------------------------------------------
    def create_training_buffer(self):
        """reference ace_trainer.py:293-452.

        Same loader, generators and call order as the reference (=> the same images in the same order and bit-exact patch
        indices); what differs is the execution: consecutive loader items of equal image size share ONE encoder launch
        (the reference encodes at batch 1, :366-367; `ACEZ_FILL_BATCH`, default 8, 1 = per image), images go host->device
        asynchronously from the loader's pinned tensors straight into the batch slot, the per-image matrices of a group
        travel as one pinned row block, an all-true mask costs no resize / copy, and one fused kernel per image scatters
        the sampled rows into all 8 buffer arrays. No host synchronisation per image.

        With a GpuImageDataset the loader items carry raw uint8 pixels and the drawn augmentation parameters: the mask
        cells are computed on the device for every image (every rank), and the owned images of a group are resized,
        jittered, normalised and rotated by the csrc/imageprep.cu kernels straight into the batch slot.
        """
        o = self.options
        max_batch = max(1, int(os.environ.get("ACEZ_FILL_BATCH", "8") or 8))
        batch_sampler = sampler.BatchSampler(sampler.RandomSampler(self.dataset, generator=self.batch_generator),
                                             batch_size=1, drop_last=False)

        def seed_worker(worker_id):
            worker_seed = torch.initial_seed() % 2 ** 32
            np.random.seed(worker_seed)
            random.seed(worker_seed)

        loader = DataLoader(dataset=self.dataset, sampler=batch_sampler, batch_size=None, worker_init_fn=seed_worker,
                            generator=self.loader_generator, pin_memory=True, num_workers=self.num_data_loader_workers,
                            persistent_workers=self.num_data_loader_workers > 0,
                            timeout=60 if self.num_data_loader_workers > 0 else 0)
        _logger.info("Starting creation of the training buffer.")
        size = min(o.max_dataset_passes * len(self.dataset) * o.samples_per_image, o.max_training_buffer_size)
        rank, world = self.rank, self.world
        # data parallel: this rank fills a LOCAL staging buffer with the rows of its own images (every world-th non-empty
        # image of the loader order); single GPU: local == the final buffer
        local_cap = size if world == 1 else rows_capacity_per_rank(size, o.samples_per_image, world)
        d = self.device
        gpu_images = self.gpu_images
        prep = ImagePrep(d) if gpu_images else None
        buf = self._alloc_buffer(local_cap)
        lib = _lib.load()
        enc = self.regressor.encoder
        self.sample_log = []  # (image index, sampled cells) — kept for the bit-exactness tests
        keep_log = bool(getattr(o, "keep_sample_log", False))
        buffer_idx, passes, image_counter = 0, 0, 0
        records = []                 # (owner rank, first global row, rows, first local row) of every image in the buffer
        local_rows = [0] * world
        n_encoded = 0
        ones_cache = {}
        # pinned staging of the per-image matrices (aug_inv 12 | pose_inv 16 | K 9 | Kinv 9), one block per group; a block
        # is reused only after the copy that read it has completed
        n_stage = 4
        mats_host = [torch.zeros((max_batch, 46), dtype=torch.float32).pin_memory() for _ in range(n_stage)]
        mats_np = [m.numpy() for m in mats_host]
        mats_dev = [torch.zeros((max_batch, 46), dtype=torch.float32, device=d) for _ in range(n_stage)]
        stage_events = [None] * n_stage
        stage_next = [0]
        group = []                   # owned loader items waiting for the shared encoder launch

        def flush():
            nonlocal n_encoded
            if not group:
                return
            n = len(group)
            H_img, W_img = group[0]["shape"][2], group[0]["shape"][3]
            images = torch.empty((n, 1, H_img, W_img), dtype=torch.float16 if gpu_images else group[0]["image"].dtype,
                                 device=d)
            sl = stage_next[0]
            stage_next[0] = (sl + 1) % n_stage
            if stage_events[sl] is not None:
                stage_events[sl].synchronize()
            else:
                stage_events[sl] = torch.cuda.Event()
            for k, g in enumerate(group):
                if not gpu_images:
                    images[k].copy_(g["image"][0], non_blocking=True)         # pinned (loader) -> device, asynchronous
                mats_np[sl][k] = g["mats"]
            mats_dev[sl][:n].copy_(mats_host[sl][:n], non_blocking=True)
            stage_events[sl].record()
            if gpu_images:
                prep.prepare([g["item"] for g in group], images)
            feats = enc.forward_nhwc(images)                                  # [n,h,w,512] fp16: ONE launch sequence
            _, H, W, C = feats.shape
            for k, g in enumerate(group):
                assert (H, W) == g["hw"]
                crds_d = g["crds"][0].float().contiguous().to(d, non_blocking=True) if self.use_depth else None
                rc = lib.acez_buffer_fill(_lib.ptr(feats[k]), _lib.ptr(g["sample_idxs"]), g["n_sel"], W, H * W,
                                          Regressor.OUTPUT_SUBSAMPLE, _lib.ptr(mats_dev[sl][k]), _lib.ptr(crds_d), g["idx"],
                                          g["local_row0"], _lib.ptr(buf['features']), _lib.ptr(buf['target_px']),
                                          _lib.ptr(buf['aug_poses_inv']), _lib.ptr(buf['poses_inv']),
                                          _lib.ptr(buf['intrinsics']), _lib.ptr(buf['intrinsics_inv']),
                                          _lib.ptr(buf['target_crds']), _lib.ptr(buf['pose_idx']), _lib.stream_ptr())
                _lib.check(rc, "acez_buffer_fill")
            n_encoded += n
            group.clear()

        with torch.no_grad():
            while buffer_idx < o.max_training_buffer_size and passes < o.max_dataset_passes:
                passes += 1
                for item in loader:
                    if gpu_images:
                        image, crds, idx, B = None, None, item["idx"], 1
                        shape = (1, 1) + tuple(item["size"])
                        H, W = encoder_out_hw(shape[2], shape[3])
                        if item["rotate"] and item["angle"] != 0.0:
                            weights = prep.mask_cells(item, H, W)   # never empty (GpuImageDataset checks the size)
                        else:
                            if (H, W) not in ones_cache:
                                ones_cache[(H, W)] = torch.ones(H * W, dtype=torch.float32, device=d)
                            weights = ones_cache[(H, W)]
                        mats = np.asarray(item["mats"], dtype=np.float32)
                    else:
                        image, mask, pose_inv, aug_pose_inv, K, Kinv, crds, _, idx = item
                        shape = tuple(image.shape)
                        B = image.shape[0]
                        assert B == 1, "the buffer is filled image by image (batch_size=1 sampler, reference :298-300)"
                        H, W = encoder_out_hw(image.shape[2], image.shape[3])
                        # mask at output resolution (reference :373-378), decided on the CPU copy: no GPU sync. An all-true
                        # mask (no rotation augmentation) stays all-true under NEAREST resizing: no resize, no host->device copy
                        if mask.numpy().all():
                            if (H, W) not in ones_cache:
                                ones_cache[(H, W)] = torch.ones(H * W, dtype=torch.float32, device=d)
                            weights = ones_cache[(H, W)]
                        else:
                            m = TF.resize(mask, [H, W], interpolation=TF.InterpolationMode.NEAREST).bool()
                            if m.sum() == 0:
                                continue
                            weights = m.float().view(-1).to(d, non_blocking=True)
                    n_sel = min(o.samples_per_image * B, o.max_training_buffer_size - buffer_idx)
                    # EVERY rank draws the indices of EVERY image: the CUDA generator advances exactly as in a single-GPU run
                    sample_idxs = torch.multinomial(weights, n_sel, replacement=True,
                                                    generator=self.sampling_generator)     # reference :423-426
                    if keep_log:
                        self.sample_log.append((int(idx), sample_idxs.cpu()))
                    owner = image_counter % world
                    image_counter += 1
                    if owner == rank:
                        if group and (group[0]["shape"] != shape or len(group) == max_batch):
                            flush()
                        if not gpu_images:
                            mats = np.concatenate([aug_pose_inv.numpy()[0, :3].ravel(), pose_inv.numpy()[0].ravel(),
                                                   K.numpy()[0].ravel(), Kinv.numpy()[0].ravel()]).astype(np.float32)
                        group.append({"image": image, "item": item if gpu_images else None, "shape": shape, "mats": mats,
                                      "crds": crds, "idx": int(idx), "sample_idxs": sample_idxs, "n_sel": n_sel,
                                      "local_row0": local_rows[rank], "hw": (H, W)})
                    records.append((owner, buffer_idx, n_sel, local_rows[owner]))
                    local_rows[owner] += n_sel
                    buffer_idx += n_sel
                    if buffer_idx >= o.max_training_buffer_size:
                        break
                flush()
        self.training_buffer_size = min(buffer_idx, o.max_training_buffer_size)
        self.images_encoded = n_encoded
        if world == 1:
            self.training_buffer = {k: v[:self.training_buffer_size] for k, v in buf.items()}
        else:
            from acezero_b200.parallel import allgather_buffer_rows
            self.training_buffer = allgather_buffer_rows(buf, records, local_rows, self.training_buffer_size, world,
                                                         permute_rows=_permute_rows_gpu)
        gb = sum(v.element_size() * v.nelement() for v in self.training_buffer.values()) / 1024 ** 3
        _logger.info(f"Created buffer of {gb:.2f}GB with {passes} passes over the training data"
                     + (f" (rank {rank} of {world} encoded {n_encoded} of {image_counter} images)." if world > 1 else "."))

    def _alloc_buffer(self, size):
        """The 8 arrays of the reference's buffer dict (ace_trainer.py:330-340), `size` rows."""
        d = self.device
        return {
            'features': torch.empty((size, self.regressor.feature_dim), dtype=torch.float16, device=d),
            'target_px': torch.empty((size, 2), dtype=torch.float32, device=d),
            'aug_poses_inv': torch.empty((size, 3, 4), dtype=torch.float32, device=d),
            'poses_inv': torch.empty((size, 4, 4), dtype=torch.float32, device=d),
            'intrinsics': torch.empty((size, 3, 3), dtype=torch.float32, device=d),
            'intrinsics_inv': torch.empty((size, 3, 3), dtype=torch.float32, device=d),
            'target_crds': torch.empty((size, 3), dtype=torch.float32, device=d),
            'pose_idx': torch.empty((size, 1), dtype=torch.int16, device=d),
        }

    # ------------------------------------------------------------------------------------------------------------
    def save_model(self):
        """fp16 head state dict, reference ace_trainer.py:681-694."""
        head_state_dict = self.regressor.heads.state_dict()
        for k in head_state_dict:
            head_state_dict[k] = head_state_dict[k].half()
        torch.save(head_state_dict, self.options.output_map_file)
        _logger.info(f"Saved trained head weights to: {self.options.output_map_file}")

    def save_poses(self):
        """reference ace_trainer.py:696-728: world-to-cam lines, confidence inf."""
        pose_file = self.options.output_map_file.parent / f"poses_{self.options.output_map_file.stem}_preliminary.txt"
        with open(pose_file, 'w') as f:
            output_poses = self.pose_refiner.get_all_current_poses()
            for i in range(output_poses.shape[0]):
                focal = float(self.K_optimizer.get_focal_length()) if self.K_optimizer is not None \
                    else self.dataset.get_focal_length(i)
                posefile.write_pose_to_pose_file(f, rgb_file=self.dataset.rgb_files[i],
                                                 pose=output_poses[i].cpu().detach().numpy(), confidence=float('inf'),
                                                 focal_length=focal)
        _logger.info(f"Saved refined poses to: {pose_file}")
