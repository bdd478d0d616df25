"""Training loop core of ACE mapping on the sm_100a kernels: the part of the reference's `TrainerACE` that runs per
iteration (ace_trainer.py:454-640) — epoch permutation, batch gather, head forward/backward with the fused
reprojection loss, GradScaler + AdamW — with the patch buffer resident in HBM, one CUDA graph per iteration and no
host synchronisation (the reference syncs >= 3 times per iteration, ace_trainer.py:578,586,615).

Data parallel (world_size > 1): every rank holds the same buffer and draws the same permutation
(`training_generator`, ace_trainer.py:79-80,466); rank r processes rows [r*b/G, (r+1)*b/G) of each batch; the loss
divisor stays the global batch size (ace_trainer.py:613); head gradients are summed with one NCCL all-reduce and the
GradScaler inf flag / loss statistics with a second, tiny one.
"""
import ctypes as C
import math

import numpy as np
import torch

from . import _lib
from .head import HeadEngine

BUFFER_KEYS = ("features", "target_px", "aug_poses_inv", "poses_inv", "intrinsics", "intrinsics_inv", "target_crds",
               "pose_idx")
IDX_RING = 16
ROW_BYTES = {"features": 1024, "target_px": 8, "aug_poses_inv": 48, "poses_inv": 64, "intrinsics": 36,
             "intrinsics_inv": 36, "target_crds": 12, "pose_idx": 2}  # 1230 B / row (ace_trainer.py:330-340)


# ----------------------------------------------------------------------------------------------------------------
# learning-rate / loss schedules as functions of the iteration (ace_schedule.py:22-69, ace_loss.py:53-69)
# ----------------------------------------------------------------------------------------------------------------
def one_cycle_lr(max_lr, total_steps, pct_start=0.3, div_factor=25.0, final_div_factor=1e4):
    """torch.optim.lr_scheduler.OneCycleLR(max_lr, total_steps, cycle_momentum=False) with torch defaults
    (ace_schedule.py:62-69): the lr used by the optimiser step of iteration i."""
    initial, minimum = max_lr / div_factor, max_lr / div_factor / final_div_factor
    up_end = float(pct_start * total_steps) - 1
    down_end = total_steps - 1

    def cos(a, b, pct):
        return b + (a - b) / 2.0 * (math.cos(math.pi * pct) + 1)

    def fn(i):
        i = min(i, total_steps - 1)
        if i <= up_end:
            return cos(initial, max_lr, i / up_end)
        return cos(max_lr, minimum, (i - up_end) / (down_end - up_end))
    return fn


class Schedule:
    """ScheduleACE semantics (ace_schedule.py:8-126) without torch's scheduler objects: lr(i), cooldown trigger and
    the mutable max_iterations."""

    def __init__(self, o):
        self.schedule = o.learning_rate_schedule
        if self.schedule not in ("circle", "constant", "1cyclepoly"):
            raise ValueError(f"Unknown learning rate schedule: {self.schedule}")
        self.max_iterations = o.iterations
        self.lr_min, self.lr_max = o.learning_rate_min, o.learning_rate_max
        self.in_cooldown_phase = False
        self.cooldown_start = None
        self.buffer = []
        if self.schedule == "circle":
            self._fn = one_cycle_lr(self.lr_max, self.max_iterations)
        elif self.schedule == "1cyclepoly":
            self.warmup_iterations = o.learning_rate_warmup_iterations
            self.warmup_lr = o.learning_rate_warmup_learning_rate
            self.cooldown_iterations = o.learning_rate_cooldown_iterations
            self.trigger = o.learning_rate_cooldown_trigger_percent_threshold
        self.steps = 0  # scheduler.step() calls so far

    @property
    def needs_inliers(self):
        """Only 1cyclepoly consumes the per-iteration inlier fraction (cooldown trigger, ace_schedule.py:91-101)."""
        return self.schedule == "1cyclepoly" and not self.in_cooldown_phase

    def lr(self):
        s = self.steps
        if self.schedule == "constant":
            return self.lr_min
        if self.schedule == "circle":
            return self._fn(s)
        if not self.in_cooldown_phase:  # LinearLR warm-up (start_factor = warmup_lr / lr_max, end_factor 1)
            f0 = self.warmup_lr / self.lr_max
            f = f0 + (1.0 - f0) * min(s, self.warmup_iterations) / self.warmup_iterations
            return self.lr_max * f
        # LinearLR cool-down (1 -> lr_min / lr_max over cooldown_iterations). torch's LinearLR is applied
        # multiplicatively to the lr it finds, and warm-up has finished before a cool-down can start (:81), so the
        # base is lr_max. The cool-down scheduler object was created at t=0 and its own counter starts at 0.
        k = min(self.steps - self.cooldown_start, self.cooldown_iterations)
        f1 = self.lr_min / self.lr_max
        return self.lr_max * (1.0 + (f1 - 1.0) * k / self.cooldown_iterations)

    def check_and_set_cooldown(self, iteration):
        """ace_schedule.py:72-101."""
        if self.schedule != "1cyclepoly" or self.in_cooldown_phase or iteration < self.warmup_iterations:
            return
        by_duration = iteration >= (self.max_iterations - self.cooldown_iterations)
        dynamic = min(self.buffer) > self.trigger
        if by_duration or dynamic:
            self.max_iterations = iteration + self.cooldown_iterations
            self.in_cooldown_phase = True
            self.cooldown_start = self.steps

    def step(self, batch_inliers):
        """ace_schedule.py:115-126 (the optimiser part runs on the device)."""
        if self.schedule == "constant":
            return
        self.steps += 1
        if self.schedule == "1cyclepoly":
            self.buffer.append(batch_inliers)
            if len(self.buffer) > 100:
                self.buffer = self.buffer[1:]


def loss_weight(o, iteration):
    """ace_loss.py:53-69 (tanh weight of iteration); soft_clamp for the l1 family."""
    if o.repro_loss_type == "dyntanh":
        w = iteration / o.iterations
        if o.repro_loss_schedule == "circle":
            w = 1 - np.sqrt(1 - w ** 2)
        return float((1 - w) * o.repro_loss_soft_clamp + o.repro_loss_soft_clamp_min)
    return float(o.repro_loss_soft_clamp)


# ----------------------------------------------------------------------------------------------------------------
class TrainLoop:
    def __init__(self, head: HeadEngine, options, buffer, use_depth=False, rank=0, world_size=1, use_graph=True,
                 device=None, pose_refiner=None, K_optimizer=None):
        self.o = options
        self.head = head
        self.lib = head.lib
        self.device = head.device if device is None else torch.device(device)
        self.use_depth = use_depth
        self.rank, self.world = rank, world_size
        self.b_global = options.batch_size
        if self.b_global % world_size != 0:
            raise ValueError("batch_size must be divisible by the number of ranks")
        self.b = self.b_global // world_size
        # The head kernels compute with fp16 operands in either mode, so dynamic loss scaling + the skip-on-overflow check stay
        # on for `--use_half False` too (the reference trains in fp32 there, ace_trainer.py:517, ace_schedule.py:70; an
        # unscaled fp16 backward underflows, and without the check one overflow would write NaN into the weights)
        self.use_scaler = True
        self.schedule = Schedule(options)
        self.iteration = 0
        self.epoch = 0
        self.training_generator = torch.Generator()
        self.training_generator.manual_seed(options.base_seed + 8191)  # ace_trainer.py:79-80
        self.pose_refiner = pose_refiner if (pose_refiner is not None and pose_refiner.active) else None
        self.K_optimizer = K_optimizer
        self.refining = self.pose_refiner is not None or self.K_optimizer is not None
        # pose / calibration refinement runs PyTorch autograd + torch optimisers (capturable) between the kernels: on one GPU
        # the whole iteration, refiners included, is still ONE captured CUDA graph (two variants: with / without the pose
        # optimiser step, ace_trainer.py:634-636); under data parallelism it stays eager (NCCL calls between the pieces)
        self.use_graph = use_graph and not (self.refining and world_size > 1)
        self._graph = None
        self._warm = 0
        self._refine_graphs = {}
        self._refine_warm = {}
        # peer-memory optimiser (csrc/adamw_dp.cu) when the head was created over symmetric memory (HeadEngine(peer_group=...))
        self._dp_peers = world_size > 1 and getattr(head, "_symm", None) is not None and not self.refining
        if self._dp_peers and head.peer is None:
            head.setup_peers()
        self._graph_host = None
        self._warm_host = 0
        self.set_buffer(buffer)
        if head.max_rows < self.b or not head.training:
            raise ValueError("head engine must be created with training=True and max_rows >= per-rank batch")
        # static per-iteration tensors (graph-stable addresses)
        d = self.device
        self.idx_dev = torch.zeros(self.b, dtype=torch.int64, device=d)
        # ring of pinned index rows: queued H2D copies read the pinned row when the DMA executes, possibly many host
        # iterations later, so a row is reused only after the copy that read it has completed
        self.idx_host = torch.zeros((IDX_RING, self.b), dtype=torch.int64).pin_memory()
        self._idx_events = [None] * IDX_RING
        self._idx_slot = 0
        # one packed allocation; the per-key tensors are typed views (so a host batch can arrive as ONE copy)
        self._aux_off, off = {}, 0
        for k in BUFFER_KEYS[1:]:
            self._aux_off[k] = off
            off += (ROW_BYTES[k] * self.b + 255) // 256 * 256
        self._aux_bytes = off
        self._aux = torch.zeros(off, dtype=torch.uint8, device=d)
        self.batch = self._aux_views(self._aux)
        if self.refining:
            self.d_P = torch.zeros((self.b, 3, 4), device=d)
            self.d_Kdiag = torch.zeros((self.b, 2), device=d)
        self.loss_w_host = None
        # ---- the schedule lives on the device (csrc/schedule.cu): lr, loss weight, cool-down trigger, max_iterations ----
        o = options
        sp = _lib.ScheduleParams()
        sp.kind = _lib.SCHED_KINDS[o.learning_rate_schedule]
        sp.iterations = int(o.iterations)
        sp.lr_min, sp.lr_max = float(o.learning_rate_min), float(o.learning_rate_max)
        sp.warmup_iterations = int(getattr(o, "learning_rate_warmup_iterations", 1) or 1)
        sp.warmup_lr = float(getattr(o, "learning_rate_warmup_learning_rate", o.learning_rate_min))
        sp.cooldown_iterations = int(getattr(o, "learning_rate_cooldown_iterations", 1) or 1)
        sp.cooldown_trigger = float(getattr(o, "learning_rate_cooldown_trigger_percent_threshold", 2.0))
        sp.batch_global = int(self.b_global)
        sp.loss_dyntanh = int(o.repro_loss_type == "dyntanh")
        sp.loss_schedule_circle = int(getattr(o, "repro_loss_schedule", "circle") == "circle")
        sp.soft_clamp, sp.soft_clamp_min = float(o.repro_loss_soft_clamp), float(o.repro_loss_soft_clamp_min)
        self._sp = sp
        self.sched_state = torch.zeros(_lib.SCHED_STATE_FLOATS, dtype=torch.float32, device=d)
        _lib.check(self.lib.acez_schedule_init(C.byref(sp), _lib.ptr(self.sched_state), _lib.stream_ptr()), "acez_schedule_init")
        # the host mirrors max_iterations / the cool-down flag from snapshots read back with a bounded lag (never a sync)
        self._poll_every = max(1, min(64, sp.cooldown_iterations // 4)) if sp.kind == 2 else 0
        self._poll_ring = [torch.zeros(16, dtype=torch.float32).pin_memory() for _ in range(4)]
        self._poll_events = [None] * 4
        self._poll_pending = []   # slots in flight, oldest first
        self._poll_slot = 0
        self.stats_host = torch.zeros(4, dtype=torch.float32).pin_memory()
        self._last_lw = None
        self.last_stats = None

    _AUX_SHAPES = {"target_px": ((2,), torch.float32), "aug_poses_inv": ((3, 4), torch.float32),
                   "poses_inv": ((4, 4), torch.float32), "intrinsics": ((3, 3), torch.float32),
                   "intrinsics_inv": ((3, 3), torch.float32), "target_crds": ((3,), torch.float32),
                   "pose_idx": ((1,), torch.int16)}

    def _aux_views(self, packed_u8):
        out = {}
        for k in BUFFER_KEYS[1:]:
            shape, dt = self._AUX_SHAPES[k]
            o = self._aux_off[k]
            out[k] = packed_u8[o:o + ROW_BYTES[k] * self.b].view(dt).view((self.b,) + shape)
        return out

    def new_host_batch(self):
        """A pinned host batch laid out like the device staging area: dict of typed views (fill them in place) over ONE
        pinned allocation, so that `prefetch_host_batch` moves it with a single host->device copy."""
        nf = self.b * ROW_BYTES["features"]
        packed = torch.zeros(nf + self._aux_bytes, dtype=torch.uint8).pin_memory()
        hb = {"features": packed[:nf].view(torch.float16).view(self.b, 512)}
        hb.update(self._aux_views(packed[nf:]))
        hb["_packed"] = packed
        return hb

    # ------------------------------------------------------------------ buffer
    def set_buffer(self, buffer):
        """buffer: dict with the reference's keys/shapes/dtypes (ace_trainer.py:330-340), CUDA-resident."""
        for k in BUFFER_KEYS:
            t = buffer[k]
            if not t.is_cuda:
                raise ValueError(f"training buffer '{k}' must live on the GPU (180 GB of HBM hold the 9.8 GB maximum)")
            if t.element_size() * t[0].numel() != ROW_BYTES[k]:
                raise ValueError(f"training buffer '{k}' has {t.element_size() * t[0].numel()} B rows, expected {ROW_BYTES[k]}")
        self.buffer = {k: buffer[k].contiguous() for k in BUFFER_KEYS}
        self.buffer_size = self.buffer["features"].shape[0]

    def _gather(self, stream=None, with_schedule=False):
        """Batch rows of all 8 buffer arrays in one launch; with_schedule: the device-side schedule step rides in its first
        block (then the iteration needs no separate schedule kernel)."""
        keys = list(BUFFER_KEYS)
        n = len(keys)
        srcs = (C.c_void_p * n)(*[self.buffer[k].data_ptr() for k in keys])
        dsts = (C.c_void_p * n)(*([self.head.input_buffer(self.b).data_ptr()] + [self.batch[k].data_ptr() for k in keys[1:]]))
        rbs = (C.c_int * n)(*[ROW_BYTES[k] for k in keys])
        if with_schedule:
            h = self.head
            src = h.stats.data_ptr() + 4 if self.world == 1 else h.grads_full.data_ptr() + 4 * (h.n_params + 2)
            rc = self.lib.acez_gather_rows_multi_sched(srcs, dsts, rbs, n, _lib.ptr(self.idx_dev), self.b, C.byref(self._sp),
                                                       _lib.ptr(self.sched_state), C.c_void_p(src), _lib.ptr(h.hyper),
                                                       _lib.stream_ptr(stream))
            _lib.check(rc, "acez_gather_rows_multi_sched")
            return
        rc = self.lib.acez_gather_rows_multi(srcs, dsts, rbs, n, _lib.ptr(self.idx_dev), self.b, _lib.stream_ptr(stream))
        _lib.check(rc, "acez_gather_rows_multi")

    # ------------------------------------------------------------------ one iteration
    def _enqueue_compute(self, P=None, d_P=None, d_Kdiag=None, gather=True, part="all"):
        """gather + forward + loss + backward (+ all-reduce) + GradScaler/AdamW on the current stream."""
        o, h = self.o, self.head
        lp = h.loss_params(o.repro_loss_type, 0.0, self.b_global, self.use_depth, o.depth_min, o.depth_max,
                           float(o.repro_loss_hard_clamp), float(o.learning_rate_cooldown_trigger_px_threshold),
                           o.depth_target, 1.0)
        if part in ("all", "fwd_bwd"):
            if gather:
                self._gather(with_schedule=True)
            else:
                self._enqueue_schedule()
        bt = self.batch
        # data parallel: the fp16-overflow check must see the SUMMED gradient (a per-rank partial can pass while the sum
        # overflows), so the optimiser runs its own check pass, which also reads the flag slot behind the gradient (the ranks'
        # local flags); single GPU: the backward kernels' folded check is complete
        flag_complete = self.world == 1
        if part == "optimizer":
            h.adamw_step(use_scaler=self.use_scaler, flag_complete=flag_complete, check_flag_slot=self.world > 1)
            return
        h.train_fwd_bwd(self.b, lp, bt["target_px"], bt["intrinsics"], bt["intrinsics_inv"],
                        aug_inv=bt["aug_poses_inv"], pose_inv=bt["poses_inv"], P=P,
                        target_crds=bt["target_crds"] if self.use_depth else None, features=None, d_P=d_P,
                        d_Kdiag=d_Kdiag, use_device_scale=True, use_device_loss_weight=True)
        if self.world > 1 and not self._dp_peers:
            self._dp_pack_flag()   # (the peer-memory optimiser packs the spare slots itself)
        if part == "fwd_bwd":
            return
        if self._dp_peers:
            h.adamw_step_peers()   # reduce-scatter + AdamW + weight all-gather over NVLink peer memory (csrc/adamw_dp.cu)
            return
        if self.world > 1:
            self._dp_allreduce()
        h.adamw_step(use_scaler=self.use_scaler, flag_complete=flag_complete, check_flag_slot=self.world > 1)

    def _enqueue_schedule(self):
        """First kernel of the iteration: device-side lr / loss weight / cool-down trigger (csrc/schedule.cu). It books the
        PREVIOUS iteration's inlier count, which under data parallelism is the all-reduced one riding behind the gradient."""
        h = self.head
        src = h.stats.data_ptr() + 4 if self.world == 1 else h.grads_full.data_ptr() + 4 * (h.n_params + 2)
        rc = self.lib.acez_schedule_step(C.byref(self._sp), _lib.ptr(self.sched_state), C.c_void_p(src), _lib.ptr(h.hyper),
                                         _lib.stream_ptr())
        _lib.check(rc, "acez_schedule_step")

    def _poll_schedule(self, force=False):
        """Host mirror of the device schedule: enqueue a 64-byte snapshot every `_poll_every` iterations and consume the
        snapshots whose copies have completed (event query, no wait). `force`: synchronous read (end of training / logging)."""
        sch = self.schedule
        if force:
            st = self.sched_state[:16].cpu()
            self._apply_snapshot(st)
            return
        if self._poll_every and self.iteration % self._poll_every == 0 and len(self._poll_pending) < len(self._poll_ring):
            k = self._poll_slot
            self._poll_slot = (k + 1) % len(self._poll_ring)
            if k not in self._poll_pending:
                self._poll_ring[k].copy_(self.sched_state[:16], non_blocking=True)
                if self._poll_events[k] is None:
                    self._poll_events[k] = torch.cuda.Event()
                self._poll_events[k].record()
                self._poll_pending.append(k)
        while self._poll_pending and self._poll_events[self._poll_pending[0]].query():
            self._apply_snapshot(self._poll_ring[self._poll_pending.pop(0)])

    def _apply_snapshot(self, st):
        sch = self.schedule
        if int(st[2]) and not sch.in_cooldown_phase:
            sch.in_cooldown_phase = True
            sch.cooldown_start = int(st[3])
        sch.max_iterations = min(sch.max_iterations, int(st[4]))

    def finish(self):
        """End of training: wait for the device, take over its final schedule state (iterations the host enqueued beyond the
        device's max_iterations ran with lr = 0 and changed nothing)."""
        torch.cuda.current_stream().synchronize()
        self._poll_schedule(force=True)
        self.iteration = min(self.iteration, int(self.sched_state[0].item()))
        return self.iteration

    def _run_refined_graphed(self, step_poses):
        """Refinement iteration as one CUDA graph per variant (captured after two eager runs of THAT variant, so that the torch
        optimisers' lazily created state exists and every kernel attribute is set)."""
        g = self._refine_graphs.get(step_poses)
        if g is None:
            if self._refine_warm.get(step_poses, 0) < 2:
                self._refine_warm[step_poses] = self._refine_warm.get(step_poses, 0) + 1
                self._enqueue_refined(step_poses)
                return
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._enqueue_refined(step_poses)
            self._refine_graphs[step_poses] = g
        g.replay()

    def _enqueue_refined(self, step_poses=True):
        """Iteration with pose and / or calibration refinement (reference ace_trainer.py:527-540, 620-640): the refined
        per-image poses and the refined intrinsics are PyTorch-autograd values; the fused kernel consumes the composed
        P = A * T and K' and returns dL/dP, dL/dK00, dL/dK11, which are pushed back through autograd."""
        o, h, bt = self.o, self.head, self.batch
        self._gather(with_schedule=True)
        lp = h.loss_params(o.repro_loss_type, 0.0, self.b_global, self.use_depth, o.depth_min, o.depth_max,
                           float(o.repro_loss_hard_clamp), float(o.learning_rate_cooldown_trigger_px_threshold),
                           o.depth_target, 1.0)
        with torch.enable_grad():
            if self.pose_refiner is not None:
                cur_b34 = self.pose_refiner.current_poses_n34()[bt["pose_idx"].view(-1).long()]
                poses_b44 = torch.cat([cur_b34, bt["poses_inv"][:, 3:4, :]], dim=1)        # refined [R|t], row (0,0,0,1)
            else:
                poses_b44 = bt["poses_inv"]
            P = torch.bmm(bt["aug_poses_inv"], poses_b44)                                   # :530
            K = self.K_optimizer.get_refined_calibration_matrices(bt["intrinsics"]) if self.K_optimizer is not None \
                else bt["intrinsics"]                                                        # :536-540
        h.train_fwd_bwd(self.b, lp, bt["target_px"], K.detach().contiguous(), bt["intrinsics_inv"],
                        P=P.detach().contiguous(), target_crds=bt["target_crds"] if self.use_depth else None,
                        features=None, d_P=self.d_P, d_Kdiag=self.d_Kdiag, use_device_scale=True,
                        use_device_loss_weight=True)
        if self.pose_refiner is not None:
            self.pose_refiner.zero_grad(set_to_none=True)                                   # :621
        if self.K_optimizer is not None:
            self.K_optimizer.zero_grad()                                                    # :623-624
        outs, grads = [], []
        if P.requires_grad:
            outs.append(P); grads.append(self.d_P)
        if K.requires_grad:
            gK = torch.zeros_like(K)
            gK[:, 0, 0] = self.d_Kdiag[:, 0]
            gK[:, 1, 1] = self.d_Kdiag[:, 1]
            outs.append(K); grads.append(gK)
        if outs:
            torch.autograd.backward(outs, grads)
        if self.world > 1:
            import torch.distributed as dist
            from .parallel import allreduce_training_state
            allreduce_training_state(h.grads, h.stats, h.found_inf)
            h.grads_full[h.n_params + 1:h.n_params + 4].copy_(h.stats[:3])   # the device schedule books the global inlier count
            extra = []
            if self.pose_refiner is not None and self.pose_refiner.pose_optimizer is not None:
                extra += [p for g in self.pose_refiner.pose_optimizer.param_groups for p in g["params"]]
            if self.K_optimizer is not None:
                extra.append(self.K_optimizer.global_f)
            for p in extra:
                if p.grad is not None:
                    dist.all_reduce(p.grad)
        h.adamw_step(use_scaler=self.use_scaler, flag_complete=self.world == 1)             # :632
        if self.pose_refiner is not None and step_poses:                                   # :634-636
            self.pose_refiner.step()
        if self.K_optimizer is not None:                                                    # :638-640
            self.K_optimizer.step()

    # ---- data parallel: ONE all-reduce per iteration. The local GradScaler flag rides in a spare slot behind the
    # gradient (+inf when set: any rank's inf makes the sum non-finite); statistics are reduced only when someone reads them
    def _dp_pack_flag(self):
        h = self.head
        if not hasattr(self, "_inf_c"):
            self._inf_c = torch.tensor([float("inf")], device=self.device)
            self._zero_c = torch.zeros(1, device=self.device)
        torch.where(h.found_inf > 0, self._inf_c, self._zero_c, out=h.grads_full[h.n_params:h.n_params + 1])
        # loss sum / inlier count / valid count ride along: the device schedule books the GLOBAL inlier count
        h.grads_full[h.n_params + 1:h.n_params + 4].copy_(h.stats[:3])

    def _dp_allreduce(self):
        import torch.distributed as dist
        dist.all_reduce(self.head.grads_full)

    def _dp_reduce_stats(self):
        """Global [loss sum, inlier count, valid count, non-finite flag]: the three sums travelled behind the gradient through
        the iteration's all-reduce (no extra collective); a non-finite loss on any rank makes the summed loss non-finite."""
        h = self.head
        st = torch.empty(4, device=self.device, dtype=torch.float32)
        st[:3] = h.grads_full[h.n_params + 1:h.n_params + 4]
        st[3] = (~torch.isfinite(st[0])).float()
        return st

    def train_iteration(self, indices, want_stats=False):
        """indices: int64 CPU tensor of the GLOBAL batch (b_global entries of the epoch permutation). Learning rate, loss
        weight and the cool-down trigger are evaluated on the device (first kernel of the iteration); the host only mirrors
        max_iterations from snapshots read back with a bounded lag."""
        sch = self.schedule
        self._poll_schedule()
        if self.iteration >= sch.max_iterations:                      # ace_trainer.py:509
            return False
        from .parallel import shard_bounds
        lo, hi = shard_bounds(self.rank, self.world, self.b_global)
        slot = self._idx_slot
        self._idx_slot = (slot + 1) % IDX_RING
        if self._idx_events[slot] is None:
            self._idx_events[slot] = torch.cuda.Event()
        else:
            self._idx_events[slot].synchronize()
        self.idx_host[slot].copy_(indices[lo:hi])
        self.idx_dev.copy_(self.idx_host[slot], non_blocking=True)
        self._idx_events[slot].record()
        if self.refining:
            step_poses = self.pose_refiner is not None and self.iteration > self.o.pose_refinement_wait   # :634-636
            if self.use_graph:
                self._run_refined_graphed(step_poses)
            else:
                self._enqueue_refined(step_poses)
        elif self.use_graph:
            self._run_graphed()
        else:
            self._enqueue_compute()
        if want_stats:
            src = self._dp_reduce_stats() if self.world > 1 else self.head.stats
            self.stats_host.copy_(src, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            self.last_stats = self.stats_host.clone()
            self._poll_schedule(force=True)
        self.iteration += 1
        return True

    def train_step_from_host(self, host_batch, read_loss=True):
        """End-to-end step with HOST inputs (the reference's `--training_buffer_cpu` path, ace_trainer.py:485-494):
        the batch rows arrive in pinned host memory, are copied to the device, trained on, and the loss statistics
        are read back. Returns (loss, inlier fraction)."""
        self.head.input_buffer(self.b).copy_(host_batch["features"], non_blocking=True)
        for k in BUFFER_KEYS[1:]:
            self.batch[k].copy_(host_batch[k], non_blocking=True)
        return self._step_on_static_batch(read_loss)

    def _step_on_static_batch(self, read_loss):
        """One iteration on whatever the static batch tensors hold (no gather); reads the loss statistics back."""
        # (NCCL all-reduces are not captured: that data-parallel path runs eagerly; the peer-memory optimiser is plain kernels
        # on this stream and is captured like the single-GPU iteration)
        if self.use_graph and (self.world == 1 or self._dp_peers):
            if self._graph_host is None:
                if self._warm_host < 2:
                    self._warm_host += 1
                    self._enqueue_compute(gather=False)
                else:
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g):
                        self._enqueue_compute(gather=False)
                    self._graph_host = g
                    g.replay()
            else:
                self._graph_host.replay()
        else:
            self._enqueue_compute(gather=False)
        out = None
        if read_loss:
            self.stats_host.copy_(self._dp_reduce_stats() if self.world > 1 else self.head.stats, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            out = (float(self.stats_host[0]), float(self.stats_host[1]) / self.b_global)
        self.iteration += 1
        return out

    # ---- pipelined host-batch path: the H2D copy of step i+1 runs on a copy stream while step i computes
    def prefetch_host_batch(self, host_batch):
        """Start the (asynchronous) host->device copy of a batch into the free staging slot. Call it for batch i+1 before
        `train_step_prefetched()` of batch i so that the copy overlaps the compute. Batches made by `new_host_batch()`
        travel as one copy; plain dicts of pinned tensors key by key."""
        nf = self.b * ROW_BYTES["features"]
        if not hasattr(self, "_stage"):
            self._copy_stream = torch.cuda.Stream(device=self.device)
            self._stage = [torch.empty(nf + self._aux_bytes, dtype=torch.uint8, device=self.device) for _ in range(2)]
            self._stage_views = []
            for st in self._stage:
                v = {"features": st[:nf].view(torch.float16).view(self.b, 512)}
                v.update(self._aux_views(st[nf:]))
                self._stage_views.append(v)
            self._stage_ev = [torch.cuda.Event(), torch.cuda.Event()]
            self._stage_free = [torch.cuda.Event(), torch.cuda.Event()]
            self._stage_w = 0   # next slot to fill
            self._stage_r = 0   # next slot to consume
            self._stage_used = [False, False]
        slot = self._stage_w
        with torch.cuda.stream(self._copy_stream):
            if self._stage_used[slot]:
                self._copy_stream.wait_event(self._stage_free[slot])   # the step that read this slot has consumed it
            if "_packed" in host_batch:
                self._stage[slot].copy_(host_batch["_packed"], non_blocking=True)
            else:
                for k in BUFFER_KEYS:
                    self._stage_views[slot][k].copy_(host_batch[k], non_blocking=True)
            self._stage_ev[slot].record(self._copy_stream)
        self._stage_used[slot] = True
        self._stage_w ^= 1

    def train_step_prefetched(self, read_loss=True, lag=0):
        """Train on the oldest prefetched batch (two device->device moves, 6.3 MB, into the graph's static tensors, then
        the captured iteration) and read the loss statistics back: returns (loss, inlier fraction).

        lag=0: the result of THIS step (host waits for the step). lag=1: this step is enqueued, then the result of the
        PREVIOUS step is returned (None on the first call; `drain_prefetched()` returns the last one), so the host
        never leaves the device idle. Every step's statistics are read in either mode. The 1cyclepoly schedule needs
        the inlier fraction of step i before the learning rate of step i+1 (ace_schedule.py:91-101) and forces lag=0."""
        slot = self._stage_r
        nf = self.b * ROW_BYTES["features"]
        cur = torch.cuda.current_stream()
        cur.wait_event(self._stage_ev[slot])
        st = self._stage[slot]
        self.head.input_buffer(self.b).view(torch.uint8).view(-1).copy_(st[:nf], non_blocking=True)
        self._aux.copy_(st[nf:], non_blocking=True)
        self._stage_free[slot].record(cur)
        self._stage_r ^= 1
        if not read_loss or lag == 0 or (self.world > 1 and not self._dp_peers):
            return self._step_on_static_batch(read_loss)
        if not hasattr(self, "_lag_stats"):
            self._lag_stats = torch.zeros((2, 4), dtype=torch.float32).pin_memory()
            self._lag_ev = [torch.cuda.Event(), torch.cuda.Event()]
            self._lag_n = 0
        self._step_on_static_batch(False)
        k = self._lag_n & 1
        self._lag_stats[k].copy_(self._dp_reduce_stats() if self.world > 1 else self.head.stats, non_blocking=True)
        self._lag_ev[k].record(cur)
        self._lag_n += 1
        return self._read_lagged(k ^ 1) if self._lag_n > 1 else None

    def _read_lagged(self, k):
        self._lag_ev[k].synchronize()
        return float(self._lag_stats[k, 0]), float(self._lag_stats[k, 1]) / self.b_global

    def drain_prefetched(self):
        """Result of the last step enqueued with lag=1 (None if there is none)."""
        if getattr(self, "_lag_n", 0) == 0:
            return None
        out = self._read_lagged((self._lag_n - 1) & 1)
        self._lag_n = 0
        return out

    def _run_graphed(self):
        """The whole iteration (gather, 8+7+1 GEMMs, tail, memsets, check/AdamW/scaler) as one CUDA graph; the
        per-iteration scalars (indices, lr, loss weight, grad scale) are read from device memory."""
        if self._graph is None:
            if self._warm < 2:  # eager iterations first: one-time kernel attribute setup, tensor maps
                self._warm += 1
                self._enqueue_compute()
                return
            if self.world == 1 or self._dp_peers:
                # data parallel over peer memory: the optimiser kernels and their cross-GPU synchronisation are kernels on this
                # stream, so the whole iteration is ONE graph, as on one GPU
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self._enqueue_compute()
                self._graph = (g,)
            else:
                # data parallel through NCCL: the all-reduce stays outside the graphs (two graphs around it)
                ga, gb = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
                with torch.cuda.graph(ga):
                    self._enqueue_compute(part="fwd_bwd")
                with torch.cuda.graph(gb):
                    self._enqueue_compute(part="optimizer")
                self._graph = (ga, gb)
        if len(self._graph) == 1:
            self._graph[0].replay()
        else:
            self._graph[0].replay()
            self._dp_allreduce()
            self._graph[1].replay()

    # ------------------------------------------------------------------ epochs
    def run_epoch(self, on_iteration=None):
        """ace_trainer.py:454-497."""
        if self.iteration >= self.schedule.max_iterations:
            return False
        self.epoch += 1
        perm = torch.randperm(self.buffer_size, generator=self.training_generator)     # :466
        bg = self.b_global
        for start in range(0, self.buffer_size, bg):                                   # :469
            if start + bg > self.buffer_size:                                          # :473 drop ragged tail
                continue
            want = on_iteration is not None and (self.iteration % self.o.iterations_output == 0)
            ran = self.train_iteration(perm[start:start + bg], want_stats=want)
            if ran and want:
                on_iteration(self)
            if not ran:
                # the reference keeps calling training_step for the rest of the epoch; each call returns at once
                break
        if self.iteration >= self.schedule.max_iterations:
            self.finish()
        return True
