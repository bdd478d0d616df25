"""Host side of the ACE head: owns the flat fp32 parameter / gradient / AdamW-state buffers and the plan of
libacez.so (C ABI `acez_head_*`, `acez_adamw_step`). Mirrors the role of `ace_network.Head` + `ScheduleACE`'s
optimiser and GradScaler in the reference (ace_network.py:62-149, ace_schedule.py:106-126).
"""
import ctypes as C
import math

import torch

from . import _lib

HEAD_CHANNELS = 512
LAYER_STRIDE = 512 * 512 + 512

LOSS_TYPES = {"tanh": 0, "dyntanh": 0, "l1": 1, "l1+sqrt": 2, "l1+logl1": 3, "l1+log": 3}


def head_layer_names(num_head_blocks):
    names = ["res3_conv1", "res3_conv2", "res3_conv3"]
    for b in range(num_head_blocks):
        names += [f"{b}c0", f"{b}c1", f"{b}c2"]
    return names + ["fc1", "fc2"]


HYPER_RING = 64


class HeadEngine:
    """Flat-buffer head. `params` is one fp32 CUDA tensor; `views()` exposes reference-named tensors aliasing it."""

    def __init__(self, num_head_blocks=1, use_homogeneous=True, mean=(0.0, 0.0, 0.0), max_rows=5120, training=False,
                 homogeneous_min_scale=0.01, homogeneous_max_scale=4.0, device="cuda", h_beta=None, max_inv_scale=None,
                 min_inv_scale=None, peer_group=None):
        self.lib = _lib.load()
        _lib.check(self.lib.acez_device_check(), "acez_device_check")
        self.device = torch.device(device)
        self.num_head_blocks = num_head_blocks
        self.use_homogeneous = bool(use_homogeneous)
        self.max_rows = int(max_rows)
        self.training = bool(training)
        self.names = head_layer_names(num_head_blocks)
        self.L = len(self.names)
        self.C3 = 4 if use_homogeneous else 3
        # the de-homogenisation constants the reference's forward reads are BUFFERS of the state dict (ace_network.py:108-114,
        # 139-144): a checkpoint stored in fp16 carries h_beta = 0.92432 and min_inv_scale = 100.0, not the values recomputed
        # from max_scale / min_scale — callers that hold the buffers pass them
        self.max_inv_scale = 1.0 / homogeneous_max_scale if max_inv_scale is None else float(max_inv_scale)
        self.min_inv_scale = 1.0 / homogeneous_min_scale if min_inv_scale is None else float(min_inv_scale)
        self.h_beta = math.log(2) / (1.0 - self.max_inv_scale) if h_beta is None else float(h_beta)
        self.mean = torch.as_tensor(mean, dtype=torch.float32).reshape(3).clone()
        self.cfg = self._config()
        self.n_params = int(self.lib.acez_head_param_count(C.byref(self.cfg)))
        assert self.n_params == self.L * LAYER_STRIDE + self.C3 * 512 + self.C3
        # Data parallel over NVLink peer memory (peer_group = a torch.distributed group of the GPUs of this box): parameters,
        # gradient and workspace are symmetric-memory allocations, so that the optimiser kernels of csrc/adamw_dp.cu can read
        # the other ranks' gradients and write the other ranks' weights directly
        self.peer = None
        self._symm = None
        if peer_group is not None and training:
            import torch.distributed._symmetric_memory as symm_mem
            self._symm = symm_mem
            self._peer_group = peer_group
            self.params = symm_mem.empty(self.n_params, dtype=torch.float32, device=self.device).zero_()
            self.grads_full = symm_mem.empty(self.n_params + 4, dtype=torch.float32, device=self.device).zero_()
        else:
            self.params = torch.zeros(self.n_params, device=self.device, dtype=torch.float32)
        # 4 spare floats behind the gradient: data-parallel runs carry the GradScaler flag and the loss statistics through the
        # SAME reduction as the gradient
        if self._symm is None:
            self.grads_full = torch.zeros(self.n_params + 4, device=self.device, dtype=torch.float32) if training else None
        self.grads = self.grads_full[:self.n_params] if training else None
        self.exp_avg = torch.zeros_like(self.params) if training else None
        self.exp_avg_sq = torch.zeros_like(self.params) if training else None
        self.plan = None
        self._build_plan()
        # device-resident optimiser / GradScaler state (no host sync in the step)
        # hyper: lr, beta1, beta2, eps, weight_decay (read by acez_adamw_step), [5] = loss weight of the iteration
        self.hyper = torch.tensor([1e-3, 0.9, 0.999, 1e-8, 0.01, 50.0, 0.0, 0.0], device=self.device, dtype=torch.float32)
        self.scaler_state = torch.tensor([65536.0, 0.0, 0.0, 0.0], device=self.device, dtype=torch.float32)
        self.found_inf = torch.zeros(1, device=self.device, dtype=torch.int32)
        self.stats = torch.zeros(4, device=self.device, dtype=torch.float32)
        # ring of pinned staging rows: the host may run many iterations ahead of the device, and every queued copy
        # must still find ITS iteration's scalars when the DMA finally executes
        self._hyper_host = torch.tensor([1e-3, 0.9, 0.999, 1e-8, 0.01, 50.0, 0.0, 0.0]).repeat(HYPER_RING, 1).pin_memory()
        self._hyper_events = [None] * HYPER_RING
        self._hyper_slot = 0

    # ------------------------------------------------------------------ plan / buffers
    def _config(self):
        cfg = _lib.HeadConfig()
        cfg.num_res_blocks = 1 + self.num_head_blocks
        cfg.use_homogeneous = int(self.use_homogeneous)
        cfg.max_rows = self.max_rows
        cfg.training = int(self.training)
        for i in range(3):
            cfg.mean[i] = float(self.mean[i])
        cfg.h_beta = self.h_beta
        cfg.max_inv_scale = self.max_inv_scale
        cfg.min_inv_scale = self.min_inv_scale
        return cfg

    def _build_plan(self):
        if self.plan is not None:
            self.lib.acez_head_plan_destroy(self.plan)
            self.plan = None
        self.cfg = self._config()
        ws_bytes = int(self.lib.acez_head_workspace_bytes(C.byref(self.cfg)))
        if getattr(self, "workspace", None) is None or self.workspace.numel() < ws_bytes:
            if self._symm is not None:
                if getattr(self, "workspace", None) is not None:
                    raise RuntimeError("a peer-memory head cannot grow its workspace (create it with the final max_rows)")
                self.workspace = self._symm.empty(ws_bytes, dtype=torch.uint8, device=self.device)
            else:
                self.workspace = torch.empty(ws_bytes, device=self.device, dtype=torch.uint8)
        plan = C.c_void_p()
        rc = self.lib.acez_head_plan_create(C.byref(self.cfg), _lib.ptr(self.params), _lib.ptr(self.grads),
                                            _lib.ptr(self.workspace), ws_bytes, C.byref(plan))
        _lib.check(rc, "acez_head_plan_create")
        self.plan = plan
        in_ptr = self.lib.acez_head_input_ptr(self.plan)
        self._input_off = in_ptr - self.workspace.data_ptr()

    @property
    def fused_chain(self):
        """True when the plan runs each pass over the hidden layers as one fused cluster kernel (head_chain4.cu)."""
        return bool(self.lib.acez_head_plan_fused_chain(self.plan))

    def chain_kernel_symbol(self):
        """Name of the kernel that runs the forward pass over the hidden layers (for profile bookkeeping in bench.py)."""
        return "head_chain4_kernel<FWD>" if self.fused_chain else "gemm_tcgen05_kernel<FWD>"

    def resize(self, max_rows):
        if max_rows > self.max_rows:
            self.max_rows = int(max_rows)
            self.workspace = None
            self._build_plan()
            self.sync_weights()

    def set_mean(self, mean):
        self.mean = torch.as_tensor(mean, dtype=torch.float32).reshape(3).clone().cpu()
        self._build_plan()

    def __del__(self):
        try:
            if self.plan is not None:
                self.lib.acez_head_plan_destroy(self.plan)
        except Exception:
            pass

    def input_buffer(self, rows):
        """fp16 [rows,512] view of the plan's input activation buffer (write features here to skip a copy)."""
        n = rows * 512 * 2
        return self.workspace[self._input_off:self._input_off + n].view(torch.float16).view(rows, 512)

    # ------------------------------------------------------------------ parameters
    def views(self):
        """dict name -> tensor view into `params` with the reference's state_dict names and OIHW shapes."""
        out = {}
        for l, n in enumerate(self.names):
            o = l * LAYER_STRIDE
            out[n + ".weight"] = self.params[o:o + 512 * 512].view(512, 512, 1, 1)
            out[n + ".bias"] = self.params[o + 512 * 512:o + LAYER_STRIDE]
        o = self.L * LAYER_STRIDE
        out["fc3.weight"] = self.params[o:o + self.C3 * 512].view(self.C3, 512, 1, 1)
        out["fc3.bias"] = self.params[o + self.C3 * 512:o + self.C3 * 512 + self.C3]
        return out

    def grad_views(self):
        out = {}
        for l, n in enumerate(self.names):
            o = l * LAYER_STRIDE
            out[n + ".weight"] = self.grads[o:o + 512 * 512].view(512, 512, 1, 1)
            out[n + ".bias"] = self.grads[o + 512 * 512:o + LAYER_STRIDE]
        o = self.L * LAYER_STRIDE
        out["fc3.weight"] = self.grads[o:o + self.C3 * 512].view(self.C3, 512, 1, 1)
        out["fc3.bias"] = self.grads[o + self.C3 * 512:o + self.C3 * 512 + self.C3]
        return out

    def load_state(self, sd):
        v = self.views()
        with torch.no_grad():
            for k, t in v.items():
                t.copy_(sd[k].to(self.device, torch.float32).reshape(t.shape))
        if "mean" in sd:
            self.set_mean(sd["mean"].reshape(3).float().cpu())
        self.sync_weights()

    def sync_weights(self, stream=None):
        _lib.check(self.lib.acez_head_sync_weights(self.plan, _lib.stream_ptr(stream)), "acez_head_sync_weights")

    # ------------------------------------------------------------------ forward
    def forward(self, features, out=None, stream=None):
        """features: fp16 CUDA [rows,512] (or None = already written to input_buffer). Returns fp32 [rows,3]."""
        rows = features.shape[0] if features is not None else out.shape[0]
        if rows > self.max_rows:
            self.resize(rows)
        if features is not None:
            if features.dtype != torch.float16:
                features = features.half()
            features = features.contiguous()
        if out is None:
            out = torch.empty((rows, 3), device=self.device, dtype=torch.float32)
        rc = self.lib.acez_head_forward(self.plan, _lib.ptr(features), rows, _lib.ptr(out), _lib.stream_ptr(stream))
        _lib.check(rc, "acez_head_forward")
        return out

    # ------------------------------------------------------------------ training
    def loss_params(self, loss_type, loss_weight, divisor, use_depth=False, depth_min=0.1, depth_max=1000.0,
                    hard_clamp=1000.0, inlier_px=10.0, depth_target=10.0, grad_scale=1.0):
        return _lib.LossParams(LOSS_TYPES[loss_type], float(loss_weight), depth_min, depth_max, hard_clamp, inlier_px,
                               depth_target, int(use_depth), float(grad_scale), int(divisor))

    def train_fwd_bwd(self, rows, lp, target_px, K, Kinv, aug_inv=None, pose_inv=None, P=None, target_crds=None,
                      features=None, d_P=None, d_Kdiag=None, sc_out=None, use_device_scale=True,
                      use_device_loss_weight=False, stream=None):
        tb = _lib.TrainBatch()
        tb.features = features.data_ptr() if features is not None else None
        tb.target_px_b2 = target_px.data_ptr()
        tb.P_b34 = P.data_ptr() if P is not None else None
        tb.aug_inv_b34 = aug_inv.data_ptr() if aug_inv is not None else None
        tb.pose_inv_b44 = pose_inv.data_ptr() if pose_inv is not None else None
        tb.K_b33 = K.data_ptr()
        tb.Kinv_b33 = Kinv.data_ptr()
        tb.target_crds_b3 = target_crds.data_ptr() if target_crds is not None else None
        tb.d_P_b34 = d_P.data_ptr() if d_P is not None else None
        tb.d_Kdiag_b2 = d_Kdiag.data_ptr() if d_Kdiag is not None else None
        tb.sc_out_b3 = sc_out.data_ptr() if sc_out is not None else None
        tb.grad_scale_dev = self.scaler_state.data_ptr() if use_device_scale else None
        tb.loss_weight_dev = (self.hyper.data_ptr() + 20) if use_device_loss_weight else None
        rc = self.lib.acez_head_train_fwd_bwd(self.plan, rows, C.byref(lp), C.byref(tb), _lib.ptr(self.stats),
                                              _lib.ptr(self.found_inf), _lib.stream_ptr(stream))
        _lib.check(rc, "acez_head_train_fwd_bwd")

    def set_hyper(self, lr, loss_weight=None, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=0.01):
        """Stage this iteration's host-computed scalars (pinned -> device, asynchronous, stream ordered)."""
        slot = self._hyper_slot
        prev = self._hyper_host[slot - 1]
        self._hyper_slot = (slot + 1) % HYPER_RING
        ev = self._hyper_events[slot]
        if ev is None:
            ev = self._hyper_events[slot] = torch.cuda.Event()
        else:
            ev.synchronize()          # the copy that last used this row (HYPER_RING iterations ago) has executed
        h = self._hyper_host[slot]
        h[0], h[1], h[2], h[3], h[4] = lr, beta1, beta2, eps, weight_decay
        h[5] = float(prev[5]) if loss_weight is None else loss_weight
        self.hyper.copy_(h, non_blocking=True)
        ev.record()

    # ------------------------------------------------------------------ data parallel over peer memory
    def setup_peers(self):
        """Rendezvous of the symmetric allocations (collective over the peer group): peer pointers of every rank's parameters,
        gradient, fp16 weight shadows and flag array."""
        import torch.distributed as dist
        sm, g = self._symm, self._peer_group
        world, rank = dist.get_world_size(g), dist.get_rank(g)
        # [0, 8) shard verdicts, [16, 40) three rows of epoch signals written by the peers (csrc/adamw_dp.cu)
        self.dp_flags = sm.empty(64, dtype=torch.int32, device=self.device).zero_()
        self.dp_sync_state = torch.zeros(4, dtype=torch.int32, device=self.device)
        import os
        torch.cuda.synchronize()
        hp = sm.rendezvous(self.params, g)
        hg = sm.rendezvous(self.grads_full, g)
        hw = sm.rendezvous(self.workspace, g)
        hf = sm.rendezvous(self.dp_flags, g)
        off16 = int(self.lib.acez_head_w16_ptr(self.plan, 0)) - self.workspace.data_ptr()
        off3 = int(self.lib.acez_head_w16_ptr(self.plan, 1)) - self.workspace.data_ptr()
        arr = lambda ptrs: (C.c_void_p * world)(*[int(p) for p in ptrs])
        shard = int(self.lib.acez_adamw_dp_shard(self.n_params, world))
        # NVLink SHARP: multicast addresses of the same buffers when the fabric provides them (torch symmetric memory binds a
        # multicast object to every allocation if it can); ACEZ_DP_MULTICAST=0 forces the peer-to-peer path
        mc = None
        try:
            mcp = [int(getattr(h, "multicast_ptr", 0) or 0) for h in (hg, hw, hp)]
            # measured (round 2): at 2 GPUs the switch reduction is slower than peer loads (the same bytes cross the links twice),
            # from 4 GPUs on a rank receives 1/G of the gradient instead of pulling (G-1)/G of it
            want = os.environ.get("ACEZ_DP_MULTICAST", "auto")
            if all(mcp) and (want == "1" or (want == "auto" and world >= 4)):
                mc = (C.c_void_p * 4)(mcp[0], mcp[1] + off16, mcp[1] + off3, mcp[2])
        except Exception:  # noqa: BLE001  (older torch: no multicast support)
            mc = None
        self.dp_multicast = mc
        self.peer = {
            "world": world, "rank": rank, "shard": shard, "handles": (hp, hg, hw, hf),
            "params": arr(hp.buffer_ptrs), "grads": arr(hg.buffer_ptrs), "flags": arr(hf.buffer_ptrs),
            "w16": arr([p + off16 for p in hw.buffer_ptrs]), "w3h": arr([p + off3 for p in hw.buffer_ptrs]),
            "reduced": torch.zeros(shard + 4, device=self.device, dtype=torch.float32),
        }
        return self.peer

    def adamw_step_peers(self, stream=None):
        """Optimiser step of one data-parallel iteration over peer memory (csrc/adamw_dp.cu): reduce this rank's shard of the
        gradient from all ranks, AdamW on the shard + the new fp16 weights to all ranks, synchronised across the GPUs inside
        the kernels (no host-side barrier: the step can be captured in a CUDA graph)."""
        P = self.peer
        _lib.check(self.lib.acez_adamw_dp_step(P["grads"], P["flags"], P["w16"], P["w3h"], P["params"], P["world"], P["rank"],
                                               self.n_params, _lib.ptr(P["reduced"]), _lib.ptr(self.params), _lib.ptr(self.exp_avg),
                                               _lib.ptr(self.exp_avg_sq), _lib.ptr(self.hyper), _lib.ptr(self.scaler_state),
                                               _lib.ptr(self.found_inf), C.c_void_p(self.grads_full.data_ptr() + 4 * self.n_params),
                                               _lib.ptr(self.dp_sync_state), _lib.ptr(self.stats), self.dp_multicast, self.L, self.C3,
                                               _lib.stream_ptr(stream)),
                   "acez_adamw_dp_step")

    def gather_params_from_shards(self):
        """fp32 master weights live on their owner rank during peer-memory training: collect them on every rank (export)."""
        if self.peer is None:
            return
        import torch.distributed as dist
        P = self.peer
        world, rank, shard = P["world"], P["rank"], P["shard"]
        mine = torch.zeros(shard, device=self.device, dtype=torch.float32)
        lo = rank * shard
        hi = min(lo + shard, self.n_params)
        if hi > lo:
            mine[:hi - lo] = self.params[lo:hi]
        full = torch.empty(world * shard, device=self.device, dtype=torch.float32)
        dist.all_gather_into_tensor(full, mine, group=self._peer_group)
        self.params.copy_(full[:self.n_params])

    def adamw_step(self, use_scaler=True, flag_complete=True, stream=None, check_flag_slot=False):
        """flag_complete: found_inf already covers all gradients (true after train_fwd_bwd).
        check_flag_slot (data parallel through NCCL): the check pass also covers grads_full[n_params], the slot the ranks'
        local flags travelled in (+inf when set), so no separate unpack kernels are needed."""
        rc = self.lib.acez_adamw_step(_lib.ptr(self.params), _lib.ptr(self.grads), _lib.ptr(self.exp_avg),
                                      _lib.ptr(self.exp_avg_sq), self.n_params, _lib.ptr(self.hyper),
                                      _lib.ptr(self.scaler_state), _lib.ptr(self.found_inf),
                                      (2 if flag_complete else (3 if check_flag_slot else 1)) if use_scaler else 0, self.plan,
                                      _lib.stream_ptr(stream))
        _lib.check(rc, "acez_adamw_step")
