"""Timing probe of the fused layer-chain kernels (head_chain4.cu): CUDA-event timings of the forward chain and of the full
forward + tail + backward, plus the in-kernel clock64 timeline of one launch (ACEZ_CHAIN_DBG=1 is set here).

    python tools/probe_chain_time.py
"""
import ctypes as C
import os
import sys

os.environ["ACEZ_CHAIN_DBG"] = "1"
os.environ["ACEZ_HEAD_CHAIN"] = "1"
sys.path.insert(0, ".")
import numpy as np
import torch

import bench
from acezero_b200 import _lib
from acezero_b200.head import HeadEngine
from oracle import ace_ref

B = 5120
SLOTS = 8 + 8 * 20
dev = torch.device("cuda")


def timeit(fn, reps=30):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    e0.record()
    for _ in range(reps):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1000.0


def stamps(lib):
    buf = np.zeros(1024 * SLOTS, dtype=np.int64)
    n = C.c_int(0)
    _lib.check(lib.acez_debug_chain_clocks(buf.ctypes.data_as(C.c_void_p), buf.size, C.byref(n)))
    return buf[:n.value * SLOTS].reshape(n.value, SLOTS)


def show(st, cta, n_steps, title):
    t0 = st[cta, 0]
    print(f"  {title} CTA {cta}: total {st[cta, 1] - t0} cycles")
    print("   step  mma:own0  peer0  peer3 retired | epi:start peerfree  box0   box2")
    for s in range(n_steps):
        r = st[cta, 8 + 8 * s: 16 + 8 * s] - t0
        print(f"   {s:3d} " + " ".join(f"{int(x):7d}" for x in r[:4]) + " | " + " ".join(f"{int(x):7d}" for x in r[4:8]))


def main():
    bt = {k: v.to(dev) for k, v in ace_ref.synth_batch(5, B).items()}
    head = HeadEngine(1, True, (0, 0, 0), max_rows=B, training=True)
    head.load_state(ace_ref.make_head_state(200, 1, True))
    assert head.fused_chain
    lib = head.lib
    head.input_buffer(B).copy_(bt["features"])
    lp = head.loss_params("dyntanh", 30.0, B)

    def fwd():
        _lib.check(lib.acez_head_forward(head.plan, None, B, None, _lib.stream_ptr()))

    def full():
        head.train_fwd_bwd(B, lp, bt["target_px"], bt["intrinsics"], bt["intrinsics_inv"], aug_inv=bt["aug_poses_inv"],
                           pose_inv=bt["poses_inv"], use_device_scale=True)

    t_f = timeit(fwd)
    t_a = timeit(full)
    fwd()
    torch.cuda.synchronize()
    st_f = stamps(lib)
    tot_f = st_f[:, 1] - st_f[:, 0]
    full()
    torch.cuda.synchronize()
    st = stamps(lib)   # the last chain launch of `full` is the dgrad chain
    tot_d = st[:, 1] - st[:, 0]
    print(f"forward chain {t_f:7.1f} us  fwd+tail+bwd {t_a:7.1f} us | median CTA cycles "
          f"fwd {int(np.median(tot_f))} dgrad {int(np.median(tot_d))}", flush=True)
    show(st_f, 0, head.L, "fwd")
    show(st, 0, head.L - 1, "dgrad")


if __name__ == "__main__":
    main()
