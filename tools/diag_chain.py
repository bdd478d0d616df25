"""Localise a mismatch of the fused layer-chain kernels (head_chain4.cu) against the per-layer GEMM path.

Runs one training forward + backward with both paths on the same inputs and prints, per layer buffer (ACT / XTRA / DZ)
and per 64-column box, the worst relative difference -- so that a failure points at a role (own half vs. peer half of
a tile = DSMEM exchange; first layer vs. later = operand publication; all boxes = descriptors).
    python tools/diag_chain.py [rows]
"""
import os
import sys

sys.path.insert(0, ".")
import torch

from oracle import ace_ref

rows = int(sys.argv[1]) if len(sys.argv) > 1 else 384
nb = int(sys.argv[2]) if len(sys.argv) > 2 else 1


def run(chain):
    os.environ["ACEZ_HEAD_CHAIN"] = str(chain)
    from acezero_b200.head import HeadEngine
    sd = ace_ref.make_head_state(200, nb, True)
    eng = HeadEngine(nb, True, (0.0, 0.0, 0.0), max_rows=rows, training=True)
    eng.load_state(sd)
    eng.scaler_state[0] = 1024.0
    bt = {k: v.cuda() for k, v in ace_ref.synth_batch(301, rows).items()}
    lp = eng.loss_params("dyntanh", 30.0, rows)
    eng.workspace.zero_()
    eng.sync_weights()
    eng.train_fwd_bwd(rows, lp, bt["target_px"], bt["intrinsics"], bt["intrinsics_inv"], aug_inv=bt["aug_poses_inv"],
                      pose_inv=bt["poses_inv"], target_crds=bt["target_crds"], features=bt["features"])
    torch.cuda.synchronize()
    ws = eng.workspace.clone()
    grads = eng.grads.clone()
    return eng, ws, grads


def main():
    print(f"rows={rows} nb={nb}", flush=True)
    e0, ws0, g0 = run(0)
    print("layer path done", flush=True)
    e1, ws1, g1 = run(1)
    print("chain path done", flush=True)
    L = e0.L
    n = e0.max_rows * 512 * 2
    nres = 1 + nb

    def view(ws, off, i):
        o = off + i * n
        return ws[o:o + rows * 512 * 2].view(torch.float16).view(rows, 512).float()

    # workspace layout (head.cu head_layout), offsets from the plan's 1024-aligned base: w16 | w3h | act | resx | xtra | dz
    def up(v):
        return (v + 1023) // 1024 * 1024
    act_rel = up(L * 512 * 512 * 2) + up(4 * 512 * 2)
    base0, base1 = e0._input_off - act_rel, e1._input_off - act_rel
    xtra_rel = up(act_rel + (L + 1) * n)
    dz_rel = up(xtra_rel + nres * n)
    # (XTRA is only written by the per-layer path: the chain keeps ReLU masks as bit words)
    bufs = [("ACT", act_rel, L + 1), ("DZ", dz_rel, L)]
    for name, off, cnt in bufs:
        for i in range(cnt):
            a, b = view(ws1, base1 + off, i), view(ws0, base0 + off, i)
            scale = float(b.abs().max()) + 1e-20
            d = (a - b).abs() / scale
            per_box = [float(d[:, 64 * k:64 * k + 64].max()) for k in range(8)]
            per_tile = [float(d[t:t + 128].max()) for t in range(0, rows, 128)]
            nz = float((a != 0).float().mean())
            print(f"{name}[{i}] scale {scale:.3e} nonzero {nz:.2f} max rel diff per box: " +
                  " ".join(f"{x:.1e}" for x in per_box) + " | per tile: " + " ".join(f"{x:.1e}" for x in per_tile[:6]),
                  flush=True)
    rel = float((g1 - g0).norm() / (g0.norm() + 1e-20))
    print(f"grads rel L2 diff {rel:.3e}; stats layer {e0.stats.tolist()} chain {e1.stats.tolist()}", flush=True)


if __name__ == "__main__":
    main()
