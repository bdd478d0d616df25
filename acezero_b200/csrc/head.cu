// ACE head (reference ace_network.py:62-149) forward / backward on sm_100a, plus the fused "tail" kernel that
// joins fc3, the homogeneous de-normalisation (ace_network.py:139-147) and the reprojection loss + backward
// (ace_trainer.py:521-613) into one pass over the last hidden activation.
//
// Data layout in HBM (all caller-owned; see acez_head_workspace_bytes):
//   params / grads : flat fp32, per hidden layer W[512,512] then b[512]; fc3 W[C3,512], b[C3] last
//   W16            : [L][512][512] fp16 shadow of the hidden-layer weights (autocast's cast of the conv weights)
//   W3h            : [4][512] fp16 shadow of fc3
//   ACT            : [L+1][max_rows][512] fp16; ACT[l] is the input of hidden layer l, ACT[L] feeds fc3
//   XTRA           : [nres][max_rows][512] fp16 post-ReLU output of the last conv of each residual block (ReLU mask)
//   DZ             : [L][max_rows][512] fp16 gradient w.r.t. the pre-activation of each hidden layer (x grad_scale)
//   GRES           : [max_rows][512] fp16 running skip-path gradient
//   MASKB          : [L+1][max_rows][64 B] one bit per channel: ReLU masks written by the fused forward chain and read
//                    by the fused dgrad chain (head_chain4.cu); MASKB[l] belongs to ACT[l]
#include <stdlib.h>

#include <vector>

#include "adamw.cuh"
#include "gemm.cuh"
#include "gemm2cta.cuh"
#include "schedule.cuh"
#include "head_chain.cuh"
#include "repro_loss.cuh"

namespace acez {

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

}  // namespace acez

struct acez_head_plan {
  acez_head_config cfg;
  int L, nres, C3;
  size_t n_params;
  float* params;
  float* grads;
  __half* W16;
  __half* W3h;
  __half* ACT;
  __half* XTRA;
  __half* DZ;
  __half* GRES;
  uint8_t* MASKB;
  float* G3;
  float* FC3PART;
  float* WBIAS;
  float* BLKPART;
  unsigned int* BLKCOUNT;
  bool counters_zeroed;
  size_t act_stride;  // max_rows * 512
  int prepared_rows;
  int prepared_training;
  std::vector<acez::GemmLaunch> fwd;
  std::vector<acez::GemmLaunch> dgrad;
  acez::GemmLaunch wgrad;    // per-layer plans: all weight gradients in one cta_group::1 launch (grid.z = layer)
  // fused layer chains (head_chain4.cu): one launch for all hidden layers of a pass
  int use_chain;
  acez::ChainLaunch chain_fwd, chain_bwd;
  acez::Gemm2Launch wgrad2;  // chain plans: all weight gradients in one cta_group::2 launch (gemm2cta.cu)
};

namespace acez {

struct HeadLayout {
  size_t w16, w3h, act, xtra, dz, gres, maskb, g3, fc3part, wbias, blkpart, total;
};

static HeadLayout head_layout(const acez_head_config& cfg) {
  const int nres = cfg.num_res_blocks;
  const int L = 3 * nres + 2;
  const size_t rows = (size_t)cfg.max_rows;
  HeadLayout o{};
  size_t off = 0;
  o.w16 = off; off = align_up(off + (size_t)L * kC * kC * 2, 1024);
  o.w3h = off; off = align_up(off + 4 * kC * 2, 1024);
  o.act = off; off = align_up(off + (size_t)(L + 1) * rows * kC * 2, 1024);
  if (cfg.training) {
    o.xtra = off; off = align_up(off + (size_t)nres * rows * kC * 2, 1024);
    o.dz = off; off = align_up(off + (size_t)L * rows * kC * 2, 1024);
    o.gres = off; off = align_up(off + rows * kC * 2, 1024);
    o.maskb = off; off = align_up(off + (size_t)(L + 1) * rows * 64, 1024);
    o.g3 = off; off = align_up(off + rows * 4 * sizeof(float), 1024);
    o.fc3part = off; off = align_up(off + ((rows + 31) / 32) * (size_t)(4 * kC + 4) * sizeof(float), 1024);
    o.wbias = off; off = align_up(off + (size_t)L * 2 * 4 * 256 * sizeof(float), 1024);  // wgrad bias partials [L][2][<=4][256]
  }
  o.blkpart = off; off = align_up(off + 4096 * 8 * sizeof(float) + 4096, 1024);  // tail per-block partials + 1024 counters
  o.total = off;
  return o;
}

// ----------------------------------------------------------------------------------------------
// small kernels
// ----------------------------------------------------------------------------------------------
__global__ void cast_weights_kernel(const float* __restrict__ params, __half* __restrict__ W16,
                                    __half* __restrict__ W3h, int L, int C3) {
  const size_t n_hidden = (size_t)L * kC * kC;
  const size_t n_total = n_hidden + (size_t)4 * kC;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_total; i += (size_t)gridDim.x * blockDim.x) {
    if (i < n_hidden) {
      const size_t l = i / ((size_t)kC * kC), r = i % ((size_t)kC * kC);
      W16[i] = __float2half_rn(params[l * kLayerStride + r]);
    } else {
      const size_t r = i - n_hidden;  // [4][512]
      const size_t row = r / kC;
      W3h[r] = (row < (size_t)C3) ? __float2half_rn(params[(size_t)L * kLayerStride + r]) : __float2half_rn(0.f);
    }
  }
}

__global__ void gather_rows_kernel(const uint8_t* __restrict__ src, const int64_t* __restrict__ idx, int rows,
                                   int row_bytes, uint8_t* __restrict__ dst) {
  // one warp per row, 16-byte vectors when the row size allows
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= rows) return;
  const uint8_t* s = src + (size_t)idx[warp] * row_bytes;
  uint8_t* d = dst + (size_t)warp * row_bytes;
  if ((row_bytes & 15) == 0 && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0) {
    for (int o = lane * 16; o < row_bytes; o += 512) *reinterpret_cast<uint4*>(d + o) = *reinterpret_cast<const uint4*>(s + o);
  } else if ((row_bytes & 3) == 0) {
    for (int o = lane * 4; o < row_bytes; o += 128) *reinterpret_cast<uint32_t*>(d + o) = *reinterpret_cast<const uint32_t*>(s + o);
  } else {
    for (int o = lane * 2; o < row_bytes; o += 64) *reinterpret_cast<uint16_t*>(d + o) = *reinterpret_cast<const uint16_t*>(s + o);
  }
}

// All arrays of the patch buffer in one launch: blockIdx.y selects the array (reference ace_trainer.py:485-494
// issues 8 index kernels + 8 H2D index copies per iteration).
struct MultiGather {
  const uint8_t* src[8];
  uint8_t* dst[8];
  int row_bytes[8];
};
// Optional rider of the batch gather: the device-side schedule of the iteration (schedule.cuh) evaluated by thread 0 of
// block 0, so that the first kernel of the iteration's graph does both (a separate one-thread kernel costs ~3 us of launch)
struct GatherSched {
  int enabled;
  acez_schedule_params p;
  float* state;
  const float* inlier_count;
  float* hyper;
};
__global__ void gather_rows_multi_kernel(const MultiGather g, const int64_t* __restrict__ idx, int rows, int n_arrays,
                                         const GatherSched sch) {
  pdl_wait();
  pdl_launch_dependents();
  // the schedule rides in an EXTRA block at the end of the grid (its serial double-precision chain would otherwise lengthen a
  // block that also gathers rows: measured +2 us)
  if (sch.enabled && blockIdx.x == gridDim.x - 1) {
    if (threadIdx.x == 0) schedule_step_device(sch.p, sch.state, sch.inlier_count, sch.hyper);
    return;
  }
  // one warp per batch row, all arrays: the 1 KB feature row moves as 2 x 16 B per lane, the small arrays as words
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= rows) return;
  const size_t src_row = (size_t)idx[warp];
  // Two passes: ALL loads of the row (every array) are issued before the first store, so the row costs one memory round trip
  // instead of one per array (round 2: 8.6 us for 6.3 MB with the arrays copied one after the other). Register paths: array 0
  // (the 1 KB feature row) as up to two 16-byte trips of the warp, the small arrays as one 4-byte (<= 128 B rows) or one 2-byte
  // (<= 64 B rows) trip; anything else takes the plain loop in the second pass.
  uint4 f16[2];
  uint32_t v4[8];
  uint16_t v2[8];
  const int rb0 = g.row_bytes[0];
  const bool big0 = (rb0 & 15) == 0 && rb0 <= 1024 && ((reinterpret_cast<uintptr_t>(g.src[0]) | reinterpret_cast<uintptr_t>(g.dst[0])) & 15) == 0;
  if (big0) {
    const uint8_t* s = g.src[0] + src_row * rb0;
    if (lane * 16 < rb0) f16[0] = *reinterpret_cast<const uint4*>(s + lane * 16);
    if (lane * 16 + 512 < rb0) f16[1] = *reinterpret_cast<const uint4*>(s + lane * 16 + 512);
  }
#pragma unroll
  for (int a = 0; a < 8; ++a) {
    if (a >= n_arrays || (a == 0 && big0)) continue;
    const int rb = g.row_bytes[a];
    const uint8_t* s = g.src[a] + src_row * rb;
    if ((rb & 3) == 0 && rb <= 128) {
      if (lane * 4 < rb) v4[a] = *reinterpret_cast<const uint32_t*>(s + lane * 4);
    } else if ((rb & 1) == 0 && rb <= 64) {
      if (lane * 2 < rb) v2[a] = *reinterpret_cast<const uint16_t*>(s + lane * 2);
    }
  }
  if (big0) {
    uint8_t* d = g.dst[0] + (size_t)warp * rb0;
    if (lane * 16 < rb0) *reinterpret_cast<uint4*>(d + lane * 16) = f16[0];
    if (lane * 16 + 512 < rb0) *reinterpret_cast<uint4*>(d + lane * 16 + 512) = f16[1];
  }
#pragma unroll
  for (int a = 0; a < 8; ++a) {
    if (a >= n_arrays || (a == 0 && big0)) continue;
    const int rb = g.row_bytes[a];
    uint8_t* d = g.dst[a] + (size_t)warp * rb;
    if ((rb & 3) == 0 && rb <= 128) {
      if (lane * 4 < rb) *reinterpret_cast<uint32_t*>(d + lane * 4) = v4[a];
    } else if ((rb & 1) == 0 && rb <= 64) {
      if (lane * 2 < rb) *reinterpret_cast<uint16_t*>(d + lane * 2) = v2[a];
    } else {
      const uint8_t* s = g.src[a] + src_row * rb;
      if ((rb & 15) == 0 && ((reinterpret_cast<uintptr_t>(g.src[a]) | reinterpret_cast<uintptr_t>(g.dst[a])) & 15) == 0) {
        for (int o = lane * 16; o < rb; o += 512) *reinterpret_cast<uint4*>(d + o) = *reinterpret_cast<const uint4*>(s + o);
      } else if ((rb & 3) == 0) {
        for (int o = lane * 4; o < rb; o += 128) *reinterpret_cast<uint32_t*>(d + o) = *reinterpret_cast<const uint32_t*>(s + o);
      } else if ((rb & 1) == 0) {
        for (int o = lane * 2; o < rb; o += 64) *reinterpret_cast<uint16_t*>(d + o) = *reinterpret_cast<const uint16_t*>(s + o);
      } else {
        for (int o = lane; o < rb; o += 32) d[o] = s[o];
      }
    }
  }
}

// ----------------------------------------------------------------------------------------------
// tail kernel: fc3 + homogeneous + (loss + backward into DZ[L-1]) + per-block partial of the fc3 weight gradient.
// One block = 40 rows (8 warps x 5), three phases:
//   A  warp w, rows 5w..5w+4: the 4 fc3 dot products of a row (lane owns columns [16 lane, 16 lane + 16), its slice of the fc3
//      weights in registers, the 4 rows' activations stay in registers for phase C) -> shared memory
//   B  ONE THREAD PER ROW (warps 0, 1): de-homogenisation, pose compose, reprojection loss and its analytic backward, back through
//      the de-homogenisation -> g[4]. The per-row chain (divisions, exp / log / tanh) is latency bound; 32 rows advance in
//      parallel instead of one per warp with all lanes redundant (round 1: 20 us for 5120 rows)
//   C  warp w, rows 5w..5w+4: dX = g W3 with the ReLU mask -> DZ[L-1] (1 KB per row, coalesced) and the warp's partial of
//      dW3 = sum_rows g x^T; block partial -> FC3PART[block] (summed by fc3_reduce_kernel)
// ----------------------------------------------------------------------------------------------
struct TailArgs {
  int rows, C3, use_homogeneous, training;
  float mean[3], h_beta, max_inv_scale, min_inv_scale;
  const __half* x;      // ACT[L]  [rows,512]
  const __half* W3h;    // [4,512] fp16
  const float* b3;      // [C3] fp32
  float* sc_out;        // [rows,3] nullable
  // training
  acez_loss_params lp;
  const float* grad_scale_dev;  // nullable: overrides lp.grad_scale (GradScaler state lives on the device)
  const float* loss_weight_dev; // nullable: overrides lp.loss_weight (per-iteration dyntanh weight, graph-stable)
  const float* tpx; const float* Pin; const float* A; const float* T; const float* K; const float* Kinv; const float* G;
  float* d_P; float* d_Kdiag;
  const float* d_sc_in; // training == 2: gradient w.r.t. the scene coordinates supplied by the caller (autograd)
  __half* dz;           // DZ[L-1] [rows,512]
  float* fc3_part;      // nullable: [gridDim.x][4*512+4] per-block partials of dW3 / db3
  float* stats;         // [4]: written (not accumulated) by the last block to finish; [3] is a latch (OR with its old value)
  int* nonfinite;       // written (not OR-ed) by the last block: later kernels of the iteration OR into it
  float* blk_part;      // [gridDim.x][8] per-block partial sums
  unsigned int* blk_count;  // self-resetting completion counter
};

static constexpr int kTailThreads = 256;
static constexpr int kTailRW = 5;                                      // rows per warp
static constexpr int kTailRows = (kTailThreads / 32) * kTailRW;        // 40 rows per block: 128 blocks for 5120 rows = ONE wave on 148 SMs
                                                                       // (round 2: 32 rows = 160 blocks = two waves, 18 us instead of 9)
static constexpr int kTailAccBytes = (kTailThreads / 32) * 4 * kC * 4;  // dynamic smem of the fc3-gradient variant: 64 KB

__global__ void __launch_bounds__(kTailThreads) head_tail_kernel(const TailArgs a) {
  extern __shared__ float sAcc[];              // [8 warps][4][512] (only when a.fc3_part != nullptr)
  __shared__ float sS[kTailRows][4];           // fc3 outputs (fp16-rounded, as the autocast conv produces them)
  __shared__ float sG[kTailRows][4];           // gradient w.r.t. the fc3 outputs (fp16-rounded values)
  __shared__ float sRed[2][3];
  __shared__ int sLast;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int r0 = blockIdx.x * kTailRows;
  pdl_wait();
  pdl_launch_dependents();

  // ---- phase-B threads prefetch their row's geometry (212 B from 5 arrays) before the dot products ----
  const int brow = r0 + tid;
  const bool b_active = tid < kTailRows && brow < a.rows;
  float geoA[12], geoT[16], Kr[9], Ki[9], tpx0 = 0.f, tpx1 = 0.f;
  if (b_active && a.training == 1) {
    if (a.Pin != nullptr) {
#pragma unroll
      for (int k = 0; k < 3; ++k) *reinterpret_cast<float4*>(&geoA[4 * k]) = *reinterpret_cast<const float4*>(a.Pin + 12 * (size_t)brow + 4 * k);
    } else {
#pragma unroll
      for (int k = 0; k < 3; ++k) *reinterpret_cast<float4*>(&geoA[4 * k]) = *reinterpret_cast<const float4*>(a.A + 12 * (size_t)brow + 4 * k);
#pragma unroll
      for (int k = 0; k < 4; ++k) *reinterpret_cast<float4*>(&geoT[4 * k]) = *reinterpret_cast<const float4*>(a.T + 16 * (size_t)brow + 4 * k);
    }
#pragma unroll
    for (int k = 0; k < 9; ++k) { Kr[k] = a.K[9 * (size_t)brow + k]; Ki[k] = a.Kinv[9 * (size_t)brow + k]; }
    const float2 tp = *reinterpret_cast<const float2*>(a.tpx + 2 * (size_t)brow);
    tpx0 = tp.x; tpx1 = tp.y;
  }

  // ---- phase A: fc3 dot products ----
  __half2 w[4][8];   // this lane's slice of the fc3 weights: 4 rows x 16 columns
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const uint4* wp = reinterpret_cast<const uint4*>(a.W3h + j * kC + lane * 16);
    const uint4 t0 = wp[0], t1 = wp[1];
    const __half2* h0 = reinterpret_cast<const __half2*>(&t0);
    const __half2* h1 = reinterpret_cast<const __half2*>(&t1);
#pragma unroll
    for (int k = 0; k < 4; ++k) { w[j][k] = h0[k]; w[j][4 + k] = h1[k]; }
  }
  uint4 xr[kTailRW][2];
#pragma unroll
  for (int i = 0; i < kTailRW; ++i) {
    const int row = r0 + kTailRW * warp + i;
    if (row < a.rows) {
      const uint4* xp = reinterpret_cast<const uint4*>(a.x + (size_t)row * kC + lane * 16);
      xr[i][0] = xp[0]; xr[i][1] = xp[1];
    } else {
      xr[i][0] = make_uint4(0u, 0u, 0u, 0u); xr[i][1] = xr[i][0];
    }
  }
#pragma unroll
  for (int i = 0; i < kTailRW; ++i) {
    const __half2* xh = reinterpret_cast<const __half2*>(xr[i]);
    float d[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float2 xf = __half22float2(xh[k]);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 wf = __half22float2(w[j][k]);
        d[j] = fmaf(xf.x, wf.x, d[j]);
        d[j] = fmaf(xf.y, wf.y, d[j]);
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) d[j] = warp_sum(d[j]);
    if (lane < 4) {
      const float dj = lane == 0 ? d[0] : (lane == 1 ? d[1] : (lane == 2 ? d[2] : d[3]));
      const float bj = (lane < a.C3) ? __half2float(__float2half_rn(a.b3[lane])) : 0.f;
      sS[kTailRW * warp + i][lane] = __half2float(__float2half_rn(dj + bj));
    }
  }
  __syncthreads();

  // ---- phase B: one thread per row ----
  float loss_sum = 0.f, inl_sum = 0.f, valid_sum = 0.f;
  bool bad = false, bad_g = false;
  if (tid < kTailRows) {
    float g[4] = {0.f, 0.f, 0.f, 0.f};
    if (b_active) {
      acez_loss_params lp = a.lp;
      if (a.training && a.grad_scale_dev != nullptr) lp.grad_scale = *a.grad_scale_dev;
      if (a.training && a.loss_weight_dev != nullptr) lp.loss_weight = *a.loss_weight_dev;
      const float s0 = sS[tid][0], s1 = sS[tid][1], s2 = sS[tid][2], s3 = sS[tid][3];
      const float sv[3] = {s0, s1, s2};
      // homogeneous -> 3-D (ace_network.py:139-147), fp32
      float X[3], h = 1.f, sig = 0.f;
      bool h_pass = true;
      if (a.use_homogeneous) {
        const float bx = a.h_beta * s3;
        float sp;
        if (bx > 20.f) { sp = s3; sig = 1.f; }               // torch softplus threshold
        else { sp = log1pf(expf(bx)) / a.h_beta; sig = 1.f / (1.f + expf(-bx)); }
        h = sp + a.max_inv_scale;
        h_pass = h <= a.min_inv_scale;                          // clamp_(max=) backward mask
        h = fminf(h, a.min_inv_scale);
#pragma unroll
        for (int i = 0; i < 3; ++i) X[i] = sv[i] / h + a.mean[i];
      } else {
#pragma unroll
        for (int i = 0; i < 3; ++i) X[i] = sv[i] + a.mean[i];
      }
      if (a.sc_out != nullptr) {
        a.sc_out[(size_t)brow * 3 + 0] = X[0]; a.sc_out[(size_t)brow * 3 + 1] = X[1]; a.sc_out[(size_t)brow * 3 + 2] = X[2];
      }
      if (a.training) {
        RowLoss o;
        if (a.training == 2) {
          // external gradient (torch.autograd through the Regressor module): skip the loss, take dL/dX from the caller
#pragma unroll
          for (int i = 0; i < 3; ++i) o.gX[i] = a.d_sc_in[3 * (size_t)brow + i];
          o.loss = 0.f; o.valid = true; o.inlier = false; o.gK00 = o.gK11 = 0.f;
          o.gc[0] = o.gc[1] = o.gc[2] = 0.f;
        } else {
          float P[12];
          if (a.Pin != nullptr) {
#pragma unroll
            for (int k = 0; k < 12; ++k) P[k] = geoA[k];
          } else {
            compose_pose(geoA, geoT, P);
          }
          repro_row(lp, X, P, Kr, Ki, tpx0, tpx1, (lp.use_depth && a.G) ? a.G + 3 * (size_t)brow : nullptr, o);
          loss_sum = o.loss / (float)lp.divisor;
          inl_sum = o.inlier ? 1.f : 0.f;
          valid_sum = o.valid ? 1.f : 0.f;
          bad = !isfinite(o.loss);
          if (a.d_Kdiag != nullptr) { a.d_Kdiag[2 * (size_t)brow] = o.gK00; a.d_Kdiag[2 * (size_t)brow + 1] = o.gK11; }
          if (a.d_P != nullptr) {
#pragma unroll
            for (int r = 0; r < 3; ++r)
              *reinterpret_cast<float4*>(a.d_P + 12 * (size_t)brow + 4 * r) = make_float4(o.gc[r] * X[0], o.gc[r] * X[1], o.gc[r] * X[2], o.gc[r]);
          }
        }
        // back through the de-homogenisation to the 4 fc3 outputs; rounded to fp16 like autograd's cast
        if (a.use_homogeneous) {
          const float ih = 1.f / h;
          float gh = 0.f;
#pragma unroll
          for (int i = 0; i < 3; ++i) { g[i] = o.gX[i] * ih; gh -= o.gX[i] * sv[i] * ih * ih; }
          g[3] = h_pass ? gh * sig : 0.f;
        } else {
#pragma unroll
          for (int i = 0; i < 3; ++i) g[i] = o.gX[i];
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          g[j] = __half2float(__float2half_rn(g[j]));
          bad_g |= !isfinite(g[j]);
        }
      }
    }
    *reinterpret_cast<float4*>(&sG[tid][0]) = make_float4(g[0], g[1], g[2], g[3]);
  }
  if (a.training == 1 && warp < 2) {   // warps 0 and 1 hold the block's 40 rows (idle lanes carry zeros)
    loss_sum = warp_sum(loss_sum); inl_sum = warp_sum(inl_sum); valid_sum = warp_sum(valid_sum);
    if (lane == 0) { sRed[warp][0] = loss_sum; sRed[warp][1] = inl_sum; sRed[warp][2] = valid_sum; }
  }
  if (!a.training) return;
  __syncthreads();

  // ---- phase C: dX8 = g W3 (fp16 result), masked by the ReLU of x8 -> DZ[L-1]; fc3 weight-gradient partial ----
  float acc[4][16];
  if (a.fc3_part != nullptr) {
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int k = 0; k < 16; ++k) acc[j][k] = 0.f;
  }
#pragma unroll
  for (int i = 0; i < kTailRW; ++i) {
    const int row = r0 + kTailRW * warp + i;
    if (row >= a.rows) continue;
    const float4 gv = *reinterpret_cast<const float4*>(&sG[kTailRW * warp + i][0]);
    const float g[4] = {gv.x, gv.y, gv.z, gv.w};
    const __half2* xh = reinterpret_cast<const __half2*>(xr[i]);
    uint4 outv[2];
    __half2* oh = reinterpret_cast<__half2*>(outv);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float2 xf = __half22float2(xh[k]);
      float d0 = 0.f, d1 = 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 wf = __half22float2(w[j][k]);
        d0 = fmaf(g[j], wf.x, d0);
        d1 = fmaf(g[j], wf.y, d1);
        if (a.fc3_part != nullptr) {
          acc[j][2 * k] = fmaf(g[j], xf.x, acc[j][2 * k]);
          acc[j][2 * k + 1] = fmaf(g[j], xf.y, acc[j][2 * k + 1]);
        }
      }
      __half2 hv = __floats2half2_rn(d0, d1);
      const float2 hf = __half22float2(hv);
      bad_g |= !(isfinite(hf.x) && isfinite(hf.y));
      if (!(xf.x > 0.f)) hv.x = __float2half_rn(0.f);
      if (!(xf.y > 0.f)) hv.y = __float2half_rn(0.f);
      oh[k] = hv;
    }
    uint4* dzp = reinterpret_cast<uint4*>(a.dz + (size_t)row * kC + lane * 16);
    dzp[0] = outv[0];
    dzp[1] = outv[1];
  }
  if (a.fc3_part != nullptr) {
    float* mine = sAcc + (size_t)warp * 4 * kC;
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int k = 0; k < 4; ++k)
        *reinterpret_cast<float4*>(mine + j * kC + lane * 16 + 4 * k) = make_float4(acc[j][4 * k], acc[j][4 * k + 1], acc[j][4 * k + 2], acc[j][4 * k + 3]);
  }
  const int any_bad = __syncthreads_or(bad ? 1 : 0);
  const int any_bad_g = __syncthreads_or(bad_g ? 1 : 0);
  if (a.fc3_part != nullptr) {
    float* out = a.fc3_part + (size_t)blockIdx.x * (4 * kC + 4);
    for (int idx = tid; idx < 4 * kC; idx += kTailThreads) {
      float t = 0.f;
#pragma unroll
      for (int wv = 0; wv < kTailThreads / 32; ++wv) t += sAcc[(size_t)wv * 4 * kC + idx];
      out[idx] = t;
    }
    if (tid < 4) {
      float t = 0.f;
      for (int r = 0; r < kTailRows; ++r) t += sG[r][tid];
      out[4 * kC + tid] = t;
    }
  }
  // per-block partials, then the last block to finish writes the totals (no pre-zeroing, deterministic order)
  if (tid == 0) {
    float* p = a.blk_part + 8 * (size_t)blockIdx.x;
    p[0] = a.training == 1 ? sRed[0][0] + sRed[1][0] : 0.f; p[1] = a.training == 1 ? sRed[0][1] + sRed[1][1] : 0.f;
    p[2] = a.training == 1 ? sRed[0][2] + sRed[1][2] : 0.f;
    p[3] = any_bad ? 1.f : 0.f; p[4] = any_bad_g ? 1.f : 0.f;
    __threadfence();
    const unsigned int done = atomicAdd(a.blk_count, 1u);
    sLast = (done == gridDim.x - 1);
  }
  __syncthreads();
  if (sLast) {
    __threadfence();
    float accs[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
    for (int b = tid; b < (int)gridDim.x; b += kTailThreads) {
      const volatile float* p = a.blk_part + 8 * (size_t)b;
#pragma unroll
      for (int k = 0; k < 5; ++k) accs[k] += p[k];
    }
    __shared__ float sTot[5][kTailThreads / 32];
#pragma unroll
    for (int k = 0; k < 5; ++k) {
      const float wsum = warp_sum(accs[k]);
      if (lane == 0) sTot[k][warp] = wsum;
    }
    __syncthreads();
    if (tid == 0) {
      float t[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
      for (int k = 0; k < 5; ++k)
        for (int wv = 0; wv < kTailThreads / 32; ++wv) t[k] += sTot[k][wv];
      if (a.stats != nullptr) {
        // stats[3] latches: a non-finite loss of any iteration stays visible until the host clears it (the reference
        // checks the loss every iteration, ace_trainer.py:615-617; here the host reads it only when it logs)
        const float was = a.stats[3];
        a.stats[0] = t[0]; a.stats[1] = t[1]; a.stats[2] = t[2]; a.stats[3] = (t[3] > 0.f || was > 0.f) ? 1.f : 0.f;
      }
      if (a.nonfinite != nullptr) *a.nonfinite = t[4] > 0.f ? 1 : 0;
      *a.blk_count = 0u;  // ready for the next launch
    }
  }
}

__global__ void fc3_reduce_kernel(const float* __restrict__ part, int nblk, int C3, float* __restrict__ gW3,
                                  float* __restrict__ gb3, int* __restrict__ nonfinite) {
  pdl_wait();
  pdl_launch_dependents();
  // 8 threads per output element (strided over the slab partials), 3 shuffles to combine
  const int gt = blockIdx.x * blockDim.x + threadIdx.x;
  const int idx = gt >> 3, sub = gt & 7;
  const int total = 4 * kC + 4;
  float s = 0.f;
  if (idx < total)
    for (int b = sub; b < nblk; b += 8) s += part[(size_t)b * total + idx];
  s += __shfl_xor_sync(0xffffffffu, s, 1);
  s += __shfl_xor_sync(0xffffffffu, s, 2);
  s += __shfl_xor_sync(0xffffffffu, s, 4);
  bool bad = false;
  if (idx < total && sub == 0) {
    if (idx < 4 * kC) {
      if (idx < C3 * kC) { gW3[idx] = s; bad = fp16_grad_overflow(s); }
    } else if (idx - 4 * kC < C3) {
      gb3[idx - 4 * kC] = s;
      bad = fp16_grad_overflow(s);
    }
  }
  if (__syncthreads_or(bad ? 1 : 0) && threadIdx.x == 0 && nonfinite != nullptr) atomicOr(nonfinite, 1);
}

// ----------------------------------------------------------------------------------------------
// GradScaler inf check + AdamW + GradScaler.update, all on the device (no host sync)
//   scaler_state: [0] scale S, [1] growth tracker, [2] optimizer step count t
// ----------------------------------------------------------------------------------------------
__global__ void grad_check_kernel(const float* __restrict__ g, size_t n, int* __restrict__ found_inf) {
  pdl_wait();
  pdl_launch_dependents();
  bool bad = false;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    bad |= fp16_grad_overflow(g[i]);
  if (__syncthreads_or(bad ? 1 : 0) && threadIdx.x == 0) atomicOr(found_inf, 1);
}

__global__ void adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                             float* __restrict__ v, size_t n, const float* __restrict__ hyper,
                             float* __restrict__ scaler_state, const int* __restrict__ found_inf,
                             int use_scaler, __half* __restrict__ W16, __half* __restrict__ W3h, int L, int C3) {
  pdl_wait();
  pdl_launch_dependents();
  const int found = use_scaler ? *found_inf : 0;
  if (!found) {  // GradScaler.step skips optimizer.step() on inf/nan
    const AdamWStep adamw(hyper, scaler_state, use_scaler);
    const size_t n4 = n / 4;
    const size_t wsz = (size_t)kC * kC;
    const size_t tstride = (size_t)gridDim.x * blockDim.x;
    for (size_t q0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q0 < n4; q0 += 2 * tstride) {
     // two independent groups per trip: 8 loads in flight per thread
     float4 G[2], P[2], M[2], V[2];
#pragma unroll
     for (int u = 0; u < 2; ++u) {
       const size_t q = q0 + u * tstride;
       if (q < n4) {
         G[u] = reinterpret_cast<const float4*>(g)[q]; P[u] = reinterpret_cast<float4*>(p)[q];
         M[u] = reinterpret_cast<float4*>(m)[q]; V[u] = reinterpret_cast<float4*>(v)[q];
       }
     }
#pragma unroll
     for (int u = 0; u < 2; ++u) {
      const size_t q = q0 + u * tstride;
      if (q >= n4) continue;
      const float4 g4 = G[u];
      float4 p4 = P[u], m4 = M[u], v4 = V[u];
      adamw.update(g4.x, p4.x, m4.x, v4.x);
      adamw.update(g4.y, p4.y, m4.y, v4.y);
      adamw.update(g4.z, p4.z, m4.z, v4.z);
      adamw.update(g4.w, p4.w, m4.w, v4.w);
      reinterpret_cast<float4*>(p)[q] = p4;
      reinterpret_cast<float4*>(m)[q] = m4;
      reinterpret_cast<float4*>(v)[q] = v4;
      if (W16 != nullptr) {  // refresh the fp16 shadow the next forward reads (layer strides are multiples of 4)
        const size_t i = 4 * q, l = i / kLayerStride, r = i % kLayerStride;
        __half2 lo = __floats2half2_rn(p4.x, p4.y), hi = __floats2half2_rn(p4.z, p4.w);
        uint2 pk = make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
        if (l < (size_t)L) {
          if (r < wsz) *reinterpret_cast<uint2*>(W16 + l * wsz + r) = pk;
        } else if (r + 3 < (size_t)C3 * kC) {
          *reinterpret_cast<uint2*>(W3h + r) = pk;
        } else {
          const float pv[4] = {p4.x, p4.y, p4.z, p4.w};
          for (int k = 0; k < 4; ++k)
            if (r + k < (size_t)C3 * kC) W3h[r + k] = __float2half_rn(pv[k]);
        }
      }
     }
    }
    for (size_t i = 4 * n4 + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
      float pi = p[i], mi = m[i], vi = v[i];
      adamw.update(g[i], pi, mi, vi);
      p[i] = pi; m[i] = mi; v[i] = vi;
      if (W16 != nullptr) {
        const size_t l = i / kLayerStride, r = i % kLayerStride;
        if (l >= (size_t)L && r < (size_t)C3 * kC) W3h[r] = __float2half_rn(pi);
      }
    }
  }
  // the last block to finish applies GradScaler.update() (scale / growth tracker / step count); the completion
  // counter lives in scaler_state[3] (bit pattern, starts at 0) and resets itself
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    unsigned int* cnt = reinterpret_cast<unsigned int*>(scaler_state + 3);
    if (atomicAdd(cnt, 1u) == gridDim.x - 1) {
      scaler_update(scaler_state, found, use_scaler);
      *cnt = 0u;
    }
  }
}

// ----------------------------------------------------------------------------------------------
// plan
// ----------------------------------------------------------------------------------------------
static int head_prepare(acez_head_plan* h, int rows, int training) {
  if (h->prepared_rows == rows && h->prepared_training >= training) return ACEZ_OK;
  const int L = h->L;
  h->fwd.assign(L, GemmLaunch{});
  for (int l = 0; l < L; ++l) {
    GemmProblem p{};
    p.A = h->ACT + (size_t)l * h->act_stride;
    p.B = h->W16 + (size_t)l * kC * kC;
    p.a_mn = 0; p.b_mn = 0;
    p.M = rows; p.N = kC; p.K = kC; p.batch = 1;
    p.lda = kC; p.ldb = kC;
    p.bn = 0;
    p.epi = EPI_FWD;
    int rc = gemm_prepare(&h->fwd[l], p);
    if (rc) return rc;
    GemmArgs& a = h->fwd[l].args;
    a.bias = h->params + (size_t)l * kLayerStride + (size_t)kC * kC;
    a.relu = 1;
    a.ldo = kC;
    const bool res_end = (l % 3 == 2) && (l < 3 * h->nres);
    if (res_end) {
      const int k = l / 3;
      // x -> XTRA[k] (ReLU mask for the backward), res = ACT[l-2] + x -> ACT[l+1]   (ace_network.py:126,133)
      a.out = (h->XTRA != nullptr) ? h->XTRA + (size_t)k * h->act_stride : nullptr;  // nullptr: x is not kept
      a.resid = h->ACT + (size_t)(l - 2) * h->act_stride;
      a.out2 = h->ACT + (size_t)(l + 1) * h->act_stride;
    } else {
      a.out = h->ACT + (size_t)(l + 1) * h->act_stride;
    }
    rc = gemm_finalize(&h->fwd[l]);
    if (rc) return rc;
  }
  if (training) {
    h->dgrad.assign(L, GemmLaunch{});
    for (int l = L - 1; l >= 1; --l) {
      // gradient w.r.t. ACT[l] = DZ[l] * W_l, then through the ReLU of the layer that produced ACT[l]
      GemmProblem p{};
      p.A = h->DZ + (size_t)l * h->act_stride;
      p.B = h->W16 + (size_t)l * kC * kC;  // [out, in] row-major: contraction over rows -> MN-major B
      p.a_mn = 0; p.b_mn = 1;
      p.M = rows; p.N = kC; p.K = kC; p.batch = 1;
      p.lda = kC; p.ldb = kC;
      p.bn = 0;
      p.epi = EPI_DGRAD;
      int rc = gemm_prepare(&h->dgrad[l], p);
      if (rc) return rc;
      GemmArgs& a = h->dgrad[l].args;
      a.ldo = kC;
      a.out = h->DZ + (size_t)(l - 1) * h->act_stride;
      a.nonfinite = nullptr;  // patched per call
      const bool is_res = (l % 3 == 0) && (l <= 3 * h->nres);
      if (is_res) {
        const int k = l / 3;  // ACT[l] = res_k = res_{k-1} + x_{l-1}
        a.mask = h->XTRA + (size_t)(k - 1) * h->act_stride;
        a.addend = (k < h->nres) ? h->GRES : nullptr;   // skip gradient from res_{k+1}
        a.out2 = (k >= 2) ? h->GRES : nullptr;          // res_{k-1} needs it (res_0 = features has no grad)
      } else {
        a.mask = h->ACT + (size_t)l * h->act_stride;
      }
      rc = gemm_finalize(&h->dgrad[l]);
      if (rc) return rc;
    }
    // all weight gradients in one launch: grid.z = layer, dZ and X MN-major, plain fp32 stores. Contraction rows beyond `rows`
    // must read as zero: the operand maps carry the true row count so that TMA zero-fills
    const uint64_t dims[3] = {(uint64_t)kC, (uint64_t)rows, (uint64_t)L};
    const uint64_t strides[2] = {(uint64_t)kC * 2, (uint64_t)h->act_stride * 2};
    const uint32_t box[3] = {64, 64, 1};
    if (h->use_chain) {
      // 256 x 256 tiles of CTA pairs with an on-chip split-K 2: a cluster of four = two pairs per tile, 128 CTAs; the tensor pipe
      // runs at 87 % per CTA instead of the 50 % of 128-column tiles (round-2 cycle counters) and the second pair's accumulator
      // travels through distributed shared memory. Measured (round 2, warm graph replays): 171.0 us per iteration against 180.6 us
      // with 256 x 128 tiles and no split; the launch alone takes ~35 us against 44.7 us for the cta_group::1 kernel below
      Gemm2Launch& W = h->wgrad2;
      W = Gemm2Launch{};
      int rc = make_tensor_map(&W.tmA, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, h->DZ, dims, strides, box, nullptr,
                               CU_TENSOR_MAP_SWIZZLE_128B);
      if (rc) return rc;
      rc = make_tensor_map(&W.tmB, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, h->ACT, dims, strides, box, nullptr,
                           CU_TENSOR_MAP_SWIZZLE_128B);
      if (rc) return rc;
      W.batch = L;
      Gemm2Args& g = W.args;
      g.M = kC; g.N = kC; g.k_blocks = (rows + 63) / 64;
      g.tiles_n = kC / kGemm2BN;
      g.out32 = h->grads; g.out32_zstride = (long long)kLayerStride; g.ldo32 = kC;
      g.bias_grad = h->grads + (size_t)kC * kC; g.bias_grad_zstride = (long long)kLayerStride;
      g.bias_part = h->WBIAS;
      g.bias_count = h->BLKCOUNT + 8;   // [L][2] arrival counters behind the tail's; zeroed once with it (launch_tail)
      g.split_k = g.k_blocks >= 2 ? 2 : 1;
      g.a_lbo = 8192; g.a_sbo = 1024; g.a_kstep = 2048;
      g.b_lbo = 8192; g.b_sbo = 1024; g.b_kstep = 2048;
    } else {
      // measured (round 1, warm graph replays): 128 x 128 tiles / 128 CTAs: 220 us per iteration, 128 x 256 / 64 CTAs: 231 us
      GemmProblem p{};
      p.A = h->DZ; p.B = h->ACT;
      p.a_mn = 1; p.b_mn = 1;
      p.M = kC; p.N = kC; p.K = (rows + 63) / 64 * 64; p.batch = L;
      p.a_zstride = (long long)h->act_stride; p.b_zstride = (long long)h->act_stride;
      p.lda = kC; p.ldb = kC;
      p.bn = 128;
      p.epi = EPI_WGRAD;
      int rc = gemm_prepare(&h->wgrad, p);
      if (rc) return rc;
      rc = make_tensor_map(&h->wgrad.tmA, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, h->DZ, dims, strides, box, nullptr,
                           CU_TENSOR_MAP_SWIZZLE_128B);
      if (rc) return rc;
      rc = make_tensor_map(&h->wgrad.tmB, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, h->ACT, dims, strides, box, nullptr,
                           CU_TENSOR_MAP_SWIZZLE_128B);
      if (rc) return rc;
      GemmArgs& a = h->wgrad.args;
      a.out32 = h->grads;
      a.out32_zstride = (long long)kLayerStride;
      a.ldo32 = kC;
      a.bias_grad = h->grads + (size_t)kC * kC;
      a.bias_grad_zstride = (long long)kLayerStride;
      rc = gemm_finalize(&h->wgrad);
      if (rc) return rc;
    }
  }
  if (h->use_chain) {
    // ---- fused forward chain: step l = hidden layer l ----
    int rc = chain_prepare(&h->chain_fwd, CHAIN_FWD, h->ACT, h->W16, L, h->ACT, (long long)h->act_stride, L + 1, rows);
    if (rc) return rc;
    ChainArgs& f = h->chain_fwd.args;
    f.n_steps = L;
    f.flags |= kChainFlagResInit;
    const size_t mask_stride = (size_t)h->cfg.max_rows * 64;
    for (int l = 0; l < L; ++l) {
      ChainStep st{};
      st.w_layer = l;
      st.relu = 1;
      st.bias = h->params + (size_t)l * kLayerStride + (size_t)kC * kC;
      st.out_slot = (h->XTRA != nullptr || l == L - 1) ? l + 1 : -1;  // inference plans keep the tiles on chip
      st.res_add = ((l % 3 == 2) && (l < 3 * h->nres)) ? 1 : 0;        // res_{k+1} = res_k + x (ace_network.py:126,133)
      st.mask_out = (h->MASKB != nullptr) ? h->MASKB + (size_t)(l + 1) * mask_stride : nullptr;
      f.step[l] = st;
    }
    if (training) {
      // ---- fused dgrad chain: step s handles layer l = L-1-s (gradient w.r.t. ACT[l], through the ReLU below) ----
      rc = chain_prepare(&h->chain_bwd, CHAIN_DGRAD, h->DZ + (size_t)(L - 1) * h->act_stride, h->W16, L, h->DZ,
                         (long long)h->act_stride, L, rows);
      if (rc) return rc;
      ChainArgs& b = h->chain_bwd.args;
      b.n_steps = L - 1;
      for (int l = L - 1; l >= 1; --l) {
        ChainStep st{};
        st.w_layer = l;
        st.out_slot = l - 1;
        st.mask_in = h->MASKB + (size_t)l * mask_stride;  // (x > 0) of the layer that produced ACT[l]
        const bool is_res = (l % 3 == 0) && (l <= 3 * h->nres);
        if (is_res) {
          const int k = l / 3;              // ACT[l] = res_k = res_{k-1} + x_{l-1}
          st.res_add = (k < h->nres) ? 1 : 0;   // + skip gradient from res_{k+1}
          st.res_save = (k >= 2) ? 1 : 0;       // res_{k-1} needs it (res_0 = features has no gradient)
        }
        b.step[L - 1 - l] = st;
      }
    }
  }
  h->prepared_rows = rows;
  h->prepared_training = training;
  return ACEZ_OK;
}

static void fill_tail_common(const acez_head_plan* h, int rows, TailArgs& t) {
  t.rows = rows;
  t.C3 = h->C3;
  t.use_homogeneous = h->cfg.use_homogeneous;
  for (int i = 0; i < 3; ++i) t.mean[i] = h->cfg.mean[i];
  t.h_beta = h->cfg.h_beta;
  t.max_inv_scale = h->cfg.max_inv_scale;
  t.min_inv_scale = h->cfg.min_inv_scale;
  t.x = h->ACT + (size_t)h->L * h->act_stride;
  t.W3h = h->W3h;
  t.b3 = h->params + (size_t)h->L * kLayerStride + (size_t)h->C3 * kC;
}

static int tail_grid(int rows) { return (rows + kTailRows - 1) / kTailRows; }

// tail (+ fc3 gradient) launch sequence shared by the training entries
static int launch_tail(acez_head_plan* h, TailArgs& t, int rows, cudaStream_t s, int* nonfinite, bool with_fc3_grad,
                       bool pdl) {
  if (!h->counters_zeroed) {  // once per plan: the completion counter is self-resetting afterwards
    ACEZ_CUDA(cudaMemsetAsync(h->BLKCOUNT, 0, 4096, s));   // tail counter [0], wgrad bias counters [8..), split-K sync [64..)
    h->counters_zeroed = true;
    pdl = false;  // predecessor is a memset
  }
  ACEZ_REQUIRE(tail_grid(rows) <= 4096, "head tail: %d rows exceed the per-block partial buffer (131072 rows)", rows);
  t.blk_part = h->BLKPART;
  t.blk_count = h->BLKCOUNT;
  t.fc3_part = with_fc3_grad ? h->FC3PART : nullptr;
  int rc = set_max_dynamic_smem<head_tail_kernel>(kTailAccBytes);
  if (rc) return rc;
  rc = launch_kernel(head_tail_kernel, dim3(tail_grid(rows)), dim3(kTailThreads), with_fc3_grad ? (size_t)kTailAccBytes : 0, s, pdl, t);
  if (rc) return rc;
  if (with_fc3_grad) {
    const int nblk = tail_grid(rows);
    float* gW3 = h->grads + (size_t)h->L * kLayerStride;
    const int total = 4 * kC + 4;
    rc = launch_kernel(fc3_reduce_kernel, dim3((total * 8 + 255) / 256), dim3(256), 0, s, true, (const float*)h->FC3PART, nblk, h->C3, gW3,
                       gW3 + (size_t)h->C3 * kC, nonfinite);
    if (rc) return rc;
  }
  return ACEZ_OK;
}

// dgrad pass + weight gradients
static int launch_backward_gemms(acez_head_plan* h, cudaStream_t s, int* nonfinite) {
  if (h->use_chain) {
    h->chain_bwd.args.nonfinite = nonfinite;
    int rc = chain_launch(h->chain_bwd, s, /*pdl=*/true);  // predecessor: fc3_reduce_kernel
    if (rc) return rc;
    h->wgrad2.args.nonfinite = nonfinite;  // fp16-overflow / inf check of the weight gradients in the epilogue
    return gemm2_launch(h->wgrad2, s, /*pdl=*/true);
  }
  for (int l = h->L - 1; l >= 1; --l) {
    h->dgrad[l].args.nonfinite = nonfinite;
    int rc = gemm_launch(h->dgrad[l], s);
    if (rc) return rc;
  }
  h->wgrad.args.nonfinite = nonfinite;
  return gemm_launch(h->wgrad, s);
}

}  // namespace acez

// ----------------------------------------------------------------------------------------------
// C ABI
// ----------------------------------------------------------------------------------------------
using namespace acez;

extern "C" size_t acez_head_param_count(const acez_head_config* cfg) {
  if (!cfg || cfg->num_res_blocks < 1) return 0;
  const int L = 3 * cfg->num_res_blocks + 2;
  const int C3 = cfg->use_homogeneous ? 4 : 3;
  return head_param_count(L, C3);
}

extern "C" size_t acez_head_workspace_bytes(const acez_head_config* cfg) {
  if (!cfg || cfg->num_res_blocks < 1 || cfg->max_rows < 1) return 0;
  return head_layout(*cfg).total + 1024;
}

extern "C" int acez_head_plan_create(const acez_head_config* cfg, float* params, float* grads, void* workspace,
                                     size_t workspace_bytes, acez_head_plan** out) {
  ACEZ_REQUIRE(cfg && params && workspace && out, "head_plan_create: null argument");
  ACEZ_REQUIRE(cfg->num_res_blocks >= 1 && cfg->num_res_blocks <= 16, "head_plan_create: num_res_blocks out of range");
  ACEZ_REQUIRE(cfg->max_rows >= 1, "head_plan_create: max_rows must be positive");
  ACEZ_REQUIRE(!cfg->training || grads != nullptr, "head_plan_create: training plan needs a gradient buffer");
  ACEZ_REQUIRE(workspace_bytes >= acez_head_workspace_bytes(cfg), "head_plan_create: workspace too small (%zu < %zu)",
               workspace_bytes, acez_head_workspace_bytes(cfg));
  {
    // The chain / GEMM kernels run with the maximum shared-memory carve-out (227 KB per SM). A kernel that prefers another
    // L1 / shared split makes the SMs re-partition between launches; the small kernels of the iteration stream their data and
    // gain nothing from L1, so they ask for the same carve-out (ACEZ_SMEM_CARVEOUT=0 leaves the driver's default).
    static bool done = false;
    const char* e = getenv("ACEZ_SMEM_CARVEOUT");
    if (!done && (e == nullptr || atoi(e) != 0)) {
      const int pct = cudaSharedmemCarveoutMaxShared;
      cudaFuncSetAttribute(gather_rows_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
      cudaFuncSetAttribute(gather_rows_multi_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
      cudaFuncSetAttribute(head_tail_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
      cudaFuncSetAttribute(fc3_reduce_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
      cudaFuncSetAttribute(grad_check_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
      cudaFuncSetAttribute(adamw_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);
      cudaGetLastError();   // a hint: failures are not errors
      done = true;
    }
  }
  acez_head_plan* h = new acez_head_plan();
  h->cfg = *cfg;
  h->nres = cfg->num_res_blocks;
  h->L = 3 * h->nres + 2;
  h->C3 = cfg->use_homogeneous ? 4 : 3;
  h->n_params = acez_head_param_count(cfg);
  h->params = params;
  h->grads = grads;
  uint8_t* base = reinterpret_cast<uint8_t*>(align_up(reinterpret_cast<uintptr_t>(workspace), 1024));
  const HeadLayout lo = head_layout(*cfg);
  h->W16 = reinterpret_cast<__half*>(base + lo.w16);
  h->W3h = reinterpret_cast<__half*>(base + lo.w3h);
  h->ACT = reinterpret_cast<__half*>(base + lo.act);
  h->XTRA = cfg->training ? reinterpret_cast<__half*>(base + lo.xtra) : nullptr;
  h->DZ = cfg->training ? reinterpret_cast<__half*>(base + lo.dz) : nullptr;
  h->GRES = cfg->training ? reinterpret_cast<__half*>(base + lo.gres) : nullptr;
  h->MASKB = cfg->training ? base + lo.maskb : nullptr;
  h->G3 = cfg->training ? reinterpret_cast<float*>(base + lo.g3) : nullptr;
  h->FC3PART = cfg->training ? reinterpret_cast<float*>(base + lo.fc3part) : nullptr;
  h->WBIAS = cfg->training ? reinterpret_cast<float*>(base + lo.wbias) : nullptr;
  h->BLKPART = reinterpret_cast<float*>(base + lo.blkpart);
  h->BLKCOUNT = reinterpret_cast<unsigned int*>(base + lo.blkpart + 4096 * 8 * sizeof(float));
  h->counters_zeroed = false;
  {
    // Default: all hidden layers of the forward / dgrad pass in one cluster kernel each (head_chain4.cu); measured on
    // B200 (round 1, b = 5120): 0.212 ms per training iteration against 0.232 ms with one GEMM launch per layer.
    // ACEZ_HEAD_CHAIN=0 selects the per-layer tcgen05 GEMM path (also used when the head is deeper than the chain holds).
    const char* e = getenv("ACEZ_HEAD_CHAIN");
    h->use_chain = ((e == nullptr || atoi(e) != 0) && h->L <= kChainMaxSteps) ? 1 : 0;
  }
  h->act_stride = (size_t)cfg->max_rows * kC;
  h->prepared_rows = -1;
  h->prepared_training = 0;
  *out = h;
  return ACEZ_OK;
}

extern "C" void acez_head_plan_destroy(acez_head_plan* plan) {
  delete plan;
}

extern "C" int acez_head_sync_weights(acez_head_plan* h, acez_stream_t stream) {
  ACEZ_REQUIRE(h != nullptr, "head_sync_weights: null plan");
  int rc = acez_device_check();
  if (rc) return rc;
  cast_weights_kernel<<<4 * sm_count(), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(h->params, h->W16, h->W3h,
                                                                                          h->L, h->C3);
  ACEZ_CUDA(cudaGetLastError());
  return ACEZ_OK;
}

extern "C" void* acez_head_input_ptr(acez_head_plan* h) { return h ? h->ACT : nullptr; }

extern "C" void* acez_head_w16_ptr(acez_head_plan* h, int which) {
  if (h == nullptr) return nullptr;
  return which == 0 ? static_cast<void*>(h->W16) : static_cast<void*>(h->W3h);
}

extern "C" int acez_head_plan_fused_chain(const acez_head_plan* h) { return (h != nullptr && h->use_chain) ? 1 : 0; }

extern "C" int acez_debug_chain_clocks(long long* host_out, size_t max_slots, int* n_ctas) {
  return chain_debug_read(host_out, max_slots, n_ctas);
}

static int head_run_forward(acez_head_plan* h, const void* features, int rows, int training, cudaStream_t s) {
  ACEZ_REQUIRE(rows >= 1 && rows <= h->cfg.max_rows, "head: rows=%d outside [1, %d]", rows, h->cfg.max_rows);
  int rc = head_prepare(h, rows, training);
  if (rc) return rc;
  if (features != nullptr && features != h->ACT)
    ACEZ_CUDA(cudaMemcpyAsync(h->ACT, features, (size_t)rows * kC * 2, cudaMemcpyDeviceToDevice, s));
  if (h->use_chain) return chain_launch(h->chain_fwd, s);
  for (int l = 0; l < h->L; ++l) {
    rc = gemm_launch(h->fwd[l], s, /*pdl=*/l > 0);  // the first kernel of the call follows a copy / foreign work
    if (rc) return rc;
  }
  return ACEZ_OK;
}

extern "C" int acez_head_forward(acez_head_plan* h, const void* features, int rows, float* sc_out,
                                 acez_stream_t stream) {
  ACEZ_REQUIRE(h != nullptr, "head_forward: null plan");
  int rc = acez_device_check();
  if (rc) return rc;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  rc = head_run_forward(h, features, rows, 0, s);
  if (rc) return rc;
  if (sc_out == nullptr) return ACEZ_OK;  // GEMM chain only (profiling)
  TailArgs t{};
  fill_tail_common(h, rows, t);
  t.training = 0;
  t.sc_out = sc_out;
  return launch_tail(h, t, rows, s, nullptr, false, true);
}

extern "C" int acez_head_train_fwd_bwd(acez_head_plan* h, int rows, const acez_loss_params* lp,
                                       const acez_train_batch* b, float* stats, int* nonfinite,
                                       acez_stream_t stream) {
  ACEZ_REQUIRE(h && lp && b && stats && nonfinite, "head_train_fwd_bwd: null argument");
  ACEZ_REQUIRE(h->cfg.training && h->grads, "head_train_fwd_bwd: plan was not created for training");
  ACEZ_REQUIRE(b->target_px_b2 && b->K_b33 && b->Kinv_b33, "head_train_fwd_bwd: missing batch tensors");
  ACEZ_REQUIRE(b->P_b34 || (b->aug_inv_b34 && b->pose_inv_b44), "head_train_fwd_bwd: need P_b34 or aug_inv+pose_inv");
  ACEZ_REQUIRE(!lp->use_depth || b->target_crds_b3, "head_train_fwd_bwd: use_depth needs target_crds_b3");
  ACEZ_REQUIRE(lp->divisor > 0, "head_train_fwd_bwd: divisor must be positive");
  int rc = acez_device_check();
  if (rc) return rc;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  rc = head_run_forward(h, b->features, rows, 1, s);
  if (rc) return rc;
  const int L = h->L;
  TailArgs t{};
  fill_tail_common(h, rows, t);
  t.training = 1;
  t.sc_out = b->sc_out_b3;
  t.lp = *lp;
  t.tpx = b->target_px_b2; t.Pin = b->P_b34; t.A = b->aug_inv_b34; t.T = b->pose_inv_b44;
  t.K = b->K_b33; t.Kinv = b->Kinv_b33; t.G = b->target_crds_b3;
  t.d_P = b->d_P_b34; t.d_Kdiag = b->d_Kdiag_b2;
  t.grad_scale_dev = b->grad_scale_dev;
  t.loss_weight_dev = b->loss_weight_dev;
  t.dz = h->DZ + (size_t)(L - 1) * h->act_stride;
  t.stats = stats;
  t.nonfinite = nonfinite;
  rc = launch_tail(h, t, rows, s, nonfinite, true, true);
  if (rc) return rc;
  return launch_backward_gemms(h, s, nonfinite);
}

extern "C" int acez_head_backward(acez_head_plan* h, int rows, const float* d_sc_b3, int* nonfinite,
                                  acez_stream_t stream) {
  ACEZ_REQUIRE(h && d_sc_b3 && nonfinite, "head_backward: null argument");
  ACEZ_REQUIRE(h->cfg.training && h->grads, "head_backward: plan was not created for training");
  ACEZ_REQUIRE(h->prepared_rows == rows && h->prepared_training >= 1,
               "head_backward: call acez_head_forward_train with the same row count first");
  int rc = acez_device_check();
  if (rc) return rc;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const int L = h->L;
  TailArgs t{};
  fill_tail_common(h, rows, t);
  t.training = 2;
  t.lp.grad_scale = 1.f; t.lp.divisor = 1;
  t.d_sc_in = d_sc_b3;
  t.dz = h->DZ + (size_t)(L - 1) * h->act_stride;
  t.stats = nullptr;
  t.nonfinite = nonfinite;
  rc = launch_tail(h, t, rows, s, nonfinite, true, false);  // first kernel of this call
  if (rc) return rc;
  return launch_backward_gemms(h, s, nonfinite);
}

extern "C" int acez_head_forward_train(acez_head_plan* h, const void* features, int rows, float* sc_out,
                                       acez_stream_t stream) {
  ACEZ_REQUIRE(h != nullptr && sc_out != nullptr, "head_forward_train: null argument");
  ACEZ_REQUIRE(h->cfg.training && h->grads, "head_forward_train: plan was not created for training");
  int rc = acez_device_check();
  if (rc) return rc;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  rc = head_run_forward(h, features, rows, 1, s);
  if (rc) return rc;
  TailArgs t{};
  fill_tail_common(h, rows, t);
  t.training = 0;
  t.sc_out = sc_out;
  return launch_tail(h, t, rows, s, nullptr, false, true);
}

extern "C" int acez_gather_rows(const void* src, const int64_t* idx, int rows, int row_bytes, void* dst,
                                acez_stream_t stream) {
  ACEZ_REQUIRE(src && idx && dst && rows >= 0 && row_bytes > 0 && (row_bytes & 1) == 0, "gather_rows: bad arguments");
  int rc = acez_device_check();
  if (rc) return rc;
  if (rows == 0) return ACEZ_OK;
  const int threads = 256;
  const int grid = (rows * 32 + threads - 1) / threads;
  gather_rows_kernel<<<grid, threads, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const uint8_t*>(src), idx, rows, row_bytes, reinterpret_cast<uint8_t*>(dst));
  ACEZ_CUDA(cudaGetLastError());
  return ACEZ_OK;
}

static int gather_multi_impl(const void* const* srcs, void* const* dsts, const int* row_bytes, int n_arrays, const int64_t* idx,
                             int rows, const acez::GatherSched& sch, acez_stream_t stream);

extern "C" int acez_gather_rows_multi(const void* const* srcs, void* const* dsts, const int* row_bytes, int n_arrays,
                                      const int64_t* idx, int rows, acez_stream_t stream) {
  acez::GatherSched sch{};
  return gather_multi_impl(srcs, dsts, row_bytes, n_arrays, idx, rows, sch, stream);
}

extern "C" int acez_gather_rows_multi_sched(const void* const* srcs, void* const* dsts, const int* row_bytes, int n_arrays,
                                            const int64_t* idx, int rows, const acez_schedule_params* p, float* state_dev,
                                            const float* inlier_count_dev, float* hyper_dev, acez_stream_t stream) {
  ACEZ_REQUIRE(p && state_dev && inlier_count_dev && hyper_dev, "gather_rows_multi_sched: null schedule argument");
  ACEZ_REQUIRE(p->kind >= ACEZ_SCHED_CONSTANT && p->kind <= ACEZ_SCHED_1CYCLEPOLY && p->batch_global > 0 && rows >= 1,
               "gather_rows_multi_sched: bad schedule parameters");
  acez::GatherSched sch{};
  sch.enabled = 1; sch.p = *p; sch.state = state_dev; sch.inlier_count = inlier_count_dev; sch.hyper = hyper_dev;
  return gather_multi_impl(srcs, dsts, row_bytes, n_arrays, idx, rows, sch, stream);
}

static int gather_multi_impl(const void* const* srcs, void* const* dsts, const int* row_bytes, int n_arrays, const int64_t* idx,
                             int rows, const acez::GatherSched& sch, acez_stream_t stream) {
  ACEZ_REQUIRE(srcs && dsts && row_bytes && idx && n_arrays >= 1 && n_arrays <= 8 && rows >= 0,
               "gather_rows_multi: bad arguments");
  MultiGather g{};
  for (int a = 0; a < n_arrays; ++a) {
    ACEZ_REQUIRE(srcs[a] && dsts[a] && row_bytes[a] > 0 && (row_bytes[a] & 1) == 0, "gather_rows_multi: bad array %d", a);
    g.src[a] = reinterpret_cast<const uint8_t*>(srcs[a]);
    g.dst[a] = reinterpret_cast<uint8_t*>(dsts[a]);
    g.row_bytes[a] = row_bytes[a];
  }
  int rc = acez_device_check();
  if (rc) return rc;
  if (rows == 0) return ACEZ_OK;
  const int threads = 256;
  dim3 grid((rows * 32 + threads - 1) / threads + (sch.enabled ? 1 : 0));
  return launch_kernel(gather_rows_multi_kernel, grid, dim3(threads), 0, reinterpret_cast<cudaStream_t>(stream), false, g, idx, rows,
                       n_arrays, sch);
}

extern "C" int acez_adamw_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, size_t n,
                               const float* hyper_dev, float* scaler_state_dev, int* found_inf_dev, int use_scaler,
                               acez_head_plan* plan, acez_stream_t stream) {
  ACEZ_REQUIRE(params && grads && exp_avg && exp_avg_sq && hyper_dev && scaler_state_dev && found_inf_dev,
               "adamw_step: null argument");
  ACEZ_REQUIRE(plan == nullptr || (plan->params == params && plan->n_params == n),
               "adamw_step: plan does not own this parameter buffer");
  int rc = acez_device_check();
  if (rc) return rc;
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const int grid = 8 * sm_count();
  if (use_scaler == 1 || use_scaler == 3) {  // 2 = the caller's flag already covers every gradient (acez_head_train_fwd_bwd does)
    // 3 (data parallel through NCCL): one more element behind the gradient is checked too - the slot in which the ranks'
    // local GradScaler flags travelled through the all-reduce (+inf when any rank overflowed)
    rc = launch_kernel(grad_check_kernel, dim3(grid), dim3(256), 0, s, false, grads, n + (use_scaler == 3 ? 1 : 0), found_inf_dev);
    if (rc) return rc;
  }
  rc = launch_kernel(adamw_kernel, dim3(grid), dim3(256), 0, s, false, params, grads, exp_avg, exp_avg_sq, n, hyper_dev,
                     scaler_state_dev, (const int*)found_inf_dev, use_scaler ? 1 : 0, plan ? plan->W16 : (__half*)nullptr,
                     plan ? plan->W3h : (__half*)nullptr, plan ? plan->L : 0, plan ? plan->C3 : 0);
  if (rc) return rc;
  return ACEZ_OK;
}
