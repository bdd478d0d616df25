/*
 * acez.h — C ABI of libacez.so, the sm_100a (B200) implementation of the ACE Zero hot path.
 *
 * This is the drop-in boundary for the one native operator of the reference (the `dsacstar` pybind11 module,
 * reference dsacstar/dsacstar.cpp:898-899, built by dsacstar/setup.py:28-38) and for the PyTorch library calls the
 * reference's training / registration loops make on the hot path (ace_trainer.py:499-640, ace_network.py:41-149,
 * ace_loss.py:39-90, ace_schedule.py:106-126, register_mapping.py:201-251).
 *
 * Conventions
 *   - plain C: raw device pointers + sizes, `int` status return (0 = ok), no exceptions, no torch types;
 *   - every buffer is caller-owned (the Python side allocates them with torch); the library never allocates
 *     device memory. Opaque `*_plan` handles hold only host-side metadata (TMA tensor maps, pointers);
 *   - `acez_stream_t` is a `cudaStream_t`; all work is enqueued on it, nothing synchronises the host
 *     unless documented;
 *   - there is no CPU path: without an sm_100a device every compute entry returns ACEZ_ERR_NO_DEVICE /
 *     ACEZ_ERR_UNSUPPORTED and sets acez_last_error().
 */
#ifndef ACEZ_H_
#define ACEZ_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ACEZ_VERSION 100

#define ACEZ_OK 0
#define ACEZ_ERR_INVALID 1
#define ACEZ_ERR_CUDA 2
#define ACEZ_ERR_UNSUPPORTED 3
#define ACEZ_ERR_NO_DEVICE 4

typedef void* acez_stream_t; /* cudaStream_t */

int acez_version(void);
/* Thread-local message of the last failing call. */
const char* acez_last_error(void);
/* 0 iff a compute-capability-10.x device is current. */
int acez_device_check(void);

/* ------------------------------------------------------------------------------------------------------------
 * Generic fp16 tensor-core GEMM (tcgen05 + TMA). Building block of the head and encoder; exported for the parity
 * tests. D[z] = A[z] * B[z]; K-major operand = [rows, K] row-major, MN-major operand = [K, rows] row-major.
 * Replaces: cuDNN/cuBLAS dispatches of nn.Conv2d(…,1,1,0) in reference ace_network.py:122-137.
 * ---------------------------------------------------------------------------------------------------------- */
#define ACEZ_EPI_FWD 0   /* out = fp16(act(acc + fp16(bias))), out2 = fp16(resid + out) */
#define ACEZ_EPI_DGRAD 1 /* v = fp16(acc) (+ addend); out2 = v; out = mask > 0 ? v : 0 */
#define ACEZ_EPI_F32 2   /* out32 = acc; optional bias_grad[m] = sum_k A[m,k] */

typedef struct acez_gemm_desc {
  const void* A; /* fp16 */
  const void* B; /* fp16 */
  int a_mn_major, b_mn_major;
  int M, N, K, batch;
  long long a_zstride, b_zstride; /* elements, used when batch > 1 */
  int lda, ldb;                   /* elements */
  int bn;                         /* 0 = auto, else 64 / 128 / 256 */
  int epilogue;
  const float* bias;  /* [N] fp32, nullable */
  const void* resid;  /* fp16 [M,ldo], nullable */
  const void* mask;   /* fp16 [M,ldo], ACEZ_EPI_DGRAD */
  const void* addend; /* fp16 [M,ldo], nullable */
  void* out;          /* fp16 [M,ldo] */
  void* out2;         /* fp16 [M,ldo], nullable */
  int ldo;
  int relu;
  int* nonfinite; /* nullable */
  float* out32;   /* ACEZ_EPI_F32: [batch][M,ldo32] */
  long long out32_zstride;
  int ldo32;
  float* bias_grad; /* nullable, [batch][M] */
  long long bias_grad_zstride;
  /* 0 = library defaults; non-zero values override the UMMA shared-memory descriptor constants (test probing) */
  unsigned a_lbo, a_sbo, a_kstep, b_lbo, b_sbo, b_kstep;
  void* dbg_clock; /* nullable: int64 [CTAs][8] clock64() stamps (entry, prologue, dependency, first tile, MMA issued,
                      accumulator ready, epilogue done, exit) */
} acez_gemm_desc;

int acez_gemm_f16(const acez_gemm_desc* d, acez_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Fused reprojection loss + backward.
 * Replaces: reference ace_trainer.py:521-613 (pose compose, projection, masks, loss) + ace_loss.py:39-90 and
 * the autograd backward of that graph (ace_schedule.py:106-107), ~40 ATen kernels and 3 host syncs.
 * ---------------------------------------------------------------------------------------------------------- */
#define ACEZ_LOSS_TANH 0    /* w * tanh(r / w); dyntanh = same with the host-computed per-iteration weight */
#define ACEZ_LOSS_L1 1      /* r where r <= soft_clamp */
#define ACEZ_LOSS_L1_SQRT 2 /* + sqrt(soft_clamp * r) above */
#define ACEZ_LOSS_L1_LOG 3  /* + log(1 + soft_clamp * r) above */

typedef struct acez_loss_params {
  int loss_type;
  float loss_weight;   /* tanh weight (ace_loss.py:53-69) or soft_clamp for the l1 family (ace_loss.py:72-90) */
  float depth_min;     /* 0.1  train_ace.py depth_min  */
  float depth_max;     /* 1000 */
  float hard_clamp;    /* 1000 repro_loss_hard_clamp */
  float inlier_px;     /* 10   learning_rate_cooldown_trigger_px_threshold */
  float depth_target;  /* 10 */
  int use_depth;       /* GT scene coordinates present (ace_trainer.py:567-574, 602-609) */
  float grad_scale;    /* GradScaler scale S (ace_schedule.py:107); gradients are emitted multiplied by it */
  int divisor;         /* batch size b of `loss /= batch_size` (ace_trainer.py:613); the GLOBAL b under data parallel */
} acez_loss_params;

/* stats[0] += sum of per-row losses / divisor (unscaled), stats[1] += #valid rows with r < inlier_px,
 * stats[2] += #valid rows, stats[3] = 1 if any non-finite loss term was seen. Caller zeroes stats. */
int acez_repro_loss_fwd_bwd(const acez_loss_params* p, int rows,
                            const float* sc_b3,          /* predicted scene coordinates */
                            const float* target_px_b2,   /* pixel targets */
                            const float* P_b34,          /* nullable: composed world->cam; else aug_inv * pose_inv */
                            const float* aug_inv_b34, const float* pose_inv_b44,
                            const float* K_b33, const float* Kinv_b33,
                            const float* target_crds_b3, /* nullable unless use_depth */
                            float* d_sc_b3,              /* out */
                            float* d_P_b34,              /* out, nullable */
                            float* d_Kdiag_b2,           /* out, nullable: dL/dK00, dL/dK11 per row */
                            float* stats, acez_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * ACE head (ace_network.Head, reference ace_network.py:62-149): plan-based forward / training step.
 * Flat fp32 parameter layout (shared by params, grads, exp_avg, exp_avg_sq):
 *   for each hidden layer l in [res3_conv1, res3_conv2, res3_conv3, {i}c0, {i}c1, {i}c2 ..., fc1, fc2]:
 *        W_l [512,512] row-major (out, in), then b_l [512]
 *   then fc3: W [C3,512], b [C3]   (C3 = 4 homogeneous, else 3)
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct acez_head_plan acez_head_plan;

typedef struct acez_head_config {
  int num_res_blocks;   /* 1 + num_head_blocks */
  int use_homogeneous;
  int max_rows;         /* capacity of one forward / training batch (multiple of 128 recommended) */
  int training;         /* allocate backward buffers */
  float mean[3];
  float h_beta;         /* ace_network.py:113 */
  float max_inv_scale;  /* ace_network.py:112 */
  float min_inv_scale;  /* ace_network.py:114 */
} acez_head_config;

size_t acez_head_param_count(const acez_head_config* cfg);
size_t acez_head_workspace_bytes(const acez_head_config* cfg);

int acez_head_plan_create(const acez_head_config* cfg, float* params, float* grads /* nullable unless training */,
                          void* workspace, size_t workspace_bytes, acez_head_plan** out);
void acez_head_plan_destroy(acez_head_plan* plan);

/* fp32 master weights -> fp16 shadow copies the GEMMs read (autocast's weight cast). */
int acez_head_sync_weights(acez_head_plan* plan, acez_stream_t stream);
/* Device pointer of the plan's input activation buffer [max_rows,512] fp16 (gather target). */
void* acez_head_input_ptr(acez_head_plan* plan);
/* 1 if the plan runs all hidden layers of a pass (ace_network.py:120-136 and its autograd transpose) as ONE fused
 * cluster kernel per pass (csrc/head_chain4.cu), 0 if it launches one tcgen05 GEMM per layer (csrc/gemm.cu). Both are
 * sm_100a paths with identical semantics; the fused chain is the default, ACEZ_HEAD_CHAIN=0 at plan creation selects
 * the per-layer path. */
int acez_head_plan_fused_chain(const acez_head_plan* plan);
/* Profiling probe of the fused chain kernel (ACEZ_CHAIN_DBG=1): clock64 stamps of the most recent launch,
 * [n_ctas][8 + 8 * 20] (layout in csrc/head_chain4.cu), copied to host memory. */
int acez_debug_chain_clocks(long long* host_out, size_t max_slots, int* n_ctas);

/* Forward only (registration; ace_network.py:120-149 under autocast): features -> scene coordinates.
 * features: fp16 [rows,512] (nullable = already in the plan's input buffer); sc_out: fp32 [rows,3]
 * (nullable: run only the hidden-layer GEMM chain, used by bench.py to time that kernel alone). */
int acez_head_forward(acez_head_plan* plan, const void* features, int rows, float* sc_out, acez_stream_t stream);

/* The same forward on a training plan, keeping what the backward needs (activations, ReLU masks), followed by the
 * backward from an externally supplied dL/d(scene coordinates) [rows,3] (unscaled or pre-scaled by the caller) into
 * `grads` — the pair torch.autograd needs when the reference's own training loop drives `Regressor`
 * (ace_trainer.py:516-518 forward, :627 backward). */
int acez_head_forward_train(acez_head_plan* plan, const void* features, int rows, float* sc_out, acez_stream_t stream);
int acez_head_backward(acez_head_plan* plan, int rows, const float* d_sc_b3, int* nonfinite, acez_stream_t stream);

typedef struct acez_train_batch {
  const void* features;        /* fp16 [rows,512]; nullable = already in the plan's input buffer */
  const float* target_px_b2;
  const float* P_b34;          /* nullable (see acez_repro_loss_fwd_bwd) */
  const float* aug_inv_b34;
  const float* pose_inv_b44;
  const float* K_b33;
  const float* Kinv_b33;
  const float* target_crds_b3; /* nullable */
  float* d_P_b34;              /* nullable out */
  float* d_Kdiag_b2;           /* nullable out */
  float* sc_out_b3;            /* nullable out: predicted scene coordinates (fp32) */
  const float* grad_scale_dev; /* nullable: device scalar overriding loss_params.grad_scale (= scaler_state[0]) */
  const float* loss_weight_dev; /* nullable: device scalar overriding loss_params.loss_weight (dyntanh schedule) */
} acez_train_batch;

/* One head forward + reprojection loss + full backward into `grads` (overwritten, scaled by grad_scale).
 * stats: [4] floats as in acez_repro_loss_fwd_bwd; [0..2] are overwritten by the call, [3] (non-finite loss seen) is a LATCH:
 * it is OR-ed with its previous value, so a caller that reads the statistics only every n-th iteration cannot miss a NaN
 * (the reference checks every iteration, ace_trainer.py:615-617); the caller zeroes it. nonfinite (int, device) is overwritten: 1 if
 * any activation gradient or (fp16-rounded) weight gradient is inf/nan — the complete GradScaler found_inf of this
 * backward pass. Replaces ace_trainer.py:516-627. */
int acez_head_train_fwd_bwd(acez_head_plan* plan, int rows, const acez_loss_params* lp, const acez_train_batch* batch,
                            float* stats, int* nonfinite, acez_stream_t stream);

/* Gather rows of the patch buffer into a batch (reference ace_trainer.py:485-494, 8 index kernels):
 * dst[i, :] = src[idx[i], :], row_bytes multiple of 2. */
int acez_gather_rows(const void* src, const int64_t* idx, int rows, int row_bytes, void* dst, acez_stream_t stream);
/* The same for up to 8 arrays sharing one index vector, in ONE launch (all arrays of the patch buffer). */
int acez_gather_rows_multi(const void* const* srcs, void* const* dsts, const int* row_bytes, int n_arrays,
                           const int64_t* idx, int rows, acez_stream_t stream);

/* Patch-buffer fill for one image (reference ace_trainer.py:381-436, ~12 small kernels): writes the rows
 * [row0, row0 + n_samples) of all 8 buffer arrays for the cells `sample_idx` (the int64 output of torch.multinomial,
 * ace_trainer.py:423-426 — the caller keeps torch's generator and call order, so indices stay bit-exact).
 * feat_rows: fp16 NHWC rows [cells,512] of the image; mats46: device floats aug_inv(12) | pose_inv(16) | K(9) | Kinv(9);
 * target_crds_3hw: planar [3,cells] or NULL (zeros, dataset.py returns zeros without depth). */
int acez_buffer_fill(const void* feat_rows, const int64_t* sample_idx, int n_samples, int map_w, int cells, int subsample,
                     const float* mats46, const float* target_crds_3hw, int pose_idx, long long row0, void* d_features,
                     float* d_target_px, float* d_aug_inv, float* d_pose_inv, float* d_K, float* d_Kinv,
                     float* d_target_crds, int16_t* d_pose_idx, acez_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * GradScaler unscale + inf check + AdamW + GradScaler.update, entirely on the device (CUDA-graph capturable, no
 * host sync). Replaces ace_schedule.py:109-113 (scaler.step(optimizer); scaler.update()) with torch.optim.AdamW
 * defaults semantics (ace_schedule.py:15,30,63) and torch.cuda.amp.GradScaler defaults (init 65536, x2 / 2000 clean
 * steps, x0.5 on inf, step skipped on inf).
 *   hyper_dev        float[5]: lr, beta1, beta2, eps, weight_decay (host-written per iteration)
 *   scaler_state_dev float[4]: [0] scale S, [1] growth tracker, [2] optimizer step count t (bias correction), [3] -
 *   found_inf_dev    int: OR-ed with the grads' non-finite / fp16-overflow check; must already hold the activation-
 *                    gradient overflow flag of acez_head_train_fwd_bwd (same pointer). Not cleared by this call.
 *   use_scaler       0: plain AdamW (use_half False): no check, no unscale, no skip; 1: check grads here;
 *                    3: like 1, and grads[n] (one spare element behind the gradient: the data-parallel flag slot) is checked too
 *                    2: found_inf_dev is already complete (acez_head_train_fwd_bwd folds the check of every gradient
 *                    into the kernels that produce it), no extra pass over the gradients
 *   scaler_state_dev[3] is a completion counter used by the kernel (keep it 0).
 * Also refreshes the head's fp16 weight shadow when `plan` is non-null.
 * ---------------------------------------------------------------------------------------------------------- */
int acez_adamw_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, size_t n,
                    const float* hyper_dev, float* scaler_state_dev, int* found_inf_dev, int use_scaler,
                    acez_head_plan* plan, acez_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Training schedule on the device. Replaces the per-iteration host logic of ScheduleACE (ace_schedule.py:22-126:
 * OneCycleLR / LinearLR warm-up + cool-down, the cool-down trigger on the last 100 batch-inlier fractions, the mutable
 * max_iterations) and the loss-weight schedule of ReproLoss (ace_loss.py:53-69). acez_schedule_step enqueues a one-thread
 * kernel that (1) books the PREVIOUS iteration's inlier count (*inlier_count_dev / batch_global) into the ring, (2) runs
 * check_and_set_cooldown for the current iteration, (3) writes hyper_dev[0] = lr (0 once iteration >= max_iterations: later
 * optimiser steps leave the weights unchanged) and hyper_dev[5] = loss weight, (4) advances the iteration counter.
 * It is meant to be the first node of the iteration's CUDA graph: no host -> device traffic and no read-back per iteration.
 * state_dev: ACEZ_SCHED_STATE_FLOATS floats, initialised by acez_schedule_init; layout (integers stored as floats):
 *   [0] iteration  [1] scheduler steps  [2] in cool-down  [3] cool-down start (steps)  [4] max_iterations
 *   [5] ring fill  [6] ring position    [7] done          [8] lr of the last step      [9] loss weight   [16..116) ring
 * ---------------------------------------------------------------------------------------------------------- */
#define ACEZ_SCHED_RING 100
#define ACEZ_SCHED_STATE_FLOATS 128
enum { ACEZ_SCHED_CONSTANT = 0, ACEZ_SCHED_CIRCLE = 1, ACEZ_SCHED_1CYCLEPOLY = 2 };
typedef struct acez_schedule_params {
  int kind;                 /* ACEZ_SCHED_* : --learning_rate_schedule constant | circle | 1cyclepoly */
  int iterations;           /* --iterations (OneCycleLR total_steps; initial max_iterations; loss-weight horizon) */
  float lr_min, lr_max;     /* --learning_rate_min / --learning_rate_max */
  int warmup_iterations;    /* 1cyclepoly */
  float warmup_lr;
  int cooldown_iterations;
  float cooldown_trigger;   /* --learning_rate_cooldown_trigger_percent_threshold */
  int batch_global;         /* divisor of the inlier count (ace_trainer.py:586) */
  int loss_dyntanh;         /* 1: dyntanh weight schedule, 0: constant soft clamp */
  int loss_schedule_circle; /* --repro_loss_schedule circle (1) | linear (0) */
  float soft_clamp, soft_clamp_min;
} acez_schedule_params;

int acez_schedule_init(const acez_schedule_params* p, float* state_dev, acez_stream_t stream);
int acez_schedule_step(const acez_schedule_params* p, float* state_dev, const float* inlier_count_dev, float* hyper_dev,
                       acez_stream_t stream);
/* acez_gather_rows_multi with the schedule step riding in its first block: the first kernel of a training iteration then does
 * both (one launch less in the iteration's graph). */
int acez_gather_rows_multi_sched(const void* const* srcs, void* const* dsts, const int* row_bytes, int n_arrays,
                                 const int64_t* idx, int rows, const acez_schedule_params* p, float* state_dev,
                                 const float* inlier_count_dev, float* hyper_dev, acez_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Data-parallel optimiser step over NVLink peer memory (G ranks of one box, one process per GPU): replaces "NCCL all-reduce
 * of the 8.4 MB gradient + replicated AdamW" with kernels that read / write the other GPUs' buffers directly, synchronised
 * across the GPUs inside the kernels (no caller barriers: the step is captured in ONE CUDA graph with the rest of the iteration).
 * Rank r owns the parameter shard [r S, (r+1) S), S = acez_adamw_dp_shard(n, G). One step:
 *   - reduce: sum over ranks of the gradient of this rank's shard; the 4 spare floats behind the gradient (+inf marker of the
 *     local GradScaler flag, loss / inlier / valid sums) are summed too; the fp16-range / inf verdict of the summed shard goes to
 *     EVERY rank
 *   - apply: found = any rank's verdict | non-finite marker; unless found: unscale + AdamW on the shard (params / moments of
 *     this rank), the new weights rounded to fp16 and stored into EVERY rank's fp16 shadows (peer_w16 / peer_w3h), the biases
 *     (the kernels read them in fp32) into every rank's parameters (peer_params); GradScaler.update(); the summed spare slots are
 *     copied to local_extras[0..4) (= this rank's grads + n); *found_inf_dev = found
 * peer_* are HOST arrays of G device pointers (peer mappings of the same buffer on every rank).
 * fp32 master weights and moments are valid on their owner rank only.
 * ---------------------------------------------------------------------------------------------------------- */
size_t acez_adamw_dp_shard(size_t n, int world);
/* Every rank's flag array (peer_flags) holds 64 ints, zero before the first step: [0, G) the verdict flags, [16, 16+G) /
 * [24, 24+G) / [32, 32+G) epoch signals "gradient complete" / "shard reduced" / "weights written", stored by the peers over
 * NVLink (st.release.sys) and polled locally (ld.acquire.sys). sync_state_dev: unsigned[4] of this rank, zero before the first
 * step ([0] = completed steps, the rest block counters). When the call's last kernel completes, every rank's shard of the new
 * weights has landed in this rank's buffers. A peer that never signals traps after ~20 s instead of hanging.
 * local_stats_dev (nullable): float[3] loss / inlier / valid sums of this rank's backward pass; when given, the step packs the
 * four spare slots behind this rank's gradient itself (+inf marker from *found_inf_dev, then the three sums) and runs as ONE
 * kernel when the shard fits a co-resident grid's registers; otherwise (or without it) as a reduce kernel and an apply kernel.
 * multicast (nullable): host array of 4 NVSwitch multicast addresses of the gradient, fp16 hidden weights, fp16 fc3 weights and
 * parameter buffers (NVLink SHARP): the gradient is then summed inside the switch (multimem.ld_reduce) and the new weights reach
 * all ranks with one store each (multimem.st); the summation order inside the switch is the hardware's, every element is still
 * reduced exactly once (by its owner), so all ranks hold identical weights. */
int acez_adamw_dp_step(const void* const* peer_grads, void* const* peer_flags, void* const* peer_w16, void* const* peer_w3h,
                       void* const* peer_params, int world, int rank, size_t n, float* reduced_shard, float* params,
                       float* exp_avg, float* exp_avg_sq, const float* hyper_dev, float* scaler_state_dev, int* found_inf_dev,
                       float* local_extras, unsigned int* sync_state_dev, const float* local_stats_dev,
                       const void* const* multicast, int L, int C3, acez_stream_t stream);
/* Device pointers of the plan's fp16 weight shadows (which = 0: hidden layers [L][512][512], 1: fc3 [4][512]); they live in the
 * caller's workspace, so a peer's copy sits at the same offset of the peer's workspace. */
void* acez_head_w16_ptr(acez_head_plan* plan, int which);

/* ------------------------------------------------------------------------------------------------------------
 * DSAC* pose solver. Replaces the reference's native operator:
 *   dsacstar.forward_rgb(sceneCoordinates[1,3,H,W] f32 CPU, outPose[4,4] f32 CPU, ransacHypotheses, inlierThreshold,
 *                        focalLength, ppointX, ppointY, inlierAlpha, maxReproj, subSampling, randomSeed,
 *                        max_hypotheses_tries) -> int inliers          (dsacstar/dsacstar.cpp:66-186, 898-899)
 * batched over n images, device pointers, per-image intrinsics.
 *   - sampling RNG: counter-based, keyed (seed, image key, hypothesis, try, draw) with image key = image_index[i] when
 *     that array is given (any order: a shuffled micro-batch of register_mapping.py:147 is ONE launch), else
 *     image_index_base + i — results do not depend on batch composition or GPU count (the reference's
 *     mt19937-per-OMP-thread stream is not reproducible across machines; SURVEY.md §9.3);
 *   - injected_idx (nullable) int32 [n, hyps, 4, 2] = (x, y) cell of each of the 4 correspondences: overrides the
 *     RNG and disables retries (parity tests feed the oracle's minimal sets);
 *   - out_pose: camera->world 4x4 row-major float (dsacstar.cpp:177-182); out_inliers: size of the inlier set the
 *     final pose was fitted to (dsacstar.cpp:185).
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct acez_dsac_params {
  int hyps;
  float inlier_threshold; /* px */
  float inlier_alpha;
  float max_reproj;
  int subsample;          /* 8 */
  uint64_t seed;
  int max_tries;
  int max_refine_steps;   /* reference MAX_REF_STEPS = 100 (dsacstar.cpp:47) */
  int image_index_base;   /* added to the in-batch image index for RNG keying (used when image_index is NULL) */
  const int* image_index; /* nullable, device int32 [n]: RNG key of image i (dataset index), overrides image_index_base + i */
} acez_dsac_params;

typedef struct acez_dsac_debug { /* all nullable; device pointers */
  float* hyp_poses;  /* [n, hyps, 6]: rvec(3), tvec(3) scene->camera of every hypothesis */
  float* hyp_scores; /* [n, hyps] soft inlier scores */
  int* best;         /* [n] index of the winning hypothesis */
  int* hyp_tries;    /* [n, hyps] number of tries used */
  int* refine_rounds;/* [n] accepted refinement rounds */
} acez_dsac_debug;

size_t acez_dsac_workspace_bytes(int n, int h, int w, int hyps);

int acez_dsac_forward_rgb_batch(const float* sc /* [n,3,h,w] device */, int n, int h, int w,
                                const float* focal /* [n] */, const float* ppx /* [n] */, const float* ppy /* [n] */,
                                const acez_dsac_params* p, const int* injected_idx, float* out_pose /* [n,4,4] */,
                                int* out_inliers /* [n] */, const acez_dsac_debug* dbg, void* workspace,
                                size_t workspace_bytes, acez_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * ACE encoder (ace_network.Encoder, reference ace_network.py:14-59): 11 convolutions, 1 -> 512 channels at 1/8
 * resolution. Weights are frozen; the plan packs them to fp16 once.
 * image: fp16 or fp32 [n,1,H,W]; features out: fp16 NHWC [n, h8, w8, 512] == the reference's `normalize_shape`
 * row order per image (ace_trainer.py:399-401).
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct acez_encoder_plan acez_encoder_plan;

size_t acez_encoder_workspace_bytes(int max_n, int max_h, int max_w);
/* weights: 22 device pointers in state_dict order (conv1.weight, conv1.bias, ..., res2_skip.weight, res2_skip.bias),
 * fp32, PyTorch OIHW layout. */
int acez_encoder_plan_create(const float* const* weights, int max_n, int max_h, int max_w, void* workspace,
                             size_t workspace_bytes, acez_stream_t stream, acez_encoder_plan** out);
void acez_encoder_plan_destroy(acez_encoder_plan* plan);
int acez_encoder_out_hw(int H, int W, int* h8, int* w8);
int acez_encoder_forward(acez_encoder_plan* plan, const void* image, int image_is_fp16, int n, int H, int W,
                         void* features_out, acez_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Point-cloud export metrics (reference ace_vis_util.py:431-592): per cell of n predicted scene-coordinate maps
 * [n,3,h,w] (device), under the mapping poses pose_inv [n,3,4] (world -> camera) and intrinsics K [n,3,3]:
 *   err   [n,h*w]  L1 reprojection error against the cell's pixel subsample * (x + 0.5, y + 0.5)  (:489-503)
 *   grad  [n,h*w]  max(|X(x,y) - X(x-1,y)|, |X(x,y) - X(x,y-1)|), reflect-padded first column / row  (:506-515)
 *   depth [n,h*w]  camera-space z                                                                   (:528)
 * ---------------------------------------------------------------------------------------------------------- */
int acez_pointcloud_metrics(const float* sc, int n, int h, int w, const float* pose_inv_n34, const float* K_n33,
                            int subsample, float* err, float* grad, float* depth, acez_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Augmented training images (reference dataset.py `_get_single_item` without depth, csrc/imageprep.cu): PIL bilinear
 * resize of the decoded uint8 image, convert("L"), ColorJitter(brightness, contrast) through PIL ImageEnhance,
 * ToTensor + Normalize(0.4, 0.25), scikit-image order-1 rotate (mode 'reflect', clip) and the fp16 store, bit for bit.
 * All images of one call share the output size. Coefficient tables (acezero_b200/imageprep.py `resize_coeffs`) are
 * int32 [out, 2 + k]: first source index, tap count, k Q22 weights.
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct {
  const uint8_t* src;        /* device [h_in, w_in, channels], channels 1 (gray) or 3 (RGB) */
  int h_in, w_in, channels;
  const int32_t* coef_x;     /* device [w_out, 2 + kx]; NULL exactly when w_in == w_out (PIL skips that pass) */
  const int32_t* coef_y;     /* device [h_out, 2 + ky]; NULL exactly when h_in == h_out */
  int kx, ky;
  int contrast_first;        /* ColorJitter's randperm puts contrast before brightness */
  float brightness, contrast;/* jitter factors; 1, 1 = no jitter */
  int rotate;                /* 0: no rotation (augmentation off) */
  double affine[6];          /* inverse map (col, row)_out -> (col, row)_in: the first two rows of skimage's matrix */
} acez_image_prep_desc;

size_t acez_image_prep_workspace_bytes(const acez_image_prep_desc* descs, int n, int h_out, int w_out);
/* out: fp16 [n, 1, h_out, w_out] device. descs: host array. */
int acez_image_prep(const acez_image_prep_desc* descs, int n, int h_out, int w_out, void* workspace,
                    size_t workspace_bytes, void* out_f16, acez_stream_t stream);
/* cells [h8*w8] float 0/1: the reference's rotated mask of an h x w image (affine6 as above, host memory) after
 * TF.resize(mask, [h8, w8], NEAREST). */
int acez_image_mask_cells(const double* affine6, int h, int w, int h8, int w8, float* cells, acez_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* ACEZ_H_ */
