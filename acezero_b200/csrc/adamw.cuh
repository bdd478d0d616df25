// The optimiser semantics both AdamW kernels implement: the single-GPU adamw_kernel (head.cu) and the data-parallel kernels
// (adamw_dp.cu). torch.optim.AdamW defaults and torch.cuda.amp.GradScaler defaults (reference: ace_schedule.py:15,30,63,70,106-113).
#pragma once
#include "common.cuh"

namespace acez {

// Flat parameter layout of the head (params / grads / exp_avg / exp_avg_sq): per hidden layer W[kC][kC] then b[kC]; fc3 W[C3][kC]
// and b[C3] last.
static constexpr int kC = 512;  // head width, hard-coded in the reference (ace_network.py:76)
static constexpr size_t kLayerStride = (size_t)kC * kC + kC;
__host__ __device__ constexpr size_t head_param_count(int L, int C3) {
  return (size_t)L * kLayerStride + (size_t)C3 * kC + (size_t)C3;
}

#ifdef __CUDACC__
// torch.cuda.amp.GradScaler.update(): backoff 0.5 on inf, growth x2 every 2000 clean steps
//   st: [0] scale S, [1] growth tracker, [2] optimizer step count t
__device__ __forceinline__ void scaler_update(float* st, int found, int use_scaler) {
  if (use_scaler && found) {
    st[0] *= 0.5f;
    st[1] = 0.f;
  } else {
    st[2] += 1.f;
    if (use_scaler) {
      st[1] += 1.f;
      if (st[1] >= 2000.f) { st[0] *= 2.f; st[1] = 0.f; }
    }
  }
}

// One optimizer.step() of AdamW: the step's constants, read once from hyper = [lr, beta1, beta2, eps, weight_decay] and the
// GradScaler state, and the element update. With use_scaler the gradient is the fp16 weight gradient of the autocast conv, scaled.
struct AdamWStep {
  float lr, b1, b2, eps, wd, inv_scale, step_size, bc2_sqrt;
  bool use_scaler;
  __device__ __forceinline__ AdamWStep(const float* hyper, const float* scaler_state, bool use_scaler_) : use_scaler(use_scaler_) {
    lr = hyper[0]; b1 = hyper[1]; b2 = hyper[2]; eps = hyper[3]; wd = hyper[4];
    inv_scale = use_scaler ? 1.f / scaler_state[0] : 1.f;
    const float t = scaler_state[2] + 1.f;  // this step's index (torch: state['step'] += 1 before use)
    const float bc1 = 1.f - powf(b1, t), bc2 = 1.f - powf(b2, t);
    step_size = lr / bc1;
    bc2_sqrt = sqrtf(bc2);
  }
  __device__ __forceinline__ void update(float gi, float& pi, float& mi, float& vi) const {
    if (use_scaler) gi = __half2float(__float2half_rn(gi));  // fp16 weight gradient of the autocast conv
    gi *= inv_scale;                                          // GradScaler.unscale_
    pi *= (1.f - lr * wd);                                    // decoupled weight decay (torch adamw)
    mi = mi + (1.f - b1) * (gi - mi);                         // exp_avg.lerp_(grad, 1 - beta1)
    vi = b2 * vi + (1.f - b2) * gi * gi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    pi -= step_size * (mi / denom);
  }
};
#endif  // __CUDACC__

}  // namespace acez
