// Data-parallel optimiser step over NVLink peer memory (acez_adamw_dp_step): the gradient all-reduce, GradScaler check, AdamW and
// the broadcast of the new fp16 weights by kernels that read / write the other GPUs' buffers directly (symmetric-memory peer
// pointers), instead of an NCCL all-reduce of the full 8.4 MB gradient followed by a replicated AdamW over all 2.1 M parameters
// (reference: ace_schedule.py:106-113 on one GPU; SURVEY.md section 8e for the sharding). Rank r owns the parameter shard
// [r S, (r+1) S), S = ceil(n / G / 8) * 8, and every rank computes the sum of ITS shard exactly once, in rank order, so all GPUs
// see bit-identical weights. The ranks synchronise through epoch signals inside the kernels (below), so one call is a plain
// sequence of kernels on the caller's stream and is captured in the iteration's CUDA graph.
//
// The step is ONE kernel (adamw_dp_fused_kernel) when the shard's parameter groups fit the registers of one co-resident grid.
// Otherwise it runs as two kernels:
//   reduce  block 0 packs the 4 spare slots behind this rank's gradient (+inf marker of the local GradScaler flag, loss / inlier /
//           valid sums) and signals "gradient complete"; every block waits for every rank's signal. g_sum[i] = sum_q grads_q[i]
//           for i in the shard; fp16-range / inf check of the summed shard -> this rank's flag, stored into EVERY rank's flag
//           array (remote 4-byte stores); the spare slots are summed by every rank for itself. The last block signals "shard
//           reduced".
//   apply   waits for every rank's "shard reduced": found = any rank's shard flag | non-finite flag slot; unless found: unscale,
//           AdamW on the shard's fp32 master weights / moments (local), new weights rounded to fp16 and stored into EVERY rank's
//           fp16 shadow (the operand the forward / dgrad GEMMs read), the biases (read in fp32) into every rank's parameter
//           buffer; GradScaler.update() on every rank (same inputs, same state). The last block signals "weights written" and
//           waits for everybody's.
// Traffic per GPU and iteration: (G-1)/G * 8.4 MB of gradient reads + (G-1)/G * 4.2 MB of weight writes over NVLink, AdamW
// state traffic 1/G of the single-GPU kernel. fp32 master weights are valid on their owner only (gathered when exported).
#include "adamw.cuh"

namespace acez {

static constexpr int kMaxRanks = 8;

// Cross-GPU synchronisation INSIDE the kernels: every rank's flag array (symmetric memory, int[kDpFlagInts]) also carries three
// rows of epoch signals, written by the peers with st.release.sys over NVLink and polled locally with ld.acquire.sys:
//   [kSigGrads + q]   rank q's gradient of this iteration is complete        (sent by block 0 of q's reduce kernel)
//   [kSigReduced + q] rank q has reduced its shard, its verdict flag is out  (sent by the last block of q's reduce kernel)
//   [kSigApplied + q] rank q has written its shard of the new weights        (sent by the last block of q's apply kernel, which
//                     then waits for everybody's: when the apply kernel completes, every rank's weights have landed here)
// The epoch (iterations completed) lives in device memory and advances once per step, so a captured CUDA graph replays it.
static constexpr int kSigGrads = 16, kSigReduced = 24, kSigApplied = 32;
static constexpr long long kDpWatchdogCycles = 40000000000ll;   // ~20 s: a peer that never signals is a dead job, not a stall

__device__ __forceinline__ void st_release_sys(int* p, int v) {
  asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// plain system-scope store: for signals sent after ONE explicit __threadfence_system() (a st.release.sys per peer would pay one
// system-scope membar per store on the critical path) and for signals that publish no data (the verdict)
__device__ __forceinline__ void st_relaxed_sys(int* p, int v) {
  asm volatile("st.relaxed.sys.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ int ld_acquire_sys(const int* p) {
  int v;
  asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// thread q < world waits until rank q's signal of row `row` has reached epoch e
__device__ __forceinline__ void dp_wait_row(const int* my_flags, int row, int q, int e) {
  const int* p = my_flags + row + q;
  if (ld_acquire_sys(p) - e >= 0) return;
  const long long t0 = clock64();
  while (ld_acquire_sys(p) - e < 0) {
    __nanosleep(40);
    if (clock64() - t0 > kDpWatchdogCycles) {
      printf("acez: data-parallel optimiser: rank %d never signalled row %d of epoch %d\n", q, row, e);
      __trap();
    }
  }
}

// The four spare slots behind each rank's flat gradient: [n] +inf if the rank's local backward overflowed (GradScaler flag), else 0;
// [n+1 .. n+3] the loss / inlier / valid sums of its local backward pass. Summed over the ranks, the first slot is non-zero or not
// finite when any rank overflowed.
__device__ __forceinline__ void pack_spare_slots(float* my_grads, size_t n, const int* local_found_inf, const float* local_stats) {
  my_grads[n] = (*local_found_inf != 0) ? __int_as_float(0x7f800000) : 0.f;
  my_grads[n + 1] = local_stats[0]; my_grads[n + 2] = local_stats[1]; my_grads[n + 3] = local_stats[2];
}
__device__ __forceinline__ bool overflow_marked(float slot) { return !isfinite(slot) || slot != 0.f; }

// NVLink SHARP (multicast objects of the NVSwitch, PTX multimem.*): one load returns the sum over all GPUs' copies of an address
// (the reduction happens in the switch: a GPU receives 1/G of the gradient instead of reading (G-1)/G of it from its peers, which a
// pull over NVLink delivered at only ~220 GB/s here), one store writes all GPUs' copies.
__device__ __forceinline__ float4 mm_ld_reduce_f32x4(const float* mc) {
  float4 r;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(mc) : "memory");
  return r;
}
__device__ __forceinline__ float mm_ld_reduce_f32(const float* mc) {
  float r;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.f32 %0, [%1];" : "=f"(r) : "l"(mc) : "memory");
  return r;
}
__device__ __forceinline__ void mm_st_b128(void* mc, uint4 v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc), "f"(__uint_as_float(v.x)),
               "f"(__uint_as_float(v.y)), "f"(__uint_as_float(v.z)), "f"(__uint_as_float(v.w)) : "memory");
}
__device__ __forceinline__ void mm_st_f32(float* mc, float v) {
  asm volatile("multimem.st.relaxed.sys.global.f32 [%0], %1;" ::"l"(mc), "f"(v) : "memory");
}

struct DpPeers {
  // multicast addresses of the same four buffers (nullptr: no NVLink SHARP, peer-to-peer loads / stores instead)
  const float* mc_grads;
  __half* mc_w16;
  __half* mc_w3h;
  float* mc_params;
  const float* grads[kMaxRanks];   // every rank's flat gradient (+4 spare floats)
  int* flags[kMaxRanks];           // every rank's flag array [world]
  __half* w16[kMaxRanks];          // every rank's fp16 hidden-layer weights [L][512][512]
  __half* w3h[kMaxRanks];          // every rank's fp16 fc3 weights [4][512]
  float* params[kMaxRanks];        // every rank's fp32 parameters: the BIASES are read in fp32 by the kernels, so they travel too
};

__global__ void __launch_bounds__(256)
adamw_dp_reduce_kernel(const DpPeers P, int world, int rank, size_t n, size_t shard, float* __restrict__ reduced,
                       float* __restrict__ my_grads /* nullable: this rank's gradient buffer (the spare slots are packed here) */,
                       const int* __restrict__ local_found_inf, const float* __restrict__ local_stats,
                       unsigned int* __restrict__ sync_state /* [0] epoch, [1] block counter */) {
  pdl_wait();
  const int epoch = (int)sync_state[0] + 1;
  // this rank's gradient is complete (stream order / the wait above): pack the spare slots behind it (the +inf marker of the
  // local GradScaler flag, the loss / inlier / valid sums of the local backward pass), tell everybody, wait for everybody's
  if (blockIdx.x == 0 && threadIdx.x == 0 && my_grads != nullptr) pack_spare_slots(my_grads, n, local_found_inf, local_stats);
  if (blockIdx.x == 0) {
    __syncthreads();
    if (threadIdx.x < world) {
      __threadfence_system();
      st_release_sys(P.flags[threadIdx.x] + kSigGrads + rank, epoch);
    }
  }
  if (threadIdx.x < world) dp_wait_row(P.flags[rank], kSigGrads, threadIdx.x, epoch);
  __syncthreads();
  const size_t lo = (size_t)rank * shard;
  const size_t hi = lo + shard < n ? lo + shard : n;
  bool bad = false;
  const size_t n4 = hi > lo ? (hi - lo) / 4 : 0;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  // two groups of four parameters per trip, the loads of ALL ranks issued before the first add: a peer read over NVLink takes
  // ~1-2 us, one dependent round trip per rank and group (round 2, first version) made the kernel latency bound
  for (size_t q0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q0 < n4; q0 += 2 * stride) {
    float4 g[2][kMaxRanks];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const size_t q = q0 + u * stride;
#pragma unroll
      for (int r = 0; r < kMaxRanks; ++r)
        if (r < world && q < n4) g[u][r] = __ldcg(reinterpret_cast<const float4*>(P.grads[r] + lo) + q);
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const size_t q = q0 + u * stride;
      if (q >= n4) continue;
      float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int r = 0; r < kMaxRanks; ++r)   // fixed order: the sum does not depend on who computes it
        if (r < world) { s.x += g[u][r].x; s.y += g[u][r].y; s.z += g[u][r].z; s.w += g[u][r].w; }
      reinterpret_cast<float4*>(reduced)[q] = s;
      // fp16_grad_overflow() of the four sums, written out: through the helper nvcc schedules this loop differently
      bad |= !isfinite(s.x) || fabsf(s.x) > 65504.f || !isfinite(s.y) || fabsf(s.y) > 65504.f;
      bad |= !isfinite(s.z) || fabsf(s.z) > 65504.f || !isfinite(s.w) || fabsf(s.w) > 65504.f;
    }
  }
  for (size_t i = lo + 4 * n4 + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += stride) {
    float s = 0.f;
    for (int r = 0; r < world; ++r) s += __ldcg(P.grads[r] + i);
    reduced[i - lo] = s;
    bad |= fp16_grad_overflow(s);
  }
  if (blockIdx.x == 0 && threadIdx.x < 4) {   // the spare slots: every rank for itself (all ranks get the same sums)
    float s = 0.f;
    for (int r = 0; r < world; ++r) s += __ldcg(P.grads[r] + n + threadIdx.x);
    reduced[shard + threadIdx.x] = s;         // kept next to the shard until the apply kernel copies them home (the peers may
  }                                           // still be reading this rank's gradient buffer)
  if (__syncthreads_or(bad ? 1 : 0) && threadIdx.x == 0) {
    for (int r = 0; r < world; ++r) *reinterpret_cast<volatile int*>(P.flags[r] + rank) = 1;   // remote stores: every rank learns this shard's verdict
  }
  if (threadIdx.x == 0) {
    __threadfence_system();   // this block's verdict stores before its arrival
    if (atomicAdd(sync_state + 1, 1u) == gridDim.x - 1) {
      sync_state[1] = 0u;
      __threadfence_system();
      for (int r = 0; r < world; ++r) st_release_sys(P.flags[r] + kSigReduced + rank, epoch);
    }
  }
}

__global__ void adamw_dp_apply_kernel(const DpPeers P, int world, int rank, size_t n, size_t shard, const float* __restrict__ reduced,
                                      float* __restrict__ p, float* __restrict__ m, float* __restrict__ v,
                                      const float* __restrict__ hyper, float* __restrict__ scaler_state, int* __restrict__ my_flags,
                                      int* __restrict__ found_inf_out, float* __restrict__ local_extras, int L, int C3,
                                      unsigned int* __restrict__ sync_state /* [0] epoch */) {
  pdl_wait();
  const int epoch = (int)sync_state[0] + 1;
  // every rank has reduced its shard: all verdict flags are final, and nobody computes with the old weights any more
  if (threadIdx.x < world) dp_wait_row(my_flags, kSigReduced, threadIdx.x, epoch);
  __syncthreads();
  int found = 0;
  for (int r = 0; r < world; ++r) found |= my_flags[r];
  const float flag_slot = reduced[shard];    // sum of the ranks' +inf markers (local backward overflow)
  if (!isfinite(flag_slot) || flag_slot != 0.f) found = 1;   // overflow_marked(), written out: nvcc compiles the helper differently here
  const size_t lo = (size_t)rank * shard;
  const size_t hi = lo + shard < n ? lo + shard : n;
  if (!found) {
    const AdamWStep adamw(hyper, scaler_state, true);
    const size_t wsz = (size_t)kC * kC;
    // groups of 8 consecutive parameters (shard bounds, layer strides and the weight / bias boundaries are multiples of 8): the
    // fp16 shadow travels to every rank as ONE 16-byte store per group and peer
    const size_t n8 = hi > lo ? (hi - lo) / 8 : 0;
    for (size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x; q < n8; q += (size_t)gridDim.x * blockDim.x) {
      const size_t i = lo + 8 * q;
      float g8[8], p8[8], m8[8], v8[8];
      *reinterpret_cast<float4*>(g8) = reinterpret_cast<const float4*>(reduced)[2 * q];
      *reinterpret_cast<float4*>(g8 + 4) = reinterpret_cast<const float4*>(reduced)[2 * q + 1];
      *reinterpret_cast<float4*>(p8) = *reinterpret_cast<const float4*>(p + i);
      *reinterpret_cast<float4*>(p8 + 4) = *reinterpret_cast<const float4*>(p + i + 4);
      *reinterpret_cast<float4*>(m8) = *reinterpret_cast<const float4*>(m + i);
      *reinterpret_cast<float4*>(m8 + 4) = *reinterpret_cast<const float4*>(m + i + 4);
      *reinterpret_cast<float4*>(v8) = *reinterpret_cast<const float4*>(v + i);
      *reinterpret_cast<float4*>(v8 + 4) = *reinterpret_cast<const float4*>(v + i + 4);
#pragma unroll
      for (int k = 0; k < 8; ++k) adamw.update(g8[k], p8[k], m8[k], v8[k]);
      *reinterpret_cast<float4*>(p + i) = *reinterpret_cast<float4*>(p8);
      *reinterpret_cast<float4*>(p + i + 4) = *reinterpret_cast<float4*>(p8 + 4);
      *reinterpret_cast<float4*>(m + i) = *reinterpret_cast<float4*>(m8);
      *reinterpret_cast<float4*>(m + i + 4) = *reinterpret_cast<float4*>(m8 + 4);
      *reinterpret_cast<float4*>(v + i) = *reinterpret_cast<float4*>(v8);
      *reinterpret_cast<float4*>(v + i + 4) = *reinterpret_cast<float4*>(v8 + 4);
      uint4 pk;
      __half2 h0 = __floats2half2_rn(p8[0], p8[1]), h1 = __floats2half2_rn(p8[2], p8[3]);
      __half2 h2 = __floats2half2_rn(p8[4], p8[5]), h3 = __floats2half2_rn(p8[6], p8[7]);
      pk.x = *reinterpret_cast<uint32_t*>(&h0); pk.y = *reinterpret_cast<uint32_t*>(&h1);
      pk.z = *reinterpret_cast<uint32_t*>(&h2); pk.w = *reinterpret_cast<uint32_t*>(&h3);
      const size_t l = i / kLayerStride, r = i % kLayerStride;
      if (l < (size_t)L) {
        if (r < wsz) {
          for (int qq = 0; qq < world; ++qq) *reinterpret_cast<uint4*>(P.w16[qq] + l * wsz + r) = pk;
        } else {   // a bias group: the fp32 values go to every rank's parameter buffer (the kernels read biases in fp32)
          for (int qq = 0; qq < world; ++qq) {
            if (qq == rank) continue;
            *reinterpret_cast<float4*>(P.params[qq] + i) = *reinterpret_cast<float4*>(p8);
            *reinterpret_cast<float4*>(P.params[qq] + i + 4) = *reinterpret_cast<float4*>(p8 + 4);
          }
        }
      } else if (r + 8 <= (size_t)C3 * kC) {
        for (int qq = 0; qq < world; ++qq) *reinterpret_cast<uint4*>(P.w3h[qq] + r) = pk;
      } else {
        for (int k = 0; k < 8; ++k) {
          if (r + k < (size_t)C3 * kC) { for (int qq = 0; qq < world; ++qq) P.w3h[qq][r + k] = __float2half_rn(p8[k]); }
          else if (i + k < n) { for (int qq = 0; qq < world; ++qq) if (qq != rank) P.params[qq][i + k] = p8[k]; }   // fc3 bias
        }
      }
    }
    for (size_t i = lo + 8 * n8 + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += (size_t)gridDim.x * blockDim.x) {
      float pi = p[i], mi = m[i], vi = v[i];
      adamw.update(reduced[i - lo], pi, mi, vi);
      p[i] = pi; m[i] = mi; v[i] = vi;
      const size_t l = i / kLayerStride, r = i % kLayerStride;
      const __half hv = __float2half_rn(pi);
      if (l < (size_t)L) {
        if (r < wsz) { for (int qq = 0; qq < world; ++qq) P.w16[qq][l * wsz + r] = hv; }
        else { for (int qq = 0; qq < world; ++qq) if (qq != rank) P.params[qq][i] = pi; }
      } else if (r < (size_t)C3 * kC) {
        for (int qq = 0; qq < world; ++qq) P.w3h[qq][r] = hv;
      } else {
        for (int qq = 0; qq < world; ++qq) if (qq != rank) P.params[qq][i] = pi;   // fc3 bias
      }
    }
  }
  // bookkeeping by one thread: summed spare slots home (statistics / schedule read them there), flags cleared for the next
  // iteration, GradScaler.update()
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    for (int k = 0; k < 4; ++k) local_extras[k] = reduced[shard + k];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence_system();   // this block's remote weight stores before its arrival
    unsigned int* cnt = reinterpret_cast<unsigned int*>(scaler_state + 3);
    if (atomicAdd(cnt, 1u) == gridDim.x - 1) {
      scaler_update(scaler_state, found, 1);
      *found_inf_out = found;
      for (int r = 0; r < world; ++r) my_flags[r] = 0;   // every block has read them (this is the last block to get here)
      *cnt = 0u;
      sync_state[0] = (unsigned int)epoch;
      __threadfence_system();
      for (int r = 0; r < world; ++r) st_release_sys(P.flags[r] + kSigApplied + rank, epoch);
      // the kernel completes only when every rank's shard of the new weights has landed in THIS rank's buffers: whatever
      // follows in stream order (the next iteration's forward) may read them
      for (int r = 0; r < world; ++r) dp_wait_row(my_flags, kSigApplied, r, epoch);
    }
  }
}


// ----------------------------------------------------------------------------------------------------------------------------
// ONE kernel for the whole data-parallel optimiser step (acez_adamw_dp_step when every parameter group of the shard fits a thread's
// registers): gradient reduction over NVLink, global GradScaler verdict, AdamW on the shard, fp16 weights pushed to every rank.
// The reduced gradient never leaves the registers, and the verdict exchange (an NVLink round trip) overlaps the loads of the master
// weights / moments and the AdamW arithmetic; only the stores wait for it.
//   1  block 0 packs the spare slots behind this rank's gradient and signals "gradient complete" to every rank; every block waits
//      for every rank's signal
//   2  each thread: all ranks' values of its parameter groups (8 consecutive parameters each) + its p / m / v -> registers; sum in
//      rank order; fp16-range check
//   3  last block to get here sends this rank's verdict (epoch * 2 + bad) to every rank
//   4  each thread computes the AdamW update in registers, then waits for every rank's verdict (and has read every rank's +inf
//      marker of the local GradScaler flags directly): found = any
//   5  unless found: p / m / v stored, fp16 weights (fp32 biases) stored into every rank's buffers
//   6  last block: GradScaler.update(), summed spare slots home, epoch, "weights written" signal to every rank, wait for everybody's
// Steps 3 -> 4 make every block wait for all blocks of all GPUs: the grid must be co-resident (sized from the occupancy query, and
// launched plainly, i.e. after the previous kernel of the stream has drained).
// ----------------------------------------------------------------------------------------------------------------------------
template <int GPT /* groups per thread */, int MAXW /* ranks held in registers */>
__global__ void __launch_bounds__(256, 2)
adamw_dp_fused_kernel(const DpPeers P, int world, int rank, size_t n, size_t shard, float* __restrict__ p, float* __restrict__ m,
                      float* __restrict__ v, const float* __restrict__ hyper, float* __restrict__ scaler_state,
                      int* __restrict__ found_inf_io /* in: flag of the local backward, out: the global verdict */,
                      float* __restrict__ my_grads, const float* __restrict__ local_stats, float* __restrict__ scratch /* [4] */,
                      unsigned int* __restrict__ sync_state /* [0] epoch, [1] block counter, [2] verdict bits, [3] block counter 2 */,
                      unsigned long long* __restrict__ stamps /* [8] %globaltimer (ns) at the phase boundaries, block 0 / the last block */,
                      int L, int C3) {
  const bool stamp0 = blockIdx.x == 0 && threadIdx.x == 0;
  auto now = [] { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; };
  if (stamp0) stamps[0] = now();
  const int epoch = (int)sync_state[0] + 1;
  int* my_flags = P.flags[rank];
  // ---- 1: gradient complete ----
  if (blockIdx.x == 0) {
    if (threadIdx.x == 0) {
      pack_spare_slots(my_grads, n, found_inf_io, local_stats);
      __threadfence_system();   // ONE system-scope fence, then plain signal stores (the gradient itself is complete by stream order)
      for (int r = 0; r < world; ++r) st_relaxed_sys(P.flags[r] + kSigGrads + rank, epoch);
    }
  }
  if (threadIdx.x < world) dp_wait_row(my_flags, kSigGrads, threadIdx.x, epoch);
  __syncthreads();
  if (stamp0) stamps[1] = now();
  // ---- 2: loads ----
  const size_t lo = (size_t)rank * shard;
  const size_t hi = lo + shard < n ? lo + shard : n;
  const size_t cnt = hi > lo ? hi - lo : 0;
  const size_t n8 = (cnt + 7) / 8;               // the last group of the last rank may be partial (n is not a multiple of 8)
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  const size_t q_first = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  float g8[GPT][8], p8[GPT][8], m8[GPT][8], v8[GPT][8];
  const bool mc = P.mc_grads != nullptr;
  const int wsum = mc ? 1 : world;   // multicast: the switch has summed already, slot 0 holds the total
  float marker = 0.f;
  if (mc) { if (threadIdx.x == 0) marker = mm_ld_reduce_f32(P.mc_grads + n); }
  else if (threadIdx.x < world) marker = __ldcg(P.grads[threadIdx.x] + n);   // +inf if that rank's local backward overflowed
  {
    float gr[GPT][MAXW][8];
#pragma unroll
    for (int k = 0; k < GPT; ++k) {
      const size_t q = q_first + k * stride;
      if (q >= n8) continue;
      const size_t i = lo + 8 * q;
      if (i + 8 <= hi) {
        if (mc) {
          *reinterpret_cast<float4*>(&gr[k][0][0]) = mm_ld_reduce_f32x4(P.mc_grads + i);
          *reinterpret_cast<float4*>(&gr[k][0][4]) = mm_ld_reduce_f32x4(P.mc_grads + i + 4);
        } else {
#pragma unroll
          for (int r = 0; r < MAXW; ++r) {
            if (r < world) {
              *reinterpret_cast<float4*>(&gr[k][r][0]) = __ldcg(reinterpret_cast<const float4*>(P.grads[r] + i));
              *reinterpret_cast<float4*>(&gr[k][r][4]) = __ldcg(reinterpret_cast<const float4*>(P.grads[r] + i) + 1);
            }
          }
        }
        *reinterpret_cast<float4*>(&p8[k][0]) = *reinterpret_cast<const float4*>(p + i);
        *reinterpret_cast<float4*>(&p8[k][4]) = *reinterpret_cast<const float4*>(p + i + 4);
        *reinterpret_cast<float4*>(&m8[k][0]) = *reinterpret_cast<const float4*>(m + i);
        *reinterpret_cast<float4*>(&m8[k][4]) = *reinterpret_cast<const float4*>(m + i + 4);
        *reinterpret_cast<float4*>(&v8[k][0]) = *reinterpret_cast<const float4*>(v + i);
        *reinterpret_cast<float4*>(&v8[k][4]) = *reinterpret_cast<const float4*>(v + i + 4);
      } else {
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const bool ok = i + e < hi;
#pragma unroll
          for (int r = 0; r < MAXW; ++r)
            if (r < wsum) gr[k][r][e] = ok ? (mc ? mm_ld_reduce_f32(P.mc_grads + i + e) : __ldcg(P.grads[r] + i + e)) : 0.f;
          p8[k][e] = ok ? p[i + e] : 0.f; m8[k][e] = ok ? m[i + e] : 0.f; v8[k][e] = ok ? v[i + e] : 0.f;
        }
      }
    }
    bool bad = false;
#pragma unroll
    for (int k = 0; k < GPT; ++k) {
      const size_t q = q_first + k * stride;
      if (q >= n8) continue;
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        float sum = 0.f;
#pragma unroll
        for (int r = 0; r < MAXW; ++r)   // fixed order: the sum does not depend on who computes it
          if (r < wsum) sum += gr[k][r][e];
        g8[k][e] = sum;
        bad |= fp16_grad_overflow(sum);
      }
    }
    if (blockIdx.x == 0 && threadIdx.x >= 32 && threadIdx.x < 36) {   // the spare slots: every rank for itself (same sums everywhere)
      float sum = 0.f;
      if (mc) sum = mm_ld_reduce_f32(P.mc_grads + n + (threadIdx.x - 32));
      else for (int r = 0; r < world; ++r) sum += __ldcg(P.grads[r] + n + (threadIdx.x - 32));
      scratch[threadIdx.x - 32] = sum;   // copied home in step 6 (the peers may still be reading this rank's gradient buffer)
    }
    // ---- 3: this rank's verdict ----
    const int bad_block = __syncthreads_or(bad ? 1 : 0);
    if (stamp0) stamps[2] = now();
    if (threadIdx.x == 0) {
      if (bad_block) atomicOr(sync_state + 2, 1u);
      __threadfence();
      if (atomicAdd(sync_state + 1, 1u) == gridDim.x - 1) {
        __threadfence();
        const int verdict = epoch * 2 + (int)(atomicExch(sync_state + 2, 0u) & 1u);
        sync_state[1] = 0u;
        for (int r = 0; r < world; ++r) st_relaxed_sys(P.flags[r] + kSigReduced + rank, verdict);   // publishes no data
      }
    }
  }
  // ---- 4: AdamW in registers, then the global verdict ----
  {
    const AdamWStep adamw(hyper, scaler_state, true);
#pragma unroll
    for (int k = 0; k < GPT; ++k)
#pragma unroll
      for (int e = 0; e < 8; ++e) adamw.update(g8[k][e], p8[k][e], m8[k][e], v8[k][e]);
  }
  int found_t = 0;
  if (mc && threadIdx.x == 0) found_t = overflow_marked(marker) ? 1 : 0;
  if (threadIdx.x < world) {
    const int* sp = my_flags + kSigReduced + threadIdx.x;
    int val = ld_acquire_sys(sp);
    if ((val >> 1) - epoch < 0) {
      const long long t0 = clock64();
      while (((val = ld_acquire_sys(sp)) >> 1) - epoch < 0) {
        __nanosleep(40);
        if (clock64() - t0 > kDpWatchdogCycles) {
          printf("acez: data-parallel optimiser: rank %d never sent its verdict of epoch %d\n", (int)threadIdx.x, epoch);
          __trap();
        }
      }
    }
    found_t |= (val & 1) | (overflow_marked(marker) ? 1 : 0);
  }
  const int found = __syncthreads_or(found_t);
  if (stamp0) stamps[3] = now();
  // ---- 5: stores ----
  if (!found) {
    const size_t wsz = (size_t)kC * kC;
#pragma unroll
    for (int k = 0; k < GPT; ++k) {
      const size_t q = q_first + k * stride;
      if (q >= n8) continue;
      const size_t i = lo + 8 * q;
      const size_t l = i / kLayerStride, r = i % kLayerStride;
      if (i + 8 <= hi) {
        *reinterpret_cast<float4*>(p + i) = *reinterpret_cast<float4*>(&p8[k][0]);
        *reinterpret_cast<float4*>(p + i + 4) = *reinterpret_cast<float4*>(&p8[k][4]);
        *reinterpret_cast<float4*>(m + i) = *reinterpret_cast<float4*>(&m8[k][0]);
        *reinterpret_cast<float4*>(m + i + 4) = *reinterpret_cast<float4*>(&m8[k][4]);
        *reinterpret_cast<float4*>(v + i) = *reinterpret_cast<float4*>(&v8[k][0]);
        *reinterpret_cast<float4*>(v + i + 4) = *reinterpret_cast<float4*>(&v8[k][4]);
      }
      if (i + 8 <= hi && (l < (size_t)L ? (r < wsz) : (r + 8 <= (size_t)C3 * kC))) {
        // a group of weights: one 16-byte fp16 store per rank (group bounds never straddle the weight / bias boundary)
        uint4 pk;
        __half2 h0 = __floats2half2_rn(p8[k][0], p8[k][1]), h1 = __floats2half2_rn(p8[k][2], p8[k][3]);
        __half2 h2 = __floats2half2_rn(p8[k][4], p8[k][5]), h3 = __floats2half2_rn(p8[k][6], p8[k][7]);
        pk.x = *reinterpret_cast<uint32_t*>(&h0); pk.y = *reinterpret_cast<uint32_t*>(&h1);
        pk.z = *reinterpret_cast<uint32_t*>(&h2); pk.w = *reinterpret_cast<uint32_t*>(&h3);
        __half* const* dst = l < (size_t)L ? P.w16 : P.w3h;
        const size_t off = l < (size_t)L ? l * wsz + r : r;
        if (mc) mm_st_b128((l < (size_t)L ? P.mc_w16 : P.mc_w3h) + off, pk);
        else for (int qq = 0; qq < world; ++qq) *reinterpret_cast<uint4*>(dst[qq] + off) = pk;
      } else {
        // biases (fp32, read by the kernels in fp32: they travel to every rank's parameter buffer), the fc3 tail, a partial group
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const size_t ie = i + e;
          if (ie >= hi) continue;
          if (i + 8 > hi) { p[ie] = p8[k][e]; m[ie] = m8[k][e]; v[ie] = v8[k][e]; }
          const size_t le = ie / kLayerStride, re = ie % kLayerStride;
          if (mc) {
            if (le < (size_t)L) {
              // (single fp16 elements only occur in a partial group: multimem.st has no 16-bit form, plain peer stores)
              if (re < wsz) { for (int qq = 0; qq < world; ++qq) P.w16[qq][le * wsz + re] = __float2half_rn(p8[k][e]); }
              else mm_st_f32(P.mc_params + ie, p8[k][e]);
            } else if (re < (size_t)C3 * kC) {
              for (int qq = 0; qq < world; ++qq) P.w3h[qq][re] = __float2half_rn(p8[k][e]);
            } else {
              mm_st_f32(P.mc_params + ie, p8[k][e]);   // fc3 bias
            }
          } else if (le < (size_t)L) {
            if (re < wsz) { for (int qq = 0; qq < world; ++qq) P.w16[qq][le * wsz + re] = __float2half_rn(p8[k][e]); }
            else { for (int qq = 0; qq < world; ++qq) if (qq != rank) P.params[qq][ie] = p8[k][e]; }
          } else if (re < (size_t)C3 * kC) {
            for (int qq = 0; qq < world; ++qq) P.w3h[qq][re] = __float2half_rn(p8[k][e]);
          } else {
            for (int qq = 0; qq < world; ++qq) if (qq != rank) P.params[qq][ie] = p8[k][e];   // fc3 bias
          }
        }
      }
    }
  }
  // ---- 6: bookkeeping by the last block ----
  __syncthreads();
  if (stamp0) stamps[4] = now();
  if (threadIdx.x == 0) {
    __threadfence_system();   // this block's remote weight stores before its arrival
    if (stamp0) stamps[5] = now();
    if (atomicAdd(sync_state + 3, 1u) == gridDim.x - 1) {
      sync_state[3] = 0u;
      scaler_update(scaler_state, found, 1);
      *found_inf_io = found;
      for (int k = 0; k < 4; ++k) my_grads[n + k] = scratch[k];   // every rank has read this rank's slots (its verdict came after)
      sync_state[0] = (unsigned int)epoch;
      __threadfence_system();
      for (int r = 0; r < world; ++r) st_relaxed_sys(P.flags[r] + kSigApplied + rank, epoch);
      stamps[6] = now();
      // the kernel completes only when every rank's shard of the new weights has landed in THIS rank's buffers
      for (int r = 0; r < world; ++r) dp_wait_row(my_flags, kSigApplied, r, epoch);
      stamps[7] = now();
    }
  }
}

}  // namespace acez

using namespace acez;

extern "C" size_t acez_adamw_dp_shard(size_t n, int world) {
  if (world < 1) return 0;
  const size_t per = (n + (size_t)world - 1) / (size_t)world;
  return (per + 7) / 8 * 8;
}

extern "C" int acez_adamw_dp_step(const void* const* peer_grads, void* const* peer_flags, void* const* peer_w16, void* const* peer_w3h,
                                  void* const* peer_params, int world, int rank, size_t n, float* reduced_shard, float* params,
                                  float* exp_avg, float* exp_avg_sq, const float* hyper_dev, float* scaler_state_dev,
                                  int* found_inf_dev, float* local_extras, unsigned int* sync_state_dev, const float* local_stats_dev,
                                  const void* const* multicast, int L, int C3, acez_stream_t stream) {
  ACEZ_REQUIRE(peer_grads && peer_flags && peer_w16 && peer_w3h && peer_params && reduced_shard && params && exp_avg && exp_avg_sq &&
                   hyper_dev && scaler_state_dev && found_inf_dev && local_extras && sync_state_dev,
               "adamw_dp_step: null argument");
  ACEZ_REQUIRE(world >= 1 && world <= kMaxRanks && rank >= 0 && rank < world && L >= 1 && (C3 == 3 || C3 == 4),
               "adamw_dp_step: bad arguments");
  ACEZ_REQUIRE(n == head_param_count(L, C3), "adamw_dp_step: parameter count does not match the head");
  int rc = acez_device_check();
  if (rc) return rc;
  DpPeers P{};
  for (int r = 0; r < world; ++r) {
    ACEZ_REQUIRE(peer_grads[r] && peer_flags[r] && peer_w16[r] && peer_w3h[r] && peer_params[r], "adamw_dp_step: null peer pointer %d", r);
    P.grads[r] = reinterpret_cast<const float*>(peer_grads[r]);
    P.flags[r] = reinterpret_cast<int*>(peer_flags[r]);
    P.w16[r] = reinterpret_cast<__half*>(peer_w16[r]);
    P.w3h[r] = reinterpret_cast<__half*>(peer_w3h[r]);
    P.params[r] = reinterpret_cast<float*>(peer_params[r]);
  }
  if (multicast != nullptr && multicast[0] && multicast[1] && multicast[2] && multicast[3]) {
    P.mc_grads = reinterpret_cast<const float*>(multicast[0]);
    P.mc_w16 = reinterpret_cast<__half*>(const_cast<void*>(multicast[1]));
    P.mc_w3h = reinterpret_cast<__half*>(const_cast<void*>(multicast[2]));
    P.mc_params = reinterpret_cast<float*>(const_cast<void*>(multicast[3]));
  }
  const size_t shard = acez_adamw_dp_shard(n, world);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (local_stats_dev != nullptr) {
    // the one-kernel step, when the shard's parameter groups (gpt per thread) fit the registers of one co-resident grid; scratch =
    // the four floats behind the reduced-shard buffer. Launched plainly (no programmatic dependent launch): the grid starts only
    // after the previous kernel of the stream has drained, so all of it is resident.
    const int gpt = world <= 2 ? 2 : 1;
    const auto kern = world <= 2 ? &adamw_dp_fused_kernel<2, 2> : world <= 4 ? &adamw_dp_fused_kernel<1, 4> : &adamw_dp_fused_kernel<1, 8>;
    int per_sm = 0;
    ACEZ_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 256, 0));
    if (per_sm > 2) per_sm = 2;
    const size_t threads = (size_t)per_sm * sm_count() * 256;
    if (per_sm >= 1 && (shard + 7) / 8 <= (size_t)gpt * threads)
      return launch_kernel(kern, dim3(per_sm * sm_count()), dim3(256), 0, st, false, P, world, rank, n, shard, params, exp_avg,
                           exp_avg_sq, hyper_dev, scaler_state_dev, found_inf_dev, local_extras - n, local_stats_dev,
                           reduced_shard + shard, sync_state_dev, reinterpret_cast<unsigned long long*>(reduced_shard), L, C3);
  }
  // (blocks that poll a signal wait for REMOTE progress only, and the signals are sent by block 0 / the last block to finish:
  // no block of these grids waits for another block of its own GPU, so residency is not a correctness condition)
  const int grid = 2 * sm_count();
  // local_extras = this rank's gradient + n: the four spare slots; local_stats_dev (nullable): pack them here instead of in
  // separate kernels (found_inf_dev still holds the local backward's flag at this point)
  float* my_grads = local_stats_dev != nullptr ? local_extras - n : nullptr;
  rc = launch_kernel(adamw_dp_reduce_kernel, dim3(grid), dim3(256), 0, st, false, P, world, rank, n, shard, reduced_shard, my_grads,
                     found_inf_dev, local_stats_dev, sync_state_dev);
  if (rc) return rc;
  return launch_kernel(adamw_dp_apply_kernel, dim3(grid), dim3(256), 0, st, false, P, world, rank, n, shard, reduced_shard, params,
                       exp_avg, exp_avg_sq, hyper_dev, scaler_state_dev, P.flags[rank], found_inf_dev, local_extras, L, C3,
                       sync_state_dev);
}
