// Fused layer chain of the ACE head on tcgen05 cta_group::2 (the default head path; design: DESIGN.md section 3.8, interface:
// head_chain.cuh): ALL hidden 512 x 512 layers of one pass (forward: 8, dgrad: 7) in ONE launch.
//
// Why cta_group::2: the round-1 chain on cta_group::1 (a cluster of two CTAs per 128-row tile) was bound by the shared-memory
// port (per layer and CTA 384 KB of UMMA operand reads + 256 KB of weight fill + 4 x 64 KB of box traffic against 4.1 k cycles of
// UMMA issue). With cta_group::2 the two CTAs of an SM pair share every weight k-block (each stages HALF of it, the hardware feeds
// both tensor cores from both halves): 128 KB of weight fill and 256 KB of operand reads per layer and CTA, and the same 96 KB ring
// holds twice as many k-blocks in flight. Measured (round 2): 43-45 us per forward chain against 55.6 us.
//
// Decomposition: a cluster of FOUR CTAs owns TWO 128-row tiles. rank = 2 c + r:
//   r = row tile inside the cluster, c = channel half. Pair P_c = {2c, 2c+1} (an SM pair) runs
//   tcgen05.mma.cta_group::2 with M = 256 (CTA r contributes its row tile's 128 x 512 A buffer), N = 256 (output channels
//   [256 c, 256 c + 256) of the layer; CTA r stages weight rows [256 c + 128 r, +128) of every k-block). Accumulators:
//   each CTA's TMEM holds ITS rows x the pair's 256 channels, double buffered.
// Roles: warp 0 TMA producer (both CTAs: own A tile, own half of every weight k-block, completing on the LEADER's barrier);
//   warp 1 of the pair leader (r = 0) issues the UMMAs; warp 1 of the other CTA is a RELAY: the leader cannot wait on a
//   remote mbarrier, so the partner forwards "my k-block j is in place" to the leader's partner_ready[j];
//   warps 2..9: epilogue, two groups of four warps (one warp per TMEM lane quarter), BOTH groups on the same 64-column box (32
//   columns each), box after box: TMEM -> registers -> bias / ReLU / residual (or ReLU-mask bits) -> fp16 -> the box of the A buffer
//   that is k-block (4 c + box) of the NEXT layer; one thread then publishes the box to the local MMA warp (mbarrier), copies it
//   into the exchange partner's (rank ^ 2: same row tile, other channel half) A buffer (bulk DSMEM copy completing on the partner's
//   mbarrier) and stores it to HBM (TMA store).
// tcgen05.commit ... multicast::cluster (mask of the pair) releases weight stages / publishes accumulators to both CTAs.
//
// Hazards and how they are ordered (s = step index, one step = one layer):
//   * MMA s+1 reads box j            after  a_ready[j] phase s+1 (own box: epilogue arrive; partner's box: complete_tx) on BOTH CTAs
//                                           of the pair (partner_ready[j] relays the other CTA's)
//   * epilogue s overwrites own box  after  tmem_full[s&1] (all MMAs of step s retired => A_s fully consumed), after the TMA store
//                                           that last read it (cp.async.bulk.wait_group.read) and after peer_free phase s (the
//                                           exchange partner consumed the DSMEM copy that read it)
//   * copy into the partner's box    after  peer_free phase s (= the partner's MMAs of step s retired)
//   * TMEM buffer s&1 rewritten by MMA s+2: needs every box of epilogue s+1, which follows epilogue s in program order
// The protocol is model-checked under random interleavings by tools/sim_chain4_protocol.py.
// The host side (tensor maps of a pass, the launch, the profiling probe's stamp buffer) is at the end of this file.
#include <stdlib.h>

#include "cluster2.cuh"
#include "head_chain.cuh"

namespace acez {

static constexpr int kC = 512;
static constexpr int CM = 128, CN = 256, CK = 64;
static constexpr int kKB = kC / CK;
static constexpr int kBoxBytes = CM * CK * 2;        // 16 KB
static constexpr int kABytes = kKB * kBoxBytes;      // 128 KB
static constexpr int kBHalf = (CN / 2) * CK * 2;     // 16 KB: this CTA's half of a weight k-block
static constexpr int kBStages = 6;
static constexpr int kSmem4 = kABytes + kBStages * kBHalf + 1024 /*fp32 bias slice*/ + 384 /*barriers*/ + 1024 /*align*/;
static_assert(kSmem4 <= 232448, "shared memory budget");
static constexpr uint32_t kSw128 = 2;

__device__ __forceinline__ bool c4_try_wait(uint64_t* bar, uint32_t parity, int sem /*0 cta acquire, 2 cluster relaxed*/) {
  if (sem == 0) return mbar_try_wait(bar, parity);
  uint32_t ok;
  asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.relaxed.cluster.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
               : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __noinline__ void c4_timeout(uint32_t tag, uint32_t parity) {
  printf("acez: chain4 wait timeout: kind %u step %u index %u parity %u (block %d, cta rank %d, thread %d)\n", tag >> 16,
         (tag >> 8) & 0xFF, tag & 0xFF, parity, blockIdx.x, (int)cluster_ctarank(), threadIdx.x);
  __trap();
}
// kinds: 1 a_ready, 2 b_full, 3 b_empty, 4 tmem_full, 5 peer_free, 7 partner_ready
template <int SEM>
__device__ __forceinline__ void c4_wait(uint64_t* bar, uint32_t parity, uint32_t tag) {
  if (c4_try_wait(bar, parity, SEM)) return;
  const long long t0 = clock64();
  while (!c4_try_wait(bar, parity, SEM)) {
    if (clock64() - t0 > kChainWatchdogCycles) c4_timeout(tag, parity);
  }
}
// consumption order of the 8 k-blocks. Two epilogue groups publish own boxes 0,1 first and 2,3 one box time later, so the
// ARRIVAL order is own 0,1 | exchange partner's 0,1 | own 2,3 | partner's 2,3. The alternative (own_first: own 0..3 | partner's
// 0..3, the order of the cta_group::1 chain; four groups publish all own boxes together) sums the k-blocks in an order
// closer to the index order of the per-layer kernels / the CPU oracle: same arithmetic, different fp32 summation order.
__device__ __forceinline__ int c4_order(int i, int c, bool own_first) {
  if (own_first) return (i < 4 ? c : (c ^ 1)) * 4 + (i & 3);
  const int b = ((i >> 2) << 1) | (i & 1);
  return ((i & 2) ? (c ^ 1) : c) * 4 + b;
}
__device__ __forceinline__ bool c4_is_partner_box(int i, bool own_first) { return own_first ? i >= 4 : (i & 2) != 0; }

// prmt.b32 with the sign-replicate bit (8) in the selector nibbles: byte <- 0xFF / 0x00 from the msb of the selected byte
__device__ __forceinline__ uint32_t c4_prmt(uint32_t a, uint32_t b, uint32_t sel) {
  uint32_t d;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
  return d;
}

// ---- epilogue arithmetic of one 32-column half of a box (thread = one accumulator row) ----
// ReLU-mask bit layout (MASKB, 64 B per row and layer = 8 B per box): one 32-bit word per 32-column half; bit t = column 2t,
// bit 16 + t = column 2t + 1 (t = 0..15). A packed half2 compare (HSET2: 0xFFFF per true half) then needs ONE LOP3 per column
// pair to deposit both bits, and the dgrad side one shift + one prmt (sign replication) to expand them again.
template <bool RES_ADD, bool WANT_MASK>
__device__ __forceinline__ void c4_fwd_half(const uint32_t (&vv)[32], uint32_t* __restrict__ res /*16 words: this half*/, const int hf,
                                            const uint32_t bias_addr, const uint32_t dst, const uint32_t swz, uint32_t& bits) {
  const __half2 zero2 = __floats2half2_rn(0.f, 0.f);
  uint32_t word = 0u;
#pragma unroll
  for (int q4 = 0; q4 < 4; ++q4) {
    const int q = hf * 4 + q4;
    const float4 bf0 = lds_128f(bias_addr + 4u * (uint32_t)(q * 8));
    const float4 bf1 = lds_128f(bias_addr + 4u * (uint32_t)(q * 8 + 4));
    const float bq[8] = {bf0.x, bf0.y, bf0.z, bf0.w, bf1.x, bf1.y, bf1.z, bf1.w};
    uint4 o;
    uint32_t* ob = reinterpret_cast<uint32_t*>(&o);
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int vc = q4 * 8 + 2 * t;
      const int tt = q4 * 4 + t;   // column pair inside the half
      // single rounding of (acc + bias) to fp16; ReLU on the rounded value gives the same result as before it
      __half2 h = __hmax2(__floats2half2_rn(__uint_as_float(vv[vc]) + bq[2 * t], __uint_as_float(vv[vc + 1]) + bq[2 * t + 1]), zero2);
      if (WANT_MASK) word |= __hgt2_mask(h, zero2) & ((1u << tt) | (1u << (16 + tt)));   // pre-residual x > 0
      if (RES_ADD) {
        uint32_t& rs = res[4 * q4 + t];
        h = __hadd2(*reinterpret_cast<const __half2*>(&rs), h);  // residual sum in fp16, as the reference's `res + x`
        rs = *reinterpret_cast<const uint32_t*>(&h);
      }
      ob[t] = *reinterpret_cast<const uint32_t*>(&h);
    }
    sts_128(dst + ((((uint32_t)q) ^ swz) << 4), o);
  }
  bits = word;
}

template <bool RES_ADD, bool RES_SAVE>
__device__ __forceinline__ void c4_dgrad_half(const uint32_t (&vv)[32], uint32_t* __restrict__ res /*16 words: this half*/, const int hf,
                                              const uint32_t mask_word, const uint32_t dst, const uint32_t swz, uint32_t& badbits) {
#pragma unroll
  for (int q4 = 0; q4 < 4; ++q4) {
    const int q = hf * 4 + q4;
    uint4 o;
    uint32_t* ob = reinterpret_cast<uint32_t*>(&o);
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int vc = q4 * 8 + 2 * t;
      const int tt = q4 * 4 + t;
      uint32_t& rs = res[4 * q4 + t];
      // autograd: the conv-backward result is rounded to fp16 first, the skip gradient is added in fp16
      __half2 h = __floats2half2_rn(__uint_as_float(vv[vc]), __uint_as_float(vv[vc + 1]));
      if (RES_ADD) h = __hadd2(h, *reinterpret_cast<const __half2*>(&rs));
      const uint32_t hb = *reinterpret_cast<const uint32_t*>(&h);
      if (RES_SAVE) rs = hb;   // the unmasked sum is the skip-path gradient of the block below
      badbits |= ((hb & 0x7C007C00u) + 0x04000400u) & 0x80008000u;  // exponent all ones: inf / nan
      // bits tt / 16 + tt -> the sign bits of bytes 0 / 2, replicated over each half by prmt
      const uint32_t x = (tt <= 7) ? (mask_word << (7 - tt)) : (mask_word >> (tt - 7));
      ob[t] = hb & c4_prmt(x, x, 0xAA88u);
    }
    sts_128(dst + ((((uint32_t)q) ^ swz) << 4), o);
  }
}

template <int MODE>
__global__ void __launch_bounds__(320, 1)
head_chain4_kernel(const __grid_constant__ CUtensorMap tmIn, const __grid_constant__ CUtensorMap tmW,
                   const __grid_constant__ CUtensorMap tmOut, const __grid_constant__ ChainArgs args) {
  constexpr int G = 2;          // epilogue groups (4 warps each, one per TMEM lane quarter)
  constexpr bool SPLIT = true;  // both groups on the same box, 32 columns each (the whole-box-per-group and four-group variants
                                // measured slower in round 2 and were removed)
  constexpr bool kDgrad = (MODE == CHAIN_DGRAD);
  constexpr int NB = 4;         // boxes a group touches per step (half of each of the four)
  constexpr int kEpiThreads = 128 * G;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;
  uint8_t* sB = smem + kABytes;
  float* sBiasF = reinterpret_cast<float*>(sB + kBStages * kBHalf);
  uint64_t* a_ready = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(sBiasF) + 1024);
  uint64_t* partner_ready = a_ready + kKB;   // leader only: the other CTA of the pair has k-block j in place
  uint64_t* b_full = partner_ready + kKB;    // leader only (count 2)
  uint64_t* b_empty = b_full + kBStages;
  uint64_t* tmem_full = b_empty + kBStages;
  uint64_t* peer_free = tmem_full + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(peer_free + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rank = (int)cluster_ctarank();
  const int c = rank >> 1, r = rank & 1;
  const bool leader = r == 0;
  const int xpeer = rank ^ 2;               // exchange partner: same row tile, other channel half
  const uint16_t pair_mask = (uint16_t)(0x3u << (2 * c));
  const int m0 = ((int)(blockIdx.x >> 2) * 2 + r) * CM;
  const int n_base = c * CN;                // the pair's output channels of every layer
  const int nb_half = n_base + r * (CN / 2);
  const int n_steps = args.n_steps;
  const bool own_first = (args.flags & kChainFlagOwnFirst) != 0;   // k-block consumption order
  long long* dbg = args.dbg != nullptr ? args.dbg + (size_t)blockIdx.x * kChainDbgSlots : nullptr;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmIn);
    tma_prefetch_desc(&tmW);
    tma_prefetch_desc(&tmOut);
    for (int i = 0; i < kKB; ++i) {
      mbar_init(&a_ready[i], 1);
      mbar_init(&partner_ready[i], 1);
    }
    for (int i = 0; i < kBStages; ++i) {
      mbar_init(&b_full[i], 2);   // leader: arrive.expect_tx (both halves) + the partner's arrive
      mbar_init(&b_empty[i], 1);  // multicast commit
    }
    mbar_init(&tmem_full[0], 1);
    mbar_init(&tmem_full[1], 1);
    mbar_init(peer_free, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc_pair(tmem_ptr, 512);
  tcgen05_fence_before();
  __syncwarp();
  cluster_sync();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  // programmatic dependent launch: everything above overlapped the predecessor's tail; its global writes are visible from
  // here on. (A plain launch returns from the wait at once.) The successor may be scheduled as soon as SMs free up.
  pdl_wait();
  pdl_launch_dependents();
  if (dbg && threadIdx.x == 0) dbg[0] = clock64();

  if (warp == 0) {
    // ------------------------------ TMA producer ------------------------------
    if (elect_one()) {
      for (int i = 0; i < kKB; ++i) {
        const int j = c4_order(i, c, own_first);
        mbar_arrive_expect_tx(&a_ready[j], kBoxBytes);
        tma_load_3d(sA + j * kBoxBytes, &tmIn, &a_ready[j], j * CK, m0, 0);
      }
      int stage = 0;
      uint32_t phase = 0;
      for (int s = 0; s < n_steps; ++s) {
        const int wl = args.step[s].w_layer;
        for (int i = 0; i < kKB; ++i) {
          const int j = c4_order(i, c, own_first);
          c4_wait<0>(&b_empty[stage], phase ^ 1, (3u << 16) | ((uint32_t)s << 8) | (uint32_t)i);
          if (leader) mbar_arrive_expect_tx(&b_full[stage], 2 * kBHalf);
          else mbar_arrive_leader(&b_full[stage]);
          uint8_t* dst = sB + stage * kBHalf;
          if (!kDgrad) {
            tma_load_3d_pair(dst, &tmW, &b_full[stage], j * CK, nb_half, wl);  // 128 weight rows x 64 input channels
          } else {
#pragma unroll
            for (int t = 0; t < 2; ++t) tma_load_3d_pair(dst + t * 8192, &tmW, &b_full[stage], nb_half + 64 * t, j * CK, wl);
          }
          if (++stage == kBStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    const uint32_t xpeer_free = mapa_cluster(smem_u32(peer_free), (uint32_t)xpeer);
    if (leader) {
      // ------------------------------ UMMA issuer (pair leader) ------------------------------
      constexpr uint32_t idesc = make_idesc_f16(2 * CM, CN, false, kDgrad);
      constexpr uint32_t b_lbo = kDgrad ? 8192u : 0u;
      constexpr uint32_t b_kstep = kDgrad ? 2048u : 32u;
      int stage = 0;
      uint32_t phase = 0;
      for (int s = 0; s < n_steps; ++s) {
        const uint32_t d_tmem = tmem_base + (uint32_t)((s & 1) * CN);
        for (int i = 0; i < kKB; ++i) {
          const int j = c4_order(i, c, own_first);
          c4_wait<0>(&a_ready[j], (uint32_t)(s & 1), (1u << 16) | ((uint32_t)s << 8) | (uint32_t)j);
          if (c4_is_partner_box(i, own_first) && s + 1 < n_steps && lane == 0) mbar_arrive_expect_tx(&a_ready[j], kBoxBytes);  // arm the next phase
          c4_wait<2>(&partner_ready[j], (uint32_t)(s & 1), (7u << 16) | ((uint32_t)s << 8) | (uint32_t)j);
          c4_wait<0>(&b_full[stage], phase, (2u << 16) | ((uint32_t)s << 8) | (uint32_t)i);
          tcgen05_fence_after();
          if (dbg && lane == 0 && (i == 0 || i == 2 || i == 7)) dbg[8 + 8 * s + (i == 0 ? 0 : (i == 7 ? 2 : 1))] = clock64();
          if (elect_one()) {
            const uint32_t a_addr = smem_u32(sA + j * kBoxBytes);
            const uint32_t b_addr = smem_u32(sB + stage * kBHalf);
#pragma unroll
            for (int k = 0; k < CK / 16; ++k) {
              const uint64_t da = make_smem_desc(a_addr + k * 32, 0, 1024, kSw128);
              const uint64_t db = make_smem_desc(b_addr + k * b_kstep, b_lbo, 1024, kSw128);
              umma_f16_pair(d_tmem, da, db, idesc, (i | k) != 0 ? 1u : 0u);
            }
          }
          __syncwarp();
          if (elect_one()) {
            tcgen05_commit_pair(&b_empty[stage], pair_mask);
            if (i == kKB - 1) tcgen05_commit_pair(&tmem_full[s & 1], pair_mask);
          }
          __syncwarp();
          if (++stage == kBStages) { stage = 0; phase ^= 1; }
        }
        c4_wait<0>(&tmem_full[s & 1], (uint32_t)((s >> 1) & 1), (4u << 16) | ((uint32_t)s << 8) | 1u);
        if (lane == 0) {
          mbar_arrive_remote_relaxed(xpeer_free);
          if (dbg) dbg[8 + 8 * s + 3] = clock64();
        }
        __syncwarp();
      }
    } else {
      // ------------------------------ relay (the other CTA of the pair) ------------------------------
      for (int s = 0; s < n_steps; ++s) {
        for (int i = 0; i < kKB; ++i) {
          const int j = c4_order(i, c, own_first);
          c4_wait<0>(&a_ready[j], (uint32_t)(s & 1), (1u << 16) | ((uint32_t)s << 8) | (uint32_t)j);
          if (lane == 0) {
            if (c4_is_partner_box(i, own_first) && s + 1 < n_steps) mbar_arrive_expect_tx(&a_ready[j], kBoxBytes);  // arm the next phase
            // my k-block j of step s is in place IN MY OWN shared memory (generic-proxy writes were fenced by their writers,
            // async copies completed on the barrier) and it is my own tensor core that will read it: the signal to the
            // leader, which issues the UMMAs for both CTAs, carries no data - relaxed, no fence (a release at cluster scope
            // costs a MEMBAR.ALL.GPU per k-block here; measured ~600 cycles per handshake in the 2-CTA chain)
            mbar_arrive_remote_relaxed(mapa_cluster(smem_u32(&partner_ready[j]), (uint32_t)(rank & ~1)));
          }
          __syncwarp();
        }
        c4_wait<0>(&tmem_full[s & 1], (uint32_t)((s >> 1) & 1), (4u << 16) | ((uint32_t)s << 8) | 1u);
        if (lane == 0) mbar_arrive_remote_relaxed(xpeer_free);
        __syncwarp();
      }
    }
  } else {
    // ------------------------------ epilogue (exchange partner = rank ^ 2) ------------------------------
    const int quarter = warp & 3;
    const int grp = (warp - 2) >> 2;                 // 0 .. G-1
    const int rr = quarter * 32 + lane;
    const int row = m0 + rr;
    const bool row_ok = row < args.rows;
    const int etid = threadIdx.x - 64;
    // one issuing thread per group, on different warps / SM sub-partitions
    const bool issuer = lane == 0 && grp == 0 && quarter == 2;   // the one thread that issues the copies of a finished box
    const uint32_t swz = (uint32_t)(rr & 7);
    const uint32_t t_row = tmem_base + ((uint32_t)(quarter * 32) << 16);
    const uint32_t sA_u32 = smem_u32(sA), sBias_u32 = smem_u32(sBiasF);
    auto bar_group = [&]() { asm volatile("bar.sync %0, 128;" ::"r"(grp + 1) : "memory"); };
    auto bar_all = [&]() { asm volatile("bar.sync 6, %0;" ::"n"(kEpiThreads) : "memory"); };
    uint32_t badbits = 0;
    // residual stream (forward) / skip-path gradient (dgrad) of this thread's row and boxes: stays in registers
    uint32_t res[NB][16];
#pragma unroll
    for (int sl = 0; sl < NB; ++sl)
#pragma unroll
      for (int t = 0; t < 16; ++t) res[sl][t] = 0u;
    if (!kDgrad && (args.flags & kChainFlagResInit)) {
      // res_0 = the input tile: this thread's row, its 32-column half of each of the CTA's four boxes
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int j = c * 4 + b;
        c4_wait<0>(&a_ready[j], 0u, (1u << 16) | (0xFFu << 8) | (uint32_t)j);
        const uint32_t src = sA_u32 + (uint32_t)(j * kBoxBytes + rr * 128);
#pragma unroll
        for (int q4 = 0; q4 < 4; ++q4) {
          const uint4 t = lds_128(src + ((((uint32_t)(grp * 4 + q4)) ^ swz) << 4));
          res[b][4 * q4] = t.x; res[b][4 * q4 + 1] = t.y; res[b][4 * q4 + 2] = t.z; res[b][4 * q4 + 3] = t.w;
        }
      }
    }
    for (int s = 0; s < n_steps; ++s) {
      const ChainStep& st = args.step[s];
      const int tbuf = s & 1;
      const bool last = (s == n_steps - 1);
      if (!kDgrad) {
        // fp32 copy of the fp16-rounded bias slice (autocast casts the bias to fp16 before the conv adds it); every
        // epilogue warp must have finished the previous step's boxes before it is overwritten
        if (s > 0) bar_all();
        if (etid < CN) sts_f32(sBias_u32 + 4u * (uint32_t)etid, __half2float(__float2half_rn(st.bias != nullptr ? __ldg(st.bias + n_base + etid) : 0.f)));
      }
      // ReLU-mask word of this thread's row and half for each box (dgrad): in flight while the accumulator is computed
      uint32_t mwb[4] = {0u, 0u, 0u, 0u};
      if (kDgrad && row_ok) {
#pragma unroll
        for (int b = 0; b < 4; ++b) mwb[b] = __ldcg(reinterpret_cast<const uint32_t*>(st.mask_in + (size_t)row * 64 + (c * 4 + b) * 8 + 4 * grp));
      }
      if (issuer) {
        // peer_free phase s: the exchange partner's MMAs of step s have retired, i.e. it has consumed the boxes copied to it during
        // step s-1 (those copies no longer read the boxes rewritten below) and its A buffer may be overwritten
        c4_wait<2>(peer_free, (uint32_t)(s & 1), (5u << 16) | ((uint32_t)s << 8));
        // the TMA stores of the previous step (issued one whole step ago) have finished reading the boxes
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        if (dbg) dbg[8 + 8 * s + 5] = clock64();
      }
      c4_wait<0>(&tmem_full[tbuf], (uint32_t)((s >> 1) & 1), (4u << 16) | ((uint32_t)s << 8));
      tcgen05_fence_after();
      if (dbg && etid == 0) dbg[8 + 8 * s + 4] = clock64();
      bar_all();   // bias slice visible; the issuer's permissions hold for every epilogue thread
      const int res_add = st.res_add, res_save = st.res_save;
      const bool want_mask = !kDgrad && st.mask_out != nullptr;
      uint32_t vv[2][32];
      tmem_ld_32x32(t_row + (uint32_t)(tbuf * CN + grp * 32), vv[0]);
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int j = c * 4 + b;
        tmem_ld_wait_for(vv[b & 1]);
        if (b + 1 < 4) tmem_ld_32x32(t_row + (uint32_t)(tbuf * CN + (b + 1) * 64 + grp * 32), vv[(b + 1) & 1]);
        const uint32_t dst = sA_u32 + (uint32_t)(j * kBoxBytes + rr * 128);
        if (!kDgrad) {
          uint32_t word = 0u;
          const uint32_t bias_addr = sBias_u32 + 4u * (uint32_t)(b * 64);
          if (res_add) {
            if (want_mask) c4_fwd_half<true, true>(vv[b & 1], res[b], grp, bias_addr, dst, swz, word);
            else c4_fwd_half<true, false>(vv[b & 1], res[b], grp, bias_addr, dst, swz, word);
          } else {
            if (want_mask) c4_fwd_half<false, true>(vv[b & 1], res[b], grp, bias_addr, dst, swz, word);
            else c4_fwd_half<false, false>(vv[b & 1], res[b], grp, bias_addr, dst, swz, word);
          }
          if (want_mask && row_ok) *reinterpret_cast<uint32_t*>(st.mask_out + (size_t)row * 64 + j * 8 + 4 * grp) = word;
        } else {
          if (res_add) {
            if (res_save) c4_dgrad_half<true, true>(vv[b & 1], res[b], grp, mwb[b], dst, swz, badbits);
            else c4_dgrad_half<true, false>(vv[b & 1], res[b], grp, mwb[b], dst, swz, badbits);
          } else {
            if (res_save) c4_dgrad_half<false, true>(vv[b & 1], res[b], grp, mwb[b], dst, swz, badbits);
            else c4_dgrad_half<false, false>(vv[b & 1], res[b], grp, mwb[b], dst, swz, badbits);
          }
        }
        // box complete once both groups are here. Its TMEM columns are rewritten by the MMAs of step s+2, which are released
        // (transitively) by the barrier arrival below: order the completed tcgen05.ld before it
        tcgen05_fence_before();
        fence_proxy_async();   // publish the half box to the tensor core / copy engines (async proxy)
        bar_all();
        if (issuer) {
          const uint32_t box_addr = smem_u32(sA + j * kBoxBytes);
          if (!last) {
            mbar_arrive(&a_ready[j]);
            dsmem_copy(mapa_cluster(box_addr, (uint32_t)xpeer), box_addr, kBoxBytes, mapa_cluster(smem_u32(&a_ready[j]), (uint32_t)xpeer));
          }
          if (st.out_slot >= 0) tma_store_3d(&tmOut, sA + j * kBoxBytes, n_base + b * 64, m0, st.out_slot);
          tma_store_commit();
          if (dbg && (b == 0 || b == 2)) dbg[8 + 8 * s + (b == 0 ? 6 : 7)] = clock64();
        }
      }
    }
    if (issuer) tma_store_wait_all();
    if (kDgrad && args.nonfinite != nullptr) {
      if (__any_sync(0xffffffffu, badbits != 0) && lane == 0) atomicOr(args.nonfinite, 1);
    }
  }

  if (dbg && threadIdx.x == 0) dbg[1] = clock64();
  __syncwarp();
  tcgen05_fence_before();
  cluster_sync();
  if (warp == 1) {
    tcgen05_fence_after();
    tmem_dealloc_pair(tmem_base, 512);
  }
}

// ----------------------------------------------------------------------------------------------
// host side
// ----------------------------------------------------------------------------------------------
int chain_prepare(ChainLaunch* C, int mode, const __half* in, const __half* W16, int L, __half* out_base,
                  long long out_zstride, int out_slots, int rows) {
  ACEZ_REQUIRE(C && in && W16 && out_base && rows >= 1 && L >= 1 && out_slots >= 1, "chain_prepare: bad arguments");
  C->mode = mode;
  int rc;
  {
    uint64_t dims[3] = {(uint64_t)kC, (uint64_t)rows, 1};
    uint64_t strides[2] = {(uint64_t)kC * 2, (uint64_t)rows * kC * 2};
    uint32_t box[3] = {64, (uint32_t)CM, 1};
    rc = make_tensor_map(&C->tmIn, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, in, dims, strides, box, nullptr,
                         CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
  }
  {
    uint64_t dims[3] = {(uint64_t)kC, (uint64_t)kC, (uint64_t)L};
    uint64_t strides[2] = {(uint64_t)kC * 2, (uint64_t)kC * kC * 2};
    uint32_t box[3] = {64, (uint32_t)(mode == CHAIN_FWD ? CN / 2 : 64), 1};
    rc = make_tensor_map(&C->tmW, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, W16, dims, strides, box, nullptr,
                         CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
  }
  {
    uint64_t dims[3] = {(uint64_t)kC, (uint64_t)rows, (uint64_t)out_slots};
    uint64_t strides[2] = {(uint64_t)kC * 2, (uint64_t)out_zstride * 2};
    uint32_t box[3] = {64, (uint32_t)CM, 1};
    rc = make_tensor_map(&C->tmOut, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, out_base, dims, strides, box, nullptr,
                         CU_TENSOR_MAP_SWIZZLE_128B);
    if (rc) return rc;
  }
  static const bool own_first = [] {
    // default: own boxes first (the summation order closest to the per-layer kernels / the oracle; all parity tests hold
    // their round-1 tolerances). ACEZ_CHAIN_ORDER=arrival consumes the k-blocks as they arrive (measured 3 us / iteration
    // faster; first-layer weight gradients then differ from the oracle by 3.2e-2 instead of <= 3e-2 relative L2)
    const char* e = getenv("ACEZ_CHAIN_ORDER");
    return e == nullptr || e[0] != 'a';
  }();
  C->args.rows = rows;
  C->args.n_steps = 0;
  C->args.flags = own_first ? kChainFlagOwnFirst : 0;
  C->args.nonfinite = nullptr;
  C->args.dbg = nullptr;
  return ACEZ_OK;
}

static long long* g_chain_dbg = nullptr;
static int g_chain_dbg_ctas = 0;
static constexpr int kChainDbgMaxCtas = 1024;

// profiling probe: device buffer for the clock64 stamps of a launch with `ctas` CTAs (nullptr unless ACEZ_CHAIN_DBG=1)
static long long* chain_debug_buffer(int ctas) {
  static const bool want_dbg = [] {
    const char* e = getenv("ACEZ_CHAIN_DBG");
    return e != nullptr && atoi(e) != 0;
  }();
  if (!want_dbg || ctas > kChainDbgMaxCtas) return nullptr;
  if (g_chain_dbg == nullptr && cudaMalloc(&g_chain_dbg, (size_t)kChainDbgMaxCtas * kChainDbgSlots * sizeof(long long)) != cudaSuccess)
    return nullptr;
  g_chain_dbg_ctas = ctas;
  return g_chain_dbg;
}

int chain_debug_read(long long* host_out, size_t max_slots, int* n_ctas) {
  ACEZ_REQUIRE(host_out != nullptr && n_ctas != nullptr, "chain_debug_read: null argument");
  *n_ctas = 0;
  if (g_chain_dbg == nullptr) return ACEZ_OK;
  ACEZ_CUDA(cudaDeviceSynchronize());
  size_t n = (size_t)g_chain_dbg_ctas * kChainDbgSlots;
  if (n > max_slots) n = max_slots;
  ACEZ_CUDA(cudaMemcpy(host_out, g_chain_dbg, n * sizeof(long long), cudaMemcpyDeviceToHost));
  *n_ctas = g_chain_dbg_ctas;
  return ACEZ_OK;
}

template <int MODE>
static int chain_launch_mode(const ChainLaunch& C, cudaStream_t stream, bool pdl) {
  constexpr auto kern = head_chain4_kernel<MODE>;
  int rc = set_max_dynamic_smem<kern>(kSmem4);
  if (rc) return rc;
  const int tiles = (C.args.rows + CM - 1) / CM;
  const int ctas = 4 * ((tiles + 1) / 2);   // a cluster of four per two row tiles
  ChainArgs args = C.args;
  args.dbg = chain_debug_buffer(ctas);   // nullptr unless ACEZ_CHAIN_DBG=1 (tools/probe_chain_time.py)
  return launch_kernel<4>(kern, dim3(ctas), dim3(320), kSmem4, stream, pdl, C.tmIn, C.tmW, C.tmOut, args);
}

int chain_launch(const ChainLaunch& C, cudaStream_t stream, bool pdl) {
  ACEZ_REQUIRE(C.args.n_steps >= 1 && C.args.n_steps <= kChainMaxSteps, "chain_launch: %d steps", C.args.n_steps);
  if (C.mode == CHAIN_FWD) return chain_launch_mode<CHAIN_FWD>(C, stream, pdl);
  return chain_launch_mode<CHAIN_DGRAD>(C, stream, pdl);
}

}  // namespace acez
