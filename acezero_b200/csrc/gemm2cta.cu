// tcgen05 GEMM with cta_group::2: the batched weight-gradient GEMM of the training step with the fused layer chain (DESIGN.md
// section 3.9).
//
//   D[z][M,N] (fp32) = A[z] * B[z]      fp16 operands, fp32 accumulation in TMEM, operand layouts as in gemm.cuh
//
// One thread-block CLUSTER of two CTAs (an SM pair of one TPC) computes one 256 x 256 output tile with
// tcgen05.mma.cta_group::2 (M = 256: 128 rows per CTA; N = 256). CTA r of the pair stages, per 64-wide k-block,
//   * its own half of A (rows m0 + 128 r ..) : 16 KB - read only by its own tensor core
//   * ITS HALF OF B (rows n0 + 128 r ..)     : 16 KB - the hardware feeds both tensor cores from both halves
// i.e. 32 KB per CTA and k-block for 128 x 256 x 64 MACs per CTA: half the shared-memory fill and half the operand reads
// per MAC of the cta_group::1 kernel with 128 x 128 tiles (round-1 measurement: the batched weight-gradient GEMM and the
// fused layer chain are bound by the shared-memory port, DESIGN.md section 7). The 2-CTA primitives (cluster2.cuh) are shared
// with the layer chain of head_chain4.cu.
#include "cluster2.cuh"
#include "gemm2cta.cuh"

namespace acez {

static constexpr int T2_BM = 128;   // rows per CTA (256 per pair)
static constexpr int T2_BK = 64;
static constexpr int T2_STAGES = 6;
static constexpr int T2_ASTAGE = T2_BM * T2_BK * 2;        // 16 KB
static constexpr int T2_THREADS = 320;
// BN = columns per pair (256 or 128); each CTA stages BN / 2 rows of B per k-block
template <int BN>
struct T2Cfg {
  static constexpr int kBStage = (BN / 2) * T2_BK * 2;  // 16 KB / 8 KB (this CTA's half of B)
  static constexpr int kStage = T2_ASTAGE + kBStage;
  static constexpr int kSmem = T2_STAGES * kStage + 1024 /*ones tile*/ + 256 + 1024;
};
// C4 = false: one CTA pair per 256 x BN tile (cluster of 2). C4 = true: cluster of FOUR CTAs = two pairs on the same tile, each
// contracting half of the k-blocks into its own TMEM (split-K 2); pair B then ships its accumulator to pair A through
// distributed shared memory (bulk copies into the drained pipeline stages) and pair A adds and stores: the reduction never
// leaves the chip (a split-K through a global workspace cost more than it saved, round 2).
template <bool A_MN, bool B_MN, int T2_BN, bool C4>
__global__ void __launch_bounds__(T2_THREADS, 1)
gemm2cta_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const Gemm2Args args) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr int T2_BSTAGE = T2Cfg<T2_BN>::kBStage;
  constexpr int T2_STAGE = T2Cfg<T2_BN>::kStage;
  uint8_t* sA = smem;
  uint8_t* sB = smem + T2_STAGES * T2_ASTAGE;
  uint8_t* sOnes = smem + T2_STAGES * T2_STAGE;  // 8 rows x 64 halves of 1.0: this CTA's half of the N = 16 bias-gradient operand
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(sOnes + 1024);
  uint64_t* empty_bar = full_bar + T2_STAGES;
  uint64_t* tmem_full_bar = empty_bar + T2_STAGES;
  uint64_t* part_bar = tmem_full_bar + 1;   // C4, pair A: the partner pair's accumulator has landed in this CTA's staging area
  uint64_t* free_bar = part_bar + 1;        // C4, pair B: pair A's pipeline stages are drained, its staging area may be written
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(free_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int crank = (int)cluster_ctarank();
  const int rank = crank & 1;               // CTA inside its pair
  const int kpair = C4 ? (crank >> 1) : 0;  // C4: 0 = pair A (first half of K, stores), 1 = pair B (second half, ships)
  const bool leader = rank == 0;
  const int tile = C4 ? (int)(blockIdx.x >> 2) : (int)(blockIdx.x >> 1);
  const uint16_t pair_mask = (uint16_t)(0x3u << (2 * kpair));
  const int m0 = (tile / args.tiles_n) * (2 * T2_BM) + rank * T2_BM;  // this CTA's 128 rows
  const int n0 = (tile % args.tiles_n) * T2_BN;
  const int nb0 = n0 + rank * (T2_BN / 2);                            // this CTA's half of B
  const int z = blockIdx.z;
  const int split = kpair, n_split = C4 ? 2 : 1;
  const int kb_begin = (int)((long long)args.k_blocks * split / n_split);
  const int kb_end = (int)((long long)args.k_blocks * (split + 1) / n_split);
  const int k_blocks = args.k_blocks;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < T2_STAGES; ++s) {
      mbar_init(&full_bar[s], 2);   // leader: arrive.expect_tx (all bytes of the pair) + the peer's arrive
      mbar_init(&empty_bar[s], 1);  // multicast commit from the leader's MMA warp
    }
    mbar_init(tmem_full_bar, 1);
    mbar_init(part_bar, 1);
    mbar_init(free_bar, 1);
    fence_barrier_init();
  }
  constexpr uint32_t kTmemCols = (T2_BN + 32 <= 256) ? 256u : 512u;  // accumulator + the bias-gradient column block
  if (warp == 1) tmem_alloc_pair(tmem_ptr, kTmemCols);
  // bias gradient dZ^T 1: one extra N = 16 UMMA per k-step against a ones tile (TMEM columns BN..BN+15). Every column tile of
  // an M-tile sees the same A operand, so the work is SPLIT over them: tile tn takes the k-blocks kb % tiles_n == tn (round 2
  // profile: with the whole column on the n0 == 0 tiles those CTAs ran 1.5x longer than the rest and set the kernel time);
  // the partial sums meet in a workspace and the last tile to arrive adds them in a fixed order (deterministic).
  const bool bias_col = args.bias_grad != nullptr;
  const int tn = tile % args.tiles_n, tm = tile / args.tiles_n;
  if (bias_col && warp >= 2) {
    __half2* o = reinterpret_cast<__half2*>(sOnes);
    for (int i = threadIdx.x - 64; i < 1024 / 4; i += 256) o[i] = __floats2half2_rn(1.f, 1.f);
    fence_proxy_async();
  }
  tcgen05_fence_before();
  __syncwarp();
  cluster_sync();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  pdl_wait();               // the set-up above overlapped the predecessor's tail; its writes are visible from here on
  pdl_launch_dependents();

  if (warp == 0) {
    // ------------------------------ TMA producer (both CTAs) ------------------------------
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      long long t_wait = 0;
      const long long t_begin = args.dbg ? clock64() : 0;
      for (int kb = kb_begin; kb < kb_end; ++kb) {
        const long long t0 = args.dbg ? clock64() : 0;
        mbar_wait(&empty_bar[stage], phase ^ 1);
        if (args.dbg) t_wait += clock64() - t0;
        if (leader) mbar_arrive_expect_tx(&full_bar[stage], 2 * T2_STAGE);
        else mbar_arrive_leader(&full_bar[stage]);
        uint8_t* a_dst = sA + stage * T2_ASTAGE;
        uint8_t* b_dst = sB + stage * T2_BSTAGE;
        if (A_MN) {
#pragma unroll
          for (int i = 0; i < T2_BM / 64; ++i) tma_load_3d_pair(a_dst + i * 8192, &tmA, &full_bar[stage], m0 + 64 * i, kb * T2_BK, z);
        } else {
          tma_load_3d_pair(a_dst, &tmA, &full_bar[stage], kb * T2_BK, m0, z);
        }
        if (B_MN) {
#pragma unroll
          for (int i = 0; i < T2_BN / 128; ++i) tma_load_3d_pair(b_dst + i * 8192, &tmB, &full_bar[stage], nb0 + 64 * i, kb * T2_BK, z);
        } else {
          tma_load_3d_pair(b_dst, &tmB, &full_bar[stage], kb * T2_BK, nb0, z);
        }
        if (++stage == T2_STAGES) { stage = 0; phase ^= 1; }
      }
      if (args.dbg) {
        long long* d = args.dbg + 8 * ((size_t)blockIdx.z * gridDim.x + blockIdx.x);
        d[2] = t_wait; d[3] = clock64() - t_begin;
      }
    }
  } else if (warp == 1 && leader) {
    // ------------------------------ UMMA issuer (leader CTA only) ------------------------------
    constexpr uint32_t idesc = make_idesc_f16(2 * T2_BM, T2_BN, A_MN, B_MN);
    constexpr uint32_t idesc_ones = make_idesc_f16(2 * T2_BM, 16, A_MN, false);
    int stage = 0;
    uint32_t phase = 0;
    uint32_t bias_started = 0u;
    long long t_wait = 0;
    const long long t_begin = args.dbg ? clock64() : 0;
    for (int kb = kb_begin; kb < kb_end; ++kb) {
      const long long t0 = args.dbg ? clock64() : 0;
      mbar_wait(&full_bar[stage], phase);
      if (args.dbg) t_wait += clock64() - t0;
      tcgen05_fence_after();
      const bool do_bias = bias_col && (kb % args.tiles_n) == tn;
      if (elect_one()) {
        const uint32_t a_addr = smem_u32(sA + stage * T2_ASTAGE);
        const uint32_t b_addr = smem_u32(sB + stage * T2_BSTAGE);
#pragma unroll
        for (int k = 0; k < T2_BK / 16; ++k) {
          const uint64_t da = make_smem_desc(a_addr + k * args.a_kstep, args.a_lbo, args.a_sbo, 2);
          const uint64_t db = make_smem_desc(b_addr + k * args.b_kstep, args.b_lbo, args.b_sbo, 2);
          umma_f16_pair(tmem_base, da, db, idesc, (kb != kb_begin || k != 0) ? 1u : 0u);
          if (do_bias) {
            const uint64_t d1 = make_smem_desc(smem_u32(sOnes) + k * 32, 0, 1024, 2);
            umma_f16_pair(tmem_base + T2_BN, da, d1, idesc_ones, (bias_started | (uint32_t)k) != 0u ? 1u : 0u);
          }
        }
      }
      if (do_bias) bias_started = 1u;
      __syncwarp();
      if (elect_one()) {
        tcgen05_commit_pair(&empty_bar[stage], pair_mask);
        if (kb == kb_end - 1) tcgen05_commit_pair(tmem_full_bar, pair_mask);
      }
      __syncwarp();
      if (++stage == T2_STAGES) { stage = 0; phase ^= 1; }
    }
    if (args.dbg && lane == 0) {
      long long* d = args.dbg + 8 * ((size_t)blockIdx.z * gridDim.x + blockIdx.x);
      d[0] = t_wait; d[1] = clock64() - t_begin;
    }
  } else if (warp >= 2) {
    // ------------------------------ epilogue (both CTAs: 128 rows x 256 columns each) ------------------------------
    const int quarter = warp & 3;
    const int grp = (warp - 2) >> 2;
    const int row = m0 + quarter * 32 + lane;
    mbar_wait(tmem_full_bar, 0);
    tcgen05_fence_after();
    const long long t_epi = args.dbg ? clock64() : 0;
    const uint32_t t_row = tmem_base + ((uint32_t)(quarter * 32) << 16);
    bool bad = false;
    const int lrow = quarter * 32 + lane;   // row inside this CTA's 128-row half
    // C4: staging area in the drained pipeline stages, [128 rows][BN floats] with a 16-byte pad per row (conflict-free
    // 128-bit accesses by a quarter warp), followed by the 128 partial row sums of the bias column
    constexpr uint32_t kPitch = T2_BN * 4 + 16;
    constexpr uint32_t kStageBytes = T2_BM * kPitch + T2_BM * 4;
    static_assert(!C4 || kStageBytes <= (uint32_t)(T2_STAGES * T2Cfg<T2_BN>::kStage), "staging area exceeds the pipeline stages");
    const uint32_t stg = smem_u32(smem);
    const bool my_bias = bias_col && [&] { bool anyb = false; for (int kb = kb_begin; kb < kb_end; ++kb) anyb |= (kb % args.tiles_n) == tn; return anyb; }();
    if (C4 && kpair == 1) {
      // ---- pair B: accumulator -> own staging -> bulk copies into the partner's staging ----
#pragma unroll 1
      for (int c = grp; c < T2_BN / 32; c += 2) {
        uint32_t v[32];
        tmem_ld_32x32(t_row + c * 32, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 8; ++j)
          sts_128(stg + (uint32_t)lrow * kPitch + (uint32_t)(c * 128 + j * 16), make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]));
      }
      if (grp == 0) {
        float g = 0.f;
        if (my_bias) {
          uint32_t v[32];
          tmem_ld_32x32(t_row + T2_BN, v);
          tmem_ld_wait();
          g = __uint_as_float(v[0]);
        }
        sts_f32(stg + T2_BM * kPitch + 4u * (uint32_t)lrow, g);
      }
      fence_proxy_async();   // generic-proxy writes -> visible to the bulk-copy engine
      asm volatile("bar.sync 2, 256;" ::: "memory");
      if (warp == 2 && lane == 0) {
        mbar_wait(free_bar, 0);   // pair A has retired all its MMAs: its stages are free
        const uint32_t dst_rank = (uint32_t)(crank - 2);
        const uint32_t dst = mapa_cluster(stg, dst_rank);
        const uint32_t bar = mapa_cluster(smem_u32(part_bar), dst_rank);
        constexpr uint32_t kChunk = 32 * kPitch;   // 4 copies of 32 rows + the bias rows
#pragma unroll
        for (uint32_t o = 0; o < T2_BM * kPitch; o += kChunk) dsmem_copy(dst + o, stg + o, kChunk, bar);
        dsmem_copy(dst + T2_BM * kPitch, stg + T2_BM * kPitch, (uint32_t)(T2_BM * 4), bar);
      }
    } else {
      float bias_partner = 0.f;
      if (C4) {
        // ---- pair A: arm the landing barrier, tell the partner that the stages are free, wait for its accumulator ----
        if (warp == 2 && lane == 0) {
          mbar_arrive_expect_tx(part_bar, kStageBytes);
          mbar_arrive_remote_release(mapa_cluster(smem_u32(free_bar), (uint32_t)(crank + 2)));
        }
        mbar_wait(part_bar, 0);
        if (grp == 0) {
          float t;
          asm volatile("ld.shared.f32 %0, [%1];" : "=f"(t) : "r"(stg + T2_BM * kPitch + 4u * (uint32_t)lrow) : "memory");
          bias_partner = t;
        }
      }
#pragma unroll 1
      for (int c = grp; c < T2_BN / 32; c += 2) {
        uint32_t v[32];
        tmem_ld_32x32(t_row + c * 32, v);
        tmem_ld_wait();
        if (C4) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 pq = lds_128f(stg + (uint32_t)lrow * kPitch + (uint32_t)(c * 128 + j * 16));
            v[4 * j] = __float_as_uint(__uint_as_float(v[4 * j]) + pq.x);
            v[4 * j + 1] = __float_as_uint(__uint_as_float(v[4 * j + 1]) + pq.y);
            v[4 * j + 2] = __float_as_uint(__uint_as_float(v[4 * j + 2]) + pq.z);
            v[4 * j + 3] = __float_as_uint(__uint_as_float(v[4 * j + 3]) + pq.w);
          }
        }
        const int ncol = n0 + c * 32;
        if (row >= args.M || ncol >= args.N) continue;
        // 256-bit stores: one full 32-byte sector per lane and instruction (with 16-byte stores every warp store touched 32
        // half-written sectors and the epilogue ran at the L1 -> L2 request rate: 8.8 k cycles for a 128 x 256 tile, round 2)
        float* dst = args.out32 + (long long)z * args.out32_zstride + (long long)row * args.ldo32 + ncol;
        if ((reinterpret_cast<uintptr_t>(dst) & 31) == 0) {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst + 8 * j), "r"(v[8 * j]), "r"(v[8 * j + 1]),
                         "r"(v[8 * j + 2]), "r"(v[8 * j + 3]), "r"(v[8 * j + 4]), "r"(v[8 * j + 5]), "r"(v[8 * j + 6]), "r"(v[8 * j + 7])
                         : "memory");
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j)
            reinterpret_cast<float4*>(dst)[j] = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                                            __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
        }
        if (args.nonfinite != nullptr) {  // GradScaler check folded in
#pragma unroll
          for (int j = 0; j < 32; ++j) bad |= fp16_grad_overflow(__uint_as_float(v[j]));
        }
      }
    if (bias_col && grp == 0) {
      __shared__ int s_last;
      const int tiles_m = (int)(gridDim.x >> (C4 ? 2 : 1)) / args.tiles_n;
      const int r_in_tile = rank * T2_BM + quarter * 32 + lane;            // 0..255 inside the pair's M-tile
      const int slots = args.tiles_n;                                      // partial row sums per M-tile: one per column tile
      float* part = args.bias_part + ((size_t)(z * tiles_m + tm) * slots) * (2 * T2_BM);
      float g = bias_partner;
      if (my_bias) {   // this CTA pair issued bias UMMAs
        uint32_t v[32];
        tmem_ld_32x32(t_row + T2_BN, v);  // columns BN..BN+15 hold the partial row sum (all equal); 32 columns are allocated
        tmem_ld_wait();
        g += __uint_as_float(v[0]);
      }
      part[(size_t)tn * (2 * T2_BM) + r_in_tile] = g;
      __threadfence();
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (quarter == 0 && lane == 0) {
        const unsigned int done = atomicAdd(args.bias_count + z * tiles_m + tm, 1u);
        s_last = (done == 2u * (unsigned int)slots - 1u) ? 1 : 0;   // both CTAs of all column tiles have stored
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (s_last) {
        __threadfence();
        const int t128 = quarter * 32 + lane;
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          const int rt = half * T2_BM + t128;
          float sum = 0.f;
          for (int j = 0; j < slots; ++j) sum += __ldcg(part + (size_t)j * (2 * T2_BM) + rt);
          const int grow = tm * 2 * T2_BM + rt;
          if (grow < args.M) {
            args.bias_grad[(long long)z * args.bias_grad_zstride + grow] = sum;
            bad |= fp16_grad_overflow(sum);
          }
        }
        if (t128 == 0) args.bias_count[z * tiles_m + tm] = 0u;   // ready for the next launch
      }
    }
    }   // pair A / plain pair
    if (args.nonfinite != nullptr) {
      if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(args.nonfinite, 1);
    }
    if (args.dbg && warp == 2 && lane == 0) args.dbg[8 * ((size_t)blockIdx.z * gridDim.x + blockIdx.x) + 4] = clock64() - t_epi;
  }

  __syncwarp();
  tcgen05_fence_before();
  cluster_sync();  // both tensor cores are done with both CTAs' shared memory and TMEM
  if (warp == 1) {
    tcgen05_fence_after();
    tmem_dealloc_pair(tmem_base, kTmemCols);
  }
}

// MN-major operands (the weight gradient's dZ and X), 256-column tiles per CTA pair
template <bool C4>
static int launch2(const CUtensorMap& tmA, const CUtensorMap& tmB, const Gemm2Args& a, int batch, cudaStream_t stream, bool pdl) {
  constexpr auto kern = gemm2cta_kernel<true, true, kGemm2BN, C4>;
  constexpr int T2_SMEM = T2Cfg<kGemm2BN>::kSmem;
  int rc = set_max_dynamic_smem<kern>(T2_SMEM);
  if (rc) return rc;
  constexpr int kCluster = C4 ? 4 : 2;   // CTAs per output tile
  const int tiles_m = (a.M + 2 * T2_BM - 1) / (2 * T2_BM);
  return launch_kernel<kCluster>(kern, dim3(kCluster * tiles_m * a.tiles_n, 1, batch), dim3(T2_THREADS), T2_SMEM, stream, pdl, tmA,
                                 tmB, a);
}

int gemm2_launch(const Gemm2Launch& L, cudaStream_t s, bool pdl) {
  if (L.args.split_k == 2) {   // on-chip split-K 2: cluster of four (two pairs per tile)
    ACEZ_REQUIRE(L.args.k_blocks >= 2, "gemm2cta: split-K 2 needs at least two k-blocks");
    return launch2<true>(L.tmA, L.tmB, L.args, L.batch, s, pdl);
  }
  return launch2<false>(L.tmA, L.tmB, L.args, L.batch, s, pdl);
}

}  // namespace acez
