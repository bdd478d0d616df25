// tcgen05 + TMA GEMM for sm_100a. See gemm.cuh for the operand conventions.
//
// One CTA computes one 128 x BN output tile: warp 0 = TMA producer, warp 1 = TMEM owner + single-thread UMMA
// issuer, warps 2..9 = epilogue (TMEM -> registers -> swizzled smem -> TMA store; two groups of four warps, one per
// TMEM lane quarter each, splitting the 64-column boxes). A ring of kStages shared-memory stages is handed
// between producer and issuer with full/empty mbarriers; tcgen05.commit releases stages and publishes the
// accumulator to the epilogue warps.
#include "gemm.cuh"

namespace acez {

static constexpr int BM = 128;
static constexpr int BK = 64;  // 64 fp16 = one 128-byte swizzle row
static constexpr int kThreads = 320;  // warp 0 TMA, warp 1 MMA, warps 2-5 and 6-9: two epilogue groups (2 warps per SMSP)
static constexpr uint32_t kSw128 = 2;

template <int BN, int EPI>
struct GemmCfg {
  static constexpr int kAStage = BM * BK * 2;
  static constexpr int kBStage = BN * BK * 2;
  static constexpr int kStage = kAStage + kBStage;
  // fp16 epilogues reserve one 128 x BN operand tile (residual / ReLU mask, prefetched by TMA during the main loop) and
  // reuse the pipeline stages as staging for the TMA stores of up to two output tiles
  static constexpr int kOpBytes = (EPI == EPI_WGRAD) ? 0 : BM * BN * 2;
  static constexpr int kStages = (EPI == EPI_WGRAD) ? (BN >= 256 ? 4 : 6) : ((BN >= 256) ? 3 : (BN >= 128 ? 4 : 6));
  static constexpr int kOnesBytes = 16 * BK * 2;  // 16 x 64 tile of 1.0 for the bias-gradient column
  static constexpr int kSmem =
      kStages * kStage + kOpBytes + kOnesBytes + BN * 4 /*bias*/ + 256 /*barriers*/ + 1024 /*align*/;
  static_assert(EPI == EPI_WGRAD || kStages * kStage >= 2 * BM * BN * 2, "stage memory must hold two output tiles");
};

template <int BN, bool A_MN, bool B_MN, int EPI>
__global__ void __launch_bounds__(kThreads, 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                    const __grid_constant__ CUtensorMap tmOut, const __grid_constant__ CUtensorMap tmOut2,
                    const __grid_constant__ CUtensorMap tmOp, const GemmArgs args) {
  using Cfg = GemmCfg<BN, EPI>;
  constexpr int kStages = Cfg::kStages;
  constexpr bool kBiasCol = (EPI == EPI_WGRAD);
  constexpr uint32_t kTmemCols = kBiasCol ? (BN >= 256 ? 512 : 2 * BN) : (BN < 32 ? 32 : BN);
  static_assert(!(kBiasCol && BN > 256), "tmem");

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;
  uint8_t* sB = smem + kStages * Cfg::kAStage;
  uint8_t* sOp = smem + kStages * Cfg::kStage;
  uint8_t* sOnes = sOp + Cfg::kOpBytes;
  float* sBias = reinterpret_cast<float*>(sOnes + Cfg::kOnesBytes);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(sBias + BN);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* tmem_full_bar = empty_bar + kStages;
  uint64_t* op_bar = tmem_full_bar + 1;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(op_bar + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  long long* dbg = args.dbg_clock
                       ? args.dbg_clock + 8 * ((size_t)(blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x)
                       : nullptr;
  if (dbg && threadIdx.x == 0) dbg[0] = clock64();
  const int n0 = blockIdx.x * BN;
  const int m0 = blockIdx.y * BM;
  const int z = blockIdx.z;
  const int k_blocks = args.k_blocks;
  // implicit-GEMM tile coordinates (conv front end)
  int c_tx = 0, c_ty = 0, c_img = 0;
  if (args.conv.enabled) {
    const ConvGeom& cg = args.conv;
    const int tile = blockIdx.y;
    c_tx = tile % cg.tiles_x; c_ty = (tile / cg.tiles_x) % cg.tiles_y; c_img = tile / (cg.tiles_x * cg.tiles_y);
  }

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (EPI != EPI_WGRAD) {
      if (args.st_out) tma_prefetch_desc(&tmOut);
      if (args.st_out2) tma_prefetch_desc(&tmOut2);
      if (args.ld_op) tma_prefetch_desc(&tmOp);
    }
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(tmem_full_bar, 1);
    mbar_init(op_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_ptr, kTmemCols);
  if (kBiasCol && warp >= 2) {
    // ones tile: layout irrelevant (all entries equal)
    __half2* o = reinterpret_cast<__half2*>(sOnes);
    for (int i = threadIdx.x - 64; i < Cfg::kOnesBytes / 4; i += 256) o[i] = __floats2half2_rn(1.f, 1.f);
    fence_proxy_async();  // generic-proxy writes -> visible to the tensor core (async proxy)
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr;
  if (dbg && threadIdx.x == 0) dbg[1] = clock64();
  // Programmatic dependent launch: everything above (barrier init, TMEM allocation, descriptor prefetch) overlaps the
  // tail of the previous kernel in the stream; global memory is only touched after the dependency has resolved.
  pdl_wait();
  pdl_launch_dependents();
  if (dbg && threadIdx.x == 0) dbg[2] = clock64();

  if (warp == 0) {
    // ------------------------------ TMA producer ------------------------------
    if (elect_one()) {
      if (EPI != EPI_WGRAD && args.ld_op) {
        // epilogue operand tile (residual / ReLU mask): lands while the main loop runs
        mbar_arrive_expect_tx(op_bar, BM * BN * 2);
#pragma unroll
        for (int b = 0; b < BN / 64; ++b) {
          if (args.conv.enabled)
            tma_load_4d(sOp + b * 16384, &tmOp, op_bar, n0 + 64 * b, c_tx * kConvTileW, c_ty * kConvTileH, c_img);
          else
            tma_load_3d(sOp + b * 16384, &tmOp, op_bar, n0 + 64 * b, m0, 0);
        }
      }
      int stage = 0;
      uint32_t phase = 0;
      for (int kb = 0; kb < k_blocks; ++kb) {
        mbar_wait(&empty_bar[stage], phase ^ 1);
        mbar_arrive_expect_tx(&full_bar[stage], Cfg::kStage);
        uint8_t* a_dst = sA + stage * Cfg::kAStage;
        uint8_t* b_dst = sB + stage * Cfg::kBStage;
        if (A_MN) {
#pragma unroll
          for (int i = 0; i < BM / 64; ++i) tma_load_3d(a_dst + i * 8192, &tmA, &full_bar[stage], m0 + 64 * i, kb * BK, z);
        } else if (args.conv.enabled) {
          // implicit GEMM: k-block = (filter tap, 64-channel chunk); one 4-D box = 16 x 8 pixels x 64 channels
          const ConvGeom& cg = args.conv;
          const int tap = kb / cg.cin_blocks, cb = kb - tap * cg.cin_blocks;
          const int ky = tap / cg.ksize, kx = tap - ky * cg.ksize;
          tma_load_4d(a_dst, &tmA, &full_bar[stage], cb * 64, c_tx * kConvTileW * cg.stride + kx - cg.pad,
                      c_ty * kConvTileH * cg.stride + ky - cg.pad, c_img);
        } else {
          tma_load_3d(a_dst, &tmA, &full_bar[stage], kb * BK, m0, z);
        }
        if (B_MN) {
#pragma unroll
          for (int i = 0; i < BN / 64; ++i) tma_load_3d(b_dst + i * 8192, &tmB, &full_bar[stage], n0 + 64 * i, kb * BK, z);
        } else {
          tma_load_3d(b_dst, &tmB, &full_bar[stage], kb * BK, n0, z);
        }
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ------------------------------ UMMA issuer ------------------------------
    constexpr uint32_t idesc = make_idesc_f16(BM, BN, A_MN, B_MN);
    constexpr uint32_t idesc_ones = make_idesc_f16(BM, 16, A_MN, false);
    int stage = 0;
    uint32_t phase = 0;
    for (int kb = 0; kb < k_blocks; ++kb) {
      mbar_wait(&full_bar[stage], phase);
      tcgen05_fence_after();
      if (dbg && kb == 0 && lane == 0) dbg[3] = clock64();
      if (elect_one()) {
        const uint32_t a_addr = smem_u32(sA + stage * Cfg::kAStage);
        const uint32_t b_addr = smem_u32(sB + stage * Cfg::kBStage);
#pragma unroll
        for (int k = 0; k < BK / 16; ++k) {
          const uint64_t da = make_smem_desc(a_addr + k * args.a_kstep, args.a_lbo, args.a_sbo, kSw128);
          const uint64_t db = make_smem_desc(b_addr + k * args.b_kstep, args.b_lbo, args.b_sbo, kSw128);
          umma_f16(tmem_base, da, db, idesc, (kb | k) != 0 ? 1u : 0u);
          if (kBiasCol && n0 == 0 && args.bias_grad != nullptr) {
            const uint64_t d1 = make_smem_desc(smem_u32(sOnes) + k * 32, 0, 1024, kSw128);
            umma_f16(tmem_base + BN, da, d1, idesc_ones, (kb | k) != 0 ? 1u : 0u);
          }
        }
      }
      __syncwarp();
      if (elect_one()) {
        tcgen05_commit(&empty_bar[stage]);                     // stage free once the MMAs above retire
        if (kb == k_blocks - 1) tcgen05_commit(tmem_full_bar);  // accumulator complete
      }
      __syncwarp();
      if (++stage == kStages) { stage = 0; phase ^= 1; }
    }
    if (dbg && lane == 0) dbg[4] = clock64();
  } else {
    // ------------------------------ epilogue (4 warps <-> 4 TMEM lane quarters) ------------------------------
    const int quarter = warp & 3;
    const int grp = (warp - 2) >> 2;     // epilogue group 0 / 1: boxes (chunks) are interleaved between the groups
    const int r = quarter * 32 + lane;  // row inside the tile
    int row = m0 + r;
    bool row_ok = row < args.M;
    if (args.conv.enabled) {
      const ConvGeom& cg = args.conv;
      const int py = c_ty * kConvTileH + r / kConvTileW, px = c_tx * kConvTileW + r % kConvTileW;
      row_ok = (py < cg.Ho) && (px < cg.Wo);
      row = (c_img * cg.Ho + py) * cg.Wo + px;  // NHWC pixel index
    }
    if (EPI == EPI_FWD) {
      for (int i = threadIdx.x - 64; i < BN; i += 256) {
        const int n = n0 + i;
        // autocast casts the fp32 bias to fp16 before the conv adds it
        sBias[i] = (args.bias != nullptr && n < args.N) ? __half2float(__float2half_rn(__ldcg(args.bias + n))) : 0.f;
      }
      asm volatile("bar.sync 3, 256;" ::: "memory");  // all epilogue warps
    }
    if (EPI != EPI_WGRAD && args.ld_op) mbar_wait(op_bar, 0);
    mbar_wait(tmem_full_bar, 0);
    tcgen05_fence_after();
    if (dbg && threadIdx.x == 64) dbg[5] = clock64();
    const bool issuer = (lane == 0) && (quarter == 2 - 2 * grp);  // first warp of the group: warp 2 / warp 6
    const uint32_t t_row = tmem_base + ((uint32_t)(quarter * 32) << 16);
    // all pipeline stages are drained by now: their memory stages the output tiles for the TMA stores
    uint8_t* sOut = smem;
    uint8_t* sOut2 = smem + BM * BN * 2;
    const uint32_t sOut_u32 = smem_u32(sOut), sOut2_u32 = smem_u32(sOut2), sOp_u32 = smem_u32(sOp), sBias_u32 = smem_u32(sBias);
    const uint32_t swz = (uint32_t)(r & 7);
    bool bad = false;
    if (EPI == EPI_WGRAD) {
#pragma unroll 1
      for (int c = grp; c < BN / 32; c += 2) {
        uint32_t v[32];
        tmem_ld_32x32(t_row + c * 32, v);
        tmem_ld_wait();
        const int ncol = n0 + c * 32;
        if (!row_ok || ncol >= args.N) continue;
        float4* dst = reinterpret_cast<float4*>(args.out32 + (long long)z * args.out32_zstride +
                                                (long long)row * args.ldo32 + ncol);
#pragma unroll
        for (int j = 0; j < 8; ++j)
          dst[j] = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                               __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
        if (args.nonfinite != nullptr) {  // GradScaler check folded in
#pragma unroll
          for (int j = 0; j < 32; ++j) bad |= fp16_grad_overflow(__uint_as_float(v[j]));
        }
      }
    } else {
      uint32_t badbits = 0;
      const bool has_add = (EPI == EPI_DGRAD) && args.addend != nullptr;
#pragma unroll 1
      for (int box = grp; box < BN / 64; box += 2) {
        // one 64-column box per iteration: a single TMEM load, 8 swizzled 16-byte chunks per tile row
        uint32_t v[64];
        tmem_ld_32x64(t_row + box * 64, v);
        tmem_ld_wait();
        const uint32_t row_off = (uint32_t)box * 16384u + (uint32_t)r * 128u;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const uint32_t off = row_off + ((((uint32_t)q) ^ swz) << 4);
          uint4 opv = make_uint4(0, 0, 0, 0);
          if (args.ld_op) opv = lds_128(sOp_u32 + off);   // explicit shared-space access (a generic pointer compiles to LD.E / ST.E)
          const __half2* ph = reinterpret_cast<const __half2*>(&opv);
          uint4 o, o2;
          __half2* oh = reinterpret_cast<__half2*>(&o);
          __half2* o2h = reinterpret_cast<__half2*>(&o2);
          if (EPI == EPI_FWD) {
            const float4 bf0 = lds_128f(sBias_u32 + 4u * (uint32_t)(box * 64 + q * 8));
            const float4 bf1 = lds_128f(sBias_u32 + 4u * (uint32_t)(box * 64 + q * 8 + 4));
            const float bq[8] = {bf0.x, bf0.y, bf0.z, bf0.w, bf1.x, bf1.y, bf1.z, bf1.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int col = q * 8 + 2 * j;
              float a = __uint_as_float(v[col]) + bq[2 * j];
              float b = __uint_as_float(v[col + 1]) + bq[2 * j + 1];
              if (args.relu) { a = fmaxf(a, 0.f); b = fmaxf(b, 0.f); }
              const __half2 h = __floats2half2_rn(a, b);
              oh[j] = h;
              o2h[j] = __hadd2(ph[j], h);  // residual sum in fp16, as the reference's `res + x`
            }
          } else {  // EPI_DGRAD
            uint4 ad = make_uint4(0, 0, 0, 0);
            if (has_add && row_ok) {  // L2 load: the kernel may have been launched early (PDL)
              ad = __ldcg(reinterpret_cast<const uint4*>(args.addend + (long long)row * args.ldo + n0 + box * 64 + q * 8));
            }
            const __half2* ah = reinterpret_cast<const __half2*>(&ad);
            const __half2 zero2 = __floats2half2_rn(0.f, 0.f);
            uint32_t* ob = reinterpret_cast<uint32_t*>(&o);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int col = q * 8 + 2 * j;
              // autograd: the conv-backward result is rounded to fp16 first, the skip gradient is added in fp16
              __half2 h = __floats2half2_rn(__uint_as_float(v[col]), __uint_as_float(v[col + 1]));
              if (has_add) h = __hadd2(h, ah[j]);
              o2h[j] = h;
              const uint32_t hb = *reinterpret_cast<const uint32_t*>(&h);
              badbits |= ((hb & 0x7C007C00u) + 0x04000400u) & 0x80008000u;  // exponent all ones: inf / nan
              ob[j] = hb & __hgt2_mask(ph[j], zero2);                       // ReLU mask from the saved activation
            }
          }
          if (args.st_out) sts_128(sOut_u32 + off, o);
          if (args.st_out2) sts_128(sOut2_u32 + off, o2);
        }
        // the box is complete in shared memory: hand it to the TMA store engine
        fence_proxy_async();
        if (grp == 0) asm volatile("bar.sync 1, 128;" ::: "memory");
        else asm volatile("bar.sync 2, 128;" ::: "memory");
        if (issuer) {
          if (args.conv.enabled) {
            if (args.st_out) tma_store_4d(&tmOut, sOut + box * 16384, n0 + 64 * box, c_tx * kConvTileW, c_ty * kConvTileH, c_img);
            if (args.st_out2) tma_store_4d(&tmOut2, sOut2 + box * 16384, n0 + 64 * box, c_tx * kConvTileW, c_ty * kConvTileH, c_img);
          } else {
            if (args.st_out) tma_store_3d(&tmOut, sOut + box * 16384, n0 + 64 * box, m0, 0);
            if (args.st_out2) tma_store_3d(&tmOut2, sOut2 + box * 16384, n0 + 64 * box, m0, 0);
          }
          tma_store_commit();
        }
      }
      bad = badbits != 0;
    }
    if (EPI != EPI_WGRAD && issuer) tma_store_wait_all();
    if (kBiasCol && grp == 0 && n0 == 0 && args.bias_grad != nullptr) {
      uint32_t v[32];
      tmem_ld_32x32(t_row + BN, v);
      tmem_ld_wait();
      if (row_ok) {
        const float g = __uint_as_float(v[0]);
        args.bias_grad[(long long)z * args.bias_grad_zstride + row] = g;
        bad |= fp16_grad_overflow(g);
      }
    }
    if (EPI != EPI_FWD && args.nonfinite != nullptr) {
      if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(args.nonfinite, 1);
    }
    if (dbg && threadIdx.x == 64) dbg[6] = clock64();
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
  if (dbg && threadIdx.x == 0) dbg[7] = clock64();
}

// ----------------------------------------------------------------------------------------------
// host side
// ----------------------------------------------------------------------------------------------
static int encode_operand(CUtensorMap* tm, const __half* base, int mn_major, int rows_mn, int K, int ld, int batch,
                          long long zstride, int tile_mn) {
  // K-major : memory [batch][rows_mn][ld], inner = K,       box {64, tile_mn, 1}
  // MN-major: memory [batch][K][ld],       inner = rows_mn, box {64, 64, 1}
  uint64_t dims[3];
  uint64_t strides[2];
  uint32_t box[3];
  if (!mn_major) {
    dims[0] = (uint64_t)K; dims[1] = (uint64_t)rows_mn; dims[2] = (uint64_t)batch;
    box[0] = 64; box[1] = (uint32_t)tile_mn; box[2] = 1;
  } else {
    dims[0] = (uint64_t)rows_mn; dims[1] = (uint64_t)K; dims[2] = (uint64_t)batch;
    box[0] = 64; box[1] = 64; box[2] = 1;
  }
  strides[0] = (uint64_t)ld * 2;
  strides[1] = (uint64_t)(batch > 1 ? zstride : (long long)dims[1] * ld) * 2;
  return make_tensor_map(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, base, dims, strides, box, nullptr,
                         CU_TENSOR_MAP_SWIZZLE_128B);
}

int gemm_prepare(GemmLaunch* L, const GemmProblem& p) {
  ACEZ_REQUIRE(p.M > 0 && p.N > 0 && p.K > 0 && p.batch >= 1, "gemm: bad shape %d %d %d x%d", p.M, p.N, p.K, p.batch);
  ACEZ_REQUIRE(p.K % BK == 0, "gemm: K=%d must be a multiple of %d", p.K, BK);
  ACEZ_REQUIRE(p.lda % 8 == 0 && p.ldb % 8 == 0, "gemm: leading dimensions must be multiples of 8 elements");
  int bn = p.bn;
  if (bn == 0) bn = (p.N % 256 == 0 && p.epi != EPI_WGRAD) ? 256 : (p.N % 128 == 0 ? 128 : 64);
  ACEZ_REQUIRE(bn == 64 || bn == 128 || bn == 256, "gemm: unsupported BN=%d", bn);
  ACEZ_REQUIRE(p.N % 32 == 0, "gemm: N=%d must be a multiple of 32", p.N);
  L->bn = bn;
  L->a_mn = p.a_mn;
  L->b_mn = p.b_mn;
  L->epi = p.epi;
  L->batch = p.batch;
  GemmArgs a{};
  a.M = p.M;
  a.N = p.N;
  a.k_blocks = p.K / BK;
  // K-major, SWIZZLE_128B: 8-row groups 1024 B apart, k-step of 16 elements = 32 B inside the swizzle row.
  // MN-major, SWIZZLE_128B: 64-element MN atoms 64 rows * 128 B = 8192 B apart (LBO), 8-row K groups 1024 B apart
  // (SBO), k-step of 16 rows = 2048 B.
  a.a_lbo = p.a_mn ? 8192 : 0; a.a_sbo = 1024; a.a_kstep = p.a_mn ? 2048 : 32;
  a.b_lbo = p.b_mn ? 8192 : 0; a.b_sbo = 1024; a.b_kstep = p.b_mn ? 2048 : 32;
  L->args = a;
  int rc = encode_operand(&L->tmA, p.A, p.a_mn, p.M, p.K, p.lda, p.batch, p.a_zstride, BM);
  if (rc) return rc;
  return encode_operand(&L->tmB, p.B, p.b_mn, p.N, p.K, p.ldb, p.batch, p.b_zstride, bn);
}

// Tensor maps of the fp16 epilogue: out / out2 (TMA stores from the staged tile) and the prefetched operand tile
// (residual for EPI_FWD, ReLU mask for EPI_DGRAD). All are [rows, ldo] row-major fp16 with the output's geometry.
static int encode_tile_map(CUtensorMap* tm, const void* base, const GemmArgs& a, int batch_images) {
  if (a.conv.enabled) {
    uint64_t dims[4] = {(uint64_t)a.N, (uint64_t)a.conv.Wo, (uint64_t)a.conv.Ho, (uint64_t)batch_images};
    uint64_t strides[3] = {(uint64_t)a.ldo * 2, (uint64_t)a.conv.Wo * a.ldo * 2, (uint64_t)a.conv.Ho * a.conv.Wo * a.ldo * 2};
    uint32_t box[4] = {64, (uint32_t)kConvTileW, (uint32_t)kConvTileH, 1};
    return make_tensor_map(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, base, dims, strides, box, nullptr,
                           CU_TENSOR_MAP_SWIZZLE_128B);
  }
  uint64_t dims[3] = {(uint64_t)a.N, (uint64_t)a.M, 1};
  uint64_t strides[2] = {(uint64_t)a.ldo * 2, (uint64_t)a.M * a.ldo * 2};
  uint32_t box[3] = {64, (uint32_t)BM, 1};
  return make_tensor_map(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, base, dims, strides, box, nullptr,
                         CU_TENSOR_MAP_SWIZZLE_128B);
}

int gemm_finalize(GemmLaunch* L) {
  GemmArgs& a = L->args;
  a.st_out = a.st_out2 = a.ld_op = 0;
  if (L->epi == EPI_WGRAD) return ACEZ_OK;
  ACEZ_REQUIRE(a.N % 64 == 0 && a.ldo % 8 == 0, "gemm: fp16 epilogue needs N %% 64 == 0 and ldo %% 8 == 0 (N=%d ldo=%d)", a.N, a.ldo);
  const int imgs = a.conv.enabled ? L->batch : 1;
  int rc;
  const __half* op = (L->epi == EPI_FWD) ? a.resid : a.mask;
  if (a.out != nullptr) {
    if ((rc = encode_tile_map(&L->tmOut, a.out, a, imgs))) return rc;
    a.st_out = 1;
  }
  const bool want2 = a.out2 != nullptr && (L->epi == EPI_DGRAD || a.resid != nullptr);
  if (want2) {
    if ((rc = encode_tile_map(&L->tmOut2, a.out2, a, imgs))) return rc;
    a.st_out2 = 1;
  }
  if (op != nullptr) {
    if ((rc = encode_tile_map(&L->tmOp, op, a, imgs))) return rc;
    a.ld_op = 1;
  }
  ACEZ_REQUIRE(L->epi != EPI_DGRAD || a.ld_op, "gemm: dgrad epilogue needs a mask");
  // unused maps must still be valid kernel parameters
  if (!a.st_out) L->tmOut = a.st_out2 ? L->tmOut2 : L->tmA;
  if (!a.st_out2) L->tmOut2 = L->tmOut;
  if (!a.ld_op) L->tmOp = L->tmOut;
  return ACEZ_OK;
}

template <int BN, bool A_MN, bool B_MN, int EPI>
static int launch_variant(const GemmLaunch& L, cudaStream_t stream, bool pdl) {
  constexpr auto kern = gemm_tcgen05_kernel<BN, A_MN, B_MN, EPI>;
  int rc = set_max_dynamic_smem<kern>(GemmCfg<BN, EPI>::kSmem);
  if (rc) return rc;
  dim3 grid((L.args.N + BN - 1) / BN, (L.args.M + BM - 1) / BM, L.batch);
  if (L.args.conv.enabled) grid.y = L.args.conv.tiles_x * L.args.conv.tiles_y * L.batch, grid.z = 1;
  return launch_kernel(kern, grid, dim3(kThreads), GemmCfg<BN, EPI>::kSmem, stream, pdl, L.tmA, L.tmB, L.tmOut, L.tmOut2, L.tmOp,
                       L.args);
}

int gemm_launch(const GemmLaunch& L, cudaStream_t stream, bool pdl) {
#define ACEZ_GEMM_CASE(BN_, AMN_, BMN_, EPI_) \
  if (L.bn == BN_ && L.a_mn == AMN_ && L.b_mn == BMN_ && L.epi == EPI_) return launch_variant<BN_, AMN_, BMN_, EPI_>(L, stream, pdl);
  ACEZ_GEMM_CASE(256, false, false, EPI_FWD)
  ACEZ_GEMM_CASE(128, false, false, EPI_FWD)
  ACEZ_GEMM_CASE(64, false, false, EPI_FWD)
  ACEZ_GEMM_CASE(256, false, true, EPI_DGRAD)
  ACEZ_GEMM_CASE(128, false, true, EPI_DGRAD)
  ACEZ_GEMM_CASE(128, true, true, EPI_WGRAD)
  ACEZ_GEMM_CASE(256, true, true, EPI_WGRAD)
  // generic fp32-output variants (tests / probing of operand layouts)
  ACEZ_GEMM_CASE(128, false, false, EPI_WGRAD)
  ACEZ_GEMM_CASE(128, false, true, EPI_WGRAD)
  ACEZ_GEMM_CASE(128, true, false, EPI_WGRAD)
#undef ACEZ_GEMM_CASE
  set_error("gemm: no kernel variant for bn=%d a_mn=%d b_mn=%d epi=%d", L.bn, L.a_mn, L.b_mn, L.epi);
  return ACEZ_ERR_UNSUPPORTED;
}

}  // namespace acez

// ----------------------------------------------------------------------------------------------
// C ABI: generic GEMM entry (tests, probing)
// ----------------------------------------------------------------------------------------------

extern "C" int acez_gemm_f16(const acez_gemm_desc* d, acez_stream_t stream) {
  using namespace acez;
  ACEZ_REQUIRE(d != nullptr, "gemm: null desc");
  int rc = acez_device_check();
  if (rc) return rc;
  GemmProblem p{};
  p.A = reinterpret_cast<const __half*>(d->A);
  p.B = reinterpret_cast<const __half*>(d->B);
  p.a_mn = d->a_mn_major;
  p.b_mn = d->b_mn_major;
  p.M = d->M; p.N = d->N; p.K = d->K;
  p.batch = d->batch > 0 ? d->batch : 1;
  p.a_zstride = d->a_zstride; p.b_zstride = d->b_zstride;
  p.lda = d->lda; p.ldb = d->ldb;
  p.bn = d->bn;
  p.epi = d->epilogue;
  GemmLaunch L;
  rc = gemm_prepare(&L, p);
  if (rc) return rc;
  GemmArgs& a = L.args;
  a.bias = d->bias;
  a.resid = reinterpret_cast<const __half*>(d->resid);
  a.mask = reinterpret_cast<const __half*>(d->mask);
  a.addend = reinterpret_cast<const __half*>(d->addend);
  a.out = reinterpret_cast<__half*>(d->out);
  a.out2 = reinterpret_cast<__half*>(d->out2);
  a.ldo = d->ldo;
  a.relu = d->relu;
  a.nonfinite = d->nonfinite;
  a.out32 = d->out32;
  a.out32_zstride = d->out32_zstride;
  a.ldo32 = d->ldo32;
  a.bias_grad = d->bias_grad;
  a.bias_grad_zstride = d->bias_grad_zstride;
  a.dbg_clock = reinterpret_cast<long long*>(d->dbg_clock);
  if (d->a_lbo) a.a_lbo = d->a_lbo;
  if (d->a_sbo) a.a_sbo = d->a_sbo;
  if (d->a_kstep) a.a_kstep = d->a_kstep;
  if (d->b_lbo) a.b_lbo = d->b_lbo;
  if (d->b_sbo) a.b_sbo = d->b_sbo;
  if (d->b_kstep) a.b_kstep = d->b_kstep;
  if (d->epilogue == ACEZ_EPI_F32) {
    ACEZ_REQUIRE(d->out32 != nullptr && d->ldo32 % 4 == 0, "gemm: fp32 epilogue needs out32 with ldo32 %% 4 == 0");
  } else {
    ACEZ_REQUIRE((d->out != nullptr || d->out2 != nullptr) && d->ldo % 8 == 0, "gemm: fp16 epilogue needs out with ldo %% 8 == 0");
    ACEZ_REQUIRE(d->epilogue != ACEZ_EPI_DGRAD || d->mask != nullptr, "gemm: dgrad epilogue needs a mask");
  }
  rc = gemm_finalize(&L);
  if (rc) return rc;
  return gemm_launch(L, reinterpret_cast<cudaStream_t>(stream), /*pdl=*/false);
}
