// cta_group::2 GEMM (gemm2cta.cu): launch descriptor of the batched weight gradient that head.cu runs after the fused dgrad chain.
#pragma once
#include "gemm.cuh"

namespace acez {

struct Gemm2Args {
  int M, N, k_blocks;
  int tiles_n;           // column tiles (bn wide) per row of tiles
  float* out32;          // [z][M][ldo32]
  long long out32_zstride;
  int ldo32;
  float* bias_grad;      // [z][M] nullable: column sum over the contraction dimension of A
  long long bias_grad_zstride;
  float* bias_part;      // with bias_grad: workspace [z][tiles_m][tiles_n][256] partial column sums (one per column tile)
  unsigned int* bias_count;  // with bias_grad: [z][tiles_m] self-resetting arrival counters (zero before the first launch)
  int* nonfinite;        // nullable: OR-ed with 1 if a stored value is non-finite or exceeds the fp16 range
  uint32_t a_lbo, a_sbo, a_kstep, b_lbo, b_sbo, b_kstep;
  int split_k;           // 1, or 2 (256-column tiles only): a cluster of four CTAs = two pairs per tile, each contracting half of the
                         // k-blocks; the second pair's accumulator travels to the first through distributed shared memory
  long long* dbg;        // nullable (no caller sets it): per CTA [0] MMA-warp cycles waiting for operands, [1] MMA loop cycles,
                         // [2] producer cycles waiting for free stages, [3] producer loop cycles, [4] epilogue cycles
};

static constexpr int kGemm2BN = 256;  // columns per CTA pair

struct Gemm2Launch {
  CUtensorMap tmA, tmB;  // MN-major operands [z][K][M] / [z][K][N], 64 x 64 boxes
  Gemm2Args args;
  int batch;
};

// pdl: programmatic dependent launch (only when the stream predecessor is a kernel)
int gemm2_launch(const Gemm2Launch& L, cudaStream_t stream, bool pdl = false);

}  // namespace acez
