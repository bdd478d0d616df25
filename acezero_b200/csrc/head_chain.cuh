// Fused layer chain of the ACE head (reference ace_network.py:120-136 forward; its autograd transpose for the dgrad
// pass): ALL hidden 512x512 layers of one pass in ONE kernel launch.
//
// The per-layer GEMMs (gemm.cu) are row-tile independent: output rows [m0, m0+128) of layer l+1 depend only on the
// same rows of layer l. So a 128-row tile never has to leave the chip between layers. A thread-block cluster of FOUR CTAs
// owns two row tiles; the SM pair of a channel half computes output channels [256c, 256c+256) of every layer for both
// tiles with tcgen05.mma.cta_group::2 (M = 256, N = 256; accumulators double-buffered in TMEM) and the CTAs of a row tile
// exchange their halves of the new activation tile through distributed shared memory (cp.async.bulk shared::cta ->
// shared::cluster, completing on the partner's mbarrier), 64-column box by box, so the next layer's MMAs start while the
// epilogue of the current one is still draining. Weights stream from L2 through a TMA ring that runs ahead across layer
// boundaries. Every new activation tile is also written to HBM (TMA store) because the weight-gradient GEMM contracts over
// ALL rows and stays a separate kernel. Kernel and host side: head_chain4.cu.
#pragma once
#include "common.cuh"

namespace acez {

enum ChainMode : int { CHAIN_FWD = 0, CHAIN_DGRAD = 1 };
// A barrier wait of the chain kernels that lasts longer than this is reported (tag of the wait, step, index) and trapped
// instead of hanging the GPU: ~10 s at 1.9 GHz, far above any legitimate stall (profiler replay, time slicing, throttling);
// the clock is only read on the slow path, after a first failed try_wait.
static constexpr long long kChainWatchdogCycles = 20000000000ll;
static constexpr int kChainMaxSteps = 20;      // hidden layers handled by one launch (3 * res blocks + 2 <= 20)
static constexpr int kChainFlagResInit = 64;    // ChainArgs.flags: FWD has residual layers, res_0 = the input tile
static constexpr int kChainFlagOwnFirst = 256;  // ChainArgs.flags: consume the own boxes' k-blocks first (default;
                                                // ACEZ_CHAIN_ORDER=arrival clears it: they are consumed as they arrive)

// One GEMM of the chain, in execution order.
struct ChainStep {
  int w_layer;             // index into W16 [L][512][512]
  int out_slot;            // z index in the output tensor map the new tile is stored to; < 0: not stored
  int relu;                // FWD
  int res_add;             // FWD: residual-closing layer, tile = res + x and res = tile (ace_network.py:126,133)
                           // DGRAD: add the skip-path gradient before masking
  int res_save;            // DGRAD: keep the unmasked sum as the skip-path gradient for the block below
  const float* bias;       // FWD: fp32 master bias [512] (rounded to fp16 before the add, autocast semantics)
  uint8_t* mask_out;       // FWD: [rows][64 B] one bit per channel, (pre-residual x > 0): the ReLU mask of the backward (nullable)
  const uint8_t* mask_in;  // DGRAD: the bit mask of the activation the gradient flows into
};

static constexpr int kChainDbgSlots = 8 + 8 * kChainMaxSteps;  // clock64 stamps per CTA (profiling probe)

struct ChainArgs {
  int rows;
  int n_steps;
  int flags;       // kChainFlagResInit | kChainFlagOwnFirst
  int* nonfinite;  // DGRAD: OR-ed with 1 if a stored gradient is inf / nan (nullable)
  long long* dbg;  // nullable: [gridDim.x][kChainDbgSlots] clock64 stamps (ACEZ_CHAIN_DBG=1, tools/probe_chain_time.py)
  ChainStep step[kChainMaxSteps];
};

struct ChainLaunch {
  CUtensorMap tmIn;   // first A tile: [rows, 512], box {64, 128, 1}
  CUtensorMap tmW;    // W16 [L][512][512], half a k-block per CTA of a pair: FWD box {64, 128, 1} (K-major B), DGRAD box
                      // {64, 64, 1} (MN-major B, two boxes per half)
  CUtensorMap tmOut;  // [slots][rows][512], box {64, 128, 1}
  ChainArgs args;
  int mode;
};

// in: the first A operand [rows,512]; out_base/out_zstride(elements)/out_slots: where new tiles are stored.
int chain_prepare(ChainLaunch* C, int mode, const __half* in, const __half* W16, int L, __half* out_base,
                  long long out_zstride, int out_slots, int rows);
// pdl: launch with the programmatic-dependent-launch attribute (only when the stream predecessor is a kernel)
int chain_launch(const ChainLaunch& C, cudaStream_t stream, bool pdl = false);
// profiling probe: copies the stamps of the most recent launch with ACEZ_CHAIN_DBG=1 to host memory
int chain_debug_read(long long* host_out, size_t max_slots, int* n_ctas);

}  // namespace acez
