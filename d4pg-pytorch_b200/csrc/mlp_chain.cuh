// Cluster-fused MLP chains (exact fp32): a whole actor/critic network chain per launch.
#pragma once
#include "gemm_ffma.cuh"
#include "adam.cuh"

namespace d4pg {

constexpr int CHAIN_MAX_SLOTS = 8;     // layers per chain (actor_target -> critic_target is 8)
constexpr int CHAIN_MAX = 3;           // chains per launch (forward: target / critic / policy)
constexpr int CHAIN_CLUSTER = 8;       // CTAs per cluster = 32-column slices of a 256-wide layer
constexpr int CHAIN_ROWS = 32;         // batch rows owned by one cluster
constexpr int CHAIN_PLANE = D4PG_HIDDEN * CHAIN_ROWS;   // floats of one exchange plane [256][32]

// One layer of a chain.  The A operand (activations / deltas of the cluster's 32 rows) comes either
// from a row-major global array (`Ag`, first layer of a chain, replay actions, logit gradients) or
// from the k-major exchange plane written by an earlier slot of the same cluster (`src`); a
// concatenated layer (critic fc2, models.py:80) takes its first K1 rows of K from the first source
// and the rest from the second.
struct ChainSlot {
  const float* W; const float* bias; const float* aux;
  const float* Ag; const float* A2g;
  float* C;                       // row-major output [B][ldc] (nullptr: exchange only)
  int ldw, ldaux, ldag, lda2g, ldc;
  int N, K, K1;
  int src, src2;                  // exchange-plane slot of the first / second A source (-1: global)
  int mode, epi;                  // GEMM_FWD / GEMM_DX, GemmEpi
  int publish;                    // 1: also store the output tile k-major for later slots
  // Optional PRE-LAYER (fp32 path): a layer at most 8 columns wide (actor fc3, the d-action step of the policy
  // backward) that every CTA of the cluster evaluates redundantly at the start of this slot, from plane `pre_src`,
  // into rows [pre_row, pre_row + pre_N) of its own A operand -- instead of a slot of its own (barrier + exchange
  // for a 32 x 6 result).  src2 == -2 (FWD: the pre-layer is the concatenated tail) or src == -2 with a_row0 =
  // pre_row (DX: the pre-layer is the whole A operand).  Rank 0 also stores it row-major to pre_C.
  int has_pre, pre_src, pre_row, a_row0;
  const float* pre_W; const float* pre_bias; const float* pre_aux; float* pre_C;
  int pre_ldw, pre_ldaux, pre_ldc, pre_N, pre_K, pre_epi;
};

struct ChainArgs {
  ChainSlot slot[CHAIN_MAX][CHAIN_MAX_SLOTS];
  int nslots[CHAIN_MAX];
  int nchains, B, row_blocks;
  int precision;                  // 0 exact fp32 FFMA tile, 1 3xTF32 / 2 TF32 mma.sync tile
  int a_floats, w_floats;         // shared memory: resident A plane, one weight-slice buffer (two are kept)
  float* xchg;                    // [nchains][row_blocks][CHAIN_MAX_SLOTS][CHAIN_PLANE]
  unsigned long long* trace;      // optional phase stamps of CTA 0 (D4PG_TC_TRACE), 6 per slot
  int trace_base;                 // first stamp index of this launch in the debug buffer
  unsigned long long* step_trace; int step_slot;
  int trace_cta;                  // which CTA writes the per-slot stamps (env D4PG_TRACE_CTA, default 0)   // step timeline stamp (entry / exit of CTA 0)
};

int64_t chain_xchg_floats(int B);
void chain_args_begin(ChainArgs& a, int B, float* xchg, int precision = 0);   // 0 fp32 FFMA, 1 3xTF32 mma.sync, 2 TF32 mma.sync
// add a slot to chain `c`; returns its slot index
int chain_add(ChainArgs& a, int c, const ChainSlot& s);
ChainSlot chain_fwd(const float* W, int ldw, const float* bias, int N, int K, int epi, float* C, int ldc, int publish);
ChainSlot chain_dx(const float* W, int ldw, int N_in, int K_out, int epi, const float* aux, int ldaux,
                   float* C, int ldc, int publish);
void chain_src_global(ChainSlot& s, const float* Ag, int ldag);
void chain_src_plane(ChainSlot& s, int slot);
void chain_src2_global(ChainSlot& s, int K1, const float* A2g, int lda2g);
void chain_src2_plane(ChainSlot& s, int K1, int slot);
void chain_pre_layer(ChainSlot& s, const float* W, int ldw, const float* bias, const float* aux, int ldaux, int N, int K, int epi,
                     float* C, int ldc, int src_slot, int pre_row, bool whole_operand);
int launch_mlp_chain(ChainArgs& a, cudaStream_t st);

// dW level of the whole step in one launch (up to 12 problems, no TMA descriptors in the parameters)
constexpr int GEMM_WIDE_MAX = 12;
struct GemmWideBatch {
  GemmProblem p[GEMM_WIDE_MAX];
  int n, total_tiles;
  unsigned long long* trace;
  // data parallel over peer memory: the last CTA to finish publishes "this rank's gradient half is complete"
  // ([0] published step count, [1] local step count, [2] CTA ticket), see comm.cu
  PeerSignal peer_sig; int has_peer_sig;
};
void gemm_wide_begin(GemmWideBatch& b, const PeerSignal* sig = nullptr);
void gemm_wide_add(GemmWideBatch& b, const GemmProblem& p);
int gemm_wide_launch(GemmWideBatch& b, cudaStream_t st);

}  // namespace d4pg
