// tcgen05 cluster chains: a whole actor/critic network chain per launch with every layer on the 5th-generation
// tensor cores (models.py:32-41,76-88 forward; autograd of ddpg.py:230,242 backward).  See mlp_tc_chain.cu.
#pragma once
#include "gemm_ffma.cuh"

namespace d4pg {

constexpr int TCC_ROWS = 64;          // batch rows owned by one cluster (= UMMA M)
constexpr int TCC_CLUSTER = 8;        // CTAs per cluster: CTA r owns output features [32r, 32r+32) of a layer
constexpr int TCC_BN = 32;            // UMMA N of one group
constexpr int TCC_KC = 32;            // k per chunk (one 128-B SWIZZLE_128B row of tf32)
constexpr int TCC_ABUFS = 9;          // A-chunk buffers per CTA: 0..7 one per K chunk of a 256-wide plane, 8 = the resident / tail chunk
constexpr int TCC_MAX_SLOTS = 8, TCC_MAX_CHAINS = 3, TCC_MAX_GROUPS = 2, TCC_MAX_CHUNKS = 9, TCC_PLANES = 8;
constexpr uint32_t TCC_A_HALF = TCC_ROWS * 128, TCC_A_CHUNK = 2 * TCC_A_HALF;      // hi image then lo image
constexpr uint32_t TCC_W_HALF = TCC_BN * 128, TCC_W_CHUNK = 2 * TCC_W_HALF;
constexpr uint32_t TCC_PLANE_BYTES = TCC_CLUSTER * TCC_A_CHUNK;                    // one published layer output
constexpr int TCC_THREADS = 320;      // warp 0 loader, warp 1 MMA issuer / TMEM owner, warps 2..9 epilogue

enum { TCC_SRC_IMG = 0, TCC_SRC_X = 1, TCC_SRC_PRE = 2 };

// One output of a slot: a 32-column slice per CTA of `N` output features.
struct TccGroup {
  const uint8_t* wimg;            // packed weight images [slices][nchunks][TCC_W_CHUNK] (tcc_pack_kernel)
  const float* bias;              // forward epilogues
  const float* aux; int ldaux;    // backward masks: row-major forward activations
  float* C; int ldc;              // row-major fp32 output (nullptr: exchange only)
  int N, epi, kchunks;           // kchunks: K chunks of the weight image (= the slot's A chunk count)
  int pub;                        // plane the output is published to for later slots (-1: none)
};
struct TccChunk { short kind, plane, chunk, buf; };      // buf: A buffer the chunk occupies (assigned at launch)
// one bulk copy: `count` consecutive chunks of a plane into consecutive A buffers, completion on full[buf0]
struct TccLoad { short plane, chunk0, buf0, count; };
// One layer slot: every group contracts the same A operand (the chunk list) with its own weights.
struct TccSlot {
  TccGroup g[TCC_MAX_GROUPS];
  TccChunk ch[TCC_MAX_CHUNKS];
  TccLoad ld[TCC_MAX_CHUNKS];
  int ngroups, nchunks, nloads;
  int nacc;                              // TMEM accumulators per group (1)
  int boff; unsigned wait_mask;          // MMA issuer: chunk c <-> A buffer c + boff; bit c: wait on full[c + boff] first
  const float* xsrc; int xld, xcols;     // after this slot's MMAs: re-convert the resident X chunk from this array
};
struct TccChain {
  TccSlot slot[TCC_MAX_SLOTS];
  int nslots, nplanes;
  const float* x0; int x0ld, x0cols;     // resident X chunk (<= 32 columns) converted at kernel start
  const float* pre; int preld, precols;  // first-slot operand converted into ring buffers 0.. at kernel start
};
struct TccArgs {
  TccChain chain[TCC_MAX_CHAINS];
  int nchains, B, row_blocks;
  int passes;                     // 3 = 3xTF32 (fp32-accurate), 1 = one TF32 pass
  // host pipeline: the batch is sampled on another stream; every CTA first waits until wait_epoch[0..wait_n) >= *wait_clock + 1
  const unsigned long long* wait_epoch; const long long* wait_clock; int wait_n;
  uint8_t* xchg;                  // [nchains][row_blocks][TCC_PLANES][TCC_PLANE_BYTES]
  unsigned long long* trace; int trace_cta;
  unsigned long long* step_trace; int step_slot;
  unsigned long long* watchdog;   // host-mapped record written by a wait that timed out (see tcc_wait)
};

// ---- packed weight images ---------------------------------------------------------------------------
// A "use" is one weight matrix in one role: FWD rows = output features j, k = input features (W[j][k]);
// DX rows = input features n, k = output features (W[k][n]).  Image = [cdiv(N,32)][cdiv(K,32)][hi 4 KB | lo 4 KB],
// every block a zero-padded 32 x 32 K-major SWIZZLE_128B tile of tf32 hi / lo parts.
struct TccPackUse {
  const float* W; int ldw, mode, N, K;
  int nslices, nchunks, block_begin;
  long long dst_off;              // bytes into the image buffer
};
constexpr int TCC_MAX_USES = 32;
struct TccPackArgs {
  TccPackUse use[TCC_MAX_USES];
  int n, total_blocks;
  uint8_t* dst;
};
void tcc_pack_begin(TccPackArgs& p, uint8_t* dst);
// returns the use index.  Several pack sets may share one image buffer: `first_block` = blocks already taken
int tcc_pack_add(TccPackArgs& p, const float* W, int ldw, int mode, int N, int K);
void tcc_pack_set_base(TccPackArgs& p, uint8_t* dst, long long first_byte);
long long tcc_pack_bytes(const TccPackArgs& p);
struct TccImage { const uint8_t* ptr; int N, kchunks; };      // one packed weight image: N output rows, kchunks K chunks
static inline TccImage tcc_image(const TccPackArgs& p, int use) { return TccImage{p.dst + p.use[use].dst_off, p.use[use].N, p.use[use].nchunks}; }
int launch_tcc_pack(const TccPackArgs& p, cudaStream_t st);

// ---- chain construction -----------------------------------------------------------------------------
int64_t tcc_xchg_floats(int B);
void tcc_args_begin(TccArgs& a, int B, uint8_t* xchg, int passes);
void tcc_chain_x0(TccArgs& a, int c, const float* src, int ld, int cols);
void tcc_chain_pre(TccArgs& a, int c, const float* src, int ld, int cols);
// start a slot of chain c; returns the slot index
int tcc_slot_begin(TccArgs& a, int c);
void tcc_slot_src_x(TccArgs& a, int c, int slot);
void tcc_slot_src_pre(TccArgs& a, int c, int slot);                          // all pre chunks of the chain
void tcc_slot_src_plane(TccArgs& a, int c, int slot, int plane, int nchunks);
void tcc_slot_reconvert_x(TccArgs& a, int c, int slot, const float* src, int ld, int cols);
// add an output group; publish != 0 allocates a plane and returns its id (else -1)
int tcc_slot_group(TccArgs& a, int c, int slot, const TccImage& img, int epi, const float* bias,
                   const float* aux, int ldaux, float* C, int ldc, int publish);
int launch_mlp_tc_chain(TccArgs& a, cudaStream_t st);
unsigned long long* tcc_watchdog_device();      // host-mapped watchdog record (allocate outside of stream capture)

}  // namespace d4pg
