// Host interface of the tensor-core layer GEMM (tc_gemm.cu): a batch of independent problems -> one launch.
#pragma once
#include "mlp_kernels.cuh"

namespace cur {

constexpr int TC_MAX_PROBS = 16;
constexpr int TC_COLSUM_ROWS = 256;      // rows per partial row reduction

struct TcReduce {
  const float* part; float* out;
  int64_t count, stride;                 // floats per slice (multiple of 4), distance between slices
  int splits, block_begin, vec;
};
struct TcReduceBatch {
  TcReduce p[2 * TC_MAX_PROBS];
  int n;
};

bool tc_supported(const GemmProb& p);     // shape / alignment fit the tcgen05 kernel
int tc_pick_splits(const GemmProb& p);
int64_t tc_partial_floats(const GemmProb& p);   // floats of split-K workspace the problem needs (0: none)
int64_t tc_rowred_partial_floats(int64_t rows, int M, int NJ);
bool tc_skinny_supported(const GemmProb& p);

struct TcLauncher {
  struct { int n, total_tiles; } G;
  TcReduceBatch R;
  struct RowRedDesc { const float* X; int64_t ldx; const float* Y; int64_t ldy; int64_t rows; int M, NJ, chunks; float* part; }
      rowred[TC_MAX_PROBS];
  int n_rowred;
  struct SkinnyDesc { GemmProb p; } skinny[TC_MAX_PROBS];
  int n_skinny;
  bool pair;                 // launch the CTA-pair (cta_group::2) kernel: every problem of the batch needs M % 256 == 0
  int level;                 // flushes so far; partial workspaces alternate between two sets (level & 1)
  bool red_pending[2];       // deferred reductions reading partial set 0 / 1 are still in flight on the side stream
  alignas(64) unsigned char storage[TC_MAX_PROBS * (4 * 128 + 128) + 64];   // TcBatch (tensor maps + problems)
  TcLauncher();
  int add(const GemmProb& p, float* partial);
  // out[m][j] = sum_r X[r][m] * Y[r][j] (j < NJ <= 4), or the column sums of X when Y == NULL;
  // partial: tc_rowred_partial_floats(rows, M, NJ) floats
  int add_rowred(const float* X, int64_t ldx, int M, const float* Y, int64_t ldy, int NJ, int64_t rows, float* out,
                 float* partial);
  // bandwidth-bound problems with N <= 4 (output layers) or K <= 4 (backward through them), see tc_skinny_kernel
  int add_skinny(const GemmProb& p);
  int flush(cudaStream_t s);
  int finish(cudaStream_t s);        // join the deferred reductions (call once after the last flush)
  bool empty() const { return G.n == 0 && R.n == 0 && n_rowred == 0 && n_skinny == 0; }
};

// ---- the fused actor / critic chain kernel (tc_chain.cu)
struct TcChainIO {
  int64_t n, grad_rows;
  const float *mQ, *mP, *tQ, *tP;                       // parameter blocks of the four nets
  const float *Xpi, *Xg, *XQu, *Xpi_t, *Xg_t;           // prepared first-layer inputs [n][ld]
  const float *XQpi, *XQ_t;                             // ... (action columns: taken from the policy output in the kernel)
  float* wsplit;                                        // 4 x arena floats: main hi | main lo | target hi | target lo
  int ld_spi, ld_sq, ld_g, lddy;
  // TRANSPOSED copies [H][n] the weight gradients need: activations (main.pi, main.Q(u)), deltas (critic, actor chain)
  float *hp[CUR_MAX_LAYERS], *hq[CUR_MAX_LAYERS], *dc[CUR_MAX_LAYERS], *dp[CUR_MAX_LAYERS];
  uint32_t *mp, *mq, *mqp;                              // ReLU mask words [layers][H / 32][n] of main.pi, main.Q(u), main.Q(pi)
  float *Q, *Qt, *dQ, *dy, *q_pi;
  const float* r;
  float gamma, clip_return, action_l2;
  int clip_pos;
  float *loss_part;                                     // [n / 128][4]
  float *q_loss, *pi_loss;
  int64_t* step_counter;
  int loss_ring;
  int side_ok;                                          // one agent, launched on the caller's stream: the weight split may have run on
                                                        // the side stream (tc_chain_presplit_async) and the loss fold goes with the row sums
  int presplit;                                         // wsplit already holds the halves (tc_chain_presplit_group_async, then
                                                        // tc_chain_presplit_wait on the stream the lanes fork from)
};
// bias / output-layer weight gradients from the transposed copies (tc_chain_rowsum_kernel)
struct TcRowSum {
  const float* XT; int64_t ld;      // [M][rows] (NULL: ones)
  const float* Y; int ldy, NJ;      // optional [rows][NJ <= 4]
  float* out; int M, block_begin;
};
struct TcRowSumBatch {
  TcRowSum p[24];
  int n;
  int64_t rows;
};
int tc_chain_rowsums(cudaStream_t s, TcRowSumBatch& R);   // on a side stream forked from `s`
int tc_chain_join(cudaStream_t s);                        // ... which `s` waits for here
// concurrent chain launches of several experts: fork from `s`, expert i's stream, join back into `s`
int tc_chain_lanes_fork(cudaStream_t s);
int tc_chain_lane(int i, cudaStream_t* out);
int tc_chain_lanes_join(cudaStream_t s);
bool tc_chain_width_supported(const cur_net_desc& d, int64_t n);   // hidden 64, 128 or 256
bool tc_chain_supported(const cur_net_desc& d, int64_t n);         // ... hidden 256 only (cur_ddpg_grads)
int tc_chain_launch(cudaStream_t s, const cur_net_desc& d, const TcChainIO& io);
int tc_chain_presplit_async(cudaStream_t s, const float* mQ, const float* tQ, float* wsplit, int64_t arena);
// several experts: ONE launch on the side stream splits every expert's weights into its own wsplit; `s` waits for it in
// tc_chain_presplit_wait
int tc_chain_presplit_group_async(cudaStream_t s, int n_e, const float* const* mQ, const float* const* tQ,
                                  float* const* wsplit, int64_t arena);
int tc_chain_presplit_wait(cudaStream_t s);
void tc_chain_set_timeline(long long* dev);             // 128 x int64 debug stamps (CTA 0 / CTA 1) or NULL
// row-major [rows][cols] fp32 operand as a TMA tensor map in the layouts the tcgen05 descriptors expect (tc_gemm.cu)
int tc_make_map(void* map /* CUtensorMap */, const float* ptr, int64_t rows, int64_t cols, int64_t ld, int box_rows,
                bool mn_major);

}  // namespace cur
