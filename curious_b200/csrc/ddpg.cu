// DDPG / UVFA actor-critic: forward, losses, backward into a flat GetFlat-ordered gradient (sm_100a).
//
// Replaces (reference flowersteam/curious):
//   baselines/her/util.py:56-107           nn / nn_modular_her
//   baselines/her/actor_critic.py:5-98     ActorCritic / MultiTaskActorCritic
//   baselines/her/ddpg.py:412-449          losses + tf.gradients + flatten_grads
//   baselines/her/ddpg.py:129-146          get_actions forward
//
// Schedule: the DDPG graph is cut into dependency levels; each level is ONE grouped-GEMM launch
// (mlp_kernels.cuh) covering all independent nets of that level:
//   fwd-1 : main.pi | target.pi | main.Q(o,g,u)        (L layers + output layer)
//   fwd-2 : main.Q(o,g,pi) | target.Q(o2,g2,pi_t)      (L layers + output layer)
//   loss  : target = clip(r + gamma*Q_t), Q_loss, pi_loss, dQ, dQ_pi
//   bwd-1 : critic chain (dX + [dW;db]) | actor-through-Q chain (dX only)
//   bwd-2 : actor chain (dX + [dW;db])
// [dW;db] blocks are written straight into the flat gradient vector in GetFlat order, because
// kernel [in,out] followed by bias [out] is exactly one contiguous (in+1) x out matrix there.
#include <string.h>

#include <stdlib.h>

#include "net_layout.cuh"
#include "tc_gemm.cuh"

namespace cur {

// Workspace carve-up (floats).  All leading dimensions are multiples of 4.
struct Workspace {
  int ld_spi, ld_sq, ld_g, H;
  float *Xpi, *Xg, *XQu, *XQpi, *Xpi_t, *Xg_t, *XQ_t;
  float *hp[CUR_MAX_LAYERS], *hq[CUR_MAX_LAYERS], *hqp[CUR_MAX_LAYERS], *ht[CUR_MAX_LAYERS], *htq[CUR_MAX_LAYERS];
  float *Q, *Qt, *dQ, *dQpi, *dy;
  float *dc[2], *da[2], *dp[2];
  float *dcl[CUR_MAX_LAYERS], *dpl[CUR_MAX_LAYERS];   // chain schedule (tc_chain.cu): one delta buffer per layer
  float* chain_loss;                                   // ... and its per-tile loss partials [n / 128][4]
  float* chain_wsplit;                                 // ... the parameters of both arenas as 3xTF32 halves (4 x arena)
  uint32_t *chain_mp, *chain_mq, *chain_mqp;           // ... ReLU mask words [layers][H / 32][n] (main.pi, main.Q(u), main.Q(pi))
  float* chain_dwpart;                                 // ... hidden < 256: K-slice partials of the FFMA weight gradients
  // tensor-core path (large batch only): split-K partial tiles / partial row reductions, TC_SLOTS problems per level
  float *tc_part, *tc_rowpart;
  int64_t tc_part_stride, tc_rowpart_stride;
  float* loss_part;                // multi-CTA loss (large batch): LOSS_MAX_CTAS x 4 partial sums
  unsigned int* loss_ticket;       // self-resetting completion ticket (the workspace is zero-initialised by the caller)
  int64_t total;
};

// Batches this large run their layer GEMMs on the tensor cores (tc_gemm.cu); below it every GEMM of a level is
// latency-bound and the FFMA grouped kernel wins (measured us/update, FFMA vs tcgen05: 512: 203 / 268, 1024: 332 / 277,
// 1536: 454 / 281, 2048: 556 / 287, 4096: 1161 / 319, 16384: 4130 / 688).  CUR_DDPG_TC=0 or cur_ddpg_set_tensor_cores(0) forces the
// FFMA path, cur_ddpg_set_tensor_cores(1) forces the tensor cores for every eligible shape (A/B measurements, tests).
constexpr int64_t TC_MIN_BATCH = 1024;
constexpr int LOSS_MAX_CTAS = 128;
constexpr int64_t LOSS_MC_MIN_BATCH = 1024;   // from here the loss / backward-seed kernel runs on several CTAs
constexpr int TC_SLOTS = 8;          // split-K weight gradients / row reductions per dependency level (chain: per net)
static int g_tc_mode = -1;          // -1: environment (default on), 0: off, 1: on  (cur_ddpg_set_tensor_cores)
static bool tc_enabled() {
  if (g_tc_mode >= 0) return g_tc_mode == 1;
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("CUR_DDPG_TC");     // "0": FFMA only, "2": force the tensor cores for every eligible shape
    v = (e && e[0] == '0') ? 0 : 1;
    if (e && e[0] == '2') g_tc_mode = 1;
  }
  return v == 1;
}
static bool tc_shape_ok(const cur_net_desc& d, int64_t n) { return n >= 256 && (n % 128) == 0 && d.hidden == 256; }
static bool use_tc(const cur_net_desc& d, int64_t n) {
  if (!tc_shape_ok(d, n) || !tc_enabled()) return false;
  return g_tc_mode == 1 || n >= TC_MIN_BATCH;
}

// The fused chain kernel (tc_chain.cu) replaces the forward / loss / dX levels whenever the tensor-core path is on and the
// shape fits; CUR_DDPG_CHAIN=0 or cur_ddpg_set_chain(0) keeps the level-by-level schedule (A/B measurements, tests).
static int g_chain_mode = -1;
static bool chain_enabled() {
  if (g_chain_mode >= 0) return g_chain_mode == 1;
  static int v = -1;
  if (v < 0) { const char* e = getenv("CUR_DDPG_CHAIN"); v = (e && e[0] == '0') ? 0 : 1; }
  return v == 1;
}
static bool use_chain(const cur_net_desc& d, int64_t n) {
  if (!use_tc(d, n) || !tc_chain_supported(d, n)) return false;
  return chain_enabled();
}
// Hidden 64 / 128 on the chain kernel (cur_ddpg_chain_grads): the weight gradients are too narrow for the 128 x 256 tile
// of tc_gemm_kernel and run on the FFMA grouped GEMM, K split into at most this many slices of the batch
constexpr int CH_DW_MAX_SPLITS = 8;
static bool narrow_chain_ok(const cur_net_desc& d, int64_t n) {
  return d.hidden < 256 && tc_chain_width_supported(d, n) && chain_enabled();
}
static int64_t chain_dw_floats(const cur_net_desc& d) {     // sum of M x N over the weight gradients of both nets
  int64_t f = 0;
  for (int which = 0; which < 2; ++which) {
    const NetLayout q = net_layout(d, which);
    f += (int64_t)(d.layers - 1) * d.hidden * d.hidden + (int64_t)(q.in_s + q.in_g) * d.hidden;
  }
  return f;
}

// narrow_chain: also carve the chain buffers of a net narrower than 256 (cur_ddpg_chain_workspace_floats)
static Workspace carve(const cur_net_desc& d, int64_t n, float* base, bool narrow_chain = false) {
  Workspace w;
  const NetLayout q = net_layout(d, 0), p = net_layout(d, 1);
  w.ld_spi = (int)r4(p.in_s);
  w.ld_sq = (int)r4(q.in_s);
  w.ld_g = (int)r4(d.modular ? d.dimg : 0);
  w.H = d.hidden;
  int64_t o = 0;
  auto take = [&](int64_t floats) {
    float* ptr = base ? base + o : nullptr;
    o += r4(floats);
    return ptr;
  };
  w.Xpi = take(n * w.ld_spi);
  w.Xg = take(n * w.ld_g);
  w.XQu = take(n * w.ld_sq);
  w.XQpi = take(n * w.ld_sq);
  w.Xpi_t = take(n * w.ld_spi);
  w.Xg_t = take(n * w.ld_g);
  w.XQ_t = take(n * w.ld_sq);
  for (int l = 0; l < d.layers; ++l) {
    w.hp[l] = take(n * w.H);
    w.hq[l] = take(n * w.H);
    w.hqp[l] = take(n * w.H);
    w.ht[l] = take(n * w.H);
    w.htq[l] = take(n * w.H);
  }
  w.Q = take(n);
  w.Qt = take(n);
  w.dQ = take(n);
  w.dQpi = take(n);
  w.dy = take(n * r4(d.dimu));
  for (int i = 0; i < 2; ++i) {
    w.dc[i] = take(n * w.H);
    w.da[i] = take(n * w.H);
    w.dp[i] = take(n * w.H);
  }
  w.loss_ticket = reinterpret_cast<unsigned int*>(take(4));
  w.loss_part = take(LOSS_MAX_CTAS * 4);
  w.tc_part = w.tc_rowpart = nullptr;
  w.tc_part_stride = w.tc_rowpart_stride = 0;
  for (int l = 0; l < CUR_MAX_LAYERS; ++l) w.dcl[l] = w.dpl[l] = nullptr;
  w.chain_loss = nullptr;
  w.chain_mp = w.chain_mq = w.chain_mqp = nullptr;
  w.chain_wsplit = nullptr;
  w.chain_dwpart = nullptr;
  const bool narrow = narrow_chain && d.hidden < 256 && tc_chain_width_supported(d, n);
  if (tc_chain_supported(d, n) || narrow) {
    for (int l = 0; l < d.layers; ++l) { w.dcl[l] = take(n * w.H); w.dpl[l] = take(n * w.H); }
    w.chain_loss = take((n / 128) * 4);
    w.chain_wsplit = take(4 * (r4(q.total) + r4(p.total)));
    w.chain_mp = reinterpret_cast<uint32_t*>(take((int64_t)d.layers * (w.H / 32) * n));
    w.chain_mq = reinterpret_cast<uint32_t*>(take((int64_t)d.layers * (w.H / 32) * n));
    w.chain_mqp = reinterpret_cast<uint32_t*>(take((int64_t)d.layers * (w.H / 32) * n));
  }
  if (narrow) w.chain_dwpart = take(CH_DW_MAX_SPLITS * chain_dw_floats(d));
  if (tc_shape_ok(d, n)) {      // carved whenever the shape is eligible: the workspace size does not depend on the toggle
    GemmProb dwp = zero_prob();
    dwp.M = w.H; dwp.N = w.H; dwp.K = (int)n; dwp.a_trans = 1;
    w.tc_part_stride = r4(tc_partial_floats(dwp));
    w.tc_rowpart_stride = r4(tc_rowred_partial_floats(n, w.H, 4));
    w.tc_part = take(2 * TC_SLOTS * w.tc_part_stride);          // two sets: the reductions of a level are deferred
    w.tc_rowpart = take(2 * TC_SLOTS * w.tc_rowpart_stride);    // (TcLauncher::flush), the next level uses the other set
  }
  w.total = o;
  return w;
}

// ------------------------------------------------------------------------------------------------
// prep: build the first-layer input matrices (normalise/clip o,g; append task_descr and action)
// ------------------------------------------------------------------------------------------------
struct PrepParams {
  cur_net_desc d;
  const float *o, *g, *u, *td, *o_2, *g_2;
  const float *ag;           // actions path only: relative goals g <- g - ag (ddpg.py:119-124)
  float clip_obs;            // actions path only: clip o,g to +-clip_obs first (ddpg.py:125-126); <=0: off
  const float *o_mean, *o_std, *g_mean, *g_std;
  int64_t n;
  int ld_spi, ld_sq, ld_g;
  float *Xpi, *Xg, *XQu, *XQpi, *Xpi_t, *Xg_t, *XQ_t;   // any may be NULL
};

__device__ __forceinline__ float norm1(float x, const float* mean, const float* std, int k, float clip) {
  float v = __fdiv_rn(__fsub_rn(x, mean[k]), std[k]);          // normalizer.py:72-77
  return fminf(fmaxf(v, -clip), clip);
}

__global__ void __launch_bounds__(256) prep_kernel(const __grid_constant__ PrepParams P) {
  const cur_net_desc& d = P.d;
  const int in_o = d.dimo;
  const int in_spi = d.modular ? d.dimo + d.dimtd : d.dimo + d.dimg;
  const int width = in_spi + d.dimu;   // columns of the widest matrix (XQ*)
  const int64_t total = P.n * width;
  const bool nrm = d.normalize_obs != 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / width;
    const int k = (int)(i - r * width);
    float v = 0.f, v2 = 0.f;   // main-side / target-side value of column k
    if (k < in_o) {
      v = P.o[r * d.dimo + k];
      if (P.clip_obs > 0.f) v = fminf(fmaxf(v, -P.clip_obs), P.clip_obs);
      if (nrm) v = norm1(v, P.o_mean, P.o_std, k, d.norm_clip);
      if (P.o_2) {
        v2 = P.o_2[r * d.dimo + k];
        if (nrm) v2 = norm1(v2, P.o_mean, P.o_std, k, d.norm_clip);
      }
    } else if (k < in_spi) {
      const int j = k - in_o;
      if (d.modular) {
        v = P.td[r * d.dimtd + j];      // task descriptor is never normalised (actor_critic.py:79,88)
        v2 = v;
      } else {
        v = P.g[r * d.dimg + j];
        if (P.ag) v = __fsub_rn(v, P.ag[r * d.dimg + j]);
        if (P.clip_obs > 0.f) v = fminf(fmaxf(v, -P.clip_obs), P.clip_obs);
        if (nrm) v = norm1(v, P.g_mean, P.g_std, j, d.norm_clip);
        if (P.g_2) {
          v2 = P.g_2[r * d.dimg + j];
          if (nrm) v2 = norm1(v2, P.g_mean, P.g_std, j, d.norm_clip);
        }
      }
    } else {
      const int j = k - in_spi;
      if (P.u && P.XQu) P.XQu[r * P.ld_sq + k] = __fdiv_rn(P.u[r * d.dimu + j], d.max_u);   // u / max_u
      continue;
    }
    if (P.Xpi) P.Xpi[r * P.ld_spi + k] = v;
    if (P.XQu) P.XQu[r * P.ld_sq + k] = v;
    if (P.XQpi) P.XQpi[r * P.ld_sq + k] = v;
    if (P.Xpi_t) P.Xpi_t[r * P.ld_spi + k] = v2;
    if (P.XQ_t) P.XQ_t[r * P.ld_sq + k] = v2;
  }
  if (d.modular) {
    const int64_t totg = P.n * d.dimg;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < totg;
         i += (int64_t)gridDim.x * blockDim.x) {
      const int64_t r = i / d.dimg;
      const int j = (int)(i - r * d.dimg);
      float v = P.g[i];
      if (P.ag) v = __fsub_rn(v, P.ag[i]);
      if (P.clip_obs > 0.f) v = fminf(fmaxf(v, -P.clip_obs), P.clip_obs);
      if (nrm) v = norm1(v, P.g_mean, P.g_std, j, d.norm_clip);
      if (P.Xg) P.Xg[r * P.ld_g + j] = v;
      if (P.g_2 && P.Xg_t) {
        float v2 = P.g_2[i];
        if (nrm) v2 = norm1(v2, P.g_mean, P.g_std, j, d.norm_clip);
        P.Xg_t[r * P.ld_g + j] = v2;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// losses (ddpg.py:436-441) + the two seeds of the backward pass.  One CTA.
// ------------------------------------------------------------------------------------------------
struct LossParams {
  const float *r, *Q, *Qpi, *Qt, *th;
  int ldth, dimu;
  int64_t n;
  float gamma, clip_return, action_l2;
  int clip_pos;
  float *dQ, *dQpi, *q_loss, *pi_loss;
  int64_t grad_rows;       // rows one loss mean runs over for the GRADIENT seeds (n, or the per-worker batch when the
                           // launch carries several reference workers, cur_ddpg_hyper.loss_rows)
  int64_t* step_counter;   // optional: losses go to slot (*step % ring), then *step += 1
  int ring;
};

__global__ void __launch_bounds__(1024) loss_kernel(const __grid_constant__ LossParams P) {
  __shared__ float red[3][32];
  float ssq = 0.f, sq = 0.f, sth = 0.f;
  const float inv_n = 1.0f / (float)P.n;
  const float inv_g = 1.0f / (float)P.grad_rows;
  const float hi = P.clip_pos ? 0.f : INFINITY;
  for (int64_t i = threadIdx.x; i < P.n; i += blockDim.x) {
    float tgt = fminf(fmaxf(P.r[i] + P.gamma * P.Qt[i], -P.clip_return), hi);   // ddpg.py:436-438
    float diff = tgt - P.Q[i];
    ssq += diff * diff;
    sq += P.Qpi[i];
    P.dQ[i] = -2.0f * inv_g * diff;      // d mean((tgt - Q)^2) / dQ
    P.dQpi[i] = -inv_g;                  // d (-mean(Q_pi)) / dQ_pi
  }
  for (int64_t i = threadIdx.x; i < P.n * P.dimu; i += blockDim.x) {
    int64_t r = i / P.dimu;
    float t = P.th[r * P.ldth + (i - r * P.dimu)];
    sth += t * t;
  }
  for (int o = 16; o > 0; o >>= 1) {
    ssq += __shfl_xor_sync(0xffffffffu, ssq, o);
    sq += __shfl_xor_sync(0xffffffffu, sq, o);
    sth += __shfl_xor_sync(0xffffffffu, sth, o);
  }
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { red[0][w] = ssq; red[1][w] = sq; red[2][w] = sth; }
  __syncthreads();
  if (w == 0) {
    const int nw = blockDim.x >> 5;
    ssq = l < nw ? red[0][l] : 0.f;
    sq = l < nw ? red[1][l] : 0.f;
    sth = l < nw ? red[2][l] : 0.f;
    for (int o = 16; o > 0; o >>= 1) {
      ssq += __shfl_xor_sync(0xffffffffu, ssq, o);
      sq += __shfl_xor_sync(0xffffffffu, sq, o);
      sth += __shfl_xor_sync(0xffffffffu, sth, o);
    }
    if (l == 0) {
      long long slot = 0;
      if (P.step_counter) {
        const long long st = *P.step_counter;
        slot = P.ring > 0 ? st % P.ring : 0;
        *P.step_counter = st + 1;
      }
      if (P.q_loss) P.q_loss[slot] = ssq * inv_n;                                           // ddpg.py:439
      if (P.pi_loss) P.pi_loss[slot] = -sq * inv_n + P.action_l2 * sth / (float)(P.n * P.dimu);   // :440-441
    }
  }
}

// Same computation on several CTAs (batch >= LOSS_MC_MIN_BATCH; one CTA takes 53 us at batch 16384): every CTA reduces a
// contiguous slice of rows, the last one to finish (ticket) folds the per-CTA partials in CTA order - deterministic.
struct LossMcParams {
  LossParams L;
  float* part;
  unsigned int* ticket;
};
__global__ void __launch_bounds__(512) loss_mc_kernel(const __grid_constant__ LossMcParams M) {
  const LossParams& P = M.L;
  __shared__ float red[3][16];
  __shared__ unsigned int s_last;
  const int64_t per = (P.n + gridDim.x - 1) / gridDim.x;
  const int64_t r0 = per * blockIdx.x, r1 = (r0 + per < P.n) ? r0 + per : P.n;
  float ssq = 0.f, sq = 0.f, sth = 0.f;
  const float inv_n = 1.0f / (float)P.n;
  const float inv_g = 1.0f / (float)P.grad_rows;
  const float hi = P.clip_pos ? 0.f : INFINITY;
  for (int64_t i = r0 + threadIdx.x; i < r1; i += blockDim.x) {
    float tgt = fminf(fmaxf(P.r[i] + P.gamma * P.Qt[i], -P.clip_return), hi);   // ddpg.py:436-438
    float diff = tgt - P.Q[i];
    ssq += diff * diff;
    sq += P.Qpi[i];
    P.dQ[i] = -2.0f * inv_g * diff;
    P.dQpi[i] = -inv_g;
    for (int j = 0; j < P.dimu; ++j) {
      const float t = P.th[i * P.ldth + j];
      sth += t * t;
    }
  }
  for (int o = 16; o > 0; o >>= 1) {
    ssq += __shfl_xor_sync(0xffffffffu, ssq, o);
    sq += __shfl_xor_sync(0xffffffffu, sq, o);
    sth += __shfl_xor_sync(0xffffffffu, sth, o);
  }
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { red[0][w] = ssq; red[1][w] = sq; red[2][w] = sth; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f, b = 0.f, c = 0.f;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) { a += red[0][i]; b += red[1][i]; c += red[2][i]; }
    M.part[4 * blockIdx.x + 0] = a; M.part[4 * blockIdx.x + 1] = b; M.part[4 * blockIdx.x + 2] = c;
    __threadfence();
    s_last = (atomicAdd(M.ticket, 1u) == gridDim.x - 1) ? 1u : 0u;
  }
  __syncthreads();
  if (s_last && threadIdx.x == 0) {
    __threadfence();
    float a = 0.f, b = 0.f, c = 0.f;
    for (int i = 0; i < (int)gridDim.x; ++i) {
      a += ((volatile float*)M.part)[4 * i + 0]; b += ((volatile float*)M.part)[4 * i + 1]; c += ((volatile float*)M.part)[4 * i + 2];
    }
    long long slot = 0;
    if (P.step_counter) {
      const long long st = *P.step_counter;
      slot = P.ring > 0 ? st % P.ring : 0;
      *P.step_counter = st + 1;
    }
    if (P.q_loss) P.q_loss[slot] = a * inv_n;                                           // ddpg.py:439
    if (P.pi_loss) P.pi_loss[slot] = -b * inv_n + P.action_l2 * c / (float)(P.n * P.dimu);   // :440-441
    *M.ticket = 0u;
  }
}

// One dependency level: problems that fit the tensor-core kernel go there when the batch is large, everything else
// (output layers at small batch, batches below the crossover) to the FFMA grouped kernel.
struct Batcher {
  GemmBatch G;
  TcLauncher T;
  cudaStream_t s;
  bool tc;
  float *tc_part, *tc_rowpart;
  int64_t part_stride, rowpart_stride;
  int rc, parts_used, rowparts_used;
  explicit Batcher(cudaStream_t st) : s(st), tc(false), tc_part(nullptr), tc_rowpart(nullptr), part_stride(0),
                                      rowpart_stride(0), rc(CUR_OK), parts_used(0), rowparts_used(0) {
    G.n = 0; G.total_tiles = 0;
  }
  Batcher(cudaStream_t st, bool use_tensor_cores, const Workspace& w)
      : s(st), tc(use_tensor_cores && w.tc_part != nullptr), tc_part(w.tc_part), tc_rowpart(w.tc_rowpart),
        part_stride(w.tc_part_stride), rowpart_stride(w.tc_rowpart_stride), rc(CUR_OK), parts_used(0), rowparts_used(0) {
    G.n = 0; G.total_tiles = 0;
  }
  void add(const GemmProb& p) {
    if (tc && tc_skinny_supported(p)) {               // before the tensor-core test: K <= 4 outer products fit both
      const int r = T.add_skinny(p);
      if (r != CUR_OK) rc = r;
      return;
    }
    if (tc && !p.ones_a && tc_supported(p)) {
      const bool split = tc_pick_splits(p) > 1;
      if (!split || (parts_used < TC_SLOTS && tc_partial_floats(p) <= part_stride)) {
        const int r = T.add(p, split ? tc_part + ((T.level & 1) * TC_SLOTS + parts_used) * part_stride : nullptr);
        if (r != CUR_OK) rc = r;
        if (split) ++parts_used;
        return;
      }
    }
    // K = batch reductions with a skinny output: bias gradients (column sums) and the output-layer weight gradients
    const bool colsum = p.ones_a && p.N <= 256;
    const bool skinny = !p.ones_a && p.a_trans && !p.b_trans && p.N <= 4 && p.K2 == 0 && p.ldc == p.N && p.epi == EPI_NONE &&
                        p.bias == nullptr && p.C2 == nullptr;
    if (tc && (colsum || skinny) && rowparts_used < TC_SLOTS) {
      float* part = tc_rowpart + ((T.level & 1) * TC_SLOTS + rowparts_used) * rowpart_stride;
      const int r = colsum ? T.add_rowred(p.B, p.ldb, p.N, nullptr, 0, 1, p.K, p.C, part)
                           : T.add_rowred(p.A, p.lda, p.M, p.B, p.ldb, p.N, p.K, p.C, part);
      if (r != CUR_OK) rc = r;
      ++rowparts_used;
      return;
    }
    G.p[G.n++] = p;
  }
  int flush() {
    if (rc != CUR_OK) return rc;
    int r = launch_gemm_batch(G, s);
    G.n = 0;
    if (r != CUR_OK) return r;
    parts_used = rowparts_used = 0;
    return T.empty() ? CUR_OK : T.flush(s);
  }
};

static int grid_prep(int64_t work) {
  int64_t b = (work + 255) / 256;
  int64_t cap = (int64_t)sm_count() * 4;
  return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}

// ------------------------------------------------------------------------------------------------
// Weight gradients of the chain schedule at hidden 64 / 128: dW = X^T dY (K = batch) as FFMA grouped-GEMM tiles over K
// slices of the batch, each slice into its own partial block, then the slices summed in slice order (deterministic).
// Without the split the few 32 x 32 tiles of H-wide gradients (4 per hidden layer at H = 64) occupy a handful of SMs for
// the whole batch.
// ------------------------------------------------------------------------------------------------
struct DwSliceSum {
  const float* part;        // [splits][count]
  float* out;               // [count]
  int64_t count;
  int splits;
};
constexpr int DW_PER_AGENT = 2 * (CUR_MAX_LAYERS + 1);   // weight-gradient problems of one agent, at most
// CAP entries: one agent's (DW_PER_AGENT) or a grouped update's (CUR_MAX_TASKS x DW_PER_AGENT)
template <int CAP>
struct DwSliceSumBatch {
  DwSliceSum p[CAP];
  int n;
};
template <int CAP>
__global__ void __launch_bounds__(256) dw_slice_sum_kernel(const __grid_constant__ DwSliceSumBatch<CAP> R) {
  for (int i = 0; i < R.n; ++i) {
    const DwSliceSum& P = R.p[i];
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < P.count; e += (int64_t)gridDim.x * blockDim.x) {
      float v = P.part[e];
      for (int s = 1; s < P.splits; ++s) v += P.part[(int64_t)s * P.count + e];
      P.out[e] = v;
    }
  }
}
template <int CAP>
static int dw_slice_sum_launch(cudaStream_t s, const DwSliceSum* sums, int count) {
  CUR_REQUIRE(count <= CAP, "too many weight-gradient problems");
  DwSliceSumBatch<CAP> R;
  R.n = count;
  for (int i = 0; i < count; ++i) R.p[i] = sums[i];
  dw_slice_sum_kernel<CAP><<<2 * sm_count(), 256, 0, s>>>(R);
  CUR_CHECK_LAUNCH();
  return CUR_OK;
}

// The K slices of one agent's problem list: enough for two CTAs per SM (the grouped GEMM's occupancy), each at least 256
// rows, in whole GK chunks.  Every expert of a grouped update gets the slices it would get alone.
struct DwSlicePlan {
  int splits;
  int64_t ks;              // rows per slice (the last one takes the rest)
};
static DwSlicePlan chain_dw_plan(const GemmProb* probs, int np, int64_t n) {
  int tiles = 0;
  for (int i = 0; i < np; ++i) tiles += ((probs[i].M + GT - 1) / GT) * ((probs[i].N + GT - 1) / GT);
  int splits = (2 * sm_count() + tiles - 1) / (tiles > 0 ? tiles : 1);
  if (splits > CH_DW_MAX_SPLITS) splits = CH_DW_MAX_SPLITS;
  if (splits > n / 256) splits = (int)(n / 256);
  if (splits < 1) splits = 1;
  DwSlicePlan pl;
  pl.ks = ((n + splits - 1) / splits + GK - 1) / GK * GK;
  pl.splits = (int)((n + pl.ks - 1) / pl.ks);
  return pl;
}

// probs: n_e lists of np dW problems each (expert i's from probs + i * np, all lists of one shape) with contiguous outputs
// (ldc == N), K = n, B K-major [N][n]; A K-major [M][n] (a_trans 0) or the input matrix [n][lda] (a_trans 1).  parts[i]:
// expert i's CH_DW_MAX_SPLITS x (sum of M x N) floats.  The slice GEMMs of all experts share the grouped-GEMM launches
// and one slice-sum launch adds every expert's slices.
static int chain_dw_ffma(cudaStream_t s, const GemmProb* probs, int np, int n_e, int64_t n, float* const* parts) {
  CUR_REQUIRE(np <= DW_PER_AGENT && n_e >= 1 && n_e <= CUR_MAX_TASKS, "bad weight-gradient list");
  GemmBatch G;
  G.n = 0; G.total_tiles = 0;
  DwSliceSum R[CUR_MAX_TASKS * DW_PER_AGENT];
  int nr = 0;
  for (int x = 0; x < n_e; ++x) {
    const GemmProb* pr = probs + x * np;
    const DwSlicePlan pl = chain_dw_plan(pr, np, n);
    const int splits = pl.splits;
    const int64_t ks = pl.ks;
    float* pp = parts[x];
    CUR_REQUIRE(pp != nullptr, "bad weight-gradient list");
    for (int i = 0; i < np; ++i) {
      const GemmProb& q = pr[i];
      CUR_REQUIRE(q.ldc == q.N && q.b_trans == 1 && q.K == n, "bad weight-gradient problem");
      const int64_t count = (int64_t)q.M * q.N;
      for (int sl = 0; sl < splits; ++sl) {
        const int64_t k0 = sl * ks;
        GemmProb p = q;
        p.split_k = 0;
        p.K = (int)(k0 + ks <= n ? ks : n - k0);
        p.A = q.a_trans ? q.A + k0 * q.lda : q.A + k0;
        p.B = q.B + k0;
        p.C = pp + sl * count;
        G.p[G.n++] = p;
        if (G.n == GEMM_MAX_PROBS) {
          CUR_TRY(launch_gemm_batch(G, s));
          G.n = 0;
        }
      }
      DwSliceSum& r = R[nr++];
      r.part = pp; r.out = q.C; r.count = count; r.splits = splits;
      pp += splits * count;
    }
  }
  if (G.n > 0) CUR_TRY(launch_gemm_batch(G, s));
  if (n_e == 1) return dw_slice_sum_launch<DW_PER_AGENT>(s, R, nr);
  return dw_slice_sum_launch<CUR_MAX_TASKS * DW_PER_AGENT>(s, R, nr);
}

}  // namespace cur

using namespace cur;

extern "C" int64_t cur_net_param_count(const cur_net_desc* d, int which) {
  if (check_desc(d) != CUR_OK || (which != 0 && which != 1)) return -1;
  return net_layout(*d, which).total;
}

extern "C" int64_t cur_theta_pi_offset(const cur_net_desc* d, int64_t* total) {
  if (check_desc(d) != CUR_OK) return -1;
  const int64_t off = r4(net_layout(*d, 0).total);
  if (total) *total = off + r4(net_layout(*d, 1).total);
  return off;
}

extern "C" int cur_ddpg_set_tensor_cores(int mode) {
  CUR_REQUIRE(mode >= -1 && mode <= 1, "mode must be -1 (default), 0 (off) or 1 (on)");
  g_tc_mode = mode;
  return CUR_OK;
}

extern "C" int cur_ddpg_set_chain(int mode) {
  CUR_REQUIRE(mode >= -1 && mode <= 1, "mode must be -1 (default), 0 (off) or 1 (on)");
  g_chain_mode = mode;
  return CUR_OK;
}

extern "C" int cur_ddpg_uses_chain(const cur_net_desc* d, int64_t batch) {
  if (check_desc(d) != CUR_OK || batch <= 0) return 0;
  return use_chain(*d, batch) ? 1 : 0;
}

extern "C" int cur_ddpg_uses_tensor_cores(const cur_net_desc* d, int64_t batch) {
  if (check_desc(d) != CUR_OK || batch <= 0) return 0;
  return use_tc(*d, batch) ? 1 : 0;
}

extern "C" int64_t cur_ddpg_workspace_floats(const cur_net_desc* d, int64_t batch) {
  if (check_desc(d) != CUR_OK || batch <= 0) return -1;
  return carve(*d, batch, nullptr).total;
}

extern "C" int cur_ddpg_actions(void* stream, const cur_net_desc* d, const float* theta,
                                const cur_norm_stats* stats, const float* o, const float* ag, const float* g,
                                const float* td, int64_t n, float clip_obs, float* workspace, float* out_pi,
                                float* out_q) {
  CUR_TRY(check_desc(d));
  CUR_REQUIRE(theta && o && g && workspace && out_pi, "NULL argument");
  CUR_REQUIRE(!d->modular || td, "task_descr required for a modular net");
  CUR_REQUIRE(n > 0 && n < (1 << 30), "bad batch");
  if (d->normalize_obs)
    CUR_REQUIRE(stats && stats->o_mean && stats->o_std && stats->g_mean && stats->g_std, "normalizer stats required");
  cudaStream_t s = (cudaStream_t)stream;
  const NetLayout LQ = net_layout(*d, 0), LP = net_layout(*d, 1);
  const float* thQ = theta;
  const float* thP = theta + r4(LQ.total);
  Workspace w = carve(*d, n, workspace);

  PrepParams P;
  memset(&P, 0, sizeof(P));
  P.d = *d; P.o = o; P.g = g; P.td = td; P.n = n;
  P.ag = ag; P.clip_obs = clip_obs;
  if (stats) { P.o_mean = stats->o_mean; P.o_std = stats->o_std; P.g_mean = stats->g_mean; P.g_std = stats->g_std; }
  P.ld_spi = w.ld_spi; P.ld_sq = w.ld_sq; P.ld_g = w.ld_g;
  P.Xpi = w.Xpi; P.Xg = w.Xg; P.XQpi = out_q ? w.XQpi : nullptr;
  prep_kernel<<<grid_prep(n * (LQ.in_s)), 256, 0, s>>>(P);
  CUR_CHECK_LAUNCH();

  Batcher B(s);
  B.add(fwd0(LP, thP, w.Xpi, w.ld_spi, w.Xg, w.ld_g, w.hp[0], n));
  CUR_TRY(B.flush());
  for (int l = 1; l < LP.L; ++l) {
    B.add(fwdl(LP, thP, l, w.hp[l - 1], w.hp[l], n));
    CUR_TRY(B.flush());
  }
  {
    // th = tanh(.) goes into the action columns of the critic input; pi = max_u * th to the caller
    GemmProb p = fwdout(LP, thP, w.hp[LP.L - 1], w.XQpi + LP.in_s, w.ld_sq, EPI_TANH, n);
    p.C2 = out_pi; p.ldc2 = d->dimu; p.scale2 = d->max_u;
    B.add(p);
    CUR_TRY(B.flush());
  }
  if (out_q) {
    B.add(fwd0(LQ, thQ, w.XQpi, w.ld_sq, w.Xg, w.ld_g, w.hqp[0], n));
    CUR_TRY(B.flush());
    for (int l = 1; l < LQ.L; ++l) {
      B.add(fwdl(LQ, thQ, l, w.hqp[l - 1], w.hqp[l], n));
      CUR_TRY(B.flush());
    }
    B.add(fwdout(LQ, thQ, w.hqp[LQ.L - 1], out_q, 1, EPI_NONE, n));
    CUR_TRY(B.flush());
  }
  return CUR_OK;
}

// One expert (= one DDPG agent) of a grouped update: its parameters, staged batch, outputs and workspace.
struct Expert {
  Workspace w;
  const float *mQ, *mP, *tQ, *tP;
  float *gQ, *gP;
  const cur_batch* batch;
  const cur_norm_stats* stats;
  const cur_ddpg_hyper* h;
  float *q_loss, *pi_loss, *q_pi;
  float* th;                           // tanh output = action columns of main.Q's input
  int parts_used, rowparts_used;       // split-K / row-reduction workspace slots taken in the current level
};

// Level batcher over several experts: every add() names the expert whose workspace slots the problem may use.
struct GroupBatcher {
  Batcher B;
  Expert* e;
  int n_e;
  GroupBatcher(cudaStream_t s, bool tc, Expert* experts, int n) : B(s), e(experts), n_e(n) {
    B.tc = tc && experts[0].w.tc_part != nullptr;
  }
  int add(int i, const GemmProb& p) {
    // flush early when a launch is full (many experts): problems of one level are independent, so splitting a level
    // over several launches is always legal
    if (B.G.n >= GEMM_MAX_PROBS - 1 || B.T.G.n >= TC_MAX_PROBS - 1 || B.T.R.n >= 2 * TC_MAX_PROBS - 2 ||
        B.T.n_rowred >= TC_MAX_PROBS - 1 || B.T.n_skinny >= TC_MAX_PROBS - 1)
      CUR_TRY(flush());
    Expert& x = e[i];
    B.tc_part = x.w.tc_part; B.tc_rowpart = x.w.tc_rowpart;
    B.part_stride = x.w.tc_part_stride; B.rowpart_stride = x.w.tc_rowpart_stride;
    B.parts_used = x.parts_used; B.rowparts_used = x.rowparts_used;
    B.add(p);
    x.parts_used = B.parts_used; x.rowparts_used = B.rowparts_used;
    return B.rc;
  }
  int flush() {
    CUR_TRY(B.flush());
    for (int i = 0; i < n_e; ++i) e[i].parts_used = e[i].rowparts_used = 0;
    return CUR_OK;
  }
};

// DDPG._grads for n_e experts of identical shape: every dependency level is ONE launch (per kernel kind) over all
// experts - the grouped-GEMM form of structure='task_experts' (train.py:287-289 builds one DDPG per module).
// narrow_chain: agents of hidden 64 / 128 on the chain schedule (cur_ddpg_chain_grads, cur_ddpg_chain_grads_group)
static int grads_levels(cudaStream_t s, const cur_net_desc* d, Expert* E, int n_e, int64_t n, bool narrow_chain = false) {
  const NetLayout LQ = net_layout(*d, 0), LP = net_layout(*d, 1);
  const int L = d->layers, H = d->hidden;
  const bool chain = narrow_chain || use_chain(*d, n);
  // the chain lanes of several narrow experts start from weights split by one launch beside the input preparation
  const bool group_split = narrow_chain && n_e > 1;
  // ---- chain schedule, one agent: the 3xTF32 weight halves are split on a side stream beside the input preparation
  if (n_e == 1 && chain)
    CUR_TRY(tc_chain_presplit_async(s, E[0].mQ, E[0].tQ, E[0].w.chain_wsplit, r4(LQ.total) + r4(LP.total)));
  if (group_split) {
    const float *mQ[CUR_MAX_TASKS], *tQ[CUR_MAX_TASKS];
    float* ws[CUR_MAX_TASKS];
    for (int i = 0; i < n_e; ++i) { mQ[i] = E[i].mQ; tQ[i] = E[i].tQ; ws[i] = E[i].w.chain_wsplit; }
    CUR_TRY(tc_chain_presplit_group_async(s, n_e, mQ, tQ, ws, r4(LQ.total) + r4(LP.total)));
  }
  // ---- inputs
  for (int i = 0; i < n_e; ++i) {
    Expert& x = E[i];
    PrepParams P;
    memset(&P, 0, sizeof(P));
    const cur_batch* b = x.batch;
    P.d = *d; P.o = b->o; P.g = b->g; P.u = b->u; P.td = b->td; P.o_2 = b->o_2; P.g_2 = b->g_2;
    P.n = n;
    if (x.stats) { P.o_mean = x.stats->o_mean; P.o_std = x.stats->o_std; P.g_mean = x.stats->g_mean; P.g_std = x.stats->g_std; }
    P.ld_spi = x.w.ld_spi; P.ld_sq = x.w.ld_sq; P.ld_g = x.w.ld_g;
    P.Xpi = x.w.Xpi; P.Xg = x.w.Xg; P.XQu = x.w.XQu; P.XQpi = x.w.XQpi; P.Xpi_t = x.w.Xpi_t; P.Xg_t = x.w.Xg_t; P.XQ_t = x.w.XQ_t;
    prep_kernel<<<grid_prep(n * LQ.in_s), 256, 0, s>>>(P);
    CUR_CHECK_LAUNCH();
    x.th = x.w.XQpi + LP.in_s;
    x.parts_used = x.rowparts_used = 0;
  }
  GroupBatcher B(s, use_tc(*d, n), E, n_e);
#define FOR_EXPERTS for (int i = 0; i < n_e; ++i)
#define ADD(prob) CUR_TRY(B.add(i, (prob)))
  if (chain) {
    // ---- chain schedule (tc_chain.cu): forward nets, losses and the data-gradient chains of a 128-row tile in one
    // CTA per chain, then every weight / bias gradient as split-K tensor-core GEMMs + row reductions, one level per net
    // (hidden 64 / 128: the weight gradients as K-sliced FFMA GEMMs, chain_dw_ffma)
    GemmProb dw_ffma[CUR_MAX_TASKS * DW_PER_AGENT];
    int n_dw_ffma = 0;
#define ADD_DW(prob) do { if (narrow_chain) dw_ffma[n_dw_ffma++] = (prob); else ADD(prob); } while (0)
    if (group_split) CUR_TRY(tc_chain_presplit_wait(s));
    if (n_e > 1) CUR_TRY(tc_chain_lanes_fork(s));
    FOR_EXPERTS {
      Expert& x = E[i]; const Workspace& w = x.w;
      TcChainIO io;
      memset(&io, 0, sizeof(io));
      io.n = n; io.grad_rows = x.h->loss_rows > 0 ? x.h->loss_rows : n;
      io.mQ = x.mQ; io.mP = x.mP; io.tQ = x.tQ; io.tP = x.tP;
      io.Xpi = w.Xpi; io.Xg = w.Xg; io.XQu = w.XQu; io.Xpi_t = w.Xpi_t; io.Xg_t = w.Xg_t; io.XQpi = w.XQpi; io.XQ_t = w.XQ_t;
      io.ld_spi = w.ld_spi; io.ld_sq = w.ld_sq; io.ld_g = w.ld_g; io.lddy = (int)r4(d->dimu);
      // (the chain keeps hp / hq / dcl / dpl TRANSPOSED, [H][n]: K-major operands of the weight-gradient GEMMs)
      for (int l = 0; l < L; ++l) { io.hp[l] = w.hp[l]; io.hq[l] = w.hq[l]; io.dc[l] = w.dcl[l]; io.dp[l] = w.dpl[l]; }
      io.mp = w.chain_mp; io.mq = w.chain_mq; io.mqp = w.chain_mqp; io.wsplit = w.chain_wsplit;
      io.Q = w.Q; io.Qt = w.Qt; io.dQ = w.dQ; io.dy = w.dy; io.q_pi = x.q_pi; io.r = x.batch->r;
      io.gamma = x.h->gamma; io.clip_return = x.h->clip_return; io.action_l2 = x.h->action_l2; io.clip_pos = x.h->clip_pos_returns;
      io.loss_part = w.chain_loss; io.q_loss = x.q_loss; io.pi_loss = x.pi_loss;
      io.step_counter = x.h->step_counter; io.loss_ring = x.h->loss_ring;
      io.side_ok = n_e == 1 ? 1 : 0;
      io.presplit = group_split ? 1 : 0;
      cudaStream_t cs = s;                         // several experts: independent chains on concurrent streams
      if (n_e > 1) CUR_TRY(tc_chain_lane(i, &cs));
      CUR_TRY(tc_chain_launch(cs, *d, io));
    }
    if (n_e > 1) CUR_TRY(tc_chain_lanes_join(s));
    const int lddy = (int)r4(d->dimu);
    // dW = X^T dY with both operands K-major (K = batch): A = hT [H][n], B = dT [H][n]; first layers: A = X [n][in]
    auto dw_t = [&](const float* XT, int m_rows, const float* DT, float* dW) {
      GemmProb p = zero_prob();
      p.A = XT; p.lda = (int)n; p.a_trans = 0; p.K = (int)n; p.split_k = 2;
      p.B = DT; p.ldb = (int)n; p.b_trans = 1;
      p.C = dW; p.ldc = H; p.M = m_rows; p.N = H;
      return p;
    };
    auto dw_x = [&](const float* X, int ldx, int n_in, const float* DT, float* dW) {
      GemmProb p = zero_prob();
      p.A = X; p.lda = ldx; p.a_trans = 1; p.K = (int)n; p.split_k = 2;
      p.B = DT; p.ldb = (int)n; p.b_trans = 1;
      p.C = dW; p.ldc = H; p.M = n_in; p.N = H;
      return p;
    };
    FOR_EXPERTS {
      Expert& x = E[i]; const Workspace& w = x.w;
      TcRowSumBatch RS;
      RS.n = 0; RS.rows = n;
      auto rowsum = [&](const float* XT, int M, const float* Y, int ldy, int NJ, float* out) {
        TcRowSum& r = RS.p[RS.n++];
        r.XT = XT; r.ld = n; r.Y = Y; r.ldy = ldy; r.NJ = NJ; r.out = out; r.M = M; r.block_begin = 0;
      };
      // main.Q from the critic chain
      rowsum(w.hq[L - 1], H, w.dQ, 1, 1, x.gQ + LQ.off_Wout);                  // dWout = h^T dQ
      rowsum(nullptr, 1, w.dQ, 1, 1, x.gQ + LQ.off_bout);                      // dbout = sum dQ
      for (int l = L - 1; l >= 1; --l) {
        ADD_DW(dw_t(w.hq[l - 1], H, w.dcl[l], x.gQ + LQ.off_W[l]));
        rowsum(w.dcl[l], H, nullptr, 0, 1, x.gQ + LQ.off_b[l]);
      }
      ADD_DW(dw_x(w.XQu, w.ld_sq, LQ.in_s, w.dcl[0], x.gQ + LQ.off_W0));
      rowsum(w.dcl[0], H, nullptr, 0, 1, x.gQ + LQ.off_b0);
      if (LQ.in_g > 0) ADD_DW(dw_x(w.Xg, w.ld_g, LQ.in_g, w.dcl[0], x.gQ + LQ.off_W0g));
      // main.pi from the actor chain
      rowsum(w.hp[L - 1], H, w.dy, lddy, d->dimu, x.gP + LP.off_Wout);
      rowsum(nullptr, 1, w.dy, lddy, d->dimu, x.gP + LP.off_bout);
      for (int l = L - 1; l >= 1; --l) {
        ADD_DW(dw_t(w.hp[l - 1], H, w.dpl[l], x.gP + LP.off_W[l]));
        rowsum(w.dpl[l], H, nullptr, 0, 1, x.gP + LP.off_b[l]);
      }
      ADD_DW(dw_x(w.Xpi, w.ld_spi, LP.in_s, w.dpl[0], x.gP + LP.off_W0));
      rowsum(w.dpl[0], H, nullptr, 0, 1, x.gP + LP.off_b0);
      if (LP.in_g > 0) ADD_DW(dw_x(w.Xg, w.ld_g, LP.in_g, w.dpl[0], x.gP + LP.off_W0g));
      CUR_TRY(tc_chain_rowsums(s, RS));             // side stream: next to the GEMM launches
    }
#undef ADD_DW
    if (narrow_chain) {
      float* parts[CUR_MAX_TASKS];
      for (int i = 0; i < n_e; ++i) parts[i] = E[i].w.chain_dwpart;
      CUR_TRY(chain_dw_ffma(s, dw_ffma, n_dw_ffma / n_e, n_e, n, parts));
    }
    CUR_TRY(B.flush());                             // (the batcher also flushes whenever a launch is full)
    CUR_TRY(B.B.T.finish(s));
    CUR_TRY(tc_chain_join(s));
    return CUR_OK;
  }
  // ---- fwd-1: main.pi | target.pi | main.Q(o,g,u)
  FOR_EXPERTS {
    Expert& x = E[i]; const Workspace& w = x.w;
    ADD(fwd0(LP, x.mP, w.Xpi, w.ld_spi, w.Xg, w.ld_g, w.hp[0], n));
    ADD(fwd0(LP, x.tP, w.Xpi_t, w.ld_spi, w.Xg_t, w.ld_g, w.ht[0], n));
    ADD(fwd0(LQ, x.mQ, w.XQu, w.ld_sq, w.Xg, w.ld_g, w.hq[0], n));
  }
  CUR_TRY(B.flush());
  for (int l = 1; l < L; ++l) {
    FOR_EXPERTS {
      Expert& x = E[i]; const Workspace& w = x.w;
      ADD(fwdl(LP, x.mP, l, w.hp[l - 1], w.hp[l], n));
      ADD(fwdl(LP, x.tP, l, w.ht[l - 1], w.ht[l], n));
      ADD(fwdl(LQ, x.mQ, l, w.hq[l - 1], w.hq[l], n));
    }
    CUR_TRY(B.flush());
  }
  FOR_EXPERTS {
    Expert& x = E[i]; const Workspace& w = x.w;
    ADD(fwdout(LP, x.mP, w.hp[L - 1], x.th, w.ld_sq, EPI_TANH, n));
    ADD(fwdout(LP, x.tP, w.ht[L - 1], w.XQ_t + LP.in_s, w.ld_sq, EPI_TANH, n));
    ADD(fwdout(LQ, x.mQ, w.hq[L - 1], w.Q, 1, EPI_NONE, n));
  }
  CUR_TRY(B.flush());
  // ---- fwd-2: main.Q(o,g,pi) | target.Q(o2,g2,pi_t)   (same u and td for the target, ddpg.py:427-431)
  FOR_EXPERTS {
    Expert& x = E[i]; const Workspace& w = x.w;
    ADD(fwd0(LQ, x.mQ, w.XQpi, w.ld_sq, w.Xg, w.ld_g, w.hqp[0], n));
    ADD(fwd0(LQ, x.tQ, w.XQ_t, w.ld_sq, w.Xg_t, w.ld_g, w.htq[0], n));
  }
  CUR_TRY(B.flush());
  for (int l = 1; l < L; ++l) {
    FOR_EXPERTS {
      Expert& x = E[i]; const Workspace& w = x.w;
      ADD(fwdl(LQ, x.mQ, l, w.hqp[l - 1], w.hqp[l], n));
      ADD(fwdl(LQ, x.tQ, l, w.htq[l - 1], w.htq[l], n));
    }
    CUR_TRY(B.flush());
  }
  FOR_EXPERTS {
    Expert& x = E[i]; const Workspace& w = x.w;
    ADD(fwdout(LQ, x.mQ, w.hqp[L - 1], x.q_pi, 1, EPI_NONE, n));
    ADD(fwdout(LQ, x.tQ, w.htq[L - 1], w.Qt, 1, EPI_NONE, n));
  }
  CUR_TRY(B.flush());

  // ---- losses and backward seeds
  FOR_EXPERTS {
    Expert& x = E[i]; const Workspace& w = x.w;
    LossParams LPm;
    LPm.r = x.batch->r; LPm.Q = w.Q; LPm.Qpi = x.q_pi; LPm.Qt = w.Qt; LPm.th = x.th; LPm.ldth = w.ld_sq; LPm.dimu = d->dimu;
    LPm.n = n; LPm.gamma = x.h->gamma; LPm.clip_return = x.h->clip_return; LPm.action_l2 = x.h->action_l2;
    LPm.clip_pos = x.h->clip_pos_returns; LPm.dQ = w.dQ; LPm.dQpi = w.dQpi; LPm.q_loss = x.q_loss; LPm.pi_loss = x.pi_loss;
    LPm.step_counter = x.h->step_counter; LPm.ring = x.h->loss_ring;
    LPm.grad_rows = x.h->loss_rows > 0 ? x.h->loss_rows : n;
    if (n >= LOSS_MC_MIN_BATCH) {
      LossMcParams MC;
      MC.L = LPm; MC.part = w.loss_part; MC.ticket = w.loss_ticket;
      int ctas = (int)((n + 511) / 512);
      if (ctas > LOSS_MAX_CTAS) ctas = LOSS_MAX_CTAS;
      loss_mc_kernel<<<ctas, 512, 0, s>>>(MC);
    } else {
      loss_kernel<<<1, 1024, 0, s>>>(LPm);
    }
    CUR_CHECK_LAUNCH();
  }

  // ---- bwd-1: critic chain (weights grads of main/Q) | actor-through-Q chain (data grads only)
  int cur = 0;
  FOR_EXPERTS {
    Expert& x = E[i]; const Workspace& w = x.w;
    ADD(bwd_dx(w.dQ, 1, x.mQ + LQ.off_Wout, H, 1, w.hq[L - 1], H, w.dc[0], H, n));
    ADD(bwd_dw(w.hq[L - 1], H, H, w.dQ, 1, 1, x.gQ + LQ.off_Wout, n));
    ADD(bwd_db(w.dQ, 1, 1, x.gQ + LQ.off_bout, n));
    ADD(bwd_dx(w.dQpi, 1, x.mQ + LQ.off_Wout, H, 1, w.hqp[L - 1], H, w.da[0], H, n));
  }
  CUR_TRY(B.flush());
  for (int l = L - 1; l >= 1; --l) {
    FOR_EXPERTS {
      Expert& x = E[i]; const Workspace& w = x.w;
      ADD(bwd_dx(w.dc[cur], H, x.mQ + LQ.off_W[l], H, H, w.hq[l - 1], H, w.dc[cur ^ 1], H, n));
      ADD(bwd_dw(w.hq[l - 1], H, H, w.dc[cur], H, H, x.gQ + LQ.off_W[l], n));
      ADD(bwd_db(w.dc[cur], H, H, x.gQ + LQ.off_b[l], n));
      ADD(bwd_dx(w.da[cur], H, x.mQ + LQ.off_W[l], H, H, w.hqp[l - 1], H, w.da[cur ^ 1], H, n));
    }
    CUR_TRY(B.flush());
    cur ^= 1;
  }
  FOR_EXPERTS {
    Expert& x = E[i]; const Workspace& w = x.w;
    ADD(bwd_dw(w.XQu, w.ld_sq, LQ.in_s, w.dc[cur], H, H, x.gQ + LQ.off_W0, n));
    ADD(bwd_db(w.dc[cur], H, H, x.gQ + LQ.off_b0, n));
    if (LQ.in_g > 0) ADD(bwd_dw(w.Xg, w.ld_g, LQ.in_g, w.dc[cur], H, H, x.gQ + LQ.off_W0g, n));
    // d pi_loss / d(pre-tanh) = (dL/d(pi/max_u) + action_l2 * 2/(B*dimu) * th) * (1 - th^2)
    GemmProb p = bwd_dx(w.da[cur], H, x.mQ + LQ.off_W0 + (int64_t)LP.in_s * H, d->dimu, H, nullptr, 0, w.dy,
                        (int)r4(d->dimu), n);
    p.epi = EPI_ACTOR_DY; p.aux = x.th; p.ldaux = w.ld_sq;
    p.coef = x.h->action_l2 * 2.0f / (float)((x.h->loss_rows > 0 ? x.h->loss_rows : n) * d->dimu);
    ADD(p);
  }
  CUR_TRY(B.flush());
  // ---- bwd-2: actor chain (weight grads of main/pi)
  const int lddy = (int)r4(d->dimu);
  cur = 0;
  FOR_EXPERTS {
    Expert& x = E[i]; const Workspace& w = x.w;
    ADD(bwd_dx(w.dy, lddy, x.mP + LP.off_Wout, H, d->dimu, w.hp[L - 1], H, w.dp[0], H, n));
    ADD(bwd_dw(w.hp[L - 1], H, H, w.dy, lddy, d->dimu, x.gP + LP.off_Wout, n));
    ADD(bwd_db(w.dy, lddy, d->dimu, x.gP + LP.off_bout, n));
  }
  CUR_TRY(B.flush());
  for (int l = L - 1; l >= 1; --l) {
    FOR_EXPERTS {
      Expert& x = E[i]; const Workspace& w = x.w;
      ADD(bwd_dx(w.dp[cur], H, x.mP + LP.off_W[l], H, H, w.hp[l - 1], H, w.dp[cur ^ 1], H, n));
      ADD(bwd_dw(w.hp[l - 1], H, H, w.dp[cur], H, H, x.gP + LP.off_W[l], n));
      ADD(bwd_db(w.dp[cur], H, H, x.gP + LP.off_b[l], n));
    }
    CUR_TRY(B.flush());
    cur ^= 1;
  }
  FOR_EXPERTS {
    Expert& x = E[i]; const Workspace& w = x.w;
    ADD(bwd_dw(w.Xpi, w.ld_spi, LP.in_s, w.dp[cur], H, H, x.gP + LP.off_W0, n));
    ADD(bwd_db(w.dp[cur], H, H, x.gP + LP.off_b0, n));
    if (LP.in_g > 0) ADD(bwd_dw(w.Xg, w.ld_g, LP.in_g, w.dp[cur], H, H, x.gP + LP.off_W0g, n));
  }
  CUR_TRY(B.flush());
  CUR_TRY(B.B.T.finish(s));               // deferred reductions of the last levels -> gradients complete on `s`
#undef FOR_EXPERTS
#undef ADD
  return CUR_OK;
}

static int fill_expert(Expert& x, const cur_net_desc* d, const float* theta_main, const float* theta_target,
                       const cur_norm_stats* stats, const cur_batch* batch, const cur_ddpg_hyper* h, float* workspace,
                       float* grads, float* q_loss, float* pi_loss, float* q_pi, bool narrow_chain = false) {
  CUR_REQUIRE(theta_main && theta_target && batch && h && workspace && grads && q_pi, "NULL argument");
  CUR_REQUIRE(batch->o && batch->g && batch->u && batch->o_2 && batch->g_2 && batch->r, "NULL batch array");
  CUR_REQUIRE(!d->modular || batch->td, "task_descr required for a modular net");
  CUR_REQUIRE(batch->n > 0 && batch->n < (1 << 30), "bad batch");
  if (d->normalize_obs)
    CUR_REQUIRE(stats && stats->o_mean && stats->o_std && stats->g_mean && stats->g_std, "normalizer stats required");
  const int64_t offP = r4(net_layout(*d, 0).total);
  x.w = carve(*d, batch->n, workspace, narrow_chain);
  x.mQ = theta_main; x.mP = theta_main + offP; x.tQ = theta_target; x.tP = theta_target + offP;
  x.gQ = grads; x.gP = grads + offP;
  x.batch = batch; x.stats = stats; x.h = h; x.q_loss = q_loss; x.pi_loss = pi_loss; x.q_pi = q_pi;
  x.th = nullptr; x.parts_used = x.rowparts_used = 0;
  return CUR_OK;
}

extern "C" int cur_ddpg_grads(void* stream, const cur_net_desc* d, const float* theta_main,
                              const float* theta_target, const cur_norm_stats* stats, const cur_batch* batch,
                              const cur_ddpg_hyper* h, float* workspace, float* grads, float* q_loss,
                              float* pi_loss, float* q_pi) {
  CUR_TRY(check_desc(d));
  Expert x;
  CUR_TRY(fill_expert(x, d, theta_main, theta_target, stats, batch, h, workspace, grads, q_loss, pi_loss, q_pi));
  return grads_levels((cudaStream_t)stream, d, &x, 1, batch->n);
}

extern "C" int cur_ddpg_grads_group(void* stream, const cur_net_desc* d, int n_experts, const cur_ddpg_expert* experts) {
  CUR_TRY(check_desc(d));
  CUR_REQUIRE(experts != nullptr && n_experts >= 1 && n_experts <= CUR_MAX_TASKS, "bad expert list");
  Expert E[CUR_MAX_TASKS];
  for (int i = 0; i < n_experts; ++i) {
    const cur_ddpg_expert& a = experts[i];
    CUR_REQUIRE(a.batch.n == experts[0].batch.n, "all experts must train on the same batch size");
    CUR_TRY(fill_expert(E[i], d, a.theta_main, a.theta_target, a.has_stats ? &a.stats : nullptr, &a.batch, &a.hyper,
                        a.workspace, a.grads, a.q_loss, a.pi_loss, a.q_pi));
  }
  return grads_levels((cudaStream_t)stream, d, E, n_experts, experts[0].batch.n);
}

extern "C" int cur_ddpg_chain_supported(const cur_net_desc* d, int64_t batch) {
  if (check_desc(d) != CUR_OK || batch <= 0) return 0;
  if (d->hidden == 256) return use_chain(*d, batch) ? 1 : 0;
  return narrow_chain_ok(*d, batch) ? 1 : 0;
}

extern "C" int64_t cur_ddpg_chain_workspace_floats(const cur_net_desc* d, int64_t batch) {
  if (check_desc(d) != CUR_OK || batch <= 0) return -1;
  return carve(*d, batch, nullptr, true).total;
}

extern "C" int cur_ddpg_chain_grads(void* stream, const cur_net_desc* d, const float* theta_main,
                                    const float* theta_target, const cur_norm_stats* stats, const cur_batch* batch,
                                    const cur_ddpg_hyper* h, float* workspace, float* grads, float* q_loss,
                                    float* pi_loss, float* q_pi) {
  CUR_TRY(check_desc(d));
  CUR_REQUIRE(batch != nullptr && cur_ddpg_chain_supported(d, batch->n), "shape not taken by the chain schedule");
  Expert x;
  CUR_TRY(fill_expert(x, d, theta_main, theta_target, stats, batch, h, workspace, grads, q_loss, pi_loss, q_pi, true));
  return grads_levels((cudaStream_t)stream, d, &x, 1, batch->n, d->hidden < 256);
}

extern "C" int cur_ddpg_chain_grads_group(void* stream, const cur_net_desc* d, int n_experts,
                                          const cur_ddpg_expert* experts) {
  CUR_TRY(check_desc(d));
  CUR_REQUIRE(d->hidden < 256, "hidden-256 experts reach the chain schedule through cur_ddpg_grads_group");
  CUR_REQUIRE(experts != nullptr && n_experts >= 1 && n_experts <= CUR_MAX_TASKS, "bad expert list");
  const int64_t n = experts[0].batch.n;
  CUR_REQUIRE(cur_ddpg_chain_supported(d, n), "shape not taken by the chain schedule");
  for (int i = 1; i < n_experts; ++i)
    CUR_REQUIRE(experts[i].batch.n == n, "all experts must train on the same batch size");
  Expert E[CUR_MAX_TASKS];
  for (int i = 0; i < n_experts; ++i) {
    const cur_ddpg_expert& a = experts[i];
    CUR_TRY(fill_expert(E[i], d, a.theta_main, a.theta_target, a.has_stats ? &a.stats : nullptr, &a.batch, &a.hyper,
                        a.workspace, a.grads, a.q_loss, a.pi_loss, a.q_pi, true));
  }
  return grads_levels((cudaStream_t)stream, d, E, n_experts, n, true);
}
