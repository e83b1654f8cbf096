// DDPG / UVFA update at large batch: the whole actor or critic CHAIN of one 128-row tile in ONE CTA on the 5th-generation
// tensor cores (sm_100a) - forward nets, losses, backward (dX) chains - with the activations never leaving the SM
// between layers.
//
// Replaces (reference flowersteam/curious), for batches of 512 rows and more (BASELINE configs 4 and 5: the 19-worker
// job, the per-GPU batch sweep):
//   baselines/her/actor_critic.py:5-98, util.py:56-107   networks (forward)
//   baselines/her/ddpg.py:412-449                        losses + the data-gradient half of tf.gradients
// The weight gradients (dW = X^T dY, K = batch) follow as split-K tcgen05 GEMMs (tc_gemm.cu) on the activations /
// deltas this kernel leaves in the workspace; at hidden 64 / 128 (the kernel is a template on the width H, every `256`
// below reads H) as K-sliced FFMA grouped GEMMs (ddpg.cu: chain_dw_ffma).
//
// Why: rows of the batch are independent until dW (the insight behind the rows schedule, ddpg_rows.cu), but that
// schedule re-streams all weights per 4 rows (cost grows linearly with the rows), and the dependency-level schedule
// (ddpg.cu) pays ~16 us of launch / prologue / epilogue / global round trip per level x 17 levels.  Here a CTA owns 128
// rows and one chain.  Per layer it streams the weight matrix ONCE as ready-made 3xTF32 halves (x = hi + lo, split once
// per update by tc_chain_presplit_kernel: 2 x 32 KB per 32-k block through a 2-stage TMA ring - a first version split the
// raw tile in shared memory with four warps and sat at the 128 B/clk shared-memory limit, 304 KB of traffic per
// k-block) and issues tcgen05.mma M=128 N=256 K=8 (hi*hi + lo*hi + hi*lo) into a TMEM accumulator; the NEXT layer's A
// operand is produced straight from that accumulator: eight "feeder" warps (two per TMEM lane quarter taking alternate
// 32-column chunks, thread = batch row) read the accumulator with tcgen05.ld, apply bias / ReLU (forward) or the ReLU
// mask (backward), keep the copy the weight-gradient GEMMs need - TRANSPOSED, [256 units][n rows], so that a warp
// (32 consecutive rows) writes one full 128-byte line per unit instead of 32 partial lines (measured: row-major
// 16-byte-per-lane stores cost ~1 k cycles of L1 transactions per chunk) - and the ReLU masks as one 32-bit word per row
// and chunk, split the values into hi / lo and write them as the next k-block of the A operand in the K-major
// 128-byte-swizzled layout the MMA descriptors expect.  Layer l + 1 accumulates into the other half of TMEM (2 x 256
// columns, ping-pong) while layer l's accumulator is being drained chunk by chunk, so feeders, TMA and tensor pipe
// overlap across the layer boundary.  Output layers (N = 1 / dimu), tanh, the TD / actor losses and the backward seeds
// are per-row dot products inside the feeder threads (partial over the chunks of a warp pair, combined through 2 KB of
// shared memory in fixed order).
//
//   warp 0      TMA producer (weights, the B operand): cp.async.bulk.tensor.2d into the B ring, mbarrier complete_tx
//   warp 1      MMA issuer (one lane), owns the TMEM allocation; tcgen05.commit frees A / B stages, publishes accumulators
//   warps 2-9   feeders (A operand + everything row-wise), see above
//
// Even CTAs run the actor chain (main.pi -> main.Q(o,g,pi) -> actor loss -> backward through main.Q and main.pi), odd
// CTAs the critic chain (target.pi -> target.Q -> main.Q(o,g,u) -> TD loss -> backward through main.Q); nothing is
// exchanged between them.  One accumulator per layer (main and cross terms together): 7.8e-7 of sum|a||b| at K = 256
// instead of 3.0e-7 with two (DESIGN.md 3.3) - the price of the ping-pong that hides the accumulator drain.
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include "net_layout.cuh"
#include "tc_gemm.cuh"
#include "tc_ptx.cuh"

namespace cur {

// The hidden width H (64, 128 or 256) is the N of every tcgen05.mma and a template parameter of the kernel and of the
// feeder helpers; everything else (128 rows per CTA, the rings, the warp roles, 3xTF32) is the same at every width.
constexpr int CH_BM = 128, CH_BK = 32;
constexpr int CH_A_HALF = CH_BM * CH_BK * 4;              // 16 KB: one k-block of the A operand (hi or lo)
constexpr int CH_A_STAGE = 2 * CH_A_HALF;                 // hi | lo
constexpr int CH_NA = 2, CH_NB = 2;                       // ring depths: 64 KB + 2 x 2 x 16 H bytes (A: one stage per feeder parity)
constexpr int CH_MNBLK = 32 * 128;                        // bytes of one 32-wide N block of an MN-major weight tile
constexpr int CH_WARP_FEED0 = 2, CH_FEED_WARPS = 8;
constexpr int CH_THREADS = (CH_WARP_FEED0 + CH_FEED_WARPS) * 32;     // 320
constexpr int CH_MAX_GEMM = 16, CH_MAX_MAPS = 40;         // (hi, lo) map pairs
template <int H>
struct ChW {
  static_assert(H == 64 || H == 128 || H == 256, "hidden widths of the chain kernel");
  static constexpr int B_HALF = H * CH_BK * 4;            // one k-block of the B operand (hi or lo): 32 x H
  static constexpr int B_STAGE = 2 * B_HALF;              // hi | lo
  static constexpr size_t SMEM_BYTES = (size_t)CH_NA * CH_A_STAGE + (size_t)CH_NB * B_STAGE + 1024 /* alignment */ + 256;
  static constexpr int NCH = H / 32;                      // 32-column chunks of a layer output
  static constexpr int VEC_FLOATS = 3 * 4 * H + 2 * 4 * H + 2 * H;   // 3 nets x <= 4 biases, 2 x [H][4], 2 x [H]
};

struct ChGemm {
  int map1, nkb1, map2, nkb2;     // weight tensor maps (hi; lo = + 1) of the (up to two) K segments, their k-block counts
  int b_mn;                       // 1: weights stored [K][N] (forward), 0: stored [N][K] (dX = dY W^T)
};
struct ChProg {
  int n;
  ChGemm g[CH_MAX_GEMM];
};

struct __align__(64) ChainParams {
  CUtensorMap maps[2][CH_MAX_MAPS];
  ChProg prog[2];                 // [0] actor chain, [1] critic chain
  cur_net_desc d;
  int L, in_sp, in_sq, in_g, ld_spi, ld_sq, ld_g, lddy;
  int64_t n, grad_rows;
  const float *Xpi, *Xg, *XQu, *XQpi, *Xpi_t, *Xg_t, *XQ_t;
  const float *bP[CUR_MAX_LAYERS], *bPT[CUR_MAX_LAYERS], *bQ[CUR_MAX_LAYERS], *bQT[CUR_MAX_LAYERS];
  const float *WoutP, *boutP, *WoutPT, *boutPT, *WoutQ, *boutQ, *WoutQT, *boutQT;
  const float* W0Q_act;           // main.Q first-layer rows of the action inputs: [dimu][H]
  // transposed copies [H][n] for the weight-gradient GEMMs: activations (hp, hq) and deltas (dc, dp)
  float *hp[CUR_MAX_LAYERS], *hq[CUR_MAX_LAYERS], *dc[CUR_MAX_LAYERS], *dp[CUR_MAX_LAYERS];
  // ReLU masks [layer][chunk][n] (H / 32 chunks), bit i of a word = unit 32 chunk + i is active
  uint32_t *mp, *mq, *mqp;
  float *Q, *Qt, *dQ, *dy, *q_pi;
  const float* r;
  float gamma, clip_return, action_l2;
  int clip_pos;
  float* loss_part;               // [tiles][4]: ssq (critic), sum Q_pi, sum th^2 (actor)
  long long* tl;                  // debug timeline (clock64 stamps of CTA 0 / 1), normally NULL
  int dbg;                        // measurement switches (CUR_CHAIN_DBG): 1 no transposed copies, 2 masks all ones
};

// ---------------------------------------------------------------------------------------------------- feeder
struct Feeder {
  uint8_t* a_gen;                 // generic address of the A ring
  float (*s_x)[4];                // [128][4] exchange buffer of the warp pairs
  uint32_t a_full, a_empty, acc_full;
  uint32_t tmem_lane;             // TMEM address of this thread's lane, column 0
  int lane, r, par;               // lane in warp, row in tile, parity of the k-blocks / chunks this warp takes
  int64_t row;                    // batch row
  int a_cnt;                      // k-blocks of the A operand so far (both parities count all of them)
  long long* tl;                  // debug stamps (first feeder warp, lane 0) or NULL
  int dbg;
  int n_stamp;
  __device__ __forceinline__ void stamp() { if (tl && n_stamp < 100) tl[400 + n_stamp++] = clock64(); }

  __device__ __forceinline__ bool mine() const { return (a_cnt & 1) == par; }
  __device__ __forceinline__ void wait_acc(int g) const {
    tc_bar_wait(acc_full + 8 * (g & 1), (uint32_t)(g >> 1) & 1u);
    tc_fence_after();
  }
  // 32 accumulator columns of GEMM g, chunk c, for this thread's row (accumulators g & 1 = 0 / 1 at columns 0 / H)
  template <int H>
  __device__ __forceinline__ void ld_chunk(int g, int c, float (&v)[32]) const {
    uint32_t x[32];
    tc_ld32(tmem_lane + (uint32_t)((g & 1) * H + c * 32), x);
    tc_ld_wait();
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(x[i]);
  }
  // the next k-block of the A operand (it must be `mine()`): this thread's row of 32 values, split, K-major SWIZZLE_128B
  __device__ __forceinline__ void push_A(const float (&v)[32]) {
    const int s = a_cnt % CH_NA, round = a_cnt / CH_NA;
    if (round > 0) tc_bar_wait(a_empty + 8 * s, (uint32_t)(round - 1) & 1u);
    float* hi = reinterpret_cast<float*>(a_gen + s * CH_A_STAGE);
    float* lo = hi + CH_A_HALF / 4;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      float4 h, l;
      tc_split1(v[4 * c], h.x, l.x); tc_split1(v[4 * c + 1], h.y, l.y);
      tc_split1(v[4 * c + 2], h.z, l.z); tc_split1(v[4 * c + 3], h.w, l.w);
      const int off = r * 32 + ((c ^ (r & 7)) << 2);
      *reinterpret_cast<float4*>(hi + off) = h;
      *reinterpret_cast<float4*>(lo + off) = l;
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();
    if (tl && a_cnt < 88) tl[96 + a_cnt] = clock64();
    if (lane == 0) tc_bar_arrive(a_full + 8 * s);
    ++a_cnt;
  }
  // Partial per-row sums of the two warps of a lane quarter -> the same total in both (fixed order: parity 0 + parity 1)
  template <int NJ>
  __device__ __forceinline__ void combine(float (&out)[NJ]) const {
    if (par == 1) {
#pragma unroll
      for (int j = 0; j < NJ; ++j) s_x[r][j] = out[j];
    }
    asm volatile("bar.sync 3, 256;" ::: "memory");
    if (par == 0) {
#pragma unroll
      for (int j = 0; j < NJ; ++j) { out[j] += s_x[r][j]; s_x[r][j] = out[j]; }
    }
    asm volatile("bar.sync 3, 256;" ::: "memory");
    if (par == 1) {
#pragma unroll
      for (int j = 0; j < NJ; ++j) out[j] = s_x[r][j];
    }
  }
};

__device__ __forceinline__ void ch_load32(const float* src, float (&v)[32]) {
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const float4 x = *reinterpret_cast<const float4*>(src + 4 * q);
    v[4 * q] = x.x; v[4 * q + 1] = x.y; v[4 * q + 2] = x.z; v[4 * q + 3] = x.w;
  }
}
// transposed copy: unit 32 c + i of this thread's row -> T[(32 c + i) * n + row]; the 32 lanes of a warp write one line
__device__ __forceinline__ void ch_store_t(float* T, int64_t n, int64_t row, int c, const float (&v)[32]) {
  float* dst = T + (int64_t)(32 * c) * n + row;
#pragma unroll
  for (int i = 0; i < 32; ++i) dst[(int64_t)i * n] = v[i];
}
__device__ __forceinline__ uint32_t ch_mask_word(const float (&v)[32]) {
  uint32_t w = 0;
#pragma unroll
  for (int i = 0; i < 32; ++i) w |= (v[i] > 0.f ? 1u : 0u) << i;
  return w;
}
// A operand of a first layer: k-blocks of the thread's row of a prepared input matrix X [n][ld] (columns >= kcols are 0);
// columns [a0, a0 + na) are taken from `act` (the tanh output of the policy net just evaluated) instead
__device__ __forceinline__ void ch_feed_x(Feeder& F, const float* X, int ld, int kcols, int a0, int na, const float (&act)[4]) {
  const int nkb = (kcols + CH_BK - 1) / CH_BK;
  const float* xr = X + F.row * ld;
#pragma unroll 1
  for (int kb = 0; kb < nkb; ++kb) {
    if (!F.mine()) { ++F.a_cnt; continue; }
    float v[32];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const int k = kb * CH_BK + 4 * q;
      float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
      if (k < ld) x = *reinterpret_cast<const float4*>(xr + k);          // ld is a multiple of 4
      v[4 * q] = k < kcols ? x.x : 0.f; v[4 * q + 1] = k + 1 < kcols ? x.y : 0.f;
      v[4 * q + 2] = k + 2 < kcols ? x.z : 0.f; v[4 * q + 3] = k + 3 < kcols ? x.w : 0.f;
    }
    if (na > 0 && a0 < (kb + 1) * CH_BK && a0 + na > kb * CH_BK) {
#pragma unroll
      for (int i = 0; i < 32; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (j < na && kb * CH_BK + i == a0 + j) v[i] = act[j];
    }
    F.push_A(v);
  }
}

// Forward hidden layer boundary: h = relu(acc(g) + bias) -> mask word, optional transposed copy -> A operand of the next GEMM
template <int H>
__device__ __forceinline__ void ch_feed_relu(Feeder& F, int g, const float* bias, float* HT, uint32_t* mask,
                                             int64_t n) {
  F.wait_acc(g);
#pragma unroll 1
  for (int c = 0; c < ChW<H>::NCH; ++c) {
    if (!F.mine()) { ++F.a_cnt; continue; }
    float v[32], b[32];
    ch_load32(bias + 32 * c, b);
    F.ld_chunk<H>(g, c, v);
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i] + b[i], 0.f);
    if (mask) mask[(int64_t)c * n + F.row] = ch_mask_word(v);
    if (HT && !(F.dbg & 1)) ch_store_t(HT, n, F.row, c, v);
    F.push_A(v);
  }
}

// Output layer on the last hidden activation: h = relu(acc(g) + bias) (mask word, optional transposed copy),
// out[j] = sum_c h[c] Wout[c][j] (the chunks of this warp's parity, then combined over the warp pair)
template <int H, int NJMAX>
__device__ __forceinline__ void ch_out_layer(Feeder& F, int g, const float* bias, float* HT, uint32_t* mask,
                                             int64_t n, const float* Wout, int nj, float (&out)[NJMAX]) {
#pragma unroll
  for (int j = 0; j < NJMAX; ++j) out[j] = 0.f;
  F.wait_acc(g);
#pragma unroll 1
  for (int c = F.par; c < ChW<H>::NCH; c += 2) {
    float v[32], b[32];
    ch_load32(bias + 32 * c, b);
    F.ld_chunk<H>(g, c, v);
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = fmaxf(v[i] + b[i], 0.f);
    if (mask) mask[(int64_t)c * n + F.row] = ch_mask_word(v);
    if (HT && !(F.dbg & 1)) ch_store_t(HT, n, F.row, c, v);
    if (NJMAX == 1) {
      float w[32];
      ch_load32(Wout + 32 * c, w);
#pragma unroll
      for (int i = 0; i < 32; ++i) out[0] = fmaf(v[i], w[i], out[0]);
    } else if (nj == 4) {
      // one broadcast 16-byte load per hidden unit: Wout[c][0..3]
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const float4 w = *(reinterpret_cast<const float4*>(Wout) + 32 * c + i);
        out[0] = fmaf(v[i], w.x, out[0]); out[1] = fmaf(v[i], w.y, out[1]);
        out[2] = fmaf(v[i], w.z, out[2]); out[3] = fmaf(v[i], w.w, out[3]);
      }
    } else {
#pragma unroll
      for (int i = 0; i < 32; ++i)
#pragma unroll
        for (int j = 0; j < NJMAX; ++j)
          if (j < nj) out[j] = fmaf(v[i], Wout[(32 * c + i) * nj + j], out[j]);
    }
  }
  F.combine<NJMAX>(out);
}

// Backward seed through an output layer: d[c] = (sum_j dout[j] Wout[c][j]) where the mask word says the unit is active
// -> optional transposed copy -> A
template <int H, int NJMAX>
__device__ __forceinline__ void ch_seed(Feeder& F, const float (&dout)[NJMAX], int nj, const float* Wout,
                                        const uint32_t* mask, float* DT, int64_t n) {
#pragma unroll 1
  for (int c = 0; c < ChW<H>::NCH; ++c) {
    if (!F.mine()) { ++F.a_cnt; continue; }
    float v[32];
    const uint32_t mw = (F.dbg & 2) ? 0xFFFFFFFFu : mask[(int64_t)c * n + F.row];
    if (NJMAX == 1) {
      float w[32];
      ch_load32(Wout + 32 * c, w);
#pragma unroll
      for (int i = 0; i < 32; ++i) v[i] = ((mw >> i) & 1u) ? dout[0] * w[i] : 0.f;
    } else if (nj == 4) {
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const float4 w = *(reinterpret_cast<const float4*>(Wout) + 32 * c + i);
        const float s = fmaf(dout[3], w.w, fmaf(dout[2], w.z, fmaf(dout[1], w.y, dout[0] * w.x)));
        v[i] = ((mw >> i) & 1u) ? s : 0.f;
      }
    } else {
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        float s = 0.f;
#pragma unroll
        for (int j = 0; j < NJMAX; ++j)
          if (j < nj) s = fmaf(dout[j], Wout[(32 * c + i) * nj + j], s);
        v[i] = ((mw >> i) & 1u) ? s : 0.f;
      }
    }
    if (DT && !(F.dbg & 1)) ch_store_t(DT, n, F.row, c, v);
    F.push_A(v);
  }
}

// Backward hidden layer boundary: d = acc(g) where the mask word says the unit was active -> optional transposed copy ->
// (optionally) A of the next GEMM
template <int H>
__device__ __forceinline__ void ch_feed_mask(Feeder& F, int g, const uint32_t* mask, float* DT, int64_t n, bool push) {
  F.wait_acc(g);
#pragma unroll 1
  for (int c = 0; c < ChW<H>::NCH; ++c) {
    if (push ? !F.mine() : ((c & 1) != F.par)) {
      if (push) ++F.a_cnt;
      continue;
    }
    float v[32];
    const uint32_t mw = (F.dbg & 2) ? 0xFFFFFFFFu : mask[(int64_t)c * n + F.row];
    F.ld_chunk<H>(g, c, v);
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = ((mw >> i) & 1u) ? v[i] : 0.f;
    if (DT && !(F.dbg & 1)) ch_store_t(DT, n, F.row, c, v);
    if (push) F.push_A(v);
  }
}

// sum over the 128 rows of the tile in fixed order (warp shuffle tree, then the 4 warps of parity 0 in order); called by
// the parity-0 feeder warps only
__device__ __forceinline__ float ch_tile_sum(float x, float* s_red, int fw, int lane) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  asm volatile("bar.sync 2, 128;" ::: "memory");
  if (lane == 0) s_red[fw] = x;
  asm volatile("bar.sync 2, 128;" ::: "memory");
  return (s_red[0] + s_red[1]) + (s_red[2] + s_red[3]);
}

template <int H>
__global__ void __launch_bounds__(CH_THREADS, 1) tc_chain_kernel(const __grid_constant__ ChainParams P) {
  using W = ChW<H>;
  extern __shared__ uint8_t ch_smem_raw[];
  __shared__ uint32_t s_tmem;
  __shared__ float s_red[4];
  __shared__ float s_x[CH_BM][4];
  __shared__ __align__(16) float s_vec[W::VEC_FLOATS];   // biases / output-layer weights of this chain (see `stage`)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int role = blockIdx.x & 1;                      // 0: actor chain, 1: critic chain
  const int tile = blockIdx.x >> 1;
  const ChProg& prog = P.prog[role];
  const cur_net_desc& d = P.d;
  const int L = P.L;

  const uint32_t base = (tc_smem(ch_smem_raw) + 1023u) & ~1023u;
  uint8_t* gen_base = ch_smem_raw + (base - tc_smem(ch_smem_raw));
  const uint32_t a_ring = base, b_ring = base + CH_NA * CH_A_STAGE;
  const uint32_t bars = b_ring + CH_NB * W::B_STAGE;
  const uint32_t a_full = bars, a_empty = bars + 8 * CH_NA, b_full = bars + 16 * CH_NA, b_empty = b_full + 8 * CH_NB,
                 acc_full = b_full + 16 * CH_NB;
  long long* tl = (P.tl != nullptr && tile == 0 && lane == 0) ? P.tl + 512 * role : nullptr;   // [role][512] stamps
  if (tl && warp == 0) tl[0] = clock64();

  if (threadIdx.x == 0) {
    for (int s = 0; s < CH_NA; ++s) { tc_bar_init(a_full + 8 * s, CH_FEED_WARPS / 2); tc_bar_init(a_empty + 8 * s, 1); }
    for (int s = 0; s < CH_NB; ++s) { tc_bar_init(b_full + 8 * s, 1); tc_bar_init(b_empty + 8 * s, 1); }
    tc_bar_init(acc_full, 1); tc_bar_init(acc_full + 8, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tc_smem(&s_tmem)), "n"(2 * H) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = s_tmem;

  if (warp == 0) {
    // =============================================================== TMA producer: the weight tiles (hi, lo) of every GEMM
    if (lane == 0) {
      int cnt = 0;
      for (int g = 0; g < prog.n; ++g) {
        const ChGemm G = prog.g[g];
        const int nkb = G.nkb1 + G.nkb2;
        for (int kb = 0; kb < nkb; ++kb, ++cnt) {
          const int s = cnt % CH_NB, round = cnt / CH_NB;
          if (round > 0) tc_bar_wait(b_empty + 8 * s, (uint32_t)(round - 1) & 1u);
          const uint32_t dst = b_ring + s * W::B_STAGE;
          const bool seg2 = kb >= G.nkb1;
          const CUtensorMap* mh = &P.maps[role][seg2 ? G.map2 : G.map1];
          const CUtensorMap* ml = mh + 1;
          const int k0 = (seg2 ? kb - G.nkb1 : kb) * CH_BK;
          if (tl && cnt < 88) tl[288 + cnt] = clock64();
          tc_bar_expect_tx(b_full + 8 * s, W::B_STAGE);                // zero-filled out-of-bounds rows count too
          if (G.b_mn) {
            for (int j = 0; j < H / 32; ++j) {                                                                 // [32 k][32 n]
              tc_tma_2d(dst + j * CH_MNBLK, mh, 32 * j, k0, b_full + 8 * s);
              tc_tma_2d(dst + W::B_HALF + j * CH_MNBLK, ml, 32 * j, k0, b_full + 8 * s);
            }
          } else {
            tc_tma_2d(dst, mh, k0, 0, b_full + 8 * s);                                                         // [H n][32 k]
            tc_tma_2d(dst + W::B_HALF, ml, k0, 0, b_full + 8 * s);
          }
        }
      }
    }
  } else if (warp == 1) {
    // =============================================================== MMA issuer
    int cnt = 0;
    for (int g = 0; g < prog.n; ++g) {
      const ChGemm G = prog.g[g];
      const int nkb = G.nkb1 + G.nkb2;
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)G.b_mn << 16) | ((uint32_t)(H >> 3) << 17) |
                             ((uint32_t)(CH_BM >> 4) << 24);
      const uint32_t b_step = G.b_mn ? 1024u : 32u, b_lbo = G.b_mn ? (uint32_t)CH_MNBLK : 16u, b_sbo = G.b_mn ? 512u : 1024u,
                     b_lt = G.b_mn ? 1u : 2u;
      const uint32_t acc = tmem + (uint32_t)((g & 1) * H);
      for (int kb = 0; kb < nkb; ++kb, ++cnt) {
        const int sa = cnt % CH_NA, ra = cnt / CH_NA, sb = cnt % CH_NB, rb = cnt / CH_NB;
        tc_bar_wait(b_full + 8 * sb, (uint32_t)rb & 1u);
        tc_bar_wait(a_full + 8 * sa, (uint32_t)ra & 1u);
        tc_fence_after();
        if (lane == 0) {
          if (tl && cnt < 88) tl[8 + cnt] = clock64();
          const uint32_t a_hi = a_ring + sa * CH_A_STAGE, a_lo = a_hi + CH_A_HALF;
          const uint32_t b_hi = b_ring + sb * W::B_STAGE, b_lo = b_hi + W::B_HALF;
#pragma unroll
          for (int ks = 0; ks < CH_BK / 8; ++ks) {
            const uint64_t dah = tc_desc(a_hi + ks * 32, 16u, 1024u, 2u), dal = tc_desc(a_lo + ks * 32, 16u, 1024u, 2u);
            const uint64_t dbh = tc_desc(b_hi + ks * b_step, b_lbo, b_sbo, b_lt), dbl = tc_desc(b_lo + ks * b_step, b_lbo, b_sbo, b_lt);
            tc_mma_tf32(acc, dal, dbh, idesc, (kb | ks) != 0);        // cross terms first, the main term on top
            tc_mma_tf32(acc, dah, dbl, idesc, 1u);
            tc_mma_tf32(acc, dah, dbh, idesc, 1u);
          }
          tc_commit(a_empty + 8 * sa);
          tc_commit(b_empty + 8 * sb);
          if (kb == nkb - 1) tc_commit(acc_full + 8 * (g & 1));
        }
        __syncwarp();
      }
    }
  } else {
    // =============================================================== feeders: thread = batch row, two warps per lane quarter
    Feeder F;
    const int q = warp & 3;                               // a warp may only touch TMEM lanes 32 (warp % 4) .. + 31
    F.par = (warp - CH_WARP_FEED0) >> 2;
    const int fw = (warp - CH_WARP_FEED0) & 3;            // index among the warps of its parity
    F.a_gen = gen_base;
    F.s_x = s_x;
    F.a_full = a_full; F.a_empty = a_empty; F.acc_full = acc_full;
    F.lane = lane; F.r = 32 * q + lane;
    F.tmem_lane = tmem + ((uint32_t)(32 * q) << 16);
    F.row = (int64_t)tile * CH_BM + F.r;
    F.a_cnt = 0;
    F.dbg = P.dbg;
    F.n_stamp = 0;
    F.tl = (tl && warp == CH_WARP_FEED0) ? tl : nullptr;
    const int64_t row = F.row, n = P.n;
    const bool lead = F.par == 0;                         // the warp of a pair that writes the per-row results
    const float inv_n = 1.0f / (float)P.grad_rows;
    const float none[4] = {0.f, 0.f, 0.f, 0.f};
#define MW(l) ((int64_t)(l) * W::NCH * n)            /* mask words of layer l */
    int g = 0;                                            // index of the GEMM whose accumulator is read next
    // The small vectors every row needs (biases, output-layer weights) go to shared memory once: read from global per
    // chunk they cost an exposed L2 round trip each (measured 0.6 - 1.5 k cycles per chunk in the output-layer passes).
    int v_off = 0;
    const int ft = threadIdx.x - CH_WARP_FEED0 * 32;
    auto stage = [&](const float* src, int count) -> const float* {
      float* dst = s_vec + v_off;
      for (int i = ft; i < count; i += CH_FEED_WARPS * 32) dst[i] = __ldg(src + i);
      v_off += (count + 3) & ~3;
      return dst;
    };
    const float *sbA[CUR_MAX_LAYERS], *sbB[CUR_MAX_LAYERS], *sbC[CUR_MAX_LAYERS];
    if (role == 0) {
      // ---------------- actor chain: main.pi (the first A operand goes out before anything else: the tensor pipe starts)
      ch_feed_x(F, P.Xpi, P.ld_spi, P.in_sp, 0, 0, none);
      if (P.in_g > 0) ch_feed_x(F, P.Xg, P.ld_g, P.in_g, 0, 0, none);
      for (int l = 0; l < L; ++l) sbA[l] = stage(P.bP[l], H);
      const float* sWoutP = stage(P.WoutP, H * d.dimu);
      for (int l = 0; l < L; ++l) sbB[l] = stage(P.bQ[l], H);
      const float* sWoutQ = stage(P.WoutQ, H);
      const float* sW0act = stage(P.W0Q_act, d.dimu * H);
      asm volatile("bar.sync 3, 256;" ::: "memory");
      for (int l = 1; l < L; ++l, ++g) ch_feed_relu<H>(F, g, sbA[l - 1], P.hp[l - 1], P.mp + MW(l - 1), n);
      float th[4];
      ch_out_layer<H, 4>(F, g, sbA[L - 1], P.hp[L - 1], P.mp + MW(L - 1), n, sWoutP, d.dimu, th);
      ++g;
      float sth = 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        th[j] = j < d.dimu ? tanhf(th[j] + __ldg(P.boutP + j)) : 0.f;       // actor_critic.py:89 (pi / max_u)
        sth += th[j] * th[j];
      }
      // ---------------- main.Q(o, g, pi): the action columns of the input come from `th`
      ch_feed_x(F, P.XQpi, P.ld_sq, P.in_sq, P.in_sp, d.dimu, th);
      if (P.in_g > 0) ch_feed_x(F, P.Xg, P.ld_g, P.in_g, 0, 0, none);
      for (int l = 1; l < L; ++l, ++g) ch_feed_relu<H>(F, g, sbB[l - 1], nullptr, P.mqp + MW(l - 1), n);
      float qv[1];
      ch_out_layer<H, 1>(F, g, sbB[L - 1], nullptr, P.mqp + MW(L - 1), n, sWoutQ, 1, qv);
      ++g;
      const float q_pi = qv[0] + __ldg(P.boutQ);
      if (lead) {
        P.q_pi[row] = q_pi;
        // ---------------- actor loss terms (ddpg.py:440-441), per-tile partial sums in fixed order
        const float sq = ch_tile_sum(q_pi, s_red, fw, lane);
        const float st = ch_tile_sum(sth, s_red, fw, lane);
        if (fw == 0 && lane == 0) { P.loss_part[4 * tile + 1] = sq; P.loss_part[4 * tile + 2] = st; }
      }
      // ---------------- backward through main.Q (actor-through-critic chain, data gradients only)
      {
        float dq[1] = {-inv_n};                                            // d(-mean(Q_pi)) / dQ_pi
        ch_seed<H, 1>(F, dq, 1, sWoutQ, P.mqp + MW(L - 1), nullptr, n);
      }
      for (int l = L - 1; l >= 2; --l, ++g) ch_feed_mask<H>(F, g, P.mqp + MW(l - 1), nullptr, n, true);
      // gradient wrt the action inputs: d h0 (masked) . W0[action rows]^T, then through tanh and the action penalty
      float dy[4] = {0.f, 0.f, 0.f, 0.f};
      F.wait_acc(g);
#pragma unroll 1
      for (int c = F.par; c < ChW<H>::NCH; c += 2) {
        float v[32];
        const uint32_t mw = (F.dbg & 2) ? 0xFFFFFFFFu : P.mqp[(int64_t)c * n + row];
        F.ld_chunk<H>(g, c, v);
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = ((mw >> i) & 1u) ? v[i] : 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (j < d.dimu) {
            float w[32];
            ch_load32(sW0act + j * H + 32 * c, w);
#pragma unroll
            for (int i = 0; i < 32; ++i) dy[j] = fmaf(v[i], w[i], dy[j]);
          }
        }
      }
      ++g;
      F.combine<4>(dy);
      {
        const float coef = P.action_l2 * 2.0f / (float)(P.grad_rows * d.dimu);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          dy[j] = j < d.dimu ? (dy[j] + coef * th[j]) * (1.f - th[j] * th[j]) : 0.f;
          if (lead && j < P.lddy) P.dy[row * P.lddy + j] = dy[j];
        }
      }
      // ---------------- backward through main.pi
      ch_seed<H, 4>(F, dy, d.dimu, sWoutP, P.mp + MW(L - 1), P.dp[L - 1], n);
      for (int l = L - 1; l >= 1; --l, ++g) ch_feed_mask<H>(F, g, P.mp + MW(l - 1), P.dp[l - 1], n, l >= 2);
    } else {
      // ---------------- critic chain: target.pi
      ch_feed_x(F, P.Xpi_t, P.ld_spi, P.in_sp, 0, 0, none);
      if (P.in_g > 0) ch_feed_x(F, P.Xg_t, P.ld_g, P.in_g, 0, 0, none);
      for (int l = 0; l < L; ++l) sbA[l] = stage(P.bPT[l], H);
      const float* sWoutPT = stage(P.WoutPT, H * d.dimu);
      for (int l = 0; l < L; ++l) sbB[l] = stage(P.bQT[l], H);
      const float* sWoutQT = stage(P.WoutQT, H);
      for (int l = 0; l < L; ++l) sbC[l] = stage(P.bQ[l], H);
      const float* sWoutQ = stage(P.WoutQ, H);
      asm volatile("bar.sync 3, 256;" ::: "memory");
      for (int l = 1; l < L; ++l, ++g) ch_feed_relu<H>(F, g, sbA[l - 1], nullptr, nullptr, n);
      float th[4];
      ch_out_layer<H, 4>(F, g, sbA[L - 1], nullptr, nullptr, n, sWoutPT, d.dimu, th);
      ++g;
#pragma unroll
      for (int j = 0; j < 4; ++j) th[j] = j < d.dimu ? tanhf(th[j] + __ldg(P.boutPT + j)) : 0.f;
      // ---------------- target.Q(o_2, g_2, pi_target) with the same td (ddpg.py:427-431)
      ch_feed_x(F, P.XQ_t, P.ld_sq, P.in_sq, P.in_sp, d.dimu, th);
      if (P.in_g > 0) ch_feed_x(F, P.Xg_t, P.ld_g, P.in_g, 0, 0, none);
      for (int l = 1; l < L; ++l, ++g) ch_feed_relu<H>(F, g, sbB[l - 1], nullptr, nullptr, n);
      float qt[1];
      ch_out_layer<H, 1>(F, g, sbB[L - 1], nullptr, nullptr, n, sWoutQT, 1, qt);
      ++g;
      const float q_t = qt[0] + __ldg(P.boutQT);
      // ---------------- main.Q(o, g, u)
      ch_feed_x(F, P.XQu, P.ld_sq, P.in_sq, 0, 0, none);
      if (P.in_g > 0) ch_feed_x(F, P.Xg, P.ld_g, P.in_g, 0, 0, none);
      for (int l = 1; l < L; ++l, ++g) ch_feed_relu<H>(F, g, sbC[l - 1], P.hq[l - 1], P.mq + MW(l - 1), n);
      float qv[1];
      ch_out_layer<H, 1>(F, g, sbC[L - 1], P.hq[L - 1], P.mq + MW(L - 1), n, sWoutQ, 1, qv);
      ++g;
      const float q = qv[0] + __ldg(P.boutQ);
      // ---------------- TD loss (ddpg.py:436-439) and its backward seed
      const float hi_clip = P.clip_pos ? 0.f : INFINITY;
      const float tgt = fminf(fmaxf(P.r[row] + P.gamma * q_t, -P.clip_return), hi_clip);
      const float diff = tgt - q;
      float dq[1] = {-2.0f * inv_n * diff};                                // d mean((tgt - Q)^2) / dQ
      if (lead) {
        P.Qt[row] = q_t; P.Q[row] = q; P.dQ[row] = dq[0];
        const float ssq = ch_tile_sum(diff * diff, s_red, fw, lane);
        if (fw == 0 && lane == 0) P.loss_part[4 * tile] = ssq;
      }
      // ---------------- backward through main.Q (critic chain)
      ch_seed<H, 1>(F, dq, 1, sWoutQ, P.mq + MW(L - 1), P.dc[L - 1], n);
      for (int l = L - 1; l >= 1; --l, ++g) ch_feed_mask<H>(F, g, P.mq + MW(l - 1), P.dc[l - 1], n, l >= 2);
    }
#undef MW
    tc_fence_before();
  }
  __syncthreads();
  if (tl && warp == 0) tl[1] = clock64();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(2 * H) : "memory");
  }
}

// Once per update: every parameter of the four nets as the two TF32 halves of 3xTF32 (tc_ptx.cuh: tc_split1), laid out
// like the parameter arenas themselves: out = [main hi | main lo | target hi | target lo], `arena` floats each
__device__ __forceinline__ void ch_presplit(const float* __restrict__ theta_main, const float* __restrict__ theta_target,
                                            float* __restrict__ out, int64_t arena4) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 2 * arena4) return;
  const bool tgt = i >= arena4;
  const int64_t k = tgt ? i - arena4 : i;
  const float4 x = reinterpret_cast<const float4*>(tgt ? theta_target : theta_main)[k];
  float4 h, l;
  tc_split1(x.x, h.x, l.x); tc_split1(x.y, h.y, l.y); tc_split1(x.z, h.z, l.z); tc_split1(x.w, h.w, l.w);
  float4* o = reinterpret_cast<float4*>(out) + (tgt ? 2 * arena4 : 0);
  o[k] = h;
  o[arena4 + k] = l;
}
__global__ void __launch_bounds__(256) tc_chain_presplit_kernel(const float* __restrict__ theta_main,
                                                                 const float* __restrict__ theta_target, float* __restrict__ out,
                                                                 int64_t arena4) {
  ch_presplit(theta_main, theta_target, out, arena4);
}
// the same for several experts of one shape, expert = blockIdx.y, each into its own buffer
struct ChainPresplitGroup {
  const float* mQ[CUR_MAX_TASKS];
  const float* tQ[CUR_MAX_TASKS];
  float* out[CUR_MAX_TASKS];
  int64_t arena4;
};
__global__ void __launch_bounds__(256) tc_chain_presplit_group_kernel(const __grid_constant__ ChainPresplitGroup P) {
  const int e = blockIdx.y;
  ch_presplit(P.mQ[e], P.tQ[e], P.out[e], P.arena4);
}

// per-tile loss partials -> Q_loss / pi_loss (ring slot of the device step counter), fixed order; bumps the counter
struct ChainLossParams {
  const float* part;
  int tiles, dimu, ring;
  int64_t n;
  float action_l2;
  float *q_loss, *pi_loss;
  int64_t* step_counter;
};
__global__ void __launch_bounds__(32) tc_chain_loss_kernel(const __grid_constant__ ChainLossParams P) {
  // lane l folds tiles l, l + 32, ... in order, then a fixed shuffle tree
  float ssq = 0.f, sq = 0.f, sth = 0.f;
  for (int t = threadIdx.x; t < P.tiles; t += 32) { ssq += P.part[4 * t]; sq += P.part[4 * t + 1]; sth += P.part[4 * t + 2]; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ssq += __shfl_xor_sync(0xffffffffu, ssq, o);
    sq += __shfl_xor_sync(0xffffffffu, sq, o);
    sth += __shfl_xor_sync(0xffffffffu, sth, o);
  }
  if (threadIdx.x != 0) return;
  long long slot = 0;
  if (P.step_counter) {
    const long long st = *P.step_counter;
    slot = P.ring > 0 ? st % P.ring : 0;
    *P.step_counter = st + 1;
  }
  const float inv_n = 1.0f / (float)P.n;
  if (P.q_loss) P.q_loss[slot] = ssq * inv_n;                                                // ddpg.py:439
  if (P.pi_loss) P.pi_loss[slot] = -sq * inv_n + P.action_l2 * sth / (float)(P.n * P.dimu);   // ddpg.py:440-441
}

// Row sums over the batch of the TRANSPOSED copies (bias gradients, output-layer weight gradients; K = batch):
//   out[m * NJ + j] = sum_r XT[m][r] * Y[r][j]   (Y == NULL: plain row sums; XT == NULL: ones, i.e. column sums of Y)
// One CTA per output row m, fixed summation order (thread t takes r = t, t + 256, ...; fixed-order fold).
__global__ void __launch_bounds__(256) tc_chain_rowsum_kernel(const __grid_constant__ TcRowSumBatch R) {
  __shared__ float red[256][4];
  int pi = 0;
#pragma unroll 1
  while (pi + 1 < R.n && (int)blockIdx.x >= R.p[pi + 1].block_begin) ++pi;
  const TcRowSum& P = R.p[pi];
  const int m = blockIdx.x - P.block_begin;
  const float* x = P.XT ? P.XT + (int64_t)m * P.ld : nullptr;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  if (x != nullptr && P.Y == nullptr) {
    // plain row sum: 16-byte loads (rows is a multiple of 128, every row of XT starts 16-byte aligned)
    for (int64_t r = 4 * (int64_t)threadIdx.x; r < R.rows; r += 1024) {
      const float4 v = *reinterpret_cast<const float4*>(x + r);
      acc[0] += (v.x + v.y) + (v.z + v.w);
    }
  } else {
    for (int64_t r = threadIdx.x; r < R.rows; r += 256) {
      const float xv = x ? x[r] : 1.f;
      if (P.Y) {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (j < P.NJ) acc[j] = fmaf(xv, P.Y[r * P.ldy + j], acc[j]);
      } else {
        acc[0] += xv;
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) red[threadIdx.x][j] = acc[j];
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) {
#pragma unroll
      for (int j = 0; j < 4; ++j) red[threadIdx.x][j] += red[threadIdx.x + o][j];
    }
    __syncthreads();
  }
  if ((int)threadIdx.x < P.NJ) P.out[(int64_t)m * P.NJ + threadIdx.x] = red[0][threadIdx.x];
}

// The row sums only depend on the chain kernel's outputs: they run on a side stream next to the weight-gradient GEMMs
// (fork / join with events - capturable, inside a CUDA graph the two become parallel branches).
struct ChainSide {
  cudaStream_t stream = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
  cudaEvent_t fork0 = nullptr, split_done = nullptr;   // the weight split runs beside the input preparation
  int device = -1;
  bool pending = false;
  bool split_pending = false;                          // tc_chain_presplit_async ran: tc_chain_launch waits instead of splitting
  bool loss_deferred = false;                          // the loss fold of the last chain launch goes with the row sums
  ChainLossParams loss;
};
static int chain_side(ChainSide** out) {
  static thread_local ChainSide ss;
  int dev = 0;
  CUR_CUDA_TRY(cudaGetDevice(&dev));
  if (ss.stream == nullptr || ss.device != dev) {
    CUR_CUDA_TRY(cudaStreamCreateWithFlags(&ss.stream, cudaStreamNonBlocking));
    CUR_CUDA_TRY(cudaEventCreateWithFlags(&ss.fork, cudaEventDisableTiming));
    CUR_CUDA_TRY(cudaEventCreateWithFlags(&ss.join, cudaEventDisableTiming));
    CUR_CUDA_TRY(cudaEventCreateWithFlags(&ss.fork0, cudaEventDisableTiming));
    CUR_CUDA_TRY(cudaEventCreateWithFlags(&ss.split_done, cudaEventDisableTiming));
    ss.device = dev;
    ss.pending = false;
    ss.split_pending = false;
    ss.loss_deferred = false;
  }
  *out = &ss;
  return CUR_OK;
}

// Several agents (task_experts): the chain kernels of different experts are independent and one expert's tiles do not
// fill the GPU, so expert i launches on lane i % 4; fork once before the first, join after the last.
constexpr int CH_LANES = 4;
struct ChainLanes {
  cudaStream_t stream[CH_LANES] = {nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t fork = nullptr, done[CH_LANES] = {nullptr, nullptr, nullptr, nullptr};
  bool used[CH_LANES] = {false, false, false, false};
  int device = -1;
};
static int chain_lanes(ChainLanes** out) {
  static thread_local ChainLanes L;
  int dev = 0;
  CUR_CUDA_TRY(cudaGetDevice(&dev));
  if (L.fork == nullptr || L.device != dev) {
    for (int i = 0; i < CH_LANES; ++i) {
      CUR_CUDA_TRY(cudaStreamCreateWithFlags(&L.stream[i], cudaStreamNonBlocking));
      CUR_CUDA_TRY(cudaEventCreateWithFlags(&L.done[i], cudaEventDisableTiming));
      L.used[i] = false;
    }
    CUR_CUDA_TRY(cudaEventCreateWithFlags(&L.fork, cudaEventDisableTiming));
    L.device = dev;
  }
  *out = &L;
  return CUR_OK;
}
int tc_chain_lanes_fork(cudaStream_t s) {
  ChainLanes* L = nullptr;
  CUR_TRY(chain_lanes(&L));
  CUR_CUDA_TRY(cudaEventRecord(L->fork, s));
  for (int i = 0; i < CH_LANES; ++i) L->used[i] = false;
  return CUR_OK;
}
int tc_chain_lane(int i, cudaStream_t* out) {
  ChainLanes* L = nullptr;
  CUR_TRY(chain_lanes(&L));
  const int k = i % CH_LANES;
  if (!L->used[k]) {
    CUR_CUDA_TRY(cudaStreamWaitEvent(L->stream[k], L->fork, 0));
    L->used[k] = true;
  }
  *out = L->stream[k];
  return CUR_OK;
}
int tc_chain_lanes_join(cudaStream_t s) {
  ChainLanes* L = nullptr;
  CUR_TRY(chain_lanes(&L));
  for (int k = 0; k < CH_LANES; ++k) {
    if (!L->used[k]) continue;
    CUR_CUDA_TRY(cudaEventRecord(L->done[k], L->stream[k]));
    CUR_CUDA_TRY(cudaStreamWaitEvent(s, L->done[k], 0));
    L->used[k] = false;
  }
  return CUR_OK;
}

int tc_chain_rowsums(cudaStream_t s, TcRowSumBatch& R) {
  if (R.n == 0) return CUR_OK;
  int blocks = 0;
  for (int i = 0; i < R.n; ++i) { R.p[i].block_begin = blocks; blocks += R.p[i].M; }
  ChainSide* ss = nullptr;
  CUR_TRY(chain_side(&ss));
  CUR_CUDA_TRY(cudaEventRecord(ss->fork, s));
  CUR_CUDA_TRY(cudaStreamWaitEvent(ss->stream, ss->fork, 0));
  if (ss->loss_deferred) {                       // the loss fold only needs the chain kernel's partials: off the GEMM's path
    tc_chain_loss_kernel<<<1, 32, 0, ss->stream>>>(ss->loss);
    CUR_CHECK_LAUNCH();
    ss->loss_deferred = false;
  }
  tc_chain_rowsum_kernel<<<blocks, 256, 0, ss->stream>>>(R);
  CUR_CHECK_LAUNCH();
  CUR_CUDA_TRY(cudaEventRecord(ss->join, ss->stream));
  ss->pending = true;
  return CUR_OK;
}

// the caller's stream waits for the row sums launched since the last join
int tc_chain_join(cudaStream_t s) {
  ChainSide* ss = nullptr;
  CUR_TRY(chain_side(&ss));
  if (ss->pending) {
    CUR_CUDA_TRY(cudaStreamWaitEvent(s, ss->join, 0));
    ss->pending = false;
  }
  return CUR_OK;
}

// ---------------------------------------------------------------------------------------------------- host side
bool tc_chain_width_supported(const cur_net_desc& d, int64_t n) {
  if ((d.hidden != 64 && d.hidden != 128 && d.hidden != 256) || n < CH_BM || (n % CH_BM) != 0 || d.dimu > 4 ||
      d.layers < 2 || d.layers > 4)
    return false;
  const NetLayout q = net_layout(d, 0), p = net_layout(d, 1);
  if ((q.in_s + 31) / 32 + (q.in_g + 31) / 32 > 8) return false;
  // TMA: 16-byte aligned rows and bases of every weight block
  if ((q.off_W0 % 4) || (q.off_W0g % 4) || (p.off_W0 % 4) || (p.off_W0g % 4)) return false;
  for (int l = 1; l < d.layers; ++l)
    if ((q.off_W[l] % 4) || (p.off_W[l] % 4)) return false;
  return n / CH_BM <= (1 << 20);
}
bool tc_chain_supported(const cur_net_desc& d, int64_t n) { return d.hidden == 256 && tc_chain_width_supported(d, n); }

// The 3xTF32 halves of the weights only depend on the previous update: split them on the side stream while the caller's
// stream prepares the inputs (call before the input preparation is launched; tc_chain_launch then waits for the event).
int tc_chain_presplit_async(cudaStream_t s, const float* mQ, const float* tQ, float* wsplit, int64_t arena) {
  ChainSide* ss = nullptr;
  CUR_TRY(chain_side(&ss));
  CUR_CUDA_TRY(cudaEventRecord(ss->fork0, s));
  CUR_CUDA_TRY(cudaStreamWaitEvent(ss->stream, ss->fork0, 0));
  const int64_t arena4 = arena / 4;
  tc_chain_presplit_kernel<<<(unsigned)((2 * arena4 + 255) / 256), 256, 0, ss->stream>>>(mQ, tQ, wsplit, arena4);
  CUR_CHECK_LAUNCH();
  CUR_CUDA_TRY(cudaEventRecord(ss->split_done, ss->stream));
  ss->split_pending = true;
  return CUR_OK;
}

int tc_chain_presplit_group_async(cudaStream_t s, int n_e, const float* const* mQ, const float* const* tQ,
                                  float* const* wsplit, int64_t arena) {
  CUR_REQUIRE(n_e >= 1 && n_e <= CUR_MAX_TASKS, "bad expert count");
  ChainSide* ss = nullptr;
  CUR_TRY(chain_side(&ss));
  ChainPresplitGroup P;
  for (int i = 0; i < n_e; ++i) { P.mQ[i] = mQ[i]; P.tQ[i] = tQ[i]; P.out[i] = wsplit[i]; }
  P.arena4 = arena / 4;
  CUR_CUDA_TRY(cudaEventRecord(ss->fork0, s));
  CUR_CUDA_TRY(cudaStreamWaitEvent(ss->stream, ss->fork0, 0));
  tc_chain_presplit_group_kernel<<<dim3((unsigned)((2 * P.arena4 + 255) / 256), (unsigned)n_e), 256, 0, ss->stream>>>(P);
  CUR_CHECK_LAUNCH();
  CUR_CUDA_TRY(cudaEventRecord(ss->split_done, ss->stream));
  ss->split_pending = true;
  return CUR_OK;
}

int tc_chain_presplit_wait(cudaStream_t s) {
  ChainSide* ss = nullptr;
  CUR_TRY(chain_side(&ss));
  if (ss->split_pending) {
    CUR_CUDA_TRY(cudaStreamWaitEvent(s, ss->split_done, 0));
    ss->split_pending = false;
  }
  return CUR_OK;
}

static long long* g_chain_timeline = nullptr;
void tc_chain_set_timeline(long long* dev) { g_chain_timeline = dev; }

template <int H>
static int ch_kernel_launch(cudaStream_t s, int tiles, const ChainParams& P) {
  static bool configured = false;
  if (!configured) {
    CUR_CUDA_TRY(cudaFuncSetAttribute(tc_chain_kernel<H>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)ChW<H>::SMEM_BYTES));
    configured = true;
  }
  tc_chain_kernel<H><<<2 * tiles, CH_THREADS, ChW<H>::SMEM_BYTES, s>>>(P);
  CUR_CHECK_LAUNCH();
  return CUR_OK;
}

int tc_chain_launch(cudaStream_t s, const cur_net_desc& d, const TcChainIO& io) {
  CUR_REQUIRE(tc_chain_width_supported(d, io.n), "shape not supported by the chain kernel");
  const NetLayout LQ = net_layout(d, 0), LP = net_layout(d, 1);
  const int L = d.layers, H = d.hidden;
  static thread_local ChainParams P;                      // 12 KB: kept off the stack; rebuilt on every call
  memset(&P.prog, 0, sizeof(P.prog));
  P.d = d; P.L = L;
  P.in_sp = LP.in_s; P.in_sq = LQ.in_s; P.in_g = LQ.in_g;
  P.ld_spi = io.ld_spi; P.ld_sq = io.ld_sq; P.ld_g = io.ld_g; P.lddy = io.lddy;
  P.n = io.n; P.grad_rows = io.grad_rows;
  P.Xpi = io.Xpi; P.Xg = io.Xg; P.XQu = io.XQu; P.Xpi_t = io.Xpi_t; P.Xg_t = io.Xg_t; P.XQpi = io.XQpi; P.XQ_t = io.XQ_t;
  const float *mQ = io.mQ, *mP = io.mP, *tQ = io.tQ, *tP = io.tP;
  for (int l = 0; l < CUR_MAX_LAYERS; ++l) {
    const bool on = l < L;
    const int64_t bq = (l == 0) ? LQ.off_b0 : LQ.off_b[l], bp = (l == 0) ? LP.off_b0 : LP.off_b[l];
    P.bP[l] = on ? mP + bp : nullptr; P.bPT[l] = on ? tP + bp : nullptr;
    P.bQ[l] = on ? mQ + bq : nullptr; P.bQT[l] = on ? tQ + bq : nullptr;
    P.hp[l] = on ? io.hp[l] : nullptr; P.hq[l] = on ? io.hq[l] : nullptr;
    P.dc[l] = on ? io.dc[l] : nullptr; P.dp[l] = on ? io.dp[l] : nullptr;
  }
  P.WoutP = mP + LP.off_Wout; P.boutP = mP + LP.off_bout; P.WoutPT = tP + LP.off_Wout; P.boutPT = tP + LP.off_bout;
  P.WoutQ = mQ + LQ.off_Wout; P.boutQ = mQ + LQ.off_bout; P.WoutQT = tQ + LQ.off_Wout; P.boutQT = tQ + LQ.off_bout;
  P.W0Q_act = mQ + LQ.off_W0 + (int64_t)LP.in_s * H;
  P.mp = io.mp; P.mq = io.mq; P.mqp = io.mqp;
  P.Q = io.Q; P.Qt = io.Qt; P.dQ = io.dQ; P.dy = io.dy; P.q_pi = io.q_pi; P.r = io.r;
  P.gamma = io.gamma; P.clip_return = io.clip_return; P.action_l2 = io.action_l2; P.clip_pos = io.clip_pos;
  P.loss_part = io.loss_part;
  P.tl = g_chain_timeline;
  static const int dbg = getenv("CUR_CHAIN_DBG") ? atoi(getenv("CUR_CHAIN_DBG")) : 0;
  P.dbg = dbg;

  // ---- the weights as 3xTF32 halves, once per call (the weights change with every update)
  const int64_t arena = r4(LQ.total) + r4(LP.total);
  CUR_REQUIRE(io.wsplit != nullptr && io.mP == io.mQ + r4(LQ.total) && io.tP == io.tQ + r4(LQ.total), "parameter arenas expected");
  ChainSide* side = nullptr;
  CUR_TRY(chain_side(&side));
  if (io.presplit) {
    // split by tc_chain_presplit_group_async; the launch stream forked after tc_chain_presplit_wait
  } else if (io.side_ok && side->split_pending) {
    CUR_CUDA_TRY(cudaStreamWaitEvent(s, side->split_done, 0));      // split by tc_chain_presplit_async
    side->split_pending = false;
  } else {
    const int64_t arena4 = arena / 4;
    tc_chain_presplit_kernel<<<(unsigned)((2 * arena4 + 255) / 256), 256, 0, s>>>(io.mQ, io.tQ, io.wsplit, arena4);
    CUR_CHECK_LAUNCH();
  }
  // ---- the GEMM programs and their weight tensor maps (pairs: hi, lo)
  int n_maps[2] = {0, 0};
  auto map_pair = [&](int role, const float* w, int64_t rows, int box_rows, bool mn) -> int {
    const bool is_target = (w >= io.tQ && w < io.tQ + arena);
    const int64_t off = is_target ? w - io.tQ : w - io.mQ;
    CUR_REQUIRE(off >= 0 && off < arena && n_maps[role] + 2 <= CH_MAX_MAPS, "bad weight block");
    const float* hi = io.wsplit + (is_target ? 2 * arena : 0) + off;
    CUR_TRY(tc_make_map(&P.maps[role][n_maps[role]++], hi, rows, H, H, box_rows, mn));
    CUR_TRY(tc_make_map(&P.maps[role][n_maps[role]++], hi + arena, rows, H, H, box_rows, mn));
    return CUR_OK;
  };
  auto fwd_net = [&](int role, const float* th, const NetLayout& NL) -> int {
    ChProg& pr = P.prog[role];
    ChGemm& g0 = pr.g[pr.n++];
    g0.b_mn = 1;
    g0.map1 = n_maps[role]; g0.nkb1 = (NL.in_s + CH_BK - 1) / CH_BK;
    CUR_TRY(map_pair(role, th + NL.off_W0, NL.in_s, CH_BK, true));
    g0.map2 = 0; g0.nkb2 = 0;
    if (NL.in_g > 0) {
      g0.map2 = n_maps[role]; g0.nkb2 = (NL.in_g + CH_BK - 1) / CH_BK;
      CUR_TRY(map_pair(role, th + NL.off_W0g, NL.in_g, CH_BK, true));
    }
    for (int l = 1; l < L; ++l) {
      ChGemm& g = pr.g[pr.n++];
      g.b_mn = 1; g.map1 = n_maps[role]; g.nkb1 = H / CH_BK; g.map2 = 0; g.nkb2 = 0;
      CUR_TRY(map_pair(role, th + NL.off_W[l], H, CH_BK, true));
    }
    return CUR_OK;
  };
  auto bwd_net = [&](int role, const float* th, const NetLayout& NL) -> int {   // dX through W_{L-1} .. W_1
    ChProg& pr = P.prog[role];
    for (int l = L - 1; l >= 1; --l) {
      ChGemm& g = pr.g[pr.n++];
      g.b_mn = 0; g.map1 = n_maps[role]; g.nkb1 = H / CH_BK; g.map2 = 0; g.nkb2 = 0;
      CUR_TRY(map_pair(role, th + NL.off_W[l], H, H, false));
    }
    return CUR_OK;
  };
  static_assert(3 * 4 + 3 <= CH_MAX_GEMM && 2 * (6 + 4 * 3) <= CH_MAX_MAPS, "programs of up to 4 hidden layers fit");
  CUR_TRY(fwd_net(0, mP, LP)); CUR_TRY(fwd_net(0, mQ, LQ)); CUR_TRY(bwd_net(0, mQ, LQ)); CUR_TRY(bwd_net(0, mP, LP));
  CUR_TRY(fwd_net(1, tP, LP)); CUR_TRY(fwd_net(1, tQ, LQ)); CUR_TRY(fwd_net(1, mQ, LQ)); CUR_TRY(bwd_net(1, mQ, LQ));
  CUR_REQUIRE(P.prog[0].n <= CH_MAX_GEMM && P.prog[1].n <= CH_MAX_GEMM, "chain program too long");

  const int tiles = (int)(io.n / CH_BM);
  if (H == 64) CUR_TRY(ch_kernel_launch<64>(s, tiles, P));
  else if (H == 128) CUR_TRY(ch_kernel_launch<128>(s, tiles, P));
  else CUR_TRY(ch_kernel_launch<256>(s, tiles, P));
  ChainLossParams LPm;
  LPm.part = io.loss_part; LPm.tiles = tiles; LPm.dimu = d.dimu; LPm.ring = io.loss_ring; LPm.n = io.n;
  LPm.action_l2 = io.action_l2; LPm.q_loss = io.q_loss; LPm.pi_loss = io.pi_loss; LPm.step_counter = io.step_counter;
  if (io.side_ok) {                              // one agent on the caller's stream: the fold travels with the row sums
    side->loss = LPm;
    side->loss_deferred = true;
  } else {
    tc_chain_loss_kernel<<<1, 32, 0, s>>>(LPm);
    CUR_CHECK_LAUNCH();
  }
  return CUR_OK;
}

}  // namespace cur

// debug: `device_buffer` = 1024 x int64 (clock64 stamps of the first actor / critic CTA: [role][512] = start, end,
// [8..) MMA issue, [96..) A stage ready (first feeder warp: its parity only), [288..) TMA issue per k-block), or NULL
extern "C" int cur_tc_chain_timeline(long long* device_buffer_1024) {
  cur::tc_chain_set_timeline(device_buffer_1024);
  return CUR_OK;
}
