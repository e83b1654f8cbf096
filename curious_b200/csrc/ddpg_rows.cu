// DDPG / UVFA update, "rows" schedule (sm_100a): the whole actor-critic graph of one update in TWO launches
// (three when the optimiser is not fused).
//
// Replaces (reference flowersteam/curious), like ddpg.cu but with a latency-oriented schedule:
//   baselines/her/actor_critic.py:5-98, util.py:56-107   networks
//   baselines/her/ddpg.py:412-449                        losses + tf.gradients + flatten_grads
//   baselines/common/mpi_adam.py:30-35                   Adam (fused into the weight-gradient launch)
//
// Why: at the reference batch (256 rows, 3x256 MLPs) one update is 0.73 GFLOP - ~10 us of FFMA - but the
// dependency-level schedule of ddpg.cu needs 17 dependent launches (140 us).  Rows of the batch are
// independent until the weight gradient, so the data path is run "decode style":
//
//   launch 0  transpose_kernel   W_l^T of the hidden layers of main.Q / main.pi (operands of the backward
//             streams), 0.5 MB.  Only when the optimiser is NOT fused into launch 2: the fused Adam epilogue
//             writes the transposed copy of every stepped hidden-layer tile itself (cur_adam_fused.transposes_valid).
//   launch 1  ddpg_stream_kernel two independent CTAs per 4 batch rows, no inter-CTA communication at all:
//               actor CTA   main.pi -> main.Q(o,g,pi) -> actor loss -> backward through main.Q and main.pi
//               critic CTA  target.pi -> target.Q -> main.Q(o,g,u) -> TD loss -> critic backward through main.Q
//             Each CTA walks its whole chain for its rows while a producer warp streams every weight matrix it
//             needs (2.2 / 2.3 MB per update) from L2 through a 4 x 32 KB shared-memory ring with TMA bulk copies
//             (cp.async.bulk + mbarrier full/empty pairs).  8 consumer warps do GEMV-like FFMA: a thread owns 4
//             output columns and a quarter of the chunk's k rows, reads W as LDS.128 and the (transposed)
//             activations as one broadcast LDS.128 per k; activations never leave shared memory between
//             layers.  History (profiles/README.md): column split over an 8-CTA cluster with a per-layer
//             exchange (lost to the synchronisation), one CTA for everything, main / target CTA pair with
//             main.Q streamed once for 8 stacked rows (FFMA-bound passes, idle target CTA), this split; round 2:
//             ddpg_stream_pair_kernel, the columns of every layer split over a 2-CTA cluster (half the weight
//             bytes per SM, st.async exchange through distributed shared memory) - correct, slower, opt-in.
//   launch 2  rows_dw_kernel     every dW = X^T dY and db = 1^T dY of both nets as one grouped GEMM with
//             the full batch as K (deterministic, no atomics), written into the flat GetFlat-ordered
//             gradient arena; optionally Adam is applied to the element in the same epilogue (world
//             size 1: no all-reduce between gradient and step).  One extra CTA without a tile folds the
//             per-CTA loss partials and bumps the device step counter beside the tiles.
//
// All arithmetic is FP32 FFMA (IEEE); see DESIGN.md section 4 for why tensor cores do not apply here.
// The stream and action kernels are instantiated for hidden 64, 128 and 256 (Width<H>); the numbers above are for 256.
#include <stdlib.h>

#include "her_device.cuh"
#include "net_layout.cuh"
#include "tc_gemm.cuh"
#include "tc_ptx.cuh"

namespace cur {

constexpr int S_ROWS = 4;                // batch rows per CTA
constexpr int S_H = 256;                 // hidden units of the widest instantiation (also 64 and 128, see Width)
constexpr int S_KIN = 256;               // widest first-layer input (may exceed a narrow hidden width: Arm8 is 100)
constexpr int S_CONSUMERS = 256;         // 8 consumer warps
constexpr int S_THREADS = S_CONSUMERS + 32;   // + 1 producer warp
constexpr int S_CK = 32;                 // k rows per weight chunk
constexpr int S_NSLOT = 4;               // ring slots (a fifth slot - one more chunk in flight while the CTA samples its rows - measured no gain)
constexpr int S_SLOT = S_CK * S_H;       // floats per slot (32 KB)
constexpr int S_MAXL = 4;                // hidden layers supported by this schedule
constexpr int S_MAXCHUNK = 128;          // weight chunks of the main CTA (L = 4: 2 * 33 + 2 * 24 = 114)
constexpr int S_MAXCHUNK_T = 128;        // weight chunks of the critic CTA (L = 4: 3 * 33 + 24 = 123)
constexpr int S_DU = 8;                  // max action dim
constexpr int S_XT = S_H * 8;            // floats of one transposed activation buffer [256 k][<= 8 rows]
constexpr int S_RED = 4 * 8 * S_H;       // split-K partials [4 k-slices][<= 8 rows][256]
constexpr int S_MISC = 2048;              // small per-CTA state + the staged HER images of the 4 rows
constexpr int S_STAGE_OFF = 256;          // float offset of the HER stage inside misc
constexpr size_t S_SMEM_BYTES = (size_t)(S_NSLOT * S_SLOT + 2 * S_XT + S_RED + S_MISC) * 4 + 128;   // + 9 mbarriers

// The stream / action kernels at hidden width H in {64, 128, 256} (pad_hidden='native' runs a narrow net at its true
// width).  A thread owns 4 output columns: H / 4 column groups, and the 256 consumer threads split a chunk's k rows into
// KS = 1024 / H k-slices of RK rows each.  A chunk fills a 32 KB slot (32 rows at 256, 64 at 128); at 64 a hidden layer
// has only 64 k rows, so its chunk is the whole 16 KB layer and a thread takes 4 of them instead of 8.  The KS partial
// sums of a column are added in a fixed pairwise tree (TreeSum): the same bits on every run.
template <int H>
struct Width {
  static_assert(H == 64 || H == 128 || H == 256, "instantiated widths");
  static constexpr int CG = H / 4;                              // column groups
  static constexpr int KS = S_CONSUMERS / CG;                   // k-slices
  static constexpr int CK = (S_SLOT / H < H) ? S_SLOT / H : H;  // k rows per weight chunk
  static constexpr int RK = CK / KS;                            // k rows of one thread per chunk
  static_assert(KS * RK == CK && KS * 4 * H <= S_RED, "chunk split / partials fit");
};
static int chunk_rows(int H) { return H == 64 ? Width<64>::CK : H == 128 ? Width<128>::CK : Width<256>::CK; }

template <int N>
struct TreeSum {   // ((p[0] + p[s]) + (p[2s] + p[3s])) + ...: a fixed summation order of N partials
  __device__ __forceinline__ static float run(const float* p, int s) {
    return TreeSum<N / 2>::run(p, s) + TreeSum<N / 2>::run(p + (N / 2) * s, s);
  }
};
template <>
struct TreeSum<1> {
  __device__ __forceinline__ static float run(const float* p, int) { return p[0]; }
};

struct SChunk {
  const float* src;   // nrows x H floats, contiguous
  int nrows;          // <= Width<H>::CK
  int k0;             // first k row of the layer this chunk covers
};

struct StreamParams {
  cur_net_desc d;
  int in_sp, in_sq, in_g, KP, L, nchunks, nchunks_t;
  int64_t n;
  int64_t grad_rows;         // rows one loss mean runs over for the backward seeds (n, or cur_ddpg_hyper.loss_rows)
  const float *o, *g, *u, *td, *o_2, *g_2, *r;
  const float *o_mean, *o_std, *g_mean, *g_std;
  float gamma, clip_return, action_l2;
  int clip_pos;
  const float *bP[S_MAXL], *bPT[S_MAXL], *bQ[S_MAXL], *bQT[S_MAXL];
  const float *WoutP, *boutP, *WoutPT, *boutPT, *WoutQ, *boutQ, *WoutQT, *boutQT;
  const float* W0Q_act;      // main Q first-layer rows of the action inputs: [dimu][H]
  int ch0[2];                // chunks of a first layer: [0] pi nets, [1] Q nets
  float *Xp, *Xq;            // [n][KP] first-layer inputs of main.pi / main.Q(u)   (weight-gradient operands)
  float *hp[S_MAXL], *hq[S_MAXL], *hqp[S_MAXL], *dc[S_MAXL], *dp[S_MAXL];   // row-major [n][H]
  float *dQ, *dy;            // [n], [n][lddy]
  int lddy;
  float* loss_part;          // [n / 4][4]
  float* q_pi;               // [n]
  long long* tl;             // optional debug timeline (clock64 stamps of CTA 0), CUR_ROWS_TIMELINE=1
  int dbg_skip_math;         // debug: consumers only wait/release (measures the pure streaming rate)
  const int64_t* tl_step;    // debug: device step counter (update number of the timeline marks) or NULL
  int pdl_late;              // programmatic dependent launch: trigger the next kernel when this CTA is done (not at its start)
  int fused_her;             // sample the CTA's 4 rows here (her, plan) instead of reading a staged batch
  HerPlan plan;
  cur_her_args her;
  SChunk chunks[S_MAXCHUNK];       // actor CTA: main.pi fwd, main.Q fwd, main.Q^T bwd, main.pi^T bwd
  SChunk chunks_t[S_MAXCHUNK_T];   // critic CTA: target.pi fwd, target.Q fwd, main.Q fwd, main.Q^T bwd
};

#define S_TL(i)                                                                   \
  do {                                                                            \
    if (P.tl != nullptr && threadIdx.x == 0 && blockIdx.x == 0) P.tl[i] = clock64(); \
  } while (0)

// ---------------------------------------------------------------- mbarrier / bulk-copy primitives
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAIT_DONE;\n"
      "bra WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(bar), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t map_to_cta(uint32_t local_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void st_remote_f32(uint32_t remote_addr, float v) {
  asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(remote_addr), "f"(v) : "memory");
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t remote_bar) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote_bar) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAITC_LOOP:\n"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAITC_DONE;\n"
      "bra WAITC_LOOP;\n"
      "WAITC_DONE:\n"
      "}\n" ::"r"(bar), "r"(parity)
      : "memory");
}
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void st_ll(unsigned long long* p, float v, uint32_t flag) {
  const unsigned long long w = ((unsigned long long)flag << 32) | (unsigned long long)__float_as_uint(v);
  asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(w) : "memory");
}
// Programmatic dependent launch: the next kernel of the stream may be scheduled while this one still runs (its CTAs
// take SMs as they free up and park in pdl_wait); pdl_wait returns once the previous kernel has completed and its
// writes are visible.  Both are no-ops for a launch without the attribute.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void consumer_sync() { asm volatile("bar.sync 1, %0;" ::"n"(S_CONSUMERS) : "memory"); }


// debug (CUR_ROWS_TIMELINE=1): first start / last end of the two launches of an update on the %globaltimer clock, in a ring
// of 8 updates at tl[64 + 2048 + 4 * (update & 7)] = {stream first start, stream last end, dw first start, dw last end}
constexpr int TL_MARKS = 64 + 2048;
__device__ __forceinline__ void tl_mark_min(long long* p) {
  atomicMin(reinterpret_cast<unsigned long long*>(p), (unsigned long long)globaltimer_ns());
}
__device__ __forceinline__ void tl_mark_max(long long* p) {
  atomicMax(reinterpret_cast<unsigned long long*>(p), (unsigned long long)globaltimer_ns());
}

struct Ring {
  const SChunk* chunks;     // this CTA's chunk list (kernel-parameter space)
  const float* slots;
  uint32_t full, empty;     // shared addresses of the barrier arrays (8 bytes per slot)
  int cons;                 // chunks consumed so far
};

// ---------------------------------------------------------------- the GEMV core
// Blackwell issues a scalar FFMA only every other cycle per scheduler; full FP32 rate needs the packed FFMA2
// (fma.rn.f32x2, __ffma2_rn): two IEEE fmas per lane per instruction.  Accumulators are therefore kept as row
// pairs: acc[p][c] = (row 2p, row 2p+1) of column 4cg + c, the activation pair comes straight out of the
// transposed tile's float4 and only the weight is duplicated.  Each half is a plain fma.rn, so results are
// bit-identical to the scalar form.
template <int NR>
__device__ __forceinline__ void fma_row(float2 (&acc)[NR / 2][4], const float* __restrict__ xs, float4 w) {
  const float2 w0 = make_float2(w.x, w.x), w1 = make_float2(w.y, w.y), w2 = make_float2(w.z, w.z),
               w3 = make_float2(w.w, w.w);
#pragma unroll
  for (int q = 0; q < NR / 4; ++q) {
    const float4 v = *reinterpret_cast<const float4*>(xs + 4 * q);
    const float2 xa = make_float2(v.x, v.y), xb = make_float2(v.z, v.w);
    acc[2 * q][0] = __ffma2_rn(xa, w0, acc[2 * q][0]);
    acc[2 * q][1] = __ffma2_rn(xa, w1, acc[2 * q][1]);
    acc[2 * q][2] = __ffma2_rn(xa, w2, acc[2 * q][2]);
    acc[2 * q][3] = __ffma2_rn(xa, w3, acc[2 * q][3]);
    acc[2 * q + 1][0] = __ffma2_rn(xb, w0, acc[2 * q + 1][0]);
    acc[2 * q + 1][1] = __ffma2_rn(xb, w1, acc[2 * q + 1][1]);
    acc[2 * q + 1][2] = __ffma2_rn(xb, w2, acc[2 * q + 1][2]);
    acc[2 * q + 1][3] = __ffma2_rn(xb, w3, acc[2 * q + 1][3]);
  }
}

// acc += sum over this thread's k rows of the next `nchunks` weight chunks of  xT[k][r] * W[k][4cg + c]
template <int H, int NR, class PT>
__device__ __forceinline__ void gemv_chunks(const PT& P, Ring& rg, int nchunks, const float* __restrict__ xT,
                                            float2 (&acc)[NR / 2][4]) {
  using Wd = Width<H>;
  constexpr int RK = Wd::RK;
  const int cg = threadIdx.x % Wd::CG, ks = threadIdx.x / Wd::CG;
#pragma unroll 1
  for (int c = 0; c < nchunks; ++c) {
    const int slot = rg.cons % S_NSLOT;
    const int nrows = rg.chunks[rg.cons].nrows, k0 = rg.chunks[rg.cons].k0;
    mbar_wait(rg.full + 8 * slot, (rg.cons / S_NSLOT) & 1);
    const float* ws = rg.slots + slot * S_SLOT + 4 * cg;
    const float* xs = xT + (k0 + ks * RK) * NR;
    if (P.dbg_skip_math) {
    } else if (nrows == Wd::CK) {
      // full chunk (all but the ragged first-layer blocks): no guards, so the LDS.128 of the thread's RK k rows
      // are issued up front and the FFMA2s run back to back
      float4 w[RK];
#pragma unroll
      for (int kk = 0; kk < RK; ++kk) w[kk] = *reinterpret_cast<const float4*>(ws + (ks * RK + kk) * H);
#pragma unroll
      for (int kk = 0; kk < RK; ++kk) fma_row<NR>(acc, xs + kk * NR, w[kk]);
    } else {
#pragma unroll 1
      for (int kk = 0; kk < RK; ++kk)
        if (ks * RK + kk < nrows)
          fma_row<NR>(acc, xs + kk * NR, *reinterpret_cast<const float4*>(ws + (ks * RK + kk) * H));
    }
    __syncwarp();
    if ((threadIdx.x & 31) == 0) mbar_arrive(rg.empty + 8 * slot);
    ++rg.cons;
  }
}

// A consumer thread that owns an output column: all of them at H = 256; below, threads H.. only take part in the
// k-slices of the GEMV and in the barriers.
template <int H>
__device__ __forceinline__ bool owns_col(int col) { return H == S_CONSUMERS || col < H; }

// One dense layer for NR rows: chunks -> split-K partials -> fixed-order sum.  Returns, for the thread's column
// `col = tid` (if owns_col), the NR pre-activation sums in v[] (without bias).
template <int H, int NR, class PT>
__device__ __forceinline__ void layer_gemv(const PT& P, Ring& rg, int nchunks, const float* xT, float* red,
                                           float (&v)[NR]) {
  using Wd = Width<H>;
  float2 acc[NR / 2][4];
#pragma unroll
  for (int p = 0; p < NR / 2; ++p)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[p][c] = make_float2(0.f, 0.f);
  gemv_chunks<H, NR>(P, rg, nchunks, xT, acc);
  const int cg = threadIdx.x % Wd::CG, ks = threadIdx.x / Wd::CG;
#pragma unroll
  for (int p = 0; p < NR / 2; ++p) {
    *reinterpret_cast<float4*>(red + (ks * NR + 2 * p) * H + 4 * cg) =
        make_float4(acc[p][0].x, acc[p][1].x, acc[p][2].x, acc[p][3].x);
    *reinterpret_cast<float4*>(red + (ks * NR + 2 * p + 1) * H + 4 * cg) =
        make_float4(acc[p][0].y, acc[p][1].y, acc[p][2].y, acc[p][3].y);
  }
  consumer_sync();
  const int col = threadIdx.x;
  if (owns_col<H>(col)) {
#pragma unroll
    for (int r = 0; r < NR; ++r) v[r] = TreeSum<Wd::KS>::run(red + r * H + col, NR * H);
  } else {
#pragma unroll
    for (int r = 0; r < NR; ++r) v[r] = 0.f;
  }
}

// write the layer output: transposed into shared memory for the next layer, row-major to global for launch 2
template <int H, int NR>
__device__ __forceinline__ void put_xT(float* yT, const float (&v)[NR]) {
  const int col = threadIdx.x;
  if (!owns_col<H>(col)) return;
#pragma unroll
  for (int q = 0; q < NR / 4; ++q)
    *reinterpret_cast<float4*>(yT + col * NR + 4 * q) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
}

__device__ __forceinline__ float norm1s(float x, const float* mean, const float* std, int k, float clip) {
  float v = __fdiv_rn(__fsub_rn(x, mean[k]), std[k]);          // normalizer.py:72-77
  return fminf(fmaxf(v, -clip), clip);
}

// Element (row, column k) of a first-layer input [o | task_descr | action | g] (modular) or [o | g | action]
// (flat), zero beyond the fan-in (actor_critic.py:76-91).  act_kind: 0 none (pi net), 1 u / max_u, 2 `ths`.
// The batch values come from the staged batch arrays, or - fused HER sampling - from the relabelled row image
// `st` in shared memory, preprocessed exactly like the HER kernel's outputs (ddpg.py:118-127: relative goals,
// clip to +-clip_obs).
__device__ __forceinline__ float x_elem(const StreamParams& P, int64_t row, int r, int k, bool target, int act_kind,
                                        const float* ths, const float* st) {
  const cur_net_desc& d = P.d;
  const bool nrm = d.normalize_obs != 0;
  const int in_s = P.in_sp + (act_kind ? d.dimu : 0);
  const HerPlan& pl = P.plan;
  const float clip = P.her.clip_obs;
  float v = 0.f;
  int gj = -1, aj = -1;
  if (k < d.dimo) {
    if (st) {
      v = st[(target ? pl.iO2 : pl.iO) + k];
      if (clip > 0.f) v = fminf(fmaxf(v, -clip), clip);
    } else {
      v = (target ? P.o_2 : P.o)[row * d.dimo + k];
    }
    if (nrm) v = norm1s(v, P.o_mean, P.o_std, k, d.norm_clip);
  } else if (d.modular) {
    if (k < d.dimo + d.dimtd) {
      const int j = k - d.dimo;
      v = st ? st[pl.iTD + j] : P.td[row * d.dimtd + j];       // never normalised
    } else if (k < in_s) aj = k - d.dimo - d.dimtd;
    else if (k < in_s + d.dimg) gj = k - in_s;
  } else {
    if (k < d.dimo + d.dimg) gj = k - d.dimo;
    else if (k < in_s) aj = k - d.dimo - d.dimg;
  }
  if (gj >= 0) {
    if (st) {
      v = st[pl.iG + gj];
      if (P.her.relative_goals) v -= st[(target ? pl.iAG2 : pl.iAG) + gj];
      if (clip > 0.f) v = fminf(fmaxf(v, -clip), clip);
    } else {
      v = (target ? P.g_2 : P.g)[row * d.dimg + gj];
    }
    if (nrm) v = norm1s(v, P.g_mean, P.g_std, gj, d.norm_clip);
  }
  if (aj >= 0) {
    if (act_kind == 1) v = __fdiv_rn(st ? st[pl.iU + aj] : P.u[row * d.dimu + aj], d.max_u);
    else v = ths[r * S_DU + aj];
  }
  return v;
}

// transposed first-layer input xT[k][NR] for rows [roff, roff + 4) of the buffer; optional row-major global copy
__device__ __noinline__ void build_x(const StreamParams& P, float* xT, int NR, int roff, int64_t row0, bool target,
                                     int act_kind, const float* ths, float* gout, const float* stage) {
  const int ss = P.plan.stage_stride;
  for (int idx = threadIdx.x; idx < S_ROWS * P.KP; idx += S_CONSUMERS) {
    const int k = idx >> 2, r = idx & 3;
    xT[k * NR + roff + r] = x_elem(P, row0 + r, r, k, target, act_kind, ths, stage ? stage + r * ss : nullptr);
  }
  if (gout) {
    for (int idx = threadIdx.x; idx < S_ROWS * P.KP; idx += S_CONSUMERS) {
      const int r = idx / P.KP, k = idx - r * P.KP;
      gout[(row0 + r) * P.KP + k] = x_elem(P, row0 + r, r, k, target, act_kind, ths, stage ? stage + r * ss : nullptr);
    }
  }
}

// Fused HER sampling of the CTA's 4 rows: draws -> cp.async gather of the row images -> relabel + reward, with
// the same per-row device functions as her_sample_kernel (bit-identical batches).  Both CTAs of a pair sample the
// same rows (a 4 x ~0.5 KB gather).
__device__ __forceinline__ void sample_rows(const StreamParams& P, int64_t row0, float* stage, const float** m_src,
                                            float* s_r, float* scratch /* >= 1 KB, 16-byte aligned */, int nrows = S_ROWS) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const HerPlan& pl = P.plan;
  HerRow row;
  row.ft = -1; row.choice = -1; row.ep = 0; row.t = 0; row.ttr = -1; row.her = false;
  // the device control block of the sampler (counts, sizes, cdf, the step counter behind a pointer) in TWO round trips: the
  // draw below used to read it in place, ~7 dependent L2 round trips in front of every chain
  static_assert(sizeof(cur_her_dyn) % 4 == 0 && sizeof(cur_her_dyn) + 8 <= 4 * 256, "control block copy fits the scratch area");
  cur_her_dyn* dyn_s = reinterpret_cast<cur_her_dyn*>(scratch);
  int64_t* step_s = reinterpret_cast<int64_t*>(scratch + sizeof(cur_her_dyn) / 4);
  if (P.her.dyn != nullptr) {
    if (tid < (int)(sizeof(cur_her_dyn) / 4))
      reinterpret_cast<uint32_t*>(dyn_s)[tid] = __ldcg(reinterpret_cast<const uint32_t*>(P.her.dyn) + tid);
    consumer_sync();
    if (tid == 0) *step_s = __ldcg(reinterpret_cast<const long long*>(dyn_s->step));
    consumer_sync();
  }
  if (tid < nrows) her_draw_row(P.her, pl, row0 + tid, row, m_src + 3 * tid, dyn_s, step_s);
  consumer_sync();
  if (warp < nrows) {
    const int per_row = pl.img4 + pl.fut4 + pl.cold4;   // (cold rows only for an `info` reward or relative goals)
    float* dst = stage + warp * pl.stage_stride;
    for (int c = lane; c < per_row; c += 32) {
      int sel = 0, q = c, doff = 4 * c;
      if (c >= pl.img4 + pl.fut4) { sel = 2; q = c - pl.img4 - pl.fut4; doff = pl.cold_off + 4 * q; }
      else if (c >= pl.img4) { sel = 1; q = c - pl.img4; doff = pl.fut_off + 4 * q; }
      const float* src = m_src[3 * warp + sel];
      if (src != nullptr) cp16_zfill(dst + doff, src + 4 * q, true);
    }
  }
  cp_commit();
  cp_wait0();
  consumer_sync();
  if (tid < nrows) {
    int relab;
    s_r[tid] = her_relabel_row(P.her, pl, stage + tid * pl.stage_stride, row, &relab);
  }
  consumer_sync();
}

// y[r][j] = sum_k xT[k][r] * W[k * ldk + j * ldj] + bias[j]  for r < NR, j < nout (NR * nout <= 32), K = H.
// 8 k-parts per output (interleaved k), combined with a fixed shuffle tree; every thread must call it.
template <int H>
__device__ __noinline__ void small_out(const float* xT, int NR, int roff, int nr, const float* __restrict__ W, int ldk,
                                       int ldj, int nout, const float* bias, float* out /* [r][S_DU] */) {
  const int kp = threadIdx.x & 7, oj = threadIdx.x >> 3;
  const int r = oj / nout, j = oj - r * nout;
  const bool on = r < nr;
  float acc = 0.f;
  if (on) {
    // all 32 weight loads of the thread in flight at once: one exposed L2 round trip instead of four (the loop is on the
    // critical path of every net: nothing else runs in the CTA meanwhile)
    float wv[H / 8];
#pragma unroll
    for (int kk = 0; kk < H / 8; ++kk) wv[kk] = __ldg(W + (int64_t)(kp + 8 * kk) * ldk + (int64_t)j * ldj);
#pragma unroll
    for (int kk = 0; kk < H / 8; ++kk) acc = fmaf(xT[(kp + 8 * kk) * NR + roff + r], wv[kk], acc);
  }
  acc += __shfl_xor_sync(0xffffffffu, acc, 1);
  acc += __shfl_xor_sync(0xffffffffu, acc, 2);
  acc += __shfl_xor_sync(0xffffffffu, acc, 4);
  if (on && kp == 0) out[r * S_DU + j] = acc + (bias ? bias[j] : 0.f);
}

__device__ __forceinline__ float relu_mask(float v, float m) { return m > 0.f ? v : 0.f; }

// One forward net for NR rows: L hidden layers (bias + ReLU) from the first-layer input already in `xa`; optional
// row-major copies of every hidden activation (rows 0-3 -> h_a, rows 4-7 -> h_b).  Returns the buffer that holds
// the last hidden activations (transposed).
template <int H, int NR, class PT>
__device__ __forceinline__ float* forward_net(const PT& P, Ring& rg, int ch0, float* xa, float* xb, float* red,
                                              const float* const* bias, float* const* h_a, float* const* h_b,
                                              int64_t row0) {
  const int col = threadIdx.x;
  const bool on = owns_col<H>(col);
  float* xin = xa;
  float* xout = xb;
  for (int l = 0; l < P.L; ++l) {
    float v[NR];
    const float b = on ? bias[l][col] : 0.f;      // in flight during the layer (an exposed L2 round trip otherwise)
    layer_gemv<H, NR>(P, rg, l == 0 ? ch0 : H / Width<H>::CK, xin, red, v);
#pragma unroll
    for (int r = 0; r < NR; ++r) v[r] = fmaxf(v[r] + b, 0.f);
    if (on && h_a != nullptr) {
#pragma unroll
      for (int r = 0; r < 4; ++r) h_a[l][(row0 + r) * H + col] = v[r];
    }
    if (on && NR == 8 && h_b != nullptr) {
#pragma unroll
      for (int r = 0; r < 4; ++r) h_b[l][(row0 + r) * H + col] = v[NR - 4 + r];
    }
    put_xT<H, NR>(xout, v);
    consumer_sync();
    float* t = xin; xin = xout; xout = t;
  }
  return xin;
}

// Two CTAs per 4 batch rows, fully independent of each other:
//   even CTA (actor):  main.pi -> main.Q(o,g,pi) -> actor loss -> backward through main.Q (action gradient) and main.pi
//   odd CTA (critic):  target.pi -> target.Q -> main.Q(o,g,u) -> TD loss -> backward through main.Q (critic chain)
// Each SM ingests 2.2-2.3 MB of weights for FOUR rows at a time (per-SM L2 -> shared bandwidth is what bounds this
// kernel; the earlier main / target split streamed main.Q once for 8 stacked rows, which made those passes FFMA-bound
// and left the target CTA idle for 40 % of the kernel).
template <int H>
__global__ void __launch_bounds__(S_THREADS, 1)
ddpg_stream_kernel(const __grid_constant__ StreamParams P) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float* ringf = reinterpret_cast<float*>(smem_raw);
  float* xa = ringf + S_NSLOT * S_SLOT;
  float* xb = xa + S_XT;
  float* red = xb + S_XT;
  float* misc = red + S_RED;
  uint64_t* bars = reinterpret_cast<uint64_t*>(misc + S_MISC);      // full[4], empty[4], qt
  float* s_th = misc;                 // [4][8] tanh output of this CTA's pi net (= pi / max_u)
  float* s_q = misc + 64;             // [8][8]: rows 0-3 main.Q(o,g,u), rows 4-7 main.Q(o,g,pi)
  float* s_qt = misc + 128;           // [4][8] target.Q (written by the target CTA through DSMEM)
  float* s_dq = misc + 160;           // [8]: dQ (rows 0-3), dQ_pi (rows 4-7);  [8..12): squared TD error
  float* s_dy = misc + 192;           // [4][8]
  float* s_r = misc + 224;            // [4] rewards of the rows (fused HER sampling)
  const float** m_src = reinterpret_cast<const float**>(misc + 228);     // [4][3] source addresses
  float* her_stage = misc + S_STAGE_OFF;                                  // [4][stage_stride]

  const int tid = threadIdx.x;
  if (P.tl != nullptr && tid == 0 && blockIdx.x < 512) P.tl[64 + 2 * blockIdx.x] = (long long)globaltimer_ns();
  if (P.tl != nullptr && P.tl_step != nullptr && tid == 0) tl_mark_min(P.tl + TL_MARKS + 4 * (int)(*P.tl_step & 7));
  const uint32_t role = blockIdx.x & 1;                      // 0: actor chain, 1: critic chain (independent CTAs)
  const int64_t row0 = (int64_t)(blockIdx.x >> 1) * S_ROWS;
  const cur_net_desc& d = P.d;
  const int L = P.L;
  const uint32_t full = smem_addr(bars), empty = smem_addr(bars + S_NSLOT);

  if (tid == 0) {
    for (int i = 0; i < S_NSLOT; ++i) {
      mbar_init(full + 8 * i, 1);
      mbar_init(empty + 8 * i, S_CONSUMERS / 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (!P.pdl_late) pdl_launch_dependents();
  pdl_wait();               // everything below reads what the previous kernel (weight gradients + Adam of the last update) wrote
  __syncthreads();          // barriers initialised before the producer / consumers use them

  const SChunk* my_chunks = role == 0 ? P.chunks : P.chunks_t;
  if (tid >= S_CONSUMERS) {
    // ------------------------------------------------------------ producer warp: stream every weight chunk
    if (tid == S_CONSUMERS) {
      const uint32_t ring_s = smem_addr(ringf);
      const int total = role == 0 ? P.nchunks : P.nchunks_t;
      for (int i = 0; i < total; ++i) {
        const int slot = i % S_NSLOT, round = i / S_NSLOT;
        if (round > 0) mbar_wait(empty + 8 * slot, (round - 1) & 1);
        const uint32_t bytes = (uint32_t)my_chunks[i].nrows * H * 4;
        mbar_expect_tx(full + 8 * slot, bytes);
        bulk_g2s(ring_s + slot * S_SLOT * 4, my_chunks[i].src, bytes, full + 8 * slot);
      }
    }
    return;
  }

  // -------------------------------------------------------------- consumers
  Ring rg;
  rg.chunks = my_chunks; rg.slots = ringf; rg.full = full; rg.empty = empty; rg.cons = 0;
  const int col = tid;
  const bool on = owns_col<H>(col);      // this thread owns an output column of the hidden layers
  const float inv_n = 1.0f / (float)P.grad_rows;      // scale of the backward seeds
  const float* stage = nullptr;
  if (P.fused_her) {
    sample_rows(P, row0, her_stage, m_src, s_r, red);
    stage = her_stage;
  }

  const float hi_clip = P.clip_pos ? 0.f : INFINITY;
  if (role == 1) {
    // ===== critic CTA: target.pi -> target.Q(o2, g2, pi_target) with the same u-slot and td (ddpg.py:427-431),
    // main.Q(o, g, u), the TD loss and the critic's backward chain.  Nothing is exchanged with the actor CTA.
    build_x(P, xa, 4, 0, row0, true, 0, nullptr, nullptr, stage);
    consumer_sync();
    float* xl = forward_net<H, 4>(P, rg, P.ch0[0], xa, xb, red, P.bPT, nullptr, nullptr, row0);
    small_out<H>(xl, 4, 0, 4, P.WoutPT, d.dimu, 1, d.dimu, P.boutPT, s_th);
    consumer_sync();
    if (tid < S_ROWS * S_DU && (tid & (S_DU - 1)) < d.dimu) s_th[tid] = tanhf(s_th[tid]);
    consumer_sync();
    build_x(P, xa, 4, 0, row0, true, 2, s_th, nullptr, stage);
    consumer_sync();
    xl = forward_net<H, 4>(P, rg, P.ch0[1], xa, xb, red, P.bQT, nullptr, nullptr, row0);
    small_out<H>(xl, 4, 0, 4, P.WoutQT, 1, 1, 1, P.boutQT, s_qt);
    consumer_sync();
    // main.Q(o, g, u)
    build_x(P, xa, 4, 0, row0, false, 1, nullptr, P.Xq, stage);
    consumer_sync();
    xl = forward_net<H, 4>(P, rg, P.ch0[1], xa, xb, red, P.bQ, P.hq, nullptr, row0);
    small_out<H>(xl, 4, 0, 4, P.WoutQ, 1, 1, 1, P.boutQ, s_q);
    consumer_sync();
    // critic loss (ddpg.py:436-439) and its backward seed
    if (tid < S_ROWS) {
      const int64_t row = row0 + tid;
      const float rew = stage ? s_r[tid] : P.r[row];
      const float tgt = fminf(fmaxf(rew + P.gamma * s_qt[tid * S_DU], -P.clip_return), hi_clip);
      const float diff = tgt - s_q[tid * S_DU];
      s_dq[tid] = -2.0f * inv_n * diff;          // d mean((tgt - Q)^2) / dQ
      s_dq[8 + tid] = diff * diff;
      P.dQ[row] = s_dq[tid];
    }
    consumer_sync();
    if (tid == 0) {
      float ssq = 0.f;
      for (int r = 0; r < S_ROWS; ++r) ssq += s_dq[8 + r];
      P.loss_part[(int64_t)(blockIdx.x >> 1) * 4] = ssq;
    }
    // backward through main.Q (critic chain): gradient at the last hidden layer is dQ * Wout^T (Wout is [H][1])
    float* xin = xa; float* xout = xb;
    if (on) {
      const float wq = __ldg(P.WoutQ + col);
      float v[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        v[r] = relu_mask(s_dq[r] * wq, __ldcg(P.hq[L - 1] + (row0 + r) * H + col));
        P.dc[L - 1][(row0 + r) * H + col] = v[r];
      }
      put_xT<H, 4>(xin, v);
    }
    consumer_sync();
    for (int l = L - 1; l >= 1; --l) {
      float m[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) m[r] = on ? __ldcg(P.hq[l - 1] + (row0 + r) * H + col) : 0.f;   // ReLU masks of layer l-1
      float v[4];
      layer_gemv<H, 4>(P, rg, H / Width<H>::CK, xin, red, v);
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        v[r] = relu_mask(v[r], m[r]);
        if (on) P.dc[l - 1][(row0 + r) * H + col] = v[r];
      }
      put_xT<H, 4>(xout, v);
      consumer_sync();
      float* t = xin; xin = xout; xout = t;
    }
    if (P.tl != nullptr && tid == 0 && blockIdx.x < 512) P.tl[65 + 2 * blockIdx.x] = (long long)globaltimer_ns();
    if (P.tl != nullptr && P.tl_step != nullptr && tid == 0) tl_mark_max(P.tl + TL_MARKS + 4 * (int)(*P.tl_step & 7) + 1);
    pdl_launch_dependents();
    return;
  }

  // ===== actor CTA: main.pi -> main.Q(o, g, pi) -> actor loss -> backward through main.Q and main.pi =====
  S_TL(0);
  build_x(P, xa, 4, 0, row0, false, 0, nullptr, P.Xp, stage);
  consumer_sync();
  S_TL(1);
  {
    float* xl = forward_net<H, 4>(P, rg, P.ch0[0], xa, xb, red, P.bP, P.hp, nullptr, row0);
    small_out<H>(xl, 4, 0, 4, P.WoutP, d.dimu, 1, d.dimu, P.boutP, s_th);
    consumer_sync();
    if (tid < S_ROWS * S_DU && (tid & (S_DU - 1)) < d.dimu) s_th[tid] = tanhf(s_th[tid]);   // actor_critic.py:89
    consumer_sync();
  }
  S_TL(2);
  S_TL(3);
  build_x(P, xa, 4, 0, row0, false, 2, s_th, nullptr, stage);
  consumer_sync();
  {
    float* xl = forward_net<H, 4>(P, rg, P.ch0[1], xa, xb, red, P.bQ, P.hqp, nullptr, row0);
    small_out<H>(xl, 4, 0, 4, P.WoutQ, 1, 1, 1, P.boutQ, s_q);
    consumer_sync();
  }
  S_TL(4);
  S_TL(5);
  // ===== actor loss terms (ddpg.py:440-441) and backward seed =====
  if (tid < S_ROWS) {
    s_dq[tid] = -inv_n;                        // d (-mean(Q_pi)) / dQ_pi
    P.q_pi[row0 + tid] = s_q[tid * S_DU];
  }
  if (tid == 0) {
    float sq = 0.f, sth = 0.f;
    for (int r = 0; r < S_ROWS; ++r) {
      sq += s_q[r * S_DU];
      for (int j = 0; j < d.dimu; ++j) sth += s_th[r * S_DU + j] * s_th[r * S_DU + j];
    }
    float* lp = P.loss_part + (int64_t)(blockIdx.x >> 1) * 4;
    lp[1] = sq; lp[2] = sth; lp[3] = 0.f;
  }
  consumer_sync();
  // ===== backward through main.Q, actor-through-critic chain =====
  {
    float* xin = xa; float* xout = xb;
    if (on) {
      const float wq = __ldg(P.WoutQ + col);
      float v[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) v[r] = relu_mask(s_dq[r] * wq, __ldcg(P.hqp[L - 1] + (row0 + r) * H + col));
      put_xT<H, 4>(xin, v);
    }
    consumer_sync();
    for (int l = L - 1; l >= 1; --l) {
      float m[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) m[r] = on ? __ldcg(P.hqp[l - 1] + (row0 + r) * H + col) : 0.f;
      float v[4];
      layer_gemv<H, 4>(P, rg, H / Width<H>::CK, xin, red, v);
#pragma unroll
      for (int r = 0; r < 4; ++r) v[r] = relu_mask(v[r], m[r]);
      put_xT<H, 4>(xout, v);
      consumer_sync();
      float* t = xin; xin = xout; xout = t;
    }
    // gradient wrt the action inputs of main.Q, then through tanh and the action penalty (ddpg.py:440-441):
    // d pi_loss/d(pre-tanh) = (dL/d(pi/max_u) + action_l2*2/(B*dimu)*th) * (1 - th^2)
    small_out<H>(xin, 4, 0, 4, P.W0Q_act, 1, H, d.dimu, nullptr, s_dy);
    consumer_sync();
    if (tid < S_ROWS * S_DU) {
      const int r = tid >> 3, j = tid & (S_DU - 1);
      float v = 0.f;
      if (j < d.dimu) {
        const float coef = P.action_l2 * 2.0f / (float)(P.grad_rows * d.dimu);
        const float th = s_th[tid];
        v = (s_dy[tid] + coef * th) * (1.f - th * th);
      }
      s_dy[tid] = v;
      if (j < P.lddy) P.dy[(row0 + r) * P.lddy + j] = v;
    }
    consumer_sync();
  }
  S_TL(6);
  // ===== backward through main.pi =====
  {
    float* xin = xa; float* xout = xb;
    if (on) {
      float v[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) v[r] = 0.f;
      for (int j = 0; j < d.dimu; ++j) {
        const float wj = __ldg(P.WoutP + (int64_t)col * d.dimu + j);
#pragma unroll
        for (int r = 0; r < 4; ++r) v[r] = fmaf(s_dy[r * S_DU + j], wj, v[r]);
      }
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        v[r] = relu_mask(v[r], __ldcg(P.hp[L - 1] + (row0 + r) * H + col));
        P.dp[L - 1][(row0 + r) * H + col] = v[r];
      }
      put_xT<H, 4>(xin, v);
    }
    consumer_sync();
    for (int l = L - 1; l >= 1; --l) {
      float m[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) m[r] = on ? __ldcg(P.hp[l - 1] + (row0 + r) * H + col) : 0.f;
      float v[4];
      layer_gemv<H, 4>(P, rg, H / Width<H>::CK, xin, red, v);
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        v[r] = relu_mask(v[r], m[r]);
        if (on) P.dp[l - 1][(row0 + r) * H + col] = v[r];
      }
      put_xT<H, 4>(xout, v);
      consumer_sync();
      float* t = xin; xin = xout; xout = t;
    }
  }
  S_TL(7);
  if (P.tl != nullptr && tid == 0 && blockIdx.x < 512) P.tl[65 + 2 * blockIdx.x] = (long long)globaltimer_ns();
  if (P.tl != nullptr && P.tl_step != nullptr && tid == 0) tl_mark_max(P.tl + TL_MARKS + 4 * (int)(*P.tl_step & 7) + 1);
  pdl_launch_dependents();
}

// ------------------------------------------------------------------------------------------------
// CTA-PAIR form of the stream kernel (batch a multiple of 8): a 2-CTA cluster walks one chain for EIGHT rows, and each CTA
// owns HALF the output columns of every hidden layer.  An SM then ingests only half of its chain's weights (1.1 MB
// instead of 2.2 MB - per-SM L2 -> shared bandwidth, ~42 B/clk, is what bounds the 4-row kernel) while doing the same
// number of FMAs (8 rows x 128 columns; scratch/micro/gemv_micro.cu: 690 cycles per 32 KB chunk against ~780 of ingest).
// After every layer the two CTAs swap their halves of the activations through distributed shared memory: each thread
// stores its 16 bytes into both CTAs' transposed activation buffer and arrives on the partner's mbarrier; the next layer
// starts with the k rows of the CTA's OWN columns (already local) and only then waits for the partner's half, so the
// exchange latency hides behind half a layer.  Weight chunks are 64 k rows x 128 columns = 32 KB, one 2-D TMA box each
// (64 bulk copies of 512 bytes per chunk, the first version, ran at ~8 B/clk: 100 us per update).
constexpr int PR_ROWS = 8;                // batch rows per CTA pair
constexpr int PR_NC = 128;                // output columns per CTA
constexpr int PR_CK = 64;                 // k rows per weight chunk (64 x 128 floats = S_SLOT)
constexpr int PR_MAXCHUNK = 64;           // chunks per (chain, rank): L = 4, 256 first-layer inputs -> 3 * 17 + 12 = 63
constexpr int PR_MISC = 4096;             // floats of small per-CTA state + the staged HER images of the 8 rows
constexpr int PR_STAGE_OFF = 512;
constexpr size_t PR_SMEM_BYTES = (size_t)(S_NSLOT * S_SLOT + 2 * S_XT + S_RED + PR_MISC) * 4 + 128;
static_assert(PR_CK * PR_NC == S_SLOT && PR_ROWS * S_H == S_XT && 8 * PR_ROWS * PR_NC == S_RED, "pair kernel reuses the ring / xT / partial areas");

constexpr int PR_MAXMAPS = 28;            // weight blocks of the four nets + the transposes (L = 4: 4 * 5 + 2 * 3 = 26)

struct PairChunk {
  int map;            // tensor map of the weight block [rows][256] this chunk comes from
  int krow;           // first row of the block
  short nrows;        // rows of the chunk that exist (<= 64; the TMA unit zero-fills the rest of the box)
  short wait;         // 1: the first chunk of a layer whose k rows are the PARTNER's columns of the previous layer
  int k0;             // first k row of the layer this chunk covers
};

struct PairParams {
  StreamParams S;
  int nch[2][2];                          // [role][rank]
  int pch0[2];                            // chunks of a first layer: [0] pi nets, [1] Q nets
  PairChunk ch[2][2][PR_MAXCHUNK];        // [role: actor, critic][cluster rank]
  alignas(64) CUtensorMap maps[PR_MAXMAPS];   // box = 128 columns x 64 rows, dense
};

struct PairRing {
  const PairChunk* chunks;
  const float* slots;
  uint32_t full, empty;
  int cons;
};

// the activation exchange of a CTA pair (see above); every consumer thread holds the same state.  A thread's 16 bytes
// travel as ONE st.async that also counts its bytes on the receiver's mbarrier (complete_tx, like a TMA copy): no
// release / acquire round trip and no per-thread arrive (256 remote arrives per layer cost ~4 k cycles, measured).
struct PairX {
  uint32_t bar_local[2], bar_remote[2];   // mbarriers (count 1 = the receiver's own expect_tx), alternating per exchange
  uint32_t x_local, x_remote;             // shared address of xa here / in the partner (xb follows at + S_XT floats)
  uint32_t word_remote;                   // a scratch word of the partner (payload of a data-less rendezvous)
  int step;                               // exchanges issued so far
  bool pending;                           // the partner's half of exchange `step - 1` has not been waited for yet
  long long* dbg;                         // debug stamps (thread 0 of CTA 0, CUR_ROWS_TIMELINE=1) or nullptr
  __device__ __forceinline__ void stamp() {
    if (dbg != nullptr) *dbg++ = clock64();
  }
  __device__ __forceinline__ void wait() {
    if (pending) {
      const int s = step - 1;
      stamp();
      mbar_wait_cluster(bar_local[s & 1], (uint32_t)((s >> 1) & 1));
      stamp();
      pending = false;
    }
  }
  // 4 rows (4 * rh ..) of column `gcol` of the layer output: into both CTAs' transposed buffer `xT`
  __device__ __forceinline__ void put(float* xT, int gcol, int rh, const float (&v)[4]) {
    float* dst = xT + gcol * PR_ROWS + 4 * rh;
    *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
    const uint32_t ra = x_remote + (smem_addr(dst) - x_local);
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.f32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(ra),
                 "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "r"(bar_remote[step & 1])
                 : "memory");
    if (threadIdx.x == 0) mbar_expect_tx(bar_local[step & 1], S_CONSUMERS * 16);     // what the partner sends me
    ++step;
    pending = true;
  }
  // pair-wide rendezvous of the consumers without data: nobody passes before both CTAs are done with what they read
  // so far (a first layer / a backward seed does not depend on the partner, so it could otherwise overwrite a buffer the
  // partner is still reading)
  __device__ __forceinline__ void sync() {
    wait();
    consumer_sync();                      // every thread of this CTA is done reading
    if (threadIdx.x == 0) {
      asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.f32 [%0], %1, [%2];" ::"r"(word_remote),
                   "f"(0.f), "r"(bar_remote[step & 1])
                   : "memory");
      mbar_expect_tx(bar_local[step & 1], 4);
    }
    ++step;
    pending = true;
    wait();
  }
};

template <class PT>
__device__ __forceinline__ void pair_gemv_chunks(const PT& P, PairRing& rg, PairX& X, int nchunks, const float* __restrict__ xT,
                                                 float2 (&acc)[4][4]) {
  const int cg = threadIdx.x & 31, ks = threadIdx.x >> 5;
#pragma unroll 1
  for (int c = 0; c < nchunks; ++c) {
    const int slot = rg.cons % S_NSLOT;
    const int nrows = rg.chunks[rg.cons].nrows, k0 = rg.chunks[rg.cons].k0;
    if (rg.chunks[rg.cons].wait) X.wait();
    mbar_wait(rg.full + 8 * slot, (rg.cons / S_NSLOT) & 1);
    const float* ws = rg.slots + slot * S_SLOT + 4 * cg;
    const float* xs = xT + (k0 + ks * 8) * PR_ROWS;
    if (P.dbg_skip_math) {
    } else if (ks * 8 < nrows) {
      // a ragged first-layer block: the TMA unit zero-filled the box rows beyond nrows and pair_build_x zeroed the x
      // rows beyond the fan-in, so a k-slice that starts inside the block runs unguarded (warp-uniform test)
      float4 w[8];
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) w[kk] = *reinterpret_cast<const float4*>(ws + (ks * 8 + kk) * PR_NC);
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) fma_row<PR_ROWS>(acc, xs + kk * PR_ROWS, w[kk]);
    }
    __syncwarp();
    if ((threadIdx.x & 31) == 0) mbar_arrive(rg.empty + 8 * slot);
    ++rg.cons;
  }
}

// One dense layer for the pair's 8 rows and this CTA's 128 columns.  Returns, for the thread's column `tid & 127` and
// its 4 rows 4 * (tid >> 7) .., the pre-activation sums (without bias).
template <class PT>
__device__ __forceinline__ void pair_layer_gemv(const PT& P, PairRing& rg, PairX& X, int nchunks, const float* xT, float* red,
                                                float (&v)[4]) {
  float2 acc[4][4];
#pragma unroll
  for (int p = 0; p < 4; ++p)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[p][c] = make_float2(0.f, 0.f);
  X.stamp();
  pair_gemv_chunks(P, rg, X, nchunks, xT, acc);
  X.stamp();
  const int cg = threadIdx.x & 31, ks = threadIdx.x >> 5;
#pragma unroll
  for (int p = 0; p < 4; ++p) {
    *reinterpret_cast<float4*>(red + (ks * PR_ROWS + 2 * p) * PR_NC + 4 * cg) =
        make_float4(acc[p][0].x, acc[p][1].x, acc[p][2].x, acc[p][3].x);
    *reinterpret_cast<float4*>(red + (ks * PR_ROWS + 2 * p + 1) * PR_NC + 4 * cg) =
        make_float4(acc[p][0].y, acc[p][1].y, acc[p][2].y, acc[p][3].y);
  }
  consumer_sync();
  const int col = threadIdx.x & (PR_NC - 1), rh = threadIdx.x >> 7;
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const float* p = red + (4 * rh + r) * PR_NC + col;
    constexpr int SL = PR_ROWS * PR_NC;             // one k-slice of partials
    v[r] = ((p[0] + p[SL]) + (p[2 * SL] + p[3 * SL])) + ((p[4 * SL] + p[5 * SL]) + (p[6 * SL] + p[7 * SL]));
  }
}

// One forward net for the pair's 8 rows (first-layer input already in `xa` of both CTAs).  Returns the buffer that holds
// the last hidden activations; the partner's half of it is still in flight (X.wait() before reading all of it).
template <class PT>
__device__ __forceinline__ float* pair_forward_net(const PT& P, PairRing& rg, PairX& X, int ch0, int L, int gc0, float* xa,
                                                   float* xb, float* red, const float* const* bias, float* const* h_out,
                                                   int64_t row0) {
  const int col = threadIdx.x & (PR_NC - 1), rh = threadIdx.x >> 7, gcol = gc0 + col;
  float* xin = xa;
  float* xout = xb;
  for (int l = 0; l < L; ++l) {
    float v[4];
    const float b = bias[l][gcol];                // in flight during the layer (an exposed L2 round trip otherwise)
    pair_layer_gemv(P, rg, X, l == 0 ? ch0 : S_H / PR_CK, xin, red, v);
#pragma unroll
    for (int r = 0; r < 4; ++r) v[r] = fmaxf(v[r] + b, 0.f);
    if (h_out != nullptr) {
#pragma unroll
      for (int r = 0; r < 4; ++r) h_out[l][(row0 + 4 * rh + r) * S_H + gcol] = v[r];
    }
    X.put(xout, gcol, rh, v);
    consumer_sync();
    X.stamp();
    float* t = xin; xin = xout; xout = t;
  }
  return xin;
}

// backward through the hidden layers L-1 .. 1 of one net from the seed already exchanged into `xin`: masks from the
// row-major activations `h`, deltas optionally stored row-major into `dout`
template <class PT>
__device__ __forceinline__ float* pair_backward_net(const PT& P, PairRing& rg, PairX& X, int L, int gc0, float* xin, float* xout,
                                                    float* red, float* const* h, float* const* dout, int64_t row0) {
  const int col = threadIdx.x & (PR_NC - 1), rh = threadIdx.x >> 7, gcol = gc0 + col;
  for (int l = L - 1; l >= 1; --l) {
    float m[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) m[r] = __ldcg(h[l - 1] + (row0 + 4 * rh + r) * S_H + gcol);   // ReLU masks of layer l-1
    float v[4];
    pair_layer_gemv(P, rg, X, S_H / PR_CK, xin, red, v);
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      v[r] = relu_mask(v[r], m[r]);
      if (dout != nullptr) dout[l - 1][(row0 + 4 * rh + r) * S_H + gcol] = v[r];
    }
    X.put(xout, gcol, rh, v);
    consumer_sync();
    float* t = xin; xin = xout; xout = t;
  }
  return xin;
}

// first-layer input of the pair's 8 rows (two 4-row halves of build_x); the row-major global copy only from rank 0
__device__ __forceinline__ void pair_build_x(const StreamParams& P, float* xT, int64_t row0, bool target, int act_kind,
                                             const float* ths, float* gout, const float* stage) {
  const int ss = P.plan.stage_stride;
  build_x(P, xT, PR_ROWS, 0, row0, target, act_kind, ths, gout, stage);
  build_x(P, xT, PR_ROWS, 4, row0 + 4, target, act_kind, ths ? ths + 4 * S_DU : nullptr, gout,
          stage ? stage + 4 * ss : nullptr);
  // k rows [KP, KP + 64) are multiplied with zero-filled weight rows of the ragged first-layer chunks: keep them finite
  const int kend = (P.KP + PR_CK < S_H) ? P.KP + PR_CK : S_H;
  for (int i = P.KP * PR_ROWS + threadIdx.x; i < kend * PR_ROWS; i += S_CONSUMERS) xT[i] = 0.f;
}

__device__ __forceinline__ void pair_consumer(const PairParams& PP, float* ringf, float* xa, float* xb, float* red,
                                              float* misc, uint32_t full, uint32_t empty, uint32_t xbar) {
  const StreamParams& P = PP.S;
  float* s_th = misc;                 // [8][8] tanh output of this chain's pi net (= pi / max_u)
  float* s_q = misc + 64;             // [8][8] main.Q of the 8 rows
  float* s_qt = misc + 128;           // [8][8] target.Q
  float* s_dq = misc + 192;           // [8] backward seed; [8..16): squared TD error
  float* s_dy = misc + 256;           // [8][8]
  float* s_r = misc + 320;            // [8] rewards of the rows (fused HER sampling)
  const float** m_src = reinterpret_cast<const float**>(misc + 336);     // [8][3] source addresses
  float* her_stage = misc + PR_STAGE_OFF;                                 // [8][stage_stride]

  const int tid = threadIdx.x;
  const uint32_t rank = cluster_ctarank();
  const uint32_t pair = blockIdx.x >> 1;
  const uint32_t role = pair & 1;                              // 0: actor chain, 1: critic chain (independent pairs)
  const int64_t row0 = (int64_t)(pair >> 1) * PR_ROWS;
  const cur_net_desc& d = P.d;
  const int L = P.L;
  const int gc0 = (int)rank * PR_NC, col = tid & (PR_NC - 1), rh = tid >> 7, gcol = gc0 + col;
  const bool lead = rank == 0;                                 // writes what both CTAs compute redundantly

  PairRing rg;
  rg.chunks = PP.ch[role][rank]; rg.slots = ringf; rg.full = full; rg.empty = empty; rg.cons = 0;
  PairX X;
  X.bar_local[0] = xbar; X.bar_local[1] = xbar + 8;
  X.bar_remote[0] = map_to_cta(xbar, rank ^ 1u); X.bar_remote[1] = map_to_cta(xbar + 8, rank ^ 1u);
  X.x_local = smem_addr(xa); X.x_remote = map_to_cta(X.x_local, rank ^ 1u);
  X.word_remote = map_to_cta(smem_addr(misc + 400), rank ^ 1u);
  X.step = 0; X.pending = false;
  X.dbg = nullptr;

  const float inv_n = 1.0f / (float)P.grad_rows;      // scale of the backward seeds
  const float* stage = nullptr;
  if (P.fused_her) {
    sample_rows(P, row0, her_stage, m_src, s_r, red, PR_ROWS);
    stage = her_stage;
  }
  const float hi_clip = P.clip_pos ? 0.f : INFINITY;
  const bool tl_on = P.tl != nullptr && blockIdx.x == 0 && tid == 0;
#define PR_TL(i) do { if (tl_on) P.tl[i] = clock64(); } while (0)

  if (role == 1) {
    // ===== critic pair: target.pi -> target.Q(o2, g2, pi_target), main.Q(o, g, u), TD loss, the critic's backward chain
    pair_build_x(P, xa, row0, true, 0, nullptr, nullptr, stage);
    consumer_sync();
    float* xl = pair_forward_net(P, rg, X, PP.pch0[0], L, gc0, xa, xb, red, P.bPT, nullptr, row0);
    X.wait();
    small_out<S_H>(xl, PR_ROWS, 0, PR_ROWS, P.WoutPT, d.dimu, 1, d.dimu, P.boutPT, s_th);
    consumer_sync();
    if (tid < PR_ROWS * S_DU && (tid & (S_DU - 1)) < d.dimu) s_th[tid] = tanhf(s_th[tid]);
    X.sync();
    consumer_sync();
    pair_build_x(P, xa, row0, true, 2, s_th, nullptr, stage);
    consumer_sync();
    xl = pair_forward_net(P, rg, X, PP.pch0[1], L, gc0, xa, xb, red, P.bQT, nullptr, row0);
    X.wait();
    small_out<S_H>(xl, PR_ROWS, 0, PR_ROWS, P.WoutQT, 1, 1, 1, P.boutQT, s_qt);
    X.sync();
    consumer_sync();
    // main.Q(o, g, u)
    pair_build_x(P, xa, row0, false, 1, nullptr, lead ? P.Xq : nullptr, stage);
    consumer_sync();
    xl = pair_forward_net(P, rg, X, PP.pch0[1], L, gc0, xa, xb, red, P.bQ, P.hq, row0);
    X.wait();
    small_out<S_H>(xl, PR_ROWS, 0, PR_ROWS, P.WoutQ, 1, 1, 1, P.boutQ, s_q);
    consumer_sync();
    // critic loss (ddpg.py:436-439) and its backward seed
    if (tid < PR_ROWS) {
      const int64_t row = row0 + tid;
      const float rew = stage ? s_r[tid] : P.r[row];
      const float tgt = fminf(fmaxf(rew + P.gamma * s_qt[tid * S_DU], -P.clip_return), hi_clip);
      const float diff = tgt - s_q[tid * S_DU];
      s_dq[tid] = -2.0f * inv_n * diff;          // d mean((tgt - Q)^2) / dQ
      s_dq[8 + tid] = diff * diff;
      if (lead) P.dQ[row] = s_dq[tid];
    }
    X.sync();
    consumer_sync();
    if (lead && tid < 2) {                        // per 4 rows, like the 4-row kernel (same fold in rows_dw_kernel)
      float ssq = 0.f;
      for (int r = 0; r < 4; ++r) ssq += s_dq[8 + 4 * tid + r];
      P.loss_part[((row0 >> 2) + tid) * 4] = ssq;
    }
    // backward through main.Q (critic chain): gradient at the last hidden layer is dQ * Wout^T (Wout is [H][1])
    {
      const float wq = __ldg(P.WoutQ + gcol);
      float v[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        v[r] = relu_mask(s_dq[4 * rh + r] * wq, __ldcg(P.hq[L - 1] + (row0 + 4 * rh + r) * S_H + gcol));
        P.dc[L - 1][(row0 + 4 * rh + r) * S_H + gcol] = v[r];
      }
      X.put(xa, gcol, rh, v);
      consumer_sync();
    }
    pair_backward_net(P, rg, X, L, gc0, xa, xb, red, P.hq, P.dc, row0);
    X.wait();
    return;
  }

  // ===== actor pair: main.pi -> main.Q(o, g, pi) -> actor loss -> backward through main.Q and main.pi =====
  PR_TL(0);
  pair_build_x(P, xa, row0, false, 0, nullptr, lead ? P.Xp : nullptr, stage);
  consumer_sync();
  PR_TL(1);
  {
    if (tl_on) X.dbg = P.tl + 8;          // main.pi forward in detail: 24 stamps at most
    X.stamp();
    float* xl = pair_forward_net(P, rg, X, PP.pch0[0], L, gc0, xa, xb, red, P.bP, P.hp, row0);
    X.wait();
    X.dbg = nullptr;
    small_out<S_H>(xl, PR_ROWS, 0, PR_ROWS, P.WoutP, d.dimu, 1, d.dimu, P.boutP, s_th);
    consumer_sync();
    if (tid < PR_ROWS * S_DU && (tid & (S_DU - 1)) < d.dimu) s_th[tid] = tanhf(s_th[tid]);   // actor_critic.py:89
    X.sync();
    consumer_sync();
  }
  PR_TL(2);
  PR_TL(3);
  pair_build_x(P, xa, row0, false, 2, s_th, nullptr, stage);
  consumer_sync();
  {
    float* xl = pair_forward_net(P, rg, X, PP.pch0[1], L, gc0, xa, xb, red, P.bQ, P.hqp, row0);
    X.wait();
    small_out<S_H>(xl, PR_ROWS, 0, PR_ROWS, P.WoutQ, 1, 1, 1, P.boutQ, s_q);
    consumer_sync();
  }
  PR_TL(4);
  PR_TL(5);
  // ===== actor loss terms (ddpg.py:440-441) and backward seed =====
  if (tid < PR_ROWS) {
    s_dq[tid] = -inv_n;                        // d (-mean(Q_pi)) / dQ_pi
    if (lead) P.q_pi[row0 + tid] = s_q[tid * S_DU];
  }
  if (lead && tid < 2) {
    float sq = 0.f, sth = 0.f;
    for (int r = 4 * tid; r < 4 * tid + 4; ++r) {
      sq += s_q[r * S_DU];
      for (int j = 0; j < d.dimu; ++j) sth += s_th[r * S_DU + j] * s_th[r * S_DU + j];
    }
    float* lp = P.loss_part + ((row0 >> 2) + tid) * 4;
    lp[1] = sq; lp[2] = sth; lp[3] = 0.f;
  }
  X.sync();
  consumer_sync();
  // ===== backward through main.Q, actor-through-critic chain =====
  {
    {
      const float wq = __ldg(P.WoutQ + gcol);
      float v[4];
#pragma unroll
      for (int r = 0; r < 4; ++r)
        v[r] = relu_mask(s_dq[4 * rh + r] * wq, __ldcg(P.hqp[L - 1] + (row0 + 4 * rh + r) * S_H + gcol));
      X.put(xa, gcol, rh, v);
      consumer_sync();
    }
    float* xin = pair_backward_net(P, rg, X, L, gc0, xa, xb, red, P.hqp, nullptr, row0);
    X.wait();
    // gradient wrt the action inputs of main.Q, then through tanh and the action penalty (ddpg.py:440-441):
    // d pi_loss/d(pre-tanh) = (dL/d(pi/max_u) + action_l2*2/(B*dimu)*th) * (1 - th^2)
    small_out<S_H>(xin, PR_ROWS, 0, PR_ROWS, P.W0Q_act, 1, S_H, d.dimu, nullptr, s_dy);
    consumer_sync();
    if (tid < PR_ROWS * S_DU) {
      const int r = tid >> 3, j = tid & (S_DU - 1);
      float v = 0.f;
      if (j < d.dimu) {
        const float coef = P.action_l2 * 2.0f / (float)(P.grad_rows * d.dimu);
        const float th = s_th[tid];
        v = (s_dy[tid] + coef * th) * (1.f - th * th);
      }
      s_dy[tid] = v;
      if (lead && j < P.lddy) P.dy[(row0 + r) * P.lddy + j] = v;
    }
    X.sync();
    consumer_sync();
  }
  PR_TL(6);
  // ===== backward through main.pi =====
  {
    {
      float v[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) v[r] = 0.f;
      for (int j = 0; j < d.dimu; ++j) {
        const float wj = __ldg(P.WoutP + (int64_t)gcol * d.dimu + j);
#pragma unroll
        for (int r = 0; r < 4; ++r) v[r] = fmaf(s_dy[(4 * rh + r) * S_DU + j], wj, v[r]);
      }
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        v[r] = relu_mask(v[r], __ldcg(P.hp[L - 1] + (row0 + 4 * rh + r) * S_H + gcol));
        P.dp[L - 1][(row0 + 4 * rh + r) * S_H + gcol] = v[r];
      }
      X.put(xa, gcol, rh, v);
      consumer_sync();
    }
    pair_backward_net(P, rg, X, L, gc0, xa, xb, red, P.hp, P.dp, row0);
    X.wait();
  }
  PR_TL(7);
#undef PR_TL
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(S_THREADS, 1)
ddpg_stream_pair_kernel(const __grid_constant__ PairParams PP) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float* ringf = reinterpret_cast<float*>(smem_raw);
  float* xa = ringf + S_NSLOT * S_SLOT;
  float* xb = xa + S_XT;
  float* red = xb + S_XT;
  float* misc = red + S_RED;
  uint64_t* bars = reinterpret_cast<uint64_t*>(misc + PR_MISC);      // full[4], empty[4], xchg[2]
  const int tid = threadIdx.x;
  const uint32_t full = smem_addr(bars), empty = smem_addr(bars + S_NSLOT), xbar = smem_addr(bars + 2 * S_NSLOT);
  if (tid == 0) {
    for (int i = 0; i < S_NSLOT; ++i) {
      mbar_init(full + 8 * i, 1);
      mbar_init(empty + 8 * i, S_CONSUMERS / 32);
    }
    mbar_init(xbar, 1);
    mbar_init(xbar + 8, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  pdl_launch_dependents();
  pdl_wait();               // everything below reads what the previous kernel (weight gradients + Adam of the last update) wrote
  cluster_sync_all();       // both CTAs' barriers are initialised before anybody arrives on them (locally or remotely)

  if (tid >= S_CONSUMERS) {
    // ------------------------------------------------------------ producer warp: stream this CTA's half of every chunk
    if (tid == S_CONSUMERS) {
      const uint32_t rank = cluster_ctarank(), role = (blockIdx.x >> 1) & 1;
      const PairChunk* my = PP.ch[role][rank];
      const int total = PP.nch[role][rank];
      const uint32_t ring_s = smem_addr(ringf);
      for (int i = 0; i < total; ++i) {
        const int slot = i % S_NSLOT, round = i / S_NSLOT;
        if (round > 0) mbar_wait(empty + 8 * slot, (round - 1) & 1);
        mbar_expect_tx(full + 8 * slot, (uint32_t)S_SLOT * 4);          // a box always counts in full (zero-filled rows too)
        tc_tma_2d(ring_s + slot * S_SLOT * 4, &PP.maps[my[i].map], (int)rank * PR_NC, my[i].krow, full + 8 * slot);
      }
    }
  } else {
    pair_consumer(PP, ringf, xa, xb, red, misc, full, empty, xbar);
  }
  cluster_sync_all();       // neither CTA leaves while the partner may still store into it / arrive on its barriers
}

// ------------------------------------------------------------------------------------------------
// get_actions as ONE launch (ddpg.py:129-146 with _preprocess_og, :118-127): one CTA per 4 rows walks pi (and, for
// compute_Q, Q on the noise-free action) with the same weight ring / GEMV core as the update kernel.  Inputs may
// live in mapped pinned HOST memory (zero-copy over PCIe: a rollout step is n = 2 rows, 0.5 KB) and so may the outputs;
// the last CTA to finish then stores the call's sequence number into a host-visible word the caller polls - no
// memcpy calls, no stream synchronisation on the critical path of a rollout step (rollout.py:217,226).
constexpr int A_MAXCHUNK = 64;          // pi + Q forward chunks (L = 4: 2 * 27)

struct ActParams {
  cur_net_desc d;
  int in_sp, in_g, KP, L, nchunks;
  int dbg_skip_math;         // (read by the shared GEMV core)
  int ch0[2];                // chunks of the first layer: [0] pi, [1] Q
  int64_t n;
  const float *o, *g, *td;
  const float* ag;           // relative goals: g <- g - ag (ddpg.py:120-125), else NULL
  const float *o_mean, *o_std, *g_mean, *g_std;
  float clip;                // clip o, g to +-clip (<= 0: off)
  uint32_t seq;              // != 0: outputs are 8-byte words {float32 bits | seq << 32} the host polls ("LL" words)
  const float *bP[S_MAXL], *bQ[S_MAXL];
  const float *WoutP, *boutP, *WoutQ, *boutQ;
  void *pi, *q;              // [n][dimu], [n] (or NULL): float32, or LL words when seq != 0
  long long* tl;
  SChunk chunks[A_MAXCHUNK];
};

// (the normaliser statistics are arguments: the routed kernel takes them from its CTA's expert)
template <class PT>
__device__ __forceinline__ float act_x_elem(const PT& P, const float* o_mean, const float* o_std, const float* g_mean,
                                            const float* g_std, int64_t row, int r, int k, int act_kind, const float* ths) {
  const cur_net_desc& d = P.d;
  const bool nrm = d.normalize_obs != 0;
  const int in_s = P.in_sp + (act_kind ? d.dimu : 0);
  const float clip = P.clip;
  float v = 0.f;
  int gj = -1, aj = -1;
  if (k < d.dimo) {
    v = P.o[row * d.dimo + k];
    if (clip > 0.f) v = fminf(fmaxf(v, -clip), clip);
    if (nrm) v = norm1s(v, o_mean, o_std, k, d.norm_clip);
  } else if (d.modular) {
    if (k < d.dimo + d.dimtd) v = P.td[row * d.dimtd + (k - d.dimo)];       // never normalised
    else if (k < in_s) aj = k - d.dimo - d.dimtd;
    else if (k < in_s + d.dimg) gj = k - in_s;
  } else {
    if (k < d.dimo + d.dimg) gj = k - d.dimo;
    else if (k < in_s) aj = k - d.dimo - d.dimg;
  }
  if (gj >= 0) {
    v = P.g[row * d.dimg + gj];
    if (P.ag) v = __fsub_rn(v, P.ag[row * d.dimg + gj]);
    if (clip > 0.f) v = fminf(fmaxf(v, -clip), clip);
    if (nrm) v = norm1s(v, g_mean, g_std, gj, d.norm_clip);
  }
  if (aj >= 0) v = ths[r * S_DU + aj];
  return v;
}

// an output element: plain float32, or - seq != 0 - one naturally aligned 8-byte word {value | seq << 32}: a 64-bit
// store is single-copy atomic (also across PCIe), so the host polls the data words themselves and the kernel needs
// neither a system fence nor a completion ticket
__device__ __forceinline__ void put_out(void* base, int64_t i, float v, uint32_t seq) {
  if (seq == 0) reinterpret_cast<float*>(base)[i] = v;
  else st_ll(reinterpret_cast<unsigned long long*>(base) + i, v, seq);
}

template <int H>
__global__ void __launch_bounds__(S_THREADS, 1)
actions_stream_kernel(const __grid_constant__ ActParams P) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float* ringf = reinterpret_cast<float*>(smem_raw);
  float* xa = ringf + S_NSLOT * S_SLOT;
  float* xb = xa + S_XT;
  float* red = xb + S_XT;
  float* misc = red + S_RED;
  uint64_t* bars = reinterpret_cast<uint64_t*>(misc + S_MISC);
  float* s_th = misc;                 // [4][8] tanh output
  float* s_q = misc + 64;             // [4][8]
  const int tid = threadIdx.x;
  const int64_t row0 = (int64_t)blockIdx.x * S_ROWS;
  const cur_net_desc& d = P.d;
  const uint32_t full = smem_addr(bars), empty = smem_addr(bars + S_NSLOT);
  if (tid == 0) {
    for (int i = 0; i < S_NSLOT; ++i) {
      mbar_init(full + 8 * i, 1);
      mbar_init(empty + 8 * i, S_CONSUMERS / 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (tid >= S_CONSUMERS) {
    if (tid == S_CONSUMERS) {
      const uint32_t ring_s = smem_addr(ringf);
      for (int i = 0; i < P.nchunks; ++i) {
        const int slot = i % S_NSLOT, round = i / S_NSLOT;
        if (round > 0) mbar_wait(empty + 8 * slot, (round - 1) & 1);
        const uint32_t bytes = (uint32_t)P.chunks[i].nrows * H * 4;
        mbar_expect_tx(full + 8 * slot, bytes);
        bulk_g2s(ring_s + slot * S_SLOT * 4, P.chunks[i].src, bytes, full + 8 * slot);
      }
    }
    return;
  }
  Ring rg;
  rg.chunks = P.chunks; rg.slots = ringf; rg.full = full; rg.empty = empty; rg.cons = 0;
  const int nr = (int)((P.n - row0 < S_ROWS) ? P.n - row0 : S_ROWS);      // rows of this CTA that exist
#define A_TL(i)                                                                              \
  do {                                                                                       \
    if (P.tl != nullptr && tid == 0 && blockIdx.x == 0) P.tl[i] = (long long)globaltimer_ns(); \
  } while (0)
  A_TL(0);
  auto build = [&](int act_kind) {
    for (int idx = tid; idx < S_ROWS * P.KP; idx += S_CONSUMERS) {
      const int k = idx >> 2, r = idx & 3;
      xa[k * 4 + r] = act_x_elem(P, P.o_mean, P.o_std, P.g_mean, P.g_std, row0 + (r < nr ? r : nr - 1), r, k, act_kind,
                                 s_th);
    }
  };
  build(0);
  consumer_sync();
  A_TL(1);
  float* xl = forward_net<H, 4>(P, rg, P.ch0[0], xa, xb, red, P.bP, nullptr, nullptr, row0);
  small_out<H>(xl, 4, 0, 4, P.WoutP, d.dimu, 1, d.dimu, P.boutP, s_th);
  consumer_sync();
  A_TL(2);
  if (tid < S_ROWS * S_DU && (tid & (S_DU - 1)) < d.dimu) {
    const float th = tanhf(s_th[tid]);                                  // actor_critic.py:89
    s_th[tid] = th;
    const int r = tid >> 3, j = tid & (S_DU - 1);
    if (r < nr) put_out(P.pi, (row0 + r) * d.dimu + j, d.max_u * th, P.seq);
  }
  consumer_sync();
  if (P.q != nullptr) {
    build(2);                                                          // Q(o, g, pi / max_u): the noise-free action
    consumer_sync();
    xl = forward_net<H, 4>(P, rg, P.ch0[1], xa, xb, red, P.bQ, nullptr, nullptr, row0);
    small_out<H>(xl, 4, 0, 4, P.WoutQ, 1, 1, 1, P.boutQ, s_q);
    consumer_sync();
    if (tid < nr) put_out(P.q, row0 + tid, s_q[tid * S_DU], P.seq);
  }
  A_TL(3);
#undef A_TL
}

// ------------------------------------------------------------------------------------------------
// The routed form (a task-experts evaluation step, rollout.py:211-223: each row is acted on by the expert of its module):
// the same CTA per 4 rows, ring and GEMV core, but every CTA tile belongs to one expert and takes that expert's weights
// and normaliser statistics from a per-launch table.  The host groups the rows by expert (each group padded to a multiple
// of 4) into a row map; inputs are read from and outputs written to the rows' original positions.  All experts share one
// cur_net_desc, so the chunk list is one list of offsets into any expert's theta.
constexpr int G_MAXROWS = 512;                                   // rows per routed launch
constexpr int G_MAXTILES = G_MAXROWS / S_ROWS + CUR_MAX_TASKS;   // each expert's group rounds up to whole tiles

struct ActExpert {
  const float* theta;
  const float *o_mean, *o_std, *g_mean, *g_std;
  const float *bP[S_MAXL], *bQ[S_MAXL];
  const float *WoutP, *boutP, *WoutQ, *boutQ;
};

struct ActGroupParams {
  cur_net_desc d;
  int in_sp, in_g, KP, L, nchunks;
  int dbg_skip_math;         // (read by the shared GEMV core)
  int ch0[2];
  const float *o, *g, *td, *ag;
  float clip;
  uint32_t seq;
  void *pi, *q;
  SChunk chunks[A_MAXCHUNK];           // nrows / k0 of every chunk (src unused: see coff)
  int32_t coff[A_MAXCHUNK];            // float offset of every chunk in an expert's theta
  ActExpert ex[CUR_MAX_TASKS];
  uint8_t tile_ex[G_MAXTILES];         // expert of every CTA
  int16_t tile_row[G_MAXTILES][S_ROWS];   // original row of every slot; -1: padding (valid slots come first)
};

template <int H>
__global__ void __launch_bounds__(S_THREADS, 1)
actions_group_kernel(const __grid_constant__ ActGroupParams P) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float* ringf = reinterpret_cast<float*>(smem_raw);
  float* xa = ringf + S_NSLOT * S_SLOT;
  float* xb = xa + S_XT;
  float* red = xb + S_XT;
  float* misc = red + S_RED;
  uint64_t* bars = reinterpret_cast<uint64_t*>(misc + S_MISC);
  float* s_th = misc;                 // [4][8] tanh output
  float* s_q = misc + 64;             // [4][8]
  const int tid = threadIdx.x;
  const ActExpert& E = P.ex[P.tile_ex[blockIdx.x]];
  const cur_net_desc& d = P.d;
  const uint32_t full = smem_addr(bars), empty = smem_addr(bars + S_NSLOT);
  if (tid == 0) {
    for (int i = 0; i < S_NSLOT; ++i) {
      mbar_init(full + 8 * i, 1);
      mbar_init(empty + 8 * i, S_CONSUMERS / 32);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (tid >= S_CONSUMERS) {
    if (tid == S_CONSUMERS) {
      const uint32_t ring_s = smem_addr(ringf);
      for (int i = 0; i < P.nchunks; ++i) {
        const int slot = i % S_NSLOT, round = i / S_NSLOT;
        if (round > 0) mbar_wait(empty + 8 * slot, (round - 1) & 1);
        const uint32_t bytes = (uint32_t)P.chunks[i].nrows * H * 4;
        mbar_expect_tx(full + 8 * slot, bytes);
        bulk_g2s(ring_s + slot * S_SLOT * 4, E.theta + P.coff[i], bytes, full + 8 * slot);
      }
    }
    return;
  }
  Ring rg;
  rg.chunks = P.chunks; rg.slots = ringf; rg.full = full; rg.empty = empty; rg.cons = 0;
  const int16_t* tile = P.tile_row[blockIdx.x];
  int nr = 0;
#pragma unroll
  for (int r = 0; r < S_ROWS; ++r) nr += tile[r] >= 0;
  auto row_of = [&](int r) -> int64_t { return tile[r] >= 0 ? tile[r] : tile[0]; };   // padding repeats the first row
  auto build = [&](int act_kind) {
    for (int idx = tid; idx < S_ROWS * P.KP; idx += S_CONSUMERS) {
      const int k = idx >> 2, r = idx & 3;
      xa[k * 4 + r] = act_x_elem(P, E.o_mean, E.o_std, E.g_mean, E.g_std, row_of(r), r, k, act_kind, s_th);
    }
  };
  build(0);
  consumer_sync();
  float* xl = forward_net<H, 4>(P, rg, P.ch0[0], xa, xb, red, E.bP, nullptr, nullptr, 0);
  small_out<H>(xl, 4, 0, 4, E.WoutP, d.dimu, 1, d.dimu, E.boutP, s_th);
  consumer_sync();
  if (tid < S_ROWS * S_DU && (tid & (S_DU - 1)) < d.dimu) {
    const float th = tanhf(s_th[tid]);                                  // actor_critic.py:89
    s_th[tid] = th;
    const int r = tid >> 3, j = tid & (S_DU - 1);
    if (r < nr) put_out(P.pi, row_of(r) * d.dimu + j, d.max_u * th, P.seq);
  }
  consumer_sync();
  if (P.q != nullptr) {
    build(2);                                                          // Q(o, g, pi / max_u): the noise-free action
    consumer_sync();
    xl = forward_net<H, 4>(P, rg, P.ch0[1], xa, xb, red, E.bQ, nullptr, nullptr, 0);
    small_out<H>(xl, 4, 0, 4, E.WoutQ, 1, 1, 1, E.boutQ, s_q);
    consumer_sync();
    if (tid < nr) put_out(P.q, row_of(tid), s_q[tid * S_DU], P.seq);
  }
}

// W^T of the hidden layers (operands of the backward streams): dst[m][j][i] = src_m[i][j], H x H each
struct TransposeParams {
  const float* src[2 * S_MAXL];
  float* dst[2 * S_MAXL];
};

template <int H>
__global__ void __launch_bounds__(256) transpose_kernel(const __grid_constant__ TransposeParams T) {
  __shared__ float tile[32][33];
  const float* src = T.src[blockIdx.z];
  float* dst = T.dst[blockIdx.z];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int i0 = blockIdx.y * 32, j0 = blockIdx.x * 32;
#pragma unroll
  for (int q = 0; q < 4; ++q) tile[ty + 8 * q][tx] = src[(int64_t)(i0 + ty + 8 * q) * H + j0 + tx];
  __syncthreads();
#pragma unroll
  for (int q = 0; q < 4; ++q) dst[(int64_t)(j0 + ty + 8 * q) * H + i0 + tx] = tile[tx][ty + 8 * q];
}

static void launch_transposes(const TransposeParams& TP, int m, int H, cudaStream_t s) {
  const dim3 grid(H / 32, H / 32, m);
  if (H == 64) transpose_kernel<64><<<grid, 256, 0, s>>>(TP);
  else if (H == 128) transpose_kernel<128><<<grid, 256, 0, s>>>(TP);
  else transpose_kernel<256><<<grid, 256, 0, s>>>(TP);
}

// ------------------------------------------------------------------------------------------------
// launch 2: all weight gradients (+ optional Adam), loss fold, step counter
// ------------------------------------------------------------------------------------------------
// ---------------------------------------------------------------- tile-level gradient exchange (several ranks)
// cur_xchg_ctx resolved for the device: every element travels as ONE naturally aligned 8-byte word
// {float32 bits | update number << 32} ("LL" protocol): a scalar 64-bit store is single-copy atomic, so the
// receiver polls the data words themselves - no flag round, no system fence on the critical path.
struct XchgDev {
  int rank, world, mode;
  unsigned long long* part[CUR_MAX_RANKS];   // partial slots of rank r's region: [world][arena]
  unsigned long long* res[CUR_MAX_RANKS];    // result slots of rank r's region: [arena]
  int64_t arena;
  long long* tl;                             // optional [tiles][4] %globaltimer stamps
  int* error_flag;
  // mode 2 (NVLS): the regions are ONE symmetric allocation with a multicast mapping - a load from part_mc is reduced by
  // the NVSwitch over every rank's copy, a store to res_mc lands in every rank's copy
  const float2* part_mc;                     // multicast alias of the partial slots [arena] {value, update number as float}
  unsigned long long* res_mc;                // multicast alias of the result slots [arena]
};

__device__ __forceinline__ unsigned long long ld_ll(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
// a peer that does not show up for ~20 s is dead or diverged: fail loudly (the host sees a launch failure)
__device__ __noinline__ void xchg_timeout_check(unsigned long long t0, int* error_flag) {
  if (globaltimer_ns() - t0 > 20000000000ull) {
    if (error_flag) *error_flag = 1;
    __threadfence_system();
    __trap();
  }
}

struct DwTail {
  int dbg_skip_stage;              // debug (CUR_DW_SKIP_STAGE=1): tiles run on whatever their shared memory holds
  int pdl_late;                    // trigger the dependent launch when the tile is done (not at the start)
  AdamCtx ax;                      // ax.theta == NULL: gradients only
  const float* neg_a_table;
  int table_len;
  int64_t* step_counter;           // may be NULL
  int ring;
  unsigned int* ticket;
  const float* loss_part;
  int n_clusters;
  int64_t n;
  int dimu;
  float action_l2;
  float *q_loss, *pi_loss;
  long long* tl;                   // debug timeline (CUR_ROWS_TIMELINE)
  int tl_skinny_block;
  int64_t parity_stride;           // > 0: gradients go to C + ((update + 1) & 1) * parity_stride (peer-memory exchange)
  int micro;                       // micro-batches (workers) per update: launch j = step % micro accumulates for j > 0
  int chunk, last_chunk;           // batches > 256 rows: one launch per 256-row K chunk; chunks > 0 accumulate, only the
                                   // last one runs the optimiser epilogue, folds the losses and bumps the step counter
  int xc_on;                       // several ranks: exchange the tiles with the peers before the step (xc)
  XchgDev xc;
};

// Epilogue context of one CTA (shared memory), resolved once from DwTail and the device step counter.
struct DwCtx {
  AdamCtx ax;
  int opt;                         // the optimiser runs in this launch (last chunk, last micro-batch of the update)
  int xc_on;                       // ... after the tile went through the exchange
  int own;                         // this rank reduces the tile
  int owner;                       // the rank that does (mode 1)
  uint32_t flag;                   // update number travelling with the data
  long long* tl;                   // this tile's stamps or NULL
  long long* dbg;                  // debug: clock64 stamps inside a traced full-K tile ([4..7] of its timeline row) or NULL
};

// Sum of the world's partial tiles in rank order (bit-identical on every reducer): g[e] holds this rank's partial on
// entry and the sum on return.  All peers' words of two elements are requested before the first check, so a tile
// whose data has landed costs two L2 round trips, not 4 x (W - 1).
template <int NE>
__device__ __forceinline__ void xchg_reduce(const XchgDev& xc, uint32_t flag, const int64_t (&off)[NE],
                                            const bool (&ok)[NE], float (&g)[NE]) {
  const unsigned long long* mine = xc.part[xc.rank];
  constexpr int EB = NE >= 2 ? 2 : 1;
#pragma unroll
  for (int e0 = 0; e0 < NE; e0 += EB) {
    unsigned long long x[EB][CUR_MAX_RANKS];
    bool all;
    unsigned int spins = 0;
    unsigned long long t0 = 0;
    do {
      all = true;
#pragma unroll
      for (int q = 0; q < EB; ++q)
#pragma unroll
        for (int r = 0; r < CUR_MAX_RANKS; ++r)
          if (r < xc.world && r != xc.rank && ok[e0 + q]) x[q][r] = ld_ll(mine + (int64_t)r * xc.arena + off[e0 + q]);
#pragma unroll
      for (int q = 0; q < EB; ++q)
#pragma unroll
        for (int r = 0; r < CUR_MAX_RANKS; ++r)
          if (r < xc.world && r != xc.rank && ok[e0 + q]) all = all && ((uint32_t)(x[q][r] >> 32) == flag);
      if (!all && (++spins & 0x3FFFu) == 0) {
        if (t0 == 0) t0 = globaltimer_ns();
        xchg_timeout_check(t0, xc.error_flag);
      }
    } while (!all);
#pragma unroll
    for (int q = 0; q < EB; ++q) {
      if (!ok[e0 + q]) continue;
      float s = 0.f;
#pragma unroll
      for (int r = 0; r < CUR_MAX_RANKS; ++r)
        if (r < xc.world) {
          const float xr = (r == xc.rank) ? g[e0 + q] : __uint_as_float((uint32_t)x[q][r]);
          s = (r == 0) ? xr : __fadd_rn(s, xr);
        }
      g[e0 + q] = s;
    }
  }
}

// mode 1, not the owner: the stepped parameters of the tile as pushed by the owner
template <int NE>
__device__ __forceinline__ void xchg_wait_result(const XchgDev& xc, uint32_t flag, const int64_t (&off)[NE],
                                                 const bool (&ok)[NE], float (&th)[NE]) {
  const unsigned long long* mine = xc.res[xc.rank];
  unsigned long long x[NE];
  bool all;
  unsigned int spins = 0;
  unsigned long long t0 = 0;
  do {
    all = true;
#pragma unroll
    for (int e = 0; e < NE; ++e)
      if (ok[e]) x[e] = ld_ll(mine + off[e]);
#pragma unroll
    for (int e = 0; e < NE; ++e)
      if (ok[e]) all = all && ((uint32_t)(x[e] >> 32) == flag);
    if (!all && (++spins & 0x3FFFu) == 0) {
      if (t0 == 0) t0 = globaltimer_ns();
      xchg_timeout_check(t0, xc.error_flag);
    }
  } while (!all);
#pragma unroll
  for (int e = 0; e < NE; ++e)
    if (ok[e]) th[e] = __uint_as_float((uint32_t)x[e]);
}

// mode 2, the owner: ONE multimem.ld_reduce per element returns the switch-reduced sum of the world's {value, number}
// pairs - the value half is the gradient sum, the number half equals world x number exactly once every rank's pair of
// THIS update has landed (a pair is one naturally aligned 8-byte store; older pairs carry a smaller number).
template <int NE>
__device__ __forceinline__ void xchg_reduce_nvls(const XchgDev& xc, float want, const int64_t (&off)[NE],
                                                 const bool (&ok)[NE], float (&g)[NE]) {
  float sv[NE], sf[NE];
  bool all;
  unsigned int spins = 0;
  unsigned long long t0 = 0;
  do {
    all = true;
#pragma unroll
    for (int e = 0; e < NE; ++e)
      if (ok[e])
        asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v2.f32 {%0, %1}, [%2];"
                     : "=f"(sv[e]), "=f"(sf[e]) : "l"(xc.part_mc + off[e]) : "memory");
#pragma unroll
    for (int e = 0; e < NE; ++e)
      if (ok[e]) all = all && (sf[e] == want);
    if (!all && (++spins & 0x3FFu) == 0) {
      if (t0 == 0) t0 = globaltimer_ns();
      xchg_timeout_check(t0, xc.error_flag);
    }
  } while (!all);
#pragma unroll
  for (int e = 0; e < NE; ++e)
    if (ok[e]) g[e] = sv[e];
}

// The end of every weight-gradient element: local gradient (accumulated over micro-batches / K chunks), exchange with
// the peers, Adam.  v[e] is the tile value of this launch, c[e] its place in the local gradient arena; th[e] returns
// the stepped parameter (undefined unless cx.opt).
template <int NE>
__device__ __forceinline__ void dw_finish(const DwTail& T, const DwCtx& cx, float* const (&c)[NE], const bool (&ok)[NE],
                                          bool accumulate, float (&v)[NE], float (&th)[NE]) {
  int64_t off[NE];
#pragma unroll
  for (int e = 0; e < NE; ++e) {
    off[e] = 0; th[e] = 0.f;
    if (ok[e]) {
      if (accumulate) v[e] += *c[e];   // micro-batch j > 0 / K chunk > 0 adds to the running sum
      *c[e] = v[e];
      off[e] = c[e] - cx.ax.grads;
    }
  }
  if (!cx.opt) return;
  if (cx.xc_on) {
    const XchgDev& xc = T.xc;
    if (cx.tl && threadIdx.x == 0) cx.tl[1] = (long long)globaltimer_ns();
    if (xc.mode == 0) {
#pragma unroll
      for (int r = 0; r < CUR_MAX_RANKS; ++r)
        if (r < xc.world && r != xc.rank) {
          unsigned long long* dst = xc.part[r] + (int64_t)xc.rank * xc.arena;
#pragma unroll
          for (int e = 0; e < NE; ++e)
            if (ok[e]) st_ll(dst + off[e], v[e], cx.flag);
        }
    } else if (xc.mode == 2) {
      // NVLS: every rank (the owner too) publishes its partial in its OWN slots; the number travels as a float so that
      // the switch can add it up (exact: world x 2^20 < 2^24)
      const float nf = (float)((cx.flag & 0xFFFFFu) + 1u);
      unsigned long long* dst = xc.part[xc.rank];
#pragma unroll
      for (int e = 0; e < NE; ++e)
        if (ok[e]) st_ll(dst + off[e], v[e], __float_as_uint(nf));
    } else if (!cx.own) {
      unsigned long long* dst = xc.part[cx.owner] + (int64_t)xc.rank * xc.arena;
#pragma unroll
      for (int e = 0; e < NE; ++e)
        if (ok[e]) st_ll(dst + off[e], v[e], cx.flag);
    }
    if (cx.own) {
      if (xc.mode == 2) xchg_reduce_nvls<NE>(xc, (float)xc.world * (float)((cx.flag & 0xFFFFFu) + 1u), off, ok, v);
      else xchg_reduce<NE>(xc, cx.flag, off, ok, v);
      if (cx.tl && threadIdx.x == 0) cx.tl[2] = (long long)globaltimer_ns();
    } else {
      xchg_wait_result<NE>(xc, cx.flag, off, ok, th);
      if (cx.tl && threadIdx.x == 0) cx.tl[2] = (long long)globaltimer_ns();
#pragma unroll
      for (int e = 0; e < NE; ++e)
        if (ok[e]) cx.ax.theta[off[e]] = th[e];
      return;
    }
  }
#pragma unroll
  for (int e = 0; e < NE; ++e)
    if (ok[e]) {
      float t = cx.ax.theta[off[e]], mm = cx.ax.m[off[e]], vv = cx.ax.v[off[e]];
      adam_elem(t, v[e], mm, vv, cx.ax.neg_a, cx.ax.b1, cx.ax.omb1, cx.ax.b2, cx.ax.omb2, cx.ax.eps);
      cx.ax.theta[off[e]] = t; cx.ax.m[off[e]] = mm; cx.ax.v[off[e]] = vv;
      th[e] = t;
    }
  if (cx.xc_on && T.xc.mode == 1) {
    const XchgDev& xc = T.xc;
#pragma unroll
    for (int r = 0; r < CUR_MAX_RANKS; ++r)
      if (r < xc.world && r != xc.rank) {
#pragma unroll
        for (int e = 0; e < NE; ++e)
          if (ok[e]) st_ll(xc.res[r] + off[e], th[e], cx.flag);
      }
  } else if (cx.xc_on && T.xc.mode == 2) {
    // one store to the multicast alias: the switch delivers the stepped parameter to every rank's result slot
#pragma unroll
    for (int e = 0; e < NE; ++e)
      if (ok[e]) st_ll(T.xc.res_mc + off[e], th[e], cx.flag);
  }
}

// Tile kinds of the weight-gradient launch (K = batch <= 256 is the reduction dimension):
//   DW_FULLK   C[32x32 tile] = A^T B, A = X [K][M] and B = dY [K][N] both staged for the WHOLE K with one burst of
//              cp.async (one L2 round trip instead of a multi-stage pipeline of dependent ones), 4-way split-K
//              inside the CTA, packed FFMA2; 3 CTAs per SM so that all ~330 tiles are co-resident (one wave)
//   DW_SKINNY  N <= 4 (output layers): 32 rows of C per tile, 8 k-parts per row
//   DW_COLSUM  C[n] = sum_k B[k][n] (bias gradients), 32 columns per tile, 8 k-parts per column
// (A 64 x 64 / 8 x 8-micro-tile variant, which is not bound by shared-memory wavefronts, measured slower here:
//  88 fat CTAs leave 60 SMs idle and cannot overlap staging with compute - see profiles/README.md.)
enum { DW_FULLK = 0, DW_SKINNY = 1, DW_COLSUM = 2 };
constexpr int DW_KMAX = 256;
constexpr int DW_LD = GT + 4;                                   // row stride of a staged [k][32] tile
constexpr size_t DW_SMEM_BYTES = (size_t)2 * DW_KMAX * DW_LD * 4;

// ---- stage A[k][m0..m0+32) and B[k][n0..n0+32) for every k (zero fill past the edges); issued before anything that
// depends on the device step counter, so that the two dependent round trips of that setup overlap this one
// (Committing the burst as 4 groups of 64 k rows and running the math of a group while the later ones travel was measured
// SLOWER - 55.3 instead of 53.4 us per update: the last operands land at +12.3 k cycles instead of +8.2 k, the cp.async
// writes and the LDS of the math share the same shared-memory pipe.)
__device__ __forceinline__ void dw_stage_fullk(const GemmProb& P, float* As, float* Bs, int m0, int n0) {
  const int tid = threadIdx.x;
#pragma unroll
  for (int j = 0; j < (DW_KMAX * 8) / GEMM_THREADS; ++j) {
    const int f = tid + j * GEMM_THREADS;
    const int k = f >> 3, c4 = (f & 7) << 2;
    const bool oka = (k < P.K) && (m0 + c4 < P.M);
    cp16_zfill(As + k * DW_LD + c4, P.A + (oka ? (int64_t)k * P.lda + (m0 + c4) : 0), oka);
    const bool okb = (k < P.K) && (n0 + c4 < P.N);
    cp16_zfill(Bs + k * DW_LD + c4, P.B + (okb ? (int64_t)k * P.ldb + (n0 + c4) : 0), okb);
  }
  cp_commit();
}

__device__ __forceinline__ void dw_tile_fullk(const GemmProb& P, float* As, float* Bs, int m0, int n0, const DwTail& T,
                                              const DwCtx& cx) {
  const int tid = threadIdx.x;
  cp_wait0();
  __syncthreads();
  if (tid == 0 && cx.dbg) cx.dbg[4] = clock64();
  const int kg = tid >> 6, lt = tid & 63, ty = lt >> 3, tx = lt & 7;
  float2 acc[4][2];
#pragma unroll
  for (int i = 0; i < 4; ++i) acc[i][0] = acc[i][1] = make_float2(0.f, 0.f);
  const float* ap = As + (kg * (DW_KMAX / 4)) * DW_LD + 4 * ty;
  const float* bp = Bs + (kg * (DW_KMAX / 4)) * DW_LD + 4 * tx;
#pragma unroll 8
  for (int k = 0; k < DW_KMAX / 4; ++k) {
    const float4 a = *reinterpret_cast<const float4*>(ap + k * DW_LD);
    const float4 b = *reinterpret_cast<const float4*>(bp + k * DW_LD);
    const float2 b01 = make_float2(b.x, b.y), b23 = make_float2(b.z, b.w);
    acc[0][0] = __ffma2_rn(make_float2(a.x, a.x), b01, acc[0][0]);
    acc[0][1] = __ffma2_rn(make_float2(a.x, a.x), b23, acc[0][1]);
    acc[1][0] = __ffma2_rn(make_float2(a.y, a.y), b01, acc[1][0]);
    acc[1][1] = __ffma2_rn(make_float2(a.y, a.y), b23, acc[1][1]);
    acc[2][0] = __ffma2_rn(make_float2(a.z, a.z), b01, acc[2][0]);
    acc[2][1] = __ffma2_rn(make_float2(a.z, a.z), b23, acc[2][1]);
    acc[3][0] = __ffma2_rn(make_float2(a.w, a.w), b01, acc[3][0]);
    acc[3][1] = __ffma2_rn(make_float2(a.w, a.w), b23, acc[3][1]);
  }
  __syncthreads();                       // everybody is done with the staged tiles: reuse them for the partials
  if (tid == 0 && cx.dbg) cx.dbg[5] = clock64();
  float* red = As;                       // 4 x [32][32]
#pragma unroll
  for (int i = 0; i < 4; ++i)
    *reinterpret_cast<float4*>(red + kg * (GT * GT) + (4 * ty + i) * GT + 4 * tx) =
        make_float4(acc[i][0].x, acc[i][0].y, acc[i][1].x, acc[i][1].y);
  __syncthreads();
  // hidden layers with the fused optimiser: keep W^T (the backward operand of the next update's stream kernel) current
  // right here instead of re-transposing every update; the stepped tile is turned in shared memory (Bs is free by
  // now) so that the transposed stores are as coalesced as the direct ones
  const bool keep_t = cx.opt && P.C2 != nullptr;
  float* tt = Bs;                        // [32 n][33]
  constexpr int NE = (GT * GT) / GEMM_THREADS;
  float* c[NE];
  bool ok[NE];
  float v[NE], th[NE];
#pragma unroll
  for (int j = 0; j < NE; ++j) {
    const int i = tid + j * GEMM_THREADS;
    const int gm = m0 + (i >> 5), gn = n0 + (i & 31);
    ok[j] = gm < P.M && gn < P.N;
    c[j] = P.C + (int64_t)gm * P.ldc + gn;
    v[j] = (red[i] + red[GT * GT + i]) + (red[2 * GT * GT + i] + red[3 * GT * GT + i]);
  }
  if (tid == 0 && cx.dbg) cx.dbg[6] = clock64();
  dw_finish<NE>(T, cx, c, ok, P.accumulate != 0, v, th);
  if (tid == 0 && cx.dbg) cx.dbg[7] = clock64();
  if (keep_t) {
#pragma unroll
    for (int j = 0; j < NE; ++j) {
      const int i = tid + j * GEMM_THREADS;
      if (ok[j]) tt[(i & 31) * (GT + 1) + (i >> 5)] = th[j];
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < NE; ++j) {
      const int i = tid + j * GEMM_THREADS;
      const int gn = n0 + (i >> 5), gm = m0 + (i & 31);
      if (gm < P.M && gn < P.N) P.C2[(int64_t)gn * P.ldc2 + gm] = tt[(i >> 5) * (GT + 1) + (i & 31)];
    }
  }
}

// C[m][j] = sum_k A[k][m] * B[k*ldb + j], j < N <= 4, for the 32 rows m0.. of C; 8 interleaved k-parts per row.
// Both operands are staged for the whole K in ONE round trip (A with cp.async like a full-K tile, B with one plain load
// per thread): the first version took its operands in four dependent batches of loads, each queued behind the 128 KB of
// staging traffic of the two full-K tiles on the same SM - 18.5 k cycles, the longest tile of the launch.
__device__ __forceinline__ void dw_stage_skinny(const GemmProb& P, float* As, float* Bs, int m0) {
  const int tid = threadIdx.x;
  const int N = P.N;
#pragma unroll
  for (int j = 0; j < (DW_KMAX * 8) / GEMM_THREADS; ++j) {
    const int f = tid + j * GEMM_THREADS;
    const int k = f >> 3, c4 = (f & 7) << 2;
    const bool oka = (k < P.K) && (m0 + c4 < P.M) && P.lda % 4 == 0;
    cp16_zfill(As + k * DW_LD + c4, P.A + (oka ? (int64_t)k * P.lda + (m0 + c4) : 0), oka);
  }
  cp_commit();
  {
    const int k = tid;                                       // GEMM_THREADS == DW_KMAX: one B row per thread
    float b[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) b[j] = (k < P.K && j < N) ? __ldg(P.B + (int64_t)k * P.ldb + j) : 0.f;
    *reinterpret_cast<float4*>(Bs + 4 * k) = make_float4(b[0], b[1], b[2], b[3]);
  }
  if (P.lda % 4 != 0) {                                      // (never for the shapes of the rows schedule: ld = 256)
    for (int f = tid; f < DW_KMAX * GT; f += GEMM_THREADS) {
      const int k = f >> 5, mm = f & 31;
      As[k * DW_LD + mm] = (k < P.K && m0 + mm < P.M) ? __ldg(P.A + (int64_t)k * P.lda + m0 + mm) : 0.f;
    }
  }
}

__device__ __forceinline__ void dw_tile_skinny(const GemmProb& P, float* As, float* Bs, int m0, const DwTail& T,
                                               const DwCtx& cx) {
  const int tid = threadIdx.x, m = tid & 31, kp = tid >> 5;
  cp_wait0();
  __syncthreads();
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 8
  for (int t = 0; t < DW_KMAX / 8; ++t) {                    // k = kp, kp + 8, ...: the summation order of the first version
    const int k = kp + 8 * t;
    const float a = As[k * DW_LD + m];
    const float4 b = *reinterpret_cast<const float4*>(Bs + 4 * k);
    acc[0] = fmaf(a, b.x, acc[0]); acc[1] = fmaf(a, b.y, acc[1]); acc[2] = fmaf(a, b.z, acc[2]); acc[3] = fmaf(a, b.w, acc[3]);
  }
  __syncthreads();                                            // everybody is done with the staged operands
  float* red = As;
#pragma unroll
  for (int j = 0; j < 4; ++j) red[(kp * 32 + m) * 4 + j] = acc[j];
  __syncthreads();
  if (tid < 32 * 4) {
    const int mm = tid >> 2, j = tid & 3;
    float* c[1] = {P.C + (int64_t)(m0 + mm) * P.ldc + j};
    const bool ok[1] = {m0 + mm < P.M && j < P.N};
    float v[1] = {0.f}, th[1];
    if (ok[0]) {
#pragma unroll
      for (int q = 0; q < 8; ++q) v[0] += red[(q * 32 + mm) * 4 + j];
    }
    dw_finish<1>(T, cx, c, ok, P.accumulate != 0, v, th);
  }
}

// C[n] = sum_k B[k][n] for the 32 columns n0.. : 8 k-parts per column, the 32 loads of a thread in flight at once (the
// first version - one thread per column walking K in steps of 4 - was a chain of 64 dependent round trips: 15 k cycles)
constexpr int DW_CS_COLS = 32;
__device__ __forceinline__ void dw_tile_colsum(const GemmProb& P, float* red, int n0, const DwTail& T, const DwCtx& cx) {
  const int tid = threadIdx.x, nn = tid & 31, kp = tid >> 5;
  const int n = n0 + nn;
  float x[DW_KMAX / 8];
#pragma unroll
  for (int t = 0; t < DW_KMAX / 8; ++t) {
    const int k = kp * (DW_KMAX / 8) + t;
    x[t] = (n < P.N && k < P.K) ? __ldg(P.B + (int64_t)k * P.ldb + n) : 0.f;
  }
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
  for (int t = 0; t < DW_KMAX / 8; t += 4) { s0 += x[t]; s1 += x[t + 1]; s2 += x[t + 2]; s3 += x[t + 3]; }
  red[kp * 32 + nn] = (s0 + s1) + (s2 + s3);
  __syncthreads();
  if (tid < 32) {
    float* c[1] = {P.C + n};
    const bool ok[1] = {n < P.N};
    float v[1], th[1];
    v[0] = ((red[nn] + red[32 + nn]) + (red[64 + nn] + red[96 + nn])) +
           ((red[128 + nn] + red[160 + nn]) + (red[192 + nn] + red[224 + nn]));
    dw_finish<1>(T, cx, c, ok, P.accumulate != 0, v, th);
  }
}

__global__ void __launch_bounds__(GEMM_THREADS, 3)
rows_dw_kernel(const __grid_constant__ GemmBatch G, const __grid_constant__ DwTail T) {
  extern __shared__ __align__(16) float dw_smem[];
  float* As = dw_smem;
  float* Bs = dw_smem + DW_KMAX * DW_LD;
  __shared__ GemmProb Ps;
  __shared__ DwCtx cx;
  // The launch that completes an update carries one extra CTA without a tile (the last block): it folds the loss partials
  // of the stream kernel and bumps the device step counter once every tile CTA has read it.  (First version: every CTA
  // fenced and took a ticket AFTER its tile and the last one to finish did the fold - ~3 us behind the slowest tile.)
  const unsigned int n_tile_ctas = gridDim.x - (T.last_chunk ? 1u : 0u);
  if (blockIdx.x >= n_tile_ctas) {
    pdl_wait();
    const long long st = T.step_counter ? *T.step_counter : 0;   // value BEFORE this update's bump
    float* lp = As;                                              // the partials travel in parallel (one round trip) ...
    for (int i = threadIdx.x; i < 4 * T.n_clusters; i += GEMM_THREADS) lp[i] = __ldcg(T.loss_part + i);
    __syncthreads();
    if (threadIdx.x == 0) {
      float ssq = 0.f, sq = 0.f, sth = 0.f;                      // ... and are added in the fixed order c = 0, 1, ...
      for (int c = 0; c < T.n_clusters; ++c) {
        ssq += lp[4 * c + 0];
        sq += lp[4 * c + 1];
        sth += lp[4 * c + 2];
      }
      const float inv_n = 1.0f / (float)T.n;
      const long long slot = (T.step_counter && T.ring > 0) ? st % T.ring : 0;
      if (T.q_loss) T.q_loss[slot] = ssq * inv_n;                                                   // ddpg.py:439
      if (T.pi_loss) T.pi_loss[slot] = -sq * inv_n + T.action_l2 * sth / (float)(T.n * T.dimu);     // ddpg.py:440-441
      if (T.tl != nullptr) {
        long long* nx = T.tl + TL_MARKS + 4 * (int)((st + 2) & 7);
        nx[0] = 0x7fffffffffffffffLL; nx[1] = 0; nx[2] = 0x7fffffffffffffffLL; nx[3] = 0;
      }
      // a tile CTA takes its ticket after it has read the step counter: only then may the counter move
      volatile unsigned int* tk = T.ticket;
      while (*tk < n_tile_ctas) { }
      if (T.step_counter) *T.step_counter = st + 1;
      *T.ticket = 0u;
      __threadfence();
    }
    pdl_launch_dependents();
    return;
  }
  long long* tl = nullptr;
  if (T.tl != nullptr && threadIdx.x == 0) {
    if (blockIdx.x == 0) tl = T.tl + 32;
    else if ((int)blockIdx.x == T.tl_skinny_block) tl = T.tl + 40;
    else if (blockIdx.x == n_tile_ctas - 1) tl = T.tl + 48;
  }
  if (tl) tl[0] = clock64();
  if (T.tl != nullptr && threadIdx.x == 0 && blockIdx.x < 512) T.tl[1088 + 2 * blockIdx.x] = (long long)globaltimer_ns();
  if (!T.pdl_late) pdl_launch_dependents();
  pdl_wait();                                                    // activations / deltas of the stream kernel, the step counter
  int pi = 0;
  {
    // the problem of this tile: last p with tile_begin[p] <= blockIdx.x (bisection: a linear walk over the ~30 problems
    // cost the last blocks of the grid - the ones that finish last - ~2 k cycles of dependent constant-bank reads)
    int lo = 0, hi = G.n - 1;
#pragma unroll 1
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if ((int)blockIdx.x >= G.p[mid].tile_begin) lo = mid; else hi = mid - 1;
    }
    pi = lo;
  }
  {
    const int* src = reinterpret_cast<const int*>(&G.p[pi]);
    int* dst = reinterpret_cast<int*>(&Ps);
    for (int i = threadIdx.x; i < (int)(sizeof(GemmProb) / 4); i += GEMM_THREADS) dst[i] = src[i];
  }
  __syncthreads();
  const GemmProb& P = Ps;
  const int tile = blockIdx.x - P.tile_begin;
  const int tm = (P.variant == DW_FULLK) ? tile / P.tiles_n : 0, tn = tile - tm * P.tiles_n;
  // ---- the operands first (one round trip) ...
  if (T.dbg_skip_stage) {                                        // debug: what the launch costs without its operand traffic
  } else if (P.variant == DW_FULLK) dw_stage_fullk(P, As, Bs, tm * GT, tn * GT);
  else if (P.variant == DW_SKINNY) dw_stage_skinny(P, As, Bs, tile * GT);
  // ---- ... and what depends on the device step counter (two dependent round trips of thread 0) while they travel
  long long st = 0;
  if (threadIdx.x == 0) {
    st = T.step_counter ? *T.step_counter : 0;                    // value BEFORE this update's bump
    // several workers per rank (SURVEY 8e: 19-worker-equivalent batches): the device counter counts micro-batches,
    // update u = st / micro, launch j = st % micro of it adds its gradient to the sum of launches 0..j-1
    const long long upd = st / T.micro, mb = st - upd * T.micro;
    if (T.tl != nullptr) tl_mark_min(T.tl + TL_MARKS + 4 * (int)(st & 7) + 2);
    cx.ax = T.ax;
    cx.opt = (T.ax.theta != nullptr && T.last_chunk && mb == T.micro - 1) ? 1 : 0;
    if (cx.opt && T.neg_a_table != nullptr) {
      long long t = upd + 1;                                      // Adam's 1-based step of this update
      cx.ax.neg_a = T.neg_a_table[(t <= T.table_len ? t : (long long)T.table_len) - 1];
    }
    cx.xc_on = (cx.opt && T.xc_on) ? 1 : 0;
    cx.owner = (int)(blockIdx.x % (unsigned)(T.xc_on ? T.xc.world : 1));
    cx.own = (!T.xc_on || T.xc.mode == 0 || cx.owner == T.xc.rank) ? 1 : 0;
    cx.flag = (uint32_t)(upd + 1);
    cx.tl = (cx.xc_on && T.xc.tl != nullptr) ? T.xc.tl + 4 * (int64_t)blockIdx.x : nullptr;
    cx.dbg = tl;
    if (cx.tl) cx.tl[0] = (long long)globaltimer_ns();
    if (T.parity_stride > 0) Ps.C += ((upd + 1) & 1) * T.parity_stride;
    Ps.accumulate = (mb > 0 || T.chunk > 0) ? 1 : 0;
    if (T.last_chunk) atomicAdd(T.ticket, 1u);                    // the step counter has been read (its value is in use above)
  }
  if (tl) tl[1] = clock64();
  // (every tile function starts with a __syncthreads before it reads cx / Ps.C / Ps.accumulate)
  if (P.variant == DW_FULLK) {
    dw_tile_fullk(P, As, Bs, tm * GT, tn * GT, T, cx);
  } else if (P.variant == DW_SKINNY) {
    dw_tile_skinny(P, As, Bs, tile * GT, T, cx);
  } else {
    dw_tile_colsum(P, As, tile * DW_CS_COLS, T, cx);
  }
  if (tl) tl[2] = clock64();
  if (cx.tl && threadIdx.x == 0) cx.tl[3] = (long long)globaltimer_ns();
  if (T.tl != nullptr && threadIdx.x == 0) {
    if (blockIdx.x < 512) T.tl[1089 + 2 * blockIdx.x] = (long long)globaltimer_ns();
    tl_mark_max(T.tl + TL_MARKS + 4 * (int)(st & 7) + 3);
  }
  pdl_launch_dependents();
  if (tl) tl[3] = clock64();
}

// tile plan of the weight-gradient launch; returns the grid size, or -1 if a problem does not fit a tile kind
static int plan_dw_batch(GemmBatch& G) {
  int t = 0;
  for (int i = 0; i < G.n; ++i) {
    GemmProb& P = G.p[i];
    P.tile_begin = t;
    if (P.ones_a) {
      P.variant = DW_COLSUM; P.tiles_n = (P.N + DW_CS_COLS - 1) / DW_CS_COLS;
      t += P.tiles_n;
    } else if (P.N <= 4) {
      P.variant = DW_SKINNY; P.tiles_n = 1;
      t += (P.M + GT - 1) / GT;
    } else {
      if (!(P.a_trans && !P.b_trans && al16(P.A) && al16(P.B) && P.lda % 4 == 0 && P.ldb % 4 == 0 && P.M % 4 == 0 &&
            P.N % 4 == 0 && P.K <= DW_KMAX))
        return -1;
      P.variant = DW_FULLK; P.tiles_n = (P.N + GT - 1) / GT;
      t += ((P.M + GT - 1) / GT) * P.tiles_n;
    }
  }
  G.total_tiles = t;
  return t;
}

// ------------------------------------------------------------------------------------------------
struct RowsWorkspace {
  unsigned int* ticket;
  float* loss_part;
  float *Xp, *Xq;
  float *hp[S_MAXL], *hq[S_MAXL], *hqp[S_MAXL], *dc[S_MAXL], *dp[S_MAXL];   // row-major [n][H]
  float *TQ[S_MAXL], *TP[S_MAXL];                                            // W_l^T [H][H], l = 1..L-1
  float *dQ, *dy;
  int KP, lddy;
  int64_t total;
};

static RowsWorkspace carve_rows(const cur_net_desc& d, int64_t n, float* base) {
  RowsWorkspace w;
  const NetLayout q = net_layout(d, 0);
  const int K0q = q.in_s + q.in_g;
  w.KP = (int)r4(K0q);
  w.lddy = (int)r4(d.dimu);
  const int64_t H = d.hidden;
  int64_t o = 0;
  auto take = [&](int64_t floats) {
    float* ptr = base ? base + o : nullptr;
    o += r4(floats);
    return ptr;
  };
  w.ticket = reinterpret_cast<unsigned int*>(take(4));
  w.loss_part = take((n / S_ROWS) * 4);
  w.Xp = take(n * w.KP);
  w.Xq = take(n * w.KP);
  for (int l = 0; l < d.layers; ++l) {
    w.hp[l] = take(n * H); w.hq[l] = take(n * H); w.hqp[l] = take(n * H);
    w.dc[l] = take(n * H); w.dp[l] = take(n * H);
    w.TQ[l] = (l >= 1) ? take(H * H) : nullptr;
    w.TP[l] = (l >= 1) ? take(H * H) : nullptr;
  }
  w.dQ = take(n);
  w.dy = take(n * w.lddy);
  w.total = o;
  return w;
}

// Batches above 256 rows run the stream kernel in several waves and the weight-gradient launch once per 256-row K chunk.
// Measured against the tensor-core levels schedule (us/update): 512: see profiles/README.md.
constexpr int64_t ROWS_MAX_BATCH = 1024;

static bool rows_supported(const cur_net_desc* d, int64_t n) {
  if (check_desc(d) != CUR_OK) return false;
  // hidden 256, and 64 / 128 for networks run at their true width (pad_hidden='native'; the CTA-pair kernel is 256 only)
  if ((d->hidden != 64 && d->hidden != 128 && d->hidden != S_H) || d->layers < 1 || d->layers > S_MAXL) return false;
  if (d->dimu > S_DU || n <= 0 || (n % S_ROWS) != 0 || n > ROWS_MAX_BATCH) return false;
  const NetLayout q = net_layout(*d, 0), p = net_layout(*d, 1);
  if (q.in_s + q.in_g > S_KIN) return false;        // the transposed first-layer input buffer, not the hidden width
  // operands of the first-layer weight gradients must be 16-byte aligned column blocks of X
  if ((q.in_s % 4) != 0 || (p.in_s % 4) != 0 || (q.in_g % 4) != 0) return false;
  if (d->dimu > 4 && (d->dimu % 4) != 0) return false;
  return true;
}

// the weight-gradient problems of both nets for the batch rows [r0, r0 + rows), in launch order
static void build_dw_batch(GemmBatch& G, const NetLayout& LQ, const NetLayout& LP, const RowsWorkspace& w, int L, int H,
                           float* gQ, float* gP, int64_t r0, int64_t rows, bool keep_transposes) {
  G.n = 0; G.total_tiles = 0;
  auto add = [&](const GemmProb& p) { G.p[G.n++] = p; };
  auto net_grads = [&](const NetLayout& NL, float* gN, const float* X0, float* const* hN, float* const* dN,
                       const float* dOut, int lddo) {
    const float* dO = dOut + r0 * lddo;
    add(bwd_dw(hN[L - 1] + r0 * H, H, H, dO, lddo, NL.out, gN + NL.off_Wout, rows));
    add(bwd_db(dO, lddo, NL.out, gN + NL.off_bout, rows));
    for (int l = L - 1; l >= 1; --l) {
      GemmProb p = bwd_dw(hN[l - 1] + r0 * H, H, H, dN[l] + r0 * H, H, H, gN + NL.off_W[l], rows);
      if (keep_transposes) { p.C2 = (&NL == &LQ) ? w.TQ[l] : w.TP[l]; p.ldc2 = H; }   // transposed copy of the stepped weights
      add(p);
      add(bwd_db(dN[l] + r0 * H, H, H, gN + NL.off_b[l], rows));
    }
    add(bwd_dw(X0 + r0 * w.KP, w.KP, NL.in_s, dN[0] + r0 * H, H, H, gN + NL.off_W0, rows));
    add(bwd_db(dN[0] + r0 * H, H, H, gN + NL.off_b0, rows));
    if (NL.in_g > 0) add(bwd_dw(X0 + r0 * w.KP + NL.in_s, w.KP, NL.in_g, dN[0] + r0 * H, H, H, gN + NL.off_W0g, rows));
  };
  net_grads(LQ, gQ, w.Xq, w.hq, w.dc, w.dQ, 1);
  net_grads(LP, gP, w.Xp, w.hp, w.dp, w.dy, w.lddy);
}

template <int H>
static int launch_stream(cudaLaunchConfig_t& cfg, const StreamParams& P) {
  static bool configured = false;
  if (!configured) {
    CUR_CUDA_TRY(cudaFuncSetAttribute(ddpg_stream_kernel<H>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)S_SMEM_BYTES));
    configured = true;
  }
  CUR_CUDA_TRY(cudaLaunchKernelEx(&cfg, ddpg_stream_kernel<H>, P));
  return CUR_OK;
}

template <int H>
static auto act_kernel(const ActParams*) { return actions_stream_kernel<H>; }
template <int H>
static auto act_kernel(const ActGroupParams*) { return actions_group_kernel<H>; }

template <int H, class PT>
static int launch_actions(unsigned blocks, cudaStream_t s, const PT& P) {
  static bool configured = false;
  const auto kernel = act_kernel<H>(&P);
  if (!configured) {
    CUR_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S_SMEM_BYTES));
    configured = true;
  }
  kernel<<<blocks, S_THREADS, S_SMEM_BYTES, s>>>(P);
  return CUR_OK;
}

// launch configuration; CUR_PDL=1 adds programmatic stream serialisation (measured: batch 256 60.2 us with, 58.3 us
// without - the early-scheduled CTAs of the next kernel do not pay for what they displace - so it is off by default)
static void pdl_config(cudaLaunchConfig_t& cfg, cudaLaunchAttribute* at, unsigned grid, unsigned block, size_t smem,
                       cudaStream_t s, int which = 0 /* 0: stream kernel, 1: weight-gradient launch */) {
  // CUR_PDL: 1 both launches may start early (trigger at the start of the previous kernel), 2 both with the trigger at the
  // END of the previous kernel's CTAs, 3 only the weight-gradient launch, 4 only the stream kernel
  static const char mode = getenv("CUR_PDL") != nullptr ? getenv("CUR_PDL")[0] : '0';
  const bool on = mode == '1' || mode == '2' || (mode == '3' && which == 1) || (mode == '4' && which == 0);
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(grid, 1, 1);
  cfg.blockDim = dim3(block, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = on ? 1 : 0;
  cfg.attrs = at;
  cfg.numAttrs = on ? 1 : 0;
}

}  // namespace cur

using namespace cur;

static long long* g_rows_tl = nullptr;     // debug timeline buffer of cur_ddpg_rows_step (CUR_ROWS_TIMELINE=1)

// debug: after a run with CUR_ROWS_TIMELINE=1 (CUDA graph or not), print where the last updates spent their time on the
// %globaltimer clock: per update the span of the two launches and the gaps between them
extern "C" int cur_rows_timeline_dump(void) {
  CUR_REQUIRE(g_rows_tl != nullptr, "no timeline recorded (set CUR_ROWS_TIMELINE=1 before the first update)");
  CUR_CUDA_TRY(cudaDeviceSynchronize());
  long long m[32];
  CUR_CUDA_TRY(cudaMemcpy(m, g_rows_tl + TL_MARKS, sizeof(m), cudaMemcpyDeviceToHost));
  // order the ring by the stream kernel's start
  int idx[8], n = 0;
  for (int i = 0; i < 8; ++i)
    if (m[4 * i] != 0x7fffffffffffffffLL && m[4 * i + 1] != 0 && m[4 * i + 3] != 0) idx[n++] = i;
  for (int i = 0; i < n; ++i)
    for (int j = i + 1; j < n; ++j)
      if (m[4 * idx[j]] < m[4 * idx[i]]) { int t = idx[i]; idx[i] = idx[j]; idx[j] = t; }
  for (int i = 0; i < n; ++i) {
    const long long* q = m + 4 * idx[i];
    fprintf(stderr, "[update marks] stream %lld ns | gap %lld | dw %lld ns", q[1] - q[0], q[2] - q[1], q[3] - q[2]);
    if (i + 1 < n) fprintf(stderr, " | gap to the next update's stream kernel %lld ns | update period %lld ns",
                           m[4 * idx[i + 1]] - q[3], m[4 * idx[i + 1]] - q[0]);
    fprintf(stderr, "\n");
  }
  return CUR_OK;
}

extern "C" int cur_ddpg_rows_owner_map(const cur_net_desc* d, int64_t batch, int world, int32_t* owner) {
  CUR_TRY(check_desc(d));
  CUR_REQUIRE(owner != nullptr && world >= 1 && world <= CUR_MAX_RANKS, "bad argument");
  CUR_REQUIRE(rows_supported(d, batch), "shape not supported by the rows schedule");
  const NetLayout LQ = net_layout(*d, 0), LP = net_layout(*d, 1);
  const int64_t offP = r4(LQ.total), arena = offP + r4(LP.total);
  // the plan only depends on shapes: build it over a dummy workspace / gradient arena that is never dereferenced
  float* ws = reinterpret_cast<float*>(malloc(16));
  float* grads = reinterpret_cast<float*>(malloc((size_t)arena * 4));
  CUR_REQUIRE(ws && grads, "out of host memory");
  const RowsWorkspace w = carve_rows(*d, batch, ws);
  GemmBatch G;
  const int64_t rows = batch < DW_KMAX ? batch : DW_KMAX;
  build_dw_batch(G, LQ, LP, w, d->layers, d->hidden, grads, grads + offP, 0, rows, false);
  const int tiles = plan_dw_batch(G);
  if (tiles <= 0) { free(ws); free(grads); return invalid("weight-gradient problems do not fit the rows schedule"); }
  for (int64_t i = 0; i < arena; ++i) owner[i] = -1;
  for (int pi = 0; pi < G.n; ++pi) {
    const GemmProb& P = G.p[pi];
    const int64_t base = P.C - grads;
    const int n_tiles = (pi + 1 < G.n ? G.p[pi + 1].tile_begin : tiles) - P.tile_begin;
    for (int t = 0; t < n_tiles; ++t) {
      const int own = (P.tile_begin + t) % world;
      if (P.variant == DW_FULLK) {
        const int tm = t / P.tiles_n, tn = t - tm * P.tiles_n;
        for (int m = tm * GT; m < (tm + 1) * GT && m < P.M; ++m)
          for (int n = tn * GT; n < (tn + 1) * GT && n < P.N; ++n) owner[base + (int64_t)m * P.ldc + n] = own;
      } else if (P.variant == DW_SKINNY) {
        for (int m = t * GT; m < (t + 1) * GT && m < P.M; ++m)
          for (int n = 0; n < P.N; ++n) owner[base + (int64_t)m * P.ldc + n] = own;
      } else {
        for (int n = t * DW_CS_COLS; n < (t + 1) * DW_CS_COLS && n < P.N; ++n) owner[base + n] = own;
      }
    }
  }
  free(ws); free(grads);
  return CUR_OK;
}

extern "C" int cur_ddpg_rows_supported(const cur_net_desc* d, int64_t batch) { return rows_supported(d, batch) ? 1 : 0; }

extern "C" int64_t cur_ddpg_rows_workspace_floats(const cur_net_desc* d, int64_t batch) {
  if (!rows_supported(d, batch)) return -1;
  return carve_rows(*d, batch, nullptr).total;
}

extern "C" int cur_ddpg_rows_step(void* stream, const cur_net_desc* d, float* theta_main, const float* theta_target,
                                  const cur_norm_stats* stats, const cur_batch* batch, const cur_ddpg_hyper* h,
                                  float* workspace, float* grads, float* q_loss, float* pi_loss, float* q_pi,
                                  const cur_adam_fused* adam, const cur_her_args* her) {
  CUR_TRY(check_desc(d));
  CUR_REQUIRE(theta_main && theta_target && batch && h && workspace && grads && q_pi, "NULL argument");
  if (her == nullptr) {
    CUR_REQUIRE(batch->o && batch->g && batch->u && batch->o_2 && batch->g_2 && batch->r, "NULL batch array");
    CUR_REQUIRE(!d->modular || batch->td, "task_descr required for a modular net");
  }
  CUR_REQUIRE(rows_supported(d, batch->n), "shape not supported by the rows schedule (see cur_ddpg_rows_supported)");
  if (d->normalize_obs)
    CUR_REQUIRE(stats && stats->o_mean && stats->o_std && stats->g_mean && stats->g_std, "normalizer stats required");
  if (adam) {
    CUR_REQUIRE(adam->m && adam->v && adam->neg_a_table && adam->table_len > 0, "incomplete Adam block");
    CUR_REQUIRE(h->step_counter != nullptr, "fused Adam needs the device step counter");
  }
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t n = batch->n;
  const NetLayout LQ = net_layout(*d, 0), LP = net_layout(*d, 1);
  const int64_t offP = r4(LQ.total);
  const float *mQ = theta_main, *mP = theta_main + offP, *tQ = theta_target, *tP = theta_target + offP;
  float *gQ = grads, *gP = grads + offP;
  const RowsWorkspace w = carve_rows(*d, n, workspace);
  const int L = d->layers, H = d->hidden;

  // ---- launch 0: W_l^T of the hidden layers of main.Q and main.pi.  With the fused optimiser the weight-gradient
  // epilogue of the previous call already left the transposes of the stepped weights in the workspace; the caller says
  // so with adam->transposes_valid (and refreshes them with cur_ddpg_rows_refresh after any other change of theta).
  const bool keep_wT = adam != nullptr ? adam->transposes_valid != 0 : h->transposes_valid != 0;
  if (L > 1 && !keep_wT) {
    TransposeParams TP;
    memset(&TP, 0, sizeof(TP));
    int m = 0;
    for (int l = 1; l < L; ++l) {
      TP.src[m] = mQ + LQ.off_W[l]; TP.dst[m++] = w.TQ[l];
      TP.src[m] = mP + LP.off_W[l]; TP.dst[m++] = w.TP[l];
    }
    launch_transposes(TP, m, H, s);
    CUR_CHECK_LAUNCH();
  }

  StreamParams P;
  memset(&P, 0, sizeof(P));
  P.d = *d;
  P.in_sp = LP.in_s; P.in_sq = LQ.in_s; P.in_g = LQ.in_g; P.KP = w.KP; P.L = L;
  P.n = n;
  P.grad_rows = h->loss_rows > 0 ? h->loss_rows : n;
  P.o = batch->o; P.g = batch->g; P.u = batch->u; P.td = batch->td; P.o_2 = batch->o_2; P.g_2 = batch->g_2;
  P.r = batch->r;
  if (stats) { P.o_mean = stats->o_mean; P.o_std = stats->o_std; P.g_mean = stats->g_mean; P.g_std = stats->g_std; }
  P.gamma = h->gamma; P.clip_return = h->clip_return; P.action_l2 = h->action_l2; P.clip_pos = h->clip_pos_returns;
  for (int l = 0; l < L; ++l) {
    const int64_t bq = (l == 0) ? LQ.off_b0 : LQ.off_b[l], bp = (l == 0) ? LP.off_b0 : LP.off_b[l];
    P.bP[l] = mP + bp; P.bPT[l] = tP + bp; P.bQ[l] = mQ + bq; P.bQT[l] = tQ + bq;
    P.hp[l] = w.hp[l]; P.hq[l] = w.hq[l]; P.hqp[l] = w.hqp[l]; P.dc[l] = w.dc[l]; P.dp[l] = w.dp[l];
  }
  P.WoutP = mP + LP.off_Wout; P.boutP = mP + LP.off_bout; P.WoutPT = tP + LP.off_Wout; P.boutPT = tP + LP.off_bout;
  P.WoutQ = mQ + LQ.off_Wout; P.boutQ = mQ + LQ.off_bout; P.WoutQT = tQ + LQ.off_Wout; P.boutQT = tQ + LQ.off_bout;
  P.W0Q_act = mQ + LQ.off_W0 + (int64_t)LP.in_s * H;
  P.Xp = w.Xp; P.Xq = w.Xq; P.dQ = w.dQ; P.dy = w.dy; P.lddy = w.lddy;
  P.loss_part = w.loss_part; P.q_pi = q_pi;
  if (her != nullptr) {
    // fused sampling: the rows of the batch are drawn, gathered and relabelled in the kernel's prologue
    CUR_REQUIRE(her->batch == n, "HER args must describe exactly this batch");
    CUR_REQUIRE(her->L.dimo == d->dimo && her->L.dimg == d->dimg && her->L.dimu == d->dimu &&
                her->L.dimtd == (d->modular ? d->dimtd : her->L.dimtd), "HER layout does not match the networks");
    CUR_REQUIRE(!her->relative_goals || her->L.dimag == her->L.dimg, "relative goals need dimg == dimag");
    P.her = *her;
    P.her.change = nullptr; P.her.info = nullptr;         // cold rows travel only for an INFO reward (make_plan)
    P.her.ag = nullptr;                                    // (ag_t is staged iff relative_goals)
    make_plan(P.her, &P.plan);
    CUR_REQUIRE(S_ROWS * P.plan.stage_stride <= S_MISC - S_STAGE_OFF, "transition too wide for the fused HER stage");
    if (P.plan.cold4 > 0)
      for (int i = 0; i < her->n_segments; ++i)
        CUR_REQUIRE(her->seg[i].cold != nullptr, "an INFO reward needs the cold rows of every segment");
    P.fused_her = 1;
  }

  // ---- weight chunks in consumption order
  int nc = 0;
  SChunk* list = P.chunks;
  const int CK = chunk_rows(H);
  auto rows_of = [&](const float* src, int nrows, int k0) {      // a row block as chunks of <= CK rows
    for (int r = 0; r < nrows; r += CK) {
      SChunk& C = list[nc++];
      C.src = src + (int64_t)r * H; C.nrows = (nrows - r < CK) ? nrows - r : CK; C.k0 = k0 + r;
    }
  };
  auto forward_net = [&](const float* th, const NetLayout& NL) {
    const int before = nc;
    rows_of(th + NL.off_W0, NL.in_s, 0);
    if (NL.in_g > 0) rows_of(th + NL.off_W0g, NL.in_g, NL.in_s);
    const int first = nc - before;
    for (int l = 1; l < L; ++l) rows_of(th + NL.off_W[l], H, 0);
    return first;
  };
  P.ch0[0] = forward_net(mP, LP);
  P.ch0[1] = forward_net(mQ, LQ);
  for (int l = L - 1; l >= 1; --l) rows_of(w.TQ[l], H, 0);
  for (int l = L - 1; l >= 1; --l) rows_of(w.TP[l], H, 0);
  CUR_REQUIRE(nc <= S_MAXCHUNK, "too many weight chunks for the rows schedule");
  P.nchunks = nc;
  nc = 0;
  list = P.chunks_t;
  forward_net(tP, LP);
  forward_net(tQ, LQ);
  forward_net(mQ, LQ);                                            // critic CTA: main.Q(o,g,u) ...
  for (int l = L - 1; l >= 1; --l) rows_of(w.TQ[l], H, 0);        // ... and its backward chain
  CUR_REQUIRE(nc <= S_MAXCHUNK_T, "too many weight chunks for the rows schedule");
  P.nchunks_t = nc;

  long long*& tl_dev = g_rows_tl;
  static int tl_calls = 0;
  const bool tl_on = getenv("CUR_ROWS_TIMELINE") != nullptr;
  if (tl_on && tl_dev == nullptr) {
    CUR_CUDA_TRY(cudaMalloc(&tl_dev, (TL_MARKS + 32) * sizeof(long long)));
    CUR_CUDA_TRY(cudaMemset(tl_dev, 0, (TL_MARKS + 32) * sizeof(long long)));
    long long init[32];
    for (int i = 0; i < 32; ++i) init[i] = (i & 1) ? 0 : 0x7fffffffffffffffLL;
    CUR_CUDA_TRY(cudaMemcpy(tl_dev + TL_MARKS, init, sizeof(init), cudaMemcpyHostToDevice));
  }
  P.tl = tl_on ? tl_dev : nullptr;
  P.tl_step = h->step_counter;
  P.dbg_skip_math = getenv("CUR_ROWS_SKIP_MATH") != nullptr;
  static const int pdl_late = (getenv("CUR_PDL") != nullptr && getenv("CUR_PDL")[0] == '2') ? 1 : 0;
  P.pdl_late = pdl_late;

  const unsigned int n_ctas = (unsigned int)(n / S_ROWS);
  // CTA-pair form (column split over a 2-CTA cluster, 8 rows per pair): half the weight bytes per SM
  static const int pair_mode = getenv("CUR_ROWS_PAIR") ? atoi(getenv("CUR_ROWS_PAIR")) : 0;   // measured slower, see profiles/README.md
  const bool use_pair = pair_mode != 0 && H == S_H && (n % PR_ROWS) == 0 && d->dimu <= 4 &&
                        (her == nullptr || PR_ROWS * P.plan.stage_stride <= PR_MISC - PR_STAGE_OFF);
  if (use_pair) {
    static bool pair_configured = false;
    if (!pair_configured) {
      CUR_CUDA_TRY(cudaFuncSetAttribute(ddpg_stream_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)PR_SMEM_BYTES));
      pair_configured = true;
    }
    static thread_local PairParams PP;                       // ~20 KB: kept off the stack; rebuilt on every call
    PP.S = P;
    // one tensor map per weight block (encoded once per address: the arenas and the workspace do not move)
    struct MapKey { const float* ptr; int rows; };
    static thread_local MapKey cache_key[256];
    static thread_local CUtensorMap cache_map[256];
    static thread_local int cache_n = 0;
    int n_maps = 0;
    MapKey used[PR_MAXMAPS];
    auto map_of = [&](const float* ptr, int rows, int* out) -> int {
      for (int i = 0; i < n_maps; ++i)
        if (used[i].ptr == ptr && used[i].rows == rows) { *out = i; return CUR_OK; }
      CUR_REQUIRE(n_maps < PR_MAXMAPS, "too many weight blocks for the CTA-pair rows schedule");
      int hit = -1;
      for (int i = 0; i < cache_n; ++i)
        if (cache_key[i].ptr == ptr && cache_key[i].rows == rows) { hit = i; break; }
      if (hit < 0) {
        hit = cache_n < 256 ? cache_n++ : 0;
        CUR_TRY(tc_make_plain_map(&cache_map[hit], ptr, rows, H, H, PR_NC, PR_CK));
        cache_key[hit].ptr = ptr; cache_key[hit].rows = rows;
      }
      PP.maps[n_maps] = cache_map[hit];
      used[n_maps].ptr = ptr; used[n_maps].rows = rows;
      *out = n_maps++;
      return CUR_OK;
    };
    for (int rank = 0; rank < 2; ++rank) {
      int m = 0;
      PairChunk* pl = nullptr;
      // a row block [nrows][256] as chunks of <= 64 rows of this rank's 128 columns; `exchanged`: the k rows are the
      // columns of the previous layer's output, so the rank's own half comes first and the partner's half waits
      auto rows_of = [&](const float* src, int nrows, int k0, bool exchanged) -> int {
        int mi = 0;
        CUR_TRY(map_of(src, nrows, &mi));
        if (!exchanged) {
          for (int r = 0; r < nrows; r += PR_CK) {
            CUR_REQUIRE(m < PR_MAXCHUNK, "too many weight chunks for the CTA-pair rows schedule");
            PairChunk& C = pl[m++];
            C.map = mi; C.krow = r; C.nrows = (short)((nrows - r < PR_CK) ? nrows - r : PR_CK); C.wait = 0; C.k0 = k0 + r;
          }
          return CUR_OK;
        }
        for (int half = 0; half < 2; ++half) {
          const int hk = (half == 0 ? rank : 1 - rank) * PR_NC;          // first k row of this half
          for (int r = 0; r < PR_NC; r += PR_CK) {
            CUR_REQUIRE(m < PR_MAXCHUNK, "too many weight chunks for the CTA-pair rows schedule");
            PairChunk& C = pl[m++];
            C.map = mi; C.krow = hk + r; C.nrows = PR_CK; C.wait = (short)((half == 1 && r == 0) ? 1 : 0); C.k0 = k0 + hk + r;
          }
        }
        return CUR_OK;
      };
      auto forward_net = [&](const float* th, const NetLayout& NL, int* first) -> int {
        const int before = m;
        CUR_TRY(rows_of(th + NL.off_W0, NL.in_s, 0, false));
        if (NL.in_g > 0) CUR_TRY(rows_of(th + NL.off_W0g, NL.in_g, NL.in_s, false));
        if (first) *first = m - before;
        for (int l = 1; l < L; ++l) CUR_TRY(rows_of(th + NL.off_W[l], H, 0, true));
        return CUR_OK;
      };
      pl = PP.ch[0][rank]; m = 0;
      CUR_TRY(forward_net(mP, LP, &PP.pch0[0]));
      CUR_TRY(forward_net(mQ, LQ, &PP.pch0[1]));
      for (int l = L - 1; l >= 1; --l) CUR_TRY(rows_of(w.TQ[l], H, 0, true));
      for (int l = L - 1; l >= 1; --l) CUR_TRY(rows_of(w.TP[l], H, 0, true));
      PP.nch[0][rank] = m;
      pl = PP.ch[1][rank]; m = 0;
      CUR_TRY(forward_net(tP, LP, nullptr));
      CUR_TRY(forward_net(tQ, LQ, nullptr));
      CUR_TRY(forward_net(mQ, LQ, nullptr));                                      // critic pair: main.Q(o,g,u) ...
      for (int l = L - 1; l >= 1; --l) CUR_TRY(rows_of(w.TQ[l], H, 0, true));     // ... and its backward chain
      PP.nch[1][rank] = m;
    }
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute at[1];
    pdl_config(cfg, at, (unsigned)(n / PR_ROWS) * 4u, S_THREADS, PR_SMEM_BYTES, s);   // (actor, critic) x (rank 0, rank 1)
    CUR_CUDA_TRY(cudaLaunchKernelEx(&cfg, ddpg_stream_pair_kernel, PP));
  } else {
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute at[1];
    pdl_config(cfg, at, 2 * n_ctas, S_THREADS, S_SMEM_BYTES, s);
    if (H == 64) CUR_TRY(launch_stream<64>(cfg, P));                     // (actor, critic) CTA pairs
    else if (H == 128) CUR_TRY(launch_stream<128>(cfg, P));
    else CUR_TRY(launch_stream<256>(cfg, P));
  }
  CUR_CHECK_LAUNCH();
  if (tl_on && ++tl_calls == 40) {          // debug only: one warmed-up timeline of CTA 0
    long long t[64];
    CUR_CUDA_TRY(cudaStreamSynchronize(s));
    CUR_CUDA_TRY(cudaMemcpy(t, tl_dev, sizeof(t), cudaMemcpyDeviceToHost));
    fprintf(stderr, "[rows timeline] build %lld | main.pi %lld | main.Q x2 %lld | wait target.Q %lld | "
                    "loss+bwd Q %lld | bwd pi %lld | total %lld cycles\n",
            t[1] - t[0], t[2] - t[1], t[4] - t[3], t[5] - t[4], t[6] - t[5], t[7] - t[6], t[7] - t[0]);
    if (use_pair) {
      fprintf(stderr, "[pair main.pi stamps, cycles after build]");
      for (int i = 8; i < 32 && t[i] != 0; ++i) fprintf(stderr, " %lld", t[i] - t[1]);
      fprintf(stderr, "\n");
    }
  }

  // ---- launch 2: weight gradients, one launch per 256-row chunk of the batch (K of the tiles)
  DwTail T;
  memset(&T, 0, sizeof(T));
  if (adam) {
    T.ax.grads = grads; T.ax.theta = theta_main; T.ax.m = adam->m; T.ax.v = adam->v;
    T.ax.b1 = (float)adam->beta1; T.ax.omb1 = (float)(1.0 - adam->beta1);
    T.ax.b2 = (float)adam->beta2; T.ax.omb2 = (float)(1.0 - adam->beta2);
    T.ax.eps = (float)adam->eps;
    T.neg_a_table = adam->neg_a_table; T.table_len = adam->table_len;
  }
  T.step_counter = h->step_counter; T.ring = h->loss_ring;
  T.ticket = w.ticket; T.loss_part = w.loss_part; T.n_clusters = (int)n_ctas; T.n = n; T.dimu = d->dimu;
  T.action_l2 = h->action_l2; T.q_loss = q_loss; T.pi_loss = pi_loss;
  T.parity_stride = h->grads_parity_stride;
  T.micro = h->micro_batches > 1 ? h->micro_batches : 1;
  CUR_REQUIRE(T.micro == 1 || h->step_counter != nullptr, "several micro-batches per update need the step counter");
  CUR_REQUIRE(T.parity_stride == 0 || (h->step_counter != nullptr && adam == nullptr),
              "gradient double buffering needs the step counter and excludes the fused Adam epilogue");
  static bool dw_configured = false;
  static int dw_resident = 0;              // CTAs of the weight-gradient launch that are co-resident on the device
  if (!dw_configured) {
    CUR_CUDA_TRY(cudaFuncSetAttribute(rows_dw_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)DW_SMEM_BYTES));
    int per_sm = 0;
    CUR_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, rows_dw_kernel, GEMM_THREADS, DW_SMEM_BYTES));
    dw_resident = per_sm * sm_count();
    dw_configured = true;
  }
  if (adam != nullptr && adam->xchg != nullptr && adam->xchg->world > 1) {
    const cur_xchg_ctx* x = adam->xchg;
    CUR_REQUIRE(x->world <= CUR_MAX_RANKS && x->rank >= 0 && x->rank < x->world, "bad rank / world of the exchange");
    CUR_REQUIRE(x->mode >= 0 && x->mode <= 2, "bad exchange mode");
    CUR_REQUIRE(x->mode != 2 || x->mc_region != nullptr, "exchange mode 2 needs the multicast mapping of the regions");
    CUR_REQUIRE(x->arena >= r4(LQ.total) + r4(LP.total), "exchange arena smaller than the gradient arena");
    T.xc_on = 1;
    T.xc.rank = x->rank; T.xc.world = x->world; T.xc.mode = x->mode; T.xc.arena = x->arena;
    T.xc.tl = reinterpret_cast<long long*>(x->timeline); T.xc.error_flag = x->error_flag;
    for (int r = 0; r < x->world; ++r) {
      CUR_REQUIRE(x->region[r] != nullptr, "peer region not mapped");
      T.xc.part[r] = reinterpret_cast<unsigned long long*>(x->region[r]);
      T.xc.res[r] = T.xc.part[r] + (int64_t)(x->mode == 2 ? 1 : x->world) * x->arena;
    }
    T.xc.part_mc = reinterpret_cast<const float2*>(x->mc_region);
    T.xc.res_mc = x->mc_region ? reinterpret_cast<unsigned long long*>(x->mc_region) + x->arena : nullptr;
  }
  T.tl = tl_on ? tl_dev : nullptr;
  T.pdl_late = pdl_late;
  T.dbg_skip_stage = getenv("CUR_DW_SKIP_STAGE") != nullptr;
  const AdamCtx ax_full = T.ax;
  const int n_chunks = (int)((n + DW_KMAX - 1) / DW_KMAX);
  for (int c = 0; c < n_chunks; ++c) {
    const int64_t r0 = (int64_t)c * DW_KMAX;
    const int64_t rows = (n - r0 < DW_KMAX) ? n - r0 : DW_KMAX;
    const bool last = c == n_chunks - 1;
    GemmBatch G;
    build_dw_batch(G, LQ, LP, w, L, H, gQ, gP, r0, rows, adam != nullptr && last);
    const int tiles = plan_dw_batch(G);
    CUR_REQUIRE(tiles > 0, "weight-gradient problems do not fit the rows schedule (unaligned dims)");
    // CTAs of the exchange spin on their peers: every tile of the launch must be resident at once
    CUR_REQUIRE(!T.xc_on || tiles + 1 <= dw_resident, "too many weight-gradient tiles for the in-launch gradient exchange");
    T.chunk = c; T.last_chunk = last ? 1 : 0;
    T.ax = ax_full;
    if (!last) T.ax.theta = nullptr;             // the optimiser runs once, on the complete sum
    T.tl_skinny_block = 0;
    for (int i = 0; i < G.n; ++i)
      if (G.p[i].variant == DW_FULLK) { T.tl_skinny_block = G.p[i].tile_begin; break; }
    {
      cudaLaunchConfig_t cfg;
      cudaLaunchAttribute at[1];
      pdl_config(cfg, at, (unsigned)tiles + (last ? 1u : 0u), GEMM_THREADS, DW_SMEM_BYTES, s, 1);   // + the bookkeeping CTA
      CUR_CUDA_TRY(cudaLaunchKernelEx(&cfg, rows_dw_kernel, G, T));
    }
    CUR_CHECK_LAUNCH();
  }
  if (tl_on && tl_calls == 40) {
    long long t[64];
    CUR_CUDA_TRY(cudaStreamSynchronize(s));
    CUR_CUDA_TRY(cudaMemcpy(t, tl_dev, sizeof(t), cudaMemcpyDeviceToHost));
    {
      // wall-clock spans (%globaltimer, ns) of every CTA of the two launches of this update
      static long long sp[2048];
      CUR_CUDA_TRY(cudaMemcpy(sp, tl_dev + 64, sizeof(sp), cudaMemcpyDeviceToHost));
      for (int k = 0; k < 2; ++k) {
        long long s0 = 0, e1 = 0, dmin = 1LL << 60, dmax = 0, dsum = 0; int cnt = 0;
        for (int b = 0; b < 512; ++b) {
          const long long a = sp[1024 * k + 2 * b], e = sp[1024 * k + 2 * b + 1];
          if (a == 0 || e == 0) continue;
          if (cnt == 0 || a < s0) s0 = a;
          if (e > e1) e1 = e;
          const long long dd = e - a;
          dmin = dd < dmin ? dd : dmin; dmax = dd > dmax ? dd : dmax; dsum += dd; ++cnt;
        }
        if (cnt) fprintf(stderr, "[spans] %s: %d CTAs, CTA span min %lld / mean %lld / max %lld ns, first start -> last end %lld ns%s",
                         k == 0 ? "stream kernel" : "dw kernel", cnt, dmin, dsum / cnt, dmax, e1 - s0, k == 0 ? "" : "\n");
        if (k == 0) { fprintf(stderr, ", "); sp[2047] = e1; } else fprintf(stderr, "[spans] stream last end -> dw first start %lld ns\n", s0 - sp[2047]);
      }
    }
    for (int b = 0; b < 3; ++b) {
      const long long* q = t + 32 + 8 * b;
      fprintf(stderr, "[dw timeline] %s: prologue %lld | tile %lld | tail %lld | total %lld cycles (start +%lld after block 0)\n",
              b == 0 ? "block 0 (output-layer tile)" : b == 1 ? "first full-K tile" : "last block", q[1] - q[0], q[2] - q[1],
              q[3] - q[2], q[3] - q[0], q[0] - t[32]);
      if (b > 0) fprintf(stderr, "              operands landed +%lld | math done +%lld | partials summed +%lld | finish (Adam) done +%lld | end +%lld\n",
                         q[4] - q[0], q[5] - q[0], q[6] - q[0], q[7] - q[0], q[2] - q[0]);
    }
  }
  CUR_CHECK_LAUNCH();
  return CUR_OK;
}

extern "C" int cur_ddpg_rows_refresh(void* stream, const cur_net_desc* d, const float* theta_main, float* workspace,
                                     int64_t batch) {
  CUR_TRY(check_desc(d));
  CUR_REQUIRE(theta_main && workspace, "NULL argument");
  CUR_REQUIRE(rows_supported(d, batch), "shape not supported by the rows schedule");
  const NetLayout LQ = net_layout(*d, 0), LP = net_layout(*d, 1);
  const float *mQ = theta_main, *mP = theta_main + r4(LQ.total);
  const RowsWorkspace w = carve_rows(*d, batch, workspace);
  const int L = d->layers, H = d->hidden;
  if (L <= 1) return CUR_OK;
  TransposeParams TP;
  memset(&TP, 0, sizeof(TP));
  int m = 0;
  for (int l = 1; l < L; ++l) {
    TP.src[m] = mQ + LQ.off_W[l]; TP.dst[m++] = w.TQ[l];
    TP.src[m] = mP + LP.off_W[l]; TP.dst[m++] = w.TP[l];
  }
  launch_transposes(TP, m, H, (cudaStream_t)stream);
  CUR_CHECK_LAUNCH();
  return CUR_OK;
}

extern "C" int cur_ddpg_rows_transposes(const cur_net_desc* d, float* workspace, int64_t batch, cur_p2p_transposes* out) {
  CUR_TRY(check_desc(d));
  CUR_REQUIRE(workspace && out, "NULL argument");
  CUR_REQUIRE(rows_supported(d, batch), "shape not supported by the rows schedule");
  const NetLayout LQ = net_layout(*d, 0), LP = net_layout(*d, 1);
  const int64_t offP = r4(LQ.total);
  const RowsWorkspace w = carve_rows(*d, batch, workspace);
  memset(out, 0, sizeof(*out));
  out->H = d->hidden;
  for (int l = 1; l < d->layers; ++l) {
    CUR_REQUIRE(out->n + 2 <= CUR_P2P_MAX_TRANSPOSES, "too many hidden layers for the transposes table");
    out->begin[out->n] = LQ.off_W[l]; out->dst[out->n++] = w.TQ[l];
    out->begin[out->n] = offP + LP.off_W[l]; out->dst[out->n++] = w.TP[l];
  }
  return CUR_OK;
}


// bias and output-layer pointers of the forward nets of `theta` (ActParams, ActExpert)
template <class T>
static void act_net_ptrs(T& P, const cur_net_desc& d, const float* theta) {
  const NetLayout LQ = net_layout(d, 0), LP = net_layout(d, 1);
  const float *thQ = theta, *thP = theta + r4(LQ.total);
  for (int l = 0; l < S_MAXL; ++l) {
    P.bP[l] = l < d.layers ? thP + ((l == 0) ? LP.off_b0 : LP.off_b[l]) : nullptr;
    P.bQ[l] = l < d.layers ? thQ + ((l == 0) ? LQ.off_b0 : LQ.off_b[l]) : nullptr;
  }
  P.WoutP = thP + LP.off_Wout; P.boutP = thP + LP.off_bout;
  P.WoutQ = thQ + LQ.off_Wout; P.boutQ = thQ + LQ.off_bout;
}

// What ActParams and ActGroupParams share: the shape, the inputs, the outputs and the weight chunks of `theta`
template <class PT>
static int act_common(PT& P, const cur_net_desc* d, const float* theta, const float* o, const float* ag, const float* g,
                      const float* td, float clip_obs, void* out_pi, void* out_q, uint32_t seq) {
  const NetLayout LQ = net_layout(*d, 0), LP = net_layout(*d, 1);
  const float *thQ = theta, *thP = theta + r4(LQ.total);
  const int L = d->layers, H = d->hidden;
  P.d = *d;
  P.in_sp = LP.in_s; P.in_g = LQ.in_g; P.L = L;
  P.KP = (LQ.in_s + LQ.in_g + 3) / 4 * 4;
  P.dbg_skip_math = 0;
  P.o = o; P.g = g; P.td = td; P.ag = ag; P.clip = clip_obs; P.seq = seq;
  P.pi = out_pi; P.q = out_q;
  int nc = 0;
  const int CK = chunk_rows(H);
  auto rows_of = [&](const float* src, int nrows, int k0) {
    for (int r = 0; r < nrows; r += CK) {
      SChunk& C = P.chunks[nc++];
      C.src = src + (int64_t)r * H; C.nrows = (nrows - r < CK) ? nrows - r : CK; C.k0 = k0 + r;
    }
  };
  auto forward_net = [&](const float* th, const NetLayout& NL) {
    const int before = nc;
    rows_of(th + NL.off_W0, NL.in_s, 0);
    if (NL.in_g > 0) rows_of(th + NL.off_W0g, NL.in_g, NL.in_s);
    const int first = nc - before;
    for (int l = 1; l < L; ++l) rows_of(th + NL.off_W[l], H, 0);
    return first;
  };
  CUR_REQUIRE((out_q ? 2 : 1) * (4 + (L - 1) * (H / CK)) <= A_MAXCHUNK, "too many weight chunks");
  P.ch0[0] = forward_net(thP, LP);
  P.ch0[1] = out_q != nullptr ? forward_net(thQ, LQ) : 0;
  P.nchunks = nc;
  return CUR_OK;
}

// One launch for DDPG.get_actions (see actions_stream_kernel).  o / ag / g / td / out_pi / out_q may be device
// pointers of mapped pinned host memory.  seq != 0: the outputs are 8-byte words {float32 bits | seq << 32}.
extern "C" int cur_ddpg_actions_rows(void* stream, const cur_net_desc* d, const float* theta, const cur_norm_stats* stats,
                                     const float* o, const float* ag, const float* g, const float* td, int64_t n,
                                     float clip_obs, void* out_pi, void* out_q, uint32_t seq) {
  CUR_TRY(check_desc(d));
  CUR_REQUIRE(theta && o && g && out_pi, "NULL argument");
  CUR_REQUIRE(!d->modular || td, "task_descr required for a modular net");
  CUR_REQUIRE(n > 0 && n <= 4096, "bad row count (the one-launch action path covers up to 4096 rows)");
  CUR_REQUIRE(rows_supported(d, S_ROWS), "shape not supported by the rows schedule (see cur_ddpg_rows_supported)");
  if (d->normalize_obs)
    CUR_REQUIRE(stats && stats->o_mean && stats->o_std && stats->g_mean && stats->g_std, "normalizer stats required");
  const int H = d->hidden;
  static const bool tl_on = getenv("CUR_ACTIONS_TIMELINE") != nullptr;
  ActParams P;
  CUR_TRY(act_common(P, d, theta, o, ag, g, td, clip_obs, out_pi, out_q, seq));
  P.n = n;
  P.o_mean = P.o_std = P.g_mean = P.g_std = nullptr;
  if (stats) { P.o_mean = stats->o_mean; P.o_std = stats->o_std; P.g_mean = stats->g_mean; P.g_std = stats->g_std; }
  act_net_ptrs(P, *d, theta);
  static long long* tl_dev = nullptr;
  static int tl_calls = 0;
  if (tl_on && tl_dev == nullptr) {
    CUR_CUDA_TRY(cudaMalloc(&tl_dev, 8 * sizeof(long long)));
    CUR_CUDA_TRY(cudaMemset(tl_dev, 0, 8 * sizeof(long long)));
  }
  P.tl = tl_on ? tl_dev : nullptr;
  const unsigned blocks = (unsigned)((n + S_ROWS - 1) / S_ROWS);
  if (H == 64) CUR_TRY(launch_actions<64>(blocks, (cudaStream_t)stream, P));
  else if (H == 128) CUR_TRY(launch_actions<128>(blocks, (cudaStream_t)stream, P));
  else CUR_TRY(launch_actions<256>(blocks, (cudaStream_t)stream, P));
  CUR_CHECK_LAUNCH();
  if (tl_on && ++tl_calls == 100) {          // debug only: one warmed-up timeline of CTA 0 (%globaltimer, ns)
    long long t[8];
    CUR_CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    CUR_CUDA_TRY(cudaMemcpy(t, tl_dev, sizeof(t), cudaMemcpyDeviceToHost));
    fprintf(stderr, "[actions timeline] inputs %lld | pi forward %lld | outputs (+ Q) %lld | total %lld ns\n", t[1] - t[0],
            t[2] - t[1], t[3] - t[2], t[3] - t[0]);
  }
  return CUR_OK;
}

// The routed form of cur_ddpg_actions_rows (see actions_group_kernel): row i is acted on by experts[row_expert[i]].  The
// rows of each expert fill whole 4-row tiles in their original order; outputs go to the rows' original positions.
extern "C" int cur_ddpg_actions_rows_group(void* stream, const cur_net_desc* d, int n_experts,
                                           const cur_actions_expert* experts, const int32_t* row_expert, const float* o,
                                           const float* ag, const float* g, const float* td, int64_t n, float clip_obs,
                                           void* out_pi, void* out_q, uint32_t seq) {
  CUR_TRY(check_desc(d));
  CUR_REQUIRE(n_experts >= 1 && n_experts <= CUR_MAX_TASKS, "n_experts must be 1..CUR_MAX_TASKS");
  CUR_REQUIRE(experts && row_expert && o && g && out_pi, "NULL argument");
  CUR_REQUIRE(!d->modular || td, "task_descr required for a modular net");
  CUR_REQUIRE(n > 0 && n <= G_MAXROWS, "bad row count (the routed action launch covers up to 512 rows)");
  CUR_REQUIRE(rows_supported(d, S_ROWS), "shape not supported by the rows schedule (see cur_ddpg_rows_supported)");
  int count[CUR_MAX_TASKS] = {0};
  for (int64_t i = 0; i < n; ++i) {
    CUR_REQUIRE(row_expert[i] >= 0 && row_expert[i] < n_experts, "row_expert entry out of range");
    ++count[row_expert[i]];
  }
  int first = -1;
  for (int e = 0; e < n_experts; ++e) {
    if (count[e] == 0) continue;
    const cur_actions_expert& X = experts[e];
    CUR_REQUIRE(X.theta, "NULL theta");
    if (d->normalize_obs)
      CUR_REQUIRE(X.stats.o_mean && X.stats.o_std && X.stats.g_mean && X.stats.g_std, "normalizer stats required");
    if (first < 0) first = e;
  }
  ActGroupParams P;
  memset(&P, 0, sizeof(P));
  const float* theta0 = experts[first].theta;
  CUR_TRY(act_common(P, d, theta0, o, ag, g, td, clip_obs, out_pi, out_q, seq));
  for (int i = 0; i < P.nchunks; ++i) {
    P.coff[i] = (int32_t)(P.chunks[i].src - theta0);
    P.chunks[i].src = nullptr;
  }
  int base[CUR_MAX_TASKS], fill[CUR_MAX_TASKS] = {0}, tiles = 0;
  for (int e = 0; e < n_experts; ++e) {
    base[e] = tiles;
    tiles += (count[e] + S_ROWS - 1) / S_ROWS;
    if (count[e] == 0) continue;
    ActExpert& E = P.ex[e];
    E.theta = experts[e].theta;
    E.o_mean = experts[e].stats.o_mean; E.o_std = experts[e].stats.o_std;
    E.g_mean = experts[e].stats.g_mean; E.g_std = experts[e].stats.g_std;
    act_net_ptrs(E, *d, E.theta);
  }
  for (int t = 0; t < tiles; ++t)
    for (int r = 0; r < S_ROWS; ++r) P.tile_row[t][r] = -1;
  for (int64_t i = 0; i < n; ++i) {
    const int e = row_expert[i], k = fill[e]++;
    P.tile_ex[base[e] + k / S_ROWS] = (uint8_t)e;
    P.tile_row[base[e] + k / S_ROWS][k % S_ROWS] = (int16_t)i;
  }
  const int H = d->hidden;
  if (H == 64) CUR_TRY(launch_actions<64>((unsigned)tiles, (cudaStream_t)stream, P));
  else if (H == 128) CUR_TRY(launch_actions<128>((unsigned)tiles, (cudaStream_t)stream, P));
  else CUR_TRY(launch_actions<256>((unsigned)tiles, (cudaStream_t)stream, P));
  CUR_CHECK_LAUNCH();
  return CUR_OK;
}

// Mapped pinned host memory for the zero-copy action path: *host_ptr is the CPU address, *dev_ptr the address the
// kernels use (equal under unified addressing).  Freed with cur_host_free.
extern "C" int cur_host_alloc(int64_t bytes, void** host_ptr, void** dev_ptr) {
  CUR_REQUIRE(bytes > 0 && host_ptr && dev_ptr, "bad argument");
  CUR_CUDA_TRY(cudaHostAlloc(host_ptr, (size_t)bytes, cudaHostAllocMapped | cudaHostAllocPortable));
  CUR_CUDA_TRY(cudaHostGetDevicePointer(dev_ptr, *host_ptr, 0));
  memset(*host_ptr, 0, (size_t)bytes);
  return CUR_OK;
}

// cudaMemcpyAsync(host -> device) on `stream` (`src` from cur_host_alloc, so the copy is asynchronous)
extern "C" int cur_copy_h2d(void* stream, void* dst, const void* src, int64_t bytes) {
  CUR_REQUIRE(dst && src && bytes >= 0, "bad argument");
  CUR_CUDA_TRY(cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream));
  return CUR_OK;
}

extern "C" int cur_host_free(void* host_ptr) {
  if (host_ptr) CUR_CUDA_TRY(cudaFreeHost(host_ptr));
  return CUR_OK;
}

static inline float __uint_as_float_host(uint32_t b) {
  float f;
  memcpy(&f, &b, sizeof(f));
  return f;
}

// Host-side tail of the zero-copy action path (DDPG.get_actions, ddpg.py:147-155): wait until every one of the n_out
// 8-byte output words {float32 bits | seq << 32} written by actions_stream_kernel carries this call's number, then apply
// the reference's post-processing with the caller's draws (np.random, taken in reference order while the launch was in
// flight).  The arithmetic restates NumPy's evaluation of the reference statements, type for type:
//   u += noise_eps * max_u * randn           float32 array += float64 array: float64 add, rounded to float32
//   u = clip(u, -max_u, max_u)               float32 (the Python float bound is a weak scalar)
//   u += explore[:, None] * (u_rand - u)     int64 * (float64 - float32) -> float64 add, rounded to float32
// Returns CUR_OK, or CUR_ERR_UNSUPPORTED if the words did not arrive within max_spins polls (the caller synchronises the
// stream to let a launch failure surface and calls again).  No CUDA call is made here.
extern "C" int cur_actions_finish_host(const void* out_words, int64_t n, int dimu, int with_q, uint32_t seq,
                                       const double* randn, const int64_t* explore, const double* u_rand, double noise_scale,
                                       double max_u, float* u_out, float* q_out, int64_t max_spins) {
  CUR_REQUIRE(out_words && u_out && n > 0 && dimu > 0, "bad argument");
  CUR_REQUIRE(!with_q || q_out, "q_out required");
  CUR_REQUIRE((randn == nullptr) == (explore == nullptr) && (randn == nullptr) == (u_rand == nullptr),
              "the three draws come together");
  const volatile unsigned long long* w = reinterpret_cast<const volatile unsigned long long*>(out_words);
  const int64_t n_pi = n * dimu, n_out = n_pi + (with_q ? n : 0);
  int64_t spins = 0, done = 0;
  while (done < n_out) {
    if ((uint32_t)(w[done] >> 32) == seq) { ++done; continue; }
    if (++spins > max_spins) return CUR_ERR_UNSUPPORTED;
  }
  const float lim = (float)max_u;
  for (int64_t r = 0; r < n; ++r) {
    for (int j = 0; j < dimu; ++j) {
      const int64_t i = r * dimu + j;
      float u = __uint_as_float_host((uint32_t)w[i]);
      if (randn != nullptr) {
        const double noise = noise_scale * randn[i];
        u = (float)((double)u + noise);
        if (u < -lim) u = -lim;                       // np.maximum / np.minimum: NaN stays NaN
        if (u > lim) u = lim;
        const double step = (double)explore[r] * (u_rand[i] - (double)u);
        u = (float)((double)u + step);
      }
      u_out[i] = u;
    }
    if (with_q) q_out[r] = __uint_as_float_host((uint32_t)w[n_pi + r]);
  }
  return CUR_OK;
}
