// Replay storage + fused HER relabel / gather / reward / preprocess kernel (sm_100a).
//
// Replaces (reference flowersteam/curious, paths relative to its root):
//   baselines/her/replay_buffer.py:57-72      store_episode           -> cur_store_episodes
//   baselines/her/her.py:20-66, 99-183        _sample_her_transitions -> cur_her_sample
//   baselines/her/ddpg.py:325-345, 350-353    per-buffer loop, concat, shuffle, _preprocess_og
//   config.py:158-159 reward_fun              restated module-distance reward (DESIGN.md)
//
// Kernel design (HBM bound, one ~0.5 KB gather per transition; ncu history in profiles/):
//   * one CTA = TILE consecutive OUTPUT rows, 4 warps;
//   * warp 0 decodes the per-row draws (injected stream or Philox4x32-10), one lane per row, and
//     publishes three source addresses per row (main span, future achieved goal, cold row);
//   * all warps then copy global -> shared with per-lane 16-byte cp.async (SASS LDGSTS, L2-only
//     `.cg`): a transition is ONE 64-byte aligned row of the transition-major storage, so a
//     single warp-wide LDGSTS moves an Arm4 transition (28 lanes row + 3 lanes future goal);
//     no register staging, ~16 KB in flight per CTA, up to 14 CTAs per SM;
//   * relabel (g, task_descr), the float64 reward and the clip are evaluated straight out of shared
//     memory and every output array is written as contiguous, fully coalesced 16-byte stores.
#include "her_device.cuh"

namespace cur {

thread_local char g_last_error[256] = {0};

int sm_count() {
  static int cached = 0;
  if (cached == 0) {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) == cudaSuccess &&
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
      cached = n;
    else
      return 148;
  }
  return cached;
}

// CTA shape of the sampling kernel: TILE transitions, HER_THREADS threads (template parameters of the kernel)

struct HerKernelParams {
  cur_her_args a;
  HerPlan p;
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void cp_async16(void* dst_smem, const void* src_gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst_smem)), "l"(src_gmem)
               : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
  asm volatile("cp.async.commit_group;\n cp.async.wait_group 0;" ::: "memory");
}

__device__ __forceinline__ float clipf(float x, float c) { return fminf(fmaxf(x, -c), c); }

// Cooperative, coalesced write of `nrows` rows of `dim` floats starting at output row j0 by threads t = 0 .. nt-1.
// src(tr, k) returns element k of tile-row tr.  The output span is contiguous and 128-byte aligned
// (j0 is a multiple of TILE), so dim % 4 == 0 takes the 16-byte path.
template <typename Src4, typename Src1>
__device__ __forceinline__ void emit(float* __restrict__ out, int dim, int64_t j0, int nrows, int t, int nt,
                                     Src4 src4, Src1 src1) {
  if (out == nullptr || dim <= 0) return;
  float* dst = out + j0 * (int64_t)dim;
  if ((dim & 3) == 0) {
    const int d4 = dim >> 2;
    const float inv = 1.0f / (float)d4;
    const int n4 = nrows * d4;
    for (int i = t; i < n4; i += nt) {
      int tr = __float2int_rz(((float)i + 0.5f) * inv);
      int k4 = i - tr * d4;
      reinterpret_cast<float4*>(dst)[i] = src4(tr, k4 << 2);
    }
  } else {
    const float inv = 1.0f / (float)dim;
    const int n = nrows * dim;
    for (int i = t; i < n; i += nt) {
      int tr = __float2int_rz(((float)i + 0.5f) * inv);
      int k = i - tr * dim;
      dst[i] = src1(tr, k);
    }
  }
}

// Two outputs of the same width sharing the index arithmetic (o/o_2, g/g_2, ag/ag_2).
template <typename A4, typename B4, typename A1, typename B1>
__device__ __forceinline__ void emit2(float* __restrict__ outa, float* __restrict__ outb, int dim, int64_t j0,
                                      int nrows, int t, int nt, A4 a4, B4 b4, A1 a1, B1 b1) {
  if (outa == nullptr) { emit(outb, dim, j0, nrows, t, nt, b4, b1); return; }
  if (outb == nullptr) { emit(outa, dim, j0, nrows, t, nt, a4, a1); return; }
  if (dim <= 0) return;
  float* da = outa + j0 * (int64_t)dim;
  float* db = outb + j0 * (int64_t)dim;
  if ((dim & 3) == 0) {
    const int d4 = dim >> 2;
    const float inv = 1.0f / (float)d4;
    const int n4 = nrows * d4;
    for (int i = t; i < n4; i += nt) {
      int tr = __float2int_rz(((float)i + 0.5f) * inv);
      int k = (i - tr * d4) << 2;
      reinterpret_cast<float4*>(da)[i] = a4(tr, k);
      reinterpret_cast<float4*>(db)[i] = b4(tr, k);
    }
  } else {
    const float inv = 1.0f / (float)dim;
    const int n = nrows * dim;
    for (int i = t; i < n; i += nt) {
      int tr = __float2int_rz(((float)i + 0.5f) * inv);
      int k = i - tr * dim;
      da[i] = a1(tr, k);
      db[i] = b1(tr, k);
    }
  }
}

// One CTA = one tile of TILE output rows, one shared-memory stage (~16 KB: 12 - 14 CTAs per SM overlap their phases):
//   draws (warp 0) | gather (all warps, cp.async) | relabel + reward (warp 0) NEXT TO the outputs that do not depend on it
//   (o, o_2, u, ag, ag_2, change, info: warps 1 - 3) | the relabelled outputs (g, g_2, task_descr: all warps).
// (A persistent double-buffered variant - draws and gather of tile i+1 issued before tile i is waited for - was measured
// slower, 70 % vs 81 % of the HBM peak: throughput follows the number of resident tiles per SM, profiles/README.md.)
// draw(j, row, src): her_draw_row of output row j (her_draw_row_worker in the worker-major form).
template <int TILE, int HER_THREADS, class Draw>
__device__ __forceinline__ void her_tile(const cur_her_args& a, const HerPlan& pl, Draw draw) {
  constexpr int HER_WARPS = HER_THREADS / 32;
  const cur_layout& L = a.L;
  extern __shared__ __align__(128) unsigned char smem_raw[];

  float* stage = reinterpret_cast<float*>(smem_raw);                              // TILE * stage_stride
  // per row: source address of [0] the transition row, [1] the future achieved goal (NULL: not a HER
  // row), [2] the cold row (NULL: not requested)
  const float** m_src = reinterpret_cast<const float**>(stage + TILE * pl.stage_stride);    // TILE * 3

  const int tid = threadIdx.x;
  const int lane = tid & 31, warp = tid >> 5;
  const int64_t j0 = (int64_t)blockIdx.x * TILE;
  const int nrows = (int)min((int64_t)TILE, a.batch - j0);
  const int ss = pl.stage_stride;

  // ---------------------------------------------------------------- phase A: draws (warp 0)
  HerRow row;
  row.ft = -1; row.choice = -1; row.ep = 0; row.t = 0; row.ttr = -1; row.her = false;
  if (warp == 0 && lane < nrows) draw(j0 + lane, row, m_src + 3 * lane);
  __syncthreads();

  // ---------------------------------------------------------------- copies: global -> shared
  // Each lane owns a fixed 16-byte chunk slot of the per-transition stage (region, index in region,
  // destination offset are loop invariant); per row it only fetches the region's source address.
  {
    const int per_row = pl.img4 + pl.fut4 + pl.cold4;
    const uint32_t stage_s = smem_u32(stage);
    for (int c0 = 0; c0 < per_row; c0 += 32) {
      const int ch = c0 + lane;
      int sel = 0, q = ch, doff = 4 * ch;
      if (ch >= pl.img4 + pl.fut4) { sel = 2; q = ch - pl.img4 - pl.fut4; doff = pl.cold_off + 4 * q; }
      else if (ch >= pl.img4) { sel = 1; q = ch - pl.img4; doff = pl.fut_off + 4 * q; }
      const bool active = ch < per_row;
      uint32_t dst = stage_s + 4u * (uint32_t)(warp * ss + doff);
      const uint32_t dstep = 4u * (uint32_t)(HER_WARPS * ss);
      for (int r = warp; r < nrows; r += HER_WARPS, dst += dstep) {
        const float* src = m_src[3 * r + sel];
        if (active && src != nullptr)
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src + 4 * q) : "memory");
      }
    }
    cp_async_wait_all();
  }
  __syncthreads();

  // image indices (HerPlan): o(t) first, then the step block; ag(t) sits in the cold part of the image
  const int iG = pl.iG, iU = pl.iU, iTD = pl.iTD, iAG2 = pl.iAG2, iO2 = pl.iO2, iO = pl.iO, iAG = pl.iAG;
  const float c = a.clip_obs;
  const bool do_clip = c > 0.0f;
  auto ld4 = [&](int tr, int off) {
    return *reinterpret_cast<const float4*>(stage + tr * ss + off);
  };
  auto clip4 = [&](float4 v) {
    if (do_clip) { v.x = clipf(v.x, c); v.y = clipf(v.y, c); v.z = clipf(v.z, c); v.w = clipf(v.w, c); }
    return v;
  };
  auto clip1 = [&](float v) { return do_clip ? clipf(v, c) : v; };
  auto sub4 = [&](float4 x, float4 y) { return make_float4(x.x - y.x, x.y - y.y, x.z - y.z, x.w - y.w); };

  if (warp == 0) {
    // ---------------------------------------------------------------- module decisions + reward (one lane per row)
    if (lane < nrows) {
      int relab_out = -1;
      const float rew1 = her_relabel_row(a, pl, stage + lane * ss, row, &relab_out);
      if (a.idx_out) {
        int32_t* io = a.idx_out + (j0 + lane) * 4;
        io[0] = row.ep; io[1] = row.t; io[2] = row.ft;
        io[3] = row.her ? ((a.mode == CUR_MODE_FLAT) ? 0 : relab_out) : -1;
      }
      if (a.r != nullptr) a.r[j0 + lane] = rew1;
    }
  } else {
    // ---------------------------------------------------------------- outputs the relabelling does not touch
    const int t = tid - 32, nt = HER_THREADS - 32;
    emit2(a.o, a.o_2, L.dimo, j0, nrows, t, nt,
          [&](int tr, int k) { return clip4(ld4(tr, iO + k)); },
          [&](int tr, int k) { return clip4(ld4(tr, iO2 + k)); },
          [&](int tr, int k) { return clip1(stage[tr * ss + iO + k]); },
          [&](int tr, int k) { return clip1(stage[tr * ss + iO2 + k]); });
    emit(a.u, L.dimu, j0, nrows, t, nt,
         [&](int tr, int k) { return ld4(tr, iU + k); },
         [&](int tr, int k) { return stage[tr * ss + iU + k]; });
    emit2(a.ag, a.ag_2, L.dimag, j0, nrows, t, nt,
          [&](int tr, int k) { return ld4(tr, iAG + k); },
          [&](int tr, int k) { return ld4(tr, iAG2 + k); },
          [&](int tr, int k) { return stage[tr * ss + iAG + k]; },
          [&](int tr, int k) { return stage[tr * ss + iAG2 + k]; });
    emit(a.change, L.dimchange, j0, nrows, t, nt,
         [&](int tr, int k) { return ld4(tr, pl.cold_off + L.off_change + k); },
         [&](int tr, int k) { return stage[tr * ss + pl.cold_off + L.off_change + k]; });
    emit(a.info, L.diminfo, j0, nrows, t, nt,
         [&](int tr, int k) { return ld4(tr, pl.cold_off + L.off_info + k); },
         [&](int tr, int k) { return stage[tr * ss + pl.cold_off + L.off_info + k]; });
  }
  __syncthreads();

  // ---------------------------------------------------------------- the relabelled outputs
  emit(a.td, L.dimtd, j0, nrows, tid, HER_THREADS,
       [&](int tr, int k) { return ld4(tr, iTD + k); },
       [&](int tr, int k) { return stage[tr * ss + iTD + k]; });
  // g / g_2 (ddpg.py:350-353): optional relative goals, then clip
  if (a.relative_goals) {
    emit2(a.g, a.g_2, L.dimg, j0, nrows, tid, HER_THREADS,
          [&](int tr, int k) { return clip4(sub4(ld4(tr, iG + k), ld4(tr, iAG + k))); },
          [&](int tr, int k) { return clip4(sub4(ld4(tr, iG + k), ld4(tr, iAG2 + k))); },
          [&](int tr, int k) { return clip1(stage[tr * ss + iG + k] - stage[tr * ss + iAG + k]); },
          [&](int tr, int k) { return clip1(stage[tr * ss + iG + k] - stage[tr * ss + iAG2 + k]); });
  } else {
    emit2(a.g, a.g_2, L.dimg, j0, nrows, tid, HER_THREADS,
          [&](int tr, int k) { return clip4(ld4(tr, iG + k)); },
          [&](int tr, int k) { return clip4(ld4(tr, iG + k)); },
          [&](int tr, int k) { return clip1(stage[tr * ss + iG + k]); },
          [&](int tr, int k) { return clip1(stage[tr * ss + iG + k]); });
  }
}

template <int TILE, int HER_THREADS>
__global__ void __launch_bounds__(HER_THREADS)
her_sample_kernel(const __grid_constant__ HerKernelParams P) {
  const cur_her_args& a = P.a;
  const HerPlan& pl = P.p;
  her_tile<TILE, HER_THREADS>(a, pl, [&](int64_t j, HerRow& row, const float** src) { her_draw_row(a, pl, j, row, src); });
}

struct HerWorkersParams {
  cur_her_args a;
  HerPlan p;
  int32_t rows_per_worker;
  const cur_her_worker_dyn* dyn;
  const int64_t* step;
  HerWorkerTab w[CUR_MAX_WORKERS];
};
static_assert(sizeof(HerWorkersParams) <= 32764, "kernel parameter limit");

// cur_her_sample_workers: the tile of her_sample_kernel, each row drawn from its worker's segments and stream.
template <int TILE, int HER_THREADS>
__global__ void __launch_bounds__(HER_THREADS)
her_sample_workers_kernel(const __grid_constant__ HerWorkersParams P) {
  const cur_her_args& a = P.a;
  const HerPlan& pl = P.p;
  her_tile<TILE, HER_THREADS>(a, pl, [&](int64_t j, HerRow& row, const float** src) {
    her_draw_row_worker(a, pl, j, P.rows_per_worker, P.w, P.dyn, P.step, row, src);
  });
}

// ------------------------------------------------------------------------------------------------
// store: pack key-major episodes into transition / cold rows, one CTA per (transition, copy)
// ------------------------------------------------------------------------------------------------
struct StoreParams {
  cur_layout L;
  cur_episode_src src;
  int n_copies;
  int32_t copy_src[CUR_MAX_COPIES];
  float* copy_hot[CUR_MAX_COPIES];
  float* copy_cold[CUR_MAX_COPIES];
  int64_t copy_slot[CUR_MAX_COPIES];
};

__global__ void __launch_bounds__(128) store_episodes_kernel(const __grid_constant__ StoreParams S) {
  const cur_layout& L = S.L;
  const int t = blockIdx.x;        // transition 0..T-1
  const int cpy = blockIdx.y;
  const int e = S.copy_src[cpy];
  float* dst = S.copy_hot[cpy] + (S.copy_slot[cpy] * L.T + t) * (int64_t)L.trans_stride;
  const int64_t rt = (int64_t)e * L.T + t;                 // step t of the key-major [n_ep, T, dim] arrays
  const int64_t rcur = (int64_t)e * (L.T + 1) + t;         // row t of the [n_ep, T+1, dim] arrays
  const int dimo_pad = round_up4(L.dimo);
  for (int k = threadIdx.x; k < L.trans_stride; k += blockDim.x) {
    float v = 0.0f;
    if (k < dimo_pad) {
      if (k < L.dimo) v = S.src.o[rcur * L.dimo + k];
    } else {
      const int b = k - dimo_pad;                          // inside the step block
      int j;
      if ((j = b - L.off_g) >= 0 && j < L.dimg) v = S.src.g[rt * L.dimg + j];
      else if ((j = b - L.off_u) >= 0 && j < L.dimu) v = S.src.u[rt * L.dimu + j];
      else if ((j = b - L.off_td) >= 0 && j < L.dimtd) { if (S.src.td) v = S.src.td[rt * L.dimtd + j]; }
      else if ((j = b - L.off_ag) >= 0 && j < L.dimag) v = S.src.ag[(rcur + 1) * L.dimag + j];
      else if ((j = b - L.off_o) >= 0 && j < L.dimo) v = S.src.o[(rcur + 1) * L.dimo + j];
    }
    dst[k] = v;
  }
  if (S.copy_cold[cpy] != nullptr) {
    float* cd = S.copy_cold[cpy] + (S.copy_slot[cpy] * L.T + t) * (int64_t)L.cold_stride;
    for (int k = threadIdx.x; k < L.cold_stride; k += blockDim.x) {
      float v = 0.0f;
      int j;
      if ((j = k - L.off_change) >= 0 && j < L.dimchange) { if (S.src.change) v = S.src.change[rt * L.dimchange + j]; }
      else if ((j = k - L.off_info) >= 0 && j < L.diminfo) { if (S.src.info) v = S.src.info[rt * L.diminfo + j]; }
      else if ((j = k - L.off_agc) >= 0 && j < L.dimag) v = S.src.ag[rcur * L.dimag + j];
      cd[k] = v;
    }
  }
}

}  // namespace cur

using namespace cur;

extern "C" int cur_abi_version(void) { return CUR_ABI_VERSION; }
extern "C" const char* cur_last_error(void) { return g_last_error; }

extern "C" int cur_device_info(int* sms, int* major, int* minor) {
  int dev = 0;
  CUR_CUDA_TRY(cudaGetDevice(&dev));
  if (sms) CUR_CUDA_TRY(cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev));
  if (major) CUR_CUDA_TRY(cudaDeviceGetAttribute(major, cudaDevAttrComputeCapabilityMajor, dev));
  if (minor) CUR_CUDA_TRY(cudaDeviceGetAttribute(minor, cudaDevAttrComputeCapabilityMinor, dev));
  return CUR_OK;
}

extern "C" int cur_layout_init(cur_layout* L, int T, int dimo, int dimag, int dimg, int dimu, int dimtd,
                               int dimchange, int diminfo) {
  CUR_REQUIRE(L != nullptr, "layout is NULL");
  CUR_REQUIRE(T > 0 && dimo > 0 && dimag > 0 && dimg > 0 && dimu > 0, "T and o/ag/g/u dims must be > 0");
  CUR_REQUIRE(dimtd >= 0 && dimchange >= 0 && diminfo >= 0, "negative dim");
  CUR_REQUIRE(dimtd <= CUR_MAX_TASKS, "too many modules");
  L->T = T;
  L->dimo = dimo; L->dimag = dimag; L->dimg = dimg; L->dimu = dimu;
  L->dimtd = dimtd; L->dimchange = dimchange; L->diminfo = diminfo;
  // Step block: g, u, task_descr, ag(t+1) in the order that makes the ag(t+1) block - the one a HER row of ANOTHER
  // transition gathers on its own - straddle the fewest 64-byte DRAM atoms of the transition row; o(t+1) stays last.
  // Ties keep the earliest order in the enumeration below (g, u, td, ag first).
  const int dimo_pad = round_up4(dimo);
  const int w[4] = {round_up4(dimg), round_up4(dimu), round_up4(dimtd), round_up4(dimag)};   // g u td ag
  static const int perms[24][4] = {{0, 1, 2, 3}, {0, 1, 3, 2}, {0, 2, 1, 3}, {0, 2, 3, 1}, {0, 3, 1, 2}, {0, 3, 2, 1},
                                   {1, 0, 2, 3}, {1, 0, 3, 2}, {1, 2, 0, 3}, {1, 2, 3, 0}, {1, 3, 0, 2}, {1, 3, 2, 0},
                                   {2, 0, 1, 3}, {2, 0, 3, 1}, {2, 1, 0, 3}, {2, 1, 3, 0}, {2, 3, 0, 1}, {2, 3, 1, 0},
                                   {3, 0, 1, 2}, {3, 0, 2, 1}, {3, 1, 0, 2}, {3, 1, 2, 0}, {3, 2, 0, 1}, {3, 2, 1, 0}};
  int best = 0, best_atoms = 1 << 30;
  for (int p = 0; p < 24; ++p) {
    int off = 0, ag_at = 0;
    for (int i = 0; i < 4; ++i) {
      if (perms[p][i] == 3) ag_at = off;
      off += w[perms[p][i]];
    }
    const int first = (dimo_pad + ag_at) / 16, last = (dimo_pad + ag_at + w[3] - 1) / 16;
    if (last - first + 1 < best_atoms) { best_atoms = last - first + 1; best = p; }
  }
  int off = 0;
  int32_t* slot[4] = {&L->off_g, &L->off_u, &L->off_td, &L->off_ag};
  for (int i = 0; i < 4; ++i) { *slot[perms[best][i]] = off; off += w[perms[best][i]]; }
  L->off_o = off; off += dimo_pad;
  L->row_stride = off;
  L->trans_stride = (dimo_pad + off + 15) / 16 * 16;
  off = 0;
  L->off_change = off; off += round_up4(dimchange);
  L->off_info = off; off += round_up4(diminfo);
  L->off_agc = off; off += round_up4(dimag);
  L->cold_stride = off;
  return CUR_OK;
}

extern "C" int cur_store_episodes(void* stream, const cur_layout* L, const cur_episode_src* src, int n_ep,
                                  int n_copies, const int32_t* copy_src, float* const* copy_hot,
                                  float* const* copy_cold, const int64_t* copy_slot) {
  CUR_REQUIRE(L && src && copy_src && copy_hot && copy_slot, "NULL argument");
  CUR_REQUIRE(src->o && src->ag && src->g && src->u, "o/ag/g/u sources are required");
  CUR_REQUIRE(n_copies >= 0 && n_ep > 0, "bad counts");
  CUR_REQUIRE(copy_cold != nullptr, "cold destinations required");
  cudaStream_t s = (cudaStream_t)stream;
  for (int done = 0; done < n_copies; done += CUR_MAX_COPIES) {
    StoreParams S;
    S.L = *L;
    S.src = *src;
    S.n_copies = (n_copies - done < CUR_MAX_COPIES) ? n_copies - done : CUR_MAX_COPIES;
    for (int i = 0; i < S.n_copies; ++i) {
      CUR_REQUIRE(copy_src[done + i] >= 0 && copy_src[done + i] < n_ep, "copy_src out of range");
      CUR_REQUIRE(copy_hot[done + i] != nullptr && copy_slot[done + i] >= 0, "bad destination");
      S.copy_src[i] = copy_src[done + i];
      S.copy_hot[i] = copy_hot[done + i];
      CUR_REQUIRE(copy_cold[done + i] != nullptr, "bad cold destination");
      S.copy_cold[i] = copy_cold[done + i];
      S.copy_slot[i] = copy_slot[done + i];
    }
    dim3 grid(L->T, S.n_copies);
    store_episodes_kernel<<<grid, 128, 0, s>>>(S);
    CUR_CHECK_LAUNCH();
  }
  return CUR_OK;
}

// Checks shared by both sampling entries: mode, reward table, injected stream, relative goals.
static int check_her_common(const cur_her_args& a) {
  CUR_REQUIRE(a.mode >= CUR_MODE_BUFFER && a.mode <= CUR_MODE_FLAT, "unknown mode");
  CUR_REQUIRE(a.tasks.n_tasks >= 0 && a.tasks.n_tasks <= CUR_MAX_TASKS, "n_tasks out of range");
  CUR_REQUIRE(a.mode == CUR_MODE_FLAT || a.tasks.n_tasks == a.L.dimtd, "n_tasks must equal dimtd");
  CUR_REQUIRE(a.L.row_stride > 0 && (a.L.row_stride & 3) == 0, "layout not initialised");
  for (int m = 0; m < a.tasks.n_tasks; ++m) {
    CUR_REQUIRE(a.tasks.len[m] >= 0 && a.tasks.len[m] <= CUR_MAX_SLICE, "module slice too long");
    for (int k = 0; k < a.tasks.len[m]; ++k) {
      CUR_REQUIRE(a.tasks.g_idx[m][k] >= 0 && a.tasks.g_idx[m][k] < a.L.dimg, "g index out of range");
      CUR_REQUIRE(a.tasks.ag_idx[m][k] >= 0 && a.tasks.ag_idx[m][k] < a.L.dimag, "ag index out of range");
      if (a.tasks.kind[m] == CUR_REWARD_PAIR)
        CUR_REQUIRE(a.tasks.ref_idx[m][k] >= 0 && a.tasks.ref_idx[m][k] < a.L.dimag, "reference ag index out of range");
    }
    CUR_REQUIRE(a.tasks.kind[m] >= CUR_REWARD_DISTANCE && a.tasks.kind[m] <= CUR_REWARD_INFO, "unknown reward kind");
    if (a.tasks.kind[m] == CUR_REWARD_INFO)
      CUR_REQUIRE(a.tasks.info_col[m] >= 0 && a.tasks.info_col[m] < a.L.diminfo, "info column out of range");
  }
  if (a.inj_ep != nullptr)
    CUR_REQUIRE(a.inj_t && a.inj_u_her && a.inj_u_off, "incomplete injected stream");
  if (a.relative_goals) CUR_REQUIRE(a.L.dimg == a.L.dimag, "relative goals need dimg == dimag");
  return CUR_OK;
}

// CTA shape: 32 rows / 128 threads.  16 / 64 and 32 / 64 measured the same (Arm4 0.827 / 0.828 vs 0.830 of the HBM peak),
// 16 / 128 slower (0.655): at full size the kernel sits at the DRAM pipe, not at its own latency (profiles/README.md)
constexpr int HER_TILE = 32, HER_THREADS = 128;

template <class Params>
static int launch_her(void (*kernel)(Params), const Params& P, int64_t batch, cudaStream_t stream, size_t* configured) {
  size_t smem = (size_t)HER_TILE * P.p.stage_stride * 4 + 3 * HER_TILE * sizeof(void*) + 16;
  if (smem > 48 * 1024 && smem > *configured) {
    CUR_REQUIRE(smem <= 227 * 1024, "row too large for the shared-memory stage");
    CUR_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    *configured = smem;
  }
  const int64_t blocks = (batch + HER_TILE - 1) / HER_TILE;
  CUR_REQUIRE(blocks <= 0x7fffffff, "batch too large for one launch");
  kernel<<<(unsigned)blocks, HER_THREADS, smem, stream>>>(P);
  CUR_CHECK_LAUNCH();
  return CUR_OK;
}

extern "C" int cur_her_sample(void* stream, const cur_her_args* args) {
  CUR_REQUIRE(args != nullptr, "args is NULL");
  const cur_her_args& a = *args;
  CUR_REQUIRE(a.batch >= 0, "negative batch");
  if (a.batch == 0) return CUR_OK;
  CUR_REQUIRE(a.n_segments >= 1 && a.n_segments <= CUR_MAX_SEGMENTS, "n_segments out of range");
  if (int st = check_her_common(a)) return st;
  int64_t total = 0;
  for (int i = 0; i < a.n_segments; ++i) {
    CUR_REQUIRE(a.seg[i].count >= 0, "negative segment count");
    if (a.dyn != nullptr) {
      CUR_REQUIRE(a.seg[i].base != nullptr, "segment base is NULL");
    } else if (a.seg[i].count > 0) {
      CUR_REQUIRE(a.seg[i].base != nullptr, "segment base is NULL");
      CUR_REQUIRE(a.seg[i].n_episodes > 0, "sampling from an empty buffer (replay_buffer.py:43)");
      CUR_REQUIRE(a.seg[i].task_to_replay < a.tasks.n_tasks, "task_to_replay out of range");
    }
    total += a.seg[i].count;
  }
  CUR_REQUIRE(a.dyn != nullptr || total == a.batch, "segment counts must sum to batch (ddpg.py:323)");
  CUR_REQUIRE(a.dyn == nullptr || a.inj_ep == nullptr, "a device control block implies Philox draws");

  HerKernelParams P;
  P.a = a;
  make_plan(a, &P.p);
  if (P.p.cold4 > 0)
    for (int i = 0; i < a.n_segments; ++i)
      CUR_REQUIRE(a.seg[i].count == 0 || a.seg[i].cold != nullptr, "change/info/ag requested but segment has no cold rows");
  static size_t configured = 0;
  return launch_her(her_sample_kernel<HER_TILE, HER_THREADS>, P, a.batch, (cudaStream_t)stream, &configured);
}

extern "C" int cur_her_sample_workers(void* stream, const cur_her_args* args, int n_workers, int rows_per_worker,
                                      const cur_her_worker* w, const cur_her_worker_dyn* dyn, const int64_t* step) {
  CUR_REQUIRE(args != nullptr && w != nullptr && dyn != nullptr, "NULL argument");
  CUR_REQUIRE(n_workers >= 1 && n_workers <= CUR_MAX_WORKERS, "n_workers out of range (1..CUR_MAX_WORKERS)");
  CUR_REQUIRE(rows_per_worker >= 1, "rows_per_worker must be positive");
  const cur_her_args& a = *args;
  CUR_REQUIRE(a.batch == (int64_t)n_workers * rows_per_worker, "batch must equal n_workers * rows_per_worker");
  if (int st = check_her_common(a)) return st;
  HerWorkersParams P;
  P.a = a;
  make_plan(a, &P.p);
  for (int j = 0; j < n_workers; ++j) {
    const cur_her_worker& wj = w[j];
    CUR_REQUIRE(wj.n_segments >= 1 && wj.n_segments <= CUR_MAX_SEGMENTS, "a worker has n_segments outside 1..17");
    int64_t total = 0;
    HerWorkerTab& t = P.w[j];
    t.seed = wj.seed;
    t.n_segments = wj.n_segments;
    for (int i = 0; i < wj.n_segments; ++i) {
      const cur_segment& sg = wj.seg[i];
      CUR_REQUIRE(sg.count >= 0, "negative segment count");
      CUR_REQUIRE(sg.base != nullptr, "segment base is NULL");
      CUR_REQUIRE(sg.count == 0 || sg.n_episodes > 0, "sampling from an empty buffer (replay_buffer.py:43)");
      CUR_REQUIRE(sg.task_to_replay < a.tasks.n_tasks, "task_to_replay out of range");
      CUR_REQUIRE(P.p.cold4 == 0 || sg.count == 0 || sg.cold != nullptr,
                  "change/info/ag requested but segment has no cold rows");
      t.base[i] = sg.base;
      t.cold[i] = sg.cold;
      t.ttr[i] = sg.task_to_replay;
      total += sg.count;
    }
    CUR_REQUIRE(total == rows_per_worker, "a worker's segment counts must sum to rows_per_worker");
  }
  P.rows_per_worker = rows_per_worker;
  P.dyn = dyn;
  P.step = step;
  static size_t configured = 0;
  return launch_her(her_sample_workers_kernel<HER_TILE, HER_THREADS>, P, a.batch, (cudaStream_t)stream, &configured);
}

// ---------------------------------------------------------------- known-answer access to the generator
__global__ void philox_kat_kernel(const uint32_t* __restrict__ in, int64_t n, uint32_t* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t* c = in + 6 * i;
  const cur::Philox x = cur::philox4x32_10(c[0], c[1], c[2], c[3], c[4], c[5]);
  for (int k = 0; k < 4; ++k) out[4 * i + k] = x.x[k];
}

extern "C" int cur_philox4x32_10(void* stream, const uint32_t* in, int64_t n, uint32_t* out) {
  CUR_REQUIRE(n >= 0 && (n == 0 || (in != nullptr && out != nullptr)), "bad arguments");
  if (n == 0) return CUR_OK;
  philox_kat_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(in, n, out);
  CUR_CHECK_LAUNCH();
  return CUR_OK;
}
