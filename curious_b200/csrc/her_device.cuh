// Per-row pieces of the fused HER relabel kernel, shared by her.cu (the batched kernel) and ddpg_rows.cu (which
// samples its own 4 rows in the prologue of the update kernel).  Same draws, same relabelling, same reward:
// the two callers are bit-identical by construction.
//
// Reference: baselines/her/her.py:108-118 (draws), :129-164 (relabel), :174-176 + config.py:158-159 (reward),
// ddpg.py:326-345 (segment table).
#pragma once
#include "common.cuh"

namespace cur {

struct HerPlan {
  // shared-memory image of one transition = its transition row [o(t) | step block] (without the 64-byte tail padding),
  // then the future achieved goal, then (optionally) the cold row [change | info | ag(t)]
  int img4;         // 16-byte chunks of the transition row that are copied
  int fut_off, fut4;
  int cold_off, cold4;   // cold4 == 0 when neither change / info / ag(t) are needed
  int stage_stride; // floats per transition in shared memory
  int dimg_pad;
  // image indices of the sections
  int iO, iG, iU, iTD, iAG2, iO2;
  int iAG;          // ag(t): inside the cold part, valid only when cold4 > 0
};


struct HerRow {
  int ep, t, ft, choice, ttr;
  bool her;
};

// Draws of one row whose segment is known (base, E episodes): c indexes the injected stream, (ctr, call_offset) is the
// Philox counter under `seed`; then the three source addresses.  cdf(k): the CP_TASK cdf, cold(): the segment's cold rows.
template <class Cdf, class Cold>
__device__ __forceinline__ void her_draw_at(const cur_her_args& a, const HerPlan& pl, int64_t c, int64_t ctr,
                                            uint64_t call_offset, uint64_t seed, const float* base, int E, HerRow& row,
                                            const float** src, Cdf cdf, Cold cold) {
  const cur_layout& L = a.L;
  double u_her, u_off;
  if (a.inj_ep != nullptr) {
    row.ep = a.inj_ep[c];
    row.t = a.inj_t[c];
    u_her = a.inj_u_her[c];
    u_off = a.inj_u_off[c];
    if (a.inj_choice) row.choice = a.inj_choice[c];
  } else {
    Philox x = philox4x32_10((uint32_t)ctr, (uint32_t)(ctr >> 32), (uint32_t)call_offset, (uint32_t)(call_offset >> 32),
                             (uint32_t)seed, (uint32_t)(seed >> 32));
    row.ep = (int)mulhi32(x.x[0], (uint32_t)E);
    row.t = (int)mulhi32(x.x[1], (uint32_t)L.T);
    u_her = u01_from_u32(x.x[2]);
    u_off = u01_from_u32(x.x[3]);
    if (a.mode == CUR_MODE_RANDOM_TASK || a.mode == CUR_MODE_CP_TASK) {
      Philox y = philox4x32_10((uint32_t)ctr, (uint32_t)(ctr >> 32), (uint32_t)call_offset,
                               (uint32_t)(call_offset >> 32) ^ 0x80000000u, (uint32_t)seed,
                               (uint32_t)(seed >> 32));
      if (a.mode == CUR_MODE_RANDOM_TASK) {
        row.choice = (int)mulhi32(y.x[0], (uint32_t)a.tasks.n_tasks);
      } else {
        // np.random.choice(p=): cdf.searchsorted(u, side='right')
        double u = u01_from_u32(y.x[0]);
        int k = 0;
        while (k < a.tasks.n_tasks - 1 && cdf(k) <= u) ++k;
        row.choice = k;
      }
    }
  }
  row.her = u_her < a.future_p;                                                   // her.py:115
  row.ft = row.her ? row.t + 1 + (int)(u_off * (double)(L.T - row.t)) : -1;       // her.py:116-118
  const int64_t tr = (int64_t)row.ep * L.T + row.t;
  src[0] = base + tr * (int64_t)L.trans_stride;
  // ag(future_t) is the ag(t+1) block of transition future_t - 1 (future_t >= 1)
  src[1] = row.her ? base + ((int64_t)row.ep * L.T + (row.ft - 1)) * (int64_t)L.trans_stride + pl.iAG2 : nullptr;
  src[2] = (pl.cold4 > 0) ? cold() + tr * (int64_t)L.cold_stride : nullptr;
}

// Draws of concat row j (injected stream or Philox), segment lookup, and the three source addresses of the row:
// src[0] main span, src[1] future achieved goal (NULL: not a HER row), src[2] cold row (NULL: not requested).
// dyn_copy / step_val (optional): the caller's copy of the device control block and of *dyn->step, fetched up front in two round
// trips (the rows kernels draw on the critical path of every update; read in place the block costs ~7 dependent ones).
__device__ __forceinline__ void her_draw_row(const cur_her_args& a, const HerPlan& pl, int64_t j, HerRow& row,
                                             const float** src, const cur_her_dyn* dyn_copy = nullptr,
                                             const int64_t* step_val = nullptr) {
  const int64_t c = a.perm ? (int64_t)a.perm[j] : j;
  // segment lookup: concat rows are the segments' counts laid end to end (ddpg.py:326-345)
  // (with a device control block - CUDA-graph replays - counts / sizes / counter come from memory)
  const cur_her_dyn* dyn = (a.dyn != nullptr && dyn_copy != nullptr) ? dyn_copy : a.dyn;
  int s = 0;
  int64_t acc = 0;
  while (s + 1 < a.n_segments) {
    const int cnt = dyn ? dyn->count[s] : a.seg[s].count;
    if (c < acc + cnt) break;
    acc += cnt;
    ++s;
  }
  const float* base = a.seg[s].base;
  const int E = dyn ? dyn->n_episodes[s] : a.seg[s].n_episodes;
  row.ttr = a.seg[s].task_to_replay;
  row.choice = -1;
  const uint64_t call_offset = a.call_offset + (dyn ? (uint64_t)(step_val ? *step_val : *dyn->step) : 0ull);
  her_draw_at(a, pl, c, c, call_offset, a.seed, base, E, row, src,
              [&](int k) { return dyn ? dyn->cdf[k] : a.tasks.cdf[k]; }, [&]() { return a.seg[s].cold; });
}

// One worker of cur_her_sample_workers: its Philox key and its own segments (the counts and sizes are read from the
// worker's device control block).
struct HerWorkerTab {
  uint64_t seed;
  int32_t n_segments;
  int32_t ttr[CUR_MAX_SEGMENTS];
  const float* base[CUR_MAX_SEGMENTS];
  const float* cold[CUR_MAX_SEGMENTS];
};

// her_draw_row of the worker-major form: concat row c = perm ? perm[j] : j belongs to worker c / rpw at local row
// i = c % rpw, which is looked up in that worker's segments and drawn at Philox counter (i, call_offset + *step) under its key.
__device__ __forceinline__ void her_draw_row_worker(const cur_her_args& a, const HerPlan& pl, int64_t j, int rpw,
                                                    const HerWorkerTab* wt, const cur_her_worker_dyn* dyn,
                                                    const int64_t* step, HerRow& row, const float** src) {
  const int64_t c = a.perm ? (int64_t)a.perm[j] : j;
  const int w = (int)(c / rpw);
  const int64_t i = c - (int64_t)w * rpw;
  const HerWorkerTab& t = wt[w];
  const cur_her_worker_dyn& d = dyn[w];
  int s = 0;
  int64_t acc = 0;
  while (s + 1 < t.n_segments) {
    const int cnt = d.count[s];
    if (i < acc + cnt) break;
    acc += cnt;
    ++s;
  }
  row.ttr = t.ttr[s];
  row.choice = -1;
  const uint64_t call_offset = a.call_offset + (step ? (uint64_t)*step : 0ull);
  her_draw_at(a, pl, c, i, call_offset, t.seed, t.base[s], d.n_episodes[s], row, src, [&](int k) { return d.cdf[k]; },
              [&]() { return t.cold[s]; });
}

// Squared distance of module m (float64, NumPy's operation order: difference, square, running sum - no FMA
// contraction), added to d2.  PAIR compares the OFFSET between two achieved-goal sub-slices with the goal slice.
__device__ __forceinline__ double reward_d2(const cur_task_table& tt, int m, const float* ag2, const float* gf, double d2) {
  const int kind = tt.kind[m];
  if (kind == CUR_REWARD_INFO) return d2;
  for (int k = 0; k < tt.len[m]; ++k) {
    double av = (double)ag2[tt.ag_idx[m][k]];
    if (kind == CUR_REWARD_PAIR) av = av - (double)ag2[tt.ref_idx[m][k]];
    const double diff = av - (double)gf[tt.g_idx[m][k]];
    d2 = __dadd_rn(d2, __dmul_rn(diff, diff));
  }
  return d2;
}

// Relabel the staged image of one row in place (g, task_descr) and return its reward.
// image indices come from the plan.  *relab_out receives the module whose goal slice was relabelled (-1: none).
__device__ __forceinline__ float her_relabel_row(const cur_her_args& a, const HerPlan& pl, float* st, const HerRow& row,
                                                 int* relab_out) {
  const cur_layout& L = a.L;
  const int iG = pl.iG, iTD = pl.iTD, iAG2 = pl.iAG2;
  const bool wipe = (a.mode == CUR_MODE_BUFFER || a.mode == CUR_MODE_RANDOM_TASK || a.mode == CUR_MODE_CP_TASK);
  int own = -1;
  for (int k = 0; k < L.dimtd; ++k)
    if (st[iTD + k] == 1.0f) { own = k; break; }                 // argwhere(td == 1) (her.py:134)
  int relab = -1, newtd = -1;
  if (row.her) {
    switch (a.mode) {
      case CUR_MODE_BUFFER: relab = (row.ttr >= 0) ? row.ttr : own; newtd = relab; break;
      case CUR_MODE_RANDOM_TASK:
      case CUR_MODE_CP_TASK: relab = row.choice; newtd = relab; break;
      case CUR_MODE_CURRENT_TASK: relab = own; newtd = -1; break;
      default: break;                          // FLAT handled below
    }
    // relabel IN PLACE in the staged image (this lane owns the row)
    const float* fut = st + pl.fut_off;
    if (a.mode == CUR_MODE_FLAT) {
      for (int m = 0; m < a.tasks.n_tasks; ++m)                   // her.py:43-47
        for (int k = 0; k < a.tasks.len[m]; ++k) st[iG + a.tasks.g_idx[m][k]] = fut[a.tasks.ag_idx[m][k]];
    } else if (relab >= 0) {
      if (wipe) {
        for (int k = 0; k < L.dimg; ++k) st[iG + k] = 0.0f;       // her.py:151
        for (int k = 0; k < L.dimtd; ++k) st[iTD + k] = (k == newtd) ? 1.0f : 0.0f;   // her.py:152,155
      }
      for (int k = 0; k < a.tasks.len[relab]; ++k)                // her.py:154 / 163
        st[iG + a.tasks.g_idx[relab][k]] = fut[a.tasks.ag_idx[relab][k]];
    } else if (wipe) {
      // HER row whose module could not be determined (task_descr not one-hot): the reference would
      // raise; clear like her.py:151-152 so the output is at least well defined
      for (int k = 0; k < L.dimg; ++k) st[iG + k] = 0.0f;
      for (int k = 0; k < L.dimtd; ++k) st[iTD + k] = 0.0f;
    }
  }
  *relab_out = relab;
  // reward on (ag_2, relabelled g, final task_descr[, info]) - the module's row of the reward table
  const float* ag2 = st + iAG2;
  const float* gf = st + iG;
  if (a.mode == CUR_MODE_FLAT) {
    double d2 = 0.0;
    for (int m = 0; m < a.tasks.n_tasks; ++m) d2 = reward_d2(a.tasks, m, ag2, gf, d2);
    return (sqrt(d2) > a.tasks.flat_threshold) ? -1.0f : 0.0f;
  }
  const int m = (newtd >= 0) ? newtd : own;
  if (m >= 0 && a.tasks.kind[m] == CUR_REWARD_INFO)
    return (float)((double)st[pl.cold_off + L.off_info + a.tasks.info_col[m]] - 1.0);
  const double d2 = (m >= 0) ? reward_d2(a.tasks, m, ag2, gf, 0.0) : 0.0;
  return (sqrt(d2) > a.tasks.threshold[m >= 0 ? m : 0]) ? -1.0f : 0.0f;
}

// true when some module's reward reads the stored info row (the cold row then travels with every transition)
inline bool reward_needs_info(const cur_task_table& tt) {
  for (int m = 0; m < tt.n_tasks; ++m)
    if (tt.kind[m] == CUR_REWARD_INFO) return true;
  return false;
}

inline int make_plan(const cur_her_args& a, HerPlan* p) {
  const cur_layout& L = a.L;
  const bool need_ag_t = (a.ag != nullptr) || a.relative_goals;
  const bool need_cold = (a.change != nullptr && L.dimchange > 0) || (a.info != nullptr && L.diminfo > 0) ||
                         (reward_needs_info(a.tasks) && L.diminfo > 0);
  const int dimo_pad = round_up4(L.dimo);
  p->img4 = (dimo_pad + L.row_stride) / 4;
  p->fut_off = dimo_pad + L.row_stride;
  p->fut4 = round_up4(L.dimag) / 4;
  p->cold_off = p->fut_off + 4 * p->fut4;
  p->cold4 = (need_cold || need_ag_t) ? L.cold_stride / 4 : 0;
  p->stage_stride = p->cold_off + 4 * p->cold4;
  // one lane per row walks its image in the draw / relabel passes: an odd number of 16-byte units per row keeps the
  // rows of a warp off the same shared-memory banks (128 floats per row would be a 32-way conflict)
  if ((p->stage_stride / 4) % 2 == 0) p->stage_stride += 4;
  p->iO = 0;
  p->iG = dimo_pad + L.off_g; p->iU = dimo_pad + L.off_u; p->iTD = dimo_pad + L.off_td;
  p->iAG2 = dimo_pad + L.off_ag; p->iO2 = dimo_pad + L.off_o;
  p->iAG = p->cold_off + L.off_agc;
  p->dimg_pad = round_up4(L.dimg);
  return CUR_OK;
}


}  // namespace cur
