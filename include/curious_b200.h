/*
 * curious_b200 C ABI - the drop-in boundary of the B200-native CURIOUS training hot path.
 *
 * The reference (flowersteam/curious) has no FFI: its hot path is Python/NumPy/TF1 behind the
 * duck-typed plugin surface wired by baselines/her/experiment/config.py:152-253.  This header is
 * the C-ABI a maintainer binds (ctypes stub in INTEGRATION.md) so that surface runs on one B200 per
 * rank.  Every entry point:
 *   - is `extern "C"`, takes plain pointers / sizes / a `cudaStream_t` passed as `void*`;
 *   - returns an int status (CUR_OK == 0); never throws; never allocates persistent memory;
 *   - works on DEVICE pointers unless the parameter is documented as host;
 *   - is asynchronous on `stream`.
 * Each declaration cites the reference code it replaces (paths relative to the reference root).
 */
#ifndef CURIOUS_B200_H
#define CURIOUS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CUR_ABI_VERSION 4

#define CUR_OK 0
#define CUR_ERR_INVALID 1   /* bad argument (dims, null pointer, table overflow)   */
#define CUR_ERR_CUDA 2      /* a CUDA runtime call failed; see cur_last_error()    */
#define CUR_ERR_UNSUPPORTED 3

#define CUR_MAX_TASKS 16    /* modules (nb_tasks)                                   */
#define CUR_MAX_SLICE 8     /* entries of one module's goal slice (tasks_g_id[m])   */
#define CUR_MAX_SEGMENTS 17 /* per-module buffers + buffer 0 (ddpg.py:255)          */
#define CUR_MAX_COPIES 64   /* (episode, destination) pairs per cur_store_episodes  */
#define CUR_MAX_LAYERS 8
#define CUR_MAX_RANKS 8      /* GPUs of one NVLink domain                            */

int cur_abi_version(void);
const char* cur_last_error(void);          /* message of the last CUR_ERR_CUDA on this thread */
int cur_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ------------------------------------------------------------------------------------------
 * Replay storage layout.  Replaces the float64 dict-of-arrays storage of
 * baselines/her/replay_buffer.py:23-24 by TWO float32 arrays per buffer:
 *
 *   hot  [E][T][trans_stride]   transition t = [ o(t) | step block ],  step block = g(t), u(t), task_descr(t),
 *                               ag(t+1), o(t+1) at off_g / off_u / off_td / off_ag / off_o (o(t+1) last)
 *   cold [E][T][cold_stride]    row t = [ change(t) | info(t) | ag(t) ]
 *
 * TRANSITION-major: everything a training transition needs (o_t, g_t, u_t, td_t, ag_{t+1}, o_{t+1}) is ONE row,
 * padded to a multiple of 64 bytes - the DRAM access granularity - so a sampled transition costs exactly
 * trans_stride * 4 bytes of DRAM reads (Arm4: 448 B = 7 atoms; the episode-major rows of round 1, 72 floats with the
 * span starting on a 32-byte boundary, cost 480 B on average), at the price of storing o twice (o(t+1) of transition t
 * is o(t) of transition t + 1; 1e6 Arm4 transitions: 0.45 GB hot + 0.11 GB cold).  The future achieved goal of a HER
 * row is the ag(t+1) block of transition future_t - 1; cur_layout_init places that block inside the step block so that
 * it straddles as few 64-byte atoms as possible (Arm4: one).  Sections are padded to multiples of 4 floats.
 * `change` / `info` / ag(t) are only read by the API-parity sampler, the store-time routing, relative goals and an
 * INFO reward rule; keeping them out of the hot rows keeps those free of dead bytes.
 * ------------------------------------------------------------------------------------------ */
typedef struct cur_layout {
  int32_t T;
  int32_t dimo, dimag, dimg, dimu, dimtd, dimchange, diminfo;
  int32_t off_g, off_u, off_td, off_ag, off_o; /* floats, inside the step block of a transition row; o last */
  int32_t row_stride;                          /* floats of the step block, multiple of 4 */
  int32_t off_change, off_info;                /* floats, inside a cold row */
  int32_t cold_stride;                         /* floats per cold row */
  int32_t trans_stride;                        /* floats per transition row: round_up16(round_up4(dimo) + row_stride) */
  int32_t off_agc;                             /* ag(t) inside a cold row */
} cur_layout;

/* Fills offsets/strides.  dimtd/dimchange/diminfo may be 0 (flat structure). */
int cur_layout_init(cur_layout* L, int T, int dimo, int dimag, int dimg, int dimu, int dimtd,
                    int dimchange, int diminfo);

/* ------------------------------------------------------------------------------------------
 * cur_store_episodes - ReplayBuffer.store_episode (replay_buffer.py:57-72) + the per-module
 * duplication of DDPG.store_episode (ddpg.py:187-197).  Packs `n_ep` episodes given as key-major
 * float32 device arrays ([n_ep,T+1,dimo], [n_ep,T+1,dimag], [n_ep,T,dim*]...) into transition rows and writes
 * copy i of episode copy_src[i] to slot copy_slot[i] of the buffer (copy_hot[i], copy_cold[i]).
 * Slot choice (_get_storage_idx, replay_buffer.py:90-109) stays on the host: it consumes the
 * caller's np.random stream.  copy_* are HOST arrays of length n_copies <= CUR_MAX_COPIES.
 * ------------------------------------------------------------------------------------------ */
typedef struct cur_episode_src {
  const float* o;      /* [n_ep, T+1, dimo]   */
  const float* ag;     /* [n_ep, T+1, dimag]  */
  const float* g;      /* [n_ep, T,   dimg]   */
  const float* u;      /* [n_ep, T,   dimu]   */
  const float* td;     /* [n_ep, T,   dimtd]     or NULL */
  const float* change; /* [n_ep, T,   dimchange] or NULL */
  const float* info;   /* [n_ep, T,   diminfo]   or NULL */
} cur_episode_src;

int cur_store_episodes(void* stream, const cur_layout* L, const cur_episode_src* src, int n_ep,
                       int n_copies, const int32_t* copy_src, float* const* copy_hot,
                       float* const* copy_cold /* entries may be NULL when cold_stride == 0 */,
                       const int64_t* copy_slot);

/* ------------------------------------------------------------------------------------------
 * cur_her_sample - ONE fused kernel for
 *   _sample_her_transitions           (her.py:20-66 flat, her.py:99-183 multi-task)
 *   + reward_fun / compute_reward     (config.py:158-159; restated rule, see DESIGN.md)
 *   + the per-buffer loop, concat and shuffle of DDPG.sample_batch (ddpg.py:325-345)
 *   + DDPG._preprocess_og             (ddpg.py:118-127, 350-353)
 * Row j of every output is concat-row c = perm ? perm[j] : j; concat rows are the segments'
 * `count`s laid end to end (buffer order).  Per concat row:
 *   draws (ep, t, u_her, u_off[, choice]) come from the injected arrays (bit-exact replay of the
 *   reference's np.random stream) or, when inj_ep == NULL, from Philox4x32-10 keyed by `seed` with
 *   counter (c, call_offset) - see DESIGN.md for the exact mapping;
 *   her = u_her < future_p;  future_t = t + 1 + (int)(u_off * (T - t))  in float64 (her.py:115-118);
 *   HER rows get g/task_descr relabelled per `mode` (her.py:129-164 / her.py:43-47);
 *   r is recomputed for every row from (ag_2, relabelled g, task_descr) (her.py:174-176).
 * Any output pointer may be NULL (not produced).  Outputs are float32 [batch, dim] row-major.
 * ------------------------------------------------------------------------------------------ */
enum {
  CUR_MODE_BUFFER = 0,       /* 'buffer' in task_replay: module = segment.task_to_replay, or the
                                row's own module when task_to_replay < 0      (her.py:131-136) */
  CUR_MODE_RANDOM_TASK = 1,  /* replay_random_task_transition                 (her.py:138-139) */
  CUR_MODE_CP_TASK = 2,      /* replay_cp_task_transition, p = cp_proba       (her.py:141-142) */
  CUR_MODE_CURRENT_TASK = 3, /* replay_current_task_transition                (her.py:158-164) */
  CUR_MODE_FLAT = 4          /* make_sample_her_transitions                   (her.py:43-47)   */
};

typedef struct cur_segment {
  const float* base;      /* transition rows of the buffer                                   */
  const float* cold;      /* cold rows (read for change / info / ag outputs, relative goals, INFO rewards) */
  int32_t n_episodes;     /* current_size: episodes are drawn from [0, n_episodes)            */
  int32_t count;          /* rows sampled from this buffer (proportions[i], ddpg.py:326-336)  */
  int32_t task_to_replay; /* module forced on HER rows, or -1 for None                        */
  int32_t _pad;
} cur_segment;

/* Reward rule of one module (config.py:158-159 hands the sampler gym_flowers' compute_reward; the rule arrives here as
 * DATA, one row of this table per module - SURVEY 8c).  All kinds yield r in {-1, 0}, evaluated in float64:
 *   DISTANCE  d = || ag_2[ag_idx[m]] - g[g_idx[m]] ||_2                       r = -1 if d > threshold[m] else 0
 *   PAIR      d = || (ag_2[ag_idx[m]] - ag_2[ref_idx[m]]) - g[g_idx[m]] ||_2  same compare: the goal is the wanted
 *             OFFSET between two achieved-goal sub-slices (one object placed relative to another, Stack-style)
 *   INFO      r = info[info_col[m]] - 1: the success flag stored with the transition passes through             */
enum { CUR_REWARD_DISTANCE = 0, CUR_REWARD_PAIR = 1, CUR_REWARD_INFO = 2 };

typedef struct cur_task_table {
  int32_t n_tasks;
  int32_t _pad;
  int32_t len[CUR_MAX_TASKS];        /* len(tasks_g_id[m])                                    */
  int16_t g_idx[CUR_MAX_TASKS][CUR_MAX_SLICE];  /* tasks_g_id[m][k]                           */
  int16_t ag_idx[CUR_MAX_TASKS][CUR_MAX_SLICE]; /* tasks_ag_id[m][k], truncated to len[m]     */
  int16_t ref_idx[CUR_MAX_TASKS][CUR_MAX_SLICE]; /* PAIR: second achieved-goal slice           */
  int32_t kind[CUR_MAX_TASKS];       /* CUR_REWARD_*                                          */
  int32_t info_col[CUR_MAX_TASKS];   /* INFO: column inside the concatenated info_* row       */
  double threshold[CUR_MAX_TASKS];   /* per module                                            */
  double flat_threshold;             /* task_descr = None (flat sampler, her.py:56-59): every module's difference
                                        vector enters ONE distance, compared with this           */
  double cdf[CUR_MAX_TASKS];         /* CP_TASK: normalised cumsum(cp_proba) (np.random.choice) */
} cur_task_table;

/* Device-resident control block for CUDA-graph replays: the values that change between launches are
 * read from memory instead of from the (frozen) kernel arguments.  `step` is the shared train-step
 * counter: the Philox counter of a launch is call_offset + *step; cur_ddpg_grads bumps it. */
typedef struct cur_her_dyn {
  const int64_t* step;                   /* device pointer                                    */
  int32_t n_episodes[CUR_MAX_SEGMENTS];  /* overrides seg[i].n_episodes                       */
  int32_t count[CUR_MAX_SEGMENTS];       /* overrides seg[i].count; must sum to batch         */
  double cdf[CUR_MAX_TASKS];             /* overrides tasks.cdf (CP_TASK mode)                */
} cur_her_dyn;

typedef struct cur_her_args {
  cur_layout L;
  cur_task_table tasks;
  int32_t mode;
  int32_t n_segments;
  cur_segment seg[CUR_MAX_SEGMENTS];
  int64_t batch;          /* total rows == sum of seg[i].count                                */
  double future_p;        /* 1 - 1/(1+k) or 0                            (her.py:86-89)       */
  /* injected draws, indexed by CONCAT row; all NULL => Philox */
  const int32_t* inj_ep;
  const int32_t* inj_t;
  const double* inj_u_her;
  const double* inj_u_off;
  const int32_t* inj_choice; /* resolved np.random.choice result per row, -1 if none; may be NULL */
  uint64_t seed;
  uint64_t call_offset;
  const int32_t* perm;    /* shuffle_inds (ddpg.py:338-345) or NULL                           */
  float clip_obs;         /* clip o,g,o_2,g_2 to +-clip_obs; <= 0 disables (raw sampler output) */
  int32_t relative_goals; /* g <- g - ag (g_2 <- g - ag_2) before clipping                    */
  float *o, *ag, *g, *u, *td, *change, *info, *o_2, *ag_2, *g_2, *r;
  int32_t* idx_out;       /* optional [batch,4]: ep, t, future_t (-1 if not HER), module (-1) */
  const cur_her_dyn* dyn; /* optional DEVICE control block (Philox mode only), see cur_her_dyn  */
} cur_her_args;

int cur_her_sample(void* stream, const cur_her_args* args);

/* Worker-major form of cur_her_sample: one launch samples the batches of n_workers reference workers, each from its own
 * buffers with its own random stream (the reference's MPI workers, train.py:221-243, hosted on one rank).  Concat row c
 * belongs to worker j = c / rows_per_worker, at local row i = c % rows_per_worker; the segment lookup runs over worker
 * j's own segments (w[j].seg: base, cold, task_to_replay; the counts and sizes the kernel reads are dyn[j]'s).
 *   Philox draws: key w[j].seed, counter (i, a->call_offset + (step ? *step : 0)) - the position a lone agent keyed
 *   w[j].seed draws its row i from at the same update.
 *   Injected draws (a->inj_*) and a->perm stay indexed by the concat row: the caller lays worker j's draws and its
 *   shuffle out in rows [j * rows_per_worker, (j + 1) * rows_per_worker).
 * Everything else (relabelling, reward table, clip, outputs, idx_out) is cur_her_sample's with a->batch ==
 * n_workers * rows_per_worker; a->seg, a->n_segments, a->seed and a->dyn are ignored.  `dyn` (DEVICE, n_workers entries)
 * and `step` (DEVICE or NULL) are read at run time, so a CUDA graph replays with frozen arguments.  w is a HOST array
 * whose seg[].count / seg[].n_episodes are checked here; refused before any launch: n_workers outside
 * 1..CUR_MAX_WORKERS, a worker with n_segments outside 1..CUR_MAX_SEGMENTS, counts of a worker that do not sum to
 * rows_per_worker, a->batch != n_workers * rows_per_worker. */
#define CUR_MAX_WORKERS 64
typedef struct cur_her_worker {
  uint64_t seed;                       /* Philox key of this worker's draws                         */
  int32_t n_segments;
  int32_t _pad;
  cur_segment seg[CUR_MAX_SEGMENTS];   /* the worker's buffers, in buffer order                      */
} cur_her_worker;
typedef struct cur_her_worker_dyn {
  int32_t n_episodes[CUR_MAX_SEGMENTS];
  int32_t count[CUR_MAX_SEGMENTS];     /* sums to rows_per_worker                                   */
  double cdf[CUR_MAX_TASKS];           /* CP_TASK mode: normalised cumsum(cp_proba)                  */
} cur_her_worker_dyn;
int cur_her_sample_workers(void* stream, const cur_her_args* a, int n_workers, int rows_per_worker,
                           const cur_her_worker* w, const cur_her_worker_dyn* dyn /* device */,
                           const int64_t* step /* device or NULL */);

/* The kernels' counter-based generator on its own: out[i] = Philox4x32-10(counter = in[i][0..3], key = in[i][4..5])
 * evaluated ON THE DEVICE by the same device function the sampling and exploration-noise kernels call (known-answer
 * tests against the Random123 vectors; the reference draws from np.random, her.py:108-116, which this mode replaces). */
int cur_philox4x32_10(void* stream, const uint32_t* in /* [n][6] device */, int64_t n, uint32_t* out /* [n][4] device */);

/* ------------------------------------------------------------------------------------------
 * Normalizer (baselines/her/normalizer.py:10-118).  State is float32 on the device.
 * ------------------------------------------------------------------------------------------ */
/* update(v): local_sum += v.sum(0); local_sumsq += (v*v).sum(0); local_count += n  (:64-70).
 * `partial` = [sum(dim) | sumsq(dim) | count(1)] float32. */
int cur_norm_accumulate(void* stream, const float* v, int64_t n, int dim, float* partial);
/* recompute_stats (:96-118, :50-61): running += partial / world   (partial already SUMMED over
 * ranks; `buf /= size`, :84-88); mean = sum/count; std = sqrt(max(eps^2, sumsq/count - mean^2));
 * partial <- 0.  `running` = [sum | sumsq | count] (count initialised to 1 by the caller, :37-39). */
int cur_norm_recompute(void* stream, float* running, float* partial, float world, float eps,
                       int dim, float* mean, float* std);
/* normalize(v) = clip((v-mean)/std, +-clip) (:72-77); denormalize (:79-82). In place allowed. */
int cur_norm_apply(void* stream, const float* v, int64_t n, int dim, const float* mean,
                   const float* std, float clip, float* out);
int cur_norm_invert(void* stream, const float* v, int64_t n, int dim, const float* mean,
                    const float* std, float* out);

/* ------------------------------------------------------------------------------------------
 * Flat-vector optimiser pieces (baselines/common/mpi_adam.py:21-35, ddpg.py:456-462).
 * ------------------------------------------------------------------------------------------ */
/* m = b1*m + (1-b1)*g; v = b2*v + (1-b2)*g*g; theta += neg_a*m/(sqrt(v)+eps).  Unfused IEEE
 * float32 operations in NumPy's order (bit-exact with the float32 NumPy evaluation).
 * neg_a = float32(-(stepsize*sqrt(1-b2^t)/(1-b1^t))) is computed by the caller in float64.
 * grad_div: divide the (already all-reduced) gradient by this first (scale_grad_by_procs,
 * mpi_adam.py:27-28); 1 = no division.  betas/eps are doubles so (1-beta) is rounded to float32
 * from the exact python value, as NumPy does. */
int cur_adam_step(void* stream, float* theta, const float* grad, float* m, float* v, int64_t n,
                  float neg_a, double beta1, double beta2, double eps, float grad_div);
/* Same, but CUDA-graph friendly: the step scale is read from a device table indexed by the shared
 * device train-step counter, which cur_ddpg_grads has ALREADY bumped for this step, so Adam's 1-based
 * t equals *step_counter and the scale is neg_a_table[min(t, table_len) - 1].  Beyond the table the
 * last entry is used (the bias correction is exactly 1 in float64 after ~4e4 steps). */
int cur_adam_step_graph(void* stream, float* theta, const float* grad, float* m, float* v,
                        int64_t n, const float* neg_a_table, int table_len,
                        const int64_t* step_counter, double beta1, double beta2, double eps,
                        float grad_div, int32_t step_div /* t = *step_counter / step_div; 1 normally */);
/* target = polyak*target + (1-polyak)*main (ddpg.py:461-462); polyak == 0 is the init copy. */
int cur_polyak(void* stream, float* target, const float* main_, int64_t n, double polyak);
/* Order-independent 64-bit checksum of a float32 vector (for check_synced, mpi_adam.py:42-50). */
int cur_checksum(void* stream, const float* x, int64_t n, uint64_t* out);

/* ------------------------------------------------------------------------------------------
 * Actor-critic networks (baselines/her/actor_critic.py:5-98, util.py:56-107) and the DDPG graph
 * (ddpg.py:412-449).  Parameters live in flat float32 vectors in GetFlat order
 * (util.py:49-53, tf_util.py:221-244):
 *    modular net:  W0s[in_s,H] b0[H] W0g[dimg,H] W1[H,H] b1[H] ... Wout[H,out] bout[out]
 *    flat net:     W0[in,H]    b0[H]             W1[H,H] b1[H] ... Wout[H,out] bout[out]
 * `theta` = [Q | pi] (ddpg.py:456), same for target, grads and Adam state.
 * ------------------------------------------------------------------------------------------ */
typedef struct cur_net_desc {
  int32_t modular;  /* 1: MultiTaskActorCritic / nn_modular_her; 0: ActorCritic / nn          */
  int32_t dimo, dimg, dimu, dimtd;
  int32_t hidden, layers; /* `layers` hidden layers of `hidden` units (+ the output layer)    */
  float max_u;
  int32_t normalize_obs;  /* apply o_stats/g_stats.normalize to o,g (actor_critic.py:31-36)   */
  float norm_clip;
} cur_net_desc;

int64_t cur_net_param_count(const cur_net_desc* d, int which /*0: Q, 1: pi*/);
/* Flat arena used by every theta-like vector (main, target, grads, Adam m/v):
 *   [ Q params | zero pad to a multiple of 4 floats | pi params | zero pad ]
 * so that both nets start 16-byte aligned and one elementwise launch / one all-reduce covers both.
 * Returns the float offset of the pi block; *total (optional) receives the arena length. */
int64_t cur_theta_pi_offset(const cur_net_desc* d, int64_t* total);
/* floats of scratch needed by cur_ddpg_grads / cur_ddpg_actions for `batch` rows; the caller zero-initialises it
 * once (it holds a self-resetting completion ticket of the multi-CTA loss kernel) */
int64_t cur_ddpg_workspace_floats(const cur_net_desc* d, int64_t batch);

typedef struct cur_norm_stats {
  const float *o_mean, *o_std, *g_mean, *g_std; /* may be NULL when normalize_obs == 0 */
} cur_norm_stats;

/* get_actions forward (ddpg.py:129-146) including _preprocess_og (ddpg.py:118-127):
 * g <- g - ag if `ag` != NULL (relative goals); o,g clipped to +-clip_obs (if > 0); optional
 * normalisation; pi = max_u*tanh(net(o,g,td)) and optionally Q(o,g,td,pi).
 * The host-side exploration noise / eps-greedy (ddpg.py:148-152) stays with the caller's RNG. */
int cur_ddpg_actions(void* stream, const cur_net_desc* d, const float* theta,
                     const cur_norm_stats* stats, const float* o, const float* ag /* or NULL */,
                     const float* g, const float* td, int64_t n, float clip_obs, float* workspace,
                     float* out_pi, float* out_q /* or NULL */);

/* The same forward as ONE launch for the rollout's per-step call (rollout.py:217,226: n = rollout_batch_size rows, 50
 * calls per episode; hidden 64, 128 or 256, see cur_ddpg_rows_supported): one CTA per 4 rows streams the net through
 * shared memory.
 * Every data pointer may address MAPPED PINNED HOST memory (cur_host_alloc) - inputs are then read and actions written
 * over PCIe by the kernel itself.  seq == 0: out_pi / out_q are float32 arrays.  seq != 0: they are arrays of 8-byte words
 * {float32 bits | seq << 32}; an aligned 64-bit store is single-copy atomic, so a caller that owns the (host-visible)
 * buffer polls the words for its call number instead of issuing copies and a stream synchronisation.  n <= 4096. */
int cur_ddpg_actions_rows(void* stream, const cur_net_desc* d, const float* theta, const cur_norm_stats* stats,
                          const float* o, const float* ag /* or NULL */, const float* g, const float* td, int64_t n,
                          float clip_obs, void* out_pi, void* out_q /* or NULL */, uint32_t seq);
/* The routed form of cur_ddpg_actions_rows for a task-experts evaluation step: row i is acted on by
 * experts[row_expert[i]] (its main or target theta and its normaliser statistics), all experts of one shape `d`.  One
 * launch: the rows of each expert fill whole 4-row CTA tiles, and every output lands at the row's original position, in
 * the same two forms (seq == 0: float32; seq != 0: {float32 bits | seq << 32} words for cur_actions_finish_host).
 * row_expert is a HOST array of n entries; the other pointers follow cur_ddpg_actions_rows.  Refused before any launch:
 * n_experts outside 1..CUR_MAX_TASKS, a row_expert entry outside 0..n_experts-1, a shape cur_ddpg_rows_supported(d, 4)
 * refuses, n outside 1..CUR_ACTIONS_GROUP_MAX_ROWS. */
#define CUR_ACTIONS_GROUP_MAX_ROWS 512
typedef struct cur_actions_expert {
  const float* theta;
  cur_norm_stats stats;            /* may hold NULLs when normalize_obs == 0 */
} cur_actions_expert;
int cur_ddpg_actions_rows_group(void* stream, const cur_net_desc* d, int n_experts, const cur_actions_expert* experts,
                                const int32_t* row_expert, const float* o, const float* ag /* or NULL */, const float* g,
                                const float* td, int64_t n, float clip_obs, void* out_pi, void* out_q /* or NULL */,
                                uint32_t seq);
/* Host-side tail of a seq != 0 call of cur_ddpg_actions_rows (ddpg.py:147-155): polls the n * dimu (+ n with_q) output
 * words in the mapped buffer until all carry `seq`, then applies the reference's exploration post-processing with the
 * caller's np.random draws (randn [n, dimu] float64, explore [n] int64 = binomial(1, random_eps), u_rand [n, dimu] float64 =
 * uniform(-max_u, max_u); all three NULL: no post-processing, e.g. device-side noise) in NumPy's own evaluation types:
 *   u = (float)((double)u + noise_scale * randn); u = clip(u, +-(float)max_u); u = (float)((double)u + explore * (u_rand - u))
 * with noise_scale = noise_eps * max_u.  Writes float32 u_out [n, dimu] and q_out [n].  CUR_ERR_UNSUPPORTED: the words did
 * not arrive within max_spins polls (synchronise the stream so that a launch failure surfaces, then call again).
 * Pure host code: no CUDA call, no device work. */
int cur_actions_finish_host(const void* out_words, int64_t n, int dimu, int with_q, uint32_t seq, const double* randn,
                            const int64_t* explore, const double* u_rand, double noise_scale, double max_u, float* u_out,
                            float* q_out /* or NULL */, int64_t max_spins);
/* cudaHostAlloc(mapped | portable): *host_ptr for the CPU, *dev_ptr for the kernels; zero-filled. */
int cur_host_alloc(int64_t bytes, void** host_ptr, void** dev_ptr);
int cur_host_free(void* host_ptr);
/* cudaMemcpyAsync(host -> device) on `stream`; `src` from cur_host_alloc */
int cur_copy_h2d(void* stream, void* dst, const void* src, int64_t bytes);

/* Device-side option for the exploration noise of get_actions (ddpg.py:147-152; SURVEY 8f row 1), in place on
 * u [n, dimu] (the out_pi of cur_ddpg_actions): Gaussian noise noise_eps * max_u * N(0,1), clip to +-max_u, then with
 * probability random_eps per row the action is replaced by a uniform one in [-max_u, max_u].  Draws are Philox4x32-10
 * blocks keyed by `seed`, counter (row, component pair, call) - the caller passes a fresh `call` per get_actions.
 * The default path keeps the noise on the host (the caller's np.random stream, like the reference). */
int cur_action_noise(void* stream, float* u, int64_t n, int dimu, float max_u, double noise_eps,
                     double random_eps, uint64_t seed, uint64_t call);
/* The same noise with per-row keys: row r gets what the one-row call cur_action_noise(u + r * dimu, 1, ..., seed[r],
 * call[r]) would give it (counter row 0).  seed / call: n entries each, readable by the device (device memory or
 * mapped pinned host memory).  Stands for a loop of one-row get_actions calls of different agents. */
int cur_action_noise_rows(void* stream, float* u, int64_t n, int dimu, float max_u, double noise_eps,
                          double random_eps, const uint64_t* seed, const uint64_t* call);

typedef struct cur_batch {
  const float *o, *g, *u, *td, *o_2, *g_2, *r; /* staged batch (ddpg.py:75-83); td NULL if flat */
  int64_t n;
} cur_batch;

typedef struct cur_ddpg_hyper {
  float gamma, clip_return, action_l2;
  int32_t clip_pos_returns;
  /* CUDA-graph replays (both optional): when step_counter != NULL the loss kernel writes q_loss /
   * pi_loss to slot (*step_counter % loss_ring) of the arrays passed to cur_ddpg_grads and then
   * increments *step_counter (after the HER kernel of this step read it, before Adam reads it). */
  int64_t* step_counter;
  int32_t loss_ring;
  /* rows schedule only, > 1 (requires step_counter): the update is the SUM of `micro_batches` consecutive launches'
   * gradients - several reference workers (each a batch of 256 with its own loss mean, ddpg.py:439-441) on one rank,
   * SURVEY 8e "19-worker-equivalent".  The device counter then counts launches: launch j = counter % micro_batches
   * overwrites the gradient for j == 0 and adds to it otherwise; consumers derive the update number as
   * counter / micro_batches (step_div of cur_adam_step_graph / cur_p2p_ctx). */
  int32_t micro_batches;
  /* rows schedule only: when > 0 (requires step_counter) the gradient of update s is written to
   * grads + (s & 1) * grads_parity_stride floats, s = update number (counter / micro_batches) after this update's bump
   * (double buffering for cur_p2p_allreduce_adam).  0: always `grads`. */
  int64_t grads_parity_stride;
  /* > 0: the batch holds batch / loss_rows reference workers (SURVEY 8e) - the backward seeds
   * are scaled by 1 / loss_rows instead of 1 / batch, so that the gradient is the SUM of the workers' single-batch
   * gradients (each loss a mean over loss_rows rows, ddpg.py:439-441 + the SUM all-reduce of ddpg.py:452-453).  The
   * reported losses stay means over the whole batch (= the average worker's loss).  0: loss_rows = batch. */
  int64_t loss_rows;
  /* rows schedule, without the fused optimiser: 1 = the transposed hidden-layer weights in the workspace are current
   * (maintained by cur_p2p_allreduce_adam_t or cur_ddpg_rows_refresh), the transpose launch is skipped. */
  int32_t transposes_valid;
  int32_t _pad;
} cur_ddpg_hyper;

/* DDPG._grads (ddpg.py:235-243): writes grads = [Q_grad | pi_grad] (flat), Q_loss (1 float),
 * pi_loss (1 float) and main.Q_pi [n,1]. */
int cur_ddpg_grads(void* stream, const cur_net_desc* d, const float* theta_main,
                   const float* theta_target, const cur_norm_stats* stats, const cur_batch* batch,
                   const cur_ddpg_hyper* h, float* workspace, float* grads, float* q_loss,
                   float* pi_loss, float* q_pi);

/* structure='task_experts' (train.py:287-289: one DDPG per module, all of the same shape): DDPG._grads of
 * n_experts agents as ONE sequence of grouped launches - every dependency level of the graph covers the
 * problems of all experts (FFMA grouped GEMM at batch 256, tcgen05 batch at batch >= 1024).  Semantically
 * `for p in policies: p._grads()`; each expert keeps its own parameters, batch, losses and workspace
 * (cur_ddpg_workspace_floats(d, batch) floats each). */
typedef struct cur_ddpg_expert {
  const float* theta_main;
  const float* theta_target;
  cur_norm_stats stats;
  int32_t has_stats;
  int32_t _pad;
  cur_batch batch;
  cur_ddpg_hyper hyper;
  float* workspace;
  float* grads;
  float* q_loss;
  float* pi_loss;
  float* q_pi;
} cur_ddpg_expert;
int cur_ddpg_grads_group(void* stream, const cur_net_desc* d, int n_experts, const cur_ddpg_expert* experts);


/* ------------------------------------------------------------------------------------------
 * "Rows" schedule of the same update (csrc/ddpg_rows.cu): DDPG._grads (ddpg.py:235-243) and,
 * optionally, both MpiAdam.update calls of DDPG._update (ddpg.py:246-248, mpi_adam.py:30-35) in
 * TWO launches: a thread-block-cluster kernel that runs the whole forward / backward data path for
 * 16-row groups of the batch, then one grouped weight-gradient GEMM over the full batch that
 * applies Adam in its epilogue.  Supported shapes: hidden 64, 128 or 256 (the kernels are instantiated
 * for each; the optional CTA-pair form is 256 only), layers <= 4, dimu <= 8, first-layer fan-in <= 256
 * whatever the hidden width, batch a multiple of 4 up to 1024 (cur_ddpg_rows_supported); anything else
 * uses cur_ddpg_grads.  Same outputs as cur_ddpg_grads.
 *
 * `workspace` must be ZERO-INITIALISED once by the caller (it holds a completion ticket).
 * With h->step_counter != NULL the losses go to slot (*step_counter % loss_ring) and the counter is
 * incremented at the end of the second launch.  With `adam` != NULL (requires step_counter) the
 * parameters theta_main and the moments are stepped in place with
 * neg_a_table[min(*step_counter + 1, table_len) - 1]; use it only when no gradient all-reduce is
 * needed between _grads and _update (world size 1) and both nets share the step size.
 * With `her` != NULL the batch is not read from `batch` (only batch->n is used): every CTA draws,
 * gathers and relabels its own rows in the kernel prologue with the code of cur_her_sample (same
 * Philox counters / injected draws / control block, bit-identical transitions); output pointers
 * inside `her` are ignored.
 * ------------------------------------------------------------------------------------------ */
/* Tile-level gradient exchange INSIDE the weight-gradient launch (csrc/ddpg_rows.cu, several ranks; replaces the
 * Allreduce(SUM) of mpi_adam.py:24-28 between _grads and _update, scale_grad_by_procs=False).  Every rank runs the same
 * tile grid; as soon as a CTA has its tile of dW it pushes the tile to the rank(s) that reduce it with "LL" stores over
 * NVLink peer memory - each element travels as one 8-byte {float32 bits, update number} word, so the receiver polls the
 * data words themselves and no flag round / memory fence sits on the critical path.  The reducer adds the world's tiles in
 * rank order (bit-identical on every reducer), applies Adam in the same epilogue and keeps W^T current, exactly like
 * the one-rank launch.
 *   mode 0  every rank reduces every tile: partials are pushed to ALL peers (one NVLink hop; (W-1) x arena x 8 bytes
 *           out per rank and update) and every rank keeps the full Adam state - best for 2 ranks;
 *   mode 1  tile t is reduced by rank t % world, which pushes the stepped parameters back to all peers (two hops,
 *           2 x (W-1)/W x arena x 8 bytes out per rank); Adam moments exist only on the owner of an element
 *           (cur_ddpg_rows_owner_map tells which) - best for 4..8 ranks;
 *   mode 2  NVLS: as mode 1, but the owner reads the tile with multimem.ld_reduce - the NVSwitch adds the world's partials
 *           (each rank keeps its partial in its OWN slots, {value, update number as float}: the number half of the reduced
 *           word equals world x number once every rank's pair has landed) - and publishes the stepped parameters with ONE
 *           store to the multicast mapping (mc_region).  (W-1)/W x arena x 8 bytes in, arena / W x 8 bytes out per rank
 *           instead of 2 x (W-1)/W x arena x 8 each way; the order of the in-switch summation is the hardware's, so the
 *           parameters are identical on every rank but not bit-equal to the rank-ordered sum of modes 0 / 1.
 * Region of a rank (zero-initialised): modes 0 / 1 (cur_p2p_alloc / cur_p2p_open, cur_xchg_region_bytes bytes)
 *   [ partial slots: world x arena x 8 bytes, block s written by rank s | result slots: arena x 8 bytes ]
 * mode 2 (symmetric memory with a multicast mapping)
 *   [ partial slots: arena x 8 bytes, written by the rank itself | result slots: arena x 8 bytes ]
 * The update number travelling with the data is (device step counter / micro_batches) + 1; it never repeats as long
 * as the counter only grows (zero the regions collectively before moving the counter backwards).  A rank that waits
 * longer than ~20 s for a peer sets *error_flag (if given) and traps. */
typedef struct cur_xchg_ctx {
  int32_t rank, world;
  int32_t mode;
  int32_t _pad;
  void* region[CUR_MAX_RANKS]; /* region[r] as mapped in this process; region[rank] is the local one */
  int64_t arena;               /* floats of the gradient / parameter arena */
  int64_t* timeline;           /* optional DEVICE buffer [tiles][4] of %globaltimer stamps (ns): CTA start, tile computed and
                                  pushed, reduced tile available (partials landed / result landed), CTA end */
  int32_t* error_flag;         /* optional device int */
  void* mc_region;             /* mode 2: the multicast (NVLS) mapping of the regions - one symmetric allocation, e.g.
                                  torch.distributed._symmetric_memory (rendezvous(...).multicast_ptr); NULL otherwise */
} cur_xchg_ctx;
int64_t cur_xchg_region_bytes(int64_t arena_floats, int world);

typedef struct cur_adam_fused {
  float *m, *v;               /* Adam moments, same arena layout as theta */
  const float* neg_a_table;   /* float32(-a_t), t = 1..table_len (see cur_adam_step_graph) */
  int32_t table_len;
  /* 1: the transposed hidden-layer weights in `workspace` are current (the previous call on this workspace was a
   * fused-Adam call, whose epilogue writes them next to the stepped weights, or cur_ddpg_rows_refresh ran after the
   * last outside change of theta_main) - the transpose launch is skipped.  0: re-transpose first. */
  int32_t transposes_valid;
  double beta1, beta2, eps;
  const cur_xchg_ctx* xchg;   /* several ranks: exchange the gradient tiles before the step (see cur_xchg_ctx); NULL: one rank */
} cur_adam_fused;

int cur_ddpg_rows_supported(const cur_net_desc* d, int64_t batch);
/* (Re)build the transposed hidden-layer weights of main.Q / main.pi in a rows-schedule workspace (see
 * cur_adam_fused.transposes_valid). */
int cur_ddpg_rows_refresh(void* stream, const cur_net_desc* d, const float* theta_main, float* workspace,
                          int64_t batch);
int64_t cur_ddpg_rows_workspace_floats(const cur_net_desc* d, int64_t batch);
/* Which rank reduces (and holds the Adam moments of) every element of the arena under cur_xchg_ctx mode 1: writes
 * owner[arena] (HOST int32; -1 for padding) for the tile plan of this net / batch. */
int cur_ddpg_rows_owner_map(const cur_net_desc* d, int64_t batch, int world, int32_t* owner /* host */);
int cur_ddpg_rows_step(void* stream, const cur_net_desc* d, float* theta_main,
                       const float* theta_target, const cur_norm_stats* stats,
                       const cur_batch* batch, const cur_ddpg_hyper* h, float* workspace,
                       float* grads, float* q_loss, float* pi_loss, float* q_pi,
                       const cur_adam_fused* adam /* or NULL: gradients only */,
                       const cur_her_args* her /* or NULL: read `batch` */);

/* ------------------------------------------------------------------------------------------
 * Data-parallel gradient exchange over NVLink peer memory, fused with Adam (csrc/p2p.cu).
 * Replaces MpiAdam.update's Allreduce(SUM) + Adam (mpi_adam.py:24-35, scale_grad_by_procs=False)
 * on the CUDA-graph path: no host involvement, no NCCL, bit-identical parameters on every rank.
 *
 * Every rank allocates a region with cur_p2p_alloc (cudaMalloc + cudaIpcGetMemHandle, zeroed),
 * sends the 64-byte handle to its peers (any transport; curious_b200/parallel.py uses
 * torch.distributed all_gather_object) and maps theirs with cur_p2p_open.  Region layout:
 *   [ 256 bytes of flags | gradient arena buffer 0 | gradient arena buffer 1 | parameter staging ]   (arena floats each)
 * The gradient of update s (s = value of the device step counter AFTER the weight-gradient launch
 * bumped it) must be in buffer (s & 1) of the rank's own region; cur_ddpg_rows_step does that when
 * h->grads_parity_stride = arena and `grads` points at buffer 0.  cur_p2p_allreduce_adam then
 * signals the peers, waits for them, sums the world's gradients in rank order out of peer memory
 * and steps theta / m / v (same arithmetic as cur_adam_step_graph).
 * ------------------------------------------------------------------------------------------ */
typedef struct cur_p2p_ctx {
  int32_t rank, world;
  void* region[CUR_MAX_RANKS]; /* region[r] as mapped in this process; region[rank] is the local one */
  int64_t arena;               /* floats per gradient buffer, multiple of 4 */
  int32_t step_div;            /* update number = *step_counter / step_div (cur_ddpg_hyper.micro_batches); 0 or 1: none */
  int32_t _pad;
} cur_p2p_ctx;

int64_t cur_p2p_region_bytes(int64_t arena_floats);
int cur_p2p_alloc(int64_t bytes, void** ptr, unsigned char* handle64);
int cur_p2p_open(const unsigned char* handle64, void** ptr);
int cur_p2p_close(void* ptr);
int cur_p2p_free(void* ptr);
int cur_p2p_zero(void* stream, void* ptr, int64_t bytes); /* cudaMemsetAsync(0) of (a part of) an own region */
int cur_p2p_allreduce_adam(void* stream, const cur_p2p_ctx* ctx, float* theta, float* m, float* v,
                           const float* neg_a_table, int table_len, const int64_t* step_counter,
                           double beta1, double beta2, double eps, int32_t* error_flag /* or NULL */);
/* Same, and for up to CUR_P2P_MAX_TRANSPOSES H x H blocks of the arena (hidden-layer kernels) the stepped values are
 * also written transposed to dst[b] - the backward operands W^T that the rows schedule would otherwise rebuild with a
 * transpose launch at the start of every update (cur_ddpg_hyper.transposes_valid). */
#define CUR_P2P_MAX_TRANSPOSES 8
typedef struct cur_p2p_transposes {
  int32_t n, H;
  int64_t begin[CUR_P2P_MAX_TRANSPOSES];   /* float offset of the block inside the arena, multiple of 4 */
  float* dst[CUR_P2P_MAX_TRANSPOSES];      /* H x H floats each */
} cur_p2p_transposes;
int cur_p2p_allreduce_adam_t(void* stream, const cur_p2p_ctx* ctx, float* theta, float* m, float* v,
                             const float* neg_a_table, int table_len, const int64_t* step_counter,
                             double beta1, double beta2, double eps, int32_t* error_flag /* or NULL */,
                             const cur_p2p_transposes* transposes /* or NULL */);
/* The table for this rank's rows-schedule workspace (hidden-layer blocks of main.Q / main.pi -> their W^T buffers). */
int cur_ddpg_rows_transposes(const cur_net_desc* d, float* workspace, int64_t batch, cur_p2p_transposes* out);
/* Sharded form of the same step (reduce-scatter by peer loads, Adam on the rank's own slice of the arena,
 * all-gather by peer stores into the staging arenas, second flag round, local copy): (W-1)/W of one arena
 * in each direction per rank instead of W-1 arenas of loads.  Same result on every rank, bit-identical to
 * cur_p2p_allreduce_adam; m / v are only maintained for the rank's own slice. */
int cur_p2p_sharded_adam(void* stream, const cur_p2p_ctx* ctx, float* theta, float* m, float* v,
                         const float* neg_a_table, int table_len, const int64_t* step_counter,
                         double beta1, double beta2, double eps, int32_t* error_flag /* or NULL */);

/* ------------------------------------------------------------------------------------------
 * Tensor-core layer GEMM for large batches (csrc/tc_gemm.cu): tcgen05 (kind::tf32) with TMEM
 * accumulators, TMA operand staging and error-compensated 3xTF32 operands (fp32-level accuracy).
 * The dense layers of util.py:56-107 and their gradients (ddpg.py:443-449) at batch >= 1024 -
 * cur_ddpg_grads routes its hidden-layer problems here; this entry point exposes one problem:
 *   C[M,N] = epi( opA(A)[M,K] * opB(B)[K,N] + bias[N] )
 *   a_trans: A is stored [K][M] (lda >= M);  b_trans: B is stored [N][K] (ldb >= K)
 *   epilogue: 0 none, 1 ReLU, 2 gate by aux[M][N] > 0 (ReLU backward)
 * Shape: N == 256, any M and K (tiles of 128 x 256 x 32; tails are zero-filled by the TMA unit);
 * 16-byte aligned pointers, leading dimensions % 4.  a_trans with M < 1024 splits K over CTAs (weight
 * gradients, K = batch): `workspace` must then hold cur_tc_gemm_workspace_floats(M, N, K, a_trans)
 * floats, C must be contiguous (ldc == N) and bias / epilogue must be unset.
 * ------------------------------------------------------------------------------------------ */
int cur_tc_gemm_supported(int64_t M, int64_t N, int64_t K);
/* debug: CTA 0 of every following tensor-core launch writes clock64() stamps of its warp roles into
 * device_buffer_128 (128 x int64); NULL switches it off */
int cur_tc_gemm_timeline(long long* device_buffer_128);
/* cur_ddpg_grads runs its layer GEMMs on the tensor cores when batch >= 1024, batch % 128 == 0 and
 * hidden == 256.  mode: -1 default (on unless the environment says CUR_DDPG_TC=0), 0 FFMA only,
 * 1 tensor cores for every eligible shape (batch >= 256, batch % 128 == 0, hidden == 256). */
int cur_ddpg_set_tensor_cores(int mode);
int cur_ddpg_uses_tensor_cores(const cur_net_desc* d, int64_t batch);
/* Large batches (a multiple of 128 rows, hidden 256, 2-4 hidden layers) with the tensor cores on: forward nets, losses
 * and the data-gradient chains run as ONE launch - a CTA per 128-row tile and chain (csrc/tc_chain.cu) - followed by the
 * split-K weight-gradient GEMMs.  mode -1: default (on; CUR_DDPG_CHAIN=0 turns it off), 0: level-by-level schedule, 1: on. */
int cur_ddpg_set_chain(int mode);
int cur_ddpg_uses_chain(const cur_net_desc* d, int64_t batch);
/* The same chain schedule at the net's own hidden width: DDPG._grads (ddpg.py:235-243: actor_critic.py:5-98 and
 * util.py:56-107 forward, ddpg.py:412-449 losses and gradients) for hidden 64 or 128 without zero-padding to 256.
 * cur_ddpg_uses_chain stays 0 for those nets and cur_ddpg_grads keeps the level-by-level schedule for them.
 * cur_ddpg_chain_supported: 1 when cur_ddpg_chain_grads takes the desc and batch - hidden 64 or 128 (and the chain is on,
 * cur_ddpg_set_chain), a batch that is a multiple of 128, dimu <= 4, 2-4 hidden layers; for hidden 256 the answer of
 * cur_ddpg_uses_chain.  cur_ddpg_chain_grads: the arguments and outputs of cur_ddpg_grads, with a workspace of
 * cur_ddpg_chain_workspace_floats(d, batch) floats; the weight gradients of a narrow net run as K-sliced FFMA GEMMs. */
int cur_ddpg_chain_supported(const cur_net_desc* d, int64_t batch);
int64_t cur_ddpg_chain_workspace_floats(const cur_net_desc* d, int64_t batch);
int cur_ddpg_chain_grads(void* stream, const cur_net_desc* d, const float* theta_main,
                         const float* theta_target, const cur_norm_stats* stats, const cur_batch* batch,
                         const cur_ddpg_hyper* h, float* workspace, float* grads, float* q_loss,
                         float* pi_loss, float* q_pi);
/* cur_ddpg_grads_group on the narrow chain: n_experts (1..CUR_MAX_TASKS) agents of hidden 64 or 128 and one batch size
 * that cur_ddpg_chain_supported takes, each with a workspace of cur_ddpg_chain_workspace_floats(d, batch) floats.  The
 * experts' chain kernels run side by side, their K-sliced weight-gradient GEMMs share grouped launches; every expert gets
 * the bits cur_ddpg_chain_grads gives it alone.  Hidden 256, a shape the chain does not take and differing batch sizes
 * are refused before anything is launched. */
int cur_ddpg_chain_grads_group(void* stream, const cur_net_desc* d, int n_experts, const cur_ddpg_expert* experts);
/* debug: after updates run with CUR_ROWS_TIMELINE=1 (rows schedule, CUDA graph or not), print to stderr the %globaltimer
 * span of the two launches of the last updates and the gaps between them */
int cur_rows_timeline_dump(void);
/* debug: in-kernel clock64 timeline of the chain kernel's first actor / critic CTA (1024 x int64 device buffer, or NULL) */
int cur_tc_chain_timeline(long long* device_buffer_1024);
int64_t cur_tc_gemm_workspace_floats(int64_t M, int64_t N, int64_t K, int a_trans);
int cur_tc_gemm(void* stream, const float* A, int64_t lda, int a_trans, const float* B, int64_t ldb,
                int b_trans, float* C, int64_t ldc, int64_t M, int64_t N, int64_t K, const float* bias,
                const float* aux, int64_t ldaux, int epilogue, float* workspace);

#ifdef __cplusplus
}
#endif
#endif /* CURIOUS_B200_H */
