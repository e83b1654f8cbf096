"""HER samplers - drop-in for reference baselines/her/her.py.

    make_sample_her_transitions(goal_replay, her_replay_k, reward_fun, task_replay='', ...)   her.py:5
    make_sample_multi_task_her_transitions(goal_replay, her_replay_k, task_replay, reward_fun, ...)  her.py:72

Both return a callable `f(episode_batch, batch_size_in_transitions, task_to_replay=None,
cp_proba=None) -> {key: array[batch, dim]}` exactly like the reference closures, but the work is
done by ONE fused CUDA kernel (cur_her_sample in csrc/her.cu): index draws, gather, goal/task
relabel, reward.  `episode_batch` is either the device view a curious_b200 ReplayBuffer hands over or
a dict of host arrays (the DDPG.store_episode normaliser path, ddpg.py:209-215), which is uploaded
and packed first.

RNG modes (attribute `rng`):
  'numpy'  (default) the four draws of her.py:108-116 (and the np.random.choice draws of
           her.py:139,142) are made on the host from the global np.random stream in the reference's
           order and injected into the kernel: same seed => bit-identical output to the reference.
  'philox' the kernel draws with counter-based Philox4x32-10 (no host RNG, no H2D traffic).
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from .reward import as_reward_spec

OUT_KEYS = ('o', 'ag', 'g', 'u', 'td', 'change', 'info', 'o_2', 'ag_2', 'g_2', 'r')


class DeviceEpisodes:
    """What ReplayBuffer.sample passes to the sampler instead of the reference's dict of views
    (replay_buffer.py:44-48): the packed device buffer and how many episodes are valid."""

    def __init__(self, storage, cold, n_episodes, layout, info_keys, has_td, has_change):
        self.storage, self.cold, self.n_episodes, self.layout = storage, cold, n_episodes, layout
        self.info_keys, self.has_td, self.has_change = info_keys, has_td, has_change


def future_probability(goal_replay, her_replay_k):
    return 1 - (1. / (1 + her_replay_k)) if goal_replay == 'her' else 0      # her.py:86-89


def mode_of(task_replay, flat):
    if flat:
        return _lib.MODE_FLAT
    if 'buffer' in task_replay or task_replay == 'hand_designed':               # her.py:94
        return _lib.MODE_BUFFER
    if task_replay == 'replay_random_task_transition':
        return _lib.MODE_RANDOM_TASK
    if task_replay == 'replay_cp_task_transition':
        return _lib.MODE_CP_TASK
    if task_replay == 'replay_current_task_transition':
        return _lib.MODE_CURRENT_TASK
    raise ValueError("task_replay %r selects no module for HER rows (the reference raises "
                     "UnboundLocalError at her.py:144)" % (task_replay,))


class HostDraws:
    """The reference's np.random draws for one sampler call, made on the host in reference order."""

    def __init__(self, E, T, B):
        self.ep = np.random.randint(0, E, B)                 # her.py:108
        self.t = np.random.randint(T, size=B)                # her.py:109
        self.u_her = np.random.uniform(size=B)               # her.py:115
        self.u_off = np.random.uniform(size=B)               # her.py:116
        self.choice = None

    def draw_choices(self, mode, future_p, nb_tasks, cp_proba):
        """np.random.choice once per HER row, in row order (her.py:129-142)."""
        if mode not in (_lib.MODE_RANDOM_TASK, _lib.MODE_CP_TASK):
            return
        B = self.ep.shape[0]
        self.choice = np.full(B, -1, np.int32)
        for row in np.where(self.u_her < future_p)[0]:
            if mode == _lib.MODE_RANDOM_TASK:
                self.choice[row] = np.random.choice(range(nb_tasks))
            else:
                self.choice[row] = np.random.choice(range(nb_tasks), p=cp_proba)


def upload_draws(draws_list, device):
    """Concatenate per-segment draws and upload as one blob.  Returns dict of device tensors."""
    ep = np.concatenate([d.ep for d in draws_list]).astype(np.int32)
    t = np.concatenate([d.t for d in draws_list]).astype(np.int32)
    uh = np.concatenate([d.u_her for d in draws_list]).astype(np.float64)
    uo = np.concatenate([d.u_off for d in draws_list]).astype(np.float64)
    B = ep.shape[0]
    has_choice = any(d.choice is not None for d in draws_list)
    n64 = 2 * B
    n32 = 2 * B + (B if has_choice else 0)
    blob = torch.empty(n64 * 8 + n32 * 4, dtype=torch.uint8, pin_memory=True)
    hb = blob.numpy()
    hb[:8 * B].view(np.float64)[:] = uh
    hb[8 * B:16 * B].view(np.float64)[:] = uo
    i32 = hb[16 * B:].view(np.int32)
    i32[:B] = ep
    i32[B:2 * B] = t
    if has_choice:
        i32[2 * B:3 * B] = np.concatenate(
            [d.choice if d.choice is not None else np.full(d.ep.shape[0], -1, np.int32) for d in draws_list])
    dev = blob.to(device, non_blocking=True)
    out = dict(u_her=dev[:8 * B], u_off=dev[8 * B:16 * B], ep=dev[16 * B:20 * B], t=dev[20 * B:24 * B],
               choice=dev[24 * B:28 * B] if has_choice else None, _keep=(blob, dev))
    return out


class HerSampler:
    """The callable returned by make_sample_*_her_transitions."""

    def __init__(self, goal_replay, her_replay_k, task_replay, reward_fun, tasks_ag_id, tasks_g_id, flat):
        self.goal_replay, self.her_replay_k, self.task_replay = goal_replay, her_replay_k, task_replay
        self.flat = flat
        self.future_p = future_probability(goal_replay, her_replay_k)
        self.tasks_ag_id, self.tasks_g_id = tasks_ag_id, tasks_g_id
        self.nb_tasks = len(tasks_ag_id) if tasks_ag_id is not None else 0
        self.reward = as_reward_spec(reward_fun, tasks_ag_id, tasks_g_id)
        self.mode = mode_of(task_replay, flat) if (flat or task_replay != '') else None
        self.task_table = self.reward.task_table()
        self._info_layout = None        # 'info' reward rules: columns resolved against the first buffer sampled
        self.rng = 'numpy'
        self.seed = 0
        self.calls = 0
        self.out_dtype = np.float64     # the reference returns the buffers' float64 (replay_buffer.py:23)
        self.device = None

    # ---- low level: any number of segments, device tensors out ------------------------------------
    def sample_device(self, segments, B, *, cp_proba=None, draws=None, perm=None, clip_obs=0.0,
                      relative_goals=False, want=('o', 'ag', 'g', 'u', 'td', 'change', 'info', 'o_2',
                                                  'ag_2', 'r'),
                      want_idx=False, out=None, stream=None, dyn=None, call_offset=None, args_only=False):
        """segments: list of (DeviceEpisodes, count, task_to_replay or None).
        Returns {key: float32 cuda tensor [B, dim]} (+ 'idx' int32 [B,4] if want_idx)."""
        if self.mode is None:
            mode_of(self.task_replay, self.flat)
        lib = _lib.load()
        first = segments[0][0]
        a = _lib.HerArgs()
        a.n_segments = len(segments)
        if len(segments) > _lib.CUR_MAX_SEGMENTS:
            raise ValueError('too many buffers in one sample call')
        total = 0
        for i, (epi, count, ttr) in enumerate(segments):
            if count > 0 and epi.n_episodes <= 0:
                raise AssertionError('sampling from an empty buffer')      # replay_buffer.py:43
            a.seg[i].base = epi.storage.data_ptr()
            a.seg[i].cold = None if epi.cold is None else epi.cold.data_ptr()
            a.seg[i].n_episodes = int(epi.n_episodes)
            a.seg[i].count = int(count)
            a.seg[i].task_to_replay = -1 if ttr is None else int(ttr)
            total += int(count)
        assert dyn is not None or total == B                                 # ddpg.py:323
        a.dyn = dyn
        a.seed = int(self.seed) & 0xFFFFFFFFFFFFFFFF
        res, keep = self._fill_args(a, first, B, cp_proba, draws, perm, call_offset, clip_obs, relative_goals, want,
                                    want_idx, out)
        if args_only:
            # the caller launches a kernel that samples for itself (cur_ddpg_rows_step with `her`)
            res['_keep'] = keep
            return a, res
        _lib.check(lib.cur_her_sample(_lib.stream_ptr(stream), C.byref(a)), 'cur_her_sample')
        res['_keep'] = keep
        return res

    def _fill_args(self, a, first, B, cp_proba, draws, perm, call_offset, clip_obs, relative_goals, want, want_idx, out):
        """The cur_her_args fields both sampling entries share: layout, reward table, draws, shuffle, outputs."""
        L = first.layout
        dev = first.storage.device
        if self.reward.needs_info() and self._info_layout != first.info_keys:
            self._info_layout = first.info_keys
            self.task_table = self.reward.task_table(first.info_keys)
        a.L = L
        a.tasks = self.task_table
        if cp_proba is not None:
            _lib.set_cdf(a.tasks, cp_proba)
        elif self.mode == _lib.MODE_CP_TASK:
            # np.random.choice(range(n), p=None) is uniform (the store_episode stats path, ddpg.py:213)
            _lib.set_cdf(a.tasks, np.ones(max(self.nb_tasks, 1)) / max(self.nb_tasks, 1))
        a.mode = self.mode
        a.batch = B
        a.future_p = float(self.future_p)
        keep = []
        if draws is not None:
            d = upload_draws(draws, dev) if isinstance(draws, (list, tuple)) else draws
            keep.append(d)
            a.inj_ep, a.inj_t = d['ep'].data_ptr(), d['t'].data_ptr()
            a.inj_u_her, a.inj_u_off = d['u_her'].data_ptr(), d['u_off'].data_ptr()
            a.inj_choice = d['choice'].data_ptr() if d.get('choice') is not None else None
        else:
            a.call_offset = self.calls if call_offset is None else call_offset
        if call_offset is None:
            self.calls += 1
        if perm is not None:
            if not torch.is_tensor(perm):
                perm = torch.from_numpy(np.ascontiguousarray(perm, dtype=np.int32)).to(dev, non_blocking=True)
            keep.append(perm)
            a.perm = perm.data_ptr()
        a.clip_obs = float(clip_obs) if clip_obs and np.isfinite(clip_obs) else 0.0
        a.relative_goals = 1 if relative_goals else 0
        dims = dict(o=L.dimo, ag=L.dimag, g=L.dimg, u=L.dimu, td=L.dimtd, change=L.dimchange, info=L.diminfo,
                    o_2=L.dimo, ag_2=L.dimag, g_2=L.dimg, r=1)
        res = {} if out is None else out
        for k in want:
            if dims[k] <= 0:
                continue
            if k not in res:
                res[k] = torch.empty((B, dims[k]), dtype=torch.float32, device=dev)
            setattr(a, k, res[k].data_ptr())
        if want_idx:
            res['idx'] = torch.empty((B, 4), dtype=torch.int32, device=dev)
            a.idx_out = res['idx'].data_ptr()
        return res, keep

    def sample_workers(self, workers, rows_per_worker, *, dyn=None, step=None, cdf=None, draws=None, perm=None,
                       clip_obs=0.0, relative_goals=False, want=('o', 'ag', 'g', 'u', 'td', 'change', 'info', 'o_2',
                                                                  'ag_2', 'r'),
                       want_idx=False, out=None, stream=None, call_offset=None):
        """Worker-major form (cur_her_sample_workers): `workers` = [(philox_key, [(DeviceEpisodes, count, ttr), ...])],
        one entry per worker; worker j's rows are [j * rows_per_worker, (j + 1) * rows_per_worker) of every output.
        dyn: device address of len(workers) cur_her_worker_dyn (CUDA graph: the caller rewrites it between replays);
        None = built from the segments' counts / sizes and `cdf` and uploaded for this call.  step: device int64 counter
        added to the Philox call offset, or None.  draws: the workers' HostDraws, worker after worker; perm: the
        permutation of all concat rows (worker j's shuffle inside its own block)."""
        lib = _lib.load()
        n = len(workers)
        B = n * rows_per_worker
        first = workers[0][1][0][0]
        W = (_lib.HerWorker * max(n, 1))()
        host_dyn = (_lib.HerWorkerDyn * max(n, 1))()
        for j, (key, segs) in enumerate(workers):
            if len(segs) > _lib.CUR_MAX_SEGMENTS:
                raise ValueError('worker %d has %d buffers; at most %d' % (j, len(segs), _lib.CUR_MAX_SEGMENTS))
            W[j].seed = int(key) & 0xFFFFFFFFFFFFFFFF
            W[j].n_segments = len(segs)
            for i, (epi, count, ttr) in enumerate(segs):
                s = W[j].seg[i]
                s.base = epi.storage.data_ptr()
                s.cold = None if epi.cold is None else epi.cold.data_ptr()
                s.n_episodes = host_dyn[j].n_episodes[i] = int(epi.n_episodes)
                s.count = host_dyn[j].count[i] = int(count)
                s.task_to_replay = -1 if ttr is None else int(ttr)
            if cdf is not None:
                _lib.set_cdf(host_dyn[j], cdf)
        a = _lib.HerArgs()
        res, keep = self._fill_args(a, first, B, None, draws, perm, call_offset, clip_obs, relative_goals, want,
                                    want_idx, out)
        if dyn is None:
            if cdf is None and self.mode == _lib.MODE_CP_TASK:
                for j in range(n):
                    host_dyn[j].cdf = a.tasks.cdf
            blob = torch.frombuffer(bytearray(host_dyn), dtype=torch.uint8).pin_memory()
            dev = blob.to(first.storage.device, non_blocking=True)
            keep.append((blob, dev))
            dyn = dev.data_ptr()
        _lib.check(lib.cur_her_sample_workers(_lib.stream_ptr(stream), C.byref(a), n, rows_per_worker, W, dyn, step),
                   'cur_her_sample_workers')
        res['_keep'] = keep
        return res

    # ---- the reference closure signature -----------------------------------------------------------
    def __call__(self, episode_batch, batch_size_in_transitions, task_to_replay=None, cp_proba=None):
        B = int(batch_size_in_transitions)
        if isinstance(episode_batch, DeviceEpisodes):
            epi = episode_batch
        else:
            from .replay_buffer import episodes_to_device
            epi = episodes_to_device(episode_batch, self.device)
        L = epi.layout
        draws = None
        if self.rng == 'numpy':
            d = HostDraws(epi.n_episodes, L.T, B)
            d.draw_choices(self.mode, self.future_p, self.nb_tasks, cp_proba)
            draws = [d]
        res = self.sample_device([(epi, B, task_to_replay)], B, cp_proba=cp_proba, draws=draws)
        return self.to_host_dict(res, epi)

    def to_host_dict(self, res, epi):
        """Device result -> the reference's transitions dict (host arrays, reference key names)."""
        torch.cuda.current_stream().synchronize()
        out = {}
        for k in ('o', 'u', 'g', 'ag', 'o_2', 'ag_2', 'r'):
            out[k] = res[k].cpu().numpy().astype(self.out_dtype)
        if epi.has_td and 'td' in res:
            out['task_descr'] = res['td'].cpu().numpy().astype(self.out_dtype)
        if epi.has_change and 'change' in res:
            out['change'] = res['change'].cpu().numpy().astype(self.out_dtype)
        if epi.info_keys and 'info' in res:
            info = res['info'].cpu().numpy().astype(self.out_dtype)
            k0 = 0
            for key, dim in epi.info_keys:
                out[key] = info[:, k0:k0 + dim]
                k0 += dim
        return out


def make_sample_her_transitions(goal_replay, her_replay_k, reward_fun, task_replay='', tasks_ag_id=None,
                                tasks_g_id=None):
    """Flat HER sampler (reference her.py:5-68)."""
    return HerSampler(goal_replay, her_replay_k, task_replay, reward_fun, tasks_ag_id, tasks_g_id, flat=True)


def make_sample_multi_task_her_transitions(goal_replay, her_replay_k, task_replay, reward_fun,
                                           tasks_ag_id=None, tasks_g_id=None):
    """Modular HER sampler (reference her.py:72-185)."""
    return HerSampler(goal_replay, her_replay_k, task_replay, reward_fun, tasks_ag_id, tasks_g_id, flat=False)
