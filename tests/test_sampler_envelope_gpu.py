"""HER sampling and episode storage at the edges of the layouts they accept, through the C ABI, against the NumPy oracle.

tests/test_her_gpu.py runs the sampler at the Arm4 / Arm8 shapes the project trains on.  Here the layouts and task tables
are written out by hand (cur_layout_init, cur_task_table) so that every limit of include/curious_b200.h is reached:
16 modules with 8-entry slices, 17 segments, 64 workers, per-row outputs at every width mod 4, a shared-memory stage over
48 KB and the largest one the 227 KB limit admits, tiles cut at 1 / 31 / 32 / 33 / 4097 rows, episodes of 1 and 200
steps.  The fused prologue of the rows update kernel (cur_ddpg_rows_step with `her`) is compared with the standalone
sampler feeding the same update, and cur_store_episodes with a NumPy packing at the cur_layout_init offsets.

Reference: oracle/philox_oracle.draws for the draws of every concat row, oracle/her_oracle fed those draws one segment
at a time, concatenated and shuffled like DDPG.sample_batch (reference ddpg.py:325-345), oracle/reward_oracle for the
DISTANCE / PAIR / INFO rules and oracle/ddpg_oracle.preprocess_og (relative goals, clip) evaluated in float64.

Every comparison is exact.  The sampler only gathers float32 data, computes its reward in float64 in NumPy's operation
order and clips elementwise; the one float32 operation it does, g - ag of relative goals, is exact in float64 and
correctly rounded in float32, so the float64 difference rounded to float32 equals it as long as the float64 difference
is exact - which the data guarantee: every goal and achieved-goal value has a magnitude in [1/8, 4), a few binades apart.
Outputs are pre-filled with NaN and followed by NaN guard rows; idx_out is requested wherever draws matter and compared
with the oracle's draws.  Every refusal tested returns before any launch.
"""
import ctypes as C
import zlib

import numpy as np
import pytest

from curious_b200 import _lib

GUARD = 8
K = 4                                      # her_replay_k: future_p = 0.8 (reference her.py:86-89)
FUTURE_P = 1 - 1. / (1 + K)
F32 = np.float32
KEYS = ('o', 'ag', 'g', 'u', 'td', 'change', 'info', 'o_2', 'ag_2', 'g_2', 'r')
TASK_REPLAY = {_lib.MODE_BUFFER: 'replay_task_cp_buffer', _lib.MODE_RANDOM_TASK: 'replay_random_task_transition',
               _lib.MODE_CP_TASK: 'replay_cp_task_transition', _lib.MODE_CURRENT_TASK: 'replay_current_task_transition'}
KIND = {'distance': _lib.REWARD_DISTANCE, 'pair': _lib.REWARD_PAIR, 'info': _lib.REWARD_INFO}
HER_SMEM_LIMIT = 227 * 1024


def r4(x):
    return (x + 3) // 4 * 4


# ------------------------------------------------------------------------------------------------
# data
# ------------------------------------------------------------------------------------------------
def signed(rng, shape, lo, hi):
    return (rng.uniform(lo, hi, shape) * rng.choice([-1.0, 1.0], shape)).astype(F32)


def make_episodes(rng, E, dims, modules=None):
    """Key-major episodes {o [E,T+1,dimo], ag [E,T+1,dimag], g, u, td, change, info [E,T,dim]}: td one-hot and constant
    over an episode (episode e in module modules[e], or a drawn one), ag a slow random walk (HER rows land on both sides
    of the reward thresholds), goal values with magnitudes in [1/8, 4) (module docstring), info flags in {0, 1}."""
    T, dimo, dimag, dimg, dimu, dimtd, dimchange, diminfo = dims
    ag = signed(rng, (E, 1, dimag), 0.5, 1.5) + np.concatenate(
        [np.zeros((E, 1, dimag)), np.cumsum(rng.normal(0, 0.02, (E, T, dimag)), axis=1)], axis=1)
    ag = np.copysign(np.clip(np.abs(ag), 0.125, 3.5), ag).astype(F32)
    ep = dict(o=signed(rng, (E, T + 1, dimo), 0.0, 2.0), ag=ag, g=signed(rng, (E, T, dimg), 0.125, 2.0),
              u=signed(rng, (E, T, dimu), 0.0, 1.0), td=None, change=None, info=None)
    if dimtd:
        mods = rng.randint(0, dimtd, E) if modules is None else np.asarray(modules)
        ep['td'] = np.repeat(np.eye(dimtd, dtype=F32)[mods][:, None, :], T, axis=1)
    if dimchange:
        ep['change'] = rng.standard_normal((E, T, dimchange)).astype(F32)
    if diminfo:
        ep['info'] = (rng.uniform(size=(E, T, diminfo)) < 0.5).astype(F32)
    return ep


def pack(L, ep):
    """NumPy packing of key-major episodes at the cur_layout_init offsets: transition rows [o(t) | g u td ag(t+1) o(t+1)]
    and cold rows [change | info | ag(t)], padding zero."""
    E, T = ep['u'].shape[:2]
    dp = r4(L.dimo)
    hot = np.zeros((E, T, L.trans_stride), F32)
    hot[..., :L.dimo] = ep['o'][:, :T]
    blocks = [(L.off_g, ep['g']), (L.off_u, ep['u']), (L.off_td, ep['td']), (L.off_ag, ep['ag'][:, 1:]),
              (L.off_o, ep['o'][:, 1:])]
    for off, v in blocks:
        if v is not None and v.shape[-1]:
            hot[..., dp + off:dp + off + v.shape[-1]] = v
    cold = np.zeros((E, T, L.cold_stride), F32)
    for off, v in ((L.off_change, ep['change']), (L.off_info, ep['info']), (L.off_agc, ep['ag'][:, :T])):
        if v is not None and v.shape[-1]:
            cold[..., off:off + v.shape[-1]] = v
    return hot, cold


def stage_floats(L, cold):
    """Floats per transition of the sampler's shared-memory stage (make_plan, csrc/her_device.cuh)."""
    ss = r4(L.dimo) + L.row_stride + r4(L.dimag) + (L.cold_stride if cold else 0)
    return ss + 4 if (ss // 4) % 2 == 0 else ss


def her_smem(L, cold):
    return 32 * stage_floats(L, cold) * 4 + 3 * 32 * 8 + 16      # launch_her, csrc/her.cu


class Tasks(object):
    """One reward table, for the kernel (cur_task_table) and for the oracle (reward_oracle.ModuleRewardTable).
    An INFO module reads the last column of the info row, which the oracle sees as key 'info_is_success'."""

    def __init__(self, g_ids, ag_ids, thresholds, kinds=None, ref_ids=None, cp=None, flat_threshold=0.5, diminfo=0):
        n = len(g_ids)
        self.g_ids, self.ag_ids, self.cp = g_ids, ag_ids, cp
        self.kinds = kinds or ['distance'] * n
        self.ref_ids = ref_ids or [None] * n
        self.thresholds, self.flat_threshold = thresholds, flat_threshold
        self.table = _lib.make_task_table(ag_ids, g_ids, threshold=thresholds, kinds=[KIND[k] for k in self.kinds],
                                          ref_ag_id=self.ref_ids, info_cols=[diminfo - 1] * n, cp_proba=cp,
                                          flat_threshold=flat_threshold)

    def cdf(self):
        return None if self.cp is None else np.cumsum(self.cp) / np.cumsum(self.cp)[-1]

    def oracle_reward(self):
        from oracle.reward_oracle import ModuleRewardTable
        return ModuleRewardTable(self.ag_ids, self.g_ids, threshold=self.thresholds, kinds=self.kinds,
                                 ref_ag_id=self.ref_ids, info_keys=['is_success' if k == 'info' else None
                                                                    for k in self.kinds],
                                 flat_threshold=self.flat_threshold)


def slices(n, length, dim, rng=None):
    """n module slices of `length` entries covering a permutation of range(n * length) (consecutive without rng)."""
    ids = np.arange(n * length) if rng is None else rng.permutation(n * length)
    assert n * length <= dim
    return [list(map(int, ids[m * length:(m + 1) * length])) for m in range(n)]


class Seg(object):
    """A buffer on the device (packed by pack()) and its row of the segment table."""

    def __init__(self, L, ep, count, ttr=-1, n_episodes=None):
        import torch
        self.ep, self.count, self.ttr = ep, int(count), int(ttr)
        self.E = int(n_episodes if n_episodes is not None else ep['u'].shape[0])
        hot, cold = pack(L, ep)
        self.hot, self.cold = torch.from_numpy(hot).cuda(), torch.from_numpy(cold).cuda()


class Case(object):
    def __init__(self, dims, tasks, mode, segs, clip_obs=0.0, relative_goals=False, seed=0x5EED0123456789AB,
                 call_offset=7, perm=None):
        self.dims, self.tasks, self.mode, self.segs = dims, tasks, mode, segs
        self.L = _lib.make_layout(*dims)
        self.T = dims[0]
        self.clip_obs, self.relative_goals, self.seed, self.call_offset, self.perm = (
            clip_obs, relative_goals, seed, call_offset, perm)

    @property
    def B(self):
        return sum(s.count for s in self.segs)

    def dim(self, k):
        L = self.L
        return dict(o=L.dimo, ag=L.dimag, g=L.dimg, u=L.dimu, td=L.dimtd, change=L.dimchange, info=L.diminfo,
                    o_2=L.dimo, ag_2=L.dimag, g_2=L.dimg, r=1)[k]

    def args(self, outs=None, draws=None):
        """cur_her_args of this case; outs: {key: tensor}; draws: injected {ep, t, u_her, u_off, choice} tensors."""
        a = _lib.HerArgs()
        a.L = self.L
        a.tasks = self.tasks.table
        a.mode = self.mode
        a.n_segments = len(self.segs)
        for i, s in enumerate(self.segs):
            a.seg[i].base, a.seg[i].cold = s.hot.data_ptr(), s.cold.data_ptr()
            a.seg[i].n_episodes, a.seg[i].count, a.seg[i].task_to_replay = s.E, s.count, s.ttr
        a.batch = self.B
        a.future_p = FUTURE_P
        a.seed, a.call_offset = self.seed, self.call_offset
        if self.perm is not None:
            a.perm = self.perm.data_ptr()
        a.clip_obs = self.clip_obs
        a.relative_goals = 1 if self.relative_goals else 0
        for k, t in (outs or {}).items():
            setattr(a, 'idx_out' if k == 'idx' else k, t.data_ptr())
        if draws is not None:
            a.inj_ep, a.inj_t = draws['ep'].data_ptr(), draws['t'].data_ptr()
            a.inj_u_her, a.inj_u_off = draws['u_her'].data_ptr(), draws['u_off'].data_ptr()
            a.inj_choice = draws['choice'].data_ptr()
        return a

    def philox_draws(self):
        """philox_oracle.draws of every concat row, one dict per segment."""
        from oracle import philox_oracle
        name = {_lib.MODE_RANDOM_TASK: 'random', _lib.MODE_CP_TASK: 'cp'}.get(self.mode)
        out, acc = [], 0
        for s in self.segs:
            out.append(philox_oracle.draws(np.arange(acc, acc + s.count), np.full(s.count, s.E), self.T, self.seed,
                                           self.call_offset, mode=name, n_tasks=self.tasks.table.n_tasks,
                                           cdf=self.tasks.cdf()))
            acc += s.count
        return out


def nan_outputs(case, keys, B=None):
    import torch
    B = case.B if B is None else B
    outs = {k: torch.full((B + GUARD, case.dim(k)), float('nan'), dtype=torch.float32, device='cuda')
            for k in keys if case.dim(k) > 0}
    outs['idx'] = torch.full((B + GUARD, 4), -12345, dtype=torch.int32, device='cuda')
    return outs


def fetch(outs, B):
    """Host copies of the outputs; the guard rows must be untouched."""
    import torch
    torch.cuda.synchronize()
    res = {}
    for k, t in outs.items():
        h = t.cpu().numpy()
        guard = h[B:]
        assert (np.isnan(guard).all() if k != 'idx' else (guard == -12345).all()), '%s written past row %d' % (k, B)
        res[k] = h[:B]
    return res


def sample(case, keys=KEYS, draws=None, dyn=None):
    """cur_her_sample of the case into NaN-filled outputs; returns the host outputs."""
    outs = nan_outputs(case, keys)
    a = case.args(outs, draws)
    if dyn is not None:
        a.dyn = dyn.data_ptr()
    _lib.check(_lib.load().cur_her_sample(_lib.stream_ptr(), C.byref(a)), 'cur_her_sample')
    return fetch(outs, case.B)


def upload_draws(d):
    import torch
    return dict(ep=torch.from_numpy(d['ep'].astype(np.int32)).cuda(), t=torch.from_numpy(d['t'].astype(np.int32)).cuda(),
                u_her=torch.from_numpy(d['u_her'].astype(np.float64)).cuda(),
                u_off=torch.from_numpy(d['u_off'].astype(np.float64)).cuda(),
                choice=torch.from_numpy(np.where(d['u_her'] < FUTURE_P, d['choice'], -1).astype(np.int32)).cuda())


# ------------------------------------------------------------------------------------------------
# the oracle side
# ------------------------------------------------------------------------------------------------
def oracle_batch(ep, diminfo):
    """The reference's episode dict of one buffer (replay_buffer.py:44-48): o_2 / ag_2 are the shifted views."""
    b = dict(o=ep['o'], ag=ep['ag'], g=ep['g'], u=ep['u'], o_2=ep['o'][:, 1:], ag_2=ep['ag'][:, 1:])
    if ep['td'] is not None:
        b['task_descr'] = ep['td']
    if ep['change'] is not None:
        b['change'] = ep['change']
    if diminfo:
        if diminfo > 1:
            b['info_a'] = ep['info'][..., :diminfo - 1]
        b['info_is_success'] = ep['info'][..., diminfo - 1:]
    return b


def oracle(case, draws):
    """her_oracle fed the draws one segment at a time, concatenated, shuffled and preprocessed (ddpg.py:325-353)."""
    from oracle import ddpg_oracle, her_oracle
    tk = case.tasks
    reward = tk.oracle_reward()
    if case.mode == _lib.MODE_FLAT:
        s = her_oracle.make_sample_her_transitions('her', K, reward, '', tasks_ag_id=tk.ag_ids, tasks_g_id=tk.g_ids)
    else:
        s = her_oracle.make_sample_multi_task_her_transitions('her', K, TASK_REPLAY[case.mode], reward,
                                                              tasks_ag_id=tk.ag_ids, tasks_g_id=tk.g_ids)
    parts = []
    for seg, d in zip(case.segs, draws):
        n = d['ep'].shape[0]
        if n == 0:
            continue
        her = d['u_her'] < FUTURE_P
        stream = her_oracle.HerStream(d['ep'].astype(np.int64), d['t'].astype(np.int64), d['u_her'], d['u_off'],
                                      np.where(her, d['choice'], -1).astype(np.int64))
        out = s(oracle_batch(seg.ep, case.L.diminfo), n, task_to_replay=None if seg.ttr < 0 else seg.ttr,
                cp_proba=tk.cp, stream=stream)
        ft = np.where(her, d['t'] + 1 + (d['u_off'] * (case.T - d['t'])).astype(int), -1)
        if case.mode == _lib.MODE_FLAT:
            mod = np.where(her, 0, -1)
        else:
            mod = np.where(her, np.argmax(out['task_descr'], axis=1), -1)
        p = dict(o=out['o'], ag=out['ag'], g=out['g'], u=out['u'], o_2=out['o_2'], ag_2=out['ag_2'], r=out['r'],
                 idx=np.stack([d['ep'], d['t'], ft, mod], axis=1).astype(np.int32))
        if 'task_descr' in out:
            p['td'] = out['task_descr']
        if 'change' in out:
            p['change'] = out['change']
        if case.L.diminfo:
            p['info'] = np.concatenate([out[k] for k in ('info_a', 'info_is_success') if k in out], axis=1)
        parts.append(p)
    ref = {k: np.concatenate([p[k] for p in parts]) for k in parts[0]}
    if case.perm is not None:
        perm = case.perm.cpu().numpy()
        ref = {k: v[perm] for k, v in ref.items()}
    clip = case.clip_obs if case.clip_obs > 0 else np.inf
    f64 = {k: np.asarray(ref[k], np.float64) for k in ('o', 'ag', 'g', 'o_2', 'ag_2')}
    o, g = ddpg_oracle.preprocess_og(f64['o'], f64['ag'], f64['g'], clip, case.relative_goals)
    o_2, g_2 = ddpg_oracle.preprocess_og(f64['o_2'], f64['ag_2'], f64['g'], clip, case.relative_goals)
    ref.update(o=o, g=g, o_2=o_2, g_2=g_2)
    ref['r'] = np.asarray(ref['r']).reshape(-1, 1)
    return {k: (v if k == 'idx' else np.asarray(v, np.float64).astype(F32)) for k, v in ref.items()}


def assert_equal(got, ref, label=''):
    assert got, 'no output'
    for k, v in got.items():
        assert k in ref, (label, k)
        assert v.shape == ref[k].shape, (label, k, v.shape, ref[k].shape)
        bad = np.argwhere(v != ref[k])                # a NaN (an element never written) differs from everything
        assert bad.size == 0, '%s %s: %d elements differ, first at %s: %r vs %r' % (
            label, k, len(bad), bad[0], v[tuple(bad[0])], ref[k][tuple(bad[0])])


def check_case(case, keys=KEYS, label=''):
    """Philox draws of the kernel against the oracle; returns the host outputs."""
    got = sample(case, keys)
    ref = oracle(case, case.philox_draws())
    assert_equal(got, ref, label)
    return got


def make_perm(rng, B):
    import torch
    return torch.from_numpy(rng.permutation(B).astype(np.int32)).cuda()


# ------------------------------------------------------------------------------------------------
# the fused-prologue predicate (CPU: the library answers without a device)
# ------------------------------------------------------------------------------------------------
def _net(modular, dimo, dimg, dimu, dimtd, hidden=256, layers=3):
    return _lib.NetDesc(modular, dimo, dimg, dimu, dimtd, hidden, layers, 1.0, 0, 5.0)


def _her(L, batch, tasks=None, relative_goals=0, cold=True, n_segments=2):
    a = _lib.HerArgs()
    a.L = L
    a.batch = batch
    a.n_segments = n_segments
    a.relative_goals = relative_goals
    if tasks is not None:
        a.tasks = tasks
    for i in range(n_segments):
        a.seg[i].base = 256                     # never dereferenced: the predicate makes no CUDA call
        a.seg[i].cold = 512 if cold else None
    return a


def _arm(n_modules, dimo, info_module=None):
    """(net, layout, task table) of tests/ddpg_util.ddpg_kwargs(n_modules, dimo=dimo)."""
    from curious_b200 import synth
    dims = synth.arm_dims(n_modules, dimo)
    ag_ids, g_ids = synth.arm_task_ids(n_modules)
    kinds = [_lib.REWARD_INFO if m == info_module else _lib.REWARD_DISTANCE for m in range(n_modules)]
    L = _lib.make_layout(50, dims['o'], dims['ag'], dims['g'], dims['u'], dims['task_descr'], dims['ag'], 1)
    return (_net(1, dims['o'], dims['g'], dims['u'], dims['task_descr']), L,
            _lib.make_task_table(ag_ids, g_ids, kinds=kinds, info_cols=[0] * n_modules))


def test_fused_her_predicate_at_the_edges():
    """cur_ddpg_rows_her_supported: 1 exactly when the rows update kernel samples the batch in its prologue.  The 4-row
    HER stage holds 448 floats per transition; Arm4 at dimo 200 needs 444, at dimo 204 452 (csrc/her_device.cuh)."""
    lib = _lib.load()
    K256 = _net(1, 212, 28, 8, 8)                         # Q fan-in 256: rows-supported, stage 524 floats
    K256_L = _lib.make_layout(50, 212, 28, 28, 8, 8, 28, 1)
    FLAT256 = _net(0, 200, 48, 8, 0)
    FLAT256_L = _lib.make_layout(50, 200, 48, 48, 8, 0, 0, 0)
    rows = []
    for dimo, want in ((40, 1), (200, 1), (204, 0)):
        d, L, tt = _arm(4, dimo)
        rows.append(('arm4 dimo %d' % dimo, d, _her(L, 256, tt), want))
    d, L, tt = _arm(8, 220)
    rows.append(('arm8 dimo 220 (Q fan-in 256)', d, _her(L, 256, tt), 0))
    rows.append(('K256', K256, _her(K256_L, 256), 0))
    rows.append(('FLAT256', FLAT256, _her(FLAT256_L, 256), 0))
    d, L, tt = _arm(4, 200, info_module=2)                # the cold row of an INFO reward tips the stage over
    rows.append(('arm4 dimo 200, INFO reward', d, _her(L, 256, tt), 0))
    d, L, tt = _arm(4, 40, info_module=2)
    rows.append(('arm4 dimo 40, INFO reward', d, _her(L, 256, tt), 1))
    rows.append(('arm4 dimo 40, INFO reward, a segment without cold rows', d, _her(L, 256, tt, cold=False), 0))
    d, L, tt = _arm(4, 40)
    rows.append(('arm4 dimo 40, relative goals', d, _her(L, 256, tt, relative_goals=1), 1))
    d, L, tt = _arm(4, 200)
    rows.append(('arm4 dimo 200, relative goals (cold row staged)', d, _her(L, 256, tt, relative_goals=1), 0))
    d, L, tt = _arm(4, 40)
    for n, want in ((4, 1), (1024, 1), (254, 0), (1028, 0), (0, 0)):
        rows.append(('arm4 dimo 40, batch %d' % n, d, _her(L, n, tt), want))
    for field, value in (('dimo', 44), ('dimg', 16), ('dimu', 8), ('dimtd', 5)):
        L2 = _lib.make_layout(*[50] + [value if f == field else getattr(L, f) for f in
                                       ('dimo', 'dimag', 'dimg', 'dimu', 'dimtd', 'dimchange', 'diminfo')])
        rows.append(('layout %s %d against the net' % (field, value), d, _her(L2, 256, tt), 0))
    L3 = _lib.make_layout(50, 40, 16, 12, 4, 4, 16, 1)     # dimag != dimg
    rows.append(('relative goals, dimag 16 != dimg 12', d, _her(L3, 256, tt, relative_goals=1), 0))
    rows.append(('same layout without relative goals', d, _her(L3, 256, tt), 1))
    rows.append(('hidden 64', _net(1, 40, 12, 4, 4, 64, 2), _her(L, 256, tt), 1))
    bad = [(label, got, want) for label, d, a, want in rows
           for got in [lib.cur_ddpg_rows_her_supported(C.byref(d), C.byref(a))] if got != want]
    assert not bad, bad
    assert lib.cur_ddpg_rows_her_supported(C.byref(_arm(4, 40)[0]), None) == 0


def test_stage_arithmetic_of_the_shapes_below():
    """The shapes of test_shared_memory_stage_sizes_in_one_process sit where their names say (CPU)."""
    small, wide, widest, past = (_lib.make_layout(5, dimo, 4, 4, 4, 0, 0, 0) for dimo in (8, 200, 892, 893))
    assert her_smem(small, False) <= 48 * 1024 < her_smem(wide, False)
    assert her_smem(widest, False) <= HER_SMEM_LIMIT < her_smem(past, False)
    assert stage_floats(past, False) - stage_floats(widest, False) == 8      # the next admissible stage stride


# ------------------------------------------------------------------------------------------------
# GPU: the sampling kernels against the oracle
# ------------------------------------------------------------------------------------------------
DIMS16 = (20, 10, 136, 128, 3, 16, 5, 3)                  # T, dimo, dimag > dimg, dimg = 16 x 8, dimu, dimtd, change, info


def tasks16(rng, mode):
    """16 modules of 8 entries: permuted g slices (consecutive for FLAT, whose oracle writes g as one block), ag slices
    overlapping each other, per-module thresholds, a PAIR module (3, modular modes) and an INFO module (5, last info
    column)."""
    n = 16
    g_ids = slices(n, 8, 128) if mode == _lib.MODE_FLAT else slices(n, 8, 128, rng)
    ag_ids = [list(map(int, rng.randint(0, 136, 8))) for _ in range(n)]
    kinds = ['distance'] * n
    kinds[5] = 'info'
    if mode != _lib.MODE_FLAT:                  # (the flat distance sums every module: a pair slice would dominate it)
        kinds[3] = 'pair'
    ref = [None] * n
    ref[3] = list(map(int, rng.randint(0, 136, 8)))
    thr = [0.03 + 0.01 * m for m in range(n)]
    thr[3] = 2.5
    cp = np.array([0, 0] + list(rng.uniform(0.5, 2.0, 12)) + [0, 0])
    return Tasks(g_ids, ag_ids, thr, kinds, ref, cp=cp if mode == _lib.MODE_CP_TASK else None, flat_threshold=1.0,
                 diminfo=3)


@pytest.mark.gpu
@pytest.mark.parametrize('mode,ttr', [(_lib.MODE_BUFFER, (15, -1)), (_lib.MODE_RANDOM_TASK, (-1,)),
                                      (_lib.MODE_CP_TASK, (-1,)), (_lib.MODE_CURRENT_TASK, (-1,)),
                                      (_lib.MODE_FLAT, (-1,))])
def test_task_table_limits(mode, ttr):
    """16 modules (tasks16) in every mode: BUFFER with task_to_replay 15 and -1, RANDOM over 16 modules, CP_TASK with
    probability 0 for the first and last two modules, CURRENT, FLAT."""
    rng = np.random.RandomState(100 + mode)
    tk = tasks16(rng, mode)
    dims = DIMS16 if mode != _lib.MODE_FLAT else DIMS16[:5] + (0,) + DIMS16[6:]
    segs = [Seg(_lib.make_layout(*dims), make_episodes(rng, 40, dims, np.arange(40) % 16), 700, t) for t in ttr]
    case = Case(dims, tk, mode, segs, clip_obs=1.5, perm=make_perm(rng, 700 * len(ttr)))
    got = check_case(case, label='mode %d' % mode)
    her = got['idx'][:, 2] >= 0
    assert set(np.unique(got['r'])) == {-1.0, 0.0}
    if mode == _lib.MODE_BUFFER:
        first = case.perm.cpu().numpy() < 700                   # rows of the segment with task_to_replay 15
        assert (got['idx'][her & first, 3] == 15).all() and (got['td'][her & first, 15] == 1).all()
        assert len(np.unique(got['idx'][her & ~first, 3])) == 16        # the rows' own modules
    if mode == _lib.MODE_CP_TASK:
        chosen = set(np.unique(got['idx'][her, 3]))
        assert chosen == set(range(2, 14)), chosen               # probability 0: modules 0, 1, 14, 15 never
    if mode in (_lib.MODE_BUFFER, _lib.MODE_RANDOM_TASK, _lib.MODE_CURRENT_TASK):
        mod = np.argmax(got['td'], axis=1)
        for m, kind in ((3, 'pair'), (5, 'info')):
            assert (her & (mod == m)).sum() > 5, (kind, m)


@pytest.mark.gpu
def test_seventeen_segments():
    """17 buffers of 1 to 300 episodes with zero counts first, in the middle and last, a task_to_replay per buffer,
    shuffled rows."""
    rng = np.random.RandomState(3)
    dims = (10, 9, 6, 6, 2, 3, 0, 0)
    tk = Tasks(slices(3, 2, 6, rng), [[0, 1], [2, 3], [4, 5]], [0.04, 0.05, 0.06])
    L = _lib.make_layout(*dims)
    counts = [0, 31, 1, 0, 64, 9, 0, 0, 120, 2, 33, 0, 77, 5, 16, 40, 0]
    sizes = [3, 1, 300, 2, 7, 1, 250, 4, 120, 9, 30, 1, 64, 2, 200, 11, 5]
    ttrs = [-1, 0, 2, 1, -1, 1, 0, -1, 2, 0, -1, 1, 2, -1, 0, 1, 2]
    segs = [Seg(L, make_episodes(rng, E, dims), c, t) for c, E, t in zip(counts, sizes, ttrs)]
    case = Case(dims, tk, _lib.MODE_BUFFER, segs, clip_obs=1.0, perm=make_perm(rng, sum(counts)))
    assert len(segs) == _lib.CUR_MAX_SEGMENTS
    check_case(case)


WIDTHS = {0: (8, 4, 4, 4, 8, 4, 4, 4), 1: (8, 1, 5, 5, 1, 5, 1, 1), 2: (8, 2, 6, 6, 2, 2, 2, 2),
          3: (8, 3, 7, 7, 3, 3, 3, 3)}


@pytest.mark.gpu
@pytest.mark.parametrize('relative_goals', [False, True])
@pytest.mark.parametrize('residue', [0, 1, 2, 3])
def test_output_widths(residue, relative_goals):
    """Every per-row output at a width of `residue` mod 4: the 16-byte path (0) and the scalar path of emit / emit2."""
    rng = np.random.RandomState(10 + residue)
    dims = WIDTHS[residue]
    n = dims[5]
    g = slices(n, 1, dims[3])
    tk = Tasks(g, [[int(x)] for x in rng.randint(0, dims[2], n)], [0.05] * n, kinds=['info'] + ['distance'] * (n - 1),
               diminfo=dims[7])
    segs = [Seg(_lib.make_layout(*dims), make_episodes(rng, 30, dims), c, t) for c, t in ((70, -1), (63, 0))]
    case = Case(dims, tk, _lib.MODE_BUFFER, segs, clip_obs=1.0, relative_goals=relative_goals,
                perm=make_perm(rng, 133))
    check_case(case)


@pytest.mark.gpu
@pytest.mark.parametrize('keys', [('r',), ('g_2', 'td'), ('g',), ('o_2', 'ag')])
def test_selective_outputs(keys):
    """Only some outputs passed: those are exact and their guard rows intact (idx_out always)."""
    rng = np.random.RandomState(21)
    dims = WIDTHS[3]
    tk = Tasks(slices(3, 1, 7), [[0], [1], [2]], [0.05] * 3, diminfo=3)
    segs = [Seg(_lib.make_layout(*dims), make_episodes(rng, 20, dims), 77)]
    case = Case(dims, tk, _lib.MODE_RANDOM_TASK, segs, clip_obs=1.0, relative_goals=True)
    got = check_case(case, keys)
    assert set(got) == set(keys) | {'idx'}


@pytest.mark.gpu
def test_shared_memory_stage_sizes_in_one_process():
    """The sampler keeps its configured dynamic shared-memory size between calls: a small stage, one over 48 KB (the
    opt-in), the largest the 227 KB limit admits, the small one again; one step past the limit is refused before any
    launch."""
    rng = np.random.RandomState(5)
    tk = Tasks([[0, 1, 2, 3]], [[3, 2, 1, 0]], [0.1])
    keys = ('o', 'g', 'u', 'o_2', 'ag_2', 'g_2', 'r')            # no cold row in the stage
    for dimo in (8, 200, 892, 8):
        dims = (5, dimo, 4, 4, 4, 0, 0, 0)
        segs = [Seg(_lib.make_layout(*dims), make_episodes(rng, 6, dims), 70)]
        check_case(Case(dims, tk, _lib.MODE_FLAT, segs, clip_obs=1.0), keys, label='dimo %d' % dimo)
    dims = (5, 893, 4, 4, 4, 0, 0, 0)
    case = Case(dims, tk, _lib.MODE_FLAT, [Seg(_lib.make_layout(*dims), make_episodes(rng, 6, dims), 70)])
    outs = nan_outputs(case, keys)
    assert _lib.load().cur_her_sample(_lib.stream_ptr(), C.byref(case.args(outs))) == 1
    got = fetch(outs, case.B)
    assert all(np.isnan(v).all() for k, v in got.items() if k != 'idx') and (got['idx'] == -12345).all()


@pytest.mark.gpu
@pytest.mark.parametrize('T', [1, 200])
def test_tiles_and_episode_lengths(T):
    """Batches that end a 32-row tile early, exactly, one row into the next, and 4097; every future t is 1 when T = 1."""
    rng = np.random.RandomState(T)
    dims = (T, 6, 6, 6, 4, 2, 0, 0)
    tk = Tasks([[0, 1, 2], [3, 4, 5]], [[0, 1, 2], [3, 4, 5]], [0.05, 0.08])
    L = _lib.make_layout(*dims)
    ep = make_episodes(rng, 25, dims)
    for B in (1, 31, 32, 33, 4097):
        got = check_case(Case(dims, tk, _lib.MODE_BUFFER, [Seg(L, ep, B, -1)], perm=make_perm(rng, B)),
                         label='B %d' % B)
        if T == 1:
            her = got['idx'][:, 2] >= 0
            assert (got['idx'][her, 2] == 1).all() and (got['idx'][:, 1] == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize('clip_obs', [0.75, 0.0])
def test_relative_goals_and_clip(clip_obs):
    """Relative goals (g - ag, g - ag_2) with a clip that binds on part of o, g, o_2 and g_2, and without a clip."""
    rng = np.random.RandomState(8)
    dims = (12, 9, 9, 9, 4, 3, 0, 0)
    tk = Tasks(slices(3, 3, 9, rng), slices(3, 3, 9, rng), [0.05, 0.05, 0.1])
    segs = [Seg(_lib.make_layout(*dims), make_episodes(rng, 30, dims), 300, t) for t in (-1, 1)]
    case = Case(dims, tk, _lib.MODE_BUFFER, segs, clip_obs=clip_obs, relative_goals=True, perm=make_perm(rng, 600))
    got = check_case(case)
    for k in ('o', 'g', 'o_2', 'g_2'):
        at = np.abs(got[k]) == clip_obs
        if clip_obs:
            assert 0.05 < at.mean() < 0.95, (k, at.mean())
        else:
            assert np.abs(got[k]).max() > 1.0


@pytest.mark.gpu
def test_device_control_block():
    """cur_her_dyn with counts, sizes and a cdf that differ from the arguments, and a step pointer: the same call with
    those values in seg[] / tasks.cdf and call_offset + step."""
    import torch
    rng = np.random.RandomState(12)
    dims = (15, 7, 8, 8, 3, 4, 0, 2)
    tk = Tasks(slices(4, 2, 8, rng), slices(4, 2, 8, rng), [0.05] * 4, kinds=['distance', 'info', 'distance', 'pair'],
               ref_ids=[None, None, None, [7, 6]], cp=np.array([1.0, 2.0, 3.0, 4.0]), diminfo=2)
    L = _lib.make_layout(*dims)
    segs = [Seg(L, make_episodes(rng, 50, dims), c) for c in (10, 20, 30, 40, 28)]
    case = Case(dims, tk, _lib.MODE_CP_TASK, segs, clip_obs=1.0, call_offset=11, perm=make_perm(rng, 128))
    counts, sizes, cp = [0, 64, 0, 50, 14], [3, 50, 1, 17, 2], np.array([0.5, 0.0, 2.0, 1.0])
    cdf = np.cumsum(cp) / np.cumsum(cp)[-1]
    step = torch.tensor([5], dtype=torch.int64, device='cuda')
    dyn = _lib.HerDyn()
    dyn.step = step.data_ptr()
    for i in range(5):
        dyn.n_episodes[i], dyn.count[i] = sizes[i], counts[i]
    for k in range(4):
        dyn.cdf[k] = cdf[k]
    dyn_dev = torch.frombuffer(bytearray(dyn), dtype=torch.uint8).cuda()
    got = sample(case, dyn=dyn_dev)
    for s, c, E in zip(segs, counts, sizes):
        s.count, s.E = c, E
    _lib.set_cdf(tk.table, cp)
    tk.cp = cp
    case.call_offset = 16
    want = sample(case)
    assert_equal(got, want, 'control block')
    assert_equal(want, oracle(case, case.philox_draws()))
    assert int(step.item()) == 5


@pytest.mark.gpu
@pytest.mark.parametrize('rows_per_worker', [5, 1])
def test_workers_equal_single_worker_calls(rows_per_worker):
    """cur_her_sample_workers with 64 workers of 1-17 segments each (5 rows: tiles straddle workers) equals the 64
    cur_her_sample calls with each worker's key, segments and cdf, concatenated."""
    import torch
    rng = np.random.RandomState(40 + rows_per_worker)
    dims = (9, 5, 6, 6, 3, 3, 0, 0)
    L = _lib.make_layout(*dims)
    pool = [Seg(L, make_episodes(rng, E, dims), 0) for E in rng.randint(1, 40, _lib.CUR_MAX_SEGMENTS)]
    tk = Tasks(slices(3, 2, 6, rng), [[0, 1], [2, 3], [4, 5]], [0.05] * 3, cp=np.array([1.0, 1.0, 1.0]))
    n = _lib.CUR_MAX_WORKERS
    W = (_lib.HerWorker * n)()
    wdyn = (_lib.HerWorkerDyn * n)()
    singles = []
    for j in range(n):
        nseg = 1 + j % _lib.CUR_MAX_SEGMENTS
        counts = rng.multinomial(rows_per_worker, np.ones(nseg) / nseg)
        cp = rng.uniform(0.0, 1.0, 3)
        W[j].seed = int(rng.randint(0, 2 ** 62)) * 3 + 1
        W[j].n_segments = nseg
        segs = []
        for i in range(nseg):
            src = pool[(i + j) % len(pool)]
            seg = Seg.__new__(Seg)
            seg.ep, seg.hot, seg.cold = src.ep, src.hot, src.cold
            seg.count, seg.ttr, seg.E = int(counts[i]), int(rng.randint(-1, 3)), int(rng.randint(1, src.E + 1))
            W[j].seg[i].base, W[j].seg[i].cold = seg.hot.data_ptr(), seg.cold.data_ptr()
            W[j].seg[i].count, W[j].seg[i].n_episodes, W[j].seg[i].task_to_replay = seg.count, seg.E, seg.ttr
            wdyn[j].count[i], wdyn[j].n_episodes[i] = seg.count, seg.E
            segs.append(seg)
        cdf = np.cumsum(cp) / np.cumsum(cp)[-1]
        for k in range(3):
            wdyn[j].cdf[k] = cdf[k]
        singles.append((W[j].seed, segs, cp))
    step = torch.tensor([2], dtype=torch.int64, device='cuda')
    dyn_dev = torch.frombuffer(bytearray(wdyn), dtype=torch.uint8).cuda()
    case = Case(dims, tk, _lib.MODE_CP_TASK, [], clip_obs=1.0, call_offset=9)
    B = n * rows_per_worker
    outs = nan_outputs(case, KEYS, B)
    a = case.args(outs)
    a.batch = B
    _lib.check(_lib.load().cur_her_sample_workers(_lib.stream_ptr(), C.byref(a), n, rows_per_worker, W,
                                                  dyn_dev.data_ptr(), step.data_ptr()), 'cur_her_sample_workers')
    got = fetch(outs, B)
    parts = []
    for seed, segs, cp in singles:
        _lib.set_cdf(tk.table, cp)
        single = Case(dims, tk, _lib.MODE_CP_TASK, segs, clip_obs=1.0, seed=seed, call_offset=11)
        parts.append(sample(single))
    want = {k: np.concatenate([p[k] for p in parts]) for k in parts[0]}
    assert_equal(got, want, 'workers')


# ------------------------------------------------------------------------------------------------
# GPU: cur_store_episodes
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('dims,null_src', [(DIMS16, False), (WIDTHS[1], False), (WIDTHS[3], False),
                                           ((7, 13, 5, 5, 3, 2, 4, 3), True)],
                         ids=['16-modules', 'widths-1', 'widths-3', 'flat-td-change-info-null'])
def test_store_episodes(dims, null_src):
    """130 copies (three launches) of 9 episodes into two NaN-filled buffers, the last slot of each included: the
    targeted slots equal the NumPy packing, every other slot stays NaN (null_src: td, change and info passed as NULL,
    zeros stored).  Then every stored (slot, t) is sampled with injected draws and compared with the oracle fed the
    source episodes."""
    import torch
    rng = np.random.RandomState(sum(dims))
    T = dims[0]
    L = _lib.make_layout(*dims)
    src = make_episodes(rng, 9, dims)
    if null_src:
        src = dict(src, td=None, change=None, info=None)
    sizes = (100, 45)
    hot = [torch.full((E, T, L.trans_stride), float('nan'), device='cuda') for E in sizes]
    cold = [torch.full((E, T, L.cold_stride), float('nan'), device='cuda') for E in sizes]
    slots = [list(rng.permutation(E - 1)[:k - 1]) + [E - 1] for E, k in zip(sizes, (90, 40))]
    copies = [(int(rng.randint(0, 9)), b, int(s)) for b in (0, 1) for s in slots[b]]
    copies = [copies[i] for i in rng.permutation(len(copies))]
    assert len(copies) == 130
    dev = {k: (None if v is None else torch.from_numpy(np.ascontiguousarray(v)).cuda()) for k, v in src.items()}
    es = _lib.EpisodeSrc(*[_lib.ptr(dev[k]) for k in ('o', 'ag', 'g', 'u', 'td', 'change', 'info')])
    n = len(copies)
    c_src = (C.c_int32 * n)(*[c[0] for c in copies])
    c_hot = (C.c_void_p * n)(*[hot[c[1]].data_ptr() for c in copies])
    c_cold = (C.c_void_p * n)(*[cold[c[1]].data_ptr() for c in copies])
    c_slot = (C.c_int64 * n)(*[c[2] for c in copies])
    _lib.check(_lib.load().cur_store_episodes(_lib.stream_ptr(), C.byref(L), C.byref(es), 9, n, c_src, c_hot, c_cold,
                                              c_slot), 'cur_store_episodes')
    torch.cuda.synchronize()
    ph, pc = pack(L, src)
    for b in (0, 1):
        h, c = hot[b].cpu().numpy(), cold[b].cpu().numpy()
        owner = {s: e for e, bb, s in copies if bb == b}
        for s in range(sizes[b]):
            if s in owner:
                assert np.array_equal(h[s], ph[owner[s]]) and np.array_equal(c[s], pc[owner[s]]), (b, s)
            else:
                assert np.isnan(h[s]).all() and np.isnan(c[s]).all(), (b, s)
    # every stored transition of buffer 0, against the oracle fed the source episodes laid out by slot
    owner = {s: e for e, bb, s in copies if bb == 0}
    stored = np.array(sorted(owner), np.int64)
    by_slot = {}
    for k, dim in (('o', dims[1]), ('ag', dims[2]), ('g', dims[3]), ('u', dims[4]), ('td', dims[5]),
                   ('change', dims[6]), ('info', dims[7])):
        by_slot[k] = np.zeros((sizes[0], T + (k in ('o', 'ag')), dim), F32) if dim else None
        if dim and src[k] is not None:
            for s, e in owner.items():
                by_slot[k][s] = src[k][e]
    seg = Seg.__new__(Seg)
    seg.ep, seg.hot, seg.cold, seg.ttr, seg.E, seg.count = by_slot, hot[0], cold[0], -1, sizes[0], len(stored) * T
    B = seg.count
    d = dict(ep=np.repeat(stored, T), t=np.tile(np.arange(T), len(stored)), u_her=rng.uniform(size=B),
             u_off=rng.uniform(size=B), choice=np.full(B, -1))
    if null_src:                                # FLAT: the goal is the concatenation of the module slices
        tk = Tasks([list(range(dims[3]))], [[(dims[3] - 1 - k) % dims[2] for k in range(dims[3])]], [0.1])
        mode = _lib.MODE_FLAT
    else:
        tk = Tasks(slices(dims[5], 1, dims[3]), [[m % dims[2]] for m in range(dims[5])], [0.05] * dims[5],
                   diminfo=dims[7])
        mode = _lib.MODE_BUFFER
    case = Case(dims, tk, mode, [seg], clip_obs=1.0)
    got = sample(case, draws=upload_draws(d))
    assert_equal(got, oracle(case, [d]), 'stored transitions')
    assert np.array_equal(got['idx'][:, :2], np.stack([d['ep'], d['t']], axis=1))


# ------------------------------------------------------------------------------------------------
# GPU: the fused prologue of the rows update kernel against the standalone sampler
# ------------------------------------------------------------------------------------------------
def _fused_case(name):
    """(case, net desc, injected draws | 'dyn' (device control block) | None)."""
    rng = np.random.RandomState(zlib.crc32(name.encode()))
    if name == '16-modules-cp':
        dims = (20, 16, 36, 32, 4, 16, 0, 0)
        cp = np.array([0, 0] + list(rng.uniform(0.5, 2.0, 12)) + [0, 0])
        tk = Tasks(slices(16, 2, 32, rng), [list(map(int, rng.randint(0, 36, 2))) for _ in range(16)],
                   [0.03 + 0.005 * m for m in range(16)], cp=cp)
        segs = [Seg(_lib.make_layout(*dims), make_episodes(rng, 40, dims), 256)]
        return Case(dims, tk, _lib.MODE_CP_TASK, segs, clip_obs=1.5), _net(1, 16, 32, 4, 16, 256, 3), None
    if name == '17-segments':
        dims = (10, 9, 8, 8, 4, 3, 0, 0)
        tk = Tasks(slices(3, 2, 8, rng), [[0, 1], [2, 3], [4, 5]], [0.04, 0.05, 0.06])
        L = _lib.make_layout(*dims)
        counts = [0, 40, 0, 16, 0, 0, 64, 8, 0, 32, 24, 0, 20, 12, 20, 20, 0]
        segs = [Seg(L, make_episodes(rng, int(rng.randint(1, 60)), dims), c, int(rng.randint(-1, 3))) for c in counts]
        return Case(dims, tk, _lib.MODE_BUFFER, segs, clip_obs=1.0), _net(1, 9, 8, 4, 3, 64, 2), None
    if name == 'relative-clip-normalize':
        dims = (16, 20, 12, 12, 4, 4, 0, 0)
        tk = Tasks(slices(4, 3, 12), slices(4, 3, 12), [0.05, 0.06, 0.07, 0.08])
        L = _lib.make_layout(*dims)
        segs = [Seg(L, make_episodes(rng, 30, dims), 64, t) for t in (-1, 3)]
        d = _lib.NetDesc(1, 20, 12, 4, 4, 128, 2, 1.0, 1, 5.0)
        return Case(dims, tk, _lib.MODE_BUFFER, segs, clip_obs=0.75, relative_goals=True), d, None
    if name == 'info-reward-injected':
        dims = (12, 40, 12, 12, 4, 4, 12, 3)
        tk = Tasks(slices(4, 3, 12), slices(4, 3, 12), [0.05] * 4, kinds=['distance', 'distance', 'info', 'pair'],
                   ref_ids=[None, None, None, [11, 10, 9]], diminfo=3)
        segs = [Seg(_lib.make_layout(*dims), make_episodes(rng, 10, dims), 4)]
        d = dict(ep=rng.randint(0, 10, 4), t=rng.randint(0, 12, 4), u_her=np.array([0.1, 0.9, 0.5, 0.2]),
                 u_off=rng.uniform(size=4), choice=np.array([2, 0, 3, 2]))
        return Case(dims, tk, _lib.MODE_RANDOM_TASK, segs, clip_obs=1.0), _net(1, 40, 12, 4, 4, 256, 3), d
    if name == 'flat-1024':
        dims = (25, 20, 12, 12, 4, 0, 0, 0)
        tk = Tasks(slices(4, 3, 12), [[2, 1, 0], [5, 4, 3], [8, 7, 6], [11, 10, 9]], [0.05] * 4, flat_threshold=0.1)
        segs = [Seg(_lib.make_layout(*dims), make_episodes(rng, 60, dims), 1024)]
        return Case(dims, tk, _lib.MODE_FLAT, segs, clip_obs=1.0), _net(0, 20, 12, 4, 0, 256, 2), None
    if name == 'control-block-step':
        dims = (14, 12, 8, 8, 8, 4, 0, 0)
        tk = Tasks(slices(4, 2, 8, rng), slices(4, 2, 8, rng), [0.05] * 4)
        L = _lib.make_layout(*dims)
        segs = [Seg(L, make_episodes(rng, 40, dims), c) for c in (100, 100, 312)]
        return Case(dims, tk, _lib.MODE_CURRENT_TASK, segs, clip_obs=1.0), _net(1, 12, 8, 8, 4, 64, 3), 'dyn'
    if name == 'widest-stage-arm4-dimo200':
        from curious_b200 import synth
        ag_ids, g_ids = synth.arm_task_ids(4)
        dims = (50, 200, 12, 12, 4, 4, 12, 1)
        tk = Tasks(g_ids, ag_ids, [0.05] * 4)
        L = _lib.make_layout(*dims)
        assert stage_floats(L, False) == 444
        segs = [Seg(L, make_episodes(rng, 8, dims), c, t) for c, t in ((128, 2), (128, -1))]
        return Case(dims, tk, _lib.MODE_BUFFER, segs, clip_obs=1.5), _net(1, 200, 12, 4, 4, 256, 3), None
    raise KeyError(name)


FUSED_CASES = ['16-modules-cp', '17-segments', 'relative-clip-normalize', 'info-reward-injected', 'flat-1024',
               'control-block-step', 'widest-stage-arm4-dimo200']


def _rows_update(d, n, theta, target, stats, step, her=None, batch=None):
    """One cur_ddpg_rows_step (gradients only) on fresh NaN-filled outputs with the step counter at 3."""
    import torch
    lib = _lib.load()
    _, total = _arena(d)
    grads = torch.full((total,), float('nan'), device='cuda')
    q_ring, pi_ring = (torch.full((4,), float('nan'), device='cuda') for _ in range(2))
    q_pi = torch.full((n + GUARD,), float('nan'), device='cuda')
    ws = torch.zeros(lib.cur_ddpg_rows_workspace_floats(C.byref(d), n), dtype=torch.float32, device='cuda')
    step.fill_(3)
    h = _lib.DdpgHyper(gamma=0.98, clip_return=3.0, action_l2=0.5, clip_pos_returns=1, step_counter=step.data_ptr(),
                       loss_ring=4, micro_batches=0, grads_parity_stride=0, loss_rows=0, transposes_valid=0)
    cb = batch if batch is not None else _lib.Batch(None, None, None, None, None, None, None, n)
    _lib.check(lib.cur_ddpg_rows_step(_lib.stream_ptr(), C.byref(d), theta.data_ptr(), target.data_ptr(),
                                      C.byref(stats[0]) if stats else None, C.byref(cb), C.byref(h), ws.data_ptr(),
                                      grads.data_ptr(), q_ring.data_ptr(), pi_ring.data_ptr(), q_pi.data_ptr(), None,
                                      C.byref(her) if her is not None else None), 'cur_ddpg_rows_step')
    torch.cuda.synchronize()
    return dict(grads=grads.cpu().numpy(), q_ring=q_ring.cpu().numpy(), pi_ring=pi_ring.cpu().numpy(),
                q_pi=q_pi.cpu().numpy(), step=int(step.item()))


def _arena(d):
    total = C.c_int64(0)
    pi = _lib.load().cur_theta_pi_offset(C.byref(d), C.byref(total))
    return pi, total.value


@pytest.mark.gpu
@pytest.mark.parametrize('name', FUSED_CASES)
def test_fused_prologue_equals_standalone_sampler(name):
    """cur_ddpg_rows_step sampling its own rows (her != NULL) against the same update fed the batch cur_her_sample
    produced from the same args: gradients, loss rings, Q_pi and the step counter bit for bit."""
    import torch
    lib = _lib.load()
    case, d, extra = _fused_case(name)
    n = case.B
    _, total = _arena(d)
    rng = np.random.RandomState(n)
    scale = float(np.sqrt(6.0 / (2 * d.hidden)))
    theta, target = (torch.from_numpy(rng.uniform(-scale, scale, total).astype(F32)).cuda() for _ in range(2))
    stats = None
    if d.normalize_obs:
        keep = [torch.from_numpy(v.astype(F32)).cuda() for v in (rng.normal(0, 0.3, d.dimo), rng.uniform(0.5, 2, d.dimo),
                                                                   rng.normal(0, 0.3, d.dimg), rng.uniform(0.5, 2, d.dimg))]
        stats = (_lib.NormStats(*[t.data_ptr() for t in keep]), keep)
    step = torch.zeros(1, dtype=torch.int64, device='cuda')
    draws = upload_draws(extra) if isinstance(extra, dict) else None
    dyn_dev = None
    if extra == 'dyn':
        counts, sizes = [0, 200, 312], [1, 17, 40]
        dyn = _lib.HerDyn()
        dyn.step = step.data_ptr()
        for i in range(3):
            dyn.count[i], dyn.n_episodes[i] = counts[i], sizes[i]
        dyn_dev = torch.frombuffer(bytearray(dyn), dtype=torch.uint8).cuda()
    her = case.args(draws=draws)
    if dyn_dev is not None:
        her.dyn = dyn_dev.data_ptr()
    assert lib.cur_ddpg_rows_her_supported(C.byref(d), C.byref(her)) == 1
    fused = _rows_update(d, n, theta, target, stats, step, her=her)
    # the standalone sampler into a batch, then the same update reading it
    keys = ('o', 'g', 'u', 'td', 'o_2', 'g_2', 'r')
    outs = {k: torch.full((n, case.dim(k)), float('nan'), device='cuda') for k in keys if case.dim(k) > 0}
    a = case.args(outs, draws)
    if dyn_dev is not None:
        a.dyn = dyn_dev.data_ptr()
    step.fill_(3)
    _lib.check(lib.cur_her_sample(_lib.stream_ptr(), C.byref(a)), 'cur_her_sample')
    cb = _lib.Batch(outs['o'].data_ptr(), outs['g'].data_ptr(), outs['u'].data_ptr(), _lib.ptr(outs.get('td')),
                    outs['o_2'].data_ptr(), outs['g_2'].data_ptr(), outs['r'].data_ptr(), n)
    unfused = _rows_update(d, n, theta, target, stats, step, batch=cb)
    assert np.isfinite(fused['q_pi'][:n]).all() and np.isnan(fused['q_pi'][n:]).all()
    for k in ('grads', 'q_ring', 'pi_ring', 'q_pi'):
        assert np.array_equal(fused[k], unfused[k], equal_nan=True), (name, k)
    assert fused['step'] == unfused['step'] == 4
    r = outs['r'].cpu().numpy()
    assert n < 8 or set(np.unique(r)) == {-1.0, 0.0}
