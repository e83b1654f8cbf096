"""structure='task_experts' acting: an evaluation step routes each row to the expert of its module in ONE launch
(TaskExperts.get_actions -> cur_ddpg_actions_rows_group), bit for bit the loop of one-row get_actions calls it stands for
(rollout.py:211-223): actions, Q, the np.random stream and every expert's device-noise counter.  Also against the NumPy
oracle, through RolloutWorker(eval=True) on whole rollouts, and the refusals / fall-backs on the CPU.  Every GPU test
carries its own mark."""
import ctypes as C

import numpy as np
import pytest

from tests.ddpg_util import ddpg_kwargs, episode_stream, make_gpu_agent, make_oracle_agent


def _loop(policies, o, ag, g, td, **kw):
    """The per-row loop the routed launch stands for (rollout.py:211-223 as RolloutWorker._act wrote it)."""
    u = np.zeros((len(o), policies[0].dimu))
    q = np.zeros((len(o), 1))
    for i in range(len(o)):
        out = policies[int(np.argmax(td[i]))].get_actions(o[i:i + 1], ag[i:i + 1], g[i:i + 1], task_descr=td[i:i + 1], **kw)
        if kw.get('compute_Q'):
            u[i], q[i, 0] = out[0], np.asarray(out[1]).reshape(-1)[0]
        else:
            u[i] = out
    return [u, q] if kw.get('compute_Q') else u


def _experts(n_exp, n_modules, hidden, normalize_obs, relative_goals, **extra):
    kw, dims, ag_ids, g_ids = ddpg_kwargs(n_modules, structure='task_experts', task_replay='replay_current_task_buffer',
                                          hidden=hidden, normalize_obs=normalize_obs, relative_goals=relative_goals)
    ps = []
    for t in range(n_exp):
        k = dict(kw)
        k['t_id'] = t
        p = make_gpu_agent(k, dims, ag_ids, g_ids, seed=30 + t, **extra)
        # per-expert statistics and a target net that differs from the main one
        p.o_stats.load_state_list([np.zeros(dims['o']), np.zeros(dims['o']), np.ones(1),
                                   np.linspace(-0.5, 0.5, dims['o']) + 0.1 * t, np.linspace(0.5, 2.0, dims['o']) + 0.2 * t])
        p.g_stats.load_state_list([np.zeros(dims['g']), np.zeros(dims['g']), np.ones(1),
                                   np.linspace(-0.1, 0.1, dims['g']) - 0.05 * t, np.linspace(0.05, 0.3, dims['g']) + 0.1 * t])
        p.set_flat('Q', p.get_flat('Q') * 1.5, target=True)
        p.set_flat('pi', p.get_flat('pi') * 0.5, target=True)
        ps.append(p)
    return ps, dims


def _inputs(rng, dims, n, n_modules, modules):
    o = rng.standard_normal((n, dims['o'])).astype(np.float32) * 3
    g = rng.uniform(-0.3, 0.3, (n, dims['g'])).astype(np.float32)
    ag = rng.uniform(-0.3, 0.3, (n, dims['ag'])).astype(np.float32)
    td = np.eye(n_modules, dtype=np.float32)[modules]
    return o, ag, g, td


def _same(a, b):
    if isinstance(a, list):
        return all(np.array_equal(x, y) and x.dtype == y.dtype and x.shape == y.shape for x, y in zip(a, b))
    return np.array_equal(a, b) and a.dtype == b.dtype and a.shape == b.shape


# (experts, modules, hidden, pad_hidden, normalize_obs, relative_goals, action_noise)
CASES = [(3, 4, 64, 'native', False, False, 'host'),
         (4, 4, 128, 'native', True, True, 'host'),
         (5, 8, 256, 'auto', True, False, 'host'),
         (4, 4, 64, True, False, True, 'host'),          # zero-padded to 256
         (4, 4, 256, 'auto', False, True, 'device'),
         (3, 8, 128, 'native', True, False, 'device')]


@pytest.mark.gpu
@pytest.mark.parametrize('case', range(len(CASES)))
def test_routed_actions_equal_the_per_row_loop(monkeypatch, case):
    """The routed launch against the loop on the same experts and inputs, np.random seeded alike: u, q (dtype and shape
    too), the np.random state afterwards and - device noise - every expert's _action_calls.  Mixed modules per step, one
    expert taking every row, n = 1 ... 512, compute_Q and use_target_net on and off, non-zero and zero eps."""
    from curious_b200 import _lib
    from curious_b200.experts import TaskExperts
    n_exp, n_mod, hidden, pad, normalize_obs, relative_goals, noise = CASES[case]
    ps, dims = _experts(n_exp, n_mod, hidden, normalize_obs, relative_goals, pad_hidden=pad, action_noise=noise)
    te = TaskExperts(ps)
    assert te._routed_ok()
    calls = []
    lib = _lib.load()
    fn = lib.cur_ddpg_actions_rows_group
    monkeypatch.setattr(lib, 'cur_ddpg_actions_rows_group', lambda *a: (calls.append(1), fn(*a))[1])
    rng = np.random.RandomState(100 + case)
    for n in (1, 2, 38, 100, 512):
        for spread in ('mixed', 'one'):
            modules = rng.randint(0, n_exp, n) if spread == 'mixed' else np.full(n, rng.randint(0, n_exp))
            o, ag, g, td = _inputs(rng, dims, n, n_mod, modules)
            for compute_Q in (False, True):
                for use_target in (False, True):
                    for eps in ((0.2, 0.3), (0., 0.)):
                        kw = dict(noise_eps=eps[0], random_eps=eps[1], use_target_net=use_target, compute_Q=compute_Q)
                        before = [p._action_calls for p in ps]
                        np.random.seed(n + 7)
                        want = _loop(ps, o, ag, g, td, **kw)
                        st_loop = np.random.get_state()
                        after = [p._action_calls for p in ps]
                        for p, c in zip(ps, before):
                            p._action_calls = c
                        np.random.seed(n + 7)
                        got = te.get_actions(o, ag, g, td, **kw)
                        st_routed = np.random.get_state()
                        what = (n, spread, compute_Q, use_target, eps)
                        assert _same(got, want), what
                        assert np.array_equal(st_loop[1], st_routed[1]) and st_loop[2:] == st_routed[2:], what
                        assert [p._action_calls for p in ps] == after, what
                        if noise == 'device':
                            assert after == [c + int((modules == e).sum()) for e, c in enumerate(before)], what
    assert len(calls) == 5 * 2 * 2 * 2 * 2                 # every step above was ONE routed launch
    # the experts act differently: a routing mistake could not pass unnoticed
    o, ag, g, td = _inputs(rng, dims, 4, n_mod, np.zeros(4, int))
    u0 = te.get_actions(o, ag, g, td)
    u1 = te.get_actions(o, ag, g, np.roll(td, 1, axis=1))
    assert not np.array_equal(u0, u1)


@pytest.mark.gpu
@pytest.mark.parametrize('hidden,pad,n_modules', [(64, 'native', 4), (128, 'native', 8), (256, 'auto', 4)])
def test_routed_actions_against_oracle(hidden, pad, n_modules):
    """Each expert's rows of a routed step against that expert's oracle forward (its weights, its statistics), with the
    tolerance of test_ddpg_gpu.py::test_get_actions_against_oracle."""
    from curious_b200.experts import TaskExperts
    n_exp = 3
    kw, dims, ag_ids, g_ids = ddpg_kwargs(n_modules, structure='task_experts', task_replay='replay_current_task_buffer',
                                          hidden=hidden, normalize_obs=True, relative_goals=True)
    episodes = episode_stream(dims, kw['T'], 3)
    oras, gpus = [], []
    for t in range(n_exp):
        k = dict(kw)
        k['t_id'] = t
        ora = make_oracle_agent(k, dims, ag_ids, g_ids, seed=40 + t)
        gpu = make_gpu_agent(k, dims, ag_ids, g_ids, seed=40 + t, pad_hidden=pad)
        for a in (ora, gpu):
            np.random.seed(60 + t)
            n = 0
            for ep in episodes[:t + 1]:                             # different statistics per expert
                n += 2
                a.store_episode({key: v.copy() for key, v in ep.items()}, np.zeros(n_modules), n)
        for a, b in ((gpu.o_stats, ora.o_stats), (gpu.g_stats, ora.g_stats)):
            a.load_state_list([b.sum, b.sumsq, b.count, b.mean, b.std])
        oras.append(ora)
        gpus.append(gpu)
    te = TaskExperts(gpus)
    rng = np.random.RandomState(5)
    for n in (1, 2, 38, 100, 512):
        modules = rng.randint(0, n_exp, n)
        o = rng.standard_normal((n, dims['o'])).astype(np.float32) * 100
        g = rng.uniform(-1, 1, (n, dims['g'])).astype(np.float32)
        ag = rng.uniform(-1, 1, (n, dims['ag'])).astype(np.float32)
        td = np.eye(n_modules, dtype=np.float32)[modules]
        for use_target in (False, True):
            u, q = te.get_actions(o, ag, g, td, use_target_net=use_target, compute_Q=True)
            for e in range(n_exp):
                rows = np.flatnonzero(modules == e)
                if len(rows) == 0:
                    continue
                u_o, q_o = oras[e].get_actions(o[rows], ag[rows], g[rows], task_descr=td[rows], use_target_net=use_target,
                                               compute_Q=True)
                tol = 1e-6 if n < 100 else 1e-5
                assert np.allclose(u[rows], np.asarray(u_o).reshape(len(rows), -1), rtol=1e-5, atol=tol), (n, e)
                assert np.allclose(q[rows], np.asarray(q_o).reshape(len(rows), 1), rtol=1e-5, atol=tol), (n, e)


@pytest.mark.gpu
@pytest.mark.parametrize('rollout_batch_size', [2, 38])
def test_evaluator_routed_equals_the_loop(rollout_batch_size):
    """RolloutWorker(eval=True) over the experts of make_experiment on envs.ModularPointEnv, whole rollouts: once through
    the routed launch, once through the per-row loop.  Episodes, Q values, competence records and np.random agree."""
    from curious_b200.train import make_experiment
    runs = []
    for forced_loop in (False, True):
        exp = make_experiment(nb_tasks=4, structure='task_experts', task_selection='active_competence_progress',
                              task_replay='replay_current_task_buffer', buffer_size=20000, rollout_batch_size=rollout_batch_size,
                              seed=3)
        ev = exp['evaluator']
        for i, p in enumerate(exp['policy']):                  # the experts share the seed: make them act differently
            p.set_flat('pi', p.get_flat('pi') * (1.0 + 0.5 * i))
            p.set_flat('Q', p.get_flat('Q') * (1.0 - 0.1 * i))
            p.set_flat('pi', p.get_flat('pi') * 0.8, target=True)
        if forced_loop:
            ev._router = (ev.policy, None)
        else:
            assert ev._expert_router() is not None
        np.random.seed(11)
        eps = [ev.generate_rollouts()[0] for _ in range(3)]
        runs.append((eps, list(ev.Q_history), list(ev.success_history), np.array(ev.get_C()), ev.tracker.state(),
                     np.random.get_state()))
    (ea, qa, sa, ca, ta, ra), (eb, qb, sb, cb, tb, rb) = runs
    for x, y in zip(ea, eb):
        assert x.keys() == y.keys()
        for key in x:
            assert x[key].dtype == y[key].dtype and np.array_equal(x[key], y[key]), key
    assert qa == qb and sa == sb and np.array_equal(ca, cb)
    assert repr(ta) == repr(tb)
    assert np.array_equal(ra[1], rb[1]) and ra[2:] == rb[2:]


# ------------------------------------------------------------------------------------------------ CPU
def test_actions_rows_group_refuses_bad_arguments():
    """Every refusal returns a non-zero status and a message before any device call, so it runs without a GPU (the
    pointers are never dereferenced)."""
    from curious_b200 import _lib
    lib = _lib.load()

    def desc(hidden=64, layers=3):
        return _lib.NetDesc(1, 40, 12, 4, 4, hidden, layers, 1.0, 0, 5.0)

    fake = 0x10000000
    experts = (_lib.ActionsExpert * 17)()
    for e in experts:
        e.theta = fake

    def refused(d, n_experts, rows, n=None):
        which = np.asarray(rows, np.int32)
        n = len(which) if n is None else n
        status = lib.cur_ddpg_actions_rows_group(None, C.byref(d), n_experts, experts, which.ctypes.data, fake, None, fake,
                                                 fake, n, 200.0, fake, fake, 1)
        return status != 0 and bool(lib.cur_last_error())

    for hidden in (64, 128, 256):
        assert lib.cur_ddpg_rows_supported(C.byref(desc(hidden)), 4) == 1
        assert refused(desc(hidden), 0, [0, 0])                             # n_experts outside 1..16
        assert refused(desc(hidden), 17, [0, 16])
        assert refused(desc(hidden), 3, [0, 3, 1])                          # row_expert out of range
        assert refused(desc(hidden), 3, [0, -1, 1])
        assert refused(desc(hidden), 2, np.zeros(513, np.int32))            # above 512 rows
        assert refused(desc(hidden), 2, [0], n=0)
    for d in (desc(96), desc(64, layers=5)):                                # shapes the rows schedule does not take
        assert lib.cur_ddpg_rows_supported(C.byref(d), 4) == 0
        assert refused(d, 2, [0, 1])
    seeds = np.zeros(2, np.uint64)
    assert lib.cur_action_noise_rows(None, None, 2, 4, 1.0, 0.1, 0.1, seeds.ctypes.data, seeds.ctypes.data) != 0
    assert lib.cur_action_noise_rows(None, fake, 2, 4, 1.0, 0.1, 0.1, None, seeds.ctypes.data) != 0


class _StandIn(object):
    """A DDPG look-alike for the host logic of TaskExperts.get_actions: records its one-row calls."""
    ACTION_ROWS_MAX = 512

    def __init__(self, t, rows_ok, log):
        from curious_b200 import _lib
        self.t, self.rows_ok, self.log = t, rows_ok, log
        self.net = type('Net', (), {'desc': _lib.NetDesc(1, 10, 3, 4, 2, 64, 3, 1.0, 0, 5.0)})()
        self.batch_size, self.device = 256, 'cpu'
        self.dimo, self.dimg, self.dimu = 10, 3, 4
        self.clip_obs, self.relative_goals, self.modular, self.action_noise = 200., False, True, 'host'

    def _action_rows_ok(self):
        return self.rows_ok

    def get_actions(self, o, ag, g, task_descr=None, noise_eps=0., random_eps=0., use_target_net=False, compute_Q=False):
        assert o.shape == (1, self.dimo) and task_descr.shape == (1, 2)
        self.log.append(self.t)
        u = np.full(self.dimu, self.t, np.float32) + np.random.randn(self.dimu).astype(np.float32)
        return [u, np.full((1, 1), -self.t, np.float32)] if compute_Q else u


@pytest.mark.parametrize('n,rows_ok', [(513, True), (2, False), (40, False)])
def test_expert_actions_fall_back_to_the_loop(monkeypatch, n, rows_ok):
    """More than ACTION_ROWS_MAX rows, or an expert off the one-launch path (action_path='levels'): the per-row loop, in
    row order, by the row's expert; no routed launch is attempted."""
    from curious_b200 import experts as X
    monkeypatch.setattr(X, '_Route', lambda *a: pytest.fail('routed launch attempted'))
    log = []
    te = X.TaskExperts([_StandIn(0, True, log), _StandIn(1, rows_ok, log)])
    rng = np.random.RandomState(0)
    modules = rng.randint(0, 2, n)
    o = rng.standard_normal((n, 10)).astype(np.float32)
    ag = g = np.zeros((n, 3), np.float32)
    td = np.eye(2, dtype=np.float32)[modules]
    np.random.seed(1)
    u, q = te.get_actions(o, ag, g, td, compute_Q=True)
    np.random.seed(1)
    want = _loop(te.policies, o, ag, g, td, compute_Q=True)
    assert log == list(modules) * 2
    assert _same([u, q], want) and u.dtype == np.float64 and q.shape == (n, 1)


def test_rollout_keeps_the_loop_for_other_policy_lists():
    """RolloutWorker routes only lists of DDPG agents of one shape; anything else keeps the loop."""
    from curious_b200.experts import TaskExperts
    log = []
    assert TaskExperts.router([_StandIn(0, True, log), _StandIn(1, True, log)]) is None
    assert TaskExperts.router(object()) is None
    assert TaskExperts.router([]) is None
