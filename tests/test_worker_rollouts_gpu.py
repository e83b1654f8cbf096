"""Virtual workers on the GPU: the noisy action launch (cur_ddpg_actions_rows_noisy) against the action launch +
cur_action_noise of each worker, DDPG.get_actions_workers against a lone agent per worker, and make_experiment /
train() with workers_per_rank=k end to end."""
import ctypes as C

import numpy as np
import pytest
import torch

from tests.ddpg_util import ddpg_kwargs, make_gpu_agent

pytestmark = pytest.mark.gpu

NOISE_EPS, RANDOM_EPS = 0.2, 0.3


def _agent(hidden, **extra):
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4, hidden=hidden)
    if hidden != 256:
        extra['pad_hidden'] = 'native'
    return make_gpu_agent(kw, dims, ag_ids, g_ids, buffer_episodes=4, seed=2, **extra), dims


def _inputs(dims, n, seed):
    rng = np.random.RandomState(seed)
    o = rng.randn(n, dims['o']).astype(np.float32)
    g = rng.randn(n, dims['g']).astype(np.float32)
    td = np.eye(dims['task_descr'], dtype=np.float32)[rng.randint(0, dims['task_descr'], n)]
    return [torch.from_numpy(x.reshape(-1)).cuda() for x in (o, g, td)], (o, g, td)


@pytest.mark.parametrize('hidden', [64, 128, 256])
@pytest.mark.parametrize('compute_Q', [False, True])
@pytest.mark.parametrize('B', [1, 2])
@pytest.mark.parametrize('k', [1, 3, 19])
def test_noisy_launch_is_launch_plus_noise_per_worker(k, B, compute_Q, hidden):
    """Worker j's rows == cur_action_noise(u_j, B, ..., key_j, call_j) after the plain launch, bit for bit; a worker with
    noisy = 0 keeps the noise-free action; a zero-noise call is the plain launch.  Q is the noise-free action's."""
    from curious_b200 import _lib
    lib = _lib.load()
    a, dims = _agent(hidden)
    n, du = k * B, a.dimu
    (o, g, td), _ = _inputs(dims, n, 10 * k + B)
    s = _lib.stream_ptr()
    keys = [(1000003 * (j + 1)) ^ (0xABCDEF << 40) for j in range(k)]
    calls = [7 + 3 * j for j in range(k)]
    noisy = [j % 3 != 1 for j in range(k)]                    # worker 1, 4, ... exploit

    def launch(noise, ne, re):
        out = torch.full((n * (du + 1),), float('nan'), device='cuda')
        q = out.data_ptr() + 4 * n * du if compute_Q else None
        args = (s, C.byref(a.net.desc), a.theta_main.data_ptr(), C.byref(a._stats), o.data_ptr(), None, g.data_ptr(),
                td.data_ptr(), n, float(a.clip_obs))
        if noise is None:
            _lib.check(lib.cur_ddpg_actions_rows(*args, out.data_ptr(), q, 0), 'plain')
        else:
            _lib.check(lib.cur_ddpg_actions_rows_noisy(*args, ne, re, noise, out.data_ptr(), q, 0), 'noisy')
        return out

    rows = (_lib.NoiseRow * n)()
    for j in range(k):
        for i in range(B):
            rows[j * B + i] = _lib.NoiseRow(keys[j], calls[j], i, 1 if noisy[j] else 0)
    rows_dev = torch.frombuffer(bytearray(rows), dtype=torch.uint8).cuda()
    want = launch(None, 0., 0.)
    for j in range(k):
        if noisy[j]:
            _lib.check(lib.cur_action_noise(s, want.data_ptr() + 4 * j * B * du, B, du, float(a.max_u), NOISE_EPS, RANDOM_EPS,
                                            keys[j], calls[j]), 'cur_action_noise')
    got = launch(rows_dev.data_ptr(), NOISE_EPS, RANDOM_EPS)
    torch.cuda.synchronize()
    m = n * (du + (1 if compute_Q else 0))
    assert torch.equal(got[:m].view(torch.int32), want[:m].view(torch.int32))
    assert any(noisy) and not torch.equal(got[:n * du], launch(None, 0., 0.)[:n * du]) or not any(noisy)
    # zero noise: the plain launch
    plain = launch(None, 0., 0.)
    zero = launch(rows_dev.data_ptr(), 0., 0.)
    torch.cuda.synchronize()
    assert torch.equal(zero[:m].view(torch.int32), plain[:m].view(torch.int32))


def test_noisy_launch_refusals():
    """Refused before any launch: a shape the row kernels do not take, n outside 1..512, bad noise parameters, no rows."""
    from curious_b200 import _lib
    lib = _lib.load()
    a, dims = _agent(256)
    (o, g, td), _ = _inputs(dims, 4, 0)
    rows = torch.zeros(24 * 600, dtype=torch.uint8, device='cuda')
    out = torch.zeros(600 * 9, device='cuda')

    def call(desc, n, ne=0.2, re=0.3, r=rows.data_ptr()):
        return lib.cur_ddpg_actions_rows_noisy(_lib.stream_ptr(), C.byref(desc), a.theta_main.data_ptr(), C.byref(a._stats),
                                               o.data_ptr(), None, g.data_ptr(), td.data_ptr(), n, 200., ne, re, r,
                                               out.data_ptr(), None, 0)
    d = a.net.desc
    bad_h = _lib.NetDesc.from_buffer_copy(d)
    bad_h.hidden = 96
    bad_u = _lib.NetDesc.from_buffer_copy(d)
    bad_u.dimu = 9
    for status in (call(d, 0), call(d, 513), call(bad_h, 4), call(bad_u, 4), call(d, 4, ne=-1.), call(d, 4, re=1.5),
                   call(d, 4, r=None)):
        assert status == 1                                   # CUR_ERR_INVALID
    torch.cuda.synchronize()
    assert torch.count_nonzero(out) == 0


@pytest.mark.parametrize('noise', ['host', 'device'])
@pytest.mark.parametrize('k,B', [(3, 2), (19, 2), (19, 4)])
def test_get_actions_workers_equals_lone_agents(k, B, noise):
    """DDPG.get_actions_workers == a lone agent of each worker's reference rank (same weights; its np.random stream for host
    noise, its key and call number for device noise), for exploring and exploiting workers, over several calls; every
    worker's stream ends where the lone agent's does.  k = 19, B = 4 (76 rows) runs through device memory."""
    import copy
    from curious_b200.workers import WorkerStreams
    own, dims = _agent(256, action_noise=noise)
    lone, _ = _agent(256, action_noise=noise)
    streams = WorkerStreams(5, k)
    ref = copy.deepcopy(streams)
    n = k * B
    for step in range(4):
        _, (o, g, td) = _inputs(dims, n, 100 + step)
        exploit = [(j + step) % 4 == 0 for j in range(k)]
        ne = [0. if x else NOISE_EPS for x in exploit]
        re = [0. if x else RANDOM_EPS for x in exploit]
        compute_Q = step % 2 == 1
        u, q = own.get_actions_workers(o, o[:, :3], g, td, noise_eps=ne, random_eps=re, streams=streams, compute_Q=compute_Q)
        for j in range(k):
            rows = slice(j * B, (j + 1) * B)
            lone.noise_seed, lone._action_calls = streams.philox_key(j), step
            with ref.use(j):
                out = lone.get_actions(o[rows], o[rows, :3], g[rows], task_descr=td[rows], noise_eps=ne[j],
                                       random_eps=re[j], compute_Q=compute_Q)
            lu, lq = (out[0], out[1]) if compute_Q else (out, None)
            assert np.array_equal(u[rows], np.asarray(lu).reshape(B, -1)), (step, j)
            assert u.dtype == np.asarray(lu).dtype
            if compute_Q:
                assert np.array_equal(q[rows], np.asarray(lq).reshape(B, 1)), (step, j)
    assert own._action_calls == (4 if noise == 'device' else 0)
    for j in range(k):
        st, want = streams.state(j), ref.state(j)
        assert np.array_equal(st[1], want[1]) and st[2:] == want[2:], j


# ------------------------------------------------------------------------------------------------ end to end
def _experiment(seed=3, **kw):
    from curious_b200.train import make_experiment
    args = dict(nb_tasks=4, structure='curious', task_selection='active_competence_progress',
                task_replay='replay_task_cp_buffer', buffer_size=20000, n_cycles=3, n_batches=8, n_test_rollouts=2,
                seed=seed)
    args.update(kw)
    return make_experiment(**args)


def _run(exp, n_epochs=2, logdir=None):
    from curious_b200.train import train
    hist = train(n_epochs=n_epochs, logdir=logdir, initial_evaluation=False, clear_eval_competence=True, **exp)
    torch.cuda.synchronize()
    return hist


def test_one_worker_is_todays_run(tmp_path):
    """make_experiment(workers_per_rank=1) + train() == the default experiment from the same seed: history, progress.csv,
    losses and final parameters bit for bit."""
    runs = []
    for i, extra in enumerate(({}, {'workers_per_rank': 1})):
        np.random.seed(0)
        exp = _experiment(**extra)
        hist = _run(exp, logdir=str(tmp_path / str(i)))
        rows = open(str(tmp_path / str(i) / 'progress.csv')).read().splitlines()
        pol = exp['policy']
        runs.append((hist, [r.split(',')[:-1] for r in rows], pol.get_flat('Q'), pol.get_flat('pi'),
                     [float(v) for _, v in pol.logs()]))
    (h0, r0, q0, p0, l0), (h1, r1, q1, p1, l1) = runs
    for a, b in zip(h0, h1):
        for key in a:
            assert np.array_equal(np.asarray(a[key]), np.asarray(b[key])), key
    assert r0 == r1                                          # every column but the wall-clock Time
    assert np.array_equal(q0, q1) and np.array_equal(p0, p1) and l0 == l1


def _recording(worker):
    """Wrap generate_rollouts so that every episode batch it returns is kept."""
    episodes = []
    real = worker.generate_rollouts

    def gen():
        ep, cp, n = real()
        episodes.append({key: v.copy() for key, v in ep.items()})
        return ep, cp, n
    worker.generate_rollouts = gen
    return episodes


def test_three_workers_end_to_end():
    """k = 3: worker j's buffers hold exactly worker j's rollouts, two runs from one seed are identical, and
    device-noise runs too."""
    from curious_b200 import apportion
    k = 3
    runs = []
    for _ in range(2):
        exp = _experiment(workers_per_rank=k)
        assert exp['params']['num_cpu'] == k and len(exp['rollout_worker'].envs) == k * 2
        episodes = _recording(exp['rollout_worker'])
        hist = _run(exp)
        runs.append((hist, exp, episodes))
    (h0, e0, eps0), (h1, e1, _) = runs
    for a, b in zip(h0, h1):
        for key in a:
            assert np.array_equal(np.asarray(a[key]), np.asarray(b[key])), key
    for which in ('Q', 'pi'):
        assert np.array_equal(e0['policy'].get_flat(which), e1['policy'].get_flat(which))
    pol, rb = e0['policy'], 2
    for j in range(k):
        mine = [ep['u'][b].astype(np.float64) for ep in eps0 for b in range(j * rb, (j + 1) * rb)]
        routed = sum(len(apportion.active_modules(ep['change'][b, -1], pol.tasks_ag_id, pol.tasks_g_id))
                     for ep in eps0 for b in range(j * rb, (j + 1) * rb))
        bufs = pol.worker_buffer_set(j)
        assert sum(b.current_size for b in bufs[1:]) == routed > 0
        for b in bufs[1:]:
            stored = b.buffers['u'][:b.current_size]
            for s in stored:
                assert any(np.array_equal(s, m) for m in mine), j     # only worker j's rollouts
    # device-side noise: one noisy launch per step
    np.random.seed(0)
    exp = _experiment(workers_per_rank=k, policy_kwargs=dict(action_noise='device'))
    hist = _run(exp, n_epochs=1)
    assert exp['policy']._action_calls == (3 + 2) * exp['rollout_worker'].T and np.isfinite(hist[0]['test_mean_Q'])


def test_three_workers_learn_reach():
    """A short k = 3 run on ModularPointEnv learns the reach module, as the one-worker loop does (test_train_loop_gpu)."""
    from curious_b200.train import make_experiment, train
    np.random.seed(0)
    exp = make_experiment(nb_tasks=4, n_controllable=3, structure='curious', task_selection='active_competence_progress',
                          task_replay='replay_task_cp_buffer', buffer_size=100000, n_cycles=10, n_batches=40,
                          n_test_rollouts=10, seed=0, workers_per_rank=3)
    hist = train(n_epochs=12, initial_evaluation=False, clear_eval_competence=True, **exp)
    C = np.array([h['C'] for h in hist])
    assert C[-3:, 0].mean() >= 0.8, C[:, 0]
    assert C[-3:, 3].mean() <= 0.3, C[:, 3]
    assert np.isfinite(exp['policy'].get_flat('Q')).all()


def test_train_refuses_what_the_learner_refuses(tmp_path):
    from curious_b200.train import make_experiment, train
    exp = _experiment(workers_per_rank=3)
    for extra in (dict(checkpoint_interval=1, logdir=str(tmp_path)), dict(resume=True, logdir=str(tmp_path))):
        with pytest.raises(ValueError):
            train(n_epochs=1, **extra, **exp)
    with pytest.raises(ValueError):                           # first-layer fan-in 21: not a shape of the action kernel
        make_experiment(nb_tasks=3, structure='curious', buffer_size=5000, workers_per_rank=3)
    with pytest.raises(ValueError):
        make_experiment(nb_tasks=3, structure='task_experts', task_replay='replay_current_task_buffer', buffer_size=5000,
                        workers_per_rank=3)
    import curious_b200.train as tr
    real = tr._world
    tr._world = lambda comm=None: (None, 2)
    try:
        with pytest.raises(ValueError):
            train(n_epochs=1, **exp)
    finally:
        tr._world = real
