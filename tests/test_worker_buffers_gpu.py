"""worker_buffers='own' on the GPU: a k-worker agent against k lone agents, each seeded as the reference rank the worker
stands for (rank_seed(seed, j): its np.random stream and its Philox key) and fed that worker's episodes."""
import contextlib

import numpy as np
import pytest

from tests.ddpg_util import ddpg_kwargs, episode_stream, make_gpu_agent, rel_err

pytestmark = pytest.mark.gpu

SEED = 3
SHAPES = {'arm4': dict(n_modules=4), 'arm8': dict(n_modules=8),
          'flat': dict(n_modules=4, structure='flat', task_replay='')}
ALL = ('o', 'g', 'u', 'td', 'o_2', 'g_2', 'r', 'ag', 'ag_2')


@contextlib.contextmanager
def _stream(states, j):
    saved = np.random.get_state()
    np.random.set_state(states[j])
    try:
        yield
    finally:
        states[j] = np.random.get_state()
        np.random.set_state(saved)


class Setup:
    """One k-worker agent and k lone agents with the same stores."""

    def __init__(self, k, shape, her_rng, buffer_episodes=6, **extra):
        from curious_b200.parallel import rank_seed
        kw, self.dims, ag_ids, g_ids = ddpg_kwargs(**SHAPES[shape], **{x: extra.pop(x) for x in ('hidden',) if x in extra})
        self.kw, self.k, self.flat = kw, k, shape == 'flat'
        self.cp = np.linspace(0.05, 0.3, len(g_ids))
        self.own = make_gpu_agent(kw, self.dims, ag_ids, g_ids, buffer_episodes=buffer_episodes, seed=SEED,
                                  her_rng=her_rng, workers_per_rank=k, worker_buffers='own', **extra)
        lone_extra = {x: v for x, v in extra.items() if x not in ('workers_mode',)}
        self.lone = []
        for j in range(k):
            a = make_gpu_agent(kw, self.dims, ag_ids, g_ids, buffer_episodes=buffer_episodes, seed=SEED, her_rng=her_rng,
                               **lone_extra)
            a.sample_transitions.seed = rank_seed(SEED, j)
            self.lone.append(a)
        self.states = [np.random.RandomState(rank_seed(SEED, j) % 2 ** 32).get_state() for j in range(k)]
        self.streams = [episode_stream(self.dims, kw['T'], 12, seed=100 + j, flat=self.flat) for j in range(k)]
        self.n_stored = 0

    def store(self, n_calls):
        for _ in range(n_calls):
            c = self.n_stored
            self.n_stored += 1
            eps = [self.streams[j][c] for j in range(self.k)]
            n = 2 * self.n_stored
            stacked = {key: np.concatenate([e[key] for e in eps]) for key in eps[0]}
            np.random.seed(1234 + c)
            caller = np.random.get_state()
            self.own.store_episode(stacked, self.cp, n)
            now = np.random.get_state()
            assert np.array_equal(now[1], caller[1]) and now[2:] == caller[2:], 'the caller stream moved'
            for j, a in enumerate(self.lone):
                with _stream(self.states, j):
                    a.store_episode({key: v.copy() for key, v in eps[j].items()}, self.cp, n)


def _bufs(b):
    return b if isinstance(b, list) else [b]


def _check_stores(s):
    import torch
    for j, lone in enumerate(s.lone):
        for mine, ref in zip(_bufs(s.own.worker_buffer_set(j)), _bufs(lone.buffer)):
            assert mine is not ref
            assert mine.current_size == ref.current_size and mine.n_transitions_stored == ref.n_transitions_stored
            n, L = ref.current_size, ref.layout
            assert torch.equal(mine.storage[:n * L.T * L.trans_stride], ref.storage[:n * L.T * L.trans_stride])
            assert torch.equal(mine.cold[:n * L.T * L.cold_stride], ref.cold[:n * L.T * L.cold_stride])
        st, want = s.own.worker_streams.state(j), s.states[j]
        assert np.array_equal(st[1], want[1]) and st[2:] == want[2:], j


def _check_batches(s, got, refs, what):
    B = s.kw['batch_size']
    for j, ref in enumerate(refs):
        for key in ref:
            if key == '_keep':
                continue
            assert np.array_equal(got[key][j * B:(j + 1) * B].cpu().numpy(), ref[key].cpu().numpy()), (what, j, key)


CASES = [(k, 'arm4', rng) for k in (1, 2, 3, 19) for rng in ('philox', 'numpy')] + \
        [(3, shape, rng) for shape in ('arm8', 'flat') for rng in ('philox', 'numpy')]


@pytest.mark.parametrize('k,shape,her_rng', CASES)
def test_sampler_and_stores_against_lone_agents(k, shape, her_rng):
    """Rows [256 j, 256 j + 256) of the k-worker batch == lone agent j's batch, bit for bit (every output and idx_out),
    at the 1st and 50th sampling call, with buffers partly filled and again past the random-overwrite point; the buffers,
    fill levels and np.random states of every worker == its lone agent's, the caller's stream untouched."""
    import torch
    s = Setup(k, shape, her_rng)
    for n_calls in (2, 8):                       # 6-episode buffers: partly filled, then overwritten at random slots
        s.store(n_calls)
        _check_stores(s)
        want = tuple(x for x in ALL if not (s.flat and x == 'td'))
        for call in range(50):
            got = s.own._sample_device(want, want_idx=True)
            refs = []
            for j, a in enumerate(s.lone):
                with _stream(s.states, j):
                    refs.append(a._sample_device(want, want_idx=True))
            if call in (0, 49):
                torch.cuda.synchronize()
                _check_batches(s, got, refs, (n_calls, call))
        _check_stores(s)


@pytest.mark.parametrize('k,shape', [(1, 'arm4'), (2, 'arm4'), (3, 'arm4'), (19, 'arm4'), (3, 'arm8'), (3, 'flat')])
def test_graph_sampler_against_lone_agents(k, shape):
    """Through the CUDA graph: the batch the k-worker update sampled at update 1 and update 50 == each lone agent's
    (its graph with the unfused sampler, so that the batch is materialised)."""
    import torch
    s = Setup(k, shape, 'philox')
    s.store(8)
    for a in s.lone:
        a.fuse_her = False
    B = s.kw['batch_size']
    for u in range(50):
        s.own.train()
        for a in s.lone:
            a.train()
        if u in (0, 49):
            torch.cuda.synchronize()
            for j, a in enumerate(s.lone):
                for key, t in a._gbatch.items():
                    if key == '_keep':              # the sampler's host references, not an output
                        continue
                    assert torch.equal(s.own._gbatch[key][j * B:(j + 1) * B], t), (u, j, key)


def test_normaliser_is_the_mean_over_workers():
    """After k-worker stores, mean / std == the reference's mean over k ranks (normalizer.py:84-118: running += summed
    partials / k) of the k lone agents' normaliser batches, within float32 summation order."""
    k = 3
    s = Setup(k, 'arm4', 'numpy')
    s.store(3)
    for name in ('o_stats', 'g_stats'):
        lone = [getattr(a, name).state_list() for a in s.lone]
        # each lone running sum is its own partials (count starts at 1): mean over ranks of the partials
        tot = sum(np.asarray(x[0], np.float64) for x in lone) / k
        totsq = sum(np.asarray(x[1], np.float64) for x in lone) / k
        cnt = 1.0 + sum(float(x[2][0]) - 1.0 for x in lone) / k
        mean = tot / cnt
        std = np.sqrt(np.maximum(s.own.o_stats.eps ** 2, totsq / cnt - mean ** 2))
        mine = getattr(s.own, name).state_list()
        assert abs(float(mine[2][0]) - cnt) <= 1e-6 * cnt
        assert rel_err(mine[3], mean) <= 1e-5, name
        assert rel_err(mine[4], std) <= 1e-5, name


@pytest.mark.parametrize('k,hidden', [(2, 256), (19, 256), (5, 64)])
def test_update_is_the_sum_of_the_workers_gradients(k, hidden):
    """Every update's gradient == the sum of the k lone agents' single-batch gradients (same weights, each from its own
    buffers and draws), over 4 updates (hidden 256: rows schedule at k = 2, chain at k = 19; hidden 64: narrow chain at
    k = 5); and the CUDA-graph update gives the same bits as the eager one on the same Philox stream."""
    import torch
    from curious_b200.ddpg import DDPG
    extra = dict(hidden=hidden)
    if hidden != 256:
        extra['pad_hidden'] = 'native'
    s = Setup(k, 'arm4', 'numpy', **extra)
    s.store(4)
    for step in range(4):
        lone_g = []
        for j, a in enumerate(s.lone):
            for which in ('Q', 'pi'):
                a.set_flat(which, s.own.get_flat(which))
            with _stream(s.states, j):
                a.stage_batch()
            a._grads()
            lone_g.append(a.grads.double())
        with np.errstate(all='ignore'):
            s.own.train()
        want = torch.stack(lone_g).sum(0)
        for which in ('Q', 'pi'):
            got = s.own._view(s.own.grads, which).cpu().numpy()
            ref = s.own._view(want, which).cpu().numpy()
            assert rel_err(got, ref) <= 5e-4, (step, which, rel_err(got, ref))
    # graph == eager, bit for bit
    agents = []
    for use_graph in (True, False):
        g = Setup(k, 'arm4', 'philox', use_cuda_graph=use_graph, **extra)
        g.store(4)
        agents.append(g.own)
    g, e = agents
    e.sample_transitions.calls = DDPG.GRAPH_STREAM_OFFSET
    for step in range(4):
        lg, qg = g.train()
        le, qe = e.train()
        assert float(lg) == float(le), step
        assert np.asarray(qg).shape == (k * 256, 1)
        assert np.array_equal(np.asarray(qg), np.asarray(qe)), step
    for which in ('Q', 'pi'):
        assert np.array_equal(g.get_flat(which), e.get_flat(which)), which


def test_shared_default_is_unchanged():
    """worker_buffers='shared' (the default) gives the bits of an agent built without the option."""
    import torch
    runs = []
    for extra in ({}, {'worker_buffers': 'shared'}):
        kw, dims, ag_ids, g_ids = ddpg_kwargs(4)
        a = make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='philox', workers_per_rank=3, **extra)
        np.random.seed(8)
        for c, ep in enumerate(episode_stream(dims, kw['T'], 4)):
            a.store_episode(ep, np.linspace(0.05, 0.3, 4), 2 * (c + 1))
        losses = [float(a.train()[0]) for _ in range(3)]
        torch.cuda.synchronize()
        runs.append((losses, a.get_flat('Q'), a.get_flat('pi')))
    assert runs[0][0] == runs[1][0]
    assert np.array_equal(runs[0][1], runs[1][1]) and np.array_equal(runs[0][2], runs[1][2])


def test_refusals():
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4)
    with pytest.raises(ValueError):
        make_gpu_agent(kw, dims, ag_ids, g_ids, workers_per_rank=2, worker_buffers='own', workers_mode='micro')
    with pytest.raises(ValueError):
        make_gpu_agent(kw, dims, ag_ids, g_ids, worker_buffers='mine')
    k2 = dict(kw, structure='task_experts', task_replay='replay_current_task_buffer')
    with pytest.raises(ValueError):
        make_gpu_agent(k2, dims, ag_ids, g_ids, workers_per_rank=2, worker_buffers='own', t_id=0)
    a = make_gpu_agent(kw, dims, ag_ids, g_ids, workers_per_rank=2, worker_buffers='own')
    with pytest.raises(ValueError):
        a.save_checkpoint('/nonexistent/ckpt')
    with pytest.raises(ValueError):
        a.load_checkpoint('/nonexistent/ckpt')


def test_refuses_several_ranks():
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4)
    from curious_b200 import ddpg as ddpg_mod
    real = ddpg_mod._world
    ddpg_mod._world = lambda comm: (None, 2)
    try:
        with pytest.raises(ValueError):
            make_gpu_agent(kw, dims, ag_ids, g_ids, workers_per_rank=2, worker_buffers='own')
    finally:
        ddpg_mod._world = real
