"""Virtual workers of RolloutWorker (workers=k, streams=WorkerStreams) against the reference's k MPI ranks, on CPU.

A world of k gloo processes runs one plain RolloutWorker per rank, rank j seeded rank_seed(seed, j) like the reference
(train.py:241-243, 332, 335); one process runs a k-worker RolloutWorker on WorkerStreams(seed, k).  The policy is a
stand-in that draws its exploration noise like DDPG.get_actions (ddpg.py:147-152): from np.random on a rank, from
worker j's stream for worker j's rows.  Exploration and evaluation workers alternate on the same streams, as in train().
Everything must be bit-equal: episodes, CP, p, C, histories, logs() (the mean over ranks train.py logs) and every
worker's final stream state.
"""
import os
import pickle
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEED, ENV_SEED, CYCLES, B, T = 11, 40, 12, 2, 8


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    p = s.getsockname()[1]
    s.close()
    return p


class _Policy(object):
    """get_actions / get_actions_workers of a deterministic actor with DDPG's host noise in reference order."""

    def __init__(self, dimu):
        self.dimu = dimu

    def _act(self, o, g, noise_eps, random_eps, rng):
        u = np.tanh(o[:, :self.dimu] + 3.0 * g[:, :self.dimu]).astype(np.float32)
        n = len(o)
        randn, explore, u_rand = rng.randn(n, self.dimu), rng.binomial(1, random_eps, n), rng.uniform(-1., 1., (n, self.dimu))
        u += noise_eps * 1.0 * randn
        u = np.clip(u, -1., 1.)
        u += explore.reshape(-1, 1) * (u_rand - u)
        return u, np.sum(o, axis=1, keepdims=True).astype(np.float32)

    def get_actions(self, o, ag, g, task_descr=None, noise_eps=0., random_eps=0., use_target_net=False, compute_Q=False):
        u, q = self._act(o, g, noise_eps, random_eps, np.random)
        return (u, q) if compute_Q else u

    def get_actions_workers(self, o, ag, g, task_descr=None, noise_eps=(), random_eps=(), streams=None,
                            use_target_net=False, compute_Q=False):
        k = len(noise_eps)
        rb = len(o) // k
        outs = [self._act(o[j * rb:(j + 1) * rb], g[j * rb:(j + 1) * rb], noise_eps[j], random_eps[j], streams.rng(j))
                for j in range(k)]
        return np.concatenate([x[0] for x in outs]), (np.concatenate([x[1] for x in outs]) if compute_Q else None)


def make_env():
    from curious_b200.envs import ModularPointEnv
    return ModularPointEnv(3, max_episode_steps=T)


def _dims(structure):
    from curious_b200.train import configure_dims
    dims = configure_dims(make_env(), structure)
    if structure == 'flat':
        dims.pop('task_descr', None)
    return dims


def _workers(structure, dims=None, **extra):
    """The exploration / evaluation pair of train.py:268-337.  Like the reference, build it after seeding: its
    constructor already draws the first assignment."""
    from curious_b200.rollout import RolloutWorker
    dims = dims or _dims(structure)
    policy = _Policy(dims['u'])
    kw = dict(dims=dims, logger=None, T=T, rollout_batch_size=B, structure=structure,
              task_selection='active_competence_progress', queue_length=6, **extra)
    explore = RolloutWorker(make_env, policy, exploit=False, noise_eps=0.2, random_eps=0.3, **kw)
    evaluator = RolloutWorker(make_env, policy, exploit=True, compute_Q=True, eval=True, **kw)
    explore.seed(ENV_SEED)
    evaluator.seed(ENV_SEED + 100)
    return explore, evaluator


def _record(w):
    """What one rank (or every virtual worker) carries after a generate_rollouts."""
    virtual = w.streams is not None
    triples = w.worker_histories if virtual else [(w.success_history, w.reward_history, w.Q_history)]
    hist = [(list(s), [r.tolist() for r in rw], list(q)) for s, rw, q in triples]
    p = None if not w.modular else [np.array(x) for x in (w.worker_p if virtual else [w.p])]
    return dict(p=p, CP=np.array(w.CP), C=np.array(w.C), hist=hist, exploit=list(w.worker_exploit if virtual else [w.exploit]),
                tasks=list(w.task_history), goals=[np.asarray(x).tolist() for x in w.goal_history], logs=w.logs('x'),
                n=w.n_episodes)


def _run_cycles(explore, evaluator):
    out = []
    for c in range(CYCLES):
        ep, cp, n = explore.generate_rollouts()
        out.append(('train', {k: v.copy() for k, v in ep.items()}, np.array(cp), n, _record(explore)))
        if c % 3 == 2:
            evaluator.clear_history()
            for _ in range(2):
                ep, cp, n = evaluator.generate_rollouts()
                out.append(('eval', {k: v.copy() for k, v in ep.items()}, np.array(cp), n, _record(evaluator)))
    return out


def _rank_body(rank, world, port, structure, out_dir):
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    import torch.distributed as dist
    from curious_b200.parallel import rank_seed
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        dims = _dims(structure)
        np.random.seed(rank_seed(SEED, rank) % 2 ** 32)                 # train.py:241-243
        explore, evaluator = _workers(structure, dims)
        for w, s in ((explore, ENV_SEED), (evaluator, ENV_SEED + 100)):
            w.seed(rank_seed(s, rank))                                  # train.py:332,335 on rank `rank`
        res = dict(cycles=_run_cycles(explore, evaluator), state=np.random.get_state())
        with open(os.path.join(out_dir, 'r%d.pkl' % rank), 'wb') as f:
            pickle.dump(res, f)
    finally:
        dist.destroy_process_group()


def _world(structure, k, tmp_path):
    import torch.multiprocessing as mp
    mp.spawn(_rank_body, args=(k, _free_port(), structure, str(tmp_path)), nprocs=k, join=True)
    out = []
    for r in range(k):
        with open(os.path.join(str(tmp_path), 'r%d.pkl' % r), 'rb') as f:
            out.append(pickle.load(f))
    return out


def _pooled(values):
    """mpi_average of one scalar per rank: the sum in rank order over the count."""
    total = 0.0
    for v in values:
        total += float(v)
    return total / len(values)


@pytest.mark.parametrize('structure', ['curious', 'flat'])
@pytest.mark.parametrize('k', [2, 3])
def test_virtual_workers_equal_reference_ranks(k, structure, tmp_path):
    from curious_b200.workers import WorkerStreams
    ranks = _world(structure, k, tmp_path)
    streams = WorkerStreams(SEED, k)
    dims = _dims(structure)
    np.random.seed(5)
    caller = np.random.get_state()
    explore, evaluator = _workers(structure, dims, workers=k, streams=streams)
    mine = _run_cycles(explore, evaluator)
    now = np.random.get_state()
    assert np.array_equal(now[1], caller[1]) and now[2:] == caller[2:], 'the caller stream moved'
    assert len(mine) == len(ranks[0]['cycles'])
    n_exploit = 0
    for step, got in enumerate(mine):
        kind, ep, cp, n, rec = got
        w = explore if kind == 'train' else evaluator
        for j, rank in enumerate(ranks):
            r_kind, r_ep, r_cp, r_n, r_rec = rank['cycles'][step]
            assert kind == r_kind and n == r_n, (step, j)
            for key in r_ep:
                assert np.array_equal(ep[key][j * B:(j + 1) * B], r_ep[key]), (step, j, key)
            assert np.array_equal(cp, r_cp), (step, j)
            assert rec['hist'][j] == r_rec['hist'][0], (step, j)           # success / reward / Q histories
            assert rec['exploit'][j] == r_rec['exploit'][0], (step, j)
            if rec['p'] is not None:
                assert np.array_equal(rec['p'][j], r_rec['p'][0]), (step, j)
        # per worker: p, histories; C and the task / goal histories are rank 0's (the queues live there)
        assert np.array_equal(rec['C'], ranks[0]['cycles'][step][4]['C']), step
        assert rec['tasks'] == ranks[0]['cycles'][step][4]['tasks'] and rec['goals'] == ranks[0]['cycles'][step][4]['goals']
        for j, rank in enumerate(ranks):
            r_rec = rank['cycles'][step][4]
            if j > 0:
                assert r_rec['tasks'] == [] and r_rec['goals'] == []
        assert rec['n'] == ranks[0]['cycles'][step][4]['n']
        # logs: the mean over ranks of every rank's own values (train.py: mpi_average)
        want = [(key, _pooled([rank['cycles'][step][4]['logs'][i][1] for rank in ranks]))
                for i, (key, _) in enumerate(ranks[0]['cycles'][step][4]['logs'])]
        got_logs = [(key, float(v)) for key, v in rec['logs']]
        assert [x[0] for x in got_logs] == [x[0] for x in want]
        for (key, a), (_, b) in zip(got_logs, want):
            assert a == b or (np.isnan(a) and np.isnan(b)), (step, key, a, b)
        if structure == 'curious' and kind == 'train':
            n_exploit += sum(rec['exploit'])
    for j, rank in enumerate(ranks):
        st, want = streams.state(j), rank['state']
        assert np.array_equal(st[1], want[1]) and st[2:] == want[2:], j
    if structure == 'curious':
        assert n_exploit > 0, 'no worker exploited: the exploit branch went untested'


def test_state_round_trip_covers_the_workers():
    """state() / load_state() carry every worker's exploit flag, p and histories: a worker restored from the state of
    another continues exactly like it (given the same streams)."""
    import copy
    from curious_b200.workers import WorkerStreams
    a_streams = WorkerStreams(SEED, 3)
    a, _ = _workers('curious', workers=3, streams=a_streams)
    for _ in range(5):
        a.generate_rollouts()
    st = a.state()
    b, _ = _workers('curious', workers=3, streams=WorkerStreams(SEED, 3))
    b.load_state(copy.deepcopy(st))
    b.streams = copy.deepcopy(a_streams)             # (the streams are the policy's: its own state, not the worker's)
    for _ in range(3):
        ea, cpa, na = a.generate_rollouts()
        eb, cpb, nb = b.generate_rollouts()
        for key in ea:
            assert np.array_equal(ea[key], eb[key]), key
        assert np.array_equal(cpa, cpb) and na == nb
    assert a.worker_exploit == b.worker_exploit
    for j in range(3):
        assert np.array_equal(a.worker_p[j], b.worker_p[j])
        assert [list(h) for h in a.worker_histories[j][:1]] == [list(h) for h in b.worker_histories[j][:1]]


def test_virtual_workers_refusals():
    from curious_b200.workers import WorkerStreams
    with pytest.raises(ValueError):
        _workers('curious', workers=3)                                  # no streams
    with pytest.raises(ValueError):
        _workers('curious', workers=3, streams=WorkerStreams(SEED, 2))  # one stream per worker
