"""Hidden-64 / hidden-128 networks at their true width on the row kernels (update) and the one-launch action kernel
(DDPG(pad_hidden='native'), csrc/ddpg_rows.cu instantiated for H = 64 / 128): against the reference's recorded outputs, the
CPU oracle, the zero-padded path and the dependency-level kernels; CUDA graph against eager, checkpoint resume, the tile
exchange of two ranks.  Every GPU test carries its own mark: the selection test without one runs on the CPU."""
import ctypes as C
import os
import pickle
import socket
import sys

import numpy as np
import pytest

from tests import ref_graph_util as R
from tests.ddpg_util import ddpg_kwargs, episode_stream, make_gpu_agent, make_oracle_agent, rel_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LOSS_RTOL = 1e-5
GRAD_RTOL = 2e-5           # test_ddpg_gpu.py: max-abs error over max|grad|, 5e-4 when an oracle unit sits at the ReLU kink
PARAM_RTOL = 2e-5


def _fill(agent, episodes, cp):
    n = 0
    for ep in episodes:
        n += 2
        agent.store_episode({k: v.copy() for k, v in ep.items()}, cp, n)


def _check_grad(got, want, relu_margin, what):
    err = rel_err(got, want)
    if err > GRAD_RTOL:
        assert relu_margin <= 2e-6 and err <= 5e-4, (what, err, relu_margin)


def _check_params(got, want, what, steps):
    """Parameters after `steps` Adam updates fed by each side's own gradients.  Adam scales every step to ~lr whatever the
    gradient's size, so an element whose gradient is rounding noise may step differently: the bulk (99.9 %) is held to
    PARAM_RTOL of the parameter scale, the stragglers to the steps of lr = 1e-3 themselves."""
    err = np.abs(np.asarray(got, np.float64) - np.asarray(want, np.float64))
    scale = np.abs(np.asarray(want, np.float64)).max()
    assert np.quantile(err, 0.999) <= PARAM_RTOL * scale, (what, np.quantile(err, 0.999), scale)
    assert err.max() <= steps * 1e-3 * 1.01, (what, err.max())


# ------------------------------------------------------------------------------------------------ 6. selection (CPU)
def test_rows_supported_answers_for_each_width():
    """cur_ddpg_rows_supported takes hidden 64 / 128 / 256 and nothing else; the library loads without a device."""
    from curious_b200 import _lib
    lib = _lib.load()
    for hidden, want in ((64, 1), (128, 1), (256, 1), (96, 0), (512, 0)):
        for modular, dimo, dimg, dimu, dimtd in ((1, 40, 12, 4, 4), (0, 40, 12, 4, 0), (1, 80, 12, 8, 8)):
            d = _lib.NetDesc(modular, dimo, dimg, dimu, dimtd, hidden, 3, 1.0, 0, 5.0)
            for n in (4, 256, 1024):
                assert lib.cur_ddpg_rows_supported(C.byref(d), n) == want, (hidden, modular, dimo, n)
            assert lib.cur_ddpg_rows_supported(C.byref(d), 1028) == 0
            assert lib.cur_ddpg_rows_supported(C.byref(d), 6) == 0


@pytest.mark.gpu
@pytest.mark.parametrize('hidden', [64, 128])
def test_default_and_unpadded_agents_keep_their_paths(hidden):
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4, hidden=hidden)
    auto = make_gpu_agent(kw, dims, ag_ids, g_ids, buffer_episodes=2)
    assert auto.net.padded and auto._use_rows(256) and auto._action_rows_ok()
    flat = make_gpu_agent(kw, dims, ag_ids, g_ids, buffer_episodes=2, pad_hidden=False)
    assert not flat.net.padded and not flat._use_rows(256) and not flat._action_rows_ok()
    with pytest.raises(ValueError):             # the row kernels are asked for explicitly, but not at this width
        make_gpu_agent(kw, dims, ag_ids, g_ids, buffer_episodes=2, update_schedule='rows', pad_hidden=False)._use_rows(256)
    native = make_gpu_agent(kw, dims, ag_ids, g_ids, buffer_episodes=2, pad_hidden='native')
    assert not native.net.padded and int(native.net.desc.hidden) == hidden
    assert native._use_rows(256) and native._use_rows(1024) and native._action_rows_ok()
    assert not native._use_rows(2048)               # the chain kernel needs 256 columns: levels at the true width
    kw96, dims96, ag96, g96 = ddpg_kwargs(4, hidden=96)
    with pytest.raises(ValueError):
        make_gpu_agent(kw96, dims96, ag96, g96, buffer_episodes=2, pad_hidden='native')


# ------------------------------------------------------------------------------------------------ 1. reference, hidden 64
class GpuAdapter(R.Adapter):
    def __init__(self, agent):
        self.a = agent

    def set_flat(self, which, flat, target):
        self.a.set_flat(which, flat, target)

    def get_flat(self, which, target):
        return self.a.get_flat(which, target)

    def set_stats(self, which, arrays):
        (self.a.o_stats if which == 'o' else self.a.g_stats).load_state_list(arrays)

    def grads(self, batch):
        self.a.stage_batch(batch)
        ql, qpi, gq, gp = self.a._grads()
        self._g = (gq, gp)
        return dict(Q_loss=float(ql), pi_loss=float(self.a._pi_loss), Q_pi=qpi.cpu().numpy(),
                    Q_grad=self.a.ref_flat(self.a.grads, 'Q').cpu().numpy(),
                    pi_grad=self.a.ref_flat(self.a.grads, 'pi').cpu().numpy())

    def apply(self):
        self.a._update(*self._g)


H64_CASES = [n for n in R.cases() if '_h64' in n and R.load(n)[0]['case']['layers'] <= 4 and
             R.load(n)[0]['case']['batch'] <= 1024]


@pytest.mark.gpu
@pytest.mark.parametrize('name', H64_CASES)
def test_native_h64_against_reference_fixtures(name, tmp_path):
    meta, z = R.load(name)
    case = meta['case']
    kw, dims, ag_ids, g_ids = R.case_kwargs(case)
    mk = lambda: make_gpu_agent(kw, dims, ag_ids, g_ids, buffer_episodes=2, her_rng='numpy', update_schedule='rows',
                                pad_hidden='native')
    gpu = mk()
    assert not gpu.net.padded and int(gpu.net.desc.hidden) == 64 and gpu._use_rows(case['batch'])
    meta, z, worst = R.walk(name, GpuAdapter(gpu), gpu)
    R.check_actions(name, gpu, z, dims, meta['seed'])
    if 'weights_pkl' in z.files:
        base = str(tmp_path / 'ref_policy')
        open(base + '_weights.pkl', 'wb').write(z['weights_pkl'].tobytes())
        fresh = mk()
        fresh.load_weights(base)
        for w in ('Q', 'pi'):
            for tgt in (False, True):
                assert np.array_equal(fresh.get_flat(w, tgt)[::meta['stride']], z['%s_%s_after' % ('target' if tgt else 'main', w)])
        R.check_actions(name, fresh, z, dims, meta['seed'], rtol=2e-5)
        fresh.save_weights(str(tmp_path / 'mine'))
        mine = pickle.load(open(str(tmp_path / 'mine') + '_weights.pkl', 'rb'))
        theirs = pickle.loads(z['weights_pkl'].tobytes())
        for a, b in zip(mine, theirs):
            for x, y in zip(a, b):
                assert np.shape(x) == np.shape(y) and np.array_equal(np.asarray(x, np.float32), np.asarray(y, np.float32))


@pytest.mark.gpu
@pytest.mark.parametrize('name', [n for n in R.agent_cases() if '_h64' in n])
def test_native_h64_agent_against_reference_trajectories(name):
    from oracle.gen_golden_ddpg import agent_kwargs
    meta, _ = R.load(name)
    kw, dims, ag_ids, g_ids = agent_kwargs(meta['case'])
    gpu = make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='numpy', pad_hidden='native')
    assert not gpu.net.padded and gpu._use_rows(kw['batch_size'])

    def stats_of(tag):
        s = gpu.o_stats if tag == 'o' else gpu.g_stats
        return s.mean.cpu().numpy(), s.std.cpu().numpy(), float(s.count.cpu()[0])
    R.walk_agent(name, gpu, gpu.get_flat, gpu.set_flat, stats_of)


# ------------------------------------------------------------------------------------------------ 2. oracle, hidden 128
@pytest.mark.gpu
@pytest.mark.parametrize('structure,n_modules,layers,normalize_obs,relative_goals',
                         [('curious', 4, 3, False, False), ('curious', 8, 2, True, False), ('flat', 4, 2, True, False),
                          ('curious', 4, 4, False, True), ('flat', 4, 4, False, False)])
def test_native_h128_against_oracle(structure, n_modules, layers, normalize_obs, relative_goals):
    import torch
    task_replay = '' if structure == 'flat' else 'replay_task_cp_buffer'
    kw, dims, ag_ids, g_ids = ddpg_kwargs(n_modules, structure=structure, task_replay=task_replay, hidden=128,
                                          layers=layers, normalize_obs=normalize_obs, relative_goals=relative_goals)
    flat = structure == 'flat'
    episodes = episode_stream(dims, kw['T'], 8, flat=flat)
    cp = np.zeros(n_modules) if flat else np.linspace(0.05, 0.3, n_modules)
    ora = make_oracle_agent(kw, dims, ag_ids, g_ids)
    gpu = make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='numpy', update_schedule='rows', pad_hidden='native')
    assert not gpu.net.padded and gpu._use_rows(kw['batch_size'])
    for agent in (ora, gpu):
        np.random.seed(31)
        _fill(agent, episodes, cp)
    if normalize_obs:
        for a, b in ((gpu.o_stats, ora.o_stats), (gpu.g_stats, ora.g_stats)):
            a.load_state_list([b.sum, b.sumsq, b.count, b.mean, b.std])
    assert np.array_equal(gpu.get_flat('Q'), ora.Q_adam.theta) and np.array_equal(gpu.get_flat('pi'), ora.pi_adam.theta)
    for step in range(3):
        np.random.seed(500 + step)
        ob = ora.sample_batch()
        np.random.seed(500 + step)
        gb = gpu.sample_batch()
        for key, x, y in zip(ora.stage_keys, gb, ob):
            # relative goals: g - ag is formed in float32 on the device (as in test_chain_kernel_network_variants)
            assert np.allclose(x, np.asarray(y, np.float64), rtol=0, atol=1e-7 if relative_goals else 0), key
        gpu.stage_batch(gb)
        ql, qpi, gq, gp = gpu._grads()
        ref = ora.grads(ob)
        tol = LOSS_RTOL if step == 0 else 2e-4          # from update 1 on: a trajectory check (see ref_graph_util.walk)
        assert abs(float(ql) - ref['Q_loss']) <= tol * abs(ref['Q_loss']) + 1e-7, step
        assert abs(float(gpu._pi_loss) - ref['pi_loss']) <= tol * abs(ref['pi_loss']) + 1e-7, step
        if step == 0:
            assert rel_err(qpi.cpu().numpy(), ref['Q_pi']) <= 1e-5
            _check_grad(gq.cpu().numpy(), ref['Q_grad'], ref['relu_margin'], 'Q')
            _check_grad(gp.cpu().numpy(), ref['pi_grad'], ref['relu_margin'], 'pi')
        gpu._update(gq, gp)
        ora.train(ob)
    _check_params(gpu.get_flat('Q'), ora.Q_adam.theta, 'Q', 3)
    _check_params(gpu.get_flat('pi'), ora.pi_adam.theta, 'pi', 3)
    assert torch.isfinite(gpu.theta_main).all()


# ------------------------------------------------------------------------------------------------ 3. native vs padded
@pytest.mark.gpu
@pytest.mark.parametrize('hidden,batch_size,workers', [(64, 256, 1), (64, 512, 1), (128, 256, 1), (128, 512, 1),
                                                       (64, 256, 2), (128, 256, 2)])
def test_native_equals_padded(hidden, batch_size, workers):
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4, hidden=hidden, batch_size=batch_size, normalize_obs=True)
    episodes = episode_stream(dims, kw['T'], 8)
    cp = np.array([0.05, 0.2, 0.1, 0.0])
    agents = [make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='numpy', seed=3, pad_hidden=p, workers_per_rank=workers)
              for p in ('native', 'auto')]
    nat, pad = agents
    assert not nat.net.padded and pad.net.padded
    rows = batch_size * workers
    assert nat._use_rows(rows) and pad._use_rows(rows)
    for agent in agents:
        np.random.seed(7)
        _fill(agent, episodes, cp)
    if workers == 1:
        batches = []
        for agent in agents:                             # the sampler is untouched: the staged batch is the same bits
            np.random.seed(9)
            batches.append(agent.sample_batch())
        for x, y in zip(*batches):
            assert np.array_equal(x, y)
    out = []
    for agent in agents:
        np.random.seed(8)
        out.append([agent.train() for _ in range(4)])
    for k, ((la, qa), (lb, qb)) in enumerate(zip(*out)):
        tol = LOSS_RTOL if k == 0 else 2e-4
        assert abs(float(la) - float(lb)) <= tol * abs(float(lb)) + 1e-7, (k, float(la), float(lb))
        assert rel_err(np.asarray(qa), np.asarray(qb)) <= 10 * tol, k
    for which in ('Q', 'pi'):
        _check_params(nat.get_flat(which), pad.get_flat(which), which, 4)


# ------------------------------------------------------------------------------------------------ 4. graph / eager / resume
@pytest.mark.gpu
@pytest.mark.parametrize('hidden', [64, 128])
def test_native_graph_equals_eager_bit_for_bit(hidden):
    import torch
    from curious_b200.ddpg import DDPG
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4, hidden=hidden)
    episodes = episode_stream(dims, kw['T'], 6)

    def run(use_graph):
        ag = make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='philox', use_cuda_graph=use_graph, pad_hidden='native')
        assert not ag.net.padded and ag._use_rows(kw['batch_size'])
        np.random.seed(4)
        _fill(ag, episodes, np.array([0.05, 0.2, 0.1, 0.0]))
        if not use_graph:
            ag.sample_transitions.calls = DDPG.GRAPH_STREAM_OFFSET
        out = [(float(lg), np.asarray(qg).copy()) for lg, qg in (ag.train() for _ in range(6))]
        ag.update_target_net()
        return ag, out
    g, og = run(True)
    e, oe = run(False)
    g2, og2 = run(True)
    assert g._graph is not None and e._graph is None
    for k, ((la, qa), (lb, qb), (lc, qc)) in enumerate(zip(og, oe, og2)):
        assert la == lb == lc, k
        assert np.array_equal(qa, qb) and np.array_equal(qa, qc), k
    for which in ('Q', 'pi'):
        for tgt in (False, True):
            assert np.array_equal(g.get_flat(which, tgt), e.get_flat(which, tgt)), (which, tgt)
            assert np.array_equal(g.get_flat(which, tgt), g2.get_flat(which, tgt)), (which, tgt)
    assert torch.equal(g._adam_m, e._adam_m) and torch.equal(g._adam_v, e._adam_v)


@pytest.mark.gpu
def test_native_checkpoint_resume_continues_bit_for_bit(tmp_path):
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4, hidden=64, normalize_obs=True)
    first = episode_stream(dims, kw['T'], 12, seed=5)
    later = episode_stream(dims, kw['T'], 3, seed=6)
    cp = np.array([0.05, 0.2, 0.1, 0.0])

    def run_on(agent, n_ep0):
        out = []
        for k, ep in enumerate(later):
            agent.store_episode({key: v.copy() for key, v in ep.items()}, cp, n_ep0 + 2 * (k + 1))
            for _ in range(4):
                loss, q = agent.train()
                out.append((float(loss), np.asarray(q).copy()))
            agent.update_target_net()
        return out
    mk = lambda seed: make_gpu_agent(kw, dims, ag_ids, g_ids, buffer_episodes=10, her_rng='philox', seed=seed,
                                     pad_hidden='native')
    a = mk(1)
    np.random.seed(11)
    _fill(a, first, cp)
    for _ in range(9):
        a.train()
    a.update_target_net()
    path = str(tmp_path / 'ckpt.pt')
    a.save_checkpoint(path)
    cont = run_on(a, 24)
    b = mk(2)
    np.random.seed(99)
    b.load_checkpoint(path)
    resumed = run_on(b, 24)
    for k, ((la, qa), (lb, qb)) in enumerate(zip(cont, resumed)):
        assert la == lb and np.array_equal(qa, qb), k
    for which in ('Q', 'pi'):
        for tgt in (False, True):
            assert np.array_equal(a.get_flat(which, tgt), b.get_flat(which, tgt)), (which, tgt)
    # a padded agent's checkpoint does not load into a native one (and the other way round)
    c = make_gpu_agent(kw, dims, ag_ids, g_ids, buffer_episodes=10, her_rng='philox')
    assert c.net.padded
    with pytest.raises(ValueError):
        c.load_checkpoint(path)
    c.save_checkpoint(str(tmp_path / 'padded.pt'))
    with pytest.raises(ValueError):
        mk(3).load_checkpoint(str(tmp_path / 'padded.pt'))
    # the reference's weight format interchanges between the two
    a.save_weights(str(tmp_path / 'w'))
    c.load_weights(str(tmp_path / 'w'))
    for which in ('Q', 'pi'):
        for tgt in (False, True):
            assert np.array_equal(a.get_flat(which, tgt), c.get_flat(which, tgt)), (which, tgt)


# ------------------------------------------------------------------------------------------------ 5. get_actions
@pytest.mark.gpu
@pytest.mark.parametrize('hidden,structure,normalize_obs,relative_goals,action_noise',
                         [(64, 'curious', True, False, 'host'), (128, 'curious', False, True, 'device'),
                          (64, 'flat', False, False, 'device'), (128, 'flat', True, False, 'host')])
def test_native_one_launch_actions_equal_the_level_kernels(hidden, structure, normalize_obs, relative_goals, action_noise):
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4, structure=structure, hidden=hidden, normalize_obs=normalize_obs,
                                          relative_goals=relative_goals,
                                          task_replay='' if structure == 'flat' else 'replay_task_cp_buffer')
    a = make_gpu_agent(kw, dims, ag_ids, g_ids, seed=3, action_noise=action_noise, pad_hidden='native')
    b = make_gpu_agent(kw, dims, ag_ids, g_ids, seed=3, action_noise=action_noise, pad_hidden='native',
                       action_path='levels')
    assert a._action_rows_ok() and not b._action_rows_ok() and not a.net.padded
    for ag_ in (a, b):
        ag_.o_stats.load_state_list([np.zeros(dims['o']), np.zeros(dims['o']), np.ones(1),
                                     np.linspace(-0.5, 0.5, dims['o']), np.linspace(0.5, 2.0, dims['o'])])
        ag_.g_stats.load_state_list([np.zeros(dims['g']), np.zeros(dims['g']), np.ones(1),
                                     np.linspace(-0.1, 0.1, dims['g']), np.linspace(0.05, 0.3, dims['g'])])
        ag_.set_flat('Q', ag_.get_flat('Q') * 1.5, target=True)
        ag_.set_flat('pi', ag_.get_flat('pi') * 0.5, target=True)
    rng = np.random.RandomState(11)
    flat = structure == 'flat'
    for n in (1, 2, 38, 100, 512, 2):
        o = rng.standard_normal((n, dims['o'])).astype(np.float32) * 3
        g = rng.uniform(-0.3, 0.3, (n, dims['g'])).astype(np.float32)
        ag = rng.uniform(-0.3, 0.3, (n, dims['ag'])).astype(np.float32)
        td = None if flat else np.eye(4, dtype=np.float32)[rng.randint(0, 4, n)]
        for use_target in (False, True):
            for compute_Q in (False, True):
                outs = []
                for ag_ in (a, b):
                    np.random.seed(4)
                    outs.append(ag_.get_actions(o, ag, g, task_descr=td, noise_eps=0.1, random_eps=0.2,
                                                use_target_net=use_target, compute_Q=compute_Q))
                if compute_Q:
                    (ua, qa), (ub, qb) = outs
                    # Q is a sum of terms far larger than a Q near zero: the error is bounded against the scale of the
                    # outputs (two summation orders differ by a few 1e-7 of it)
                    assert qa.shape == qb.shape == (n, 1) and rel_err(qa, qb) <= 1e-5, (n, use_target, rel_err(qa, qb))
                else:
                    ua, ub = outs
                assert ua.shape == ub.shape and np.allclose(ua, ub, rtol=1e-5, atol=2e-6), \
                    (n, use_target, compute_Q, np.abs(ua - ub).max())
    assert a._action_calls == b._action_calls


# ------------------------------------------------------------------------------------------------ 7. two ranks
def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out_dir, grad_exchange):
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    os.environ.pop('CUR_XCHG_MODE', None)
    torch.cuda.set_device(rank)
    dev = torch.device('cuda', rank)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=dev)
    try:
        from curious_b200 import parallel
        parallel.ORDERED_ALLREDUCE = True
        kw, dims, ag_ids, g_ids = ddpg_kwargs(4, hidden=64)
        agent = make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='philox', seed=rank, device=dev,
                               grad_exchange=grad_exchange, pad_hidden='native')
        assert not agent.net.padded and agent._use_rows(kw['batch_size'])
        np.random.seed(parallel.rank_seed(0, rank))
        n = 0
        for ep in episode_stream(dims, kw['T'], 6, seed=123 + rank):
            n += 2
            agent.store_episode(ep, np.array([0.05, 0.2, 0.1, 0.0]), n)
        for _ in range(60):
            agent.train()
        assert (agent._xchg is not None) == (grad_exchange == 'tile')
        agent.update_target_net()
        torch.cuda.synchronize()
        fp = agent.theta_main.clone()
        parallel.assert_synced(fp)
        np.save(os.path.join(out_dir, 'theta%d.npy' % rank), fp.cpu().numpy())
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
def test_native_h64_tile_exchange_equals_rank_ordered_allreduce(tmp_path):
    """Two ranks, hidden 64 at the true width: the in-launch tile exchange (sum in rank order, Adam + W^T in the epilogue)
    against an all-gather + rank-ordered sum + Adam launch: bit-identical parameters on both ranks and both paths."""
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    thetas = {}
    for mode in ('tile', 'nccl'):
        d = tmp_path / mode
        d.mkdir()
        mp.spawn(_worker, args=(2, _free_port(), str(d), mode), nprocs=2, join=True)
        thetas[mode] = [np.load(os.path.join(str(d), 'theta%d.npy' % r)) for r in range(2)]
        assert np.array_equal(thetas[mode][0], thetas[mode][1])
    assert np.array_equal(thetas['tile'][0], thetas['nccl'][0])
