"""GPU parity of the DDPG path (store_episode / sample_batch / train / update_target_net / get_actions,
Normalizer, MpiAdam) against the CPU oracle.

Tolerances (float32 path, summation order differs from NumPy/Eigen):
  losses                 rel 1e-5
  gradients              max-abs error <= 2e-5 * max|grad| (per flat vector).  ONLY when that bound fails and a hidden
                         pre-activation of the oracle lies within 2e-6 of the ReLU kink (such a unit may land on the
                         other side of the kink in any float32 re-implementation - different summation order - and
                         flips a whole row of dW) the update is held to 5e-4 instead; how often that fallback is TAKEN is
                         counted, reported and bounded (<= 10 % of the checks) by the last test of this file
  weights after a step   rel 1e-5 of max|theta| ... Adam's m/sqrt(v) normalisation can flip tiny gradients,
                         so the step itself is additionally checked with the ORACLE's gradient (bit exact)
"""
import os

import numpy as np
import pytest

from tests.ddpg_util import ddpg_kwargs, episode_stream, make_gpu_agent, make_oracle_agent, rel_err

pytestmark = pytest.mark.gpu
LOSS_RTOL = 1e-5
GRAD_RTOL = 2e-5
# how often the ReLU-kink fallback was taken, per category ('b256': the reference batch; 'large': 512 - 4864 rows, where
# a pre-activation within float32 rounding of 0 exists in practically every batch); reported by the last test
ESCAPES = {c: {'checks': 0, 'near_kink': 0, 'escapes': 0, 'worst_strict': 0.0, 'taken': []} for c in ('b256', 'large')}


def _check_grad(got, want, relu_margin, what='', cat='b256'):
    """max-abs error of a flat gradient <= GRAD_RTOL * max|grad|.  Only when that fails AND a hidden pre-activation of
    the oracle sits within 2e-6 of the ReLU kink (module docstring) the comparison falls back to 5e-4; how often that
    fallback is actually TAKEN is counted and bounded in test_zz_gradient_escape_frequency."""
    err = rel_err(got, want)
    E = ESCAPES[cat]
    E['checks'] += 1
    E['near_kink'] += int(relu_margin <= 2e-6)
    if err <= GRAD_RTOL:
        E['worst_strict'] = max(E['worst_strict'], float(err))
        return
    assert relu_margin <= 2e-6, (what, err, relu_margin)
    E['escapes'] += 1
    E['taken'].append((what, float(err), float(relu_margin)))
    assert err <= 5e-4, (what, err, relu_margin)


def _fill(agent, episodes, cp):
    n = 0
    for ep in episodes:
        n += ep['u'].shape[0]
        agent.store_episode({k: v.copy() for k, v in ep.items()}, cp, n)


@pytest.mark.parametrize('schedule', ['levels', 'rows'])
@pytest.mark.parametrize('normalize_obs', [False, True])
@pytest.mark.parametrize('n_modules', [4, 8])
def test_store_sample_train_against_oracle(normalize_obs, n_modules, schedule):
    """Same seeds on both sides: buffers, normaliser stats, sampled batch (bit exact), losses, gradients and
    updated weights (tolerance) must agree over several updates."""
    import torch
    kw, dims, ag_ids, g_ids = ddpg_kwargs(n_modules, normalize_obs=normalize_obs)
    cp = np.linspace(0.0, 0.3, n_modules)
    episodes = episode_stream(dims, kw['T'], 12)
    ora = make_oracle_agent(kw, dims, ag_ids, g_ids)
    gpu = make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='numpy', update_schedule=schedule)
    np.random.seed(2024)
    _fill(ora, episodes, cp)
    np.random.seed(2024)
    _fill(gpu, episodes, cp)
    # routing + duplication + distractor aliasing (ddpg.py:107-110,181-195)
    for i in range(n_modules + 1):
        assert gpu.buffer[i].current_size == ora.buffer[i].current_size, i
        if ora.buffer[i].current_size:
            hb = gpu.buffer[i].buffers
            for k in ('o', 'g', 'ag', 'u', 'task_descr', 'change'):
                n = ora.buffer[i].current_size
                assert np.array_equal(hb[k][:n], ora.buffer[i].buffers[k][:n]), (i, k)
    assert gpu.buffer[0].current_size == 0
    if n_modules == 8:
        assert gpu.buffer[6] is gpu.buffer[5] and gpu.buffer[8] is gpu.buffer[5]
    # normaliser statistics (fp32 accumulations in a different order)
    for a, b in ((gpu.o_stats, ora.o_stats), (gpu.g_stats, ora.g_stats)):
        assert np.allclose(a.mean.cpu().numpy(), b.mean, rtol=1e-5, atol=1e-6)
        assert np.allclose(a.std.cpu().numpy(), b.std, rtol=1e-5, atol=1e-6)
        assert float(a.count.cpu()[0]) == float(b.count[0])
    # identical initial weights
    assert np.array_equal(gpu.get_flat('Q'), ora.Q_adam.theta)
    assert np.array_equal(gpu.get_flat('pi'), ora.pi_adam.theta)
    # make the comparison independent of the tiny stats difference
    if normalize_obs:
        gpu.o_stats.load_state_list([ora.o_stats.sum, ora.o_stats.sumsq, ora.o_stats.count, ora.o_stats.mean,
                                     ora.o_stats.std])
        gpu.g_stats.load_state_list([ora.g_stats.sum, ora.g_stats.sumsq, ora.g_stats.count, ora.g_stats.mean,
                                     ora.g_stats.std])
    for step in range(4):
        np.random.seed(100 + step)
        ob = ora.sample_batch()
        np.random.seed(100 + step)
        gb = gpu.sample_batch()
        assert list(gpu.stage_shapes.keys()) == ora.stage_keys
        for key, x, y in zip(ora.stage_keys, gb, ob):
            assert x.shape == y.shape, key
            assert np.array_equal(x, np.asarray(y, np.float64)), key        # bit exact staged batch
        assert np.array_equal(gpu.proportions, ora.proportions)
        gpu.stage_batch(gb)
        ql, qpi, gq, gp = gpu._grads()
        ref = ora.grads(ob)
        assert abs(float(ql) - ref['Q_loss']) <= LOSS_RTOL * abs(ref['Q_loss']) + 1e-7
        assert abs(float(gpu._pi_loss) - ref['pi_loss']) <= LOSS_RTOL * abs(ref['pi_loss']) + 1e-7
        assert rel_err(qpi.cpu().numpy(), ref['Q_pi']) <= 1e-5
        _check_grad(gq.cpu().numpy(), ref['Q_grad'], ref['relu_margin'], 'Q')
        _check_grad(gp.cpu().numpy(), ref['pi_grad'], ref['relu_margin'], 'pi')
        # Adam with the oracle's own gradient: bit exact
        gpu.grads.zero_()
        gpu._view(gpu.grads, 'Q').copy_(torch.from_numpy(ref['Q_grad']).cuda())
        gpu._view(gpu.grads, 'pi').copy_(torch.from_numpy(ref['pi_grad']).cuda())
        gpu._update(gpu._view(gpu.grads, 'Q'), gpu._view(gpu.grads, 'pi'))
        ora.train(ob)
        assert np.array_equal(gpu.get_flat('Q'), ora.Q_adam.theta)
        assert np.array_equal(gpu.get_flat('pi'), ora.pi_adam.theta)
        assert np.array_equal(gpu.Q_adam.m.cpu().numpy(), ora.Q_adam.m)
        assert np.array_equal(gpu.pi_adam.v.cpu().numpy(), ora.pi_adam.v)
    gpu.update_target_net()
    ora.update_target_net()
    from oracle.ddpg_oracle import flatten
    assert np.array_equal(gpu.get_flat('Q', target=True), flatten(ora.target_Q))      # polyak: bit exact
    assert np.array_equal(gpu.get_flat('pi', target=True), flatten(ora.target_pi))


@pytest.mark.parametrize('schedule', ['levels', 'rows'])
@pytest.mark.parametrize('normalize_obs', [False, True])
def test_flat_network_step_against_oracle(normalize_obs, schedule):
    """The flat `ActorCritic` + `nn` (actor_critic.py:5-48, util.py:56-71) at the default width (hidden 256, batch 256),
    per step: staged batch bit-exact, losses rel 1e-5, Q_pi, both gradients, Adam with the oracle's gradient bit-exact."""
    import torch
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4, structure='flat', task_replay='', normalize_obs=normalize_obs)
    episodes = episode_stream(dims, kw['T'], 10, flat=True)
    cp = np.zeros(4)
    ora = make_oracle_agent(kw, dims, ag_ids, g_ids)
    gpu = make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='numpy', update_schedule=schedule)
    assert gpu._use_rows(kw['batch_size']) == (schedule == 'rows')
    np.random.seed(31)
    _fill(ora, episodes, cp)
    np.random.seed(31)
    _fill(gpu, episodes, cp)
    if normalize_obs:
        for a, b in ((gpu.o_stats, ora.o_stats), (gpu.g_stats, ora.g_stats)):
            a.load_state_list([b.sum, b.sumsq, b.count, b.mean, b.std])
    assert np.array_equal(gpu.get_flat('Q'), ora.Q_adam.theta) and np.array_equal(gpu.get_flat('pi'), ora.pi_adam.theta)
    for step in range(4):
        np.random.seed(500 + step)
        ob = ora.sample_batch()
        np.random.seed(500 + step)
        gb = gpu.sample_batch()
        for key, x, y in zip(ora.stage_keys, gb, ob):
            assert np.array_equal(x, np.asarray(y, np.float64)), key
        gpu.stage_batch(gb)
        ql, qpi, gq, gp = gpu._grads()
        ref = ora.grads(ob)
        assert abs(float(ql) - ref['Q_loss']) <= LOSS_RTOL * abs(ref['Q_loss']) + 1e-7
        assert abs(float(gpu._pi_loss) - ref['pi_loss']) <= LOSS_RTOL * abs(ref['pi_loss']) + 1e-7
        assert rel_err(qpi.cpu().numpy(), ref['Q_pi']) <= 1e-5
        _check_grad(gq.cpu().numpy(), ref['Q_grad'], ref['relu_margin'], 'Q')
        _check_grad(gp.cpu().numpy(), ref['pi_grad'], ref['relu_margin'], 'pi')
        gpu.grads.zero_()
        gpu._view(gpu.grads, 'Q').copy_(torch.from_numpy(ref['Q_grad']).cuda())
        gpu._view(gpu.grads, 'pi').copy_(torch.from_numpy(ref['pi_grad']).cuda())
        gpu._update(gpu._view(gpu.grads, 'Q'), gpu._view(gpu.grads, 'pi'))
        ora.train(ob)
        assert np.array_equal(gpu.get_flat('Q'), ora.Q_adam.theta)
        assert np.array_equal(gpu.get_flat('pi'), ora.pi_adam.theta)
    gpu.update_target_net()
    ora.update_target_net()
    from oracle.ddpg_oracle import flatten
    assert np.array_equal(gpu.get_flat('Q', target=True), flatten(ora.target_Q))
    assert np.array_equal(gpu.get_flat('pi', target=True), flatten(ora.target_pi))


@pytest.mark.parametrize('structure,task_replay', [('curious', 'replay_task_random_buffer'),
                                                   ('curious', 'replay_cp_task_transition'),
                                                   ('curious', 'replay_random_task_transition'),
                                                   ('curious', 'replay_current_task_transition'),
                                                   ('task_experts', 'replay_current_task_buffer'),
                                                   ('flat', '')])
def test_training_trajectory_all_options(structure, task_replay):
    """train() end to end (own gradients) for every structure / task_replay option: weights after 5 updates
    stay within tolerance of the oracle trajectory."""
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4, structure=structure, task_replay=task_replay, hidden=64, batch_size=128)
    if structure == 'task_experts':
        kw['t_id'] = 1
    cp = np.array([0.05, 0.2, 0.1, 0.0])
    episodes = episode_stream(dims, kw['T'], 6, flat=structure == 'flat')
    ora = make_oracle_agent(kw, dims, ag_ids, g_ids)
    gpu = make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='numpy')
    np.random.seed(7)
    _fill(ora, episodes, cp)
    np.random.seed(7)
    _fill(gpu, episodes, cp)
    np.random.seed(8)
    for _ in range(5):
        ql_o, qpi_o = ora.train()
    ora.update_target_net()
    np.random.seed(8)
    for _ in range(5):
        ql_g, qpi_g = gpu.train()
    gpu.update_target_net()
    assert abs(float(ql_g) - ql_o) <= 1e-4 * abs(ql_o) + 1e-6
    assert np.asarray(qpi_g).shape == qpi_o.shape == (kw['batch_size'], 1)
    # 5 Adam steps of size ~1e-3 each: compare against the size of the accumulated update
    for which, adam in (('Q', ora.Q_adam), ('pi', ora.pi_adam)):
        got = gpu.get_flat(which)
        assert np.abs(got - adam.theta).max() <= 2e-4, which


def test_get_actions_against_oracle():
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4, normalize_obs=True)
    ora = make_oracle_agent(kw, dims, ag_ids, g_ids)
    gpu = make_gpu_agent(kw, dims, ag_ids, g_ids)
    episodes = episode_stream(dims, kw['T'], 3)
    cp = np.zeros(4)
    np.random.seed(1)
    _fill(ora, episodes, cp)
    np.random.seed(1)
    _fill(gpu, episodes, cp)
    gpu.o_stats.load_state_list([ora.o_stats.sum, ora.o_stats.sumsq, ora.o_stats.count, ora.o_stats.mean, ora.o_stats.std])
    gpu.g_stats.load_state_list([ora.g_stats.sum, ora.g_stats.sumsq, ora.g_stats.count, ora.g_stats.mean, ora.g_stats.std])
    rng = np.random.RandomState(5)
    for n in (1, 2, 38, 203, 700):               # <= 512 rows: the one-launch path, above: the level kernels
        o = rng.standard_normal((n, dims['o'])).astype(np.float32) * 100
        g = rng.uniform(-1, 1, (n, dims['g'])).astype(np.float32)
        ag = rng.uniform(-1, 1, (n, dims['ag'])).astype(np.float32)
        td = np.eye(4, dtype=np.float32)[rng.randint(0, 4, n)]
        for use_target in (False, True):
            np.random.seed(9)
            u_o, q_o = ora.get_actions(o, ag, g, task_descr=td, noise_eps=0.2, random_eps=0.3,
                                       use_target_net=use_target, compute_Q=True)
            np.random.seed(9)
            u_g, q_g = gpu.get_actions(o, ag, g, task_descr=td, noise_eps=0.2, random_eps=0.3,
                                       use_target_net=use_target, compute_Q=True)
            assert u_g.shape == u_o.shape and (n > 1 or u_g.ndim == 1)
            assert np.allclose(u_g, u_o, rtol=1e-5, atol=1e-6 if n < 100 else 1e-5)      # (see the note below)
            assert np.allclose(q_g, q_o, rtol=1e-5, atol=1e-6 if n < 100 else 1e-5)
        np.random.seed(10)
        # raw network output: inputs here are 100x out of distribution (clipped to +-200, normalised,
        # clipped to +-5), so pre-tanh sums of ~45 terms of magnitude ~5; 1e-5 of the action range max_u
        assert np.allclose(gpu.get_actions(o, ag, g, task_descr=td), ora.get_actions(o, ag, g, task_descr=td),
                           rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize('structure,relative_goals,normalize_obs,action_noise',
                         [('curious', False, False, 'host'), ('curious', True, True, 'host'), ('flat', False, True, 'host'),
                          ('curious', False, True, 'device'), ('task_experts', False, False, 'host')])
def test_one_launch_actions_equal_the_level_kernels(structure, relative_goals, normalize_obs, action_noise):
    """The rollout-step path (cur_ddpg_actions_rows: one launch, zero-copy host buffers, polled completion word) against
    the multi-launch forward of the same library on the same weights: every option that changes the network input, both
    nets, with and without Q, row counts that are not multiples of the 4-row CTA, repeated calls (buffer reuse)."""
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4, structure=structure, task_replay='' if structure == 'flat' else
                                          ('replay_current_task_buffer' if structure == 'task_experts' else
                                           'replay_task_cp_buffer'), normalize_obs=normalize_obs,
                                          relative_goals=relative_goals)
    if structure == 'task_experts':
        kw['t_id'] = 2
    a = make_gpu_agent(kw, dims, ag_ids, g_ids, seed=3, action_noise=action_noise)
    b = make_gpu_agent(kw, dims, ag_ids, g_ids, seed=3, action_noise=action_noise, action_path='levels')
    assert a._action_rows_ok() and not b._action_rows_ok()
    for ag_ in (a, b):                                             # non-trivial statistics and a target net that differs
        ag_.o_stats.load_state_list([np.zeros(dims['o']), np.zeros(dims['o']), np.ones(1),
                                     np.linspace(-0.5, 0.5, dims['o']), np.linspace(0.5, 2.0, dims['o'])])
        ag_.g_stats.load_state_list([np.zeros(dims['g']), np.zeros(dims['g']), np.ones(1),
                                     np.linspace(-0.1, 0.1, dims['g']), np.linspace(0.05, 0.3, dims['g'])])
        ag_.set_flat('Q', ag_.get_flat('Q') * 1.5, target=True)
        ag_.set_flat('pi', ag_.get_flat('pi') * 0.5, target=True)
    rng = np.random.RandomState(11)
    flat = structure == 'flat'
    for n in (1, 2, 3, 4, 5, 38, 2, 511, 2):
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
                    assert qa.shape == qb.shape == (n, 1) and np.allclose(qa, qb, rtol=1e-5, atol=2e-6)
                else:
                    ua, ub = outs
                assert ua.shape == ub.shape and np.allclose(ua, ub, rtol=1e-5, atol=2e-6), (n, use_target, compute_Q)
    assert a._action_calls == b._action_calls


def test_device_side_exploration_noise_against_oracle():
    """action_noise='device' (SURVEY 8f row 1): ddpg.py:147-152 applied on the device from Philox draws, checked against the
    NumPy restatement on the same counters; the host np.random stream is left alone and every call draws afresh."""
    from oracle.philox_oracle import action_noise
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4, hidden=64)
    gpu = make_gpu_agent(kw, dims, ag_ids, g_ids, seed=5, action_noise='device')
    rng = np.random.RandomState(1)
    call = 0
    for n in (1, 3, 38, 5000):
        o = rng.standard_normal((n, dims['o'])).astype(np.float32)
        g = rng.uniform(-1, 1, (n, dims['g'])).astype(np.float32)
        ag = rng.uniform(-1, 1, (n, dims['ag'])).astype(np.float32)
        td = np.eye(4, dtype=np.float32)[rng.randint(0, 4, n)]
        np.random.seed(3)
        before = np.random.get_state()[1].copy()
        clean, q_clean = gpu.get_actions(o, ag, g, task_descr=td, compute_Q=True)             # call `call`: no noise asked
        noisy, q = gpu.get_actions(o, ag, g, task_descr=td, noise_eps=0.2, random_eps=0.3, compute_Q=True)
        assert np.array_equal(np.random.get_state()[1], before), 'device noise must not touch the host stream'
        assert np.array_equal(q, q_clean)                                                     # Q of the noise-free action
        want, explored = action_noise(np.asarray(clean, np.float32).reshape(n, -1), 1.0, 0.2, 0.3, 5, call + 1)
        noisy = np.asarray(noisy).reshape(n, -1)
        assert np.allclose(noisy, want, rtol=0, atol=1e-6), np.abs(noisy - want).max()
        assert np.abs(noisy).max() <= 1.0
        again = np.asarray(gpu.get_actions(o, ag, g, task_descr=td, noise_eps=0.2, random_eps=0.3)).reshape(n, -1)
        assert not np.array_equal(again, noisy)                                               # a fresh counter per call
        call += 3
        if n == 5000:
            assert abs(explored.mean() - 0.3) < 0.03
            kept = ~explored
            resid = (noisy - np.asarray(clean).reshape(n, -1))[kept]
            inside = np.abs(np.asarray(clean).reshape(n, -1)[kept]) < 0.3                       # clipping cannot bite there
            assert abs(resid[inside].std() - 0.2) < 0.01 and abs(resid[inside].mean()) < 0.01
            assert np.abs(noisy[explored]).mean() > 0.4                                       # uniform in [-1, 1]: mean |u| = 0.5


def test_normalizer_and_adam_primitives():
    import torch
    from curious_b200.mpi_adam import MpiAdam
    from curious_b200.normalizer import Normalizer
    from oracle.ddpg_oracle import MpiAdamOracle, NormalizerOracle
    rng = np.random.RandomState(0)
    for dim, rows in ((40, 100), (12, 100), (3, 7), (300, 5000)):
        a, b = Normalizer(dim, 0.01, 5), NormalizerOracle(dim, 0.01, 5)
        for _ in range(3):
            v = (rng.standard_normal((rows, dim)) * 3 + 1).astype(np.float32)
            a.update(v)
            b.update(v)
            a.recompute_stats()
            b.recompute_stats()
        assert np.allclose(a.mean.cpu().numpy(), b.mean, rtol=2e-6, atol=1e-6)
        assert np.allclose(a.std.cpu().numpy(), b.std, rtol=2e-5, atol=1e-6)
        x = rng.standard_normal((17, dim)).astype(np.float32) * 10
        a.load_state_list([b.sum, b.sumsq, b.count, b.mean, b.std])
        assert np.array_equal(a.normalize(x).cpu().numpy(), b.normalize(x))
        assert np.array_equal(a.denormalize(x).cpu().numpy(), b.denormalize(x))
    # Adam on the reference's own test problem: sum(a^2) + sum(sin(b))  (mpi_adam.py:54-63), bit exact
    np.random.seed(0)
    a0 = np.random.randn(3).astype('float32')
    b0 = np.random.randn(2, 5).astype('float32')
    theta0 = np.concatenate([a0, b0.reshape(-1)])
    ora = MpiAdamOracle(theta0)
    flat = torch.zeros(16, dtype=torch.float32, device='cuda')[:13]
    flat.copy_(torch.from_numpy(theta0))
    gpu = MpiAdam([flat])
    for i in range(10):
        th = ora.theta
        grad = np.concatenate([2 * th[:3], np.cos(th[3:])]).astype(np.float32)
        ora.update(grad, 1e-2)
        gpu.update(grad, 1e-2)
        assert np.array_equal(gpu.getflat(), ora.theta), i


def test_save_load_weights_roundtrip(tmp_path):
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4, hidden=64)
    a = make_gpu_agent(kw, dims, ag_ids, g_ids, seed=1)
    b = make_gpu_agent(kw, dims, ag_ids, g_ids, seed=2)
    a.update_target_net()
    path = str(tmp_path / 'policy')
    a.save_weights(path)
    import pickle
    with open(path + '_weights.pkl', 'rb') as f:
        w = pickle.load(f)
    # reference layout: 4 lists of per-variable arrays + 2 normaliser lists (ddpg.py:481-497)
    assert len(w) == 6 and [x.shape for x in w[0]] == [(48, 64), (64,), (12, 64), (64, 64), (64,), (64, 64), (64,),
                                                      (64, 1), (1,)]
    assert [x.shape for x in w[4]] == [(40,), (40,), (1,), (40,), (40,)]
    b.load_weights(path)
    for which in ('Q', 'pi'):
        for tgt in (False, True):
            assert np.array_equal(a.get_flat(which, tgt), b.get_flat(which, tgt))


@pytest.mark.parametrize('structure,layers,batch_size', [('curious', 3, 256), ('curious', 3, 640), ('flat', 2, 64), ('task_experts', 1, 32),
                                                         ('curious', 4, 16)])
def test_rows_schedule_trajectory(structure, layers, batch_size):
    """The cluster ("rows") schedule end to end through train(): modular and flat nets, 1-4 hidden layers,
    batches of 1..16 clusters; weights after 5 updates within tolerance of the oracle trajectory, and the
    levels schedule fed the same batches lands on the same weights within the same tolerance."""
    task_replay = {'curious': 'replay_task_cp_buffer', 'flat': '', 'task_experts': 'replay_current_task_buffer'}[structure]
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4, structure=structure, task_replay=task_replay, hidden=256, layers=layers,
                                          batch_size=batch_size)
    if structure == 'task_experts':
        kw['t_id'] = 2
    cp = np.array([0.05, 0.2, 0.1, 0.0])
    episodes = episode_stream(dims, kw['T'], 6, flat=structure == 'flat')
    ora = make_oracle_agent(kw, dims, ag_ids, g_ids)
    gpus = [make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='numpy', update_schedule=s) for s in ('rows', 'levels')]
    for agent in [ora] + gpus:
        np.random.seed(7)
        _fill(agent, episodes, cp)
    np.random.seed(8)
    for _ in range(5):
        ql_o, qpi_o = ora.train()
    for gpu in gpus:
        np.random.seed(8)
        for _ in range(5):
            ql_g, qpi_g = gpu.train()
        assert abs(float(ql_g) - ql_o) <= 1e-4 * abs(ql_o) + 1e-6
        assert rel_err(np.asarray(qpi_g), qpi_o) <= 5e-4     # 5 Adam steps amplify summation-order differences
        for which, adam in (('Q', ora.Q_adam), ('pi', ora.pi_adam)):
            # Adam normalises every step to ~lr whatever the gradient's size, so a gradient element that is
            # pure rounding noise may step the other way in a re-implementation with a different summation
            # order: bound the bulk tightly and the stragglers by the 5 steps of lr = 1e-3 themselves
            err = np.abs(gpu.get_flat(which) - adam.theta)
            assert np.quantile(err, 0.999) <= 2e-4, which
            assert err.max() <= 5 * 1e-3 * 1.01, which


def test_policy_pickle_roundtrip():
    """Policies are pickled for playing (ddpg.py:511-537, rollout.py:429-431, experiment/play.py:30-33): weights and
    normaliser statistics travel, buffers / optimiser / sampler do not."""
    import pickle
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4, hidden=64, normalize_obs=True)
    a = make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='philox', seed=3)
    _fill(a, episode_stream(dims, kw['T'], 3), np.array([0.05, 0.2, 0.1, 0.0]))
    for _ in range(3):
        a.train()
    a.update_target_net()
    b = pickle.loads(pickle.dumps(a))
    assert b.sample_transitions is None and not hasattr(b, 'buffer')
    for which in ('Q', 'pi'):
        for tgt in (False, True):
            assert np.array_equal(a.get_flat(which, tgt), b.get_flat(which, tgt))
    rng = np.random.RandomState(0)
    o, ag, g = rng.randn(7, dims['o']), rng.randn(7, dims['ag']), rng.randn(7, dims['g'])
    td = np.eye(4)[rng.randint(0, 4, 7)]
    for tgt in (False, True):
        ua, qa = a.get_actions(o, ag, g, task_descr=td, use_target_net=tgt, compute_Q=True)
        ub, qb = b.get_actions(o, ag, g, task_descr=td, use_target_net=tgt, compute_Q=True)
        assert np.array_equal(ua, ub) and np.array_equal(qa, qb)


@pytest.mark.parametrize('use_graph', [True, False])
def test_checkpoint_resume_continues_bit_for_bit(use_graph, tmp_path):
    """save_checkpoint / load_checkpoint (true resume: the reference only keeps weights + normaliser statistics,
    ddpg.py:481-497): a fresh agent that loads the checkpoint - other initial weights, empty buffers - continues
    exactly like the agent that never stopped: same losses, parameters, Adam moments, normaliser statistics and the same
    buffer slots overwritten (the buffers are small enough to be full, so slot choice consumes np.random)."""
    import torch
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4, normalize_obs=True)
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

    a = make_gpu_agent(kw, dims, ag_ids, g_ids, buffer_episodes=10, her_rng='philox', seed=1, use_cuda_graph=use_graph)
    np.random.seed(11)
    _fill(a, first, cp)
    for _ in range(9):
        a.train()
    a.update_target_net()
    assert any(b.full for b in a.buffer[1:]), 'the test wants random slot overwrites after the resume'
    path = str(tmp_path / 'ckpt.pt')
    a.save_checkpoint(path)
    cont = run_on(a, 24)

    b = make_gpu_agent(kw, dims, ag_ids, g_ids, buffer_episodes=10, her_rng='philox', seed=2, use_cuda_graph=use_graph)
    np.random.seed(99)
    b.load_checkpoint(path)
    assert b.Q_adam.t == 9 and int(b._step.item()) == 9
    assert [x.current_size for x in b.buffer] == [x.current_size for x in a.buffer]
    resumed = run_on(b, 24)
    for k, ((la, qa), (lb, qb)) in enumerate(zip(cont, resumed)):
        assert la == lb, k
        assert np.array_equal(qa, qb), k
    for which in ('Q', 'pi'):
        for tgt in (False, True):
            assert np.array_equal(a.get_flat(which, tgt), b.get_flat(which, tgt)), (which, tgt)
    assert torch.equal(a._adam_m, b._adam_m) and torch.equal(a._adam_v, b._adam_v)
    assert torch.equal(a.o_stats._running, b.o_stats._running) and torch.equal(a.g_stats.std, b.g_stats.std)
    for x, y in zip(a.buffer, b.buffer):
        assert x.n_transitions_stored == y.n_transitions_stored
        n = x.current_size * x.layout.T * x.layout.trans_stride
        assert torch.equal(x.storage[:n], y.storage[:n])
    # a checkpoint of another architecture is refused
    kw2, dims2, ag2, g2 = ddpg_kwargs(4, hidden=64)
    c = make_gpu_agent(kw2, dims2, ag2, g2, her_rng='philox')
    with pytest.raises(ValueError):
        c.load_checkpoint(path)


@pytest.mark.parametrize('schedule', ['levels', 'rows'])
@pytest.mark.parametrize('task_replay', ['replay_task_cp_buffer', 'replay_cp_task_transition'])
def test_cuda_graph_path_equals_eager_path(task_replay, schedule):
    """train() through the captured CUDA graph (device control block, device step counter, Adam table)
    must be bit-identical to the launch-by-launch path fed with the same Philox counters."""
    import torch
    from curious_b200.ddpg import DDPG
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4, task_replay=task_replay)
    episodes = episode_stream(dims, kw['T'], 6)
    agents = []
    for use_graph in (True, False):
        ag = make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='philox', use_cuda_graph=use_graph,
                            update_schedule=schedule)
        np.random.seed(4)
        _fill(ag, episodes, np.array([0.05, 0.2, 0.1, 0.0]))
        agents.append(ag)
    g, e = agents
    # the normaliser stats of the two agents were fed by identical Philox samples
    assert torch.equal(g.o_stats.mean, e.o_stats.mean)
    e.sample_transitions.calls = DDPG.GRAPH_STREAM_OFFSET
    for step in range(7):
        if step == 4:      # change the LP weights and the buffer contents mid-way: the control block must follow
            for ag in agents:
                np.random.seed(5)
                _fill(ag, episode_stream(dims, kw['T'], 2, seed=77), np.array([0.3, 0.0, 0.1, 0.2]))
            e.sample_transitions.calls = DDPG.GRAPH_STREAM_OFFSET + step
        lg, qg = g.train()
        le, qe = e.train()
        assert float(lg) == float(le), step
        assert np.array_equal(np.asarray(qg), np.asarray(qe)), step
    for which in ('Q', 'pi'):
        assert np.array_equal(g.get_flat(which), e.get_flat(which)), which
    assert torch.equal(g.Q_adam.m, e.Q_adam.m) and torch.equal(g.pi_adam.v, e.pi_adam.v)
    assert int(g._step.item()) == int(e._step.item()) == 7
    # weights changed from outside (load_weights / set_flat): the rows graph keeps W^T of the hidden layers in its
    # workspace (maintained by the fused Adam epilogue) and must rebuild it before the next replay
    for ag in agents:
        ag.set_flat('Q', (ag.get_flat('Q') * np.float32(0.5)))
        ag.set_flat('pi', (ag.get_flat('pi') * np.float32(1.25)))
    for step in range(2):
        lg, qg = g.train()
        le, qe = e.train()
        assert float(lg) == float(le), step
    for which in ('Q', 'pi'):
        assert np.array_equal(g.get_flat(which), e.get_flat(which)), which
    g.update_target_net()
    e.update_target_net()
    assert np.array_equal(g.get_flat('Q', True), e.get_flat('Q', True))


@pytest.mark.parametrize('n_modules,dimo,fused', [(8, 220, False), (4, 204, False), (4, 200, True)])
def test_graph_path_when_a_transition_does_not_fit_the_fused_stage(n_modules, dimo, fused):
    """Default options (Philox draws, CUDA graph, rows schedule at batch 256).  Arm8 at dimo 220 (Q fan-in exactly 256)
    and Arm4 at dimo 204 are nets the rows kernel takes whose transitions do not fit its 4-row HER stage: the graph
    samples them with the standalone kernel.  Arm4 at dimo 200 is the widest that fits and samples in the prologue.
    Either way the graph path equals the launch-by-launch path bit for bit."""
    import torch
    from curious_b200.ddpg import DDPG
    kw, dims, ag_ids, g_ids = ddpg_kwargs(n_modules, dimo=dimo)
    episodes = episode_stream(dims, kw['T'], 6)
    cp = np.resize([0.05, 0.2, 0.1, 0.0], n_modules)
    agents = []
    for use_graph in (True, False):
        ag = make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='philox', use_cuda_graph=use_graph)
        np.random.seed(4)
        _fill(ag, episodes, cp)
        agents.append(ag)
    g, e = agents
    e.sample_transitions.calls = DDPG.GRAPH_STREAM_OFFSET
    for step in range(5):
        lg, qg = g.train()
        le, qe = e.train()
        assert float(lg) == float(le), step
        assert np.array_equal(np.asarray(qg), np.asarray(qe)), step
    for which in ('Q', 'pi'):
        assert np.array_equal(g.get_flat(which), e.get_flat(which)), which
    for adam in ('Q_adam', 'pi_adam'):
        assert torch.equal(getattr(g, adam).m, getattr(e, adam).m) and torch.equal(getattr(g, adam).v, getattr(e, adam).v)
    segs = [(buf.device_view(), 0, ttr) for buf, ttr in g._all_segments()]
    assert (g._fused_her_args(segs) is not None) == fused


@pytest.mark.parametrize('batch_size', [512, 1024, 1280, 2560, 4096, 4864])
def test_large_batch_tensor_core_update_against_oracle(batch_size):
    """BASELINE configs 4 / 5 (19 workers x 256 = 4864 rows; batch sweep): at large batch the update runs on tcgen05
    (3xTF32) - by default as the fused chain kernel (csrc/tc_chain.cu: forward, losses and dX chains of a 128-row tile in
    one CTA) followed by split-K weight-gradient GEMMs, alternatively level by level (csrc/tc_gemm.cu).  Same tolerances
    as the batch-256 path versus the oracle for both, and both must agree with the FFMA path of the same library on the
    same batch."""
    import ctypes as C
    from curious_b200 import _lib
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4, batch_size=batch_size)
    cp = np.linspace(0.0, 0.3, 4)
    episodes = episode_stream(dims, kw['T'], 12)
    ora = make_oracle_agent(kw, dims, ag_ids, g_ids)
    gpu = make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='numpy', update_schedule='levels')
    np.random.seed(7)
    _fill(ora, episodes, cp)
    np.random.seed(7)
    _fill(gpu, episodes, cp)
    lib = _lib.load()
    modes = [('chain', 1, 1), ('levels', 1, 0), ('ffma', 0, 0)] if batch_size % 128 == 0 else [('ffma', 0, 0)]
    try:
        for step in range(2):
            np.random.seed(300 + step)
            ob = ora.sample_batch()
            np.random.seed(300 + step)
            gb = gpu.sample_batch()
            for key, x, y in zip(ora.stage_keys, gb, ob):
                assert np.array_equal(x, np.asarray(y, np.float64)), key
            ref = ora.grads(ob)
            got = {}
            for name, tc, chain in modes:
                _lib.check(lib.cur_ddpg_set_tensor_cores(tc), 'cur_ddpg_set_tensor_cores')
                _lib.check(lib.cur_ddpg_set_chain(chain), 'cur_ddpg_set_chain')
                assert lib.cur_ddpg_uses_tensor_cores(C.byref(gpu.net.desc), batch_size) == tc
                assert lib.cur_ddpg_uses_chain(C.byref(gpu.net.desc), batch_size) == chain
                gpu.grads.zero_()
                gpu.stage_batch(gb)
                ql, qpi, gq, gp = gpu._grads()
                got[name] = (float(ql), float(gpu._pi_loss), qpi.cpu().numpy().copy(), gq.cpu().numpy().copy(),
                             gp.cpu().numpy().copy())
            for name, _, _ in modes:
                ql, pl, qpi, gq, gp = got[name]
                assert abs(ql - ref['Q_loss']) <= LOSS_RTOL * abs(ref['Q_loss']) + 1e-7, name
                assert abs(pl - ref['pi_loss']) <= LOSS_RTOL * abs(ref['pi_loss']) + 1e-7, name
                assert rel_err(qpi, ref['Q_pi']) <= 1e-5, name
                _check_grad(gq, ref['Q_grad'], ref['relu_margin'], 'Q %s' % name, 'large')        # see the module docstring
                _check_grad(gp, ref['pi_grad'], ref['relu_margin'], 'pi %s' % name, 'large')
            for name in ('chain', 'levels'):
                _check_grad(got[name][3], got['ffma'][3], ref['relu_margin'], 'Q %s vs ffma' % name, 'large')
                _check_grad(got[name][4], got['ffma'][4], ref['relu_margin'], 'pi %s vs ffma' % name, 'large')
            # step both sides with the ORACLE's gradient (Adam's m / sqrt(v) turns last-bit gradient noise into
            # +-lr parameter differences on the first steps, see the module docstring): bit exact
            import torch
            gpu.grads.zero_()
            gpu._view(gpu.grads, 'Q').copy_(torch.from_numpy(ref['Q_grad']).cuda())
            gpu._view(gpu.grads, 'pi').copy_(torch.from_numpy(ref['pi_grad']).cuda())
            gpu._update(gpu._view(gpu.grads, 'Q'), gpu._view(gpu.grads, 'pi'))
            ora.train(ob)
            assert np.array_equal(gpu.get_flat('Q'), ora.Q_adam.theta)
            assert np.array_equal(gpu.get_flat('pi'), ora.pi_adam.theta)
    finally:
        lib.cur_ddpg_set_tensor_cores(-1)
        lib.cur_ddpg_set_chain(-1)


@pytest.mark.parametrize('structure,n_modules,layers,normalize_obs,relative_goals',
                         [('flat', 4, 3, False, False), ('curious', 8, 3, True, False), ('curious', 4, 2, False, True),
                          ('curious', 4, 4, True, False), ('task_experts', 4, 3, False, False)])
def test_chain_kernel_network_variants(structure, n_modules, layers, normalize_obs, relative_goals):
    """The fused chain kernel on every network shape it accepts: the flat nets (one K segment in the first layers), the
    Arm8 dims (three k-blocks of state input), 2 and 4 hidden layers, normalised inputs, relative goals - losses, Q_pi and
    both gradients at 1024 rows against the oracle and against the FFMA path of the same library."""
    import ctypes as C
    from curious_b200 import _lib
    task_replay = '' if structure == 'flat' else ('replay_current_task_buffer' if structure == 'task_experts'
                                                   else 'replay_task_cp_buffer')
    kw, dims, ag_ids, g_ids = ddpg_kwargs(n_modules, structure=structure, task_replay=task_replay, batch_size=1024,
                                          layers=layers, normalize_obs=normalize_obs, relative_goals=relative_goals)
    if structure == 'task_experts':
        kw['t_id'] = 1
    cp = np.linspace(0.0, 0.3, n_modules)
    episodes = episode_stream(dims, kw['T'], 12, flat=structure == 'flat')
    ora = make_oracle_agent(kw, dims, ag_ids, g_ids)
    gpu = make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='numpy', update_schedule='levels')
    np.random.seed(17)
    _fill(ora, episodes, cp)
    np.random.seed(17)
    _fill(gpu, episodes, cp)
    if normalize_obs:
        for a, b in ((gpu.o_stats, ora.o_stats), (gpu.g_stats, ora.g_stats)):
            a.load_state_list([b.sum, b.sumsq, b.count, b.mean, b.std])
    lib = _lib.load()
    try:
        np.random.seed(400)
        ob = ora.sample_batch()
        np.random.seed(400)
        gb = gpu.sample_batch()
        for key, x, y in zip(ora.stage_keys, gb, ob):
            if relative_goals and key in ('g', 'g_2'):        # g - ag: float32 on the device, float64 in the reference
                assert np.allclose(x, np.asarray(y, np.float64), rtol=0, atol=1e-7), key
            else:
                assert np.array_equal(x, np.asarray(y, np.float64)), key
        ref = ora.grads(ob)
        got = {}
        for name, tc, chain in (('chain', 1, 1), ('ffma', 0, 0)):
            _lib.check(lib.cur_ddpg_set_tensor_cores(tc), 'cur_ddpg_set_tensor_cores')
            _lib.check(lib.cur_ddpg_set_chain(chain), 'cur_ddpg_set_chain')
            assert lib.cur_ddpg_uses_chain(C.byref(gpu.net.desc), 1024) == chain
            gpu.grads.zero_()
            gpu.stage_batch(gb)
            ql, qpi, gq, gp = gpu._grads()
            got[name] = (float(ql), float(gpu._pi_loss), qpi.cpu().numpy().copy(), gq.cpu().numpy().copy(),
                         gp.cpu().numpy().copy())
        for name in ('chain', 'ffma'):
            ql, pl, qpi, gq, gp = got[name]
            assert abs(ql - ref['Q_loss']) <= LOSS_RTOL * abs(ref['Q_loss']) + 1e-7, name
            assert abs(pl - ref['pi_loss']) <= LOSS_RTOL * abs(ref['pi_loss']) + 1e-7, name
            assert rel_err(qpi, ref['Q_pi']) <= 1e-5, name
            _check_grad(gq, ref['Q_grad'], ref['relu_margin'], 'Q %s' % name, 'large')
            _check_grad(gp, ref['pi_grad'], ref['relu_margin'], 'pi %s' % name, 'large')
        _check_grad(got['chain'][3], got['ffma'][3], ref['relu_margin'], 'Q chain vs ffma', 'large')
        _check_grad(got['chain'][4], got['ffma'][4], ref['relu_margin'], 'pi chain vs ffma', 'large')
    finally:
        lib.cur_ddpg_set_tensor_cores(-1)
        lib.cur_ddpg_set_chain(-1)


@pytest.mark.parametrize('batch_size,use_graph', [(256, True), (256, False), (2048, True)])
def test_task_experts_grouped_update_equals_sequential(batch_size, use_graph):
    """structure='task_experts': TaskExperts.train() steps all experts with grouped launches (one launch per
    dependency level over every expert's problems, cur_ddpg_grads_group).  It must be `for p in policies:
    p.train()` - bit-identical parameters and losses to stepping the same experts one after the other on the
    levels schedule (same Philox streams, same per-problem arithmetic)."""
    import torch
    from curious_b200.experts import TaskExperts
    n_exp = 3
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4, structure='task_experts', task_replay='replay_current_task_buffer',
                                          batch_size=batch_size)
    cp = np.array([0.05, 0.2, 0.1, 0.0])
    episodes = episode_stream(dims, kw['T'], 8)

    def build(use_cuda_graph):
        agents = []
        for t in range(n_exp):
            k = dict(kw)
            k['t_id'] = t
            a = make_gpu_agent(k, dims, ag_ids, g_ids, her_rng='philox', seed=10 + t, update_schedule='levels',
                               use_cuda_graph=use_cuda_graph)
            np.random.seed(7)
            _fill(a, episodes, cp)
            agents.append(a)
        return agents

    seq = build(use_graph)
    grp = TaskExperts(build(use_graph), use_cuda_graph=use_graph)
    losses_seq, losses_grp = [], []
    for _ in range(4):
        losses_seq.append([float(p.train()[0]) for p in seq])
        losses_grp.append([float(x[0]) for x in grp.train()])
    torch.cuda.synchronize()
    assert np.array_equal(np.array(losses_seq), np.array(losses_grp))
    for a, b in zip(seq, grp.policies):
        assert torch.equal(a.theta_main, b.theta_main)
        assert torch.equal(a._adam_v, b._adam_v)
        assert a.Q_adam.t == b.Q_adam.t == 4
    # different experts do learn different things
    assert not torch.equal(grp[0].theta_main, grp[1].theta_main)


def test_workers_per_rank_sums_single_batch_gradients():
    """SURVEY 8e: the reference's 19 MPI workers become ceil(19 / G) workers per GPU.  `workers_per_rank=k` makes one
    update the SUM of k batch-256 gradients, each with its own loss mean - what MpiAdam's SUM all-reduce over k
    single-batch workers produces (mpi_adam.py:24-28 with scale_grad_by_procs=False, ddpg.py:452-453).
      (1) eager path with the reference's np.random draws == oracle emulating k workers (Adam fed the summed gradient)
      (2) CUDA-graph path (k launches accumulating in the weight-gradient epilogue, Adam's t = counter / k)
          == eager path, bit for bit, on the same Philox stream."""
    import torch
    from curious_b200.ddpg import DDPG
    from oracle.ddpg_oracle import unflatten
    k = 3
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4)
    cp = np.array([0.05, 0.2, 0.1, 0.0])
    episodes = episode_stream(dims, kw['T'], 8)
    # ---- (1) against the oracle
    ora = make_oracle_agent(kw, dims, ag_ids, g_ids)
    gpu = make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='numpy', workers_per_rank=k)
    for a in (ora, gpu):
        np.random.seed(11)
        _fill(a, episodes, cp)
    for step in range(3):
        np.random.seed(500 + step)
        outs = [ora.grads(ora.sample_batch()) for _ in range(k)]
        gq = np.sum([o['Q_grad'] for o in outs], axis=0, dtype=np.float32)
        gp = np.sum([o['pi_grad'] for o in outs], axis=0, dtype=np.float32)
        np.random.seed(500 + step)
        gpu.train()
        margin = min(o['relu_margin'] for o in outs)
        _check_grad(gpu._view(gpu.grads, 'Q').cpu().numpy(), gq, margin, 'Q workers')
        _check_grad(gpu._view(gpu.grads, 'pi').cpu().numpy(), gp, margin, 'pi workers')
        # keep both sides on the oracle's trajectory (see the module docstring about Adam and tiny gradients)
        ora.main_Q = unflatten(ora.Q_adam.update(gq, ora.Q_lr), ora.ac.Q_shapes)
        ora.main_pi = unflatten(ora.pi_adam.update(gp, ora.pi_lr), ora.ac.pi_shapes)
        gpu.set_flat('Q', ora.Q_adam.theta)
        gpu.set_flat('pi', ora.pi_adam.theta)
        gpu.Q_adam.m.copy_(torch.from_numpy(ora.Q_adam.m).cuda()); gpu.Q_adam.v.copy_(torch.from_numpy(ora.Q_adam.v).cuda())
        gpu.pi_adam.m.copy_(torch.from_numpy(ora.pi_adam.m).cuda()); gpu.pi_adam.v.copy_(torch.from_numpy(ora.pi_adam.v).cuda())
    assert gpu.Q_adam.t == ora.Q_adam.t == 3 and int(gpu._step.item()) == 3 * k
    # ---- (2) graph == eager
    agents = []
    for use_graph in (True, False):
        ag = make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='philox', use_cuda_graph=use_graph, workers_per_rank=k,
                            workers_mode='micro')
        np.random.seed(4)
        _fill(ag, episodes, cp)
        agents.append(ag)
    g, e = agents
    e.sample_transitions.calls = DDPG.GRAPH_STREAM_OFFSET
    for step in range(5):
        lg, qg = g.train()
        le, qe = e.train()
        assert float(lg) == float(le), step
        assert np.array_equal(np.asarray(qg), np.asarray(qe)), step
    for which in ('Q', 'pi'):
        assert np.array_equal(g.get_flat(which), e.get_flat(which)), which
    assert torch.equal(g.Q_adam.m, e.Q_adam.m) and torch.equal(g.pi_adam.v, e.pi_adam.v)
    assert int(g._step.item()) == int(e._step.item()) == 5 * k and g.Q_adam.t == 5


def test_wide_batch_of_workers_equals_sum_of_single_batch_gradients():
    """workers_per_rank as ONE wide batch (k x 256 >= 1024 rows on the tensor-core levels schedule): with the
    backward seeds scaled by 1 / 256 (cur_ddpg_hyper.loss_rows) the gradient of the wide batch is the SUM of the k
    single-batch gradients - the reference's SUM all-reduce over k workers (ddpg.py:452-453)."""
    import torch
    from curious_b200 import _lib
    k = 4
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4)
    cp = np.array([0.05, 0.2, 0.1, 0.0])
    a = make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='numpy', update_schedule='levels')
    np.random.seed(21)
    _fill(a, episode_stream(dims, kw['T'], 8), cp)
    np.random.seed(22)
    batches = [a.sample_batch() for _ in range(k)]
    lib = _lib.load()
    try:
        lib.cur_ddpg_set_tensor_cores(0)
        total, losses = None, []
        for b in batches:
            a.stage_batch(b)
            ql, _, _, _ = a._grads()
            losses.append(float(ql))
            total = a.grads.clone() if total is None else total + a.grads
        wide = [np.concatenate([b[i] for b in batches], axis=0) for i in range(len(batches[0]))]
        for mode, tol in ((0, 2e-6), (1, GRAD_RTOL)):          # FFMA: summation order only; tcgen05: 3xTF32
            lib.cur_ddpg_set_tensor_cores(mode)
            a._hyper.loss_rows = kw['batch_size']
            a.stage_batch(wide)
            ql, qpi, _, _ = a._grads()
            a._hyper.loss_rows = 0
            assert qpi.shape == (k * kw['batch_size'], 1)
            assert abs(float(ql) - np.mean(losses)) <= 1e-5 * abs(np.mean(losses))      # mean over all workers' rows
            for which in ('Q', 'pi'):
                assert rel_err(a._view(a.grads, which).cpu().numpy(), a._view(total, which).cpu().numpy()) <= tol, (mode, which)
    finally:
        lib.cur_ddpg_set_tensor_cores(-1)
        a._hyper.loss_rows = 0
    # the CUDA-graph path picks the wide form on its own and counts one device step / one Adam step per update
    g = make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='philox', workers_per_rank=k, update_schedule='rows')
    np.random.seed(21)
    _fill(g, episode_stream(dims, kw['T'], 8), cp)
    out = [float(g.train()[0]) for _ in range(5)]
    assert g._wide and g._graph_rows == k * kw['batch_size'] and np.isfinite(out).all()
    assert int(g._step.item()) == 5 and g.Q_adam.t == 5
    # the same wide batches on the schedule 'auto' picks from 1024 rows - the fused tcgen05 chain kernel (same Philox stream,
    # other kernels): the trajectories stay together
    lv = make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='philox', workers_per_rank=k)
    np.random.seed(21)
    _fill(lv, episode_stream(dims, kw['T'], 8), cp)
    out_lv = [float(lv.train()[0]) for _ in range(5)]
    assert lv._wide and not lv._use_rows(lv._graph_rows) and g._use_rows(g._graph_rows)
    from curious_b200 import _lib as _l
    import ctypes as _C
    assert _l.load().cur_ddpg_uses_chain(_C.byref(lv.net.desc), lv._graph_rows) == 1
    assert np.allclose(out, out_lv, rtol=2e-3), (out, out_lv)
    for which in ('Q', 'pi'):
        err = np.abs(g.get_flat(which) - lv.get_flat(which))
        assert np.quantile(err, 0.999) <= 2e-4 and err.max() <= 5 * 1e-3 * 1.01, which
    big = make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='philox', workers_per_rank=8)        # 2048 rows: tensor-core levels
    np.random.seed(21)
    _fill(big, episode_stream(dims, kw['T'], 8), cp)
    assert np.isfinite(float(big.train()[0])) and big._wide and not big._use_rows(big._graph_rows)



def test_store_episode_issues_one_packed_statistics_collective(monkeypatch):
    """SURVEY 8e: per store_episode ONE all-reduce of [sum_o|sumsq_o|count_o|sum_g|sumsq_g|count_g] (the reference: six,
    normalizer.py:84-94), and the statistics equal those of two separately synchronised normalisers."""
    import torch
    from curious_b200 import normalizer
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4)
    gpu = make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='numpy')
    calls = []
    real = normalizer.allreduce_sum_

    def counting(t, comm=None):
        calls.append(int(t.numel()))
        return real(t, comm)

    monkeypatch.setattr(normalizer, 'allreduce_sum_', counting)
    eps = episode_stream(dims, kw['T'], 3)
    np.random.seed(3)
    for i, ep in enumerate(eps):
        gpu.store_episode({k: v.copy() for k, v in ep.items()}, np.array([0.05, 0.2, 0.1, 0.0]), 2 * (i + 1))
    assert calls == [2 * (dims['o'] + dims['g']) + 2] * 3
    # the same updates through stand-alone normalisers (one collective each)
    ref_o = normalizer.Normalizer(dims['o'], kw['norm_eps'], kw['norm_clip'])
    ref_g = normalizer.Normalizer(dims['g'], kw['norm_eps'], kw['norm_clip'])
    twin = make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='numpy')
    twin.o_stats.update = lambda v, _u=twin.o_stats.update: (ref_o.update(v.clone()), _u(v))[1]
    twin.g_stats.update = lambda v, _u=twin.g_stats.update: (ref_g.update(v.clone()), _u(v))[1]
    np.random.seed(3)
    for i, ep in enumerate(eps):
        twin.store_episode({k: v.copy() for k, v in ep.items()}, np.array([0.05, 0.2, 0.1, 0.0]), 2 * (i + 1))
        ref_o.recompute_stats()
        ref_g.recompute_stats()
    for a, b in ((gpu.o_stats, ref_o), (gpu.g_stats, ref_g)):
        assert torch.equal(a.mean, b.mean) and torch.equal(a.std, b.std) and torch.equal(a.count, b.count)


def test_zz_gradient_escape_frequency():
    """Runs last in this file: how many of the per-step gradient comparisons above needed the ReLU-kink fallback (5e-4)
    because the strict bound (2e-5 of max|grad|) failed.  Printed (pytest -rP), written next to the other run records
    when the directory exists, and bounded at the reference batch: the fallback is for the rare flipped unit, not a
    second tolerance.  (At 512 - 4864 rows a unit within float32 rounding of the kink exists in nearly every batch -
    millions of pre-activations - so the large-batch category is reported, not bounded.)"""
    import json
    import os
    for cat, E in ESCAPES.items():
        print('[%s] gradient checks: %d; with a pre-activation within 2e-6 of the kink: %d; strict bound failed and the '
              'fallback was taken: %d; worst error among the strict passes: %.3g; worst error with the fallback: %.3g'
              % (cat, E['checks'], E['near_kink'], E['escapes'], E['worst_strict'], max([t[1] for t in E['taken']] + [0.0])))
    out = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'gpurun_out')
    if os.path.isdir(out):
        json.dump(dict(ESCAPES, tolerance=GRAD_RTOL, escape_tolerance=5e-4, margin_threshold=2e-6),
                  open(os.path.join(out, 'grad_escape_frequency.json'), 'w'))
    E = ESCAPES['b256']
    if E['checks'] >= 20:
        assert E['escapes'] <= 0.1 * E['checks'], (E['checks'], E['escapes'], E['taken'])
