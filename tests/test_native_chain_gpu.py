"""Hidden-64 / hidden-128 networks at their true width on the tcgen05 chain kernel above 1024 rows
(DDPG(pad_hidden='native') -> cur_ddpg_chain_grads, csrc/tc_chain.cu instantiated for H = 64 / 128): the library's shape
query, the CPU oracle and the dependency-level kernels of the same library, the path each setting selects, CUDA graph
against eager, the 19-worker wide batch, checkpoint resume and short trajectories against the level kernels.  Every GPU
test carries its own mark: the query test runs on the CPU."""
import ctypes as C

import numpy as np
import pytest

from tests.ddpg_util import ddpg_kwargs, episode_stream, make_gpu_agent, make_oracle_agent, rel_err

LOSS_RTOL = 1e-5
GRAD_RTOL = 2e-5           # test_ddpg_gpu.py: max-abs error over max|grad|, 5e-4 when an oracle unit sits at the ReLU kink
PARAM_RTOL = 2e-5
CP = np.array([0.05, 0.2, 0.1, 0.0])


def _fill(agent, episodes, cp):
    n = 0
    for ep in episodes:
        n += 2
        agent.store_episode({k: v.copy() for k, v in ep.items()}, cp, n)


def _check_grad(got, want, relu_margin, what):
    err = rel_err(got, want)
    if err > GRAD_RTOL:
        assert relu_margin <= 2e-6 and err <= 5e-4, (what, err, relu_margin)


def _check_params(got, want, what, steps, rtol=PARAM_RTOL):
    """As in test_native_hidden_gpu.py: the bulk (99.9 %) within rtol of the parameter scale, the stragglers (elements
    whose gradient is rounding noise, which Adam scales up to ~lr) within the steps of lr = 1e-3."""
    err = np.abs(np.asarray(got, np.float64) - np.asarray(want, np.float64))
    scale = np.abs(np.asarray(want, np.float64)).max()
    assert np.quantile(err, 0.999) <= rtol * scale, (what, np.quantile(err, 0.999), scale)
    assert err.max() <= steps * 1e-3 * 1.01, (what, err.max())


def _desc(hidden, layers=3, modular=1, dimo=40, dimg=12, dimu=4, dimtd=4):
    from curious_b200 import _lib
    return _lib.NetDesc(modular, dimo, dimg, dimu, dimtd, hidden, layers, 1.0, 0, 5.0)


# ------------------------------------------------------------------------------------------------ query (CPU)
def test_chain_supported_answers_for_each_width():
    """cur_ddpg_chain_supported takes hidden 64 / 128 at any multiple of 128 rows and follows cur_ddpg_uses_chain at hidden
    256; cur_ddpg_uses_chain itself still refuses the narrow nets.  The library loads without a device."""
    from curious_b200 import _lib
    lib = _lib.load()
    for hidden in (64, 128):
        for modular, dimo, dimg, dimu, dimtd in ((1, 40, 12, 4, 4), (0, 40, 12, 4, 0), (1, 80, 12, 4, 8)):
            for layers in (2, 3, 4):
                d = _desc(hidden, layers, modular, dimo, dimg, dimu, dimtd)
                for n in (128, 1152, 2048, 4864):
                    assert lib.cur_ddpg_chain_supported(C.byref(d), n) == 1, (hidden, modular, layers, n)
                    assert lib.cur_ddpg_uses_chain(C.byref(d), n) == 0, (hidden, n)
                    assert lib.cur_ddpg_chain_workspace_floats(C.byref(d), n) > lib.cur_ddpg_workspace_floats(C.byref(d), n)
                for n in (1000, 1153, 64):
                    assert lib.cur_ddpg_chain_supported(C.byref(d), n) == 0, (hidden, n)
        for layers in (1, 5):
            assert lib.cur_ddpg_chain_supported(C.byref(_desc(hidden, layers)), 2048) == 0, layers
        assert lib.cur_ddpg_chain_supported(C.byref(_desc(hidden, dimu=8, dimtd=8)), 2048) == 0
    for hidden in (96, 512):
        assert lib.cur_ddpg_chain_supported(C.byref(_desc(hidden)), 2048) == 0, hidden
    d256 = _desc(256)
    for n in (256, 1024, 2048, 4864):
        assert lib.cur_ddpg_chain_supported(C.byref(d256), n) == lib.cur_ddpg_uses_chain(C.byref(d256), n), n
        assert lib.cur_ddpg_chain_workspace_floats(C.byref(d256), n) == lib.cur_ddpg_workspace_floats(C.byref(d256), n)
    assert lib.cur_ddpg_chain_supported(C.byref(d256), 2048) == 1
    try:
        lib.cur_ddpg_set_chain(0)                                 # the chain switch turns the narrow chain off too
        assert lib.cur_ddpg_chain_supported(C.byref(_desc(64)), 2048) == 0
    finally:
        lib.cur_ddpg_set_chain(-1)


# ------------------------------------------------------------------------------------------------ oracle parity
VARIANTS = [('curious', 4, 3, False, False), ('curious', 8, 3, True, False), ('flat', 4, 3, False, False),
            ('curious', 4, 2, False, True), ('curious', 4, 4, True, False)]
ROWS = (1152, 2048, 4864)


@pytest.mark.gpu
@pytest.mark.parametrize('hidden', [64, 128])
@pytest.mark.parametrize('variant', range(len(VARIANTS)))
def test_native_chain_against_oracle_and_levels(hidden, variant):
    """Losses, Q_pi and both gradients of one batch on the narrow chain against the oracle and against the FFMA level
    kernels of the same library (cur_ddpg_set_chain(0)); the variants cycle through 1152, 2048 and 4864 rows."""
    from curious_b200 import _lib
    structure, n_modules, layers, normalize_obs, relative_goals = VARIANTS[variant]
    rows = ROWS[(variant + (hidden == 128)) % len(ROWS)]
    task_replay = '' if structure == 'flat' else 'replay_task_cp_buffer'
    kw, dims, ag_ids, g_ids = ddpg_kwargs(n_modules, structure=structure, task_replay=task_replay, batch_size=rows,
                                          hidden=hidden, layers=layers, normalize_obs=normalize_obs,
                                          relative_goals=relative_goals)
    cp = np.zeros(n_modules) if structure == 'flat' else np.linspace(0.0, 0.3, n_modules)
    episodes = episode_stream(dims, kw['T'], 12, flat=structure == 'flat')
    ora = make_oracle_agent(kw, dims, ag_ids, g_ids)
    gpu = make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='numpy', pad_hidden='native')
    assert not gpu.net.padded and int(gpu.net.desc.hidden) == hidden
    for a in (ora, gpu):
        np.random.seed(17)
        _fill(a, episodes, cp)
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
            assert np.allclose(x, np.asarray(y, np.float64), rtol=0, atol=1e-7 if relative_goals else 0), key
        ref = ora.grads(ob)
        got = {}
        for name, chain in (('chain', -1), ('levels', 0)):
            lib.cur_ddpg_set_chain(chain)
            assert gpu._use_native_chain(rows) == (chain != 0) and not gpu._use_rows(rows)
            gpu.grads.zero_()
            gpu.stage_batch(gb)
            ql, qpi, gq, gp = gpu._grads()
            got[name] = (float(ql), float(gpu._pi_loss), qpi.cpu().numpy().copy(),
                         gpu.ref_flat(gpu.grads, 'Q').cpu().numpy(), gpu.ref_flat(gpu.grads, 'pi').cpu().numpy())
        for name in ('chain', 'levels'):
            ql, pl, qpi, gq, gp = got[name]
            assert abs(ql - ref['Q_loss']) <= LOSS_RTOL * abs(ref['Q_loss']) + 1e-7, name
            assert abs(pl - ref['pi_loss']) <= LOSS_RTOL * abs(ref['pi_loss']) + 1e-7, name
            assert rel_err(qpi, ref['Q_pi']) <= 1e-5, name
            _check_grad(gq, ref['Q_grad'], ref['relu_margin'], 'Q %s' % name)
            _check_grad(gp, ref['pi_grad'], ref['relu_margin'], 'pi %s' % name)
        _check_grad(got['chain'][3], got['levels'][3], ref['relu_margin'], 'Q chain vs levels')
        _check_grad(got['chain'][4], got['levels'][4], ref['relu_margin'], 'pi chain vs levels')
    finally:
        lib.cur_ddpg_set_chain(-1)


# ------------------------------------------------------------------------------------------------ path selection
@pytest.mark.gpu
@pytest.mark.parametrize('hidden', [64, 128])
def test_each_setting_keeps_its_path(hidden):
    from curious_b200 import _lib
    lib = _lib.load()
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4, hidden=hidden)
    native = make_gpu_agent(kw, dims, ag_ids, g_ids, buffer_episodes=2, pad_hidden='native')
    assert native._use_rows(1024) and not native._use_native_chain(1024)       # rows up to 1024 rows, as before
    assert not native._use_rows(2048) and native._use_native_chain(2048)
    flat = make_gpu_agent(kw, dims, ag_ids, g_ids, buffer_episodes=2, pad_hidden=False)
    assert not flat._use_rows(2048) and not flat._use_native_chain(2048)       # dependency levels at the true width
    auto = make_gpu_agent(kw, dims, ag_ids, g_ids, buffer_episodes=2)
    assert auto.net.padded and not auto._use_native_chain(2048)
    assert lib.cur_ddpg_uses_chain(C.byref(auto.net.desc), 2048) == 1           # the 256-wide chain, as before
    assert lib.cur_ddpg_uses_chain(C.byref(native.net.desc), 2048) == 0
    # update_schedule='levels': the level kernels at the true width up to 1024 rows (cur_ddpg_grads), as before; above, the
    # narrow chain, as a hidden-256 net reaches its chain through cur_ddpg_grads
    lv = make_gpu_agent(kw, dims, ag_ids, g_ids, buffer_episodes=2, pad_hidden='native', update_schedule='levels')
    for n in (128, 256, 512, 1024):
        assert not lv._use_rows(n) and not lv._use_native_chain(n), n
    assert lv._use_native_chain(1152) and lv._use_native_chain(2048)


# ------------------------------------------------------------------------------------------------ graph / eager / resume
@pytest.mark.gpu
@pytest.mark.parametrize('hidden', [64, 128])
def test_native_chain_graph_equals_eager_bit_for_bit(hidden):
    import torch
    from curious_b200.ddpg import DDPG
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4, hidden=hidden, batch_size=2048)
    episodes = episode_stream(dims, kw['T'], 6)

    def run(use_graph):
        ag = make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='philox', use_cuda_graph=use_graph, pad_hidden='native')
        assert ag._use_native_chain(2048)
        np.random.seed(4)
        _fill(ag, episodes, CP)
        if not use_graph:
            ag.sample_transitions.calls = DDPG.GRAPH_STREAM_OFFSET
        out = [(float(lg), np.asarray(qg).copy()) for lg, qg in (ag.train() for _ in range(4))]
        ag.update_target_net()
        return ag, out
    g, og = run(True)
    e, oe = run(False)
    assert g._graph is not None and e._graph is None
    for k, ((la, qa), (lb, qb)) in enumerate(zip(og, oe)):
        assert la == lb and np.array_equal(qa, qb), k
    for which in ('Q', 'pi'):
        for tgt in (False, True):
            assert np.array_equal(g.get_flat(which, tgt), e.get_flat(which, tgt)), (which, tgt)
    assert torch.equal(g._adam_m, e._adam_m) and torch.equal(g._adam_v, e._adam_v)


@pytest.mark.gpu
def test_native_chain_checkpoint_resume_continues_bit_for_bit(tmp_path):
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4, hidden=64, batch_size=2048, normalize_obs=True)
    first = episode_stream(dims, kw['T'], 12, seed=5)
    later = episode_stream(dims, kw['T'], 2, seed=6)

    def run_on(agent, n_ep0):
        out = []
        for k, ep in enumerate(later):
            agent.store_episode({key: v.copy() for key, v in ep.items()}, CP, n_ep0 + 2 * (k + 1))
            for _ in range(3):
                loss, q = agent.train()
                out.append((float(loss), np.asarray(q).copy()))
            agent.update_target_net()
        return out
    mk = lambda seed: make_gpu_agent(kw, dims, ag_ids, g_ids, buffer_episodes=10, her_rng='philox', seed=seed,
                                     pad_hidden='native')
    a = mk(1)
    assert a._use_native_chain(2048)
    np.random.seed(11)
    _fill(a, first, CP)
    for _ in range(5):
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


# ------------------------------------------------------------------------------------------------ 19 workers, wide
@pytest.mark.gpu
def test_native_nineteen_workers_run_one_wide_chain_update():
    """workers_per_rank=19 at batch 256: one 4864-row update on the narrow chain with 1 / 256 loss seeds.  Its gradient
    is the SUM of the 19 workers' single-batch gradients, of the oracle and of the row kernels (the sum the 19 accumulating
    launches of workers_mode='micro' form); the CUDA-graph agent picks this wide form on its own."""
    k = 19
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4, hidden=64)
    episodes = episode_stream(dims, kw['T'], 8)
    # ---- the wide batch of 19 workers' batches against the oracle emulating 19 workers
    ora = make_oracle_agent(kw, dims, ag_ids, g_ids)
    gpu = make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='numpy', pad_hidden='native')
    for a in (ora, gpu):
        np.random.seed(11)
        _fill(a, episodes, CP)
    np.random.seed(500)
    outs = [ora.grads(ora.sample_batch()) for _ in range(k)]
    np.random.seed(500)
    gbs = [gpu.sample_batch() for _ in range(k)]
    wide_batch = [np.concatenate([b[i] for b in gbs], axis=0) for i in range(len(gbs[0]))]
    rows = k * kw['batch_size']
    assert gpu._use_native_chain(rows)
    try:
        gpu._hyper.loss_rows = kw['batch_size']                 # 1 / 256 loss seeds: the sum of the workers' gradients
        gpu.stage_batch(wide_batch)
        ql, qpi, _, _ = gpu._grads()
    finally:
        gpu._hyper.loss_rows = 0
    assert qpi.shape == (rows, 1)
    ref_loss = np.mean([o['Q_loss'] for o in outs])
    assert abs(float(ql) - ref_loss) <= LOSS_RTOL * abs(ref_loss) + 1e-7
    margin = min(o['relu_margin'] for o in outs)
    _check_grad(gpu.ref_flat(gpu.grads, 'Q').cpu().numpy(), np.sum([o['Q_grad'] for o in outs], axis=0), margin, 'Q')
    _check_grad(gpu.ref_flat(gpu.grads, 'pi').cpu().numpy(), np.sum([o['pi_grad'] for o in outs], axis=0), margin, 'pi')
    wide = {w: gpu.ref_flat(gpu.grads, w).cpu().numpy().copy() for w in ('Q', 'pi')}
    micro = {w: 0.0 for w in ('Q', 'pi')}
    for b in gbs:                                               # the row kernels, one worker's batch at a time
        gpu.stage_batch(b)
        assert gpu._use_rows(kw['batch_size'])
        gpu._grads()
        for w in ('Q', 'pi'):
            micro[w] = micro[w] + gpu.ref_flat(gpu.grads, w).cpu().numpy()
    for w in ('Q', 'pi'):
        _check_grad(wide[w], micro[w], margin, '%s wide vs micro' % w)
    # ---- the CUDA-graph agent: one wide chain update per train(), one device step and one Adam step
    g = make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='philox', workers_per_rank=k, pad_hidden='native')
    np.random.seed(21)
    _fill(g, episodes, CP)
    out = [float(g.train()[0]) for _ in range(4)]
    assert g._wide and g._graph_rows == rows and g._use_native_chain(rows) and np.isfinite(out).all()
    assert int(g._step.item()) == 4 and g.Q_adam.t == 4


# ------------------------------------------------------------------------------------------------ chain vs levels
@pytest.mark.gpu
@pytest.mark.parametrize('hidden', [64, 128])
def test_native_chain_follows_the_level_kernels_for_four_updates(hidden):
    """3xTF32 chain against FFMA levels from the same seed.  Their gradients agree within 2e-5 of max|grad| per batch
    (test above), but Adam scales every step to ~lr, so elements with small gradients drift further than between two FFMA
    paths.  The bulk tolerance is therefore WIDENED from the 2e-5 of the parameter scale that test_native_hidden_gpu.py
    holds native and padded (both FFMA) to 4e-4, the order of the 2e-4 absolute that test_ddpg_gpu.py holds the 256-wide
    chain against the rows schedule to.  Seen on a B200: 0.9e-4 (hidden 64) and 1.0e-4 (hidden 128) at this shape;
    1e-7 - 5e-5 at the shapes of profiles/r04_native_chain.json ('agreement')."""
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4, hidden=hidden, batch_size=2048, normalize_obs=True)
    episodes = episode_stream(dims, kw['T'], 8)
    agents = [make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='numpy', seed=3, pad_hidden=p) for p in ('native', False)]
    chain, levels = agents
    assert chain._use_native_chain(2048) and not levels._use_native_chain(2048) and not levels._use_rows(2048)
    out = []
    for agent in agents:
        np.random.seed(7)
        _fill(agent, episodes, CP)
        np.random.seed(8)
        out.append([agent.train() for _ in range(4)])
    for k, ((la, qa), (lb, qb)) in enumerate(zip(*out)):
        tol = LOSS_RTOL if k == 0 else 2e-4
        assert abs(float(la) - float(lb)) <= tol * abs(float(lb)) + 1e-7, (k, float(la), float(lb))
        assert rel_err(np.asarray(qa), np.asarray(qb)) <= 10 * tol, k
    for which in ('Q', 'pi'):
        _check_params(chain.get_flat(which), levels.get_flat(which), which, 4, rtol=4e-4)
