"""structure='task_experts' with hidden-64 / hidden-128 experts built with pad_hidden='native' above 1024 rows: one grouped
round on the narrow chain (TaskExperts -> cur_ddpg_chain_grads_group) against stepping the experts one after the other
(each on its own cur_ddpg_chain_grads), against the NumPy oracle, which entry point each setting calls, and the refusals
of the new entry point.  Every GPU test carries its own mark: the refusals run on the CPU."""
import ctypes as C

import numpy as np
import pytest

from tests.ddpg_util import ddpg_kwargs, episode_stream, make_gpu_agent, make_oracle_agent, rel_err

LOSS_RTOL = 1e-5
GRAD_RTOL = 2e-5           # as test_native_chain_gpu.py (near the ReLU kink: _check_grads)


def _fill(agent, episodes, cp):
    n = 0
    for ep in episodes:
        n += 2
        agent.store_episode({k: v.copy() for k, v in ep.items()}, cp, n)


KINK = 2e-6                # a hidden pre-activation this close to 0 may land on the other side of the ReLU in float32
KINK_UNITS = 6             # at most this many of the closest such units are tried on both sides


def _oracle_kink_sides(ora, batch):
    """The oracle's gradients for every way the KINK_UNITS hidden units closest to the ReLU kink (within KINK) of the
    three differentiated evaluations (main.pi, main.Q(pi), main.Q(u)) can fall: a re-implementation whose sums round
    differently may put such a unit on the other side, which changes a whole row's contribution to the gradient.  Returns
    one oracle result per side assignment.  oracle.ddpg_oracle.mlp_forward is replaced by the same computation with the
    chosen units moved across the kink while this runs."""
    from oracle import ddpg_oracle as D
    f32 = np.float32
    st = dict(call=0, flip=frozenset(), near={})

    def forward(net, modular, x_state, x_goal):
        call = st['call']
        st['call'] += 1

        def relu(pre, layer):
            h = np.maximum(pre, 0).astype(f32)
            for r, c in np.argwhere(np.abs(pre) <= KINK):
                key = (call, layer, int(r), int(c))
                st['near'].setdefault(key, float(abs(pre[r, c])))
                if key in st['flip']:
                    h[r, c] = 0 if h[r, c] > 0 else max(abs(pre[r, c]), f32(1e-30))
            return h
        if modular:
            pre = x_state @ net[0] + net[1] + x_goal @ net[2]
            rest, x0 = net[3:], (x_state, x_goal)
        else:
            x = np.concatenate([x_state, x_goal], axis=1)
            pre = x @ net[0] + net[1]
            rest, x0 = net[2:], (x,)
        margin = float(np.abs(pre).min())
        h = relu(pre, 0)
        acts = [h]
        n_rest = len(rest) // 2
        for i in range(n_rest):
            pre = h @ rest[2 * i] + rest[2 * i + 1]
            if i < n_rest - 1:
                margin = min(margin, float(np.abs(pre).min()))
                h = relu(pre, i + 1)
                acts.append(h)
            else:
                h = pre.astype(f32)
        return h, (x0, acts, margin)

    orig = D.mlp_forward
    D.mlp_forward = forward
    try:
        ora.grads(batch)
        near = sorted((k for k in st['near'] if k[0] < 3), key=lambda k: st['near'][k])[:KINK_UNITS]
        sides = []
        for bits in range(1, 1 << len(near)):
            st['call'] = 0
            st['flip'] = frozenset(k for i, k in enumerate(near) if (bits >> i) & 1)
            sides.append(ora.grads(batch))
    finally:
        D.mlp_forward = orig
    return sides


def _check_grads(got_q, got_pi, ref, ora, batch, what):
    """Both gradients within GRAD_RTOL of the oracle (max-abs error over max|grad|, as test_native_chain_gpu.py).  Only when
    that fails and an oracle unit lies within KINK of the ReLU kink, they must be within GRAD_RTOL of the oracle with some
    of the closest such units on the other side of the kink (_oracle_kink_sides)."""
    err = max(rel_err(got_q, ref['Q_grad']), rel_err(got_pi, ref['pi_grad']))
    if err <= GRAD_RTOL:
        return
    assert ref['relu_margin'] <= KINK, (what, err, ref['relu_margin'])
    side = min(max(rel_err(got_q, s['Q_grad']), rel_err(got_pi, s['pi_grad'])) for s in _oracle_kink_sides(ora, batch))
    assert side <= GRAD_RTOL, (what, err, side, ref['relu_margin'])


def _experts(kw, dims, ag_ids, g_ids, n_exp, episodes, **extra):
    cp = np.linspace(0.05, 0.3, len(g_ids))
    agents = []
    for t in range(n_exp):
        k = dict(kw)
        k['t_id'] = t
        a = make_gpu_agent(k, dims, ag_ids, g_ids, seed=10 + t, **extra)
        np.random.seed(7)
        _fill(a, episodes, cp)
        agents.append(a)
    return agents


# ------------------------------------------------------------------------------------------------ grouped == sequential
CASES = [(3, 1152), (3, 2048), (3, 4864), (5, 2048)]     # 5 experts: more experts than chain lanes (and modules of Arm4)


@pytest.mark.gpu
@pytest.mark.parametrize('schedule', ['auto', 'levels'])
@pytest.mark.parametrize('use_graph', [False, True])
@pytest.mark.parametrize('case', range(len(CASES)))
@pytest.mark.parametrize('hidden', [64, 128])
def test_native_experts_grouped_chain_equals_sequential(hidden, case, use_graph, schedule):
    """TaskExperts.train() on the grouped narrow chain is `for p in policies: p.train()` bit for bit: losses, parameters,
    both Adam moments and the Adam step count after 4 updates."""
    import torch
    from curious_b200.experts import TaskExperts
    n_exp, rows = CASES[case]
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4 if n_exp <= 4 else 8, structure='task_experts',
                                          task_replay='replay_current_task_buffer', batch_size=rows, hidden=hidden)
    episodes = episode_stream(dims, kw['T'], 8)
    extra = dict(her_rng='philox', pad_hidden='native', update_schedule=schedule, use_cuda_graph=use_graph)
    seq = _experts(kw, dims, ag_ids, g_ids, n_exp, episodes, **extra)
    grp = TaskExperts(_experts(kw, dims, ag_ids, g_ids, n_exp, episodes, **extra), use_cuda_graph=use_graph)
    assert grp._native_chain() and all(p._use_native_chain(rows) for p in seq)
    losses_seq, losses_grp = [], []
    for _ in range(4):
        losses_seq.append([float(p.train()[0]) for p in seq])
        losses_grp.append([float(x[0]) for x in grp.train()])
    torch.cuda.synchronize()
    assert (grp._graph is not None) == use_graph
    assert np.array_equal(np.array(losses_seq), np.array(losses_grp))
    for a, b in zip(seq, grp.policies):
        assert torch.equal(a.theta_main, b.theta_main)
        assert torch.equal(a._adam_m, b._adam_m)
        assert torch.equal(a._adam_v, b._adam_v)
        assert a.Q_adam.t == b.Q_adam.t == 4
    for i in range(1, n_exp):                               # the experts learn different things
        assert not torch.equal(grp[0].theta_main, grp[i].theta_main), i


# ------------------------------------------------------------------------------------------------ oracle parity
@pytest.mark.gpu
@pytest.mark.parametrize('hidden,n_modules,rows,normalize_obs', [(64, 4, 1152, False), (128, 8, 4864, True),
                                                                 (64, 8, 2048, True), (128, 4, 2048, False)])
def test_native_experts_grouped_chain_against_oracle(hidden, n_modules, rows, normalize_obs):
    """One grouped round of 3 experts, each on its own batch: every expert's losses, Q_pi and both gradients against the
    oracle, and bit for bit against the expert's own cur_ddpg_chain_grads on the same batch."""
    from curious_b200.experts import TaskExperts
    n_exp = 3
    kw, dims, ag_ids, g_ids = ddpg_kwargs(n_modules, structure='task_experts', task_replay='replay_current_task_buffer',
                                          batch_size=rows, hidden=hidden, normalize_obs=normalize_obs)
    cp = np.linspace(0.0, 0.3, n_modules)
    episodes = episode_stream(dims, kw['T'], 12)
    oras, gpus = [], []
    for t in range(n_exp):
        k = dict(kw)
        k['t_id'] = t
        ora = make_oracle_agent(k, dims, ag_ids, g_ids, seed=20 + t)
        gpu = make_gpu_agent(k, dims, ag_ids, g_ids, her_rng='numpy', seed=20 + t, pad_hidden='native')
        for a in (ora, gpu):
            np.random.seed(17 + t)
            _fill(a, episodes, cp)
        if normalize_obs:
            for a, b in ((gpu.o_stats, ora.o_stats), (gpu.g_stats, ora.g_stats)):
                a.load_state_list([b.sum, b.sumsq, b.count, b.mean, b.std])
        oras.append(ora)
        gpus.append(gpu)
    refs, obs = [], []
    for t, (ora, gpu) in enumerate(zip(oras, gpus)):
        np.random.seed(400 + t)
        ob = ora.sample_batch()
        obs.append(ob)
        np.random.seed(400 + t)
        gb = gpu.sample_batch()
        for key, x, y in zip(ora.stage_keys, gb, ob):
            assert np.array_equal(x, np.asarray(y, np.float64)), key
        refs.append(ora.grads(ob))
        gpu.grads.zero_()
        gpu.stage_batch(gb)
    te = TaskExperts(gpus, use_cuda_graph=False)
    assert te._native_chain()
    arr = te._expert_array(False, True)
    te._grads_group(arr, True)
    grouped = [(float(g._q_loss), float(g._pi_loss), g._q_pi_eager.cpu().numpy().copy(),
                g.ref_flat(g.grads, 'Q').cpu().numpy().copy(), g.ref_flat(g.grads, 'pi').cpu().numpy().copy()) for g in gpus]
    for t, (gpu, ref) in enumerate(zip(gpus, refs)):
        ql, pl, qpi, gq, gp = grouped[t]
        assert abs(ql - ref['Q_loss']) <= LOSS_RTOL * abs(ref['Q_loss']) + 1e-7, t
        assert abs(pl - ref['pi_loss']) <= LOSS_RTOL * abs(ref['pi_loss']) + 1e-7, t
        assert rel_err(qpi, ref['Q_pi']) <= 1e-5, t
        _check_grads(gq, gp, ref, oras[t], obs[t], 'expert %d' % t)
        gpu.grads.zero_()
        ql1, qpi1, _, _ = gpu._grads()                   # the same staged batch through cur_ddpg_chain_grads alone
        assert ql == float(ql1) and pl == float(gpu._pi_loss) and np.array_equal(qpi, qpi1.cpu().numpy()), t
        assert np.array_equal(gq, gpu.ref_flat(gpu.grads, 'Q').cpu().numpy()), t
        assert np.array_equal(gp, gpu.ref_flat(gpu.grads, 'pi').cpu().numpy()), t
    assert not np.array_equal(grouped[0][3], grouped[1][3])


# ------------------------------------------------------------------------------------------------ path selection
@pytest.mark.gpu
@pytest.mark.parametrize('use_graph', [False, True])
def test_native_experts_path_selection(monkeypatch, use_graph):
    """Native experts from 1152 rows call cur_ddpg_chain_grads_group and never cur_ddpg_grads_group; at 1024 rows,
    hidden 256, pad_hidden=False and with the chain switched off (cur_ddpg_set_chain(0)) they keep cur_ddpg_grads_group."""
    from curious_b200 import _lib
    from curious_b200.experts import TaskExperts
    lib = _lib.load()
    calls = []
    for name in ('cur_ddpg_grads_group', 'cur_ddpg_chain_grads_group'):
        fn = getattr(lib, name)
        monkeypatch.setattr(lib, name, lambda *a, _fn=fn, _name=name: (calls.append(_name), _fn(*a))[1])

    def called(hidden, rows, **extra):
        kw, dims, ag_ids, g_ids = ddpg_kwargs(4, structure='task_experts', task_replay='replay_current_task_buffer',
                                              batch_size=rows, hidden=hidden)
        episodes = episode_stream(dims, kw['T'], 6)
        te = TaskExperts(_experts(kw, dims, ag_ids, g_ids, 2, episodes, her_rng='philox', use_cuda_graph=use_graph,
                                  **extra), use_cuda_graph=use_graph)
        del calls[:]
        for _ in range(2):
            out = te.train()
            assert all(np.isfinite(float(x[0])) for x in out)
        return set(calls)

    for hidden in (64, 128):
        assert called(hidden, 1152, pad_hidden='native') == {'cur_ddpg_chain_grads_group'}, hidden
        assert called(hidden, 2048, pad_hidden='native', update_schedule='levels') == {'cur_ddpg_chain_grads_group'}
        assert called(hidden, 1024, pad_hidden='native') == {'cur_ddpg_grads_group'}, hidden
        assert called(hidden, 2048, pad_hidden=False) == {'cur_ddpg_grads_group'}, hidden
    assert called(256, 2048, pad_hidden='native') == {'cur_ddpg_grads_group'}
    try:
        lib.cur_ddpg_set_chain(0)
        assert called(64, 2048, pad_hidden='native') == {'cur_ddpg_grads_group'}
    finally:
        lib.cur_ddpg_set_chain(-1)


# ------------------------------------------------------------------------------------------------ refusals (CPU)
def test_chain_grads_group_refuses_bad_arguments():
    """Every refusal returns a non-zero status and a message before any device call, so it runs without a GPU (the
    pointers are never dereferenced)."""
    from curious_b200 import _lib
    lib = _lib.load()

    def desc(hidden):
        return _lib.NetDesc(1, 40, 12, 4, 4, hidden, 3, 1.0, 0, 5.0)

    def experts(count, rows):
        arr = (_lib.DdpgExpert * max(count, 1))()
        for i, e in enumerate(arr):
            fake = 0x10000000 * (i + 1)
            e.theta_main = e.theta_target = fake
            e.has_stats = 0
            e.batch = _lib.Batch(fake, fake, fake, fake, fake, fake, fake, rows[i] if i < len(rows) else rows[-1])
            e.workspace = e.grads = e.q_loss = e.pi_loss = e.q_pi = fake
        return arr

    def refused(d, n_experts, arr):
        status = lib.cur_ddpg_chain_grads_group(None, C.byref(d), n_experts, arr)
        return status != 0 and bool(lib.cur_last_error())

    assert refused(desc(256), 2, experts(2, [2048]))                        # hidden 256: cur_ddpg_grads_group
    for hidden in (64, 128):
        assert refused(desc(hidden), 2, experts(2, [1000]))                 # not a multiple of 128
        assert refused(desc(hidden), 0, experts(1, [2048]))
        assert refused(desc(hidden), 17, experts(17, [2048]))               # more than CUR_MAX_TASKS
        assert refused(desc(hidden), 3, experts(3, [2048, 2048, 1152]))     # batch sizes differ
        assert lib.cur_ddpg_chain_supported(C.byref(desc(hidden)), 2048) == 1
