"""CPU-only tests: C-ABI library loads and exports every declared symbol, ctypes mirrors match the header,
host apportioning logic equals the oracle, oracle backward pass equals torch autograd."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from curious_b200 import _lib
    lib = _lib.load()
    header = open(os.path.join(ROOT, 'include', 'curious_b200.h')).read()
    declared = set(re.findall(r'\b(cur_[a-z0-9_]+)\s*\(', header))
    declared -= {'cur_layout', 'cur_segment', 'cur_her_dyn'}
    assert len(declared) >= 18
    for name in declared:
        assert hasattr(lib, name), name
        assert name in _lib.SIGNATURES, 'ctypes signature missing for ' + name
    assert lib.cur_abi_version() == 4


def test_ctypes_structs_match_header(tmp_path):
    from curious_b200 import _lib
    src = tmp_path / 'sz.cpp'
    src.write_text('#include "%s"\n#include <stdio.h>\nint main(){printf("%%zu %%zu %%zu %%zu %%zu %%zu %%zu %%zu %%zu %%zu %%zu %%zu %%zu %%zu\\n",'
                   'sizeof(cur_layout),sizeof(cur_task_table),sizeof(cur_segment),sizeof(cur_her_args),'
                   'sizeof(cur_net_desc),sizeof(cur_batch),sizeof(cur_ddpg_hyper),sizeof(cur_norm_stats),'
                   'sizeof(cur_episode_src),sizeof(cur_her_dyn),sizeof(cur_adam_fused),sizeof(cur_p2p_ctx),sizeof(cur_ddpg_expert),sizeof(cur_xchg_ctx));}\n' % os.path.join(ROOT, 'include', 'curious_b200.h'))
    exe = tmp_path / 'sz'
    subprocess.check_call(['g++', str(src), '-o', str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    want = [C.sizeof(t) for t in (_lib.Layout, _lib.TaskTable, _lib.Segment, _lib.HerArgs, _lib.NetDesc, _lib.Batch,
                                  _lib.DdpgHyper, _lib.NormStats, _lib.EpisodeSrc, _lib.HerDyn, _lib.AdamFused,
                                  _lib.P2PCtx, _lib.DdpgExpert, _lib.XchgCtx)]
    assert got == want


def test_layout_and_param_counts_without_gpu():
    from curious_b200 import _lib
    L = _lib.make_layout(50, 40, 12, 12, 4, 4, 12, 1)
    # Arm4: the transition row is exactly 7 x 64 bytes and the ag(t+1) block (floats 52..63 of it) sits inside ONE
    # 64-byte atom - the order g, ag, u, td is the first of the enumeration that achieves it
    assert (L.off_g, L.off_ag, L.off_u, L.off_td, L.off_o, L.row_stride, L.trans_stride) == (0, 12, 24, 28, 32, 72, 112)
    assert (40 + L.off_ag) // 16 == (40 + L.off_ag + 11) // 16
    assert (L.off_change, L.off_info, L.off_agc, L.cold_stride) == (0, 12, 16, 28)
    L = _lib.make_layout(10, 25, 3, 3, 4)          # unaligned dims get padded sections; flat: the cold row is ag(t) alone
    assert (L.off_g, L.off_u, L.off_td, L.off_ag, L.off_o, L.row_stride, L.trans_stride) == (0, 4, 8, 8, 12, 40, 80)
    assert (L.off_change, L.off_info, L.off_agc, L.cold_stride) == (0, 0, 0, 4)
    L = _lib.make_layout(50, 64, 24, 24, 4, 8, 0, 0)   # Arm8: 24 floats of ag(t+1) cannot fit one atom; two is the minimum
    assert (64 + L.off_ag) // 16 + 1 == (64 + L.off_ag + 23) // 16
    lib = _lib.load()
    d = _lib.NetDesc(1, 40, 12, 4, 4, 256, 3, 1.0, 0, 5.0)
    assert lib.cur_net_param_count(C.byref(d), 0) == 147457      # SURVEY 8a (a8)
    assert lib.cur_net_param_count(C.byref(d), 1) == 147204
    bad = _lib.NetDesc(1, 40, 12, 4, 4, 250, 3, 1.0, 0, 5.0)
    assert lib.cur_net_param_count(C.byref(bad), 0) == -1
    with pytest.raises(_lib.CuriousLibError):
        _lib.check(lib.cur_layout_init(C.byref(_lib.Layout()), 0, 1, 1, 1, 1, 0, 0, 0), 'cur_layout_init')


def test_apportioning_equals_oracle():
    from curious_b200 import apportion
    from oracle import ddpg_oracle
    rng = np.random.RandomState(0)
    for _ in range(300):
        N = rng.choice([2, 4, 8])
        sizes = [0] + list(rng.randint(0, 6, N) * (rng.uniform(size=N) < 0.7))
        if sum(sizes[1:]) == 0:
            sizes[1 + rng.randint(N)] = 3
        cp = rng.uniform(size=N) * (rng.uniform(size=N) < 0.6)
        B = int(rng.choice([100, 256, 257]))
        for tr in ('replay_task_random_buffer', 'replay_task_cp_buffer'):
            a = apportion.proportions_curious(sizes, 50, B, tr, cp, 0.4)
            b = ddpg_oracle.apportion_curious(sizes, 50, B, tr, cp, 0.4)
            assert np.array_equal(a, b) and a.sum() == B and a[0] == 0
            assert all(a[i] == 0 for i in range(1, N + 1) if sizes[i] == 0)
        t_id = int(rng.randint(N))
        a = apportion.proportions_task_expert(sizes, 50, B, t_id)
        assert np.array_equal(a, ddpg_oracle.apportion_task_expert(sizes, 50, B, t_id))
        assert a.sum() == B
        if sizes[t_id + 1] > 0:
            assert a[t_id + 1] == B
    with pytest.raises(RuntimeError):
        apportion.proportions_curious([0, 0, 0], 50, 256, 'replay_task_cp_buffer', np.zeros(2), 0.4)
    with pytest.raises(NameError):
        apportion.proportions_curious([0, 1, 0], 50, 256, 'hand_designed', np.zeros(2), 0.4)
    p = apportion.cp_probabilities([0.05, 0.2, 0.1, 0.0], 0.4)
    assert abs(p.sum() - 1) < 1e-15 and np.allclose(p, 0.1 + 0.6 * np.array([0.05, 0.2, 0.1, 0]) / 0.35)
    ch = np.zeros(24, bool)
    ch[[0, 16, 21]] = True
    ids = [[3 * j, 3 * j + 1, 3 * j + 2] for j in range(8)]
    assert apportion.active_modules(ch, ids, ids) == [0]          # modules 5 and 7 moved but j<5 only (ddpg.py:183)
    assert apportion.active_modules(ch[:12], ids[:4], ids[:4]) == [0]


@pytest.mark.parametrize('modular', [True, False])
@pytest.mark.parametrize('normalize_obs', [False, True])
def test_oracle_gradients_equal_torch_autograd(modular, normalize_obs):
    """The hand-written NumPy backward pass of the oracle vs torch CPU autograd of the same graph
    (ddpg.py:412-449)."""
    import torch
    from oracle import ddpg_oracle as D
    rng = np.random.RandomState(1)
    dimo, dimg, dimu, dimtd, H, L, B = 10, 6, 4, 2 if modular else 0, 32, 3, 64
    o_stats, g_stats = D.NormalizerOracle(dimo, 0.01, 5), D.NormalizerOracle(dimg, 0.01, 5)
    o_stats.update(rng.standard_normal((50, dimo)).astype(np.float32)); o_stats.recompute_stats()
    g_stats.update(rng.standard_normal((50, dimg)).astype(np.float32)); g_stats.recompute_stats()
    ac = D.ActorCriticOracle(modular, dimo, dimg, dimu, dimtd, H, L, 1.0, normalize_obs, o_stats, g_stats)
    nets = [D.xavier_uniform_net(rng, s) for s in (ac.Q_shapes, ac.pi_shapes, ac.Q_shapes, ac.pi_shapes)]
    for net in nets:     # non-zero biases so their gradients are exercised
        for v in net:
            if v.ndim == 1:
                v += rng.standard_normal(v.shape).astype(np.float32) * 0.1
    batch = dict(o=rng.standard_normal((B, dimo)), g=rng.standard_normal((B, dimg)), u=rng.uniform(-1, 1, (B, dimu)),
                 o_2=rng.standard_normal((B, dimo)), g_2=rng.standard_normal((B, dimg)),
                 r=-(rng.uniform(size=(B, 1)) < 0.5).astype(np.float64))
    batch = {k: v.astype(np.float32) for k, v in batch.items()}
    if modular:
        batch['task_descr'] = np.eye(dimtd, dtype=np.float32)[rng.randint(0, dimtd, B)]
    out = D.ddpg_losses_and_grads(ac, nets[0], nets[1], nets[2], nets[3], batch, 0.98, 50., True, 1.0)

    t = lambda a: torch.tensor(a, dtype=torch.float64)
    tn = [[t(v).requires_grad_(True) for v in net] for net in nets]

    def norm(x, st):
        return torch.clamp((x - t(st.mean)) / t(st.std), -5, 5) if normalize_obs else x

    def mlp(net, xs, xg):
        if modular:
            h = torch.relu(xs @ net[0] + net[1] + xg @ net[2]); rest = net[3:]
        else:
            h = torch.relu(torch.cat([xs, xg], 1) @ net[0] + net[1]); rest = net[2:]
        for i in range(len(rest) // 2):
            h = h @ rest[2 * i] + rest[2 * i + 1]
            if i < len(rest) // 2 - 1:
                h = torch.relu(h)
        return h

    def pi_fn(net, o, g, td):
        return torch.tanh(mlp(net, torch.cat([o, td], 1), g) if modular else mlp(net, o, g))

    def q_fn(net, o, g, td, a):
        if modular:
            return mlp(net, torch.cat([o, td, a], 1), g)
        return mlp(net, torch.cat([o, g, a], 1), torch.zeros(o.shape[0], 0, dtype=torch.float64))

    o, g, o2, g2 = norm(t(batch['o']), o_stats), norm(t(batch['g']), g_stats), norm(t(batch['o_2']), o_stats), \
        norm(t(batch['g_2']), g_stats)
    td = t(batch['task_descr']) if modular else None
    pi = pi_fn(tn[1], o, g, td)
    Q_pi = q_fn(tn[0], o, g, td, pi)
    Q = q_fn(tn[0], o, g, td, t(batch['u']))
    with torch.no_grad():
        tgt = torch.clamp(t(batch['r']) + 0.98 * q_fn(tn[2], o2, g2, td, pi_fn(tn[3], o2, g2, td)), -50., 0.)
    Q_loss = ((tgt - Q) ** 2).mean()
    pi_loss = -Q_pi.mean() + (pi ** 2).mean()
    gQ = torch.autograd.grad(Q_loss, tn[0], retain_graph=True)
    gP = torch.autograd.grad(pi_loss, tn[1])
    flat = lambda gs: np.concatenate([x.numpy().reshape(-1) for x in gs])
    assert abs(out['Q_loss'] - Q_loss.item()) < 1e-5 * abs(Q_loss.item())
    assert abs(out['pi_loss'] - pi_loss.item()) < 1e-5 * abs(pi_loss.item()) + 1e-7
    for got, want in ((out['Q_grad'], flat(gQ)), (out['pi_grad'], flat(gP))):
        assert np.abs(got - want).max() <= 2e-5 * np.abs(want).max()


def test_adam_oracle_on_reference_test_problem():
    """The problem of the reference's print-only test_MpiAdam (mpi_adam.py:54-63): 10 steps on
    sum(a^2)+sum(sin(b)) must track an independent float64 Adam (TF's epsilon-hat formulation)."""
    from oracle.ddpg_oracle import MpiAdamOracle
    np.random.seed(0)
    a = np.random.randn(3).astype('float32')
    b = np.random.randn(2, 5).astype('float32')
    th0 = np.concatenate([a, b.reshape(-1)])
    ora = MpiAdamOracle(th0)
    th = th0.astype(np.float64)
    m = np.zeros_like(th); v = np.zeros_like(th)
    losses = []
    for t in range(1, 11):
        g = np.concatenate([2 * th[:3], np.cos(th[3:])])
        losses.append((th[:3] ** 2).sum() + np.sin(th[3:]).sum())
        m = 0.9 * m + 0.1 * g; v = 0.999 * v + 0.001 * g * g
        th = th - 1e-2 * np.sqrt(1 - 0.999 ** t) / (1 - 0.9 ** t) * m / (np.sqrt(v) + 1e-8)
        g32 = np.concatenate([2 * ora.theta[:3], np.cos(ora.theta[3:])]).astype(np.float32)
        ora.update(g32, 1e-2)
        assert ora.theta.dtype == np.float32 and ora.m.dtype == np.float32
        assert np.allclose(ora.theta, th, rtol=1e-5, atol=1e-6)
    assert losses[-1] < losses[0]


def test_product_never_imports_the_oracle():
    """oracle/ is test infrastructure: nothing under curious_b200/ (nor its CUDA sources) may import,
    call or link it, and the product must not read /root/reference at run time."""
    import os
    import re
    root = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'curious_b200')
    pat = re.compile(r'^\s*(from|import)\s+oracle\b|/root/reference', re.M)
    for dirpath, _, files in os.walk(root):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.h')):
                src = open(os.path.join(dirpath, f)).read()
                assert not pat.search(src), os.path.join(dirpath, f)


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    """No CPU fallback: with the shared library absent the binding raises instead of degrading."""
    from curious_b200 import _lib
    monkeypatch.setattr(_lib, 'LIB_PATH', str(tmp_path / 'nope.so'))
    monkeypatch.setattr(_lib, '_lib', None)
    import pytest
    with pytest.raises((OSError, RuntimeError)):
        _lib.load()


def test_action_noise_oracle_statistics():
    """The NumPy restatement of the device-side exploration noise (oracle/philox_oracle.action_noise, ddpg.py:147-152):
    standard-normal Box-Muller pairs, eps-greedy rate, clipping, determinism in (seed, call)."""
    from oracle.philox_oracle import action_noise
    u = np.zeros((40000, 4), np.float32)
    a, explored = action_noise(u, 1.0, 0.2, 0.0, seed=7, call=3)
    assert a.dtype == np.float32 and not explored.any()
    assert abs(a.std() - 0.2) < 2e-3 and abs(a.mean()) < 2e-3
    assert abs(np.corrcoef(a[:, 0], a[:, 1])[0, 1]) < 0.02 and abs(np.corrcoef(a[:-1, 0], a[1:, 0])[0, 1]) < 0.02
    b, explored = action_noise(u, 1.0, 0.2, 0.3, seed=7, call=3)
    assert abs(explored.mean() - 0.3) < 0.01
    assert np.array_equal(b[~explored], a[~explored]) and np.abs(b).max() <= 1.0
    assert abs(np.abs(b[explored]).mean() - 0.5) < 0.01
    c, _ = action_noise(u, 1.0, 0.2, 0.3, seed=7, call=4)
    assert not np.array_equal(b, c)
    d, _ = action_noise(u[:, :3], 1.0, 5.0, 0.0, seed=7, call=3)          # odd dimu; heavy noise is clipped
    assert d.shape == (40000, 3) and np.abs(d).max() == 1.0


def test_bench_roofline_arithmetic_matches_the_survey():
    """SURVEY 8(d): 828 B / transition (Arm4-shaped), 1340 B (Arm8-shaped), ~0.73 GFLOP per batch-256 update - the
    figures `roofline.achieved` and the TFLOP/s columns of bench.py are computed from."""
    import bench
    from curious_b200 import synth
    d4, d8 = synth.arm_dims(4), synth.arm_dims(8)
    assert (d4['o'], d4['g'], d4['ag'], d4['u']) == (40, 12, 12, 4) and (d8['o'], d8['g']) == (64, 24)
    assert bench.algorithmic_bytes_per_transition(d4, 4) == 424 + 404 == 828
    assert bench.algorithmic_bytes_per_transition(d8, 8) == 680 + 660 == 1340
    f = bench.update_flops(d4, 4, 256)
    f_pi = 2 * 256 * ((44 + 12) * 256 + 2 * 256 * 256 + 256 * 4)
    f_q = 2 * 256 * ((48 + 12) * 256 + 2 * 256 * 256 + 256)
    assert abs(f_pi - 75.0e6) < 0.1e6 and abs(f_q - 75.1e6) < 0.1e6          # SURVEY: F_pi = 75.0 M, F_Q = 75.1 M
    assert 0.72e9 < f < 0.74e9 and bench.update_flops(d4, 4, 512) == 2 * f
    # the clocks object of the JSON line keeps its keys without a GPU (no samples, no crash)
    sampler = bench.ClockSampler(0)
    sampler.start()
    line = sampler.stop()
    assert set(line) >= {'sm_mhz', 'sm_max_mhz', 'reasons', 'samples', 'source'}


def test_product_slot_policy_equals_the_live_reference():
    """ReplayBuffer._get_storage_idx of the drop-in (host logic, consumes the caller's np.random) against the unmodified
    reference method on random sequences - no device needed: the object is built without its CUDA storage.  Without a
    reference checkout, against the slot sequences recorded from that method (tests/golden/storage_*.npz)."""
    import importlib.util
    import json
    from curious_b200.replay_buffer import ReplayBuffer
    from tests.ddpg_util import REFERENCE_ROOT
    if not os.path.isdir(os.path.join(REFERENCE_ROOT, 'baselines', 'her')):
        state = np.random.get_state()
        try:
            for name in ('storage_single', 'storage_batched'):
                z = np.load(os.path.join(ROOT, 'tests', 'golden', name + '.npz'))
                meta = json.loads(str(z['meta']))
                mine = ReplayBuffer.__new__(ReplayBuffer)
                mine.size, mine.T, mine.current_size, mine.n_transitions_stored = meta['size_ep'], meta['T'], 0, 0
                np.random.seed(meta['seed'])
                for k, inc in enumerate(meta['increments']):
                    assert np.array_equal(np.atleast_1d(mine._get_storage_idx(inc)), z['idx_%d' % k]), (name, k)
                    assert mine.current_size == z['sizes'][k], (name, k)
        finally:
            np.random.set_state(state)
        return
    spec = importlib.util.spec_from_file_location('gen_golden', os.path.join(ROOT, 'oracle', 'gen_golden.py'))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    _, ref_rb = gen.import_reference()
    rng = np.random.RandomState(5)
    state = np.random.get_state()
    try:
        for case in range(40):
            T, size_ep = int(rng.randint(1, 6)), int(rng.randint(1, 12))
            ref = ref_rb.ReplayBuffer({'u': (T, 1)}, size_ep * T, T, None)
            mine = ReplayBuffer.__new__(ReplayBuffer)
            mine.size, mine.T, mine.current_size, mine.n_transitions_stored = size_ep, T, 0, 0
            seed = int(rng.randint(1 << 30))
            incs = [int(rng.randint(1, size_ep + 1)) for _ in range(int(rng.randint(3, 30)))]
            out = []
            for buf in (ref, mine):
                np.random.seed(seed)
                seq = []
                for inc in incs:
                    idx = buf._get_storage_idx(inc)
                    seq.append((np.atleast_1d(idx).tolist(), np.ndim(idx), buf.current_size))
                out.append((seq, np.random.get_state()[1].copy()))
            assert out[0][0] == out[1][0], (case, incs)
            assert np.array_equal(out[0][1], out[1][1])
            with pytest.raises(AssertionError):
                mine._get_storage_idx(size_ep + 1)
    finally:
        np.random.set_state(state)


def test_host_draws_replay_the_reference_stream():
    """curious_b200.her.HostDraws (the `her_rng='numpy'` path: the reference's np.random draws made on the host in reference
    order, her.py:108-116,129-142) against the RNG stream recorded from the unmodified reference in every fixture."""
    from curious_b200 import her
    from tests.golden_util import load_case, sampler_cases
    state = np.random.get_state()
    try:
        n_choice_cases = 0
        for name in sampler_cases():
            meta, eps, stream, ref = load_case(name)
            np.random.seed(meta['seed'])
            d = her.HostDraws(meta['E'], meta['T'], meta['B'])
            d.draw_choices(her.mode_of(meta['task_replay'], meta['flat']),
                           her.future_probability(meta['goal_replay'], meta['her_replay_k']), meta['n_modules'], meta['cp_proba'])
            assert np.array_equal(d.ep, stream['s_ep']) and np.array_equal(d.t, stream['s_t']), name
            assert np.array_equal(d.u_her, stream['s_uher']) and np.array_equal(d.u_off, stream['s_uoff']), name
            seq = stream['s_choice_seq']
            if seq.size:
                n_choice_cases += 1
                assert np.array_equal(d.choice[d.choice >= 0], seq), name
            else:
                assert d.choice is None or (d.choice < 0).all(), name
        assert n_choice_cases >= 5
    finally:
        np.random.set_state(state)


def test_library_sass_is_blackwell_native():
    """B200_PROFILING.md "What proves a Blackwell-native kernel": the SASS of the in-tree library holds tcgen05 MMAs
    (UTC*MMA) with TMEM loads (LDTM), TMA tensor and bulk copies (UTMALDG / UBLKCP) with their mbarrier waits (SYNCS), the
    cta_group::2 commit of the pair kernel (UTCBAR.2CTA), packed FP32 FMAs (FFMA2) and the in-switch reduction of the NVLS
    gradient exchange (multimem.ld_reduce = LDGMC.E.ADD) inside the weight-gradient kernel - and no legacy HMMA tensor path."""
    import shutil
    import subprocess
    from curious_b200 import _lib
    tool = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'
    if not os.path.exists(tool) or not os.path.exists(_lib.LIB_PATH):
        pytest.skip('cuobjdump or the built library is not available')
    sass = subprocess.run([tool, '-sass', _lib.LIB_PATH], capture_output=True, text=True, timeout=300).stdout
    assert 'sm_100a' in sass
    import re
    count = lambda pattern: len(re.findall(pattern, sass))
    assert count(r'\bUTC[A-Z]*MMA') >= 6                 # 3xTF32: three MMAs per k-step, single-CTA and pair kernels
    assert count(r'\bLDTM') >= 8 and count(r'\bUTMALDG') >= 8 and count(r'\bUBLKCP') >= 1
    assert count(r'\bUTCBAR\.2CTA') >= 1 and count(r'\bSYNCS\.') >= 20 and count(r'\bFFMA2\b') >= 500
    assert count(r'\bLDGMC\.E\.ADD\.F32') >= 3         # FULLK / SKINNY / COLSUM tile epilogues of rows_dw_kernel
    assert count(r'\bHMMA\b') == 0 and count(r'\bHGMMA\b') == 0


def test_owner_map_of_the_tile_exchange_covers_every_parameter():
    """cur_ddpg_rows_owner_map (host only): under mode 1 of the tile exchange every real parameter of the arena is reduced
    by exactly one rank, the padding by none, and the tiles are spread round-robin (balanced to a few percent)."""
    from curious_b200 import _lib
    lib = _lib.load()
    for d in (_lib.NetDesc(1, 40, 12, 4, 4, 256, 3, 1.0, 0, 5.0), _lib.NetDesc(1, 64, 24, 4, 8, 256, 3, 1.0, 1, 5.0),
              _lib.NetDesc(0, 40, 12, 4, 0, 256, 2, 1.0, 0, 5.0)):
        total = C.c_int64()
        off_pi = lib.cur_theta_pi_offset(C.byref(d), C.byref(total))
        nq, npi = lib.cur_net_param_count(C.byref(d), 0), lib.cur_net_param_count(C.byref(d), 1)
        for world in (1, 2, 8):
            owner = np.full(total.value, -7, np.int32)
            _lib.check(lib.cur_ddpg_rows_owner_map(C.byref(d), 256, world, owner.ctypes.data), 'cur_ddpg_rows_owner_map')
            real = np.zeros(total.value, bool)
            real[:nq] = True
            real[off_pi:off_pi + npi] = True
            assert ((owner >= 0) == real).all()
            assert owner[real].max() == world - 1
            counts = np.bincount(owner[real], minlength=world)
            assert counts.min() > 0.8 * counts.mean()


def test_zero_padded_network_index_map():
    """actor_critic._NetSpec(kernel_hidden=256): where every element of the reference's flat vector (hidden wide) sits in
    the 256-wide kernel-side vector - injective, inside the padded net, rows / columns of every layer preserved."""
    from curious_b200.actor_critic import ActorCritic, MultiTaskActorCritic
    for cls, kw in ((MultiTaskActorCritic, dict(dimtd=4)), (ActorCritic, {})):
        for hidden, layers in ((64, 3), (128, 2), (60, 4)):
            net = cls(40, 12, 4, 1.0, hidden, layers, kernel_hidden=256, **kw)
            assert net.padded and net.desc.hidden == 256
            for which, n_pad in (('Q', net.n_Q), ('pi', net.n_pi)):
                idx = net.ref_index(which)
                ref = [int(np.prod(s)) for s in net.var_shapes(which)]
                assert idx.size == sum(ref) and len(set(idx.tolist())) == idx.size and idx.max() < n_pad
                # walk the layers: element (i, j) of a [r, c] kernel lands at base + i * padded_c + j
                flat = np.arange(sum(ref), dtype=np.float64) + 1.0
                padded = np.zeros(n_pad)
                padded[idx] = flat
                k = kp = 0
                for s, ps in zip(net.var_shapes(which), net.var_shapes(which, 256)):
                    a = flat[k:k + int(np.prod(s))].reshape(s)
                    b = padded[kp:kp + int(np.prod(ps))].reshape(ps)
                    if len(s) == 2:
                        assert np.array_equal(b[:s[0], :s[1]], a) and b[s[0]:].sum() == 0 and b[:, s[1]:].sum() == 0
                    else:
                        assert np.array_equal(b[:s[0]], a) and b[s[0]:].sum() == 0
                    k += int(np.prod(s))
                    kp += int(np.prod(ps))
        same = cls(40, 12, 4, 1.0, 256, 3, kernel_hidden=256, **kw)
        assert not same.padded and np.array_equal(same.ref_index('Q'), np.arange(same.n_Q))


def _reference_action_postprocessing(u, randn, explore, u_rand, noise_eps, max_u):
    """ddpg.py:147-151 as NumPy evaluates the reference statements on the float32 policy output."""
    u = u.copy()
    noise = noise_eps * max_u * randn
    u += noise
    u = np.clip(u, -max_u, max_u)
    u += explore.reshape(-1, 1) * (u_rand - u)
    return u


@pytest.mark.parametrize('n,dimu,with_q', [(1, 4, False), (2, 4, False), (2, 4, True), (38, 4, True), (7, 3, True)])
def test_host_action_tail_equals_the_reference_statements(n, dimu, with_q):
    """cur_actions_finish_host (the host tail of the zero-copy get_actions path, pure host code) against the reference's own
    NumPy statements, bit for bit: float32 += float64, float32 clip, int64 * (float64 - float32)."""
    from curious_b200 import _lib
    lib = _lib.load()
    rng = np.random.RandomState(n * 10 + dimu)
    for trial in range(20):
        seq = 1 + trial
        max_u = [1.0, 0.7, 2.5][trial % 3]
        noise_eps = [0.2, 0.0, 1.3][trial % 3]
        u = (max_u * np.tanh(rng.randn(n, dimu) * 2)).astype(np.float32)
        q = rng.randn(n).astype(np.float32)
        words = np.zeros((n * (dimu + 1), 2), np.uint32)
        words[:n * dimu, 0] = u.reshape(-1).view(np.uint32)
        words[n * dimu:, 0] = q.view(np.uint32)
        words[:n * dimu + (n if with_q else 0), 1] = seq
        randn = rng.randn(n, dimu)
        explore = rng.binomial(1, 0.3, n).astype(np.int64)
        u_rand = rng.uniform(-max_u, max_u, (n, dimu))
        u_out = np.full((n, dimu), np.nan, np.float32)
        q_out = np.full(n, np.nan, np.float32)
        rc = lib.cur_actions_finish_host(words.ctypes.data, n, dimu, int(with_q), seq, randn.ctypes.data, explore.ctypes.data,
                                         u_rand.ctypes.data, float(noise_eps) * float(max_u), float(max_u), u_out.ctypes.data,
                                         q_out.ctypes.data if with_q else None, 1000)
        assert rc == 0
        want = _reference_action_postprocessing(u, randn, explore, u_rand, noise_eps, max_u)
        assert want.dtype == np.float32 and np.array_equal(u_out, want)
        if with_q:
            assert np.array_equal(q_out, q)
        # no draws (device-side noise or a caller that only wants the policy output): plain copy
        rc = lib.cur_actions_finish_host(words.ctypes.data, n, dimu, 0, seq, None, None, None, 0.0, float(max_u),
                                         u_out.ctypes.data, None, 1000)
        assert rc == 0 and np.array_equal(u_out, u)
        # one word still carries the previous call's number: the poll gives up after max_spins
        words[n * dimu - 1, 1] = seq - 1
        rc = lib.cur_actions_finish_host(words.ctypes.data, n, dimu, 0, seq, None, None, None, 0.0, float(max_u),
                                         u_out.ctypes.data, None, 1000)
        assert rc == 3


def test_scalar_randint_is_the_size_one_draw():
    """ReplayBuffer._get_storage_idx draws the slot of a full buffer with the scalar form of np.random.randint: same value,
    same stream position as the reference's np.random.randint(0, size, 1) (replay_buffer.py:99-102) for every size class."""
    rng = np.random.RandomState(0)
    sizes = [1, 2, 3, 5, 8, 9, 255, 256, 257, 1000, 20000, 65535, 65536, 65537, 10 ** 6, 2 ** 31 - 1, 2 ** 31, 2 ** 32 - 1,
             2 ** 32, 2 ** 32 + 5, 2 ** 40]
    for _ in range(400):
        n = int(rng.choice(sizes))
        seed = int(rng.randint(0, 2 ** 31 - 1))
        np.random.seed(seed)
        a = [int(np.random.randint(0, n, 1)[0]) for _ in range(4)]
        sa = np.random.get_state()
        np.random.seed(seed)
        b = [int(np.random.randint(0, n)) for _ in range(4)]
        sb = np.random.get_state()
        assert a == b and np.array_equal(sa[1], sb[1]) and sa[2:] == sb[2:], (n, seed)


def test_timeline_dump_without_a_recorded_timeline_is_an_error_not_a_crash():
    """cur_rows_timeline_dump (debug export) refuses politely when no update ran with CUR_ROWS_TIMELINE=1 (no CUDA call)."""
    from curious_b200 import _lib
    lib = _lib.load()
    assert lib.cur_rows_timeline_dump() == 1                      # CUR_ERR_INVALID
    assert b'timeline' in (lib.cur_last_error() or b'')
