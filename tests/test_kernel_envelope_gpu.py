"""The DDPG update and action kernels at the edges of the shapes they accept, through the C ABI, against the float64
reference of tests/ddpg_f64.py.

The agent-level tests build every net from tests/ddpg_util.ddpg_kwargs (dimu 4, fan-in <= 100, max_u 1, action_l2 1, a
clip_return that never binds).  Here the net descriptions are written out by hand so that each kernel path runs at the
shapes it is sized for: a first layer exactly 256 wide (the rows kernel's input buffer and chunk budget), 8-wide action
heads, the chain kernel at exactly 8 input k-blocks and with tail columns in both input blocks, dimu 1-3, level kernels
at hidden 100 / 8 layers and at 1 or 3 rows.  Every case runs at max_u = 2.5, gamma = 0.9 and a clip_return that binds on
part of the rows, with action_l2, clip_pos_returns and normalize_obs varied across the cases.

Each case first asserts which path the library takes for it (cur_ddpg_rows_supported, cur_ddpg_chain_supported,
cur_ddpg_uses_chain, cur_ddpg_uses_tensor_cores), so that a changed predicate fails here instead of moving the case to
another kernel.  The batches are drawn kink-free (ddpg_f64.make_case), so every comparison is strict:
  losses            |got - ref| <= 1e-5 * (their magnitude scale, ddpg_f64.losses_and_grads)
  Q_pi, Q           |got - ref| <= 1e-5 * (magnitude sum of the output layer), per row
  gradients         max|got - ref| <= 2e-5 * scale(block), per named block, FFMA and 3xTF32 alike
  actions           |got - ref| <= 1e-5 * max_u
Outputs are pre-filled with NaN and followed by NaN guard rows: an element a kernel forgets, or a store past row n, fails.
Run with -rP to see the worst error of each case as a fraction of its bound, and the acceptance rate of the kink-free draw.
"""
import ctypes as C
import zlib

import numpy as np
import pytest

from curious_b200 import _lib
from tests import ddpg_f64 as F

MAX_U = 2.5
GAMMA = 0.9
NORM_CLIP = 3.0
GRAD_TOL = 2e-5         # the suite's GRAD_RTOL, now per block against the block's magnitude scale
LOSS_TOL = 1e-5
ACT_TOL = 1e-5
GUARD = 8               # NaN rows after every per-row output


def desc_of(modular, dimo, dimg, dimu, dimtd, hidden, layers, normalize_obs=0):
    return _lib.NetDesc(modular, dimo, dimg, dimu, dimtd, hidden, layers, MAX_U, normalize_obs, NORM_CLIP)


def predicates(d, n):
    lib = _lib.load()
    return dict(rows=lib.cur_ddpg_rows_supported(C.byref(d), n), chain=lib.cur_ddpg_chain_supported(C.byref(d), n),
                uses_chain=lib.cur_ddpg_uses_chain(C.byref(d), n), tc=lib.cur_ddpg_uses_tensor_cores(C.byref(d), n))


class switches(object):
    """cur_ddpg_set_tensor_cores / cur_ddpg_set_chain for the duration of a block; always back to the defaults."""

    def __init__(self, tc=-1, chain=-1):
        self.tc, self.chain = tc, chain

    def __enter__(self):
        lib = _lib.load()
        _lib.check(lib.cur_ddpg_set_tensor_cores(self.tc), 'cur_ddpg_set_tensor_cores')
        _lib.check(lib.cur_ddpg_set_chain(self.chain), 'cur_ddpg_set_chain')

    def __exit__(self, *exc):
        lib = _lib.load()
        lib.cur_ddpg_set_tensor_cores(-1)
        lib.cur_ddpg_set_chain(-1)
        return False


# ------------------------------------------------------------------------------------------------
# the support predicates at each edge (CPU: the library answers without a device)
# ------------------------------------------------------------------------------------------------
K256 = (1, 212, 28, 8, 8)          # modular, Q fan-in 228 + 28 = 256 exactly, dimu 8
FLAT256 = (0, 200, 48, 8, 0)       # flat, Q fan-in 200 + 48 + 8 = 256
K260 = (1, 216, 28, 8, 8)          # one column past the rows kernel's input buffer
KB8 = (1, 180, 64, 4, 8)           # chain: Q in_s 192 + in_g 64 = 8 k-blocks of 32 exactly
KB9 = (1, 181, 64, 4, 8)           # 9 k-blocks
TAILS = (1, 150, 33, 3, 8)         # Q in_s 161, in_g 33: tail columns in both input blocks
SMALL1 = (1, 25, 3, 1, 1)          # small odd inputs, dimu 1
DIMU3 = (1, 40, 12, 3, 4)          # dimu 3: the 16-byte column blocks of the rows kernel do not fit
LEVEL = (1, 25, 3, 6, 2)           # level kernels only

# (dims, hidden, layers, n, switches (tc, chain)) -> (rows_supported, chain_supported, uses_chain, uses_tensor_cores)
PREDICATE_TABLE = [
    (K256, 256, 4, 4, (-1, -1), (1, 0, 0, 0)),
    (K256, 256, 4, 12, (-1, -1), (1, 0, 0, 0)),
    (K256, 256, 4, 1020, (-1, -1), (1, 0, 0, 0)),
    (K256, 256, 4, 1024, (-1, -1), (1, 0, 0, 1)),
    (K256, 256, 4, 1028, (-1, -1), (0, 0, 0, 0)),
    (FLAT256, 256, 4, 4, (-1, -1), (1, 0, 0, 0)),
    (FLAT256, 256, 4, 1024, (-1, -1), (1, 0, 0, 1)),
    (K260, 256, 4, 256, (-1, -1), (0, 0, 0, 0)),
    (K256, 64, 1, 4, (-1, -1), (1, 0, 0, 0)),
    (K256, 64, 1, 256, (-1, -1), (1, 0, 0, 0)),
    (KB8, 256, 4, 1024, (-1, -1), (1, 1, 1, 1)),
    (KB8, 256, 4, 1152, (-1, -1), (0, 1, 1, 1)),
    (KB8, 256, 4, 256, (-1, -1), (1, 0, 0, 0)),
    (KB8, 256, 4, 256, (1, -1), (1, 1, 1, 1)),
    (KB9, 256, 4, 1024, (-1, -1), (0, 0, 0, 1)),
    (TAILS, 256, 3, 1024, (-1, -1), (0, 1, 1, 1)),
    (TAILS, 256, 3, 1024, (-1, 0), (0, 0, 0, 1)),
    (SMALL1, 64, 2, 128, (-1, -1), (0, 1, 0, 0)),
    (SMALL1, 64, 2, 1152, (-1, -1), (0, 1, 0, 0)),
    (SMALL1, 128, 2, 1152, (-1, -1), (0, 1, 0, 0)),
    (SMALL1, 64, 2, 1152, (-1, 0), (0, 0, 0, 0)),
    (DIMU3, 256, 2, 256, (-1, -1), (0, 0, 0, 0)),
    (LEVEL, 100, 8, 1, (-1, -1), (0, 0, 0, 0)),
    (LEVEL, 100, 8, 3, (-1, -1), (0, 0, 0, 0)),
    (LEVEL, 100, 8, 257, (-1, -1), (0, 0, 0, 0)),
]


def test_support_predicates_at_the_edges():
    bad = []
    for dims, hidden, layers, n, (tc, chain), want in PREDICATE_TABLE:
        with switches(tc, chain):
            p = predicates(desc_of(*dims, hidden, layers), n)
        got = (p['rows'], p['chain'], p['uses_chain'], p['tc'])
        if got != want:
            bad.append((dims, hidden, layers, n, (tc, chain), got, want))
    assert not bad, bad


# ------------------------------------------------------------------------------------------------
# the float64 reference itself (CPU)
# ------------------------------------------------------------------------------------------------
def test_f64_reference_against_finite_differences():
    """Central differences of the reference's own losses at a tiny net with every option on: the gradients it reports
    are d loss / d theta times batch / loss_rows (the loss_rows seed scaling)."""
    d = desc_of(1, 5, 3, 2, 2, 8, 2, normalize_obs=1)
    case, _ = F.make_case(d, 4, seed=7, gamma=GAMMA, clip_pos_returns=True, action_l2=0.37, loss_rows=2)
    kw = dict(case['hyper'])
    offs, _ = F.arena_offsets(d)
    ref = F.losses_and_grads(d, case['main'], case['target'], case['batch'], case['stats'], **kw)
    assert ref['lo_clip'] > 0 and ref['hi_clip'] > 0 and ref['lo_clip'] + ref['hi_clip'] < 1
    theta = case['main'].astype(np.float64)
    factor = 4 / 2.0
    h = 1e-6
    for which, loss in (('Q', 'Q_loss'), ('pi', 'pi_loss')):
        k = offs[which]
        for name, s in zip(F.block_names(d), F.shapes(d, which)):
            size = int(np.prod(s))
            fd = np.empty(size)
            for i in range(size):
                tp, tm = theta.copy(), theta.copy()
                tp[k + i] += h
                tm[k + i] -= h
                lp = F.losses_and_grads(d, tp, case['target'], case['batch'], case['stats'], **kw)[loss]
                lm = F.losses_and_grads(d, tm, case['target'], case['batch'], case['stats'], **kw)[loss]
                fd[i] = (lp - lm) / (2 * h) * factor
            got = ref[which + '_grad'][name].reshape(-1)
            scale = max(ref[which + '_scale'][name], 1e-12)
            assert np.abs(fd - got).max() <= 1e-7 * scale, (which, name, np.abs(fd - got).max(), scale)
            k += size


def test_f64_reference_matches_the_float32_oracle_at_arm4():
    from oracle import ddpg_oracle as O
    d = desc_of(1, 40, 12, 4, 4, 256, 3, normalize_obs=1)
    case, _ = F.make_case(d, 256, seed=5, gamma=GAMMA, clip_pos_returns=True, action_l2=0.37)
    hyp = case['hyper']
    st = case['stats']
    o_stats, g_stats = O.NormalizerOracle(d.dimo, default_clip_range=NORM_CLIP), O.NormalizerOracle(
        d.dimg, default_clip_range=NORM_CLIP)
    o_stats.mean, o_stats.std, g_stats.mean, g_stats.std = st['o_mean'], st['o_std'], st['g_mean'], st['g_std']
    ac = O.ActorCriticOracle(True, d.dimo, d.dimg, d.dimu, d.dimtd, d.hidden, d.layers, MAX_U, True, o_stats, g_stats)
    offs, _ = F.arena_offsets(d)
    nets = {}
    for tag, theta in (('main', case['main']), ('target', case['target'])):
        for w, shp in (('Q', ac.Q_shapes), ('pi', ac.pi_shapes)):
            n_w = sum(int(np.prod(s)) for s in shp)
            nets[tag, w] = O.unflatten(theta[offs[w]:offs[w] + n_w], shp)
    b = case['batch']
    batch = dict(o=b['o'], g=b['g'], u=b['u'], task_descr=b['td'], o_2=b['o_2'], g_2=b['g_2'], r=b['r'])
    want = O.ddpg_losses_and_grads(ac, nets['main', 'Q'], nets['main', 'pi'], nets['target', 'Q'], nets['target', 'pi'],
                                   batch, hyp['gamma'], hyp['clip_return'], hyp['clip_pos_returns'], hyp['action_l2'])
    ref = F.losses_and_grads(d, case['main'], case['target'], b, st, **hyp)
    assert abs(ref['Q_loss'] - want['Q_loss']) <= LOSS_TOL * ref['Q_loss_scale']
    assert abs(ref['pi_loss'] - want['pi_loss']) <= LOSS_TOL * ref['pi_loss_scale']
    assert np.all(np.abs(ref['Q_pi'] - want['Q_pi']) <= LOSS_TOL * ref['Q_pi_mag'])
    for which in ('Q', 'pi'):
        flat = np.zeros(max(offs.values()) + 1 + want[which + '_grad'].size, np.float32)
        flat[offs[which]:offs[which] + want[which + '_grad'].size] = want[which + '_grad']
        got = F.split(d, flat, which, offs[which])
        for name, g in ref[which + '_grad'].items():
            assert np.abs(got[name] - g).max() <= GRAD_TOL * ref[which + '_scale'][name], (which, name)


# ------------------------------------------------------------------------------------------------
# GPU plumbing
# ------------------------------------------------------------------------------------------------
def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda()


def _nan(n):
    import torch
    return torch.full((n,), float('nan'), dtype=torch.float32, device='cuda')


def _stats(case):
    st = case['stats']
    if st is None:
        return None, None
    keep = {k: _dev(v) for k, v in st.items()}
    return _lib.NormStats(keep['o_mean'].data_ptr(), keep['o_std'].data_ptr(), keep['g_mean'].data_ptr(),
                          keep['g_std'].data_ptr()), keep


def _batch(case):
    b = {k: (None if v is None else _dev(v)) for k, v in case['batch'].items()}
    cb = _lib.Batch(b['o'].data_ptr(), b['g'].data_ptr(), b['u'].data_ptr(), _lib.ptr(b['td']), b['o_2'].data_ptr(),
                    b['g_2'].data_ptr(), b['r'].data_ptr(), case['n'])
    return cb, b


def _hyper(case, step=None, loss_ring=0, transposes_valid=0):
    h = case['hyper']
    return _lib.DdpgHyper(gamma=h['gamma'], clip_return=h['clip_return'], action_l2=h['action_l2'],
                          clip_pos_returns=1 if h['clip_pos_returns'] else 0, step_counter=_lib.ptr(step),
                          loss_ring=loss_ring, micro_batches=0, grads_parity_stride=0, loss_rows=h['loss_rows'],
                          transposes_valid=transposes_valid)


def run_update(case, path):
    """One cur_ddpg_rows_step / cur_ddpg_chain_grads / cur_ddpg_grads call on fresh NaN-filled outputs."""
    import torch
    lib = _lib.load()
    d, n = case['desc'], case['n']
    _, total = F.arena_offsets(d)
    main, target = _dev(case['main']), _dev(case['target'])
    stats, keep_s = _stats(case)
    cb, keep_b = _batch(case)
    hyper = _hyper(case)
    grads, q_pi, q_loss, pi_loss = _nan(total), _nan(n + GUARD), _nan(1), _nan(1)
    sp = C.byref(stats) if stats is not None else None
    args = (_lib.stream_ptr(), C.byref(d), main.data_ptr(), target.data_ptr(), sp, C.byref(cb), C.byref(hyper))
    outs = (grads.data_ptr(), q_loss.data_ptr(), pi_loss.data_ptr(), q_pi.data_ptr())
    if path == 'rows':
        ws = torch.zeros(lib.cur_ddpg_rows_workspace_floats(C.byref(d), n), dtype=torch.float32, device='cuda')
        _lib.check(lib.cur_ddpg_rows_step(*args, ws.data_ptr(), *outs, None, None), 'cur_ddpg_rows_step')
    elif path == 'chain':
        ws = torch.zeros(lib.cur_ddpg_chain_workspace_floats(C.byref(d), n), dtype=torch.float32, device='cuda')
        _lib.check(lib.cur_ddpg_chain_grads(*args, ws.data_ptr(), *outs), 'cur_ddpg_chain_grads')
    else:
        ws = torch.zeros(lib.cur_ddpg_workspace_floats(C.byref(d), n), dtype=torch.float32, device='cuda')
        _lib.check(lib.cur_ddpg_grads(*args, ws.data_ptr(), *outs), 'cur_ddpg_grads')
    torch.cuda.synchronize()
    return dict(grads=grads.cpu().numpy(), q_pi=q_pi.cpu().numpy(), q_loss=float(q_loss.item()),
                pi_loss=float(pi_loss.item()))


def check_update(case, got, label, acceptance):
    """Every bound of the module docstring; returns and prints the worst error as a fraction of its bound."""
    d, n = case['desc'], case['n']
    ref = F.losses_and_grads(d, case['main'], case['target'], case['batch'], case['stats'], **case['hyper'])
    offs, _ = F.arena_offsets(d)
    ratios = {}
    ratios['Q_loss'] = abs(got['q_loss'] - ref['Q_loss']) / (LOSS_TOL * ref['Q_loss_scale'])
    ratios['pi_loss'] = abs(got['pi_loss'] - ref['pi_loss']) / (LOSS_TOL * ref['pi_loss_scale'])
    ratios['Q_pi'] = float((np.abs(got['q_pi'][:n] - ref['Q_pi'][:, 0]) / (LOSS_TOL * ref['Q_pi_mag'][:, 0])).max())
    assert np.isnan(got['q_pi'][n:]).all(), '%s: q_pi written past row n' % label
    for which in ('Q', 'pi'):
        blocks = F.split(d, got['grads'], which, offs[which])
        for name, want in ref[which + '_grad'].items():
            g = blocks[name]
            assert not np.isnan(g).any(), '%s: %s.%s not (entirely) written' % (label, which, name)
            ratios[which + '.' + name] = float(np.abs(g - want).max() / (GRAD_TOL * max(ref[which + '_scale'][name],
                                                                                        1e-30)))
    worst = max(ratios, key=ratios.get)
    print('[%s] worst %s at %.3f of its bound; kink-free draw accepted %.1f%% of rows; lower clip on %.0f%%, '
          'upper clip on %.0f%% of rows' % (label, worst, ratios[worst], 100 * acceptance, 100 * ref['lo_clip'],
                                            100 * ref['hi_clip']))
    bad = {k: v for k, v in ratios.items() if not v <= 1.0}
    assert not bad, (label, bad)
    return ratios


# ------------------------------------------------------------------------------------------------
# update cases: (name, dims, hidden, layers, n, path, switches, predicates (rows, chain, uses_chain, tc), options)
# options: normalize_obs, clip_pos_returns, action_l2, loss_rows
# ------------------------------------------------------------------------------------------------
UPDATE_CASES = [
    # rows schedule
    ('rows_k256_h256_l4_n1024', K256, 256, 4, 1024, 'rows', (-1, -1), (1, 0, 0, 1), (1, 1, 0.37, 0)),
    ('rows_k256_h256_l4_n4', K256, 256, 4, 4, 'rows', (-1, -1), (1, 0, 0, 0), (0, 0, 0.0, 0)),
    ('rows_k256_h256_l4_n1024_loss_rows', K256, 256, 4, 1024, 'rows', (-1, -1), (1, 0, 0, 1), (0, 1, 0.37, 256)),
    ('rows_k256_h256_l1_n1020', K256, 256, 1, 1020, 'rows', (-1, -1), (1, 0, 0, 0), (1, 0, 0.37, 0)),
    ('rows_k256_h128_l4_n12', K256, 128, 4, 12, 'rows', (-1, -1), (1, 0, 0, 0), (0, 1, 0.0, 0)),
    ('rows_k256_h128_l1_n252', K256, 128, 1, 252, 'rows', (-1, -1), (1, 0, 0, 0), (1, 1, 0.37, 0)),
    ('rows_k256_h64_l4_n20', K256, 64, 4, 20, 'rows', (-1, -1), (1, 0, 0, 0), (1, 0, 0.37, 0)),
    ('rows_k256_h64_l1_n1024', K256, 64, 1, 1024, 'rows', (-1, -1), (1, 0, 0, 0), (0, 1, 0.0, 0)),
    ('rows_flat256_h256_l4_n1024', FLAT256, 256, 4, 1024, 'rows', (-1, -1), (1, 0, 0, 1), (1, 1, 0.37, 0)),
    ('rows_flat256_h256_l4_n4', FLAT256, 256, 4, 4, 'rows', (-1, -1), (1, 0, 0, 0), (0, 0, 0.0, 0)),
    ('rows_dimu4_h256_l2_n252', KB8, 256, 2, 252, 'rows', (-1, -1), (1, 0, 0, 0), (1, 1, 0.37, 0)),
    # hidden-256 chain kernel through cur_ddpg_grads
    ('chain_kb8_l4_n1024', KB8, 256, 4, 1024, 'grads', (-1, -1), (1, 1, 1, 1), (1, 1, 0.37, 0)),
    ('chain_kb8_l2_n1152', KB8, 256, 2, 1152, 'grads', (-1, -1), (0, 1, 1, 1), (0, 0, 0.0, 0)),
    ('chain_kb8_l4_n256_tc', KB8, 256, 4, 256, 'grads', (1, -1), (1, 1, 1, 1), (0, 1, 0.37, 0)),
    ('chain_tails_dimu3_l3_n1024', TAILS, 256, 3, 1024, 'grads', (-1, -1), (0, 1, 1, 1), (1, 0, 0.37, 0)),
    ('chain_tails_dimu2_l2_n1152', (1, 150, 33, 2, 8), 256, 2, 1152, 'grads', (-1, -1), (0, 1, 1, 1), (1, 1, 0.0, 0)),
    ('chain_small_dimu1_l4_n1024', SMALL1, 256, 4, 1024, 'grads', (-1, -1), (0, 1, 1, 1), (0, 1, 0.37, 0)),
    # narrow chain (cur_ddpg_chain_grads)
    ('narrow_h64_l2_n128', SMALL1, 64, 2, 128, 'chain', (-1, -1), (0, 1, 0, 0), (1, 1, 0.37, 0)),
    ('narrow_h64_l4_n1152', SMALL1, 64, 4, 1152, 'chain', (-1, -1), (0, 1, 0, 0), (0, 0, 0.0, 0)),
    ('narrow_h128_l2_n128', SMALL1, 128, 2, 128, 'chain', (-1, -1), (0, 1, 0, 0), (0, 1, 0.37, 0)),
    ('narrow_h128_l2_n1152', SMALL1, 128, 2, 1152, 'chain', (-1, -1), (0, 1, 0, 0), (1, 0, 0.37, 0)),
    # level kernels
    ('levels_h100_l8_n1', LEVEL, 100, 8, 1, 'grads', (-1, -1), (0, 0, 0, 0), (1, 1, 0.37, 0)),
    ('levels_h100_l8_n3', LEVEL, 100, 8, 3, 'grads', (-1, -1), (0, 0, 0, 0), (0, 0, 0.0, 0)),
    ('levels_h100_l8_n257', LEVEL, 100, 8, 257, 'grads', (-1, -1), (0, 0, 0, 0), (1, 0, 0.37, 0)),
    ('levels_tc_tails_l3_n1024', TAILS, 256, 3, 1024, 'grads', (-1, 0), (0, 0, 0, 1), (0, 1, 0.37, 0)),
]


def build_case(name, dims, hidden, layers, n, opts):
    normalize, clip_pos, l2, loss_rows = opts
    d = desc_of(*dims, hidden, layers, normalize_obs=normalize)
    return F.make_case(d, n, seed=zlib.crc32(name.encode()) & 0xffff, gamma=GAMMA, clip_pos_returns=bool(clip_pos),
                       action_l2=l2, loss_rows=loss_rows)


@pytest.mark.gpu
@pytest.mark.parametrize('name,dims,hidden,layers,n,path,sw,want,opts', UPDATE_CASES, ids=[c[0] for c in UPDATE_CASES])
def test_update_kernel_against_f64(name, dims, hidden, layers, n, path, sw, want, opts):
    case, acceptance = build_case(name, dims, hidden, layers, n, opts)
    with switches(*sw):
        p = predicates(case['desc'], n)
        assert (p['rows'], p['chain'], p['uses_chain'], p['tc']) == want, (name, p)
        got = run_update(case, path)
    check_update(case, got, name, acceptance)


# ------------------------------------------------------------------------------------------------
# rows schedule with the fused optimiser
# ------------------------------------------------------------------------------------------------
def _np_adam(theta, g, m, v, neg_a, b1, b2, eps):
    """MpiAdamOracle.update's float32 arithmetic with the step scale neg_a = float32(-a_t)."""
    f = np.float32
    m = (f(b1) * m + f(1 - b1) * g).astype(f)
    v = (f(b2) * v + f(1 - b2) * (g * g)).astype(f)
    step = (f(neg_a) * m / (np.sqrt(v) + f(eps))).astype(f)
    return (theta + step).astype(f), m, v


@pytest.mark.gpu
def test_rows_fused_adam_at_fan_in_256():
    """The stepped theta / m / v equal float32 NumPy Adam of the gradient the same kernel writes without the optimiser,
    bit for bit; a second step that trusts the W^T tiles the first step's epilogue wrote equals a second step on a fresh
    workspace that transposes theta itself, bit for bit."""
    import torch
    lib = _lib.load()
    d = desc_of(*K256, 256, 4, normalize_obs=1)
    n = 256
    case, _ = F.make_case(d, n, seed=11, gamma=GAMMA, clip_pos_returns=True, action_l2=0.37)
    offs, total = F.arena_offsets(d)
    nets = [(offs[w], offs[w] + sum(int(np.prod(s)) for s in F.shapes(d, w))) for w in ('Q', 'pi')]
    rng = np.random.RandomState(12)
    m0 = (rng.standard_normal(total) * 1e-3).astype(np.float32)
    v0 = (rng.uniform(0.0, 1e-5, total)).astype(np.float32)
    b1, b2, eps = 0.9, 0.999, 1e-8
    table = np.array([-1e-3, -7e-4, -5e-4], np.float32)
    stats, keep_s = _stats(case)
    cb, keep_b = _batch(case)
    target = _dev(case['target'])
    tab = _dev(table)
    sp = C.byref(stats)

    def call(theta, m, v, ws, step, adam_valid=None):
        hyper = _hyper(case, step=step, loss_ring=1)
        grads, q_pi, ql, pl = _nan(total), _nan(n + GUARD), _nan(1), _nan(1)
        adam = None
        if adam_valid is not None:
            adam = _lib.AdamFused(m.data_ptr(), v.data_ptr(), tab.data_ptr(), len(table), adam_valid, b1, b2, eps, None)
        _lib.check(lib.cur_ddpg_rows_step(_lib.stream_ptr(), C.byref(d), theta.data_ptr(), target.data_ptr(), sp,
                                          C.byref(cb), C.byref(hyper), ws.data_ptr(), grads.data_ptr(), ql.data_ptr(),
                                          pl.data_ptr(), q_pi.data_ptr(), C.byref(adam) if adam else None, None),
                   'cur_ddpg_rows_step')
        torch.cuda.synchronize()
        assert np.isnan(q_pi[n:].cpu().numpy()).all()
        return grads.cpu().numpy()

    def ws_new():
        return torch.zeros(lib.cur_ddpg_rows_workspace_floats(C.byref(d), n), dtype=torch.float32, device='cuda')

    assert lib.cur_ddpg_rows_supported(C.byref(d), n) == 1
    step = torch.zeros(1, dtype=torch.int64, device='cuda')
    g = call(_dev(case['main']), None, None, ws_new(), step)
    for a, b in nets:
        assert not np.isnan(g[a:b]).any()
    # first fused step, t = 1
    theta, m, v = _dev(case['main']), _dev(m0), _dev(v0)
    ws = ws_new()
    step.zero_()
    call(theta, m, v, ws, step, adam_valid=0)
    assert int(step.item()) == 1
    want_t, want_m, want_v = _np_adam(case['main'], g, m0, v0, table[0], b1, b2, eps)
    for got, want, what in ((theta, want_t, 'theta'), (m, want_m, 'm'), (v, want_v, 'v')):
        got = got.cpu().numpy()
        for a, b in nets:
            assert np.array_equal(got[a:b].view(np.uint32), want[a:b].view(np.uint32)), what
    # second step, t = 2: transposes from the epilogue vs. a fresh workspace
    theta1, m1, v1 = theta.clone(), m.clone(), v.clone()
    call(theta, m, v, ws, step, adam_valid=1)
    step2 = torch.ones(1, dtype=torch.int64, device='cuda')
    call(theta1, m1, v1, ws_new(), step2, adam_valid=0)
    for x, y, what in ((theta, theta1, 'theta'), (m, m1, 'm'), (v, v1, 'v')):
        x, y = x.cpu().numpy(), y.cpu().numpy()
        for a, b in nets:
            assert np.array_equal(x[a:b].view(np.uint32), y[a:b].view(np.uint32)), what
    print('[rows fused Adam] step 1 equals NumPy Adam of the gradients-only call bit for bit; step 2 with '
          'transposes_valid = 1 equals a fresh workspace bit for bit')


# ------------------------------------------------------------------------------------------------
# action kernels
# ------------------------------------------------------------------------------------------------
def action_inputs(d, n, seed):
    rng = np.random.RandomState(seed)
    o = 2.5 * rng.standard_normal((n, d.dimo))
    o[::7] *= 3.0                                          # rows past clip_obs
    ag = rng.uniform(-1.5, 1.5, (n, d.dimg))
    g = rng.uniform(-2.0, 2.0, (n, d.dimg))
    td = np.eye(d.dimtd)[rng.randint(0, d.dimtd, n)] if d.modular else None
    return {k: (None if v is None else v.astype(np.float32)) for k, v in dict(o=o, ag=ag, g=g, td=td).items()}


CLIP_OBS = 5.0


def _decode(words, count, seq):
    w = words.view(np.uint32).reshape(-1, 2)
    assert (w[:count, 1] == seq).all(), 'a word without the call number'
    return w[:count, 0].copy().view(np.float32)


def check_actions(d, theta, stats, inp, pi, q, label):
    n = inp['o'].shape[0]
    ref_pi, ref_q, qmag = F.forward(d, theta, inp['o'], inp['g'], inp['td'], stats, ag=inp['ag'], clip_obs=CLIP_OBS)
    r_pi = float(np.abs(pi.reshape(n, d.dimu) - ref_pi).max() / (ACT_TOL * MAX_U))
    r_q = 0.0 if q is None else float((np.abs(q.reshape(n, 1) - ref_q) / (ACT_TOL * qmag)).max())
    print('[%s] pi at %.3f, Q at %.3f of its bound' % (label, r_pi, r_q))
    assert r_pi <= 1.0 and r_q <= 1.0, (label, r_pi, r_q)


ACTION_N = [1, 3, 5, 4093, 4096]


@pytest.mark.gpu
@pytest.mark.parametrize('n', ACTION_N)
def test_action_kernels_at_fan_in_256(n):
    """cur_ddpg_actions_rows (float32 and word forms, with and without Q) and cur_ddpg_actions against the float64
    forward: dimu 8, first-layer fan-in 256, relative goals, a binding clip_obs and a binding norm_clip."""
    import torch
    lib = _lib.load()
    d = desc_of(*K256, 256, 4, normalize_obs=1)
    rng = np.random.RandomState(n)
    theta = F.random_theta(rng, d)
    st = F.random_stats(rng, d)
    inp = action_inputs(d, n, seed=100 + n)
    o_cl = np.clip(inp['o'], -CLIP_OBS, CLIP_OBS)
    assert (o_cl != inp['o']).any() and (np.abs((o_cl - st['o_mean']) / st['o_std']) > NORM_CLIP).any()
    stats, keep_s = _stats(dict(stats=st))
    dev = {k: _dev(v) for k, v in inp.items()}
    th = _dev(theta)
    ptrs = (dev['o'].data_ptr(), dev['ag'].data_ptr(), dev['g'].data_ptr(), dev['td'].data_ptr())
    for with_q in (False, True):
        for seq in (0, 7):
            if seq == 0:
                pi, q = _nan(n * d.dimu + GUARD), (_nan(n + GUARD) if with_q else None)
            else:
                pi = torch.full((n * d.dimu + GUARD,), -1, dtype=torch.int64, device='cuda')
                q = torch.full((n + GUARD,), -1, dtype=torch.int64, device='cuda') if with_q else None
            _lib.check(lib.cur_ddpg_actions_rows(_lib.stream_ptr(), C.byref(d), th.data_ptr(), C.byref(stats), *ptrs, n,
                                                 CLIP_OBS, pi.data_ptr(), _lib.ptr(q), seq), 'cur_ddpg_actions_rows')
            torch.cuda.synchronize()
            pi_h = pi.cpu().numpy()
            q_h = None if q is None else q.cpu().numpy()
            if seq == 0:
                assert np.isnan(pi_h[n * d.dimu:]).all() and (q_h is None or np.isnan(q_h[n:]).all())
                got_pi, got_q = pi_h[:n * d.dimu], (None if q_h is None else q_h[:n])
            else:
                assert (pi_h[n * d.dimu:] == -1).all() and (q_h is None or (q_h[n:] == -1).all())
                got_pi = _decode(pi_h, n * d.dimu, seq)
                got_q = None if q_h is None else _decode(q_h, n, seq)
            check_actions(d, theta, st, inp, got_pi, got_q, 'actions_rows n=%d q=%d seq=%d' % (n, with_q, seq))
    ws = torch.zeros(lib.cur_ddpg_workspace_floats(C.byref(d), n), dtype=torch.float32, device='cuda')
    pi, q = _nan(n * d.dimu + GUARD), _nan(n + GUARD)
    _lib.check(lib.cur_ddpg_actions(_lib.stream_ptr(), C.byref(d), th.data_ptr(), C.byref(stats), *ptrs, n, CLIP_OBS,
                                    ws.data_ptr(), pi.data_ptr(), q.data_ptr()), 'cur_ddpg_actions')
    torch.cuda.synchronize()
    pi_h, q_h = pi.cpu().numpy(), q.cpu().numpy()
    assert np.isnan(pi_h[n * d.dimu:]).all() and np.isnan(q_h[n:]).all()
    check_actions(d, theta, st, inp, pi_h[:n * d.dimu], q_h[:n], 'actions levels n=%d' % n)


@pytest.mark.gpu
def test_routed_action_launch_with_empty_experts():
    """cur_ddpg_actions_rows_group: 512 rows over 16 experts of their own weights and statistics, three experts
    without a row; every row against the float64 forward of its expert."""
    import torch
    lib = _lib.load()
    d = desc_of(*K256, 128, 2, normalize_obs=1)
    n, n_e = 512, 16
    rng = np.random.RandomState(21)
    thetas = [F.random_theta(rng, d) for _ in range(n_e)]
    sts = [F.random_stats(rng, d) for _ in range(n_e)]
    live = [e for e in range(n_e) if e not in (3, 7, 12)]
    row_expert = np.asarray(rng.choice(live, n), np.int32)
    inp = action_inputs(d, n, seed=22)
    dev = {k: _dev(v) for k, v in inp.items()}
    keep, experts = [], (_lib.ActionsExpert * n_e)()
    for e in range(n_e):
        t = _dev(thetas[e])
        s, ks = _stats(dict(stats=sts[e]))
        keep += [t, ks]
        experts[e].theta = t.data_ptr()
        experts[e].stats = s
    for seq in (0, 9):
        if seq == 0:
            pi, q = _nan(n * d.dimu + GUARD), _nan(n + GUARD)
        else:
            pi = torch.full((n * d.dimu + GUARD,), -1, dtype=torch.int64, device='cuda')
            q = torch.full((n + GUARD,), -1, dtype=torch.int64, device='cuda')
        _lib.check(lib.cur_ddpg_actions_rows_group(_lib.stream_ptr(), C.byref(d), n_e, experts,
                                                   row_expert.ctypes.data, dev['o'].data_ptr(), dev['ag'].data_ptr(),
                                                   dev['g'].data_ptr(), dev['td'].data_ptr(), n, CLIP_OBS, pi.data_ptr(),
                                                   q.data_ptr(), seq), 'cur_ddpg_actions_rows_group')
        torch.cuda.synchronize()
        pi_h, q_h = pi.cpu().numpy(), q.cpu().numpy()
        if seq == 0:
            assert np.isnan(pi_h[n * d.dimu:]).all() and np.isnan(q_h[n:]).all()
            got_pi, got_q = pi_h[:n * d.dimu].reshape(n, d.dimu), q_h[:n]
        else:
            assert (pi_h[n * d.dimu:] == -1).all() and (q_h[n:] == -1).all()
            got_pi, got_q = _decode(pi_h, n * d.dimu, seq).reshape(n, d.dimu), _decode(q_h, n, seq)
        for e in live:
            rows = np.nonzero(row_expert == e)[0]
            sub = {k: v[rows] for k, v in inp.items()}
            check_actions(d, thetas[e], sts[e], sub, got_pi[rows], got_q[rows],
                          'actions group expert %d (%d rows) seq=%d' % (e, len(rows), seq))
