"""Float64 restatement of DDPG._grads and the get_actions forward on the library's flat arenas, and a seeded case
generator whose rows stay clear of the ReLU kinks.

The update follows oracle/ddpg_oracle.ddpg_losses_and_grads term for term (normalise then clip, u / max_u in the critic
input, the target clip, the 2 / (B * dimu) L2 seed, and the loss_rows seed scaling of cur_ddpg_hyper), but evaluates
everything in float64 and splits each gradient into its named blocks.  Every block comes with a magnitude scale - the
largest entry of |X|^T |dY| for a weight block, of sum |dY| for a bias block - so that a kernel can be held to
`max|got - ref| <= tol * scale` block by block: an error in a small block (the bias of an 8-wide action head) does not
hide under the largest element of the flat vector, and cancellation in a bias sum does not make the bound flaky.

The generator (make_case) redraws every batch row in which a hidden pre-activation of a differentiated evaluation
(main pi, main Q(u), main Q(pi)) lies closer to zero than delta times its own magnitude sum: a float32 kernel then puts
every unit on the same side of the kink as this reference, and the comparison needs no fallback tolerance.
"""
import numpy as np

from oracle.ddpg_oracle import net_shapes

F64 = np.float64


# ------------------------------------------------------------------------------------------------
# arena layout
# ------------------------------------------------------------------------------------------------
def net_dims(desc, which):
    """(in_s, in_g, out) of net `which` ('Q' | 'pi') as the library lays it out (csrc/net_layout.cuh)."""
    act = desc.dimu if which == 'Q' else 0
    if desc.modular:
        return desc.dimo + desc.dimtd + act, desc.dimg, (1 if which == 'Q' else desc.dimu)
    return desc.dimo + desc.dimg + act, 0, (1 if which == 'Q' else desc.dimu)


def shapes(desc, which):
    in_s, in_g, out = net_dims(desc, which)
    return net_shapes(bool(desc.modular), in_s, in_g, desc.hidden, desc.layers, out)


def block_names(desc):
    head = ['W0s', 'b0', 'W0g'] if desc.modular else ['W0', 'b0']
    mid = []
    for l in range(1, desc.layers):
        mid += ['W%d' % l, 'b%d' % l]
    return head + mid + ['Wout', 'bout']


def arena_offsets(desc):
    """{'Q': offset, 'pi': offset} and the arena length, from the library (cur_theta_pi_offset)."""
    import ctypes as C
    from curious_b200 import _lib
    total = C.c_int64()
    off_pi = _lib.load().cur_theta_pi_offset(C.byref(desc), C.byref(total))
    assert off_pi >= 0
    n_q = _lib.load().cur_net_param_count(C.byref(desc), 0)
    n_pi = _lib.load().cur_net_param_count(C.byref(desc), 1)
    assert n_q == sum(int(np.prod(s)) for s in shapes(desc, 'Q'))
    assert n_pi == sum(int(np.prod(s)) for s in shapes(desc, 'pi'))
    return {'Q': 0, 'pi': int(off_pi)}, int(total.value)


def split(desc, flat, which, offset):
    """The blocks of net `which` in an arena-shaped vector, as float64 arrays keyed by block name."""
    out, k = {}, offset
    for name, s in zip(block_names(desc), shapes(desc, which)):
        n = int(np.prod(s))
        out[name] = np.asarray(flat[k:k + n], F64).reshape(s)
        k += n
    return out


def join(desc, blocks, which, arena, offset):
    k = offset
    for name, s in zip(block_names(desc), shapes(desc, which)):
        n = int(np.prod(s))
        arena[k:k + n] = np.asarray(blocks[name]).reshape(-1)
        k += n


# ------------------------------------------------------------------------------------------------
# forward / backward in float64
# ------------------------------------------------------------------------------------------------
def mlp(net, modular, layers, xs, xg):
    """Returns (y, cache).  cache: inputs, post-ReLU activations, and per hidden layer the pre-activation z and its
    magnitude sum sum_k |x_k w_k| + |b| (the scale of float32 rounding in z)."""
    if modular:
        z = xs @ net['W0s'] + net['b0'] + xg @ net['W0g']
        mag = np.abs(xs) @ np.abs(net['W0s']) + np.abs(net['b0']) + np.abs(xg) @ np.abs(net['W0g'])
        k0 = xs.shape[1] + xg.shape[1] + 1
    else:
        z = xs @ net['W0'] + net['b0']
        mag = np.abs(xs) @ np.abs(net['W0']) + np.abs(net['b0'])
        k0 = xs.shape[1] + 1
    pres, acts, ks = [(z, mag)], [], [k0]
    h = np.maximum(z, 0.0)
    acts.append(h)
    for l in range(1, layers):
        W, b = net['W%d' % l], net['b%d' % l]
        z = h @ W + b
        pres.append((z, np.abs(h) @ np.abs(W) + np.abs(b)))
        ks.append(h.shape[1] + 1)
        h = np.maximum(z, 0.0)
        acts.append(h)
    y = h @ net['Wout'] + net['bout']
    ymag = np.abs(h) @ np.abs(net['Wout']) + np.abs(net['bout'])
    return y, dict(xs=xs, xg=xg, acts=acts, pres=pres, ks=ks, ymag=ymag)


def mlp_back(net, modular, layers, cache, dy, want_params=True):
    """Backprop dy.  Returns (grads {name: array}, scales {name: float}, dxs)."""
    acts = cache['acts']
    g, sc = {}, {}

    def wblock(name, x, d):
        if want_params:
            g[name] = x.T @ d
            sc[name] = float((np.abs(x).T @ np.abs(d)).max()) if x.shape[1] else 0.0

    def bblock(name, d):
        if want_params:
            g[name] = d.sum(axis=0)
            sc[name] = float(np.abs(d).sum(axis=0).max())

    d = dy
    wblock('Wout', acts[-1], d)
    bblock('bout', d)
    d = (d @ net['Wout'].T) * (acts[-1] > 0)
    for l in range(layers - 1, 0, -1):
        wblock('W%d' % l, acts[l - 1], d)
        bblock('b%d' % l, d)
        d = (d @ net['W%d' % l].T) * (acts[l - 1] > 0)
    if modular:
        wblock('W0s', cache['xs'], d)
        bblock('b0', d)
        wblock('W0g', cache['xg'], d)
        dxs = d @ net['W0s'].T
    else:
        wblock('W0', cache['xs'], d)
        bblock('b0', d)
        dxs = d @ net['W0'].T
    return g, sc, dxs


def preprocess(desc, o, g, stats, ag=None, clip_obs=0.0):
    """get_actions / staged-batch preprocessing: relative goal, clip to +-clip_obs, then normalise and clip to
    +-norm_clip (ddpg.py:118-127, actor_critic.py:31-36; normalizer.py:72-77)."""
    o = np.asarray(o, F64)
    g = np.asarray(g, F64)
    if ag is not None:
        g = g - np.asarray(ag, F64)
    if clip_obs > 0:
        o = np.clip(o, -clip_obs, clip_obs)
        g = np.clip(g, -clip_obs, clip_obs)
    if desc.normalize_obs:
        c = float(desc.norm_clip)
        o = np.clip((o - stats['o_mean']) / stats['o_std'], -c, c)
        g = np.clip((g - stats['g_mean']) / stats['g_std'], -c, c)
    return o, g


def _pi(desc, net, o, g, td):
    xs, xg = (np.concatenate([o, td], axis=1), g) if desc.modular else (np.concatenate([o, g], axis=1), None)
    y, cache = mlp(net, desc.modular, desc.layers, xs, xg)
    th = np.tanh(y)
    return th, cache


def _q(desc, net, o, g, td, a):
    """Q(o, g, a) with a = u / max_u already applied."""
    if desc.modular:
        xs, xg = np.concatenate([o, td, a], axis=1), g
    else:
        xs, xg = np.concatenate([o, g, a], axis=1), None
    return mlp(net, desc.modular, desc.layers, xs, xg)


def nets(desc, theta):
    offs, _ = arena_offsets(desc)
    return {w: split(desc, theta, w, offs[w]) for w in ('Q', 'pi')}


def forward(desc, theta, o, g, td, stats=None, ag=None, clip_obs=0.0):
    """get_actions forward: (pi = max_u * tanh(net), Q(o, g, pi / max_u), the Q output's magnitude sum)."""
    N = nets(desc, theta)
    o, g = preprocess(desc, o, g, stats, ag, clip_obs)
    td = None if td is None else np.asarray(td, F64)
    th, _ = _pi(desc, N['pi'], o, g, td)
    q, qc = _q(desc, N['Q'], o, g, td, th)
    return float(desc.max_u) * th, q, qc['ymag']


def losses_and_grads(desc, theta_main, theta_target, batch, stats=None, gamma=0.98, clip_return=50.0,
                     clip_pos_returns=True, action_l2=1.0, loss_rows=0):
    """DDPG._grads in float64.  batch: dict o, g, u, td (or None), o_2, g_2, r.  Returns a dict with Q_loss, pi_loss,
    Q_pi [n, 1], Q_pi_mag (per-row magnitude sum of the Q_pi output), target, Q_grad / pi_grad / Q_scale / pi_scale
    ({block: array / float}), Q_loss_scale / pi_loss_scale (the loss plus the first-order change that per-row Q errors of
    one magnitude sum of the Q output would cause: mean(diff^2) + 2 mean(|diff| * mag(Q)), mean(mag(Q_pi)) +
    |action_l2| mean(th^2)), and per-row kink ratios (kink: min over the differentiated hidden units of
    |z| / (magnitude sum * sqrt(K) * 2^-24))."""
    max_u = float(desc.max_u)
    M, T = nets(desc, theta_main), nets(desc, theta_target)
    n = batch['o'].shape[0]
    Bl = loss_rows if loss_rows > 0 else n
    td = None if batch.get('td') is None else np.asarray(batch['td'], F64)
    o, g = preprocess(desc, batch['o'], batch['g'], stats)
    o2, g2 = preprocess(desc, batch['o_2'], batch['g_2'], stats)
    u = np.asarray(batch['u'], F64)
    r = np.asarray(batch['r'], F64).reshape(-1, 1)

    th, pi_cache = _pi(desc, M['pi'], o, g, td)
    Q_pi, qpi_cache = _q(desc, M['Q'], o, g, td, th)
    Q, q_cache = _q(desc, M['Q'], o, g, td, u / max_u)
    th_t, _ = _pi(desc, T['pi'], o2, g2, td)
    Q_t, _ = _q(desc, T['Q'], o2, g2, td, th_t)

    hi = 0.0 if clip_pos_returns else np.inf
    target = np.clip(r + gamma * Q_t, -clip_return, hi)
    diff = target - Q
    Q_loss = float(np.mean(diff * diff))
    pi_loss = float(-np.mean(Q_pi) + action_l2 * np.mean(th * th))

    dQ = (-2.0 / Bl) * diff
    Q_grad, Q_scale, _ = mlp_back(M['Q'], desc.modular, desc.layers, q_cache, dQ)
    dQpi = np.full((n, 1), -1.0 / Bl)
    _, _, dxs = mlp_back(M['Q'], desc.modular, desc.layers, qpi_cache, dQpi, want_params=False)
    in_s_pi = net_dims(desc, 'pi')[0]
    d_a = dxs[:, in_s_pi:in_s_pi + desc.dimu]          # action columns of the critic input: d pi_loss / d (pi / max_u)
    d_th = d_a + action_l2 * (2.0 / (Bl * desc.dimu)) * th
    dy = d_th * (1.0 - th * th)
    pi_grad, pi_scale, _ = mlp_back(M['pi'], desc.modular, desc.layers, pi_cache, dy)

    kink = np.full(n, np.inf)
    for c in (pi_cache, q_cache, qpi_cache):
        for (z, mag), k in zip(c['pres'], c['ks']):
            bound = np.maximum(mag, 1e-300) * np.sqrt(k) * 2.0 ** -24
            kink = np.minimum(kink, (np.abs(z) / bound).min(axis=1))
    return dict(Q_loss=Q_loss, pi_loss=pi_loss, Q_pi=Q_pi, Q_pi_mag=qpi_cache['ymag'], Q=Q, target=target,
                pi=max_u * th, Q_grad=Q_grad, pi_grad=pi_grad, Q_scale=Q_scale, pi_scale=pi_scale,
                pi_loss_scale=float(np.mean(qpi_cache['ymag']) + abs(action_l2) * np.mean(th * th)),
                Q_loss_scale=float(np.mean(diff * diff) + 2.0 * np.mean(np.abs(diff) * q_cache['ymag'])), kink=kink,
                lo_clip=float(np.mean(r + gamma * Q_t < -clip_return)),
                hi_clip=float(np.mean(r + gamma * Q_t > 0.0)) if clip_pos_returns else 0.0)


# ------------------------------------------------------------------------------------------------
# seeded cases
# ------------------------------------------------------------------------------------------------
KINK_FACTOR = 10.0      # delta = KINK_FACTOR * sqrt(K) * 2^-24: ten times the float32 rounding bound of a K-term sum


def random_net(rng, desc, which, bias=0.1):
    """Xavier-uniform kernels and non-zero uniform biases, in block order."""
    out = {}
    for name, s in zip(block_names(desc), shapes(desc, which)):
        if len(s) == 2:
            lim = np.sqrt(6.0 / (s[0] + s[1]))
            out[name] = rng.uniform(-lim, lim, s)
        else:
            out[name] = rng.uniform(-bias, bias, s)
    return out


def random_theta(rng, desc, q_out_scale=1.0, q_out_shift=0.0):
    offs, total = arena_offsets(desc)
    theta = np.zeros(total, np.float32)
    for w in ('Q', 'pi'):
        blocks = random_net(rng, desc, w)
        if w == 'Q':
            blocks['Wout'] = blocks['Wout'] * q_out_scale
            blocks['bout'] = blocks['bout'] * q_out_scale + q_out_shift
        join(desc, {k: v.astype(np.float32) for k, v in blocks.items()}, w, theta, offs[w])
    return theta


def random_stats(rng, desc):
    return {'o_mean': rng.normal(0.0, 0.5, desc.dimo).astype(np.float32),
            'o_std': rng.uniform(0.5, 2.0, desc.dimo).astype(np.float32),
            'g_mean': rng.normal(0.0, 0.3, desc.dimg).astype(np.float32),
            'g_std': rng.uniform(0.3, 1.5, desc.dimg).astype(np.float32)}


def random_rows(rng, desc, n):
    """o, o_2 ~ 2.5 N(0, 1) (large enough for a norm_clip of 3 to bind), goals ~ U(-1, 1), u ~ U(-max_u, max_u), one-hot
    task_descr, r in {-1, 0}."""
    max_u = float(desc.max_u)
    b = dict(o=2.5 * rng.standard_normal((n, desc.dimo)), o_2=2.5 * rng.standard_normal((n, desc.dimo)),
             g=rng.uniform(-1, 1, (n, desc.dimg)), g_2=rng.uniform(-1, 1, (n, desc.dimg)),
             u=rng.uniform(-max_u, max_u, (n, desc.dimu)), r=-(rng.uniform(0, 1, (n, 1)) < 0.5).astype(F64))
    b['td'] = np.eye(desc.dimtd)[rng.randint(0, desc.dimtd, n)] if desc.modular else None
    return {k: (None if v is None else v.astype(np.float32)) for k, v in b.items()}


def make_case(desc, n, seed, gamma=0.9, clip_pos_returns=True, action_l2=0.37, loss_rows=0, q_spread=4.0):
    """A kink-free case: main and target arenas (different draws), normaliser statistics, a batch of n rows, the
    hyperparameters, and the clip_return that binds on part of the rows.  Returns (case dict, acceptance rate)."""
    rng = np.random.RandomState(seed)
    main = random_theta(rng, desc)
    stats = random_stats(rng, desc) if desc.normalize_obs else None
    # target Q scaled and shifted so that Q_t spreads over about +-q_spread around 0: clip_return = 2 binds below on
    # part of the rows, and with clip_pos_returns the upper clip at 0 binds on the rows with a positive return
    target = random_theta(np.random.RandomState(seed + 1), desc)
    probe = random_rows(rng, desc, 256)
    q_t = forward(desc, target, probe['o_2'], probe['g_2'], probe['td'], stats)[1]
    scale = q_spread / max(float(np.std(q_t)), 1e-6)
    target = random_theta(np.random.RandomState(seed + 1), desc, q_out_scale=scale,
                          q_out_shift=-scale * float(np.median(q_t)))
    clip_return = 2.0
    hyper = dict(gamma=gamma, clip_return=clip_return, clip_pos_returns=clip_pos_returns, action_l2=action_l2,
                 loss_rows=loss_rows)
    rows, drawn, passed = {}, 0, 0
    need = n
    parts = []
    while need > 0:
        cand = random_rows(rng, desc, max(2 * need, 16))
        drawn += cand['o'].shape[0]
        ok = np.nonzero(losses_and_grads(desc, main, target, cand, stats, **hyper)['kink'] > KINK_FACTOR)[0]
        passed += len(ok)
        ok = ok[:need]
        parts.append({k: (None if v is None else v[ok]) for k, v in cand.items()})
        need -= len(ok)
        assert drawn < 100 * n + 1000, 'kink-free rows are too rare for this net'
    for k in parts[0]:
        rows[k] = None if parts[0][k] is None else np.concatenate([p[k] for p in parts])
    accepted = passed / float(drawn)
    return dict(desc=desc, n=n, main=main, target=target, stats=stats, batch=rows, hyper=hyper), accepted
