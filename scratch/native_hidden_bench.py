"""Hidden 64 / 128 at the true width (DDPG pad_hidden='native') against the zero-padded row kernels (pad_hidden='auto') and
the dependency-level kernels at the true width (pad_hidden=False), in ONE process: device-timed train() (CUDA graph, fused
HER + Adam) at batch 256 / 512 for Arm4 and Arm8 shapes, get_actions wall clock at n = 2 / 38.  The three arms run
alternately, REPS times each, on agents built from the same seed.  Afterwards native and padded agents of every shape are
checked against each other (losses and parameters after a few updates from the same start).

    python scratch/native_hidden_bench.py --out profiles/r03_native_hidden.json [--iters 200] [--reps 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from tests.ddpg_util import ddpg_kwargs, episode_stream, make_gpu_agent  # noqa: E402

ARMS = {'native': dict(pad_hidden='native'), 'padded': dict(pad_hidden='auto'), 'levels': dict(pad_hidden=False)}


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return dict(nvidia_smi=q.stdout.strip(), torch_name=torch.cuda.get_device_name(0))


def make(n_modules, hidden, batch, arm, seed=0):
    kw, dims, ag_ids, g_ids = ddpg_kwargs(n_modules, hidden=hidden, batch_size=batch)
    ag = make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='philox', buffer_episodes=200, seed=seed, **ARMS[arm])
    np.random.seed(0)
    n = 0
    cp = np.linspace(0.05, 0.3, n_modules)
    for ep in episode_stream(dims, kw['T'], 10):
        n += 2
        ag.store_episode(ep, cp, n)
    return ag, dims


def time_train(ag, iters):
    for _ in range(5):
        ag.train()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        ag.train()
    e1.record()
    torch.cuda.synchronize()
    return 1e3 * e0.elapsed_time(e1) / iters


def time_actions(ag, dims, n, calls):
    rng = np.random.RandomState(1)
    o = rng.standard_normal((n, dims['o'])).astype(np.float32)
    g = rng.uniform(-0.3, 0.3, (n, dims['g'])).astype(np.float32)
    a = rng.uniform(-0.3, 0.3, (n, dims['ag'])).astype(np.float32)
    td = np.eye(dims['task_descr'], dtype=np.float32)[rng.randint(0, dims['task_descr'], n)]
    for _ in range(20):
        ag.get_actions(o, a, g, task_descr=td, noise_eps=0.2, random_eps=0.3)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(calls):
        ag.get_actions(o, a, g, task_descr=td, noise_eps=0.2, random_eps=0.3)
    return 1e6 * (time.perf_counter() - t0) / calls


def agreement(n_modules, hidden, batch, steps=4):
    """native vs padded from the same seed: the same Philox batches; losses per update and parameters after `steps`."""
    (nat, _), (pad, _) = make(n_modules, hidden, batch, 'native', 5), make(n_modules, hidden, batch, 'padded', 5)
    losses = [[float(a.train()[0]) for _ in range(steps)] for a in (nat, pad)]
    out = dict(loss_rel=[abs(x - y) / max(abs(y), 1e-30) for x, y in zip(*losses)])
    for w in ('Q', 'pi'):
        a, b = nat.get_flat(w).astype(np.float64), pad.get_flat(w).astype(np.float64)
        err = np.abs(a - b)
        out[w] = dict(max_abs=float(err.max()), q999_over_scale=float(np.quantile(err, 0.999) / np.abs(b).max()))
    out['ok'] = bool(out['loss_rel'][0] <= 1e-5 and all(out[w]['q999_over_scale'] <= 2e-5 and
                                                         out[w]['max_abs'] <= steps * 1e-3 * 1.01 for w in ('Q', 'pi')))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True, help='path of the JSON record')
    ap.add_argument('--iters', type=int, default=200)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--calls', type=int, default=300)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'needs a CUDA device'
    rec = dict(gpu=gpu_info(), iters=args.iters, reps=args.reps, train_us={}, actions_us={}, paths={}, agreement={})
    for hidden in (64, 128):
        for n_modules in (4, 8):
            for batch in (256, 512):
                key = 'h%d_arm%d_b%d' % (hidden, n_modules, batch)
                agents = {arm: make(n_modules, hidden, batch, arm) for arm in ARMS}
                rec['paths'][key] = {arm: dict(padded=bool(a.net.padded), rows=bool(a._use_rows(batch)),
                                               action_rows=bool(a._action_rows_ok())) for arm, (a, _) in agents.items()}
                times = {arm: [] for arm in ARMS}
                for _ in range(args.reps):
                    for arm, (a, _) in agents.items():
                        times[arm].append(time_train(a, args.iters))
                rec['train_us'][key] = times
                print(key, {arm: ['%.1f' % t for t in v] for arm, v in times.items()}, flush=True)
                if batch == 256:
                    for n in (2, 38):
                        at = {arm: [] for arm in ARMS}
                        for _ in range(args.reps):
                            for arm, (a, dims) in agents.items():
                                at[arm].append(time_actions(a, dims, n, args.calls))
                        rec['actions_us']['h%d_arm%d_n%d' % (hidden, n_modules, n)] = at
                        print('  get_actions n=%d' % n, {arm: ['%.1f' % t for t in v] for arm, v in at.items()}, flush=True)
                rec['agreement'][key] = agreement(n_modules, hidden, batch)
                print('  agreement', rec['agreement'][key], flush=True)
                del agents
                torch.cuda.empty_cache()
    rec['gpu_after'] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(rec, f, indent=1)
    print('wrote', args.out)


if __name__ == '__main__':
    main()
