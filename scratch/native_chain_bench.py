"""Hidden 64 / 128 above 1024 rows: the chain kernel at the true width (DDPG pad_hidden='native', cur_ddpg_chain_grads)
against the dependency-level kernels at the true width (pad_hidden=False, what 'native' ran there before) and the
zero-padded 256-wide chain (pad_hidden=True), in ONE process: device-timed train() through the CUDA graph (one rank, Adam in
the graph) for Arm4 and Arm8 shapes at 1152 / 2048 / 4096 / 4864 rows, plus the update of workers_per_rank=19 at batch 256
(native: one 4864-row chain update; native micro: 19 accumulating row-kernel launches, what 'native' ran before; padded:
the 256-wide chain).  The arms run alternately, REPS times each, on agents built from the same seed; the record keeps every
repetition and the median.

    python scratch/native_chain_bench.py --out profiles/r04_native_chain.json [--iters 100] [--reps 3]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from tests.ddpg_util import ddpg_kwargs, episode_stream, make_gpu_agent  # noqa: E402

ARMS = {'native': dict(pad_hidden='native'), 'levels': dict(pad_hidden=False), 'padded': dict(pad_hidden=True)}
WORKER_ARMS = {'native': dict(pad_hidden='native'), 'native_micro': dict(pad_hidden='native', workers_mode='micro'),
               'padded': dict(pad_hidden=True)}


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return dict(nvidia_smi=q.stdout.strip(), torch_name=torch.cuda.get_device_name(0))


def make(n_modules, hidden, batch, extra, workers=1, seed=0):
    kw, dims, ag_ids, g_ids = ddpg_kwargs(n_modules, hidden=hidden, batch_size=batch)
    ag = make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='philox', buffer_episodes=200, seed=seed,
                        workers_per_rank=workers, **extra)
    np.random.seed(0)
    n = 0
    cp = np.linspace(0.05, 0.3, n_modules)
    for ep in episode_stream(dims, kw['T'], 10):
        n += 2
        ag.store_episode(ep, cp, n)
    return ag


def path_of(ag, rows):
    if ag._use_rows(rows):
        return 'rows'
    if ag._use_native_chain(rows):
        return 'chain_native'
    return 'chain_256' if ag.net.padded else 'levels'


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


def run_arms(agents, iters, reps):
    times = {arm: [] for arm in agents}
    for _ in range(reps):
        for arm, a in agents.items():
            times[arm].append(time_train(a, iters))
    return dict(reps=times, median={arm: float(np.median(v)) for arm, v in times.items()})


def agreement(n_modules, hidden, rows, steps=4):
    """native chain vs levels at the true width from the same seed (same Philox batches): loss per update, parameters after
    `steps` updates as the 99.9 % quantile and the maximum of |difference| (test_native_chain_gpu.py holds the quantile to
    4e-4 of the parameter scale)."""
    a, b = make(n_modules, hidden, rows, ARMS['native'], seed=5), make(n_modules, hidden, rows, ARMS['levels'], seed=5)
    losses = [[float(x.train()[0]) for _ in range(steps)] for x in (a, b)]
    out = dict(loss_rel=[abs(x - y) / max(abs(y), 1e-30) for x, y in zip(*losses)])
    for w in ('Q', 'pi'):
        p, q = a.get_flat(w).astype(np.float64), b.get_flat(w).astype(np.float64)
        err = np.abs(p - q)
        out[w] = dict(max_abs=float(err.max()), q999_over_scale=float(np.quantile(err, 0.999) / np.abs(q).max()))
    return out


def kernel_profile(n_modules, hidden, rows, iters=20):
    """Device time per eager update of every kernel of the native chain schedule (torch.profiler, its own pass): shows
    what the K-sliced FFMA weight gradients (grouped_gemm_kernel, dw_slice_sum_kernel) cost next to the chain kernel."""
    from torch.profiler import ProfilerActivity, profile
    kw, dims, ag_ids, g_ids = ddpg_kwargs(n_modules, hidden=hidden, batch_size=rows)
    ag = make_gpu_agent(kw, dims, ag_ids, g_ids, her_rng='numpy', buffer_episodes=200, pad_hidden='native')
    np.random.seed(0)
    for i, ep in enumerate(episode_stream(dims, kw['T'], 10)):
        ag.store_episode(ep, np.linspace(0.05, 0.3, n_modules), 2 * (i + 1))
    assert ag._use_native_chain(rows)
    ag.stage_batch(ag.sample_batch())
    for _ in range(3):
        ag._grads()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            ag._grads()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, 'device_time_total', None)
        if t is None:
            t = e.cuda_time_total
        if t > 0:
            out[e.key[:80]] = dict(us_per_update=float(t) / iters, launches_per_update=e.count / iters)
    return out


def save(path, rec):
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, 'w') as f:
        json.dump(rec, f, indent=1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True, help='path of the JSON record')
    ap.add_argument('--iters', type=int, default=100)
    ap.add_argument('--reps', type=int, default=3)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'needs a CUDA device'
    rec = dict(gpu=gpu_info(), iters=args.iters, reps=args.reps, unit='us per train() update, CUDA graph, device events',
               train_us={}, paths={}, workers19_us={}, workers19_paths={}, agreement={}, kernels={})
    for hidden in (64, 128):
        for n_modules in (4, 8):
            for rows in (1152, 2048, 4096, 4864):
                key = 'h%d_arm%d_b%d' % (hidden, n_modules, rows)
                agents = {arm: make(n_modules, hidden, rows, extra) for arm, extra in ARMS.items()}
                rec['paths'][key] = {arm: path_of(a, rows) for arm, a in agents.items()}
                rec['train_us'][key] = run_arms(agents, args.iters, args.reps)
                print(key, rec['paths'][key], {k: '%.1f' % v for k, v in rec['train_us'][key]['median'].items()},
                      flush=True)
                del agents
                torch.cuda.empty_cache()
                save(args.out, rec)                   # partial records survive an interrupted run
                if n_modules == 4 and rows in (1152, 4864):
                    rec['agreement'][key] = agreement(n_modules, hidden, rows)
                    rec['kernels'][key] = kernel_profile(n_modules, hidden, rows)
                    print('  agreement', rec['agreement'][key], flush=True)
                    print('  kernels', {k: '%.1f' % v['us_per_update'] for k, v in rec['kernels'][key].items()}, flush=True)
        for n_modules in (4, 8):
            key = 'h%d_arm%d_b256_w19' % (hidden, n_modules)
            agents = {arm: make(n_modules, hidden, 256, extra, workers=19) for arm, extra in WORKER_ARMS.items()}
            rec['workers19_us'][key] = run_arms(agents, max(10, args.iters // 2), args.reps)
            rec['workers19_paths'][key] = {arm: dict(wide=bool(a._wide), graph_rows=int(a._graph_rows),
                                                     path=path_of(a, a._graph_rows)) for arm, a in agents.items()}
            print(key, rec['workers19_paths'][key],
                  {k: '%.1f' % v for k, v in rec['workers19_us'][key]['median'].items()}, flush=True)
            del agents
            torch.cuda.empty_cache()
    sel = [k for k, p in rec['paths'].items() if p['native'] == 'chain_native']
    rec['native_chain_faster_than_levels'] = {k: bool(rec['train_us'][k]['median']['native'] <
                                                      rec['train_us'][k]['median']['levels']) for k in sel}
    rec['gpu_after'] = gpu_info()
    save(args.out, rec)
    print('wrote', args.out)


if __name__ == '__main__':
    main()
