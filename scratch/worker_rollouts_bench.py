"""Virtual workers (RolloutWorker(workers=k), make_experiment(workers_per_rank=k)) on one GPU:

  * the acting step, host to host: DDPG.get_actions_workers over k * B rows (one launch) against a loop of k
    get_actions calls of B rows (what k lone agents cost), host and device noise, k = 1, 3, 19;
  * one training cycle (k-worker rollouts + store_episode + n_batches updates + update_target_net) and one epoch
    (n_cycles cycles + n_test_rollouts evaluation rollouts), k = 1, 3, 19 (k = 1: today's make_experiment);
  * the GPU name, power limit and SM clock, read in the same run.

    python scratch/worker_rollouts_bench.py --out profiles/r10_worker_rollouts.json
"""
import argparse
import json
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, __file__.rsplit('/scratch/', 1)[0])


def gpu_info():
    q = 'name,power.limit,clocks.sm,clocks.max.sm'
    out = subprocess.run(['nvidia-smi', '--query-gpu=' + q, '--format=csv,noheader'], capture_output=True, text=True)
    return dict(zip(q.split(','), [x.strip() for x in out.stdout.strip().splitlines()[0].split(',')])) if out.stdout else {}


def acting(k, noise, B=2, steps=300, warmup=50):
    from curious_b200.train import make_experiment
    from curious_b200.workers import WorkerStreams
    exp = make_experiment(nb_tasks=4, structure='curious', buffer_size=10000, seed=0,
                          policy_kwargs=dict(action_noise=noise))
    pol = exp['policy']
    d = pol.input_dims
    streams = WorkerStreams(0, k)
    rng = np.random.RandomState(0)
    n = k * B
    o, g = rng.randn(n, d['o']).astype(np.float32), rng.randn(n, d['g']).astype(np.float32)
    td = np.eye(d['task_descr'], dtype=np.float32)[rng.randint(0, d['task_descr'], n)]
    ne, re = [0.2] * k, [0.3] * k

    def one():
        pol.get_actions_workers(o, o, g, td, noise_eps=ne, random_eps=re, streams=streams)

    def loop():
        for j in range(k):
            rows = slice(j * B, (j + 1) * B)
            with streams.use(j):
                pol.get_actions(o[rows], o[rows], g[rows], task_descr=td[rows], noise_eps=0.2, random_eps=0.3)
    res = {}
    for name, fn in (('one_launch', one), ('loop_of_k_calls', loop)):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()                          # every call returns host actions: host to host
        torch.cuda.synchronize()
        res[name + '_us'] = round(1e6 * (time.perf_counter() - t0) / steps, 2)
    return res


def training(k, n_cycles=10, n_batches=40, n_test_rollouts=10):
    from curious_b200.train import _evaluate, make_experiment
    np.random.seed(0)
    exp = make_experiment(nb_tasks=4, n_controllable=3, structure='curious', buffer_size=100000, n_cycles=n_cycles,
                          n_batches=n_batches, n_test_rollouts=n_test_rollouts, seed=0, workers_per_rank=k)
    pol, w, ev = exp['policy'], exp['rollout_worker'], exp['evaluator']

    def cycle():
        ep, cp, n = w.generate_rollouts()
        pol.store_episode(ep, cp, n)
        for _ in range(n_batches):
            pol.train()
        pol.update_target_net()
    for _ in range(3):                    # warm-up: graph capture, workspaces, slots
        cycle()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    reps = 5
    for _ in range(reps):
        cycle()
    torch.cuda.synchronize()
    t_cycle = (time.perf_counter() - t0) / reps
    t0 = time.perf_counter()
    for _ in range(n_cycles):
        cycle()
    _evaluate(ev, n_test_rollouts)
    torch.cuda.synchronize()
    t_epoch = time.perf_counter() - t0
    T = w.T
    return dict(cycle_ms=round(1e3 * t_cycle, 2), epoch_s=round(t_epoch, 3), n_cycles=n_cycles, n_batches=n_batches,
                n_test_rollouts=n_test_rollouts, rollout_batch_size=w.rollout_batch_size, T=T,
                env_steps_per_cycle=k * w.rollout_batch_size * T)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--workers', default='1,3,19')
    args = ap.parse_args()
    ks = [int(x) for x in args.workers.split(',')]
    rec = dict(command=' '.join(['python'] + sys.argv), gpu_before=gpu_info(), acting={}, training={})
    for k in ks:
        for noise in ('host', 'device'):
            rec['acting']['k%d_%s' % (k, noise)] = acting(k, noise)
            print('acting', k, noise, rec['acting']['k%d_%s' % (k, noise)], flush=True)
    for k in ks:
        rec['training']['k%d' % k] = training(k)
        print('training', k, rec['training']['k%d' % k], flush=True)
    rec['gpu_after'] = gpu_info()
    print(json.dumps(rec))
    if args.out:
        with open(args.out, 'w') as f:
            json.dump(rec, f, indent=1)


if __name__ == '__main__':
    main()
