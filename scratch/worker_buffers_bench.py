"""worker_buffers='own' against 'shared' on Arm4 (hidden 256, batch 256 per worker, CUDA graph, Philox draws).

Arms, alternated `--rounds` times in one process, medians reported:
  train_us[k][mode]   device time of one train() (CUDA events around --updates back-to-back updates), k = 1, 3, 19
  store_us[mode]      store_episode host to host (perf_counter around the call + a device synchronise) at k = 19:
                      'own' stores 19 workers x 2 episodes into 19 buffer sets, 'shared' the 2 episodes of one rank

    python scratch/worker_buffers_bench.py --out profiles/r07_worker_buffers.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip()


def make(k, mode, episodes):
    from tests.ddpg_util import ddpg_kwargs, make_gpu_agent
    kw, dims, ag_ids, g_ids = ddpg_kwargs(4)
    a = make_gpu_agent(kw, dims, ag_ids, g_ids, buffer_episodes=200, seed=0, her_rng='philox', workers_per_rank=k,
                       worker_buffers=mode)
    cp = np.linspace(0.05, 0.3, 4)
    per_call = k if mode == 'own' else 1
    for c in range(40):
        eps = [episodes[(c * per_call + j) % len(episodes)] for j in range(per_call)]
        a.store_episode({key: np.concatenate([e[key] for e in eps]) for key in eps[0]}, cp, 2 * (c + 1))
    return a, cp


def time_train(a, n):
    import torch
    for _ in range(20):
        a.train()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(n):
        a.train()
    t1.record()
    torch.cuda.synchronize()
    return 1e3 * t0.elapsed_time(t1) / n


def time_store(a, k, mode, episodes, cp, n):
    import torch
    per_call = k if mode == 'own' else 1
    out = []
    for c in range(n):
        eps = [episodes[(c * per_call + j) % len(episodes)] for j in range(per_call)]
        batch = {key: np.concatenate([e[key] for e in eps]) for key in eps[0]}
        torch.cuda.synchronize()
        t = time.perf_counter()
        a.store_episode(batch, cp, 100 + c)
        torch.cuda.synchronize()
        out.append(1e6 * (time.perf_counter() - t))
    return float(np.median(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--updates', type=int, default=200)
    ap.add_argument('--stores', type=int, default=30)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('needs a CUDA device')
    from curious_b200 import synth
    from tests.ddpg_util import episode_stream
    dims = synth.arm_dims(4, None)
    episodes = episode_stream(dims, 50, 64, seed=5)
    agents = {(k, m): make(k, m, episodes) for k in (1, 3, 19) for m in ('shared', 'own')}
    train = {(k, m): [] for k, m in agents}
    store = {'shared': [], 'own': []}
    for _ in range(args.rounds):
        for k in (1, 3, 19):
            for m in ('shared', 'own'):
                train[(k, m)].append(time_train(agents[(k, m)][0], args.updates))
        for m in ('shared', 'own'):
            a, cp = agents[(19, m)]
            store[m].append(time_store(a, 19, m, episodes, cp, args.stores))
    rec = dict(gpu=gpu_info(), torch=torch.__version__, workload='Arm4, hidden 256, 3 layers, batch 256 per worker, '
               'CUDA graph, Philox draws; buffers of 200 episodes per module, 40 stores before timing',
               rounds=args.rounds, updates_per_window=args.updates,
               train_us={'k%d' % k: {m: float(np.median(train[(k, m)])) for m in ('shared', 'own')} for k in (1, 3, 19)},
               train_us_all={'k%d_%s' % (k, m): v for (k, m), v in train.items()},
               store_us_k19={m: float(np.median(v)) for m, v in store.items()},
               store_us_k19_all=store)
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(args.out) or '.', exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(json.dumps(rec, indent=1) + '\n')


if __name__ == '__main__':
    main()
