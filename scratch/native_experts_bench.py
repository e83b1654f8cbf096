"""structure='task_experts' with 4 native hidden-64 / 128 experts (DDPG pad_hidden='native'): one TaskExperts.train() round
as the grouped narrow chain (cur_ddpg_chain_grads_group) against the same experts stepped one after the other, each on its
own narrow chain (mode='sequential'), and against today's grouped level kernels at the true width (pad_hidden=False,
cur_ddpg_grads_group).  Device-timed rounds through the CUDA graph (one rank, Adam in the graph) for Arm4 and Arm8 shapes at
1024 / 1152 / 2048 / 4096 / 4864 rows, in ONE process: the arms run alternately, REPS times each, on experts built from
the same seeds; the record keeps every repetition and the median.  1024 rows is below the narrow chain: there the native
experts keep their paths (grouped level kernels / rows schedule), recorded for reference.  After the timing the grouped and
the sequential chain experts have taken the same number of updates from the same seeds, and the record says whether their
parameters are bit-identical.

    python scratch/native_experts_bench.py --out profiles/r05_native_experts.json [--iters 50] [--reps 3]
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

N_EXPERTS = 4
ARMS = {'grouped_chain': ('native', 'grouped'), 'sequential_chain': ('native', 'sequential'),
        'grouped_levels': (False, 'grouped')}


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return dict(nvidia_smi=q.stdout.strip(), torch_name=torch.cuda.get_device_name(0))


def make(n_modules, hidden, rows, pad_hidden, mode):
    from curious_b200.experts import TaskExperts
    kw, dims, ag_ids, g_ids = ddpg_kwargs(n_modules, structure='task_experts', task_replay='replay_current_task_buffer',
                                          batch_size=rows, hidden=hidden)
    cp = np.linspace(0.05, 0.3, n_modules)
    episodes = episode_stream(dims, kw['T'], 10)
    agents = []
    for t in range(N_EXPERTS):
        k = dict(kw)
        k['t_id'] = t
        ag = make_gpu_agent(k, dims, ag_ids, g_ids, her_rng='philox', buffer_episodes=200, seed=10 + t,
                            pad_hidden=pad_hidden)
        np.random.seed(0)
        for i, ep in enumerate(episodes):
            ag.store_episode(ep, cp, 2 * (i + 1))
        agents.append(ag)
    return TaskExperts(agents, mode=mode)


def path_of(te, rows):
    p = te.policies[0]
    if te.mode == 'sequential':
        if p._use_rows(rows):
            return 'sequential_rows'
        return 'sequential_chain_native' if p._use_native_chain(rows) else 'sequential_levels'
    return 'grouped_chain_native' if te._native_chain() else 'grouped_levels'


def time_rounds(te, iters):
    for _ in range(5):
        te.train()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        te.train()
    e1.record()
    torch.cuda.synchronize()
    return 1e3 * e0.elapsed_time(e1) / iters


def save(path, rec):
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, 'w') as f:
        json.dump(rec, f, indent=1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True, help='path of the JSON record')
    ap.add_argument('--iters', type=int, default=50)
    ap.add_argument('--reps', type=int, default=3)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'needs a CUDA device'
    rec = dict(gpu=gpu_info(), experts=N_EXPERTS, iters=args.iters, reps=args.reps,
               unit='us per TaskExperts.train() round of %d experts, CUDA graph, device events' % N_EXPERTS,
               round_us={}, paths={}, grouped_equals_sequential={})
    for hidden in (64, 128):
        for n_modules in (4, 8):
            for rows in (1024, 1152, 2048, 4096, 4864):
                key = 'h%d_arm%d_b%d' % (hidden, n_modules, rows)
                tes = {arm: make(n_modules, hidden, rows, pad, mode) for arm, (pad, mode) in ARMS.items()}
                rec['paths'][key] = {arm: path_of(te, rows) for arm, te in tes.items()}
                times = {arm: [] for arm in tes}
                for _ in range(args.reps):
                    for arm, te in tes.items():
                        times[arm].append(time_rounds(te, args.iters))
                rec['round_us'][key] = dict(reps=times, median={arm: float(np.median(v)) for arm, v in times.items()})
                a, b = tes['grouped_chain'].policies, tes['sequential_chain'].policies
                rec['grouped_equals_sequential'][key] = bool(all(
                    torch.equal(x.theta_main, y.theta_main) and torch.equal(x._adam_v, y._adam_v) for x, y in zip(a, b)))
                print(key, rec['paths'][key], {k: '%.1f' % v for k, v in rec['round_us'][key]['median'].items()},
                      'bit-identical' if rec['grouped_equals_sequential'][key] else 'DIFFERENT', flush=True)
                del tes, a, b
                torch.cuda.empty_cache()
                save(args.out, rec)                   # partial records survive an interrupted run
    rec['gpu_after'] = gpu_info()
    save(args.out, rec)
    print('wrote', args.out)


if __name__ == '__main__':
    main()
