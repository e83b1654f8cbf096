"""structure='task_experts' acting: one evaluator step (TaskExperts.get_actions with the evaluator's arguments: no noise,
compute_Q) as ONE routed launch (cur_ddpg_actions_rows_group) against the per-row loop of one-row get_actions calls it
replaces (rollout.py:211-223).  Host to host per step, each step ending in a device synchronise, for 4 experts on Arm4 and
8 experts on Arm8, n = 2 / 38 / 100 rows spread over the experts at random, hidden 64 (pad_hidden='native') and 256.  The
two arms alternate REPS times in one process on the same experts and inputs; the record keeps every repetition, the
median, whether both arms gave the same bits, and the GPU name and power limit read in the same run.

    python scratch/expert_actions_bench.py --out profiles/r06_expert_actions.json [--iters 200] [--reps 3]
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

from tests.ddpg_util import ddpg_kwargs, make_gpu_agent  # noqa: E402

SHAPES = [(4, 4), (8, 8)]                                    # (experts, modules): Arm4, Arm8
WIDTHS = [(64, 'native'), (256, 'auto')]
ROWS = [2, 38, 100]


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return dict(nvidia_smi=q.stdout.strip(), torch_name=torch.cuda.get_device_name(0))


def make(n_exp, n_modules, hidden, pad):
    from curious_b200.experts import TaskExperts
    kw, dims, ag_ids, g_ids = ddpg_kwargs(n_modules, structure='task_experts', task_replay='replay_current_task_buffer',
                                          hidden=hidden)
    ps = []
    for t in range(n_exp):
        k = dict(kw)
        k['t_id'] = t
        ps.append(make_gpu_agent(k, dims, ag_ids, g_ids, seed=10 + t, pad_hidden=pad))
    return TaskExperts(ps), dims


def step_fn(te, arm, o, ag, g, td):
    which = np.argmax(td, axis=1).astype(np.int32)
    if arm == 'routed':
        return lambda: te.get_actions(o, ag, g, td, compute_Q=True)
    return lambda: te._actions_loop(o, ag, g, td, which, 0., 0., False, True)


def time_steps(fn, iters):
    for _ in range(10):
        fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(iters):
        fn()
        torch.cuda.synchronize()
    return 1e6 * (time.perf_counter() - t0) / iters


def save(path, rec):
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, 'w') as f:
        json.dump(rec, f, indent=1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True, help='path of the JSON record')
    ap.add_argument('--iters', type=int, default=200)
    ap.add_argument('--reps', type=int, default=3)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'needs a CUDA device'
    rec = dict(gpu=gpu_info(), iters=args.iters, reps=args.reps,
               unit='us per evaluator step (TaskExperts.get_actions, compute_Q, no noise), host to host incl. a device '
                    'synchronise', step_us={}, same_bits={})
    for n_exp, n_modules in SHAPES:
        for hidden, pad in WIDTHS:
            te, dims = make(n_exp, n_modules, hidden, pad)
            assert te._routed_ok()
            for n in ROWS:
                key = 'arm%d_%dexperts_h%d_n%d' % (n_modules, n_exp, hidden, n)
                rng = np.random.RandomState(n)
                o = rng.standard_normal((n, dims['o'])).astype(np.float32)
                g = rng.uniform(-1, 1, (n, dims['g'])).astype(np.float32)
                ag = rng.uniform(-1, 1, (n, dims['ag'])).astype(np.float32)
                td = np.eye(n_modules, dtype=np.float32)[rng.randint(0, n_exp, n)]
                fns = {arm: step_fn(te, arm, o, ag, g, td) for arm in ('routed', 'loop')}
                outs = {arm: fn() for arm, fn in fns.items()}
                rec['same_bits'][key] = bool(all(np.array_equal(a, b) for a, b in zip(outs['routed'], outs['loop'])))
                times = {arm: [] for arm in fns}
                for _ in range(args.reps):
                    for arm, fn in fns.items():
                        times[arm].append(time_steps(fn, args.iters))
                rec['step_us'][key] = dict(reps=times, median={arm: float(np.median(v)) for arm, v in times.items()})
                print(key, {k: '%.1f' % v for k, v in rec['step_us'][key]['median'].items()},
                      'same bits' if rec['same_bits'][key] else 'DIFFERENT', flush=True)
                save(args.out, rec)
            del te
            torch.cuda.empty_cache()
    rec['gpu_after'] = gpu_info()
    save(args.out, rec)
    print('wrote', args.out)


if __name__ == '__main__':
    main()
