import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from tests.ddpg_util import ddpg_kwargs, episode_stream, make_gpu_agent, make_oracle_agent, rel_err
from curious_b200 import _lib
from curious_b200.experts import TaskExperts
from tests.test_native_experts_gpu import _fill
for hidden, n_modules, rows, normalize_obs in [(64, 8, 2048, True), (128, 4, 2048, False)]:
    n_exp = 3
    kw, dims, ag_ids, g_ids = ddpg_kwargs(n_modules, structure='task_experts', task_replay='replay_current_task_buffer',
                                          batch_size=rows, hidden=hidden, normalize_obs=normalize_obs)
    cp = np.linspace(0.0, 0.3, n_modules)
    episodes = episode_stream(dims, kw['T'], 12)
    oras, gpus = [], []
    for t in range(n_exp):
        k = dict(kw); k['t_id'] = t
        ora = make_oracle_agent(k, dims, ag_ids, g_ids, seed=20 + t)
        gpu = make_gpu_agent(k, dims, ag_ids, g_ids, her_rng='numpy', seed=20 + t, pad_hidden='native')
        for a in (ora, gpu):
            np.random.seed(17 + t); _fill(a, episodes, cp)
        if normalize_obs:
            for a, b in ((gpu.o_stats, ora.o_stats), (gpu.g_stats, ora.g_stats)):
                a.load_state_list([b.sum, b.sumsq, b.count, b.mean, b.std])
        oras.append(ora); gpus.append(gpu)
    refs, gbs = [], []
    for t, (ora, gpu) in enumerate(zip(oras, gpus)):
        np.random.seed(400 + t); ob = ora.sample_batch()
        np.random.seed(400 + t); gb = gpu.sample_batch()
        refs.append(ora.grads(ob)); gbs.append(gb)
        gpu.grads.zero_(); gpu.stage_batch(gb)
    te = TaskExperts(gpus, use_cuda_graph=False)
    te._grads_group(te._expert_array(False, True), True)
    grp = [(gpu.ref_flat(gpu.grads, 'Q').cpu().numpy().copy(), gpu.ref_flat(gpu.grads, 'pi').cpu().numpy().copy()) for gpu in gpus]
    lib = _lib.load()
    for t, gpu in enumerate(gpus):
        ref = refs[t]
        out = {}
        for name, ch in (('single_chain', -1), ('levels', 0)):
            lib.cur_ddpg_set_chain(ch)
            gpu.grads.zero_(); gpu.stage_batch(gbs[t]); gpu._grads()
            out[name] = (gpu.ref_flat(gpu.grads, 'Q').cpu().numpy().copy(), gpu.ref_flat(gpu.grads, 'pi').cpu().numpy().copy())
        lib.cur_ddpg_set_chain(-1)
        print(hidden, n_modules, rows, 'expert', t, 'margin %.3g' % ref['relu_margin'],
              'grouped==single Q %s pi %s' % (np.array_equal(grp[t][0], out['single_chain'][0]), np.array_equal(grp[t][1], out['single_chain'][1])),
              'err vs oracle Q/pi: grouped %.3g/%.3g single %.3g/%.3g levels %.3g/%.3g' % (
                  rel_err(grp[t][0], ref['Q_grad']), rel_err(grp[t][1], ref['pi_grad']),
                  rel_err(out['single_chain'][0], ref['Q_grad']), rel_err(out['single_chain'][1], ref['pi_grad']),
                  rel_err(out['levels'][0], ref['Q_grad']), rel_err(out['levels'][1], ref['pi_grad'])),
              'chain vs levels pi %.3g' % rel_err(out['single_chain'][1], out['levels'][1]), flush=True)
