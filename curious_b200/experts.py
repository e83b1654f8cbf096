"""structure='task_experts' as one grouped update - the B200 form of the reference's per-module experts.

The reference builds one DDPG per module over shared per-module buffers (train.py:287-289, ddpg.py:302-318) and
trains ONE of them per epoch (`policy[i_policy].train()`, train.py:108-113).  On a B200 a batch-256 update of one
expert leaves the GPU mostly idle (every GEMM level is latency-bound), so `TaskExperts.train()` steps ALL experts
in one sequence of grouped launches: every dependency level of the DDPG graph is one launch over the problems of all
experts (csrc/ddpg.cu cur_ddpg_grads_group; FFMA grouped GEMM at batch 256, the tcgen05 batch at batch >= 1024).
Experts built with pad_hidden='native' at hidden 64 / 128 that train on the narrow chain (from 1152 rows) run
cur_ddpg_chain_grads_group instead: their chain kernels side by side, their K-sliced weight gradients in shared launches.
Semantically it is `for p in policies: p.train()` - every expert keeps its own parameters, Adam state, Philox
stream, LP apportioning and buffers, and the result is bit-identical to stepping them one after the other on the
levels schedule, or on the narrow chain for native experts.

Acting (`get_actions`, the evaluation step of the experts, rollout.py:211-223) routes each row to the expert of its
module in ONE launch (cur_ddpg_actions_rows_group): bit for bit the loop of one-row get_actions calls it stands for,
np.random stream and device-noise counters included.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from .parallel import allreduce_sum_, world as _world
from .util import LazyHost, capture_graph


class TaskExperts(object):
    def __init__(self, policies, use_cuda_graph=True, mode='auto'):
        """mode: 'grouped' = grouped launches; 'sequential' = p.train() one after the other; 'auto' = sequential
        when every expert runs the rows schedule at batch <= 512 (one expert's row CTAs already fill the 148 SMs;
        measured per round of 4 experts: batch 256 237 us vs 322 us grouped, 512 435 vs 524, 1024 841 vs 372),
        grouped otherwise.  Native hidden-64 / 128 experts on the narrow chain give the same bits either way and grouped
        is faster at every measured shape (one B200, 1000 W, profiles/r05_native_experts.json, 4 experts, Arm4, us per
        round grouped vs sequential: hidden 64 1152 rows 191 vs 344, 4864 rows 460 vs 529; hidden 128 233 vs 429 and
        589 vs 694; Arm8 alike), so they run grouped."""
        assert len(policies) >= 1 and mode in ('auto', 'grouped', 'sequential')
        self.mode = mode
        p0 = policies[0]
        for p in policies:
            assert bytes(p.net.desc) == bytes(p0.net.desc), 'experts must share the network shape'
            assert p.batch_size == p0.batch_size and p.device == p0.device
        self.policies = list(policies)
        self.use_cuda_graph = use_cuda_graph
        self._graph = None
        self._experts = None

    @staticmethod
    def router(policies):
        """A TaskExperts over `policies` when they are DDPG agents of one network shape on one device (their evaluation
        step can then be one routed launch); None for any other list."""
        from .ddpg import DDPG
        if isinstance(policies, TaskExperts):
            return policies
        if not isinstance(policies, (list, tuple)):
            return None
        ps = list(policies)
        if not ps or len(ps) > _lib.CUR_MAX_TASKS or not all(isinstance(p, DDPG) for p in ps):
            return None
        p0 = ps[0]
        if not all(bytes(p.net.desc) == bytes(p0.net.desc) and p.batch_size == p0.batch_size and p.device == p0.device
                   for p in ps):
            return None
        return TaskExperts(ps)

    def __len__(self):
        return len(self.policies)

    def __getitem__(self, i):
        return self.policies[i]

    # ------------------------------------------------------------------------------------------
    def _native_chain(self):
        """Every expert is a native hidden-64 / 128 net that trains on the narrow chain at its batch size
        (DDPG._use_native_chain): the round runs as cur_ddpg_chain_grads_group, bit for bit what each expert's own
        cur_ddpg_chain_grads gives."""
        return all(p._use_native_chain(p.batch_size) for p in self.policies)

    def _grads_group(self, arr, chain):
        lib = _lib.load()
        fn, name = ((lib.cur_ddpg_chain_grads_group, 'cur_ddpg_chain_grads_group') if chain else
                    (lib.cur_ddpg_grads_group, 'cur_ddpg_grads_group'))
        _lib.check(fn(_lib.stream_ptr(), C.byref(self.policies[0].net.desc), len(arr), arr), name)

    def _expert_array(self, graph, chain):
        arr = (_lib.DdpgExpert * len(self.policies))()
        for e, p in zip(arr, self.policies):
            n = p.batch_size
            b = p._gbatch if graph else p._batch
            g2 = b['g_2'] if (not graph or p.relative_goals) else b['g']
            e.theta_main = p.theta_main.data_ptr()
            e.theta_target = p.theta_target.data_ptr()
            e.stats = p._stats
            e.has_stats = 1
            e.batch = _lib.Batch(b['o'].data_ptr(), b['g'].data_ptr(), b['u'].data_ptr(),
                                 b['td'].data_ptr() if p.modular else None, b['o_2'].data_ptr(), g2.data_ptr(),
                                 b['r'].data_ptr(), n)
            e.hyper = p._ghyper if graph else p._hyper
            e.workspace = (p._workspace_chain(n) if chain else p._workspace(n)).data_ptr()
            e.grads = p.grads.data_ptr()
            if graph:
                e.q_loss, e.pi_loss, e.q_pi = p._q_ring.data_ptr(), p._pi_ring.data_ptr(), p._q_pi.data_ptr()
            else:
                p._q_pi_eager = torch.empty((n, 1), dtype=torch.float32, device=p.device)
                e.q_loss, e.pi_loss, e.q_pi = p._q_loss.data_ptr(), p._pi_loss.data_ptr(), p._q_pi_eager.data_ptr()
        return arr

    def _launch(self, graph):
        """HER sample per expert, grouped gradients, then (single rank) Adam per expert."""
        for p in self.policies:
            if graph:
                segs = [(buf.device_view(), 0, ttr) for buf, ttr in p._all_segments()]
                p.sample_transitions.sample_device(segs, p.batch_size, clip_obs=p.clip_obs,
                                                   relative_goals=p.relative_goals, want=p._gwant, out=p._gbatch,
                                                   dyn=p._dyn_dev.data_ptr(), call_offset=p.GRAPH_STREAM_OFFSET)
            else:
                p.stage_batch()
        chain = self._native_chain()
        arr = self._expert_array(graph, chain)
        self._keep = arr
        self._grads_group(arr, chain)

    def _build_graph(self):
        chain = self._native_chain()
        for p in self.policies:
            p.grad_exchange = 'nccl'          # several ranks: NCCL all-reduce + Adam after the graph
            p._prepare_graph_state()
            (p._workspace_chain if chain else p._workspace)(p.batch_size)
        dev = self.policies[0].device
        torch.cuda.current_stream().synchronize()
        states = [(p.theta_main.clone(), p._adam_m.clone(), p._adam_v.clone(), p._step.clone()) for p in self.policies]
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):                       # warm-up outside capture
            self._launch(True)
            for p in self.policies:
                p._launch_adam()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize(dev)
        for p, st in zip(self.policies, states):
            p.theta_main.copy_(st[0])
            for dst, src in zip((p._adam_m, p._adam_v, p._step), st[1:]):
                dst.copy_(src)
        self._single_rank = _world(self.policies[0].comm)[1] == 1
        g = torch.cuda.CUDAGraph()
        with capture_graph(g):
            self._launch(True)
            if self._single_rank:
                for p in self.policies:
                    p._launch_adam()
        self._graph = g

    def train(self, stage=True):
        """One update of every expert.  Returns [(critic_loss, actor_loss), ...] like DDPG.train (ddpg.py:368-373)."""
        ps = self.policies
        if self.mode == 'sequential' or (self.mode == 'auto' and all(
                p.update_schedule != 'levels' and p.batch_size <= 512 and p._use_rows(p.batch_size) for p in ps)):
            return [p.train(stage) for p in ps]
        graph = stage and self.use_cuda_graph and all(p.her_rng == 'philox' for p in ps)
        if graph:
            if self._graph is None:
                self._build_graph()
            for p in ps:
                if p.Q_adam.t % 100 == 0:
                    p.Q_adam.check_synced()
                    p.pi_adam.check_synced()
                p._refresh_dyn()
            slots = [p._n_updates % p.LOSS_RING for p in ps]
            self._graph.replay()
            if not self._single_rank:
                for p in ps:
                    allreduce_sum_(p.grads, p.comm)          # SUM, not mean (ddpg.py:452-453)
                    p._launch_adam()
            out = []
            for p, slot in zip(ps, slots):
                p._n_updates += 1
                p.Q_adam.t += 1
                p.pi_adam.t += 1
                out.append((LazyHost(p._q_ring[slot]), LazyHost(p._q_pi)))
            return out
        if stage:
            self._launch(False)
        else:
            chain = self._native_chain()
            arr = self._expert_array(False, chain)
            self._keep = arr
            self._grads_group(arr, chain)
        out = []
        for p in ps:
            p._update(p._view(p.grads, 'Q'), p._view(p.grads, 'pi'))
            p._step += 1
            p._n_updates += 1
            out.append((LazyHost(p._q_loss.clone().reshape(())), LazyHost(p._q_pi_eager)))
        return out

    def update_target_net(self):
        for p in self.policies:
            p.update_target_net()

    # ------------------------------------------------------------------------------------------ acting
    def _routed_ok(self):
        """Every expert would take the one-launch action path, and the options the launch shares agree."""
        ps = self.policies
        p0 = ps[0]
        return len(ps) <= _lib.CUR_MAX_TASKS and all(
            p._action_rows_ok() and (p.clip_obs, p.relative_goals, p.modular, p.action_noise) ==
            (p0.clip_obs, p0.relative_goals, p0.modular, p0.action_noise) for p in ps)

    def get_actions(self, o, ag, g, task_descr, noise_eps=0., random_eps=0., use_target_net=False, compute_Q=False):
        """Each row acted on by policies[argmax(task_descr[row])] (rollout.py:211-223).  Returns u float64 [n, dimu], and
        with compute_Q [u, q float64 [n, 1]]: exactly what a loop of one-row get_actions calls builds, including the
        np.random draws (per row: randn, binomial, uniform) and every expert's device-noise counter.  Up to
        ACTION_ROWS_MAX rows of experts on the one-launch path: ONE routed launch (cur_ddpg_actions_rows_group);
        otherwise that loop."""
        p0 = self.policies[0]
        o = np.asarray(o, np.float32).reshape(-1, p0.dimo)
        n = o.shape[0]
        g = np.asarray(g, np.float32).reshape(n, p0.dimg)
        td = np.asarray(task_descr, np.float32).reshape(n, -1)
        which = np.argmax(td, axis=1).astype(np.int32)
        if n > p0.ACTION_ROWS_MAX or not self._routed_ok():
            return self._actions_loop(o, ag, g, td, which, noise_eps, random_eps, use_target_net, compute_Q)
        device_noise = p0.action_noise == 'device'
        route = _Route(self.policies, which, use_target_net)
        res, finished = p0._actions_one_launch(o, ag, g, td, n, None, compute_Q, device_noise, noise_eps, random_eps,
                                               route=route)
        if device_noise:                                   # one call per row in the loop
            for p, c in zip(self.policies, np.bincount(which, minlength=len(self.policies))):
                p._action_calls += int(c)
        if not finished:
            res = p0._finish_actions(res, n, compute_Q, device_noise, noise_eps, random_eps, draw=route.draw)
        u = np.asarray(res[0] if compute_Q else res, np.float64).reshape(n, p0.dimu)
        return [u, np.asarray(res[1], np.float64).reshape(n, 1)] if compute_Q else u

    def _actions_loop(self, o, ag, g, td, which, noise_eps, random_eps, use_target_net, compute_Q):
        """One get_actions call per row, by the row's expert (rollout.py:211-223)."""
        n = len(o)
        u = np.zeros((n, self.policies[0].dimu))
        q = np.zeros((n, 1))
        for i in range(n):
            out = self.policies[which[i]].get_actions(
                o[i:i + 1], None if ag is None else ag[i:i + 1], g[i:i + 1], task_descr=td[i:i + 1], noise_eps=noise_eps,
                random_eps=random_eps, use_target_net=use_target_net, compute_Q=compute_Q)
            if compute_Q:
                u[i], q[i, 0] = out[0], np.asarray(out[1]).reshape(-1)[0]
            else:
                u[i] = out
        return [u, q] if compute_Q else u


class _Route(object):
    """One routed action launch as DDPG._actions_one_launch asks for it: the launch (cur_ddpg_actions_rows_group), the
    device-side noise pass and the host draws, each as the loop of one-row calls would have made them."""

    def __init__(self, policies, which, use_target_net):
        self.policies, self.which = policies, which
        self.arr = (_lib.ActionsExpert * len(policies))()
        for e, p in zip(self.arr, policies):
            e.theta = (p.theta_target if use_target_net else p.theta_main).data_ptr()
            e.stats = p._stats

    def launch(self, o, ag, g, td, n, clip_obs, out_pi, out_q, seq):
        ps = self.policies
        _lib.check(_lib.load().cur_ddpg_actions_rows_group(
            _lib.stream_ptr(), C.byref(ps[0].net.desc), len(ps), self.arr, self.which.ctypes.data, o, ag, g, td, n,
            clip_obs, out_pi, out_q, seq), 'cur_ddpg_actions_rows_group')

    def noise(self, out, n, noise_eps, random_eps):
        """Row i is the k-th one-row call of its expert in this step: Philox key = the expert's noise_seed, call number =
        its _action_calls + k (cur_action_noise_rows)."""
        ps = self.policies
        keys = np.empty((2, n), np.uint64)
        taken = [0] * len(ps)
        for i, e in enumerate(self.which):
            p = ps[e]
            keys[0, i] = int(p.noise_seed) & (2 ** 64 - 1)
            keys[1, i] = p._action_calls + taken[e]
            taken[e] += 1
        dev = torch.from_numpy(keys.view(np.int64)).to(ps[0].device)
        p0 = ps[0]
        _lib.check(_lib.load().cur_action_noise_rows(_lib.stream_ptr(), out, n, p0.dimu, float(p0.max_u), float(noise_eps),
                                                     float(random_eps), dev[0].data_ptr(), dev[1].data_ptr()),
                   'cur_action_noise_rows')

    def draw(self, n, random_eps):
        """The host draws of the loop: per row, the row's expert's _draw_action_noise(1, random_eps)."""
        rows = [self.policies[e]._draw_action_noise(1, random_eps) for e in self.which]
        return tuple(np.concatenate([r[k] for r in rows]) for k in range(3))
