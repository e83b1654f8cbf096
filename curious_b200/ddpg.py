"""DDPG + HER agent on one B200 per rank - drop-in for reference baselines/her/ddpg.py:18-537.

Same constructor arguments, same methods (get_actions / store_episode / sample_batch / stage_batch /
train / update_target_net / get_current_buffer_size / clear_buffer / logs / save_weights / load_weights /
pickling).  What moved to the device:
  sample_batch      one fused kernel over all LP-apportioned module buffers     (csrc/her.cu)
  _grads            grouped-GEMM forward/backward into a flat gradient          (csrc/ddpg.cu)
  _update           NCCL all-reduce(SUM) + fused Adam on the flat arena         (csrc/norm_adam.cu)
  update_target_net fused polyak on the flat arena
  o_stats/g_stats   device normalisers, one packed all-reduce per store_episode
Host keeps: the LP apportioning arithmetic (<= 9 integers, ddpg.py:255-286), buffer slot choice and
the exploration noise of get_actions - they consume the caller's np.random stream in reference order.

Extra keyword arguments (all optional): device, comm (torch.distributed group; default WORLD when
initialised), her_rng ('philox' default | 'numpy' = replay the reference's np.random draws),
action_noise ('host' default | 'device': exploration noise of get_actions from counter-based draws on the device),
seed (Xavier init seed; the reference uses TF's graph seed), workers_per_rank / workers_mode / worker_buffers
('shared' default | 'own': every hosted worker with its own buffers and random streams, DESIGN.md section 7).
"""
import ctypes as C
import pickle
from collections import OrderedDict

import numpy as np
import torch

from . import _lib, apportion
from .her import DeviceEpisodes, HostDraws
from .mpi_adam import MpiAdam, adam_step_scale
from .normalizer import Normalizer, recompute_stats_packed
from .parallel import allreduce_sum_, world as _world
from .replay_buffer import StagedEpisodes, episodes_to_device
from .util import LazyHost, capture_graph, dims_to_shapes, import_function, store_args, transitions_in_episode_batch


_ADAM_TABLES = {}


def _adam_table(lr, beta1, beta2, n):
    """float32(-a_t) for t = 1..n with a_t evaluated exactly like MpiAdam.update does it on the host
    (python float pow, mpi_adam.py:31), so the graph path and the eager path step identically."""
    key = (float(lr), float(beta1), float(beta2), int(n))
    if key not in _ADAM_TABLES:
        _ADAM_TABLES[key] = np.array([np.float32(-adam_step_scale(lr, beta1, beta2, t)) for t in range(1, n + 1)],
                                     np.float32)
    return _ADAM_TABLES[key]


class DDPG(object):
    @store_args
    def __init__(self, input_dims, hidden, layers, network_class, polyak, batch_size,
                 Q_lr, pi_lr, norm_eps, norm_clip, max_u, action_l2, clip_obs, scope, T,
                 rollout_batch_size, subtract_goals, relative_goals, clip_pos_returns, clip_return,
                 normalize_obs, sample_transitions, gamma, buffers=None, reuse=False, tasks_ag_id=None,
                 tasks_g_id=None, task_replay='', t_id=None, eps_task=None, **kwargs):
        """See reference ddpg.py:25-60 for the meaning of every argument."""
        if self.clip_return is None:
            self.clip_return = np.inf
        self.structure = kwargs.get('structure', getattr(self, 'structure', 'curious'))
        self.device = kwargs.get('device') or torch.device('cuda', torch.cuda.current_device())
        self.comm = kwargs.get('comm')
        self.her_rng = kwargs.get('her_rng', 'philox')
        self.seed = kwargs.get('seed', 0)
        # key of the device-side exploration noise (action_noise='device'); per rank in make_experiment, like the
        # reference's rank_seed (train.py:242), while `seed` (weight init) is the same on every rank
        self.noise_seed = kwargs.get('noise_seed', self.seed)
        self.use_cuda_graph = kwargs.get('use_cuda_graph', True)
        # 'rows' (cluster kernel + fused dW/Adam, 2 launches), 'levels' (one grouped GEMM per dependency
        # level) or 'auto' (rows whenever the shape is supported)
        self.update_schedule = kwargs.get('update_schedule', 'auto')
        self.fuse_her = kwargs.get('fuse_her', True)      # rows schedule: sample inside the update kernel
        # hidden widths below 256 (config.py:25 is a user parameter), four values:
        #   'auto'    run zero-padded to 256 on the hand-written row / chain / action kernels whenever they take the padded
        #             shape (actor_critic._NetSpec; same results, 59 instead of 140 us per batch-256 update)
        #   True      always zero-padded to 256
        #   False     never: dependency-level kernels at the true width
        #   'native'  hidden 64 / 128 at the true width on the row kernels (train() up to 1024 rows, with the CUDA graph,
        #             fused HER and fused Adam / the tile exchange), on the tcgen05 chain kernel above (a multiple of 128
        #             rows, cur_ddpg_chain_grads; weight gradients on K-sliced FFMA GEMMs, all-reduce + Adam after the graph
        #             with several ranks, workers_per_rank > 1 as one wide batch) and on the one-launch action kernel
        #             (get_actions up to 512 rows, compute_Q included).  Batches neither takes run the dependency-level
        #             kernels at the true width, like False.  Hidden 256 runs as always; any other width raises ValueError.
        self.pad_hidden = kwargs.get('pad_hidden', 'auto')
        if self.pad_hidden == 'native' and self.hidden not in self.NATIVE_HIDDEN:
            raise ValueError("pad_hidden='native' needs hidden in %s, not %r" % (self.NATIVE_HIDDEN, self.hidden))
        # several ranks: 'tile' = the gradient tiles are exchanged over NVLink peer memory INSIDE the weight-gradient
        # launch, Adam and W^T stay in its epilogue (csrc/ddpg_rows.cu, parallel.TileGradExchange: 2 launches per update
        # like one rank), 'p2p' = one exchange + Adam kernel after the weight-gradient launch (csrc/p2p.cu: every rank
        # sums all peers' gradients in rank order), 'p2p_sharded' = reduce-scatter by loads, Adam on the own slice,
        # all-gather by stores, 'nccl' = NCCL all-reduce + Adam launch after the graph, 'auto' = tile when the rows
        # schedule runs on an NCCL (one GPU per rank) group
        self.grad_exchange = kwargs.get('grad_exchange', 'auto')
        # mode of the in-launch tile exchange: 'auto' (0 for two ranks, 1 above), 0, 1, or 2 / 'nvls' (NVSwitch multicast:
        # multimem.ld_reduce does the sum; parallel.TileGradExchange)
        self.xchg_mode = kwargs.get('xchg_mode', 'auto')
        assert self.grad_exchange in ('auto', 'tile', 'p2p', 'p2p_sharded', 'nccl')
        self.xchg_timeline_tiles = int(kwargs.get('xchg_timeline_tiles', 0))      # debug: per-tile %globaltimer stamps
        # reference workers hosted by this rank (SURVEY 8e: the 19 MPI workers become ceil(19 / G) workers per GPU):
        # every update is the SUM of `workers_per_rank` batch-256 gradients, each with its own loss mean, exactly what
        # the reference's SUM all-reduce over that many single-batch workers produces (ddpg.py:452-453)
        self.workers_per_rank = int(kwargs.get('workers_per_rank', 1))
        assert self.workers_per_rank >= 1
        # 'wide' = the workers' batches as one batch with 1 / batch_size loss seeds, 'micro' = one accumulating launch
        # pair per worker (same Philox stream positions as the launch-by-launch path), 'auto' = wide when a schedule
        # takes workers x batch_size rows
        self.workers_mode = kwargs.get('workers_mode', 'auto')
        assert self.workers_mode in ('auto', 'wide', 'micro')
        # 'shared' = the k workers of a rank sample their batches from the rank's one buffer set; 'own' = every worker j has
        # its own buffers, np.random stream and Philox key (reference rank r * k + j, train.py:221-243; workers.py), its
        # own episodes in store_episode and its own share of the normaliser batch - one rank only, learner only
        self.worker_buffers = kwargs.get('worker_buffers', 'shared')
        if self.worker_buffers not in ('shared', 'own'):
            raise ValueError("worker_buffers must be 'shared' or 'own', not %r" % (self.worker_buffers,))
        # exploration noise of get_actions (ddpg.py:147-152): 'host' = the caller's np.random stream in reference order,
        # 'device' = counter-based draws applied on the device before the one D2H copy (SURVEY 8f row 1)
        # train() on the CUDA-graph path returns views of fixed device buffers (no copy per update); True = owned copies
        self.own_train_outputs = bool(kwargs.get('own_train_outputs', False))
        self.action_noise = kwargs.get('action_noise', 'host')
        assert self.action_noise in ('host', 'device')
        self._action_calls = 0
        self.action_path = kwargs.get('action_path', 'auto')   # 'levels': always the multi-launch forward
        self._action_rows = None
        self._action_slots = {}
        self.create_actor_critic = import_function(self.network_class)

        self.dimo = self.input_dims['o']
        self.dimg = self.input_dims['g']
        self.dimag = self.input_dims['ag']
        self.dimu = self.input_dims['u']
        self.modular = self.structure in ('curious', 'task_experts')
        if self.modular:
            self.dimtd = self.input_dims['task_descr']
        else:
            self.dimtd = 0

        # staged batch layout (ddpg.py:73-83)
        input_shapes = dims_to_shapes(self.input_dims)
        stage_shapes = OrderedDict()
        for key in sorted(self.input_dims.keys()):
            if key.startswith('info_'):
                continue
            stage_shapes[key] = (None, *input_shapes[key])
        for key in ['o', 'g']:
            stage_shapes[key + '_2'] = stage_shapes[key]
        stage_shapes['r'] = (None, 1)
        self.stage_shapes = stage_shapes

        if t_id is not None:
            self.scope += str(t_id)

        if self.modular:
            self.nb_tasks = len(tasks_g_id)
        if buffers is not None:
            self.buffer = buffers
            if type(self.buffer) is list and len(self.buffer) > 5:
                for i in range(6, len(self.buffer)):        # distractor buffers are one buffer (ddpg.py:104-110)
                    self.buffer[i] = self.buffer[5]
        self._create_network(reuse=reuse)
        if self.worker_buffers == 'own':
            self._init_own_workers()
        self.first = True
        self.cp = None
        self._staged = None

    # ------------------------------------------------------------------------------------------
    def _create_network(self, reuse=False):
        dev = self.device
        mk = lambda kh: self.create_actor_critic(dimo=self.dimo, dimg=self.dimg, dimu=self.dimu, dimtd=self.dimtd,
                                                 max_u=self.max_u, hidden=self.hidden, layers=self.layers,
                                                 normalize_obs=self.normalize_obs, norm_clip=self.norm_clip,
                                                 kernel_hidden=kh)
        self.net = mk(None)
        if (self.pad_hidden and self.pad_hidden != 'native' and self.hidden < self.KERNEL_HIDDEN and
                self.update_schedule != 'levels'):
            wide = mk(self.KERNEL_HIDDEN)
            rows = self.batch_size * max(1, int(getattr(self, 'workers_per_rank', 1)))
            if self.pad_hidden is True or _lib.load().cur_ddpg_rows_supported(C.byref(wide.desc), min(rows, 256)):
                self.net = wide
        if self.net.modular != self.modular:
            raise ValueError('network_class %s does not fit structure %r' % (self.network_class, self.structure))
        net = self.net
        self._ref_idx = None
        if net.padded:
            self._ref_idx = {w: torch.from_numpy(net.ref_index(w)).to(dev) for w in ('Q', 'pi')}
        # running averages (ddpg.py:402-409)
        # both normalisers accumulate into ONE packed buffer [sum_o|sumsq_o|count_o|sum_g|sumsq_g|count_g]: one collective
        # per store_episode (normalizer.recompute_stats_packed)
        no, ng = 2 * self.dimo + 1, 2 * self.dimg + 1
        self._stats_partial = torch.zeros(no + ng, dtype=torch.float32, device=dev)
        self.o_stats = Normalizer(self.dimo, self.norm_eps, self.norm_clip, device=dev, comm=self.comm,
                                  partial=self._stats_partial[:no])
        self.g_stats = Normalizer(self.dimg, self.norm_eps, self.norm_clip, device=dev, comm=self.comm,
                                  partial=self._stats_partial[no:])
        self._stats = _lib.NormStats(self.o_stats.mean.data_ptr(), self.o_stats.std.data_ptr(),
                                     self.g_stats.mean.data_ptr(), self.g_stats.std.data_ptr())
        # flat arenas: [Q | pad | pi | pad]
        self.theta_main = torch.zeros(net.arena, dtype=torch.float32, device=dev)
        self.theta_target = torch.zeros(net.arena, dtype=torch.float32, device=dev)
        self.grads = torch.zeros(net.arena, dtype=torch.float32, device=dev)
        self._init_weights()
        # optimisers (ddpg.py:451-453): separate Adam state and step counters for Q and pi
        self._adam_m = torch.zeros(net.arena, dtype=torch.float32, device=dev)
        self._adam_v = torch.zeros(net.arena, dtype=torch.float32, device=dev)
        self.Q_adam = MpiAdam([self._view(self.theta_main, 'Q')], scale_grad_by_procs=False, comm=self.comm,
                              m=self._view(self._adam_m, 'Q'), v=self._view(self._adam_v, 'Q'))
        self.pi_adam = MpiAdam([self._view(self.theta_main, 'pi')], scale_grad_by_procs=False, comm=self.comm,
                               m=self._view(self._adam_m, 'pi'), v=self._view(self._adam_v, 'pi'))
        self.Q_adam.on_change = self.pi_adam.on_change = self._mark_weights_changed
        self._hyper = _lib.DdpgHyper(float(self.gamma), float(min(self.clip_return, 3.0e38)), float(self.action_l2),
                                     1 if self.clip_pos_returns else 0)
        self._ws = {}
        self._sync_optimizers()
        self._init_target_net()
        self._q_loss = torch.zeros(1, dtype=torch.float32, device=dev)
        self._pi_loss = torch.zeros(1, dtype=torch.float32, device=dev)
        self._batch = None
        # shared device train-step counter (Philox counter of the HER kernel, Adam's t, loss ring slot)
        self._step = torch.zeros(1, dtype=torch.int64, device=dev)
        self._n_updates = 0
        self._graph = None
        self._graph_sig = None
        self._graph_fused = False
        self._wT_dirty = True

    def _init_own_workers(self):
        """worker_buffers='own': worker 0 keeps the buffers the caller passed, workers 1.. get buffers of the same shapes
        and sizes (buffers 6.. aliasing 5 like the caller's, ddpg.py:104-110)."""
        if _world(self.comm)[1] > 1:
            raise ValueError("worker_buffers='own' runs on one rank")
        if self.structure == 'task_experts':
            raise ValueError("worker_buffers='own' does not take structure='task_experts'")
        if self.workers_mode == 'micro':
            raise ValueError("worker_buffers='own' runs the workers as one wide batch, not workers_mode='micro'")
        if getattr(self, 'buffer', None) is None:
            raise ValueError("worker_buffers='own' needs the buffers")
        from .replay_buffer import ReplayBuffer
        from .workers import WorkerStreams
        k = self.workers_per_rank
        new = lambda b: ReplayBuffer(b.buffer_shapes, b.size * b.T, b.T, b.sample_transitions, device=b.device)
        self._worker_buffers = [self.buffer]
        for _ in range(1, k):
            if isinstance(self.buffer, list):
                bufs = []
                for i, b in enumerate(self.buffer):
                    bufs.append(bufs[5] if i > 5 else new(b))
            else:
                bufs = new(self.buffer)
            self._worker_buffers.append(bufs)
        self.worker_streams = WorkerStreams(self.seed, k)
        self._hyper.loss_rows = self.batch_size        # each worker's loss is a mean over its own batch

    def worker_buffer_set(self, j):
        """Worker j's buffers (worker_buffers='own'): a list like `buffers`, or one ReplayBuffer."""
        return self._worker_buffers[j]

    def _own(self):
        return self.worker_buffers == 'own'

    def _mark_weights_changed(self):
        """theta_main was written outside the fused update: W^T kept by the rows graph must be rebuilt (_refresh_wT)."""
        self._wT_dirty = True

    def _view(self, arena, which):
        net = self.net
        return arena[:net.n_Q] if which == 'Q' else arena[net.pi_offset:net.pi_offset + net.n_pi]

    def _init_weights(self):
        """tf.contrib.layers.xavier_initializer() (uniform) kernels, zero biases (util.py:63), drawn on the
        host in flat order main/Q then main/pi and uploaded."""
        rng = np.random.RandomState(self.seed)
        for which in ('Q', 'pi'):
            chunks = []
            for s in self.net.var_shapes(which):
                if len(s) == 2:
                    lim = np.sqrt(6.0 / (s[0] + s[1]))
                    chunks.append(rng.uniform(-lim, lim, s).astype(np.float32).reshape(-1))
                else:
                    chunks.append(np.zeros(s, np.float32))
            self.set_flat(which, np.concatenate(chunks))

    KERNEL_HIDDEN = 256        # width of the hand-written row / chain / action kernels
    NATIVE_HIDDEN = (64, 128, 256)   # widths the row / action kernels are instantiated for (pad_hidden='native')

    def ref_flat(self, arena, which):
        """The `which` net of an arena-shaped tensor (parameters, gradients, Adam moments) as a device vector in the
        reference's GetFlat order - a view, or a gather when the net runs zero-padded."""
        v = self._view(arena, which)
        return v if self._ref_idx is None else v[self._ref_idx[which]]

    # flat parameter access in GetFlat order (tf_util.py:221-244)
    def get_flat(self, which, target=False):
        return self.ref_flat(self.theta_target if target else self.theta_main, which).detach().cpu().numpy().copy()

    def set_flat(self, which, values, target=False):
        v = torch.from_numpy(np.ascontiguousarray(values, dtype=np.float32)).to(self.device)
        dst = self._view(self.theta_target if target else self.theta_main, which)
        if self._ref_idx is None:
            dst.copy_(v)
        else:
            dst.zero_()                                   # the padding stays exactly zero
            dst[self._ref_idx[which]] = v
        self._wT_dirty = True

    def _workspace(self, n):
        if n not in self._ws:
            floats = _lib.load().cur_ddpg_workspace_floats(C.byref(self.net.desc), n)
            self._ws[n] = torch.zeros(floats, dtype=torch.float32, device=self.device)     # holds a ticket: zeroed
        return self._ws[n]

    def _rows_shape_ok(self, n):
        """cur_ddpg_rows_supported for this agent's net and n rows.  The library also takes hidden 64 / 128; an agent
        runs a net of any width but 256 on the row / action kernels only when it was built with pad_hidden='native'."""
        if int(self.net.desc.hidden) != self.KERNEL_HIDDEN and self.pad_hidden != 'native':
            return False
        return bool(_lib.load().cur_ddpg_rows_supported(C.byref(self.net.desc), n))

    def _use_rows(self, n):
        if self.update_schedule == 'levels':
            return False
        lib = _lib.load()
        ok = self._rows_shape_ok(n)
        if self.update_schedule == 'rows':
            if not ok:
                raise ValueError('update_schedule="rows" does not support this network / batch shape')
            return True
        # auto: from 1024 rows the fused tcgen05 chain kernel (csrc/tc_chain.cu) is faster than re-streaming the weights per
        # 4 rows (measured us / update, rows vs chain: 512 110 / 165, 768 160 / 166, 1024 208 / 166)
        if ok and n >= self.CHAIN_MIN_ROWS and lib.cur_ddpg_uses_chain(C.byref(self.net.desc), n):
            return False
        return ok

    def _use_native_chain(self, n):
        """A 'native' net narrower than 256 runs a batch of NATIVE_CHAIN_MIN_ROWS rows or more that the rows schedule does
        not take on the chain kernel at its own width (cur_ddpg_chain_grads) when the library takes the shape - under
        update_schedule 'auto' and 'levels' alike, as a hidden-256 net reaches the chain through cur_ddpg_grads from 1024
        rows.  Smaller batches keep the paths they had: rows, or the level kernels at the true width."""
        if (self.pad_hidden != 'native' or int(self.net.desc.hidden) >= self.KERNEL_HIDDEN or
                n < self.NATIVE_CHAIN_MIN_ROWS or self._use_rows(n)):
            return False
        return bool(_lib.load().cur_ddpg_chain_supported(C.byref(self.net.desc), n))

    def _workspace_chain(self, n):
        key = ('chain', n)
        if key not in self._ws:
            floats = _lib.load().cur_ddpg_chain_workspace_floats(C.byref(self.net.desc), n)
            self._ws[key] = torch.zeros(floats, dtype=torch.float32, device=self.device)
        return self._ws[key]

    def _workspace_rows(self, n):
        key = ('rows', n)
        if key not in self._ws:
            floats = _lib.load().cur_ddpg_rows_workspace_floats(C.byref(self.net.desc), n)
            self._ws[key] = torch.zeros(floats, dtype=torch.float32, device=self.device)   # holds a ticket: zeroed
        return self._ws[key]

    # ------------------------------------------------------------------------------------------
    def _random_action(self, n):
        return np.random.uniform(low=-self.max_u, high=self.max_u, size=(n, self.dimu))

    def _preprocess_og(self, o, ag, g):
        """Host version kept for API parity (ddpg.py:118-127); the device paths fuse it into their kernels."""
        if self.relative_goals:
            g_shape = g.shape
            g = g.reshape(-1, self.dimg)
            ag = ag.reshape(-1, self.dimag)
            g = self.subtract_goals(g, ag)
            g = g.reshape(*g_shape)
        o = np.clip(o, -self.clip_obs, self.clip_obs)
        g = np.clip(g, -self.clip_obs, self.clip_obs)
        return o, g

    def _action_slot(self, n):
        """Persistent mapped pinned buffers of the one-launch action path for n rows: the inputs, and the outputs as
        8-byte words {float32 | call number} (cur_ddpg_actions_rows)."""
        slot = self._action_slots.get(n)
        if slot is None:
            lib = _lib.load()
            sizes = [('o', n * self.dimo), ('g', n * self.dimg)]
            if self.relative_goals:
                sizes.append(('ag', n * self.dimag))
            if self.modular:
                sizes.append(('td', n * self.dimtd))
            sizes += [('out', 2 * n * (self.dimu + 1))]           # [pi words | q words]
            total = sum((sz + 3) // 4 * 4 for _, sz in sizes)
            hp, dp = C.c_void_p(), C.c_void_p()
            _lib.check(lib.cur_host_alloc(4 * total, C.byref(hp), C.byref(dp)), 'cur_host_alloc')
            host = np.ctypeslib.as_array((C.c_float * total).from_address(hp.value))
            slot = dict(host_ptr=hp.value, seq=0)
            k = 0
            for name, sz in sizes:
                slot[name] = host[k:k + sz]
                slot['d_' + name] = dp.value + 4 * k
                k += (sz + 3) // 4 * 4
            words = slot['out'].reshape(n * (self.dimu + 1), 2)
            slot['val'] = words[:, 0]                              # float32 values: n * dimu actions, then n Q values
            slot['tag'] = words[:, 1].view(np.uint32)              # the call number each word was written by
            slot['d_q'] = slot['d_out'] + 8 * n * self.dimu
            slot['h_out'] = hp.value + (slot['d_out'] - dp.value)
            # host post-processing (cur_actions_finish_host): the caller's draws and the finished float32 [pi | q]
            slot['randn'] = np.empty((n, self.dimu), np.float64)
            slot['explore'] = np.empty(n, np.int64)
            slot['u_rand'] = np.empty((n, self.dimu), np.float64)
            slot['fin'] = np.empty(n * (self.dimu + 1), np.float32)
            slot['fin_u'] = slot['fin'][:n * self.dimu].reshape(n, self.dimu)
            slot['fin_q'] = slot['fin'][n * self.dimu:].reshape(n, 1)
            for name in ('randn', 'explore', 'u_rand', 'fin'):
                slot['p_' + name] = slot[name].ctypes.data
            slot['p_fin_q'] = slot['p_fin'] + 4 * n * self.dimu
            slot['refs'] = (C.byref(self.net.desc), C.byref(self._stats))
            self._action_slots[n] = slot
        return slot

    def _actions_one_launch(self, o, ag, g, task_descr, n, theta, compute_Q, device_noise, noise_eps, random_eps,
                            route=None):
        """cur_ddpg_actions_rows: inputs read from / actions written to mapped pinned memory by the kernel; completion =
        every output word carries this call's number (no copies, no stream synchronisation, no fence).  Returns
        (result, finished): the finished get_actions result on the zero-copy path (post-processing included), else the
        flat [pi | q] host array that `_finish_actions` still has to post-process.  `route` (experts._Route): the rows
        go to several experts of this shape in one routed launch, with its own noise pass and host draws."""
        lib = _lib.load()
        slot = self._action_slot(n)
        np.copyto(slot['o'], o.reshape(-1))
        np.copyto(slot['g'], g.reshape(-1))
        if self.relative_goals:
            np.copyto(slot['ag'], np.asarray(ag, np.float32).reshape(-1))
        if self.modular:
            np.copyto(slot['td'], np.asarray(task_descr, np.float32).reshape(-1))
        n_out = n * (self.dimu + (1 if compute_Q else 0))
        noisy = device_noise and (noise_eps != 0. or random_eps != 0.)
        if noisy or n > self.ACTION_ZERO_COPY_MAX:
            # plain float32 outputs in device memory, one D2H copy: device-side noise works in place on the device array
            # (Q is evaluated on the noise-free action, like the reference's Q_pi_tf, ddpg.py:138-146), and above a few
            # dozen rows 4-byte accesses over PCIe cost more than one bulk copy each way
            out = torch.empty(n * (self.dimu + 1), dtype=torch.float32, device=self.device)
            base = slot['d_o']
            if n > self.ACTION_ZERO_COPY_MAX:
                if 'dev_in' not in slot:
                    slot['n_in'] = (slot['d_out'] - slot['d_o']) // 4
                    slot['dev_in'] = torch.empty(slot['n_in'], dtype=torch.float32, device=self.device)
                _lib.check(lib.cur_copy_h2d(_lib.stream_ptr(), slot['dev_in'].data_ptr(), slot['d_o'], 4 * slot['n_in']),
                           'cur_copy_h2d')
                base = slot['dev_in'].data_ptr()
            rel = lambda name: base + (slot[name] - slot['d_o'])
            ptrs = (base, rel('d_ag') if self.relative_goals else None, rel('d_g'), rel('d_td') if self.modular else None,
                    n, float(self.clip_obs), out.data_ptr(), out.data_ptr() + 4 * n * self.dimu if compute_Q else None, 0)
            if route is None:
                _lib.check(lib.cur_ddpg_actions_rows(_lib.stream_ptr(), C.byref(self.net.desc), theta.data_ptr(),
                                                     C.byref(self._stats), *ptrs), 'cur_ddpg_actions_rows')
            else:
                route.launch(*ptrs)
            if noisy and route is None:
                _lib.check(lib.cur_action_noise(_lib.stream_ptr(), out.data_ptr(), n, self.dimu, float(self.max_u),
                                                float(noise_eps), float(random_eps), int(self.noise_seed) & (2 ** 64 - 1),
                                                self._action_calls), 'cur_action_noise')
            elif noisy:
                route.noise(out.data_ptr(), n, noise_eps, random_eps)
            return out[:n_out].cpu().numpy(), False
        slot['seq'] = seq = slot['seq'] % 0xFFFFFFF0 + 1
        if route is None:
            desc_ref, stats_ref = slot['refs']
            _lib.check(lib.cur_ddpg_actions_rows(
                _lib.stream_ptr(), desc_ref, theta.data_ptr(), stats_ref, slot['d_o'],
                slot['d_ag'] if self.relative_goals else None, slot['d_g'], slot['d_td'] if self.modular else None, n,
                float(self.clip_obs), slot['d_out'], slot['d_q'] if compute_Q else None, seq), 'cur_ddpg_actions_rows')
        else:
            route.launch(slot['d_o'], slot['d_ag'] if self.relative_goals else None, slot['d_g'],
                         slot['d_td'] if self.modular else None, n, float(self.clip_obs), slot['d_out'],
                         slot['d_q'] if compute_Q else None, seq)
        # The host RNG draws of ddpg.py:148-151 do not depend on the kernel's answer: take them (in reference order) while
        # the launch is in flight - ~10 us of NumPy calls hidden behind ~15 us of launch latency + weight stream.  The
        # arithmetic on the answer is one C call (cur_actions_finish_host: poll the words, NumPy's own evaluation types).
        p_randn = p_explore = p_u_rand = None
        if not device_noise:
            randn, explore, u_rand = (self._draw_action_noise if route is None else route.draw)(n, random_eps)
            np.copyto(slot['randn'], randn)
            np.copyto(slot['explore'], explore)
            np.copyto(slot['u_rand'], u_rand)
            p_randn, p_explore, p_u_rand = slot['p_randn'], slot['p_explore'], slot['p_u_rand']
        finish = (slot['h_out'], n, self.dimu, 1 if compute_Q else 0, seq, p_randn, p_explore, p_u_rand,
                  float(noise_eps) * float(self.max_u), float(self.max_u), slot['p_fin'],
                  slot['p_fin_q'] if compute_Q else None, 20000000)          # ~0.1 s of polls
        status = lib.cur_actions_finish_host(*finish)
        if status == 3:                     # no answer: let a launch failure surface, then give up
            torch.cuda.current_stream().synchronize()
            status = lib.cur_actions_finish_host(*finish)
            if status == 3:
                raise RuntimeError('cur_ddpg_actions_rows did not complete')
        _lib.check(status, 'cur_actions_finish_host')
        u = slot['fin_u']
        u = u[0].copy() if n == 1 else u.copy()                                            # ddpg.py:152-154
        return ([u, slot['fin_q'].copy()] if compute_Q else u), True

    CHAIN_MIN_ROWS = 1024      # update_schedule='auto': rows schedule below, tcgen05 chain kernel from here
    # pad_hidden='native', hidden 64 / 128: the narrow chain kernel from here (the rows schedule ends at 1024 rows and the
    # chain takes multiples of 128; profiles/r04_native_chain.json)
    NATIVE_CHAIN_MIN_ROWS = 1152
    ACTION_ROWS_MAX = 512      # rows per call served by the one-launch path (one CTA per 4 rows)
    ACTION_ZERO_COPY_MAX = 64  # ... of which up to this many rows travel zero-copy (kernel reads / writes host memory)

    def get_actions(self, o, ag, g, task_descr=None, noise_eps=0., random_eps=0., use_target_net=False,
                    compute_Q=False):
        """ddpg.py:129-161.  Up to ACTION_ROWS_MAX rows (the rollout's per-step call): ONE launch that reads the host
        arrays and writes the host actions itself (`_actions_one_launch`); larger batches: one H2D blob, prep + MLP level
        kernels, one D2H.  Exploration noise on the host RNG (default) or on the device (`action_noise='device'`)."""
        o = np.asarray(o, np.float32).reshape(-1, self.dimo)
        g = np.asarray(g, np.float32).reshape(-1, self.dimg)
        n = o.shape[0]
        theta = self.theta_target if use_target_net else self.theta_main
        device_noise = self.action_noise == 'device'
        if n <= self.ACTION_ROWS_MAX and self._action_rows_ok():
            res, finished = self._actions_one_launch(o, ag, g, task_descr, n, theta, compute_Q, device_noise, noise_eps,
                                                     random_eps)
            if device_noise:
                self._action_calls += 1
            return res if finished else self._finish_actions(res, n, compute_Q, device_noise, noise_eps, random_eps)
        parts = [o, g]
        if self.relative_goals:
            parts.append(np.asarray(ag, np.float32).reshape(-1, self.dimag))
        if self.modular:
            parts.append(np.asarray(task_descr, np.float32).reshape(-1, self.dimtd))
        sizes = [p.size for p in parts]
        host = torch.empty(sum(sizes), dtype=torch.float32, pin_memory=True)
        hv = host.numpy()
        k = 0
        for p, s in zip(parts, sizes):
            hv[k:k + s] = p.reshape(-1)
            k += s
        dev = host.to(self.device, non_blocking=True)
        base, k = dev.data_ptr(), 0
        ptrs = []
        for s in sizes:
            ptrs.append(base + 4 * k)
            k += s
        p_o, p_g = ptrs[0], ptrs[1]
        idx = 2
        p_ag = None
        if self.relative_goals:
            p_ag = ptrs[idx]
            idx += 1
        p_td = ptrs[idx] if self.modular else None
        out = torch.empty(n * (self.dimu + (1 if compute_Q else 0)), dtype=torch.float32, device=self.device)
        _lib.check(_lib.load().cur_ddpg_actions(
            _lib.stream_ptr(), C.byref(self.net.desc), theta.data_ptr(), C.byref(self._stats), p_o, p_ag, p_g, p_td, n,
            float(self.clip_obs), self._workspace(n).data_ptr(), out.data_ptr(),
            out.data_ptr() + 4 * n * self.dimu if compute_Q else None), 'cur_ddpg_actions')
        if device_noise:
            # Q above was evaluated on the noise-free action, like the reference's Q_pi_tf (ddpg.py:138-146)
            if noise_eps != 0. or random_eps != 0.:
                _lib.check(_lib.load().cur_action_noise(_lib.stream_ptr(), out.data_ptr(), n, self.dimu, float(self.max_u),
                                                        float(noise_eps), float(random_eps), int(self.noise_seed) & (2 ** 64 - 1),
                                                        self._action_calls), 'cur_action_noise')
            self._action_calls += 1
        return self._finish_actions(out.cpu().numpy(), n, compute_Q, device_noise, noise_eps, random_eps)

    def get_actions_workers(self, o, ag, g, task_descr=None, noise_eps=(), random_eps=(), streams=None,
                            use_target_net=False, compute_Q=False):
        """get_actions for the k reference workers this rank hosts, as ONE action launch over their k * B rows: rows
        [j * B, (j + 1) * B) are worker j's, acting with noise_eps[j] / random_eps[j] (0 for a worker that exploits).
        Worker j's exploration noise is what a lone agent of its reference rank gets (ddpg.py:147-152): host noise drawn
        from streams.rng(j) in reference order (randn, binomial, uniform; also when its eps are 0), taken while the
        launch is in flight; device noise (action_noise='device') keyed by streams.philox_key(j) at counter rows 0..B-1
        and this agent's call number, applied inside the launch (cur_ddpg_actions_rows_noisy).  Up to
        ACTION_ZERO_COPY_MAX rows zero-copy, up to ACTION_ROWS_MAX through device memory; anything the one-launch
        action kernel does not take raises ValueError.  Returns (u [k * B, dimu] float32, q [k * B, 1] or None)."""
        k = len(noise_eps)
        o = np.asarray(o, np.float32).reshape(-1, self.dimo)
        g = np.asarray(g, np.float32).reshape(-1, self.dimg)
        n = o.shape[0]
        if k == 0 or len(random_eps) != k or streams is None or len(streams) != k or n % k:
            raise ValueError('get_actions_workers takes k * B rows, k noise_eps / random_eps and the k workers\' streams')
        if n > self.ACTION_ROWS_MAX or not self._action_rows_ok():
            raise ValueError('get_actions_workers runs the one-launch action kernel (up to %d rows of a shape '
                             'cur_ddpg_rows_supported takes)' % self.ACTION_ROWS_MAX)
        B = n // k
        device_noise = self.action_noise == 'device'
        noisy = [float(ne) != 0. or float(re) != 0. for ne, re in zip(noise_eps, random_eps)]
        eps = {(float(ne), float(re)) for ne, re, on in zip(noise_eps, random_eps, noisy) if on}
        if device_noise and len(eps) > 1:
            raise ValueError('device noise: the workers that explore share one noise_eps / random_eps')
        lib = _lib.load()
        slot = self._action_slot(n)
        np.copyto(slot['o'], o.reshape(-1))
        np.copyto(slot['g'], g.reshape(-1))
        if self.relative_goals:
            np.copyto(slot['ag'], np.asarray(ag, np.float32).reshape(-1))
        if self.modular:
            np.copyto(slot['td'], np.asarray(task_descr, np.float32).reshape(-1))
        zero_copy = n <= self.ACTION_ZERO_COPY_MAX
        if zero_copy:
            slot['seq'] = seq = slot['seq'] % 0xFFFFFFF0 + 1
            base, out_pi, out_q = slot['d_o'], slot['d_out'], slot['d_q'] if compute_Q else None
        else:
            # above a few dozen rows: inputs and float32 outputs through device memory (as get_actions does)
            seq, out = 0, torch.empty(n * (self.dimu + 1), dtype=torch.float32, device=self.device)
            if 'dev_in' not in slot:
                slot['n_in'] = (slot['d_out'] - slot['d_o']) // 4
                slot['dev_in'] = torch.empty(slot['n_in'], dtype=torch.float32, device=self.device)
            _lib.check(lib.cur_copy_h2d(_lib.stream_ptr(), slot['dev_in'].data_ptr(), slot['d_o'], 4 * slot['n_in']),
                       'cur_copy_h2d')
            base = slot['dev_in'].data_ptr()
            out_pi, out_q = out.data_ptr(), out.data_ptr() + 4 * n * self.dimu if compute_Q else None
        rel = lambda name: base + (slot[name] - slot['d_o'])
        theta = self.theta_target if use_target_net else self.theta_main
        args = (_lib.stream_ptr(), C.byref(self.net.desc), theta.data_ptr(), C.byref(self._stats), base,
                rel('d_ag') if self.relative_goals else None, rel('d_g'), rel('d_td') if self.modular else None, n,
                float(self.clip_obs))
        if device_noise and eps:
            rows = self._noise_rows(slot, n)
            rows['seed'] = np.repeat(np.array([streams.philox_key(j) for j in range(k)], np.uint64), B)
            rows['call'] = self._action_calls
            rows['ctr'] = np.tile(np.arange(B, dtype=np.uint32), k)
            rows['noisy'] = np.repeat(np.array(noisy, np.uint32), B)
            ne, re = eps.pop()
            _lib.check(lib.cur_ddpg_actions_rows_noisy(*args, ne, re, slot['d_noise_rows'], out_pi, out_q, seq),
                       'cur_ddpg_actions_rows_noisy')
        else:
            _lib.check(lib.cur_ddpg_actions_rows(*args, out_pi, out_q, seq), 'cur_ddpg_actions_rows')
        if device_noise:
            self._action_calls += 1
        else:
            # every worker's draws from its own stream, in reference order, while the launch is in flight; the noise is
            # scaled here (noise_eps * max_u * randn, ddpg.py:148) because the workers' scales differ
            randn, explore, u_rand = slot['randn'], slot['explore'], slot['u_rand']
            for j in range(k):
                rng, s = streams.rng(j), slice(j * B, (j + 1) * B)
                np.multiply(float(noise_eps[j]) * self.max_u, rng.randn(B, self.dimu), out=randn[s])
                explore[s] = rng.binomial(1, random_eps[j], B)
                u_rand[s] = rng.uniform(low=-self.max_u, high=self.max_u, size=(B, self.dimu))
        if not zero_copy:
            res = out[:n * (self.dimu + (1 if compute_Q else 0))].cpu().numpy()
            u = res[:n * self.dimu].reshape(n, self.dimu)
            if not device_noise:
                u += slot['randn']                                                          # ddpg.py:148-149
                np.minimum(np.maximum(u, -self.max_u, out=u), self.max_u, out=u)            # ddpg.py:150
                u += slot['explore'].reshape(-1, 1) * (slot['u_rand'] - u)                  # ddpg.py:151
            return u.copy(), (res[n * self.dimu:].reshape(n, 1).copy() if compute_Q else None)
        draws = (None,) * 3 if device_noise else (slot['p_randn'], slot['p_explore'], slot['p_u_rand'])
        finish = (slot['h_out'], n, self.dimu, 1 if compute_Q else 0, seq, *draws, 1.0, float(self.max_u), slot['p_fin'],
                  slot['p_fin_q'] if compute_Q else None, 20000000)
        status = lib.cur_actions_finish_host(*finish)
        if status == 3:                     # no answer: let a launch failure surface, then give up
            torch.cuda.current_stream().synchronize()
            status = lib.cur_actions_finish_host(*finish)
            if status == 3:
                raise RuntimeError('the action launch did not complete')
        _lib.check(status, 'cur_actions_finish_host')
        return slot['fin_u'].copy(), (slot['fin_q'].copy() if compute_Q else None)

    def _noise_rows(self, slot, n):
        """The per-row {seed, call, ctr, noisy} table of cur_ddpg_actions_rows_noisy, in mapped pinned memory of the slot."""
        if 'noise_rows' not in slot:
            hp, dp = C.c_void_p(), C.c_void_p()
            size = C.sizeof(_lib.NoiseRow)
            _lib.check(_lib.load().cur_host_alloc(size * n, C.byref(hp), C.byref(dp)), 'cur_host_alloc')
            dt = np.dtype({'names': ['seed', 'call', 'ctr', 'noisy'], 'formats': ['<u8', '<u8', '<u4', '<u4'],
                           'offsets': [_lib.NoiseRow.seed.offset, _lib.NoiseRow.call.offset, _lib.NoiseRow.ctr.offset,
                                       _lib.NoiseRow.noisy.offset], 'itemsize': size})
            slot['noise_rows'] = np.ctypeslib.as_array((C.c_uint8 * (size * n)).from_address(hp.value)).view(dt)
            slot['d_noise_rows'] = dp.value
        return slot['noise_rows']

    def _action_rows_ok(self):
        if self._action_rows is None:
            self._action_rows = bool(self.action_path != 'levels' and self._rows_shape_ok(4))
        return self._action_rows

    def _draw_action_noise(self, n, random_eps):
        """The host RNG draws of ddpg.py:148-151 in the order the reference consumes np.random: randn (Gaussian noise),
        binomial (which rows act randomly), uniform (_random_action) - also when the eps are 0, like the reference."""
        return np.random.randn(n, self.dimu), np.random.binomial(1, random_eps, n), self._random_action(n)

    def _finish_actions(self, res, n, compute_Q, device_noise, noise_eps, random_eps, draw=None):
        """Action postprocessing (ddpg.py:147-155) on the flat [pi | q] host array `res` (owned by this call); the
        zero-copy path does the same arithmetic in cur_actions_finish_host (compared in tests/test_host_logic.py).
        `draw`: the host draws, when they are not this agent's _draw_action_noise (a routed expert step)."""
        u = res[:n * self.dimu].reshape(n, self.dimu)
        if not device_noise:
            randn, explore, u_rand = (draw or self._draw_action_noise)(n, random_eps)
            u += noise_eps * self.max_u * randn                                             # ddpg.py:148-149
            lim = self.max_u
            np.minimum(np.maximum(u, -lim, out=u), lim, out=u)                              # np.clip, ddpg.py:150
            u += explore.reshape(-1, 1) * (u_rand - u)                                      # ddpg.py:151
        u = u[0].copy() if n == 1 else u.copy()                                            # ddpg.py:152-154
        if not compute_Q:
            return u
        return [u, res[n * self.dimu:].reshape(n, 1).copy()]

    # ------------------------------------------------------------------------------------------
    def _multi_buffer(self):
        return 'buffer' in self.task_replay or self.task_replay == 'hand_designed'

    def store_episode(self, episode_batch, cp, n_ep, update_stats=True):
        """episode_batch: {key: [rollout_batch_size, T or T+1, dim]} (ddpg.py:163-223).  worker_buffers='own': the k
        workers' episodes stacked worker-major, [k * rollout_batch_size, ...]; episode b belongs to worker
        b // rollout_batch_size."""
        if self._own():
            return self._store_episode_own(episode_batch, cp, n_ep, update_stats)
        batch_size = episode_batch['ag'].shape[0]
        self.cp = cp
        self.n_episodes = n_ep
        some_buffer = self.buffer[1] if type(self.buffer) is list else self.buffer
        keys = list(some_buffer.buffer_shapes.keys())
        staged = StagedEpisodes({k: episode_batch[k] for k in keys}, some_buffer.layout, some_buffer.info_keys,
                                some_buffer.has_td, some_buffer.has_change, self.device)
        copies = []
        self._route_episodes(episode_batch, staged, range(batch_size), self.buffer, copies)
        staged.store(copies)
        self._staged = staged

        if update_stats:
            # HER-sample rollout_batch_size*T transitions of the fresh episodes and feed the preprocessed
            # o,g to the normalisers (ddpg.py:206-223)
            episode_batch['o_2'] = episode_batch['o'][:, 1:, :]
            episode_batch['ag_2'] = episode_batch['ag'][:, 1:, :]
            num = transitions_in_episode_batch(episode_batch)
            epi = episodes_to_device({k: episode_batch[k] for k in keys}, self.device, staged=staged)
            sampler = self.sample_transitions
            draws = None
            if self.her_rng == 'numpy':
                d = HostDraws(epi.n_episodes, epi.layout.T, num)
                d.draw_choices(sampler.mode, sampler.future_p, getattr(self, 'nb_tasks', 0), None)
                draws = [d]
            res = sampler.sample_device([(epi, num, None)], num, draws=draws, clip_obs=self.clip_obs,
                                        relative_goals=self.relative_goals, want=('o', 'g'))
            self.o_stats.update(res['o'])
            self.g_stats.update(res['g'])
            recompute_stats_packed((self.o_stats, self.g_stats), self._stats_partial, self.comm)

    def _route_episodes(self, episode_batch, staged, episodes, buffer, copies):
        """Slot choice of every episode in `episodes` into `buffer` (a list of module buffers, or one), appended to
        `copies` as store_staged descriptors."""
        if self.modular:
            change = np.asarray(episode_batch['change'])
            for b in episodes:
                active_tasks = apportion.active_modules(change[b, -1], self.tasks_ag_id, self.tasks_g_id)
                # (the reference all-reduces an unused counter here, ddpg.py:185 - dropped)
                if self._multi_buffer():
                    for task in active_tasks:                        # buffer[0] is never written (ddpg.py:191-195)
                        copies.append(buffer[task + 1].store_staged(staged, b))
                else:
                    copies.append(buffer.store_staged(staged, b))
        else:
            for b in episodes:
                copies.append(buffer.store_staged(staged, b))

    def _store_episode_own(self, episode_batch, cp, n_ep, update_stats):
        """store_episode of k workers with their own buffers: each worker routes its episodes into its buffers, slot draws
        from its own stream; one upload, the copies in as few cur_store_episodes launches as CUR_MAX_COPIES allows.  The
        normaliser batch: every worker HER-samples rollout_batch_size * T fresh transitions of its own episodes with its
        own draws, all into the one packed partial, which recompute divides by k (the reference's mean over ranks,
        normalizer.py:84-94)."""
        k = self.workers_per_rank
        n_total = episode_batch['ag'].shape[0]
        if n_total % k:
            raise ValueError('store_episode with %d workers needs k * rollout_batch_size episodes, got %d' % (k, n_total))
        rb = n_total // k
        self.cp = cp
        self.n_episodes = n_ep
        some_buffer = self.buffer[1] if type(self.buffer) is list else self.buffer
        keys = list(some_buffer.buffer_shapes.keys())
        staged = StagedEpisodes({key: episode_batch[key] for key in keys}, some_buffer.layout, some_buffer.info_keys,
                                some_buffer.has_td, some_buffer.has_change, self.device)
        copies = []
        for j in range(k):
            with self.worker_streams.use(j):
                self._route_episodes(episode_batch, staged, range(j * rb, (j + 1) * rb), self._worker_buffers[j], copies)
        staged.store(copies)
        self._staged = staged
        if not update_stats:
            return
        episode_batch['o_2'] = episode_batch['o'][:, 1:, :]
        episode_batch['ag_2'] = episode_batch['ag'][:, 1:, :]
        per = transitions_in_episode_batch(episode_batch) // k
        epi = episodes_to_device({key: episode_batch[key] for key in keys}, self.device, staged=staged)
        sampler = self.sample_transitions
        L = epi.layout
        hot, cold = L.T * L.trans_stride * rb, L.T * L.cold_stride * rb
        workers, draws = [], None if self.her_rng != 'numpy' else []
        for j in range(k):
            part = DeviceEpisodes(epi.storage[j * hot:(j + 1) * hot], epi.cold[j * cold:(j + 1) * cold], rb, L,
                                  epi.info_keys, epi.has_td, epi.has_change)
            workers.append((self.worker_streams.philox_key(j), [(part, per, None)]))
            if draws is not None:
                with self.worker_streams.use(j):
                    d = HostDraws(rb, L.T, per)
                    d.draw_choices(sampler.mode, sampler.future_p, getattr(self, 'nb_tasks', 0), None)
                draws.append(d)
        res = sampler.sample_workers(workers, per, draws=draws, clip_obs=self.clip_obs,
                                     relative_goals=self.relative_goals, want=('o', 'g'))
        self.o_stats.update(res['o'])
        self.g_stats.update(res['g'])
        recompute_stats_packed((self.o_stats, self.g_stats), self._stats_partial, self.comm, workers=k)

    def get_current_buffer_size(self):
        return sum([self.buffer[i].get_current_size() for i in range(self.nb_tasks)])

    def _sync_optimizers(self):
        self.Q_adam.sync()
        self.pi_adam.sync()
        self._wT_dirty = True

    # ------------------------------------------------------------------------------------------
    def _proportions(self, buffers=None):
        """LP-weighted apportioning of the batch over the module buffers (ddpg.py:255-286, 302-318); `buffers`: a
        worker's buffer set (worker_buffers='own': shared cp, that worker's fill levels)."""
        buffers = self.buffer if buffers is None else buffers
        sizes = [buffers[i].current_size for i in range(self.nb_tasks + 1)]
        if self.structure == 'curious':
            prop = apportion.proportions_curious(sizes, self.T, self.batch_size, self.task_replay, self.cp,
                                                 self.eps_task)
        else:
            prop = apportion.proportions_task_expert(sizes, self.T, self.batch_size, self.t_id)
        self.proportions = prop
        return prop

    def _sample_device(self, want, rng=None, want_idx=False):
        """Run the fused HER kernel for one batch; returns {key: float32 cuda tensor} (+ 'idx' with want_idx)."""
        rng = rng or self.her_rng
        if self._own():
            return self._sample_workers(want, rng, want_idx=want_idx)
        sampler = self.sample_transitions
        B = self.batch_size
        cp_proba = None
        perm = None
        if self.modular and self._multi_buffer() and (
                self.structure == 'curious' or self.task_replay == 'replay_current_task_buffer'):
            prop = self._proportions()
            segs = []
            for i in range(self.nb_tasks + 1):
                if prop[i] > 0:
                    if self.structure == 'curious':
                        ttr = i - 1 if i > 0 else None
                    else:
                        ttr = self.t_id
                    assert self.buffer[i].current_size > 0
                    segs.append((self.buffer[i].device_view(), int(prop[i]), ttr))
            shuffle = True
        else:
            buf = self.buffer
            assert buf.current_size > 0
            if self.modular and self.structure == 'curious' and self.task_replay == 'replay_cp_task_transition':
                cp_proba = apportion.cp_probabilities(self.cp, self.eps_task)       # ddpg.py:288-296
            segs = [(buf.device_view(), B, None)]
            shuffle = False
        draws = None
        if rng == 'numpy':
            draws = []
            for epi, count, ttr in segs:      # one sampler call per non-empty buffer, in buffer order
                d = HostDraws(epi.n_episodes, epi.layout.T, count)
                d.draw_choices(sampler.mode, sampler.future_p, getattr(self, 'nb_tasks', 0), cp_proba)
                draws.append(d)
            if shuffle:
                perm = np.arange(B)
                np.random.shuffle(perm)                                   # ddpg.py:338-339
                self._last_perm = perm
        return sampler.sample_device(segs, B, cp_proba=cp_proba, draws=draws, perm=perm, clip_obs=self.clip_obs,
                                     relative_goals=self.relative_goals, want=want, want_idx=want_idx)

    def _worker_segments(self, j):
        """Worker j's (buffer, count, task_to_replay) table over ALL its buffers in buffer order (count 0 where nothing is
        sampled), the apportioning of `_sample_device`, whether the batch is shuffled, and cp_proba as `_sample_device`
        passes it to the sampler."""
        bufs = self._worker_buffers[j]
        cp_proba = None
        if self.modular and self._multi_buffer() and (
                self.structure == 'curious' or self.task_replay == 'replay_current_task_buffer'):
            prop = self._proportions(bufs)
            segs = []
            for i in range(self.nb_tasks + 1):
                ttr = (i - 1 if i > 0 else None) if self.structure == 'curious' else self.t_id
                segs.append((bufs[i], int(prop[i]), ttr))
            return segs, True, cp_proba
        if self.modular and self.structure == 'curious' and self.task_replay == 'replay_cp_task_transition':
            cp_proba = apportion.cp_probabilities(self.cp, self.eps_task)       # ddpg.py:288-296
        return [(bufs, self.batch_size, None)], False, cp_proba

    def _sample_workers(self, want, rng=None, want_idx=False, out=None, dyn=None, step=None, call_offset=None):
        """worker_buffers='own': the batches of the k workers, each from its own buffers with its own draws, as one
        cur_her_sample_workers launch; rows [j * batch_size, (j + 1) * batch_size) are worker j's batch."""
        rng = rng or self.her_rng
        sampler = self.sample_transitions
        B = self.batch_size
        workers, draws, perms, cp_proba = [], [], [], None
        for j in range(self.workers_per_rank):
            segs, shuffle, cp_proba = self._worker_segments(j)
            for buf, count, _ in segs:
                assert count == 0 or buf.current_size > 0
            workers.append((self.worker_streams.philox_key(j), [(b.device_view(), c, t) for b, c, t in segs]))
            if rng == 'numpy':
                with self.worker_streams.use(j):
                    for b, count, _ in segs:          # one sampler call per non-empty buffer, in buffer order
                        if count > 0:
                            d = HostDraws(b.current_size, b.T, count)
                            d.draw_choices(sampler.mode, sampler.future_p, getattr(self, 'nb_tasks', 0), cp_proba)
                            draws.append(d)
                    if shuffle:
                        perm = np.arange(B)
                        np.random.shuffle(perm)                           # ddpg.py:338-339
                        perms.append(perm + j * B)
        perm = np.concatenate(perms) if perms else None
        if perm is not None:
            self._last_perm = perm[:B]
        return sampler.sample_workers(workers, B, dyn=dyn, step=step, cdf=cp_proba, draws=draws if rng == 'numpy' else None,
                                      perm=perm, clip_obs=self.clip_obs, relative_goals=self.relative_goals, want=want,
                                      want_idx=want_idx, out=out, call_offset=call_offset)

    _STAGE_TO_KERNEL = {'ag': 'ag', 'g': 'g', 'o': 'o', 'task_descr': 'td', 'u': 'u', 'o_2': 'o_2', 'g_2': 'g_2',
                        'r': 'r'}

    def sample_batch(self):
        """Returns the staged batch as a list of host arrays in stage_shapes order (ddpg.py:251-360)."""
        want = tuple(self._STAGE_TO_KERNEL[k] for k in self.stage_shapes.keys())
        res = self._sample_device(want)
        torch.cuda.current_stream().synchronize()
        B = self.batch_size                # worker_buffers='own': worker 0's batch
        return [res[self._STAGE_TO_KERNEL[k]][:B].cpu().numpy().astype(np.float64) for k in self.stage_shapes.keys()]

    def stage_batch(self, batch=None):
        """ddpg.py:362-366.  With batch=None the batch is sampled on the device and never leaves it."""
        if batch is None:
            want = ('o', 'g', 'u', 'td', 'o_2', 'g_2', 'r') if self.modular else ('o', 'g', 'u', 'o_2', 'g_2', 'r')
            self._batch = self._sample_device(want)
            return
        assert len(self.stage_shapes) == len(batch)
        dev = {}
        for key, arr in zip(self.stage_shapes.keys(), batch):
            dev[self._STAGE_TO_KERNEL[key]] = torch.from_numpy(
                np.ascontiguousarray(arr, dtype=np.float32)).to(self.device, non_blocking=True)
        self._batch = dev

    def _grads(self):
        b = self._batch
        n = b['o'].shape[0]
        cb = _lib.Batch(b['o'].data_ptr(), b['g'].data_ptr(), b['u'].data_ptr(),
                        b['td'].data_ptr() if self.modular else None, b['o_2'].data_ptr(), b['g_2'].data_ptr(),
                        b['r'].data_ptr(), n)
        q_pi = torch.empty((n, 1), dtype=torch.float32, device=self.device)
        if self._use_rows(n):
            _lib.check(_lib.load().cur_ddpg_rows_step(
                _lib.stream_ptr(), C.byref(self.net.desc), self.theta_main.data_ptr(), self.theta_target.data_ptr(),
                C.byref(self._stats), C.byref(cb), C.byref(self._hyper), self._workspace_rows(n).data_ptr(),
                self.grads.data_ptr(), self._q_loss.data_ptr(), self._pi_loss.data_ptr(), q_pi.data_ptr(), None, None),
                'cur_ddpg_rows_step')
        elif self._use_native_chain(n):
            _lib.check(_lib.load().cur_ddpg_chain_grads(
                _lib.stream_ptr(), C.byref(self.net.desc), self.theta_main.data_ptr(), self.theta_target.data_ptr(),
                C.byref(self._stats), C.byref(cb), C.byref(self._hyper), self._workspace_chain(n).data_ptr(),
                self.grads.data_ptr(), self._q_loss.data_ptr(), self._pi_loss.data_ptr(), q_pi.data_ptr()),
                'cur_ddpg_chain_grads')
        else:
            _lib.check(_lib.load().cur_ddpg_grads(
                _lib.stream_ptr(), C.byref(self.net.desc), self.theta_main.data_ptr(), self.theta_target.data_ptr(),
                C.byref(self._stats), C.byref(cb), C.byref(self._hyper), self._workspace(n).data_ptr(),
                self.grads.data_ptr(), self._q_loss.data_ptr(), self._pi_loss.data_ptr(), q_pi.data_ptr()),
                'cur_ddpg_grads')
        return self._q_loss, q_pi, self._view(self.grads, 'Q'), self._view(self.grads, 'pi')

    def _update(self, Q_grad, pi_grad):
        """Q_adam.update + pi_adam.update (ddpg.py:246-248).  Both vectors live in one arena, so the two
        MPI all-reduces of the reference become ONE NCCL all-reduce, and when both nets share the step
        size one fused Adam launch covers the arena."""
        group, world = _world(self.comm)
        self._wT_dirty = True
        if self.Q_adam.t % 100 == 0:
            self.Q_adam.check_synced()
            self.pi_adam.check_synced()
        allreduce_sum_(self.grads, self.comm)                     # SUM, not mean (ddpg.py:452-453)
        self.Q_adam.t += 1
        self.pi_adam.t += 1
        lib = _lib.load()
        for adam, grad, lr in ((self.Q_adam, Q_grad, self.Q_lr), (self.pi_adam, pi_grad, self.pi_lr)):
            a = adam_step_scale(lr, adam.beta1, adam.beta2, adam.t)
            _lib.check(lib.cur_adam_step(_lib.stream_ptr(), adam.theta.data_ptr(), grad.data_ptr(),
                                         adam.m.data_ptr(), adam.v.data_ptr(), adam.theta.numel(),
                                         float(np.float32(-a)), adam.beta1, adam.beta2, adam.epsilon, 1.0),
                       'cur_adam_step')

    # ------------------------------------------------------------------------------------------
    # CUDA-graph fast path: HER sample -> grads -> all-reduce -> Adam captured once, replayed per update.
    # Everything that changes between updates lives in device memory (cur_her_dyn control block, the
    # shared step counter, the Adam step-scale table), so the frozen kernel arguments stay valid.
    LOSS_RING = 4096
    ADAM_TABLE = 65536
    GRAPH_STREAM_OFFSET = 1 << 40          # Philox call_offset base of the train-step stream

    def _all_segments(self):
        """Fixed segment table over every buffer (count 0 where nothing is sampled)."""
        if self.modular and self._multi_buffer():
            segs = []
            for i in range(self.nb_tasks + 1):
                ttr = (i - 1 if i > 0 else None) if self.structure == 'curious' else self.t_id
                segs.append((self.buffer[i], ttr))
            return segs
        return [(self.buffer, None)]

    def _dyn_signature(self):
        cp = None if self.cp is None else tuple(np.asarray(self.cp, np.float64).tolist())
        if self._own():
            sets = [b if isinstance(b, list) else [b] for b in self._worker_buffers]
            return tuple(b.current_size for bufs in sets for b in bufs), cp
        segs = self._all_segments()
        return tuple(b.current_size for b, _ in segs), cp

    def _refresh_dyn(self):
        """Recompute the LP apportioning (ddpg.py:255-318) and push it to the device control block."""
        sig = self._dyn_signature()
        if sig == self._graph_sig:
            return
        if self._own():
            self._refresh_worker_dyn()
            self._graph_sig = sig
            return
        segs = self._all_segments()
        d = self._dyn_struct
        if self.modular and self._multi_buffer():
            prop = self._proportions()
        else:
            assert self.buffer.current_size > 0
            prop = [self.batch_size]
            if self.modular and self.structure == 'curious' and self.task_replay == 'replay_cp_task_transition':
                _lib.set_cdf(d, apportion.cp_probabilities(self.cp, self.eps_task))
            elif self.sample_transitions.mode == _lib.MODE_CP_TASK:
                _lib.set_cdf(d, np.ones(self.nb_tasks) / self.nb_tasks)
        mult = self._graph_rows // self.batch_size          # wide batch: every worker's apportioning, k times
        for i, (buf, _) in enumerate(segs):
            d.n_episodes[i] = int(buf.current_size)
            d.count[i] = int(prop[i]) * mult
        C.memmove(self._dyn_host.data_ptr(), C.addressof(d), C.sizeof(d))
        self._dyn_dev.copy_(self._dyn_host, non_blocking=True)
        self._graph_sig = sig

    def _refresh_worker_dyn(self):
        """worker_buffers='own': every worker's apportioning (shared cp, its own fill levels) and cdf into the device
        control blocks of the captured worker sampler."""
        d = self._wdyn_struct
        for j in range(self.workers_per_rank):
            segs, _, cp_proba = self._worker_segments(j)
            for i, (buf, count, _) in enumerate(segs):
                d[j].n_episodes[i] = int(buf.current_size)
                d[j].count[i] = int(count)
            if cp_proba is not None:
                _lib.set_cdf(d[j], cp_proba)
            elif self.sample_transitions.mode == _lib.MODE_CP_TASK:
                _lib.set_cdf(d[j], np.ones(self.nb_tasks) / self.nb_tasks)
        C.memmove(self._wdyn_host.data_ptr(), C.addressof(d), C.sizeof(d))
        self._wdyn_dev.copy_(self._wdyn_host, non_blocking=True)

    def _prepare_graph_state(self):
        """Device-resident state of the graph path (control block, loss rings, Adam tables, fixed batch buffers)."""
        dev = self.device
        # several workers per rank as ONE wide batch: same gradient as k single-batch launches (loss seeds scaled by
        # 1 / batch_size, cur_ddpg_hyper.loss_rows) on the rows schedule up to 1024 rows or the tensor-core levels
        # schedule above (3x faster at 19 workers), or the chain kernel at a native width; otherwise k accumulating
        # launches of the rows schedule
        k = self.workers_per_rank
        lib = _lib.load()
        wide_rows = k * self.batch_size
        self._wide = bool(k > 1 and self.workers_mode != 'micro' and (
            (self.update_schedule != 'levels' and self._rows_shape_ok(wide_rows)) or
            lib.cur_ddpg_uses_tensor_cores(C.byref(self.net.desc), wide_rows) or self._use_native_chain(wide_rows)))
        if self._own() and k > 1 and not self._wide:
            raise ValueError("worker_buffers='own' needs a schedule that takes workers x batch_size rows in one update "
                             "(rows up to 1024, the chain kernel or the tensor-core levels schedule above)")
        self._graph_rows = self.batch_size * (k if self._wide else 1)
        self._micro = 1 if self._wide else k
        B = self._graph_rows
        L = self._all_segments()[0][0].layout
        self._dyn_struct = _lib.HerDyn()
        self._dyn_struct.step = self._step.data_ptr()
        nbytes = C.sizeof(_lib.HerDyn)
        self._dyn_host = torch.zeros(nbytes, dtype=torch.uint8, pin_memory=True)
        self._dyn_dev = torch.zeros(nbytes, dtype=torch.uint8, device=dev)
        if self._own():
            self._wdyn_struct = (_lib.HerWorkerDyn * k)()
            self._wdyn_host = torch.zeros(C.sizeof(self._wdyn_struct), dtype=torch.uint8, pin_memory=True)
            self._wdyn_dev = torch.zeros(C.sizeof(self._wdyn_struct), dtype=torch.uint8, device=dev)
        self._q_ring = torch.zeros(self.LOSS_RING, dtype=torch.float32, device=dev)
        self._pi_ring = torch.zeros(self.LOSS_RING, dtype=torch.float32, device=dev)
        self._q_pi = torch.zeros((B, 1), dtype=torch.float32, device=dev)
        self._adam_tables = [torch.from_numpy(_adam_table(lr, adam.beta1, adam.beta2, self.ADAM_TABLE)).to(dev)
                             for adam, lr in ((self.Q_adam, self.Q_lr), (self.pi_adam, self.pi_lr))]
        dims = dict(o=L.dimo, g=L.dimg, u=L.dimu, td=L.dimtd, o_2=L.dimo, r=1)
        want = [k for k in ('o', 'g', 'u', 'td', 'o_2', 'r') if dims[k] > 0]
        if self.relative_goals:
            want.append('g_2')
            dims['g_2'] = L.dimg
        self._gbatch = {k: torch.empty((B, dims[k]), dtype=torch.float32, device=dev) for k in want}
        self._gwant = tuple(want)
        self._ghyper = _lib.DdpgHyper(self._hyper.gamma, self._hyper.clip_return, self._hyper.action_l2,
                                      self._hyper.clip_pos_returns, self._step.data_ptr(), self.LOSS_RING,
                                      self._micro if self._micro > 1 else 0)
        if self._wide or self._own():
            self._ghyper.loss_rows = self.batch_size
        if self._micro > 1 and not self._use_rows(B):
            raise ValueError('workers_per_rank > 1 on the CUDA-graph path needs the rows schedule or a batch the '
                             'tensor-core levels schedule takes (workers x batch_size >= 1024, a multiple of 128)')
        if self._use_rows(B):
            self._workspace_rows(B)
        elif self._use_native_chain(B):
            self._workspace_chain(B)
        else:
            self._workspace(B)
        self._peer = None
        self._xchg = None
        kind = self._exchange_kind()
        if kind == 'tile':
            from .parallel import TileGradExchange
            self._xchg = TileGradExchange(self.net.arena, self.comm, mode=self.xchg_mode,
                                          timeline_tiles=self.xchg_timeline_tiles)
        elif kind is not None:
            from .parallel import PeerGradExchange
            # the sharded exchange moves 8x fewer bytes at 8 GPUs but measured no faster (2 GPUs: 83 us full / 91 us
            # sharded, 8 GPUs: 97.3 / 98.2): the exchange is latency / straggler bound, so the one-round kernel is default
            self._peer = PeerGradExchange(self.net.arena, self.comm, sharded=self.grad_exchange == 'p2p_sharded')
            self._peer.ctx.step_div = self._micro
            # the one-round exchange kernel also writes W^T of the stepped hidden layers: no transpose launch per update
            self._peer_wT = None
            import os
            # opt-in (CUR_P2P_WT=1): measured 4 us SLOWER per update on 2 GPUs than the separate 2.5 us transpose
            # launch (the tile phase runs behind the linear phase on the kernel's 148 CTAs)
            if not self._peer.sharded and os.environ.get('CUR_P2P_WT', '0') == '1':
                self._peer_wT = _lib.P2PTransposes()
                _lib.check(lib.cur_ddpg_rows_transposes(C.byref(self.net.desc), self._workspace_rows(B).data_ptr(), B,
                                                        C.byref(self._peer_wT)), 'cur_ddpg_rows_transposes')
            self._ghyper.grads_parity_stride = self.net.arena
        self._graph_sig = None
        self._refresh_dyn()
        self._graph_state_ready = True

    def _build_graph(self):
        dev = self.device
        self._prepare_graph_state()
        torch.cuda.current_stream().synchronize()
        # warm-up run outside capture (lazy module loading, cudaFuncSetAttribute)
        state = (self.theta_main.clone(), self._adam_m.clone(), self._adam_v.clone(), self._step.clone())
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            fused = self._launch_sample_and_grads(solo=True)
            if not fused:
                self._launch_adam(warmup=True)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize(dev)
        self.theta_main.copy_(state[0])
        for dst, src in zip((self._adam_m, self._adam_v, self._step), state[1:]):
            dst.copy_(src)
        # One rank: the whole update is one graph.  Several ranks: the graph ends after the gradients; the
        # NCCL all-reduce and the Adam launch follow on the same stream (collectives are kept out of the
        # capture: a captured torch NCCL all-reduce dead-locked on the 2-GPU box).
        # With the peer-memory exchange the all-reduce IS the Adam kernel and the whole update is one graph again.
        self._graph_has_adam = _world(self.comm)[1] == 1 or self._peer is not None or self._xchg is not None
        keeps_wT = self._peer is not None and getattr(self, '_peer_wT', None) is not None
        if keeps_wT:
            self._ghyper.transposes_valid = 1
        g = torch.cuda.CUDAGraph()
        with capture_graph(g):
            # fused Adam: its epilogue keeps W^T current, so the captured update has no transpose launch
            fused = self._launch_sample_and_grads(keep_wT=fused)
            if self._graph_has_adam and not fused:
                self._launch_adam()
        self._graph = g
        self._graph_fused = fused or keeps_wT
        self._wT_dirty = True            # the warm-up stepped (and we restored) theta: rebuild W^T before the first replay
        if self._peer is not None or self._xchg is not None:
            import torch.distributed as dist
            torch.cuda.synchronize(dev)
            dist.barrier(group=_world(self.comm)[0])

    def _exchange_kind(self):
        """None (one rank, or NCCL after the graph) | 'tile' | 'p2p' | 'p2p_sharded'."""
        group, n = _world(self.comm)
        if n <= 1 or self.grad_exchange == 'nccl':
            return None
        import torch.distributed as dist
        ok = (self._use_rows(self._graph_rows) and self._same_rule() and n <= _lib.CUR_MAX_RANKS and
              dist.get_backend(group) == 'nccl')
        if self.grad_exchange != 'auto' and not ok:
            raise ValueError('grad_exchange=%r needs the rows schedule, one Adam rule for both nets and an NCCL '
                             'group of <= %d ranks' % (self.grad_exchange, _lib.CUR_MAX_RANKS))
        if not ok:
            return None
        return 'tile' if self.grad_exchange == 'auto' else self.grad_exchange

    def _same_rule(self):
        qa, pa = self.Q_adam, self.pi_adam
        return (self.Q_lr, qa.beta1, qa.beta2, qa.epsilon) == (self.pi_lr, pa.beta1, pa.beta2, pa.epsilon)

    def _launch_sample_and_grads(self, keep_wT=False, solo=False):
        """HER sample + gradients of one update, all parameters frozen / device-resident (capturable).
        Returns True when Adam was fused into the weight-gradient launch.  keep_wT: the transposed hidden-layer
        weights in the rows workspace are current (maintained by the fused Adam epilogue, see _refresh_wT).
        solo: the warm-up run outside capture - no peer is touched with an update that is discarded afterwards."""
        lib = _lib.load()
        sampler = self.sample_transitions
        segs = [(buf.device_view(), 0, ttr) for buf, ttr in self._all_segments()]
        her_args = None
        if self._own():
            # the workers' batches: one standalone sampler launch (not fused into the rows prologue)
            self._sample_workers(self._gwant, rng='philox', out=self._gbatch, dyn=self._wdyn_dev.data_ptr(),
                                 step=self._step.data_ptr(), call_offset=self.GRAPH_STREAM_OFFSET)
        else:
            her_args = self._fused_her_args(segs)
            if her_args is None:
                sampler.sample_device(segs, self._graph_rows, clip_obs=self.clip_obs,
                                      relative_goals=self.relative_goals, want=self._gwant, out=self._gbatch,
                                      dyn=self._dyn_dev.data_ptr(), call_offset=self.GRAPH_STREAM_OFFSET)
        b = self._gbatch
        n = self._graph_rows
        g2 = b['g_2'] if self.relative_goals else b['g']       # g_2 == g without relative goals (ddpg.py:353)
        cb = _lib.Batch(b['o'].data_ptr(), b['g'].data_ptr(), b['u'].data_ptr(),
                        b['td'].data_ptr() if self.modular else None, b['o_2'].data_ptr(), g2.data_ptr(),
                        b['r'].data_ptr(), n)
        qa = self.Q_adam
        if self._use_rows(n):
            # with one rank there is no all-reduce between _grads and _update: Adam runs in the epilogue of
            # the weight-gradient launch (2 launches per update after the HER kernel)
            # ... and with several ranks when the tiles are exchanged inside that launch (TileGradExchange); with
            # several workers per rank the epilogue of the update's last launch steps the complete sum
            fuse = self._same_rule() and (_world(self.comm)[1] == 1 or self._xchg is not None)
            adam = _lib.AdamFused(self._adam_m.data_ptr(), self._adam_v.data_ptr(), self._adam_tables[0].data_ptr(),
                                  self.ADAM_TABLE, 1 if keep_wT else 0, qa.beta1, qa.beta2, qa.epsilon,
                                  C.pointer(self._xchg.ctx) if (self._xchg is not None and not solo) else None) \
                if fuse else None
            base_valid = self._ghyper.transposes_valid
            for j in range(self._micro):
                # the weights do not change between the workers of one update: only the first launch re-transposes
                self._ghyper.transposes_valid = 1 if (j > 0 or base_valid) else 0
                if fuse:
                    adam.transposes_valid = 1 if (j > 0 or keep_wT) else 0
                if j > 0 and her_args is None:            # unfused sampling: a fresh batch for every worker
                    sampler.sample_device(segs, self._graph_rows, clip_obs=self.clip_obs,
                                          relative_goals=self.relative_goals, want=self._gwant, out=self._gbatch,
                                          dyn=self._dyn_dev.data_ptr(), call_offset=self.GRAPH_STREAM_OFFSET)
                _lib.check(lib.cur_ddpg_rows_step(
                    _lib.stream_ptr(), C.byref(self.net.desc), self.theta_main.data_ptr(), self.theta_target.data_ptr(),
                    C.byref(self._stats), C.byref(cb), C.byref(self._ghyper), self._workspace_rows(n).data_ptr(),
                    self._peer.grads_ptr(0) if self._peer is not None else self.grads.data_ptr(),
                    self._q_ring.data_ptr(), self._pi_ring.data_ptr(), self._q_pi.data_ptr(),
                    C.byref(adam) if fuse else None, C.byref(her_args) if her_args is not None else None),
                    'cur_ddpg_rows_step')
            self._ghyper.transposes_valid = base_valid
            return fuse
        if self._use_native_chain(n):
            _lib.check(lib.cur_ddpg_chain_grads(
                _lib.stream_ptr(), C.byref(self.net.desc), self.theta_main.data_ptr(), self.theta_target.data_ptr(),
                C.byref(self._stats), C.byref(cb), C.byref(self._ghyper), self._workspace_chain(n).data_ptr(),
                self.grads.data_ptr(), self._q_ring.data_ptr(), self._pi_ring.data_ptr(), self._q_pi.data_ptr()),
                'cur_ddpg_chain_grads')
            return False
        _lib.check(lib.cur_ddpg_grads(
            _lib.stream_ptr(), C.byref(self.net.desc), self.theta_main.data_ptr(), self.theta_target.data_ptr(),
            C.byref(self._stats), C.byref(cb), C.byref(self._ghyper), self._workspace(n).data_ptr(),
            self.grads.data_ptr(), self._q_ring.data_ptr(), self._pi_ring.data_ptr(), self._q_pi.data_ptr()),
            'cur_ddpg_grads')
        return False

    def _fused_her_args(self, segs):
        """The sampler's cur_her_args for the rows update kernel to sample its own rows in its prologue (no separate HER
        launch), or None: the rows schedule does not run, fusing is off, or a transition does not fit that kernel's HER
        stage (cur_ddpg_rows_her_supported) - the batch is then sampled into _gbatch by the standalone kernel."""
        if not (self._use_rows(self._graph_rows) and self.fuse_her):
            return None
        her_args, keep = self.sample_transitions.sample_device(
            segs, self._graph_rows, clip_obs=self.clip_obs, relative_goals=self.relative_goals, want=(),
            dyn=self._dyn_dev.data_ptr(), call_offset=self.GRAPH_STREAM_OFFSET, args_only=True)
        if not _lib.load().cur_ddpg_rows_her_supported(C.byref(self.net.desc), C.byref(her_args)):
            return None
        self._her_keep = keep
        return her_args

    def _launch_adam(self, warmup=False):
        """Adam on the (already all-reduced) gradient arena; the step scale is read from the device table with
        the device step counter, so the launch is identical every update."""
        lib = _lib.load()
        qa = self.Q_adam
        if self._peer is not None:
            # sum the world's gradients out of peer memory and step, one kernel (csrc/p2p.cu).  The warm-up run
            # outside capture uses a world-of-one context so that no peer is signalled with a discarded update.
            if warmup:
                solo = _lib.P2PCtx()
                solo.rank, solo.world, solo.arena = 0, 1, self._peer.arena
                solo.step_div = self._micro
                solo.region[0] = self._peer.own
                _lib.check(lib.cur_p2p_allreduce_adam(
                    _lib.stream_ptr(), C.byref(solo), self.theta_main.data_ptr(), self._adam_m.data_ptr(),
                    self._adam_v.data_ptr(), self._adam_tables[0].data_ptr(), self.ADAM_TABLE, self._step.data_ptr(),
                    qa.beta1, qa.beta2, qa.epsilon, None), 'cur_p2p_allreduce_adam')
            else:
                self._peer.allreduce_adam(_lib.stream_ptr(), self.theta_main, self._adam_m, self._adam_v,
                                          self._adam_tables[0], self.ADAM_TABLE, self._step, qa.beta1, qa.beta2,
                                          qa.epsilon, transposes=self._peer_wT)
            return
        if self._same_rule():
            # same step rule for both nets: ONE launch over the whole [Q | pad | pi] arena (padding has zero
            # gradient and stays zero)
            _lib.check(lib.cur_adam_step_graph(
                _lib.stream_ptr(), self.theta_main.data_ptr(), self.grads.data_ptr(), self._adam_m.data_ptr(),
                self._adam_v.data_ptr(), self.theta_main.numel(), self._adam_tables[0].data_ptr(), self.ADAM_TABLE,
                self._step.data_ptr(), qa.beta1, qa.beta2, qa.epsilon, 1.0, self._micro), 'cur_adam_step_graph')
            return
        for adam, which, table in ((self.Q_adam, 'Q', self._adam_tables[0]), (self.pi_adam, 'pi', self._adam_tables[1])):
            _lib.check(lib.cur_adam_step_graph(
                _lib.stream_ptr(), adam.theta.data_ptr(), self._view(self.grads, which).data_ptr(), adam.m.data_ptr(),
                adam.v.data_ptr(), adam.theta.numel(), table.data_ptr(), self.ADAM_TABLE, self._step.data_ptr(),
                adam.beta1, adam.beta2, adam.epsilon, 1.0, self._micro), 'cur_adam_step_graph')

    def _refresh_wT(self):
        """Rebuild the transposed hidden-layer weights in the rows workspace after theta_main changed outside the
        fused update (initial weights, set_flat / load_weights, broadcast from rank 0, launch-by-launch updates)."""
        B = self._graph_rows                 # the workspace of the captured update (workers x batch_size rows when wide)
        _lib.check(_lib.load().cur_ddpg_rows_refresh(_lib.stream_ptr(), C.byref(self.net.desc), self.theta_main.data_ptr(),
                                                     self._workspace_rows(B).data_ptr(), B), 'cur_ddpg_rows_refresh')
        self._wT_dirty = False

    def _train_graph(self):
        if self._graph is None:
            self._build_graph()
        if self.Q_adam.t % 100 == 0:
            if self._peer is not None:
                self._peer.check()
            self.Q_adam.check_synced()
            self.pi_adam.check_synced()
        self._refresh_dyn()
        if self._graph_fused and self._wT_dirty:          # (only the rows schedule with the fused optimiser)
            self._refresh_wT()
        k = self._micro                    # the loss of the rank's last worker (device ring slot = launch index % ring)
        slot = (self._n_updates * k + k - 1) % self.LOSS_RING
        self._graph.replay()
        if not self._graph_has_adam:
            allreduce_sum_(self.grads, self.comm)                 # SUM, not mean (ddpg.py:452-453)
            self._launch_adam()
        self._n_updates += 1
        self.Q_adam.t += 1
        self.pi_adam.t += 1
        if self.own_train_outputs:        # owned copies like the reference's arrays (one small device copy per update)
            return LazyHost(self._q_ring[slot].clone()), LazyHost(self._q_pi.clone())
        # views of the graph's fixed output buffers: the loss slot is reused after LOSS_RING updates, Q_pi by the very
        # next one - a stale read raises (LazyHost) instead of returning a later update's values
        n = self._n_updates
        return (LazyHost(self._q_ring[slot], lambda: self._n_updates - n < self.LOSS_RING),
                LazyHost(self._q_pi, lambda: self._n_updates == n))

    def train(self, stage=True):
        """One DDPG update (ddpg.py:368-373).  Returns (critic_loss, actor_loss) as lazily synchronising
        host values; like the reference, "actor_loss" is main.Q_pi, the whole [B,1] array (ddpg.py:237-243)."""
        if stage and self.use_cuda_graph and self.her_rng == 'philox':
            return self._train_graph()
        if stage:
            self.stage_batch()
        critic_loss, actor_loss, Q_grad, pi_grad = self._grads()
        if self.workers_per_rank > 1 and not self._own():
            # several reference workers on this rank: sum of their single-batch gradients (ddpg.py:452-453)
            assert stage, 'workers_per_rank > 1 samples its own batches'
            total = self.grads.clone()
            for _ in range(self.workers_per_rank - 1):
                self.stage_batch()
                critic_loss, actor_loss, Q_grad, pi_grad = self._grads()
                total += self.grads
            self.grads.copy_(total)
        self._update(Q_grad, pi_grad)
        # the device counter counts sampled batches (Philox stream position); the workers of 'own' are one wide batch
        self._step += 1 if self._own() else self.workers_per_rank
        self._n_updates += 1
        return LazyHost(critic_loss.clone().reshape(())), LazyHost(actor_loss)

    def _init_target_net(self):
        _lib.check(_lib.load().cur_polyak(_lib.stream_ptr(), self.theta_target.data_ptr(), self.theta_main.data_ptr(),
                                          self.theta_main.numel(), 0.0), 'cur_polyak')

    def update_target_net(self):
        if getattr(self, '_peer', None) is not None:
            self._peer.check()              # (once per cycle: a timed-out exchange must not survive into the target net)
        _lib.check(_lib.load().cur_polyak(_lib.stream_ptr(), self.theta_target.data_ptr(), self.theta_main.data_ptr(),
                                          self.theta_main.numel(), float(self.polyak)), 'cur_polyak')

    def clear_buffer(self):
        for bufs in (self._worker_buffers if self._own() else [self.buffer]):
            for i in range(self.nb_tasks):
                bufs[i].clear_buffer()

    # ------------------------------------------------------------------------------------------
    def logs(self, prefix=''):
        logs = []
        logs += [('stats_o/mean', float(self.o_stats.mean.mean().item()))]
        logs += [('stats_o/std', float(self.o_stats.std.mean().item()))]
        logs += [('stats_g/mean', float(self.g_stats.mean.mean().item()))]
        logs += [('stats_g/std', float(self.g_stats.std.mean().item()))]
        if prefix != '' and not prefix.endswith('/'):
            return [(prefix + '/' + key, val) for key, val in logs]
        return logs

    def _vars_list(self, which, target=False):
        flat = self.get_flat(which, target)
        out, k = [], 0
        for s in self.net.var_shapes(which):
            n = int(np.prod(s))
            out.append(flat[k:k + n].reshape(s).copy())
            k += n
        return out

    def save_weights(self, path):
        """<path>_weights.pkl = [main/Q, main/pi, target/Q, target/pi, o_stats, g_stats] as lists of arrays
        (ddpg.py:481-497) - the reference's on-disk format."""
        to_save = [self._vars_list('Q'), self._vars_list('pi'), self._vars_list('Q', True),
                   self._vars_list('pi', True), self.o_stats.state_list(), self.g_stats.state_list()]
        with open(path + '_weights.pkl', 'wb') as f:
            pickle.dump(to_save, f)

    def load_weights(self, path):
        with open(path + '_weights.pkl', 'rb') as f:
            weights = pickle.load(f)
        for i, (which, target) in enumerate((('Q', False), ('pi', False), ('Q', True), ('pi', True))):
            self.set_flat(which, np.concatenate([np.asarray(v, np.float32).reshape(-1) for v in weights[i]]), target)
        self.o_stats.load_state_list(weights[4])
        self.g_stats.load_state_list(weights[5])

    # ------------------------------------------------------------------------------------------ resume
    def _unique_buffers(self):
        """The distinct ReplayBuffer objects behind self.buffer (Arm8: buffers 6.. alias 5, ddpg.py:107-110)."""
        seen, out = set(), []
        for i, b in enumerate(self.buffer if isinstance(self.buffer, (list, tuple)) else [self.buffer]):
            if id(b) not in seen:
                seen.add(id(b))
                out.append((i, b))
        return out

    def _gather_adam_state(self):
        """Owner mode of the tile exchange (cur_xchg_ctx mode 1) keeps the Adam moments of an element only on the rank
        that reduces it: assemble the full vectors on every rank (COLLECTIVE - every rank saves its own checkpoint,
        train.py of this package; also needed before switching to another update path)."""
        x = getattr(self, '_xchg', None)
        if x is None or x.mode not in (1, 2):
            return
        owner = np.empty(int(self.net.arena), np.int32)
        _lib.check(_lib.load().cur_ddpg_rows_owner_map(C.byref(self.net.desc), self._graph_rows, x.world,
                                                       owner.ctypes.data), 'cur_ddpg_rows_owner_map')
        mine = torch.from_numpy((owner == x.rank).astype(np.float32)).to(self.device)
        for t in (self._adam_m, self._adam_v):
            t.mul_(mine)
            allreduce_sum_(t, self.comm)        # x + 0 + ... + 0 is exact

    def save_checkpoint(self, path, buffers=True, numpy_rng=True):
        """Everything a run needs to continue bit for bit: parameters, Adam moments and step counters, normaliser
        accumulators, the Philox stream positions and (optionally) the replay buffers and the host np.random state.
        The reference can only save weights + normaliser statistics (ddpg.py:481-497, SURVEY 8f row 3): its Adam
        state, replay data and RNG position are lost on restart.  One torch.save file, tensors on the host."""
        if self._own():
            raise ValueError("save_checkpoint does not cover worker_buffers='own' (per-worker buffers and streams)")
        self._gather_adam_state()
        cpu = lambda t: t.detach().cpu().clone()
        st = dict(format=1, arena=int(self.net.arena), net=self._net_signature(), theta_main=cpu(self.theta_main), theta_target=cpu(self.theta_target),
                  adam_m=cpu(self._adam_m), adam_v=cpu(self._adam_v), adam_t=(int(self.Q_adam.t), int(self.pi_adam.t)),
                  step=int(self._step.item()), n_updates=int(self._n_updates),
                  sampler=dict(calls=int(self.sample_transitions.calls), seed=int(self.sample_transitions.seed)),
                  norm={k: dict(running=cpu(n._running), partial=cpu(n._partial), mean=cpu(n.mean), std=cpu(n.std))
                        for k, n in (('o', self.o_stats), ('g', self.g_stats))})
        if numpy_rng:
            st['numpy_rng'] = np.random.get_state()
        if buffers:
            st['buffers'] = []
            for i, b in self._unique_buffers():
                L, n = b.layout, b.current_size
                st['buffers'].append(dict(
                    index=i, current_size=n, n_transitions_stored=b.n_transitions_stored, layout=bytes(L),
                    hot=cpu(b.storage[:n * L.T * L.trans_stride]),
                    cold=None if b.cold is None else cpu(b.cold[:n * L.T * L.cold_stride])))
        torch.save(st, path)

    def _net_signature(self):
        """What has to agree between a checkpoint and the agent it is loaded into (a hidden-64 net zero-padded to the
        kernels' width has the arena size of a hidden-256 one)."""
        n = self.net
        return (bool(n.modular), int(n.dimo), int(n.dimg), int(n.dimu), int(n.dimtd), int(n.hidden), int(n.kernel_hidden),
                int(n.layers))

    def load_checkpoint(self, path):
        """Inverse of save_checkpoint on an agent built with the same arguments (checked: arena size, buffer layouts)."""
        if self._own():
            raise ValueError("load_checkpoint does not cover worker_buffers='own' (per-worker buffers and streams)")
        st = torch.load(path, map_location='cpu', weights_only=False)
        if st.get('format') != 1 or st['arena'] != int(self.net.arena) or st.get('net', self._net_signature()) != \
                self._net_signature():
            raise ValueError('checkpoint %s does not fit this agent (arena %s vs %d, network %s vs %s)' % (
                path, st.get('arena'), self.net.arena, st.get('net'), self._net_signature()))
        if getattr(self, '_peer', None) is not None and st['step'] < int(self._step.item()):
            # the peer-memory exchange counts updates in its NVLink flags (csrc/p2p.cu): they cannot run backwards
            raise ValueError('load the checkpoint into a freshly built agent when the peer-memory exchange is active')
        if getattr(self, '_xchg', None) is not None:
            self._xchg.reset()            # (collective) the update numbers travelling with the tiles start over
        for dst, key in ((self.theta_main, 'theta_main'), (self.theta_target, 'theta_target'),
                         (self._adam_m, 'adam_m'), (self._adam_v, 'adam_v')):
            dst.copy_(st[key].to(self.device))
        self.Q_adam.t, self.pi_adam.t = st['adam_t']
        self._step.fill_(st['step'])
        self._n_updates = st['n_updates']
        self.sample_transitions.calls = st['sampler']['calls']
        self.sample_transitions.seed = st['sampler']['seed']
        for k, n in (('o', self.o_stats), ('g', self.g_stats)):
            for dst, key in ((n._running, 'running'), (n._partial, 'partial'), (n.mean, 'mean'), (n.std, 'std')):
                dst.copy_(st['norm'][k][key].to(self.device))
        if 'buffers' in st:
            mine = dict(self._unique_buffers())
            for rec in st['buffers']:
                b = mine.get(rec['index'])
                if b is None or bytes(b.layout) != rec['layout'] or rec['current_size'] > b.size:
                    raise ValueError('checkpoint buffer %d does not fit this agent' % rec['index'])
                with b.lock:
                    b.storage[:rec['hot'].numel()].copy_(rec['hot'].to(self.device))
                    if rec['cold'] is not None:
                        b.cold[:rec['cold'].numel()].copy_(rec['cold'].to(self.device))
                    b.current_size = rec['current_size']
                    b.n_transitions_stored = rec['n_transitions_stored']
        if 'numpy_rng' in st:
            np.random.set_state(st['numpy_rng'])
        self._mark_weights_changed()
        self._graph_sig = None            # buffer sizes changed: the graph's control block is rewritten on the next train()

    def __getstate__(self):
        """Policies can be pickled for playing; training state (Adam, buffers) is not saved (ddpg.py:511-521)."""
        excluded_subnames = ['_tf', '_op', '_vars', '_adam', 'buffer', 'sess', '_stats', 'main', 'target', 'lock',
                             'env', 'sample_transitions', 'stage_shapes', 'create_actor_critic']      # ddpg.py:514-516
        device_state = ('net', 'device', 'comm', 'grads', 'kwargs')     # this implementation's own (exact names + _private)
        state = {k: v for k, v in self.__dict__.items() if not k.startswith('_') and k not in device_state and
                 all([subname not in k for subname in excluded_subnames])}
        state['weights'] = [self.get_flat('Q'), self.get_flat('pi'), self.get_flat('Q', True), self.get_flat('pi', True),
                            self.o_stats.state_list(), self.g_stats.state_list()]
        return state

    def __setstate__(self, state):
        if 'sample_transitions' not in state:
            state['sample_transitions'] = None      # not needed for playing the policy
        weights = state.pop('weights')
        extra = {k: state.pop(k) for k in list(state.keys())
                 if k not in DDPG.__init__.__wrapped__.__code__.co_varnames and
                 k not in ('structure', 'her_rng', 'seed', 'noise_seed')}
        self.__init__(**state)
        self.__dict__.update(extra)
        for i, (which, target) in enumerate((('Q', False), ('pi', False), ('Q', True), ('pi', True))):
            self.set_flat(which, weights[i], target)
        self.o_stats.load_state_list(weights[4])
        self.g_stats.load_state_list(weights[5])
