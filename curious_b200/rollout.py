"""RolloutWorker - the caller of DDPG.get_actions and the producer of DDPG.store_episode's input.

Same constructor arguments, public methods and episode dictionary as reference baselines/her/rollout.py:13-491, for
environments with the gym_flowers attribute contract (curious_b200.envs.ModularPointEnv here: gym_flowers / MuJoCo
are absent).  Built around fixed batch-major arrays instead of per-step Python lists:

  * all `rollout_batch_size` environments of the rank are stepped on host cores, with ONE batched
    `policy.get_actions` device forward per timestep (north_star: "MuJoCo stepping stays on host cores, with
    batched get_actions on device"),
  * the episode is written straight into [B, T(+1), dim] arrays (what store_episode wants; the reference builds
    time-major lists and transposes them, util.py:174-184),
  * task / goal draws for every rank are made on rank 0 in one go and scattered (rollout.py:118-140), the LP block
    (rollout.py:316-404) lives in curious_b200.queues.CompetenceTracker; MPI collectives become torch.distributed
    object collectives,
  * SAGG-RIAC goal selection (`goal_selection='active'`) is not supported (readme.md:19 marks it unsupported).

Virtual workers (`workers=k`, `streams=` a workers.WorkerStreams; one rank): the worker holds the environments of the k
reference workers the rank hosts, worker j standing for reference rank j with `rollout_batch_size` environments
[j * B, (j + 1) * B).  Each worker keeps what a reference rank keeps - its exploit flag, p and success / reward / Q
histories - and draws everything a rank draws from its own stream (streams.rng(j)): the exploit draw, and through
`policy.get_actions_workers` the exploration noise of its rows, all k workers acting in one launch per step.  Worker 0
draws the task / goal assignment of every worker (as rank 0 does for every rank), the competence queues take the
exploit rollouts of all workers in worker order, and generate_rollouts returns the worker-major episode batch of
DDPG.store_episode with worker_buffers='own'.  logs() and current_success_rate() / current_mean_Q() are the mean over
workers (mpi_average over the reference's ranks).  One deviation: a NaN observation restarts every worker's rollouts,
where a reference rank restarts only its own.

Pinned against the reference class itself, compiled from its unmodified source and run on the same environments and
np.random stream (tests/test_reference_live.py::test_rollout_worker_equals_reference_class).
"""
import pickle
from collections import deque

import numpy as np

from .parallel import rank as _rank, rank_seed, world as _world
from .queues import CompetenceTracker
from .util import store_args


class RolloutWorker(object):
    @store_args
    def __init__(self, make_env, policy, dims, logger, T, rollout_batch_size=1, exploit=False, use_target_net=False,
                 compute_Q=False, noise_eps=0, random_eps=0, history_len=100, render=False, structure='curious',
                 task_selection='random', goal_selection='random', queue_length=500, eval=False, unique_task=None,
                 temperature=None, workers=1, streams=None, **kwargs):
        """Arguments as in reference rollout.py:19-41; `workers` / `streams`: virtual workers (module docstring)."""
        if goal_selection == 'active':
            raise ValueError("goal_selection='active' (SAGG-RIAC) is unsupported, as in the reference readme")
        assert T > 0
        self.comm = kwargs.get('comm')
        self.rank, self.nb_cpu = _rank(self.comm), _world(self.comm)[1]
        if streams is not None or workers != 1:
            if streams is None or len(streams) != workers:
                raise ValueError('%d virtual workers need a WorkerStreams of %d streams' % (workers, workers))
            if self.nb_cpu > 1:
                raise ValueError('virtual workers run on one rank')
            if structure == 'task_experts':
                raise ValueError("virtual workers do not take structure='task_experts'")
            self.nb_cpu = workers                           # the reference ranks the workers stand for
        self.envs = [make_env() for _ in range(rollout_batch_size * workers)]
        core = self.envs[0].unwrapped
        self.nb_tasks = core.nb_tasks
        self.modular = structure in ('curious', 'task_experts')
        self.info_keys = [k[len('info_'):] for k in dims if k.startswith('info_')]
        self.n_episodes = 0
        self.nb_goals_per_rollout = self.nb_cpu * rollout_batch_size
        B = rollout_batch_size * workers
        self.g = np.zeros((B, dims['g']), np.float32)
        self.initial_o = np.zeros((B, dims['o']), np.float32)
        self.initial_ag = np.zeros((B, dims['ag']), np.float32)
        self.task_descr = np.zeros((B, self.nb_tasks), np.float32)
        self.C, self.CP = np.zeros(self.nb_tasks), np.zeros(self.nb_tasks)
        if self.streams is None:
            self.success_history, self.reward_history, self.Q_history = (deque(maxlen=history_len) for _ in range(3))
        else:
            # per worker: (success, reward, Q) histories, exploit flag, p (self.p is worker 0's, which draws the tasks)
            self.worker_histories = [tuple(deque(maxlen=history_len) for _ in range(3)) for _ in range(workers)]
            self.worker_exploit = [exploit] * workers
        self.task_history, self.goal_history = deque(), deque()
        if self.modular:
            self.tasks_ag_id, self.tasks_g_id = core.tasks_ag_id, core.tasks_g_id
            self.tracker = CompetenceTracker(self.nb_tasks, queue_length=queue_length, task_selection=task_selection,
                                             structure=structure, unique_task=unique_task, eval=eval, comm=self.comm)
            self.competence_computers = self.tracker.competence_computers
            self.p = self.tracker.p.copy()
            if self.streams is not None:
                self.worker_p = [self.p] + [self.tracker.p.copy() for _ in range(1, workers)]
        else:
            for env in self.envs:
                env.unwrapped.set_flat_env()
        self.stochastic_reset = False
        self.count = -1
        self.reset_all_rollouts()

    # ---------------------------------------------------------------------------------------- tasks and goals
    def _from_rank0(self, make):
        """`make()` runs on rank 0 and returns one entry per rank; every rank gets its own (scatter)."""
        if self.nb_cpu == 1:
            return make()[0]
        import torch.distributed as dist
        group = _world(self.comm)[0]
        box = [make() if self.rank == 0 else None]
        dist.broadcast_object_list(box, src=0 if group is None else dist.get_global_rank(group, 0), group=group)
        return box[0][self.rank]

    def _draw_assignment(self, i, rng=np.random):
        """Rank 0 picks (task, goal) for rollout slot i of every rank, in the reference's draw order (rollout.py:118-140):
        all tasks in one np.random.choice(p=self.p, size=nb_cpu), then one uniform goal in [-1, 1]^len(g_id) per rank.
        `rng`: rank 0's stream (virtual workers: worker 0's)."""
        core = self.envs[i].unwrapped
        if self.modular:
            tasks = rng.choice(range(self.nb_tasks), p=self.p, size=self.nb_cpu).tolist()
            goals = [rng.uniform(-1, 1, len(self.tasks_g_id[tasks[cpu]])) for cpu in range(self.nb_cpu)]
        else:
            tasks = [0] * self.nb_cpu
            goals = [rng.uniform(-1, 1, self.dims['g']) for _ in range(self.nb_cpu)]
        for cpu in range(self.nb_cpu):
            slot = cpu * self.rollout_batch_size + i
            if self.modular:
                self.tasks[slot] = tasks[cpu]
                self.goals[slot] = core._compute_goal(goals[cpu], tasks[cpu], eval=self.eval)[0][self.tasks_g_id[tasks[cpu]]]
            else:
                self.goals[slot] = core._compute_goal(goals[cpu], 0)[0]
        return list(zip(tasks, goals))

    def reset_rollout(self, i):
        """Reset environment i and give it its next task and goal (rollout.py:104-165)."""
        env = self.envs[i]
        if self.eval or not self.stochastic_reset or np.random.rand() < 0.3 or self.exploit:
            env.reset()
        task, goal = self._from_rank0(lambda: self._draw_assignment(i))
        self.count += 1
        self._start(i, task, goal)

    def _start(self, i, task, goal):
        env = self.envs[i]
        if self.modular:
            obs = env.unwrapped.reset_task_goal(goal=goal, task=task, directly=False, eval=self.eval)
            self.task_descr[i] = obs['mask']
        else:
            obs = env.unwrapped.reset_task_goal(goal=goal)
        self.initial_o[i], self.initial_ag[i], self.g[i] = obs['observation'], obs['achieved_goal'], obs['desired_goal']

    def _reset_rollout_workers(self, i):
        """reset_rollout(i) of every virtual worker: worker j resets its environment i as rank j does, worker 0 draws
        the assignment of slot i for all of them."""
        B = self.rollout_batch_size
        for j in range(self.workers):
            if (self.eval or not self.stochastic_reset or self.streams.rng(j).rand() < 0.3 or
                    self.worker_exploit[j]):
                self.envs[j * B + i].reset()
        assignment = self._draw_assignment(i, self.streams.rng(0))
        self.count += 1
        for j, (task, goal) in enumerate(assignment):
            self._start(j * B + i, task, goal)

    def reset_all_rollouts(self):
        self.goals = [None] * self.nb_goals_per_rollout
        self.tasks = [None] * self.nb_goals_per_rollout
        for i in range(self.rollout_batch_size):
            if self.streams is None:
                self.reset_rollout(i)
            else:
                self._reset_rollout_workers(i)

    # ---------------------------------------------------------------------------------------------- acting
    def _act(self, o, ag):
        """One device forward for all environments of the rank -> (u [B, dimu], Q [B, 1] or None)."""
        if self.streams is not None:            # every virtual worker's rows in one launch, each with its own noise
            return self.policy.get_actions_workers(
                o, ag, self.g, task_descr=self.task_descr if self.modular else None,
                noise_eps=[0. if x else self.noise_eps for x in self.worker_exploit],
                random_eps=[0. if x else self.random_eps for x in self.worker_exploit], streams=self.streams,
                use_target_net=self.use_target_net, compute_Q=self.compute_Q)
        quiet = self.exploit
        kw = dict(compute_Q=self.compute_Q, noise_eps=0. if quiet else self.noise_eps,
                  random_eps=0. if quiet else self.random_eps, use_target_net=self.use_target_net)
        if self.structure == 'task_experts' and self.eval:
            # evaluation of experts: the expert of the demanded task acts (rollout.py:211-223)
            experts = self._expert_router()
            if experts is not None:             # one routed launch, bit for bit the loop below
                out = experts.get_actions(o, ag, self.g, self.task_descr, **kw)
                return (out[0], out[1]) if self.compute_Q else (out, None)
            u = np.zeros((len(o), self.dims['u']))
            q = np.zeros((len(o), 1))
            for i in range(len(o)):
                expert = self.policy[int(np.argmax(self.task_descr[i]))]
                out = expert.get_actions(o[i:i + 1], ag[i:i + 1], self.g[i:i + 1], task_descr=self.task_descr[i:i + 1], **kw)
                if self.compute_Q:
                    u[i], q[i, 0] = out[0], np.asarray(out[1]).reshape(-1)[0]
                else:
                    u[i] = out
            return u, (q if self.compute_Q else None)
        out = self.policy.get_actions(o, ag, self.g, task_descr=self.task_descr if self.modular else None, **kw)
        u, q = (out if self.compute_Q else (out, None))
        return np.asarray(u).reshape(len(o), -1), q

    def _expert_router(self):
        """experts.TaskExperts over the policy list when it is made of DDPG agents of one shape, else None (the loop)."""
        if getattr(self, '_router', (None,))[0] is not self.policy:
            from .experts import TaskExperts
            self._router = (self.policy, TaskExperts.router(self.policy))
        return self._router[1]

    def generate_rollouts(self):
        """`rollout_batch_size` episodes of T steps with the current policy (rollout.py:178-406).
        Returns (episode {key: [B, T(+1), dim]}, CP, n_episodes); virtual workers: B = workers * rollout_batch_size,
        worker-major."""
        if self.streams is not None:
            self._draw_exploit_workers()
        else:
            if self.eval:
                self.exploit = True
            elif self.modular:
                self.exploit = bool(np.random.random() < 0.1)       # competence is measured on noise-free rollouts
            if self.modular and self.exploit and (self.eval or self.structure == 'curious'):
                self.p = np.ones(self.nb_tasks) / self.nb_tasks
        self.reset_all_rollouts()
        B, T, d = len(self.envs), self.T, self.dims
        # observations, achieved goals, goals and task descriptors are float32 like the reference's working arrays
        # (rollout.py:50-52,194-197); actions keep the dtype the policy returns
        ep = {'o': np.zeros((B, T + 1, d['o']), np.float32), 'ag': np.zeros((B, T + 1, d['ag']), np.float32), 'u': None,
              'g': np.zeros((B, T, d['g']), np.float32)}
        if self.modular:
            ep['task_descr'] = np.zeros((B, T, self.nb_tasks), np.float32)
            ep['change'] = np.zeros((B, T, d['ag']), bool)
        for key in self.info_keys:
            ep['info_' + key] = np.zeros((B, T, d['info_' + key]), np.float32)
        ep['o'][:, 0], ep['ag'][:, 0] = self.initial_o, self.initial_ag
        success = np.zeros(B)
        env_reward = np.zeros(B)
        Qs = []
        for t in range(T):
            u, q = self._act(ep['o'][:, t].copy(), ep['ag'][:, t].copy())
            if q is not None:
                Qs.append(q)
            if ep['u'] is None:
                ep['u'] = np.zeros((B, T, d['u']), np.asarray(u).dtype)
            ep['u'][:, t], ep['g'][:, t] = u, self.g
            if self.modular:
                ep['task_descr'][:, t] = self.task_descr
            for i, env in enumerate(self.envs):
                obs, env_reward[i], _, info = env.step(u[i])        # the reward is recomputed by the HER sampler
                success[i] = info.get('is_success', 0.0)
                ep['o'][i, t + 1], ep['ag'][i, t + 1] = obs['observation'], obs['achieved_goal']
                self.g[i] = obs['desired_goal']
                for key in self.info_keys:
                    ep['info_' + key][i, t] = info[key]
            if np.isnan(ep['o'][:, t + 1]).any():
                self.reset_all_rollouts()
                return self.generate_rollouts()
            if self.modular:                                        # did the outcome move since the start? (routing)
                ep['change'][:, t] = np.abs(ep['ag'][:, 0] - ep['ag'][:, t + 1]) > 1e-3
        self.initial_o[:] = ep['o'][:, T]
        if self.streams is None:
            self.success_history.append(float(success.mean()))
            self.reward_history.append(env_reward.copy())
            if self.compute_Q:
                self.Q_history.append(np.mean(Qs))
        else:
            rb = self.rollout_batch_size
            for j, (succ_h, reward_h, q_h) in enumerate(self.worker_histories):
                rows = slice(j * rb, (j + 1) * rb)
                succ_h.append(float(success[rows].mean()))
                reward_h.append(env_reward[rows].copy())
                if self.compute_Q:
                    q_h.append(np.mean([q[rows] for q in Qs]))
        self.n_episodes += self.rollout_batch_size * self.nb_cpu
        if self.modular:
            self._update_competence(success)
        return ep, self.CP, self.n_episodes

    def _draw_exploit_workers(self):
        """The start of generate_rollouts on every virtual worker: its exploit draw from its own stream, and p uniform
        on a worker that exploits (rollout.py:180-190)."""
        for j in range(self.workers):
            if self.eval:
                self.worker_exploit[j] = True
            elif self.modular:
                self.worker_exploit[j] = bool(self.streams.rng(j).random() < 0.1)
            if self.modular and self.worker_exploit[j] and (self.eval or self.structure == 'curious'):
                self.worker_p[j] = np.ones(self.nb_tasks) / self.nb_tasks
        if self.modular:
            self.p = self.worker_p[0]

    def _update_competence(self, success):
        """rollout.py:316-404: only noise-free rollouts count; rank 0 owns the queues, everybody gets CP and p back.
        Virtual workers: the exploit rollouts of every worker, in worker order (the reference's gather in rank order)."""
        if self.streams is not None:
            rb, tasks, succ = self.rollout_batch_size, [], []
            for j in range(self.workers):
                if self.worker_exploit[j]:
                    tasks += [int(env.unwrapped.task) for env in self.envs[j * rb:(j + 1) * rb]]
                    succ += success[j * rb:(j + 1) * rb].tolist()
        elif self.exploit:
            tasks, succ = [int(env.unwrapped.task) for env in self.envs], success.tolist()
        else:
            tasks, succ = [], []
        if self.rank == 0:
            self.task_history.extend(t for t in self.tasks if t is not None)
            self.goal_history.extend(g for g in self.goals if g is not None)
        self.CP, p = self.tracker.update(tasks, succ)
        self.C = self.tracker.C
        if not self.eval:
            self.p = np.array(p, np.float64)
            if self.streams is not None:                            # p is broadcast to every rank
                self.worker_p = [self.p] + [np.array(p, np.float64) for _ in range(1, self.workers)]

    # ------------------------------------------------------------------------------------------ bookkeeping
    def _own_histories(self):
        """(success, reward, Q) histories of the rank, one triple per virtual worker."""
        if self.streams is None:
            return [(self.success_history, self.reward_history, self.Q_history)]
        return self.worker_histories

    def _mean_over_workers(self, which):
        """Virtual workers: mpi_average over the ranks they stand for of each one's mean history `which` (summed in
        worker order)."""
        total = 0.0
        for hs in self.worker_histories:
            total += float(np.mean(hs[which]))
        return total / self.workers

    def clear_history(self):
        for hs in self._own_histories():
            for h in hs:
                h.clear()

    def clear_competence_queue(self):
        self.tracker.clear_competence_queue()

    def current_success_rate(self):
        return np.mean(self.success_history) if self.streams is None else self._mean_over_workers(0)

    def current_mean_Q(self):
        return np.mean(self.Q_history) if self.streams is None else self._mean_over_workers(2)

    def get_CP(self):
        return self.tracker.get_CP()

    def get_C(self):
        return self.tracker.get_C()

    def seed(self, seed):
        """Environment idx of the rank: seed + 1000 * idx (train.py:332,335).  Virtual worker j seeds its environments
        as rank j does, from rank_seed(seed, j)."""
        rb = self.rollout_batch_size
        for idx, env in enumerate(self.envs):
            if self.streams is None:
                env.seed(seed + 1000 * idx)
            else:
                env.seed(rank_seed(seed, idx // rb) + 1000 * (idx % rb))

    def save_policy(self, path):
        with open(path, 'wb') as f:
            pickle.dump(self.policy, f)
        if hasattr(self.policy, 'save_weights'):
            self.policy.save_weights(path)

    # resume support (beyond the reference): what generate_rollouts carries from one call to the next
    def state(self):
        own = (self.success_history, self.reward_history, self.Q_history) if self.streams is None else ((), (), ())
        st = dict(n_episodes=self.n_episodes, count=self.count, p=np.array(self.p, np.float64) if self.modular else None,
                  CP=np.array(self.CP, np.float64), C=np.array(self.C, np.float64), exploit=self.exploit,
                  histories=[list(h) for h in own + (self.task_history, self.goal_history)],
                  initial_o=self.initial_o.copy(), initial_ag=self.initial_ag.copy(), g=self.g.copy(),
                  tracker=self.tracker.state() if self.modular else None,
                  env_rng=[e.unwrapped.rng.get_state() if hasattr(getattr(e.unwrapped, 'rng', None), 'get_state') else None
                           for e in self.envs])
        if self.streams is not None:
            st['workers'] = dict(exploit=list(self.worker_exploit),
                                 p=[np.array(p, np.float64) for p in self.worker_p] if self.modular else None,
                                 histories=[[list(h) for h in hs] for hs in self.worker_histories])
        return st

    def load_state(self, st):
        self.n_episodes, self.count, self.exploit = st['n_episodes'], st['count'], st['exploit']
        self.CP, self.C = st['CP'].copy(), st['C'].copy()
        own = ((self.success_history, self.reward_history, self.Q_history) if self.streams is None else
               (deque(), deque(), deque()))
        for h, saved in zip(own + (self.task_history, self.goal_history), st['histories']):
            h.clear()
            h.extend(saved)
        self.initial_o[:], self.initial_ag[:], self.g[:] = st['initial_o'], st['initial_ag'], st['g']
        if self.modular:
            self.p = st['p'].copy()
            self.tracker.load_state(st['tracker'])
        for e, rng in zip(self.envs, st['env_rng']):
            if rng is not None:
                e.unwrapped.rng.set_state(rng)
        if self.streams is not None:
            w = st['workers']
            self.worker_exploit = list(w['exploit'])
            for hs, saved in zip(self.worker_histories, w['histories']):
                for h, s in zip(hs, saved):
                    h.clear()
                    h.extend(s)
            if self.modular:
                self.worker_p = [p.copy() for p in w['p']]
                self.p = self.worker_p[0]

    def save_goal_task_history(self, path):
        """No-op, like the reference's (rollout.py:437-449: body commented out); kept for the train loop's call."""

    def _prefixed(self, items, prefix):
        return [((prefix.rstrip('/') + '/' + k) if prefix else k, v) for k, v in items]

    def logs(self, prefix='worker'):
        """Virtual workers: the mean over workers of each value, what train.py logs over ranks (mpi_average)."""
        if self.streams is None:
            items = [('success_rate', np.mean(self.success_history)), ('avg_reward', np.mean(self.reward_history))]
            if self.compute_Q:
                items.append(('mean_Q', np.mean(self.Q_history)))
        else:
            items = [('success_rate', self._mean_over_workers(0)), ('avg_reward', self._mean_over_workers(1))]
            if self.compute_Q:
                items.append(('mean_Q', self._mean_over_workers(2)))
        items.append(('episode', self.n_episodes))
        return self._prefixed(items, prefix)

    def additional_logs(self, prefix='worker'):
        items = []
        if self.modular:
            C, CP = self.get_C(), self.get_CP()
            for i in range(self.nb_tasks):
                items.append(('C_task%d' % i, '%.3g' % C[i]))
                if not self.eval:
                    share = np.mean(np.array(self.task_history)[-100:] == i) if len(self.task_history) else 0.0
                    items += [('CP_task%d' % i, '%.3g' % CP[i]), ('%%_task%d' % i, '%.3g' % share),
                              ('p_task%d' % i, '%.3g' % self.p[i])]
        return self._prefixed(items, prefix)
