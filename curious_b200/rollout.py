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

Pinned against the reference class itself, compiled from its unmodified source and run on the same environments and
np.random stream (tests/test_reference_live.py::test_rollout_worker_equals_reference_class).
"""
import pickle
from collections import deque

import numpy as np

from .parallel import rank as _rank, world as _world
from .queues import CompetenceTracker
from .util import store_args


class RolloutWorker(object):
    @store_args
    def __init__(self, make_env, policy, dims, logger, T, rollout_batch_size=1, exploit=False, use_target_net=False,
                 compute_Q=False, noise_eps=0, random_eps=0, history_len=100, render=False, structure='curious',
                 task_selection='random', goal_selection='random', queue_length=500, eval=False, unique_task=None,
                 temperature=None, **kwargs):
        """Arguments as in reference rollout.py:19-41."""
        if goal_selection == 'active':
            raise ValueError("goal_selection='active' (SAGG-RIAC) is unsupported, as in the reference readme")
        assert T > 0
        self.comm = kwargs.get('comm')
        self.rank, self.nb_cpu = _rank(self.comm), _world(self.comm)[1]
        self.envs = [make_env() for _ in range(rollout_batch_size)]
        core = self.envs[0].unwrapped
        self.nb_tasks = core.nb_tasks
        self.modular = structure in ('curious', 'task_experts')
        self.info_keys = [k[len('info_'):] for k in dims if k.startswith('info_')]
        self.n_episodes = 0
        self.nb_goals_per_rollout = self.nb_cpu * rollout_batch_size
        B = rollout_batch_size
        self.g = np.zeros((B, dims['g']), np.float32)
        self.initial_o = np.zeros((B, dims['o']), np.float32)
        self.initial_ag = np.zeros((B, dims['ag']), np.float32)
        self.task_descr = np.zeros((B, self.nb_tasks), np.float32)
        self.C, self.CP = np.zeros(self.nb_tasks), np.zeros(self.nb_tasks)
        self.success_history, self.reward_history, self.Q_history = (deque(maxlen=history_len) for _ in range(3))
        self.task_history, self.goal_history = deque(), deque()
        if self.modular:
            self.tasks_ag_id, self.tasks_g_id = core.tasks_ag_id, core.tasks_g_id
            self.tracker = CompetenceTracker(self.nb_tasks, queue_length=queue_length, task_selection=task_selection,
                                             structure=structure, unique_task=unique_task, eval=eval, comm=self.comm)
            self.competence_computers = self.tracker.competence_computers
            self.p = self.tracker.p.copy()
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

    def _draw_assignment(self, i):
        """Rank 0 picks (task, goal) for rollout slot i of every rank, in the reference's draw order (rollout.py:118-140):
        all tasks in one np.random.choice(p=self.p, size=nb_cpu), then one uniform goal in [-1, 1]^len(g_id) per rank."""
        core = self.envs[i].unwrapped
        if self.modular:
            tasks = np.random.choice(range(self.nb_tasks), p=self.p, size=self.nb_cpu).tolist()
            goals = [np.random.uniform(-1, 1, len(self.tasks_g_id[tasks[cpu]])) for cpu in range(self.nb_cpu)]
        else:
            tasks = [0] * self.nb_cpu
            goals = [np.random.uniform(-1, 1, self.dims['g']) for _ in range(self.nb_cpu)]
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
        if self.modular:
            obs = env.unwrapped.reset_task_goal(goal=goal, task=task, directly=False, eval=self.eval)
            self.task_descr[i] = obs['mask']
        else:
            obs = env.unwrapped.reset_task_goal(goal=goal)
        self.initial_o[i], self.initial_ag[i], self.g[i] = obs['observation'], obs['achieved_goal'], obs['desired_goal']

    def reset_all_rollouts(self):
        self.goals = [None] * self.nb_goals_per_rollout
        self.tasks = [None] * self.nb_goals_per_rollout
        for i in range(self.rollout_batch_size):
            self.reset_rollout(i)

    # ---------------------------------------------------------------------------------------------- acting
    def _act(self, o, ag):
        """One device forward for all environments of the rank -> (u [B, dimu], Q [B, 1] or None)."""
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
        Returns (episode {key: [B, T(+1), dim]}, CP, n_episodes)."""
        if self.eval:
            self.exploit = True
        elif self.modular:
            self.exploit = bool(np.random.random() < 0.1)       # competence is measured on noise-free rollouts
        if self.modular and self.exploit and (self.eval or self.structure == 'curious'):
            self.p = np.ones(self.nb_tasks) / self.nb_tasks
        self.reset_all_rollouts()
        B, T, d = self.rollout_batch_size, self.T, self.dims
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
        self.success_history.append(float(success.mean()))
        self.reward_history.append(env_reward.copy())
        if self.compute_Q:
            self.Q_history.append(np.mean(Qs))
        self.n_episodes += B * self.nb_cpu
        if self.modular:
            self._update_competence(success)
        return ep, self.CP, self.n_episodes

    def _update_competence(self, success):
        """rollout.py:316-404: only noise-free rollouts count; rank 0 owns the queues, everybody gets CP and p back."""
        if self.exploit:
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

    # ------------------------------------------------------------------------------------------ bookkeeping
    def clear_history(self):
        for h in (self.success_history, self.reward_history, self.Q_history):
            h.clear()

    def clear_competence_queue(self):
        self.tracker.clear_competence_queue()

    def current_success_rate(self):
        return np.mean(self.success_history)

    def current_mean_Q(self):
        return np.mean(self.Q_history)

    def get_CP(self):
        return self.tracker.get_CP()

    def get_C(self):
        return self.tracker.get_C()

    def seed(self, seed):
        for idx, env in enumerate(self.envs):
            env.seed(seed + 1000 * idx)

    def save_policy(self, path):
        with open(path, 'wb') as f:
            pickle.dump(self.policy, f)
        if hasattr(self.policy, 'save_weights'):
            self.policy.save_weights(path)

    # resume support (beyond the reference): what generate_rollouts carries from one call to the next
    def state(self):
        st = dict(n_episodes=self.n_episodes, count=self.count, p=np.array(self.p, np.float64) if self.modular else None,
                  CP=np.array(self.CP, np.float64), C=np.array(self.C, np.float64), exploit=self.exploit,
                  histories=[list(h) for h in (self.success_history, self.reward_history, self.Q_history,
                                               self.task_history, self.goal_history)],
                  initial_o=self.initial_o.copy(), initial_ag=self.initial_ag.copy(), g=self.g.copy(),
                  tracker=self.tracker.state() if self.modular else None,
                  env_rng=[e.unwrapped.rng.get_state() if hasattr(getattr(e.unwrapped, 'rng', None), 'get_state') else None
                           for e in self.envs])
        return st

    def load_state(self, st):
        self.n_episodes, self.count, self.exploit = st['n_episodes'], st['count'], st['exploit']
        self.CP, self.C = st['CP'].copy(), st['C'].copy()
        for h, saved in zip((self.success_history, self.reward_history, self.Q_history, self.task_history,
                             self.goal_history), st['histories']):
            h.clear()
            h.extend(saved)
        self.initial_o[:], self.initial_ag[:], self.g[:] = st['initial_o'], st['initial_ag'], st['g']
        if self.modular:
            self.p = st['p'].copy()
            self.tracker.load_state(st['tracker'])
        for e, rng in zip(self.envs, st['env_rng']):
            if rng is not None:
                e.unwrapped.rng.set_state(rng)

    def save_goal_task_history(self, path):
        """No-op, like the reference's (rollout.py:437-449: body commented out); kept for the train loop's call."""

    def _prefixed(self, items, prefix):
        return [((prefix.rstrip('/') + '/' + k) if prefix else k, v) for k, v in items]

    def logs(self, prefix='worker'):
        items = [('success_rate', np.mean(self.success_history)), ('avg_reward', np.mean(self.reward_history))]
        if self.compute_Q:
            items.append(('mean_Q', np.mean(self.Q_history)))
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
