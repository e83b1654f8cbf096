"""Driver loop: reference baselines/her/experiment/train.py:48-170 and the pieces of config.py it needs
(config.py:20-90 defaults, :110-170 configure_her, :184-214 configure_buffer, :219-253 configure_ddpg, :257-275
configure_dims) for environments with the gym_flowers attribute contract (SURVEY 8f row 4).

    exp = make_experiment(nb_tasks=4, structure='curious', task_selection='active_competence_progress',
                          task_replay='replay_task_cp_buffer')
    history = train(**exp, n_epochs=10)

Process launch (`mpirun -np N` -> `python -m torch.distributed.run --nproc-per-node N`) is the caller's business
(INTEGRATION.md).  With `logdir=` the loop writes the reference's run records (progress.csv, params.json,
policy_latest / policy_best / policy_<epoch>.pkl, train.py:53-55,171-206,264-266 - see runlog.py) and, beyond the
reference, a resumable checkpoint per epoch (`checkpoint_interval`, DDPG.save_checkpoint).
"""
import os
import pickle
import time

import numpy as np

from . import her
from .ddpg import DDPG
from .envs import ModularPointEnv
from .replay_buffer import ReplayBuffer
from .rollout import RolloutWorker
from .parallel import assert_rank_streams_differ, bcast_object, rank as _rank, rank_seed, world as _world
from .runlog import RunLog, mpi_average

MULTI_TASK_PARAMS = {            # config.py:56-90
    'max_u': 1., 'layers': 3, 'hidden': 256, 'network_class': 'baselines.her.actor_critic:MultiTaskActorCritic',
    'Q_lr': 0.001, 'pi_lr': 0.001, 'buffer_size': int(1E6), 'polyak': 0.95, 'action_l2': 1.0, 'clip_obs': 200.,
    'scope': 'ddpg', 'relative_goals': False, 'n_cycles': 25, 'rollout_batch_size': 2, 'n_batches': 100,
    'batch_size': 256, 'n_test_rollouts': 5, 'test_with_polyak': False, 'random_eps': 0.3, 'noise_eps': 0.2,
    'her_replay_k': 4, 'norm_eps': 0.01, 'norm_clip': 5,
    'her_sampling_func': 'baselines.her.her:make_sample_multi_task_her_transitions', 'queue_length': 300, 'eps_task': 0.4,
}
FLAT_PARAMS = dict(MULTI_TASK_PARAMS, network_class='baselines.her.actor_critic:ActorCritic',
                   her_sampling_func='baselines.her.her:make_sample_her_transitions', queue_length=200)


def simple_goal_subtract(a, b):
    """config.py:177-179 (a module-level function, so that policies pickle)."""
    assert a.shape == b.shape
    return a - b


def configure_dims(env, structure):
    """config.py:257-275: dims from one reset + step of the environment."""
    env.reset()
    obs, _, _, info = env.step(env.action_space.sample())
    dims = {'o': obs['observation'].shape[0], 'u': env.action_space.shape[0], 'g': obs['desired_goal'].shape[0],
            'ag': obs['achieved_goal'].shape[0]}
    if structure != 'flat':
        dims['task_descr'] = env.unwrapped.nb_tasks
    for key, value in info.items():
        value = np.array(value)
        if value.ndim == 0:
            value = value.reshape(1)
        dims['info_{}'.format(key)] = value.shape[0]
    return dims


def configure_buffer(dims, T, sampler, buffer_size, structure, task_replay, nb_tasks, device=None):
    """config.py:184-214: one buffer, or one per module + buffer 0 for the *_buffer replay modes."""
    shapes = {key: (T if key != 'o' and key != 'ag' else T + 1, val) for key, val in dims.items()}
    if structure != 'flat':
        shapes['change'] = (T, dims['ag'])
    if structure != 'flat' and ('buffer' in task_replay or task_replay == 'hand_designed'):
        return [ReplayBuffer(shapes, buffer_size, T, sampler, device=device) for _ in range(nb_tasks + 1)]
    return ReplayBuffer(shapes, buffer_size, T, sampler, device=device)


def make_experiment(nb_tasks=4, n_controllable=None, structure='curious', task_selection='active_competence_progress',
                    goal_replay='her', task_replay='replay_task_cp_buffer', seed=0, device=None, normalize_obs=False,
                    make_env=None, policy_kwargs=None, workers_per_rank=1, **overrides):
    """config.prepare_params + configure_* + the RolloutWorker pair of train.py:268-337.  Returns the keyword
    arguments of train().  workers_per_rank=k > 1: the rank hosts k reference workers (worker j = reference rank j, one
    rank only): DDPG(workers_per_rank=k, worker_buffers='own') with k-worker exploration and evaluation RolloutWorkers on
    the policy's worker streams; the run parameters record num_cpu = k."""
    if workers_per_rank != 1:
        if structure == 'task_experts':
            raise ValueError("workers_per_rank > 1 does not take structure='task_experts'")
        if _world((policy_kwargs or {}).get('comm'))[1] > 1:
            raise ValueError('workers_per_rank > 1 runs on one rank')
    params = dict(FLAT_PARAMS if structure == 'flat' else MULTI_TASK_PARAMS)
    params.update(overrides)
    # train.py:241-243: every rank seeds everything with rank_seed = seed + 1000000 * rank (set_global_seeds: np.random
    # and random), so that ranks explore, draw tasks / goals / replay slots and sample replay differently; only the weight
    # initialisation keeps `seed` (rank 0's weights are broadcast anyway, ddpg.py:466)
    import random
    rs = rank_seed(seed, _rank((policy_kwargs or {}).get('comm')))
    np.random.seed(rs % (2 ** 32))
    random.seed(rs)
    if make_env is None:
        def make_env():
            return ModularPointEnv(nb_tasks, n_controllable)
    env = make_env()
    T = env._max_episode_steps
    gamma = 1. - 1. / T                                             # config.py:127
    dims = configure_dims(env, structure)
    ag_ids, g_ids = env.unwrapped.tasks_ag_id, env.unwrapped.tasks_g_id
    reward = env.unwrapped.reward_spec                              # config.py:158-159 as data (see reward.py)
    if structure == 'flat':
        sampler = her.make_sample_her_transitions(goal_replay, params['her_replay_k'], reward, '', tasks_ag_id=ag_ids,
                                                  tasks_g_id=g_ids)
        task_replay = ''
    else:
        sampler = her.make_sample_multi_task_her_transitions(goal_replay, params['her_replay_k'], task_replay, reward,
                                                             tasks_ag_id=ag_ids, tasks_g_id=g_ids)
    ddpg_kw = dict(input_dims=dims, hidden=params['hidden'], layers=params['layers'], network_class=params['network_class'],
                   polyak=params['polyak'], batch_size=params['batch_size'], Q_lr=params['Q_lr'], pi_lr=params['pi_lr'],
                   norm_eps=params['norm_eps'], norm_clip=params['norm_clip'], max_u=params['max_u'],
                   action_l2=params['action_l2'], clip_obs=params['clip_obs'], scope=params['scope'], T=T,
                   rollout_batch_size=params['rollout_batch_size'], subtract_goals=simple_goal_subtract,
                   relative_goals=params['relative_goals'], clip_pos_returns=True, clip_return=1. / (1. - gamma),
                   normalize_obs=normalize_obs, sample_transitions=sampler, gamma=gamma, tasks_ag_id=ag_ids, tasks_g_id=g_ids,
                   task_replay=task_replay, eps_task=params.get('eps_task'), structure=structure, her_rng='philox',
                   seed=seed, device=device)
    ddpg_kw['noise_seed'] = rs                      # key of the device-side exploration noise (action_noise='device')
    ddpg_kw.update(policy_kwargs or {})             # this implementation's extras: action_noise, update_schedule, comm, ...
    if workers_per_rank != 1:
        ddpg_kw.update(workers_per_rank=workers_per_rank, worker_buffers='own')
    sampler.seed = rs                               # Philox key of the HER draws
    buffer_size = (params['buffer_size'] // params['rollout_batch_size']) * params['rollout_batch_size']    # config.py:204
    buffers = configure_buffer({k: v for k, v in dims.items() if structure != 'flat' or k != 'task_descr'}, T, sampler,
                               buffer_size, structure, task_replay, nb_tasks, device=device)
    rollout_kw = dict(dims=dims, logger=None, T=T, rollout_batch_size=params['rollout_batch_size'], structure=structure,
                      task_selection=task_selection, queue_length=params['queue_length'])
    explore = dict(rollout_kw, exploit=False, use_target_net=False, compute_Q=False, noise_eps=params['noise_eps'],
                   random_eps=params['random_eps'])
    test = dict(rollout_kw, exploit=True, use_target_net=params['test_with_polyak'], compute_Q=True, eval=True)
    if structure == 'task_experts':                                 # train.py:287-289,325-331
        policy = [DDPG(buffers=buffers, t_id=i, **ddpg_kw) for i in range(nb_tasks)]
        for i, pol in enumerate(policy):
            # the experts share one sampler (one Philox key): give each its own counter range on the train-step stream
            pol.GRAPH_STREAM_OFFSET = DDPG.GRAPH_STREAM_OFFSET + (i << 36)
            pol.noise_seed = rs + i
        rollout_worker = [RolloutWorker(make_env, policy[i], unique_task=i, **explore) for i in range(nb_tasks)]
        for i, w in enumerate(rollout_worker):
            w.seed(rs + i)                                          # train.py:328-329
    else:
        policy = DDPG(buffers=buffers, **ddpg_kw)
        if workers_per_rank != 1:               # every worker acts, stores and samples on its own stream
            if not policy._action_rows_ok():
                raise ValueError('workers_per_rank > 1 acts through the one-launch action kernel, which does not take this '
                                 'network shape (see cur_ddpg_rows_supported)')
            explore = dict(explore, workers=workers_per_rank, streams=policy.worker_streams)
            test = dict(test, workers=workers_per_rank, streams=policy.worker_streams)
        rollout_worker = RolloutWorker(make_env, policy, **explore)
        rollout_worker.seed(rs)                                     # train.py:332
    evaluator = RolloutWorker(make_env, policy, **test)
    evaluator.seed(rs + 100)                                        # train.py:335
    run_params = dict(params, structure=structure, task_selection=task_selection, goal_selection='random',
                      goal_replay=goal_replay, task_replay=task_replay, normalize_obs=normalize_obs, seed=seed,
                      nb_tasks=nb_tasks, T=T, gamma=gamma, clip_return=1. / (1. - gamma),
                      env_name=type(env).__name__, num_cpu=evaluator.nb_cpu)
    return dict(policy=policy, rollout_worker=rollout_worker, evaluator=evaluator, n_cycles=params['n_cycles'],
                n_batches=params['n_batches'], n_test_rollouts=params['n_test_rollouts'], structure=structure,
                task_selection=task_selection, eps_task=params.get('eps_task', 0.4), params=run_params)


def _evaluate(evaluator, n_test_rollouts, clear_competence=False):
    """train.py:157-160: the evaluator's histories restart every epoch, its competence queues do not (they keep a running
    window over the evaluation rollouts of all epochs) unless `clear_competence` asks for a per-epoch measurement."""
    evaluator.clear_history()
    if clear_competence and evaluator.modular:
        evaluator.clear_competence_queue()
    for _ in range(n_test_rollouts):
        evaluator.generate_rollouts()
    out = dict(test_success_rate=float(evaluator.current_success_rate()), test_mean_Q=float(evaluator.current_mean_Q()))
    if evaluator.modular:
        out['C'] = np.asarray(evaluator.get_C(), np.float64).copy()
    return out


class _EpochRecords(object):
    """train.py:171-206 (`logs`): the tabular row of one epoch and the policy files, written by rank 0; plus (beyond the
    reference) the resumable state of the run, written by every rank for its own buffers, RNG streams and workers."""

    def __init__(self, logdir, evaluator, params, policy_save_interval, save_policies, checkpoint_interval, echo,
                 workers=(), resumed=None):
        self.evaluator = evaluator
        self.workers = list(workers)
        self.rank = evaluator.rank
        self.suffix = '' if self.rank == 0 else '_rank%d' % self.rank
        self.log = RunLog(logdir, rank=self.rank, echo=echo,
                          resume_after_epoch=None if resumed is None else resumed['epoch'])
        self.save_policies, self.interval = save_policies, policy_save_interval
        self.checkpoint_interval = checkpoint_interval
        self.best = -1 if resumed is None else resumed['best']
        self.t0 = time.time() - (0.0 if resumed is None else resumed['elapsed'])
        if params is not None:
            self.log.write_params(params)
        self.log.info('Training...' if resumed is None else 'Resuming after epoch %d...' % resumed['epoch'])

    def _path(self, name):
        return os.path.join(self.log.get_dir(), name)

    @staticmethod
    def load_run_state(logdir, rank):
        path = os.path.join(logdir, 'run_state%s.pkl' % ('' if rank == 0 else '_rank%d' % rank))
        if not os.path.exists(path):
            return None
        with open(path, 'rb') as f:
            return pickle.load(f)

    def _save_run_state(self, epoch, policy):
        """One resumable file per policy and one run_state per rank (every rank owns its replay buffers and RNG streams);
        written to a temporary name first so that a crash mid-write leaves the previous checkpoint intact."""
        os.makedirs(self.log.get_dir(), exist_ok=True)
        for i, pol in enumerate(policy if isinstance(policy, list) else [policy]):
            path = self._path('checkpoint_%d%s.pt' % (i, self.suffix))
            pol.save_checkpoint(path + '.tmp')
            os.replace(path + '.tmp', path)
        state = dict(epoch=epoch, best=self.best, elapsed=time.time() - self.t0,
                     workers=[w.state() for w in self.workers], evaluator=self.evaluator.state())
        path = self._path('run_state%s.pkl' % self.suffix)
        with open(path + '.tmp', 'wb') as f:
            pickle.dump(state, f)
        os.replace(path + '.tmp', path)

    def epoch(self, epoch, rollout_worker, policy, i_policy=None):
        log, comm = self.log, self.evaluator.comm
        log.record_tabular('epoch', epoch)
        for key, val in self.evaluator.logs('test'):
            log.record_tabular(key, '%.3g' % mpi_average(val, comm))
        for key, val in rollout_worker.logs('train'):
            log.record_tabular(key, '%.3g' % mpi_average(val, comm))
        for key, val in (policy[i_policy] if isinstance(policy, list) else policy).logs():
            log.record_tabular(key, '%.3g' % mpi_average(val, comm))
        if i_policy is not None:
            log.record_tabular('IND_TASK_rollout', i_policy)
        for key, val in rollout_worker.additional_logs('train') + self.evaluator.additional_logs('test'):
            log.record_tabular(key, val)
        log.record_tabular('Time', time.time() - self.t0)
        log.dump_tabular()
        rollout_worker.save_goal_task_history(log.get_dir())
        success = mpi_average(self.evaluator.current_success_rate(), comm)
        if getattr(self.evaluator, 'streams', None) is None:
            assert_rank_streams_differ(comm)                                   # train.py:207-212
        else:
            self.evaluator.streams.assert_differ()                             # ... on every virtual worker's stream
        if log.active and self.save_policies:
            if success >= self.best:
                self.best = success
                log.info('New best success rate: {}. Saving policy to {} ...'.format(success, self._path('policy_best.pkl')))
                self.evaluator.save_policy(self._path('policy_best.pkl'))
            if self.interval > 0 and epoch % self.interval == 0:
                self.evaluator.save_policy(self._path('policy_%d.pkl' % epoch))
                self.evaluator.save_policy(self._path('policy_latest.pkl'))
        if self.checkpoint_interval > 0 and epoch % self.checkpoint_interval == 0 and log.get_dir() is not None:
            self._save_run_state(epoch, policy)


def train(policy, rollout_worker, evaluator, n_epochs, n_test_rollouts, n_cycles, n_batches, structure='curious',
          task_selection='active_competence_progress', eps_task=0.4, log=None, logdir=None, params=None,
          policy_save_interval=5, save_policies=True, checkpoint_interval=0, echo=False, resume=False,
          experts_follow_cp=False, initial_evaluation=True, clear_eval_competence=False):
    """train.py:48-170: per epoch n_cycles x (rollouts -> store_episode -> n_batches x train -> update_target_net),
    then n_test_rollouts evaluation rollouts.  Returns one dict per epoch; with `logdir` also writes the reference's
    run records (see module docstring).  `resume=True` continues the run whose checkpoints (`checkpoint_interval`) are in
    `logdir` from the epoch after the last one: policies, buffers, optimiser, RNG streams, competence queues and the
    files pick up where they were (the returned history covers the new epochs).
    Like the reference, a fresh run starts with one evaluation of the untrained policy, recorded as epoch -1
    (train.py:62-75,125-135; `initial_evaluation=False` skips it), and the evaluator's competence queues run over all epochs
    (`clear_eval_competence=True` restarts them at every evaluation instead)."""
    hosted = getattr(evaluator, 'streams', None) is not None or getattr(policy, 'worker_buffers', 'shared') == 'own'
    if hosted:
        # what the learner refuses for worker_buffers='own' (DDPG), refused before the first rollout instead of mid-run
        if checkpoint_interval > 0 or resume:
            raise ValueError('checkpoints do not cover virtual workers (worker_buffers=\'own\')')
        if structure == 'task_experts' or isinstance(policy, list):
            raise ValueError("virtual workers do not take structure='task_experts'")
        if _world(evaluator.comm)[1] > 1:
            raise ValueError('virtual workers run on one rank')
    history = []
    records = None
    resumed_run = None
    start_epoch = 0
    workers = rollout_worker if isinstance(rollout_worker, list) else [rollout_worker]
    if logdir is not None:
        resumed = resumed_run = _EpochRecords.load_run_state(logdir, evaluator.rank) if resume else None
        if resumed is not None:
            suffix = '' if evaluator.rank == 0 else '_rank%d' % evaluator.rank
            for i, pol in enumerate(policy if isinstance(policy, list) else [policy]):
                pol.load_checkpoint(os.path.join(logdir, 'checkpoint_%d%s.pt' % (i, suffix)))
            for w, st in zip(workers, resumed['workers']):
                w.load_state(st)
            evaluator.load_state(resumed['evaluator'])
            start_epoch = resumed['epoch'] + 1
        records = _EpochRecords(logdir, evaluator, params, policy_save_interval, save_policies, checkpoint_interval, echo,
                                workers=workers, resumed=resumed)
    if initial_evaluation and start_epoch == 0 and resumed_run is None:   # (a run resumed from its epoch -1 checkpoint
        # must not evaluate the untrained policy a second time)
        # train.py:62-75 / 125-135: epoch -1.  The experts' branch also restarts the evaluator's competence queues here and
        # logs the LAST expert's worker and policy (i_policy = -1 indexes the lists from the end)
        evaluator.clear_history()
        if structure == 'task_experts' and evaluator.modular:
            evaluator.clear_competence_queue()
        for _ in range(n_test_rollouts):
            evaluator.generate_rollouts()
        if records:
            if structure == 'task_experts':
                records.epoch(-1, rollout_worker[-1], policy, -1)
            else:
                records.epoch(-1, rollout_worker, policy)
    if structure == 'task_experts':
        nb_tasks = len(policy)
        p = 1 / nb_tasks * np.ones([nb_tasks])
        for epoch in range(start_epoch, n_epochs):
            proba = p.copy()
            if task_selection == 'random':
                i_policy = epoch % nb_tasks                                  # train.py:79-81
            else:
                # train.py:83-104: rank 0 draws the expert, everybody follows
                if evaluator.rank == 0:
                    cps = [np.array([rollout_worker[i].get_CP()]).squeeze()[i] for i in range(nb_tasks)]
                    CP = np.array(cps).copy()
                    if CP.sum() == 0:
                        proba = (1 / nb_tasks) * np.ones([nb_tasks])
                    else:
                        proba = eps_task * (1 / nb_tasks) * np.ones([nb_tasks]) + (1 - eps_task) * CP / CP.sum()
                    # The reference computes `proba` and then normalises and draws from `p`, which is never assigned from it
                    # (train.py:91-100): its experts are picked uniformly whatever their competence progress.  Kept as it
                    # behaves; experts_follow_cp=True draws from `proba`, which is what the code reads like it meant.
                    if experts_follow_cp:
                        p = proba.copy()
                    if p.sum() > 1:
                        p[np.argmax(p)] -= p.sum() - 1
                    elif p.sum() < 1:
                        p[-1] = 1 - p[:-1].sum()
                    i_policy = int(np.random.choice(range(nb_tasks), p=p))
                else:
                    i_policy = 0
                i_policy = int(bcast_object(i_policy, evaluator.comm))
            rollout_worker[i_policy].clear_history()
            for _ in range(n_cycles):
                episode, cp, n_ep = rollout_worker[i_policy].generate_rollouts()
                policy[i_policy].store_episode(episode, cp, n_ep)
                for _ in range(n_batches):
                    policy[i_policy].train()
                policy[i_policy].update_target_net()
            rec = dict(epoch=epoch, i_policy=i_policy, p=p.copy(), proba=proba.copy(), **_evaluate(evaluator, n_test_rollouts, clear_eval_competence))
            history.append(rec)
            if log:
                log(rec)
            if records:
                records.epoch(epoch, rollout_worker[i_policy], policy, i_policy)
        if records:
            records.log.close()
        return history
    for epoch in range(start_epoch, n_epochs):                                            # train.py:125-166
        rollout_worker.clear_history()
        for _ in range(n_cycles):
            episode, cp, n_ep = rollout_worker.generate_rollouts()
            policy.store_episode(episode, cp, n_ep)
            for _ in range(n_batches):
                policy.train()
            policy.update_target_net()
        rec = dict(epoch=epoch, train_success_rate=float(rollout_worker.current_success_rate()),
                   **_evaluate(evaluator, n_test_rollouts, clear_eval_competence))
        if rollout_worker.modular:
            rec['CP'] = np.asarray(rollout_worker.get_CP(), np.float64).copy()
            rec['p'] = np.asarray(rollout_worker.p, np.float64).copy()
        history.append(rec)
        if log:
            log(rec)
        if records:
            records.epoch(epoch, rollout_worker, policy)
    if records:
        records.log.close()
    return history
