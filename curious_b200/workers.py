"""Host random streams of the reference workers one rank hosts (DDPG(worker_buffers='own'), RolloutWorker(workers=k)).

The reference runs one MPI worker per process and seeds each with rank_seed = seed + 1000000 * rank (train.py:241-243):
every host draw a worker makes - its exploit draw and the exploration noise of its rollouts (rollout.py:178-230,
ddpg.py:147-152), replay slots once its buffers are full (replay_buffer.py:99-102), the HER sampler's draws
(her.py:108-116) and the batch shuffle (ddpg.py:338-339) - comes from that worker's own np.random stream.  With k
workers on rank r, worker j stands for reference rank r * k + j.  Its stream is one np.random.RandomState: rollout code
draws from it directly (`rng(j)`), the learner's np.random code paths see it as the global stream inside `use(j)`, so
the caller's global stream comes back exactly as it was and both views advance one stream.
"""
import contextlib

import numpy as np

from .parallel import rank_seed


class WorkerStreams:
    def __init__(self, seed, n_workers, rank=0):
        self.seeds = [rank_seed(int(seed), rank * n_workers + j) for j in range(n_workers)]
        # np.random.seed takes 32 bits (make_experiment seeds the same way, train.py of this package)
        self._rngs = [np.random.RandomState(s % (2 ** 32)) for s in self.seeds]

    def __len__(self):
        return len(self._rngs)

    def philox_key(self, j):
        """Key of worker j's device draws: a lone agent of that rank is keyed with its rank seed (make_experiment)."""
        return self.seeds[j] & 0xFFFFFFFFFFFFFFFF

    def rng(self, j):
        """Worker j's stream as a np.random.RandomState: its methods draw what the np.random functions of the same name
        draw from the global stream in that state."""
        return self._rngs[j]

    def state(self, j):
        """Worker j's np.random state, in np.random.get_state() form."""
        return self._rngs[j].get_state()

    @contextlib.contextmanager
    def use(self, j):
        """np.random is worker j's stream inside the block; the caller's state is restored afterwards."""
        saved = np.random.get_state()
        np.random.set_state(self._rngs[j].get_state())
        try:
            yield
        finally:
            self._rngs[j].set_state(np.random.get_state())
            np.random.set_state(saved)

    def assert_differ(self):
        """train.py:207-212 for the hosted workers: each draws one uniform from its own stream, and workers seeded like
        worker 0 are caught.  Consumes one draw of every worker's stream, like the reference on every rank."""
        draws = [float(r.uniform(size=(1,))[0]) for r in self._rngs]
        for j in range(1, len(draws)):
            assert draws[j] != draws[0], 'worker %d draws the same np.random stream as worker 0 (train.py:211-212)' % j
        return draws
