"""Host random streams of the reference workers one rank hosts (DDPG(worker_buffers='own')).

The reference runs one MPI worker per process and seeds each with rank_seed = seed + 1000000 * rank (train.py:241-243):
every host draw a worker makes - replay slots once its buffers are full (replay_buffer.py:99-102), the HER sampler's
draws (her.py:108-116) and the batch shuffle (ddpg.py:338-339) - comes from that worker's own np.random stream.  With k
workers on rank r, worker j stands for reference rank r * k + j.  Its stream is kept here as a saved np.random state
and swapped into np.random only around that worker's draws, so the caller's global stream (which the rollouts draw
from) comes back exactly as it was.
"""
import contextlib

import numpy as np

from .parallel import rank_seed


class WorkerStreams:
    def __init__(self, seed, n_workers, rank=0):
        self.seeds = [rank_seed(int(seed), rank * n_workers + j) for j in range(n_workers)]
        # np.random.seed takes 32 bits (make_experiment seeds the same way, train.py of this package)
        self._states = [np.random.RandomState(s % (2 ** 32)).get_state() for s in self.seeds]

    def __len__(self):
        return len(self._states)

    def philox_key(self, j):
        """Key of worker j's device draws: a lone agent of that rank is keyed with its rank seed (make_experiment)."""
        return self.seeds[j] & 0xFFFFFFFFFFFFFFFF

    def state(self, j):
        """Worker j's np.random state, in np.random.get_state() form."""
        return self._states[j]

    @contextlib.contextmanager
    def use(self, j):
        """np.random is worker j's stream inside the block; the caller's state is restored afterwards."""
        saved = np.random.get_state()
        np.random.set_state(self._states[j])
        try:
            yield
        finally:
            self._states[j] = np.random.get_state()
            np.random.set_state(saved)
