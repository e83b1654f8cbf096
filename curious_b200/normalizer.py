"""Running-statistics normaliser on the device - drop-in for reference baselines/her/normalizer.py.

State (sum, sumsq, count, mean, std) is float32 on the GPU.  `update` is a column-reduction kernel,
`recompute_stats` packs (sum | sumsq | count) of all ranks into ONE all-reduce (the reference issues
three blocking MPI all-reduces per normaliser, normalizer.py:84-94) followed by one fused kernel for
`+=`, mean and std (normalizer.py:50-61).
"""
import threading

import numpy as np
import torch

from . import _lib


from .parallel import allreduce_sum_, world as _world


class Normalizer:
    def __init__(self, size, eps=1e-2, default_clip_range=np.inf, sess=None, device=None, comm=None, partial=None):
        """Same arguments as the reference (normalizer.py:11); `sess` is accepted and ignored.  `partial`: a float32
        device view of 2 * size + 1 zeros to accumulate into - several normalisers handed slices of ONE buffer are
        synchronised with a single collective (`recompute_stats_packed`)."""
        self.size = size
        self.eps = eps
        self.default_clip_range = default_clip_range
        self.sess = sess
        self.device = device or torch.device('cuda', torch.cuda.current_device())
        self.comm = comm
        # [sum | sumsq | count]; count starts at ONE with sum = 0 (normalizer.py:31-39)
        self._partial = partial if partial is not None else torch.zeros(2 * size + 1, dtype=torch.float32, device=self.device)
        assert self._partial.numel() == 2 * size + 1 and self._partial.dtype == torch.float32
        self._running = torch.zeros(2 * size + 1, dtype=torch.float32, device=self.device)
        self._running[2 * size] = 1.0
        self.mean = torch.zeros(size, dtype=torch.float32, device=self.device)
        self.std = torch.ones(size, dtype=torch.float32, device=self.device)
        self.lock = threading.Lock()

    # reference attribute names, as device views
    @property
    def local_sum(self):
        return self._partial[:self.size]

    @property
    def local_sumsq(self):
        return self._partial[self.size:2 * self.size]

    @property
    def local_count(self):
        return self._partial[2 * self.size:]

    @property
    def sum(self):
        return self._running[:self.size]

    @property
    def sumsq(self):
        return self._running[self.size:2 * self.size]

    @property
    def count(self):
        return self._running[2 * self.size:]

    def _as_device(self, v):
        if torch.is_tensor(v):
            return v.to(self.device, torch.float32).contiguous()
        return torch.from_numpy(np.ascontiguousarray(v, dtype=np.float32)).to(self.device)

    def update(self, v):
        v = self._as_device(v).reshape(-1, self.size)                 # normalizer.py:64-70
        with self.lock:
            _lib.check(_lib.load().cur_norm_accumulate(_lib.stream_ptr(), v.data_ptr(), v.shape[0], self.size,
                                                       self._partial.data_ptr()), 'cur_norm_accumulate')

    def normalize(self, v, clip_range=None):
        if clip_range is None:
            clip_range = self.default_clip_range
        v = self._as_device(v)
        out = torch.empty_like(v)
        n = v.numel() // self.size
        clip = float(clip_range) if np.isfinite(clip_range) else float(np.finfo(np.float32).max)
        _lib.check(_lib.load().cur_norm_apply(_lib.stream_ptr(), v.data_ptr(), n, self.size, self.mean.data_ptr(),
                                              self.std.data_ptr(), clip, out.data_ptr()), 'cur_norm_apply')
        return out

    def denormalize(self, v):
        v = self._as_device(v)
        out = torch.empty_like(v)
        n = v.numel() // self.size
        _lib.check(_lib.load().cur_norm_invert(_lib.stream_ptr(), v.data_ptr(), n, self.size, self.mean.data_ptr(),
                                               self.std.data_ptr(), out.data_ptr()), 'cur_norm_invert')
        return out

    def synchronize(self, local_sum=None, local_sumsq=None, local_count=None, root=None):
        """Cross-rank SUM of the packed partials (the division by the world size, normalizer.py:87,
        happens in recompute).  Arguments are accepted for signature parity; the packed device buffer
        is what is reduced."""
        return allreduce_sum_(self._partial, self.comm)

    def recompute_stats(self, world=None):
        """normalizer.py:96-118.  `world`: the partials were already summed over that many ranks (packed path)."""
        with self.lock:
            if world is None:
                world = self.synchronize()
            _lib.check(_lib.load().cur_norm_recompute(_lib.stream_ptr(), self._running.data_ptr(),
                                                      self._partial.data_ptr(), float(world), float(self.eps),
                                                      self.size, self.mean.data_ptr(), self.std.data_ptr()),
                       'cur_norm_recompute')

    # (de)serialisation in the reference's global-variable order: sum, sumsq, count, mean, std
    # (normalizer.py:31-45; used by DDPG.save_weights, ddpg.py:481-497)
    def state_list(self):
        return [t.detach().cpu().numpy().copy() for t in (self.sum, self.sumsq, self.count, self.mean, self.std)]

    def load_state_list(self, arrays):
        s, q, c, m, sd = [np.asarray(a, np.float32) for a in arrays]
        self._running[:self.size] = torch.from_numpy(s).to(self.device)
        self._running[self.size:2 * self.size] = torch.from_numpy(q).to(self.device)
        self._running[2 * self.size:] = torch.from_numpy(c.reshape(1)).to(self.device)
        self.mean.copy_(torch.from_numpy(m).to(self.device))
        self.std.copy_(torch.from_numpy(sd).to(self.device))


def recompute_stats_packed(normalizers, packed, comm=None, workers=1):
    """`recompute_stats` of several normalisers whose partials are slices of `packed`: ONE all-reduce for all of them
    per store_episode (the reference issues three blocking all-reduces per normaliser, normalizer.py:84-94, six per
    store; SURVEY 8e asks for one packed collective), then each one's `+=` / mean / std kernel.  `workers`: reference
    workers per rank whose batches all went into the partials - the mean is over workers x ranks."""
    world = allreduce_sum_(packed, comm)
    for nz in normalizers:
        nz.recompute_stats(world=world * workers)
    return world


class IdentityNormalizer:
    """reference normalizer.py:121-140"""

    def __init__(self, size, std=1.):
        self.size = size
        self.mean = torch.zeros(size, dtype=torch.float32)
        self.std = std * torch.ones(size, dtype=torch.float32)

    def update(self, x):
        pass

    def normalize(self, x, clip_range=None):
        return x / self.std

    def denormalize(self, x):
        return self.std * x

    def synchronize(self):
        pass

    def recompute_stats(self):
        pass
