"""CPU tests of worker_buffers='own': the host random streams of the hosted workers, the ctypes mirror of the new
structs, and the refusals of cur_her_sample_workers (checked before any launch, so the library answers without a
device)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_worker_streams_are_independently_seeded_rank_streams():
    from curious_b200.parallel import rank_seed
    from curious_b200.workers import WorkerStreams
    k, seed = 3, 17
    ws = WorkerStreams(seed, k)
    ref = [np.random.RandomState(rank_seed(seed, j) % 2 ** 32) for j in range(k)]
    np.random.seed(99)
    caller = np.random.get_state()
    # interleaved draws of different sizes: each worker continues its own stream, the caller's stream is untouched
    for rnd in range(4):
        for j in (2, 0, 1):
            with ws.use(j):
                got = np.random.randint(0, 1000, rnd + j + 1)
                got_u = np.random.uniform(size=2)
            assert np.array_equal(got, ref[j].randint(0, 1000, rnd + j + 1))
            assert np.array_equal(got_u, ref[j].uniform(size=2))
            now = np.random.get_state()
            assert now[0] == caller[0] and np.array_equal(now[1], caller[1]) and now[2:] == caller[2:]
    for j in range(k):
        st, want = ws.state(j), ref[j].get_state()
        assert np.array_equal(st[1], want[1]) and st[2:] == want[2:]
        assert ws.philox_key(j) == rank_seed(seed, j)


def test_worker_streams_restore_the_caller_state_on_error():
    from curious_b200.workers import WorkerStreams
    ws = WorkerStreams(0, 2)
    np.random.seed(5)
    before = np.random.get_state()
    with pytest.raises(RuntimeError):
        with ws.use(1):
            np.random.uniform()
            raise RuntimeError('boom')
    after = np.random.get_state()
    assert np.array_equal(before[1], after[1]) and before[2:] == after[2:]


def test_worker_structs_match_header(tmp_path):
    from curious_b200 import _lib
    src = tmp_path / 'sz.cpp'
    src.write_text('#include "%s"\n#include <stdio.h>\nint main(){printf("%%zu %%zu %%d\\n",'
                   'sizeof(cur_her_worker),sizeof(cur_her_worker_dyn),CUR_MAX_WORKERS);}\n'
                   % os.path.join(ROOT, 'include', 'curious_b200.h'))
    exe = tmp_path / 'sz'
    subprocess.check_call(['g++', str(src), '-o', str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert got == [C.sizeof(_lib.HerWorker), C.sizeof(_lib.HerWorkerDyn), _lib.CUR_MAX_WORKERS]


def _args(batch):
    from curious_b200 import _lib
    a = _lib.HerArgs()
    a.L = _lib.make_layout(50, 10, 3, 3, 4)
    a.mode = _lib.MODE_FLAT
    a.batch = batch
    return a


def _workers(n, counts, n_segments=1):
    from curious_b200 import _lib
    W = (_lib.HerWorker * n)()
    for j in range(n):
        W[j].seed = j
        W[j].n_segments = n_segments
        for i in range(min(n_segments, _lib.CUR_MAX_SEGMENTS)):
            W[j].seg[i].base = 256          # never dereferenced: every case is refused before a launch
            W[j].seg[i].n_episodes = 4
            W[j].seg[i].count = counts[j] if i == 0 else 0
    return W


@pytest.mark.parametrize('case', ['n_workers_0', 'n_workers_65', 'segments_18', 'segments_0', 'counts', 'batch'])
def test_sample_workers_refusals(case):
    from curious_b200 import _lib
    lib = _lib.load()
    n, R = 2, 8
    counts = [R] * 65
    a, W, nw, rows = _args(n * R), None, n, R
    if case == 'n_workers_0':
        nw, a = 0, _args(0)
    elif case == 'n_workers_65':
        nw, a = 65, _args(65 * R)
        W = _workers(65, counts)
    elif case == 'segments_18':
        W = _workers(n, counts)
        W[1].n_segments = 18
    elif case == 'segments_0':
        W = _workers(n, counts)
        W[0].n_segments = 0
    elif case == 'counts':
        W = _workers(n, [R, R - 1])
    elif case == 'batch':
        a = _args(n * R + 4)
    if W is None:
        W = _workers(max(nw, 1), counts)
    dyn = C.c_void_p(4096)                  # a device address in real use; not read when the call is refused
    status = lib.cur_her_sample_workers(None, C.byref(a), nw, rows, W, dyn, None)
    assert status == 1, case                 # CUR_ERR_INVALID
