"""ctypes binding of libcurious_b200.so (the C ABI declared in include/curious_b200.h).

There is NO CPU fallback: if the library is missing or a call fails, this module raises.
torch is used only for device memory and streams (tensor.data_ptr(), current stream).
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, 'libcurious_b200.so')

CUR_MAX_TASKS = 16
CUR_MAX_SLICE = 8
CUR_MAX_SEGMENTS = 17
CUR_MAX_COPIES = 64
CUR_MAX_WORKERS = 64

MODE_BUFFER, MODE_RANDOM_TASK, MODE_CP_TASK, MODE_CURRENT_TASK, MODE_FLAT = range(5)

f32p = C.POINTER(C.c_float)


class Layout(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        'T', 'dimo', 'dimag', 'dimg', 'dimu', 'dimtd', 'dimchange', 'diminfo',
        'off_g', 'off_u', 'off_td', 'off_ag', 'off_o', 'row_stride',
        'off_change', 'off_info', 'cold_stride', 'trans_stride', 'off_agc')]


class EpisodeSrc(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ('o', 'ag', 'g', 'u', 'td', 'change', 'info')]


class Segment(C.Structure):
    _fields_ = [('base', C.c_void_p), ('cold', C.c_void_p), ('n_episodes', C.c_int32), ('count', C.c_int32),
                ('task_to_replay', C.c_int32), ('_pad', C.c_int32)]


REWARD_DISTANCE, REWARD_PAIR, REWARD_INFO = 0, 1, 2


class TaskTable(C.Structure):
    _fields_ = [('n_tasks', C.c_int32), ('_pad', C.c_int32),
                ('len', C.c_int32 * CUR_MAX_TASKS),
                ('g_idx', (C.c_int16 * CUR_MAX_SLICE) * CUR_MAX_TASKS),
                ('ag_idx', (C.c_int16 * CUR_MAX_SLICE) * CUR_MAX_TASKS),
                ('ref_idx', (C.c_int16 * CUR_MAX_SLICE) * CUR_MAX_TASKS),
                ('kind', C.c_int32 * CUR_MAX_TASKS),
                ('info_col', C.c_int32 * CUR_MAX_TASKS),
                ('threshold', C.c_double * CUR_MAX_TASKS),
                ('flat_threshold', C.c_double),
                ('cdf', C.c_double * CUR_MAX_TASKS)]


class HerDyn(C.Structure):
    _fields_ = [('step', C.c_void_p), ('n_episodes', C.c_int32 * CUR_MAX_SEGMENTS),
                ('count', C.c_int32 * CUR_MAX_SEGMENTS), ('cdf', C.c_double * CUR_MAX_TASKS)]


class HerArgs(C.Structure):
    _fields_ = [('L', Layout), ('tasks', TaskTable), ('mode', C.c_int32), ('n_segments', C.c_int32),
                ('seg', Segment * CUR_MAX_SEGMENTS), ('batch', C.c_int64), ('future_p', C.c_double),
                ('inj_ep', C.c_void_p), ('inj_t', C.c_void_p), ('inj_u_her', C.c_void_p),
                ('inj_u_off', C.c_void_p), ('inj_choice', C.c_void_p),
                ('seed', C.c_uint64), ('call_offset', C.c_uint64), ('perm', C.c_void_p),
                ('clip_obs', C.c_float), ('relative_goals', C.c_int32),
                ('o', C.c_void_p), ('ag', C.c_void_p), ('g', C.c_void_p), ('u', C.c_void_p),
                ('td', C.c_void_p), ('change', C.c_void_p), ('info', C.c_void_p), ('o_2', C.c_void_p),
                ('ag_2', C.c_void_p), ('g_2', C.c_void_p), ('r', C.c_void_p), ('idx_out', C.c_void_p),
                ('dyn', C.c_void_p)]


class HerWorker(C.Structure):
    _fields_ = [('seed', C.c_uint64), ('n_segments', C.c_int32), ('_pad', C.c_int32), ('seg', Segment * CUR_MAX_SEGMENTS)]


class HerWorkerDyn(C.Structure):
    _fields_ = [('n_episodes', C.c_int32 * CUR_MAX_SEGMENTS), ('count', C.c_int32 * CUR_MAX_SEGMENTS),
                ('cdf', C.c_double * CUR_MAX_TASKS)]


class NetDesc(C.Structure):
    _fields_ = [('modular', C.c_int32), ('dimo', C.c_int32), ('dimg', C.c_int32), ('dimu', C.c_int32),
                ('dimtd', C.c_int32), ('hidden', C.c_int32), ('layers', C.c_int32), ('max_u', C.c_float),
                ('normalize_obs', C.c_int32), ('norm_clip', C.c_float)]


class NormStats(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ('o_mean', 'o_std', 'g_mean', 'g_std')]


class ActionsExpert(C.Structure):
    _fields_ = [('theta', C.c_void_p), ('stats', NormStats)]


class Batch(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ('o', 'g', 'u', 'td', 'o_2', 'g_2', 'r')] + [('n', C.c_int64)]


class DdpgHyper(C.Structure):
    _fields_ = [('gamma', C.c_float), ('clip_return', C.c_float), ('action_l2', C.c_float),
                ('clip_pos_returns', C.c_int32), ('step_counter', C.c_void_p), ('loss_ring', C.c_int32),
                ('micro_batches', C.c_int32), ('grads_parity_stride', C.c_int64), ('loss_rows', C.c_int64),
                ('transposes_valid', C.c_int32), ('_pad2', C.c_int32)]


class DdpgExpert(C.Structure):
    _fields_ = [('theta_main', C.c_void_p), ('theta_target', C.c_void_p), ('stats', NormStats), ('has_stats', C.c_int32),
                ('_pad', C.c_int32), ('batch', Batch), ('hyper', DdpgHyper), ('workspace', C.c_void_p),
                ('grads', C.c_void_p), ('q_loss', C.c_void_p), ('pi_loss', C.c_void_p), ('q_pi', C.c_void_p)]


CUR_MAX_RANKS = 8


class XchgCtx(C.Structure):
    _fields_ = [('rank', C.c_int32), ('world', C.c_int32), ('mode', C.c_int32), ('_pad', C.c_int32),
                ('region', C.c_void_p * CUR_MAX_RANKS), ('arena', C.c_int64), ('timeline', C.c_void_p),
                ('error_flag', C.c_void_p), ('mc_region', C.c_void_p)]


class AdamFused(C.Structure):
    _fields_ = [('m', C.c_void_p), ('v', C.c_void_p), ('neg_a_table', C.c_void_p), ('table_len', C.c_int32),
                ('transposes_valid', C.c_int32), ('beta1', C.c_double), ('beta2', C.c_double), ('eps', C.c_double),
                ('xchg', C.POINTER(XchgCtx))]


CUR_P2P_MAX_TRANSPOSES = 8


class P2PTransposes(C.Structure):
    _fields_ = [('n', C.c_int32), ('H', C.c_int32), ('begin', C.c_int64 * CUR_P2P_MAX_TRANSPOSES),
                ('dst', C.c_void_p * CUR_P2P_MAX_TRANSPOSES)]


class P2PCtx(C.Structure):
    _fields_ = [('rank', C.c_int32), ('world', C.c_int32), ('region', C.c_void_p * CUR_MAX_RANKS),
                ('arena', C.c_int64), ('step_div', C.c_int32), ('_pad', C.c_int32)]


# name -> (restype, argtypes); every symbol include/curious_b200.h declares
SIGNATURES = {
    'cur_abi_version': (C.c_int, []),
    'cur_last_error': (C.c_char_p, []),
    'cur_device_info': (C.c_int, [C.POINTER(C.c_int)] * 3),
    'cur_layout_init': (C.c_int, [C.POINTER(Layout)] + [C.c_int] * 8),
    'cur_store_episodes': (C.c_int, [C.c_void_p, C.POINTER(Layout), C.POINTER(EpisodeSrc), C.c_int, C.c_int,
                                     C.POINTER(C.c_int32), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                     C.POINTER(C.c_int64)]),
    'cur_her_sample': (C.c_int, [C.c_void_p, C.POINTER(HerArgs)]),
    'cur_her_sample_workers': (C.c_int, [C.c_void_p, C.POINTER(HerArgs), C.c_int, C.c_int, C.POINTER(HerWorker),
                                         C.c_void_p, C.c_void_p]),
    'cur_philox4x32_10': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    'cur_norm_accumulate': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    'cur_norm_recompute': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_int,
                                     C.c_void_p, C.c_void_p]),
    'cur_norm_apply': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p,
                                 C.c_float, C.c_void_p]),
    'cur_norm_invert': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p,
                                  C.c_void_p]),
    'cur_adam_step': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                C.c_float, C.c_double, C.c_double, C.c_double, C.c_float]),
    'cur_adam_step_graph': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                      C.c_void_p, C.c_int, C.c_void_p, C.c_double, C.c_double, C.c_double,
                                      C.c_float, C.c_int32]),
    'cur_polyak': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_double]),
    'cur_checksum': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    'cur_ddpg_actions_rows': (C.c_int, [C.c_void_p, C.POINTER(NetDesc), C.c_void_p, C.POINTER(NormStats), C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_float, C.c_void_p, C.c_void_p,
                                        C.c_uint32]),
    'cur_ddpg_actions_rows_group': (C.c_int, [C.c_void_p, C.POINTER(NetDesc), C.c_int, C.POINTER(ActionsExpert),
                                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                              C.c_float, C.c_void_p, C.c_void_p, C.c_uint32]),
    'cur_actions_finish_host':(C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_uint32, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_double, C.c_double, C.c_void_p, C.c_void_p, C.c_int64]),
    'cur_host_alloc': (C.c_int, [C.c_int64, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
    'cur_host_free': (C.c_int, [C.c_void_p]),
    'cur_copy_h2d': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]),
    'cur_action_noise': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_float, C.c_double, C.c_double,
                                   C.c_uint64, C.c_uint64]),
    'cur_action_noise_rows': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_float, C.c_double, C.c_double,
                                        C.c_void_p, C.c_void_p]),
    'cur_net_param_count': (C.c_int64, [C.POINTER(NetDesc), C.c_int]),
    'cur_theta_pi_offset': (C.c_int64, [C.POINTER(NetDesc), C.POINTER(C.c_int64)]),
    'cur_ddpg_workspace_floats': (C.c_int64, [C.POINTER(NetDesc), C.c_int64]),
    'cur_ddpg_actions': (C.c_int, [C.c_void_p, C.POINTER(NetDesc), C.c_void_p, C.POINTER(NormStats),
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_float,
                                   C.c_void_p, C.c_void_p, C.c_void_p]),
    'cur_ddpg_grads': (C.c_int, [C.c_void_p, C.POINTER(NetDesc), C.c_void_p, C.c_void_p,
                                 C.POINTER(NormStats), C.POINTER(Batch), C.POINTER(DdpgHyper), C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'cur_ddpg_rows_supported': (C.c_int, [C.POINTER(NetDesc), C.c_int64]),
    'cur_ddpg_rows_workspace_floats': (C.c_int64, [C.POINTER(NetDesc), C.c_int64]),
    'cur_ddpg_rows_step': (C.c_int, [C.c_void_p, C.POINTER(NetDesc), C.c_void_p, C.c_void_p,
                                     C.POINTER(NormStats), C.POINTER(Batch), C.POINTER(DdpgHyper), C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(AdamFused),
                                     C.POINTER(HerArgs)]),
    'cur_ddpg_rows_refresh': (C.c_int, [C.c_void_p, C.POINTER(NetDesc), C.c_void_p, C.c_void_p, C.c_int64]),
    'cur_ddpg_grads_group': (C.c_int, [C.c_void_p, C.POINTER(NetDesc), C.c_int, C.POINTER(DdpgExpert)]),
    'cur_ddpg_set_tensor_cores': (C.c_int, [C.c_int]),
    'cur_tc_chain_timeline': (C.c_int, [C.c_void_p]),
    'cur_rows_timeline_dump': (C.c_int, []),
    'cur_ddpg_set_chain': (C.c_int, [C.c_int]),
    'cur_ddpg_uses_chain': (C.c_int, [C.POINTER(NetDesc), C.c_int64]),
    'cur_ddpg_uses_tensor_cores': (C.c_int, [C.POINTER(NetDesc), C.c_int64]),
    'cur_ddpg_chain_supported': (C.c_int, [C.POINTER(NetDesc), C.c_int64]),
    'cur_ddpg_chain_workspace_floats': (C.c_int64, [C.POINTER(NetDesc), C.c_int64]),
    'cur_ddpg_chain_grads': (C.c_int, [C.c_void_p, C.POINTER(NetDesc), C.c_void_p, C.c_void_p,
                                       C.POINTER(NormStats), C.POINTER(Batch), C.POINTER(DdpgHyper), C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'cur_ddpg_chain_grads_group': (C.c_int, [C.c_void_p, C.POINTER(NetDesc), C.c_int, C.POINTER(DdpgExpert)]),
    'cur_tc_gemm_timeline': (C.c_int, [C.c_void_p]),
    'cur_tc_gemm_supported': (C.c_int, [C.c_int64, C.c_int64, C.c_int64]),
    'cur_tc_gemm_workspace_floats': (C.c_int64, [C.c_int64, C.c_int64, C.c_int64, C.c_int]),
    'cur_tc_gemm': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int64, C.c_int, C.c_void_p,
                              C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_int,
                              C.c_void_p]),
    'cur_ddpg_rows_owner_map': (C.c_int, [C.POINTER(NetDesc), C.c_int64, C.c_int, C.c_void_p]),
    'cur_xchg_region_bytes': (C.c_int64, [C.c_int64, C.c_int]),
    'cur_p2p_region_bytes': (C.c_int64, [C.c_int64]),
    'cur_p2p_alloc': (C.c_int, [C.c_int64, C.POINTER(C.c_void_p), C.c_char_p]),
    'cur_p2p_open': (C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]),
    'cur_p2p_close': (C.c_int, [C.c_void_p]),
    'cur_p2p_free': (C.c_int, [C.c_void_p]),
    'cur_p2p_zero': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64]),
    'cur_p2p_allreduce_adam': (C.c_int, [C.c_void_p, C.POINTER(P2PCtx), C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_int, C.c_void_p, C.c_double, C.c_double, C.c_double,
                                         C.c_void_p]),
    'cur_p2p_allreduce_adam_t': (C.c_int, [C.c_void_p, C.POINTER(P2PCtx), C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_int, C.c_void_p, C.c_double, C.c_double, C.c_double,
                                           C.c_void_p, C.POINTER(P2PTransposes)]),
    'cur_ddpg_rows_transposes': (C.c_int, [C.POINTER(NetDesc), C.c_void_p, C.c_int64, C.POINTER(P2PTransposes)]),
    'cur_p2p_sharded_adam': (C.c_int, [C.c_void_p, C.POINTER(P2PCtx), C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_int, C.c_void_p, C.c_double, C.c_double, C.c_double,
                                       C.c_void_p]),
}

_lib = None


class CuriousLibError(RuntimeError):
    pass


def load():
    """Load the shared library (once).  Raises if it has not been built - there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CuriousLibError(
            '%s not found: build it with `python -m curious_b200.build` (or __graft_entry__.build()). '
            'curious_b200 has no CPU fallback.' % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status, what):
    if status != 0:
        msg = load().cur_last_error()
        raise CuriousLibError('%s failed with status %d: %s' % (what, status, (msg or b'').decode()))


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    return None if t is None else t.data_ptr()


def stream_ptr(stream=None):
    """cudaStream_t of `stream` or of torch's current stream (the raw-handle query: torch.cuda.current_stream() builds a
    Stream object per call, ~5 us - more than a kernel launch)."""
    if stream is not None:
        return stream.cuda_stream
    import torch
    try:
        return torch._C._cuda_getCurrentRawStream(torch._C._cuda_getDevice())
    except AttributeError:
        return torch.cuda.current_stream().cuda_stream


def make_layout(T, dimo, dimag, dimg, dimu, dimtd=0, dimchange=0, diminfo=0):
    L = Layout()
    check(load().cur_layout_init(C.byref(L), T, dimo, dimag, dimg, dimu, dimtd, dimchange, diminfo),
          'cur_layout_init')
    return L


def make_task_table(tasks_ag_id, tasks_g_id, threshold=0.05, cp_proba=None, kinds=None, ref_ag_id=None, info_cols=None,
                    flat_threshold=None):
    """cur_task_table: per module the goal / achieved-goal columns and its reward rule (kind, threshold, and for PAIR the
    second achieved-goal slice, for INFO the column of the stored info row).  `threshold` is a scalar or one per module."""
    tt = TaskTable()
    n = len(tasks_g_id) if tasks_g_id is not None else 0
    if n > CUR_MAX_TASKS:
        raise ValueError('at most %d modules are supported' % CUR_MAX_TASKS)
    tt.n_tasks = n
    thr = np.broadcast_to(np.asarray(threshold, np.float64), (n,)) if n else np.zeros(0)
    tt.flat_threshold = float(flat_threshold if flat_threshold is not None else (thr[0] if n else 0.05))
    for m in range(n):
        g_ids = list(tasks_g_id[m])
        ag_ids = list(tasks_ag_id[m])[:len(g_ids)]     # her.py:147-148
        if len(g_ids) > CUR_MAX_SLICE:
            raise ValueError('module goal slices longer than %d are not supported' % CUR_MAX_SLICE)
        tt.len[m] = len(g_ids)
        tt.kind[m] = int(kinds[m]) if kinds is not None else REWARD_DISTANCE
        tt.threshold[m] = float(thr[m])
        tt.info_col[m] = int(info_cols[m]) if info_cols is not None and info_cols[m] is not None else 0
        for k, (gi, ai) in enumerate(zip(g_ids, ag_ids)):
            tt.g_idx[m][k] = int(gi)
            tt.ag_idx[m][k] = int(ai)
        if tt.kind[m] == REWARD_PAIR:
            ref = list(ref_ag_id[m])[:len(g_ids)]
            if len(ref) != len(g_ids):
                raise ValueError('module %d: the PAIR reward needs a reference slice as long as the goal slice' % m)
            for k, ri in enumerate(ref):
                tt.ref_idx[m][k] = int(ri)
    if cp_proba is not None:
        set_cdf(tt, cp_proba)
    return tt


def set_cdf(tt, cp_proba):
    # np.random.choice(p=): cdf = p.cumsum(); cdf /= cdf[-1]
    p = np.asarray(cp_proba, np.float64)
    cdf = p.cumsum()
    cdf /= cdf[-1]
    for k in range(len(cdf)):
        tt.cdf[k] = float(cdf[k])
