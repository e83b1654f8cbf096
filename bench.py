"""bench.py - CURIOUS training hot path on B200 (contract: see the repository prompt / DESIGN.md section 6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

metric   HER-relabelled transitions/s (BASELINE.json), Arm4-shaped synthetic replay:
         4 module buffers x 1e6 transitions (20 000 episodes x T=50, dimo=40, dimg=dimag=12, dimu=4, N=4).
step     ONE launch of the fused HER relabel+gather+reward+clip kernel over ROWS_PER_STEP rows
         (4096 batches of 256), LP-apportioned over the module buffers, Philox draws, producing the
         staged training batch (o, g, u, task_descr, o_2, r).
value    rows / device time (CUDA events), inputs resident in HBM, max over ranks, whole job.
e2e      the reference's training cycle (experiment/train.py:148-155) through the public plugin API with HOST episode
         buffers: DDPG.store_episode(host episodes) + 100 x DDPG.train() + DDPG.update_target_net() + device->host read
         of the critic losses; transitions consumed per second.
--impl reference   the oracle port of that SAME cycle (same n_batches) on the host cores (the reference is pure
         Python; TF1/mpi4py/gym_flowers are not installable, see DESIGN.md), one process per core up to 19.
Also on the line: update_us / updates_per_s (device-timed train()), get_actions latency (n = 2, 38; host in -> host
out), a rollout-inclusive cycle (50 x get_actions + store + 100 x train), the 19-worker-equivalent update, all of it
again on the Arm8 shape (BASELINE config 4), and - several ranks - the bit-exact parity of the in-launch gradient
exchange against an all-gather + rank-ordered sum (`exchange_parity`) and the per-rank scaling of the update.
--dump-outputs DIR   after the timed steps, rank 0 writes the staged batch of the last step (o, g, u, td, o_2, r) as
         DIR/<name>.npy, float32, the same seeded sample of DUMP_ROWS rows from every array (53 MB in all).  The inputs
         are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_MODULES = 4
T = 50
BUFFER_TRANSITIONS = 1000000
BATCH = 256
ROWS_PER_STEP = 1 << 20
CP = [0.05, 0.2, 0.1, 0.0]
CP8 = [0.05, 0.2, 0.1, 0.0, 0.0, 0.0, 0.0, 0.0]
EPS_TASK = 0.4
N_BATCHES = 100                # config.py:72 - the SAME cycle in both arms: store_episode + N_BATCHES x train + polyak
ROLLOUT_STEPS = T              # get_actions calls per rollout (rollout.py:217,226: one per env step)
HER_OUTPUTS = ('o', 'g', 'u', 'td', 'o_2', 'r')   # the staged training batch one HER step produces
DUMP_ROWS = 1 << 17            # --dump-outputs: rows sampled from the ROWS_PER_STEP of a step (x 101 floats x 4 B = 53 MB)
DUMP_SEED = 0


def workload_config():
    """The `config` of the JSON line - identical in both arms (--impl ours / reference)."""
    return {'workload': 'arm4-shaped: 4 module buffers x 1e6 transitions (T=50, dimo=40, dimg=12, dimu=4, N=4), '
                        'LP-apportioned (replay_task_cp_buffer, cp=%s, eps_task=%s), batch 256' % (CP, EPS_TASK),
            'cycle': 'store_episode(2 host episodes) + %d x train + update_target_net (experiment/train.py:148-155)'
                     % N_BATCHES,
            'her_step': '%d rows per fused HER launch (= %d batches of 256), Philox draws' % (ROWS_PER_STEP,
                                                                                              ROWS_PER_STEP // BATCH),
            'l2': 'inputs (1.44 GB of replay rows per rank) and outputs (0.42 GB) exceed the 126 MB L2',
            'rows_per_step': ROWS_PER_STEP, 'batch': BATCH, 'n_batches': N_BATCHES}


def algorithmic_bytes_per_transition(dims, n_modules, g_len=3):
    """SURVEY 8(d): reads o,o_2,u,td,g and the module slices of ag_2 / future ag; writes o,o_2,g,u,td,r."""
    rd = 4 * (2 * dims['o'] + dims['u'] + n_modules + dims['g'] + 2 * g_len)
    wr = 4 * (2 * dims['o'] + dims['g'] + dims['u'] + n_modules + 1)
    return rd + wr


class ClockSampler(threading.Thread):
    """SM clocks / throttle reasons while the timed region runs (B200_PROFILING.md's clocks line).  Sampled through NVML
    in-process every 4 ms (the HER region lasts ~10 ms; one `nvidia-smi` call takes longer than that), falling back to
    an `nvidia-smi --query-gpu` loop when pynvml is unavailable."""
    Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
    REASON_BITS = (('hw_slowdown', 0x8), ('hw_thermal_slowdown', 0x40), ('sw_thermal_slowdown', 0x20),
                   ('sw_power_cap', 0x4))

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.samples, self._stop_evt = index, [], threading.Event()
        self.source = 'nvidia-smi'
        self._nvml = self._handle = None
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            handle = None
            try:                                     # CUDA_VISIBLE_DEVICES may renumber: go by UUID when torch exposes it
                uuid = str(torch.cuda.get_device_properties(index).uuid)
                handle = pynvml.nvmlDeviceGetHandleByUUID(('GPU-' + uuid) if not uuid.startswith('GPU-') else uuid)
            except Exception:
                handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            pynvml.nvmlDeviceGetClockInfo(handle, pynvml.NVML_CLOCK_SM)
            self._nvml, self._handle, self.source = pynvml, handle, 'nvml'
        except Exception:
            self._nvml = None

    def _sample_nvml(self):
        n, h = self._nvml, self._handle
        sm = n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM)
        try:
            mask = n.nvmlDeviceGetCurrentClocksEventReasons(h)
        except Exception:
            mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        return [str(sm), str(mx)] + ['Active' if mask & bit else 'Not Active' for _, bit in self.REASON_BITS]

    def run(self):
        while not self._stop_evt.is_set():
            try:
                if self._nvml is not None:
                    self.samples.append(self._sample_nvml())
                else:
                    out = subprocess.check_output(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                                   '--format=csv,noheader,nounits'], timeout=5).decode().strip()
                    self.samples.append([x.strip() for x in out.split(',')])
            except Exception:
                pass
            self._stop_evt.wait(0.004 if self._nvml is not None else 0.05)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        sm, mx, reasons = [], 0, set()
        for s in self.samples:
            try:
                sm.append(float(s[0]))
                mx = max(mx, float(s[1]))
            except Exception:
                continue
            for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), s[2:]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': mx or None,
                'reasons': sorted(reasons), 'samples': len(sm), 'source': self.source}


TRAFFIC_FILE = 'profiles/r02_her_traffic.json'


def her_traffic_per_launch(rows_per_step):
    """DRAM bytes of one fused HER launch from the committed `ncu --set full` capture (profiles/), scaled to the
    rows of this launch; None if the capture is missing."""
    p = os.path.join(ROOT, TRAFFIC_FILE)
    try:
        t = json.load(open(p))
        return (t['dram_bytes_read'] + t['dram_bytes_write']) * rows_per_step / t['rows_per_launch']
    except Exception:
        return None


def measured_peak_hbm():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        try:
            return float(json.load(open(p))['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
        except Exception:
            pass
    return 6650.0, 'fallback (B200_PROFILING.md)'


# ------------------------------------------------------------------------------------------------
# workload construction
# ------------------------------------------------------------------------------------------------
def synth_dims(n_modules=N_MODULES):
    from curious_b200 import synth
    dims = synth.arm_dims(n_modules)
    ag_ids, g_ids = synth.arm_task_ids(n_modules)
    return dims, ag_ids, g_ids


def fill_buffer_on_device(buf, dims, seed):
    """Fill a ReplayBuffer to capacity with Arm-shaped synthetic episodes generated ON the device (same value
    structure as curious_b200.synth.make_episodes; input generation only)."""
    import torch
    from curious_b200.replay_buffer import StagedEpisodes
    g = torch.Generator(device=buf.device)
    g.manual_seed(seed)
    E, N = buf.size, dims['task_descr']
    chunk = 2000
    dev = buf.device
    for e0 in range(0, E, chunk):
        n = min(chunk, E - e0)
        o = torch.randn((n, T + 1, dims['o']), generator=g, device=dev).clamp_(-5, 5)
        ag0 = (torch.rand((n, 1, dims['ag']), generator=g, device=dev) - 0.5) * 0.3
        moving = (torch.rand((n, N), generator=g, device=dev) >= 0.3).float().repeat_interleave(dims['ag'] // N, dim=1)
        steps = torch.randn((n, T, dims['ag']), generator=g, device=dev) * 0.02 * moving[:, None, :]
        ag = torch.cat([ag0, ag0 + torch.cumsum(steps, dim=1)], dim=1).contiguous()
        task = torch.randint(0, N, (n,), generator=g, device=dev)
        td = torch.nn.functional.one_hot(task, N).float()[:, None, :].expand(n, T, N).contiguous()
        gv = (torch.rand((n, dims['g']), generator=g, device=dev) - 0.5) * 0.3
        gmask = td[:, 0, :].repeat_interleave(dims['g'] // N, dim=1)
        gg = (gv * gmask)[:, None, :].expand(n, T, dims['g']).contiguous()
        u = torch.rand((n, T, dims['u']), generator=g, device=dev) * 2 - 1
        change = ((ag[:, :1, :] - ag[:, 1:, :]).abs() > 1e-3).float().contiguous()
        info = (torch.rand((n, T, 1), generator=g, device=dev) < 0.25).float()
        staged = StagedEpisodes.from_device(dict(o=o.contiguous(), ag=ag, g=gg, u=u.contiguous(), task_descr=td,
                                                 change=change, info=info), buf.layout)
        staged.store([(i, buf.storage, buf.cold, e0 + i) for i in range(n)])
        torch.cuda.synchronize()
    buf.current_size = E
    buf.n_transitions_stored = E * T


def build_gpu_workload(device, seed, n_modules=N_MODULES):
    """Arm4-shaped (BASELINE configs 2/3) or Arm8-shaped (config 4: 4 distractor modules, buffers 6..8 alias buffer 5,
    ddpg.py:104-110) replay + agent factory."""
    from curious_b200 import her, synth
    from curious_b200.ddpg import DDPG
    from curious_b200.replay_buffer import ReplayBuffer
    from curious_b200.reward import ModuleDistanceReward
    dims, ag_ids, g_ids = synth_dims(n_modules)
    sampler = her.make_sample_multi_task_her_transitions('her', 4, 'replay_task_cp_buffer',
                                                         ModuleDistanceReward(ag_ids, g_ids), tasks_ag_id=ag_ids,
                                                         tasks_g_id=g_ids)
    sampler.rng = 'philox'
    sampler.seed = seed
    shapes = synth.buffer_shapes(dims, T)
    n_real = min(n_modules, 5)                         # modules >= 5 are never stored (ddpg.py:183): buffers 6.. alias 5
    buffers = [ReplayBuffer(shapes, BUFFER_TRANSITIONS if 0 < i <= n_real else T, T, sampler, device=device)
               for i in range(n_modules + 1)]          # buffer 0 is never written by the reference (ddpg.py:191)
    for i in range(1, n_real + 1):
        fill_buffer_on_device(buffers[i], dims, seed * 100 + i + 10 * n_modules)
    for i in range(6, n_modules + 1):
        buffers[i] = buffers[5]
    gamma = 1. - 1. / T
    cp = np.array(CP if n_modules == 4 else CP8)

    def make_agent(batch_size=BATCH, structure='curious', task_replay='replay_task_cp_buffer', hidden=256, **extra):
        extra.setdefault('grad_exchange', os.environ.get('CUR_GRAD_EXCHANGE', 'auto'))
        a = DDPG(input_dims=dims, hidden=hidden, layers=3, network_class='baselines.her.actor_critic:MultiTaskActorCritic',
                 polyak=0.95, batch_size=batch_size, Q_lr=0.001, pi_lr=0.001, norm_eps=0.01, norm_clip=5, max_u=1.,
                 action_l2=1.0, clip_obs=200., scope='ddpg', T=T, rollout_batch_size=2,
                 subtract_goals=lambda a, b: a - b, relative_goals=False, clip_pos_returns=True,
                 clip_return=1. / (1. - gamma), normalize_obs=False, sample_transitions=sampler, gamma=gamma,
                 buffers=list(buffers), tasks_ag_id=ag_ids, tasks_g_id=g_ids, task_replay=task_replay,
                 eps_task=EPS_TASK, structure=structure, her_rng='philox', seed=0, device=device, **extra)
        a.cp = cp
        return a

    agent = make_agent()
    agent.make_agent = make_agent
    agent.bench_cp = cp
    return agent, sampler, buffers, dims, ag_ids, g_ids


def update_flops(dims, n_modules, batch, hidden=256):
    """SURVEY 8(d): algorithmic FLOPs of one DDPG update (forward of main/target pi and the three Q passes, critic,
    actor-through-critic and actor backward chains)."""
    H, B = hidden, batch
    s_pi, s_q = dims['o'] + n_modules, dims['o'] + n_modules + dims['u']
    f_pi = 2 * B * ((s_pi + dims['g']) * H + 2 * H * H + H * dims['u'])
    f_q = 2 * B * ((s_q + dims['g']) * H + 2 * H * H + H)
    fwd = 2 * f_pi + 3 * f_q
    bwd = (2 * f_q - 2 * B * (s_q + dims['g']) * H) + (f_q - 2 * B * (s_q + dims['g'] - dims['u']) * H) + \
          (2 * f_pi - 2 * B * (s_pi + dims['g']) * H)
    return fwd + bwd


def time_updates(fn, n, torch):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def schedule_name(a, rows):
    """Which implementation of the update DDPG.train() runs at `rows` rows per launch."""
    import ctypes as C
    from curious_b200 import _lib
    if a._use_rows(rows):
        return 'rows (FFMA2 row clusters)'
    lib = _lib.load()
    if lib.cur_ddpg_uses_chain(C.byref(a.net.desc), rows):
        return 'chain (tcgen05, fused actor / critic chains + split-K weight gradients)'
    if lib.cur_ddpg_uses_tensor_cores(C.byref(a.net.desc), rows):
        return 'levels (tcgen05)'
    return 'levels (FFMA)'


def large_batch_sweep(agent, dims, torch):
    """BASELINE config 5: per-GPU batch sweep of the DDPG update through DDPG.train() (HER sample + grads + Adam in
    one CUDA graph) and structure='task_experts' as grouped launches.  At batch >= 1024 the hidden-layer GEMMs run on
    tcgen05 (3xTF32): `tensor_frac` = 3 x algorithmic FLOP/s / (measured dense bf16 peak / 2), i.e. against the TF32
    rate of the tensor pipe, all 3 error-compensation passes counted."""
    from curious_b200 import _lib
    from curious_b200.experts import TaskExperts
    import ctypes as C
    try:
        bf16 = float(json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))['bf16_tflops'])
    except Exception:
        bf16 = 2250.0 * 0.745
    sweep = []
    for b in (256, 512, 1024, 2048, 4096, 4864, 16384):
        a = agent if b == BATCH else agent.make_agent(batch_size=b)
        ms = time_updates(a.train, 200 if b <= 1024 else 40, torch)
        fl = update_flops(dims, N_MODULES, b)
        tc = bool(_lib.load().cur_ddpg_uses_tensor_cores(C.byref(a.net.desc), b)) and not a._use_rows(b)
        sweep.append({'batch': b, 'update_us': 1e3 * ms, 'updates_per_s': 1e3 / ms, 'transitions_per_s': 1e3 * b / ms,
                      'tflops': fl / (ms * 1e-3) / 1e12, 'schedule': schedule_name(a, b),
                      'tensor_cores': tc, 'tensor_frac': (3 * fl / (ms * 1e-3) / 1e12) / (bf16 / 2) if tc else None})
        if b != BATCH:
            del a
            torch.cuda.empty_cache()
    # hidden widths other than the default (config.py:25): zero-padded onto the 256-wide kernels (DDPG pad_hidden) next to
    # the dependency-level kernels at the true width
    widths = []
    for h in (64, 128):
        rec = {'hidden': h, 'batch': BATCH}
        for tag, kw in (('padded_rows_update_us', dict(pad_hidden='auto')), ('levels_update_us', dict(pad_hidden=False))):
            a = agent.make_agent(hidden=h, **kw)
            rec[tag] = 1e3 * time_updates(a.train, 200, torch)
            rec[tag.replace('update_us', 'schedule')] = schedule_name(a, BATCH)
            del a
            torch.cuda.empty_cache()
        widths.append(rec)
    experts = []
    for b in (256, 4096):
        ps = [agent.make_agent(batch_size=b, structure='task_experts', task_replay='replay_current_task_buffer', t_id=t,
                               update_schedule='auto') for t in range(N_MODULES)]
        for p in ps:
            p.cp = np.array(CP)
        grp = TaskExperts(ps)
        ms = time_updates(grp.train, 100 if b <= 1024 else 20, torch)
        experts.append({'experts': N_MODULES, 'batch': b, 'round_us': 1e3 * ms, 'expert_updates_per_s': 1e3 * N_MODULES / ms,
                        'mode': 'sequential rows' if all(p._use_rows(b) for p in ps) else 'grouped levels'})
        del grp, ps
        torch.cuda.empty_cache()
    return {'batch_sweep': sweep, 'hidden_widths': widths, 'task_experts': experts, 'tf32_peak_tflops_assumed': bf16 / 2}


def her_step_segments(buffers, rows, cp):
    """LP apportioning of `rows` over the DISTINCT module buffers (aliased distractor buffers are sampled through every
    module that points at them, like DDPG.sample_batch does, ddpg.py:326-336)."""
    from curious_b200 import apportion
    sizes = [b.current_size for b in buffers]
    prop = apportion.proportions_curious(sizes, T, rows, 'replay_task_cp_buffer', np.array(cp), EPS_TASK)
    return [(buffers[i].device_view(), int(prop[i]), i - 1) for i in range(1, len(buffers)) if prop[i] > 0]


def her_line(sampler, buffers, dims, n_modules, cp, torch, label):
    """One fused HER launch over ROWS_PER_STEP rows on this shape: transitions/s and fraction of the HBM roofline."""
    segs = her_step_segments(buffers, ROWS_PER_STEP, cp)
    out = {}
    want = HER_OUTPUTS
    ms = time_updates(lambda: sampler.sample_device(segs, ROWS_PER_STEP, clip_obs=200.0, want=want, out=out), 20, torch)
    bpt = algorithmic_bytes_per_transition(dims, n_modules)
    peak, _ = measured_peak_hbm()
    achieved = bpt * ROWS_PER_STEP / (ms * 1e-3) / 1e9
    del out
    torch.cuda.empty_cache()
    return {'transitions_per_s': ROWS_PER_STEP / (ms * 1e-3), 'ms_per_launch': ms, 'algorithmic_bytes_per_transition': bpt,
            'achieved_gbs': achieved, 'frac_of_hbm_peak': achieved / peak, 'workload': label}


def dump_outputs(out, directory):
    """The arrays one HER step hands its caller (sample_device's dict of [ROWS_PER_STEP, dim] float32 device tensors),
    as directory/<name>.npy: the rows of a fixed seeded sample, the same rows in every array."""
    import torch
    os.makedirs(directory, exist_ok=True)
    rows = np.sort(np.random.RandomState(DUMP_SEED).choice(ROWS_PER_STEP, DUMP_ROWS, replace=False))
    sel = None
    for name, t in out.items():
        if name.startswith('_'):                          # references the launch keeps alive, not outputs
            continue
        if sel is None:
            sel = torch.from_numpy(rows).to(t.device)
        np.save(os.path.join(directory, name + '.npy'), t.index_select(0, sel).cpu().numpy().astype(np.float32))


def build_cpu_workload(seed, episodes_per_buffer):
    from curious_b200 import synth
    from oracle import ddpg_oracle, her_oracle, replay_oracle
    from oracle.reward_oracle import ModuleDistanceReward
    dims, ag_ids, g_ids = synth_dims()
    sampler = her_oracle.make_sample_multi_task_her_transitions('her', 4, 'replay_task_cp_buffer',
                                                                ModuleDistanceReward(ag_ids, g_ids),
                                                                tasks_ag_id=ag_ids, tasks_g_id=g_ids)
    shapes = synth.buffer_shapes(dims, T)
    buffers = [replay_oracle.ReplayBufferOracle(shapes, (episodes_per_buffer if i > 0 else 1) * T, T, sampler)
               for i in range(N_MODULES + 1)]
    rng = np.random.RandomState(seed)
    for i in range(1, N_MODULES + 1):
        for e0 in range(0, episodes_per_buffer, 2000):
            n = min(2000, episodes_per_buffer - e0)
            buffers[i].store_episode(synth.make_episodes(rng, n, T, dims))
    gamma = 1. - 1. / T
    agent = ddpg_oracle.DDPGOracle(
        input_dims=dims, hidden=256, layers=3, polyak=0.95, batch_size=BATCH, Q_lr=0.001, pi_lr=0.001, norm_eps=0.01,
        norm_clip=5, max_u=1., action_l2=1.0, clip_obs=200., T=T, rollout_batch_size=2, relative_goals=False,
        clip_pos_returns=True, clip_return=1. / (1. - gamma), normalize_obs=False, sample_transitions=sampler,
        gamma=gamma, buffers=buffers, structure='curious', tasks_ag_id=ag_ids, tasks_g_id=g_ids,
        task_replay='replay_task_cp_buffer', eps_task=EPS_TASK, weights_rng=np.random.RandomState(0))
    agent.cp = np.array(CP)
    return agent, dims


def cpu_sampler_baseline(seconds=12.0):
    """The oracle's DDPG.sample_batch (apportion + per-buffer HER sampler + concat + shuffle + preprocess) on one
    core, full-size buffers: transitions/s.  kind = 'port' (restatement of her.py / replay_buffer.py / ddpg.py)."""
    import contextlib
    try:
        from threadpoolctl import threadpool_limits
        ctx = threadpool_limits(limits=1)
    except Exception:
        ctx = contextlib.nullcontext()
    with ctx:
        agent, _ = build_cpu_workload(0, BUFFER_TRANSITIONS // T)
        np.random.seed(0)
        for _ in range(20):
            agent.sample_batch()
        n, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < seconds:
            agent.sample_batch()
            n += 1
        dt = time.perf_counter() - t0
    return {'value': n * BATCH / dt, 'unit': 'transitions/s', 'cores': 1, 'kind': 'port',
            'sample': '%d sample_batch calls x %d rows on 4 x 1e6-transition float64 buffers, 1 thread '
                      '(oracle port of her.py/replay_buffer.py/ddpg.py sample_batch)' % (n, BATCH)}


def _ref_worker(rank, n_steps, n_warm, updates, episodes_per_buffer, q):
    os.environ['OMP_NUM_THREADS'] = '1'
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=1)
    except Exception:
        pass
    agent, dims = build_cpu_workload(rank, episodes_per_buffer)
    from curious_b200 import synth
    rng = np.random.RandomState(1000 + rank)
    np.random.seed(1000000 * rank)
    q.put(('ready', rank))
    times = []
    for s in range(n_warm + n_steps):
        ep = synth.make_episodes(rng, 2, T, dims, change_dtype=bool)
        t0 = time.perf_counter()
        agent.store_episode(ep, np.array(CP), 2 * (s + 1))
        for _ in range(updates):
            agent.train()
        agent.update_target_net()
        times.append(time.perf_counter() - t0)
    q.put(('done', rank, times[n_warm:]))


def run_reference_arm(args):
    """The training cycle of the reference restated on the CPU (oracle port), one single-threaded process per
    worker like the reference's `mpirun -np 19 --bind-to core` (train.py:221-231); no all-reduce is modelled, so
    this over-estimates the CPU arm.  Each step is ONE cycle of the ours-arm's e2e: store_episode + N_BATCHES x train +
    update_target_net (a bounded sample of the job: `steps` cycles per worker)."""
    import multiprocessing as mp
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    procs = max(1, min(19, cores))
    episodes = BUFFER_TRANSITIONS // T
    # bound memory: each worker owns 4 float64 buffers of 0.69 GB
    try:
        import psutil
        avail = psutil.virtual_memory().available
        procs = max(1, min(procs, int(avail * 0.6 // (4 * 0.7e9))))
    except Exception:
        pass
    ctx = mp.get_context('fork')
    q = ctx.Queue()
    workers = [ctx.Process(target=_ref_worker, args=(r, args.steps, args.warmup, N_BATCHES, episodes, q))
               for r in range(procs)]
    for w in workers:
        w.start()
    done = {}
    while len(done) < procs:
        msg = q.get()
        if msg[0] == 'done':
            done[msg[1]] = msg[2]
    for w in workers:
        w.join()
    per_step = np.max(np.array([done[r] for r in range(procs)]), axis=0)      # slowest worker per step
    total = float(per_step.sum())
    value = procs * N_BATCHES * BATCH * args.steps / total
    line = {
        'impl': 'reference', 'metric': 'HER-relabelled transitions/s', 'value': value, 'unit': 'transitions/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * total / args.steps,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(),
        'what': 'CPU arm: the training cycle of `config.cycle` on %d single-threaded worker processes (one per core up '
                'to 19, like mpirun -np 19 --bind-to core); value = transitions consumed by the updates per second, '
                'all workers' % procs,
        'cpu_baseline': {'value': value, 'unit': 'transitions/s', 'cores': procs, 'kind': 'port',
                         'sample': '%d single-threaded worker processes x %d cycles x %d updates of batch %d (oracle '
                                   'NumPy port of her.py/replay_buffer.py/ddpg.py/mpi_adam.py; TF1 graph restated in '
                                   'float32 NumPy/BLAS; no all-reduce modelled)' % (procs, args.steps, N_BATCHES, BATCH)},
        'e2e': {'value': value, 'unit': 'transitions/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'updates_per_s': procs * N_BATCHES * args.steps / total,
        'update_us_per_worker': 1e6 * total / (N_BATCHES * args.steps),
        'host_cores': cores,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
def measure_agent(agent, dims, n_modules, world, rank, barrier, torch, dist, device, full=True):
    """Everything the line reports per shape (Arm4 / Arm8): device-timed update, the e2e training cycle through the
    plugin API with host episodes, get_actions latency, the rollout-inclusive cycle, the 19-worker-equivalent update."""
    from curious_b200 import synth
    cp = agent.bench_cp
    res = {}
    # ---- DDPG updates/s: device-timed train() (sample + grads + gradient exchange + Adam) through the public API
    for _ in range(5):
        agent.train()
    barrier()
    n_upd = 200
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n_upd):
        agent.train()
    e1.record()
    barrier()
    upd_ms = e0.elapsed_time(e1)
    # ---- e2e: training cycles through the plugin API with host episode buffers
    rng = np.random.RandomState(99 + rank)
    host_eps = [synth.make_episodes(rng, 2, T, dims, change_dtype=bool) for _ in range(8)]
    h2d = sum(np.asarray(v).size * 4 for v in host_eps[0].values())

    def cycle(i):
        agent.store_episode({k: v for k, v in host_eps[i % len(host_eps)].items()}, cp, 2 * (i + 1))
        losses = [agent.train()[0] for _ in range(N_BATCHES)]
        agent.update_target_net()
        return torch.stack([l.tensor for l in losses]).cpu().numpy()          # device->host read of the results

    for i in range(3):
        cycle(i)
    barrier()
    n_cyc = 10
    t0 = time.perf_counter()
    for i in range(n_cyc):
        out = cycle(3 + i)
    barrier()
    cyc_s = time.perf_counter() - t0
    # ---- get_actions latency, host arrays in -> host actions out (rollout.py:217,226: one call per env step; n = 2 is
    # the reference's rollout_batch_size, n = 38 the 19 workers' environments batched on one rank)
    ga = {}
    for n in (2, 38):
        o = rng.standard_normal((n, dims['o'])).astype(np.float32)
        ag = rng.uniform(-0.15, 0.15, (n, dims['ag'])).astype(np.float32)
        g = rng.uniform(-0.15, 0.15, (n, dims['g'])).astype(np.float32)
        td = np.eye(n_modules, dtype=np.float32)[rng.randint(0, n_modules, n)]
        for _ in range(20):
            agent.get_actions(o, ag, g, task_descr=td, noise_eps=0.2, random_eps=0.3)
        reps = 300
        t0 = time.perf_counter()
        for _ in range(reps):
            agent.get_actions(o, ag, g, task_descr=td, noise_eps=0.2, random_eps=0.3)
        dt = time.perf_counter() - t0
        ga['n%d' % n] = {'us_per_call': 1e6 * dt / reps, 'actions_per_s': n * reps / dt}
    # ---- rollout-inclusive cycle: ROLLOUT_STEPS x get_actions(n = 2) (the device round trips of one rollout; the
    # environment itself stays on the host and is not modelled) + store_episode + N_BATCHES x train + update_target_net
    o2 = rng.standard_normal((2, dims['o'])).astype(np.float32)
    ag2 = rng.uniform(-0.15, 0.15, (2, dims['ag'])).astype(np.float32)
    g2 = rng.uniform(-0.15, 0.15, (2, dims['g'])).astype(np.float32)
    td2 = np.eye(n_modules, dtype=np.float32)[[0, 1]]

    def rollout_cycle(i):
        for _ in range(ROLLOUT_STEPS):
            agent.get_actions(o2, ag2, g2, task_descr=td2, noise_eps=0.2, random_eps=0.3)
        return cycle(i)

    rollout_cycle(0)
    barrier()
    n_rc = 5
    t0 = time.perf_counter()
    for i in range(n_rc):
        rollout_cycle(20 + i)
    barrier()
    rc_s = time.perf_counter() - t0
    # ---- 19-worker-equivalent (BASELINE config 4 / SURVEY 8e): the reference's 19 MPI workers spread over the ranks,
    # ceil(19 / world) batch-256 workers per GPU, gradients summed per rank and across ranks, one Adam step
    k19 = -(-19 // world)
    agent19 = agent.make_agent(workers_per_rank=k19)
    for _ in range(3):
        agent19.train()
    barrier()
    n19 = 30
    e0.record()
    for _ in range(n19):
        agent19.train()
    e1.record()
    barrier()
    upd19_ms = e0.elapsed_time(e1)
    sched19 = schedule_name(agent19, agent19._graph_rows)
    exch19 = 'tile' if agent19._xchg is not None else ('p2p' if agent19._peer is not None else ('nccl' if world > 1 else None))
    del agent19
    torch.cuda.empty_cache()
    vals = [upd_ms, cyc_s, upd19_ms, rc_s, ga['n2']['us_per_call'], ga['n38']['us_per_call']]
    if world > 1:
        tt = torch.tensor(vals, device=device, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        vals = [float(x) for x in tt.cpu()]
    upd_ms, cyc_s, upd19_ms, rc_s, ga2, ga38 = vals
    res['update_us'] = 1e3 * upd_ms / n_upd
    res['updates_per_s'] = world * n_upd / (upd_ms * 1e-3)
    res['update_schedule'] = schedule_name(agent, BATCH)
    res['grad_exchange'] = ('tile' if getattr(agent, '_xchg', None) is not None else
                            'p2p' if getattr(agent, '_peer', None) is not None else 'nccl') if world > 1 else None
    if getattr(agent, '_xchg', None) is not None:
        res['grad_exchange_mode'] = int(agent._xchg.mode)
    res['e2e'] = {'value': world * n_cyc * N_BATCHES * BATCH / cyc_s, 'unit': 'transitions/s',
                  'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': int(out.nbytes),
                  'what': 'DDPG.store_episode(host) + %d x DDPG.train() + update_target_net + loss readback per cycle'
                          % N_BATCHES, 'cycle_ms': 1e3 * cyc_s / n_cyc,
                  'updates_per_s': world * n_cyc * N_BATCHES / cyc_s}
    res['get_actions'] = {'n2_us_per_call': ga2, 'n38_us_per_call': ga38, 'n38_actions_per_s': 38 * 1e6 / ga38,
                          'what': 'DDPG.get_actions(host o, ag, g, task_descr; noise_eps 0.2, random_eps 0.3) -> host '
                                  'actions, wall clock per call, max over ranks'}
    res['rollout_cycle'] = {'cycle_ms': 1e3 * rc_s / n_rc,
                            'transitions_per_s': world * n_rc * N_BATCHES * BATCH / rc_s,
                            'what': '%d x get_actions(n = 2) + store_episode + %d x train + update_target_net + loss '
                                    'readback (environment stepping not modelled)' % (ROLLOUT_STEPS, N_BATCHES)}
    res['workers19_equivalent'] = {'workers_per_rank': k19, 'workers': k19 * world, 'global_batch': k19 * world * BATCH,
                                   'update_us': 1e3 * upd19_ms / n19, 'updates_per_s': n19 / (upd19_ms * 1e-3),
                                   'transitions_per_s': k19 * world * BATCH * n19 / (upd19_ms * 1e-3),
                                   'schedule': sched19, 'grad_exchange': exch19}
    return res


def exchange_parity(agent, world, rank, torch, dist, device, n_updates=8):
    """Several ranks: the same updates through the in-launch tile exchange and through an all-gather + RANK-ORDERED sum +
    Adam launch on identical gradients (fresh twin agents: same weights, same replay, same Philox counters).  The
    peer-memory forms of the exchange (modes 0 / 1) sum in rank order: bit-identical parameters on every rank, asserted
    bit for bit.  The NVLS form (mode 2, the default from 4 ranks) sums in the switch: parameters bit-identical on every
    rank and within 1e-6 of the rank-ordered result; the mode-1 bit-for-bit check runs beside it.  Also reports the
    distance to NCCL's own all-reduce, whose summation order is its algorithm's (equal for 2 ranks, a few ulp otherwise)."""
    from curious_b200 import parallel
    thetas, modes = {}, {}
    for name, kw, ordered in (('tile', dict(grad_exchange='auto'), False), ('ordered', dict(grad_exchange='nccl'), True),
                              ('nccl', dict(grad_exchange='nccl'), False), ('mode1', dict(grad_exchange='auto', xchg_mode=1), False)):
        if name == 'mode1' and modes.get('tile') != 2:
            continue
        parallel.ORDERED_ALLREDUCE = ordered
        a = agent.make_agent(**kw)
        for _ in range(n_updates):
            a.train()
        a.update_target_net()
        torch.cuda.synchronize()
        thetas[name] = a.theta_main.clone()
        kind = 'tile' if a._xchg is not None else ('p2p' if a._peer is not None else 'nccl')
        modes[name] = int(a._xchg.mode) if a._xchg is not None else None
        if name == 'tile':
            used = kind
        del a
        torch.cuda.empty_cache()
        dist.barrier()
    parallel.ORDERED_ALLREDUCE = False
    nvls = modes['tile'] == 2
    d_ord = (thetas['tile'] - thetas['ordered']).abs().max()
    dist.all_reduce(d_ord, op=dist.ReduceOp.MAX)
    if nvls:
        bad = torch.tensor([0 if float(d_ord.item()) <= 1e-6 else 1], device=device)
        bad += 0 if torch.equal(thetas['mode1'], thetas['ordered']) else 1
    else:
        bad = torch.tensor([0 if torch.equal(thetas['tile'], thetas['ordered']) else 1], device=device)
    # ... and every rank holds rank 0's parameters
    ref = thetas['tile'].clone()
    dist.broadcast(ref, src=0)
    bad += 0 if torch.equal(ref, thetas['tile']) else 1
    dist.all_reduce(bad)
    diff = (thetas['tile'] - thetas['nccl']).abs().max()
    dist.all_reduce(diff, op=dist.ReduceOp.MAX)
    return {'exchange_parity': int(bad.item()) == 0, 'exchange': used, 'exchange_mode': modes['tile'], 'updates': n_updates,
            'exchange_parity_rule': ('parameters bit-identical on every rank and within 1e-6 of the rank-ordered sum (NVLS: '
                                     'the switch fixes the summation order); the peer-memory mode 1 bit-equal to the '
                                     'rank-ordered sum in the same run' if nvls else
                                     'parameters bit-equal to the rank-ordered sum on every rank'),
            'max_abs_diff_vs_rank_ordered_sum': float(d_ord.item()),
            'max_abs_diff_vs_nccl_allreduce': float(diff.item()),
            'against': 'all-gather + rank-ordered float32 sum + Adam launch (parallel.ORDERED_ALLREDUCE)'}


def nvls_exchange(agent, world, torch, dist, device, n_updates=8):
    """Several ranks: the NVLS form of the tile exchange (cur_xchg_ctx mode 2: multimem.ld_reduce through the NVSwitch,
    one multicast store for the result) next to the default - per-rank update time, parameters identical on every rank,
    distance to the rank-ordered sum (the in-switch summation order is the hardware's)."""
    from curious_b200 import parallel
    try:
        a = agent.make_agent(grad_exchange='tile', xchg_mode='nvls')
    except Exception as e:                      # no multicast support on this system / torch build
        return {'unavailable': '%s: %s' % (type(e).__name__, str(e)[:200])}
    for _ in range(n_updates):
        a.train()
    a.update_target_net()
    torch.cuda.synchronize()
    theta = a.theta_main.clone()
    parallel.ORDERED_ALLREDUCE = True
    b = agent.make_agent(grad_exchange='nccl')
    for _ in range(n_updates):
        b.train()
    b.update_target_net()
    torch.cuda.synchronize()
    parallel.ORDERED_ALLREDUCE = False
    diff = (theta - b.theta_main).abs().max()
    dist.all_reduce(diff, op=dist.ReduceOp.MAX)
    del b
    ref = theta.clone()
    dist.broadcast(ref, src=0)
    bad = torch.tensor([0 if torch.equal(ref, theta) else 1], device=device)
    dist.all_reduce(bad)
    for _ in range(5):
        a.train()
    ms = time_updates(a.train, 200, torch)
    tt = torch.tensor([ms], device=device, dtype=torch.float64)
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    del a
    torch.cuda.empty_cache()
    dist.barrier()
    b = agent.make_agent(grad_exchange='tile', xchg_mode=1 if world > 2 else 0)
    for _ in range(5):
        b.train()
    ms1 = time_updates(b.train, 200, torch)
    t1 = torch.tensor([ms1], device=device, dtype=torch.float64)
    dist.all_reduce(t1, op=dist.ReduceOp.MAX)
    del b
    torch.cuda.empty_cache()
    dist.barrier()
    return {'per_rank_update_us': 1e3 * float(tt.item()), 'peer_memory_mode_per_rank_update_us': 1e3 * float(t1.item()),
            'identical_on_every_rank': int(bad.item()) == 0,
            'max_abs_diff_vs_rank_ordered_sum': float(diff.item()), 'updates': n_updates,
            'what': 'tile exchange mode 2: partials in place, multimem.ld_reduce by the owning rank, Adam, one multicast '
                    'store of the stepped parameters (csrc/ddpg_rows.cu, parallel.TileGradExchange(mode="nvls"))'}


def run_ours(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    device = torch.device('cuda', local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=device)
    from curious_b200 import _lib
    _lib.load()
    agent, sampler, buffers, dims, ag_ids, g_ids = build_gpu_workload(device, seed=1 + rank)
    segs = her_step_segments(buffers, ROWS_PER_STEP, CP)
    want = HER_OUTPUTS
    out = {}

    def her_step():
        return sampler.sample_device(segs, ROWS_PER_STEP, clip_obs=200.0, want=want, out=out)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        her_step()
    barrier()
    clocks = ClockSampler(local)
    clocks.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(args.steps):
        her_step()
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    if args.dump_outputs and rank == 0:
        dump_outputs(out, args.dump_outputs)
    del out
    arm4 = measure_agent(agent, dims, N_MODULES, world, rank, barrier, torch, dist, device)
    clock_info = clocks.stop()
    if world > 1:
        tt = torch.tensor([ms], device=device, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt.item())
    # ---- several ranks: how much one rank's update costs next to a world of one on the same GPU, and the parity check
    scaling = parity = nvls = None
    if world > 1:
        solo = agent.make_agent(comm=False)
        for _ in range(5):
            solo.train()
        solo_ms = time_updates(solo.train, 200, torch)
        del solo
        tt = torch.tensor([solo_ms], device=device, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        solo_us = 1e3 * float(tt.item())
        scaling = {'single_rank_update_us': solo_us, 'per_rank_update_us': arm4['update_us'],
                   'efficiency': solo_us / arm4['update_us'],
                   'what': 'device-timed train() of one rank alone (comm=False, same GPU, same run) / the same inside the '
                           '%d-rank job: the weak-scaling efficiency of the path that has a collective' % world}
        parity = exchange_parity(agent, world, rank, torch, dist, device)
        # the NVLS form of the exchange next to the default: opt-in (its setup goes through the system's multicast support)
        nvls = nvls_exchange(agent, world, torch, dist, device) if os.environ.get('CUR_BENCH_NVLS') == '1' else None
    # ---- BASELINE config 4: the Arm8 shape (dimo 64, dimg 24, N 8, buffers 6..8 aliased), same measurements
    agent8, sampler8, buffers8, dims8, _, _ = build_gpu_workload(device, seed=50 + rank, n_modules=8)
    arm8 = measure_agent(agent8, dims8, 8, world, rank, barrier, torch, dist, device)
    her8 = None
    if world == 1:
        her8 = her_line(sampler8, buffers8, dims8, 8, CP8, torch,
                        'arm8-shaped: 5 distinct module buffers x 1e6 transitions (dimo=64, dimg=24, dimu=4, N=8), '
                        '%d rows per launch' % ROWS_PER_STEP)
    if world > 1 and parity is not None and not parity['exchange_parity']:
        if rank == 0:
            print(json.dumps({'error': 'exchange_parity failed', 'detail': parity}))
        dist.destroy_process_group()
        sys.exit(3)
    if rank == 0:
        peak, peak_src = measured_peak_hbm()
        bpt = algorithmic_bytes_per_transition(dims, N_MODULES)
        kernel_ms = ms / args.steps                       # one step == one launch of the fused kernel
        achieved = bpt * ROWS_PER_STEP / (kernel_ms * 1e-3) / 1e9
        line = {
            'metric': 'HER-relabelled transitions/s', 'value': world * ROWS_PER_STEP * args.steps / (ms * 1e-3),
            'unit': 'transitions/s', 'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3),
            'ms_per_step': kernel_ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic',
            'config': workload_config(),
            'roofline': {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                         'traffic': her_traffic_per_launch(ROWS_PER_STEP),
                         'traffic_source': 'static: dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` '
                                           'capture of this kernel on this workload (%s), scaled to the rows of a '
                                           'launch; not measured in this run' % TRAFFIC_FILE,
                         'peak_source': peak_src,
                         'algorithmic_bytes': bpt * ROWS_PER_STEP, 'algorithmic_bytes_per_transition': bpt,
                         'kernel': 'her_sample_kernel'},
            'e2e': arm4['e2e'],
            'gpu_launches': args.steps,
            'clocks': clock_info,
            'updates_per_s': arm4['updates_per_s'], 'update_us': arm4['update_us'],
            'update_schedule': arm4['update_schedule'], 'grad_exchange': arm4['grad_exchange'],
            'get_actions': arm4['get_actions'], 'rollout_cycle': arm4['rollout_cycle'],
            'workers19_equivalent': arm4['workers19_equivalent'],
            'arm8': dict(arm8, workload='arm8-shaped (BASELINE config 4): dimo=64, dimg=dimag=24, dimu=4, N=8, 5 distinct '
                                        'module buffers x 1e6 transitions, buffers 6..8 alias buffer 5, modules >= 5 never '
                                        'stored (ddpg.py:104-110,183), cp=%s' % CP8),
        }
        if 'grad_exchange_mode' in arm4:
            line['grad_exchange_mode'] = arm4['grad_exchange_mode']
        if scaling is not None:
            line['scaling_e2e'] = scaling
            line.update(parity)
            if nvls is not None:
                line['nvls_exchange'] = nvls
        if her8 is not None:
            line['her_arm8'] = her8
        if world == 1 and not args.no_sweep:
            line['ddpg_update'] = large_batch_sweep(agent, dims, torch)
        if world == 1 and not args.no_cpu_baseline:
            line['cpu_baseline'] = cpu_sampler_baseline()
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=50)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-sweep', action='store_true', help='skip the batch sweep / task_experts section')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write a seeded sample of the last timed step\'s outputs as DIR/<name>.npy (float32)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes the outputs of --impl ours')
    if args.impl == 'reference':
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
