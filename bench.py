#!/usr/bin/env python
"""bench.py -- agent-steps/s of the mrs-gym step path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload c5|c2|c3|c4] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

Workload (default c5 = BASELINE.json configs[4], the config the metric is quoted on; it fits one
GPU): 65536 envs x 8 agents PER GPU (weak scaling), ACTION_TYPE set_speeds, K_HOPS=3, COMM_RANGE 2.0
(RETURN_A), built-in state_fn cat(pos, vel).  A "step" is one env.step of all envs = ONE launch of
step_group_kernel that reads and writes the whole state in HBM.

Timed region: `steps` steps issued as CUDA-graph replays of T-step rollouts (T = min(steps, 100);
Swarm.capture_rollout; actions of every step are distinct device buffers) plus steps % T plain
launches, bracketed by barrier + synchronize, CUDA events
on the launching stream, max over ranks.  L2: no flush in the headline loop -- per step the kernel
streams actions + X + A (38 MB at c5) that are distinct every step, while the 27 MB state is
re-read from wherever the previous step left it (that is the real access pattern of a rollout);
`l2_flushed` reports the same step timed one launch at a time with a 512 MB read-flush in between.

e2e: the same steps through mrs_step_host (C ABI, pinned HOST buffers): H2D actions, step, D2H of the
newest X and A slices, stream sync -- every step.

--dump-outputs DIR: after the timed region, what its last step handed the caller -- the newest X and A slices
and the swarm state -- is written as DIR/<name>.npy (float32; rank 0's shard).  The inputs are seeded, so two
builds run with the same arguments can be compared output for output.  The benchmark writes nothing else: the
tree it runs from may be read-only.

--impl reference: the CPU arm.  The reference is pure Python over PyBullet (not installable here,
no network), so the CPU implementation that can run is the oracle port (oracle/spec.py, numpy,
float64 Bullet restatement) on all host cores, one process per core, on a bounded sample of the
same workload.  The verbatim reference Python is ~100x slower than this port (BASELINE.md §2).
"""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import sys
import threading
import time

sys.dont_write_bytecode = True      # no __pycache__ in the tree the benchmark runs from
_REPO = os.path.dirname(os.path.abspath(__file__))
for _p in (_REPO, os.path.join(_REPO, 'mrs-gym_b200'), os.path.join(_REPO, 'tests')):
    if _p not in sys.path:
        sys.path.insert(0, _p)

HOVER = 14475.809

CPU_REPS = 24        # rollouts per process of the cpu_baseline leg (see cpu_sample_sizes)
WORKLOADS = {
    # name: E (per GPU), N, mode, K, comm_range, spacing, z0, algorithmic bytes / agent-step (SURVEY.md §8d)
    'c5': dict(E=65536, N=8, mode='set_speeds', K=3, R=2.0, spacing=1.0, z0=2.5, B=176,
               desc='65536 envs x 8 agents per GPU, set_speeds, K_HOPS=3, RETURN_A COMM_RANGE=2.0 (BASELINE configs[4])'),
    'c2': dict(E=256, N=32, mode='set_target_pos', K=3, R=2.0, spacing=1.0, z0=2.5, B=316,
               desc='256 envs x 32 agents, set_target_pos, K_HOPS=3, RETURN_A COMM_RANGE=2.0 (BASELINE configs[1])'),
    'c3': dict(E=4096, N=16, mode='set_control', K=0, R=float('inf'), spacing=0.7, z0=1.0, B=144, A=False,
               desc='4096 envs x 16 agents, set_control, ground + agent contact, RETURN_A off (BASELINE configs[2]; '
                    'SURVEY.md 8d counts no A bytes for it)'),
    # not BASELINE configs: the C5 shape with the PID action modes (profiling the controller path)
    'c5v': dict(E=65536, N=8, mode='set_target_vel', K=3, R=2.0, spacing=1.0, z0=2.5, B=296,
                desc='65536 envs x 8 agents per GPU, set_target_vel, K_HOPS=3, RETURN_A COMM_RANGE=2.0'),
    'c5p': dict(E=65536, N=8, mode='set_target_pos', K=3, R=2.0, spacing=1.0, z0=2.5, B=220,
                desc='65536 envs x 8 agents per GPU, set_target_pos, K_HOPS=3, RETURN_A COMM_RANGE=2.0'),
    # not a BASELINE config: a mid-size swarm at scale (thread-per-agent kernels of the 32 < N <= 128 range)
    'm64': dict(E=1024, N=64, mode='set_target_vel', K=1, R=2.0, spacing=1.0, z0=2.5, B=104 + 12 + 120 + 24 + 256,
                desc='1024 envs x 64 agents, set_target_vel, K_HOPS=1, RETURN_A COMM_RANGE=2.0'),
    'c4': dict(E=1, N=4096, mode='set_force', K=0, R=2.0, spacing=1.0, z0=2.0, B=16548,
               desc='1 env x 4096 agents, set_force, adjacency dominated (BASELINE configs[3])'),
}


def workload_config(w, E, world):
    return {'workload': w['desc'], 'envs_per_gpu': E, 'agents_per_env': w['N'], 'action_type': w['mode'],
            'k_hops': w['K'], 'comm_range': w['R'], 'state_fn': 'cat(pos,vel) D=6',
            'parallelism': 'env-shard x%d' % world}


def kernel_sources_hash():
    """sha256 over the CUDA sources of the library (csrc/*.cu, *.cuh, include/mrs_b200.h)."""
    import hashlib
    h = hashlib.sha256()
    csrc = os.path.join(_REPO, 'mrs-gym_b200', 'csrc')
    files = [os.path.join(csrc, f) for f in sorted(os.listdir(csrc)) if f.endswith(('.cu', '.cuh'))]
    files.append(os.path.join(_REPO, 'include', 'mrs_b200.h'))
    for f in files:
        h.update(open(f, 'rb').read())
    return h.hexdigest()


# ------------------------------------------------------------------------------ synthetic inputs
def make_inputs(w, E, T, seed):
    import numpy as np
    import helpers as H
    rng = np.random.default_rng(seed)
    N = w['N']
    st = H.random_state(rng, E, N, spacing=w['spacing'], z0=w['z0'], jitter=0.1, tilt=0.0, vel=0.0, angvel=0.0)
    mode = w['mode']
    if mode == 'set_speeds':
        act = (HOVER * (1 + 0.05 * rng.standard_normal((T, E, N, 4), dtype=np.float32))).astype(np.float32)
    elif mode == 'set_target_pos':
        act = np.broadcast_to((st['pos'] + rng.normal(0, 0.5, (E, N, 3)).astype(np.float32))[None], (T, E, N, 3)).copy()
    elif mode == 'set_target_vel':
        act = (rng.standard_normal((1, E, N, 3), dtype=np.float32) * 0.5).repeat(T, 0)
    elif mode == 'set_control':
        act = np.concatenate([9.81 + rng.uniform(-1, 1, (T, E, N, 1)), rng.uniform(-1, 1, (T, E, N, 3))],
                             axis=-1).astype(np.float32)
    elif mode == 'set_force':
        act = rng.normal(0, 0.02, (T, E, N, 3)).astype(np.float32)
    else:
        act = H.random_actions(rng, mode, T, E, N, start_pos=st['pos'])
    return st, act


# ------------------------------------------------------------------------------ CPU arm (oracle port)
def _cpu_worker(args):
    """`reps` rollouts of a cache-sized batch (E envs), each W untimed warm-up steps then T timed steps: the sum of the
    timed stretches.  Every rollout starts from a fresh start state, so all of them cover the same stretch of the
    trajectory as the GPU's timed region."""
    wname, E, T, seed, W, reps = args
    os.environ.setdefault('OMP_NUM_THREADS', '1')
    import numpy as np
    import helpers as H
    w = WORKLOADS[wname]
    spent = 0.0
    for r in range(reps):
        st, act = make_inputs(w, E, T + W, seed + 1000 * r)
        env = H.make_spec(E, w['N'], w['mode'], w['K'], w['R'], st)
        for t in range(W):                     # untimed warm-up steps (imports, scipy caches)
            env.step(act[t])
        t0 = time.perf_counter()
        for t in range(T):
            env.step(act[W + t])
        spent += time.perf_counter() - t0
    return spent


def cpu_port_throughput(wname, procs, E_per_proc, T, seed=4321, warmup=1, reps=1):
    """agent-steps/s of the oracle port on `procs` host processes (slowest worker's timed seconds)."""
    w = WORKLOADS[wname]
    ctx = mp.get_context('spawn')
    t0 = time.perf_counter()
    with ctx.Pool(procs) as pool:
        walls = pool.map(_cpu_worker, [(wname, E_per_proc, T, seed + i, max(1, warmup), reps) for i in range(procs)])
    total = procs * E_per_proc * w['N'] * T * reps
    return total / max(walls), max(walls), time.perf_counter() - t0


def _verbatim_worker(args):
    """One process = one reference MRS env (the reference holds one global PyBullet client), stepped verbatim."""
    wname, T, seed = args
    os.environ.setdefault('OMP_NUM_THREADS', '1')
    import numpy as np
    import torch
    torch.set_num_threads(1)
    from oracle import ref_runner
    w = WORKLOADS[wname]
    mrsgym, fake = ref_runner.load_reference()
    N = min(w['N'], 32)
    rng = np.random.default_rng(seed)
    env = ref_runner.make_env(mrsgym, fake, N, w['mode'] if w['mode'] != 'set_force' else 'set_target_accel', K=w['K'],
                              comm_range=w['R'])
    adim = 4 if w['mode'] in ('set_speeds', 'set_control') else 3
    if w['mode'] == 'set_speeds':
        acts = (HOVER * (1 + 0.05 * rng.standard_normal((T + 1, N, adim)))).astype(np.float32)
    elif w['mode'] == 'set_control':
        acts = np.concatenate([9.81 + rng.uniform(-1, 1, (T + 1, N, 1)), rng.uniform(-1, 1, (T + 1, N, 3))], -1).astype(np.float32)
    else:
        acts = rng.normal(0, 0.3, (T + 1, N, adim)).astype(np.float32)
    env.step(torch.tensor(acts[0]))
    t0 = time.perf_counter()
    for t in range(T):
        env.step(torch.tensor(acts[1 + t]))
    return time.perf_counter() - t0, N


def cpu_verbatim_throughput(wname, procs, T=10):
    """The reference's own Python, imported where it lies and run verbatim on the oracle's fake pybullet backend
    (BASELINE.md 4.2): one env per process.  None when no reference tree is present (the GPU box has none)."""
    try:
        from oracle import ref_runner
        if ref_runner.reference_root() is None:
            return None
        ctx = mp.get_context('spawn')
        with ctx.Pool(procs) as pool:
            res = pool.map(_verbatim_worker, [(wname, T, 99 + i) for i in range(procs)])
        wall = max(r[0] for r in res)
        N = res[0][1]
        return {'value': procs * N * T / wall, 'unit': 'agent-steps/s', 'cores': procs,
                'kind': 'reference python + restated Bullet (oracle/fake_pybullet; PyBullet itself is not installable)',
                'sample': '%d processes x 1 env x %d agents x %d steps, the reference imported from %s'
                          % (procs, N, T, ref_runner.reference_root())}
    except Exception as exc:                    # the verbatim leg is a courtesy: never take the bench line down
        return {'unavailable': '%s: %s' % (type(exc).__name__, exc)}


def cpu_sample_sizes(wname):
    w = WORKLOADS[wname]
    if w['N'] >= 1024:
        return 1, 2          # one env of 4096 agents: ~N^2 pair arrays in numpy
    # a cache-sized batch per process (4096 agents), 40 steps per rollout: the SAME stretch of the rollout as the
    # GPU's timed region -- the first steps, before the synthetic swarm collapses (the oracle's sequential-impulse
    # solver in numpy is an order of magnitude slower per step once every agent is in contact).  cpu_baseline
    # repeats such rollouts (CPU_REPS) to reach ~10 s of CPU work per process at ~5e5 agent-steps/s/core.
    return max(1, 4096 // w['N']), 40


# ------------------------------------------------------------------------------ clocks
class ClockSampler:
    """Samples SM clock + throttle reasons of one GPU through NVML while a region runs."""

    def __init__(self, index, period=0.01):
        self.index, self.period = index, period
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {'hw_slowdown': 0x8, 'sw_power_cap': 0x4, 'hw_thermal_slowdown': 0x40, 'sw_thermal_slowdown': 0x20,
                 'hw_power_brake_slowdown': 0x80, 'sync_boost': 0x10}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for n, bit in names.items():
                    if r & bit:
                        self.reasons.add(n)
            except Exception:
                pass
            self._stop.wait(self.period)

    def __enter__(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thr is not None:
            self._thr.join()

    def summary(self):
        s = sorted(self.samples)
        return {'sm_mhz': (s[len(s) // 2] if s else None), 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons),
                'samples': len(s)}


def physical_gpu_index(local):
    vis = os.environ.get('CUDA_VISIBLE_DEVICES')
    if vis:
        try:
            return int(vis.split(',')[local])
        except Exception:
            return local
    return local


# ------------------------------------------------------------------------------ --dump-outputs
DUMP_BYTES = 64 * 10 ** 6     # at most this much in all (C5: 56.6 MB, written whole)


def last_step_outputs(sw):
    """What the timed path hands its caller after its last step, copied to the host: the newest slice of the
    observation window X [E,N,6], of the adjacency window A [E,N,N] (absent with RETURN_A off) and the state
    [E,N,13] (pos, quat xyzw, vel, angvel)."""
    out = {'X': sw.X_window()[0], 'state': sw.state.t().reshape(sw.E, sw.N, -1)}
    if sw.A_tape is not None:
        out['A'] = sw.A_window()[0]
    return {k: v.cpu().numpy() for k, v in out.items()}


def dump_outputs(dirname, arrays, budget=DUMP_BYTES):
    """DIR/<name>.npy for every array.  Larger than `budget` together: every array keeps the same fraction of its
    rows (flattened to [rows, last axis]), picked with a fixed seed, so runs with the same arguments keep the same
    rows."""
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    os.makedirs(dirname, exist_ok=True)
    for name, a in sorted(arrays.items()):
        if total > budget:
            rows = a.reshape(-1, a.shape[-1])
            pick = np.random.default_rng(0).choice(len(rows), max(1, len(rows) * budget // total), replace=False)
            a = rows[np.sort(pick)]
        np.save(os.path.join(dirname, name + '.npy'), a)


# ------------------------------------------------------------------------------ GPU arm
def run_gpu(args):
    import numpy as np
    import torch
    import __graft_entry__
    __graft_entry__.build()
    import mrsgym_b200 as M
    from mrsgym_b200 import dist as D
    import helpers as H

    rank, world = D.init_from_env()
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    numa_bound = D.bind_to_gpu_numa(physical_gpu_index(local)) if world > 1 else False
    w = WORKLOADS[args.workload]
    E0 = args.envs or w['E']
    E = E0 if args.scaling == 'weak' else max(1, E0 // world)
    N, K = w['N'], w['K']
    steps, warmup = args.steps, max(args.warmup, 3)
    # the timed region is `replays` replays of a T-step graph plus `rem` plain single-step launches at its end
    T = min(steps, args.graph_steps)
    replays, rem = steps // T, steps % T

    st, act_np = make_inputs(w, E, T, seed=1234 + 4 + rank)
    use_graph = T >= K + 1
    sw = M.Swarm(E, N, K, w['mode'], M._abi.X_POS_VEL, w['R'], tape_slots=T if use_graph else 2 * K + 2, ring=use_graph,
                 want_A=w.get('A', True) and not os.environ.get('MRS_EXP_NO_A'))
    H.upload_state(sw, st)
    actions = torch.from_numpy(act_np).to(dev)
    # the one exchange of the path: the per-rollout statistics reduction, as the library's peer-memory kernel
    # (mrs_stats_allreduce) at the end of every graph replay; torch.distributed / NCCL stays the plumbing
    comm, comm_note = None, 'single GPU: no exchange'
    if world > 1:
        try:
            comm = D.PeerComm()
            comm_note = ('mrs_stats_allreduce: peer-memory kernel (NVLink P2P stores into the peers\' mailboxes, 64 B per '
                         'rank, one 32-thread launch per GPU) as the last node of every rollout graph; NCCL only for '
                         'rendezvous, handle exchange and the max over ranks of the timings')
        except Exception as exc:                       # no peer access on this box: NCCL does the reduction
            comm, comm_note = None, 'NCCL all-reduce after the rollout (PeerComm unavailable: %s)' % exc
    if use_graph:
        roll = sw.capture_rollout(actions, T, stats_comm=comm)
    else:                                   # fewer steps than the observation window: plain launches
        class _Plain:
            launches_per_replay = T

            def replay(self):
                sw.step_many_single(actions, T)
        _Plain.launches_per_replay = T * sw._step_launches()
        roll = _Plain()

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize(dev)

    # ---- headline: device-resident inputs, graph replays.
    # Every timed region is a defined stretch of ONE rollout: the bench's start state is uploaded again, the warm-up
    # steps follow, then the timed steps.  The synthetic C5 swarm -- open-loop rotor speeds with 5 % noise -- tumbles
    # into itself after ~60 steps and lies on the ground after ~200 (SURVEY.md 8d workload), so "the step" would
    # otherwise depend on how much ran before it; with the driver's protocol the region is steps 21-40, free flight.
    # The contact-dominated regime of the same swarm is reported separately (`contact_regime`).
    if not os.environ.get('BENCH_NO_REUPLOAD'):
        H.upload_state(sw, st)
    for _ in range(max(1, -(-warmup // T))):
        roll.replay()
    sw.stats.zero_()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(physical_gpu_index(local))
    tiny = torch.zeros(1, device=dev)
    in_graph = use_graph and comm is not None

    def reduce_stats():
        return sw.allreduce_stats(comm) if (comm is not None or world == 1) else sw.allreduce_stats()

    barrier()
    with sampler:
        if world > 1:
            # The region starts ON THE DEVICE: the stream first spins ~0.5 ms (the host enqueues the whole region
            # behind it), then passes a device-side barrier across the ranks, then records e0 -- so every rank's
            # clock starts when the last rank arrives, not when its host thread happened to wake up from the
            # host barrier.  The statistics reduction at the end of the rollout aligns the ends the same way.
            torch.cuda._sleep(int(0.5e-3 * 1.9e9))
            if comm is not None:
                comm.barrier()
            else:
                torch.distributed.all_reduce(tiny)
        e0.record()
        for _ in range(replays):
            roll.replay()
        for t in range(rem):                      # only when `steps` is not a multiple of the graph length
            sw.step(actions[t])
        if world > 1 and (rem or not in_graph):
            reduce_stats()                        # (inside the graph otherwise)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        timed_stats = sw.read_stats()
        outputs = last_step_outputs(sw) if args.dump_outputs else None
        # keep the same load running long enough for NVML to see the clocks under load
        t_end = time.time() + args.clock_seconds
        while time.time() < t_end:
            for _ in range(max(1, 2000 // T)):
                roll.replay()
            torch.cuda.synchronize(dev)
    stats_check = None
    if world > 1:
        # the peer-memory reduction against NCCL on the same counters (outside the timed region)
        mine = reduce_stats().clone()
        ref = sw.stats.clone()
        torch.distributed.all_reduce(ref)
        stats_check = 'ok' if bool((mine == ref).all()) else 'MISMATCH %s vs %s' % (mine.tolist(), ref.tolist())
    gpu_launches = replays * roll.launches_per_replay + rem * sw._step_launches()
    ms = D.max_over_ranks(ms, dev)
    agent_steps = float(E) * N * steps * world
    value = agent_steps / (ms * 1e-3)
    sw_status = sw.read_status()

    # ---- the same rollout graph on the swarm as the clock-sampling loop left it: thousands of steps in, every agent
    # rests on the ground or against a neighbour, every warp-chunk takes the contact path (solver sweeps)
    contact_regime = None
    if use_graph:
        sw.stats.zero_()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        roll.replay()
        g1.record()
        torch.cuda.synchronize(dev)
        cs = sw.read_stats()
        cms = g0.elapsed_time(g1) / T
        contact_regime = {'ms_per_step': cms, 'value': float(E) * N / (cms * 1e-3), 'unit': 'agent-steps/s (this rank)',
                          'contact_chunk_steps': cs.get('contact_chunks'), 'solver_sweeps': cs.get('solver_sweeps'),
                          'note': 'same graph, swarm collapsed onto the ground (after the clock-sampling loop)'}
    # ---- same step, one launch at a time with an L2 flush in between (per-launch events), again from the bench's
    # start state
    H.upload_state(sw, st)
    flush = torch.zeros(512 * 1024 * 1024 // 4, device=dev, dtype=torch.float32)
    n_f = min(steps, 20)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_f)]
    sink = torch.zeros((), device=dev)
    for i in range(n_f):
        sink += flush.sum()                 # READ 512 MB: evicts L2 with clean lines (no write-back debt)
        evs[i][0].record()
        sw.step(actions[i % T])
        evs[i][1].record()
    torch.cuda.synchronize(dev)
    flushed_ms = sorted(a.elapsed_time(b) for a, b in evs)
    flushed_med = flushed_ms[len(flushed_ms) // 2]
    del flush

    # ---- multi-step launch (mrs_step_many: state stays in registers for T steps)
    many = None
    if N <= 32:
        H.upload_state(sw, st)
        sw.step_many(actions, T)
        torch.cuda.synchronize(dev)
        m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        m0.record()
        sw.step_many(actions, T)
        m1.record()
        torch.cuda.synchronize(dev)
        mm = m0.elapsed_time(m1)
        many = {'value': float(E) * N * T / (mm * 1e-3), 'unit': 'agent-steps/s (this rank)', 'T': T,
                'note': 'one launch for T steps, state on chip; streams only actions in and X/A out'}

    # ---- e2e through the C ABI with host buffers
    adim = M._abi.ACTION_DIMS[sw.cfg.action_type]
    n_e = min(steps, args.e2e_steps)
    h2d = E * N * adim * 4
    d2h = E * N * (6 + (N if sw.A_tape is not None else 0)) * 4
    e2e_value = e2e_pipe_value = e2e_compact = pcie_gbs = None
    if n_e > 0:
        host_act = [torch.from_numpy(act_np[i % T]).pin_memory() for i in range(min(n_e, T))]
        dev_act = torch.empty(E, N, max(adim, 1), device=dev)
        Xh = torch.empty(E, N, 6).pin_memory()
        Ah = torch.empty(E, N, N).pin_memory() if sw.A_tape is not None else None
        for i in range(3):
            sw.step_host(host_act[i % len(host_act)], dev_act, Xh, Ah)
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for i in range(n_e):
            sw.step_host(host_act[i % len(host_act)], dev_act, Xh, Ah)
        c1.record()
        barrier()
        e2e_ms = D.max_over_ranks(c0.elapsed_time(c1), dev)
        e2e_value = float(E) * N * n_e * world / (e2e_ms * 1e-3)
        # pipelined variant: mrs_rollout_host, copies of neighbouring steps overlap the kernels
        n_p = min(n_e, T)
        ah = torch.from_numpy(act_np[:n_p]).pin_memory()
        Xhh = torch.empty(n_p, E, N, 6).pin_memory()
        Ahh = torch.empty(n_p, E, N, N).pin_memory() if sw.A_tape is not None else None
        dev2 = torch.empty(2, E, N, max(adim, 1), device=dev)
        sw.rollout_host(ah, dev2, Xhh, Ahh)
        barrier()
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record()
        sw.rollout_host(ah, dev2, Xhh, Ahh)
        p1.record()
        barrier()
        pipe_ms = D.max_over_ranks(p0.elapsed_time(p1), dev)
        e2e_pipe_value = float(E) * N * n_p * world / (pipe_ms * 1e-3)
        # opt-in compact adjacency on the wire: one bit per entry instead of one float32 (mrs_pack_adjacency)
        e2e_compact = None
        if sw.A_tape is not None:
            Wd = (N + 31) // 32
            Bhh = torch.empty(n_p, E, N, Wd, dtype=torch.int32).pin_memory()
            devB = torch.empty(2, E, N, Wd, dtype=torch.int32, device=dev)
            sw.rollout_host(ah, dev2, Xhh, None, Bhh, devB)
            barrier()
            q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            q0.record()
            sw.rollout_host(ah, dev2, Xhh, None, Bhh, devB)
            q1.record()
            barrier()
            cms = D.max_over_ranks(q0.elapsed_time(q1), dev)
            d2h_c = E * N * (6 + Wd) * 4
            e2e_compact = {'value': float(E) * N * n_p * world / (cms * 1e-3), 'unit': 'agent-steps/s',
                           'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h_c,
                           'pcie_gbs_per_rank': (h2d + d2h_c) * n_p / (cms * 1e-3) / 1e9,
                           'api': 'mrs_rollout_host with Abits_host: newest X slice + the adjacency bit-packed (u32 per row)'}
            del Bhh, devB
        pcie_gbs = (h2d + d2h) * n_p / (pipe_ms * 1e-3) / 1e9
        del ah, Xhh, Ahh

    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    if rank != 0:
        return
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    peaks_path = os.path.join(_REPO, 'MEASURED_PEAKS.json')
    if os.path.isfile(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    else:
        peak, peak_src = 6650.0, 'fallback (B200_PROFILING.md)'
    ms_per_step = ms / steps
    bytes_per_launch = float(E) * N * w['B']
    achieved = bytes_per_launch / (ms_per_step * 1e-3) / 1e9
    # DRAM bytes per launch of the dominant kernel come from an ncu --set full capture (profiles/traffic.json, written
    # by tools/evidence_collect.py together with the hash of the kernel sources it was taken with): reported only
    # when that hash matches the sources of the library that just ran, null otherwise -- never a stale number
    traffic = None
    tp = os.path.join(_REPO, 'profiles', 'traffic.json')
    if os.path.isfile(tp):
        tj = json.load(open(tp))
        if tj.get('kernel_sources_sha256') == kernel_sources_hash():
            traffic = tj.get(args.workload)
    if N <= 32:
        kernel = 'step_group_kernel<%s>' % w['mode']
    elif N <= 128 and E * N >= 32768:
        kernel = 'step_env_kernel<%s> (one CTA per env, the whole step)' % w['mode']
    elif N <= 128:
        kernel = 'step_pre_kernel + contact_env_kernel + step_post_kernel + adjacency kernel (the step = their sum)'
    else:
        kernel = 'pair_tile_kernel + agent_pre_kernel + contact_env_kernel + step_post_kernel + adjacency_tiled_kernel (the step = their sum)'
    out = {
        'metric': 'agent-steps/sec', 'value': value, 'unit': 'agent-steps/s', 'n_gpus': world, 'steps': steps,
        'warmup': warmup, 'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': args.scaling,
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(w, E, world),
        'notes': {'launch': (('CUDA graph of %d single-step launches, %d replays' if use_graph else '%d plain launches x %d') % (T, replays))
                            + (' + %d plain launches' % rem if rem else ''),
                  'l2': 'inputs larger than L2: the timed region consumes %.0f MB of distinct action buffers and writes '
                        '%.0f MB of distinct X/A tape slots (L2 = 126 MB); no buffer is re-read across iterations -- the '
                        'state is loop-carried (written by step t, read by step t+1, as in any rollout).  l2_flushed '
                        'reports the same step one launch at a time behind a 512 MB read-flush'
                        % (T * E * N * max(M._abi.ACTION_DIMS[sw.cfg.action_type], 1) * 4 / 1e6,
                           steps * E * N * (6 + (N if sw.A_tape is not None else 0)) * 4 / 1e6),
                  'timed_region': ('device-aligned: spin + device barrier across ranks, e0, %d steps, statistics reduction, e1; '
                                   'max over ranks' % steps) if world > 1 else 'e0, %d steps, e1 (CUDA events on the launch stream)' % steps,
                  'collective': comm_note, 'stats_allreduce_check': stats_check},
        'roofline': {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                     'traffic': traffic, 'kernel': kernel, 'peak_source': peak_src,
                     'algorithmic_bytes_per_agent_step': w['B'], 'agent_steps_per_launch': E * N,
                     'launch_ms': ms_per_step},
        'l2_flushed': {'ms_per_step_median': flushed_med, 'ms_min': flushed_ms[0], 'n': n_f,
                       'value': float(E) * N / (flushed_med * 1e-3),
                       'achieved_gbs': bytes_per_launch / (flushed_med * 1e-3) / 1e9,
                       'frac': bytes_per_launch / (flushed_med * 1e-3) / 1e9 / peak},
        'step_many': many,
        'contact_regime': contact_regime,
        'stats_timed_region': timed_stats,
        'e2e': {'value': e2e_pipe_value, 'unit': 'agent-steps/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                'steps': n_e, 'api': 'mrs_rollout_host (C ABI, pinned host buffers; every step: H2D actions, kernel, D2H '
                                     'newest X and A; copies of neighbouring steps overlap the kernels)',
                'sync_per_step': {'value': e2e_value, 'api': 'mrs_step_host (same copies, stream sync after every step)'},
                'numa_bound': numa_bound, 'pcie_gbs_per_rank': pcie_gbs},
        'e2e_compactA': e2e_compact,
        'gpu_launches': gpu_launches,
        'clocks': sampler.summary(),
        'status_word': sw_status,
    }
    if world == 1 and not args.no_cpu:
        procs = min(os.cpu_count() or 1, 64)
        Ep, Tc = cpu_sample_sizes(args.workload)
        reps = 1 if w['N'] >= 1024 else (4 if w['spacing'] < 0.75 else CPU_REPS)
        v, wall, total = cpu_port_throughput(args.workload, procs, Ep, Tc, warmup=max(args.warmup, 3), reps=reps)
        out['cpu_baseline'] = {'value': v, 'unit': 'agent-steps/s', 'cores': procs, 'kind': 'port',
                               'sample': '%d processes x %d rollouts x %d envs x %d agents x %d steps (after %d warm-up '
                                         'steps each) of the same workload (oracle/spec.py, numpy float64); %.1f s'
                                         % (procs, reps, Ep, w['N'], Tc, max(args.warmup, 3), total)}
        verb = cpu_verbatim_throughput(args.workload, procs)
        if verb is not None:
            out['cpu_baseline_verbatim'] = verb
    emit(out)


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    w = WORKLOADS[args.workload]
    procs = min(os.cpu_count() or 1, 64)
    Ep, _ = cpu_sample_sizes(args.workload)
    steps, warmup = args.steps, max(args.warmup, 3)      # the same floor as the GPU arm
    # bounded: each "step" here is one env.step of the sample batch (procs x Ep envs)
    Tc = max(1, min(steps, 200))
    v, wall, total = cpu_port_throughput(args.workload, procs, Ep, Tc, warmup=min(warmup, 20))
    out = {
        'impl': 'reference', 'metric': 'agent-steps/sec', 'value': v, 'unit': 'agent-steps/s',
        'n_gpus': int(os.environ.get('WORLD_SIZE', '1')), 'steps': Tc, 'warmup': warmup,
        'ms_per_step': wall / Tc * 1e3, 'higher_is_better': True, 'scaling': args.scaling, 'vs_baseline': None,
        'dtype': 'f64', 'data': 'synthetic',
        'config': workload_config(w, args.envs or w['E'], int(os.environ.get('WORLD_SIZE', '1'))),
        'notes': {'cpu_sample': 'bounded sample of the workload: %d processes x %d envs per step' % (procs, Ep)},
        'cpu_baseline': {'value': v, 'unit': 'agent-steps/s', 'cores': procs, 'kind': 'port',
                         'sample': '%d processes x %d envs x %d agents x %d steps (oracle/spec.py numpy port of the '
                                   'reference step + restated Bullet; PyBullet itself is not installable here)'
                                   % (procs, Ep, w['N'], Tc)},
        'e2e': {'value': v, 'unit': 'agent-steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    emit(out)


_REAL_STDOUT = None


def _quiet_stdout():
    """Everything except the final JSON line goes to stderr (NCCL / torch banners print to fd 1)."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), 'w')
        os.dup2(2, 1)


def emit(obj):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(obj) + '\n')
    out.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='c5', choices=sorted(WORKLOADS))
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'])
    ap.add_argument('--graph-steps', type=int, default=100, help='steps per captured CUDA graph')
    ap.add_argument('--e2e-steps', type=int, default=50)
    ap.add_argument('--clock-seconds', type=float, default=1.0)
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--envs', type=int, default=0, help='override envs per GPU (size sweeps; not the BASELINE config)')
    ap.add_argument('--dump-outputs', metavar='DIR', default='',
                    help='write what the last timed step computed as DIR/<name>.npy (at most 64 MB)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs records the GPU path (--impl b200)')
    _quiet_stdout()
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == '__main__':
    main()
