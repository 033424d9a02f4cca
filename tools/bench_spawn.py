#!/usr/bin/env python
"""Start-state sampling on the device against the host sampler, and what it does to rollouts with auto-reset.

    python tools/bench_spawn.py [--reps 5] [--rollout-steps 200] [--out profiles/r3_spawn.json]

  * mrs_spawn kernel time (CUDA events around back-to-back launches of one seed, a preallocated failure counter) at
    the shapes of the parity tests: 1024 x 64, 64 x 200, 1 x 4096, 4 x 33 and 2 x 1500, each in a region that holds it;
  * the host sampler (spawn.sample_start_pos, torch on the CPU) at the same shapes, host clock;
  * rollout(env, reynolds_policy(), T, episode_length=50) at 1024 x 64, set_target_vel, COMM_RANGE 2.0, with
    DefaultSpawn (device spawn) and with the same distribution behind a wrapper MRS does not recognise (host sampler
    + upload), alternated over `reps` repetitions, each from a fresh full reset outside the timed region; also the
    same rollout without resets.  Host clock around the rollout with a device synchronise on both ends.
  * the device name and power limit, read in the same run.
Writes one JSON file (--out) and prints it.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

sys.dont_write_bytecode = True
_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (_REPO, os.path.join(_REPO, 'mrs-gym_b200'), os.path.join(_REPO, 'tools')):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from bench_neighbors import device_info, spread  # noqa: E402

R_AGENT = 0.3
# (E, N, (z_lo, z_hi, xy_radius)): the host sampler converges in all of them
SHAPES = [(1024, 64, (1.0, 5.0, 3.0)), (64, 200, (1.0, 5.0, 4.0)), (1, 4096, (1.0, 17.0, 16.0)),
          (4, 33, (1.0, 5.0, 3.0)), (2, 1500, (1.0, 9.0, 9.0))]


class HostOnly:
    """DefaultSpawn's distribution behind a type MRS does not recognise: MRS.reset samples it on the host."""

    def __init__(self, dist):
        self.dist = dist

    def sample(self, sample_shape=()):
        return self.dist.sample(sample_shape)


def kernel_time(E, N, region, reps):
    import torch
    import mrsgym_b200 as M
    sw = M.Swarm(E, N, 0, 'set_target_vel', M._abi.X_POS_VEL, want_A=False)
    failed = torch.zeros(1, dtype=torch.int32, device='cuda')
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    z_lo, z_hi, R = region

    def launch():
        return sw.lib.mrs_spawn(C.byref(sw.cfg), C.byref(sw.bufs), None, C.c_ulonglong(1), C.c_ulonglong(0), z_lo, z_hi, R, R,
                                -1.5707963, 1.5707963, 256, C.c_void_p(failed.data_ptr()), stream)
    for _ in range(3):
        assert launch() == 0
    torch.cuda.synchronize()
    failed.zero_()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    launch()
    e1.record()
    torch.cuda.synchronize()
    one = e0.elapsed_time(e1)
    n = max(5, min(200, int(200.0 / max(one, 1e-3))))        # about 0.2 s of launches per round
    us = []
    for _ in range(reps):
        e0.record()
        for _ in range(n):
            launch()
        e1.record()
        torch.cuda.synchronize()
        us.append(e0.elapsed_time(e1) * 1e3 / n)
    return {'us_per_launch': spread(us), 'launches_per_round': n, 'failed_envs': int(failed.item())}


def host_time(E, N, region, reps):
    import torch
    from mrsgym_b200 import DefaultSpawn, sample_start_pos
    dist = DefaultSpawn(N, region[0], region[1], region[2])
    s = []
    for _ in range(reps):
        t0 = time.perf_counter()
        sample_start_pos(dist, E, N, R_AGENT)
        s.append(time.perf_counter() - t0)
    return {'s_per_call': spread(s), 'torch_threads': torch.get_num_threads()}


def rollouts(T, reps):
    import torch
    import mrsgym_b200 as M
    E, N = 1024, 64
    kw = dict(N_AGENTS=N, N_ENVS=E, COMM_RANGE=2.0, ACTION_TYPE='set_target_vel', SEED=1)
    dist = M.DefaultSpawn(N, 1.0, 5.0, 3.0)
    envs = {'device_spawn': M.MRS(START_POS=dist, **kw), 'host_sampler': M.MRS(START_POS=HostOnly(dist), **kw)}
    pol = M.reynolds_policy()
    variants = [('device_spawn', 50), ('host_sampler', 50), ('no_reset', None)]
    secs = {v: [] for v, _ in variants}
    for rep in range(reps + 1):                                   # rep 0 warms every path up
        for v, ep in variants:
            env = envs['device_spawn' if v == 'no_reset' else v]
            env.reset()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            M.rollout(env, pol, T, episode_length=ep)
            torch.cuda.synchronize()
            if rep:
                secs[v].append(time.perf_counter() - t0)
            env.check_status()
    res = {v: {'s_per_rollout': spread(s), 'agent_steps_per_s': spread([T * E * N / x for x in s])} for v, s in secs.items()}
    res['speedup_device_over_host'] = statistics.median(secs['host_sampler']) / statistics.median(secs['device_spawn'])
    res['setup'] = {'E': E, 'N': N, 'T': T, 'episode_length': 50, 'resets_per_rollout': T // 50,
                    'region': '(z 1..5, xy radius 3)', 'COMM_RANGE': 2.0, 'ACTION_TYPE': 'set_target_vel',
                    'recorded': 'X, A, action, reward, done (rollout defaults)'}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--rollout-steps', type=int, default=200)
    ap.add_argument('--out', default=os.path.join(_REPO, 'profiles', 'r3_spawn.json'))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit('bench_spawn needs a CUDA device')
    import __graft_entry__
    __graft_entry__.build()
    torch.cuda.set_device(0)
    out = {'device': device_info(), 'spawn': {}, 'rollout': None}
    for E, N, region in SHAPES:
        key = '%dx%d' % (E, N)
        out['spawn'][key] = {'E': E, 'N': N, 'region': {'z': region[:2], 'xy_radius': region[2]},
                             'device': kernel_time(E, N, region, args.reps),
                             'host': host_time(E, N, region, min(args.reps, 3))}
        out['spawn'][key]['speedup'] = (out['spawn'][key]['host']['s_per_call']['median'] * 1e6 /
                                        out['spawn'][key]['device']['us_per_launch']['median'])
        torch.cuda.empty_cache()
    out['rollout'] = rollouts(args.rollout_steps, args.reps)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as fp:
        json.dump(out, fp, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == '__main__':
    main()
