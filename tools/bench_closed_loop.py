#!/usr/bin/env python
"""The closed loop of rollout(): host-driven (graph=False) against one CUDA graph with on-device auto-reset (graph=True).

    python tools/bench_closed_loop.py [--reps 7] [--steps 100] [--out profiles/r3_closed_loop.json]

  * rollout(env, reynolds_policy(), T, episode_length=50) at 65536 x 8 and 1024 x 64 agents, set_target_vel,
    K_HOPS 3, COMM_RANGE 2.0, TAPE_SLOTS = T, with graph=False and graph=True on two envs of the same settings,
    alternated over `reps` repetitions (plus one untimed warm-up that also captures the graph), each from a fresh
    full reset outside the timed region.  Host clock around the rollout with a device synchronise on both ends;
    us per step = that time / T.  Median, min and max.
  * the mrs_autoreset kernel alone (CUDA events around back-to-back launches) at the same shapes with 0 %, ~2 % and
    100 % of the envs resetting (done_in masks).
  * the device name and power limit, read in the same run.
Writes one JSON file (--out) and prints it.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

sys.dont_write_bytecode = True
_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (_REPO, os.path.join(_REPO, 'mrs-gym_b200'), os.path.join(_REPO, 'tools')):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from bench_neighbors import device_info, spread  # noqa: E402

# (E, N, (z_lo, z_hi, xy_radius)): the start region of each shape
SHAPES = [(65536, 8, (1.0, 3.0, 1.0)), (1024, 64, (1.0, 5.0, 3.0))]
K_HOPS, COMM_RANGE, EPISODE_LENGTH = 3, 2.0, 50


def rollouts(E, N, region, T, reps):
    import torch
    import mrsgym_b200 as M
    kw = dict(N_AGENTS=N, N_ENVS=E, K_HOPS=K_HOPS, COMM_RANGE=COMM_RANGE, ACTION_TYPE='set_target_vel', SEED=1,
              START_POS=M.DefaultSpawn(N, *region), TAPE_SLOTS=T)
    envs = {'eager': M.MRS(**kw), 'graph': M.MRS(**kw)}
    pol = M.reynolds_policy()
    secs = {v: [] for v in envs}
    for rep in range(reps + 1):                                   # rep 0 warms both paths up and captures the graph
        for v, env in envs.items():
            env.reset()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            M.rollout(env, pol, T, episode_length=EPISODE_LENGTH, graph=(v == 'graph'))
            torch.cuda.synchronize()
            if rep:
                secs[v].append(time.perf_counter() - t0)
            env.check_status()
    res = {v: {'us_per_step': spread([s * 1e6 / T for s in x])} for v, x in secs.items()}
    res['speedup_graph_over_eager'] = res['eager']['us_per_step']['median'] / res['graph']['us_per_step']['median']
    res['setup'] = {'E': E, 'N': N, 'T': T, 'K_HOPS': K_HOPS, 'COMM_RANGE': COMM_RANGE,
                    'episode_length': EPISODE_LENGTH, 'resets_per_rollout': T // EPISODE_LENGTH,
                    'region': {'z': region[:2], 'xy_radius': region[2]}, 'ACTION_TYPE': 'set_target_vel',
                    'policy': 'reynolds_policy()', 'recorded': 'X, A, action, reward, done (rollout defaults)'}
    del envs
    torch.cuda.empty_cache()
    return res


def kernel_time(E, N, region, reps):
    import torch
    import mrsgym_b200 as M
    sw = M.Swarm(E, N, K_HOPS, 'set_target_vel', M._abi.X_POS_VEL, COMM_RANGE, tape_slots=2 * K_HOPS + 2, ring=True)
    dev = sw.device
    sw.spawn(1, z=region[:2], xy_radius=region[2], xy_sigma=region[2])
    steps = torch.zeros(E, dtype=torch.int32, device=dev)
    episode = torch.zeros(E, dtype=torch.int32, device=dev)
    done = torch.zeros(E, dtype=torch.bool, device=dev)
    failed = torch.zeros(1, dtype=torch.int32, device=dev)
    out = {}
    for name, frac in (('0%', 0.0), ('2%', 0.02), ('100%', 1.0)):
        mask = torch.zeros(E, dtype=torch.bool, device=dev)
        mask[torch.randperm(E, device=dev)[:int(round(frac * E))]] = True

        def launch():
            sw.autoreset(1, steps, episode, done, done_in=mask, slot_x=0, slot_a=0, z=region[:2], xy_radius=region[2],
                         xy_sigma=region[2], max_rounds=10000 if N > 32 else 256, failed=failed)
        for _ in range(3):
            launch()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n = 50
        us = []
        for _ in range(reps):
            e0.record()
            for _ in range(n):
                launch()
            e1.record()
            torch.cuda.synchronize()
            us.append(e0.elapsed_time(e1) * 1e3 / n)
        out[name] = {'resetting_envs': int(mask.sum()), 'us_per_launch': spread(us)}
    out['failed_envs'] = int(failed.item())
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=7)
    ap.add_argument('--steps', type=int, default=100)
    ap.add_argument('--out', default=os.path.join(_REPO, 'profiles', 'r3_closed_loop.json'))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit('bench_closed_loop needs a CUDA device')
    import __graft_entry__
    __graft_entry__.build()
    torch.cuda.set_device(0)
    out = {'device': device_info(), 'rollout': {}, 'autoreset_kernel': {}}
    for E, N, region in SHAPES:
        key = '%dx%d' % (E, N)
        out['rollout'][key] = rollouts(E, N, region, args.steps, args.reps)
        out['autoreset_kernel'][key] = kernel_time(E, N, region, args.reps)
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as fp:
        json.dump(out, fp, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == '__main__':
    main()
