#!/usr/bin/env python
"""Cost of the external wrench (MrsBuffers.wrench): per-step time without a wrench, with a zero wrench and with a
random one.

    python tools/bench_wrench.py [--reps 9] [--steps 20] [--out profiles/r3_wrench.json]

(profiles/r3_wrench_100steps.json: --steps 100 --reps 7, long enough for the synthetic C5 swarm to tumble into contact)

  * bench.py's C5 workload (65536 x 8, set_speeds, K_HOPS 3, A on) and its m64 workload (1024 x 64 = 65536 agents,
    set_target_vel, K_HOPS 1: the fused step_env_kernel), each as a CUDA-graphed `steps`-step mrs_rollout
    (Swarm.capture_rollout) on three swarms of the same settings and start state: no wrench bound, a zero wrench, and
    a random one (|F| <= 0.1 N, |tau| <= 1e-5 N m per component, fixed seed).  The three replays are alternated over
    `reps` repetitions, each from the same start state uploaded outside the timed region; CUDA events around the
    replay, us per step = that time / steps.  Median, min and max.
  * the device name and power limit, read in the same run.
Writes one JSON file (--out) and prints it.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

sys.dont_write_bytecode = True
_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (_REPO, os.path.join(_REPO, 'mrs-gym_b200'), os.path.join(_REPO, 'tools'), os.path.join(_REPO, 'tests')):
    if _p not in sys.path:
        sys.path.insert(0, _p)

from bench_neighbors import device_info, spread  # noqa: E402

VARIANTS = ('none', 'zero', 'random')


def run(name, steps, reps):
    import numpy as np
    import torch
    import bench
    import helpers as H
    import mrsgym_b200 as M
    w = bench.WORKLOADS[name]
    E, N, K = w['E'], w['N'], w['K']
    st, act_np = bench.make_inputs(w, E, steps, seed=1234 + 4)
    acts = torch.from_numpy(act_np).cuda()
    rng = np.random.default_rng(7)
    F = torch.from_numpy(rng.uniform(-0.1, 0.1, (E, N, 3)).astype(np.float32)).cuda()
    Tq = torch.from_numpy(rng.uniform(-1e-5, 1e-5, (E, N, 3)).astype(np.float32)).cuda()
    swarms, graphs = {}, {}
    for v in VARIANTS:
        sw = swarms[v] = M.Swarm(E, N, K, w['mode'], M._abi.X_POS_VEL, w['R'], tape_slots=steps, ring=True)
        if v == 'zero':
            sw.set_external_wrench(torch.zeros(3, device='cuda'), torch.zeros(3, device='cuda'))
        elif v == 'random':
            sw.set_external_wrench(F, Tq)
        H.upload_state(sw, st)
        graphs[v] = sw.capture_rollout(acts, steps)
    us = {v: [] for v in VARIANTS}
    for _ in range(reps):
        for v, sw in swarms.items():
            H.upload_state(sw, st)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            graphs[v].replay()
            e1.record()
            torch.cuda.synchronize()
            us[v].append(e0.elapsed_time(e1) * 1e3 / steps)
    res = {v: {'us_per_step': spread(x)} for v, x in us.items()}
    base = res['none']['us_per_step']['median']
    for v in ('zero', 'random'):
        res[v]['ratio_to_none'] = res[v]['us_per_step']['median'] / base
    res['setup'] = {'workload': name, 'desc': w['desc'], 'E': E, 'N': N, 'steps': steps, 'reps': reps,
                    'form': 'Swarm.capture_rollout (mrs_rollout in a CUDA graph)',
                    'random_wrench': '|F| <= 0.1 N, |tau| <= 1e-5 N m per component, seed 7',
                    'extra_bytes_per_agent_step': 24}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=9)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--out', default=os.path.join(_REPO, 'profiles', 'r3_wrench.json'))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('bench_wrench.py measures on a CUDA device; none is visible')
    out = {'device': device_info(), 'c5': run('c5', args.steps, args.reps), 'm64': run('m64', args.steps, args.reps)}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == '__main__':
    main()
