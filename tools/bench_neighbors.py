#!/usr/bin/env python
"""Dense A against neighbour lists on one GPU: the cost of A_FORMAT='neighbors' per step and per kernel.

    python tools/bench_neighbors.py [--workloads c4,m64,c5] [--steps 50] [--reps 7] [--out profiles/r3_neighbors.json]

For every workload of bench.py (its WORKLOADS / make_inputs, seeded like bench.py's rank 0):
  * us per step of CUDA-graph rollouts (Swarm.capture_rollout, ring tapes of `steps` slots), dense mode against
    neighbour mode (M = min(N - 1, 64)), the two alternated over `reps` repetitions, every repetition from the same
    uploaded start state; median, min and max;
  * kernel time of mrs_neighbors against mrs_adjacency on the same positions (CUDA events around 200 launches each);
  * bytes the step writes for A (4 N per agent against 4 (M + 1)), the largest degree and the overflow counter;
  * the device name and power limit, read in the same run.
Writes one JSON file (--out) and prints it.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

sys.dont_write_bytecode = True
_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (_REPO, os.path.join(_REPO, 'mrs-gym_b200'), os.path.join(_REPO, 'tests')):
    if _p not in sys.path:
        sys.path.insert(0, _p)


def device_info():
    import torch
    info = {'name': torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i',
                            os.environ.get('CUDA_VISIBLE_DEVICES', '0').split(',')[0]],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info['nvidia_smi'] = q
    except (OSError, subprocess.SubprocessError) as exc:
        info['nvidia_smi'] = 'unavailable: %s' % exc
    return info


def spread(xs):
    return {'median': statistics.median(xs), 'min': min(xs), 'max': max(xs), 'n': len(xs)}


def run(name, steps, reps):
    import torch
    import bench
    import helpers as H
    import mrsgym_b200 as M
    w = bench.WORKLOADS[name]
    E, N, K = w['E'], w['N'], w['K']
    Mx = min(N - 1, 64)
    st, act_np = bench.make_inputs(w, E, steps, seed=1234 + 4)
    acts = torch.from_numpy(act_np).cuda()
    mk = lambda **kw: M.Swarm(E, N, K, w['mode'], M._abi.X_POS_VEL, w['R'], tape_slots=steps, ring=True, **kw)
    swarms = {'dense': mk(), 'neighbors': mk(neighbors=Mx)}
    graphs = {}
    for k, sw in swarms.items():
        H.upload_state(sw, st)
        graphs[k] = sw.capture_rollout(acts, steps)
    ms = {k: [] for k in swarms}
    for _ in range(reps):
        for k, sw in swarms.items():                       # alternated: both modes see the same box state
            H.upload_state(sw, st)
            sw.stats.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            graphs[k].replay()
            e1.record()
            torch.cuda.synchronize()
            ms[k].append(e0.elapsed_time(e1) * 1e3 / steps)
    nb = swarms['neighbors']
    win = nb.N_window()
    max_deg = int(win.count.max())
    overflow_rows = int(nb.read_stats()['neighbor_overflow'])
    status = nb.read_status()
    # kernels on the same positions (the state the timed rollouts left)
    sw = swarms['dense']
    pos = sw.get_pos().contiguous()
    A = torch.empty(E, N, N, device='cuda')
    idx = torch.empty(E, N, Mx, dtype=torch.int32, device='cuda')
    cnt = torch.empty(E, N, dtype=torch.int32, device='cuda')
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    cfg, bufs = C.byref(sw.cfg), C.byref(sw.bufs)
    calls = {
        'mrs_adjacency': lambda: sw.lib.mrs_adjacency(cfg, C.c_void_p(pos.data_ptr()), C.c_void_p(A.data_ptr()), stream),
        'mrs_neighbors': lambda: sw.lib.mrs_neighbors(cfg, bufs, Mx, C.c_void_p(idx.data_ptr()), C.c_void_p(cnt.data_ptr()),
                                                      stream),
    }
    kern = {k: [] for k in calls}
    for _ in range(3):
        for k, fn in calls.items():
            for _ in range(10):
                assert fn() == 0
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(200):
                fn()
            e1.record()
            torch.cuda.synchronize()
            kern[k].append(e0.elapsed_time(e1) * 1e3 / 200)
    assert torch.equal(M.Neighbors(idx, cnt).to_dense(), A), 'neighbour lists differ from the dense A'
    S = E * N
    return {
        'workload': w['desc'], 'E': E, 'N': N, 'K': K, 'M': Mx, 'graph_steps': steps, 'reps': reps,
        'us_per_step': {k: spread(v) for k, v in ms.items()},
        'step_ratio_neighbors_over_dense': statistics.median(ms['neighbors']) / statistics.median(ms['dense']),
        'kernel_us': {k: spread(v) for k, v in kern.items()},
        'kernel_note': 'CUDA events around 200 back-to-back launches, 3 rounds alternated; positions after the rollouts',
        'A_bytes_written_per_step': {'dense': 4 * S * N, 'neighbors': 4 * S * (Mx + 1)},
        'max_degree': max_deg, 'overflow_rows': overflow_rows, 'status': status,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--workloads', default='c4,m64,c5')
    ap.add_argument('--steps', type=int, default=50, help='steps per captured rollout graph')
    ap.add_argument('--reps', type=int, default=7)
    ap.add_argument('--out', default=os.path.join(_REPO, 'profiles', 'r3_neighbors.json'))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit('bench_neighbors needs a CUDA device')
    import __graft_entry__
    __graft_entry__.build()
    torch.cuda.set_device(0)
    out = {'device': device_info(), 'results': {}}
    for name in args.workloads.split(','):
        out['results'][name] = run(name, args.steps, args.reps)
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as fp:
        json.dump(out, fp, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == '__main__':
    main()
