"""Shared fixtures of the parity tests: seeded start states / actions fed identically to the
CUDA path (through the C ABI) and to the CPU oracle (oracle/spec.py).  Nothing here reads
/root/reference."""
from __future__ import annotations

import numpy as np

# torch and the oracle are imported lazily: bench.py's CPU workers use the input generators of this
# module and should not pay for a torch import each; bench.py's GPU arm must not pull the oracle in

HOVER = 14475.809
MODES = ['set_target_vel', 'set_target_pos', 'set_target_accel', 'set_force', 'set_target_ori', 'set_control',
         'set_speeds']


def grid_positions(E, N, spacing=1.0, z0=2.0, jitter=0.1, rng=None):
    g = int(np.ceil(N ** (1 / 3)))
    grid = np.array([[i, j, k] for k in range(g) for j in range(g) for i in range(g)][:N], dtype=np.float64)
    pos = grid[None] * spacing + np.array([0, 0, z0])
    if rng is not None and jitter > 0:
        pos = pos + rng.uniform(-jitter, jitter, (E, N, 3))
    else:
        pos = np.broadcast_to(pos, (E, N, 3)).copy()
    return pos


def random_state(rng, E, N, spacing=1.0, z0=2.0, jitter=0.1, tilt=0.15, vel=0.3, angvel=0.5):
    """float32-representable start state (so GPU and oracle start from identical numbers)."""
    from scipy.spatial.transform import Rotation as R
    pos = grid_positions(E, N, spacing, z0, jitter, rng)
    rpy = np.concatenate([rng.uniform(-tilt, tilt, (E * N, 2)), rng.uniform(-np.pi / 2, np.pi / 2, (E * N, 1))], axis=1)
    quat = R.from_euler('xyz', rpy).as_quat().reshape(E, N, 4)
    st = dict(pos=pos, quat=quat, vel=rng.uniform(-vel, vel, (E, N, 3)), angvel=rng.uniform(-angvel, angvel, (E, N, 3)))
    return {k: v.astype(np.float32) for k, v in st.items()}


def random_actions(rng, mode, T, E, N, start_pos=None):
    if mode == 'set_target_vel':
        a = rng.normal(0, 0.5, (1, E, N, 3)).repeat(T, 0) + rng.normal(0, 0.05, (T, E, N, 3))
    elif mode == 'set_target_pos':
        a = (start_pos + rng.normal(0, 0.5, (E, N, 3)))[None].repeat(T, 0)
    elif mode == 'set_target_accel':
        a = rng.normal(0, 1.0, (T, E, N, 3))
    elif mode == 'set_force':
        a = rng.normal(0, 0.02, (T, E, N, 3))
    elif mode == 'set_target_ori':
        a = rng.uniform(-0.2, 0.2, (1, E, N, 3)).repeat(T, 0)
    elif mode == 'set_control':
        a = np.stack([9.81 + rng.uniform(-1, 1, (T, E, N)), rng.uniform(-1, 1, (T, E, N)),
                      rng.uniform(-1, 1, (T, E, N)), rng.uniform(-1, 1, (T, E, N))], axis=-1)
        a[::5, :, :, 1:] *= 60.0          # some rows in the NNLS branch
    elif mode == 'set_speeds':
        a = HOVER * (1 + 0.05 * rng.normal(0, 1, (T, E, N, 4)))
    else:
        raise ValueError(mode)
    return a.astype(np.float32)


def upload_state(swarm, st):
    """Exact float32 upload into the SoA planes (bypasses the euler conversion of set_state)."""
    import torch
    S = swarm.S
    planes = np.concatenate([st['pos'].reshape(S, 3), st['quat'].reshape(S, 4), st['vel'].reshape(S, 3),
                             st['angvel'].reshape(S, 3)], axis=1).T.copy()
    swarm.state.copy_(torch.from_numpy(planes))
    swarm.reset_windows()


def read_state(swarm):
    p = swarm.state.detach().cpu().numpy().astype(np.float64)
    S, E, N = swarm.S, swarm.E, swarm.N
    return dict(pos=p[0:3].T.reshape(E, N, 3), quat=p[3:7].T.reshape(E, N, 4), vel=p[7:10].T.reshape(E, N, 3),
                angvel=p[10:13].T.reshape(E, N, 3))


def make_spec(E, N, mode, K, comm_range, st, agent_radius=0.3, dt=0.01, **phys):
    from oracle import spec
    from oracle import bullet_model as bm
    phys.setdefault('contact_radius', agent_radius)
    P = bm.PhysicsParams(agent_radius=agent_radius, **phys)
    env = spec.SpecEnv(E, N, mode, K=K, comm_range=comm_range, dt=dt, phys=P)
    env.set_state(pos=st['pos'].astype(np.float64), quat=st['quat'].astype(np.float64),
                  vel=st['vel'].astype(np.float64), angvel=st['angvel'].astype(np.float64))
    env.reset_rings()
    return env


def spec_state(env):
    return dict(pos=env.pos.copy(), quat=env.quat.copy(), vel=env.vel.copy(), angvel=env.angvel.copy())


# One-step delta bar of the parity tests: |d_gpu - d_ref| <= REL * |d_ref| + floor, both deltas measured from the
# common float32 start state; the floor is the float32 resolution of the stored quantity (pos: also one ulp of the
# coordinate)
REL = 1e-4
FLOOR = dict(pos=5e-7, vel=5e-7, angvel=1e-5, quat=3e-7)


def delta_ratio(s0, r1, g1):
    """{quantity: largest |(g1 - s0) - (r1 - s0)| in multiples of the bar around the reference r1}"""
    worst = {}
    for k in ('pos', 'vel', 'angvel', 'quat'):
        base = s0[k].astype(np.float64)
        dg, dr = g1[k] - base, r1[k] - base
        if k == 'quat':       # q and -q are the same rotation
            flip = np.sum(g1[k] * r1[k], axis=-1, keepdims=True) < 0
            dg = np.where(flip, -g1[k], g1[k]) - base
        err = np.abs(dg - dr)
        floor = FLOOR[k]
        if k == 'pos':     # one float32 ulp of the stored coordinate (5e-7 m up to 8 m, 1e-6 m up to 16 m, ...)
            floor = np.maximum(floor, np.spacing(np.abs(g1[k]).astype(np.float32)).astype(np.float64))
        tol = REL * np.abs(dr) + floor
        worst[k] = float(np.max(err / tol)) if err.size else 0.0
        if not np.all(np.isfinite(err)):
            worst[k] = float('inf')
    return worst


def check_delta(tag, s0, g1, r1):
    """one-step deltas, GPU (g1) vs oracle (r1), both measured from the common start state s0"""
    worst = delta_ratio(s0, r1, g1)
    for k, w in worst.items():
        assert w <= 1.0, '%s: %s delta off by %.3g x tolerance' % (tag, k, w)
    return worst


def quat_angle(q1, q2):
    """Rotation angle between unit quaternions (rad), sign-insensitive."""
    d = np.abs(np.sum(q1 * q2, axis=-1)) / (np.linalg.norm(q1, axis=-1) * np.linalg.norm(q2, axis=-1))
    return 2.0 * np.arccos(np.clip(d, 0.0, 1.0))


def torch_cpu_adjacency(pos32, comm_range):
    """MRS.calc_A exactly as the reference computes it (MRS.py:117-124,166-170), on torch CPU."""
    import torch
    pos = torch.as_tensor(pos32, dtype=torch.float32)
    N = pos.shape[-2]
    if comm_range == float('inf'):
        return (torch.ones(N, N) - torch.eye(N)).expand(*pos.shape[:-2], N, N).clone()
    out = []
    for p in pos.reshape(-1, N, 3):
        posi = p.unsqueeze(1).expand(-1, N, -1)
        posj = p.unsqueeze(0).expand(N, -1, -1)
        codist = (posi - posj).norm(dim=2)
        codist.diagonal().fill_(float('inf'))
        out.append((codist <= comm_range).float())
    return torch.stack(out).reshape(*pos.shape[:-2], N, N)


def downwash_sensitivity(pos):
    """max over agent pairs of |d(downwash force)/d(dz)| [N/m] at positions [N,3]
    (Quadcopter.py:99-115: F = -dw1 (pr/(4 dz))^2 exp(-0.5 (dxy/(dw2 dz + dw3))^2), dz > 0).  The
    force is singular at dz -> 0+: a trajectory that passes such a point amplifies float32
    position rounding (1e-7 m) into a visible velocity kick, in the reference's own dynamics."""
    p = np.asarray(pos, np.float64)
    rel = p[None, :, :] - p[:, None, :]
    dz = rel[..., 2]
    dxy = np.sqrt(rel[..., 0] ** 2 + rel[..., 1] ** 2)
    def F(dz):
        with np.errstate(all='ignore'):
            a = 2267.18 * (2.31348e-2 / (4 * dz)) ** 2
            b = 0.16 * dz - 0.11
            return np.where((dz > 0) & (dxy < 10), a * np.exp(-0.5 * (dxy / b) ** 2), 0.0)
    h = 1e-6
    with np.errstate(all='ignore'):
        S = np.abs(F(dz + h) - F(dz - h)) / (2 * h)
    S = np.where(np.isfinite(S), S, np.inf)
    np.fill_diagonal(S, 0.0)
    return float(S.max())


def first_singular_step(g, limit=1.0e3):
    """first step of a golden trajectory whose PRE-step positions have a downwash sensitivity above
    `limit` N/m (a 2e-7 m position rounding then changes the force by > 2e-4 N = 0.1 % of the
    weight); T if none."""
    T = int(g['T'])
    prev = g['start_pos']
    for t in range(T):
        if downwash_sensitivity(prev) > limit:
            return t
        prev = g['pos'][t]
    return T
