"""numpy restatement of the wide start-state sampler (`spawn_wide_kernel`, mrs_spawn for N > 32).

splitmix64 runs in uint64, so the uniform variates are the kernel's bits exactly; the draws and the pair tests run in
float32.  Every pair test made is reported through its margin |d^2 - 4 r^2|: a GPU that rounds a few ulp differently
can only flip a test whose margin is of that order, so a test holds the GPU to this restatement when the smallest
margin is well above float32 rounding.
"""
from __future__ import annotations

import numpy as np

_U64 = np.uint64
_F32 = np.float32
YAW_ROUND = 0xFFFFFFFF          # the yaw's key domain: a round index no draw uses (max_rounds is an int)


def splitmix64(x):
    x = np.asarray(x, dtype=_U64)
    with np.errstate(over='ignore'):
        x = x + _U64(0x9E3779B97F4A7C15)
        x = (x ^ (x >> _U64(30))) * _U64(0xBF58476D1CE4E5B9)
        x = (x ^ (x >> _U64(27))) * _U64(0x94D049BB133111EB)
    return x ^ (x >> _U64(31))


def pre_hash(agent, rnd):
    """The word under the per-env hash: (agent << 32) | round, injective for agent < 2^32 and round < 2^32."""
    return (np.asarray(agent, dtype=_U64) << _U64(32)) | np.asarray(rnd, dtype=_U64)


def key(seed, global_env, agent, rnd):
    return splitmix64(_U64(seed) ^ splitmix64(splitmix64(_U64(global_env)) ^ pre_hash(agent, rnd)))


def warp_pre_hash(global_env, lane, rnd):
    """The N <= 32 kernel's packing (spawn_kernel): aliases once lane >= 256 or round >= 4096."""
    return ((np.asarray(global_env, dtype=_U64) << _U64(20)) ^ (np.asarray(lane, dtype=_U64) << _U64(12))
            ^ np.asarray(rnd, dtype=_U64))


def u01(h):
    return ((np.asarray(h, dtype=_U64) >> _U64(40)).astype(_F32) + _F32(0.5)) * _F32(1.0 / 16777216.0)


def draw(k, z_lo, z_hi, xy_radius, xy_sigma):
    """Box-Muller xy (sigma xy_sigma) pulled onto the disc of radius xy_radius, z ~ U[z_lo, z_hi]: float32."""
    u1 = u01(k)
    u2 = u01(splitmix64(k))
    u3 = u01(splitmix64(k ^ _U64(0x5851F42D4C957F2D)))
    r = _F32(xy_sigma) * np.sqrt(_F32(-2.0) * np.log(u1))
    ang = _F32(6.28318530717958647692) * u2
    x, y = r * np.cos(ang), r * np.sin(ang)
    R = _F32(xy_radius)
    mag = np.maximum(np.sqrt(x * x + y * y), R)
    x, y = x / mag * R, y / mag * R
    z = _F32(z_lo) + (_F32(z_hi) - _F32(z_lo)) * u3
    return np.stack([x, y, z], axis=-1).astype(_F32)


def spawn_env(seed, global_env, N, agent_radius, z=(1.0, 3.0), xy_radius=1.0, xy_sigma=1.0,
              yaw=(-np.pi / 2, np.pi / 2), max_rounds=256):
    """One env -> (pos [N, 3] f32, yaw [N] f32, failed bool, smallest margin of the pair tests made, rounds)."""
    lim2 = _F32(4.0) * _F32(agent_radius) * _F32(agent_radius)
    agents = np.arange(N)
    pos = np.zeros((N, 3), _F32)
    moved = np.ones(N, bool)
    margin = np.inf
    failed = True
    rounds = 0
    for rnd in range(max_rounds):
        rounds = rnd + 1
        m = np.flatnonzero(moved)
        pos[m] = draw(key(seed, global_env, m, rnd), z[0], z[1], xy_radius, xy_sigma)
        # every pair with a mover: two agents that did not move were apart in the previous round already
        flagged = np.zeros(N, bool)
        for c0 in range(0, len(m), 512):
            mc = m[c0:c0 + 512]
            d = pos[mc][:, None, :] - pos[None, :, :]
            d2 = d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1] + d[..., 2] * d[..., 2]
            tested = mc[:, None] != agents[None, :]
            if tested.any():
                margin = min(margin, float(np.abs(d2[tested].astype(np.float64) - float(lim2)).min()))
            close = tested & (d2 < lim2)
            flagged[np.maximum(mc[:, None], agents[None, :])[close]] = True     # the higher agent of a close pair
        moved = flagged
        if not flagged.any():
            failed = False
            break
    ky = key(seed, global_env, agents, YAW_ROUND)
    yaws = _F32(yaw[0]) + (_F32(yaw[1]) - _F32(yaw[0])) * u01(ky)
    return pos, yaws.astype(_F32), failed, margin, rounds


def spawn(seed, E, N, agent_radius, env_offset=0, **kw):
    """E envs -> (pos [E, N, 3], yaw [E, N], failed [E] bool, smallest margin over all envs)."""
    pos = np.zeros((E, N, 3), _F32)
    yaws = np.zeros((E, N), _F32)
    failed = np.zeros(E, bool)
    margin = np.inf
    for e in range(E):
        pos[e], yaws[e], failed[e], mg, _ = spawn_env(seed, env_offset + e, N, agent_radius, **kw)
        margin = min(margin, mg)
    return pos, yaws, failed, margin
