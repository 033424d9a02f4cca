"""numpy restatement of the on-device auto-reset (mrs_autoreset): the episode-keyed start-state draws and the done rule.

The draws and the rejection rule are those of mrs_spawn (spawn_spec.py); only the key differs: ONE packing for every
N, (agent, round) under a hash of (global env, episode), so a reset depends on (seed, env_offset + e, episode) alone.
splitmix64 runs in uint64, the draws and pair tests in float32, and the smallest margin |d^2 - 4 r^2| of the pair
tests made is reported as in spawn_spec.
"""
from __future__ import annotations

import numpy as np

from spawn_spec import YAW_ROUND, draw, pre_hash, splitmix64, u01

_U64 = np.uint64
_F32 = np.float32
EPISODE_SALT = 0xD1B54A32D192ED03


def env_hash(global_env, episode):
    """The per-(env, episode) hash the (agent, round) word is packed under."""
    return splitmix64(splitmix64(np.asarray(global_env, dtype=_U64))
                      ^ splitmix64(_U64(EPISODE_SALT) ^ np.asarray(episode, dtype=_U64)))


def key(seed, global_env, episode, agent, rnd):
    return splitmix64(_U64(seed) ^ splitmix64(env_hash(global_env, episode) ^ pre_hash(agent, rnd)))


def reset_env(seed, global_env, episode, N, agent_radius, z=(1.0, 3.0), xy_radius=1.0, xy_sigma=1.0,
              yaw=(-np.pi / 2, np.pi / 2), max_rounds=256):
    """Start of episode `episode` of one env -> (pos [N, 3] f32, yaw [N] f32, failed, smallest margin, rounds)."""
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
        pos[m] = draw(key(seed, global_env, episode, m, rnd), z[0], z[1], xy_radius, xy_sigma)
        d = pos[m][:, None, :] - pos[None, :, :]
        d2 = d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1] + d[..., 2] * d[..., 2]
        tested = m[:, None] != agents[None, :]
        if tested.any():
            margin = min(margin, float(np.abs(d2[tested].astype(np.float64) - float(lim2)).min()))
        close = tested & (d2 < lim2)
        flagged = np.zeros(N, bool)
        flagged[np.maximum(m[:, None], agents[None, :])[close]] = True          # the higher agent of a close pair
        moved = flagged
        if not flagged.any():
            failed = False
            break
    yaws = _F32(yaw[0]) + (_F32(yaw[1]) - _F32(yaw[0])) * u01(key(seed, global_env, episode, agents, YAW_ROUND))
    return pos, yaws.astype(_F32), failed, margin, rounds


def done_rule(n, done_in=False, episode_length=0, max_timesteps=-1):
    """done of one env whose count since its last reset is n BEFORE this step: done_fn's verdict, MAX_TIMESTEPS as the
    default done_fn sees it (the count before the step's increment), episode_length on the count after it."""
    return bool(done_in) or (max_timesteps >= 0 and n >= max_timesteps) or (episode_length > 0 and n + 1 >= episode_length)


def run_counters(T, n0=0, done_in=None, episode_length=0, max_timesteps=-1):
    """T steps of one env's bookkeeping from count n0 -> (done [T] bool, count after every step [T])."""
    done, counts, n = [], [], n0
    for t in range(T):
        d = done_rule(n, False if done_in is None else done_in[t], episode_length, max_timesteps)
        n = 0 if d else n + 1
        done.append(d)
        counts.append(n)
    return np.array(done), np.array(counts)
