"""The wide start-state sampler's specification (spawn_spec.py, the numpy restatement of mrs_spawn for N > 32), with
no GPU: its RNG key packing, its output distribution against the host sampler, and its failure count."""
import numpy as np
import torch
from scipy import stats

import spawn_spec as S


def test_key_packing_is_injective_past_the_warp_packing_limits():
    """(agent, round) -> pre-hash word is injective on a grid that crosses agent 256 and round 4096, where the
    N <= 32 kernel's packing (ge << 20) ^ (lane << 12) ^ round aliases; the full keys of several envs are distinct."""
    agent, rnd = np.meshgrid(np.arange(0, 300), np.concatenate([np.arange(0, 40), np.arange(4080, 4110)]), indexing='ij')
    agent, rnd = agent.ravel(), rnd.ravel()
    assert len(np.unique(S.pre_hash(agent, rnd))) == agent.size
    # the old packing collides there: lane 256 of env 0 is lane 0 of env 1, round 4096 of lane 0 is round 0 of lane 1
    assert S.warp_pre_hash(0, 256, 7) == S.warp_pre_hash(1, 0, 7)
    assert S.warp_pre_hash(3, 0, 4096) == S.warp_pre_hash(3, 1, 0)
    old = np.concatenate([S.warp_pre_hash(e, agent, rnd) for e in range(3)])
    assert len(np.unique(old)) < old.size
    # the full 64-bit keys of three envs (plus the yaw domain) on that grid: all distinct
    keys = np.concatenate([S.key(99, e, agent, rnd) for e in range(3)] +
                          [S.key(99, e, np.arange(300), S.YAW_ROUND) for e in range(3)])
    assert len(np.unique(keys)) == keys.size
    # extremes of the domain stay distinct
    ext = S.pre_hash(np.array([0, 2**31 - 1, 0, 1]), np.array([2**32 - 1, 0, 0, 0]))
    assert len(np.unique(ext)) == 4


def test_splitmix64_matches_the_reference_vectors():
    """splitmix64 as published (Steele, Lea, Flood 2014; Vigna's splitmix64.c): state 0 -> 0xE220A8397B1DCDAF."""
    assert int(S.splitmix64(0)) == 0xE220A8397B1DCDAF
    assert int(S.splitmix64(0x9E3779B97F4A7C15)) == 0x6E789E6AA1B965F4


def test_restatement_output_is_collision_free_in_region_and_uniform():
    E, N, r = 64, 64, 0.3
    z, R = (1.0, 5.0), 3.0
    pos, yaw, failed, margin = S.spawn(5, E, N, r, z=z, xy_radius=R, xy_sigma=R)
    assert not failed.any()
    d = np.linalg.norm(pos[:, :, None] - pos[:, None], axis=-1) + 10 * np.eye(N)
    assert d.min() >= 2 * r - 1e-6
    assert np.linalg.norm(pos[..., :2], axis=-1).max() <= R * (1 + 1e-6)
    assert z[0] <= pos[..., 2].min() and pos[..., 2].max() <= z[1]
    assert yaw.min() >= -np.pi / 2 and yaw.max() <= np.pi / 2
    # z and yaw uniform: Kolmogorov-Smirnov against U[lo, hi] (4096 samples; the rejection thins z only slightly)
    assert stats.kstest(pos[..., 2].ravel(), 'uniform', args=(z[0], z[1] - z[0])).pvalue > 1e-3
    assert stats.kstest(yaw.ravel(), 'uniform', args=(-np.pi / 2, np.pi)).pvalue > 1e-3
    # the same distribution as the host sampler: mean xy radius at N = 64
    torch.manual_seed(0)
    from mrsgym_b200 import DefaultSpawn, sample_start_pos
    host = sample_start_pos(DefaultSpawn(N, z[0], z[1], R), 256, N, r).numpy()
    rs, rh = np.linalg.norm(pos[..., :2], axis=-1), np.linalg.norm(host[..., :2], axis=-1)
    # per-sample sd ~0.65 m over 4096 (restatement) and 16384 (host) samples: 0.05 m is > 4 sigma
    assert abs(rs.mean() - rh.mean()) < 0.05


def test_restatement_is_keyed_by_global_env():
    a = S.spawn(3, 4, 40, 0.3, z=(1.0, 5.0), xy_radius=3.0, xy_sigma=3.0)
    b = S.spawn(3, 2, 40, 0.3, env_offset=2, z=(1.0, 5.0), xy_radius=3.0, xy_sigma=3.0)
    assert np.array_equal(a[0][2:], b[0]) and np.array_equal(a[1][2:], b[1])
    assert not np.array_equal(a[0][0], a[0][1])


def test_infeasible_density_fails_every_env():
    """The reference's default region (r = 1 m disc, z in [1, 3]) cannot hold 64 agents 0.6 m apart."""
    pos, yaw, failed, _ = S.spawn(1, 3, 64, 0.3, max_rounds=50)
    assert failed.all()
    assert np.isfinite(pos).all() and np.isfinite(yaw).all()
