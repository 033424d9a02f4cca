"""The auto-reset restatement (autoreset_spec.py) without a GPU: key distinctness, the draw distribution against the
host sampler, and the done rule's off-by-one on hand-worked tables."""
import numpy as np
import pytest
import torch

import autoreset_spec as AR
import spawn_spec as S


def test_keys_distinct_across_episodes_envs_and_agents():
    # agents 0..599 (the warp packing of mrs_spawn aliases from 256 on), 16 episodes, 24 envs, 3 rounds + the yaw
    ep, env, agent, rnd = np.meshgrid(np.arange(16), np.arange(24), np.arange(600), np.array([0, 1, 2, S.YAW_ROUND]),
                                      indexing='ij')
    k = AR.key(7, env.ravel(), ep.ravel(), agent.ravel(), rnd.ravel())
    assert np.unique(k).size == k.size
    # the warp packing of mrs_spawn does alias there: agent 256 of env 0 is agent 0 of env 1
    w = S.warp_pre_hash(np.array([0, 1]), np.array([256, 0]), np.array([0, 0]))
    assert w[0] == w[1]
    # episode 0 of env e is not mrs_spawn's stream of env e
    assert AR.key(7, 3, 0, 0, 0) != S.key(7, 3, 0, 0)


def test_the_episode_changes_every_draw():
    a = AR.reset_env(5, 2, 1, 8, 0.3)[0]
    b = AR.reset_env(5, 2, 2, 8, 0.3)[0]
    c = AR.reset_env(5, 3, 1, 8, 0.3)[0]
    assert not np.any(a == b) and not np.any(a == c)
    assert np.array_equal(a, AR.reset_env(5, 2, 1, 8, 0.3)[0])


def test_distribution_matches_sample_start_pos():
    from scipy import stats
    from mrsgym_b200.spawn import DefaultSpawn, sample_start_pos
    E, N = 1500, 6
    ours = np.stack([AR.reset_env(11, e, 1 + e % 3, N, 0.3)[0] for e in range(E)])
    torch.manual_seed(0)
    host = sample_start_pos(DefaultSpawn(N), E, N, 0.3).numpy()
    for name, f in (('x', lambda p: p[..., 0]), ('y', lambda p: p[..., 1]), ('z', lambda p: p[..., 2]),
                    ('radius', lambda p: np.linalg.norm(p[..., :2], axis=-1)),
                    ('agent 0 radius', lambda p: np.linalg.norm(p[:, 0, :2], axis=-1)),
                    ('agent N-1 radius', lambda p: np.linalg.norm(p[:, -1, :2], axis=-1))):
        assert stats.ks_2samp(f(ours).ravel(), f(host).ravel()).pvalue > 1e-3, name
    d = np.linalg.norm(ours[:, :, None] - ours[:, None], axis=-1) + 10 * np.eye(N)
    assert d.min() >= 0.6 * (1 - 1e-6)
    assert np.linalg.norm(ours[..., :2], axis=-1).max() <= 1.0 + 1e-6


# (n before the step, done_fn, episode_length, max_timesteps) -> done; worked by hand from the two readings of the
# count: MRS.step calls done_fn before `steps += 1` (env.py), rollout() tests episode_length after it
TABLE = [
    (0, False, 0, -1, False),      # no limit at all
    (0, True, 0, -1, True),        # done_fn alone
    (0, False, 1, -1, True),       # episode_length 1: every step ends an episode
    (1, False, 3, -1, False),      # second step of an episode of 3
    (2, False, 3, -1, True),       # third step: count after = 3 >= 3
    (2, False, 0, 3, False),       # MAX_TIMESTEPS 3 sees 2 before the increment
    (3, False, 0, 3, True),        # ... and ends on the fourth step
    (0, False, 0, 0, True),        # MAX_TIMESTEPS 0: done at once
    (2, False, 3, 3, True),        # episode_length wins by one step
    (4, False, 10, 5, False),
    (5, False, 10, 5, True),
    (8, False, 10, 50, False),
    (9, False, 10, 50, True),
]


@pytest.mark.parametrize('n,done_in,episode_length,max_timesteps,want', TABLE)
def test_done_rule_table(n, done_in, episode_length, max_timesteps, want):
    assert AR.done_rule(n, done_in, episode_length, max_timesteps) == want


def test_done_rule_over_episodes():
    # episode_length 3: steps 2, 5, 8 end an episode; MAX_TIMESTEPS 3: steps 3, 7
    done, counts = AR.run_counters(10, episode_length=3)
    assert np.flatnonzero(done).tolist() == [2, 5, 8]
    assert counts.tolist() == [1, 2, 0, 1, 2, 0, 1, 2, 0, 1]
    done, _ = AR.run_counters(10, max_timesteps=3)
    assert np.flatnonzero(done).tolist() == [3, 7]
    # an env that enters the loop 4 steps into its episode ends on its 6th step of episode_length 6 = loop step 1
    done, _ = AR.run_counters(8, n0=4, episode_length=6)
    assert np.flatnonzero(done).tolist() == [1, 7]
    # done_fn at step 4 restarts the count
    fn = np.zeros(10, bool)
    fn[4] = True
    done, _ = AR.run_counters(10, done_in=fn, episode_length=4)
    assert np.flatnonzero(done).tolist() == [3, 4, 8]
