"""mrs_spawn for N > 32 (spawn_wide_kernel, a CTA per env) on the GPU: parity with the numpy restatement
(spawn_spec.py), invariants, determinism across batch shapes and masks, the failure count, and MRS.reset / rollout()
with DefaultSpawn at N > 32 without the host sampler."""
import numpy as np
import pytest
import torch

import spawn_spec as S

pytestmark = pytest.mark.gpu

R_AGENT = 0.3
# (E, N, (z_lo, z_hi, xy_radius), seed): N not a multiple of 32, N above the CTA size (1024), one env of 4096 agents.
# The seeds are those whose smallest pair-test margin clears the rounding bound below with the most room.
SHAPES = [(1024, 64, (1.0, 5.0, 3.0), 14), (64, 200, (1.0, 5.0, 4.0), 8), (1, 4096, (1.0, 17.0, 16.0), 4),
          (4, 33, (1.0, 5.0, 3.0), 1), (2, 1500, (1.0, 9.0, 9.0), 12)]


def _rounding_bound(region):
    """The largest |d^2 - 4 r^2| a float32 restatement and the GPU can disagree on: each coordinate within 8 ulp of
    the region's largest coordinate (the draw is a handful of correctly or nearly correctly rounded float32 ops),
    so |d| moves by at most 2 sqrt(3) such errors near d = 2r, plus the rounding of d^2 itself."""
    cmax = max(abs(region[1]), region[2])
    eps = 8 * 2.0 ** -24 * cmax
    return 2 * (2 * R_AGENT) * 2 * np.sqrt(3) * eps + 8 * 2.0 ** -24 * 4 * R_AGENT ** 2


def _swarm(E, N):
    import mrsgym_b200 as M
    return M.Swarm(E, N, 0, 'set_target_vel', M._abi.X_POS_VEL, want_A=False)


def _spawn(sw, seed, region, **kw):
    z_lo, z_hi, R = region
    return sw.spawn(seed, z=(z_lo, z_hi), xy_radius=R, xy_sigma=R, **kw)


def _planes(sw):
    return sw.state.reshape(13, sw.E, sw.N)


@pytest.mark.parametrize('E,N,region,seed', SHAPES)
def test_matches_the_restatement(E, N, region, seed):
    pos, yaw, failed, margin = S.spawn(seed, E, N, R_AGENT, z=region[:2], xy_radius=region[2], xy_sigma=region[2])
    assert not failed.any()
    # no pair test of the restatement is a rounding tie: a GPU mismatch below is a defect
    assert margin > _rounding_bound(region), (margin, _rounding_bound(region))
    sw = _swarm(E, N)
    f = _spawn(sw, seed, region)
    torch.cuda.synchronize()
    assert int(f.item()) == 0
    np.testing.assert_allclose(sw.get_pos().cpu().numpy(), pos, rtol=0, atol=1e-5)
    q = sw.get_quat().cpu().numpy().astype(np.float64)
    np.testing.assert_allclose(2 * np.arctan2(q[..., 2], q[..., 3]), yaw, rtol=0, atol=1e-6)


@pytest.mark.parametrize('E,N,region,seed', SHAPES)
def test_invariants(E, N, region, seed):
    z_lo, z_hi, R = region
    sw = _swarm(E, N)
    f = _spawn(sw, seed + 1000, region)
    assert int(f.item()) == 0
    p = sw.get_pos().double()
    d2 = ((p.unsqueeze(2) - p.unsqueeze(1)) ** 2).sum(-1) + 100 * torch.eye(N, device=p.device, dtype=p.dtype)
    assert float(d2.min()) >= 4 * R_AGENT ** 2 * (1 - 1e-6)
    assert float(p[..., :2].norm(dim=-1).max()) <= R * (1 + 1e-6)
    assert z_lo <= float(p[..., 2].min()) and float(p[..., 2].max()) <= z_hi
    q = sw.get_quat()
    assert float(q[..., :2].abs().max()) == 0.0
    assert float((q.norm(dim=-1) - 1).abs().max()) < 1e-6
    yaw = 2 * torch.atan2(q[..., 2].double(), q[..., 3].double())
    assert float(yaw.abs().max()) <= np.pi / 2 + 1e-6
    assert float(sw.get_vel().abs().max()) == 0.0 and float(sw.get_angvel().abs().max()) == 0.0


def test_determinism_batch_and_mask():
    E, N, region = 48, 100, (1.0, 5.0, 3.0)
    sw = _swarm(E, N)
    _spawn(sw, 21, region)
    ref = sw.state.clone()
    _spawn(sw, 21, region)
    assert torch.equal(sw.state, ref), 'the same seed twice'
    # env e of the batch = a one-env spawn with env_offset = e
    one = _swarm(1, N)
    for e in (0, 17, 47):
        _spawn(one, 21, region, env_offset=e)
        assert torch.equal(_planes(one)[:, 0], _planes(sw)[:, e])
    # a masked spawn writes the selected envs as an unmasked spawn with that seed does, and no others
    other = _swarm(E, N)
    _spawn(other, 77, region)
    full77 = other.state.clone()
    mask = torch.zeros(E, dtype=torch.bool)
    mask[::5] = True
    mask[7] = True
    _spawn(sw, 77, region, env_mask=mask)
    m = mask.cuda()
    assert torch.equal(_planes(sw)[:, m], full77.reshape(13, E, N)[:, m])
    assert torch.equal(_planes(sw)[:, ~m], ref.reshape(13, E, N)[:, ~m])


def test_infeasible_density_counts_every_env():
    E, N = 6, 64
    sw = _swarm(E, N)
    f = sw.spawn(3, max_rounds=40)          # the reference's default region: r = 1 m, z in [1, 3]
    assert int(f.item()) == E
    assert bool(torch.isfinite(sw.state).all())
    pos, yaw, failed, _ = S.spawn(3, E, N, R_AGENT, max_rounds=40)
    assert failed.all()
    # a masked call counts only the selected envs
    mask = torch.tensor([True, False, True, False, False, False])
    f2 = sw.spawn(4, env_mask=mask, max_rounds=40)
    assert int(f2.item()) == 2


def test_mrs_default_region_at_64_agents_raises():
    import mrsgym_b200 as M
    with pytest.raises(RuntimeError, match='did not converge'):
        M.MRS(N_AGENTS=64)


def _mrs(**kw):
    import mrsgym_b200 as M
    base = dict(N_AGENTS=64, N_ENVS=1024, START_POS=M.DefaultSpawn(64, 1, 5, 3), COMM_RANGE=2.0,
                ACTION_TYPE='set_target_vel', SEED=9)
    base.update(kw)
    return M.MRS(**base)


def test_mrs_resets_on_the_device(monkeypatch):
    import mrsgym_b200 as M

    def host_sampler(*a, **k):
        raise AssertionError('sample_start_pos called for DefaultSpawn')
    monkeypatch.setattr(M.spawn, 'sample_start_pos', host_sampler)
    env = _mrs()
    assert int(env.spawn_failed.item()) == 0
    rng = torch.get_rng_state()
    env.reset()
    mask = torch.zeros(1024, dtype=torch.bool)
    mask[::3] = True
    env.reset(env_mask=mask)
    assert torch.equal(torch.get_rng_state(), rng), 'the device spawn touched the CPU generator'
    p = env.env.get_pos()
    d = (p.unsqueeze(2) - p.unsqueeze(1)).norm(dim=-1) + 10 * torch.eye(64, device=p.device)
    assert float(d.min()) >= 2 * R_AGENT - 1e-6
    # same SEED => same start; ENV_OFFSET shards are the halves of the whole
    a, b = _mrs(), _mrs()
    assert torch.equal(a.swarm.state, b.swarm.state)
    lo, hi = _mrs(N_ENVS=512, ENV_OFFSET=0), _mrs(N_ENVS=512, ENV_OFFSET=512)
    pw = a.env.get_pos()
    assert torch.equal(pw[:512], lo.env.get_pos()) and torch.equal(pw[512:], hi.env.get_pos())
    assert not torch.equal(lo.env.get_pos(), hi.env.get_pos())


def test_rollout_auto_resets_only_finished_envs(monkeypatch):
    import mrsgym_b200 as M

    def host_sampler(*a, **k):
        raise AssertionError('sample_start_pos called for DefaultSpawn')
    monkeypatch.setattr(M.spawn, 'sample_start_pos', host_sampler)
    E, N = 1024, 64
    env = _mrs(K_HOPS=1)
    pol = M.reynolds_policy()
    for _ in range(3):
        env.step(pol(env.get_Xk(), env.calc_Ak()))
    odd = torch.arange(E) % 2 == 1
    env.reset(env_mask=~odd)          # even envs restart: odd envs are 3 steps ahead
    env.refresh_A(~odd)
    oc, ec = odd.cuda(), (~odd).cuda()
    # three steps: the odd envs reach episode_length 6 after the last one and are reset
    first = M.rollout(env, pol, 3, episode_length=6)
    assert torch.equal(first['done'].cpu(), torch.stack([torch.zeros(E, dtype=torch.bool)] * 2 + [odd]))
    W = env.get_Xk()                   # [E, 2, N, 6], newest first
    # the reset envs: both slices are the new start; the others keep their history (newest before it = step 2's input)
    assert torch.equal(W[oc][:, 0], W[oc][:, 1])
    assert torch.equal(W[ec][:, 1], first['X'][2][ec])
    assert not torch.equal(W[ec][:, 0], W[ec][:, 1])
    second = M.rollout(env, pol, 5, episode_length=6)
    data = {k: torch.cat([first[k], second[k]]) for k in ('X', 'done')}
    done = data['done'].cpu()
    assert torch.equal(done[5], ~odd) and not done[[0, 1, 3, 4, 6, 7]].any()
    X = data['X']
    # the odd envs start again at step 3: a fresh collision-free draw with zero velocity, in the region
    fresh = X[3][oc]
    assert float(fresh[..., 3:6].abs().max()) == 0.0
    p = fresh[..., :3]
    d = (p.unsqueeze(2) - p.unsqueeze(1)).norm(dim=-1) + 10 * torch.eye(N, device=p.device)
    assert float(d.min()) >= 2 * R_AGENT - 1e-6
    assert float(p[..., :2].norm(dim=-1).max()) <= 3.0 + 1e-5
    # the even envs keep flying: no jump between steps 2 and 3 (|v| <= ~1 m/s, dt = 0.01 s)
    assert float((X[3][ec][..., :3] - X[2][ec][..., :3]).norm(dim=-1).max()) < 0.05
    assert float(X[3][ec][..., 3:6].abs().max()) > 0.0
    assert env.env_steps[ec].eq(2).all() and env.env_steps[oc].eq(5).all()
    env.check_status()
