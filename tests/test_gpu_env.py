"""The reference-facing Python surface (mrsgym_b200.make('mrs-v0') / MRS.step) on the GPU:
shapes, callback order, error behaviour and the README example against the golden the
reference's own Python produced."""
import os

import numpy as np
import pytest
import torch

import helpers as H
from conftest import GOLDEN

pytestmark = pytest.mark.gpu


def test_readme_example_c1_vs_golden():
    """BASELINE configs[0]: 'simple' env, N_AGENTS=3, set_target_vel, K_HOPS=0 (README.md:21-40)."""
    import mrsgym_b200 as mrsgym
    g = np.load(os.path.join(GOLDEN, 'ref_c1_vel.npz'))
    env = mrsgym.make('mrs-v0', state_fn=lambda quad: torch.cat([quad.get_pos(), quad.get_vel()]),
                      N_AGENTS=3, K_HOPS=0, ACTION_TYPE='set_target_vel', HEADLESS=True,
                      START_POS=torch.tensor(g['start_pos'], dtype=torch.float32), START_ORI=torch.zeros(3, 3))
    assert env.STATE_SIZE == 6
    X0 = env.reset()
    assert tuple(X0.shape) == (1, 3, 6)
    np.testing.assert_allclose(X0.cpu().numpy(), g['X0'], atol=1e-6)
    for t in range(int(g['T'])):
        X, reward, done, info = env.step(torch.tensor(g['actions'][t]))
        assert tuple(X.shape) == (1, 3, 6) and tuple(info['A'].shape) == (1, 3, 3)
        assert reward == 0.0 and done is False
    np.testing.assert_allclose(X.cpu().numpy(), g['X'][-1], atol=1e-3)
    np.testing.assert_array_equal(info['A'].cpu().numpy(), g['A'][-1])


def test_callbacks_order_and_arguments():
    import mrsgym_b200 as mrsgym
    log = []

    def update_fn(**kw):
        log.append(('update', kw['steps_since_reset'], kw['Xlast'] is kw['X']))

    def reward_fn(**kw):
        log.append(('reward', kw['steps_since_reset'], kw['Xlast'] is kw['X']))
        return 1.5

    def info_fn(**kw):
        log.append(('info', kw['steps_since_reset'], kw['Xlast'] is kw['X']))
        return {'n': kw['env'].get_pos().shape[0]}

    def done_fn(**kw):
        log.append(('done', kw['steps_since_reset'], kw['Xlast'] is kw['X']))
        return kw['steps_since_reset'] >= 1

    env = mrsgym.MRS(state_fn='pos_vel', reward_fn=reward_fn, info_fn=info_fn, update_fn=update_fn, done_fn=done_fn,
                     N_AGENTS=4, K_HOPS=2, COMM_RANGE=5.0, START_POS=torch.tensor(H.grid_positions(1, 4)[0]),
                     START_ORI=torch.zeros(4, 3))
    X, r, d, info = env.step(torch.zeros(4, 3))
    # reference order: update, reward, (last_obs := X), info, done; callbacks see the pre-increment
    # counter; info_fn / done_fn see Xlast is X (MRS.py:260-274)
    assert [l[0] for l in log] == ['update', 'reward', 'info', 'done']
    assert [l[1] for l in log] == [0, 0, 0, 0]
    assert [l[2] for l in log] == [False, False, True, True]
    assert r == 1.5 and d is False and info['n'] == 4 and 'A' in info
    assert env.steps_since_reset == 1
    X, r, d, info = env.step(torch.zeros(12))          # flat actions are reshaped (MRS.py:245-246)
    assert d is True
    assert tuple(X.shape) == (3, 4, 6) and tuple(info['A'].shape) == (3, 4, 4)


def test_error_behaviour():
    import mrsgym_b200 as mrsgym
    env = mrsgym.MRS(N_AGENTS=2, START_POS=torch.tensor([[0., 0, 1], [1, 0, 1]]), START_ORI=torch.zeros(2, 3))
    with pytest.raises(Exception, match='NaN'):
        env.step(torch.tensor([[float('nan'), 0, 0], [0, 0, 0]]))
    with pytest.raises(AttributeError):
        env.step(torch.zeros(2, 3), ACTION_TYPE='set_nothing')
    # device-resident NaN actions: flagged by the kernel, raised lazily
    env.step(torch.full((2, 3), float('nan'), device='cuda'))
    with pytest.raises(Exception, match='NaN'):
        env.check_status()
    with pytest.raises(mrsgym.MrsError):
        mrsgym.Swarm(1, 2, device='cpu')
    # raw-pointer boundary: wrong shape / dtype / device never reaches the C ABI
    sw = mrsgym.Swarm(4, 2, 0, 'set_speeds')
    for bad in (torch.zeros(4, 2, 3, device='cuda'), torch.zeros(4, 2, 4, device='cuda', dtype=torch.float64),
                torch.zeros(4, 2, 4), torch.zeros(4, 2, 8, device='cuda')[..., ::2], None):
        with pytest.raises(ValueError):
            sw.step(bad)
    lib = mrsgym._abi.lib()
    import ctypes
    assert lib.mrs_step(ctypes.byref(sw.cfg), ctypes.byref(sw.bufs), None, 0, 0, None) == -1      # NULL actions
    assert lib.mrs_step(ctypes.byref(sw.cfg), ctypes.byref(sw.bufs), ctypes.c_void_p(sw.state.data_ptr()), sw.L, 0, None) == -1   # slot out of range


def test_batched_env_shapes_and_modes():
    import mrsgym_b200 as mrsgym
    E, N, K = 16, 8, 3
    pos = torch.tensor(H.grid_positions(E, N, z0=3.0), dtype=torch.float32)
    env = mrsgym.make('mrs-v0', N_ENVS=E, N_AGENTS=N, K_HOPS=K, COMM_RANGE=2.0, ACTION_TYPE='set_target_pos',
                      START_POS=pos, state_fn='full')
    X, r, d, info = env.step(pos.cuda() + 0.1)
    assert tuple(X.shape) == (E, K + 1, N, 13) and tuple(info['A'].shape) == (E, K + 1, N, N)
    for mode, adim in [('set_speeds', 4), ('set_control', 4), ('set_force', 3), ('set_target_ori', 3),
                       ('set_target_accel', 3), ('set_target_vel', 3)]:
        a = torch.zeros(E, N, adim)
        if mode == 'set_speeds':
            a += H.HOVER
        if mode == 'set_control':
            a[..., 0] = 9.81
        X, r, d, info = env.step(a, ACTION_TYPE=mode)
        assert env.ACTION_DIM == adim
    assert torch.isfinite(X).all()
    env.check_status()
    # no action at all (MRS.step(None)): free fall, still returns observations
    z0 = env.env.get_pos()[..., 2].clone()
    env.step(None)
    assert bool((env.env.get_pos()[..., 2] < z0).all())
    # calc_Ak outside step shifts only the A ring (DataGenerator.py:23)
    Xk = env.get_Xk().clone()
    Ak = env.calc_Ak()
    assert torch.equal(env.get_Xk(), Xk) and torch.equal(Ak[:, 0], Ak[:, 1])


def test_default_reset_spawns_collision_free():
    import mrsgym_b200 as mrsgym
    env = mrsgym.MRS(N_ENVS=8, N_AGENTS=6)
    p = env.env.get_pos()
    d = (p.unsqueeze(2) - p.unsqueeze(1)).norm(dim=-1) + 10 * torch.eye(6, device=p.device)
    assert float(d.min()) >= 2 * env.AGENT_RADIUS
    yaw = env.env.get_ori()[..., 2]
    assert float(yaw.abs().max()) <= np.pi / 2 + 1e-5
    X = env.reset()
    assert tuple(X.shape) == (8, 1, 6, 6)


def test_device_spawn_distribution_and_determinism():
    """mrs_spawn: the reference's default start distribution (MRS.py:69-78,127-161) sampled on the
    device -- separation >= 2*AGENT_RADIUS, xy inside the unit disc, z ~ U[1,3], yaw ~ U[-pi/2, pi/2],
    zero velocities; reproducible from the seed; masked resets touch only the selected envs."""
    import mrsgym_b200 as mrsgym
    E, N = 4096, 8
    sw = mrsgym.Swarm(E, N, 0, 'set_speeds')
    failed = sw.spawn(seed=123)
    p = sw.get_pos()
    assert int(failed.item()) == 0
    d = (p.unsqueeze(2) - p.unsqueeze(1)).norm(dim=-1) + 10 * torch.eye(N, device=p.device)
    assert float(d.min()) >= 0.6 - 1e-6
    assert float(p[..., :2].norm(dim=-1).max()) <= 1.0 + 1e-5
    z = p[..., 2].flatten()
    assert 1.0 <= float(z.min()) and float(z.max()) <= 3.0
    # uniformity of z and yaw (KS distance against the uniform CDF; 32768 samples => 0.01 is > 5 sigma)
    for v, lo, hi in ((z, 1.0, 3.0), (sw.get_ori()[..., 2].flatten(), -np.pi / 2, np.pi / 2)):
        u = ((v - lo) / (hi - lo)).sort().values.cpu().double()
        n = u.numel()
        ks = (u - (torch.arange(n, dtype=torch.float64) + 0.5) / n).abs().max()
        assert float(ks) < 0.015
    assert float(sw.get_vel().abs().max()) == 0.0 and float(sw.get_angvel().abs().max()) == 0.0
    assert float((sw.get_quat().norm(dim=-1) - 1).abs().max()) < 1e-6
    # against the host sampler of the reference's distribution: same marginal radius statistics
    host = mrsgym.sample_start_pos(mrsgym.DefaultSpawn(N), 2048, N, 0.3)
    assert abs(float(host[..., :2].norm(dim=-1).mean()) - float(p[..., :2].norm(dim=-1).mean())) < 0.02
    # determinism and masking
    ref = sw.state.clone()
    sw.spawn(seed=123)
    assert torch.equal(sw.state, ref)
    mask = torch.zeros(E, dtype=torch.bool)
    mask[::3] = True
    sw.spawn(seed=999, env_mask=mask)
    new = sw.state.reshape(13, E, N)
    old = ref.reshape(13, E, N)
    assert torch.equal(new[:, ~mask.cuda()], old[:, ~mask.cuda()])
    assert not torch.equal(new[0, mask.cuda()], old[0, mask.cuda()])


def test_masked_reset_keeps_other_envs_history():
    import mrsgym_b200 as mrsgym
    E, N, K = 6, 4, 2
    env = mrsgym.MRS(N_ENVS=E, N_AGENTS=N, K_HOPS=K, COMM_RANGE=3.0, ACTION_TYPE='set_target_vel', SEED=5)
    for _ in range(4):
        X, r, d, info = env.step(torch.zeros(E, N, 3))
    Xb, Ab = env.get_Xk().clone(), env.get_Ak().clone()
    mask = torch.tensor([True, False, False, True, False, False])
    X = env.reset(env_mask=mask)
    keep = ~mask.cuda()
    assert torch.equal(X[keep], Xb[keep]) and torch.equal(env.get_Ak()[keep], Ab[keep])
    # the reset envs: X history = copies of the new X0, A history = zeros, step counter back to 0
    assert torch.equal(X[mask.cuda()][:, 0], X[mask.cuda()][:, K])
    assert float(env.get_Ak()[mask.cuda()].abs().sum()) == 0.0
    assert env.env_steps.tolist() == [0, 4, 4, 0, 4, 4]
    assert not torch.equal(X[mask.cuda()][:, 0], Xb[mask.cuda()][:, 0])
    env.step(torch.zeros(E, N, 3))
    env.check_status()


def test_on_device_rollout_with_reynolds_policy():
    """rollout(): closed loop policy -> step on the device with per-env auto-reset and a dataset of
    device tensors (the generate_mrs loop of examples/simulating_data/helper/DataGenerator.py:8-48)."""
    import mrsgym_b200 as mrsgym
    E, N, K, T = 64, 8, 1, 30
    env = mrsgym.MRS(N_ENVS=E, N_AGENTS=N, K_HOPS=K, COMM_RANGE=2.5, ACTION_TYPE='set_target_vel', SEED=11,
                     reward_fn=lambda **kw: -kw['X'][:, 0, :, 3:6].norm(dim=-1).mean(dim=-1),
                     done_fn=lambda **kw: kw['X'][:, 0, :, 2].min(dim=-1).values < 0.6)
    pol = mrsgym.reynolds_policy()
    data = mrsgym.rollout(env, pol, T, episode_length=12)
    assert tuple(data['X'].shape) == (T, E, N, 6) and tuple(data['A'].shape) == (T, E, N, N)
    assert tuple(data['action'].shape) == (T, E, N, 3) and tuple(data['reward'].shape) == (T, E)
    assert data['done'].dtype == torch.bool and all(v.is_cuda for v in data.values())
    # episode_length 12 => every env is reset at steps 11 and 23 (0-based), and starts again from a
    # collision-free draw with zero velocity
    assert bool(data['done'][11].all()) and bool(data['done'][23].all())
    assert float(data['X'][12][..., 3:6].abs().max()) == 0.0
    p = data['X'][12][..., :3]
    d = (p.unsqueeze(2) - p.unsqueeze(1)).norm(dim=-1) + 10 * torch.eye(N, device=p.device)
    assert float(d.min()) >= 0.6 - 1e-6
    # the recorded A is the adjacency of the recorded X
    from oracle import spec
    np.testing.assert_array_equal(data['A'][5].cpu().numpy(), spec.adjacency(data['X'][5][..., :3].cpu().numpy(), 2.5))
    # flocking: commanded speeds are bounded, the swarm stays finite
    assert float(data['action'].norm(dim=-1).max()) <= 1.0 + 1e-5 and bool(torch.isfinite(data['X']).all())
    env.check_status()
    # reproducible from the seed
    env2 = mrsgym.MRS(N_ENVS=E, N_AGENTS=N, K_HOPS=K, COMM_RANGE=2.5, ACTION_TYPE='set_target_vel', SEED=11,
                      reward_fn=lambda **kw: -kw['X'][:, 0, :, 3:6].norm(dim=-1).mean(dim=-1),
                      done_fn=lambda **kw: kw['X'][:, 0, :, 2].min(dim=-1).values < 0.6)
    data2 = mrsgym.rollout(env2, pol, T, episode_length=12)
    assert torch.equal(data['X'], data2['X']) and torch.equal(data['action'], data2['action'])


def test_rllib_style_wrappers():
    """flat-numpy and dict-per-agent adapters (reference MRSWrapper.py:11-55), no ray needed"""
    import mrsgym_b200 as mrsgym
    pos = torch.tensor(H.grid_positions(1, 3)[0], dtype=torch.float32)
    cfg = dict(N_AGENTS=3, K_HOPS=1, ACTION_TYPE='set_target_vel', START_POS=pos, START_ORI=torch.zeros(3, 3),
               action_fn=lambda a: np.asarray(a) * 0.5)
    flat = mrsgym.make('mrs-rllib-v0', config=cfg)
    obs = flat.reset()
    assert isinstance(obs, np.ndarray) and obs.shape == (2 * 3 * 6,)
    obs, r, d, info = flat.step(np.ones((3, 3), np.float32))
    assert obs.shape == (36,) and 'A' in info
    multi = mrsgym.make('mrs-rllib-multiagent-v0', config=cfg)
    o = multi.reset()
    assert set(o) == {'agent1', 'agent2', 'agent3'} and o['agent2'].shape == (6,)
    o, r, d, info = multi.step({'agent1': [1.0, 0, 0], 'agent3': [0, 1.0, 0]})
    assert set(o) == {'agent1', 'agent2', 'agent3'}
    # both wrappers drive the same dynamics: agent 1 was commanded +x
    for _ in range(20):
        o, r, d, info = multi.step({'agent1': [1.0, 0, 0]})
    assert o['agent1'][3] > 0.05 and abs(o['agent2'][3]) < 0.02


def test_analytic_sensors_vs_oracle():
    """mrs_proximity / mrs_raycast (Object.collision / get_dist / raycast on the simple world's
    primitives) against oracle/sensors.py"""
    import mrsgym_b200 as mrsgym
    import sensor_cases as SC
    E, N = 7, 12
    rng = np.random.default_rng(91)
    st = H.random_state(rng, E, N, spacing=0.62, z0=0.56, jitter=0.05, tilt=0.4)
    st['pos'][:, 6:, 2] += 1.5                               # half of them well above the ground
    sw = mrsgym.Swarm(E, N, 0, 'set_speeds')
    SC.apply(sw, 'r30')
    H.upload_state(sw, st)
    P = SC.phys('r30')
    # margin rule (sensor_cases.py): decisions that clear their float32 bound agree exactly, values within the bound
    p = sw.proximity(0.04)
    v = SC.proximity_verdict(st['pos'], st['quat'], P, 0.04)
    assert (np.abs(p['gap_agent'].cpu().numpy() - v['gap_agent']) <= v['ga_bound']).all()
    assert (np.abs(p['gap_ground'].cpu().numpy() - v['gap_ground']) <= v['gg_bound']).all()
    np.testing.assert_array_equal(p['nearest'].cpu().numpy()[v['nearest_ok']], v['nearest'][v['nearest_ok']])
    np.testing.assert_array_equal(p['collision'].cpu().numpy()[v['collision_ok']], v['collision'][v['collision_ok']])
    assert v['collision'].any() and (~v['collision']).any()
    dirs = np.array([[1, 0, 0], [0, 0, -1], [0.3, -0.5, -0.2], [-1, 1, 0.1], [0, 0, 1]], np.float32)
    for body in (True, False):
        r = sw.raycast(dirs, offset=(0.0, 0.0, -0.02), body=body, RANGE=30.0)
        v = SC.ray_verdict(st['pos'], st['quat'], dirs, body, 30.0, P, offset=(0.0, 0.0, -0.02))
        got_d, got_o = r['dist'].cpu().numpy(), r['object'].cpu().numpy()
        c, obj = v['certain'], v['obj']
        np.testing.assert_array_equal(got_o[c], obj[c])
        hit = c & np.isfinite(v['dist'])
        with np.errstate(invalid='ignore'):            # inf - inf off the hits
            assert (np.abs(got_d - v['dist'])[hit] <= v['bound'][hit]).all()
        assert np.all(np.isinf(got_d[c & ~np.isfinite(v['dist'])]))
        assert (obj == N).any() and ((obj >= 0) & (obj < N)).any() and (obj == -1).any()
    # the env-level view used by reward functions (magent.py:42: -1 if agent.collision() else 0)
    env = mrsgym.MRS(N_ENVS=3, N_AGENTS=4, START_POS=torch.tensor([[0., 0, 0.52], [0.5, 0, 2], [3, 0, 2], [3, 0.5, 2.]]),
                     START_ORI=torch.zeros(4, 3))
    c = env.env.collision()
    assert tuple(c.shape) == (3, 4) and bool(c[:, 0].all())
    assert bool(c[:, 2].all()) and bool(c[:, 3].all()) and not bool(c[:, 1].any())


def test_gym_spaces_like_the_reference():
    """observation_space / action_space as MRS.py:51-52 builds them (flat boxes, the reference's own length
    expression K_HOPS + 1 * N_AGENTS * STATE_SIZE), per-agent boxes on the multi-agent wrapper."""
    import mrsgym_b200 as mrsgym
    from mrsgym_b200.wrappers import MRS_RLlib, MRS_RLlib_MultiAgent
    env = mrsgym.MRS(N_AGENTS=3, K_HOPS=2, START_POS=torch.tensor(H.grid_positions(1, 3)[0]), START_ORI=torch.zeros(3, 3))
    assert env.observation_space.shape == (2 + 1 * 3 * 6,)
    assert env.action_space.shape == (12,)
    np.testing.assert_allclose(env.action_space.low[:4], [8.81, -1, -1, -1], rtol=1e-6)
    np.testing.assert_allclose(env.action_space.high[4:8], [10.81, 1, 1, 1], rtol=1e-6)
    a = env.action_space.sample()
    assert a.shape == (12,) and env.action_space.contains(a)
    cfg = dict(N_AGENTS=3, START_POS=torch.tensor(H.grid_positions(1, 3)[0]), START_ORI=torch.zeros(3, 3))
    flat = MRS_RLlib(dict(cfg))
    assert flat.observation_space.shape == (0 + 18,) and flat.action_space.shape == (12,)
    multi = MRS_RLlib_MultiAgent(dict(cfg, ACTION_TYPE='set_control'))
    assert multi.observation_space.shape == (6,) and multi.action_space.shape == (4,)


def test_get_ori_mat_for_state_fn():
    """Object.get_ori(mat=True) (Object.py:90-95) in a reference-style state_fn: [3, 3, E*N] body->world matrices."""
    import mrsgym_b200 as mrsgym
    from scipy.spatial.transform import Rotation as R
    rpy = torch.tensor([[0.1, -0.2, 0.3], [0.0, 0.4, -1.0], [-0.3, 0.1, 2.0]])

    def state_fn(quad):
        m = quad.get_ori(mat=True)                       # [3, 3, S]
        return torch.cat([quad.get_pos(), m[:, 2, :]])   # position + body z axis in world coordinates

    env = mrsgym.MRS(state_fn=state_fn, N_AGENTS=3, START_POS=torch.tensor(H.grid_positions(1, 3)[0]), START_ORI=rpy)
    X = env.reset()
    assert tuple(X.shape) == (1, 3, 6)
    want = R.from_euler('xyz', rpy.numpy()).as_matrix()[:, :, 2]
    np.testing.assert_allclose(X[0, :, 3:].cpu().numpy(), want, atol=1e-6)
    np.testing.assert_allclose(env.env.get_ori(mat=True).cpu().numpy(), R.from_euler('xyz', rpy.numpy()).as_matrix(), atol=1e-6)


def test_contact_points_and_closest_objects():
    """Object.get_contact_points / get_closest_objects (Object.py:100-141) on the contact geometry of the step"""
    import mrsgym_b200 as mrsgym
    pos = torch.tensor([[0.0, 0.0, 0.5135], [0.55, 0.0, 0.5135], [3.0, 0.0, 2.0]])      # two resting and touching, one aloft
    env = mrsgym.MRS(N_AGENTS=3, START_POS=pos, START_ORI=torch.zeros(3, 3))
    env.reset()
    c = env.env.get_contact_points()
    assert tuple(c['object'].shape) == (3, 5) and tuple(c['pos'].shape) == (3, 5, 3)
    obj = c['object'].cpu().numpy()
    assert obj[0, 0] == 1 and obj[1, 0] == 0 and obj[2, 0] == -1          # sphere contact 0 <-> 1
    assert (obj[0, 1:] == 3).all() and (obj[1, 1:] == 3).all() and (obj[2, 1:] == -1).all()   # 3 = N_AGENTS = the ground
    np.testing.assert_allclose(c['distance'][0, 0].item(), 0.55 - 0.6, atol=1e-6)
    np.testing.assert_allclose(c['distance'][0, 1:].cpu().numpy(), 0.5135 - 0.0125 - 0.001 - 0.5, atol=1e-6)
    np.testing.assert_allclose(c['pos'][0, 1].cpu().numpy(), [0.06, 0.0, 0.501], atol=1e-6)
    np.testing.assert_allclose(c['normal'][0, 0].cpu().numpy(), [-1.0, 0.0, 0.0], atol=1e-6)
    cb = env.env.get_contact_points(body=True)
    np.testing.assert_allclose(cb['pos'][1, 3].cpu().numpy(), [-0.06, 0.0, -0.0125], atol=1e-6)
    near = env.env.get_closest_objects(0.1)
    assert near['mask'].cpu().numpy().tolist() == [[False, True, False], [True, False, False], [False, False, False]]


def test_rpm_mirror_matches_the_reference_anchors():
    """Swarm(keep_rpm=True): the rotor speeds the GPU controller commands against the reference's own numbers for the
    seven anchor cases of SURVEY.md 8(c) (tests/golden/ref_anchor_*.npz, generated from /root/reference)."""
    import glob
    import mrsgym_b200 as M
    files = sorted(glob.glob(os.path.join(GOLDEN, 'ref_anchor_*.npz')))
    assert len(files) >= 7
    for f in files:
        g = np.load(f)
        N, mode = int(g['N']), str(g['mode'])
        sw = M.Swarm(1, N, 0, mode, M._abi.X_POS_VEL, float(g['comm_range']), keep_rpm=True)
        st = {k: g['start_' + k][None].astype(np.float32) for k in ('pos', 'quat', 'vel', 'angvel')}
        H.upload_state(sw, st)
        sw.step(torch.from_numpy(g['actions'][0][None]).cuda())
        rpm = sw.rpm.cpu().numpy().T.reshape(N, 4)
        np.testing.assert_allclose(rpm, g['rpm'][0], rtol=2e-5, err_msg=os.path.basename(f))


def test_shards_spawn_different_environments():
    """mrs_spawn keys its draws by seed and GLOBAL env index: two shards of a job (ENV_OFFSET = the shard's first
    env) sample different start states, and a shard equals the matching slice of the unsharded batch."""
    import mrsgym_b200 as mrsgym
    whole = mrsgym.MRS(N_AGENTS=4, N_ENVS=64, SEED=7)
    lo = mrsgym.MRS(N_AGENTS=4, N_ENVS=32, SEED=7, ENV_OFFSET=0)
    hi = mrsgym.MRS(N_AGENTS=4, N_ENVS=32, SEED=7, ENV_OFFSET=32)
    pw, pl, ph = whole.env.get_pos(), lo.env.get_pos(), hi.env.get_pos()
    assert torch.equal(pw[:32], pl) and torch.equal(pw[32:], ph)
    assert not torch.equal(pl, ph)


def test_batched_default_done_is_per_env():
    import mrsgym_b200 as mrsgym
    env = mrsgym.MRS(N_AGENTS=2, N_ENVS=3, MAX_TIMESTEPS=2)
    a = torch.zeros(3, 2, 3, device='cuda')
    for _ in range(2):
        X, r, done, info = env.step(a)
    assert done.tolist() == [False, False, False]         # evaluated before the counter is incremented (MRS.py:272-274)
    env.reset(env_mask=torch.tensor([False, True, False]))
    X, r, done, info = env.step(a)
    assert done.tolist() == [True, False, True]


def test_device_nan_action_does_not_poison_the_state():
    """A NaN in a device-resident action cannot raise before the step (MRS.py:247-248 does for host actions): that
    agent steps without rotor forces, keeps its PID state, the status bit is raised -- everything stays finite."""
    import mrsgym_b200 as M
    for N in (8, 40):
        sw = M.Swarm(4, N, 0, 'set_target_vel', M._abi.X_POS_VEL, 2.0)
        rng = np.random.default_rng(3)
        st = H.random_state(rng, 4, N)
        H.upload_state(sw, st)
        act = torch.zeros(4, N, 3, device='cuda')
        act[1, 2, 0] = float('nan')
        ctrl0 = sw.ctrl.clone()
        sw.step(act)
        assert bool(torch.isfinite(sw.state).all())
        s = 1 * N + 2
        assert torch.equal(sw.ctrl[:, s].nan_to_num(nan=-7.0), ctrl0[:, s].nan_to_num(nan=-7.0))     # PID state untouched
        assert sw.read_status() & M._abi.STATUS_NAN_ACTION
        # the agent fell freely: no thrust
        assert float(sw.state[9, s]) < float(st['vel'][1, 2, 2]) - 0.09


def test_misaligned_action_views_are_handled():
    import mrsgym_b200 as mrsgym
    import mrsgym_b200 as M
    env = mrsgym.MRS(N_AGENTS=2, N_ENVS=2, ACTION_TYPE='set_speeds', START_POS=torch.tensor(H.grid_positions(1, 2)[0]),
                     START_ORI=torch.zeros(2, 3))
    buf = torch.full((1 + 16,), 14475.8, device='cuda')
    view = buf[1:].view(2, 2, 4)                      # 4 bytes into its storage: the kernels read float4 actions
    assert view.data_ptr() % 16 != 0
    env.step(view)                                    # MRS.step re-aligns
    with pytest.raises(ValueError, match='16-byte'):
        env.swarm.step(view)                          # the raw Swarm refuses instead of faulting


def test_single_env_windows_stay_valid_without_a_copy_per_step():
    """N_ENVS = 1 hands out fresh tensors like the reference (MRS.py:87-110 builds X and A anew every step): a held
    observation never changes afterwards, across tape renewals and resets, and equals what a copying env returns."""
    import mrsgym_b200 as mrsgym
    start = torch.tensor([[0., 0, 2], [1, 0, 2], [0, 1, 2.5], [1, 1, 3]])
    kw = dict(N_AGENTS=4, K_HOPS=2, COMM_RANGE=1.2, ACTION_TYPE='set_target_vel', START_POS=start, START_ORI=torch.zeros(4, 3),
              TAPE_SLOTS=8)
    env = mrsgym.make('mrs-v0', **kw)
    ref = mrsgym.make('mrs-v0', BATCHED=False, COPY_OBS=False, **kw)
    assert env.swarm.fresh and not env._clone and not ref.swarm.fresh
    g = torch.Generator().manual_seed(5)
    held, want = [], []
    gen0 = env.swarm.generation
    for t in range(40):
        if t == 25:
            held.append((env.reset(), None)); want.append((ref.reset().clone(), None))
        a = torch.randn(4, 3, generator=g) * 0.5
        X, _, _, info = env.step(a)
        Xr, _, _, infor = ref.step(a)
        held.append((X, info['A'])); want.append((Xr.clone(), infor['A'].clone()))
    assert env.swarm.generation > gen0 + 4          # the 8-slot tapes were renewed several times
    for (X, A), (Xr, Ar) in zip(held, want):
        assert torch.equal(X, Xr)
        assert A is None or torch.equal(A, Ar)


def test_bench_dump_outputs_are_the_last_timed_step(tmp_path):
    """bench.py --dump-outputs: two runs with the same arguments write the same arrays, and they are X, A and the state
    after the warm-up replay and exactly --steps timed steps from the bench's start state."""
    import json
    import subprocess
    import sys
    import bench
    import mrsgym_b200 as M
    from conftest import _REPO
    E, T = 256, 7
    dumps = []
    for i in range(2):
        d = tmp_path / str(i)
        r = subprocess.run([sys.executable, os.path.join(_REPO, 'bench.py'), '--envs', str(E), '--steps', str(T),
                            '--warmup', '1', '--no-cpu', '--clock-seconds', '0', '--e2e-steps', '0', '--dump-outputs', str(d)],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])['steps'] == T
        dumps.append({k: np.load(d / (k + '.npy')) for k in ('X', 'A', 'state')})
    a, b = dumps
    for k in a:
        assert a[k].dtype == np.float32 and np.array_equal(a[k], b[k]), k
    # the same inputs through plain single-step launches: one warm-up replay of T steps, then the T timed steps
    w = bench.WORKLOADS['c5']
    st, act = bench.make_inputs(w, E, T, seed=1234 + 4)
    sw = M.Swarm(E, w['N'], w['K'], w['mode'], M._abi.X_POS_VEL, w['R'])
    H.upload_state(sw, st)
    actions = torch.from_numpy(act).cuda()
    for t in range(2 * T):
        sw.step(actions[t % T])
    np.testing.assert_array_equal(a['state'], sw.state.t().reshape(E, w['N'], 13).cpu().numpy())
    np.testing.assert_array_equal(a['X'], sw.X_window()[0].cpu().numpy())
    np.testing.assert_array_equal(a['A'], sw.A_window()[0].cpu().numpy())
