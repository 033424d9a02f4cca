"""mrs_autoreset and rollout(graph=True) on the GPU: the kernel against the numpy restatement (autoreset_spec.py), the
captured closed loop against the same body run eagerly and against rollout(), replays, determinism, sharding, the
spawn failure contract, capturable callbacks and the refusals."""
import math

import numpy as np
import pytest
import torch

import autoreset_spec as AR

pytestmark = pytest.mark.gpu

R_AGENT = 0.3
SEED, OFFSET, K, L = 1, 100, 2, 5
# N -> (E, (z_lo, z_hi, xy_radius)); with SEED / OFFSET / the episodes below every pair test of the restatement clears
# the rounding bound (asserted in the test)
CASES = {3: (50, (1.0, 3.0, 1.0)), 8: (41, (1.0, 3.0, 1.0)), 16: (30, (1.0, 5.0, 3.0)), 32: (22, (1.0, 5.0, 3.0)),
         33: (9, (1.0, 5.0, 3.0)), 64: (10, (1.0, 5.0, 3.0)), 200: (5, (1.0, 5.0, 4.0))}


def _rounding_bound(region):
    """As test_gpu_spawn_wide: the largest |d^2 - 4 r^2| a float32 restatement and the GPU can disagree on."""
    cmax = max(abs(region[1]), region[2])
    eps = 8 * 2.0 ** -24 * cmax
    return 2 * (2 * R_AGENT) * 2 * np.sqrt(3) * eps + 8 * 2.0 ** -24 * 4 * R_AGENT ** 2


def _swarm(E, N, layout=None, comm_range=2.0):
    import mrsgym_b200 as M
    sw = M.Swarm(E, N, K, 'set_target_vel', M._abi.X_POS_VEL if layout is None else layout, comm_range,
                 tape_slots=L, ring=True)
    g = torch.Generator(device=sw.device).manual_seed(N)
    for t in (sw.state, sw.ctrl, sw.X_tape, sw.A_tape):
        t.copy_(torch.rand(t.shape, generator=g, device=sw.device) * 4 - 2)
    return sw


def _counters(E, dev):
    e = torch.arange(E, device=dev)
    steps = (e % 9).to(torch.int32)                    # episode_length 8: n = 7, 8 end their episode
    episode = ((e * 7) % 5).to(torch.int32)
    done_in = (e % 3 == 0)
    return steps, episode, done_in


@pytest.mark.parametrize('N', sorted(CASES))
@pytest.mark.parametrize('slot', [0, 3])                 # slot 3: the window (3, 4, 0) wraps the ring of 5
def test_kernel_matches_the_restatement(N, slot):
    E, region = CASES[N]
    z_lo, z_hi, R = region
    sw = _swarm(E, N)
    dev = sw.device
    steps, episode, done_in = _counters(E, dev)
    st0, ct0, X0, A0, ep0, n0 = (sw.state.clone(), sw.ctrl.clone(), sw.X_tape.clone(), sw.A_tape.clone(),
                                 episode.clone(), steps.clone())
    done_out = torch.full((E,), 7, dtype=torch.uint8, device=dev)
    failed = torch.zeros(1, dtype=torch.int32, device=dev)
    rounds = 10000 if N > 32 else 256
    sw.autoreset(SEED, steps, episode, done_out, done_in=done_in, slot_x=slot, slot_a=slot, z=(z_lo, z_hi), xy_radius=R,
                 xy_sigma=R, max_rounds=rounds, env_offset=OFFSET, episode_length=8, failed=failed)
    torch.cuda.synchronize()
    want = np.array([AR.done_rule(int(n), bool(d), 8) for n, d in zip(n0.tolist(), done_in.tolist())])
    assert want.any() and not want.all()
    m = torch.from_numpy(want).to(dev)
    assert torch.equal(done_out.bool(), m)
    assert int(failed.item()) == 0
    # counters
    assert torch.equal(episode, torch.where(m, ep0 + 1, ep0))
    assert torch.equal(steps, torch.where(m, torch.zeros_like(n0), n0 + 1))
    # untouched envs: every byte of state, PID planes and every tape slot
    stE, st0E = sw.state.reshape(13, E, N), st0.reshape(13, E, N)
    assert torch.equal(stE[:, ~m], st0E[:, ~m])
    assert torch.equal(sw.ctrl, ct0), 'the PID planes are left alone (also for reset envs)'
    assert torch.equal(sw.X_tape[:, ~m], X0[:, ~m]) and torch.equal(sw.A_tape[:, ~m], A0[:, ~m])
    # reset envs: the restatement's draw of episode + 1
    pos, q = sw.get_pos().cpu().numpy(), sw.get_quat().cpu().numpy().astype(np.float64)
    margin = np.inf
    for e in np.flatnonzero(want):
        p, yaw, f, mg, _ = AR.reset_env(SEED, OFFSET + e, int(ep0[e]) + 1, N, R_AGENT, z=(z_lo, z_hi), xy_radius=R,
                                        xy_sigma=R, max_rounds=rounds)
        assert not f
        margin = min(margin, mg)
        np.testing.assert_allclose(pos[e], p, rtol=0, atol=1e-5)
        np.testing.assert_allclose(2 * np.arctan2(q[e, :, 2], q[e, :, 3]), yaw, rtol=0, atol=1e-6)
    assert margin > _rounding_bound(region), (margin, _rounding_bound(region))
    assert float(np.abs(q[want][..., :2]).max()) == 0.0
    assert float(sw.get_vel()[m].abs().max()) == 0.0 and float(sw.get_angvel()[m].abs().max()) == 0.0
    # windows: K+1 copies of X0; A0 = mrs_adjacency of the new positions in the newest slot, zeros in the K older ones
    x0 = torch.cat([sw.get_pos(), sw.get_vel()], dim=-1)[m]
    win = [(slot + k) % L for k in range(K + 1)]
    for k, sl in enumerate(win):
        assert torch.equal(sw.X_tape[sl][m], x0), ('X slot', sl)
        if k == 0:
            assert torch.equal(sw.A_tape[sl][m], sw.adjacency(sw.get_pos())[m])
        else:
            assert float(sw.A_tape[sl][m].abs().max()) == 0.0, ('A slot', sl)
    for sl in set(range(L)) - set(win):
        assert torch.equal(sw.X_tape[sl], X0[sl]) and torch.equal(sw.A_tape[sl], A0[sl])


@pytest.mark.parametrize('N', [8, 64])
def test_kernel_full_layout_max_timesteps_and_infinite_range(N):
    import mrsgym_b200 as M
    E, region = CASES[N][0], CASES[N][1]
    sw = _swarm(E, N, layout=M._abi.X_FULL, comm_range=float('inf'))
    steps, episode, _ = _counters(E, sw.device)
    n0 = steps.clone()
    done = torch.empty(E, dtype=torch.bool, device=sw.device)
    sw.autoreset(SEED, steps, episode, done, slot_x=1, slot_a=2, z=region[:2], xy_radius=region[2],
                 xy_sigma=region[2], max_rounds=10000, max_timesteps=6)
    m = n0 >= 6                                          # MAX_TIMESTEPS sees the count before the increment
    assert torch.equal(done, m)
    full = torch.cat([sw.get_pos(), sw.get_quat(), sw.get_vel(), sw.get_angvel()], dim=-1)[m]
    for k in range(K + 1):
        assert torch.equal(sw.X_tape[(1 + k) % L][m], full)
    eye = torch.eye(N, device=sw.device)
    assert torch.equal(sw.A_tape[2][m], (1 - eye).expand(int(m.sum()), N, N))


def test_kernel_refuses_bad_arguments():
    import ctypes as C
    import mrsgym_b200 as M
    sw = _swarm(4, 8)
    a = M._abi.MrsAutoResetArgs(1, 0, 1.0, 3.0, 1.0, 1.0, 0.0, 0.0, 16, 0, -1)
    z32 = torch.zeros(4, dtype=torch.int32, device=sw.device)
    d = torch.zeros(4, dtype=torch.uint8, device=sw.device)
    p = lambda t: C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)  # noqa: E731
    call = lambda st, ep, do, sx, sa: sw.lib.mrs_autoreset(sw._cfg_ref, sw._bufs_ref, C.byref(a), None, p(st), p(ep),  # noqa: E731
                                                          p(do), sx, sa, None, sw._stream())
    assert call(z32, z32.clone(), d, 0, 0) == 0
    for args in ((None, z32, d, 0, 0), (z32, None, d, 0, 0), (z32, z32, None, 0, 0), (z32, z32, d, L, 0),
                 (z32, z32, d, 0, -1)):
        assert call(*args) == -1, args
    sw.cfg.state_layout = M._abi.X_NONE
    assert call(z32, z32, d, 0, 0) == -1
    sw.cfg.state_layout = M._abi.X_POS_VEL
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------- rollout(graph=True)
def _env(E, N, T_slots=8, **kw):
    import mrsgym_b200 as M
    R = 4.0 if N > 64 else (3.0 if N > 8 else 1.0)
    base = dict(N_AGENTS=N, N_ENVS=E, K_HOPS=2, COMM_RANGE=2.0, ACTION_TYPE='set_target_vel', SEED=5,
                START_POS=M.DefaultSpawn(N, 1.0, 5.0, R), TAPE_SLOTS=T_slots)
    base.update(kw)
    return M.MRS(**base)


def _state(env):
    return (env.swarm.state.clone(), env.swarm.ctrl.clone(), env.episode.clone(), env.env_steps.clone())


GRAPH_SHAPES = [(256, 8), (100, 16), (64, 64), (4, 200)]


@pytest.mark.parametrize('E,N', GRAPH_SHAPES)
def test_graph_equals_the_eager_body(E, N):
    import mrsgym_b200 as M
    pol = M.reynolds_policy()
    T = 16                                                # 2 L, resets at steps 4, 9, 14
    a, b = _env(E, N), _env(E, N)
    da = M.rollout(a, pol, T, episode_length=5, graph=True)
    db = M.ClosedLoopGraph(b, pol, T, episode_length=5, capture=False).run()
    assert set(da) == {'X', 'A', 'action', 'reward', 'done'} == set(db)
    for k in da:
        assert torch.equal(da[k], db[k]), k
    for x, y in zip(_state(a), _state(b)):
        assert torch.equal(x, y)
    assert torch.equal(a.get_Xk(), b.get_Xk()) and torch.equal(a.get_Ak(), b.get_Ak())
    assert da['done'].any(dim=1).cpu().tolist() == [t in (4, 9, 14) for t in range(T)]
    assert torch.equal(a.episode.cpu(), torch.full((E,), 3, dtype=torch.int32))


def test_graph_matches_rollout_without_resets():
    import mrsgym_b200 as M
    pol = M.reynolds_policy()
    a, b = _env(128, 8), _env(128, 8)
    da = M.rollout(a, pol, 16, episode_length=40, graph=True)
    db = M.rollout(b, pol, 16, episode_length=40)
    for k in ('X', 'A', 'action', 'reward', 'done'):
        assert torch.equal(da[k], db[k]), k
    assert not da['done'].any()
    assert torch.equal(a.swarm.state, b.swarm.state) and torch.equal(a.env_steps, b.env_steps)


@pytest.mark.parametrize('E,N', [(96, 8), (16, 64)])
def test_graph_resets_on_the_steps_rollout_does(E, N):
    import mrsgym_b200 as M
    pol = M.reynolds_policy()
    a, b = _env(E, N), _env(E, N)
    # envs enter the loop at different points of their episodes
    for env in (a, b):
        env.step(pol(env.get_Xk(), env.get_Ak()))
        half = torch.arange(E) % 2 == 0
        env.reset(env_mask=half)
        env.refresh_A(half)
    da = M.rollout(a, pol, 16, episode_length=4, graph=True)
    db = M.rollout(b, pol, 16, episode_length=4)
    assert torch.equal(da['done'], db['done'])
    assert torch.equal(a.env_steps, b.env_steps)
    for data, env in ((da, a), (db, b)):
        done = data['done']
        for t in range(15):
            m = done[t]
            if not m.any():
                continue
            x = data['X'][t + 1][m]                      # the first observation of the new episode: X0
            assert float(x[..., 3:6].abs().max()) == 0.0
            assert torch.equal(data['A'][t + 1][m], env.swarm.adjacency(data['X'][t + 1][..., :3])[m])
            p = x[..., :3]
            d = (p.unsqueeze(2) - p.unsqueeze(1)).norm(dim=-1) + 10 * torch.eye(N, device=p.device)
            assert float(d.min()) >= 2 * R_AGENT - 1e-6
    # the last step ends an episode for the envs that entered on a fresh start: their final windows are the reset's
    m = da['done'][15]
    assert m.any()
    for env in (a, b):
        X, A = env.get_Xk(), env.get_Ak()
        assert torch.equal(X[m][:, 1], X[m][:, 0]) and torch.equal(X[m][:, 2], X[m][:, 0])
        assert float(A[m][:, 1:].abs().max()) == 0.0
        assert torch.equal(A[m][:, 0], env.swarm.adjacency(env.swarm.get_pos())[m])


def test_replays_start_new_episodes_and_are_deterministic():
    import mrsgym_b200 as M
    pol = M.reynolds_policy()
    a, b = _env(64, 16), _env(64, 16)
    first = {k: v.clone() for k, v in M.rollout(a, pol, 8, episode_length=3, graph=True).items()}
    ep1 = a.episode.clone()
    second = M.rollout(a, pol, 8, episode_length=3, graph=True)
    assert len(a._graphs) == 1, 'the second call replays the cached graph'
    # episode_length 3 counts across calls: resets at steps 2 and 5 of the first call, 0, 3 and 6 of the second
    assert torch.equal(ep1, torch.full_like(ep1, 2)) and torch.equal(a.episode, ep1 + 3)
    assert not torch.equal(first['X'][3], second['X'][1])
    # a second env with the same SEED replays the same two calls
    b1 = {k: v.clone() for k, v in M.rollout(b, pol, 8, episode_length=3, graph=True).items()}
    b2 = M.rollout(b, pol, 8, episode_length=3, graph=True)
    for k in first:
        assert torch.equal(first[k], b1[k]) and torch.equal(second[k], b2[k]), k
    assert torch.equal(a.swarm.state, b.swarm.state)
    # out= receives a copy
    out = {}
    M.rollout(a, pol, 8, episode_length=3, graph=True, out=out)
    assert out['X'].data_ptr() != a._graphs[next(iter(a._graphs))].data['X'].data_ptr()


def test_shards_equal_slices_of_the_whole():
    import mrsgym_b200 as M

    def pol(X, A):                                       # per agent: no reduction whose order could depend on E
        return (0.5 * X[:, 0, :, 3:6] - 0.25 * X[:, 0, :, :3]).contiguous()
    full = _env(64, 8)
    lo, hi = _env(32, 8, ENV_OFFSET=0), _env(32, 8, ENV_OFFSET=32)
    df = M.rollout(full, pol, 16, episode_length=3, graph=True)
    dl = M.rollout(lo, pol, 16, episode_length=3, graph=True)
    dh = M.rollout(hi, pol, 16, episode_length=3, graph=True)
    for k in ('X', 'A', 'action', 'done'):
        assert torch.equal(df[k][:, :32], dl[k]) and torch.equal(df[k][:, 32:], dh[k]), k
    assert not torch.equal(dl['X'][4], dh['X'][4])


def test_infeasible_density_raises_after_replay():
    import mrsgym_b200 as M
    env = _env(4, 64)
    env.START_POS = M.DefaultSpawn(64)                  # r = 1 m, z in [1, 3]: 64 agents do not fit
    with pytest.raises(RuntimeError, match='did not converge'):
        M.rollout(env, M.reynolds_policy(), 8, episode_length=2, graph=True)


def test_small_envs_count_failures_lazily():
    import mrsgym_b200 as M
    env = _env(8, 32, START_POS=M.DefaultSpawn(32, 1.0, 5.0, 3.0))
    env.START_POS = M.DefaultSpawn(32, 1.0, 1.0, 0.4)   # a flat disc of 0.4 m: 32 agents never fit
    M.rollout(env, M.reynolds_policy(), 8, episode_length=4, graph=True)
    assert int(env.spawn_failed.item()) == 2 * 8


def test_tensor_done_fn_triggers_resets():
    import mrsgym_b200 as M
    pol = M.reynolds_policy()
    holder = {}

    def done_fn(X, **kw):
        return holder['env'].env_steps >= 3                  # a device tensor; the device counter inside the graph
    a, b = _env(32, 8, done_fn=done_fn), _env(32, 8, done_fn=done_fn)
    holder['env'] = a
    da = M.rollout(a, pol, 16, graph=True)
    holder['env'] = b
    db = M.rollout(b, pol, 16)
    assert torch.equal(da['done'], db['done'])
    assert da['done'].any(dim=1).cpu().tolist() == [t in (3, 7, 11, 15) for t in range(16)]
    assert torch.equal(a.episode.cpu(), torch.full((32,), 4, dtype=torch.int32))
    # constant verdicts and rewards are filled in
    c = _env(16, 8, done_fn=lambda **kw: True, reward_fn=lambda X, **kw: X[:, 0, :, 2].mean(-1))
    dc = M.rollout(c, pol, 8, graph=True)
    assert bool(dc['done'].all()) and torch.equal(c.episode.cpu(), torch.full((16,), 8, dtype=torch.int32))
    assert float(dc['reward'].min()) >= 0.5


@pytest.mark.parametrize('kw,match', [
    (dict(A_FORMAT='neighbors'), "A_FORMAT='dense'"),
    (dict(state_fn=lambda q: torch.cat([q.get_pos(), q.get_vel()])), 'fused state_fn'),
    (dict(N_ENVS=1), 'COPY_OBS=False'),
    (dict(TAPE_SLOTS=12), 'multiple of the tape size'),
    (dict(START_ORI=torch.tensor([0.1, 0, 0, 0.1, 0, 0])), 'default START_POS'),
    (dict(update_fn=lambda **kw: None), 'update_fn'),
    (dict(info_fn=lambda **kw: {}), 'info_fn'),
])
def test_refusals(kw, match):
    import mrsgym_b200 as M
    env = _env(4, 8, **kw)
    with pytest.raises(ValueError, match=match):
        M.rollout(env, M.reynolds_policy(), 8, graph=True)


def test_tensor_start_pos_is_refused():
    import mrsgym_b200 as M
    env = _env(4, 8)
    env.START_POS = torch.zeros(8, 3) + torch.arange(8).unsqueeze(1)
    with pytest.raises(ValueError, match='default START_POS'):
        M.rollout(env, M.reynolds_policy(), 8, graph=True)


def test_unbatched_env_without_copies():
    import mrsgym_b200 as M
    pol = M.reynolds_policy()
    a, b = _env(1, 8, COPY_OBS=False), _env(1, 8, COPY_OBS=False)
    da = M.rollout(a, pol, 16, episode_length=6, graph=True)
    db = M.ClosedLoopGraph(b, pol, 16, episode_length=6, capture=False).run()
    for k in da:
        assert torch.equal(da[k], db[k]), k
    assert da['X'].shape == (16, 1, 8, 6) and int(a.episode.item()) == 2
    assert math.isclose(float(a.env_steps.item()), 4)


def test_capture_after_dropping_an_env_with_a_cached_graph():
    import gc
    import mrsgym_b200 as M
    pol = M.reynolds_policy()
    old = _env(16, 8)
    M.rollout(old, pol, 8, episode_length=3, graph=True)
    del old                                     # a dead reference cycle that still holds a captured graph
    threshold = gc.get_threshold()
    gc.set_threshold(1)                         # the cyclic collector would run at every allocation
    try:
        new = _env(16, 8)
        data = M.rollout(new, pol, 8, episode_length=3, graph=True)
    finally:
        gc.set_threshold(*threshold)
    assert data['done'].any(dim=1).cpu().tolist() == [t in (2, 5) for t in range(8)]
