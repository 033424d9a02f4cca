"""The external wrench (MrsBuffers.wrench, Swarm.set_external_wrench) on every kernel the step can pick with one bound,
against the CPU oracle (wrench_cases.step_with_wrench): N <= 32 run-time-width kernels at every width and at a
size that would otherwise take SM-sized CTAs, the multi-step and chained forms, and the N > 32 lanes-per-agent, fused,
three-kernel and tiled paths.  Free-flight scenes are held to the one-step delta bar, contact scenes to the contact
band of test_gpu_physics_variants.py; A is bit-exact on the GPU's own X.  The scenes (wrench_cases.py) are >= 10 bars
away from each wrong kernel they name (test_cpu_wrench.py)."""
import numpy as np
import pytest
import torch

import helpers as H
import physics_variants as V
import wrench_cases as W
from oracle import spec

pytestmark = pytest.mark.gpu

R_COMM = 1.5


def _big_cta_envs():
    from test_gpu_physics_variants import _big_cta_envs as f
    return f()


def _swarm(E, N, mode, **kw):
    import mrsgym_b200 as M
    return M.Swarm(E, N, 0, mode, M._abi.X_POS_VEL, R_COMM, **kw)


def _dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def _run(kind, E, N, mode=None, how='step', T=1, picks=None, seed=0, fused=None, monkeypatch=None):
    """Step a scene with its wrench on the GPU and compare with the oracle; returns the swarm"""
    if fused is not None:
        monkeypatch.setenv('MRS_B200_FUSED_MID', fused)
    contact = W.KINDS[kind][0]
    st, F, Tq = W.make_case(kind, E, N, seed=seed + N)
    acts = W.mode_actions(mode, E, N, st, seed=seed + 1, T=T)
    sw = _swarm(E, N, mode)
    H.upload_state(sw, st)
    sw.set_external_wrench(_dev(F), _dev(Tq))
    a_dev = None if acts is None else _dev(acts)
    if how == 'step':
        for t in range(T):
            sw.step(None if a_dev is None else a_dev[t].contiguous())
    elif how == 'many':
        sw.step_many(a_dev, T)
    else:
        sw.rollout(a_dev, T)
    picks = list(range(E)) if picks is None else picks
    sub = lambda d: {k: v[picks] for k, v in d.items()}
    g = sub(H.read_state(sw))
    s0 = sub(st)
    ref = W.oracle_step(s0, mode, None if acts is None else acts[:, picks], F[picks], Tq[picks], T=T)
    if T == 1:
        r = W.bar_ratio(s0, ref, g, contact)
        assert r <= 1.0, (kind, mode, how, E, N, r)
    else:
        for k, tol in V.TRAJ_BAR:
            assert float(np.max(np.abs(g[k] - ref[k]))) <= tol, (kind, k)
    X = sw.X_window()[0]
    np.testing.assert_array_equal(sw.A_window()[0][picks].cpu().numpy(), spec.adjacency(X[picks][..., :3].cpu().numpy(), R_COMM))
    assert sw.read_status() == 0
    return sw


SMALL = [(12, 5), (67, 8), (10, 16), (4, 32)]
KINDS = list(W.KINDS)


# ------------------------------------------------------------------------------ N <= 32
@pytest.mark.parametrize('kind', KINDS)
@pytest.mark.parametrize('E,N', SMALL)
def test_group_kernels(kind, E, N):
    """the run-time-width wrench kernel at every width; 67 x 8 has a ragged last chunk"""
    _run(kind, E, N)


@pytest.mark.parametrize('kind', ['tilted', 'pressed', 'collide'])
def test_group_kernel_at_sm_sized_cta_scale(kind):
    """N = 8 with enough warp-chunks that the step without a wrench takes SM-sized CTAs"""
    E = _big_cta_envs()
    _run(kind, E, 8, picks=[0, 1, 2, 3, E // 2 + 1, E - 1])


@pytest.mark.parametrize('mode', H.MODES + [None])
@pytest.mark.parametrize('E,N', [(12, 5), (6, 48)])
def test_every_action_mode(mode, E, N):
    """every action mode (and NO_ACTION) with the wrench, on an N <= 32 and an N > 32 shape"""
    _run('tilted', E, N, mode=mode)


@pytest.mark.parametrize('kind', ['tilted', 'collide', 'slide_above'])
@pytest.mark.parametrize('E,N', [(67, 8), (9, 16)])
def test_multi_step_forms(kind, E, N):
    """mrs_step_many within 2e-5 of plain steps (float32 rounding of the MANY kernels), mrs_rollout bit for bit"""
    T = 3
    plain = _run(kind, E, N, how='step', T=T)
    many = _run(kind, E, N, how='many', T=T)
    roll = _run(kind, E, N, how='rollout', T=T)
    assert torch.equal(plain.state, roll.state)
    assert float((plain.state.double() - many.state.double()).abs().max()) < 2e-5


# ------------------------------------------------------------------------------ N > 32
@pytest.mark.parametrize('kind', KINDS)
def test_lanes_per_agent_kernels(kind):
    _run(kind, 6, 48)


@pytest.mark.parametrize('fused', ['1', '0'])
@pytest.mark.parametrize('kind', KINDS)
def test_one_cta_per_env_kernels(kind, fused, monkeypatch):
    """>= 32768 agents: step_env_kernel, and the three-kernel path (MRS_B200_FUSED_MID=0)"""
    _run(kind, 520, 64, picks=[0, 1, 259, 519], fused=fused, monkeypatch=monkeypatch)


@pytest.mark.parametrize('kind', KINDS)
@pytest.mark.parametrize('E,N', [(2, 200), (1, 1030)])
def test_tiled_kernels(kind, E, N):
    if kind == 'collide' and N > 1024:
        pytest.skip('1030 agents in contact: more than the per-env solver holds (MRS_STATUS_CONTACT_OVERFLOW)')
    _run(kind, E, N)


# ------------------------------------------------------------------------------ zero wrench, clear, persistence
def _zero_vs_none(E, N, mode, baked=True):
    st, _, _ = W.make_case('tilted', E, N, seed=21)
    acts = W.mode_actions(mode, E, N, st, seed=22)
    out = []
    for zero in (False, True):
        sw = _swarm(E, N, mode)
        if not baked:       # AGENT_RADIUS only sizes the spawn: a config that is not the baked one, same physics
            sw.cfg.phys.agent_radius = 0.31
            assert sw.lib.mrs_config_is_baked(sw._cfg_ref) == 0
        H.upload_state(sw, st)
        if zero:
            sw.set_external_wrench(torch.zeros(3, device='cuda'), torch.zeros(3, device='cuda'))
        sw.step(None if acts is None else _dev(acts[0]))
        out.append(sw)
    return out


# A zero wrench adds exact zeros, but the kernels with and without EXT are different binaries: ptxas contracts some
# multiply-adds of the rotor wrench differently in the two (as in the fused and three-kernel N > 32 paths for
# set_control), so the two runs agree to float32 rounding, not to the bit.
@pytest.mark.parametrize('E,N', [(6, 48), (520, 64), (2, 200)])
def test_zero_wrench_equals_none_wide(E, N):
    a, b = _zero_vs_none(E, N, 'set_speeds')
    assert float((a.state.double() - b.state.double()).abs().max()) < 2e-5


def test_zero_wrench_equals_none_generic_group():
    """N = 5 under a non-baked configuration: both runs take generic run-time-width kernels"""
    a, b = _zero_vs_none(12, 5, 'set_speeds', baked=False)
    assert float((a.state.double() - b.state.double()).abs().max()) < 2e-5


def test_zero_wrench_near_baked_at_n8():
    """N = 8 default config: the baked unrolled kernel against the generic wrench kernel, within the tolerance of
    test_baked_kernels_agree_with_generic_kernels"""
    a, b = _zero_vs_none(64, 8, 'set_target_vel')
    assert float((a.state.double() - b.state.double()).abs().max()) < 2e-5


@pytest.mark.parametrize('E,N', [(12, 8), (6, 48)])
def test_clear_restores_the_plain_step(E, N):
    """after clear_external_wrench() the results are bit-identical to a swarm that never had one"""
    st, F, Tq = W.make_case('tilted', E, N, seed=31)
    acts = _dev(W.mode_actions('set_speeds', E, N, st, seed=32, T=2))
    a, b = _swarm(E, N, 'set_speeds'), _swarm(E, N, 'set_speeds')
    for s in (a, b):
        H.upload_state(s, st)
    b.set_external_wrench(_dev(F), _dev(Tq))
    ptr = b.wrench.data_ptr()
    b.clear_external_wrench()
    for t in range(2):
        a.step(acts[t].contiguous())
        b.step(acts[t].contiguous())
    assert torch.equal(a.state, b.state) and torch.equal(a.A_tape, b.A_tape)
    b.set_external_wrench(torque=_dev(Tq))
    assert b.wrench.data_ptr() == ptr and b.wrench_bound


def test_set_external_wrench_shapes_and_mask():
    E, N = 3, 4
    sw = _swarm(E, N, None)
    sw.set_external_wrench(torch.tensor([1.0, 2.0, 3.0], device='cuda'))
    w = sw.wrench.view(6, E, N)
    assert torch.equal(w[0], torch.ones(E, N, device='cuda')) and torch.equal(w[3:], torch.zeros(3, E, N, device='cuda'))
    per_env = torch.arange(E * 3, dtype=torch.float32, device='cuda').reshape(E, 1, 3)
    sw.set_external_wrench(torque=per_env, env_mask=torch.tensor([True, False, True], device='cuda'))
    assert torch.equal(w[3:, 0], per_env[0, 0][:, None].expand(3, N))
    assert torch.equal(w[3:, 1], torch.zeros(3, N, device='cuda'))
    assert torch.equal(w[0], torch.ones(E, N, device='cuda'))       # force kept


def test_wrench_survives_reset_and_env_api():
    """MRS.set_external_wrench ([N, 3] unbatched) persists through reset(); NO_ACTION with F = m g z hovers"""
    import mrsgym_b200 as M
    env = M.MRS(N_AGENTS=4, N_ENVS=1, ACTION_TYPE='set_speeds', COMM_RANGE=R_COMM)
    env.set_external_wrench(torch.tensor([[0.0, 0.0, W.WEIGHT]] * 4, device='cuda'))
    env.reset()
    assert env.swarm.wrench_bound
    env.swarm.set_action_type(None)
    z0 = env.swarm.get_pos()[..., 2].clone()
    env.swarm.step(None)
    assert float((env.swarm.get_vel()).abs().max()) < 1e-5
    assert torch.allclose(env.swarm.get_pos()[..., 2], z0, atol=1e-6)
    env.clear_external_wrench()
    assert not env.swarm.wrench_bound


# ------------------------------------------------------------------------------ NaN actions and non-finite wrenches
@pytest.mark.parametrize('E,N', [(12, 8), (12, 5), (6, 48), (520, 64), (2, 200)])
def test_nan_action_keeps_the_wrench(E, N):
    """a NaN-action agent gets no rotor wrench but the external one; status bit and counter as without a wrench"""
    st, F, Tq = W.make_case('tilted', E, N, seed=41)
    acts = W.mode_actions('set_speeds', E, N, st, seed=42)
    acts[0, 1, 3, 2] = np.nan
    sw = _swarm(E, N, 'set_speeds')
    H.upload_state(sw, st)
    sw.set_external_wrench(_dev(F), _dev(Tq))
    sw.step(_dev(acts[0]))
    picks = sorted({0, 1, min(2, E - 1), E - 1})
    sub = lambda d: {k: v[picks] for k, v in d.items()}
    ref = W.oracle_step(sub(st), 'set_speeds', acts[:, picks], F[picks], Tq[picks])
    assert W.bar_ratio(sub(st), ref, sub(H.read_state(sw)), False) <= 1.0
    assert sw.read_status() == 1 and sw.read_stats()['nan_actions'] == 1


@pytest.mark.parametrize('E,N', [(12, 8), (6, 48), (2, 200)])
def test_nonfinite_wrench_meets_the_clamp(E, N):
    """NaN / inf wrench components are not special-cased: like any non-finite acceleration they meet the
    +-max_coord_vel clamp (fminf / fmaxf return the bound for NaN), so those agents move at the clamp velocity, stay
    finite and raise no status; the other envs step exactly as with a finite wrench"""
    st, F, Tq = W.make_case('tilted', E, N, seed=51)
    bad_F, bad_T = F.copy(), Tq.copy()
    e_bad = 5 % E
    bad_F[e_bad, 1, 0] = np.nan
    bad_T[e_bad, 2, 2] = np.inf
    out = []
    for f, t in ((F, Tq), (bad_F, bad_T)):
        sw = _swarm(E, N, None)
        H.upload_state(sw, st)
        sw.set_external_wrench(_dev(f), _dev(t))
        sw.step(None)
        out.append(sw)
    a, b = out
    assert a.read_status() == 0 and b.read_status() == 0 and b.read_stats()['nonfinite'] == 0
    sa, sb = a.state.view(13, E, N), b.state.view(13, E, N)
    others = [e for e in range(E) if e != e_bad]
    assert torch.equal(sa[:, others], sb[:, others])
    assert bool(torch.isfinite(sb).all())
    assert float(sb[7, e_bad, 1].abs()) == 100.0 and float(sb[12, e_bad, 2].abs()) == 100.0


# ------------------------------------------------------------------------------ graphs
def test_graph_rollout_refuses_a_bind_change():
    E, N, T = 12, 8, 4
    sw = _swarm(E, N, None, tape_slots=T)
    st, F, Tq = W.make_case('tilted', E, N, seed=61)
    H.upload_state(sw, st)
    g = sw.capture_rollout(None, T)
    g.replay()
    sw.set_external_wrench(_dev(F), _dev(Tq))
    with pytest.raises(RuntimeError):
        g.replay()
    g2 = sw.capture_rollout(None, T)
    g2.replay()
    sw.clear_external_wrench()
    with pytest.raises(RuntimeError):
        g2.replay()


@pytest.mark.parametrize('N', [8, 48])
def test_closed_loop_graph_with_a_time_varying_wrench(N):
    """rollout(graph=True) whose policy rewrites the wrench every step: the replay equals the eager body bit for bit;
    the wrench survives the on-device auto-reset; binding or unbinding captures again"""
    import mrsgym_b200 as M
    E, T = 16, 8

    def make():
        env = M.MRS(N_AGENTS=N, N_ENVS=E, ACTION_TYPE='set_speeds', COMM_RANGE=R_COMM, TAPE_SLOTS=T, SEED=5,
                    START_POS=M.DefaultSpawn(N, 1.0, 5.0, 3.0))
        env.set_external_wrench(torch.zeros(3, device='cuda'))
        return env
    gust = torch.tensor([0.05, -0.02, 0.1], device='cuda')

    def policy(X, A, env=None):      # a wind that follows the swarm's mean height: a new wrench every step
        h = X[:, 0, :, 2].mean(dim=1).reshape(E, 1, 1)
        env.set_external_wrench(gust * torch.sin(7.0 * h))
        return torch.full((E, N, 4), H.HOVER, device='cuda')
    outs = []
    for capture in (True, False):
        env = make()
        pol = lambda X, A, **kw: policy(X, A, env=env)
        g = M.ClosedLoopGraph(env, pol, T, episode_length=3, capture=capture)
        d = g.run()
        outs.append((env.swarm.state.clone(), env.swarm.wrench.clone(), d))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    assert bool(outs[0][1].abs().sum() > 0)
    env = make()
    pol = lambda X, A, **kw: policy(X, A, env=env)
    M.rollout(env, pol, T, episode_length=3, graph=True)
    n = len(env._graphs)
    env.clear_external_wrench()
    with pytest.raises(RuntimeError):
        M.rollout(env, pol, T, episode_length=3, graph=True)     # the policy binds it again inside the loop
    env.set_external_wrench(torch.zeros(3, device='cuda'))
    env.swarm.clear_external_wrench()
    M.rollout(env, lambda X, A, **kw: torch.full((E, N, 4), H.HOVER, device='cuda'), T, episode_length=3, graph=True)
    assert len(env._graphs) == n + 1
