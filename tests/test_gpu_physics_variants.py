"""The CUDA contact solve under non-default physics (tests/physics_variants.py) against the CPU oracle, on every
kernel the step can pick: N <= 32 run-time-width, unrolled full-chunk and SM-sized-CTA kernels, the multi-step and
chained forms, the 33-128 agent kernels (lanes per agent, fused one CTA per env, thread per agent) and the N > 128
tiled pair pass; plus N > 4096 agents in one env, the sensors at a contact radius below the agent radius, and the
status bits of non-finite states and of a per-env pair overflow.  Every comparison is preceded by a check that the
oracle under the variant is at least 10 bars away from the oracle under the default physics (and, for a sweep cap
k, from k + 1), so a kernel that ignored the field would fail."""
import os
import re

import numpy as np
import pytest
import torch

import helpers as H
import physics_variants as V
from oracle import bullet_model as bm
from oracle import spec

pytestmark = pytest.mark.gpu

R_COMM, K = 1.5, 1
ALL = list(V.VARIANTS)


def _swarm(E, N, fields, layout=None, **kw):
    import mrsgym_b200 as M
    sw = M.Swarm(E, N, K, None, M._abi.X_POS_VEL if layout is None else layout, R_COMM, **kw)
    V.apply(sw, fields)
    return sw


def _big_cta_envs():
    """E at N = 8 above the SM-sized-CTA threshold of launch_group (nwork > 2 * sms * kBig warp-chunks, kBig =
    4 * ModeTraits<MRS_NO_ACTION>::minb), read from the source and the device"""
    src = open(os.path.join(os.path.dirname(__file__), '..', 'mrs-gym_b200', 'csrc', 'mrs_device.cuh')).read()
    minb = int(re.search(r'struct ModeTraits<MRS_NO_ACTION>.*?minb = (\d+);', src).group(1))
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    return 4 * (2 * sms * 4 * minb + 256)          # 4 envs per warp-chunk at N = 8


def _check_variant(name, E, N, how='step', T=1, picks=None, layout=None, seed=0):
    import mrsgym_b200 as M
    fields, kind = V.VARIANTS[name]
    st = V.make_state(kind, E, N, seed=seed + N)
    picks = list(range(E)) if picks is None else picks
    sub = {k: v[picks] for k, v in st.items()}
    # discrimination first: the variant must move the oracle's first step by >= 10 bars
    disc, ref1 = V.discrimination(sub, fields)
    assert min(disc.values()) >= 10, (name, disc)
    sw = _swarm(E, N, fields, layout)
    H.upload_state(sw, st)
    if how == 'step':
        for _ in range(T):
            sw.step(None)
    elif how == 'many':
        sw.step_many(None, T)
    else:
        sw.rollout(None, T)
    g = H.read_state(sw)
    gs = {k: v[picks] for k, v in g.items()}
    ref = ref1 if T == 1 else V.oracle_steps(sub, fields, T)
    bar = V.CONTACT_BAND if T == 1 else V.TRAJ_BAR
    for k, tol in bar:
        err = float(np.max(np.abs(gs[k] - ref[k])))
        assert err <= tol, (name, how, E, N, k, err)
    X = sw.X_window()[0]
    np.testing.assert_array_equal(sw.A_window()[0][picks].cpu().numpy(), spec.adjacency(X[picks][..., :3].cpu().numpy(), R_COMM))
    if layout == M._abi.X_FULL:
        assert torch.equal(X, sw.state.t().reshape(E, N, 13))
    assert sw.read_status() == 0
    stats = sw.read_stats()
    if fields.get('ground_contact', 1) == 0:
        assert stats['ground_contacts'] == 0
    if fields.get('agent_contact', 1) == 0:
        assert stats['agent_contact_rows'] == 0
    if N <= 32:
        iters = fields.get('solver_iters', 50)
        assert stats['solver_sweeps'] <= iters * stats['contact_chunks'], stats
    return sw, st


# ------------------------------------------------------------------------------ N <= 32
@pytest.mark.parametrize('name', ALL)
@pytest.mark.parametrize('E,N', [(12, 5), (8, 12)])
def test_runtime_width_kernel(name, E, N):
    """GT = 0: group width chosen at run time (N not a power of two), 4 or 2 envs per warp-chunk"""
    _check_variant(name, E, N)


@pytest.mark.parametrize('name', ALL)
@pytest.mark.parametrize('E,N', [(67, 8), (10, 16), (4, 32)])
def test_unrolled_full_chunk_kernels(name, E, N):
    """GT = 8 / 16 / 32 on full chunks; at E = 67, N = 8 the ragged last chunk runs the run-time-width kernel"""
    import mrsgym_b200 as M
    _check_variant(name, E, N, layout=M._abi.X_FULL if N == 16 else None)


@pytest.mark.parametrize('name', ['iters3', 'loose_tol', 'erp2', 'hull_contact'])
def test_sm_sized_cta_kernel(name):
    """N = 8 with enough warp-chunks for one SM-sized CTA per SM and the parked-chunk hand-out; the oracle runs a
    converged / capped mix of envs from the first warp-chunk and envs far into the batch"""
    E = _big_cta_envs()
    _check_variant(name, E, 8, picks=[0, 1, 2, 3, E // 2 + 1, E - 1])


@pytest.mark.parametrize('name', ['iters1', 'mu_agent1', 'small_agents', 'dt_mars'])
@pytest.mark.parametrize('E,N', [(67, 8), (9, 16)])
def test_multi_step_forms(name, E, N):
    """mrs_step_many (MANY kernels, state in registers across steps) and the chained mrs_rollout: within the
    contact-grade trajectory bar of the oracle after 3 steps; mrs_rollout bit for bit equal to plain steps, the MANY
    kernels to float32 rounding"""
    T = 3
    plain, st = _check_variant(name, E, N, how='step', T=T)
    many, _ = _check_variant(name, E, N, how='many', T=T)
    roll, _ = _check_variant(name, E, N, how='rollout', T=T)
    assert torch.equal(plain.state, roll.state)
    assert float((plain.state.double() - many.state.double()).abs().max()) < 2e-5


# ------------------------------------------------------------------------------ 33 <= N <= 128
@pytest.mark.parametrize('name', ALL)
def test_lanes_per_agent_wide_kernels(name):
    """few agents: step_pre_kernel<8> + contact_env_kernel + step_post_kernel"""
    _check_variant(name, 6, 48)


@pytest.mark.parametrize('fused', ['1', '0'])
@pytest.mark.parametrize('name', ['hull_contact', 'iters3', 'mu_ground15', 'no_pairs', 'small_agents'])
def test_one_cta_per_env_kernels(name, fused, monkeypatch):
    """>= 32768 agents: the fused step_env_kernel, and the three-kernel path (MRS_B200_FUSED_MID=0)"""
    import mrsgym_b200 as M
    monkeypatch.setenv('MRS_B200_FUSED_MID', fused)
    _check_variant(name, 520, 64, picks=[0, 1, 259, 519], layout=M._abi.X_FULL if fused == '1' else None)


# ------------------------------------------------------------------------------ N > 128
@pytest.mark.parametrize('name', ALL)
def test_tiled_pair_kernels(name):
    """pair_tile_kernel + agent_pre_kernel"""
    _check_variant(name, 2, 200)


@pytest.mark.parametrize('name', ['hull_contact', 'erp2', 'margin'])
def test_tiled_pair_kernels_1030(name):
    """states with fewer than the 1024 agents in contact the per-env solver holds"""
    _check_variant(name, 1, 1030)


# ------------------------------------------------------------------------------ more than 4096 agents in one env
def _wide_state(N, clump, seed):
    """lattice 1 m apart; pairs of the last tournament round (>= 4096 for N > 4096) and of lower rounds moved to
    0.5 m (spheres overlap by 0.1 m); clump: 9 last-round pairs packed into one 18-agent clump (17 pairs per agent:
    the round walk).  Returns the state and the rounds of the pairs in contact."""
    rng = np.random.default_rng(seed)
    st = H.random_state(rng, 1, N, spacing=1.0, z0=2.0, jitter=0.0, tilt=0.02, vel=0.1, angvel=0.1)
    part = bm.tournament_partner(N)
    last = part.shape[0] - 1
    used = np.zeros(N, bool)
    chosen = []
    for r in [last] * 80 + list(rng.integers(0, last, 80)):
        i = int(rng.integers(0, N))
        for _ in range(N):
            j = int(part[r, i])
            if j != i and not used[i] and not used[j]:
                break
            i = (i + 1) % N
        else:
            continue
        used[i] = used[j] = True
        chosen.append((min(i, j), max(i, j), r))
    pos = st['pos'][0]
    off = np.float32(0.5 / np.sqrt(3))
    for i, j, r in chosen:
        pos[j] = pos[i] + off
    if clump:
        lo = [i for i in range(N) if not used[i] and part[last, i] > i and not used[part[last, i]]][:9]
        cl = np.array([[a, b, c] for a in range(3) for b in range(3) for c in range(2)], np.float32) * 0.2
        for q, i in enumerate(lo):
            j = int(part[last, i])
            pos[i] = cl[2 * q] + np.array([-6.0, -6.0, 6.0], np.float32)
            pos[j] = cl[2 * q + 1] + np.array([-6.0, -6.0, 6.0], np.float32)
            chosen.append((i, j, last))
    st['pos'][0] = pos
    return st, np.array([r for _, _, r in chosen])


@pytest.mark.parametrize('N', [4097, 4100])
@pytest.mark.parametrize('clump', [False, True])
def test_more_than_4096_agents(N, clump):
    """One env of N > 4096 agents (contact_env_kernel: its bit mask of occupied rounds must cover rounds >= 4096).
    Sparse pairs take the level walk, the clump the round walk; both hold pairs of the last round.  One step against
    the oracle, A bit-exact, and the same step again bit for bit."""
    import mrsgym_b200 as M
    st, rounds = _wide_state(N, clump, 4097 + N)
    assert np.sum(rounds >= 4096) >= 9 and np.sum(rounds < 4096) >= 9
    out = []
    for rep in range(2):
        sw = M.Swarm(1, N, K, None, M._abi.X_POS_VEL, R_COMM)
        H.upload_state(sw, st)
        sw.step(None)
        out.append(sw)
    assert torch.equal(out[0].state, out[1].state)
    sw = out[0]
    g1 = H.read_state(sw)
    r1 = V.oracle_steps(st, {})
    scale = max(1.0, float(np.max(np.abs(r1['vel']))))
    for k, tol in V.CONTACT_BAND:
        err = float(np.max(np.abs(g1[k] - r1[k])))
        assert err <= tol * scale, (k, err, scale)
    X = sw.X_window()[0].cpu().numpy()
    np.testing.assert_array_equal(sw.A_window()[0].cpu().numpy(), spec.adjacency(X[..., :3], R_COMM))
    assert sw.read_status() == 0 and sw.read_stats()['agent_contact_rows'] >= len(rounds)


# ------------------------------------------------------------------------------ sensors and MRS
def test_sensors_use_the_contact_radius():
    """CONTACT_RADIUS = 0.06 below AGENT_RADIUS = 0.3: mrs_proximity / mrs_raycast match oracle/sensors.py, and
    collision(), get_contact_points, get_closest_objects and the step agree on which pairs touch."""
    import mrsgym_b200 as M
    from oracle import sensors
    env = M.MRS(N_AGENTS=4, N_ENVS=2, CONTACT_RADIUS=0.06, ACTION_TYPE='set_speeds', HEADLESS=True)
    sw = env.swarm
    pos = np.array([[[0, 0, 2], [0.2, 0, 2], [5, 0, 2], [5, 5, 2]],        # a pair 0.2 m apart: no contact
                    [[0, 0, 2], [0.1, 0, 2], [5, 0, 2], [5, 5, 2]]], np.float32)   # 0.10 m: contact
    st = dict(pos=pos, quat=np.tile(np.array([0, 0, 0, 1], np.float32), (2, 4, 1)), vel=np.zeros((2, 4, 3), np.float32),
              angvel=np.zeros((2, 4, 3), np.float32))
    st['vel'][:, 0, 0], st['vel'][:, 1, 0] = 0.2, -0.2
    H.upload_state(sw, st)
    P = bm.PhysicsParams(contact_radius=0.06)
    ga, ne, gg, co = sensors.proximity(pos, st['quat'], P)
    pr = sw.proximity()
    np.testing.assert_allclose(pr['gap_agent'].cpu().numpy(), ga, atol=1e-6)
    np.testing.assert_array_equal(pr['nearest'].cpu().numpy(), ne)
    np.testing.assert_array_equal(pr['collision'].cpu().numpy().astype(bool), co)
    dirs = np.array([[1.0, 0, 0], [-1.0, 0, 0], [0, 0, -1.0]], np.float32)
    rc = sw.raycast(torch.from_numpy(dirs).cuda(), (0.0, 0.0, 0.0), False, 100.0)
    d_ref, o_ref = sensors.raycast(pos, st['quat'], dirs, (0, 0, 0), False, 100.0, P)
    np.testing.assert_array_equal(rc['object'].cpu().numpy().reshape(o_ref.shape), o_ref)
    fin = np.isfinite(d_ref)
    np.testing.assert_allclose(rc['dist'].cpu().numpy().reshape(d_ref.shape)[fin], d_ref[fin], atol=1e-5)
    assert d_ref[0, 0, 0] == pytest.approx(0.2 - 0.06) and d_ref[1, 0, 0] == pytest.approx(0.1 - 0.06)
    col = env.env.collision().cpu().numpy()
    cp = env.env.get_contact_points()
    cl = env.env.get_closest_objects(0.02)['mask'].cpu().numpy()
    assert not col[0, :2].any() and col[1, :2].all()
    assert (cp['object'][0, :2, 0].cpu().numpy() == -1).all() and (cp['object'][1, :2, 0].cpu().numpy() == [1, 0]).all()
    assert not cl[0, 0, 1] and cl[1, 0, 1]
    for e in range(2):          # the step applies a pair row exactly where the sensors report a contact
        one = M.Swarm(1, 4, 0, None, M._abi.X_POS_VEL, contact_radius=0.06)
        H.upload_state(one, {k: v[e:e + 1] for k, v in st.items()})
        one.step(None)
        assert (one.read_stats()['agent_contact_rows'] > 0) == (e == 1)


def test_mrs_physics_options_reach_the_step():
    """MRS(CONTACT_RADIUS=, SOLVER_ITERS=, DT=) steps like a Swarm with the same fields, and SOLVER_ITERS set after
    construction takes effect at the next step"""
    import mrsgym_b200 as M
    E, N = 12, 5
    st = V.make_state('heap', E, N, seed=3)
    fields = dict(contact_radius=0.06, solver_iters=3, dt=0.005)
    env = M.MRS(N_AGENTS=N, N_ENVS=E, CONTACT_RADIUS=0.06, SOLVER_ITERS=3, DT=0.005, ACTION_TYPE='set_speeds')
    sw = _swarm(E, N, fields)
    for s in (env.swarm, sw):
        H.upload_state(s, st)
    env.step(None)
    sw.step(None)
    assert torch.equal(env.swarm.state, sw.state)
    env.SOLVER_ITERS = 1
    env.step(None)
    V.apply(sw, dict(solver_iters=1))
    sw.step(None)
    assert torch.equal(env.swarm.state, sw.state)


# ------------------------------------------------------------------------------ status bits
@pytest.mark.parametrize('E,N', [(12, 8), (6, 48), (2, 200)])
def test_nonfinite_state_sets_the_status(E, N):
    """+inf position and NaN velocity in one agent of env 5 % E: MRS_STATUS_NONFINITE, stats['nonfinite'] = the
    non-finite agents after the step; envs outside that env's warp-chunk (N <= 32) or other envs (N > 32) step
    exactly as without the bad agent, the others of its chunk to float32 rounding"""
    st = V.make_state('heap', E, N, seed=11)
    bad = dict((k, v.copy()) for k, v in st.items())
    e_bad = 5 % E
    bad['pos'][e_bad, 1, 0] = np.inf
    bad['vel'][e_bad, 1, 2] = np.nan
    a, b = _swarm(E, N, {}), _swarm(E, N, {})
    H.upload_state(a, st)
    H.upload_state(b, bad)
    a.step(None)
    b.step(None)
    assert b.read_status() & 2
    gb = H.read_state(b)
    nonfinite = int(np.sum(~np.all(np.isfinite(np.concatenate([gb[k] for k in ('pos', 'vel', 'angvel', 'quat')], -1)), -1)))
    assert nonfinite >= 1 and b.read_stats()['nonfinite'] == nonfinite
    sa, sb = a.state.view(13, E, N), b.state.view(13, E, N)
    per_chunk = 32 // (1 << (N - 1).bit_length()) if N <= 32 else 1
    c0 = (e_bad // per_chunk) * per_chunk
    others = [e for e in range(E) if not c0 <= e < c0 + per_chunk]
    assert torch.equal(sa[:, others], sb[:, others])
    mates = [e for e in range(c0, min(E, c0 + per_chunk)) if e != e_bad]
    if mates:
        assert float((sa[:, mates].double() - sb[:, mates].double()).abs().max()) < 2e-5


def test_pair_overflow_sets_the_status():
    """N = 48, a clump of 30 agents all in range of each other: 435 pairs > 4 * 64 = 256 the per-env solver holds"""
    import mrsgym_b200 as M
    E, N = 2, 48
    rng = np.random.default_rng(9)
    st = H.random_state(rng, E, N, spacing=1.5, z0=3.0, jitter=0.05, tilt=0.05, vel=0.1, angvel=0.1)
    cl = np.array([[a, b, c] for a in range(5) for b in range(3) for c in range(2)], np.float32) * 0.12
    st['pos'][0, :30] = cl + np.array([20.0, 20.0, 3.0], np.float32)
    sw = _swarm(E, N, {})
    H.upload_state(sw, st)
    sw.step(None)
    assert sw.read_status() & M._abi.STATUS_CONTACT_OVERFLOW
    assert bool(torch.isfinite(sw.state).all())
