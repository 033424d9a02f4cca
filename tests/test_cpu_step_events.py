"""The scenes and expected counts of tests/step_events.py, and the oracle paths they use, on the CPU: every decision a
count depends on sits clear of its threshold (float32 cannot flip it), every scene tells a plausible wrong count from
the right one, and the counting / NaN-aware oracle paths reduce to the plain ones."""
import numpy as np
import pytest

import helpers as H
import physics_variants as V
import step_events as SE
from oracle import bullet_model as bm

NS = (5, 8, 12, 16, 32, 48, 64, 200)
Z_MARGIN, D2_MARGIN, LAM_MARGIN, TOL_FACTOR = 1e-3, 1e-4, 1e-6, 10.0


@pytest.fixture(scope='module')
def thr():
    return SE.thresholds()


def _run(kind, N, mode=None, T=3, nan_steps=(0,)):
    st = SE.make_scene(kind, N)
    acts = None
    if kind == 'nan_chunk':
        mode = mode or 'set_speeds'
        acts = H.random_actions(np.random.default_rng(N), mode, T, SE.E0, N, st['pos'])
        SE.plant_nans(acts, N, nan_steps)
    return st, acts, SE.oracle_run(st, mode, acts, T, **SE.SCENE_PHYS.get(kind, {}))


@pytest.mark.parametrize('N', NS)
@pytest.mark.parametrize('kind', SE.SCENES)
def test_scene_margins(kind, N, thr):
    """heights, pair distances, impulses and the sweep-exit test all clear of their thresholds"""
    gz, lim2 = thr
    _, _, (_, steps) = _run(kind, N)
    m = SE.margins(steps, gz, lim2, N)
    assert m['z'] >= Z_MARGIN and m['d2'] >= D2_MARGIN and m['lam'] >= LAM_MARGIN, m
    tol = bm.PhysicsParams().solver_tol
    for s in steps:
        c = s['counts']
        for w in (c['worst'] if c else []):
            w = w[c['active'] & (w > 0)]
            assert np.all((w >= TOL_FACTOR * tol) | (w <= tol / TOL_FACTOR)), w


@pytest.mark.parametrize('mode', H.MODES)
@pytest.mark.parametrize('N', (5, 8, 16, 48))
def test_nan_scene_margins_every_mode(mode, N, thr):
    """...and no pair sits near the downwash singularity at dz -> 0+, where float32 rounding of the positions would
    decide the trajectory (the scene steps with rotor forces)"""
    gz, lim2 = thr
    for nan_steps in ((0,), (1,)):
        _, _, (_, steps) = _run('nan_chunk', N, mode, nan_steps=nan_steps)
        m = SE.margins(steps, gz, lim2, N)
        assert m['z'] >= Z_MARGIN and m['d2'] >= D2_MARGIN and m['lam'] >= LAM_MARGIN, (nan_steps, m)
        for s in steps:
            assert max(H.downwash_sensitivity(p) for p in s['pre']) <= 1e3, nan_steps


@pytest.mark.parametrize('N', (5, 8, 12, 16))
def test_scenes_discriminate(N, thr):
    """per-chunk and per-agent counting differ; rows in range and rows that pushed differ; free flight counts 0"""
    gz, lim2 = thr
    gpw = SE.chunk_envs(N)
    _, _, (_, steps) = _run('nan_chunk', N)
    ex = SE.expected_stats(steps, N, gz, lim2)
    per_chunk = len({e // gpw for e, _ in SE.NAN_AGENTS})
    assert ex['nan_actions'] == len(SE.NAN_AGENTS) > per_chunk
    assert ex['agent_contact_rows'] > 0 and ex['nonfinite'] == 0
    _, _, (_, steps) = _run('nonfinite', N)
    ex = SE.expected_stats(steps, N, gz, lim2)
    per_chunk = len({e // gpw for e, _ in SE.BAD_AGENTS})
    assert ex['nonfinite'] == 3 * len(SE.BAD_AGENTS) and per_chunk < len(SE.BAD_AGENTS)
    for kind in ('separating', 'lifting'):
        _, _, (_, steps) = _run(kind, N)
        ex = SE.expected_stats(steps, N, gz, lim2)
        rows_in_range = sum(int(np.sum(s['counts']['active'])) for s in steps)
        assert rows_in_range > 0 and 0 < ex['solver_sweeps'] <= ex['contact_chunks']
        assert ex['agent_contact_rows'] == 0 and ex['ground_contacts'] == 0, (kind, ex)
    _, _, (_, steps) = _run('heap', N)
    ex = SE.expected_stats(steps, N, gz, lim2)
    assert ex['agent_contact_rows'] > 0 and ex['ground_contacts'] > 0 and 0 < ex['solver_sweeps'] <= 3 * ex['contact_chunks']
    _, _, (_, steps) = _run('free', N)
    assert all(v == 0 for v in SE.expected_stats(steps, N, gz, lim2).values())
    assert SE.expected_stats(steps, N, gz, lim2, 'many') == SE.expected_stats(steps, N, gz, lim2)


@pytest.mark.parametrize('N', (5, 8, 12, 16, 32))
def test_nan_alone_needs_the_hand_off(N, thr):
    """At every width of the N <= 32 kernels the NaN scene has a warp-chunk that only its NaN agent sends to the contact
    path: with the NaN at step 1, a kernel whose NaN test never hands a chunk over counts fewer contact chunk-steps --
    1 per such chunk for single steps, 2 (T - 1) for mrs_step_many"""
    gz, lim2 = thr
    _, _, (_, steps) = _run('nan_chunk', N, nan_steps=(1,))
    lone = {f: SE.expected_stats(steps, N, gz, lim2, f)['contact_chunks'] -
            SE.expected_stats(steps, N, gz, lim2, f, nan_hands_off=False)['contact_chunks'] for f in ('single', 'many')}
    assert lone['single'] >= 1 and lone['many'] == 2 * lone['single'], lone


@pytest.mark.parametrize('mode', H.MODES)
def test_nan_oracle_discriminates(mode):
    """The NaN agents' one-step result is >= 10 bars from a step that gives them the downwash of the others, and
    from one that applies the rotor wrench of their action with the NaN read as 0"""
    N = 8
    st, acts, (env, steps) = _run('nan_chunk', N, mode, T=1)
    nan = steps[0]['nan']
    got = H.spec_state(env)
    # the downwash received: the other agents' rotor speeds of the right step, 0 for the NaN agents, as set_speeds
    dw = H.make_spec(SE.E0, N, 'set_speeds', 0, float('inf'), st)
    dw.step(np.where(nan[..., None], 0.0, steps[0]['rpm']).astype(np.float32))
    wrench = H.make_spec(SE.E0, N, mode, 0, float('inf'), st)
    wrench.step(np.nan_to_num(acts[0], nan=0.0))
    for other in (H.spec_state(dw), H.spec_state(wrench)):
        sub = {k: v[nan] for k, v in got.items()}
        assert V.band_ratio(sub, {k: v[nan] for k, v in other.items()}) >= 10


def test_counts_none_is_todays_solve():
    """counts=None leaves solve_contacts bit for bit as it is, and counts does not change the result"""
    st = V.make_state('heap', 8, 8, seed=5)
    P = bm.PhysicsParams()
    pos, quat = st['pos'].astype(np.float64), st['quat'].astype(np.float64)
    v1, w1 = bm.unconstrained_velocities(quat, st['vel'].astype(np.float64), st['angvel'].astype(np.float64),
                                         np.zeros((8, 8, 3)), np.zeros((8, 8, 3)), P, 0.01, 9.81)
    a = bm.solve_contacts(pos, quat, v1, w1, P, 0.01)
    counts = {}
    b = bm.solve_contacts(pos, quat, v1, w1, P, 0.01, counts)
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x, y)
    assert counts['sweeps'].shape == (8,) and counts['pair_rows'].shape == (8, 8)
    assert np.all(counts['pair_rows'].sum(-1) % 2 == 0)      # both agents of a pushing pair count it


@pytest.mark.parametrize('mode', H.MODES)
def test_nan_policy_reduces_to_the_plain_step(mode):
    """No NaN: nan_policy='agent_none' is bit for bit step(actions).  Every agent NaN: the state equals step(None)
    and the controller state is unchanged (also before the controller's first call)."""
    rng = np.random.default_rng(7)
    E, N, T = 3, 5, 3
    st = H.random_state(rng, E, N)
    acts = H.random_actions(rng, mode, T, E, N, st['pos'])
    a, b = H.make_spec(E, N, mode, 0, float('inf'), st), H.make_spec(E, N, mode, 0, float('inf'), st)
    for t in range(T):
        a.step(acts[t])
        b.step(acts[t], nan_policy='agent_none')
    for k, v in H.spec_state(a).items():
        np.testing.assert_array_equal(v, H.spec_state(b)[k])
    assert a.ctrl.keys() == b.ctrl.keys() and all(np.array_equal(a.ctrl[k], b.ctrl[k]) for k in a.ctrl)
    for warm in (0, 1):
        c, d = H.make_spec(E, N, mode, 0, float('inf'), st), H.make_spec(E, N, mode, 0, float('inf'), st)
        for t in range(warm):
            c.step(acts[t])
            d.step(acts[t])
        before = {k: np.array(v, copy=True) for k, v in d.ctrl.items()}
        c.step(None)
        d.step(np.full_like(acts[0], np.nan), nan_policy='agent_none')
        for k, v in H.spec_state(c).items():
            np.testing.assert_array_equal(v, H.spec_state(d)[k])
        assert d.ctrl.keys() == before.keys()
        for k in before:
            np.testing.assert_array_equal(np.broadcast_to(before[k], d.ctrl[k].shape), d.ctrl[k])
        assert np.all(d.last['rpm'] == 0.0)
    with pytest.raises(Exception, match='contains NaN'):
        c.step(np.full_like(acts[0], np.nan))


def test_nan_agent_first_call_is_per_agent():
    """set_target_vel: an agent whose first controller call was a NaN step starts its derivative afresh at its next
    finite step, exactly like an oracle that never saw the NaN step for it"""
    rng = np.random.default_rng(3)
    E, N = 1, 2
    st = H.random_state(rng, E, N, spacing=3.0)
    acts = H.random_actions(rng, 'set_target_vel', 2, E, N)
    acts[0, 0, 0, 1] = np.nan
    env = H.make_spec(E, N, 'set_target_vel', 0, float('inf'), st)
    env.step(acts[0], nan_policy='agent_none')
    assert np.isnan(env.ctrl['last_vel_e'][0, 0, 0]) and not np.isnan(env.ctrl['last_vel_e'][0, 1, 0])
    env.step(acts[1], nan_policy='agent_none')
    assert np.all(np.isfinite(env.ctrl['d_vel_e'])) and np.all(np.isfinite(env.vel))
