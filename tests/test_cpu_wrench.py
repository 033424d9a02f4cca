"""The external wrench in the CPU oracle (wrench_cases.step_with_wrench): a zero wrench changes nothing, two analytic
anchors, and every scene of wrench_cases.py at least 10 bars away from each wrong kernel it is built to catch, so that
test_gpu_wrench.py fails a kernel that makes one of those mistakes."""
import numpy as np
import pytest

import helpers as H
import wrench_cases as W
from oracle import bullet_model as bm


def _modes_for(kind):
    return [None] if W.KINDS[kind][0] or kind == 'weightless' else [None, 'set_speeds', 'set_target_vel']


@pytest.mark.parametrize('mode', [None, 'set_speeds', 'set_target_vel', 'set_control'])
def test_zero_wrench_is_bit_identical(mode):
    """the oracle step with a zero wrench (and with None) gives the numbers of the plain step bit for bit"""
    E, N = 3, 6
    st, F, Tq = W.make_case('tilted', E, N, seed=1)
    acts = W.mode_actions(mode, E, N, st, seed=2, T=2)
    out = []
    zero = np.zeros((E, N, 3))
    for wrench in ('plain', (None, None), (zero, zero)):
        env = H.make_spec(E, N, mode or 'set_speeds', 1, 1.5, st)
        for t in range(2):
            a = None if acts is None else acts[t]
            X, A = env.step(a) if wrench == 'plain' else W.step_with_wrench(env, a, *wrench)
        out.append((H.spec_state(env), X, A))
    out = [out[0], out[1], out[0], out[2]]
    for i in (0, 2):
        for k in out[i][0]:
            np.testing.assert_array_equal(out[i][0][k], out[i + 1][0][k])
        np.testing.assert_array_equal(out[i][1], out[i + 1][1])
        np.testing.assert_array_equal(out[i][2], out[i + 1][2])


@pytest.mark.parametrize('mode', [None, 'set_speeds'])
def test_uniform_lift_equals_lower_gravity(mode):
    """F = m delta z on every agent steps like gravity g - delta (free flight), to float64 rounding"""
    E, N, delta = 2, 5, 3.2
    st, _, _ = W.make_case('tilted', E, N, seed=3)
    acts = W.mode_actions(mode, E, N, st, seed=4)
    F = np.zeros((E, N, 3))
    F[..., 2] = W.MASS * delta
    a = W.oracle_step(st, mode, acts, F, np.zeros((E, N, 3)))
    from oracle import spec
    env = spec.SpecEnv(E, N, mode or 'set_speeds', gravity=W.G - delta, phys=bm.PhysicsParams())
    env.set_state(**{k: v.astype(np.float64) for k, v in st.items()})
    env.step(None if acts is None else acts[0])
    dt = 0.01
    assert np.max(np.abs(a['vel'] - env.vel)) * W.MASS / dt <= 1e-12 * W.WEIGHT
    assert np.max(np.abs(a['angvel'] - env.angvel)) == 0.0


def test_torque_at_rest_without_damping():
    """at rest, zero damping, gyro off: dw = dt R I^-1 R^T tau"""
    E, N = 2, 6
    st, _, Tq = W.make_case('tilted', E, N, seed=5)
    st['angvel'][:] = 0.0
    st['vel'][:] = 0.0
    P = dict(lin_damping=0.0, ang_damping=0.0, gyro=0)
    got = W.oracle_step(st, None, None, np.zeros((E, N, 3)), Tq, **P)
    R = W.rotmat(st['quat'])
    I = bm.PhysicsParams(**P).inertia_diag()
    want = 0.01 * np.einsum('...ij,...j->...i', R, np.einsum('...ji,...j->...i', R, Tq.astype(np.float64)) / I)
    np.testing.assert_allclose(got['angvel'], want, rtol=1e-12, atol=0)
    assert np.max(np.abs(want)) > 10 * H.FLOOR['angvel']


@pytest.mark.parametrize('kind', list(W.KINDS))
def test_cases_tell_wrong_kernels_apart(kind):
    """each scene lands >= 10 bars away from every wrong kernel it names, in every mode it runs in"""
    contact, wrongs = W.KINDS[kind]
    E, N = 4, 8
    st, F, Tq = W.make_case(kind, E, N, seed=7)
    for mode in _modes_for(kind):
        acts = W.mode_actions(mode, E, N, st, seed=8)
        ref = W.oracle_step(st, mode, acts, F, Tq)
        for wrong in wrongs:
            bad = W.oracle_step(st, mode, acts, F, Tq, wrong=wrong)
            r = W.bar_ratio(st, ref, bad, contact)
            assert r >= 10, (kind, mode, wrong, r)


def test_nan_action_keeps_the_wrench():
    """a NaN-action agent loses its rotor wrench but keeps the external one: >= 10 bars from zeroing it"""
    E, N = 2, 8
    st, F, Tq = W.make_case('tilted', E, N, seed=9)
    acts = W.mode_actions('set_speeds', E, N, st, seed=10)
    acts[0, 1, 3, 2] = np.nan
    ref = W.oracle_step(st, 'set_speeds', acts, F, Tq)
    for wrong in ('none', 'nan_zeroed'):
        bad = W.oracle_step(st, 'set_speeds', acts, F, Tq, wrong=wrong)
        assert W.bar_ratio(st, ref, bad, False) >= 10, wrong


def test_friction_margins():
    """the slide scenes sit a factor 2 from the friction limit of the ground rows, both ways: below it the agents stay
    put, above it they slide"""
    E, N = 2, 6
    for kind, moves in (('slide_below', False), ('slide_above', True)):
        st, F, Tq = W.make_case(kind, E, N, seed=11)
        got = W.oracle_step(st, None, None, F, Tq)
        vxy = np.linalg.norm(got['vel'][..., :2], axis=-1)
        free = 0.01 * np.linalg.norm(F[..., :2], axis=-1) / W.MASS          # the push with no friction at all
        if moves:
            assert np.all(vxy > 0.2 * free), kind
        else:
            assert np.all(vxy < 1e-6), kind
