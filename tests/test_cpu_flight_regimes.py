"""Oracle-only checks behind test_gpu_flight_regimes.py: in every free-flight case (tests/flight_regimes.py), at the
shapes and seeds the GPU tests use, the oracle's step lands at least 10 one-step delta bars (helpers.delta_ratio) away
from what a subtly wrong kernel would compute -- the field at its default, the feature switched off, the other side of
a cut-off, or the attitude series cut after x^2 -- so such a kernel fails there.  Also: every MrsPhysicsParams field
is varied by the contact variants or by these cases, or excused."""
import numpy as np
import pytest

import flight_regimes as F
import physics_variants as V


def _discrimination(name, E, N, seed, picks=None):
    st, rpm, probe = F.make_case(name, E, N, seed=seed)
    if picks is not None:
        st = {k: v[picks] for k, v in st.items()}
        rpm = None if rpm is None else rpm[picks]
        probe = probe[picks]
    ref = F.oracle_step(st, F.fields_of(name), rpm)
    assert all(np.all(np.isfinite(v)) for v in ref.values()), name
    assert picks is None or name != 'ring'          # the flipped ring is rebuilt at the full shape
    wrong = F.wrong_results(name, st, rpm, probe, seed, E, N)
    return {k: max(F.probe_ratio(st, ref, o, p).values()) for k, (o, p) in wrong.items()}


@pytest.mark.parametrize('name', list(F.CASES))
@pytest.mark.parametrize('E,N', F.SHAPES)
def test_case_is_far_from_a_wrong_kernel(name, E, N):
    disc = _discrimination(name, E, N, seed=N)
    if name in F.CONTINUITY:
        assert not disc
        return
    assert disc and min(disc.values()) >= 10, disc


@pytest.mark.parametrize('name', ['spin_below', 'spin_above', 'clamp', 'attitude', 'ring', 'downwash_near',
                                  'threshold_high', 'mass'])
def test_case_is_far_from_a_wrong_kernel_1030(name):
    disc = _discrimination(name, 1, 1030, seed=1030)
    assert min(disc.values()) >= 10, disc


@pytest.mark.parametrize('name', ['spin_above', 'clamp', 'hclip', 'downwash_near', 'clamp5', 'mass'])
def test_case_is_far_from_a_wrong_kernel_520x64(name):
    disc = _discrimination(name, 520, 64, seed=64, picks=[0, 1, 259, 519])
    assert min(disc.values()) >= 10, disc


def test_only_fixed_geometry_is_excused():
    """the free-flight fields are varied here; what stays excused is the inertia (derived from the mass, which the
    mass case sets with it), the ground plane and the collision cylinder"""
    from mrsgym_b200 import _abi
    fields = {f for f, _ in _abi.MrsPhysicsParams._fields_}
    flight = set().union(*(set(f) for _, f, _ in F.CASES.values())) - set(F.TOP_LEVEL)
    assert {'mass', 'lin_damping', 'ang_damping', 'max_coord_vel', 'gyro', 'ang_motion_threshold'} <= flight
    assert set(V.NOT_VARIED) == {'inertia', 'ground_z', 'col_radius', 'col_halfheight', 'col_margin'}
    assert set(V.PHYS_FIELDS) | flight | set(V.NOT_VARIED) == fields


def test_states_reach_the_edges():
    """the start states sit where the issue of each case is: spin on both sides of the cap and within 1e-6 of it,
    coordinates at the clamp, rolls on both sides of pi/2 and pi, propellers below the clip, partners 9.99 / 10.01 m
    off, dz = 0, one ulp, 1-10 mm and beta ~ 0; every coordinate below 128 m"""
    from oracle import bullet_model as bm
    dt = 0.01
    wdt = lambda n: np.linalg.norm(F.make_case(n, 6, 48, seed=1)[0]['angvel'].astype(np.float64), axis=-1) * dt
    a = wdt('spin_below')
    assert a.min() >= 0.4 and a.max() <= 0.78
    assert wdt('spin_above').min() > np.pi / 4
    assert np.max(np.abs(wdt('spin_at_cap') / (np.pi / 4) - 1)) < 2e-6
    st, _, _ = F.make_case('clamp', 6, 48, seed=1)
    assert np.all(st['vel'][..., 2] < -99.9) and np.all(np.max(np.abs(st['angvel']), -1) > 99.4)
    st, _, _ = F.make_case('attitude', 6, 48, seed=1)
    R = bm.quat_to_mat(st['quat'].astype(np.float64))
    assert (R[..., 2, 2] > 0).any() and (R[..., 2, 2] < 0).any() and np.all(st['pos'][..., 2] >= 0.65)
    st, _, _ = F.make_case('ring', 2, 200, seed=1)
    p = st['pos'].astype(np.float64)
    dxy = np.linalg.norm(p[:, :, None, :2] - p[:, None, :, :2], axis=-1)
    dz = p[:, None, :, 2] - p[:, :, None, 2]
    near = dxy[(dz > 30)]
    assert np.any(np.abs(near - 9.99) < 1e-4) and np.any(np.abs(near - 10.01) < 1e-4)
    st, _, _ = F.make_case('downwash_near', 2, 200, seed=1)
    p = st['pos']
    dz = (p[:, None, :, 2] - p[:, :, None, 2]).astype(np.float32)
    dxy = np.linalg.norm(p[:, :, None, :2].astype(np.float64) - p[:, None, :, :2], axis=-1)
    close = dxy < 1.0
    np.fill_diagonal(close[0], False)
    np.fill_diagonal(close[1], False)
    z32 = np.abs(p[:, :, 2]).max()
    assert np.any(close & (dz == 0)) and np.any(close & (dz > 0) & (dz <= np.spacing(np.float32(z32))))
    assert np.any(close & (dz >= 1e-3) & (dz <= 1e-2)) and np.any((dxy == 0) & (np.abs(dz - 0.6875) < 1e-3))
    for name in F.CASES:
        assert np.all(np.abs(F.make_case(name, 2, 200, seed=2)[0]['pos']) < 128.0)
