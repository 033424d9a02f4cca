"""Oracle-only checks behind test_gpu_physics_variants.py: every physics variant, in the start state the GPU tests
use it in, moves the oracle's step far beyond the bar the GPU is held to (so a kernel that ignored the field would
fail there), and every MrsPhysicsParams field is varied here or by the free-flight cases, or excused by name."""
import dataclasses

import numpy as np
import pytest

import physics_variants as V
from oracle import bullet_model as bm
from oracle import sensors

# (E, N) of the GPU tests that run every variant on all of their envs
SHAPES = [(12, 5), (8, 12), (67, 8), (10, 16), (4, 32), (6, 48), (2, 200)]


def test_every_physics_field_is_varied_or_excused():
    """varied by a contact variant here, by a free-flight case (flight_regimes.py), or excused by name"""
    from mrsgym_b200 import _abi
    import flight_regimes as F
    fields = {f for f, _ in _abi.MrsPhysicsParams._fields_}
    flight = set().union(*(set(f) for _, f, _ in F.CASES.values())) - set(F.TOP_LEVEL)
    assert set(V.PHYS_FIELDS) | flight | set(V.NOT_VARIED) == fields
    assert not (set(V.PHYS_FIELDS) | flight) & set(V.NOT_VARIED)
    oracle_fields = {f.name for f in dataclasses.fields(bm.PhysicsParams)}
    assert set(V.PHYS_FIELDS.values()) <= oracle_fields
    varied = set()
    for fields_, kind in V.VARIANTS.values():
        assert set(fields_) <= set(V.PHYS_FIELDS) | set(V.TOP_LEVEL) and kind in V.STATE_UNITS
        varied |= set(fields_)
    assert varied == set(V.PHYS_FIELDS) | set(V.TOP_LEVEL)


@pytest.mark.parametrize('name', list(V.VARIANTS))
@pytest.mark.parametrize('E,N', SHAPES)
def test_variant_moves_the_oracle_beyond_the_bar(name, E, N):
    fields, kind = V.VARIANTS[name]
    st = V.make_state(kind, E, N, seed=N)
    disc, _ = V.discrimination(st, fields)
    assert min(disc.values()) >= 10, disc


@pytest.mark.parametrize('name', ['hull_contact', 'erp2', 'margin'])
def test_variant_moves_the_oracle_beyond_the_bar_1030(name):
    fields, kind = V.VARIANTS[name]
    disc, _ = V.discrimination(V.make_state(kind, 1, 1030, seed=1030), fields)
    assert min(disc.values()) >= 10, disc


@pytest.mark.parametrize('name', ['hull_contact', 'iters3', 'mu_ground15', 'no_pairs', 'small_agents'])
def test_variant_moves_the_oracle_beyond_the_bar_520x64(name):
    fields, kind = V.VARIANTS[name]
    st = V.make_state(kind, 520, 64, seed=64)
    disc, _ = V.discrimination({k: v[[0, 1, 259, 519]] for k, v in st.items()}, fields)
    assert min(disc.values()) >= 10, disc


def test_heap_state_mixes_converged_and_capped_envs():
    """under a sweep cap of 3 the first warp-chunk at N = 8 holds envs that converge earlier and envs the cap stops"""
    st = V.make_state('heap', 4, 8, seed=8)
    capped = V.oracle_steps(st, dict(solver_iters=3))
    free = V.oracle_steps(st, dict(solver_iters=50))
    per_env = np.max(np.abs(capped['vel'] - free['vel']), axis=(1, 2))
    assert (per_env == 0).any() and (per_env > 1e-2).any(), per_env


def test_sensor_oracle_uses_the_contact_radius():
    """agents are CONTACT_RADIUS spheres for the sensors, as for the step's pair rows; AGENT_RADIUS is the spawn
    separation only"""
    P = bm.PhysicsParams(agent_radius=0.3, contact_radius=0.06)
    pos = np.array([[[0, 0, 2], [0.2, 0, 2], [0.2, 3, 2]]], float)
    quat = np.tile([0.0, 0.0, 0.0, 1.0], (1, 3, 1))
    ga, ne, gg, co = sensors.proximity(pos, quat, P)
    np.testing.assert_allclose(ga[0, :2], 0.2 - 0.12)
    assert list(ne[0, :2]) == [1, 0] and not co[0, :2].any()
    d, o = sensors.raycast(pos, quat, np.array([[1.0, 0, 0]]), (0, 0, 0), False, 100.0, P)
    assert o[0, 0, 0] == 1 and d[0, 0, 0] == pytest.approx(0.2 - 0.06)
