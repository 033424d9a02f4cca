"""Free-flight step at the edges of its range: spin below / at / above the attitude cap, the +-max_coord_vel clamp,
the gyroscopic term, attitudes past 90 degrees with the rotors on, the ground-effect clip and the downwash cut-offs
(dxy < 10, dz > 0, dz -> 0+, beta = dw2 dz + dw3 ~ 0), plus the free-flight MrsPhysicsParams fields the contact tests
leave at their defaults.  One dict of fields per case, applied to both the CUDA step (the MrsConfig of a Swarm) and
the CPU oracle, and seeded float32 start states with their set_speeds actions.  Shared by test_cpu_flight_regimes.py
(oracle only) and test_gpu_flight_regimes.py."""
from __future__ import annotations

import contextlib
import math

import numpy as np

import helpers as H

# ------------------------------------------------------------------------------ cases
# name -> (unit kinds an env cycles through, physics fields, actions: 'hover' = set_speeds at HOVER +- 2 %,
# None = NO_ACTION)
REGIMES = {
    'spin_below': (['spin_below'], {}, 'hover'),        # |w| dt in [0.4, 0.78]: the Taylor series, x up to pi/8
    'spin_above': (['spin_above'], {}, 'hover'),        # |w| 80-170 rad/s: the capped step
    'spin_at_cap': (['spin_at_cap'], {}, 'hover'),      # |w| dt = pi/4 (1 +- 1e-6): continuity across the cap
    'spin_free': (['spin_below', 'spin_above'], {}, None),
    'gyro': (['gyro'], {}, 'hover'),
    # At 100 m/s the default damping (0.04 (1 + |v|) v = 404 m/s^2, and the rotor drag) outweighs every force the
    # rotors can produce, so the clamp binds only undamped and unpowered: gravity takes v_z past -100 and the gyro term
    # moves an angular coordinate past +-100
    'clamp': (['clamp100'], dict(lin_damping=0.0, ang_damping=0.0), None),
    'attitude': (['roll', 'pitch'], {}, 'hover'),       # roll around +-pi/2 and pi, pitch near +-pi/2, z 0.65-1
    'hclip': (['hclip'], dict(ground_contact=0), 'hover'),      # propellers below gnd_hclip (no ground rows)
    'ring': (['ring'], {}, 'hover'),                    # partners 9.99 / 10.01 m off, 40-60 m higher
    'downwash_near': (['dz0', 'dz_ulp', 'dz_small', 'beta0_axis', 'beta0_off'], {}, 'hover'),
}

# the free-flight MrsPhysicsParams fields off their defaults (the generic kernels; the baked ones never see them)
VARIANTS = {
    'lin_damping': (['spin_below'], dict(lin_damping=0.5), 'hover'),
    'ang_damping': (['spin_below'], dict(ang_damping=0.5), 'hover'),
    'no_gyro': (['gyro'], dict(gyro=0), 'hover'),
    'clamp5': (['clamp5'], dict(max_coord_vel=5.0), 'hover'),
    'threshold_low': (['spin_below'], dict(ang_motion_threshold=0.3), 'hover'),     # binds early, jumps to pi/4
    'threshold_high': (['spin_wide'], dict(ang_motion_threshold=3.0, dt=0.02), 'hover'),   # series up to x = 1.5
    'mass': (['spin_below'], dict(mass=0.04), 'hover'),         # inertia follows the mass on both sides
}

CASES = dict(REGIMES, **VARIANTS)

# cases in which no field or boundary can be moved without changing the answer by design: they check that the
# step is continuous across the attitude cap, and finite where the downwash has its singular points
CONTINUITY = ('spin_at_cap',)

TOP_LEVEL = ('dt', 'gravity')
HOVER_SPREAD = 0.02

# (E, N) of the GPU tests that run the cases on all of their envs
SHAPES = [(12, 5), (67, 8), (10, 16), (4, 32), (6, 48), (2, 200)]


def apply(sw, fields):
    """Write a case's fields into a Swarm's MrsConfig.  A mass also sets the inertia, as the oracle derives it from
    the mass (PhysicsParams.inertia_diag)."""
    from oracle import bullet_model as bm
    for k, v in fields.items():
        if k in TOP_LEVEL:
            setattr(sw.cfg, k, float(v))
        else:
            cur = getattr(sw.cfg.phys, k)
            setattr(sw.cfg.phys, k, type(cur)(v))
        if k == 'mass':
            I = bm.PhysicsParams(mass=float(v)).inertia_diag()
            for i in range(3):
                sw.cfg.phys.inertia[i] = float(np.float32(I[i]))


# ------------------------------------------------------------------------------ oracle
@contextlib.contextmanager
def _integrator(fn):
    """run bullet_step with another integrate_positions (a test-local wrong kernel)"""
    from oracle import bullet_model as bm
    keep = bm.integrate_positions
    if fn is not None:
        bm.integrate_positions = fn
    try:
        yield
    finally:
        bm.integrate_positions = keep


def oracle_step(st, fields, rpm, dt_override=None, integrate=None, no_hclip=False, flip_gnd=False, no_downwash=False):
    """One oracle step from the float32 state st under `fields` (rpm None: NO_ACTION).  The keyword switches give the
    result of a subtly wrong kernel: another integrator, no ground-effect clip, the ground-effect predicate inverted,
    no downwash."""
    from oracle import bullet_model as bm
    from oracle import spec
    E, N = st['pos'].shape[:2]
    phys = {k: v for k, v in fields.items() if k not in TOP_LEVEL}
    dt = float(fields.get('dt', 0.01))
    quad = bm.QuadParams(dw1=0.0) if no_downwash else None
    env = spec.SpecEnv(E, N, 'set_speeds', dt=dt, gravity=float(fields.get('gravity', 9.81)),
                       phys=bm.PhysicsParams(**phys), quad=quad)
    env.set_state(pos=st['pos'].astype(np.float64), quat=st['quat'].astype(np.float64),
                  vel=st['vel'].astype(np.float64), angvel=st['angvel'].astype(np.float64))
    if no_hclip:
        env.der['GroundEffectHClip'] = 0.0
    if flip_gnd:            # get_ori feeds only the ground-effect test `roll < pi/2 and pitch < pi/2` under set_speeds
        get_ori = env.get_ori

        def flipped():
            o = get_ori()
            ok = (o[..., 0] < np.float32(np.pi / 2)) & (o[..., 1] < np.float32(np.pi / 2))
            o = o.copy()
            o[..., 0] = np.where(ok, np.float32(3.0), np.float32(0.0))
            o[..., 1] = 0.0
            return o
        env.get_ori = flipped
    with _integrator(integrate):
        env.step(None if rpm is None else rpm)
    return H.spec_state(env)


def probe_ratio(s0, ref, other, probe):
    """how far (in delta bars, helpers.delta_ratio) `other` lands from the oracle `ref`, over the probe agents"""
    sub = lambda d: {k: v[probe] for k, v in d.items()}
    return H.delta_ratio(sub(s0), sub(ref), sub(other))


# ------------------------------------------------------------------------------ start states
# An env is a lattice of cells 30 m apart (centres within +-105 m, so every coordinate stays below 128 m).  A cell
# holds one unit: a block of sub-units 2.5 m apart at one height (agents at equal heights feel no downwash from each
# other; 1.5 m or more apart at height differences below ~0.8 m, it underflows), or one downwash ring.  Cells are far
# enough apart that no agent sees the downwash of another cell, and every agent flies clear of the ground and of
# contact except in the 'attitude' (0.65-1 m) and 'hclip' (no ground rows) units.  Agents are shuffled in each env.
CELL = 30.0
CELLS = 8                       # per side
SUB = 2.5


def _rand_rot(rng, n):
    from scipy.spatial.transform import Rotation
    return Rotation.random(n, random_state=rng).as_quat()


def _euler(rpy):
    from scipy.spatial.transform import Rotation
    return Rotation.from_euler('xyz', np.atleast_2d(rpy)).as_quat()


def _spin(rng, lo, hi, dt=0.01):
    """angular velocity of magnitude |w| dt in [lo, hi] about a random axis, denser towards hi (where the higher
    terms of the attitude series weigh most)"""
    a = rng.normal(size=3)
    return a / np.linalg.norm(a) * (lo + (hi - lo) * np.sqrt(rng.uniform())) / dt


def _hover(rng, n):
    return H.HOVER * (1 + HOVER_SPREAD * rng.uniform(-1, 1, (n, 4)))


def _agent(p, q, v, w, rpm):
    return dict(pos=np.atleast_2d(p), quat=np.atleast_2d(q), vel=np.atleast_2d(v), angvel=np.atleast_2d(w),
                rpm=np.atleast_2d(rpm))


def _sub_unit(kind, rng, z, flip):
    """agents of one sub-unit around (0, 0, z)"""
    v = rng.uniform(-0.3, 0.3, 3)
    if kind in ('spin_below', 'spin_above', 'spin_at_cap', 'spin_wide', 'gyro'):
        if kind == 'spin_below':
            w = _spin(rng, 0.4, 0.78)
        elif kind == 'spin_above':
            w = _spin(rng, 0.8, 1.7)
        elif kind == 'spin_at_cap':
            w = _spin(rng, 1.0, 1.0) * (np.pi / 4) * (1 + rng.choice([-1e-6, 1e-6]))
        elif kind == 'spin_wide':       # dt = 0.02: |w| dt in [1, 2.95], below a threshold of 3
            w = _spin(rng, 1.0, 2.95, dt=0.02)
        else:                           # fast spin about an axis off the principal axes
            w = _spin(rng, 0.4, 0.7)
        return _agent([0, 0, z], _rand_rot(rng, 1), v, w, _hover(rng, 1))
    if kind == 'clamp100':              # falling at 99.91-99.99 m/s, one angular coordinate at 99.5-99.99 rad/s
        w = rng.uniform(-30, 30, 3)
        i = rng.integers(0, 3)
        w[i] = rng.choice([-1, 1]) * rng.uniform(99.5, 99.99)
        return _agent([0, 0, z], _rand_rot(rng, 1), [v[0], v[1], -rng.uniform(99.91, 99.99)], w, np.zeros(4))
    if kind == 'clamp5':                # upside down: thrust and gravity take v_z past -5, a roll torque w_x past 5
        q = _euler([np.pi, rng.uniform(-0.05, 0.05), rng.uniform(-0.05, 0.05)])
        w = np.array([rng.uniform(4.9, 4.99), rng.uniform(-1, 1), rng.uniform(-1, 1)])
        rpm = H.HOVER * np.array([1.03, 1.03, 0.97, 0.97])
        return _agent([0, 0, z], q, [v[0], v[1], -rng.uniform(4.95, 4.99)], w, rpm)
    if kind in ('roll', 'pitch'):       # rotors on at 0.65-1 m: the ground-effect predicate
        # The reference tests roll < f32(pi/2) on the euler angles of the float32 quaternion, the kernels the sign of
        # R22 / R21; in a window of ~4e-8 rad just above pi/2 the two disagree by construction, so no state sits there
        if kind == 'roll':
            rpy = [rng.choice([np.pi / 2, np.pi, -np.pi / 2]) + rng.choice([-1e-3, 1e-3]), rng.uniform(-0.3, 0.3),
                   rng.uniform(-np.pi, np.pi)]
        else:
            rpy = [rng.uniform(-0.3, 0.3), rng.choice([-1, 1]) * (np.pi / 2 - 1e-3), rng.uniform(-np.pi, np.pi)]
        return _agent([0, 0, z], _euler(rpy), v, rng.uniform(-0.5, 0.5, 3), _hover(rng, 1))
    if kind == 'hclip':                 # propellers 1-3 cm high, below gnd_hclip = 3.8 cm
        rpy = [rng.uniform(-0.05, 0.05), rng.uniform(-0.05, 0.05), rng.uniform(-np.pi, np.pi)]
        return _agent([0, 0, z], _euler(rpy), v, rng.uniform(-0.5, 0.5, 3), _hover(rng, 1))
    # downwash pairs: the lower agent at (0, 0, z), the upper one dxy away horizontally, dz higher
    if kind == 'dz0':                   # equal heights: no downwash either way (the kernels' dz > 0 test)
        dxy, dz = rng.uniform(0.65, 0.8), 0.0
    elif kind == 'dz_ulp':              # one float32 ulp apart: alpha ~ 3e11 N, the exponential makes it 1e-3 - 1 N
        dxy, dz = rng.uniform(0.8, 0.9), None
    elif kind == 'dz_small':            # dz -> 0+: ~1e-4 N near 1 mm, below the bar near 1 cm
        dxy, dz = rng.uniform(0.65, 0.8), rng.uniform(1e-3, 1e-2)
    elif kind == 'beta0_axis':          # beta ~ 0 straight above: exp(0) = 1, the full alpha ~ 0.16 N
        dxy, dz = 0.0, 0.6875 + rng.choice([-1, 1]) * rng.uniform(1e-5, 1e-3)
    elif kind == 'beta0_off':           # beta ~ 0 off axis: dxy / beta in [0.3, 1.5] (|beta| >= 2e-4 keeps the
        s = rng.choice([-1, 1]) * rng.uniform(1.25e-3, 6.25e-3)     # float32 rounding of beta below 1e-4 relative)
        dz = 0.6875 + s
        dxy = abs(0.16 * s) * rng.uniform(0.3, 1.5)
    else:
        raise ValueError(kind)
    a = rng.uniform(0, 2 * np.pi)
    up = np.array([dxy * np.cos(a), dxy * np.sin(a), 0.0])
    v2 = rng.uniform(-0.3, 0.3, 3)
    q = _euler([[rng.uniform(-0.1, 0.1), rng.uniform(-0.1, 0.1), rng.uniform(-3, 3)] for _ in range(2)])
    w = rng.uniform(-0.5, 0.5, (2, 3))
    z32 = np.float32(z)
    if dz is None:
        z_up = np.nextafter(z32, np.float32(np.inf)) if rng.integers(0, 2) else z32
        z_lo = z32 if z_up != z32 else np.nextafter(z32, np.float32(-np.inf))
        p = np.array([[0, 0, z_lo], up + [0, 0, z_up]], np.float64)
    else:
        p = np.array([[0, 0, z], up + [0, 0, z + dz]])
    return _agent(p, q, np.stack([v, v2]), w, _hover(rng, 2))


def _cell(kind, rng, m, flip, k):
    """one cell of the lattice (positions relative to its centre); `probe` marks the agents the discrimination of a
    flipped state compares"""
    if kind == 'ring':
        # the centre agent feels the downwash of P partners 40-60 m above it (one height, so the partners feel
        # nothing from each other), all at 9.99 m or all at 10.01 m, alternating per cell; `flip` swaps the radii
        P = max(8, m - 1)
        z = rng.uniform(3, 5)
        r = 9.99 if (k % 2 == 0) != flip else 10.01
        ang = rng.uniform(0, 2 * np.pi) + 2 * np.pi * np.arange(P) / P
        zp = z + rng.uniform(45, 60)     # where one partner's force peaks at dxy = 10 m (~1.2e-5 N)
        p = np.concatenate([[[0, 0, z]], np.stack([r * np.cos(ang), r * np.sin(ang), np.full(P, zp)], 1)])
        # the centre flies upright: the downwash acts along body z, so all of it shows in one velocity coordinate
        q = np.concatenate([_euler([rng.uniform(-0.1, 0.1), rng.uniform(-0.1, 0.1), rng.uniform(-3, 3)]),
                            _rand_rot(rng, P)])
        out = _agent(p, q, rng.uniform(-0.3, 0.3, (P + 1, 3)), rng.uniform(-0.5, 0.5, (P + 1, 3)),
                     _hover(rng, P + 1))
        out['probe'] = np.arange(P + 1) == 0
        return out
    z = {'roll': (0.65, 1.0), 'pitch': (0.65, 1.0), 'hclip': (0.01, 0.03),
         'clamp100': (50, 60), 'clamp5': (10, 20)}.get(kind, (3, 8))
    z = rng.uniform(*z)
    side = int(np.ceil(np.sqrt(m)))
    parts = []
    for s in range(m):
        u = _sub_unit(kind, rng, z, flip)
        u['pos'] = u['pos'] + np.array([(s % side - (side - 1) / 2) * SUB, (s // side - (side - 1) / 2) * SUB, 0.0])
        parts.append(u)
    out = {key: np.concatenate([u[key] for u in parts]) for key in parts[0]}
    out['probe'] = np.ones(len(out['pos']), bool)
    return out


def make_case(name, E, N, seed=0, flip=False):
    """float32 start state [E, N, ...] of a case, its set_speeds actions [E, N, 4] (None for NO_ACTION) and the
    probe mask [E, N]"""
    kinds, _, act = CASES[name]
    rng = np.random.default_rng(seed)
    m = max(1, int(np.ceil(N / 48)))
    keys = ('pos', 'quat', 'vel', 'angvel', 'rpm', 'probe')
    out = {key: np.zeros((E, N) + ((3,) if key in ('pos', 'vel', 'angvel') else (4,) if key in ('quat', 'rpm') else ()),
                         bool if key == 'probe' else np.float64) for key in keys}
    for e in range(E):
        i, k = 0, 0
        while i < N:
            assert k < CELLS * CELLS, (name, N)
            c = _cell(kinds[(k + e) % len(kinds)], rng, m, flip, k)
            n = min(len(c['pos']), N - i)
            c['pos'] = c['pos'] + np.array([(k % CELLS - (CELLS - 1) / 2) * CELL, (k // CELLS - (CELLS - 1) / 2) * CELL, 0])
            for key in keys:
                out[key][e, i:i + n] = c[key][:n]
            i += n
            k += 1
        perm = rng.permutation(N)
        for key in keys:
            out[key][e] = out[key][e, perm]
    st = {key: out[key].astype(np.float32) for key in ('pos', 'quat', 'vel', 'angvel')}
    assert np.all(np.abs(st['pos']) < 128.0)
    rpm = out['rpm'].astype(np.float32) if act == 'hover' else None
    return st, rpm, out['probe']


def fields_of(name):
    return CASES[name][1]


# ------------------------------------------------------------------------------ what a wrong kernel would compute
def wrong_results(name, st, rpm, probe, seed, E, N):
    """{label: (state of a subtly wrong kernel, probe mask)} for a case: the same oracle with the field at its
    default or the feature switched off, the other side of a boundary, or a truncated attitude series"""
    fields = fields_of(name)
    base = {k: v for k, v in fields.items()}
    out = {}
    kinds = CASES[name][0]
    if name in VARIANTS:
        dflt = {k: v for k, v in fields.items() if k == 'dt'}
        out['default'] = (oracle_step(st, dflt, rpm), probe)
    if name in ('spin_below', 'spin_free', 'threshold_high'):
        out['series_x2'] = (oracle_step(st, base, rpm, integrate=integrate_series_x2), probe)
    if 'spin_above' in kinds:
        out['no_cap'] = (oracle_step(st, dict(base, ang_motion_threshold=math.inf), rpm), probe)
    if name in ('gyro', 'spin_above'):
        out['no_gyro'] = (oracle_step(st, dict(base, gyro=False), rpm), probe)
    if name == 'clamp' or name == 'clamp5':
        out['no_clamp'] = (oracle_step(st, dict(base, max_coord_vel=math.inf), rpm), probe)
    if name == 'attitude':
        out['gnd_predicate'] = (oracle_step(st, base, rpm, flip_gnd=True), probe)
    if name == 'hclip':
        out['no_hclip'] = (oracle_step(st, base, rpm, no_hclip=True), probe)
    if name == 'downwash_near':
        out['no_downwash'] = (oracle_step(st, base, rpm, no_downwash=True), probe)
    if name == 'ring':
        st2, rpm2, probe2 = make_case(name, E, N, seed=seed, flip=True)
        assert np.array_equal(probe, probe2)
        for k in st:
            assert np.array_equal(st[k][probe], st2[k][probe])
        out['other_radius'] = (oracle_step(st2, base, rpm2), probe)
    return out


def integrate_series_x2(pos, quat, v, w, P, dt):
    """bullet_model.integrate_positions with sin(x)/x and cos(x) cut after the x^2 term (a kernel that lost the
    higher terms of its series), below the cap"""
    from oracle import bullet_model as bm
    pos1 = pos + dt * v
    ang = np.sqrt(np.sum(w * w, axis=-1, keepdims=True))
    capped = ang * dt > P.ang_motion_threshold
    ang_c = np.where(capped, 0.5 * (0.5 * math.pi) / dt, ang)
    x = 0.5 * ang_c * dt
    with np.errstate(invalid='ignore', divide='ignore'):
        k_exact = np.sin(x) / ang_c
    k = np.where(capped, k_exact, 0.5 * dt * (1 - x * x / 6))
    c = np.where(capped, np.cos(x), 1 - x * x / 2)
    dq = np.concatenate([w * np.where(ang_c < 1e-3, 0.5 * dt, k), c], axis=-1)
    q1 = bm.quat_mul(dq, quat)
    return pos1, q1 / np.sqrt(np.sum(q1 * q1, axis=-1, keepdims=True))
