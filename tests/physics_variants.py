"""Non-default physics for the contact tests: one dict per variant, applied to both the CUDA step (the
MrsConfig of a Swarm) and the CPU oracle (bullet_model.PhysicsParams + spec.SpecEnv), plus seeded start states in
which each variant changes the result.  Shared by test_cpu_physics_variants.py (oracle only) and
test_gpu_physics_variants.py."""
from __future__ import annotations

import numpy as np

# MrsConfig top-level fields a variant may set (SpecEnv takes them as arguments)
TOP_LEVEL = ('dt', 'gravity')

# every MrsPhysicsParams field a variant sets -> its PhysicsParams counterpart
PHYS_FIELDS = {
    'erp2': 'erp2', 'slop': 'slop', 'contact_margin': 'contact_margin', 'mu_ground': 'mu_ground',
    'mu_agent': 'mu_agent', 'ground_contact': 'ground_contact', 'agent_contact': 'agent_contact',
    'agent_radius': 'agent_radius', 'contact_radius': 'contact_radius', 'solver_iters': 'solver_iters',
    'solver_tol': 'solver_tol',
}

# MrsPhysicsParams fields neither these variants nor the free-flight cases (flight_regimes.py) set, and why
NOT_VARIED = {
    'inertia': 'derived from the mass and the collision box in both models (PhysicsParams.inertia_diag), not a free '
               'setting; the mass case of flight_regimes.py sets it with the mass',
    'ground_z': 'scene geometry of plane.urdf, fixed by the reference world',
    'col_radius': 'cf2x collision cylinder, fixed by the reference model',
    'col_halfheight': 'cf2x collision cylinder, fixed by the reference model',
    'col_margin': 'Bullet collision margin of the cylinder, fixed by the reference model',
}

# name -> (fields, state kind the fields matter in)
VARIANTS = {
    'hull_contact': (dict(contact_radius=0.06), 'hull'),
    'iters1': (dict(solver_iters=1), 'heap'),
    'iters3': (dict(solver_iters=3), 'heap'),
    'loose_tol': (dict(solver_tol=1e-2), 'heap_only'),
    'mu_ground0': (dict(mu_ground=0.0), 'touchdown'),
    'mu_ground15': (dict(mu_ground=1.5), 'touchdown'),
    'mu_agent0': (dict(mu_agent=0.0), 'graze'),
    'mu_agent1': (dict(mu_agent=1.0), 'graze'),
    'erp2': (dict(erp2=0.2), 'baumgarte'),
    'margin': (dict(contact_margin=0.05), 'baumgarte'),
    'slop': (dict(slop=1e-3), 'baumgarte'),
    'no_ground': (dict(ground_contact=0), 'sunk'),
    'no_pairs': (dict(agent_contact=0), 'baumgarte'),
    'dt_mars': (dict(dt=0.005, gravity=3.71), 'heap'),
    'small_agents': (dict(agent_radius=0.1, contact_radius=0.1), 'small'),
}

# One-step band of the contact tests (test_gpu_parity.CONTACT_BAND) and the contact-grade trajectory bar of a few
# steps (test_gpu_parity.test_full_size_c3_control_with_contact)
CONTACT_BAND = (('vel', 3e-4), ('pos', 3e-6), ('angvel', 1e-3))
TRAJ_BAR = (('pos', 5e-2), ('vel', 0.5))


def apply(sw, fields):
    """Write a variant into a Swarm's MrsConfig (read by every following step)."""
    for k, v in fields.items():
        if k in TOP_LEVEL:
            setattr(sw.cfg, k, float(v))
        else:
            cur = getattr(sw.cfg.phys, k)
            setattr(sw.cfg.phys, k, type(cur)(v))


def spec_env(E, N, st, fields, K=0, comm_range=float('inf')):
    """The oracle under a variant (NO_ACTION steps: ref.step(None)), started from the float32 state st."""
    from oracle import bullet_model as bm
    from oracle import spec
    phys = {PHYS_FIELDS[k]: v for k, v in fields.items() if k not in TOP_LEVEL}
    top = {k: float(v) for k, v in fields.items() if k in TOP_LEVEL}
    env = spec.SpecEnv(E, N, 'set_speeds', K=K, comm_range=comm_range, dt=top.get('dt', 0.01),
                       gravity=top.get('gravity', 9.81), phys=bm.PhysicsParams(**phys))
    env.set_state(pos=st['pos'].astype(np.float64), quat=st['quat'].astype(np.float64),
                  vel=st['vel'].astype(np.float64), angvel=st['angvel'].astype(np.float64))
    env.reset_rings()
    return env


def oracle_steps(st, fields, T=1):
    E, N = st['pos'].shape[:2]
    env = spec_env(E, N, st, fields)
    for _ in range(T):
        env.step(None)
    return dict(pos=env.pos.copy(), quat=env.quat.copy(), vel=env.vel.copy(), angvel=env.angvel.copy())


def band_ratio(a, b, bar=CONTACT_BAND):
    """largest |a - b| over the bar, in multiples of the bar"""
    return max(float(np.max(np.abs(a[k] - b[k]))) / tol for k, tol in bar)


def discrimination(st, fields, T=1, bar=CONTACT_BAND):
    """How far (in bars) the oracle under `fields` lands from the oracle under the default physics and, for a sweep
    cap k, from the cap k + 1.  A kernel that ignored the field would be off by this much."""
    got = oracle_steps(st, fields, T)
    out = {'default': band_ratio(got, oracle_steps(st, {}, T), bar)}
    if 'solver_iters' in fields:
        nxt = dict(fields, solver_iters=fields['solver_iters'] + 1)
        out['next_iters'] = band_ratio(got, oracle_steps(st, nxt, T), bar)
    return out, got


# ------------------------------------------------------------------------------ start states
# A state is built from small groups of agents ("units") on a horizontal lattice, 1.4 m apart (no contact between
# units at the default radius); the agents of an env are then shuffled so that partners sit at arbitrary indices.
SPACING = 1.4
Z_AIR = 2.0
Z_TOUCH = 0.5 + 0.0125 + 0.001 + 0.004      # collision-cylinder rim 4 mm above the ground: within the contact margin


def _dir(rng):
    a = rng.uniform(0, 2 * np.pi)
    e = rng.uniform(-0.3, 0.3)
    return np.array([np.cos(a) * np.cos(e), np.sin(a) * np.cos(e), np.sin(e)])


def _pair(rng, sep, z, approach, tangential=0.0):
    """two agents `sep` apart around (0, 0, z), closing at `approach` m/s, sliding past each other at `tangential`"""
    n = _dir(rng)
    t = np.cross(n, [0.0, 0.0, 1.0])
    t /= np.linalg.norm(t)
    p = np.array([[0, 0, z], [0, 0, z]]) + np.outer([-0.5, 0.5], n) * sep
    v = np.outer([0.5, -0.5], n) * approach + np.outer([0.5, -0.5], t) * tangential
    return p, v


def _unit(kind, rng, k):
    if kind == 'free':
        return np.array([[0.0, 0.0, 3.0]]), rng.uniform(-0.2, 0.2, (1, 3))
    if kind == 'hull':      # in hull contact (0.09-0.13 m) or in contact only at the default radius (0.3-0.6 m)
        sep = rng.uniform(0.09, 0.13) if k % 2 == 0 else rng.uniform(0.3, 0.6)
        return _pair(rng, sep, Z_AIR, 0.3)
    if kind == 'small':     # 0.18-0.3 m: in contact as 0.1 m spheres near the low end, as 0.3 m spheres always
        return _pair(rng, rng.uniform(0.18, 0.3), Z_AIR, 0.3)
    if kind == 'graze':     # sphere gap -10..+10 mm at the default radius, 1 m/s tangential relative velocity
        return _pair(rng, rng.uniform(0.59, 0.61), Z_AIR, 0.2, tangential=1.0)
    if kind == 'overlap':   # penetrating by 1-5 cm
        return _pair(rng, rng.uniform(0.55, 0.59), Z_AIR, 0.1)
    if kind == 'speculative':       # 30-45 mm gap closing at 6 m/s: a row only with a margin above the gap
        return _pair(rng, rng.uniform(0.63, 0.645), Z_AIR, 6.0)
    if kind == 'touchdown':         # landing at 0.5 m/s with 1 m/s horizontal velocity
        a = rng.uniform(0, 2 * np.pi)
        return np.array([[0.0, 0.0, Z_TOUCH]]), np.array([[np.cos(a), np.sin(a), -0.5]])
    if kind == 'pressed':           # resting 2-5 mm deep in the ground
        return np.array([[0.0, 0.0, Z_TOUCH - 0.004 - rng.uniform(0.002, 0.005)]]), np.zeros((1, 3))
    if kind == 'sunk':              # well below the ground plane
        return np.array([[0.0, 0.0, 0.45]]), np.array([[0.0, 0.0, -0.2]])
    if kind == 'heap':              # 2 x 2 agents 0.45 m apart (spheres overlap by 0.15 m) landing at 1 m/s
        g = np.array([[0, 0], [1, 0], [0, 1], [1, 1]], float) * 0.45 - 0.225
        p = np.concatenate([g + rng.uniform(-0.02, 0.02, (4, 2)), Z_TOUCH + rng.uniform(0, 0.01, (4, 1))], axis=1)
        v = np.concatenate([rng.uniform(-0.1, 0.1, (4, 2)), np.full((4, 1), -1.0)], axis=1)
        return p, v
    raise ValueError(kind)


# state kind -> the unit kinds its envs cycle through (env e takes row e % len(rows)); 'free' rows and a 'touchdown'
# row put converged envs next to ones the sweep cap binds in, in one warp-chunk
STATE_UNITS = {
    'hull': [['hull']],
    'heap': [['heap'], ['free'], ['heap', 'touchdown'], ['touchdown']],
    # N > 32 solves an agent that touches only the ground on its own, with its own early exit, where the oracle stops
    # all rows of an env together: under a loose tolerance the two stopping rules differ by up to the tolerance, so
    # the tolerance variant runs on heaps without lone ground contacts
    'heap_only': [['heap'], ['free'], ['heap', 'free']],
    'touchdown': [['touchdown']],
    'graze': [['graze']],
    'baumgarte': [['overlap', 'speculative', 'pressed']],
    'sunk': [['sunk', 'overlap']],
    'small': [['small']],
}


def make_state(kind, E, N, seed=0):
    """float32 start state [E, N, ...] of a state kind (see STATE_UNITS)."""
    from scipy.spatial.transform import Rotation
    rng = np.random.default_rng(seed)
    rows = STATE_UNITS[kind]
    cols = int(np.ceil(np.sqrt(N)))
    pos = np.zeros((E, N, 3))
    vel = np.zeros((E, N, 3))
    for e in range(E):
        units = rows[e % len(rows)]
        i, k = 0, 0
        while i < N:
            p, v = _unit(units[k % len(units)], rng, k)
            if i + len(p) > N:
                p, v = _unit('free', rng, k)
            c = (np.array([k % cols, k // cols, 0.0]) - np.array([cols / 2, cols / 2, 0.0])) * SPACING
            pos[e, i:i + len(p)] = p + c
            vel[e, i:i + len(p)] = v
            i += len(p)
            k += 1
        perm = rng.permutation(N)
        pos[e], vel[e] = pos[e, perm], vel[e, perm]
    rpy = np.concatenate([rng.uniform(-0.05, 0.05, (E * N, 2)), rng.uniform(-np.pi, np.pi, (E * N, 1))], axis=1)
    quat = Rotation.from_euler('xyz', rpy).as_quat().reshape(E, N, 4)
    st = dict(pos=pos, quat=quat, vel=vel, angvel=rng.uniform(-0.1, 0.1, (E, N, 3)))
    return {k: v.astype(np.float32) for k, v in st.items()}
