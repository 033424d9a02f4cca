"""Cases of the analytic sensors (mrs_proximity / mrs_raycast) and the float32 bounds they are judged by.

Shared by test_cpu_sensors.py (oracle and float32 emulation only) and test_gpu_sensors.py.  A case is a small group
of agents built around one env (its agents take slots 0..n-1; the rest of the env is parked on a far lattice), for a
sensor configuration (CONFIGS: the MrsPhysicsParams fields the sensors read), a ray frame (body or world) and a
range.  The rays of a call are one direction set for every agent (directions()); the hand-built cases place their
partners so that chosen (agent, ray) pairs hit or miss an edge on purpose, and list those pairs as `edges`.

The answer is oracle/sensors.py in float64 on the float32 inputs.  Every decision an answer depends on is reported
through its margin (hit/miss r^2 - d^2, t against 0 and the range, the ground box edge 15 - |h|, the start above the
ground sz - ground_z, the runner-up partner, gap - threshold) next to a bound on what float32 rounding can move it
by.  The bounds are operation counts times EPS (the unit roundoff of float32) times the coordinate scale of the
decision; they are zero where every operation of the kernel is exact on the given numbers (dyadic geometry).  A
decision is certain when its margin clears its bound; the kernel must then agree exactly, and a distance must be
within its bound.
"""
from __future__ import annotations

import dataclasses

import numpy as np

from oracle import bullet_model as bm
from oracle import sensors

EPS = 2.0 ** -24
F32 = np.float32
# error of a unit ray direction in the kernel (division by the largest component, rotation by R, rsqrtf, scaling)
DIR_ERR = 16 * EPS
BOX = 15.0

# MrsPhysicsParams fields the sensor kernels read, and their defaults
SENSOR_FIELDS = {'ground_z': 0.5, 'col_radius': 0.06, 'col_halfheight': 0.0125, 'col_margin': 0.001,
                 'contact_radius': 0.3, 'agent_radius': 0.3}
CONFIGS = {
    'r30': {},
    'r06': dict(contact_radius=0.06),
    # every field off its default, on a dyadic grid so that hand-built ties are exact in float32
    'moved': dict(ground_z=0.25, col_radius=0.0625, col_halfheight=0.015625, col_margin=0.00390625,
                  contact_radius=0.125, agent_radius=0.2),
}
OFFSET = (0.03125, -0.0625, 0.015625)                     # ray start in the body frame: dyadic, nonzero
RAY_CALLS = ((False, 100.0), (True, float('inf')))        # (body, range) of the two raycast calls per scene
THRESHOLD = 0.04


def fields(cfg):
    """float32 values of every sensor field under a configuration"""
    return {k: float(F32(CONFIGS[cfg].get(k, v))) for k, v in SENSOR_FIELDS.items()}


def phys(cfg):
    return bm.PhysicsParams(**fields(cfg))


def apply(sw, cfg):
    """Write a configuration into a Swarm's MrsConfig (every field, so that both sides use the same float32 values)."""
    for k, v in fields(cfg).items():
        setattr(sw.cfg.phys, k, v)


def tie_threshold(cfg):
    """the gap of two agents 1 m apart: the threshold of the exact-tie case (float32)"""
    r = F32(fields(cfg)['contact_radius'])
    return float(F32(1.0) - F32(2.0) * r)


# ------------------------------------------------------------------------------ directions
def _unit(v):
    v = np.asarray(v, np.float64)
    return v / np.linalg.norm(v)


W_FAR = {30.0: _unit([0.8, 0.6, 0.05]), 60.0: _unit([-0.6, 0.8, 0.05]), 99.0: _unit([-0.8, -0.6, 0.05])}
FAR_RAYS = 32                                             # rays per far target, impact parameters 0 .. 1.2 r
FAR0 = 9


def directions(cfg, n=129, seed=5):
    """The direction set of every raycast call under a configuration (the first n):
    0 the far direction (magnitude 2.5), 1 down, 2 +x (dz = 0), 3 a 1e-30 direction, 4 a 1e30 direction, 5 zero,
    6 NaN, 7 +x with dz = -1 ulp, 8 +y, 9.. rays aimed at the far targets at impact parameters 0 .. 1.2 r, then
    seeded directions."""
    rng = np.random.default_rng(seed)
    r = fields(cfg)['contact_radius']
    d = [2.5 * W_FAR[30.0], [0, 0, -1], [1, 0, 0], 1e-30 * np.array([0.6, 0, -0.8]), 1e30 * np.array([0.2, 0.9, -0.3]),
         [0, 0, 0], [np.nan, 0.5, -0.5], [1, 0, -2.0 ** -23], [0, 1, 0]]
    for L, w in W_FAR.items():
        for k in range(FAR_RAYS):
            e = np.cross(w, rng.normal(size=3))
            e /= np.linalg.norm(e)
            b = 1.2 * r * k / (FAR_RAYS - 1)
            d.append(L * w + b * e)
    while len(d) < 129:
        v = rng.normal(size=3)
        v[2] = -abs(v[2]) if rng.uniform() < 0.7 else v[2]
        d.append(v * rng.choice([0.5, 1.0, 3.0]))
    return np.array(d, np.float64).astype(F32)[:n]


# ------------------------------------------------------------------------------ cases
ID = np.array([0, 0, 0, 1], F32)


def _quat(axis, angle):
    from scipy.spatial.transform import Rotation
    return Rotation.from_rotvec(_unit(axis) * angle).as_quat().astype(F32)


@dataclasses.dataclass
class Case:
    pos: np.ndarray                # [n, 3] float32
    quat: np.ndarray               # [n, 4] float32
    edges: list                    # hand-built (agent, ray) pairs that must be certain
    prox_edges: list = dataclasses.field(default_factory=list)    # hand-built agents whose proximity must be certain


def _case(agents, edges=(), prox_edges=()):
    pos = np.array([a[0] for a in agents], np.float64).astype(F32)
    quat = np.array([a[1] if len(a) > 1 else ID for a in agents], F32)
    return Case(pos, quat, list(edges), list(prox_edges))


def _start(p, body, q=ID):
    """ray start of an agent at p (float64 of the float32 start the kernel forms from p and OFFSET)"""
    R = bm.quat_to_mat(np.asarray(q, np.float64)) if body else np.eye(3)
    return np.asarray(p, np.float64) + R @ np.asarray(OFFSET)


def case_far(cfg, body, rng, seed):
    """a shooter and targets at 30, 60 and 99 m, hit by rays 0 and 9.. at impact parameters 0 .. 1.2 r"""
    g = np.random.default_rng(seed)
    p = np.array([g.uniform(-5, 5), g.uniform(-5, 5), 20.0], F32)
    s = _start(p, body)
    agents = [(p,)] + [(s + L * w,) for L, w in W_FAR.items()]
    edges = [(0, 0)] + [(0, FAR0 + k) for k in range(3 * FAR_RAYS)]
    return _case(agents, edges)


def case_range(cfg, body, rng, seed):
    """hits 2 mm inside and 2 mm beyond the range (+x rays); at an infinite range both at 50 m"""
    r = fields(cfg)['contact_radius']
    agents, edges = [], []
    for k, delta in enumerate((-0.002, 0.002)):
        p = np.array([-20.0, 4.0 * k - 2, 3.0], F32)
        s = _start(p, body)
        L = (rng + delta + r) if np.isfinite(rng) else 50.0 + 10 * k
        agents += [(p,), (s + [L, 0, 0],)]
        edges.append((2 * k, 2))
    return _case(agents, edges)


def case_tolerance(cfg, body, rng, seed):
    """a start inside a partner's sphere and a partner 0.5 m behind the start: +x misses both; down hits the ground"""
    r = fields(cfg)['contact_radius']
    pa, pb = np.array([-3.0, 6.0, 5.0], F32), np.array([-3.0, 9.0, 5.0], F32)
    agents = [(pa,), (_start(pa, body) + [0.5 * r, 0, 0],), (pb,), (_start(pb, body) - [0.5, 0, 0],)]
    return _case(agents, [(0, 2), (2, 2), (0, 1), (2, 1)])


def case_occlusion(cfg, body, rng, seed):
    """three partners on one +x ray; a partner in front of and one behind the ground on a down-slanted ray; a 1e30 ray"""
    gz = fields(cfg)['ground_z']
    agents = []
    p1 = np.array([-10.0, -6.0, 4.0], F32)
    agents += [(p1,)] + [(_start(p1, body) + [L, 0.01 * L, 0],) for L in (2.0, 4.0, 6.0)]
    u3 = _unit([0.6, 0, -0.8])
    for k, frac in enumerate((0.5, 1.5)):
        p = np.array([-5.0, -9.0 + 3 * k, 3.0], F32)
        s = _start(p, body)
        tg = (s[2] - gz) / 0.8
        agents += [(p,), (s + frac * tg * u3,)]
    p4 = np.array([-8.0, -12.0, 6.0], F32)
    agents += [(p4,), (_start(p4, body) + 2.0 * _unit([0.2, 0.9, -0.3]),)]
    return _case(agents, [(0, 2), (4, 3), (6, 3), (8, 4)])


def case_box(cfg, body, rng, seed):
    """down rays 3 mm inside / outside |x| = 15 and |y| = 15; a start exactly at ground_z and one below it; rays
    from 5 cm above the ground with dz = 0 and dz = -1 ulp"""
    gz = fields(cfg)['ground_z']
    o = np.asarray(OFFSET)
    agents = []
    for x, y in ((BOX - 0.003 - o[0], 1.0), (BOX + 0.003 - o[0], 3.0), (-5.0, -BOX + 0.003 - o[1]),
                 (-7.0, -BOX - 0.003 - o[1])):
        agents.append(([x, y, 2.0],))
    agents.append(([0.5, 7.0, gz - o[2]],))             # start exactly at ground_z (dyadic: exact in float32)
    agents.append(([0.5, 9.0, gz - 0.2],))              # start below the ground
    agents.append(([-12.0, 11.0, gz + 0.05],))          # grazing the ground: horizontal rays
    edges = [(k, 1) for k in range(6)] + [(6, 2), (6, 7)]
    return _case(agents, edges)


def case_frames(cfg, body, rng, seed):
    """tilted, inverted and on-side agents (the offset and body-frame rays turn with them) near the ground"""
    g = np.random.default_rng(seed)
    qs = [_quat([1, 0, 0], 0.4), _quat([1, 1, 0], 2.0), _quat([1, 0, 0], np.pi), _quat([0, 1, 0], np.pi / 2),
          _quat(g.normal(size=3), g.uniform(0, np.pi)), _quat([0, 0, 1], 1.0)]
    agents = [(np.array([3.0 + 0.9 * (k % 3), -3.0 + 0.9 * (k // 3), 1.0 + 0.3 * k]), q) for k, q in enumerate(qs)]
    return _case(agents)


def case_lone(cfg, body, rng, seed):
    return _case([([1.0, 2.0, 3.0], _quat([1, 2, 0], 0.3))], prox_edges=[0])


def case_coincident(cfg, body, rng, seed):
    """two agents at one point and one 0.5 m away"""
    return _case([([2.0, 2.0, 2.0],), ([2.5, 2.0, 2.0],), ([2.0, 2.0, 2.0],)], prox_edges=[0, 1, 2])


def case_lattice(cfg, body, rng, seed):
    """a 2 x 2 x 2 lattice of 0.75 m: every agent has three nearest partners at exactly the same distance"""
    pts = [[4 + 0.75 * i, 4 + 0.75 * j, 2 + 0.75 * k] for k in range(2) for j in range(2) for i in range(2)]
    return _case([(p,) for p in pts], prox_edges=list(range(8)))


def case_far_swarm(cfg, body, rng, seed):
    """eight agents 2 km from the origin, 0.4 - 1 m apart"""
    g = np.random.default_rng(seed)
    pts = np.array([2000.0, -1500.0, 3.0]) + g.uniform(-0.7, 0.7, (8, 3))
    return _case([(p, _quat(g.normal(size=3), 0.3)) for p in pts])


def case_tie(cfg, body, rng, seed):
    """two agents exactly 1 m apart (gap_agent == tie_threshold) and one whose ground gap equals it (identity)"""
    f = fields(cfg)
    thr = tie_threshold(cfg)
    ext = float(F32(f['col_halfheight']) + F32(f['col_margin']))
    zg = float(F32(f['ground_z'] + ext + thr))
    # a tie by design only where the kernel's arithmetic is exact on these numbers (float32 = float64)
    edges = [0, 1] if thr == 1.0 - 2.0 * f['contact_radius'] else []
    if ext == f['col_halfheight'] + f['col_margin'] and zg - ext - f['ground_z'] == thr:
        edges.append(2)
    return _case([([6.0, -6.0, 3.0],), ([7.0, -6.0, 3.0],), ([6.0, -2.0, zg],)], prox_edges=edges)


def case_tilts(cfg, body, rng, seed):
    """ground gaps of a few cm under tilts about axis-aligned and diagonal axes: near-level, 0.2 rad, 30 deg, on its
    side, inverted"""
    gz = fields(cfg)['ground_z']
    qs = [_quat([1, 1, 0], 1e-3), _quat([1, 0, 0], 0.2), _quat([1, 1, 0], 0.2), _quat([1, 1, 0], np.pi / 6),
          _quat([1, 1, 0], np.pi / 2), _quat([1, 0, 0], np.pi / 2), _quat([1, 0, 0], np.pi), _quat([1, 1, 0], np.pi)]
    xs = [-6.0, -5.0, -3.7, -2.6, -1.1, 0.0, 1.6, 2.7]             # distinct spacings: no near-ties of `nearest`
    agents = [([x, 12.0, gz + 0.02 + 0.006 * k], q) for k, (x, q) in enumerate(zip(xs, qs))]
    return _case(agents, prox_edges=list(range(8)))


CASES = {'far': case_far, 'range': case_range, 'tolerance': case_tolerance, 'occlusion': case_occlusion,
         'box': case_box, 'frames': case_frames, 'lone': case_lone, 'coincident': case_coincident,
         'lattice': case_lattice, 'far_swarm': case_far_swarm, 'tie': case_tie, 'tilts': case_tilts}


def case_sizes():
    return {k: len(f('r30', False, 100.0, 0).pos) for k, f in CASES.items()}


# ------------------------------------------------------------------------------ assembled scenes
@dataclasses.dataclass
class Scene:
    pos: np.ndarray        # [E, N, 3] float32
    quat: np.ndarray       # [E, N, 4] float32
    names: list            # case of each env
    edges: list            # (env, agent, ray) that must be certain
    prox_edges: list       # (env, agent) whose proximity must be certain


def parked(N):
    """slots a case does not use: a lattice 4 m apart, 1 km away (exact distances: lattice ties)"""
    k = np.arange(N)
    return np.stack([1000.0 + 4.0 * (k % 16), 1000.0 + 4.0 * ((k // 16) % 16), 500.0 + 4.0 * (k // 256)], -1)


def passes(E, N):
    """the case names each pass of an (E, N) shape holds per env (cases that need more than N agents are left out)"""
    fit = [k for k, n in case_sizes().items() if n <= N]
    P = -(-len(fit) // E)
    return [[fit[(p * E + e) % len(fit)] for e in range(E)] for p in range(P)]


def scene(cfg, names, N, body, rng):
    E = len(names)
    pos = np.broadcast_to(parked(N), (E, N, 3)).astype(F32)
    quat = np.broadcast_to(ID, (E, N, 4)).copy()
    edges, prox = [], []
    for e, name in enumerate(names):
        c = CASES[name](cfg, body, rng, 1000 + e)
        n = len(c.pos)
        pos[e, :n], quat[e, :n] = c.pos, c.quat
        edges += [(e, a, r) for a, r in c.edges]
        prox += [(e, a) for a in c.prox_edges]
    return Scene(pos, quat, names, edges, prox)


# ------------------------------------------------------------------------------ proximity: answer, margins, bounds
def _exact(x64):
    """float32 rounding leaves x unchanged"""
    return np.asarray(x64, np.float64) == np.asarray(x64, np.float64).astype(F32).astype(np.float64)


def proximity_verdict(pos, quat, P, thr, agents=None):
    """oracle answer + certainty of `agents` (default all): {'gap_agent', 'nearest', 'gap_ground', 'collision',
    'ga_bound', 'gg_bound', 'nearest_ok', 'collision_ok', 'ga_margin', 'gg_margin'} over [E, k]"""
    pos = np.asarray(pos, np.float64)
    E, N, _ = pos.shape
    agents = np.arange(N) if agents is None else np.asarray(agents)
    k = len(agents)
    thr = float(F32(thr))
    ga, ne, gg, co = sensors.proximity(pos, quat, P, thr, agents)
    dif = pos[:, agents, None, :] - pos[:, None, :, :]
    d2 = np.sum(dif * dif, -1)
    ex_d2 = np.all(_exact(dif) & _exact(dif * dif), -1) & _exact(d2)
    d2[:, np.arange(k), agents] = np.inf
    order = np.argsort(d2, axis=-1, kind='stable')[..., :2]
    first = np.take_along_axis(d2, order[..., :1], -1)[..., 0]
    if N > 2:
        second = np.take_along_axis(d2, order[..., 1:2], -1)[..., 0]
        exact_pair = (np.take_along_axis(ex_d2, order[..., :1], -1) & np.take_along_axis(ex_d2, order[..., 1:2], -1))[..., 0]
        nb = np.where(exact_pair, 0.0, 8 * EPS * (first + second))
        nearest_ok = (second - first > nb) | ((nb == 0) & (second >= first))
    else:
        nearest_ok = np.ones((E, k), bool)
    d1 = np.sqrt(first)
    r2 = 2.0 * P.contact_radius
    ex_ga = (np.take_along_axis(ex_d2, order[..., :1], -1)[..., 0] & _exact(d1) & _exact(d1 - r2)) | (N == 1)
    with np.errstate(invalid='ignore'):
        ga_bound = np.where(ex_ga, 0.0, 8 * EPS * (d1 + r2))
    q = np.asarray(quat, np.float64)[:, agents]
    ident = np.all(q == ID, axis=-1)
    ext = P.col_halfheight + P.col_margin
    z = pos[:, agents, 2]
    ex_gg = ident & _exact(ext) & _exact(z - ext) & _exact(z - ext - P.ground_z)
    gg_bound = np.where(ex_gg, 0.0, 4 * EPS * (np.abs(z) + abs(P.ground_z) + P.col_radius + P.col_halfheight
                                               + P.col_margin) + 16 * EPS * (P.col_radius + P.col_halfheight))
    with np.errstate(invalid='ignore'):
        a_true, g_true = ga - thr < -ga_bound, gg - thr < -gg_bound
        a_false = (ga - thr > ga_bound) | ((ga_bound == 0) & (ga >= thr))
        g_false = (gg - thr > gg_bound) | ((gg_bound == 0) & (gg >= thr))
    collision_ok = a_true | g_true | (a_false & g_false)
    return dict(gap_agent=ga, nearest=ne, gap_ground=gg, collision=co, ga_bound=ga_bound, gg_bound=gg_bound,
                nearest_ok=nearest_ok, collision_ok=collision_ok, ga_margin=ga - thr, gg_margin=gg - thr)


# ------------------------------------------------------------------------------ rays: answer, margins, bounds
def ray_verdict(pos, quat, dirs, body, rng, P, agents=None, offset=OFFSET, chunk=1 << 21):
    """oracle answer + certainty for the rays of `agents` (default all): {'dist', 'obj', 'certain', 'bound'} over
    [E, k, R].  certain: every decision the answer depends on clears its bound (the hit/miss and t decisions of the
    winner, the runner-up partner, every candidate that could take its place); bound: the float32 bound of the
    winner's distance (including the grazing term)."""
    pos = np.asarray(pos, np.float64)
    E, N, _ = pos.shape
    agents = np.arange(N) if agents is None else np.asarray(agents)
    s, u, ok = sensors.ray_frames(pos, quat, dirs, offset, body, agents)
    Rn = u.shape[2]
    out = {k: np.empty((E, len(agents), Rn)) for k in ('dist', 'bound')}
    out['obj'] = np.empty((E, len(agents), Rn), np.int64)
    out['certain'] = np.empty((E, len(agents), Rn), bool)
    q = np.asarray(quat, np.float64)[:, agents]
    p = pos[:, agents]
    off = np.asarray(offset, np.float64)
    if body:
        ex_s = np.all(q == ID, -1)[..., None] & _exact(p + off)
    else:
        ex_s = _exact(p + off)
    ds = np.where(np.all(ex_s, -1), 0.0, 8 * EPS * (np.linalg.norm(p, axis=-1) + 3 * np.linalg.norm(off)))   # [E,k]
    r2 = P.contact_radius ** 2
    step = max(1, chunk // max(1, E * Rn * N))
    for a0 in range(0, len(agents), step):
        sl = slice(a0, a0 + step)
        S, U, dS = s[:, sl], u[:, sl], ds[:, sl, None]
        t_g, h, tc, d2 = sensors.ray_candidates(pos, S, U, agents[sl], P)
        T = sensors.candidate_times(S, t_g, h, tc, d2, rng, P)
        k = np.argmin(T, axis=-1)
        best = np.take_along_axis(T, k[..., None], -1)[..., 0]
        # ---- agent candidates: t and its bound, certainly valid / invalid
        C = np.linalg.norm(pos[:, None, None, :, :] - S[:, :, None, None, :], axis=-1)
        own = ~np.isfinite(d2)
        d2f = np.where(own, 0.0, d2)
        dc = dS[..., None] + 2 * EPS * C
        dtc = dc + C * (DIR_ERR + 4 * EPS)
        dq = dc + dtc + np.abs(tc) * DIR_ERR + 4 * EPS * C
        bh = 2 * np.sqrt(d2f) * dq + dq * dq + 4 * EPS * d2f + 2 * EPS * r2
        mh = r2 - d2f
        ta = tc - np.sqrt(np.maximum(mh, 0.0))
        dta = dtc + bh / (2 * np.sqrt(np.maximum(mh, bh))) + 2 * EPS * np.abs(ta)
        fin_rng = rng if np.isfinite(rng) else np.inf
        a_valid = (mh > bh) & (ta > dta) & (fin_rng - ta > dta + EPS * (fin_rng if np.isfinite(fin_rng) else 0))
        a_invalid = own | (mh < -bh) | (ta < -dta) | (ta - fin_rng > dta)
        # ---- the ground
        gz = P.ground_z
        sz = S[:, :, None, 2]
        dz = U[..., 2]
        with np.errstate(invalid='ignore', divide='ignore'):
            dtg = (dS + 2 * EPS * np.abs(gz - sz)) / np.abs(dz) + np.where(np.isfinite(t_g), t_g, 0) * (DIR_ERR / np.abs(dz) + 2 * EPS)
            dh = dS + np.where(np.isfinite(t_g), t_g, 0) * DIR_ERR + dtg + 2 * EPS * np.abs(h[..., :2]).max(-1)
            box_m = BOX - np.abs(h[..., :2]).max(-1)
            start_m = sz - gz
            down = dz < 0
            g_valid = (down & (-dz > DIR_ERR) & ((start_m > dS) | ((dS == 0) & (start_m > 0))) & (box_m > dh)
                       & (fin_rng - t_g > dtg))
            # a ray within DIR_ERR of horizontal: whatever sign the kernel gives dz, a ground hit would lie beyond the box
            horizontal_far = (np.abs(dz) <= DIR_ERR) & (start_m > DIR_ERR * (2 * BOX + np.abs(S[:, :, None, :2]).max(-1)))
            below = (start_m < -dS) | ((dS == 0) & (start_m <= 0))
            g_invalid = ((dz > DIR_ERR) | horizontal_far | below
                         | (down & ((box_m < -dh) | (t_g - fin_rng > dtg))))
        tt = np.concatenate([np.where(np.isfinite(t_g), t_g, np.inf)[..., None], ta], -1)
        dt = np.concatenate([np.where(np.isfinite(dtg), dtg, np.inf)[..., None], dta], -1)
        valid = np.concatenate([g_valid[..., None], a_valid], -1)
        invalid = np.concatenate([g_invalid[..., None], a_invalid], -1)
        hit = np.isfinite(best)
        tw = np.take_along_axis(tt, k[..., None], -1)
        dtw = np.take_along_axis(dt, k[..., None], -1)
        others = np.ones_like(invalid)
        np.put_along_axis(others, k[..., None], False, -1)
        with np.errstate(invalid='ignore'):
            clear = invalid | (tt - tw > dt + dtw)                  # cannot take the winner's place
        win_ok = np.take_along_axis(valid, k[..., None], -1)[..., 0]
        certain = np.where(hit, win_ok & np.all(clear | ~others, -1), np.all(invalid, -1))
        certain |= ~ok[None, None, :]
        out['dist'][:, sl] = np.where(hit & ok, best, np.inf)
        out['obj'][:, sl] = np.where(hit & ok, np.where(k == 0, N, k - 1), -1)
        out['certain'][:, sl] = certain
        out['bound'][:, sl] = np.where(hit & ok, dtw[..., 0], 0.0)
    return out
