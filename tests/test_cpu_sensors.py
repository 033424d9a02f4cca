"""The sensor specification (oracle/sensors.py) and its cases (sensor_cases.py) without a GPU:

- the vectorised oracle equals a literal loop restatement of the sensors;
- every hand-built decision clears its float32 bound, and the exact ties are exact;
- each case set lands far (10 bars, or a certain decision) from what a subtly wrong kernel computes;
- a float32 emulation of raycast_kernel / proximity_kernel stays inside the bars, while the |c|^2 - tc^2 form of the
  squared miss distance (the kernel before the perpendicular form) does not at far range.
"""
import dataclasses

import numpy as np
import pytest

import sensor_cases as SC
from oracle import bullet_model as bm
from oracle import sensors

F32 = np.float32
SHAPE_N = 16                         # every case fits; one env per case


def _scenes():
    """(cfg, scene, body, range, P, dirs) for every configuration and ray call at one env per case"""
    E = len(SC.CASES)
    for cfg in SC.CONFIGS:
        P, dirs = SC.phys(cfg), SC.directions(cfg)
        for body, rng in SC.RAY_CALLS:
            yield cfg, SC.scene(cfg, list(SC.CASES), SHAPE_N, body, rng), body, rng, P, dirs
    assert E == len(SC.passes(E, SHAPE_N)[0])


# ------------------------------------------------------------------------------ oracle vs its loop restatement
def loop_raycast(pos, quat, directions, offset, body, rng, P):
    """The sensors' rays one at a time (the statement the vectorised oracle must equal)."""
    pos = np.asarray(pos, np.float64)
    E, N, _ = pos.shape
    dirs = np.asarray(directions, np.float64).reshape(-1, 3)
    Rm = bm.quat_to_mat(np.asarray(quat, np.float64))
    dist = np.full((E, N, len(dirs)), np.inf)
    obj = np.full((E, N, len(dirs)), -1, np.int64)
    off = np.asarray(offset, np.float64)
    for e in range(E):
        for i in range(N):
            for r in range(len(dirs)):
                dvec, o = dirs[r], off
                big = np.max(np.abs(dvec))
                if not (np.all(np.isfinite(dvec)) and big > 0):
                    continue
                dvec = dvec / big
                if body:
                    dvec, o = Rm[e, i] @ dvec, Rm[e, i] @ off
                dvec = dvec / np.linalg.norm(dvec)
                s = pos[e, i] + o
                best, bid = rng, -1
                if dvec[2] < 0 and s[2] > P.ground_z:
                    t = (P.ground_z - s[2]) / dvec[2]
                    h = s + t * dvec
                    if t < best and abs(h[0]) <= 15 and abs(h[1]) <= 15:
                        best, bid = t, N
                for j in range(N):
                    if j == i:
                        continue
                    c = pos[e, j] - s
                    tc = c @ dvec
                    d2 = c @ c - tc * tc
                    if d2 > P.contact_radius ** 2:
                        continue
                    t = tc - np.sqrt(P.contact_radius ** 2 - d2)
                    if 0 <= t < best:
                        best, bid = t, j
                if bid >= 0:
                    dist[e, i, r], obj[e, i, r] = best, bid
    return dist, obj


@pytest.mark.parametrize('body,rng', [(False, 30.0), (True, 30.0), (True, float('inf'))])
def test_vectorised_raycast_equals_the_loop(body, rng):
    g = np.random.default_rng(3)
    E, N = 3, 7
    pos = (g.uniform(-4, 4, (E, N, 3)) + [0, 0, 3.0]).astype(F32)
    quat = g.normal(size=(E, N, 4))
    quat = (quat / np.linalg.norm(quat, axis=-1, keepdims=True)).astype(F32)
    dirs = SC.directions('r30', 24)
    P = bm.PhysicsParams(contact_radius=0.7)
    d0, o0 = loop_raycast(pos, quat, dirs, SC.OFFSET, body, rng, P)
    d1, o1 = sensors.raycast(pos, quat, dirs, SC.OFFSET, body, rng, P)
    np.testing.assert_array_equal(o1, o0)
    np.testing.assert_allclose(d1, d0, rtol=1e-12, atol=1e-12)
    assert (o0 == N).any() and ((o0 >= 0) & (o0 < N)).any() and (o0 == -1).any()
    sub = np.array([5, 1])
    d2, o2 = sensors.raycast(pos, quat, dirs, SC.OFFSET, body, rng, P, agents=sub)
    np.testing.assert_array_equal(o2, o0[:, sub])


def test_gap_ground_is_the_lowest_rim_point_of_the_step():
    """gap_ground = the smallest of the ground rows' gaps (bullet_model.ground_rim, used by solve_contacts) =
    z - r max(|R20|, |R21|) - h |R22| - margin - ground_z; about a diagonal axis it lies r (1 - 1/sqrt 2) sin(tilt)
    above the continuous support the sensors used before"""
    sc = SC.scene('r06', ['tilts'], 8, False, 100.0)
    P = SC.phys('r06')
    _, _, gg, _ = sensors.proximity(sc.pos, sc.quat, P)
    R = bm.quat_to_mat(sc.quat.astype(np.float64))
    want = (sc.pos[..., 2] - P.col_radius * np.maximum(np.abs(R[..., 2, 0]), np.abs(R[..., 2, 1]))
            - P.col_halfheight * np.abs(R[..., 2, 2]) - P.col_margin - P.ground_z)
    np.testing.assert_allclose(gg, want, atol=1e-15)
    R22 = R[..., 2, 2]
    cont = sc.pos[..., 2] - P.col_radius * np.sqrt(1 - R22 ** 2) - P.col_halfheight * np.abs(R22) - P.col_margin - P.ground_z
    tilt = np.arccos(np.clip(R22, -1, 1))[0, 3]               # 30 degrees about (1, 1, 0)
    assert gg[0, 3] - cont[0, 3] == pytest.approx(P.col_radius * (1 - 2 ** -0.5) * np.sin(tilt), rel=1e-6)


# ------------------------------------------------------------------------------ the cases themselves
def test_hand_built_decisions_clear_their_bounds():
    for cfg, sc, body, rng, P, dirs in _scenes():
        v = SC.ray_verdict(sc.pos, sc.quat, dirs, body, rng, P)
        bad = [(sc.names[e], a, r) for e, a, r in sc.edges if not v['certain'][e, a, r]]
        assert not bad, (cfg, body, bad)
        assert v['certain'].mean() > 0.99, (cfg, body, v['certain'].mean())
        hit = np.isfinite(v['dist'])
        assert (v['obj'] == SHAPE_N).any() and (v['obj'][hit] < SHAPE_N).any() and (~hit).any()
        for thr in (SC.THRESHOLD, SC.tie_threshold(cfg)):
            p = SC.proximity_verdict(sc.pos, sc.quat, P, thr)
            bad = [(sc.names[e], a) for e, a in sc.prox_edges if not (p['nearest_ok'][e, a] and p['collision_ok'][e, a])]
            assert not bad, (cfg, thr, bad)


def test_exact_ties_are_exact():
    """lattice and coincident ties, gap_agent == threshold and gap_ground == threshold hold in float32 arithmetic with
    no rounding at all (bound 0), so the kernel must break them exactly as the specification does"""
    names = list(SC.CASES)
    sc = SC.scene('moved', names, SHAPE_N, False, 100.0)
    p = SC.proximity_verdict(sc.pos, sc.quat, SC.phys('moved'), SC.tie_threshold('moved'))
    lat, tie, coi = names.index('lattice'), names.index('tie'), names.index('coincident')
    assert (p['ga_bound'][lat, :8] == 0).all() and list(p['nearest'][lat, :8]) == [1, 0, 0, 1, 0, 1, 2, 3]
    assert p['nearest'][coi, 0] == 2 and p['nearest'][coi, 2] == 0 and p['nearest'][coi, 1] == 0
    assert p['ga_margin'][tie, 0] == 0 and p['ga_bound'][tie, 0] == 0 and not p['collision'][tie, 0]
    assert p['gg_margin'][tie, 2] == 0 and p['gg_bound'][tie, 2] == 0 and not p['collision'][tie, 2]
    lone = SC.scene('r30', ['lone'], 1, False, 100.0)
    q = SC.proximity_verdict(lone.pos, lone.quat, SC.phys('r30'), SC.THRESHOLD)
    assert q['nearest'][0, 0] == -1 and np.isinf(q['gap_agent'][0, 0])


def test_every_sensor_field_is_varied():
    for k, v in SC.SENSOR_FIELDS.items():
        assert any(SC.fields(cfg)[k] != float(F32(v)) for cfg in SC.CONFIGS), k
        assert hasattr(bm.PhysicsParams(), k)


def test_directions_cover_the_edges():
    d = SC.directions('r30')
    assert len(d) == 129 and not np.isfinite(d[6]).all() and not d[5].any()
    assert np.abs(d[3]).max() < 1e-29 and np.abs(d[4]).max() > 1e29
    assert d[2][2] == 0 and d[7][2] == -2.0 ** -23 and abs(np.linalg.norm(d[0]) - 2.5) < 1e-6


# ------------------------------------------------------------------------------ subtly wrong kernels
RAY_MUTANTS = ['agent_radius', 'unbounded_ground', 'offset_unrotated', 'unnormalised_t', 'dropped_t_ge0', 'last_hit',
               'ground_z_ignored']
PROX_MUTANTS = ['agent_radius', 'ground_z_ignored', 'abs_R22_dropped', 'continuous_support', 'last_index_ties',
                'le_threshold']


def mutant_raycast(pos, quat, dirs, body, rng, P, mut):
    """the oracle's rays with one defect"""
    pos = np.asarray(pos, np.float64)
    N = pos.shape[1]
    if mut == 'agent_radius':
        P = dataclasses.replace(P, contact_radius=P.agent_radius)
    if mut == 'ground_z_ignored':
        P = dataclasses.replace(P, ground_z=0.0)
    s, u, ok = sensors.ray_frames(pos, quat, dirs, SC.OFFSET, body)
    if mut == 'offset_unrotated':
        s = pos + np.asarray(SC.OFFSET)
    t_g, h, tc, d2 = sensors.ray_candidates(pos, s, u, np.arange(N), P)
    if mut == 'unbounded_ground':
        h = np.zeros_like(h)
    tmin = -1.0 if mut == 'dropped_t_ge0' else 0.0
    r2 = P.contact_radius ** 2
    g = np.where((t_g < rng) & (np.abs(h[..., 0]) <= 15) & (np.abs(h[..., 1]) <= 15), t_g, np.inf)
    with np.errstate(invalid='ignore'):
        t = tc - np.sqrt(np.maximum(r2 - d2, 0.0))
    t = np.where((d2 <= r2) & (t > tmin if tmin < 0 else t >= 0) & (t < rng), t, np.inf)
    T = np.concatenate([g[..., None], t], -1)
    if mut == 'last_hit':
        k = np.argmax(np.where(np.isfinite(T), T, -np.inf), -1)
    else:
        k = np.argmin(T, -1)
    best = np.take_along_axis(T, k[..., None], -1)[..., 0]
    hit = np.isfinite(best) & ok
    dist = np.where(hit, best, np.inf)
    if mut == 'unnormalised_t':                      # t along the raw (rotated) direction instead of the unit one
        raw = np.linalg.norm(np.nan_to_num(np.asarray(dirs, np.float64), posinf=0, neginf=0), axis=-1)
        dist = dist / np.where(raw > 0, raw, 1.0)
    return dist, np.where(hit, np.where(k == 0, N, k - 1), -1)


def mutant_proximity(pos, quat, P, thr, mut):
    pos = np.asarray(pos, np.float64)
    E, N, _ = pos.shape
    thr = float(F32(thr))
    if mut == 'ground_z_ignored':
        P = dataclasses.replace(P, ground_z=0.0)
    rc = P.agent_radius if mut == 'agent_radius' else P.contact_radius
    d = np.linalg.norm(pos[:, :, None] - pos[:, None], axis=-1)
    d[:, np.arange(N), np.arange(N)] = np.inf
    if mut == 'last_index_ties':
        ne = N - 1 - np.argmin(d[..., ::-1], -1)
    else:
        ne = d.argmin(-1)
    ne = np.where(N > 1, ne, -1)
    ga = d.min(-1) - 2 * rc
    R = bm.quat_to_mat(np.asarray(quat, np.float64))
    R20, R21, R22 = R[..., 2, 0], R[..., 2, 1], R[..., 2, 2]
    side = P.col_radius * (np.sqrt(np.maximum(1 - R22 ** 2, 0)) if mut == 'continuous_support'
                           else np.maximum(np.abs(R20), np.abs(R21)))
    ext = side + P.col_halfheight * (R22 if mut == 'abs_R22_dropped' else np.abs(R22)) + P.col_margin
    gg = pos[..., 2] - ext - P.ground_z
    co = ((ga <= thr) | (gg <= thr)) if mut == 'le_threshold' else ((ga < thr) | (gg < thr))
    return ga, ne, gg, co


def _ray_caught(v, dist, obj):
    c = v['certain']
    flip = c & (obj != v['obj'])
    same = c & (obj == v['obj']) & np.isfinite(v['dist'])
    with np.errstate(invalid='ignore'):
        far = same & (np.abs(dist - v['dist']) > np.maximum(10 * v['bound'], 0)) & (dist != v['dist'])
    return int(flip.sum()), int(far.sum())


@pytest.mark.parametrize('mut', RAY_MUTANTS)
def test_rays_catch_a_subtly_wrong_kernel(mut):
    caught = {}
    for cfg, sc, body, rng, P, dirs in _scenes():
        v = SC.ray_verdict(sc.pos, sc.quat, dirs, body, rng, P)
        dist, obj = mutant_raycast(sc.pos, sc.quat, dirs, body, rng, P, mut)
        flips, far = _ray_caught(v, dist, obj)
        caught[(cfg, body)] = (flips, far)
    assert any(f + d > 0 for f, d in caught.values()), caught


@pytest.mark.parametrize('mut', PROX_MUTANTS)
def test_proximity_catches_a_subtly_wrong_kernel(mut):
    caught = {}
    for cfg in SC.CONFIGS:
        sc = SC.scene(cfg, list(SC.CASES), SHAPE_N, False, 100.0)
        P = SC.phys(cfg)
        for thr in (SC.THRESHOLD, SC.tie_threshold(cfg)):
            v = SC.proximity_verdict(sc.pos, sc.quat, P, thr)
            ga, ne, gg, co = mutant_proximity(sc.pos, sc.quat, P, thr, mut)
            n = int((v['nearest_ok'] & (ne != v['nearest'])).sum()) + int((v['collision_ok'] & (co != v['collision'])).sum())
            with np.errstate(invalid='ignore'):
                n += int(((np.abs(ga - v['gap_agent']) > 10 * v['ga_bound']) & (ga != v['gap_agent'])).sum())
                n += int(((np.abs(gg - v['gap_ground']) > 10 * v['gg_bound']) & (gg != v['gap_ground'])).sum())
            caught[(cfg, thr)] = n
    assert any(caught.values()), caught


# ------------------------------------------------------------------------------ float32 emulation of the kernels
class Arith:
    """float32 arithmetic of nvcc's output, with (fma=True) or without contraction of a * b + c"""

    def __init__(self, fma):
        self.fma = fma

    def mad(self, a, b, c):
        if self.fma:
            return (np.asarray(a, np.float64) * np.asarray(b, np.float64) + np.asarray(c, np.float64)).astype(F32)
        return F32(a) * F32(b) + F32(c) if np.isscalar(a) and np.isscalar(b) else a * b + c

    def dot(self, ax, ay, az, bx, by, bz):
        return self.mad(az, bz, self.mad(ay, by, ax * bx))


def _mat(q, A):
    x, y, z, w = (q[..., k] for k in range(4))
    one, two = F32(1), F32(2)
    return [one - two * A.mad(z, z, y * y), two * A.mad(-z, w, x * y), two * A.mad(y, w, x * z),
            two * A.mad(z, w, x * y), one - two * A.mad(z, z, x * x), two * A.mad(-x, w, y * z),
            two * A.mad(-y, w, x * z), two * A.mad(x, w, y * z), one - two * A.mad(y, y, x * x)]


def emulate_raycast(pos, quat, dirs, body, rng, P, form='perp', fma=True):
    """raycast_kernel in numpy float32, over [E, N, R] (rsqrtf as a correctly rounded 1/sqrt)"""
    A = Arith(fma)
    pos, quat, dirs = (np.asarray(x, F32) for x in (pos, quat, dirs))
    E, N, _ = pos.shape
    gz, rc = F32(P.ground_z), F32(P.contact_radius)
    with np.errstate(all='ignore'):
        big = np.max(np.abs(dirs), -1)
        ok = (big > 0) & np.all(np.isfinite(dirs), -1)
        d = dirs / np.where(ok, big, F32(1))[:, None]
        dx, dy, dz = (np.broadcast_to(d[:, k], (E, N, len(d))) for k in range(3))
        ox, oy, oz = (np.full((E, N, 1), F32(v)) for v in SC.OFFSET)
        if body:
            R = [m[..., None] for m in _mat(quat, A)]
            dx, dy, dz = (A.dot(R[3 * i], R[3 * i + 1], R[3 * i + 2], dx, dy, dz) for i in range(3))
            ox, oy, oz = (A.dot(R[3 * i], R[3 * i + 1], R[3 * i + 2], ox, oy, oz) for i in range(3))
        inv = (1.0 / np.sqrt(A.dot(dx, dy, dz, dx, dy, dz).astype(np.float64))).astype(F32)
        dx, dy, dz = dx * inv, dy * inv, dz * inv
        sx, sy, sz = ox + pos[..., 0:1], oy + pos[..., 1:2], oz + pos[..., 2:3]
        best = np.full((E, N, len(d)), F32(rng))
        idx = np.full((E, N, len(d)), -1)
        tg = (gz - sz) / dz
        hx, hy = A.mad(tg, dx, sx), A.mad(tg, dy, sy)
        g = (dz < 0) & (sz > gz) & (tg < best) & (np.abs(hx) <= 15) & (np.abs(hy) <= 15)
        best, idx = np.where(g, tg, best), np.where(g, N, idx)
        rad2 = rc * rc
        for j in range(N):
            cx, cy, cz = (pos[:, j:j + 1, k:k + 1] - s for k, s in enumerate((sx, sy, sz)))
            tc = A.dot(cx, cy, cz, dx, dy, dz)
            if form == 'perp':
                ex, ey, ez = A.mad(-tc, dx, cx), A.mad(-tc, dy, cy), A.mad(-tc, dz, cz)
                d2 = A.dot(ex, ey, ez, ex, ey, ez)
            else:                                       # the form before: |c|^2 - tc^2
                d2 = A.mad(-tc, tc, A.dot(cx, cy, cz, cx, cy, cz))
            t = tc - np.sqrt(rad2 - d2)
            take = (d2 <= rad2) & (t >= 0) & (t < best) & (np.arange(N) != j)[None, :, None]
            best, idx = np.where(take, t, best), np.where(take, j, idx)
    hit = (idx >= 0) & ok
    return np.where(hit, best, np.inf).astype(np.float64), np.where(hit, idx, -1)


def emulate_proximity(pos, quat, P, thr, fma=True):
    A = Arith(fma)
    pos, quat = np.asarray(pos, F32), np.asarray(quat, F32)
    E, N, _ = pos.shape
    dif = pos[:, :, None] - pos[:, None]
    d2 = A.dot(*(dif[..., k] for k in range(3)), *(dif[..., k] for k in range(3)))
    d2[:, np.arange(N), np.arange(N)] = np.inf
    ne = np.where(N > 1, d2.argmin(-1), -1)
    ga = np.sqrt(d2.min(-1)) - F32(2) * F32(P.contact_radius)
    R = _mat(quat, A)
    ext = A.mad(F32(P.col_halfheight), np.abs(R[8]), F32(P.col_radius) * np.maximum(np.abs(R[6]), np.abs(R[7])))
    ext = ext + F32(P.col_margin)
    gg = pos[..., 2] - ext - F32(P.ground_z)
    return ga.astype(np.float64), ne, gg.astype(np.float64), (ga < F32(thr)) | (gg < F32(thr))


def _ray_misses(v, dist, obj):
    """certain rays where the emulation disagrees with the verdict, and the worst distance error in bounds"""
    c = v['certain']
    wrong = c & (obj != v['obj'])
    both = c & (obj == v['obj']) & np.isfinite(v['dist'])
    ratio = np.abs(dist - v['dist'])[both] / np.maximum(v['bound'][both], 1e-300)
    return int(wrong.sum()), float(ratio.max()) if ratio.size else 0.0


@pytest.mark.parametrize('fma', [True, False])
def test_emulated_kernels_stay_inside_the_bars(fma):
    """The arithmetic of the fixed kernels, rounded in float32 as the GPU rounds it, agrees with the specification
    on every certain decision and stays within every distance bound, at every case and configuration."""
    for cfg, sc, body, rng, P, dirs in _scenes():
        v = SC.ray_verdict(sc.pos, sc.quat, dirs, body, rng, P)
        wrong, worst = _ray_misses(v, *emulate_raycast(sc.pos, sc.quat, dirs, body, rng, P, 'perp', fma))
        assert wrong == 0 and worst <= 1.0, (cfg, body, wrong, worst)
        for thr in (SC.THRESHOLD, SC.tie_threshold(cfg)):
            p = SC.proximity_verdict(sc.pos, sc.quat, P, thr)
            ga, ne, gg, co = emulate_proximity(sc.pos, sc.quat, P, thr, fma)
            assert (ne == p['nearest'])[p['nearest_ok']].all() and (co == p['collision'])[p['collision_ok']].all()
            fin = np.isfinite(p['gap_agent'])
            assert (np.abs(ga - p['gap_agent'])[fin] <= p['ga_bound'][fin]).all(), cfg
            assert (np.abs(gg - p['gap_ground']) <= p['gg_bound']).all(), cfg
            assert (np.isinf(ga) == ~fin).all()


@pytest.mark.parametrize('fma', [True, False])
def test_cancelling_miss_distance_fails_the_bars_at_far_range(fma):
    """|c|^2 - tc^2 loses the squared miss distance to cancellation at 30 - 99 m: the bars of the far cases catch it
    (decisions flip or distances leave their bounds), while the perpendicular form stays inside them."""
    out = {}
    for cfg in ('r06', 'r30'):
        sc = SC.scene(cfg, ['far'] * 4, 4, False, 100.0)
        P, dirs = SC.phys(cfg), SC.directions(cfg)
        v = SC.ray_verdict(sc.pos, sc.quat, dirs, False, 100.0, P)
        out[cfg] = {form: _ray_misses(v, *emulate_raycast(sc.pos, sc.quat, dirs, False, 100.0, P, form, fma))
                    for form in ('cancel', 'perp')}
    for cfg, r in out.items():
        assert r['perp'][0] == 0 and r['perp'][1] <= 1.0, out
    wrong, worst = out['r06']['cancel']
    assert wrong > 0 or worst > 1.0, out
