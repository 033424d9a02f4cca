"""mrs_proximity / mrs_raycast and the torch helpers built on them against the sensor specification
(oracle/sensors.py through sensor_cases.py) at every size class of the kernels' indexing, at the edges of their
geometry and under non-default configurations.

Bars: ids, `nearest` and `collision` exactly equal wherever the decision clears its float32 bound; distances and gaps
within their bounds; the hand-built edge decisions are never excused (their certainty is checked here on the
assembled scene, and on the CPU by test_cpu_sensors.py)."""
import ctypes as C

import numpy as np
import pytest
import torch

import sensor_cases as SC

pytestmark = pytest.mark.gpu

F32 = np.float32
# (E, N, rays): 1 / 7 / 128 / 129 rays, N around the 32-agent warp boundary, E*N beyond one block and past 2^15
SHAPES = [(1, 1, 129), (3, 1, 7), (1, 2, 128), (7, 12, 129), (5, 31, 1), (4, 32, 128), (3, 33, 129), (2, 129, 7),
          (1, 1030, 128), (1, 4097, 129), (4101, 8, 129)]


def _subset(E, N, seed):
    """envs and agents compared: all of them at small shapes, else every case agent plus a seeded sample"""
    g = np.random.default_rng(seed)
    envs = np.arange(E)
    if E > 64:
        envs = np.unique(np.concatenate([np.arange(2 * len(SC.CASES)), g.choice(E, 48, replace=False), [E - 1]]))
    agents = np.arange(N)
    if N > 129:
        agents = np.unique(np.concatenate([np.arange(max(SC.case_sizes().values())), g.choice(N, 12, replace=False),
                                           [N - 1]]))
    return envs, agents


def _upload(sw, pos, quat):
    import helpers as H
    z = np.zeros(pos.shape, F32)
    H.upload_state(sw, dict(pos=pos, quat=quat, vel=z, angvel=z))


def check_proximity(sw, sc, P, thr, envs, agents, tag):
    got = sw.proximity(thr)
    w = SC.proximity_verdict(sc.pos[envs], sc.quat[envs], P, thr, agents)
    g = {k: t.cpu().numpy()[np.ix_(envs, agents)] for k, t in got.items()}
    bad = w['nearest_ok'] & (g['nearest'] != w['nearest'])
    assert not bad.any(), (tag, 'nearest', np.argwhere(bad)[:5])
    bad = w['collision_ok'] & (g['collision'] != w['collision'])
    assert not bad.any(), (tag, 'collision', np.argwhere(bad)[:5])
    fin = np.isfinite(w['gap_agent'])
    assert (np.isinf(g['gap_agent']) == ~fin).all() and not np.isnan(g['gap_agent']).any(), tag
    with np.errstate(invalid='ignore'):
        err = np.abs(g['gap_agent'] - w['gap_agent'])[fin]
    assert (err <= w['ga_bound'][fin]).all(), (tag, 'gap_agent', float((err / np.maximum(w['ga_bound'][fin], 1e-30)).max()))
    err = np.abs(g['gap_ground'] - w['gap_ground'])
    assert (err <= w['gg_bound']).all(), (tag, 'gap_ground worst error %.3g m' % err.max(),
                                          float((err / np.maximum(w['gg_bound'], 1e-30)).max()))
    pe = [(np.searchsorted(envs, e), np.searchsorted(agents, a)) for e, a in sc.prox_edges
          if e in envs and a in agents]
    for e, a in pe:       # hand-built: never excused
        assert w['nearest_ok'][e, a] and w['collision_ok'][e, a], (tag, sc.names[envs[e]], agents[a])


def check_rays(sw, sc, P, dirs, body, rng, envs, agents, tag):
    got = sw.raycast(torch.from_numpy(dirs).cuda(), SC.OFFSET, body, rng)
    d = got['dist'].cpu().numpy()[np.ix_(envs, agents)]
    o = got['object'].cpu().numpy()[np.ix_(envs, agents)]
    v = SC.ray_verdict(sc.pos[envs], sc.quat[envs], dirs, body, rng, P, agents)
    c = v['certain']
    assert not np.isnan(d).any(), tag
    wrong = c & (o != v['obj'])
    assert not wrong.any(), (tag, 'object', [(sc.names[envs[e]], agents[a], r, o[e, a, r], v['obj'][e, a, r])
                                             for e, a, r in np.argwhere(wrong)[:6]], int(wrong.sum()))
    hit = c & np.isfinite(v['dist'])
    with np.errstate(invalid='ignore'):
        err = np.abs(d - v['dist'])[hit]
    ratio = err / np.maximum(v['bound'][hit], 1e-30)
    assert (ratio <= 1.0).all(), (tag, 'dist: worst %.3g bars, worst error %.3g m' % (ratio.max(), err.max()))
    assert np.isinf(d[c & ~np.isfinite(v['dist'])]).all(), tag
    for e, a, r in sc.edges:
        if e in envs and a in agents and r < len(dirs):
            assert c[np.searchsorted(envs, e), np.searchsorted(agents, a), r], (tag, sc.names[e], a, r)


@pytest.mark.parametrize('E,N,R', SHAPES, ids=['%dx%d-r%d' % s for s in SHAPES])
def test_sensors_vs_oracle_at_every_shape(E, N, R):
    import mrsgym_b200 as M
    sw = M.Swarm(E, N, 0, 'set_speeds', M._abi.X_POS_VEL, want_A=False)
    envs, agents = _subset(E, N, E * 7919 + N)
    for cfg in SC.CONFIGS:
        SC.apply(sw, cfg)
        P, dirs = SC.phys(cfg), SC.directions(cfg, R)
        for p, names in enumerate(SC.passes(E, N)):
            for body, rng in SC.RAY_CALLS:
                sc = SC.scene(cfg, names, N, body, rng)
                _upload(sw, sc.pos, sc.quat)
                check_rays(sw, sc, P, dirs, body, rng, envs, agents, (cfg, p, body, rng))
            sc = SC.scene(cfg, names, N, False, 100.0)
            _upload(sw, sc.pos, sc.quat)
            for thr in (SC.THRESHOLD, SC.tie_threshold(cfg)):
                check_proximity(sw, sc, P, thr, envs, agents, (cfg, p, thr))
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------ torch helpers
def _pairs_scene(N, centre, seed, r):
    """N agents in pairs whose sphere gaps straddle 0.02 m, pairs 1 m apart, tilted up to 0.5 rad, near `centre`"""
    from scipy.spatial.transform import Rotation
    g = np.random.default_rng(seed)
    cols = int(np.ceil(np.sqrt(N / 2)))
    pos = np.zeros((N, 3))
    for k in range(0, N, 2):
        c = np.array([(k // 2) % cols, (k // 2) // cols, 0.0]) + centre
        n = SC._unit(g.normal(size=3))
        sep = 2 * r + g.uniform(-0.01, 0.05)
        pos[k] = c - 0.5 * sep * n
        if k + 1 < N:
            pos[k + 1] = c + 0.5 * sep * n
    quat = Rotation.from_rotvec(g.normal(size=(N, 3)) * 0.25).as_quat()
    return pos.astype(F32), quat.astype(F32)


def _contact_points_ref(pos, quat, P, thr, body):
    """Environment.get_contact_points restated in float64 numpy: slot 0 the nearest agent's sphere contact, slots 1-4
    the lower-rim points of the collision cylinder against the ground"""
    from oracle import bullet_model as bm
    from oracle import sensors
    pos = np.asarray(pos, np.float64)
    E, N, _ = pos.shape
    ga, ne, _, _ = sensors.proximity(pos, quat, P, thr)
    R = bm.quat_to_mat(np.asarray(quat, np.float64))
    c, _, gd = bm.ground_rim(pos, R, P)
    pj = np.take_along_axis(pos, np.maximum(ne, 0)[..., None].repeat(3, -1), 1)
    n = pos - pj
    n = n / np.maximum(np.linalg.norm(n, axis=-1, keepdims=True), 1e-12)
    P0 = pos - n * P.contact_radius
    Pw = pos[:, :, None] + np.einsum('enij,enpj->enpi', R, c)
    obj = np.concatenate([np.where((ne >= 0) & (ga < thr), ne, -1)[..., None], np.where(gd < thr, N, -1)], -1)
    Pt = np.concatenate([P0[:, :, None], Pw], 2)
    nrm = np.zeros((E, N, 5, 3))
    nrm[..., 0, :] = n
    nrm[..., 1:, 2] = 1.0
    if body:
        Pt = np.einsum('enji,enpj->enpi', R, Pt - pos[:, :, None])
        nrm = np.einsum('enji,enpj->enpi', R, nrm)
    return dict(object=obj, pos=Pt, normal=nrm, distance=np.concatenate([ga[..., None], gd], -1))


@pytest.mark.parametrize('N', [40, 300])
@pytest.mark.parametrize('cfg', ['r30', 'r06'])
def test_contact_points_and_closest_objects_vs_numpy(N, cfg):
    """get_contact_points (world and body frame) and get_closest_objects on a swarm near the ground at the origin and
    one 100 m away, against float64 numpy: decisions that clear their bound equal, gaps within float32 bounds"""
    import mrsgym_b200 as M
    from mrsgym_b200.env import Environment
    P = SC.phys(cfg)
    r = P.contact_radius
    pos, quat = zip(*[_pairs_scene(N, np.array(c), 11 + k, r) for k, c in enumerate([(-8.0, -8.0, 0.565), (100.0, -80.0, 40.0)])])
    pos, quat = np.stack(pos), np.stack(quat)
    sw = M.Swarm(2, N, 0, 'set_speeds', M._abi.X_POS_VEL, want_A=False)
    SC.apply(sw, cfg)
    _upload(sw, pos, quat)
    env = Environment(sw, False)
    thr = float(F32(P.contact_margin))
    v = SC.proximity_verdict(pos, quat, P, thr)
    # the helper forms world points pos + R c in float32 and body-frame ones from them: both carry the rounding of the
    # world coordinates, and a normal carries that of pos - pos_j over the partner distance
    scale = np.abs(pos).max(-1) + 1.0
    pos_tol = (32 * SC.EPS * scale)[..., None, None]
    nrm_tol = (8 * SC.EPS * scale / (v['gap_agent'] + 2 * r) + 8 * SC.EPS)[..., None, None]
    for body in (False, True):
        got = {k: t.cpu().numpy() for k, t in env.get_contact_points(body=body).items()}
        want = _contact_points_ref(pos, quat, P, thr, body)
        ok0 = v['collision_ok'] & (np.abs(v['ga_margin']) > v['ga_bound'])
        np.testing.assert_array_equal(got['object'][..., 0][ok0], want['object'][..., 0][ok0])
        gb = v['gg_bound'][..., None]
        okg = np.abs(want['distance'][..., 1:] - thr) > gb
        np.testing.assert_array_equal(got['object'][..., 1:][okg], want['object'][..., 1:][okg])
        assert (np.abs(got['distance'][..., 0] - want['distance'][..., 0]) <= v['ga_bound']).all()
        assert (np.abs(got['distance'][..., 1:] - want['distance'][..., 1:]) <= gb).all()
        err = np.abs(got['pos'] - want['pos'])
        assert (err <= pos_tol).all(), (body, float(err.max()), float((err / pos_tol).max()))
        err = np.abs(got['normal'] - want['normal'])[..., :1, :]
        assert (err <= nrm_tol).all(), (body, float(err.max()), float((err / nrm_tol).max()))
        assert (np.abs(got['normal'][..., 1:, :] - want['normal'][..., 1:, :]) <= 16 * SC.EPS).all()     # rows of R in float32
        assert (got['object'][..., 0] >= 0).any() and (got['object'][..., 1:] == N).any()
    radius = 0.02
    cl = {k: t.cpu().numpy() for k, t in env.get_closest_objects(radius).items()}
    p64 = pos.astype(np.float64)
    d = np.linalg.norm(p64[:, :, None] - p64[:, None], axis=-1)
    gap = d - 2 * r
    bound = 8 * SC.EPS * (d + 2 * r)
    err = np.abs(cl['gap'] - gap)
    assert (err <= bound).all(), 'get_closest_objects: worst gap error %.3g m (%.3g bars)' % (err.max(), (err / bound).max())
    mask = (gap < radius) & ~np.eye(N, dtype=bool)
    sure = np.abs(gap - radius) > bound
    np.testing.assert_array_equal(cl['mask'][sure], mask[sure])
    assert mask.any() and (~mask).any()


# ------------------------------------------------------------------------------ index range near 2^32
def test_ray_index_range_near_2_32():
    """E*N = 2^26 agents (N = 8) and 63 rays: E*N*R = 4.23e9 thread indices, checked on the first, a middle and the
    last env against the oracle; 64 rays (E*N*R = 2^32) are refused with MRS_ERR_UNSUPPORTED before any output is
    touched.  Full-size device buffers."""
    import mrsgym_b200 as M
    from mrsgym_b200 import _abi
    from mrsgym_b200.core import _ptr
    E, N = 1 << 23, 8
    S = E * N
    footprint = (_abi.STATE_PLANES + _abi.CTRL_PLANES) * S * 4 + 64 * S * 8
    free = torch.cuda.mem_get_info()[0]
    if free < footprint + (8 << 30):
        pytest.skip('needs %.1f GB of free device memory (%.1f GB free)' % ((footprint + (8 << 30)) / 1e9, free / 1e9))
    cfg = 'r06'
    P = SC.phys(cfg)
    sw = dist = obj = None
    try:
        sw = M.Swarm(E, N, 0, 'set_speeds', _abi.X_NONE, want_A=False)
        SC.apply(sw, cfg)
        sc = SC.scene(cfg, ['far', 'tolerance', 'box'], N, False, 100.0)
        base = sc.pos[1], sc.quat[1]
        for k in range(3):
            sw.state[k].view(E, N).copy_(torch.from_numpy(base[0][:, k].copy()).cuda().expand(E, N))
        for k in range(4):
            sw.state[3 + k].view(E, N).copy_(torch.from_numpy(base[1][:, k].copy()).cuda().expand(E, N))
        for e, src in ((0, 0), (E - 1, 2)):
            for k in range(3):
                sw.state[k, e * N:(e + 1) * N] = torch.from_numpy(sc.pos[src, :, k].copy()).cuda()
            for k in range(4):
                sw.state[3 + k, e * N:(e + 1) * N] = torch.from_numpy(sc.quat[src, :, k].copy()).cuda()
        dirs = torch.from_numpy(SC.directions(cfg, 64)).cuda()
        dist = torch.full((S * 64,), -7.5, dtype=torch.float32, device='cuda')
        obj = torch.full((S * 64,), -7, dtype=torch.int32, device='cuda')
        off = (C.c_float * 3)(*SC.OFFSET)
        rc = sw.lib.mrs_raycast(sw._cfg_ref, sw._bufs_ref, _ptr(dirs), 64, off, 0, 100.0, _ptr(dist), _ptr(obj),
                                sw._stream())
        assert rc == -3                                        # MRS_ERR_UNSUPPORTED
        torch.cuda.synchronize()
        for part in dist.split(1 << 28):
            assert bool((part == -7.5).all())
        for part in obj.split(1 << 28):
            assert bool((part == -7).all())
        R = 63
        _abi.check(sw.lib.mrs_raycast(sw._cfg_ref, sw._bufs_ref, _ptr(dirs), R, off, 0, 100.0, _ptr(dist), _ptr(obj),
                                      sw._stream()), 'mrs_raycast')
        torch.cuda.synchronize()
        assert bool((dist[S * R:S * R + (1 << 20)] == -7.5).all()) and bool((dist[-(1 << 20):] == -7.5).all())
        mid = E // 2
        rows = {0: 0, mid: 1, E - 1: 2}
        pos = np.stack([sc.pos[0], base[0], sc.pos[2]])
        quat = np.stack([sc.quat[0], base[1], sc.quat[2]])
        v = SC.ray_verdict(pos, quat, SC.directions(cfg, R), False, 100.0, P)
        for e, i in rows.items():
            lo = e * N * R
            d = dist[lo:lo + N * R].view(N, R).cpu().numpy().astype(np.float64)
            o = obj[lo:lo + N * R].view(N, R).cpu().numpy()
            c = v['certain'][i]
            assert (o == v['obj'][i])[c].all(), e
            hit = c & np.isfinite(v['dist'][i])
            with np.errstate(invalid='ignore'):            # inf - inf off the hits
                assert (np.abs(d - v['dist'][i])[hit] <= v['bound'][i][hit]).all(), e
        assert (v['obj'][0] >= 0).any() and (v['obj'][2] == N).any()
    finally:
        del sw, dist, obj
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
