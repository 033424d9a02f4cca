"""TEST INFRASTRUCTURE -- CPU oracle of the analytic sensors (not product code).

Restates Object.collision / get_dist / raycast (/root/reference/mrsgym/Object.py:98-174) on the
primitives the B200 step uses for contact: ground = top face (z = ground_z, |x|,|y| <= 15) of the
30 x 30 x 1 box of plane.urdf:21-26, agents = CONTACT_RADIUS spheres (the spheres the step's pair rows use;
AGENT_RADIUS is only the spawn separation), the quad's own ground gap = the lowest of the four rim points of the
step's ground rows (bullet_model.ground_rim, the code solve_contacts uses).
PARITY UNPINNED against PyBullet: the reference answers these queries on Bullet's hull geometry
(getClosestPoints / rayTestBatch), which cannot be run here; this is the specification the kernels
are tested against.  float64 numpy, vectorised over partners and rays.

Ray semantics: a direction counts by its orientation only (any finite nonzero magnitude gives the result of its
unit vector); a zero or non-finite direction hits nothing.  A ray starts at position + offset (offset and
direction rotated by the agent's orientation with body=True) and reports the first of: the ground face when the
ray points down from above it and meets it inside the box, and agent spheres met at t >= 0, all at t < range.
Ties go to the ground, then to the lowest agent index.
"""
from __future__ import annotations

import numpy as np

from . import bullet_model as bm


def proximity(pos, quat, P: bm.PhysicsParams, threshold=0.04, agents=None):
    """pos [E,N,3], quat [E,N,4] -> gap_agent [E,k], nearest [E,k], gap_ground [E,k], collision [E,k] of `agents`
    (default all N)"""
    pos = np.asarray(pos, np.float64)
    E, N, _ = pos.shape
    agents = np.arange(N) if agents is None else np.asarray(agents)
    d = np.linalg.norm(pos[:, agents, None, :] - pos[:, None, :, :], axis=-1)
    d[:, np.arange(len(agents)), agents] = np.inf
    nearest = np.where(N > 1, d.argmin(axis=-1), -1)
    gap_agent = d.min(axis=-1) - 2.0 * P.contact_radius
    gap_ground = ground_rim_gaps(pos[:, agents], np.asarray(quat)[:, agents], P).min(axis=-1)
    return gap_agent, nearest, gap_ground, (gap_agent < threshold) | (gap_ground < threshold)


def ground_rim_gaps(pos, quat, P: bm.PhysicsParams):
    """gap of each of the four lower-rim points of the collision cylinder to the ground [E,N,4]"""
    pos = np.asarray(pos, np.float64)
    return bm.ground_rim(pos, bm.quat_to_mat(np.asarray(quat, np.float64)), P)[2]


def unit_directions(directions):
    """[R,3] -> (unit float64 directions [R,3] (zero where not usable), usable [R] bool)"""
    d = np.asarray(directions, np.float64).reshape(-1, 3)
    big = np.max(np.abs(d), axis=-1)
    ok = np.all(np.isfinite(d), axis=-1) & (big > 0)
    with np.errstate(invalid='ignore', divide='ignore'):
        u = d / np.where(ok, big, 1.0)[:, None]
        u = u / np.linalg.norm(u, axis=-1, keepdims=True)
    return np.where(ok[:, None], u, 0.0), ok


def ray_frames(pos, quat, directions, offset, body, agents=None):
    """starts s [E,k,3] and unit directions u [E,k,R,3] of the rays of agents (default all), usable [R]"""
    pos = np.asarray(pos, np.float64)
    agents = np.arange(pos.shape[1]) if agents is None else np.asarray(agents)
    u, ok = unit_directions(directions)
    off = np.asarray(offset, np.float64)
    p = pos[:, agents]
    if body:
        Rm = bm.quat_to_mat(np.asarray(quat, np.float64)[:, agents])
        s = p + np.einsum('ekij,j->eki', Rm, off)
        u = np.einsum('ekij,rj->ekri', Rm, u)
        u = u / np.where(ok[:, None], np.linalg.norm(u, axis=-1, keepdims=True), 1.0)
    else:
        s = p + off
        u = np.broadcast_to(u, p.shape[:2] + u.shape).copy()
    return s, u, ok


def ray_candidates(pos, s, u, agents, P: bm.PhysicsParams):
    """Every candidate of every ray: the ground (t_g [E,k,R] and the hit point h [E,k,R,3], t_g = inf when the ray
    does not point down from above the ground) and every agent sphere (tc = closest approach along the ray and
    d2 = squared miss distance, [E,k,R,N]).  The own agent of a ray has d2 = inf."""
    pos = np.asarray(pos, np.float64)
    dz = u[..., 2]
    down = (dz < 0) & (s[:, :, None, 2] > P.ground_z)
    with np.errstate(invalid='ignore', divide='ignore'):
        t_g = np.where(down, (P.ground_z - s[:, :, None, 2]) / np.where(down, dz, -1.0), np.inf)
        h = s[:, :, None, :] + np.where(down, t_g, 0.0)[..., None] * u
    c = pos[:, None, None, :, :] - s[:, :, None, None, :]                  # [E,k,1,N,3]
    tc = np.einsum('ekrnj,ekrj->ekrn', np.broadcast_to(c, u.shape[:3] + c.shape[3:]), u)
    q = c - tc[..., None] * u[:, :, :, None, :]
    d2 = np.sum(q * q, axis=-1)
    d2[:, np.arange(len(agents)), :, np.asarray(agents)] = np.inf
    return t_g, h, tc, d2


def candidate_times(s, t_g, h, tc, d2, rng, P: bm.PhysicsParams):
    """hit time of every candidate, inf where it is not hit within range: [E,k,R,1+N] (column 0 = the ground)"""
    r2 = P.contact_radius ** 2
    g = np.where((t_g < rng) & (np.abs(h[..., 0]) <= 15) & (np.abs(h[..., 1]) <= 15), t_g, np.inf)
    with np.errstate(invalid='ignore'):
        t = tc - np.sqrt(np.maximum(r2 - d2, 0.0))
    t = np.where((d2 <= r2) & (t >= 0) & (t < rng), t, np.inf)
    return np.concatenate([g[..., None], t], axis=-1)


def raycast(pos, quat, directions, offset, body, rng, P: bm.PhysicsParams, agents=None, chunk=1 << 22):
    """-> dist [E,k,R] (inf = no hit), obj [E,k,R] (-1 none, N ground, j agent) for the rays of `agents`
    (default all N)"""
    pos = np.asarray(pos, np.float64)
    E, N, _ = pos.shape
    agents = np.arange(N) if agents is None else np.asarray(agents)
    s, u, ok = ray_frames(pos, quat, directions, offset, body, agents)
    Rn = u.shape[2]
    dist = np.full((E, len(agents), Rn), np.inf)
    obj = np.full((E, len(agents), Rn), -1, np.int64)
    step = max(1, chunk // max(1, E * Rn * N))
    for a0 in range(0, len(agents), step):
        sl = slice(a0, a0 + step)
        T = candidate_times(s[:, sl], *ray_candidates(pos, s[:, sl], u[:, sl], agents[sl], P), rng, P)
        k = np.argmin(T, axis=-1)                              # first occurrence: ground, then the lowest index
        best = np.take_along_axis(T, k[..., None], -1)[..., 0]
        hit = np.isfinite(best) & ok
        dist[:, sl] = np.where(hit, best, np.inf)
        obj[:, sl] = np.where(hit, np.where(k == 0, N, k - 1), -1)
    return dist, obj
