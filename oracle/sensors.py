"""TEST INFRASTRUCTURE -- CPU oracle of the analytic sensors (not product code).

Restates Object.collision / get_dist / raycast (/root/reference/mrsgym/Object.py:98-174) on the
primitives the B200 step uses for contact: ground = top face (z = ground_z, |x|,|y| <= 15) of the
30 x 30 x 1 box of plane.urdf:21-26, agents = CONTACT_RADIUS spheres (the spheres the step's pair rows use;
AGENT_RADIUS is only the spawn separation),
the quad's own ground gap = collision-cylinder support extent as in bullet_model.ground_contact.
PARITY UNPINNED against PyBullet: the reference answers these queries on Bullet's hull geometry
(getClosestPoints / rayTestBatch), which cannot be run here; this is the specification the kernels
are tested against.  float64 numpy, loops over rays are fine at test sizes.
"""
from __future__ import annotations

import numpy as np

from . import bullet_model as bm


def proximity(pos, quat, P: bm.PhysicsParams, threshold=0.04):
    """pos [E,N,3], quat [E,N,4] -> gap_agent [E,N], nearest [E,N], gap_ground [E,N], collision [E,N]"""
    pos = np.asarray(pos, np.float64)
    E, N, _ = pos.shape
    d = np.linalg.norm(pos[:, :, None, :] - pos[:, None, :, :], axis=-1)
    d[:, np.arange(N), np.arange(N)] = np.inf
    nearest = np.where(N > 1, d.argmin(axis=-1), -1)
    gap_agent = d.min(axis=-1) - 2.0 * P.contact_radius
    R22 = bm.quat_to_mat(np.asarray(quat, np.float64))[..., 2, 2]
    ext = P.col_radius * np.sqrt(np.maximum(1 - R22 * R22, 0)) + P.col_halfheight * np.abs(R22) + P.col_margin
    gap_ground = pos[..., 2] - ext - P.ground_z
    return gap_agent, nearest, gap_ground, (gap_agent < threshold) | (gap_ground < threshold)


def raycast(pos, quat, directions, offset, body, rng, P: bm.PhysicsParams):
    """-> dist [E,N,R] (inf = no hit), obj [E,N,R] (-1 none, N ground, j agent)"""
    pos = np.asarray(pos, np.float64)
    E, N, _ = pos.shape
    dirs = np.asarray(directions, np.float64).reshape(-1, 3)
    Rn = dirs.shape[0]
    Rm = bm.quat_to_mat(np.asarray(quat, np.float64))
    dist = np.full((E, N, Rn), np.inf)
    obj = np.full((E, N, Rn), -1, np.int64)
    off = np.asarray(offset, np.float64)
    for e in range(E):
        for i in range(N):
            for r in range(Rn):
                dvec, o = dirs[r], off
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
