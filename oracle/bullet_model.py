"""TEST INFRASTRUCTURE -- CPU oracle, not product code.

float64 numpy restatement of what ``p.stepSimulation()`` does to the
``'simple'`` mrs-gym scene (N x cf2x.urdf multibodies + plane.urdf), i.e. the
call at /root/reference/mrsgym/BulletSim.py:46-47.

The arithmetic lives in the third-party ``pybullet`` wheel (Bullet3 C++,
``btMultiBodyDynamicsWorld``).  It is NOT vendored under /root/reference and is
un-pinned (reference setup.py:5 ``install_requires=[..., 'pybullet', ...]``; the
shipped .pyc files are cpython-37 => pybullet 3.0-3.1 era).  pybullet is not
installable here (no network) so this file restates Bullet's published
algorithm from the bullet3 sources as recalled:

  btMultiBodyDynamicsWorld::solveConstraints         gravity -> ABA -> v += dt*a
  btMultiBody::computeAccelerationsArticulatedBody…  damping 0.04, gyro term
  btMultiBody::applyDeltaVeeMultiDof                 +-100 coordinate clamp
  btMultiBodyConstraintSolver::setupMultiBodyContactConstraint   erp2 / slop rhs
  btMultiBody::stepPositionsMultiDof                 p += dt*v, exp-map quaternion
  URDF2Bullet / btCompoundShape::calculateLocalInertia   AABB box inertia

PARITY UNPINNED for this file: the reference holds no tests / golden vectors
and real PyBullet cannot be run here.  Every constant is a field of
``PhysicsParams`` (loadable from the JSON that tools/pin_bullet.py writes when a real
pybullet is importable) so a pinned run can correct it without code changes.

Contact (SURVEY.md §8a-P item 4) is a velocity-level sequential-impulse solver, restitution 0,
Baumgarte push-out erp2, ``solver_iters`` Gauss-Seidel sweeps with early exit below
``solver_tol``, mirrored row for row by the CUDA kernels:
  * ground: the collision cylinder touches the ground box with up to four points of its lower
    rim (Bullet keeps <= 4 manifold points); each point is a normal row applied AT the point, so a
    tilted landing produces a righting torque; two Coulomb friction rows (world x, y) at the CoM,
    each bounded by mu_ground * (sum of the agent's normal impulses);
  * agent-agent: the north star's CONTACT_RADIUS sphere-sphere simplification of the hull
    contact: central normal row + two Coulomb friction rows (mu_agent) on the CoM velocities (the
    proxy sphere carries no rotational coupling);
  * sweep order: all ground rows (point 0..3 normal, then friction x, y), then the pair rows in
    round-robin-tournament order (round r pairs i with (2r - i) mod (M-1); rows of one round touch
    disjoint bodies, so they can be processed in parallel without changing the result).

All arrays are ``[..., 3]`` / ``[..., 4]`` (quaternion order xyzw, as PyBullet)
with arbitrary leading batch dims; agent-agent contact couples the second to
last axis (``[..., N, 3]``).
"""
from __future__ import annotations

import dataclasses
import math

import numpy as np


@dataclasses.dataclass
class QuadParams:
    """cf2x.urdf constants (/root/reference/mrsgym/models/cf2x.urdf:5,11-12,31-36,42-78)
    and the derived ones of Quadcopter.calculate_parameters
    (/root/reference/mrsgym/Quadcopter.py:153-168)."""
    mass: float = 0.027
    arm: float = 0.0397
    kf: float = 3.16e-10
    km: float = 7.94e-12
    thrust2weight: float = 2.25
    ixx: float = 1.4e-5          # file inertia: used by set_control only
    iyy: float = 1.4e-5
    izz: float = 2.17e-5
    gnd_eff_coeff: float = 11.36859
    prop_radius: float = 2.31348e-2
    drag_xy: float = 9.1785e-7
    drag_z: float = 10.311e-7
    dw1: float = 2267.18
    dw2: float = 0.16
    dw3: float = -0.11
    col_radius: float = 0.06
    col_length: float = 0.025
    # prop link CoM offsets, cf2x.urdf:42,54,66,78
    prop_xy: tuple = ((0.028, 0.028), (-0.028, 0.028), (-0.028, -0.028), (0.028, -0.028))
    # QuadControl gains (/root/reference/mrsgym/QuadControl.py:14-32)
    pos_p: float = 1.5
    pos_i: float = 0.001
    pos_d: float = 1.0
    vel_p: float = 3.0
    vel_i: float = 0.1
    vel_d: float = 1.0
    ori_p: tuple = (70000.0, 70000.0, 60000.0)
    ori_i: tuple = (0.0, 0.0, 500.0)
    ori_d: tuple = (20000.0, 20000.0, 12000.0)
    min_pwm: float = 20000.0
    max_pwm: float = 65535.0
    pwm2rpm_a: float = 0.2685
    pwm2rpm_b: float = 4070.3
    ctrl_dt: float = 0.01        # QuadControl always uses DefaultSim (QuadControl.py:10)
    ctrl_gravity: float = 9.81

    def derived(self, gravity: float = 9.81) -> dict:
        g = gravity * self.mass
        max_rpm = math.sqrt(self.thrust2weight * g / (4 * self.kf))
        max_thrust = 4.0 * self.kf * max_rpm ** 2
        hclip = 0.25 * self.prop_radius * math.sqrt(
            (15 * max_rpm ** 2 * self.kf * self.gnd_eff_coeff) / max_thrust)
        return dict(GravityForce=g, HoverRPM=math.sqrt(g / (4 * self.kf)), MaxRPM=max_rpm,
                    MaxThrust=max_thrust, GroundEffectHClip=hclip)


@dataclasses.dataclass
class PhysicsParams:
    """Bullet-side constants.  [Bullet, unverified] unless noted."""
    mass: float = 0.027
    # collision AABB half extents used for the default (no URDF_USE_INERTIA_FROM_FILE)
    # inertia: cylinder hull r=.06, half-length .0125; margins: hull recalcLocalAabb
    # (+.001) + btTransformAabb (+.001) + compound getAabb (+.001) => 3 margins.
    inertia_margins: int = 3
    col_margin: float = 0.001
    col_radius: float = 0.06
    col_halfheight: float = 0.0125
    lin_damping: float = 0.04
    ang_damping: float = 0.04
    max_coord_vel: float = 100.0
    gyro: bool = True
    ang_motion_threshold: float = 0.25 * math.pi
    # contact solver (PhysicsServerCommandProcessor defaults)
    erp2: float = 0.08
    slop: float = 1e-5
    contact_margin: float = 0.02     # contact breaking threshold: speculative contacts
    mu_ground: float = 0.75          # plane 1.5 (plane.urdf:4-6) x link default 0.5
    ground_z: float = 0.5            # plane.urdf:21-26 box 30x30x1 centred at z=0
    mu_agent: float = 0.25           # quad-quad: link default 0.5 x 0.5
    ground_contact: bool = True
    agent_contact: bool = True
    agent_radius: float = 0.3        # MRS.AGENT_RADIUS (/root/reference/mrsgym/MRS.py:28): spawn separation
    contact_radius: float = 0.3      # radius of the agent-agent contact sphere (north star: = AGENT_RADIUS;
                                     # 0.06 gives the size of the reference's cf2x collision cylinder)
    solver_iters: int = 50           # Bullet numSolverIterations
    solver_tol: float = 1e-6         # early exit: largest change of a row's contact-point velocity in a sweep [m/s]

    @classmethod
    def from_json(cls, path):
        """PhysicsParams from the JSON tools/pin_bullet.py writes (unknown keys are ignored)."""
        import json
        d = json.load(open(path))
        d = d.get('PhysicsParams', d)
        known = {f.name for f in dataclasses.fields(cls)}
        return cls(**{k: v for k, v in d.items() if k in known})

    def inertia_diag(self) -> np.ndarray:
        hx = self.col_radius + self.inertia_margins * self.col_margin
        hz = self.col_halfheight + self.inertia_margins * self.col_margin
        lx, lz = 2 * hx, 2 * hz
        return np.array([self.mass / 12.0 * (lx * lx + lz * lz),
                         self.mass / 12.0 * (lx * lx + lz * lz),
                         self.mass / 12.0 * (lx * lx + lx * lx)])


# ----------------------------------------------------------------------------- rotations
def quat_to_mat(q: np.ndarray) -> np.ndarray:
    """xyzw unit quaternion -> body->world rotation matrix [..., 3, 3]."""
    x, y, z, w = q[..., 0], q[..., 1], q[..., 2], q[..., 3]
    R = np.empty(q.shape[:-1] + (3, 3), dtype=q.dtype)
    R[..., 0, 0] = 1 - 2 * (y * y + z * z)
    R[..., 0, 1] = 2 * (x * y - z * w)
    R[..., 0, 2] = 2 * (x * z + y * w)
    R[..., 1, 0] = 2 * (x * y + z * w)
    R[..., 1, 1] = 1 - 2 * (x * x + z * z)
    R[..., 1, 2] = 2 * (y * z - x * w)
    R[..., 2, 0] = 2 * (x * z - y * w)
    R[..., 2, 1] = 2 * (y * z + x * w)
    R[..., 2, 2] = 1 - 2 * (x * x + y * y)
    return R


def quat_mul(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """Hamilton product a (x) b, xyzw."""
    ax, ay, az, aw = a[..., 0], a[..., 1], a[..., 2], a[..., 3]
    bx, by, bz, bw = b[..., 0], b[..., 1], b[..., 2], b[..., 3]
    return np.stack([aw * bx + ax * bw + ay * bz - az * by,
                     aw * by - ax * bz + ay * bw + az * bx,
                     aw * bz + ax * by - ay * bx + az * bw,
                     aw * bw - ax * bx - ay * by - az * bz], axis=-1)


def _norm(v):
    return np.sqrt(np.sum(v * v, axis=-1, keepdims=True))


def matvec(R, v):
    return np.einsum('...ij,...j->...i', R, v)


def matTvec(R, v):
    return np.einsum('...ji,...j->...i', R, v)


# ----------------------------------------------------------------------------- step pieces
def unconstrained_velocities(quat, vel, angvel, force_w, torque_w, P: PhysicsParams,
                             dt: float, gravity: float):
    """Bullet solveConstraints front half: gravity, ABA for a free base with damping
    and gyroscopic term, v += dt*a, +-max_coord_vel clamp per coordinate."""
    I = P.inertia_diag()
    R = quat_to_mat(quat)
    F = force_w.copy()
    F[..., 2] -= P.mass * gravity
    k = P.lin_damping
    a = F / P.mass - vel * (k + k * _norm(vel))
    w_b = matTvec(R, angvel)
    tau_b = matTvec(R, torque_w)
    Iw = I * w_b
    ka = P.ang_damping
    rhs = tau_b - Iw * (ka + ka * _norm(w_b))
    if P.gyro:
        rhs = rhs - np.cross(w_b, Iw)
    wdot_w = matvec(R, rhs / I)
    v1 = np.clip(vel + dt * a, -P.max_coord_vel, P.max_coord_vel)
    w1 = np.clip(angvel + dt * wdot_w, -P.max_coord_vel, P.max_coord_vel)
    return v1, w1


def _contact_bias(dist, P: PhysicsParams, dt: float):
    """Velocity bound b of a normal row (vn >= b after the solve), after
    btMultiBodyConstraintSolver::setupMultiBodyContactConstraint with restitution 0:
    penetration = dist + slop; an open gap may close within the step (b = -pen/dt < 0), a
    penetrating one is pushed out Baumgarte style (b = -pen*erp2/dt > 0)."""
    pen = dist + P.slop
    return np.where(pen > 0.0, -pen / dt, -pen * P.erp2 / dt)


# lower-rim contact points of the collision cylinder in the body frame (unit radius / half height)
RIM = np.array([[1.0, 0.0], [0.0, 1.0], [-1.0, 0.0], [0.0, -1.0]])


def plane_space(n):
    """btPlaneSpace1: two unit tangents p, q of the unit normal n ([..., 3])."""
    nx, ny, nz = n[..., 0], n[..., 1], n[..., 2]
    big = np.abs(nz) > 0.7071067811865475
    with np.errstate(invalid='ignore', divide='ignore'):
        a1 = ny * ny + nz * nz
        k1 = 1.0 / np.sqrt(a1)
        p1 = np.stack([np.zeros_like(nx), -nz * k1, ny * k1], axis=-1)
        q1 = np.stack([a1 * k1, -nx * p1[..., 2], nx * p1[..., 1]], axis=-1)
        a2 = nx * nx + ny * ny
        k2 = 1.0 / np.sqrt(a2)
        p2 = np.stack([-ny * k2, nx * k2, np.zeros_like(nx)], axis=-1)
        q2 = np.stack([-nz * p2[..., 1], nz * p2[..., 0], a2 * k2], axis=-1)
    return np.where(big[..., None], p1, p2), np.where(big[..., None], q1, q2)


def tournament_partner(N):
    """Round-robin tournament (circle method) over M = N rounded up to even: partner[r, i] for rounds
    r = 0 .. M-2; i == partner means i sits out (odd N).  Every unordered pair meets exactly once."""
    M = N + (N & 1)
    if M < 2:
        return np.zeros((0, N), dtype=np.int64)
    part = np.empty((M - 1, M), dtype=np.int64)
    for r in range(M - 1):
        for i in range(M - 1):
            j = (2 * r - i) % (M - 1)
            part[r, i] = (M - 1) if j == i else j
        part[r, M - 1] = r
    part = part[:, :N].copy()
    idx = np.arange(N)[None, :]
    part = np.where(part >= N, idx, part)             # the dummy of an odd N: sit out
    return part


def ground_rim(pos, R, P: PhysicsParams):
    """The four lower-rim points of the collision cylinder (the face that looks down) for positions [E,N,3] and
    body->world rotations [E,N,3,3]: body-frame points c [E,N,4,3], world z in the body frame nb [E,N,3] (row 2 of
    R) and each point's gap to the ground [E,N,4] (collision margin included)."""
    E, N = pos.shape[:2]
    sgn = np.where(R[..., 2, 2] >= 0.0, 1.0, -1.0)
    c = np.empty((E, N, 4, 3))                         # body-frame contact points
    c[..., 0] = P.col_radius * RIM[:, 0]
    c[..., 1] = P.col_radius * RIM[:, 1]
    c[..., 2] = (-P.col_halfheight * sgn)[..., None]
    nb = R[..., 2, :]                                  # world z in the body frame (row 2 of R)
    zoff = np.einsum('enk,enpk->enp', nb, c)           # height of the point above the CoM
    return c, nb, pos[..., 2, None] + zoff - P.col_margin - P.ground_z


def solve_contacts(pos, quat, v1, w1, P: PhysicsParams, dt: float, counts: dict | None = None):
    """Sequential-impulse contact solve on the unconstrained velocities (see the module
    docstring for the row set and the sweep order).  Returns (v, w) world frame.

    counts (optional dict): filled with what the kernels count (include/mrs_b200.h, stats slots), shaped like the
    leading dims of pos:
      'sweeps'    [...]     sweeps run while the env was alive (0 for an env that had no row when no env had one);
      'active'    [...]     the env had an active row (ground point within the margin, or a pair in range);
      'worst'     [s][...]  largest row change of every sweep s (all envs, alive or not);
      'ground'    [..., N]  the agent's ground rows pushed (sum of its four normal impulses > 0);
      'pair_rows' [..., N]  pair rows of the agent with normal impulse > 0 (a pushing pair counts for both agents);
      'g_lam'     [..., N, 4] final normal impulses of the ground rows (0 where no row);
      'p_lam'     list of [...] final normal impulses of the active pair rows (inactive rows are 0)."""
    lead = pos.shape[:-2]
    N = pos.shape[-2]
    pos = pos.reshape(-1, N, 3)
    quat = quat.reshape(-1, N, 4)
    v = np.array(v1, np.float64).reshape(-1, N, 3)
    w = np.array(w1, np.float64).reshape(-1, N, 3)
    E = pos.shape[0]
    im = 1.0 / P.mass
    invI = 1.0 / P.inertia_diag()
    R = quat_to_mat(quat)
    wb = matTvec(R, w)                                     # body-frame angular velocity during the solve
    # ---- ground rows: four lower-rim points (the face that looks down)
    g_act = np.zeros((E, N, 4), dtype=bool)
    if P.ground_contact:
        c, nb, dist = ground_rim(pos, R, P)
        g_act = dist < P.contact_margin
        g_bias = _contact_bias(dist, P, dt)
        g_a = np.cross(c, nb[..., None, :])                # (c x n)_body
        g_K = im + np.sum(g_a * g_a * invI, axis=-1)
        g_lam = np.zeros((E, N, 4))
        f_lam = np.zeros((E, N, 2))
    # ---- pair rows
    part = tournament_partner(N) if (P.agent_contact and N > 1) else np.zeros((0, N), dtype=np.int64)
    rounds = []
    for r in range(part.shape[0]):
        pr = part[r]
        lo = np.nonzero(pr > np.arange(N))[0]              # the lower index of each pair of the round
        hi = pr[lo]
        d = pos[:, lo] - pos[:, hi]
        dd = np.sqrt(np.sum(d * d, axis=-1))
        act = (dd - 2.0 * P.contact_radius < P.contact_margin) & (dd > 0.0)
        if not act.any():
            continue
        with np.errstate(invalid='ignore', divide='ignore'):
            n = np.where(act[..., None], d / dd[..., None], np.array([0.0, 0.0, 1.0]))
        t1, t2 = plane_space(n)
        rounds.append(dict(lo=lo, hi=hi, act=act, n=n, t1=t1, t2=t2,
                           bias=_contact_bias(dd - 2.0 * P.contact_radius, P, dt),
                           lam=np.zeros(act.shape), lt1=np.zeros(act.shape), lt2=np.zeros(act.shape)))
    if counts is not None:
        p_act = np.zeros(E, dtype=bool)
        for rd in rounds:
            p_act |= rd['act'].any(axis=-1)
        counts.update(sweeps=np.zeros(lead, np.int64), active=(g_act.any(axis=(-2, -1)) | p_act).reshape(lead),
                      worst=[], ground=np.zeros(lead + (N,), bool), pair_rows=np.zeros(lead + (N,), np.int64),
                      g_lam=np.zeros(lead + (N, 4)), p_lam=[])
    if not (g_act.any() or rounds):
        return np.array(v1, np.float64).reshape(lead + (N, 3)), np.array(w1, np.float64).reshape(lead + (N, 3))
    alive = np.ones(E, dtype=bool)                         # envs that have not converged yet
    sweeps = np.zeros(E, np.int64)
    for it in range(int(P.solver_iters)):
        sweeps += alive
        worst = np.zeros(E)
        am = alive[:, None]
        if P.ground_contact:
            for p in range(4):
                a = g_a[..., p, :]
                vn = v[..., 2] + np.sum(a * wb, axis=-1)
                lam_new = np.maximum(g_lam[..., p] + (g_bias[..., p] - vn) / g_K[..., p], 0.0)
                dl = np.where(g_act[..., p] & am, lam_new - g_lam[..., p], 0.0)
                g_lam[..., p] += dl
                v[..., 2] += dl * im
                wb += (a * invI) * dl[..., None]
                worst = np.maximum(worst, np.max(np.abs(dl) * g_K[..., p], axis=-1))
            lim = P.mu_ground * np.sum(g_lam, axis=-1)
            for k in range(2):
                lam_new = np.clip(f_lam[..., k] - v[..., k] / im, -lim, lim)
                dl = np.where(am, lam_new - f_lam[..., k], 0.0)
                f_lam[..., k] += dl
                v[..., k] += dl * im
                worst = np.maximum(worst, np.max(np.abs(dl) * im, axis=-1))
        for rd in rounds:
            lo, hi, act = rd['lo'], rd['hi'], rd['act'] & am
            for key, lkey in (('n', 'lam'), ('t1', 'lt1'), ('t2', 'lt2')):
                u = rd[key]
                vr = np.sum(u * (v[:, lo] - v[:, hi]), axis=-1)
                if key == 'n':
                    lam_new = np.maximum(rd['lam'] + (rd['bias'] - vr) / (2.0 * im), 0.0)
                else:
                    lim = P.mu_agent * rd['lam']
                    lam_new = np.clip(rd[lkey] - vr / (2.0 * im), -lim, lim)
                dl = np.where(act, lam_new - rd[lkey], 0.0)
                rd[lkey] = rd[lkey] + dl
                v[:, lo] += u * (dl * im)[..., None]
                v[:, hi] -= u * (dl * im)[..., None]
                if dl.shape[1]:
                    worst = np.maximum(worst, np.max(np.abs(dl) * 2.0 * im, axis=-1))
        if counts is not None:
            counts['worst'].append(worst.reshape(lead))
        alive = alive & ~(worst < P.solver_tol)
        if not alive.any():
            break
    if counts is not None:
        counts['sweeps'] = sweeps.reshape(lead)
        pair_rows = np.zeros((E, N), np.int64)
        for rd in rounds:
            pushed = (rd['lam'] > 0.0).astype(np.int64)
            pair_rows[:, rd['lo']] += pushed
            pair_rows[:, rd['hi']] += pushed
            counts['p_lam'].append(np.where(rd['act'], rd['lam'], 0.0).reshape(lead + (-1,)))
        counts['pair_rows'] = pair_rows.reshape(lead + (N,))
        if P.ground_contact:
            counts['ground'] = (np.sum(g_lam, axis=-1) > 0.0).reshape(lead + (N,))
            counts['g_lam'] = g_lam.reshape(lead + (N, 4))
    w = matvec(R, wb)
    return v.reshape(lead + (N, 3)), w.reshape(lead + (N, 3))


def integrate_positions(pos, quat, v, w, P: PhysicsParams, dt: float):
    """btMultiBody::stepPositionsMultiDof for the base: p += dt*v; world-frame
    exponential map q <- dq(w*dt) (x) q with |w|dt capped at pi/4 and a Taylor branch
    below 1e-3 rad/s, then normalise."""
    pos1 = pos + dt * v
    ang = _norm(w)
    ang = np.where(ang * dt > P.ang_motion_threshold, 0.5 * (0.5 * math.pi) / dt, ang)
    with np.errstate(invalid='ignore', divide='ignore'):
        big = np.sin(0.5 * ang * dt) / ang
    small = 0.5 * dt - (dt * dt * dt) * 0.020833333333 * ang * ang
    axis = w * np.where(ang < 0.001, small, big)
    dq = np.concatenate([axis, np.cos(0.5 * ang * dt)], axis=-1)
    q1 = quat_mul(dq, quat)
    q1 = q1 / _norm(q1)
    return pos1, q1


def bullet_step(pos, quat, vel, angvel, force_w, torque_w, P: PhysicsParams,
                dt: float = 0.01, gravity: float = 9.81, counts: dict | None = None):
    """One ``stepSimulation`` (numSubSteps=0).  Inputs float64, world frame; force/torque
    are the summed external wrench about the CoM.  Returns (pos, quat, vel, angvel).
    counts: see solve_contacts (left empty when both contact kinds are off)."""
    v1, w1 = unconstrained_velocities(quat, vel, angvel, force_w, torque_w, P, dt, gravity)
    if P.ground_contact or P.agent_contact:
        v1, w1 = solve_contacts(pos, quat, v1, w1, P, dt, counts)
    pos1, q1 = integrate_positions(pos, quat, v1, w1, P, dt)
    return pos1, q1, v1, w1
