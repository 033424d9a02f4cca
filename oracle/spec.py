"""TEST INFRASTRUCTURE -- CPU oracle ("port"), not product code.

Batched ``[E, N]`` numpy restatement of the mrs-gym per-step hot path.  Every function
cites the reference lines it follows; dtypes (float32 getters, float64 numpy promotion)
are mirrored so that one env of this model reproduces the reference's own Python run
verbatim on ``oracle/fake_pybullet`` (tests/test_oracle_golden.py pins it against
tests/golden/ref_*.npz, which ``oracle/make_golden.py`` generated from /root/reference).

  MRS.step / calc_Xk / calc_Ak / calc_A        /root/reference/mrsgym/MRS.py:87-124,240-277
  Environment.set_actions / get_X              /root/reference/mrsgym/Environment.py:84-94
  Quadcopter.set_* / dynamics / nnlsRPM        /root/reference/mrsgym/Quadcopter.py:26-115,172-208
  QuadControl.*                                /root/reference/mrsgym/QuadControl.py:35-127
  Object getters (float32)                     /root/reference/mrsgym/Object.py:78-97
  p.stepSimulation                             oracle/bullet_model.py (PARITY UNPINNED part)
"""
from __future__ import annotations

import math

import numpy as np
from scipy.optimize import nnls
from scipy.spatial.transform import Rotation as R

from . import bullet_model as bm

f32 = np.float32

ACTION_DIMS = dict(set_target_vel=3, set_target_pos=3, set_target_accel=3, set_force=3,
                   set_target_ori=3, set_control=4, set_speeds=4)


# ----------------------------------------------------------------------------- adjacency
def fma32(a, b, c):
    """Correctly rounded float32 fma(a,b,c) from float64 arithmetic: a*b is exact in
    float64; the sum is rounded to odd (TwoSum error as sticky bit) so the final
    float32 rounding is the single correct one."""
    a, b, c = np.broadcast_arrays(np.asarray(a, f32), np.asarray(b, f32), np.asarray(c, f32))
    shape = a.shape
    a = a.astype(np.float64).ravel()
    b = b.astype(np.float64).ravel()
    c = c.astype(np.float64).ravel()
    p = a * b
    s = p + c
    bb = s - p
    err = (p - (s - bb)) + (c - bb)
    bits = s.view(np.int64).copy()
    inexact = (err != 0) & np.isfinite(s)
    even = (bits & 1) == 0
    # the odd neighbour lies in err's direction: larger magnitude iff sign(err)==sign(s)
    away = (err > 0) == (s > 0)
    bits = np.where(inexact & even, bits + np.where(away, 1, -1), bits)
    return bits.view(np.float64).astype(f32).reshape(shape)


def adjacency(pos32, comm_range):
    """MRS.calc_A (/root/reference/mrsgym/MRS.py:117-124) on float32 positions
    ``[..., N, 3]``: d = ||p_i - p_j||_2 in float32 (torch CPU ``norm``: sqrt_rn of
    fma(dz,dz,fma(dy,dy,dx*dx)), SURVEY.md §8a row a15), diagonal -> inf,
    A = (d <= float32(COMM_RANGE)).  NaN distance -> 0."""
    pos32 = np.asarray(pos32, f32)
    N = pos32.shape[-2]
    if comm_range == float('inf'):
        A = np.ones(pos32.shape[:-2] + (N, N), f32) - np.eye(N, dtype=f32)
        return A
    d = pos32[..., :, None, :] - pos32[..., None, :, :]
    dx, dy, dz = d[..., 0], d[..., 1], d[..., 2]
    s = fma32(dz, dz, fma32(dy, dy, (dx * dx).astype(f32)))
    dist = np.sqrt(s.astype(f32)).astype(f32)
    with np.errstate(invalid='ignore'):
        A = (dist <= f32(comm_range))
    A = A & ~np.eye(N, dtype=bool)
    return A.astype(f32)


# ----------------------------------------------------------------------------- mixer
MIX_A = np.array([[1, 1, 1, 1],
                  [1 / np.sqrt(2), 1 / np.sqrt(2), -1 / np.sqrt(2), -1 / np.sqrt(2)],
                  [-1 / np.sqrt(2), 1 / np.sqrt(2), 1 / np.sqrt(2), -1 / np.sqrt(2)],
                  [-1, 1, -1, 1]])          # Quadcopter.py:164
MIX_AINV = np.linalg.inv(MIX_A)


def nnls_subset_tables():
    """For each of the 16 column subsets S of MIX_A: the 4x4 matrix P_S with
    x = P_S @ B the unconstrained least-squares solution on S (zero off S).  The
    NNLS optimum is the primal-feasible subset solution of least residual."""
    tabs = np.zeros((16, 4, 4))
    for m in range(16):
        cols = [c for c in range(4) if (m >> c) & 1]
        if cols:
            As = MIX_A[:, cols]
            tabs[m][cols, :] = np.linalg.solve(As.T @ As, As.T)
    return tabs


def nnls_rpm(B):
    """nnlsRPM (/root/reference/mrsgym/Quadcopter.py:172-208): sq = Ainv@B; if any
    negative -> scipy nnls(A, B, maxiter=12); rpm = sqrt(sq).  B: [M,4] float64."""
    sq = B @ MIX_AINV.T
    out = sq.copy()
    for m in np.nonzero(sq.min(axis=1) < 0)[0]:
        out[m], _ = nnls(MIX_A, B[m], maxiter=3 * 4)
    return np.sqrt(out)


# ----------------------------------------------------------------------------- the env model
class SpecEnv:
    """E independent 'simple' worlds of N cf2x quads.  State float64 like Bullet's."""

    def __init__(self, E, N, action_type='set_target_vel', K=0, comm_range=float('inf'),
                 dt=0.01, gravity=9.81, phys: bm.PhysicsParams | None = None,
                 quad: bm.QuadParams | None = None):
        self.E, self.N, self.K = E, N, K
        self.action_type = action_type
        self.comm_range = comm_range
        self.dt, self.gravity = dt, gravity
        self.P = phys or bm.PhysicsParams()
        self.Q = quad or bm.QuadParams()
        self.der = self.Q.derived(gravity)
        z = np.zeros((E, N, 3))
        self.pos, self.vel, self.angvel = z.copy(), z.copy(), z.copy()
        self.quat = np.zeros((E, N, 4))
        self.quat[..., 3] = 1.0
        self.speeds = np.zeros((E, N, 4))          # Quadcopter.speeds (Quadcopter.py:19)
        self.ctrl = {}                               # lazily created like QuadControl's hasattr
        self.X, self.A = [], []
        self.last = {}

    # ---- Object getters (/root/reference/mrsgym/Object.py:78-97): float32 views
    def get_pos(self):
        return self.pos.astype(f32)

    def get_vel(self):
        return self.vel.astype(f32)

    def get_angvel(self):
        return self.angvel.astype(f32)

    def _rot(self):
        q32 = self.quat.astype(f32).astype(np.float64).reshape(-1, 4)
        return R.from_quat(q32)

    def get_ori(self):
        return self._rot().as_euler('xyz').astype(f32).reshape(self.E, self.N, 3)

    def get_ori_mat(self):
        return self._rot().as_matrix().astype(f32).reshape(self.E, self.N, 3, 3)

    def set_state(self, pos=None, quat=None, vel=None, angvel=None, ori_euler=None):
        if pos is not None:
            self.pos = np.array(pos, np.float64).reshape(self.E, self.N, 3)
        if ori_euler is not None:    # Object.set_state: euler 'xyz' -> quat (Object.py:54-56)
            e = np.array(ori_euler, np.float64).reshape(-1, 3)
            quat = R.from_euler('xyz', e).as_quat().reshape(self.E, self.N, 4)
        if quat is not None:
            q = np.array(quat, np.float64).reshape(self.E, self.N, 4)
            self.quat = q / np.linalg.norm(q, axis=-1, keepdims=True)
        if vel is not None:
            self.vel = np.array(vel, np.float64).reshape(self.E, self.N, 3)
        if angvel is not None:
            self.angvel = np.array(angvel, np.float64).reshape(self.E, self.N, 3)

    # ---- QuadControl (/root/reference/mrsgym/QuadControl.py)
    def _pos_control(self, target_pos):                       # :35-48
        pos, vel = self.get_pos(), self.get_vel()
        target_pos = np.asarray(target_pos)
        pos_e = target_pos - pos
        if 'integral_pos_e' not in self.ctrl:
            self.ctrl['integral_pos_e'] = np.zeros((self.E, self.N, 3))
        d_pos_e = np.zeros(3) - vel
        self.ctrl['integral_pos_e'] = self.ctrl['integral_pos_e'] + pos_e * self.Q.ctrl_dt
        ta = (self.Q.pos_p * np.ones(3)) * pos_e + (self.Q.pos_i * np.ones(3)) * self.ctrl['integral_pos_e'] \
            + (self.Q.pos_d * np.ones(3)) * d_pos_e
        return self._accel_control(ta)

    def _vel_control(self, target_vel):                       # :51-70
        vel = self.get_vel()
        target_vel = np.asarray(target_vel)
        vel_e = target_vel - vel
        c = self.ctrl
        if 'last_vel_e' not in c:
            c['last_vel_e'] = vel_e
            c['d_vel_e'] = np.zeros((self.E, self.N, 3))
        elif np.isnan(c['last_vel_e'][..., 0]).any():
            # rows of agents whose controller has never run (step(nan_policy='agent_none') put the marker back):
            # their first call, per agent, like the device's last_vel_e.x = NaN marker
            first = np.isnan(c['last_vel_e'][..., 0])[..., None]
            c['last_vel_e'] = np.where(first, vel_e, c['last_vel_e'])
            c['d_vel_e'] = np.where(first, 0.0, c['d_vel_e'])
            c['last_target_vel'] = np.where(first, target_vel, c['last_target_vel'])
        if 'last_target_vel' not in c:
            c['last_target_vel'] = target_vel
        if 'integral_vel_e' not in c:
            c['integral_vel_e'] = np.zeros((self.E, self.N, 3))
        DT = self.Q.ctrl_dt
        c['d_vel_e'] = (((vel_e - c['last_vel_e']) - (target_vel - c['last_target_vel'])) / DT) * 0.5 \
            + c['d_vel_e'] * 0.5
        c['last_vel_e'] = vel_e
        c['last_target_vel'] = target_vel
        c['integral_vel_e'] = c['integral_vel_e'] + vel_e * DT
        ta = (self.Q.vel_p * np.ones(3)) * vel_e + (self.Q.vel_i * np.ones(3)) * c['integral_vel_e'] \
            + (self.Q.vel_d * np.ones(3)) * c['d_vel_e']
        return self._accel_control(ta)

    def _accel_control(self, target_accel):                   # :73-90
        ori = self.get_ori()
        ta = np.asarray(target_accel) + np.array([0.0, 0.0, self.Q.ctrl_gravity])
        ta = np.broadcast_to(ta, (self.E, self.N, 3)).astype(np.float64)
        rot32 = R.from_euler('xyz', ori.reshape(-1, 3).astype(np.float64)).as_matrix().astype(f32)
        rot32 = rot32.reshape(self.E, self.N, 3, 3)
        with np.errstate(invalid='ignore', divide='ignore'):
            tz = ta / np.linalg.norm(ta, axis=-1, keepdims=True)
        bad = np.any(np.isnan(tz), axis=-1)
        tz[bad] = np.array([0.0, 0.0, 1.0])
        tx = np.cross(rot32[..., :, 1], tz)
        ty = np.cross(tz, tx)
        tr = np.stack([tx, ty, tz], axis=-1)
        target_ori = R.from_matrix(tr.reshape(-1, 3, 3)).as_euler('xyz').reshape(self.E, self.N, 3)
        return self._attitude_control(target_ori, ta)

    def _attitude_control(self, target_ori, target_accel):    # :93-127
        Q = self.Q
        ori = self.get_ori()
        angvel = self.get_angvel()
        target_accel = np.broadcast_to(np.asarray(target_accel, np.float64), (self.E, self.N, 3))
        rot = R.from_euler('xyz', ori.reshape(-1, 3).astype(np.float64)).as_matrix().reshape(self.E, self.N, 3, 3)
        trot = R.from_euler('xyz', np.asarray(target_ori).reshape(-1, 3).astype(np.float64)).as_matrix()
        trot = trot.reshape(self.E, self.N, 3, 3)
        rme = np.einsum('...ji,...jk->...ik', trot, rot) - np.einsum('...ji,...jk->...ik', rot, trot)
        rot_e = np.stack([rme[..., 2, 1], rme[..., 0, 2], rme[..., 1, 0]], axis=-1)
        if 'integral_ori_e' not in self.ctrl:
            self.ctrl['integral_ori_e'] = np.zeros((self.E, self.N, 3))
        angvel_e = np.array([0, 0, 0]) - angvel
        ie = self.ctrl['integral_ori_e'] - rot_e * Q.ctrl_dt
        ie = np.clip(ie, -1500.0, 1500.0)
        ie[..., 0:2] = np.clip(ie[..., 0:2], -1.0, 1.0)
        self.ctrl['integral_ori_e'] = ie
        tt = -np.array(Q.ori_p) * rot_e + np.array(Q.ori_i) * ie + np.array(Q.ori_d) * angvel_e
        tt = np.clip(tt, -3200, 3200)
        nrm = np.linalg.norm(target_accel, axis=-1)
        with np.errstate(invalid='ignore', divide='ignore'):
            cosang = np.sum(target_accel / nrm[..., None] * rot[..., :, 2], axis=-1)
            ratio = 1.0 / np.maximum(cosang, 0.2)
            scalar_thrust = np.where(nrm != 0, ratio * nrm * Q.mass, 0.0)
        thrust = (np.sqrt(scalar_thrust / (4 * Q.kf)) - Q.pwm2rpm_b) / Q.pwm2rpm_a
        mixer = np.array([[.5, -.5, -1], [.5, .5, 1], [-.5, .5, -1], [-.5, -.5, 1]])
        pwm = thrust[..., None] + np.einsum('mk,...k->...m', mixer, tt)
        pwm = np.clip(pwm, Q.min_pwm, Q.max_pwm)
        return Q.pwm2rpm_a * pwm + Q.pwm2rpm_b

    # ---- Quadcopter action modes (/root/reference/mrsgym/Quadcopter.py:26-65)
    def _set_control(self, control):
        Q = self.Q
        control = np.asarray(control)
        if control.dtype == f32:     # torch f32 scalar * python float -> f32
            comp = np.stack([control[..., 0] * f32(Q.mass), control[..., 1] * f32(Q.ixx),
                             control[..., 2] * f32(Q.iyy), control[..., 3] * f32(Q.izz)], axis=-1)
        else:
            comp = control * np.array([Q.mass, Q.ixx, Q.iyy, Q.izz])
        bcoeff = np.array([1 / Q.kf, 1 / (Q.kf * Q.arm), 1 / (Q.kf * Q.arm), 1 / Q.km])
        B = comp.astype(np.float64) * bcoeff
        return nnls_rpm(B.reshape(-1, 4)).reshape(self.E, self.N, 4)

    def _apply_speeds(self, speeds):
        """set_speeds (Quadcopter.py:38-45): rotor thrust along link z at the prop-link
        CoM + yaw torque on link 4, both LINK_FRAME.  Returns body-frame wrench."""
        Q = self.Q
        self.speeds = np.array(speeds)
        forces = np.array(self.speeds ** 2) * Q.kf
        torques = np.array(self.speeds ** 2) * Q.km
        z_torque = (-torques[..., 0] + torques[..., 1] - torques[..., 2] + torques[..., 3])
        return forces.astype(np.float64), z_torque.astype(np.float64)

    # ---- one env.step (MRS.step, /root/reference/mrsgym/MRS.py:240-277)
    def step(self, actions, action_type=None, nan_policy='raise', counts=None):
        """nan_policy: 'raise' (MRS.py:247-248) or 'agent_none', the rule of the CUDA step for device-resident actions:
        an agent with a NaN in any action component steps like MRS.step(None) -- no rotor wrench (thrust, drag,
        ground effect) and no downwash received, its controller state as before the step, its rotor speeds 0 -- while
        it still casts downwash onto the others.  counts: see bullet_model.solve_contacts."""
        mode = action_type or self.action_type
        Q, E, N = self.Q, self.E, self.N
        nan_rows = None
        if actions is not None:
            actions = np.asarray(actions)
            if np.any(np.isnan(actions)):
                if nan_policy != 'agent_none':
                    raise Exception('The given action contains NaN')
                actions = actions.reshape(E, N, -1)
                nan_rows = np.any(np.isnan(actions), axis=-1)
                actions = np.where(nan_rows[..., None], actions.dtype.type(0), actions)
                saved = {k: np.array(v, copy=True) for k, v in self.ctrl.items()}
            actions = actions.reshape(E, N, -1)
            if mode == 'set_target_vel':
                rpm = self._vel_control(actions)
            elif mode == 'set_target_pos':
                rpm = self._pos_control(actions)
            elif mode == 'set_target_accel':
                rpm = self._accel_control(actions)
            elif mode == 'set_force':      # README alias; := set_target_accel(F/Mass) (SURVEY §0.4)
                rpm = self._accel_control(actions / actions.dtype.type(Q.mass))
            elif mode == 'set_target_ori':
                rpm = self._attitude_control(actions, np.array([0.0, 0.0, 9.81]))
            elif mode == 'set_control':
                rpm = self._set_control(actions)
            elif mode == 'set_speeds':
                rpm = actions
            else:
                raise AttributeError("'Quadcopter' object has no attribute '%s'" % mode)
            forces, z_torque = self._apply_speeds(rpm)
            Fw, Tw = self._wrench(forces, z_torque)
            if nan_rows is not None:
                Fw[nan_rows] = 0.0
                Tw[nan_rows] = 0.0
                self.speeds = np.array(self.speeds, np.float64)
                self.speeds[nan_rows] = 0.0
                for k in list(self.ctrl):
                    v = np.array(np.broadcast_to(self.ctrl[k], (E, N, 3)), copy=True)
                    if k in saved:
                        v[nan_rows] = saved[k][nan_rows]
                    elif nan_rows.all():
                        del self.ctrl[k]
                        continue
                    else:       # created by this step: the agents back to "never called"
                        v[nan_rows] = np.nan if k == 'last_vel_e' else 0.0
                    self.ctrl[k] = v
        else:
            Fw = np.zeros((E, N, 3))
            Tw = np.zeros((E, N, 3))
        self.last = dict(rpm=np.array(self.speeds, np.float64), force=Fw, torque=Tw)
        self.pos, self.quat, self.vel, self.angvel = bm.bullet_step(
            self.pos, self.quat, self.vel, self.angvel, Fw, Tw, self.P, self.dt, self.gravity, counts)
        X = self.calc_X()
        self.X.insert(0, X)
        del self.X[self.K + 1:]
        while len(self.X) < self.K + 1:
            self.X.append(X)
        A = adjacency(self.get_pos(), self.comm_range)
        self.A.insert(0, A)
        del self.A[self.K + 1:]
        while len(self.A) < self.K + 1:
            self.A.append(np.zeros((E, N, N), f32))
        return np.stack(self.X, axis=1), np.stack(self.A, axis=1)   # [E,K+1,N,D], [E,K+1,N,N]

    def reset_rings(self):
        """MRS.reset/set tail (MRS.py:185-192): clear rings, refill X with copies."""
        self.X, self.A = [], []
        X = self.calc_X()
        self.X = [X] * (self.K + 1)
        return np.stack(self.X, axis=1)

    def calc_X(self):
        """state_fn = cat(get_pos, get_vel) (README.md:28-29) -> [E,N,6] float32."""
        return np.concatenate([self.get_pos(), self.get_vel()], axis=-1)

    # ---- forces of set_speeds + Quadcopter.dynamics (Quadcopter.py:38-45,69-115)
    def _wrench(self, forces, z_torque):
        Q, E, N = self.Q, self.E, self.N
        R64 = bm.quat_to_mat(self.quat)                     # backend applies LINK_FRAME with exact state
        offs = np.array([[x, y, 0.0] for x, y in Q.prop_xy])  # [4,3]
        zb = np.array([0.0, 0.0, 1.0])
        # rotor thrust: force f_i*z_body at r_i
        Fb = np.zeros((E, N, 3))
        Tb = np.zeros((E, N, 3))
        for i in range(4):
            fi = forces[..., i, None] * zb
            Fb += fi
            Tb += np.cross(offs[i], fi)
        Tb[..., 2] += z_torque
        # ground effect (:70-87)
        pos64 = self.pos
        heights = np.stack([(pos64 + bm.matvec(R64, offs[i]))[..., 2] for i in range(4)], axis=-1)
        heights = np.clip(heights, self.der['GroundEffectHClip'], np.inf)
        gnd = np.array(self.speeds ** 2) * Q.kf * Q.gnd_eff_coeff * (Q.prop_radius / (4 * heights)) ** 2
        ori = self.get_ori()
        ok = (ori[..., 0] < f32(np.pi / 2)) & (ori[..., 1] < f32(np.pi / 2))
        gnd = np.where(ok[..., None], gnd, 0.0).astype(np.float64)
        for i in range(4):
            gi = gnd[..., i, None] * zb
            Fb += gi
            Tb += np.cross(offs[i], gi)
        # drag (:88-98): R32 @ (c * v32), applied again in LINK_FRAME
        rot32 = self.get_ori_mat()
        vel32 = self.get_vel()
        s = np.sum(np.array(2 * np.pi * self.speeds / 60), axis=-1)
        drag_factors = -1 * np.array([Q.drag_xy, Q.drag_xy, Q.drag_z]) * s[..., None]
        drag = np.einsum('...ij,...j->...i', rot32.astype(np.float64), drag_factors * vel32)
        Fb += drag
        # downwash (:99-115) -- float32 arithmetic as in the reference
        pos32 = self.get_pos()
        rel = pos32[:, None, :, :] - pos32[:, :, None, :]          # [E,i,j] = p_j - p_i
        dz = rel[..., 2]
        dxy = np.sqrt((rel[..., 0] * rel[..., 0] + rel[..., 1] * rel[..., 1]).astype(f32)).astype(f32)
        with np.errstate(invalid='ignore', divide='ignore', over='ignore'):
            # torch evaluates `scalar / tensor` as tensor.reciprocal() * scalar (float32)
            r = (f32(1) / (f32(4) * dz)) * f32(Q.prop_radius)
            alpha = f32(Q.dw1) * (r * r)
            beta = f32(Q.dw2) * dz + f32(Q.dw3)
            q = (f32(1) / beta) * dxy
            dw = -alpha * np.exp(f32(-.5) * (q * q))
        mask = (dz > 0) & (dxy < 10)
        dw = np.where(mask, dw, f32(0)).astype(np.float64)
        Fb[..., 2] += dw.sum(axis=-1)
        Fw = bm.matvec(R64, Fb)
        Tw = bm.matvec(R64, Tb)
        return Fw, Tw
