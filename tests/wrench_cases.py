"""Seeded scenes for the external wrench (MrsBuffers.wrench, Swarm.set_external_wrench): float32 start states and
float32 world-frame forces / torques fed identically to the CUDA step and to the CPU oracle, plus the wrong kernels a
test must tell apart from the right one.  The oracle's step (oracle/spec.py SpecEnv.step) knows no external wrench:
step_with_wrench() runs it with bullet_model.bullet_step wrapped so that the wrench is added in float64 to the
agent's own world-frame wrench -- after the NaN-action zeroing and also without actions, where the kernels add it.  Shared by test_cpu_wrench.py (oracle
only) and test_gpu_wrench.py."""
from __future__ import annotations

from unittest import mock

import numpy as np

import helpers as H
import physics_variants as V

MASS, G = 0.027, 9.81
WEIGHT = MASS * G                 # 0.265 N
SPACING = 1.4                     # lattice pitch: no two scene units within contact range (0.62 m)
Z_AIR = 3.0
Z_REST = V.Z_TOUCH - 0.004        # collision-cylinder rim on the ground (resting, rows active)
MU_GROUND = 0.75

# kind -> (contact scene, wrong kernels the kind must be >= 10 bars away from)
KINDS = {
    'tilted': (False, ('none', 'body_force', 'torque_unrotated')),      # up to 60 deg, every other agent inverted
    'weightless': (False, ('none', 'body_force')),                      # F = m g z on agents tilted 40 deg
    'clamp': (False, ('none',)),                                        # a push past max_coord_vel
    'pressed': (True, ('none', 'after_contact')),                       # grounded, pushed down
    'slide_below': (True, ('after_contact',)),                          # grounded, sideways at half the friction limit
    'slide_above': (True, ('none', 'after_contact')),                   # grounded, sideways at twice the limit
    'collide': (True, ('none', 'after_contact')),                       # pairs in contact pushed into each other
}
WRONG = ('none', 'body_force', 'torque_unrotated', 'after_contact', 'nan_zeroed')


def _lattice(E, N, z):
    cols = int(np.ceil(np.sqrt(N)))
    k = np.arange(N)
    p = np.stack([(k % cols) * SPACING, (k // cols) * SPACING, np.full(N, z)], axis=-1)
    return np.broadcast_to(p, (E, N, 3)).copy()


def make_case(kind, E, N, seed=0):
    """(state, force [E,N,3], torque [E,N,3]) of a scene kind, float32.  Every scene carries torques that move w by
    >= 10 one-step bars (1e-4 N m: ~0.03 rad/s in a step against a 1e-5 rad/s floor)."""
    from scipy.spatial.transform import Rotation
    rng = np.random.default_rng(seed)
    S = E * N
    yaw = rng.uniform(-np.pi, np.pi, S)
    roll = rng.uniform(-0.05, 0.05, S)
    pitch = rng.uniform(-0.05, 0.05, S)
    vel = rng.uniform(-0.2, 0.2, (E, N, 3))
    torque = rng.uniform(-2e-4, 2e-4, (E, N, 3))
    force = np.zeros((E, N, 3))
    pos = _lattice(E, N, Z_AIR)
    if kind == 'tilted':
        roll = rng.uniform(-np.pi / 3, np.pi / 3, S)
        pitch = rng.uniform(-np.pi / 3, np.pi / 3, S)
        roll[1::2] += np.pi                                        # inverted: body z points down
        d = rng.normal(0, 1, (E, N, 3))
        force = d / np.linalg.norm(d, axis=-1, keepdims=True) * rng.uniform(0.05, WEIGHT, (E, N, 1))
    elif kind == 'weightless':
        roll = rng.choice([-1.0, 1.0], S) * np.radians(40)
        force[..., 2] = WEIGHT
    elif kind == 'clamp':
        vel[..., 0] = 99.9
        force[..., 0] = 2.0                                        # dv = 0.74 m/s: v* = 100 (clamped)
    elif kind in ('pressed', 'slide_below', 'slide_above'):
        pos[..., 2] = Z_REST
        vel[:] = 0.0
        torque *= 0.1
        if kind == 'pressed':
            force[..., 2] = -0.5
        else:
            # friction limit of the ground rows of a resting agent under its weight alone: mu m g (NO_ACTION scenes)
            f = (0.5 if kind == 'slide_below' else 2.0) * MU_GROUND * WEIGHT
            a = rng.uniform(0, 2 * np.pi, (E, N))
            force[..., 0], force[..., 1] = f * np.cos(a), f * np.sin(a)
    elif kind == 'collide':
        vel[:] = 0.0
        for i in range(0, N - 1, 2):                               # agent i + 1 sits 0.58 m from i (overlap 2 cm)
            d = rng.normal(0, 1, (E, 3))
            d[:, 2] *= 0.3
            d /= np.linalg.norm(d, axis=-1, keepdims=True)
            pos[:, i + 1] = pos[:, i] + 0.58 * d
            force[:, i] = 0.2 * d
            force[:, i + 1] = -0.2 * d
    else:
        raise ValueError(kind)
    quat = Rotation.from_euler('xyz', np.stack([roll, pitch, yaw], -1)).as_quat().reshape(E, N, 4)
    st = dict(pos=pos, quat=quat, vel=vel, angvel=rng.uniform(-0.3, 0.3, (E, N, 3)))
    return ({k: v.astype(np.float32) for k, v in st.items()}, force.astype(np.float32), torque.astype(np.float32))


def rotmat(quat):
    """R of the float32 quaternion as the oracle holds it (normalised in float64)"""
    from oracle import bullet_model as bm
    q = np.asarray(quat, np.float64)
    return bm.quat_to_mat(q / np.linalg.norm(q, axis=-1, keepdims=True))


def _with_wrench(F, Tq):
    """bullet_step with F / Tq [E, N, 3] added to the summed applied wrench (the right kernel)"""
    from oracle import bullet_model as bm
    real = bm.bullet_step

    def step(pos, quat, vel, angvel, force_w, torque_w, P, dt=0.01, gravity=9.81, counts=None):
        return real(pos, quat, vel, angvel, force_w + F, torque_w + Tq, P, dt, gravity, counts)
    return step


def step_with_wrench(env, actions, force, torque, **kw):
    """one SpecEnv.step with the external wrench force / torque ([E, N, 3], world frame; None: none)"""
    from oracle import spec
    if force is None and torque is None:
        return env.step(actions, **kw)
    shape = (env.E, env.N, 3)
    F = np.broadcast_to(np.asarray(0.0 if force is None else force, np.float64), shape)
    Tq = np.broadcast_to(np.asarray(0.0 if torque is None else torque, np.float64), shape)
    with mock.patch.object(spec.bm, 'bullet_step', _with_wrench(F, Tq)):
        return env.step(actions, **kw)


def _after_contact(F, Tq):
    """bullet_step with the external wrench added to the velocities AFTER the contact solve (a wrong kernel)"""
    from oracle import bullet_model as bm

    def step(pos, quat, vel, angvel, force_w, torque_w, P, dt=0.01, gravity=9.81, counts=None):
        v1, w1 = bm.unconstrained_velocities(quat, vel, angvel, force_w, torque_w, P, dt, gravity)
        if P.ground_contact or P.agent_contact:
            v1, w1 = bm.solve_contacts(pos, quat, v1, w1, P, dt, counts)
        R = bm.quat_to_mat(quat)
        v1 = np.clip(v1 + dt * F / P.mass, -P.max_coord_vel, P.max_coord_vel)
        w1 = np.clip(w1 + dt * bm.matvec(R, bm.matTvec(R, Tq) / P.inertia_diag()), -P.max_coord_vel, P.max_coord_vel)
        pos1, q1 = bm.integrate_positions(pos, quat, v1, w1, P, dt)
        return pos1, q1, v1, w1
    return step


def oracle_step(st, mode, actions, force, torque, wrong=None, T=1, **phys):
    """State after T oracle steps from the float32 state st (mode None: NO_ACTION) under the external wrench, or
    under one of the WRONG kernels."""
    from oracle import spec
    E, N = st['pos'].shape[:2]
    env = H.make_spec(E, N, mode or 'set_speeds', 0, float('inf'), st, **phys)
    F = np.asarray(force, np.float64)
    Tq = np.asarray(torque, np.float64)
    R = rotmat(st['quat'])
    if wrong == 'body_force':
        F = np.einsum('...ij,...j->...i', R, F)
    elif wrong == 'torque_unrotated':
        Tq = np.einsum('...ij,...j->...i', R, Tq)
    elif wrong == 'nan_zeroed' and actions is not None:
        bad = np.any(np.isnan(np.asarray(actions[0])), axis=-1)[..., None]
        F, Tq = np.where(bad, 0.0, F), np.where(bad, 0.0, Tq)
    for t in range(T):
        a = None if actions is None else actions[t]
        if wrong == 'none':
            env.step(a, nan_policy='agent_none')
        elif wrong == 'after_contact':
            with mock.patch.object(spec.bm, 'bullet_step', _after_contact(F, Tq)):
                env.step(a, nan_policy='agent_none')
        else:
            step_with_wrench(env, a, F, Tq, nan_policy='agent_none')
    return H.spec_state(env)


def bar_ratio(s0, ref, got, contact):
    """largest distance of `got` from `ref` in bars: the one-step delta bar in free flight, the contact band of the
    contact tests otherwise"""
    if contact:
        return V.band_ratio(got, ref)
    return max(H.delta_ratio(s0, ref, got).values())


def mode_actions(mode, E, N, st, seed=0, T=1):
    if mode is None:
        return None
    return H.random_actions(np.random.default_rng(seed), mode, T, E, N, start_pos=st['pos'])
