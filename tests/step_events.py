"""Scenes for the step's event outputs -- the sticky status word and the stats counters (include/mrs_b200.h) -- and the
NaN-action rule, plus the counts each kernel form must report for them, derived from the CPU oracle.  Shared by
test_cpu_step_events.py (oracle only) and test_gpu_step_events.py.

Every scene is built so that a plausible wrong count gives a different integer: several NaN or non-finite agents in
one warp-chunk (per-chunk counting gives 1, per-agent counting gives the number of agents), pairs and ground points
whose rows are in range but do not push (rows in range != rows that pushed), and free flight where every counter is
0.  Agents outside the units of a scene fly on a 2 m lattice at one height: no contact, no downwash between them."""
from __future__ import annotations

import ctypes as C

import numpy as np

import physics_variants as V

SPACING = 2.0
Z_AIR = 3.0
SCENES = ('free', 'separating', 'lifting', 'heap', 'nonfinite', 'nan_chunk')
E0 = 12             # envs of one scene block; larger batches tile the block (E0 is a multiple of every chunk's env count,
                    # and holds three warp-chunks at N = 5 and 8)

# unit kind -> (positions, velocities) around the unit's lattice cell at height Z_AIR.  The partners of a pair differ
# in height by 0.3 m or more: at a height difference near 0 the downwash (~ 1 / dz^2) is singular and float32 rounding
# of the positions decides the trajectory (helpers.downwash_sensitivity).
#   separate: 0.60 m apart along (0.8, 0, 0.6) (inside the contact range, sphere gap 0), moving apart at 0.6 m/s: rows
#             active, never push
#   press:    0.55 m apart along (0, 0.8, 0.6) (spheres overlap by 5 cm), closing at 0.2 m/s: a pushing pair
#   under:    the first agent 1 m straight below the second: it sits in the second's downwash
#   lift:     0.525 m (rim 11.5 mm above the ground: ground rows active), climbing at 1 m/s: rows never push
_SEP, _PRESS = np.array([0.8, 0.0, 0.6]), np.array([0.0, 0.8, 0.6])
UNITS = {
    'separate': (np.outer([-0.3, 0.3], _SEP), np.outer([-0.3, 0.3], _SEP)),
    'press': (np.outer([-0.275, 0.275], _PRESS), np.outer([0.1, -0.1], _PRESS)),
    'under': (np.array([[0.0, 0.0, 0.0], [0.0, 0.0, 1.0]]), np.zeros((2, 3))),
    'lift': (np.array([[0.0, 0.0, 0.525 - Z_AIR]]), np.array([[0.0, 0.0, 1.0]])),
}

# scene -> units of env e (row e % E0; rows not listed fly free)
LAYOUT = {
    'free': {},
    'separating': {0: ['separate'], 2: ['separate', 'separate'], 5: ['separate']},
    'lifting': {1: ['lift'], 2: ['lift', 'lift'], 6: ['lift']},
    'heap': {0: ['heap'], 2: ['heap', 'touchdown'], 3: ['touchdown'], 5: ['press'], 9: ['heap']},
    'nonfinite': {},
    'nan_chunk': {0: ['under'], 1: ['press'], 2: ['press'], 3: ['press']},
}
# physics a scene runs under: the heap with a cap of 3 sweeps, which binds in every heap env -- at the default cap its
# last sweeps end within a few percent of solver_tol, where float32 could stop one sweep earlier or later
SCENE_PHYS = {'heap': dict(solver_iters=3)}
# nan_chunk: (env, agent) of the NaN agents; the k-th gets its NaN in action component k % A.  Four in envs 0-3 (one
# warp-chunk at N = 5 and 8, two at N = 12 and 16), where pairs push: env 0 agent 0 flies under agent 1, env 1 agent 0
# is one side of a pushing pair.  One alone in env 6, whose warp-chunk (envs 4-7, 6-7 or 6 alone) has no other contact
# candidate: at every width only the NaN hands it to the contact path, so mrs_step_many with the NaN at step 1 parks
# it at step 1 (contact_chunks T - 1) and single steps count it once.  Envs 8-11 stay clean.
NAN_AGENTS = ((0, 0), (1, 0), (2, 2), (3, 1), (6, 1))
LONE_NAN_ENV = 6
# nonfinite: (env, agent) given +inf x and NaN vz: two in env 0 (one warp-chunk), one in env 4 (another one for N <= 8)
BAD_AGENTS = ((0, 1), (0, 2), (4, 0))


def chunk_envs(N):
    """envs per warp-chunk of the N <= 32 kernels (32 / pow2ceil(N)); None for the wide kernels"""
    return 32 // (1 << (N - 1).bit_length()) if N <= 32 else None


def _unit(kind, rng, k):
    if kind in UNITS:
        p, v = UNITS[kind]
        return p + np.array([0.0, 0.0, Z_AIR]), v.copy()
    return V._unit(kind, rng, k)          # heap (2 x 2 landing agents), touchdown (one landing agent)


def make_scene(kind, N, E=E0, seed=0):
    """float32 start state [E, N, ...] of a scene: the block of E0 envs, repeated (and cut) to E envs."""
    from scipy.spatial.transform import Rotation
    rng = np.random.default_rng(seed * 1000 + N)
    cols = int(np.ceil(np.sqrt(N)))
    pos = np.zeros((E0, N, 3))
    vel = rng.uniform(-0.2, 0.2, (E0, N, 3))
    for e in range(E0):
        units = LAYOUT[kind].get(e, [])
        i = k = 0
        while i < N:
            p, v = _unit(units[k], rng, k) if k < len(units) else _unit('free', rng, k)
            if i + len(p) > N:
                p, v = _unit('free', rng, k)
            c = np.array([k % cols, k // cols, 0.0]) * SPACING
            pos[e, i:i + len(p)] = p + c
            vel[e, i:i + len(p)] = v
            i += len(p)
            k += 1
    rpy = np.concatenate([rng.uniform(-0.05, 0.05, (E0 * N, 2)), rng.uniform(-np.pi, np.pi, (E0 * N, 1))], axis=1)
    quat = Rotation.from_euler('xyz', rpy).as_quat().reshape(E0, N, 4)
    st = dict(pos=pos, quat=quat, vel=vel, angvel=rng.uniform(-0.1, 0.1, (E0, N, 3)))
    if kind == 'nonfinite':
        for e, a in BAD_AGENTS:
            pos[e, a, 0] = np.inf
            vel[e, a, 2] = np.nan
    return {k: np.ascontiguousarray(np.tile(v.astype(np.float32), (-(-E // E0), 1, 1))[:E]) for k, v in st.items()}


def plant_nans(actions, N, steps):
    """actions [T, E, N, A] (float32, modified in place): the NaN agents get a NaN in component k % A at each of
    `steps`"""
    A = actions.shape[-1]
    for t in steps:
        for k, (e, a) in enumerate(NAN_AGENTS):
            actions[t, e::E0, a, k % A] = np.nan
    return actions


# ------------------------------------------------------------------------------ the library's own thresholds
def thresholds():
    """(gnd_skip_z, lim2) of the default config, from the library's own derivation (mrs_debug_derived)"""
    from mrsgym_b200 import _abi
    d = _abi.Derived()
    _abi.check(_abi.lib().mrs_debug_derived(C.byref(_abi.default_config()), C.byref(d), C.sizeof(d)), 'mrs_debug_derived')
    return float(d.gnd_skip_z), float(d.lim2)


# ------------------------------------------------------------------------------ oracle runs and expected counts
def oracle_run(st, mode, actions, T, K=0, comm_range=float('inf'), **phys):
    """T oracle steps (actions [T, E, N, A] or None; NaN entries follow the device rule).  Returns the final state
    and, per step, the pre-step positions, the NaN mask, the contact counts and the non-finite mask after the step."""
    import helpers as H
    E, N = st['pos'].shape[:2]
    env = H.make_spec(E, N, mode or 'set_speeds', K, comm_range, st, **phys)
    steps = []
    for t in range(T):
        counts = {}
        pre = env.pos.copy()
        a = None if actions is None else actions[t]
        nan = np.zeros((E, N), bool) if a is None else np.any(np.isnan(a), axis=-1)
        env.step(a, nan_policy='agent_none', counts=counts)
        fin = np.all(np.isfinite(np.concatenate([env.pos, env.quat, env.vel, env.angvel], -1)), -1)
        steps.append(dict(pre=pre, nan=nan, counts=counts, bad=~fin, rpm=env.last['rpm'].copy()))
    return env, steps


def expected_stats(steps, N, gnd_skip_z, lim2, form='single', nan_hands_off=True):
    """The stats a step form must report for oracle steps (oracle_run).  form: 'single' (single-step launches and the
    chained rollout) or 'many' (the MANY kernels of mrs_step_many, N <= 32: a parked chunk counts T - first step).
    nan_hands_off=False: contact_chunks of a kernel whose NaN actions did not send a chunk to the contact path (the
    tests show that the scenes tell the two apart)."""
    E = steps[0]['pre'].shape[0]
    T = len(steps)
    out = dict(agent_contact_rows=0, ground_contacts=0, nonfinite=0, nan_actions=0, contact_chunks=0, solver_sweeps=0)
    gpw = chunk_envs(N)
    cand = np.zeros((T, E), bool)
    for t, s in enumerate(steps):
        c = s['counts']
        out['agent_contact_rows'] += int(c['pair_rows'].sum()) if c else 0
        out['ground_contacts'] += int(c['ground'].sum()) if c else 0
        out['nonfinite'] += int(s['bad'].sum())
        out['nan_actions'] += int(s['nan'].sum())
        p = s['pre']
        with np.errstate(invalid='ignore'):
            low = np.any(p[..., 2] < gnd_skip_z, axis=-1)
            d = p[:, :, None, :] - p[:, None, :, :]
            d2 = np.sum(d * d, -1)
            d2[:, np.arange(N), np.arange(N)] = np.inf
            near = np.any(d2 < lim2, axis=(-2, -1))
        cand[t] = low | near | (np.any(s['nan'], -1) & nan_hands_off)
    if gpw is None:
        return out
    nch = (E + gpw - 1) // gpw
    ch = np.zeros((T, nch), bool)
    sweeps = np.zeros((T, nch), np.int64)
    for t, s in enumerate(steps):
        c = s['counts']
        for k in range(nch):
            ch[t, k] = cand[t, k * gpw:(k + 1) * gpw].any()
            if c:
                sw = np.where(c['active'], c['sweeps'], 0)[k * gpw:(k + 1) * gpw]
                sweeps[t, k] = sw.max()
    if form == 'many':
        first = np.where(ch.any(0), np.argmax(ch, axis=0), T)
        out['contact_chunks'] = int(np.sum(T - first))
    else:
        out['contact_chunks'] = int(ch.sum())
    out['solver_sweeps'] = int(sweeps.sum())
    return out


def margins(steps, gnd_skip_z, lim2, N):
    """The smallest distance of any decision a count depends on from its threshold: pre-step heights from gnd_skip_z
    and squared pair distances from lim2 (finite agents only), and every nonzero final normal impulse"""
    out = dict(z=np.inf, d2=np.inf, lam=np.inf)
    for s in steps:
        p = s['pre']
        ok = np.all(np.isfinite(p), -1)
        z = np.abs(p[..., 2] - gnd_skip_z)[ok]
        out['z'] = min(out['z'], float(z.min()) if z.size else np.inf)
        with np.errstate(invalid='ignore'):
            d = p[:, :, None, :] - p[:, None, :, :]
            d2 = np.sum(d * d, -1)
        both = ok[:, :, None] & ok[:, None, :] & ~np.eye(N, dtype=bool)
        if both.any():
            out['d2'] = min(out['d2'], float(np.abs(d2 - lim2)[both].min()))
        c = s['counts']
        if c:
            lams = [c['g_lam'].ravel()] + [l.ravel() for l in c['p_lam']]
            lam = np.concatenate(lams)
            lam = lam[lam != 0.0]
            if lam.size:
                out['lam'] = min(out['lam'], float(lam.min()))
    return out
