"""GPU parity tests proper: the CUDA path (through the C ABI, via mrsgym_b200.Swarm / MRS)
against the CPU oracle on identical seeded inputs and against the committed golden vectors that
the reference's own Python produced (tests/golden/ref_*.npz).

Tolerances (BASELINE.json north_star):
  * adjacency A: bit-exact given identical positions;
  * one-step state deltas: |d_gpu - d_ref| <= 1e-4 * |d_ref| + floor, the floor being the float32
    resolution of the stored quantity (the GPU state is float32, Bullet's is float64):
    pos max(5e-7 m, 1 ulp of the coordinate), vel 5e-7 m/s, angvel 1e-5 rad/s, quaternion 3e-7;
  * 100-step free-flight trajectories: position <= 1e-3 m, attitude <= 1e-3 rad;
    contact trajectories (approximate by design): position <= 5e-2 m.
"""
import glob
import os

import numpy as np
import pytest
import torch

import helpers as H
from conftest import GOLDEN
from oracle import spec

pytestmark = pytest.mark.gpu


def _swarm(E, N, mode, K=0, comm_range=float('inf'), layout=None, **kw):
    import mrsgym_b200 as M
    layout = M._abi.X_POS_VEL if layout is None else layout
    return M.Swarm(E, N, K, mode, layout, comm_range, **kw)


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


# ------------------------------------------------------------------------------ adjacency
@pytest.mark.parametrize('E,N,R', [(1, 3, 1.5), (64, 8, 2.0), (16, 32, 2.0), (7, 5, 0.9), (3, 33, 1.7), (5, 64, 2.0),
                                   (9, 36, 1.2), (3, 100, float('inf')), (700, 64, 2.0), (2, 124, 1.6),
                                   (2, 128, 2.0), (1, 500, 3.0), (1, 4096, 2.0), (4, 16, float('inf')),
                                   (1, 256, float('inf'))])
def test_adjacency_bit_exact_vs_torch_cpu(E, N, R):
    rng = np.random.default_rng(1000 + N)
    # lattice points (distances hit COMM_RANGE exactly) + jitter on half of the envs
    pos = H.grid_positions(E, N, spacing=0.5, z0=1.0, jitter=0.0)
    pos[E // 2:] += rng.uniform(-0.3, 0.3, pos[E // 2:].shape)
    pos32 = pos.astype(np.float32)
    sw = _swarm(E, N, 'set_speeds', 0, R)
    A = sw.adjacency(_dev(pos32)).cpu()
    ref = H.torch_cpu_adjacency(pos32, R)
    assert A.shape == ref.shape
    assert int((A != ref).sum()) == 0
    np.testing.assert_array_equal(A.numpy(), spec.adjacency(pos32, R))
    assert torch.equal(A, A.transpose(-1, -2)) and float(torch.diagonal(A, dim1=-2, dim2=-1).abs().sum()) == 0.0


def test_adjacency_threshold_edges():
    """distances one float32 ulp either side of COMM_RANGE, NaN positions, zero range"""
    R = 2.0
    base = np.zeros((1, 8, 3), np.float32)
    d = np.float32(R)
    offs = [np.nextafter(d, np.float32(0)), d, np.nextafter(d, np.float32(10)), np.float32(1.9999), np.float32(2.0001)]
    for i, o in enumerate(offs):
        base[0, i + 1, 0] = o
    base[0, 7] = np.nan
    sw = _swarm(1, 8, 'set_speeds', 0, R)
    A = sw.adjacency(_dev(base)).cpu()
    assert int((A != H.torch_cpu_adjacency(base, R)).sum()) == 0
    assert float(A[0, 7].sum()) == 0.0
    for Rz in (0.0, 1e-30, 1e30):
        sw = _swarm(1, 8, 'set_speeds', 0, Rz)
        A = sw.adjacency(_dev(base)).cpu()
        assert int((A != H.torch_cpu_adjacency(base, Rz)).sum()) == 0


# ------------------------------------------------------------------------------ one step
@pytest.mark.parametrize('mode', H.MODES)
@pytest.mark.parametrize('E,N', [(64, 8), (5, 3), (8, 32), (3, 40), (2, 100), (1, 300)])
def test_one_step_delta_vs_oracle(mode, E, N):
    rng = np.random.default_rng(sum(map(ord, mode)) * 1000 + E * 37 + N)
    st = H.random_state(rng, E, N, spacing=0.9)
    act = H.random_actions(rng, mode, 1, E, N, start_pos=st['pos'])
    sw = _swarm(E, N, mode, 1, 1.5)
    H.upload_state(sw, st)
    sw.step(_dev(act[0]))
    torch.cuda.synchronize()
    g1 = H.read_state(sw)
    ref = H.make_spec(E, N, mode, 1, 1.5, st)
    Xr, Ar = ref.step(act[0])
    H.check_delta('%s E%d N%d' % (mode, E, N), st, g1, H.spec_state(ref))
    # observation written by the same launch: X = float32 state, A = adjacency of ITS positions
    X = sw.X_window()[0].cpu().numpy()
    np.testing.assert_array_equal(X[..., :3], g1['pos'].astype(np.float32))
    np.testing.assert_array_equal(X[..., 3:], g1['vel'].astype(np.float32))
    A = sw.A_window()[0].cpu().numpy()
    np.testing.assert_array_equal(A, spec.adjacency(X[..., :3], 1.5))
    assert sw.read_status() == 0


@pytest.mark.parametrize('mode', ['set_target_vel', 'set_target_pos'])
def test_controller_state_carries_over_steps(mode):
    """second and third controller calls use the stored PID planes (integrators, d_vel_e, last_*)"""
    E, N, T = 16, 8, 3
    rng = np.random.default_rng(77)
    st = H.random_state(rng, E, N)
    act = H.random_actions(rng, mode, T, E, N, start_pos=st['pos'])
    sw = _swarm(E, N, mode, 0)
    H.upload_state(sw, st)
    ref = H.make_spec(E, N, mode, 0, float('inf'), st)
    for t in range(T):
        s0 = H.read_state(sw)
        # restart the oracle from the GPU's float32 state so that each step is a one-step test
        ref.set_state(pos=s0['pos'], quat=s0['quat'], vel=s0['vel'], angvel=s0['angvel'])
        sw.step(_dev(act[t]))
        ref.step(act[t])
        H.check_delta('%s step %d' % (mode, t), {k: v.astype(np.float32) for k, v in s0.items()}, H.read_state(sw),
                     H.spec_state(ref))


def test_no_action_step_is_free_fall():
    E, N = 4, 8
    rng = np.random.default_rng(5)
    st = H.random_state(rng, E, N)
    sw = _swarm(E, N, 'set_speeds')
    H.upload_state(sw, st)
    sw.set_action_type(None)
    sw.step(None)
    ref = H.make_spec(E, N, 'set_speeds', 0, float('inf'), st)
    ref.step(None)
    H.check_delta('no action', st, H.read_state(sw), H.spec_state(ref))


# ------------------------------------------------------------------------------ contact
# One-step band of the contact tests.  A normal row's bias is penetration / dt (x erp2): the float32 resolution of a
# height near 0.5 m (6e-8 m) is 6e-6 m/s of bias; through the point's effective mass (K ~ 140 / kg) and the angular
# Jacobian (|a| / I ~ 1700) that is up to ~1e-4 rad/s of angular velocity per row, and the solver stops sweeping
# below solver_tol = 1e-6 m/s wherever float32 and float64 happen to cross it.
CONTACT_BAND = (('vel', 3e-4), ('pos', 3e-6), ('angvel', 1e-3))


@pytest.mark.parametrize('N', [4, 16, 48, 200])
def test_contact_one_step(N):
    """ground landing + AGENT_RADIUS sphere-sphere rows (C3 regime: 0.55 m spacing < 2*0.3)"""
    E = 32
    rng = np.random.default_rng(300 + N)
    st = H.random_state(rng, E, N, spacing=0.55, z0=0.53, jitter=0.03, tilt=0.05, vel=0.5, angvel=0.2)
    st['vel'][..., 2] -= 1.0
    act = H.random_actions(rng, 'set_control', 1, E, N)
    sw = _swarm(E, N, 'set_control', 0)
    H.upload_state(sw, st)
    sw.step(_dev(act[0]))
    ref = H.make_spec(E, N, 'set_control', 0, float('inf'), st)
    ref.step(act[0])
    g1, r1 = H.read_state(sw), H.spec_state(ref)
    # contact rows switch on thresholds (dist < margin, rhs > 0): allow a float32-sized band
    for k, tol in CONTACT_BAND:
        assert np.max(np.abs(g1[k] - r1[k])) <= tol, k
    stats = sw.read_stats()
    assert stats['agent_contact_rows'] > 0 and stats['ground_contacts'] > 0


def _heap_state(E, N, side, rng):
    g = np.array([[i, j] for i in range(side) for j in range(side)][:N], float)
    pos = np.zeros((E, N, 3))
    pos[..., :2] = g * 0.5 + rng.uniform(-0.02, 0.02, (E, N, 2))
    pos[..., 2] = 0.56 + rng.uniform(0, 0.05, (E, N))
    from scipy.spatial.transform import Rotation as R
    rpy = np.concatenate([rng.uniform(-0.1, 0.1, (E * N, 2)), rng.uniform(-1, 1, (E * N, 1))], 1)
    st = dict(pos=pos, quat=R.from_euler('xyz', rpy).as_quat().reshape(E, N, 4), vel=np.zeros((E, N, 3)),
              angvel=np.zeros((E, N, 3)))
    return {k: v.astype(np.float32) for k, v in st.items()}


@pytest.mark.parametrize('N,side', [(16, 4), (48, 7)])
def test_resting_heap_stays_put(N, side):
    """Agents dropped 0.5 m apart (contact spheres of 2 x 0.3 m overlap) are pushed apart to 0.6 m by the
    sequential-impulse solver and then REST: within a millimetre over 1000 further steps, no jitter, on the
    rim points of the collision cylinder (VERDICT r1 #2).  N = 16: in-warp solve, N = 48: contact_env_kernel."""
    E = 6
    st = _heap_state(E, N, side, np.random.default_rng(5))
    sw = _swarm(E, N, None, 0)
    H.upload_state(sw, st)
    for t in range(600):
        sw.step(None)
    p0 = sw.get_pos().clone()
    for t in range(1000):
        sw.step(None)
    p1 = sw.get_pos()
    assert float((p1 - p0).abs().max()) < 1e-3
    d = torch.cdist(p1, p1) + 9 * torch.eye(N, device='cuda')
    assert float(d.min()) > 0.6 - 1e-3
    assert float((p1[..., 2] - 0.51349).abs().max()) < 2e-5
    assert float(sw.get_vel().abs().max()) < 1e-3
    assert sw.read_status() == 0
    # the first 60 steps against the oracle (contact-grade tolerance)
    sw2 = _swarm(E, N, None, 0)
    H.upload_state(sw2, st)
    ref = H.make_spec(E, N, 'set_speeds', 0, float('inf'), st)
    for t in range(60):
        sw2.step(None)
        ref.step(None)
    assert np.max(np.abs(H.read_state(sw2)['pos'] - ref.pos)) < 5e-3


@pytest.mark.parametrize('N', [3, 40])
def test_tilted_landing_rights_itself(N):
    """The ground impulses act at the rim points of the collision cylinder: a quad that lands tilted is turned
    flat, one that lands upside down rests on its top face."""
    from scipy.spatial.transform import Rotation as R
    E = 4
    pos = H.grid_positions(E, N, spacing=1.0, z0=0.62, jitter=0.0)
    pos[..., 2] = 0.62
    rpy = np.tile(np.array([0.4, 0.2, 0.1]), (E * N, 1))
    rpy[1::2] = np.array([np.pi - 0.3, 0.1, 0.0])
    st = dict(pos=pos, quat=R.from_euler('xyz', rpy).as_quat().reshape(E, N, 4), vel=np.zeros((E, N, 3)),
              angvel=np.zeros((E, N, 3)))
    st = {k: v.astype(np.float32) for k, v in st.items()}
    sw = _swarm(E, N, None, 0)
    H.upload_state(sw, st)
    for t in range(200):
        sw.step(None)
    q = sw.get_quat().reshape(-1, 4)
    R22 = 1 - 2 * (q[:, 0] ** 2 + q[:, 1] ** 2)
    assert float((R22[0::2] - 1).abs().max()) < 1e-5 and float((R22[1::2] + 1).abs().max()) < 1e-5
    assert float((sw.get_pos()[..., 2] - 0.51349).abs().max()) < 2e-5


# ------------------------------------------------------------------------------ goldens
TRAJ = sorted(glob.glob(os.path.join(GOLDEN, 'ref_*.npz')))


@pytest.mark.parametrize('path', TRAJ, ids=[os.path.basename(f)[4:-4] for f in TRAJ])
def test_trajectory_vs_reference_golden(path):
    """GPU rollout from the golden start state with the golden actions vs the trajectory the
    reference's own Python produced (oracle/make_golden.py)."""
    g = np.load(path)
    N, K, T, mode = int(g['N']), int(g['K']), int(g['T']), str(g['mode'])
    R = float(g['comm_range'])
    st = dict(pos=g['start_pos'][None], quat=g['start_quat'][None], vel=g['start_vel'][None],
              angvel=g['start_angvel'][None])
    st = {k: v.astype(np.float32) for k, v in st.items()}
    sw = _swarm(1, N, mode, K, R, agent_radius=float(g['agent_radius']), dt=float(g['dt']), gravity=float(g['gravity']))
    none_steps = set(int(t) for t in g['none_steps'])
    H.upload_state(sw, st)
    contact = 'contact' in path
    ptol, atol = (5e-2, 5e-2) if contact else (1e-3, 1e-3)
    # free flight is tightly checked up to the first downwash singularity of the reference
    # trajectory (an agent crossing just under another: force ~ 1/dz^2); from there on the
    # reference dynamics itself amplifies float32 rounding and the contact-grade tolerance applies
    t_sing = H.first_singular_step(g)
    worst_p = worst_a = 0.0
    for t in range(T):
        if t == t_sing:
            assert worst_p <= ptol and worst_a <= atol, (worst_p, worst_a)
            ptol, atol = 5e-2, 5e-2
        if t in none_steps:                 # MRS.step(None): no forces on this step
            sw.set_action_type(None)
            sw.step(None)
            sw.set_action_type(mode)
        else:
            sw.step(_dev(g['actions'][t][None]))
        s = H.read_state(sw)
        worst_p = max(worst_p, float(np.abs(s['pos'][0] - g['pos'][t]).max()))
        worst_a = max(worst_a, float(H.quat_angle(s['quat'][0], g['quat'][t]).max()))
        if t == 0 and not contact:
            # first step: rpm-level agreement shows up as a tight velocity match
            assert np.abs(s['vel'][0] - g['vel'][0]).max() < 2e-6
            assert np.abs(s['angvel'][0] - g['angvel'][0]).max() < 5e-5
    assert worst_p <= ptol, 'position drift %.3g m' % worst_p
    assert worst_a <= atol, 'attitude drift %.3g rad' % worst_a
    # observation windows of the last step: ring order newest-first, K+1 deep
    X = sw.X_window()[:, 0].cpu().numpy()
    assert X.shape == g['X'][-1].shape
    np.testing.assert_allclose(X, g['X'][-1], atol=20 * ptol, rtol=0)
    A = sw.A_window()[:, 0].cpu().numpy()
    assert A.shape == g['A'][-1].shape
    for k in range(K + 1):
        np.testing.assert_array_equal(A[k], spec.adjacency(X[k][:, :3], R))
    assert sw.read_status() == 0


# ------------------------------------------------------------------------------ rings / many / shards
def test_ring_semantics_match_reference():
    """X padded with copies of X0, A padded with zeros, newest first, independent heads
    (MRS.py:87-114; SURVEY.md rows a14/a15), across several tape wrap-arounds."""
    E, N, K, T = 3, 8, 3, 40
    rng = np.random.default_rng(11)
    st = H.random_state(rng, E, N)
    act = H.random_actions(rng, 'set_speeds', T, E, N)
    sw = _swarm(E, N, 'set_speeds', K, 1.2, tape_slots=2 * K + 2)
    H.upload_state(sw, st)
    X0 = sw.X_window().clone()
    assert all(torch.equal(X0[0], X0[k]) for k in range(K + 1))
    newest_X, newest_A = [X0[0]], []
    for t in range(T):
        sw.step(_dev(act[t]))
        Xw, Aw = sw.X_window().clone(), sw.A_window().clone()
        newest_X.insert(0, Xw[0])
        newest_A.insert(0, Aw[0])
        for k in range(K + 1):
            want = newest_X[k] if k < len(newest_X) else newest_X[-1]
            assert torch.equal(Xw[k], want), (t, k)
            if k < len(newest_A):
                assert torch.equal(Aw[k], newest_A[k]), (t, k)
            else:
                assert float(Aw[k].abs().sum()) == 0.0, (t, k)


@pytest.mark.parametrize('N,mode', [(8, 'set_speeds'), (32, 'set_target_pos'), (3, 'set_target_vel'), (40, 'set_control'),
                                    (16, 'set_control'), (150, 'set_force')])
def test_step_many_equals_repeated_step(N, mode):
    E, K, T = 33, 2, 23
    rng = np.random.default_rng(21)
    st = H.random_state(rng, E, N)
    act = _dev(H.random_actions(rng, mode, T, E, N, start_pos=st['pos']))
    a = _swarm(E, N, mode, K, 1.5, tape_slots=12)
    b = _swarm(E, N, mode, K, 1.5, tape_slots=12)
    H.upload_state(a, st)
    H.upload_state(b, st)
    for t in range(T):
        a.step(act[t])
    b.step_many(act, T)
    if N > 32:
        # wide path: mrs_step_many issues the same per-step kernels -> bit for bit
        assert torch.equal(a.state, b.state)
        assert torch.equal(a.ctrl.nan_to_num(nan=-7.0), b.ctrl.nan_to_num(nan=-7.0))
        assert torch.equal(a.X_window(), b.X_window()) and torch.equal(a.A_window(), b.A_window())
        return
    # N <= 32: the multi-step kernel (state in registers across steps) is compiled separately from the single-step
    # kernel, so the compiler's FMA contraction may differ: float32 rounding level, not bit for bit
    # (mrs_rollout -- chained single-step launches -- is the bit-identical multi-step form, see
    # test_chained_rollout_equals_plain_steps)
    sa, sb = a.state.double(), b.state.double()
    assert float((sa - sb).abs().max()) < 2e-5, float((sa - sb).abs().max())
    ca, cb = a.ctrl.nan_to_num(nan=-7.0).double(), b.ctrl.nan_to_num(nan=-7.0).double()
    assert float(((ca - cb).abs() / (1.0 + ca.abs())).max()) < 2e-5
    assert float((a.X_window() - b.X_window()).abs().max()) < 2e-5
    # every A slice is the exact adjacency of the X slice written with it
    from oracle import spec
    Xb, Ab = b.X_window().cpu().numpy(), b.A_window().cpu().numpy()
    for k in range(K + 1):
        assert np.array_equal(Ab[k], spec.adjacency(Xb[k][..., :3], 1.5)), k


@pytest.mark.parametrize('N', [8, 40, 130])
def test_env_shards_are_independent(N):
    """1-GPU result == concatenation of per-shard results, bit for bit (SURVEY.md §8e)."""
    import mrsgym_b200 as M
    E, T = 50, 5
    rng = np.random.default_rng(31)
    st = H.random_state(rng, E, N)
    act = H.random_actions(rng, 'set_target_vel', T, E, N)
    full = _swarm(E, N, 'set_target_vel', 1, 1.5)
    H.upload_state(full, st)
    full.step_many(_dev(act), T)
    parts = []
    for r in range(3):
        lo, hi = M.shard_range(E, r, 3)
        sh = _swarm(hi - lo, N, 'set_target_vel', 1, 1.5)
        H.upload_state(sh, {k: v[lo:hi] for k, v in st.items()})
        sh.step_many(_dev(act[:, lo:hi]), T)
        parts.append(sh)
    S = full.S
    cat = torch.cat([p.state for p in parts], dim=1)
    assert torch.equal(full.state, cat)
    assert torch.equal(full.A_window(), torch.cat([p.A_window() for p in parts], dim=1))
    assert torch.equal(full.X_window(), torch.cat([p.X_window() for p in parts], dim=1))


def test_set_state_euler_and_mask():
    from scipy.spatial.transform import Rotation as R
    E, N = 6, 5
    rng = np.random.default_rng(41)
    sw = _swarm(E, N, 'set_speeds')
    pos = rng.uniform(-2, 2, (E, N, 3)).astype(np.float32)
    ori = rng.uniform(-1.4, 1.4, (E, N, 3)).astype(np.float32)
    vel = rng.uniform(-1, 1, (E, N, 3)).astype(np.float32)
    sw.set_state(pos=pos, ori=ori, vel=vel, angvel=None)
    s = H.read_state(sw)
    np.testing.assert_array_equal(s['pos'].astype(np.float32), pos)
    q = R.from_euler('xyz', ori.reshape(-1, 3).astype(np.float64)).as_quat().reshape(E, N, 4)
    assert np.max(H.quat_angle(s['quat'], q)) < 1e-6
    np.testing.assert_allclose(sw.get_ori().cpu().numpy(), ori, atol=2e-6)
    # masked update touches only the selected envs; None keeps the component
    mask = np.array([1, 0, 0, 1, 0, 0], np.uint8)
    sw.set_state(pos=np.zeros((E, N, 3), np.float32), env_mask=mask)
    s2 = H.read_state(sw)
    assert np.all(s2['pos'][mask == 1] == 0) and np.array_equal(s2['pos'][mask == 0], s['pos'][mask == 0])
    np.testing.assert_array_equal(s2['vel'], s['vel'])
    np.testing.assert_array_equal(s2['quat'], s['quat'])


def test_step_host_roundtrip():
    E, N, K = 128, 8, 1
    rng = np.random.default_rng(51)
    st = H.random_state(rng, E, N)
    act = H.random_actions(rng, 'set_speeds', 1, E, N)
    a = _swarm(E, N, 'set_speeds', K, 2.0)
    b = _swarm(E, N, 'set_speeds', K, 2.0)
    H.upload_state(a, st)
    H.upload_state(b, st)
    a.step(_dev(act[0]))
    ah = torch.from_numpy(act[0]).pin_memory()
    Xh = torch.empty(E, N, 6).pin_memory()
    Ah = torch.empty(E, N, N).pin_memory()
    b.step_host(ah, torch.empty(E, N, 4, device='cuda'), Xh, Ah)
    assert torch.equal(a.state, b.state)
    assert torch.equal(Xh, a.X_window()[0].cpu()) and torch.equal(Ah, a.A_window()[0].cpu())


@pytest.mark.parametrize('N,mode', [(8, 'set_speeds'), (40, 'set_target_vel')])
def test_graph_rollout_ring_mode_equals_steps(N, mode):
    """capture_rollout: CUDA graph of T steps on a ring tape (tape_slots = T, nothing is ever moved);
    two replays == 2 T plain steps, bit for bit, windows included"""
    E, K, T = 48, 3, 8
    rng = np.random.default_rng(53)
    st = H.random_state(rng, E, N)
    act = _dev(H.random_actions(rng, mode, T, E, N, start_pos=st['pos']))
    a = _swarm(E, N, mode, K, 1.5)
    b = _swarm(E, N, mode, K, 1.5, tape_slots=T, ring=True)
    H.upload_state(a, st)
    H.upload_state(b, st)
    roll = b.capture_rollout(act, T)
    H.upload_state(b, st)                     # the capture warm-up stepped b: start again from st
    b.ctrl.copy_(a.ctrl)
    for rep in range(2):
        for t in range(T):
            a.step(act[t])
        roll.replay()
        assert torch.equal(a.state, b.state), rep
        assert torch.equal(a.X_window(), b.X_window()) and torch.equal(a.A_window(), b.A_window()), rep
    with pytest.raises(ValueError):
        b.capture_rollout(act[:5], 5)


def test_rollout_host_pipelined_equals_steps():
    E, N, K, T = 256, 8, 2, 37
    rng = np.random.default_rng(52)
    st = H.random_state(rng, E, N)
    act = H.random_actions(rng, 'set_speeds', T, E, N)
    a = _swarm(E, N, 'set_speeds', K, 2.0, tape_slots=16)
    b = _swarm(E, N, 'set_speeds', K, 2.0, tape_slots=16)
    H.upload_state(a, st)
    H.upload_state(b, st)
    Xs, As = [], []
    for t in range(T):
        a.step(_dev(act[t]))
        Xs.append(a.X_window()[0].cpu())
        As.append(a.A_window()[0].cpu())
    ah = torch.from_numpy(act).pin_memory()
    Xh = torch.empty(T, E, N, 6).pin_memory()
    Ah = torch.empty(T, E, N, N).pin_memory()
    b.rollout_host(ah, torch.empty(2, E, N, 4, device='cuda'), Xh, Ah)
    assert torch.equal(a.state, b.state)
    assert torch.equal(Xh, torch.stack(Xs)) and torch.equal(Ah, torch.stack(As))
    assert torch.equal(a.X_window(), b.X_window()) and torch.equal(a.A_window(), b.A_window())


def test_full_size_properties_c5():
    """BASELINE configs[4] at full size (65536 envs x 8): properties that need no oracle run --
    A symmetric with zero diagonal and equal to the oracle adjacency of the GPU's own X on a
    sample of envs; unit quaternions; every env of a replicated batch evolves identically."""
    E, N, K, T = 65536, 8, 3, 20
    rng = np.random.default_rng(61)
    one = H.random_state(rng, 1, N, spacing=1.0, z0=2.5)
    st = {k: np.repeat(v, E, axis=0) for k, v in one.items()}
    a1 = H.random_actions(rng, 'set_speeds', T, 1, N)
    act = _dev(np.repeat(a1, E, axis=1))
    sw = _swarm(E, N, 'set_speeds', K, 2.0)
    H.upload_state(sw, st)
    sw.step_many(act, T)
    A = sw.A_window()
    X = sw.X_window()
    assert torch.equal(A, A.transpose(-1, -2))
    assert float(torch.diagonal(A, dim1=-2, dim2=-1).abs().sum()) == 0.0
    assert torch.equal(X, X[:, :1].expand_as(X)) and torch.equal(A, A[:, :1].expand_as(A))
    q = sw.get_quat()
    assert float((q.norm(dim=-1) - 1).abs().max()) < 1e-5
    idx = torch.tensor([0, 1, E // 2, E - 1])
    Xs = X[:, idx].cpu().numpy()
    np.testing.assert_array_equal(A[:, idx].cpu().numpy(), spec.adjacency(Xs[..., :3], 2.0))
    # and the replicated env agrees with the oracle trajectory
    ref = H.make_spec(1, N, 'set_speeds', K, 2.0, one)
    for t in range(T):
        ref.step(a1[t])
    assert np.abs(sw.get_pos()[0].cpu().numpy() - ref.pos[0]).max() < 1e-4
    assert sw.read_status() == 0


# ------------------------------------------------------------------------------ BASELINE configs at full size
def _subset_vs_oracle(E, N, mode, K, R, T, spacing, z0, pick, seed, ptol, vtol, step_many=True, noise=None):
    """Envs are independent: run the GPU on the full batch and the oracle on a handful of its envs
    with the same inputs; trajectories must agree within the free-flight / contact tolerance."""
    rng = np.random.default_rng(seed)
    st = H.random_state(rng, E, N, spacing=spacing, z0=z0, jitter=0.1, tilt=0.02, vel=0.05, angvel=0.05)
    act = H.random_actions(rng, mode, T, E, N, start_pos=st['pos'])
    if mode == 'set_control':
        act[::5, :, :, 1:] /= 60.0                      # keep C3 in the regular mixer branch mostly
    if noise is not None:
        act = noise(rng, act)
    sw = _swarm(E, N, mode, K, R)
    H.upload_state(sw, st)
    if step_many:
        sw.step_many(_dev(act), T)
    else:
        for t in range(T):
            sw.step(_dev(act[t]))
    g = H.read_state(sw)
    sub = {k: v[pick] for k, v in st.items()}
    ref = H.make_spec(len(pick), N, mode, K, R, sub)
    for t in range(T):
        Xr, Ar = ref.step(act[t][pick])
    assert np.abs(g['pos'][pick] - ref.pos).max() <= ptol
    assert np.abs(g['vel'][pick] - ref.vel).max() <= vtol
    X = sw.X_window()[:, pick].cpu().numpy()
    A = sw.A_window()[:, pick].cpu().numpy()
    for k in range(K + 1):
        np.testing.assert_array_equal(A[k], spec.adjacency(X[k][..., :3], R))
    assert sw.read_status() == 0
    return sw


def test_full_size_c2_swarm32_target_pos():
    """BASELINE configs[1]: 256 envs x 32 agents, set_target_pos, K_HOPS=3, COMM_RANGE=2.0"""
    _subset_vs_oracle(256, 32, 'set_target_pos', 3, 2.0, T=15, spacing=1.0, z0=3.0, pick=[0, 17, 255], seed=71,
                      ptol=1e-4, vtol=2e-3)


def test_full_size_c3_control_with_contact():
    """BASELINE configs[2]: 4096 envs x 16 agents, set_control, ground + agent-agent contact"""
    sw = _subset_vs_oracle(4096, 16, 'set_control', 0, float('inf'), T=12, spacing=0.58, z0=0.56, pick=[0, 1000, 4095],
                           seed=72, ptol=5e-2, vtol=0.5, step_many=False)
    stats = sw.read_stats()
    assert stats['agent_contact_rows'] > 0 and stats['ground_contacts'] > 0


def test_full_size_c4_single_env_4096_agents():
    """BASELINE configs[3]: one env of 4096 agents, set_force, adjacency dominated -- one step against the
    oracle (float64 pair arrays of 4096^2), A bit-exact on the GPU's own positions"""
    E, N, R = 1, 4096, 2.0
    rng = np.random.default_rng(73)
    st = H.random_state(rng, E, N, spacing=1.0, z0=2.0, jitter=0.2, tilt=0.02, vel=0.1, angvel=0.1)
    act = H.random_actions(rng, 'set_force', 1, E, N)
    sw = _swarm(E, N, 'set_force', 0, R)
    H.upload_state(sw, st)
    sw.step(_dev(act[0]))
    ref = H.make_spec(E, N, 'set_force', 0, R, st)
    ref.step(act[0])
    H.check_delta('c4', st, H.read_state(sw), H.spec_state(ref))
    X = sw.X_window()[0].cpu().numpy()
    A = sw.A_window()[0].cpu()
    assert int((A != H.torch_cpu_adjacency(X[..., :3], R)).sum()) == 0
    deg = A.sum(-1)
    assert 3 <= float(deg.mean()) <= 40            # ~ tens of neighbours at COMM_RANGE 2.0 on a 1 m lattice


def test_full_size_c5_subset_vs_oracle():
    """BASELINE configs[4]: 65536 envs x 8 agents, set_speeds, K_HOPS=3 -- three envs of the full batch
    against the oracle over 40 steps (free flight)"""
    _subset_vs_oracle(65536, 8, 'set_speeds', 3, 2.0, T=40, spacing=1.0, z0=3.0, pick=[0, 31337, 65535], seed=74,
                      ptol=1e-4, vtol=1e-3)


@pytest.mark.parametrize('E,N', [(1, 1), (3, 31), (2, 33), (1, 2), (257, 5), (3, 8), (1, 16), (4101, 8), (9, 16)])
def test_ragged_shapes_one_step(E, N):
    """group widths that do not fill a warp, the first wide-path size, single agent; N = 8 / 16 with a ragged
    last warp-chunk (full chunks go to the unrolled kernel, the tail to the run-time-width kernel)"""
    rng = np.random.default_rng(80 + N)
    st = H.random_state(rng, E, N, spacing=0.9)
    act = H.random_actions(rng, 'set_target_vel', 1, E, N)
    sw = _swarm(E, N, 'set_target_vel', 1, 1.5)
    H.upload_state(sw, st)
    sw.step(_dev(act[0]))
    ref = H.make_spec(E, N, 'set_target_vel', 1, 1.5, st)
    ref.step(act[0])
    H.check_delta('ragged E%d N%d' % (E, N), st, H.read_state(sw), H.spec_state(ref))
    X = sw.X_window()[0].cpu().numpy()
    np.testing.assert_array_equal(sw.A_window()[0].cpu().numpy(), spec.adjacency(X[..., :3], 1.5))


@pytest.mark.parametrize('mode', ['set_speeds', 'set_target_pos', 'set_target_vel', 'set_control', 'set_target_ori', 'set_force'])
@pytest.mark.parametrize('E,N', [(67, 8), (5, 3)])
def test_baked_kernels_agree_with_generic_kernels(mode, E, N):
    """The default model runs kernels with the constants as immediates (mrs_config_is_baked); a configuration
    that differs in a field this mode never reads runs the generic kernels on the same numbers.  Same
    arithmetic: A bit-exact, states equal to float32 rounding of differently contracted expressions."""
    import ctypes
    T, K, R = 12, 2, 1.5
    rng = np.random.default_rng(91)
    st = H.random_state(rng, E, N, spacing=0.8)
    act = _dev(H.random_actions(rng, mode, T, E, N, start_pos=st['pos']))
    a = _swarm(E, N, mode, K, R, tape_slots=T + K + 1)
    b = _swarm(E, N, mode, K, R, tape_slots=T + K + 1)
    assert a.lib.mrs_config_is_baked(ctypes.byref(a.cfg)) == 1
    if mode == 'set_control':
        b.cfg.quad.pos_p = 1.25          # position gain: unused by set_control
    else:
        b.cfg.quad.arm = 0.04            # arm length: only set_control scales torques with it
    assert b.lib.mrs_config_is_baked(ctypes.byref(b.cfg)) == 0
    H.upload_state(a, st)
    H.upload_state(b, st)
    a.step(act[0])
    b.step(act[0])
    ga, gb = H.read_state(a), H.read_state(b)
    for k in ('pos', 'vel', 'angvel', 'quat'):
        np.testing.assert_allclose(ga[k], gb[k], rtol=2e-6, atol=1e-6, err_msg='%s %s' % (mode, k))
    a.step_many(act[1:].contiguous(), T - 1)
    b.step_many(act[1:].contiguous(), T - 1)
    ga, gb = H.read_state(a), H.read_state(b)
    for k in ('pos', 'vel'):
        np.testing.assert_allclose(ga[k], gb[k], rtol=1e-4, atol=1e-4, err_msg='%s %s after %d steps' % (mode, k, T))
    assert a.read_status() == 0 and b.read_status() == 0


@pytest.mark.parametrize('E,N,mode', [(2, 1100, 'set_target_vel'), (1, 1024, 'set_control'), (3, 1025, 'set_speeds')])
def test_tiled_pair_path_ragged(E, N, mode):
    """N >= 1024 (pair_tile_kernel + agent_pre_kernel): agent tiles and partner slices that do not divide N,
    several envs per launch, sparse contact (spacing 0.8 +- 0.24: about one agent in six within 2 * AGENT_RADIUS +
    margin of a neighbour; the per-env solver holds 1024 agents in contact) -- one step against the oracle, then
    the same step again from the same state must reproduce bit for bit (fixed-order partial sums)."""
    rng = np.random.default_rng(97 + N)
    st = H.random_state(rng, E, N, spacing=0.8, jitter=0.12)
    act = H.random_actions(rng, mode, 1, E, N, start_pos=st['pos'])
    sw = _swarm(E, N, mode, 1, 1.5)
    H.upload_state(sw, st)
    sw.step(_dev(act[0]))
    ref = H.make_spec(E, N, mode, 1, 1.5, st)
    ref.step(act[0])
    g1, r1 = H.read_state(sw), H.spec_state(ref)
    # contact rows switch on thresholds (dist < margin, rhs > 0): allow a float32-sized band
    for k, tol in CONTACT_BAND:
        assert np.max(np.abs(g1[k] - r1[k])) <= tol, k
    X = sw.X_window()[0].cpu().numpy()
    np.testing.assert_array_equal(sw.A_window()[0].cpu().numpy(), spec.adjacency(X[..., :3], 1.5))
    assert sw.read_stats()['agent_contact_rows'] > 0        # sphere contact rows fired
    sw2 = _swarm(E, N, mode, 1, 1.5)
    H.upload_state(sw2, st)
    sw2.step(_dev(act[0]))
    assert torch.equal(sw.state, sw2.state)


def test_wide_contact_dense_cluster_uses_the_round_walk():
    """N > 32 with an agent that has more than 16 pairs in range (a clump of 18 agents, all within the 0.62 m contact
    range of each other: 17 pairs each, 153 in the env): the per-env solver's level schedule does not apply and it
    walks the tournament rounds instead -- same rows, same order as the oracle.  The overlaps are deep (impulses of
    tens of m/s), so the comparison is relative to the largest velocity."""
    E, N = 3, 48
    rng = np.random.default_rng(4848)
    st = H.random_state(rng, E, N, spacing=1.5, z0=3.0, jitter=0.05, tilt=0.05, vel=0.2, angvel=0.2)
    clump = np.array([[i, j, k] for i in range(3) for j in range(3) for k in range(2)], np.float32) * 0.2
    where = rng.permutation(N)[:18]
    st['pos'][:, where] = (clump + np.array([10., 10., 3.], np.float32))[None] + rng.uniform(-0.004, 0.004, (E, 18, 3)).astype(np.float32)
    act = H.random_actions(rng, 'set_target_vel', 1, E, N)
    sw = _swarm(E, N, 'set_target_vel', 0)
    H.upload_state(sw, st)
    sw.step(_dev(act[0]))
    ref = H.make_spec(E, N, 'set_target_vel', 0, float('inf'), st)
    ref.step(act[0])
    g1, r1 = H.read_state(sw), H.spec_state(ref)
    scale = float(np.max(np.abs(r1['vel'])))
    assert scale > 1.0 and sw.read_stats()['agent_contact_rows'] > 20 * E
    assert sw.read_status() == 0
    np.testing.assert_allclose(g1['vel'], r1['vel'], rtol=0, atol=3e-4 * scale)
    np.testing.assert_allclose(g1['pos'], r1['pos'], rtol=0, atol=3e-6 * scale)


def test_capture_rollout_leaves_the_swarm_untouched():
    """capture_rollout warms the launch path up outside the capture; that must not advance the swarm: a captured
    twin replayed once equals T plain steps from the same start, windows included."""
    E, N, K, T = 37, 8, 2, 12
    rng = np.random.default_rng(123)
    st = H.random_state(rng, E, N)
    act = _dev(H.random_actions(rng, 'set_target_vel', T, E, N))
    a = _swarm(E, N, 'set_target_vel', K, 1.5, tape_slots=T, ring=True)
    b = _swarm(E, N, 'set_target_vel', K, 1.5, tape_slots=T, ring=True)
    for sw in (a, b):
        H.upload_state(sw, st)
        sw.step(act[0])                     # some history in the windows
    before = (a.state.clone(), a.ctrl.clone().nan_to_num(nan=-7.0), a.X_window().clone(), a.A_window().clone())
    roll = a.capture_rollout(act, T)
    assert torch.equal(a.state, before[0]) and torch.equal(a.ctrl.nan_to_num(nan=-7.0), before[1])
    assert torch.equal(a.X_window(), before[2]) and torch.equal(a.A_window(), before[3])
    roll.replay()
    for t in range(T):
        b.step(act[t])
    assert torch.equal(a.state, b.state)
    assert torch.equal(a.X_window(), b.X_window()) and torch.equal(a.A_window(), b.A_window())
    assert a.read_stats() == b.read_stats()


@pytest.mark.parametrize('E,N,mode,spacing', [(512, 64, 'set_target_vel', 0.55), (328, 100, 'set_control', 0.8),
                                              (1000, 33, 'set_speeds', 0.55), (256, 128, 'set_target_pos', 2.0)])
def test_fused_env_kernel_equals_the_three_kernel_path(E, N, mode, spacing, monkeypatch):
    """32 < N <= 128 with >= 32768 agents: step_env_kernel (one CTA per env, one launch per step) against the
    pre / contact / post / adjacency kernels it replaces (MRS_B200_FUSED_MID=0) -- state, controller state, rpm
    mirror, X and A windows and the statistics bit for bit over several steps (set_control: to float32 rounding), in
    contact (0.55 m), near the ground without pair rows (0.8 m) and in free flight (2 m), with a NaN action on the way."""
    import mrsgym_b200 as M
    rng = np.random.default_rng(77 + N)
    st = H.random_state(rng, E, N, spacing=spacing, jitter=0.05, z0=0.6 if spacing < 1 else 2.0)
    T = 4
    act = _dev(H.random_actions(rng, mode, T, E, N, start_pos=st['pos']))
    act[2, 3, 5, 0] = float('nan')
    out = []
    for fused in ('1', '0'):
        monkeypatch.setenv('MRS_B200_FUSED_MID', fused)
        sw = M.Swarm(E, N, 2, mode, M._abi.X_FULL, 1.5, keep_rpm=True)
        H.upload_state(sw, st)
        sw.reset_windows()
        for t in range(T):
            sw.step(act[t])
        out.append((sw.state.clone(), sw.ctrl.clone().view(torch.int32), sw.rpm.clone(), sw.X_window().clone(),
                    sw.A_window().clone(), sw.read_stats(), sw.read_status()))
    a, b = out
    if mode == 'set_control':
        # the mixer's NNLS branch is inlined into two different kernels and contracted into FMAs differently: equal to
        # float32 rounding, not to the bit
        for x, y in zip(a[:4], b[:4]):
            x, y = (t.view(torch.float32).nan_to_num(nan=-7.0) for t in (x, y))
            assert float((x - y).abs().max()) <= 2e-6 * max(1.0, float(y.abs().max())), float((x - y).abs().max())
        assert torch.equal(a[4], b[4])
    else:
        for x, y in zip(a[:5], b[:5]):
            assert torch.equal(x, y)
    assert (mode == 'set_control' or a[5] == b[5]) and a[6] == b[6] == M._abi.STATUS_NAN_ACTION
    assert a[5]['nan_actions'] == 1 and (spacing > 0.6 or a[5]['agent_contact_rows'] > 0)


@pytest.mark.parametrize('E,N,mode', [(512, 64, 'set_target_vel'), (400, 100, 'set_control'), (1000, 33, 'set_speeds'),
                                      (260, 128, 'set_target_pos')])
def test_thread_per_agent_mid_path(E, N, mode):
    """32 < N <= 128 with >= 32768 agents: step_mid_pre_kernel + step_post_kernel<1> (one thread per agent, the
    CTA's 128 slots span several envs).  One step in the contact regime against the oracle, A bit-exact, and a
    3-step mrs_step_many equal to three single steps."""
    rng = np.random.default_rng(11 + N)
    st = H.random_state(rng, E, N, spacing=0.55, jitter=0.05)
    act = H.random_actions(rng, mode, 3, E, N, start_pos=st['pos'])
    sw = _swarm(E, N, mode, 1, 1.5)
    H.upload_state(sw, st)
    sw.step(_dev(act[0]))
    ref = H.make_spec(E, N, mode, 1, 1.5, st)
    ref.step(act[0])
    g1, r1 = H.read_state(sw), H.spec_state(ref)
    # contact rows switch on thresholds (dist < margin, rhs > 0): among tens of thousands of agents a few sit
    # within float32 rounding of one, so the band of the small contact test holds for all but a handful
    for k, tol in CONTACT_BAND:
        err = np.abs(g1[k] - r1[k]).max(axis=-1)
        assert np.mean(err > tol) < 1e-3 and err.max() <= 50 * tol, (k, float(err.max()), float(np.mean(err > tol)))
    X = sw.X_window()[0].cpu().numpy()
    np.testing.assert_array_equal(sw.A_window()[0].cpu().numpy(), spec.adjacency(X[..., :3], 1.5))
    assert sw.read_stats()['agent_contact_rows'] > 0
    sw.step(_dev(act[1]))
    sw.step(_dev(act[2]))
    sw2 = _swarm(E, N, mode, 1, 1.5)
    H.upload_state(sw2, st)
    sw2.step_many(_dev(act), 3)
    assert torch.equal(sw.state, sw2.state) and torch.equal(sw.A_window(), sw2.A_window())


@pytest.mark.parametrize('N,mode,E', [(8, 'set_speeds', 40000), (16, 'set_target_pos', 21000), (8, 'set_target_vel', 36001)])
def test_chained_rollout_equals_plain_steps(N, mode, E):
    """mrs_rollout: single-step launches whose chunk ranges are handed from launch to launch through
    bufs.sync (no grid-wide dependency) == the same steps as plain stream-ordered mrs_step launches, bit for
    bit, eagerly and as CUDA-graph replays; sizes that take the SM-sized-CTA path (one with a ragged tail)."""
    K, T = 2, 12
    rng = np.random.default_rng(71)
    st = H.random_state(rng, E, N)
    act = _dev(H.random_actions(rng, mode, T, E, N, start_pos=st['pos']))
    a = _swarm(E, N, mode, K, 1.5, tape_slots=T, ring=True)
    b = _swarm(E, N, mode, K, 1.5, tape_slots=T, ring=True)
    H.upload_state(a, st)
    H.upload_state(b, st)
    for t in range(T):
        a.step(act[t])
    b.rollout(act, T)
    torch.cuda.synchronize()
    bits = lambda t: t.view(torch.int32)       # the PID planes carry a NaN marker
    assert torch.equal(a.state, b.state) and torch.equal(bits(a.ctrl), bits(b.ctrl))
    assert torch.equal(a.X_tape, b.X_tape) and torch.equal(a.A_tape, b.A_tape)
    roll = b.capture_rollout(act, T)          # leaves b where it was
    for rep in range(3):
        for t in range(T):
            a.step(act[t])
        roll.replay()
    torch.cuda.synchronize()
    assert torch.equal(a.state, b.state) and torch.equal(bits(a.ctrl), bits(b.ctrl))
    assert torch.equal(a.X_tape, b.X_tape) and torch.equal(a.A_tape, b.A_tape)
    assert a.read_status() == 0 and b.read_status() == 0
    assert a.read_stats() == b.read_stats()


@pytest.mark.parametrize('E,N', [(256, 8), (33, 16), (7, 32), (5, 40), (3, 100)])
def test_packed_adjacency_on_the_wire_equals_float_adjacency(E, N):
    """Opt-in compact adjacency of the host paths (mrs_pack_adjacency): unpacked bits == the float32 A the step wrote,
    bit for bit, through mrs_step_host and the pipelined mrs_rollout_host (which may deliver both forms at once)."""
    from mrsgym_b200.core import unpack_adjacency
    K, T = 1, 7
    rng = np.random.default_rng(5 + N)
    st = H.random_state(rng, E, N)
    act = H.random_actions(rng, 'set_speeds', T, E, N)
    sw = _swarm(E, N, 'set_speeds', K, 1.3, tape_slots=16)
    H.upload_state(sw, st)
    W = (N + 31) // 32
    ah = torch.from_numpy(act).pin_memory()
    Xh = torch.empty(T, E, N, 6).pin_memory()
    Ah = torch.empty(T, E, N, N).pin_memory()
    Bh = torch.empty(T, E, N, W, dtype=torch.int32).pin_memory()
    sw.rollout_host(ah, torch.empty(2, E, N, 4, device='cuda'), Xh, Ah, Bh, torch.empty(2, E, N, W, dtype=torch.int32, device='cuda'))
    assert torch.equal(unpack_adjacency(Bh, N), Ah)
    assert float(Ah.sum()) > 0 and float((1 - Ah).sum()) > 0            # the case has both zeros and ones
    # compact form only, one synchronous step
    B1 = torch.empty(E, N, W, dtype=torch.int32).pin_memory()
    sw.step_host(ah[0], torch.empty(E, N, 4, device='cuda'), Xh[0], None, B1, torch.empty(E, N, W, dtype=torch.int32, device='cuda'))
    assert torch.equal(unpack_adjacency(B1, N).cuda(), sw.A_window()[0])
    assert torch.equal(unpack_adjacency(sw.pack_adjacency(sw.A_window()[0]), N), sw.A_window()[0])
