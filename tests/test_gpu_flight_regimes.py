"""The CUDA free-flight step at the edges of its range (tests/flight_regimes.py) against the CPU oracle, on every
kernel the step can pick: N <= 32 run-time-width, unrolled (pair-once downwash with the shuffle to the lower agent)
and SM-sized-CTA kernels, mrs_step_many and the chained mrs_rollout, the 33-128 agent kernels (lanes per agent, fused
one CTA per env and the three-kernel path) and the N > 128 tiled pair pass.  The bar is the one-step delta bar of
test_gpu_parity.py (helpers.check_delta); A must be bit-exact on the GPU's own X and the status 0.
test_cpu_flight_regimes.py shows, at these shapes and seeds, that every case lands >= 10 bars away from what a subtly
wrong kernel would compute."""
import numpy as np
import pytest
import torch

import flight_regimes as F
import helpers as H
from oracle import spec
from test_gpu_physics_variants import _big_cta_envs

pytestmark = pytest.mark.gpu

R_COMM, K = 12.0, 1
ALL = list(F.CASES)


def _swarm(E, N, name, layout=None):
    import mrsgym_b200 as M
    act = 'set_speeds' if F.CASES[name][2] == 'hover' else None
    sw = M.Swarm(E, N, K, act, M._abi.X_POS_VEL if layout is None else layout, R_COMM)
    F.apply(sw, F.fields_of(name))
    return sw


def _dev(a):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _check_step(tag, sw, s0, rpm, fields, picks):
    """one step of sw (already taken) from the float32 state s0 against the oracle, on the envs `picks`"""
    sub = lambda d: {k: v[picks] for k, v in d.items()}
    ref = F.oracle_step(sub(s0), fields, None if rpm is None else rpm[picks])
    g = sub(H.read_state(sw))
    H.check_delta(tag, sub(s0), g, ref)
    X = sw.X_window()[0]
    np.testing.assert_array_equal(X[..., :3].cpu().numpy(), H.read_state(sw)['pos'].astype(np.float32))
    np.testing.assert_array_equal(sw.A_window()[0][picks].cpu().numpy(),
                                  spec.adjacency(X[picks][..., :3].cpu().numpy(), R_COMM))
    assert sw.read_status() == 0, tag


def _run(name, E, N, picks=None, layout=None, tile=None, T=1):
    """T plain steps, each a one-step test restarted from the GPU's float32 state"""
    st, rpm, _ = F.make_case(name, *(tile or (E, N)), seed=N)
    if tile:                # envs repeat with period tile[0]: the oracle runs the picked ones
        reps = -(-E // tile[0])
        st = {k: np.ascontiguousarray(np.tile(v, (reps,) + (1,) * (v.ndim - 1))[:E]) for k, v in st.items()}
        rpm = None if rpm is None else np.ascontiguousarray(np.tile(rpm, (reps, 1, 1))[:E])
    picks = list(range(E)) if picks is None else picks
    sw = _swarm(E, N, name, layout)
    H.upload_state(sw, st)
    fields = F.fields_of(name)
    a = _dev(rpm)
    for t in range(T):
        s0 = {k: v.astype(np.float32) for k, v in H.read_state(sw).items()}
        sw.step(a)
        _check_step('%s E%d N%d step %d' % (name, E, N, t), sw, s0, rpm, fields, picks)
    return sw, st, rpm


# ------------------------------------------------------------------------------ N <= 32
@pytest.mark.parametrize('name', ALL)
def test_runtime_width_kernel(name):
    """GT = 0: group width chosen at run time (N = 5), 4 envs per warp-chunk"""
    _run(name, 12, 5)


@pytest.mark.parametrize('name', ALL)
@pytest.mark.parametrize('E,N', [(67, 8), (10, 16), (4, 32)])
def test_unrolled_full_chunk_kernels(name, E, N):
    """GT = 8 / 16 / 32: each pair's downwash evaluated once with |dz| and handed to the lower agent by shuffle; at
    E = 67, N = 8 the ragged last chunk runs the run-time-width kernel"""
    import mrsgym_b200 as M
    _run(name, E, N, layout=M._abi.X_FULL if N == 16 else None)


@pytest.mark.parametrize('name', ['spin_below', 'spin_above', 'clamp', 'attitude', 'downwash_near', 'threshold_high',
                                  'mass'])
def test_sm_sized_cta_kernel(name):
    """N = 8 with enough warp-chunks for one SM-sized CTA per SM; the oracle runs envs of the first warp-chunk and
    envs far into the batch"""
    E = _big_cta_envs()
    _run(name, E, 8, picks=[0, 1, 2, 3, E // 2 + 1, E - 1], tile=(64, 8))


@pytest.mark.parametrize('name', ['spin_below', 'spin_above', 'gyro', 'clamp', 'ring', 'downwash_near', 'clamp5',
                                  'threshold_high'])
@pytest.mark.parametrize('E,N', [(67, 8), (9, 16)])
def test_multi_step_forms(name, E, N):
    """three plain steps, each a one-step test from the GPU's float32 state; mrs_rollout bit for bit equal to them,
    mrs_step_many (state in registers across steps) to float32 rounding"""
    T = 3
    plain, st, rpm = _run(name, E, N, T=T)
    acts = None if rpm is None else _dev(np.ascontiguousarray(np.broadcast_to(rpm, (T,) + rpm.shape)))
    out = {}
    for how in ('many', 'rollout'):
        sw = _swarm(E, N, name)
        H.upload_state(sw, st)
        (sw.step_many if how == 'many' else sw.rollout)(acts, T)
        assert sw.read_status() == 0, how
        out[how] = sw
    assert torch.equal(plain.state, out['rollout'].state)
    # float32 rounding relative to each agent's vector (pos, quat, vel, angvel): a spin of 100+ rad/s carries ulps of
    # 8e-6 into all three of its coordinates, and the gyro term feeds them back
    p, m = plain.state.double(), out['many'].state.double()
    for name_, lo, hi in (('pos', 0, 3), ('quat', 3, 7), ('vel', 7, 10), ('angvel', 10, 13)):
        scale = p[lo:hi].norm(dim=0).clamp(min=1.0)
        rel = float(((p[lo:hi] - m[lo:hi]).abs() / scale).max())
        assert rel < 2e-5, (name_, rel)


# ------------------------------------------------------------------------------ 33 <= N <= 128
@pytest.mark.parametrize('name', ALL)
def test_lanes_per_agent_wide_kernels(name):
    """few agents: step_pre_kernel<8> + contact_env_kernel + step_post_kernel"""
    _run(name, 6, 48)


@pytest.mark.parametrize('fused', ['1', '0'])
@pytest.mark.parametrize('name', ['spin_above', 'clamp', 'hclip', 'downwash_near', 'clamp5', 'mass'])
def test_one_cta_per_env_kernels(name, fused, monkeypatch):
    """>= 32768 agents: the fused step_env_kernel, and the three-kernel path (MRS_B200_FUSED_MID=0)"""
    import mrsgym_b200 as M
    monkeypatch.setenv('MRS_B200_FUSED_MID', fused)
    _run(name, 520, 64, picks=[0, 1, 259, 519], layout=M._abi.X_FULL if fused == '1' else None)


# ------------------------------------------------------------------------------ N > 128
@pytest.mark.parametrize('name', ALL)
def test_tiled_pair_kernels(name):
    """pair_tile_kernel + agent_pre_kernel"""
    _run(name, 2, 200)


@pytest.mark.parametrize('name', ['spin_below', 'spin_above', 'clamp', 'attitude', 'ring', 'downwash_near',
                                  'threshold_high', 'mass'])
def test_tiled_pair_kernels_1030(name):
    _run(name, 1, 1030)
