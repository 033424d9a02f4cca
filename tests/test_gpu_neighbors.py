"""mrs_neighbors on the device: the lists against mrs_adjacency and torch CPU (bit-exact graph, ascending rows, -1
padding, degrees), threshold edges, overflow, determinism; MRS(A_FORMAT='neighbors') against the dense mode on the
same seed; graph-captured rollouts; reynolds_policy / rollout() on lists; the C4 swarm at full size."""
import ctypes

import numpy as np
import pytest
import torch

import helpers as H
from oracle import spec

pytestmark = pytest.mark.gpu


def _swarm(E, N, R, **kw):
    import mrsgym_b200 as M
    return M.Swarm(E, N, 0, 'set_speeds', M._abi.X_POS_VEL, R, **kw)


def _upload_pos(sw, pos32):
    sw.state[0:3] = torch.from_numpy(np.ascontiguousarray(pos32.reshape(-1, 3).T)).cuda()


def _check_lists(nb, A, M):
    """nb = Neighbors [E, N, M] / [E, N] on the device, A = the dense {0,1} A [E, N, N] (CPU)."""
    idx, cnt = nb.idx.cpu(), nb.count.cpu()
    N = A.shape[-1]
    assert torch.equal(cnt, A.sum(-1).to(torch.int32))
    j = torch.arange(N).expand_as(A)
    want = torch.where(A != 0, j, j + N).sort(dim=-1).values[..., :M]
    want = torch.where(want < N, want, torch.full_like(want, -1)).to(torch.int32)
    if M > N:
        want = torch.cat([want, torch.full((*want.shape[:-1], M - N), -1, dtype=torch.int32)], -1)
    assert torch.equal(idx, want)


SHAPES = [(1, 3, 1.5), (64, 8, 2.0), (16, 32, 2.0), (7, 5, 0.9), (3, 33, 1.7), (5, 64, 2.0), (9, 36, 1.2),
          (3, 100, float('inf')), (700, 64, 2.0), (2, 124, 1.6), (2, 128, 2.0), (1, 500, 3.0), (1, 4096, 2.0),
          (4, 16, float('inf')), (1, 256, float('inf'))]


@pytest.mark.parametrize('E,N,R', SHAPES)
def test_neighbors_equal_adjacency(E, N, R):
    rng = np.random.default_rng(1000 + N)
    pos = H.grid_positions(E, N, spacing=0.5, z0=1.0, jitter=0.0)
    pos[E // 2:] += rng.uniform(-0.3, 0.3, pos[E // 2:].shape)
    pos32 = pos.astype(np.float32)
    sw = _swarm(E, N, R)
    _upload_pos(sw, pos32)
    A = sw.adjacency(torch.from_numpy(pos32).cuda()).cpu()
    assert torch.equal(A, H.torch_cpu_adjacency(pos32, R))
    M = N - 1 if N <= 65 else int(A.sum(-1).max())
    nb = sw.neighbors(M)
    _check_lists(nb, A, M)
    assert sw.read_status() == 0 and sw.read_stats()['neighbor_overflow'] == 0
    assert torch.equal(nb.to_dense().cpu(), A)


def test_neighbor_threshold_edges():
    R = 2.0
    base = np.zeros((1, 8, 3), np.float32)
    d = np.float32(R)
    offs = [np.nextafter(d, np.float32(0)), d, np.nextafter(d, np.float32(10)), np.float32(1.9999), np.float32(2.0001)]
    for i, o in enumerate(offs):
        base[0, i + 1, 0] = o
    base[0, 7] = np.nan
    for Rz in (R, 0.0, 1e-30, 1e30):
        sw = _swarm(1, 8, Rz)
        _upload_pos(sw, base)
        A = H.torch_cpu_adjacency(base, Rz)
        assert torch.equal(sw.adjacency(torch.from_numpy(base).cuda()).cpu(), A)
        _check_lists(sw.neighbors(7), A, 7)
        _check_lists(sw.neighbors(12), A, 12)
        assert sw.read_status() == 0


@pytest.mark.parametrize('E,N', [(50, 8), (6, 20), (4, 64), (1, 300)])
def test_neighbor_overflow_degrees_only_and_determinism(E, N):
    import mrsgym_b200 as M
    rng = np.random.default_rng(N)
    pos32 = H.grid_positions(E, N, spacing=0.4, z0=1.0, jitter=0.1, rng=rng).astype(np.float32)
    sw = _swarm(E, N, 1.0)
    _upload_pos(sw, pos32)
    A = H.torch_cpu_adjacency(pos32, 1.0)
    deg = A.sum(-1)
    m = 3
    assert int((deg > m).sum()) > 0
    sw.stats.zero_()
    nb = sw.neighbors(m)
    _check_lists(nb, A, m)                                   # first m neighbours, true degree
    assert sw.read_status() & M._abi.STATUS_NEIGHBOR_OVERFLOW
    assert sw.read_stats()['neighbor_overflow'] == int((deg > m).sum())
    nb2 = sw.neighbors(m)
    assert torch.equal(nb.idx, nb2.idx) and torch.equal(nb.count, nb2.count)
    assert sw.read_status() & M._abi.STATUS_NEIGHBOR_OVERFLOW            # the second call overflows as well (clears)
    sw.stats.zero_()
    d0 = sw.neighbors(0)                                     # degrees only: no idx, no overflow
    assert d0.idx.shape == (E, N, 0) and torch.equal(d0.count.cpu(), deg.to(torch.int32))
    assert sw.read_status() == 0 and sw.read_stats()['neighbor_overflow'] == 0
    # argument checks of the C ABI
    cnt = torch.empty(E, N, dtype=torch.int32, device='cuda')
    lib, s = sw.lib, ctypes.c_void_p(0)
    assert lib.mrs_neighbors(ctypes.byref(sw.cfg), ctypes.byref(sw.bufs), -1, None, ctypes.c_void_p(cnt.data_ptr()), s) == -1
    assert lib.mrs_neighbors(ctypes.byref(sw.cfg), ctypes.byref(sw.bufs), 4, None, ctypes.c_void_p(cnt.data_ptr()), s) == -1
    assert lib.mrs_neighbors(ctypes.byref(sw.cfg), ctypes.byref(sw.bufs), 0, None, None, s) == -1


def _pair(N, K, E, seed=5):
    import mrsgym_b200 as M
    kw = dict(N_AGENTS=N, N_ENVS=E, K_HOPS=K, COMM_RANGE=1.2, ACTION_TYPE='set_target_vel', SEED=seed, AGENT_RADIUS=0.1)
    if N > 32:      # host-side start states: fixed positions and attitudes, so that both envs start alike
        kw['START_POS'] = torch.from_numpy(H.grid_positions(E, N, spacing=0.7, z0=2.0, jitter=0.1,
                                                            rng=np.random.default_rng(seed)).astype(np.float32))
        kw['START_ORI'] = torch.zeros(N, 3)
    return M.MRS(**kw), M.MRS(A_FORMAT='neighbors', **kw)


def _same_window(d, n, M):
    assert n.idx.shape[-1] == M
    assert torch.equal(n.to_dense(), d), 'neighbour window differs from the dense window'


@pytest.mark.parametrize('N', [3, 8, 33, 64, 200])
@pytest.mark.parametrize('K', [0, 3])
@pytest.mark.parametrize('E', [1, 5])
def test_mrs_neighbor_mode_matches_dense(N, K, E):
    dense, nbr = _pair(N, K, E)
    M = min(N - 1, 64)
    rng = np.random.default_rng(N * 10 + K)
    for env in (dense, nbr):
        env.calc_Ak()
    _same_window(dense.get_Ak(), nbr.get_Ak(), M)
    for t in range(40):
        act = torch.from_numpy(rng.normal(0, 0.4, (E, N, 3)).astype(np.float32)).cuda()
        act = act if E > 1 else act[0]
        Xd, _, _, infod = dense.step(act)
        Xn, _, _, infon = nbr.step(act)
        assert torch.equal(Xd, Xn)
        assert torch.equal(dense.swarm.state, nbr.swarm.state)          # A never feeds back into the physics
        _same_window(infod['A'], infon['A'], M)
        if t == 15:
            dense.reset(); nbr.reset()
            assert torch.equal(dense.swarm.state, nbr.swarm.state)
            _same_window(dense.get_Ak(), nbr.get_Ak(), M)
            dense.calc_Ak(); nbr.calc_Ak()
        if t == 25 and E > 1:
            mask = torch.zeros(E, dtype=torch.bool)
            mask[1::2] = True
            dense.reset(env_mask=mask); nbr.reset(env_mask=mask)
            _same_window(dense.get_Ak(), nbr.get_Ak(), M)
            _same_window(dense.refresh_A(mask), nbr.refresh_A(mask), M)
    nbr.check_status()
    Ad = dense.calc_A()
    assert torch.equal(Ad, nbr.calc_A())                                  # calc_A stays dense


@pytest.mark.parametrize('N', [8, 64])
def test_capture_rollout_neighbor_mode(N):
    import mrsgym_b200 as M
    E, K, T = 32, 2, 8
    rng = np.random.default_rng(N)
    st = H.random_state(rng, E, N, spacing=0.8)
    act = torch.from_numpy(H.random_actions(rng, 'set_speeds', T, E, N)).cuda()
    a = M.Swarm(E, N, K, 'set_speeds', M._abi.X_POS_VEL, 1.5, tape_slots=T, ring=True, neighbors=N - 1)
    b = M.Swarm(E, N, K, 'set_speeds', M._abi.X_POS_VEL, 1.5, tape_slots=T, neighbors=N - 1)
    H.upload_state(a, st)
    H.upload_state(b, st)
    g = a.capture_rollout(act, T)
    for rep in range(2):
        g.replay()
        for t in range(T):
            b.step(act[t])
        torch.cuda.synchronize()
        assert torch.equal(a.state, b.state)
        wa, wb = a.N_window(), b.N_window()
        assert torch.equal(wa.idx, wb.idx) and torch.equal(wa.count, wb.count)
        X = a.X_window()[0].cpu().numpy()
        assert np.array_equal(wa.to_dense()[0].cpu().numpy(), spec.adjacency(X[..., :3], 1.5))


def test_rollout_reynolds_on_lists():
    import mrsgym_b200 as M
    E, N, T = 16, 12, 30
    kw = dict(N_AGENTS=N, N_ENVS=E, K_HOPS=1, COMM_RANGE=1.5, ACTION_TYPE='set_target_vel', SEED=3, MAX_TIMESTEPS=20)
    dense, nbr = M.MRS(**kw), M.MRS(A_FORMAT='neighbors', **kw)
    pol = M.reynolds_policy()
    # the same X through both windows: the policy agrees to rounding
    dense.calc_Ak(); nbr.calc_Ak()
    out_d, out_n = pol(dense.get_Xk(), dense.get_Ak()), pol(nbr.get_Xk(), nbr.get_Ak())
    torch.testing.assert_close(out_n, out_d, rtol=1e-6, atol=1e-6)
    data = M.rollout(nbr, pol, T, episode_length=12)
    assert 'A' not in data and data['A_idx'].shape == (T, E, N, N - 1) and data['A_cnt'].shape == (T, E, N)
    X = data['X'].cpu().numpy()
    A = spec.adjacency(X[..., :3], 1.5)
    assert np.array_equal(M.Neighbors(data['A_idx'], data['A_cnt']).to_dense().cpu().numpy(), A)
    assert np.array_equal(data['A_cnt'].cpu().numpy(), A.sum(-1).astype(np.int32))
    hist = M.to_trainer_history(data, envs=[0, 3])
    assert len(hist['A']) == 2 * T and np.array_equal(hist['A'][T + 4].numpy(), A[4, 3])


def test_c4_full_size():
    import bench
    import mrsgym_b200 as M
    w = bench.WORKLOADS['c4']
    E, N = w['E'], w['N']
    st, act = bench.make_inputs(w, E, 5, seed=1234 + 4)
    dense = M.Swarm(E, N, 0, w['mode'], M._abi.X_POS_VEL, w['R'], tape_slots=8)
    nbr = M.Swarm(E, N, 0, w['mode'], M._abi.X_POS_VEL, w['R'], tape_slots=8, neighbors=64)
    H.upload_state(dense, st)
    H.upload_state(nbr, st)
    acts = torch.from_numpy(act).cuda()
    maxdeg = 0
    for t in range(5):
        dense.step(acts[t])
        nbr.step(acts[t])
        w_n = nbr.N_window()
        assert torch.equal(w_n.to_dense(), dense.A_window())
        maxdeg = max(maxdeg, int(w_n.count.max()))
    assert torch.equal(dense.state, nbr.state)
    assert 0 < maxdeg <= 64 and nbr.read_status() == 0 and nbr.read_stats()['neighbor_overflow'] == 0
    print('c4: max degree %d at M = 64, no overflow' % maxdeg)
