"""Host side of the neighbour-list form of A, on CPU: Neighbors.to_dense / edge_index on hand-built lists, the
neighbour tapes' heads against the reference's deque semantics (MRS.py:87-114) with a test double standing in for
mrs_step / mrs_neighbors (in the style of test_cpu_tapes.py), and reynolds_policy / to_trainer_history on lists."""
import ctypes
import random
from collections import deque

import numpy as np
import pytest
import torch

import helpers as H
from mrsgym_b200 import _abi, Neighbors
from mrsgym_b200.core import Swarm
from mrsgym_b200.rollout import reynolds_policy, to_trainer_history


def lists_of(A, M):
    """Neighbors of a dense {0,1} A [..., N, N] (the definition mrs_neighbors implements)."""
    A = torch.as_tensor(A)
    N = A.shape[-1]
    cnt = (A != 0).sum(-1).to(torch.int32)
    j = torch.arange(N).expand_as(A)
    key = torch.where(A != 0, j, j + N)                     # hits first, in ascending j
    order = key.sort(dim=-1).values[..., :M]
    idx = torch.where(order < N, order, torch.full_like(order, -1)).to(torch.int32)
    if M > N:
        idx = torch.cat([idx, torch.full((*idx.shape[:-1], M - N), -1, dtype=torch.int32)], dim=-1)
    return Neighbors(idx, cnt)


# ------------------------------------------------------------------------------ Neighbors
def test_to_dense_and_edge_index_hand_built():
    # one env, 4 agents: 0-1, 0-3, 2-3
    idx = torch.tensor([[1, 3, -1], [0, -1, -1], [3, -1, -1], [0, 2, -1]], dtype=torch.int32)
    cnt = torch.tensor([2, 1, 1, 2], dtype=torch.int32)
    nb = Neighbors(idx, cnt)
    A = nb.to_dense()
    assert A.dtype == torch.float32 and A.shape == (4, 4)
    want = torch.zeros(4, 4)
    for i, j in ((0, 1), (0, 3), (2, 3)):
        want[i, j] = want[j, i] = 1.0
    assert torch.equal(A, want)
    ei = nb.edge_index(None)
    assert ei.dtype == torch.int64
    assert ei.tolist() == [[0, 0, 1, 2, 3, 3], [1, 3, 0, 3, 0, 2]]
    # windows: [K+1, N, M] (one env) and [E, K+1, N, M]; node index e*N + i
    win = Neighbors(torch.stack([idx, torch.full_like(idx, -1)]), torch.stack([cnt, torch.zeros_like(cnt)]))
    assert torch.equal(win.edge_index(0), ei) and win.edge_index(1).shape == (2, 0)
    bat = Neighbors(torch.stack([win.idx, win.idx.flip(0)]), torch.stack([win.count, win.count.flip(0)]))
    assert bat.edge_index(0).tolist() == ei.tolist()            # env 1's hop 0 is empty
    e1 = bat.edge_index(1)
    assert torch.equal(e1, ei + 4)                                # env 1's hop 1 = the lists, offset by N
    assert torch.equal(bat.to_dense()[1, 1], want) and float(bat.to_dense()[1, 0].sum()) == 0.0


@pytest.mark.parametrize('E,N,M', [(3, 5, 4), (2, 9, 3), (1, 40, 64), (4, 1, 0), (2, 33, 32)])
def test_lists_roundtrip_random_graphs(E, N, M):
    g = torch.Generator().manual_seed(E * 100 + N)
    A = (torch.rand(E, 2, N, N, generator=g) < 0.3).float()
    A = ((A + A.transpose(-1, -2)) > 0).float()
    A.diagonal(dim1=-2, dim2=-1).zero_()
    nb = lists_of(A, M)
    assert nb.idx.shape == (E, 2, N, M)
    if M >= N - 1:
        assert torch.equal(nb.to_dense(), A)
        for k in range(2):
            want = A[:, k].nonzero()
            ei = nb.edge_index(k)
            assert torch.equal(ei[0], want[:, 0] * N + want[:, 1]) and torch.equal(ei[1], want[:, 0] * N + want[:, 2])
    else:       # truncated rows keep their first M neighbours
        D = nb.to_dense()
        assert torch.equal(D * A, D) and torch.equal(D.sum(-1), nb.count.clamp(max=M).float())


# ------------------------------------------------------------------------------ tapes
class FakeNbrLib:
    """mrs_step writes the step's serial number into X; mrs_neighbors writes 2 * serial (+1 when called outside a
    step, i.e. calc_Ak / push_A) into the count and index slot it was pointed at."""

    def __init__(self, sw):
        self.sw = sw
        self.serial = 0
        self.after_step = False
        self.calls = []

    def mrs_step(self, cfg, bufs, actions, slot_x, slot_a, stream):
        assert self.sw.A_tape is None and not self.sw.bufs.A_tape          # no dense A in neighbour mode
        self.serial += 1
        assert 0 <= slot_x < self.sw.L and 0 <= slot_a < self.sw.L
        self.sw.X_tape[slot_x] = float(self.serial)
        self.after_step = True
        self.calls.append('step')
        return 0

    def mrs_neighbors(self, cfg, bufs, M, idx, cnt, stream):
        sw = self.sw
        slot, rem = divmod(cnt.value - sw.N_cnt.data_ptr(), 4 * sw.S)
        assert rem == 0 and 0 <= slot < sw.L
        assert idx.value == sw.N_idx.data_ptr() + 4 * slot * sw.S * M
        v = 2 * self.serial + (0 if self.after_step else 1)
        sw.N_cnt[slot] = v
        sw.N_idx[slot] = v
        self.after_step = False
        self.calls.append('nbr')
        return 0

    def mrs_observe(self, cfg, bufs, slot, write_X, write_A, stream):
        assert not write_A
        if write_X:
            self.sw.X_tape[slot] = float(self.serial)
        return 0

    def mrs_tape_fill(self, cfg, bufs, which, src, dst_first, count, stream):
        assert which == 1, 'the neighbour tapes are moved with torch copies'
        for i in range(count):
            self.sw.X_tape[dst_first + i] = self.sw.X_tape[src] if src >= 0 else 0.0
        return 0


def make_nbr_swarm(K, L, M=2, ring=False, fresh=False):
    sw = object.__new__(Swarm)              # bypass the CUDA-only constructor: host logic only
    sw.E, sw.N, sw.K, sw.L, sw.S, sw.D = 1, 1, K, L, 1, 1
    sw.cfg = _abi.MrsConfig()
    sw.cfg.E = sw.cfg.N = 1
    sw.cfg.K, sw.cfg.L = K, L
    sw.cfg.action_type = _abi.NO_ACTION
    sw.cfg.state_layout = _abi.X_POS_VEL
    sw.bufs = _abi.MrsBuffers()
    sw.X_tape = torch.full((L, 1, 1, 1), -1.0)
    sw.A_tape = None
    sw.nbr = M
    sw.N_idx = torch.full((L, 1, 1, M), -7, dtype=torch.int32)
    sw.N_cnt = torch.full((L, 1, 1), -7, dtype=torch.int32)
    sw.device = torch.device('cpu')
    sw.launches = 0
    sw.hx = sw.ha = L - K - 1
    sw.ring = ring
    sw.fresh = fresh and not ring
    sw.generation = 0
    sw.a_empty = True
    sw.lib = FakeNbrLib(sw)
    sw._stream = lambda: None
    sw._mrs_step = sw.lib.mrs_step
    sw._cfg_ref, sw._bufs_ref = ctypes.byref(sw.cfg), ctypes.byref(sw.bufs)
    sw._launches_per_step = 1
    return sw


class RefRings:
    """The reference's two deques (MRS.calc_Xk / calc_Ak / reset, MRS.py:87-114,185-192); an empty A entry is a
    list with count 0."""

    def __init__(self, K):
        self.K = K
        self.X, self.A = deque(), deque()

    def reset(self, x0):
        self.X, self.A = deque(), deque()
        self.push_X(x0)

    def push_X(self, x):
        self.X.appendleft(x)
        if len(self.X) > self.K + 1:
            self.X.pop()
        while len(self.X) < self.K + 1:
            self.X.append(x)

    def push_A(self, a):
        self.A.appendleft(a)
        if len(self.A) > self.K + 1:
            self.A.pop()
        while len(self.A) < self.K + 1:
            self.A.append(0)


def window_lists(sw):
    idx, cnt = sw.N_window()
    return idx.reshape(sw.K + 1, -1), cnt.flatten().tolist()


def assert_matches(sw, ref, it):
    assert sw.X_window().flatten().tolist() == list(ref.X), (it, 'X')
    if len(ref.A) == 0:
        assert sw.a_empty
        return
    idx, cnt = window_lists(sw)
    assert not sw.a_empty and cnt == list(ref.A), (it, 'cnt')
    for k, v in enumerate(ref.A):
        assert idx[k].tolist() == [v if v else -1] * sw.nbr, (it, 'idx', k)


@pytest.mark.parametrize('mode', ['plain', 'ring', 'fresh'])
@pytest.mark.parametrize('K', [0, 1, 2, 3, 4, 5])
def test_neighbor_tapes_follow_the_reference_deques(K, mode):
    L = (K + 1 if mode == 'ring' else 2 * K + 2) + K % 3 + 1
    rnd = random.Random(K * 10 + len(mode))
    sw = make_nbr_swarm(K, L, M=3, ring=mode == 'ring', fresh=mode == 'fresh')
    ref = RefRings(K)
    held = []
    sw.reset_windows()
    ref.reset(float(sw.lib.serial))
    for it in range(300):
        op = rnd.random()
        if op < 0.45:
            sw.step(None)
            ref.push_X(float(sw.lib.serial))
            ref.push_A(2 * sw.lib.serial)
        elif op < 0.6:
            T = rnd.randint(1, 2 * L)
            (sw.step_many if op < 0.52 else sw.rollout)(None, T)       # per-step launches in neighbour mode
            for s in range(sw.lib.serial - T + 1, sw.lib.serial + 1):
                ref.push_X(float(s))
                ref.push_A(2 * s)
        elif op < 0.85:
            sw.push_A()                                  # calc_Ak outside step: only the A ring shifts
            ref.push_A(2 * sw.lib.serial + 1)
        elif op < 0.92 and mode == 'fresh':
            sw.renew_tapes()
        else:
            sw.reset_windows()
            ref.reset(float(sw.lib.serial))
        assert_matches(sw, ref, it)
        assert 0 <= sw.hx < L and 0 <= sw.ha <= L
        if mode == 'fresh' and not sw.a_empty:
            held.append((sw.N_window(), list(ref.A)))
    # every step is mrs_step followed by mrs_neighbors
    calls = sw.lib.calls
    assert all(calls[i + 1] == 'nbr' for i, c in enumerate(calls) if c == 'step')
    for w, want in held:                                # fresh tapes: windows handed out earlier never change
        assert w.count.flatten().tolist() == want
    assert mode != 'fresh' or sw.generation > 300 // L


def test_masked_windows_slots_and_graph_keep_cover_neighbor_tapes():
    sw = make_nbr_swarm(2, 8, M=2)
    sw.reset_windows()
    for _ in range(3):
        sw.step(None)
    assert sw.window_slots(2) == list(range(sw.ha, sw.ha + 3))
    idx, cnt = sw.N_window()
    assert idx.shape == (3, 1, 1, 2) and cnt.shape == (3, 1, 1)
    assert cnt.flatten().tolist() == [6, 4, 2]
    with pytest.raises(_abi.MrsError):
        sw.step_host(torch.zeros(0), None, None, None)


# ------------------------------------------------------------------------------ policy and dataset
@pytest.mark.parametrize('E,N,R', [(3, 8, 1.5), (1, 40, 2.0), (2, 5, float('inf'))])
def test_reynolds_policy_lists_match_dense(E, N, R):
    rng = np.random.default_rng(N)
    pos = H.grid_positions(E, N, spacing=0.7, z0=1.0, jitter=0.2, rng=rng).astype(np.float32)
    vel = rng.normal(0, 0.5, (E, N, 3)).astype(np.float32)
    X = torch.from_numpy(np.concatenate([pos, vel], -1)).unsqueeze(1).repeat(1, 2, 1, 1)     # [E, K+1, N, 6]
    A = H.torch_cpu_adjacency(pos, R).unsqueeze(1).repeat(1, 2, 1, 1)
    nb = lists_of(A, N - 1)
    pol = reynolds_policy()
    dense, lists = pol(X, A), pol(X, nb)
    assert dense.shape == lists.shape == (E, N, 3)
    torch.testing.assert_close(lists, dense, rtol=1e-6, atol=1e-6)
    torch.testing.assert_close(pol(X[0], Neighbors(nb.idx[0], nb.count[0])), dense[:1], rtol=1e-6, atol=1e-6)


def test_trainer_history_expands_lists():
    T, E, N = 3, 2, 5
    g = torch.Generator().manual_seed(3)
    A = (torch.rand(T, E, N, N, generator=g) < 0.4).float()
    A = ((A + A.transpose(-1, -2)) > 0).float()
    A.diagonal(dim1=-2, dim2=-1).zero_()
    nb = lists_of(A, N - 1)
    X = torch.rand(T, E, N, 6, generator=g)
    dense = to_trainer_history({'X': X, 'A': A})
    lists = to_trainer_history({'X': X, 'A_idx': nb.idx, 'A_cnt': nb.count})
    assert len(lists['A']) == T * E
    for a, b in zip(dense['A'], lists['A']):
        assert a.shape == (N, N) and torch.equal(a, b)
    assert dense['done'] == lists['done']
