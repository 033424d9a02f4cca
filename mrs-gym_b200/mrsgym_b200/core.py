"""Swarm: the batched [envs x agents] device state store and its C-ABI calls.

Replaces, for the step path only, the reference's BulletSim + Environment + Quadcopter +
QuadControl object graph (/root/reference/mrsgym/BulletSim.py, Environment.py:84-124,
Quadcopter.py, QuadControl.py).  PyTorch owns every device buffer (the library never
allocates); all launches go on torch's current stream.

Observation history ("tapes"): X_tape [L][E][N][D] and A_tape [L][E][N][N].  Time runs towards
LOWER slot indices: a step writes slot head-1, so slots [head, head+K] are exactly the
reference's newest-first K_HOPS+1 window (MRS.get_Xk / get_Ak, MRS.py:98-114) as a zero-copy
view.  When a head reaches 0 the K newest slots are moved to the top of the tape.  X and A keep
separate heads because the reference shifts its two deques independently (calc_Ak can be called
without calc_Xk, examples/simulating_data/helper/DataGenerator.py:23).

Neighbour mode (Swarm(..., neighbors=M)): the A tape is replaced by two int32 tapes, N_idx [L][E][N][M] and
N_cnt [L][E][N] (mrs_neighbors), that follow the A head through every rule above.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import NamedTuple

import torch

from . import _abi


# torch.cuda.current_stream() builds a Stream object (~7 us per call, a tenth of a small env.step); the raw
# handle is all the C ABI needs
_raw_stream = getattr(torch._C, '_cuda_getCurrentRawStream', None) or (
    lambda idx: torch.cuda.current_stream(idx).cuda_stream)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def unpack_adjacency(bits, N: int):
    """Inverse of mrs_pack_adjacency: int32 [..., N, ceil(N/32)] -> float32 {0,1} [..., N, N]."""
    b = bits.to(torch.int64) & 0xffffffff
    j = torch.arange(N, device=bits.device)
    return ((b[..., j // 32] >> (j % 32)) & 1).to(torch.float32)


class Neighbors(NamedTuple):
    """The COMM_RANGE graph as neighbour lists (mrs_neighbors): idx int32 [..., N, M] holds the neighbours of every
    agent in ascending order, padded with -1; count int32 [..., N] the true degree (count > M: the list was truncated
    to its first M entries).  Windows of MRS are [E, K+1, N, M] / [E, K+1, N] (unbatched [K+1, N, M] / [K+1, N]),
    newest first; a snapshot of Swarm.neighbors is [E, N, M] / [E, N]."""
    idx: torch.Tensor
    count: torch.Tensor

    def to_dense(self):
        """float32 {0,1} A [..., N, N] of the listed neighbours: the dense A of the same step when no row overflowed."""
        idx = self.idx.long()
        N = idx.shape[-2]
        A = torch.zeros(*idx.shape[:-1], N + 1, dtype=torch.float32, device=idx.device)
        A.scatter_(-1, torch.where(idx >= 0, idx, torch.full_like(idx, N)), 1.0)     # padding lands in column N
        return A[..., :N].contiguous()

    def edge_index(self, k=0):
        """int64 [2, nnz] edge list of hop slice k over the node index e*N + i: edge_index[0] = i (the agent whose
        list it is), edge_index[1] = j (its neighbour), in the row-major order of A.nonzero().  The graph is
        symmetric, so this is also PyG's source -> target list.  idx [E, K+1, N, M] or [K+1, N, M] (one env);
        k=None: no hop axis, [E, N, M] or [N, M] (a snapshot of Swarm.neighbors)."""
        idx = self.idx
        if k is not None:
            idx = idx.select(-3, k)
        N, M = idx.shape[-2], idx.shape[-1]
        idx = idx.reshape(math.prod(idx.shape[:-1]), M).long()
        rows = torch.arange(idx.shape[0], device=idx.device).unsqueeze(1).expand(-1, M)
        keep = idx >= 0
        return torch.stack([rows[keep], (rows - rows % N + idx)[keep]])


def shard_range(E_total: int, rank: int, world: int):
    """Contiguous env block owned by `rank` (SURVEY.md §8e): [lo, hi)."""
    base, rem = divmod(E_total, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


class Swarm:
    # neighbour mode (neighbors=M): lists per agent instead of the dense A tape (class defaults: dense mode)
    nbr = None
    N_idx = None
    N_cnt = None

    def __init__(self, E: int, N: int, K: int = 0, action_type='set_target_vel', state_layout=_abi.X_POS_VEL,
                 comm_range=float('inf'), dt=0.01, gravity=9.81, agent_radius=0.3, device='cuda', contact_radius=None,
                 tape_slots=None, want_A=True, custom_D=0, keep_rpm=False, ring=False, fresh_tapes=False, neighbors=None):
        """neighbors=M: the COMM_RANGE graph is kept as neighbour lists of at most M entries per agent (tapes N_idx
        [L][E][N][M] / N_cnt [L][E][N], mrs_neighbors) and no dense A tape is allocated.  Every stepping call then
        runs mrs_step without A followed by one mrs_neighbors launch per step, for every N: the one-launch
        mrs_step_many and the chained hand-over of mrs_rollout (N <= 32) never store the intermediate positions
        the lists are built from, so step_many / rollout / capture_rollout become per-step launches."""
        self.lib = _abi.lib()
        self.device = torch.device(device)
        if self.device.type != 'cuda':
            raise _abi.MrsError('mrsgym_b200 runs on CUDA devices only (no CPU fallback); got %s' % device)
        if self.device.index is None:
            self.device = torch.device('cuda', torch.cuda.current_device())
        if self.device.index != torch.cuda.current_device():
            # kernels are launched on the CURRENT device with raw pointers: one process per GPU
            raise _abi.MrsError('the swarm lives on %s but the current CUDA device is %d: call '
                                'torch.cuda.set_device first (one process per GPU)' % (self.device, torch.cuda.current_device()))
        self.E, self.N, self.K = int(E), int(N), int(K)
        self.S = self.E * self.N
        if neighbors is not None:
            if int(neighbors) < 0:
                raise ValueError('neighbors (list length M) must be >= 0')
            self.nbr = int(neighbors)
            want_A = False
        self.cfg = _abi.default_config()
        self.cfg.E, self.cfg.N, self.cfg.K = self.E, self.N, self.K
        self.set_action_type(action_type)
        self.cfg.state_layout = state_layout
        self.cfg.comm_range = float(comm_range)
        self.cfg.dt, self.cfg.gravity = float(dt), float(gravity)
        self.cfg.phys.agent_radius = float(agent_radius)
        # the agent-agent contact sphere: AGENT_RADIUS unless told otherwise (0.06 = the cf2x collision cylinder)
        self.cfg.phys.contact_radius = float(agent_radius if contact_radius is None else contact_radius)
        self.D = _abi.STATE_DIMS[state_layout] if state_layout != _abi.X_NONE else int(custom_D)
        if tape_slots:
            self.L = int(tape_slots)
        else:
            # default history depth: when a head reaches slot 0 the K newest slots move to the top (K copies of
            # a whole slice), so the move is amortised over L - K steps; deep tapes make it negligible.  Up to
            # 256 slots within a ~2 GB budget for X and A together (C5: 29 MB per slot -> 68 slots).
            D_ = _abi.STATE_DIMS[state_layout] if state_layout != _abi.X_NONE else int(custom_D)
            slot_bytes = 4 * self.S * (max(D_, 0) + (self.N if want_A else 0) + (self.nbr + 1 if self.nbr is not None else 0))
            self.L = max(2 * self.K + 2, 16, min(256, int(2e9 // max(slot_bytes, 1))))
        if self.L < (self.K + 1 if ring else 2 * self.K + 2):
            raise ValueError('tape_slots must be >= 2*K_HOPS+2 (K_HOPS+1 in ring mode)')
        self.cfg.L = self.L
        dev = self.device
        z = dict(device=dev, dtype=torch.float32)
        self.state = torch.zeros(_abi.STATE_PLANES, self.S, **z)
        self.state[6].fill_(1.0)                                  # identity quaternion (xyzw)
        self.ctrl = torch.zeros(_abi.CTRL_PLANES, self.S, **z)
        self.ctrl[9].fill_(float('nan'))                          # last_vel_e.x = NaN: never called
        self.rpm = torch.zeros(4, self.S, **z) if keep_rpm else None
        self.X_tape = torch.zeros(self.L, self.E, self.N, max(self.D, 1), **z) if self.D > 0 else None
        self.A_tape = torch.zeros(self.L, self.E, self.N, self.N, **z) if want_A else None
        if self.nbr is not None:
            self.N_idx = torch.full((self.L, self.E, self.N, self.nbr), -1, device=dev, dtype=torch.int32)
            self.N_cnt = torch.zeros(self.L, self.E, self.N, device=dev, dtype=torch.int32)
        self.scratch = torch.zeros(self.lib.mrs_scratch_planes(self.E, self.N), self.S, **z) if self.N > 32 else None
        self.status = torch.zeros(1, device=dev, dtype=torch.int32)
        self.stats = torch.zeros(_abi.STATS_SLOTS, device=dev, dtype=torch.int64)
        self.sync = torch.zeros(_abi.SYNC_WORDS, device=dev, dtype=torch.int64)    # range hand-over of mrs_rollout
        self.bufs = _abi.MrsBuffers()
        self._cfg_ref, self._bufs_ref = C.byref(self.cfg), C.byref(self.bufs)     # reused by the per-step calls
        self._mrs_step = self.lib.mrs_step
        self._bind()
        self.hx = self.L - self.K - 1
        self.ha = self.L - self.K - 1
        self.ring = bool(ring)     # True: heads wrap around the tape, nothing is ever moved (graph rollouts)
        # fresh tapes: a tape that has been written down to slot 0 (or is re-initialised by a reset) is not reused --
        # the next slots come from a NEW tensor, so a window view handed out earlier is never overwritten and stays
        # valid for as long as somebody holds it (reference semantics: every step returns fresh tensors) without a
        # copy per step.  Only for small slots: one held view keeps its whole tape generation alive.
        slot_bytes = 4 * self.S * (max(self.D, 0) + (self.N if want_A else 0) + (self.nbr + 1 if self.nbr is not None else 0))
        self.fresh = bool(fresh_tapes) and not self.ring and slot_bytes * self.L <= (64 << 20)
        self.generation = 0        # bumped whenever a fresh tape replaces the current one
        self.a_empty = True        # no A slice pushed since the last full reset (MRS.py:186)
        self._stats_sum = None     # result buffer of allreduce_stats(comm)
        self.launches = 0          # kernel launches issued through the ABI (bench: gpu_launches)
        self._launches_per_step = self._step_launches()

    # ------------------------------------------------------------------ plumbing
    def _bind(self):
        b = self.bufs
        b.state, b.ctrl = self.state.data_ptr(), self.ctrl.data_ptr()
        b.rpm = self.rpm.data_ptr() if self.rpm is not None else None
        b.X_tape = self.X_tape.data_ptr() if (self.X_tape is not None and self.cfg.state_layout != _abi.X_NONE) else None
        b.A_tape = self.A_tape.data_ptr() if self.A_tape is not None else None
        b.scratch = self.scratch.data_ptr() if self.scratch is not None else None
        b.status, b.stats = self.status.data_ptr(), self.stats.data_ptr()
        b.sync = self.sync.data_ptr()

    def _stream(self):
        if torch.cuda.current_device() != self.device.index:
            raise _abi.MrsError('current CUDA device changed to %d; the swarm lives on %s' % (torch.cuda.current_device(), self.device))
        return C.c_void_p(_raw_stream(self.device.index))

    def set_action_type(self, action_type):
        if action_type is None:
            self.cfg.action_type = _abi.NO_ACTION
        elif isinstance(action_type, str):
            if action_type not in _abi.ACTION_TYPES:
                # the reference dispatches with getattr(agent, behaviour) (Environment.py:92)
                raise AttributeError("'Quadcopter' object has no attribute '%s'" % action_type)
            self.cfg.action_type = _abi.ACTION_TYPES[action_type]
        else:
            self.cfg.action_type = int(action_type)
        return _abi.ACTION_DIMS[self.cfg.action_type]

    @property
    def action_dim(self):
        return _abi.ACTION_DIMS[self.cfg.action_type]

    # ------------------------------------------------------------------ tapes
    def _make_room(self, which: int, need: int = 1):
        """Ensure `need` free slots below the head of tape `which` (1 = X, 2 = A)."""
        head = self.hx if which == 1 else self.ha
        if head >= need:
            return head
        K, L = self.K, self.L
        if self.ring:                # ring mode (graph rollouts): wrap around, nothing is moved
            return L
        tape = self.X_tape if which == 1 else self.A_tape
        if which == 2 and self.N_idx is not None:     # neighbour tapes: torch copies of the K newest slots
            if self.fresh:
                new = (torch.empty_like(self.N_idx), torch.empty_like(self.N_cnt))
                if K > 0:
                    new[0][L - K:L], new[1][L - K:L] = self.N_idx[head:head + K], self.N_cnt[head:head + K]
                self._swap_nbr(*new)
            elif K > 0:
                self.N_idx[L - K:L] = self.N_idx[head:head + K].clone()
                self.N_cnt[L - K:L] = self.N_cnt[head:head + K].clone()
        elif tape is not None and self.fresh:
            new = torch.empty_like(tape)
            if K > 0:
                new[L - K:L] = tape[head:head + K]
            self._swap_tape(which, new)
        elif tape is not None and K > 0 and which == 1 and self.cfg.state_layout == _abi.X_NONE:
            tape[L - K:L] = tape[head:head + K].clone()      # python-written X (custom state_fn)
        elif tape is not None and K > 0:
            for i in range(K - 1, -1, -1):           # move the K newest slots to the top
                _abi.check(self.lib.mrs_tape_fill(C.byref(self.cfg), C.byref(self.bufs), which, head + i,
                                                  L - K + i, 1, self._stream()), 'mrs_tape_fill')
                self.launches += 1
        head = L - K
        if which == 1:
            self.hx = head
        else:
            self.ha = head
        return head

    def _swap_tape(self, which, new):
        if which == 1:
            self.X_tape = new
            if self.cfg.state_layout != _abi.X_NONE:
                self.bufs.X_tape = new.data_ptr()
        else:
            self.A_tape = new
            self.bufs.A_tape = new.data_ptr()
        self.generation += 1

    def _swap_nbr(self, new_idx, new_cnt):
        self.N_idx, self.N_cnt = new_idx, new_cnt
        self.generation += 1

    def _has_A(self):
        """An A history is kept: the dense A tape or the neighbour tapes."""
        return self.A_tape is not None or self.N_idx is not None

    def _push_neighbors(self, slot):
        """mrs_neighbors of the current positions into neighbour-tape slot `slot`."""
        S, M = self.S, self.nbr
        idx = self.N_idx.data_ptr() + 4 * slot * S * M
        rc = self.lib.mrs_neighbors(self._cfg_ref, self._bufs_ref, M, C.c_void_p(idx if M else 0),
                                    C.c_void_p(self.N_cnt.data_ptr() + 4 * slot * S), self._stream())
        if rc:
            _abi.check(rc, 'mrs_neighbors')
        self.launches += 1

    def renew_tapes(self):
        """Fresh-tape mode: continue on new tapes (the current windows move to their top), so that an in-place edit
        of the history -- a masked reset -- does not show through windows handed out earlier."""
        if not self.fresh:
            return
        if self.N_idx is not None:
            n = min(self.K + 1, self.L - self.ha)
            new = (torch.empty_like(self.N_idx), torch.empty_like(self.N_cnt))
            new[0][self.L - n:], new[1][self.L - n:] = self.N_idx[self.ha:self.ha + n], self.N_cnt[self.ha:self.ha + n]
            self._swap_nbr(*new)
            self.ha = self.L - n
        for which in (1, 2):
            tape = self.X_tape if which == 1 else self.A_tape
            if tape is None:
                continue
            head = self.hx if which == 1 else self.ha
            n = min(self.K + 1, self.L - head)
            new = torch.empty_like(tape)
            new[self.L - n:] = tape[head:head + n]
            self._swap_tape(which, new)
            if which == 1:
                self.hx = self.L - n
            else:
                self.ha = self.L - n

    def max_chunk(self):
        """Largest T a single mrs_step_many may take with this tape size."""
        return self.L - self.K

    def reset_windows(self, write_X=True):
        """Ring state after MRS.reset/set (MRS.py:185-192): X window = K+1 copies of X0, A window
        empty (reads as zeros, MRS.py:107-108)."""
        K, L = self.K, self.L
        self.hx = self.ha = L - K - 1
        st = self._stream()
        if self.fresh:             # the windows handed out before the reset keep their contents
            if self.X_tape is not None:
                self._swap_tape(1, torch.empty_like(self.X_tape))
            if self.A_tape is not None:
                self._swap_tape(2, torch.empty_like(self.A_tape))
            if self.N_idx is not None:
                self._swap_nbr(torch.empty_like(self.N_idx), torch.empty_like(self.N_cnt))
        if self.X_tape is not None:
            if write_X and self.cfg.state_layout != _abi.X_NONE:
                _abi.check(self.lib.mrs_observe(C.byref(self.cfg), C.byref(self.bufs), self.hx, 1, 0, st), 'mrs_observe')
                self.launches += 1
            if K > 0 and self.cfg.state_layout != _abi.X_NONE:
                _abi.check(self.lib.mrs_tape_fill(C.byref(self.cfg), C.byref(self.bufs), 1, self.hx, self.hx + 1, K, st),
                           'mrs_tape_fill')
                self.launches += 1
        if self.A_tape is not None:
            _abi.check(self.lib.mrs_tape_fill(C.byref(self.cfg), C.byref(self.bufs), 2, -1, self.ha, K + 1, st),
                       'mrs_tape_fill')
            self.launches += 1
            self.ha += 1          # empty deque: the first push lands on slot L-K-1
        if self.N_idx is not None:    # empty window: no neighbours, cnt = 0
            self.N_idx[self.ha:self.ha + K + 1].fill_(-1)
            self.N_cnt[self.ha:self.ha + K + 1].zero_()
            self.ha += 1
        self.a_empty = True

    def fill_X_history(self):
        """Custom state_fn path: replicate slot hx into the K older slots (python wrote X0 there)."""
        for sl in self.window_slots(1)[1:]:
            self.X_tape[sl] = self.X_tape[self.hx]

    def window_slots(self, which: int):
        """Tape slots of the newest-first K+1 window of tape `which` (1 = X, 2 = A)."""
        h = self.hx if which == 1 else self.ha
        return [(h + k) % self.L for k in range(self.K + 1)] if self.ring else list(range(h, min(h + self.K + 1, self.L)))

    def _window(self, tape, h):
        if self.ring and h + self.K + 1 > self.L:      # wrapped: the only case that copies
            return torch.cat([tape[h:], tape[:h + self.K + 1 - self.L]], dim=0)
        return tape[h:h + self.K + 1]

    def X_window(self):
        return self._window(self.X_tape, self.hx)                 # [K+1, E, N, D], newest first

    def A_window(self):
        return self._window(self.A_tape, self.ha)                 # [K+1, E, N, N]

    def N_window(self):
        """Neighbour mode: the newest-first K+1 window as Neighbors([K+1, E, N, M], [K+1, E, N])."""
        return Neighbors(self._window(self.N_idx, self.ha), self._window(self.N_cnt, self.ha))

    def neighbors(self, M):
        """mrs_neighbors of the current positions, one-off (any mode): Neighbors([E, N, M], [E, N]).  A degree above
        M sets STATUS_NEIGHBOR_OVERFLOW (read_status) and counts in read_stats()['neighbor_overflow']."""
        M = int(M)
        idx = torch.empty(self.E, self.N, M, dtype=torch.int32, device=self.device)
        cnt = torch.empty(self.E, self.N, dtype=torch.int32, device=self.device)
        _abi.check(self.lib.mrs_neighbors(self._cfg_ref, self._bufs_ref, M, _ptr(idx) if M else C.c_void_p(0), _ptr(cnt),
                                          self._stream()), 'mrs_neighbors')
        self.launches += 1
        return Neighbors(idx, cnt)

    # ------------------------------------------------------------------ the step
    def _check_actions(self, actions, T=1, host=False):
        """The C ABI reads raw pointers: refuse anything that is not float32, contiguous, of the
        right size and on the right device before it gets there."""
        adim = self.action_dim
        if adim == 0:
            return
        if actions is None:
            raise ValueError('ACTION_TYPE needs actions of shape [%d, %d, %d]' % (self.E, self.N, adim))
        if actions.dtype != torch.float32 or not actions.is_contiguous():
            raise ValueError('actions must be a contiguous float32 tensor')
        if actions.numel() != T * self.S * adim:
            raise ValueError('actions has %d elements, expected %d x %d x %d x %d' % (actions.numel(), T, self.E, self.N, adim))
        if host:
            if actions.is_cuda or not actions.is_pinned():
                raise ValueError('host actions must live in pinned host memory')
        elif actions.device != self.device:
            raise ValueError('actions live on %s, the swarm on %s' % (actions.device, self.device))
        if (adim == 4 or self.N in (8, 16, 32)) and actions.data_ptr() % 16:
            # these shapes read actions with 16-byte cp.async / float4 loads: a misaligned pointer would be a sticky
            # CUDA fault instead of a Python exception (3-component actions of other swarm sizes are read per float)
            raise ValueError('actions must start on a 16-byte boundary (got a view at offset %d of its storage); '
                             'pass actions.clone()' % actions.storage_offset())

    def _dense_only(self, what):
        if self.nbr is not None:
            raise _abi.MrsError('%s copies dense A slices to the host; it has no neighbour-list form (build the swarm '
                                'without neighbors=)' % what)

    def _step_launches(self, n=1, fused=False):
        """Kernels the library launches for n steps (bench: gpu_launches).  N <= 32: one fused kernel per step
        (per call when `fused`: mrs_step_many), plus one for a ragged last warp-chunk when N is 8, 16 or 32 and E
        is not a multiple of 32 / N.  N > 32: pre (+ per-agent kernel for N > 128), per-env contact, post, adjacency per
        step; 32 < N <= 128 with >= 32768 agents: one fused launch per step."""
        if self.N <= 32:
            gpw = 32 // self.N if self.N in (8, 16, 32) else 0
            per = 1 + (1 if gpw and self.E % gpw and self.E >= gpw else 0)
            return per if fused else per * n
        if self.N <= 128 and self.S >= 32768:
            return n                     # one CTA per env: the whole step incl. the A slice in one launch (step_env_kernel)
        return n * ((3 if self.N > 128 else 2) + (1 if self.N > 1 else 0) + (1 if self.A_tape is not None else 0))

    def step(self, actions):
        """One env.step for all envs.  actions: device float32 [E,N,A] contiguous, or None."""
        self._check_actions(actions)
        hx = self._make_room(1) - 1 if self.X_tape is not None else 0
        ha = self._make_room(2) - 1 if self._has_A() else 0
        rc = self._mrs_step(self._cfg_ref, self._bufs_ref, _ptr(actions), hx, ha, self._stream())
        if rc:
            _abi.check(rc, 'mrs_step')
        self.launches += self._launches_per_step
        if self.nbr is not None:
            self._push_neighbors(ha)
        if self.X_tape is not None:
            self.hx = hx
        if self._has_A():
            self.ha = ha
            self.a_empty = False

    def step_many(self, actions, T: int):
        """T steps with pre-computed actions [T,E,N,A]; chunks at tape wrap-arounds.  Neighbour mode: T steps of
        step() (the lists need the positions of every step)."""
        self._check_actions(actions, T)
        if self.nbr is not None:
            return self.step_many_single(actions, T)
        done = 0
        while done < T:
            hx = self._make_room(1) if self.X_tape is not None else T
            ha = self._make_room(2) if self.A_tape is not None else T
            n = min(T - done, hx, ha)
            a = actions[done:done + n] if actions is not None else None
            _abi.check(self.lib.mrs_step_many(C.byref(self.cfg), C.byref(self.bufs), _ptr(a), n, hx - 1, ha - 1,
                                              self._stream()), 'mrs_step_many')
            self.launches += self._step_launches(n, fused=True)
            if self.X_tape is not None:
                self.hx = hx - n
            if self.A_tape is not None:
                self.ha = ha - n
                self.a_empty = False
            done += n

    def step_many_single(self, actions, T: int):
        """T steps as T separate mrs_step launches (each reads and writes the state in HBM)."""
        for t in range(T):
            self.step(actions[t] if actions is not None else None)

    def rollout(self, actions, T: int):
        """mrs_rollout: T steps as T single-step launches issued by ONE C call; for N in {8, 16, 32} at scale the
        launches are chained (range hand-over through `sync`, no grid-wide dependency).  Chunks at tape wrap-arounds.
        Neighbour mode: T steps of step() (mrs_step + mrs_neighbors each, never chained)."""
        self._check_actions(actions, T)
        if self.nbr is not None:
            return self.step_many_single(actions, T)
        done = 0
        while done < T:
            hx = self._make_room(1) if self.X_tape is not None else T
            ha = self._make_room(2) if self.A_tape is not None else T
            n = min(T - done, hx, ha)
            a = actions[done:done + n] if actions is not None else None
            _abi.check(self.lib.mrs_rollout(self._cfg_ref, self._bufs_ref, _ptr(a), n, hx - 1, ha - 1, self._stream()),
                       'mrs_rollout')
            self.launches += self._step_launches(n)
            if self.X_tape is not None:
                self.hx = hx - n
            if self.A_tape is not None:
                self.ha = ha - n
                self.a_empty = False
            done += n

    def capture_rollout(self, actions, T: int, stats_comm=None):
        """CUDA-graph a T-step rollout (launch-bound loops belong in graphs): returns a
        GraphRollout whose replay() advances all envs by T steps reading actions[t] from the
        given device buffer (refill it between replays).  Capturing itself leaves the swarm where it was.  The swarm switches to ring mode (tape heads
        wrap around, no slots are moved); T must be a multiple of the tape size, so every replay
        ends on the slots it started from (pass tape_slots=T to the constructor).  stats_comm (dist.PeerComm):
        the per-rollout statistics reduction becomes the last node of the graph (result: swarm._stats_sum)."""
        return GraphRollout(self, actions, T, stats_comm)

    def push_A(self):
        """MRS.calc_Ak outside step: adjacency (neighbour mode: the neighbour lists) of the current positions becomes
        the newest slot."""
        ha = self._make_room(2) - 1
        if self.nbr is not None:
            self._push_neighbors(ha)
        else:
            _abi.check(self.lib.mrs_observe(C.byref(self.cfg), C.byref(self.bufs), ha, 0, 1, self._stream()), 'mrs_observe')
            self.launches += 1
        self.ha = ha
        self.a_empty = False

    def push_X(self):
        hx = self._make_room(1) - 1
        if self.cfg.state_layout != _abi.X_NONE:
            _abi.check(self.lib.mrs_observe(C.byref(self.cfg), C.byref(self.bufs), hx, 1, 0, self._stream()), 'mrs_observe')
            self.launches += 1
        self.hx = hx
        return hx

    def step_host(self, actions_host, dev_actions, X_host, A_host, Abits_host=None, dev_Abits=None):
        """mrs_step_host: pinned host actions in, newest X/A slice out, synchronous.  Abits_host (pinned int32
        [E,N,ceil(N/32)]) + dev_Abits (device staging of the same shape): the adjacency bit-packed for the wire."""
        self._check_actions(actions_host, host=True)
        self._dense_only('step_host')
        hx = self._make_room(1) - 1 if self.X_tape is not None else 0
        ha = self._make_room(2) - 1 if self.A_tape is not None else 0
        _abi.check(self.lib.mrs_step_host(C.byref(self.cfg), C.byref(self.bufs), _ptr(actions_host), _ptr(dev_actions),
                                          _ptr(X_host), _ptr(A_host), _ptr(Abits_host), _ptr(dev_Abits), hx, ha, self._stream()),
                   'mrs_step_host')
        self.launches += self._step_launches()
        if self.X_tape is not None:
            self.hx = hx
        if self.A_tape is not None:
            self.ha = ha
            self.a_empty = False

    def rollout_host(self, actions_host, dev_actions2, X_host=None, A_host=None, Abits_host=None, dev_Abits2=None):
        """mrs_rollout_host: T steps from pinned host actions [T,E,N,A] with the newest X / A slice of
        every step copied to pinned host arrays [T,E,N,D] / [T,E,N,N] (and / or the adjacency bit-packed:
        Abits_host int32 [T,E,N,ceil(N/32)] with dev_Abits2 [2,E,N,ceil(N/32)] device staging); copies overlap the kernels.
        Chunks at tape wrap-arounds."""
        T = int(actions_host.shape[0])
        self._check_actions(actions_host, T, host=True)
        self._dense_only('rollout_host')
        done = 0
        while done < T:
            hx = self._make_room(1) if self.X_tape is not None else T
            ha = self._make_room(2) if self.A_tape is not None else T
            n = min(T - done, hx, ha)
            _abi.check(self.lib.mrs_rollout_host(
                C.byref(self.cfg), C.byref(self.bufs), _ptr(actions_host[done:done + n]), _ptr(dev_actions2),
                _ptr(X_host[done:done + n]) if X_host is not None else C.c_void_p(0),
                _ptr(A_host[done:done + n]) if A_host is not None else C.c_void_p(0),
                _ptr(Abits_host[done:done + n]) if Abits_host is not None else C.c_void_p(0), _ptr(dev_Abits2),
                n, hx - 1, ha - 1, self._stream()), 'mrs_rollout_host')
            self.launches += self._step_launches(n)
            if self.X_tape is not None:
                self.hx = hx - n
            if self.A_tape is not None:
                self.ha = ha - n
                self.a_empty = False
            done += n

    # ------------------------------------------------------------------ state access
    def set_state(self, pos=None, ori=None, vel=None, angvel=None, env_mask=None):
        """Environment.set_state -> Object.set_state (Environment.py:97-103, Object.py:42-65).
        Each of pos/ori(euler xyz)/vel/angvel: [E,N,3] (or [N,3], broadcast over envs) or None = keep."""
        def prep(x):
            if x is None:
                return None
            x = torch.as_tensor(x, dtype=torch.float32).to(self.device)
            if x.dim() == 2:
                x = x.unsqueeze(0).expand(self.E, -1, -1)
            return x.reshape(self.E, self.N, 3).contiguous()
        pos, ori, vel, angvel = prep(pos), prep(ori), prep(vel), prep(angvel)
        if env_mask is not None:
            env_mask = torch.as_tensor(env_mask).to(self.device).to(torch.uint8).reshape(self.E).contiguous()
        _abi.check(self.lib.mrs_set_state(C.byref(self.cfg), C.byref(self.bufs), _ptr(pos), _ptr(ori), _ptr(vel),
                                          _ptr(angvel), _ptr(env_mask), self._stream()), 'mrs_set_state')
        self.launches += 1

    def spawn(self, seed, env_mask=None, z=(1.0, 3.0), xy_radius=1.0, xy_sigma=1.0, yaw=(-math.pi / 2, math.pi / 2),
              max_rounds=256, env_offset=0):
        """On-device reset with the reference's default start distribution (mrs_spawn), any N: a warp per env for
        N <= 32, a CTA per env above.  Agents closer than 2*agent_radius to a lower-indexed agent of their env are
        re-drawn, for at most max_rounds rounds.  env_offset: global index of this shard's first env (the draws are
        keyed by seed and GLOBAL env index, so the ranks of a sharded job sample different environments; the result
        does not depend on E or env_mask).  Returns the device counter of envs whose rejection sampling did not
        converge within max_rounds (read it lazily); those envs keep their last draw."""
        if env_mask is not None:
            env_mask = torch.as_tensor(env_mask).to(self.device).to(torch.uint8).reshape(self.E).contiguous()
        failed = torch.zeros(1, device=self.device, dtype=torch.int32)
        _abi.check(self.lib.mrs_spawn(C.byref(self.cfg), C.byref(self.bufs), _ptr(env_mask), C.c_ulonglong(int(seed)),
                                      C.c_ulonglong(int(env_offset)), float(z[0]), float(z[1]), float(xy_radius), float(xy_sigma), float(yaw[0]),
                                      float(yaw[1]), int(max_rounds), _ptr(failed), self._stream()), 'mrs_spawn')
        self.launches += 1
        return failed

    def autoreset(self, seed, env_steps, episode, done_out, done_in=None, slot_x=None, slot_a=None, z=(1.0, 3.0),
                  xy_radius=1.0, xy_sigma=1.0, yaw=(-math.pi / 2, math.pi / 2), max_rounds=256, env_offset=0,
                  episode_length=0, max_timesteps=-1, failed=None):
        """mrs_autoreset: the per-step episode bookkeeping of a closed loop, after the step.  env_steps (int32 [E]) and
        episode (int32 [E], read as unsigned) are device counters updated in place; done_out (uint8 / bool [E]) receives
        done[t]; done_in (bool / uint8 [E] or None) is the done_fn result.  Done envs are redrawn with the default start
        distribution keyed by (seed, env_offset + e, episode + 1), their K+1 X window becomes X0 and their A window
        A0 followed by K zero slices; the other envs only count the step.  slot_x / slot_a: the newest slots of the
        windows (default: the current heads).  failed (int32 [1], added to): envs whose rejection sampling did not
        converge.  Stream-ordered and capturable."""
        for t, what in ((env_steps, 'env_steps'), (episode, 'episode')):
            if t.dtype != torch.int32 or not t.is_contiguous() or t.numel() != self.E or t.device != self.device:
                raise ValueError('%s must be a contiguous int32 [%d] tensor on %s' % (what, self.E, self.device))
        if done_out.dtype not in (torch.uint8, torch.bool) or not done_out.is_contiguous() or done_out.numel() != self.E:
            raise ValueError('done_out must be a contiguous uint8 / bool [%d] tensor' % self.E)
        if done_in is not None and (done_in.dtype not in (torch.uint8, torch.bool) or not done_in.is_contiguous()
                                    or done_in.numel() != self.E):
            raise ValueError('done_in must be a contiguous uint8 / bool [%d] tensor' % self.E)
        a = _abi.MrsAutoResetArgs(int(seed), int(env_offset), float(z[0]), float(z[1]), float(xy_radius), float(xy_sigma),
                                  float(yaw[0]), float(yaw[1]), int(max_rounds), int(episode_length), int(max_timesteps))
        _abi.check(self.lib.mrs_autoreset(self._cfg_ref, self._bufs_ref, C.byref(a), _ptr(done_in), _ptr(env_steps),
                                          _ptr(episode), _ptr(done_out), self.hx if slot_x is None else int(slot_x),
                                          self.ha if slot_a is None else int(slot_a), _ptr(failed), self._stream()),
                   'mrs_autoreset')
        self.launches += 1

    def set_quat(self, quat):
        """Exact quaternion upload (xyzw), bypassing the euler conversion (tests / checkpoints)."""
        q = torch.as_tensor(quat, dtype=torch.float32).to(self.device).reshape(self.S, 4)
        self.state[3:7] = q.t()

    def _planes(self, lo, hi):
        return self.state[lo:hi].t().reshape(self.E, self.N, hi - lo)

    def get_pos(self):
        return self._planes(0, 3)

    def get_quat(self):
        return self._planes(3, 7)

    def get_vel(self):
        return self._planes(7, 10)

    def get_angvel(self):
        return self._planes(10, 13)

    def get_ori(self):
        """euler 'xyz' [roll, pitch, yaw] as scipy's as_euler('xyz') (Object.get_ori, Object.py:90-97)."""
        x, y, z, w = (self.state[i] for i in range(3, 7))
        roll = torch.atan2(2 * (w * x + y * z), 1 - 2 * (x * x + y * y))
        pitch = torch.asin(torch.clamp(2 * (w * y - z * x), -1.0, 1.0))
        yaw = torch.atan2(2 * (w * z + x * y), 1 - 2 * (y * y + z * z))
        return torch.stack([roll, pitch, yaw], dim=-1).reshape(self.E, self.N, 3)

    def get_rotmat(self):
        """body->world rotation matrices [E, N, 3, 3] (Object.get_ori(mat=True), Object.py:90-95)."""
        x, y, z, w = (self.state[i] for i in range(3, 7))
        R = torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w),
                         2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w),
                         2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)], dim=-1)
        return R.reshape(self.E, self.N, 3, 3)

    def contact_points(self, body=False, threshold=None):
        """Contact candidates of every agent on the contact geometry of the step (see Environment.get_contact_points):
        slot 0 the nearest other agent (contact spheres), slots 1-4 the lower-rim points of the collision cylinder
        against the ground.  Derived from the device state with torch ops (a diagnostic, not on the step path)."""
        ph = self.cfg.phys
        thr = float(ph.contact_margin if threshold is None else threshold)
        pr = self.proximity(thr)
        pos, R = self.get_pos(), self.get_rotmat()
        E, N, dev = self.E, self.N, self.device
        j = pr['nearest'].long().clamp(min=0)
        pj = torch.gather(pos, 1, j.unsqueeze(-1).expand(E, N, 3))
        d = pos - pj
        dist = d.norm(dim=-1, keepdim=True).clamp(min=1e-12)
        n_a = d / dist                                                    # on the agent: away from the partner
        rc = float(ph.contact_radius)
        p_a = pos - n_a * rc
        has_a = (pr['nearest'] >= 0) & (pr['gap_agent'] < thr)
        # rim points: c = (+-r, 0, cz), (0, +-r, cz), cz = -h sign(R22)
        r_, h_ = float(ph.col_radius), float(ph.col_halfheight)
        sgn = torch.where(R[..., 2, 2] >= 0, 1.0, -1.0)
        c = torch.zeros(E, N, 4, 3, device=dev)
        c[..., 0, 0], c[..., 1, 1], c[..., 2, 0], c[..., 3, 1] = r_, r_, -r_, -r_
        c[..., 2] = (-h_ * sgn).unsqueeze(-1)
        pw = pos.unsqueeze(2) + torch.einsum('enij,enpj->enpi', R, c)
        gdist = pw[..., 2] - float(ph.col_margin) - float(ph.ground_z)
        obj = torch.full((E, N, 5), -1, dtype=torch.int64, device=dev)
        obj[..., 0] = torch.where(has_a, pr['nearest'].long(), torch.full_like(j, -1))
        obj[..., 1:] = torch.where(gdist < thr, torch.full_like(gdist, float(N)).long(), torch.full_like(gdist, -1.0).long())
        P = torch.cat([p_a.unsqueeze(2), pw], dim=2)
        nrm = torch.zeros(E, N, 5, 3, device=dev)
        nrm[..., 0, :] = n_a
        nrm[..., 1:, 2] = 1.0
        D = torch.cat([pr['gap_agent'].unsqueeze(-1), gdist], dim=-1)
        if body:
            P = torch.einsum('enji,enpj->enpi', R, P - pos.unsqueeze(2))
            nrm = torch.einsum('enji,enpj->enpi', R, nrm)
        return {'object': obj, 'pos': P, 'normal': nrm, 'distance': D, 'mask': obj >= 0}

    def adjacency(self, pos):
        """MRS.calc_A on arbitrary float32 positions [E,N,3] -> [E,N,N] (bit-exact with torch CPU)."""
        pos = torch.as_tensor(pos, dtype=torch.float32).to(self.device).reshape(self.E, self.N, 3).contiguous()
        A = torch.empty(self.E, self.N, self.N, device=self.device, dtype=torch.float32)
        _abi.check(self.lib.mrs_adjacency(C.byref(self.cfg), _ptr(pos), _ptr(A), self._stream()), 'mrs_adjacency')
        self.launches += 1
        return A

    def pack_adjacency(self, A):
        """mrs_pack_adjacency: float32 A [E,N,N] on the device -> int32 [E,N,ceil(N/32)] (bit j of word w = A[..., 32w+j])."""
        A = A.contiguous()
        out = torch.empty(self.E, self.N, (self.N + 31) // 32, dtype=torch.int32, device=self.device)
        _abi.check(self.lib.mrs_pack_adjacency(self._cfg_ref, _ptr(A), _ptr(out), self._stream()), 'mrs_pack_adjacency')
        self.launches += 1
        return out

    def proximity(self, threshold=0.04):
        """mrs_proximity: dict of [E,N] tensors -- 'gap_agent' (to the nearest other agent), 'nearest'
        (its index, -1 if N == 1), 'gap_ground', 'collision' (bool, any gap < threshold)."""
        z = dict(device=self.device)
        ga = torch.empty(self.E, self.N, dtype=torch.float32, **z)
        ne = torch.empty(self.E, self.N, dtype=torch.int32, **z)
        gg = torch.empty(self.E, self.N, dtype=torch.float32, **z)
        co = torch.empty(self.E, self.N, dtype=torch.uint8, **z)
        _abi.check(self.lib.mrs_proximity(C.byref(self.cfg), C.byref(self.bufs), float(threshold), _ptr(ga), _ptr(ne),
                                          _ptr(gg), _ptr(co), self._stream()), 'mrs_proximity')
        self.launches += 1
        return {'gap_agent': ga, 'nearest': ne, 'gap_ground': gg, 'collision': co.bool()}

    def raycast(self, directions, offset=(0.0, 0.0, 0.0), body=True, RANGE=100.0):
        """mrs_raycast: directions [R,3] (body or world frame) for every agent -> {'dist' [E,N,R] (inf =
        no hit), 'object' [E,N,R] int (-1 none, N ground, j agent j)} (Object.raycast, Object.py:143-174)."""
        d = torch.as_tensor(directions, dtype=torch.float32).reshape(-1, 3).to(self.device).contiguous()
        R = d.shape[0]
        dist = torch.empty(self.E, self.N, R, dtype=torch.float32, device=self.device)
        obj = torch.empty(self.E, self.N, R, dtype=torch.int32, device=self.device)
        off = (C.c_float * 3)(*[float(v) for v in offset])
        _abi.check(self.lib.mrs_raycast(C.byref(self.cfg), C.byref(self.bufs), _ptr(d), R, off, 1 if body else 0,
                                        float(RANGE), _ptr(dist), _ptr(obj), self._stream()), 'mrs_raycast')
        self.launches += 1
        return {'dist': dist, 'object': obj}

    def read_status(self, clear=True):
        v = int(self.status.item())
        if clear and v:
            self.status.zero_()
        return v

    def read_stats(self):
        v = self.stats.tolist()
        return {n: v[i] for i, n in enumerate(_abi.STAT_NAMES)}

    def allreduce_stats(self, comm=None, group=None):
        """Per-rollout statistics reduction across env shards: the ONLY exchange of the path (SURVEY.md §8e).
        comm = dist.PeerComm: the library's peer-memory kernel (mrs_stats_allreduce) on the current stream, no
        host involvement, capturable in a CUDA graph; the result tensor is reused between calls.
        comm = None: torch.distributed all-reduce (gloo in the CPU tests, NCCL otherwise)."""
        if comm is not None:
            if self._stats_sum is None:
                self._stats_sum = torch.zeros_like(self.stats)
            _abi.check(self.lib.mrs_stats_allreduce(self._cfg_ref, self._bufs_ref, comm.handle, _ptr(self._stats_sum),
                                                    self._stream()), 'mrs_stats_allreduce')
            self.launches += 1
            return self._stats_sum
        from .dist import allreduce_stats
        return allreduce_stats(self.stats, group)


class GraphRollout:
    def __init__(self, swarm: Swarm, actions, T: int, stats_comm=None):
        sw = self.swarm = swarm
        self.stats_comm = stats_comm
        if T < 1 or T % sw.L != 0:
            raise ValueError('capture_rollout: T=%d must be a multiple of the tape size (%d slots); build the '
                             'swarm with tape_slots=T' % (T, sw.L))
        if sw.X_tape is not None and sw.cfg.state_layout == _abi.X_NONE:
            raise RuntimeError('capture_rollout needs a fused state layout')
        if actions is not None and tuple(actions.shape[:3]) != (T, sw.E, sw.N):
            raise ValueError('actions must be [T, E, N, A]')
        self.T, self.actions = T, actions
        sw.ring = True
        self.launches_per_replay = 0
        torch.cuda.synchronize(sw.device)
        self.graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(device=sw.device)
        side.wait_stream(torch.cuda.current_stream(sw.device))
        with torch.cuda.stream(side):
            # warm-up outside capture (lazy module load, per-function attributes): it advances the swarm by T
            # steps, so everything a later step can read is put back afterwards -- state, PID planes, counters
            # and the K+1 observation windows (the rest of the tapes is history nobody can reach any more)
            keep = [(t, t.clone()) for t in (sw.state, sw.ctrl, sw.status, sw.stats, sw.rpm) if t is not None]
            for tape, which in ((sw.X_tape, 1), (sw.A_tape, 2), (sw.N_idx, 2), (sw.N_cnt, 2)):
                if tape is not None:
                    keep += [(tape[sl], tape[sl].clone()) for sl in sw.window_slots(which)]
            heads = (sw.hx, sw.ha, sw.a_empty, sw.launches)
            self._body()
            for dst, src in keep:
                dst.copy_(src)
            sw.hx, sw.ha, sw.a_empty, sw.launches = heads
            torch.cuda.synchronize(sw.device)
            with torch.cuda.graph(self.graph, stream=side):
                before = sw.launches
                self._body()        # the heads come back to where they were: T is a multiple of L
                self.launches_per_replay = sw.launches - before
        torch.cuda.current_stream(sw.device).wait_stream(side)
        torch.cuda.synchronize(sw.device)

    def _body(self):
        sw = self.swarm
        if sw.nbr is not None:
            sw.step_many_single(self.actions, self.T)   # mrs_step + mrs_neighbors per step
        elif sw.N > 32:
            sw.step_many(self.actions, self.T)       # wide path: per-step kernels anyway, adjacency overlapped
        else:
            sw.rollout(self.actions, self.T)             # single-step launches, chained where the shape allows
        if self.stats_comm is not None:
            sw.allreduce_stats(self.stats_comm)

    def replay(self):
        self.graph.replay()
        self.swarm.launches += self.launches_per_replay
        self.swarm.a_empty = False
