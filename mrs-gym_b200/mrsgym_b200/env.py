"""MRS: the reference's Gym environment class, batched over N_ENVS and running on the B200.

Mirrors /root/reference/mrsgym/MRS.py:12-293 for the step path: same constructor kwargs
(N_AGENTS, K_HOPS, COMM_RANGE, ACTION_TYPE, AGENT_RADIUS, MAX_TIMESTEPS, START_POS, START_ORI,
DT, GRAVITY, ...), same `step(actions, ACTION_TYPE=None) -> (X, reward, done, info)` with
info["A"], same callback order (update -> reward -> last_obs := X -> info -> done ->
steps_since_reset += 1, MRS.py:260-274), same ring semantics (X padded with copies, A with
zeros).  New kwargs: N_ENVS (batch of independent worlds; default 1 = reference shapes),
DEVICE, TAPE_SLOTS, CHECK_NAN, COPY_OBS, A_FORMAT, MAX_NEIGHBORS.

Shapes: N_ENVS == 1 -> X (K+1, N, D), A (K+1, N, N) exactly like the reference;
        N_ENVS  > 1 -> X [E, K+1, N, D], A [E, K+1, N, N] (zero-copy views of the device tapes
        unless COPY_OBS; a view stays valid for at least TAPE_SLOTS - 2*K_HOPS - 2 further steps).

A_FORMAT='neighbors': get_Ak(), info['A'], the A= argument of the callbacks, calc_Ak() and refresh_A() return
Neighbors windows instead of the dense A: idx [E, K+1, N, M] (neighbours in ascending order, -1 padded) and count
[E, K+1, N] (unbatched [K+1, N, M] / [K+1, N]), newest first, M = MAX_NEIGHBORS (default min(N_AGENTS - 1, 64)).
No dense A history is kept; calc_A() stays dense.  Neighbors.to_dense() gives the dense window back,
Neighbors.edge_index(k) the edge list of hop k.
"""
from __future__ import annotations

import math
import time

import numpy as np
import torch

from . import _abi
from .core import Swarm, Neighbors
from . import spawn as _spawn
from .spaces import Box

_LAYOUTS = {'pos_vel': _abi.X_POS_VEL, 'full': _abi.X_FULL}


class AgentBatch:
    """What a reference-style ``state_fn(quad)`` receives: the getters of Object
    (/root/reference/mrsgym/Object.py:78-97) for ALL agents at once, component-major
    ([3, E*N]) so that 1-D code such as ``torch.cat([quad.get_pos(), quad.get_vel()])``
    (README.md:28-29) works unchanged and yields [D, E*N]."""

    def __init__(self, swarm: Swarm):
        self._s = swarm

    def get_pos(self):
        return self._s.state[0:3]

    def get_vel(self):
        return self._s.state[7:10]

    def get_angvel(self):
        return self._s.state[10:13]

    def get_quat(self):
        return self._s.state[3:7]

    def get_ori(self, mat=False):
        """euler 'xyz' [3, E*N], or with mat=True the body->world rotation matrices [3, 3, E*N]
        (Object.get_ori, Object.py:90-97: R.from_quat(q).as_matrix())."""
        if mat:
            return self._s.get_rotmat().reshape(self._s.S, 3, 3).permute(1, 2, 0)
        return self._s.get_ori().reshape(self._s.S, 3).t()


class Environment:
    """Batched stand-in for the reference's Environment on the step path
    (/root/reference/mrsgym/Environment.py:84-124): getters return [E, N, 3] device tensors
    ([N, 3] when N_ENVS == 1, like the reference)."""

    def __init__(self, swarm: Swarm, squeeze: bool):
        self.swarm = swarm
        self._squeeze = squeeze
        self.data = {}
        self.agents = AgentBatch(swarm)
        self.objects = []
        self.controlled = []
        self.object_dict = {}

    def _out(self, x):
        return x[0] if self._squeeze else x

    def get_pos(self):
        return self._out(self.swarm.get_pos())

    def get_vel(self):
        return self._out(self.swarm.get_vel())

    def get_angvel(self):
        return self._out(self.swarm.get_angvel())

    def get_ori(self, mat=False):
        return self._out(self.swarm.get_rotmat() if mat else self.swarm.get_ori())

    def get_quat(self):
        return self._out(self.swarm.get_quat())

    def set_state(self, pos=None, ori=None, vel=None, angvel=None, env_mask=None):
        self.swarm.set_state(pos=pos, ori=ori, vel=vel, angvel=angvel, env_mask=env_mask)

    def set_data(self, name, val):
        self.data[name] = val

    def get_data(self, name):
        return self.data.get(name, None)

    # analytic sensors on the simple world's primitives (Object.py:98-174), all agents at once
    def collision(self, threshold=0.04):
        """Object.collision (Object.py:136-137): any contact closer than 0.04 -> bool [E,N] ([N])."""
        return self._out(self.swarm.proximity(threshold)['collision'])

    def get_dist(self):
        """Gap to the nearest other agent and to the ground, [E,N] each (Object.get_dist, Object.py:118-133)."""
        p = self.swarm.proximity()
        return {k: self._out(v) for k, v in p.items()}

    def raycast(self, directions, offset=(0.0, 0.0, 0.0), body=True, RANGE=100.0):
        r = self.swarm.raycast(directions, offset, body, RANGE)
        return {k: self._out(v) for k, v in r.items()}

    def get_contact_points(self, body=False, threshold=None):
        """Object.get_contact_points (Object.py:100-116) on the contact geometry of the step, all agents at once.
        Per agent up to 1 + 4 candidate contacts are reported as padded arrays with a mask: the nearest other agent
        (contact spheres of CONTACT_RADIUS) and the four lower-rim points of the collision cylinder against the
        ground.  Keys: 'object' int [..., 5] (agent index, N_AGENTS = ground, -1 = no contact), 'pos' [..., 5, 3]
        (world, or body frame with body=True), 'normal' [..., 5, 3] unit normal on the agent, 'distance' [..., 5],
        'mask' bool [..., 5].  A contact exists where the gap is below `threshold` (default: the solver's contact
        margin, like Bullet's manifold).  'normal force' magnitudes are not kept by the step; the solver's
        impulses are internal."""
        return {k: self._out(v) for k, v in self.swarm.contact_points(body=body, threshold=threshold).items()}

    def get_closest_objects(self, radius):
        """Object.get_closest_objects (Object.py:139-141): for every agent the other agents whose contact
        spheres come within `radius` of its own, as a bool mask [..., N, N] plus the gaps [..., N, N]."""
        sw = self.swarm
        p = sw.get_pos()
        gap = torch.cdist(p, p) - 2.0 * float(sw.cfg.phys.contact_radius)
        eye = torch.eye(sw.N, dtype=torch.bool, device=p.device)
        mask = (gap < float(radius)) & ~eye
        return {'mask': self._out(mask), 'gap': self._out(gap)}

    # GUI / debug helpers of the reference (Environment.py:127-306) are no-ops headless
    def draw_links(self, A):
        pass

    def get_keyboard_events(self):
        return {}

    def get_mouse_events(self):
        return {}


class _Sim:
    """BulletSim constants holder (/root/reference/mrsgym/BulletSim.py:8-24)."""

    def __init__(self, **kwargs):
        self.REAL_TIME = False
        self.HEADLESS = True
        self.GRAVITY = 9.81
        self.DT = 0.01
        for name, val in kwargs.items():
            if name in self.__dict__:
                self.__dict__[name] = val

    def stop(self):
        pass


def _zero_reward(**kwargs):
    """Default reward_fn (MRS.py:37): 0."""
    return 0.0


def _no_info(**kwargs):
    """Default info_fn (MRS.py:40): no extra info."""
    return {}


class MRS:
    metadata = {'render.modes': ['headless', 'bullet']}

    def __init__(self, state_fn=None, reward_fn=None, done_fn=None, info_fn=None, update_fn=None, start_fn=None,
                 env='simple', **kwargs):
        # Constants (MRS.py:24-35) + the batching ones
        self.N_AGENTS = 1
        self.K_HOPS = 0
        self.STATE_SIZE = 0
        self.ACTION_DIM = 0
        self.AGENT_RADIUS = 0.3
        self.CONTACT_RADIUS = None   # agent-agent contact sphere; None = AGENT_RADIUS (0.06 = the cf2x collision hull)
        self.SOLVER_ITERS = None     # contact solver sweeps; None = Bullet's 50
        self.COMM_RANGE = float('inf')
        self.RETURN_A = False
        self.RETURN_EVENTS = False
        self.ACTION_TYPE = 'set_target_vel'
        self.HEADLESS = True
        self.MAX_TIMESTEPS = float('inf')
        self.N_ENVS = 1
        self.DEVICE = 'cuda'
        self.TAPE_SLOTS = None
        self.CHECK_NAN = 'auto'
        self.COPY_OBS = None
        self.BATCHED = None          # None: batched shapes iff N_ENVS > 1
        self.SEED = 0                # seed of the on-device start-state sampler
        self.ENV_OFFSET = None       # global index of this process's first env; None: shard_range(rank) under torchrun
        self.A_FORMAT = 'dense'      # 'neighbors': A windows as neighbour lists (Neighbors), no dense A history
        self.MAX_NEIGHBORS = None    # list length M of A_FORMAT='neighbors'; None: min(N_AGENTS - 1, 64)
        self.set_constants(kwargs)
        if env != 'simple':
            raise NotImplementedError("only the 'simple' world (N x cf2x + ground plane, EnvCreator.py:7-13) is in scope")
        self.state_fn = state_fn
        self.reward_fn = reward_fn if (reward_fn is not None) else _zero_reward
        # default done: steps since the last reset >= MAX_TIMESTEPS (MRS.py:39); batched: per env ([E] bool tensor,
        # a masked reset restarts the count of the selected envs only)
        self.done_fn = done_fn if (done_fn is not None) else self._default_done
        self.info_fn = info_fn if (info_fn is not None) else _no_info
        self.update_fn = update_fn
        self.start_fn = start_fn
        self.sim = _Sim(**kwargs)
        self.START_POS = _spawn.DefaultSpawn(self.N_AGENTS)
        self.START_ORI = torch.tensor([0, 0, -np.pi / 2, 0, 0, np.pi / 2]).expand(self.N_AGENTS, -1)
        self.set_constants(kwargs)
        if isinstance(self.START_ORI, torch.Tensor) and self.START_ORI.dim() == 1:
            self.START_ORI = self.START_ORI.expand(self.N_AGENTS, -1)
        self._batched = (self.N_ENVS > 1) if self.BATCHED is None else bool(self.BATCHED)
        self._copy = (not self._batched) if self.COPY_OBS is None else bool(self.COPY_OBS)
        self._views = {}
        self._bases = {}
        # state_fn: None / 'pos_vel' / 'full' -> fused in the step kernel; callable -> python
        if state_fn is None:
            state_fn = 'pos_vel'
        if isinstance(state_fn, str):
            layout, custom_D = _LAYOUTS[state_fn], 0
        else:
            layout = _abi.X_NONE
            custom_D = self.STATE_SIZE
        self._layout = layout
        self.swarm = None
        self._spawn_count = 0
        self.spawn_failed = None
        self._build(layout, custom_D)
        # Gym spaces, literally as the reference builds them (MRS.py:51-52): a flat observation box whose length is
        # the reference's own expression K_HOPS + 1 * N_AGENTS * STATE_SIZE (operator precedence included) and the
        # set_control-style action box [9.81 -+ 1, -+1, -+1, -+1] tiled over the agents
        n_obs = self.K_HOPS + 1 * self.N_AGENTS * self.STATE_SIZE
        self.observation_space = Box(np.full((n_obs,), -np.inf, dtype=np.float32), np.full((n_obs,), np.inf, dtype=np.float32))
        self.action_space = Box(np.tile(np.array([9.81 - 1, -1., -1., -1.], dtype=np.float32), self.N_AGENTS),
                                np.tile(np.array([9.81 + 1, 1., 1., 1.], dtype=np.float32), self.N_AGENTS))
        # per-env steps since that env's last reset = _steps_total - _steps_at_reset[e]: stepping costs a Python
        # increment, not a device launch; the tensor is materialised when somebody reads env_steps
        self._steps_total = 0
        self._steps_at_reset = torch.zeros(self.N_ENVS, dtype=torch.int64, device=self.swarm.device)
        self._uniform_reset = True      # no masked reset since the last full one: env_steps is the same for all envs
        # rollout(graph=True): the graph's device step counter, which env_steps reports while the graph's body runs,
        # the index of every env's current episode (advanced by the on-device auto-reset, the key of its draws) and
        # the captured closed loops of this env
        self._dev_steps = None
        self.episode = torch.zeros(self.N_ENVS, dtype=torch.int32, device=self.swarm.device)
        self._graphs = {}
        self._done_const = {}
        self.steps_since_reset = 0
        self.last_action = None
        self.last_obs = None
        self.last_loop_time = time.monotonic()
        self.is_initialised = False
        self.reset()

    # ------------------------------------------------------------------ construction
    def set_constants(self, kwargs):
        for name, val in kwargs.items():
            if name in self.__dict__:
                self.__dict__[name] = val

    def _build(self, layout, custom_D):
        if layout == _abi.X_NONE and custom_D <= 0:
            # probe the user's state_fn once on a throw-away one-env swarm to learn D
            probe = Swarm(1, self.N_AGENTS, 0, self.ACTION_TYPE, _abi.X_POS_VEL, device=self.DEVICE, want_A=False)
            custom_D = int(self._call_state_fn(probe).shape[-1])
        if self.A_FORMAT not in ('dense', 'neighbors'):
            raise ValueError("A_FORMAT must be 'dense' or 'neighbors', got %r" % (self.A_FORMAT,))
        nbr = None
        if self.A_FORMAT == 'neighbors':
            nbr = min(self.N_AGENTS - 1, 64) if self.MAX_NEIGHBORS is None else int(self.MAX_NEIGHBORS)
        self.swarm = Swarm(self.N_ENVS, self.N_AGENTS, self.K_HOPS, self.ACTION_TYPE, layout, self.COMM_RANGE,
                           dt=self.sim.DT, gravity=self.sim.GRAVITY, agent_radius=self.AGENT_RADIUS,
                           device=self.DEVICE, tape_slots=self.TAPE_SLOTS, want_A=True, custom_D=custom_D,
                           contact_radius=self.CONTACT_RADIUS, fresh_tapes=self._copy, neighbors=nbr)
        self._clone = self._copy and not self.swarm.fresh      # fresh tapes: views stay valid, no copy per step
        self.STATE_SIZE = self.swarm.D
        self.ACTION_DIM = self.swarm.action_dim
        self.env = Environment(self.swarm, squeeze=not self._batched)
        self._built_K = self.K_HOPS
        self._cfg_key = None
        self._last_mode = None

    def _call_state_fn(self, swarm):
        """User state_fn on the whole batch -> [E, N, D] float32."""
        out = self.state_fn(AgentBatch(swarm))
        out = torch.as_tensor(out, dtype=torch.float32, device=swarm.device)
        if out.dim() == 2 and out.shape[1] == swarm.S:        # [D, E*N] (reference-style 1-D code)
            out = out.t()
        return out.reshape(swarm.E, swarm.N, -1)

    def _sync_cfg(self):
        """Attributes are mutable after construction in the reference (e.g. analytics.py:40).  The C struct is
        rewritten only when one of them changed (a tuple compare per step instead of six ctypes stores)."""
        if self.K_HOPS != self._built_K:
            raise RuntimeError('K_HOPS cannot change after construction (tape geometry); build a new MRS')
        key = (self.COMM_RANGE, self.AGENT_RADIUS, self.CONTACT_RADIUS, self.sim.DT, self.sim.GRAVITY, self.SOLVER_ITERS)
        if key == self._cfg_key:
            return
        self._cfg_key = key
        c = self.swarm.cfg
        c.comm_range = float(self.COMM_RANGE)
        c.phys.agent_radius = float(self.AGENT_RADIUS)
        c.phys.contact_radius = float(self.AGENT_RADIUS if self.CONTACT_RADIUS is None else self.CONTACT_RADIUS)
        if self.SOLVER_ITERS is not None:
            c.phys.solver_iters = int(self.SOLVER_ITERS)
        c.dt, c.gravity = float(self.sim.DT), float(self.sim.GRAVITY)

    def _default_done(self, **kwargs):
        """MRS.py:39: steps since the last reset >= MAX_TIMESTEPS; batched: [E] bool.  While every env was last reset
        at the same step (no masked reset since) the answer is one Python compare and a cached constant tensor."""
        if not self._batched:
            return kwargs['steps_since_reset'] >= self.MAX_TIMESTEPS
        if self._uniform_reset:
            flag = kwargs['steps_since_reset'] >= self.MAX_TIMESTEPS
            t = self._done_const.get(flag)
            if t is None:
                t = self._done_const[flag] = torch.full((self.N_ENVS,), flag, dtype=torch.bool, device=self.swarm.device)
            return t
        return self.env_steps >= self.MAX_TIMESTEPS

    @property
    def env_steps(self):
        """[E] int64: steps since each env's last (masked) reset."""
        if self._dev_steps is not None:          # inside the body of rollout(graph=True): the device counter
            return self._dev_steps.long()
        return self._steps_total - self._steps_at_reset

    # ------------------------------------------------------------------ observation windows
    def _shape(self, w):
        # w: [K+1, E, N, *] tape view, newest first
        if self._batched:
            w = w.permute(1, 0, 2, 3)
        else:
            w = w[:, 0]
        return w.clone() if self._clone else w

    def _window(self, which):
        """Newest-first K+1 window of tape `which` in the reference's layout.  The window of a given head slot
        is always the same view of the (static) tape, so views are built once per head position: a training
        loop pays a dict lookup instead of slicing + permuting two tensors per step."""
        sw = self.swarm
        head = sw.hx if which == 1 else sw.ha
        tape = sw.X_tape if which == 1 else sw.A_tape
        if tape is None or (sw.ring and head + sw.K + 1 > sw.L):          # wrapped windows are assembled afresh
            return self._shape(sw.X_window() if which == 1 else sw.A_window())
        if self._copy:
            # one slice of a per-tape base view ([E, L, N, *] or, unbatched, [L, N, *]) instead of slice + index
            b = self._bases.get(which)
            if b is None or b[0] is not tape:
                b = self._bases[which] = (tape, tape.permute(1, 0, 2, 3) if self._batched else tape[:, 0])
            w = b[1][:, head:head + sw.K + 1] if self._batched else b[1][head:head + sw.K + 1]
            return w.clone() if self._clone else w
        key = (which, head, tape.data_ptr())
        v = self._views.get(key)
        if v is None:
            if len(self._views) > 4 * sw.L + 8:
                self._views.clear()
            v = self._views[key] = self._shape(sw.X_window() if which == 1 else sw.A_window())
        return v

    def get_Xk(self):
        return self._window(1)

    def get_Ak(self):
        if self.swarm.nbr is not None:
            return self._nbr_window()
        return self._window(2)

    def _nbr_window(self):
        """Neighbors window in the reference's layout: [E, K+1, N, M] / [E, K+1, N] (unbatched [K+1, N, M] / [K+1, N])."""
        idx, cnt = self.swarm.N_window()
        if self._batched:
            idx, cnt = idx.transpose(0, 1), cnt.transpose(0, 1)
        else:
            idx, cnt = idx[:, 0], cnt[:, 0]
        if self._clone:
            idx, cnt = idx.clone(), cnt.clone()
        return Neighbors(idx, cnt)

    def calc_Xk(self):
        """MRS.calc_Xk (MRS.py:87-95): push X of the current state."""
        hx = self.swarm.push_X()
        if self._layout == _abi.X_NONE:
            self.swarm.X_tape[hx] = self._call_state_fn(self.swarm)
        return self.get_Xk()

    def calc_Ak(self):
        """MRS.calc_Ak (MRS.py:102-110): push A of the current positions."""
        self._sync_cfg()
        self.swarm.push_A()
        return self.get_Ak()

    def refresh_A(self, env_mask=None):
        """After a reset the reference's callers push A0 with calc_Ak() (DataGenerator.py:23).  Batched
        form: env_mask=None pushes for every env; with a mask only the NEWEST slice of the selected
        envs is replaced by the adjacency of their current positions (the others keep their ring)."""
        if env_mask is None:
            return self.calc_Ak()
        self._sync_cfg()
        sw = self.swarm
        m = torch.as_tensor(env_mask).to(sw.device).bool().reshape(sw.E)
        if sw.nbr is not None:
            new = sw.neighbors(sw.nbr)
            sw.N_idx[sw.ha][m] = new.idx[m]
            sw.N_cnt[sw.ha][m] = new.count[m]
            return self.get_Ak()
        A0 = sw.adjacency(sw.get_pos())
        sw.A_tape[sw.ha][m] = A0[m]
        return self.get_Ak()

    def a_ring_empty(self):
        """True right after a full reset / set: no A slice has been pushed yet (MRS.py:186)."""
        return self.swarm.a_empty

    def calc_A(self):
        self._sync_cfg()
        A = self.swarm.adjacency(self.swarm.get_pos())
        return A if self._batched else A[0]

    def get_relative_position(self, pos):
        N = pos.shape[-2]
        return pos.unsqueeze(-2).expand(*pos.shape[:-2], N, N, 3) - pos.unsqueeze(-3).expand(*pos.shape[:-2], N, N, 3)

    # ------------------------------------------------------------------ reset / set
    def generate_start_pos(self):
        """MRS.generate_start_pos (MRS.py:127-154), batched: tensor START_POS is used as is;
        a distribution is sampled per env with the same 2*AGENT_RADIUS rejection rule."""
        if isinstance(self.START_POS, torch.Tensor):
            return self.START_POS
        return _spawn.sample_start_pos(self.START_POS, self.N_ENVS, self.N_AGENTS, self.AGENT_RADIUS)

    def generate_start_ori(self):
        ori = torch.as_tensor(self.START_ORI, dtype=torch.float32)
        if ori.shape[-1] == 3:
            return ori
        lo, hi = ori[..., :3], ori[..., 3:]
        shape = (self.N_ENVS,) + tuple(lo.shape) if lo.dim() == 2 else tuple(lo.shape)
        return lo + (hi - lo) * torch.rand(shape)

    def _after_state_change(self):
        """Tail of MRS.reset / MRS.set (MRS.py:185-192): clear rings, steps := 0, start_fn, X0."""
        self.steps_since_reset = 0
        self._steps_total = 0
        self._steps_at_reset.zero_()
        self._uniform_reset = True
        if self.start_fn is not None:
            self.start_fn(self)
        self.swarm.reset_windows()
        if self._layout == _abi.X_NONE:
            self.swarm.X_tape[self.swarm.hx] = self._call_state_fn(self.swarm)
            self.swarm.fill_X_history()
        Xk = self.get_Xk()
        self.last_obs = Xk
        return Xk

    def _env_offset(self):
        """Global index of this process's first env: ENV_OFFSET, else RANK * N_ENVS under torchrun (every rank of
        the documented one-process-per-GPU layout owns an equal shard), else 0."""
        if self.ENV_OFFSET is not None:
            return int(self.ENV_OFFSET)
        import os
        return int(os.environ.get('RANK', '0')) * self.N_ENVS if int(os.environ.get('WORLD_SIZE', '1')) > 1 else 0

    def _device_spawn_ok(self):
        """The default START_POS / START_ORI (MRS.py:53-54) can be sampled on the device."""
        if not isinstance(self.START_POS, _spawn.DefaultSpawn):
            return False
        ori = torch.as_tensor(self.START_ORI, dtype=torch.float32)
        if ori.dim() != 2 or ori.shape[-1] != 6:
            return False
        same = bool((ori == ori[0]).all())
        return same and bool((ori[0, [0, 1, 3, 4]] == 0).all())

    def _after_masked_state_change(self, env_mask):
        """Per-env reset in a batch: only the selected envs get their rings re-initialised (X history
        := copies of X0, A history := zeros); the other envs keep theirs.  The reference has one env
        per process, so this is the batched reading of MRS.reset's tail (MRS.py:185-192)."""
        sw = self.swarm
        sw.renew_tapes()
        m = torch.as_tensor(env_mask).to(sw.device).bool().reshape(sw.E)
        self._steps_at_reset[m] = self._steps_total
        self._uniform_reset = False
        if self.start_fn is not None:
            self.start_fn(self)
        if sw.X_tape is not None:
            if self._layout == _abi.X_NONE:
                X0 = self._call_state_fn(sw)
            elif self._layout == _abi.X_POS_VEL:
                X0 = torch.cat([sw.get_pos(), sw.get_vel()], dim=-1)
            else:
                X0 = torch.cat([sw.get_pos(), sw.get_quat(), sw.get_vel(), sw.get_angvel()], dim=-1)
            for sl in sw.window_slots(1):
                sw.X_tape[sl][m] = X0[m].to(sw.X_tape.dtype)
        if sw.A_tape is not None:
            for sl in sw.window_slots(2):
                sw.A_tape[sl][m] = 0
        if sw.N_idx is not None:
            for sl in sw.window_slots(2):
                sw.N_idx[sl][m] = -1
                sw.N_cnt[sl][m] = 0
        Xk = self.get_Xk()
        self.last_obs = Xk
        return Xk

    def reset(self, pos=None, ori=None, vel=None, angvel=None, env_mask=None):
        """MRS.reset (MRS.py:174-192).  PID integrators are NOT reset (reference behaviour).
        env_mask ([E] bool) resets only the selected envs of the batch and keeps the rings of the rest.
        With the default START_POS / START_ORI the start state is sampled on the device (mrs_spawn)."""
        self.is_initialised = True
        if pos is None and ori is None and self._device_spawn_ok():
            ori6 = torch.as_tensor(self.START_ORI, dtype=torch.float32)[0]
            sp = self.START_POS
            self._spawn_count += 1
            # N > 32 keeps the host sampler's failure contract (10000 rounds, then RuntimeError): one synchronising
            # read of the counter per reset.  N <= 32 keeps its lazy counter and 256 rounds.
            wide = self.N_AGENTS > 32
            self.spawn_failed = self.swarm.spawn(self.SEED * 1000003 + self._spawn_count, env_mask=env_mask,
                                                 z=(sp.z_low, sp.z_high), xy_radius=sp.xy_radius, xy_sigma=sp.xy_radius,
                                                 yaw=(float(ori6[2]), float(ori6[5])), env_offset=self._env_offset(),
                                                 max_rounds=10000 if wide else 256)
            if wide and int(self.spawn_failed.item()):
                raise RuntimeError('start-position rejection sampling did not converge (N_AGENTS too dense for START_POS)')
            if vel is not None or angvel is not None:
                self.swarm.set_state(vel=vel, angvel=angvel, env_mask=env_mask)
        else:
            if pos is None:
                pos = self.generate_start_pos()
            if ori is None:
                ori = self.generate_start_ori()
            if vel is None:
                vel = torch.zeros(self.N_AGENTS, 3)
            if angvel is None:
                angvel = torch.zeros(self.N_AGENTS, 3)
            self.swarm.set_state(pos=pos, ori=ori, vel=vel, angvel=angvel, env_mask=env_mask)
        if env_mask is not None:
            return self._after_masked_state_change(env_mask)
        return self._after_state_change()

    def set(self, pos=None, ori=None, vel=None, angvel=None, env_mask=None):
        """MRS.set (MRS.py:196-205): like reset, but None keeps the current value."""
        self.swarm.set_state(pos=pos, ori=ori, vel=vel, angvel=angvel, env_mask=env_mask)
        if env_mask is not None:
            return self._after_masked_state_change(env_mask)
        return self._after_state_change()

    # ------------------------------------------------------------------ step
    def _prep_actions(self, actions):
        adim = self.swarm.action_dim
        sw = self.swarm
        # fast path of a training loop: a float32 device tensor of the right size needs no conversion at all
        if (isinstance(actions, torch.Tensor) and actions.is_cuda and actions.dtype == torch.float32
                and actions.is_contiguous() and actions.numel() == sw.S * adim and actions.device == sw.device
                and not actions.requires_grad and self.CHECK_NAN is not True and actions.data_ptr() % 16 == 0):
            if actions.dim() == (3 if self._batched else 2):      # already in the shape the callbacks see: no view at all
                self.last_action = actions
                return actions
            return actions.view(self.N_ENVS, self.N_AGENTS, adim)
        host = not (isinstance(actions, torch.Tensor) and actions.is_cuda)
        actions = torch.as_tensor(actions).detach()
        if actions.dtype != torch.float32:
            actions = actions.to(torch.float32)
        check = self.CHECK_NAN
        if (check == 'auto' and host) or check is True:
            if bool(torch.isnan(actions).any()):
                raise Exception('The given action contains NaN:\n %s' % str(actions))      # MRS.py:247-248
        actions = actions.to(self.swarm.device).reshape(self.N_ENVS, self.N_AGENTS, adim).contiguous()
        if actions.data_ptr() % 16:          # a view into the middle of a buffer: the kernels need 16-byte alignment
            actions = actions.clone()
        return actions

    def step(self, actions, ACTION_TYPE=None):
        """MRS.step (MRS.py:240-277)."""
        self._sync_cfg()
        if actions is not None:
            if ACTION_TYPE is None:
                ACTION_TYPE = self.ACTION_TYPE
            if ACTION_TYPE != self._last_mode:
                self.ACTION_DIM = self.swarm.set_action_type(ACTION_TYPE)
                self._last_mode = ACTION_TYPE
            self.last_action = None
            actions = self._prep_actions(actions)
            if self.last_action is None:
                self.last_action = actions if self._batched else actions[0]
        else:
            self.swarm.set_action_type(None)
            self._last_mode = None
        self.swarm.step(actions)
        if self._layout == _abi.X_NONE:
            self.swarm.X_tape[self.swarm.hx] = self._call_state_fn(self.swarm)
        Xk = self.get_Xk()
        Ak = self.get_Ak()
        kw = dict(env=self.env, A=Ak, action=self.last_action, steps_since_reset=self.steps_since_reset)
        if self.update_fn is not None:
            self.update_fn(X=Xk, Xlast=self.last_obs, **kw)
        reward = self.reward_fn(X=Xk, Xlast=self.last_obs, **kw)
        self.last_obs = Xk
        info = self.info_fn(X=Xk, Xlast=self.last_obs, **kw)
        info['A'] = Ak
        if self.RETURN_EVENTS:
            info['keyboard_events'] = self.env.get_keyboard_events()
            info['mouse_events'] = self.env.get_mouse_events()
        done = self.done_fn(X=Xk, Xlast=self.last_obs, **kw)
        self.last_loop_time = time.monotonic()
        self.steps_since_reset += 1
        self._steps_total += 1
        return Xk, reward, done, info

    def step_many(self, actions, ACTION_TYPE=None):
        """T steps with pre-computed actions [T, E, N, A] in one launch (state stays on chip);
        the rollout loop of examples/simulating_data/helper/DataGenerator.py:8-48 without the
        per-step host round trip.  Returns the final (X, A) windows; callbacks are not called."""
        self._sync_cfg()
        if self._layout == _abi.X_NONE:
            raise RuntimeError('step_many needs a fused state layout (state_fn "pos_vel" or "full")')
        if ACTION_TYPE is None:
            ACTION_TYPE = self.ACTION_TYPE
        adim = self.swarm.set_action_type(ACTION_TYPE)
        self._last_mode = ACTION_TYPE
        actions = torch.as_tensor(actions, dtype=torch.float32).to(self.swarm.device)
        T = actions.shape[0]
        actions = actions.reshape(T, self.N_ENVS, self.N_AGENTS, adim).contiguous()
        self.swarm.step_many(actions, T)
        self.steps_since_reset += T
        self._steps_total += T
        Xk = self.get_Xk()
        self.last_obs = Xk
        return Xk, self.get_Ak()

    def check_status(self):
        """Lazy NaN / non-finite guard for device-resident actions (synchronises)."""
        v = self.swarm.read_status()
        if v & _abi.STATUS_NAN_ACTION:
            raise Exception('The given action contains NaN')
        if v & _abi.STATUS_NONFINITE:
            raise FloatingPointError('simulation state left the finite range')
        if v & _abi.STATUS_NEIGHBOR_OVERFLOW:
            raise OverflowError('an agent had more neighbours within COMM_RANGE than MAX_NEIGHBORS = %d: its list was '
                                'truncated (count holds the true degree); raise MAX_NEIGHBORS' % self.swarm.nbr)

    # ------------------------------------------------------------------ misc API parity
    def set_data(self, name, val):
        self.env.set_data(name, val)

    def get_data(self, name):
        return self.env.get_data(name)

    def close(self):
        pass

    def render(self, mode='bullet', close=False):
        if close:
            self.close()

    def wait(self, dt=None):
        if dt is None:
            dt = self.sim.DT
        diff = time.monotonic() - self.last_loop_time
        time.sleep(max(dt - diff, 0))

    def get_env(self):
        return self.env

    def get_objects(self):
        return self.env.objects

    def get_agents(self):
        return self.env.agents

    def get_controlled(self):
        return self.env.controlled

    def get_object_dict(self):
        return self.env.object_dict
