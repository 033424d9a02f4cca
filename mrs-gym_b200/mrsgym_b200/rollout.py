"""On-device rollout driver and dataset format (SURVEY.md §8f rank 2).

The reference's only rollout loop is examples/simulating_data/helper/DataGenerator.py:8-48
(`generate_mrs`): reset -> calc_Ak -> model.forward(A, X) -> trainer.set_state(...) -> env.step(action)
until enough datapoints, resetting every `episode_length` steps or on `done`.  Here the same loop runs
for all envs of the batch with the policy, the environment and the dataset on the GPU: no host round
trip per step, per-env auto-reset through MRS.reset(env_mask=...).

Dataset = dict of device tensors (torch.save-able, the counterpart of Trainer.history /
Trainer.save_trainer, helper/Trainer.py:43-108):
  X [T, E, N, D]   newest observation slice before the action of step t
  A [T, E, N, N]   newest adjacency slice before the action of step t; with A_FORMAT='neighbors' instead
                   A_idx [T, E, N, M] and A_cnt [T, E, N], the same slice as neighbour lists (Neighbors)
  action [T, E, N, ACTION_DIM], reward [T, E] (or [T]), done [T, E] bool (episode ended AFTER step t)
"""
from __future__ import annotations

import gc
import math

import torch

from . import _abi
from .core import Neighbors
from .env import _no_info


def reynolds_policy(cohesion=0.5, separation=0.6, alignment=0.5, sep_dist=0.9, v_max=1.0):
    """Classic Reynolds flocking (cohesion / separation / alignment over the COMM_RANGE neighbours)
    as a batched policy for ACTION_TYPE='set_target_vel' with state_fn = cat(pos, vel).
    X: [E, K+1, N, 6] or [K+1, N, 6]; A: [E, K+1, N, N] or [K+1, N, N], or a Neighbors window (A_FORMAT='neighbors',
    aggregated with gathers over the lists, no N x N intermediate)  ->  target velocities [E, N, 3]."""

    def limit(vel, centre, push, align):
        v = vel + cohesion * centre + separation * push + alignment * align
        speed = v.norm(dim=-1, keepdim=True).clamp_min(1e-6)
        return v * (speed.clamp_max(v_max) / speed)

    def policy_lists(X, A):
        if X.dim() == 3:
            X, A = X.unsqueeze(0), Neighbors(A.idx.unsqueeze(0), A.count.unsqueeze(0))
        x, idx = X[:, 0], A.idx[:, 0].long()          # newest slice; idx [E, N, M]
        pos, vel = x[..., :3], x[..., 3:6]
        E, N, M = idx.shape
        ok = idx >= 0
        a = ok.to(pos.dtype).unsqueeze(-1)             # [E, N, M, 1]
        flat = idx.clamp_min(0).reshape(E, N * M, 1).expand(-1, -1, 3)
        rel = torch.gather(pos, 1, flat).reshape(E, N, M, 3) - pos.unsqueeze(2)      # p_j - p_i
        dvel = torch.gather(vel, 1, flat).reshape(E, N, M, 3) - vel.unsqueeze(2)
        deg = a.sum(dim=2).clamp_min(1.0)
        centre = (a * rel).sum(dim=2) / deg
        dist = rel.norm(dim=-1, keepdim=True).clamp_min(1e-6)
        push = (a * (dist < sep_dist) * (sep_dist - dist) / dist * (-rel)).sum(dim=2)
        align = (a * dvel).sum(dim=2) / deg
        return limit(vel, centre, push, align)

    def policy(X, A):
        if isinstance(A, Neighbors):
            return policy_lists(X, A)
        if X.dim() == 3:
            X, A = X.unsqueeze(0), A.unsqueeze(0)
        x, a = X[:, 0], A[:, 0]                       # newest slice
        pos, vel = x[..., :3], x[..., 3:6]
        deg = a.sum(dim=-1, keepdim=True).clamp_min(1.0)
        rel = pos.unsqueeze(1) - pos.unsqueeze(2)     # rel[e, i, j] = p_j - p_i
        centre = (a.unsqueeze(-1) * rel).sum(dim=2) / deg
        dist = rel.norm(dim=-1).clamp_min(1e-6)
        push = (a * (dist < sep_dist) * (sep_dist - dist) / dist).unsqueeze(-1) * (-rel)
        align = (a.unsqueeze(-1) * (vel.unsqueeze(1) - vel.unsqueeze(2))).sum(dim=2) / deg
        return limit(vel, centre, push.sum(dim=2), align)

    return policy


def rollout(env, policy, T, episode_length=None, record=('X', 'A', 'action', 'reward', 'done'), out=None, graph=False):
    """Closed-loop rollout of `T` steps for all envs of `env` (an mrsgym_b200.MRS).

    policy(X, A) -> actions, all on the device (A: a Neighbors window when env.A_FORMAT == 'neighbors'; the dataset
    then records A_idx / A_cnt instead of A).  An env is reset (masked, on-device spawn when the
    default start distribution is in use) when its `done` entry is True or after `episode_length`
    steps.  Returns the dataset dict described in the module docstring; pass `out` to append into
    preallocated buffers of a previous call.

    graph=True: the T steps run as ONE CUDA graph with the episode bookkeeping and the masked reset on the device
    (mrs_autoreset): no host decision and no synchronisation per step.  The first call for a (policy, T,
    episode_length, record) captures the graph (the capture leaves the env where it was) and caches it on the env;
    later calls replay it.  The done rule and the windows after a reset are those of graph=False; the start states
    of reset envs are drawn on the device keyed by (SEED, global env index, env.episode), so they differ from
    graph=False's draws but not between runs.  The returned tensors are the graph's own buffers: the next replay
    overwrites them (copy what you keep, or pass `out`).  reward_fn / done_fn run inside the graph: they must return
    device tensors or constants and must not synchronise (capture fails loudly if they do); they see the per-env
    count as env.env_steps (the host-side steps_since_reset argument is frozen at capture).  After a replay an env
    of more than 32 agents raises RuntimeError when a reset's rejection sampling did not converge; smaller envs count
    such resets in env.spawn_failed (read it lazily).  Needs the default START_POS / START_ORI, a fused state_fn,
    A_FORMAT='dense', no update_fn / info_fn, no fresh tapes (COPY_OBS=False when N_ENVS = 1) and T a multiple of the
    tape size (TAPE_SLOTS=T): the graph runs the tapes as rings, like Swarm.capture_rollout."""
    if graph:
        data = closed_loop_graph(env, policy, T, episode_length, record).run()
        if out is None:
            return data
        for k, v in data.items():
            if k in out:
                out[k].copy_(v)
            else:
                out[k] = v.clone()
        return out
    sw = env.swarm
    E, N = sw.E, sw.N
    dev = sw.device
    X = env.get_Xk()
    if env.a_ring_empty():            # right after reset: push A0 like DataGenerator.py:23
        env.calc_Ak()
    A = env.get_Ak()
    data = out if out is not None else {}
    batched = env._batched

    def as_batch(t):
        return t if batched else t.unsqueeze(0)

    for t in range(T):
        actions = policy(X, A)
        adim = actions.shape[-1]
        if 'X' in record:
            data.setdefault('X', torch.empty(T, E, N, sw.D, device=dev))[t] = as_batch(X)[:, 0]
        if 'A' in record and isinstance(A, Neighbors):
            idx, cnt = (A.idx, A.count) if batched else (A.idx.unsqueeze(0), A.count.unsqueeze(0))
            data.setdefault('A_idx', torch.empty(T, E, N, idx.shape[-1], dtype=torch.int32, device=dev))[t] = idx[:, 0]
            data.setdefault('A_cnt', torch.empty(T, E, N, dtype=torch.int32, device=dev))[t] = cnt[:, 0]
        elif 'A' in record:
            data.setdefault('A', torch.empty(T, E, N, N, device=dev))[t] = as_batch(A)[:, 0]
        if 'action' in record:
            data.setdefault('action', torch.empty(T, E, N, adim, device=dev))[t] = actions.reshape(E, N, adim)
        X, reward, done, info = env.step(actions if batched else actions.reshape(N, adim))
        A = info['A']
        done_t = torch.as_tensor(done, device=dev)
        done_e = done_t.reshape(-1)[:E].bool() if done_t.numel() >= E else done_t.reshape(1).bool().expand(E)
        if episode_length is not None:
            done_e = done_e | (env.env_steps >= episode_length)
        if 'reward' in record:
            r = torch.as_tensor(reward, dtype=torch.float32, device=dev)
            data.setdefault('reward', torch.empty(T, E, device=dev))[t] = r if r.numel() == E else r.reshape(-1)[:1].expand(E)
        if 'done' in record:
            data.setdefault('done', torch.empty(T, E, dtype=torch.bool, device=dev))[t] = done_e
        if bool(done_e.any()):
            X = env.reset(env_mask=done_e)
            A = env.refresh_A(done_e)
    return data


def closed_loop_graph(env, policy, T, episode_length=None, record=('X', 'A', 'action', 'reward', 'done')):
    """The ClosedLoopGraph of rollout(graph=True), from the env's cache or captured now."""
    env._sync_cfg()
    if env.a_ring_empty():            # right after reset: push A0 like DataGenerator.py:23 (eager, before the graph)
        env.calc_Ak()
    sw = env.swarm
    sp = env.START_POS
    spawn = (env.SEED, env._env_offset(), getattr(sp, 'z_low', None), getattr(sp, 'z_high', None),
             getattr(sp, 'xy_radius', None))
    # the captured step kernels read the external wrench iff it was bound at capture
    key = (policy, int(T), episode_length, tuple(record), sw.hx, sw.ha, env._cfg_key, env.ACTION_TYPE, spawn, sw.bufs.wrench)
    g = env._graphs.get(key)
    if g is None:
        g = env._graphs[key] = ClosedLoopGraph(env, policy, T, episode_length, record)
    return g


class ClosedLoopGraph:
    """T closed-loop steps (policy -> mrs_step -> reward_fn / done_fn -> mrs_autoreset) with on-device episode
    bookkeeping, captured in one torch.cuda.CUDAGraph (capture=False: the same body run eagerly on every run(), the
    reference the graph is tested against).  See rollout(graph=True)."""

    def __init__(self, env, policy, T, episode_length=None, record=('X', 'A', 'action', 'reward', 'done'), capture=True):
        sw = env.swarm
        self._refuse(env, T)
        env._sync_cfg()
        if env.a_ring_empty():        # right after reset: push A0 like DataGenerator.py:23
            env.calc_Ak()
        self.env, self.policy, self.T, self.record = env, policy, int(T), tuple(record)
        if env.ACTION_TYPE != env._last_mode:
            env.ACTION_DIM = sw.set_action_type(env.ACTION_TYPE)
            env._last_mode = env.ACTION_TYPE
        E, N, dev = sw.E, sw.N, sw.device
        self.adim = sw.action_dim
        # the done rule: episode_length counts after the step's increment (0 = none; <= 0 ends every step as
        # env_steps >= episode_length does), the default done_fn's MAX_TIMESTEPS before it (-1 = never)
        self.episode_length = 0 if episode_length is None else max(int(math.ceil(episode_length)), 1)
        self.default_done = env.done_fn == env._default_done
        mt = env.MAX_TIMESTEPS
        self.max_timesteps = -1 if (not self.default_done or mt == float('inf')) else max(int(math.ceil(mt)), 0)
        sp = env.START_POS
        ori6 = torch.as_tensor(env.START_ORI, dtype=torch.float32)[0]
        self.spawn = dict(seed=int(env.SEED), env_offset=env._env_offset(), z=(sp.z_low, sp.z_high),
                          xy_radius=sp.xy_radius, xy_sigma=sp.xy_radius, yaw=(float(ori6[2]), float(ori6[5])),
                          max_rounds=10000 if N > 32 else 256)
        z = dict(device=dev)
        self.data = {}
        if 'X' in record:
            self.data['X'] = torch.empty(T, E, N, sw.D, **z)
        if 'A' in record:
            self.data['A'] = torch.empty(T, E, N, N, **z)
        if 'action' in record:
            self.data['action'] = torch.empty(T, E, N, self.adim, **z)
        if 'reward' in record:
            self.data['reward'] = torch.empty(T, E, **z)
        self.done = torch.zeros(T, E, dtype=torch.bool, **z)          # mrs_autoreset's done_out of every step
        if 'done' in record:
            self.data['done'] = self.done
        self.done_in = torch.zeros(E, dtype=torch.bool, **z)
        self.steps = torch.zeros(E, dtype=torch.int32, **z)           # env_steps on the device during a run
        self.failed = torch.zeros(1, dtype=torch.int32, **z)
        self.last_action = None
        sw.ring = True                 # heads wrap around: T is a multiple of L, so every run ends where it started
        self.graph = None
        self.launches_per_run = 0
        if capture:
            self._capture()

    @staticmethod
    def _refuse(env, T):
        sw = env.swarm
        if sw.nbr is not None:
            raise ValueError("rollout(graph=True) needs A_FORMAT='dense' (neighbour lists are not in graph mode yet); "
                             "use graph=False")
        if env._layout == _abi.X_NONE:
            raise ValueError("rollout(graph=True) needs a fused state_fn ('pos_vel' or 'full'); a callable state_fn "
                             "runs with graph=False")
        if sw.fresh:
            raise ValueError('rollout(graph=True) cannot run on fresh tapes (N_ENVS = 1 with the default COPY_OBS): '
                             'build the env with COPY_OBS=False')
        if T < 1 or T % sw.L:
            raise ValueError('rollout(graph=True): T=%d must be a multiple of the tape size (%d slots); build the env '
                             'with TAPE_SLOTS=T' % (T, sw.L))
        if not env._device_spawn_ok():
            raise ValueError('rollout(graph=True) resets with the default START_POS / START_ORI only; use graph=False '
                             'for a custom start distribution')
        if env.update_fn is not None or env.info_fn is not _no_info:
            raise ValueError('rollout(graph=True) does not call update_fn / info_fn; build the env without them or use '
                             'graph=False')
        if env.done_fn == env._default_done and not env._batched and env.MAX_TIMESTEPS != float('inf'):
            raise ValueError('rollout(graph=True) counts MAX_TIMESTEPS per env: build the env with BATCHED=True')

    def _body(self):
        env, sw, T = self.env, self.env.swarm, self.T
        E, N, adim, batched = sw.E, sw.N, self.adim, env._batched
        d = self.data
        env._dev_steps = self.steps
        try:
            X, A = env.get_Xk(), env.get_Ak()
            env.last_obs = X
            for t in range(T):
                actions = self.policy(X, A)
                if 'X' in d:
                    d['X'][t] = X[:, 0] if batched else X[0].unsqueeze(0)
                if 'A' in d:
                    d['A'][t] = A[:, 0] if batched else A[0].unsqueeze(0)
                if 'action' in d:
                    d['action'][t] = actions.reshape(E, N, adim)
                env.last_action = None
                acts = env._prep_actions(actions if batched else actions.reshape(N, adim))
                if env.last_action is None:
                    env.last_action = acts if batched else acts[0]
                sw.step(acts)
                Xk, Ak = env.get_Xk(), env.get_Ak()
                kw = dict(env=env.env, A=Ak, action=env.last_action, steps_since_reset=env.steps_since_reset)
                reward = env.reward_fn(X=Xk, Xlast=env.last_obs, **kw)
                env.last_obs = Xk
                done_in = None
                if not self.default_done:
                    done_in = self._as_done(env.done_fn(X=Xk, Xlast=env.last_obs, **kw), E)
                sw.autoreset(done_out=self.done[t], done_in=done_in, env_steps=self.steps, episode=env.episode,
                             episode_length=self.episode_length, max_timesteps=self.max_timesteps, failed=self.failed,
                             **self.spawn)
                if 'reward' in d:
                    self._put_reward(d['reward'][t], reward, E)
                X, A = env.get_Xk(), env.get_Ak()
                env.last_obs = X
            self.last_action = env.last_action
        finally:
            env._dev_steps = None

    def _as_done(self, done, E):
        """done_fn's result as the kernel's done_in [E] (rollout()'s reading: [E] per env, or one value for all)."""
        if isinstance(done, torch.Tensor):
            done = done.reshape(-1)
            self.done_in.copy_(done[:E] if done.numel() >= E else done[:1].expand(E))
        else:
            self.done_in.fill_(bool(done))
        return self.done_in

    @staticmethod
    def _put_reward(dst, reward, E):
        if isinstance(reward, torch.Tensor):
            r = reward.reshape(-1)
            dst.copy_(r if r.numel() == E else r[:1].expand(E))
        else:
            dst.fill_(float(reward))

    def _capture(self):
        """Warm up outside capture (lazy module loads, the policy's first calls), put back everything the warm-up
        touched, then capture; as GraphRollout."""
        env, sw = self.env, self.env.swarm
        torch.cuda.synchronize(sw.device)
        self.graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(device=sw.device)
        side.wait_stream(torch.cuda.current_stream(sw.device))
        with torch.cuda.stream(side):
            keep = [(t, t.clone()) for t in (sw.state, sw.ctrl, sw.status, sw.stats, sw.rpm, sw.wrench, env.episode,
                                             self.steps, self.failed) if t is not None]
            bound = sw.bufs.wrench
            for tape, which in ((sw.X_tape, 1), (sw.A_tape, 2)):
                if tape is not None:
                    keep += [(tape[sl], tape[sl].clone()) for sl in sw.window_slots(which)]
            host = (sw.hx, sw.ha, sw.a_empty, sw.launches, env.last_obs, env.last_action)
            self._prologue()
            self._body()
            for dst, src in keep:
                dst.copy_(src)
            sw.hx, sw.ha, sw.a_empty, sw.launches, env.last_obs, env.last_action = host
            if sw.bufs.wrench != bound:
                raise RuntimeError('the policy bound or cleared the external wrench: bind it (set_external_wrench) '
                                   'before rollout(graph=True); inside the loop only write it')
            torch.cuda.synchronize(sw.device)
            # an MRS is a reference cycle (its default done_fn is one of its bound methods), so a dropped env and the
            # CUDA graphs it cached are freed by the cyclic collector; freeing a graph or its memory pool while this
            # capture runs would invalidate the capture: collect the dead cycles now and let no collection run inside
            gc.collect()
            gc_was_enabled = gc.isenabled()
            gc.disable()
            try:
                with torch.cuda.graph(self.graph, stream=side):
                    before = sw.launches
                    self._body()        # the heads come back to where they were: T is a multiple of L
                    self.launches_per_run = sw.launches - before
            except RuntimeError as ex:
                raise RuntimeError('rollout(graph=True): capturing the closed loop failed: %s.  The policy, reward_fn '
                                   'and done_fn run inside the CUDA graph: they must return device tensors or '
                                   'constants and must not synchronise with the host (no .item(), bool(tensor), '
                                   '.cpu() or host tensors)' % ex) from ex
            finally:
                if gc_was_enabled:
                    gc.enable()
                sw.hx, sw.ha, sw.a_empty, sw.launches, env.last_obs, env.last_action = host
        torch.cuda.current_stream(sw.device).wait_stream(side)
        torch.cuda.synchronize(sw.device)

    def _prologue(self):
        env = self.env
        self.steps.copy_(env.env_steps)
        self.failed.zero_()

    def run(self):
        """T closed-loop steps from where the env is: the graph's replay (or the eager body).  Returns the dataset
        dict (the graph's own buffers)."""
        env, sw = self.env, self.env.swarm
        if env.a_ring_empty():        # (closed_loop_graph has done this before it looked the graph up)
            env.calc_Ak()
        self._prologue()
        if self.graph is not None:
            self.graph.replay()
            sw.launches += self.launches_per_run
        else:
            self._body()
        env._steps_total += self.T
        env.steps_since_reset += self.T
        env._steps_at_reset = env._steps_total - self.steps.long()
        env._uniform_reset = False
        sw.a_empty = False
        env.last_obs = env.get_Xk()
        env.last_action = self.last_action
        if sw.N > 32:
            # the eager path's failure contract (10000 rounds, then RuntimeError): one read per run
            if int(self.failed.item()):
                raise RuntimeError('start-position rejection sampling did not converge (N_AGENTS too dense for START_POS)')
        else:
            env.spawn_failed = self.failed
        return self.data


def to_trainer_history(data, envs=None):
    """The batched dataset of rollout() in the layout of the reference's replay store, `Trainer.history`
    (examples/simulating_data/helper/Trainer.py:89-108: parallel lists `X` (N, D), `A` (N, N), `expert` (N, ACTION_DIM),
    `done`, `context`, one entry per time step, episodes back to back).  The envs of the batch are laid end to end;
    the last recorded step of every env is marked `done` (as Trainer.save_trainer does for the last entry, :44-45), so
    that a K-step window (`Trainer.get_state`, :112-125) never straddles two envs.  The result can be handed to
    `Trainer.load_trainer_dict({'history': ...})` or saved with torch.save; tensors are moved to the CPU like the
    reference's `.cpu()` calls in DataGenerator.py:41.  A dataset recorded in neighbour mode (A_idx / A_cnt) is
    expanded to the reference's dense (N, N) entries."""
    X = data['X']
    A = data['A'] if 'A' in data else Neighbors(data['A_idx'].cpu(), data['A_cnt'].cpu()).to_dense()
    T, E = X.shape[0], X.shape[1]
    envs = range(E) if envs is None else envs
    done = data['done'] if 'done' in data else torch.zeros(T, E, dtype=torch.bool)
    act = data.get('action')
    Xc, Ac, dc = X.cpu(), A.cpu(), done.cpu()
    ac = act.cpu() if act is not None else None
    hist = {'done': [], 'A': [], 'X': [], 'context': [], 'expert': []}
    for e in envs:
        for t in range(T):
            hist['X'].append(Xc[t, e])
            hist['A'].append(Ac[t, e])
            hist['expert'].append(ac[t, e] if ac is not None else None)
            hist['context'].append({})
            hist['done'].append(bool(dc[t, e]) or t == T - 1)
    return hist


def save_dataset(data, path):
    """torch.save of the dataset dict (device tensors are written as they are; load with map_location as needed)."""
    with open(path, 'wb') as fp:
        torch.save(data, fp)
