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

import torch

from .core import Neighbors


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


def rollout(env, policy, T, episode_length=None, record=('X', 'A', 'action', 'reward', 'done'), out=None):
    """Closed-loop rollout of `T` steps for all envs of `env` (an mrsgym_b200.MRS).

    policy(X, A) -> actions, all on the device (A: a Neighbors window when env.A_FORMAT == 'neighbors'; the dataset
    then records A_idx / A_cnt instead of A).  An env is reset (masked, on-device spawn when the
    default start distribution is in use) when its `done` entry is True or after `episode_length`
    steps.  Returns the dataset dict described in the module docstring; pass `out` to append into
    preallocated buffers of a previous call."""
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
