"""The step's event outputs -- the sticky status word and every stats counter -- and the NaN-action rule against the
CPU oracle, on every kernel the step can pick (tests/step_events.py builds the scenes and the expected counts):
N <= 32 run-time width, unrolled 8 / 16 / 32 and SM-sized CTAs; 33-128 lanes per agent, fused and three-kernel one
CTA per env; N > 128 tiled; and the multi-step forms (mrs_step_many, chained mrs_rollout, graph replay).  Every
counter is compared as an exact integer."""
import numpy as np
import pytest
import torch

import helpers as H
import physics_variants as V
import step_events as SE

pytestmark = pytest.mark.gpu

STAT_KEYS = ('agent_contact_rows', 'ground_contacts', 'nonfinite', 'nan_actions', 'contact_chunks', 'solver_sweeps')
T = 3


def _big_cta_envs():
    from test_gpu_physics_variants import _big_cta_envs as big
    return -(-big() // SE.E0) * SE.E0


# path -> (E, N, MRS_B200_FUSED_MID)
PATHS = {
    'runtime5': (12, 5, None), 'runtime12': (12, 12, None),
    'unrolled8': (12, 8, None), 'unrolled16': (12, 16, None), 'unrolled32': (12, 32, None),
    'sm_cta': ('big', 8, None),
    'lanes48': (12, 48, None), 'fused64': (520, 64, '1'), 'three64': (520, 64, '0'),
    'thread64': (512, 64, '0'), 'thread33': (1000, 33, '0'),
    'tiled200': (2, 200, None), 'tiled1030': (1, 1030, None),
}
NAN_PATHS = ('runtime5', 'unrolled8', 'unrolled16', 'sm_cta', 'lanes48', 'fused64', 'thread64', 'tiled200')


@pytest.fixture(scope='module')
def thr():
    return SE.thresholds()


def _shape(path, monkeypatch):
    E, N, fused = PATHS[path]
    if fused is not None:
        monkeypatch.setenv('MRS_B200_FUSED_MID', fused)
    return (_big_cta_envs() if E == 'big' else E), N


def _swarm(E, N, mode, kind, **kw):
    import mrsgym_b200 as M
    sw = M.Swarm(E, N, 0, mode, M._abi.X_POS_VEL, float('inf'), keep_rpm=True, **kw)
    V.apply(sw, SE.SCENE_PHYS.get(kind, {}))
    return sw


def _dev(a):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _stats(sw):
    s = sw.read_stats()
    return {k: s[k] for k in STAT_KEYS}


def _expect(kind, E, N, mode, acts, thr, form='single', **kw):
    """expected stats, from the oracle on one scene block times the number of whole blocks (envs are independent and
    a block holds whole warp-chunks), plus the oracle on the envs of the last, cut block"""
    out = None
    for Eo, times in ((min(E, SE.E0), E // SE.E0 or 1), (E % SE.E0 if E > SE.E0 else 0, 1)):
        if not Eo:
            continue
        a = None if acts is None else acts[:, :Eo]
        _, steps = SE.oracle_run(SE.make_scene(kind, N, Eo), mode, a, acts.shape[0] if acts is not None else T,
                                 **SE.SCENE_PHYS.get(kind, {}))
        ex = SE.expected_stats(steps, N, *thr, form=form, **kw)
        out = {k: v * times + (out[k] if out else 0) for k, v in ex.items()}
    return out


def _actions(kind, mode, Tn, E, N, st, nan_steps=(0,)):
    if kind != 'nan_chunk':
        return None
    acts = H.random_actions(np.random.default_rng(N), mode, Tn, SE.E0, N, SE.make_scene(kind, N)['pos'])
    acts = np.ascontiguousarray(np.tile(acts, (1, -(-E // SE.E0), 1, 1))[:, :E])
    return SE.plant_nans(acts, N, nan_steps)


# ------------------------------------------------------------------------------ counters on every path
@pytest.mark.parametrize('kind', SE.SCENES)
@pytest.mark.parametrize('path', list(PATHS))
def test_counters_on_every_path(path, kind, thr, monkeypatch):
    """T single steps: every counter equals the oracle's count; the counters accumulate across launches"""
    E, N = _shape(path, monkeypatch)
    mode = 'set_speeds' if kind == 'nan_chunk' else None
    st = SE.make_scene(kind, N, E)
    acts = _actions(kind, mode, T, E, N, st)
    sw = _swarm(E, N, mode, kind)
    H.upload_state(sw, st)
    sw.stats.zero_()
    sw.read_status()
    for t in range(T):
        sw.step(_dev(acts[t]) if acts is not None else None)
    ex = _expect(kind, E, N, mode, acts, thr)
    assert _stats(sw) == ex, (path, kind, _stats(sw), ex)
    status = sw.read_status()
    want = (2 if ex['nonfinite'] else 0) | (1 if ex['nan_actions'] else 0)
    assert status & 3 == want, (status, want)


# ------------------------------------------------------------------------------ multi-step forms
@pytest.mark.parametrize('kind', ['heap', 'nan_chunk', 'nonfinite', 'lifting'])
@pytest.mark.parametrize('E,N', [(12, 8), (12, 5), (12, 16), (40000, 8)])
def test_forms_agree(E, N, kind, thr):
    """T plain steps, mrs_rollout (chained at 40000 x 8), graph replay and mrs_step_many: equal contact, ground,
    non-finite and NaN counts; contact_chunks and solver_sweeps follow each form's rule.  NaN at step 1: the warp-chunk
    of the lone NaN agent is a candidate only through the NaN, so the fast path must hand it over in the middle of a
    mrs_step_many launch (T - 1 = 2 contact chunk-steps) and the single-step forms count it once."""
    mode = 'set_speeds' if kind == 'nan_chunk' else None
    st = SE.make_scene(kind, N, E)
    acts = _actions(kind, mode, T, E, N, st, nan_steps=(1,))
    single = _expect(kind, E, N, mode, acts, thr)
    many = _expect(kind, E, N, mode, acts, thr, form='many')
    if kind == 'nan_chunk':
        lone = len(range(SE.LONE_NAN_ENV, E, SE.E0))
        lone_single = single['contact_chunks'] - _expect(kind, E, N, mode, acts, thr, nan_hands_off=False)['contact_chunks']
        lone_many = many['contact_chunks'] - _expect(kind, E, N, mode, acts, thr, 'many', nan_hands_off=False)['contact_chunks']
        assert lone_single == lone and lone_many == 2 * lone, (lone_single, lone_many, lone)
    got, states = {}, {}
    for form in ('step', 'rollout', 'graph', 'many'):
        # the graph replays T steps on a ring of T slots; the other forms get deep tapes, so that Swarm.step_many issues
        # ONE mrs_step_many launch of T steps (it splits a launch where a tape wraps, and T - t0 counts per launch)
        sw = _swarm(E, N, mode, kind, **(dict(tape_slots=T) if form == 'graph' else {}))
        H.upload_state(sw, st)
        a = _dev(acts)
        if form == 'graph':
            g = sw.capture_rollout(a, T)
            sw.stats.zero_()
            g.replay()
        else:
            sw.stats.zero_()
            if form == 'step':
                for t in range(T):
                    sw.step(a[t] if a is not None else None)
            elif form == 'rollout':
                sw.rollout(a, T)
            else:
                sw.step_many(a, T)
        got[form] = _stats(sw)
        states[form] = sw.state.clone()
    for form in ('step', 'rollout', 'graph'):
        assert got[form] == single, (form, got[form], single)
    assert got['many'] == many, (got['many'], many)
    for form in ('rollout', 'graph'):
        assert torch.equal(states['step'].nan_to_num(nan=-7.0), states[form].nan_to_num(nan=-7.0)), form


# ------------------------------------------------------------------------------ the NaN-action rule
def _ctrl_eq(a, b):
    return torch.equal(a.nan_to_num(nan=-7.0), b.nan_to_num(nan=-7.0))


@pytest.mark.parametrize('path', NAN_PATHS)
@pytest.mark.parametrize('mode', H.MODES)
def test_nan_action_single_step(mode, path, thr, monkeypatch):
    """NaN at step 0: the NaN agents step like the oracle's agent_none rule, keep their 18 PID planes bit for bit (and
    evolve them at the next finite step), mirror rpm 0, raise NAN_ACTION and not NONFINITE; envs outside their
    warp-chunk (N <= 32) or env (N > 32) equal a run with the NaN entries replaced by finite ones, bit for bit"""
    import mrsgym_b200 as M
    E, N = _shape(path, monkeypatch)
    st = SE.make_scene('nan_chunk', N, E)
    acts = _actions('nan_chunk', mode, 2, E, N, st)
    nan = np.any(np.isnan(acts[0]), -1)
    sw, clean = _swarm(E, N, mode, 'nan_chunk'), _swarm(E, N, mode, 'nan_chunk')
    for s in (sw, clean):
        H.upload_state(s, st)
        s.stats.zero_()
    ctrl0 = sw.ctrl.clone()
    sw.rpm.fill_(1.0)
    sw.step(_dev(acts[0]))
    clean.step(_dev(np.nan_to_num(acts[0], nan=0.25)))
    Eo = min(E, SE.E0)
    sub = {k: v[:Eo] for k, v in st.items()}
    env, steps = SE.oracle_run(sub, mode, acts[:1, :Eo], 1)
    g = H.read_state(sw)
    ref = H.spec_state(env)
    for k, tol in V.CONTACT_BAND:
        err = float(np.max(np.abs(g[k][:Eo] - ref[k])))
        assert err <= tol, (k, err)
    idx = torch.from_numpy(np.nonzero(nan.ravel())[0]).cuda()
    assert _ctrl_eq(sw.ctrl[:, idx], ctrl0[:, idx])
    assert float(sw.rpm[:, idx].abs().max()) == 0.0
    assert sw.read_stats()['nan_actions'] == int(nan.sum())
    status = sw.read_status(clear=False)
    assert status & M._abi.STATUS_NAN_ACTION and not status & M._abi.STATUS_NONFINITE
    gpw = SE.chunk_envs(N) or 1
    hit = {e // gpw for e in np.nonzero(nan.any(-1))[0]}
    others = [e for e in range(E) if e // gpw not in hit]
    sa, sb = sw.state.view(13, E, N), clean.state.view(13, E, N)
    assert torch.equal(sa[:, others], sb[:, others])
    assert _ctrl_eq(sw.ctrl.view(18, E, N)[:, others], clean.ctrl.view(18, E, N)[:, others])
    # a finite step: the NaN agents' controller runs again; the status bit stays (sticky) until it is read
    ctrl1 = sw.ctrl.clone()
    sw.step(_dev(np.nan_to_num(acts[1], nan=0.25)))
    if mode not in ('set_control', 'set_speeds'):
        assert not _ctrl_eq(sw.ctrl[:, idx], ctrl1[:, idx])
    # ... from the restored state: the two steps follow the NaN-aware oracle
    env2, _ = SE.oracle_run(sub, mode, acts[:2, :Eo], 2)
    g, ref = H.read_state(sw), H.spec_state(env2)
    for k, tol in V.TRAJ_BAR:
        err = float(np.max(np.abs(g[k][:Eo] - ref[k])))
        assert err <= tol, ('after the finite step', k, err)
    assert sw.read_stats()['nan_actions'] == int(nan.sum())
    assert sw.read_status(clear=False) & M._abi.STATUS_NAN_ACTION


@pytest.mark.parametrize('form', ['many', 'rollout'])
@pytest.mark.parametrize('path', ['runtime5', 'unrolled8', 'unrolled16', 'lanes48', 'tiled200'])
@pytest.mark.parametrize('mode', H.MODES)
def test_nan_action_mid_launch(mode, path, form, thr, monkeypatch):
    """NaN at step 1 of a 3-step mrs_step_many / mrs_rollout (the prefetched action and the mid-launch hand-off of the
    lone NaN agent's warp-chunk): within the trajectory bar of the oracle, every counter exact under the form's rule,
    NAN_ACTION without NONFINITE"""
    import mrsgym_b200 as M
    E, N = _shape(path, monkeypatch)
    st = SE.make_scene('nan_chunk', N, E)
    acts = _actions('nan_chunk', mode, T, E, N, st, nan_steps=(1,))
    sw = _swarm(E, N, mode, 'nan_chunk')
    H.upload_state(sw, st)
    sw.stats.zero_()
    (sw.step_many if form == 'many' else sw.rollout)(_dev(acts), T)
    env, steps = SE.oracle_run(st, mode, acts, T)
    g, ref = H.read_state(sw), H.spec_state(env)
    for k, tol in V.TRAJ_BAR:
        err = float(np.max(np.abs(g[k] - ref[k])))
        assert err <= tol, (k, err)
    ex = _expect('nan_chunk', E, N, mode, acts, thr, form=form if form == 'many' else 'single')
    assert _stats(sw) == ex, (_stats(sw), ex)
    assert ex['nan_actions'] == int(np.isnan(acts).any(-1).sum())
    status = sw.read_status()
    assert status & M._abi.STATUS_NAN_ACTION and not status & M._abi.STATUS_NONFINITE


def test_check_status_raises_the_reference_exception():
    import mrsgym_b200 as M
    env = M.MRS(N_AGENTS=8, N_ENVS=4, ACTION_TYPE='set_target_vel')
    a = torch.zeros(4, 8, 3, device='cuda')
    a[2, 3, 1] = float('nan')
    env.step(a)
    env.step(torch.zeros(4, 8, 3, device='cuda'))      # a later clean step leaves the bit set
    with pytest.raises(Exception, match='^The given action contains NaN$'):
        env.check_status()


# ------------------------------------------------------------------------------ NULL status / stats through the C ABI
@pytest.mark.parametrize('path', ['runtime5', 'unrolled8', 'lanes48', 'fused64', 'tiled200'])
def test_null_status_or_stats(path, monkeypatch):
    """status = NULL: the NaN actions are still counted; stats = NULL: the step runs and gives the same state"""
    E, N = _shape(path, monkeypatch)
    mode = 'set_speeds'
    st = SE.make_scene('nan_chunk', N, E)
    acts = _actions('nan_chunk', mode, 1, E, N, st)
    full, nostatus, nostats = (_swarm(E, N, mode, 'nan_chunk') for _ in range(3))
    nostatus.bufs.status = None
    nostats.bufs.stats = None
    for s in (full, nostatus, nostats):
        H.upload_state(s, st)
        s.stats.zero_()
        s.step(_dev(acts[0]))
    n = int(np.isnan(acts[0]).any(-1).sum())
    assert full.read_stats()['nan_actions'] == n and nostatus.read_stats()['nan_actions'] == n
    assert nostatus.read_status() == 0 and nostats.read_stats()['nan_actions'] == 0
    assert torch.equal(full.state, nostatus.state) and torch.equal(full.state, nostats.state)
