"""CPU-only checks of the host side: the C-ABI library loads and exports every symbol
include/mrs_b200.h declares, the ctypes mirror matches the compiled structs, compute calls
fail loudly without a GPU (no fallback), env sharding and the statistics reduction (gloo,
world_size 2)."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import _REPO

HEADER = os.path.join(_REPO, 'include', 'mrs_b200.h')


def _lib():
    from mrsgym_b200 import _abi
    if not os.path.isfile(_abi.LIB_PATH):
        sys.path.insert(0, _REPO)
        import __graft_entry__
        __graft_entry__.build()
    return _abi


def test_header_symbols_are_exported():
    _abi = _lib()
    text = open(HEADER).read()
    names = set(re.findall(r'^\s*(?:int|size_t|const char\*|void\*)\s+(mrs_\w+)\s*\(', text, flags=re.M))
    assert len(names) >= 13
    handle = ctypes.CDLL(_abi.LIB_PATH)
    for n in names:
        assert hasattr(handle, n), n
    assert names == set(_abi.EXPORTS)


def test_struct_mirror_and_defaults():
    _abi = _lib()
    lib = _abi.lib()
    assert lib.mrs_abi_version() == _abi.ABI_VERSION
    assert lib.mrs_sizeof_config() == ctypes.sizeof(_abi.MrsConfig)
    assert lib.mrs_sizeof_buffers() == ctypes.sizeof(_abi.MrsBuffers)
    cfg = _abi.default_config()
    from oracle import bullet_model as bm, spec
    Q, P = bm.QuadParams(), bm.PhysicsParams()
    assert cfg.quad.mass == np.float32(Q.mass) and cfg.quad.kf == np.float32(Q.kf)
    assert abs(cfg.quad.gnd_hclip - Q.derived()['GroundEffectHClip']) < 1e-8
    np.testing.assert_allclose(list(cfg.phys.inertia), P.inertia_diag(), rtol=1e-6)
    np.testing.assert_allclose(np.array(list(cfg.quad.nnls_tab)).reshape(16, 4, 4), spec.nnls_subset_tables(), atol=1e-7)
    np.testing.assert_allclose(np.array(list(cfg.quad.mix_ainv)).reshape(4, 4), spec.MIX_AINV, atol=1e-7)
    for mode, code in _abi.ACTION_TYPES.items():
        assert lib.mrs_action_dim(code) == spec.ACTION_DIMS[mode]
    assert lib.mrs_state_dim(_abi.X_POS_VEL) == 6 and lib.mrs_state_dim(_abi.X_FULL) == 13


def test_baked_constants_match_the_library_defaults():
    """csrc/mrs_baked.cuh (immediates of the specialised kernels) is generated from the library's own
    mrs_default_config + host derivation: the committed header must be current, the default configuration
    must select the baked kernels and any other value must not."""
    _abi = _lib()
    lib = _abi.lib()
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    rc = subprocess.run([sys.executable, os.path.join(root, 'tools', 'gen_baked.py'), '--check']).returncode
    assert rc == 0, 'mrs_baked.cuh is stale: run tools/gen_baked.py and rebuild'
    cfg = _abi.default_config()
    cfg.E, cfg.N, cfg.K, cfg.L = 7, 5, 2, 9                       # run-time fields do not matter
    cfg.comm_range = 1.25
    assert lib.mrs_config_is_baked(ctypes.byref(cfg)) == 1
    for poke in ('dt', 'gravity'):
        c2 = _abi.default_config()
        setattr(c2, poke, float(np.nextafter(np.float32(getattr(c2, poke)), np.float32(np.inf))))
        assert lib.mrs_config_is_baked(ctypes.byref(c2)) == 0, poke
    c3 = _abi.default_config()
    c3.quad.kf = float(np.nextafter(np.float32(c3.quad.kf), np.float32(1)))
    assert lib.mrs_config_is_baked(ctypes.byref(c3)) == 0
    c4 = _abi.default_config()
    c4.phys.gyro = 0
    assert lib.mrs_config_is_baked(ctypes.byref(c4)) == 0
    c5 = _abi.default_config()
    c5.quad.nnls_tab[3] = 0.5                                      # tables are read at run time: still baked
    assert lib.mrs_config_is_baked(ctypes.byref(c5)) == 1


def test_scratch_planes_follow_the_pair_slices():
    """mrs_scratch_planes(E, N): nothing for the one-warp envs, 7 planes for the lanes-per-agent / thread-per-agent
    kernels (N <= 128), 7 + 2 per partner slice for the tiled pair pass -- at most 32 slices, at most one per 128
    partners, fewer as the env count alone fills the GPU."""
    lib = _lib().lib()
    assert lib.mrs_scratch_planes(10, 8) == 0 and lib.mrs_scratch_planes(1, 32) == 0
    for N in (33, 64, 128):
        assert lib.mrs_scratch_planes(1, N) == 7 and lib.mrs_scratch_planes(5000, N) == 7
    assert lib.mrs_scratch_planes(1, 4096) == 7 + 2 * 32
    assert lib.mrs_scratch_planes(1, 129) == 7 + 2 * 2          # two tiles of 128: two slices at most
    assert lib.mrs_scratch_planes(1, 1024) == 7 + 2 * 8
    last = None
    for E in (1, 2, 8, 64, 1000, 100000):
        p = lib.mrs_scratch_planes(E, 2048)
        assert 9 <= p <= 7 + 2 * 16 and (p - 7) % 2 == 0
        assert last is None or p <= last                         # more envs never need more slices
        last = p
    assert lib.mrs_scratch_planes(100000, 2048) == 9
    assert lib.mrs_scratch_planes(0, 64) == 0


@pytest.mark.skipif(torch.cuda.is_available(), reason='checks the no-GPU behaviour')
def test_no_cpu_fallback():
    import mrsgym_b200 as M
    with pytest.raises(Exception):
        M.Swarm(1, 3)
    with pytest.raises(M.MrsError):
        M.Swarm(1, 3, device='cpu')
    # argument errors are reported, not crashed on
    _abi = M._abi
    assert _abi.lib().mrs_step(None, None, None, 0, 0, None) == -1
    assert b'argument' in _abi.lib().mrs_strerror(-1)


def test_shard_range_partitions_envs():
    from mrsgym_b200 import shard_range
    for E in (1, 7, 64, 65536, 65537):
        for W in (1, 2, 3, 8):
            spans = [shard_range(E, r, W) for r in range(W)]
            assert spans[0][0] == 0 and spans[-1][1] == E
            assert all(spans[i][1] == spans[i + 1][0] for i in range(W - 1))
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1


def test_spawn_rejection_sampler():
    from mrsgym_b200 import DefaultSpawn, sample_start_pos
    torch.manual_seed(0)
    d = DefaultSpawn(6)
    s = d.sample()
    assert s.shape == (6, 3)
    assert float(s[:, :2].norm(dim=-1).max()) <= 1.0 + 1e-6 and 1.0 <= float(s[:, 2].min()) and float(s[:, 2].max()) <= 3.0
    pos = sample_start_pos(d, 32, 6, 0.3)
    dist = (pos.unsqueeze(2) - pos.unsqueeze(1)).norm(dim=-1) + 10 * torch.eye(6)
    assert float(dist.min()) >= 0.6


_WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, os.path.join(%(repo)r, 'mrs-gym_b200'))
from mrsgym_b200.core import shard_range
from mrsgym_b200.dist import allreduce_stats, init_from_env
rank, world = init_from_env(backend='gloo')
lo, hi = shard_range(10, rank, world)
stats = torch.tensor([hi - lo, rank + 1, 0, 0, 0, 0, 0, 0], dtype=torch.int64)
out = allreduce_stats(stats)
assert out.tolist()[:2] == [10, 3], out
dist.destroy_process_group()
print('ok', rank)
'''


def test_stats_allreduce_gloo_world2(tmp_path):
    script = tmp_path / 'w.py'
    script.write_text(_WORKER % dict(repo=_REPO))
    env = dict(os.environ, MASTER_ADDR='127.0.0.1', MASTER_PORT='29591', WORLD_SIZE='2')
    procs = [subprocess.Popen([sys.executable, str(script)], env=dict(env, RANK=str(r), LOCAL_RANK=str(r)),
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT) for r in range(2)]
    outs = [p.communicate(timeout=120)[0].decode() for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    assert all('ok' in o for o in outs)


def test_header_is_plain_c():
    """include/mrs_b200.h is the drop-in boundary for non-Python callers (cgo / JNI / N-API): it must compile as
    C99 and as C++ without any CUDA or torch type."""
    import shutil
    import subprocess
    if shutil.which('gcc') is None:
        pytest.skip('no gcc')
    for cmd in (['gcc', '-std=c99', '-Wall', '-Wextra', '-pedantic', '-Werror', '-fsyntax-only', '-x', 'c', HEADER],
                ['g++', '-std=c++11', '-Wall', '-Werror', '-fsyntax-only', '-x', 'c++', HEADER]):
        r = subprocess.run(cmd, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
    text = open(HEADER).read()
    assert '#include <cuda' not in text and '#include <torch' not in text and 'at::Tensor' not in text


def test_reference_arm_prints_the_bench_contract():
    """bench.py --impl reference runs on the CPU alone (oracle port on all host cores, a bounded sample) and prints
    ONE JSON line on stdout with the contract's keys; under torchrun only rank 0 prints."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--impl', 'reference', '--steps', '2', '--warmup', '1'],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-500:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ('impl', 'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
              'vs_baseline', 'dtype', 'data', 'config', 'cpu_baseline', 'e2e'):
        assert k in d, k
    assert d['impl'] == 'reference' and d['metric'] == 'agent-steps/sec' and d['value'] > 0
    assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1 and d['cpu_baseline']['value'] == d['value']
    assert d['e2e'] == {'value': d['value'], 'unit': d['unit'], 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    env = dict(os.environ, RANK='1', WORLD_SIZE='2')
    r1 = subprocess.run([sys.executable, os.path.join(root, 'bench.py'), '--impl', 'reference', '--steps', '2'],
                        capture_output=True, text=True, timeout=120, env=env)
    assert r1.returncode == 0 and r1.stdout.strip() == ''


def test_bench_dump_outputs_within_the_budget(tmp_path):
    """bench.py --dump-outputs: arrays are written whole when they fit the budget; otherwise every array keeps the
    same fraction of its rows, the same rows on every run, and all of them together fit."""
    import bench
    rng = np.random.default_rng(1)
    arrays = {'A': rng.random((2, 32, 64), dtype=np.float32), 'X': rng.random((2, 32, 6), dtype=np.float32)}
    bench.dump_outputs(str(tmp_path / 'whole'), arrays)
    for k, a in arrays.items():
        np.testing.assert_array_equal(np.load(tmp_path / 'whole' / (k + '.npy')), a)
    budget = 8000
    for d in ('s1', 's2'):
        bench.dump_outputs(str(tmp_path / d), arrays, budget=budget)
    got = {k: np.load(tmp_path / 's1' / (k + '.npy')) for k in arrays}
    assert 0 < sum(a.nbytes for a in got.values()) <= budget
    total = sum(a.nbytes for a in arrays.values())
    for k, a in got.items():
        rows = arrays[k].reshape(-1, arrays[k].shape[-1])
        assert a.dtype == np.float32 and a.shape == (len(rows) * budget // total, rows.shape[1])
        assert all((rows == r).all(axis=1).any() for r in a)
        np.testing.assert_array_equal(np.load(tmp_path / 's2' / (k + '.npy')), a)


def test_plain_c_caller_links_and_runs(tmp_path):
    """examples/c_abi_smoke.c: a C99 program with no CUDA headers links against libmrs_b200.so and uses the
    configuration / validation entry points (the part of the ABI that needs no device)."""
    import shutil
    import subprocess
    _abi = _lib()
    if shutil.which('gcc') is None:
        pytest.skip('no gcc')
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    libdir = os.path.dirname(_abi.LIB_PATH)
    exe = str(tmp_path / 'c_abi_smoke')
    r = subprocess.run(['gcc', '-std=c99', '-Wall', '-Werror', '-I', os.path.join(root, 'include'),
                        os.path.join(root, 'examples', 'c_abi_smoke.c'), '-o', exe, '-L', libdir, '-lmrs_b200',
                        '-Wl,-rpath,' + libdir], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert 'baked 1' in r.stdout and 'action dim 4' in r.stdout


def test_box_shim():
    from mrsgym_b200.spaces import Box
    b = Box(np.array([0.0, -1.0], dtype=np.float32), np.array([1.0, 1.0], dtype=np.float32))
    assert b.shape == (2,)
    x = b.sample()
    assert x.shape == (2,) and b.contains(x) and not b.contains(np.array([2.0, 0.0], dtype=np.float32))
    u = Box(np.full((3,), -np.inf, dtype=np.float32), np.full((3,), np.inf, dtype=np.float32))
    assert u.sample().shape == (3,)


def test_pin_bullet_runs_on_the_fake_backend():
    """tools/pin_bullet.py (SURVEY.md 8a-P 'pin these first') is exercised on oracle/fake_pybullet so that it is known
    to run the day a real pybullet wheel is importable; on the fake backend it reads the oracle's constants back."""
    sys.path.insert(0, os.path.join(_REPO, 'tools'))
    import importlib
    pin = importlib.import_module('pin_bullet')
    from oracle import bullet_model as bm
    doc = pin.main(['--backend', 'fake', '--models', '/nonexistent/models'])
    assert doc['backend'] == 'fake'
    pp, pr = doc['PhysicsParams'], doc['probes']
    P = bm.PhysicsParams()
    assert abs(pr['gravity'] - 9.81) < 1e-9
    assert abs(pp['lin_damping'] - P.lin_damping) < 1e-6 and abs(pp['ang_damping'] - P.ang_damping) < 1e-6
    assert abs(pr['link0_arm_x'] - 0.028) < 1e-9 and abs(pr['link0_arm_y'] - 0.028) < 1e-9
    assert pp['max_coord_vel'] == P.max_coord_vel and pp['gyro'] is True
    np.testing.assert_allclose(pp['measured_inertia_diag'], P.inertia_diag(), rtol=1e-12)
    assert abs(pr['rest']['height'] - (P.ground_z + P.col_halfheight + P.col_margin - P.slop)) < 1e-6
    assert pr['tilted_landing']['body_z_dot_world_z'] > 0.999999
    assert len(pr['one_step_goldens']) == 8
    # the JSON loads back into the oracle's parameter set
    import json, tempfile
    with tempfile.NamedTemporaryFile('w', suffix='.json', delete=False) as f:
        json.dump(doc, f)
    P2 = bm.PhysicsParams.from_json(f.name)
    assert P2.solver_iters == 50 and abs(P2.mu_ground - 0.75) < 1e-12


def test_rollout_dataset_in_the_reference_trainer_layout(tmp_path):
    """to_trainer_history: the batched dataset as Trainer.history (helper/Trainer.py:89-108) -- the valid K-step windows
    that Trainer.update_valid_idxs (:128-138) derives from the `done` list never straddle two envs or two episodes."""
    import mrsgym_b200 as M
    T, E, N, D, K = 7, 3, 4, 6, 2
    g = torch.Generator().manual_seed(3)
    data = {'X': torch.randn(T, E, N, D, generator=g), 'A': (torch.rand(T, E, N, N, generator=g) < 0.5).float(),
            'action': torch.randn(T, E, N, 3, generator=g), 'done': torch.zeros(T, E, dtype=torch.bool)}
    data['done'][3, 1] = True                           # env 1 ends an episode after step 3
    h = M.to_trainer_history(data)
    assert len(h['X']) == len(h['A']) == len(h['expert']) == len(h['done']) == len(h['context']) == T * E
    assert h['X'][T + 4].shape == (N, D) and torch.equal(h['X'][T + 4], data['X'][4, 1])
    assert torch.equal(h['A'][2 * T + 6], data['A'][6, 2]) and torch.equal(h['expert'][0], data['action'][0, 0])
    assert [i for i, d in enumerate(h['done']) if d] == [T - 1, T + 3, 2 * T - 1, 3 * T - 1]
    # the reference's window bookkeeping, restated: an entry is a valid window end when K earlier entries of the same
    # episode precede it
    valid, since = [], -1
    for idx, d in enumerate(h['done']):
        since = -1 if d else since + 1
        if since >= K:
            valid.append(idx)
    for idx in valid:
        env = idx // T
        assert all((idx - k) // T == env for k in range(K + 1))
        assert not any(h['done'][idx - k] for k in range(K + 1))
    M.save_dataset(data, str(tmp_path / 'd.pt'))
    back = torch.load(str(tmp_path / 'd.pt'))
    assert all(torch.equal(back[k], data[k]) for k in data)
