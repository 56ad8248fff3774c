"""bench.py contract: the reference arm (`--impl reference`, the CPU oracle port on a bounded sample) prints one JSON line with the keys
of the task statement, and under a multi-rank launch only rank 0 prints it; --dump-outputs writes what the last timed step computed,
the same for the same arguments, and on the GPU the engine arm's dump agrees with the reference arm's on the same problems."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_ARGS = ['--impl', 'reference', '--steps', '2', '--warmup', '3', '--ref-problems', '8']


def _run(env_extra=None, args=REF_ARGS):
    env = dict(os.environ)
    for k in ('RANK', 'LOCAL_RANK', 'WORLD_SIZE'):
        env.pop(k, None)
    env.update(env_extra or {})
    cmd = [sys.executable, os.path.join(ROOT, 'bench.py')] + list(args)
    return subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)


def _dump(path, B, N=45):
    """the arrays of one --dump-outputs directory, with their dtype and shapes checked"""
    shapes = {'x': (B, 10), 'u': (B, 5), 'terminated': (B,), 'x_guess': (B, N + 1, 10), 'u_guess': (B, N, 5), 'status': (B,),
              'problem_index': (B,)}
    assert sorted(os.listdir(path)) == sorted(k + '.npy' for k in shapes)
    out = {k: np.load(os.path.join(path, k + '.npy')) for k in shapes}
    for k, a in out.items():
        assert a.dtype == np.float64 and a.shape == shapes[k], (k, a.dtype, a.shape)
        assert np.isfinite(a).all(), k
    np.testing.assert_array_equal(out['problem_index'], np.arange(B))
    return out


def test_reference_arm_line():
    res = _run()
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.startswith('{')]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['metric'] == 'rti_iterations_per_sec' and d['higher_is_better'] is True
    assert d['steps'] == 2 and d['warmup'] == 3 and d['n_gpus'] == 1 and d['dtype'] == 'f64' and d['vs_baseline'] is None
    assert d['value'] > 0 and abs(d['ms_per_step'] * d['steps'] * 1e-3 * d['value'] - 8 * 2) < 1e-6 * 16      # 8 problems x 2 steps, one solve each
    cb = d['cpu_baseline']
    assert cb['kind'] == 'port' and cb['cores'] >= 1 and cb['value'] == d['value'] and '8 problems x 2' in cb['sample']
    assert d['e2e'] == {'value': d['value'], 'unit': d['unit'], 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    assert 'cfg1' in d['config']['workload'] and 'model' not in d['config']


def test_reference_arm_only_rank_zero_prints():
    res = _run({'RANK': '1', 'LOCAL_RANK': '1', 'WORLD_SIZE': '2', 'MASTER_ADDR': '127.0.0.1', 'MASTER_PORT': '29571'})
    assert res.returncode == 0, res.stderr[-2000:]
    assert not [l for l in res.stdout.splitlines() if l.startswith('{')]


def test_reference_arm_dumps_the_last_timed_step(tmp_path):
    """the same arguments give the same arrays; the dump follows warmup + steps closed-loop steps (3 + 2 = 2 + 3), one more step moves it"""
    runs = {'a': REF_ARGS, 'b': REF_ARGS, 'split': REF_ARGS[:2] + ['--steps', '3', '--warmup', '2'] + REF_ARGS[6:],
            'longer': REF_ARGS[:2] + ['--steps', '3'] + REF_ARGS[4:]}
    out = {}
    for name, args in runs.items():
        res = _run(args=args + ['--dump-outputs', str(tmp_path / name)])
        assert res.returncode == 0, res.stderr[-2000:]
        out[name] = _dump(tmp_path / name, 8)
    for k in out['a']:
        np.testing.assert_array_equal(out['a'][k], out['b'][k], err_msg=k)
        np.testing.assert_array_equal(out['a'][k], out['split'][k], err_msg=k)
    assert not np.array_equal(out['a']['x'], out['longer']['x'])


@pytest.mark.gpu
def test_engine_arm_dump_matches_the_reference_arm(tmp_path):
    """the timed closed loop of the CUDA engine and of the CPU oracle on the same 32 problems (same seeds): the dumped last step agrees to
    the parity tolerances of tests/test_gpu_parity.py, statuses identical"""
    common = ['--steps', '2', '--warmup', '3']
    eng = _run(args=common + ['--batch', '32', '--no-e2e', '--no-cpu', '--no-mlp', '--probe-steps', '1', '--dump-outputs', str(tmp_path / 'eng')])
    assert eng.returncode == 0, eng.stderr[-2000:]
    assert json.loads([l for l in eng.stdout.splitlines() if l.startswith('{')][0])['steps'] == 2
    ref = _run(args=common + ['--impl', 'reference', '--ref-problems', '32', '--dump-outputs', str(tmp_path / 'ref')])
    assert ref.returncode == 0, ref.stderr[-2000:]
    g, o = _dump(tmp_path / 'eng', 32), _dump(tmp_path / 'ref', 32)
    np.testing.assert_array_equal(g['status'], o['status'])
    np.testing.assert_array_equal(g['terminated'], o['terminated'])
    for k, tol in (('x', 1e-6), ('u', 1e-5), ('x_guess', 1e-5), ('u_guess', 1e-5)):
        a, b = g[k], o[k]
        err = float(np.abs(a - b).max()) / max(1.0, float(np.abs(b).max()))
        assert err <= tol, f'{k}: max rel err {err:.3e} > {tol}'
