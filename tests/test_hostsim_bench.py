"""bench.py's own control flow on the CPU: the headline benchmark script run end to end on the stand-in CUDA runtime
(tests/hostsim, launches recorded and checked but not interpreted -- timings are meaningless there).  Checks the JSON
contract of the line it prints and that no launch, copy or tensor map of the benchmark-sized run breaks a runtime rule
(the run that first showed a dataset conversion launch beyond the grid limit)."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def load_bench():
    """bench.py as a new module: its constants read the environment at import, and an earlier test may hold an import of it"""
    spec = importlib.util.spec_from_file_location('bench_under_test', os.path.join(ROOT, 'bench.py'))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


RUNNER = r'''
import sys, runpy, ctypes as C
sys.path[:0] = [{root!r}, {pkg!r}]
from boltzmann_machines import _native
sim = _native.load_library({sim!r})
sim.fakecuda_violation.restype = C.c_char_p
_native._lib = sim
sys.argv = ['bench.py', '--steps', '6', '--warmup', '3', '--no-cpu-baseline', '--dump-outputs', {dump!r}]
try:
    runpy.run_path({bench!r}, run_name='__main__')
finally:
    print('VIOLATIONS=' + sim.fakecuda_violation().decode())
'''


def test_bench_contract_on_the_host_simulation(tmp_path):
    obj = os.path.join(ROOT, 'boltzmann-machines_b200', 'build')
    if not (os.path.isdir(obj) and any(f.endswith('.o') for f in os.listdir(obj))):
        pytest.skip('library objects not built (run build.sh / __graft_entry__.build())')
    subprocess.check_call(['bash', os.path.join(ROOT, 'tests', 'hostsim', 'build.sh')], stdout=subprocess.DEVNULL)
    code = RUNNER.format(root=ROOT, pkg=os.path.join(ROOT, 'boltzmann-machines_b200'),
                         sim=os.path.join(ROOT, 'tests', 'hostsim', '_build', 'libbm_hostsim.so'), bench=os.path.join(ROOT, 'bench.py'),
                         dump=str(tmp_path / 'outputs'))
    # 20 batches = 81920 rows: still taller than grid.y can index (the refused-launch case), half the host-side data shuffling
    env = dict(os.environ, BM_BENCH_BATCHES='20')
    res = subprocess.run([sys.executable, '-c', code], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600, cwd=str(tmp_path), env=env)
    assert res.returncode == 0, res.stdout[-3000:]
    assert 'VIOLATIONS=\n' in res.stdout + '\n', res.stdout[-1500:]
    line = [l for l in res.stdout.splitlines() if l.startswith('{"metric"')]
    assert len(line) == 1, res.stdout[-1500:]
    out = json.loads(line[0])
    for key in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling', 'vs_baseline',
                'dtype', 'data', 'config', 'gpu_launches', 'clocks', 'roofline', 'e2e'):
        assert key in out, key
    assert out['n_gpus'] == 1 and out['steps'] == 6 and out['higher_is_better'] is True and out['scaling'] == 'weak'
    assert out['config']['workload'].startswith('BernoulliRBM 784-1024') and 'model' not in out['config']
    assert set(out['roofline']) >= {'bound', 'achieved', 'peak', 'unit', 'frac', 'traffic'}
    assert set(out['e2e']) >= {'value', 'unit', 'h2d_bytes_per_step', 'd2h_bytes_per_step'}
    assert out['e2e']['h2d_bytes_per_step'] == 4096 * 784          # one byte per visible unit and row
    assert 'fit_region_failed' not in out['e2e'] and out['e2e']['path'].startswith('Model(**kwargs).fit(X)')
    assert out['gpu_launches'] == 2 * out['steps']                  # the step's program and the update kernel
    assert out['e2e']['steps'] == out['steps']                       # fit() runs exactly the K steps it was given
    shapes = {'W': (784, 1024), 'dW': (784, 1024), 'vb': (784,), 'dvb': (784,), 'hb': (1024,), 'dhb': (1024,), 'q_means': (1024,)}
    dumped = {f[:-4]: np.load(str(tmp_path / 'outputs' / f)) for f in os.listdir(str(tmp_path / 'outputs'))}
    assert {k: (a.shape, a.dtype) for k, a in dumped.items()} == {k: (s, np.float32) for k, s in shapes.items()}


def test_reference_arm_prints_the_same_config_and_runs_exactly_the_steps_it_was_given(tmp_path, monkeypatch):
    """`bench.py --impl reference --steps K --warmup W`: the oracle port on the host cores; same `config` object as the b200 arm,
    exactly K timed steps (each a bounded sample of the workload's step when K full steps would not fit the time budget), and the
    cpu_baseline / e2e objects the contract asks of this arm."""
    env = dict(os.environ, BM_BENCH_REFERENCE_SECONDS='3', BM_BENCH_BATCHES='20')
    res = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '7', '--warmup', '2'],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600, cwd=str(tmp_path), env=env)
    assert res.returncode == 0, res.stdout[-3000:]
    out = json.loads([l for l in res.stdout.splitlines() if l.startswith('{"impl"')][0])
    assert out['impl'] == 'reference' and out['steps'] == 7 and out['warmup'] == 2 and out['n_gpus'] == 1
    assert out['metric'] == 'gibbs_updates_per_sec' and out['unit'] == 'updates/s' and out['higher_is_better'] is True
    monkeypatch.setenv('BM_BENCH_BATCHES', '20')
    assert out['config'] == load_bench().rbm_config('cfg2', 1)
    assert out['cpu_baseline']['kind'] == 'port' and out['cpu_baseline']['value'] == out['value'] and out['cpu_baseline']['cores'] >= 1
    assert 'rows each of the batch of 4096' in out['cpu_baseline']['sample']          # 9 full steps do not fit 3 seconds
    assert out['e2e'] == {'value': out['value'], 'unit': 'updates/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}


def test_bench_with_two_ranks_on_the_host_simulation(tmp_path):
    """the launch the driver uses for N > 1 (torchrun, one rank per GPU) with both ranks on the stand-in runtime and the shared-memory
    stand-in for NCCL: rank 0 prints one line for the whole job, the engine-level regions and fit() run data parallel, nothing
    breaks a runtime rule"""
    pytest.importorskip('torch')
    obj = os.path.join(ROOT, 'boltzmann-machines_b200', 'build')
    if not (os.path.isdir(obj) and any(f.endswith('.o') for f in os.listdir(obj))):
        pytest.skip('library objects not built (run build.sh / __graft_entry__.build())')
    subprocess.check_call(['bash', os.path.join(ROOT, 'tests', 'hostsim', 'build.sh')], stdout=subprocess.DEVNULL)
    env = dict(os.environ, BM_BENCH_BATCHES='4',
               BM_NCCL_LIB=os.path.join(ROOT, 'tests', 'hostsim', '_build', 'libfakenccl.so'))
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr', '127.0.0.1',
           '--master-port', str(29900 + os.getpid() % 90), os.path.join(ROOT, 'tools', 'hostsim_run.py'), os.path.join(ROOT, 'bench.py'),
           '--gpus', '2', '--steps', '6', '--warmup', '3', '--no-cpu-baseline']
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900, cwd=str(tmp_path), env=env)
    assert res.returncode == 0, res.stdout[-3000:]
    lines = [l for l in res.stdout.splitlines() if l.startswith('{"metric"')]
    assert len(lines) == 1, res.stdout[-2000:]
    out = json.loads(lines[0])
    assert out['n_gpus'] == 2 and out['steps'] == 6 and out['scaling'] == 'weak'
    assert out['config']['parallelism'] == 'dp2' and out['config']['global_batch'] == 2 * 4096
    assert out['e2e']['h2d_bytes_per_step'] == 2 * 4096 * 784 and out['e2e']['steps'] == 6 and 'fit_region_failed' not in out['e2e']
    assert res.stdout.count('violations: none') == 2, res.stdout[-2000:]


def test_dump_outputs_keeps_the_same_sample_within_64_mb(tmp_path):
    """`--dump-outputs` past 64 MB in all: each array keeps the same seeded sample of its rows, in its own dtype"""
    bench = load_bench()
    rng = np.random.RandomState(1)
    arrays = {'W': rng.rand(5000, 4096).astype(np.float32), 'logw': rng.randn(20000)}       # 78 MB + 0.16 MB
    for d in ('a', 'b'):
        bench.dump_outputs(arrays, str(tmp_path / d))
    a = {k: np.load(str(tmp_path / 'a' / (k + '.npy'))) for k in arrays}
    b = {k: np.load(str(tmp_path / 'b' / (k + '.npy'))) for k in arrays}
    assert sum(x.nbytes for x in a.values()) <= 64 * 2 ** 20 < sum(x.nbytes for x in arrays.values())
    for k, x in arrays.items():
        assert a[k].dtype == x.dtype and a[k].shape[1:] == x.shape[1:] and 0.8 * len(x) < len(a[k]) < len(x)
        assert np.array_equal(a[k], b[k])
        first = lambda m: m.reshape(len(m), -1)[:, 0]
        assert np.isin(first(a[k]), first(x)).all()                 # rows of the output, not new values
