"""TEST INFRASTRUCTURE: the float64 oracle's AIS log-weights for the tensor-core ladder's parity tests
(tests/test_zz_dbm_tc_ais_gpu.py), committed as tests/golden/ais_tc_cases.json because the oracle needs up to minutes per case.

The parameters are rounded to bf16 (and stored as float32), so every GEMM operand of the tensor-core ladder is exact: states
are 0/1 and W is already bf16.  The engine and the float64 oracle then see the same model and the same Philox uniforms, and
their chains part only where a uniform lands within rounding of its probability -- the log-weights can be compared run by
run.  The shapes put ragged tails on the column tiles of both unit ops, K across two 64-element chunks, runs across the
256-row blocks; the ladders take the series form (>= 400 temperatures), the closed form, both, and the degenerate 2 and 3;
k = 4 puts the 90-op launch boundary inside a temperature step.  H1 <= 14 keeps log Z exactly enumerable (v and h2 sum
out analytically).

Each case stores the oracle's log-weights of runs [0, 64) and of a window across the 256-row boundary, the log-mean-exp,
mean and standard deviation over all its runs, the exact log Z where H1 <= 14, and a digest of its parameters.
tests/test_oracle_fixtures.py re-derives two runs of one wide case (runs are independent chains: a subset recomputed with
`first_run` is exact) and the parameters.

    python tests/golden/make_ais_tc_oracle.py [case ...]       (about a minute on 8 cores; byte-identical output)
"""
import hashlib
import json
import os
import sys

for _v in ('OPENBLAS_NUM_THREADS', 'OMP_NUM_THREADS', 'MKL_NUM_THREADS'):
    os.environ.setdefault(_v, '1')

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (ROOT, os.path.join(ROOT, 'boltzmann-machines_b200')):
    if p not in sys.path:
        sys.path.insert(0, p)

OUT = os.path.join(HERE, 'ais_tc_cases.json')
AIS_SEED = 2222
WINDOWS = ((0, 64), (240, 300))         # runs compared one by one: the first block, and across the 256-row boundary


def _case(name, V, Hs, n_betas, k=1, R=300, sample_v=True, sample_h=(True, True), scale=1.0):
    return dict(name=name, V=V, Hs=list(Hs), n_betas=n_betas, k=k, R=R, sample_v=sample_v, sample_h=list(sample_h),
                scale=scale, seed=AIS_SEED)


CASES = [
    # all sampled: compared run by run
    _case('ragged_series', 300, (12, 530), 1000),            # ragged multi-tile on both unit ops, series form
    _case('ragged_closed', 300, (12, 530), 200),             # the same model, closed form
    _case('edge_mixed', 129, (14, 257), 400),                # one past a tile / chunk edge; series and closed forms mixed
    _case('bench_widths', 784, (10, 1000), 1000),            # the benchmark's widths
    _case('tile_multiples_k2', 256, (8, 512), 200, k=2),     # exact tile multiples, two sweeps per temperature
    _case('k_two_chunks', 200, (70, 300), 200),              # K = 70 spans two 64-element chunks (no enumeration)
    _case('ladder_2', 300, (12, 530), 2),                    # degenerate ladders
    _case('ladder_3_one_run', 129, (14, 257), 3, R=1),
    _case('k4_launch_cut', 300, (12, 530), 50, k=4),         # 12 ops per temperature: the 90-op launch cut is mid-step
    # mean-valued units: chains part early, compared in distribution
    _case('mean_v', 300, (12, 530), 200, sample_v=False),
    _case('mean_h2', 300, (12, 530), 200, sample_h=(True, False)),
    _case('mean_h1_passes', 300, (12, 530), 200, sample_h=(False, True)),
]
CASE = {c['name']: c for c in CASES}


def weight_seed(case):
    """one seed per case, from its name (stable under reordering of CASES)"""
    return int(hashlib.sha256(case['name'].encode()).hexdigest()[:8], 16)


def params(case):
    """W_i ~ scale N(0, 1) / sqrt(H1), biases 0.1 N(0, 1); all rounded to bf16, stored as float32"""
    from oracle.rbm import bf16_round
    rng = np.random.RandomState(weight_seed(case))
    V, (H1, H2) = case['V'], case['Hs']
    s = case['scale'] / np.sqrt(H1)
    d = {'vb': 0.1 * rng.randn(V), 'W': s * rng.randn(V, H1), 'hb': 0.1 * rng.randn(H1),
         'W_1': s * rng.randn(H1, H2), 'hb_1': 0.1 * rng.randn(H2)}
    return {n: bf16_round(a.astype(np.float32)) for n, a in d.items()}


def params_digest(d):
    h = hashlib.sha256()
    for n in sorted(d):
        h.update(n.encode()); h.update(np.ascontiguousarray(d[n], dtype=np.float32).tobytes())
    return h.hexdigest()


def cfg(case, dtype='float64', compute='fp32'):
    return dict(n_visible=case['V'], n_hiddens=list(case['Hs']), v_kind='bernoulli', h_kinds=['bernoulli'] * 2,
                h_n_samples=[100.] * 2, dtype=dtype, compute=compute, n_particles=4, batch_size=4, max_mf_updates=6,
                mf_tol=1e-6, l2=1e-4, max_norm=3.0, sample_v=case['sample_v'], sample_h=list(case['sample_h']),
                sparsity_target=[0.2] * 2, sparsity_cost=[0.01] * 2, sparsity_damping=0.9)


def log_weights(case, n_runs=None, first_run=0):
    """the float64 oracle's log Z estimates of runs [first_run, first_run + n_runs)"""
    from oracle.dbm import OracleDBM
    ref = OracleDBM(cfg(case))
    ref.set_params({n: a.astype(np.float64) for n, a in params(case).items()})
    n = case['R'] if n_runs is None else n_runs
    return np.asarray(ref.ais(n, case['n_betas'], case['k'], case['seed'], first_run=first_run), dtype=np.float64)


def exact_log_z(case):
    """log Z of the binary 2-layer DBM by enumeration over h1 (v and h2 summed out analytically); None past H1 = 14"""
    H1 = case['Hs'][0]
    if H1 > 14:
        return None
    d = {n: a.astype(np.float64) for n, a in params(case).items()}
    X = ((np.arange(2 ** H1)[:, None] >> np.arange(H1)[None, :]) & 1).astype(np.float64)
    t = X @ d['hb'] + np.logaddexp(0, X @ d['W'].T + d['vb']).sum(axis=1) + np.logaddexp(0, X @ d['W_1'] + d['hb_1']).sum(axis=1)
    return float(np.logaddexp.reduce(t))


def lme(v):
    v = np.asarray(v, dtype=np.float64)
    return float(np.logaddexp.reduce(v) - np.log(len(v)))


def windows(case):
    return [(lo, min(hi, case['R'])) for lo, hi in WINDOWS if lo < case['R']]


def run_case(case):
    v = log_weights(case)
    return dict(case, weight_seed=weight_seed(case), params_sha256=params_digest(params(case)),
                windows=[dict(first=lo, log_weights=[float(x) for x in v[lo:hi]]) for lo, hi in windows(case)],
                lme=lme(v), mean=float(v.mean()), std=float(v.std()), exact_log_z=exact_log_z(case))


def load():
    with open(OUT) as fh:
        return json.load(fh)


if __name__ == '__main__':
    import time
    from concurrent.futures import ProcessPoolExecutor
    names = sys.argv[1:] or [c['name'] for c in CASES]
    t0 = time.time()
    with ProcessPoolExecutor(max_workers=min(len(names), os.cpu_count() or 1)) as ex:
        got = dict(zip(names, ex.map(run_case, [CASE[n] for n in names])))
    old = {c['name']: c for c in load()['cases']} if os.path.isfile(OUT) and len(names) < len(CASES) else {}
    old.update(got)
    out = dict(generated_by='tests/golden/make_ais_tc_oracle.py (oracle/dbm.py, float64)', windows=[list(w) for w in WINDOWS],
               cases=[old[c['name']] for c in CASES])
    with open(OUT, 'w') as fh:
        json.dump(out, fh, indent=1)
        fh.write('\n')
    for n in names:
        c = got[n]
        ex_ = c['exact_log_z']
        print('%-18s lme %.4f  exact %s  lme-exact %s  std %.3f' % (
            n, c['lme'], 'n/a' if ex_ is None else '%.4f' % ex_, 'n/a' if ex_ is None else '%+.4f' % (c['lme'] - ex_), c['std']))
    print('%.0f s' % (time.time() - t0))
