"""The tensor-core AIS ladder (bm_dbm_tc.cuh DbmTC::ais_local: the importance weights accumulated inside the epilogues of the
tcgen05 program kernel, bm_tc.cu MODE_AIS_*) run by run against the float64 oracle and against exact log Z.

The models have bf16-exact parameters (tests/golden/make_ais_tc_oracle.py), so every GEMM operand of the ladder is exact
and the engine and the oracle run the same chains on the same Philox uniforms: a chain parts from the oracle's only where a
uniform lands within rounding of its probability (a parted chain then differs by about 0.1 nats).  The other runs must agree
to fp32 summation error, which checks every column tile's share of a run's log-weight, the masks of the ragged tails, the
256-row blocks, the series and closed forms of the increment and the launch cuts of the ladder -- errors far below the
+-1-nat gate at the benchmark shape.  The oracle's log-weights are the committed fixture tests/golden/ais_tc_cases.json.

Not caught at these tolerances: errors of the increment below about 1e-5 relative, such as dropping the series' second-order
term (AIS_MAX_CT / AIS_MAX_CD in bm_tc.cu bound the form's own error at 3e-6)."""
import importlib.util
import os

import numpy as np
import pytest

from boltzmann_machines import _native

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
_spec = importlib.util.spec_from_file_location('make_ais_tc_oracle', os.path.join(HERE, 'golden', 'make_ais_tc_oracle.py'))
G = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(G)

FX = {c['name']: c for c in G.load()['cases']}
SAMPLED = [n for n, c in FX.items() if c['sample_v'] and all(c['sample_h'])]
UNSAMPLED = [n for n in FX if n not in SAMPLED]
EXACT = [n for n in SAMPLED if FX[n]['exact_log_z'] is not None]

# per-run agreement: |a - b| <= ATOL + RTOL |b| for at least FRAC of the compared runs, and no run a nat off.  On a B200 at
# most one chain of 124 parted from the oracle's (a 1000-temperature ladder, 0.1 nats); the others agreed to 1e-4 at most
# (1000 temperatures) and 2e-5 (200).  Crediting only the first column tile, or one form of the increment where the other
# belongs, moves every run by 0.05 to 190 nats.
ATOL, RTOL, FRAC = 2e-3, 1e-5, 0.97


def engine(case):
    eng = _native.CudaDBM(G.cfg(case, dtype='float32', compute='bf16'))
    assert eng.compute == 'bf16'
    eng.set_params(G.params(case))
    return eng


_LADDER = {}


def ladder(name, monkeypatch=None, **env):
    """the engine's log-weights of all the runs of a case (the default ladder is shared by the tests)"""
    key = (name, tuple(sorted(env.items())))
    if key not in _LADDER:
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        case = FX[name]
        eng = engine(case)
        try:
            _LADDER[key] = eng.ais(case['R'], case['n_betas'], case['k'], case['seed'])
        finally:
            eng.close()
            for k in env:
                monkeypatch.delenv(k)
    return _LADDER[key]


def oracle_runs(case):
    """(run indices, the oracle's log-weights) of the fixture's windows"""
    idx = np.concatenate([np.arange(w['first'], w['first'] + len(w['log_weights'])) for w in case['windows']])
    return idx, np.concatenate([np.asarray(w['log_weights'], dtype=np.float64) for w in case['windows']])


def agree(a, b, what):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    d = np.abs(a - b)
    ok = d <= ATOL + RTOL * np.abs(b)
    print('\n[ais-tc] %s: %d of %d runs agree (%.3f), median |diff| %.2e, max %.2e' % (what, ok.sum(), ok.size, ok.mean(),
                                                                                    np.median(d), d.max()))
    assert ok.mean() >= FRAC, (what, ok.mean(), np.sort(d)[-10:])
    assert d.max() < 1.0, (what, d.max())


@pytest.mark.parametrize('name', SAMPLED)
def test_ais_runs_match_the_float64_oracle(monkeypatch, name):
    case = FX[name]
    a = ladder(name, monkeypatch)
    assert a.shape == (case['R'],) and np.all(np.isfinite(a))
    idx, b = oracle_runs(case)
    agree(a[idx], b, name)


@pytest.mark.parametrize('name', EXACT)
def test_ais_log_z_is_as_close_to_exact_as_the_oracles(monkeypatch, name):
    """AIS's own error is not the engine's: the gate is the oracle's estimate on the same seeds and its distance to exact
    log Z (the 2- and 3-temperature ladders are far from it, the 1000-temperature ones within a few tenths)."""
    case = FX[name]
    a = ladder(name, monkeypatch)
    exact, b = case['exact_log_z'], case['lme']
    print('\n[ais-tc] %s: lme %.4f, oracle %.4f, exact %.4f' % (name, G.lme(a), b, exact))
    assert abs(G.lme(a) - b) < 0.02, (G.lme(a), b)
    assert abs(G.lme(a) - exact) <= abs(b - exact) + 0.05, (G.lme(a), b, exact)


@pytest.mark.parametrize('name', UNSAMPLED)
def test_ais_with_mean_valued_units_matches_the_oracle_in_distribution(monkeypatch, name):
    """sample_v=False / sample_h[1]=False take the closed-form units op with mean outputs; sample_h[0]=False the pass-per-
    kernel ladder.  Mean-valued units are rounded to bf16 before the next GEMM, so the chains part early: compared by
    their log-mean-exp against exact log Z and by their mean against the oracle's."""
    case = FX[name]
    a = ladder(name, monkeypatch)
    R, exact = case['R'], case['exact_log_z']
    print('\n[ais-tc] %s: lme %.4f (oracle %.4f, exact %.4f), mean %.4f (oracle %.4f +- %.4f)' % (
        name, G.lme(a), case['lme'], exact, a.mean(), case['mean'], case['std'] / np.sqrt(R)))
    assert np.all(np.isfinite(a))
    assert abs(G.lme(a) - exact) <= abs(case['lme'] - exact) + 0.1, (G.lme(a), case['lme'], exact)
    assert abs(a.mean() - case['mean']) <= 4 * case['std'] / np.sqrt(R) + 0.02, (a.mean(), case['mean'], case['std'])


@pytest.mark.parametrize('name', ['ragged_closed', 'k4_launch_cut'])
def test_launch_cuts_do_not_change_the_ladder(monkeypatch, name):
    """BM_DBM_AIS_OPS=7 cuts the ladder into launches of 7 ops, between the U and T ops of a temperature step (and, at
    k = 4, inside the step's sweeps); the default's 90-op cut falls inside a step at k = 4.  The same draws: only the order
    of the fp64 atomics may differ."""
    np.testing.assert_allclose(ladder(name, monkeypatch, BM_DBM_AIS_OPS='7'), ladder(name, monkeypatch), rtol=0, atol=1e-6)


@pytest.mark.parametrize('env', [dict(BM_DBM_AIS_EPILOGUE='0'), dict(BM_DBM_AIS_EPILOGUE='0', BM_DBM_AIS_FUSED='0')],
                         ids=['fused', 'passes'])
def test_pass_per_kernel_variants_match_the_epilogue_ladder(monkeypatch, env):
    """the kernel-per-pass ladders draw the same units but take the closed form on fp32 pre-activations where the default
    takes the series: held to the per-run tolerance, against the default and against the oracle"""
    name = 'ragged_series'
    a, d = ladder(name, monkeypatch, **env), ladder(name, monkeypatch)
    agree(a, d, '%s %s vs epilogue' % (name, '+'.join(sorted(env))))
    idx, b = oracle_runs(FX[name])
    agree(a[idx], b, '%s %s vs oracle' % (name, '+'.join(sorted(env))))


@pytest.mark.parametrize('first,n', [(0, 64), (250, 50)])
def test_first_run_computes_those_runs_of_the_ladder(monkeypatch, first, n):
    """ais(n, first_run=f) on the tensor-core engine (bm_dbm_ais_rows, how ranks shard the runs): runs [f, f + n) of the
    whole ladder, also when they straddle a 256-row block"""
    name = 'ragged_closed'
    case = FX[name]
    whole = ladder(name, monkeypatch)
    eng = engine(case)
    got = eng.ais(n, case['n_betas'], case['k'], case['seed'], first_run=first)
    eng.close()
    np.testing.assert_allclose(got, whole[first:first + n], rtol=0, atol=1e-6)


def test_ladders_past_32768_runs_go_in_chunks_keyed_by_the_run():
    """ais_slice runs long ladders in chunks of 32768 runs; run r draws from row r whatever the chunk.  At V=7, Hs=(5, 4)
    the float64 oracle is cheap enough to compute here."""
    case = dict(name='chunked', V=7, Hs=[5, 4], n_betas=10, k=1, R=32768 + 300, sample_v=True, sample_h=[True, True],
                scale=1.0, seed=2222)
    eng = engine(case)
    a = eng.ais(case['R'], case['n_betas'], case['k'], case['seed'])
    lo = 32768 - 150
    b = G.log_weights(case, n_runs=300, first_run=lo)
    agree(a[lo:lo + 300], b, 'chunked ladder, runs [%d, %d)' % (lo, lo + 300))
    tail = eng.ais(case['R'] - 32760, case['n_betas'], case['k'], case['seed'], first_run=32760)
    eng.close()
    np.testing.assert_allclose(tail, a[32760:], rtol=0, atol=1e-6)
