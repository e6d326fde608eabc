"""Fixtures that hold OUTPUTS OF THE ORACLE (not of the reference): they exist because the oracle needs minutes for them and the GPU
box should spend its time on the GPU.  Each one is re-derived here, in part, so that the file cannot drift from oracle/."""
import json
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))


def test_benchmark_shape_ais_fixture_is_the_float64_oracles():
    """tests/golden/ais_benchmark_shape_oracle.json: chains are independent (Philox counters carry the chain index), so two chains
    from the middle of the ladder, recomputed alone, must reproduce the stored float64 log-weights bit for bit."""
    import importlib.util
    spec = importlib.util.spec_from_file_location('make_ais_benchmark_oracle', os.path.join(HERE, 'golden', 'make_ais_benchmark_oracle.py'))
    M = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(M)
    fx = json.load(open(os.path.join(HERE, 'golden', 'ais_benchmark_shape_oracle.json')))
    assert fx['shape'] == {k: (list(v) if isinstance(v, tuple) else v) for k, v in M.SHAPE.items()}
    assert len(fx['log_weights']) == fx['n_runs'] == 256
    got = M.log_weights(2, first_run=200)
    np.testing.assert_array_equal(got, np.asarray(fx['log_weights'][200:202]))
    # and the parameters are the ones the GPU test hands to the engines
    import sys
    sys.path.insert(0, HERE)
    d = M.weights()
    rng = np.random.RandomState(0)
    assert np.array_equal(d['vb'], (0.1 * rng.randn(784)).astype(np.float32))


def test_tensor_core_ais_fixture_is_the_float64_oracles():
    """tests/golden/ais_tc_cases.json: the case matrix and parameters are the generator's, the parameters are exact in bf16,
    two runs of a wide case across the 256-row boundary recomputed alone reproduce the stored log-weights bit for bit, and
    the stored exact log Z is the enumeration's."""
    import importlib.util
    from oracle.rbm import bf16_round
    spec = importlib.util.spec_from_file_location('make_ais_tc_oracle', os.path.join(HERE, 'golden', 'make_ais_tc_oracle.py'))
    M = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(M)
    fx = M.load()
    assert [c['name'] for c in fx['cases']] == [c['name'] for c in M.CASES]
    for case, got in zip(M.CASES, fx['cases']):
        assert {k: got[k] for k in case} == case, case['name']
        d = M.params(case)
        assert got['params_sha256'] == M.params_digest(d), case['name']
        for n, a in d.items():
            assert a.dtype == np.float32 and np.array_equal(bf16_round(a), a), (case['name'], n)
        assert [(w['first'], w['first'] + len(w['log_weights'])) for w in got['windows']] == M.windows(case), case['name']
        assert (got['exact_log_z'] is None) == (case['Hs'][0] > 14), case['name']
    byname = {c['name']: c for c in fx['cases']}
    case = byname['bench_widths']
    w = [w for w in case['windows'] if w['first'] <= 255 < w['first'] + len(w['log_weights'])][0]
    got = M.log_weights(M.CASE['bench_widths'], n_runs=2, first_run=255)
    np.testing.assert_array_equal(got, np.asarray(w['log_weights'][255 - w['first']:257 - w['first']]))
    assert M.exact_log_z(M.CASE['edge_mixed']) == byname['edge_mixed']['exact_log_z']
