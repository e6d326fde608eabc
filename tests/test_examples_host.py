"""The reference's own example scripts against this package (north_star; SURVEY.md section 8 f.1).  The scripts are the original
project's source and stay out of this repository: tests/golden/make_example_traces.py ran them UNCHANGED (Python-2 syntax rewritten
in memory, Keras / the MNIST loader replaced by stand-ins: tests/example_runner.py), twice each -- training, then the rerun that
takes the load_model branches -- and recorded every call they made into the package.  These tests make the same calls, on the
CPU with the oracle engines (the host logic is the same whichever engine computes), and check what the scripts went on to use."""
import json
import os

import numpy as np

from example_runner import replay, translate

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def replay_example(name, workdir):
    with open(os.path.join(GOLDEN, 'example_{0}_trace.json'.format(name))) as fh:
        calls = json.load(fh)['calls']
    with np.load(os.path.join(GOLDEN, 'example_{0}_trace.npz'.format(name))) as z:
        arrays = {k: z[k] for k in z.files}
    results = replay(calls, arrays, str(workdir))
    return {c['method']: [r for d, r in zip(calls, results) if d['method'] == c['method']] for c in calls}


def test_translate_handles_the_two_python2_constructs_of_the_examples():
    src = 'print __doc__\ndef f((a, b), c,\n      (d, e), k=1):\n    print "x: {0}".format(a)\n    return a + e\n'
    g = {'__doc__': 'doc'}
    exec(compile(translate(src), '<t>', 'exec'), g)
    assert g['f']((1, 2), 3, (4, 5)) == 6


def test_rbm_mnist_example_runs_unchanged(oracle_engines, tmp_path):
    got = replay_example('rbm_mnist', tmp_path)
    params = json.load(open(str(tmp_path / 'rbm' / 'params.json')))
    assert params['n_hidden'] == 48 and params['epoch_'] == 2
    trained, loaded = got['get_tf_params']                # what the script hands to Keras: the trained RBM weights
    assert trained['W'].shape == (784, 48) and np.abs(trained['W']).max() > 0.011
    # the rerun finds the model directory and takes the script's load_model branch
    assert len(got['load_model']) == 1 and all(np.array_equal(trained[k], loaded[k]) for k in trained)


def test_dbm_mnist_example_runs_unchanged(oracle_engines, tmp_path):
    got = replay_example('dbm_mnist', tmp_path)
    assert len(got['fit']) == 3 and len(got['transform']) == 2          # RBM #1, RBM #2 (each feeding the next), the DBM
    params = json.load(open(str(tmp_path / 'dbm' / 'params.json')))
    assert params['n_hiddens_'] == [32, 24] and params['epoch_'] == 2
    trained, loaded = got['get_tf_params']
    assert trained['W'].shape == (784, 32) and trained['W_1'].shape == (32, 24)
    # the rerun loads every model from disk, `dbm.load_rbms(rbms)` included (dbm_mnist.py:133-134)
    assert len(got['load_model']) == 3 and len(got['load_rbms']) == 1
    assert all(np.array_equal(trained[k], loaded[k]) for k in trained)
