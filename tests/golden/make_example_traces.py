"""Records tests/golden/example_{rbm,dbm}_mnist_trace.json (+ .npz): every call the original project's example scripts
examples/rbm_mnist.py and examples/dbm_mnist.py make into this package, each script run UNCHANGED (tests/example_runner.py) on
the oracle engines, twice -- training, then the rerun that loads the saved models.  tests/test_examples_host.py replays the calls.
The scripts stay in the original's checkout; run where one exists:

    python tests/golden/make_example_traces.py <examples/ directory of a checkout of yell/boltzmann-machines>
"""
import contextlib
import io
import json
import os
import shutil
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'boltzmann-machines_b200'), os.path.dirname(HERE)]

from example_runner import Recorder, run_example                     # noqa: E402

# the command lines the scripts run with; {workdir} is the directory the models are written to
ARGS = {
    'rbm_mnist': ['--n-train', '512', '--n-val', '128', '--n-hidden', '48', '--epochs', '2', '--batch-size', '64',
                  '--model-dirpath', '{workdir}/rbm/', '--mlp-save-prefix', '{workdir}/rbm_', '--mlp-epochs', '1'],
    'dbm_mnist': ['--n-train', '256', '--n-val', '64', '--n-hiddens', '32', '24', '--epochs', '1', '1', '2',
                  '--batch-size', '32', '32', '32', '--increase-n-gibbs-steps-every', '1', '--n-particles', '32',
                  '--max-mf-updates', '5', '--rbm1-dirpath', '{workdir}/rbm1/', '--rbm2-dirpath', '{workdir}/rbm2/',
                  '--dbm-dirpath', '{workdir}/dbm/', '--mlp-save-prefix', '{workdir}/dbm_', '--mlp-epochs', '1'],
}
# what the script prints on its first and second run (the second takes the load_model branches)
PRINTS = {'rbm_mnist': (('Training model', 'Test accuracy'), ('Loading model',)),
          'dbm_mnist': (('Training RBM #1', 'Training RBM #2', 'Training DBM', 'Test accuracy'), ('Loading RBM #1', 'Loading DBM'))}


def record(examples, name):
    from boltzmann_machines.base import set_engine_factory
    from oracle.dbm import dbm_factory
    from oracle.rbm import rbm_factory
    set_engine_factory('rbm', rbm_factory)
    set_engine_factory('dbm', dbm_factory)
    workdir = tempfile.mkdtemp(prefix='bm_example_')
    try:
        argv = [a.replace('{workdir}', workdir) for a in ARGS[name]]
        with Recorder(workdir) as rec:
            for expected in PRINTS[name]:
                out = io.StringIO()
                with contextlib.redirect_stdout(out):
                    run_example(os.path.join(examples, name + '.py'), argv)
                missing = [p for p in expected if p not in out.getvalue()]
                assert not missing, '{0}: the script did not print {1}'.format(name, missing)
    finally:
        shutil.rmtree(workdir, ignore_errors=True)
    with open(os.path.join(HERE, 'example_{0}_trace.json'.format(name)), 'w') as fh:
        json.dump({'source': 'examples/{0}.py of yell/boltzmann-machines, run twice: {1}'.format(name, ' '.join(ARGS[name])),
                   'calls': rec.calls}, fh, indent=1)
    np.savez_compressed(os.path.join(HERE, 'example_{0}_trace.npz'.format(name)), **rec.arrays)
    print(name, len(rec.calls), 'calls,', len(rec.arrays), 'arrays')


if __name__ == '__main__':
    for n in ARGS:
        record(sys.argv[1], n)
