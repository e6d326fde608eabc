"""TEST INFRASTRUCTURE: runs the reference's example scripts (examples/rbm_mnist.py, examples/dbm_mnist.py) UNCHANGED against
this repository's `boltzmann_machines` package.

The scripts are Python 2 (print statements, tuple parameters) and import Keras and an MNIST loader, none of which exist in
this image, so the runner
  * reads the script from the reference checkout (never copied into the repository) and rewrites, in memory, exactly the two
    Python-2 constructs the examples use -- `print x` statements and tuple parameters in `def` headers;
  * provides stand-ins for what is out of scope of the hot path (SURVEY.md section 8): `keras` (the MLP fine-tuning: fit is a
    no-op, predict is uniform), `boltzmann_machines.utils.dataset.load_mnist` (synthetic binary 'MNIST'), the Keras optimizer
    `MultiAdam`, and the examples' `env` path shim;
  * executes the script as `__main__` with the given command line.
Everything the script does with BernoulliRBM / DBM -- constructor keywords, fit, transform, load_model, load_rbms,
get_tf_params -- goes through the package under test.
"""
import ast
import os
import re
import sys
import types

import numpy as np


# ---- Python 2 -> 3, for the constructs the examples use ------------------------------------------------------------------
def _split_top_level(text):
    parts, depth, cur = [], 0, ''
    for ch in text:
        if ch in '([{':
            depth += 1
        elif ch in ')]}':
            depth -= 1
        if ch == ',' and depth == 0:
            parts.append(cur)
            cur = ''
        else:
            cur += ch
    if cur.strip():
        parts.append(cur)
    return parts


def translate(src):
    """`print x` -> `print(x)`; `def f((a, b), c):` -> `def f(_t0, c):` + `a, b = _t0` as the first statement."""
    out, lines, i = [], src.split('\n'), 0
    while i < len(lines):
        line = lines[i]
        m = re.match(r'^(\s*)print\s+(?!\()(.*\S)\s*$', line) or re.match(r'^(\s*)print\s+(\(.*\)\s*%.*|".*)$', line)
        if m and not line.lstrip().startswith('#'):
            out.append('{0}print({1})'.format(m.group(1), m.group(2)))
            i += 1
            continue
        if re.match(r'^\s*def\s+\w+\s*\(', line):
            header, j = line, i
            while header.count('(') != header.count(')') or not header.rstrip().endswith(':'):
                j += 1
                header += '\n' + lines[j]
            indent = re.match(r'^(\s*)', line).group(1)
            name, rest = re.match(r'^\s*def\s+(\w+)\s*\((.*)\)\s*:\s*$', header, flags=re.S).groups()
            args, unpack = [], []
            for a in _split_top_level(rest):
                a = a.strip()
                if a.startswith('('):
                    tmp = '_t{0}'.format(len(unpack))
                    unpack.append('{0}    {1} = {2}'.format(indent, a, tmp))
                    args.append(tmp)
                elif a:
                    args.append(a)
            out.append('{0}def {1}({2}):'.format(indent, name, ', '.join(args)))
            out.extend(unpack)
            i = j + 1
            continue
        out.append(line)
        i += 1
    return '\n'.join(out)


# ---- stand-ins ---------------------------------------------------------------------------------------------------------
def synthetic_mnist(n, seed):
    """binary 'digits' in 0 / 255 from a random 784-32 teacher RBM + labels derived from the hidden code"""
    rng = np.random.RandomState(seed)
    W = 0.6 * rng.randn(784, 32)
    h = (rng.rand(n, 32) < 0.5).astype(np.float64)
    p = 1.0 / (1.0 + np.exp(-(h @ W.T - 2.0)))
    X = (rng.rand(n, 784) < p).astype(np.float32) * 255.0
    y = (h[:, :4] @ np.array([1, 2, 4, 8])).astype(np.int64) % 10
    return X, y


def _stub_modules(n_train, n_test):
    mods = {}

    def mod(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        mods[name] = m
        return m

    class Layer(object):
        def __init__(self, *a, **kw):
            self.units = a[0] if a else None
            w = kw.get('weights')
            self._weights = [np.asarray(w[0]), np.asarray(w[1])] if w is not None else [np.zeros((1, 1)), np.zeros(1)]

        def get_weights(self):
            return self._weights

    class Sequential(object):
        def __init__(self, layers=()):
            self.layers = list(layers)

        def compile(self, *a, **kw):
            pass

        def fit(self, *a, **kw):
            print('[stand-in keras] MLP fine-tuning is out of scope: fit() skipped')

        def predict(self, X):
            return np.full((len(X), 10), 0.1)

    class Anything(object):
        def __init__(self, *a, **kw):
            pass

    keras = mod('keras')
    keras.regularizers = mod('keras.regularizers', l2=lambda *a, **kw: None)
    keras.callbacks = mod('keras.callbacks', EarlyStopping=Anything, ReduceLROnPlateau=Anything)
    keras.initializers = mod('keras.initializers', glorot_uniform=lambda *a, **kw: None)
    keras.models = mod('keras.models', Sequential=Sequential)
    keras.layers = mod('keras.layers', Dense=Layer, Activation=Layer)
    mod('env')

    def load_mnist(mode='train', path='.'):
        return synthetic_mnist(n_train if mode == 'train' else n_test, 7 if mode == 'train' else 8)
    mod('boltzmann_machines.utils.dataset', load_mnist=load_mnist)
    mod('boltzmann_machines.utils.optimizers', MultiAdam=Anything)
    return mods


def run_example(path, argv, n_train=640, n_test=128):
    """Executes the example at `path` as __main__ with command line `argv`.  Returns the script's globals."""
    src = open(path).read()
    py3 = translate(src)
    code = compile(py3, path, 'exec')
    stubs = _stub_modules(n_train, n_test)
    saved = {k: sys.modules.get(k) for k in stubs}
    old_argv = sys.argv
    sys.modules.update(stubs)
    sys.argv = [os.path.basename(path)] + list(argv)
    g = {'__name__': '__main__', '__file__': path, '__doc__': ast.get_docstring(ast.parse(py3))}
    try:
        exec(code, g)
    finally:
        sys.argv = old_argv
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    return g


# ---- what a script does with the package, recorded and replayed ---------------------------------------------------------
# the package names the examples import; a trace refers to them by name
ENTRY_POINTS = {'BernoulliRBM': ('boltzmann_machines.rbm', 'BernoulliRBM'), 'logit_mean': ('boltzmann_machines.rbm', 'logit_mean'),
                'DBM': ('boltzmann_machines', 'DBM')}


def summary(v):
    """what a call returned, as far as a trace keeps it: shape and dtype of arrays, through dicts, lists and tuples"""
    if isinstance(v, np.ndarray):
        return {'shape': list(v.shape), 'dtype': v.dtype.name}
    if isinstance(v, dict):
        return {k: summary(x) for k, x in sorted(v.items())}
    if isinstance(v, (list, tuple)):
        return [summary(x) for x in v]
    return None


class _Model(object):
    """a model the package returned to the script: its method calls are recorded"""

    def __init__(self, recorder, obj, index):
        self._recorder, self._obj, self._index = recorder, obj, index

    def __getattr__(self, name):
        attr = getattr(self._obj, name)
        if not callable(attr):
            return attr
        return lambda *a, **kw: self._recorder.call({'call': self._index}, name, attr, a, kw)


class _Entry(object):
    """an entry point of the package as the script imports it: calling it, or a class method of it, is recorded"""

    def __init__(self, recorder, name, real):
        self._recorder, self._name, self._real = recorder, name, real

    def __call__(self, *a, **kw):
        return self._recorder.call({'entry': self._name}, '__call__', self._real, a, kw)

    def __getattr__(self, attr):
        real = getattr(self._real, attr)
        return lambda *a, **kw: self._recorder.call({'entry': self._name}, attr, real, a, kw)


def _unwrap(v):
    if isinstance(v, _Model):
        return v._obj
    if isinstance(v, (list, tuple)):
        return type(v)(_unwrap(x) for x in v)
    if isinstance(v, dict):
        return {k: _unwrap(x) for k, x in v.items()}
    return v


class Recorder(object):
    """While active, the entry points of ENTRY_POINTS are wrappers that log every call into the package: the target (entry
    point, or the model an earlier call returned), the method, the arguments and a summary of the result.  Arguments that are
    results of earlier calls are referenced by call index, other arrays are kept in `arrays`, and paths are written relative to
    `workdir`."""

    def __init__(self, workdir):
        self.workdir, self.calls, self.arrays, self._results, self._saved = workdir, [], {}, [], []

    def __enter__(self):
        import importlib
        for name, (mod, attr) in ENTRY_POINTS.items():
            m = importlib.import_module(mod)
            self._saved.append((m, attr, getattr(m, attr)))
            setattr(m, attr, _Entry(self, name, getattr(m, attr)))
        return self

    def __exit__(self, *exc):
        for m, attr, real in self._saved:
            setattr(m, attr, real)

    def _encode(self, v):
        if isinstance(v, _Model):
            return {'call': v._index}
        if isinstance(v, np.ndarray):
            for i, r in enumerate(self._results):
                if isinstance(r, np.ndarray) and (r is v or (r.shape == v.shape and r.dtype == v.dtype and np.array_equal(r, v))):
                    return {'call': i}
            for key, a in self.arrays.items():
                if a.shape == v.shape and a.dtype == v.dtype and np.array_equal(a, v):
                    return {'array': key}
            key = 'a{0}'.format(len(self.arrays))
            self.arrays[key] = v.copy()
            return {'array': key}
        if isinstance(v, (list, tuple)):
            return {type(v).__name__: [self._encode(x) for x in v]}
        if isinstance(v, dict):
            return {'dict': {k: self._encode(x) for k, x in v.items()}}
        if isinstance(v, str):
            return v.replace(self.workdir, '{workdir}')
        if isinstance(v, np.generic):
            return v.item()
        if v is None or isinstance(v, (bool, int, float)):
            return v
        raise TypeError('a trace cannot hold an argument of type {0}'.format(type(v)))

    def call(self, target, method, fn, args, kwargs):
        rec = {'target': target, 'method': method, 'args': [self._encode(a) for a in args],
               'kwargs': {k: self._encode(v) for k, v in sorted(kwargs.items())}}
        out = fn(*_unwrap(args), **_unwrap(kwargs))
        rec['returned'] = summary(out)
        self.calls.append(rec)
        self._results.append(out)
        if type(out).__module__.startswith('boltzmann_machines'):
            return _Model(self, out, len(self.calls) - 1)
        return out


def replay(calls, arrays, workdir):
    """Makes the calls of a trace on the package, in order, and checks that each returns what it returned when recorded (shapes
    and dtypes of its arrays).  Returns every call's result."""
    import importlib
    results = []

    def decode(v):
        if isinstance(v, str):
            return v.replace('{workdir}', workdir)
        if not isinstance(v, dict):
            return v
        (tag, x), = v.items()
        if tag == 'call':
            return results[x]
        if tag == 'array':
            return arrays[x]
        if tag == 'dict':
            return {k: decode(y) for k, y in x.items()}
        return {'list': list, 'tuple': tuple}[tag](decode(y) for y in x)

    for c in calls:
        t = c['target']
        obj = getattr(importlib.import_module(ENTRY_POINTS[t['entry']][0]), ENTRY_POINTS[t['entry']][1]) if 'entry' in t else results[t['call']]
        fn = obj if c['method'] == '__call__' else getattr(obj, c['method'])
        out = fn(*[decode(a) for a in c['args']], **{k: decode(v) for k, v in c['kwargs'].items()})
        assert summary(out) == c['returned'], (len(results), c['method'], summary(out), c['returned'])
        results.append(out)
    return results
