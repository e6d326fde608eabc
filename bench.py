#!/usr/bin/env python
"""Benchmarks of the hot path on N B200s of one node, one JSON line on stdout (rank 0).

    python bench.py --gpus N --steps K --warmup W                 # headline: BASELINE.json configs[1] (cfg2)
    python bench.py --config cfg3|cfg4|cfg4-ais|cfg5|cfg5-pcd      # the other BASELINE.json configurations
    python bench.py --impl reference [--config ...]                # the reference's CPU path (oracle restatement), host cores

cfg2      BernoulliRBM 784-1024, batch 4096 per GPU, CD-5               metric: Gibbs updates/s (batch x k)
cfg3      GaussianRBM 3072-5000, batch 2048, CD-1                        metric: Gibbs updates/s
cfg4      DBM 784-512-1024, batch = particles = 1024, <=25 mean-field updates, 1 PCD sweep   metric: batch rows/s
cfg4-ais  AIS on that DBM, 20000 runs x 1000 betas                       metric: chain transitions/s
cfg5      BernoulliRBM 784-4096, batch 4096 per GPU, 25 Gibbs steps (chains of the RBM engine, started at the data)
cfg5-pcd  the same shard as the reference runs PCD: its DBM class with ONE hidden layer (README.md:96), 4096 particles per GPU

A "step" = one full training step of the configuration (AIS: one whole ladder).  See DESIGN.md "Measurement" for every field.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, 'boltzmann-machines_b200')):
    if _p not in sys.path:
        sys.path.insert(0, _p)

# ---- the headline workload (kept as module constants: tools/ and tests/ import them) -------------------------
V, H, B, K_GIBBS = 784, 1024, 4096, 5
N_BATCHES = int(os.environ.get('BM_BENCH_BATCHES', '40'))    # resident dataset: 40 x 4096 rows = 257 MB of bf16 > 126 MB L2
#                                      (BM_BENCH_BATCHES: dry runs on the host simulation only -- `config.l2_policy` states the size)
LR, MOMENTUM, L2 = 0.05, 0.5, 1e-5
REFERENCE_BUDGET_S = float(os.environ.get('BM_BENCH_REFERENCE_SECONDS', '40'))   # --impl reference: timed + warm-up steps together
DUMP_BYTES = 64 * 2 ** 20                                     # --dump-outputs: at most this much in all
FLOP_PER_STEP = 2.0 * B * V * H * (2 * K_GIBBS + 3)      # SURVEY.md §8(d): (2k+3) GEMMs of 2BVH

RBM_WORKLOADS = {
    # name: (kind, V, H, batch, k, lr, W init stddev, resident batches, description)
    'cfg2': ('bernoulli', 784, 1024, 4096, 5, 0.05, 0.01, N_BATCHES,
             'BernoulliRBM 784-1024, batch 4096 per GPU, CD-5 (BASELINE.json configs[1])'),
    'cfg3': ('gaussian', 3072, 5000, 2048, 1, 5e-4, 0.0008, max(2, min(N_BATCHES, 12)),
             'GaussianRBM 3072-5000, batch 2048, CD-1 (BASELINE.json configs[2])'),
    'cfg5': ('bernoulli', 784, 4096, 4096, 25, 0.01, 0.01, N_BATCHES,
             'BernoulliRBM 784-4096, batch 4096 per GPU, 25 Gibbs steps per update (BASELINE.json configs[4], chains of the RBM '
             'engine started at the data; the persistent-particle variant is --config cfg5-pcd)'),
}
DBM_SHAPE = (784, [512, 1024], 1024)          # cfg4: V, hidden layers, batch = particles


def synth_mnist(n_rows, seed=1337, gibbs=30, n_vis=V):
    """Binary 'MNIST-shaped' data: samples of a random teacher RBM n_vis-64 with a 13% on-rate bias
    (SURVEY.md §8d), generated once for `base` rows and tiled."""
    rng = np.random.RandomState(seed)
    base = min(n_rows, 8192)
    Wt = (0.5 * rng.randn(n_vis, 64)).astype(np.float32)
    bt = np.float32(np.log(0.13 / 0.87))
    v = (rng.rand(base, n_vis) < 0.5).astype(np.float32)
    for _ in range(gibbs):
        h = (rng.rand(base, 64) < 1.0 / (1.0 + np.exp(-(v @ Wt)))).astype(np.float32)
        v = (rng.rand(base, n_vis) < 1.0 / (1.0 + np.exp(-(h @ Wt.T + bt)))).astype(np.float32)
    reps = (n_rows + base - 1) // base
    return np.ascontiguousarray(np.tile(v, (reps, 1))[:n_rows])


def synth_cifar(n_rows, n_vis=3072, seed=1338):
    """Real-valued 'CIFAR-shaped' data (SURVEY.md §8d): X = Z A + 0.3 E with a 64-dimensional latent, standardised per
    feature like examples/dbm_cifar_naive.py:358-371 does."""
    rng = np.random.RandomState(seed)
    base = min(n_rows, 4096)
    Z = rng.randn(base, 64).astype(np.float32)
    A = rng.randn(64, n_vis).astype(np.float32)
    X = Z @ A + 0.3 * rng.randn(base, n_vis).astype(np.float32)
    X = (X - X.mean(axis=0)) / (X.std(axis=0) + 1e-6)
    reps = (n_rows + base - 1) // base
    return np.ascontiguousarray(np.tile(X.astype(np.float32), (reps, 1))[:n_rows])


def model_cfg(compute='bf16', name='cfg2'):
    kind, v, h, b = RBM_WORKLOADS[name][:4]
    cfg = dict(n_visible=v, n_hidden=h, v_kind=kind, h_kind='bernoulli', dtype='float32',
               compute=compute, l2=L2, sample_v=False, sample_h=True, max_batch=b,
               sparsity_target=0.1, sparsity_cost=0.0, sparsity_damping=0.9)
    if kind == 'gaussian':
        cfg['sigma'] = np.ones(v)
    return cfg


def dbm_cfg(compute='bf16', n_hiddens=None, rows=None, n_visible=None, pcd_only=False):
    v, hs, b = DBM_SHAPE
    hs = list(n_hiddens or hs)
    b = rows or b
    v = n_visible or v
    L = len(hs)
    cfg = dict(compute=compute, n_visible=v, n_hiddens=hs, v_kind='bernoulli', h_kinds=['bernoulli'] * L, h_n_samples=[100.] * L,
               dtype='float32', n_particles=b, batch_size=b, max_mf_updates=25, mf_tol=1e-7, l2=1e-7, max_norm=6.0,
               sample_v=True, sample_h=[True] * L, sparsity_target=[0.2, 0.1][:L], sparsity_cost=[1e-4, 5e-5][:L],
               sparsity_damping=0.9)
    if pcd_only:                      # cfg5-pcd: one hidden layer, the positive phase is a single pass
        cfg.update(max_mf_updates=1, l2=1e-5, max_norm=1e9, sample_v=False, sparsity_cost=[0.0])
    return cfg


def dbm_params(cfg, seed=2, scale=0.02):
    rng = np.random.RandomState(seed)
    sizes = [cfg['n_visible']] + list(cfg['n_hiddens'])
    d = {'vb': np.zeros(sizes[0], np.float32)}
    for i in range(len(sizes) - 1):
        s = '' if i == 0 else '_%d' % i
        d['W' + s] = (scale * rng.randn(sizes[i], sizes[i + 1])).astype(np.float32)
        d['hb' + s] = np.zeros(sizes[i + 1], np.float32)
    return d


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons, one sample every 100 ms from before the warm-up to the end
    of the run; every sample is stamped on arrival and only those that fall inside a timed region
    (`mark()` ... `unmark()`) are reported, i.e. the median is a median UNDER LOAD."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
         'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, device):
        self.device, self.proc, self.samples, self.windows, self._t0 = device, None, [], [], None

    def start(self):
        import threading
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.device), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, bufsize=1)
        except OSError:
            self.proc = None
            return

        def pump():
            for line in self.proc.stdout:
                self.samples.append((time.perf_counter(), line))
        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def mark(self):
        self._t0 = time.perf_counter()

    def unmark(self):
        self.windows.append((self._t0, time.perf_counter()))

    def n_loaded(self):
        return sum(1 for t, _ in self.samples if any(a + 0.05 <= t <= b for a, b in self.windows))

    def stop(self):
        if not self.proc:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        self.thread.join(timeout=2)
        sm, mx, pw, reasons = [], [], [], set()
        names = ('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap')
        for t, line in self.samples:
            # a sample describes the 100 ms before it: require it to lie well inside a loaded window
            if not any(a + 0.05 <= t <= b for a, b in self.windows):
                continue
            f = [x.strip() for x in line.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            try:
                pw.append(float(f[3]))
            except ValueError:
                pass
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': float(np.median(sm)) if sm else None,
                'sm_max_mhz': float(max(mx)) if mx else None,
                'power_w_max': float(max(pw)) if pw else None,
                'samples': len(sm), 'reasons': sorted(reasons)}


def measured_peaks():
    """(burst TF/s, sustained TF/s, source).  The program kernel is timed inside a long step, but the steps measured here
    last a few milliseconds at full clocks -- the burst regime -- so `roofline.frac` is quoted against the BURST figure and
    `frac_sustained` beside it."""
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.isfile(p):
        with open(p) as fh:
            d = json.load(fh)
        burst = float(d.get('bf16_tflops', 1590.0))
        return burst, float(d.get('bf16_tflops_sustained', burst)), 'measured (MEASURED_PEAKS.json bf16_tflops / bf16_tflops_sustained)'
    return 1590.0, 1400.0, 'fallback (B200_PROFILING.md: 1.59 PFLOP/s burst, ~1.4 sustained)'


def recorded_traffic(kernel_key):
    """dram bytes per launch of the dominant kernel from the committed `ncu --set full` capture (profiles/...traffic.json states
    the commit it was taken at); None when this configuration has no capture."""
    p = os.path.join(ROOT, 'profiles', 'tc_program_kernel_traffic.json')
    if os.path.isfile(p):
        with open(p) as fh:
            d = json.load(fh)
        if kernel_key in d:
            return d[kernel_key]
        if kernel_key == 'cfg2':
            return d.get('dram_bytes_per_launch')
    return None


def dump_outputs(arrays, out_dir):
    """Writes each array as out_dir/<name>.npy.  Past DUMP_BYTES in all, every array keeps the same fraction of its rows, a fixed
    seeded sample, so that the files of two builds of the project compare element for element."""
    total = sum(a.nbytes for a in arrays.values())
    keep = min(1.0, DUMP_BYTES / total)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if keep < 1.0:
            a = a[np.sort(np.random.RandomState(0).choice(len(a), int(len(a) * keep), replace=False))]
        np.save(os.path.join(out_dir, name + '.npy'), a)


def blas_threads():
    try:
        from threadpoolctl import threadpool_limits
        return threadpool_limits
    except ImportError:
        return None


def time_cpu(step, n_steps, warmup, calibrate=True, threads=None):
    """Times `step(i)` (the oracle, numpy/OpenBLAS + C Philox) on the host cores.  OpenBLAS with every hardware thread of
    a 128-core host is several times SLOWER on these GEMMs than with a few dozen threads, so the BLAS pool size is calibrated
    first (one step per candidate) and the fastest setting is the one reported -- the CPU arm at its best."""
    limits = blas_threads()
    n_cpu = os.cpu_count() or 1
    threads = n_cpu
    tick = [0]

    def run(n, limit):
        t0 = time.perf_counter()
        for _ in range(n):
            if limits is not None:
                with limits(limits=limit, user_api='blas'):
                    step(tick[0])
            else:
                step(tick[0])
            tick[0] += 1
        return time.perf_counter() - t0

    if threads is not None:                       # pool size already calibrated by an earlier call
        run(warmup, threads)
        return run(n_steps, threads), threads
    run(max(1, warmup), n_cpu)
    if calibrate and limits is not None and n_cpu > 8:
        cands = sorted({c for c in (8, 16, 32, 64, n_cpu) if c <= n_cpu})
        times = {c: run(1, c) for c in cands}
        threads = min(times, key=times.get)
    dt = run(n_steps, threads)
    return dt, threads


# --------------------------------------------------------------------------------------------
# workloads: each returns a dict of callables / constants the driver below times
# --------------------------------------------------------------------------------------------
def rbm_config(name, world):
    """the `config` object of an RBM workload's JSON line -- the same in both arms (`--impl reference` prints this too)"""
    kind, v, h, b, k, lr, w_std, n_batches, descr = RBM_WORKLOADS[name]
    ldv = -(-(v + 2) // 64) * 64
    return {'workload': descr, 'parallelism': 'dp{0}'.format(world),
            'l2_policy': 'inputs larger than L2: resident dataset {0} MB bf16, batches cycle'.format(b * n_batches * ldv * 2 // 2 ** 20),
            'flop_per_step': 2.0 * b * v * h * (2 * k + 3), 'global_batch': b * world, 'k': k}


def rbm_workload(name, ctx, rank, world, compute):
    from boltzmann_machines import _native
    kind, v, h, b, k, lr, w_std, n_batches, descr = RBM_WORKLOADS[name]
    n_rows = b * n_batches
    X = synth_cifar(n_rows, v, seed=1338 + rank) if kind == 'gaussian' else synth_mnist(n_rows, seed=1337 + rank, n_vis=v)
    eng = _native.CudaRBM(model_cfg(compute, name), ctx=ctx)
    eng.init_normal_W(w_std, 1337)
    if kind != 'gaussian':
        # (data parallel: every replica starts from the same parameters -- the visible bias comes from rank 0's rows on every rank)
        X0 = X if rank == 0 else synth_mnist(8192, seed=1337, n_vis=v)
        p = np.clip(X0[:8192].mean(axis=0), 1e-7, 1 - 1e-7)
        eng.set_params({'vb': np.log(p / (1 - p)).astype(np.float32)})
    eng.set_data(X)
    seed = 20260922
    ldv = -(-(v + 2) // 64) * 64
    wl = dict(name=name, descr=descr, eng=eng, units_per_step=b * k, unit='updates/s', metric='gibbs_updates_per_sec',
              flop_per_step=2.0 * b * v * h * (2 * k + 3), n_batches=n_batches, batch=b,
              l2_policy='inputs larger than L2: resident dataset {0} MB bf16, batches cycle'.format(n_rows * ldv * 2 // 2 ** 20),
              cfg_extra={'global_batch': b * world, 'k': k},
              kernel='bm::tc_program_kernel<2>')
    wl['step'] = lambda i: eng.train_step_at((i % n_batches) * b, b, lr, MOMENTUM, k, seed, i)
    wl['outputs'] = eng.get_params                      # the trained variables: what the caller of a training step reads back

    def e2e_factory(kind_of_feed):
        # 'native': what fit() feeds for this data (bytes for binary data); 'float32': the same rows as grey levels --
        # real-valued data, which the bf16 engine takes as bfloat16 (half the reference's float32 feed_dict bytes)
        Xh = eng.pin(X) if kind_of_feed == 'native' else eng.pin(np.ascontiguousarray(X * np.float32(0.75)))

        def run(n_steps, t0):
            done = 0
            while done < n_steps:
                nb = min(n_batches, n_steps - done)
                eng.train_epoch(Xh[:nb * b], b, lr, MOMENTUM, k, seed, t0 + done, metrics=('msre',), every=1)
                done += nb
        return Xh, run
    wl['e2e_factory'] = e2e_factory
    wl['h2d_native'] = lambda Xh: b * v * Xh.dtype.itemsize * world
    wl['d2h'] = 64 * world

    def fit_e2e(n_steps, before_close=None):
        """The call a user of the library makes: Model(**kwargs).fit(X) on a HOST float32 array -- engine construction, weight
        initialisation, packing + page-locking of the training set, the epochs (every step uploads its own batch and reads its
        MSRE back) and the final save are all inside the timed region.  Exactly `n_steps` steps: whole epochs over the first
        `nb` batches of the dataset, `nb` the largest divisor of n_steps that it holds.  Returns (seconds, steps run, bytes up
        per step)."""
        import shutil
        import tempfile
        from boltzmann_machines.rbm import BernoulliRBM, GaussianRBM
        nb = max(d for d in range(1, min(n_batches, n_steps) + 1) if n_steps % d == 0)
        epochs = n_steps // nb
        tmp = tempfile.mkdtemp(prefix='bm_bench_fit_')
        kw = dict(n_visible=v, n_hidden=h, W_init=w_std, hb_init=0., n_gibbs_steps=k, learning_rate=lr, momentum=MOMENTUM,
                  max_epoch=epochs, batch_size=b, l2=L2, sample_v_states=False, sample_h_states=True,
                  metrics_config=dict(msre=True, pll=False, feg=False, l2_loss=False, train_metrics_every_iter=1),
                  verbose=False, save_after_each_epoch=False, random_seed=1337, dtype='float32', model_path=tmp + '/')
        if kind == 'gaussian':
            model = GaussianRBM(sigma=1., **kw)
        else:
            pm = np.clip(X0[:8192].mean(axis=0), 1e-7, 1 - 1e-7)
            model = BernoulliRBM(vb_init=np.log(pm / (1 - pm)).astype(np.float32), **kw)
        old = _native.Context._default.get(None)
        _native.Context._default[None] = ctx            # the model's engine lives on this rank's context (and communicator)
        # where the one-time costs go: wall time inside engine.pin (packing + page-locking) and the model saves
        from boltzmann_machines.base.native_model import NativeModel
        spent = {'pin': 0.0, 'save': 0.0}
        real_pin, real_save = _native.CudaRBM.pin, NativeModel._save_model

        def timed(key, fn):
            def wrapper(*a, **kw):
                t = time.perf_counter()
                try:
                    return fn(*a, **kw)
                finally:
                    spent[key] += time.perf_counter() - t
            return wrapper
        _native.CudaRBM.pin, NativeModel._save_model = timed('pin', real_pin), timed('save', real_save)
        try:
            t0 = time.perf_counter()
            model.fit(X[:nb * b])
            ctx.sync()
            dt = time.perf_counter() - t0
            fit_e2e.breakdown_ms = {'pack_and_pin_training_set': 1e3 * spent['pin'], 'model_saves': 1e3 * spent['save'],
                                    'everything_else (engine construction, init, epochs)': 1e3 * (dt - spent['pin'] - spent['save'])}
        finally:
            _native.CudaRBM.pin, NativeModel._save_model = real_pin, real_save
            # data parallel: the final save reads the other ranks' weight rows through peer memory -- every rank must have
            # finished reading before any rank frees its model (INTEGRATION.md, peer exchange)
            if before_close is not None:
                before_close()
            model.close() if hasattr(model, 'close') else None
            if old is None:
                _native.Context._default.pop(None, None)
            else:
                _native.Context._default[None] = old
            shutil.rmtree(tmp, ignore_errors=True)
        byte_valued = _native.as_bytes(X[:64]) is not None
        return dt, epochs * nb, b * v * (1 if byte_valued else 2)
    wl['fit_e2e'] = fit_e2e

    def quality():
        # held-out rows of the same generator: validation PLL / MSRE of the model as trained by the timed regions
        Xv = (synth_cifar(b, v, seed=99) if kind == 'gaussian' else synth_mnist(b, seed=99, n_vis=v))
        m = eng.metrics(Xv, 1, seed, 10 ** 6, ('msre', 'pll'))
        return {'val_msre': float(m['msre']), 'val_pll': float(m['pll'])}
    wl['quality'] = quality
    return wl


def dbm_workload(name, ctx, rank, world, compute, ais_runs, ais_betas):
    from boltzmann_machines import _native
    if name == 'cfg5-pcd':
        v, hs, b, k = 784, [4096], 4096, 25
        cfg = dbm_cfg(compute, hs, b, v, pcd_only=True)
        descr = ('BernoulliRBM 784-4096 as the reference runs PCD-25: its DBM class with one hidden layer (README.md:96), batch 4096 '
                 'and 4096 persistent particles per GPU (BASELINE.json configs[4])')
        lr = 0.01
    else:
        v, hs, b = DBM_SHAPE
        k = 1
        cfg = dbm_cfg(compute)
        descr = 'DBM 784-512-1024, batch = particles = 1024, <=25 mean-field updates, 1 PCD sweep (BASELINE.json configs[3])'
        lr = 2e-3
    eng = _native.CudaDBM(cfg, ctx=ctx)
    eng.set_params(dbm_params(cfg, scale=0.01 if name == 'cfg5-pcd' else 0.02))
    eng.init_particles(4242)
    n_batches = 8
    X = synth_mnist(b * n_batches, seed=1337 + rank, n_vis=v)
    Xpin = _native.pinned_copy(X)
    seed = 99
    if name == 'cfg4-ais':
        H1, H2 = hs
        flop = float(ais_runs) * (ais_betas - 1) * (4.0 * H1 * v + 4.0 * H1 * H2)          # SURVEY 8(d), fused count
        last = {}

        def step(i):
            last['logw'] = eng.ais(ais_runs, ais_betas, 1, 2222)
        wl = dict(name=name, descr='AIS on the DBM 784-512-1024: {0} runs x {1} betas, 1 Gibbs step per temperature '
                                   '(BASELINE.json configs[3])'.format(ais_runs, ais_betas),
                  eng=eng, units_per_step=ais_runs * (ais_betas - 1), unit='chain transitions/s',
                  metric='ais_chain_transitions_per_sec', flop_per_step=flop, n_batches=1, batch=ais_runs,
                  l2_policy='no input: every temperature rewrites the {0} MB of chain states and pre-activations (> L2)'.format(
                      ais_runs * (v + H1 + H2) * 6 // 2 ** 20),
                  cfg_extra={'n_runs': ais_runs, 'n_betas': ais_betas}, kernel='bm::tc_program_kernel<2>', step=step)
        wl['e2e_step'] = step                       # the call a user makes returns the log-weights to the host: same path
        wl['outputs'] = lambda: {'logw': last['logw']}
        wl['h2d'] = 0
        wl['d2h'] = 8 * ais_runs

        def quality():
            lw = last.get('logw')
            if lw is None:
                return {}
            return {'log_Z': float(np.logaddexp.reduce(lw) - np.log(len(lw)))}
        wl['quality'] = quality
        wl['sync_each_step'] = True
        return wl
    sizes = [v] + hs
    pairs = sum(sizes[i] * sizes[i + 1] for i in range(len(hs)))
    if name == 'cfg5-pcd':
        flop = 2.0 * b * v * hs[0] * (2 * k + 3 + 1)      # k sweeps, positive pass + its init pass, two gradient GEMMs
    else:
        H1, H2 = hs
        mf = 2.0 * b * (v * H1 + 2 * H1 * H2) * 25 + 2.0 * b * (v * H1 + H1 * H2)     # as written in the reference (SURVEY 8d)
        flop = mf + 2.0 * b * 2 * pairs + 2.0 * b * 2 * pairs
    nmf = {}

    def step(i):
        eng.train_step(Xpin[(i % n_batches) * b:(i % n_batches + 1) * b], lr, MOMENTUM, k, seed, i)

    def e2e_step(i):
        nmf.update(eng.train_step(Xpin[(i % n_batches) * b:(i % n_batches + 1) * b], lr, MOMENTUM, k, seed, i,
                                  metrics=('msre', 'n_mf_updates')))
    wl = dict(name=name, descr=descr, eng=eng, units_per_step=b * (k if name == 'cfg5-pcd' else 1),
              unit='updates/s' if name == 'cfg5-pcd' else 'rows/s',
              metric='gibbs_updates_per_sec' if name == 'cfg5-pcd' else 'dbm_train_rows_per_sec',
              flop_per_step=flop, n_batches=n_batches, batch=b,
              l2_policy='the DBM entry point takes host batches: every step uploads its batch (value and e2e differ by the '
                        'metric read-back only); weights + activations of a step: {0} MB'.format(
                            (4 * pairs * 3 + 2 * b * sum(sizes) * 6) // 2 ** 20),
              cfg_extra={'global_batch': b * world, 'k': k, 'max_mf_updates': cfg['max_mf_updates']},
              kernel='bm::tc_program_kernel<2>', step=step, e2e_step=e2e_step, outputs=eng.get_params)
    wl['h2d'] = b * v * 4 * world
    wl['d2h'] = 16 * world
    wl['quality'] = lambda: {key: float(val) for key, val in nmf.items()}
    return wl


# --------------------------------------------------------------------------------------------
# CPU side: the oracle (numpy + C Philox) timed on the host cores
# --------------------------------------------------------------------------------------------
def cpu_arm(name, n_steps, warmup, ais_runs, ais_betas, budget_s=None):
    """(value in the metric's unit, seconds per step, threads, sample description, quality dict).  `budget_s` (RBM workloads): run
    EXACTLY n_steps timed steps, each on as many rows of the batch as keeps the timed region near that many seconds -- a step is then
    a bounded sample of the workload's step (same model, same k, fewer rows), and the rate is rows * k / time as always."""
    n_cpu = os.cpu_count()
    if name in RBM_WORKLOADS:
        from oracle.rbm import OracleRBM
        kind, v, h, b, k, lr, w_std, _, _ = RBM_WORKLOADS[name]
        X = synth_cifar(b * 2, v) if kind == 'gaussian' else synth_mnist(b * 2, n_vis=v)
        ora = OracleRBM(model_cfg('fp32', name))
        rng = np.random.RandomState(0)
        ora.set_params({'W': (w_std * rng.randn(v, h)).astype(np.float32)})
        rows, pool = b, None
        if budget_s is not None:
            # one full step per BLAS pool size first (it is also the pool calibration); then the rows that fit the budget
            t_full, pool = time_cpu(lambda i: ora.train_step(X[:b], lr, MOMENTUM, k, 1, 10 ** 6 + i), 1, 1)
            rows = int(min(b, max(64, b * budget_s / (max(1, n_steps + warmup) * t_full)))) // 64 * 64
        dt, threads = time_cpu(lambda i: ora.train_step(X[(i % 2) * b:(i % 2) * b + rows], lr, MOMENTUM, k, 1, i), n_steps, warmup,
                               threads=pool)
        Xv = synth_cifar(b, v, seed=99) if kind == 'gaussian' else synth_mnist(b, seed=99, n_vis=v)
        m = ora.metrics(Xv, 1, 1, 10 ** 6, ('msre', 'pll'))
        q = {'val_msre': float(m['msre']), 'val_pll': float(m['pll']), 'train_steps': n_steps + max(1, warmup) + 4}
        sample = '{0} CD-{1} steps of batch {2} ({3}-{4}) on the oracle (numpy/OpenBLAS + C Philox)'.format(n_steps, k, b, v, h)
        if rows != b:
            sample = ('{0} CD-{1} steps on {5} rows each of the batch of {2} ({3}-{4}) on the oracle (numpy/OpenBLAS + C Philox): a '
                      'full step takes {6:.2f} s here, the sample keeps the run within its time budget').format(n_steps, k, b, v, h, rows, t_full)
        return n_steps * rows * k / dt, dt / n_steps, threads, sample, q
    from oracle.dbm import OracleDBM
    if name == 'cfg4-ais':
        cfg = dbm_cfg('fp32')
        ora = OracleDBM(cfg)
        ora.set_params(dbm_params(cfg))
        runs, betas = min(ais_runs, 400), min(ais_betas, 60)                    # bounded sample of the same ladder shape
        out = {}
        dt, threads = time_cpu(lambda i: out.update(lw=ora.ais(runs, betas, 1, 2222)), 1, 0, calibrate=False)
        lw = out['lw']
        q = {'log_Z_of_the_sample_ladder': float(np.logaddexp.reduce(lw) - np.log(len(lw)))}
        sample = 'one AIS ladder of {0} runs x {1} betas on the oracle (fp32 numpy/OpenBLAS + C Philox)'.format(runs, betas)
        return runs * (betas - 1) / dt, dt, threads, sample, q
    if name == 'cfg5-pcd':
        cfg = dbm_cfg('fp32', [4096], 4096, 784, pcd_only=True)
        k, lr = 25, 0.01
    else:
        cfg = dbm_cfg('fp32')
        k, lr = 1, 2e-3
    b, v = cfg['batch_size'], cfg['n_visible']
    ora = OracleDBM(cfg)
    ora.set_params(dbm_params(cfg, scale=0.01 if name == 'cfg5-pcd' else 0.02))
    ora.init_particles(4242)
    X = synth_mnist(b, n_vis=v)
    n_steps = max(1, min(n_steps, 3))
    dt, threads = time_cpu(lambda i: ora.train_step(X, lr, MOMENTUM, k, 99, i), n_steps, min(warmup, 1), calibrate=False)
    units = b * (k if name == 'cfg5-pcd' else 1)
    sample = '{0} training steps of batch {1} on the oracle (numpy/OpenBLAS + C Philox)'.format(n_steps, b)
    return n_steps * units / dt, dt / n_steps, threads, sample, {}


WORKLOAD_NAMES = ('cfg2', 'cfg3', 'cfg4', 'cfg4-ais', 'cfg5', 'cfg5-pcd')
METRICS = {'cfg4': ('dbm_train_rows_per_sec', 'rows/s'), 'cfg4-ais': ('ais_chain_transitions_per_sec', 'chain transitions/s')}


def run_reference(args):
    """The reference arm: the reference's own CPU path (oracle/ -- TF 1.3 / Python 2 cannot run in this image, DESIGN section 6) on
    the host cores, with the BLAS pool at its fastest size.  Same `config`, `metric`, `unit` as the b200 arm; RBM workloads run
    exactly --steps timed and --warmup untimed steps, each a bounded sample of the workload's step (cpu_arm)."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    note = 'TF1/py2 reference cannot run in this image; timed: oracle/ restatement of its CPU path'
    if args.config in RBM_WORKLOADS:
        steps, warm = max(1, args.steps), max(0, args.warmup)
        val, sec, cores, sample, quality = cpu_arm(args.config, steps, warm, args.ais_runs, args.ais_betas, budget_s=REFERENCE_BUDGET_S)
        config = rbm_config(args.config, args.gpus)
    else:
        steps = max(1, min(args.steps, 12))
        warm = max(1, min(args.warmup, 2))
        val, sec, cores, sample, quality = cpu_arm(args.config, steps, warm, args.ais_runs, args.ais_betas)
        config = {'workload': args.config}
    metric, unit = METRICS.get(args.config, ('gibbs_updates_per_sec', 'updates/s'))
    sample += '; BLAS pool {0} of {1} hardware threads'.format(cores, os.cpu_count())
    print(json.dumps({
        'impl': 'reference', 'metric': metric, 'value': val, 'unit': unit,
        'n_gpus': args.gpus, 'steps': steps, 'warmup': warm, 'ms_per_step': 1e3 * sec,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': config, 'note': note,
        'quality': quality,
        'cpu_baseline': {'value': val, 'unit': unit, 'cores': cores, 'kind': 'port', 'sample': sample},
        'e2e': {'value': val, 'unit': unit, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }))


# --------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=None)
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--impl', default='b200')
    ap.add_argument('--config', default='cfg2', choices=WORKLOAD_NAMES)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--compute', default='bf16')
    ap.add_argument('--ais-runs', type=int, default=20000)
    ap.add_argument('--ais-betas', type=int, default=1000)
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed step computed as DIR/<name>.npy (at most 64 MB: a fixed sample of larger outputs)')
    args = ap.parse_args()
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs: the reference arm times a sample of each step, not the outputs of the timed path')
    if args.steps is None:
        args.steps = {'cfg2': 2000, 'cfg3': 500, 'cfg5': 300, 'cfg5-pcd': 200, 'cfg4': 300, 'cfg4-ais': 3}[args.config]
    if args.impl == 'reference':
        return run_reference(args)
    args.warmup = max(args.warmup, 3)
    if args.config == 'cfg4-ais':
        args.warmup = min(args.warmup, 3)

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    dist = None
    if world > 1:
        import torch.distributed as dist            # plumbing only: rendezvous, barrier, max-reduce
        dist.init_process_group('gloo')

    from boltzmann_machines import _native
    ctx = _native.Context(local)
    if world > 1:
        uid = [_native.Context.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        ctx.comm_init(uid[0], rank, world)

    def barrier():
        ctx.sync()
        if dist is not None:
            dist.barrier()

    def max_over_ranks(x):
        if dist is None:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    if args.config in RBM_WORKLOADS:
        wl = rbm_workload(args.config, ctx, rank, world, args.compute)
    else:
        wl = dbm_workload(args.config, ctx, rank, world, args.compute, args.ais_runs, args.ais_betas)
    step = wl['step']
    units = wl['units_per_step']
    tick = [0]

    def run_steps(n, fn=None):
        fn = fn or step
        for _ in range(n):
            fn(tick[0])
            tick[0] += 1

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    run_steps(args.warmup)
    barrier()

    # ---- timed region 1: the hot path with its inputs where the engine keeps them (RBM: resident in HBM) -------------
    l0 = ctx.launch_count()
    barrier()
    sampler.mark()
    ctx.timer_start()
    run_steps(args.steps)
    ms = ctx.timer_stop()
    barrier()
    sampler.unmark()
    launches = ctx.launch_count() - l0
    ms = max_over_ranks(ms)
    value = args.steps * units * world / (ms * 1e-3)
    if args.dump_outputs:
        # read before the regions below train on; the other ranks wait, since the read may reach their weight rows
        if rank == 0:
            dump_outputs(wl['outputs'](), args.dump_outputs)
        barrier()

    # ---- region 2: same steps with per-launch CUDA events on the tensor-core kernel ---------------------------------
    ctx.profile_tc(True)
    sampler.mark()
    run_steps(args.steps if args.config != 'cfg4-ais' else 1)
    flops, tc_ms, tc_launches = ctx.profile_read()
    sampler.unmark()
    ctx.profile_tc(False)
    peak, peak_sustained, peak_src = measured_peaks()
    achieved = flops / (tc_ms * 1e-3) / 1e12 if tc_ms > 0 else 0.0

    # ---- region 3: end to end through the call a user of the library makes, HOST buffers in, result back -------------
    e2e = {}
    if 'e2e_factory' in wl:
        # RBM: bm_rbm_train_epoch[_u8] on the array BaseRBM._fit pinned with engine.pin -- every step uploads its own batch
        # from pinned host memory (double-buffered against the previous step's compute) and reads its MSRE back
        for key, feed in (('e2e', 'native'), ('e2e_float32', 'float32')):
            Xh, run = wl['e2e_factory'](feed)
            if key == 'e2e_float32' and 'e2e' in e2e and e2e['e2e']['feed_dtype'] != 'uint8':
                _native.pinned_free(np.asarray(Xh))
                continue                               # real-valued data: the native feed already is float32
            run(max(wl['n_batches'], args.warmup), tick[0]); tick[0] += max(wl['n_batches'], args.warmup)
            passes = []
            for _ in range(2):                         # two timed passes of exactly K steps; both are reported
                barrier()
                sampler.mark()
                ctx.timer_start()
                run(args.steps, tick[0]); tick[0] += args.steps
                t = ctx.timer_stop()
                barrier()
                sampler.unmark()
                passes.append(max_over_ranks(t))
            t = min(passes)
            e2e[key] = {'value': args.steps * units * world / (t * 1e-3), 'unit': wl['unit'],
                        'h2d_bytes_per_step': int(wl['h2d_native'](Xh)), 'd2h_bytes_per_step': wl['d2h'],
                        'ms_per_step': t / args.steps, 'timed_passes_ms_per_step': [x / args.steps for x in passes],
                        'reported': 'faster of two passes of K steps',
                        'feed_dtype': 'bfloat16' if isinstance(Xh, _native.Bf16Array) else str(Xh.dtype),
                        'path': 'bm_rbm_train_epoch{0} on a pinned host dataset (what BaseRBM._train_epoch calls), msre read back every '
                                'step'.format('_u8' if Xh.dtype == np.uint8 else '_bf16' if isinstance(Xh, _native.Bf16Array) else '')}
            _native.pinned_free(np.asarray(Xh))
        # the headline end-to-end number goes through the public API itself: Model(...).fit(X)
        e2e['e2e_epoch_call'] = e2e.pop('e2e')
        barrier()
        # fit() runs exactly K steps; its one-time costs (engine construction, packing and page-locking the training set, the
        # save: about 0.1 s for the 514 MB float32 set of 40 batches) weigh less the larger K is
        try:
            fit_s, fit_steps, up = wl['fit_e2e'](min(args.steps, 2 * wl['n_batches']), barrier)          # (warm: library loaded, CUDA context up)
            passes = []
            for _ in range(2):
                barrier()
                sampler.mark()
                fit_s, fit_steps, up = wl['fit_e2e'](args.steps, barrier)
                barrier()
                sampler.unmark()
                passes.append(max_over_ranks(fit_s))
            t = min(passes)
            e2e['e2e'] = {'value': fit_steps * units * world / t, 'unit': wl['unit'], 'h2d_bytes_per_step': int(up) * world,
                          'd2h_bytes_per_step': wl['d2h'], 'ms_per_step': 1e3 * t / fit_steps, 'steps': fit_steps,
                          'timed_passes_ms_per_step': [1e3 * x / fit_steps for x in passes], 'reported': 'faster of two fits',
                          'timing': 'host wall clock around fit() (+ device sync), max over ranks',
                          'fit_breakdown_ms_rank0_last_fit': getattr(wl['fit_e2e'], 'breakdown_ms', None),
                          'path': 'Model(**kwargs).fit(X) on a host float32 array, metrics_config msre every iteration: engine construction, '
                                  'weight init, packing + page-locking of the training set, the epochs (one native call each: per-step batch '
                                  'upload + msre read-back), final save -- all inside the timed region; e2e_epoch_call is the steady-state '
                                  'epoch call alone'}
        except Exception as exc:          # (every rank runs the same code on the same shapes: a failure here is common to all)
            sys.stderr.write('[bench] the fit() region failed ({0!r}); e2e falls back to the epoch-call measurement\n'.format(exc))
            e2e['e2e'] = dict(e2e['e2e_epoch_call'], fit_region_failed=repr(exc))
    else:
        n = args.steps
        passes = []
        for _ in range(2):
            barrier()
            sampler.mark()
            ctx.timer_start()
            run_steps(n, wl['e2e_step'])
            t = ctx.timer_stop()
            barrier()
            sampler.unmark()
            passes.append(max_over_ranks(t))
        t = min(passes)
        e2e['e2e'] = {'value': n * units * world / (t * 1e-3), 'unit': wl['unit'], 'h2d_bytes_per_step': wl['h2d'],
                      'd2h_bytes_per_step': wl['d2h'], 'ms_per_step': t / n, 'timed_passes_ms_per_step': [x / n for x in passes],
                      'reported': 'faster of two passes of K steps',
                      'path': 'the engine call the host mirror makes per step, pinned host batch in, metrics / log-weights back'}

    quality = wl['quality']() if 'quality' in wl else {}
    quality['train_steps'] = tick[0]

    # clock probe: when K is so small that no 100 ms sample fell inside a timed region, keep the
    # same load running (untimed) until a few samples exist -- same work, same clocks
    # (with peers every step is a collective: rank 0 decides, every rank runs the same number of probe steps)
    def rank0_says(flag):
        if dist is None:
            return flag
        box = [bool(flag) if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        return box[0]

    probe = 0
    if rank == 0:
        sampler.mark()
    t_end = time.perf_counter() + 3.0
    chunk = 50 if args.config != 'cfg4-ais' else 1
    while rank0_says(rank == 0 and sampler.n_loaded() < 5 and time.perf_counter() < t_end):
        run_steps(chunk)
        ctx.sync()
        if rank == 0:
            sampler.windows.append((sampler._t0, time.perf_counter()))
        probe += chunk
    clocks = None
    if rank == 0:
        clocks = sampler.stop()
        clocks['probe_steps_after_timed_regions'] = probe
    barrier()

    try:
        wl['eng'].close()            # (releases the peer-memory exchange; BM_PEER_PROFILE prints its averages here)
    except Exception:
        pass
    if rank != 0:
        return
    flop_step = wl['flop_per_step']
    step_tflops = flop_step * args.steps / (ms * 1e-3) / 1e12
    config = {'workload': wl['descr'], 'parallelism': 'dp{0}'.format(world), 'l2_policy': wl['l2_policy'],
              'flop_per_step': flop_step}
    config.update(wl['cfg_extra'])
    if args.config in RBM_WORKLOADS:
        config = rbm_config(args.config, world)      # (the same object the reference arm prints)
    out = {
        'metric': wl['metric'], 'value': value, 'unit': wl['unit'],
        'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms / args.steps,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'bf16' if args.compute == 'bf16' else 'f32', 'data': 'synthetic',
        'config': config,
        'gpu_launches': int(launches),
        'clocks': clocks,
        'roofline': {'bound': 'tensor', 'achieved': achieved, 'peak': peak, 'unit': 'TFLOP/s',
                     'frac': achieved / peak if peak else None,
                     'peak_sustained': peak_sustained, 'frac_sustained': achieved / peak_sustained if peak_sustained else None,
                     'traffic': recorded_traffic(args.config),
                     'kernel': wl['kernel'], 'launches': int(tc_launches), 'peak_source': peak_src,
                     'achieved_is': 'algorithmic FLOPs of the tensor-core launches / their CUDA-event time (region 2)',
                     'step_tflops': step_tflops, 'step_frac': step_tflops / peak, 'step_frac_sustained': step_tflops / peak_sustained},
        'quality': quality,
    }
    out.update(e2e)
    
    if world == 1 and not args.no_cpu_baseline:
        cpu_steps = {'cfg2': 8, 'cfg3': 3, 'cfg5': 2, 'cfg5-pcd': 1, 'cfg4': 3, 'cfg4-ais': 1}[args.config]
        val, sec, cores, sample, q = cpu_arm(args.config, cpu_steps, 1, args.ais_runs, args.ais_betas)
        out['cpu_baseline'] = {'value': val, 'unit': wl['unit'], 'cores': cores, 'kind': 'port',
                               'sample': sample + '; BLAS pool calibrated to its fastest size ({0} of {1} hardware threads)'.format(
                                   cores, os.cpu_count()), 'quality': q}
    print(json.dumps(out))


if __name__ == '__main__':
    main()
