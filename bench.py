#!/usr/bin/env python
"""Benchmark of the ciMRGP VI hot path (BASELINE.json: VI iterations/sec at N = 1e6, 10 resolutions; batched
Cholesky GFLOP/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

One "step" is one full variational sweep (`_fit()`, MRGP.py:571-652) over all 10 layers of the config-4 workload
(N = 1e6 samples, dx = 1, dy = 2, M = 30, 1023 regions, ci mode, fp64, static basis intervals).  Prints ONE JSON line.

GPU arm.  `value`: sweeps per second with everything resident in HBM, CUDA events on the engine's stream around every
step, L2 flushed (256 MB write) between steps, max over ranks.  `e2e`: the same sweep through the drop-in API with
NEW OBSERVATIONS every step at unchanged inputs: 16 MB of y copied from pinned host memory, the layer-0 statistics pass
over x and y, the sweep, the six ELBO terms per layer read back.  `roofline`: the streaming kernel that remains on the
path, k_ystats (24 B per sample), against the measured HBM peak; the steady-state sweep itself is ONE latency-bound
kernel (k_ci_sweep) that touches no sample (DESIGN.md §4), reported next to it.  `cpu_baseline` / `--impl reference`:
the multi-threaded C restatement of the sweep (oracle/mrgp_port.c, kind "port") on the host cores, at the FULL config
(no extrapolation), plus - when the reference itself travelled (oracle/_ref, bytecode compiled by build()) - one sweep of
the UNMODIFIED reference at config-3 size as the calibration.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np


def _finite(o):
    """JSON has no NaN / inf: map them to null."""
    if isinstance(o, dict):
        return {k: _finite(v) for k, v in o.items()}
    if isinstance(o, (list, tuple)):
        return [_finite(v) for v in o]
    if isinstance(o, (float, np.floating)):
        return float(o) if np.isfinite(o) else None
    if isinstance(o, np.integer):
        return int(o)
    return o


ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests', 'golden'))

N_SAMPLES = 1000000
N_LAYERS = 10
N_BASIS = 30
DY = 2
METRIC = 'ciMRGP VI iters/sec at N=1e6, R=10'
WORKLOAD = 'config4: synthetic 1-D nonstationary signal (script-1 f, seed 10), N=1e6, dx=1, dy=2, M=30, ' \
           '10 resolutions (1023 regions), ciMRGP, fp64, static basis intervals'
# the same `config` object on both arms (the driver compares them)
CONFIG = {'workload': WORKLOAD, 'l2': 'GPU arm: L2 flushed between timed steps (256 MB write); CPU arm: n/a'}
# algorithmic HBM bytes per sample-layer (SURVEY.md §8d): phase A 8(dx+2dy) = 40, phase B 8(dx+2dy+1) + 8(dy+1) = 72
BYTES_SWEEP_PER_SAMPLE_LAYER = 112
# --dump-outputs: the latent functions have one row per sample (240 MB at N = 1e6 over 10 layers); a fixed sample of
# DUMP_ROWS rows keeps the whole dump near 35 MB, under DUMP_BYTES
DUMP_ROWS = 1 << 17
DUMP_BYTES = 64 << 20


def engine_outputs(eng):
    """What a caller reads back after a sweep: every array of Engine.state() (per-layer posteriors, shared Bingham / ARD /
    omega state, latent functions) and the six ELBO terms per layer.  Per-sample arrays are cut to a seeded sample of rows,
    whose indices are returned as `latent_rows`."""
    rows = np.sort(np.random.RandomState(0).choice(eng.N, min(eng.N, DUMP_ROWS), replace=False))
    out = {k: v[rows] if k.endswith(('.fbar', '.fvar')) else v for k, v in eng.state(latent=True).items()}
    out['latent_rows'] = rows
    out['elbo'] = eng.elbo()
    return out


def dump_outputs(out_dir, arrays):
    """One float64 DIR/<name>.npy per array, so that two builds can be compared output for output."""
    arrays = {k: np.ascontiguousarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_BYTES:
        raise ValueError('outputs of %d bytes exceed the dump limit of %d' % (total, DUMP_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + '.npy'), v)


def peaks():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    except Exception:
        return 6650.0, 'fallback (B200_PROFILING.md)'


def ncu_traffic(kernel):
    """dram bytes per launch of `kernel` from the tracked ncu summary (profiles/r02_ncu_traffic.json), or None."""
    try:
        with open(os.path.join(ROOT, 'profiles', 'r02_ncu_traffic.json')) as f:
            return json.load(f).get(kernel)
    except Exception:
        return None


class ClockSampler(object):
    """SM clock and throttle reasons sampled DURING the timed region: NVML from a polling thread (one sample
    every ~2 ms; the timed region of this benchmark lasts tens of milliseconds, too short for `nvidia-smi -lms`),
    with the nvidia-smi one-shot query of B200_PROFILING.md as the fallback."""
    REASONS = (('hw_slowdown', 0x8), ('hw_thermal_slowdown', 0x40), ('sw_thermal_slowdown', 0x20), ('sw_power_cap', 0x4))

    def __init__(self, index):
        self.index, self.sm, self.mask, self.max_sm, self.stop_flag, self.thread, self.nvml = index, [], 0, None, False, None, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.dev = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.dev, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
        except Exception:
            self.nvml = None

    def _poll(self):
        nv = self.nvml
        while not self.stop_flag:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.dev, nv.NVML_CLOCK_SM)))
                get = getattr(nv, 'nvmlDeviceGetCurrentClocksEventReasons', None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
                self.mask |= int(get(self.dev))
            except Exception:
                pass
            time.sleep(0.002)

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.thread.join(timeout=2)
            return {'sm_mhz': float(np.median(self.sm)) if self.sm else None, 'sm_max_mhz': self.max_sm,
                    'reasons': [n for n, bit in self.REASONS if self.mask & bit], 'samples': len(self.sm), 'source': 'nvml'}
        try:
            q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
                'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
            out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + q, '--format=csv,noheader,nounits'],
                                 capture_output=True, text=True, timeout=10).stdout.strip().split(',')
            names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
            return {'sm_mhz': float(out[0]), 'sm_max_mhz': float(out[1]),
                    'reasons': [n for k, n in enumerate(names) if out[2 + k].strip() == 'Active'], 'samples': 1,
                    'source': 'nvidia-smi after the timed region'}
        except Exception:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvml and nvidia-smi unavailable'], 'samples': 0}


def make_model(n, layers, device, fi=False, distributed=False, n_basis=N_BASIS, seed=10):
    import workloads
    from cimrgp_b200 import IndexSetUniform, LaplacianEigenpairs, MaternKernel
    from cimrgp_b200.MRGP import MultiResolutionGaussianProcess
    x, y = workloads.workload1(n, seed=seed)
    return MultiResolutionGaussianProcess([x, y], n_basis, IndexSetUniform(n, layers - 1, 2), LaplacianEigenpairs(),
                                          MaternKernel(nu=1, l=1, sf=1), forced_independence=fi, device=device,
                                          distributed=distributed)


# ------------------------------------------------------------------------------------------------------------------
# CPU arms
# ------------------------------------------------------------------------------------------------------------------
def port_sweeps(n, layers, warmup, steps, dump=None):
    """The C restatement of the ci sweep (oracle/mrgp_port.c, OpenMP over all host threads) at FULL size n: seconds of
    each of `steps` sweeps after `warmup` sweeps, the threads it used, the seconds of its constructor.  dump: directory
    that receives the state after the last sweep."""
    import workloads
    from oracle import mrgp_oracle as O
    from oracle import port_c
    x, y = workloads.workload1(n)
    t0 = time.perf_counter()
    p = port_c.PortC(x, y, N_BASIS, O.uniform_offsets(n, layers - 1, 2))
    t_ctor = time.perf_counter() - t0
    p.sweep(warmup)
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        p.sweep(1)
        times.append(time.perf_counter() - t0)
    threads = p.threads
    if dump:
        dump_outputs(dump, p.state())
    p.close()
    return times, threads, t_ctor


class _BytecodeFinder(object):
    """Imports the reference's modules from their compiled bytecode under oracle/_ref/<name>.bytecode."""

    def __init__(self, path):
        self.path = path

    def find_spec(self, name, path=None, target=None):
        import importlib.machinery
        import importlib.util
        f = os.path.join(self.path, name + '.bytecode')
        if '.' in name or not os.path.exists(f):
            return None
        return importlib.util.spec_from_file_location(name, f, loader=importlib.machinery.SourcelessFileLoader(name, f))


def load_reference():
    """The UNMODIFIED reference: /root/reference/src in the build container, its bytecode under oracle/_ref (compiled by
    __graft_entry__.build(), git-ignored, travels with the snapshot) on the GPU box.  None when neither is there."""
    import types
    import warnings
    src, byt = '/root/reference/src', os.path.join(ROOT, 'oracle', '_ref')
    if os.path.exists(os.path.join(src, 'MRGP.py')):
        path = src
        if path not in sys.path:
            sys.path.insert(0, path)
    elif os.path.exists(os.path.join(byt, 'MRGP.bytecode')):
        path = byt
        sys.meta_path.insert(0, _BytecodeFinder(byt))
    else:
        return None
    import scipy.misc
    import scipy.special
    scipy.misc.logsumexp = scipy.special.logsumexp          # Stats.py:4
    for name in ('GPy', 'gpflow'):                           # RegressionInput.py:4-5 (only used with adaptive_inputs)
        sys.modules.setdefault(name, types.ModuleType(name))
    warnings.filterwarnings('ignore')
    mods = {name: __import__(name) for name in ('IndexSetGenerator', 'KernelClass', 'MRGP')}
    return types.SimpleNamespace(path=path, **mods)


def reference_calibration(n=100000, layers=8):
    """One `_fit()` of the unmodified reference at config-3 size (N = 1e5, 8 resolutions) next to the C port at the same
    size: how far the port is from the reference's own speed."""
    R = load_reference()
    if R is None:
        return {'available': False, 'why': 'neither /root/reference/src nor oracle/_ref is present on this host'}
    import workloads
    x, y = workloads.workload1(n)
    t0 = time.perf_counter()
    m = R.MRGP.MultiResolutionGaussianProcess(
        train_xy=[x, y], n_basis=N_BASIS, index_set_obj=R.IndexSetGenerator.IndexSetUniform(sample_length=n, resolution=layers - 1, divider=2),
        basis_function_obj=R.KernelClass.LaplacianEigenpairs(), spectral_density_obj=R.KernelClass.MaternKernel(nu=1, l=1, sf=1),
        adaptive_inputs=False, standard_normalized_inputs=True, basis_interval_obj=None, interval_factor=1, forced_independence=False)
    t_ctor = time.perf_counter() - t0
    t0 = time.perf_counter()
    m._fit()
    t_fit = time.perf_counter() - t0
    times, threads, _ = port_sweeps(n, layers, 1, 3)
    return {'available': True, 'kind': 'reference', 'source': R.path, 'workload': 'config3: N=1e5, 8 resolutions (255 regions), M=30, ci',
            'cores': 1, 'constructor_s': t_ctor, 's_per_sweep': t_fit, 'it_per_s': 1.0 / t_fit,
            'port_same_size': {'s_per_sweep': float(np.mean(times)), 'cores': threads},
            'port_speedup_over_reference': t_fit / float(np.mean(times))}


def run_reference(args, rank, world):
    """--impl reference: the CPU implementation of the path on the host cores, at the full config (rank 0 only)."""
    if rank != 0:
        return
    times, threads, t_ctor = port_sweeps(N_SAMPLES, N_LAYERS, args.warmup, args.steps, dump=args.dump_outputs)
    total = float(np.sum(times))
    value = args.steps / total
    calib = None if args.no_calibration else reference_calibration()
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': 'it/s', 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': 1e3 * total / args.steps, 'step_ms': [round(1e3 * t, 2) for t in times],
        'steps_timed': args.steps, 'extrapolated': False,
        'higher_is_better': True, 'scaling': 'weak' if world > 1 else 'strong', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': CONFIG,
        'cpu_baseline': {'value': value, 'unit': 'it/s', 'cores': threads, 'kind': 'port', 'host_cores': os.cpu_count(),
                         'sample': '%d full sweeps at the stated config (N=1e6, 10 layers, every layer streams its samples twice, as '
                                   'the reference does) of oracle/mrgp_port.c, OpenMP over %d threads; constructor %.1f s not '
                                   'included' % (args.steps, threads, t_ctor)},
        'e2e': {'value': value, 'unit': 'it/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'reference_unmodified': calib,
        'note': 'kind "port": the reference is single-threaded Python (295 s per sweep at this config in the survey container); '
                'its own speed is calibrated under reference_unmodified'
                + ('' if world == 1 else '; --gpus %d: the GPU arm runs %d independent models (one per GPU) - on the host they share the '
                   'same cores, so the aggregate CPU rate of %d models is the rate of one model on all cores, which is what is timed' % (world, world, world)),
    }
    print(json.dumps(_finite(line)))


# ------------------------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------------------------
def flush_l2(eng, flush, torch):
    """256 MB of HBM writes ON THE ENGINE'S STREAM: evicts L2 and keeps the GPU busy while the host queues the timed work
    behind it, so that the CUDA events around a step bracket device time only (no launch latency of an idle queue)."""
    with torch.cuda.stream(eng.stream):
        flush.zero_()


def timed_sweeps(eng, steps, flush, barrier, max_over_ranks, torch):
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    barrier()
    for k in range(steps):
        flush_l2(eng, flush, torch)       # stream order: after the previous timed sweep, before this one
        ev[k][0].record(eng.stream)
        eng.sweep(1)
        ev[k][1].record(eng.stream)
    barrier()
    return [max_over_ranks(a.elapsed_time(b)) for a, b in ev]


def time_call(eng, fn, flush, torch, reps):
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    torch.cuda.synchronize()
    for k in range(reps):
        if flush is not None:
            flush_l2(eng, flush, torch)
        else:
            eng.sweep(1)                  # keeps the queue busy (warm-L2 timing of back-to-back sweeps)
        ev[k][0].record(eng.stream)
        fn()
        ev[k][1].record(eng.stream)
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in ev]


def cholesky_grid(lib, torch, fp64_peak_tflops):
    """mrgp_batched_cholesky over n x batch: GFLOP/s (n^3 / 3 per matrix) and fraction of the measured FP64 peak."""
    import ctypes as C
    out = []
    rng = np.random.RandomState(0)
    for n in (2, 4, 8, 16, 32):
        for batch in (1000, 10000, 100000, 1000000):
            if n * n * batch * 8 > 2 ** 31:
                continue
            a = rng.randn(min(batch, 4096), n, n + 2)
            a = a @ np.swapaxes(a, 1, 2) + n * np.eye(n)
            base = torch.as_tensor(a, device='cuda')
            src = base.repeat((batch + base.shape[0] - 1) // base.shape[0], 1, 1)[:batch].contiguous()
            work = torch.empty_like(src)
            info = torch.zeros(batch, dtype=torch.int32, device='cuda')
            st = torch.cuda.current_stream()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            best = None
            for rep in range(4):
                work.copy_(src)
                e0.record(st)
                lib.mrgp_batched_cholesky(C.c_void_p(st.cuda_stream), C.c_void_p(work.data_ptr()), n, batch, C.c_void_p(info.data_ptr()))
                e1.record(st)
                e1.synchronize()
                t = e0.elapsed_time(e1)
                best = t if best is None or t < best else best
            gflops = (n ** 3 / 3.0) * batch / (best * 1e-3) / 1e9
            out.append({'n': n, 'batch': batch, 'ms': round(best, 4), 'gflops': round(gflops, 2),
                        'frac_fp64_peak': gflops / (fp64_peak_tflops * 1e3), 'gbs': round(2 * n * n * 8 * batch / (best * 1e-3) / 1e9, 1)})
    return out


def extras_single_gpu(args, torch, local_rank, flush):
    """BASELINE configs 3, 4 (fi) and 5 on the same GPU, short runs: it/s of a sweep, L2 flushed between timed sweeps."""
    out = {}

    def rate(m, steps=10, warm=4):
        eng = m._engine
        eng.sweep(warm)
        eng.synchronize()
        ms = timed_sweeps(eng, steps, flush, torch.cuda.synchronize, lambda v: v, torch)
        return {'it_per_s': steps / (sum(ms) / 1e3), 'ms_per_sweep': float(np.mean(ms)), 'ms_median': float(np.median(ms))}
    m = make_model(100000, 8, local_rank)
    out['config3_ci'] = dict(rate(m), workload='N=1e5, 8 resolutions (255 regions), M=30, ci')
    del m
    m = make_model(N_SAMPLES, N_LAYERS, local_rank, fi=True)
    r = rate(m, steps=8, warm=3)
    r['hbm_gbs_contract'] = BYTES_SWEEP_PER_SAMPLE_LAYER * N_SAMPLES * N_LAYERS / (r['ms_per_sweep'] * 1e-3) / 1e9
    r['workload'] = 'config 4 in fi mode: every layer streams its samples twice (112 B per sample-layer, SURVEY.md §8d)'
    out['config4_fi'] = r
    del m
    if args.config5_series > 0:
        out['config5'] = config5(args.config5_series, local_rank, torch)
    return out


def config5(n_series, device, torch, rank=0, world=1, n_iter=6, fi_series=1024):
    """Batch of independent series (N = 2048, 6 resolutions, M = 30): seconds per iteration of the whole batch."""
    import workloads
    from cimrgp_b200 import LaplacianEigenpairs, MaternKernel, SeriesBatch
    xs, ys = [], []
    lo, hi = (rank * n_series) // world, ((rank + 1) * n_series) // world
    for s in range(lo, hi):
        x, y = workloads.workload1(2048, seed=10 + s)
        xs.append(x)
        ys.append(y)
    res = {'series_total': n_series, 'series_this_rank': hi - lo, 'workload': 'N=2048, 6 resolutions (63 regions), M=30 per series',
           'fi_series_this_rank': min(hi - lo, max(1, fi_series // world))}
    for fi in (False, True):
        t0 = time.perf_counter()
        n_use = res['fi_series_this_rank'] if fi else hi - lo      # fi: a 1024-series sample of the batch (its cost is linear in the series)
        batch = SeriesBatch(xs[:n_use], ys[:n_use], N_BASIS, 5, LaplacianEigenpairs(), MaternKernel(nu=1, l=1, sf=1), forced_independence=fi,
                            device=device)
        t_build = time.perf_counter() - t0
        batch.fit(3)
        torch.cuda.synchronize()
        l0 = batch.launch_count()
        t0 = time.perf_counter()
        batch.fit(n_iter)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / n_iter
        res['fi' if fi else 'ci'] = {'series': n_use, 'ms_per_batch_iteration': 1e3 * dt, 'series_sweeps_per_s': n_use / dt,
                                     'launches_per_iteration': (batch.launch_count() - l0) / n_iter, 'build_s': t_build}
        batch.close()
        del batch
    return res


def measure_e2e(m, eng, steps, flush, barrier, max_over_ranks, torch, scale=1):
    """End to end through the public API: new observations from pinned host memory every step, statistics pass, sweep, ELBO
    terms back.  Two loops over the same work: (serial) upload, then compute, then read - the latency of one data set;
    (pipelined) the double-buffered upload of the API: the copy of step k + 1 is started before the sweep of step k, which
    reads no sample - the throughput of a stream of data sets, which is what `value` counts.  scale: models working in
    parallel (replicas, one per GPU)."""
    e2e_ms = []
    for k in range(steps):
        barrier()
        flush_l2(eng, flush, torch)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(eng.stream)
        eng.upload_observations()                      # H2D of this rank's rows of y (n, 2) from pinned memory
        m.fit(n_iter=1, tol=1e-300, min_iter=1)        # statistics pass + one sweep + the six ELBO terms per layer, read back
        b.record(eng.stream)
        b.synchronize()
        e2e_ms.append(max_over_ranks(a.elapsed_time(b)))
    # pipelined: ONE timed region around all K steps (L2 flushes included - nothing is subtracted); every step's copy,
    # statistics pass, sweep and read-back happen inside it
    # (three runs of K steps, the median run is reported and all three are listed: one timed region per run has no per-step
    # median to absorb a stall of the host - a 4-GPU run showed one run of 1.65 ms per step between two of 0.42 / 0.47)
    runs = []
    for rep in range(3):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        eng.synchronize()
        a.record(eng.stream)
        eng.prefetch_observations()                        # observations of step 0
        bounds = []
        for k in range(steps):
            flush_l2(eng, flush, torch)
            eng.refresh_statistics()                       # takes over set k: waits for its copy, statistics pass
            if k + 1 < steps:
                eng.prefetch_observations()                # copy of set k + 1 on the copy stream, beside the sweep of set k
            eng.sweep(1)                                   # one sweep ...
            eng.elbo_async(k & 1)                          # ... and its ELBO terms into pinned host memory
            if k > 0:
                bounds.append(eng.elbo_result((k - 1) & 1))   # the bound of step k - 1 is read while step k runs
        bounds.append(eng.elbo_result((steps - 1) & 1))
        b.record(eng.stream)
        b.synchronize()
        assert len(bounds) == steps and all(np.all(np.isfinite(v)) for v in bounds)
        runs.append(max_over_ranks(a.elapsed_time(b)) / steps)
    pipe_ms = float(np.median(runs))
    return {'value': scale * 1e3 / pipe_ms, 'unit': 'it/s', 'h2d_bytes_per_step': scale * eng.N * DY * 8,
            'd2h_bytes_per_step': scale * N_LAYERS * 6 * 8, 'ms_per_step': pipe_ms, 'ms_per_step_runs': [round(v, 4) for v in runs],
            'serial': {'value': scale * steps / (sum(e2e_ms) / 1e3), 'ms_per_step': float(np.mean(e2e_ms)),
                       'what': 'upload, statistics pass, sweep, read-back one after the other (L2 flush before each step, not timed)'},
            'what': 'new observations y every step at UNCHANGED inputs x (x-derived tables are reused; new inputs need the '
                    'basis rebuilt, include/cimrgp.h): y from pinned host memory through the double-buffered upload of the API '
                    '(mrgp_prefetch_observations_host: the copy of step k + 1 overlaps the sweep of step k, which reads no '
                    'sample), layer-0 statistics pass over x and y, one sweep, ELBO terms back (the terms of every step are read on the host, '
                    'one step late: mrgp_elbo_async / mrgp_elbo_wait); one timed region around all '
                    'steps of a run, the L2 flush of every step included; median of three runs',
            'lower_bound_layer0': m.lower_bound_layer[0][-1]}


def run_gpu(args, rank, world, local_rank):
    import ctypes as C
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    multi = world > 1
    if multi:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    # N > 1: one model per GPU (a series of its own per rank, same configuration): the steady-state ci sweep reads no sample,
    # so nothing of one model is left to shard (DESIGN.md §5) and independent series are the natural shard of the workload
    # (BASELINE config 5).  No data-path collective; barrier + max over ranks around the timed regions.  The SAMPLE-sharded
    # single model (statistics pass and uploads split over the GPUs, the sweep replicated) is measured after it and goes
    # into extras.sample_sharded.
    m = make_model(N_SAMPLES, N_LAYERS, local_rank, seed=10 + rank)
    eng = m._engine
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device='cuda')
    peak, peak_src = peaks()

    def barrier():
        torch.cuda.synchronize()
        if multi:
            dist.barrier()
            torch.cuda.synchronize()

    def max_over_ranks(v):
        if not multi:
            return v
        t = torch.tensor([v], dtype=torch.float64, device='cuda')
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    warm = max(args.warmup, 3)
    eng.sweep(warm)
    eng.synchronize()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # ---- device-resident timing -------------------------------------------------------------------------------
    l0 = eng.launch_count()
    step_ms = timed_sweeps(eng, args.steps, flush, barrier, max_over_ranks, torch)
    launches = eng.launch_count() - l0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, engine_outputs(eng))     # before the e2e loops sweep the model further
    total_s = sum(step_ms) / 1e3
    value = (world if multi else 1) * args.steps / total_s

    e2e = None if args.no_e2e else measure_e2e(m, eng, args.steps, flush, barrier, max_over_ranks, torch, scale=world if multi else 1)
    clocks = sampler.stop() if rank == 0 else None

    # ---- kernels -------------------------------------------------------------------------------------------------
    # k_ystats: the streaming pass of the path (per data set; every step of e2e).  Timed alone, L2 flushed before each launch.
    ys_ms = [max_over_ranks(v) for v in time_call(eng, eng.refresh_statistics, flush, torch, 7)]
    ys_med = float(np.median(ys_ms))
    ys_bytes = 24 * eng.N                                  # x (8) + y (16) per sample
    achieved = ys_bytes / (ys_med * 1e-3) / 1e9
    # k_ci_sweep: the whole steady-state sweep, warm L2 (back-to-back sweeps as in fit(n_iter))
    warm_ms = [max_over_ranks(v) for v in time_call(eng, lambda: eng.sweep(1), None, torch, 9)]
    sink = torch.zeros(8, dtype=torch.float64, device='cuda')
    ms = C.c_float()
    iters = 200000
    torch.cuda.synchronize()
    eng.lib.mrgp_fp64_probe(None, iters, C.c_void_p(sink.data_ptr()), C.byref(ms))
    sms = torch.cuda.get_device_properties(local_rank).multi_processor_count
    fp64_peak = sms * 4 * 256 * iters * 8 * 2 / (ms.value * 1e-3) / 1e12
    ys_flops = (3 * N_BASIS + 22 + 5) * 2 * eng.N          # per sample: recurrence M, Phi^T y 2M, sincospi 22, sums 5 (FMA = 2 flop)
    roofline = {
        'bound': 'hbm', 'kernel': 'k_ystats<2,30> (layer-0 sufficient statistics of y: the streaming kernel of the path)',
        'achieved': achieved * (world if multi else 1), 'peak': peak * (world if multi else 1), 'peak_source': peak_src, 'unit': 'GB/s',
        'frac': achieved / peak,
        'traffic': ncu_traffic('k_ystats'), 'traffic_source': 'ncu --set full, profiles/r02_ncu_traffic.json',
        'bytes_per_launch': ys_bytes, 'ms_per_launch': ys_med,
        'fp64': {'peak_tflops_measured': fp64_peak, 'achieved_tflops': ys_flops / (ys_med * 1e-3) / 1e12,
                 'frac': ys_flops / (ys_med * 1e-3) / 1e12 / fp64_peak},
        'sweep_kernel': {'kernel': 'k_ci_sweep<30> (one cluster of %s CTAs, all 10 layers)' % os.environ.get('MRGP_CHAIN_CLUSTER', '16'),
                         'ms_warm_l2': float(np.median(warm_ms)), 'ms_flushed_l2_median': float(np.median(step_ms)),
                         'traffic': ncu_traffic('k_ci_sweep'),
                         'note': 'latency-bound chain of small-matrix steps (Bingham, ARD, omega): no sample is read; the '
                                 '112 B per sample-layer of SURVEY.md §8d are not moved any more'},
    }
    if multi:
        line = None
        if rank == 0:
            line = {
                'metric': METRIC, 'value': value, 'unit': 'it/s', 'n_gpus': world, 'steps': args.steps, 'warmup': warm,
                'ms_per_step': 1e3 * total_s / args.steps, 'ms_per_step_median': float(np.median(step_ms)),
                'step_ms': [round(v, 4) for v in step_ms],
                'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
                'config': dict(CONFIG, parallelism='replicas only: %d independent series of the stated configuration, one model per '
                               'GPU, no data-path collective (value = models x sweeps / slowest rank). One model cannot use more '
                               'GPUs in the steady state: its sweep reads no sample; extras.sample_sharded has that arm' % world),
                'clocks': clocks, 'e2e': e2e, 'gpu_launches': launches * world, 'roofline': roofline, 'cpu_baseline': None,
            }
        # ---- the sample-sharded single model (strong scaling of ONE N = 1e6 problem) ---------------------------------
        sharded = None
        if not args.no_extras:
            eng.close()
            del m
            ms_ = make_model(N_SAMPLES, N_LAYERS, local_rank, distributed=True)
            es = ms_._engine
            es.sweep(warm)
            es.synchronize()
            st = timed_sweeps(es, 10, flush, barrier, max_over_ranks, torch)
            e2 = measure_e2e(ms_, es, 10, flush, barrier, max_over_ranks, torch)
            wm = [max_over_ranks(v) for v in time_call(es, lambda: es.sweep(1), None, torch, 9)]
            ysm = [max_over_ranks(v) for v in time_call(es, es.refresh_statistics, flush, torch, 7)]
            sharded = {'value': 10 / (sum(st) / 1e3), 'ms_per_step': float(np.mean(st)), 'e2e': {k: e2[k] for k in ('value', 'ms_per_step', 'serial')},
                       'h2d_bytes_per_step_per_gpu': es.N * DY * 8,
                       'amdahl': {'serial_us': 1e3 * float(np.median(wm)), 'statistics_pass_us': 1e3 * float(np.median(ysm)),
                                  'note': 'samples split into %d contiguous chunks (x, y never leave their GPU); the small-matrix sweep '
                                          'is replicated (serial_us); the sharded work is the statistics pass per data set with one '
                                          'exchange of 63 doubles over NVLink peer memory. Strong scaling of the sweep rate is flat by '
                                          'construction' % world}}
            eng = es
        extras = None
        if args.config5_series > 0 and not args.no_extras:
            torch.cuda.synchronize()
            c5 = config5(args.config5_series, local_rank, torch, rank=rank, world=world)
            # whole-job throughput: series of all ranks / slowest rank
            t = torch.tensor([c5['ci']['ms_per_batch_iteration'], c5['fi']['ms_per_batch_iteration']], dtype=torch.float64, device='cuda')
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            extras = {'config5_series_sharded': {'series_total': args.config5_series, 'ranks': world, 'collectives': 'none (replicas only)',
                                                 'ci_ms_per_batch_iteration': float(t[0]), 'ci_series_sweeps_per_s': args.config5_series / (float(t[0]) * 1e-3),
                                                 'fi_series': c5['fi']['series'] * world, 'fi_ms_per_batch_iteration': float(t[1]),
                                                 'fi_series_sweeps_per_s': c5['fi']['series'] * world / (float(t[1]) * 1e-3)}}
        if rank == 0:
            if extras is not None or sharded is not None:
                extras = dict(extras or {}, sample_sharded=sharded)
            line['extras'] = extras
            print(json.dumps(_finite(line)))
            sys.stdout.flush()
        barrier()
        eng.close()
        sys.stdout.flush()
        os._exit(0)

    cpu = None
    if not args.no_cpu_baseline:
        times, threads, t_ctor = port_sweeps(N_SAMPLES, N_LAYERS, 1, 5)
        cpu = {'value': 5 / float(np.sum(times)), 'unit': 'it/s', 'cores': threads, 'kind': 'port', 'host_cores': os.cpu_count(),
               'sample': '5 full sweeps at the stated config (N=1e6, 10 layers) of oracle/mrgp_port.c, OpenMP over %d threads, %.2f s per '
                         'sweep; not extrapolated' % (threads, float(np.mean(times)))}
    chol_total = eng.cholesky_count()
    omega_iters = [int(v) for v in eng.get(-1, 51, (N_LAYERS,))]
    extras = None if args.no_extras else extras_single_gpu(args, torch, local_rank, flush)
    grid = None if args.no_extras else cholesky_grid(eng.lib, torch, fp64_peak)
    line = {
        'metric': METRIC, 'value': value, 'unit': 'it/s', 'n_gpus': 1, 'steps': args.steps, 'warmup': warm,
        'ms_per_step': 1e3 * total_s / args.steps, 'ms_per_step_median': float(np.median(step_ms)),
        'ms_per_step_settled': float(np.mean(step_ms[len(step_ms) // 2:])),
        'step_ms': [round(v, 4) for v in step_ms],
        'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': CONFIG, 'clocks': clocks, 'e2e': e2e, 'gpu_launches': launches, 'roofline': roofline, 'cpu_baseline': cpu,
        'omega_iters_last_sweep': omega_iters,
        'batched_cholesky': {
            'in_sweep': {'n': DY, 'factorisations_per_sweep': N_BASIS * N_LAYERS,
                         'gflops': (DY ** 3 / 3.0) * N_BASIS * N_LAYERS / (float(np.median(step_ms)) * 1e-3) / 1e9,
                         'count_total': chol_total,
                         'note': 'the path has one Cholesky: the dy x dy PD test of the Bingham update (SanityCheck.py:59-65), M per '
                                 'layer in ci mode; it lives in registers inside k_ci_sweep and is < 1 % of a sweep'},
            'unit': 'GFLOP/s (n^3 / 3 per matrix)', 'fp64_peak_tflops_measured': fp64_peak, 'grid': grid},
        'extras': extras,
    }
    print(json.dumps(_finite(line)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-extras', action='store_true')
    ap.add_argument('--no-calibration', action='store_true')
    ap.add_argument('--config5-series', type=int, default=4096, help='series of the config-5 extra (BASELINE: 4096; fi mode runs on 1024 of them)')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write what the last timed step computed to DIR/<name>.npy (float64); '
                                                          'the inputs are seeded, so two builds can be compared file by file')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if args.impl == 'reference':
        run_reference(args, rank, world)
    else:
        run_gpu(args, rank, world, local_rank)


if __name__ == '__main__':
    main()
