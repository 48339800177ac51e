#!/usr/bin/env python
"""Benchmark of the sGDML hot paths on B200 (contract: see the task's bench.py section).

Metric (BASELINE.json): force predictions/s (the `value`) and K-assembly + solve wall-time
(the `train` object), on BASELINE config 2 -- synthetic aspirin, 21 atoms, 1000 training
points, 6 permutations, sigma 20 (SURVEY.md section 8d) -- unless --workload says otherwise.

A "step" is one pass of the prediction path over one batch of `--batch` synthetic query
geometries per GPU.  `value` times K steps with inputs resident in HBM; `e2e` times the same
steps through the public API ``GDMLPredict.predict`` with HOST buffers (pinned), host<->device
copies inside the timed region.  The training path (GDMLTrain.train: descriptors, assembly of
K in HBM, FP64 Cholesky, model, integration constant) runs once on rank 0 before the
prediction steps, produces the model they use, and is reported under `train`.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl engine|reference] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
"""

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (config key in sgdml_b200.synth.CONFIGS, BASELINE.json config it stands for)
    'aspirin': ('aspirin', 'configs[1]: aspirin 21 atoms, 1000 train, 6 perms (synthetic, SURVEY 8d)'),
    'ethanol': ('ethanol', 'configs[0]: ethanol 9 atoms, 200 train, 6 perms (synthetic, SURVEY 8d)'),
    # prediction only (random coefficients): training at this size needs the iterative solver
    'ac-ala3-nhme': ('ac-ala3-nhme', 'configs[2]: Ac-Ala3-NHMe 42 atoms, 2000 train, 243 perms, predict at batch 4096 (synthetic, SURVEY 8d)'),
    'synthetic100': ('synthetic100', 'configs[3]: synthetic 100-atom molecule, 5000 train, 12 perms, predict at batch 512 (synthetic, SURVEY 8d)'),
    'c60': ('c60', 'configs[4]: buckyball C60, 3000 train, 120 perms (I_h), predict at batch 256 (synthetic, SURVEY 8d)'),
}
PREDICT_ONLY = {'ac-ala3-nhme': 4096, 'synthetic100': 512, 'c60': 256}  # workload -> default batch


T0 = time.perf_counter()


def log(msg):
    sys.stderr.write('[bench %7.1fs] %s\n' % (time.perf_counter() - T0, msg))
    sys.stderr.flush()


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='engine', choices=['engine', 'reference'])
    ap.add_argument('--workload', default='aspirin', choices=sorted(WORKLOADS))
    ap.add_argument('--batch', type=int, default=65536, help='query geometries per GPU per step')
    ap.add_argument('--n-train', type=int, default=None, help='override the number of training points')
    ap.add_argument('--no-train', action='store_true', help='skip the training leg (random-coefficient model)')
    ap.add_argument('--cpu-seconds', type=float, default=15.0, help='target duration of the cpu_baseline sample')
    ap.add_argument('--no-cpu-baseline', action='store_true', help='skip the cpu_baseline leg (profiling runs)')
    ap.add_argument('--ref-batch', type=int, default=None, help='queries per step of the reference arm')
    ap.add_argument('--no-extras', action='store_true', help='skip the ethanol and sharded-path legs of the default run')
    ap.add_argument('--sharded-workload', default='c60', choices=['c60', 'synthetic100', 'ac-ala3-nhme'])
    ap.add_argument('--sharded-n-train', type=int, default=None)
    ap.add_argument('--sharded-batch', type=int, default=64, help='query geometries of the training-point-sharded predictor leg')
    ap.add_argument('--sharded-iters', type=int, default=3, help='PCG iterations timed in the sharded leg')
    ap.add_argument('--sharded-inducing', type=int, default=4096, help='columns of the (synthetic) Nystroem factor in the sharded leg')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last one returned (E.npy, F.npy; float64, a fixed seeded row '
                    'sample above %d MB) and the alphas_F of the timed training run (train_alphas_F.npy) to DIR'
                    % (DUMP_BYTES >> 20))
    ap.add_argument('--ref-torch-worker', default=None, help=argparse.SUPPRESS)  # internal: reference torch-CUDA arm
    ap.add_argument('--ref-worker', default=None, help=argparse.SUPPRESS)  # internal: JSON spec of a reference-arm subprocess
    ap.add_argument('--ref-train-worker', default=None, help=argparse.SUPPRESS)  # internal: reference training sample
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    return args


DUMP_BYTES = 64 << 20  # cap of everything --dump-outputs writes


def dump_outputs(out_dir, E, F, alphas_F=None):
    """Writes the prediction outputs E (B,), F (B, 3N) and, when the model was trained in this run, its alphas_F as
    float64 .npy files.  If they exceed DUMP_BYTES together, E and F are cut to the same fixed, seeded sample of rows
    (sorted), so that two builds run with the same arguments write comparable files."""
    os.makedirs(out_dir, exist_ok=True)
    E = E.detach().cpu().numpy()
    F = F.detach().cpu().numpy()
    arrays = {}
    budget = DUMP_BYTES - 3 * 4096  # room for the .npy headers
    if alphas_F is not None:
        arrays['train_alphas_F'] = np.asarray(alphas_F, dtype=np.float64)
        budget -= arrays['train_alphas_F'].nbytes
    rows = min(E.shape[0], budget // (8 * (1 + F.shape[1])))
    if rows < E.shape[0]:
        keep = np.sort(np.random.default_rng(0).choice(E.shape[0], size=rows, replace=False))
        E, F = E[keep], F[keep]
    arrays['E'], arrays['F'] = E, F
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), np.ascontiguousarray(a, dtype=np.float64))
    log('outputs written to %s: %s' % (out_dir, ', '.join('%s %s' % (k, a.shape) for k, a in arrays.items())))


# --------------------------------------------------------------------------- clocks
class ClockSampler(object):
    """Samples nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    Q = (
        'index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
        'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
        'clocks_event_reasons.sw_power_cap'
    )

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '-i', str(self.gpu_index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits', '-lms', '100'],
                stdout=subprocess.PIPE,
                stderr=subprocess.DEVNULL,
                text=True,
            )
            self.thread = threading.Thread(target=self._reader, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _reader(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            f = [x.strip() for x in r.split(',')]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for nm, val in zip(names, f[4:8]):
                if val.lower().startswith('active'):
                    reasons.add(nm)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no samples']}
        # "under load": samples in the upper half of the observed power range
        thr = 0.5 * (max(power) + min(power))
        load = [s for s, p in zip(sm, power) if p >= thr] or sm
        return {
            'sm_mhz': float(np.median(load)),
            'sm_max_mhz': float(max(smax)),
            'power_w_max': float(max(power)),
            'samples': len(sm),
            'reasons': sorted(reasons),
        }


# --------------------------------------------------------------------------- workload
def workload_cfg(args):
    from sgdml_b200 import synth

    cfg = dict(synth.CONFIGS[WORKLOADS[args.workload][0]])
    if args.n_train is not None:
        cfg['n_train'] = args.n_train
    cfg['name'] = WORKLOADS[args.workload][0]
    return cfg


def algorithmic_flops_per_query(cfg, S):
    N = cfg['n_atoms']
    D = N * (N - 1) // 2
    return 9.0 * cfg['n_train'] * S * D  # SURVEY.md 8d: W_P = 9 M S D


# --------------------------------------------------------------------------- reference arm (CPU)
def oracle_random_model(cfg, perms):
    """Random-coefficient model of the workload's shape built with the ORACLE (CPU) code:
    prediction cost does not depend on the coefficient values."""
    from oracle import desc as odesc
    from sgdml_b200 import synth

    N, M = cfg['n_atoms'], cfg['n_train']
    R = synth.geometries(N, M, 0, r0=synth.config_perms_and_r0(cfg['name'])[1]).reshape(M, -1)
    rng = np.random.default_rng(99)
    alphas = rng.standard_normal(M * 3 * N)
    x, g = odesc.from_R(R)
    return {
        'type': 'm',
        'z': np.ones(N, dtype=np.int64),
        'R_desc': x.T.copy(),
        'R_d_desc_alpha': odesc.d_desc_dot_vec(g, alphas.reshape(M, -1)),
        'alphas_F': alphas,
        'c': 0.0,
        'std': 1.0,
        'sig': cfg['sig'],
        'lam': 1e-10,
        'perms': perms,
        'tril_perms_lin': odesc.tril_perms_lin(perms),
        'use_E': True,
    }


def cpu_workers(cfg, n_perms):
    """Worker processes of the CPU arm: all host threads, unless the per-worker permuted caches
    (2 * M*S*D doubles, predict.py:426-441) would not fit in ~128 GB of host memory together."""
    cores = os.cpu_count() or 1
    D = cfg['n_atoms'] * (cfg['n_atoms'] - 1) // 2
    cache = 2.0 * cfg['n_train'] * n_perms * D * 8
    return int(max(1, min(cores, 128e9 // cache)))


class CpuPredictor(object):
    """The CPU arm: oracle port of predict.py:84-245 on a persistent pool over the host threads."""

    def __init__(self, model, cfg, n_procs):
        from oracle import predict as opredict

        self.cfg = cfg
        self.pp = opredict.ParallelPredictor(model, n_procs)

    def rate(self, n_queries, seed=1):
        from sgdml_b200 import synth

        r0 = synth.config_perms_and_r0(self.cfg['name'])[1]
        Rq = synth.geometries(self.cfg['n_atoms'], n_queries, seed, r0=r0).reshape(n_queries, -1)
        t0 = time.perf_counter()
        self.pp.predict(Rq)
        return n_queries / (time.perf_counter() - t0)

    def close(self):
        self.pp.close()


# The UNMODIFIED reference (stefanch/sGDML v1.0.3) lives in baseline/_ref when it was installed in the
# build container (git-ignored, but it travels to the GPU box with the snapshot).  It is run in a fresh
# interpreter: its worker pool forks (predict.py:36), which must not happen in a process that has
# initialised CUDA or torch's thread pools.
REF_DIR = os.path.join(ROOT, 'baseline', '_ref')


def reference_available():
    if os.environ.get('SGDML_B200_NO_REFERENCE'):  # tests: force the oracle-port fallback
        return False
    return os.path.isfile(os.path.join(REF_DIR, 'sgdml', 'predict.py'))


def ref_worker_main(spec):
    """Runs inside the subprocess: GDMLPredict(model, use_torch=False) of the reference, its own process
    pool over the host threads in bulk mode (predict.py:1236-1256); prints one JSON line."""
    import logging

    sys.path.insert(0, REF_DIR)
    from sgdml.predict import GDMLPredict  # the reference, not this repo

    from sgdml_b200 import synth

    cfg = spec['cfg']
    perms, r0 = synth.config_perms_and_r0(cfg['name'])
    model = oracle_random_model(cfg, perms)
    N = cfg['n_atoms']
    cores = int(spec['cores'])
    pred = GDMLPredict(model, max_processes=cores, use_torch=False, log_level=logging.CRITICAL)

    def rate(n_queries, seed):
        Rq = synth.geometries(N, n_queries, seed, r0=r0).reshape(n_queries, -1)
        t0 = time.perf_counter()
        pred.predict(Rq)
        return n_queries / (time.perf_counter() - t0)

    # The reference tunes (bulk mode, workers, chunk size) with prepare_parallel (predict.py:776-1044), whose
    # run time is unbounded on a many-core host; the same three knobs are set here through the same setters
    # from a short list, keeping the fastest.
    pred._set_bulk_mp(True)
    pred._set_num_workers(max(cores - 1, 1))
    best = (0.0, None)
    n_probe = max(2 * cores, 64)
    rate(n_probe, 3)  # spin the pool up
    for chunk in [None, 256, 64, 16]:
        if chunk is not None and chunk >= cfg['n_train']:
            continue
        pred._set_chunk_size(chunk)
        r = rate(n_probe, 5)
        if r > best[0]:
            best = (r, chunk)
    pred._set_chunk_size(best[1])
    per_step = int(spec['per_step'] or max(cores, min(200000, best[0] * float(spec['seconds_per_step']))))
    for _ in range(int(spec['warmup'])):
        rate(per_step, 7)
    t0 = time.perf_counter()
    for k in range(int(spec['steps'])):
        rate(per_step, 11 + k)
    dt = time.perf_counter() - t0
    # parity of the arm itself: the reference against this repo's oracle on a few queries
    from oracle import predict as opredict

    Rq = synth.geometries(N, 4, 1, r0=r0).reshape(4, -1)
    _, F_ref = pred.predict(Rq)
    _, F_orc = opredict.Predictor(model).predict(Rq)
    dev = float(np.max(np.abs(F_ref - F_orc)) / np.max(np.abs(F_orc)))
    print(json.dumps({'per_step': per_step, 'steps': int(spec['steps']), 'seconds': dt, 'chunk_size': best[1],
                      'workers': int(pred.num_workers), 'oracle_vs_reference_rel': dev}))
    sys.stdout.flush()
    os._exit(0)  # the reference's pool has no clean shutdown path (predict.py:462-470)


def ref_train_worker_main(spec):
    """Runs inside a subprocess: the reference's training path on a BOUNDED sample (SURVEY.md section 8d).
    part 'assemble': GDMLTrain._assemble_kernel_mat (train.py:1260-1535) for the first k block-columns, its
    own process pool over the host threads; part 'cholesky': scipy.linalg.cho_factor + cho_solve
    (analytic.py:94-99) at a reduced n.  The caller scales by M/k and (n/n_s)^3."""
    sys.path.insert(0, REF_DIR)
    from sgdml_b200 import synth

    cfg = spec['cfg']
    N, M = cfg['n_atoms'], cfg['n_train']
    if spec['part'] == 'assemble':
        from sgdml.train import GDMLTrain
        from sgdml.utils.desc import Desc

        cores = int(spec['cores'])
        perms, r0 = synth.config_perms_and_r0(cfg['name'])
        R = synth.geometries(N, M, 0, r0=r0).reshape(M, -1)
        desc = Desc(N, max_processes=cores)
        t0 = time.perf_counter()
        R_desc, R_d_desc = desc.from_R(R, max_processes=cores)
        t_desc = time.perf_counter() - t0
        tril_perms = np.array([Desc.perm(p) for p in perms])
        tril_perms_lin = (tril_perms + np.arange(len(perms))[:, None] * desc.dim).flatten('F')
        gdml = GDMLTrain(max_processes=cores, use_torch=False)
        k, t = 1, 0.0
        k_max = max(1, min(M, int(4e9 / (8.0 * 3 * N * M * 3 * N))))  # the host copy of the sampled columns stays below 4 GB
        while True:  # grow the sample until it takes a few seconds
            t0 = time.perf_counter()
            gdml._assemble_kernel_mat(R_desc, R_d_desc, tril_perms_lin, cfg['sig'], desc, col_idxs=np.s_[: k * 3 * N])
            t = time.perf_counter() - t0
            if t >= float(spec['seconds']) or k >= k_max:
                break
            k = min(k_max, max(k + 1, int(k * min(8.0, 1.3 * float(spec['seconds']) / max(t, 1e-3)))))
        print(json.dumps({'col_points': k, 'seconds': t, 'desc_seconds': t_desc, 'workers': cores}))
    else:
        import scipy.linalg

        n_s = int(spec['n_sample'])
        rng = np.random.default_rng(0)
        A = rng.standard_normal((n_s, n_s))
        A = A @ A.T + n_s * np.eye(n_s)
        y = rng.standard_normal(n_s)
        t0 = time.perf_counter()
        L, lower = scipy.linalg.cho_factor(A, overwrite_a=True, check_finite=False)  # analytic.py:94-96
        scipy.linalg.cho_solve((L, lower), y, overwrite_b=True, check_finite=False)  # analytic.py:97-99
        print(json.dumps({'n_sample': n_s, 'seconds': time.perf_counter() - t0}))
    sys.stdout.flush()
    os._exit(0)


def reference_train_estimate(cfg, cores, seconds=6.0):
    """CPU time of the reference's K assembly + Cholesky solve for this workload, EXTRAPOLATED from bounded
    samples run with the unmodified reference (None if it is not installed)."""
    if not reference_available():
        return None
    N, M = cfg['n_atoms'], cfg['n_train']
    n = 3 * N * M
    out = {}
    for part, threads in (('assemble', '1'), ('cholesky', None)):
        spec = {'cfg': cfg, 'cores': cores, 'part': part, 'seconds': seconds, 'n_sample': min(n, 12000)}
        env = dict(os.environ)
        for k in ('OMP_NUM_THREADS', 'OPENBLAS_NUM_THREADS', 'MKL_NUM_THREADS'):
            if threads is None:
                env.pop(k, None)  # LAPACK on all the threads it wants
            else:
                env[k] = threads  # pool of single-threaded workers
        env['CUDA_VISIBLE_DEVICES'] = ''
        for k in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK'):
            env.pop(k, None)
        try:
            res = subprocess.run([sys.executable, os.path.abspath(__file__), '--ref-train-worker', json.dumps(spec)],
                                 env=env, capture_output=True, text=True, timeout=90 + 10 * seconds)
            out[part] = json.loads(res.stdout.strip().splitlines()[-1])
        except Exception as e:  # noqa: BLE001 -- a reported baseline must never take the benchmark down
            log('reference training sample (%s) failed: %r' % (part, e))
            return None
    a, c = out['assemble'], out['cholesky']
    assemble_s = a['seconds'] * M / a['col_points']
    solve_s = c['seconds'] * (n / c['n_sample']) ** 3
    return {
        'kind': 'reference',
        'extrapolated': True,
        'cores': cores,
        'assemble_s': assemble_s,
        'solve_s': solve_s,
        'total_s': assemble_s + solve_s,
        'sample': 'unmodified reference: GDMLTrain._assemble_kernel_mat on the first %d of %d block-columns (%.1f s, %d worker '
        'processes) scaled by M/k; scipy cho_factor + cho_solve at n = %d (%.2f s, LAPACK threads unrestricted) scaled by (n/n_s)^3'
        % (a['col_points'], M, a['seconds'], a['workers'], c['n_sample'], c['seconds']),
    }


def ref_torch_worker_main(spec):
    """Runs inside a subprocess WITH the GPU visible: the reference's own torch engine on CUDA --
    GDMLPredict(model, use_torch=True).predict (predict.py:358-421, torchtools.py:877-1128; inputs are downcast to
    float32 by the reference itself, predict.py:1197-1201, the model stays float64) and GDMLTorchAssemble through
    GDMLTrain(use_torch=True)._assemble_kernel_mat (train.py:1412-1482, torchtools.py:110-392) on a bounded number
    of block-columns.  Prints one JSON line."""
    import logging

    sys.path.insert(0, REF_DIR)
    import torch

    from sgdml_b200 import synth

    cfg = spec['cfg']
    perms, r0 = synth.config_perms_and_r0(cfg['name'])
    N, M = cfg['n_atoms'], cfg['n_train']
    out = {'device': torch.cuda.get_device_name(0) if torch.cuda.is_available() else 'cpu'}
    try:
        from sgdml.predict import GDMLPredict  # the reference, not this repo

        model = oracle_random_model(cfg, perms)
        pred = GDMLPredict(model, use_torch=True, log_level=logging.CRITICAL)
        Bq = int(spec['batch'])
        Rq = synth.geometries(N, Bq, 1, r0=r0).reshape(Bq, -1)
        pred.predict(Rq)  # warm-up (its own batch-size back-off happens here)
        torch.cuda.synchronize()
        n_done, t0 = 0, time.perf_counter()
        while time.perf_counter() - t0 < float(spec['seconds']):
            E, F = pred.predict(Rq)
            n_done += Bq
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        from oracle import predict as opredict

        _, F_orc = opredict.Predictor(model).predict(Rq[:4])
        out['predict'] = {'value': n_done / dt, 'unit': 'predictions/s', 'batch': Bq, 'seconds': dt,
                          'rel_dev_from_f64_oracle': float(np.max(np.abs(F[:4] - F_orc)) / np.max(np.abs(F_orc)))}
    except Exception as e:  # noqa: BLE001
        out['predict'] = {'unavailable': repr(e)[:300]}
    try:
        from sgdml.train import GDMLTrain
        from sgdml.utils.desc import Desc

        R = synth.geometries(N, M, 0, r0=r0).reshape(M, -1)
        desc = Desc(N, max_processes=1)
        R_desc, R_d_desc = desc.from_R(R, max_processes=1)
        tril_perms = np.array([Desc.perm(p) for p in perms])
        tril_perms_lin = (tril_perms + np.arange(len(perms))[:, None] * desc.dim).flatten('F')
        gdml = GDMLTrain(max_processes=1, use_torch=True)
        k = max(1, min(M, int(spec['col_points'])))
        gdml._assemble_kernel_mat(R_desc, R_d_desc, tril_perms_lin, cfg['sig'], desc, col_idxs=np.s_[: 3 * N])  # warm-up
        t0 = time.perf_counter()
        gdml._assemble_kernel_mat(R_desc, R_d_desc, tril_perms_lin, cfg['sig'], desc, col_idxs=np.s_[: k * 3 * N])
        dt = time.perf_counter() - t0
        out['assemble'] = {'col_points': k, 'seconds': dt, 'extrapolated_full_s': dt * M / k}
    except Exception as e:  # noqa: BLE001
        out['assemble'] = {'unavailable': repr(e)[:300]}
    print(json.dumps(out))
    sys.stdout.flush()
    os._exit(0)


def reference_torch_cuda(cfg, gpu_index, seconds=5.0):
    """The reference's own torch-CUDA path timed on this B200 (BASELINE.md section 3, SURVEY 8d "existing GPU
    implementation" bar); None if the reference is not installed, {'unavailable': why} if it cannot run."""
    if not reference_available():
        return None
    spec = {'cfg': cfg, 'batch': 1024, 'seconds': seconds, 'col_points': 16}
    env = dict(os.environ)
    env['CUDA_VISIBLE_DEVICES'] = str(gpu_index)
    for k in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK'):
        env.pop(k, None)
    try:
        res = subprocess.run([sys.executable, os.path.abspath(__file__), '--ref-torch-worker', json.dumps(spec)],
                             env=env, capture_output=True, text=True, timeout=240)
        for ln in reversed(res.stdout.strip().splitlines()):
            try:
                out = json.loads(ln)
                out['kind'] = 'reference (unmodified, its torch engine on cuda:%d of this box)' % gpu_index
                return out
            except ValueError:
                continue
        return {'unavailable': 'no output; stderr tail: ' + res.stderr.strip()[-300:]}
    except Exception as e:  # noqa: BLE001
        return {'unavailable': repr(e)[:300]}


def run_reference_subprocess(cfg, cores, warmup, steps, per_step, seconds_per_step, timeout_s):
    """-> dict (see ref_worker_main) or None if the reference is not installed / failed / timed out."""
    if not reference_available():
        return None
    spec = {'cfg': cfg, 'cores': cores, 'warmup': warmup, 'steps': steps, 'per_step': per_step,
            'seconds_per_step': seconds_per_step}
    env = dict(os.environ)
    for k in ('OMP_NUM_THREADS', 'OPENBLAS_NUM_THREADS', 'MKL_NUM_THREADS'):
        env[k] = '1'  # one BLAS thread per worker process: the pool already uses every host thread
    env['CUDA_VISIBLE_DEVICES'] = ''
    for k in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK'):
        env.pop(k, None)
    try:
        out = subprocess.run([sys.executable, os.path.abspath(__file__), '--ref-worker', json.dumps(spec)],
                             env=env, capture_output=True, text=True, timeout=timeout_s)
    except subprocess.TimeoutExpired:
        log('reference subprocess timed out after %.0f s' % timeout_s)
        return None
    if out.returncode != 0:
        log('reference subprocess failed: %s' % out.stderr.strip()[-400:])
        return None
    for ln in reversed(out.stdout.strip().splitlines()):
        try:
            return json.loads(ln)
        except ValueError:
            continue
    return None


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the prediction path on all host
    threads -- the unmodified reference from baseline/_ref when it is installed (kind "reference"),
    otherwise the oracle port of predict.py:84-245 (kind "port").  Under torchrun only rank 0 works."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    from sgdml_b200 import synth

    cfg = workload_cfg(args)
    perms, _ = synth.config_perms_and_r0(cfg['name'])
    S = len(perms)
    cores = os.cpu_count() or 1
    # each step a bounded sample (~4 s) so that warmup + steps stay within a few minutes
    res = run_reference_subprocess(cfg, cores, args.warmup, args.steps, args.ref_batch, 4.0,
                                   timeout_s=120 + 30.0 * (args.warmup + args.steps))
    if res is not None:
        kind = 'reference'
        per_step, dt = res['per_step'], res['seconds']
        sample = ('%d steps x %d query geometries, unmodified reference GDMLPredict(use_torch=False).predict, bulk mode, '
                  '%d worker processes (1 BLAS thread each), chunk_size %s; oracle vs reference on 4 queries: %.1e rel'
                  % (args.steps, per_step, res['workers'], res['chunk_size'], res['oracle_vs_reference_rel']))
    else:
        kind = 'port'
        model = oracle_random_model(cfg, perms)
        cores = cpu_workers(cfg, S)
        cpu = CpuPredictor(model, cfg, cores)
        cpu.rate(cores, seed=3)  # spin the pool up
        rate_probe = cpu.rate(4 * cores, seed=5)
        per_step = args.ref_batch or int(max(cores, min(200000, rate_probe * 4.0)))
        for _ in range(args.warmup):
            cpu.rate(per_step, seed=7)
        t0 = time.perf_counter()
        for k in range(args.steps):
            cpu.rate(per_step, seed=11 + k)
        dt = time.perf_counter() - t0
        cpu.close()
        sample = '%d steps x %d query geometries, NumPy oracle port, process pool over all host threads (1 BLAS thread each)' % (args.steps, per_step)
    value = per_step * args.steps / dt
    line = {
        'impl': 'reference',
        'metric': 'force_predictions_per_s',
        'value': value,
        'unit': 'predictions/s',
        'n_gpus': args.gpus,
        'steps': args.steps,
        'warmup': args.warmup,
        'ms_per_step': 1e3 * dt / args.steps,
        'higher_is_better': True,
        'scaling': 'weak',
        'vs_baseline': None,
        'dtype': 'f64',
        'data': 'synthetic',
        'config': {
            'workload': WORKLOADS[args.workload][1],
            'n_atoms': cfg['n_atoms'],
            'n_train': cfg['n_train'],
            'n_perms': S,
            'sig': cfg['sig'],
            'batch_per_step': per_step,
        },
        'cpu_baseline': {
            'value': value,
            'unit': 'predictions/s',
            'cores': cores,
            'kind': kind,
            'sample': sample,
        },
        'e2e': {'value': value, 'unit': 'predictions/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line))


# --------------------------------------------------------------------------- engine arm
def _barrier(world):
    import torch
    import torch.distributed as dist

    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def _max_over_ranks(seconds, world):
    import torch
    import torch.distributed as dist

    t = torch.tensor([seconds], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def measure_workload(args, workload, batch, steps, warmup, world, rank, local_rank, compact=False, dump_dir=None):
    """One full measurement of a named workload: training leg (rank 0), device-resident prediction steps,
    end-to-end steps through the public API with host buffers, roofline of the dominant kernel and (not compact)
    the CPU / reference baselines.  With `dump_dir`, rank 0 writes the outputs of the last device-resident step
    (dump_outputs).  Returns the JSON line as a dict on rank 0, None elsewhere."""
    import torch
    import torch.distributed as dist

    import sgdml_b200
    from sgdml_b200 import _lib, synth
    from sgdml_b200.diagnostics import residual_report

    L = _lib.lib()
    wargs = argparse.Namespace(**vars(args))
    wargs.workload = workload
    cfg = workload_cfg(wargs)
    no_train = args.no_train or workload in PREDICT_ONLY
    N, M = cfg['n_atoms'], cfg['n_train']
    D = N * (N - 1) // 2
    perms, r0 = synth.config_perms_and_r0(cfg['name'])
    S = len(perms)
    n = 3 * N * M

    # ---------------- training leg (rank 0), model broadcast to the other ranks
    train_info = None
    task = synth.make_task(N, M, perms, cfg['sig'], r0=r0)
    trainer = sgdml_b200.GDMLTrain()
    if no_train:
        model = synth.random_model(N, M, perms, cfg['sig'], r0=r0)
    else:
        alphas_t = torch.empty(n + 2, dtype=torch.float64, device='cuda')
        if rank == 0:
            # warm-up: a small training run (kernel load, context, allocator), then ONE untimed pass of the timed
            # configuration itself -- the training step's warm-up step.  Its wall time is reported as `cold_run`: it
            # carries the first-use costs (31.8 GB K buffer, factorisation workspaces, first launches at this size),
            # which were measured between 0.03 and 0.9 s depending on the box.
            log('[%s] warm-up training run' % workload)
            trainer.train(synth.make_task(N, min(M, 40), perms, cfg['sig'], r0=r0))
            cold_run = None
            if not compact:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                trainer.train(task)
                torch.cuda.synchronize()
                cold_run = {'total_s': time.perf_counter() - t0, 'timings': {k: float(v) for k, v in trainer.timings.items()}}
                log('[%s] cold training run (untimed warm-up step): %.3f s (%s)' % (workload, cold_run['total_s'], trainer.timings))
            log('[%s] timed training run: n = %d' % (workload, n))
            # clocks / power / throttle reasons during the training run too: the int8 trailing updates draw far more
            # power than the FP64 DMMA kernels, so a power or thermal cap would show here and not in the predict phase
            tsampler = ClockSampler(local_rank)
            tsampler.start()
            time.sleep(0.5)
            tsampler.rows.clear()
            torch.cuda.synchronize()
            L.sgdml_b200_profile_reset()
            t0 = time.perf_counter()
            model0 = trainer.train(task)
            torch.cuda.synchronize()
            train_s = time.perf_counter() - t0
            train_clocks = tsampler.stop()
            log('[%s] training done in %.3f s (%s)' % (workload, train_s, trainer.timings))
            snap = _lib.profile_snapshot()
            tm = trainer.timings
            hbm_peak, hbm_src = measured_peak('hbm_gbs', 6650.0)
            fp64_peak = fp64_peak_tflops(L)
            asm_bytes = 8.0 * n * n + 8.0 * M * 4 * D
            asm_flops = float(M) * M * 2.0 * D * 3 * N * (S + 6)  # SURVEY 8d: W_K = 2 D 3N (S + 6) per block
            # independent check of the benchmarked training run: (K - lam I) alphas against the labels through the
            # predictor kernels (none of the assembly / Cholesky code), and the forces on the training points
            chk = residual_report(model0, task)
            chk['ok'] = bool(chk['residual_rel'] < 1e-8 and chk['force_rel_max_train'] < 1e-3)
            log('[%s] solution check: %s' % (workload, chk))
            train_info = {
                'metric': 'K-assembly+solve wall-time',
                'unit': 's',
                'higher_is_better': False,
                'n': n,
                'K_bytes': 8 * n * n,
                'total_s': train_s,
                'clocks': train_clocks,
                'assemble_s': tm['assemble_s'],
                'solve_s': tm['solve_s'],
                'what': 'GDMLTrain.train(task): host R/F/E in -> model dict out (descriptors, K assembly in HBM, '
                'FP64 Cholesky + 2 triangular solves, R_d_desc_alpha, integration constant)',
                'gpu_launches': int(sum(v[2] for v in snap.values())),
                'solution_check': dict(
                    chk,
                    what='||(K - lam I) alphas - y|| / ||y|| with K.alphas evaluated by the predictor kernels '
                    '(K.v identity, iterative.py:183-204): independent of the assembly and Cholesky kernels; '
                    'force_rel_max_train = max |F_pred - F_label| / max |F_label| on ALL training points',
                ),
                'roofline_assemble': {
                    'bound': 'hbm',
                    'achieved': asm_bytes / tm['assemble_s'] * 1e-9,
                    'peak': hbm_peak,
                    'unit': 'GB/s',
                    'frac': asm_bytes / tm['assemble_s'] * 1e-9 / hbm_peak,
                    'peak_source': hbm_src,
                    'algorithmic_bytes': asm_bytes,
                    'fp64': {
                        'algorithmic_flops': asm_flops,
                        'achieved_tflops': asm_flops / tm['assemble_s'] * 1e-12,
                        'frac_of_fp64_peak': asm_flops / tm['assemble_s'] * 1e-12 / fp64_peak,
                        'note': 'SURVEY 8d: above ~5 flop/B the FP64 pipe governs; both terms are reported, '
                        'the larger fraction names the binding roofline',
                    },
                },
                'roofline_solve': {
                    'bound': 'fp64-tensor (DMMA)',
                    'achieved': (n**3 / 3.0) / tm['solve_s'] * 1e-12,
                    'peak': fp64_peak,
                    'unit': 'TFLOP/s',
                    'frac': (n**3 / 3.0) / tm['solve_s'] * 1e-12 / fp64_peak,
                    'peak_source': 'live DMMA m8n8k4 probe (sgdml_b200_fp64_peak_tflops); MEASURED_PEAKS.json has no FP64 entry',
                    'algorithmic_flops': n**3 / 3.0,
                    'trailing_update': 'FP64 DMMA',
                    'note': 'whole solve (potf2 + TRSM strips + trailing updates + 2 triangular solves) over n^3/3; a '
                    'fraction above 1 means the trailing updates ran on the int8 tensor cores (error-free slicing)',
                },
            }
            slices_env = os.environ.get('SGDML_B200_OZAKI_SLICES')
            int8_default = slices_env is None and n >= 16384
            if int8_default or (slices_env not in (None, '', '0')):
                train_info['roofline_solve']['trailing_update'] = (
                    'tcgen05.mma kind::i8 on %s signed 7-bit slices per operand (exact int32 accumulation in tensor memory, '
                    'FP64 level sums); default for n >= 16384, sgdml_b200_set_solve_slices(0) / SGDML_B200_OZAKI_SLICES=0 = FP64 DMMA'
                    % (slices_env or '7'))
                train_info['roofline_solve']['bound'] = 'int8 tensor pipe + shared-memory operand bandwidth (csrc/ozaki.cu); fraction quoted against the FP64 DMMA peak it replaces'
            if cold_run is not None:
                train_info['cold_run'] = cold_run
            if int8_default and not compact:
                # the same training run with all-FP64 trailing updates, for comparison (and as a second, independent solution)
                L.sgdml_b200_set_solve_slices(0)
                try:
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    model_fp64 = trainer.train(task)
                    torch.cuda.synchronize()
                    t_fp64 = time.perf_counter() - t0
                    chk64 = residual_report(model_fp64, task)
                    a0, a1 = model0['alphas_F'], model_fp64['alphas_F']
                    train_info['fp64_dmma'] = {
                        'total_s': t_fp64,
                        'solve_s': trainer.timings['solve_s'],
                        'timings': {k: float(v) for k, v in trainer.timings.items()},
                        'residual_rel': chk64['residual_rel'],
                        'force_rel_max_train': chk64['force_rel_max_train'],
                        'solve_tflops': (n**3 / 3.0) / trainer.timings['solve_s'] * 1e-12,
                        'frac_of_fp64_peak': (n**3 / 3.0) / trainer.timings['solve_s'] * 1e-12 / fp64_peak,
                        'alphas_rel_diff_int8_vs_fp64': float(np.max(np.abs(a0 - a1)) / np.max(np.abs(a1))),
                        'what': 'the same GDMLTrain.train with sgdml_b200_set_solve_slices(0): every trailing update on the FP64 DMMA pipe',
                    }
                    log('[%s] FP64-DMMA training run: %.3f s (solve %.3f s)' % (workload, t_fp64, trainer.timings['solve_s']))
                finally:
                    L.sgdml_b200_set_solve_slices(-1)
            alphas_t[:n] = torch.from_numpy(model0['alphas_F']).cuda()
            alphas_t[n] = float(model0['c'])
            alphas_t[n + 1] = float(model0['std'])
        if world > 1:
            dist.broadcast(alphas_t, src=0)
        if rank == 0:
            model = model0
        else:
            host = alphas_t.cpu().numpy()
            desc = sgdml_b200.desc.Desc(N)
            R_desc, R_d_desc = desc.from_R(task['R_train'].reshape(M, -1))
            from sgdml_b200.desc import tril_perms_lin

            model = trainer.create_model(task, 'analytic', R_desc, R_d_desc, tril_perms_lin(perms), float(host[n + 1]), host[:n].copy())
            model['c'] = float(host[n])

    predictor = sgdml_b200.GDMLPredict(model)
    log('[%s] predictor ready; batch %d' % (workload, batch))

    # ---------------- prediction steps, inputs resident in HBM
    B = batch
    Rq_host = synth.geometries(N, B, 1 + rank, r0=r0).reshape(B, -1)
    Rq_dev = torch.from_numpy(Rq_host).cuda()
    # the clock sampler (an nvidia-smi child process) is started BEFORE the warm-up so that its
    # start-up (fork, NVML initialisation) cannot disturb the timed region
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.5)
    for _ in range(max(warmup, 3)):
        predictor.predict(Rq_dev)
    _barrier(world)
    if rank == 0:
        sampler.rows.clear()
    # one more untimed step is queued right before the start event: the device then has ~25 ms of work in front of the
    # timed steps, so a host hiccup while they are being enqueued (observed once on a loaded box: 28 ms, 10 % of a
    # 10-step region) cannot leave the GPU idle inside the timed region.  The region itself is K steps of device work
    # between two CUDA events on the launching stream.
    predictor.predict(Rq_dev)
    L.sgdml_b200_profile_reset()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        E_dev, F_dev = predictor.predict(Rq_dev)
    e1.record()
    _barrier(world)
    clocks = sampler.stop() if rank == 0 else None
    dt = _max_over_ranks(e0.elapsed_time(e1) * 1e-3, world)
    launches_timed = int(sum(v[2] for v in _lib.profile_snapshot().values()))
    value = world * B * steps / dt
    log('[%s] device-resident steps done: %.3e predictions/s' % (workload, value))
    if dump_dir is not None and rank == 0:
        dump_outputs(dump_dir, E_dev, F_dev, None if no_train else model['alphas_F'])

    # ---------------- end to end through the public API with pinned HOST buffers
    R_pin = torch.from_numpy(Rq_host).pin_memory()
    out_pin = (torch.empty(B, dtype=torch.float64).pin_memory(), torch.empty((B, 3 * N), dtype=torch.float64).pin_memory())
    for _ in range(2):
        predictor.predict(R_pin, out=out_pin)
    _barrier(world)
    t0 = time.perf_counter()
    for _ in range(steps):
        E_h, F_h = predictor.predict(R_pin, out=out_pin)
        _ = float(E_h[0])  # the step's result is read on the host
    torch.cuda.synchronize()
    dt_e2e = _max_over_ranks(time.perf_counter() - t0, world)
    e2e_value = world * B * steps / dt_e2e
    log('[%s] e2e steps done: %.3e predictions/s' % (workload, e2e_value))

    # ---------------- the same through the reference-shaped call: NumPy array in, NEW NumPy arrays out (pageable)
    for _ in range(2):
        predictor.predict(Rq_host)
    _barrier(world)
    t0 = time.perf_counter()
    for _ in range(steps):
        E_n, F_n = predictor.predict(Rq_host)
        _ = float(E_n[0])
    dt_np = _max_over_ranks(time.perf_counter() - t0, world)
    e2e_numpy = world * B * steps / dt_np
    log('[%s] e2e (NumPy in/out) steps done: %.3e predictions/s' % (workload, e2e_numpy))

    # parity spot check of the benchmarked path (tiny, after the timed regions)
    assert np.allclose(F_h[:8].numpy(), F_dev[:8].cpu().numpy(), rtol=0, atol=0), 'host and device paths disagree'
    assert np.array_equal(F_n[:8], F_h[:8].numpy()), 'NumPy and pinned-tensor paths disagree'

    # ---------------- roofline of the dominant kernel (rank 0): device time of k_predict_main
    roofline = None
    cpu_baseline = None
    ref_torch = None
    if rank == 0:
        L.sgdml_b200_profile_reset()
        L.sgdml_b200_profile_enable(1)
        reps = 3
        for _ in range(reps):
            predictor.predict(Rq_dev)
        torch.cuda.synchronize()
        L.sgdml_b200_profile_enable(0)
        snap = _lib.profile_snapshot()
        main_ms, main_scopes, main_launches = snap['predict_main']
        aux_ms = snap['predict_aux'][0] + snap['desc'][0]
        flops_step = algorithmic_flops_per_query(cfg, S) * B
        t_step = main_ms * 1e-3 / reps
        fp64_peak = fp64_peak_tflops(L)
        achieved = flops_step / t_step * 1e-12
        # flops the kernels actually issue on the DMMA pipe: the GEMM form needs 8 per (row, m, d)
        # (2 GEMMs in, 2 GEMMs out) instead of the 9 of the reference's elementwise form (SURVEY 8d),
        # on descriptors padded to the tile width
        fused = D <= 256
        DP = next(p for p in (40, 72, 112, 160, 224, 256) if p >= D) if fused else (D + 3) // 4 * 4
        executed = 8.0 * M * S * DP * B / t_step * 1e-12
        roofline = {
            'bound': 'tensor',
            'pipe': 'fp64 tensor pipe (mma.sync.m8n8k4.f64 -> DMMA); tcgen05 has no f64 kind',
            'kernel': 'k_predict_main' if fused else 'GEMM-composed predictor: 4 x k_gemm_nt_tma + k_transform_rows + k_combine_rows',
            'achieved': achieved,
            'peak': fp64_peak,
            'unit': 'TFLOP/s',
            'frac': achieved / fp64_peak,
            'executed_tflops': executed,
            'frac_executed': executed / fp64_peak,
            'note': 'achieved counts the algorithmic 9*M*S*D flops per query of SURVEY 8d; the kernels issue 8*M*S*DP '
            '(GEMM form, padded D), so frac can exceed frac_executed (= DMMA-pipe utilisation) by up to 9/8',
            'peak_source': 'live DMMA m8n8k4 probe (sgdml_b200_fp64_peak_tflops), burst; MEASURED_PEAKS.json carries only HBM and bf16 peaks',
            'algorithmic_flops_per_step': flops_step,
            'kernel_ms_per_step': t_step * 1e3,
            'launches_per_step': main_launches / reps,
            'kernel_share_of_step': main_ms / max(main_ms + aux_ms, 1e-9),
            'traffic': ncu_traffic(workload, B / max(main_launches / reps, 1)),
        }
        log('[%s] roofline probe done' % workload)
        if world == 1 and not args.no_cpu_baseline and not compact:
            cfg_named = dict(cfg)
            all_cores = os.cpu_count() or 1
            # the unmodified reference on all host threads when baseline/_ref is installed (one step of
            # ~cpu_seconds), otherwise the oracle port
            res = run_reference_subprocess(cfg_named, all_cores, 0, 1, None, args.cpu_seconds, timeout_s=120 + 4 * args.cpu_seconds)
            if res is not None:
                rate = res['per_step'] * res['steps'] / res['seconds']
                log('cpu baseline (reference): %.1f predictions/s' % rate)
                cpu_baseline = {
                    'value': rate,
                    'unit': 'predictions/s',
                    'cores': all_cores,
                    'kind': 'reference',
                    'sample': '%d query geometries of the same workload, unmodified reference GDMLPredict(use_torch=False).predict in bulk mode, '
                    '%d worker processes (1 BLAS thread each), chunk_size %s; oracle vs reference on 4 queries: %.1e rel'
                    % (res['per_step'], res['workers'], res['chunk_size'], res['oracle_vs_reference_rel']),
                }
            else:
                cores = cpu_workers(cfg, S)
                cmodel = oracle_random_model(cfg, perms)
                cpu = CpuPredictor(cmodel, cfg, cores)
                cpu.rate(cores, seed=3)  # spin the pool up
                rate_probe = cpu.rate(4 * cores, seed=5)
                nq = int(max(cores, min(400000, rate_probe * args.cpu_seconds)))
                log('cpu baseline: %d queries on %d threads (probe rate %.1f/s)' % (nq, cores, rate_probe))
                rate = cpu.rate(nq)
                cpu.close()
                log('cpu baseline done: %.1f predictions/s' % rate)
                cpu_baseline = {
                    'value': rate,
                    'unit': 'predictions/s',
                    'cores': cores,
                    'kind': 'port',
                    'sample': '%d query geometries of the same workload, NumPy oracle port of predict.py:84-245, process pool over all host threads (1 BLAS thread each)'
                    % nq,
                }
            # the reference's OWN GPU path (torch, CUDA) on this B200: the "existing GPU implementation" bar
            ref_torch = reference_torch_cuda(cfg_named, local_rank)
            log('reference torch-CUDA arm: %s' % (ref_torch,))

    if rank == 0 and world == 1 and train_info is not None and not args.no_cpu_baseline and not compact:
        # the reference's own CPU training path beside it (bounded samples, extrapolated: SURVEY.md section 8d)
        train_info['cpu_reference'] = reference_train_estimate(dict(cfg), os.cpu_count() or 1)
        log('reference training estimate: %s' % (train_info['cpu_reference'],))

    del predictor
    if rank != 0:
        return None
    return {
        'metric': 'force_predictions_per_s',
        'value': value,
        'unit': 'predictions/s',
        'n_gpus': world,
        'steps': steps,
        'warmup': max(warmup, 3),
        'ms_per_step': 1e3 * dt / steps,
        'higher_is_better': True,
        'scaling': 'weak',
        'vs_baseline': None,
        'dtype': 'f64',
        'data': 'synthetic',
        'config': {
            'workload': WORKLOADS[workload][1],
            'n_atoms': N,
            'n_train': M,
            'n_perms': S,
            'sig': cfg['sig'],
            'batch_per_gpu_per_step': B,
            'parallelism': 'query batch sharded over %d GPU(s), model replicated, no data-path collective' % world,
            'l2': 'no explicit flush: each step streams >= %.0f MB of per-row workspace (query rows + partial forces, > 126 MB L2); '
            'the %.1f MB model is L2-resident by design' % (B * S * D * 8 * 2 / 1e6, 2 * M * D * 8 / 1e6),
            'model': 'trained by the engine in this run' if not no_train else 'random coefficients',
        },
        'e2e': {
            'value': e2e_value,
            'unit': 'predictions/s',
            'h2d_bytes_per_step': B * 3 * N * 8,
            'd2h_bytes_per_step': B * (3 * N + 1) * 8,
            'what': 'GDMLPredict.predict(pinned host R, out=pinned host E/F); H2D and D2H copies inside the timed region',
            'numpy': {
                'value': e2e_numpy,
                'unit': 'predictions/s',
                'what': 'the reference-shaped call: GDMLPredict.predict(np.ndarray) -> NEW NumPy arrays (pageable host '
                'memory both ways, output allocation inside the timed region)',
            },
        },
        'gpu_launches': launches_timed,
        'clocks': clocks,
        'roofline': roofline,
        'cpu_baseline': cpu_baseline,
        'ref_torch_cuda': ref_torch,
        'train': train_info,
    }


def measure_sharded(args, world, rank, local_rank):
    """The north-star splits (SURVEY 8e) on a large-molecule shape, at ANY number of GPUs (1 = the base of the
    strong-scaling curve): (i) prediction with the TRAINING POINTS sharded over the ranks -- every rank evaluates the
    whole batch against its M/G points, then ONE all-reduce of B*(3N+1) doubles on the device; (ii) iterations of
    the device-resident PCG with row-sharded K.v (all-gather of n doubles) and row-sharded Nystroem factor
    (all-reduce of m doubles + all-gather of n doubles).  Random coefficients / a random factor: the cost of both
    paths does not depend on the values.  Timed with CUDA events, max over ranks."""
    import ctypes

    import torch

    import sgdml_b200
    from sgdml_b200 import _lib, synth
    from sgdml_b200 import dist as sdist
    from sgdml_b200.desc import Desc

    name = args.sharded_workload
    cfg = dict(synth.CONFIGS[name])
    if args.sharded_n_train:
        cfg['n_train'] = args.sharded_n_train
    N, M = cfg['n_atoms'], cfg['n_train']
    perms, r0 = synth.config_perms_and_r0(name)
    S = len(perms)
    dim_i = 3 * N
    n = dim_i * M
    D = N * (N - 1) // 2
    L = _lib.lib()
    model = synth.random_model(N, M, perms, cfg['sig'], r0=r0)
    out = {'workload': WORKLOADS[name][1], 'n_atoms': N, 'n_train': M, 'n_perms': S, 'n': n, 'n_gpus': world}

    # ---- (i) prediction sharded over training points
    B = args.sharded_batch
    tp = sdist.TrainPointShardedPredictor(model, sgdml_b200.GDMLPredict)
    Rq = torch.from_numpy(synth.geometries(N, B, 1, r0=r0).reshape(B, -1)).cuda()
    for _ in range(2):
        tp.predict(Rq)
    _barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 3
    e0.record()
    for _ in range(reps):
        E, F = tp.predict(Rq)
    e1.record()
    _barrier(world)
    dt = _max_over_ranks(e0.elapsed_time(e1) * 1e-3, world) / reps
    flops = 9.0 * M * S * D * B
    fp64_peak = fp64_peak_tflops(L)
    out['train_point_sharded_predict'] = {
        'batch': B,
        'ms_per_batch': dt * 1e3,
        'predictions_per_s': B / dt,
        'collective': 'one all-reduce (NCCL, device buffers) of B*(3N+1) doubles per batch',
        'allreduce_bytes': B * (dim_i + 1) * 8,
        'tflops_algorithmic_total': flops / dt * 1e-12,
        'frac_of_fp64_peak_per_gpu': flops / dt * 1e-12 / world / fp64_peak,
    }
    del tp

    # ---- (ii) PCG iterations, K.v rows and factor rows sharded by training point
    lo, hi = sdist.shard_bounds(M, world, rank)
    pred = sgdml_b200.GDMLPredict(model)
    _, R_d_desc = Desc(N).from_R(synth.geometries(N, M, 0, r0=r0).reshape(M, -1))
    pred.set_R_d_desc(R_d_desc)
    del R_d_desc
    m_ind = args.sharded_inducing
    n_loc = (hi - lo) * dim_i
    ldx = (m_ind + 1) // 2 * 2
    X = 1e-3 * torch.randn((max(n_loc, 1), ldx), dtype=torch.float64, device='cuda')
    y = np.random.default_rng(3).standard_normal(n)
    check_every = 4
    wsd = int(L.sgdml_b200_pcg_workspace_doubles(n, n_loc, m_ind, check_every))
    ws = torch.empty(wsd, dtype=torch.float64, device='cuda')

    def _exchange(_ctx, op, buf, count):
        sdist.exchange_on_workspace(ws, (int(buf) - ws.data_ptr()) // 8, int(count), int(op), M, dim_i)
        return 0

    exch = _lib.EXCHANGE_FN(_exchange) if world > 1 else ctypes.cast(None, _lib.EXCHANGE_FN)
    prog = ctypes.cast(None, _lib.PROGRESS_FN)
    x = np.zeros(n)
    iters, resid = ctypes.c_int64(0), ctypes.c_double(0.0)

    def run(n_it):
        _lib.check(
            L.sgdml_b200_pcg(pred._handle, lo if world > 1 else 0, hi if world > 1 else M, X.data_ptr(), m_ind, ldx, 1e-10,
                             _lib.ptr(y), _lib.ptr(x), 1, 0.0, n_it, check_every, ws.data_ptr(), wsd, exch, None, prog, None,
                             ctypes.byref(iters), ctypes.byref(resid), _lib.current_stream()),
            'pcg',
        )

    run(1)  # warm-up (also the set-up: r0, z0, p0)
    _barrier(world)
    n_it = args.sharded_iters
    # set-up cost (one P.v, no K.v) is measured separately and subtracted
    e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    e[0].record()
    run(0)
    e[1].record()
    run(n_it)
    e[2].record()
    _barrier(world)
    t_setup = _max_over_ranks(e[0].elapsed_time(e[1]) * 1e-3, world)
    t_total = _max_over_ranks(e[1].elapsed_time(e[2]) * 1e-3, world)
    per_iter = max(t_total - t_setup, 1e-9) / max(int(iters.value), 1)
    kv_flops = 9.0 * M * M * S * D
    out['pcg_iteration'] = {
        'iterations_timed': int(iters.value),
        'ms_per_iteration': per_iter * 1e3,
        'inducing_columns': m_ind,
        'collectives_per_iteration': 'all-gather of n doubles (K.v rows), all-reduce of m doubles + all-gather of n doubles (P.v); '
        'NCCL on device buffers inside the solver workspace, enqueued by the exchange hook of sgdml_b200_pcg',
        'allgather_bytes_per_iteration': 2 * n * 8,
        'allreduce_bytes_per_iteration': m_ind * 8,
        'kv_tflops_algorithmic_total': kv_flops / per_iter * 1e-12,
        'frac_of_fp64_peak_per_gpu': kv_flops / per_iter * 1e-12 / world / fp64_peak,
        'limiting': 'K.v (FP64 tensor pipe); the collectives move %.1f MB per iteration' % ((2 * n + m_ind) * 8 / 1e6),
    }
    del pred, X, ws
    torch.cuda.empty_cache()
    return out if rank == 0 else None


def nccl_log_dir():
    """Per-launch directory for the NCCL logs: every rank of one torchrun launch sees the same run id and port."""
    import tempfile

    run = '%s_%s' % (os.environ.get('TORCHELASTIC_RUN_ID', 'run'), os.environ.get('MASTER_PORT', '0'))
    return os.path.join(tempfile.gettempdir(), 'sgdml_b200_nccl_%s' % run)


def run_engine(args):
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    nccl_log = None
    if world > 1:
        # NCCL's INFO log (rank count, rings/trees, NVLS) goes to a FILE per rank so that stdout stays the single
        # JSON line and the communicator can still be verified (comm_nranks).  Set BEFORE torch is imported:
        # NCCL latches its debug settings at its first call.  The directory is outside the source tree (which may be
        # read-only) and shared by the ranks of one launch.
        nccl_dir = nccl_log_dir()
        os.makedirs(nccl_dir, exist_ok=True)
        if os.environ.get('NCCL_DEBUG', '').upper() not in ('INFO', 'TRACE'):
            os.environ['NCCL_DEBUG'] = 'INFO'  # (a pre-set WARN / VERSION would leave the rank count unobservable)
            os.environ.setdefault('NCCL_DEBUG_SUBSYS', 'INIT,ENV')
        os.environ.setdefault('NCCL_DEBUG_FILE', os.path.join(nccl_dir, 'nccl_n%d_%%h_%%p.log' % world))
        nccl_log = os.environ['NCCL_DEBUG_FILE']
    import torch
    import torch.distributed as dist

    torch.cuda.set_device(local_rank)
    if world > 1:
        import datetime

        # a mismatched collective must fail in minutes, not in NCCL's default 10 (the slowest legitimate wait is rank > 0
        # waiting for rank 0's training legs: a few seconds)
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank), timeout=datetime.timedelta(seconds=240))
        # the communicator, checked directly: a sum of ones over the ranks and the distinct devices behind them
        ones = torch.ones(1, dtype=torch.float64, device='cuda')
        dist.all_reduce(ones)
        uuids = [None] * world
        dist.all_gather_object(uuids, str(torch.cuda.get_device_properties(local_rank).uuid))
        nccl_check = {
            'backend': dist.get_backend(),
            'world_size': dist.get_world_size(),
            'allreduce_of_ones': float(ones.item()),
            'distinct_devices': len(set(uuids)),
            'nccl_version': '.'.join(str(v) for v in torch.cuda.nccl.version()),
        }

    line = measure_workload(args, args.workload, args.batch, args.steps, args.warmup, world, rank, local_rank,
                            dump_dir=args.dump_outputs)
    default_run = args.workload == 'aspirin' and not args.no_train and args.n_train is None
    if default_run and world == 1 and not args.no_extras:
        # north_star's own target (ethanol: train < 1 s, >= 1e6 predictions/s at >= 60 % of the roofline) in the same
        # driver-recorded line
        eth = measure_workload(args, 'ethanol', args.batch, max(3, args.steps // 2), 3, world, rank, local_rank, compact=True)
        if rank == 0:
            line['north_star_ethanol'] = eth
    if not args.no_extras and (world > 1 or default_run):
        sh = measure_sharded(args, world, rank, local_rank)
        if rank == 0:
            line['sharded'] = sh
            if nccl_log:
                line['sharded']['nccl_debug_file'] = nccl_log
    if world > 1 and rank == 0:
        # NCCL's own account of the communicator: the init lines of every rank's INFO log, echoed to stderr (stdout
        # stays the one JSON line) and counted in the line
        import glob

        init_lines = []
        for fn in sorted(glob.glob(os.path.join(nccl_log_dir(), 'nccl_n%d_*.log' % world))):
            try:
                with open(fn) as f:
                    init_lines += [ln.strip() for ln in f if ('nranks' in ln or 'NVLS' in ln or 'Connected all' in ln)]
            except OSError:
                pass
        for ln in init_lines[:24]:
            print('[nccl] ' + ln, file=sys.stderr)
        nccl_check['debug_file'] = nccl_log
        nccl_check['init_lines_with_nranks'] = sum(1 for ln in init_lines if 'nranks %d' % world in ln or 'nranks=%d' % world in ln)
        line['nccl'] = nccl_check
    if rank == 0:
        print(json.dumps(line))
        sys.stdout.flush()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def ncu_traffic(workload, queries_per_launch):
    """DRAM bytes per launch of k_predict_main from the committed ncu capture (profiles/r02_traffic.json),
    scaled to this run's launch size; None if no capture exists for the workload."""
    try:
        with open(os.path.join(ROOT, 'profiles', 'r02_traffic.json')) as f:
            return float(json.load(f)[workload]['bytes_per_query']) * queries_per_launch
    except Exception:
        return None


def measured_peak(key, fallback):
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    try:
        with open(path) as f:
            return float(json.load(f)[key]), 'MEASURED_PEAKS.json (%s, of measured)' % key
    except Exception:
        return fallback, 'fallback from B200_PROFILING.md (of fallback)'


def fp64_peak_tflops(L):
    import ctypes

    v = ctypes.c_double()
    rc = L.sgdml_b200_fp64_peak_tflops(ctypes.byref(v))
    if rc != 0 or not (v.value > 0):
        raise RuntimeError('fp64 peak probe failed')
    return v.value


def main():
    args = parse_args()
    if args.ref_worker is not None:
        ref_worker_main(json.loads(args.ref_worker))
        return
    if args.ref_train_worker is not None:
        ref_train_worker_main(json.loads(args.ref_train_worker))
        return
    if args.ref_torch_worker is not None:
        ref_torch_worker_main(json.loads(args.ref_torch_worker))
        return
    if args.workload in PREDICT_ONLY:
        args.no_train = True
        if args.batch == 65536:
            args.batch = PREDICT_ONLY[args.workload]
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_engine(args)


if __name__ == '__main__':
    main()
