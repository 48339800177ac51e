"""Analytic Hessian against central differences of the forces, on BASELINE configs 1 (ethanol) and 2 (aspirin) with
the synthetic random-coefficient models bench.py uses (sgdml_b200.synth), at B = 1, 64 and 1024 queries.

Per (config, B), in one process on one GPU:
  * Hessians/s of GDMLPredict.predict_hessian (device tensors in and out), CUDA events around each call;
  * the same from central differences: one GDMLPredict.predict call on the 6N displaced geometries per query
    (h = 1e-4, displaced geometries built before the timed region), alternated call by call with the analytic one;
  * the max difference between the two Hessians, relative to max |H|;
  * flop counts from shapes (below) and their rates against the live FP64 DMMA peak: for the Gram kernel alone
    (k_hess_gram, device time from the library's profiling scopes, in a separate untimed pass) and end to end;
  * GPU name and power limit, read in the same run.

    python tools/hessian_probe.py --out profiles/r03_hessian_probe.json
"""

import argparse
import ctypes
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402


def flops(N, M, S):
    """Per Hessian, from shapes: Gram 4 M S (3N)^2 (A^T B over 2 M S rows), u / v construction 24 M S D (two sparse
    J^T products of 6 D multiply-adds each), weight GEMMs 4 M S D; a prediction is 9 M S D."""
    D = N * (N - 1) // 2
    gram = 4.0 * M * S * (3 * N) ** 2
    return {'gram': gram, 'construct': 24.0 * M * S * D, 'weights': 4.0 * M * S * D,
            'total': gram + 28.0 * M * S * D, 'prediction': 9.0 * M * S * D}


def gpu_info():
    import torch

    info = {'device': torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader,nounits'],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(',')
        info['power_limit_w'] = float(q[0])
        info['sm_clock_max_mhz'] = float(q[1])
    except Exception as e:  # noqa: BLE001
        info['power_limit_w'] = None
        info['nvidia_smi_error'] = str(e)
    return info


def run_case(p, N, R, h, reps):
    import torch

    from sgdml_b200 import _lib

    B, n = R.shape
    dev = R.device
    Ha = torch.empty((B, n, n), dtype=torch.float64, device=dev)
    Ea = torch.empty(B, dtype=torch.float64, device=dev)
    Fa = torch.empty((B, n), dtype=torch.float64, device=dev)
    eye = torch.eye(n, dtype=torch.float64, device=dev) * h
    Rcd = torch.stack([R[:, None, :] + eye[None], R[:, None, :] - eye[None]], dim=1).reshape(-1, n).contiguous()
    Fcd = torch.empty_like(Rcd)
    Ecd = torch.empty(Rcd.shape[0], dtype=torch.float64, device=dev)

    def analytic():
        p.predict_hessian(R, out=(Ea, Fa, Ha))

    def central():
        p.predict(Rcd, out=(Ecd, Fcd))

    for _ in range(3):  # warm-up of both shapes
        analytic()
        central()
    torch.cuda.synchronize()
    t_a, t_c = [], []
    for _ in range(reps):  # alternated
        for fn, acc in ((analytic, t_a), (central, t_c)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            acc.append(e0.elapsed_time(e1))
    Fc = Fcd.reshape(B, 2, n, n)
    Hcd = -(Fc[:, 0] - Fc[:, 1]) / (2 * h)  # [b, j, i] = -dF_i / dR_j
    diff = float((Ha - Hcd.transpose(1, 2)).abs().max() / Ha.abs().max())
    # Gram kernel device time: profiling scopes (synchronising), separate from the timed calls above
    L = _lib.lib()
    L.sgdml_b200_profile_enable(1)
    L.sgdml_b200_profile_reset()
    n_prof = max(3, min(reps, 10))
    for _ in range(n_prof):
        analytic()
    torch.cuda.synchronize()
    snap = _lib.profile_snapshot()
    L.sgdml_b200_profile_enable(0)
    gram_ms = snap['hessian'][0] / n_prof
    return {
        'analytic_ms_median': float(np.median(t_a)),
        'analytic_ms_all': [round(x, 4) for x in t_a],
        'central_ms_median': float(np.median(t_c)),
        'central_ms_all': [round(x, 4) for x in t_c],
        'gram_kernel_ms': gram_ms,
        'max_rel_diff_analytic_vs_central': diff,
        'H_max_abs': float(Ha.abs().max()),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None, help='JSON output path (default: stdout only)')
    ap.add_argument('--batches', default='1,64,1024')
    ap.add_argument('--configs', default='ethanol,aspirin')
    ap.add_argument('--h', type=float, default=1e-4)
    args = ap.parse_args()

    import torch

    import sgdml_b200
    from sgdml_b200 import _lib, synth

    _lib.require_gpu()
    info = gpu_info()
    peak = ctypes.c_double()
    _lib.check(_lib.lib().sgdml_b200_fp64_peak_tflops(ctypes.byref(peak)), 'fp64_peak')
    info['fp64_dmma_peak_tflops_live'] = peak.value
    results = []
    for name in args.configs.split(','):
        cfg = synth.CONFIGS[name]
        N, M = cfg['n_atoms'], cfg['n_train']
        perms, r0 = synth.config_perms_and_r0(name)
        S = perms.shape[0]
        model = synth.random_model(N, M, perms, cfg['sig'], r0=r0)
        p = sgdml_b200.GDMLPredict(model)
        fl = flops(N, M, S)
        for B in (int(b) for b in args.batches.split(',')):
            R = torch.from_numpy(synth.geometries(N, B, 1, r0=r0).reshape(B, -1)).cuda()
            reps = 30 if B <= 64 else 10
            r = run_case(p, N, R, args.h, reps)
            ta, tc, tg = r['analytic_ms_median'] * 1e-3, r['central_ms_median'] * 1e-3, r['gram_kernel_ms'] * 1e-3
            r.update({
                'config': name, 'n_atoms': N, 'n_train': M, 'n_perms': S, 'B': B,
                'flops_per_hessian': fl,
                'analytic_hessians_per_s': B / ta,
                'central_hessians_per_s': B / tc,
                'speedup_analytic_over_central': tc / ta,
                'gram_kernel_dmma_flops_tflops': fl['gram'] * B / tg * 1e-12 if tg > 0 else None,
                'gram_kernel_share_of_fp64_peak': fl['gram'] * B / tg * 1e-12 / peak.value if tg > 0 else None,
                'end_to_end_tflops': fl['total'] * B / ta * 1e-12,
                'end_to_end_share_of_fp64_peak': fl['total'] * B / ta * 1e-12 / peak.value,
            })
            results.append(r)
            print('%-8s B %5d  analytic %9.3f ms (%10.1f H/s)  central %9.3f ms (%10.1f H/s)  x%.1f  gram %.3f ms '
                  '(%.1f%% of peak)  e2e %.1f%%  diff %.1e' % (
                      name, B, r['analytic_ms_median'], r['analytic_hessians_per_s'], r['central_ms_median'],
                      r['central_hessians_per_s'], r['speedup_analytic_over_central'], r['gram_kernel_ms'],
                      100 * (r['gram_kernel_share_of_fp64_peak'] or 0), 100 * r['end_to_end_share_of_fp64_peak'],
                      r['max_rel_diff_analytic_vs_central']), flush=True)
        del p
    out = {'gpu': info, 'h': args.h, 'results': results}
    print(json.dumps(info))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(out, f, indent=1)


if __name__ == '__main__':
    main()
