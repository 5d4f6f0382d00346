"""Fine-level kernels of the V-cycle at the bench size: the per-kernel path (probe modes 0-3: residual, Chebyshev steps,
fused pre-smoother) against the two level sweeps of mgsweep.cuh (modes 6 / 7).

Builds bench.py's n = 4000 problem, runs one bench step, then times each kernel over 50 launches with CUDA events (every
input is larger than L2) and reports algorithmic bytes, GB/s and the fraction of the HBM copy peak.  The card's name,
power limit and maximum SM clock are recorded with the numbers.

    python scripts/mgsweep_probe.py --out DIR [--n 4000] [--reps 50]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402

KERNELS = {0: 'k_dia_apply<DIA_PLAIN,7> (residual)', 1: 'k_dia_apply<DIA_CHEB0,7>', 2: 'k_dia_apply<DIA_CHEBK,7>',
           3: 'k_dia_apply<DIA_PRE2,7>', 6: 'k_mg_down (PRE2 + residual + restriction)',
           7: 'k_mg_up (prolongation + CHEB0 + CHEBK)'}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--n', type=int, default=bench.N_DEFAULT)
    ap.add_argument('--reps', type=int, default=50)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device')
    os.makedirs(a.out, exist_ok=True)
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip()
    peaks = {}
    pk = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(pk):
        peaks = json.load(open(pk))
    peak = float(peaks.get('hbm_gbs', 6650.0))
    es = bench.EngineStep(a.n, 0)
    es.step()
    p = es.p
    rows = []
    for mode, name in KERNELS.items():
        alg, _ = p.vcycle_op_probe(mode)
        t = bench._time_launches(torch, lambda: p.vcycle_op_probe(mode), a.reps)
        gbs = alg / t / 1e9
        rows.append(dict(mode=mode, kernel=name, launch_us=t * 1e6, algorithmic_bytes=alg,
                         bytes_per_row=alg / p.N, achieved_gbs=gbs, frac_of_peak=gbs / peak))
        print('%-45s %8.1f us  %6.1f B/row  %7.0f GB/s  %.3f of peak' % (name, t * 1e6, alg / p.N, gbs, gbs / peak),
              flush=True)
    old = sum(r['launch_us'] for r in rows if r['mode'] in (0, 1, 2, 3))
    new = sum(r['launch_us'] for r in rows if r['mode'] in (6, 7))
    out = dict(gpu=gpu, n=a.n, dofs=p.N, reps=a.reps, peak_gbs=peak, kernels=rows,
               per_kernel_operator_us=old, sweeps_us=new,
               note='per-kernel sum excludes k_restrict_nested / k_prolong_nested (no probe mode)')
    print('gpu: %s ; operator kernels of the per-kernel visit %.1f us, two sweeps %.1f us' % (gpu, old, new))
    json.dump(out, open(os.path.join(a.out, 'mgsweep_probe.json'), 'w'), indent=1)


if __name__ == '__main__':
    main()
