"""Per-kernel breakdown of bench.py's engine step with torch.profiler (CUDA activities).

Builds bench.py's EngineStep, warms up, then profiles --steps steps and writes to --out DIR:
  step_kernels.csv   kernel, launches per step, total us per step, share of the summed kernel time
  step_profile.json  the same per kernel, plus device-to-host copies, stream / device synchronisations and
                     host-to-device copies per step, summed kernel time against the profiled wall time, and the card's
                     name, power limit and maximum SM clock read in the same run

Kernel times come from the profiler's CUDA activity records of a warm, back-to-back step; the profiler slows the host, so
the wall time per step here is not bench.py's value.

    python scripts/step_profile.py --out DIR [--n 4000] [--workload p1] [--steps 3] [--warmup 3]
"""
import argparse
import collections
import csv
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402

SYNCS = ('cudaStreamSynchronize', 'cudaDeviceSynchronize', 'cudaEventSynchronize')


def kernel_name(name):
    """'void femo::k_spmv<false, 0, double, false>(int const*, ...)' -> 'k_spmv<false, 0, double, false>'"""
    s = name
    if s.startswith('void '):
        s = s[5:]
    depth = 0
    for i, ch in enumerate(s):
        if ch == '<':
            depth += 1
        elif ch == '>':
            depth -= 1
        elif ch == '(' and depth == 0:
            s = s[:i]
            break
    return s.replace('femo::', '')


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True)
    ap.add_argument('--n', type=int, default=None)
    ap.add_argument('--workload', default='p1', choices=['p1', 'p2', 'hex'])
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=3)
    a = ap.parse_args()
    import torch
    from torch.profiler import ProfilerActivity, profile
    from torch.autograd import DeviceType
    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device')
    n = a.n or dict(p1=bench.N_DEFAULT, p2=2000, hex=256)[a.workload]
    os.makedirs(a.out, exist_ok=True)
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip()
    es = bench.EngineStep(n, 0, kind=a.workload)
    for _ in range(a.warmup):
        es.step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        t0 = time.perf_counter()
        for _ in range(a.steps):
            es.step()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
    kern = collections.defaultdict(lambda: [0, 0.0])
    copies = collections.Counter()
    api = collections.Counter()
    for e in prof.events():
        if e.device_type == DeviceType.CUDA:
            if e.name.startswith('Memcpy') or e.name.startswith('Memset'):
                copies[e.name] += 1
            else:
                k = kern[kernel_name(e.name)]
                k[0] += 1
                k[1] += e.time_range.elapsed_us()
        elif e.name in SYNCS or e.name.startswith('cudaMemcpy'):
            api[e.name] += 1
    total = sum(v[1] for v in kern.values())
    rows = sorted(((name, c / a.steps, us / a.steps, us / total) for name, (c, us) in kern.items()), key=lambda r: -r[2])
    with open(os.path.join(a.out, 'step_kernels.csv'), 'w', newline='') as f:
        w = csv.writer(f)
        w.writerow(['kernel', 'launches_per_step', 'us_per_step', 'share'])
        for r in rows:
            w.writerow([r[0], '%g' % r[1], '%.1f' % r[2], '%.4f' % r[3]])
    per_step = lambda c: {k: v / a.steps for k, v in sorted(c.items())}   # noqa: E731
    d2h = sum(v for k, v in copies.items() if 'DtoH' in k) / a.steps
    syncs = sum(api[k] for k in SYNCS) / a.steps
    out = dict(gpu=gpu, workload=a.workload, n=n, steps=a.steps, warmup=a.warmup, step_info=es.info,
               kernel_ms_per_step=total / a.steps / 1e3, profiled_wall_ms_per_step=wall / a.steps * 1e3,
               launches_per_step=sum(r[1] for r in rows), d2h_copies_per_step=d2h, syncs_per_step=syncs,
               copies_per_step=per_step(copies), runtime_calls_per_step=per_step(api),
               kernels=[dict(kernel=r[0], launches_per_step=r[1], us_per_step=r[2], share=r[3]) for r in rows])
    json.dump(out, open(os.path.join(a.out, 'step_profile.json'), 'w'), indent=1)
    print('gpu: %s ; %s n=%d ; kernels %.2f ms/step (profiled wall %.2f ms), %d launches, %.1f D2H copies, %.1f syncs per step'
          % (gpu, a.workload, n, out['kernel_ms_per_step'], out['profiled_wall_ms_per_step'], out['launches_per_step'], d2h, syncs))
    for r in rows[:25]:
        print('%-60s %7g %9.1f us %6.2f %%' % (r[0][:60], r[1], r[2], 100 * r[3]))


if __name__ == '__main__':
    main()
