"""Cost of project_T_each_iter in the block order at config-3 shape (200000 x 20000, k = 64, fp32).

    python tools/bench_simplex_hals.py [--reps 5] [--sweeps 10] [--profile-dir DIR]

Times ms per sweep (CUDA events around RRIEngine.sweeps, the variants alternating, after a warm-up of each) of
    hals_tf32            block order, TF32 contractions, no constraint
    hals_tf32_fused      + project_T_each_iter, fused cooperative T update (the default where it applies)
    hals_tf32_chain      + project_T_each_iter, per-topic launch chain (RRI_SIMPLEX_FUSED=0)
    rri_simplex          interleaved order + project_T_each_iter, IEEE fp32, on the same data
and the device time of the constrained T update's own kernels (torch.profiler over one sweep of each block-order
variant).  X (16 GB) is larger than L2, so every sweep streams it from HBM.  Prints the GPU name and power limit."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench                     # noqa: E402
import rri_nmf_b200 as R         # noqa: E402


def gpu_info():
    try:
        return subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                              stdout=subprocess.PIPE, universal_newlines=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as ex:
        return 'nvidia-smi unavailable (%s)' % ex


def ms_per_sweep(eng, W, T, n, params, chain):
    if chain:
        os.environ['RRI_SIMPLEX_FUSED'] = '0'
    try:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        flags = eng.sweeps(W, T, n, params)
        e1.record()
        e1.synchronize()
    finally:
        os.environ.pop('RRI_SIMPLEX_FUSED', None)
    return e0.elapsed_time(e1) / n, flags


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--sweeps', type=int, default=10)
    ap.add_argument('--rri-sweeps', type=int, default=2)
    ap.add_argument('--profile-dir', default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device: this measurement needs the GPU')
    dev = torch.device('cuda:0')
    print('gpu: %s' % gpu_info(), flush=True)
    cfg = dict(bench.CONFIGS['cfg3'])
    X, W0, T0 = bench.gen_shard(torch, cfg, cfg['n'], 0, dev)
    k = cfg['k']
    hals = R.RRIEngine(X, k, order='hals', math='tf32')
    rri = R.RRIEngine(X, k, order='rri', math='ieee')
    hals.project_rows_simplex(T0, 1.0)
    free, cons = hals.params(), hals.params(ub_t=1.0, simplex_T=True)
    variants = [('hals_tf32', hals, free, False, a.sweeps), ('hals_tf32_fused', hals, cons, False, a.sweeps),
                ('hals_tf32_chain', hals, cons, True, a.sweeps), ('rri_simplex', rri, cons, False, a.rri_sweeps)]
    state = {}
    for name, eng, p, chain, _ in variants:           # warm-up: 2 sweeps of every variant from the same start
        W, T = W0.clone(), T0.clone()
        ms_per_sweep(eng, W, T, 2, p, chain)
        state[name] = (W, T)
    times = {v[0]: [] for v in variants}
    for rep in range(a.reps):
        for name, eng, p, chain, ns in variants:
            W, T = state[name]
            ms, flags = ms_per_sweep(eng, W, T, ns, p, chain)
            times[name].append(ms)
            print('rep %d %-16s %8.3f ms/sweep flags=%d' % (rep, name, ms, flags), flush=True)
    # launches per block-order sweep (the fused kernel is one launch; the chain 2k + 1)
    launches = {}
    for name, eng, p, chain, _ in variants[:3]:
        W, T = state[name]
        l0 = eng.stats()['kernel_launches']
        ms_per_sweep(eng, W, T, 1, p, chain)
        launches[name] = eng.stats()['kernel_launches'] - l0
    # device time of the constrained update's own kernels, one sweep each under the profiler
    from torch.profiler import profile, ProfilerActivity
    kern_us = {}
    for name, eng, p, chain, _ in variants[1:3]:
        W, T = state[name]
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            ms_per_sweep(eng, W, T, 1, p, chain)
            torch.cuda.synchronize()
        tot, cnt = 0.0, 0
        for ev in prof.key_averages():
            if 'simplex' in ev.key:
                tot += ev.device_time_total if hasattr(ev, 'device_time_total') else ev.cuda_time_total
                cnt += ev.count
        kern_us[name] = (tot, cnt)
        if a.profile_dir:
            os.makedirs(a.profile_dir, exist_ok=True)
            with open(os.path.join(a.profile_dir, 'simplex_%s_kernels.txt' % name), 'w') as f:
                f.write(prof.key_averages().table(sort_by='cuda_time_total', row_limit=25))
    res = {'gpu': gpu_info(), 'shape': [cfg['n'], cfg['d'], k], 'dtype': 'f32', 'reps': a.reps}
    for name in times:
        m = float(np.median(times[name]))
        res[name] = {'ms_per_sweep_median': round(m, 3), 'ms_per_sweep_min': round(float(np.min(times[name])), 3),
                     'ms_per_sweep_max': round(float(np.max(times[name])), 3), 'sweeps_per_s': round(1000.0 / m, 1)}
    for name, l in launches.items():
        res[name]['launches_per_sweep'] = l
    for name, (us, cnt) in kern_us.items():
        res[name]['constrained_update_kernel_ms_per_sweep'] = round(us / 1000.0, 3)
        res[name]['constrained_update_kernels_per_sweep'] = cnt
    base = res['hals_tf32']['ms_per_sweep_median']
    res['extra_ms_per_sweep_fused'] = round(res['hals_tf32_fused']['ms_per_sweep_median'] - base, 3)
    res['extra_ms_per_sweep_chain'] = round(res['hals_tf32_chain']['ms_per_sweep_median'] - base, 3)
    print(json.dumps(res), flush=True)
    hals.close()
    rri.close()


if __name__ == '__main__':
    main()
