"""16-bit against fp32 storage of X for the block-order TF32 sweeps, on the same data and the same card in one process.

    python tools/bench_x16.py [--config cfg3] [--rows N] [--reps 5] [--sweeps 100] [--out FILE]

Two engines on one seeded matrix (bench.gen_shard): one bound by default (16-bit copies of X and X', rri_bind decides
from the data), one bound with RRI_X16=0 (fp32 X'; the contractions stream fp32 X through the TF32 tensor map).  Per
arm: ms per sweep (CUDA events around one engine call of --sweeps sweeps; the arms alternate, --reps times, from the
same starting factors), the contraction times from profile_kernel('gemm_w' / 'gemm_t'), the bytes of X each
contraction reads and the rate that makes, and the relative difference of the factors after the first repetition.
X is larger than L2 at the benchmark shapes, so every sweep streams it from HBM.  Prints the GPU name, power limit
and clocks with the result (one JSON line, also written to --out)."""
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
        return subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.sm,clocks.max.sm,clocks.mem',
                               '--format=csv,noheader'], stdout=subprocess.PIPE, universal_newlines=True,
                              timeout=30).stdout.strip().splitlines()[0]
    except Exception as ex:
        return 'nvidia-smi unavailable (%s)' % ex


def timed(eng, W, T, n, params):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    eng.sweeps(W, T, n, params, want_flags=False)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--config', default='cfg3', choices=['cfg3', 'cfg5'])
    ap.add_argument('--rows', type=int, default=None, help='rows of the shard (config 5 on 8 GPUs: 125000 per GPU)')
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--sweeps', type=int, default=100)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device: this measurement needs the GPU')
    dev = torch.device('cuda:0')
    cfg = dict(bench.CONFIGS[a.config])
    if a.rows:
        cfg['n'] = a.rows
    n, d, k = cfg['n'], cfg['d'], cfg['k']
    X, W0, T0 = bench.gen_shard(torch, cfg, n, 0, dev)
    engines = {}
    for arm in ('f16', 'f32'):
        if arm == 'f32':
            os.environ['RRI_X16'] = '0'
        try:
            torch.cuda.synchronize()
            b0 = torch.cuda.Event(enable_timing=True)
            b1 = torch.cuda.Event(enable_timing=True)
            b0.record()
            eng = R.RRIEngine(X, k, order='hals', math='tf32')
            b1.record()
            b1.synchronize()
        finally:
            os.environ.pop('RRI_X16', None)
        engines[arm] = (eng, b0.elapsed_time(b1))
    res = {'gpu': gpu_info(), 'config': a.config, 'shape': [n, d, k], 'reps': a.reps, 'sweeps_per_rep': a.sweeps,
           'torch': torch.__version__}
    params = engines['f16'][0].params()
    state = {}
    for arm, (eng, _) in engines.items():           # warm-up: 3 sweeps of each arm
        W, T = W0.clone(), T0.clone()
        timed(eng, W, T, 3, params)
    times = {arm: [] for arm in engines}
    first = {}
    for rep in range(a.reps):
        for arm, (eng, _) in engines.items():
            W, T = W0.clone(), T0.clone()
            ms = timed(eng, W, T, a.sweeps, params)
            times[arm].append(ms)
            if rep == 0:
                first[arm] = (W.double(), T.double(), eng.rel_error(W, T))
            state[arm] = (W, T)
            print('rep %d %s %8.3f ms/sweep' % (rep, arm, ms), flush=True)
    for arm, (eng, bind_ms) in engines.items():
        W, T = state[arm]
        gw = eng.profile_kernel('gemm_w', W, T, 20)
        gt = eng.profile_kernel('gemm_t', W, T, 20)
        xb = n * d * (2 if eng.stats()['x_operand'] == 'f16' else 4)
        m = float(np.median(times[arm]))
        res[arm] = {'x_operand': eng.stats()['x_operand'], 'bind_ms': round(bind_ms, 2),
                    'ms_per_sweep_median': round(m, 4), 'ms_per_sweep_min': round(float(np.min(times[arm])), 4),
                    'ms_per_sweep_max': round(float(np.max(times[arm])), 4), 'ms_per_sweep_all': [round(t, 4) for t in times[arm]],
                    'sweeps_per_s': round(1000.0 / m, 1),
                    'gemm_w_ms': round(gw, 4), 'gemm_t_ms': round(gt, 4),
                    'x_bytes_per_contraction': xb,
                    'x_read_gbs_gemm_w': round(xb / (gw * 1e-3) / 1e9, 1), 'x_read_gbs_gemm_t': round(xb / (gt * 1e-3) / 1e9, 1),
                    'final_rel_error_rep0': first[arm][2]}
    Wa, Ta, _ = first['f16']
    Wb, Tb, _ = first['f32']
    res['rel_diff_W'] = float(torch.linalg.norm(Wa - Wb) / torch.linalg.norm(Wb))
    res['rel_diff_T'] = float(torch.linalg.norm(Ta - Tb) / torch.linalg.norm(Tb))
    res['speedup_median'] = round(res['f32']['ms_per_sweep_median'] / res['f16']['ms_per_sweep_median'], 3)
    res['gpu_after'] = gpu_info()
    line = json.dumps(res)
    print(line, flush=True)
    if a.out:
        with open(a.out, 'w') as f:
            f.write(line + '\n')
    for eng, _ in engines.values():
        eng.close()


if __name__ == '__main__':
    main()
