"""Several block-order models per pass over X against the same models run one after another, on one card in one process.

    python tools/bench_models.py [--config cfg3] [--ks 16,32,64] [--reps 5] [--sweeps 20] [--out FILE]

For each storage of X (the 16-bit copies, and fp32 with RRI_X16=0), each rank k and each number of models
b in {1, 2, 4, 256/k}: one engine with models=b and one single-model engine, both TF32.  Per repetition, from the same
seeded starting factors: one call of --sweeps sweeps of the batched engine, then --sweeps sweeps of each of the b models
on the single-model engine (CUDA events around the engine calls; the two arms alternate, --reps times).  Reported: ms
per sweep of all b models and per model for both arms, their ratio, the contraction time of both half-steps at the
batched width N = b*k (profile_kernel 'gemm_w' / 'gemm_t') and the bytes of X per second that makes, and every model's
final relative error against its single-model run after the first repetition.  X is larger than L2: every sweep streams
it from HBM.  Prints the GPU name and power limit read in the same call (one JSON line per configuration, all of them
also written to --out)."""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))
import bench                     # noqa: E402
import rri_nmf_b200 as R         # noqa: E402
from bench_x16 import gpu_info   # noqa: E402


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1)


def starts(n, d, k, b, dev):
    Ws, Ts = [], []
    for m in range(b):
        g = torch.Generator(device=dev)
        g.manual_seed(1000 + 17 * k + m)
        Ws.append(torch.rand((n, k), generator=g, device=dev, dtype=torch.float32))
        Ts.append(torch.rand((k, d), generator=g, device=dev, dtype=torch.float32))
    return Ws, Ts


def engine(X, k, models, x16):
    if not x16:
        os.environ['RRI_X16'] = '0'
    try:
        return R.RRIEngine(X, k, order='hals', math='tf32', models=models)
    finally:
        os.environ.pop('RRI_X16', None)


def run_config(X, k, b, x16, single, reps, sweeps, dev):
    n, d = int(X.shape[0]), int(X.shape[1])
    Ws, Ts = starts(n, d, k, b, dev)
    eng = engine(X, k, b, x16)
    prm = eng.params()
    Wb0, Tb0 = torch.stack(Ws).contiguous(), torch.stack(Ts).contiguous()
    Wb, Tb = Wb0.clone(), Tb0.clone()
    eng.sweeps(Wb, Tb, 3, prm, want_flags=False)                  # warm-up of both arms
    W, T = Ws[0].clone(), Ts[0].clone()
    single.sweeps(W, T, 3, prm, want_flags=False)
    t_batch, t_single = [], []
    err_batch = err_single = None
    for rep in range(reps):
        Wb, Tb = Wb0.clone(), Tb0.clone()
        t_batch.append(timed(lambda: eng.sweeps(Wb, Tb, sweeps, prm, want_flags=False)) / sweeps)
        Wsd = [w.clone() for w in Ws]
        Tsd = [t.clone() for t in Ts]

        def singles():
            for m in range(b):
                single.sweeps(Wsd[m], Tsd[m], sweeps, prm, want_flags=False)
        t_single.append(timed(singles) / sweeps)
        if rep == 0:
            err_batch = eng.rel_error(Wb, Tb)
            err_single = [single.rel_error(Wsd[m], Tsd[m]) for m in range(b)]
        print('k=%d b=%d x16=%d rep %d: batched %.3f ms/sweep, %d single %.3f ms/sweep'
              % (k, b, x16, rep, t_batch[-1], b, t_single[-1]), flush=True)
    gw = eng.profile_kernel('gemm_w', Wb, Tb, 20)
    gt = eng.profile_kernel('gemm_t', Wb, Tb, 20)
    xb = n * d * (2 if eng.stats()['x_operand'] == 'f16' else 4)
    mb, ms = float(np.median(t_batch)), float(np.median(t_single))
    out = {'k': k, 'models': b, 'N': b * k, 'x_operand': eng.stats()['x_operand'],
           'batched_ms_per_sweep': round(mb, 4), 'batched_ms_per_model_sweep': round(mb / b, 4),
           'separate_ms_per_sweep': round(ms, 4), 'separate_ms_per_model_sweep': round(ms / b, 4),
           'speedup': round(ms / mb, 3),
           'batched_all': [round(t, 4) for t in t_batch], 'separate_all': [round(t, 4) for t in t_single],
           'gemm_w_ms': round(gw, 4), 'gemm_t_ms': round(gt, 4),
           'x_read_gbs_gemm_w': round(xb / (gw * 1e-3) / 1e9, 1), 'x_read_gbs_gemm_t': round(xb / (gt * 1e-3) / 1e9, 1),
           'max_abs_rel_error_diff': float(np.max(np.abs(np.array(err_batch) - np.array(err_single)))),
           'rel_error_batched': err_batch, 'rel_error_separate': err_single}
    eng.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--config', default='cfg3', choices=sorted(bench.CONFIGS))
    ap.add_argument('--ks', default='16,32,64')
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--sweeps', type=int, default=20)
    ap.add_argument('--storage', default='f16,f32')
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device: this measurement needs the GPU')
    dev = torch.device('cuda:0')
    cfg = dict(bench.CONFIGS[a.config])
    n, d = cfg['n'], cfg['d']
    X, _, _ = bench.gen_shard(torch, cfg, n, 0, dev)
    lines = []
    head = {'gpu': gpu_info(), 'config': a.config, 'shape': [n, d], 'reps': a.reps, 'sweeps_per_rep': a.sweeps,
            'torch': torch.__version__}
    print(json.dumps(head), flush=True)
    lines.append(head)
    for storage in a.storage.split(','):
        x16 = storage == 'f16'
        for k in [int(v) for v in a.ks.split(',')]:
            single = engine(X, k, None, x16)
            for b in sorted({1, 2, 4, 256 // k}):
                res = run_config(X, k, b, x16, single, a.reps, a.sweeps, dev)
                res['config'] = a.config
                print(json.dumps(res), flush=True)
                lines.append(res)
            single.close()
    tail = {'gpu_after': gpu_info()}
    print(json.dumps(tail), flush=True)
    lines.append(tail)
    if a.out:
        with open(a.out, 'w') as f:
            for r in lines:
                f.write(json.dumps(r) + '\n')


if __name__ == '__main__':
    main()
