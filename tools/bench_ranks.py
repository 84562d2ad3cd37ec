"""A rank sweep (models of different ranks of one X) per pass over X against the same ranks fitted one after another, on
one card in one process.

    python tools/bench_ranks.py [--config cfg3] [--sets 2-20,10-60,pow2] [--reps 5] [--sweeps 20] [--out FILE]

For each storage of X (the 16-bit copies, and fp32 with RRI_X16=0) and each rank set -- 2..20 (width 209), 10, 20, ..,
60 (width 210), 8, 16, 32, 64, 128 (width 248), and the control (64,)*4 through the rank list against models=4 -- one
ranks engine and one single-model TF32 engine per rank.  Per repetition, from the same seeded starting factors: one call
of --sweeps sweeps of the ranks engine, then --sweeps sweeps of every rank on its own engine (CUDA events around the
sweep calls, summed over the ranks; each single-model engine holds its own copy of Xᵀ, so one at a time is created,
warmed up and closed outside the timed calls; the two arms alternate, --reps times).  Reported: ms per sweep of all
models for both arms and their ratio, the contraction time of both half-steps at the batch width (profile_kernel 'gemm_w' / 'gemm_t'), the rest of a
batched sweep (row updates, transposes, factor conversions), and every model's final relative error against its own
run after the first repetition.  X is larger than L2.  Prints the GPU name and power limit read in the same call."""
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
from bench_models import timed   # noqa: E402

SETS = {'2-20': list(range(2, 21)), '10-60': list(range(10, 61, 10)), 'pow2': [8, 16, 32, 64, 128],
        'control': [64] * 4}


def starts(n, d, ranks, dev):
    Ws, Ts = [], []
    for m, k in enumerate(ranks):
        g = torch.Generator(device=dev)
        g.manual_seed(2000 + 17 * k + m)
        Ws.append(torch.rand((n, k), generator=g, device=dev, dtype=torch.float32))
        Ts.append(torch.rand((k, d), generator=g, device=dev, dtype=torch.float32))
    return Ws, Ts


def engine(X, k, x16, models=None):
    if not x16:
        os.environ['RRI_X16'] = '0'
    try:
        return R.RRIEngine(X, k, order='hals', math='tf32', models=models)
    finally:
        os.environ.pop('RRI_X16', None)


def run_set(X, name, ranks, x16, reps, sweeps, dev):
    n, d = int(X.shape[0]), int(X.shape[1])
    Ws, Ts = starts(n, d, ranks, dev)
    eng = engine(X, ranks, x16)
    prm = eng.params()
    W0, T0 = eng.pack(Ws, Ts)
    if name == 'control':                  # the other arm: the same models as models=4 of rank 64
        other = engine(X, 64, x16, models=4)
        Wo0, To0 = torch.stack(Ws).contiguous(), torch.stack(Ts).contiguous()
        other.sweeps(Wo0.clone(), To0.clone(), 3, prm, want_flags=False)
    W, T = W0.clone(), T0.clone()
    eng.sweeps(W, T, 3, prm, want_flags=False)                    # warm-up
    t_batch, t_other = [], []
    err_batch = err_other = None
    for rep in range(reps):
        W, T = W0.clone(), T0.clone()
        t_batch.append(timed(lambda: eng.sweeps(W, T, sweeps, prm, want_flags=False)) / sweeps)
        if name == 'control':
            Wo, To = Wo0.clone(), To0.clone()
            t_other.append(timed(lambda: other.sweeps(Wo, To, sweeps, prm, want_flags=False)) / sweeps)
        else:
            tot, errs = 0.0, []
            for m, k in enumerate(ranks):
                single = engine(X, k, x16)
                single.sweeps(Ws[m].clone(), Ts[m].clone(), 3, prm, want_flags=False)     # warm-up
                Wm, Tm = Ws[m].clone(), Ts[m].clone()
                tot += timed(lambda: single.sweeps(Wm, Tm, sweeps, prm, want_flags=False))
                if rep == 0:
                    errs.append(single.rel_error(Wm, Tm))
                single.close()
            t_other.append(tot / sweeps)
        if rep == 0:
            err_batch = eng.rel_error(W, T)
            err_other = other.rel_error(Wo, To) if name == 'control' else errs
        print('%s x16=%d rep %d: batch %.3f ms/sweep, other arm %.3f ms/sweep'
              % (name, x16, rep, t_batch[-1], t_other[-1]), flush=True)
    gw = eng.profile_kernel('gemm_w', W, T, 20)
    gt = eng.profile_kernel('gemm_t', W, T, 20)
    mb, mo = float(np.median(t_batch)), float(np.median(t_other))
    out = {'set': name, 'ranks': ranks, 'width': sum(ranks), 'x_operand': eng.stats()['x_operand'],
           'batch_ms_per_sweep': round(mb, 4), 'other_arm': 'models=4' if name == 'control' else 'one engine per rank',
           'other_ms_per_sweep': round(mo, 4), 'speedup': round(mo / mb, 3),
           'batch_all': [round(t, 4) for t in t_batch], 'other_all': [round(t, 4) for t in t_other],
           'gemm_w_ms': round(gw, 4), 'gemm_t_ms': round(gt, 4), 'beyond_contraction_ms': round(mb - gw - gt, 4),
           'max_abs_rel_error_diff': float(np.max(np.abs(np.array(err_batch) - np.array(err_other)))),
           'rel_error_batch': err_batch, 'rel_error_other': err_other}
    eng.close()
    if name == 'control':
        other.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--config', default='cfg3', choices=sorted(bench.CONFIGS))
    ap.add_argument('--sets', default='2-20,10-60,pow2,control')
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
        for name in a.sets.split(','):
            res = run_set(X, name, SETS[name], storage == 'f16', a.reps, a.sweeps, dev)
            res['config'] = a.config
            print(json.dumps(res), flush=True)
            lines.append(res)
    tail = {'gpu_after': gpu_info()}
    print(json.dumps(tail), flush=True)
    lines.append(tail)
    if a.out:
        with open(a.out, 'w') as f:
            for r in lines:
                f.write(json.dumps(r) + '\n')


if __name__ == '__main__':
    main()
