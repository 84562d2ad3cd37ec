"""Observed-entries data with a weight w0 on the unstored entries (RRIEngine(X_csr, k, unstored_weight=w0),
rri_set_unstored_weight) against the same call with w0 = 0 and against the dense masked engine on the densified X with a
real-valued W_mat.

    python tools/bench_sparse_implicit.py [--shapes cfg4,big] [--sweeps 10] [--reps 2] [--no-dense] [--out DIR]

    cfg4  100 000 x 20 000, k = 50, fp32, 5 % nominal observed (the data of tools/bench_sparse.py), w0 = 0.05, unweighted
          and with entry weights 1 + alpha r (alpha = 0.5, r = the stored value over its mean); the arms w0 = 0 / w0 > 0
          run alternating, --reps times each.  The dense masked engine (math='ieee', both X and M dense: 16 GB) runs once
          from the same start, for its time and the output gap.
    big   1 000 000 x 100 000, k = 50, fp32, 0.1 % stored (1e8 entries; dense X and M would be 800 GB): w0 = 0 and 0.05,
          unweighted.
Per arm: ms per sweep (CUDA events around --sweeps sweeps in one call, after one warm-up sweep), launches per sweep, the
time of one T- and one W-half-step of topic 0 (rri_profile_kernel 'masked_t' / 'masked_w': pack + pass + (Gram row) +
solve, 20 launches each) and the final relative error sqrt(2 obj / sum M x^2).  The GPU name, power limit and max SM
clock are read in the same call."""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))
from bench_sparse_zero import _rel_err, _timed, gpu_info      # noqa: E402


def cfg4_data(dev):
    n, d, k, density = 100000, 20000, 50, 0.05
    g = torch.Generator(device=dev)
    g.manual_seed(0)
    U = torch.rand(n, k, generator=g, device=dev)
    V = torch.rand(k, d, generator=g, device=dev)
    X = U @ V
    X += 0.05 * X.mean() * torch.rand(n, d, generator=g, device=dev)
    M = torch.rand(n, d, generator=g, device=dev) < density
    W0 = torch.rand(n, k, generator=g, device=dev)
    T0 = torch.rand(k, d, generator=g, device=dev)
    Xs = (X * M).to_sparse_csr()
    del U, V, X, M
    torch.cuda.empty_cache()
    return Xs, W0, T0, k


def big_data(dev):
    n, d, k, per_row = 1000000, 100000, 50, 100
    g = torch.Generator(device=dev)
    g.manual_seed(1)
    U = torch.rand(n, k, generator=g, device=dev)
    Vt = torch.rand(d, k, generator=g, device=dev)
    rows = torch.arange(n, device=dev).repeat_interleave(per_row)
    cols = torch.randint(0, d, (n * per_row,), generator=g, device=dev)
    key = torch.unique(rows * d + cols)                               # sorted, duplicates merged
    del rows, cols
    r, c = key // d, key % d
    vals = torch.empty(key.numel(), device=dev)
    for a in range(0, key.numel(), 10000000):
        vals[a:a + 10000000] = (U[r[a:a + 10000000]] * Vt[c[a:a + 10000000]]).sum(1)
    crow = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    crow[1:] = torch.cumsum(torch.bincount(r, minlength=n), 0)
    Xs = torch.sparse_csr_tensor(crow, c, vals, size=(n, d), check_invariants=False)
    del U, Vt, key, r
    W0 = torch.rand(n, k, generator=g, device=dev)
    T0 = torch.rand(k, d, generator=g, device=dev)
    torch.cuda.empty_cache()
    return Xs, W0, T0, k


def arm(R, eng, W0, T0, sweeps):
    W, T = W0.clone(), T0.clone()
    p = eng.params()
    _timed(eng, W, T, 1, p)                                           # warm-up
    a = eng.stats()['kernel_launches']
    ms = _timed(eng, W, T, sweeps, p)
    out = {'ms_per_sweep': ms, 'launches_per_sweep': (eng.stats()['kernel_launches'] - a) / sweeps,
           'final_rel_err': _rel_err(eng, W, T)}
    Wp, Tp = W0.clone(), T0.clone()
    out['t_half_step_ms'] = eng.profile_kernel('masked_t', Wp, Tp, iters=20)
    out['w_half_step_ms'] = eng.profile_kernel('masked_w', Wp, Tp, iters=20)
    return out


def run_shape(R, shape, Xs, W0, T0, k, w0, sweeps, reps, weights, dense):
    nnz = int(Xs.values().numel())
    n, d = int(Xs.shape[0]), int(Xs.shape[1])
    base = {'shape': shape, 'n': n, 'd': d, 'k': k, 'nnz': nnz, 'stored': nnz / (float(n) * d), 'dtype': 'float32',
            'w0': w0, 'sweeps': sweeps}
    recs = []
    for wname, wts in weights:
        engines = {0.0: R.RRIEngine(Xs, k, W_mat=wts), w0: R.RRIEngine(Xs, k, W_mat=wts, unstored_weight=w0)}
        res = {0.0: [], w0: []}
        for _ in range(reps):                                         # alternating arms
            for w in (0.0, w0):
                res[w].append(arm(R, engines[w], W0, T0, sweeps))
        for e in engines.values():
            e.close()
        rec = dict(base, weights=wname)
        rec['unstored_weight_0'] = res[0.0]
        rec['unstored_weight_w0'] = res[w0]
        m0 = min(r['ms_per_sweep'] for r in res[0.0])
        m1 = min(r['ms_per_sweep'] for r in res[w0])
        rec['ratio_w0_over_0'] = m1 / m0
        rec['extra_launches_per_sweep'] = res[w0][0]['launches_per_sweep'] - res[0.0][0]['launches_per_sweep']
        if dense:
            # the dense masked problem the sparse one stands for: X and M = w0 + (m - w0) at the stored entries, n x d
            Xd = Xs.to_dense()
            Md = torch.full((n, d), w0, device=Xd.device)
            vals = torch.ones(nnz, device=Xd.device) if wts is None else wts
            Md.view(-1)[(torch.arange(n, device=Xd.device).repeat_interleave(Xs.crow_indices().diff()) * d
                         + Xs.col_indices()).long()] = vals
            ed = R.RRIEngine(Xd, k, W_mat=Md)
            W, T = W0.clone(), T0.clone()
            p = ed.params()
            _timed(ed, W, T, 1, p)
            dms = _timed(ed, W, T, sweeps, p)
            rec['dense_masked_ieee'] = {'ms_per_sweep': dms, 'final_rel_err': _rel_err(ed, W, T)}
            ed.close()
            del Xd, Md, ed
            torch.cuda.empty_cache()
            rec['rel_err_gap_vs_dense'] = abs(res[w0][0]['final_rel_err'] - rec['dense_masked_ieee']['final_rel_err'])
            rec['speedup_vs_dense'] = dms / m1
        recs.append(rec)
        print(json.dumps(rec), flush=True)
    return recs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--shapes', default='cfg4,big')
    ap.add_argument('--w0', type=float, default=0.05)
    ap.add_argument('--sweeps', type=int, default=10)
    ap.add_argument('--reps', type=int, default=2)
    ap.add_argument('--no-dense', action='store_true')
    ap.add_argument('--out', default=None, help='directory for the JSON lines (default: stdout only)')
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device: this measurement needs the GPU')
    import rri_nmf_b200 as R
    dev = torch.device('cuda:0')
    info = gpu_info()
    print('gpu: %s' % info, flush=True)
    recs = []
    for shape in a.shapes.split(','):
        if shape == 'cfg4':
            Xs, W0, T0, k = cfg4_data(dev)
            v = Xs.values()
            weights = [('none', None), ('1+0.5r', 1.0 + 0.5 * v / v.mean())]
            recs += run_shape(R, shape, Xs, W0, T0, k, a.w0, a.sweeps, a.reps, weights, not a.no_dense)
        elif shape == 'big':
            Xs, W0, T0, k = big_data(dev)
            recs += run_shape(R, shape, Xs, W0, T0, k, a.w0, max(2, a.sweeps // 3), 1, [('none', None)], False)
        else:
            raise SystemExit('unknown shape %r' % shape)
        del Xs, W0, T0
        torch.cuda.empty_cache()
    for r in recs:
        r['gpu'] = info
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, 'sparse_implicit_bench.jsonl'), 'w') as f:
            for r in recs:
                f.write(json.dumps(r) + '\n')


if __name__ == '__main__':
    main()
