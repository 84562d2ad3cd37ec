"""Observed-entries data with rank-one weights on the unstored entries (RRIEngine(X_csr, k, unstored_weight=w0,
unstored_row_weight=a, unstored_col_weight=b), rri_set_unstored_weight_vectors) against the scalar-w0 call and against the
dense masked engine on the densified X and M.

    python tools/bench_sparse_implicit_vectors.py [--sweeps 10] [--reps 3] [--no-dense] [--out DIR]

Config-4 shape: 100 000 x 20 000, k = 50, fp32, 5 % nominal observed (the data of tools/bench_sparse_implicit.py),
w0 = 0.05.  b follows item popularity, b_j = f_j^alpha / mean(f^alpha) with f_j the stored entries of column j and
alpha = 0.5; a (user activity, the same rule over the rows) is given in the arm 'a+b' only.  Unweighted and with entry
weights 1 + 0.5 r (r = the stored value over its mean), the arms scalar w0 / b / a+b run alternating, --reps times each.
The dense masked engine (math='ieee', dense X and M = w0 a_i b_j off the stored entries: 16 GB) runs once on the
unweighted 'a+b' problem from the same start, for its time and the output gap.
Per arm: ms per sweep (CUDA events around --sweeps sweeps in one call, after one warm-up sweep), launches per sweep, the
time of one T- and one W-half-step of topic 0 (rri_profile_kernel 'masked_t' / 'masked_w', 20 launches each) and the
final relative error sqrt(2 obj / sum M x^2).  The GPU name, power limit and max SM clock are read in the same call."""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))
from bench_sparse_implicit import arm, cfg4_data                  # noqa: E402
from bench_sparse_zero import _rel_err, _timed, gpu_info          # noqa: E402


def popularity(counts, alpha):
    """f^alpha / mean(f^alpha): the item-popularity weights of He et al. (SIGIR 2016), scaled to mean 1"""
    p = counts.double() ** alpha
    return (p / p.mean()).float()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--w0', type=float, default=0.05)
    ap.add_argument('--alpha', type=float, default=0.5)
    ap.add_argument('--sweeps', type=int, default=10)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--no-dense', action='store_true')
    ap.add_argument('--out', default=None, help='directory for the JSON lines (default: stdout only)')
    o = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device: this measurement needs the GPU')
    import rri_nmf_b200 as R
    dev = torch.device('cuda:0')
    info = gpu_info()
    print('gpu: %s' % info, flush=True)
    Xs, W0, T0, k = cfg4_data(dev)
    n, d, nnz = int(Xs.shape[0]), int(Xs.shape[1]), int(Xs.values().numel())
    b = popularity(torch.bincount(Xs.col_indices().long(), minlength=d), o.alpha)
    a = popularity(Xs.crow_indices().diff(), o.alpha)
    v = Xs.values()
    base = {'shape': 'cfg4', 'n': n, 'd': d, 'k': k, 'nnz': nnz, 'dtype': 'float32', 'w0': o.w0, 'alpha': o.alpha,
            'sweeps': o.sweeps}
    vecs = {'scalar': (None, None), 'b': (None, b), 'a+b': (a, b)}
    recs = []
    for wname, wts in (('none', None), ('1+0.5r', 1.0 + 0.5 * v / v.mean())):
        engines = {name: R.RRIEngine(Xs, k, W_mat=wts, unstored_weight=o.w0, unstored_row_weight=ra,
                                     unstored_col_weight=cb) for name, (ra, cb) in vecs.items()}
        res = {name: [] for name in vecs}
        for _ in range(o.reps):                                       # alternating arms
            for name in vecs:
                res[name].append(arm(R, engines[name], W0, T0, o.sweeps))
        for e in engines.values():
            e.close()
        rec = dict(base, weights=wname, arms=res)
        best = {name: min(r['ms_per_sweep'] for r in res[name]) for name in vecs}
        rec['best_ms_per_sweep'] = best
        rec['ratio_b_over_scalar'] = best['b'] / best['scalar']
        rec['ratio_ab_over_scalar'] = best['a+b'] / best['scalar']
        rec['extra_launches_per_sweep_ab'] = res['a+b'][0]['launches_per_sweep'] - res['scalar'][0]['launches_per_sweep']
        if wname == 'none' and not o.no_dense:
            # the dense masked problem the sparse one stands for: X and M = w0 a_i b_j off the stored entries, 1 on them
            Xd = Xs.to_dense()
            Md = o.w0 * torch.outer(a, b)
            Md.view(-1)[(torch.arange(n, device=dev).repeat_interleave(Xs.crow_indices().diff()) * d
                         + Xs.col_indices()).long()] = 1.0
            ed = R.RRIEngine(Xd, k, W_mat=Md)
            W, T = W0.clone(), T0.clone()
            p = ed.params()
            _timed(ed, W, T, 1, p)
            dms = _timed(ed, W, T, o.sweeps, p)
            rec['dense_masked_ieee'] = {'ms_per_sweep': dms, 'final_rel_err': _rel_err(ed, W, T)}
            ed.close()
            del Xd, Md, ed
            torch.cuda.empty_cache()
            rec['rel_err_gap_vs_dense'] = abs(res['a+b'][0]['final_rel_err'] - rec['dense_masked_ieee']['final_rel_err'])
            rec['speedup_vs_dense'] = dms / best['a+b']
        rec['gpu'] = info
        recs.append(rec)
        print(json.dumps(rec), flush=True)
    if o.out:
        os.makedirs(o.out, exist_ok=True)
        with open(os.path.join(o.out, 'sparse_implicit_vectors_bench.jsonl'), 'w') as f:
            for r in recs:
                f.write(json.dumps(r) + '\n')


if __name__ == '__main__':
    main()
