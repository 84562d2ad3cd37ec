"""Block-order sweeps on zero-filled sparse data (RRIEngine(..., unstored='zero'), spmm_kernels.cu) against the dense
block order on the same matrix densified.

    python tools/bench_sparse_zero.py [--shapes cfg3,big] [--densities 0.001,0.01,0.05] [--sweeps 10] [--out DIR]

The matrix comes from `text_like`: a seeded document-term-like generator (nothing is downloaded).  Column popularity
follows a Zipf law (exponent 1), row lengths vary around density * d, and the stored values come from a planted
non-negative rank-k model plus noise, so the fit error actually falls.  Shapes:
    cfg3  200 000 x 20 000, k = 64, fp32, at each density (the config-3 shape of bench.py)
    big   2 000 000 x 200 000, k = 64, fp32, 0.05 % (nnz ≈ 1.6e8 once duplicates are merged; 1.6 TB if dense: the sparse run only)
Per case it prints one JSON line: ms per sweep (unconstrained and with project_T_each_iter), the SpMM time of each
half-step (CUDA events through rri_profile_kernel), achieved HBM and gather GB/s from the algorithmic bytes, launches
per sweep, the dense block order (TF32 and IEEE) on the densified matrix where it fits, and the final relative errors of
the sparse and the dense IEEE runs from the same start (they must agree within 1e-4).  The GPU name, power limit and
max SM clock are read in the same call."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def text_like(n, d, density, k, seed=0, device='cpu', dtype=torch.float32, noise=0.1):
    """Seeded document-term-like sparse matrix as a torch sparse CSR tensor on `device` (rows ascending, columns
    strictly ascending inside a row).  Zipf(1) column popularity over a seeded permutation of the columns, log-normal
    row lengths around density * d (duplicates merged), values W0[i] . H0[:, j] * (1 + noise * N(0, 1)), clipped at 0."""
    dev = torch.device(device)
    g = torch.Generator(device=dev).manual_seed(int(seed))
    p = 1.0 / torch.arange(1, d + 1, device=dev, dtype=torch.float64)
    cdf = torch.cumsum(p, 0)
    cdf = cdf / cdf[-1]
    perm = torch.randperm(d, generator=g, device=dev)
    z = torch.randn(n, generator=g, device=dev, dtype=torch.float64)
    lens = torch.round(density * d * torch.exp(0.5 * z - 0.125)).clamp_(0, d).to(torch.int64)
    total = int(lens.sum())
    rows = torch.repeat_interleave(torch.arange(n, device=dev), lens)
    u = torch.rand(total, generator=g, device=dev, dtype=torch.float64)
    cols = perm[torch.searchsorted(cdf, u).clamp_(max=d - 1)]
    key = torch.unique(rows * d + cols)                  # sorted: row-major order, duplicates merged
    del rows, cols, u
    rows, cols = key // d, key % d
    del key
    W0 = torch.rand(n, k, generator=g, device=dev, dtype=torch.float32) ** 2
    H0 = (torch.rand(k, d, generator=g, device=dev, dtype=torch.float32) ** 2).t().contiguous()
    val = torch.empty(rows.numel(), device=dev, dtype=torch.float32)
    step = 1 << 23
    for b in range(0, rows.numel(), step):
        e = min(b + step, rows.numel())
        v = (W0[rows[b:e]] * H0[cols[b:e]]).sum(1)
        val[b:e] = (v * (1 + noise * torch.randn(e - b, generator=g, device=dev))).clamp_(min=0)
    crow = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    crow[1:] = torch.cumsum(torch.bincount(rows, minlength=n), 0)
    del rows, W0, H0
    return torch.sparse_csr_tensor(crow, cols, val.to(dtype), size=(n, d), check_invariants=False)


def gpu_info():
    try:
        return subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                              stdout=subprocess.PIPE, universal_newlines=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as ex:
        return 'nvidia-smi unavailable (%s)' % ex


def _timed(eng, W, T, n, params):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    eng.sweeps(W, T, n, params)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / n


def _rel_err(eng, W, T):
    v = eng.objective_terms(W, T)
    return float(np.sqrt(2.0 * v[0] / v[1]))


def run_engine(R, eng, W0, T0, sweeps, halves):
    """ms / sweep unconstrained and with the simplex-constrained T update, the final relative error of the
    unconstrained run, launches per sweep and (halves) the SpMM / half-step times"""
    out = {}
    W, T = W0.clone(), T0.clone()
    free = eng.params()
    _timed(eng, W.clone(), T.clone(), 1, free)                         # warm-up
    a = eng.stats()['kernel_launches']
    out['ms_per_sweep'] = _timed(eng, W, T, sweeps, free)
    out['launches_per_sweep'] = (eng.stats()['kernel_launches'] - a) / sweeps
    out['final_rel_err'] = _rel_err(eng, W, T)
    Wc, Tc = W0.clone(), T0.clone()
    eng.project_rows_simplex(Tc, 1.0)
    cons = eng.params(ub_t=1.0, simplex_T=True)
    _timed(eng, Wc, Tc, 1, cons)
    out['ms_per_sweep_simplex_T'] = _timed(eng, Wc, Tc, sweeps, cons)
    if halves:
        for name in ('gemm_w', 'gemm_t', 'w_half', 't_half'):
            out['ms_' + name] = eng.profile_kernel(name, W.clone(), T.clone(), iters=20)
    return out


def case(R, shape, n, d, density, k, sweeps, dense_ok):
    dev = torch.device('cuda:0')
    X = text_like(n, d, density, k, seed=1, device=dev)
    nnz = int(X.values().numel())
    g = torch.Generator(device=dev).manual_seed(2)
    # uniform start whose product has the mean of X over all n * d entries
    scale = 2.0 * float(np.sqrt(X.values().double().mean().item() * nnz / (float(n) * d) / k)) or 1.0
    W0 = (torch.rand(n, k, generator=g, device=dev) * scale).contiguous()
    T0 = (torch.rand(k, d, generator=g, device=dev) * scale).contiguous()
    rec = {'shape': shape, 'n': n, 'd': d, 'k': k, 'density': density, 'nnz': nnz, 'dtype': 'float32',
           'sweeps': sweeps}
    eng = R.RRIEngine(X, k, order='hals', unstored='zero')
    rec['workspace_bytes'] = eng.stats()['workspace_bytes']
    rec['sparse'] = run_engine(R, eng, W0, T0, sweeps, True)
    eng.close()
    s = 4
    # algorithmic bytes per half-step: value + index streams, segment pointers, output, one read of the gathered factor
    hbm_w = nnz * (s + 4) + (n + 1) * 8 + n * k * s + d * k * s
    hbm_t = nnz * (s + 4) + (d + 1) * 8 + d * k * s + n * k * s
    gather = nnz * k * s
    sp_ = rec['sparse']
    rec['bytes'] = {'hbm_w_half': hbm_w, 'hbm_t_half': hbm_t, 'gather_per_half': gather,
                    'gathered_factor_w_half': d * k * s, 'gathered_factor_t_half': n * k * s}
    rec['achieved_GBps'] = {'hbm_w': hbm_w / sp_['ms_gemm_w'] / 1e6, 'hbm_t': hbm_t / sp_['ms_gemm_t'] / 1e6,
                            'gather_w': gather / sp_['ms_gemm_w'] / 1e6, 'gather_t': gather / sp_['ms_gemm_t'] / 1e6}
    if dense_ok:
        Xd = X.to_dense()
        del X
        for math in ('tf32', 'ieee'):
            e2 = R.RRIEngine(Xd, k, order='hals', math=math)
            rec['dense_' + math] = run_engine(R, e2, W0, T0, sweeps, False)
            e2.close()
            torch.cuda.empty_cache()
        del Xd
        rec['rel_err_diff_vs_dense_ieee'] = abs(sp_['final_rel_err'] - rec['dense_ieee']['final_rel_err'])
        rec['outputs_agree'] = rec['rel_err_diff_vs_dense_ieee'] <= 1e-4
        rec['speedup_vs_dense_tf32'] = rec['dense_tf32']['ms_per_sweep'] / sp_['ms_per_sweep']
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--shapes', default='cfg3,big')
    ap.add_argument('--densities', default='0.001,0.01,0.05')
    ap.add_argument('--sweeps', type=int, default=10)
    ap.add_argument('--out', default=None, help='directory for the JSON lines (default: stdout only)')
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device: this measurement needs the GPU')
    import rri_nmf_b200 as R
    info = gpu_info()
    print('gpu: %s' % info, flush=True)
    recs = []
    for shape in a.shapes.split(','):
        if shape == 'cfg3':
            cases = [(200000, 20000, float(x), 64, True) for x in a.densities.split(',')]
        elif shape == 'big':
            cases = [(2000000, 200000, 0.0005, 64, False)]
        else:
            raise SystemExit('unknown shape %r' % shape)
        for n, d, dens, k, dense_ok in cases:
            rec = case(R, shape, n, d, dens, k, a.sweeps, dense_ok)
            rec['gpu'] = info
            recs.append(rec)
            print(json.dumps(rec), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, 'sparse_zero_bench.jsonl'), 'w') as f:
            for r in recs:
                f.write(json.dumps(r) + '\n')


if __name__ == '__main__':
    main()
