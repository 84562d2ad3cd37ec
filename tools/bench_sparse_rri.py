"""The interleaved (reference) order on zero-filled sparse data (RRIEngine(..., order='rri', unstored='zero'),
sparse_rri_kernels.cu) against the same order on the matrix densified and against the sparse block order.

    python tools/bench_sparse_rri.py [--shapes cfg3,big] [--densities 0.001,0.01,0.05] [--sweeps 10] [--out DIR]

Matrices come from `tools/bench_sparse_zero.text_like` (seeded, nothing is downloaded).  Shapes:
    cfg3  200 000 x 20 000, k = 64, fp32, at each density; the dense interleaved order runs on X.to_dense() (16 GB)
    big   2 000 000 x 200 000, k = 64, fp32, 0.05 % (1.6 TB if dense: the sparse runs only)
Per case one JSON line: ms per sweep (CUDA events, one warm-up sweep, then --sweeps timed sweeps in one call), the fused
pass's time (rri_profile_kernel which = 0, 20 launches), its algorithmic bytes with the HBM and gather rates, launches
per sweep, the sparse block order and the dense interleaved order, and the final relative errors of the sparse and the
dense interleaved runs from the same start, in fp32 and in fp64 (`rel_err_f64`: the same runs on the fp64 copies of X
and of the start, which separates the sparse path from the fp32 rounding of the iteration).  `launch_floor_ms_per_sweep` is a sweep of the same k on a 512 x 512
matrix with 2 % stored entries: the cost of the 3k + 3 launches alone.  The GPU name, power limit and max SM clock
are read in the same call."""
import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))
from bench_sparse_zero import _rel_err, _timed, gpu_info, text_like      # noqa: E402


def run(eng, W0, T0, sweeps):
    W, T = W0.clone(), T0.clone()
    p = eng.params()
    _timed(eng, W, T, 1, p)                                             # warm-up (the same start for every engine)
    a = eng.stats()['kernel_launches']
    ms = _timed(eng, W, T, sweeps, p)
    return {'ms_per_sweep': ms, 'launches_per_sweep': (eng.stats()['kernel_launches'] - a) / sweeps,
            'final_rel_err': _rel_err(eng, W, T)}, W, T


def case(R, shape, n, d, density, k, sweeps, dense_ok):
    dev = torch.device('cuda:0')
    X = text_like(n, d, density, k, seed=1, device=dev)
    nnz = int(X.values().numel())
    g = torch.Generator(device=dev).manual_seed(2)
    scale = 2.0 * float(np.sqrt(X.values().double().mean().item() * nnz / (float(n) * d) / k)) or 1.0
    W0 = (torch.rand(n, k, generator=g, device=dev) * scale).contiguous()
    T0 = (torch.rand(k, d, generator=g, device=dev) * scale).contiguous()
    s = 4
    rec = {'shape': shape, 'n': n, 'd': d, 'k': k, 'density': density, 'nnz': nnz, 'stored': nnz / (float(n) * d),
           'dtype': 'float32', 'sweeps': sweeps}
    eng = R.RRIEngine(X, k, order='rri', unstored='zero')
    rec['workspace_bytes'] = eng.stats()['workspace_bytes']
    rec['sparse_rri'], W, T = run(eng, W0, T0, sweeps)
    rec['pass_ms'] = eng.profile_kernel('rri_pass', W, T, iters=20)
    eng.close()
    # per topic: value + index streams of both orientations, their segment pointers, the two outputs
    hbm = 2 * nnz * (s + 4) + (n + d + 2) * 8 + (n + d) * s
    rec['bytes_per_pass'] = {'hbm': hbm, 'gather': 2 * nnz * s, 'per_sweep_hbm': k * hbm}
    rec['achieved_GBps'] = {'hbm': hbm / rec['pass_ms'] / 1e6, 'gather': 2 * nnz * s / rec['pass_ms'] / 1e6}
    rec['pass_share_of_sweep'] = k * rec['pass_ms'] / rec['sparse_rri']['ms_per_sweep']
    eng = R.RRIEngine(X, k, order='hals', unstored='zero')
    rec['sparse_hals'], _, _ = run(eng, W0, T0, sweeps)
    eng.close()
    if dense_ok:
        X64 = torch.sparse_csr_tensor(X.crow_indices(), X.col_indices(), X.values().double(), size=X.shape)
        Xd = X.to_dense()
        del X
        e2 = R.RRIEngine(Xd, k, order='rri')
        rec['dense_rri'], _, _ = run(e2, W0, T0, sweeps)
        e2.close()
        f64 = {}
        e2 = R.RRIEngine(Xd.double(), k, order='rri')
        f64['dense_rri'] = run(e2, W0.double(), T0.double(), sweeps)[0]['final_rel_err']
        e2.close()
        del Xd, e2
        torch.cuda.empty_cache()
        Xs = X64
        e2 = R.RRIEngine(Xs, k, order='rri', unstored='zero')
        f64['sparse_rri'] = run(e2, W0.double(), T0.double(), sweeps)[0]['final_rel_err']
        e2.close()
        f64['diff'] = abs(f64['sparse_rri'] - f64['dense_rri'])
        rec['rel_err_f64'] = f64
        rec['rel_err_diff_vs_dense_rri'] = abs(rec['sparse_rri']['final_rel_err'] - rec['dense_rri']['final_rel_err'])
        rec['outputs_agree'] = rec['rel_err_diff_vs_dense_rri'] <= 1e-4
        rec['speedup_vs_dense_rri'] = rec['dense_rri']['ms_per_sweep'] / rec['sparse_rri']['ms_per_sweep']
    rec['slowdown_vs_sparse_hals'] = rec['sparse_rri']['ms_per_sweep'] / rec['sparse_hals']['ms_per_sweep']
    torch.cuda.empty_cache()
    return rec


def launch_floor(R, k, sweeps):
    dev = torch.device('cuda:0')
    X = text_like(512, 512, 0.02, k, seed=3, device=dev)
    g = torch.Generator(device=dev).manual_seed(4)
    W0 = torch.rand(512, k, generator=g, device=dev) * 0.1
    T0 = torch.rand(k, 512, generator=g, device=dev) * 0.1
    eng = R.RRIEngine(X, k, order='rri', unstored='zero')
    out, _, _ = run(eng, W0, T0, sweeps)
    eng.close()
    return out


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
    floor = launch_floor(R, 64, a.sweeps)
    print(json.dumps({'launch_floor_k64': floor, 'gpu': info}), flush=True)
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
            rec['launch_floor_ms_per_sweep'] = floor['ms_per_sweep']
            rec['launch_floor_share'] = floor['ms_per_sweep'] / rec['sparse_rri']['ms_per_sweep']
            rec['gpu'] = info
            recs.append(rec)
            print(json.dumps(rec), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, 'sparse_rri_bench.jsonl'), 'w') as f:
            for r in recs:
                f.write(json.dumps(r) + '\n')


if __name__ == '__main__':
    main()
