"""NNDSVD initialisation of sparse X on the device (rri_spmm through RRIEngine.products, _device_init.py) against the
host initialisation (`_host.initialize_nmf`: sklearn's randomized_svd on the scipy matrix).

    python tools/bench_sparse_init.py [--cases cfg3,cfg4,big] [--densities 0.001,0.01,0.05] [--dtypes f32,f64]
                                      [--sweeps 50] [--out DIR]

The matrices come from `text_like` of tools/bench_sparse_zero.py (seeded, Zipf column popularity, planted rank-k
values; nothing is downloaded).  Cases:
    cfg3  200 000 x 20 000, k = 64, zero-filled (unstored='zero', block order), at each density and dtype
    cfg4  100 000 x 20 000, k = 50, fp32, 5 % nominal, observed entries (the recommender setting, interleaved order)
    big   2 000 000 x 200 000, k = 64, fp32, 0.05 % nominal, zero-filled: device only (the host SVD takes minutes)
Per case one JSON line: host initialize_nmf seconds (measured once), device initialisation seconds (median of 3, split
into the 2 n_iter + 2 sparse products and the rest: QR / SVD / NNDSVD steps), ms per rri_spmm at width k + 10 (padded
to a 16-byte row as RRIEngine.products does; CUDA events, median of 20 launches per orientation), the end-to-end
nmf(..., max_iter=--sweeps) wall time with each initialisation, and the relative gap between the final
reconstruction errors of the two runs.  The GPU name, power limit and max SM clock are read in the same call."""
import argparse
import json
import os
import sys
import time

import numpy as np
import scipy.sparse as sp
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))

from bench_sparse_zero import gpu_info, text_like      # noqa: E402


class _TimedProducts(object):
    """the engine's products with a device synchronise around each call: seconds spent in them"""

    def __init__(self, P):
        self.P, self.s, self.calls = P, 0.0, 0

    def _run(self, f, Q):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = f(Q)
        torch.cuda.synchronize()
        self.s += time.perf_counter() - t0
        self.calls += 1
        return out

    def right(self, Q):
        return self._run(self.P.right, Q)

    def left(self, Q):
        return self._run(self.P.left, Q)


def _spmm_ms(R, eng, width, dtype, iters=20):
    """median ms of one rri_spmm launch per orientation at `width` columns, padded as RRIEngine.products pads"""
    import ctypes as C
    v = 16 // torch.tensor([], dtype=dtype).element_size()
    ld = (width + v - 1) // v * v
    out = {'width': width, 'ld': ld}
    for name, t, rin, rout in (('right', 0, eng.d, eng.n), ('left', 1, eng.n, eng.d)):
        B = torch.rand(rin, ld, device=eng.device, dtype=dtype)
        Cm = torch.empty(rout, ld, device=eng.device, dtype=dtype)
        args = (eng.h, t, C.c_void_p(B.data_ptr()), ld, C.c_void_p(Cm.data_ptr()), ld, ld, eng._stream())
        R._lib.check(eng.lib.rri_spmm(*args))                       # warm-up (and the first-call plan build)
        ts = []
        for _ in range(iters):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            R._lib.check(eng.lib.rri_spmm(*args))
            e1.record()
            e1.synchronize()
            ts.append(e0.elapsed_time(e1))
        out['ms_' + name] = float(np.median(ts))
    return out


def _scipy(X, dtype):
    Xc = X.cpu()
    return sp.csr_matrix((Xc.values().numpy().astype(dtype), Xc.col_indices().numpy().astype(np.int32),
                          Xc.crow_indices().numpy()), shape=tuple(X.shape))


def case(R, name, n, d, density, k, dtype, unstored, sweeps, host):
    from rri_nmf_b200._device_init import initialize_nmf_torch
    from rri_nmf_b200._host import initialize_nmf
    dev = torch.device('cuda:0')
    tdt = torch.float32 if dtype == 'f32' else torch.float64
    X = text_like(n, d, density, k, seed=1, device=dev, dtype=tdt)
    nnz = int(X.values().numel())
    rec = {'case': name, 'n': n, 'd': d, 'k': k, 'density': density, 'nnz': nnz, 'dtype': dtype, 'unstored': unstored}
    order = 'hals' if unstored == 'zero' else 'rri'
    eng = R.RRIEngine(X, k, order=order, unstored=unstored)
    rec['spmm'] = _spmm_ms(R, eng, k + 10, tdt)
    dev_s, prod_s, calls = [], [], 0
    for rep in range(4):                                              # one warm-up, then 3 timed
        P = _TimedProducts(eng.products())
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        W, T = initialize_nmf_torch(X, k, 'nndsvd', random_state=0, products=P)
        torch.cuda.synchronize()
        if rep:
            dev_s.append(time.perf_counter() - t0)
            prod_s.append(P.s)
        calls = P.calls
    del W, T
    eng.close()
    rec['device_init'] = {'s_median': float(np.median(dev_s)), 's_all': dev_s, 'products_s_median': float(np.median(prod_s)),
                          'qr_svd_nndsvd_s_median': float(np.median(np.array(dev_s) - np.array(prod_s))),
                          'products': calls}
    Xh = _scipy(X, np.float32 if dtype == 'f32' else np.float64)
    del X
    torch.cuda.empty_cache()
    if host:
        t0 = time.perf_counter()
        initialize_nmf(Xh, k, 'nndsvd', random_state=0)
        rec['host_init_s'] = time.perf_counter() - t0
        rec['init_speedup'] = rec['host_init_s'] / rec['device_init']['s_median']
    kw = dict(max_iter=sweeps, random_state=0, reset_topic_method=None, max_time=1e9, return_reconstruction_err=True)
    if unstored == 'zero':
        kw.update(update_order='hals', unstored='zero')
    e2e = {}
    for arm in (('device', 'host') if host else ('device',)):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = R.nmf(Xh, k, init_on_device=arm == 'device', **kw)
        torch.cuda.synchronize()
        e2e[arm] = {'s': time.perf_counter() - t0, 'init_on_device_s': out['timing'].get('init_on_device_s'),
                    'solve_s': out['timing'].get('solve_s'), 'reconstruction_err': out['reconstruction_err']}
    rec['e2e_%d_sweeps' % sweeps] = e2e
    if host:
        a, b = e2e['device']['reconstruction_err'], e2e['host']['reconstruction_err']
        rec['final_err_rel_gap'] = abs(a - b) / b
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--cases', default='cfg3,cfg4,big')
    ap.add_argument('--densities', default='0.001,0.01,0.05')
    ap.add_argument('--dtypes', default='f32,f64')
    ap.add_argument('--sweeps', type=int, default=50)
    ap.add_argument('--rows-scale', type=float, default=1.0, help='scale n (a quick rehearsal; the line then says so)')
    ap.add_argument('--out', default=None, help='directory for the JSON lines (default: stdout only)')
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('no CUDA device: this measurement needs the GPU')
    import rri_nmf_b200 as R
    info = gpu_info()
    print('gpu: %s' % info, flush=True)
    sc = a.rows_scale
    todo = []
    for c in a.cases.split(','):
        if c == 'cfg3':
            todo += [('cfg3', int(200000 * sc), 20000, float(x), 64, dt, 'zero', True)
                     for x in a.densities.split(',') for dt in a.dtypes.split(',')]
        elif c == 'cfg4':
            todo.append(('cfg4', int(100000 * sc), 20000, 0.05, 50, 'f32', 'missing', True))
        elif c == 'big':
            todo.append(('big', int(2000000 * sc), 200000, 0.0005, 64, 'f32', 'zero', False))
        else:
            raise SystemExit('unknown case %r' % c)
    recs = []
    for name, n, d, dens, k, dt, unstored, host in todo:
        rec = case(R, name, n, d, dens, k, dt, unstored, a.sweeps, host)
        rec['gpu'] = info
        if sc != 1.0:
            rec['rows_scale'] = sc
        recs.append(rec)
        print(json.dumps(rec), flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, 'sparse_init_bench.jsonl'), 'w') as f:
            for r in recs:
                f.write(json.dumps(r) + '\n')


if __name__ == '__main__':
    main()
