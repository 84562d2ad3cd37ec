"""NNDSVD initialisation of sparse X on the device: rri_spmm (the SpMM kernel of spmm_kernels.cu with leading dimensions
and column panels) against scipy on both sparse handle kinds, its determinism and its errors, and nmf() / the
estimators with init_on_device=True against the host initialisation."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from conftest import ROOT, relfro

sys.path.insert(0, os.path.join(ROOT, 'tools'))
from bench_sparse_zero import text_like      # noqa: E402

pytestmark = pytest.mark.gpu

WIDTHS = [1, 3, 17, 74, 138, 266]


@pytest.fixture(scope='module')
def R(cuda_device):
    import rri_nmf_b200
    return rri_nmf_b200


def zipf_csr(n=3000, d=2000, per_row=12, seed=0):
    """Zipf column popularity (the first columns hold far more than 1024 entries), one row longer than 1024 entries,
    empty rows 0..6 and empty columns d-5..d-1; sorted, duplicates merged"""
    rs = np.random.RandomState(seed)
    p = 1.0 / np.arange(1, d - 4)
    p /= p.sum()
    rows = np.repeat(np.arange(7, n), rs.poisson(per_row, n - 7))
    cols = rs.choice(d - 5, size=rows.size, p=p)
    rows = np.concatenate([rows, np.full(d - 5, 9)])
    cols = np.concatenate([cols, np.arange(d - 5)])
    X = sp.csr_matrix((rs.rand(rows.size) + 0.1, (rows, cols)), shape=(n, d))
    X.sum_duplicates()
    X.sort_indices()
    assert np.diff(X.indptr).max() > 1024 and np.bincount(X.indices, minlength=d).max() > 1024
    return X


def engine(R, X, kind, dtype, k=8):
    """(engine, matrix it applies as scipy fp64): kind in zero / observed / weighted"""
    dev = torch.device('cuda:0')
    Xt = R.RRIEngine.csr_tensor(X.indptr, X.indices, X.data, X.shape, dev, dtype)
    if kind == 'zero':
        return R.RRIEngine(Xt, k, order='hals', unstored='zero'), X
    if kind == 'observed':
        return R.RRIEngine(Xt, k), X
    w = np.random.RandomState(5).rand(X.nnz)
    Xw = X.copy()
    Xw.data = Xw.data * w
    return R.RRIEngine(Xt, k, W_mat=torch.from_numpy(w).to(dev)), Xw


def spmm(eng, transpose, B, ldb, Cm, ldc, width, boff=0, coff=0):
    es = B.element_size()
    return eng.lib.rri_spmm(eng.h, transpose, C.c_void_p(B.data_ptr() + boff * es), ldb,
                            C.c_void_p(Cm.data_ptr() + coff * es), ldc, width, eng._stream())


@pytest.mark.parametrize('dtype', [torch.float64, torch.float32])
@pytest.mark.parametrize('kind', ['zero', 'observed', 'weighted'])
def test_spmm_matches_scipy(R, kind, dtype):
    X = zipf_csr()
    eng, Xr = engine(R, X, kind, dtype)
    tol = 1e-12 if dtype == torch.float64 else 1e-5
    rs = np.random.RandomState(1)
    n, d = X.shape
    for width in WIDTHS:
        for transpose in (0, 1):
            rin, rout = (n, d) if transpose else (d, n)
            Bh = rs.rand(rin, width)
            ref = (Xr.T if transpose else Xr) @ Bh
            B = torch.from_numpy(Bh).to('cuda', dtype)
            Cm = torch.full((rout, width), float('nan'), dtype=dtype, device='cuda')
            R._lib.check(spmm(eng, transpose, B, width, Cm, width, width))
            assert relfro(Cm.cpu().numpy(), ref) <= tol, (width, transpose)
            P = eng.products()
            out = P.left(B) if transpose else P.right(B)
            assert tuple(out.shape) == (rout, width)
            assert relfro(out.cpu().numpy(), ref) <= tol, (width, transpose)
    eng.close()


@pytest.mark.parametrize('kind', ['zero', 'weighted'])
def test_spmm_column_panels_through_ld(R, kind):
    """C[:, 3:3+w] = X B[:, 8:8+w] inside wider operands; the other columns of C are left alone"""
    X = zipf_csr(seed=2)
    eng, Xr = engine(R, X, kind, torch.float64)
    n, d = X.shape
    rs = np.random.RandomState(3)
    for width in (17, 74, 266):
        Bh = rs.rand(d, width + 13)
        B = torch.from_numpy(Bh).cuda()
        Cm = torch.full((n, width + 9), -7.0, dtype=torch.float64, device='cuda')
        R._lib.check(spmm(eng, 0, B, width + 13, Cm, width + 9, width, boff=8, coff=3))
        got = Cm.cpu().numpy()
        assert relfro(got[:, 3:3 + width], Xr @ Bh[:, 8:8 + width]) <= 1e-12
        assert (got[:, :3] == -7.0).all() and (got[:, 3 + width:] == -7.0).all()
    eng.close()


def test_spmm_deterministic_and_sweeps_unchanged(R):
    """two identical calls give identical bits; block-order sweeps of a zero-filled handle give identical bits before and
    after rri_spmm calls on the same handle (the shared chunk slots and arrival counters are left clean)"""
    X = zipf_csr(seed=4)
    eng, _ = engine(R, X, 'zero', torch.float32, k=8)
    n, d = X.shape
    g = torch.Generator(device='cuda').manual_seed(0)
    W0 = torch.rand(n, 8, generator=g, device='cuda')
    T0 = torch.rand(8, d, generator=g, device='cuda')
    W1, T1 = W0.clone(), T0.clone()
    eng.sweeps(W1, T1, 3, eng.params())
    P = eng.products()
    for width in (5, 8, 74, 266):
        Q = torch.rand(d, width, generator=g, device='cuda')
        a, b = P.right(Q), P.right(Q)
        assert torch.equal(a, b)
        Q2 = torch.rand(n, width, generator=g, device='cuda')
        assert torch.equal(P.left(Q2), P.left(Q2))
    W2, T2 = W0.clone(), T0.clone()
    eng.sweeps(W2, T2, 3, eng.params())
    assert torch.equal(W1, W2) and torch.equal(T1, T2)
    eng.close()


def test_spmm_errors(R):
    X = zipf_csr(seed=5)
    n, d = X.shape
    eng, _ = engine(R, X, 'observed', torch.float64)
    B = torch.zeros(d, 16, dtype=torch.float64, device='cuda')
    Cm = torch.zeros(n, 16, dtype=torch.float64, device='cuda')
    for args in [(0, B, 16, Cm, 16, 0), (0, B, 16, Cm, 16, -3),        # width < 1
                 (0, B, 8, Cm, 16, 16), (0, B, 16, Cm, 15, 16),          # ld shorter than the width
                 (2, B, 16, Cm, 16, 16)]:                                 # no such orientation
        assert spmm(eng, *args) != 0
        assert len(R._lib.load().rri_last_error()) > 0
    assert eng.lib.rri_spmm(eng.h, 0, None, 16, C.c_void_p(Cm.data_ptr()), 16, 16, eng._stream()) != 0
    assert b'null' in eng.lib.rri_last_error()
    assert eng.lib.rri_spmm(eng.h, 0, C.c_void_p(B.data_ptr() + 4), 16, C.c_void_p(Cm.data_ptr()), 16, 8,
                            eng._stream()) != 0                           # misaligned operand
    assert b'aligned' in eng.lib.rri_last_error()
    with pytest.raises(ValueError):
        eng.products().right(torch.zeros(d + 1, 4, dtype=torch.float64, device='cuda'))
    eng.close()
    dense = R.RRIEngine(torch.rand(50, 40, dtype=torch.float64, device='cuda'), 4, order='hals')
    B = torch.zeros(40, 4, dtype=torch.float64, device='cuda')
    Cm = torch.zeros(50, 4, dtype=torch.float64, device='cuda')
    with pytest.raises(R._lib.RriError, match='sparse'):
        R._lib.check(spmm(dense, 0, B, 4, Cm, 4, 4))
    dense.close()


def test_cuda_sparse_without_engine_products_is_refused(R):
    from rri_nmf_b200._device_init import randomized_svd_torch
    X = text_like(200, 150, 0.05, 4, seed=1, device='cuda', dtype=torch.float64)
    with pytest.raises(ValueError):
        randomized_svd_torch(X, 4, random_state=0)


def _tl(n, d, density, k, seed):
    X = text_like(n, d, density, k, seed=seed, dtype=torch.float64)
    return sp.csr_matrix((X.values().numpy(), X.col_indices().numpy(), X.crow_indices().numpy()), shape=(n, d))


@pytest.mark.parametrize('init', ['nndsvd', 'nndsvda', 'nndsvdar'])
@pytest.mark.parametrize('case', ['zero_hals', 'observed_rri', 'observed_weighted'])
def test_nmf_device_init_equals_host_init(R, case, init):
    X = _tl(500, 320, 0.06, 6, seed=21)
    kw = dict(max_iter=5, random_state=3, init=init, eps_stop=-1.0, reset_topic_method=None, max_time=1e9)
    if case == 'zero_hals':
        kw.update(unstored='zero', update_order='hals')
    elif case == 'observed_weighted':
        Wm = X.copy()
        Wm.data = np.random.RandomState(2).rand(X.nnz) + 0.5
        kw.update(W_mat=Wm)
    a = R.nmf(X, 6, init_on_device=True, **kw)
    b = R.nmf(X, 6, init_on_device=False, **kw)
    assert 'init_on_device_s' in a['timing'] and 'init_on_device_s' not in b['timing']
    assert isinstance(a['W'], np.ndarray) and a['W'].dtype == np.float64
    assert relfro(a['W'], b['W']) <= 1e-6 and relfro(a['T'], b['T']) <= 1e-6, (relfro(a['W'], b['W']),
                                                                               relfro(a['T'], b['T']))


def test_cuda_sparse_tensor_initialised_on_device_by_default(R):
    Xh = _tl(400, 300, 0.05, 5, seed=3)
    Xd = R.RRIEngine.csr_tensor(Xh.indptr, Xh.indices, Xh.data, Xh.shape, torch.device('cuda:0'), torch.float64)
    out = R.nmf(Xd, 5, max_iter=2, random_state=0, unstored='zero', update_order='hals', reset_topic_method=None)
    assert 'init_on_device_s' in out['timing']
    assert isinstance(out['W'], torch.Tensor) and out['W'].is_cuda
    small = R.nmf(Xh, 5, max_iter=2, random_state=0, unstored='zero', update_order='hals', reset_topic_method=None)
    assert 'init_on_device_s' not in small['timing']          # small host input: the host path, as before
    assert relfro(out['W'].cpu().numpy(), small['W']) <= 1e-6


def test_tm_estimator_either_initialisation(R):
    from rri_nmf_b200 import NMF_TM_Estimator
    X = _tl(400, 350, 0.04, 6, seed=13)
    Xnew = _tl(120, 350, 0.04, 6, seed=14)
    kw = dict(handle_tfidf=True, handle_normalization=True, max_iter=5, update_order='hals', random_state=0)
    ed = NMF_TM_Estimator(400, 350, 6, nmf_kwargs={'init_on_device': True}, **kw).fit(X)
    eh = NMF_TM_Estimator(400, 350, 6, nmf_kwargs={'init_on_device': False}, **kw).fit(X)
    assert 'init_on_device_s' in ed.nmf_outputs['timing'] and 'init_on_device_s' not in eh.nmf_outputs['timing']
    assert relfro(ed.W, eh.W) <= 1e-6 and relfro(ed.T, eh.T) <= 1e-6
    assert abs(ed.score(Xnew) - eh.score(Xnew)) <= 1e-6


def test_rs_estimator_sparse_either_initialisation(R):
    from rri_nmf_b200 import NMF_RS_Estimator
    X = _tl(300, 200, 0.08, 5, seed=31)
    I, J = X.nonzero()
    ij = np.column_stack([I, J])
    y = np.asarray(X[I, J]).ravel()
    kw = dict(max_iter=5, random_state=0, sparse=True, use_validation_early_stopping=False)
    ed = NMF_RS_Estimator(300, 200, 5, nmf_kwargs={'init_on_device': True}, **kw).fit(ij, y)
    eh = NMF_RS_Estimator(300, 200, 5, nmf_kwargs={'init_on_device': False}, **kw).fit(ij, y)
    assert 'init_on_device_s' in ed.nmf_outputs['timing'] and 'init_on_device_s' not in eh.nmf_outputs['timing']
    assert relfro(ed.W, eh.W) <= 1e-6 and relfro(ed.T, eh.T) <= 1e-6
    assert abs(ed.score(ij, y) - eh.score(ij, y)) <= 1e-6


def test_beyond_dense_capacity_initialises_on_device(R):
    """1 000 000 x 1 000 000 with 1e7 stored entries (4 TB if dense), k = 16: the NNDSVD runs on the device and torch's
    allocations grow by less than 1 GB (the engine's own workspace is allocated outside torch)"""
    dev = torch.device('cuda:0')
    n = d = 1000000
    X = text_like(n, d, 1e-5, 16, seed=7, device=dev)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated(dev)
    torch.cuda.reset_peak_memory_stats(dev)
    out = R.nmf(X, 16, max_iter=1, random_state=0, unstored='zero', update_order='hals', reset_topic_method=None)
    torch.cuda.synchronize()
    assert 'init_on_device_s' in out['timing']
    assert torch.cuda.max_memory_allocated(dev) - base < (1 << 30), torch.cuda.max_memory_allocated(dev) - base
    assert bool(torch.isfinite(out['W']).all()) and bool(torch.isfinite(out['T']).all())
    assert float(out['T'].sum()) > 0
