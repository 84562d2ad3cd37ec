"""Zero-filled sparse data (nmf(..., unstored='zero'), RRIEngine(..., unstored='zero'), rri_bind_csr_zero): the block
order with the sparse x dense contraction of spmm_kernels.cu against the oracle on X.toarray(), against the dense
engine, its determinism, launch count, capacity beyond dense, transform(), the estimator and the argument errors."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import torch

import rri_oracle as orc
from conftest import ROOT, relfro

sys.path.insert(0, os.path.join(ROOT, 'tools'))
from bench_sparse_zero import text_like      # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def R(cuda_device):
    import rri_nmf_b200
    return rri_nmf_b200


def _scipy(X, dtype=np.float64):
    """scipy CSR copy of a torch sparse CSR tensor (generated on the CPU)"""
    return sp.csr_matrix((X.values().numpy().astype(dtype), X.col_indices().numpy(), X.crow_indices().numpy()),
                         shape=tuple(X.shape))


def _case(n, d, k, density=0.05, seed=0, dtype=np.float64):
    X = _scipy(text_like(n, d, density, k, seed=seed), dtype)
    from rri_nmf_b200._host import initialize_nmf
    W0, T0 = initialize_nmf(X, k, 'nndsvda', random_state=0)
    return X, W0.astype(dtype), T0.astype(dtype)


def _vs_oracle(R, X, k, W0, T0, sweeps, tol, **kw):
    Xd = X.toarray()
    for ns in range(1, sweeps + 1):
        o = orc.nmf_oracle(Xd, k, W0, T0, max_iter=ns, order='hals', **kw)
        g = R.nmf(X, k, W_in=W0, T_in=T0, max_iter=ns, update_order='hals', unstored='zero', reset_topic_method=None,
                  **kw)
        assert relfro(g['T'], o['T']) <= tol, (ns, relfro(g['T'], o['T']))
        assert relfro(g['W'], o['W']) <= tol, (ns, relfro(g['W'], o['W']))
        if 'obj_history' in o:
            assert np.allclose(g['obj_history'], o['obj_history'], rtol=tol, atol=0)
    return g, o


@pytest.mark.parametrize('k,kw', [
    (16, {}),
    (16, dict(reg_w_l1=0.01, reg_w_l2=0.1, reg_t_l1=0.02, reg_t_l2=0.2)),
    (16, dict(project_T_each_iter=True, t_row_sum=1.0)),     # fused simplex T update
    (7, dict(project_T_each_iter=True, t_row_sum=1.0)),      # per-topic chain (k odd)
    (12, dict(w_row_sum=1.0, do_final_project_W=True)),
    (9, dict(w_row_sum=1.0, project_W_each_iter=True)),
])
def test_parity_with_oracle_fp64(R, k, kw):
    """after each of sweeps 1..3 the factors are within 1e-9 of the oracle's block order on X.toarray()"""
    X, W0, T0 = _case(300, 517, k, seed=k)
    _vs_oracle(R, X, k, W0, T0, 3, 1e-9, **kw)


def test_same_as_dense_engine(R):
    """fp64: within 1e-9 of nmf(X.toarray(), update_order='hals', math='ieee'); fp32: final relative errors within 1e-4"""
    X, W0, T0 = _case(700, 900, 10, density=0.02, seed=3)
    kw = dict(W_in=W0, T_in=T0, max_iter=8, update_order='hals', reset_topic_method=None, return_reconstruction_err=True)
    g = R.nmf(X, 10, unstored='zero', **kw)
    o = R.nmf(X.toarray(), 10, math='ieee', **kw)
    assert relfro(g['W'], o['W']) <= 1e-9 and relfro(g['T'], o['T']) <= 1e-9
    assert abs(g['reconstruction_err'] / o['reconstruction_err'] - 1) <= 1e-9
    X32 = X.astype(np.float32)
    kw32 = dict(kw, W_in=W0.astype(np.float32), T_in=T0.astype(np.float32), max_iter=20)
    g = R.nmf(X32, 10, unstored='zero', **kw32)
    o = R.nmf(X32.toarray(), 10, math='ieee', **kw32)
    assert g['W'].dtype == np.float32
    xn = float(np.sqrt(X.multiply(X).sum()))
    assert abs(g['reconstruction_err'] - o['reconstruction_err']) / xn <= 1e-4


def test_objective_and_stopping_rule(R):
    X, W0, T0 = _case(400, 300, 8, seed=5)
    kw = dict(compute_obj_each_iter=True, eps_stop=1e-2, reg_w_l2=0.05)     # (the oracle stops after 11 sweeps)
    g, o = _vs_oracle(R, X, 8, W0, T0, 1, 1e-9, **kw)
    o = orc.nmf_oracle(X.toarray(), 8, W0, T0, max_iter=60, order='hals', **kw)
    g = R.nmf(X, 8, W_in=W0, T_in=T0, max_iter=60, update_order='hals', unstored='zero', reset_topic_method=None,
              return_reconstruction_err=True, **kw)
    assert len(g['obj_history']) == len(o['obj_history']) < 60
    assert np.allclose(g['obj_history'], o['obj_history'], rtol=1e-9, atol=0)
    # the calculator outlives the engine: it rebuilds a zero-filled block-order engine on demand
    assert abs(g['obj_calculator'].true_objective() / g['obj_history'][-1] - 1) <= 1e-9
    d = R.nmf(X.toarray(), 8, W_in=W0, T_in=T0, max_iter=60, update_order='hals', math='ieee',
              reset_topic_method=None, return_reconstruction_err=True, **kw)
    assert abs(g['reconstruction_err'] / d['reconstruction_err'] - 1) <= 1e-9


def _special_matrix():
    """200 100 x 3 000: column 7 stored in every non-empty row (chunked and fixed up), row 11 stored in every non-empty
    column, rows 20..29 and columns 100..109 empty, ~5 random entries per row otherwise"""
    rng = np.random.RandomState(0)
    n, d = 200100, 3000
    nr = 5 * n
    r = rng.randint(0, n, nr)
    c = rng.randint(0, d, nr)
    r = np.concatenate([r, np.arange(n), np.full(d, 11)])
    c = np.concatenate([c, np.full(n, 7), np.arange(d)])
    keep = ~(((r >= 20) & (r < 30)) | ((c >= 100) & (c < 110)))
    keep &= ~((r == 11) & (c >= 100) & (c < 110))
    X = sp.csr_matrix((rng.rand(keep.sum()) + 0.1, (r[keep], c[keep])), shape=(n, d))
    X.sum_duplicates()
    X.sort_indices()
    return X


@pytest.mark.parametrize('k', [1, 7, 64, 128])
def test_bitwise_reentrance_fp32(R, k):
    """4 sweeps in one call == 4 calls of one sweep, bit for bit (also run to run)"""
    X = _special_matrix()
    assert np.diff(X.tocsc().indptr).max() >= 200000
    dev = torch.device('cuda:0')
    Xt = R.RRIEngine.csr_tensor(X.indptr, X.indices, X.data, X.shape, dev, torch.float32)
    rng = np.random.RandomState(k)
    W0 = torch.from_numpy(rng.rand(X.shape[0], k).astype(np.float32) * 0.1).to(dev)
    T0 = torch.from_numpy(rng.rand(k, X.shape[1]).astype(np.float32) * 0.1).to(dev)
    eng = R.RRIEngine(Xt, k, order='hals', unstored='zero')
    assert eng.sparse and not eng.masked
    p = eng.params(reg_w_l2=0.01, reg_t_l2=0.01)
    W1, T1 = W0.clone(), T0.clone()
    eng.sweeps(W1, T1, 4, p)
    W2, T2 = W0.clone(), T0.clone()
    for _ in range(4):
        eng.sweeps(W2, T2, 1, p)
    W3, T3 = W0.clone(), T0.clone()
    eng.sweeps(W3, T3, 4, p)
    assert torch.equal(W1, W2) and torch.equal(T1, T2)
    assert torch.equal(W1, W3) and torch.equal(T1, T3)
    # empty rows / columns have a zero contraction: their factor entries collapse (up to the rounding of the
    # update's numerator, ~1e-32 in fp32)
    Wh, Th = W1.double().cpu().numpy(), T1.double().cpu().numpy()
    assert np.all(np.isfinite(Wh)) and np.all(np.isfinite(Th))
    assert np.abs(Wh[20:30]).max() <= 1e-20 and np.abs(Th[:, 100:110]).max() <= 1e-20
    eng.close()


def test_contraction_and_partials_against_host(R):
    """X T' / X' W through the profile and partials entry points, with a chunked column, vs scipy in fp64"""
    X = _special_matrix()
    k = 5
    dev = torch.device('cuda:0')
    Xt = R.RRIEngine.csr_tensor(X.indptr, X.indices, X.data, X.shape, dev, torch.float64)
    rng = np.random.RandomState(1)
    Wn, Tn = rng.rand(X.shape[0], k), rng.rand(k, X.shape[1])
    W, T = torch.from_numpy(Wn).to(dev), torch.from_numpy(Tn).to(dev)
    eng = R.RRIEngine(Xt, k, order='hals', unstored='zero')
    for t in (0, 3):
        wR, nw = eng.partials_T(W, T, t)
        assert nw.numel() == 1
        G = Wn.T @ Wn
        ref = X.T @ Wn[:, t] - sum(G[j, t] * Tn[j] for j in range(k) if j != t)
        assert relfro(wR.cpu().numpy(), ref) <= 1e-12
        assert abs(float(nw[0]) / G[t, t] - 1) <= 1e-12
    v = eng.objective_terms(W, T)
    xsq = X.multiply(X).sum()
    ref = 0.5 * (xsq - 2 * np.sum((X @ Tn.T) * Wn) + np.sum((Wn.T @ Wn) * (Tn @ Tn.T)))
    assert abs(v[0] / ref - 1) <= 1e-9
    assert abs(v[1] / X.multiply(X).sum() - 1) <= 1e-12
    for name in ('gemm_w', 'gemm_t', 'w_half', 't_half'):
        assert eng.profile_kernel(name, W.clone(), T.clone(), iters=2) > 0
    eng.close()


def test_launches_independent_of_k(R):
    dev = torch.device('cuda:0')
    X = text_like(3000, 2000, 0.01, 8, seed=2).to(dev)
    per = []
    for k in (8, 32):
        eng = R.RRIEngine(X, k, order='hals', unstored='zero')
        W = torch.rand(3000, k, device=dev)
        T = torch.rand(k, 2000, device=dev)
        a = eng.stats()['kernel_launches']
        eng.sweeps(W, T, 1, eng.params())
        per.append(eng.stats()['kernel_launches'] - a)
        eng.close()
    assert per[0] == per[1], per


def test_beyond_dense_capacity(R):
    """1 000 000 x 1 000 000 with 1e7 stored entries (4 TB if dense), k = 16, fp32"""
    dev = torch.device('cuda:0')
    n = d = 1000000
    X = text_like(n, d, 1e-5, 16, seed=7, device=dev)
    assert X.values().numel() > 5e6
    k = 16
    g = torch.Generator(device=dev).manual_seed(0)
    W = torch.rand(n, k, generator=g, device=dev) * 0.05
    T = torch.rand(k, d, generator=g, device=dev) * 0.05
    eng = R.RRIEngine(X, k, order='hals', unstored='zero')
    assert eng.stats()['workspace_bytes'] < (1 << 30)
    o0 = eng.objective(W, T)
    flags = eng.sweeps(W, T, 2, eng.params())
    o1 = eng.objective(W, T)
    assert o1 < o0 and np.isfinite(o1), (o0, o1, flags)
    assert eng.stats()['workspace_bytes'] < (1 << 30)
    eng.close()


@pytest.mark.parametrize('order', ['hals', 'rri'])
def test_transform_fix_T(R, order):
    X, W0, T0 = _case(300, 400, 6, seed=11)
    from rri_nmf_b200._host import normalize
    T0 = normalize(T0)
    kw = dict(max_iter=4, fix_T=True, T_in=T0, w_row_sum=1.0, t_row_sum=1.0, update_order=order, random_state=0)
    g = R.nmf(X, 6, unstored='zero', **kw)
    o = R.nmf(X.toarray(), 6, **kw)
    assert relfro(g['W'], o['W']) <= 1e-9
    assert np.array_equal(g['T'], o['T'])


def test_tm_estimator_hals_sparse_equals_dense(R):
    from rri_nmf_b200 import NMF_TM_Estimator
    X, _, _ = _case(400, 350, 6, density=0.03, seed=13)
    Xnew, _, _ = _case(120, 350, 6, density=0.03, seed=14)
    kw = dict(handle_tfidf=True, handle_normalization=True, max_iter=5, update_order='hals', random_state=0)
    es = NMF_TM_Estimator(400, 350, 6, **kw).fit(X)
    ed = NMF_TM_Estimator(400, 350, 6, **kw).fit(X.toarray())
    assert relfro(es.W, ed.W) <= 1e-9 and relfro(es.T, ed.T) <= 1e-9
    assert abs(es.reconstruction_err_ / ed.reconstruction_err_ - 1) <= 1e-9
    assert relfro(es.transform(Xnew), ed.transform(Xnew.toarray())) <= 1e-9
    assert abs(es.score(Xnew) - ed.score(Xnew.toarray())) <= 1e-9
    es.one_iter(X)
    ed.one_iter(X.toarray())
    assert relfro(es.T, ed.T) <= 1e-9


def test_tm_estimator_rri_densifies(R):
    from rri_nmf_b200 import NMF_TM_Estimator
    X, _, _ = _case(200, 150, 4, density=0.05, seed=15)
    kw = dict(handle_tfidf=True, handle_normalization=True, max_iter=3, random_state=0)
    es = NMF_TM_Estimator(200, 150, 4, **kw)
    ed = NMF_TM_Estimator(200, 150, 4, **kw)
    Ws = es.fit_transform(X)
    Wd = ed.fit_transform(X.toarray())
    assert np.array_equal(Ws, Wd) and np.array_equal(es.T, ed.T)
    assert np.array_equal(es.transform(X), ed.transform(X.toarray()))
    assert es.score(X) == ed.score(X.toarray())


def test_argument_errors(R):
    from rri_nmf_b200 import _lib
    X, W0, T0 = _case(100, 80, 4, seed=17)
    with pytest.raises(NotImplementedError, match="update_order='hals'.*toarray"):
        R.nmf(X, 4, W_in=W0, T_in=T0, max_iter=1, unstored='zero')
    with pytest.raises(ValueError, match='ieee'):
        R.nmf(X.astype(np.float32), 4, max_iter=1, unstored='zero', update_order='hals', math='tf32')
    with pytest.raises(ValueError, match='W_mat'):
        R.nmf(X, 4, max_iter=1, unstored='zero', update_order='hals', W_mat=X)
    with pytest.raises(ValueError, match='unstored'):
        R.nmf(X, 4, max_iter=1, unstored='nan', update_order='hals')
    dev = torch.device('cuda:0')
    crow = torch.tensor([0, 2, 3], dtype=torch.int64)
    bad_order = torch.sparse_csr_tensor(crow, torch.tensor([3, 1, 0]), torch.ones(3, dtype=torch.float64), size=(2, 5),
                                        check_invariants=False).to(dev)
    with pytest.raises(_lib.RriError, match='strictly ascending'):
        R.RRIEngine(bad_order, 2, order='hals', unstored='zero')
    bad_col = torch.sparse_csr_tensor(crow, torch.tensor([1, 5, 0]), torch.ones(3, dtype=torch.float64), size=(2, 5),
                                      check_invariants=False).to(dev)
    with pytest.raises(_lib.RriError, match=r'outside \[0,d\)'):
        R.RRIEngine(bad_col, 2, order='hals', unstored='zero')
    Xt = R.RRIEngine.csr_tensor(X.indptr, X.indices, X.data, X.shape, dev)
    eng = R.RRIEngine(Xt, 4, order='hals', unstored='zero')
    W = torch.rand(100, 4, device=dev, dtype=torch.float64)
    T = torch.rand(4, 80, device=dev, dtype=torch.float64)
    with pytest.raises(_lib.RriError, match='rri_topics'):
        eng.topics(W, T, 0, 1, eng.params())
    buf = (C.c_char * 64)()
    assert eng.lib.rri_peer_export(eng.h, buf) != 0
    assert b'NCCL all-reduce' in eng.lib.rri_last_error()
    eng.close()


def test_row_sharded_parity(cuda_device):
    ngpu = torch.cuda.device_count()
    if ngpu < 2:
        pytest.skip('needs 2 GPUs')
    r = subprocess.run([sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2',
                        '--master-addr', '127.0.0.1', '--master-port', '29541',
                        os.path.join(ROOT, 'tests', 'multi_gpu_sparse_zero_check.py')],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, universal_newlines=True, timeout=600)
    assert 'MULTI_GPU_SPARSE_ZERO PASS' in r.stdout, r.stdout[-3000:]
