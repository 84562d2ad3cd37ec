"""The interleaved order on zero-filled sparse data (nmf(..., unstored='zero', update_order='rri'),
RRIEngine(..., order='rri', unstored='zero'), sparse_rri_pass_kernel): against the oracle's interleaved order on
X.toarray(), against the dense engine, its determinism, statistics, objective, topic reset, the estimator, launch count,
capacity beyond dense and the argument policy."""
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import torch

import rri_oracle as orc
from conftest import ROOT, golden, relfro
from test_gpu_sparse_zero import _case, _special_matrix

sys.path.insert(0, os.path.join(ROOT, 'tools'))
from bench_sparse_zero import text_like      # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def R(cuda_device):
    import rri_nmf_b200
    return rri_nmf_b200


def _vs_oracle(R, X, k, W0, T0, sweeps, tol, **kw):
    Xd = X.toarray()
    for ns in range(1, sweeps + 1):
        o = orc.nmf_oracle(Xd, k, W0, T0, max_iter=ns, order='rri', **kw)
        g = R.nmf(X, k, W_in=W0, T_in=T0, max_iter=ns, update_order='rri', unstored='zero', reset_topic_method=None,
                  **kw)
        assert relfro(g['T'], o['T']) <= tol, (ns, relfro(g['T'], o['T']))
        assert relfro(g['W'], o['W']) <= tol, (ns, relfro(g['W'], o['W']))
        if 'obj_history' in o:
            assert np.allclose(g['obj_history'], o['obj_history'], rtol=tol, atol=0)
    return g, o


@pytest.mark.parametrize('k,kw', [
    (16, {}),
    (16, dict(reg_w_l1=0.01, reg_w_l2=0.1, reg_t_l1=0.02, reg_t_l2=0.2)),
    (16, dict(project_T_each_iter=True, t_row_sum=1.0)),
    (12, dict(w_row_sum=1.0, do_final_project_W=True)),
    (9, dict(w_row_sum=1.0, project_W_each_iter=True)),
    (7, {}),
    (1, {}),
])
def test_parity_with_oracle_fp64(R, k, kw):
    """after each of sweeps 1..3 the factors are within 1e-9 of the oracle's interleaved order on X.toarray()"""
    X, W0, T0 = _case(300, 517, k, seed=k)
    _vs_oracle(R, X, k, W0, T0, 3, 1e-9, **kw)


def test_same_as_dense_engine(R):
    """fp64: within 1e-9 of nmf(X.toarray(), update_order='rri'); fp32: final relative errors within 1e-4"""
    X, W0, T0 = _case(700, 900, 10, density=0.02, seed=3)
    kw = dict(W_in=W0, T_in=T0, max_iter=8, update_order='rri', reset_topic_method=None, return_reconstruction_err=True)
    g = R.nmf(X, 10, unstored='zero', **kw)
    o = R.nmf(X.toarray(), 10, **kw)
    assert relfro(g['W'], o['W']) <= 1e-9 and relfro(g['T'], o['T']) <= 1e-9
    assert abs(g['reconstruction_err'] / o['reconstruction_err'] - 1) <= 1e-9
    X32 = X.astype(np.float32)
    kw32 = dict(kw, W_in=W0.astype(np.float32), T_in=T0.astype(np.float32), max_iter=20)
    g = R.nmf(X32, 10, unstored='zero', **kw32)
    o = R.nmf(X32.toarray(), 10, **kw32)
    assert g['W'].dtype == np.float32
    xn = float(np.sqrt(X.multiply(X).sum()))
    assert abs(g['reconstruction_err'] - o['reconstruction_err']) / xn <= 1e-4


@pytest.mark.parametrize('k', [1, 7, 64])
def test_bitwise_reentrance_fp32(R, k):
    """4 sweeps in one call == 4 calls of one sweep == a second run, bit for bit, on a matrix with a chunked column,
    a row stored in every column and empty rows and columns"""
    X = _special_matrix()
    assert np.diff(X.tocsc().indptr).max() >= 200000
    dev = torch.device('cuda:0')
    Xt = R.RRIEngine.csr_tensor(X.indptr, X.indices, X.data, X.shape, dev, torch.float32)
    rng = np.random.RandomState(k)
    W0 = torch.from_numpy(rng.rand(X.shape[0], k).astype(np.float32) * 0.1).to(dev)
    T0 = torch.from_numpy(rng.rand(k, X.shape[1]).astype(np.float32) * 0.1).to(dev)
    eng = R.RRIEngine(Xt, k, order='rri', unstored='zero')
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
    Wh, Th = W1.double().cpu().numpy(), T1.double().cpu().numpy()
    assert np.all(np.isfinite(Wh)) and np.all(np.isfinite(Th))
    assert np.abs(Wh[20:30]).max() <= 1e-20 and np.abs(Th[:, 100:110]).max() <= 1e-20
    eng.close()


def test_statistics_against_scipy(R):
    """partials_T, the objective terms and both products of an rri-order engine, with a chunked column, vs scipy in
    fp64; the fused pass can be timed"""
    X = _special_matrix()
    k = 5
    dev = torch.device('cuda:0')
    Xt = R.RRIEngine.csr_tensor(X.indptr, X.indices, X.data, X.shape, dev, torch.float64)
    rng = np.random.RandomState(1)
    Wn, Tn = rng.rand(X.shape[0], k), rng.rand(k, X.shape[1])
    W, T = torch.from_numpy(Wn).to(dev), torch.from_numpy(Tn).to(dev)
    eng = R.RRIEngine(Xt, k, order='rri', unstored='zero')
    G = Wn.T @ Wn
    for t in (0, 3):
        wR, nw = eng.partials_T(W, T, t)
        ref = X.T @ Wn[:, t] - sum(G[j, t] * Tn[j] for j in range(k) if j != t)
        assert relfro(wR.cpu().numpy(), ref) <= 1e-12
        assert abs(float(nw[0]) / G[t, t] - 1) <= 1e-12
    v = eng.objective_terms(W, T)
    xsq = X.multiply(X).sum()
    ref = 0.5 * (xsq - 2 * np.sum((X @ Tn.T) * Wn) + np.sum((Wn.T @ Wn) * (Tn @ Tn.T)))
    assert abs(v[0] / ref - 1) <= 1e-9 and abs(v[1] / xsq - 1) <= 1e-12
    P = eng.products()
    assert relfro(P.right(T.t()).cpu().numpy(), X @ Tn.T) <= 1e-12
    assert relfro(P.left(W).cpu().numpy(), X.T @ Wn) <= 1e-12
    assert eng.profile_kernel('rri_pass', W.clone(), T.clone(), iters=3) > 0
    eng.close()


def test_objective_and_stopping_rule(R):
    X, W0, T0 = _case(400, 300, 8, seed=5)
    kw = dict(compute_obj_each_iter=True, eps_stop=1e-2, reg_w_l2=0.05)
    o = orc.nmf_oracle(X.toarray(), 8, W0, T0, max_iter=60, order='rri', **kw)
    g = R.nmf(X, 8, W_in=W0, T_in=T0, max_iter=60, update_order='rri', unstored='zero', reset_topic_method=None,
              return_reconstruction_err=True, **kw)
    assert len(g['obj_history']) == len(o['obj_history']) < 60
    assert np.allclose(g['obj_history'], o['obj_history'], rtol=1e-9, atol=0)
    assert relfro(g['W'], o['W']) <= 1e-9 and relfro(g['T'], o['T']) <= 1e-9
    # the calculator outlives the engine: it rebuilds a zero-filled engine on demand
    assert abs(g['obj_calculator'].true_objective() / g['obj_history'][-1] - 1) <= 1e-9


def test_topic_reset_golden_all_entries_stored(R):
    """the X of reset_rri_f64.npz as CSR with every entry stored reproduces the unmodified reference's run, in which a
    topic empties in the first sweep and is re-seeded from the max-residual document"""
    g = golden('reset_rri_f64.npz')
    rs = np.random.RandomState(33 + 57)
    X, W0, T0 = rs.rand(33, 57), rs.rand(33, 8), rs.rand(8, 57)
    Xs = sp.csr_matrix(X)
    assert Xs.nnz == X.size
    out = R.nmf(Xs, 8, W_in=W0, T_in=T0, max_iter=6, compute_obj_each_iter=True, eps_stop=-1.0, unstored='zero',
                update_order='rri')
    assert np.allclose(out['obj_history'], g['obj_history'], rtol=1e-9, atol=0)
    assert relfro(out['W'], g['W']) <= 1e-9 and relfro(out['T'], g['T']) <= 1e-9


@pytest.mark.parametrize('method', ['max_resid_document', 'random'])
def test_topic_reset_with_zeros_equals_dense(R, monkeypatch, method):
    """on a matrix with unstored zeros where a topic empties (the oracle, which applies no reset, raises), the sparse
    run re-seeds it exactly as the dense device path does"""
    nmf_mod = sys.modules['rri_nmf_b200.nmf']          # (the package exports the function under the same name)
    rs = np.random.RandomState(33 + 57)
    X, W0, T0 = rs.rand(33, 57), rs.rand(33, 8), rs.rand(8, 57)
    X[X < 0.4] = 0
    with pytest.raises(ValueError):
        orc.nmf_oracle(X, 8, W0, T0, max_iter=6)
    calls = []
    inner = nmf_mod.max_resid_document_sparse
    monkeypatch.setattr(nmf_mod, 'max_resid_document_sparse', lambda *a, **k: calls.append(1) or inner(*a, **k))
    kw = dict(W_in=W0, T_in=T0, max_iter=6, compute_obj_each_iter=True, eps_stop=-1.0, update_order='rri',
              reset_topic_method=method, fix_reset_seed=True)
    s = R.nmf(sp.csr_matrix(X), 8, unstored='zero', **kw)
    d = R.nmf(X, 8, **kw)
    if method == 'max_resid_document':
        assert len(calls) >= 1
    assert np.allclose(s['obj_history'], d['obj_history'], rtol=1e-9, atol=0)
    assert relfro(s['W'], d['W']) <= 1e-9 and relfro(s['T'], d['T']) <= 1e-9


def test_tm_estimator_sparse_equals_dense(R):
    from rri_nmf_b200 import NMF_TM_Estimator
    X, _, _ = _case(400, 350, 6, density=0.03, seed=13)
    Xnew, _, _ = _case(120, 350, 6, density=0.03, seed=14)
    kw = dict(handle_tfidf=True, handle_normalization=True, max_iter=5, random_state=0)
    es = NMF_TM_Estimator(400, 350, 6, sparse=True, **kw).fit(X)
    ed = NMF_TM_Estimator(400, 350, 6, **kw).fit(X.toarray())
    assert relfro(es.W, ed.W) <= 1e-9 and relfro(es.T, ed.T) <= 1e-9
    assert abs(es.reconstruction_err_ / ed.reconstruction_err_ - 1) <= 1e-9
    assert relfro(es.transform(Xnew), ed.transform(Xnew.toarray())) <= 1e-9
    assert abs(es.score(Xnew) - ed.score(Xnew.toarray())) <= 1e-9
    es.one_iter(X)
    ed.one_iter(X.toarray())
    assert relfro(es.W, ed.W) <= 1e-9 and relfro(es.T, ed.T) <= 1e-9


def test_tm_estimator_sparse_never_densifies(R, monkeypatch):
    from rri_nmf_b200 import NMF_TM_Estimator
    X, _, _ = _case(300, 250, 5, density=0.04, seed=23)

    def refuse(self, *a, **k):
        raise AssertionError('X was densified')
    for cls in (sp.csr_matrix, sp.csc_matrix, sp.coo_matrix):
        monkeypatch.setattr(cls, 'toarray', refuse)
        monkeypatch.setattr(cls, 'todense', refuse)
    e = NMF_TM_Estimator(300, 250, 5, sparse=True, handle_tfidf=True, handle_normalization=True, max_iter=3,
                         random_state=0).fit(X)
    assert np.all(np.isfinite(e.W)) and np.isfinite(e.score(X))
    R.nmf(X, 5, max_iter=2, unstored='zero', update_order='rri', random_state=0)


def test_launches_per_sweep(R):
    """3 launches per topic and sweep (T-step, fused pass, W-step) plus a constant per call"""
    dev = torch.device('cuda:0')
    X = text_like(3000, 2000, 0.01, 8, seed=2).to(dev)
    extra = []
    for k in (8, 32):
        eng = R.RRIEngine(X, k, order='rri', unstored='zero')
        W = torch.rand(3000, k, device=dev)
        T = torch.rand(k, 2000, device=dev)
        per = []
        for ns in (1, 3):
            a = eng.stats()['kernel_launches']
            eng.sweeps(W, T, ns, eng.params())
            per.append(eng.stats()['kernel_launches'] - a)
        assert per[1] - per[0] == 2 * 3 * k, (k, per)
        extra.append(per[0] - 3 * k)
        eng.close()
    assert extra[0] == extra[1], extra


def test_beyond_dense_capacity(R):
    """1 000 000 x 1 000 000 with 1e7 stored entries (4 TB if dense), k = 16, fp32, interleaved order"""
    dev = torch.device('cuda:0')
    n = d = 1000000
    X = text_like(n, d, 1e-5, 16, seed=7, device=dev)
    assert X.values().numel() > 5e6
    k = 16
    g = torch.Generator(device=dev).manual_seed(0)
    W = torch.rand(n, k, generator=g, device=dev) * 0.05
    T = torch.rand(k, d, generator=g, device=dev) * 0.05
    eng = R.RRIEngine(X, k, order='rri', unstored='zero')
    assert eng.stats()['workspace_bytes'] < (1 << 30)
    o0 = eng.objective(W, T)
    flags = eng.sweeps(W, T, 1, eng.params())
    o1 = eng.objective(W, T)
    assert o1 < o0 and np.isfinite(o1), (o0, o1, flags)
    assert eng.stats()['workspace_bytes'] < (1 << 30)
    eng.close()


def test_argument_policy(R):
    X, W0, T0 = _case(100, 80, 4, seed=17)
    with pytest.raises(ValueError, match='ieee'):
        R.nmf(X.astype(np.float32), 4, max_iter=1, unstored='zero', update_order='rri', math='tf32')
    dev = torch.device('cuda:0')
    Xt = R.RRIEngine.csr_tensor(X.indptr, X.indices, X.data, X.shape, dev)
    eng = R.RRIEngine(Xt, 4, order='rri', unstored='zero')
    W = torch.from_numpy(W0).to(dev).contiguous()
    T = torch.from_numpy(T0).to(dev).contiguous()
    p = eng.params()
    W1, T1 = W.clone(), T.clone()
    eng.topics(W1, T1, 0, 2, p)
    eng.topics(W1, T1, 2, 4, p)
    W2, T2 = W.clone(), T.clone()
    eng.sweeps(W2, T2, 1, p)
    assert relfro(W1.cpu().numpy(), W2.cpu().numpy()) <= 1e-14 and relfro(T1.cpu().numpy(), T2.cpu().numpy()) <= 1e-14
    eng.close()


@pytest.mark.parametrize('init', ['nndsvd', 'nndsvda'])
def test_device_init_equals_host_init(R, init):
    X, _, _ = _case(500, 320, 6, density=0.06, seed=21)
    kw = dict(max_iter=5, random_state=3, init=init, eps_stop=-1.0, reset_topic_method=None, max_time=1e9,
              unstored='zero', update_order='rri')
    a = R.nmf(X, 6, init_on_device=True, **kw)
    b = R.nmf(X, 6, init_on_device=False, **kw)
    assert 'init_on_device_s' in a['timing'] and 'init_on_device_s' not in b['timing']
    assert relfro(a['W'], b['W']) <= 1e-6 and relfro(a['T'], b['T']) <= 1e-6


def test_row_sharded_parity(cuda_device):
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    r = subprocess.run([sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2',
                        '--master-addr', '127.0.0.1', '--master-port', '29543',
                        os.path.join(ROOT, 'tests', 'multi_gpu_sparse_rri_check.py')],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, universal_newlines=True, timeout=600)
    assert 'MULTI_GPU_SPARSE_RRI PASS' in r.stdout, r.stdout[-3000:]
