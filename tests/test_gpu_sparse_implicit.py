"""Observed-entries data with a weight on the unstored entries (nmf(X_sparse, ..., unstored_weight=w0),
RRIEngine(..., unstored_weight=w0), rri_set_unstored_weight): against the oracle's masked iteration on the densified X and
M (M = w0 at every unstored entry), against the dense masked engine, its determinism, topics, initialisation, objective,
the recommender estimator and the ABI refusals."""
import ctypes as C
import importlib

import numpy as np
import pytest
import scipy.sparse as sp
import torch

import rri_oracle as orc
from conftest import relfro
from test_sparse_implicit_scheme_cpu import dense_M, implicit_case

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def R(cuda_device):
    import rri_nmf_b200
    return rri_nmf_b200


def _case(n, d, k, w0, weighted, density=0.12, seed=0, dtype=np.float64):
    """(X csr, weights csr or None, dense X, dense M, W0, T0)"""
    I, J, vals, wts, W0, T0 = implicit_case(n, d, k, density, seed, weighted, stored_zeros=5)
    X = sp.csr_matrix((vals, (I, J)), shape=(n, d), dtype=dtype)
    assert X.nnz == len(vals)                                   # the explicit zeros stay stored
    Wm = None if wts is None else sp.csr_matrix((wts, (I, J)), shape=(n, d), dtype=dtype)
    Xd = np.zeros((n, d))
    Xd[I, J] = vals
    return X, Wm, Xd, dense_M(I, J, n, d, w0, wts), W0.astype(dtype), T0.astype(dtype)


CASES = [
    ('rri', 0.05, False, 7, {}),
    ('rri', 0.5, True, 5, {}),
    ('rri', 2.0, True, 1, {}),
    ('hals', 1.0, False, 3, {}),
    ('hals', 0.3, True, 5, {}),
    ('rri', 0.2, True, 6, dict(reg_w_l1=0.01, reg_w_l2=0.1, reg_t_l1=0.02, reg_t_l2=0.2)),
    ('hals', 0.2, False, 6, dict(reg_w_l1=0.01, reg_w_l2=0.1, reg_t_l1=0.02, reg_t_l2=0.2)),
    ('rri', 0.1, False, 8, dict(project_T_each_iter=True, t_row_sum=1.0)),
    ('rri', 0.1, True, 6, dict(w_row_sum=1.0)),
    ('rri', 0.1, True, 5, dict(fix_T=True)),
    ('hals', 0.1, False, 5, dict(fix_T=True)),
]


@pytest.mark.parametrize('order,w0,weighted,k,kw', CASES)
def test_parity_with_oracle_fp64(R, order, w0, weighted, k, kw):
    """after each of sweeps 1..3 the factors, and the objective history, are within 1e-9 of the oracle's masked
    iteration on X.toarray() with the dense M"""
    X, Wm, Xd, M, W0, T0 = _case(300, 220, k, w0, weighted, seed=k)
    for ns in (1, 2, 3):
        o = orc.nmf_oracle(Xd, k, W0, T0, max_iter=ns, W_mat=M, order=order, compute_obj_each_iter=True, eps_stop=0,
                           **kw)
        g = R.nmf(X, k, W_mat=Wm, W_in=W0, T_in=T0, max_iter=ns, update_order=order, reset_topic_method=None,
                  compute_obj_each_iter=True, eps_stop=0, unstored_weight=w0, **kw)
        assert relfro(g['W'], o['W']) <= 1e-9, (ns, relfro(g['W'], o['W']))
        assert relfro(g['T'], o['T']) <= 1e-9, (ns, relfro(g['T'], o['T']))
        assert np.allclose(g['obj_history'], o['obj_history'], rtol=1e-9, atol=0)
    # the detached calculator rebuilds an engine with the same unstored weight
    regs = {a: b for a, b in kw.items() if a.startswith('reg')}
    assert abs(g['obj_calculator'].true_objective() / orc.objective(Xd, g['W'], g['T'], M, **regs) - 1) <= 1e-9


def test_objective_terms_and_reconstruction_error(R):
    X, Wm, Xd, M, W0, T0 = _case(260, 310, 6, 0.07, True, seed=3)
    g = R.nmf(X, 6, W_mat=Wm, W_in=W0, T_in=T0, max_iter=4, reset_topic_method=None, unstored_weight=0.07,
              return_reconstruction_err=True)
    ref = np.sqrt(np.sum(M * (Xd - g['W'].dot(g['T'])) ** 2))
    assert abs(g['reconstruction_err'] / ref - 1) <= 1e-9
    import rri_nmf_b200.engine as E
    Xt = E.RRIEngine.csr_tensor(X.indptr, X.indices, X.data, X.shape, 'cuda:0', torch.float64)
    eng = E.RRIEngine(Xt, 6, W_mat=torch.as_tensor(Wm.data, device='cuda:0'), unstored_weight=0.07)
    try:
        Wd, Td = torch.as_tensor(g['W'], device='cuda:0'), torch.as_tensor(g['T'], device='cuda:0')
        v = eng.objective_terms(Wd, Td)
    finally:
        eng.close()
    R2 = (Xd - g['W'].dot(g['T'])) ** 2
    want = [0.5 * np.sum(M * R2), np.sum(M * Xd ** 2), np.sum(g['W'] ** 2), np.abs(g['W']).sum(),
            np.sum(g['T'] ** 2), np.abs(g['T']).sum()]
    assert np.allclose(v, want, rtol=1e-9, atol=0)


@pytest.mark.parametrize('order', ['rri', 'hals'])
def test_same_as_dense_masked_engine(R, order):
    """fp64: within 1e-9 of nmf(X.toarray(), W_mat=M) on the dense masked engine; fp32: the final relative errors
    after 20 sweeps agree within 1e-4"""
    X, Wm, Xd, M, W0, T0 = _case(500, 420, 8, 0.05, True, density=0.08, seed=4)
    kw = dict(W_in=W0, T_in=T0, max_iter=6, update_order=order, reset_topic_method=None, return_reconstruction_err=True)
    g = R.nmf(X, 8, W_mat=Wm, unstored_weight=0.05, **kw)
    o = R.nmf(Xd, 8, W_mat=M, **kw)
    assert relfro(g['W'], o['W']) <= 1e-9 and relfro(g['T'], o['T']) <= 1e-9
    assert abs(g['reconstruction_err'] / o['reconstruction_err'] - 1) <= 1e-9
    kw32 = dict(kw, W_in=W0.astype(np.float32), T_in=T0.astype(np.float32), max_iter=20)
    g = R.nmf(X.astype(np.float32), 8, W_mat=Wm.astype(np.float32), unstored_weight=0.05, **kw32)
    o = R.nmf(Xd.astype(np.float32), 8, W_mat=M.astype(np.float32), **kw32)
    assert g['W'].dtype == np.float32
    xn = float(np.sqrt(np.sum(M * Xd ** 2)))
    assert abs(g['reconstruction_err'] - o['reconstruction_err']) / xn <= 1e-4


def test_zero_weight_is_bit_identical(R):
    """unstored_weight=0 is the plain observed-entries call: same bits"""
    X, Wm, _, _, W0, T0 = _case(400, 330, 7, 0.0, True, seed=6, dtype=np.float32)
    for order in ('rri', 'hals'):
        kw = dict(W_mat=Wm, W_in=W0, T_in=T0, max_iter=5, update_order=order, reset_topic_method=None)
        a = R.nmf(X, 7, **kw)
        b = R.nmf(X, 7, unstored_weight=0, **kw)
        assert np.array_equal(a['W'], b['W']) and np.array_equal(a['T'], b['T'])


def _engine(R, X, Wm, k, w0, order='rri', dtype=torch.float32):
    from rri_nmf_b200.engine import RRIEngine
    Xt = RRIEngine.csr_tensor(X.indptr, X.indices, X.data, X.shape, 'cuda:0', dtype)
    wt = None if Wm is None else torch.as_tensor(Wm.data, device='cuda:0', dtype=dtype)
    return RRIEngine(Xt, k, W_mat=wt, order=order, unstored_weight=w0)


@pytest.mark.parametrize('order', ['rri', 'hals'])
@pytest.mark.parametrize('weighted', [False, True])
def test_n_sweeps_in_one_call_equal_n_calls(R, order, weighted):
    X, Wm, _, _, W0, T0 = _case(700, 520, 9, 0.05, weighted, seed=8, dtype=np.float32)
    eng = _engine(R, X, Wm, 9, 0.05, order)
    try:
        p = eng.params()
        W1, T1 = torch.as_tensor(W0, device='cuda:0').clone(), torch.as_tensor(T0, device='cuda:0').clone()
        W2, T2 = W1.clone(), T1.clone()
        eng.sweeps(W1, T1, 4, p)
        for _ in range(4):
            eng.sweeps(W2, T2, 1, p)
        torch.cuda.synchronize()
        assert torch.equal(W1, W2) and torch.equal(T1, T2)
    finally:
        eng.close()


def test_refresh_every_8_fp64(R):
    X, Wm, _, _, W0, T0 = _case(600, 450, 8, 0.1, True, seed=9)
    kw = dict(W_mat=Wm, W_in=W0, T_in=T0, max_iter=10, reset_topic_method=None, unstored_weight=0.1, sweeps_per_call=10)
    a = R.nmf(X, 8, **kw)
    b = R.nmf(X, 8, sparse_refresh_every=8, **kw)
    assert relfro(b['W'], a['W']) <= 1e-9 and relfro(b['T'], a['T']) <= 1e-9


def test_topics_in_two_ranges(R):
    """rri_topics over [0, t) and then [t, k) is one interleaved sweep of the oracle"""
    X, Wm, Xd, M, W0, T0 = _case(320, 270, 7, 0.3, True, seed=10)
    eng = _engine(R, X, Wm, 7, 0.3, dtype=torch.float64)
    try:
        W = torch.as_tensor(W0, device='cuda:0').clone()
        T = torch.as_tensor(T0, device='cuda:0').clone()
        p = eng.params()
        eng.topics(W, T, 0, 3, p)
        eng.topics(W, T, 3, 7, p)
        Wo, To = W0.copy(), T0.copy()
        orc.sweep(Xd, Wo, To, M)
        assert relfro(W.cpu().numpy(), Wo) <= 1e-9 and relfro(T.cpu().numpy(), To) <= 1e-9
    finally:
        eng.close()


def test_device_init_scipy_and_torch_csr(R):
    """the device NNDSVD starts from W_mat o X (the unstored weight does not enter it); the sweeps from there follow the
    oracle, and a torch CSR input on the device gives the same factors as the scipy input"""
    X, Wm, Xd, M, _, _ = _case(400, 300, 6, 0.08, True, seed=12)
    kw = dict(W_mat=Wm, random_state=3, init_on_device=True, reset_topic_method=None, unstored_weight=0.08)
    i0 = R.nmf(X, 6, max_iter=0, **kw)
    i00 = R.nmf(X, 6, max_iter=0, **dict(kw, unstored_weight=0.0))
    assert np.array_equal(i0['W'], i00['W']) and np.array_equal(i0['T'], i00['T'])
    g = R.nmf(X, 6, max_iter=3, **kw)
    o = orc.nmf_oracle(Xd, 6, i0['W'], i0['T'], max_iter=3, W_mat=M)
    assert relfro(g['W'], o['W']) <= 1e-9 and relfro(g['T'], o['T']) <= 1e-9
    from rri_nmf_b200.engine import RRIEngine
    Xt = RRIEngine.csr_tensor(X.indptr, X.indices, X.data, X.shape, 'cuda:0', torch.float64)
    gt = R.nmf(Xt, 6, max_iter=3, **dict(kw, W_mat=torch.as_tensor(Wm.data, device='cuda:0')))
    assert isinstance(gt['W'], torch.Tensor) and gt['W'].is_cuda
    assert relfro(gt['W'].cpu().numpy(), g['W']) <= 1e-12 and relfro(gt['T'].cpu().numpy(), g['T']) <= 1e-12


def test_rs_estimator_through_nmf_kwargs(R, monkeypatch):
    """NMF_RS_Estimator(sparse=True, nmf_kwargs={'unstored_weight': w0}) is nmf(..., unstored_weight=w0); its validation
    early stop is handed the device tensors"""
    si = importlib.import_module('rri_nmf_b200.sklearn_interface')
    rs = np.random.RandomState(0)
    n, d, k = 300, 200, 5
    U, V = rs.rand(n, 3), rs.rand(3, d)
    mask = rs.rand(n, d) < 0.1
    I, J = np.nonzero(mask)
    y = np.clip(np.round(1 + 4 * (U.dot(V))[I, J] / 3), 1, 5)
    ij = np.column_stack([I, J])
    kw = dict(random_state=0, max_iter=8, sparse=True, nmf_kwargs={'unstored_weight': 0.05})
    E = R.NMF_RS_Estimator(n, d, k, use_validation_early_stopping=False, **kw).fit(ij, y)
    F = R.NMF_RS_Estimator(n, d, k, use_validation_early_stopping=False, **kw)
    W_in, T_in = F._warm_start()
    direct = R.nmf(F._observed(ij, y), k, max_iter=8, max_time=7200, compute_obj_each_iter=True,
                   reset_topic_method=None, early_stop=False, project_T_each_iter=False, t_row_sum=1.0,
                   project_W_each_iter=False, w_row_sum=None, W_mat=None, W_in=W_in, T_in=T_in, reg_w_l1=0,
                   reg_t_l1=0, random_state=0, return_reconstruction_err=True, unstored_weight=0.05,
                   **F._device_kwargs())
    assert np.array_equal(E.W, direct['W']) and np.array_equal(E.T, direct['T'])
    seen = []
    real = si.nmf

    def spy(*a, **kws):
        cb = kws.get('early_stop')
        if callable(cb):
            def wrapped(X, W, T):
                seen.append((type(W), getattr(W, 'is_cuda', False)))
                return cb(X, W, T)
            wrapped.device_tensors = getattr(cb, 'device_tensors', False)
            kws['early_stop'] = wrapped
        assert kws.get('unstored_weight') == 0.05
        return real(*a, **kws)
    monkeypatch.setattr(si, 'nmf', spy)
    R.NMF_RS_Estimator(n, d, k, use_validation_early_stopping=True, **kw).fit(ij, y)
    assert seen and all(t is torch.Tensor and cuda for t, cuda in seen)


def test_abi_refusals(R):
    """the entry points that do not serve an unstored weight refuse it, and a bad weight is refused"""
    from rri_nmf_b200 import _lib
    from rri_nmf_b200.engine import RRIEngine
    lib = _lib.load()

    def handle():
        h = C.c_void_p()
        _lib.check(lib.rri_create(C.byref(h), 40, 30, 4, _lib.RRI_F64, _lib.RRI_MATH_IEEE, _lib.RRI_ORDER_RRI, 0))
        return h
    h = handle()
    try:
        for bad in (-1.0, float('nan'), float('inf')):
            assert lib.rri_set_unstored_weight(h, bad) != 0
        assert lib.rri_set_unstored_weight(h, 0.1) == 0
        X = torch.rand(40, 30, dtype=torch.float64, device='cuda:0')
        assert lib.rri_bind(h, C.c_void_p(X.data_ptr()), 30, None, _lib.RRI_MASK_NONE, 0, None) != 0
        rowptr = torch.zeros(41, dtype=torch.int64, device='cuda:0')
        assert lib.rri_bind_csr_zero(h, 0, C.c_void_p(rowptr.data_ptr()), None, None, None) != 0
        assert lib.rri_set_models(h, 2) != 0
        assert lib.rri_set_comm(h, None, 0, 2, None) != 0
    finally:
        lib.rri_destroy(h)
    X, Wm, _, _, W0, T0 = _case(40, 30, 4, 0.1, False, density=0.3, seed=1)
    eng = _engine(R, X, Wm, 4, 0.1, dtype=torch.float64)
    try:
        W = torch.as_tensor(W0, device='cuda:0').contiguous()
        T = torch.as_tensor(T0, device='cuda:0').contiguous()
        with pytest.raises(_lib.RriError):
            eng.partials_T(W, T, 0)
        assert lib.rri_set_unstored_weight(eng.h, 0.2) != 0            # after the binding
        eng.sweeps(W, T, 1, eng.params())                               # the handle still works
        st = eng.stats()
        assert st['kernel_launches'] > 0
    finally:
        eng.close()
    with pytest.raises(ValueError):
        RRIEngine(torch.rand(40, 30, device='cuda:0'), 4, unstored_weight=0.1)
