"""Observed-entries data with rank-one weights on the unstored entries (nmf(X_sparse, ..., unstored_weight=w0,
unstored_row_weight=a, unstored_col_weight=b), rri_set_unstored_weight_vectors): against the oracle's masked iteration on
the densified X and M (M = w0 a_i b_j at every unstored entry), against the dense masked engine and the scalar-w0
handle, its determinism, topics, initialisation, objective, the recommender estimator and the ABI refusals."""
import ctypes as C
import importlib
import pickle

import numpy as np
import pytest
import scipy.sparse as sp
import torch

import rri_oracle as orc
from conftest import relfro
from test_sparse_implicit_vectors_scheme_cpu import dense_M_vectors, vectors_case

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def R(cuda_device):
    import rri_nmf_b200
    return rri_nmf_b200


def _case(n, d, k, w0, weighted, which, density=0.12, seed=0, dtype=np.float64):
    """(X csr, weights csr or None, dense X, dense M, W0, T0, a, b)"""
    I, J, vals, wts, W0, T0, a, b = vectors_case(n, d, k, density, seed, weighted, which)
    X = sp.csr_matrix((vals, (I, J)), shape=(n, d), dtype=dtype)
    assert X.nnz == len(vals)                                   # the explicit zeros stay stored
    Wm = None if wts is None else sp.csr_matrix((wts, (I, J)), shape=(n, d), dtype=dtype)
    Xd = np.zeros((n, d))
    Xd[I, J] = vals
    cast = lambda v: None if v is None else v.astype(dtype)
    return (X, Wm, Xd, dense_M_vectors(I, J, n, d, w0, cast(a), cast(b), wts), W0.astype(dtype), T0.astype(dtype),
            cast(a), cast(b))


CASES = [
    ('rri', 0.05, False, 'b', 7, {}),
    ('rri', 0.5, True, 'a', 5, {}),
    ('rri', 0.3, True, 'ab', 1, {}),
    ('hals', 1.0, False, 'ab', 3, {}),
    ('hals', 0.3, True, 'b', 5, {}),
    ('rri', 0.2, True, 'ab', 6, dict(reg_w_l1=0.01, reg_w_l2=0.1, reg_t_l1=0.02, reg_t_l2=0.2)),
    ('hals', 0.2, False, 'ab', 6, dict(reg_w_l1=0.01, reg_w_l2=0.1, reg_t_l1=0.02, reg_t_l2=0.2)),
    ('rri', 0.1, False, 'ab', 8, dict(project_T_each_iter=True, t_row_sum=1.0)),
    ('rri', 0.1, True, 'b', 6, dict(w_row_sum=1.0)),
    ('rri', 0.1, True, 'ab', 5, dict(fix_T=True)),
    ('hals', 0.1, False, 'a', 5, dict(fix_T=True)),
]


@pytest.mark.parametrize('order,w0,weighted,which,k,kw', CASES)
def test_parity_with_oracle_fp64(R, order, w0, weighted, which, k, kw):
    """after each of sweeps 1..3 the factors, and the objective history, are within 1e-9 of the oracle's masked
    iteration on X.toarray() with the dense M"""
    X, Wm, Xd, M, W0, T0, a, b = _case(300, 220, k, w0, weighted, which, seed=k)
    for ns in (1, 2, 3):
        o = orc.nmf_oracle(Xd, k, W0, T0, max_iter=ns, W_mat=M, order=order, compute_obj_each_iter=True, eps_stop=0,
                           **kw)
        g = R.nmf(X, k, W_mat=Wm, W_in=W0, T_in=T0, max_iter=ns, update_order=order, reset_topic_method=None,
                  compute_obj_each_iter=True, eps_stop=0, unstored_weight=w0, unstored_row_weight=a,
                  unstored_col_weight=b, **kw)
        assert relfro(g['W'], o['W']) <= 1e-9, (ns, relfro(g['W'], o['W']))
        assert relfro(g['T'], o['T']) <= 1e-9, (ns, relfro(g['T'], o['T']))
        assert np.allclose(g['obj_history'], o['obj_history'], rtol=1e-9, atol=0)
    # the detached calculator keeps the vectors as host arrays (it pickles) and rebuilds an engine with them
    calc = pickle.loads(pickle.dumps(g['obj_calculator']))
    regs = {x: y for x, y in kw.items() if x.startswith('reg')}
    assert abs(calc.true_objective() / orc.objective(Xd, g['W'], g['T'], M, **regs) - 1) <= 1e-9


def test_objective_terms_and_reconstruction_error(R):
    X, Wm, Xd, M, W0, T0, a, b = _case(260, 310, 6, 0.07, True, 'ab', seed=3)
    g = R.nmf(X, 6, W_mat=Wm, W_in=W0, T_in=T0, max_iter=4, reset_topic_method=None, unstored_weight=0.07,
              unstored_row_weight=a, unstored_col_weight=b, return_reconstruction_err=True)
    ref = np.sqrt(np.sum(M * (Xd - g['W'].dot(g['T'])) ** 2))
    assert abs(g['reconstruction_err'] / ref - 1) <= 1e-9


@pytest.mark.parametrize('order', ['rri', 'hals'])
def test_same_as_dense_masked_engine(R, order):
    """fp64: within 1e-9 of nmf(X.toarray(), W_mat=M) on the dense masked engine; fp32: the final relative errors
    after 20 sweeps agree within 1e-4"""
    X, Wm, Xd, M, W0, T0, a, b = _case(500, 420, 8, 0.05, True, 'ab', density=0.08, seed=4)
    kw = dict(W_in=W0, T_in=T0, max_iter=6, update_order=order, reset_topic_method=None, return_reconstruction_err=True)
    g = R.nmf(X, 8, W_mat=Wm, unstored_weight=0.05, unstored_row_weight=a, unstored_col_weight=b, **kw)
    o = R.nmf(Xd, 8, W_mat=M, **kw)
    assert relfro(g['W'], o['W']) <= 1e-9 and relfro(g['T'], o['T']) <= 1e-9
    assert abs(g['reconstruction_err'] / o['reconstruction_err'] - 1) <= 1e-9
    kw32 = dict(kw, W_in=W0.astype(np.float32), T_in=T0.astype(np.float32), max_iter=20)
    g = R.nmf(X.astype(np.float32), 8, W_mat=Wm.astype(np.float32), unstored_weight=0.05,
              unstored_row_weight=a.astype(np.float32), unstored_col_weight=b.astype(np.float32), **kw32)
    o = R.nmf(Xd.astype(np.float32), 8, W_mat=M.astype(np.float32), **kw32)
    assert g['W'].dtype == np.float32
    xn = float(np.sqrt(np.sum(M * Xd ** 2)))
    assert abs(g['reconstruction_err'] - o['reconstruction_err']) / xn <= 1e-4


@pytest.mark.parametrize('order', ['rri', 'hals'])
def test_vectors_of_ones_are_the_scalar_handle(R, order):
    X, Wm, _, _, W0, T0, _, _ = _case(400, 330, 7, 0.2, True, 'ab', seed=6)
    kw = dict(W_mat=Wm, W_in=W0, T_in=T0, max_iter=5, update_order=order, reset_topic_method=None, unstored_weight=0.2,
              compute_obj_each_iter=True, eps_stop=0)
    s = R.nmf(X, 7, **kw)
    v = R.nmf(X, 7, unstored_row_weight=np.ones(400), unstored_col_weight=np.ones(330), **kw)
    assert relfro(v['W'], s['W']) <= 1e-12 and relfro(v['T'], s['T']) <= 1e-12
    assert np.allclose(v['obj_history'], s['obj_history'], rtol=1e-12, atol=0)


def _engine(X, Wm, k, w0, a=None, b=None, order='rri', dtype=torch.float32):
    from rri_nmf_b200.engine import RRIEngine
    Xt = RRIEngine.csr_tensor(X.indptr, X.indices, X.data, X.shape, 'cuda:0', dtype)
    wt = None if Wm is None else torch.as_tensor(Wm.data, device='cuda:0', dtype=dtype)
    return RRIEngine(Xt, k, W_mat=wt, order=order, unstored_weight=w0, unstored_row_weight=a, unstored_col_weight=b)


@pytest.mark.parametrize('order', ['rri', 'hals'])
def test_null_vectors_are_the_scalar_handle_bit_for_bit(R, order, monkeypatch):
    """rri_set_unstored_weight_vectors(h, NULL, NULL) leaves the scalar-w0 handle: the same launches, the same bits"""
    from rri_nmf_b200 import _lib
    X, Wm, _, _, W0, T0, _, _ = _case(700, 520, 9, 0.05, True, 'ab', seed=8, dtype=np.float32)
    lib = _lib.load()

    def run():
        eng = _engine(X, Wm, 9, 0.05, order=order)
        try:
            W = torch.as_tensor(W0, device='cuda:0').clone()
            T = torch.as_tensor(T0, device='cuda:0').clone()
            eng.sweeps(W, T, 3, eng.params())
            v = eng.objective_terms(W, T)
            torch.cuda.synchronize()
            return W.cpu(), T.cpu(), v, eng.stats()['kernel_launches']
        finally:
            eng.close()
    Wa, Ta, va, na = run()
    real = lib.rri_set_unstored_weight

    def with_null_vectors(h, w0):
        rc = real(h, w0)
        return rc or lib.rri_set_unstored_weight_vectors(h, None, None)
    monkeypatch.setattr(lib, 'rri_set_unstored_weight', with_null_vectors)
    Wb, Tb, vb, nb = run()
    assert torch.equal(Wa, Wb) and torch.equal(Ta, Tb)
    assert list(va) == list(vb) and na == nb


@pytest.mark.parametrize('order', ['rri', 'hals'])
@pytest.mark.parametrize('weighted', [False, True])
def test_n_sweeps_in_one_call_equal_n_calls(R, order, weighted):
    X, Wm, _, _, W0, T0, a, b = _case(700, 520, 9, 0.05, weighted, 'ab', seed=8, dtype=np.float32)
    eng = _engine(X, Wm, 9, 0.05, a, b, order)
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
    X, Wm, Xd, M, W0, T0, a, b = _case(600, 450, 8, 0.1, True, 'ab', seed=9)
    kw = dict(W_mat=Wm, W_in=W0, T_in=T0, max_iter=10, reset_topic_method=None, unstored_weight=0.1,
              unstored_row_weight=a, unstored_col_weight=b, sweeps_per_call=10)
    g = R.nmf(X, 8, **kw)
    o = orc.nmf_oracle(Xd, 8, W0, T0, max_iter=10, W_mat=M)
    assert relfro(g['W'], o['W']) <= 1e-9 and relfro(g['T'], o['T']) <= 1e-9
    e8 = R.nmf(X, 8, sparse_refresh_every=8, **kw)
    assert relfro(e8['W'], g['W']) <= 1e-9 and relfro(e8['T'], g['T']) <= 1e-9


def test_topics_in_two_ranges(R):
    """rri_topics over [0, t) and then [t, k) is one interleaved sweep of the oracle"""
    X, Wm, Xd, M, W0, T0, a, b = _case(320, 270, 7, 0.3, True, 'ab', seed=10)
    eng = _engine(X, Wm, 7, 0.3, a, b, dtype=torch.float64)
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


def test_device_init_scipy_and_torch_csr_with_cuda_vectors(R):
    """the device NNDSVD starts from W_mat o X (the unstored weights do not enter it); the sweeps from there follow the
    oracle, and a torch CSR input with CUDA-tensor vectors gives the same factors as the scipy input"""
    X, Wm, Xd, M, _, _, a, b = _case(400, 300, 6, 0.08, True, 'ab', seed=12)
    kw = dict(W_mat=Wm, random_state=3, init_on_device=True, reset_topic_method=None, unstored_weight=0.08)
    i0 = R.nmf(X, 6, max_iter=0, unstored_row_weight=a, unstored_col_weight=b, **kw)
    i00 = R.nmf(X, 6, max_iter=0, **kw)
    assert np.array_equal(i0['W'], i00['W']) and np.array_equal(i0['T'], i00['T'])
    g = R.nmf(X, 6, max_iter=3, unstored_row_weight=a, unstored_col_weight=b, **kw)
    o = orc.nmf_oracle(Xd, 6, i0['W'], i0['T'], max_iter=3, W_mat=M)
    assert relfro(g['W'], o['W']) <= 1e-9 and relfro(g['T'], o['T']) <= 1e-9
    from rri_nmf_b200.engine import RRIEngine
    Xt = RRIEngine.csr_tensor(X.indptr, X.indices, X.data, X.shape, 'cuda:0', torch.float64)
    gt = R.nmf(Xt, 6, max_iter=3, unstored_row_weight=torch.as_tensor(a, device='cuda:0'),
               unstored_col_weight=torch.as_tensor(b, device='cuda:0'),
               **dict(kw, W_mat=torch.as_tensor(Wm.data, device='cuda:0')))
    assert isinstance(gt['W'], torch.Tensor) and gt['W'].is_cuda
    assert relfro(gt['W'].cpu().numpy(), g['W']) <= 1e-12 and relfro(gt['T'].cpu().numpy(), g['T']) <= 1e-12


def test_rs_estimator_through_nmf_kwargs(R, monkeypatch):
    """NMF_RS_Estimator(sparse=True, nmf_kwargs={...vectors...}) is nmf(..., the vectors); transform() folds in new
    rows with w0 and the column weights and drops the row weights"""
    si = importlib.import_module('rri_nmf_b200.sklearn_interface')
    rs = np.random.RandomState(0)
    n, d, k = 300, 200, 5
    U, V = rs.rand(n, 3), rs.rand(3, d)
    mask = rs.rand(n, d) < 0.1
    I, J = np.nonzero(mask)
    y = np.clip(np.round(1 + 4 * (U.dot(V))[I, J] / 3), 1, 5)
    ij = np.column_stack([I, J])
    a = rs.uniform(0.5, 2.0, n)
    b = np.bincount(J, minlength=d).astype(np.float64) ** 0.5 + 0.1      # item popularity
    nk = {'unstored_weight': 0.05, 'unstored_row_weight': a, 'unstored_col_weight': b}
    kw = dict(random_state=0, max_iter=8, sparse=True, nmf_kwargs=nk)
    E = R.NMF_RS_Estimator(n, d, k, use_validation_early_stopping=False, **kw).fit(ij, y)
    F = R.NMF_RS_Estimator(n, d, k, use_validation_early_stopping=False, **kw)
    W_in, T_in = F._warm_start()
    direct = R.nmf(F._observed(ij, y), k, max_iter=8, max_time=7200, compute_obj_each_iter=True,
                   reset_topic_method=None, early_stop=False, project_T_each_iter=False, t_row_sum=1.0,
                   project_W_each_iter=False, w_row_sum=None, W_mat=None, W_in=W_in, T_in=T_in, reg_w_l1=0,
                   reg_t_l1=0, random_state=0, return_reconstruction_err=True, **dict(nk, **F._device_kwargs()))
    assert np.array_equal(E.W, direct['W']) and np.array_equal(E.T, direct['T'])
    Xnew = sp.csr_matrix((y[:40], (I[:40] % 17, J[:40])), shape=(17, d))
    seen = []
    real = si.nmf

    def spy(*args, **kws):
        seen.append(dict(kws))
        return real(*args, **kws)
    monkeypatch.setattr(si, 'nmf', spy)
    Wn = E.transform(Xnew)
    assert Wn.shape == (17, k)
    assert 'unstored_row_weight' not in seen[-1] and seen[-1]['unstored_col_weight'] is b
    assert seen[-1]['unstored_weight'] == 0.05 and seen[-1]['fix_T']


def test_abi_refusals(R):
    """the calls the rank-one weights do not serve are refused, and bad vectors fail the binding"""
    from rri_nmf_b200 import _lib
    from rri_nmf_b200.engine import RRIEngine
    lib = _lib.load()

    def handle(order=_lib.RRI_ORDER_RRI):
        h = C.c_void_p()
        _lib.check(lib.rri_create(C.byref(h), 40, 30, 4, _lib.RRI_F64, _lib.RRI_MATH_IEEE, order, 0))
        return h
    av = torch.ones(40, dtype=torch.float64, device='cuda:0')
    bv = torch.ones(30, dtype=torch.float64, device='cuda:0')
    pa, pb = C.c_void_p(av.data_ptr()), C.c_void_p(bv.data_ptr())
    h = handle()
    try:
        assert lib.rri_set_unstored_weight_vectors(h, pa, pb) != 0          # no w0 > 0
        assert lib.rri_set_unstored_weight(h, 0.1) == 0
        assert lib.rri_set_unstored_weight_vectors(h, pa, pb) == 0
        X = torch.rand(40, 30, dtype=torch.float64, device='cuda:0')
        assert lib.rri_bind(h, C.c_void_p(X.data_ptr()), 30, None, _lib.RRI_MASK_NONE, 0, None) != 0
        rowptr = torch.zeros(41, dtype=torch.int64, device='cuda:0')
        assert lib.rri_bind_csr_zero(h, 0, C.c_void_p(rowptr.data_ptr()), None, None, None) != 0
        assert lib.rri_set_models(h, 2) != 0
        assert lib.rri_set_comm(h, None, 0, 2, None) != 0
    finally:
        lib.rri_destroy(h)
    h = handle(_lib.RRI_ORDER_HALS)
    try:
        assert lib.rri_set_models(h, 2) == 0
        assert lib.rri_set_unstored_weight_vectors(h, pa, pb) != 0          # a handle of several models
    finally:
        lib.rri_destroy(h)
    X, Wm, _, _, W0, T0, a, b = _case(40, 30, 4, 0.1, False, 'ab', density=0.3, seed=1)
    for bad in (-1.0, float('nan'), float('inf')):                          # checked on the device at bind
        bb = b.copy()
        bb[3] = bad
        with pytest.raises(_lib.RriError):
            _bind_unchecked(X, a, bb)
    eng = _engine(X, Wm, 4, 0.1, a, b, dtype=torch.float64)
    try:
        W = torch.as_tensor(W0, device='cuda:0').contiguous()
        T = torch.as_tensor(T0, device='cuda:0').contiguous()
        with pytest.raises(_lib.RriError):
            eng.partials_T(W, T, 0)
        assert lib.rri_set_unstored_weight_vectors(eng.h, pa, pb) != 0     # after the binding
        eng.sweeps(W, T, 1, eng.params())                                   # the handle still works
        assert eng.stats()['kernel_launches'] > 0
    finally:
        eng.close()
    with pytest.raises(ValueError):
        RRIEngine(torch.rand(40, 30, device='cuda:0'), 4, unstored_weight=0.1, unstored_col_weight=np.ones(30))


def _bind_unchecked(X, a, b):
    """rri_create + rri_set_unstored_weight(_vectors) + rri_bind_csr on the raw ABI (no host-side check of the vectors)"""
    from rri_nmf_b200 import _lib
    lib = _lib.load()
    h = C.c_void_p()
    _lib.check(lib.rri_create(C.byref(h), X.shape[0], X.shape[1], 4, _lib.RRI_F64, _lib.RRI_MATH_IEEE,
                              _lib.RRI_ORDER_RRI, 0))
    try:
        av = torch.as_tensor(a, device='cuda:0', dtype=torch.float64)
        bv = torch.as_tensor(b, device='cuda:0', dtype=torch.float64)
        _lib.check(lib.rri_set_unstored_weight(h, 0.1))
        _lib.check(lib.rri_set_unstored_weight_vectors(h, C.c_void_p(av.data_ptr()), C.c_void_p(bv.data_ptr())))
        del av, bv                                                          # the engine keeps its own copies
        rp = torch.as_tensor(X.indptr, device='cuda:0', dtype=torch.int64)
        ci = torch.as_tensor(X.indices, device='cuda:0', dtype=torch.int32)
        va = torch.as_tensor(X.data, device='cuda:0', dtype=torch.float64)
        _lib.check(lib.rri_bind_csr(h, X.nnz, C.c_void_p(rp.data_ptr()), C.c_void_p(ci.data_ptr()),
                                    C.c_void_p(va.data_ptr()), None, None))
    finally:
        lib.rri_destroy(h)
