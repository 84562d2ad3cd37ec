"""GPU parity tests of the observed-entries (sparse CSR/CSC) WRRI path -- SURVEY.md §8 row f4 -- through the
C-ABI (rri_bind_csr + the masked entry points), against the golden vectors of the unmodified reference and
the NumPy oracle run on the densified data.

Tolerances as for the dense path: FP64 relative Frobenius <= 1e-9; FP32 final relative error within 1e-4.
"""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

import rri_oracle as orc
from conftest import golden, relfro

pytestmark = pytest.mark.gpu

F64_TOL = 1e-9


@pytest.fixture(scope='module')
def R(cuda_device):
    import rri_nmf_b200
    return rri_nmf_b200


def run(R, X, k, W0, T0, **kw):
    kw.setdefault('reset_topic_method', None)
    kw.setdefault('max_time', 1e9)
    kw.setdefault('eps_stop', -1.0)
    return R.nmf(X, k, W_in=W0, T_in=T0, **kw)


def observed(X, M):
    """CSR of the entries where M != 0 (values may be anything, also 0)"""
    I, J = np.nonzero(M)
    return sp.csr_matrix((X[I, J], (I, J)), shape=X.shape)


@pytest.mark.parametrize('name,regs', [('plain', {}), ('l1both', {'reg_w_l1': 0.1, 'reg_t_l1': 0.1}),
                                        ('l1w', {'reg_w_l1': 0.1}), ('l1t', {'reg_t_l1': 0.1})])
def test_recsys_sparse_matches_reference(R, name, regs):
    g = golden('recsys_wrri_f64.npz')
    X = g['X']
    out = run(R, sp.csr_matrix(X), 7, g['W0'], g['T0'], max_iter=15, compute_obj_each_iter=True, t_row_sum=1.0,
              **regs)
    assert relfro(out['W'], g['W_' + name]) < F64_TOL and relfro(out['T'], g['T_' + name]) < F64_TOL
    assert np.allclose(out['obj_history'], g['obj_' + name], rtol=1e-9)
    assert np.all(np.diff(out['obj_history']) <= 1e-9)        # reference tests/test_nmf.py:78
    assert out['T'].max() <= 1.0                              # ub clip (optimization.py:82-83)


def test_sparse_entry_weights_both_orders(R):
    X, W0, T0, Mb = orc.synth(120, 90, 5, 6, sigma=0.05, seed=5, mask_density=0.3)
    Mw = Mb * np.random.RandomState(9).rand(120, 90) * 2.0
    Xs, Ws = observed(X, Mb), observed(Mw, Mb)
    g = golden('weighted_wrri_f64.npz')
    out = run(R, Xs, 6, W0, T0, max_iter=8, W_mat=Ws, compute_obj_each_iter=True)
    assert relfro(out['W'], g['W']) < F64_TOL and relfro(out['T'], g['T']) < F64_TOL
    assert np.allclose(out['obj_history'], g['obj_history'], rtol=1e-9)
    gh = golden('weighted_wrri_hals_f64.npz')
    out = run(R, Xs, 6, W0, T0, max_iter=5, W_mat=Ws, update_order='hals')
    assert relfro(out['W'], gh['W']) < F64_TOL and relfro(out['T'], gh['T']) < F64_TOL


@pytest.mark.parametrize('n,d,density', [(700, 1900, 0.3),     # rows >= 512 entries: a block per row, a warp per column
                                          (1900, 700, 0.3),     # the other way round
                                          (257, 131, 0.05),     # short, ragged segments; empty rows and columns
                                          (9000, 300, 0.05),    # the gathered factor spans several shared-memory blocks
                                          (300, 9000, 0.05),    # (4096 records each in fp64), in either orientation
                                          (48, 270000, 0.001),  # more than 64 such blocks: the direct pass, gathering
                                          (270000, 48, 0.001)]) # from global memory, in either orientation
@pytest.mark.parametrize('order', ['rri', 'hals'])
def test_sparse_matches_oracle_fp64(R, n, d, density, order):
    k = 8 if n > 500 else 7        # odd k: zero pad columns in the restart's 16-byte gathers of T' rows
    X, W0, T0, M = orc.synth(n, d, k, k, sigma=0.05, seed=n + d, mask_density=density)
    M[5, :] = 0
    M[:, 3] = 0                                               # an unobserved row and column
    o = orc.nmf_oracle(X, k, W0, T0, max_iter=3, W_mat=M, order=order)
    out = run(R, observed(X, M), k, W0, T0, max_iter=3, update_order=order)
    assert relfro(out['W'], o['W']) < F64_TOL and relfro(out['T'], o['T']) < F64_TOL
    assert np.all(out['T'][:, 3] == 0) and np.all(out['W'][5, :] == 0)


def test_sparse_fp32_relerr_and_resume(R):
    X, W0, T0, M = orc.synth(600, 400, 12, 12, sigma=0.05, seed=21, mask_density=0.15)
    o = orc.nmf_oracle(X, 12, W0, T0, max_iter=10, W_mat=M)
    Xs = observed(X, M).astype(np.float32)
    W32, T32 = W0.astype(np.float32), T0.astype(np.float32)
    out = run(R, Xs, 12, W32, T32, max_iter=10)
    assert out['W'].dtype == np.float32
    re_o = orc.rel_error(X, o['W'], o['T'], M)
    re_g = orc.rel_error(X, out['W'].astype(np.float64), out['T'].astype(np.float64), M)
    assert abs(re_o - re_g) < 1e-4, (re_o, re_g)
    # N sweeps == N x one sweep, bit for bit (tests/test_nmf.py:97-109): the residual restarts every sweep
    W, T = W32, T32
    for _ in range(10):
        r = run(R, Xs, 12, W, T, max_iter=1)
        W, T = r['W'], r['T']
    assert np.array_equal(W, out['W']) and np.array_equal(T, out['T'])


def test_sparse_fix_T_is_transform(R):
    """W-only sweeps (sklearn_interface.py:144-156) read the row orientation only"""
    X, W0, T0, M = orc.synth(300, 200, 6, 6, sigma=0.05, seed=4, mask_density=0.2)
    o = orc.nmf_oracle(X, 6, W0, T0, max_iter=4, W_mat=M, fix_T=True)
    out = run(R, observed(X, M), 6, W0, T0, max_iter=4, fix_T=True)
    assert relfro(out['W'], o['W']) < F64_TOL
    assert np.array_equal(out['T'], np.maximum(T0, 0))


def test_sparse_partials_and_objective_match_dense_engine(R, cuda_device):
    X, W0, T0, M = orc.synth(257, 131, 5, 7, sigma=0.05, seed=8, mask_density=0.3)
    dev = cuda_device
    Wd, Td = torch.from_numpy(np.maximum(W0, 0)).to(dev), torch.from_numpy(np.maximum(T0, 0)).to(dev)
    Xs = observed(X, M)
    Xc = R.RRIEngine.csr_tensor(Xs.indptr, Xs.indices, Xs.data, Xs.shape, dev)
    es = R.RRIEngine(Xc, 7)
    ed = R.RRIEngine(torch.from_numpy(X).to(dev), 7, W_mat=torch.from_numpy(M).to(dev))
    try:
        for t in (0, 3, 6):
            a, b = es.partials_T(Wd, Td, t)
            c, e = ed.partials_T(Wd, Td, t)
            # nmf.py:697-699: wR = W[:,t]' Rt, nw = (W[:,t]^2)' M
            assert relfro(a.cpu().numpy(), c.cpu().numpy()) < F64_TOL and relfro(b.cpu().numpy(), e.cpu().numpy()) < F64_TOL
        vs, vd = es.objective_terms(Wd, Td), ed.objective_terms(Wd, Td)
        assert np.allclose(vs, vd, rtol=1e-12)
        assert abs(es.rel_error(Wd, Td) - orc.rel_error(X, np.maximum(W0, 0), np.maximum(T0, 0), M)) < 1e-12
        assert es.masked and es.sparse and es.stats()['kernel_launches'] > 0
    finally:
        es.close()
        ed.close()


def test_sparse_rejects_malformed_csr(R, cuda_device):
    dev = cuda_device
    crow = np.array([0, 2, 3])
    val = np.array([1.0, 2.0, 3.0])

    def engine(cols, ncols=4, **kw):
        return R.RRIEngine(R.RRIEngine.csr_tensor(crow, np.array(cols), val, (2, ncols), dev, kw.pop('dtype', None)), 2, **kw)

    with pytest.raises(RuntimeError, match='ascending'):
        engine([2, 1, 0])                       # unsorted row
    with pytest.raises(RuntimeError, match='ascending'):
        engine([1, 1, 0])                       # duplicate entry
    e = engine([0, 3, 1])
    e.close()
    with pytest.raises(RuntimeError, match='outside'):
        engine([0, 4, 1])                       # column index >= d
    with pytest.raises(ValueError):
        engine([0, 3, 1], dtype=torch.float32, math='tf32')


def test_RS_estimator_sparse_equals_dense(R):
    """the estimator keeps the ratings sparse end to end with sparse=True; same fit as the densifying default"""
    X = golden('recsys_wrri_f64.npz')['X']
    n, d = X.shape
    for early in (False, True):
        Ed = R.NMF_RS_Estimator(n, d, 5, random_state=0, max_iter=12, use_validation_early_stopping=early).fit_from_Xtr(X)
        Es = R.NMF_RS_Estimator(n, d, 5, random_state=0, max_iter=12, use_validation_early_stopping=early,
                                sparse=True).fit_from_Xtr(sp.csr_matrix(X))
        assert relfro(Es.W, Ed.W) < 1e-8 and relfro(Es.T, Ed.T) < 1e-8
        assert abs(Es.reconstruction_err_ - Ed.reconstruction_err_) < 1e-8 * Ed.reconstruction_err_
        assert Es.score(X) < 1.0
    assert relfro(Es.transform(sp.csr_matrix(X)), Ed.transform(X)) < 1e-8


def test_sparse_residual_carried_across_sweeps(cuda_device):
    """sparse_refresh_every > 1: the two residual copies continue from sweep to sweep inside one engine call (with the
    pending rank-one record crossing the sweep boundary) instead of being rebuilt from the factors; in fp64 the
    iterates agree with the restart-every-sweep run to rounding, and the call is still exact against the oracle."""
    import scipy.sparse as sp
    import rri_nmf_b200 as R
    X, W0, T0, M = orc.synth(300, 210, 6, 7, sigma=0.05, seed=21, mask_density=0.2)
    Xs = sp.csr_matrix(X * M)
    o = orc.nmf_oracle(X, 7, W0, T0, max_iter=9, W_mat=M, t_row_sum=1.0)
    kw = dict(W_in=W0, T_in=T0, max_iter=9, t_row_sum=1.0, reset_topic_method=None, max_time=1e9, sweeps_per_call=16)
    a = R.nmf(Xs, 7, sparse_refresh_every=1, **kw)
    b = R.nmf(Xs, 7, sparse_refresh_every=4, **kw)
    assert relfro(a['W'], o['W']) < 1e-9 and relfro(a['T'], o['T']) < 1e-9
    assert relfro(b['W'], o['W']) < 1e-9 and relfro(b['T'], o['T']) < 1e-9
    assert relfro(b['W'], a['W']) < 1e-11


@pytest.mark.parametrize('weighted', [False, True])
def test_sparse_fp32_long_factor_streamlined_pass(R, weighted):
    """fp32 with a gathered factor longer than one 64 KB staging block (9000 rows -> two blocks of 4500 records on the
    column side): the T-steps run through sp_pass_stream_kernel (16 entries per lane and batch; 8 with entry weights),
    the W-steps through the two-CTA kernel.  Final relative error within 1e-4 of the fp64 oracle, factors within 1e-3."""
    n, d, k = 9000, 160, 4
    X, W0, T0, Mb = orc.synth(n, d, k, k, sigma=0.05, seed=33, mask_density=0.06)
    kw = {}
    M = Mb
    if weighted:
        M = Mb * (0.5 + np.random.RandomState(4).rand(n, d))
        kw['W_mat'] = observed(M, Mb).astype(np.float32)
    o = orc.nmf_oracle(X, k, W0, T0, max_iter=4, W_mat=M)
    out = run(R, observed(X, Mb).astype(np.float32), k, W0.astype(np.float32), T0.astype(np.float32), max_iter=4, **kw)
    re_o = orc.rel_error(X, o['W'], o['T'], Mb)
    re_g = orc.rel_error(X, out['W'].astype(np.float64), out['T'].astype(np.float64), Mb)
    assert abs(re_o - re_g) < 1e-4, (re_o, re_g)
    assert relfro(out['W'], o['W']) < 1e-3 and relfro(out['T'], o['T']) < 1e-3
