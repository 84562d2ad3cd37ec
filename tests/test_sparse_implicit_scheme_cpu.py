"""Observed-entries WRRI with a weight w0 on the unstored entries (nmf(..., unstored_weight=w0), rri_set_unstored_weight):
the scheme of rri_nmf_b200/csrc/sparse_kernels.cu + api.cu -- residual copies holding the shifted residual
S = (m - w0) E + w0 x, plus one Gram row per half-step -- modelled in NumPy and checked on the CPU against the oracle's
masked iteration on the densified X and M (M = w0 at every unstored entry).

`SparseImplicitWRRI` is also the CPU model the GPU tests (test_gpu_sparse_implicit.py) import."""
import numpy as np
import pytest

import rri_oracle as orc
from conftest import relfro
from sparse_scheme import EPS, Side, SparseWRRI, solve_vector_c


class ImplicitSide(Side):
    """one orientation whose copy holds S = mt E + w0 x, mt = m - w0 (m = 1 without entry weights)"""

    def __init__(self, seg, idx, x, wgt, nseg, w0):
        super(ImplicitSide, self).__init__(seg, idx, x, wgt, nseg)
        self.w0 = w0
        self.mt = (np.ones_like(self.x) if self.wgt is None else self.wgt) - w0

    def residual(self, A, B):
        """sp_residual_rows_kernel / sp_residual_kernel in shifted mode"""
        E = self.x - np.einsum('el,el->e', A[self.seg], B[self.idx])
        self.E = self.mt * E + self.w0 * self.x

    def half_step(self, pend_other, pend_own, oth_old, oth_new, own_cur):
        """sp_entry in shifted mode: the stored-entry part of (numer, denom)"""
        if pend_own is not None:
            opo, opn = pend_own
            qa, qb = pend_other
            self.E = self.E + self.mt * (qa[self.idx] * opo[self.seg] - qb[self.idx] * opn[self.seg])
        ehs = self.E + self.mt * own_cur[self.seg] * oth_old[self.idx]
        g = oth_new[self.idx]
        numer = np.bincount(self.seg, weights=g * ehs, minlength=self.nseg)
        denom = np.bincount(self.seg, weights=self.mt * g * g, minlength=self.nseg)
        return numer, denom


class SparseImplicitWRRI(SparseWRRI):
    """the scheme with unstored weight w0: per half-step the stored-entry sums of the shifted copies plus the rank-k part
    -w0 sum_{s!=t} G_ts F_s (numer) and +w0 G_tt (denom) from one Gram row (sp_gram_rows_kernel,
    sp_implicit_final_kernel)"""

    def __init__(self, rows, cols, vals, n, d, weights=None, unstored_weight=0.0):
        self.n, self.d = n, d
        self.allreduce = None
        self.w0 = float(unstored_weight)
        self.csr = ImplicitSide(rows, cols, vals, weights, n, self.w0)
        self.csc = ImplicitSide(cols, rows, vals, weights, d, self.w0)

    def _T_step(self, W, T, t, S, reg_l1, reg_l2, ub):
        wt = W[:, t].copy()
        pend = S['csc']
        told = T[t].copy()
        numer, denom = self.csc.half_step(None if pend is None else (pend[0], pend[1]),
                                          None if pend is None else (pend[2], pend[3]), wt, wt, told)
        g = wt.dot(W)                                  # w_t' W
        go = g.copy()
        go[t] = 0
        numer = numer - self.w0 * go.dot(T)
        denom = denom + self.w0 * g[t]
        T[t] = solve_vector_c(numer - reg_l1, denom + reg_l2, EPS, ub)
        S['csc'] = (wt, wt, told, T[t].copy())
        S['told_cur'] = told

    def _W_step(self, W, T, t, S, reg_l1, reg_l2, ub):
        trow = T[t].copy()
        told = S['told_cur'] if S['told_cur'] is not None else trow
        pend = S['csr']
        wold = W[:, t].copy()
        numer, denom = self.csr.half_step(None if pend is None else (pend[2], pend[3]),
                                          None if pend is None else (pend[0], pend[1]), told, trow, wold)
        h = T.dot(trow)                                # T t_t' (this topic's row already updated)
        ho = h.copy()
        ho[t] = 0
        numer = numer - self.w0 * W.dot(ho)
        denom = denom + self.w0 * h[t]
        W[:, t] = solve_vector_c(numer - reg_l1, denom + reg_l2, EPS, ub)
        S['csr'] = (wold, W[:, t].copy(), told, trow)
        if S['told_cur'] is not None:
            S['csc'] = S['csr']
        S['told_cur'] = None

    def objective_terms(self, W, T):
        """(0.5 sum M (X - W T)^2 over all n x d entries, sum M X^2) without an n x d pass:
        0.5 [sum m E^2 + w0 (<W'W, T T'> - sum (x - E)^2)] over the stored entries"""
        c = self.csr
        E = c.x - np.einsum('el,el->e', W[c.seg], T.T[c.idx])
        m = 1.0 if c.wgt is None else c.wgt
        gh = float(np.sum(W.T.dot(W) * T.dot(T.T)))
        return (0.5 * float(np.sum(m * E ** 2) + self.w0 * (gh - np.sum((c.x - E) ** 2))),
                float(np.sum(m * c.x ** 2)))


def dense_M(I, J, n, d, w0, weights=None):
    """the dense weight matrix the sparse problem stands for: w0 everywhere, the entry weights (or 1) where stored"""
    M = np.full((n, d), float(w0))
    M[I, J] = 1.0 if weights is None else weights
    return M


def implicit_case(n, d, k, density, seed, weighted, stored_zeros=0, empty=True):
    """X sparse (I, J, vals) with an empty row and column and explicitly stored zeros, entry weights in [0.2, 3) when
    weighted (part of them below any w0 >= 0.2), W0, T0 >= 0"""
    rs = np.random.RandomState(seed)
    X, W0, T0 = orc.synth(n, d, max(1, k), k, sigma=0.1, seed=seed)
    mask = rs.rand(n, d) < density
    if empty:
        mask[rs.randint(n), :] = False
        mask[:, rs.randint(d)] = False
    I, J = np.nonzero(mask)
    vals = X[I, J].copy()
    if stored_zeros:
        vals[rs.choice(len(vals), stored_zeros, replace=False)] = 0.0
    wts = rs.uniform(0.2, 3.0, size=len(vals)) if weighted else None
    return I, J, vals, wts, W0, T0


@pytest.mark.parametrize('order', ['rri', 'hals'])
@pytest.mark.parametrize('weighted', [False, True])
@pytest.mark.parametrize('w0', [0.01, 0.5, 1.0, 2.0])
@pytest.mark.parametrize('k', [1, 3])
def test_scheme_matches_dense_oracle(order, weighted, w0, k):
    """after each of 3 sweeps the scheme equals the oracle's masked iteration on (X.toarray(), M) within 1e-12"""
    n, d = 37, 29
    I, J, vals, wts, W0, T0 = implicit_case(n, d, k, 0.3, seed=11 * k + int(10 * w0), weighted=weighted, stored_zeros=3)
    S = SparseImplicitWRRI(I, J, vals, n, d, weights=wts, unstored_weight=w0)
    Xd = np.zeros((n, d))
    Xd[I, J] = vals
    M = dense_M(I, J, n, d, w0, wts)
    W, T = np.maximum(W0, 0).copy(), np.maximum(T0, 0).copy()
    Wo, To = W.copy(), T.copy()
    for _ in range(3):
        S.sweeps(W, T, 1, order=order, check_copies=order == 'rri')
        orc.sweep(Xd, Wo, To, M, order=order)
        assert relfro(W, Wo) <= 1e-12 and relfro(T, To) <= 1e-12, (relfro(W, Wo), relfro(T, To))
    half, xsq = S.objective_terms(W, T)
    assert abs(half - 0.5 * np.sum(M * (Xd - W.dot(T)) ** 2)) <= 1e-12 * half
    assert abs(xsq - np.sum(M * Xd ** 2)) <= 1e-12 * xsq


@pytest.mark.parametrize('kw', [dict(reg_w_l1=0.01, reg_w_l2=0.1, reg_t_l1=0.02, reg_t_l2=0.2),
                                dict(ub_t=1.0), dict(fix_T=True)])
def test_scheme_regularisers_bounds_fix_T(kw):
    n, d, k = 41, 33, 3
    I, J, vals, wts, W0, T0 = implicit_case(n, d, k, 0.25, seed=5, weighted=True)
    S = SparseImplicitWRRI(I, J, vals, n, d, weights=wts, unstored_weight=0.3)
    Xd = np.zeros((n, d))
    Xd[I, J] = vals
    M = dense_M(I, J, n, d, 0.3, wts)
    W, T = np.maximum(W0, 0).copy(), np.maximum(T0, 0).copy()
    o = orc.nmf_oracle(Xd, k, W0, T0, max_iter=3, W_mat=M, fix_T=kw.get('fix_T', False), t_row_sum=kw.get('ub_t'),
                       **{a: b for a, b in kw.items() if a.startswith('reg')})
    S.sweeps(W, T, 3, **kw)
    assert relfro(W, o['W']) <= 1e-12 and relfro(T, o['T']) <= 1e-12


def test_zero_weight_is_the_observed_entries_scheme():
    """w0 = 0: the shifted copies are the plain residual and the rank-k part vanishes"""
    n, d, k = 30, 26, 4
    I, J, vals, wts, W0, T0 = implicit_case(n, d, k, 0.3, seed=2, weighted=True)
    a = SparseImplicitWRRI(I, J, vals, n, d, weights=wts, unstored_weight=0.0)
    b = SparseWRRI(I, J, vals, n, d, weights=wts)
    Wa, Ta = np.maximum(W0, 0).copy(), np.maximum(T0, 0).copy()
    Wb, Tb = Wa.copy(), Ta.copy()
    a.sweeps(Wa, Ta, 2)
    b.sweeps(Wb, Tb, 2)
    assert relfro(Wa, Wb) <= 1e-14 and relfro(Ta, Tb) <= 1e-14
