"""Observed-entries WRRI with rank-one weights on the unstored entries (nmf(..., unstored_weight=w0,
unstored_row_weight=a, unstored_col_weight=b), rri_set_unstored_weight_vectors): the unstored entry (i, j) weighs
u_ij = w0 a_i b_j.  The scheme of rri_nmf_b200/csrc/sparse_kernels.cu + api.cu -- residual copies holding
S = mt E + u x with mt = m - u per stored entry, plus one weighted Gram row per half-step scaled per column (T-steps) or
per row (W-steps) -- modelled in NumPy and checked on the CPU against the oracle's masked iteration on the densified X
and M (M = u at every unstored entry).

`SparseImplicitVectorsWRRI` is also the CPU model the GPU tests (test_gpu_sparse_implicit_vectors.py) import."""
import numpy as np
import pytest

import rri_oracle as orc
from conftest import relfro
from sparse_scheme import EPS, solve_vector_c
from test_sparse_implicit_scheme_cpu import ImplicitSide, SparseImplicitWRRI, implicit_case


class RankOneSide(ImplicitSide):
    """one orientation whose copy holds S = mt E + u x, u = w0 a_i b_j, mt = m - u (m = 1 without entry weights)"""

    def __init__(self, seg, idx, x, wgt, nseg, w0, vseg, vidx):
        super(RankOneSide, self).__init__(seg, idx, x, wgt, nseg, w0)
        self.u = w0 * (vseg[self.seg] * vidx[self.idx])         # (a_i b_j: the same bits in both orientations)
        self.mt = (np.ones_like(self.x) if self.wgt is None else self.wgt) - self.u

    def residual(self, A, B):
        """sp_residual_rows_kernel / sp_residual_kernel in rank-one mode"""
        E = self.x - np.einsum('el,el->e', A[self.seg], B[self.idx])
        self.E = self.mt * E + self.u * self.x


class SparseImplicitVectorsWRRI(SparseImplicitWRRI):
    """the scheme with rank-one unstored weights: per half-step the stored-entry sums of the shifted copies (sp_entry with
    mt streamed as the weights) plus -w0 b_j sum_{s!=t} G^a_ts T_sj, +w0 b_j G^a_tt with G^a = W' diag(a) W in a T-step,
    and -w0 a_i sum_{s!=t} H^b_ts W_is, +w0 a_i H^b_tt with H^b = T diag(b) T' in a W-step"""

    def __init__(self, rows, cols, vals, n, d, weights=None, unstored_weight=0.0, a=None, b=None):
        self.n, self.d = n, d
        self.allreduce = None
        self.w0 = float(unstored_weight)
        self.a = np.ones(n) if a is None else np.asarray(a, dtype=np.float64)
        self.b = np.ones(d) if b is None else np.asarray(b, dtype=np.float64)
        self.csr = RankOneSide(rows, cols, vals, weights, n, self.w0, self.a, self.b)
        self.csc = RankOneSide(cols, rows, vals, weights, d, self.w0, self.b, self.a)

    def _T_step(self, W, T, t, S, reg_l1, reg_l2, ub):
        wt = W[:, t].copy()
        pend = S['csc']
        told = T[t].copy()
        numer, denom = self.csc.half_step(None if pend is None else (pend[0], pend[1]),
                                          None if pend is None else (pend[2], pend[3]), wt, wt, told)
        g = (wt * self.a).dot(W)                       # row t of W' diag(a) W
        go = g.copy()
        go[t] = 0
        numer = numer - self.w0 * self.b * go.dot(T)
        denom = denom + self.w0 * self.b * g[t]
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
        h = T.dot(trow * self.b)                       # row t of T diag(b) T' (this topic's row already updated)
        ho = h.copy()
        ho[t] = 0
        numer = numer - self.w0 * self.a * W.dot(ho)
        denom = denom + self.w0 * self.a * h[t]
        W[:, t] = solve_vector_c(numer - reg_l1, denom + reg_l2, EPS, ub)
        S['csr'] = (wold, W[:, t].copy(), told, trow)
        if S['told_cur'] is not None:
            S['csc'] = S['csr']
        S['told_cur'] = None

    def objective_terms(self, W, T):
        """0.5 [sum m E^2 + w0 (<W' diag(a) W, T diag(b) T'> - sum a_i b_j (x - E)^2)] over the stored entries"""
        c = self.csr
        E = c.x - np.einsum('el,el->e', W[c.seg], T.T[c.idx])
        m = 1.0 if c.wgt is None else c.wgt
        ab = self.a[c.seg] * self.b[c.idx]
        gh = float(np.sum((W.T * self.a).dot(W) * (T * self.b).dot(T.T)))
        return (0.5 * float(np.sum(m * E ** 2) + self.w0 * (gh - np.sum(ab * (c.x - E) ** 2))),
                float(np.sum(m * c.x ** 2)))


def dense_M_vectors(I, J, n, d, w0, a, b, weights=None):
    """the dense weight matrix of the rank-one scheme: w0 a_i b_j everywhere, the entry weights (or 1) where stored"""
    M = float(w0) * np.outer(np.ones(n) if a is None else a, np.ones(d) if b is None else b)
    M[I, J] = 1.0 if weights is None else weights
    return M


def vectors_case(n, d, k, density, seed, weighted, which, zeros=True):
    """implicit_case (an empty row and column, 3 stored zeros, entry weights in [0.2, 3)) plus a over the rows and b
    over the columns in [0, 4) (`which` in 'a', 'b', 'ab'), with zeros inside both at rows / columns that hold entries;
    b follows item popularity (column counts ** 0.5, rescaled), so that some u exceed the entry weights"""
    I, J, vals, wts, W0, T0 = implicit_case(n, d, k, density, seed, weighted, stored_zeros=3)
    rs = np.random.RandomState(seed + 1000)
    a = rs.uniform(0.1, 4.0, n) if 'a' in which else None
    b = None
    if 'b' in which:
        cnt = np.bincount(J, minlength=d).astype(np.float64)
        b = cnt ** 0.5
        b = 3.0 * b / b.max() + rs.uniform(0.0, 0.5, d)
    if zeros:
        if a is not None:
            a[np.unique(I)[:2]] = 0.0
        if b is not None:
            b[np.unique(J)[-2:]] = 0.0
    return I, J, vals, wts, W0, T0, a, b


@pytest.mark.parametrize('order', ['rri', 'hals'])
@pytest.mark.parametrize('weighted', [False, True])
@pytest.mark.parametrize('which', ['a', 'b', 'ab'])
@pytest.mark.parametrize('k', [1, 3])
def test_scheme_matches_dense_oracle(order, weighted, which, k):
    """after each of 3 sweeps the scheme equals the oracle's masked iteration on (X.toarray(), M) within 1e-12, and the
    objective formula equals the dense one"""
    n, d, w0 = 37, 29, 0.4
    I, J, vals, wts, W0, T0, a, b = vectors_case(n, d, k, 0.3, 7 * k + len(which), weighted, which)
    S = SparseImplicitVectorsWRRI(I, J, vals, n, d, weights=wts, unstored_weight=w0, a=a, b=b)
    Xd = np.zeros((n, d))
    Xd[I, J] = vals
    M = dense_M_vectors(I, J, n, d, w0, a, b, wts)
    if weighted:
        assert np.any(wts < M.max())                       # entry weights below some u: mt < 0 there
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
    I, J, vals, wts, W0, T0, a, b = vectors_case(n, d, k, 0.25, 5, True, 'ab')
    S = SparseImplicitVectorsWRRI(I, J, vals, n, d, weights=wts, unstored_weight=0.3, a=a, b=b)
    Xd = np.zeros((n, d))
    Xd[I, J] = vals
    M = dense_M_vectors(I, J, n, d, 0.3, a, b, wts)
    W, T = np.maximum(W0, 0).copy(), np.maximum(T0, 0).copy()
    o = orc.nmf_oracle(Xd, k, W0, T0, max_iter=3, W_mat=M, fix_T=kw.get('fix_T', False), t_row_sum=kw.get('ub_t'),
                       **{x: y for x, y in kw.items() if x.startswith('reg')})
    S.sweeps(W, T, 3, **kw)
    assert relfro(W, o['W']) <= 1e-12 and relfro(T, o['T']) <= 1e-12


@pytest.mark.parametrize('order', ['rri', 'hals'])
def test_vectors_of_ones_are_the_scalar_scheme(order):
    """a = 1 and b = 1 give the scalar-w0 scheme (every formula reduces to it)"""
    n, d, k = 30, 26, 4
    I, J, vals, wts, W0, T0 = implicit_case(n, d, k, 0.3, seed=2, weighted=True)
    v = SparseImplicitVectorsWRRI(I, J, vals, n, d, weights=wts, unstored_weight=0.2, a=np.ones(n), b=np.ones(d))
    s = SparseImplicitWRRI(I, J, vals, n, d, weights=wts, unstored_weight=0.2)
    Wa, Ta = np.maximum(W0, 0).copy(), np.maximum(T0, 0).copy()
    Wb, Tb = Wa.copy(), Ta.copy()
    v.sweeps(Wa, Ta, 2, order=order)
    s.sweeps(Wb, Tb, 2, order=order)
    assert relfro(Wa, Wb) <= 1e-14 and relfro(Ta, Tb) <= 1e-14
    assert abs(v.objective_terms(Wa, Ta)[0] / s.objective_terms(Wb, Tb)[0] - 1) <= 1e-14
