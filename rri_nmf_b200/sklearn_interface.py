"""sklearn-style estimators over the device sweep engine -- the surface of the reference's
src/rri_nmf/sklearn_interface.py (NMF_TM_Estimator :185-345, NMF_RS_Estimator :14-182): same constructor
parameters, methods and attributes (`W`, `T`, `nmf_outputs`, `idf`, `min_rating`, `max_rating`, `Xpred`),
plus the sklearn-conventional read-only aliases `components_` (= T), `n_components` (= k) and
`reconstruction_err_` that BASELINE.json's north_star asks for.

Additional constructor arguments: `device`, `update_order`, `math` (forwarded to `nmf`); `NMF_RS_Estimator` also
takes `sparse=True` to keep the (i, j, rating) triples sparse all the way to the device (observed-entries engine,
traffic proportional to the number of ratings) instead of densifying them as the reference does; `NMF_TM_Estimator`
takes `sparse=True` to keep scipy.sparse document-term matrices sparse in the interleaved order (see below).

`NMF_TM_Estimator` takes scipy.sparse document-term matrices in fit, fit_transform, one_iter, transform and score.  With
update_order='hals' X stays sparse all the way to the device (nmf(..., unstored='zero'): unstored entries are zeros).
With the default update_order='rri' the estimator densifies X and runs the reference-exact interleaved order, unless it
was built with `sparse=True`: then X stays sparse in that order too (one pass over the stored entries per topic).
"""
import numpy as np
import scipy.sparse as sp
import sklearn.base
from sklearn.model_selection import train_test_split
from sklearn.utils.validation import check_X_y, check_array

import torch

from ._host import normalize, tfidf
from .nmf import nmf

_EMPTY = np.array([])


def _np(a):
    return a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else a


def _r2_sparse(X, W, T):
    """1 - SSE / SST of sklearn_interface.py:339-345 for a scipy.sparse X without an n x d temporary, in fp64:
    SST = ||X||^2 - n ||mean||^2,  SSE = ||X||^2 - 2 <X T', W> + <W'W, T T'>"""
    W = np.asarray(W, dtype=np.float64)
    T = np.asarray(T, dtype=np.float64)
    xsq = float(X.multiply(X).sum())
    mean = np.asarray(X.mean(axis=0)).ravel()
    SST = xsq - X.shape[0] * float(mean @ mean)
    SSE = xsq - 2.0 * float(np.sum(np.asarray(X @ T.T) * W)) + float(np.sum((W.T @ W) * (T @ T.T)))
    return 1 - SSE / SST


class _FactorMixin(object):
    """W/T bookkeeping shared by the two estimators (sparsify/densify: sklearn_interface.py:42-57)."""

    def sparsify(self):
        self.W = sp.csr_matrix(self.W) if not sp.issparse(self.W) else self.W.tocsr()
        self.T = sp.csr_matrix(self.T) if not sp.issparse(self.T) else self.T.tocsr()

    def densify(self):
        if sp.issparse(self.W):
            self.W = self.W.toarray()
        if sp.issparse(self.T):
            self.T = self.T.toarray()

    def _warm_start(self):
        """continue from a previous fit when W/T are populated (sklearn_interface.py:104-112, :253-261)"""
        self.densify()
        W_in = self.W if np.size(self.W) > 0 else []
        T_in = self.T if np.size(self.T) > 0 else []
        return W_in, T_in

    def _device_kwargs(self):
        return dict(device=self.device, update_order=self.update_order, math=self.math)

    # sklearn-conventional aliases
    @property
    def components_(self):
        return self.T

    @property
    def n_components(self):
        return self.k

    @property
    def reconstruction_err_(self):
        """||M o (X - WT)||_F of the last fit (M = observed-entry mask for the recommender)."""
        return getattr(self, '_reconstruction_err', None)


class NMF_TM_Estimator(_FactorMixin, sklearn.base.BaseEstimator, sklearn.base.TransformerMixin):
    """Topic-model NMF: rows of W and T on the simplex (sklearn_interface.py:185-345)."""

    def __init__(self, n, d, k, wr1=0, wr2=0, tr1=0, tr2=0, random_state=0, handle_tfidf=False,
                 handle_normalization=False, max_iter=300, W=_EMPTY, T=_EMPTY, nmf_kwargs={},
                 do_final_project_W=True, device=None, update_order='rri', math='ieee', sparse=False):
        self.n, self.d, self.k = n, d, k
        self.wr1, self.wr2, self.tr1, self.tr2 = wr1, wr2, tr1, tr2
        self.random_state = random_state
        self.handle_tfidf = handle_tfidf
        self.handle_normalization = handle_normalization
        self.max_iter = max_iter
        self.W, self.T = W, T
        self.nmf_kwargs = nmf_kwargs
        self.do_final_project_W = do_final_project_W
        self.device, self.update_order, self.math = device, update_order, math
        self.sparse = sparse

    def _keep_sparse(self, X):
        """sparse X goes to the device as it is in block order, and in the interleaved order with sparse=True;
        otherwise the interleaved order runs on its dense form"""
        return sp.issparse(X) and (self.update_order == 'hals' or self.sparse)

    def _prep(self, X, fit):
        if self._keep_sparse(X):
            X = sp.csr_matrix(X)
            if self.handle_tfidf:
                if fit:
                    X, self.idf = tfidf(X, return_idf=True)
                else:
                    X = X.multiply(self.idf[None, :]).tocsr()
            if self.handle_normalization:
                X = normalize(X)
            return X
        X = np.asarray(X.toarray() if sp.issparse(X) else _np(X))
        if self.handle_tfidf:
            if fit:
                X, self.idf = tfidf(X, return_idf=True)
            else:
                X = X * self.idf
        if self.handle_normalization:
            X = normalize(X)
        return X

    def _run(self, X, max_iter, max_time):
        W_in, T_in = self._warm_start()
        X = self._prep(X, fit=True)
        kw = dict(self._device_kwargs())
        if sp.issparse(X):
            kw['unstored'] = 'zero'
        kw.update(self.nmf_kwargs)
        # sklearn_interface.py:269-276 / :300-308
        soln = nmf(X, self.k, max_iter=max_iter, max_time=max_time, project_W_each_iter=False, w_row_sum=1.0,
                   project_T_each_iter=True, t_row_sum=1.0, do_final_project_W=self.do_final_project_W,
                   W_in=W_in, T_in=T_in, reg_w_l1=self.wr1, reg_w_l2=self.wr2, reg_t_l1=self.tr1,
                   reg_t_l2=self.tr2, random_state=self.random_state, return_reconstruction_err=True, **kw)
        self.W = soln.pop('W')
        self.T = soln.pop('T')
        # ||X - W T||_F of the returned factors, evaluated by the engine on the device copy of X before it was
        # released (no n x d host temporary, no host GEMM)
        self._reconstruction_err = soln.pop('reconstruction_err')
        self.nmf_outputs = soln
        return self

    def fit_transform(self, X, y=None):
        Xv = X.data if sp.issparse(X) else np.asarray(_np(X))
        assert np.all(Xv >= 0), 'X must be non-negative'                      # sklearn_interface.py:251
        self._run(X, self.max_iter, 7200)
        return self.W

    def fit(self, X, y=None):
        self.fit_transform(X, y)
        return self

    def one_iter(self, X):
        """one more sweep from the current (W, T): sweep-level resume (sklearn_interface.py:284-314)"""
        return self._run(X, 1, 240)

    def transform(self, Xnew):
        """express Xnew in terms of the fitted topics: 4 W-only sweeps (sklearn_interface.py:320-334)"""
        Xnew = self._prep(Xnew, fit=False)
        kw = dict(self._device_kwargs(), unstored='zero') if sp.issparse(Xnew) else self._device_kwargs()
        soln = nmf(Xnew, self.k, max_iter=4, max_time=7200, project_W_each_iter=False, w_row_sum=1.0,
                   t_row_sum=1.0, T_in=self.T, do_final_project_W=self.do_final_project_W, fix_T=True,
                   reg_w_l1=self.wr1, reg_w_l2=self.wr2, reg_t_l1=self.tr1, reg_t_l2=self.tr2,
                   random_state=self.random_state, **kw)
        return soln['W']

    def constrained_transform(self, X):
        return self.transform(X)

    def score(self, X, y=None):
        """R^2 of the reconstruction of new X (sklearn_interface.py:339-345).  Sparse X kept sparse (block order, or
        sparse=True): no n x d array is formed -- SST = ||X||^2 - n ||mean||^2 and SSE = ||X||^2 - 2 <X T', W> + <W'W, T T'>, in fp64 on the host."""
        if self._keep_sparse(X):
            X = sp.csr_matrix(X, dtype=np.float64)
            return _r2_sparse(X, self.transform(X), self.T)
        X = np.asarray(X.toarray() if sp.issparse(X) else _np(X))
        SST = ((X - np.mean(X, axis=0)) ** 2).sum()
        W = self.transform(X)
        SSE = ((X - np.dot(W, self.T)) ** 2).sum()
        return 1 - SSE / SST


class NMF_RS_Estimator(_FactorMixin, sklearn.base.BaseEstimator):
    """Recommender NMF on observed (i, j, rating) entries: the masked WRRI path
    (sklearn_interface.py:14-182)."""

    def __init__(self, n, d, k, wr1=0, tr1=0, random_state=0, W=_EMPTY, T=_EMPTY, max_iter=30, nmf_kwargs={},
                 use_validation_early_stopping=True, device=None, update_order='rri', math='ieee', sparse=False):
        self.n, self.d, self.k = n, d, k
        self.max_iter = max_iter
        self.wr1, self.tr1 = wr1, tr1
        self.random_state = random_state
        self.min_rating = None
        self.max_rating = None
        self.Xpred = _EMPTY
        self.use_validation_early_stopping = use_validation_early_stopping
        self.W, self.T = W, T
        self.nmf_kwargs = nmf_kwargs
        self.device, self.update_order, self.math = device, update_order, math
        self.sparse = sparse

    def _observed(self, ij, r):
        """n*d matrix of the ratings: duplicates summed, zero ratings unobserved -- what
        coo_matrix(...).toarray() followed by `Xtr != 0` gives in the reference (sklearn_interface.py:78-83, :100-102)"""
        M = sp.coo_matrix((np.asarray(r, dtype=np.float64), (ij[:, 0], ij[:, 1])), shape=(self.n, self.d)).tocsr()
        M.sum_duplicates()
        M.eliminate_zeros()
        M.sort_indices()
        return M

    def fit(self, X, y=None):
        """X: (m, 2) integer (i, j) pairs; y: (m,) ratings (sklearn_interface.py:59-128)"""
        X, y = check_X_y(X, y)
        X = X.astype(np.int64)
        self.min_rating, self.max_rating = np.min(y), np.max(y)
        if self.use_validation_early_stopping:
            UItr, UIval, Rtr, Rval = train_test_split(X, y, test_size=0.05, random_state=0, stratify=None)
            Xtr = self._observed(UItr, Rtr)
            Xv = self._observed(UIval, Rval)
            Iv, Jv = Xv.nonzero()
            held = np.asarray(Xv[Iv, Jv]).ravel()
            lo, hi = float(self.min_rating), float(self.max_rating)

            held_dev = {}

            def RMSE_val(Xign, W, T):
                # validation RMSE over the held-out entries only, with the rating clip of
                # sklearn_interface.py:85-91; evaluated where W and T live.  nmf() hands this callback the device
                # tensors (`device_tensors`): W, T and X never return to the host between sweeps, and the held-out
                # triples are uploaded once.
                if isinstance(W, torch.Tensor):
                    if W.device not in held_dev:
                        held_dev[W.device] = (torch.as_tensor(Iv, device=W.device), torch.as_tensor(Jv, device=W.device),
                                              torch.as_tensor(held, device=W.device, dtype=W.dtype))
                    ii, jj, ref = held_dev[W.device]
                    pred = (W[ii, :] * T[:, jj].t()).sum(1).clamp(lo, hi)
                    return float(torch.sqrt(torch.mean((pred - ref) ** 2)))
                pred = np.clip(np.einsum('ik,ki->i', W[Iv, :], T[:, Jv]), lo, hi)
                return float(np.sqrt(np.mean((pred - held) ** 2)))

            RMSE_val.device_tensors = True
            self.early_stop = RMSE_val
        else:
            self.early_stop = False
            Xtr = self._observed(X, y)
        W_in, T_in = self._warm_start()
        kw = dict(self._device_kwargs())
        kw.update(self.nmf_kwargs)
        if self.sparse:
            data, W_mat_tr = Xtr, None                                # stored entries = observed entries
        else:
            data = Xtr.toarray()
            W_mat_tr = torch.from_numpy((data != 0).astype(np.uint8))   # sklearn_interface.py:100-102
        soln = nmf(data, self.k, max_iter=self.max_iter, max_time=7200, compute_obj_each_iter=True,
                   reset_topic_method=None, early_stop=self.early_stop, project_T_each_iter=False,
                   t_row_sum=1.0, project_W_each_iter=False, w_row_sum=None,
                   W_mat=W_mat_tr, W_in=W_in, T_in=T_in, reg_w_l1=self.wr1,
                   reg_t_l1=self.tr1, random_state=self.random_state, return_reconstruction_err=True,
                   **kw)   # sklearn_interface.py:116-123
        self.W = soln.pop('W')
        self.T = soln.pop('T')
        self._reconstruction_err = soln.pop('reconstruction_err')     # over the observed training entries, on device
        self.nmf_outputs = soln
        self.Xpred = _EMPTY
        return self

    def fit_from_Xtr(self, Xtr):
        """build the (i, j), rating lists from a (sparse or dense) n*d matrix (sklearn_interface.py:130-142)"""
        Xtr = Xtr.tocsr() if sp.issparse(Xtr) else sp.csr_matrix(Xtr)
        I, J = Xtr.nonzero()
        return self.fit(np.column_stack([I, J]), np.asarray(Xtr[I, J]).ravel())

    def transform(self, Xnew):
        """express Xnew in terms of the fitted topics (sklearn_interface.py:144-156).  Of the rank-one unstored weights
        in nmf_kwargs, the new rows keep unstored_weight and unstored_col_weight (the items); unstored_row_weight belongs
        to the fitted rows and is dropped."""
        if self.sparse:
            Xnew = sp.csr_matrix(Xnew, dtype=np.float64)
            Xnew.eliminate_zeros()
            mask = None
        else:
            Xnew = np.asarray(Xnew.toarray() if sp.issparse(Xnew) else Xnew, dtype=np.float64)
            mask = torch.from_numpy((Xnew != 0).astype(np.uint8))
        soln = nmf(Xnew, self.k, max_iter=4, max_time=7200, project_W_each_iter=False,
                   project_T_each_iter=False, W_mat=mask, T_in=self.T, fix_T=True, reg_w_l1=self.wr1,
                   reg_t_l1=self.tr1, t_row_sum=1.0, w_row_sum=None, reset_topic_method='random',
                   random_state=self.random_state,
                   **dict(self._device_kwargs(), **{a: b for a, b in self.nmf_kwargs.items() if a != 'unstored_row_weight'}))
        return soln['W']

    def make_Xpred(self):
        if np.size(self.Xpred) == 0:
            self.Xpred = np.clip(np.dot(self.W, self.T), a_min=self.min_rating, a_max=self.max_rating)

    def predict(self, X):
        self.make_Xpred()
        X = check_array(X).astype(np.int64)
        return self.Xpred[X[:, 0], X[:, 1]]

    def score(self, X, y=_EMPTY):
        """RMSE of the predictions (sklearn_interface.py:172-182)"""
        self.make_Xpred()
        if sp.issparse(X):
            X = X.toarray()
        if np.size(y) > 0:
            return np.sqrt(np.mean((y - self.predict(X)) ** 2))
        I, J = np.asarray(X).nonzero()
        return np.sqrt(np.mean((np.asarray(X)[I, J] - self.Xpred[I, J]) ** 2))
