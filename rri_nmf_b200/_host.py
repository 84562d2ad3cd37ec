"""Host-side helpers around the device sweep: initialisation and the two preprocessing options of the
estimators.  They run once per fit, outside the hot path (SURVEY.md §2: out of scope for the device),
and are written against NumPy/SciPy only.

Behavioural references: initialization.py:9-163 (`initialize_nmf`), matrixops.py:124-179
(`normalize`, `tfidf`).
"""
import numpy as np


def _rng(random_state):
    if isinstance(random_state, np.random.RandomState):
        return random_state
    return np.random.RandomState(random_state)


def initialize_nmf(X, n_components, init=None, eps=1e-6, random_state=None, row_normalize=False):
    """Initial (W, T) for X ~ W T.  init in {None, 'random', 'smart_random', 'nndsvd', 'nndsvda',
    'nndsvdar'} with the semantics of initialization.py:80-163 (NNDSVD: Boutsidis & Gallopoulos 2008
    on a randomized partial SVD).  X may be a scipy.sparse matrix (never densified)."""
    import scipy.sparse as sp
    if not sp.issparse(X):
        X = np.asarray(X)
    n, d = X.shape
    k = int(n_components)
    if init is None:
        init = 'nndsvd' if k < d else 'random'
    if init == 'random':
        rng = _rng(random_state)
        T = rng.rand(k, d)            # T is drawn first (initialization.py:84-85)
        W = rng.rand(n, k)
    elif init == 'smart_random':
        rng = _rng(random_state)
        scale = np.sqrt(X.mean() / k)
        T = np.abs(scale * rng.randn(k, d))
        W = np.abs(scale * rng.randn(n, k))
    elif init in ('nndsvd', 'nndsvda', 'nndsvdar'):
        from sklearn.utils.extmath import randomized_svd
        U, S, Vt = randomized_svd(X, k, random_state=random_state)
        # split every singular pair into its positive and negative parts and keep, per component,
        # the sign pattern carrying more mass; the leading pair is non-negative up to a global sign
        Up, Un = np.maximum(U, 0), np.maximum(-U, 0)
        Vp, Vn = np.maximum(Vt, 0), np.maximum(-Vt, 0)
        nup, nun = np.linalg.norm(Up, axis=0), np.linalg.norm(Un, axis=0)
        nvp, nvn = np.linalg.norm(Vp, axis=1), np.linalg.norm(Vn, axis=1)
        mp, mn = nup * nvp, nun * nvn
        W = np.zeros_like(U)
        T = np.zeros_like(Vt)
        W[:, 0] = np.sqrt(S[0]) * np.abs(U[:, 0])
        T[0, :] = np.sqrt(S[0]) * np.abs(Vt[0, :])
        for j in range(1, k):
            if mp[j] > mn[j]:
                u, v, sig = Up[:, j] / nup[j], Vp[j] / nvp[j], mp[j]
            else:
                u, v, sig = Un[:, j] / nun[j], Vn[j] / nvn[j], mn[j]
            lam = np.sqrt(S[j] * sig)
            W[:, j], T[j, :] = lam * u, lam * v
        W[W < eps] = 0
        T[T < eps] = 0
        if init == 'nndsvda':
            avg = X.mean()
            W[W == 0] = avg
            T[T == 0] = avg
        elif init == 'nndsvdar':
            rng = _rng(random_state)
            avg = X.mean()
            W[W == 0] = np.abs(avg * rng.randn(int((W == 0).sum())) / 100)
            T[T == 0] = np.abs(avg * rng.randn(int((T == 0).sum())) / 100)
    else:
        raise ValueError('Invalid init parameter: got %r instead of one of %r'
                         % (init, (None, 'random', 'smart_random', 'nndsvd', 'nndsvda', 'nndsvdar')))
    if row_normalize:
        T = normalize(T)
    return W, T


def normalize(X, dim=1, zero_sum_fix=True):
    """Scale rows (dim=1) or columns (dim=0) to sum to 1; all-zero vectors become uniform
    (matrixops.py:124-163).  A scipy.sparse X gives a CSR matrix equal to the dense result (an all-zero row then
    stores its d uniform entries)."""
    import scipy.sparse as sp
    if sp.issparse(X):
        return _normalize_sparse(X, dim, zero_sum_fix)
    X = np.asarray(X, dtype=float)
    if dim == 0:
        return normalize(X.T, 1, zero_sum_fix).T
    if dim != 1:
        raise Exception('Unknown dim=%r' % (dim,))
    s = X.sum(1) + np.spacing(1)
    out = X / s[:, None]
    if zero_sum_fix:
        out[s < 1e-10, :] = 1.0 / X.shape[1]
    return out


def _normalize_sparse(X, dim, zero_sum_fix):
    import scipy.sparse as sp
    if dim == 0:
        return _normalize_sparse(X.T, 1, zero_sum_fix).T.tocsr()
    if dim != 1:
        raise Exception('Unknown dim=%r' % (dim,))
    X = sp.csr_matrix(X, dtype=float, copy=True)
    n, d = X.shape
    s = np.asarray(X.sum(1)).ravel() + np.spacing(1)
    X.data = X.data / np.repeat(s, np.diff(X.indptr))
    if not zero_sum_fix:
        return X
    zero = np.flatnonzero(s < 1e-10)
    if zero.size == 0:
        return X
    keep = np.ones(n)
    keep[zero] = 0.0
    uni = sp.csr_matrix((np.full(zero.size * d, 1.0 / d), (np.repeat(zero, d), np.tile(np.arange(d), zero.size))),
                        shape=(n, d))
    out = (sp.diags(keep) @ X + uni).tocsr()
    out.sort_indices()
    return out


def tfidf(X, return_idf=False):
    """tf-idf with idf = log(n / df) (matrixops.py:166-179).  A scipy.sparse X gives a CSR matrix equal to the dense
    result."""
    import scipy.sparse as sp
    if sp.issparse(X):
        X = sp.csr_matrix(X)
        idf = np.log(X.shape[0] / (np.asarray((X > 0).sum(0)).ravel() + np.spacing(1)))
        out = X.multiply(idf[None, :]).tocsr()
        return (out, idf) if return_idf else out
    X = np.asarray(X)
    n = X.shape[0]
    idf = np.log(n / ((X > 0).sum(0) + np.spacing(1)))
    out = X * idf
    return (out, idf) if return_idf else out
