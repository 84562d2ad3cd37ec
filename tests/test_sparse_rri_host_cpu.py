"""Host side of the interleaved order on zero-filled sparse data: the update_order policy of nmf() (the caller names the
order on zero-filled data) and the sparse max-residual-document search of the topic reset against NumPy on the
densified matrix."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

import rri_nmf_b200 as R
from rri_nmf_b200 import _lib
from rri_nmf_b200.nmf import max_resid_document_sparse


def _matrix(seed=0, n=60, d=45, density=0.15):
    A = sp.random(n, d, density=density, random_state=np.random.RandomState(seed), format='lil') * 3
    A[5, :] = 0                      # empty row
    A[:, 9] = 0                      # empty column
    A = A.tocsr()
    A.sort_indices()
    return A


def test_zero_filled_needs_an_explicit_order():
    X = _matrix()
    kw = dict(W_in=np.ones((60, 3)), T_in=np.ones((3, 45)), max_iter=1, unstored='zero')
    with pytest.raises(NotImplementedError, match="update_order='hals'.*toarray") as ei:
        R.nmf(X, 3, **kw)
    assert "update_order='rri'" in str(ei.value) and '\n' not in str(ei.value)
    with pytest.raises(ValueError, match="update_order"):
        R.nmf(X, 3, update_order='block', **kw)


@pytest.mark.skipif(torch.cuda.is_available(), reason='checks the behaviour on a CPU-only host')
def test_explicit_rri_order_reaches_the_device_path():
    X = _matrix()
    kw = dict(W_in=np.ones((60, 3)), T_in=np.ones((3, 45)), max_iter=1, unstored='zero')
    for order in ('rri', 'hals'):
        with pytest.raises(_lib.RriError):
            R.nmf(X, 3, update_order=order, **kw)
    with pytest.raises(_lib.RriError):            # fix_T (transform) needs no order
        R.nmf(X, 3, fix_T=True, **kw)


@pytest.mark.parametrize('seed,chunk', [(0, None), (1, 7), (2, 1), (3, 1000)])
@pytest.mark.parametrize('dtype', [torch.float64, torch.float32])
def test_max_resid_document_sparse_equals_dense(seed, chunk, dtype):
    X = _matrix(seed)
    rng = np.random.RandomState(seed + 10)
    k = 4
    W = rng.rand(X.shape[0], k) * 0.3
    T = rng.rand(k, X.shape[1]) * 0.3
    Rd = np.maximum(X.toarray() - W @ T, 0)
    ref_i = int(np.argmax((Rd ** 2).sum(1)))
    mi, cols, vals = max_resid_document_sparse(torch.from_numpy(X.indptr.astype(np.int64)),
                                               torch.from_numpy(X.indices.astype(np.int32)),
                                               torch.from_numpy(X.data).to(dtype), torch.from_numpy(W).to(dtype),
                                               torch.from_numpy(T).to(dtype), chunk_entries=chunk)
    assert mi == ref_i
    row = np.zeros(X.shape[1])
    row[cols.numpy()] = vals.double().numpy()
    tol = 1e-12 if dtype == torch.float64 else 1e-5
    assert np.max(np.abs(row - Rd[ref_i])) <= tol * max(1.0, np.abs(Rd[ref_i]).max())


def test_max_resid_document_first_of_ties():
    """identical rows: the first index wins, as np.argmax / torch.argmax on the dense residual"""
    X = sp.csr_matrix(np.array([[0, 0, 0], [1.0, 0, 2.0], [0, 0, 0], [1.0, 0, 2.0]]))
    W = np.zeros((4, 1))
    T = np.zeros((1, 3))
    mi, cols, vals = max_resid_document_sparse(torch.from_numpy(X.indptr.astype(np.int64)),
                                               torch.from_numpy(X.indices.astype(np.int32)), torch.from_numpy(X.data),
                                               torch.from_numpy(W), torch.from_numpy(T))
    assert mi == 1 and cols.tolist() == [0, 2] and vals.tolist() == [1.0, 2.0]
