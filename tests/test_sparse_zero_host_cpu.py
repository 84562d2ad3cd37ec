"""Host side of zero-filled sparse data: the sparse branches of tfidf / normalize equal the dense helpers (all-zero
rows and columns included), and the sparse R^2 formula of NMF_TM_Estimator.score equals the dense computation."""
import numpy as np
import pytest
import scipy.sparse as sp

from rri_nmf_b200._host import normalize, tfidf
from rri_nmf_b200.sklearn_interface import _r2_sparse


def _matrix(seed=0, n=40, d=25):
    rng = np.random.RandomState(seed)
    A = sp.random(n, d, density=0.2, random_state=rng, format='lil') * 5
    A[3, :] = 0                      # all-zero row
    A[:, 4] = 0                      # all-zero column
    A = A.tocsr()
    A[7, 2] = 0.0                    # an explicitly stored zero
    return A


@pytest.mark.filterwarnings('ignore::scipy.sparse.SparseEfficiencyWarning')
def test_tfidf_sparse_equals_dense():
    A = _matrix()
    out, idf = tfidf(A, return_idf=True)
    ref, ref_idf = tfidf(A.toarray(), return_idf=True)
    assert sp.isspmatrix_csr(out) or sp.issparse(out)
    assert np.array_equal(idf, ref_idf)
    assert np.array_equal(out.toarray(), ref)


@pytest.mark.filterwarnings('ignore::scipy.sparse.SparseEfficiencyWarning')
@pytest.mark.parametrize('dim', [1, 0])
def test_normalize_sparse_equals_dense(dim):
    A = _matrix(1)
    out = normalize(A, dim)
    ref = normalize(A.toarray(), dim)
    assert sp.issparse(out)
    np.testing.assert_allclose(out.toarray(), ref, rtol=1e-14, atol=1e-16)
    if dim == 1:
        assert out[3].nnz == A.shape[1]                   # the zero row becomes the stored uniform row 1/d
        np.testing.assert_array_equal(out[3].toarray(), np.full((1, A.shape[1]), 1.0 / A.shape[1]))
    np.testing.assert_allclose(normalize(tfidf(A)).toarray(), normalize(tfidf(A.toarray())), rtol=1e-14, atol=1e-16)


@pytest.mark.filterwarnings('ignore::scipy.sparse.SparseEfficiencyWarning')
def test_sparse_score_formula_equals_dense():
    """the R^2 that score() takes on sparse input (SST and SSE from ||X||^2, the column mean and the k x k products)
    against the dense sums of sklearn_interface.py:339-345"""
    A = _matrix(2)
    rng = np.random.RandomState(3)
    W, T = rng.rand(A.shape[0], 4), rng.rand(4, A.shape[1])
    X = A.toarray()
    SST = ((X - np.mean(X, axis=0)) ** 2).sum()
    SSE = ((X - W @ T) ** 2).sum()
    assert abs(_r2_sparse(A, W, T) - (1 - SSE / SST)) < 1e-12
