"""The device-resident NNDSVD initialisation on sparse X (rri_nmf_b200/_device_init.py with a torch sparse CSR tensor):
the same torch code, run on the CPU with the two products served by torch sparse ops or by scipy, against the host
implementation on the scipy matrix (`_host.initialize_nmf`, sklearn's randomized_svd).  X is never densified."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

from conftest import relfro
from rri_nmf_b200._device_init import initialize_nmf_torch, randomized_svd_torch
from rri_nmf_b200._host import initialize_nmf, normalize

INITS = ['nndsvd', 'nndsvda', 'nndsvdar', 'random', 'smart_random']


def sparse_data(n, d, density, seed=0, dtype=np.float64):
    """non-negative low-rank-ish CSR matrix with empty rows and columns"""
    rs = np.random.RandomState(seed)
    X = sp.random(n, d, density=density, format='csr', random_state=rs, dtype=np.float64)
    X.data = (X.data + rs.rand(X.nnz) * (1 + (X.indices % 7))).astype(dtype)
    X = X.tocsr()
    X.sort_indices()
    return X


def to_torch(X):
    return torch.sparse_csr_tensor(torch.from_numpy(X.indptr).long(), torch.from_numpy(X.indices).long(),
                                   torch.from_numpy(X.data), size=X.shape, check_invariants=False)


class ScipyProducts(object):
    """X @ Q and X' @ Q by scipy on the host matrix"""

    def __init__(self, X):
        self.X = X
        self.calls = 0

    def right(self, Q):
        self.calls += 1
        return torch.from_numpy(np.asarray(self.X @ Q.numpy()))

    def left(self, Q):
        self.calls += 1
        return torch.from_numpy(np.asarray(self.X.T @ Q.numpy()))


@pytest.mark.parametrize('init', INITS)
@pytest.mark.parametrize('shape', [(300, 120), (90, 400)])
@pytest.mark.parametrize('via', ['torch', 'scipy'])
def test_sparse_initialize_matches_host(init, shape, via):
    n, d = shape
    X = sparse_data(n, d, 0.08, seed=1)
    W, T = initialize_nmf(X, 7, init, random_state=5)
    P = ScipyProducts(X) if via == 'scipy' else None
    Wt, Tt = initialize_nmf_torch(to_torch(X), 7, init, random_state=5, products=P)
    assert Wt.shape == (n, 7) and Tt.shape == (7, d)
    assert Wt.dtype == torch.float64 and Tt.dtype == torch.float64
    assert relfro(Wt.numpy(), W) <= 1e-8 and relfro(Tt.numpy(), T) <= 1e-8
    assert (Wt >= 0).all() and (Tt >= 0).all()
    if P is not None and init.startswith('nndsvd'):
        assert P.calls == 2 * 7 + 2 or P.calls == 2 * 4 + 2       # 2 * n_iter + 2 passes over X


def test_sparse_randomized_svd_matches_sklearn():
    from sklearn.utils.extmath import randomized_svd
    X = sparse_data(250, 140, 0.1, seed=3)
    U, s, Vt = randomized_svd(X, 6, random_state=3)
    Ut, st, Vtt = randomized_svd_torch(to_torch(X), 6, random_state=3)
    assert np.allclose(st.numpy(), s, rtol=1e-10)
    assert relfro(Ut.numpy(), U) <= 1e-8 and relfro(Vtt.numpy(), Vt) <= 1e-8


@pytest.mark.parametrize('weighted', [False, True])
def test_nmf_device_initialisation_step_sparse(weighted):
    """nmf()'s device-side initialisation step on a sparse X with optional 1-D entry weights (W_mat o X, NNDSVD, row
    normalisations: nmf.py:840-850) against the host path, on CPU tensors"""
    from rri_nmf_b200.nmf import _initialize_on_device
    X = sparse_data(200, 90, 0.1, seed=4)
    w = np.random.RandomState(1).rand(X.nnz) if weighted else None
    Xh = X.copy()
    if weighted:
        Xh.data = Xh.data * w
    W, T = initialize_nmf(Xh, 6, 'nndsvda', random_state=2)
    T = normalize(T) * 1.0
    W = normalize(W) * 2.0
    Wt, Tt = _initialize_on_device(to_torch(X), torch.from_numpy(w) if weighted else None, 6, 'nndsvda', 2, 1.0, 2.0,
                                   products=ScipyProducts(Xh))
    assert relfro(Wt.numpy(), W) <= 1e-8 and relfro(Tt.numpy(), T) <= 1e-8


def test_mean_is_over_all_entries():
    """'nndsvda' fills the zeros of W and T with sum(stored values) / (n * d)"""
    X = sparse_data(120, 80, 0.05, seed=6)
    Wt, Tt = initialize_nmf_torch(to_torch(X), 4, 'nndsvda', random_state=0)
    avg = X.data.sum() / (120 * 80)
    filled = np.concatenate([Wt.numpy().ravel(), Tt.numpy().ravel()])
    assert np.isclose(filled, avg, rtol=1e-12, atol=0).any()


def test_no_dense_n_by_d_is_formed():
    """1 000 000 x 500 000 (4 TB if dense) with 20 000 stored entries initialises in O((n + d) (k + 10) + nnz)"""
    n, d = 1000000, 500000
    rs = np.random.RandomState(0)
    rows = np.sort(rs.randint(0, n, 20000))
    cols = rs.randint(0, d, 20000)
    X = sp.csr_matrix((rs.rand(20000) + 0.5, (rows, cols)), shape=(n, d))
    X.sum_duplicates()
    X.sort_indices()
    Wt, Tt = initialize_nmf_torch(to_torch(X), 2, 'nndsvd', random_state=0)
    assert Wt.shape == (n, 2) and Tt.shape == (2, d)
    assert bool(torch.isfinite(Wt).all()) and bool(torch.isfinite(Tt).all())
    assert float(Wt.sum()) > 0 and float(Tt.sum()) > 0

