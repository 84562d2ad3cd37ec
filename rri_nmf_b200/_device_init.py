"""NNDSVD initialisation with every pass over X on the device that holds X (SURVEY.md §8 row f3).

Behavioural reference: initialization.py:80-163 -- Boutsidis & Gallopoulos NNDSVD on a randomized partial SVD
(`sklearn.utils.extmath.randomized_svd`: Gaussian test matrix from the NumPy generator, normalised power
iterations, QR, SVD of the (k+10)-row projection, `svd_flip`).  The host version in `_host.py` needs X in host
memory and, at 200k x 20k, minutes of CPU time; here X stays where the sweep engine will read it, the 2*n_iter+2
streaming passes over it run through the engine's own contraction kernel (rri_gemm_nt with k+10 columns; library
GEMMs only when no engine is at hand: CPU tensors, the masked product W_mat o X), the small factorisations are
`torch.linalg.qr/svd`.  The same torch code runs on CPU tensors, which is how it is checked
against `_host.initialize_nmf` without a GPU (tests/test_device_init_cpu.py).

X may also be a torch sparse CSR tensor.  It is never densified: shape, dtype and device come from the tensor, the means
of 'nndsvda' / 'nndsvdar' / 'smart_random' are (sum of the stored values) / (n*d), and on a CUDA device the products
must come from the sweep engine (`RRIEngine.products` on a sparse handle: rri_spmm, the SpMM kernel of the zero-filled
block order).  The workspace is O((n + d) * (k + 10) + nnz).
"""
import numpy as np
import torch

from ._host import _rng


def _span_normalize(A):
    """Orthonormal basis of the columns of A.  sklearn's default normaliser between power iterations is
    scipy.linalg.lu(A, permute_l=True)[0]; any basis of the same column space gives the same final factors up to
    rounding, and the thin QR needs no n x n permutation matrix (torch.linalg.lu returns P dense: 160 GB at
    n = 200 000)."""
    Q, _ = torch.linalg.qr(A, mode='reduced')
    return Q


def _is_sparse(M):
    return M.layout != torch.strided


def _mean(M):
    """mean over all n*d entries; the unstored entries of a sparse M are zeros"""
    if _is_sparse(M):
        return M.values().sum() / (M.shape[0] * M.shape[1])
    return M.mean()


class _TorchProducts(object):
    """the two streaming products of the randomized SVD as library GEMMs (CPU tensors, or no engine at hand)"""

    def __init__(self, M):
        if _is_sparse(M) and M.is_cuda:
            raise ValueError('a sparse X on a CUDA device needs the engine products (RRIEngine.products: rri_spmm)')
        self.M = M

    def right(self, Q):          # M @ Q      [n, r]
        return self.M @ Q

    def left(self, Q):           # M' @ Q     [d, r]
        return self.M.t() @ Q


def randomized_svd_torch(M, n_components, random_state=None, n_oversamples=10, products=None):
    """sklearn.utils.extmath.randomized_svd(M, n_components, random_state=...) with its defaults
    (n_iter='auto', transpose='auto', flip_sign=True; the power iterations are re-orthonormalised by a thin QR where
    sklearn's 'auto' uses LU -- same subspace) on M's device.
    M: dense 2-D torch tensor (float32 or float64) or sparse CSR tensor; it is only ever used as a product operand (no
    copy, no transpose materialised).  `products` (optional): object with right(Q) = M @ Q and left(Q) = M' @ Q -- the sweep engine's
    own streaming contraction (`RRIEngine.products`, rri_gemm_nt: the tcgen05 kernel in TF32 mode, the IEEE SIMT
    kernel otherwise) -- so that the 2*n_iter + 2 passes over X run through the repo's kernels.
    Returns (U[n,k], s[k], Vt[k,d])."""
    P = products if products is not None else _TorchProducts(M)
    rs = _rng(random_state)
    n_random = n_components + n_oversamples
    n_samples, n_features = M.shape
    n_iter = 7 if n_components < 0.1 * min(M.shape) else 4
    transpose = n_samples < n_features
    # A = M' when transposed: A @ Q = M' @ Q (left product), A' @ Q = M @ Q (right product)
    A_mm = P.left if transpose else P.right
    At_mm = P.right if transpose else P.left
    A_cols = n_samples if transpose else n_features
    Q = rs.normal(size=(A_cols, n_random))
    if M.dtype == torch.float32:
        Q = Q.astype(np.float32, copy=False)
    Q = torch.from_numpy(Q).to(M.device)
    normalize = _span_normalize if n_iter > 2 else (lambda x: x)
    for _ in range(n_iter):
        Q = normalize(A_mm(Q))
        Q = normalize(At_mm(Q))
    Q, _ = torch.linalg.qr(A_mm(Q), mode='reduced')
    Bt = At_mm(Q)                            # A'Q, the transpose of Q'A
    if _is_sparse(M):
        # The factors of a sparse X can be far larger than X: the SVD of the r x A_cols matrix Q'A through a thin QR
        # of its transpose, A'Q = Qb Rb, and the r x r SVD of Rb' (a library SVD of the wide matrix itself needs
        # several copies of it).  Same factorisation up to rounding; the signs are fixed by svd_flip below.
        Qb, Rb = torch.linalg.qr(Bt, mode='reduced')
        del Bt
        Uhat, s, Vrt = torch.linalg.svd(Rb.t())
        Vt = Vrt @ Qb.t()
        del Qb
    else:
        Uhat, s, Vt = torch.linalg.svd(Bt.t(), full_matrices=False)
        del Bt
    U = Q @ Uhat
    del Q
    # svd_flip: u_based_decision unless transposed (then the rows of Vt are the columns of the caller's U)
    if not transpose:
        idx = U.abs().argmax(dim=0)
        signs = torch.sign(U[idx, torch.arange(U.shape[1], device=U.device)])
    else:
        idx = Vt.abs().argmax(dim=1)
        signs = torch.sign(Vt[torch.arange(Vt.shape[0], device=Vt.device), idx])
    U.mul_(signs[None, :])
    Vt.mul_(signs[:, None])
    k = n_components
    if transpose:
        return Vt[:k, :].t(), s[:k], U[:, :k].t()
    return U[:, :k], s[:k], Vt[:k, :]


def initialize_nmf_torch(X, n_components, init=None, eps=1e-6, random_state=None, products=None):
    """initialize_nmf (initialization.py:9-163, `_host.initialize_nmf`) for a dense or sparse CSR torch tensor X on any device;
    returns torch tensors (W[n,k], T[k,d]) on X's device.  'random' / 'smart_random' draw from the NumPy generator
    on the host exactly like the reference (n*k + k*d numbers) and upload."""
    n, d = X.shape
    k = int(n_components)
    if init is None:
        init = 'nndsvd' if k < d else 'random'
    dev, dt = X.device, X.dtype
    if init == 'random':
        rng = _rng(random_state)
        T = rng.rand(k, d)                       # T is drawn first (initialization.py:84-85)
        W = rng.rand(n, k)
        return torch.from_numpy(W).to(dev), torch.from_numpy(T).to(dev)
    if init == 'smart_random':
        rng = _rng(random_state)
        scale = float(torch.sqrt(_mean(X) / k))
        T = np.abs(scale * rng.randn(k, d))
        W = np.abs(scale * rng.randn(n, k))
        return torch.from_numpy(W).to(dev), torch.from_numpy(T).to(dev)
    if init not in ('nndsvd', 'nndsvda', 'nndsvdar'):
        raise ValueError('Invalid init parameter: got %r instead of one of %r'
                         % (init, (None, 'random', 'smart_random', 'nndsvd', 'nndsvda', 'nndsvdar')))
    U, S, Vt = randomized_svd_torch(X, k, random_state=random_state, products=products)
    U, Vt = U.contiguous(), Vt.contiguous()
    # every singular pair is split into its positive and negative parts; per component the sign pattern carrying
    # more mass is kept (initialization.py:113-139); the leading pair is used as is up to sign (:108-109)
    # (one n x k / k x d temporary at a time: the factors of a sparse X can be far larger than X)
    nup, nun = torch.linalg.norm(U.clamp(min=0), dim=0), torch.linalg.norm((-U).clamp(min=0), dim=0)
    nvp, nvn = torch.linalg.norm(Vt.clamp(min=0), dim=1), torch.linalg.norm((-Vt).clamp(min=0), dim=1)
    mp, mn = nup * nvp, nun * nvn
    pos = mp > mn
    tiny = torch.finfo(dt).tiny
    sgn = torch.where(pos, 1.0, -1.0).to(dt)
    lam = torch.sqrt(S * torch.where(pos, mp, mn))
    W = (U * sgn[None, :]).clamp_(min=0).div_(torch.where(pos, nup, nun).clamp(min=tiny)[None, :]).mul_(lam[None, :])
    T = (Vt * sgn[:, None]).clamp_(min=0).div_(torch.where(pos, nvp, nvn).clamp(min=tiny)[:, None]).mul_(lam[:, None])
    W[:, 0] = torch.sqrt(S[0]) * U[:, 0].abs()
    T[0, :] = torch.sqrt(S[0]) * Vt[0, :].abs()
    W[W < eps] = 0
    T[T < eps] = 0
    if init == 'nndsvda':
        avg = _mean(X)
        W[W == 0] = avg
        T[T == 0] = avg
    elif init == 'nndsvdar':
        rng = _rng(random_state)
        avg = float(_mean(X))
        zw, zt = W == 0, T == 0
        # the reference fills W's zeros first, then T's, in C order (initialization.py:150-151)
        W[zw] = torch.from_numpy(np.abs(avg * rng.randn(int(zw.sum())) / 100)).to(device=dev, dtype=dt)
        T[zt] = torch.from_numpy(np.abs(avg * rng.randn(int(zt.sum())) / 100)).to(device=dev, dtype=dt)
    return W, T
