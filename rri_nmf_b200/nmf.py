"""`nmf(X, k, **kwargs) -> dict` -- the reference's solver entry point (src/rri_nmf/nmf.py:98-560) with
its two inner loops (`for iter_no ... for t in range(k)`, :377, :415-476) running on the B200 through
librri_b200.so.  The outer shell stays Python: argument validation, initialisation, stopping policy,
early stop, topic reset, return dict -- same names, meaning and error behaviour as the reference.

Additional keyword-only arguments select the device path:
    device        torch device (default 'cuda'); there is NO CPU fallback
    update_order  'rri'  -- the reference's interleaved order (exact drop-in), or
                  'hals' -- block order: all T-steps then all W-steps (2 passes over X per sweep), or
                  None   -- the default: 'rri' for every input except zero-filled sparse data (unstored='zero'), where
                            the caller names the order (the two cost very different amounts there, see below)
    math          'ieee' (default) or 'tf32' (tcgen05 tensor-core contractions; float32 + 'hals')
    comm          engine.NcclComm for a row-sharded multi-GPU run (X, W_in, W_mat are the local shards)
    objective     how `obj_history` is evaluated: 'exact' = an explicit pass over X per evaluation (the reference's
                  TrueObjComputer, nmf.py:71-94); 'contraction' = ||X||^2 - 2<X T', W> + <W'W, T T'> from the block-order
                  sweep's own contraction (no extra pass over X; unmasked dense data, update_order='hals'); 'auto'
                  (default) = 'contraction' where it applies with IEEE arithmetic (fp64 / math='ieee'), else 'exact'.
                  With math='tf32' the contraction form carries the TF32 rounding of <X T', W> amplified by
                  ||X||^2 / ||X - WT||^2 (~1e-3 relative at a 3 % residual): ask for it explicitly.
    sparse_refresh_every  observed-entries (sparse X) engines, interleaved order: rebuild the maintained residual from the
                  factors every this many sweeps of one engine call (default 1: every sweep, bitwise re-entrant; larger
                  values skip 17 % of a sweep at config-4 shape and let fp rounding of the rank-one updates accumulate
                  over that many sweeps)
    return_reconstruction_err  also return 'reconstruction_err' = ||M^(1/2) o (X - W T)||_F of the returned factors,
                  evaluated on the device before the engine is released (the estimators' `reconstruction_err_`)
    init_on_device  where the NNDSVD initialisation runs when W_in/T_in are not both given: True = on the GPU that
                  holds X (`_device_init.py`; X never returns to the host), False = on the host (`_host.py`, NumPy /
                  sklearn, as the reference does), None (default) = on the device when X is already a CUDA tensor or
                  has 2^26 or more elements (n * d, stored or not), on the host otherwise.  Sparse X follows the same
                  rule; on the device its products go through rri_spmm and it is never densified.  Row-sharded runs
                  (comm=...) take W_in / T_in and initialise nothing.

X may also be a scipy.sparse matrix or a torch sparse CSR tensor, never densified.  What its unstored entries mean is
set by the keyword-only argument `unstored`:
    'missing' (default)  the STORED entries are the observed ones (the recommender setting of
                  sklearn_interface.py:78-102 without densifying the (i, j, rating) triples and without a dense W_mat);
                  W_mat is then None or a sparse matrix of the same structure holding entry weights.
    'zero'        X is an ordinary non-negative matrix stored sparsely (a tf-idf document-term matrix): every entry is
                  fitted, the unstored ones as 0 -- the result equals nmf(X.toarray(), ..., update_order=<the same>,
                  math='ieee') up to the summation order.  Needs math='ieee', no W_mat, and an explicit update_order
                  (fix_T=True runs the W-only sweeps whatever the order):
                  'hals'  the block-order half-steps take X T' and X' W from a sparse x dense contraction; the fast
                          choice (two passes over the stored entries per sweep).  Topic reset is not applied (an
                          emptied topic raises, as on the dense block order).
                  'rri'   the reference's interleaved order: per topic one pass over the stored entries in both
                          orientations (k passes per sweep, an order of magnitude slower than 'hals', an order of
                          magnitude faster than the densified matrix).  Topic reset works as on dense data: the
                          residual document is found over the stored entries, never densifying X.
                  Traffic grows with the stored entries, not with n * d.
With unstored='missing', the keyword-only `unstored_weight` w0 >= 0 (default 0) gives the unstored entries a weight of
their own (implicit feedback, one-class recommenders: unobserved pairs count as zeros of small weight w0, observed
ones with their W_mat weight, 1 without W_mat).  The result equals nmf(X.toarray(), ..., W_mat=M) with the dense M that
holds w0 at every unstored entry, up to the summation order, in both orders -- but nothing of size n x d is formed:
per entry the sweep moves the bytes of w0 = 0, plus O((n + d) k) per topic.  One GPU (no comm), no fix_W.
The keyword-only `unstored_row_weight` a (length n) and `unstored_col_weight` b (length d), NumPy or torch vectors >= 0,
make that weight rank-one: the unstored entry (i, j) weighs w0 a_i b_j (user- / item-oriented and item-popularity
schemes of one-class collaborative filtering; None = ones).  The result equals nmf(X.toarray(), ..., W_mat=M) with that
M; an unweighted sweep then streams the bytes of a weighted one.  They need unstored_weight > 0.
"""
import logging
import time

import numpy as np
import scipy.sparse as sp
import torch

from . import _lib
from ._device_init import initialize_nmf_torch
from ._host import initialize_nmf, normalize
from .engine import RRIEngine, EPS_DIV_BY_ZERO, check_unstored_weight, check_unstored_vectors

logger = logging.getLogger(__name__)
eps_div_by_zero = EPS_DIV_BY_ZERO          # nmf.py:52


class DeviceObjective(object):
    """Stand-in for the reference's TrueObjComputer (nmf.py:58-94) returned as 'obj_calculator'.

    While nmf() runs it evaluates the objective on the live engine.  When nmf() returns, the engine (and with it the
    device copy of X, the mask and the workspace) is released: the calculator keeps the value of the last
    evaluation and references to the caller's X / W_mat and the returned factors, and `true_objective()` rebuilds a
    short-lived engine on demand -- like the reference's object, which holds plain arrays.  Picklable."""

    def __init__(self, engine, W, T, regs, via_contraction=False):
        self.engine, self.W, self.T, self.regs = engine, W, T, regs
        self.obj = np.inf
        self._rebuild = None
        self.via_contraction = via_contraction      # unmasked block order: objective from the sweep's own contraction
        self._after_sweep = False                   # set by nmf() for the evaluation that directly follows a sweep

    def true_objective(self):
        if self.engine is not None:
            self.obj = self.engine.objective(self.W, self.T, via_contraction=self.via_contraction,
                                             reuse_last_sweep=self._after_sweep, **self.regs)
            self._after_sweep = False
        elif self._rebuild is not None:
            X, W_mat, device, dtype, order, unstored, unstored_weight, vectors = self._rebuild
            device = torch.device(device)
            with torch.cuda.device(device):
                if _is_sparse(X):
                    Xd, Md = _sparse_to_device(X, W_mat, device, dtype)
                else:
                    Xd, Md = _to_device(X, device, dtype), _mask_to_device(W_mat, device, dtype)
                # (a zero-filled sparse binding evaluates in the order of the fit; every other binding in 'rri')
                eng = RRIEngine(Xd, int(np.shape(self.W)[1]), W_mat=Md, order=order if unstored == 'zero' else 'rri',
                                unstored=unstored, unstored_weight=unstored_weight, unstored_row_weight=vectors[0],
                                unstored_col_weight=vectors[1])
                try:
                    self.obj = eng.objective(_to_device(self.W, device, dtype).contiguous(),
                                             _to_device(self.T, device, dtype).contiguous(), **self.regs)
                finally:
                    eng.close()
        return self.obj

    def _detach(self, X, W_mat, W, T, device, dtype, order, unstored='missing', unstored_weight=0.0,
                unstored_vectors=(None, None)):
        """called by nmf() before it closes the engine (the rank-one unstored weights are kept as host arrays)"""
        self.engine = None
        self.W, self.T = W, T
        vectors = tuple(None if v is None else (v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v))
                        for v in unstored_vectors)
        self._rebuild = (X, W_mat, str(device), dtype, order, unstored, unstored_weight, vectors)

    def __getstate__(self):
        st = dict(self.__dict__)
        st['engine'] = None
        return st


def _mask_to_device(W_mat, device, dtype):
    if W_mat is None:
        return None
    if isinstance(W_mat, torch.Tensor) and W_mat.dtype in (torch.uint8, torch.bool):
        return W_mat.to(device)
    return _to_device(W_mat, device, dtype)


def _universal_stopping_condition(obj_history, eps_stop=1e-4):
    """optimization.py:284-291"""
    if len(obj_history) < 2:
        return False
    return abs(obj_history[-1] - obj_history[-2]) <= eps_stop * abs(obj_history[0] - obj_history[1])


def _bcast_scalar(comm, v):
    """the same Python scalar on every rank of a row-sharded run (rank 0's)"""
    import torch.distributed as dist
    box = [v]
    dist.broadcast_object_list(box, src=0)
    return box[0]


def _all_any(comm, flag):
    """collective OR of a per-rank stop decision: the ranks must leave the sweep loop together, or the next
    exchange hangs"""
    if comm is None or getattr(comm, 'world', 1) <= 1:
        return bool(flag)
    import torch.distributed as dist
    res = [None] * comm.world
    dist.all_gather_object(res, bool(flag))
    return any(res)


def _all_mean(comm, v):
    if comm is None or getattr(comm, 'world', 1) <= 1:
        return v
    import torch.distributed as dist
    res = [None] * comm.world
    dist.all_gather_object(res, float(v))
    return float(np.mean(res))


def _is_empty(a):
    return a is None or int(np.prod(np.shape(a))) == 0


def _is_sparse(X):
    return sp.issparse(X) or (isinstance(X, torch.Tensor) and X.layout != torch.strided)


def _sparse_to_device(X, W_mat, device, dtype):
    """(torch sparse CSR tensor on `device`, 1-D entry weights or None) from a scipy.sparse matrix or a torch
    sparse tensor; indices sorted, duplicates summed (what coo_matrix(...).toarray() does in the reference,
    sklearn_interface.py:78-83)."""
    if isinstance(X, torch.Tensor):
        Xc = X.to_sparse_csr() if X.layout != torch.sparse_csr else X
        Xc = RRIEngine.csr_tensor(Xc.crow_indices(), Xc.col_indices(), Xc.values(), Xc.shape, device, dtype)
        wts = None
        if W_mat is not None:
            if not (isinstance(W_mat, torch.Tensor) and W_mat.dim() == 1):
                raise ValueError('with a sparse tensor X, W_mat is a 1-D tensor of nnz entry weights')
            wts = W_mat.to(device=device, dtype=dtype)
        return Xc, wts
    Xs = X.tocsr(copy=True)
    Xs.sum_duplicates()
    Xs.sort_indices()
    wts = None
    if W_mat is not None:
        if not sp.issparse(W_mat):
            raise ValueError('with sparse X, W_mat must be a sparse matrix with the structure of X (entry weights)')
        Ms = W_mat.tocsr(copy=True)
        Ms.sum_duplicates()
        Ms.sort_indices()
        if Ms.shape != Xs.shape or not (np.array_equal(Ms.indptr, Xs.indptr) and np.array_equal(Ms.indices, Xs.indices)):
            raise ValueError('sparse W_mat must store exactly the entries X stores')
        wts = torch.from_numpy(np.ascontiguousarray(Ms.data)).to(device=device, dtype=dtype)
    return RRIEngine.csr_tensor(Xs.indptr, Xs.indices, Xs.data, Xs.shape, device, dtype), wts


def _normalize_rows(A):
    """matrixops.py:124-163 (`normalize`, dim=1, zero_sum_fix) on a device tensor"""
    s = A.sum(1, keepdim=True) + float(np.spacing(1))
    out = A / s
    zero = (s < 1e-10).squeeze(1)
    if bool(zero.any()):
        out[zero, :] = 1.0 / A.shape[1]
    return out


def _initialize_on_device(Xd, W_mat, k, init, random_state, t_row_sum, w_row_sum, products=None):
    """nmf.py:840-850 (initialize_nmf on W_mat o X, then the row normalisations) with X staying on its device:
    initialization.py:80-163 through `_device_init.initialize_nmf_torch`.  products: the engine's streaming
    contraction for the passes over X (dense data: unmasked only, with W_mat the matrix being factorised is W_mat o X;
    sparse data: always, the engine applies the entry weights).  A sparse Xd with entry weights W_mat (1-D) is handed
    on as the CSR tensor of w o x (nnz values) for the means."""
    Xi = Xd
    if Xd.layout == torch.sparse_csr:
        if W_mat is not None:
            Xi = torch.sparse_csr_tensor(Xd.crow_indices(), Xd.col_indices(), Xd.values() * W_mat, size=tuple(Xd.shape),
                                         check_invariants=False)
    elif W_mat is not None:
        Mi = W_mat if isinstance(W_mat, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(W_mat))
        Xi = Xd * Mi.to(device=Xd.device, dtype=Xd.dtype)
        products = None
    Wi, Ti = initialize_nmf_torch(Xi, k, init, random_state=random_state, products=products)
    del Xi
    if t_row_sum is not None:
        Ti = _normalize_rows(Ti) * t_row_sum
    if w_row_sum is not None:
        Wi = _normalize_rows(Wi) * w_row_sum
    return Wi.to(Xd.dtype), Ti.to(Xd.dtype)


_STAGE = {'bufs': None, 'bytes': 0}
_STAGE_CHUNK_BYTES = 8 << 20     # measured on the B200 hosts (profiles/r02_h2d_staging_probe.txt): 4 threads x 8 MB
_STAGE_THREADS = 4               # chunks reach the pinned copy rate (53 vs 54 GB/s); torch's pageable .to(): 11 GB/s


def _stage_buffers(nbuf, nbytes):
    """module-level pinned staging buffers (page-locking host memory costs ~0.1 s per GB: pay it once per process)"""
    if _STAGE['bufs'] is None or len(_STAGE['bufs']) < nbuf or _STAGE['bytes'] < nbytes:
        _STAGE['bufs'] = [torch.empty(nbytes, dtype=torch.uint8).pin_memory() for _ in range(nbuf)]
        _STAGE['bytes'] = nbytes
    return _STAGE['bufs']


def _pageable_to_device(t, device):
    """Host -> device copy of a large PAGEABLE array (what a drop-in user passes) at close to the pinned rate:
    row chunks are copied into a few pinned staging buffers by worker threads (tensor.copy_ releases the GIL) and
    go to the device with asynchronous copies on a side stream, so the pageable -> pinned memcpy of one chunk
    overlaps the DMA of the others.  A single pin_memory() of the whole array would cost a second full host copy
    plus the page-locking of a data-sized allocation, serialised before the first byte moves."""
    import threading
    flat = t.reshape(-1).view(torch.uint8) if t.is_contiguous() else t.contiguous().reshape(-1).view(torch.uint8)
    total = flat.numel()
    out = torch.empty(t.shape, dtype=t.dtype, device=device)
    oflat = out.reshape(-1).view(torch.uint8)
    nthreads = max(1, min(_STAGE_THREADS, len(__import__('os').sched_getaffinity(0))))
    bufs = _stage_buffers(2 * nthreads, _STAGE_CHUNK_BYTES)
    nchunks = (total + _STAGE_CHUNK_BYTES - 1) // _STAGE_CHUNK_BYTES
    side = torch.cuda.Stream(device=device)
    side.wait_stream(torch.cuda.current_stream(device))
    errors = []

    def worker(w):
        try:
            torch.cuda.set_device(device)
            events = [None, None]
            for j, c in enumerate(range(w, nchunks, nthreads)):
                b = bufs[2 * w + (j & 1)]
                if events[j & 1] is not None:
                    events[j & 1].synchronize()            # the DMA that last read this buffer has finished
                lo = c * _STAGE_CHUNK_BYTES
                hi = min(total, lo + _STAGE_CHUNK_BYTES)
                b[:hi - lo].copy_(flat[lo:hi])              # pageable -> pinned (GIL released)
                with torch.cuda.stream(side):
                    oflat[lo:hi].copy_(b[:hi - lo], non_blocking=True)
                    ev = torch.cuda.Event()
                    ev.record(side)
                events[j & 1] = ev
            for ev in events:
                if ev is not None:
                    ev.synchronize()
        except Exception as ex:                             # surfaced by the caller
            errors.append(ex)

    threads = [threading.Thread(target=worker, args=(w,)) for w in range(nthreads)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    if errors:
        raise errors[0]
    torch.cuda.current_stream(device).wait_stream(side)
    return out


def _to_device(a, device, dtype):
    if isinstance(a, torch.Tensor):
        if a.device.type == 'cpu' and device.type == 'cuda' and a.dtype == dtype and not a.is_pinned() \
                and a.numel() * a.element_size() >= (64 << 20) and a.layout == torch.strided:
            return _pageable_to_device(a, device)
        return a.to(device=device, dtype=dtype, non_blocking=a.device.type == 'cpu' and a.is_pinned())
    a = np.ascontiguousarray(a)
    t = torch.from_numpy(a)
    if device.type == 'cuda' and t.dtype == dtype and not t.is_pinned() and t.numel() * t.element_size() >= (64 << 20):
        return _pageable_to_device(t, device)
    return t.to(device=device, dtype=dtype, non_blocking=True)


def nmf(X, k, w_row=None, W_mat=None, fix_W=False, fix_T=False, random_state=None, init='nndsvd', T_in=[],
        W_in=[], max_iter=200, max_time=600, eps_stop=1e-4, compute_obj_each_iter=False,
        project_W_each_iter=False, w_row_sum=None, do_final_project_W=True, project_T_each_iter=False,
        t_row_sum=None, early_stop=None, reset_topic_method='max_resid_document', fix_reset_seed=False,
        n_resets=23, reg_w_l2=0, reg_t_l2=0, reg_w_l1=0, reg_t_l1=0, diagnostics=[], store_gradients=False,
        ind_rows_to_store=None, eps_gauss_t=None, delta_gauss_t=None,
        *, device=None, update_order=None, math='ieee', comm=None, engine=None, sweeps_per_call=16,
        init_on_device=None, return_reconstruction_err=False, sparse_refresh_every=1, objective='auto',
        unstored='missing', unstored_weight=0.0, unstored_row_weight=None, unstored_col_weight=None):
    """Non-negative factorisation X ~ W T by rank-one residue iteration.  See the reference docstring
    (nmf.py:109-269) for the arguments; returns {'W', 'T', 'iter_cputime', 'random_state'[, 'obj_history',
    'obj_calculator', 'diagnostics']} (nmf.py:551-560).  W and T come back as the kind of array X was
    (NumPy in -> NumPy out, torch tensor in -> torch tensors on the device)."""
    lib = _lib.load()           # fail loudly before doing anything if the CUDA library is missing
    del lib
    if update_order not in (None, 'rri', 'hals'):
        raise ValueError("update_order must be 'rri', 'hals' or None")
    if unstored not in ('missing', 'zero'):
        raise ValueError("unstored must be 'missing' or 'zero'")
    zero_filled = unstored == 'zero' and _is_sparse(X)
    unstored_weight = check_unstored_weight(unstored_weight, _is_sparse(X), unstored)
    if unstored_weight > 0:
        if comm is not None:
            raise NotImplementedError('unstored_weight runs on one GPU (row shards are not implemented)')
        if fix_W:
            raise NotImplementedError('fix_W=True is not available with unstored_weight')
    unstored_vectors = check_unstored_vectors(unstored_row_weight, unstored_col_weight, X.shape[0], X.shape[1],
                                              unstored_weight)
    if zero_filled:
        if W_mat is not None:
            raise ValueError("unstored='zero' takes no W_mat: weights on a zero-filled matrix would be a dense n x d object")
        if math != 'ieee':
            raise ValueError("unstored='zero' runs with math='ieee' (the sparse contraction is not compute-bound)")
        if fix_W:
            raise NotImplementedError("fix_W=True is not available with unstored='zero'")
        if update_order is None and not fix_T:
            raise NotImplementedError("unstored='zero' needs an explicit order: update_order='hals' (block order, fast) or "
                                      "update_order='rri' (the reference's interleaved order, k passes per sweep), or "
                                      "densify with X.toarray()")
    if update_order is None:
        update_order = 'rri'
    n, d = X.shape
    rtv = {}
    numpy_io = not isinstance(X, torch.Tensor)

    # ---- argument policy, as nmf.py:280-315
    if project_T_each_iter and np.any([reg_w_l1, reg_t_l1]):
        logger.warning('This implementation can not solve project_T_each_iter=True with regularization. '
                       'Setting project_T_each_iter to False.')
        project_T_each_iter = False
    if (not project_T_each_iter and not t_row_sum) and (reg_t_l1 < 0 or reg_t_l2 < 0):
        logger.error('Unbounded objective. reg_t_l1=%s, reg_t_l2=%s', reg_t_l1, reg_t_l2)
        return {'W': np.ones((n, k)), 'T': np.ones((k, d)) * 1e6, 'obj_history': [-np.inf], 'iter_cputime': [0]}
    if (not project_W_each_iter and not w_row_sum) and (reg_w_l1 < 0 or reg_w_l2 < 0):
        logger.error('Unbounded objective. reg_w_l1=%s, reg_w_l2=%s', reg_w_l1, reg_w_l2)
        return {'W': np.ones((n, k)) * 1e6, 'T': np.ones((k, d)), 'obj_history': [-np.inf], 'iter_cputime': [0]}

    # ---- features of nmf() that are outside the accelerated path (SURVEY.md §2) fail loudly
    if w_row is not None:
        raise NotImplementedError('w_row (row weighting + W-only sub-solve, nmf.py:335-344, :531-539) is not '
                                  'on the device path; pre-scale X by sqrt(w_row) on the host')
    if eps_gauss_t or delta_gauss_t:
        raise NotImplementedError('the Gaussian DP mechanism (nmf.py:422-435) is not on the device path')
    if store_gradients:
        raise NotImplementedError('store_gradients: use RRIEngine.partials_T (the statistic of nmf.py:680-686)')
    if fix_W:
        # T-only sweeps: per topic the statistic comes from the engine (rri_partials_T, nmf.py:680-686 / :706-713),
        # the solve and the reference's W[:, t] *= nt1 rescaling (nmf.py:450-452) are a few device vector ops
        update_order = 'rri'
        if math != 'ieee':
            raise ValueError("fix_W=True runs with math='ieee'")
        if comm is not None:
            raise NotImplementedError('fix_W=True is not available on row shards')
    if w_row_sum is not None and not np.isscalar(w_row_sum):
        raise NotImplementedError('vector w_row_sum is not on the device path')
    sharded = comm is not None and getattr(comm, 'world', 1) > 1
    if sharded:
        # Row-sharded contract (INTEGRATION.md §4): every rank passes ITS rows of X / W_in / W_mat and the SAME T_in.
        # An initialisation computed per shard would give every rank a different T replica (garbage, silently), so
        # both factors must be given; T_in and random_state are then broadcast from rank 0 so that the replicas
        # are bit-identical from sweep 0 whatever the caller passed.
        if _is_empty(W_in) or _is_empty(T_in):
            raise ValueError('row-sharded runs (comm=...) need W_in (the local rows) and T_in (replicated): an '
                             'initialisation per shard would start the ranks from different T')
    if type(diagnostics) is not list:
        diagnostics = [diagnostics]
    if len(diagnostics) > 0:
        rtv['diagnostics'] = {f.__name__: [] for f in diagnostics}
    if random_state is None:
        random_state = int(time.time()) % 4294967296
    if sharded:
        random_state = _bcast_scalar(comm, random_state)
    t_global_start = time.time()
    max_time = max_time - 10                                     # nmf.py:333
    if n <= k:
        init = 'random'                                          # nmf.py:346-347
    start_time = time.process_time()

    # ---- device placement
    if device is None:
        device = X.device if isinstance(X, torch.Tensor) and X.is_cuda else torch.device('cuda')
    device = torch.device(device)
    if not torch.cuda.is_available():
        raise _lib.RriError('no CUDA device is available: rri_nmf_b200.nmf has no CPU fallback')
    if device.type != 'cuda':
        raise _lib.RriError('rri_nmf_b200.nmf runs on CUDA devices only (no CPU fallback)')
    if device.index is None:
        device = torch.device('cuda', torch.cuda.current_device())
    sparse_in = _is_sparse(X)
    if isinstance(X, torch.Tensor):
        dtype = X.dtype if X.dtype in (torch.float32, torch.float64) else torch.float64
    else:
        dtype = torch.float32 if (X.dtype if sparse_in else np.asarray(X).dtype) == np.float32 else torch.float64

    # ---- initialisation and validation, as nmf.py:819-880
    init_on_device = _init_on_device_rule(X, n, d, W_in, T_in, init_on_device, comm)
    W0, T0 = _host_start(X, W_mat, k, init, random_state, t_row_sum, w_row_sum, W_in, T_in, init_on_device)
    timing = {}
    _t0 = time.perf_counter()
    a_W_mat_user = W_mat
    with torch.cuda.device(device):
        if sparse_in:
            Xd, W_mat = _sparse_to_device(X, W_mat, device, dtype)
        else:
            Xd = _to_device(X, device, dtype)
        W_mat_user = a_W_mat_user
        Md = W_mat if sparse_in else _mask_to_device(W_mat, device, dtype)   # sparse: 1-D entry weights, already there
        # (no synchronisation here: the host -> device copy of X keeps running while the engine allocates its
        # workspace; the first kernel is stream-ordered behind it)
        timing['to_device_enqueue_s'] = time.perf_counter() - _t0   # host -> device copies of X (and W_mat) issued
        _t1 = time.perf_counter()
        own_engine = engine is None
        if engine is None:
            # (fix_T: the W-only sweeps are the same in both orders; on zero-filled data they run on a block-order
            # binding, which holds no interleaved-order partials)
            engine = RRIEngine(Xd, k, W_mat=Md, order='hals' if zero_filled and fix_T else update_order, math=math,
                               comm=comm, unstored=unstored, unstored_weight=unstored_weight,
                               unstored_row_weight=unstored_vectors[0], unstored_col_weight=unstored_vectors[1])
        timing['engine_setup_s'] = time.perf_counter() - _t1       # workspace, transposed copy of X, peer mapping
        try:
            W, T = _device_start(engine, Xd, W_mat, Md, k, init, random_state, t_row_sum, w_row_sum, W0, T0,
                                 init_on_device, timing)
            if sharded:
                import torch.distributed as dist
                dist.broadcast(T, src=0)
            _t2 = time.perf_counter()
            out = _solve(engine, X if sparse_in else Xd, W, T, rtv, locals())
            timing['solve_s'] = time.perf_counter() - _t2           # (rest of the H2D copy,) sweeps, device -> host copy of W, T
            out['timing'] = timing
            if return_reconstruction_err:
                Wd = W if isinstance(out['W'], np.ndarray) else out['W']
                Td = T if isinstance(out['T'], np.ndarray) else out['T']
                out['reconstruction_err'] = float(np.sqrt(2.0 * engine.objective_terms(Wd, Td)[0]))
            if 'obj_calculator' in out and own_engine:
                # the calculator outlives this call without pinning device memory (and stays picklable)
                out['obj_calculator']._detach(X, W_mat_user, out['W'], out['T'], device, dtype, engine.order,
                                              engine.unstored, engine.unstored_weight, engine.unstored_vectors)
            return out
        finally:
            if own_engine:
                _t3 = time.perf_counter()
                engine.close()
                timing['teardown_s'] = time.perf_counter() - _t3


# Widest stacked factor operand (models * k) of one models engine; more models run as groups one after another on the
# same device copy of X.  See DESIGN.md §6 for the measurement that chose it.
MODELS_WIDTH_CAP = 256


def _model_groups(n_models, k, cap=None):
    """sizes of the groups the models are run in: as many models of rank k per group as fit the width cap"""
    per = max(1, (MODELS_WIDTH_CAP if cap is None else cap) // int(k))
    return [min(per, n_models - i) for i in range(0, n_models, per)]


def _rank_groups(ranks, cap=None):
    """the groups (lists of model indices, each in caller order) that models of the given ranks run in: first fit by
    decreasing rank (ties in caller order) under the width cap"""
    cap = MODELS_WIDTH_CAP if cap is None else cap
    groups, widths = [], []
    for m in sorted(range(len(ranks)), key=lambda m: -ranks[m]):
        for g in range(len(groups)):
            if widths[g] + ranks[m] <= cap:
                groups[g].append(m)
                widths[g] += ranks[m]
                break
        else:
            groups.append([m])
            widths.append(ranks[m])
    return [sorted(g) for g in groups]


def nmf_models(X, k, random_state=None, W_in=None, T_in=None, **kwargs):
    """Several block-order factorisations of one matrix, X ~ W_m T_m for m = 0..b-1, sharing every pass over X.

    Restarts and consensus runs fit many models of one X.  Here the factors of up to MODELS_WIDTH_CAP / k models are
    stacked into one operand, so each block-order half-step reads X once for all of them (two passes per sweep instead
    of 2b); the row updates stay per model.  X is uploaded once.

    random_state: a list of seeds, one per model, and/or W_in, T_in: lists of starting factors (n x k, k x d).  The
    number of models is the length of the list(s) given.  Every other keyword argument is nmf()'s.  Each model starts
    exactly as nmf() would start it (host or device initialisation by the same rule, or its W_in / T_in), and returns
    what `nmf(X, k, random_state=s_m, update_order='hals', ...)` returns for it: a dict with 'W', 'T', 'iter_cputime',
    'random_state' and, with compute_obj_each_iter, 'obj_history'.  NNDSVD hardly depends on the seed: for restarts use
    init='random', 'smart_random' or 'nndsvdar', or pass starts.

    Each model stops on its own (the stopping rule of nmf() on its own objective history); the batch sweeps on until all
    have stopped or max_iter is reached.  A model whose sweep fails (an emptied topic, an unbounded objective,
    non-finite values) gets the dict {'error': <the exception nmf() would raise>, 'random_state': ...} and no factors;
    its factors are zeroed on the device and the others carry on.

    k may also be a sequence of ranks, one per model (choosing k: fit k = 2..20 in one call).  The lists given must then
    have its length (they may all be omitted: every model takes the time-based seed nmf() would take), W_in[m] is
    n x k[m], and the models run in groups of total width <= MODELS_WIDTH_CAP, packed first fit by decreasing rank; the
    results come back in the order of k.  With math='ieee' every model is bit-identical to its
    own nmf() run; with math='tf32' the models share the contraction's operand (and, with 16-bit copies of X, its
    power-of-two scale), which changes their rounding, not their accuracy.  The flags are read after every engine
    call: a model that produces non-finite values inside a call of several sweeps (sweeps_per_call) can disturb that
    shared scale for the rest of the call.

    Supported: dense unmasked X (fp32 / fp64), update_order='hals', math 'ieee' / 'tf32', the four regularisers,
    w_row_sum / t_row_sum as upper bounds, project_W_each_iter, do_final_project_W, compute_obj_each_iter, objective,
    eps_stop, max_iter, max_time, sweeps_per_call, init_on_device, device.  Everything else raises before any device
    work: NotImplementedError for W_mat, sparse X, unstored weight vectors, comm, update_order='rri', fix_W / fix_T, project_T_each_iter with
    t_row_sum, early_stop, diagnostics, w_row, the Gaussian mechanism, store_gradients, an engine, and
    return_reconstruction_err; ValueError for lists of different lengths and for ranks outside [1, 256].
    """
    import inspect
    defaults = {name: p.default for name, p in inspect.signature(nmf).parameters.items()
                if p.default is not inspect.Parameter.empty}
    unknown = sorted(set(kwargs) - set(defaults))
    if unknown:
        raise TypeError('nmf_models() got unexpected keyword arguments %s' % unknown)
    a = dict(defaults)
    a['update_order'] = 'hals'
    a.update(kwargs)
    lib = _lib.load()
    del lib

    # ---- what the shared contraction does not serve: refuse before any device work
    if a['W_mat'] is not None:
        raise NotImplementedError('nmf_models takes unmasked data (no W_mat)')
    if a['unstored_row_weight'] is not None or a['unstored_col_weight'] is not None:
        raise NotImplementedError('nmf_models takes dense X (no unstored weights)')
    if _is_sparse(X):
        raise NotImplementedError('nmf_models takes dense X')
    if a['comm'] is not None:
        raise NotImplementedError('nmf_models runs on one GPU (no comm)')
    if a['update_order'] == 'rri':
        raise NotImplementedError("nmf_models runs the block order (update_order='hals')")
    if a['update_order'] != 'hals':
        raise ValueError("update_order must be 'hals'")
    if a['fix_W'] or a['fix_T']:
        raise NotImplementedError('nmf_models does not take fix_W / fix_T')
    if a['project_T_each_iter'] and a['t_row_sum'] and not (a['reg_w_l1'] or a['reg_t_l1']):
        raise NotImplementedError('nmf_models does not take project_T_each_iter with t_row_sum')
    if a['early_stop']:
        raise NotImplementedError('nmf_models does not take early_stop')
    diagnostics = a['diagnostics'] if type(a['diagnostics']) is list else [a['diagnostics']]
    if diagnostics:
        raise NotImplementedError('nmf_models does not take diagnostics')
    if a['w_row'] is not None:
        raise NotImplementedError('w_row is not on the device path; pre-scale X by sqrt(w_row) on the host')
    if a['eps_gauss_t'] or a['delta_gauss_t']:
        raise NotImplementedError('the Gaussian DP mechanism (nmf.py:422-435) is not on the device path')
    if a['store_gradients']:
        raise NotImplementedError('nmf_models does not take store_gradients')
    if a['engine'] is not None:
        raise NotImplementedError('nmf_models builds its own engines (no engine=)')
    if a['return_reconstruction_err']:
        raise NotImplementedError('nmf_models does not take return_reconstruction_err')
    if a['w_row_sum'] is not None and not np.isscalar(a['w_row_sum']):
        raise NotImplementedError('vector w_row_sum is not on the device path')
    if a['math'] not in ('ieee', 'tf32'):
        raise ValueError("math must be 'ieee' or 'tf32'")
    if a['objective'] not in ('auto', 'exact', 'contraction'):
        raise ValueError("objective must be 'auto', 'exact' or 'contraction'")
    rank_list = isinstance(k, (list, tuple, np.ndarray))
    ks = [int(r) for r in k] if rank_list else [int(k)]
    for r in ks:
        if r < 1 or r > 256:
            raise ValueError('k must be in [1, 256] (got %d)' % r)
    lists = {name: v for name, v in (('random_state', random_state), ('W_in', W_in), ('T_in', T_in)) if v is not None}
    if not lists and not rank_list:
        raise ValueError('nmf_models needs a list of random_state seeds and/or lists W_in, T_in (one entry per model)')
    lengths = {name: len(v) for name, v in lists.items()}
    if rank_list:
        lengths['k'] = len(ks)
    if len(set(lengths.values())) != 1:
        raise ValueError('random_state, W_in and T_in must have one entry per model (lengths %s)' % lengths)
    b = next(iter(lengths.values()))
    if b < 1:
        raise ValueError('nmf_models needs at least one model')
    if not rank_list:
        ks = ks * b
    if rank_list:                           # (each start must have its model's rank)
        for m in range(b):
            if W_in is not None and not _is_empty(W_in[m]) and tuple(np.shape(W_in[m])) != (X.shape[0], ks[m]):
                raise ValueError('W_in[%d] must be n x k[%d] = %d x %d' % (m, m, X.shape[0], ks[m]))
            if T_in is not None and not _is_empty(T_in[m]) and tuple(np.shape(T_in[m])) != (ks[m], X.shape[1]):
                raise ValueError('T_in[%d] must be k[%d] x d = %d x %d' % (m, m, ks[m], X.shape[1]))
    seeds = list(random_state) if random_state is not None else [None] * b
    W_ins = list(W_in) if W_in is not None else [[]] * b
    T_ins = list(T_in) if T_in is not None else [[]] * b
    n, d = X.shape
    # ---- argument policy of nmf() (nmf.py:280-315)
    project_T = a['project_T_each_iter']
    if project_T and np.any([a['reg_w_l1'], a['reg_t_l1']]):
        logger.warning('This implementation can not solve project_T_each_iter=True with regularization. '
                       'Setting project_T_each_iter to False.')
        project_T = False
    if (not project_T and not a['t_row_sum']) and (a['reg_t_l1'] < 0 or a['reg_t_l2'] < 0):
        logger.error('Unbounded objective. reg_t_l1=%s, reg_t_l2=%s', a['reg_t_l1'], a['reg_t_l2'])
        return [{'W': np.ones((n, r)), 'T': np.ones((r, d)) * 1e6, 'obj_history': [-np.inf], 'iter_cputime': [0]}
                for r in ks]
    if (not a['project_W_each_iter'] and not a['w_row_sum']) and (a['reg_w_l1'] < 0 or a['reg_w_l2'] < 0):
        logger.error('Unbounded objective. reg_w_l1=%s, reg_w_l2=%s', a['reg_w_l1'], a['reg_w_l2'])
        return [{'W': np.ones((n, r)) * 1e6, 'T': np.ones((r, d)), 'obj_history': [-np.inf], 'iter_cputime': [0]}
                for r in ks]
    seeds = [int(time.time()) % 4294967296 if s is None else s for s in seeds]
    t_global_start = time.time()
    max_time = a['max_time'] - 10                                 # nmf.py:333
    inits = ['random' if n <= r else a['init'] for r in ks]       # nmf.py:346-347
    start_time = time.process_time()
    device = a['device']
    if device is None:
        device = X.device if isinstance(X, torch.Tensor) and X.is_cuda else torch.device('cuda')
    device = torch.device(device)
    if not torch.cuda.is_available():
        raise _lib.RriError('no CUDA device is available: rri_nmf_b200.nmf_models has no CPU fallback')
    if device.type != 'cuda':
        raise _lib.RriError('rri_nmf_b200.nmf_models runs on CUDA devices only (no CPU fallback)')
    if device.index is None:
        device = torch.device('cuda', torch.cuda.current_device())
    if isinstance(X, torch.Tensor):
        dtype = X.dtype if X.dtype in (torch.float32, torch.float64) else torch.float64
    else:
        dtype = torch.float32 if np.asarray(X).dtype == np.float32 else torch.float64
    numpy_io = not isinstance(X, torch.Tensor)
    w_row_sum, t_row_sum = a['w_row_sum'], a['t_row_sum']
    on_device = [_init_on_device_rule(X, n, d, W_ins[m], T_ins[m], a['init_on_device'], None) for m in range(b)]
    starts = [_host_start(X, None, ks[m], inits[m], seeds[m], t_row_sum, w_row_sum, W_ins[m], T_ins[m], on_device[m])
              for m in range(b)]
    if rank_list:
        groups = _rank_groups(ks)
    else:
        sizes = _model_groups(b, ks[0])
        groups = [list(range(sum(sizes[:i]), sum(sizes[:i + 1]))) for i in range(len(sizes))]
    results = [None] * b
    with torch.cuda.device(device):
        Xd = _to_device(X, device, dtype)
        for idx in groups:
            if rank_list:
                engine = RRIEngine(Xd, [ks[m] for m in idx], order='hals', math=a['math'])
            else:
                engine = RRIEngine(Xd, ks[0], order='hals', math=a['math'], models=len(idx))
            try:
                out = _solve_models(engine, idx, starts, on_device, seeds, inits, a, start_time, t_global_start,
                                    max_time, numpy_io)
            finally:
                engine.close()
            for m, r in zip(idx, out):
                results[m] = r
    return results


def _solve_models(engine, idx, starts, on_device, seeds, inits, a, start_time, t_global_start, max_time, numpy_io):
    """The sweep loop of _solve for the models `idx` of one models engine (equal ranks, or a ranks engine), each
    stopping on its own.  Wbuf, Tbuf are the engine's buffers; W[j], T[j] below are model j's views of them."""
    g = len(idx)
    w_row_sum, t_row_sum = a['w_row_sum'], a['t_row_sum']
    regs = dict(reg_w_l1=a['reg_w_l1'], reg_w_l2=a['reg_w_l2'], reg_t_l1=a['reg_t_l1'], reg_t_l2=a['reg_t_l2'])
    if engine.ranks is not None:
        Wbuf = torch.empty((engine.n * engine.k,), dtype=engine.dtype, device=engine.device)
        Tbuf = torch.empty((engine.k, engine.d), dtype=engine.dtype, device=engine.device)
        W, T = engine.views(Wbuf, Tbuf)
        ranks = engine.ranks
    else:
        Wbuf = torch.empty((g, engine.n, engine.k), dtype=engine.dtype, device=engine.device)
        Tbuf = torch.empty((g, engine.k, engine.d), dtype=engine.dtype, device=engine.device)
        W, T = list(Wbuf), list(Tbuf)
        ranks = [engine.k] * g
    for j, m in enumerate(idx):
        Wj, Tj = _device_start(engine, engine.X, None, None, ranks[j], inits[m], seeds[m], t_row_sum, w_row_sum,
                               starts[m][0], starts[m][1], on_device[m], {})
        W[j].copy_(Wj)
        T[j].copy_(Tj)
        del Wj, Tj
    project_W = a['project_W_each_iter'] and w_row_sum is not None
    if project_W:                                                                 # nmf.py:870-873
        for j in range(g):
            engine.project_rows_simplex(W[j], w_row_sum)
    params = engine.params(ub_w=w_row_sum, ub_t=t_row_sum, **regs)
    obj_mode = a['objective']
    via_contraction = obj_mode == 'contraction' or (obj_mode == 'auto' and engine.math == 'ieee')
    compute_obj = a['compute_obj_each_iter']
    unapplied_reset = a['reset_topic_method']
    chunk = 1 if (compute_obj or project_W) else max(1, int(a['sweeps_per_call']))
    active = [True] * g
    final = [None] * g                      # (W, T) of a model that stopped before the others
    errors = [None] * g
    hist = [[] for _ in range(g)]
    cpu = [[] for _ in range(g)]
    iter_no, max_iter = 0, a['max_iter']
    while iter_no < max_iter and any(active):
        ns = min(chunk, max_iter - iter_no)
        flags = engine.sweeps(Wbuf, Tbuf, ns, params, want_flags=True)
        sums = []

        def topic_sums(j):
            if not sums:
                sums.extend(engine.topic_sums())
            return sums[0][j], sums[1][j]
        for j in range(g):
            if not active[j]:
                if flags[j] & (_lib.FLAG_UNBOUNDED | _lib.FLAG_NONFINITE):
                    W[j].zero_()            # (a model that already stopped: its result was taken when it stopped)
                    T[j].zero_()
                continue
            exc = _flags_error(flags[j], lambda: topic_sums(j), unapplied_reset)
            if exc is not None:
                # only this model fails; zero factors keep it out of the shared operand's scale from here on
                errors[j] = exc
                active[j] = False
                W[j].zero_()
                T[j].zero_()
        iter_no += ns
        if project_W:                                                             # nmf.py:481-484
            for j in range(g):
                if active[j]:
                    engine.project_rows_simplex(W[j], w_row_sum)
        if compute_obj:                                                           # nmf.py:488-489
            objs = engine.objective(Wbuf, Tbuf, via_contraction=via_contraction, reuse_last_sweep=not project_W, **regs)
        now = time.process_time()
        for j in range(g):
            if active[j]:
                if compute_obj:
                    hist[j].append(objs[j])
                cpu[j].extend([now] * ns)
        if time.time() - t_global_start >= max_time:                             # nmf.py:506-508
            break
        if compute_obj:
            for j in range(g):
                if active[j] and _universal_stopping_condition(hist[j], a['eps_stop']):     # :510-514
                    final[j] = (W[j].clone(), T[j].clone())
                    active[j] = False
    out = []
    for j, m in enumerate(idx):
        if errors[j] is not None:
            out.append({'error': errors[j], 'random_state': seeds[m]})
            continue
        Wj, Tj = final[j] if final[j] is not None else (W[j].clone(), T[j].clone())
        if not project_W and w_row_sum is not None and a['do_final_project_W']:   # nmf.py:519-529
            engine.project_rows_simplex(Wj, w_row_sum)
        torch.cuda.current_stream(Wj.device).synchronize()
        r = {'W': Wj.cpu().numpy() if numpy_io else Wj, 'T': Tj.cpu().numpy() if numpy_io else Tj}
        if compute_obj:
            r['obj_history'] = hist[j]
        r['iter_cputime'] = [x - start_time for x in cpu[j]]
        r['random_state'] = seeds[m]
        out.append(r)
    return out


def _init_on_device_rule(X, n, d, W_in, T_in, init_on_device, comm):
    """Whether the NNDSVD initialisation runs on the device (see `init_on_device` in the module docstring)."""
    need_init = _is_empty(W_in) or _is_empty(T_in)
    if init_on_device is None:
        init_on_device = (isinstance(X, torch.Tensor) and X.is_cuda) or n * d >= (1 << 26)
    return bool(init_on_device) and need_init and comm is None


def _host_start(X, W_mat, k, init, random_state, t_row_sum, w_row_sum, W_in, T_in, init_on_device):
    """(W0, T0) of nmf.py:819-868 as far as the host makes them: the host NNDSVD (unless it runs on the device) and the
    caller's W_in / T_in after their shape check.  A factor left to the device initialisation is None."""
    n, d = X.shape
    need_init = _is_empty(W_in) or _is_empty(T_in)
    W0 = T0 = None
    if need_init and not init_on_device:
        if _is_sparse(X):
            # M o X is the sparse matrix itself (entry weights folded in): the SVD never densifies it
            if isinstance(X, torch.Tensor):
                Xc = X.detach().to_sparse_csr().cpu()
                Xh = sp.csr_matrix((Xc.values().numpy(), Xc.col_indices().numpy(), Xc.crow_indices().numpy()),
                                   shape=(n, d))
                if W_mat is not None:
                    Xh.data = Xh.data * W_mat.detach().cpu().numpy()
            else:
                Xh = X.tocsr()
                if W_mat is not None:
                    Xh = Xh.multiply(W_mat).tocsr()
            Mh = None
        else:
            Xh = X.detach().cpu().numpy() if isinstance(X, torch.Tensor) else np.asarray(X)
            Mh = None
            if W_mat is not None:
                Mh = W_mat.detach().cpu().numpy() if isinstance(W_mat, torch.Tensor) else np.asarray(W_mat)
        W0, T0 = initialize_nmf(Mh * Xh if Mh is not None else Xh, k, init, random_state=random_state,
                                row_normalize=False)
        if t_row_sum is not None:
            T0 = normalize(T0) * t_row_sum
        if w_row_sum is not None:
            W0 = normalize(W0) * w_row_sum
    if not _is_empty(W_in):
        if tuple(np.shape(W_in)) != (n, k):
            raise ValueError('W_in has wrong dimensions, must be n*k')
        W0 = W_in
    if not _is_empty(T_in):
        if tuple(np.shape(T_in)) != (k, d):
            raise ValueError('T_in has wrong dimensions, must be k*d')
        T0 = T_in
    return W0, T0


def _device_start(engine, Xd, W_mat, Md, k, init, random_state, t_row_sum, w_row_sum, W0, T0, init_on_device,
                  timing):
    """The device factors nmf() starts from: the device NNDSVD where `init_on_device` says so (its passes over X go
    through the engine's own contraction kernel), then W0 / T0 clipped at 0 in fresh device tensors."""
    device, dtype = engine.device, engine.dtype
    if init_on_device:
        _ti = time.perf_counter()
        sparse_in = Xd.layout == torch.sparse_csr
        Wi, Ti = _initialize_on_device(Xd, W_mat, k, init, random_state, t_row_sum, w_row_sum,
                                       products=engine.products() if (Md is None or sparse_in) else None)
        torch.cuda.current_stream(device).synchronize()
        timing['init_on_device_s'] = timing.get('init_on_device_s', 0.0) + time.perf_counter() - _ti
        W0 = Wi if W0 is None else W0
        T0 = Ti if T0 is None else T0
    # np.maximum(W_in, 0) makes copies: the caller's arrays are never mutated (nmf.py:867-868)
    W = _to_device(W0, device, dtype).clamp(min=0).contiguous()
    T = _to_device(T0, device, dtype).clamp(min=0).contiguous()
    if W.data_ptr() == (W0.data_ptr() if isinstance(W0, torch.Tensor) else 0):
        W = W.clone()
    if T.data_ptr() == (T0.data_ptr() if isinstance(T0, torch.Tensor) else 0):
        T = T.clone()
    return W, T


def _solve(engine, Xd, W, T, rtv, a):
    """Sweep loop and post-processing: nmf.py:351-560."""
    k, n, d = a['k'], a['n'], a['d']
    fix_T = a['fix_T']
    w_row_sum, t_row_sum = a['w_row_sum'], a['t_row_sum']
    project_T_each_iter, project_W_each_iter = a['project_T_each_iter'], a['project_W_each_iter']
    early_stop, diagnostics = a['early_stop'], a['diagnostics']
    compute_obj_each_iter, eps_stop = a['compute_obj_each_iter'], a['eps_stop']
    reset_topic_method = a['reset_topic_method']
    max_iter, max_time, t_global_start = a['max_iter'], a['max_time'], a['t_global_start']
    numpy_io = a['numpy_io']
    regs = dict(reg_w_l1=a['reg_w_l1'], reg_w_l2=a['reg_w_l2'], reg_t_l1=a['reg_t_l1'], reg_t_l2=a['reg_t_l2'])

    if project_W_each_iter and not a['fix_W'] and w_row_sum is not None:          # nmf.py:870-873
        engine.project_rows_simplex(W, w_row_sum)
    if project_T_each_iter and not fix_T and t_row_sum is not None:               # nmf.py:875-878
        engine.project_rows_simplex(T, t_row_sum)

    params = engine.params(ub_w=w_row_sum, ub_t=t_row_sum, fix_T=fix_T,
                           simplex_T=bool(project_T_each_iter and t_row_sum and not fix_T),
                           sp_refresh_every=a['sparse_refresh_every'], **regs)
    masked = engine.masked

    def host_view(t):
        return t.detach().cpu().numpy() if numpy_io else t

    # User callbacks (early_stop, diagnostics) get what the reference gives them: arrays of the kind X was.  A callback
    # carrying the attribute `device_tensors = True` (the recommender estimator's validation RMSE) is handed the
    # device-resident X, W, T instead -- nothing returns to the host between sweeps (SURVEY.md §8 f2).
    cbs = ([early_stop] if callable(early_stop) else []) + list(diagnostics)
    need_host = any(not getattr(f, 'device_tensors', False) for f in cbs)
    Xcb = None
    if cbs and need_host:
        Xcb = Xd if a['sparse_in'] else host_view(Xd)          # sparse input is handed to callbacks as given

    def call_cb(f):
        if getattr(f, 'device_tensors', False):
            return f(Xd, W, T)
        return f(Xcb, host_view(W), host_view(T))

    state = {'n_resets_remaining': a['n_resets']}
    iter_cputime = []
    obj_history = []
    obj_mode = a['objective']
    if obj_mode not in ('auto', 'exact', 'contraction'):
        raise ValueError("objective must be 'auto', 'exact' or 'contraction'")
    can_contract = engine.order == 'hals' and not masked and not fix_T
    if obj_mode == 'contraction' and not can_contract:
        raise ValueError("objective='contraction' needs unmasked dense data and update_order='hals'")
    via_contraction = can_contract and (obj_mode == 'contraction' or (obj_mode == 'auto' and engine.math == 'ieee'))
    OBJ = DeviceObjective(engine, W, T, regs, via_contraction) if compute_obj_each_iter else None
    if early_stop:
        last_score = np.inf
        W_prev, T_prev = W.clone(), T.clone()
    for f in diagnostics:
        rtv['diagnostics'][f.__name__].append(call_cb(f))

    # sweeps can be batched into one library call when nothing on the host has to look at the state
    # in between (N sweeps in one call == N calls of one sweep, bit for bit)
    comm = a['comm']
    sharded = comm is not None and getattr(comm, 'world', 1) > 1
    can_reset = reset_topic_method is not None and engine.order == 'rri' and not masked and not fix_T \
        and not a['fix_W'] and not sharded
    if reset_topic_method is not None and not can_reset and not fix_T and not a['fix_W']:
        # the reference re-seeds an emptied topic (nmf.py:762-816); here that policy exists for the unmasked,
        # unsharded interleaved order only.  Say so up front; an emptied topic then raises (see _raise_on_flags).
        logger.info("reset_topic_method=%r is only applied with update_order='rri' on unmasked, unsharded data; "
                    "on this engine an emptied topic raises instead of being re-seeded", reset_topic_method)
    per_sweep_host = bool(early_stop) or compute_obj_each_iter or bool(diagnostics) or \
        (project_W_each_iter and w_row_sum is not None) or can_reset
    chunk = 1 if per_sweep_host else max(1, int(a['sweeps_per_call']))

    iter_no = 0
    while iter_no < max_iter:
        if early_stop:                                                             # nmf.py:381-407
            if callable(early_stop):
                # row shards: every rank scores its own rows; the decision uses the mean over ranks so that all
                # ranks revert and leave together
                this_score = _all_mean(comm, call_cb(early_stop))
            else:
                this_score = obj_history[-1] if (compute_obj_each_iter and obj_history) else np.inf
            if this_score > last_score:
                W.copy_(W_prev)
                T.copy_(T_prev)
                obj_history = obj_history[:-1]
                iter_cputime = iter_cputime[:-1]
                for f in diagnostics:
                    rtv['diagnostics'][f.__name__] = rtv['diagnostics'][f.__name__][:-1]
                break
            last_score = this_score
            W_prev.copy_(W)
            T_prev.copy_(T)
        ns = min(chunk, max_iter - iter_no)
        if can_reset:
            W_save, T_save = W.clone(), T.clone()
        if a['fix_W']:
            ns = 1
            flags = 0 if fix_T else _sweep_fix_W(engine, W, T, a)
        else:
            flags = engine.sweeps(W, T, ns, params, want_flags=True)
        if flags & (_lib.FLAG_ZERO_T | _lib.FLAG_ZERO_W) and can_reset and state['n_resets_remaining'] > 0:
            # rare path: redo this sweep topic by topic with the reset policy of nmf.py:762-783, :796-816
            W.copy_(W_save)
            T.copy_(T_save)
            flags = _sweep_with_resets(engine, Xd, W, T, params, a, state)
        if fix_T and reset_topic_method is not None:
            # transform(): the reference would re-seed topic t (T row included!) when no new document uses it
            # (nmf.py:796-816 runs under fix_T as well).  Here T is left alone and the column stays zero.
            flags &= ~_lib.FLAG_ZERO_W
        if flags & _lib.FLAG_NOT_IMPLEMENTED:
            # block order with project_T_each_iter: a T denominator <= 0 and t_row_sum != 1 (optimization.py:60-74)
            raise NotImplementedError('s={} is not yet implemented'.format(t_row_sum))
        _raise_on_flags(flags, engine, reset_topic_method if not (can_reset or fix_T) else None)
        iter_no += ns
        if project_W_each_iter and not a['fix_W'] and w_row_sum is not None:      # nmf.py:481-484
            engine.project_rows_simplex(W, w_row_sum)
        if compute_obj_each_iter:                                                  # nmf.py:488-489
            # (the sweep's own contraction is still valid unless W was projected after it)
            OBJ._after_sweep = not (project_W_each_iter and w_row_sum is not None) and not a['fix_W']
            obj_history.append(OBJ.true_objective())
        now = time.process_time()
        iter_cputime.extend([now] * ns)
        for f in diagnostics:                                                      # nmf.py:495-500
            rtv['diagnostics'][f.__name__].append(call_cb(f))
        # stop decisions are collective on row shards (a rank that left alone would hang the others' exchange)
        if _all_any(comm, time.time() - t_global_start >= max_time):              # nmf.py:506-508
            break
        if compute_obj_each_iter and _universal_stopping_condition(obj_history, eps_stop):   # :510-514
            break                       # (the objective is all-reduced: the same number on every rank)
    iter_cputime = [x - a['start_time'] for x in iter_cputime]

    if (not project_W_each_iter and w_row_sum is not None and not a['fix_W'] and a['do_final_project_W']):
        engine.project_rows_simplex(W, w_row_sum)                                  # nmf.py:519-529

    torch.cuda.current_stream(W.device).synchronize()
    rtv['W'] = host_view(W)
    rtv['T'] = host_view(T)
    if compute_obj_each_iter:
        rtv['obj_history'] = obj_history
        rtv['obj_calculator'] = OBJ
    rtv['iter_cputime'] = iter_cputime
    rtv['random_state'] = a['random_state']
    return rtv


def _qf_min_device(numer, denom, s, ub, engine):
    """qf_min(-numer, denom, s=s, ub=ub) of optimization.py:12-88 on device vectors: returns (x, nx) with
    nx = sum(x) before the projection / rescaling to sum s.  denom with one element = the scalar-c branches
    (:51-74), otherwise the vector-c branch (:75-87)."""
    d = numer.numel()
    eps = eps_div_by_zero
    if s:                                                         # :43-49
        if ub:
            ub = min(ub, s)
            assert d * ub >= s
        else:
            ub = s
    if denom.numel() == 1:
        c = float(denom)
        if c > 0:                                                 # :53-59 (ub is ignored on this branch)
            x = numer.clamp(min=0) / (c + eps)
            nx = float(x.sum())
            if s is not None:
                x = engine.project_rows_simplex(x.reshape(1, -1).contiguous(), s).reshape(-1)
            return x, nx
        x = torch.zeros_like(numer)                               # :60-74
        if s is None:
            if not ub:
                raise ValueError('Minimum objective is unbounded.')
            x[(c - numer) < 0] = ub
        elif s == 1.0:
            x[int(torch.argmax(numer))] = 1.0
        else:
            raise NotImplementedError('s={} is not yet implemented'.format(s))
        return x, 1.0
    if bool((denom < 0).any()) and (s is None and ub is None):    # :76-77
        raise ValueError('Minimum objective is unbounded.')
    x = torch.where(denom > 0, numer.clamp(min=0) / (denom + eps), torch.zeros_like(numer))
    if ub is not None:
        x = x.clamp(max=ub)
    nx = float(x.sum())
    if s is not None:
        x = s * x / x.sum()
    return x, nx


def _sweep_fix_W(engine, W, T, a):
    """One T-only sweep in the reference's order (nmf.py:415-458 with fix_W=True): for every topic the shard
    statistic of rri_partials_T, the qf_min solve, and -- when no regulariser is set -- the rescaling
    W[:, t] *= nt1 of nmf.py:450-452 that keeps W T invariant under the row normalisation of T."""
    t_row_sum = a['t_row_sum']
    s = t_row_sum if a['project_T_each_iter'] else None           # nmf.py:442-445
    noreg = (abs(a['reg_w_l1']) + abs(a['reg_w_l2']) + abs(a['reg_t_l1']) + abs(a['reg_t_l2'])) == 0
    for t in range(a['k']):
        wR, nw = engine.partials_T(W, T, t)
        x, nt1 = _qf_min_device(wR - a['reg_t_l1'], nw + a['reg_t_l2'], s, t_row_sum, engine)
        T[t, :] = x
        if noreg:
            W[:, t] *= nt1
        if t_row_sum and a['project_T_each_iter'] and abs(float(T[t, :].sum()) - t_row_sum) > 1e-15:
            engine.project_rows_simplex(T[t:t + 1, :], t_row_sum)               # nmf.py:759-761
    return 0


def _raise_on_flags(flags, engine, unapplied_reset=None):
    exc = _flags_error(flags, engine.topic_sums, unapplied_reset)
    if exc is not None:
        raise exc


def _flags_error(flags, topic_sums, unapplied_reset=None):
    """The exception a sweep's flags word stands for (None: carry on); topic_sums() -> (sum_T[k], sum_W[k])"""
    if unapplied_reset is not None and flags & (_lib.FLAG_ZERO_T | _lib.FLAG_ZERO_W):
        sT, sW = topic_sums()
        if np.any(sT <= 1e-10) or np.any(sW <= 1e-10):
            return ValueError("a topic emptied (sum <= 1e-10) and reset_topic_method=%r is not applied on this engine "
                              "(resets exist for update_order='rri' on unmasked, unsharded data; nmf.py:762-816): "
                              "use that mode, other initial factors, or reset_topic_method=None" % (unapplied_reset,))
    if flags & _lib.FLAG_UNBOUNDED:
        # optimization.py:60-67 / :76-77 -> _unbounded_objective (:105-107)
        return ValueError('Minimum objective is unbounded. (a denominator became <= 0 with no upper bound; '
                          'typically a topic collapsed to zero while reset_topic_method is None)')
    if flags & _lib.FLAG_NONFINITE:
        return FloatingPointError('non-finite values produced in the sweep')
    if flags & _lib.FLAG_ZERO_W:
        if np.any(topic_sums()[1] <= 0):
            return AssertionError('W[:, t] sums to 0')                              # nmf.py:476
    return None


def _sweep_with_resets(engine, Xd, W, T, params, a, state):
    """One rri-order sweep executed topic by topic so that an emptied topic can be re-seeded exactly
    where the reference does it (nmf.py:458 -> :762-783 after the T-step, :471 -> :796-816 after the
    W-step).  The device runs the topic; the reset itself (a full residual, rare) uses torch ops."""
    k = engine.k
    flags_all = 0
    method = a['reset_topic_method']

    def reset(t):
        state['n_resets_remaining'] -= 1
        if method == 'max_resid_document':
            if engine.sparse:
                mi, cols, vals = max_resid_document_sparse(engine.crow, engine.col, engine.val, W, T)
                T[t, :] = 0
                T[t, cols] = vals
            else:
                R = (Xd - W @ T).clamp_(min=0)
                mi = int(torch.argmax((R ** 2).sum(1)))
                T[t, :] = R[mi, :]
            W[:, t] = 0
            W[mi, t] = 1.0
        elif method == 'random':
            if a['fix_reset_seed']:
                np.random.seed(t + int(torch.argmax(T[t, :])))
            r = np.random.rand(1, engine.d)
            T[t, :] = torch.from_numpy(r / r.sum()).to(T).reshape(-1)
            W[:, t] = torch.from_numpy(np.random.rand(engine.n)).to(W)
        else:
            raise ValueError('unknown reset_topic_method %r' % (method,))

    for t in range(k):
        W_save, T_save = W.clone(), T.clone()
        f = engine.topics(W, T, t, t + 1, params)
        sT, sW = engine.topic_sums()
        if sT[t] <= 1e-10 and state['n_resets_remaining'] > 0:
            # the T row came out empty: keep only the T-step of this attempt, re-seed the topic, then run the
            # W-step on the re-seeded row (the first attempt's W-step saw a zero denominator: drop its flags)
            W.copy_(W_save)
            T_new_row = T[t, :].clone()
            T.copy_(T_save)
            T[t, :] = T_new_row
            reset(t)
            _w_step_only(engine, W, T, t, params)
            f = 0
            sW_t = float(W[:, t].sum())
        else:
            sW_t = sW[t]
        if sW_t <= 1e-10 and state['n_resets_remaining'] > 0:
            reset(t)                                      # nmf.py:796-816
            f &= ~_lib.FLAG_ZERO_W
        flags_all |= f
    return flags_all


def max_resid_document_sparse(crow, col, val, W, T, chunk_entries=None):
    """(i, columns, values) for zero-filled sparse X given as CSR (crow, col, val): i is the first row of
    max(X - W T, 0) with the largest sum of squares (the reference's 'max_resid_document', nmf.py:766-770), columns and
    values are that row's stored entries of the clamped residual.  With W, T >= 0 every unstored entry of
    max(X - W T, 0) is max(-W[i] . T[:, j], 0) = 0, so the sums run over the stored entries only, in chunks of
    entries: no n x d array is formed."""
    nnz = int(val.numel())
    step = chunk_entries or max(1, (1 << 22) // max(int(W.shape[1]), 1))
    col = col.to(torch.int64)
    r = torch.empty(nnz, dtype=W.dtype, device=W.device)
    for a in range(0, nnz, step):
        b = min(a + step, nnz)
        rows = torch.searchsorted(crow, torch.arange(a, b, device=crow.device), right=True) - 1
        pred = (W[rows] * T[:, col[a:b]].t()).sum(1)
        r[a:b] = (val[a:b].to(W.dtype) - pred).clamp_(min=0)
    # (one fixed summation order per row)
    ss = torch.segment_reduce(r * r, 'sum', lengths=crow.diff(), unsafe=True)
    mi = int(torch.argmax(ss))
    lo, hi = int(crow[mi]), int(crow[mi + 1])
    return mi, col[lo:hi], r[lo:hi]


def _w_step_only(engine, W, T, t, params):
    """W-step of topic t alone (nmf.py:462-469 with the current T), used only on the rare reset path right after
    a topic was re-seeded; plain torch ops on the device tensors (X T_t' of sparse data through rri_spmm)."""
    Tt = T[t, :]
    h = T @ Tt
    nt = float(h[t])
    h[t] = 0
    xt = engine.products().right(Tt.reshape(-1, 1))[:, 0] if engine.sparse else engine.X @ Tt
    numer = xt - W @ h - params.reg_w_l1
    denom = nt + params.reg_w_l2
    if denom > 0:
        W[:, t] = numer.clamp(min=0) / (denom + params.eps)
    else:
        W[:, t] = 0
