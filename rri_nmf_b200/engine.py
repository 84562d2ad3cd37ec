"""RRIEngine -- thin object wrapper of the C-ABI handle (include/rri_b200.h) over torch-owned device
memory.  PyTorch is plumbing only here (allocation, streams, torch.distributed bootstrap): every
kernel on the sweep path is launched by librri_b200.so."""
import ctypes as C
import os

import numpy as np
import torch

from . import _lib
from ._lib import RriParams, check

EPS_DIV_BY_ZERO = float(np.spacing(10))     # reference nmf.py:52 / optimization.py:5


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


class NcclComm(object):
    """An ncclComm_t created by the engine library from an id broadcast over torch.distributed."""

    def __init__(self, device_index, group=None):
        import torch.distributed as dist
        self.rank = dist.get_rank(group)
        self.world = dist.get_world_size(group)
        self.lib = _lib.load()
        self.nccl_path = _lib.nccl_library_path()
        path = self.nccl_path.encode() if self.nccl_path else None
        idbuf = (C.c_char * 128)()
        if self.rank == 0:
            check(self.lib.rri_nccl_unique_id(idbuf, path))
        # broadcast the 128-byte id with whatever backend the group has
        backend = dist.get_backend(group)
        dev = torch.device('cuda', device_index) if backend == 'nccl' else torch.device('cpu')
        t = torch.tensor(list(bytes(idbuf)), dtype=torch.uint8, device=dev)
        dist.broadcast(t, src=0, group=group)
        raw = bytes(t.cpu().tolist())
        idbuf2 = (C.c_char * 128).from_buffer_copy(raw)
        self.comm = C.c_void_p()
        check(self.lib.rri_nccl_comm_create(C.byref(self.comm), idbuf2, self.rank, self.world,
                                            device_index, path))

    def destroy(self):
        if self.comm:
            self.lib.rri_nccl_comm_destroy(self.comm)
            self.comm = C.c_void_p()


class RRIEngine(object):
    """One sweep engine per GPU / row shard.

    X: torch tensor [n_local, d] on a CUDA device, float32 or float64, row-major (a row stride >= d
    is allowed).  W_mat: optional weights, same shape (same dtype, or uint8 0/1 mask).
    X may also be a torch sparse CSR tensor (never densified).  unstored='missing' (default): its stored entries are
    the observed ones (the recommender setting); W_mat is then an optional 1-D tensor of nnz entry weights.
    unstored='zero': X is an ordinary non-negative matrix stored sparsely (a tf-idf document-term matrix), every entry
    is fitted, the unstored ones as 0 (rri_bind_csr_zero: math='ieee', no W_mat; order='hals' contracts X T' / X' W,
    order='rri' makes one pass over the rows and the columns per topic).
    order: 'rri' (reference-exact interleaved order, nmf.py:415-476) or 'hals' (block order).
    math : 'ieee' or 'tf32' (tcgen05 tensor-core contraction; float32 + hals only).
    """

    def __init__(self, X, k, W_mat=None, order='rri', math='ieee', comm=None, unstored='missing'):
        if not isinstance(X, torch.Tensor) or not X.is_cuda:
            raise _lib.RriError('RRIEngine needs X resident on a CUDA device (no CPU fallback)')
        if X.dim() != 2:
            raise ValueError('X must be 2-D')
        if X.dtype not in (torch.float32, torch.float64):
            raise ValueError('X must be float32 or float64')
        self.sparse = X.layout == torch.sparse_csr
        if not self.sparse and X.layout != torch.strided:
            raise ValueError('X must be a dense (strided) or a sparse CSR tensor')
        if unstored not in ('missing', 'zero'):
            raise ValueError("unstored must be 'missing' or 'zero'")
        if unstored == 'zero' and self.sparse:
            if math != 'ieee':
                raise ValueError("zero-filled sparse X runs with math='ieee' (the sparse contraction is not compute-bound)")
            if W_mat is not None:
                raise ValueError('zero-filled sparse X takes no W_mat (weights on every entry would be a dense n x d object)')
        self.unstored = unstored if self.sparse else 'missing'
        if not self.sparse and X.stride(1) != 1:
            X = X.contiguous()
        self.lib = _lib.load()
        self.X = X
        self.n, self.d = int(X.shape[0]), int(X.shape[1])
        self.k = int(k)
        self.dtype = X.dtype
        self.device = X.device
        self.order = order
        self.math = math
        self.comm = comm
        self.W_mat = None
        self.Xt = None
        self.peer_exchange = False
        self.h = C.c_void_p()
        dev_index = self.device.index if self.device.index is not None else torch.cuda.current_device()
        self.dev_index = dev_index
        check(self.lib.rri_create(C.byref(self.h), self.n, self.d, self.k,
                                  _lib.RRI_F32 if self.dtype == torch.float32 else _lib.RRI_F64,
                                  {'ieee': _lib.RRI_MATH_IEEE, 'tf32': _lib.RRI_MATH_TF32}[math],
                                  {'rri': _lib.RRI_ORDER_RRI, 'hals': _lib.RRI_ORDER_HALS}[order],
                                  dev_index))
        if comm is not None and comm.world > 1:
            path = comm.nccl_path.encode() if comm.nccl_path else None
            check(self.lib.rri_set_comm(self.h, comm.comm, comm.rank, comm.world, path))
        if self.sparse:
            self._bind_csr(X, W_mat)
            return
        mk = _lib.RRI_MASK_NONE
        ldm = 0
        if W_mat is not None:
            if tuple(W_mat.shape) != (self.n, self.d):
                raise ValueError('W_mat must have the shape of X')
            if W_mat.dtype == torch.uint8 or W_mat.dtype == torch.bool:
                # byte masks are kept with a row stride that is a multiple of 16 bytes (a legal TMA row)
                ldp = (self.d + 15) // 16 * 16
                Mp = torch.zeros((self.n, ldp), dtype=torch.uint8, device=W_mat.device)
                Mp[:, :self.d] = W_mat.to(torch.uint8)
                W_mat = Mp[:, :self.d]
                mk = _lib.RRI_MASK_U8
            else:
                W_mat = W_mat.to(self.dtype).contiguous()
                mk = _lib.RRI_MASK_REAL
            self.W_mat = W_mat
            ldm = int(W_mat.stride(0))
        if order == 'hals' and self.W_mat is None:
            # the transposed copy of X lives in a torch tensor: allocation and release go through the caching
            # allocator instead of a cudaMalloc/cudaFree of a data-sized buffer per engine.  With math='tf32' the library
            # may keep 16-bit copies of X and X' there instead (rri_set_transpose_storage): the row stride leaves room
            # for them where n or d is not a multiple of 8
            v = 16 // X.element_size()
            ldxt = (self.n + v - 1) // v * v
            if math == 'tf32':
                b16 = 2 * (self.n * ((self.d + 7) // 8 * 8) + self.d * ((self.n + 7) // 8 * 8))
                ldxt = max(ldxt, (-(-b16 // (4 * self.d)) + v - 1) // v * v)
            self.Xt = torch.empty((self.d, ldxt), dtype=self.dtype, device=self.device)
            check(self.lib.rri_set_transpose_storage(self.h, _ptr(self.Xt), ldxt))
        check(self.lib.rri_bind(self.h, _ptr(self.X), int(self.X.stride(0)), _ptr(self.W_mat), mk, ldm,
                                self._stream()))
        if (comm is not None and comm.world > 1 and order == 'hals' and self.W_mat is None
                and os.environ.get('RRI_P2P', '1') != '0'):
            self._setup_peer_exchange(comm)

    def _bind_csr(self, X, weights):
        """Observed-entries binding (rri_bind_csr): X is a torch sparse CSR tensor whose stored entries are the
        observed ones; `weights` (optional) is a 1-D tensor of nnz entry weights in the order of X.values().
        With unstored='zero': the zero-filled binding (rri_bind_csr_zero)."""
        if self.math != 'ieee':
            raise ValueError("sparse (observed-entries) data runs with math='ieee'")
        self.crow = X.crow_indices().to(torch.int64).contiguous()
        self.col = X.col_indices().to(torch.int32).contiguous()
        self.val = X.values().contiguous()
        self.nnz = int(self.val.numel())
        if self.unstored == 'zero':
            self.entry_weights = None
            check(self.lib.rri_bind_csr_zero(self.h, self.nnz, _ptr(self.crow), _ptr(self.col), _ptr(self.val),
                                             self._stream()))
            return
        self.entry_weights = None
        if weights is not None:
            if weights.dim() != 1 or int(weights.numel()) != self.nnz:
                raise ValueError('with sparse X, W_mat is a 1-D tensor of nnz entry weights (the order of X.values())')
            self.entry_weights = weights.to(device=self.device, dtype=self.dtype).contiguous()
        check(self.lib.rri_bind_csr(self.h, self.nnz, _ptr(self.crow), _ptr(self.col), _ptr(self.val),
                                    _ptr(self.entry_weights), self._stream()))

    @staticmethod
    def csr_tensor(indptr, indices, data, shape, device, dtype=None):
        """torch sparse CSR tensor on `device` from host or device index/value arrays (the form RRIEngine takes for
        observed-entries data); the three components are moved one by one, the matrix is never densified."""
        def dev(a, dt):
            t = a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a))
            return t.to(device=device, dtype=dt)
        val = dev(data, dtype)
        return torch.sparse_csr_tensor(dev(indptr, torch.int64), dev(indices, torch.int64), val,
                                       size=tuple(int(x) for x in shape), check_invariants=False)

    @property
    def masked(self):
        """True when only a subset of the entries is fitted (dense W_mat or sparse observed entries)"""
        return (self.sparse and self.unstored == 'missing') or self.W_mat is not None

    def _setup_peer_exchange(self, comm):
        """Map every rank's exchange buffer (CUDA IPC over NVLink) so that the T half-step reads the shard
        statistics of all ranks in place; falls back to the NCCL all-reduce when the mapping is refused."""
        import torch.distributed as dist
        hbuf = (C.c_char * 64)()
        ok = self.lib.rri_peer_export(self.h, hbuf) == 0
        mine = bytes(hbuf) if ok else b''
        gathered = [None] * comm.world
        dist.all_gather_object(gathered, mine)
        if not all(len(g) == 64 for g in gathered):
            return
        rc = self.lib.rri_peer_import(self.h, b''.join(gathered), comm.rank, comm.world)
        flags = [None] * comm.world
        dist.all_gather_object(flags, rc == 0)
        if all(flags):
            check(self.lib.rri_peer_enable(self.h, 1))
            self.peer_exchange = True

    # ------------------------------------------------------------------------------------------
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def close(self):
        if getattr(self, 'h', None):
            if getattr(self, 'peer_exchange', False):
                # peers may still be reading this rank's exchange buffer: leave together
                # (unmap the peers' buffers between two barriers, so that no rank frees a buffer that is still
                # mapped or being read elsewhere)
                try:
                    import torch.distributed as dist
                    if dist.is_initialized():
                        torch.cuda.synchronize(self.device)
                        dist.barrier()
                        self.lib.rri_peer_close(self.h)
                        dist.barrier()
                except Exception:
                    pass
                self.peer_exchange = False
            self.lib.rri_destroy(self.h)
            self.h = C.c_void_p()
            self.Xt = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def params(reg_w_l1=0.0, reg_w_l2=0.0, reg_t_l1=0.0, reg_t_l2=0.0, ub_w=None, ub_t=None,
               fix_W=False, fix_T=False, simplex_T=False, eps=EPS_DIV_BY_ZERO, sp_refresh_every=1):
        p = RriParams()
        p.reg_w_l1, p.reg_w_l2, p.reg_t_l1, p.reg_t_l2 = float(reg_w_l1), float(reg_w_l2), float(reg_t_l1), float(reg_t_l2)
        p.ub_w = float(ub_w) if ub_w else 0.0
        p.ub_t = float(ub_t) if ub_t else 0.0
        p.eps = float(eps)
        p.fix_W, p.fix_T, p.simplex_T = int(bool(fix_W)), int(bool(fix_T)), int(bool(simplex_T))
        p.sp_refresh_every = int(sp_refresh_every)
        return p

    def _check_factors(self, W, T):
        if tuple(W.shape) != (self.n, self.k) or tuple(T.shape) != (self.k, self.d):
            raise ValueError('W must be n*k and T must be k*d')
        for a in (W, T):
            if a.dtype != self.dtype or a.device != self.device or not a.is_contiguous():
                raise ValueError('factors must be contiguous %s tensors on %s' % (self.dtype, self.device))

    def sweeps(self, W, T, n_sweeps, params, want_flags=True):
        """n_sweeps sweeps in place on W, T.  Returns the flags word (0 if want_flags is False)."""
        self._check_factors(W, T)
        flags = C.c_int32(0)
        check(self.lib.rri_sweeps(self.h, _ptr(W), _ptr(T), int(n_sweeps), C.byref(params),
                                  C.byref(flags) if want_flags else None, self._stream()))
        return int(flags.value)

    def topics(self, W, T, t_begin, t_end, params):
        self._check_factors(W, T)
        flags = C.c_int32(0)
        check(self.lib.rri_topics(self.h, _ptr(W), _ptr(T), int(t_begin), int(t_end), C.byref(params),
                                  C.byref(flags), self._stream()))
        return int(flags.value)

    def topic_sums(self):
        sT = (C.c_double * self.k)()
        sW = (C.c_double * self.k)()
        check(self.lib.rri_topic_sums(self.h, sT, sW, self._stream()))
        return np.array(sT[:]), np.array(sW[:])

    def objective_terms(self, W, T, via_contraction=False, reuse_last_sweep=False):
        """[0.5*sum M(X-WT)^2, sum M X^2, sum W^2, sum |W|, sum T^2, sum |T|]; the first four are
        all-reduced over the row shards when a communicator is attached.
        via_contraction (unmasked dense data): ||X||^2 - 2<X T', W> + <W'W, T T'> instead of an explicit pass over X;
        reuse_last_sweep: W, T are exactly what the last block-order `sweeps` call left (its contraction is reused)."""
        self._check_factors(W, T)
        out = (C.c_double * 6)()
        if via_contraction:
            check(self.lib.rri_objective_contraction(self.h, _ptr(W), _ptr(T), int(bool(reuse_last_sweep)), out,
                                                     self._stream()))
        else:
            check(self.lib.rri_objective(self.h, _ptr(W), _ptr(T), out, self._stream()))
        v = np.array(out[:])
        if self.comm is not None and self.comm.world > 1:
            import torch.distributed as dist
            t = torch.tensor(v[:4], dtype=torch.float64, device=self.device)
            dist.all_reduce(t)
            v[:4] = t.cpu().numpy()
        return v

    def objective(self, W, T, reg_w_l1=0.0, reg_w_l2=0.0, reg_t_l1=0.0, reg_t_l2=0.0, via_contraction=False,
                  reuse_last_sweep=False):
        """nmf.py:71-94"""
        v = self.objective_terms(W, T, via_contraction, reuse_last_sweep)
        return float(v[0] + 0.5 * reg_w_l2 * v[2] + 0.5 * reg_t_l2 * v[4] + reg_t_l1 * v[5] + reg_w_l1 * v[3])

    def rel_error(self, W, T):
        """||M^(1/2) o (X - WT)||_F / ||M^(1/2) o X||_F"""
        v = self.objective_terms(W, T)
        return float(np.sqrt(2.0 * v[0] / v[1]))

    def partials_T(self, W, T, t):
        """Shard statistic of nmf.py:680-686 / :706-713 for topic t: (wR[d], nw[1 or d])."""
        self._check_factors(W, T)
        wR = torch.empty(self.d, dtype=self.dtype, device=self.device)
        nw = torch.empty(self.d if self.masked else 1, dtype=self.dtype, device=self.device)
        check(self.lib.rri_partials_T(self.h, _ptr(W), _ptr(T), int(t), _ptr(wR), _ptr(nw), self._stream()))
        return wR, nw

    def project_rows_simplex(self, A, s=1.0):
        if A.dtype != self.dtype or not A.is_contiguous() or A.dim() != 2:
            raise ValueError('A must be a contiguous 2-D tensor of the engine dtype')
        check(self.lib.rri_project_rows_simplex(self.h, _ptr(A), int(A.shape[0]), int(A.shape[1]), float(s),
                                                self._stream()))
        return A

    def gemm_nt(self, A, B):
        """C = A @ B.T through the engine's contraction kernel (unit tests / roofline)."""
        M, K = A.shape
        N = B.shape[0]
        if A.stride(1) != 1 or B.stride(1) != 1 or B.shape[1] != K:
            raise ValueError('gemm_nt takes K-contiguous operands A[M,K], B[N,K]')
        Cm = torch.empty(M, N, dtype=A.dtype, device=A.device)
        check(self.lib.rri_gemm_nt(self.h, _ptr(A), int(A.stride(0)), _ptr(B), int(B.stride(0)), _ptr(Cm), N,
                                   M, N, K, self._stream()))
        return Cm

    def contract_x(self, B, transpose=False):
        """C = X @ B.T (transpose=False) or X.T @ B.T (True) through the operand copies the block-order sweeps read
        (rri_contract_x; dense unmasked hals engines).  B [N, K] with unit column stride, N <= k + 16."""
        K = self.n if transpose else self.d
        if B.dim() != 2 or int(B.shape[1]) != K or B.stride(1) != 1:
            raise ValueError('B must be [N, %d] with unit column stride' % K)
        N = int(B.shape[0])
        Cm = torch.empty((self.d if transpose else self.n), N, dtype=self.dtype, device=self.device)
        check(self.lib.rri_contract_x(self.h, int(bool(transpose)), _ptr(B), int(B.stride(0)), N, _ptr(Cm),
                                      self._stream()))
        return Cm

    def products(self):
        """The two streaming products of a randomized SVD of X through the engine's contraction kernel (used by the
        device-resident NNDSVD initialisation, SURVEY.md §8 f3): right(Q) = X @ Q, left(Q) = X' @ Q.  The transposed
        product needs the engine's K-contiguous copy of X' (block-order handles); without it that one product is
        a library GEMM.  On a sparse handle both products are rri_spmm (the zero-filled matrix of the stored entries,
        times the entry weights when given); Q is padded to a 16-byte row internally."""
        eng = self
        v = 16 // self.X.element_size()
        if self.sparse:
            def spmm(Q, transpose):
                rows_in, rows_out = (eng.n, eng.d) if transpose else (eng.d, eng.n)
                if Q.dim() != 2 or int(Q.shape[0]) != rows_in:
                    raise ValueError('the operand must have %d rows' % rows_in)
                r = int(Q.shape[1])
                ld = (r + v - 1) // v * v
                B = Q.to(device=eng.device, dtype=eng.dtype)
                if ld != r or not B.is_contiguous():
                    Bp = torch.zeros((rows_in, ld), dtype=eng.dtype, device=eng.device)
                    Bp[:, :r] = B
                    B = Bp
                Cm = torch.empty((rows_out, ld), dtype=eng.dtype, device=eng.device)
                check(eng.lib.rri_spmm(eng.h, int(transpose), _ptr(B), ld, _ptr(Cm), ld, ld, eng._stream()))
                return Cm[:, :r]

            class _S(object):
                def right(self, Q):
                    return spmm(Q, 0)

                def left(self, Q):
                    return spmm(Q, 1)
            return _S()

        def kmajor(Q):
            """Q' [r, K] with a 16-byte aligned row stride (a legal TMA operand)"""
            K, r = Q.shape
            ld = (K + v - 1) // v * v
            B = torch.zeros((r, ld), dtype=eng.dtype, device=eng.device)
            B[:, :K] = Q.t()
            return B[:, :K]

        aligned = self.X.stride(0) % v == 0 and self.X.data_ptr() % 16 == 0

        class _P(object):
            def right(self, Q):
                if not aligned or Q.shape[1] > 256:
                    return eng.X @ Q.to(eng.dtype)
                return eng.gemm_nt(eng.X, kmajor(Q))

            def left(self, Q):
                if eng.Xt is None or Q.shape[1] > 256:
                    return eng.X.t() @ Q.to(eng.dtype)
                return eng.contract_x(kmajor(Q), transpose=True)
        return _P()

    def profile_kernel(self, which, W, T, iters=5):
        """average launch duration (ms) of the dominant streaming kernel, timed with CUDA events on the
        launching stream: which in {'rri_pass', 'gemm_w', 'gemm_t'}; 't_half' / 'w_half' time a whole
        block-order half-step (they advance W, T and are collective on row shards)"""
        self._check_factors(W, T)
        ms = C.c_float(0)
        idx = {'rri_pass': 0, 'gemm_w': 1, 'gemm_t': 2, 't_half': 3, 'w_half': 4, 'masked_t': 5, 'masked_w': 6}[which]
        check(self.lib.rri_profile_kernel(self.h, idx, _ptr(W), _ptr(T), int(iters), C.byref(ms), self._stream()))
        return float(ms.value)

    def stats(self):
        a, b = C.c_int64(0), C.c_int64(0)
        check(self.lib.rri_stats(self.h, C.byref(a), C.byref(b)))
        bits = C.c_int32(0)
        check(self.lib.rri_x_operand_bits(self.h, C.byref(bits)))
        return {'kernel_launches': int(a.value), 'workspace_bytes': int(b.value), 'x_operand': 'f%d' % bits.value}
