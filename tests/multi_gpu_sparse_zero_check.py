"""Row-sharded parity of zero-filled sparse data (run under torch.distributed.run, one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29541 \
        tests/multi_gpu_sparse_zero_check.py

Every rank binds the CSR rows of its shard with unstored='zero'; the T half-step all-reduces [X_i'W_i | W_i'W_i] over
NCCL (the peer-memory exchange serves dense data only).  Rank 0 compares the gathered factors and the objective with the
unsharded NumPy oracle on X.toarray() (fp64, 1e-9); the T replicas must be bit-identical on every rank."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'oracle'))
sys.path.insert(0, os.path.join(ROOT, 'tools'))
import rri_oracle as orc                      # noqa: E402
import scipy.sparse as sp                     # noqa: E402
import rri_nmf_b200 as R                      # noqa: E402
from bench_sparse_zero import text_like       # noqa: E402
from rri_nmf_b200._host import initialize_nmf  # noqa: E402
from rri_nmf_b200.engine import NcclComm      # noqa: E402
from rri_nmf_b200.sharding import shard_bounds  # noqa: E402


def main():
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    rank, world = dist.get_rank(), dist.get_world_size()
    comm = NcclComm(local)
    ok = True

    def gather_rows(Wl):
        parts = [None] * world
        dist.all_gather_object(parts, Wl)
        return np.vstack(parts)

    def replicas_identical(Tnp):
        tt = torch.from_numpy(np.ascontiguousarray(Tnp)).cuda()
        t0 = tt.clone()
        dist.broadcast(t0, src=0)
        flag = torch.tensor([1 if torch.equal(t0, tt) else 0], device='cuda')
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        return bool(flag.item())

    n = 1003
    for d, k, kw in ((517, 16, {}), (517, 7, dict(project_T_each_iter=True, t_row_sum=1.0, w_row_sum=1.0))):
        Xt = text_like(n, d, 0.05, k, seed=k)
        X = sp.csr_matrix((Xt.values().numpy().astype(np.float64), Xt.col_indices().numpy(), Xt.crow_indices().numpy()),
                          shape=(n, d))
        W0, T0 = initialize_nmf(X, k, 'nndsvda', random_state=0)
        b, e = shard_bounds(n, world)[rank]
        kw = dict(kw, compute_obj_each_iter=True, eps_stop=-1.0)
        o = orc.nmf_oracle(X.toarray(), k, W0, T0, max_iter=3, order='hals', **kw)
        g = R.nmf(X[b:e], k, W_in=W0[b:e], T_in=T0, max_iter=3, update_order='hals', unstored='zero',
                  reset_topic_method=None, comm=comm, device='cuda:%d' % local, **kw)
        Wg = gather_rows(g['W'])
        rw = np.linalg.norm(Wg - o['W']) / np.linalg.norm(o['W'])
        rt = np.linalg.norm(g['T'] - o['T']) / np.linalg.norm(o['T'])
        ro = np.max(np.abs(np.array(g['obj_history']) / np.array(o['obj_history']) - 1))
        same = replicas_identical(g['T'])
        good = rw < 1e-9 and rt < 1e-9 and ro < 1e-9 and same
        ok = ok and good
        if rank == 0:
            print('sparse zero d=%d k=%d relW=%.2e relT=%.2e relObj=%.2e replicas identical: %s %s'
                  % (d, k, rw, rt, ro, same, 'ok' if good else 'FAIL'), flush=True)
    flag = torch.tensor([1 if ok else 0], device='cuda')
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    comm.destroy()
    dist.destroy_process_group()
    if rank == 0:
        print('MULTI_GPU_SPARSE_ZERO %s (world=%d)' % ('PASS' if int(flag.item()) else 'FAIL', world), flush=True)
    sys.exit(0 if int(flag.item()) else 1)


if __name__ == '__main__':
    main()
