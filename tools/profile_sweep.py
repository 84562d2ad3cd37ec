"""Kernel times of block-order sweeps at a bench configuration (torch.profiler, CUDA activities): one table of the
kernels of `--sweeps` sweeps issued by one engine call, after a warm-up call.  Run from the repository root."""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--config', default='cfg3')
    ap.add_argument('--sweeps', type=int, default=10)
    a = ap.parse_args()
    import torch
    import bench
    import rri_nmf_b200 as R
    cfg = dict(bench.CONFIGS[a.config])
    dev = torch.device('cuda', 0)
    X, W, T = bench.gen_shard(torch, cfg, cfg['n'], 0, dev)
    eng = R.RRIEngine(X, cfg['k'], order='hals', math='tf32')
    p = eng.params()
    eng.sweeps(W, T, 3, p, want_flags=False)
    torch.cuda.synchronize()
    from torch.profiler import profile, ProfilerActivity
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        eng.sweeps(W, T, a.sweeps, p, want_flags=False)
        torch.cuda.synchronize()
    print(prof.key_averages().table(sort_by='cuda_time_total', row_limit=25, max_name_column_width=70))
    print('per sweep: divide the totals by', a.sweeps)


if __name__ == '__main__':
    main()
