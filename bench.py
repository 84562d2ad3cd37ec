#!/usr/bin/env python
"""bench.py -- RRI sweeps/sec + achieved HBM GB/s on BASELINE.json's headline configuration
(dense 200k x 20k low-rank-plus-noise, k=64, fp32, row-sharded over N GPUs of one box).

    python bench.py --gpus N --steps K --warmup W            (N>1: launched under torch.distributed.run)
    python bench.py --impl reference --gpus N --steps K --warmup W

A "step" is one full sweep (k T-steps and k W-steps) over the whole data set.  Prints ONE JSON line.
See DESIGN.md "Measurement" for what each key means.  --dump-outputs DIR also writes the factors W and T of the
last timed step (the inputs are seeded, so two builds run with the same arguments can be compared output for output).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # name: n, d, k (= planted rank), noise, dtype            (BASELINE.json "configs")
    'cfg1': dict(n=500, d=300, k=10, sigma=0.0, dtype='f64'),
    'cfg2': dict(n=20000, d=5000, k=32, sigma=0.05, dtype='f64'),
    'cfg3': dict(n=200000, d=20000, k=64, sigma=0.05, dtype='f32'),
    'cfg5': dict(n=1000000, d=20000, k=128, sigma=0.05, dtype='f32'),
    # config 4: masked WRRI recommender, 5 % observed; --masked dense (0/1 byte mask next to a dense X, the reference's
    # own data layout) or --masked sparse (the observed entries as CSR, rri_bind_csr)
    'cfg4': dict(n=100000, d=20000, k=50, sigma=0.05, dtype='f32', density=0.05),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=100)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', default='cfg3', choices=sorted(CONFIGS))
    ap.add_argument('--order', default=None, choices=['hals', 'rri'],
                    help="update order: default 'hals' (block order), for config 4 'rri' (the reference's interleaved order)")
    ap.add_argument('--math', default=None, choices=['ieee', 'tf32'])
    ap.add_argument('--rows', type=int, default=None, help='override n (debugging; the line then says so)')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-pageable', action='store_true', help='skip the e2e run from pageable host arrays')
    ap.add_argument('--no-rri', action='store_true', help='skip the side measurement of the reference-exact order')
    ap.add_argument('--cpu-rows', type=int, default=None)
    ap.add_argument('--masked', default='dense', choices=['dense', 'sparse'], help='config 4: data layout of the observed entries')
    ap.add_argument('--refresh-every', type=int, default=1, help='config 4 sparse: residual restart period (sweeps)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the factors the timed sweeps produced as DIR/W.npy and DIR/T.npy (at most 64 MB; '
                         'a fixed seeded sample of the rows of W when it does not fit)')
    a = ap.parse_args()
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    if a.order is None:
        a.order = 'rri' if a.config == 'cfg4' else 'hals'
    return a


# ------------------------------------------------------------------------------------------------
def load_traffic(key):
    """DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture of this
    configuration (profiles/traffic.json: dram__bytes_read.sum + dram__bytes_write.sum), or None"""
    p = os.path.join(ROOT, 'profiles', 'traffic.json')
    try:
        return json.load(open(p)).get(key)
    except Exception:
        return None


def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.isfile(p):
        try:
            j = json.load(open(p))
            return float(j['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
        except Exception:
            pass
    return 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region: the poller runs from program
    start (nvidia-smi takes a while to come up); `window()` keeps the samples whose host arrival time
    falls inside the timed region (or the nearest one when the region is shorter than a poll period)."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
         'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '50'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, universal_newlines=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(',')]))

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()

    def window(self, t0, t1):
        if self.proc is None or not self.rows:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable'], 'samples': 0}
        inside = [r for (t, r) in self.rows if t0 <= t <= t1 + 0.06]
        if not inside:
            mid = 0.5 * (t0 + t1)
            inside = [min(self.rows, key=lambda tr: abs(tr[0] - mid))[1]]
        sm, mx, pw, reasons = [], [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in inside:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                pw.append(float(r[3]))
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith('active'):
                        reasons.add(nm)
            except Exception:
                pass
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'power_w_max': max(pw) if pw else None, 'reasons': sorted(reasons), 'samples': len(sm)}


DUMP_BYTES = 64 * 10 ** 6


def _dump_sample(count, keep, seed):
    """indices 0..count-1, or a fixed seeded sorted sample of `keep` of them"""
    import numpy as np
    return np.arange(count) if keep >= count else np.sort(np.random.RandomState(seed).choice(count, keep, replace=False))


def dump_outputs(dirname, n, row0, W, T, dist=None):
    """--dump-outputs: W and T (NumPy, float32 or float64) as the timed sweeps left them, written to DIR/W.npy and
    DIR/T.npy.  When the two exceed DUMP_BYTES, W.npy holds the rows of a fixed seeded sample (sorted), the same for
    every run of the same configuration; T.npy likewise holds a sample of T's columns when T alone exceeds half of
    DUMP_BYTES.  With row shards every rank passes its rows [row0, row0 + len(W)) of the n global ones (collective)
    and rank 0 writes."""
    import numpy as np
    T = T[:, _dump_sample(T.shape[1], (DUMP_BYTES // 2) // (T.shape[0] * T.itemsize), 1)]
    keep = (DUMP_BYTES - T.nbytes - 4096) // (W.shape[1] * W.itemsize)       # 4 KB for the two .npy headers
    rows = _dump_sample(n, keep, 0)
    Ws = W[rows[(rows >= row0) & (rows < row0 + W.shape[0])] - row0]
    if dist is not None:
        parts = [None] * dist.get_world_size()
        dist.all_gather_object(parts, Ws)
        if dist.get_rank() != 0:
            return
        Ws = np.concatenate(parts)
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, 'W.npy'), Ws)
    np.save(os.path.join(dirname, 'T.npy'), T)


GEN_BLOCK = 8192


def gen_shard(torch, cfg, rows, row0, device, seed=None):
    """Rows [row0, row0+rows) of the GLOBAL matrix X = U V + sigma*mean(UV)*E (uniform factors, SURVEY.md §8d),
    generated on the device.  Every block of GEN_BLOCK global rows has its own generator seed, so the matrix (and
    W0) do not depend on how the rows are sharded: N = 1, 2, 4, 8 ranks factorise the SAME matrix and the line's
    `final_rel_error` must agree across N.  (`seed` is accepted for older callers and ignored.)"""
    d, r = cfg['d'], cfg['k']
    dt = torch.float32 if cfg['dtype'] == 'f32' else torch.float64
    g = torch.Generator(device=device)
    g.manual_seed(4242)
    V = torch.rand(r, d, generator=g, device=device, dtype=dt)          # shared by all shards
    X = torch.empty(rows, d, device=device, dtype=dt)
    W0 = torch.empty(rows, cfg['k'], device=device, dtype=dt)
    mean_uv = 0.25 * r                                                    # E[u v] * r for U[0,1) factors
    Xb = torch.empty(GEN_BLOCK, d, device=device, dtype=dt)
    for gb in range(row0 // GEN_BLOCK, (row0 + rows + GEN_BLOCK - 1) // GEN_BLOCK):
        # the whole block is generated with block-independent shapes (same cuBLAS kernel, same Philox stream on
        # every rank) and the shard's slice of it is kept
        g.manual_seed(100000 + gb)
        U = torch.rand(GEN_BLOCK, r, generator=g, device=device, dtype=dt)
        torch.matmul(U, V, out=Xb)
        if cfg['sigma']:
            Xb.add_(torch.rand(GEN_BLOCK, d, generator=g, device=device, dtype=dt), alpha=cfg['sigma'] * mean_uv)
        Wb = torch.rand(GEN_BLOCK, cfg['k'], generator=g, device=device, dtype=dt)
        lo, hi = max(row0, gb * GEN_BLOCK), min(row0 + rows, (gb + 1) * GEN_BLOCK)
        X[lo - row0:hi - row0] = Xb[lo - gb * GEN_BLOCK:hi - gb * GEN_BLOCK]
        W0[lo - row0:hi - row0] = Wb[lo - gb * GEN_BLOCK:hi - gb * GEN_BLOCK]
    del Xb
    g.manual_seed(77)
    T0 = torch.rand(cfg['k'], d, generator=g, device=device, dtype=dt)   # replicated
    return X, W0, T0


# ------------------------------------------------------------------------------------------------
REF_COPY = os.path.join(ROOT, 'oracle', '_ref')      # build-time copy of the reference's sources (git-ignored)


def _load_cpu_arm():
    """(kind, sweep_runner): the UNMODIFIED reference `nmf()` through oracle/refshim.py when `build()` left a copy of
    its sources under oracle/_ref/ (kind 'reference'), else the NumPy restatement oracle/rri_oracle.py ('port')."""
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import rri_oracle as orc
    if os.path.isfile(os.path.join(REF_COPY, 'src', 'rri_nmf', 'nmf.py')) and not os.environ.get('RRI_BENCH_PORT'):
        try:
            os.environ['RRI_REFERENCE_ROOT'] = REF_COPY
            import refshim
            refshim.REF_ROOT = REF_COPY
            ref = refshim.load()

            def run(X, k, W, T, sweeps, M=None):
                kw = dict(W_mat=M, t_row_sum=1.0) if M is not None else {}
                r = ref.nmf.nmf(X, k, W_in=W, T_in=T, max_iter=sweeps, max_time=1e9, eps_stop=-1.0,
                                compute_obj_each_iter=False, reset_topic_method=None, **kw)
                return r['W'], r['T']
            return 'reference', run, orc
        except Exception as ex:                    # a broken copy must not take the bench line down
            sys.stderr.write('reference copy under oracle/_ref unusable (%r); timing the port\n' % (ex,))

    def run(X, k, W, T, sweeps, M=None):
        W, T = W.copy(), T.copy()
        for _ in range(sweeps):
            orc.sweep(X, W, T, M=M, order='rri', t_row_sum=1.0 if M is not None else None)
        return W, T
    return 'port', run, orc


def cpu_reference_sweeps(cfg, rows, sweeps, warm=1, dump=None):
    """Time the reference's sweep (per-topic GEMVs over X, nmf.py:415-476, interleaved order -- the only order it
    has) on ALL host cores, on a row sample of the configuration; its cost is exactly linear in n, so the
    full-size figure is the sample's rate scaled by rows/n.  BLAS threads are forced to the number of available
    cores whatever OMP_NUM_THREADS says (torch.distributed.run exports OMP_NUM_THREADS=1).  dump: directory that
    receives the sample's W and T after the timed sweeps (dump_outputs)."""
    import numpy as np
    from threadpoolctl import threadpool_info, threadpool_limits
    ncores = len(os.sched_getaffinity(0))
    kind, run, orc = _load_cpu_arm()
    dt = np.float32 if cfg['dtype'] == 'f32' else np.float64
    M = None
    if cfg.get('density'):
        X, W0, T0, M = orc.synth(rows, cfg['d'], cfg['k'], cfg['k'], sigma=cfg['sigma'], seed=0, dtype=dt,
                                 mask_density=cfg['density'])
        M = M.astype(dt)
    else:
        X, W0, T0 = orc.synth(rows, cfg['d'], cfg['k'], cfg['k'], sigma=cfg['sigma'], seed=0, dtype=dt)
    W, T = np.maximum(W0, 0), np.maximum(T0, 0)
    with threadpool_limits(limits=ncores, user_api='blas'):
        info = [i for i in threadpool_info() if i.get('user_api') == 'blas']
        blas = '%s %s' % (info[0].get('internal_api'), info[0].get('version')) if info else 'unknown BLAS'
        threads = int(info[0].get('num_threads')) if info else ncores
        if warm > 0:
            W, T = run(X, cfg['k'], W, T, warm, M) if M is not None else run(X, cfg['k'], W, T, warm)
        t0 = time.perf_counter()
        W, T = run(X, cfg['k'], W, T, sweeps, M) if M is not None else run(X, cfg['k'], W, T, sweeps)
        dtm = (time.perf_counter() - t0) / sweeps
    if dump:
        dump_outputs(dump, rows, 0, W, T)
    full = dtm * cfg['n'] / rows
    what = ('the UNMODIFIED reference nmf() (oracle/_ref copy of src/rri_nmf, py3 shim, logger at WARNING)'
            if kind == 'reference' else 'the NumPy port oracle/rri_oracle.py of the reference sweep')
    return {'value': 1.0 / full, 'unit': 'sweeps/s', 'cores': threads, 'kind': kind,
            'sample': '%s on %d of %d rows (all %d columns, k=%d, %s): %d sweeps of the interleaved reference order '
                      '(%s) timed after %d warm-up, %.3f s/sweep on the sample, scaled '
                      'linearly in n; %s with %d BLAS threads (forced with threadpoolctl); host cores available %d'
                      % (what, rows, cfg['n'], cfg['d'], cfg['k'], cfg['dtype'], sweeps,
                         'masked WRRI with a %.0f %% 0/1 W_mat, ub_t=1: 2k dense residual products, nmf.py:687-701, :735-746' % (100 * cfg['density'])
                         if M is not None else '2k GEMV passes over X, nmf.py:415-476',
                         warm, dtm, blas, threads, ncores),
            'ms_per_sweep_sample': dtm * 1e3, 'sample_rows': rows, 'blas_threads': threads,
            'host_cores': ncores}


def cpu_sample_rows(cfg, sweeps, seconds):
    """rows of the sample so that `sweeps` reference sweeps take about `seconds` of wall time (the reference moves
    2k x rows x d elements per sweep at roughly 40 GB/s on these hosts; masked: 2k dense rows x k x d products per
    sweep plus ~8 elementwise passes over rows x d)"""
    if cfg.get('density'):
        per_row = 1e-2 * cfg['k'] * cfg['k'] * cfg['d'] / (50 * 50 * 20000)      # measured: 10 ms per row and sweep, 8 cores
        return int(min(cfg['n'], max(128, seconds / (max(1, sweeps) * per_row))))
    es = 4 if cfg['dtype'] == 'f32' else 8
    per_row = 2.0 * cfg['k'] * cfg['d'] * es / 40e9
    return int(min(cfg['n'], max(256, seconds / (max(1, sweeps) * per_row))))


def main_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return 0
    cfg = dict(CONFIGS[args.config])
    if args.rows:
        cfg['n'] = args.rows
    # bounded sample: K timed sweeps (+ warm-up) stay around a minute of CPU time
    rows = args.cpu_rows or cpu_sample_rows(cfg, args.steps + min(args.warmup, 1), 60.0)
    cb = cpu_reference_sweeps(cfg, rows, sweeps=args.steps, warm=max(0, min(args.warmup, 1)), dump=args.dump_outputs)
    line = {
        'impl': 'reference', 'metric': 'RRI sweeps/sec', 'value': cb['value'], 'unit': 'sweeps/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 / cb['value'], 'higher_is_better': True,
        'scaling': 'strong', 'vs_baseline': None, 'dtype': cfg['dtype'], 'data': 'synthetic',
        'config': {'workload': '%s: dense %dx%d low-rank-plus-noise, k=%d, %s%s' % (args.config, cfg['n'], cfg['d'], cfg['k'], cfg['dtype'], ', masked WRRI (5 %% observed)' if cfg.get('density') else ''),
                   'update_order': 'rri (the reference has only the interleaved order; the GPU arm reports the same '
                                   'order under "reference_order" and the ratio under "like_for_like")',
                   'sample_rows': rows},
        'cpu_baseline': cb,
        'e2e': {'value': cb['value'], 'unit': 'sweeps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------
def main_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import rri_nmf_b200 as R
    from rri_nmf_b200.engine import NcclComm
    from rri_nmf_b200.sharding import shard_bounds

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit('--gpus %d needs torch.distributed.run --nproc-per-node %d' % (args.gpus, args.gpus))
    torch.cuda.set_device(local)
    device = torch.device('cuda', local)
    comm = None
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=device)
        comm = NcclComm(local)

    sampler = ClockSampler(local)          # started before data generation: nvidia-smi needs a second to come up
    if rank == 0:
        sampler.start()
    cfg = dict(CONFIGS[args.config])
    if args.rows:
        cfg['n'] = args.rows
    math = args.math or ('tf32' if (cfg['dtype'] == 'f32' and args.order == 'hals') else 'ieee')
    n, d, k = cfg['n'], cfg['d'], cfg['k']
    es = 4 if cfg['dtype'] == 'f32' else 8
    b, e = shard_bounds(n, world)[rank]
    X, W0, T0 = gen_shard(torch, cfg, e - b, b, device)
    eng = R.RRIEngine(X, k, order=args.order, math=math, comm=comm)
    params = eng.params()
    peer_x = bool(getattr(eng, 'peer_exchange', False))
    W, T = W0.clone(), T0.clone()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # K steps = K sweeps issued by ONE call of the engine (like nmf(max_iter=K) does): the per-call set-up
    # (transposed factor copies, flag reset) is paid once, not once per sweep
    if args.warmup > 0:
        eng.sweeps(W, T, args.warmup, params, want_flags=False)
    barrier()
    l0 = eng.stats()['kernel_launches']
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    th0 = time.time()
    ev0.record()
    eng.sweeps(W, T, args.steps, params, want_flags=False)
    ev1.record()
    barrier()
    th1 = time.time()
    ms = ev0.elapsed_time(ev1)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, n, b, W.cpu().numpy(), T.cpu().numpy(), dist if world > 1 else None)
    clocks = None
    if rank == 0:
        time.sleep(0.12)
        clocks = sampler.window(th0, th1)
        sampler.stop()
    launches = eng.stats()['kernel_launches'] - l0
    if world > 1:
        t = torch.tensor([ms], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    ms_per_step = ms / args.steps
    value = 1e3 / ms_per_step
    relerr = eng.rel_error(W, T)

    # ---- roofline of the dominant kernel (timed alone, CUDA events on the launching stream)
    peak, peak_src = load_peaks()
    passes = 2 if args.order == 'hals' else k
    if args.order == 'hals':
        kms = 0.5 * (eng.profile_kernel('gemm_w', W, T, 5) + eng.profile_kernel('gemm_t', W, T, 5))
        kname = 'tf32 tcgen05 contraction (X T\' and X\' W)' if math == 'tf32' else 'simt contraction'
    else:
        kms = eng.profile_kernel('rri_pass', W, T, 5)
        kname = 'rri_pass_kernel (y = X T_t\', p = w_t\' X)'
    alg_bytes = float(e - b) * d * es                       # one read of the local X per launch
    achieved = alg_bytes / (kms * 1e-3) / 1e9
    roofline = {'bound': 'hbm', 'kernel': kname, 'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
                'frac': achieved / peak,
                'traffic': load_traffic('%s/%s/%s/rows%d' % (args.config, args.order, math, e - b)),
                'peak_source': peak_src, 'kernel_ms': kms,
                'algorithmic_bytes_per_launch': alg_bytes, 'launches_per_sweep': passes,
                'sweep_effective_gbs': passes * alg_bytes / (ms_per_step * 1e-3) / 1e9,
                'kernel_share_of_step': passes * kms / ms_per_step}

    if args.order == 'hals':
        # whole half-steps (contraction + Gram + exchange + update), CUDA events; what is not the contraction is the
        # fixed cost that does not shrink with the shard
        try:
            Wc, Tc = W.clone(), T.clone()
            th, wh = eng.profile_kernel('t_half', Wc, Tc, 5), eng.profile_kernel('w_half', Wc, Tc, 5)
            gt, gw = eng.profile_kernel('gemm_t', Wc, Tc, 5), eng.profile_kernel('gemm_w', Wc, Tc, 5)
            roofline['half_steps_ms'] = {'t_half': th, 'w_half': wh, 'gemm_t': gt, 'gemm_w': gw,
                                         't_half_minus_contraction': th - gt, 'w_half_minus_contraction': wh - gw}
            del Wc, Tc
        except Exception as ex:
            roofline['half_steps_ms'] = {'error': repr(ex)[:200]}

    objective_cost = None
    if args.order == 'hals':
        # an objective per sweep (compute_obj_each_iter=True): the explicit pass over X against the form that
        # reuses the sweep's own contraction
        try:
            Wc, Tc = W.clone(), T.clone()

            def timed(fn, reps):
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                a0.record()
                for _ in range(reps):
                    fn()
                a1.record()
                torch.cuda.synchronize()
                return a0.elapsed_time(a1) / reps

            def sweep_and_obj():
                eng.sweeps(Wc, Tc, 1, params, want_flags=False)
                return eng.objective(Wc, Tc, via_contraction=True, reuse_last_sweep=True)

            sweep_and_obj()
            t_both = timed(sweep_and_obj, 5)
            t_sweep = timed(lambda: eng.sweeps(Wc, Tc, 1, params, want_flags=False), 5)
            eng.sweeps(Wc, Tc, 1, params, want_flags=False)
            o_fast = eng.objective(Wc, Tc, via_contraction=True, reuse_last_sweep=True)
            o_exact = eng.objective(Wc, Tc)
            t_exact = timed(lambda: eng.objective(Wc, Tc), 2)
            objective_cost = {'ms_sweep': t_sweep, 'ms_sweep_plus_objective_via_contraction': t_both,
                              'overhead_frac': t_both / t_sweep - 1.0, 'ms_explicit_objective_pass': t_exact,
                              'objective_via_contraction': o_fast, 'objective_explicit': o_exact,
                              'rel_diff': o_fast / o_exact - 1.0, 'world_local_terms_only': world > 1}
            del Wc, Tc
        except Exception as ex:
            objective_cost = {'error': repr(ex)[:200]}

    # ---- e2e: the public call with HOST buffers, copies inside the timed region.  Two figures: pinned host arrays
    # (the headline e2e) and plain pageable NumPy arrays (what a drop-in user passes; nmf() stages them through
    # its own pinned chunk buffers)
    e2e = None
    if not args.no_e2e:
        try:
            Xh = torch.empty(X.shape, dtype=X.dtype, pin_memory=True)
            Xh.copy_(X)
            Wh, Th = W0.cpu().pin_memory(), T0.cpu().pin_memory()
            eng.close()
            del eng
            torch.cuda.synchronize()
            s_e2e = args.steps

            def e2e_call(Xa, Wa, Ta):
                barrier()
                t0 = time.perf_counter()
                out = R.nmf(Xa, k, W_in=Wa, T_in=Ta, max_iter=s_e2e, reset_topic_method=None,
                            max_time=1e9, update_order=args.order, math=math, device=device, comm=comm)
                _ = float(out['W'][0, 0])
                t_call = time.perf_counter() - t0
                barrier()
                dt = time.perf_counter() - t0
                if world > 1:
                    tt = torch.tensor([dt], device=device, dtype=torch.float64)
                    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                    dt = float(tt.item())
                return dt, dict(out.get('timing', {}), call_s=t_call)

            e2e_call(Xh.numpy()[:1024], Wh.numpy()[:1024], Th.numpy())          # library/allocator warm-up, untimed
            dt, ph = e2e_call(Xh.numpy(), Wh.numpy(), Th.numpy())
            hb = (Xh.numel() + Wh.numel() + Th.numel()) * es * world
            db = (Wh.numel() + Th.numel()) * es * world
            e2e = {'value': s_e2e / dt, 'unit': 'sweeps/s', 'h2d_bytes_per_step': hb / s_e2e,
                   'd2h_bytes_per_step': db / s_e2e,
                   'what': 'rri_nmf_b200.nmf(X_host, k, W_in, T_in, max_iter=%d) from pinned host arrays: H2D of X/W/T, '
                           '%d sweeps, D2H of W/T; %.3f s total' % (s_e2e, s_e2e, dt),
                   'rank0_phases_s': ph}
            if not args.no_pageable:
                Xp = np.empty(tuple(X.shape), dtype=np.float32 if es == 4 else np.float64)   # pageable
                Xp[...] = Xh.numpy()
                Wp, Tp = np.array(Wh.numpy()), np.array(Th.numpy())
                del Xh
                dtp, php = e2e_call(Xp, Wp, Tp)
                e2e['pageable'] = {'value': s_e2e / dtp, 'unit': 'sweeps/s', 'total_s': dtp, 'rank0_phases_s': php,
                                   'what': 'the same call with plain (pageable) NumPy arrays', 'vs_pinned': dtp / dt}
                del Xp
        except Exception as ex:        # host RAM too small for a pinned copy, etc.
            e2e = {'value': None, 'unit': 'sweeps/s', 'h2d_bytes_per_step': None, 'd2h_bytes_per_step': None,
                   'error': repr(ex)[:200]}

    # ---- side measurement: the reference-exact interleaved order on the same data (k passes over X per sweep)
    rri_side = None
    if args.order == 'hals' and not args.no_rri:
        try:
            eng_r = R.RRIEngine(X, k, order='rri', math='ieee', comm=comm)
            Wr, Tr = W0.clone(), T0.clone()
            eng_r.sweeps(Wr, Tr, 1, params, want_flags=False)
            barrier()
            r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            r0.record()
            for _ in range(2):
                eng_r.sweeps(Wr, Tr, 1, params, want_flags=False)
            r1.record()
            barrier()
            rms = r0.elapsed_time(r1) / 2
            if world > 1:
                tr = torch.tensor([rms], device=device, dtype=torch.float64)
                dist.all_reduce(tr, op=dist.ReduceOp.MAX)
                rms = float(tr.item())
            pk = eng_r.profile_kernel('rri_pass', Wr, Tr, 3)
            rri_side = {'update_order': 'rri (reference-exact, nmf.py:415-476)', 'value': 1e3 / rms, 'unit': 'sweeps/s',
                        'ms_per_step': rms, 'steps': 2, 'pass_kernel_ms': pk,
                        'pass_kernel_gbs': alg_bytes / (pk * 1e-3) / 1e9, 'pass_kernel_frac': alg_bytes / (pk * 1e-3) / 1e9 / peak}
            eng_r.close()
            del Wr, Tr
        except Exception as ex:
            rri_side = {'error': repr(ex)[:200]}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        rows = args.cpu_rows or cpu_sample_rows(cfg, 6, 20.0)      # 5 timed sweeps + 1 warm-up in about 20 s
        cpu = cpu_reference_sweeps(cfg, rows, sweeps=5, warm=1)

    if rank == 0:
        line = {
            'metric': 'RRI sweeps/sec', 'value': value, 'unit': 'sweeps/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': 'strong',
            'vs_baseline': None, 'dtype': cfg['dtype'] + ('/tf32-mma' if math == 'tf32' else ''), 'data': 'synthetic',
            'config': {'workload': '%s: dense %dx%d low-rank-plus-noise (sigma=%.2f), k=%d, %s, row-sharded over %d GPU(s)'
                                   % (args.config, n, d, cfg['sigma'], k, cfg['dtype'], world),
                       'update_order': args.order, 'math': math, 'rows_per_gpu': e - b,
                       'l2_policy': 'inputs (%.1f GB/GPU) larger than L2; no flush needed' % (alg_bytes / 1e9),
                       'final_rel_error': relerr,
                       'exchange': ('nvlink peer memory (fused into the T update)' if peer_x else 'nccl all-reduce') if world > 1 else 'none'},
            'roofline': roofline, 'cpu_baseline': cpu, 'e2e': e2e, 'gpu_launches': launches, 'clocks': clocks,
            'reference_order': rri_side, 'objective_per_sweep': objective_cost,
        }
        if cpu and rri_side and rri_side.get('value'):
            # same update order on both sides: the reference's interleaved sweep on the GPU over the CPU figure
            line['like_for_like'] = {'update_order': 'rri (nmf.py:415-476) on both sides', 'gpu_value': rri_side['value'],
                                     'cpu_value': cpu['value'], 'ratio': rri_side['value'] / cpu['value'],
                                     'cpu_kind': cpu['kind'], 'cpu_cores': cpu['cores']}
        elif cpu and args.order == 'rri':
            line['like_for_like'] = {'update_order': 'rri (nmf.py:415-476) on both sides', 'gpu_value': value,
                                     'cpu_value': cpu['value'], 'ratio': value / cpu['value'],
                                     'cpu_kind': cpu['kind'], 'cpu_cores': cpu['cores']}
        print(json.dumps(line))
    if world > 1:
        if comm is not None:
            comm.destroy()
        dist.destroy_process_group()
    return 0


def gen_mask_shard(torch, cfg, rows, row0, device):
    """0/1 byte mask of the observed entries (Bernoulli(density)), per global block of GEN_BLOCK rows like gen_shard"""
    g = torch.Generator(device=device)
    M = torch.empty(rows, cfg['d'], device=device, dtype=torch.uint8)
    for gb in range(row0 // GEN_BLOCK, (row0 + rows + GEN_BLOCK - 1) // GEN_BLOCK):
        g.manual_seed(700000 + gb)
        Mb = (torch.rand(GEN_BLOCK, cfg['d'], generator=g, device=device) < cfg['density']).to(torch.uint8)
        lo, hi = max(row0, gb * GEN_BLOCK), min(row0 + rows, (gb + 1) * GEN_BLOCK)
        M[lo - row0:hi - row0] = Mb[lo - gb * GEN_BLOCK:hi - gb * GEN_BLOCK]
    return M


def main_masked(args):
    """config 4: masked WRRI sweeps (reference order by default), dense byte mask or observed entries as CSR"""
    import numpy as np
    import torch
    import rri_nmf_b200 as R
    if int(os.environ.get('WORLD_SIZE', '1')) != 1 or args.gpus != 1:
        raise SystemExit('config 4 is benchmarked on one GPU (the multi-GPU masked path is covered by tests/multi_gpu_check.py)')
    device = torch.device('cuda', 0)
    torch.cuda.set_device(0)
    sampler = ClockSampler(0)
    sampler.start()
    cfg = dict(CONFIGS['cfg4'])
    if args.rows:
        cfg['n'] = args.rows
    order = args.order
    n, d, k = cfg['n'], cfg['d'], cfg['k']
    X, W0, T0 = gen_shard(torch, cfg, n, 0, device)
    M = gen_mask_shard(torch, cfg, n, 0, device)
    sparse = args.masked == 'sparse'
    if sparse:
        Xs = (X * M).to_sparse_csr()
        nnz = int(Xs.values().numel())
        eng = R.RRIEngine(Xs, k, order=order)
        math = 'ieee'
        alg_bytes = 10.0 * nnz                          # 2 B local index + 4 B residual read + 4 B residual written
        kname = 'sp_pass_stream_kernel + solve (one T half-step of one topic over the observed entries)'
    else:
        nnz = int(M.sum())
        math = args.math or 'tf32'
        eng = R.RRIEngine(X, k, W_mat=M, order=order, math=math)
        alg_bytes = float(n) * d * 5.0                  # one read of X (fp32) and of the byte mask
        kname = 'wrri_tc_tma_kernel (masked statistics of one half-step, W T tile on tcgen05)' if math == 'tf32' else 'wrri_tstats/wstats_kernel'
    params = eng.params(ub_t=1.0, sp_refresh_every=args.refresh_every)
    W, T = W0.clone(), T0.clone()
    if args.warmup > 0:
        eng.sweeps(W, T, args.warmup, params, want_flags=False)
    torch.cuda.synchronize()
    l0 = eng.stats()['kernel_launches']
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    th0 = time.time()
    ev0.record()
    eng.sweeps(W, T, args.steps, params, want_flags=False)
    ev1.record()
    torch.cuda.synchronize()
    th1 = time.time()
    ms_per_step = ev0.elapsed_time(ev1) / args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, n, 0, W.cpu().numpy(), T.cpu().numpy())
    time.sleep(0.12)
    clocks = sampler.window(th0, th1)
    sampler.stop()
    launches = eng.stats()['kernel_launches'] - l0
    relerr = eng.rel_error(W, T)
    peak, peak_src = load_peaks()
    Wc, Tc = W.clone(), T.clone()
    kt, kw = eng.profile_kernel('masked_t', Wc, Tc, 5), eng.profile_kernel('masked_w', Wc, Tc, 5)
    kms = 0.5 * (kt + kw)
    achieved = alg_bytes / (kms * 1e-3) / 1e9
    roofline = {'bound': 'hbm', 'kernel': kname, 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                'traffic': load_traffic('cfg4/%s/%s/rows%d' % (args.masked, order, n)), 'peak_source': peak_src,
                'kernel_ms': kms, 'half_step_ms': {'t_step': kt, 'w_step': kw, 'includes': 'statistics pass + solve + sum'},
                'algorithmic_bytes_per_launch': alg_bytes, 'launches_per_sweep': 2 * k,
                'sweep_effective_gbs': 2 * k * alg_bytes / (ms_per_step * 1e-3) / 1e9,
                'kernel_share_of_step': 2 * k * kms / ms_per_step}
    del Wc, Tc
    e2e = None
    if not args.no_e2e:
        try:
            eng.close()
            Wh, Th = W0.cpu().pin_memory(), T0.cpu().pin_memory()
            if sparse:
                Xh = Xs.cpu()
                kw_ = {}
                hb = (Xh.values().numel() * 8 + Xh.crow_indices().numel() * 8 + Wh.numel() * 4 + Th.numel() * 4)
            else:
                Xp = torch.empty(X.shape, dtype=X.dtype, pin_memory=True); Xp.copy_(X)
                Mp = torch.empty(M.shape, dtype=torch.uint8, pin_memory=True); Mp.copy_(M)
                Xh, kw_ = Xp.numpy(), {'W_mat': Mp, 'math': math}
                hb = Xp.numel() * 4 + Mp.numel() + Wh.numel() * 4 + Th.numel() * 4
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = R.nmf(Xh, k, W_in=Wh.numpy(), T_in=Th.numpy(), max_iter=args.steps, reset_topic_method=None, max_time=1e9,
                        t_row_sum=1.0, update_order=order, device=device, sparse_refresh_every=args.refresh_every, **kw_)
            _ = float(out['W'][0, 0])
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            e2e = {'value': args.steps / dt, 'unit': 'sweeps/s', 'h2d_bytes_per_step': hb / args.steps,
                   'd2h_bytes_per_step': (Wh.numel() + Th.numel()) * 4 / args.steps,
                   'what': 'rri_nmf_b200.nmf(X_host, k, W_mat / sparse X, ...) from host arrays: H2D, %d sweeps, D2H of W/T; %.3f s total' % (args.steps, dt),
                   'rank0_phases_s': out.get('timing')}
        except Exception as ex:
            e2e = {'value': None, 'unit': 'sweeps/s', 'h2d_bytes_per_step': None, 'd2h_bytes_per_step': None, 'error': repr(ex)[:200]}
    cpu = None
    if not args.no_cpu:
        rows = args.cpu_rows or cpu_sample_rows(cfg, 4, 20.0)
        cpu = cpu_reference_sweeps(cfg, rows, sweeps=3, warm=1)
    line = {'metric': 'RRI sweeps/sec', 'value': 1e3 / ms_per_step, 'unit': 'sweeps/s', 'n_gpus': 1, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None,
            'dtype': 'f32' + ('/tf32-mma' if math == 'tf32' else ''), 'data': 'synthetic',
            'config': {'workload': 'cfg4: masked WRRI recommender %dx%d, %.0f %% observed (nnz = %d), k=%d, f32, ub_t=1, %s' %
                                   (n, d, 100 * cfg['density'], nnz, k, 'observed entries as CSR + CSC' if sparse else 'dense X + 0/1 byte mask'),
                       'update_order': order, 'math': math, 'masked': args.masked, 'refresh_every': args.refresh_every,
                       'l2_policy': 'inputs (%.1f GB per pass) larger than L2; no flush needed' % (alg_bytes / 1e9),
                       'final_rel_error': relerr},
            'roofline': roofline, 'cpu_baseline': cpu, 'e2e': e2e, 'gpu_launches': launches, 'clocks': clocks}
    if cpu and order == 'rri':
        line['like_for_like'] = {'update_order': 'rri (masked WRRI, nmf.py:687-701 / :735-746) on both sides',
                                 'gpu_value': line['value'], 'cpu_value': cpu['value'], 'ratio': line['value'] / cpu['value'],
                                 'cpu_kind': cpu['kind'], 'cpu_cores': cpu['cores']}
    print(json.dumps(line))
    return 0


if __name__ == '__main__':
    a = parse()
    if a.impl == 'reference':
        sys.exit(main_reference(a))
    sys.exit(main_masked(a) if a.config == 'cfg4' else main_ours(a))
