"""Block order (update_order='hals') with project_T_each_iter on unmasked dense data: the constrained T update
(simplex_kernels.cu -- one cooperative launch, or the per-topic chain) against the oracle's block-order sweep
(rri_oracle.sweep(order='hals', project_T_each_iter=True)), its dispatch, determinism and the estimator on top."""
import os

import numpy as np
import pytest
import torch

import rri_oracle as orc
import simplex_theta as sx
from conftest import golden, relfro

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def R(cuda_device):
    import rri_nmf_b200
    return rri_nmf_b200


def _nmf_vs_oracle(R, X, k, W0, T0, sweeps, tol, **kw):
    """after each of 1..sweeps sweeps: device factors within tol (relative Frobenius) of the oracle's"""
    for ns in range(1, sweeps + 1):
        o = orc.nmf_oracle(X, k, W0, T0, max_iter=ns, order='hals', project_T_each_iter=True, **kw)
        g = R.nmf(X, k, W_in=W0, T_in=T0, max_iter=ns, update_order='hals', project_T_each_iter=True,
                  reset_topic_method=None, **kw)
        assert relfro(g['T'], o['T']) <= tol, (ns, relfro(g['T'], o['T']))
        assert relfro(g['W'], o['W']) <= tol, (ns, relfro(g['W'], o['W']))
        if 'obj_history' in o:
            assert np.allclose(g['obj_history'], o['obj_history'], rtol=tol, atol=0)
    return g


def _check_simplex(T, s):
    assert np.all(T >= 0)
    assert np.max(np.abs(T.sum(1) - s)) <= 1e-12 * max(1.0, s)


@pytest.mark.parametrize('project_W', [False, True])
@pytest.mark.parametrize('reg_t_l2', [0.0, 0.1, -0.1])
def test_tm_fixture_fp64(R, project_W, reg_t_l2):
    from rri_nmf_b200._host import initialize_nmf, normalize
    X = golden('text_tm_f64.npz')['X']
    W0, T0 = initialize_nmf(X, 15, 'nndsvd', random_state=0, row_normalize=False)    # as nmf() starts (nmf.py:840-850)
    W0, T0 = normalize(W0), normalize(T0)
    out = _nmf_vs_oracle(R, X, 15, W0, T0, 3, 1e-9, w_row_sum=1.0, t_row_sum=1.0, project_W_each_iter=project_W,
                         reg_t_l2=reg_t_l2, reg_w_l2=0.1)
    _check_simplex(out['T'], 1.0)


@pytest.mark.parametrize('k,t_row_sum', [(64, 1.0), (1, 1.0), (80, 1.0), (16, 2.5), (2, 2.5)])
def test_synthetic_fp64(R, k, t_row_sum):
    """d = 517 (not a multiple of the 128-column block); k = 64 / 16 / 2 fused, k = 1 (odd) and 80 (> 64) the chain"""
    X, W0, T0 = sx.topic_data(300, 517, k, t_row_sum, seed=k)
    out = _nmf_vs_oracle(R, X, k, W0, T0, 3, 1e-9, t_row_sum=t_row_sum)
    _check_simplex(out['T'], t_row_sum)


def test_objective_auto_after_constrained_sweeps(R):
    """objective='auto' (fp64: the contraction form, reusing the sweep's own contraction) stays exact"""
    X, W0, T0 = sx.topic_data(400, 300, 12, seed=2)
    _nmf_vs_oracle(R, X, 12, W0, T0, 1, 1e-9, t_row_sum=1.0, w_row_sum=1.0, compute_obj_each_iter=True,
                   eps_stop=-1.0)
    o = orc.nmf_oracle(X, 12, W0, T0, max_iter=6, order='hals', project_T_each_iter=True, t_row_sum=1.0,
                       w_row_sum=1.0, project_W_each_iter=True, compute_obj_each_iter=True, eps_stop=-1.0)
    g = R.nmf(X, 12, W_in=W0, T_in=T0, max_iter=6, update_order='hals', project_T_each_iter=True, t_row_sum=1.0,
              w_row_sum=1.0, project_W_each_iter=True, compute_obj_each_iter=True, eps_stop=-1.0,
              reset_topic_method=None, objective='auto')
    assert np.allclose(g['obj_history'], o['obj_history'], rtol=1e-9, atol=0)
    assert relfro(g['T'], o['T']) <= 1e-9 and relfro(g['W'], o['W']) <= 1e-9


def _engine_case(R, n, d, k, dtype, math='ieee', seed=0):
    X, W0, T0 = sx.topic_data(n, d, k, seed=seed)
    dev = torch.device('cuda:0')
    Xd = torch.from_numpy(X.astype(dtype)).to(dev)
    eng = R.RRIEngine(Xd, k, order='hals', math=math)
    W = torch.from_numpy(W0.astype(dtype)).to(dev)
    T = torch.from_numpy(T0.astype(dtype)).to(dev)
    eng.project_rows_simplex(T, 1.0)
    return eng, W, T


def _launches_per_sweep(eng, W, T, params):
    a = eng.stats()['kernel_launches']
    eng.sweeps(W, T, 1, params)
    return eng.stats()['kernel_launches'] - a


@pytest.mark.parametrize('n,d,k,dtype,fused', [
    (200, 517, 64, np.float64, True),        # fp64 up to k = 64, k a multiple of 2
    (200, 517, 80, np.float64, False),       # fp64 k > 64
    (200, 517, 15, np.float64, False),       # k not a multiple of the 16-byte vector
    (200, 1000, 128, np.float32, True),      # fp32 up to k = 128
    (200, 1000, 132, np.float32, False),     # fp32 k > 128
    (16, 600000, 16, np.float32, False),     # grid too large to be co-resident
])
def test_dispatch(R, n, d, k, dtype, fused):
    """the fused kernel is one launch per T half-step (as the unconstrained row update), the chain 2k + 1"""
    eng, W, T = _engine_case(R, n, d, k, dtype)
    free = _launches_per_sweep(eng, W.clone(), T.clone(), eng.params())
    cons = _launches_per_sweep(eng, W, T, eng.params(ub_t=1.0, simplex_T=True))
    assert cons - free == (0 if fused else 2 * k), (cons, free)
    Th = T.double().cpu().numpy()
    assert np.all(Th >= 0)
    assert np.max(np.abs(Th.sum(1) - 1.0)) <= (1e-12 if dtype == np.float64 else 1e-5)
    eng.close()


def test_dispatch_switch_forces_the_chain(R, monkeypatch):
    """RRI_SIMPLEX_FUSED=0 runs the chain where the fused kernel applies; both agree to rounding"""
    eng, W, T = _engine_case(R, 300, 517, 32, np.float64)
    p = eng.params(ub_t=1.0, simplex_T=True)
    W2, T2 = W.clone(), T.clone()
    free = _launches_per_sweep(eng, W.clone(), T.clone(), eng.params())
    assert _launches_per_sweep(eng, W, T, p) == free
    monkeypatch.setenv('RRI_SIMPLEX_FUSED', '0')
    assert _launches_per_sweep(eng, W2, T2, p) == free + 2 * 32
    assert relfro(T2.cpu().numpy(), T.cpu().numpy()) < 1e-13
    assert relfro(W2.cpu().numpy(), W.cpu().numpy()) < 1e-13
    eng.close()


@pytest.mark.parametrize('k,chain', [(32, False), (32, True), (15, False)])
def test_reentrance_and_run_to_run_bitwise(R, monkeypatch, k, chain):
    if chain:
        monkeypatch.setenv('RRI_SIMPLEX_FUSED', '0')
    eng, W0, T0 = _engine_case(R, 500, 3000, k, np.float32, seed=4)
    p = eng.params(ub_t=1.0, simplex_T=True)
    W, T = W0.clone(), T0.clone()
    eng.sweeps(W, T, 5, p)
    W1, T1 = W0.clone(), T0.clone()
    for _ in range(5):
        eng.sweeps(W1, T1, 1, p)
    assert torch.equal(W, W1) and torch.equal(T, T1)
    W2, T2 = W0.clone(), T0.clone()
    eng.sweeps(W2, T2, 5, p)
    assert torch.equal(W, W2) and torch.equal(T, T2)
    eng.close()


@pytest.mark.parametrize('math', ['ieee', 'tf32'])
def test_fp32_against_fp64_oracle(R, math):
    X, W0, T0 = sx.topic_data(2048, 1024, 32, seed=8)
    o = orc.nmf_oracle(X, 32, W0, T0, max_iter=3, order='hals', project_T_each_iter=True, t_row_sum=1.0)
    g = R.nmf(X.astype(np.float32), 32, W_in=W0.astype(np.float32), T_in=T0.astype(np.float32), max_iter=3,
              update_order='hals', math=math, project_T_each_iter=True, t_row_sum=1.0, reset_topic_method=None)
    re_o = orc.rel_error(X, o['W'], o['T'])
    re_g = orc.rel_error(X, g['W'].astype(np.float64), g['T'].astype(np.float64))
    assert abs(re_g - re_o) < 1e-4, (re_g, re_o)
    assert np.all(g['T'] >= 0) and np.max(np.abs(g['T'].astype(np.float64).sum(1) - 1)) < 1e-5


def test_c_nonpositive_with_radius_not_one_raises(R):
    """a denominator ||w_t||^2 + reg_t_l2 <= 0 with t_row_sum != 1: the oracle's qf_min raises NotImplementedError"""
    X, W0, T0 = orc.synth(50, 300, 4, 4, seed=1)
    W0 = W0 * 0.01
    with pytest.raises(NotImplementedError):
        orc.nmf_oracle(X, 4, W0, T0, max_iter=1, order='hals', project_T_each_iter=True, t_row_sum=2.0, reg_t_l2=-10.0)
    with pytest.raises(NotImplementedError):
        R.nmf(X, 4, W_in=W0, T_in=T0, max_iter=1, update_order='hals', project_T_each_iter=True, t_row_sum=2.0,
              reg_t_l2=-10.0, reset_topic_method=None)


def test_c_nonpositive_with_radius_one_is_one_hot(R):
    X, W0, T0 = orc.synth(50, 300, 4, 4, seed=1)
    W0 = W0 * 0.01
    for k_case in (4, 5):           # fused (even k) and chain (odd k)
        Wk, Tk = W0, T0
        if k_case == 5:
            Wk = np.hstack([W0, W0[:, :1]])
            Tk = np.vstack([T0, T0[:1]])
        o = orc.nmf_oracle(X, k_case, Wk, Tk, max_iter=1, order='hals', project_T_each_iter=True, t_row_sum=1.0,
                           reg_t_l2=-10.0)
        g = R.nmf(X, k_case, W_in=Wk, T_in=Tk, max_iter=1, update_order='hals', project_T_each_iter=True,
                  t_row_sum=1.0, reg_t_l2=-10.0, reset_topic_method=None, do_final_project_W=False)
        assert np.all(np.count_nonzero(o['T'], axis=1) == 1)
        assert np.array_equal(g['T'], o['T'])


def test_tm_estimator_block_order(R):
    """NMF_TM_Estimator(update_order='hals'): fit, sweep-level resume (fit(2) + 8 x one_iter + final projection ==
    fit(10)), transform and reconstruction_err_"""
    X = golden('text_tm_f64.npz')['X']
    n, d = X.shape
    M = R.NMF_TM_Estimator(n, d, 6, random_state=0, max_iter=10, update_order='hals').fit(X)
    assert np.linalg.norm(X - np.dot(M.W, M.T), 'fro') < np.linalg.norm(X, 'fro')
    assert abs(M.reconstruction_err_ - np.linalg.norm(X - np.dot(M.W, M.T), 'fro')) < 1e-9
    _check_simplex(M.T, 1.0)
    M2 = R.NMF_TM_Estimator(n, d, 6, random_state=0, max_iter=2, do_final_project_W=False, update_order='hals').fit(X)
    M2.max_iter = 10
    for _ in range(8):
        M2 = M2.one_iter(X)
    M2.W = orc.proj_mat_to_simplex(M2.W)
    assert np.allclose(M2.T, M.T)
    assert np.allclose(M2.W, M.W)
    Wn = M.transform(X[:10])
    assert Wn.shape == (10, 6) and np.all(Wn >= 0)


@pytest.mark.parametrize('math', ['ieee', 'tf32'])
def test_tm_estimator_block_order_fp32(R, math):
    X = golden('text_tm_f64.npz')['X'].astype(np.float32)
    n, d = X.shape
    M = R.NMF_TM_Estimator(n, d, 8, random_state=0, max_iter=10, update_order='hals', math=math).fit(X)
    assert np.all(M.T >= 0) and np.max(np.abs(M.T.astype(np.float64).sum(1) - 1)) < 1e-5
    assert M.reconstruction_err_ < np.linalg.norm(X, 'fro')


@pytest.fixture(scope='module')
def cfg3_simplex(cuda_device):
    """config-3 shape (200000 x 20000, k = 64, fp32), topic-model-like: X = W T + noise with skewed rows of W and T on
    the simplex, and a start near them (uniform data empties topics under the constraint within a few sweeps)"""
    free, _ = torch.cuda.mem_get_info(cuda_device)
    if free < 60e9:
        pytest.skip('needs ~40 GB of device memory')
    n, d, k = 200000, 20000, 64
    g = torch.Generator(device=cuda_device)
    g.manual_seed(31)

    def rows(m, c, p):
        a = torch.rand(m, c, generator=g, device=cuda_device) ** p
        return a / a.sum(1, keepdim=True)
    Wt, Tt = rows(n, k, 8), rows(k, d, 20)
    X = Wt @ Tt
    X.add_(torch.rand(n, d, generator=g, device=cuda_device), alpha=0.05 * float(X.mean()))
    W0 = Wt + 0.2 * torch.rand(n, k, generator=g, device=cuda_device)
    W0 /= W0.sum(1, keepdim=True)
    T0 = Tt + 0.2 / d * torch.rand(k, d, generator=g, device=cuda_device)
    T0 /= T0.sum(1, keepdim=True)
    del Wt, Tt
    yield X, W0, T0
    del X, W0, T0
    torch.cuda.empty_cache()


def test_full_size_tf32_vs_ieee(R, cfg3_simplex):
    """config 3 (200000 x 20000, k = 64, fp32): the constrained block order in TF32 and IEEE arithmetic agree"""
    X, W0, T0 = cfg3_simplex
    err = {}
    for math in ('ieee', 'tf32'):
        eng = R.RRIEngine(X, 64, order='hals', math=math)
        W, T = W0.clone(), T0.clone()
        p = eng.params(ub_t=1.0, simplex_T=True)
        assert eng.sweeps(W, T, 3, p) == 0
        assert float(T.min()) >= 0.0 and float((T.double().sum(1) - 1).abs().max()) < 1e-4
        err[math] = eng.rel_error(W, T)
        eng.close()
    assert abs(err['tf32'] - err['ieee']) < 1e-4, err


@pytest.mark.parametrize('p2p', ['1', '0'])
def test_row_sharded_parity(cuda_device, p2p):
    """2 ranks: the constrained T half-step over the NCCL all-reduce, with the peer exchange mapped (1) or not (0)"""
    import subprocess
    import sys
    from conftest import ROOT
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    r = subprocess.run([sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2',
                        '--master-addr', '127.0.0.1', '--master-port', '2953%d' % int(p2p),
                        os.path.join(ROOT, 'tests', 'multi_gpu_simplex_check.py')], env=dict(os.environ, RRI_P2P=p2p),
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, universal_newlines=True, timeout=600)
    assert 'MULTI_GPU_SIMPLEX PASS' in r.stdout, r.stdout[-3000:]
