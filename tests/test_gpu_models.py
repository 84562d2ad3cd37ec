"""Several block-order models of one matrix on one binding (rri_set_models, RRIEngine(models=b), nmf_models): every
model against the oracle and against a handle of its own, per-model stopping and failure, re-entrance, groups."""
import numpy as np
import pytest
import torch

import rri_oracle as orc
from conftest import relfro

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def R(cuda_device):
    import rri_nmf_b200
    return rri_nmf_b200


def _starts(n, d, k, b, seed, dtype=np.float64):
    rs = np.random.RandomState(seed)
    return [rs.rand(n, k).astype(dtype) for _ in range(b)], [rs.rand(k, d).astype(dtype) for _ in range(b)]


def _stack(Ws, Ts, dev):
    return (torch.from_numpy(np.stack(Ws)).to(dev).contiguous(), torch.from_numpy(np.stack(Ts)).to(dev).contiguous())


REGS = [dict(), dict(reg_w_l1=0.01, reg_w_l2=0.02, reg_t_l1=0.03, reg_t_l2=0.04),
        dict(w_row_sum=2.0, t_row_sum=30.0)]


@pytest.mark.parametrize('kw', REGS)
def test_fp64_ieee_three_models_vs_oracle_and_own_handle(R, cuda_device, kw):
    """3 models of rank 8: after each of 3 sweeps every model is within 1e-9 of the oracle's block order from its own
    start and bit-identical to a handle of its own (regularisers, row-sum bounds)"""
    X, _, _ = orc.synth(300, 200, 6, 8, sigma=0.1, seed=4)
    Ws, Ts = _starts(300, 200, 8, 3, seed=5)
    Xd = torch.from_numpy(X).to(cuda_device)
    ub = dict(ub_w=kw.get('w_row_sum'), ub_t=kw.get('t_row_sum'))
    regs = {key: v for key, v in kw.items() if key.startswith('reg')}
    prm = R.RRIEngine.params(**regs, **ub)
    eng = R.RRIEngine(Xd, 8, order='hals', models=3)
    Wb, Tb = _stack(Ws, Ts, cuda_device)
    singles = [R.RRIEngine(Xd, 8, order='hals') for _ in range(3)]
    Wsd = [torch.from_numpy(w).to(cuda_device) for w in Ws]
    Tsd = [torch.from_numpy(t).to(cuda_device) for t in Ts]
    Wo, To = [w.copy() for w in Ws], [t.copy() for t in Ts]
    for _ in range(3):
        assert eng.sweeps(Wb, Tb, 1, prm) == [0, 0, 0]
        for m in range(3):
            singles[m].sweeps(Wsd[m], Tsd[m], 1, prm)
            orc.sweep(X, Wo[m], To[m], order='hals', **kw)
            assert torch.equal(Wb[m], Wsd[m]) and torch.equal(Tb[m], Tsd[m])
            assert relfro(Wb[m].cpu().numpy(), Wo[m]) < 1e-9
            assert relfro(Tb[m].cpu().numpy(), To[m]) < 1e-9
    sT, sW = eng.topic_sums()
    assert sT.shape == (3, 8) and np.allclose(sT[1], Tb[1].sum(1).cpu().numpy(), rtol=1e-12)
    for via in (False, True):
        v = eng.objective_terms(Wb, Tb, via_contraction=via)
        for m in range(3):
            assert np.array_equal(v[m], singles[m].objective_terms(Wsd[m], Tsd[m], via_contraction=via))


@pytest.mark.parametrize('math,dtype', [('ieee', np.float64), ('tf32', np.float32)])
def test_identical_starts_give_identical_models(R, cuda_device, math, dtype):
    X, _, _ = orc.synth(400, 300, 6, 16, sigma=0.1, seed=8, dtype=dtype)
    Ws, Ts = _starts(400, 300, 16, 2, seed=9, dtype=dtype)
    Wb, Tb = _stack([Ws[0], Ws[1], Ws[0]], [Ts[0], Ts[1], Ts[0]], cuda_device)
    eng = R.RRIEngine(torch.from_numpy(X).to(cuda_device), 16, order='hals', math=math, models=3)
    eng.sweeps(Wb, Tb, 5, R.RRIEngine.params())
    assert torch.equal(Wb[0], Wb[2]) and torch.equal(Tb[0], Tb[2])
    assert not torch.equal(Wb[0], Wb[1])


@pytest.mark.parametrize('x16', [True, False])
@pytest.mark.parametrize('k,b', [(32, 4), (64, 4), (16, 16)])
def test_tf32_widest_contraction_matches_own_handles(R, cuda_device, monkeypatch, x16, k, b):
    """b * k = 128 and 256 on the TF32 contraction (16-bit copies of X or fp32 storage): after 20 sweeps every model's
    relative error is within 1e-4 of a TF32 handle of its own (DESIGN.md §5)"""
    if not x16:
        monkeypatch.setenv('RRI_X16', '0')
    X, _, _ = orc.synth(3000, 1200, k, k, sigma=0.1, seed=11, dtype=np.float32)
    Ws, Ts = _starts(3000, 1200, k, b, seed=12, dtype=np.float32)
    Xd = torch.from_numpy(X).to(cuda_device)
    eng = R.RRIEngine(Xd, k, order='hals', math='tf32', models=b)
    assert eng.stats()['x_operand'] == ('f16' if x16 else 'f32')
    Wb, Tb = _stack(Ws, Ts, cuda_device)
    flags = eng.sweeps(Wb, Tb, 20, R.RRIEngine.params())
    assert flags == [0] * b
    errs = eng.rel_error(Wb, Tb)
    single = R.RRIEngine(Xd, k, order='hals', math='tf32')
    for m in range(b):
        W, T = torch.from_numpy(Ws[m]).to(cuda_device), torch.from_numpy(Ts[m]).to(cuda_device)
        single.sweeps(W, T, 20, R.RRIEngine.params())
        assert abs(errs[m] - single.rel_error(W, T)) < 1e-4


STOP = [dict(), dict(reg_w_l2=0.05, reg_t_l1=0.01, w_row_sum=1.0, project_W_each_iter=True, t_row_sum=50.0,
                     objective='exact')]


@pytest.mark.parametrize('kw', STOP)
def test_each_model_stops_as_its_own_nmf_call(R, kw):
    """fp64, compute_obj_each_iter, eps_stop: each model's obj_history, sweep count and factors equal its nmf() call"""
    X, _, _ = orc.synth(120, 90, 5, 6, sigma=0.2, seed=21)
    seeds = [3, 4, 5, 6]
    common = dict(init='random', compute_obj_each_iter=True, eps_stop=2e-3, max_iter=60, **kw)
    out = R.nmf_models(X, 6, random_state=seeds, **common)
    lens = set()
    for s, o in zip(seeds, out):
        ref = R.nmf(X, 6, random_state=s, update_order='hals', **common)
        assert 'error' not in o and o['random_state'] == s
        assert o['obj_history'] == ref['obj_history']
        assert len(o['iter_cputime']) == len(ref['iter_cputime'])
        assert np.array_equal(o['W'], ref['W']) and np.array_equal(o['T'], ref['T'])
        lens.add(len(o['obj_history']))
    assert len(lens) > 1                    # the models did stop at different sweeps


def _isolation_starts(n, d, k, dtype):
    Ws, Ts = _starts(n, d, k, 3, seed=31, dtype=dtype)
    Ws[1][:, 2] = 0                         # topic 2 of model 1 empties in its first T-step
    return Ws, Ts


def test_failed_model_leaves_the_others_bit_identical(R):
    X, _, _ = orc.synth(150, 110, 5, 7, sigma=0.1, seed=30)
    Ws, Ts = _isolation_starts(150, 110, 7, np.float64)
    out = R.nmf_models(X, 7, W_in=Ws, T_in=Ts, max_iter=12, update_order='hals')
    with pytest.raises(ValueError) as ref_err:
        R.nmf(X, 7, W_in=Ws[1], T_in=Ts[1], max_iter=12, update_order='hals')
    assert isinstance(out[1]['error'], ValueError) and 'W' not in out[1]
    assert str(out[1]['error']) == str(ref_err.value)
    for m in (0, 2):
        ref = R.nmf(X, 7, W_in=Ws[m], T_in=Ts[m], max_iter=12, update_order='hals')
        assert np.array_equal(out[m]['W'], ref['W']) and np.array_equal(out[m]['T'], ref['T'])


def test_failed_model_isolation_tf32_16bit(R, cuda_device):
    X, _, _ = orc.synth(2000, 900, 8, 16, sigma=0.1, seed=32, dtype=np.float32)
    Ws, Ts = _isolation_starts(2000, 900, 16, np.float32)
    out = R.nmf_models(X, 16, W_in=Ws, T_in=Ts, max_iter=20, math='tf32', sweeps_per_call=4)
    assert isinstance(out[1]['error'], ValueError)
    eng = R.RRIEngine(torch.from_numpy(X).to(cuda_device), 16, order='hals', math='tf32')
    assert eng.stats()['x_operand'] == 'f16'
    for m in (0, 2):
        ref = R.nmf(X, 16, W_in=Ws[m], T_in=Ts[m], max_iter=20, math='tf32', update_order='hals', sweeps_per_call=4)
        got = eng.rel_error(torch.from_numpy(out[m]['W']).to(cuda_device), torch.from_numpy(out[m]['T']).to(cuda_device))
        want = eng.rel_error(torch.from_numpy(ref['W']).to(cuda_device), torch.from_numpy(ref['T']).to(cuda_device))
        assert np.all(np.isfinite(out[m]['W'])) and abs(got - want) < 1e-4


@pytest.mark.parametrize('math,dtype', [('ieee', np.float64), ('ieee', np.float32), ('tf32', np.float32)])
def test_reentrant_on_a_models_handle(R, cuda_device, math, dtype):
    X, _, _ = orc.synth(500, 260, 6, 12, sigma=0.1, seed=40, dtype=dtype)
    Ws, Ts = _starts(500, 260, 12, 3, seed=41, dtype=dtype)
    eng = R.RRIEngine(torch.from_numpy(X).to(cuda_device), 12, order='hals', math=math, models=3)
    prm = R.RRIEngine.params(reg_w_l2=0.01)
    W1, T1 = _stack(Ws, Ts, cuda_device)
    W2, T2 = W1.clone(), T1.clone()
    eng.sweeps(W1, T1, 6, prm)
    for _ in range(6):
        eng.sweeps(W2, T2, 1, prm)
    assert torch.equal(W1, W2) and torch.equal(T1, T2)


def test_groups_above_the_cap_equal_separate_runs(R):
    """k = 100, 3 models: groups of 2 and 1 (rank 100 in fp64 takes the warp-per-row update)"""
    X, _, _ = orc.synth(400, 300, 100, 100, sigma=0.1, seed=50)
    Ws, Ts = _starts(400, 300, 100, 3, seed=51)
    out = R.nmf_models(X, 100, W_in=Ws, T_in=Ts, max_iter=3, reg_t_l2=0.1)
    fitted = 0
    for m in range(3):
        try:
            ref = R.nmf(X, 100, W_in=Ws[m], T_in=Ts[m], max_iter=3, reg_t_l2=0.1, update_order='hals')
        except ValueError as ex:            # (an emptied topic fails the model in both)
            assert str(out[m]['error']) == str(ex)
            continue
        assert np.array_equal(out[m]['W'], ref['W']) and np.array_equal(out[m]['T'], ref['T'])
        fitted += 1
    assert fitted >= 2


def test_device_initialisation_per_model(R, cuda_device):
    """starts made on the device (X is a CUDA tensor) through the models engine's contraction equal nmf()'s"""
    X, _, _ = orc.synth(300, 140, 6, 5, sigma=0.1, seed=60)
    Xd = torch.from_numpy(X).to(cuda_device)
    out = R.nmf_models(Xd, 5, random_state=[1, 2], init='nndsvdar', max_iter=4)
    for s, o in zip([1, 2], out):
        ref = R.nmf(Xd, 5, random_state=s, init='nndsvdar', max_iter=4, update_order='hals')
        assert torch.equal(o['W'], ref['W']) and torch.equal(o['T'], ref['T'])


def test_models_handle_refusals(R, cuda_device):
    import ctypes as C
    from rri_nmf_b200 import _lib
    X = torch.rand(50, 40, dtype=torch.float64, device=cuda_device)
    with pytest.raises(_lib.RriError):
        R.RRIEngine(X, 6, order='rri', models=2)
    with pytest.raises(_lib.RriError):
        R.RRIEngine(X, 6, order='hals', models=2, W_mat=torch.ones_like(X))
    with pytest.raises(_lib.RriError):
        R.RRIEngine(X.to_sparse_csr(), 6, order='hals', models=2, unstored='zero')
    eng = R.RRIEngine(X, 6, order='hals', models=2)
    W, T = torch.rand(2, 50, 6, dtype=torch.float64, device=cuda_device), torch.rand(2, 6, 40, dtype=torch.float64, device=cuda_device)
    with pytest.raises(_lib.RriError):
        eng.sweeps(W, T, 1, R.RRIEngine.params(ub_t=1.0, simplex_T=True))
    wR = torch.empty(40, dtype=torch.float64, device=cuda_device)
    assert eng.lib.rri_partials_T(eng.h, C.c_void_p(W.data_ptr()), C.c_void_p(T.data_ptr()), 0,
                                  C.c_void_p(wR.data_ptr()), C.c_void_p(wR.data_ptr()), eng._stream()) != 0
    h = C.c_void_p()
    _lib.check(eng.lib.rri_create(C.byref(h), 50, 40, 6, 1, 0, 1, cuda_device.index or 0))
    try:
        assert eng.lib.rri_set_models(h, 4) != 0          # 6 % 4 != 0
        assert eng.lib.rri_set_models(h, 3) == 0
    finally:
        eng.lib.rri_destroy(h)
