"""Models of different ranks of one matrix on one binding (rri_set_model_ranks, RRIEngine(X, [k_0, ...]),
nmf_models(X, [k_0, ...])): every model against a handle of its own and the oracle, equal ranks against models=b,
per-model stopping, failure, grouping, device starts, re-entrance and the refusals."""
import ctypes as C

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


def _starts(n, d, ranks, seed, dtype=np.float64):
    rs = np.random.RandomState(seed)
    return [rs.rand(n, k).astype(dtype) for k in ranks], [rs.rand(k, d).astype(dtype) for k in ranks]


def _dev(arrays, dev):
    return [torch.from_numpy(a).to(dev) for a in arrays]


REGS = [dict(), dict(reg_w_l1=0.01, reg_w_l2=0.02, reg_t_l1=0.03, reg_t_l2=0.04),
        dict(w_row_sum=2.0, t_row_sum=30.0)]


@pytest.mark.parametrize('kw', REGS)
def test_fp64_ieee_mixed_ranks_vs_oracle_and_own_handles(R, cuda_device, kw):
    """ranks 3, 8, 5, 16 (offsets 0, 3, 11, 16: aligned and unaligned blocks): after each of 3 sweeps every model is
    bit-identical to a handle of its own and within 1e-9 of the oracle's block order (data of true rank 16: no topic
    of any model empties on the oracle)"""
    ranks = (3, 8, 5, 16)
    X, _, _ = orc.synth(300, 200, 16, 16, sigma=0.1, seed=4)
    Ws, Ts = _starts(300, 200, ranks, seed=5)
    Xd = torch.from_numpy(X).to(cuda_device)
    ub = dict(ub_w=kw.get('w_row_sum'), ub_t=kw.get('t_row_sum'))
    regs = {key: v for key, v in kw.items() if key.startswith('reg')}
    prm = R.RRIEngine.params(**regs, **ub)
    eng = R.RRIEngine(Xd, list(ranks), order='hals')
    W, T = eng.pack(_dev(Ws, cuda_device), _dev(Ts, cuda_device))
    Wv, Tv = eng.views(W, T)
    singles = [R.RRIEngine(Xd, k, order='hals') for k in ranks]
    Wsd, Tsd = _dev(Ws, cuda_device), _dev(Ts, cuda_device)
    Wo, To = [w.copy() for w in Ws], [t.copy() for t in Ts]
    for _ in range(3):
        assert eng.sweeps(W, T, 1, prm) == [0] * 4
        for m in range(4):
            singles[m].sweeps(Wsd[m], Tsd[m], 1, prm)
            orc.sweep(X, Wo[m], To[m], order='hals', **kw)
            assert torch.equal(Wv[m], Wsd[m]) and torch.equal(Tv[m], Tsd[m])
            assert relfro(Wv[m].cpu().numpy(), Wo[m]) < 1e-9
            assert relfro(Tv[m].cpu().numpy(), To[m]) < 1e-9
    sT, sW = eng.topic_sums()
    for m in range(4):
        oT, oW = singles[m].topic_sums()
        assert np.array_equal(sT[m], oT) and np.array_equal(sW[m], oW)
    for via in (False, True):
        v = eng.objective_terms(W, T, via_contraction=via)
        assert v.shape == (4, 6)
        for m in range(4):
            assert np.array_equal(v[m], singles[m].objective_terms(Wsd[m], Tsd[m], via_contraction=via))
    assert len(eng.rel_error(W, T)) == 4


def test_fp32_ieee_mixed_ranks_bit_identical(R, cuda_device):
    ranks = (4, 12, 7)
    X, _, _ = orc.synth(400, 260, 6, 8, sigma=0.1, seed=6, dtype=np.float32)
    Ws, Ts = _starts(400, 260, ranks, seed=7, dtype=np.float32)
    Xd = torch.from_numpy(X).to(cuda_device)
    eng = R.RRIEngine(Xd, list(ranks), order='hals')
    W, T = eng.pack(_dev(Ws, cuda_device), _dev(Ts, cuda_device))
    Wv, Tv = eng.views(W, T)
    prm = R.RRIEngine.params(reg_w_l2=0.01)
    eng.sweeps(W, T, 4, prm)
    for m, k in enumerate(ranks):
        Wm, Tm = torch.from_numpy(Ws[m]).to(cuda_device), torch.from_numpy(Ts[m]).to(cuda_device)
        R.RRIEngine(Xd, k, order='hals').sweeps(Wm, Tm, 4, prm)
        assert torch.equal(Wv[m], Wm) and torch.equal(Tv[m], Tm)


@pytest.mark.parametrize('x16', [True, False])
@pytest.mark.parametrize('ranks', [tuple(range(2, 21)), (128, 64, 32, 16, 16)])
def test_tf32_rank_sweep_matches_own_handles(R, cuda_device, monkeypatch, x16, ranks):
    """total widths 209 and 256 on the TF32 contraction (16-bit copies of X or fp32 storage): after 20 sweeps every
    model keeps all its topics and its relative error is within 1e-4 of a TF32 handle of its own (data of true rank
    128: on the oracle no topic of any of these ranks empties in 20 sweeps)"""
    if not x16:
        monkeypatch.setenv('RRI_X16', '0')
    X, _, _ = orc.synth(3000, 1200, 128, 128, sigma=0.1, seed=11, dtype=np.float32)
    Ws, Ts = _starts(3000, 1200, ranks, seed=12, dtype=np.float32)
    Xd = torch.from_numpy(X).to(cuda_device)
    eng = R.RRIEngine(Xd, list(ranks), order='hals', math='tf32')
    assert eng.stats()['x_operand'] == ('f16' if x16 else 'f32')
    W, T = eng.pack(_dev(Ws, cuda_device), _dev(Ts, cuda_device))
    assert eng.sweeps(W, T, 20, R.RRIEngine.params(reg_t_l2=0.01)) == [0] * len(ranks)
    errs = eng.rel_error(W, T)
    for m, k in enumerate(ranks):
        single = R.RRIEngine(Xd, k, order='hals', math='tf32')
        Wm, Tm = torch.from_numpy(Ws[m]).to(cuda_device), torch.from_numpy(Ts[m]).to(cuda_device)
        assert single.sweeps(Wm, Tm, 20, R.RRIEngine.params(reg_t_l2=0.01)) == 0
        assert abs(errs[m] - single.rel_error(Wm, Tm)) < 1e-4


@pytest.mark.parametrize('dtype', [np.float64, np.float32])
def test_unaligned_models_take_the_staged_update_with_the_same_bits(R, cuda_device, dtype):
    """120 x 100: both IEEE contractions run as one K-slice (<= 128 K-elements per slice), so a single handle of an
    even (fp64) / multiple-of-4 (fp32) rank takes the register-resident update.  Ranks 3, 8, 4, 12: the models of
    ranks 8 and 12 start at offsets 3 and 15, off the 16-byte boundary, and take the staged update; every model must
    still be bit-identical to its own handle."""
    ranks = (3, 8, 4, 12)
    X, _, _ = orc.synth(120, 100, 12, 12, sigma=0.1, seed=70, dtype=dtype)
    Ws, Ts = _starts(120, 100, ranks, seed=71, dtype=dtype)
    Xd = torch.from_numpy(X).to(cuda_device)
    eng = R.RRIEngine(Xd, list(ranks), order='hals')
    W, T = eng.pack(_dev(Ws, cuda_device), _dev(Ts, cuda_device))
    Wv, Tv = eng.views(W, T)
    prm = R.RRIEngine.params(reg_t_l2=0.01)
    assert eng.sweeps(W, T, 5, prm) == [0] * 4
    for m, k in enumerate(ranks):
        Wm, Tm = torch.from_numpy(Ws[m]).to(cuda_device), torch.from_numpy(Ts[m]).to(cuda_device)
        assert R.RRIEngine(Xd, k, order='hals').sweeps(Wm, Tm, 5, prm) == 0
        assert torch.equal(Wv[m], Wm) and torch.equal(Tv[m], Tm)


@pytest.mark.parametrize('math,dtype', [('ieee', np.float64), ('tf32', np.float32)])
def test_equal_ranks_as_a_sequence_equal_models(R, cuda_device, math, dtype):
    X, _, _ = orc.synth(500, 300, 6, 16, sigma=0.1, seed=13, dtype=dtype)
    Ws, Ts = _starts(500, 300, (16,) * 4, seed=14, dtype=dtype)
    Xd = torch.from_numpy(X).to(cuda_device)
    er = R.RRIEngine(Xd, [16] * 4, order='hals', math=math)
    em = R.RRIEngine(Xd, 16, order='hals', math=math, models=4)
    W1, T1 = er.pack(_dev(Ws, cuda_device), _dev(Ts, cuda_device))
    W2 = torch.from_numpy(np.stack(Ws)).to(cuda_device).contiguous()
    T2 = torch.from_numpy(np.stack(Ts)).to(cuda_device).contiguous()
    er.sweeps(W1, T1, 5, R.RRIEngine.params())
    em.sweeps(W2, T2, 5, R.RRIEngine.params())
    assert torch.equal(W1, W2.reshape(-1)) and torch.equal(T1, T2.reshape(64, 300))


def test_each_rank_stops_as_its_own_nmf_call(R):
    X, _, _ = orc.synth(120, 90, 5, 6, sigma=0.2, seed=21)
    ranks, seeds = [4, 6, 9, 5], [3, 4, 5, 6]
    common = dict(init='random', compute_obj_each_iter=True, eps_stop=2e-3, max_iter=60)
    out = R.nmf_models(X, ranks, random_state=seeds, **common)
    lens = set()
    for k, s, o in zip(ranks, seeds, out):
        ref = R.nmf(X, k, random_state=s, update_order='hals', **common)
        assert 'error' not in o and o['W'].shape == (120, k)
        assert o['obj_history'] == ref['obj_history']
        assert len(o['iter_cputime']) == len(ref['iter_cputime'])
        assert np.array_equal(o['W'], ref['W']) and np.array_equal(o['T'], ref['T'])
        lens.add(len(o['obj_history']))
    assert len(lens) > 1


def test_failed_rank_leaves_the_others_bit_identical(R):
    ranks = [5, 7, 4]
    X, _, _ = orc.synth(150, 110, 5, 7, sigma=0.1, seed=30)
    Ws, Ts = _starts(150, 110, ranks, seed=31)
    Ws[1][:, 2] = 0                         # topic 2 of model 1 empties in its first T-step
    out = R.nmf_models(X, ranks, W_in=Ws, T_in=Ts, max_iter=12)
    with pytest.raises(ValueError) as ref_err:
        R.nmf(X, 7, W_in=Ws[1], T_in=Ts[1], max_iter=12, update_order='hals')
    assert isinstance(out[1]['error'], ValueError) and str(out[1]['error']) == str(ref_err.value)
    for m in (0, 2):
        ref = R.nmf(X, ranks[m], W_in=Ws[m], T_in=Ts[m], max_iter=12, update_order='hals')
        assert np.array_equal(out[m]['W'], ref['W']) and np.array_equal(out[m]['T'], ref['T'])


def test_rank_groups_equal_separate_runs(R):
    """ranks 200, 100, 50, 150: groups {200, 50} and {100, 150}; results in caller order (on the oracle ranks 200 and
    150, one of each group, keep all their topics; the others fail as their own nmf() calls do)"""
    ranks = [200, 100, 50, 150]
    X, _, _ = orc.synth(600, 400, 250, 250, sigma=0.1, seed=50)
    Ws, Ts = _starts(600, 400, ranks, seed=51)
    out = R.nmf_models(X, ranks, W_in=Ws, T_in=Ts, max_iter=3, reg_t_l2=0.1)
    fitted = 0
    for m, k in enumerate(ranks):
        try:
            ref = R.nmf(X, k, W_in=Ws[m], T_in=Ts[m], max_iter=3, reg_t_l2=0.1, update_order='hals')
        except ValueError as ex:
            assert str(out[m]['error']) == str(ex)
            continue
        assert np.array_equal(out[m]['W'], ref['W']) and np.array_equal(out[m]['T'], ref['T'])
        fitted += 1
    assert fitted >= 2


def test_device_initialisation_per_rank(R, cuda_device):
    X, _, _ = orc.synth(300, 140, 6, 5, sigma=0.1, seed=60)
    Xd = torch.from_numpy(X).to(cuda_device)
    out = R.nmf_models(Xd, [5, 3], random_state=[1, 2], init='nndsvdar', max_iter=4)
    for k, s, o in zip([5, 3], [1, 2], out):
        ref = R.nmf(Xd, k, random_state=s, init='nndsvdar', max_iter=4, update_order='hals')
        assert torch.equal(o['W'], ref['W']) and torch.equal(o['T'], ref['T'])


@pytest.mark.parametrize('math,dtype', [('ieee', np.float64), ('ieee', np.float32), ('tf32', np.float32)])
def test_reentrant_on_a_ranks_handle(R, cuda_device, math, dtype):
    ranks = [3, 12, 6]
    X, _, _ = orc.synth(500, 260, 6, 12, sigma=0.1, seed=40, dtype=dtype)
    Ws, Ts = _starts(500, 260, ranks, seed=41, dtype=dtype)
    eng = R.RRIEngine(torch.from_numpy(X).to(cuda_device), ranks, order='hals', math=math)
    prm = R.RRIEngine.params(reg_w_l2=0.01)
    W1, T1 = eng.pack(_dev(Ws, cuda_device), _dev(Ts, cuda_device))
    W2, T2 = W1.clone(), T1.clone()
    eng.sweeps(W1, T1, 6, prm)
    for _ in range(6):
        eng.sweeps(W2, T2, 1, prm)
    assert torch.equal(W1, W2) and torch.equal(T1, T2)


def test_ranks_handle_refusals(R, cuda_device):
    from rri_nmf_b200 import _lib
    X = torch.rand(50, 40, dtype=torch.float64, device=cuda_device)
    with pytest.raises(_lib.RriError):
        R.RRIEngine(X, [2, 4], order='rri')
    with pytest.raises(_lib.RriError):
        R.RRIEngine(X, [2, 4], order='hals', W_mat=torch.ones_like(X))
    with pytest.raises(_lib.RriError):
        R.RRIEngine(X.to_sparse_csr(), [2, 4], order='hals', unstored='zero')
    eng = R.RRIEngine(X, [2, 4], order='hals')
    W, T = eng.pack([torch.rand(50, 2, dtype=torch.float64, device=cuda_device),
                     torch.rand(50, 4, dtype=torch.float64, device=cuda_device)],
                    [torch.rand(2, 40, dtype=torch.float64, device=cuda_device),
                     torch.rand(4, 40, dtype=torch.float64, device=cuda_device)])
    with pytest.raises(_lib.RriError):
        eng.sweeps(W, T, 1, R.RRIEngine.params(ub_t=1.0, simplex_T=True))
    wR = torch.empty(40, dtype=torch.float64, device=cuda_device)
    assert eng.lib.rri_partials_T(eng.h, C.c_void_p(W.data_ptr()), C.c_void_p(T.data_ptr()), 0,
                                  C.c_void_p(wR.data_ptr()), C.c_void_p(wR.data_ptr()), eng._stream()) != 0
    h = C.c_void_p()
    _lib.check(eng.lib.rri_create(C.byref(h), 50, 40, 6, 1, 0, 1, cuda_device.index or 0))
    try:
        assert eng.lib.rri_set_model_ranks(h, 2, (C.c_int32 * 2)(2, 3)) != 0      # 2 + 3 != 6
        assert eng.lib.rri_set_model_ranks(h, 3, (C.c_int32 * 3)(2, 0, 4)) != 0   # a rank of 0
        assert eng.lib.rri_set_model_ranks(h, 2, (C.c_int32 * 2)(2, 4)) == 0
    finally:
        eng.lib.rri_destroy(h)
