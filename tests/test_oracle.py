"""The NumPy oracle against the golden vectors produced by the unmodified reference
(oracle/make_golden.py) and -- when the reference is present -- against the live reference."""
import numpy as np
import pytest

import rri_oracle as orc
import refshim
from conftest import golden, relfro

TOL = 1e-11     # restatement vs reference: same arithmetic, BLAS summation order may differ


def test_eps_constant():
    # nmf.py:52 / optimization.py:5
    assert orc.EPS_DIV_BY_ZERO == 1.7763568394002505e-15


def test_cfg1_rri_snapshots_and_objective():
    g = golden('cfg1_rri_f64.npz')
    X, W0, T0 = orc.synth(500, 300, 10, 10, sigma=0.0, seed=0)
    assert np.allclose([X.sum(), (X ** 2).sum()], g['x_checksum'], rtol=1e-14)
    out = orc.nmf_oracle(X, 10, W0, T0, max_iter=200, compute_obj_each_iter=True, eps_stop=-1.0,
                         snapshots=set(int(c) for c in g['counts']))
    for c in g['counts']:
        W, T = out['snapshots'][int(c)]
        assert relfro(W, g['W_%d' % c]) < TOL, c
        assert relfro(T, g['T_%d' % c]) < TOL, c
    assert np.allclose(out['obj_history'], g['obj_history'], rtol=1e-10)
    assert np.all(np.diff(out['obj_history']) <= 0)      # tests/test_nmf.py:40


def test_cfg1_hals_block_order():
    g = golden('cfg1_hals_f64.npz')
    X, W0, T0 = orc.synth(500, 300, 10, 10, sigma=0.0, seed=0)
    out = orc.nmf_oracle(X, 10, W0, T0, max_iter=50, order='hals',
                         snapshots=set(int(c) for c in g['counts']))
    for c in g['counts']:
        W, T = out['snapshots'][int(c)]
        assert relfro(W, g['W_%d' % c]) < TOL
        assert relfro(T, g['T_%d' % c]) < TOL
    # the two orders are genuinely different iterations (SURVEY.md F2)
    gr = golden('cfg1_rri_f64.npz')
    assert relfro(g['W_10'], gr['W_10']) > 1e-4


def test_cfg1_fp32_inputs_stay_fp32():
    g = golden('cfg1_rri_f32.npz')
    X, W0, T0 = orc.synth(500, 300, 10, 10, sigma=0.0, seed=0, dtype=np.float32)
    out = orc.nmf_oracle(X, 10, W0, T0, max_iter=10)
    assert out['W'].dtype == np.float32
    assert relfro(out['W'], g['W_10']) < 1e-4
    re = orc.rel_error(X.astype(np.float64), out['W'].astype(np.float64), out['T'].astype(np.float64))
    assert abs(re - float(g['relerr_10'])) < 1e-6


def test_regularised():
    g = golden('reg_rri_f64.npz')
    X, W0, T0 = orc.synth(257, 131, 6, 7, sigma=0.05, seed=3)
    rw1, rw2, rt1, rt2 = g['regs']
    out = orc.nmf_oracle(X, 7, W0, T0, max_iter=6, compute_obj_each_iter=True, eps_stop=-1.0,
                         reg_w_l1=rw1, reg_w_l2=rw2, reg_t_l1=rt1, reg_t_l2=rt2)
    assert relfro(out['W'], g['W']) < TOL
    assert relfro(out['T'], g['T']) < TOL
    assert np.allclose(out['obj_history'], g['obj_history'], rtol=1e-11)


def test_row_partials_add_up():
    """nmf.py:680-686: the row-subset statistic; partials over disjoint shards sum to the full one."""
    g = golden('partials_f64.npz')
    X, W0, T0 = orc.synth(257, 131, 6, 7, sigma=0.05, seed=3)
    s = int(g['split'][0])
    for t in (0, 3, 6):
        wa, na = orc.update_T_stats(X, W0, T0, t, rows=np.arange(0, s))
        wb, nb = orc.update_T_stats(X, W0, T0, t, rows=np.arange(s, 257))
        wf, nf = orc.update_T_stats(X, W0, T0, t)
        assert relfro(wa, g['numer_a_%d' % t]) < 1e-13
        assert relfro(wb, g['numer_b_%d' % t]) < 1e-13
        assert relfro(wf, g['numer_full_%d' % t]) < 1e-13
        assert abs(na - g['denom_a_%d' % t]) < 1e-12 and abs(nb - g['denom_b_%d' % t]) < 1e-12
        assert relfro(wa + wb, wf) < 1e-13 and abs(na + nb - nf) < 1e-12


def test_fix_T_is_clean_block_W_update():
    g = golden('fixT_f64.npz')
    X, W0, T0 = orc.synth(257, 131, 6, 7, sigma=0.05, seed=3)
    out = orc.nmf_oracle(X, 7, W0, T0, max_iter=4, fix_T=True)
    assert relfro(out['W'], g['W']) < TOL
    assert np.array_equal(out['T'], g['T'])


@pytest.mark.parametrize('name,regs', [('plain', {}), ('l1both', {'reg_w_l1': 0.1, 'reg_t_l1': 0.1}),
                                        ('l1w', {'reg_w_l1': 0.1}), ('l1t', {'reg_t_l1': 0.1})])
def test_recsys_masked_wrri(name, regs):
    g = golden('recsys_wrri_f64.npz')
    X = g['X']
    M = (X != 0).astype(np.float64)
    out = orc.nmf_oracle(X, 7, g['W0'], g['T0'], max_iter=15, W_mat=M, compute_obj_each_iter=True,
                         eps_stop=-1.0, t_row_sum=1.0, **regs)
    assert relfro(out['W'], g['W_' + name]) < 1e-10
    assert relfro(out['T'], g['T_' + name]) < 1e-10
    assert np.allclose(out['obj_history'], g['obj_' + name], rtol=1e-10)
    assert np.all(np.diff(out['obj_history']) <= 1e-9)   # tests/test_nmf.py:78
    assert out['T'].max() <= 1.0                           # ub clip, optimization.py:82-83


def test_weighted_wrri_real_weights():
    g = golden('weighted_wrri_f64.npz')
    X, W0, T0, Mb = orc.synth(120, 90, 5, 6, sigma=0.05, seed=5, mask_density=0.3)
    Mw = Mb * np.random.RandomState(9).rand(120, 90) * 2.0
    out = orc.nmf_oracle(X, 6, W0, T0, max_iter=8, W_mat=Mw, compute_obj_each_iter=True, eps_stop=-1.0)
    assert relfro(out['W'], g['W']) < 1e-10 and relfro(out['T'], g['T']) < 1e-10
    assert np.allclose(out['obj_history'], g['obj_history'], rtol=1e-10)
    gh = golden('weighted_wrri_hals_f64.npz')
    out = orc.nmf_oracle(X, 6, W0, T0, max_iter=5, W_mat=Mw, order='hals')
    assert relfro(out['W'], gh['W']) < 1e-10 and relfro(out['T'], gh['T']) < 1e-10


def test_text_topic_model_simplex():
    g = golden('text_tm_f64.npz')
    X = g['X']
    out = orc.nmf_oracle(X, 15, g['W0'], g['T0'], max_iter=15, w_row_sum=1.0, project_T_each_iter=True,
                         project_W_each_iter=True, compute_obj_each_iter=True, eps_stop=-1.0,
                         t_row_sum=1.0, reg_t_l2=0.1)
    assert relfro(out['W'], g['W_tm']) < 1e-10 and relfro(out['T'], g['T_tm']) < 1e-10
    assert np.allclose(out['obj_history'], g['obj_tm'], rtol=1e-10)
    # tests/test_nmf.py:41-54: constraint violation
    cv = np.sum(np.abs(out['W'].sum(1) - 1)) + np.sum(np.abs(out['T'].sum(1) - 1))
    assert cv <= 1e-13 * 10
    out = orc.nmf_oracle(X, 15, g['W0'], g['T0'], max_iter=10, w_row_sum=1.0, project_T_each_iter=True,
                         t_row_sum=1.0)
    assert relfro(out['W'], g['W_est']) < 1e-10 and relfro(out['T'], g['T_est']) < 1e-10


# ------------------------------------------------------------------ cases run against the live reference
# The reference sources are not part of the repository.  tests/golden/live_cases_f64.npz pins what the oracle returns
# on these inputs (oracle/make_golden.py live-pins), so every checkout checks them; with the reference present
# (RRI_REFERENCE_ROOT) the tests also compare with it directly, at the same tolerances.


@pytest.mark.parametrize('n,d,k,masked', [(64, 40, 5, False), (33, 57, 4, False), (40, 30, 4, True)])
def test_live_reference_random(n, d, k, masked):
    rs = np.random.RandomState(n + d)
    X, W0, T0 = rs.rand(n, d), rs.rand(n, k), rs.rand(k, d)
    M = (rs.rand(n, d) < 0.4).astype(float) if masked else None
    o = orc.nmf_oracle(X, k, W0, T0, max_iter=5, W_mat=M, compute_obj_each_iter=True, eps_stop=-1.0)
    g = golden('live_cases_f64.npz')
    key = '%d_%d_%d_%d' % (n, d, k, masked)
    expected = [(g['W_' + key], g['T_' + key], g['obj_' + key])]
    if refshim.available():
        r = refshim.load().nmf.nmf(X, k, W_in=W0, T_in=T0, max_iter=5, W_mat=M, reset_topic_method=None,
                                   compute_obj_each_iter=True, eps_stop=-1.0)
        expected.append((r['W'], r['T'], r['obj_history']))
    for W, T, obj in expected:
        assert relfro(o['W'], W) < TOL and relfro(o['T'], T) < TOL
        assert np.allclose(o['obj_history'], obj, rtol=1e-11)


def test_live_reference_stopping_rule():
    rs = np.random.RandomState(1)
    X, W0, T0 = rs.rand(60, 50), rs.rand(60, 4), rs.rand(4, 50)
    o = orc.nmf_oracle(X, 4, W0, T0, max_iter=200, compute_obj_each_iter=True, eps_stop=1e-3)
    assert len(o['obj_history']) == int(golden('live_cases_f64.npz')['stop_len'][0]) < 200
    if refshim.available():
        r = refshim.load().nmf.nmf(X, 4, W_in=W0, T_in=T0, max_iter=200, reset_topic_method=None,
                                   compute_obj_each_iter=True, eps_stop=1e-3)
        assert len(o['obj_history']) == len(r['obj_history'])


def test_live_reference_zero_topic_raises():
    """A topic that collapses to zero with resets disabled: the T row is all-zero -> nt = 0 ->
    the W-step takes qf_min's c<=0 branch without bounds and raises (optimization.py:60-67,105-107)."""
    rs = np.random.RandomState(33 + 57)
    X, W0, T0 = rs.rand(33, 57), rs.rand(33, 8), rs.rand(8, 57)
    with pytest.raises(ValueError):
        orc.nmf_oracle(X, 8, W0, T0, max_iter=5)
    if refshim.available():
        with pytest.raises(ValueError):
            refshim.load().nmf.nmf(X, 8, W_in=W0, T_in=T0, max_iter=5, reset_topic_method=None)
