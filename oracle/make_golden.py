"""Generate tests/golden/*.npz by running the UNMODIFIED reference (via oracle/refshim.py).

TEST INFRASTRUCTURE ONLY.  Run in the build container (needs /root/reference):

    python oracle/make_golden.py

(`python oracle/make_golden.py live-pins` writes the one file that does not come from the reference: see
live_case_pins.)

All cases pass explicit W_in/T_in (so sklearn's randomized_svd stream is not part of the
golden), `reset_topic_method=None`, logger at WARNING (SURVEY.md F4).  Inputs are stored in the
file when they are not reproducible from a NumPy RandomState seed.
"""
import os
import sys

import numpy as np
import scipy.sparse

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import refshim            # noqa: E402
import rri_oracle as orc  # noqa: E402

OUT = os.path.join(HERE, '..', 'tests', 'golden')
REF_DATA = os.path.join(refshim.REF_ROOT, 'tests', 'data')


def ref_nmf(ref, X, k, W0, T0, **kw):
    kw.setdefault('reset_topic_method', None)
    kw.setdefault('max_time', 1e9)
    kw.setdefault('eps_stop', -1.0)      # never stop on the objective: we want all sweeps
    return ref.nmf.nmf(X, k, W_in=W0, T_in=T0, **kw)


def snapshots(ref, X, k, W0, T0, counts, **kw):
    """Reference state after each sweep count in `counts` (re-entrant driver: N sweeps from
    the inputs; the reference copies W_in/T_in, nmf.py:867-868)."""
    out = {}
    W, T = W0, T0
    done = 0
    for c in sorted(counts):
        r = ref_nmf(ref, X, k, W, T, max_iter=c - done, **kw)
        W, T = r['W'], r['T']
        done = c
        out[c] = (W.copy(), T.copy())
    return out


def ref_block_sweep(ref, X, W, T, M=None, **regs):
    """The reference's own _compute_update_T/_compute_update_W/qf_min driven in BLOCK order
    (all T-steps, then all W-steps) -- the oracle for update_order='hals' (SURVEY.md F2, F5)."""
    k = W.shape[1]
    n, d = X.shape
    for t in range(k):
        wR, nw, _, _ = ref.nmf._compute_update_T(X=X, W=W, T=T, t=t, store_gradients=False,
                                                 ind_rows_to_store=None, W_mat=M)
        T[t, :], _ = ref.optimization.qf_min(-(wR - regs.get('reg_t_l1', 0)),
                                             nw + regs.get('reg_t_l2', 0), s=None,
                                             ub=regs.get('t_row_sum'))
    for t in range(k):
        Rt, nt = ref.nmf._compute_update_W(X=X, W=W, T=T, W_mat=M, t=t)
        W[:, t], _ = ref.optimization.qf_min(-(Rt - regs.get('reg_w_l1', 0)),
                                             nt + regs.get('reg_w_l2', 0), s=None,
                                             ub=regs.get('w_row_sum'))


def make_fix_W(ref):
    """fix_W=True: T-only sweeps in which, without regularisation, the reference also rescales W[:, t] by the
    T-step's sum (nmf.py:450-452, SURVEY.md F5) -- unmasked / simplex-constrained / regularised / masked."""
    X, W0, T0, M = orc.synth(120, 80, 5, 6, sigma=0.05, seed=13, mask_density=0.4)
    d = {}
    cases = (('plain', {}), ('simplex', dict(project_T_each_iter=True, t_row_sum=1.0)),
             ('reg', dict(reg_t_l1=0.01, reg_t_l2=0.05)), ('masked', dict(W_mat=M)),
             ('masked_ub', dict(W_mat=M, t_row_sum=1.0)))
    for name, kw in cases:
        r = ref_nmf(ref, X, 6, W0, T0, max_iter=3, fix_W=True, **kw)
        d['W_' + name], d['T_' + name] = r['W'], r['T']
    np.savez_compressed(os.path.join(OUT, 'fixW_f64.npz'), **d)


def estimator_goldens(ref, Xr):
    """The reference's recommender estimator on its own fixture (tests/test_nmf.py:81-88): NNDSVD init, 5 % validation
    split, validation-RMSE early stop (it stops after 2 sweeps and reverts to the state after the first).  Depends on
    sklearn's randomized_svd and train_test_split, like the replay scalars."""
    n, d = Xr.shape
    E = ref.sklearn_interface.NMF_RS_Estimator(n, d, 5, random_state=0, max_iter=20)
    E = E.fit_from_Xtr(scipy.sparse.csr_matrix(Xr))
    np.savez_compressed(os.path.join(OUT, 'rs_estimator_f64.npz'), W=E.W, T=E.T,
                        obj_history=np.array(E.nmf_outputs['obj_history']), score=np.array([E.score(Xr)]))


def main():
    ref = refshim.load()
    os.makedirs(OUT, exist_ok=True)
    make_fix_W(ref)
    if len(sys.argv) > 1 and sys.argv[1] == 'fixW':
        return

    # ---------------------------------------------------------------- cfg1: 500x300 k=10 fp64
    X, W0, T0 = orc.synth(500, 300, 10, 10, sigma=0.0, seed=0)
    counts = [1, 2, 10, 200]
    snaps = snapshots(ref, X, 10, W0, T0, counts)
    r = ref_nmf(ref, X, 10, W0, T0, max_iter=200, compute_obj_each_iter=True)
    assert np.array_equal(r['W'], snaps[200][0])
    d = {'counts': np.array(counts), 'obj_history': np.array(r['obj_history']),
         'x_checksum': np.array([X.sum(), (X ** 2).sum()])}
    for c in counts:
        d['W_%d' % c], d['T_%d' % c] = snaps[c]
    np.savez_compressed(os.path.join(OUT, 'cfg1_rri_f64.npz'), **d)

    # block order on the same inputs
    W, T = np.maximum(W0, 0), np.maximum(T0, 0)
    d = {'counts': np.array([1, 2, 10, 50])}
    for s in range(1, 51):
        ref_block_sweep(ref, X, W, T)
        if s in (1, 2, 10, 50):
            d['W_%d' % s], d['T_%d' % s] = W.copy(), T.copy()
    np.savez_compressed(os.path.join(OUT, 'cfg1_hals_f64.npz'), **d)

    # fp32 inputs straight through the reference (result dtype float32, SURVEY.md C.4)
    Xf, W0f, T0f = X.astype(np.float32), W0.astype(np.float32), T0.astype(np.float32)
    r32 = ref_nmf(ref, Xf, 10, W0f, T0f, max_iter=10)
    assert r32['W'].dtype == np.float32
    np.savez_compressed(os.path.join(OUT, 'cfg1_rri_f32.npz'), W_10=r32['W'], T_10=r32['T'],
                        relerr_10=orc.rel_error(Xf.astype(np.float64), r32['W'].astype(np.float64),
                                                r32['T'].astype(np.float64)))

    # regularised, noisy, non-square-ish case; k not a multiple of anything
    X, W0, T0 = orc.synth(257, 131, 6, 7, sigma=0.05, seed=3)
    regs = dict(reg_w_l1=0.02, reg_w_l2=0.1, reg_t_l1=0.01, reg_t_l2=0.05)
    r = ref_nmf(ref, X, 7, W0, T0, max_iter=6, compute_obj_each_iter=True, **regs)
    np.savez_compressed(os.path.join(OUT, 'reg_rri_f64.npz'), W=r['W'], T=r['T'],
                        obj_history=np.array(r['obj_history']),
                        regs=np.array([regs['reg_w_l1'], regs['reg_w_l2'], regs['reg_t_l1'],
                                       regs['reg_t_l2']]))

    # row-subset partial statistic (nmf.py:680-686) -- the multi-GPU partial (SURVEY.md F10)
    # (the reference's own store_gradients post-processing, nmf.py:541-549, passes a lambda as
    # stack_matrices' dict_key and raises; so we call _compute_update_T directly, which is where
    # the partial is defined)
    rows_a = np.arange(0, 100)
    rows_b = np.arange(100, 257)
    Wp, Tp = np.maximum(W0, 0), np.maximum(T0, 0)
    d = {'split': np.array([100])}
    for t in (0, 3, 6):
        for nm, rows in (('a', rows_a), ('b', rows_b), ('full', None)):
            wR, nw, wRs, nws = ref.nmf._compute_update_T(X=X, W=Wp, T=Tp, t=t, store_gradients=True,
                                                         ind_rows_to_store=rows, W_mat=None)
            d['numer_%s_%d' % (nm, t)] = np.asarray(wRs)
            d['denom_%s_%d' % (nm, t)] = np.asarray(nws)
    np.savez_compressed(os.path.join(OUT, 'partials_f64.npz'), **d)

    # fix_T=True (what transform() runs: sklearn_interface.py:327-334), 4 W-only sweeps
    r = ref_nmf(ref, X, 7, W0, T0, max_iter=4, fix_T=True)
    np.savez_compressed(os.path.join(OUT, 'fixT_f64.npz'), W=r['W'], T=r['T'])

    # ---------------------------------------------------------------- masked WRRI: recsys fixture
    Xr = scipy.sparse.load_npz(os.path.join(REF_DATA, 'recsys_data_train.npz')).toarray().astype(np.float64)
    M = np.zeros(Xr.shape)
    M[Xr.nonzero()] = 1.0
    rs = np.random.RandomState(11)
    W0 = rs.rand(100, 7)
    T0 = rs.rand(7, 200)
    d = {'X': Xr, 'W0': W0, 'T0': T0}
    for name, regs in (('plain', {}), ('l1both', {'reg_w_l1': 0.1, 'reg_t_l1': 0.1}),
                       ('l1w', {'reg_w_l1': 0.1}), ('l1t', {'reg_t_l1': 0.1})):
        # the RS settings of tests/test_nmf.py:66-72: ub_t = t_row_sum = 1.0, no projection
        r = ref_nmf(ref, Xr, 7, W0, T0, max_iter=15, W_mat=M, compute_obj_each_iter=True,
                    project_T_each_iter=False, t_row_sum=1.0, project_W_each_iter=False,
                    w_row_sum=None, **regs)
        d['W_' + name], d['T_' + name] = r['W'], r['T']
        d['obj_' + name] = np.array(r['obj_history'])
    np.savez_compressed(os.path.join(OUT, 'recsys_wrri_f64.npz'), **d)

    # masked, real-valued weights, no upper bound, synthetic
    X, W0, T0, Mb = orc.synth(120, 90, 5, 6, sigma=0.05, seed=5, mask_density=0.3)
    Mw = Mb * np.random.RandomState(9).rand(120, 90) * 2.0
    r = ref_nmf(ref, X, 6, W0, T0, max_iter=8, W_mat=Mw, compute_obj_each_iter=True)
    np.savez_compressed(os.path.join(OUT, 'weighted_wrri_f64.npz'), W=r['W'], T=r['T'],
                        obj_history=np.array(r['obj_history']))
    W, T = np.maximum(W0, 0), np.maximum(T0, 0)
    for s in range(5):
        ref_block_sweep(ref, X, W, T, M=Mw)
    np.savez_compressed(os.path.join(OUT, 'weighted_wrri_hals_f64.npz'), W=W, T=T)

    # ---------------------------------------------------------------- topic-model setting (simplex)
    Xt = scipy.sparse.load_npz(os.path.join(REF_DATA, 'text_data_train.npz')).toarray()
    Xt = ref.matrixops.normalize(ref.matrixops.tfidf(Xt))
    Xt = np.asarray(Xt, dtype=np.float64)
    rs = np.random.RandomState(12)
    W0 = rs.rand(100, 15)
    T0 = rs.rand(15, 200)
    d = {'X': Xt, 'W0': W0, 'T0': T0}
    # tests/test_nmf.py:30-35 settings, explicit init
    r = ref_nmf(ref, Xt, 15, W0, T0, max_iter=15, w_row_sum=1.0, project_T_each_iter=True,
                project_W_each_iter=True, compute_obj_each_iter=True, t_row_sum=1.0,
                early_stop=False, reg_t_l2=0.1)
    d['W_tm'], d['T_tm'], d['obj_tm'] = r['W'], r['T'], np.array(r['obj_history'])
    # NMF_TM_Estimator.fit settings (sklearn_interface.py:269-276): final projection only
    r = ref_nmf(ref, Xt, 15, W0, T0, max_iter=10, project_W_each_iter=False, w_row_sum=1.0,
                project_T_each_iter=True, t_row_sum=1.0, do_final_project_W=True)
    d['W_est'], d['T_est'] = r['W'], r['T']
    np.savez_compressed(os.path.join(OUT, 'text_tm_f64.npz'), **d)

    # ---------------------------------------------------------------- topic reset (default reset_topic_method)
    # a case where a topic collapses to zero in the first sweep: the reference re-seeds it from the document
    # with the largest positive residual (nmf.py:762-783)
    rs = np.random.RandomState(33 + 57)
    X, W0, T0 = rs.rand(33, 57), rs.rand(33, 8), rs.rand(8, 57)
    r = ref.nmf.nmf(X, 8, W_in=W0, T_in=T0, max_iter=6, compute_obj_each_iter=True, eps_stop=-1.0)
    np.savez_compressed(os.path.join(OUT, 'reset_rri_f64.npz'), W=r['W'], T=r['T'],
                        obj_history=np.array(r['obj_history']),
                        resets_remaining=np.array([ref.nmf.n_resets_remaining]))

    # ---------------------------------------------------------------- reference test replay (App. B.3)
    # NNDSVD-initialised (depends on sklearn's randomized_svd) -> scalar regression goldens only
    rep = {}
    Wm = np.zeros(Xr.shape)
    Wm[Xr.nonzero()] = 1.0
    for name, regs in (('rs_plain', {}), ('rs_l1both', {'reg_w_l1': 0.1, 'reg_t_l1': 0.1})):
        r = ref.nmf.nmf(Xr, k=7, max_iter=15, random_state=0, W_mat=Wm, compute_obj_each_iter=True,
                        reset_topic_method=None, early_stop=False, project_T_each_iter=False,
                        t_row_sum=1.0, project_W_each_iter=False, w_row_sum=None, **regs)
        rep[name] = np.array(r['obj_history'])
    np.savez_compressed(os.path.join(OUT, 'replay_scalars.npz'), **rep)
    estimator_goldens(ref, Xr)
    print('golden written to', os.path.abspath(OUT))
    for f in sorted(os.listdir(OUT)):
        print('  %-32s %8d B' % (f, os.path.getsize(os.path.join(OUT, f))))


# the inputs of the live-reference tests (tests/test_oracle.py, tests/test_abi_cpu.py)
LIVE_RANDOM_CASES = ((64, 40, 5, False), (33, 57, 4, False), (40, 30, 4, True))


def live_case_pins():
    """tests/golden/live_cases_f64.npz: what the ORACLE (and, for the host helpers, rri_nmf_b200._host) returns on the
    inputs of the tests that compare with the live reference, so that those tests check every checkout, also one
    without the reference.  These values are not the reference's own: the reference sources are not part of the
    repository.  With the reference present the same tests also compare with it directly.

        python oracle/make_golden.py live-pins
    """
    sys.path.insert(0, os.path.join(HERE, '..'))
    from rri_nmf_b200._host import initialize_nmf, normalize, tfidf
    d = {}
    for n, dd, k, masked in LIVE_RANDOM_CASES:
        rs = np.random.RandomState(n + dd)
        X, W0, T0 = rs.rand(n, dd), rs.rand(n, k), rs.rand(k, dd)
        M = (rs.rand(n, dd) < 0.4).astype(float) if masked else None
        o = orc.nmf_oracle(X, k, W0, T0, max_iter=5, W_mat=M, compute_obj_each_iter=True, eps_stop=-1.0)
        key = '%d_%d_%d_%d' % (n, dd, k, masked)
        d['W_' + key], d['T_' + key], d['obj_' + key] = o['W'], o['T'], np.array(o['obj_history'])
    rs = np.random.RandomState(1)
    X, W0, T0 = rs.rand(60, 50), rs.rand(60, 4), rs.rand(4, 50)
    o = orc.nmf_oracle(X, 4, W0, T0, max_iter=200, compute_obj_each_iter=True, eps_stop=1e-3)
    d['stop_len'] = np.array([len(o['obj_history'])])
    rs = np.random.RandomState(0)
    X = rs.rand(40, 30) * (rs.rand(40, 30) < 0.3)
    d['tfidf'], d['normalize'] = tfidf(X), normalize(X)
    for init in ('random', 'smart_random', 'nndsvd', 'nndsvda', 'nndsvdar'):
        d['W_' + init], d['T_' + init] = initialize_nmf(X, 5, init, random_state=3)
    np.savez_compressed(os.path.join(OUT, 'live_cases_f64.npz'), **d)


if __name__ == '__main__':
    if sys.argv[1:] == ['live-pins']:
        live_case_pins()
    else:
        main()
