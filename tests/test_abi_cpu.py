"""CPU-side checks (no GPU): the C-ABI library loads and exports every symbol include/rri_b200.h declares,
the host helpers match the reference's known-answer test, and the product path refuses to run without
a CUDA device (no CPU fallback)."""
import os
import re

import numpy as np
import pytest

from conftest import ROOT

HEADER = os.path.join(ROOT, 'include', 'rri_b200.h')


def _declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    return sorted(set(re.findall(r'\b(rri_[A-Za-z0-9_]+)\s*\(', src)))


def test_header_and_binding_agree():
    from rri_nmf_b200 import _lib
    assert _declared_symbols() == sorted(_lib.SYMBOLS)


def test_library_exports_every_declared_symbol():
    from rri_nmf_b200 import _lib
    if not os.path.isfile(_lib.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    lib = _lib.load()
    for name in _declared_symbols():
        assert hasattr(lib, name), name
    assert b'sm_100a' in lib.rri_version()


def test_struct_layout_matches_header():
    import ctypes as C
    from rri_nmf_b200._lib import RriParams
    assert C.sizeof(RriParams) == 7 * 8 + 4 * 4


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip('a GPU is present')
    import ctypes as C
    import rri_nmf_b200
    from rri_nmf_b200 import _lib
    lib = _lib.load()
    h = C.c_void_p()
    assert lib.rri_create(C.byref(h), 10, 10, 2, 0, 0, 0, 0) != 0
    assert b'no CPU fallback' in lib.rri_last_error()
    with pytest.raises(_lib.RriError):
        rri_nmf_b200.nmf(np.random.rand(10, 8), 2)
    with pytest.raises(_lib.RriError):
        rri_nmf_b200.RRIEngine(torch.zeros(4, 4), 2)


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, 'rri_nmf_b200')
    for fn in os.listdir(pkg):
        if fn.endswith('.py'):
            src = open(os.path.join(pkg, fn)).read()
            assert 'rri_oracle' not in src and 'refshim' not in src and 'import oracle' not in src, fn


def test_nndsvd_known_answer():
    """reference tests/test_nmf.py:13-19 with the golden bytes of tests/conftest.py:8-19 (decoded in
    SURVEY.md App. B.2)"""
    from rri_nmf_b200._host import initialize_nmf
    X = np.array([[1, 0], [0.5, 0.5], [0.25, 0.75]])
    Wt = np.array([[0.7731182278974053, 0], [0.6108880790649228, 0.2268147629447849],
                   [0.5297730046486816, 0.6538575655189827]])
    Tt = np.array([[0.9676003516472353, 0.5615202893907696], [0, 0.6920799467374485]])
    W, T = initialize_nmf(X, 2, init='nndsvd', random_state=0)
    assert np.allclose(Wt, W) and np.allclose(Tt, T)


def test_host_helpers_against_reference_when_present():
    """against tests/golden/live_cases_f64.npz (these helpers' own outputs, oracle/make_golden.py live-pins) and,
    when the reference is present, against its matrixops / initialization directly"""
    import refshim
    from conftest import golden
    from rri_nmf_b200._host import initialize_nmf, normalize, tfidf
    rs = np.random.RandomState(0)
    X = rs.rand(40, 30) * (rs.rand(40, 30) < 0.3)
    g = golden('live_cases_f64.npz')
    inits = ('random', 'smart_random', 'nndsvd', 'nndsvda', 'nndsvdar')
    expected = [(g['tfidf'], g['normalize'], {i: (g['W_' + i], g['T_' + i]) for i in inits})]
    if refshim.available():
        ref = refshim.load()
        expected.append((ref.matrixops.tfidf(X), ref.matrixops.normalize(X),
                         {i: ref.initialization.initialize_nmf(X, 5, i, random_state=3) for i in inits}))
    for tf, nm, init_out in expected:
        assert np.allclose(tfidf(X), tf)
        assert np.allclose(normalize(X), nm)
        for init in inits:
            a, b = initialize_nmf(X, 5, init, random_state=3), init_out[init]
            assert np.allclose(a[0], b[0]) and np.allclose(a[1], b[1]), init


def test_estimator_surface():
    """constructor parameters / attributes of sklearn_interface.py:15-38, :187-226"""
    import rri_nmf_b200 as R
    tm = R.NMF_TM_Estimator(100, 200, 5, wr1=0.1, max_iter=7)
    assert (tm.n, tm.d, tm.k, tm.wr1, tm.max_iter, tm.handle_tfidf) == (100, 200, 5, 0.1, 7, False)
    assert tm.get_params()['k'] == 5 and tm.n_components == 5
    rs = R.NMF_RS_Estimator(100, 200, 5)
    assert rs.max_iter == 30 and rs.use_validation_early_stopping and rs.Xpred.size == 0
    for m in ('fit', 'fit_transform', 'transform', 'one_iter', 'score', 'sparsify', 'densify', 'constrained_transform'):
        assert hasattr(tm, m)
    for m in ('fit', 'fit_from_Xtr', 'transform', 'predict', 'score', 'make_Xpred', 'sparsify', 'densify'):
        assert hasattr(rs, m)


def test_documented_switches_exist_in_the_sources():
    """DESIGN.md §9a lists the A/B environment switches of the library; every one of them must be read somewhere in
    csrc/ or the Python package, and every switch the CUDA sources read must be listed there."""
    design = open(os.path.join(ROOT, 'DESIGN.md')).read()
    sec = design[design.index('## 9a.'):design.index('## 10.')]
    documented = set(re.findall(r'`(RRI_[A-Z0-9_]+)', sec))
    read = set()
    pkg = os.path.join(ROOT, 'rri_nmf_b200')
    for d, _, files in os.walk(pkg):
        if os.path.basename(d) == 'build':
            continue
        for f in files:
            if f.endswith(('.cu', '.cuh', '.h', '.py')):
                src = open(os.path.join(d, f)).read()
                read |= set(re.findall(r'getenv\("(RRI_[A-Z0-9_]+)"\)', src))
                read |= set(re.findall(r"environ(?:\.get)?[\(\[]\s*'(RRI_[A-Z0-9_]+)'", src))
    assert documented <= read, sorted(documented - read)
    assert read <= documented, sorted(read - documented)
