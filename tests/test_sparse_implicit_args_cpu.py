"""nmf(..., unstored_weight=w0) on the host side (no GPU): every argument the weighted-unstored path does not take is
refused before any device work, and w0 = 0 leaves the call path as it was."""
import importlib

import numpy as np
import pytest
import scipy.sparse as sp

import rri_nmf_b200 as R

nmf_mod = importlib.import_module('rri_nmf_b200.nmf')      # (the package attribute `nmf` is the function)


@pytest.fixture
def no_device(monkeypatch):
    """any attempt to reach a device, an engine or an initialisation fails the test"""
    def boom(*a, **kw):
        raise AssertionError('device work before the argument check')
    monkeypatch.setattr(nmf_mod, 'RRIEngine', boom)
    monkeypatch.setattr(nmf_mod, '_to_device', boom)
    monkeypatch.setattr(nmf_mod, '_host_start', boom)
    monkeypatch.setattr(nmf_mod.torch.cuda, 'is_available', boom)


Xs = sp.random(20, 12, density=0.3, format='csr', random_state=0)


@pytest.mark.parametrize('X,kw', [
    (Xs.toarray(), dict(unstored_weight=0.1)),                   # dense X: the weights belong in a dense W_mat
    (Xs, dict(unstored_weight=0.1, unstored='zero')),            # zero-filled: every unstored entry has weight 1
    (Xs, dict(unstored_weight=-0.1)),
    (Xs, dict(unstored_weight=float('nan'))),
    (Xs, dict(unstored_weight=float('inf'))),
    (Xs, dict(unstored_weight='heavy')),
])
def test_bad_unstored_weight_raises_value_error(no_device, X, kw):
    with pytest.raises(ValueError):
        R.nmf(X, 3, **kw)


@pytest.mark.parametrize('kw', [dict(comm=object()), dict(fix_W=True)])
def test_unimplemented_combinations_raise(no_device, kw):
    with pytest.raises(NotImplementedError):
        R.nmf(Xs, 3, unstored_weight=0.1, **kw)


def test_zero_weight_passes_the_check():
    """w0 = 0 is accepted for every input kind (it is the default) and is the plain float 0"""
    for X, unstored in ((Xs, 'missing'), (Xs, 'zero'), (Xs.toarray(), 'missing')):
        assert nmf_mod.check_unstored_weight(0, sp.issparse(X), unstored) == 0.0
    assert nmf_mod.check_unstored_weight(np.float32(0.25), True, 'missing') == 0.25
