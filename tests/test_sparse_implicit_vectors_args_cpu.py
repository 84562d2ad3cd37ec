"""nmf(..., unstored_row_weight=a, unstored_col_weight=b) on the host side (no GPU): every argument the rank-one
unstored weights do not serve is refused before any device work, and nmf_models refuses the keywords."""
import importlib

import numpy as np
import pytest
import scipy.sparse as sp
import torch

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
a20, b12 = np.linspace(0.5, 2.0, 20), np.linspace(0.1, 1.0, 12)


@pytest.mark.parametrize('X,kw', [
    (Xs, dict(unstored_row_weight=a20)),                                        # no w0
    (Xs, dict(unstored_col_weight=b12, unstored_weight=0.0)),
    (Xs.toarray(), dict(unstored_col_weight=b12)),                              # dense X
    (Xs.toarray(), dict(unstored_col_weight=b12, unstored_weight=0.1)),
    (Xs, dict(unstored_row_weight=a20, unstored_weight=0.1, unstored='zero')),  # zero-filled
    (Xs, dict(unstored_row_weight=a20[:19], unstored_weight=0.1)),              # wrong lengths
    (Xs, dict(unstored_col_weight=a20, unstored_weight=0.1)),
    (Xs, dict(unstored_row_weight=a20.reshape(4, 5), unstored_weight=0.1)),     # not 1-D
    (Xs, dict(unstored_row_weight=np.float64(2.0), unstored_weight=0.1)),
    (Xs, dict(unstored_col_weight=np.r_[b12[:-1], -0.5], unstored_weight=0.1)),  # negative, non-finite
    (Xs, dict(unstored_col_weight=np.r_[b12[:-1], np.nan], unstored_weight=0.1)),
    (Xs, dict(unstored_row_weight=torch.from_numpy(np.r_[a20[:-1], np.inf]), unstored_weight=0.1)),
    (Xs, dict(unstored_row_weight=['x'] * 20, unstored_weight=0.1)),
])
def test_bad_vectors_raise_value_error(no_device, X, kw):
    with pytest.raises(ValueError):
        R.nmf(X, 3, **kw)


@pytest.mark.parametrize('kw', [dict(comm=object()), dict(fix_W=True)])
def test_unimplemented_combinations_raise(no_device, kw):
    with pytest.raises(NotImplementedError):
        R.nmf(Xs, 3, unstored_weight=0.1, unstored_row_weight=a20, unstored_col_weight=b12, **kw)


@pytest.mark.parametrize('kw', [dict(unstored_row_weight=a20), dict(unstored_col_weight=b12)])
def test_nmf_models_refuses_the_vectors(no_device, kw):
    with pytest.raises(NotImplementedError):
        R.nmf_models(Xs.toarray(), 3, random_state=[0, 1], **kw)


def test_accepted_vectors_come_back_as_host_arrays():
    """NumPy and CPU torch vectors (any float dtype) pass the check as float64 arrays; None stays None"""
    a, b = nmf_mod.check_unstored_vectors(torch.from_numpy(a20.astype(np.float32)), None, 20, 12, 0.1)
    assert isinstance(a, np.ndarray) and a.dtype == np.float64 and b is None
    assert np.array_equal(a, a20.astype(np.float32).astype(np.float64))
    a, b = nmf_mod.check_unstored_vectors(None, list(b12), 20, 12, 0.25)
    assert a is None and np.array_equal(b, b12)
    assert nmf_mod.check_unstored_vectors(None, None, 20, 12, 0.0) == (None, None)
