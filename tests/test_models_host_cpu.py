"""nmf_models on the host side (no GPU): every unsupported argument is refused before any device work, and the models
are grouped by the width cap of the shared contraction."""
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


X = np.random.RandomState(0).rand(20, 12)


@pytest.mark.parametrize('kw', [
    dict(W_mat=np.ones((20, 12))),
    dict(comm=object()),
    dict(update_order='rri'),
    dict(fix_W=True),
    dict(fix_T=True),
    dict(project_T_each_iter=True, t_row_sum=1.0),
    dict(early_stop=lambda X, W, T: 0.0),
    dict(diagnostics=[lambda X, W, T: 0.0]),
    dict(w_row=np.ones(20)),
    dict(store_gradients=True),
    dict(return_reconstruction_err=True),
])
def test_unsupported_arguments_raise_before_device_work(no_device, kw):
    with pytest.raises(NotImplementedError):
        R.nmf_models(X, 3, random_state=[0, 1], **kw)


def test_sparse_X_raises_before_device_work(no_device):
    with pytest.raises(NotImplementedError):
        R.nmf_models(sp.random(20, 12, density=0.3, format='csr'), 3, random_state=[0, 1])


@pytest.mark.parametrize('kw', [
    dict(random_state=[0, 1], W_in=[np.ones((20, 3))]),
    dict(W_in=[np.ones((20, 3))] * 2, T_in=[np.ones((3, 12))] * 3),
    dict(random_state=[0, 1, 2], T_in=[np.ones((3, 12))] * 2),
])
def test_list_lengths_must_agree(no_device, kw):
    with pytest.raises(ValueError):
        R.nmf_models(X, 3, **kw)


def test_rank_above_256_and_missing_lists(no_device):
    with pytest.raises(ValueError):
        R.nmf_models(X, 257, random_state=[0])
    with pytest.raises(ValueError):
        R.nmf_models(X, 3)
    with pytest.raises(ValueError):
        R.nmf_models(X, 3, random_state=[0], update_order='block')
    with pytest.raises(TypeError):
        R.nmf_models(X, 3, random_state=[0], n_init=4)


def test_groups_respect_the_width_cap():
    cap = nmf_mod.MODELS_WIDTH_CAP
    assert nmf_mod._model_groups(3, 100, cap=256) == [2, 1]
    assert nmf_mod._model_groups(8, 32, cap=256) == [8]
    assert nmf_mod._model_groups(9, 32, cap=256) == [8, 1]
    assert nmf_mod._model_groups(5, 64, cap=128) == [2, 2, 1]
    assert nmf_mod._model_groups(2, 256, cap=256) == [1, 1]
    for b, k in [(1, 1), (7, 16), (40, 8), (3, 200)]:
        g = nmf_mod._model_groups(b, k)
        assert sum(g) == b and all(x * k <= max(cap, k) for x in g)

