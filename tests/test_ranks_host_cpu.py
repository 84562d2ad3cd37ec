"""nmf_models with a list of ranks on the host side (no GPU): argument checks and unsupported arguments are refused
before any device work, and the models are packed into groups first fit by decreasing rank."""
import importlib

import numpy as np
import pytest

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
    dict(random_state=[0, 1]),                                   # 3 ranks, 2 seeds
    dict(W_in=[np.ones((20, 2)), np.ones((20, 3))], T_in=[np.ones((2, 12)), np.ones((3, 12))]),
    dict(W_in=[np.ones((20, 2)), np.ones((20, 3)), np.ones((20, 5))], random_state=[0, 1, 2]),   # W_in[2] not 20 x 4
    dict(T_in=[np.ones((2, 12)), np.ones((4, 12)), np.ones((4, 12))], random_state=[0, 1, 2]),   # T_in[1] not 3 x 12
])
def test_list_lengths_and_shapes(no_device, kw):
    with pytest.raises(ValueError):
        R.nmf_models(X, [2, 3, 4], **kw)


@pytest.mark.parametrize('ranks', [[2, 0, 3], [2, 257], [-1]])
def test_ranks_outside_range(no_device, ranks):
    with pytest.raises(ValueError):
        R.nmf_models(X, ranks)


@pytest.mark.parametrize('kw', [
    dict(W_mat=np.ones((20, 12))),
    dict(comm=object()),
    dict(update_order='rri'),
    dict(fix_W=True),
    dict(project_T_each_iter=True, t_row_sum=1.0),
    dict(early_stop=lambda X, W, T: 0.0),
    dict(diagnostics=[lambda X, W, T: 0.0]),
    dict(return_reconstruction_err=True),
])
def test_unsupported_arguments_raise_before_device_work(no_device, kw):
    with pytest.raises(NotImplementedError):
        R.nmf_models(X, [2, 3], **kw)


def test_first_fit_decreasing_groups():
    assert nmf_mod._rank_groups([200, 100, 50, 150]) == [[0, 2], [1, 3]]
    assert nmf_mod._rank_groups(list(range(2, 21))) == [list(range(19))]
    assert nmf_mod._rank_groups([128, 64, 32, 16, 16, 1]) == [[0, 1, 2, 3, 4], [5]]
    assert nmf_mod._rank_groups([3, 5, 3], cap=8) == [[0, 1], [2]]      # ties in caller order: model 0 before 2
