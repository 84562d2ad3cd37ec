"""The blocked simplex threshold of the constrained block-order T update (oracle/simplex_theta.py, the model of
simplex_kernels.cu: grid_michelot) equals the sort-based projection of the reference (euclidean_proj_simplex) for any
split of the vector into blocks."""
import numpy as np
import pytest

import rri_oracle as orc
import simplex_theta as sx

BLOCKS = [1, 2, 3, 7, 32, 148]


def _check(x, s, nblocks):
    ref = orc.euclidean_proj_simplex(np.array(x, dtype=np.float64), s)
    got = sx.blocked_proj_simplex(x, s, nblocks)
    assert np.allclose(got, ref, rtol=1e-12, atol=1e-15), (nblocks, s)
    assert abs(got.sum() - s) <= 1e-12 * max(1.0, s)
    assert np.all(got >= 0)


@pytest.mark.parametrize('nblocks', BLOCKS)
@pytest.mark.parametrize('s', [1.0, 2.5, 0.3])
def test_random_vectors(nblocks, s):
    rs = np.random.RandomState(nblocks)
    for d in (1, 5, 150, 1000):
        _check(rs.rand(d) * rs.choice([0.01, 1.0, 50.0]), s, min(nblocks, d))
        # the solve's output: many exact zeros (clipped numerators)
        _check(np.maximum(rs.randn(d), 0), s, min(nblocks, d))


@pytest.mark.parametrize('nblocks', BLOCKS)
def test_ties(nblocks):
    x = np.array([0.5, 0.5, 0.5, 0.2, 0.2, 0.0, 0.5] * 30)
    for s in (1.0, 2.5):
        _check(x, s, nblocks)


@pytest.mark.parametrize('nblocks', BLOCKS)
def test_all_zero(nblocks):
    d = 300
    _check(np.zeros(d), 1.0, nblocks)
    assert np.allclose(sx.blocked_proj_simplex(np.zeros(d), 2.5, nblocks), 2.5 / d)


@pytest.mark.parametrize('nblocks', BLOCKS)
def test_single_positive_entry(nblocks):
    x = np.zeros(400)
    x[123] = 7.0
    for s in (1.0, 2.5):
        got = sx.blocked_proj_simplex(x, s, nblocks)
        _check(x, s, nblocks)
        assert got[123] == s and np.count_nonzero(got) == 1


@pytest.mark.parametrize('nblocks', BLOCKS)
def test_sum_below_radius_negative_theta(nblocks):
    """sum(x+) < s: theta < 0 and every entry, the zeros included, is lifted"""
    rs = np.random.RandomState(3)
    x = np.maximum(rs.randn(500), 0) * 1e-3
    assert x.sum() < 1.0
    theta, _ = sx.blocked_theta(x, 1.0, nblocks)
    assert theta < 0
    _check(x, 1.0, nblocks)
    assert np.all(sx.blocked_proj_simplex(x, 1.0, nblocks) > 0)


def test_every_block_split_gives_the_same_active_set():
    rs = np.random.RandomState(11)
    x = np.maximum(rs.randn(2000), 0)
    ref = orc.euclidean_proj_simplex(x, 1.0) > 0
    for nb in range(1, 149):
        assert np.array_equal(sx.blocked_proj_simplex(x, 1.0, nb) > 0, ref), nb
