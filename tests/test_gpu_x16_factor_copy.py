"""The fp16 copy of the factor operand (f16_absmax_kernel / f16_factor_kernel, x16_kernels.cu) carries exactly the TF32
value of every factor element, on the four-element path (rows of a multiple of 4 columns) and on the element-at-a-time
path (other widths)."""
import numpy as np
import pytest
import torch

from test_gpu_x16 import _crafted, _engine
from test_x16_rule_cpu import tf32

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize('n,d', [(300, 204), (301, 203), (257, 136)])
def test_factor_copy_is_the_tf32_value(cuda_device, monkeypatch, n, d):
    """X holds one 1 per row (row i at column i mod d), so X B' returns B's entries themselves and X' W sums them per
    column: both must be bit for bit the TF32 values of the factor (30 binades: exact under one power-of-two scale)"""
    X = np.zeros((n, d), np.float32)
    X[np.arange(n), np.arange(n) % d] = 1.0
    Xd = torch.from_numpy(X).to(cuda_device)
    eng = _engine(Xd, monkeypatch=monkeypatch)
    assert eng.stats()['x_operand'] == 'f16'
    B = _crafted(16, d, 5, seed=1)
    got = eng.contract_x(torch.from_numpy(B).to(cuda_device)).cpu().numpy()
    assert np.array_equal(got.view(np.uint32), tf32(B)[:, np.arange(n) % d].T.copy().view(np.uint32))
    # X' W with the rows of W at distinct columns of X (n <= 2d: at most two nonzero terms per column, one of them 0 here)
    W = _crafted(16, n, -7, seed=2)
    W[:, d:] = 0
    got = eng.contract_x(torch.from_numpy(W).to(cuda_device), transpose=True).cpu().numpy()
    want = np.zeros((d, 16), np.float32)
    want[: min(n, d)] = tf32(W)[:, : min(n, d)].T
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    eng.close()
