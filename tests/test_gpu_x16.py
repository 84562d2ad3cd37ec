"""16-bit storage of X on TF32 hals handles (x16_kernels.cu, f16_gemm_run): the fp16 copies carry exactly the operand
the TF32 tensor map produces, the handle falls back to fp32 storage when that is not possible, and the sweeps agree
with the fp32 storage to the contraction's reordering spread."""
import numpy as np
import pytest
import torch

from test_x16_rule_cpu import tf32, x16_rule

pytestmark = pytest.mark.gpu


def _engine(X, k=16, x16=True, monkeypatch=None):
    import rri_nmf_b200 as R
    if not x16:
        monkeypatch.setenv('RRI_X16', '0')
    try:
        return R.RRIEngine(X, k, order='hals', math='tf32')
    finally:
        if not x16:
            monkeypatch.delenv('RRI_X16')


def _crafted(n, d, emax, seed=0):
    """values spread over the 30 binades [2^(emax-29), 2^(emax+1)), with TF32 rounding ties (both parities), values
    just off a tie, zeros, negatives, and both ends of the scaled fp16 range"""
    rs = np.random.RandomState(seed)
    E = rs.randint(emax - 29, emax, size=(n, d))
    hi = rs.randint(0, 1024, size=(n, d)).astype(np.uint32)              # the mantissa bits TF32 keeps
    lo = rs.choice(np.array([0, 0x1000, 0x0fff, 0x1001, 0x1fff, 1], np.uint32), size=(n, d))
    lo = np.where(rs.rand(n, d) < 0.3, rs.randint(0, 0x2000, size=(n, d)).astype(np.uint32), lo)
    mant = (hi << 13) | lo
    bits = ((E + 127).astype(np.uint32) << 23) | mant
    X = bits.view(np.float32).copy()
    X[rs.rand(n, d) < 0.3] *= -1
    X[rs.rand(n, d) < 0.1] = 0
    X[0, 0] = np.float32(2.0 ** emax * (2 - 2 ** -10))          # the largest value: 65504 once scaled
    X[1, 1] = np.float32(2.0 ** (emax - 29))                     # the smallest normal fp16 once scaled
    X[2, 2] = -X[1, 1]
    return X


def _unit_rows(idx, K, device):
    B = torch.zeros((len(idx), K), dtype=torch.float32, device=device)
    B[torch.arange(len(idx)), torch.as_tensor(idx)] = 1.0
    return B


@pytest.mark.parametrize('n,d,emax', [(300, 204, 3), (256, 136, 6), (520, 96, -20)])
def test_operand_is_the_tf32_value(cuda_device, monkeypatch, n, d, emax):
    """X (and X') against unit-vector factor rows returns the operand itself: bit for bit the TF32 value of x, from
    the 16-bit storage as from the fp32 tensor map"""
    X = _crafted(n, d, emax)
    ok, e = x16_rule(X)
    assert ok
    Xd = torch.from_numpy(X).to(cuda_device)
    eng = _engine(Xd, monkeypatch=monkeypatch)
    ref = _engine(Xd, x16=False, monkeypatch=monkeypatch)
    assert eng.stats()['x_operand'] == 'f16' and ref.stats()['x_operand'] == 'f32'
    want = tf32(X)
    N = 16
    Xt = Xd.t().contiguous()
    for c0 in range(0, d, N):
        cols = list(range(c0, min(c0 + N, d)))
        B = _unit_rows(cols, d, cuda_device)
        got = eng.contract_x(B).cpu().numpy()
        assert np.array_equal(got.view(np.uint32), want[:, cols].view(np.uint32))
        assert np.array_equal(got.view(np.uint32), ref.contract_x(B).cpu().numpy().view(np.uint32))
        assert np.array_equal(got.view(np.uint32), eng.gemm_nt(Xd, B).cpu().numpy().view(np.uint32))
    for r0 in range(0, n, 4 * N):
        rows = list(range(r0, min(r0 + N, n)))
        B = _unit_rows(rows, n, cuda_device)
        got = eng.contract_x(B, transpose=True).cpu().numpy()
        assert np.array_equal(got.view(np.uint32), want[rows, :].T.view(np.uint32))
        assert np.array_equal(got.view(np.uint32), eng.gemm_nt(Xt, B).cpu().numpy().view(np.uint32))
    eng.close()
    ref.close()


@pytest.mark.parametrize('case', ['too_wide', 'inf', 'nan', 'subnormal', 'zeros', 'env'])
def test_storage_decision(cuda_device, monkeypatch, case):
    """out-of-range or non-finite data binds on fp32 storage (and still sweeps); the decision matches the model"""
    X = _crafted(128, 64, 3)
    if case == 'too_wide':
        X[5, 5] = np.float32(2.0 ** -27)
    elif case == 'inf':
        X[5, 5] = np.inf
    elif case == 'nan':
        X[5, 5] = np.nan
    elif case == 'subnormal':
        X[5, 5] = np.float32(2.0 ** -130)
    elif case == 'zeros':
        X[:] = 0
    Xd = torch.from_numpy(X).to(cuda_device)
    eng = _engine(Xd, k=4, x16=case != 'env', monkeypatch=monkeypatch)
    expect = x16_rule(X)[0] and case != 'env'
    assert eng.stats()['x_operand'] == ('f16' if expect else 'f32')
    if case in ('too_wide', 'subnormal', 'env'):
        B = _unit_rows([5, 6, 7, 8], 64, cuda_device)
        got = eng.contract_x(B).cpu().numpy()
        assert np.array_equal(got.view(np.uint32), eng.gemm_nt(Xd, B).cpu().numpy().view(np.uint32))
    eng.close()


def test_sweeps_agree_with_fp32_storage(cuda_device, monkeypatch):
    """the block-order sweeps on 16-bit storage against fp32 storage on the same data: the contractions see the same
    operands and differ only in the order of their sums"""
    import rri_oracle as orc
    X, W0, T0 = orc.synth(3000, 1000, 16, 16, sigma=0.05, seed=3)
    X = np.abs(X).astype(np.float32)
    assert x16_rule(X)[0]
    Xd = torch.from_numpy(X).to(cuda_device)
    out = {}
    for x16 in (True, False):
        eng = _engine(Xd, k=16, x16=x16, monkeypatch=monkeypatch)
        assert eng.stats()['x_operand'] == ('f16' if x16 else 'f32')
        W = torch.from_numpy(W0.astype(np.float32)).to(cuda_device)
        T = torch.from_numpy(T0.astype(np.float32)).to(cuda_device)
        eng.sweeps(W, T, 20, eng.params())
        out[x16] = (W.cpu().numpy().astype(np.float64), T.cpu().numpy().astype(np.float64), eng.rel_error(W, T))
        # N sweeps in one call == N calls of one sweep, bit for bit
        W2 = torch.from_numpy(W0.astype(np.float32)).to(cuda_device)
        T2 = torch.from_numpy(T0.astype(np.float32)).to(cuda_device)
        for _ in range(20):
            eng.sweeps(W2, T2, 1, eng.params())
        assert torch.equal(W, W2) and torch.equal(T, T2)
        eng.close()
    (Wa, Ta, ra), (Wb, Tb, rb) = out[True], out[False]
    assert np.linalg.norm(Wa - Wb) / np.linalg.norm(Wb) < 1e-3
    assert np.linalg.norm(Ta - Tb) / np.linalg.norm(Tb) < 1e-3
    assert abs(ra - rb) < 1e-5 * ra + 1e-7
