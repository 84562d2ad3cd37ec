"""CPU model of the rule by which a TF32 hals handle keeps X as 16-bit copies (x16_kernels.cu: x16_exponent).

fp16(tf32(x) * 2^e) is exact when tf32(x) * 2^e is 0 or a normal fp16 (2^-14 <= |.| <= 65504).  The scale puts the
largest |tf32(x)| into [2^15, 2^16); the copies are taken when every other nonzero value then stays >= 2^-14, no value
is inf / nan and none is an fp32 subnormal.  tests/test_gpu_x16.py checks the device's decision against this model."""
import numpy as np


def tf32(x):
    """round float32 values to TF32 (10 mantissa bits) the way the TF32 tensor map does: nearest, ties to even"""
    b = np.asarray(x, dtype=np.float32).view(np.uint32).astype(np.uint64)
    finite = (b & 0x7f800000) != 0x7f800000
    r = np.where(finite, (b + 0xfff + ((b >> 13) & 1)) & 0xffffe000, b).astype(np.uint32)
    return r.view(np.float32)


def x16_rule(X):
    """(True, e) when X is kept as fp16(tf32(X) * 2^e), else (False, None)"""
    a = np.abs(tf32(X).astype(np.float32))
    if not np.all(np.isfinite(a)):
        return False, None
    nz = a[a != 0]
    if nz.size == 0:
        return True, 0
    if nz.min() < np.finfo(np.float32).tiny:
        return False, None
    emax, emin = int(np.frexp(nz.max())[1]) - 1, int(np.frexp(nz.min())[1]) - 1
    e = min(15 - emax, 126)
    return (emin + e >= -14), (e if emin + e >= -14 else None)


def to_x16(X, e):
    """the 16-bit copy itself, and the check that it is exact"""
    s = np.float32(2.0 ** e)
    y = (tf32(X) * s).astype(np.float16)
    assert np.array_equal(y.astype(np.float32), tf32(X) * s)
    return y


def test_tf32_rounding_ties_go_to_even():
    one = np.float32(1.0)
    ulp = np.float32(2.0 ** -10)
    x = np.array([1 + 2 ** -11, 1 + 3 * 2 ** -11, 1 + 2 ** -12, -(1 + 2 ** -11), 1 + 2 ** -11 + 2 ** -23,
                  1 + 5 * 2 ** -11, np.finfo(np.float32).max], dtype=np.float32)
    assert tf32(x).tolist() == [one, one + 2 * ulp, one, -one, one + ulp, one + 2 * ulp, np.inf]


def test_rule_edges():
    assert x16_rule(np.zeros((3, 4), np.float32)) == (True, 0)
    # values between 2 and 80 (the benchmark's data): max 80 -> scale 2^9
    ok, e = x16_rule(np.array([[2.0, 80.0], [0.0, 33.5]], np.float32))
    assert ok and e == 9
    # exactly 30 binades: [2^-26, 2^3 * (2 - 2^-10)]
    top = np.float32(8 * (2 - 2 ** -10))
    ok, e = x16_rule(np.array([top, 2.0 ** -26, -3.0], np.float32))
    assert ok and e == 12
    y = to_x16(np.array([top, 2.0 ** -26], np.float32), e)
    assert float(y[0]) == 65504.0 and float(y[1]) == 2.0 ** -14
    # one binade more is out of range
    assert x16_rule(np.array([top, 2.0 ** -27], np.float32)) == (False, None)
    # the maximum rounds up into the next binade under TF32: the scale follows the rounded value
    ok, e = x16_rule(np.array([np.float32(16 - 2 ** -20), 1.0], np.float32))
    assert ok and e == 11
    # non-finite values and fp32 subnormals keep the fp32 path
    assert x16_rule(np.array([1.0, np.inf], np.float32)) == (False, None)
    assert x16_rule(np.array([1.0, np.nan], np.float32)) == (False, None)
    assert x16_rule(np.array([2.0 ** -130, 2.0 ** -128], np.float32)) == (False, None)
    # a finite value that rounds to inf under TF32
    assert x16_rule(np.array([np.finfo(np.float32).max], np.float32)) == (False, None)
    # tiny but normal data: the scale is capped at 2^126
    ok, e = x16_rule(np.array([2.0 ** -120, 2.0 ** -125], np.float32))
    assert ok and e == 126
    assert x16_rule(np.array([2.0 ** -120, 2.0 ** -126], np.float32)) == (True, 126)
