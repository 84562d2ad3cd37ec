"""Signed bias of the block-order contraction over long K with both storages of X: the fp32 tensor map (TF32 rounding on
the way into shared memory, tcgen05.mma kind::tf32) and the 16-bit copies (kind::f16), against the fp64 product of the
same TF32-rounded operands.  The TMEM flush period (RRI_GEMM_FLUSH, in 32-wide chunks; 4 = every 128 K) bounds the
accumulation chain of either kind.
python tools/x16_bias.py      (RRI_GEMM_FLUSH=0 disables the flush)"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import rri_nmf_b200 as R         # noqa: E402


def tf32(x):
    b = x.view(torch.int32)
    return ((b + 0xfff + ((b >> 13) & 1)) & ~0x1fff).view(torch.float32)      # nearest, ties to even (finite inputs)


dev = torch.device('cuda:0')
torch.manual_seed(0)
for (M, N, K) in [(20000, 64, 20000), (20000, 64, 200000), (4096, 128, 50000)]:
    A = torch.rand(M, K, device=dev).clamp_(min=2.0 ** -20)     # (torch.rand reaches below 2^-30 of its maximum)
    B = torch.rand(N, K, device=dev)
    eng = R.RRIEngine(A, N, order='hals', math='tf32')
    assert eng.stats()['x_operand'] == 'f16'
    Cr = tf32(A).double() @ tf32(B).double().t()
    for name, C in (('f32 map', eng.gemm_nt(A, B)), ('f16 copy', eng.contract_x(B))):
        torch.cuda.synchronize()
        D = C.double() - Cr
        print('M=%d N=%d K=%d %-8s relfro=%.3e mean_signed_rel=%+.3e' % (M, N, K, name, float(D.norm() / Cr.norm()),
                                                                      float((D / Cr).mean())), flush=True)
    eng.close()
    del A, B, Cr
