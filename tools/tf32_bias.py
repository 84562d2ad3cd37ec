"""Signed bias of the TF32 contraction against an fp64 product for long K (accumulation-chain check).
python tools/tf32_bias.py"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import rri_nmf_b200 as R
dev = torch.device("cuda:0")
torch.manual_seed(0)
for (M, N, K) in [(1000, 64, 2000), (20000, 64, 20000), (20000, 64, 200000), (4096, 128, 50000), (3000, 10, 70000), (2000, 200, 30000)]:
    A = torch.rand(M, K, device=dev); B = torch.rand(N, K, device=dev)
    eng = R.RRIEngine(torch.zeros(8, 8, device=dev), N, order="hals", math="tf32")
    C = eng.gemm_nt(A, B); torch.cuda.synchronize()
    Cr = A.double() @ B.double().t()
    print("M=%d N=%d K=%d relfro=%.3e mean_signed_rel=%+.3e" % (M, N, K, float((C.double() - Cr).norm() / Cr.norm()),
                                                               float(((C.double() - Cr) / Cr).mean())), flush=True)
    eng.close(); del A, B, C, Cr
