"""rri_nmf_b200 -- B200-native (sm_100a) rank-one-residue-iteration NMF sweep engine.

Drop-in for the hot path of maksimt/rri_nmf: `nmf(X, k, **kwargs) -> dict` (reference
src/rri_nmf/nmf.py:98-560) and the sklearn-style estimators (src/rri_nmf/sklearn_interface.py),
running on hand-written CUDA kernels behind the C-ABI of include/rri_b200.h.
"""
from .nmf import nmf, nmf_models, eps_div_by_zero          # noqa: F401
from .engine import RRIEngine                               # noqa: F401
from .sklearn_interface import NMF_TM_Estimator, NMF_RS_Estimator   # noqa: F401

__all__ = ['nmf', 'nmf_models', 'RRIEngine', 'NMF_TM_Estimator', 'NMF_RS_Estimator', 'eps_div_by_zero']
