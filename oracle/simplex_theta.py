"""NumPy model of the blocked simplex threshold of the block-order T update with project_T_each_iter
(rri_nmf_b200/csrc/simplex_kernels.cu: simplex_T_fused_kernel, grid_michelot).

TEST INFRASTRUCTURE ONLY (tests/test_simplex_theta_cpu.py).  The kernel holds one entry of the vector per thread,
`nblocks` blocks of threads.  Michelot's iteration
    theta <- (sum_{x_i > theta} x_i - s) / |{x_i > theta}|,   from theta = -inf (every entry active),
stops when a round finds the active set unchanged.  Every round is one grid-wide reduction: each block sums its own
entries, the block partials go to one slot per block, and after a grid barrier every block adds the slots in block
order -- so every block derives the same theta.  The projection is max(x - theta, 0); its threshold equals the one
of the sort-based projection (rri_oracle.euclidean_proj_simplex, matrixops.py:5-69).
"""
import numpy as np


def _round(x, theta, nblocks):
    """one reduction round: (sum, count) of the active entries, block partials added in block order"""
    tot, cnt = 0.0, 0.0
    for part in np.array_split(np.asarray(x, dtype=np.float64), nblocks):
        act = part > theta
        tot += float(np.sum(part[act]))
        cnt += float(np.count_nonzero(act))
    return tot, cnt


def blocked_theta(x, s=1.0, nblocks=1, theta=-1e300, prev_cnt=-1.0):
    """the kernel's threshold for x split into nblocks blocks; returns (theta, rounds)"""
    rounds = 0
    while True:
        tot, cnt = _round(x, theta, nblocks)
        rounds += 1
        if cnt == prev_cnt or cnt == 0.0:
            return theta, rounds
        prev_cnt = cnt
        theta = (tot - s) / cnt


def blocked_proj_simplex(x, s=1.0, nblocks=1):
    """max(x - theta, 0) with the blocked threshold"""
    theta, _ = blocked_theta(x, s, nblocks)
    return np.maximum(np.asarray(x, dtype=np.float64) - theta, 0.0)


def topic_data(n, d, k, s=1.0, seed=0):
    """a topic-model-like problem for the block order with project_T_each_iter: X = W T (+ a little noise) with
    Dirichlet rows of W (sum 1) and of T (sum s), and a start (W0, T0) near them.  (Uniform synthetic data with a
    random start empties topics within a few constrained sweeps -- the reference then asserts, nmf.py:476.)"""
    rs = np.random.RandomState(seed)
    Wt = rs.dirichlet(np.full(k, 0.2), n)
    Tt = rs.dirichlet(np.full(d, 0.1), k)
    X = Wt.dot(Tt) * s + 0.01 * rs.rand(n, d) / d
    W0 = Wt + 0.2 * rs.rand(n, k)
    W0 /= W0.sum(1, keepdims=True)
    T0 = Tt + 0.2 * rs.rand(k, d) / d
    T0 *= s / T0.sum(1, keepdims=True)
    return X, W0, T0
