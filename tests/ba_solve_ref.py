"""Matrix generators and a high-precision referee for the reduced-camera-system solve (k_ba_solve, oracle ldlt_solve).

The three families cover what the solver meets and where an LDL^T without pivoting loses accuracy:
  dense_spd   M M^T / n + I: well conditioned, every entry non-zero (short panels, full trailing updates)
  ba_shaped   6x6 pose blocks, banded co-visibility with wrap-around (the windows synth.ba_problem draws), J^T J + lambda I; the relative
              constraints leave the 6-dim gauge of BA, so lambda sets the smallest eigenvalue and with it kappa (up to ~1e6, like early LM trials)
  graded      D^1/2 A D^1/2 with D log-uniform over 1e-4 .. 1e4: entries spanning 16 orders of magnitude (only a backward-error gate applies)
"""
import numpy as np

U = 2.0 ** -53          # unit roundoff of fp64
LD = np.longdouble


def dense_spd(n, seed=0):
    rng = np.random.default_rng(1000 + n + 7919 * seed)
    M = rng.standard_normal((n, n))
    return M @ M.T / n + np.eye(n)


def ba_shaped(n, kappa=1e6, band=6, seed=0):
    """Leading n x n block of a BA-shaped system over ceil(n/6) poses: pose j is co-visible with j+1 .. j+band (mod the pose count); every
    co-visible pair contributes A^T A for a random 6 x 12 relative Jacobian A (rotation columns scaled up like the image Jacobians). For n a
    multiple of 6 and at least two poses, kappa_2 is `kappa` up to rounding."""
    rng = np.random.default_rng(2000 + n + 7919 * seed)
    nb = -(-n // 6)
    H = np.zeros((6 * nb, 6 * nb))
    col = np.array([4.0, 4.0, 4.0, 1.0, 1.0, 1.0])
    pairs = sorted({(min(i, (i + d) % nb), max(i, (i + d) % nb)) for i in range(nb) for d in range(1, band + 1) if (i + d) % nb != i})
    for i, j in pairs:
        A = rng.standard_normal((6, 6)) * col
        J = np.concatenate([A, -A], 1)                # observes x_i - x_j only
        idx = np.r_[6 * i:6 * i + 6, 6 * j:6 * j + 6]
        H[np.ix_(idx, idx)] += J.T @ J
    if nb == 1:                                       # a lone pose: one absolute observation
        A = rng.standard_normal((6, 6)) * col
        H += A.T @ A
    # relative constraints leave the gauge (all poses moved together) free: lambda alone lifts it, as the LM damping does
    ev = np.linalg.eigvalsh(H)
    lam = max(ev[-1] / kappa - ev[0], ev[-1] * U)
    S = H + lam * np.eye(6 * nb)
    return np.ascontiguousarray(S[:n, :n])


def graded(n, seed=0):
    rng = np.random.default_rng(3000 + n + 7919 * seed)
    d = np.sqrt(10.0 ** rng.uniform(-4, 4, n))
    return dense_spd(n, seed) * d[:, None] * d[None, :]


FAMILIES = {"dense_spd": dense_spd, "ba_shaped": ba_shaped, "graded": graded}


def rhs(n, seed=0):
    return np.random.default_rng(4000 + n + 7919 * seed).standard_normal(n)


def pack(S, g):
    """(n+1) x n layout the solver reads: S, then g as row n."""
    return np.ascontiguousarray(np.vstack([S, g[None, :]]))


def residual(S, g, x):
    """g - S x in long double."""
    return g.astype(LD) - S.astype(LD) @ np.asarray(x).astype(LD)


def reference_solve(S, g):
    """x*: the fp64 LAPACK solve plus two steps of iterative refinement, residuals and the accumulated solution in long double."""
    x = np.linalg.solve(S, g).astype(LD)
    for _ in range(2):
        x = x + np.linalg.solve(S, residual(S, g, x).astype(np.float64)).astype(LD)
    return x


def backward_error(S, g, x):
    """Normwise backward error eta = ||g - S x||_inf / (||S||_inf ||x||_inf + ||g||_inf)."""
    r = residual(S, g, x)
    nS = np.abs(S).sum(1).max()
    return float(np.abs(r).max() / (LD(nS) * np.abs(np.asarray(x).astype(LD)).max() + LD(np.abs(g).max())))


def forward_error(x, xref):
    xref = np.asarray(xref).astype(LD)
    return float(np.abs(np.asarray(x).astype(LD) - xref).max() / np.abs(xref).max())


def kappa_inf(S):
    return float(np.abs(S).sum(1).max() * np.abs(np.linalg.inv(S)).sum(1).max())


def zero_pivot(S, k):
    """S with row and column k zeroed: the k-th pivot of any LDL^T is exactly 0."""
    S = S.copy()
    S[k, :] = 0.0
    S[:, k] = 0.0
    return S
