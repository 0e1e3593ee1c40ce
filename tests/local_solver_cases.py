"""Dense systems for the interaction-region solvers (csrc/node_kernels.cuh), a NumPy replay of the pivot decisions of
the blocked solver ``TileGJ``, and an extended-precision reference solve.

The assembly scales every row of a local system to unit 1-norm before the solve (phase 3 of ``mpfa_node``), and so do
the generators here.  ``TileGJ`` takes pivots four columns at a time (a "panel").  Its fast path accepts the panel's
natural 4 x 4 diagonal block of the current Schur complement when none of its rows has been a pivot row yet and the
largest entry of the block's inverse, rounded to float, is <= ``GROWTH``; otherwise it runs partial pivoting on the
panel (the slow path).  ``panel_paths`` replays that decision, so that each family below can state, and the tests can
check, which path every panel takes.

Families (all return ``(M, info)`` with ``M`` row-scaled, float64):

* ``family_f``  strictly diagonally dominant: the fast path on every panel.
* ``family_s``  rows of a family-F matrix shifted by four, with zero blocks that make every natural diagonal block
  exactly singular or already used: the slow path on every panel.
* ``family_m_gauss`` Gaussian; ``family_m_panel`` family F except that panel k fails the growth test.
* ``family_g``  the growth of panel 0 placed just below / just above ``GROWTH``, also across the float rounding.
* ``family_c``  family F with the four columns of one panel scaled by 10^-e (rows scaled again afterwards).
* ``singular_*`` exactly singular systems whose elimination is exact in binary floating point, so that every
  elimination order meets an exact zero pivot.  (A generic singular matrix is, after rounding, a nearly singular one
  for every LU, the reference's ``np.linalg.inv`` included: only exact structures can be required to be refused.)
* ``nonfinite`` a NaN or an Inf in the system.
"""
from __future__ import annotations

import numpy as np
import scipy.linalg as sla

GROWTH = 64.0
U = np.finfo(np.float64).eps / 2


def row_scale(M: np.ndarray) -> np.ndarray:
    s = np.abs(M).sum(axis=1)
    return M / s[:, None]


# ---------------------------------------------------------------------------------------------------------------------
# reference solve
# ---------------------------------------------------------------------------------------------------------------------
def ref_solve(M: np.ndarray, B: np.ndarray, iters: int = 4) -> np.ndarray:
    """float64 LU with partial pivoting, then iterative refinement with residuals in np.longdouble."""
    lu = sla.lu_factor(M)
    X = sla.lu_solve(lu, B)
    Ml, Bl = M.astype(np.longdouble), B.astype(np.longdouble)
    for _ in range(iters):
        R = Bl - Ml @ X.astype(np.longdouble)
        X = X + sla.lu_solve(lu, R.astype(np.float64))
    return X


def cond_inf(M: np.ndarray) -> float:
    return float(np.abs(M).sum(axis=1).max() * np.abs(np.linalg.inv(M)).sum(axis=1).max())


def error_ratio(X: np.ndarray, Xref: np.ndarray, M: np.ndarray, kappa: float | None = None) -> float:
    """max|X - Xref| / max|Xref|  over the bound 50 n u kappa_inf(M)."""
    n = M.shape[0]
    k = cond_inf(M) if kappa is None else kappa
    err = np.abs(X - Xref).max() / np.abs(Xref).max()
    return float(err / (50.0 * n * U * k))


# ---------------------------------------------------------------------------------------------------------------------
# replay of TileGJ's panel decisions
# ---------------------------------------------------------------------------------------------------------------------
def _block_growth(blk: np.ndarray) -> float:
    """invert_block: Gauss-Jordan on the 4 x 4 block in its natural row order (no pivoting), then the largest
    |entry| rounded to float32.  inf / nan when a pivot is zero or not finite."""
    m = blk.astype(np.float64).copy()
    iv = np.eye(4)
    with np.errstate(all="ignore"):
        for k in range(4):
            inv = 1.0 / m[k, k]
            m[k] *= inv
            iv[k] *= inv
            for j in range(4):
                if j != k:
                    f = m[j, k]
                    m[j] -= f * m[k]
                    iv[j] -= f * iv[k]
        a = np.abs(iv)
        if not np.all(np.isfinite(a)):
            return float("inf")
        return float(np.float32(a.max()))


def panel_paths(M: np.ndarray) -> list:
    """Per panel: "fast", "slow", or "singular" (the replay stops there).  Partial pivoting on exact magnitudes."""
    n = M.shape[0]
    S = M.astype(np.float64).copy()
    used = np.zeros(n, bool)
    out = []
    for q in range((n + 3) // 4):
        p0 = 4 * q
        pw = min(4, n - p0)
        nat = np.arange(p0, p0 + pw)
        blk = np.eye(4)
        blk[:pw, :pw] = S[np.ix_(nat, nat)]
        fast = (not used[nat].any()) and _block_growth(blk) <= GROWTH
        if fast:
            piv = list(nat)
        else:
            P = S[:, p0:p0 + pw].copy()
            avail = ~used
            piv = []
            for j in range(pw):
                mag = np.where(avail, np.abs(P[:, j]), -1.0)
                r = int(np.argmax(mag))
                if not mag[r] > 0:
                    out.append("singular")
                    return out
                piv.append(r)
                avail[r] = False
                f = P[:, j] / P[r, j]
                f[r] = 0.0
                f[~avail] = 0.0
                P -= np.outer(f, P[r])
        out.append("fast" if fast else "slow")
        piv = np.array(piv)
        A11 = S[np.ix_(piv, np.arange(p0, p0 + pw))]
        if not np.all(np.isfinite(A11)) or np.linalg.matrix_rank(A11) < pw:
            out[-1] = "singular"
            return out
        others = np.setdiff1d(np.where(~used)[0], piv)
        R = np.linalg.solve(A11, S[piv, p0:])
        S[others, p0:] -= S[others, p0:p0 + pw] @ R
        used[piv] = True
    return out


# ---------------------------------------------------------------------------------------------------------------------
# families
# ---------------------------------------------------------------------------------------------------------------------
def family_f(n: int, seed: int = 0, off: float = 0.5) -> np.ndarray:
    """Strictly diagonally dominant: off-diagonal mass `off` times the diagonal in every row, random signs."""
    rng = np.random.default_rng(seed)
    M = rng.uniform(-1.0, 1.0, (n, n))
    np.fill_diagonal(M, 0.0)
    s = np.abs(M).sum(axis=1)
    s[s == 0] = 1.0
    M *= (off / s)[:, None]
    np.fill_diagonal(M, rng.choice([-1.0, 1.0], n) * rng.uniform(1.0, 2.0, n))
    return row_scale(M)


def family_s(n: int, seed: int = 0) -> np.ndarray:
    """Rows of a family-F matrix F shifted down by four (row i of M is row i - 4 of F, cyclically), with
    F[n-4:, :4] = 0.  Panel 0's natural block (F's last four rows in its columns) is zero; from then on, panel q's
    natural rows hold F's rows of panel q - 1, which panel q - 1 has taken as pivots.  Needs n >= 8."""
    assert n >= 8
    F = family_f(n, seed)
    F[n - 4:, :4] = 0.0
    F = row_scale(F)
    return np.roll(F, 4, axis=0)


GAUSS_SEEDS = 8   # from n = 8 on, at least one of these seeds has a slow panel and every one a fast panel


def family_m_gauss(n: int, seed: int = 0) -> np.ndarray:
    return row_scale(np.random.default_rng(1000 + seed).standard_normal((n, n)))


def _bad_block(M: np.ndarray, q: int, delta: float) -> np.ndarray:
    """Rows 4q, 4q+1 of panel q become [1, 1] and [1, 1 + delta] in the panel's first two columns (plus the small
    off-diagonal rest); the other rows' entries in those columns are damped, so that partial pivoting still picks
    the natural rows while the natural-order inverse has entries of about 2 (1 + delta) / delta."""
    M = M.copy()
    n = M.shape[0]
    a, b = 4 * q, 4 * q + 1
    cols = [a, b]
    rest = np.setdiff1d(np.arange(n), [a, b])
    M[np.ix_(rest, cols)] *= 0.05
    sa = np.abs(M[a]).sum() - np.abs(M[a, cols]).sum()
    sb = np.abs(M[b]).sum() - np.abs(M[b, cols]).sum()
    M[a] *= 0.01 / max(sa, 1e-300)
    M[b] *= 0.01 / max(sb, 1e-300)
    M[a, a], M[a, b] = 1.0, 1.0
    M[b, a], M[b, b] = 1.0, 1.0 + delta
    return row_scale(M)


def family_m_panel(n: int, k: int, seed: int = 0) -> np.ndarray:
    """Family F except that panel k (which must hold at least two columns) fails the growth test."""
    return _bad_block(family_f(n, seed, off=0.2), k, 0.01)


def panel_growth(M: np.ndarray, q: int = 0) -> float:
    """Growth of panel q's natural block in double precision (before the float rounding), assuming the fast path
    on the panels before it."""
    S = M.astype(np.float64).copy()
    n = M.shape[0]
    for p in range(q):
        nat = np.arange(4 * p, min(4 * p + 4, n))
        others = np.arange(nat[-1] + 1, n)
        R = np.linalg.solve(S[np.ix_(nat, nat)], S[nat, nat[0]:])
        S[others, nat[0]:] -= S[np.ix_(others, nat)] @ R
    nat = np.arange(4 * q, min(4 * q + 4, n))
    pw = nat.size
    blk = np.eye(4)
    blk[:pw, :pw] = S[np.ix_(nat, nat)]
    return float(np.abs(np.linalg.inv(blk)).max())


# growth targets of family G: (target, path).  Float32 spacing above 64 is 2^-17 = 7.6e-6: 64 + 3e-6 rounds to 64
# (fast, although above the threshold in double), 64 + 5e-6 rounds to 64 + 7.6e-6 (slow).
G_TARGETS = ((64.0 - 1e-4, "fast"), (64.0 - 1e-9, "fast"), (64.0 + 3e-6, "fast"), (64.0 + 5e-6, "slow"),
             (64.0 + 1e-3, "slow"))


def family_g(n: int, target: float, seed: int = 0) -> np.ndarray:
    """Panel 0's growth tuned to `target` by bisection on delta of ``_bad_block``.  Needs n >= 2."""
    base = family_f(n, seed, off=0.2)
    lo, hi = 1e-4, 1.0   # growth decreases with delta
    for _ in range(200):
        mid = 0.5 * (lo + hi)
        g = panel_growth(_bad_block(base, 0, mid))
        if g > target:
            lo = mid
        else:
            hi = mid
        if hi - lo < 1e-17 * hi:
            break
    return _bad_block(base, 0, hi)


C_EXPONENTS = (0, 3, 6, 9, 12)


def graded_panel(n: int) -> int:
    return ((n + 3) // 4) // 2


def family_c(n: int, e: int, seed: int = 0):
    """Family F with the columns of panel ``graded_panel(n)`` scaled by 10^-e, rows scaled again.  Returns
    ``(M, Mu, d)``: M = Mu diag(d), Mu the row-scaled matrix before the column scaling; then  d * X(M) = X(Mu)."""
    F = family_f(n, seed)
    q = graded_panel(n)
    d = np.ones(n)
    d[4 * q:min(4 * q + 4, n)] = 10.0 ** (-e)
    s = np.abs(F * d[None, :]).sum(axis=1)
    Mu = F / s[:, None]
    return Mu * d[None, :], Mu, d


# ---- exactly singular systems (dyadic entries: every elimination order meets an exact zero pivot)
def singular_duplicate_row(n: int, seed: int = 0) -> np.ndarray:
    """Rows n-2 and n-1 identical ([0.5, 0.5] in the last two columns), a family-F block above.  Needs n >= 2."""
    M = family_f(n, seed)
    M[n - 2:, :] = 0.0
    M[n - 2:, n - 2:] = 0.5
    return M


def singular_last_panel(n: int, seed: int = 0) -> np.ndarray:
    """n = 3 mod 4: the last, partial panel (three columns) holds a rank-2 block whose third row is the difference of
    the first two; the leading (n-3) x (n-3) block is family F."""
    assert n % 4 == 3
    M = family_f(n, seed)
    M[n - 3:, :] = 0.0
    M[n - 3:, n - 3:] = [[0.5, 0.5, 0.0], [0.5, 0.0, 0.5], [0.0, -0.5, 0.5]]
    return M


def singular_zero_column(n: int, seed: int = 0) -> np.ndarray:
    """Column 4 * (last full panel) + 1 is zero (column n-1 when n < 4)."""
    M = family_f(n, seed)
    q = max(n // 4 - 1, 0)
    c = min(4 * q + 1, n - 1)
    M[:, c] = 0.0
    return row_scale(M)


def nonfinite(n: int, kind: str, seed: int = 0) -> np.ndarray:
    M = family_f(n, seed)
    i = n // 2
    M[i, (i + 1) % n] = np.nan if kind == "nan" else np.inf
    return M


def rhs(n: int, ncol: int, seed: int = 0) -> np.ndarray:
    return np.random.default_rng(500 + seed).standard_normal((n, ncol))


def sizes(max_n: int, cap: int | None = None) -> list:
    """n = 1..9, the neighbours of every multiple of 8 (tile and warp edges; all remainders mod 4 occur), and
    max_n - 1, max_n."""
    top = max_n if cap is None else min(max_n, cap)
    s = set(range(1, min(9, top) + 1))
    for m in range(8, top + 2, 8):
        s.update((m - 1, m, m + 1))
    s.update((top - 1, top))
    return sorted(x for x in s if 1 <= x <= top)
