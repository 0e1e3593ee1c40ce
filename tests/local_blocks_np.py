"""NumPy twin of ``porepy_b200.krylov.LocalBlocks`` (csrc/local_blocks.cu) for the CPU tests: the same block
gather, pivot test and application on a scipy matrix and CPU torch tensors.  Test infrastructure only: the product
never imports it."""
from __future__ import annotations

import numpy as np
import scipy.sparse as sps


def block_inverses(a, layout, pivot_rel: float = 1e-14):
    """List of B_b^-1 = A[rows_b, cols_b]^-1 (Gauss-Jordan with partial pivoting, as the kernel does it); raises the
    kernel's ``ValueError`` naming the first block with a non-finite entry, a pivot that is not finite or
    <= pivot_rel max|B_b|, or a non-finite inverse."""
    a = sps.csr_matrix(a)
    out = []
    for b in range(len(layout.ptr) - 1):
        r = layout.rows[layout.ptr[b]:layout.ptr[b + 1]]
        c = layout.cols[layout.ptr[b]:layout.ptr[b + 1]]
        B = a[r][:, c].toarray()
        s = B.shape[0]
        if not np.isfinite(B).all():
            raise ValueError(f"Error in inversion of local linear systems (block {b} is singular or not finite (a zero or non-finite pivot, entry or inverse))")
        amax = np.abs(B).max() if B.size else 0.0
        M = np.hstack((B, np.eye(s)))
        for k in range(s):
            p = k + int(np.argmax(np.abs(M[k:, k])))
            piv = M[p, k]
            if not np.isfinite(piv) or not abs(piv) > pivot_rel * amax:
                raise ValueError(f"Error in inversion of local linear systems (block {b} is singular or not finite (a zero or non-finite pivot, entry or inverse))")
            M[[k, p]] = M[[p, k]]
            M[k] /= piv
            f = M[:, k].copy()
            f[k] = 0.0
            M -= np.outer(f, M[k])
        if not np.isfinite(M[:, s:]).all():
            raise ValueError(f"Error in inversion of local linear systems (block {b} is singular or not finite (a zero or non-finite pivot, entry or inverse))")
        out.append(M[:, s:])
    return out


class NumpyLocalBlocks:
    """``factor(J)`` (scipy matrix, or anything with ``to_scipy``) / ``apply(r, out)`` on CPU torch tensors."""

    def __init__(self, layout):
        self.layout = layout
        self.n = int(layout.ptr[-1])
        self.inv = None

    def factor(self, J):
        self.inv = block_inverses(J.to_scipy() if hasattr(J, "to_scipy") else J, self.layout)
        return self

    def apply(self, r, out=None):
        import torch
        rh = r.detach().cpu().numpy()
        z = np.empty(self.n)
        L = self.layout
        for b, m in enumerate(self.inv):
            z[L.cols[L.ptr[b]:L.ptr[b + 1]]] = m @ rh[L.rows[L.ptr[b]:L.ptr[b + 1]]]
        zt = torch.as_tensor(z, dtype=r.dtype)
        if out is None:
            return zt
        out.copy_(zt)
        return out
