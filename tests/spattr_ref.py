"""ShortestPathAttr (metric=np.dot) as one dense fp64 feature matrix, on the CPU (no device, no reference needed).

The kernel is bilinear in the attributes: k(x, y) = sum_d <F_x[d], F_y[d]> with F[d] = sum_{(i,j): S[i,j]=d} a_i (x) a_j
(SPAttrOracle._maps).  `spattr_phi` lays the per-graph maps out as rows of one matrix Phi -- one flattened da x da block
per distinct path length of the union, in ascending order, as the device does -- so that

* K_ref = Phi Phi^T is the kernel matrix in fp64,
* K_abs = |Phi| |Phi|^T is the scale the tensor-core Gram's error bound is stated against (equal to K_ref when all
  attributes are non-negative),
* diag = <Phi_i, Phi_i>, correctly rounded (math.fsum), is the exact self similarity.
"""
import math

import numpy as np

from oracle.gk_oracle import SPAttrOracle


def spattr_phi(X, Y=None, algorithm_type="auto"):
    """Dense fp64 feature matrix of X (and of Y below it, the rows `transform` adds)."""
    o = SPAttrOracle(algorithm_type=algorithm_type)
    maps = o._maps(X) + (o._maps(Y) if Y is not None else [])
    dists = sorted(set().union(*(m.keys() for m in maps)))
    da = next((f.shape[0] for m in maps for f in m.values()), 1)
    col = {d: b for b, d in enumerate(dists)}
    Phi = np.zeros((len(maps), max(len(dists), 1) * da * da))
    for r, m in enumerate(maps):
        for d, f in m.items():
            b = col[d]
            Phi[r, b * da * da:(b + 1) * da * da] = np.asarray(f, dtype=float).ravel()
    return Phi


def spattr_gram_ref(Phi, n_fit=None):
    """fit_transform (n_fit None or all rows): the square K of all rows; transform: rows n_fit.. against rows ..n_fit.
    Returns (K_ref, K_abs, row self similarities, column self similarities)."""
    n = Phi.shape[0]
    n_fit = n if n_fit is None else n_fit
    diag = np.array([math.fsum(x * x for x in row) for row in Phi])
    R = Phi if n_fit == n else Phi[n_fit:]
    C = Phi[:n_fit]
    K = R @ C.T
    K_abs = np.abs(R) @ np.abs(C).T
    drow = diag if n_fit == n else diag[n_fit:]
    if n_fit == n:
        np.fill_diagonal(K, diag)
    return K, K_abs, drow, diag[:n_fit]


def spattr_ref(X, Y=None, algorithm_type="auto", normalize=False):
    """K_ref (normalised as the reference does it when `normalize`) for fit_transform(X), or for transform(Y) after
    fit(X), with its error scale K_abs (divided by the same sqrt(d_i d_j) when `normalize`) and the self similarities
    (rows, columns)."""
    Phi = spattr_phi(X, Y, algorithm_type)
    K, K_abs, drow, dcol = spattr_gram_ref(Phi, None if Y is None else len(X))
    if normalize:
        with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
            s = np.sqrt(np.outer(drow, dcol))
            K, K_abs = K / s, K_abs / s
    return K, K_abs, drow, dcol
