"""CPU restatement (numpy) of the reference's ``rdsampler`` -- TEST INFRASTRUCTURE.

Only ``tests/`` and ``profiles/`` may import this module; the product (``pygho_b200``) never
does.  Unlike ``hodata_oracle`` it has no golden vectors: ``tests/test_rd_oracle_cpu.py``
checks it against closed forms instead.
"""
from __future__ import annotations

import numpy as np


def rd_matrix(edge_index: np.ndarray, num_nodes: int) -> np.ndarray:
    """rdsampler (MaTupleSampler.py:34-57): resistance distances ``L+_ii + L+_jj - 2 L+_ij`` of
    the SIMPLE undirected graph (both directions one edge, duplicates once, self-loops dropped),
    ``L+ = pinv(D - A)`` in fp64; (n, n).

    The cutoff is 1e-10 of the largest eigenvalue, not numpy's default 1e-15: the null
    eigenvalue of a Laplacian comes out of ``eigh`` at about n * eps * lambda_max (-8.9e-15 for
    K_12, whose R is then off by 1.3e-3), while the smallest non-zero one of a graph of up to
    128 nodes is above 1e-6 of the largest."""
    n = num_nodes
    A = np.zeros((n, n), dtype=np.float64)
    A[edge_index[0], edge_index[1]] = 1.0
    A[edge_index[1], edge_index[0]] = 1.0
    np.fill_diagonal(A, 0.0)
    P = np.linalg.pinv(np.diag(A.sum(1)) - A, rcond=1e-10, hermitian=True)
    d = np.diag(P)
    R = d[:, None] + d[None, :] - 2.0 * P
    np.fill_diagonal(R, 0.0)
    return R
