"""Numpy restatement of the LOBPCG block kernels (csrc/modes.cu) -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

`NumpyBackend` has the methods of femb200.modes.DeviceBackend on [n, ld] row-major numpy arrays, so the whole driver
(femb200.modes.lobpcg) runs on a CPU-only machine and, on the GPU, each kernel can be compared with its restatement.
`assemble_bsr3` builds K and M on one node-level 3x3 block pattern from element matrices, as the device assembly does.
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp


def node_pattern(elements, n_nodes):
    """(brow [nb+1], bcol [nnzb]) int32 of the node graph of the connectivity (every node pair of an element), columns ascending."""
    e = np.asarray(elements, dtype=np.int64)
    nen = e.shape[1]
    a = np.repeat(e, nen, axis=1).reshape(-1)
    b = np.tile(e, (1, nen)).reshape(-1)
    keys = np.unique(a * n_nodes + b)
    rows, cols = keys // n_nodes, keys % n_nodes
    brow = np.zeros(n_nodes + 1, dtype=np.int64)
    np.add.at(brow, rows + 1, 1)
    return np.cumsum(brow).astype(np.int32), cols.astype(np.int32)


def assemble_bsr3(Ke, elements, n_nodes, pattern=None):
    """Block values bval [nnzb, 3, 3] of sum_e K_e on the node pattern (element-ascending sums)."""
    brow, bcol = pattern if pattern is not None else node_pattern(elements, n_nodes)
    e = np.asarray(elements, dtype=np.int64)
    M, nen = e.shape
    Ke = np.asarray(Ke, dtype=np.float64).reshape(M, nen, 3, nen, 3).transpose(0, 1, 3, 2, 4)   # [M, a, b, 3, 3]
    rows = np.repeat(e, nen, axis=1).reshape(-1)
    cols = np.tile(e, (1, nen)).reshape(-1)
    keys = np.arange(len(brow) - 1).repeat(np.diff(brow)) * n_nodes + bcol
    slot = np.searchsorted(keys, rows * n_nodes + cols)
    bval = np.zeros((bcol.size, 3, 3))
    np.add.at(bval, slot, Ke.reshape(-1, 3, 3))
    return bval


def bsr_matrix(brow, bcol, bval):
    nb = len(brow) - 1
    return sp.bsr_matrix((bval, bcol, brow), shape=(3 * nb, 3 * nb))


def dof_mask(n_nodes, fixed):
    mask = np.ones((n_nodes, 3), dtype=np.uint8)
    if fixed is not None and np.asarray(fixed).size:
        mask[np.asarray(fixed)] = 0
    return mask.reshape(-1)


class NumpyBackend:
    """femb_spmm_bsr3 / femb_mb_gram / femb_mb_combine / femb_lobpcg_residual restated with numpy."""

    def __init__(self, brow, bcol, kval, mval, mask):
        self.K = bsr_matrix(brow, bcol, kval).tocsr()
        self.M = bsr_matrix(brow, bcol, mval).tocsr()
        self.mask = np.asarray(mask, dtype=np.uint8)
        self.n = self.K.shape[0]
        d = self.K.diagonal()
        self.dinv = np.where((self.mask != 0) & (d != 0), 1.0 / np.where(d != 0, d, 1.0), 0.0)
        self.norm_K = float(abs(self.K).sum(axis=1).max())
        self.norm_M = float(abs(self.M).sum(axis=1).max())

    def zeros(self, rows, cols):
        return np.zeros((rows, cols))

    def upload(self, a):
        return np.array(a, dtype=np.float64)

    def host(self, t):
        return np.array(t)

    def mask_host(self):
        return self.mask

    def spmm(self, X, c0, k, YK, YM):
        f = self.mask[:, None].astype(np.float64)
        x = X[:, c0:c0 + k] * f
        YK[:, c0:c0 + k] = (self.K @ x) * f
        if YM is not None:
            YM[:, c0:c0 + k] = (self.M @ x) * f

    def gram(self, A, B, k, G):
        G[:k * k] = (A[:, :k].T @ B[:, :k]).reshape(-1)

    def combine(self, X, k, Cm, Y, c0, beta=0.0):
        Cm = np.asarray(Cm, dtype=np.float64)
        mc = Cm.shape[1]
        out = X[:, :k] @ Cm
        Y[:, c0:c0 + mc] = beta * Y[:, c0:c0 + mc] + out if beta != 0.0 else out

    def residual(self, X, KX, MX, m, lam, active, na, W, c0, norms):
        R = KX[:, :m] - MX[:, :m] * np.asarray(lam, dtype=np.float64)[None, :m]
        norms[:m] = (R * R).sum(axis=0)
        norms[m:2 * m] = (X[:, :m] * X[:, :m]).sum(axis=0)
        if na:
            W[:, c0:c0 + na] = self.dinv[:, None] * R[:, np.asarray(active)[:na]]

    def active_list(self, cols):
        return np.asarray(cols, dtype=np.int32)
