"""Plain NumPy / SciPy restatement of the explicit 2-form assembly of the Helmholtz family,
``alpha*inner(grad u, grad v)*dx + beta*inner(u, v)*dx`` on Q_p (x) P_p hexahedra with trilinear
geometry, as PyOP2 assembles it into a PETSc AIJ / BAIJ matrix:

* the pattern is the union over every cell of the sparsity's map of (row node, column node),
  plus the diagonal (pyop2/sparsity.pyx);
* each visited cell adds its element matrix with MatSetValuesLocal semantics: a row or column
  whose local-to-global index is negative is dropped;
* ``set_local_diagonal_entries`` then writes the diagonal of the constrained rows;
* a vector-valued space of block size bs holds A (x) I_bs.

Nothing here imports the engine, its sources or ``oracle/``: the element matrices are formed
from the 1-D tables of ``fiat_lite`` by batched float64 matmuls, the pattern by ``np.unique``.
"""
import numpy as np
import scipy.sparse as sp

from firedrake_b200.fiat_lite import interval_element

CHUNK = 64                         # cells per batched matmul


def _tables(p):
    """Reference gradients (Q, nd, 3) and values (Q, nd) of the tensor basis at the tensor Gauss
    points, the derivatives of the 8 trilinear vertex functions (Q, 8, 3), and the weights (Q,)."""
    el = interval_element(p)
    n, B, D, xq, wq = el.ndof, el.B, el.D, el.xq, el.wq
    q = np.arange(n)
    # point index (qx, qy, qz) and dof index (ax, ay, az), both z fastest
    Bx, By, Bz = B[:, None, None, :, None, None], B[None, :, None, None, :, None], B[None, None, :, None, None, :]
    Dx, Dy, Dz = D[:, None, None, :, None, None], D[None, :, None, None, :, None], D[None, None, :, None, None, :]
    Q, nd = n ** 3, n ** 3
    val = (Bx * By * Bz).reshape(Q, nd)
    gref = np.stack([(Dx * By * Bz).reshape(Q, nd), (Bx * Dy * Bz).reshape(Q, nd),
                     (Bx * By * Dz).reshape(Q, nd)], axis=-1)
    xi = np.stack(np.meshgrid(xq[q], xq[q], xq[q], indexing="ij"), axis=-1).reshape(Q, 3)
    w = (wq[:, None, None] * wq[None, :, None] * wq[None, None, :]).reshape(Q)
    dN = np.empty((Q, 8, 3))
    for bx in (0, 1):
        for by in (0, 1):
            for bz in (0, 1):
                s = [xi[:, d] if b else 1.0 - xi[:, d] for d, b in enumerate((bx, by, bz))]
                ds = [1.0 if b else -1.0 for b in (bx, by, bz)]
                v = (bx * 2 + by) * 2 + bz
                dN[:, v] = np.stack([ds[0] * s[1] * s[2], s[0] * ds[1] * s[2], s[0] * s[1] * ds[2]], axis=-1)
    return gref, val, dN, w


def element_matrices(p, X, alpha, beta):
    """Element matrices (nc, nd, nd) of cells with vertex coordinates X (nc, 8, 3), vertex v =
    (bx*2 + by)*2 + bz.  A_c = M_c^T M_c with the rows of M_c the sqrt(w |det J|)-scaled
    physical gradients (times sqrt(alpha)) and values (times sqrt(beta)) at every point."""
    assert alpha >= 0.0 and beta >= 0.0
    gref, val, dN, w = _tables(p)
    X = np.asarray(X, dtype=np.float64)
    J = np.einsum("cva,qvd->cqad", X, dN)                     # J[a][d] = dx_a / dxi_d
    K = np.linalg.inv(J)                                      # K[d][a] = dxi_d / dx_a
    s = np.sqrt(w[None, :] * np.abs(np.linalg.det(J)))        # (nc, Q)
    G = np.einsum("qid,cqda->cqai", gref, K)                  # physical gradients, (nc, Q, 3, nd)
    rows = [np.sqrt(alpha) * s[:, :, None, None] * G,
            np.sqrt(beta) * s[:, :, None, None] * val[None, :, None, :]]
    M = np.concatenate(rows, axis=2).reshape(X.shape[0], -1, val.shape[1])
    return np.matmul(M.transpose(0, 2, 1), M)


class Cells:
    """The cells one loop visits: node indices (ncells, nd) and vertex indices (ncells, 8)."""

    def __init__(self, nodes, verts):
        self.nodes = np.asarray(nodes, dtype=np.int64)
        self.verts = np.asarray(verts, dtype=np.int64)

    @classmethod
    def extruded(cls, mesh, V, cols=None):
        """Every layer of base columns ``cols`` (default all, in order): PyOP2's extruded loop
        ``for col in cols: for layer in range(nz)``, node = map[col] + offset * layer."""
        nz = mesh.nz
        cols = np.arange(mesh.num_base_cells) if cols is None else np.asarray(cols, dtype=np.int64)
        lay = np.arange(nz, dtype=np.int64)
        nodes = V.cell_node_map[cols][:, None, :].astype(np.int64) + lay[None, :, None] * V.offset[None, None, :]
        verts = (mesh.coord_map[cols][:, None, :].astype(np.int64)
                 + lay[None, :, None] * mesh.coord_offset[None, None, :])
        return cls(nodes.reshape(-1, V.arity), verts.reshape(-1, 8))

    def __len__(self):
        return len(self.nodes)


def pattern(nrows, cells):
    """CSR pattern (rowptr int64, colidx int32) of every cell's node list x itself, plus the diagonal."""
    nd = cells.nodes.shape[1]
    r = np.repeat(cells.nodes, nd, axis=1).ravel()
    c = np.tile(cells.nodes, (1, nd)).ravel()
    d = np.arange(nrows, dtype=np.int64)
    keys = np.unique(np.concatenate([r * nrows + c, d * nrows + d]))
    rows, cols = np.divmod(keys, nrows)
    rowptr = np.zeros(nrows + 1, dtype=np.int64)
    np.cumsum(np.bincount(rows, minlength=nrows), out=rowptr[1:])
    return rowptr, cols.astype(np.int32)


def assemble(p, alpha, beta, coords, rowptr, colidx, cells, row_mask=None, col_mask=None, diag_rows=(),
             diag_val=1.0):
    """Values (nnz,) of the matrix on the pattern (rowptr, colidx) after adding the element matrices of
    ``cells`` (masked rows / columns dropped) and writing ``diag_val`` on the diagonal of ``diag_rows``."""
    nrows = len(rowptr) - 1
    keys = np.repeat(np.arange(nrows, dtype=np.int64), np.diff(rowptr)) * nrows + colidx
    vals = np.zeros(len(colidx))
    nd = cells.nodes.shape[1]
    coords = np.asarray(coords).reshape(-1, 3)
    for c0 in range(0, len(cells), CHUNK):
        nodes = cells.nodes[c0:c0 + CHUNK]
        A = element_matrices(p, coords[cells.verts[c0:c0 + CHUNK]], alpha, beta)
        r = np.repeat(nodes, nd, axis=1).ravel()               # A[c, i, j]: row node i, column node j
        c = np.tile(nodes, (1, nd)).ravel()
        a = A.ravel()
        keep = np.ones(len(a), dtype=bool)
        if row_mask is not None:
            keep &= ~row_mask[r]
        if col_mask is not None:
            keep &= ~col_mask[c]
        k = r[keep] * nrows + c[keep]
        pos = np.searchsorted(keys, k)
        assert np.array_equal(keys[pos], k), "an element entry lies outside the pattern"
        vals += np.bincount(pos, weights=a[keep], minlength=len(vals))
    rows = np.asarray(diag_rows, dtype=np.int64)
    if len(rows):
        pos = np.searchsorted(keys, rows * nrows + rows)
        vals[pos] = diag_val
    return vals


def diagonal(p, alpha, beta, coords, nrows, cells):
    """diag(A) of the unmasked matrix: the element diagonals summed onto their nodes."""
    out = np.zeros(nrows)
    coords = np.asarray(coords).reshape(-1, 3)
    for c0 in range(0, len(cells), CHUNK):
        A = element_matrices(p, coords[cells.verts[c0:c0 + CHUNK]], alpha, beta)
        nodes = cells.nodes[c0:c0 + CHUNK]
        out += np.bincount(nodes.ravel(), weights=np.diagonal(A, axis1=1, axis2=2).ravel(), minlength=nrows)
    return out


def to_scipy(rowptr, colidx, vals, nrows):
    return sp.csr_matrix((vals, colidx, rowptr), shape=(nrows, nrows))


def blocked_values(vals, bs):
    """BAIJ values (nnz * bs * bs,) of A (x) I_bs on the node pattern of A."""
    out = np.zeros((len(vals), bs, bs))
    for a in range(bs):
        out[:, a, a] = vals
    return out.ravel()
