"""Explicit 2-form assembly on the GPU against the NumPy reference assembler (tests/_matrix_ref.py)
at the shapes where the element-matrix kernels and their scatters branch:

* the sum-factorised MATRIX mode of action_hex.cu and the three dense B^T D B kernels of
  bdb_matrix.cu (generic, two-cells-per-CTA p = 3, symmetric p = 4), on meshes large enough that the
  grid-stride loop of every bdb launch runs more than once, with an odd cell count;
* the per-column rank-table scatter with its layer classes (1, 2 and 3+ layers) and the binary
  search (Subsets, native hex cells; tests/_matrix_env_worker.py disables the table);
* iteration ranges [start, end) and the core / owned split;
* BC lgmaps with set_local_diagonal_entries, and mat.mult;
* the A (x) I route of vector spaces (store after a zero, accumulate otherwise, the odd-length tail);
* the diagonal mode behind getDiagonal.

The CSR pattern must equal the reference exactly, values to 1e-12 * max|A_ref| entrywise.
"""
import functools

import numpy as np
import pytest
import scipy.sparse as sp

import _matrix_ref as R
from firedrake_b200 import _lib, op2
from firedrake_b200.utility_meshes import ExtrudedHexMesh

pytestmark = pytest.mark.gpu

TOL = 1e-12
FORMS = [(1.0, 0.0), (0.0, 1.0), (1.0, 0.7)]
# meshes whose cell count is odd and exceeds what one bdb launch keeps resident (see resident_cells)
MULTIPASS = {1: (13, 11, 11), 2: (13, 11, 11), 3: (13, 11, 11), 4: (7, 5, 13)}


@pytest.fixture(params=[0, 1, -1], ids=["sumfact", "dmma", "auto"])
def any_kernel(request, engine):
    """matrix_kernel 0 / 1 as the conftest fixture, and -1: the default choice (DMMA for p >= 3)."""
    _lib.check(engine.fdb_set_option(b"matrix_kernel", request.param))
    yield request.param
    _lib.check(engine.fdb_set_option(b"matrix_kernel", -1))


def sm_count():
    import ctypes as C
    name, sms, mem = C.create_string_buffer(256), C.c_int(), C.c_size_t()
    _lib.check(_lib.lib().fdb_device_info(name, 256, C.byref(sms), C.byref(mem)), "fdb_device_info")
    return sms.value


def resident_cells(p, sym=True):
    """Upper bound on the cells one SM holds in one bdb_matrix.cu launch: CTAs of 256 threads, at most
    2048 threads and 228 KB of shared memory per SM, with the kernels' shared-memory footprints
    (BdbCfg), times the cells per CTA (two for the p = 3 kernel with the symmetric tilings on)."""
    n = p + 1
    nd = n ** 3
    npad = (nd + 31) // 32 * 32
    s, nchunk, kr = npad + 4, (nd + 3) // 4, 16
    pairs = sym and npad == 64
    if pairs:
        smem = (4 * kr * s + 2 * nchunk * 4 * 7 + 48) * 8 + 2 * npad * 12 + 16
    else:
        smem = (3 * kr * s + nchunk * 4 * 7 + 24) * 8 + npad * 12 + 16
    ctas = min(2048 // 256, 228 * 1024 // smem)
    return ctas * (2 if pairs else 1)


# ---------------------------------------------------------------------------------------- helpers
@functools.lru_cache(maxsize=None)
def mesh_of(nx, ny, nz, seed=3):
    return ExtrudedHexMesh(nx, ny, nz, warp=0.05, permute_seed=seed)


class Problem:
    """op2 objects of a scalar (or blocked) Q_p space on ``mesh`` and the reference pattern."""

    def __init__(self, mesh, p, bs=1, core=None):
        self.mesh, self.p, self.bs = mesh, p, bs
        self.V = V = mesh.function_space(p)
        ncols = mesh.num_base_cells
        base = op2.Set(ncols) if core is None else op2.Set((core, ncols, ncols))
        self.cells = op2.ExtrudedSet(base, mesh.layers)
        self.nodes = op2.Set(V.node_count)
        vnodes = op2.Set(mesh.coord_space.node_count)
        self.m0 = op2.Map(self.cells, self.nodes, V.arity, V.cell_node_map, offset=V.offset)
        self.m1 = op2.Map(self.cells, vnodes, 8, mesh.coord_map, offset=mesh.coord_offset)
        self.X = op2.Dat(op2.DataSet(vnodes, 3), mesh.coordinates)
        self.all_cells = R.Cells.extruded(mesh, V)
        self.rowptr, self.colidx = _pattern(mesh, p)

    def mat(self):
        ds = self.nodes if self.bs == 1 else op2.DataSet(self.nodes, self.bs)
        return op2.Mat(op2.Sparsity((ds, ds), [(self.m0, self.m0, None)]))

    def kernel(self, alpha, beta):
        return op2.Kernel("helmholtz", degree=self.p, alpha=alpha, beta=beta, rank=2, cdim=self.bs)

    def ref(self, alpha, beta, cols=None, mask=None, diag_rows=()):
        cells = self.all_cells if cols is None else R.Cells.extruded(self.mesh, self.V, cols)
        return R.assemble(self.p, alpha, beta, self.mesh.coordinates, self.rowptr, self.colidx, cells,
                          mask, mask, diag_rows)


@functools.lru_cache(maxsize=8)
def _pattern(mesh, p):
    return R.pattern(mesh.function_space(p).node_count, R.Cells.extruded(mesh, mesh.function_space(p)))


@functools.lru_cache(maxsize=16)
def _full_ref(mesh, p, alpha, beta):
    return Problem(mesh, p).ref(alpha, beta)


def check(mat, rowptr, colidx, ref, what=""):
    ro, co, vals = mat.csr()
    assert np.array_equal(ro, rowptr) and np.array_equal(co, colidx), f"{what}: pattern differs"
    err = np.abs(vals - ref).max()
    assert err < TOL * np.abs(ref).max(), f"{what}: max error {err:.3e} of max|A| {np.abs(ref).max():.3e}"


def assemble_full(pr, alpha, beta):
    mat = pr.mat()
    mat.zero()
    op2.par_loop(pr.kernel(alpha, beta), pr.cells, mat(op2.INC, (pr.m0, pr.m0)), pr.X(op2.READ, pr.m1))
    mat.assemble()
    return mat


# ------------------------------------------------------------------ shared with the env worker
def check_forms_multipass(p, alpha, beta, sym=True):
    mesh = mesh_of(*MULTIPASS[p])
    ncells = mesh.num_cells
    assert ncells % 2 == 1 and ncells > sm_count() * resident_cells(p, sym), (p, ncells)
    pr = Problem(mesh, p)
    check(assemble_full(pr, alpha, beta), pr.rowptr, pr.colidx, _full_ref(mesh, p, alpha, beta),
          f"p={p} ({alpha}, {beta}) {ncells} cells")


def check_short_columns(p, nz):
    pr = Problem(mesh_of(5, 4, nz), p)
    check(assemble_full(pr, 1.0, 0.7), pr.rowptr, pr.colidx, pr.ref(1.0, 0.7), f"p={p} nz={nz}")


def check_ranges(p):
    """[0, k) as the core part and [k, ncols) as the owned part of one par_loop, then [s, e) alone."""
    mesh = mesh_of(7, 7, 3)
    ncols = mesh.num_base_cells
    k = 33                                       # odd, not a multiple of 32
    pr = Problem(mesh, p, core=k)
    assert pr.cells.core_part == (0, k) and pr.cells.owned_part == (k, ncols)
    mat = assemble_full(pr, 1.0, 0.7)
    check(mat, pr.rowptr, pr.colidx, _full_ref(mesh, p, 1.0, 0.7), f"p={p} core/owned split")
    s, e = 5, 40
    mat.zero()
    gk = op2.GlobalKernel(pr.kernel(1.0, 0.7), [pr.m0, pr.m1], extruded=True)
    loop = op2.Parloop(gk, pr.cells, [mat(op2.INC, (pr.m0, pr.m0)), pr.X(op2.READ, pr.m1)])
    loop._compute((s, e))
    mat.assemble()
    check(mat, pr.rowptr, pr.colidx, pr.ref(1.0, 0.7, cols=np.arange(s, e)), f"p={p} [{s}, {e})")


def check_lgmaps(p, seed=0):
    """Bottom and top node rows plus ~10 % random nodes masked, unit diagonal on them, then mat.mult."""
    mesh = mesh_of(6, 5, 4)
    pr = Problem(mesh, p)
    V = pr.V
    rng = np.random.default_rng(seed)
    bc = np.union1d(np.union1d(V.boundary_nodes("bottom"), V.boundary_nodes("top")),
                    rng.choice(V.node_count, V.node_count // 10, replace=False)).astype(np.int32)
    lg = np.arange(V.node_count, dtype=np.int32)
    lg[bc] = -1
    mat = pr.mat()
    op2.par_loop(pr.kernel(1.0, 0.7), pr.cells, mat(op2.INC, (pr.m0, pr.m0), lgmaps=(lg, lg)),
                 pr.X(op2.READ, pr.m1))
    mat.set_local_diagonal_entries(bc, 1.0)
    mat.assemble()
    ref = pr.ref(1.0, 0.7, mask=lg < 0, diag_rows=bc)
    check(mat, pr.rowptr, pr.colidx, ref, f"p={p} lgmaps")
    A = R.to_scipy(pr.rowptr, pr.colidx, ref, V.node_count)
    xv = rng.standard_normal(V.node_count)
    y = op2.Dat(pr.nodes)
    mat.mult(op2.Dat(pr.nodes, xv.copy()), y)
    yr = A @ xv
    assert np.abs(y.data_ro - yr).max() < TOL * np.abs(yr).max()


# -------------------------------------------------------------------------------------- tests
@pytest.mark.parametrize("alpha,beta", FORMS)
@pytest.mark.parametrize("p", [1, 2, 3, 4])
def test_forms_multipass_odd(any_kernel, p, alpha, beta):
    """Every degree and both templates (beta = 0 has its own), on a mesh where each bdb launch strides
    over its cells more than once and the last p = 3 pair has one live cell."""
    check_forms_multipass(p, alpha, beta)


@pytest.mark.parametrize("p", [5])
def test_degree_5_matrix_is_refused(matrix_kernel, p):
    pr = Problem(mesh_of(2, 2, 2), p)
    mat = pr.mat()
    with pytest.raises(_lib.EngineError, match="not instantiated"):
        op2.par_loop(pr.kernel(1.0, 0.0), pr.cells, mat(op2.INC, (pr.m0, pr.m0)), pr.X(op2.READ, pr.m1))


@pytest.mark.parametrize("nz", [1, 2, 3])
@pytest.mark.parametrize("p", [1, 2, 3, 4])
def test_short_columns(matrix_kernel, p, nz):
    """Columns of 1 and 2 layers: the rank table has one class per layer (v = layer)."""
    check_short_columns(p, nz)


@pytest.mark.parametrize("p", [1, 2, 3, 4])
def test_iteration_ranges(matrix_kernel, p):
    check_ranges(p)


@pytest.mark.parametrize("p", [1, 2, 3, 4])
def test_subset_binary_search(matrix_kernel, p):
    """An op2.Subset of columns (given unsorted, with the first and the last column): binary-search scatter."""
    mesh = mesh_of(7, 7, 3)
    pr = Problem(mesh, p)
    ncols = mesh.num_base_cells
    rng = np.random.default_rng(p)
    idx = np.concatenate([[ncols - 1, 0], rng.choice(np.arange(1, ncols - 1), ncols // 2, replace=False)])
    sub = op2.Subset(pr.cells, idx)
    mat = pr.mat()
    op2.par_loop(pr.kernel(1.0, 0.7), sub, mat(op2.INC, (pr.m0, pr.m0)), pr.X(op2.READ, pr.m1))
    mat.assemble()
    check(mat, pr.rowptr, pr.colidx, pr.ref(1.0, 0.7, cols=np.sort(idx)), f"p={p} subset")


@pytest.mark.parametrize("p", [1, 2, 3, 4])
def test_native_hex_cells(matrix_kernel, p):
    """Non-extruded hexes (one map row per cell, in arbitrary order, no offsets): binary-search scatter."""
    mesh = mesh_of(5, 3, 3)
    V = mesh.function_space(p)
    full = V.full_cell_node_list()
    cfull = mesh.coord_space.full_cell_node_list()
    perm = np.random.default_rng(p).permutation(full.shape[0])
    assert full.shape[0] % 2 == 1
    cells = op2.Set(full.shape[0])
    nodes = op2.Set(V.node_count)
    vnodes = op2.Set(mesh.coord_space.node_count)
    m0 = op2.Map(cells, nodes, V.arity, full[perm])
    m1 = op2.Map(cells, vnodes, 8, cfull[perm])
    X = op2.Dat(op2.DataSet(vnodes, 3), mesh.coordinates)
    mat = op2.Mat(op2.Sparsity((nodes, nodes), [(m0, m0, None)]))
    op2.par_loop(op2.Kernel("helmholtz", degree=p, alpha=1.0, beta=0.7, rank=2), cells,
                 mat(op2.INC, (m0, m0)), X(op2.READ, m1))
    mat.assemble()
    hexes = R.Cells(full[perm], cfull[perm])
    rowptr, colidx = R.pattern(V.node_count, hexes)
    ref = R.assemble(p, 1.0, 0.7, mesh.coordinates, rowptr, colidx, hexes)
    check(mat, rowptr, colidx, ref, f"p={p} native hex")


@pytest.mark.parametrize("p", [1, 2, 3, 4])
def test_lgmaps_diagonal_and_mult(matrix_kernel, p):
    check_lgmaps(p)


@pytest.mark.parametrize("bs", [2, 3, 4])
@pytest.mark.parametrize("p", [2, 4])
def test_blocked_a_kron_identity(matrix_kernel, p, bs):
    """Vector spaces hold A (x) I_bs: a zeroed matrix is stored block by block, a second assembly without
    a zero accumulates (2A); mat.mult against kron(A, I) @ x; component-only BCs are refused."""
    mesh = mesh_of(4, 3, 3)
    pr = Problem(mesh, p, bs=bs)
    n = pr.V.node_count
    ref = _full_ref(mesh, p, 1.0, 0.7)
    if bs == 3:
        # odd nnz * bs^2: the store kernel writes pairs of doubles and copies the last entry on its own
        assert len(pr.colidx) % 2 == 1
    mat = pr.mat()
    assert mat.bs == bs and mat.nnz == len(pr.colidx)
    mat.zero()
    arg = lambda: mat(op2.INC, (pr.m0, pr.m0))
    op2.par_loop(pr.kernel(1.0, 0.7), pr.cells, arg(), pr.X(op2.READ, pr.m1))
    check(mat, pr.rowptr, pr.colidx, R.blocked_values(ref, bs), f"p={p} bs={bs} store")
    op2.par_loop(pr.kernel(1.0, 0.7), pr.cells, arg(), pr.X(op2.READ, pr.m1))
    check(mat, pr.rowptr, pr.colidx, R.blocked_values(2.0 * ref, bs), f"p={p} bs={bs} accumulate")
    rng = np.random.default_rng(bs)
    xv = rng.standard_normal((n, bs))
    y = op2.Dat(op2.DataSet(pr.nodes, bs))
    mat.mult(op2.Dat(op2.DataSet(pr.nodes, bs), xv.copy()), y)
    yr = (sp.kron(R.to_scipy(pr.rowptr, pr.colidx, 2.0 * ref, n), sp.identity(bs), format="csr")
          @ xv.ravel()).reshape(n, bs)
    assert np.abs(y.data_ro - yr).max() < TOL * np.abs(yr).max()
    # a condition on one component only is not expressible as A (x) I
    lg = np.arange(n * bs, dtype=np.int32)
    lg[pr.V.boundary_nodes("bottom").astype(np.int64) * bs] = -1
    with pytest.raises(_lib.EngineError, match="single components"):
        op2.par_loop(pr.kernel(1.0, 0.7), pr.cells, mat(op2.INC, (pr.m0, pr.m0), lgmaps=(lg, lg)),
                     pr.X(op2.READ, pr.m1))


@pytest.mark.parametrize("bcs", [False, True])
@pytest.mark.parametrize("p", [1, 2, 3])
def test_get_diagonal(p, bcs, engine):
    """Diagonal mode of the sum-factorised kernel (P.vals == nullptr) behind getDiagonal."""
    from firedrake_b200.assemble import DirichletBC, Form, FunctionSpace, assemble
    mesh = mesh_of(*MULTIPASS[p])
    V = FunctionSpace(mesh, p)
    bc = [DirichletBC(V, 0.0, ["bottom", 1, 3])] if bcs else []
    ctx = assemble(Form(V, 1.0, 0.7), bcs=bc, mat_type="matfree")
    D = ctx.getDiagonal(V.dat())
    ref = R.diagonal(p, 1.0, 0.7, mesh.coordinates, V.node_count, R.Cells.extruded(mesh, V.V))
    if bcs:
        ref[bc[0].nodes] = 1.0
    assert np.abs(D.data_ro - ref).max() < TOL * np.abs(ref).max()


@pytest.mark.parametrize("env", ["FDB_BDB_SYM=0", "FDB_MAT_NO_RANK=1"])
def test_env_selected_paths(env):
    """Kernel choices read once per process: the generic bdb kernel at p = 3 / 4 and the binary-search
    scatter on full extruded sets, in a worker process (tests/_matrix_env_worker.py)."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    name, value = env.split("=")
    r = subprocess.run([sys.executable, os.path.join(root, "tests", "_matrix_env_worker.py")],
                       env=dict(os.environ, **{name: value}), capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert f"MATRIX_ENV_OK {name}" in r.stdout
