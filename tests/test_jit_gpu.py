"""GPU run of the generic wrapper builder and of the blocked matrices.

First run on a B200 in round 2 (all 28 cases green on the first attempt; log kept in
profiles/r02_first_validation.txt), after which the round-1 gate was removed.

Each case mirrors a CPU case of tests/test_codegen.py, now through
``op2.par_loop(op2.Kernel(code, name), ...)`` -> fdb_wrapper_create (NVRTC) ->
fdb_kernel_call on device-resident Dats.
"""
import os

import numpy as np
import pytest

from firedrake_b200 import op2
from firedrake_b200.codegen import CStringKernel, PermutedMap
from firedrake_b200.fiat_lite import interval_element
from firedrake_b200.utility_meshes import ExtrudedHexMesh

import test_codegen as tc

pytestmark = [pytest.mark.gpu]

GOLD = tc.GOLD


def test_golden_mass_and_rhs(engine):
    elems, nodes, m, X, f = tc._golden_mesh()
    mass, rhs = tc._p1_kernels()
    A = op2.Mat(op2.Sparsity((nodes, nodes), [(m, m, None)]))
    A.zero()
    op2.par_loop(mass, elems, A(op2.INC, (m, m)), X(op2.READ, m))
    A.assemble()
    assert np.abs(A.values - np.array(GOLD["expected_matrix"])).max() < GOLD["expected_matrix_eps"]
    b = op2.Dat(nodes)
    op2.par_loop(rhs, elems, b(op2.INC, m), X(op2.READ, m), f(op2.READ, m))
    assert np.abs(b.data_ro - np.array(GOLD["expected_rhs"])).max() < GOLD["expected_rhs_eps"]
    # the same golden arrays through the hand-written P1 kernels agree with the generated path
    y = op2.Dat(nodes)
    A.mult(f, y)
    assert np.allclose(y.data_ro, b.data_ro, rtol=0, atol=1e-14)


def test_blocked_matrix_generic_path(engine):
    elems, nodes, m, X, _ = tc._golden_mesh()
    mass2, _ = tc._p1_kernels(cdim=2)
    d2 = op2.DataSet(nodes, 2)
    A = op2.Mat(op2.Sparsity((d2, d2), [(m, m, None)]))
    A.zero()
    lg = np.arange(8, dtype=np.int32)
    lg[7] = -1
    op2.par_loop(mass2, elems, A(op2.INC, (m, m), lgmaps=(lg, lg)), X(op2.READ, m))
    A.set_local_diagonal_entries([3], 1.0, idx=1)
    A.assemble()
    M = np.kron(np.array(GOLD["expected_matrix"]), np.eye(2))
    D = A.values
    keep = [i for i in range(8) if i != 7]
    assert np.abs(D[np.ix_(keep, keep)] - M[np.ix_(keep, keep)]).max() < 1e-5
    assert D[7, 7] == 1.0 and np.all(D[7, :7] == 0) and np.all(D[:7, 7] == 0)
    x = op2.Dat(d2, np.random.default_rng(0).standard_normal((4, 2)))
    y = op2.Dat(d2)
    A.mult(x, y)
    assert np.allclose(y.data_ro.ravel(), D @ x.data_ro.ravel(), rtol=0, atol=1e-14)


def test_access_modes(engine):
    n = 100000                                 # many warps: atomics and warp reductions matter
    it, ind, unit = op2.Set(n), op2.Set(n), op2.Set(1)
    rng = np.random.default_rng(7)
    i2i = op2.Map(it, ind, 1, rng.permutation(n))
    i2u = op2.Map(it, unit, 1, np.zeros(n, dtype=np.int32))
    x = op2.Dat(ind, np.arange(n), dtype=np.uint32)
    op2.par_loop(op2.Kernel("static void wo(unsigned int *x) { *x = 42; }", "wo"), it, x(op2.WRITE, i2i))
    assert (x.data_ro == 42).all()
    x = op2.Dat(ind, np.arange(n), dtype=np.uint32)
    op2.par_loop(op2.Kernel("static void rw(unsigned int *x) { (*x) = (*x) + 1; }", "rw"), it, x(op2.RW, i2i))
    assert int(x.data_ro.sum(dtype=np.uint64)) == n * (n + 1) // 2
    u = op2.Dat(unit, [0], dtype=np.uint32)
    op2.par_loop(op2.Kernel("static void inc(unsigned int *x) { (*x) = (*x) + 1; }", "inc"), it, u(op2.INC, i2u))
    assert u.data_ro[0] == n
    v = op2.Dat(it, rng.standard_normal(n))
    for acc, cmp, ref in ((op2.MIN, "<", v.data_ro.min()), (op2.MAX, ">", v.data_ro.max())):
        t = op2.Dat(unit, [v.data_ro[0]])
        k = op2.Kernel(f"static void mm(double *t, const double *v) {{ if (*v {cmp} *t) *t = *v; }}", "mm")
        op2.par_loop(k, it, t(acc, i2u), v(op2.READ))
        assert t.data_ro[0] == ref
        g = op2.Global(1, v.data_ro[0])
        k = op2.Kernel(f"static void gm(const double *v, double *g) {{ if (*v {cmp} *g) *g = *v; }}", "gm")
        op2.par_loop(k, it, v(op2.READ), g(acc))
        assert g.data_ro[0] == ref
    g = op2.Global(1, 0.0)
    op2.par_loop(op2.Kernel("static void gs(const double *v, double *g) { *g += *v; }", "gs"), it,
                 v(op2.READ), g(op2.INC))
    assert abs(g.data_ro[0] - v.data_ro.sum()) < 1e-9
    gi = op2.Global(1, 0, np.int64)
    w = op2.Dat(it, np.arange(n), dtype=np.int64)
    op2.par_loop(op2.Kernel("static void gl(const long long *v, long long *g) { *g += *v; }", "gl"), it,
                 w(op2.READ), gi(op2.INC))
    assert gi.data_ro[0] == n * (n - 1) // 2


def test_permuted_map_and_subset(engine):
    fromset, toset = op2.Set(1), op2.Set(4)
    d1 = op2.Dat(toset, [10, 11, 12, 13], dtype=np.int32)
    d2 = op2.Dat(toset, dtype=np.int32)
    m1 = op2.Map(fromset, toset, 4, [0, 2, 1, 3])
    m2, m3 = PermutedMap(m1, [3, 2, 1, 0]), PermutedMap(m1, [0, 2, 3, 1])
    k = op2.Kernel("void copy(int *to, const int * restrict from) { for (int i = 0; i < 4; i++) to[i] = from[i]; }",
                   "copy")
    op2.par_loop(k, fromset, d2(op2.WRITE, m2), d1(op2.READ, m3))
    expect = np.empty(4, dtype=np.int32)
    expect[m1.values_with_halo[0][m2.permutation]] = d1.data_ro[m1.values_with_halo[0][m3.permutation]]
    assert (d2.data_ro == expect).all()
    it = op2.Set(5000)
    x = op2.Dat(it, dtype=np.int32)
    sub = op2.Subset(it, np.arange(3, 5000, 7))
    op2.par_loop(op2.Kernel("static void one(int *x) { *x = 1; }", "one"), sub, x(op2.WRITE))
    assert x.data_ro.sum() == len(sub.indices) and (x.data_ro[sub.indices] == 1).all()


def test_generic_extruded_action_equals_fast_path_and_oracle(engine, oracle):
    mesh = ExtrudedHexMesh(7, 6, 9, warp=0.05, permute_seed=0)
    V = mesh.function_space(1)
    cells = op2.ExtrudedSet(op2.Set(mesh.num_base_cells), mesh.layers)
    nodes, vnodes = op2.Set(V.node_count), op2.Set(mesh.coord_space.node_count)
    m0 = op2.Map(cells, nodes, V.arity, V.cell_node_map, offset=V.offset)
    m1 = op2.Map(cells, vnodes, 8, mesh.coord_map, offset=mesh.coord_offset)
    X = op2.Dat(op2.DataSet(vnodes, 3), mesh.coordinates)
    x = op2.Dat(nodes, np.random.default_rng(3).standard_normal(V.node_count))
    yg, yf = op2.Dat(nodes), op2.Dat(nodes)
    op2.par_loop(op2.Kernel(tc.Q1_POISSON, "q1_poisson"), cells, yg(op2.INC, m0), X(op2.READ, m1), x(op2.READ, m0))
    op2.par_loop(op2.Kernel("helmholtz", degree=1), cells, yf(op2.INC, m0), X(op2.READ, m1), x(op2.READ, m0))
    yo = np.zeros(V.node_count)
    oracle.action_extruded(interval_element(1), 0, mesh.num_base_cells, [0, mesh.layers], yo, mesh.coordinates,
                           x.data_ro.copy(), V.cell_node_map, V.offset, mesh.coord_map, mesh.coord_offset)
    scale = np.abs(yo).max()
    assert np.abs(yg.data_ro - yo).max() < 1e-12 * scale
    assert np.abs(yf.data_ro - yo).max() < 1e-12 * scale


@pytest.mark.parametrize("p,cdim", [(2, 3), (1, 2), (3, 3), (4, 3)])
def test_vector_space_matrix_fast_path(engine, oracle, matrix_kernel, p, cdim):
    """assemble(a) on a VectorFunctionSpace (config 4's explicit matrix): blocked CSR ==
    kron(scalar oracle matrix, I), with node Dirichlet conditions, and SpMV == matrix-free.
    p >= 3 runs the dense B^T D B kernel on the fp64 tensor pipe (bdb_matrix.cu), (4, 3) being
    config 4's own instance; reference scatter: pyop2/codegen/builder.py:573-625."""
    from firedrake_b200.assemble import DirichletBC, FunctionSpace, assemble, helmholtz
    import test_matrix_gpu as tm
    mesh = ExtrudedHexMesh(3, 3, 4, warp=0.05, permute_seed=2) if p < 4 else \
        ExtrudedHexMesh(2, 2, 3, warp=0.05, permute_seed=2)
    V = FunctionSpace(mesh, p, cdim=cdim)
    bcs = [DirichletBC(V, 0.0, "bottom")]
    A = assemble(helmholtz(V), bcs=bcs)
    assert A.bs == cdim
    lg = np.arange(V.node_count, dtype=np.int32)
    lg[bcs[0].nodes] = -1
    rowptr, colidx, vo = tm.oracle_matrix(oracle, mesh, V.V, p, 1.0, 1.0, lg)
    r2, c2, vals = A.csr()
    assert np.array_equal(rowptr, r2) and np.array_equal(colidx, c2)
    blocks = vals.reshape(-1, cdim, cdim)
    diag_rows = np.isin(np.repeat(np.arange(V.node_count), np.diff(rowptr)), bcs[0].nodes) & \
        (colidx == np.repeat(np.arange(V.node_count), np.diff(rowptr)))
    expect = vo[:, None, None] * np.eye(cdim)[None]
    expect[diag_rows] = np.eye(cdim)
    assert np.abs(blocks - expect).max() < 1e-12 * np.abs(vo).max()
    x = V.dat(np.random.default_rng(1).standard_normal((V.node_count, cdim)))
    y1, y2 = V.dat(), V.dat()
    A.mult(x, y1)
    assemble(helmholtz(V), bcs=bcs, mat_type="matfree").mult(x, y2)
    assert np.abs(y1.data_ro - y2.data_ro).max() < 1e-11 * np.abs(y1.data_ro).max()


def test_cg4_matrix_instantiation(engine, oracle):
    """Degree-4 explicit matrix (new launch_matrix_n<5> instantiation)."""
    import test_matrix_gpu as tm
    mesh = ExtrudedHexMesh(2, 2, 3, warp=0.05, permute_seed=2)
    V, cells, nodes, m0, m1, X = tm.setup(mesh, 4)
    mat = op2.Mat(op2.Sparsity((nodes, nodes), [(m0, m0, None)]))
    mat.zero()
    op2.par_loop(op2.Kernel("helmholtz", degree=4, alpha=1.0, beta=1.0, rank=2), cells,
                 mat(op2.INC, (m0, m0)), X(op2.READ, m1))
    mat.assemble()
    _, _, vals = mat.csr()
    _, _, vo = tm.oracle_matrix(oracle, mesh, V, 4, 1.0, 1.0)
    assert np.abs(vals - vo).max() < 1e-12 * np.abs(vo).max()


def test_mult_transpose(engine):
    from firedrake_b200.assemble import DirichletBC, FunctionSpace, assemble, poisson
    mesh = ExtrudedHexMesh(3, 3, 4, warp=0.05)
    V = FunctionSpace(mesh, 2)
    bcs = [DirichletBC(V, 0.0, "top")]
    ctx = assemble(poisson(V), bcs=bcs, mat_type="matfree")
    A = assemble(poisson(V), bcs=bcs).values
    x = V.dat(np.random.default_rng(5).standard_normal(V.node_count))
    y = V.dat()
    ctx.multTranspose(x, y)
    assert np.abs(y.data_ro - A.T @ x.data_ro).max() < 1e-11 * np.abs(y.data_ro).max()


def test_expression_interpolation(engine):
    from firedrake_b200.assemble import FunctionSpace, interpolate
    mesh = ExtrudedHexMesh(5, 4, 6, warp=0.05, permute_seed=1)
    V = FunctionSpace(mesh, 3)
    u = interpolate(V, "sin(M_PI * x[0]) * cos(2 * M_PI * x[1]) * (1 + x[2])")
    P = V.V.dof_coordinates()
    ref = np.sin(np.pi * P[:, 0]) * np.cos(2 * np.pi * P[:, 1]) * (1 + P[:, 2])
    assert np.abs(u.data_ro - ref).max() < 1e-13
    W = FunctionSpace(mesh, 2, cdim=3)
    w = interpolate(W, ["x[1] * x[2]", "-x[0]", "exp(x[2])"])
    P = W.V.dof_coordinates()
    ref = np.stack([P[:, 1] * P[:, 2], -P[:, 0], np.exp(P[:, 2])], axis=1)
    assert np.abs(w.data_ro - ref).max() < 1e-13


def test_host_pointer_mode_generic(engine):
    """fdb_kernel_call(FDB_LOC_HOST) on a generated wrapper: NumPy buffers in, every written
    Dat copied back, versions tracked (two calls: the second must see the first's result)."""
    from firedrake_b200 import codegen
    elems, nodes, m, X, f = tc._golden_mesh()
    _, rhs = tc._p1_kernels()
    b = op2.Dat(nodes)
    b.data[:] = 0.0
    codegen.par_loop(rhs, elems, b(op2.INC, m), X(op2.READ, m), f(op2.READ, m), location="host")
    assert np.abs(b._data - np.array(GOLD["expected_rhs"])).max() < GOLD["expected_rhs_eps"]
    codegen.par_loop(rhs, elems, b(op2.INC, m), X(op2.READ, m), f(op2.READ, m), location="host")
    assert np.abs(b._data - 2 * np.array(GOLD["expected_rhs"])).max() < 2 * GOLD["expected_rhs_eps"]


def test_mg_transfers_on_device(engine):
    from firedrake_b200 import mg
    from firedrake_b200.assemble import FunctionSpace
    h = mg.MeshHierarchy(2, 3, 2, 1, permute_seed=4)
    Vc, Vf = FunctionSpace(h[0], 2), FunctionSpace(h[1], 2)
    T = mg.TransferManager(Vc, Vf)
    Pc, Pf = Vc.V.dof_coordinates(), Vf.V.dof_coordinates()
    poly = lambda P: (1 + P[:, 0]) ** 2 * (2 - P[:, 1]) ** 2 * (0.5 + P[:, 2]) ** 2
    uc, uf = Vc.dat(poly(Pc)), Vf.dat()
    T.prolong(uc, uf)
    assert np.abs(uf.data_ro - poly(Pf)).max() < 1e-12 * np.abs(poly(Pf)).max()
    back = Vc.dat()
    T.inject(uf, back)
    assert np.abs(back.data_ro - uc.data_ro).max() < 1e-12 * np.abs(uc.data_ro).max()
    rng = np.random.default_rng(11)
    vc, rf = Vc.dat(rng.standard_normal(Vc.node_count)), Vf.dat(rng.standard_normal(Vf.node_count))
    pv, rc = Vf.dat(), Vc.dat()
    T.prolong(vc, pv)
    T.restrict(rf, rc)
    lhs, rhs = float(pv.data_ro @ rf.data_ro), float(vc.data_ro @ rc.data_ro)
    assert abs(lhs - rhs) < 1e-11 * max(abs(lhs), 1.0)


def test_mg_preconditioned_cg_is_mesh_independent(engine):
    """demos/multigrid/geometric_multigrid.py.rst: CG preconditioned by a V-cycle converges in a
    number of iterations that does not grow under refinement (unpreconditioned CG doubles)."""
    from firedrake_b200 import mg
    from firedrake_b200.assemble import cg, helmholtz
    its, plain = [], []
    for levels in (1, 2):
        h = mg.MeshHierarchy(4, 4, 4, levels, warp=0.03)
        vc = mg.VCycle(h, 2, helmholtz, bc_domains=("bottom",))
        top = len(h) - 1
        V, A = vc.spaces[top], vc.ops[top]
        b = V.dat(np.random.default_rng(2).standard_normal(V.node_count))
        for bc in vc.bcs[top]:
            bc.zero(b)
        x = V.dat()
        x.device_ptr
        n, hist = mg.pcg(A, b, x, lambda r, z: vc.apply(top, r, z), rtol=1e-8)
        assert hist[-1] <= 1e-8 * hist[0]
        its.append(n)
        x2 = V.dat()
        x2.device_ptr
        n2, _ = cg(A, b, x2, rtol=1e-8, maxit=2000)
        plain.append(n2)
        assert np.abs(x.data_ro - x2.data_ro).max() < 1e-6 * np.abs(x2.data_ro).max()
    assert its[1] <= its[0] + 3 and its[1] < plain[1] / 3


def test_zero_forms_dx_and_exterior_facets(engine):
    """tests/firedrake/regression/test_integral_hex.py:10-23 (f*ds on the unit cube, exact
    value 2+4+2+5+2+6) on the extruded hex mesh, the per-face split, and volume / area of a
    warped mesh whose boundary is unchanged (tests/firedrake/extrusion/test_zero_forms_extrusion.py)."""
    from firedrake_b200.assemble import FunctionSpace, assemble_functional, interpolate
    mesh = ExtrudedHexMesh(2, 3, 5, permute_seed=3)
    V = FunctionSpace(mesh, 3)
    f = interpolate(V, "2 * x[0] + 3 * x[1] * x[1] + 4 * x[2] * x[2] * x[2]")
    assert abs(assemble_functional(V, f, "ds_b") - 2.0) < 1e-10
    assert abs(assemble_functional(V, f, "ds_t") - 6.0) < 1e-10
    assert abs(assemble_functional(V, f, "ds_v") - (2 + 4 + 2 + 5)) < 1e-10
    assert abs(assemble_functional(V, f, "ds") - 21.0) < 1e-10
    assert abs(assemble_functional(V, f, "dx") - (1 + 1 + 1)) < 1e-10
    wm = ExtrudedHexMesh(3, 3, 4, warp=0.05, permute_seed=1)
    W = FunctionSpace(wm, 2)
    one = interpolate(W, "1.0")
    assert abs(assemble_functional(W, one, "dx") - 1.0) < 1e-12
    assert abs(assemble_functional(W, one, "ds") - 6.0) < 1e-12


def test_dense_linear_algebra_callables(engine):
    n, N = 5000, 5
    it = op2.Set(n)
    rng = np.random.default_rng(4)
    A = rng.standard_normal((n, N, N))
    A[::3, 0, 0] = 0.0
    b = rng.standard_normal((n, N))
    dA, db = op2.Dat(op2.DataSet(it, N * N), A), op2.Dat(op2.DataSet(it, N), b)
    dinv, dx = op2.Dat(op2.DataSet(it, N * N)), op2.Dat(op2.DataSet(it, N))
    k = op2.Kernel(f"static void la(double *Ainv, double *x, const double *A, const double *b)"
                   f"{{ inverse(Ainv, A, {N}); solve(x, A, b, {N}); }}", "la")
    op2.par_loop(k, it, dinv(op2.WRITE), dx(op2.WRITE), dA(op2.READ), db(op2.READ))
    ref_inv = np.linalg.inv(A)
    ref_x = np.linalg.solve(A, b[..., None])[..., 0]
    scale = np.abs(ref_inv).max(axis=(1, 2))
    assert (np.abs(dinv.data_ro.reshape(n, N, N) - ref_inv).max(axis=(1, 2)) < 1e-10 * scale).all()
    assert (np.abs(dx.data_ro - ref_x).max(axis=1) < 1e-10 * np.abs(ref_x).max(axis=1) * np.maximum(scale, 1)).all()


@pytest.mark.parametrize("p,levels,rate", [(1, (4, 6), 1.9), (2, (2, 4), 2.9), (3, (1, 3), 3.9)])
def test_helmholtz_convergence_rates(engine, p, levels, rate):
    """tests/firedrake/extrusion/test_helmholtz_scalar.py:8-36 through the engine: f and the exact
    solution interpolated (generic path), load vector = mass action, matrix-free CG on the device,
    L2 error through the mass form."""
    from firedrake_b200.assemble import FunctionSpace, assemble, cg, helmholtz, interpolate, mass
    errs = []
    for ii in range(*levels):
        n = 2 ** ii
        V = FunctionSpace(ExtrudedHexMesh(n, n, n, permute_seed=ii), p)
        u_exact = "cos(2*M_PI*x[0]) * cos(2*M_PI*x[1]) * cos(2*M_PI*x[2])"
        exact = interpolate(V, u_exact)
        f = interpolate(V, f"(1 + 12*M_PI*M_PI) * {u_exact}")
        b = assemble(mass(V), u=f)
        A = assemble(helmholtz(V), mat_type="matfree")
        u = V.dat()
        u.device_ptr
        it, hist = cg(A, b, u, rtol=1e-12, maxit=5000)
        assert hist[-1] <= 1e-12 * hist[0]
        e = V.dat(u.data_ro - exact.data_ro)
        Me = assemble(mass(V), u=e)
        errs.append(np.sqrt(e.data_ro @ Me.data_ro))
    rates = [np.log2(errs[i] / errs[i + 1]) for i in range(len(errs) - 1)]
    assert min(rates) > rate, (errs, rates)


def test_interior_facet_functionals(engine):
    """tests/firedrake/regression/test_integral_hex.py:26-37: the jump of a continuous function
    over all interior facets vanishes; avg(1)*dS measures the interior facet area
    ((nz-1) Lx Ly horizontal + ((nx-1) + (ny-1)) vertical unit faces on the unit cube).
    Exercises ON_INTERIOR_FACETS two-layer packs and doubled '+'/'-' facet maps."""
    from firedrake_b200.assemble import FunctionSpace, assemble_functional, interpolate
    mesh = ExtrudedHexMesh(2, 3, 5, permute_seed=2)
    V = FunctionSpace(mesh, 3)
    f = interpolate(V, "2 * x[0] + 3 * x[1] * x[1] + 4 * x[2] * x[2] * x[2]")
    assert assemble_functional(V, f, "dS", integrand="jump2") ** 0.5 < 1e-13
    one = interpolate(V, "1.0")
    assert abs(assemble_functional(V, one, "dS_h") - 4.0) < 1e-12
    assert abs(assemble_functional(V, one, "dS_v") - 3.0) < 1e-12
    # avg(f) over the horizontal facets z = k/5: int 2x + 3y^2 + 4z^3 = 2 + 4 z^3
    ref = sum(2 + 4 * (k / 5) ** 3 for k in range(1, 5))
    assert abs(assemble_functional(V, f, "dS_h") - ref) < 1e-11


@pytest.mark.parametrize("p", [1, 2, 3, 4, 5])
def test_affine_cell_variant(engine, oracle, p, monkeypatch):
    """The per-cell-metric kernel variant (fdb_kernel_desc.affine_cells) on a mesh of
    parallelepipeds == the oracle (which evaluates the geometry at every quadrature point),
    Poisson and Helmholtz; the geometry check refuses a warped mesh."""
    from firedrake_b200.assemble import FunctionSpace, OneFormAssembler, helmholtz, poisson
    monkeypatch.setenv("FDB_AFFINE", "1")
    mesh = ExtrudedHexMesh(4, 3, 8, Lx=2.0, Ly=0.75, Lz=1.0, permute_seed=1)
    V = FunctionSpace(mesh, p)
    assert V.cells_are_affine()
    assert not FunctionSpace(ExtrudedHexMesh(4, 3, 8, warp=0.05), p).cells_are_affine()
    x = V.dat(np.random.default_rng(9).standard_normal(V.node_count))
    for form, (alpha, beta) in ((poisson(V), (1.0, 0.0)), (helmholtz(V), (1.0, 1.0))):
        assert form.kernel(1).affine
        y = OneFormAssembler(form, x).assemble()
        yo = np.zeros(V.node_count)
        oracle.action_extruded(interval_element(p), 0, mesh.num_base_cells, [0, mesh.layers], yo, mesh.coordinates,
                               x.data_ro.copy(), V.V.cell_node_map, V.V.offset, mesh.coord_map, mesh.coord_offset,
                               1, alpha, beta)
        assert np.abs(y.data_ro - yo).max() < 1e-12 * np.abs(yo).max()


@pytest.mark.parametrize("pc", ["none", "jacobi", "mg"])
def test_solve_front_end(engine, pc):
    """solve(a == L, u, bcs, solver_parameters) (firedrake/solving.py): the reference's
    strong-BC Poisson problem (tests/firedrake/extrusion/test_poisson_strong_bcs_extrusion.py:
    u = 0 on the bottom, 42 on the top, exact solution 42 z) with each preconditioner."""
    from firedrake_b200 import mg
    from firedrake_b200.assemble import DirichletBC, FunctionSpace, poisson, solve
    h = mg.MeshHierarchy(2, 2, 2, 2)
    V = FunctionSpace(h[2], 2)
    bcs = [DirichletBC(V, 0.0, "bottom"), DirichletBC(V, 42.0, "top")]
    u = V.dat()
    its, hist = solve(poisson(V), V.dat(), u, bcs=bcs, hierarchy=h,
                      solver_parameters={"pc_type": pc, "ksp_rtol": 1e-12})
    z = V.V.dof_coordinates()[:, 2]
    assert np.abs(u.data_ro - 42.0 * z).max() < 1e-7, (pc, its, hist[-1])
    assert its < {"none": 200, "jacobi": 200, "mg": 15}[pc]


def test_variable_coefficient_form(engine, oracle):
    """inner(kappa*grad u, grad v)*dx with a coefficient field, generic path: kappa == 1 must
    equal the hand-written Poisson kernel; kappa = 2 + x must equal 2*Poisson + the x-weighted part
    (linearity in kappa)."""
    from firedrake_b200.assemble import (FunctionSpace, OneFormAssembler, assemble_variable_coefficient,
                                         interpolate, poisson)
    mesh = ExtrudedHexMesh(4, 3, 5, warp=0.05, permute_seed=2)
    V = FunctionSpace(mesh, 2)
    u = V.dat(np.random.default_rng(0).standard_normal(V.node_count))
    one, xk, kap = interpolate(V, "1.0"), interpolate(V, "x[0]"), interpolate(V, "2.0 + x[0]")
    y1 = assemble_variable_coefficient(V, one, u)
    yf = OneFormAssembler(poisson(V), u).assemble()
    scale = np.abs(yf.data_ro).max()
    assert np.abs(y1.data_ro - yf.data_ro).max() < 1e-12 * scale
    yx = assemble_variable_coefficient(V, xk, u)
    yk = assemble_variable_coefficient(V, kap, u)
    assert np.abs(yk.data_ro - (2 * y1.data_ro + yx.data_ro)).max() < 1e-12 * scale


def test_periodic_extrusion_on_device(engine, oracle):
    """Periodic extrusion on the GPU (generic wrapper path): Q1 Poisson action on columns that are
    periodic in z -- nz dofs per vertex column, the top cell's top dofs are the bottom cell's bottom
    ones (Map.offset_quotient, pyop2/codegen/builder.py:100-123) -- against a cell-by-cell NumPy
    assembly of the oracle's element actions with wrapped indices."""
    from oracle import oracle as orc
    nx, ny, nz = 3, 2, 6
    mesh = ExtrudedHexMesh(nx, ny, nz, warp=0.0)
    V1 = mesh.coord_space
    NV = (nx + 1) * (ny + 1)
    cols = op2.ExtrudedSet(op2.Set(mesh.num_base_cells), mesh.layers, extruded_periodic=True)
    pnodes = op2.Set(NV * nz)
    vnodes = op2.Set(V1.node_count)
    # periodic numbering: vertex column v holds dofs v*nz .. v*nz + nz-1
    vcol = (V1.cell_node_map[:, ::2] // (nz + 1))            # (ncols, 4): vertex column of each (ax, ay)
    assert np.array_equal(V1.cell_node_map[:, ::2] % (nz + 1), 0 * vcol)
    pm = np.empty((mesh.num_base_cells, 8), dtype=np.int32)
    pm[:, 0::2] = vcol * nz
    pm[:, 1::2] = vcol * nz + 1
    m0 = op2.Map(cols, pnodes, 8, pm, offset=[1] * 8, offset_quotient=[0, 1] * 4)
    m1 = op2.Map(cols, vnodes, 8, mesh.coord_map, offset=mesh.coord_offset)
    rng = np.random.default_rng(5)
    u = op2.Dat(pnodes, rng.standard_normal(NV * nz))
    y = op2.Dat(pnodes)
    X = op2.Dat(op2.DataSet(vnodes, 3), mesh.coordinates)
    op2.par_loop(op2.Kernel(tc.Q1_POISSON, "q1_poisson"), cols, y(op2.INC, m0), X(op2.READ, m1), u(op2.READ, m0))
    el = interval_element(1)
    ref = np.zeros(NV * nz)
    uh = u.data_ro
    for c in range(mesh.num_base_cells):
        for l in range(nz):
            idx = pm[c] + np.array([(l + q) % nz - q for q in (0, 1)] * 4)
            cidx = mesh.coord_map[c] + mesh.coord_offset * l
            ref[idx] += orc.cell_action(el, mesh.coordinates[cidx].ravel(), uh[idx].copy())
    assert np.abs(y.data_ro - ref).max() < 1e-12 * np.abs(ref).max()
    # constants are in the null space of the periodic operator as well
    one = op2.Dat(pnodes, np.ones(NV * nz))
    z = op2.Dat(pnodes)
    op2.par_loop(op2.Kernel(tc.Q1_POISSON, "q1_poisson"), cols, z(op2.INC, m0), X(op2.READ, m1), one(op2.READ, m0))
    assert np.abs(z.data_ro).max() < 1e-12


def test_periodic_interior_horizontal_facets_on_device(engine):
    """dS_h on periodically extruded columns: a column of nz cells has nz horizontal interior
    facets, the last one joining its top cell to its bottom cell (pyop2/codegen/builder.py:800-805).
    Counted three ways: a Global INC (nz per column), the sum of the layer numbers into a Dat
    indexed by the column (0 + ... + nz-1), and a cell Dat through a periodic map that every
    facet adds 1 to below and 10 to above (11 in every cell, the bottom cell's 10 coming from
    the wrap-around facet)."""
    from firedrake_b200 import codegen
    ncol, nz = 37, 6
    cols = op2.ExtrudedSet(op2.Set(ncol), nz + 1, extruded_periodic=True)
    cells = op2.Set(ncol * nz)
    cmap = op2.Map(cols, cells, 1, np.arange(ncol) * nz, offset=[1])     # cell l of column c: c*nz + l
    k = op2.Kernel("static void k(double *g, double *s, double *c, int layer) "
                   "{ g[0] += 1.0; s[0] += layer; c[0] += 1.0; c[1] += 10.0; }", "k")
    for location in ("device", "host"):
        g = op2.Global(1, 0.0)
        s = op2.Dat(op2.DataSet(cols, 1))
        c = op2.Dat(cells)
        codegen.par_loop(k, cols, g(op2.INC), s(op2.INC), c(op2.INC, cmap), iteration_region="ON_INTERIOR_FACETS",
                         pass_layer_arg=True, location=location)
        assert g.data_ro[0] == ncol * nz, location
        assert (s.data_ro == nz * (nz - 1) // 2).all(), location
        assert (c.data_ro == 11.0).all(), location


def test_mixed_dat_parloop_and_vector_operations(engine):
    """op2.MixedDat through op2.par_loop on the device and in host-pointer mode (one local tensor
    for the kernel, one arglist pointer per block: pyop2/parloop.py:203-212), plus the block-wise
    whole-vector operations of pyop2/types/dat.py:861-."""
    from firedrake_b200 import codegen
    rng = np.random.default_rng(5)
    ncell, nv, npr = 4000, 2300, 900
    cells, vset, pset = op2.Set(ncell), op2.Set(nv), op2.Set(npr)
    mv = op2.Map(cells, vset, 3, rng.integers(0, nv, (ncell, 3)))
    mp = op2.Map(cells, pset, 2, rng.integers(0, npr, (ncell, 2)))
    u, p = op2.Dat(vset ** 2, rng.standard_normal((nv, 2))), op2.Dat(pset, rng.standard_normal(npr))
    w, r = op2.MixedDat([u, p]), op2.MixedDat(op2.MixedDataSet([vset ** 2, pset]))
    mm = op2.MixedMap([mv, mp])
    k = op2.Kernel("static void k(double *r, const double *w, const double *s) {"
                   " for (int i = 0; i < 8; ++i) r[i] += s[0]*w[i] + (i < 7 ? w[i+1] : w[0]); }", "k")
    s = op2.Global(1, 1.5)
    eu, ep = np.zeros((nv, 2)), np.zeros(npr)
    for c in range(ncell):
        loc = np.concatenate([u.data_ro[mv.values[c]].ravel(), p.data_ro[mp.values[c]].ravel()])
        out = 1.5 * loc + np.roll(loc, -1)
        np.add.at(eu, mv.values[c], out[:6].reshape(3, 2))
        np.add.at(ep, mp.values[c], out[6:])
    r.zero()
    op2.par_loop(k, cells, r(op2.INC, mm), w(op2.READ, mm), s(op2.READ))
    assert np.abs(r[0].data_ro - eu).max() < 1e-12 and np.abs(r[1].data_ro.ravel() - ep).max() < 1e-12
    r.zero()
    codegen.par_loop(k, cells, r(op2.INC, mm), w(op2.READ, mm), s(op2.READ), location="host")
    assert np.abs(r[0]._data - eu).max() < 1e-12 and np.abs(r[1]._data.ravel() - ep).max() < 1e-12
    # whole-vector operations act block by block
    w2 = op2.MixedDat(w.dataset)
    w.copy(w2)
    w2.axpy(2.0, w)
    assert abs(w2.inner(w) - 3.0 * w.inner(w)) < 1e-12 * w.inner(w)
    assert abs(w.norm() - np.sqrt((u.data_ro ** 2).sum() + (p.data_ro ** 2).sum())) < 1e-12
    w2 -= w
    w2 *= 0.5
    assert np.abs(w2[0].data_ro - u.data_ro).max() < 1e-14 and np.abs(w2[1].data_ro - p.data_ro).max() < 1e-14


@pytest.mark.parametrize("region", ["ALL", "ON_TOP", "ON_INTERIOR_FACETS"])
def test_variable_layers_on_device(engine, region):
    """Variable layers through op2.par_loop, device-resident and host-pointer mode, against the
    NumPy loop of tests/test_codegen.py::test_variable_layers at a size with uneven columns."""
    from firedrake_b200 import codegen
    lay, colstart, nnode = tc._variable_columns(seed=3, ncol=700)
    ncol = len(lay)
    cols = op2.ExtrudedSet(op2.Set(ncol), lay)
    nodes = op2.Set(nnode)
    m = op2.Map(cols, nodes, 2, colstart[:, None] + np.array([0, 1])[None, :], offset=[1, 1])
    xh = np.random.default_rng(0).standard_normal(nnode)
    x, y = op2.Dat(nodes, xh), op2.Dat(nodes)
    if region == "ON_INTERIOR_FACETS":
        k = op2.Kernel("static void k(double *y, const double *x, int layer) { for (int i = 0; i < 4; ++i) "
                       "y[i] += (i + 1) * x[3 - i] + layer; }", "k")
    else:
        k = op2.Kernel("static void k(double *y, const double *x, int layer) "
                       "{ y[0] += 2.0*x[0] + x[1] + layer; y[1] += x[0] - 3.0*x[1]; }", "k")
    ref = np.zeros(nnode)
    for c in range(ncol):
        cs, ce = lay[c, 0], lay[c, 1] - 1
        lo, hi = {"ALL": (cs, ce), "ON_TOP": (max(ce - 1, cs), ce), "ON_INTERIOR_FACETS": (cs, ce - 1)}[region]
        for l in range(lo, hi):
            b = colstart[c] + (l - cs)
            if region == "ON_INTERIOR_FACETS":
                idx = np.array([b, b + 1, b + 1, b + 2])
                np.add.at(ref, idx, np.array([(i + 1) * xh[idx[3 - i]] + l for i in range(4)]))
            else:
                ref[b] += 2 * xh[b] + xh[b + 1] + l
                ref[b + 1] += xh[b] - 3 * xh[b + 1]
    for location in ("device", "host"):
        y.zero()
        codegen.par_loop(k, cols, y(op2.INC, m), x(op2.READ, m), iteration_region=region, pass_layer_arg=True,
                         location=location)
        assert np.abs(y.data_ro - ref).max() < 1e-12

