"""Host logic of the Python layers against a MOCK engine (tests/_mock_engine.py).

Runs, on the CPU, test functions that normally need the GPU: the mock replaces the C
ABI (device memory = host memory, generated wrappers through their host build, the
hand-written Helmholtz kernels through the oracle), so what is checked here is the
Python side -- argument marshalling, residency / dat_version bookkeeping, lgmap
swapping, BC handling, the V-cycle and Krylov loops -- not the device code.

Two groups: (1) tests that already PASS on a real B200 (they calibrate the mock: if
the mock mis-emulated the ABI these would fail), (2) the tests of tests/test_jit_gpu.py
(generic wrapper path, multigrid, solve front end), which also pass on the GPU since round 2.
"""
import numpy as np
import pytest

import _mock_engine as me
import test_assemble_gpu as ta
import test_jit_gpu as tj
import test_matrix_gpu as tm
import test_zz_mixed_mat_gpu as tz


@pytest.fixture()
def mock(oracle):
    with me.install(oracle) as eng:
        yield eng


# ---- (1) calibration: GPU-validated tests must also pass on the mock
def test_mock_runs_validated_matrix_tests(mock, oracle):
    tm.test_sparsity_matches_reference_semantics(mock, oracle, 2)
    tm.test_matrix_matches_oracle(mock, oracle, -1, 2, 1.0, 1.0)     # matrix_kernel fixture value: auto
    tm.test_bc_lgmaps_diagonal_and_matvec(mock, oracle, -1)


def test_mock_runs_validated_assemble_tests(mock, oracle):
    ta.test_matfree_equals_assembled_with_bcs(mock)
    ta.test_poisson_solve_strong_bcs_extrusion(mock)
    ta.test_cg_matches_scipy(mock)
    ta.test_get_diagonal(mock)
    ta.test_submatrix_and_duplicate_of_matrix_free_context(mock)


# ---- (2) the post-budget code paths
def test_generic_parloops_host_logic(mock):
    tj.test_golden_mass_and_rhs(mock)
    tj.test_blocked_matrix_generic_path(mock)
    tj.test_permuted_map_and_subset(mock)
    tj.test_host_pointer_mode_generic(mock)


def test_access_modes_host_logic(mock):
    tj.test_access_modes(mock)


def test_mixed_dat_host_logic(mock):
    tj.test_mixed_dat_parloop_and_vector_operations(mock)


@pytest.mark.parametrize("extruded", [False, True])
def test_mixed_mat_host_logic(mock, extruded):
    """Monolithic mixed matrices: dof-expanded block maps, MatBlock arguments, block lgmaps, mult on MixedDats."""
    tz.test_mixed_mat_monolithic(mock, extruded)


@pytest.mark.parametrize("region", ["ALL", "ON_TOP", "ON_INTERIOR_FACETS"])
def test_variable_layers_host_logic(mock, region):
    tj.test_variable_layers_on_device(mock, region)


def test_periodic_extrusion_host_logic(mock, oracle):
    tj.test_periodic_extrusion_on_device(mock, oracle)


def test_generic_vs_fast_path_host_logic(mock, oracle):
    tj.test_generic_extruded_action_equals_fast_path_and_oracle(mock, oracle)
    tj.test_expression_interpolation(mock)


def test_vector_space_assemble_host_logic(mock, oracle):
    tj.test_vector_space_matrix_fast_path(mock, oracle, -1, 1, 2)
    tj.test_mult_transpose(mock)


def test_mg_transfers_host_logic(mock):
    tj.test_mg_transfers_on_device(mock)


def test_mg_vcycle_host_logic(mock):
    tj.test_mg_preconditioned_cg_is_mesh_independent(mock)


def test_zero_forms_host_logic(mock):
    tj.test_zero_forms_dx_and_exterior_facets(mock)
    tj.test_dense_linear_algebra_callables(mock)
    tj.test_interior_facet_functionals(mock)


def test_helmholtz_convergence_host_logic(mock):
    tj.test_helmholtz_convergence_rates(mock, 2, (2, 4), 2.9)
    tj.test_helmholtz_convergence_rates(mock, 3, (1, 3), 3.9)


def test_affine_variant_host_logic(mock, oracle, monkeypatch):
    tj.test_affine_cell_variant(mock, oracle, 2, monkeypatch)


def test_dat_algebra_host_logic(mock):
    """Dat.copy / += / -= / *= / maxpy (pyop2/types/dat.py:312-540) keep host and device copies and
    dat_version consistent."""
    from firedrake_b200 import op2
    s = op2.Set(50)
    rng = np.random.default_rng(0)
    a0, b0 = rng.standard_normal(50), rng.standard_normal(50)
    a, b, c = op2.Dat(s, a0.copy()), op2.Dat(s, b0.copy()), op2.Dat(s)     # Dat wraps the array it is given
    v = a.dat_version
    a += b
    assert a.dat_version > v and np.allclose(a.data_ro, a0 + b0)
    a -= b
    a *= 3.0
    a *= b
    assert np.allclose(a.data_ro, 3 * a0 * b0)
    a.copy(c)
    assert np.allclose(c.data_ro, a.data_ro)
    c.maxpy([2.0, -1.0], [a, b])
    assert np.allclose(c.data_ro, 3 * (3 * a0 * b0) - b0)
    c.data[:] = 1.0                                   # host write, then device op must see it
    c += b
    assert np.allclose(c.data_ro, 1 + b0)
    # binary operators return new Dats; scalars shift / scale
    f = a + b
    g = 2.0 * a - b + 1.5
    h = -(a / 4.0) + (1.0 - b)
    assert f is not a and np.allclose(f.data_ro, a.data_ro + b.data_ro)
    assert np.allclose(g.data_ro, 2 * a.data_ro - b.data_ro + 1.5)
    assert np.allclose(h.data_ro, -a.data_ro / 4 + 1 - b.data_ro)
    g /= 2.0
    assert np.allclose(g.data_ro, (2 * a.data_ro - b.data_ro + 1.5) / 2)
    assert a.split() == (a,) and len(a) == 1 and a[0] is a and list(a) == [a]
    # write-only host access does not download; save / load round trip
    v0 = h.dat_version
    h.data_wo[...] = 7.0
    assert h.dat_version > v0 and np.all(h.data_ro == 7.0)
    import os
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        fn = os.path.join(tmp, "dat")
        f.save(fn)
        h.load(fn)
    assert np.array_equal(h.data_ro, f.data_ro)
    # copy restricted to a subset: the other rows of the target keep their values
    sub = op2.Subset(s, np.array([3, 7, 8, 41], dtype=np.int32))
    d = op2.Dat(op2.DataSet(s, 2), rng.standard_normal((50, 2)))
    e = op2.Dat(op2.DataSet(s, 2), np.full((50, 2), -5.0))
    d.copy(e, subset=sub)
    want = np.full((50, 2), -5.0)
    want[sub.indices] = d.data_ro[sub.indices]
    assert np.array_equal(e.data_ro, want)


@pytest.mark.parametrize("pc", ["none", "jacobi", "mg"])
def test_solve_front_end_host_logic(mock, pc):
    tj.test_solve_front_end(mock, pc)


def test_variable_coefficient_host_logic(mock, oracle):
    tj.test_variable_coefficient_form(mock, oracle)


def test_mat_path_maps_must_be_the_sparsity_maps(mock):
    """``mat(op2.INC, (rmap, cmap))`` with maps other than the sparsity's raises MapValueError
    (pyop2/types/mat.py:439-441), even when they have the same iteration and target sets: the scatter
    locates entries through the sparsity's map, so another map's values would land at wrong positions."""
    from firedrake_b200 import op2
    import test_matrix_gpu as tm
    mesh = tm.ExtrudedHexMesh(3, 2, 3, warp=0.05)
    V, cells, nodes, m0, m1, X = tm.setup(mesh, 2)
    mat = op2.Mat(op2.Sparsity((nodes, nodes), [(m0, m0, None)]))
    perm = np.random.default_rng(0).permutation(mesh.num_base_cells)
    m2 = op2.Map(cells, nodes, V.arity, V.cell_node_map[perm], offset=V.offset)
    m0_copy = op2.Map(cells, nodes, V.arity, V.cell_node_map.copy(), offset=V.offset)
    for path in [(m2, m2), (m0, m2), (m2, m0), (m0_copy, m0_copy)]:
        with pytest.raises(op2.MapValueError):
            mat(op2.INC, path)
    k = op2.Kernel("helmholtz", degree=2, rank=2)
    op2.par_loop(k, cells, mat(op2.INC, (m0, m0)), X(op2.READ, m1))
    # blocked matrices take the same check
    bmat = op2.Mat(op2.Sparsity((op2.DataSet(nodes, 2), op2.DataSet(nodes, 2)), [(m0, m0, None)]))
    with pytest.raises(op2.MapValueError):
        bmat(op2.INC, (m2, m2))
    bmat(op2.INC, (m0, m0))
