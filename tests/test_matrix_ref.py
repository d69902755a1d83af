"""Pins of the NumPy reference assembler (tests/_matrix_ref.py) that the GPU matrix sweep
(tests/test_matrix_shapes_gpu.py) trusts: its element matrices against the explicit dense
evaluation of test_oracle_pins, and whole assembled matrices (pattern, values, lgmaps, ranges,
subsets) against the oracle's CSR assembly."""
import numpy as np
import pytest

import _matrix_ref as R
from firedrake_b200.fiat_lite import interval_element
from firedrake_b200.utility_meshes import ExtrudedHexMesh
from test_oracle_pins import dense_element_matrix


@pytest.mark.parametrize("p", [1, 2, 3, 4])
def test_element_matrix_vs_dense(p):
    rng = np.random.default_rng(10 + p)
    X = np.array([[bx, by, bz] for bx in (0, 1) for by in (0, 1) for bz in (0, 1)], dtype=float)
    X = X * [1.0, 0.7, 1.3] + 0.12 * rng.standard_normal((8, 3))      # non-affine hex
    for alpha, beta in [(1.0, 0.0), (0.0, 1.0), (1.0, 0.7)]:
        Aref = dense_element_matrix(p, X, alpha, beta)
        A = R.element_matrices(p, X[None], alpha, beta)[0]
        assert np.abs(A - Aref).max() < 1e-13 * np.abs(Aref).max()


def oracle_values(oracle, mesh, V, p, alpha, beta, start=0, end=None, lg=None):
    rowptr, colidx = oracle.build_sparsity(V.node_count, V.cell_node_map, V.offset, mesh.nz)
    vals = np.zeros(len(colidx))
    end = mesh.num_base_cells if end is None else end
    oracle.matrix_extruded(interval_element(p), start, end, [0, mesh.layers], rowptr, colidx, vals,
                           mesh.coordinates, V.cell_node_map, V.offset, mesh.coord_map, mesh.coord_offset,
                           lg, lg, alpha, beta)
    return rowptr, colidx, vals


MESHES = [dict(nx=3, ny=2, nz=3, warp=0.06, permute_seed=5), dict(nx=2, ny=3, nz=2, warp=0.04, permute_seed=9)]


@pytest.mark.parametrize("p", [1, 2, 3, 4])
@pytest.mark.parametrize("m", [0, 1])
def test_assembled_matrix_vs_oracle(oracle, p, m):
    mesh = ExtrudedHexMesh(**MESHES[m])
    V = mesh.function_space(p)
    cells = R.Cells.extruded(mesh, V)
    rowptr, colidx = R.pattern(V.node_count, cells)
    for alpha, beta in [(1.0, 0.0), (0.0, 1.0), (1.0, 0.7)]:
        ro, co, vo = oracle_values(oracle, mesh, V, p, alpha, beta)
        assert np.array_equal(rowptr, ro) and np.array_equal(colidx, co)
        vals = R.assemble(p, alpha, beta, mesh.coordinates, rowptr, colidx, cells)
        assert np.abs(vals - vo).max() < 1e-13 * np.abs(vo).max()
    # a range of columns, and BC masks (the oracle drops the masked entries but writes no diagonal)
    ncols = mesh.num_base_cells
    ro, co, vo = oracle_values(oracle, mesh, V, p, 1.0, 0.7, start=1, end=ncols - 1)
    vals = R.assemble(p, 1.0, 0.7, mesh.coordinates, rowptr, colidx,
                      R.Cells.extruded(mesh, V, np.arange(1, ncols - 1)))
    assert np.abs(vals - vo).max() < 1e-13 * np.abs(vo).max()
    bc = np.union1d(V.boundary_nodes("bottom"), V.boundary_nodes(3))
    lg = np.arange(V.node_count, dtype=np.int32)
    lg[bc] = -1
    mask = lg < 0
    _, _, vo = oracle_values(oracle, mesh, V, p, 1.0, 0.7, lg=lg)
    vals = R.assemble(p, 1.0, 0.7, mesh.coordinates, rowptr, colidx, cells, mask, mask)
    assert np.abs(vals - vo).max() < 1e-13 * np.abs(vo).max()
    vals = R.assemble(p, 1.0, 0.7, mesh.coordinates, rowptr, colidx, cells, mask, mask, diag_rows=bc)
    A = R.to_scipy(rowptr, colidx, vals, V.node_count)
    assert np.array_equal(A.diagonal()[bc], np.ones(len(bc)))
    # the diagonal helper is the diagonal of the unmasked matrix
    vals = R.assemble(p, 1.0, 0.7, mesh.coordinates, rowptr, colidx, cells)
    d = R.diagonal(p, 1.0, 0.7, mesh.coordinates, V.node_count, cells)
    assert np.abs(d - R.to_scipy(rowptr, colidx, vals, V.node_count).diagonal()).max() < 1e-14 * np.abs(d).max()


def test_subset_equals_sum_of_columns(oracle):
    p = 2
    mesh = ExtrudedHexMesh(**MESHES[0])
    V = mesh.function_space(p)
    rowptr, colidx = R.pattern(V.node_count, R.Cells.extruded(mesh, V))
    cols = [4, 0, 5]
    vals = R.assemble(p, 1.0, 0.0, mesh.coordinates, rowptr, colidx, R.Cells.extruded(mesh, V, cols))
    vo = sum(oracle_values(oracle, mesh, V, p, 1.0, 0.0, start=c, end=c + 1)[2] for c in cols)
    assert np.abs(vals - vo).max() < 1e-13 * np.abs(vo).max()
