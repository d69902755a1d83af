"""ctypes driver for the CPU oracle (TEST INFRASTRUCTURE -- see oracle.c header).

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s
``cpu_baseline`` / ``--impl reference`` legs may import this module.

Two builds of ``oracle.c``:

* ``_build/liboracle.so`` -- portable ``-march=x86-64-v3``; built by
  ``__graft_entry__.build()`` in the CPU container and shipped to the GPU box;
* ``-march=native`` as PyOP2's JIT uses (reference pyop2/compilation.py:341-363),
  compiled on first use in each process ON THE MACHINE THAT RUNS IT (the build
  machine's CPU may differ from the GPU host's), in a temporary directory that
  is removed once the library is loaded, so the source tree may be read-only.
  Used for timing when gcc is available, else falls back to the portable one.
"""
from __future__ import annotations

import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
BUILD = os.path.join(HERE, "_build")
SRC = [os.path.join(HERE, "oracle.c"), os.path.join(HERE, "dg_advection.c")]
BASE_FLAGS = ["-O3", "-ffast-math", "-fPIC", "-shared", "-std=gnu11", "-fopenmp",
              "-fno-math-errno"]

c_dp = ctypes.POINTER(ctypes.c_double)
c_ip = ctypes.POINTER(ctypes.c_int32)
c_lp = ctypes.POINTER(ctypes.c_int64)


def _compile(out, march):
    os.makedirs(os.path.dirname(out), exist_ok=True)
    cmd = ["gcc", *BASE_FLAGS, f"-march={march}", "-o", out, *SRC, "-lm"]
    subprocess.run(cmd, check=True, cwd=HERE, capture_output=True)
    return out


def build(force=False):
    out = os.path.join(BUILD, "liboracle.so")
    deps = SRC + [os.path.join(HERE, "hex_kernels.inc")]
    if force or not os.path.exists(out) or any(
            os.path.getmtime(d) > os.path.getmtime(out) for d in deps):
        _compile(out, "x86-64-v3")
    return out


def _load_native():
    tmp = tempfile.mkdtemp(prefix="fdb_oracle_")
    try:
        return ctypes.CDLL(_compile(os.path.join(tmp, "liboracle_native.so"), "native"))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


class _W(ctypes.Structure):
    _fields_ = [("start", ctypes.c_int), ("end", ctypes.c_int),
                ("layers", c_ip), ("y", c_dp), ("coords", c_dp), ("x", c_dp),
                ("map0", c_ip), ("off0", c_ip), ("map1", c_ip), ("off1", c_ip)]


_lib = {}


def lib(native=False):
    key = bool(native)
    if key in _lib:
        return _lib[key]
    L = None
    if native:
        try:
            L, path = _load_native(), "liboracle_native.so"
        except Exception:
            pass
    if L is None:
        path = build()
        L = ctypes.CDLL(path)
    L.orc_build_sparsity.restype = ctypes.c_int64
    L.orc_vec_dot.restype = ctypes.c_double
    _lib[key] = L
    L._path = path
    return L


def _d(a):
    assert a.dtype == np.float64 and a.flags.c_contiguous
    return a.ctypes.data_as(c_dp)


def _i(a):
    if a is None:
        return None
    assert a.dtype == np.int32 and a.flags.c_contiguous
    return a.ctypes.data_as(c_ip)


def _l(a):
    assert a.dtype == np.int64 and a.flags.c_contiguous
    return a.ctypes.data_as(c_lp)


def _tabs(el):
    """(B, D, CB, CD, wq) for a fiat_lite.Interval1D trial element; the
    coordinate element is P1 tabulated at the same points."""
    xq = el.xq
    CB = np.ascontiguousarray(np.stack([1.0 - xq, xq], axis=1))
    CD = np.ascontiguousarray(np.tile(np.array([-1.0, 1.0]), (len(xq), 1)))
    return (np.ascontiguousarray(el.B), np.ascontiguousarray(el.D), CB, CD,
            np.ascontiguousarray(el.wq))


def action_extruded(el, start, end, layers, y, coords, x, map0, off0, map1, off1,
                    cdim=1, alpha=1.0, beta=0.0, native=False):
    B, D, CB, CD, wq = _tabs(el)
    lay = np.ascontiguousarray(layers, dtype=np.int32)
    rc = lib(native).orc_wrap_action_extruded(
        el.degree, start, end, _i(lay), _d(y), _d(coords), _d(x), _i(map0), _i(off0),
        _i(map1), _i(off1), cdim, _d(B), _d(D), _d(CB), _d(CD), _d(wq),
        ctypes.c_double(alpha), ctypes.c_double(beta))
    if rc:
        raise RuntimeError(f"oracle action failed rc={rc}")
    return y


def matrix_extruded(el, start, end, layers, rowptr, colidx, vals, coords, map0, off0,
                    map1, off1, row_lgmap=None, col_lgmap=None, alpha=1.0, beta=0.0):
    B, D, CB, CD, wq = _tabs(el)
    lay = np.ascontiguousarray(layers, dtype=np.int32)
    rc = lib().orc_wrap_matrix_extruded(
        el.degree, start, end, _i(lay), len(rowptr) - 1, _l(rowptr), _i(colidx), _d(vals),
        _d(coords), _i(map0), _i(off0), _i(map1), _i(off1), _i(row_lgmap), _i(col_lgmap),
        _d(B), _d(D), _d(CB), _d(CD), _d(wq), ctypes.c_double(alpha), ctypes.c_double(beta))
    if rc:
        raise RuntimeError(f"oracle matrix assembly failed rc={rc}")
    return vals


def cell_action(el, coords24, w, alpha=1.0, beta=0.0):
    B, D, CB, CD, wq = _tabs(el)
    A = np.zeros(el.ndof ** 3)
    rc = lib().orc_cell_action(el.degree, _d(A), _d(np.ascontiguousarray(coords24)),
                               _d(np.ascontiguousarray(w)), _d(B), _d(D), _d(CB), _d(CD),
                               _d(wq), ctypes.c_double(alpha), ctypes.c_double(beta))
    assert rc == 0
    return A


def cell_matrix(el, coords24, alpha=1.0, beta=0.0):
    B, D, CB, CD, wq = _tabs(el)
    nd = el.ndof ** 3
    A = np.zeros((nd, nd))
    rc = lib().orc_cell_matrix(el.degree, _d(A), _d(np.ascontiguousarray(coords24)),
                               _d(B), _d(D), _d(CB), _d(CD), _d(wq),
                               ctypes.c_double(alpha), ctypes.c_double(beta))
    assert rc == 0
    return A


def build_sparsity(nrows, cmap, off=None, nlayers=1):
    """CSR pattern (rowptr int64, colidx int32) from a cell->node map."""
    ncells, arity = cmap.shape
    rowptr = np.zeros(nrows + 1, dtype=np.int64)
    dummy = np.zeros(1, dtype=np.int32)
    nnz = lib().orc_build_sparsity(nrows, ncells, nlayers, arity, _i(cmap), _i(off),
                                   _l(rowptr), _i(dummy), ctypes.c_int64(0))
    colidx = np.zeros(nnz, dtype=np.int32)
    rowptr[:] = 0
    lib().orc_build_sparsity(nrows, ncells, nlayers, arity, _i(cmap), _i(off),
                             _l(rowptr), _i(colidx), ctypes.c_int64(nnz))
    return rowptr, colidx


# -- P1 triangle tables -------------------------------------------------------
def tri_table_fiat(deg=2):
    """P1 basis in FIAT order (phi0 = 1-x-y, phi1 = x, phi2 = y) on a
    degree-2 exact 3-point rule (edge midpoints)."""
    pts = np.array([[0.5, 0.0], [0.5, 0.5], [0.0, 0.5]])
    w = np.full(3, 1.0 / 6.0)
    tab = np.stack([1 - pts[:, 0] - pts[:, 1], pts[:, 0], pts[:, 1]])
    dtab = np.array([[-1.0, -1.0], [1.0, 0.0], [0.0, 1.0]])
    return 3, np.ascontiguousarray(tab), np.ascontiguousarray(dtab), w


def tri_matrix(kind, start, end, rowptr, colidx, vals, coords, cmap, table,
               row_lgmap=None, col_lgmap=None, use_abs=1, beta=0.0):
    nq, tab, dtab, w = table
    rc = lib().orc_wrap_tri_matrix(
        {"mass": 0, "laplace": 1}[kind], start, end, len(rowptr) - 1, _l(rowptr),
        _i(colidx), _d(vals), _d(coords), _i(cmap), _i(row_lgmap), _i(col_lgmap),
        nq, _d(tab), _d(dtab), _d(w), use_abs, ctypes.c_double(beta))
    if rc:
        raise RuntimeError("oracle tri matrix failed")
    return vals


def tri_rhs(start, end, b, coords, f, cmap, table, use_abs=1):
    nq, tab, dtab, w = table
    lib().orc_wrap_tri_rhs(start, end, _d(b), _d(coords), _d(f), _i(cmap), nq,
                           _d(tab), _d(dtab), _d(w), use_abs)
    return b


def tri_action(start, end, y, coords, x, cmap, table, alpha=1.0, beta=0.0):
    nq, tab, dtab, w = table
    lib().orc_wrap_tri_action(start, end, _d(y), _d(coords), _d(x), _i(cmap), nq,
                              _d(tab), _d(dtab), _d(w), ctypes.c_double(alpha),
                              ctypes.c_double(beta))
    return y


def indirect_inc(start, end, cmap, edge_vals, node_vals):
    lib().orc_indirect_inc(start, end, cmap.shape[1], _i(cmap), _d(edge_vals), _d(node_vals))
    return node_vals


def action_workers(el, problems, cdim=1, alpha=1.0, beta=0.0, native=True):
    """Run one extruded action per worker thread, each on its own local
    problem dict(start,end,layers,y,coords,x,map0,off0,map1,off1)."""
    B, D, CB, CD, wq = _tabs(el)
    arr = (_W * len(problems))()
    keep = []
    for k, p in enumerate(problems):
        lay = np.ascontiguousarray(p["layers"], dtype=np.int32)
        keep.append(lay)
        arr[k] = _W(p["start"], p["end"], _i(lay), _d(p["y"]), _d(p["coords"]), _d(p["x"]),
                    _i(p["map0"]), _i(p["off0"]), _i(p["map1"]), _i(p["off1"]))
    rc = lib(native).orc_action_workers(el.degree, len(problems), arr, cdim, _d(B), _d(D),
                                        _d(CB), _d(CD), _d(wq), ctypes.c_double(alpha),
                                        ctypes.c_double(beta))
    if rc:
        raise RuntimeError("oracle workers failed")


def action_bench(el, mesh, V, x, nworkers, reps, cpu_ids=None, alpha=1.0, beta=0.0, native=True):
    """Pinned, first-touch timing of the extruded action: ``nworkers`` threads each run the
    template slab ``(mesh, V)`` on private copies, followed by the ghost-plane reduce between
    neighbouring slabs (``orc_action_bench`` in oracle.c).  Returns (times[reps], checksum)."""
    B, D, CB, CD, wq = _tabs(el)
    lay = np.ascontiguousarray([0, mesh.layers], dtype=np.int32)
    hi = np.ascontiguousarray(V.plane_nodes(mesh.nx), dtype=np.int32)
    lo = np.ascontiguousarray(V.plane_nodes(0), dtype=np.int32)
    assert hi.size == lo.size
    times = np.zeros(reps)
    chk = ctypes.c_double(0.0)
    ids = None if cpu_ids is None else np.ascontiguousarray(cpu_ids, dtype=np.int32)
    m0 = np.ascontiguousarray(V.cell_node_map, dtype=np.int32)
    m1 = np.ascontiguousarray(mesh.coord_map, dtype=np.int32)
    off0 = np.ascontiguousarray(V.offset, dtype=np.int32)
    off1 = np.ascontiguousarray(mesh.coord_offset, dtype=np.int32)
    coords = np.ascontiguousarray(mesh.coordinates, dtype=np.float64)
    L = lib(native)
    rc = L.orc_action_bench(el.degree, int(nworkers), int(reps), _i(ids), int(mesh.num_base_cells),
                            _i(lay), ctypes.c_int64(V.node_count),
                            ctypes.c_int64(mesh.coord_space.node_count), _d(coords), _d(x), _i(m0),
                            int(V.arity), _i(off0), _i(m1), _i(off1), int(hi.size), _i(hi), _i(lo),
                            _d(B), _d(D), _d(CB), _d(CD), _d(wq), ctypes.c_double(alpha),
                            ctypes.c_double(beta), _d(times), ctypes.byref(chk))
    if rc:
        raise RuntimeError("oracle action_bench failed")
    return times, chk.value


def action_extruded_parallel(el, mesh, y, coords, x, map0, off0, map1, off1, cdim=1, alpha=1.0,
                             beta=0.0, nthreads=None, native=False, ncells=None):
    """``action_extruded`` over base cells ``[0, ncells)`` of ``mesh`` with several threads:
    bands of base-cell columns (constant ``mesh.cell_ix``), even bands then odd bands
    (``orc_action_bands``).  Same result as the sequential wrapper up to summation order
    across bands.  Needs ``mesh.cell_ix`` (structured base mesh)."""
    import os
    ncells = mesh.num_base_cells if ncells is None else ncells
    ix = np.asarray(mesh.cell_ix[:ncells])
    # runs of consecutive cells with the same ix
    brk = np.flatnonzero(np.diff(ix)) + 1
    rs = np.concatenate([[0], brk]).astype(np.int32)
    re_ = np.concatenate([brk, [ncells]]).astype(np.int32)
    band_of_run = ix[rs]
    order = np.argsort(band_of_run, kind="stable")
    rs, re_, band_of_run = rs[order], re_[order], band_of_run[order]
    nb = int(band_of_run.max()) + 1 if len(band_of_run) else 0
    first = np.searchsorted(band_of_run, np.arange(nb + 1)).astype(np.int32)
    B, D, CB, CD, wq = _tabs(el)
    lay = np.ascontiguousarray([0, mesh.layers], dtype=np.int32)
    nt = nthreads or len(os.sched_getaffinity(0))
    rc = lib(native).orc_action_bands(el.degree, nb, _i(first), _i(np.ascontiguousarray(rs)),
                                      _i(np.ascontiguousarray(re_)), _i(lay), _d(y), _d(coords), _d(x),
                                      _i(map0), _i(off0), _i(map1), _i(off1), int(cdim), _d(B), _d(D),
                                      _d(CB), _d(CD), _d(wq), ctypes.c_double(alpha),
                                      ctypes.c_double(beta), int(nt))
    if rc:
        raise RuntimeError("oracle action_bands failed")
    return y


def vec_axpy(a, x, y, native=True):
    lib(native).orc_vec_axpy(ctypes.c_int64(x.size), ctypes.c_double(a), _d(x), _d(y))


def vec_aypx(a, x, y, native=True):
    lib(native).orc_vec_aypx(ctypes.c_int64(x.size), ctypes.c_double(a), _d(x), _d(y))


def vec_dot(x, y, native=True):
    return float(lib(native).orc_vec_dot(ctypes.c_int64(x.size), _d(x), _d(y)))


def num_threads():
    return lib().orc_num_threads()


# -- DG advection (reference demos/DG_advection) ------------------------------
c_up = ctypes.POINTER(ctypes.c_uint32)


def dq1_end_values(variant="gl"):
    """(2, 2): DQ1 1-D basis (nodes = 2 Gauss points for the default spectral
    variant, interval ends for "equispaced") evaluated at x = 0 and x = 1."""
    from firedrake_b200.fiat_lite import interval_element
    el = interval_element(1, 2, variant)
    B, _ = el.tabulate([0.0, 1.0])
    return np.ascontiguousarray(B)


def dg_rhs(mesh, q, u, dt, q_in=1.0, nq=3, variant="gl", out=None):
    """assemble(L1) of the DG advection demo: cell + exterior + interior facets."""
    from firedrake_b200.fiat_lite import gauss_legendre
    L = lib()
    xq, wq = gauss_legendre(nq)
    Bend = dq1_end_values(variant)
    if out is None:
        out = np.zeros(mesh.num_cells * 4)
    uu = np.ascontiguousarray(u, dtype=np.float64)
    fl_e = np.ascontiguousarray(mesh.ext_facet_local, dtype=np.uint32)
    fl_i = np.ascontiguousarray(mesh.int_facet_local, dtype=np.uint32)
    L.orc_dg_cells(0, mesh.num_cells, _d(out), _d(mesh.coordinates), _d(q), _d(uu), _i(mesh.dg1_map),
                   _i(mesh.coord_map), nq, _d(Bend), _d(wq), _d(xq), ctypes.c_double(dt))
    L.orc_dg_exterior_facets(0, len(mesh.ext_facet_cells), _d(out), _d(mesh.coordinates), _d(q), _d(uu),
                             _i(mesh.ext_facet_cells), fl_e.ctypes.data_as(c_up), _i(mesh.dg1_map),
                             _i(mesh.coord_map), nq, _d(Bend), _d(wq), _d(xq), ctypes.c_double(dt),
                             ctypes.c_double(q_in))
    L.orc_dg_interior_facets(0, len(mesh.int_facet_cells), _d(out), _d(mesh.coordinates), _d(q), _d(uu),
                             _i(mesh.int_facet_cells), fl_i.ctypes.data_as(c_up), _i(mesh.dg1_map),
                             _i(mesh.coord_map), nq, _d(Bend), _d(wq), _d(xq), ctypes.c_double(dt))
    return out
