"""TEST INFRASTRUCTURE: a host stand-in for libfdb200's C ABI, so that the PYTHON
layers (op2 / assemble / codegen / mg: argument marshalling, dat_version and
residency bookkeeping, lgmap swapping, BC handling, V-cycle and Krylov logic)
can be exercised without a GPU.  "Device" memory is host memory; generated
wrappers run through the host build of their generated body (tests/_jit_host.py),
the hand-written Helmholtz kernels are replaced by the oracle.  Nothing here is
importable from the product; `install()` monkeypatches firedrake_b200._lib for
the duration of a test only.  What this can NOT check is the device code itself
(CUDA prelude, launchers, hand-written kernels): that is what `-m gpu` is for.
"""
import ctypes as C

import numpy as np

from firedrake_b200 import _lib
from firedrake_b200.fiat_lite import interval_element

import _jit_host as jh


def _obj(x):
    """The ctypes object behind byref(x) / pointer / plain value."""
    return x._obj if hasattr(x, "_obj") else x


def _addr(p):
    if p is None:
        return 0
    if isinstance(p, int):
        return p
    if isinstance(p, C.c_void_p):
        return p.value or 0
    if hasattr(p, "contents"):                      # POINTER(...)
        return C.cast(p, C.c_void_p).value or 0
    return int(p)


def _view(addr, count, dtype=np.float64):
    if count == 0:
        return np.zeros(0, dtype=dtype)
    buf = (C.c_char * (count * np.dtype(dtype).itemsize)).from_address(_addr(addr))
    return np.frombuffer(buf, dtype=dtype, count=count)


class _Mat:
    def __init__(self, nrows, rowptr, colidx, bs, cmap, off, nlay):
        self.nrows, self.rowptr, self.colidx, self.bs = nrows, rowptr, colidx, bs
        self.vals = np.zeros(len(colidx) * bs * bs)
        self.row_lg = self.col_lg = None
        self.cmap, self.off, self.nlay = cmap, off, nlay

    def host_csr(self):
        h = jh.HostCSR.__new__(jh.HostCSR)
        h.nrows, h.bs, h.rowptr, h.colidx, h.vals = self.nrows, self.bs, self.rowptr, self.colidx, self.vals
        h.row_lg, h.col_lg = self.row_lg, self.col_lg
        return h


class MockEngine:
    def __init__(self, oracle):
        self.oracle = oracle
        self.bufs = {}          # address -> ctypes buffer (keeps "device" memory alive)
        self.kernels = {}
        self.mats = {}
        self._next = 1000
        self._err = b""
        self.launches = 0

    # ------------------------------------------------------------ runtime / memory
    def fdb_last_error(self):
        return self._err

    def _fail(self, msg):
        self._err = msg.encode()
        return 1

    def fdb_synchronize(self):
        return 0

    # timers (bench / run_configs): wall clock stands in for CUDA events
    def fdb_timer_create(self, out):
        _obj(out).value = 1
        return 0

    def fdb_timer_start(self, t):
        import time
        self._t0 = time.perf_counter()
        return 0

    def fdb_timer_stop(self, t, ms):
        import time
        _obj(ms).value = (time.perf_counter() - self._t0) * 1e3
        return 0

    def fdb_timer_destroy(self, t):
        return 0

    def fdb_set_option(self, name, value):
        return 0

    def fdb_get_option(self, name, out):
        _obj(out).value = -1
        return 0

    def fdb_launch_count(self):
        return self.launches

    def fdb_malloc(self, n):
        b = (C.c_char * max(int(n), 1))()
        a = C.addressof(b)
        self.bufs[a] = b
        return a

    fdb_host_alloc = fdb_malloc

    def fdb_free(self, p):
        self.bufs.pop(_addr(p), None)
        return 0

    fdb_host_free = fdb_free

    def fdb_memset(self, p, v, n):
        C.memset(_addr(p), v, n)
        return 0

    def _copy(self, dst, src, n):
        C.memmove(_addr(dst), _addr(src), n)
        return 0

    fdb_memcpy_h2d = fdb_memcpy_d2h = fdb_memcpy_d2d = _copy

    def fdb_zero_background(self, p, n):
        return self.fdb_memset(p, 0, n)

    def fdb_background_barrier(self):
        return 0

    def fdb_mirror_drop(self, p):
        return 0

    # ------------------------------------------------ communicator / halos over gloo
    # (set .dist = torch.distributed after init_process_group to emulate N ranks)
    dist = None

    def fdb_comm_size(self):
        return self.dist.get_world_size() if self.dist is not None else 1

    def fdb_comm_rank(self):
        return self.dist.get_rank() if self.dist is not None else 0

    def fdb_allreduce(self, dev, n, op):
        import torch
        if self.dist is None:
            return 0
        v = _view(dev, n)
        t = torch.from_numpy(v.copy())
        self.dist.all_reduce(t, op={0: self.dist.ReduceOp.SUM, 1: self.dist.ReduceOp.MIN,
                                    2: self.dist.ReduceOp.MAX}[op])
        v[:] = t.numpy()
        return 0

    def fdb_halo_create(self, nneigh, ranks, send_counts, send_idx, recv_counts, recv_idx, max_cdim, out):
        rk = _view(ranks, nneigh, np.int32)
        sc, rc = _view(send_counts, nneigh, np.int32), _view(recv_counts, nneigh, np.int32)
        si, ri = _view(send_idx, int(sc.sum()), np.int32).copy(), _view(recv_idx, int(rc.sum()), np.int32).copy()
        so, ro = np.concatenate([[0], np.cumsum(sc)]), np.concatenate([[0], np.cumsum(rc)])
        self._next += 1
        self.kernels[self._next] = [(int(rk[i]), si[so[i]:so[i + 1]], ri[ro[i]:ro[i + 1]]) for i in range(nneigh)]
        _obj(out).value = self._next
        return 0

    def fdb_halo_destroy(self, h):
        self.kernels.pop(_addr(h), None)
        return 0

    def _halo(self, h, dat, cdim, reverse):
        from _gloo_halo import exchange
        neigh = self.kernels[_addr(h)]
        top = max([int(max(s.max(initial=-1), r.max(initial=-1))) for _, s, r in neigh] + [-1]) + 1
        data = _view(dat, top * cdim).reshape(top, cdim)
        for c in range(cdim):                       # the gloo helper moves scalar fields
            col = np.ascontiguousarray(data[:, c])
            exchange(neigh, col, reverse)
            data[:, c] = col
        return 0

    def fdb_halo_global_to_local_begin(self, h, dat, cdim):
        return self._halo(h, dat, cdim, False)

    def fdb_halo_global_to_local_end(self, h, dat, cdim):
        return 0

    def fdb_halo_local_to_global_begin(self, h, dat, cdim):
        return self._halo(h, dat, cdim, True)

    def fdb_halo_local_to_global_end(self, h, dat, cdim):
        return 0

    # ---------------------------------------------------------------- vector algebra
    def fdb_vec_axpy(self, n, a, x, y):
        _view(y, n)[:] += a * _view(x, n)
        return 0

    def fdb_vec_aypx(self, n, a, x, y):
        yv = _view(y, n)
        yv[:] = _view(x, n) + a * yv
        return 0

    def fdb_vec_scale(self, n, a, x):
        _view(x, n)[:] *= a
        return 0

    def fdb_vec_gather(self, n, idx, src, dst):
        if n:
            i = np.ctypeslib.as_array(C.cast(idx, C.POINTER(C.c_int32)), (n,))
            _view(dst, n)[:] = np.ctypeslib.as_array(C.cast(src, C.POINTER(C.c_double)), (int(i.max()) + 1,))[i]
        return 0

    def fdb_vec_scatter(self, n, idx, src, dst):
        if n:
            i = np.ctypeslib.as_array(C.cast(idx, C.POINTER(C.c_int32)), (n,))
            np.ctypeslib.as_array(C.cast(dst, C.POINTER(C.c_double)), (int(i.max()) + 1,))[i] = _view(src, n)
        return 0

    def fdb_vec_fill(self, n, a, x):
        if n:
            _view(x, n)[:] = a
        return 0

    def fdb_vec_dot(self, n, x, y, out):
        _obj(out).value = float(_view(x, n) @ _view(y, n))
        return 0

    def fdb_vec_pointwise_mult(self, n, x, y, w):
        _view(w, n)[:] = _view(x, n) * _view(y, n)
        return 0

    def fdb_dat_zero_nodes(self, dat, cdim, nodes, n):
        idx = _view(nodes, n, np.int32)
        _view(dat, (int(idx.max()) + 1) * cdim if n else 0).reshape(-1, cdim)[idx] = 0.0
        return 0

    def fdb_dat_set_nodes(self, dat, src, cdim, nodes, n):
        idx = _view(nodes, n, np.int32)
        m = (int(idx.max()) + 1) * cdim if n else 0
        _view(dat, m).reshape(-1, cdim)[idx] = _view(src, m).reshape(-1, cdim)[idx]
        return 0

    def fdb_dat_set_nodes_scalar(self, dat, value, cdim, nodes, n):
        idx = _view(nodes, n, np.int32)
        _view(dat, (int(idx.max()) + 1) * cdim if n else 0).reshape(-1, cdim)[idx] = value
        return 0

    # ----------------------------------------------------------------------- matrices
    def _new_mat(self, nrows, map_host, ncols, arity, off_host, nlay, bs, out):
        cmap = _view(map_host, ncols * arity, np.int32).reshape(ncols, arity).copy()
        off = _view(off_host, arity, np.int32).copy() if _addr(off_host) else None
        rowptr, colidx = self.oracle.build_sparsity(nrows, cmap, off, nlay)
        self._next += 1
        self.mats[self._next] = _Mat(nrows, np.asarray(rowptr, dtype=np.int64),
                                     np.asarray(colidx, dtype=np.int32), bs, cmap, off, nlay)
        _obj(out).value = self._next
        return 0

    def fdb_mat_create(self, nrows, m, ncols, arity, off, nlay, out):
        return self._new_mat(nrows, m, ncols, arity, off, nlay, 1, out)

    def fdb_mat_create_blocked(self, nrows, m, ncols, arity, off, nlay, bs, out):
        return self._new_mat(nrows, m, ncols, arity, off, nlay, bs, out)

    def fdb_mat_destroy(self, h):
        self.mats.pop(_addr(h), None)
        return 0

    def fdb_mat_nnz(self, h, nnz, nrows):
        m = self.mats[_addr(h)]
        _obj(nnz).value, _obj(nrows).value = len(m.colidx), m.nrows
        return 0

    def fdb_mat_zero(self, h):
        self.mats[_addr(h)].vals[:] = 0
        return 0

    def fdb_mat_set_lgmaps(self, h, r, c):
        m = self.mats[_addr(h)]
        n = m.nrows * m.bs
        m.row_lg = _view(r, n, np.int32).copy() if _addr(r) else None
        m.col_lg = _view(c, n, np.int32).copy() if _addr(c) else None
        return 0

    def fdb_mat_set_diagonal_blocked(self, h, rows, n, value, idx):
        m = self.mats[_addr(h)]
        blocks = m.vals.reshape(-1, m.bs, m.bs)
        for r in _view(rows, n, np.int32):
            k = m.rowptr[r] + np.searchsorted(m.colidx[m.rowptr[r]:m.rowptr[r + 1]], r)
            for a in range(m.bs):
                if idx < 0 or idx == a:
                    blocks[k, a, a] = value
        return 0

    def fdb_mat_set_diagonal(self, h, rows, n, value):
        return self.fdb_mat_set_diagonal_blocked(h, rows, n, value, -1)

    def fdb_mat_get_csr(self, h, rowptr, colidx, vals):
        m = self.mats[_addr(h)]
        for dst, src in ((rowptr, m.rowptr), (colidx, m.colidx), (vals, m.vals)):
            if _addr(dst):
                C.memmove(_addr(dst), src.ctypes.data, src.nbytes)
        return 0

    def fdb_mat_mult(self, h, x, y):
        m = self.mats[_addr(h)]
        bs = m.bs
        xv = _view(x, m.nrows * bs).reshape(-1, bs)
        yv = _view(y, m.nrows * bs).reshape(-1, bs)
        blocks = m.vals.reshape(-1, bs, bs)
        rows = np.repeat(np.arange(m.nrows), np.diff(m.rowptr))
        yv[:] = 0
        np.add.at(yv, rows, np.einsum("kab,kb->ka", blocks, xv[m.colidx]))
        return 0

    def fdb_cells_are_affine(self, coords, map1, off1, start, end, nlay, result):
        off = _view(off1, 8, np.int32) if _addr(off1) else np.zeros(8, dtype=np.int32)
        m = _view(map1, end * 8, np.int32).reshape(end, 8)[start:end]
        idx = m[:, None, :] + off[None, None, :] * np.arange(nlay)[None, :, None]
        X = _view(coords, (int(idx.max()) + 1) * 3).reshape(-1, 3)[idx]          # (cols, layers, 8, 3)
        v = lambda b: X[:, :, b, :]
        bad = ((v(6) - v(4) - v(2) + v(0)) != 0) | ((v(3) - v(2) - v(1) + v(0)) != 0) | \
              ((v(5) - v(4) - v(1) + v(0)) != 0) | ((v(7) - v(6) - v(5) - v(3) + v(4) + v(2) + v(1) - v(0)) != 0)
        _obj(result).value = 0 if bad.any() else 1
        return 0

    # ------------------------------------------------------------------------ kernels
    def fdb_kernel_create(self, desc, out):
        d = _obj(desc)
        if d.form != _lib.FORM_HELMHOLTZ or d.cell != _lib.CELL_HEX_EXTRUDED:
            return self._fail("mock engine: only the extruded Helmholtz family is emulated")
        n = (d.degree + 1) ** 3
        k = dict(kind="helmholtz", degree=d.degree, rank=d.rank, cdim=d.cdim, alpha=d.alpha, beta=d.beta,
                 diagonal=d.diagonal, off0=np.array(d.offset0[:n], dtype=np.int32),
                 off1=np.array(d.offset1[:8], dtype=np.int32))
        self._next += 1
        self.kernels[self._next] = k
        _obj(out).value = self._next
        return 0

    def fdb_wrapper_create(self, desc, out):
        d = _obj(desc)
        real = self.real                                     # source generation needs no GPU
        need = C.c_size_t()
        if real.fdb_wrapper_source(C.byref(d), None, 0, C.byref(need)):
            self._err = real.fdb_last_error()
            return 1
        buf = C.create_string_buffer(need.value)
        real.fdb_wrapper_source(C.byref(d), buf, need.value, C.byref(need))
        name = d.kernel_name.decode()
        fn, keep = jh.build(buf.value.decode(), name)
        args = [(d.args[i].kind, d.args[i].access, d.args[i].dtype, d.args[i].dim) for i in range(d.nargs)]
        self._next += 1
        self.kernels[self._next] = dict(kind="jit", fn=fn, keep=keep, args=args, extruded=d.extruded,
                                        subset=d.subset, region=d.iteration_region, name=name,
                                        varlay=d.variable_layers, periodic=d.extruded_periodic)
        _obj(out).value = self._next
        return 0

    def fdb_kernel_destroy(self, h):
        self.kernels.pop(_addr(h), None)
        return 0

    def fdb_kernel_call(self, h, ca):
        k = self.kernels[_addr(h)]
        a = _obj(ca)
        self.launches += 1
        if k["kind"] == "jit":
            return self._call_jit(k, a)          # host location: "mirrors" are the host buffers themselves
        if a.location != _lib.LOC_DEVICE:
            return self._fail("mock engine: device-location calls only for the hand-written kernels")
        return self._call_helmholtz(k, a)

    def _call_jit(self, k, a):
        p = jh.WrapParams()
        p.start, p.end = a.start, a.end
        nl = 1
        if k["extruded"] and k["varlay"]:
            lay = _view(C.cast(a.layers, C.c_void_p).value, 2 * a.layers_count, np.int32).reshape(-1, 2)
            p.col_layers = lay.ctypes.data
            p.layer_lo, p.layer_hi, p.ncl = 0, jh.tallest(lay, k["region"]), 1
            nl = p.layer_hi
        elif k["extruded"]:
            cs, ce = a.layers[0], a.layers[1] - 1
            p.bottom = cs
            p.ncl = max(ce - cs, 1)
            region = ("ALL", "ON_BOTTOM", "ON_TOP", "ON_INTERIOR_FACETS")[k["region"]]
            lo, hi = jh.extents(cs, ce, region, bool(k["periodic"]))
            p.layer_lo, p.layer_hi = lo, hi
            nl = max(hi - lo, 0)
        p.subset = _addr(a.subset) or None
        nmat = 0
        for i, (kind, access, dtype, dim) in enumerate(k["args"]):
            if kind == _lib.ARG_MAT:
                m = self.mats[a.args[i]]
                v = p.mat[nmat]
                nmat += 1
                v.rowptr, v.colidx, v.vals = m.rowptr.ctypes.data, m.colidx.ctypes.data, m.vals.ctypes.data
                v.row_lg = m.row_lg.ctypes.data if m.row_lg is not None else None
                v.col_lg = m.col_lg.ctypes.data if m.col_lg is not None else None
                v.bs_r = v.bs_c = m.bs
            else:
                p.arg[i] = a.args[i]                         # Dat: "device" buffer; Global: host buffer
        for i in range(a.nmaps):
            p.map[i] = a.maps[i]
        total = (a.end - a.start) * nl
        k["fn"](C.byref(p), ((total + 127) // 128) * 128 if total else 128)
        return 0

    def _call_helmholtz(self, k, a):
        el = interval_element(k["degree"])
        orc = self.oracle
        nlayers_nodes = a.layers[1]
        nlay = nlayers_nodes - 1
        arity = (k["degree"] + 1) ** 3
        ncols = a.end
        map0 = _view(a.maps[0], ncols * arity, np.int32).reshape(ncols, arity)
        map1 = _view(a.maps[1], ncols * 8, np.int32).reshape(ncols, 8)
        nvert = int(map1.max() + k["off1"].max() * nlay) + 1
        coords = _view(a.args[1], nvert * 3).reshape(nvert, 3)
        nnode = int(map0.max() + k["off0"].max() * nlay) + 1
        if _addr(a.subset):
            cols = _view(a.subset, a.end, np.int32)[a.start:a.end]
            ranges = [(int(c), int(c) + 1) for c in cols]
        else:
            ranges = [(a.start, a.end)]
        if k["rank"] == 2:
            m = self.mats[a.args[0]]
            # node-level lgmap of the dof-level one (k_node_lgmap in csrc/mat.cu)
            lg = lambda v: None if v is None else np.where(
                (v.reshape(-1, m.bs) < 0).all(axis=1), -1, np.arange(m.nrows)).astype(np.int32)
            vals = np.zeros(len(m.colidx))
            for s, e in ranges:
                orc.matrix_extruded(el, s, e, [0, nlayers_nodes], m.rowptr, m.colidx, vals, coords, map0,
                                    k["off0"], map1, k["off1"], lg(m.row_lg), lg(m.col_lg), k["alpha"], k["beta"])
            blocks = m.vals.reshape(-1, m.bs, m.bs)
            for c in range(m.bs):
                blocks[:, c, c] += vals
            return 0
        cdim = k["cdim"]
        y = _view(a.args[0], nnode * cdim)
        if k["diagonal"]:
            for s, e in ranges:
                for c in range(s, e):
                    for l in range(nlay):
                        xv = coords[map1[c] + k["off1"] * l].ravel()
                        Ae = orc.cell_matrix(el, xv, k["alpha"], k["beta"])
                        np.add.at(y, map0[c] + k["off0"] * l, np.diag(Ae))
            return 0
        x = _view(a.args[2], nnode * cdim).copy()
        for s, e in ranges:
            orc.action_extruded(el, s, e, [0, nlayers_nodes], y, coords, x, map0, k["off0"], map1, k["off1"],
                                cdim, k["alpha"], k["beta"])
        return 0


class install:
    """Context manager: route firedrake_b200._lib to a MockEngine."""

    def __init__(self, oracle):
        self.engine = MockEngine(oracle)

    def __enter__(self):
        from firedrake_b200 import codegen
        self.engine.real = _lib.load()                       # the real library (no GPU needed to load it)
        self._saved = (_lib._lib, _lib._initialised, _lib.lib, _lib.init, _lib.check, dict(codegen._handles))
        eng = self.engine
        codegen._handles.clear()
        _lib._lib, _lib._initialised = eng, 0
        _lib.lib = lambda: eng
        _lib.init = lambda device=None: eng

        def check(rc, what=""):
            if rc != 0:
                msg = eng.fdb_last_error().decode(errors="replace")
                raise _lib.EngineError(f"{what}: {msg}" if what else msg)
        _lib.check = check
        return eng

    def __exit__(self, *exc):
        from firedrake_b200 import codegen
        import gc
        gc.collect()                                        # run __del__ of mock-backed objects now
        codegen._handles.clear()
        _lib._lib, _lib._initialised, _lib.lib, _lib.init, _lib.check, saved = self._saved
        codegen._handles.update(saved)
        return False
