"""TEST INFRASTRUCTURE: run the generic wrapper builder's GENERATED code on the
host.  The generated source (``WrapperSpec.source()``) is cut at the prelude
marker, ``tests/jit_host_prelude.h`` is prepended and the body -- the local
kernel plus the generated wrapper, byte for byte what NVRTC compiles -- is built
with g++ and called through ctypes with the same parameter block the CUDA
launcher fills (``FdbWrapParams`` in csrc/wrapper_jit.cu).  This checks packing,
unpacking, index arithmetic, iteration regions and reductions of the generated
code against the reference's semantics without a GPU; it is not a product path.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
MARKER = "/* ==== fdb200 prelude end ==== */"
_cache = {}


class MatView(C.Structure):
    _fields_ = [("rowptr", C.c_void_p), ("colidx", C.c_void_p), ("vals", C.c_void_p),
                ("row_lg", C.c_void_p), ("col_lg", C.c_void_p), ("bs_r", C.c_int), ("bs_c", C.c_int)]


class WrapParams(C.Structure):
    _fields_ = [("start", C.c_int), ("end", C.c_int), ("layer_lo", C.c_int), ("layer_hi", C.c_int),
                ("bottom", C.c_int), ("ncl", C.c_int), ("subset", C.c_void_p), ("col_layers", C.c_void_p),
                ("arg", C.c_void_p * 16), ("map", C.c_void_p * 8), ("mat", MatView * 4)]


def build(source: str, name: str):
    """Compile the body of ``source`` for the host; returns the ctypes function."""
    assert MARKER in source
    body = source.split(MARKER, 1)[1]
    text = '#include "jit_host_prelude.h"\n' + body
    key = hashlib.sha1(text.encode()).hexdigest()
    if key in _cache:
        return _cache[key]
    d = tempfile.mkdtemp(prefix="fdb_jit_host_")
    src = os.path.join(d, "wrap.cpp")
    so = os.path.join(d, "wrap.so")
    with open(src, "w") as fh:
        fh.write(text)
    r = subprocess.run(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-I", HERE, src, "-o", so],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    lib = C.CDLL(so)
    fn = getattr(lib, "wrap_" + name)
    fn.argtypes = [C.POINTER(WrapParams), C.c_longlong]
    fn.restype = None
    _cache[key] = (fn, lib)
    return fn, lib


class HostCSR:
    """Minimal host CSR with the layout of fdb_mat (node pattern, bs x bs blocks)."""

    def __init__(self, nrows, pairs, bs=1):
        rows = sorted(set((int(r), int(c)) for r, c in pairs) | {(i, i) for i in range(nrows)})
        self.nrows, self.bs = nrows, bs
        self.rowptr = np.zeros(nrows + 1, dtype=np.int64)
        for r, _ in rows:
            self.rowptr[r + 1] += 1
        self.rowptr = np.cumsum(self.rowptr).astype(np.int64)
        self.colidx = np.array([c for _, c in rows], dtype=np.int32)
        self.vals = np.zeros(len(rows) * bs * bs)
        self.row_lg = self.col_lg = None

    def dense(self):
        bs = self.bs
        A = np.zeros((self.nrows * bs, self.nrows * bs))
        blocks = self.vals.reshape(-1, bs, bs)
        for r in range(self.nrows):
            for k in range(self.rowptr[r], self.rowptr[r + 1]):
                c = self.colidx[k]
                A[r * bs:(r + 1) * bs, c * bs:(c + 1) * bs] = blocks[k]
        return A


def tallest(layers, region):
    """Layer extent of the launch grid for variable layers (fdb_jit_call)."""
    cells = layers[:, 1] - 1 - layers[:, 0]
    if region in ("ON_BOTTOM", "ON_TOP", 1, 2):
        return int((cells > 0).any())
    if region in ("ON_INTERIOR_FACETS", 3):
        return int(max(cells.max() - 1, 0))
    return int(max(cells.max(), 0))


def extents(cs, ce, region, periodic=False):
    """Layer extent of the launch grid for constant layers, cells ``[cs, ce)`` (fdb_jit_call):
    a periodic column has ``ce - cs`` interior horizontal facets, the last one wrapping round."""
    return {"ALL": (cs, ce), "ON_BOTTOM": (cs, cs + 1), "ON_TOP": (ce - 1, ce),
            "ON_INTERIOR_FACETS": (cs, ce if periodic else ce - 1)}[region]


def run(spec, start, end, args, maps, layers=None, subset=None, region="ALL", periodic=False):
    """Execute the generated wrapper on host arrays.  ``args``: one entry per
    kernel argument -- numpy array (Dat / Global) or HostCSR (Mat); ``maps``: the
    int32 map arrays in slot order; ``periodic``: the set is periodically extruded."""
    fn, _ = build(spec.source(), spec.kernel.name)
    p = WrapParams()
    p.start, p.end = start, end
    nl = 1
    if layers is not None and np.ndim(layers) == 2:
        lay = np.ascontiguousarray(layers, dtype=np.int32)
        keep_lay = lay
        p.col_layers = lay.ctypes.data
        p.layer_lo, p.layer_hi, p.ncl = 0, tallest(lay, region), 1
        nl = p.layer_hi
    elif layers is not None:
        cs, ce = int(layers[0]), int(layers[1]) - 1
        p.bottom = cs
        p.ncl = max(ce - cs, 1)
        lo, hi = extents(cs, ce, region, periodic)
        p.layer_lo, p.layer_hi = lo, hi
        nl = max(hi - lo, 0)
    keep = []
    if subset is not None:
        s = np.ascontiguousarray(subset, dtype=np.int32)
        keep.append(s)
        p.subset = s.ctypes.data
    nmat = 0
    for i, a in enumerate(args):
        if isinstance(a, HostCSR):
            v = p.mat[nmat]
            nmat += 1
            v.rowptr, v.colidx, v.vals = a.rowptr.ctypes.data, a.colidx.ctypes.data, a.vals.ctypes.data
            v.row_lg = a.row_lg.ctypes.data if a.row_lg is not None else None
            v.col_lg = a.col_lg.ctypes.data if a.col_lg is not None else None
            v.bs_r = v.bs_c = a.bs
        else:
            assert a.flags["C_CONTIGUOUS"]
            p.arg[i] = a.ctypes.data
    for i, m in enumerate(maps):
        assert m.dtype == np.int32 and m.flags["C_CONTIGUOUS"]
        p.map[i] = m.ctypes.data
    total = (end - start) * nl
    nthreads = ((total + 127) // 128) * 128 if total else 128
    fn(C.byref(p), nthreads)
