"""The generic wrapper builder (csrc/wrapper_jit.cu) against an independent
restatement of PyOP2's loop semantics (tests/_pyop2_loop.py), swept over the
cross-product of the wrapper's features: extrusion kind x iteration region,
cell layers, iteration range, access modes, Global reductions, dtypes, cdim,
permuted and multiple maps, the layer argument, thread counts round warp and
block multiples, and the location of the data.

Every input is a small integer and every kernel output depends on the entry,
slot and layer, so the results are exact whatever order the atomics run in and
the comparison is ``==``: one misplaced or missing contribution fails.

One parametrisation, three legs: ``host_harness`` runs the generated wrapper body
on the CPU (tests/_jit_host.py), ``device`` and ``host_location`` run
``codegen.par_loop`` on the GPU with device-resident Dats and with NumPy buffers
(mirror cache and write-back).
"""
from dataclasses import dataclass

import numpy as np
import pytest

from firedrake_b200 import _lib, codegen, op2
from firedrake_b200.codegen import CStringKernel, PermutedMap, WrapperSpec

import _jit_host as jh
import _pyop2_loop as ref

# ------------------------------------------------------------------------- the axes
EXTRUSIONS = ("none", "layers0", "layers2", "periodic", "periodic_oq01", "periodic_oqmix", "variable")
CELL_LAYERS = (1, 2, 3, 33)
ITERATIONS = ("full", "split", "subset", "empty")
# y's access; "direct_*": y is a Dat on the iteration set (the private-copy path when extruded)
Y_ACCESSES = ("INC", "WRITE", "RW", "MIN", "MAX", "direct_INC", "direct_WRITE")
# (access, dim, where the extreme value is): "last" = only in the last iterated entry,
# "initial" = every value is on the wrong side of the Global's initial value
GLOBALS = (None, ("INC", 1, "initial"), ("INC", 3, "initial"), ("MIN", 1, "last"), ("MIN", 3, "initial"),
           ("MAX", 1, "initial"), ("MAX", 3, "last"))
DTYPES = (np.float64, np.float32, np.int32, np.uint32, np.int64)
CDIMS = (1, 3)
X_MAPS = ("same", "permuted", "other")
THREADS = (31, 32, 33, 127, 128, 129, 255, 256, 257)

CTYPE = {np.float64: "double", np.float32: "float", np.int32: "int", np.uint32: "unsigned int",
         np.int64: "long long"}


@dataclass(frozen=True)
class Case:
    extrusion: str
    region: str
    cells: int
    iteration: str
    y_access: str
    glob: tuple
    dtype: type
    cdim: int
    x_map: str
    pass_layer: bool
    threads: int
    seed: int

    @property
    def id(self):
        g = "-" if self.glob is None else "".join(str(v) for v in self.glob)
        return (f"{self.extrusion}-{self.region}-L{self.cells}-{self.iteration}-{self.y_access}-g{g}-"
                f"{np.dtype(self.dtype).name}-c{self.cdim}-{self.x_map}-{'lay' if self.pass_layer else 'nolay'}"
                f"-t{self.threads}")

    @property
    def extruded(self):
        return self.extrusion != "none"

    @property
    def periodic(self):
        return self.extrusion.startswith("periodic")


def _cases():
    """Every extrusion x region pair three times; the other axes drawn with a fixed seed
    (test_case_matrix_covers_every_axis_value checks that every value appears), then
    moved to the nearest combination whose result is defined."""
    pairs = [("none", "ALL")] + [(e, r) for e in EXTRUSIONS[1:] for r in ref.REGIONS]
    rng = np.random.default_rng(2024)
    out = []
    for p, (ext, region) in enumerate(pairs):
        for r in range(3):
            pick = lambda vals: vals[rng.integers(len(vals))]     # noqa: E731
            cells, acc, glob, iteration = pick(CELL_LAYERS), pick(Y_ACCESSES), pick(GLOBALS), pick(ITERATIONS)
            if r == 0:
                # the first case of every pair iterates columns of several cells through a map
                cells, acc, iteration = pick((3, 33)), pick(Y_ACCESSES[:5]), pick(("full", "split"))
            if ext == "none":
                cells = 1
            elif ext.startswith("periodic"):
                cells = max(cells, 2)              # a periodic column has at least two cells
            if region == "ON_INTERIOR_FACETS" and acc in ("WRITE", "RW"):
                # the F = 2 packs of neighbouring facets share a cell: a store is not defined
                acc = {"WRITE": "INC", "RW": "MAX"}[acc]
            out.append(Case(ext, region, int(cells), iteration, acc, glob, pick(DTYPES), int(pick(CDIMS)),
                            pick(X_MAPS), bool(ext != "none" and rng.integers(2)), int(pick(THREADS)), 100 * p + r))
    # atomic contention: >= 10^5 threads onto few addresses and one Global
    out += [Case("layers0", "ALL", 33, "split", "INC", ("INC", 3, "initial"), np.int64, 1, "other", True, 102300, 1),
            Case("none", "ALL", 1, "full", "MIN", ("MAX", 1, "last"), np.float64, 3, "permuted", False, 100003, 2),
            Case("none", "ALL", 1, "subset", "INC", ("INC", 1, "initial"), np.float32, 1, "same", False, 150001, 3),
            Case("periodic_oq01", "ON_INTERIOR_FACETS", 33, "full", "MAX", ("MIN", 3, "last"), np.uint32, 1,
                 "same", True, 100000, 4)]
    return out


CASES = _cases()


# --------------------------------------------------------------- the local kernels
# Each C statement with its Python twin next to it.  y is the Dat under test, x a
# READ Dat through a map, w a READ direct Dat feeding the Global g.
def _inc(a, i, v):
    a[i] += v


def _store(a, i, v):
    a[i] = v


def _rw(a, i, v):
    a[i] = 2 * a[i] + v


def _min(a, i, v):
    if v < a[i]:
        a[i] = v


def _max(a, i, v):
    if v > a[i]:
        a[i] = v


UPDATE = {"INC": ("{a}[{i}] += {v};", _inc),
          "WRITE": ("{a}[{i}] = {v};", _store),
          "RW": ("{a}[{i}] = 2 * {a}[{i}] + {v};", _rw),
          "MIN": ("if ({v} < {a}[{i}]) {a}[{i}] = {v};", _min),
          "MAX": ("if ({v} > {a}[{i}]) {a}[{i}] = {v};", _max)}


def make_kernel(c, ny, nx, gdim):
    """(CStringKernel, Python twin) for case ``c`` with local sizes ``ny``, ``nx`` and a
    Global of ``gdim`` entries (0: none)."""
    T = CTYPE[c.dtype]
    acc = c.y_access.replace("direct_", "")
    lay = " + 7 * layer" if c.pass_layer else ""
    if c.y_access == "direct_WRITE":
        # every layer of a column stores into the same entry: the value may not depend on the layer
        yexpr, ytwin = "3 * i + 11", (lambda x, i, layer: 3 * i + 11)
    else:
        yexpr = f"(i + 1) * x[{nx} - 1 - i % {nx}] + i{lay}"
        ytwin = (lambda x, i, layer: (i + 1) * int(x[nx - 1 - i % nx]) + i + 7 * layer)
    params = [f"{T} *y", f"const {T} *x"]
    body = [f"    for (int i = 0; i < {ny}; ++i) {{ const {T} v = ({T})({yexpr}); "
            + UPDATE[acc][0].format(a="y", i="i", v="v") + " }"]
    if gdim:
        gacc = c.glob[0]
        glay = " + layer" if c.pass_layer and gacc == "INC" else ""
        params += [f"const {T} *w", f"{T} *g"]
        body.append(f"    for (int d = 0; d < {gdim}; ++d) {{ const {T} u = ({T})(w[d] + d{glay}); "
                    + UPDATE[gacc][0].format(a="g", i="d", v="u") + " }")
    if c.pass_layer:
        params.append("int layer")
    code = "static void k(" + ", ".join(params) + ")\n{\n" + "\n".join(body) + "\n}\n"

    def twin(y, x, *rest):
        layer = rest[-1] if c.pass_layer else 0
        for i in range(ny):
            UPDATE[acc][1](y, i, ytwin(x, i, layer))
        if gdim:
            w, g = rest[0], rest[1]
            glay = layer if c.glob[0] == "INC" else 0
            for d in range(gdim):
                UPDATE[c.glob[0]][1](g, d, int(w[d]) + d + glay)

    return CStringKernel(code, "k"), twin


# ------------------------------------------------------------------- the problems
def _region_layers(c):
    if not c.extruded:
        return 1
    return {"ALL": c.cells, "ON_BOTTOM": 1, "ON_TOP": 1,
            "ON_INTERIOR_FACETS": c.cells if c.periodic else c.cells - 1}[c.region]


def _maps(c, nent, rng, layers):
    """Two maps per extrusion kind, as (values, offset, offset_quotient, toset size):
    "cg" shares targets between entries and layers, "dg" is injective over the region."""
    ncl = c.cells
    n = np.arange(nent)
    if not c.extruded:
        nn = max(4, nent // 2)
        cg = (rng.integers(0, nn, (nent, 3)), None, None, nn)
        dg = (rng.permutation(2 * nent).reshape(nent, 2), None, None, 2 * nent)
        return cg, dg
    if c.extrusion == "variable":
        h = layers[:, 1] - layers[:, 0] - 1                      # cells per column
        colstart = np.concatenate([[0], np.cumsum(h + 1)[:-1]])
        cellstart = np.concatenate([[0], np.cumsum(h)[:-1]])
        cg = (np.stack([colstart, colstart + 1], 1), [1, 1], None, int((h + 1).sum()))
        dg = (cellstart[:, None], [1], None, int(h.sum()))
        return cg, dg
    # node columns of height H, entry n between node columns n and n + 1 (Q1 in the vertical)
    H = ncl if c.periodic else ncl + 1
    oq = {"periodic_oq01": [0, 1, 0, 1], "periodic_oqmix": [2, 0, 1, 3]}.get(c.extrusion)
    q = np.zeros(4, dtype=int) if oq is None else np.asarray(oq) % ncl
    if oq is None:
        q[[1, 3]] = 1
    cg = (np.stack([n * H + q[0], n * H + q[1], (n + 1) * H + q[2], (n + 1) * H + q[3]], 1), [1, 1, 1, 1], oq,
          (nent + 1) * H + 1)
    # two cell dofs per cell, DG: injective over all layers (and over a periodic column)
    dq = None if oq is None else [0, 1]
    second = 1 if dq is None else 1 + 2 * (1 % ncl)
    dg = (np.stack([2 * ncl * n, 2 * ncl * n + second], 1), [2, 2], dq, 2 * ncl * nent + 2)
    return cg, dg


class Problem:
    """One case's iteration set, maps, Dats and Global, as op2 objects and plain arrays."""

    def __init__(self, c):
        self.c = c
        rng = np.random.default_rng(c.seed)
        dt = c.dtype
        nl = _region_layers(c)
        nent = max(1, round(c.threads / max(nl, 1)))
        self.layers = None
        if c.extrusion == "variable":
            h = rng.integers(1, c.cells + 1, nent)
            h[-1] = c.cells                                    # the tallest column is iterated last
            b = rng.integers(0, 4, nent)
            self.layers = np.stack([b, b + h + 1], 1).astype(np.int32)
        elif c.extruded:
            b = 2 if c.extrusion == "layers2" else 0
            self.layers = np.array([b, b + c.cells + 1], dtype=np.int32)
        # iteration set and the [start, end) parts the parloop runs
        sizes = {"full": nent, "split": (nent // 3, nent, nent), "subset": nent, "empty": (0, 0, nent)}[c.iteration]
        base = op2.Set(sizes)
        if c.extruded:
            base = op2.ExtrudedSet(base, self.layers if c.extrusion == "variable" else c.cells + 1,
                                   extruded_periodic=c.periodic)
            if c.extrusion == "layers2":
                base.layers_array = self.layers.reshape(1, 2).copy()
        self.base = base
        self.subset = None
        self.iterset = base
        if c.iteration == "subset":
            idx = np.sort(rng.choice(nent, size=max(1, (2 * nent) // 3), replace=False))
            idx[-1] = nent - 1
            self.iterset = op2.Subset(base, idx)
            self.subset = self.iterset.indices
        self.parts = [p for p in (self.iterset.core_part, self.iterset.owned_part) if p[1] > p[0]]
        if c.iteration == "empty":
            self.parts = [(0, 0)]
        # maps
        cg, dg = _maps(c, nent, rng, self.layers)

        def mk(spec):
            vals, off, oq, ntarget = spec
            # entries past the ones the map reaches stay untouched: a wrong index that overshoots
            # lands there and shows up in the comparison rather than outside the array
            toset = op2.Set(2 * int(ntarget) + 8)
            return op2.Map(base, toset, np.asarray(vals).shape[1], vals, offset=off, offset_quotient=oq)

        acc = c.y_access.replace("direct_", "")
        ykind = "dg" if acc in ("WRITE", "RW") else "cg"
        ymap = None if c.y_access.startswith("direct_") else mk({"cg": cg, "dg": dg}[ykind])
        xbase = ymap if ymap is not None else mk(cg)
        if c.x_map == "same":
            xmap = xbase
        elif c.x_map == "permuted":
            xmap = PermutedMap(xbase, rng.permutation(xbase.arity))
        else:                                      # a second map: the other kind
            xmap = mk(cg if ymap is not None and ykind == "dg" else dg)
        self.maps = {"y": ymap, "x": xmap}
        # data
        cd = c.cdim
        ydim = op2.DataSet(base if ymap is None else ymap.toset, cd)
        lo, hi = {"INC": (0, 50), "WRITE": (1000, 2000), "RW": (1000, 2000), "MIN": (1, 2000),
                  "MAX": (1, 2000)}[acc]
        self.y = op2.Dat(ydim, rng.integers(lo, hi, (ydim.set.total_size, cd)), dtype=dt)
        self.x = op2.Dat(op2.DataSet(xmap.toset, cd), rng.integers(1, 21, (xmap.toset.total_size, cd)), dtype=dt)
        self.w = self.g = None
        if c.glob is not None:
            gacc, gdim, side = c.glob
            # float32 sums of 10^5 terms stay exact below 2**24
            wv = rng.integers(10, 60 if dt == np.float32 else 1000, (nent, gdim))
            if side == "last":
                # the last iterated entry (its column's threads end the grid) holds the extreme
                wv[nent - 1] = {"MIN": 5, "MAX": 5000}[gacc]
            self.w = op2.Dat(op2.DataSet(base, gdim), wv, dtype=dt)
            init = {("INC", "initial"): 17, ("MIN", "last"): 100000, ("MIN", "initial"): 1,
                    ("MAX", "last"): 1, ("MAX", "initial"): 100000}[(gacc, side)]
            self.g = op2.Global(gdim, init + np.arange(gdim), dtype=dt)
        F = 2 if c.region == "ON_INTERIOR_FACETS" else 1
        ny = cd if ymap is None else F * ymap.arity * cd
        self.kernel, self.twin = make_kernel(c, ny, F * xmap.arity * cd, 0 if self.g is None else c.glob[1])

    def args(self):
        acc = getattr(op2, self.c.y_access.replace("direct_", ""))
        a = [self.y(acc, self.maps["y"]), self.x(op2.READ, self.maps["x"])]
        if self.g is not None:
            a += [self.w(op2.READ), self.g(getattr(op2, self.c.glob[0]))]
        return a

    def arrays(self):
        return [self.y, self.x] + ([] if self.g is None else [self.w, self.g])

    def reference(self):
        """The expected contents of every argument after the parloop."""
        def rmap(m):
            if m is None:
                return None
            b = m.map_ if isinstance(m, PermutedMap) else m
            return ref.Map(b.values_with_halo, b.offset, b.offset_quotient,
                           m.permutation if isinstance(m, PermutedMap) else None)
        data = [np.array(d._data, copy=True) for d in self.arrays()]
        acc = [self.c.y_access.replace("direct_", ""), "READ"] + ([] if self.g is None else ["READ", self.c.glob[0]])
        maps = [rmap(self.maps["y"]), rmap(self.maps["x"]), None, None]
        args = [ref.Arg(d, a, m, is_global=(i == 3)) for i, (d, a, m) in enumerate(zip(data, acc, maps))]
        for s, e in self.parts:
            ref.par_loop(self.twin, s, e, args, layers=self.layers, region=self.c.region, periodic=self.c.periodic,
                         subset=self.subset, pass_layer=self.c.pass_layer)
        return data

    def spec(self):
        c = self.c
        return WrapperSpec(self.kernel, self.args(), extruded=c.extruded, subset=self.subset is not None,
                           iteration_region=c.region, pass_layer_arg=c.pass_layer, extruded_periodic=c.periodic,
                           constant_layers=c.extrusion != "variable")

    def run_host_harness(self):
        spec = self.spec()
        arrays = [d._data for d in self.arrays()]
        maps = [m.values_with_halo for m in spec.maps]
        layers = None if self.layers is None else (self.layers if self.layers.ndim == 2 else list(self.layers))
        for s, e in self.parts:
            jh.run(spec, s, e, arrays, maps, layers=layers, subset=self.subset, region=self.c.region,
                   periodic=self.c.periodic)
        return [np.array(a) for a in arrays]

    def run_engine(self, location):
        c = self.c
        codegen.par_loop(self.kernel, self.iterset, *self.args(), iteration_region=c.region,
                         pass_layer_arg=c.pass_layer, location=location)
        return [np.array(d.data_ro_with_halos if isinstance(d, op2.Dat) else d._data) for d in self.arrays()]


def _assert_same(c, got, want):
    names = ["y", "x", "w", "g"]
    for name, g, w in zip(names, got, want):
        g, w = np.asarray(g).reshape(w.shape), w
        if not np.array_equal(g, w):
            bad = np.argwhere(g != w)
            first = [(tuple(int(v) for v in i), g[tuple(i)].item(), w[tuple(i)].item()) for i in bad[:6]]
            pytest.fail(f"{c.id}: {name} differs in {len(bad)} of {w.size} entries; (index, got, expected): {first}")


def _check_exact(c, want):
    """All contributions are positive integers, so a float result is exact when every
    value stays below 2**mantissa bits: then no partial sum was rounded."""
    if np.dtype(c.dtype).kind == "f":
        limit = 2.0 ** np.finfo(c.dtype).nmant
        assert all(np.abs(w).max(initial=0) < limit for w in want), "case would round: shrink its data"


LEGS = ["host_harness",
        pytest.param("device", marks=pytest.mark.gpu),
        pytest.param("host_location", marks=pytest.mark.gpu)]


@pytest.mark.parametrize("leg", LEGS)
@pytest.mark.parametrize("case", CASES, ids=[c.id for c in CASES])
def test_parloop_matches_pyop2_semantics(case, leg, request):
    pb = Problem(case)
    want = pb.reference()
    _check_exact(case, want)
    if leg == "host_harness":
        got = pb.run_host_harness()
    else:
        request.getfixturevalue("engine")
        got = pb.run_engine("device" if leg == "device" else "host")
    _assert_same(case, got, want)


def test_case_matrix_covers_every_axis_value():
    """Every value of every axis, and every extrusion x region pair, is in the sweep."""
    seen = lambda f: {f(c) for c in CASES}                      # noqa: E731
    assert seen(lambda c: c.extrusion) == set(EXTRUSIONS)
    assert seen(lambda c: (c.extrusion, c.region)) == {("none", "ALL")} | {
        (e, r) for e in EXTRUSIONS[1:] for r in ref.REGIONS}
    assert seen(lambda c: c.cells) == set(CELL_LAYERS)
    assert seen(lambda c: c.iteration) == set(ITERATIONS)
    assert seen(lambda c: c.y_access) == set(Y_ACCESSES)
    assert seen(lambda c: c.glob) >= set(GLOBALS)
    assert seen(lambda c: c.dtype) == set(DTYPES)
    assert seen(lambda c: c.cdim) == set(CDIMS)
    assert seen(lambda c: c.x_map) == set(X_MAPS)
    assert seen(lambda c: c.pass_layer) == {False, True}
    assert seen(lambda c: c.threads) >= set(THREADS)
    assert min(c.cells for c in CASES if c.periodic) >= 2
    assert any(c.threads >= 10 ** 5 for c in CASES)
    for gacc in ("MIN", "MAX"):
        assert {(c.glob[2]) for c in CASES if c.glob and c.glob[0] == gacc} == {"last", "initial"}


# ------------------------------------------------------------------ refused combinations
def _refused(kind):
    """(kernel, iterset, args, par_loop keywords, message) of a parloop the engine must refuse:
    one whose result would depend on the order of the threads, or that PyOP2 cannot express."""
    cols = op2.ExtrudedSet(op2.Set(5), 4)
    plain, nodes = op2.Set(5), op2.Set(8)
    m = op2.Map(plain, nodes, 1, np.arange(5))
    d = op2.Dat(op2.DataSet(cols, 1))
    x = op2.Dat(nodes)
    g = op2.Global(1, 0.0)
    k1 = CStringKernel("static void k(double *a) { a[0] += 1.0; }", "k")
    if kind.startswith("direct_"):
        # one entry per column, shared by the threads of all its layers
        return k1, cols, [d(getattr(op2, kind[7:]))], {}, "READ, INC or WRITE"
    if kind == "periodic_variable":
        var = op2.ExtrudedSet(op2.Set(5), np.array([[0, 3]] * 5, dtype=np.int32))
        var.extruded_periodic = True               # op2.ExtrudedSet refuses this itself
        return k1, var, [op2.Dat(op2.DataSet(var, 1))(op2.INC)], {}, "periodic extrusion has constant layers"
    if kind.startswith("global_"):
        return k1, plain, [g(getattr(op2, kind[7:]))], {}, "Globals are READ, INC, MIN or MAX"
    if kind == "region_unextruded":
        return k1, plain, [x(op2.INC, m)], dict(iteration_region="ON_TOP"), "need an extruded set"
    if kind == "layer_unextruded":
        k2 = CStringKernel("static void k(double *a, int layer) { a[0] += layer; }", "k")
        return k2, plain, [x(op2.INC, m)], dict(pass_layer_arg=True), "pass_layer_arg needs an extruded"
    raise ValueError(kind)


REFUSED = ("direct_RW", "direct_MIN", "direct_MAX", "periodic_variable", "global_WRITE", "global_RW",
           "region_unextruded", "layer_unextruded")


@pytest.mark.parametrize("leg", LEGS)
@pytest.mark.parametrize("kind", REFUSED)
def test_refused_combinations_raise(kind, leg, request):
    k, iterset, args, kw, msg = _refused(kind)
    if leg == "host_harness":
        base = iterset.superset if isinstance(iterset, op2.Subset) else iterset
        spec = WrapperSpec(k, args, extruded=base._extruded, iteration_region=kw.get("iteration_region", "ALL"),
                           pass_layer_arg=kw.get("pass_layer_arg", False),
                           extruded_periodic=getattr(base, "extruded_periodic", False),
                           constant_layers=getattr(base, "constant_layers", True))
        with pytest.raises(_lib.EngineError, match=msg):
            spec.source()
        return
    request.getfixturevalue("engine")
    with pytest.raises(_lib.EngineError, match=msg):
        codegen.par_loop(k, iterset, *args, location="device" if leg == "device" else "host", **kw)


def test_periodic_variable_layers_refused_by_the_set():
    with pytest.raises(ValueError, match="periodic extrusion needs constant layers"):
        op2.ExtrudedSet(op2.Set(2), np.array([[0, 3], [0, 4]], dtype=np.int32), extruded_periodic=True)
