"""TEST INFRASTRUCTURE: a sequential restatement of one PyOP2 parloop.

This is the loop nest PyOP2's generated C runs (pyop2/codegen/builder.py), written
as plain NumPy, one iteration at a time:

* the layer extents of every iteration region (builder.py:790-812), guarded by
  ``0 <= start <= end`` as the RuntimeIndex there is;
* the extruded map indexing ``values[n, perm[j]] + offset[perm[j]] * (layer - bottom + f)``
  with its periodic remainder forms (builder.py:80-124, PMap 144-177);
* the interior-horizontal ``F = 2`` packs (builder.py:359-364, 840-844);
* the gather / scatter of each access mode for Dats (DatPack, builder.py:322-429)
  and Globals (GlobalPack, builder.py:241-319): INC and WRITE packs start from zero,
  READ / RW / MIN / MAX packs read the current value, and the unpack adds, takes the
  minimum / maximum, or stores.  A direct Dat is handed to the kernel in place.

It shares no code with the wrapper generator or with the harnesses that run the
generated code; its inputs are plain arrays: map values, offsets, offset
quotients, permutations, layers, subset indices and Dat / Global contents.
"""
from dataclasses import dataclass

import numpy as np

REGIONS = ("ALL", "ON_BOTTOM", "ON_TOP", "ON_INTERIOR_FACETS")
ACCESSES = ("READ", "WRITE", "RW", "INC", "MIN", "MAX")


@dataclass
class Map:
    values: np.ndarray                    # (iteration set size, arity)
    offset: np.ndarray = None             # (arity,), extruded maps only
    offset_quotient: np.ndarray = None    # (arity,), periodic extrusion only
    permutation: np.ndarray = None        # PermutedMap


@dataclass
class Arg:
    data: np.ndarray                      # Dat: (set size, cdim...); Global: (dim,)
    access: str
    map: Map = None
    is_global: bool = False


def layer_extents(cell_start, cell_end, region, periodic):
    """``[start, end)`` of the layer loop for one column whose cells are
    ``[cell_start, cell_end)`` (builder.py:790-812)."""
    if region == "ON_BOTTOM":
        return cell_start, cell_start + 1
    if region == "ON_TOP":
        return cell_end - 1, cell_end
    if region == "ON_INTERIOR_FACETS":
        # periodic columns have a facet between their top and bottom cells as well
        return cell_start, cell_end if periodic else cell_end - 1
    if region == "ALL":
        return cell_start, cell_end
    raise ValueError(region)


def _c_rem(a, b):
    """C's ``%`` (truncating), which is what the generated code evaluates."""
    return np.fmod(a, b)


def map_entries(m, n, layer, bottom, num_layers, F, periodic):
    """The ``F * arity`` entries a map yields for entry ``n`` at ``layer``, F-major."""
    arity = m.values.shape[1]
    perm = np.arange(arity) if m.permutation is None else np.asarray(m.permutation)
    base = m.values[n, perm].astype(np.int64)
    if layer is None or m.offset is None:
        assert F == 1
        return base
    off = np.asarray(m.offset, dtype=np.int64)[perm]
    out = []
    for k in range(F):
        o = np.full(arity, layer - bottom + k, dtype=np.int64)
        if periodic:
            if m.offset_quotient is None:
                o = _c_rem(o, num_layers)
            else:
                q = np.asarray(m.offset_quotient, dtype=np.int64)[perm]
                o = _c_rem(o + q, num_layers) - _c_rem(q, num_layers)
        out.append(base + off * o)
    return np.concatenate(out)


def par_loop(kernel, start, end, args, *, layers=None, region="ALL", periodic=False, subset=None,
             pass_layer=False, interior_horizontal=None):
    """Run ``kernel`` over iteration entries ``[start, end)`` (positions in ``subset``
    when given), updating the arrays of ``args`` in place.

    ``layers``: None (not extruded), a ``[bottom, top)`` node-layer pair (constant
    layers), or an ``(nentries, 2)`` array of such pairs (variable layers).
    ``kernel`` is called with one 1-D array per argument (a copy for packed
    arguments, a view for direct Dats and READ Globals) and, with ``pass_layer``,
    the layer number."""
    if region != "ALL" and layers is None:
        raise ValueError("iteration regions need an extruded set")
    if interior_horizontal is None:
        interior_horizontal = region == "ON_INTERIOR_FACETS"
    F = 2 if interior_horizontal else 1
    lay = None if layers is None else np.asarray(layers)
    for it in range(start, end):
        n = int(subset[it]) if subset is not None else it
        if lay is None:
            _iteration(kernel, args, n, None, 0, 1, 1, False, False)
            continue
        row = lay[n] if lay.ndim == 2 else lay
        cell_start, cell_end = int(row[0]), int(row[1]) - 1
        lo, hi = layer_extents(cell_start, cell_end, region, periodic)
        if not (0 <= lo <= hi):
            continue
        for layer in range(lo, hi):
            _iteration(kernel, args, n, layer, cell_start, cell_end - cell_start, F, periodic, pass_layer)


def _iteration(kernel, args, n, layer, bottom, num_layers, F, periodic, pass_layer):
    kargs, unpacks = [], []
    for a in args:
        if a.is_global:
            if a.access == "READ":
                kargs.append(a.data)
                continue
            t = np.zeros_like(a.data) if a.access == "INC" else a.data.copy()
            kargs.append(t)
            unpacks.append((a, None, t))
        elif a.map is None:
            kargs.append(a.data.reshape(a.data.shape[0], -1)[n])
        else:
            idx = map_entries(a.map, n, layer, bottom, num_layers, F, periodic)
            flat = a.data.reshape(a.data.shape[0], -1)
            if a.access in ("READ", "RW", "MIN", "MAX"):
                t = flat[idx].ravel().copy()
            else:
                t = np.zeros(idx.size * flat.shape[1], dtype=flat.dtype)
            kargs.append(t)
            if a.access != "READ":
                unpacks.append((a, idx, t))
    if pass_layer:
        kargs.append(layer)
    kernel(*kargs)
    for a, idx, t in unpacks:
        if idx is None:
            dst, src = a.data.reshape(-1), t.reshape(-1)
        else:
            flat = a.data.reshape(a.data.shape[0], -1)
            src = t.reshape(idx.size, flat.shape[1])
            dst = None
        if a.access == "INC":
            if dst is not None:
                dst += src
            else:
                np.add.at(flat, idx, src)
        elif a.access == "MIN":
            if dst is not None:
                np.minimum(dst, src, out=dst)
            else:
                np.minimum.at(flat, idx, src)
        elif a.access == "MAX":
            if dst is not None:
                np.maximum(dst, src, out=dst)
            else:
                np.maximum.at(flat, idx, src)
        else:                                     # WRITE, RW: store, in slot order
            if dst is not None:
                dst[...] = src
            else:
                for k in range(idx.size):
                    flat[idx[k]] = src[k]
