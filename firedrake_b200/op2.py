"""A minimal mirror of the PyOP2 object model, backed by ``libfdb200.so``.

Same names, argument meaning and call protocol as the reference for the part
of PyOP2 that sits on the assembly hot path (SURVEY.md section 8a rows A3-A9):

=================  ===========================================================
here               reference
=================  ===========================================================
``Set``            pyop2/types/set.py:18-125  (core | owned | ghost sizes)
``ExtrudedSet``    pyop2/types/set.py:306-394 (constant layers)
``Subset``         pyop2/types/set.py:397-
``DataSet``        pyop2/types/dataset.py
``Map``            pyop2/types/map.py:17-165  (values + per-dof layer offset)
``Dat``            pyop2/types/dat.py:27-712  (NumPy buffer + dat_version)
``Global``         pyop2/types/glob.py
``Kernel``         pyop2/local_kernel.py:33-43 -- here a *form descriptor*
                   instead of C/loopy source: the element kernels are
                   hand-written CUDA, selected by descriptor
``GlobalKernel``   pyop2/global_kernel.py:255-335
``Parloop``        pyop2/parloop.py:167-260
``par_loop``       pyop2/parloop.py:705-762 (legacy ``dat(access, map)`` args)
=================  ===========================================================

Two data-placement modes, chosen per parloop:

* ``"host"`` (drop-in): the arglist carries HOST pointers exactly as
  pyop2/parloop.py:203-212 builds it; the engine mirrors them on the device
  keyed on ``dat_version`` and writes the output back.
* ``"device"``: Dats own a device buffer (``Dat.device_ptr``) that stays
  resident across calls; the host copy is refreshed lazily by ``Dat.data_ro``.
"""
from __future__ import annotations

import ctypes as C
import enum
import itertools
import weakref
from dataclasses import dataclass, field

import numpy as np

from . import _lib
from ._lib import EngineError

IntType = np.int32
ScalarType = np.float64


class Access(enum.IntEnum):
    READ = 1
    WRITE = 2
    RW = 3
    INC = 4
    MIN = 5
    MAX = 6


READ, WRITE, RW, INC, MIN, MAX = (Access.READ, Access.WRITE, Access.RW, Access.INC,
                                  Access.MIN, Access.MAX)

ALL = "ALL"
ON_BOTTOM = "ON_BOTTOM"
ON_TOP = "ON_TOP"
ON_INTERIOR_FACETS = "ON_INTERIOR_FACETS"


class MapValueError(ValueError):
    pass


class DataSetTypeError(TypeError):
    pass


# Generation ids for objects whose host buffers the engine mirrors by ADDRESS (maps, subset
# index arrays): unique per object and never reused, passed as fdb_call_args.map_versions /
# subset_version so that a new object at a recycled address cannot hit the old mirror, and the
# mirror itself is released when the object dies.
_generations = itertools.count(1)


def _drop_host_mirror(ptr):
    try:
        if _lib._initialised is not None:
            _lib._lib.fdb_mirror_drop(ptr)
    except Exception:
        pass


# ---------------------------------------------------------------------- sets
class Set:
    """Iteration/data set with ``[core | owned | ghost]`` partitions."""
    _extruded = False
    owner_computes = False     # True: partitioned with exec-halo entries, INC loops need no reduce

    def __pow__(self, dim):
        """``set ** dim`` is the DataSet of that shape on the set (pyop2/types/set.py Set.__pow__)."""
        return DataSet(self, dim)

    def __init__(self, size, name=None):
        if isinstance(size, (int, np.integer)):
            size = (size, size, size)
        if len(size) == 2:
            size = (size[0], size[0], size[1])
        self.core_size, self.size, self.total_size = (int(s) for s in size)
        if not (0 <= self.core_size <= self.size <= self.total_size):
            raise ValueError("need core <= owned <= total sizes")
        self.name = name or "set"

    @property
    def sizes(self):
        return (self.core_size, self.size, self.total_size)

    # pyop2/types/set.py:119-125
    @property
    def core_part(self):
        return (0, self.core_size)

    @property
    def owned_part(self):
        return (self.core_size, self.size)

    def __call__(self, *indices):
        return Subset(self, np.asarray(indices, dtype=IntType).ravel())


class ExtrudedSet(Set):
    """A set of columns (pyop2/types/set.py:306-394).  ``layers`` is an int -- NODE layers
    per column, cells per column = layers - 1, ``layers_array`` the int[1][2] the wrapper gets
    -- or an ``(total_size, 2)`` array of ``[bottom, top)`` node layers per column (variable
    layers: every column's map row points at ITS bottom cell; generic wrapper path only)."""
    _extruded = True
    constant_layers = True

    def __init__(self, parent: Set, layers, extruded_periodic: bool = False):
        super().__init__(parent.sizes, name=parent.name + "_extruded")
        self.parent = parent
        layers = np.asarray(layers, dtype=IntType)
        if layers.shape:
            if layers.shape != (parent.total_size, 2):
                raise ValueError(f"specifying layers per entity, but provided {layers.shape}, "
                                 f"needed ({parent.total_size}, 2)")
            if extruded_periodic:
                raise ValueError("periodic extrusion needs constant layers")
            if (layers[:, 1] - layers[:, 0] < 1).any():
                raise ValueError("every column needs at least one node layer")
            self.constant_layers = False
            self.layers_array = np.ascontiguousarray(layers)
            self._generation = next(_generations)
            weakref.finalize(self, _drop_host_mirror, self.layers_array.ctypes.data)
        else:
            if layers < 2:
                raise ValueError("an extruded set needs at least 2 node layers")
            self.layers_array = np.array([[0, int(layers)]], dtype=IntType)
        # periodic in the extruded direction (pyop2/types/set.py ExtrudedSet(extruded_periodic=...)):
        # the top layer's top dofs ARE the bottom layer's bottom dofs; maps carry offset_quotient
        self.extruded_periodic = bool(extruded_periodic)

    @property
    def layers(self):
        if not self.constant_layers:
            raise ValueError("no single layer count: use layers_array")
        return int(self.layers_array[0, 1])


class Subset(Set):
    _extruded = False

    @property
    def layers(self):
        return self.superset.layers

    def __init__(self, superset: Set, indices):
        idx = np.unique(np.asarray(indices, dtype=IntType))
        if isinstance(superset, Subset):
            # a subset of a subset addresses the parent's entries (pyop2/types/set.py:413-416)
            if len(idx) and (idx[0] < 0 or idx[-1] >= superset.total_size):
                raise ValueError("subset indices out of range")
            idx = np.unique(superset.indices[idx])
            superset = superset.superset
        if len(idx) and (idx[0] < 0 or idx[-1] >= superset.total_size):
            raise ValueError("subset indices out of range")
        self.superset = superset
        self.indices = np.ascontiguousarray(idx)
        self._generation = next(_generations)
        weakref.finalize(self, _drop_host_mirror, self.indices.ctypes.data)
        core = int(np.searchsorted(idx, superset.core_size))
        owned = int(np.searchsorted(idx, superset.size))
        Set.__init__(self, (core, owned, len(idx)), name=superset.name + "_subset")
        self._extruded = superset._extruded
        if self._extruded:
            self.constant_layers = superset.constant_layers
            self.layers_array = superset.layers_array


    # set algebra on the index lists (pyop2/types/set.py:486-547); a plain Set stands for "everything"
    @property
    def owned_indices(self):
        return self.indices[self.indices < self.superset.size]

    def _other_indices(self, other):
        if other is self.superset:
            return None
        if not isinstance(other, Subset) or other.superset is not self.superset:
            raise TypeError("set operations need a subset of the same superset (or the superset itself)")
        return other.indices

    def intersection(self, other):
        o = self._other_indices(other)
        return self if o is None else Subset(self.superset, np.intersect1d(self.indices, o))

    def union(self, other):
        o = self._other_indices(other)
        return other if o is None else Subset(self.superset, np.union1d(self.indices, o))

    def difference(self, other):
        o = self._other_indices(other)
        return Subset(self.superset, [] if o is None else np.setdiff1d(self.indices, o))

    def symmetric_difference(self, other):
        o = self._other_indices(other)
        if o is None:
            return Subset(self.superset, np.setdiff1d(np.arange(self.superset.total_size, dtype=IntType), self.indices))
        return Subset(self.superset, np.setxor1d(self.indices, o))


class DataSet:
    """``halo``: a firedrake_b200.halo.Halo describing which rows of the set
    are ghost copies (reference pyop2/types/dataset.py + firedrake/halo.py)."""

    def __init__(self, iter_set: Set, dim=1, name=None, halo=None):
        self.set = iter_set
        self.dim = (dim,) if isinstance(dim, (int, np.integer)) else tuple(dim)
        self.cdim = int(np.prod(self.dim))
        self.name = name or "dset"
        self.halo = halo


def _as_dataset(s):
    return s if isinstance(s, DataSet) else DataSet(s, 1)


# ---------------------------------------------------------------------- maps
class Map:
    """``values`` has shape (iterset.total_size, arity); for extruded iteration
    sets each row addresses the BOTTOM cell of a column and ``offset[i]`` is
    added per layer (pyop2/types/map.py:36-56)."""
    _ids = itertools.count()

    def __init__(self, iterset, toset, arity, values, name=None, offset=None, offset_quotient=None):
        self.iterset, self.toset, self.arity = iterset, toset, int(arity)
        v = np.ascontiguousarray(np.asarray(values, dtype=IntType).reshape(-1, self.arity))
        if v.shape[0] != iterset.total_size:
            raise MapValueError(f"map has {v.shape[0]} rows, iterset has {iterset.total_size}")
        if v.size and (v.min() < 0 or v.max() >= toset.total_size):
            raise MapValueError("map values out of range of the target set")
        self.values_with_halo = v
        self.offset = None if offset is None else np.ascontiguousarray(offset, dtype=IntType)
        if self.offset is not None and self.offset.shape != (self.arity,):
            raise MapValueError("offset must have one entry per arity index")
        # periodic extrusion (pyop2/types/map.py: offset_quotient): 1 for dofs on the top of the cell
        self.offset_quotient = (None if offset_quotient is None
                                else np.ascontiguousarray(offset_quotient, dtype=IntType))
        if self.offset_quotient is not None and self.offset_quotient.shape != (self.arity,):
            raise MapValueError("offset_quotient must have one entry per arity index")
        self.name = name or f"map_{next(Map._ids)}"
        self._dev = None
        self._generation = next(_generations)
        weakref.finalize(self, _drop_host_mirror, self.values_with_halo.ctypes.data)

    @property
    def values(self):
        return self.values_with_halo[:self.iterset.size]

    @property
    def device_ptr(self):
        if self._dev is None:
            self._dev = DeviceArray.from_host(self.values_with_halo)
        return self._dev.ptr


class ComposedMap(Map):
    """``op2.ComposedMap(m0, m1, ..., mk)``: ``local[i] = global[m0[m1[...mk[e]...]][i]]``
    (pyop2/types/map.py:219-279): ``m0`` has the arity of the result, every inner map has arity 1 and
    lands on the iteration set of the map before it.  The reference keeps the factors and emits the
    chained indirection in the wrapper; here the composition is materialised ONCE on the host (one
    int32 gather per factor) and the device sees a plain map -- one dependent load per access instead
    of k + 1.  ``offset`` / ``offset_quotient`` are those of ``m0`` (map.py:257)."""

    def __init__(self, *maps_, name=None):
        if len(maps_) < 1 or not all(isinstance(m, Map) for m in maps_):
            raise TypeError("all factors of a ComposedMap must be Maps")
        for tomap, frommap in zip(maps_[:-1], maps_[1:]):
            if tomap.iterset is not frommap.toset:
                raise MapValueError("tomap.iterset must match frommap.toset")
            if frommap.arity != 1:
                raise MapValueError("inner maps of a ComposedMap have arity 1")
        vals = maps_[0].values_with_halo
        for m in maps_[1:]:
            vals = vals[m.values_with_halo[:, 0]]
        self.maps_ = tuple(maps_)
        super().__init__(maps_[-1].iterset, maps_[0].toset, maps_[0].arity, vals,
                         name=name or "cmap_" + "_".join(m.name for m in maps_),
                         offset=maps_[0].offset, offset_quotient=maps_[0].offset_quotient)


# -------------------------------------------------------------- device memory
class DeviceArray:
    """RAII wrapper around fdb_malloc/fdb_free."""

    def __init__(self, nbytes):
        L = _lib.lib()
        self.nbytes = int(nbytes)
        self.ptr = L.fdb_malloc(self.nbytes)
        if not self.ptr:
            raise EngineError(L.fdb_last_error().decode())

    @classmethod
    def from_host(cls, arr):
        arr = np.ascontiguousarray(arr)
        d = cls(arr.nbytes)
        _lib.check(_lib.lib().fdb_memcpy_h2d(d.ptr, arr.ctypes.data, arr.nbytes), "h2d")
        return d

    def to_host(self, out):
        _lib.check(_lib.lib().fdb_memcpy_d2h(out.ctypes.data, self.ptr, out.nbytes), "d2h")
        return out

    def __del__(self):
        try:
            if self.ptr and _lib._initialised is not None:
                _lib._lib.fdb_free(self.ptr)
        except Exception:
            pass
        self.ptr = None


class PinnedArray:
    """NumPy view of page-locked host memory (fdb_host_alloc)."""

    def __init__(self, shape, dtype):
        L = _lib.lib()
        self.dtype = np.dtype(dtype)
        self.shape = tuple(shape)
        n = int(np.prod(self.shape)) * self.dtype.itemsize
        self.ptr = L.fdb_host_alloc(max(n, 1))
        if not self.ptr:
            raise EngineError(L.fdb_last_error().decode())
        buf = (C.c_char * max(n, 1)).from_address(self.ptr)
        self.array = np.frombuffer(buf, dtype=self.dtype, count=int(np.prod(self.shape))).reshape(self.shape)

    def __del__(self):
        try:
            if self.ptr and _lib._initialised is not None:
                _lib._lib.fdb_host_free(self.ptr)
        except Exception:
            pass
        self.ptr = None


# ------------------------------------------------------------- mixed carriers
class MixedSet:
    """Tuple of Sets (pyop2/types/set.py MixedSet): the node sets of a mixed function space."""

    def __init__(self, sets):
        self._sets = tuple(sets)

    def split(self):
        return self._sets

    def __iter__(self):
        return iter(self._sets)

    def __len__(self):
        return len(self._sets)

    def __getitem__(self, i):
        return self._sets[i]


class MixedDataSet(MixedSet):
    """Tuple of DataSets (pyop2/types/dataset.py MixedDataSet)."""

    def __init__(self, dsets):
        super().__init__(_as_dataset(d) for d in dsets)


class MixedMap:
    """Tuple of Maps from ONE iteration set to the sets of a MixedSet (pyop2/types/map.py MixedMap)."""

    def __init__(self, maps):
        self._maps = tuple(maps)
        its = {id(_m.iterset) for _m in self._maps}
        if len(its) != 1:
            raise MapValueError("all maps of a MixedMap share the iteration set")
        self.iterset = self._maps[0].iterset
        self.arity = sum(m.arity for m in self._maps)

    def split(self):
        return self._maps

    def __iter__(self):
        return iter(self._maps)

    def __len__(self):
        return len(self._maps)

    def __getitem__(self, i):
        return self._maps[i]


@dataclass
class MixedArg:
    """``mixed_dat(access, mixed_map)``: expands to one wrapper argument (= one pointer in the
    arglist, pyop2/parloop.py:203-212) per sub-Dat, packed back to back into ONE local tensor."""
    data: "MixedDat"
    access: Access
    map: MixedMap

    def split(self):
        if len(self.map) != len(self.data):
            raise MapValueError("MixedMap and MixedDat have different numbers of blocks")
        out = [d(self.access, m) for d, m in zip(self.data, self.map)]
        for a in out[1:]:
            a.mixed_continuation = True
        return out


class MixedDat:
    """Tuple of Dats behaving like one vector (pyop2/types/dat.py:861-): ``split`` / indexing /
    iteration give the blocks; whole-vector operations (zero, copy, axpy, inner, norm, +=, -=, *=)
    apply block by block; ``dat(access, MixedMap)`` passes all blocks to a parloop."""

    def __init__(self, dats_or_dset):
        if isinstance(dats_or_dset, MixedDataSet):
            self._dats = tuple(Dat(ds) for ds in dats_or_dset)
        else:
            self._dats = tuple(dats_or_dset)
        if not all(isinstance(d, Dat) for d in self._dats):
            raise DataSetTypeError("MixedDat takes Dats or a MixedDataSet")
        self.dataset = MixedDataSet(d.dataset for d in self._dats)
        self.name = "mixed_" + "_".join(d.name for d in self._dats)

    def split(self):
        return self._dats

    def __iter__(self):
        return iter(self._dats)

    def __len__(self):
        return len(self._dats)

    def __getitem__(self, i):
        return self._dats[i]

    def __call__(self, access, map_=None):
        if not isinstance(map_, MixedMap):
            raise MapValueError("a MixedDat argument needs a MixedMap")
        return MixedArg(self, access, map_)

    @property
    def dat_version(self):
        return sum(d.dat_version for d in self._dats)

    @property
    def data(self):
        return tuple(d.data for d in self._dats)

    @property
    def data_ro(self):
        return tuple(d.data_ro for d in self._dats)

    @property
    def halo_valid(self):
        return all(d.halo_valid for d in self._dats)

    def zero(self, subset=None):
        if subset is not None:
            raise NotImplementedError("zero(subset) on a MixedDat: apply it to the block")
        for d in self._dats:
            d.zero()

    def copy(self, other):
        for a, b in zip(self._dats, other._dats):
            a.copy(b)

    def axpy(self, alpha, other):
        for a, b in zip(self._dats, other._dats):
            a.axpy(alpha, b)

    def inner(self, other):
        return sum(a.inner(b) for a, b in zip(self._dats, other._dats))

    def norm(self):
        return float(np.sqrt(self.inner(self)))

    def __iadd__(self, other):
        self.axpy(1.0, other)
        return self

    def __isub__(self, other):
        self.axpy(-1.0, other)
        return self

    def __imul__(self, scalar):
        for d in self._dats:
            d.__imul__(scalar)
        return self


# ----------------------------------------------------------------------- Dats
class Dat:
    """Node data: C-contiguous ``(total_size, *dim)``, owned rows first, ghosts
    at the tail, vector spaces AoS (pyop2/types/dat.py:72-96).

    ``dat_version`` follows pyop2/types/data_carrier.py:79-97: it is bumped by
    every write access to ``data`` and by every parloop that writes the Dat.
    """
    _ids = itertools.count()
    # zero() of a device-resident Dat rotates between two buffers, the idle one being
    # zeroed on a side stream while the engine stream keeps computing
    zero_rotation = False   # measured: overlapping the zeroing slows the compute kernel by as much (DESIGN.md)

    def __init__(self, dataset, data=None, dtype=ScalarType, name=None, pinned=False):
        self.dataset = _as_dataset(dataset)
        shape = (self.dataset.set.total_size,) + (self.dataset.dim if self.dataset.cdim > 1 else ())
        self._pinned = None
        if pinned:
            self._pinned = PinnedArray(shape, dtype)
            self._data = self._pinned.array
            self._data[...] = 0 if data is None else np.asarray(data, dtype=dtype).reshape(shape)
        elif data is None:
            self._data = np.zeros(shape, dtype=dtype)
        else:
            self._data = np.ascontiguousarray(np.asarray(data, dtype=dtype).reshape(shape))
        self.dtype = np.dtype(dtype)
        self.name = name or f"dat_{next(Dat._ids)}"
        self.dat_version = 0
        self._dev = None            # DeviceArray, device-resident mode
        self._spare = None          # pre-zeroed twin used by zero() (see Dat.zero_rotation)
        self._host_valid = True
        self._dev_valid = False
        self._is_zero = data is None
        self.halo_valid = True
        self.frozen_halo = False     # pyop2/types/dat.py:680-712 (skip l2g inside an assembly)

    # -- shape helpers
    @property
    def cdim(self):
        return self.dataset.cdim

    @property
    def nbytes(self):
        return self._data.nbytes

    # -- host access (pyop2/types/dat.py data / data_ro / data_with_halos)
    def _sync_host(self):
        if not self._host_valid:
            if self._is_zero:
                self._data[...] = 0          # a lazy zero() materialises here
            else:
                self._dev.to_host(self._data)
            self._host_valid = True

    @property
    def data_ro(self):
        self._sync_host()
        v = self._data[:self.dataset.set.size].view()
        v.setflags(write=False)
        return v

    @property
    def data_ro_with_halos(self):
        self._sync_host()
        v = self._data.view()
        v.setflags(write=False)
        return v

    @property
    def data(self):
        self._sync_host()
        self.increment_dat_version()
        self._dev_valid = False
        self._is_zero = False
        self.halo_valid = False      # pyop2/types/dat.py:622-678
        return self._data[:self.dataset.set.size]

    @property
    def data_with_halos(self):
        self._sync_host()
        self.increment_dat_version()
        self._dev_valid = False
        self._is_zero = False
        return self._data

    @property
    def data_wo(self):
        """Write-only host access (pyop2/types/dat.py data_wo): the caller overwrites every owned row, so
        nothing is downloaded first."""
        self._host_valid = True
        self.increment_dat_version()
        self._dev_valid = False
        self._is_zero = False
        self.halo_valid = False
        return self._data[:self.dataset.set.size]

    @property
    def data_wo_with_halos(self):
        self._host_valid = True
        self.increment_dat_version()
        self._dev_valid = False
        self._is_zero = False
        return self._data

    def increment_dat_version(self):
        self.dat_version += 1

    # -- a Dat is also the 1-tuple of itself (pyop2/types/dat.py:118-138: split / iteration / indexing)
    def split(self):
        return (self,)

    def __iter__(self):
        yield self

    def __len__(self):
        return 1

    def __getitem__(self, i):
        if i != 0:
            raise IndexError("a Dat has the block 0 only")
        return self

    def save(self, filename):
        """Owned rows to a NumPy file (pyop2/types/dat.py:286-294)."""
        np.save(filename, self.data_ro)

    def load(self, filename):
        """Owned rows from a NumPy file written by ``save`` (".npy" appended as NumPy does)."""
        import os
        if not os.path.exists(filename) and os.path.exists(str(filename) + ".npy"):
            filename = str(filename) + ".npy"
        v = np.load(filename)
        if v.shape != self._data[:self.dataset.set.size].shape:
            raise ValueError("file holds an array of a different shape")
        self.data_wo[...] = v

    # -- device residency
    @property
    def device_ptr(self):
        """Device buffer holding the current values (uploads if stale)."""
        if self._dev is None:
            self._dev = DeviceArray(self._data.nbytes)
        if not self._dev_valid:
            if self._is_zero:
                _lib.check(_lib.lib().fdb_memset(self._dev.ptr, 0, self._data.nbytes), "memset")
            else:
                _lib.check(_lib.lib().fdb_memcpy_h2d(self._dev.ptr, self._data.ctypes.data,
                                                     self._data.nbytes), "h2d")
            self._dev_valid = True
        return self._dev.ptr

    def _device_written(self, halo_valid=False):
        """The device copy was written.  As in the reference, ANY write invalidates the ghost
        rows (pyop2/types/dat.py:622-678); only ``Halo.global_to_local_end`` (or an operation
        that provably wrote current ghost values) passes ``halo_valid=True``."""
        self._host_valid = False
        self._dev_valid = True
        self._is_zero = False
        self.halo_valid = bool(halo_valid)
        self.increment_dat_version()

    def _reset_ghost_rows(self, access):
        """Before a loop that accumulates into this Dat, set its ghost rows to the identity of
        the reduction (0 for INC, +/-inf for MIN/MAX) -- what the reference's
        ``global_to_local_begin`` does for those access modes (pyop2/types/dat.py:633-636) --
        so that the local->global reduce afterwards sends THIS loop's contributions only."""
        st = self.dataset.set
        nghost = (st.total_size - st.size) * self.cdim
        if nghost <= 0 or (self._is_zero and access is INC):
            return                       # a (lazily) zeroed Dat already holds the INC identity
        ident = {INC: 0.0, MIN: float("inf"), MAX: float("-inf")}[access]
        base = self.device_ptr + st.size * self.cdim * self.dtype.itemsize
        _lib.check(_lib.lib().fdb_vec_fill(nghost, ident, base), "fdb_vec_fill")

    # -- whole-Dat operations (pyop2/types/dat.py:297-311, 354-540)
    def zero(self, subset=None):
        if subset is not None:
            if self._dev_valid and not self._host_valid:
                if not hasattr(subset, "_dev_idx"):
                    subset._dev_idx = DeviceArray.from_host(subset.indices)    # uploaded once
                _lib.check(_lib.lib().fdb_dat_zero_nodes(self._dev.ptr, self.cdim, subset._dev_idx.ptr,
                                                         len(subset.indices)), "zero_nodes")
                self.increment_dat_version()
            else:
                self.data_with_halos[subset.indices] = 0
            return
        # lazy: neither copy is touched until somebody needs it (the assembler
        # zeroes the tensor right before a parloop that overwrites it anyway)
        self._host_valid = False
        self._dev_valid = False
        self._is_zero = True
        self.increment_dat_version()
        if self._dev is not None and Dat.zero_rotation:
            # device-resident tensor: swap in a buffer that was zeroed in the
            # background (overlapping the previous kernel) and send the old one
            # to be zeroed for the next call
            L = _lib.lib()
            if self._spare is None:
                self._spare = DeviceArray(self._data.nbytes)
                _lib.check(L.fdb_zero_background(self._spare.ptr, self._data.nbytes))
            _lib.check(L.fdb_background_barrier())
            self._dev, self._spare = self._spare, self._dev
            _lib.check(L.fdb_zero_background(self._spare.ptr, self._data.nbytes))
            self._dev_valid = True

    def _vec_op(self, other, fn, *scalars):
        L = _lib.lib()
        n = self._data.size
        _lib.check(fn(n, *scalars, other.device_ptr, self.device_ptr))
        # the algebra ran over every local row: the ghost rows stay current only if they were
        # current in BOTH operands (pyop2/types/dat.py:622-678: a write invalidates the halo)
        self._device_written(halo_valid=self.halo_valid and other.halo_valid)

    def axpy(self, alpha, other):
        """self += alpha * other"""
        self._vec_op(other, _lib.lib().fdb_vec_axpy, float(alpha))

    def inner(self, other):
        out = C.c_double()
        _lib.check(_lib.lib().fdb_vec_dot(self._data.size, self.device_ptr, other.device_ptr,
                                          C.byref(out)), "dot")
        return out.value

    def norm(self):
        return float(np.sqrt(self.inner(self)))

    # in-place algebra on the device (pyop2/types/dat.py:312-352 copy, :354-540 _iop / maxpy)
    def copy(self, other, subset=None):
        """``other <- self`` (note the direction: pyop2/types/dat.py:312-330)."""
        if other.nbytes != self.nbytes:
            raise ValueError("copy between Dats of different sizes")
        if subset is not None:
            # only the rows of the subset (pyop2/types/dat.py:312-330, _copy_parloop on a Subset)
            if not hasattr(subset, "_dev_idx"):
                subset._dev_idx = DeviceArray.from_host(subset.indices)      # uploaded once
            dst, src = other.device_ptr, self.device_ptr
            _lib.check(_lib.lib().fdb_dat_set_nodes(dst, src, self.cdim, subset._dev_idx.ptr,
                                                    len(subset.indices)), "fdb_dat_set_nodes")
            other._device_written()
            return
        _lib.check(_lib.lib().fdb_memcpy_d2d(other.device_ptr, self.device_ptr, self.nbytes), "d2d")
        other._device_written(halo_valid=self.halo_valid)

    def __iadd__(self, other):
        if not isinstance(other, Dat):
            return NotImplemented
        self.axpy(1.0, other)
        return self

    def __isub__(self, other):
        if not isinstance(other, Dat):
            return NotImplemented
        self.axpy(-1.0, other)
        return self

    def __imul__(self, other):
        L = _lib.lib()
        if isinstance(other, Dat):
            _lib.check(L.fdb_vec_pointwise_mult(self._data.size, self.device_ptr, other.device_ptr,
                                                self.device_ptr), "pointwise_mult")
            hv = self.halo_valid and other.halo_valid
        else:
            _lib.check(L.fdb_vec_scale(self._data.size, float(other), self.device_ptr), "scale")
            hv = self.halo_valid          # a uniform scaling keeps current ghost rows current
        self._device_written(halo_valid=hv)
        return self

    def __itruediv__(self, other):
        if isinstance(other, Dat):
            raise NotImplementedError("pointwise division of Dats: scale by the reciprocal field")
        return self.__imul__(1.0 / float(other))

    # binary operators build a new Dat on the device (pyop2/types/dat.py:422-505)
    def _copy_of(self):
        r = Dat(self.dataset, dtype=self.dtype)
        self.copy(r)
        return r

    def _shift(self, value):
        """self += value (a scalar), through a filled temporary."""
        t = Dat(self.dataset, dtype=self.dtype)
        _lib.check(_lib.lib().fdb_vec_fill(t._data.size, float(value), t.device_ptr), "fdb_vec_fill")
        t._device_written(halo_valid=True)
        self.axpy(1.0, t)

    def __pos__(self):
        return self._copy_of()

    def __neg__(self):
        r = self._copy_of()
        r *= -1.0
        return r

    def __add__(self, other):
        r = self._copy_of()
        if isinstance(other, Dat):
            r += other
        else:
            r._shift(other)
        return r

    __radd__ = __add__

    def __sub__(self, other):
        r = self._copy_of()
        if isinstance(other, Dat):
            r -= other
        else:
            r._shift(-float(other))
        return r

    def __rsub__(self, other):
        return (-self).__add__(other)

    def __mul__(self, other):
        r = self._copy_of()
        r *= other
        return r

    __rmul__ = __mul__

    def __truediv__(self, other):
        r = self._copy_of()
        r /= other
        return r

    def maxpy(self, scalars, dats):
        """``self += sum_i scalars[i] * dats[i]`` (pyop2/types/dat.py:509-540)."""
        for a, d in zip(scalars, dats):
            self.axpy(a, d)

    def __call__(self, access, path=None):
        """Legacy parloop argument ``dat(op2.INC, map)`` (pyop2/parloop.py:709-743)."""
        return LegacyArg(self, access, path)

    def __del__(self):
        # the engine's host-pointer mirror cache is keyed on the buffer address: drop the
        # entry so that a later allocation at the same address cannot hit a stale mirror
        try:
            if _lib._initialised is not None and self._data is not None:
                _lib._lib.fdb_mirror_drop(self._data.ctypes.data)
        except Exception:
            pass


class Sparsity:
    """``op2.Sparsity((row_dset, col_dset), [(rmap, cmap, None)])``
    (pyop2/types/mat.py:27-292).  Only square single-block sparsities whose row
    and column maps coincide are supported (every form of the supported set)."""

    mixed = False

    def __init__(self, dsets, maps_and_regions, name=None):
        if isinstance(dsets, MixedDataSet):
            dsets = (dsets, dsets)
        if isinstance(dsets, (tuple, list)) and any(isinstance(d, MixedDataSet) for d in dsets):
            self._init_mixed(tuple(dsets), maps_and_regions, name)
            return
        if isinstance(dsets, DataSet) or isinstance(dsets, Set):
            dsets = (dsets, dsets)
        self.dsets = tuple(_as_dataset(d) for d in dsets)
        if self.dsets[0].set is not self.dsets[1].set:
            raise NotImplementedError("rectangular sparsities are not supported")
        if self.dsets[0].cdim != self.dsets[1].cdim:
            raise NotImplementedError("row and column block sizes must coincide")
        self.bs = self.dsets[0].cdim          # BAIJ block size (pyop2/types/mat.py:741-804)
        self.maps = []
        for entry in maps_and_regions:
            rmap, cmap = entry[0], entry[1]
            if rmap is not cmap:
                raise NotImplementedError("row and column maps must coincide")
            if rmap.toset is not self.dsets[0].set:
                raise MapValueError("sparsity map does not target the data set")
            self.maps.append(rmap)
        if len(self.maps) != 1:
            raise NotImplementedError("exactly one (rmap, cmap) pair is supported")
        self.name = name or "sparsity"

    def _init_mixed(self, dsets, maps_and_regions, name):
        """Sparsity over MixedDataSets (pyop2/types/mat.py:75-160: one block per pair of data sets).
        As the reference's default for mixed spaces (``mat_type='aij'``: ``Mat._init_monolithic``,
        pyop2/types/mat.py:660-700) the blocks live in ONE scalar CSR matrix over the concatenated dof
        numbering ``[block 0 dofs | block 1 dofs | ...]`` (dof = node * cdim + component); its pattern
        comes from the concatenation of the dof-expanded block maps, so the engine's single-map
        sparsity builder serves unchanged.  Square block structures with coinciding row / column maps
        only (as for single blocks); one rank (no halo on the blocks)."""
        rd, cd = dsets
        if not (isinstance(rd, MixedDataSet) and isinstance(cd, MixedDataSet)) or len(rd) != len(cd) or \
                any(r.set is not c.set or r.cdim != c.cdim for r, c in zip(rd, cd)):
            raise NotImplementedError("mixed sparsities must be square: the same data sets for rows and columns")
        if any(d.halo is not None for d in rd):
            raise NotImplementedError("mixed sparsities are not partitioned (no halo on the blocks)")
        if len(maps_and_regions) != 1:
            raise NotImplementedError("exactly one (rmaps, cmaps) pair is supported")
        rmaps, cmaps = maps_and_regions[0][0], maps_and_regions[0][1]
        if not (isinstance(rmaps, MixedMap) and isinstance(cmaps, MixedMap)) or len(rmaps) != len(rd) or \
                any(r is not c for r, c in zip(rmaps, cmaps)):
            raise NotImplementedError("row and column maps must be the same MixedMap blocks")
        for m, d in zip(rmaps, rd):
            if m.toset is not d.set:
                raise MapValueError("sparsity map does not target the data set of its block")
        self.mixed = True
        self.dsets = (rd, cd)
        self.maps = [rmaps]
        self.bs = 1
        self.name = name or "mixed_sparsity"
        sizes = [d.set.total_size * d.cdim for d in rd]
        self.block_offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
        self.mono_set = Set(int(self.block_offsets[-1]), name=self.name + "_dofs")
        self._expanded = {}
        parts = [self.expand_map(m, i) for i, m in enumerate(rmaps)]
        it = rmaps.iterset
        off = None
        if it._extruded:
            off = np.concatenate([e.offset for e in parts])
        self.mono_map = Map(it, self.mono_set, sum(e.arity for e in parts),
                            np.concatenate([e.values_with_halo for e in parts], axis=1),
                            name=self.name + "_map", offset=off)
        self.mono = Sparsity((self.mono_set, self.mono_set), [(self.mono_map, self.mono_map, None)],
                             name=self.name + "_monolithic")

    def expand_map(self, m, block):
        """The dof map of ``m`` (a Map into the node set of ``block``) in the monolithic numbering:
        arity * cdim entries ``offset_block + node * cdim + component``, node-major like the element
        tensors of vector-valued spaces (pyop2/codegen/builder.py:575-625)."""
        key = (id(m), block)
        hit = self._expanded.get(key)
        if hit is not None and hit[0] is m:
            return hit[1]
        d = self.dsets[0][block]
        if m.toset is not d.set:
            raise MapValueError(f"map {m.name} does not target the node set of block {block}")
        cd = d.cdim
        comp = np.arange(cd, dtype=np.int64)
        vals = (m.values_with_halo.astype(np.int64)[:, :, None] * cd + comp[None, None, :]
                + int(self.block_offsets[block])).reshape(m.values_with_halo.shape[0], -1)
        off = None if m.offset is None else np.repeat(m.offset.astype(np.int64) * cd, cd)
        if getattr(m, "offset_quotient", None) is not None:
            raise NotImplementedError("periodic extrusion in a mixed matrix")
        e = Map(m.iterset, self.mono_set, m.arity * cd, vals, name=f"{m.name}_dofs{block}", offset=off)
        self._expanded[key] = (m, e)
        return e

    @property
    def shape(self):
        if self.mixed:
            n = self.mono_set.total_size
            return (n, n)
        n = self.dsets[0].set.total_size
        return (n, n)


class Mat:
    """``op2.Mat(sparsity)`` (pyop2/types/mat.py:607-985) backed by a device CSR
    matrix instead of a PETSc AIJ one.  ``mat(op2.INC, (rmap, cmap), lgmaps=...)``
    builds the parloop argument; ``lgmaps`` = ``(row_lgmap, col_lgmap)`` NumPy
    arrays, identity except -1 on Dirichlet rows / columns."""
    _ids = itertools.count()

    def __init__(self, sparsity: Sparsity, dtype=ScalarType, name=None):
        if sparsity.mixed:
            # monolithic matrix of a mixed space: the scalar CSR of the concatenated dof numbering;
            # ``mat[i, j]`` are MatBlock views (pyop2/types/mat.py:660-700, 990-1060)
            Mat.__init__(self, sparsity.mono, dtype, name)
            self.sparsity = sparsity
            self._blocks = {}
            return
        self.sparsity = sparsity
        self.name = name or f"mat_{next(Mat._ids)}"
        m = sparsity.maps[0]
        it = m.iterset
        nlay = (it.layers - 1) if it._extruded else 1
        off = m.offset
        h = C.c_void_p()
        L = _lib.lib()
        self.bs = sparsity.bs
        if self.bs == 1:
            _lib.check(L.fdb_mat_create(sparsity.shape[0], m.values_with_halo.ctypes.data, it.total_size,
                                        m.arity, None if off is None else off.ctypes.data, nlay,
                                        C.byref(h)), "fdb_mat_create")
        else:
            _lib.check(L.fdb_mat_create_blocked(sparsity.shape[0], m.values_with_halo.ctypes.data,
                                                it.total_size, m.arity,
                                                None if off is None else off.ctypes.data, nlay, self.bs,
                                                C.byref(h)), "fdb_mat_create_blocked")
        self.handle = h
        self.dat_version = 0
        nnz = C.c_longlong()
        nr = C.c_int32()
        L.fdb_mat_nnz(h, C.byref(nnz), C.byref(nr))
        self.nnz = nnz.value
        self.nrows = nr.value

    def __call__(self, access, path, lgmaps=None):
        rmap, cmap = path
        if self._mixed:
            # the whole mixed element tensor at once: rows / columns ordered block by block
            if not (isinstance(rmap, MixedMap) and isinstance(cmap, MixedMap)):
                raise MapValueError("a mixed Mat argument needs MixedMaps (or pass mat[i, j] block by block)")
            sp = self.sparsity
            rmap = sp.mono_map if rmap is sp.maps[0] else self._mono_map_of(rmap)
            cmap = sp.mono_map if cmap is sp.maps[0] else self._mono_map_of(cmap)
        elif getattr(self, "sparsity", None) is not None and \
                not (rmap is self.sparsity.maps[0] and cmap is self.sparsity.maps[0]):
            # pyop2/types/mat.py:439-441.  The scatter finds an entry's position from the sparsity's
            # map (the rank table is per column of that map), so another map over the same sets
            # would add its values at wrong positions without any error
            raise MapValueError("Path maps not in sparsity maps")
        a = LegacyArg(self, access, rmap)
        a.cmap = cmap
        a.lgmaps = lgmaps
        return a

    @property
    def _mixed(self):
        return getattr(getattr(self, "sparsity", None), "mixed", False)

    def _mono_map_of(self, mm):
        sp = self.sparsity
        parts = [sp.expand_map(m, i) for i, m in enumerate(mm)]
        key = ("mono",) + tuple(id(m) for m in mm)
        hit = sp._expanded.get(key)
        if hit is not None and all(a is b for a, b in zip(hit[0], mm)):
            return hit[1]
        off = np.concatenate([e.offset for e in parts]) if mm.iterset._extruded else None
        e = Map(mm.iterset, sp.mono_set, sum(p.arity for p in parts),
                np.concatenate([p.values_with_halo for p in parts], axis=1), offset=off)
        sp._expanded[key] = (tuple(mm), e)
        return e

    def __getitem__(self, ij):
        """``mat[i, j]``: the block coupling row space i and column space j (pyop2 ``MatBlock``)."""
        if not self._mixed:
            if tuple(ij) != (0, 0):
                raise IndexError("a single-block Mat has the block (0, 0) only")
            return self
        i, j = ij
        nb = len(self.sparsity.dsets[0])
        if not (0 <= i < nb and 0 <= j < nb):
            raise IndexError(f"block ({i}, {j}) of a {nb} x {nb} mixed matrix")
        blk = self._blocks.get((i, j))
        if blk is None:
            blk = self._blocks[(i, j)] = MatBlock(self, i, j)
        return blk

    def zero(self):
        _lib.check(_lib.lib().fdb_mat_zero(self.handle), "fdb_mat_zero")
        self.dat_version += 1

    zeroEntries = zero

    # shape bookkeeping of pyop2/types/mat.py:820-890
    @property
    def is_mixed(self):
        return self._mixed

    @property
    def dims(self):
        d = self.sparsity.dsets
        if self._mixed:
            return tuple(tuple((r.dim, c.dim) for c in d[1]) for r in d[0])
        return (((d[0].dim, d[1].dim),),)

    @property
    def nblock_rows(self):
        return len(self.sparsity.dsets[0]) if self._mixed else 1

    @property
    def nblock_cols(self):
        return len(self.sparsity.dsets[1]) if self._mixed else 1

    @property
    def nblocks(self):
        return self.nblock_rows * self.nblock_cols

    @property
    def blocks(self):
        return [[self[i, j] for j in range(self.nblock_cols)] for i in range(self.nblock_rows)]

    def __iter__(self):
        """The blocks in row-major order (pyop2/types/mat.py:835-838)."""
        for row in self.blocks:
            yield from row

    @property
    def ncols(self):
        return self.nrows

    @property
    def shape(self):
        return (self.nrows * self.bs, self.nrows * self.bs)

    def increment_dat_version(self):
        self.dat_version += 1

    def assemble(self):
        """MatAssemblyBegin/End: nothing is stashed here (single address space
        per GPU, owner-computes across GPUs); just drain the stream."""
        _lib.check(_lib.lib().fdb_synchronize())

    def set_local_diagonal_entries(self, rows, diag_val=1.0, idx=None):
        """``rows`` are node rows; ``idx`` selects one component of a blocked
        matrix, default every component (pyop2/types/mat.py:897-937)."""
        rows = np.ascontiguousarray(rows, dtype=IntType)
        if self.bs == 1:
            _lib.check(_lib.lib().fdb_mat_set_diagonal(self.handle, rows.ctypes.data, len(rows),
                                                       float(diag_val)), "fdb_mat_set_diagonal")
        else:
            _lib.check(_lib.lib().fdb_mat_set_diagonal_blocked(
                self.handle, rows.ctypes.data, len(rows), float(diag_val), -1 if idx is None else int(idx)),
                "fdb_mat_set_diagonal_blocked")
        self.dat_version += 1

    def csr(self):
        rowptr = np.empty(self.nrows + 1, dtype=np.int64)
        colidx = np.empty(self.nnz, dtype=IntType)
        vals = np.empty(self.nnz * self.bs * self.bs, dtype=ScalarType)
        _lib.check(_lib.lib().fdb_mat_get_csr(self.handle, rowptr.ctypes.data, colidx.ctypes.data,
                                              vals.ctypes.data), "fdb_mat_get_csr")
        return rowptr, colidx, vals

    @property
    def values(self):
        """Dense copy (small matrices / tests), as ``Mat.values`` in PyOP2."""
        rowptr, colidx, vals = self.csr()
        bs = self.bs
        if bs == 1:
            A = np.zeros((self.nrows, self.nrows))
            for r in range(self.nrows):
                A[r, colidx[rowptr[r]:rowptr[r + 1]]] = vals[rowptr[r]:rowptr[r + 1]]
            return A
        A = np.zeros((self.nrows * bs, self.nrows * bs))
        blocks = vals.reshape(-1, bs, bs)
        for r in range(self.nrows):
            for k in range(rowptr[r], rowptr[r + 1]):
                c = colidx[k]
                A[r * bs:(r + 1) * bs, c * bs:(c + 1) * bs] = blocks[k]
        return A

    def mult(self, x, y):
        if self._mixed and isinstance(x, MixedDat):
            # block vectors <-> the contiguous dof vector of the monolithic matrix (device copies)
            L = _lib.lib()
            if getattr(self, "_xy", None) is None:
                self._xy = (Dat(self.sparsity.mono_set), Dat(self.sparsity.mono_set))
            xm, ym = self._xy
            offs = self.sparsity.block_offsets
            xm.zero()
            xd, yd = xm.device_ptr, ym.device_ptr
            for xb, o in zip(x, offs):           # plain device copies: no alignment demands on odd offsets
                _lib.check(L.fdb_memcpy_d2d(xd + int(o) * 8, xb.device_ptr, xb.nbytes), "pack")
            xm._device_written()
            _lib.check(L.fdb_mat_mult(self.handle, xd, yd), "fdb_mat_mult")
            ym._device_written()
            for yb, o in zip(y, offs):
                _lib.check(L.fdb_memcpy_d2d(yb.device_ptr, yd + int(o) * 8, yb.nbytes), "unpack")
                yb._device_written()
            return
        _lib.check(_lib.lib().fdb_mat_mult(self.handle, x.device_ptr, y.device_ptr), "fdb_mat_mult")
        y._device_written()

    def __del__(self):
        try:
            if self.handle is not None and _lib._initialised is not None:
                _lib._lib.fdb_mat_destroy(self.handle)
        except Exception:
            pass


class MatBlock(Mat):
    """``mixed_mat[i, j]`` (pyop2/types/mat.py MatBlock, ``MatGetLocalSubMatrix``): a VIEW of the
    monolithic matrix.  ``block(op2.INC, (rmap_i, cmap_j), lgmaps=...)`` is a parloop argument whose
    maps are the dof-expanded, offset maps of the two spaces (block size 1), so the element tensor
    of the block, rows (node, component) x columns (node, component), lands in the right rows and
    columns of the parent; ``lgmaps`` are dof-level arrays over the block's own rows / columns."""

    def __init__(self, parent, i, j):
        self.parent, self.i, self.j = parent, i, j
        self.sparsity = parent.sparsity
        self.handle = parent.handle
        self.bs = 1
        self.name = f"{parent.name}_{i}{j}"

    @property
    def dat_version(self):
        return self.parent.dat_version

    @dat_version.setter
    def dat_version(self, v):
        self.parent.dat_version = v

    @property
    def _range(self):
        o = self.sparsity.block_offsets
        return (int(o[self.i]), int(o[self.i + 1])), (int(o[self.j]), int(o[self.j + 1]))

    def __call__(self, access, path, lgmaps=None):
        rmap, cmap = path
        sp = self.sparsity
        a = LegacyArg(self, access, sp.expand_map(rmap, self.i))
        a.cmap = sp.expand_map(cmap, self.j)
        a.lgmaps = None
        if lgmaps is not None:
            n = sp.mono_set.total_size
            (r0, r1), (c0, c1) = self._range
            out = []
            for lg, lo, hi in ((lgmaps[0], r0, r1), (lgmaps[1], c0, c1)):
                lg = np.asarray(lg, dtype=np.int64).ravel()
                if lg.size != hi - lo:
                    raise ValueError(f"block lgmap has {lg.size} entries, the block has {hi - lo} dofs")
                full = np.arange(n, dtype=np.int64)
                full[lo:hi] = np.where(lg >= 0, lg + lo, -1)
                out.append(full.astype(IntType))
            a.lgmaps = tuple(out)
        return a

    _mixed = False                              # a block is a single-block matrix to its users

    def __getitem__(self, ij):
        if tuple(ij) != (0, 0):
            raise IndexError("a MatBlock has the block (0, 0) only")
        return self

    @property
    def dims(self):
        d = self.sparsity.dsets
        return (((d[0][self.i].dim, d[1][self.j].dim),),)

    @property
    def shape(self):
        (r0, r1), (c0, c1) = self._range
        return (r1 - r0, c1 - c0)

    @property
    def nrows(self):
        return self.shape[0]

    @property
    def ncols(self):
        return self.shape[1]

    def zero(self):
        raise NotImplementedError("zero the mixed Mat, not one of its blocks")

    def assemble(self):
        self.parent.assemble()

    def set_local_diagonal_entries(self, rows, diag_val=1.0, idx=None):
        """Diagonal of a diagonal block: ``rows`` are NODE rows of the block's space, ``idx`` one
        component (default all), as for blocked matrices (pyop2/types/mat.py:897-937)."""
        if self.i != self.j:
            raise ValueError("only diagonal blocks have a diagonal")
        cd = self.sparsity.dsets[0][self.i].cdim
        rows = np.asarray(rows, dtype=np.int64).ravel()
        comps = np.arange(cd) if idx is None else np.array([int(idx)])
        dofs = (rows[:, None] * cd + comps[None, :]).ravel() + self._range[0][0]
        Mat.set_local_diagonal_entries(self.parent, dofs.astype(IntType), diag_val)

    @property
    def values(self):
        (r0, r1), (c0, c1) = self._range
        return self.parent.values[r0:r1, c0:c1]

    def mult(self, x, y):
        raise NotImplementedError("multiply with the mixed Mat")

    def __del__(self):
        pass                                    # the parent owns the engine handle


class Global:
    def __init__(self, dim, data=None, dtype=ScalarType, name=None, comm=None):
        self.dim = (dim,) if isinstance(dim, (int, np.integer)) else tuple(dim)
        self._data = (np.zeros(self.dim, dtype=dtype) if data is None
                      else np.asarray(data, dtype=dtype).reshape(self.dim).copy())
        self.name = name or "global"
        self.dat_version = 0

    @property
    def data(self):
        self.dat_version += 1
        return self._data

    @property
    def data_ro(self):
        return self._data

    # host data: the vector operations of pyop2/types/glob.py:33-180 are NumPy one-liners
    @property
    def data_wo(self):
        return self.data

    @property
    def shape(self):
        return self._data.shape

    @property
    def dtype(self):
        return self._data.dtype

    @property
    def nbytes(self):
        return self._data.nbytes

    def increment_dat_version(self):
        self.dat_version += 1

    def split(self):
        return (self,)

    def zero(self, subset=None):
        if subset is not None:
            raise NotImplementedError("a Global has no subsets")
        self.data[...] = 0

    def copy(self, other, subset=None):
        """``other <- self`` (the direction of Dat.copy)."""
        other.data[...] = self._data

    def duplicate(self):
        return Global(self.dim, self._data, dtype=self._data.dtype, name=self.name + "_dup")

    def inner(self, other):
        return float(np.dot(self._data.ravel(), np.conj(other.data_ro.ravel())))

    def axpy(self, alpha, other):
        self.data[...] += alpha * other.data_ro

    def maxpy(self, scalars, globs):
        for a, g in zip(scalars, globs):
            self.axpy(a, g)

    def __call__(self, access, path=None):
        return LegacyArg(self, access, None)


@dataclass
class LegacyArg:
    data: object
    access: Access
    map: object = None
    lgmaps: object = None


# ------------------------------------------------------------------- kernels
@dataclass(frozen=True)
class Kernel:
    """The local kernel.  In the reference this wraps TSFC-generated loopy or a
    C string (pyop2/local_kernel.py:33-43, 186-207); here it names one of the
    hand-written sm_100a element kernels through a form descriptor.

    ``form``: "helmholtz" family = ``alpha*inner(grad u, grad v)*dx +
    beta*inner(u, v)*dx``.  ``rank`` 1 means the 1-form ``action(a, w)``
    (arguments: output Dat INC, coordinates READ, coefficient READ), the kernel
    TSFC names ``form0_cell_integral``.
    """
    form: str = "helmholtz"
    degree: int = 1
    alpha: float = 1.0
    beta: float = 0.0
    rank: int = 1
    cdim: int = 1
    integral: str = "cell"          # "cell" | "exterior_facet" | "interior_facet"
    cell: str = "hex"               # "hex" (extruded or native) | "triangle" (affine P1)
    diagonal: bool = False          # rank 1: diagonal of the bilinear form (args: d, coordinates)
    affine: bool = False            # rank 1 hex: promise that all cells are parallelepipeds (fdb_kernel_desc.affine_cells)
    nq: int = 0                     # 1-D quadrature points (0: the form's default)
    name: str = "form0_cell_integral"
    accesses: tuple = (INC, READ, READ)
    # tabulation: a fiat_lite.Interval1D, or None for the default GLL/Gauss pair
    element: object = field(default=None, compare=False, hash=False)

    def __new__(cls, *args, **kwargs):
        # ``op2.Kernel(code, name)`` with C source (pyop2/local_kernel.py:33-43) builds the
        # generic local kernel; form descriptors name the hand-written fast paths
        src = args[0] if args else kwargs.get("code")
        if isinstance(src, str) and ("(" in src or "code" in kwargs):
            from .codegen import CStringKernel
            return CStringKernel(*args, **kwargs)
        return super().__new__(cls)

    def __post_init__(self):
        if self.form == "dg_advection":
            # args: out, coordinates, q, u, constants (dtc, q_in) [, local facet numbers]
            extra = {"cell": 0, "exterior_facet": 1, "interior_facet": 1, "fused": 2}[self.integral]
            acc = (INC, READ, READ, READ, READ) + (READ,) * extra
            object.__setattr__(self, "accesses", acc)
            object.__setattr__(self, "name", f"form0_{self.integral}_integral")
        if self.diagonal:
            object.__setattr__(self, "accesses", (INC, READ))
        if self.rank == 2 and self.accesses == (INC, READ, READ):
            object.__setattr__(self, "accesses", (INC, READ))
            if self.name == "form0_cell_integral":
                object.__setattr__(self, "name", "form00_cell_integral")

    @property
    def num_flops(self):
        n = self.degree + 1
        return 2 * 6 * n ** 4 * 2 + 130 * n ** 3


_FORMS = {"helmholtz": _lib.FORM_HELMHOLTZ, "dg_advection": _lib.FORM_DG_ADVECTION}
_INTEGRALS = {"cell": _lib.INTEGRAL_CELL, "exterior_facet": _lib.INTEGRAL_EXTERIOR_FACET,
              "interior_facet": _lib.INTEGRAL_INTERIOR_FACET, "fused": _lib.INTEGRAL_FUSED}


class GlobalKernel:
    """pyop2/global_kernel.py:255-335: the compile-time description of a
    parloop.  ``__call__`` is the Python -> native boundary."""
    _cache = {}

    def __init__(self, local_kernel: Kernel, arguments, *, extruded=False,
                 constant_layers=True, subset=False, scatter="atomic"):
        self.local_kernel = local_kernel
        self.arguments = tuple(arguments)      # (Map, Map): argument map, coordinate map
        self.extruded = extruded
        self.constant_layers = constant_layers
        self.subset = subset
        self.scatter = scatter
        self._handle = None
        if extruded and not constant_layers:
            raise NotImplementedError("the hand-written kernels take constant layers; variable layers run "
                                      "on the generic wrapper path (op2.Kernel(code, name))")

    @property
    def name(self):
        return "wrap_" + self.local_kernel.name          # global_kernel.py:344-346

    def compile(self):
        if self._handle is not None:
            return self._handle
        from .fiat_lite import gauss_legendre, interval_element
        lk = self.local_kernel
        if lk.form == "dg_advection":
            nq = lk.nq or 3
            d = _lib.KernelDesc()
            d.form, d.rank, d.cell = _FORMS[lk.form], 1, _lib.CELL_QUAD
            d.integral = _INTEGRALS[lk.integral]
            d.degree, d.nq, d.cdim, d.scatter = 1, nq, 1, _lib.SCATTER_ATOMIC
            xq, wq = gauss_legendre(nq)
            for i in range(nq):
                d.xq[i], d.wq[i] = xq[i], wq[i]
            # DQ1: default "spectral" variant = Gauss-Legendre nodes on the interval
            el = lk.element or interval_element(1, 2, "gl")
            Bend, _ = el.tabulate([0.0, 1.0])
            for e in range(2):
                for i in range(2):
                    d.B[e * 2 + i] = Bend[e, i]
            h = C.c_void_p()
            _lib.check(_lib.lib().fdb_kernel_create(C.byref(d), C.byref(h)), "fdb_kernel_create")
            self._handle = h
            return h
        if lk.cell == "triangle":
            # P1 on affine triangles, FIAT basis order (1-x-y, x, y), 3-point
            # edge-midpoint rule (degree 2, exact for the P1 mass matrix)
            d = _lib.KernelDesc()
            d.form, d.rank, d.cell = _FORMS[lk.form], lk.rank, _lib.CELL_TRIANGLE
            d.integral, d.degree, d.nq, d.cdim, d.scatter = _lib.INTEGRAL_CELL, 1, 3, 1, _lib.SCATTER_ATOMIC
            d.alpha, d.beta = lk.alpha, lk.beta
            pts = [(0.5, 0.0), (0.5, 0.5), (0.0, 0.5)]
            for q, (x, y) in enumerate(pts):
                d.B[0 * 3 + q], d.B[1 * 3 + q], d.B[2 * 3 + q] = 1 - x - y, x, y
                d.wq[q] = 1.0 / 6.0
            for i, g in enumerate([(-1.0, -1.0), (1.0, 0.0), (0.0, 1.0)]):
                d.D[i * 2], d.D[i * 2 + 1] = g
            h = C.c_void_p()
            _lib.check(_lib.lib().fdb_kernel_create(C.byref(d), C.byref(h)), "fdb_kernel_create")
            self._handle = h
            return h
        el = lk.element or interval_element(lk.degree)
        n = lk.degree + 1
        if el.ndof != n:
            raise ValueError("element degree does not match the kernel")
        d = _lib.KernelDesc()
        d.form = _FORMS[lk.form]
        d.rank = lk.rank
        d.cell = _lib.CELL_HEX_EXTRUDED if self.extruded else _lib.CELL_HEX
        d.integral = _lib.INTEGRAL_CELL
        d.degree = lk.degree
        d.nq = el.nq
        d.cdim = lk.cdim
        d.scatter = {"atomic": _lib.SCATTER_ATOMIC, "coloured": _lib.SCATTER_COLOURED}[self.scatter]
        d.alpha, d.beta = lk.alpha, lk.beta
        d.diagonal = int(lk.diagonal)
        d.affine_cells = int(lk.affine and lk.rank == 1 and not lk.diagonal)
        for q in range(el.nq):
            d.wq[q] = el.wq[q]
            d.xq[q] = el.xq[q]
            for a in range(n):
                d.B[q * n + a] = el.B[q, a]
                d.D[q * n + a] = el.D[q, a]
        m0, m1 = self.arguments
        keep = []
        if self.extruded:
            if m0.offset is None or m1.offset is None:
                raise MapValueError("extruded parloop needs maps with offsets")
            o0 = np.ascontiguousarray(m0.offset, dtype=IntType)
            o1 = np.ascontiguousarray(m1.offset, dtype=IntType)
            keep = [o0, o1]
            d.offset0 = o0.ctypes.data_as(C.POINTER(C.c_int32))
            d.offset1 = o1.ctypes.data_as(C.POINTER(C.c_int32))
        h = C.c_void_p()
        _lib.check(_lib.lib().fdb_kernel_create(C.byref(d), C.byref(h)), "fdb_kernel_create")
        del keep
        self._handle = h
        return h

    def __call__(self, start, end, layers, subset_indices, args, arg_bytes, arg_versions,
                 maps, map_bytes, location, writeback, output_is_zero, map_versions=None,
                 subset_version=0):
        h = self.compile()
        ca = _lib.CallArgs()
        ca.start, ca.end = int(start), int(end)
        if layers is not None:
            ca.layers = layers.ctypes.data_as(C.POINTER(C.c_int32))
        ca.subset = subset_indices
        ca.nargs = len(args)
        ca.args = (C.c_void_p * len(args))(*args)
        if arg_bytes is not None:
            ca.arg_bytes = (C.c_size_t * len(args))(*arg_bytes)
            ca.arg_versions = (C.c_uint64 * len(args))(*arg_versions)
        ca.nmaps = len(maps)
        ca.maps = (C.c_void_p * len(maps))(*maps)
        if map_bytes is not None:
            ca.map_bytes = (C.c_size_t * len(maps))(*map_bytes)
        if map_versions is not None:
            ca.map_versions = (C.c_uint64 * len(maps))(*map_versions)
        ca.subset_version = int(subset_version)
        ca.location = location
        ca.writeback = int(writeback)
        ca.output_is_zero = int(output_is_zero)
        _lib.check(_lib.lib().fdb_kernel_call(h, C.byref(ca)), self.name)

    def __del__(self):
        try:
            if self._handle is not None and _lib._initialised is not None:
                _lib._lib.fdb_kernel_destroy(self._handle)
        except Exception:
            pass


class _PhaseTimer:
    """FDB_PHASE_TIMING=1: synchronise after every phase of a partitioned parloop and accumulate
    host wall time per phase (diagnostics only: the synchronisation removes all overlap)."""
    _inst = None

    def __init__(self, on):
        self.on, self.t, self.acc = on, None, {}
        if on:
            import atexit
            atexit.register(self.report)

    @classmethod
    def get(cls):
        if cls._inst is None:
            import os
            cls._inst = cls(os.environ.get("FDB_PHASE_TIMING") == "1")
        if cls._inst.on:
            import time
            _lib.check(_lib.lib().fdb_synchronize())
            cls._inst.t = time.perf_counter()
        return cls._inst

    def mark(self, name):
        if self.on:
            import time
            _lib.check(_lib.lib().fdb_synchronize())
            now = time.perf_counter()
            a = self.acc.setdefault(name, [0, 0.0])
            a[0] += 1
            a[1] += now - self.t
            self.t = now

    def report(self):
        import os
        print("phase timing rank", os.environ.get("RANK", "0"),
              {k: "%d x %.3f ms" % (n, 1e3 * t / n) for k, (n, t) in self.acc.items()}, flush=True)


class Parloop:
    """pyop2/parloop.py:167-260.  ``args`` are ``LegacyArg``s in TSFC argument
    order (output, coordinates, coefficient).  ``__call__`` follows the
    reference protocol: compute core, (halo exchanges are driven by
    firedrake_b200.halo when a halo is attached), compute owned, bump the
    version of written Dats."""

    def __init__(self, global_knl: GlobalKernel, iterset: Set, args, location="device"):
        self.global_kernel = global_knl
        self.iterset = iterset
        self.args = list(args)
        self.location = location
        self._check()

    def _check(self):
        base = self.iterset.superset if isinstance(self.iterset, Subset) else self.iterset
        if getattr(base, "extruded_periodic", False):
            raise NotImplementedError("periodic extrusion (offset_quotient) runs on the generic wrapper path: "
                                      "pass the local kernel as C source (op2.Kernel(code, name))")
        if not getattr(base, "constant_layers", True):
            raise NotImplementedError("variable layers run on the generic wrapper path: "
                                      "pass the local kernel as C source (op2.Kernel(code, name))")
        lk = self.global_kernel.local_kernel
        if len(self.args) != len(lk.accesses):
            raise ValueError(f"kernel takes {len(lk.accesses)} arguments, got {len(self.args)}")
        for a, acc in zip(self.args, lk.accesses):
            if a.access != acc:
                raise ValueError(f"argument {a.data.name}: access {a.access.name} != kernel's {acc.name}")
            if a.map is not None:
                base = self.iterset.superset if isinstance(self.iterset, Subset) else self.iterset
                if a.map.iterset is not base:
                    raise MapValueError(f"map {a.map.name} is not defined on the iteration set")
                toset = (a.data.sparsity.dsets[0].set if isinstance(a.data, Mat)
                         else a.data.dataset.set)
                if a.map.toset is not toset:
                    raise MapValueError(f"map {a.map.name} does not target {a.data.name}'s set")

    # the two compute phases of pyop2/parloop.py:250-253
    def _compute(self, part):
        start, end = part
        if end <= start:
            return
        gk = self.global_kernel
        it = self.iterset
        layers = it.layers_array.ravel() if it._extruded else None
        out = self.args[0].data
        maps = []
        for a in self.args:
            if a.map is not None and a.map not in maps:
                maps.append(a.map)       # distinct maps, first-use order
        if isinstance(out, Mat):
            # replace_lgmaps (pyop2/parloop.py:279-314): BC-masked maps for this loop only
            L = _lib.lib()
            lg = self.args[0].lgmaps
            if lg is not None:
                r, c = (np.ascontiguousarray(v, dtype=IntType) for v in lg)
                _lib.check(L.fdb_mat_set_lgmaps(out.handle, r.ctypes.data, c.ctypes.data))
            subset = None
            if isinstance(it, Subset):
                if not hasattr(it, "_dev_idx"):
                    it._dev_idx = DeviceArray.from_host(it.indices)
                subset = it._dev_idx.ptr
            coords = self.args[1].data
            try:
                gk(start, end, layers, subset, [out.handle.value, coords.device_ptr], None, None,
                   [m.device_ptr for m in maps], None, _lib.LOC_DEVICE, False, False)
            finally:
                if lg is not None:
                    _lib.check(L.fdb_mat_set_lgmaps(out.handle, None, None))
            out.dat_version += 1
            return
        if self.location == "device":
            subset = None
            if isinstance(it, Subset):
                if not hasattr(it, "_dev_idx"):
                    it._dev_idx = DeviceArray.from_host(it.indices)
                subset = it._dev_idx.ptr
            ptrs = [a.data._data.ctypes.data if isinstance(a.data, Global) else a.data.device_ptr
                    for a in self.args]
            gk(start, end, layers, subset, ptrs, None, None, [m.device_ptr for m in maps], None,
               _lib.LOC_DEVICE, False, False)
            out._device_written()
        else:
            subset = it.indices.ctypes.data if isinstance(it, Subset) else None
            lazy_zero = out._is_zero and not out._host_valid
            for a in self.args:
                if not (a.data is out and lazy_zero):
                    a.data._sync_host()
            ptrs = [a.data._data.ctypes.data for a in self.args]
            nbytes = [a.data._data.nbytes for a in self.args]
            vers = [a.data.dat_version for a in self.args]
            gk(start, end, layers, subset, ptrs, nbytes, vers,
               [m.values_with_halo.ctypes.data for m in maps],
               [m.values_with_halo.nbytes for m in maps], _lib.LOC_HOST, True, out._is_zero,
               map_versions=[m._generation for m in maps],
               subset_version=it._generation if isinstance(it, Subset) else 0)
            out.increment_dat_version()      # pyop2/parloop.py:262-272
            out._is_zero = False
            out._host_valid = True           # written back by the engine
            out._dev_valid = False

    def __call__(self):
        """pyop2/parloop.py:243-260: halo begin -> core -> halo end -> owned ->
        local-to-global reduce of INC Dats."""
        reads = [a.data for a in self.args
                 if a.access == READ and isinstance(a.data, Dat) and a.data.dataset.halo is not None
                 and not a.data.halo_valid]
        if reads and self.location != "device":
            base0 = self.iterset.superset if isinstance(self.iterset, Subset) else self.iterset
            if getattr(base0, "owner_computes", False) and len(self.args) == 3 and not isinstance(self.iterset, Subset):
                return self._call_host_partitioned()
            raise NotImplementedError("halo exchanges on host-resident Dats need an exec-halo partition "
                                      "(SlabPartition(exec_halo=True)); otherwise use location='device'")
        incs = [a.data for a in self.args
                if a.access == INC and isinstance(a.data, Dat) and a.data.dataset.halo is not None
                and not a.data.frozen_halo]
        base = self.iterset.superset if isinstance(self.iterset, Subset) else self.iterset
        if getattr(base, "owner_computes", False) and not isinstance(self.iterset, Subset):
            # the set is partitioned with EXEC-HALO entries (partition.SlabPartition(exec_halo=True),
            # flagged on every rank, including those that hold no exec cells themselves): executing
            # them redundantly completes every owned row locally, so INC Dats need no local->global
            # reduce (SURVEY.md section 8e option (ii)); their ghost rows are left holding partial
            # sums and are marked stale, as after the reference's reduce
            ph = _PhaseTimer.get()
            for d in reads:
                d.dataset.halo.global_to_local_begin(d)
            ph.mark("g2l_begin")
            self._compute(self.iterset.core_part)
            ph.mark("core")
            for d in reads:
                d.dataset.halo.global_to_local_end(d)
            ph.mark("g2l_end")
            self._compute((self.iterset.core_size, self.iterset.total_size))   # owned + exec halo
            ph.mark("owned+exec")
            for d in incs:
                d._device_written(halo_valid=False)
            return
        for d in incs:
            d._reset_ghost_rows(INC)
        for d in reads:
            d.dataset.halo.global_to_local_begin(d)
        c0, c1 = self.iterset.core_part
        if reads and incs and c1 - c0 >= 8:
            # Both exchanges are hidden behind core cells: a first slice of the
            # core part covers the global->local latency, then the cells that
            # touch ghost rows run, their contributions leave (local->global
            # begin) and the rest of the core part overlaps that exchange.  Same
            # result as the reference order (INC is order independent).
            split = c0 + max(1, (c1 - c0) // 8)
            self._compute((c0, split))
            for d in reads:
                d.dataset.halo.global_to_local_end(d)
            self._compute(self.iterset.owned_part)
            for d in incs:
                d.dataset.halo.local_to_global_begin(d)
            self._compute((split, c1))
            for d in incs:
                d.dataset.halo.local_to_global_end(d)
            return
        self._compute(self.iterset.core_part)
        for d in reads:
            d.dataset.halo.global_to_local_end(d)
        self._compute(self.iterset.owned_part)
        for d in incs:
            d.dataset.halo.local_to_global_begin(d)
            d.dataset.halo.local_to_global_end(d)

    compute = __call__

    # -- host-resident Dats on a partitioned mesh (exec-halo protocol) -------------------------------
    def _host_plan(self):
        """Row ranges of the partitioned host path, read off the map once: ``upto`` = rows the core
        cells touch (the engine's chunked pipeline uploads exactly those), ``ranges`` = owned rows the
        boundary cells (owned-non-core + exec halo) touch, merged into a few contiguous ranges."""
        if getattr(self, "_hplan", None) is None:
            it = self.iterset
            m = self.args[0].map
            mp = m.values_with_halo.astype(np.int64)
            nlay = it.layers - 1 if it._extruded else 1
            off = (m.offset if m.offset is not None else np.zeros(m.arity, dtype=IntType)).astype(np.int64)
            owned = self.args[0].data.dataset.set.size
            top = mp + off[None, :] * (nlay - 1) + 1
            upto = int(top[:it.core_size].max()) if it.core_size else 0
            lo = mp[it.core_size:].ravel()
            hi = top[it.core_size:].ravel()
            keep = lo < owned
            lo, hi = lo[keep], np.minimum(hi[keep], owned)
            order = np.argsort(lo, kind="stable")
            ranges = []
            for a, b in zip(lo[order].tolist(), hi[order].tolist()):
                if ranges and a - ranges[-1][1] <= 65536:
                    ranges[-1][1] = max(ranges[-1][1], b)
                else:
                    ranges.append([a, b])
            self._hplan = (min(upto, owned), owned, ranges)
        return self._hplan

    def _call_host_partitioned(self):
        """``location="host"`` on an exec-halo partition: pinned host Dats in, host Dats out, every
        PCIe transfer overlapped with compute where the data dependences allow --
        1. core cells through the engine's chunked pipeline (H2D of x | kernel | D2H of y, three streams),
        2. the owned rows of x the core cells never read are uploaded, ghost rows arrive from their
           owners (NCCL, device to device: the host copies of ghost rows are stale by definition),
        3. boundary cells (owned-non-core + exec halo) on the mirrors,
        4. the few row ranges of y they touch are downloaded again."""
        it = self.iterset
        out, X, x = (a.data for a in self.args)
        m0, m1 = self.args[0].map, self.args[1].map
        L = _lib.lib()
        upto, owned, ranges = self._host_plan()
        self._compute(it.core_part)                               # 1. (host path: pipelined when large)
        rowb = x.cdim * x.dtype.itemsize

        def mirror(buf, version, upload):
            d = C.c_void_p()
            _lib.check(L.fdb_mirror_acquire(buf.ctypes.data, buf.nbytes, int(version), int(upload), C.byref(d)),
                       "fdb_mirror_acquire")
            return d.value
        xd = mirror(x._data, x.dat_version, 0)
        if it.core_size == 0:                                     # nothing ran yet: whole upload, zero output
            upto = 0
            yd0 = mirror(out._data, out.dat_version, 0)
            _lib.check(L.fdb_memset(yd0, 0, out._data.nbytes))
            out.increment_dat_version()
        if owned > upto:                                          # 2.
            _lib.check(L.fdb_mirror_upload_range(x._data.ctypes.data, upto * rowb, (owned - upto) * rowb),
                       "fdb_mirror_upload_range")
        halo = x.dataset.halo
        _lib.check(L.fdb_halo_global_to_local_begin(halo.handle, xd, x.cdim))
        _lib.check(L.fdb_halo_global_to_local_end(halo.handle, xd, x.cdim))
        _lib.check(L.fdb_mirror_set_version(x._data.ctypes.data, int(x.dat_version)))
        if it.total_size > it.core_size:                          # 3.
            yd = mirror(out._data, out.dat_version, 0)
            Xd = mirror(X._data, X.dat_version, 1)
            md = [mirror(m.values_with_halo, m._generation, 1) for m in (m0, m1)]
            layers = it.layers_array.ravel() if it._extruded else None
            self.global_kernel(it.core_size, it.total_size, layers, None, [yd, Xd, xd], None, None, md, None,
                               _lib.LOC_DEVICE, False, False)
            yb = out._data
            orow = out.cdim * out.dtype.itemsize
            for k, (a, b) in enumerate(ranges):                   # 4.
                _lib.check(L.fdb_mirror_download_range(yb.ctypes.data, a * orow, (b - a) * orow,
                                                       int(k == len(ranges) - 1)), "fdb_mirror_download_range")
        out._host_valid, out._dev_valid, out._is_zero = True, False, False
        out.halo_valid = False


def par_loop(kernel: Kernel, iterset: Set, *args, location="device", scatter="atomic"):
    """``op2.par_loop(kernel, iterset, dat(op2.INC, map), ...)``
    (pyop2/parloop.py:705-762)."""
    from . import codegen
    if isinstance(kernel, codegen.CStringKernel):
        return codegen.par_loop(kernel, iterset, *args)
    maps = []
    for a in args:
        if a.map is not None and a.map not in maps:
            maps.append(a.map)
    base = iterset.superset if isinstance(iterset, Subset) else iterset
    gk = GlobalKernel(kernel, maps, extruded=base._extruded, subset=isinstance(iterset, Subset),
                      scatter=scatter)
    Parloop(gk, iterset, args, location=location)()
    return gk


def __getattr__(name):
    # lazily re-exported from codegen (which imports this module)
    if name in ("PermutedMap", "CStringKernel"):
        from . import codegen
        return getattr(codegen, name)
    raise AttributeError(name)
