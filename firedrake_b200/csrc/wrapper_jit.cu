// Generic wrapper builder: the replacement for PyOP2's code generation of the
// global kernel around an ARBITRARY local kernel
//   pyop2/codegen/builder.py:702-1008   WrapperBuilder (loops, packs, kernel call)
//   pyop2/codegen/builder.py:215-300    GlobalPack
//   pyop2/codegen/builder.py:322-429    DatPack (gather / scatter by access mode)
//   pyop2/codegen/builder.py:520-625    MatPack (MatSetValues[Blocked]Local)
//   pyop2/codegen/rep2loopy.py:409-593  lowering to C
//   pyop2/compilation.py:424-455        cc + dlopen
// Here: the local kernel's C source is wrapped into one CUDA kernel (one thread
// per iteration-set entry and layer, layers fastest so that a warp walks up a
// column: the map row is a broadcast and the Dat accesses of the 32 lanes are
// `offset[i]` apart), compiled with NVRTC for sm_100a and loaded with the
// runtime's library API.  The hand-written kernels in action_hex.cu etc. are the
// fast path for the forms they cover; this file is the general path, so the
// engine never needs a CPU to run a parloop.
//
// The generated text has two parts separated by a marker line: a prelude
// (types, parameter block, atomics, reductions, the kernel entry macro) and a
// flavour-independent body (local kernel + wrapper).  tests/ re-compile the body
// with g++ against a host prelude to check the generated packing/unpacking code
// against the reference's golden arrays without a GPU.
#include <ctype.h>
#include <dlfcn.h>
#include <stdarg.h>
#include <stdlib.h>

#include <algorithm>
#include <sstream>
#include <string>
#include <vector>

#include "common.cuh"

using namespace fdb;

// ---------------------------------------------------------------------------
// parameter block shared by the launcher and the generated kernel (the prelude
// below restates it textually; tests/ mirror it with ctypes)
struct FdbMatView {
    const long long *rowptr;
    const int *colidx;
    double *vals;
    const int *row_lg;     // dof-level (nrows*bs_r) or NULL = identity
    const int *col_lg;
    int bs_r, bs_c;
};

struct FdbWrapParams {
    int start, end;        // iteration range
    int layer_lo, layer_hi;  // cell layers iterated: [layer_lo, layer_hi)
    int bottom;            // layers[0]
    int ncl;               // cell layers per column (the modulus of periodic extrusion)
    const int *subset;
    const int *col_layers; // variable layers: int[ncolumns][2] node-layer extents, else NULL
    void *arg[FDB_WRAP_MAX_ARGS];
    const int *map[FDB_WRAP_MAX_MAPS];
    FdbMatView mat[FDB_WRAP_MAX_MATS];
};

namespace {

const char *kPreludeEnd = "/* ==== fdb200 prelude end ==== */";

const char *kPrelude = R"PRELUDE(
// ---- fdb200 generated global kernel: CUDA prelude ----
typedef signed char int8_t;
typedef unsigned char uint8_t;
typedef short int16_t;
typedef unsigned short uint16_t;
typedef int int32_t;
typedef unsigned int uint32_t;
typedef long long int64_t;
typedef unsigned long long uint64_t;
typedef unsigned long size_t;
typedef double PetscScalar;
typedef double PetscReal;
typedef int PetscInt;
#define restrict __restrict__
#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif
#define FDB_DEVICE __device__ __forceinline__
#define FDB_CONST __device__ const
#define FDB_ABORT() __trap()

struct FdbMatView {
    const long long *rowptr;
    const int *colidx;
    double *vals;
    const int *row_lg;
    const int *col_lg;
    int bs_r, bs_c;
};
struct FdbWrapParams {
    int start, end;
    int layer_lo, layer_hi;
    int bottom;
    int ncl;
    const int *subset;
    const int *col_layers; // variable layers: int[ncolumns][2] node-layer extents, else NULL
    void *arg[16];
    const int *map[8];
    FdbMatView mat[4];
};

// ---- scatter primitives (A5): INC / MIN / MAX on Dats are atomics
FDB_DEVICE void fdb_atomic_add(double *p, double v) { atomicAdd(p, v); }
FDB_DEVICE void fdb_atomic_add(float *p, float v) { atomicAdd(p, v); }
FDB_DEVICE void fdb_atomic_add(int *p, int v) { atomicAdd(p, v); }
FDB_DEVICE void fdb_atomic_add(unsigned int *p, unsigned int v) { atomicAdd(p, v); }
FDB_DEVICE void fdb_atomic_add(long long *p, long long v)
{
    atomicAdd((unsigned long long *)p, (unsigned long long)v);
}
FDB_DEVICE void fdb_atomic_min(int *p, int v) { atomicMin(p, v); }
FDB_DEVICE void fdb_atomic_min(unsigned int *p, unsigned int v) { atomicMin(p, v); }
FDB_DEVICE void fdb_atomic_min(long long *p, long long v) { atomicMin(p, v); }
FDB_DEVICE void fdb_atomic_max(int *p, int v) { atomicMax(p, v); }
FDB_DEVICE void fdb_atomic_max(unsigned int *p, unsigned int v) { atomicMax(p, v); }
FDB_DEVICE void fdb_atomic_max(long long *p, long long v) { atomicMax(p, v); }
FDB_DEVICE void fdb_atomic_min(double *p, double v)
{
    unsigned long long *a = (unsigned long long *)p, old = *a, seen;
    do {
        seen = old;
        if (!(v < __longlong_as_double((long long)seen))) break;
        old = atomicCAS(a, seen, (unsigned long long)__double_as_longlong(v));
    } while (old != seen);
}
FDB_DEVICE void fdb_atomic_max(double *p, double v)
{
    unsigned long long *a = (unsigned long long *)p, old = *a, seen;
    do {
        seen = old;
        if (!(v > __longlong_as_double((long long)seen))) break;
        old = atomicCAS(a, seen, (unsigned long long)__double_as_longlong(v));
    } while (old != seen);
}
FDB_DEVICE void fdb_atomic_min(float *p, float v)
{
    unsigned int *a = (unsigned int *)p, old = *a, seen;
    do {
        seen = old;
        if (!(v < __uint_as_float(seen))) break;
        old = atomicCAS(a, seen, __float_as_uint(v));
    } while (old != seen);
}
FDB_DEVICE void fdb_atomic_max(float *p, float v)
{
    unsigned int *a = (unsigned int *)p, old = *a, seen;
    do {
        seen = old;
        if (!(v > __uint_as_float(seen))) break;
        old = atomicCAS(a, seen, __float_as_uint(v));
    } while (old != seen);
}

// ---- Global reductions (pyop2/parloop.py:516-532 privatises INC globals; here the
// private copy is a thread's, combined across the warp before one atomic).
// Every lane of the warp calls these (inactive lanes pass the identity).
template <class T> FDB_DEVICE T fdb_shfl_down(T v, int o) { return __shfl_down_sync(0xffffffffu, v, o); }
template <class T> FDB_DEVICE void fdb_reduce_add(T *g, T v, bool active)
{
    if (!active) v = (T)0;
    for (int o = 16; o > 0; o >>= 1) v += fdb_shfl_down(v, o);
    if ((threadIdx.x & 31) == 0) fdb_atomic_add(g, v);
}
template <class T> FDB_DEVICE void fdb_reduce_min(T *g, T v, bool active)
{
    const unsigned m = __ballot_sync(0xffffffffu, active);
    if (m == 0) return;
    const int src = __ffs(m) - 1;
    const T first = __shfl_sync(0xffffffffu, v, src);
    if (!active) v = first;
    for (int o = 16; o > 0; o >>= 1) { T w = fdb_shfl_down(v, o); v = w < v ? w : v; }
    if ((threadIdx.x & 31) == 0) fdb_atomic_min(g, v);
}
template <class T> FDB_DEVICE void fdb_reduce_max(T *g, T v, bool active)
{
    const unsigned m = __ballot_sync(0xffffffffu, active);
    if (m == 0) return;
    const int src = __ffs(m) - 1;
    const T first = __shfl_sync(0xffffffffu, v, src);
    if (!active) v = first;
    for (int o = 16; o > 0; o >>= 1) { T w = fdb_shfl_down(v, o); v = w > v ? w : v; }
    if ((threadIdx.x & 31) == 0) fdb_atomic_max(g, v);
}

// ---- MatSetValues[Blocked]Local (A6): node row/column + component -> CSR slot by
// binary search in the (sorted) row; entries whose lgmap index is negative are
// dropped (masked lgmaps = Dirichlet rows/columns), as PETSc does.
FDB_DEVICE void fdb_mat_set(const FdbMatView &m, int rnode, int a, int cnode, int b, double v, int insert)
{
    if (m.row_lg && m.row_lg[(long long)rnode * m.bs_r + a] < 0) return;
    if (m.col_lg && m.col_lg[(long long)cnode * m.bs_c + b] < 0) return;
    long long lo = m.rowptr[rnode], hi = m.rowptr[rnode + 1];
    if (hi <= lo) return;
    while (hi - lo > 1) {
        const long long mid = (lo + hi) >> 1;
        if (m.colidx[mid] <= cnode) lo = mid; else hi = mid;
    }
    if (m.colidx[lo] != cnode) return;
    double *dst = m.vals + (lo * m.bs_r + a) * m.bs_c + b;
    if (insert) *dst = v; else atomicAdd(dst, v);
}

#define FDB_ENTRY(NAME, BODY)                                                         \
    extern "C" __global__ void __launch_bounds__(128) NAME(const FdbWrapParams p)     \
    {                                                                                 \
        BODY(p, (long long)blockIdx.x * blockDim.x + threadIdx.x);                    \
    }
)PRELUDE";

// Small dense linear algebra callable from local kernels: the `inverse` / `solve`
// entry points PyOP2 provides to Slate-generated kernels through LAPACK
// (pyop2/codegen/c/inverse.c:20-47, solve.c:20-51; SURVEY.md section 8f row f4).
// One matrix per thread = per iteration-set entry ("batched" over the parloop);
// row-major, partial pivoting.  Emitted only when the local kernel mentions them.
const char *kDenseLA = R"LA(
#define FDB_LA_MAX 32
/* Aout = A^{-1}, N x N row-major; Gauss-Jordan with partial pivoting */
FDB_DEVICE void inverse(double *Aout, const double *A, int N)
{
    if (N > FDB_LA_MAX) FDB_ABORT();
    int piv[FDB_LA_MAX];
    for (int i = 0; i < N * N; ++i) Aout[i] = A[i];
    for (int c = 0; c < N; ++c) {
        int p = c;
        double best = fabs(Aout[c * N + c]);
        for (int r = c + 1; r < N; ++r)
            if (fabs(Aout[r * N + c]) > best) { best = fabs(Aout[r * N + c]); p = r; }
        if (best == 0.0) FDB_ABORT();                  /* singular: the reference aborts too */
        piv[c] = p;
        if (p != c)
            for (int j = 0; j < N; ++j) { const double t = Aout[c * N + j]; Aout[c * N + j] = Aout[p * N + j]; Aout[p * N + j] = t; }
        const double d = 1.0 / Aout[c * N + c];
        Aout[c * N + c] = 1.0;
        for (int j = 0; j < N; ++j) Aout[c * N + j] *= d;
        for (int r = 0; r < N; ++r) {
            if (r == c) continue;
            const double f = Aout[r * N + c];
            Aout[r * N + c] = 0.0;
            for (int j = 0; j < N; ++j) Aout[r * N + j] -= f * Aout[c * N + j];
        }
    }
    for (int c = N - 1; c >= 0; --c)                   /* undo the row swaps on the columns */
        if (piv[c] != c)
            for (int r = 0; r < N; ++r) { const double t = Aout[r * N + c]; Aout[r * N + c] = Aout[r * N + piv[c]]; Aout[r * N + piv[c]] = t; }
}
/* out = A^{-1} B for one right-hand side, A row-major; LU with partial pivoting on a copy */
FDB_DEVICE void solve(double *out, const double *A, const double *B, int N)
{
    if (N > FDB_LA_MAX) FDB_ABORT();
    double W[FDB_LA_MAX * FDB_LA_MAX];
    for (int i = 0; i < N * N; ++i) W[i] = A[i];
    for (int i = 0; i < N; ++i) out[i] = B[i];
    for (int c = 0; c < N; ++c) {
        int p = c;
        double best = fabs(W[c * N + c]);
        for (int r = c + 1; r < N; ++r)
            if (fabs(W[r * N + c]) > best) { best = fabs(W[r * N + c]); p = r; }
        if (best == 0.0) FDB_ABORT();
        if (p != c) {
            for (int j = 0; j < N; ++j) { const double t = W[c * N + j]; W[c * N + j] = W[p * N + j]; W[p * N + j] = t; }
            const double t = out[c]; out[c] = out[p]; out[p] = t;
        }
        for (int r = c + 1; r < N; ++r) {
            const double f = W[r * N + c] / W[c * N + c];
            for (int j = c + 1; j < N; ++j) W[r * N + j] -= f * W[c * N + j];
            out[r] -= f * out[c];
        }
    }
    for (int r = N - 1; r >= 0; --r) {
        double v = out[r];
        for (int j = r + 1; j < N; ++j) v -= W[r * N + j] * out[j];
        out[r] = v / W[r * N + r];
    }
}
)LA";

bool mentions(const char *src, const char *word)
{
    const size_t n = strlen(word);
    for (const char *p = strstr(src, word); p; p = strstr(p + 1, word)) {
        const bool left = p == src || !(isalnum((unsigned char)p[-1]) || p[-1] == '_');
        const char *q = p + n;
        while (*q == ' ' || *q == '\t') q++;
        if (left && *q == '(') return true;
    }
    return false;
}

const char *ctype(int dt)
{
    switch (dt) {
    case FDB_F64: return "double";
    case FDB_F32: return "float";
    case FDB_I32: return "int";
    case FDB_U32: return "unsigned int";
    case FDB_I64: return "long long";
    }
    return nullptr;
}

size_t dtype_size(int dt)
{
    switch (dt) {
    case FDB_F64: case FDB_I64: return 8;
    case FDB_F32: case FDB_I32: case FDB_U32: return 4;
    }
    return 0;
}

bool valid_identifier(const char *s)
{
    if (!s || !*s) return false;
    if (!(isalpha((unsigned char)s[0]) || s[0] == '_')) return false;
    for (const char *c = s; *c; c++)
        if (!(isalnum((unsigned char)*c) || *c == '_')) return false;
    return strlen(s) < 200;
}

struct ArgInfo {
    fdb_wrapper_arg a;
    std::vector<int> off, off2, perm;
    int mat_slot = -1;
    int idx_r = -1, idx_c = -1;   // index-array ids (row / column for a Mat)
};

struct IndexSet {     // one materialised index array: map slot + offsets + permutation + f extent
    int map, arity, F;
    std::vector<int> off, perm, oq;     // oq: offset_quotient (periodic extrusion), empty = zeros
    bool same(const IndexSet &o) const
    {
        return map == o.map && arity == o.arity && F == o.F && off == o.off && perm == o.perm && oq == o.oq;
    }
};

struct Plan {
    std::string name;
    std::vector<ArgInfo> args;
    std::vector<IndexSet> idx;
    int extruded = 0, subset = 0, region = 0, nmaps = 0, nmats = 0, pass_layer = 0, periodic = 0, varlay = 0;
    // a direct Dat that is written from an extruded loop goes through a private copy
    bool private_direct(const fdb_wrapper_arg &a) const
    {
        return extruded && a.kind == FDB_ARG_DAT && a.map < 0 && a.access != FDB_READ;
    }
};

int validate(const fdb_wrapper_desc *d, Plan &pl)
{
    if (!d || !d->kernel_source || !d->args) {
        set_error("fdb_wrapper: NULL descriptor field");
        return 1;
    }
    if (!valid_identifier(d->kernel_name)) {
        set_error("fdb_wrapper: kernel_name is not a C identifier");
        return 1;
    }
    if (d->nargs < 1 || d->nargs > FDB_WRAP_MAX_ARGS) {
        set_error("fdb_wrapper: nargs %d outside 1..%d", d->nargs, FDB_WRAP_MAX_ARGS);
        return 1;
    }
    if (d->iteration_region < 0 || d->iteration_region > FDB_REGION_ON_INTERIOR_FACETS) {
        set_error("fdb_wrapper: unknown iteration region %d", d->iteration_region);
        return 1;
    }
    if (!d->extruded && d->iteration_region != FDB_REGION_ALL) {
        set_error("fdb_wrapper: iteration regions need an extruded set");
        return 1;
    }
    pl.name = d->kernel_name;
    pl.extruded = d->extruded ? 1 : 0;
    pl.subset = d->subset ? 1 : 0;
    pl.region = d->iteration_region;
    pl.pass_layer = d->pass_layer_arg ? 1 : 0;
    pl.periodic = (d->extruded && d->extruded_periodic) ? 1 : 0;
    pl.varlay = (d->extruded && d->variable_layers) ? 1 : 0;
    if (d->variable_layers && !d->extruded) {
        set_error("fdb_wrapper: variable_layers needs an extruded wrapper");
        return 1;
    }
    if (pl.varlay && pl.periodic) {
        set_error("fdb_wrapper: periodic extrusion has constant layers (pyop2/types/set.py ExtrudedSet)");
        return 1;
    }
    if (pl.pass_layer && !pl.extruded) {
        set_error("fdb_wrapper: pass_layer_arg needs an extruded set (pyop2/global_kernel.py:299-302)");
        return 1;
    }
    auto add_index = [&](int map, int arity, int F, const fdb_int *off, const fdb_int *perm,
                         const fdb_int *oq) -> int {
        IndexSet s;
        s.map = map;
        s.arity = arity;
        s.F = F;
        if (off && pl.extruded) s.off.assign(off, off + arity);
        if (oq && pl.extruded && pl.periodic) s.oq.assign(oq, oq + arity);
        if (perm) s.perm.assign(perm, perm + arity);
        for (size_t i = 0; i < pl.idx.size(); i++)
            if (pl.idx[i].same(s)) return (int)i;
        pl.idx.push_back(s);
        return (int)pl.idx.size() - 1;
    };
    for (int i = 0; i < d->nargs; i++) {
        ArgInfo ai;
        ai.a = d->args[i];
        const fdb_wrapper_arg &a = ai.a;
        const int F = a.interior_horizontal ? 2 : 1;
        if (a.interior_horizontal && !pl.extruded) {
            set_error("fdb_wrapper: arg %d: interior_horizontal needs an extruded set", i);
            return 1;
        }
        if (a.mixed_continuation) {
            // a MixedDat segment continues the previous wrapper argument's local tensor
            if (i == 0 || a.kind != FDB_ARG_DAT || a.map < 0 || d->args[i - 1].kind != FDB_ARG_DAT ||
                d->args[i - 1].map < 0 || d->args[i - 1].access != a.access || d->args[i - 1].dtype != a.dtype) {
                set_error("fdb_wrapper: arg %d: a MixedDat segment must follow an indirect Dat argument of the "
                          "same access and dtype", i);
                return 1;
            }
        }
        if (a.access < FDB_READ || a.access > FDB_MAX) {
            set_error("fdb_wrapper: arg %d: bad access %d", i, a.access);
            return 1;
        }
        if (a.kind == FDB_ARG_DAT) {
            if (!ctype(a.dtype) || a.dim < 1 || a.dim > 64) {
                set_error("fdb_wrapper: arg %d: bad dtype/dim", i);
                return 1;
            }
            if (a.map >= 0) {
                if (a.map >= FDB_WRAP_MAX_MAPS || a.arity < 1 || a.arity > 1024) {
                    set_error("fdb_wrapper: arg %d: map slot %d / arity %d out of range", i, a.map, a.arity);
                    return 1;
                }
                if (pl.extruded && !a.offset) {
                    set_error("fdb_wrapper: arg %d: extruded indirect Dat needs Map.offset", i);
                    return 1;
                }
                if (a.permutation)
                    for (int j = 0; j < a.arity; j++)
                        if (a.permutation[j] < 0 || a.permutation[j] >= a.arity) {
                            set_error("fdb_wrapper: arg %d: permutation entry out of range", i);
                            return 1;
                        }
                pl.nmaps = std::max(pl.nmaps, a.map + 1);
                ai.idx_r = add_index(a.map, a.arity, F, a.offset, a.permutation, a.offset_quotient);
            } else {
                // a direct Dat on an extruded set is indexed by the column only
                // (pyop2/codegen/builder.py:386-397): every layer of a column sees the same
                // entry, which is only race free for READ
                if (pl.extruded && a.access != FDB_READ && a.access != FDB_INC && a.access != FDB_WRITE) {
                    set_error("fdb_wrapper: arg %d: direct Dats on extruded sets are READ, INC or WRITE "
                              "(one entry per column, shared by the threads of all its layers: RW / MIN / "
                              "MAX would depend on the layer order)", i);
                    return 1;
                }
            }
        } else if (a.kind == FDB_ARG_GLOBAL) {
            if (!ctype(a.dtype) || a.dim < 1 || a.dim > 256) {
                set_error("fdb_wrapper: arg %d: bad Global dtype/dim", i);
                return 1;
            }
            if (a.access == FDB_WRITE || a.access == FDB_RW) {
                set_error("fdb_wrapper: arg %d: Globals are READ, INC, MIN or MAX "
                          "(pyop2/types/glob.py access check)", i);
                return 1;
            }
        } else if (a.kind == FDB_ARG_MAT) {
            if (a.access != FDB_INC && a.access != FDB_WRITE) {
                set_error("fdb_wrapper: arg %d: Mats are INC or WRITE (builder.py:558-563)", i);
                return 1;
            }
            if (a.map < 0 || a.map2 < 0 || a.map >= FDB_WRAP_MAX_MAPS || a.map2 >= FDB_WRAP_MAX_MAPS ||
                a.arity < 1 || a.arity2 < 1 || a.dim < 1 || a.dim2 < 1 || a.dim > 8 || a.dim2 > 8) {
                set_error("fdb_wrapper: arg %d: bad Mat maps / block sizes", i);
                return 1;
            }
            if ((long long)F * a.arity * a.dim * F * a.arity2 * a.dim2 > (1 << 16)) {
                set_error("fdb_wrapper: arg %d: element tensor too large for the generic path", i);
                return 1;
            }
            if (pl.extruded && (!a.offset || !a.offset2)) {
                set_error("fdb_wrapper: arg %d: extruded Mat needs both Map.offset arrays", i);
                return 1;
            }
            if (pl.nmats >= FDB_WRAP_MAX_MATS) {
                set_error("fdb_wrapper: more than %d Mat arguments", FDB_WRAP_MAX_MATS);
                return 1;
            }
            ai.mat_slot = pl.nmats++;
            pl.nmaps = std::max(pl.nmaps, std::max(a.map, a.map2) + 1);
            ai.idx_r = add_index(a.map, a.arity, F, a.offset, nullptr, a.offset_quotient);
            ai.idx_c = add_index(a.map2, a.arity2, F, a.offset2, nullptr, a.offset_quotient2);
        } else {
            set_error("fdb_wrapper: arg %d: unknown kind %d", i, a.kind);
            return 1;
        }
        if (a.offset && a.arity > 0) ai.off.assign(a.offset, a.offset + a.arity);
        if (a.offset2 && a.arity2 > 0) ai.off2.assign(a.offset2, a.offset2 + a.arity2);
        if (a.permutation && a.arity > 0) ai.perm.assign(a.permutation, a.permutation + a.arity);
        ai.a.offset = ai.a.offset2 = ai.a.permutation = nullptr;   // the copies above are the owners
        ai.a.offset_quotient = ai.a.offset_quotient2 = nullptr;     // (copied into the index sets)
        pl.args.push_back(ai);
    }
    return 0;
}

// the local kernel's source with preprocessor includes removed (there are no
// host headers under NVRTC; math functions and the fixed-width types are built in
// or predefined by the prelude)
std::string strip_includes(const char *src)
{
    std::istringstream in(src);
    std::ostringstream out;
    std::string line;
    while (std::getline(in, line)) {
        size_t p = line.find_first_not_of(" \t");
        if (p != std::string::npos && line.compare(p, 1, "#") == 0) {
            size_t q = line.find_first_not_of(" \t", p + 1);
            if (q != std::string::npos && line.compare(q, 7, "include") == 0) {
                out << "/* " << "include removed" << " */\n";
                continue;
            }
        }
        out << line << "\n";
    }
    return out.str();
}

void emit_int_table(std::ostringstream &o, const std::string &name, const std::vector<int> &v)
{
    o << "FDB_CONST int " << name << "[" << v.size() << "] = {";
    for (size_t i = 0; i < v.size(); i++) o << (i ? ", " : "") << v[i];
    o << "};\n";
}

std::string generate(const fdb_wrapper_desc *d, const Plan &pl)
{
    std::ostringstream o;
    o << kPrelude << "\n" << kPreludeEnd << "\n";
    if (mentions(d->kernel_source, "inverse") || mentions(d->kernel_source, "solve")) o << kDenseLA << "\n";
    o << "// ---- local kernel: " << pl.name << "\n";
    o << strip_includes(d->kernel_source) << "\n";
    o << "// ---- wrapper (generated): wrap_" << pl.name << "\n";
    // compile-time constants of the wrapper (pyop2/global_kernel.py:309-317): offsets, permutations
    for (size_t s = 0; s < pl.idx.size(); s++) {
        const IndexSet &is = pl.idx[s];
        if (!is.off.empty()) emit_int_table(o, "fdb_off" + std::to_string(s), is.off);
        if (!is.oq.empty()) emit_int_table(o, "fdb_oq" + std::to_string(s), is.oq);
        if (!is.perm.empty()) emit_int_table(o, "fdb_perm" + std::to_string(s), is.perm);
    }
    o << "FDB_DEVICE void wrap_" << pl.name << "_body(const FdbWrapParams &p, long long tid)\n{\n";
    if (pl.varlay) {
        // every column has its own extent; the grid is (entries) x (tallest column in the region),
        // threads above a column's top stay idle (pyop2/codegen/builder.py:754-812)
        o << "    const int nl = p.layer_hi - p.layer_lo;\n"
          << "    const long long total = (long long)(p.end - p.start) * (nl > 0 ? nl : 0);\n"
          << "    bool active = tid < total;\n"
          << "    const long long it = active ? tid / nl : 0;\n"
          << "    int n = p.start + (int)it;\n";
        if (pl.subset) o << "    if (active) n = p.subset[n];\n";
        o << "    const int fdb_cs = active ? p.col_layers[2 * (long long)n] : 0;\n"
          << "    const int fdb_ce = active ? p.col_layers[2 * (long long)n + 1] - 1 : 0;\n";
        switch (pl.region) {
        case FDB_REGION_ON_BOTTOM: o << "    const int fdb_lo = fdb_cs, fdb_hi = fdb_cs + 1;\n"; break;
        case FDB_REGION_ON_TOP: o << "    const int fdb_lo = fdb_ce - 1, fdb_hi = fdb_ce;\n"; break;
        case FDB_REGION_ON_INTERIOR_FACETS: o << "    const int fdb_lo = fdb_cs, fdb_hi = fdb_ce - 1;\n"; break;
        default: o << "    const int fdb_lo = fdb_cs, fdb_hi = fdb_ce;\n"; break;
        }
        o << "    const int layer = fdb_lo + (active ? (int)(tid - it * nl) : 0);\n"
          << "    active = active && layer < fdb_hi && layer >= fdb_cs && layer < fdb_ce;\n"
          << "    const int lrel = layer - fdb_cs;\n";
    } else if (pl.extruded) {
        o << "    const int nl = p.layer_hi - p.layer_lo;\n"
          << "    const long long total = (long long)(p.end - p.start) * (nl > 0 ? nl : 0);\n"
          << "    const bool active = tid < total;\n"
          << "    const long long it = active ? tid / nl : 0;\n"
          << "    const int layer = active ? p.layer_lo + (int)(tid - it * nl) : p.layer_lo;\n"
          << "    const int lrel = layer - p.bottom;\n";
    } else {
        o << "    const long long total = (long long)(p.end - p.start);\n"
          << "    const bool active = tid < total;\n"
          << "    const long long it = active ? tid : 0;\n";
    }
    if (!pl.varlay) {
        o << "    int n = p.start + (int)it;\n";
        if (pl.subset) o << "    if (active) n = p.subset[n];\n";
    }
    // MixedDat groups: a continuation segment shares the local tensor of its group head
    std::vector<int> ghead(pl.args.size()), goff(pl.args.size(), 0), gsize(pl.args.size(), 0);
    for (size_t i = 0; i < pl.args.size(); i++) {
        const fdb_wrapper_arg &a = pl.args[i].a;
        const int F = a.interior_horizontal ? 2 : 1;
        const int sz = (a.kind == FDB_ARG_DAT && a.map >= 0) ? F * a.arity * a.dim : 0;
        ghead[i] = (a.mixed_continuation && i > 0) ? ghead[i - 1] : (int)i;
        goff[i] = gsize[ghead[i]];
        gsize[ghead[i]] += sz;
    }
    auto tseg = [&](size_t i) {     // "t<head> + <offset>" of segment i
        return "(t" + std::to_string(ghead[i]) + " + " + std::to_string(goff[i]) + ")";
    };
    // declarations (function scope so that the reductions after the guarded block see them)
    for (size_t i = 0; i < pl.args.size(); i++) {
        const fdb_wrapper_arg &a = pl.args[i].a;
        const int F = a.interior_horizontal ? 2 : 1;
        if (a.kind == FDB_ARG_DAT && a.map >= 0) {
            if (ghead[i] == (int)i) o << "    " << ctype(a.dtype) << " t" << i << "[" << gsize[i] << "];\n";
        }
        else if (pl.private_direct(a))
            o << "    " << ctype(a.dtype) << " t" << i << "[" << a.dim << "];\n";
        else if (a.kind == FDB_ARG_GLOBAL && a.access != FDB_READ)
            o << "    " << ctype(a.dtype) << " t" << i << "[" << a.dim << "];\n";
        else if (a.kind == FDB_ARG_MAT)
            o << "    double t" << i << "[" << F * a.arity * a.dim * F * a.arity2 * a.dim2 << "];\n";
    }
    for (size_t s = 0; s < pl.idx.size(); s++)
        o << "    int ix" << s << "[" << pl.idx[s].F * pl.idx[s].arity << "];\n";
    // Global INC/MIN/MAX packs (all lanes: the reductions below are warp-collective)
    for (size_t i = 0; i < pl.args.size(); i++) {
        const fdb_wrapper_arg &a = pl.args[i].a;
        if (a.kind != FDB_ARG_GLOBAL || a.access == FDB_READ) continue;
        o << "    for (int d = 0; d < " << a.dim << "; ++d) t" << i << "[d] = ";
        if (a.access == FDB_INC)
            o << "(" << ctype(a.dtype) << ")0;\n";
        else
            o << "((const " << ctype(a.dtype) << " *)p.arg[" << i << "])[d];\n";
    }
    o << "    if (active) {\n";
    // index arrays: map[n][perm[i]] + offset[i] * (layer - bottom + f)
    for (size_t s = 0; s < pl.idx.size(); s++) {
        const IndexSet &is = pl.idx[s];
        o << "        for (int f = 0; f < " << is.F << "; ++f)\n"
          << "            for (int i = 0; i < " << is.arity << "; ++i)\n"
          << "                ix" << s << "[f * " << is.arity << " + i] = p.map[" << is.map
          << "][(long long)n * " << is.arity << " + ";
        if (!is.perm.empty()) o << "fdb_perm" << s << "[i]"; else o << "i";
        o << "]";
        if (!is.off.empty()) {
            if (!pl.periodic)
                o << " + fdb_off" << s << "[i] * (lrel + f)";
            else if (is.oq.empty())      // periodic, offset_quotient == 0 (builder.py:108-111)
                o << " + fdb_off" << s << "[i] * ((lrel + f) % p.ncl)";
            else                         // builder.py:112-119
                o << " + fdb_off" << s << "[i] * ((lrel + f + fdb_oq" << s << "[i]) % p.ncl - fdb_oq" << s
                  << "[i] % p.ncl)";
        }
        o << ";\n";
    }
    // packs
    for (size_t i = 0; i < pl.args.size(); i++) {
        const ArgInfo &ai = pl.args[i];
        const fdb_wrapper_arg &a = ai.a;
        const int F = a.interior_horizontal ? 2 : 1;
        if (a.kind == FDB_ARG_DAT && a.map >= 0) {
            const bool reads = a.access == FDB_READ || a.access == FDB_RW || a.access == FDB_MIN ||
                               a.access == FDB_MAX;
            o << "        for (int k = 0; k < " << F * a.arity << "; ++k)\n"
              << "            for (int c = 0; c < " << a.dim << "; ++c)\n"
              << "                " << tseg(i) << "[k * " << a.dim << " + c] = ";
            if (reads)
                o << "((const " << ctype(a.dtype) << " *)p.arg[" << i << "])[(long long)ix" << ai.idx_r
                  << "[k] * " << a.dim << " + c];\n";
            else
                o << "(" << ctype(a.dtype) << ")0;\n";
        } else if (a.kind == FDB_ARG_MAT) {
            o << "        for (int k = 0; k < " << F * a.arity * a.dim * F * a.arity2 * a.dim2 << "; ++k) t" << i
              << "[k] = 0.0;\n";
        } else if (pl.private_direct(a)) {
            o << "        for (int c = 0; c < " << a.dim << "; ++c) t" << i << "[c] = (" << ctype(a.dtype) << ")0;\n";
        }
    }
    // the local kernel
    o << "        " << pl.name << "(";
    bool first_kernel_arg = true;
    for (size_t i = 0; i < pl.args.size(); i++) {
        const fdb_wrapper_arg &a = pl.args[i].a;
        if (ghead[i] != (int)i) continue;            // continuation segment of a MixedDat: no own pointer
        if (!first_kernel_arg) o << ", ";
        first_kernel_arg = false;
        if (a.kind == FDB_ARG_DAT && a.map < 0 && !pl.private_direct(a))
            o << "((" << ctype(a.dtype) << " *)p.arg[" << i << "]) + (long long)n * " << a.dim;
        else if (a.kind == FDB_ARG_GLOBAL && a.access == FDB_READ)
            o << "(" << ctype(a.dtype) << " *)p.arg[" << i << "]";
        else
            o << "t" << i;
    }
    if (pl.pass_layer) o << ", layer";
    o << ");\n";
    // unpacks
    for (size_t i = 0; i < pl.args.size(); i++) {
        const ArgInfo &ai = pl.args[i];
        const fdb_wrapper_arg &a = ai.a;
        const int F = a.interior_horizontal ? 2 : 1;
        if (a.kind == FDB_ARG_DAT && a.map >= 0 && a.access != FDB_READ) {
            o << "        for (int k = 0; k < " << F * a.arity << "; ++k)\n"
              << "            for (int c = 0; c < " << a.dim << "; ++c) {\n"
              << "                " << ctype(a.dtype) << " *dst = ((" << ctype(a.dtype) << " *)p.arg[" << i
              << "]) + (long long)ix" << ai.idx_r << "[k] * " << a.dim << " + c;\n"
              << "                const " << ctype(a.dtype) << " v = " << tseg(i) << "[k * " << a.dim << " + c];\n";
            switch (a.access) {
            case FDB_INC: o << "                fdb_atomic_add(dst, v);\n"; break;
            case FDB_MIN: o << "                fdb_atomic_min(dst, v);\n"; break;
            case FDB_MAX: o << "                fdb_atomic_max(dst, v);\n"; break;
            default: o << "                *dst = v;\n"; break;
            }
            o << "            }\n";
        } else if (pl.private_direct(a)) {
            o << "        for (int c = 0; c < " << a.dim << "; ++c) {\n"
              << "            " << ctype(a.dtype) << " *dst = ((" << ctype(a.dtype) << " *)p.arg[" << i
              << "]) + (long long)n * " << a.dim << " + c;\n";
            if (a.access == FDB_INC) o << "            fdb_atomic_add(dst, t" << i << "[c]);\n";
            else o << "            *dst = t" << i << "[c];\n";
            o << "        }\n";
        } else if (a.kind == FDB_ARG_MAT) {
            const int nr = F * a.arity, nc = F * a.arity2;
            o << "        for (int r = 0; r < " << nr << "; ++r)\n"
              << "            for (int a = 0; a < " << a.dim << "; ++a)\n"
              << "                for (int c = 0; c < " << nc << "; ++c)\n"
              << "                    for (int b = 0; b < " << a.dim2 << "; ++b)\n"
              << "                        fdb_mat_set(p.mat[" << ai.mat_slot << "], ix" << ai.idx_r << "[r], a, ix"
              << ai.idx_c << "[c], b, t" << i << "[((r * " << a.dim << " + a) * " << nc << " + c) * " << a.dim2
              << " + b], " << (a.access == FDB_WRITE ? 1 : 0) << ");\n";
        }
    }
    o << "    }\n";
    // Global reductions
    for (size_t i = 0; i < pl.args.size(); i++) {
        const fdb_wrapper_arg &a = pl.args[i].a;
        if (a.kind != FDB_ARG_GLOBAL || a.access == FDB_READ) continue;
        const char *fn = a.access == FDB_INC ? "fdb_reduce_add" : (a.access == FDB_MIN ? "fdb_reduce_min" : "fdb_reduce_max");
        o << "    for (int d = 0; d < " << a.dim << "; ++d) " << fn << "(((" << ctype(a.dtype) << " *)p.arg[" << i
          << "]) + d, t" << i << "[d], active);\n";
    }
    o << "}\n";
    o << "FDB_ENTRY(wrap_" << pl.name << ", wrap_" << pl.name << "_body)\n";
    return o.str();
}

// ---------------------------------------------------------------------------
// NVRTC through dlopen (like NCCL in halo.cu: no link-time dependency)
typedef struct _nvrtcProgram *nvrtcProgram;
struct Nvrtc {
    void *h = nullptr;
    int (*CreateProgram)(nvrtcProgram *, const char *, const char *, int, const char *const *, const char *const *);
    int (*CompileProgram)(nvrtcProgram, int, const char *const *);
    int (*GetProgramLogSize)(nvrtcProgram, size_t *);
    int (*GetProgramLog)(nvrtcProgram, char *);
    int (*GetCUBINSize)(nvrtcProgram, size_t *);
    int (*GetCUBIN)(nvrtcProgram, char *);
    int (*DestroyProgram)(nvrtcProgram *);
    const char *(*GetErrorString)(int);
};

Nvrtc *nvrtc()
{
    static Nvrtc n;
    static bool tried = false;
    if (tried) return n.h ? &n : nullptr;
    tried = true;
    const char *names[] = {getenv("FDB200_NVRTC"), "libnvrtc.so.12", "libnvrtc.so",
                           "/usr/local/cuda/lib64/libnvrtc.so.12", "/usr/local/cuda/lib64/libnvrtc.so"};
    for (const char *nm : names) {
        if (!nm || !*nm) continue;
        n.h = dlopen(nm, RTLD_NOW | RTLD_LOCAL);
        if (n.h) break;
    }
    if (!n.h) {
        set_error("fdb_wrapper: libnvrtc not found (set FDB200_NVRTC): %s", dlerror());
        return nullptr;
    }
#define SYM(f)                                                      \
    *(void **)(&n.f) = dlsym(n.h, "nvrtc" #f);                      \
    if (!n.f) {                                                     \
        set_error("fdb_wrapper: libnvrtc lacks nvrtc" #f);          \
        dlclose(n.h);                                               \
        n.h = nullptr;                                              \
        return nullptr;                                             \
    }
    SYM(CreateProgram) SYM(CompileProgram) SYM(GetProgramLogSize) SYM(GetProgramLog) SYM(GetCUBINSize)
    SYM(GetCUBIN) SYM(DestroyProgram) SYM(GetErrorString)
#undef SYM
    return &n;
}

int compile_cubin(const std::string &src, const std::string &name, std::vector<char> &cubin)
{
    Nvrtc *n = nvrtc();
    if (!n) return 1;
    nvrtcProgram prog = nullptr;
    int rc = n->CreateProgram(&prog, src.c_str(), ("wrap_" + name + ".cu").c_str(), 0, nullptr, nullptr);
    if (rc) {
        set_error("nvrtcCreateProgram: %s", n->GetErrorString(rc));
        return 1;
    }
    // -default-device: functions without an execution-space specifier (the local
    // kernel, written as plain C) are __device__ functions
    const char *opts[] = {"--gpu-architecture=sm_100a", "-default-device", "--std=c++17", "-lineinfo",
                          "--fmad=true"};
    rc = n->CompileProgram(prog, (int)(sizeof(opts) / sizeof(opts[0])), opts);
    if (rc) {
        size_t ls = 0;
        n->GetProgramLogSize(prog, &ls);
        std::string log(ls + 1, '\0');
        if (ls) n->GetProgramLog(prog, &log[0]);
        if (log.size() > 3500) log.resize(3500);
        set_error("NVRTC failed to compile wrap_%s (%s):\n%s", name.c_str(), n->GetErrorString(rc), log.c_str());
        n->DestroyProgram(&prog);
        return 1;
    }
    size_t sz = 0;
    rc = n->GetCUBINSize(prog, &sz);
    if (rc || sz == 0) {
        set_error("nvrtcGetCUBINSize: %s", rc ? n->GetErrorString(rc) : "empty image");
        n->DestroyProgram(&prog);
        return 1;
    }
    cubin.resize(sz);
    rc = n->GetCUBIN(prog, cubin.data());
    n->DestroyProgram(&prog);
    if (rc) {
        set_error("nvrtcGetCUBIN: %s", n->GetErrorString(rc));
        return 1;
    }
    return 0;
}

}  // namespace

// the loaded kernel behind a fdb_kernel_s created by fdb_wrapper_create
struct fdb_jit_s {
    Plan plan;
    std::string source;
    cudaLibrary_t lib = nullptr;
    cudaKernel_t fn = nullptr;
    char *d_globals = nullptr;        // device copies of the Global arguments
    std::vector<size_t> gofs;         // byte offset per arg (Globals only)
    size_t gbytes = 0;
    std::vector<char> h_globals;      // staging
    // variable layers: tallest column of the last layers array seen
    const fdb_int *lay_ptr = nullptr;
    uint64_t lay_ver = 0;
    fdb_int lay_cnt = 0;
    int lay_max = 0;
};

void fdb_jit_destroy(fdb_jit_s *j)
{
    if (!j) return;
    if (ctx().ready) {
        if (j->lib) cudaLibraryUnload(j->lib);
        if (j->d_globals) cudaFree(j->d_globals);
    }
    delete j;
}

int fdb_jit_call(fdb_kernel_s *k, const fdb_call_args *a)
{
    fdb_jit_s *j = k->jit;
    const Plan &pl = j->plan;
    if (a->nargs != (int)pl.args.size() || a->nmaps < pl.nmaps) {
        set_error("wrap_%s: expected %d args and >= %d maps, got %d / %d", pl.name.c_str(), (int)pl.args.size(),
                  pl.nmaps, a->nargs, a->nmaps);
        return 1;
    }
    if (a->end < a->start) {
        set_error("wrap_%s: end < start", pl.name.c_str());
        return 1;
    }
    if (pl.extruded && !a->layers) {
        set_error("wrap_%s: extruded wrapper called without layers", pl.name.c_str());
        return 1;
    }
    if (pl.subset && !a->subset) {
        set_error("wrap_%s: wrapper was generated for a Subset but none was passed", pl.name.c_str());
        return 1;
    }
    const bool host = a->location == FDB_LOC_HOST;
    if (host && (!a->arg_bytes || !a->map_bytes)) {
        set_error("wrap_%s: host mode needs arg_bytes and map_bytes", pl.name.c_str());
        return 1;
    }
    cudaStream_t st = ctx().stream;
    FdbWrapParams p;
    memset(&p, 0, sizeof(p));
    p.start = a->start;
    p.end = a->end;
    int nl = 1;
    if (pl.varlay) {
        if (a->layers_count < a->end && !pl.subset) {
            set_error("wrap_%s: variable layers: %d rows of layers for an iteration range ending at %d",
                      pl.name.c_str(), (int)a->layers_count, (int)a->end);
            return 1;
        }
        // tallest column in the iteration region: the layer extent of the launch grid
        if (j->lay_ptr != a->layers || j->lay_ver != a->layers_version || j->lay_cnt != a->layers_count) {
            int mx = 0;
            for (fdb_int c = 0; c < a->layers_count; c++) {
                const int cs = a->layers[2 * c], ce = a->layers[2 * c + 1] - 1;
                int ext;
                switch (pl.region) {
                case FDB_REGION_ON_BOTTOM: case FDB_REGION_ON_TOP: ext = ce > cs ? 1 : 0; break;
                case FDB_REGION_ON_INTERIOR_FACETS: ext = ce - 1 - cs; break;
                default: ext = ce - cs; break;
                }
                if (ext > mx) mx = ext;
            }
            j->lay_ptr = a->layers; j->lay_ver = a->layers_version; j->lay_cnt = a->layers_count; j->lay_max = mx;
        }
        void *q;
        if (fdb_mirror_acquire(a->layers, sizeof(fdb_int) * 2 * (size_t)a->layers_count, a->layers_version, 1, &q))
            return 1;
        p.col_layers = (const int *)q;
        p.layer_lo = 0;
        p.layer_hi = nl = j->lay_max;
        p.ncl = 1;
    } else if (pl.extruded) {
        // layer extents by iteration region (pyop2/codegen/builder.py:790-812); layers[] counts
        // NODE layers, so cells are [layers[0], layers[1]-1)
        const int cs = a->layers[0], ce = a->layers[1] - 1;
        p.bottom = cs;
        p.ncl = ce - cs > 0 ? ce - cs : 1;
        switch (pl.region) {
        case FDB_REGION_ON_BOTTOM: p.layer_lo = cs; p.layer_hi = cs + 1; break;
        case FDB_REGION_ON_TOP: p.layer_lo = ce - 1; p.layer_hi = ce; break;
        // a periodic column also has the facet between its top and bottom cells: the
        // last layer's "above" cell wraps round to the bottom through the % p.ncl of the
        // map index (tests/test_wrapper_semantics.py, periodic ON_INTERIOR_FACETS cases)
        case FDB_REGION_ON_INTERIOR_FACETS: p.layer_lo = cs; p.layer_hi = pl.periodic ? ce : ce - 1; break;
        default: p.layer_lo = cs; p.layer_hi = ce; break;
        }
        nl = p.layer_hi - p.layer_lo;
        if (nl < 0) nl = 0;
    }
    const long long total = (long long)(a->end - a->start) * nl;
    if (total >= (1ll << 31) * 128) {
        set_error("wrap_%s: iteration space too large", pl.name.c_str());
        return 1;
    }
    // maps and subset
    for (int m = 0; m < pl.nmaps; m++) {
        if (host) {
            void *q;
            if (fdb_mirror_acquire(a->maps[m], a->map_bytes[m], a->map_versions ? a->map_versions[m] : 0, 1, &q)) return 1;
            p.map[m] = (const int *)q;
        } else {
            p.map[m] = a->maps[m];
        }
    }
    if (pl.subset) {
        if (host) {
            void *q;
            if (fdb_mirror_acquire(a->subset, sizeof(fdb_int) * (size_t)a->end, a->subset_version, 1, &q)) return 1;
            p.subset = (const int *)q;
        } else {
            p.subset = a->subset;
        }
    }
    // arguments
    bool any_global_out = false;
    for (size_t i = 0; i < pl.args.size(); i++) {
        const fdb_wrapper_arg &wa = pl.args[i].a;
        if (wa.kind == FDB_ARG_DAT) {
            if (host) {
                const uint64_t ver = a->arg_versions ? a->arg_versions[i] : 0;
                if (!a->arg_versions) fdb_mirror_drop(a->args[i]);
                const bool zero = (i == 0 && a->output_is_zero && wa.access == FDB_INC);
                void *q;
                if (fdb_mirror_acquire(a->args[i], a->arg_bytes[i], ver, zero ? 0 : 1, &q)) return 1;
                if (zero) FDB_CUDA(cudaMemsetAsync(q, 0, a->arg_bytes[i], st));
                p.arg[i] = q;
            } else {
                p.arg[i] = a->args[i];
            }
        } else if (wa.kind == FDB_ARG_GLOBAL) {
            // Globals always arrive as HOST pointers; a device copy lives in d_globals
            const size_t nb = dtype_size(wa.dtype) * wa.dim;
            memcpy(j->h_globals.data() + j->gofs[i], a->args[i], nb);
            p.arg[i] = j->d_globals + j->gofs[i];
            if (wa.access != FDB_READ) any_global_out = true;
        } else {
            fdb_mat_t m = (fdb_mat_t)a->args[i];
            FdbMatView &v = p.mat[pl.args[i].mat_slot];
            int bs = 1;
            if (fdb_mat_device_view(m, &v.rowptr, &v.colidx, &v.vals, &v.row_lg, &v.col_lg)) return 1;
            fdb_mat_block_size(m, &bs);
            v.bs_r = v.bs_c = bs;
            if (bs != wa.dim || bs != wa.dim2) {
                set_error("wrap_%s: arg %d: Mat block size %d != wrapper's (%d, %d)", pl.name.c_str(), (int)i, bs,
                          wa.dim, wa.dim2);
                return 1;
            }
        }
    }
    if (j->gbytes)
        FDB_CUDA(cudaMemcpyAsync(j->d_globals, j->h_globals.data(), j->gbytes, cudaMemcpyHostToDevice, st));
    if (total > 0) {
        const unsigned block = 128;
        const unsigned grid = (unsigned)((total + block - 1) / block);
        void *kargs[] = {&p};
        FDB_CUDA(cudaLaunchKernel((const void *)j->fn, dim3(grid), dim3(block), kargs, 0, st));
        FDB_LAUNCH_CHECK();
    }
    if (any_global_out) {
        // reductions return through the host Global (the caller's Iallreduce across ranks,
        // pyop2/parloop.py:411-442, follows on these values)
        FDB_CUDA(cudaMemcpyAsync(j->h_globals.data(), j->d_globals, j->gbytes, cudaMemcpyDeviceToHost, st));
        FDB_CUDA(cudaStreamSynchronize(st));
        for (size_t i = 0; i < pl.args.size(); i++) {
            const fdb_wrapper_arg &wa = pl.args[i].a;
            if (wa.kind == FDB_ARG_GLOBAL && wa.access != FDB_READ)
                memcpy(a->args[i], j->h_globals.data() + j->gofs[i], dtype_size(wa.dtype) * wa.dim);
        }
    }
    if (host && a->writeback) {
        for (size_t i = 0; i < pl.args.size(); i++) {
            const fdb_wrapper_arg &wa = pl.args[i].a;
            if (wa.kind != FDB_ARG_DAT || wa.access == FDB_READ) continue;
            if (fdb_mirror_writeback(a->args[i])) return 1;
            if (a->arg_versions) fdb_mirror_set_version(a->args[i], a->arg_versions[i] + 1);
        }
    }
    return 0;
}

extern "C" {

int fdb_wrapper_source(const fdb_wrapper_desc *d, char *buf, size_t cap, size_t *needed)
{
    Plan pl;
    if (validate(d, pl)) return 1;
    const std::string s = generate(d, pl);
    if (needed) *needed = s.size() + 1;
    if (buf && cap) {
        const size_t n = s.size() + 1 <= cap ? s.size() : cap - 1;
        memcpy(buf, s.data(), n);
        buf[n] = '\0';
    }
    return 0;
}

int fdb_wrapper_compile(const fdb_wrapper_desc *d, void *cubin, size_t cap, size_t *needed)
{
    Plan pl;
    if (validate(d, pl)) return 1;
    const std::string s = generate(d, pl);
    std::vector<char> img;
    if (compile_cubin(s, pl.name, img)) return 1;
    if (needed) *needed = img.size();
    if (cubin && cap >= img.size()) memcpy(cubin, img.data(), img.size());
    return 0;
}

int fdb_wrapper_create(const fdb_wrapper_desc *d, fdb_kernel_t *out)
{
    if (require_init()) return 1;
    if (!out) {
        set_error("fdb_wrapper_create: NULL out");
        return 1;
    }
    fdb_jit_s *j = new fdb_jit_s;
    if (validate(d, j->plan)) {
        delete j;
        return 1;
    }
    j->source = generate(d, j->plan);
    std::vector<char> img;
    if (compile_cubin(j->source, j->plan.name, img)) {
        delete j;
        return 1;
    }
    cudaError_t e = cudaLibraryLoadData(&j->lib, img.data(), nullptr, nullptr, 0, nullptr, nullptr, 0);
    if (e != cudaSuccess) {
        set_error("cudaLibraryLoadData(wrap_%s): %s", j->plan.name.c_str(), cudaGetErrorString(e));
        delete j;
        return 1;
    }
    e = cudaLibraryGetKernel(&j->fn, j->lib, ("wrap_" + j->plan.name).c_str());
    if (e != cudaSuccess) {
        set_error("cudaLibraryGetKernel(wrap_%s): %s", j->plan.name.c_str(), cudaGetErrorString(e));
        cudaLibraryUnload(j->lib);
        delete j;
        return 1;
    }
    // device staging for Globals
    j->gofs.assign(j->plan.args.size(), 0);
    size_t ofs = 0;
    for (size_t i = 0; i < j->plan.args.size(); i++) {
        const fdb_wrapper_arg &wa = j->plan.args[i].a;
        if (wa.kind != FDB_ARG_GLOBAL) continue;
        j->gofs[i] = ofs;
        ofs += (dtype_size(wa.dtype) * wa.dim + 15) & ~(size_t)15;
    }
    j->gbytes = ofs;
    if (ofs) {
        j->h_globals.assign(ofs, 0);
        if (cudaMalloc(&j->d_globals, ofs) != cudaSuccess) {
            set_error("fdb_wrapper_create: cudaMalloc of the Global staging failed");
            cudaLibraryUnload(j->lib);
            delete j;
            return 1;
        }
    }
    fdb_kernel_s *k = new fdb_kernel_s;
    memset(&k->desc, 0, sizeof(k->desc));
    k->n1d = 0;
    k->arity = 0;
    k->jit = j;
    *out = k;
    return 0;
}

}  // extern "C"
