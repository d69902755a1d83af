// "Compile" and call of a global kernel: the replacement for
// pyop2.global_kernel.compile_global_kernel + GlobalKernel.__call__
// (reference pyop2/global_kernel.py:327-335, 426-456).  fdb_kernel_create compiles
// nothing: it validates the descriptor against the set of hand-written sm_100a
// kernels and precomputes the tables they need.  Handles made by
// fdb_wrapper_create (wrapper_jit.cu: NVRTC wrapper around an arbitrary local
// kernel) are dispatched from fdb_kernel_call as well.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "common.cuh"

using namespace fdb;

namespace {

// Dt = D * B^{-1}  (collocated derivative on the quadrature points).
// Solves X B = D by Gaussian elimination with partial pivoting on B^T X^T = D^T.
int collocated_derivative(int n, const double *B, const double *D, double *Dt)
{
    double A[FDB_MAX_1D][FDB_MAX_1D], R[FDB_MAX_1D][FDB_MAX_1D];
    for (int i = 0; i < n; i++)
        for (int j = 0; j < n; j++) {
            A[i][j] = B[j * n + i];   // B^T
            R[i][j] = D[j * n + i];   // D^T
        }
    for (int c = 0; c < n; c++) {
        int piv = c;
        for (int r = c + 1; r < n; r++)
            if (fabs(A[r][c]) > fabs(A[piv][c])) piv = r;
        if (fabs(A[piv][c]) < 1e-14) return 1;
        if (piv != c)
            for (int j = 0; j < n; j++) {
                std::swap(A[piv][j], A[c][j]);
                std::swap(R[piv][j], R[c][j]);
            }
        for (int r = 0; r < n; r++) {
            if (r == c) continue;
            double f = A[r][c] / A[c][c];
            for (int j = 0; j < n; j++) {
                A[r][j] -= f * A[c][j];
                R[r][j] -= f * R[c][j];
            }
        }
    }
    for (int i = 0; i < n; i++)
        for (int j = 0; j < n; j++) Dt[j * n + i] = R[i][j] / A[i][i];   // X = (X^T)^T
    return 0;
}

// Greedy colouring of columns (base cells) so that no two columns of one
// colour share a dof column: the deterministic fallback of the north_star
// ("warp-aggregated atomic kernel with a colouring fallback").  Host side,
// once per map.
int build_colouring(fdb_kernel_s *k, const fdb_int *h_map, fdb_int ncols)
{
    const int arity = k->arity;
    fdb_int maxnode = 0;
    for (long long i = 0; i < (long long)ncols * arity; i++) maxnode = std::max(maxnode, h_map[i]);
    // node -> bitmask of colours already used by a column touching it
    std::vector<uint64_t> used((size_t)maxnode + 1, 0);
    std::vector<int> colour(ncols);
    int ncolours = 0;
    for (fdb_int c = 0; c < ncols; c++) {
        uint64_t m = 0;
        for (int i = 0; i < arity; i++) m |= used[h_map[(size_t)c * arity + i]];
        int col = 0;
        while (col < 64 && (m >> col) & 1) col++;
        if (col >= 64) {
            set_error("colouring needs more than 64 colours");
            return 1;
        }
        colour[c] = col;
        ncolours = std::max(ncolours, col + 1);
        for (int i = 0; i < arity; i++) used[h_map[(size_t)c * arity + i]] |= (uint64_t)1 << col;
    }
    std::vector<fdb_int> sorted(ncols);
    int pos = 0;
    for (int col = 0; col < ncolours; col++) {
        k->colour_start[col] = pos;
        for (fdb_int c = 0; c < ncols; c++)
            if (colour[c] == col) sorted[pos++] = c;
    }
    k->colour_start[ncolours] = pos;
    k->ncolours = ncolours;
    if (k->d_colour_cols) cudaFree(k->d_colour_cols);
    FDB_CUDA(cudaMalloc(&k->d_colour_cols, sizeof(fdb_int) * std::max(ncols, 1)));
    FDB_CUDA(cudaMemcpyAsync(k->d_colour_cols, sorted.data(), sizeof(fdb_int) * ncols,
                             cudaMemcpyHostToDevice, ctx().stream));
    FDB_CUDA(cudaStreamSynchronize(ctx().stream));
    return 0;
}

// Drop-in (host pointer) call of a 1-form with the output just zeroed by the
// assembler: instead of "upload x, compute, download y" back to back, the
// iteration range is cut into chunks of columns and three streams overlap
//     H2D of the x rows chunk k+1 needs  |  kernel on chunk k  |  D2H of the
//     y rows no later chunk can touch
// (PCIe is full duplex, so the end-to-end time tends to max(H2D, D2H) instead
// of their sum).  Which rows a chunk touches is read off the map on the host:
// with Firedrake's cell-closure numbering the touched range grows monotonically
// with the chunk index; for an arbitrary numbering the schedule degenerates to
// the monolithic one by construction (everything uploaded before chunk 0,
// downloaded after the last), never to a wrong one.
static inline uint64_t map_ver(const fdb_call_args *a, int i)
{
    return a->map_versions ? a->map_versions[i] : 0;
}

struct PipelinePlan {
    const void *map_key = nullptr;
    uint64_t map_gen = 0;
    fdb_int start = 0, end = 0;
    int nlay = 0;
    std::vector<fdb_int> c0, c1;          // column range of each chunk
    std::vector<long long> upto;          // rows [0, upto[k]) must be resident before chunk k
    std::vector<long long> final_below;   // rows [0, final_below[k]) are final after chunk k
};
static PipelinePlan g_plan;
static cudaStream_t g_h2d = nullptr, g_d2h = nullptr;
static std::vector<cudaEvent_t> g_ev_up, g_ev_done;

static int pipelined_host_action(fdb_kernel_s *k, const fdb_call_args *a, int nlay)
{
    static const int nchunks_env = getenv("FDB_PIPELINE_CHUNKS") ? atoi(getenv("FDB_PIPELINE_CHUNKS")) : 32;
    const fdb_int ncols = a->end - a->start;
    int K = nchunks_env;
    if (K <= 1 || ncols < 64 * K) return -1;
    const int arity = k->arity;
    const size_t nrows = a->arg_bytes[0] / (sizeof(double) * k->desc.cdim);
    cudaStream_t st = ctx().stream;
    if (!g_h2d) {
        FDB_CUDA(cudaStreamCreateWithFlags(&g_h2d, cudaStreamNonBlocking));
        FDB_CUDA(cudaStreamCreateWithFlags(&g_d2h, cudaStreamNonBlocking));
    }
    while ((int)g_ev_up.size() < K) {
        cudaEvent_t e1, e2;
        FDB_CUDA(cudaEventCreateWithFlags(&e1, cudaEventDisableTiming));
        FDB_CUDA(cudaEventCreateWithFlags(&e2, cudaEventDisableTiming));
        g_ev_up.push_back(e1);
        g_ev_done.push_back(e2);
    }
    PipelinePlan &pl = g_plan;
    if (pl.map_key != (const void *)a->maps[0] || pl.map_gen != map_ver(a, 0) || pl.start != a->start ||
        pl.end != a->end ||
        pl.nlay != nlay || (int)pl.c0.size() != K) {
        // host analysis of the map (cached while the same map is passed)
        const fdb_int *map = a->maps[0];
        pl = PipelinePlan();
        pl.map_key = a->maps[0];
        pl.map_gen = map_ver(a, 0);
        pl.start = a->start;
        pl.end = a->end;
        pl.nlay = nlay;
        std::vector<long long> lo(K), hi(K);
        for (int c = 0; c < K; c++) {
            fdb_int b0 = a->start + (fdb_int)((long long)ncols * c / K);
            fdb_int b1 = a->start + (fdb_int)((long long)ncols * (c + 1) / K);
            pl.c0.push_back(b0);
            pl.c1.push_back(b1);
            long long l = (long long)nrows, h = 0;
            for (fdb_int col = b0; col < b1; col++)
                for (int i = 0; i < arity; i++) {
                    long long v = map[(size_t)col * arity + i];
                    long long top = v + (long long)k->h_off0[i] * (nlay - 1);
                    if (v < l) l = v;
                    if (top + 1 > h) h = top + 1;
                }
            lo[c] = l;
            hi[c] = h;
        }
        pl.upto.resize(K);
        pl.final_below.resize(K);
        long long m = 0;
        for (int c = 0; c < K; c++) {
            if (hi[c] > m) m = hi[c];
            pl.upto[c] = m;
        }
        long long mn = (long long)nrows;
        for (int c = K - 1; c >= 0; c--) {
            pl.final_below[c] = mn;          // min over later chunks of their lowest row
            if (lo[c] < mn) mn = lo[c];
        }
        pl.final_below[K - 1] = (long long)nrows;
    }
    void *dy, *dx, *dc, *dm0, *dm1;
    // static inputs through the mirror cache (uploaded once)
    if (fdb_mirror_acquire(a->args[1], a->arg_bytes[1], a->arg_versions[1], 1, &dc)) return 1;
    if (fdb_mirror_acquire(a->maps[0], a->map_bytes[0], map_ver(a, 0), 1, &dm0)) return 1;
    if (fdb_mirror_acquire(a->maps[1], a->map_bytes[1], map_ver(a, 1), 1, &dm1)) return 1;
    if (fdb_mirror_acquire(a->args[0], a->arg_bytes[0], a->arg_versions[0], 0, &dy)) return 1;
    bool x_current = fdb_mirror_is_current(a->args[2], a->arg_bytes[2], a->arg_versions[2]);
    if (fdb_mirror_acquire(a->args[2], a->arg_bytes[2], a->arg_versions[2], 0, &dx)) return 1;
    const size_t rowb = sizeof(double) * k->desc.cdim;
    // uploads wait for whatever the engine stream was doing with these buffers
    FDB_CUDA(cudaEventRecord(g_ev_done[0], st));
    FDB_CUDA(cudaStreamWaitEvent(g_h2d, g_ev_done[0], 0));
    FDB_CUDA(cudaStreamWaitEvent(g_d2h, g_ev_done[0], 0));
    // rows above the highest touched one: never gathered, must still read as zero
    if (pl.upto[K - 1] < (long long)nrows)
        FDB_CUDA(cudaMemsetAsync((char *)dy + pl.upto[K - 1] * rowb, 0,
                                 (size_t)((long long)nrows - pl.upto[K - 1]) * rowb, st));
    long long up_done = 0, down_done = 0;
    for (int c = 0; c < K; c++) {
        if (pl.upto[c] > up_done) {
            if (!x_current)
                FDB_CUDA(cudaMemcpyAsync((char *)dx + up_done * rowb, (const char *)a->args[2] + up_done * rowb,
                                         (size_t)(pl.upto[c] - up_done) * rowb, cudaMemcpyHostToDevice, g_h2d));
            FDB_CUDA(cudaMemsetAsync((char *)dy + up_done * rowb, 0, (size_t)(pl.upto[c] - up_done) * rowb, st));
            up_done = pl.upto[c];
        }
        FDB_CUDA(cudaEventRecord(g_ev_up[c], g_h2d));
        FDB_CUDA(cudaStreamWaitEvent(st, g_ev_up[c], 0));
        if (fdb_launch_helmholtz_action(k, pl.c0[c], pl.c1[c], nlay, nullptr, (double *)dy, (const double *)dc,
                                        (const double *)dx, (const fdb_int *)dm0, (const fdb_int *)dm1))
            return 1;
        FDB_CUDA(cudaEventRecord(g_ev_done[c], st));
        if (pl.final_below[c] > down_done) {
            FDB_CUDA(cudaStreamWaitEvent(g_d2h, g_ev_done[c], 0));
            FDB_CUDA(cudaMemcpyAsync((char *)a->args[0] + down_done * rowb, (const char *)dy + down_done * rowb,
                                     (size_t)(pl.final_below[c] - down_done) * rowb, cudaMemcpyDeviceToHost, g_d2h));
            down_done = pl.final_below[c];
        }
    }
    FDB_CUDA(cudaStreamSynchronize(g_d2h));
    FDB_CUDA(cudaStreamSynchronize(st));
    if (up_done == (long long)nrows) fdb_mirror_set_version(a->args[2], a->arg_versions[2]);
    fdb_mirror_set_version(a->args[0], a->arg_versions[0] + 1);
    return 0;
}

}  // namespace

extern "C" {

int fdb_kernel_create(const fdb_kernel_desc *d, fdb_kernel_t *out)
{
    if (require_init()) return 1;
    if (!d || !out) {
        set_error("fdb_kernel_create: NULL argument");
        return 1;
    }
    if (d->form == FDB_FORM_DG_ADVECTION) {
        if (d->cell != FDB_CELL_QUAD || d->rank != 1 || d->degree != 1 || d->cdim != 1 ||
            d->nq < 1 || d->nq > FDB_MAX_1D || d->integral < 0 || d->integral > FDB_INTEGRAL_FUSED) {
            set_error("fdb_kernel_create: DG advection is DQ1 on quads, rank 1, nq <= %d", FDB_MAX_1D);
            return 1;
        }
        fdb_kernel_s *k = new fdb_kernel_s;
        k->desc = *d;
        k->n1d = 2;
        k->arity = d->integral == FDB_INTEGRAL_INTERIOR_FACET ? 8 : 4;
        k->desc.offset0 = k->desc.offset1 = nullptr;
        *out = k;
        return 0;
    }
    if (d->form == FDB_FORM_HELMHOLTZ && d->cell == FDB_CELL_TRIANGLE) {
        // affine P1 triangles: B = basis table (3, nq), D = reference gradients (3, 2)
        if (d->degree != 1 || d->cdim != 1 || d->nq < 1 || d->nq > FDB_MAX_1D ||
            (d->rank != 1 && d->rank != 2) || d->integral != FDB_INTEGRAL_CELL) {
            set_error("fdb_kernel_create: triangle kernels are P1, scalar, nq <= %d", FDB_MAX_1D);
            return 1;
        }
        fdb_kernel_s *k = new fdb_kernel_s;
        k->desc = *d;
        k->n1d = 2;
        k->arity = 3;
        k->desc.offset0 = k->desc.offset1 = nullptr;
        *out = k;
        return 0;
    }
    if (d->form != FDB_FORM_HELMHOLTZ) {
        set_error("fdb_kernel_create: form %d is not in the supported set", d->form);
        return 1;
    }
    if (d->cell != FDB_CELL_HEX_EXTRUDED && d->cell != FDB_CELL_HEX) {
        set_error("fdb_kernel_create: cell type %d not supported for form %d", d->cell, d->form);
        return 1;
    }
    if (d->integral != FDB_INTEGRAL_CELL) {
        set_error("fdb_kernel_create: Helmholtz-family forms only have cell integrals");
        return 1;
    }
    if (d->degree < 1 || d->degree > 5) {
        set_error("fdb_kernel_create: degree %d outside 1..5", d->degree);
        return 1;
    }
    if (d->nq != d->degree + 1) {
        set_error("fdb_kernel_create: hex kernels need nq == degree+1 Gauss points per axis "
                  "(got nq=%d for degree %d); pin the rule with dx(degree=2*p)",
                  d->nq, d->degree);
        return 1;
    }
    if (d->rank != 1 && d->rank != 2) {
        set_error("fdb_kernel_create: rank must be 1 or 2");
        return 1;
    }
    // 2-forms assemble the scalar matrix and add it into the block diagonals (A (x) I_cdim), so any
    // block size the blocked store / SpMV kernels of mat.cu instantiate (1..4) is fine there
    const int max_cdim = d->rank == 2 ? 4 : 3;
    if (d->cdim < 1 || d->cdim > max_cdim) {
        set_error("fdb_kernel_create: cdim %d outside 1..%d", d->cdim, max_cdim);
        return 1;
    }
    if (d->cell == FDB_CELL_HEX_EXTRUDED && (!d->offset0 || !d->offset1)) {
        set_error("fdb_kernel_create: extruded cells need offset0/offset1");
        return 1;
    }
    fdb_kernel_s *k = new fdb_kernel_s;
    k->desc = *d;
    k->n1d = d->degree + 1;
    k->arity = k->n1d * k->n1d * k->n1d;
    memset(k->h_off0, 0, sizeof(k->h_off0));
    memset(k->h_off1, 0, sizeof(k->h_off1));
    if (d->offset0) memcpy(k->h_off0, d->offset0, sizeof(fdb_int) * k->arity);
    if (d->offset1) memcpy(k->h_off1, d->offset1, sizeof(fdb_int) * 8);
    k->desc.offset0 = k->h_off0;
    k->desc.offset1 = k->h_off1;
    if (collocated_derivative(k->n1d, d->B, d->D, k->Dt)) {
        set_error("fdb_kernel_create: basis table B is singular");
        delete k;
        return 1;
    }
    FDB_CUDA(cudaMalloc(&k->d_off0, sizeof(fdb_int) * k->arity));
    FDB_CUDA(cudaMalloc(&k->d_off1, sizeof(fdb_int) * 8));
    FDB_CUDA(cudaMemcpyAsync(k->d_off0, k->h_off0, sizeof(fdb_int) * k->arity,
                             cudaMemcpyHostToDevice, ctx().stream));
    FDB_CUDA(cudaMemcpyAsync(k->d_off1, k->h_off1, sizeof(fdb_int) * 8, cudaMemcpyHostToDevice,
                             ctx().stream));
    FDB_CUDA(cudaStreamSynchronize(ctx().stream));
    *out = k;
    return 0;
}

int fdb_kernel_destroy(fdb_kernel_t k)
{
    if (!k) return 0;
    if (ctx().ready) cudaStreamSynchronize(ctx().stream);
    if (k->jit) fdb_jit_destroy(k->jit);
    if (ctx().ready) {
        if (k->d_off0) cudaFree(k->d_off0);
        if (k->d_off1) cudaFree(k->d_off1);
        if (k->d_colour_cols) cudaFree(k->d_colour_cols);
        if (k->d_bdb_table) cudaFree(k->d_bdb_table);
    }
    delete k;
    return 0;
}

int fdb_kernel_call(fdb_kernel_t k, const fdb_call_args *a)
{
    if (require_init()) return 1;
    if (!k || !a) {
        set_error("fdb_kernel_call: NULL argument");
        return 1;
    }
    fdb_mirror_new_epoch();
    if (k->jit) return fdb_jit_call(k, a);      // generated wrapper (wrapper_jit.cu)
    if (k->desc.form == FDB_FORM_DG_ADVECTION) {
        // args = [out (INC), coords, q, u, consts (HOST double[2] {dtc, q_in}), facet numbers]
        // maps = [DQ1 (facet-)node map, CG1 (facet-)node map]
        const bool facets = k->desc.integral != FDB_INTEGRAL_CELL;
        const bool fused = k->desc.integral == FDB_INTEGRAL_FUSED;
        const int want = fused ? 7 : (facets ? 6 : 5);
        if (a->nargs != want || a->nmaps != 2) {
            set_error("fdb_kernel_call: DG advection expects %d args and 2 maps", want);
            return 1;
        }
        if (a->location != FDB_LOC_DEVICE) {
            set_error("fdb_kernel_call: DG advection kernels take device-resident Dats");
            return 1;
        }
        return fdb_launch_dg_advection(k, a->start, a->end, a->subset, (double *)a->args[0],
                                       (const double *)a->args[1], (const double *)a->args[2],
                                       (const double *)a->args[3], (const double *)a->args[4],
                                       facets ? (const unsigned *)a->args[5] : nullptr, a->maps[0],
                                       a->maps[1], fused ? (const fdb_int *)a->args[6] : nullptr);
    }
    if (k->desc.cell == FDB_CELL_TRIANGLE) {
        // rank 1: args = [y, coords, x]; rank 2: args = [mat, coords]; maps[0] = cell->vertex map
        // (V and the P1 coordinate space share it; a second identical map is accepted)
        const int want = k->desc.rank == 1 ? 3 : 2;
        if (a->nargs != want || a->nmaps < 1 || a->location != FDB_LOC_DEVICE) {
            set_error("fdb_kernel_call: P1 triangle kernel expects %d device args and 1-2 maps", want);
            return 1;
        }
        if (k->desc.rank == 1)
            return fdb_launch_tri_p1(k, a->start, a->end, a->subset, (double *)a->args[0],
                                     (const double *)a->args[1], (const double *)a->args[2], a->maps[0],
                                     nullptr);
        return fdb_launch_tri_p1(k, a->start, a->end, a->subset, nullptr, (const double *)a->args[1],
                                 nullptr, a->maps[0], (fdb_mat_t)a->args[0]);
    }
    const bool extruded = k->desc.cell == FDB_CELL_HEX_EXTRUDED;
    if (extruded && !a->layers) {
        set_error("fdb_kernel_call: extruded kernel called without layers");
        return 1;
    }
    if (a->end < a->start) {
        set_error("fdb_kernel_call: end < start");
        return 1;
    }
    const int nlay = extruded ? (a->layers[1] - a->layers[0] - 1) : 1;
    if (extruded && a->layers[0] != 0) {
        set_error("fdb_kernel_call: nonzero bottom layer not supported");
        return 1;
    }
    if ((long long)(a->end - a->start) * nlay >= (1ll << 31) - 64) {
        set_error("fdb_kernel_call: iteration set too large for IntType");
        return 1;
    }
    if (k->desc.rank == 2) {
        // 2-form: args = [Mat handle (INC), coords (READ)], maps = [V map, coord map]
        // (the reference passes the PETSc Mat handle in the same slot:
        // pyop2/types/mat.py:621-623)
        if (a->nargs != 2 || a->nmaps != 2) {
            set_error("fdb_kernel_call: 2-form expects 2 args (mat, coords) and 2 maps");
            return 1;
        }
        fdb_mat_t target = (fdb_mat_t)a->args[0];
        int mat_bs = 1;
        fdb_mat_block_size(target, &mat_bs);
        if (mat_bs != k->desc.cdim) {
            set_error("fdb_kernel_call: Mat block size %d != value size %d of the argument space", mat_bs,
                      k->desc.cdim);
            return 1;
        }
        if (k->desc.scatter != FDB_SCATTER_ATOMIC) {
            set_error("fdb_kernel_call: coloured scatter is not implemented for matrices");
            return 1;
        }
        const double *dcoords;
        const fdb_int *dm[2];
        const fdb_int *dsub = a->subset;
        if (a->location == FDB_LOC_HOST) {
            void *p;
            uint64_t ver = a->arg_versions ? a->arg_versions[1] : 0;
            if (!a->arg_versions) fdb_mirror_drop(a->args[1]);
            if (fdb_mirror_acquire(a->args[1], a->arg_bytes[1], ver, 1, &p)) return 1;
            dcoords = (const double *)p;
            for (int i = 0; i < 2; i++) {
                if (fdb_mirror_acquire(a->maps[i], a->map_bytes[i], map_ver(a, i), 1, &p)) return 1;
                dm[i] = (const fdb_int *)p;
            }
            if (a->subset) {
                if (fdb_mirror_acquire(a->subset, sizeof(fdb_int) * (size_t)a->end, a->subset_version, 1, &p)) return 1;
                dsub = (const fdb_int *)p;
            }
        } else {
            dcoords = (const double *)a->args[1];
            dm[0] = a->maps[0];
            dm[1] = a->maps[1];
        }
        if (mat_bs == 1)
            return fdb_launch_helmholtz_matrix(k, a->start, a->end, nlay, dsub, target, dcoords, dm[0], dm[1],
                                               nullptr);
        // vector-valued space: the element tensor of the Helmholtz family is A_scalar (x) I_cdim
        // (off-diagonal component blocks vanish identically), so the scalar kernel assembles into
        // a scalar view of the blocked pattern, which is then added to the block diagonals
        fdb_mat_t view = nullptr;
        if (fdb_mat_scalar_view_begin(target, &view)) return 1;
        int rc = fdb_launch_helmholtz_matrix(k, a->start, a->end, nlay, dsub, view, dcoords, dm[0], dm[1], nullptr);
        int rc2 = fdb_mat_scalar_view_end(target, view);
        return rc ? rc : rc2;
    }
    if (k->desc.diagonal) {
        // args = [d (INC), coords]; device-resident only
        if (a->nargs != 2 || a->nmaps != 2 || a->location != FDB_LOC_DEVICE || k->desc.cdim != 1 ||
            k->n1d > 4) {
            set_error("fdb_kernel_call: diagonal assembly expects 2 device args, 2 maps, scalar CG1..3");
            return 1;
        }
        return fdb_launch_helmholtz_matrix(k, a->start, a->end, nlay, a->subset, nullptr,
                                           (const double *)a->args[1], a->maps[0], a->maps[1],
                                           (double *)a->args[0]);
    }
    // 1-form: args = [y (INC), coords (READ), x (READ)], maps = [V map, coord map]
    if (a->nargs != 3 || a->nmaps != 2) {
        set_error("fdb_kernel_call: 1-form expects 3 args (y, coords, x) and 2 maps, got %d/%d",
                  a->nargs, a->nmaps);
        return 1;
    }
    if (a->location == FDB_LOC_HOST && a->arg_versions && a->arg_bytes && a->map_bytes &&
        a->writeback && a->output_is_zero && !a->subset && extruded &&
        k->desc.scatter == FDB_SCATTER_ATOMIC) {
        int rc = pipelined_host_action(k, a, nlay);
        if (rc >= 0) return rc;      // -1: not applicable, fall through to the monolithic path
    }
    void *dargs[3];
    const fdb_int *dmaps[2];
    const fdb_int *dsubset = a->subset;
    if (a->location == FDB_LOC_HOST) {
        if (!a->arg_bytes || !a->map_bytes) {
            set_error("fdb_kernel_call: host mode needs arg_bytes and map_bytes");
            return 1;
        }
        for (int i = 0; i < 3; i++) {
            uint64_t ver = a->arg_versions ? a->arg_versions[i] : 0;
            // without versions every call re-uploads (drop-in default: the
            // reference hands over live NumPy buffers)
            if (!a->arg_versions) fdb_mirror_drop(a->args[i]);
            const bool zero_out = (i == 0 && a->output_is_zero);
            if (fdb_mirror_acquire(a->args[i], a->arg_bytes[i], ver, zero_out ? 0 : 1, &dargs[i]))
                return 1;
            if (zero_out)
                FDB_CUDA(cudaMemsetAsync(dargs[i], 0, a->arg_bytes[i], ctx().stream));
        }
        for (int i = 0; i < 2; i++) {
            void *p;
            if (fdb_mirror_acquire(a->maps[i], a->map_bytes[i], map_ver(a, i), 1, &p)) return 1;
            dmaps[i] = (const fdb_int *)p;
        }
        if (a->subset) {
            void *p;
            if (fdb_mirror_acquire(a->subset, sizeof(fdb_int) * (size_t)a->end, a->subset_version, 1, &p)) return 1;
            dsubset = (const fdb_int *)p;
        }
    } else {
        for (int i = 0; i < 3; i++) dargs[i] = a->args[i];
        for (int i = 0; i < 2; i++) dmaps[i] = a->maps[i];
    }
    if (k->desc.scatter == FDB_SCATTER_COLOURED &&
        (k->colour_map_key != (const void *)a->maps[0] || k->colour_map_gen != map_ver(a, 0) ||
         k->colour_end != a->end)) {
        // colouring covers columns [0, end): copy the map to the host if needed
        std::vector<fdb_int> hmap;
        const fdb_int *src = a->maps[0];
        if (a->location == FDB_LOC_DEVICE) {
            hmap.resize((size_t)a->end * k->arity);
            FDB_CUDA(cudaMemcpy(hmap.data(), a->maps[0], sizeof(fdb_int) * hmap.size(),
                                cudaMemcpyDeviceToHost));
            src = hmap.data();
        }
        if (build_colouring(k, src, a->end)) return 1;
        k->colour_map_key = (const void *)a->maps[0];
        k->colour_map_gen = map_ver(a, 0);
        k->colour_end = a->end;
    }
    if (k->desc.scatter == FDB_SCATTER_COLOURED && a->start != 0) {
        set_error("fdb_kernel_call: coloured scatter needs start == 0");
        return 1;
    }
    int rc = fdb_launch_helmholtz_action(k, a->start, a->end, nlay, dsubset, (double *)dargs[0],
                                         (const double *)dargs[1], (const double *)dargs[2],
                                         dmaps[0], dmaps[1]);
    if (rc) return rc;
    if (a->location == FDB_LOC_HOST && a->writeback) {
        // the output mirror now differs from the host copy: write it back
        if (fdb_mirror_writeback(a->args[0])) return 1;
        if (a->arg_versions) fdb_mirror_set_version(a->args[0], a->arg_versions[0] + 1);
    }
    return 0;
}

}  // extern "C"
