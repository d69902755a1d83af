#!/usr/bin/env python
"""Benchmark of the hot path: assembled DoFs/s of the Poisson CG3 1-form
``assemble(action(a, u))`` on an N^3 extruded hexahedral mesh (BASELINE.json
configs[1], N = 256), fp64.

A "step" is one assembly: zero the output Dat (firedrake/assemble.py:1042-1047),
run the global kernel (gather + element kernel + scatter-add), i.e. exactly the
work ``OneFormAssembler.assemble`` does in steady state (SURVEY.md section 3.2).

    python bench.py --gpus 1 --steps 10 --warmup 3
    python bench.py --impl reference            # CPU restatement on the host cores
    python bench.py --dump-outputs DIR          # also write the last step's result to DIR/y.npy

Prints ONE JSON line (see the key list in DESIGN.md section "Measurement").
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "assembled DoFs/sec (Poisson CG3, 256^3 hex, 1-form/action)"
DUMP_ROWS = 1 << 22          # --dump-outputs: at most 32 MiB of float64 over all ranks


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", type=int, default=256, help="cells per axis")
    ap.add_argument("--degree", type=int, default=3)
    ap.add_argument("--warp", type=float, default=0.05)
    ap.add_argument("--permute", type=int, default=-1, help="seed for a random base-cell order (-1: off)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--halo", default="exec", choices=["exec", "sum"],
                    help="partitioned runs: 'exec' = redundant execution of one exec-halo cell column per rank, "
                         "no local->global reduce (SURVEY.md 8e option ii); 'sum' = the reference's owned cells + "
                         "ghost-sum reduce")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the owned rows of the assembled vector of the last step "
                         "to DIR/y.npy (DIR/y_rank<R>.npy with several GPUs), float64; above %d rows in all, "
                         "the rows at fixed seeded indices" % DUMP_ROWS)
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


# ------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        # "under load" = upper half of the samples
        sm_sorted = sorted(sm)
        med = float(np.median(sm_sorted[len(sm_sorted) // 2:])) if sm else None
        return {"sm_mhz": med, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------- workload
def make_problem(args, rank, world, pinned):
    """Rank-local slab of the n^3 mesh in Firedrake-shaped arrays, wrapped in
    the PyOP2-mirror objects (sets ordered core | owned | ghost)."""
    from firedrake_b200 import op2
    from firedrake_b200.halo import Halo
    from firedrake_b200.partition import SlabPartition
    n, p = args.n, args.degree
    if args.permute >= 0 and world > 1:
        raise SystemExit("--permute is a single-GPU stress option")
    part = SlabPartition(n, n, n, p, rank, world, warp=args.warp, exec_halo=args.halo == "exec")
    mesh, V = part.mesh, part.V
    if args.permute >= 0:
        from firedrake_b200.utility_meshes import ExtrudedHexMesh
        mesh = ExtrudedHexMesh(n, n, n, warp=args.warp, permute_seed=args.permute)
        V = mesh.function_space(p)
    halo = Halo(part.neighbours) if world > 1 else None
    cells = op2.ExtrudedSet(op2.Set(part.cell_sizes), mesh.layers)
    cells.owner_computes = part.exec_halo
    nodes = op2.Set(part.node_sizes)
    vnodes = op2.Set(mesh.coord_space.node_count)
    m0 = op2.Map(cells, nodes, V.arity, V.cell_node_map, offset=V.offset)
    m1 = op2.Map(cells, vnodes, 8, mesh.coord_map, offset=mesh.coord_offset)
    dnodes = op2.DataSet(nodes, 1, halo=halo)
    x = op2.Dat(dnodes, pinned=pinned)
    rng = np.random.default_rng(1234 + rank)
    xa = x.data_with_halos
    chunk = 1 << 24
    for i in range(0, V.node_count, chunk):
        xa[i:i + chunk] = rng.standard_normal(min(chunk, V.node_count - i))
    y = op2.Dat(dnodes, pinned=pinned)
    X = op2.Dat(op2.DataSet(vnodes, 3), mesh.coordinates)
    return part, mesh, V, cells, m0, m1, x, y, X


def dump_outputs(out_dir, y, nowned, rank, world):
    """--dump-outputs: the owned rows of ``y`` as a caller reads them (``y.data_ro``); beyond
    DUMP_ROWS / world rows per rank, the rows at sorted indices drawn with a fixed seed, so that
    two builds run with the same arguments write the same rows."""
    rows = y.data_ro[:nowned]
    k = DUMP_ROWS // world
    if nowned > k:
        rows = rows[np.unique(np.random.default_rng(0).integers(0, nowned, k))]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "y.npy" if world == 1 else f"y_rank{rank}.npy"),
            np.asarray(rows, dtype=np.float64))


def algorithmic_bytes(V, mesh):
    """SURVEY.md section 8(d): read x + write y, coordinates, map."""
    return 16 * V.node_count + 24 * mesh.coord_space.node_count + 4 * V.arity * mesh.num_base_cells


def workload_name(args):
    n, p = args.n, args.degree
    order = "lexicographic" if args.permute < 0 else "random seed %d" % args.permute
    return (f"Poisson CG{p} 1-form assemble(action(a,u)) on {n}^3 extruded hexes "
            f"({n ** 3} cells, {(n * p + 1) ** 3} DoFs), Q1 geometry warp={args.warp}, "
            f"base-cell order={order}")


def _physical_cores(cpus):
    """One logical CPU per physical core out of ``cpus`` (sysfs topology); ``cpus`` if unknown."""
    seen, out = set(), []
    for c in cpus:
        try:
            with open(f"/sys/devices/system/cpu/cpu{c}/topology/thread_siblings_list") as f:
                key = f.read().strip()
        except OSError:
            return list(cpus)
        if key not in seen:
            seen.add(key)
            out.append(c)
    return out


def cpu_baseline(args, seconds, reps=5):
    """The oracle (CPU restatement of the PyOP2 wrapper + TSFC kernel) in the reference's MPI
    model (SURVEY.md section 8d, BASELINE.md section 3): one sequential worker PINNED to each
    host core, every worker first-touching its own ghosted slab, local loops followed by the
    ghost-plane reduce; a pass = barrier-to-barrier wall time (max over workers).  With P workers
    and n base columns along x each worker holds an (n/P) x n x n slab, i.e. the 128-core box
    runs the whole 256^3 job per pass; if that exceeds the time budget the slab is thinned and
    the sample says so."""
    from firedrake_b200.fiat_lite import interval_element
    from firedrake_b200.utility_meshes import ExtrudedHexMesh
    from oracle import oracle
    p, n = args.degree, args.n
    el = interval_element(p)
    cpus = sorted(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else list(range(os.cpu_count() or 1))
    phys = _physical_cores(cpus)
    native = True
    oracle.lib(native)

    def slab(sx):
        mesh = ExtrudedHexMesh(sx, n, n, Lx=sx / n, warp=args.warp)
        V = mesh.function_space(p)
        x = np.random.default_rng(5).standard_normal(V.node_count)
        return mesh, V, x

    # calibrate on one worker, one base row
    mesh, V, x = slab(1)
    t_row = float(oracle.action_bench(el, mesh, V, x, 1, 1, cpus[:1], native=native)[0][0])
    cands = [("one worker per logical CPU", cpus)]
    if len(phys) < len(cpus):
        cands.append(("one worker per physical core", phys))
    budget = seconds / (len(cands) * 3 + reps + 1)           # seconds per pass
    best = None
    for label, ids in cands:
        P = len(ids)
        sx_full = max(1, -(-n // P))                         # ceil: P slabs cover the mesh
        # SMT siblings share a core: allow ~2x the single-thread row time per pass
        sx = max(1, min(sx_full, int(budget / max(2.0 * t_row, 1e-9))))
        mesh, V, x = slab(sx)
        ts, _ = oracle.action_bench(el, mesh, V, x, P, 2, ids, native=native)
        owned = (sx * p) * (n * p + 1) * (n * p + 1)          # one face shared with the neighbour
        rate = P * owned / float(np.min(ts))
        if best is None or rate > best[0]:
            best = (rate, label, ids, sx, sx_full, mesh, V, x)
    _, label, ids, sx, sx_full, mesh, V, x = best
    P = len(ids)
    ts, _ = oracle.action_bench(el, mesh, V, x, P, reps, ids, native=native)
    t = float(np.median(ts))
    owned = (sx * p) * (n * p + 1) * (n * p + 1)
    value = P * owned / t
    whole = "the whole mesh" if sx == sx_full and P * sx >= n else f"{P * sx}/{n} of the mesh (time-bounded sample)"
    return {"value": value, "unit": "DoFs/s", "cores": P, "kind": "port",
            "sample": f"{P} pinned workers ({label}) x ({sx}x{n} base cells x {n} layers, CG{p}) slabs = {whole}; "
                      f"first-touch private arrays, ghost-plane reduce included, median of {reps} passes after "
                      f"warm-up, {os.path.basename(oracle.lib(native)._path)}",
            "seconds_per_pass": t, "seconds_min": float(np.min(ts)), "seconds_max": float(np.max(ts)),
            "passes": [float(v) for v in ts], "dofs_per_pass": P * owned}


def cpu_cg_baseline(mesh, V, p, b, bc_nodes, iters):
    """cpu_baseline leg of benchmarks/cg_multi.py (config 5): unpreconditioned CG on the host cores
    with the oracle's operator (banded multi-threaded action, Dirichlet rows as in
    firedrake/matrix_free/operators.py:225-239) and OpenMP vector algebra -- the reference's
    'solve stays on the host' path restated.  ``iters`` fixed iterations from x = 0; returns
    (seconds, residual history)."""
    from firedrake_b200.fiat_lite import interval_element
    from oracle import oracle
    el = interval_element(p)
    coords = np.ascontiguousarray(mesh.coordinates)
    n = V.node_count
    xin, Ap = np.empty(n), np.empty(n)

    def mult(v, out):
        np.copyto(xin, v)
        xin[bc_nodes] = 0.0
        out[:] = 0.0
        oracle.action_extruded_parallel(el, mesh, out, coords, xin, V.cell_node_map, V.offset, mesh.coord_map,
                                        mesh.coord_offset, native=True)
        out[bc_nodes] = v[bc_nodes]

    x = np.zeros(n)
    r = b.copy()
    pv = r.copy()
    t0 = time.perf_counter()
    rr = oracle.vec_dot(r, r)
    hist = [float(np.sqrt(rr))]
    for _ in range(iters):
        mult(pv, Ap)
        alpha = rr / oracle.vec_dot(pv, Ap)
        oracle.vec_axpy(alpha, pv, x)
        oracle.vec_axpy(-alpha, Ap, r)
        rr_new = oracle.vec_dot(r, r)
        oracle.vec_aypx(rr_new / rr, r, pv)
        rr = rr_new
        hist.append(float(np.sqrt(rr)))
    return time.perf_counter() - t0, hist


def run_reference(args):
    """--impl reference: K 'steps', each one bounded pass of the CPU arm (above)."""
    reps = max(5, min(args.steps, 10))
    base = cpu_baseline(args, max(args.cpu_seconds, 20.0), reps=reps)
    line = {
        "impl": "reference", "metric": METRIC, "value": base["value"], "unit": "DoFs/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": base["seconds_per_pass"] * 1e3 * ((args.n * args.degree + 1) ** 3) / base["dofs_per_pass"],
        "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args),
                   "quadrature": f"Gauss-Legendre {args.degree + 1}^3 (dx(degree={2 * args.degree}))",
                   "note": "CPU restatement of Firedrake/PyOP2/TSFC (oracle/), not Firedrake itself: omits "
                           "Python glue and PETSc; ms_per_step = time per pass scaled to the whole mesh; "
                           f"timed passes: {reps}"},
        "cpu_baseline": base,
        "e2e": {"value": base["value"], "unit": "DoFs/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def oracle_parity(args, part, mesh, V, x, y, rank, world, dist):
    """Outside the timed region: every rank compares the OWNED rows of its device result with
    the oracle run on the same slab (banded multi-threaded wrapper, oracle.action_extruded_parallel),
    after the oracle's own ghost-plane sums have gone to their owners over gloo -- the distributed
    result is checked against an independent CPU computation, not against another GPU run."""
    from firedrake_b200.fiat_lite import interval_element
    from oracle import oracle
    el = interval_element(args.degree)
    xh = np.ascontiguousarray(x.data_ro_with_halos if hasattr(x, "data_ro_with_halos") else x.data_with_halos)
    yh = np.ascontiguousarray(y.data_ro_with_halos if hasattr(y, "data_ro_with_halos") else y.data_with_halos)
    if world > 1:
        # ghost rows of x straight from their owners' HOST copies over gloo (independent of the
        # device halo exchange under test)
        import torch
        xh = xh.copy()
        flat = xh.reshape(-1)
        reqs, bufs = [], []
        for nb, send, recv in part.neighbours:
            if len(send):
                reqs.append(dist.isend(torch.from_numpy(np.ascontiguousarray(flat[send])), nb))
        for nb, send, recv in part.neighbours:
            if len(recv):
                t = torch.empty(len(recv), dtype=torch.float64)
                dist.recv(t, nb)
                flat[recv] = t.numpy()
        for r in reqs:
            r.wait()
    yo = np.zeros(V.node_count)
    ncpu = len(os.sched_getaffinity(0))
    t0 = time.perf_counter()
    oracle.action_extruded_parallel(el, mesh, yo, np.ascontiguousarray(mesh.coordinates), xh.reshape(-1),
                                    V.cell_node_map, V.offset, mesh.coord_map, mesh.coord_offset,
                                    nthreads=max(1, ncpu // world), native=True)
    t_or = time.perf_counter() - t0
    if world > 1 and not part.exec_halo:
        import torch
        # ghost plane (my left face, owned by rank-1) -> owner adds (local_to_global, SUM)
        reqs = []
        if rank > 0:
            send = torch.from_numpy(np.ascontiguousarray(yo[V.plane_nodes(0)]))
            reqs.append(dist.isend(send, rank - 1))
        if rank < world - 1:
            hi = V.plane_nodes(part.x1 - part.x0)
            recv = torch.empty(len(hi), dtype=torch.float64)
            dist.recv(recv, rank + 1)
            yo[hi] += recv.numpy()
        for r in reqs:
            r.wait()
    no = V.owned_node_count
    err = float(np.abs(yh.reshape(-1)[:no] - yo[:no]).max())
    scale = float(np.abs(yo[:no]).max())
    if dist is not None:
        import torch
        t = torch.tensor([err, scale], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        err, scale = float(t[0]), float(t[1])
    return {"rel_err": err / scale, "vs": "oracle", "tolerance": 1e-12,
            "checked": "every owned DoF of every rank (max-norm error / max-norm of the oracle result)",
            "oracle_seconds": t_or}


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        if rank == 0:
            run_reference(args)
        return
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with "
                         "python -m torch.distributed.run --nproc-per-node N bench.py --gpus N")

    import ctypes as C
    from firedrake_b200 import _lib, op2
    from firedrake_b200.halo import comm_init_from_env
    rank, world, dist = comm_init_from_env()
    L = _lib.lib()
    n, p = args.n, args.degree
    t_setup = time.perf_counter()
    part, mesh, V, cells, m0, m1, x, y, X = make_problem(args, rank, world, pinned=not args.no_e2e)
    ndof_owned = V.owned_node_count
    ndof_global = (n * p + 1) ** 3
    # the per-cell-metric kernel variant for meshes of parallelepipeds (only --warp 0 qualifies),
    # after the device-side check of the promise (DESIGN.md section 8b); FDB_AFFINE=0 opts out
    affine = False
    if os.environ.get("FDB_AFFINE", "1") != "0" and args.warp == 0.0:
        res = C.c_int()
        off1 = np.ascontiguousarray(mesh.coord_offset, dtype=np.int32)
        _lib.check(L.fdb_cells_are_affine(X.device_ptr, m1.device_ptr, off1.ctypes.data, 0, cells.total_size,
                                          mesh.nz, C.byref(res)), "fdb_cells_are_affine")
        affine = bool(res.value)
    kern = op2.Kernel("helmholtz", degree=p, alpha=1.0, beta=0.0, affine=affine)
    gk = op2.GlobalKernel(kern, [m0, m1], extruded=True)
    loop = op2.Parloop(gk, cells, [y(op2.INC, m0), X(op2.READ, m1), x(op2.READ, m0)], location="device")
    t_setup = time.perf_counter() - t_setup

    def barrier():
        _lib.check(L.fdb_synchronize())
        if dist is not None:
            dist.barrier()

    def maxreduce(v):
        if dist is None:
            return v
        import torch
        t = torch.tensor([v], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def step():
        # one assembly: zero the tensor, refresh ghost x, core cells overlapped
        # with the exchange, owned cells, ghost contributions back to owners
        x.halo_valid = world == 1      # x changes every solver iteration
        y.zero()
        loop()

    # make everything resident (inputs in HBM before the timed region)
    x.device_ptr; y.device_ptr; X.device_ptr; m0.device_ptr; m1.device_ptr
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()

    tm = C.c_void_p(); tk = C.c_void_p()
    _lib.check(L.fdb_timer_create(C.byref(tm)))
    _lib.check(L.fdb_timer_create(C.byref(tk)))
    sampler = ClockSampler(int(os.environ.get("LOCAL_RANK", "0")))
    sampler.start()
    time.sleep(0.3)
    launches0 = L.fdb_launch_count()
    ms = C.c_float()
    barrier()
    _lib.check(L.fdb_timer_start(tm))
    for _ in range(args.steps):
        step()
    _lib.check(L.fdb_timer_stop(tm, C.byref(ms)))
    barrier()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, y, ndof_owned, rank, world)
    total_ms = maxreduce(ms.value)
    launches = L.fdb_launch_count() - launches0
    # kernel-only duration (CUDA events around the global kernel alone, same
    # stream); single-GPU figure used for the roofline
    kms = []
    kloop = op2.Parloop(gk, cells, [y(op2.INC, m0), X(op2.READ, m1), x(op2.READ, m0)], location="device")
    for _ in range(args.steps):
        y.zero()
        y.device_ptr
        x.halo_valid = True
        y.frozen_halo = True
        _lib.check(L.fdb_timer_start(tk))
        kloop()
        _lib.check(L.fdb_timer_stop(tk, C.byref(ms)))
        y.frozen_halo = False
        kms.append(ms.value)
    clocks = sampler.stop()
    ms_per_step = total_ms / args.steps
    value = ndof_global / (ms_per_step * 1e-3)
    kernel_ms = maxreduce(float(np.mean(kms)))

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_gbs = peaks.get("hbm_gbs", 6650.0)
    abytes = algorithmic_bytes(V, mesh)
    hbm_achieved = abytes / (kernel_ms * 1e-3) / 1e9
    kname = f"helmholtz_action_kernel<{p + 1},false,true,3>"
    counts = {}
    try:
        counts = json.load(open(os.path.join(ROOT, "profiles", "kernel_counts.json"))).get(kname, {})
    except Exception:
        pass
    # The kernel is fp64-pipe bound (DESIGN.md section 4): the binding roofline is the fp64 FMA rate,
    # 64 lanes/clk/SM (the DMMA/DFMA microbenchmark of profiles/r01_microbench_fp64.txt reaches 37.1 of
    # these 37.2 TFLOP/s; MEASURED_PEAKS.json carries no fp64 figure).  Work = SASS-counted flops per
    # cell (profiles/kernel_counts.json) when this kernel instance has been counted, else the model.
    ctx_sm = C.c_int()
    _lib.check(L.fdb_device_info(None, 0, C.byref(ctx_sm), None), "fdb_device_info")
    sm_count = ctx_sm.value or 148
    clk_hz = (clocks.get("sm_max_mhz") or 1965.0) * 1e6
    fp64_peak = sm_count * 64 * 2 * clk_hz / 1e12
    ncell_rank = mesh.num_cells
    flop_cell = counts.get("flop_per_cell", kern.num_flops)
    tf = flop_cell * ncell_rank / (kernel_ms * 1e-3) / 1e12
    traffic = (counts.get("dram_bytes_per_launch") or {}).get(str(n)) if world == 1 else None
    roofline = {"bound": "fp64", "achieved": tf, "peak": fp64_peak, "unit": "TFLOP/s", "frac": tf / fp64_peak,
                "traffic": traffic, "kernel": kname, "kernel_ms": kernel_ms,
                "flop_per_cell": flop_cell,
                "flop_source": "SASS count (profiles/kernel_counts.json, profiles/r02_action_cg3.sass, tools/sass_loops.py)" if counts
                               else "model 24 n^4 + 130 n^3 (kernel instance not counted)",
                "peak_source": f"{sm_count} SMs x 64 fp64 FMA lanes/clk x 2 x {clk_hz / 1e9:.3f} GHz (clocks.sm_max_mhz); "
                               "microbenchmark: 37.1 TFLOP/s (profiles/r01_microbench_fp64.txt)",
                "traffic_source": "ncu --set full capture, profiles/r02s2_action_cg3_n256_summary.txt (8.783 GB read + 4.102 GB written)" if traffic else None,
                "hbm": {"achieved": hbm_achieved, "peak": peak_gbs, "unit": "GB/s", "frac": hbm_achieved / peak_gbs,
                        "algorithmic_bytes_per_launch": abytes,
                        "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650",
                        "note": "reported because the contract asks for it; with geometry recomputed at every "
                                "quadrature point this workload cannot be HBM bound (SURVEY.md section 8d)"}}
    if counts:
        # share of the fp64 pipe's issue slots actually used (2 cycles per warp instruction per SMSP)
        roofline["fp64_pipe_frac"] = (counts["fp64_instr_per_cell"] * ncell_rank / (sm_count * 64 * clk_hz)) / (kernel_ms * 1e-3)
        if "three_register_fp64_per_warp_unit" in counts:
            # a DFMA with three distinct register sources needs a third register-read cycle (measured:
            # profiles/r02_microbench_issue.txt, 3.05 cycles per DFMA against 2.0): pipe time the kernel cannot avoid
            cyc_unit = 2.0 * counts["fp64_instr_per_warp_unit"] + counts["three_register_fp64_per_warp_unit"]
            units = ncell_rank / counts["cells_per_warp_unit"]
            roofline["fp64_pipe_frac_with_operand_reads"] = (cyc_unit * units / (sm_count * 4 * clk_hz)) / (kernel_ms * 1e-3)

    e2e = None
    if not args.no_e2e:
        nst = max(1, args.steps)
        if world == 1:
            hloop = op2.Parloop(gk, cells, [y(op2.INC, m0), X(op2.READ, m1), x(op2.READ, m0)], location="host")
            def hstep():
                x.data_with_halos[0] += 0.0      # host write: bumps dat_version -> H2D of x
                y.zero()                         # assemble() zeroes the tensor (lazy here)
                hloop()                          # H2D x, device memset y, kernel, D2H y
                return float(y._data[0])
            path = ("op2.Parloop(location='host') -> fdb_kernel_call(FDB_LOC_HOST): pinned host Dats; the "
                    "engine overlaps H2D of x | kernel | D2H of y over 32 column chunks (3 streams)")
        elif args.halo == "exec":
            hloop = op2.Parloop(gk, cells, [y(op2.INC, m0), X(op2.READ, m1), x(op2.READ, m0)], location="host")
            def hstep():
                x.data_with_halos[0] += 0.0      # host write: bumps dat_version -> H2D of the local x
                x.halo_valid = False             # ... whose ghost rows are stale again
                y.zero()
                hloop()                          # Parloop._call_host_partitioned
                return float(y._data[0])
            path = ("per rank, op2.Parloop(location='host') on the exec-halo partition: core cells through the chunked "
                    "H2D x | kernel | D2H y pipeline of fdb_kernel_call(FDB_LOC_HOST), remaining owned x rows uploaded, "
                    "ghost rows over NCCL, boundary cells on the mirrors, the row ranges they touch downloaded again")
        else:
            def hstep():
                x.data_with_halos[0] += 0.0      # host write -> H2D of the local x
                x.halo_valid = False             # ... whose ghost rows are stale again
                y.zero()
                loop()                           # exchanges + kernels on device-resident mirrors
                return float(y.data_ro[0])       # D2H of the local y
            path = ("per rank: pinned host Dat -> H2D, halo exchanges + kernels, D2H of the local y; "
                    "op2.Parloop(location='device') with lazy host sync")
        hstep()
        barrier()
        t0 = time.perf_counter()
        for _ in range(nst):
            hstep()
        barrier()
        t = maxreduce((time.perf_counter() - t0) / nst)
        e2e = {"value": ndof_global / t, "unit": "DoFs/s", "h2d_bytes_per_step": x.nbytes,
               "d2h_bytes_per_step": y.nbytes, "ms_per_step": t * 1e3, "steps": nst, "path": path,
               "bytes_are": "per rank"}

    parity = None
    if not args.no_parity:
        x.halo_valid = world == 1
        y.zero()
        loop()
        parity = oracle_parity(args, part, mesh, V, x, y, rank, world, dist)

    if rank != 0:
        return
    line = {
        "metric": METRIC, "value": value, "unit": "DoFs/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args),
                   "quadrature": f"Gauss-Legendre {p + 1}^3 (dx(degree={2 * p}))",
                   "parallelism": (f"{world} slab(s) along x, NCCL halo exchange; "
                                   + ("exec-halo mode: one redundant cell column per rank, ghost reads of x only "
                                      f"({p + 1} planes of {n * p + 1}^2 dofs), no ghost-sum reduce" if args.halo == "exec"
                                      else f"one {n * p + 1}^2-dof face per neighbour each way (ghost read + ghost sum)"))
                                  if world > 1 else "single GPU",
                   "l2": "inputs (x,y: %.1f GB per rank) exceed the 126 MB L2; no flush needed"
                         % (2 * 8 * V.node_count / 1e9),
                   "setup_s": t_setup,
                   "kernel_variant": "per-cell metric (all cells checked affine)" if affine else "general (geometry at every quadrature point)"},
        "clocks": clocks, "gpu_launches": int(launches), "roofline": roofline,
    }
    if e2e:
        line["e2e"] = e2e
    if parity:
        line["parity"] = parity
    if not args.no_cpu and world == 1:
        line["cpu_baseline"] = cpu_baseline(args, args.cpu_seconds)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
