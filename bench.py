#!/usr/bin/env python
"""bench.py -- time-steps/s of the B200 hot path (assembly of the linearised Taylor-Hood system +
block-preconditioned GMRES) on the mesh-3D-20-equivalent, with the roofline of the dominant kernel,
an end-to-end number through the C ABI with host buffers, and a CPU baseline.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--level 20] [--impl reference] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  A "step" is one pass of the hot path -- nsb_assemble_linearized +
nsb_solve with the reference's stopping rule (GMRES(150), 1e-2 * ||b||, <= 200 iterations) -- on the
synthetic state of SURVEY.md 8(d) (3D-2Z parameters: dt 0.01, theta 0.5, nu 1e-3, SUPG + grad-div).
`value` keeps all inputs resident in HBM; `e2e` pushes u^n, u^{n-1} and the constraints from host buffers
and reads the solution back every step.  Inputs are far larger than L2 (12.8 GB of matrix values),
so no explicit L2 flush is needed between iterations.

`--dump-outputs DIR` writes what the timed path returned in its last timed step (the solution vector and the solve's
status) as .npy files; the inputs are seeded, so two builds run with the same arguments can be compared file by file.
Nothing is written into the source tree, which may be read-only: the generated mesh file and the line the reference arm
leaves for the GPU arm go to a private per-user directory under the temporary directory (user_cache_dir).
"""
import argparse
import hashlib
import json
import os
import stat
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
CASE = "3D-2Z"
DUMP_MAX_VALUES = 3_750_000        # float64 values per dumped array: two arrays stay under 64 MB, larger ones are sampled
DUMP_SEED = 2024


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def user_cache_dir():
    """<tmp>/nsb200-<uid>: run-time files of bench.py and the tools that share its mesh, kept out of the source tree.  Created
    with mode 0700; refused unless it is a real directory owned by this user that no one else can write to, so another
    user cannot plant a mesh or a reference-arm line in it."""
    d = os.path.join(tempfile.gettempdir(), "nsb200-%d" % os.getuid())
    os.makedirs(d, mode=0o700, exist_ok=True)
    st = os.lstat(d)
    if not stat.S_ISDIR(st.st_mode) or st.st_uid != os.getuid() or st.st_mode & 0o022:
        raise RuntimeError("%s is not a private directory of this user" % d)
    return d


def get_mesh_file(level):
    """mesh-3D-<level>-equivalent as a binary dump for the C++ host reader (generated once, cached in user_cache_dir).  The
    cache key includes a hash of the generator's sources, so checkouts with different generators never share a file."""
    from tools import meshgen, msh
    h = hashlib.sha1()
    for f in (meshgen.__file__, msh.__file__, os.path.join(os.path.dirname(meshgen.__file__), "cross_sections", "level%d.npz" % level)):
        if os.path.exists(f):
            h.update(open(f, "rb").read())
    path = os.path.join(user_cache_dir(), "mesh-3D-%d-%s.bin" % (level, h.hexdigest()[:16]))
    if not os.path.exists(path):
        t0 = time.time()
        m = meshgen.mesh_3d(level)
        tmp = "%s.%d.tmp" % (path, os.getpid())
        msh.write_bin(tmp, m)
        os.replace(tmp, path)
        log("[bench] generated mesh-3D-%d-equivalent: %d cells, %d vertices in %.1f s" % (level, m.n_cells, m.n_vertices, time.time() - t0))
    return path


def dump_outputs(out_dir, sol, n_u, converged, iterations, residual):
    """The timed path's result, float64: the velocity and the pressure part of the solution, each in full or -- when it has
    more than DUMP_MAX_VALUES entries -- at DUMP_MAX_VALUES sorted indices drawn with DUMP_SEED (the same for every run of
    the same workload), and [converged, GMRES iterations, final residual] of the solve."""
    def sample(a):
        if a.size <= DUMP_MAX_VALUES:
            return a
        return a[np.sort(np.random.default_rng(DUMP_SEED).choice(a.size, DUMP_MAX_VALUES, replace=False))]

    os.makedirs(out_dir, exist_ok=True)
    arrays = {"solution_velocity": sample(sol[:n_u]), "solution_pressure": sample(sol[n_u:]),
              "solve_status": np.array([float(converged), float(iterations), residual])}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, np.float64))
    log("[bench] outputs of the last timed step written to %s: %s" % (out_dir, ", ".join("%s %s" % (k, v.shape) for k, v in arrays.items())))


def synthetic_state(pts, comp, n_u, U_m=2.25, H=0.41):
    """u^n = inlet paraboloid * (1 + 0.1 xi), u^{n-1} likewise (seeds 1234 / 1235), p = 0."""
    N = pts.shape[0]
    prof = 16.0 * U_m * pts[:, 0] * pts[:, 1] * (H - pts[:, 0]) * (H - pts[:, 1]) / H ** 4
    base = np.where((comp == 2) & (np.arange(N) < n_u), prof, 0.0)
    un = base * (1 + 0.1 * np.random.default_rng(1234).uniform(-1, 1, N))
    unm1 = base * (1 + 0.1 * np.random.default_rng(1235).uniform(-1, 1, N))
    return un, unm1


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.rows = index, False, []

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(r[2 + k].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons}


def recorded_traffic(level, kernel, precision=32):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture
    (profiles/r02_traffic.json, keys level -> kernel[_fp<precision>]); None when no capture exists for this workload / kernel."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))[str(level)]
        return t.get("%s_fp%d" % (kernel, precision), t.get(kernel))
    except Exception:
        return None


def measured_peak():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle's C/OpenMP restatement of the reference's time step on the host cores
# ------------------------------------------------------------------------------------------------
# The reference's own mpirun path cannot be built here (deal.II + Trilinos + MPI + Boost absent), so `kind` is "port":
# oracle/c/ns_oracle_c.c = the reference's assembly loops (cpp:569-831) and its solve_linear_system (cpp:833-868,
# hpp:279-366): ILU(1) on F / ILU(0) on M_p over one row block per thread (Ifpack's per-rank ILU, overlap 0), re-factorized
# every solve like the reference, GMRES(150) to 1e-2*||b||, at most 200 iterations.  Substitutions, all stated in the
# emitted `sample`: K_p^-1 is ILU(0)-CG to 1e-4 instead of one Trilinos-ML V-cycle (a few per cent of the solve time,
# reported as kp_cg_s); M_p / K_p are assembled once outside the timed step (the reference also builds them once,
# cpp:798-829); the Schur mass coefficient is the reference's theta*nu (hpp:343).
SAMPLE_LC = float(os.environ.get("NSB_BENCH_SAMPLE_LC", "0.025"))      # cylinder mesh size of the bounded CPU sample mesh


def ref_cache():
    """The last `--impl reference` line, read back by the GPU arm."""
    return os.path.join(user_cache_dir(), "reference_arm_last.json")


def host_threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


class CpuCase:
    """Mesh, DoFs, pattern, constraints, synthetic state and the one-time pressure blocks of the CPU arm (not timed)."""

    def __init__(self, mesh):
        from oracle import assemble as asm, dofs as odofs, postprocess as pp, c_port
        c_port.set_num_threads(host_threads())            # torchrun exports OMP_NUM_THREADS=1: use the host cores anyway
        self.threads = c_port.num_threads()
        t0 = time.time()
        self.mesh = mesh
        self.dm = dm = odofs.enumerate_dofs(mesh)
        rp, col = odofs.make_sparsity_fast(dm)
        self.pat = (np.ascontiguousarray(rp, np.int64), np.ascontiguousarray(col, np.int32))
        tc = pp.TEST_CASES[CASE]
        self.con = odofs.build_constraints(mesh, dm, pp.inlet_profile(3, tc["U_m"], False, 4.0, 1.0), pp.boundary_ids(3))
        self.un, self.unm1 = synthetic_state(dm.support_points, dm.component, dm.n_u)
        self.p = asm.Params(dt=0.01, theta=0.5, nu=1e-3, use_supg=True)
        self.pp_blocks = asm.pressure_blocks(mesh, dm, self.con)
        self.setup_s = time.time() - t0

    def step(self, time_budget_s=0.0):
        """One pass of the hot path as the reference brackets it (cpp:1113-1296: assembly + preconditioner setup + GMRES)."""
        from oracle import c_port
        dm = self.dm
        t0 = time.time()
        A, b, _, _ = c_port.assemble_linearized(self.mesh, dm, self.pat, self.p, self.con, self.un, self.unm1, with_pressure_matrices=False)
        t1 = time.time()
        _, its, res, rc, tm = c_port.solve_blocks(self.pat, dm.n_dofs, dm.n_u, A, self.pp_blocks, b, self.p, max_it=200, tol_rel=1e-2,
                                                  n_tmp_vectors=150, time_budget_s=time_budget_s)
        t2 = time.time()
        r = dict(seconds=t2 - t0, assembly_s=t1 - t0, solve_s=t2 - t1, precond_setup_s=float(tm["setup"]), gmres_s=float(tm["gmres"]),
                 kp_cg_s=float(tm["kp_cg"]), gmres_iterations=int(its), converged=(rc == 0), stopped_by_time_budget=(rc == 2),
                 breakdown_nan=(rc == 3))
        log("[bench] cpu step: assembly %.1f s, ILU setup %.1f s, GMRES %.1f s (%d its, converged %s%s), K_p CG %.1f s"
            % (r["assembly_s"], r["precond_setup_s"], r["gmres_s"], its, rc == 0,
               ", STOPPED BY TIME BUDGET" if rc == 2 else ", RESIDUAL IS NaN (ILU(1) breakdown)" if rc == 3 else "", r["kp_cg_s"]))
        return r


def cpu_sample_entry(full_cells, repeats=2):
    """cpu_baseline of the GPU arm when no same-box run of `--impl reference` is available: one step on a coarser mesh of
    the same geometry and state (about 10-30 s of CPU work), scaled linearly by the cell count -- an extrapolation, marked so."""
    from tools import meshgen
    case = CpuCase(meshgen.mesh_3d(lc_cyl=SAMPLE_LC, lc_global=0.15))
    rs = [case.step() for _ in range(repeats)]
    r = rs[-1]
    factor = full_cells / case.mesh.n_cells
    return {"value": 1.0 / (r["seconds"] * factor), "unit": "steps/s", "cores": case.threads, "kind": "port", "same_config": False,
            "extrapolation_factor": round(factor, 2),
            "sample": "BOUNDED SAMPLE, EXTRAPOLATED: oracle C/OpenMP port (reference assembly loops; ILU(1)/ILU(0) per thread block, "
                      "re-factorized every solve; K_p^-1 by ILU(0)-CG 1e-4 in place of ML; GMRES(150), <= 200 its) on a %d-cell mesh of the "
                      "same geometry and state: %.1f s per step (assembly %.1f, ILU setup %.1f, GMRES %.1f incl. K_p CG %.1f), %d its, "
                      "converged=%s; scaled by cells x%.1f to the %d-cell workload.  The same-config number is the `--impl reference` line."
                      % (case.mesh.n_cells, r["seconds"], r["assembly_s"], r["precond_setup_s"], r["gmres_s"], r["kp_cg_s"],
                         r["gmres_iterations"], r["converged"], factor, full_cells)}


def cpu_memory_estimate(level):
    """Peak host bytes of CpuCase + one step at mesh-3D-<level> (measured ratios: 415 nnz per cell, ILU(1) fill 4.7 x nnz(F))."""
    cells = {5: 92136, 10: 572922, 20: 3851622, 40: 30.5e6}[level]
    nnz = 415.0 * cells
    nnzF = 0.84 * nnz
    n = 4.23 * cells
    return nnz * (8 + 4) + nnzF * 12 + 4.7 * nnzF * 12 + 150 * n * 8 + 8e3 * cells


def reference_arm(args):
    """`--impl reference`: one full time step of the CPU port on the SAME mesh-3D-<level>-equivalent, state and parameters
    as the GPU arm, on all host cores.  One step takes minutes, so the arm times exactly one step after an untimed setup
    (`steps`/`warmup` in the line are what was actually run; the requested values are under config).  GMRES is capped at the
    reference's own 200 iterations (cpp:836): a non-converged solve is what the reference executes before its fallbacks."""
    import psutil
    from tools import meshgen
    level = args.level
    avail = psutil.virtual_memory().available
    note = None
    while level > 5 and cpu_memory_estimate(level) > 0.8 * avail:
        note = "mesh-3D-%d needs about %.0f GB of host memory for the ILU(1) factors, %.0f GB available" % (level, cpu_memory_estimate(level) / 1e9, avail / 1e9)
        level = {40: 20, 20: 10, 10: 5}[level]
    t0 = time.time()
    mesh = meshgen.mesh_3d(level)
    log("[bench] reference arm: mesh-3D-%d-equivalent, %d cells (%.0f s); host threads %d, %.0f GB available"
        % (level, mesh.n_cells, time.time() - t0, host_threads(), avail / 1e9))
    case = CpuCase(mesh)
    log("[bench] reference arm: setup %.0f s (DoFs %d, nnz %d)" % (case.setup_s, case.dm.n_dofs, case.pat[1].size))
    r = case.step(time_budget_s=float(os.environ.get("NSB_BENCH_REF_BUDGET_S", "1000")))
    same = level == args.level
    value = 1.0 / r["seconds"]
    cells_full = {5: 92136, 10: 572922, 20: 3851622}.get(args.level)
    if not same and cells_full:
        value *= mesh.n_cells / cells_full
    entry = {"value": value, "unit": "steps/s", "cores": case.threads, "kind": "port", "same_config": same,
             "sample": ("one full step of the oracle C/OpenMP port (reference assembly loops; ILU(1) on F + ILU(0) on M_p per thread "
                        "block, re-factorized every solve; K_p^-1 by ILU(0)-CG 1e-4 in place of ML; GMRES(150), tol 1e-2, <= 200 its) on the "
                        "mesh-3D-%d-equivalent (%d cells, %d DoFs, %d nnz): %.1f s = assembly %.1f + ILU setup %.1f + GMRES %.1f "
                        "(K_p CG %.1f); %d its, converged=%s%s%s"
                        % (level, mesh.n_cells, case.dm.n_dofs, case.pat[1].size, r["seconds"], r["assembly_s"], r["precond_setup_s"],
                           r["gmres_s"], r["kp_cg_s"], r["gmres_iterations"], r["converged"],
                           "; GMRES stopped early by the arm's time budget, so the step time is a LOWER bound" if r["stopped_by_time_budget"] else
                           "; the ILU(1) factors of F overflow on this mesh (no pivoting, Ifpack defaults) and the residual is NaN from the first "
                           "iteration -- deal.II's SolverControl reports failure on a NaN residual, so the time is that of the reference's FIRST "
                           "attempt only (its BE fallback and dt-halving retries would repeat assembly + factorization up to 6 more times): a LOWER bound"
                           if r["breakdown_nan"] else "",
                           "; NOT the requested mesh (%s): scaled by cells" % note if not same else ""))}
    line = {
        "impl": "reference", "metric": "time-steps/s", "value": value, "unit": "steps/s", "n_gpus": args.gpus,
        "steps": 1, "warmup": 0, "ms_per_step": 1e3 / value, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args.level, mesh.n_cells if same else None, case.dm.n_dofs if same else None, case.pat[1].size if same else None),
                   "requested_steps": args.steps, "requested_warmup": args.warmup,
                   "gmres_iterations_per_step": [r["gmres_iterations"]], "converged": r["converged"], "breakdown_s": r,
                   "untimed_setup_s": round(case.setup_s, 1)},
        "cpu_baseline": entry,
        "e2e": {"value": value, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    try:
        json.dump(dict(line, when=time.time(), level=args.level), open(ref_cache(), "w"))
    except Exception:
        pass
    print(json.dumps(line), flush=True)


def workload_name(level, cells=None, dofs=None, nnz=None):
    sizes = " (%d tets, %d DoFs, %d nnz)" % (cells, dofs, nnz) if cells else ""
    return ("mesh-3D-%d-equivalent%s, 3D-2Z: CN theta=0.5, linearised, dt=0.01, SUPG+grad-div, GMRES(150) tol 1e-2*||b||, max 200 its"
            % (level, sizes))


def cpu_baseline_for(level, full_cells):
    """cpu_baseline of the GPU arm: the same-config measurement of `--impl reference` when it ran on this box within the
    last two hours (the driver runs it first), else the bounded, extrapolated sample."""
    try:
        c = json.load(open(ref_cache()))
        if c.get("level") == level and time.time() - c.get("when", 0) < 7200 and c["cpu_baseline"].get("same_config"):
            e = dict(c["cpu_baseline"])
            e["sample"] = "measured by `bench.py --impl reference` on this box: " + e["sample"]
            return e
    except Exception:
        pass
    return cpu_sample_entry(full_cells)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--level", type=int, default=20, help="mesh-3D-<level>-equivalent (5, 10, 20, 40)")
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="skip the end-to-end region (large meshes on a short GPU budget)")
    ap.add_argument("--precision", type=int, default=0,
                    help="storage of the packed operator inside the velocity polynomial: 16, 32 (or 64: the fp64 values); 0 = library default")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the solution and solve status of the last timed step to DIR/<name>.npy (float64, < 64 MB)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the GPU arm's solution; it does not apply to --impl reference")
    sys.dont_write_bytecode = True          # bench.py writes nothing into the source tree, bytecode caches of its imports included

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if rank == 0:
            reference_arm(args)
        return

    # Everything but the final JSON line goes to stderr -- including what C libraries (NCCL's version
    # banner) write to file descriptor 1.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    import torch
    import nsb200 as nsb
    dist = None
    uid = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        torch.cuda.set_device(local_rank)
        holder = [nsb.Device.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(holder, src=0)
        uid = holder[0]
    torch.cuda.set_device(local_rank)

    # ---- setup (not timed): mesh, DoFs, constraints on the host; structure upload
    if rank == 0:
        mesh_file = get_mesh_file(args.level)
    if world > 1:
        dist.barrier()
    mesh_file = get_mesh_file(args.level)
    if args.level >= 40:
        import psutil
        need = 30e9 * max(1, world)        # measured: about 25 GB of host memory per rank at mesh-3D-40 (global mesh + DoF maps per rank)
        avail = psutil.virtual_memory().available
        if avail < need:
            raise SystemExit("[bench] mesh-3D-%d needs about %.0f GB of host memory for %d ranks, %.0f GB available" % (args.level, need / 1e9, world, avail / 1e9))
    t0 = time.time()
    hs = nsb.HostSetup(mesh_file, 3)
    pts, cells = hs.mesh()
    cell_dofs = hs.cell_dofs()
    sp_pts, comp = hs.support_points()
    cdofs, cvals = hs.constraints(CASE, 1.0)
    n_u, n_p, N = hs.n_u, hs.n_p, hs.n_dofs
    log("[bench] rank %d host setup %.1f s: %d cells, %d + %d DoFs" % (rank, time.time() - t0, hs.n_cells, n_u, n_p))
    dev = nsb.Device(3, local_rank)
    if args.precision:
        dev.set_solver_opts(precond_precision=args.precision)
    part = None
    if world > 1:
        dev.comm_init(rank, world, uid)
        part = (np.arange(hs.n_cells, dtype=np.int64) * world // hs.n_cells).astype(np.int32)
    t0 = time.time()
    dev.upload_mesh(pts, cells, cell_dofs, n_u, n_p, part)
    nrows, nnz, nc = dev.sizes()
    log("[bench] rank %d structure + upload %.1f s: %d rows, %d nnz" % (rank, time.time() - t0, nrows, nnz))
    nnz_global = nnz
    if world > 1:
        t_nnz = torch.tensor([nnz], dtype=torch.int64, device="cuda")
        dist.all_reduce(t_nnz)
        nnz_global = int(t_nnz.item())
    un, unm1 = synthetic_state(sp_pts, comp, n_u)
    del pts, cells, cell_dofs, sp_pts, comp        # the device (and the host class) hold what they need
    dev.set_constraints(cdofs, cvals)
    dev.set_params(0.01, 0.5, 1e-3, 1.0, 0.1, True, False)
    dev.set_vector(nsb.NSB_SOLUTION_OLD, un)
    dev.set_vector(nsb.NSB_SOLUTION_OLD_OLD, unm1)
    dev.assemble_linearized()
    t0 = time.time()
    dev.assemble_pressure_matrices()
    log("[bench] pressure matrices + multigrid setup %.1f s" % (time.time() - t0))

    def sync_all():
        dev.synchronize()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def step_resident():
        dev.assemble_linearized()
        return dev.solve(200, 1e-2, 150)

    def step_e2e():
        dev.set_vector(nsb.NSB_SOLUTION_OLD, un)
        dev.set_vector(nsb.NSB_SOLUTION_OLD_OLD, unm1)
        dev.set_constraints(cdofs, cvals)
        dev.assemble_linearized()
        r = dev.solve(200, 1e-2, 150)
        dev.get_vector(nsb.NSB_SOLUTION, sol_host)
        return r

    sol_host = np.zeros(N)
    for _ in range(args.warmup):
        ok, its, res = step_resident()
    if args.warmup:
        log("[bench] warm-up done: converged %s, %d GMRES iterations, %s" % (ok, its, dev.solver_info()))

    # ---- timed region 1: inputs resident in HBM, per-kernel CUDA-event profile on the library's stream
    sampler = ClockSampler(local_rank)
    sampler.start()
    dev.profile_enable(True)
    dev.profile_reset()
    launches0 = dev.launch_count()
    sync_all()
    dev.timer_start()
    iters = []
    for _ in range(args.steps):
        ok, its, res = step_resident()
        iters.append(its)
    ms = dev.timer_stop()
    sync_all()
    launches = dev.launch_count() - launches0
    log("[bench] rank %d timed region done: %.1f ms for %d steps" % (rank, ms, args.steps))
    prof = dev.profile()
    dev.profile_enable(False)
    if args.dump_outputs:
        sol = dev.get_vector(nsb.NSB_SOLUTION)       # collective across ranks: every rank receives the full vector
        if rank == 0:
            dump_outputs(args.dump_outputs, sol, n_u, ok, its, res)
        del sol
    t_res = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t_res, op=dist.ReduceOp.MAX)
    ms = float(t_res.item())
    # ---- timed region 2: end to end through the C ABI with host buffers
    ms_e2e = float("nan")
    if not args.quick:
        step_e2e()
        sync_all()
        dev.timer_start()
        for _ in range(args.steps):
            step_e2e()
        ms_e2e = dev.timer_stop()
        sync_all()
    log("[bench] rank %d e2e region done: %.1f ms" % (rank, ms_e2e))
    t_e = torch.tensor([ms_e2e], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
    ms_e2e = float(t_e.item())
    sampler.stop_flag = True
    sampler.join(timeout=2)

    if rank == 0:
        peak, peak_src = measured_peak()
        tot = {k: v[0] for k, v in prof.items()}
        dom = max(("spmv_vel", "spmv", "asm_rows", "orth"), key=lambda k: tot.get(k, 0.0))
        blocks = dev.block_nnz()
        opts_eff = dev.get_solver_opts()
        vop = dev.velocity_operator_info()
        # Bytes per launch, two conventions (DESIGN.md section 3):
        #  * "performed": what the operation has to move AS IT IS PERFORMED -- the stored operator (packed fp32 / fp16 copy for
        #    the velocity block, fp64 values for A), its compressed index side, and each vector once;
        #  * "csr": SURVEY 8(d)'s figure for a textbook fp64 CSR SpMV (12 B per non-zero + vectors), kept for reference only.
        n_loc_u = n_u if world == 1 else int(nrows * n_u / N)      # owned velocity rows (exact on one GPU)
        vec_vel = (8 + 8 + 8 + 16) * n_loc_u              # x read, y write, u read, poly read + write
        bytes_perf = {
            "spmv_vel": (vop["value_bytes"] + vop["index_bytes"] if vop["precision"] != 64 else 8 * blocks["uu"] + 2 * blocks["uu"] // 9) + vec_vel,
            "spmv": 8 * nnz + 2 * (blocks["uu"] // 9 + blocks["up"]) + 32 * (nrows // 3) + 16 * nrows,
            "asm_rows": 8 * nnz + 8 * nrows + 8 * 3 * 4 * nc + 20 * 34 * nc,
        }
        bytes_csr = {
            "spmv_vel": 12 * blocks["uu"] + 16 * n_loc_u + 4 * (n_loc_u + 1),
            "spmv": 12 * nnz + 16 * nrows + 4 * (nrows + 1),
            "asm_rows": 8 * nnz + 8 * nrows + 8 * 3 * 4 * nc + 20 * 34 * nc,
        }
        kernels = {}
        for k, (t_ms, n) in prof.items():
            if n:
                kernels[k] = {"ms_total": round(t_ms, 3), "launches": n, "ms_avg": round(t_ms / n, 4)}
        prec = opts_eff["precond_precision"]
        line = {
            "metric": "time-steps/s", "value": args.steps / (ms * 1e-3), "unit": "steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None,
            "dtype": "f64" + (" (fp%d operator copy inside the velocity preconditioner)" % prec if prec != 64 else ""),
            "data": "synthetic",
            "config": {"workload": workload_name(args.level, hs.n_cells, N, nnz_global),
                       "parallelism": "1 process per GPU, contiguous cell chunks" if world > 1 else "single GPU",
                       "l2": "inputs (%.1f GB of matrix values) exceed L2; no flush needed" % (8e-9 * nnz),
                       "gmres_iterations_per_step": iters,
                       "solver": dict(dev.solver_info(), velocity_operator="packed fp%d copy of Dinv F, TMA-streamed" % prec if prec != 64 else "assembled fp64 values",
                                      velocity_operator_bytes=vop, velocity_preconditioner=dev.velocity_pc_info()),
                       "comm": dev.comm_info()},
            "gpu_launches": int(launches),
            "clocks": sampler.summary(),
            "e2e": {"value": (args.steps / (ms_e2e * 1e-3)) if ms_e2e == ms_e2e else None, "unit": "steps/s", "h2d_bytes_per_step": int(2 * 8 * N + 12 * cdofs.size),
                    "d2h_bytes_per_step": int(8 * N)},
            "kernels": kernels,
        }
        for k in ("spmv_vel", "spmv", "asm_rows"):
            if k in kernels:
                kernels[k]["performed_GBps"] = round(bytes_perf[k] / (kernels[k]["ms_avg"] * 1e-3) / 1e9, 1)
                kernels[k]["frac_of_peak"] = round(kernels[k]["performed_GBps"] / peak, 3)
        if "asm_rows" in kernels:
            t_asm = sum(kernels[k]["ms_avg"] for k in ("asm_context", "asm_rows", "asm_pack") if k in kernels)
            kernels["asm_rows"]["all_passes_ms"] = round(t_asm, 3)
            kernels["asm_rows"]["all_passes_frac_of_peak"] = round(bytes_perf["asm_rows"] / (t_asm * 1e-3) / 1e9 / peak, 3)
        # roofline of the dominant kernel
        if dom in kernels and bytes_perf.get(dom):
            ach = bytes_perf[dom] / (kernels[dom]["ms_avg"] * 1e-3) / 1e9
            tr = recorded_traffic(args.level, dom, prec) if world == 1 else None
            line["roofline"] = {"kernel": dom, "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                                "traffic": tr, "peak_source": peak_src,
                                "bytes_per_launch": int(bytes_perf[dom]),
                                "bytes_convention": "operation as performed: stored operator (packed fp%s values + metadata) + each vector once" % prec,
                                "frac_csr_convention": bytes_csr[dom] / (kernels[dom]["ms_avg"] * 1e-3) / 1e9 / peak}
            if tr:
                line["roofline"]["dram_GBps"] = tr / (kernels[dom]["ms_avg"] * 1e-3) / 1e9
                line["roofline"]["dram_frac"] = line["roofline"]["dram_GBps"] / peak
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline_for(args.level, hs.n_cells)
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    dev.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
