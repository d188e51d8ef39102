"""Multi-GPU validation (one process per GPU, launch with torchrun): every rank's owned rows of the
assembled matrix / rhs against the oracle and -- bit for bit -- against a single-GPU assembly of the same system,
the tight-tolerance solve against a sparse direct solve, the iteration count at the reference tolerance
(partition-independent preconditioner), and three time steps of the C++ host class NavierStokes<3>(make_3D_2Z)
(BASELINE config 3, "1 vs 2 GPUs") with per-rank VTU pieces.  --forcing adds a body force everywhere: each rank
samples it at its own local cells' quadrature points (owned + ghost layer), the oracle at its own, and the host class
takes it through HostSolver.set_forcing.  --forcing-source does the same with the force given as CUDA source: every rank
compiles it and evaluates it on the device at its own local cells (ghost layer included), and the slots are compared bit
for bit with the single-GPU ones, cell by cell.
  python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 tools/gpu_multi.py [--json out.json] [--forcing | --forcing-source]
tests/test_gpu_multirank.py and tests/test_gpu_forcing.py run this under pytest and assert on the JSON."""
import argparse
import json
import os
import sys
import tempfile
import xml.etree.ElementTree as ET

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from oracle import assemble as asm, dofs as odofs, postprocess as pp, solve as osolve  # noqa: E402
import nsb200 as nsb  # noqa: E402
from tests.conftest import synthetic_state  # noqa: E402
from tests.forcing_cases import ForcedOracle, quadrature_points, sample, smooth_forcing  # noqa: E402
from tests.forcing_sources import SMOOTH  # noqa: E402
from tools import meshgen, msh  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--json", default=None)
    ap.add_argument("--lc", type=float, default=0.04)
    ap.add_argument("--part", default="chunks", help="cell partition: chunks (contiguous) or metis (face-dual graph, like the reference)")
    ap.add_argument("--forcing", action="store_true", help="assemble and step with a non-zero body force")
    ap.add_argument("--forcing-source", action="store_true", help="the same body force as CUDA source evaluated on each GPU")
    args = ap.parse_args()
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    holder = [nsb.Device.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(holder, src=0)
    mesh = meshgen.mesh_3d(lc_cyl=args.lc, lc_global=0.15)
    dm = odofs.enumerate_dofs(mesh)
    pat = odofs.make_sparsity(dm)
    N = dm.n_dofs
    tc = pp.TEST_CASES["3D-2Z"]
    con = odofs.build_constraints(mesh, dm, pp.inlet_profile(3, tc["U_m"], False, 4.0, 1.0), pp.boundary_ids(3))
    un, unm1 = synthetic_state(dm, 3, tc["U_m"])
    p = asm.Params(dt=0.01, theta=0.5, nu=1e-3, use_supg=True)
    t_new, t_old = 1.0, 0.99
    forced = args.forcing or args.forcing_source
    forcing = None
    if forced:
        qp = quadrature_points(mesh)
        forcing = (sample(smooth_forcing, qp, t_new), sample(smooth_forcing, qp, t_old))
    ref = asm.assemble(mesh, dm, pat, p, con, "linearized", un, unm1, forcing=forcing) if rank == 0 else None
    holder2 = [ref]
    dist.broadcast_object_list(holder2, src=0)
    ref = holder2[0]

    def setup(dev, part):
        dev.upload_mesh(mesh.points, mesh.cells, dm.cell_dofs, dm.n_u, dm.n_p, part)
        if args.forcing:
            qd = dev.quadrature_points()
            dev.set_forcing(sample(smooth_forcing, qd, t_new), sample(smooth_forcing, qd, t_old))
        elif args.forcing_source:
            dev.set_forcing_source(SMOOTH)
            dev.eval_forcing(nsb.NSB_FORCING_NEW, t_new)
            dev.eval_forcing(nsb.NSB_FORCING_OLD, t_old)
        dev.set_constraints(con.dofs, con.val[con.dofs])
        dev.set_params(0.01, 0.5, 1e-3, 1.0, 0.1, True, False)
        dev.set_vector(nsb.NSB_SOLUTION_OLD, un)
        dev.set_vector(nsb.NSB_SOLUTION_OLD_OLD, unm1)
        dev.assemble_linearized()

    # single-GPU assembly of the same system on this rank's device (no communicator): the bit-exactness reference
    one = nsb.Device(3, local)
    setup(one, None)
    vals1 = one.matrix_values()
    rp1, _ = one.pattern()
    b1 = one.get_vector(nsb.NSB_RHS)
    if args.forcing_source:
        # the single-GPU slots, cells keyed by their quadrature points (bit-identical on every rank: same vertices, same
        # operations), so that each rank's local cells can be matched to them
        q1 = one.quadrature_points()
        fn1, fo1 = one.forcing(nsb.NSB_FORCING_NEW), one.forcing(nsb.NSB_FORCING_OLD)
        slots1 = {q1[k].tobytes(): k for k in range(q1.shape[0])}
    one.assemble_pressure_matrices()
    ok1, it1, _ = one.solve(200, 1e-2, 150)
    one.close()

    dev = nsb.Device(3, local)
    dev.comm_init(rank, world, holder[0])
    part = (np.arange(mesh.n_cells, dtype=np.int64) * world // mesh.n_cells).astype(np.int32)
    if args.part == "metis":
        tmpm = tempfile.mkdtemp(prefix="nsb_part_%d_" % rank)
        msh.write_bin(tmpm + "/m.bin", mesh)
        hsu = nsb.HostSetup(tmpm + "/m.bin", 3)
        part = hsu.partition(world, 1)
        hsu.close()
    setup(dev, part)
    nrows, nnz, nc = dev.sizes()
    rp, col = dev.pattern()
    gid = dev.row_gids()
    vals = dev.matrix_values()
    orp, ocol = pat
    errA = 0.0
    okpat, bitexact = True, True
    for k in range(nrows):
        g = gid[k]
        okpat &= np.array_equal(col[rp[k]:rp[k + 1]].astype(np.int64), ocol[orp[g]:orp[g + 1]].astype(np.int64))
        errA = max(errA, np.abs(vals[rp[k]:rp[k + 1]] - ref.A[orp[g]:orp[g + 1]]).max())
        bitexact &= np.array_equal(vals[rp[k]:rp[k + 1]], vals1[rp1[g]:rp1[g + 1]])
    errA /= np.abs(ref.A).max()
    b = dev.get_vector(nsb.NSB_RHS)
    errb = np.abs(b - ref.b).max() / np.abs(ref.b).max()
    b_bitexact = bool(np.array_equal(b, b1))
    slots_bitexact = None
    if args.forcing_source:
        qd, fnd, fod = dev.quadrature_points(), dev.forcing(nsb.NSB_FORCING_NEW), dev.forcing(nsb.NSB_FORCING_OLD)
        idx = [slots1.get(qd[k].tobytes(), -1) for k in range(qd.shape[0])]
        slots_bitexact = bool(min(idx) >= 0 and np.array_equal(fnd, fn1[idx]) and np.array_equal(fod, fo1[idx]))
    dev.assemble_pressure_matrices()
    ok, it, res = dev.solve(200, 1e-2, 150)
    ok2, it2, _ = dev.solve(3000, 1e-12, 150)
    xs = dev.get_vector(nsb.NSB_SOLUTION)
    A = asm.to_csr(pat, ref.A, N)
    xd = con.distribute(osolve.direct_solve(A, ref.b))
    ferr = float(np.linalg.norm(xs - xd) / np.linalg.norm(xd))
    rec = dict(rank=rank, world=world, rows=int(nrows), cells=int(nc), pattern_ok=bool(okpat), A_relerr=float(errA),
               A_bitexact_vs_1gpu=bool(bitexact), b_relerr=float(errb), b_bitexact_vs_1gpu=b_bitexact,
               gmres_ok=bool(ok), gmres_its=int(it), gmres_its_1gpu=int(it1), tight_ok=bool(ok2), tight_its=int(it2),
               field_relerr_vs_direct=ferr, slots_bitexact_vs_1gpu=slots_bitexact, fused=os.environ.get("NSB200_FUSED_HALO", "0"), halo=os.environ.get("NSB200_HALO", "p2p"))
    print("[rank %d/%d] " % (rank, world) + json.dumps(rec), flush=True)
    dist.barrier()
    dev.close()

    # ---- the C++ host class NavierStokes<3>(make_3D_2Z) on `world` GPUs: three time steps in parity mode
    tmp = [tempfile.mkdtemp(prefix="nsb_multi_") if rank == 0 else None]
    dist.broadcast_object_list(tmp, src=0)
    outdir = tmp[0] + "/"
    path = outdir + "mesh_%d.bin" % rank
    msh.write_bin(path, mesh)
    holder3 = [nsb.Device.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(holder3, src=0)
    hs = nsb.HostSolver("3D-2Z", path, device=local, rank=rank, nranks=world, nccl_unique_id=holder3[0], gmres_tolerance=1e-12,
                        write_vtu=True, output_dir=outdir, partitioner=1 if args.part == "metis" else 0)
    if args.forcing:
        hs.set_forcing(smooth_forcing)
    elif args.forcing_source:
        hs.set_forcing_source(SMOOTH)
    hs.initialize()
    infos = [hs.step() for _ in range(3)]
    steps = []
    if rank == 0:
        o = ForcedOracle(mesh, "3D-2Z", smooth_forcing, solver="direct") if forced else osolve.Oracle(mesh, "3D-2Z", solver="direct")
        for k, info in enumerate(infos):
            ref_ = o.step()
            errs = {key: abs(info[key] - ref_[key]) / max(abs(ref_[key]), 1e-300) for key in ("cd", "cl", "dp")}
            steps.append(dict(step=k + 1, gmres=info["gmres_iterations"], cd=info["cd"], cl=info["cl"], dp=info["dp"],
                              cl_abs=abs(ref_["cl"]), **{"err_" + a: b for a, b in errs.items()}))
        x = hs.solution()
        field = float(np.linalg.norm(x - o.current_solution) / np.linalg.norm(o.current_solution))
    dist.barrier()
    hs.close()
    recs = [None] * world
    dist.all_gather_object(recs, rec)
    if rank == 0:
        # per-rank VTU pieces: every rank's file exists, the .pvtu lists them all, owned cells sum to the mesh
        pv = ET.parse(outdir + "solution_0003.pvtu").getroot()
        pieces = [e.get("Source") for e in pv.iter("Piece")]
        ncell = 0
        for src in pieces:
            piece = ET.parse(outdir + src).getroot().find("UnstructuredGrid/Piece")
            ncell += int(piece.get("NumberOfCells"))
        summary = dict(world=world, partition=args.part, forcing=bool(args.forcing), forcing_source=bool(args.forcing_source), fused=os.environ.get("NSB200_FUSED_HALO", "0"), halo=os.environ.get("NSB200_HALO", "p2p"), mesh_cells=int(mesh.n_cells), n_dofs=int(N),
                       ranks=recs, host_class_steps=steps, host_class_field_relerr=field, vtu_pieces=pieces, vtu_cells_total=ncell)
        print("[summary] " + json.dumps(summary), flush=True)
        if args.json:
            with open(args.json, "w") as f:
                json.dump(summary, f, indent=1)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
