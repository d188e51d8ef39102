"""What a forcing term costs on the GPU path, at a size a user would run (default mesh-3D-20, 3D-2Z).

1. The assembly's first pass (`asm_context`, CUDA events through nsb_profile_*): per launch without forcing and with
   forcing (f_new != f_old), in alternating blocks so that drift of the shared machine shows up as spread, not as a
   difference.  The unforced blocks also show that the default path is untouched: its time is compared with the spread of
   its own repeats.
2. The host side of one slot through the C ABI: exporting the quadrature points, evaluating a simple analytic forcing with
   numpy and uploading it (nsb_set_forcing).
3. The same forcing as CUDA source evaluated on the device (nsb_set_forcing_source): NVRTC compile time without a GPU
   (nsb_check_forcing_source) and the first set (compile, load, geometry upload); the `forcing` kernel's time per slot
   from CUDA events, and the bytes it writes per second as a share of a device-to-device copy's bandwidth measured in the
   same run (torch copy of 2 x 2 GB buffers, larger than L2: read + write bytes over time).
4. The host class (NavierStokes<3> through HostSolver): unforced, with the Python callback (HostSolver.set_forcing) and
   with the source (set_forcing_source): the per-step time the step reports for the forcing (StepInfo::forcing_seconds),
   next to the step's wall time.
The card's name and power limit are read in the same run.
  python tools/gpu_forcing_cost.py [--level 20] [--rounds 5] [--launches 5] [--steps 2] [--evals 20] [--json out.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import postprocess as pp  # noqa: E402
from tools.gpu_check import load_nsb  # noqa: E402


def analytic_forcing(x, t):
    """A body force in the flow direction that varies across the channel and in time."""
    f = np.zeros_like(x)
    f[:, 2] = (1.0 + 0.5 * np.sin(t)) * np.sin(np.pi * x[:, 0] / 0.41) * np.sin(np.pi * x[:, 1] / 0.41)
    return f


# analytic_forcing as CUDA source (M_PI is not defined in NVRTC's built-ins)
ANALYTIC_SRC = r"""
__device__ void nsb_forcing(const double* x, double t, const double* prm, double* f) {
  const double pi = 3.141592653589793;
  f[2] = (1.0 + 0.5 * sin(t)) * sin(pi * x[0] / 0.41) * sin(pi * x[1] / 0.41);
}
"""


def copy_bandwidth(nbytes=2 << 30, reps=10):
    """Device-to-device copy: (read + write bytes) / time, CUDA events, buffers much larger than L2."""
    import torch
    a = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    for _ in range(2):
        b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        b.copy_(a)
    e1.record()
    e1.synchronize()
    return 2.0 * nbytes * reps / (e0.elapsed_time(e1) * 1e-3)


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--level", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--launches", type=int, default=5)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--evals", type=int, default=20, help="timed nsb_eval_forcing calls per slot")
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    nsb = load_nsb()
    import bench
    out = dict(card=card(), level=args.level)
    print("card:", out["card"], flush=True)
    mesh_file = bench.get_mesh_file(args.level)
    hs = nsb.HostSetup(mesh_file, 3)
    pts, cells = hs.mesh()
    sp_pts, comp = hs.support_points()
    cd, cvals = hs.constraints("3D-2Z", 1.0)
    tc = pp.TEST_CASES["3D-2Z"]
    nu = pp.viscosity(3, tc["U_m"], tc["Re"])
    dev = nsb.Device(3)
    dev.upload_mesh(pts, cells, hs.cell_dofs(), hs.n_u, hs.n_p)
    _, _, nc = dev.sizes()
    out.update(cells=int(nc), dofs=int(hs.n_dofs))
    dev.set_constraints(cd, cvals)
    un, unm1 = bench.synthetic_state(sp_pts, comp, hs.n_u)
    dev.set_params(0.01, 0.5, nu, 1.0, 0.1, True, False)
    dev.set_vector(nsb.NSB_SOLUTION_OLD, un)
    dev.set_vector(nsb.NSB_SOLUTION_OLD_OLD, unm1)

    # ---- host side of the C ABI path: points, numpy evaluation, upload (one slot)
    t0 = time.perf_counter()
    q = dev.quadrature_points()
    t1 = time.perf_counter()
    flat = q.reshape(-1, 3)
    f_new = analytic_forcing(flat, 1.0).reshape(q.shape)
    t2 = time.perf_counter()
    f_old = analytic_forcing(flat, 0.99).reshape(q.shape)
    dev.set_forcing(f_new, None)
    dev.clear_forcing()
    t3 = time.perf_counter()
    dev.set_forcing(f_new, f_old)
    dev.synchronize()
    t4 = time.perf_counter()
    dev.clear_forcing()
    out["c_abi_host"] = dict(points=q.shape[0] * q.shape[1], quadrature_points_s=t1 - t0, numpy_eval_per_slot_s=t2 - t1,
                             upload_two_slots_s=t4 - t3, bytes_per_slot=int(f_new.nbytes))
    print("C ABI host side:", json.dumps(out["c_abi_host"]), flush=True)

    # ---- asm_context with and without forcing, alternating blocks
    for _ in range(2):                                   # warm both instantiations
        dev.assemble_linearized()
        dev.set_forcing(f_new, f_old)
        dev.assemble_linearized()
        dev.clear_forcing()
    dev.synchronize()
    per = {"none": [], "forced": []}
    dev.profile_enable(True)
    for r in range(args.rounds):
        for mode in ("none", "forced"):
            if mode == "forced":
                dev.set_forcing(f_new, f_old)
            dev.synchronize()
            dev.profile_reset()
            for _ in range(args.launches):
                dev.assemble_linearized()
            dev.synchronize()
            ms, n = dev.profile()["asm_context"]
            per[mode].append(ms / n)
            if mode == "forced":
                dev.clear_forcing()
    dev.profile_enable(False)
    out["asm_context_ms"] = {k: dict(blocks=v, median=float(np.median(v)), min=float(min(v)), max=float(max(v))) for k, v in per.items()}
    extra = 2 * f_new.nbytes
    out["forcing_bytes_per_assembly"] = int(extra)
    print("asm_context per launch [ms]:", json.dumps(out["asm_context_ms"]), flush=True)
    print("extra bytes read per assembly: %.2f GB" % (extra / 1e9), flush=True)

    # ---- the same forcing evaluated on the device from CUDA source
    t0 = time.perf_counter()
    nsb.check_forcing_source(3, ANALYTIC_SRC)
    t1 = time.perf_counter()
    dev.set_forcing_source(ANALYTIC_SRC)
    t2 = time.perf_counter()
    for which, t in ((nsb.NSB_FORCING_NEW, 1.0), (nsb.NSB_FORCING_OLD, 0.99)):       # warm
        dev.eval_forcing(which, t)
    fd = dev.forcing(nsb.NSB_FORCING_NEW)
    dev_err = float(np.abs(fd - f_new).max() / np.abs(f_new).max())
    dev.profile_enable(True)
    dev.profile_reset()
    t3 = time.perf_counter()
    for k in range(args.evals):
        dev.eval_forcing(k % 2, 1.0 - 0.01 * (k % 2))
    t4 = time.perf_counter()
    ms, n = dev.profile()["forcing"]
    dev.profile_enable(False)
    bw = copy_bandwidth()
    kernel_ms = ms / n
    written = int(f_new.nbytes)
    out["device_source"] = dict(nvrtc=dev.forcing_info()["nvrtc"], compile_only_s=t1 - t0, first_set_s=t2 - t1,
                                kernel_ms_per_slot=kernel_ms, eval_call_s_per_slot=(t4 - t3) / args.evals,
                                bytes_written_per_slot=written, write_rate_GBps=written / (kernel_ms * 1e-3) / 1e9,
                                copy_bandwidth_GBps=bw / 1e9, share_of_copy_bandwidth=written / (kernel_ms * 1e-3) / bw,
                                max_rel_err_vs_numpy=dev_err)
    print("device source:", json.dumps(out["device_source"]), flush=True)
    dev.set_forcing_source(None)
    dev.close()

    # ---- the host class: evaluation + upload per step
    steps = {}
    for mode in ("none", "callback", "source"):
        s = nsb.HostSolver("3D-2Z", mesh_file)
        if mode == "callback":
            s.set_forcing(analytic_forcing)
        elif mode == "source":
            s.set_forcing_source(ANALYTIC_SRC)
        s.initialize()
        infos = [s.step() for _ in range(args.steps)]
        steps[mode] = [dict(wall_s=i["wall_seconds"], forcing_s=i["forcing_seconds"], gmres=i["gmres_iterations"]) for i in infos]
        s.close()
    out["host_class_steps"] = steps
    print("host class steps:", json.dumps(steps), flush=True)
    out["card_after"] = card()
    if args.json:
        with open(args.json, "w") as fh:
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
