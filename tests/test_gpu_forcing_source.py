"""GPU (-m gpu): the forcing term evaluated on the device from CUDA source (nsb_set_forcing_source / nsb_eval_forcing,
DeviceForcing through HostSolver.set_forcing_source), against the quadrature points, numpy, the host-supplied slots, the
oracle and the manufactured solution of tests/forcing_cases.py.  The CUDA twins live in tests/forcing_sources.py.
Tolerances: slots of f = x bit-identical to the exported points; smooth twin 1e-14 max|f| (libm vs CUDA math, FMA
contraction in the user's code); assembled A and b bit-identical to the same slots uploaded from the host and 1e-12
(max-norm scaled) from the oracle; manufactured and trajectory bounds as in test_gpu_forcing.py."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import assemble as asm, dofs as odofs
from tests.conftest import GOLDEN, ROOT
from tests.forcing_cases import ForcedOracle, Manufactured, quadrature_points, sample, smooth_forcing
from tests.forcing_sources import IDENTITY, MANUFACTURED, SCALED, SMOOTH, ZERO, manufactured_params
from tests.test_gpu_multirank import _free_port, _ngpus
from tests.test_gpu_parity import TOL_ASM, TOL_FIELD, TOL_FORCE, Case, relmax
from tools import msh

pytestmark = pytest.mark.gpu

T_NEW = 1.0


@pytest.fixture(scope="module")
def fcase2d(nsb, golden_mesh):
    c = Case(nsb, golden_mesh("mesh-2D"), "2D-2")
    yield c
    c.dev.close()


@pytest.fixture(scope="module")
def fcase3d(nsb, small_3d_mesh):
    c = Case(nsb, small_3d_mesh, "3D-2Z")
    yield c
    c.dev.close()


def _eval_both(c, src=SMOOTH, params=()):
    nsb = c.nsb
    c.dev.set_forcing_source(src, params)
    c.dev.eval_forcing(nsb.NSB_FORCING_NEW, T_NEW)
    c.dev.eval_forcing(nsb.NSB_FORCING_OLD, T_NEW - c.dt)


def _oracle_forcing(c):
    q = quadrature_points(c.mesh)
    return sample(smooth_forcing, q, T_NEW), sample(smooth_forcing, q, T_NEW - c.dt)


@pytest.mark.parametrize("which", ["2d", "3d"])
def test_identity_source_reproduces_the_quadrature_points(fcase2d, fcase3d, which):
    c = fcase2d if which == "2d" else fcase3d
    nsb = c.nsb
    try:
        c.dev.set_forcing_source(IDENTITY)
        for slot in (nsb.NSB_FORCING_NEW, nsb.NSB_FORCING_OLD):
            c.dev.eval_forcing(slot, 0.25)
            f = c.dev.forcing(slot)
            pts = c.dev.quadrature_points()
            assert f.shape == pts.shape
            assert np.array_equal(f.view(np.uint64), pts.view(np.uint64))
    finally:
        c.dev.set_forcing_source(None)


@pytest.mark.parametrize("which", ["2d", "3d"])
def test_smooth_twin_matches_numpy(fcase2d, fcase3d, which):
    c = fcase2d if which == "2d" else fcase3d
    nsb = c.nsb
    pts = c.dev.quadrature_points()
    try:
        c.dev.set_forcing_source(SMOOTH)
        for t in (0.0, 1.37):
            c.dev.eval_forcing(nsb.NSB_FORCING_NEW, t)
            f, ref = c.dev.forcing(nsb.NSB_FORCING_NEW), sample(smooth_forcing, pts, t)
            err = np.abs(f - ref).max() / np.abs(ref).max()
            print("%s t=%.2f: max error %.2e of max|f|" % (which, t, err))
            assert err <= 1e-14
    finally:
        c.dev.set_forcing_source(None)


@pytest.mark.parametrize("which", ["2d", "3d"])
@pytest.mark.parametrize("theta,first_order", [(0.5, False), (1.0, True), (0.5, True)])
def test_linearized_assembly_device_slots_vs_uploaded(fcase2d, fcase3d, which, theta, first_order):
    c = fcase2d if which == "2d" else fcase3d
    nsb = c.nsb
    con = c.constraints()
    try:
        _eval_both(c)
        p = c.linearized(theta, first_order, con)
        A1, b1 = c.dev.matrix_values(), c.dev.get_vector(nsb.NSB_RHS)
        fn, fo = c.dev.forcing(nsb.NSB_FORCING_NEW), c.dev.forcing(nsb.NSB_FORCING_OLD)
        c.dev.set_forcing_source(None)
        c.dev.set_forcing(fn, fo)
        c.linearized(theta, first_order, con)
        A2, b2 = c.dev.matrix_values(), c.dev.get_vector(nsb.NSB_RHS)
    finally:
        c.dev.set_forcing_source(None)
        c.dev.clear_forcing()
    assert np.array_equal(A1, A2) and np.array_equal(b1, b2)
    ref = asm.assemble(c.mesh, c.dm, c.pat, p, con, "linearized", c.un, c.unm1, with_pressure_matrices=False,
                       forcing=_oracle_forcing(c))
    assert relmax(A1, ref.A) < TOL_ASM and relmax(b1, ref.b) < TOL_ASM


@pytest.mark.parametrize("which", ["2d", "3d"])
def test_newton_assembly_device_slots_vs_uploaded(fcase2d, fcase3d, which):
    c = fcase2d if which == "2d" else fcase3d
    nsb = c.nsb
    con = c.constraints(homogeneous=True)
    pk = np.zeros(c.dm.n_dofs)
    pk[c.dm.n_u:] = 0.05 * np.random.default_rng(7).uniform(-1, 1, c.dm.n_p)
    cur = c.un + pk

    def assemble(theta):
        c.dev.set_params(c.dt, theta, c.nu, 1.0, 0.1, c.tc["supg"], False)
        c.dev.set_vector(nsb.NSB_CURRENT_SOLUTION, cur)
        c.dev.set_vector(nsb.NSB_SOLUTION_OLD, c.unm1)
        c.dev.assemble_newton()
        return c.dev.matrix_values(), c.dev.get_vector(nsb.NSB_RHS)

    try:
        for theta in (1.0, 0.5):
            _eval_both(c)
            A1, b1 = assemble(theta)
            fn, fo = c.dev.forcing(nsb.NSB_FORCING_NEW), c.dev.forcing(nsb.NSB_FORCING_OLD)
            c.dev.set_forcing_source(None)
            c.dev.set_forcing(fn, fo)
            A2, b2 = assemble(theta)
            c.dev.clear_forcing()
            assert np.array_equal(A1, A2) and np.array_equal(b1, b2)
            p = asm.Params(dt=c.dt, theta=theta, nu=c.nu, use_supg=c.tc["supg"])
            ref = asm.assemble(c.mesh, c.dm, c.pat, p, con, "newton", cur, c.unm1, with_pressure_matrices=False,
                               forcing=_oracle_forcing(c))
            assert relmax(A1, ref.A) < TOL_ASM and relmax(b1, ref.b) < TOL_ASM
    finally:
        c.dev.set_forcing_source(None)
        c.dev.clear_forcing()


@pytest.mark.parametrize("which", ["2d", "3d"])
def test_zero_source_and_unload_are_bit_identical_to_none(nsb, golden_mesh, small_3d_mesh, which):
    mesh = golden_mesh("mesh-2D") if which == "2d" else small_3d_mesh
    case = "2D-2" if which == "2d" else "3D-2Z"
    ref, c = Case(nsb, mesh, case), Case(nsb, mesh, case)

    def assemble(cc):
        cc.linearized(0.5, False, cc.constraints())
        return cc.dev.matrix_values(), cc.dev.get_vector(nsb.NSB_RHS)

    A0, b0 = assemble(ref)
    _eval_both(c)
    A1, b1 = assemble(c)
    assert np.array_equal(A1, A0) and not np.array_equal(b1, b0)
    _eval_both(c, ZERO)                                               # all-zero results clear both slots
    assert not c.dev.forcing(nsb.NSB_FORCING_NEW).any()
    A2, b2 = assemble(c)
    assert np.array_equal(A2, A0) and np.array_equal(b2, b0)
    _eval_both(c)
    n = c.dev.launch_count()
    c.dev.set_forcing_source(None)
    assert c.dev.launch_count() == n                                  # unloading clears without a launch
    assert not c.dev.forcing_info()["has_source"]
    A3, b3 = assemble(c)
    assert np.array_equal(A3, A0) and np.array_equal(b3, b0)
    ref.dev.close()
    c.dev.close()


def test_same_source_compiles_once_and_parameters_need_no_compile(fcase3d):
    c = fcase3d
    nsb = c.nsb
    pts = c.dev.quadrature_points()
    try:
        before = c.dev.forcing_info()
        c.dev.set_forcing_source(SCALED, [2.0, 0.0])
        c.dev.set_forcing_source(SCALED, [2.0, 0.0])
        info = c.dev.forcing_info()
        print("NVRTC %d.%d" % info["nvrtc"])
        assert info["nvrtc"][0] >= 12 and info["has_source"]
        assert info["compiles"] == before["compiles"] + 1
        c.dev.eval_forcing(nsb.NSB_FORCING_NEW, 0.5)
        f1 = c.dev.forcing(nsb.NSB_FORCING_NEW)
        c.dev.set_forcing_source(SCALED, [3.0, 1.0])
        c.dev.eval_forcing(nsb.NSB_FORCING_NEW, 0.5)
        f2 = c.dev.forcing(nsb.NSB_FORCING_NEW)
        info = c.dev.forcing_info()
        assert info["compiles"] == before["compiles"] + 1
        assert info["evaluations"] == before["evaluations"] + 2
        assert np.allclose(f1[..., 0], 2.0 * pts[..., 0], rtol=1e-15, atol=0)
        assert np.allclose(f2[..., 0], 3.0 * pts[..., 0] + 0.5, rtol=1e-15, atol=1e-15)
        assert not f2[..., 1:].any()
        c.dev.set_forcing_source(SMOOTH)
        assert c.dev.forcing_info()["compiles"] == before["compiles"] + 2
    finally:
        c.dev.set_forcing_source(None)


@pytest.mark.parametrize("which", ["2d", "3d"])
def test_manufactured_solution_with_parameters(nsb, golden_mesh, small_3d_mesh, which):
    """As test_manufactured_solution_through_the_library, with the body force evaluated on the device from prm."""
    mesh = golden_mesh("mesh-2D") if which == "2d" else small_3d_mesh
    dim, nu, dt = mesh.dim, 1e-3, 0.02
    dm = odofs.enumerate_dofs(mesh)
    ms = Manufactured(mesh, nu)
    x = ms.exact(dm)
    dev = nsb.Device(dim)
    dev.upload_mesh(mesh.points, mesh.cells, dm.cell_dofs, dm.n_u, dm.n_p)
    dev.set_forcing_source(MANUFACTURED, manufactured_params(ms))

    def forced():
        dev.eval_forcing(nsb.NSB_FORCING_NEW, 0.0)
        dev.eval_forcing(nsb.NSB_FORCING_OLD, -dt)

    forced()
    f = dev.forcing(nsb.NSB_FORCING_NEW)
    ref = sample(ms.forcing, dev.quadrature_points(), 0.0)
    assert np.abs(f - ref).max() <= 1e-13 * np.abs(ref).max()
    con = ms.constraints(dm)
    dev.set_constraints(con.dofs, con.val[con.dofs])
    for theta in (1.0, 0.5):
        forced()
        dev.set_params(dt, theta, nu, 1.0, 0.1, False, True)
        dev.set_vector(nsb.NSB_SOLUTION_OLD, x)
        dev.set_vector(nsb.NSB_SOLUTION_OLD_OLD, x)
        dev.assemble_linearized()
        dev.assemble_pressure_matrices()
        b = dev.get_vector(nsb.NSB_RHS)
        defect = np.linalg.norm(dev.spmv(np.where(con.is_c, 0.0, x)) - b) / np.linalg.norm(b)
        ok, it, _ = dev.solve(2000, 1e-12, 150)
        err = np.linalg.norm(dev.get_vector(nsb.NSB_SOLUTION) - x) / np.linalg.norm(x)
        print("%s linearised theta %.1f: defect %.2e, solve %d its, field error %.2e" % (which, theta, defect, it, err))
        assert defect < 1e-10 and ok and err < 1e-8
    hcon = odofs.build_constraints(mesh, dm, None, ms.ids, homogeneous=True)
    dev.set_constraints(hcon.dofs, hcon.val[hcon.dofs])
    for supg in ((False, True) if dim == 2 else (True,)):
        norms = []
        for on in (True, False):
            forced() if on else dev.clear_forcing()
            dev.set_params(dt, 1.0, nu, 1.0, 0.1, supg, True)
            dev.set_vector(nsb.NSB_CURRENT_SOLUTION, x)
            dev.set_vector(nsb.NSB_SOLUTION_OLD, x)
            dev.assemble_newton()
            norms.append(dev.rhs_norm())
        print("%s Newton SUPG %s: residual ratio %.2e" % (which, supg, norms[0] / norms[1]))
        assert norms[0] <= 1e-9 * norms[1]
    dev.close()


def _trajectory(nsb, case, path, mesh, steps, fail_at=None, fail_solves=0):
    """HostSolver(case) with the smooth source against ForcedOracle(direct, numpy smooth_forcing)."""
    s = nsb.HostSolver(case, path, gmres_tolerance=1e-12)
    s.set_forcing_source(SMOOTH)
    s.initialize()
    o = ForcedOracle(mesh, case, smooth_forcing, solver="direct")
    out = []
    for k in range(steps):
        if k == fail_at:
            s.set_test_fail_solves(fail_solves)
            o.fail_solves = fail_solves
        info, ref = s.step(), o.step()
        for key in ("cd", "cl", "dp"):
            assert abs(info[key] - ref[key]) <= TOL_FORCE * abs(ref[key]) + 1e-12, (case, k, key, info[key], ref[key])
        x = s.solution()
        assert np.linalg.norm(x - o.current_solution) / np.linalg.norm(o.current_solution) < TOL_FIELD, (case, k)
        out.append((info, s.device().forcing_info()))
    s.close()
    return out


def test_host_class_2d2_source_trajectory_with_halved_retry(nsb, golden_mesh, msh_file):
    traj = _trajectory(nsb, "2D-2", msh_file("mesh-2D"), golden_mesh("mesh-2D"), 3, fail_at=2, fail_solves=2)
    assert traj[2][0]["solves"] == 3
    assert traj[0][1]["compiles"] == 1 and traj[-1][1]["compiles"] == 1
    g = np.load(os.path.join(GOLDEN, "oracle_vectors.npz"))["traj_2D2"]            # the unforced trajectory
    assert abs(traj[0][0]["cd"] - g[0][1]) > 1e3 * TOL_FORCE * abs(g[0][1])


def test_host_class_2d1_newton_evaluates_twice_per_step(nsb, golden_mesh, msh_file):
    traj = _trajectory(nsb, "2D-1", msh_file("mesh-2D"), golden_mesh("mesh-2D"), 2)
    for k, (info, fi) in enumerate(traj):
        print("step %d: %d Newton iterations, %d evaluations, forcing %.4f s" % (k + 1, info["newton_iterations"], fi["evaluations"],
                                                                                info["forcing_seconds"]))
        assert fi["evaluations"] == 2 * (k + 1)
    assert traj[0][0]["newton_iterations"] >= 2


def test_host_class_3d2z_source_trajectory(nsb, small_3d_mesh, tmp_path):
    path = str(tmp_path / "m3.bin")
    msh.write_bin(path, small_3d_mesh)
    _trajectory(nsb, "3D-2Z", path, small_3d_mesh, 3)


def test_forcing_source_error_paths(nsb, golden_mesh, msh_file):
    L = nsb.lib()
    dev = nsb.Device(2)
    with pytest.raises(nsb.NsbError, match="no mesh uploaded"):
        dev.set_forcing_source(SMOOTH)
    with pytest.raises(nsb.NsbError, match="no mesh uploaded"):
        dev.eval_forcing(nsb.NSB_FORCING_NEW, 0.0)
    m = golden_mesh("mesh-2D")
    dm = odofs.enumerate_dofs(m)
    dev.upload_mesh(m.points, m.cells, dm.cell_dofs, dm.n_u, dm.n_p)
    with pytest.raises(nsb.NsbError, match="no forcing source set"):
        dev.eval_forcing(nsb.NSB_FORCING_NEW, 0.0)
    bad = "__device__ void nsb_forcing(const double* x, double t, const double* prm, double* f) {\n  f[0] = x[0] +;\n}\n"
    with pytest.raises(nsb.NsbError, match=r"nsb_forcing\.cu\(2\): error"):
        dev.set_forcing_source(bad)
    assert not dev.forcing_info()["has_source"]
    with pytest.raises(nsb.NsbError, match="n_prm"):
        dev.set_forcing_source(SMOOTH, np.zeros(17))
    assert L.nsb_set_forcing_source(dev.h, SMOOTH.encode(), None, 2) != 0
    assert "prm is NULL" in L.nsb_last_error(dev.h).decode()
    dev.set_forcing_source(SMOOTH, np.zeros(16))
    for which in (-1, 2):
        with pytest.raises(nsb.NsbError, match="which"):
            dev.eval_forcing(which, 0.0)
        with pytest.raises(nsb.NsbError, match="which"):
            dev.forcing(which)
    assert L.nsb_get_forcing(dev.h, nsb.NSB_FORCING_OLD, _buf(dev)) == 1         # clear slot: soft 1
    dev.close()
    # the host class: too many parameters fail at once, a compile error fails the step with NVRTC's log
    s = nsb.HostSolver("2D-2", msh_file("mesh-2D"))
    with pytest.raises(nsb.NsbError, match="at most 16"):
        s.set_forcing_source(SMOOTH, np.zeros(17))
    s.set_forcing_source(bad)
    s.initialize()
    with pytest.raises(nsb.NsbError, match=r"nsb_forcing\.cu\(2\)"):
        s.step()
    s.close()


def _buf(dev):
    import ctypes as C
    _, _, nc = dev.sizes()
    dev._tmp = np.empty(nc * 7 * dev.dim)
    return dev._tmp.ctypes.data_as(C.POINTER(C.c_double))


def test_multi_gpu_forcing_source_bit_exact_vs_single_gpu(tmp_path):
    """tools/gpu_multi.py --forcing-source: every rank compiles and evaluates the source on its own local cells (ghost
    layer included); its slots, A and b are bit-exact against one GPU, and the host class's steps match the oracle."""
    n = _ngpus()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    out = str(tmp_path / "multi.json")
    env = dict(os.environ, OMP_NUM_THREADS="4")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tools", "gpu_multi.py"), "--json", out, "--lc", "0.05",
           "--forcing-source"]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    s = json.load(open(out))
    assert s["forcing_source"] and s["world"] == 2
    for r_ in s["ranks"]:
        assert r_["slots_bitexact_vs_1gpu"] and r_["A_bitexact_vs_1gpu"] and r_["b_bitexact_vs_1gpu"], r_
        assert r_["A_relerr"] < 1e-12 and r_["b_relerr"] < 1e-12 and r_["field_relerr_vs_direct"] < 1e-8, r_
    for st in s["host_class_steps"]:
        assert st["err_cd"] < 1e-6 and st["err_dp"] < 1e-6, st
    assert s["host_class_field_relerr"] < 1e-8
