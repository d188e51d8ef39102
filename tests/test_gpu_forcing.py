"""GPU (-m gpu): the forcing input (nsb_get_quadrature_points / nsb_set_forcing, NavierStokes::set_forcing_term) against
the oracle and against a manufactured solution the P2/P1 space represents exactly (tests/forcing_cases.py).
Tolerances: assembled A and b relative 1e-12 (max-norm scaled); quadrature points 1e-14; manufactured: spmv defect
1e-10 ||b||, tight solve relative L2 1e-8, Newton residual 1e-9 of the unforced one; host class C_D, C_L, dp 1e-6 and
fields 1e-8 against the oracle's direct-solve trajectory."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import assemble as asm, dofs as odofs, solve as osolve
from tests.conftest import GOLDEN, ROOT
from tests.forcing_cases import ForcedOracle, Manufactured, quadrature_points, sample, smooth_forcing
from tests.test_gpu_parity import TOL_ASM, TOL_FIELD, TOL_FORCE, Case, relmax
from tests.test_gpu_multirank import _free_port, _ngpus
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


def _forcing(c, pts):
    """(f at T_NEW, f at T_NEW - dt) at pts: f_new != f_old."""
    return sample(smooth_forcing, pts, T_NEW), sample(smooth_forcing, pts, T_NEW - c.dt)


@pytest.mark.parametrize("which", ["2d", "3d"])
def test_quadrature_points_match_oracle(fcase2d, fcase3d, which):
    c = fcase2d if which == "2d" else fcase3d
    pts = c.dev.quadrature_points()
    ref = quadrature_points(c.mesh)
    assert pts.shape == ref.shape == (c.mesh.n_cells, 7 if c.dim == 2 else 10, c.dim)
    assert relmax(pts, ref) < 1e-14


@pytest.mark.parametrize("which", ["2d", "3d"])
@pytest.mark.parametrize("theta,first_order", [(0.5, False), (1.0, True), (0.5, True)])
def test_linearized_assembly_parity_with_forcing(fcase2d, fcase3d, which, theta, first_order):
    c = fcase2d if which == "2d" else fcase3d
    con = c.constraints()
    c.dev.set_forcing(*_forcing(c, c.dev.quadrature_points()))
    try:
        p = c.linearized(theta, first_order, con)
    finally:
        c.dev.clear_forcing()
    ref = asm.assemble(c.mesh, c.dm, c.pat, p, con, "linearized", c.un, c.unm1, with_pressure_matrices=False,
                       forcing=_forcing(c, quadrature_points(c.mesh)))
    A, b = c.dev.matrix_values(), c.dev.get_vector(c.nsb.NSB_RHS)
    assert relmax(A, ref.A) < TOL_ASM and relmax(b, ref.b) < TOL_ASM
    ref0 = asm.assemble(c.mesh, c.dm, c.pat, p, con, "linearized", c.un, c.unm1, with_pressure_matrices=False)
    assert np.linalg.norm(b - ref0.b) > 1e-3 * np.linalg.norm(ref0.b)         # the forcing did change the rhs
    c.dev.assemble_linearized()                                               # cleared: back to the unforced system
    assert relmax(c.dev.get_vector(c.nsb.NSB_RHS), ref0.b) < TOL_ASM


@pytest.mark.parametrize("which", ["2d", "3d"])
def test_newton_assembly_parity_with_forcing(fcase2d, fcase3d, which):
    c = fcase2d if which == "2d" else fcase3d
    nsb = c.nsb
    con = c.constraints(homogeneous=True)
    pk = np.zeros(c.dm.n_dofs)
    pk[c.dm.n_u:] = 0.05 * np.random.default_rng(7).uniform(-1, 1, c.dm.n_p)
    cur = c.un + pk
    fo = _forcing(c, quadrature_points(c.mesh))
    c.dev.set_forcing(*_forcing(c, c.dev.quadrature_points()))
    try:
        for theta in (1.0, 0.5):
            p = asm.Params(dt=c.dt, theta=theta, nu=c.nu, use_supg=c.tc["supg"])
            c.dev.set_params(c.dt, theta, c.nu, 1.0, 0.1, c.tc["supg"], False)
            c.dev.set_vector(nsb.NSB_CURRENT_SOLUTION, cur)
            c.dev.set_vector(nsb.NSB_SOLUTION_OLD, c.unm1)
            c.dev.assemble_newton()
            ref = asm.assemble(c.mesh, c.dm, c.pat, p, con, "newton", cur, c.unm1, with_pressure_matrices=False, forcing=fo)
            ref0 = asm.assemble(c.mesh, c.dm, c.pat, p, con, "newton", cur, c.unm1, with_pressure_matrices=False)
            b = c.dev.get_vector(nsb.NSB_RHS)
            assert relmax(c.dev.matrix_values(), ref.A) < TOL_ASM and relmax(b, ref.b) < TOL_ASM
            assert np.linalg.norm(b - ref0.b) > 1e-3 * np.linalg.norm(ref0.b)
    finally:
        c.dev.clear_forcing()


@pytest.mark.parametrize("which", ["2d", "3d"])
def test_zero_forcing_and_clear_are_bit_identical_to_none(nsb, golden_mesh, small_3d_mesh, which):
    mesh = golden_mesh("mesh-2D") if which == "2d" else small_3d_mesh
    case = "2D-2" if which == "2d" else "3D-2Z"
    ref, c = Case(nsb, mesh, case), Case(nsb, mesh, case)

    def assemble(cc):
        cc.linearized(0.5, False, cc.constraints())
        return cc.dev.matrix_values(), cc.dev.get_vector(nsb.NSB_RHS)

    A0, b0 = assemble(ref)
    pts = c.dev.quadrature_points()
    c.dev.set_forcing(*_forcing(c, pts))
    A1, b1 = assemble(c)
    assert np.array_equal(A1, A0) and not np.array_equal(b1, b0)
    c.dev.set_forcing(np.zeros_like(pts), np.zeros_like(pts))                 # all-zero values = no forcing
    A2, b2 = assemble(c)
    assert np.array_equal(A2, A0) and np.array_equal(b2, b0)
    c.dev.set_forcing(*_forcing(c, pts))
    n = c.dev.launch_count()
    c.dev.clear_forcing()
    assert c.dev.launch_count() == n                                          # a clear launches nothing
    A3, b3 = assemble(c)
    assert np.array_equal(A3, A0) and np.array_equal(b3, b0)
    ref.dev.close()
    c.dev.close()


@pytest.mark.parametrize("which", ["2d", "3d"])
def test_manufactured_solution_through_the_library(nsb, golden_mesh, small_3d_mesh, which):
    """Linearised step (no SUPG, see tests/forcing_cases.py) and Newton residual (SUPG in 3-D) at the exact solution."""
    mesh = golden_mesh("mesh-2D") if which == "2d" else small_3d_mesh
    dim, nu, dt = mesh.dim, 1e-3, 0.02
    dm = odofs.enumerate_dofs(mesh)
    ms = Manufactured(mesh, nu)
    x = ms.exact(dm)
    dev = nsb.Device(dim)
    dev.upload_mesh(mesh.points, mesh.cells, dm.cell_dofs, dm.n_u, dm.n_p)
    f = sample(ms.forcing, dev.quadrature_points(), 0.0)
    # linearised: A x_u = b to round-off, and the tight solve returns u
    con = ms.constraints(dm)
    dev.set_constraints(con.dofs, con.val[con.dofs])
    for theta in (1.0, 0.5):
        dev.set_forcing(f, f)
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
    # Newton: the residual vanishes at u
    hcon = odofs.build_constraints(mesh, dm, None, ms.ids, homogeneous=True)
    dev.set_constraints(hcon.dofs, hcon.val[hcon.dofs])
    for supg in ((False, True) if dim == 2 else (True,)):
        norms = []
        for forced in (True, False):
            dev.set_forcing(f, f) if forced else dev.clear_forcing()
            dev.set_params(dt, 1.0, nu, 1.0, 0.1, supg, True)
            dev.set_vector(nsb.NSB_CURRENT_SOLUTION, x)
            dev.set_vector(nsb.NSB_SOLUTION_OLD, x)
            dev.assemble_newton()
            norms.append(dev.rhs_norm())
        print("%s Newton SUPG %s: residual ratio %.2e" % (which, supg, norms[0] / norms[1]))
        assert norms[0] <= 1e-9 * norms[1]
    dev.close()


def _trajectory(nsb, case, path, mesh, steps, fail_at=None, fail_solves=0):
    """HostSolver(case) with smooth_forcing against ForcedOracle(direct) over `steps` steps; the step `fail_at` has its
    first `fail_solves` linear solves reported as failed on both sides (retry / fallback paths)."""
    s = nsb.HostSolver(case, path, gmres_tolerance=1e-12)
    s.set_forcing(smooth_forcing)
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
        out.append((info, ref, x))
    s.close()
    return out


def test_host_class_2d2_forced_trajectory_with_halved_retry(nsb, golden_mesh, msh_file):
    """Three CN steps; in the third, the solve and its BE fallback are reported as failed, so the step is redone with
    dt/2 and the forcing's old time level is re-sampled at t - dt/2."""
    traj = _trajectory(nsb, "2D-2", msh_file("mesh-2D"), golden_mesh("mesh-2D"), 3, fail_at=2, fail_solves=2)
    assert traj[2][0]["solves"] == 3
    g = np.load(os.path.join(GOLDEN, "oracle_vectors.npz"))["traj_2D2"]                  # the unforced trajectory
    for k, (info, _, _) in enumerate(traj[:2]):
        assert abs(info["cd"] - g[k][1]) > 1e3 * TOL_FORCE * abs(g[k][1]), (k, info["cd"], g[k][1])


def test_host_class_2d1_newton_forced_trajectory(nsb, golden_mesh, msh_file):
    traj = _trajectory(nsb, "2D-1", msh_file("mesh-2D"), golden_mesh("mesh-2D"), 2)
    g = np.load(os.path.join(GOLDEN, "oracle_vectors.npz"))["traj_2D1"][0]
    assert abs(traj[0][0]["cd"] - g[1]) > 1e3 * TOL_FORCE * abs(g[1])
    assert traj[0][0]["newton_iterations"] >= 1


def test_host_class_3d2z_forced_trajectory(nsb, small_3d_mesh, tmp_path):
    path = str(tmp_path / "m3.bin")
    msh.write_bin(path, small_3d_mesh)
    traj = _trajectory(nsb, "3D-2Z", path, small_3d_mesh, 3)
    o = osolve.Oracle(small_3d_mesh, "3D-2Z", solver="direct")
    o.step()
    x = traj[0][2]
    assert np.linalg.norm(x - o.current_solution) > 1e3 * TOL_FIELD * np.linalg.norm(o.current_solution)


def test_host_class_forcing_callback_error_fails_the_step(nsb, msh_file):
    s = nsb.HostSolver("2D-2", msh_file("mesh-2D"))

    def bad(x, t):
        raise ValueError("no forcing today")

    s.set_forcing(bad)
    s.initialize()
    with pytest.raises(nsb.NsbError, match="forcing callback") as e:
        s.step()
    assert isinstance(e.value.__cause__, ValueError)
    s.close()


def test_forcing_error_paths(nsb, golden_mesh):
    import ctypes as C
    L = nsb.lib()
    dev = nsb.Device(2)
    nq = C.c_int()
    assert L.nsb_set_forcing(dev.h, nsb.NSB_FORCING_NEW, None) != 0
    assert "no mesh uploaded" in L.nsb_last_error(dev.h).decode()
    assert L.nsb_get_quadrature_points(dev.h, C.byref(nq), None) != 0
    assert "no mesh uploaded" in L.nsb_last_error(dev.h).decode()
    m = golden_mesh("mesh-2D")
    dm = odofs.enumerate_dofs(m)
    dev.upload_mesh(m.points, m.cells, dm.cell_dofs, dm.n_u, dm.n_p)
    for which in (-1, 2):
        with pytest.raises(nsb.NsbError, match="which"):
            dev._ck(L.nsb_set_forcing(dev.h, which, None))
    with pytest.raises(ValueError, match="shape"):
        dev.set_forcing(np.ones((3, 7, 2)))
    dev.close()


def test_multi_gpu_forcing_bit_exact_vs_single_gpu(tmp_path):
    """tools/gpu_multi.py --forcing: per rank, A and b with forcing bit-exact against one GPU (ghost-layer cells sample
    the forcing at their own points) and within 1e-12 of the oracle; the host class's forced steps match the oracle."""
    n = _ngpus()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    out = str(tmp_path / "multi.json")
    env = dict(os.environ, OMP_NUM_THREADS="4")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tools", "gpu_multi.py"), "--json", out, "--lc", "0.05", "--forcing"]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    s = json.load(open(out))
    assert s["forcing"] and s["world"] == 2
    for r_ in s["ranks"]:
        assert r_["A_bitexact_vs_1gpu"] and r_["b_bitexact_vs_1gpu"], r_
        assert r_["A_relerr"] < 1e-12 and r_["b_relerr"] < 1e-12 and r_["field_relerr_vs_direct"] < 1e-8, r_
    for st in s["host_class_steps"]:
        assert st["err_cd"] < 1e-6 and st["err_dp"] < 1e-6, st
    assert s["host_class_field_relerr"] < 1e-8
