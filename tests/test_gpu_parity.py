"""GPU (-m gpu): the CUDA path, called through the C ABI, against the numpy oracle on the same seeded
inputs.  Tolerances: assembled matrix / rhs relative 1e-12 (max-norm scaled); fields in tight-tolerance
mode relative L2 <= 1e-8; C_D, C_L, dp relative 1e-6 (BASELINE.json north_star); integer maps bit-exact;
run-to-run bit-reproducibility."""
import os

import numpy as np
import pytest
import scipy.sparse as sp

from oracle import assemble as asm, dofs as odofs, postprocess as pp, solve as osolve
from tests.conftest import GOLDEN, synthetic_state
from tools import meshgen, msh

pytestmark = pytest.mark.gpu

TOL_ASM = 1e-12
TOL_FIELD = 1e-8
TOL_FORCE = 1e-6


def relmax(a, b):
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


class Case:
    """Mesh + oracle structures + a device with the mesh uploaded."""

    def __init__(self, nsb, mesh, case):
        self.nsb, self.mesh, self.tc = nsb, mesh, pp.TEST_CASES[case]
        self.dim = mesh.dim
        self.dm = odofs.enumerate_dofs(mesh)
        self.pat = odofs.make_sparsity(self.dm)
        self.ids = pp.boundary_ids(self.dim)
        self.nu = pp.viscosity(self.dim, self.tc["U_m"], self.tc["Re"])
        self.dev = nsb.Device(self.dim)
        self.dev.upload_mesh(mesh.points, mesh.cells, self.dm.cell_dofs, self.dm.n_u, self.dm.n_p)
        self.un, self.unm1 = synthetic_state(self.dm, self.dim, self.tc["U_m"])
        self.dt = 0.01 if self.dim == 3 else 0.02

    def constraints(self, t=1.0, homogeneous=False):
        tc = self.tc
        con = odofs.build_constraints(self.mesh, self.dm, pp.inlet_profile(self.dim, tc["U_m"], tc["time_dep"], tc["T_ramp"], t),
                                      self.ids, homogeneous=homogeneous)
        self.dev.set_constraints(con.dofs, con.val[con.dofs])
        return con

    def linearized(self, theta, first_order, con):
        nsb = self.nsb
        p = asm.Params(dt=self.dt, theta=theta, nu=self.nu, use_supg=self.tc["supg"], first_step=first_order)
        self.dev.set_params(self.dt, theta, self.nu, 1.0, 0.1, self.tc["supg"], first_order)
        self.dev.set_vector(nsb.NSB_SOLUTION_OLD, self.un)
        self.dev.set_vector(nsb.NSB_SOLUTION_OLD_OLD, self.unm1)
        self.dev.assemble_linearized()
        return p


@pytest.fixture(scope="module")
def case2d(nsb, golden_mesh):
    c = Case(nsb, golden_mesh("mesh-2D"), "2D-2")
    yield c
    c.dev.close()


@pytest.fixture(scope="module")
def case3d(nsb, small_3d_mesh):
    c = Case(nsb, small_3d_mesh, "3D-2Z")
    yield c
    c.dev.close()


@pytest.mark.parametrize("which", ["2d", "3d"])
def test_pattern_bit_exact(case2d, case3d, which):
    c = case2d if which == "2d" else case3d
    rp, col = c.dev.pattern()
    assert np.array_equal(rp, c.pat[0]) and np.array_equal(col.astype(np.int64), c.pat[1].astype(np.int64))
    assert np.array_equal(c.dev.row_gids(), np.arange(c.dm.n_dofs))


@pytest.mark.parametrize("which", ["2d", "3d"])
@pytest.mark.parametrize("theta,first_order", [(0.5, False), (1.0, True), (0.5, True)])
def test_linearized_assembly_parity(case2d, case3d, which, theta, first_order):
    c = case2d if which == "2d" else case3d
    con = c.constraints()
    p = c.linearized(theta, first_order, con)
    ref = asm.assemble(c.mesh, c.dm, c.pat, p, con, "linearized", c.un, c.unm1, with_pressure_matrices=False)
    A = c.dev.matrix_values()
    b = c.dev.get_vector(c.nsb.NSB_RHS)
    assert relmax(A, ref.A) < TOL_ASM and relmax(b, ref.b) < TOL_ASM
    assert abs(c.dev.rhs_norm() - np.linalg.norm(ref.b)) < 1e-12 * np.linalg.norm(ref.b)
    if not first_order:
        # the u* clamp (cpp:674) must fire on some but not all quadrature points for this state
        p1 = asm.Params(dt=c.dt, theta=theta, nu=c.nu, use_supg=c.tc["supg"], first_step=True)
        ref1 = asm.assemble(c.mesh, c.dm, c.pat, p1, con, "linearized", c.un, c.unm1, with_pressure_matrices=False)
        assert relmax(ref.A, ref1.A) > 1e-6


@pytest.mark.parametrize("which", ["2d", "3d"])
def test_newton_assembly_parity(case2d, case3d, which):
    c = case2d if which == "2d" else case3d
    nsb = c.nsb
    con = c.constraints(homogeneous=True)
    pk = np.zeros(c.dm.n_dofs)
    pk[c.dm.n_u:] = 0.05 * np.random.default_rng(7).uniform(-1, 1, c.dm.n_p)
    cur = c.un + pk
    for theta in (1.0, 0.5):
        p = asm.Params(dt=c.dt, theta=theta, nu=c.nu, use_supg=c.tc["supg"])
        c.dev.set_params(c.dt, theta, c.nu, 1.0, 0.1, c.tc["supg"], False)
        c.dev.set_vector(nsb.NSB_CURRENT_SOLUTION, cur)
        c.dev.set_vector(nsb.NSB_SOLUTION_OLD, c.unm1)
        c.dev.assemble_newton()
        ref = asm.assemble(c.mesh, c.dm, c.pat, p, con, "newton", cur, c.unm1, with_pressure_matrices=False)
        assert relmax(c.dev.matrix_values(), ref.A) < TOL_ASM
        assert relmax(c.dev.get_vector(nsb.NSB_RHS), ref.b) < TOL_ASM


@pytest.mark.parametrize("which", ["2d", "3d"])
def test_pressure_matrices_spmv_and_solve(case2d, case3d, which):
    c = case2d if which == "2d" else case3d
    nsb, N, n_u = c.nsb, c.dm.n_dofs, c.dm.n_u
    con = c.constraints()
    p = c.linearized(0.5, False, con)
    ref = asm.assemble(c.mesh, c.dm, c.pat, p, con, "linearized", c.un, c.unm1)
    c.dev.assemble_pressure_matrices()
    for which_m, full in ((0, ref.Mp), (1, ref.Kp)):
        rp, col, val = c.dev.pressure_matrix(which_m)
        dev_m = sp.csr_matrix((val, col, rp), shape=(c.dm.n_p, c.dm.n_p))
        or_m = asm.to_csr(c.pat, full, N)[n_u:, n_u:]
        assert abs(dev_m - or_m).max() < TOL_ASM * abs(or_m).max()
    A = asm.to_csr(c.pat, ref.A, N)
    rng = np.random.default_rng(42)
    x, y = rng.uniform(-1, 1, N), rng.uniform(-1, 1, N)
    ax, ay = c.dev.spmv(x), c.dev.spmv(y)
    assert relmax(ax, A @ x) < 1e-13
    assert relmax(c.dev.spmv(2.0 * x - 3.0 * y), 2.0 * ax - 3.0 * ay) < 1e-13          # linearity
    # reference stopping rule: converges well inside the reference's 200-iteration budget
    ok, it, res = c.dev.solve(200, 1e-2, 150)
    assert ok and 0 < it < 100 and res <= 1e-2 * np.linalg.norm(ref.b)
    # parity mode: tight tolerance against a sparse direct solve of the ORACLE's matrix
    ok, it2, _ = c.dev.solve(2000, 1e-12, 150)
    assert ok
    xs = c.dev.get_vector(nsb.NSB_SOLUTION)
    xd = con.distribute(osolve.direct_solve(A, ref.b))
    assert np.linalg.norm(xs - xd) / np.linalg.norm(xd) < TOL_FIELD
    assert np.array_equal(xs[con.is_c], con.val[con.is_c])                             # constraints.distribute
    # bit-reproducibility: same inputs -> same bits, same iteration count
    A1 = c.dev.matrix_values()
    c.dev.assemble_linearized()
    assert np.array_equal(A1, c.dev.matrix_values())
    ok, it3, _ = c.dev.solve(2000, 1e-12, 150)
    assert it3 == it2 and np.array_equal(xs, c.dev.get_vector(nsb.NSB_SOLUTION))


def test_zero_initialised_solver_opts_mean_the_defaults(nsb):
    """A zero-initialised nsb_solver_opts (what RunOptions::solver{} and the C facade pass) selects the library defaults
    for every field, including the Gram-Schmidt policy (ADVICE r1: 0 used to switch the second pass off)."""
    dev = nsb.Device(2)
    base = dev.get_solver_opts()
    dev.set_solver_opts()                     # all fields zero
    got = dev.get_solver_opts()
    assert got == base and got["reorthogonalize"] == 1 and got["velocity_cycle"] == 2 and got["precond_precision"] in (16, 32)
    dev.set_solver_opts(reorthogonalize=-1, precond_precision=64, velocity_cycle=1)
    got = dev.get_solver_opts()
    assert got["reorthogonalize"] == -1 and got["precond_precision"] == 64 and got["velocity_cycle"] == 1
    dev.close()


def test_error_paths(nsb, golden_mesh):
    m = golden_mesh("mesh-2D")
    dm = odofs.enumerate_dofs(m)
    dev = nsb.Device(2)
    with pytest.raises(nsb.NsbError, match="no assembled system"):
        dev.solve()
    bad = dm.cell_dofs.copy()
    bad[0, 0] += 1                                   # breaks the consecutive-velocity-DoF contract
    with pytest.raises(nsb.NsbError, match="node-block"):
        dev.upload_mesh(m.points, m.cells, bad, dm.n_u, dm.n_p)
    flipped = m.cells.copy()
    flipped[0, [0, 1]] = flipped[0, [1, 0]]          # negative cell measure
    dmf = odofs.enumerate_dofs(msh.Mesh(2, m.points, flipped, m.cell_tag, m.faces, m.face_tag))
    with pytest.raises(nsb.NsbError, match="non-positive measure"):
        dev.upload_mesh(m.points, flipped, dmf.cell_dofs, dmf.n_u, dmf.n_p)
    dev.upload_mesh(m.points, m.cells, dm.cell_dofs, dm.n_u, dm.n_p)
    dev.set_vector(nsb.NSB_SOLUTION_OLD, np.zeros(dm.n_dofs))
    dev.assemble_linearized()
    with pytest.raises(nsb.NsbError, match="pressure"):
        dev.solve()
    dev.close()


def test_host_class_trajectory_2d2_matches_oracle(nsb, msh_file):
    """NavierStokes<2>(make_2D_2) through the C++ host class, tight GMRES tolerance, vs the oracle's
    direct-solve trajectory (golden): first CN step as BE, second step, then extrapolated u*."""
    g = np.load(os.path.join(GOLDEN, "oracle_vectors.npz"))["traj_2D2"]
    s = nsb.HostSolver("2D-2", msh_file("mesh-2D"), gmres_tolerance=1e-12)
    s.initialize()
    for k in range(4):
        info = s.step()
        assert info["converged"] == 1
        got = np.array([info["time"], info["cd"], info["cl"], info["dp"]])
        assert np.all(np.abs(got - g[k]) <= TOL_FORCE * np.abs(g[k]) + 1e-13), (k, got, g[k])
    s.close()


def test_host_class_newton_2d1_matches_oracle(nsb, msh_file):
    g = np.load(os.path.join(GOLDEN, "oracle_vectors.npz"))["traj_2D1"][0]
    s = nsb.HostSolver("2D-1", msh_file("mesh-2D"), gmres_tolerance=1e-12)
    s.initialize()
    info = s.step()
    got = np.array([info["time"], info["cd"], info["cl"], info["dp"]])
    assert np.all(np.abs(got - g[:4]) <= TOL_FORCE * np.abs(g[:4]) + 1e-13), (got, g)
    assert info["newton_iterations"] == int(g[4])
    s.close()


def test_host_class_3d_steps_match_oracle(nsb, small_3d_mesh, tmp_path):
    path = str(tmp_path / "m3.bin")
    msh.write_bin(path, small_3d_mesh)
    s = nsb.HostSolver("3D-2Z", path, gmres_tolerance=1e-12)
    s.initialize()
    o = osolve.Oracle(small_3d_mesh, "3D-2Z", solver="direct")
    for k in range(3):
        info, ref = s.step(), o.step()
        for key in ("cd", "cl", "dp"):
            assert abs(info[key] - ref[key]) <= TOL_FORCE * abs(ref[key]) + 1e-12, (k, key, info[key], ref[key])
        x = s.solution()
        assert np.linalg.norm(x - o.current_solution) / np.linalg.norm(o.current_solution) < TOL_FIELD
    # reference stopping rule (1e-2 * ||b|| on the preconditioned residual): converged, within the 200-iteration cap, and the
    # same first step as the tight-tolerance trajectory to the accuracy that stopping rule leaves (measured on a B200: C_D
    # 2e-7, dp 1e-8 relative after 17 iterations; the bound is loose on purpose -- two preconditioners stopped at 1e-2 may
    # differ by up to that tolerance, SURVEY fact 5)
    s2 = nsb.HostSolver("3D-2Z", path)
    s2.initialize()
    info = s2.step()
    o1 = osolve.Oracle(small_3d_mesh, "3D-2Z", solver="direct")
    ref1 = o1.step()
    assert info["converged"] == 1 and 0 < info["gmres_iterations"] <= 200 and info["solves"] == 1
    loose = {key: abs(info[key] - ref1[key]) / max(abs(ref1[key]), 1e-300) for key in ("cd", "dp")}
    print("first step at the reference tolerance vs direct solve:", loose, "GMRES", info["gmres_iterations"])
    assert loose["cd"] < 5e-2 and loose["dp"] < 5e-2, loose
    x2 = s2.solution()
    assert np.linalg.norm(x2 - o1.current_solution) / np.linalg.norm(o1.current_solution) < 5e-2
    s.close()
    s2.close()


def test_full_size_properties_mesh_3d_10(nsb):
    """mesh-3D-10-equivalent (0.57 M cells, 2.45 M DoFs): size-independent properties."""
    mesh = meshgen.mesh_3d(10)
    dm = odofs.enumerate_dofs(mesh)
    N, n_u = dm.n_dofs, dm.n_u
    dev = nsb.Device(3)
    dev.upload_mesh(mesh.points, mesh.cells, dm.cell_dofs, dm.n_u, dm.n_p)
    nrows, nnz, _ = dev.sizes()
    assert nrows == N and 90 < nnz / nrows < 105
    tc = pp.TEST_CASES["3D-2Z"]
    con = odofs.build_constraints(mesh, dm, pp.inlet_profile(3, tc["U_m"], False, 4.0, 1.0), pp.boundary_ids(3))
    dev.set_constraints(con.dofs, con.val[con.dofs])
    un, unm1 = synthetic_state(dm, 3, tc["U_m"])
    dev.set_params(0.01, 0.5, 1e-3, 1.0, 0.1, True, False)
    dev.set_vector(nsb.NSB_SOLUTION_OLD, un)
    dev.set_vector(nsb.NSB_SOLUTION_OLD_OLD, unm1)
    dev.assemble_linearized()
    b1 = dev.get_vector(nsb.NSB_RHS)
    # (1) constrained rows are identity-like: A e_c = d e_c with d > 0, b_c = 0
    e = np.zeros(N)
    c0 = con.dofs[::997]
    e[c0] = 1.0
    y = dev.spmv(e)
    assert np.all(y[c0] > 0) and np.count_nonzero(y) == c0.size and np.all(b1[con.is_c] == 0)
    # (2) pressure rows of A applied to a linear velocity field give -(psi, div u) = -2 * (M_p 1) on
    #     rows whose velocity neighbours are all unconstrained
    dev.assemble_pressure_matrices()
    rp, col, val = dev.pressure_matrix(0)
    mp1 = sp.csr_matrix((val, col, rp), shape=(dm.n_p, dm.n_p)) @ np.ones(dm.n_p)
    u = np.zeros(N)
    comp = dm.component[:n_u]
    u[:n_u] = np.where(comp == 0, dm.support_points[:n_u, 0], np.where(comp == 1, dm.support_points[:n_u, 1], 0.0))
    u[con.is_c] = 0.0
    yp = dev.spmv(u)[n_u:]
    touched = np.abs(dev.spmv(np.where(con.is_c, 1.0, 0.0) * 0 + con.is_c.astype(float)))   # zero columns => 0
    assert np.count_nonzero(touched[~con.is_c]) == 0                                       # constrained columns eliminated
    # rows far from the Dirichlet boundary
    interior = np.ones(dm.n_p, bool)
    cells_b = np.isin(dm.cell_dofs, con.dofs).any(axis=1)
    interior[np.unique(dm.cell_dofs[cells_b][:, [3, 7, 11, 15]]) - n_u] = False
    assert np.abs(yp[interior] + 2.0 * mp1[interior]).max() < 1e-12 * np.abs(mp1).max() * 1e3
    # (3) linearity + run-to-run bit reproducibility of assembly
    rng = np.random.default_rng(3)
    x, z = rng.uniform(-1, 1, N), rng.uniform(-1, 1, N)
    assert relmax(dev.spmv(x + 2 * z), dev.spmv(x) + 2 * dev.spmv(z)) < 1e-13
    dev.assemble_linearized()
    assert np.array_equal(b1, dev.get_vector(nsb.NSB_RHS))
    # (4) the solve meets the reference stopping rule and its solution satisfies the constraints
    ok, it, res = dev.solve(200, 1e-2, 150)
    assert ok and res <= 1e-2 * np.linalg.norm(b1)
    xs = dev.get_vector(nsb.NSB_SOLUTION)
    assert np.array_equal(xs[con.is_c], con.val[con.is_c])
    dev.close()


def test_solver_options_reach_the_same_solution(case3d):
    """fp64 / fp32 / fp16 operator copies inside the velocity polynomial, Chebyshev vs harmonic-Ritz roots, the reference's
    theta*nu Schur scaling: different preconditioners, same linear system => same tight-tolerance solution."""
    c = case3d
    nsb = c.nsb
    con = c.constraints()
    c.linearized(0.5, False, con)
    c.dev.assemble_pressure_matrices()
    ok, it0, _ = c.dev.solve(3000, 1e-12, 150)
    x0 = c.dev.get_vector(nsb.NSB_SOLUTION)
    assert ok
    for opts in (dict(precond_precision=64), dict(poly_kind=-1), dict(poly_target=0.2, poly_degree_F=8),
                 dict(schur_mass_coeff=0.5 * c.nu), dict(precond_precision=32), dict(precond_precision=16)):
        c.dev.set_solver_opts(**opts)
        c.dev.assemble_linearized()            # refills the operator copy after a precision change
        ok, it, _ = c.dev.solve(3000, 1e-12, 150)
        x = c.dev.get_vector(nsb.NSB_SOLUTION)
        assert ok, opts
        assert np.linalg.norm(x - x0) / np.linalg.norm(x0) < 1e-9, opts
    info = c.dev.solver_info()
    assert info["amg_levels"] >= 1 and info["poly_degree"] >= 1
    c.dev.set_solver_opts()
    c.dev.assemble_linearized()


def test_newton_iterations_3d_supg_match_oracle(case3d):
    """Two Newton iterations of the 3D-1Z setting (backward Euler, SUPG with the P2 Laplacian in the strong
    residual, grad-div) driven through the C ABI: -residual norm, update and iterate against the oracle.
    (The full reference step needs all 50 Newton iterations here -- too slow for a direct-solve oracle.)"""
    c = case3d
    nsb, dm, N = c.nsb, c.dm, c.dm.n_dofs
    tc = pp.TEST_CASES["3D-1Z"]
    nu = pp.viscosity(3, tc["U_m"], tc["Re"])
    dt = 0.1
    con = odofs.build_constraints(c.mesh, dm, None, c.ids, homogeneous=True)
    c.dev.set_constraints(con.dofs, con.val[con.dofs])
    c.dev.set_params(dt, 1.0, nu, 1.0, 0.1, True, True)
    # lift the inlet profile onto a zero state (cpp:1118-1142)
    cur = np.zeros(N)
    d_in = odofs.boundary_dofs(c.mesh, dm, c.ids["inlet"])
    cur[d_in] = pp.inlet_profile(3, tc["U_m"], False, 0.0, dt)(dm.support_points[d_in], dm.component[d_in])
    old = np.zeros(N)
    p = asm.Params(dt=dt, theta=1.0, nu=nu, use_supg=True)
    c.dev.set_vector(nsb.NSB_SOLUTION_OLD, old)
    c.dev.set_vector(nsb.NSB_CURRENT_SOLUTION, cur)
    c.dev.assemble_newton()
    c.dev.assemble_pressure_matrices()
    cur_o = cur.copy()
    for it in range(2):
        c.dev.set_vector(nsb.NSB_CURRENT_SOLUTION, cur)
        c.dev.assemble_newton()
        ref = asm.assemble(c.mesh, dm, c.pat, p, con, "newton", cur_o, old, with_pressure_matrices=False)
        assert abs(c.dev.rhs_norm() - np.linalg.norm(ref.b)) < 1e-10 * np.linalg.norm(ref.b)
        ok, _, _ = c.dev.solve(3000, 1e-12, 150)
        assert ok
        upd = c.dev.get_vector(nsb.NSB_SOLUTION)
        upd_o = con.distribute(osolve.direct_solve(asm.to_csr(c.pat, ref.A, N), ref.b))
        assert np.linalg.norm(upd - upd_o) / np.linalg.norm(upd_o) < TOL_FIELD
        cur = cur + upd
        cur_o = cur_o + upd_o
    assert np.linalg.norm(cur - cur_o) / np.linalg.norm(cur_o) < TOL_FIELD


@pytest.mark.parametrize("which", ["2d", "3d"])
def test_streamed_velocity_operator_equals_assembled(case2d, case3d, which):
    """The streamed velocity operator (velstream.cuh: packed fp32 / fp16 copy of Dinv F, TMA-staged tiles, segmented warp
    scans) is the same operator as the generic fp64 row kernel on the assembled values (precond_precision=64), including
    Dinv-scaled Dirichlet rows: checked on random vectors in two u* regimes, bit-reproducible from call to call, and
    through the GMRES iteration counts at the reference's stopping rule."""
    c = case2d if which == "2d" else case3d
    nsb = c.nsb
    con = c.constraints()
    n_u = c.dm.n_u
    x = np.zeros(c.dm.n_dofs)
    x[:n_u] = np.random.default_rng(7).standard_normal(n_u)
    try:
        for theta, first in ((0.5, False), (1.0, True)):
            ys, its = {}, {}
            for prec in (64, 32, 16):
                c.dev.set_solver_opts(precond_precision=prec)
                c.linearized(theta, first, con)
                c.dev.assemble_pressure_matrices()
                ys[prec] = c.dev.apply_velocity_block(x)[:n_u]
                assert np.array_equal(ys[prec], c.dev.apply_velocity_block(x)[:n_u])
                ok, it, _ = c.dev.solve(200, 1e-2, 150)
                assert ok
                its[prec] = it
            assert np.abs(ys[64]).max() > 0
            # (the values themselves are checked row by row against the stored copy in test_gpu_preconditioner.py)
            # Dirichlet rows act as the identity after the block-Jacobi scaling
            cu = con.dofs[con.dofs < n_u]
            assert np.allclose(ys[32][cu], x[cu], rtol=1e-12, atol=0) and np.allclose(ys[16][cu], x[cu], rtol=1e-12, atol=0)
            assert abs(its[32] - its[64]) <= 1 and abs(its[16] - its[64]) <= 2, its
    finally:
        c.dev.set_solver_opts()
        c.linearized(0.5, False, con)


def _p1_prolongation(mesh, dm):
    """P1-vector -> P2-vector prolongation in the velocity numbering: vertex nodes take the vertex value, line nodes
    the mean of their two end vertices (column index dim * vertex + component)."""
    dim = mesh.dim
    nv = dim + 1
    lines = [(0, 1), (1, 2), (2, 0)] if dim == 2 else [(0, 1), (1, 2), (2, 0), (0, 3), (1, 3), (2, 3)]
    cd = dm.cell_dofs.astype(np.int64)
    cells = mesh.cells.astype(np.int64)
    rows, cols, vals = [], [], []
    for v in range(nv):
        for c in range(dim):
            rows.append(cd[:, v * (dim + 1) + c]); cols.append(dim * cells[:, v] + c); vals.append(np.ones(len(cd)))
    for l, (i, j) in enumerate(lines):
        for c in range(dim):
            r = cd[:, nv * (dim + 1) + dim * l + c]
            rows += [r, r]; cols += [dim * cells[:, i] + c, dim * cells[:, j] + c]; vals += [np.full(len(cd), 0.5)] * 2
    rows, cols, vals = np.concatenate(rows), np.concatenate(cols), np.concatenate(vals)
    _, idx = np.unique(rows * (dim * mesh.n_vertices) + cols, return_index=True)
    return sp.csr_matrix((vals[idx], (rows[idx], cols[idx])), shape=(dm.n_u, dim * mesh.n_vertices))


@pytest.mark.parametrize("which", ["2d", "3d"])
def test_coarse_operator_is_the_galerkin_product(case2d, case3d, which):
    """The coarse operator of the two-level velocity cycle, formed cell by cell from the S_ab blocks of assembly pass 1
    (twolevel.cuh), equals P^T F P computed from the ORACLE's assembled matrix on the free coarse DoFs, and is the
    identity on constrained ones -- in two u* regimes, with SUPG + grad-div in 3-D."""
    c = case2d if which == "2d" else case3d
    dim, dm, mesh = c.dim, c.dm, c.mesh
    con = c.constraints()
    P = _p1_prolongation(mesh, dm)
    # coarse DoF (vertex v, comp k) is constrained iff the vertex's own velocity DoF is
    vdof = np.zeros(dim * mesh.n_vertices, np.int64)
    for v in range(dim + 1):
        for k in range(dim):
            vdof[dim * mesh.cells[:, v].astype(np.int64) + k] = dm.cell_dofs[:, v * (dim + 1) + k]
    cfree = ~con.is_c[vdof]
    for theta, first in ((0.5, False), (1.0, True)):
        p = c.linearized(theta, first, con)
        ref = asm.assemble(mesh, dm, c.pat, p, con, "linearized", c.un, c.unm1, with_pressure_matrices=False)
        F = asm.to_csr(c.pat, ref.A, dm.n_dofs)[:dm.n_u, :dm.n_u]
        G = (P.T @ F @ P).tocsr()
        rg, rp, cg, v = c.dev.coarse_operator()
        nb = np.diff(rp)
        # pressure DoF id -> mesh vertex: pressure DoFs are numbered in vertex first-touch order = dm's vertex map
        pvert = np.zeros(dm.n_p, np.int64)
        for k in range(dim + 1):
            pvert[dm.cell_dofs[:, k * (dim + 1) + dim].astype(np.int64) - dm.n_u] = mesh.cells[:, k]
        rows_v, cols_v = pvert[np.repeat(rg, nb)], pvert[cg]
        scale = np.abs(G).max()
        worst = 0.0
        for a in range(dim):
            for b in range(dim):
                want = np.asarray(G[dim * rows_v + a, dim * cols_v + b]).ravel()
                fr, fc = cfree[dim * rows_v + a], cfree[dim * cols_v + b]
                both = fr & fc
                worst = max(worst, np.abs(v[both, a, b] - want[both]).max() / scale)
                ident = ((rows_v == cols_v) & (a == b) & ~fr).astype(float)
                assert np.array_equal(v[~both, a, b], ident[~both])
        assert worst < 1e-12, worst
        # every free-free entry of the Galerkin product lies inside the P1 pattern the kernel stores
        Gf = sp.diags(cfree.astype(float)) @ G @ sp.diags(cfree.astype(float))
        assert abs(Gf).sum() > 0
        covered = sp.csr_matrix((np.ones(len(rows_v) * dim * dim),
                                 (np.repeat(dim * rows_v, dim * dim) + np.tile(np.repeat(np.arange(dim), dim), len(rows_v)),
                                  np.repeat(dim * cols_v, dim * dim) + np.tile(np.tile(np.arange(dim), dim), len(rows_v)))),
                                shape=G.shape)
        outside = Gf - Gf.multiply(covered)
        assert abs(outside).max() < 1e-12 * scale


def test_two_level_cycle_reaches_the_same_solution(case3d):
    """Two-level cycle vs single-level polynomial inside the block preconditioner: different preconditioners, same linear
    system => the same tight-tolerance solution; the cycle is selected for the linearised 3-D system.  (Its pay-off --
    half the velocity-operator applications per solve -- shows on the large grad-div dominated meshes, profiles/README.md.)"""
    c = case3d
    nsb = c.nsb
    con = c.constraints()
    out = {}
    try:
        for cyc in (1, 2):
            for prec in (32, 16):
                c.dev.set_solver_opts(velocity_cycle=cyc, precond_precision=prec)
                c.linearized(0.5, False, con)
                c.dev.assemble_pressure_matrices()
                c.dev.profile_enable(True)
                c.dev.profile_reset()
                ok, it, _ = c.dev.solve(200, 1e-2, 150)
                napp = c.dev.profile()["spmv_vel"][1]
                c.dev.profile_enable(False)
                info = c.dev.velocity_pc_info()
                assert ok and info["two_level"] == (cyc == 2), (cyc, info)
                ok2, it2, _ = c.dev.solve(3000, 1e-12, 150)
                assert ok2
                out[(cyc, prec)] = (c.dev.get_vector(nsb.NSB_SOLUTION), it, napp, it2)
        x0 = out[(1, 32)][0]
        for k, (x, it, napp, it2) in out.items():
            assert np.linalg.norm(x - x0) / np.linalg.norm(x0) < 1e-9, k
        assert out[(2, 32)][1] <= out[(1, 32)][1] + 2, {k: v[1:] for k, v in out.items()}      # no worse as a preconditioner
        # bit-reproducible from solve to solve
        c.dev.set_solver_opts()
        c.linearized(0.5, False, con)
        a = c.dev.solve(200, 1e-2, 150)
        xa = c.dev.get_vector(nsb.NSB_SOLUTION)
        b = c.dev.solve(200, 1e-2, 150)
        assert a == b and np.array_equal(xa, c.dev.get_vector(nsb.NSB_SOLUTION))
    finally:
        c.dev.set_solver_opts()
        c.linearized(0.5, False, con)
