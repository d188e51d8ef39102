"""The forcing input of the assembly, checked on the oracle without a GPU: a manufactured steady solution that the P2/P1
space represents exactly (tests/forcing_cases.py) must solve the linearised step and zero the Newton residual to
round-off once its body force is supplied -- a correctness pin that does not depend on the oracle agreeing with itself.
The linearised checks run without SUPG: that system's SUPG rhs is not consistent with its matrix at the exact solution
(see tests/forcing_cases.py); Newton's is, and its checks run with SUPG."""
import numpy as np
import pytest

from oracle import assemble as asm, dofs as odofs
from tests.forcing_cases import Manufactured, quadrature_points, sample

NU, DT = 1e-3, 0.02
TOL_LIN, TOL_NEWTON = 1e-10, 1e-9


def _setup(mesh):
    dm = odofs.enumerate_dofs(mesh)
    pat = odofs.make_sparsity(dm)
    ms = Manufactured(mesh, NU)
    f = sample(ms.forcing, quadrature_points(mesh), 0.0)
    return dm, pat, ms, f


def linearized_defect(mesh, theta, supg=False):
    """||A x_u - b|| / ||b|| for u^n = u^{n-1} = u (x_u: u with the constrained entries zeroed, as the elimination
    needs), and the same with the forcing left out."""
    dm, pat, ms, f = _setup(mesh)
    con = ms.constraints(dm)
    x = ms.exact(dm)
    xu = np.where(con.is_c, 0.0, x)
    p = asm.Params(dt=DT, theta=theta, nu=NU, use_supg=supg, first_step=True)
    out = []
    for forcing in ((f, f), None):
        r = asm.assemble(mesh, dm, pat, p, con, "linearized", x, x, with_pressure_matrices=False, forcing=forcing)
        A = asm.to_csr(pat, r.A, dm.n_dofs)
        out.append(np.linalg.norm(A @ xu - r.b) / np.linalg.norm(r.b))
    return out


def newton_residual(mesh, theta, supg):
    """||b(u)|| / ||b(u) without the forcing||."""
    dm, pat, ms, f = _setup(mesh)
    con = odofs.build_constraints(mesh, dm, None, ms.ids, homogeneous=True)
    x = ms.exact(dm)
    p = asm.Params(dt=DT, theta=theta, nu=NU, use_supg=supg)
    b = [asm.assemble(mesh, dm, pat, p, con, "newton", x, x, with_pressure_matrices=False, forcing=fc).b
         for fc in ((f, f), None)]
    return np.linalg.norm(b[0]) / np.linalg.norm(b[1])


def test_manufactured_solution_is_exact(golden_mesh, small_3d_mesh):
    """The fields themselves: divergence-free, the outlet conditions hold, and f is what the formula says (finite
    differences of the momentum equation at random points)."""
    for mesh in (golden_mesh("mesh-2D"), small_3d_mesh):
        ms = Manufactured(mesh, NU)
        dim = mesh.dim
        rng = np.random.default_rng(5)
        x = mesh.points.min(0) + rng.uniform(0, 1, (50, dim)) * np.ptp(mesh.points, 0)
        e = 1e-4
        grad = np.zeros((50, dim, dim))                         # grad[i][c][d] = d u_c / d x_d
        lap = np.zeros((50, dim))
        gp = np.zeros((50, dim))
        for d in range(dim):
            dx = np.zeros(dim)
            dx[d] = e
            up, um, u0 = ms.velocity(x + dx), ms.velocity(x - dx), ms.velocity(x)
            grad[:, :, d] = (up - um) / (2 * e)
            lap += (up - 2 * u0 + um) / (e * e)
            gp[:, d] = (ms.pressure(x + dx) - ms.pressure(x - dx)) / (2 * e)
        u = ms.velocity(x)
        assert np.abs(np.trace(grad, axis1=1, axis2=2)).max() < 1e-9
        f = np.einsum("icd,id->ic", grad, u) - NU * lap + gp
        assert np.abs(f - ms.forcing(x)).max() < 1e-6
        out = x.copy()
        out[:, ms.ax] = ms.L                                    # on the outlet plane
        dx = np.zeros(dim)
        dx[ms.ax] = e
        dudn = (ms.velocity(out + dx) - ms.velocity(out - dx)) / (2 * e)
        assert np.abs(NU * dudn).max() < 1e-12 and np.abs(ms.pressure(out)).max() == 0.0


@pytest.mark.parametrize("theta", [1.0, 0.5])
def test_linearized_step_reproduces_manufactured_2d(golden_mesh, theta):
    forced, unforced = linearized_defect(golden_mesh("mesh-2D"), theta)
    print("mesh-2D linearised, theta %.1f: defect %.2e (without the forcing %.2e)" % (theta, forced, unforced))
    assert forced < TOL_LIN and unforced > 1e-3


@pytest.mark.parametrize("supg", [False, True])
def test_newton_residual_vanishes_at_manufactured_2d(golden_mesh, supg):
    r = newton_residual(golden_mesh("mesh-2D"), 1.0, supg)
    print("mesh-2D Newton, SUPG %s: residual ratio %.2e" % (supg, r))
    assert r < TOL_NEWTON


@pytest.mark.parametrize("theta", [1.0, 0.5])
def test_linearized_step_reproduces_manufactured_3d(small_3d_mesh, theta):
    forced, unforced = linearized_defect(small_3d_mesh, theta)
    print("3-D linearised, theta %.1f: defect %.2e (without the forcing %.2e)" % (theta, forced, unforced))
    assert forced < TOL_LIN and unforced > 1e-3


@pytest.mark.parametrize("theta", [1.0, 0.5])
def test_newton_supg_residual_vanishes_at_manufactured_3d(small_3d_mesh, theta):
    r = newton_residual(small_3d_mesh, theta, True)
    print("3-D Newton + SUPG, theta %.1f: residual ratio %.2e" % (theta, r))
    assert r < TOL_NEWTON
