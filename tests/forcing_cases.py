"""Shared pieces of the forcing tests (test_forcing_cpu.py, test_gpu_forcing.py).

- `ForcedOracle`: the oracle's time loop with a forcing term fn(points (n, dim), t) -> (n, dim), sampled at the mapped
  quadrature points at t and at t - dt of each assembly (dt of that assembly, so a halved retry samples t - dt/2) --
  the time semantics of the host class (DESIGN.md section 1).  oracle/assemble.py already takes the per-(cell, point)
  arrays; only the sampling is added here.
- `Manufactured`: a steady Navier-Stokes solution that the P2/P1 space represents exactly, with its body force.  Flow
  axis x (the outlet's normal), outlet plane x = L, transverse coordinates y (and z in 3-D):
      u_x = a + b y + c y^2,   u_y = k (x - L)^2,   (u_z = 0),   p = beta (x - L)
  u is divergence-free, nu du/dn - p n = 0 and p = 0 hold on x = L, and f = (u . grad) u - nu lap u + grad p.  Every
  other boundary takes Dirichlet data equal to u.  Galerkin integration by parts is exact for these degrees with
  QGaussSimplex(3), so a linearised step from u^n = u^{n-1} = u returns u, and the Newton residual vanishes at u.
  Newton's SUPG term vanishes there too (its strong residual has -nu lap u).  The linearised system's SUPG term does
  not: its rhs contracts the FIRST index of grad phi_i with u* (cpp:733) while its matrix uses (u* . grad) phi_i, so
  even a harmonic u leaves an O(tau) defect; the manufactured checks of that system run without SUPG (DESIGN.md s.5).
"""
import numpy as np

from oracle import assemble as asm, dofs as odofs, fe_tables as fe, postprocess as pp, solve as osolve


def quadrature_points(mesh):
    """(n_cells, n_q, dim): x_q = sum_v lambda_{q,v} X_v."""
    lam = fe.barycentric(fe.quadrature(mesh.dim)[0])
    return np.einsum("qv,cvd->cqd", lam, mesh.points[mesh.cells])


def sample(fn, pts, t):
    return np.asarray(fn(pts.reshape(-1, pts.shape[-1]), t), np.float64).reshape(pts.shape)


def smooth_forcing(x, t):
    """A smooth, time-dependent, non-polynomial body force of moderate size (|f| <~ 0.5) for parity runs."""
    s = 0.5 * (1.0 + 0.5 * np.sin(3.0 * t))
    f = np.empty_like(x)
    f[:, 0] = s * np.sin(2.0 * x[:, 0] + x[:, 1])
    f[:, 1] = s * np.cos(x[:, 0] - 3.0 * x[:, 1]) + 0.1 * t
    if x.shape[1] == 3:
        f[:, 2] = s * np.sin(4.0 * x[:, 2] + x[:, 0])
    return f


class ForcedOracle(osolve.Oracle):
    def __init__(self, mesh, case, forcing, **kw):
        super().__init__(mesh, case, **kw)
        assert not self.c_assembly, "the C assembly port has no forcing input"
        self.forcing = forcing
        self.qpts = quadrature_points(mesh)

    def forcing_arrays(self, dt):
        return sample(self.forcing, self.qpts, self.time), sample(self.forcing, self.qpts, self.time - dt)

    def assemble_linearized(self, p):
        con = odofs.build_constraints(self.mesh, self.dm, self.inlet(self.time), self.ids)
        out = asm.assemble(self.mesh, self.dm, self.pattern, p, con, "linearized", self.solution_old, self.solution_old_old,
                           with_pressure_matrices=self.Mp is None, forcing=self.forcing_arrays(p.dt))
        if self.Mp is None:
            self.Mp, self.Kp = out.Mp, out.Kp
        return out, con

    def assemble_newton(self, p):
        out = asm.assemble(self.mesh, self.dm, self.pattern, p, self.newton_constraints, "newton", self.current_solution,
                           self.solution_old, with_pressure_matrices=self.Mp is None, forcing=self.forcing_arrays(p.dt))
        if self.Mp is None:
            self.Mp, self.Kp = out.Mp, out.Kp
        return out


class Manufactured:
    def __init__(self, mesh, nu, a=0.3, b=2.0, c=-4.0, k=0.7, beta=0.5):
        dim = mesh.dim
        self.mesh, self.dim, self.nu = mesh, dim, nu
        self.ids = pp.boundary_ids(dim)
        outlet = np.unique(mesh.faces[mesh.face_tag == self.ids["outlet"]].ravel())
        X = mesh.points[outlet]
        self.ax = int(np.argmin(X.max(0) - X.min(0)))                 # the outlet is the plane x_ax = L
        assert np.ptp(X[:, self.ax]) < 1e-12 and np.ptp(X[:, self.ax - 1]) > 0
        self.L = float(X[0, self.ax])
        self.tr = [d for d in range(dim) if d != self.ax]             # y, (z)
        self.a, self.b, self.c, self.k, self.beta = a, b, c, k, beta

    def velocity(self, x):
        X, y = x[:, self.ax] - self.L, x[:, self.tr[0]]
        u = np.zeros_like(x)
        u[:, self.ax] = self.a + self.b * y + self.c * y * y
        u[:, self.tr[0]] = self.k * X * X
        return u

    def pressure(self, x):
        return self.beta * (x[:, self.ax] - self.L)

    def forcing(self, x, t=0.0):
        X, y = x[:, self.ax] - self.L, x[:, self.tr[0]]
        u = self.velocity(x)
        f = np.zeros_like(x)
        # (u . grad) u: u_x depends on y only, u_y on x only
        f[:, self.ax] = u[:, self.tr[0]] * (self.b + 2 * self.c * y) - 2 * self.nu * self.c + self.beta
        f[:, self.tr[0]] = 2 * self.k * X * u[:, self.ax] - 2 * self.nu * self.k
        return f

    def exact(self, dm):
        """u, p as a global DoF vector."""
        x = np.zeros(dm.n_dofs)
        sp_, comp = dm.support_points, dm.component
        vel = comp < self.dim
        x[vel] = self.velocity(sp_[vel])[np.arange(vel.sum()), comp[vel]]
        x[~vel] = self.pressure(sp_[~vel])
        return x

    def constraints(self, dm):
        """Dirichlet u on inlet, walls and cylinder, p = 0 on the outlet (same index sets as the test cases)."""
        x = self.exact(dm)
        con = odofs.Constraints(dm.n_dofs)
        for key in ("inlet", "wall", "cylinder"):
            d = odofs.boundary_dofs(self.mesh, dm, self.ids[key])
            con.add(d, x[d])
        con.add(odofs.boundary_dofs(self.mesh, dm, self.ids["outlet"], velocity=False, pressure=True), 0.0)
        return con
