"""GPU (-m gpu): the kernels of the block preconditioner as operators, against float64 references built from the device's
own assembled matrix (assembly itself is pinned to the oracle in test_gpu_parity.py):

  1. the packed copy of B = Dinv F (k_vel_pack, k_coarse_pack) against Dinv F rounded as the kernels round it;
  2. the persistent streamed operator k_vel_stream, MODE 2 / 3 / 4 on both levels, row by row against the fp64 product of
     the stored values, on meshes whose tiles wrap the TMA ring several times per CTA;
  3. the velocity preconditioner (product-form polynomial, two-level cycle) rebuilt from the exported roots and operators;
  4. the Schur side of the block preconditioner (k_schur_rhs, Jacobi-Chebyshev on M_p, the K_p V-cycle);
  5. the residual GMRES reports, recomputed from the returned iterate.

Tolerances were set from runs on a B200; each is stated next to the largest error measured there."""
import math

import numpy as np
import pytest
import scipy.sparse as sp

from oracle import dofs as odofs, postprocess as pp
from tests.conftest import synthetic_state
from tests.test_gpu_parity import _p1_prolongation
from tools import meshgen

pytestmark = pytest.mark.gpu

# mesh key -> (mesh, test case); the last two have enough stream tiles to wrap the ring of every CTA
MESHES = {"2d": ("mesh-2D", "2D-2"), "3d": ("small_3d", "3D-2Z"), "2d100": ("mesh-2D-100", "2D-2"), "3d5": ("mesh_3d(5)", "3D-2Z")}
RING_WRAP = ("2d100", "3d5")

# tolerances; the largest error measured on a B200 (148 SMs, 1000 W power limit) over all parametrizations is on the right
TOL_STREAM = 1e-14      # per row, relative to the row's sum of |terms|                  measured 9.9e-16
TOL_SPMV = 1e-14        # per row, relative to (|A||x|)_i                                measured 1.03e-15
TOL_PC = 1e-13          # relative L2, velocity preconditioner vs its numpy rebuild      measured 7.2e-15
TOL_ID = 1e-13          # residual-polynomial identity, relative to |z|                  measured 3.3e-15
TOL_SCHUR = 1e-13       # k_schur_rhs, M_p Chebyshev, linearity of P^-1                  measured 2.8e-15
TOL_SYM = 1e-13         # symmetry of the K_p V-cycle, relative to |Va||b|               measured 1.3e-15
TOL_GMRES = 1e-10       # reported vs recomputed preconditioned residual, relative       measured 3.3e-12
EPS = 2.0 ** -53


class System:
    """A mesh on the device with the synthetic state of the parity tests, linearised (theta = 0.5, first-order u*) or Newton."""

    def __init__(self, nsb, mesh, case):
        self.nsb, self.mesh, self.dim = nsb, mesh, mesh.dim
        self.tc = pp.TEST_CASES[case]
        self.dm = dm = odofs.enumerate_dofs(mesh)
        self.n_u, self.n_p, self.N = dm.n_u, dm.n_p, dm.n_dofs
        self.nu = pp.viscosity(self.dim, self.tc["U_m"], self.tc["Re"])
        self.dt = 0.01 if self.dim == 3 else 0.02
        self.dev = nsb.Device(self.dim)
        self.dev.upload_mesh(mesh.points, mesh.cells, dm.cell_dofs, dm.n_u, dm.n_p)
        assert np.array_equal(self.dev.row_gids(), np.arange(self.N))
        self.un, self.unm1 = synthetic_state(dm, self.dim, self.tc["U_m"])
        ids = pp.boundary_ids(self.dim)
        prof = pp.inlet_profile(self.dim, self.tc["U_m"], self.tc["time_dep"], self.tc["T_ramp"], 1.0)
        self.cons = {"lin": odofs.build_constraints(mesh, dm, prof, ids),
                     "newton": odofs.build_constraints(mesh, dm, prof, ids, homogeneous=True)}
        # pressure DoF -> mesh vertex, and the P1 prolongation with its columns in level-1 numbering (dim * pressure id + comp)
        pvert = np.zeros(self.n_p, np.int64)
        for k in range(self.dim + 1):
            pvert[dm.cell_dofs[:, k * (self.dim + 1) + self.dim].astype(np.int64) - self.n_u] = mesh.cells[:, k]
        perm = (self.dim * pvert[:, None] + np.arange(self.dim)[None, :]).ravel()
        self.P = _p1_prolongation(mesh, dm)[:, perm].tocsr()
        vdof = np.zeros(self.dim * mesh.n_vertices, np.int64)
        for v in range(self.dim + 1):
            for k in range(self.dim):
                vdof[self.dim * mesh.cells[:, v].astype(np.int64) + k] = dm.cell_dofs[:, v * (self.dim + 1) + k]
        self.vdof = vdof[perm]                      # fine velocity DoF of every coarse DoF
        self.state = None

    def assemble(self, state, pressure=True, **opts):
        nsb, dev = self.nsb, self.dev
        con = self.cons[state]
        dev.set_solver_opts(**opts)
        dev.set_constraints(con.dofs, con.val[con.dofs])
        if state == "lin":
            dev.set_params(self.dt, 0.5, self.nu, 1.0, 0.1, self.tc["supg"], True)
            dev.set_vector(nsb.NSB_SOLUTION_OLD, self.un)
            dev.set_vector(nsb.NSB_SOLUTION_OLD_OLD, self.unm1)
            dev.assemble_linearized()
        else:
            pk = np.zeros(self.N)
            pk[self.n_u:] = 0.05 * np.random.default_rng(7).uniform(-1, 1, self.n_p)
            dev.set_params(self.dt, 0.5, self.nu, 1.0, 0.1, self.tc["supg"], False)
            dev.set_vector(nsb.NSB_CURRENT_SOLUTION, self.un + pk)
            dev.set_vector(nsb.NSB_SOLUTION_OLD, self.unm1)
            dev.assemble_newton()
        if pressure:
            dev.assemble_pressure_matrices()
        self.state = state
        return con

    def matrix(self):
        rp, col = self.dev.pattern()
        return sp.csr_matrix((self.dev.matrix_values(), col.astype(np.int64), rp), shape=(self.N, self.N))


@pytest.fixture(scope="module")
def systems(nsb, golden_mesh, small_3d_mesh):
    made = {}

    def get(key):
        if key not in made:
            name, case = MESHES[key]
            mesh = small_3d_mesh if key == "3d" else meshgen.mesh_3d(5) if key == "3d5" else golden_mesh(name)
            made[key] = System(nsb, mesh, case)
        return made[key]

    yield get
    for s in made.values():
        s.dev.close()


_SMS = []


def multi_processor_count():
    if not _SMS:
        import torch
        _SMS.append(torch.cuda.get_device_properties(0).multi_processor_count)
    return _SMS[0]


def assert_regime(s, key, prec, tiles, level=0):
    """The pipeline regime a parametrization claims: ring wraps (more than 2 * STAGES tiles per CTA) on the large meshes, at most
    two tiles per CTA on the small ones (fine level).  STAGES = 2 for 3-D fp32, else 3 (VsLayout)."""
    sms = multi_processor_count()
    stages = 2 if (s.dim == 3 and prec == 32) else 3
    per_cta = math.ceil(tiles / min(tiles, sms))
    print(f"[{key} level {level} fp{prec}] stream tiles {tiles}, {sms} SMs, {stages} stages: up to {per_cta} tiles per CTA")
    if level == 0 and prec != 64:
        if key in RING_WRAP:
            assert tiles > 2 * stages * sms, (tiles, stages, sms)
        else:
            assert tiles <= 2 * sms, (tiles, sms)


# ---- block helpers ------------------------------------------------------------------------------------------------------
def node_blocks(M, dim):
    """dim x dim node blocks of a sparse matrix: sorted keys row_node * n_col_nodes + col_node, values [nblocks, dim, dim]."""
    M = M.tocoo()
    ncol = M.shape[1] // dim
    key = (M.row // dim).astype(np.int64) * ncol + M.col // dim
    uk, inv = np.unique(key, return_inverse=True)
    V = np.zeros((len(uk), dim, dim))
    V[inv, M.row % dim, M.col % dim] = M.data
    return uk, V, ncol


def block_inverse_diag(uk, V, ncol, n_nodes):
    nodes = np.arange(n_nodes, dtype=np.int64)
    pos = np.searchsorted(uk, nodes * ncol + nodes)
    assert np.array_equal(uk[pos], nodes * ncol + nodes)
    return np.linalg.inv(V[pos])


def scaled_blocks(uk, V, ncol, dinv):
    """blocks of Dinv M in the order of uk"""
    return np.einsum("nij,njk->nik", dinv[uk // ncol], V)


def blocks_to_csr(rows, cols, V, dim, n):
    r = (dim * rows)[:, None, None] + np.arange(dim)[None, :, None]
    c = (dim * cols)[:, None, None] + np.arange(dim)[None, None, :]
    r, c = np.broadcast_arrays(r, c)
    return sp.csr_matrix((V.ravel(), (r.ravel(), c.ravel())), shape=(n, n))


def block_diag_csr(dinv, dim):
    nn = len(dinv)
    return blocks_to_csr(np.arange(nn), np.arange(nn), dinv, dim, dim * nn)


def exported_keys(op, ncol):
    rows = np.repeat(op["row_gid"], np.diff(op["rowptr"]))
    return rows, rows * ncol + op["col_gid"]


def check_pack(op, uk, ref, absref, ncol, prec, what):
    """Every (node, neighbour) block present once; values finite, within one ulp of the reference rounded fp64 -> fp32 (-> fp16)
    as the pack kernels round (plus the fp64 rounding of the product, absref = |Dinv||F|: entries that cancel to zero, such as
    the off-diagonals of Dinv D = I, come out as +-1e-20 in fp64 and survive in fp32), and almost all bit-identical."""
    rows, ke = exported_keys(op, ncol)
    assert np.array_equal(np.sort(ke), uk), what
    pos = np.searchsorted(uk, ke)
    want, noise = ref[pos], 8 * EPS * absref[pos]
    r32 = want.astype(np.float32)
    r = r32.astype(np.float16) if prec == 16 else r32
    got = op["vals"]
    assert np.all(np.isfinite(got)) and np.all(np.isfinite(r)), what
    ulp = np.spacing(np.abs(r)).astype(np.float64)
    diff = np.abs(got - r.astype(np.float64))
    well = np.abs(want) > 1e6 * noise              # not a cancellation: the rounding is determined by fp64
    same = float(np.mean(diff[well] == 0))
    print(f"{what}: {len(ke)} blocks, bit-identical fraction {same:.6f} of {int(well.sum())} well-determined values, "
          f"max |diff| / (ulp + fp64 noise) {np.max(diff / (ulp + noise)):.3g}")
    assert np.all(diff <= ulp + noise), what
    assert same > 0.999, (what, same)


def check_stream(dev, level, B, Babs, n, rng, what):
    """MODE 2 / 3 / 4 of the level's operator on random vectors, per row against the fp64 product, bit-reproducible."""
    x, u, p = rng.standard_normal((3, n))
    cu, ct, cpu, cpy = cf = (0.7, -1.3, 0.4, 0.9)
    t, bt = B @ x, Babs @ np.abs(x)
    worst = 0.0
    for mode in (2, 3, 4):
        out = dev.apply_velocity_operator(level, mode, x, u, p, cf)
        again = dev.apply_velocity_operator(level, mode, x, u, p, cf)
        y, pn = out if mode == 3 else (out, None)
        if mode == 3:
            assert np.array_equal(y, again[0]) and np.array_equal(pn, again[1]), (what, mode)
        else:
            assert np.array_equal(y, again), (what, mode)
        yr, yb = (t, bt) if mode == 2 else (cu * u + ct * t, abs(cu) * np.abs(u) + abs(ct) * bt)
        e = np.abs(y - yr)
        assert np.all(e <= TOL_STREAM * yb), (what, mode, np.max(e / np.maximum(yb, 1e-300)))
        worst = max(worst, float(np.max(e / np.maximum(yb, 1e-300))))
        if mode == 3:
            pr = p + cpu * u + cpy * yr
            pb = np.abs(p) + abs(cpu) * np.abs(u) + abs(cpy) * yb
            e = np.abs(pn - pr)
            assert np.all(e <= TOL_STREAM * pb), (what, "poly", np.max(e / pb))
            worst = max(worst, float(np.max(e / pb)))
    print(f"{what}: stream MODE 2/3/4 worst row error / row bound {worst:.3g}")
    return worst


@pytest.mark.parametrize("prec", [16, 32, 64])
@pytest.mark.parametrize("state", ["lin", "newton"])
@pytest.mark.parametrize("key", ["2d", "3d", "2d100", "3d5"])
def test_packed_operator_and_stream(systems, key, state, prec):
    """Pack (k_vel_pack, k_coarse_pack) and stream (k_vel_stream MODE 2/3/4) on both levels, and nsb_spmv per row."""
    s = systems(key)
    dev, dim, n_u = s.dev, s.dim, s.n_u
    s.assemble(state, pressure=False, precond_precision=prec)
    rng = np.random.default_rng(11)
    A = s.matrix()
    F = A[:n_u, :n_u]
    uk, V, ncol = node_blocks(F, dim)
    dinv = block_inverse_diag(uk, V, ncol, n_u // dim)
    Bref = scaled_blocks(uk, V, ncol, dinv)
    op = dev.velocity_operator(0)
    assert op["precision"] == prec and op["tiles"] == dev.velocity_operator_info()["tiles"]
    assert_regime(s, key, prec, op["tiles"])
    tag = f"[{key} {state} fp{prec}]"
    if prec == 64:
        # no packed copy: the generic fp64 row kernel applies Dinv (F x)
        assert len(op["col_gid"]) == 0
        B = blocks_to_csr(uk // ncol, uk % ncol, Bref, dim, n_u)
        Babs = abs(block_diag_csr(dinv, dim)) @ abs(F)
    else:
        check_pack(op, uk, Bref, scaled_blocks(uk, np.abs(V), ncol, np.abs(dinv)), ncol, prec, tag + " fine pack")
        rows, _ = exported_keys(op, ncol)
        B = blocks_to_csr(rows, op["col_gid"], op["vals"], dim, n_u)
        Babs = abs(B)
    check_stream(dev, 0, B, Babs, n_u, rng, tag + " fine")
    if state == "lin" and prec != 64:
        # coarse level: Dinv_c times the exported Galerkin operator
        rg, rp, cg, cv = dev.coarse_operator()
        crow = np.repeat(rg, np.diff(rp))
        G = blocks_to_csr(crow, cg, cv, dim, dim * s.n_p)
        ukc, Vc, nc = node_blocks(G, dim)
        dinv_c = block_inverse_diag(ukc, Vc, nc, s.n_p)
        opc = dev.velocity_operator(1)
        assert opc["precision"] == prec
        assert_regime(s, key, prec, opc["tiles"], level=1)
        check_pack(opc, ukc, scaled_blocks(ukc, Vc, nc, dinv_c), scaled_blocks(ukc, np.abs(Vc), nc, np.abs(dinv_c)), nc, prec,
                   tag + " coarse pack")
        rows_c, _ = exported_keys(opc, nc)
        Bc = blocks_to_csr(rows_c, opc["col_gid"], opc["vals"], dim, dim * s.n_p)
        check_stream(dev, 1, Bc, abs(Bc), dim * s.n_p, rng, tag + " coarse")
    if prec == 16:
        x = rng.standard_normal(s.N)
        y = dev.spmv(x)
        e = np.abs(y - A @ x)
        bound = abs(A) @ np.abs(x)
        print(f"{tag} nsb_spmv worst row error / row bound {np.max(e / np.maximum(bound, 1e-300)):.3g}")
        assert np.all(e <= TOL_SPMV * bound)


# ---- velocity preconditioner --------------------------------------------------------------------------------------------
def poly_ref(B, roots, z0, defect=None):
    """p(B) z0 in the product form of apply_poly (Leja order, one real quadratic step per conjugate pair)."""
    if defect == "drop_root":
        roots = np.delete(roots, len(roots) // 2)
    ct = 1.0 if defect == "ct_sign" else -1.0
    prod, poly = z0.copy(), np.zeros_like(z0)
    for k, th in enumerate(roots):
        last = k + 1 == len(roots)
        a, b = th.real, th.imag
        if b == 0.0:
            poly = poly + prod / a
            if not last:
                prod = prod + ct * (B @ prod) / a
        else:
            m2 = a * a + b * b
            tmp = 2.0 * a * prod + ct * (B @ prod)
            poly = poly + tmp / m2
            if not last:
                prod = prod + ct * (B @ tmp) / m2
    return poly


def residual_poly(B, roots, z):
    """prod_k (I - B / theta_k) z, a real quadratic factor per conjugate pair"""
    r = z.copy()
    for th in roots:
        a, b = th.real, th.imag
        if b == 0.0:
            r = r - (B @ r) / a
        else:
            m2 = a * a + b * b
            Br = B @ r
            r = r - (2.0 * a / m2) * Br + (B @ Br) / m2
    return r


def velocity_pc_ref(s, L, x_u, defect=None):
    """DESIGN section 4: single level p(B) Dinv x; two-level y0 = diag(free_f) P p_c(B_c) Dinv_c diag(free_c) P^T x,
    y = y0 + q(B)(Dinv x - B y0).  Returns (y, y0)."""
    u0 = L["Dinv"] @ x_u
    if not L["two_level"]:
        return poly_ref(L["B"], L["roots"], u0, defect), np.zeros_like(x_u)
    rc = s.P.T @ x_u
    if defect != "no_mask":
        rc = np.where(L["free_c"], rc, 0.0)
    pc = poly_ref(L["Bc"], L["roots_c"], L["Dinv_c"] @ rc, "drop_root" if defect == "drop_root" else None)
    y0 = np.where(L["free_f"], s.P @ pc, 0.0)
    ct = 1.0 if defect == "ct_sign" else -1.0
    return y0 + poly_ref(L["B"], L["roots"], u0 + ct * (L["B"] @ y0)), y0


def exported_levels(s, two_level):
    dev, dim, n_u = s.dev, s.dim, s.n_u
    A = s.matrix()
    uk, V, ncol = node_blocks(A[:n_u, :n_u], dim)
    dinv = block_inverse_diag(uk, V, ncol, n_u // dim)
    op = dev.velocity_operator(0)
    rows, _ = exported_keys(op, ncol)
    L = dict(two_level=two_level, A=A, Dinv=block_diag_csr(dinv, dim), roots=dev.velocity_pc_roots(0),
             B=blocks_to_csr(rows, op["col_gid"], op["vals"], dim, n_u))
    if two_level:
        rg, rp, cg, cv = dev.coarse_operator()
        ukc, Vc, nc = node_blocks(blocks_to_csr(np.repeat(rg, np.diff(rp)), cg, cv, dim, dim * s.n_p), dim)
        opc = dev.velocity_operator(1)
        rows_c, _ = exported_keys(opc, nc)
        con = s.cons[s.state]
        L.update(Bc=blocks_to_csr(rows_c, opc["col_gid"], opc["vals"], dim, dim * s.n_p), roots_c=dev.velocity_pc_roots(1),
                 Dinv_c=block_diag_csr(block_inverse_diag(ukc, Vc, nc, s.n_p), dim),
                 free_c=~con.is_c[s.vdof], free_f=~con.is_c[:n_u])
    return L


PC_CASES = {
    "3d-lin-two-level": ("3d", "lin", {}, True),
    "3d-lin-two-level-fp32": ("3d", "lin", dict(precond_precision=32), True),
    "3d-lin-chebyshev": ("3d", "lin", dict(velocity_cycle=1), False),
    "2d-lin-harmonic-ritz": ("2d", "lin", {}, False),
    "3d-newton": ("3d", "newton", {}, False),
    "3d5-lin-two-level": ("3d5", "lin", {}, True),
    "2d100-lin-harmonic-ritz": ("2d100", "lin", {}, False),
}


@pytest.mark.parametrize("case", list(PC_CASES))
def test_velocity_preconditioner(systems, case):
    """nsb_apply_velocity_pc equals its rebuild from the exported roots and operators, satisfies the residual-polynomial
    identity, and the rebuild would see one dropped root, a missing restriction mask or a flipped sign."""
    key, state, opts, two = PC_CASES[case]
    s = systems(key)
    dev, n_u = s.dev, s.n_u
    try:
        s.assemble(state, **opts)
        ok, it, _ = dev.solve(200, 1e-2, 150)
        assert ok
        info = dev.velocity_pc_info()
        assert info["two_level"] == two, info
        L = exported_levels(s, two)
        roots = L["roots"]
        assert_regime(s, key, dev.get_solver_opts()["precond_precision"], dev.velocity_operator_info()["tiles"])
        if case.startswith("2d"):
            assert np.any(roots.imag > 0), roots          # harmonic Ritz values with complex pairs
        if "chebyshev" in case or two:
            assert np.all(roots.imag == 0), roots
        if two:
            assert len(L["roots_c"]) == info["coarse_degree"] > 0
        print(f"[{case}] {it} GMRES iterations, two-level {two}, fine roots {len(roots)} "
              f"({int(np.sum(roots.imag > 0))} pairs)" + (f", coarse roots {len(L['roots_c'])}" if two else ""))
        x = np.random.default_rng(5).standard_normal(s.N)
        y = dev.apply_velocity_pc(x)[:n_u]
        assert np.array_equal(y, dev.apply_velocity_pc(x)[:n_u])
        ref, y0 = velocity_pc_ref(s, L, x[:n_u])
        err = np.linalg.norm(y - ref) / np.linalg.norm(ref)
        # residual-polynomial identity on the smoothing / polynomial part: z - B (y - y0) = prod_k (I - B / theta_k) z
        z = L["Dinv"] @ x[:n_u] - L["B"] @ y0
        eid = np.linalg.norm(z - L["B"] @ (y - y0) - residual_poly(L["B"], roots, z)) / np.linalg.norm(z)
        print(f"[{case}] relative error vs rebuild {err:.3g}, residual-polynomial identity {eid:.3g}")
        assert err <= TOL_PC and eid <= TOL_ID, (err, eid)
        for defect in ("drop_root", "ct_sign") + (("no_mask",) if two else ()):
            bad, _ = velocity_pc_ref(s, L, x[:n_u], defect)
            d = np.linalg.norm(bad - ref) / np.linalg.norm(ref)
            print(f"[{case}] defect {defect}: relative change {d:.3g}")
            assert d >= 100 * TOL_PC, (defect, d)
    finally:
        dev.set_solver_opts()


# ---- Schur side ---------------------------------------------------------------------------------------------------------
def jacobi_chebyshev(M, lmax, degree, b):
    """csr_cheb with a zero initial guess on the interval [1.1 lmax / 6, 1.1 lmax]"""
    hi, lo = 1.1 * lmax, 1.1 * lmax / 6.0
    theta, delta = 0.5 * (hi + lo), 0.5 * (hi - lo)
    sigma = theta / delta
    rho = 1.0 / sigma
    dinv = 1.0 / M.diagonal()
    d = dinv * b / theta
    x = d.copy()
    for _ in range(1, degree):
        rho_new = 1.0 / (2.0 * sigma - rho)
        c1, c2 = rho_new * rho, 2.0 * rho_new / delta
        rho = rho_new
        d = c1 * d + c2 * dinv * (b - M @ x)
        x = x + d
    return x


@pytest.mark.parametrize("key", ["2d", "3d", "2d100", "3d5"])
def test_schur_side(systems, key):
    """P^-1 = [F~^-1, 0; -S~^-1 B F~^-1, S~^-1] with S~^-1 t = -(rho/dt) V(t) - cm C(t): velocity part bitwise the velocity
    preconditioner, pressure part a function of t = x_p - B y_u only (k_schur_rhs), C the Jacobi-Chebyshev of M_p, V a
    symmetric positive V-cycle; P^-1 linear and bit-reproducible."""
    s = systems(key)
    dev, n_u, N = s.dev, s.n_u, s.N
    rng = np.random.default_rng(13)
    try:
        s.assemble("lin")
        dev.solve(200, 1e-2, 150)            # sets the preconditioner up; its convergence is not what is checked here
        A = s.matrix()
        x = rng.standard_normal(N)
        y = dev.apply_preconditioner(x)
        yu = dev.apply_velocity_pc(x)[:n_u]
        assert np.array_equal(y[:n_u], yu)
        # k_schur_rhs: the pressure part sees x only through t = x_p - B y_u
        t = x[n_u:] - A[n_u:, :n_u] @ yu
        y2 = dev.apply_preconditioner(np.concatenate([np.zeros(n_u), t]))
        e_rhs = np.linalg.norm(y2[n_u:] - y[n_u:]) / np.linalg.norm(y[n_u:])
        # two mass coefficients isolate C(t) (M_p Chebyshev), a tiny one the V-cycle
        opts = dev.get_solver_opts()
        rp, col, val = dev.pressure_matrix(0)
        Mp = sp.csr_matrix((val, col, rp), shape=(s.n_p, s.n_p))
        lmax = dev.pressure_pc_info()["mp_lambda_max"]
        rho_dt = 1.0 / s.dt

        def pressure_part(tv, cm):
            dev.set_solver_opts(**dict(opts, schur_mass_coeff=cm))
            assert dev.pressure_pc_info()["mass_coeff"] == cm
            return dev.apply_preconditioner(np.concatenate([np.zeros(n_u), tv]))[n_u:]

        tr = rng.standard_normal(s.n_p)
        C = (pressure_part(tr, 10.0) - pressure_part(tr, 30.0)) / 20.0
        Cref = jacobi_chebyshev(Mp, lmax, opts["cheb_degree_Mp"], tr)
        e_cheb = np.linalg.norm(C - Cref) / np.linalg.norm(Cref)
        cs = 1e-8

        def vcycle(tv):
            return -(pressure_part(tv, cs) + cs * jacobi_chebyshev(Mp, lmax, opts["cheb_degree_Mp"], tv)) / rho_dt

        a, b = rng.standard_normal((2, s.n_p))
        Va, Vb = vcycle(a), vcycle(b)
        e_sym = abs(Va @ b - a @ Vb) / (np.linalg.norm(Va) * np.linalg.norm(b))
        assert Va @ a > 0 and Vb @ b > 0
        rp, col, val = dev.pressure_matrix(1)
        Kp = sp.csr_matrix((val, col, rp), shape=(s.n_p, s.n_p))
        e = rng.standard_normal(s.n_p)
        r = e - vcycle(Kp @ e)
        contraction = math.sqrt((r @ (Kp @ r)) / (e @ (Kp @ e)))
        dev.set_solver_opts(**opts)
        # linear and bit-reproducible
        z = rng.standard_normal(N)
        yz = dev.apply_preconditioner(z)
        ylin = dev.apply_preconditioner(2.0 * x - 3.0 * z)
        e_lin = np.linalg.norm(ylin - (2.0 * y - 3.0 * yz)) / np.linalg.norm(ylin)
        assert np.array_equal(yz, dev.apply_preconditioner(z))
        print(f"[{key}] k_schur_rhs {e_rhs:.3g}, M_p Chebyshev {e_cheb:.3g}, V-cycle symmetry {e_sym:.3g}, "
              f"K_p-norm contraction {contraction:.3g}, linearity {e_lin:.3g}")
        assert e_rhs <= TOL_SCHUR and e_cheb <= TOL_SCHUR and e_lin <= TOL_SCHUR and e_sym <= TOL_SYM
    finally:
        dev.set_solver_opts()


# ---- GMRES ----------------------------------------------------------------------------------------------------------------
GMRES_CASES = {
    "converged": ("lin", dict(max_it=200, tol_rel=1e-2, n_tmp_vectors=150)),
    "max_it": ("newton", dict(max_it=7, tol_rel=1e-12, n_tmp_vectors=150)),
    "restarted": ("lin", dict(max_it=200, tol_rel=1e-2, n_tmp_vectors=10)),
}
# (Far below the 1e-2 rule the two part from each other at the rounding floor of the recomputation: at 1e-8 * |b| they agreed
# to 5e-6 relative, 1e-14 of |P^-1 b|.)


@pytest.mark.parametrize("case", list(GMRES_CASES))
@pytest.mark.parametrize("key", ["2d", "3d"])
def test_gmres_reports_the_true_residual(systems, key, case):
    """The residual nsb_solve reports (what the 1e-2 stopping rule decides on) is |P^-1 (b - A x)| of the iterate it returns
    (constrained entries zero before constraints.distribute: b_c = 0, resp. homogeneous constraints)."""
    state, kw = GMRES_CASES[case]
    s = systems(key)
    dev, nsb = s.dev, s.nsb
    con = s.assemble(state)
    ok, it, res = dev.solve(**kw)
    if case == "max_it":
        assert not ok and it == 7
    else:
        assert ok
    if case == "restarted":
        assert it > kw["n_tmp_vectors"] - 2, it
    x = dev.get_vector(nsb.NSB_SOLUTION)
    b = dev.get_vector(nsb.NSB_RHS)
    assert np.all(b[con.is_c] == 0) and np.all(x[con.is_c] == con.val[con.is_c])
    x[con.is_c] = 0.0
    true = np.linalg.norm(dev.apply_preconditioner(b - dev.spmv(x)))
    rel = abs(true - res) / true
    print(f"[{key} {case}] rc {0 if ok else 1}, {it} iterations, reported {res:.6g}, recomputed {true:.6g}, relative {rel:.3g}")
    assert rel <= TOL_GMRES, (res, true)
