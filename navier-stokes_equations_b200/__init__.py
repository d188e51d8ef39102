"""ctypes bindings of libnsb200.so (include/nsb200.h) and libnsbhost.so (include/nsb200_host.h).

Thin bindings only: the product is the CUDA/C++ behind the C ABI.  There is no CPU
fallback -- loading fails loudly if the shared library is missing, and every call raises
`NsbError` with the library's own message on a non-zero/negative return code.

The directory name contains a '-', so it is imported by path: `import nsb200` (nsb200.py at the repository root).
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NSB200_LIB", os.path.join(_HERE, "libnsb200.so"))   # override: kernel-variant experiments

NSB_SOLUTION_OLD, NSB_SOLUTION_OLD_OLD, NSB_CURRENT_SOLUTION, NSB_SOLUTION, NSB_RHS = 0, 1, 2, 3, 4
NSB_FORCING_NEW, NSB_FORCING_OLD = 0, 1
PROFILE_CLASSES = ("asm_context", "asm_rows", "spmv", "spmv_vel", "schur", "amg", "orth", "other", "asm_pack", "coarse", "asm_coarse", "forcing")


class NsbError(RuntimeError):
    pass


class NsbParams(C.Structure):
    _fields_ = [("dt", C.c_double), ("theta", C.c_double), ("nu", C.c_double), ("rho", C.c_double),
                ("gamma", C.c_double), ("use_supg", C.c_int32), ("first_order_ustar", C.c_int32)]


class NsbSolverOpts(C.Structure):
    _fields_ = [("poly_degree_F", C.c_int32), ("poly_refresh", C.c_int32), ("poly_kind", C.c_int32), ("poly_target", C.c_double), ("cheb_degree_Mp", C.c_int32),
                ("amg_smoother_degree", C.c_int32), ("schur_mass_coeff", C.c_double), ("reorthogonalize", C.c_int32), ("precond_precision", C.c_int32),
                ("precond_operator", C.c_int32), ("velocity_cycle", C.c_int32), ("smoother_degree", C.c_int32),
                ("smoother_lo_frac", C.c_double), ("coarse_degree", C.c_int32), ("smoother_hi_factor", C.c_double)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NsbError("libnsb200.so is not built (run `python -c 'import __graft_entry__ as g; g.build()'`); "
                           "there is no CPU fallback")
        _lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        _lib.nsb_last_error.restype = C.c_char_p
    return _lib


def _p(a, ctype):
    return a.ctypes.data_as(C.POINTER(ctype))


def check_forcing_source(dim, src):
    """Compile a forcing source for sm_100a without a GPU (nsb_check_forcing_source); raises NsbError with NVRTC's log."""
    buf = C.create_string_buffer(1 << 16)
    if lib().nsb_check_forcing_source(int(dim), src.encode(), buf, C.c_size_t(len(buf))) != 0:
        raise NsbError(buf.value.decode())


class Device:
    """One nsb_handle.  Methods mirror include/nsb200.h one to one."""

    def __init__(self, dim, device=0):
        self.dim = dim
        self.h = C.c_void_p()
        L = lib()
        rc = L.nsb_create(dim, device, C.byref(self.h))
        if rc != 0:
            msg = L.nsb_last_error(self.h).decode() if self.h else "nsb_create failed"
            if self.h:
                L.nsb_destroy(self.h)
                self.h = None
            raise NsbError(msg)
        self.n_dofs = 0

    def _ck(self, rc, soft=()):
        if rc != 0 and rc not in soft:
            raise NsbError(lib().nsb_last_error(self.h).decode())
        return rc

    def close(self):
        if self.h:
            lib().nsb_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- setup
    def comm_init(self, rank, nranks, uid: bytes):
        buf = C.create_string_buffer(uid, 128)
        self._ck(lib().nsb_comm_init(self.h, rank, nranks, buf))

    @staticmethod
    def comm_unique_id() -> bytes:
        buf = C.create_string_buffer(128)
        if lib().nsb_comm_unique_id(buf) != 0:
            raise NsbError("ncclGetUniqueId failed")
        return buf.raw

    def upload_mesh(self, coords, cell_vertices, cell_dofs, n_u, n_p, cell_part=None):
        coords = np.ascontiguousarray(coords, np.float64)
        cv = np.ascontiguousarray(cell_vertices, np.uint32)
        cd = np.ascontiguousarray(cell_dofs, np.uint32)
        part = None if cell_part is None else np.ascontiguousarray(cell_part, np.int32)
        self.n_dofs = int(n_u + n_p)
        self._ck(lib().nsb_upload_mesh(self.h, C.c_int64(coords.shape[0]), _p(coords, C.c_double),
                                        C.c_int64(cv.shape[0]), _p(cv, C.c_uint32), _p(cd, C.c_uint32),
                                        C.c_int64(n_u), C.c_int64(n_p),
                                        _p(part, C.c_int32) if part is not None else None))

    def sizes(self):
        a, b, c = C.c_int64(), C.c_int64(), C.c_int64()
        self._ck(lib().nsb_get_sizes(self.h, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    def block_nnz(self):
        v = [C.c_int64() for _ in range(4)]
        self._ck(lib().nsb_get_block_nnz(self.h, *[C.byref(x) for x in v]))
        return dict(uu=v[0].value, up=v[1].value, pu=v[2].value, pp=v[3].value)

    def pattern(self):
        n, nnz, _ = self.sizes()
        rp = np.empty(n + 1, np.int64)
        col = np.empty(nnz, np.uint32)
        self._ck(lib().nsb_get_pattern(self.h, _p(rp, C.c_int64), _p(col, C.c_uint32)))
        return rp, col

    def row_gids(self):
        n, _, _ = self.sizes()
        g = np.empty(n, np.int64)
        self._ck(lib().nsb_get_row_gids(self.h, _p(g, C.c_int64)))
        return g

    # ---- per-step inputs
    def set_constraints(self, dofs, vals):
        d = np.ascontiguousarray(dofs, np.uint32)
        v = np.ascontiguousarray(vals, np.float64)
        self._ck(lib().nsb_set_constraints(self.h, C.c_int64(d.shape[0]), _p(d, C.c_uint32), _p(v, C.c_double)))

    def set_params(self, dt, theta, nu, rho=1.0, gamma=0.1, use_supg=False, first_order_ustar=False):
        p = NsbParams(dt, theta, nu, rho, gamma, int(use_supg), int(first_order_ustar))
        self._ck(lib().nsb_set_params(self.h, C.byref(p)))

    def set_solver_opts(self, poly_degree_F=0, poly_refresh=0, poly_kind=0, poly_target=0.0, cheb_degree_Mp=0, amg_smoother_degree=0,
                        schur_mass_coeff=0.0, reorthogonalize=0, precond_precision=0, precond_operator=0, velocity_cycle=0,
                        smoother_degree=0, smoother_lo_frac=0.0, coarse_degree=0, smoother_hi_factor=0.0):
        o = NsbSolverOpts(poly_degree_F, poly_refresh, poly_kind, poly_target, cheb_degree_Mp, amg_smoother_degree, schur_mass_coeff, reorthogonalize, precond_precision,
                          precond_operator, velocity_cycle, smoother_degree, smoother_lo_frac, coarse_degree, smoother_hi_factor)
        self._ck(lib().nsb_set_solver_opts(self.h, C.byref(o)))

    def get_solver_opts(self):
        o = NsbSolverOpts()
        self._ck(lib().nsb_get_solver_opts(self.h, C.byref(o)))
        return {k: getattr(o, k) for k, _ in NsbSolverOpts._fields_}

    def set_vector(self, which, v):
        v = np.ascontiguousarray(v, np.float64)
        assert v.shape[0] == self.n_dofs
        self._ck(lib().nsb_set_vector(self.h, which, _p(v, C.c_double)))

    def get_vector(self, which, out=None):
        out = np.zeros(self.n_dofs) if out is None else out
        self._ck(lib().nsb_get_vector(self.h, which, _p(out, C.c_double)))
        return out

    def copy_vector(self, dst, src):
        self._ck(lib().nsb_copy_vector(self.h, dst, src))

    def axpy_vector(self, dst, alpha, src):
        self._ck(lib().nsb_axpy_vector(self.h, dst, C.c_double(alpha), src))

    def quadrature_points(self):
        """Mapped quadrature points of the local cells, (n_cells_local, n_q, dim): where set_forcing's values belong."""
        _, _, nc = self.sizes()
        nq = C.c_int()
        self._ck(lib().nsb_get_quadrature_points(self.h, C.byref(nq), None))
        pts = np.empty((nc, nq.value, self.dim))
        self._ck(lib().nsb_get_quadrature_points(self.h, C.byref(nq), _p(pts, C.c_double)))
        return pts

    def set_forcing(self, f_new, f_old=None):
        """Forcing at t (f_new) and at t - dt (f_old, default: the same values) at quadrature_points(); None = zero."""
        if f_old is None:
            f_old = f_new
        for which, f in ((NSB_FORCING_NEW, f_new), (NSB_FORCING_OLD, f_old)):
            if f is None:
                self._ck(lib().nsb_set_forcing(self.h, which, None))
                continue
            a = np.ascontiguousarray(f, np.float64)
            _, _, nc = self.sizes()
            if a.size != nc * (7 if self.dim == 2 else 10) * self.dim:
                raise ValueError("forcing must have shape (n_cells_local, n_q, dim), got %s" % (a.shape,))
            self._ck(lib().nsb_set_forcing(self.h, which, _p(a, C.c_double)))

    def clear_forcing(self):
        self.set_forcing(None, None)

    def set_forcing_source(self, src, params=()):
        """Forcing as CUDA source evaluated on the device (nsb_set_forcing_source): `src` defines
        __device__ void nsb_forcing(const double* x, double t, const double* prm, double* f); params (at most 16) arrive as
        prm.  Compiles unless the same source is already loaded.  None unloads it and clears both slots."""
        prm = np.ascontiguousarray(params, np.float64).ravel()
        self._ck(lib().nsb_set_forcing_source(self.h, None if src is None else src.encode(),
                                              _p(prm, C.c_double) if prm.size else None, int(prm.size)))

    def eval_forcing(self, which, t):
        """Fill slot `which` (NSB_FORCING_NEW / NSB_FORCING_OLD) with the source's f at time t on the device."""
        self._ck(lib().nsb_eval_forcing(self.h, which, C.c_double(t)))

    def forcing(self, which):
        """Slot `which` as (n_cells_local, n_q, dim); all zeros when the slot is clear."""
        _, _, nc = self.sizes()
        f = np.empty((nc, 7 if self.dim == 2 else 10, self.dim))
        self._ck(lib().nsb_get_forcing(self.h, which, _p(f, C.c_double)), soft=(1,))
        return f

    def forcing_info(self):
        hs, nv_maj, nv_min = C.c_int(), C.c_int(), C.c_int()
        comp, ev = C.c_int64(), C.c_int64()
        self._ck(lib().nsb_forcing_info(self.h, C.byref(hs), C.byref(comp), C.byref(ev), C.byref(nv_maj), C.byref(nv_min)))
        return dict(has_source=bool(hs.value), compiles=comp.value, evaluations=ev.value, nvrtc=(nv_maj.value, nv_min.value))

    # ---- hot path
    def assemble_linearized(self):
        self._ck(lib().nsb_assemble_linearized(self.h))

    def assemble_newton(self):
        self._ck(lib().nsb_assemble_newton(self.h))

    def assemble_pressure_matrices(self):
        self._ck(lib().nsb_assemble_pressure_matrices(self.h))

    def rhs_norm(self):
        v = C.c_double()
        self._ck(lib().nsb_rhs_norm(self.h, C.byref(v)))
        return v.value

    def solve(self, max_it=200, tol_rel=1e-2, n_tmp_vectors=150):
        it, res = C.c_int(), C.c_double()
        rc = self._ck(lib().nsb_solve(self.h, max_it, C.c_double(tol_rel), n_tmp_vectors, C.byref(it), C.byref(res)), soft=(1,))
        return rc == 0, it.value, res.value

    # ---- inspection
    def matrix_values(self):
        _, nnz, _ = self.sizes()
        v = np.empty(nnz)
        self._ck(lib().nsb_get_matrix_values(self.h, _p(v, C.c_double)))
        return v

    def pressure_matrix(self, which):
        n, nnz = C.c_int64(), C.c_int64()
        self._ck(lib().nsb_get_pressure_matrix(self.h, which, C.byref(n), C.byref(nnz), None, None, None))
        rp = np.empty(n.value + 1, np.int32)
        col = np.empty(nnz.value, np.int32)
        val = np.empty(nnz.value)
        self._ck(lib().nsb_get_pressure_matrix(self.h, which, C.byref(n), C.byref(nnz), _p(rp, C.c_int32), _p(col, C.c_int32), _p(val, C.c_double)))
        return rp, col, val

    def spmv(self, x):
        x = np.ascontiguousarray(x, np.float64)
        y = np.zeros(self.n_dofs)
        self._ck(lib().nsb_spmv(self.h, _p(x, C.c_double), _p(y, C.c_double)))
        return y

    def apply_velocity_block(self, x):
        """y_u = Dinv F x_u with the operator the velocity polynomial uses (diagnostic)."""
        x = np.ascontiguousarray(x, np.float64)
        y = np.zeros(self.n_dofs)
        self._ck(lib().nsb_apply_velocity_block(self.h, _p(x, C.c_double), _p(y, C.c_double)))
        return y

    # ---- measurement
    def timer_start(self):
        self._ck(lib().nsb_timer_start(self.h))

    def timer_stop(self):
        ms = C.c_double()
        self._ck(lib().nsb_timer_stop(self.h, C.byref(ms)))
        return ms.value

    def synchronize(self):
        self._ck(lib().nsb_synchronize(self.h))

    def profile_enable(self, on=True):
        self._ck(lib().nsb_profile_enable(self.h, int(on)))

    def profile_reset(self):
        self._ck(lib().nsb_profile_reset(self.h))

    def profile(self):
        out = {}
        for name in PROFILE_CLASSES:
            ms, n = C.c_double(), C.c_int64()
            self._ck(lib().nsb_profile_get(self.h, name.encode(), C.byref(ms), C.byref(n)))
            out[name] = (ms.value, n.value)
        return out

    def solver_info(self):
        d, r, l = C.c_int(), C.c_double(), C.c_int()
        self._ck(lib().nsb_solver_info(self.h, C.byref(d), C.byref(r), C.byref(l)))
        return dict(poly_degree=d.value, poly_probe_residual=r.value, amg_levels=l.value)

    def velocity_operator_info(self):
        p = C.c_int()
        v = [C.c_int64() for _ in range(4)]
        self._ck(lib().nsb_velocity_operator_info(self.h, C.byref(p), *[C.byref(x) for x in v]))
        return dict(precision=p.value, value_bytes=v[0].value, index_bytes=v[1].value, tiles=v[2].value, blocks=v[3].value)

    def coarse_operator(self):
        """(row_gid, rowptr, col_gid, vals[nblocks, dim, dim]) of the Galerkin coarse operator (owned vertices)."""
        n, nb = C.c_int64(), C.c_int64()
        self._ck(lib().nsb_get_coarse_operator(self.h, C.byref(n), C.byref(nb), None, None, None, None))
        rg, rp, cg = np.empty(n.value, np.int64), np.empty(n.value + 1, np.int64), np.empty(nb.value, np.int64)
        v = np.empty((nb.value, self.dim, self.dim))
        self._ck(lib().nsb_get_coarse_operator(self.h, C.byref(n), C.byref(nb), _p(rg, C.c_int64), _p(rp, C.c_int64), _p(cg, C.c_int64), _p(v, C.c_double)))
        return rg, rp, cg, v

    def comm_info(self):
        a, b = C.c_int(), C.c_int()
        d = C.c_int64()
        self._ck(lib().nsb_comm_info(self.h, C.byref(a), C.byref(b), C.byref(d)))
        return dict(nranks=a.value, halo=("none", "nccl send/recv", "peer stores over NVLink (CUDA IPC)", "peer stores fused into the streamed operator")[b.value],
                    halo_doubles_per_exchange=d.value)

    def velocity_pc_info(self):
        a, b, d = C.c_int(), C.c_int(), C.c_int()
        r, v = C.c_int64(), C.c_int64()
        lm = C.c_double()
        self._ck(lib().nsb_velocity_pc_info(self.h, C.byref(a), C.byref(b), C.byref(d), C.byref(r), C.byref(v), C.byref(lm)))
        return dict(two_level=bool(a.value), smoother_degree=b.value, coarse_degree=d.value, coarse_rows=r.value,
                    coarse_value_bytes=v.value, fine_lambda_max=lm.value)

    def velocity_operator(self, level):
        """The packed B = Dinv F of `level` (0 fine, 1 coarse) as stored: dict(precision, tiles, row_gid, rowptr, col_gid,
        vals[nblocks, dim, dim]) in the level's global node numbering."""
        prec, nt, n, nb = C.c_int(), C.c_int64(), C.c_int64(), C.c_int64()
        self._ck(lib().nsb_get_velocity_operator(self.h, level, C.byref(prec), C.byref(nt), C.byref(n), C.byref(nb),
                                                 None, None, None, None))
        rg, rp, cg = np.empty(n.value, np.int64), np.empty(n.value + 1, np.int64), np.empty(nb.value, np.int64)
        v = np.empty((nb.value, self.dim, self.dim))
        self._ck(lib().nsb_get_velocity_operator(self.h, level, C.byref(prec), C.byref(nt), C.byref(n), C.byref(nb),
                                                 _p(rg, C.c_int64), _p(rp, C.c_int64), _p(cg, C.c_int64), _p(v, C.c_double)))
        return dict(precision=prec.value, tiles=nt.value, row_gid=rg, rowptr=rp, col_gid=cg, vals=v)

    def apply_velocity_operator(self, level, mode, x, u=None, poly=None, coef=(0.0, 0.0, 0.0, 0.0)):
        """One application of the level's streamed operator with epilogue `mode` (2, 3, 4; coef = cu, ct, cpu, cpy) on
        vectors in the level's global numbering.  Returns y, or (y, poly updated) for mode 3."""
        x = np.ascontiguousarray(x, np.float64)
        y = np.zeros_like(x)
        cf = np.ascontiguousarray(coef, np.float64)
        ua = None if u is None else np.ascontiguousarray(u, np.float64)
        pa = None if poly is None else np.array(poly, np.float64)
        self._ck(lib().nsb_apply_velocity_operator(self.h, level, mode, _p(cf, C.c_double), _p(x, C.c_double),
                                                   None if ua is None else _p(ua, C.c_double), _p(y, C.c_double),
                                                   None if pa is None else _p(pa, C.c_double)))
        return (y, pa) if mode == 3 else y

    def velocity_pc_roots(self, level):
        """Roots of the level's polynomial (application order, one complex entry per conjugate pair)."""
        n = C.c_int()
        self._ck(lib().nsb_get_velocity_pc_roots(self.h, level, C.byref(n), None, None))
        re, im = np.empty(n.value), np.empty(n.value)
        self._ck(lib().nsb_get_velocity_pc_roots(self.h, level, C.byref(n), _p(re, C.c_double), _p(im, C.c_double)))
        return re + 1j * im

    def apply_velocity_pc(self, x):
        x = np.ascontiguousarray(x, np.float64)
        y = np.zeros(self.n_dofs)
        self._ck(lib().nsb_apply_velocity_pc(self.h, _p(x, C.c_double), _p(y, C.c_double)))
        return y

    def apply_preconditioner(self, x):
        x = np.ascontiguousarray(x, np.float64)
        y = np.zeros(self.n_dofs)
        self._ck(lib().nsb_apply_preconditioner(self.h, _p(x, C.c_double), _p(y, C.c_double)))
        return y

    def pressure_pc_info(self):
        lm, cm = C.c_double(), C.c_double()
        self._ck(lib().nsb_pressure_pc_info(self.h, C.byref(lm), C.byref(cm)))
        return dict(mp_lambda_max=lm.value, mass_coeff=cm.value)

    def launch_count(self):
        n = C.c_int64()
        self._ck(lib().nsb_launch_count(self.h, C.byref(n)))
        return n.value


# ------------------------------------------------------------------------------------------------
# libnsbhost.so: the C++ mirror of the reference's NavierStokes<dim> class (include/nsb200_host.h)
# ------------------------------------------------------------------------------------------------
HOST_LIB_PATH = os.path.join(_HERE, "libnsbhost.so")
_hostlib = None


class NshOptions(C.Structure):
    _fields_ = [("device", C.c_int32), ("rank", C.c_int32), ("nranks", C.c_int32), ("nccl_unique_id", C.c_void_p),
                ("write_vtu", C.c_int32), ("verbose", C.c_int32), ("gmres_tolerance", C.c_double), ("deltat", C.c_double),
                ("max_steps", C.c_int32), ("output_dir", C.c_char_p), ("solver", NsbSolverOpts), ("partitioner", C.c_int32), ("test_fail_solves", C.c_int32)]


class NshStepInfo(C.Structure):
    _fields_ = [("time", C.c_double), ("cd", C.c_double), ("cl", C.c_double), ("dp", C.c_double), ("wall_seconds", C.c_double),
                ("gmres_iterations", C.c_int32), ("newton_iterations", C.c_int32), ("solves", C.c_int32), ("converged", C.c_int32),
                ("forcing_seconds", C.c_double)]


def hostlib():
    global _hostlib
    if _hostlib is None:
        lib()
        if not os.path.exists(HOST_LIB_PATH):
            raise NsbError("libnsbhost.so is not built")
        _hostlib = C.CDLL(HOST_LIB_PATH)
        _hostlib.nsh_last_error.restype = C.c_char_p
        _hostlib.nsh_device.restype = C.c_void_p
    return _hostlib


# int fn(int64_t n, const double* pts, double t, double* out, void* user)   (nsh_forcing_fn)
_FORCING_FN = C.CFUNCTYPE(C.c_int, C.c_int64, C.POINTER(C.c_double), C.c_double, C.POINTER(C.c_double), C.c_void_p)


class _BorrowedDevice(Device):
    """View of the nsb_handle owned by a HostSolver (never destroyed from Python)."""

    def __init__(self, handle, dim, n_dofs):
        self.h = C.c_void_p(handle)
        self.dim = dim
        self.n_dofs = n_dofs

    def close(self):
        self.h = None


class HostSolver:
    """NavierStokes<dim>(TestCases::make_<case>(mesh_file)) driven through the C facade."""

    def __init__(self, case, mesh_file, device=0, rank=0, nranks=1, nccl_unique_id=None, write_vtu=False, verbose=False,
                 gmres_tolerance=0.0, deltat=0.0, output_dir=None, solver_opts=None, test_fail_solves=0, partitioner=0):
        L = hostlib()
        self._uid = C.create_string_buffer(nccl_unique_id, 128) if nccl_unique_id else None
        self._outdir = output_dir.encode() if output_dir else None
        o = NshOptions(device, rank, nranks, C.cast(self._uid, C.c_void_p) if self._uid else None, int(write_vtu),
                       int(verbose), gmres_tolerance, deltat, -1, self._outdir, solver_opts or NsbSolverOpts(), partitioner, test_fail_solves)
        self.h = C.c_void_p()
        if L.nsh_create(case.encode(), mesh_file.encode(), C.byref(o), C.byref(self.h)) != 0:
            raise NsbError(L.nsh_last_error().decode())
        self.dim = 2 if case.startswith("2D") else 3
        self._forcing_cb = None
        self._forcing_error = None

    def _ck(self, rc):
        if rc != 0:
            raise NsbError(hostlib().nsh_last_error().decode())

    def initialize(self):
        self._ck(hostlib().nsh_initialize(self.h))
        v = [C.c_int64() for _ in range(4)]
        self._ck(hostlib().nsh_get_sizes(self.h, *[C.byref(x) for x in v]))
        self.n_u, self.n_p, self.n_cells, self.n_vertices = [x.value for x in v]

    def step(self):
        info = NshStepInfo()
        self._forcing_error = None
        if hostlib().nsh_step(self.h, C.byref(info)) != 0:
            msg = hostlib().nsh_last_error().decode()
            raise NsbError(msg) from self._forcing_error
        return {k: getattr(info, k) for k, _ in NshStepInfo._fields_}

    def set_forcing(self, fn):
        """Forcing term f: fn(points (n, dim), t) -> (n, dim), called at most twice per assembly (t and t - dt) on the
        quadrature points of the solver's local cells.  None restores the default zero forcing."""
        if fn is None:
            self._forcing_cb = None
            self._ck(hostlib().nsh_set_forcing(self.h, None, None))
            return
        dim = self.dim

        def cb(n, pts, t, out, user):
            try:
                x = np.ctypeslib.as_array(pts, shape=(n, dim)).copy() if n else np.empty((0, dim))
                f = np.asarray(fn(x, t), dtype=np.float64).reshape(n, dim)
                if n:
                    np.ctypeslib.as_array(out, shape=(n, dim))[:] = f
                return 0
            except Exception as e:       # reported by step() as the cause of the failed step
                self._forcing_error = e
                return 1

        self._forcing_cb = _FORCING_FN(cb)        # must outlive every step that may call it
        self._ck(hostlib().nsh_set_forcing(self.h, self._forcing_cb, None))

    def set_forcing_source(self, src, params=()):
        """Forcing term as CUDA source evaluated on the GPU (DeviceForcing; see Device.set_forcing_source for the contract).
        A compile error fails the first step that needs the forcing.  None restores the default zero forcing."""
        prm = np.ascontiguousarray(params, np.float64).ravel()
        self._forcing_cb = None
        self._ck(hostlib().nsh_set_forcing_source(self.h, None if src is None else src.encode(),
                                                  _p(prm, C.c_double) if prm.size else None, int(prm.size)))

    def set_test_fail_solves(self, k):
        self._ck(hostlib().nsh_set_test_fail_solves(self.h, int(k)))

    def solution(self):
        out = np.empty(self.n_u + self.n_p)
        self._ck(hostlib().nsh_get_solution(self.h, _p(out, C.c_double)))
        return out

    def device(self):
        return _BorrowedDevice(hostlib().nsh_device(self.h), self.dim, self.n_u + self.n_p)

    def close(self):
        if self.h:
            hostlib().nsh_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class HostSetup:
    """Host-only setup object (nshd_*): mesh reading, DoF enumeration, sparsity, constraints -- the
    integer part of the reference's setup(), no GPU involved."""

    def __init__(self, mesh_file, dim):
        L = hostlib()
        self.h = C.c_void_p()
        if L.nshd_create(mesh_file.encode(), dim, C.byref(self.h)) != 0:
            raise NsbError(L.nsh_last_error().decode())
        self.dim = dim
        v = [C.c_int64() for _ in range(5)]
        L.nshd_get_sizes(self.h, *[C.byref(x) for x in v])
        self.n_u, self.n_p, self.n_cells, self.n_vertices, self.n_boundary_faces = [x.value for x in v]
        self.n_dofs = self.n_u + self.n_p
        self.dofs_per_cell = dim * (6 if dim == 2 else 10) + dim + 1

    def cell_dofs(self):
        a = np.empty((self.n_cells, self.dofs_per_cell), np.uint32)
        hostlib().nshd_get_cell_dofs(self.h, _p(a, C.c_uint32))
        return a

    def support_points(self):
        p = np.empty((self.n_dofs, self.dim))
        c = np.empty(self.n_dofs, np.uint8)
        hostlib().nshd_get_support_points(self.h, _p(p, C.c_double), _p(c, C.c_ubyte))
        return p, c

    def pattern(self):
        nnz = C.c_int64()
        if hostlib().nshd_get_pattern(self.h, C.byref(nnz), None, None) != 0:
            raise NsbError(hostlib().nsh_last_error().decode())
        rp = np.empty(self.n_dofs + 1, np.int64)
        col = np.empty(nnz.value, np.uint32)
        hostlib().nshd_get_pattern(self.h, C.byref(nnz), _p(rp, C.c_int64), _p(col, C.c_uint32))
        return rp, col

    def constraints(self, case, t, homogeneous=False):
        n = C.c_int64()
        if hostlib().nshd_get_constraints(self.h, case.encode(), C.c_double(t), int(homogeneous), C.byref(n), None, None) != 0:
            raise NsbError(hostlib().nsh_last_error().decode())
        d = np.empty(n.value, np.uint32)
        v = np.empty(n.value)
        hostlib().nshd_get_constraints(self.h, case.encode(), C.c_double(t), int(homogeneous), C.byref(n), _p(d, C.c_uint32), _p(v, C.c_double))
        return d, v

    def partition(self, nranks, method=0):
        """Owning rank of every cell: method 0 contiguous chunks, 1 METIS on the face-dual graph."""
        part = np.empty(self.n_cells, np.int32)
        if hostlib().nshd_partition(self.h, int(nranks), int(method), _p(part, C.c_int32)) != 0:
            raise NsbError(hostlib().nsh_last_error().decode())
        return part

    def mesh(self):
        p = np.empty((self.n_vertices, self.dim))
        c = np.empty((self.n_cells, self.dim + 1), np.uint32)
        hostlib().nshd_get_mesh(self.h, _p(p, C.c_double), _p(c, C.c_uint32))
        return p, c

    def close(self):
        if self.h:
            hostlib().nshd_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
