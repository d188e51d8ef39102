/* nsb200 -- C ABI of the B200-native hot path of gdonninelli/Navier-Stokes_equations.
 *
 * Drop-in boundary (SURVEY.md section 8b): the reference has no FFI layer; its seam is the
 * protected methods of NavierStokes<dim> (reference src/classes/NavierStokes.hpp:530-553)
 * plus setup() (reference src/classes/NavierStokes.cpp:3-276).  Each entry point below names
 * the reference code it replaces.  Plain C: opaque handle, caller-owned host buffers,
 * int return codes (0 = ok, >0 = soft condition documented per call, <0 = error with
 * nsb_last_error()); no exceptions cross the boundary; no torch / C++ types.
 *
 * Numbering contract: all DoF indices are the reference's global numbering after
 * DoFRenumbering::component_wise (velocity block [0,n_u), pressure block [n_u,n_u+n_p)),
 * cell_dofs in FESystem local order (per vertex u_0..u_{d-1},p ; per line u_0..u_{d-1}).
 */
#ifndef NSB200_H
#define NSB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct nsb_ctx* nsb_handle;

/* time-stepping / stabilisation parameters read by the assembly
 * (reference NavierStokes.hpp:485-511; cpp:463,665,793) */
typedef struct nsb_params {
  double dt;                /* deltat                                               */
  double theta;             /* 1 = backward Euler, 0.5 = Crank-Nicolson              */
  double nu;                /* kinematic viscosity                                   */
  double rho;               /* density                                               */
  double gamma;             /* grad-div weight (0.1 in the reference), used iff use_supg */
  int32_t use_supg;         /* SUPG + grad-div stabilisation (3-D cases)             */
  int32_t first_order_ustar;/* first_step || second_step || BackwardEuler (cpp:665)  */
} nsb_params;

/* options of the GPU preconditioner that stands in for Ifpack ILU / ML AMG
 * (reference NavierStokes.hpp:302-315).  Zero-initialise for defaults. */
typedef struct nsb_solver_opts {
  int32_t poly_degree_F;    /* max degree of the polynomial on Dinv*F        (default 64)  */
  int32_t poly_refresh;     /* rebuild that polynomial every k-th solve      (default 1)   */
  int32_t poly_kind;        /* 0/1 = Chebyshev roots on the interval spanned by the harmonic Ritz values when the
                               spectrum is real, else the harmonic Ritz roots themselves (default);
                               <0 = always the harmonic Ritz (GMRES) polynomial                       */
  double poly_target;       /* stop growing the degree once the polynomial reduces the probe
                               vector's residual below this                  (default 0.08) */
  int32_t cheb_degree_Mp;   /* Jacobi Chebyshev degree on M_p               (default 3)   */
  int32_t amg_smoother_degree; /* Chebyshev sweeps per level, pre and post  (default 2)   */
  double schur_mass_coeff;  /* coefficient of M_p^-1; <0 = theta*nu + gamma_graddiv (default),
                               set to theta*nu for the reference's exact scaling (hpp:343) */
  int32_t reorthogonalize;  /* 0 or 1 = classical Gram-Schmidt with a second pass when the first cancelled more than half of
                               the vector (DGKS, default); 2 = always twice; <0 = always once */
  int32_t precond_precision;/* storage of the operator used INSIDE the velocity polynomial: a packed, tile-planar copy of
                               Dinv F in fp16 (16, default) or fp32 (32), streamed through shared memory with TMA bulk copies
                               (products and sums in fp64, so the preconditioner stays a fixed linear operator), or 64 = the
                               assembled fp64 values themselves.  Changing it invalidates the assembled system
                               (re-assemble before solving). */
  int32_t precond_operator; /* reserved (round 1's element-wise operator was removed); ignored */
  int32_t velocity_cycle;   /* 2 (default, also 0) = two-level cycle on the velocity block of LINEARISED systems whose scaled
                               spectrum is real: P1 coarse space (Galerkin operator, Chebyshev solve) + Chebyshev smoother;
                               1 = the single-level polynomial only.  Newton systems and complex spectra always use 1. */
  int32_t smoother_degree;  /* operator applications of the fine-level smoother per cycle      (default 14)   */
  double smoother_lo_frac;  /* smoother interval [frac * lambda_max, lambda_max]               (default 0.012)*/
  int32_t coarse_degree;    /* Chebyshev degree of the coarse solve                            (default 15)   */
  double smoother_hi_factor;/* lambda_max = this factor x the largest Ritz value of 12 Arnoldi steps (default 1.1) */
} nsb_solver_opts;

/* ---- lifetime -------------------------------------------------------------------- */
int nsb_create(int dim, int device, nsb_handle* out);
int nsb_destroy(nsb_handle h);
const char* nsb_last_error(nsb_handle h);

/* Multi-GPU: one process per GPU.  `nccl_unique_id` is the 128-byte ncclUniqueId produced by
 * rank 0 (nsb_comm_unique_id) and broadcast by the host program (MPI in the reference,
 * torch.distributed in bench.py).  Replaces the MPI communicator of reference
 * NavierStokes.hpp:401-407.  Must be called before nsb_upload_mesh. */
int nsb_comm_unique_id(void* out128);
int nsb_comm_init(nsb_handle h, int rank, int nranks, const void* nccl_unique_id);

/* ---- setup: replaces the DoF / sparsity / matrix part of setup()
 *      (reference NavierStokes.cpp:83-104, 197-225, 256-273) ------------------------- */
/* coords[V][dim], cell_vertices[C][dim+1], cell_dofs[C][dofs_per_cell] (15 / 34),
 * cell_part[C] = owning rank of each cell or NULL on one GPU
 * (GridTools::partition_triangulation, cpp:56). */
int nsb_upload_mesh(nsb_handle h, int64_t n_vertices, const double* coords, int64_t n_cells,
                    const uint32_t* cell_vertices, const uint32_t* cell_dofs, int64_t n_u, int64_t n_p,
                    const int32_t* cell_part);
/* local sizes: owned rows, stored non-zeros of the owned rows, local cells (owned + ghost layer) */
int nsb_get_sizes(nsb_handle h, int64_t* n_rows_owned, int64_t* nnz_owned, int64_t* n_cells_local);
/* stored non-zeros of the owned rows per block: velocity-velocity (F), velocity-pressure (B^T),
 * pressure-velocity (B), pressure-pressure */
int nsb_get_block_nnz(nsb_handle h, int64_t* uu, int64_t* up, int64_t* pu, int64_t* pp);
/* sparsity pattern of the owned rows as scalar CSR with GLOBAL column indices, rows in local
 * order (see nsb_get_row_gids); on one GPU this is exactly make_sparsity_pattern's result
 * (cpp:265).  rowptr[n_rows_owned+1], col[nnz_owned]. */
int nsb_get_pattern(nsb_handle h, int64_t* rowptr, uint32_t* col);
int nsb_get_row_gids(nsb_handle h, int64_t* gid);

/* ---- per-step inputs -------------------------------------------------------------- */
/* Dirichlet lines x[dof] = val: newton_constraints (cpp:229-253) or the per-step
 * system_constraints (cpp:617-639).  Replaces the previous set. */
int nsb_set_constraints(nsb_handle h, int64_t n, const uint32_t* dof, const double* val);
int nsb_set_params(nsb_handle h, const nsb_params* p);
int nsb_set_solver_opts(nsb_handle h, const nsb_solver_opts* o);
/* the options in effect (defaults resolved) */
int nsb_get_solver_opts(nsb_handle h, nsb_solver_opts* out);

enum {
  NSB_SOLUTION_OLD = 0,      /* solution_old        u^n                (hpp:578)           */
  NSB_SOLUTION_OLD_OLD = 1,  /* solution_old_old    u^{n-1}            (hpp:587)           */
  NSB_CURRENT_SOLUTION = 2,  /* current_solution    Newton iterate     (hpp:581)           */
  NSB_SOLUTION = 3,          /* solution_owned / newton_update: result of the last solve   */
  NSB_RHS = 4                /* system_rhs                                                 */
};
/* v has the GLOBAL length n_u+n_p; every rank passes the full vector (ghost import,
 * cpp:1053-1056,1299-1300). */
int nsb_set_vector(nsb_handle h, int which, const double* v_global);
/* full vector in global numbering.  With more than one rank this is a COLLECTIVE call: every rank
 * receives the whole vector (what the reference gets from its ghosted vectors + MPI). */
int nsb_get_vector(nsb_handle h, int which, double* v_global);
/* device-resident time-level bookkeeping of run() (cpp:1299-1300, 1183-1185):
 * dst = src ;  dst += alpha * src.  Ghost entries are refreshed. */
int nsb_copy_vector(nsb_handle h, int dst, int src);
int nsb_axpy_vector(nsb_handle h, int dst, double alpha, int src);

/* forcing term f of the momentum equation (reference NavierStokes.hpp:150-171), sampled by the caller at the
 * quadrature points of the LOCAL cells (owned + ghost layer, nsb_get_sizes' n_cells_local).  The assembly uses
 * f_theta = theta f(t) + (1 - theta) f(t - dt) in the rhs and in the SUPG source / strong residual
 * (linearised system cpp:688-720, 733; Newton cpp:367-370, 488-506). */
enum {
  NSB_FORCING_NEW = 0,       /* f at t          */
  NSB_FORCING_OLD = 1        /* f at t - dt     */
};
/* mapped quadrature points of the local cells, in the order nsb_set_forcing expects: pts[n_cells_local][n_q][dim],
 * x_q = sum_v lambda_{q,v} X_v of QGaussSimplex<dim>(3) (n_q = 7 in 2-D, 10 in 3-D).  pts = NULL: n_q only. */
int nsb_get_quadrature_points(nsb_handle h, int* n_q, double* pts);
/* f[n_cells_local][n_q][dim], the forcing's velocity components at those points, into slot `which`; NULL or all zero
 * clears the slot.  Both slots clear (the default) = no forcing: the kernels then read nothing and the assembled system
 * is bit-identical to one that never had forcing.  Replaces the previous values of the slot; a new mesh clears both. */
int nsb_set_forcing(nsb_handle h, int which, const double* f);

/* Forcing evaluated on the device from CUDA source compiled at run time (NVRTC, loaded on first use; without it only these
 * entries fail).  The source defines a function named nsb_forcing with this signature (the library checks it exactly):
 *     __device__ void <nsb_forcing>(const double* x, double t, const double* prm, double* f);
 * x[NSB_DIM] is a quadrature point, prm[] the parameters passed here, f[NSB_DIM] the velocity components (zeroed before the
 * call).  The library puts `#define NSB_DIM 2|3` before the text and its evaluation kernel after it.  No #include; NVRTC's
 * built-in math (sin, cos, exp, pow, sqrt, ...) is available, M_PI is not defined; helper __device__ functions and constants
 * may be defined.  Compiled with --gpu-architecture=sm_XYa of the handle's device and -std=c++17.
 *
 * Compiles `src` (or reuses the kernel when the text equals the one already loaded: nothing is compiled) and stores
 * prm[n_prm], 0 <= n_prm <= 16 (prm may be NULL when n_prm = 0).  A compile error returns < 0 and nsb_last_error carries
 * NVRTC's log, whose line numbers count the lines of `src`.  On first use the local cells' vertex coordinates and cell ->
 * vertex table are copied to the device (freed by a new mesh).  The slots keep their values until the next
 * nsb_eval_forcing / nsb_set_forcing.  src = NULL unloads the kernel and clears both slots.  Errors: no mesh uploaded,
 * n_prm out of range, prm = NULL with n_prm > 0. */
int nsb_set_forcing_source(nsb_handle h, const char* src, const double* prm, int n_prm);
/* fills slot `which` on the device with f(x_q, t) at the points of nsb_get_quadrature_points (mapped on the device with
 * the same operations in the same order: bit-identical points).  An all-zero result clears the slot as nsb_set_forcing
 * does.  Synchronises (reads back 4 bytes).  A later nsb_set_forcing of the slot replaces its values, and vice versa.
 * Errors: no mesh uploaded, bad `which`, no source set. */
int nsb_eval_forcing(nsb_handle h, int which, double t);
/* inspection: slot `which` as f[n_cells_local][n_q][dim]; returns 1 (soft) and zeros when the slot is clear */
int nsb_get_forcing(nsb_handle h, int which, double* f);
/* a source is loaded; sources compiled and slots evaluated since nsb_create; version of the NVRTC that was loaded
 * (0.0 when none could be).  NULL pointers are skipped. */
int nsb_forcing_info(nsb_handle h, int* has_source, int64_t* compiles, int64_t* evaluations, int* nvrtc_major, int* nvrtc_minor);
/* compiles a forcing source for sm_100a without a handle or a GPU: 0 when it compiles, else < 0 with the error (NVRTC's log)
 * in log[log_size] (truncated, NUL-terminated; log may be NULL) */
int nsb_check_forcing_source(int dim, const char* src, char* log, size_t log_size);

/* ---- the hot path ----------------------------------------------------------------- */
/* assemble_linearized_system()  (cpp:569-831): A, b from u^n, u^{n-1}, constraints, params */
int nsb_assemble_linearized(nsb_handle h);
/* assemble_newton_system()      (cpp:278-539): Jacobian, -residual from current/old solution */
int nsb_assemble_newton(nsb_handle h);
/* one-time M_p, K_p (+1e-6 M_p) through the current constraints (cpp:798-803, 812-829) and
 * the multigrid hierarchy that replaces the per-solve ML setup (hpp:310-315) */
int nsb_assemble_pressure_matrices(nsb_handle h);
/* system_rhs.l2_norm()  (cpp:542, 834, 1154, 1190) */
int nsb_rhs_norm(nsb_handle h, double* norm);
/* solve_linear_system() / solve_newton_system() (cpp:833-868, 541-567): left-preconditioned
 * restarted GMRES from x0 = 0, stop when the preconditioned residual <= tol_rel*||b||_2 or after
 * max_it iterations, n_tmp_vectors = SolverGMRES::AdditionalData (150), then
 * constraints.distribute(x).  Returns 0 converged, 1 not converged (SolverControl::NoConvergence). */
int nsb_solve(nsb_handle h, int max_it, double tol_rel, int n_tmp_vectors, int* iterations, double* residual);

/* ---- inspection (parity tests) ---------------------------------------------------- */
int nsb_get_matrix_values(nsb_handle h, double* vals /* [nnz_owned] */);
/* (1,1) blocks of pressure_mass / pressure_stiffness as global CSR over pressure DoFs */
int nsb_get_pressure_matrix(nsb_handle h, int which /*0 Mp, 1 Kp*/, int64_t* n, int64_t* nnz,
                            int32_t* rowptr, int32_t* col, double* val);
/* y = A x on the device; x, y global-length host vectors (owned entries of y written) */
int nsb_spmv(nsb_handle h, const double* x_global, double* y_global);
/* diagnostic: y_u = Dinv F x_u, the node-block-Jacobi scaled velocity block exactly as the velocity polynomial of the
 * preconditioner applies it (operator and precision per nsb_solver_opts); only velocity entries are read / written */
int nsb_apply_velocity_block(nsb_handle h, const double* x_global, double* y_global);

/* ---- measurement ------------------------------------------------------------------ */
/* CUDA-event timing on the library's stream */
int nsb_timer_start(nsb_handle h);
int nsb_timer_stop(nsb_handle h, double* milliseconds);
int nsb_synchronize(nsb_handle h);
/* per-kernel-class CUDA-event profile: names "asm_context","asm_rows","spmv","spmv_vel",
 * "schur","amg","orth","other","asm_pack","coarse","asm_coarse","forcing" */
int nsb_profile_enable(nsb_handle h, int on);
int nsb_profile_reset(nsb_handle h);
int nsb_profile_get(nsb_handle h, const char* name, double* total_ms, int64_t* launches);
/* what the last solve used: degree of the velocity polynomial, its residual reduction on the
 * probe vector, number of multigrid levels of K_p */
int nsb_solver_info(nsb_handle h, int* poly_degree, double* poly_probe_residual, int* amg_levels);
/* the packed velocity operator as stored: precision (16 / 32; 64 = none, the fp64 values are used), bytes of its value
 * array, bytes of its index side (block metadata, tile headers, unique-neighbour lists), tiles, (node, neighbour) blocks */
int nsb_velocity_operator_info(nsb_handle h, int* precision, int64_t* value_bytes, int64_t* index_bytes, int64_t* tiles,
                               int64_t* blocks);
/* how the ghost entries travel: halo_mode 0 = single GPU, 1 = NCCL send/recv, 2 = peer stores over NVLink (CUDA IPC; separate
 * push / wait kernels), 3 = peer stores fused into the streamed velocity operator; doubles this rank sends per velocity exchange */
int nsb_comm_info(nsb_handle h, int* nranks, int* halo_mode, int64_t* halo_doubles_per_exchange);
/* inspection (parity tests): the Galerkin coarse operator P^T F P of the two-level velocity cycle as block CSR over the owned
 * vertices -- global vertex id of every row, block row pointer, global vertex id of every block column, dim*dim values per
 * block (row-major).  NULL arrays are skipped (call once for the sizes). */
int nsb_get_coarse_operator(nsb_handle h, int64_t* n_rows, int64_t* n_blocks, int64_t* row_gid, int64_t* rowptr, int64_t* col_gid,
                            double* vals);
/* the velocity preconditioner as set up by the last solve: two-level cycle or not, smoother / coarse degrees, coarse rows,
 * bytes of the packed coarse operator, estimate of lambda_max(Dinv F) */
int nsb_velocity_pc_info(nsb_handle h, int* two_level, int* smoother_degree, int* coarse_degree, int64_t* coarse_rows,
                         int64_t* coarse_value_bytes, double* fine_lambda_max);
/* inspection (parity tests) of the velocity preconditioner's operators, one GPU only (an error with more ranks).  Vectors of a
 * level are in its own global numbering: level 0 (fine) = the velocity DoFs, level 1 (coarse P1 level of the two-level cycle) =
 * dim * vertex + component with vertex = pressure DoF - n_u.
 *
 * The packed copy of B = Dinv F of `level` exactly as the streamed operator reads it, unpacked from the tile headers, the quad
 * metadata and the unique-neighbour lists into block CSR over the owned nodes: global node id of every row, block row pointer,
 * global node id of every block column, dim*dim values per block (row-major, widened to double).  Also the level's stream
 * tile count.  At precond_precision = 64 no copy is kept: precision 64 and no blocks.  NULL arrays are skipped (call once for
 * the sizes). */
int nsb_get_velocity_operator(nsb_handle h, int level, int* precision, int64_t* tiles, int64_t* n_rows, int64_t* n_blocks,
                              int64_t* row_gid, int64_t* rowptr, int64_t* col_gid, double* vals);
/* one application of the level's operator with the fused epilogue `mode` (coef = {cu, ct, cpu, cpy}):
 *   2: y = B x ;  3: y = cu*u + ct*(B x), poly += cpu*u + cpy*y ;  4: y = cu*u + ct*(B x)
 * u is read for modes 3 and 4, poly read and written for mode 3 (coef, u and poly may be NULL where unused). */
int nsb_apply_velocity_operator(nsb_handle h, int level, int mode, const double coef[4], const double* x, const double* u, double* y,
                                double* poly);
/* roots of the level's polynomial as set up by the last nsb_solve, in application (Leja) order, one entry (re, im > 0) per
 * conjugate pair; n = 0 for level 1 when the last setup chose the single-level polynomial.  NULL arrays are skipped. */
int nsb_get_velocity_pc_roots(nsb_handle h, int level, int* n, double* re, double* im);
/* the velocity preconditioner y_u ~ F^-1 x_u / the whole block preconditioner y = P^-1 x as set up by the last nsb_solve;
 * x and y are global-length vectors (nsb_apply_velocity_pc reads and writes only their velocity entries) */
int nsb_apply_velocity_pc(nsb_handle h, const double* x_global, double* y_global);
int nsb_apply_preconditioner(nsb_handle h, const double* x_global, double* y_global);
/* the Schur side of the block preconditioner: estimate of lambda_max(diag(M_p)^-1 M_p) that bounds its Jacobi-Chebyshev
 * interval [1.1 lambda / 6, 1.1 lambda], and the coefficient of that M_p^-1 term (schur_mass_coeff resolved) */
int nsb_pressure_pc_info(nsb_handle h, double* mp_lambda_max, double* mass_coeff);
/* how many kernels this library launched since nsb_create */
int nsb_launch_count(nsb_handle h, int64_t* n);

#ifdef __cplusplus
}
#endif
#endif /* NSB200_H */
