/* nsb200_host -- C facade over the C++ host mirror of the reference's NavierStokes<dim> class
 * (navier-stokes_equations_b200/host/navier_stokes.hpp; reference src/classes/NavierStokes.hpp:225-603).
 * It exists so that non-C++ programs (bench.py, the pytest suites) can drive the same class a C++
 * user would instantiate; it adds no numerics.  The nshd_* group is host-only (no GPU needed):
 * mesh reading, DoF enumeration, sparsity, constraints -- the integer setup of
 * reference src/classes/NavierStokes.cpp:7-104, 229-273.
 */
#ifndef NSB200_HOST_H
#define NSB200_HOST_H

#include <stdint.h>

#include "nsb200.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct nsh_solver* nsh_handle;
typedef struct nshd_setup* nshd_handle;

typedef struct nsh_options {
  int32_t device;            /* CUDA device ordinal of this process                              */
  int32_t rank, nranks;      /* one process per GPU                                              */
  const void* nccl_unique_id;/* 128 bytes from nsb_comm_unique_id, broadcast by the caller       */
  int32_t write_vtu;         /* 1 = output() writes solution_NNNN.vtu/.pvtu every step (cpp:1322) */
  int32_t verbose;           /* 1 = the reference's pcout lines on rank 0                        */
  double gmres_tolerance;    /* <=0: 1e-2 (reference cpp:545, 836)                               */
  double deltat;             /* <=0: the test case's own rule (TestCases.hpp / hpp:368-375)      */
  int32_t max_steps;         /* run(): stop after this many steps; <0 = until T                  */
  const char* output_dir;    /* NULL = "./"                                                      */
  nsb_solver_opts solver;    /* zero = defaults                                                  */
  int32_t partitioner;       /* cells -> ranks: 0 contiguous chunks (default), 1 METIS on the face-dual graph (cpp:56) */
  int32_t test_fail_solves;  /* test hook: report the next k linear solves as not converged (drives the retry /
                                fallback paths of run(), cpp:1174-1198, 1223-1286); 0 in production           */
  int32_t restart_every;     /* run(): write a restart file after every step whose number is a multiple of this, and after
                                its last step; 0 = never                                                       */
  const char* restart_file;  /* where run() writes it; NULL = output_dir + "restart.nsb"                       */
} nsh_options;

typedef struct nsh_step_info {
  double time, cd, cl, dp, wall_seconds;
  int32_t gmres_iterations, newton_iterations, solves, converged;
  double forcing_seconds;    /* time of the step spent evaluating the forcing term and getting it to the device (host
                                evaluation + upload, or device evaluation + synchronise for a forcing source) */
} nsh_step_info;

const char* nsh_last_error(void);

/* test_case in {"2D-1","2D-2","2D-3","3D-1Z","3D-2Z","3D-3Z"} = TestCases::make_* (TestCases.hpp:101-306);
 * mesh_file: Gmsh MSH 2.2 ASCII (.msh) or the binary dump of tools/msh.py (.bin) */
int nsh_create(const char* test_case, const char* mesh_file, const nsh_options* opt, nsh_handle* out);
void nsh_destroy(nsh_handle h);
int nsh_initialize(nsh_handle h);                        /* setup() + initial condition (cpp:1045-1071) */
/* Restart files (NavierStokes::save_restart / resume, DESIGN.md section 12).  nsh_save_restart: call on every rank after a
 * step; rank 0 writes the file atomically (path.tmp, fsync, rename).  nsh_resume: in place of nsh_initialize; fails, naming
 * the field, when the file does not belong to this mesh / test case / dt, or is truncated or corrupt.  Set the forcing again
 * before stepping: it is not stored. */
int nsh_resume(nsh_handle h, const char* path);
int nsh_save_restart(nsh_handle h, const char* path);
int nsh_step(nsh_handle h, nsh_step_info* info);         /* one time step of run() (cpp:1074-1322)      */
int nsh_run(nsh_handle h);                               /* run()                                        */
int nsh_get_sizes(nsh_handle h, int64_t* n_u, int64_t* n_p, int64_t* n_cells, int64_t* n_vertices);
int nsh_get_solution(nsh_handle h, double* current_solution /* [n_u+n_p] */);
nsb_handle nsh_device(nsh_handle h);
/* test hook, see nsh_options.test_fail_solves */
int nsh_set_test_fail_solves(nsh_handle h, int32_t k);

/* forcing term of the momentum equation (NavierStokes::set_forcing_term, reference hpp:150-171) as a batched callback:
 * fn writes f(x_i, t) for the n points pts[n][dim] into out[n][dim] (velocity components) and returns 0; any other return
 * value fails the step that asked for it.  The solver calls fn at most twice per assembly (t and t - dt), on the
 * quadrature points of its local cells.  fn = NULL restores the default zero forcing. */
typedef int (*nsh_forcing_fn)(int64_t n, const double* pts, double t, double* out, void* user);
int nsh_set_forcing(nsh_handle h, nsh_forcing_fn fn, void* user);
/* forcing term as CUDA source evaluated on the device (DeviceForcing; source contract and parameters as for
 * nsb_set_forcing_source, at most 16).  The solver compiles it on the first step that needs it (a compile error fails that
 * step with NVRTC's log) and evaluates each time level once per assembly time.  src = NULL restores the default zero
 * forcing. */
int nsh_set_forcing_source(nsh_handle h, const char* src, const double* prm, int32_t n_prm);

/* ---- host-only setup objects -------------------------------------------------------------- */
int nshd_create(const char* mesh_file, int dim, nshd_handle* out);
void nshd_destroy(nshd_handle h);
int nshd_get_sizes(nshd_handle h, int64_t* n_u, int64_t* n_p, int64_t* n_cells, int64_t* n_vertices, int64_t* n_boundary_faces);
int nshd_get_mesh(nshd_handle h, double* points, uint32_t* cells);
int nshd_get_cell_dofs(nshd_handle h, uint32_t* cell_dofs);
int nshd_get_support_points(nshd_handle h, double* pts, unsigned char* component);
/* owning rank of every cell for `nranks` ranks: method 0 contiguous chunks, 1 METIS (GridTools::partition_triangulation, cpp:56) */
int nshd_partition(nshd_handle h, int nranks, int method, int32_t* cell_part);
/* make_sparsity_pattern(dh, bdsp, empty_constraints, true): call with NULLs to get nnz first */
int nshd_get_pattern(nshd_handle h, int64_t* nnz, int64_t* rowptr, uint32_t* col);
/* Dirichlet lines in the reference's order inlet -> walls -> cylinder (velocity), outlet (pressure).
 * homogeneous = 1: newton_constraints (cpp:229-253); else system_constraints of test_case at time t
 * (cpp:617-639).  Call with NULL arrays to get n. */
int nshd_get_constraints(nshd_handle h, const char* test_case, double t, int homogeneous, int64_t* n, uint32_t* dofs, double* vals);

#ifdef __cplusplus
}
#endif
#endif
