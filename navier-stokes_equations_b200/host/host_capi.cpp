// C facade (include/nsb200_host.h) over NavierStokes<dim>; no numerics here.
#include "../../include/nsb200_host.h"

#include <cstring>
#include <memory>
#include <string>

#include "navier_stokes.hpp"
#include "test_cases.hpp"

using namespace nsb_host;

namespace {
thread_local std::string g_err;

struct CaseSpec { int dim; };
int case_dim(const std::string& n) {
  if (n == "2D-1" || n == "2D-2" || n == "2D-3") return 2;
  if (n == "3D-1Z" || n == "3D-2Z" || n == "3D-3Z") return 3;
  return 0;
}
BenchmarkTestCase<2> make2(const std::string& n, const std::string& mesh, double dt) {
  if (n == "2D-1") return TestCases::make_2D_1(mesh, TimeScheme::BackwardEuler, NonlinearMethod::Newton, dt);
  if (n == "2D-2") return TestCases::make_2D_2(mesh, TimeScheme::CrankNicolson, NonlinearMethod::Linearized, dt);
  return TestCases::make_2D_3(mesh, TimeScheme::CrankNicolson, NonlinearMethod::Linearized, dt);
}
BenchmarkTestCase<3> make3(const std::string& n, const std::string& mesh, double dt) {
  if (n == "3D-1Z") return TestCases::make_3D_1Z(mesh, TimeScheme::BackwardEuler, NonlinearMethod::Newton, dt);
  if (n == "3D-2Z") return TestCases::make_3D_2Z(mesh, TimeScheme::CrankNicolson, NonlinearMethod::Linearized, dt);
  return TestCases::make_3D_3Z(mesh, TimeScheme::CrankNicolson, NonlinearMethod::Linearized, dt);
}
// Function<dim> over the C callback of nsh_set_forcing: vector_value_list makes one call for all points.
template <int dim> class CallbackForcing : public Function<dim> {
public:
  CallbackForcing(nsh_forcing_fn fn_, void* user_) : Function<dim>(dim + 1), fn(fn_), user(user_) {}
  double value(const Point<dim>& p, const unsigned int component) const override {
    Vector<double> v(dim + 1);
    vector_value(p, v);
    return v[component];
  }
  void vector_value(const Point<dim>& p, Vector<double>& values) const override {
    double x[3] = {0, 0, 0}, o[3] = {0, 0, 0};
    for (int d = 0; d < dim; ++d) x[d] = p[d];
    call(1, x, o);
    for (int c = 0; c < dim; ++c) values[c] = o[c];
    if (values.size() > (size_t)dim) values[dim] = 0.0;
  }
  void vector_value_list(const std::vector<Point<dim>>& points, std::vector<Vector<double>>& values) const override {
    const size_t n = points.size();
    std::vector<double> x(n * dim), o(n * dim, 0.0);
    for (size_t i = 0; i < n; ++i)
      for (int d = 0; d < dim; ++d) x[i * dim + d] = points[i][d];
    call((int64_t)n, x.data(), o.data());
    for (size_t i = 0; i < n; ++i) {
      for (int c = 0; c < dim; ++c) values[i][c] = o[i * dim + c];
      if (values[i].size() > (size_t)dim) values[i][dim] = 0.0;
    }
  }
private:
  void call(int64_t n, const double* x, double* o) const {
    const int rc = fn(n, x, this->get_time(), o, user);
    if (rc != 0)
      throw std::runtime_error("forcing callback returned " + std::to_string(rc) + " at t = " + std::to_string(this->get_time()));
  }
  nsh_forcing_fn fn;
  void* user;
};
}  // namespace

struct nsh_solver {
  int dim = 0;
  std::unique_ptr<NavierStokes<2>> s2;
  std::unique_ptr<NavierStokes<3>> s3;
};

struct nshd_setup {
  Mesh mesh;
  DofHandler dh;
  std::vector<BoundaryFace> bf;
};

#define NSH_TRY try {
#define NSH_CATCH                                              \
  }                                                            \
  catch (const std::exception& e) { g_err = e.what(); return -1; } \
  catch (...) { g_err = "unknown exception"; return -1; }

extern "C" {

const char* nsh_last_error(void) { return g_err.c_str(); }

int nsh_create(const char* test_case, const char* mesh_file, const nsh_options* o, nsh_handle* out) {
  NSH_TRY
  if (!test_case || !mesh_file || !out) { g_err = "null argument"; return -1; }
  const int dim = case_dim(test_case);
  if (!dim) { g_err = std::string("unknown test case ") + test_case; return -1; }
  RunOptions ro;
  double dt = -1.0;
  if (o) {
    ro.device = o->device; ro.rank = o->rank; ro.nranks = o->nranks > 0 ? o->nranks : 1;
    ro.nccl_unique_id = o->nccl_unique_id;
    ro.write_vtu = o->write_vtu != 0; ro.verbose = o->verbose != 0;
    if (o->gmres_tolerance > 0) ro.gmres_tolerance = o->gmres_tolerance;
    ro.max_steps = o->max_steps;
    if (o->output_dir) ro.output_dir = o->output_dir;
    ro.solver = o->solver;
    ro.partitioner = o->partitioner;
    ro.test_fail_solves = o->test_fail_solves;
    ro.restart_every = o->restart_every;
    if (o->restart_file) ro.restart_file = o->restart_file;
    dt = o->deltat;
  }
  auto h = std::make_unique<nsh_solver>();
  h->dim = dim;
  if (dim == 2) h->s2 = std::make_unique<NavierStokes<2>>(make2(test_case, mesh_file, dt), ro);
  else h->s3 = std::make_unique<NavierStokes<3>>(make3(test_case, mesh_file, dt), ro);
  *out = h.release();
  return 0;
  NSH_CATCH
}

void nsh_destroy(nsh_handle h) { delete h; }

int nsh_initialize(nsh_handle h) {
  NSH_TRY
  if (h->dim == 2) h->s2->initialize(); else h->s3->initialize();
  return 0;
  NSH_CATCH
}

int nsh_resume(nsh_handle h, const char* path) {
  if (!h || !path) { g_err = "null argument"; return -1; }
  NSH_TRY
  if (h->dim == 2) h->s2->resume(path); else h->s3->resume(path);
  return 0;
  NSH_CATCH
}

int nsh_save_restart(nsh_handle h, const char* path) {
  if (!h || !path) { g_err = "null argument"; return -1; }
  NSH_TRY
  if (h->dim == 2) h->s2->save_restart(path); else h->s3->save_restart(path);
  return 0;
  NSH_CATCH
}

int nsh_step(nsh_handle h, nsh_step_info* info) {
  NSH_TRY
  StepInfo s = h->dim == 2 ? h->s2->advance() : h->s3->advance();
  if (info) {
    info->time = s.time; info->cd = s.cd; info->cl = s.cl; info->dp = s.dp; info->wall_seconds = s.wall_seconds;
    info->gmres_iterations = s.gmres_iterations; info->newton_iterations = s.newton_iterations;
    info->solves = s.solves; info->converged = s.converged ? 1 : 0; info->forcing_seconds = s.forcing_seconds;
  }
  return 0;
  NSH_CATCH
}

int nsh_run(nsh_handle h) {
  NSH_TRY
  if (h->dim == 2) h->s2->run(); else h->s3->run();
  return 0;
  NSH_CATCH
}

int nsh_get_sizes(nsh_handle h, int64_t* n_u, int64_t* n_p, int64_t* n_cells, int64_t* n_vertices) {
  NSH_TRY
  const DofHandler& d = h->dim == 2 ? h->s2->dofs() : h->s3->dofs();
  const Mesh& m = h->dim == 2 ? h->s2->grid() : h->s3->grid();
  if (n_u) *n_u = d.n_u;
  if (n_p) *n_p = d.n_p;
  if (n_cells) *n_cells = m.n_cells();
  if (n_vertices) *n_vertices = m.n_vertices();
  return 0;
  NSH_CATCH
}

int nsh_get_solution(nsh_handle h, double* out) {
  NSH_TRY
  const std::vector<double>& s = h->dim == 2 ? h->s2->current() : h->s3->current();
  std::memcpy(out, s.data(), s.size() * sizeof(double));
  return 0;
  NSH_CATCH
}

int nsh_set_test_fail_solves(nsh_handle h, int32_t k) {
  if (!h) return -1;
  if (h->dim == 2) h->s2->options.test_fail_solves = k; else h->s3->options.test_fail_solves = k;
  return 0;
}

int nsh_set_forcing(nsh_handle h, nsh_forcing_fn fn, void* user) {
  if (!h) { g_err = "null handle"; return -1; }
  NSH_TRY
  if (h->dim == 2) h->s2->set_forcing_term(fn ? std::make_shared<CallbackForcing<2>>(fn, user) : nullptr);
  else h->s3->set_forcing_term(fn ? std::make_shared<CallbackForcing<3>>(fn, user) : nullptr);
  return 0;
  NSH_CATCH
}

int nsh_set_forcing_source(nsh_handle h, const char* src, const double* prm, int32_t n_prm) {
  if (!h) { g_err = "null handle"; return -1; }
  NSH_TRY
  if (n_prm < 0 || (n_prm > 0 && !prm)) { g_err = "nsh_set_forcing_source: bad parameter array"; return -1; }
  const std::vector<double> p(prm, prm + n_prm);
  if (h->dim == 2) h->s2->set_forcing_term(src ? std::make_shared<DeviceForcing<2>>(src, p) : nullptr);
  else h->s3->set_forcing_term(src ? std::make_shared<DeviceForcing<3>>(src, p) : nullptr);
  return 0;
  NSH_CATCH
}

nsb_handle nsh_device(nsh_handle h) { return h->dim == 2 ? h->s2->device() : h->s3->device(); }

// ---- host-only
int nshd_create(const char* mesh_file, int dim, nshd_handle* out) {
  NSH_TRY
  auto h = std::make_unique<nshd_setup>();
  h->mesh = read_mesh(mesh_file, dim);
  h->dh.distribute(h->mesh);
  h->bf = boundary_faces(h->mesh);
  const int wall = dim == 2 ? 103 : 104, cyl = dim == 2 ? 104 : 103;
  assign_boundary_ids_geometrically(h->mesh, h->bf, 101, 102, wall, cyl);
  *out = h.release();
  return 0;
  NSH_CATCH
}

void nshd_destroy(nshd_handle h) { delete h; }

int nshd_get_sizes(nshd_handle h, int64_t* n_u, int64_t* n_p, int64_t* n_cells, int64_t* n_vertices, int64_t* nbf) {
  if (n_u) *n_u = h->dh.n_u;
  if (n_p) *n_p = h->dh.n_p;
  if (n_cells) *n_cells = h->mesh.n_cells();
  if (n_vertices) *n_vertices = h->mesh.n_vertices();
  if (nbf) *nbf = (int64_t)h->bf.size();
  return 0;
}

int nshd_get_mesh(nshd_handle h, double* points, uint32_t* cells) {
  if (points) std::memcpy(points, h->mesh.points.data(), h->mesh.points.size() * sizeof(double));
  if (cells) std::memcpy(cells, h->mesh.cells.data(), h->mesh.cells.size() * sizeof(uint32_t));
  return 0;
}

int nshd_get_cell_dofs(nshd_handle h, uint32_t* cd) {
  std::memcpy(cd, h->dh.cell_dofs.data(), h->dh.cell_dofs.size() * sizeof(uint32_t));
  return 0;
}

int nshd_get_support_points(nshd_handle h, double* pts, unsigned char* comp) {
  if (pts) std::memcpy(pts, h->dh.support_points.data(), h->dh.support_points.size() * sizeof(double));
  if (comp) std::memcpy(comp, h->dh.component.data(), h->dh.component.size());
  return 0;
}

int nshd_partition(nshd_handle h, int nranks, int method, int32_t* cell_part) {
  NSH_TRY
  const std::vector<int32_t> p = partition_cells(h->mesh, nranks, method);
  std::copy(p.begin(), p.end(), cell_part);
  return 0;
  NSH_CATCH
}

int nshd_get_pattern(nshd_handle h, int64_t* nnz, int64_t* rowptr, uint32_t* col) {
  NSH_TRY
  std::vector<int64_t> rp;
  std::vector<uint32_t> cl;
  make_sparsity_pattern(h->dh, rp, cl);
  if (nnz) *nnz = (int64_t)cl.size();
  if (rowptr) std::copy(rp.begin(), rp.end(), rowptr);
  if (col) std::copy(cl.begin(), cl.end(), col);
  return 0;
  NSH_CATCH
}

int nshd_get_constraints(nshd_handle h, const char* test_case, double t, int homogeneous, int64_t* n, uint32_t* dofs, double* vals) {
  NSH_TRY
  const int dim = h->mesh.dim;
  if (case_dim(test_case) != dim) { g_err = "test case / mesh dimension mismatch"; return -1; }
  const int wall = dim == 2 ? 103 : 104, cyl = dim == 2 ? 104 : 103;
  Constraints c;
  auto zero = [](const double*, int) { return 0.0; };
  std::function<double(const double*, int)> inlet = zero;
  std::shared_ptr<Function<2>> f2;
  std::shared_ptr<Function<3>> f3;
  if (!homogeneous) {
    if (dim == 2) {
      f2 = make2(test_case, "", -1.0).inlet_velocity;
      f2->set_time(t);
      inlet = [f2](const double* x, int comp) { return f2->value(Point<2>(x[0], x[1]), (unsigned)comp); };
    } else {
      f3 = make3(test_case, "", -1.0).inlet_velocity;
      f3->set_time(t);
      inlet = [f3](const double* x, int comp) { return f3->value(Point<3>(x[0], x[1], x[2]), (unsigned)comp); };
    }
  }
  interpolate_boundary_values(h->mesh, h->dh, h->bf, 101, inlet, true, false, c);
  interpolate_boundary_values(h->mesh, h->dh, h->bf, wall, zero, true, false, c);
  interpolate_boundary_values(h->mesh, h->dh, h->bf, cyl, zero, true, false, c);
  interpolate_boundary_values(h->mesh, h->dh, h->bf, 102, zero, false, true, c);
  std::vector<uint32_t> d;
  std::vector<double> v;
  c.to_arrays(d, v);
  if (n) *n = (int64_t)d.size();
  if (dofs) std::copy(d.begin(), d.end(), dofs);
  if (vals) std::copy(v.begin(), v.end(), vals);
  return 0;
  NSH_CATCH
}

}  // extern "C"
