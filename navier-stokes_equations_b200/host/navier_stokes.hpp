// Host-side mirror of the reference's solver class (reference src/classes/NavierStokes.hpp:225-603):
// same public interface (constructors, set_*, setup / output / run, compute_default_deltat) and the
// same protected seam (assemble_newton_system, solve_newton_system, assemble_linearized_system,
// solve_linear_system, compute_lift_drag, compute_pressure_difference).  deal.II / Trilinos / MPI are
// replaced by the small host classes in this directory and by the CUDA path behind include/nsb200.h.
#pragma once
#include <chrono>
#include <cmath>
#include <fstream>
#include <iostream>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/nsb200.h"
#include "dof_handler.hpp"
#include "function.hpp"
#include "mesh.hpp"

namespace nsb_host {

enum class TimeScheme { BackwardEuler, CrankNicolson };
enum class NonlinearMethod { Newton, Linearized };

inline std::string to_string(TimeScheme s) { return s == TimeScheme::BackwardEuler ? "Backward Euler" : "Crank-Nicolson"; }
inline std::string to_string(NonlinearMethod m) { return m == NonlinearMethod::Newton ? "Newton" : "Linearized (semi-implicit)"; }

// constructor default of the reference (hpp:65-123): NB the 2-D profile uses 6 U_m, unlike TestCases
template <int dim> class InletVelocity : public Function<dim> {
public:
  InletVelocity(double H_ = 0.41, double U_m_ = 1.5, bool time_dep = true)
    : Function<dim>(dim + 1), H(H_), U_m(U_m_), time_dependent(time_dep) {}
  double value(const Point<dim>& p, const unsigned int component) const override {
    constexpr unsigned int flow_component = (dim == 2) ? 0 : 2;
    if (component != flow_component) return 0.0;
    double profile = (dim == 2) ? 6.0 * U_m * p[1] * (H - p[1]) / (H * H)
                                : 16.0 * U_m * p[0] * p[1] * (H - p[0]) * (H - p[1]) / (H * H * H * H);
    if (time_dependent) profile *= std::sin(M_PI * this->get_time() / 8.0);
    return profile;
  }
protected:
  const double H, U_m;
  const bool time_dependent;
};

template <int dim> class ZeroDirichletBC : public Function<dim> {
public:
  ZeroDirichletBC() : Function<dim>(dim + 1) {}
};
template <int dim> class ForcingTerm : public Function<dim> {
public:
  ForcingTerm() : Function<dim>(dim + 1) {}
};
// A forcing term given as CUDA source (include/nsb200.h, nsb_set_forcing_source), evaluated on the device at the
// quadrature points.  Immutable: to change the source or the parameters, call set_forcing_term with a new one.  There is
// no host evaluation.
template <int dim> class DeviceForcing : public Function<dim> {
public:
  explicit DeviceForcing(std::string source_, std::vector<double> params_ = {})
    : Function<dim>(dim + 1), src(std::move(source_)), prm(std::move(params_)) {
    if (prm.size() > 16) throw std::invalid_argument("DeviceForcing takes at most 16 parameters, got " + std::to_string(prm.size()));
  }
  double value(const Point<dim>& /*p*/, const unsigned int /*component*/ = 0) const override {
    throw std::logic_error("DeviceForcing is evaluated on the GPU only (nsb_eval_forcing)");
  }
  const std::string& source() const { return src; }
  const std::vector<double>& params() const { return prm; }
private:
  const std::string src;
  const std::vector<double> prm;
};
template <int dim> class InitialCondition : public Function<dim> {
public:
  InitialCondition() : Function<dim>(dim + 1) {}
};

// reference hpp:203-222
template <int dim> struct BenchmarkTestCase {
  std::string name, description, mesh_file;
  unsigned int degree_velocity = 2, degree_pressure = 1;
  double Re = 0, U_m = 0, T = 0, deltat = -1;
  TimeScheme time_scheme = TimeScheme::BackwardEuler;
  NonlinearMethod nonlinear_method = NonlinearMethod::Newton;
  std::shared_ptr<Function<dim>> inlet_velocity, dirichlet_bc, forcing_term, initial_condition;
  bool use_supg = false;
};

// Run-time switches that have no counterpart in the reference (its parameters are compile-time).
struct RunOptions {
  int device = 0;                 // CUDA device of this process
  int rank = 0, nranks = 1;       // one process per GPU (the reference: one MPI rank per partition)
  const void* nccl_unique_id = nullptr;
  bool write_vtu = true;          // output() every step like the reference (cpp:1321-1322); off for timing
  bool verbose = true;
  double gmres_tolerance = 1e-2;  // reference cpp:545, 836; parity mode uses 1e-12
  int max_steps = -1;             // stop run() after this many time steps (-1: until T)
  std::string output_dir = "./";
  nsb_solver_opts solver{};       // zero = library defaults
  int partitioner = 0;            // cells -> ranks: 0 = contiguous chunks, 1 = METIS on the face-dual graph (partition_cells, mesh.hpp)
  int test_fail_solves = 0;       // test hook: the next k linear solves are REPORTED as not converged (their result is kept,
                                  // as the reference keeps the iterate of a failed GMRES) -> drives run()'s retry / fallback paths
  int restart_every = 0;          // run(): save_restart after every step whose number is a multiple of this, and after the
                                  // last step of the invocation (0 = off)
  std::string restart_file;       // where run() saves; empty = output_dir + "restart.nsb"
  std::string resume_file;        // run() resumes from this file instead of initialize() (empty = initialize())
};

struct StepInfo {
  double time = 0, cd = 0, cl = 0, dp = 0, wall_seconds = 0;
  int gmres_iterations = 0, newton_iterations = 0, solves = 0;
  bool converged = true;
  double forcing_seconds = 0;     // time spent evaluating the forcing term and getting it to the device: host evaluation and
                                  // upload, or device evaluation and its synchronise for a DeviceForcing (part of wall_seconds)
};

template <int dim> class NavierStokes {
public:
  static double compute_default_deltat(double Re) {     // hpp:368-375
    if (Re <= 20) return 0.1;
    else if (Re <= 50) return 0.05;
    else if (Re <= 100) return 0.02;
    else if (Re <= 150) return 0.01;
    else return 0.005;
  }

  explicit NavierStokes(const BenchmarkTestCase<dim>& tc, const RunOptions& opt = RunOptions())
    : NavierStokes(tc.mesh_file, tc.degree_velocity, tc.degree_pressure, tc.deltat, tc.T, tc.Re, tc.U_m, tc.time_scheme,
                   tc.nonlinear_method, tc.inlet_velocity, tc.dirichlet_bc, tc.forcing_term, tc.initial_condition,
                   tc.use_supg, opt) {
    case_name = tc.name;
  }

  NavierStokes(const std::string& mesh_file_name_, const unsigned int& degree_velocity_,
               const unsigned int& degree_pressure_, const double deltat_, const double T_, const double Re_,
               const double U_m_ = 1.5, TimeScheme time_scheme_ = TimeScheme::BackwardEuler,
               NonlinearMethod nonlinear_method_ = NonlinearMethod::Newton,
               std::shared_ptr<Function<dim>> inlet_velocity_ = nullptr,
               std::shared_ptr<Function<dim>> dirichlet_bc_ = nullptr,
               std::shared_ptr<Function<dim>> forcing_term_ = nullptr,
               std::shared_ptr<Function<dim>> initial_condition_ = nullptr, bool use_supg_ = false,
               const RunOptions& opt = RunOptions());
  ~NavierStokes();
  NavierStokes(const NavierStokes&) = delete;

  void set_inlet_velocity(std::shared_ptr<Function<dim>> f) { inlet_velocity = f; }
  void set_dirichlet_bc(std::shared_ptr<Function<dim>> f) { dirichlet_bc = f; }
  void set_forcing_term(std::shared_ptr<Function<dim>> f) {
    forcing_term = f ? f : std::make_shared<ForcingTerm<dim>>();
    forcing_time[0] = forcing_time[1] = std::nan("");
  }
  void set_initial_condition(std::shared_ptr<Function<dim>> f) { initial_condition = f; }

  void setup();
  void output(const unsigned int time_step);
  void run();

  // ---- additions for drivers / tests (no counterpart in the reference) ----
  void initialize();                 // setup() + initial condition, as the head of run() (cpp:1045-1068)
  StepInfo advance();                // one pass of the while loop body of run() (cpp:1074-1322)
  // Restart files (DESIGN.md section 12).  save_restart: call on every rank after advance() returns; rank 0 writes
  // path + ".tmp", flushes, fsyncs and renames it to path, so an earlier file survives a crash mid-write.  resume: in place
  // of initialize(); checks the file against this solver (mesh, test case, Re, U_m, dt, scheme, method, SUPG) and throws,
  // naming the field, before it changes anything; continues forces.txt after its first time_step_no rows and the VTU
  // numbering at time_step_no + 1.  With the same options and forcing the continuation is bit-identical to the run that
  // was never interrupted (not with poly_refresh > 1).  The forcing term is code, not state: set it again before stepping.
  void save_restart(const std::string& path) const;
  void resume(const std::string& path);
  const std::vector<double>& current() const { return current_solution; }
  const DofHandler& dofs() const { return dof_handler; }
  const Mesh& grid() const { return mesh; }
  nsb_handle device() const { return dev; }
  double viscosity() const { return nu; }
  double time_now() const { return time; }
  RunOptions options;

protected:
  const unsigned int mpi_size, mpi_rank;
  std::ostream& pcout;
  bool pcout_active;
  const std::string mesh_file_name;
  std::string case_name;               // BenchmarkTestCase::name, written to restart files (empty without a test case)
  const unsigned int degree_velocity, degree_pressure;
  Mesh mesh;
  double Re;
  double nu = 0.001;
  double rho = 1.0;
  static constexpr double D = 0.1;
  static constexpr double H = 0.41;
  double U_m = 1.5;
  double deltat;
  double T;
  double time = 0.0;
  TimeScheme time_scheme;
  NonlinearMethod nonlinear_method;
  double theta;
  bool use_supg;
  static constexpr unsigned int newton_max_iterations = 50;
  static constexpr double newton_tolerance = 1e-8;
  static constexpr unsigned int inlet_boundary_id = 101;
  static constexpr unsigned int outlet_boundary_id = 102;
  unsigned int wall_boundary_id = (dim == 2) ? 103 : 104;
  unsigned int cylinder_boundary_id = (dim == 2) ? 104 : 103;
  std::shared_ptr<Function<dim>> inlet_velocity, dirichlet_bc, forcing_term, initial_condition;

  void compute_lift_drag(double& drag_coeff, double& lift_coeff) const;
  double compute_pressure_difference();
  void assemble_newton_system();
  void solve_newton_system();          // throws NoConvergence like SolverControl (cpp:541-567)
  void assemble_linearized_system();
  bool solve_linear_system();

  struct NoConvergence : public std::exception {
    int last_step; double last_value;
    NoConvergence(int s, double v) : last_step(s), last_value(v) {}
    const char* what() const noexcept override { return "Iterative method reported convergence failure"; }
  };

  DofHandler dof_handler;
  std::vector<BoundaryFace> bfaces;
  nsb_handle dev = nullptr;
  // host copies of the owned vectors the driver logic manipulates (hpp:575-587)
  std::vector<double> solution_owned, solution, solution_old, newton_update, current_solution, solution_backup,
      solution_old_old;
  bool first_step = true, second_step = true;
  bool pressure_matrices_assembled = false;
  Constraints newton_constraints, system_constraints;
  std::vector<int32_t> cell_part;       // owning rank of every cell (several ranks)
  std::ofstream forces_file;
  unsigned int time_step_no = 0;
  int last_gmres_iterations = 0, step_gmres_iterations = 0, step_solves = 0;
  double last_rhs_norm = 0.0;
  double step_forcing_seconds = 0.0;
  // forcing uploaded to the device: the time each slot (NSB_FORCING_NEW / _OLD) was evaluated at, NaN = not uploaded
  double forcing_time[2] = {std::nan(""), std::nan("")};
  bool forcing_on_device = false;
  std::vector<Point<dim>> forcing_points;      // quadrature points of the device's local cells (nsb_get_quadrature_points)
  std::vector<Vector<double>> forcing_values;  // vector_value_list output, kept between evaluations
  std::shared_ptr<Function<dim>> forcing_source_term;   // the DeviceForcing whose source the device holds, if any

  void push_params(bool first_order);
  void update_forcing();
  void build_system_constraints();
  uint64_t mesh_hash() const;          // FNV-1a of the vertices, cell vertex lists and boundary faces with their ids
  void ck(int rc, const char* what) const;
  std::function<double(const double*, int)> eval(const std::shared_ptr<Function<dim>>& f) const;
};

extern template class NavierStokes<2>;
extern template class NavierStokes<3>;

}  // namespace nsb_host
