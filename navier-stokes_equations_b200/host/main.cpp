// Driver with the same role as the reference's src/main.cpp:3-46, except that the test case and
// mesh are chosen on the command line instead of by editing the source:
//   navier_stokes <test case> <mesh file> [--steps N] [--no-vtu] [--tol X] [--device D]
//                 [--forcing FILE.cu [--forcing-params a,b,...]]
// --forcing: the forcing term as CUDA source evaluated on the GPU (DeviceForcing, include/nsb200.h nsb_set_forcing_source),
// with up to 16 parameters.
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <sstream>

#include "navier_stokes.hpp"
#include "test_cases.hpp"

using namespace nsb_host;

namespace {
std::string forcing_src;
std::vector<double> forcing_params;

template <int dim> void run(BenchmarkTestCase<dim> tc, const RunOptions& opt) {
  if (!forcing_src.empty()) tc.forcing_term = std::make_shared<DeviceForcing<dim>>(forcing_src, forcing_params);
  NavierStokes<dim> s(tc, opt);
  s.run();
}

std::string read_file(const char* path) {
  std::ifstream in(path);
  if (!in) throw std::runtime_error(std::string("cannot read forcing source ") + path);
  std::stringstream ss;
  ss << in.rdbuf();
  return ss.str();
}

std::vector<double> parse_list(const char* s) {
  std::vector<double> v;
  std::stringstream ss(s);
  std::string item;
  while (std::getline(ss, item, ',')) {
    char* end = nullptr;
    v.push_back(std::strtod(item.c_str(), &end));
    if (item.empty() || *end) throw std::runtime_error("--forcing-params: not a number: '" + item + "'");
  }
  return v;
}
}  // namespace

int main(int argc, char* argv[]) {
  try {
    if (argc < 3) {
      std::cerr << "usage: " << argv[0] << " <2D-1|2D-2|2D-3|3D-1Z|3D-2Z|3D-3Z> <mesh.msh|mesh.bin> [--steps N] [--no-vtu] [--tol X] [--device D]"
                << " [--forcing FILE.cu [--forcing-params a,b,...]]" << std::endl;
      return 2;
    }
    const std::string tc_name = argv[1], mesh = argv[2];
    RunOptions opt;
    for (int i = 3; i < argc; ++i) {
      if (!std::strcmp(argv[i], "--steps") && i + 1 < argc) opt.max_steps = std::atoi(argv[++i]);
      else if (!std::strcmp(argv[i], "--no-vtu")) opt.write_vtu = false;
      else if (!std::strcmp(argv[i], "--tol") && i + 1 < argc) opt.gmres_tolerance = std::atof(argv[++i]);
      else if (!std::strcmp(argv[i], "--device") && i + 1 < argc) opt.device = std::atoi(argv[++i]);
      else if (!std::strcmp(argv[i], "--forcing") && i + 1 < argc) forcing_src = read_file(argv[++i]);
      else if (!std::strcmp(argv[i], "--forcing-params") && i + 1 < argc) forcing_params = parse_list(argv[++i]);
    }
    if (!forcing_params.empty() && forcing_src.empty()) throw std::runtime_error("--forcing-params needs --forcing FILE.cu");
    if (tc_name == "2D-1") run(TestCases::make_2D_1(mesh), opt);
    else if (tc_name == "2D-2") run(TestCases::make_2D_2(mesh), opt);
    else if (tc_name == "2D-3") run(TestCases::make_2D_3(mesh), opt);
    else if (tc_name == "3D-1Z") run(TestCases::make_3D_1Z(mesh), opt);
    else if (tc_name == "3D-2Z") run(TestCases::make_3D_2Z(mesh), opt);
    else if (tc_name == "3D-3Z") run(TestCases::make_3D_3Z(mesh), opt);
    else { std::cerr << "unknown test case " << tc_name << std::endl; return 2; }
  } catch (std::exception& exc) {
    std::cerr << std::endl << "----------------------------------------------------" << std::endl;
    std::cerr << "Exception: " << exc.what() << std::endl << "Aborting!" << std::endl;
    return 1;
  } catch (...) {
    std::cerr << std::endl << "----------------------------------------------------" << std::endl;
    std::cerr << "Unknown exception! Aborting!" << std::endl;
    return 1;
  }
  return 0;
}
