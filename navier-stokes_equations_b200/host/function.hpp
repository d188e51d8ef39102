// Minimal stand-ins for the deal.II value types the reference's public interface exposes
// (dealii::Point<dim>, dealii::Function<dim>, dealii::Vector<double>): same member names and
// meaning, so user-supplied inlet / forcing / initial-condition classes written against
// reference src/classes/NavierStokes.hpp:65-195 port by changing the include.
#pragma once
#include <array>
#include <cstddef>
#include <vector>

namespace nsb_host {

template <int dim> class Point {
public:
  Point() { c.fill(0.0); }
  Point(double x, double y) { c.fill(0.0); c[0] = x; c[1] = y; }
  Point(double x, double y, double z) { c.fill(0.0); c[0] = x; c[1] = y; if (dim > 2) c[2] = z; }
  double operator[](unsigned int i) const { return c[i]; }
  double& operator[](unsigned int i) { return c[i]; }
private:
  std::array<double, 3> c;
};

template <typename T> class Vector {
public:
  explicit Vector(std::size_t n = 0) : v(n, T(0)) {}
  T& operator[](std::size_t i) { return v[i]; }
  const T& operator[](std::size_t i) const { return v[i]; }
  T& operator()(std::size_t i) { return v[i]; }
  const T& operator()(std::size_t i) const { return v[i]; }
  std::size_t size() const { return v.size(); }
private:
  std::vector<T> v;
};

template <int dim> class Function {
public:
  explicit Function(unsigned int n_components = 1, double initial_time = 0.0)
    : n_components(n_components), time(initial_time) {}
  virtual ~Function() = default;
  virtual double value(const Point<dim>& /*p*/, const unsigned int /*component*/ = 0) const { return 0.0; }
  virtual void vector_value(const Point<dim>& p, Vector<double>& values) const {
    for (unsigned int c = 0; c < n_components; ++c) values[c] = value(p, c);
  }
  // deal.II's batched evaluation: values[i] = vector_value(points[i]); values must hold points.size() vectors of
  // n_components entries.  The forcing term is evaluated through this (once per assembly time level), so a class
  // that can evaluate many points at once overrides it.
  virtual void vector_value_list(const std::vector<Point<dim>>& points, std::vector<Vector<double>>& values) const {
    for (std::size_t i = 0; i < points.size(); ++i) vector_value(points[i], values[i]);
  }
  virtual void set_time(const double t) { time = t; }
  double get_time() const { return time; }
  const unsigned int n_components;
private:
  double time;
};

namespace Functions {
template <int dim> class ZeroFunction : public Function<dim> {
public:
  explicit ZeroFunction(unsigned int n = 1) : Function<dim>(n) {}
};
}  // namespace Functions

}  // namespace nsb_host
