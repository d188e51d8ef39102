"""CUDA twins of the forcing terms in tests/forcing_cases.py, for nsb_set_forcing_source (test_forcing_source_cpu.py,
test_gpu_forcing_source.py, tools/gpu_multi.py --forcing-source)."""

# smooth_forcing(x, t)
SMOOTH = r"""
__device__ void nsb_forcing(const double* x, double t, const double* prm, double* f) {
  const double s = 0.5 * (1.0 + 0.5 * sin(3.0 * t));
  f[0] = s * sin(2.0 * x[0] + x[1]);
  f[1] = s * cos(x[0] - 3.0 * x[1]) + 0.1 * t;
#if NSB_DIM == 3
  f[2] = s * sin(4.0 * x[2] + x[0]);
#endif
}
"""

# Manufactured.forcing(x) with its coefficients in prm (manufactured_params)
MANUFACTURED = r"""
// prm = a, b, c, k, beta, nu, L (outlet plane x_ax = L), ax (flow axis); y = the first transverse coordinate
__device__ void nsb_forcing(const double* x, double t, const double* prm, double* f) {
  const double a = prm[0], b = prm[1], c = prm[2], k = prm[3], beta = prm[4], nu = prm[5], L = prm[6];
  const int ax = (int)prm[7], tr = ax == 0 ? 1 : 0;
  const double X = x[ax] - L, y = x[tr];
  const double ux = a + b * y + c * y * y, uy = k * X * X;
  f[ax] = uy * (b + 2.0 * c * y) - 2.0 * nu * c + beta;
  f[tr] = 2.0 * k * X * ux - 2.0 * nu * k;
}
"""

# f = x: the slots then hold the quadrature points themselves
IDENTITY = r"""
__device__ void nsb_forcing(const double* x, double t, const double* prm, double* f) {
  for (int k = 0; k < NSB_DIM; ++k) f[k] = x[k];
}
"""

# identically zero (f arrives zeroed; the negative zero still counts as zero)
ZERO = r"""
__device__ void nsb_forcing(const double* x, double t, const double* prm, double* f) {
  f[0] = -0.0 * x[0];
}
"""

# prm[0] * x_0 in the first component: changes with the parameters alone
SCALED = r"""
__device__ void nsb_forcing(const double* x, double t, const double* prm, double* f) {
  f[0] = prm[0] * x[0] + prm[1] * t;
}
"""


def manufactured_params(ms):
    return [ms.a, ms.b, ms.c, ms.k, ms.beta, ms.nu, ms.L, float(ms.ax)]
