// Evaluation kernel of a device-side forcing term (nsb_set_forcing_source / nsb_eval_forcing).  Not compiled by nvcc:
// the Makefile embeds this file as text in libnsb200.so, and the library compiles it with NVRTC after the user's
//   __device__ void nsb_forcing(const double* x, double t, const double* prm, double* f);
// and after its own definitions of NSB_DIM (2 or 3) and NSB_NQ (quadrature points per cell, 7 or 10).

// the user's function must have exactly the documented signature (an implicit conversion of an argument, or a result
// that is silently dropped, would otherwise compile)
template <typename A, typename B> struct nsb_same_type { static constexpr bool value = false; };
template <typename A> struct nsb_same_type<A, A> { static constexpr bool value = true; };
static_assert(nsb_same_type<decltype(&nsb_forcing), void (*)(const double*, double, const double*, double*)>::value,
              "nsb_forcing must be declared as __device__ void nsb_forcing(const double* x, double t, const double* prm, double* f)");

// barycentric coordinates lam[q][v] of the quadrature points, passed by value from the library's FE tables
struct nsb_lambda {
  double v[NSB_NQ][NSB_DIM + 1];
};

// One thread per (local cell, quadrature point) i = cell * NSB_NQ + q:
//   x_q = sum_v lam[q][v] X_v, added in vertex order with separate multiply and add (no FMA contraction), the same
//         operations in the same order as nsb_get_quadrature_points, so the points are bit-identical to the exported ones;
//   f[i][0..NSB_DIM) = nsb_forcing(x_q, t, prm), zeroed before the call;
//   *nonzero |= 1 if any component is non-zero (an OR: the flag does not depend on the order the warps finish in).
extern "C" __global__ void __launch_bounds__(256) nsb_forcing_eval(const double* __restrict__ coords, const int* __restrict__ cell_vertices,
                                                                   nsb_lambda lam, long long n_points, double t,
                                                                   const double* __restrict__ prm, double* __restrict__ f,
                                                                   unsigned int* __restrict__ nonzero) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  bool nz = false;
  if (i < n_points) {
    const long long cell = i / NSB_NQ;
    const int q = (int)(i - cell * NSB_NQ);
    double x[NSB_DIM];
#pragma unroll
    for (int k = 0; k < NSB_DIM; ++k) x[k] = 0.0;
#pragma unroll
    for (int v = 0; v <= NSB_DIM; ++v) {
      const double* X = coords + (long long)__ldg(&cell_vertices[cell * (NSB_DIM + 1) + v]) * NSB_DIM;
#pragma unroll
      for (int k = 0; k < NSB_DIM; ++k) x[k] = __dadd_rn(x[k], __dmul_rn(lam.v[q][v], __ldg(&X[k])));
    }
    double out[NSB_DIM];
#pragma unroll
    for (int k = 0; k < NSB_DIM; ++k) out[k] = 0.0;
    nsb_forcing(x, t, prm, out);
#pragma unroll
    for (int k = 0; k < NSB_DIM; ++k) {
      f[i * NSB_DIM + k] = out[k];
      nz |= out[k] != 0.0;
    }
  }
  // blockDim is a multiple of 32, so every warp is full here
  if (__any_sync(0xffffffffu, nz) && (threadIdx.x & 31) == 0) atomicOr(nonzero, 1u);
}
