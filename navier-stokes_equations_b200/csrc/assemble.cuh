// Assembly of the linearised (Oseen-type) and Newton Taylor-Hood systems.
//
// Replaces   NavierStokes<dim>::assemble_linearized_system()   reference src/classes/NavierStokes.cpp:569-831
//            NavierStokes<dim>::assemble_newton_system()       reference src/classes/NavierStokes.cpp:278-539
//            AffineConstraints::distribute_local_to_global     reference cpp:516-523, 810-817 (SURVEY.md A.5)
//
// Two passes, both deterministic and atomics-free (DESIGN.md "Assembly"):
//   1. k_cell_context : one warp per cell.  Evaluates u^n, u^{n-1} (or u^k, p^k), u*, tau at the
//      quadrature points, writes the cell's rhs vector and its context: for the linearised system
//      the finished scalar block S_ab (CtxL, 1 KB), for Newton the per-point data (Ctx).  FORCED adds a
//      user-supplied body force, given per (cell, quadrature point) at t and at t - dt (cpp:688-697, 367-370);
//      the unforced instantiations read nothing extra and are the same code as without that option.
//   2. k_node_rows    : one warp per OWNED P2 node.  Walks the node's cells in ascending order,
//      computes the dim (+1) local matrix rows of that node exploiting the component-block
//      structure  A[(a,c),(b,d)] = delta_cd S_ab + gamma G^{cd}_ab (+ T^{cd}_ab for Newton),
//      accumulates them in shared memory, applies the Dirichlet elimination and stores every
//      CSR value exactly once.  No zero-fill of the matrix, no read-modify-write of HBM.
#pragma once
#include "device.cuh"

namespace nsb {

template <int DIM> __host__ __device__ constexpr int node_i(int a) {
  if (a <= DIM) return a;
  if (DIM == 2) return (a == 3) ? 0 : (a == 4) ? 1 : 2;
  return (a == 4) ? 0 : (a == 5) ? 1 : (a == 6) ? 2 : (a == 7) ? 0 : (a == 8) ? 1 : 2;
}
template <int DIM> __host__ __device__ constexpr int node_j(int a) {
  if (a <= DIM) return a;
  if (DIM == 2) return (a == 3) ? 1 : (a == 4) ? 2 : 0;
  return (a == 4) ? 1 : (a == 5) ? 2 : (a == 6) ? 0 : 3;
}

constexpr int ASM_WARPS = 8;
#ifndef NSB_ASM_MIN_CTAS
#define NSB_ASM_MIN_CTAS 4
#endif

// The FE tables are read with lane-dependent indices all over both passes; from __constant__
// memory that serialises (one address per cycle).  Each CTA therefore keeps a copy in shared
// memory, filled with coalesced loads from an L2-resident global copy.
__device__ __forceinline__ void load_tables_to_smem(FeTables* dst, const FeTables* __restrict__ src) {
  static_assert(sizeof(FeTables) % sizeof(double) == 0, "FeTables must be a whole number of 8-byte words");
  const double* s = reinterpret_cast<const double*>(src);
  double* d = reinterpret_cast<double*>(dst);
  for (int i = threadIdx.x; i < (int)(sizeof(FeTables) / sizeof(double)); i += blockDim.x) d[i] = __ldg(s + i);
}

// per-quadrature-point scratch of pass 1 (shared memory, per warp)
template <int DIM> struct QS {
  static constexpr int NV = DIM + 1;
  static constexpr int S = 0;                      // s[NV]
  static constexpr int TW = NV;                    // tau*JxW
  static constexpr int M = NV + 1;                 // mvec[DIM]
  static constexpr int WZ = M + DIM;               // WZ[DIM][NV]
  static constexpr int HH = WZ + DIM * NV;         // H[DIM][DIM] = grad u^k  (Newton)
  static constexpr int PD = HH + DIM * DIM;        // JxW * div u^k            (Newton)
  static constexpr int JW = PD + 1;                // JxW
  static constexpr int N = JW + 1;
};

// ------------------------------------------------------------------------------------
// pass 1
// ------------------------------------------------------------------------------------
#ifndef NSB_CTX_MIN_CTAS
#define NSB_CTX_MIN_CTAS 2
#endif
template <int DIM, bool NEWTON, bool FORCED>
__global__ void __launch_bounds__(ASM_WARPS * 32, NSB_CTX_MIN_CTAS)
k_cell_context(DevMesh M, AsmParams P, const FeTables* __restrict__ gT, const double* __restrict__ vecA,
               const double* __restrict__ vecB, double* __restrict__ ctx_out, double* __restrict__ cell_rhs,
               const double* __restrict__ f_new, const double* __restrict__ f_old) {
  constexpr int NV = DIM + 1, NN = Fe<DIM>::NN, NQ = Fe<DIM>::NQ, DPC = Fe<DIM>::DPC;
  using C = Ctx<DIM>;
  using Q = QS<DIM>;
  using CL = CtxL<DIM>;
  constexpr int CTXN = NEWTON ? C::N_NEWTON : CL::N;
  constexpr int WS = NN * DIM * 2 + NV + 4 + NQ * Q::N;     // doubles per warp
  static_assert(3 * NN * NQ <= NQ * Q::N, "the per-q scratch is reused for c, PQ, QD of the S_ab sums");
  static_assert(NV * NV <= NN * DIM, "the gathered-velocity scratch is reused for grad lambda products");
  __shared__ double sm_all[ASM_WARPS * WS];
  __shared__ FeTables sT;
  load_tables_to_smem(&sT, gT);
  __syncthreads();
  const FeTables& T = sT;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (int cell = blockIdx.x * ASM_WARPS + wid; cell < M.nc; cell += gridDim.x * ASM_WARPS) {
  double* su = sm_all + wid * WS;          // vecA velocity [NN][DIM]
  double* sv = su + NN * DIM;              // vecB velocity [NN][DIM]
  double* sp = sv + NN * DIM;              // vecA pressure [NV]
  double* sq = sp + NV + 4;                // per-q blocks

  // ---- phase A: gather
  const double* geo = M.cell_geom + (size_t)cell * 16;
  double gl[NV][DIM];
#pragma unroll
  for (int v = 0; v < NV; ++v)
#pragma unroll
    for (int k = 0; k < DIM; ++k) gl[v][k] = __ldg(geo + v * DIM + k);
  const double absJ = __ldg(geo + 12), inv_h = __ldg(geo + 14);
  if (lane < NN * DIM) {
    const int a = lane / DIM, c = lane % DIM;
    const int xo = __ldg(M.cell_xoff + (size_t)cell * NN + a) + c;
    su[lane] = vecA[xo];
    sv[lane] = vecB[xo];
  }
  if (NEWTON && lane < NV) sp[lane] = vecA[__ldg(M.cell_poff + (size_t)cell * NV + lane)];
  __syncwarp();

  // ---- phase B: one lane per quadrature point
  if (lane < NQ) {
    const int q = lane;
    const double JxW = T.w[q] * absJ;
    double ua[DIM], ub[DIM], UA[DIM][NV], UB[DIM][NV];
#pragma unroll
    for (int c = 0; c < DIM; ++c) {
      ua[c] = 0; ub[c] = 0;
#pragma unroll
      for (int m = 0; m < NV; ++m) { UA[c][m] = 0; UB[c][m] = 0; }
    }
#pragma unroll
    for (int a = 0; a < NN; ++a) {
      const double ph = T.phi[q][a], d0 = T.dco[a][0][q], d1 = T.dco[a][1][q];
#pragma unroll
      for (int c = 0; c < DIM; ++c) {
        const double xa = su[a * DIM + c], xb = sv[a * DIM + c];
        ua[c] += ph * xa;
        ub[c] += ph * xb;
        UA[c][node_i<DIM>(a)] += d0 * xa;
        if (a >= NV) UA[c][node_j<DIM>(a)] += d1 * xa;
        if (NEWTON) {
          UB[c][node_i<DIM>(a)] += d0 * xb;
          if (a >= NV) UB[c][node_j<DIM>(a)] += d1 * xb;
        }
      }
    }
    double gA[DIM][DIM], gB[DIM][DIM];
#pragma unroll
    for (int c = 0; c < DIM; ++c)
#pragma unroll
      for (int k = 0; k < DIM; ++k) {
        double s = 0, t = 0;
#pragma unroll
        for (int m = 0; m < NV; ++m) { s += UA[c][m] * gl[m][k]; if (NEWTON) t += UB[c][m] * gl[m][k]; }
        gA[c][k] = s; gB[c][k] = t;
      }
    double ustar[DIM];
    if (NEWTON || P.first_order_ustar) {
#pragma unroll
      for (int c = 0; c < DIM; ++c) ustar[c] = ua[c];
    } else {
      // u* = 2u^n - u^{n-1}, clamped back to u^n when it grows by more than 20 % (cpp:668-676)
      double ns = 0, no = 0;
#pragma unroll
      for (int c = 0; c < DIM; ++c) { ustar[c] = 2.0 * ua[c] - ub[c]; ns += ustar[c] * ustar[c]; no += ua[c] * ua[c]; }
      ns = sqrt(ns); no = sqrt(no);
      if (no > 1e-12 && ns > 1.2 * no) {
#pragma unroll
        for (int c = 0; c < DIM; ++c) ustar[c] = ua[c];
      }
    }
    double tw = 0.0;
    if (P.use_supg) {
      double um = 0;
#pragma unroll
      for (int c = 0; c < DIM; ++c) um += ustar[c] * ustar[c];
      um = sqrt(um);
      const double t1 = 2.0 * P.inv_dt, t2 = 2.0 * um * inv_h, t3 = 4.0 * P.nu * inv_h * inv_h;
      tw = JxW / sqrt(t1 * t1 + t2 * t2 + t3 * t3);      // tau * JxW   (cpp:727-729)
    }
    double* o = sq + q * Q::N;
    double s[NV];
#pragma unroll
    for (int m = 0; m < NV; ++m) {
      double t = 0;
#pragma unroll
      for (int k = 0; k < DIM; ++k) t += ustar[k] * gl[m][k];
      s[m] = t; o[Q::S + m] = t;
    }
    o[Q::TW] = tw;
    o[Q::JW] = JxW;
    double convA[DIM], convB[DIM];
#pragma unroll
    for (int c = 0; c < DIM; ++c) {
      double t = 0, r = 0;
#pragma unroll
      for (int k = 0; k < DIM; ++k) { t += gA[c][k] * ua[k]; if (NEWTON) r += gB[c][k] * ub[k]; }
      convA[c] = t; convB[c] = r;
    }
    // forcing f_theta = theta f(t) + (1 - theta) f(t - dt) at this point ([cell][q][DIM], contiguous per cell); loaded
    // here rather than at the top of phase B because the gradient accumulators are dead by now (no spills)
    double fth[DIM];
    if (FORCED) {
      const size_t fo = ((size_t)cell * NQ + q) * DIM;
#pragma unroll
      for (int c = 0; c < DIM; ++c) fth[c] = P.theta * __ldg(f_new + fo + c) + (1.0 - P.theta) * __ldg(f_old + fo + c);
    }
    if (!NEWTON) {
      // rhs of the linearised system (cpp:702-745)
#pragma unroll
      for (int c = 0; c < DIM; ++c) {
        o[Q::M + c] = JxW * (P.inv_dt * ua[c] - (1.0 - P.theta) * convA[c]);
        if (FORCED) o[Q::M + c] += JxW * fth[c];
        const double E = tw * ustar[c];                    // tau u*_c JxW: first-index contraction, cpp:733
#pragma unroll
        for (int m = 0; m < NV; ++m) {
          double gg = 0, z = 0;
          if (FORCED) {
            // SUPG source with the same first-index contraction: tau u*_c grad phi_a . (f_theta + u^n / dt)   (cpp:733)
#pragma unroll
            for (int k = 0; k < DIM; ++k) { gg += gl[m][k] * gA[c][k]; z += gl[m][k] * (ua[k] * P.inv_dt + fth[k]); }
            o[Q::WZ + c * NV + m] = -JxW * (1.0 - P.theta) * P.nu * gg + E * z;
          } else {
#pragma unroll
            for (int k = 0; k < DIM; ++k) { gg += gl[m][k] * gA[c][k]; z += gl[m][k] * ua[k]; }
            o[Q::WZ + c * NV + m] = -JxW * (1.0 - P.theta) * P.nu * gg + E * (z * P.inv_dt);
          }
        }
      }
    } else {
      // -residual of the Newton system (cpp:377-418, 478-510)
      double pk = 0, gp[DIM], lap[DIM];
#pragma unroll
      for (int v = 0; v < NV; ++v) pk += T.lam[q][v] * sp[v];
#pragma unroll
      for (int k = 0; k < DIM; ++k) {
        double t = 0;
#pragma unroll
        for (int v = 0; v < NV; ++v) t += sp[v] * gl[v][k];
        gp[k] = t; lap[k] = 0;
      }
#pragma unroll
      for (int a = 0; a < NN; ++a) {
        double gg = 0;
#pragma unroll
        for (int k = 0; k < DIM; ++k) gg += gl[node_i<DIM>(a)][k] * gl[node_j<DIM>(a)][k];
        const double lapN = (a < NV ? 4.0 : 8.0) * gg;
#pragma unroll
        for (int c = 0; c < DIM; ++c) lap[c] += su[a * DIM + c] * lapN;
      }
      double tr = 0;
#pragma unroll
      for (int c = 0; c < DIM; ++c) {
        tr += gA[c][c];
        o[Q::M + c] = -JxW * ((ua[c] - ub[c]) * P.inv_dt + P.theta * convA[c] + (1.0 - P.theta) * convB[c]);
        double strong = (ua[c] - ub[c]) * P.inv_dt + convA[c] + gp[c] - P.nu * lap[c];
        if (FORCED) {
          o[Q::M + c] += JxW * fth[c];
          strong -= fth[c];                                // strong residual of the SUPG term (cpp:488-506)
        }
#pragma unroll
        for (int m = 0; m < NV; ++m) {
          double ga = 0, gb = 0;
#pragma unroll
          for (int k = 0; k < DIM; ++k) { ga += gl[m][k] * gA[c][k]; gb += gl[m][k] * gB[c][k]; }
          o[Q::WZ + c * NV + m] = -JxW * P.nu * (P.theta * ga + (1.0 - P.theta) * gb) + JxW * pk * gl[m][c] -
                                  tw * s[m] * strong;
        }
#pragma unroll
        for (int d = 0; d < DIM; ++d) o[Q::HH + c * DIM + d] = gA[c][d];
      }
      o[Q::PD] = JxW * tr;
    }
  }
  __syncwarp();

  // ---- phase C: one lane per velocity DoF: rhs entry and local diagonal
  double diag_abs = 0.0;
  if (lane < NN * DIM) {
    const int a = lane / DIM, c = lane % DIM;
    const int ia = T.idx[a][0], ja = T.idx[a][1];
    double r = 0, svar = 0, tnew = 0;
    for (int q = 0; q < NQ; ++q) {
      const double* o = sq + q * Q::N;
      const double ph = T.phi[q][a], d0 = T.dco[a][0][q], d1 = T.dco[a][1][q];
      r += ph * o[Q::M + c] + d0 * o[Q::WZ + c * NV + ia] + d1 * o[Q::WZ + c * NV + ja];
      const double ca = d0 * o[Q::S + ia] + d1 * o[Q::S + ja];
      const double Pa = o[Q::JW] * P.theta * ph, Qa = o[Q::TW] * ca;
      svar += Pa * ca + Qa * (ph * P.inv_dt + ca);
      if (NEWTON) tnew += (Pa + Qa) * ph * o[Q::HH + c * DIM + c];
    }
    cell_rhs[(size_t)cell * DPC + lane] = r;
    // G^{kk}_aa for all k (trace) and for k == c
    double trG = 0, Gcc = 0;
#pragma unroll
    for (int k = 0; k < DIM; ++k) {
      const double g0 = gl[ia][k], g1 = gl[ja][k];
      const double g = absJ * (T.Khat[a][a][0][0] * g0 * g0 + T.Khat[a][a][0][1] * g0 * g1 +
                               T.Khat[a][a][1][0] * g1 * g0 + T.Khat[a][a][1][1] * g1 * g1);
      trG += g;
      if (k == c) Gcc = g;
    }
    const double Saa = absJ * T.Mhat[a][a] * P.inv_dt + P.theta * P.nu * trG + svar;
    diag_abs = fabs(Saa + P.gamma * Gcc + tnew);
  }
  if (lane < NV) {
    double r = 0;
    if (NEWTON)
      for (int q = 0; q < NQ; ++q) r += T.lam[q][lane] * sq[q * Q::N + Q::PD];
    cell_rhs[(size_t)cell * DPC + NN * DIM + lane] = r;
  }
  const double avg = warp_sum_fixed(diag_abs) / (double)DPC;

  // ---- phase D: context
  double* co = ctx_out + (size_t)cell * CTXN;
  if (NEWTON) {
    if (lane < NV * DIM) co[C::GL + lane] = gl[lane / DIM][lane % DIM];
    if (lane == 0) { co[C::ABSJ] = absJ; co[C::AVG] = avg; }
    for (int k = lane; k < NQ * NV; k += 32) co[C::S + k] = sq[(k / NV) * Q::N + Q::S + (k % NV)];
    if (lane < NQ) co[C::TW + lane] = sq[lane * Q::N + Q::TW];
    for (int k = lane; k < NQ * DIM * DIM; k += 32) co[C::H + k] = sq[(k / (DIM * DIM)) * Q::N + Q::HH + (k % (DIM * DIM))];
  } else {
    // Linearised system: finish the quadrature sums of the delta_cd part here, once per cell, so that the
    // node-row pass (which visits the cell once per node) only combines finished numbers.
    //   c_a(q)  = u*(q) . grad phi_a(q)
    //   PQ_a(q) = JxW theta phi_a + tau JxW c_a       QD_a(q) = tau JxW c_a / dt
    //   S_ab    = |J| Mhat_ab / dt + theta nu tr G_ab + sum_q [PQ_a c_b + QD_a phi_b]      (cpp:744-786)
    if (lane < NV * DIM) co[CL::GL + lane] = gl[lane / DIM][lane % DIM];
    if (lane == 0) { co[CL::ABSJ] = absJ; co[CL::AVG] = avg; }
    constexpr int NAQ = NN * NQ, RAQ = (NAQ + 31) / 32;
    double cq_[RAQ], pq_[RAQ], qd_[RAQ];
#pragma unroll
    for (int r = 0; r < RAQ; ++r) {
      const int e = lane + 32 * r;
      cq_[r] = 0.0; pq_[r] = 0.0; qd_[r] = 0.0;
      if (e < NAQ) {
        const int a = e / NQ, q = e % NQ;
        const double* o = sq + q * Q::N;
        const double ca = T.dco[a][0][q] * o[Q::S + T.idx[a][0]] + T.dco[a][1][q] * o[Q::S + T.idx[a][1]];
        const double qa = o[Q::TW] * ca;
        cq_[r] = ca;
        pq_[r] = o[Q::JW] * P.theta * T.phi[q][a] + qa;
        qd_[r] = qa * P.inv_dt;
      }
    }
    // products of the barycentric gradients, g_k . g_l (for tr G_ab), in the dead velocity scratch
    if (lane < NV * NV) {
      const int k = lane / NV, l = lane % NV;
      double t = 0.0;
#pragma unroll
      for (int m = 0; m < DIM; ++m) t += __ldg(geo + k * DIM + m) * __ldg(geo + l * DIM + m);
      su[lane] = t;
    }
    __syncwarp();                                    // every lane is done reading the per-q scratch
    double* s_c = sq;
    double* s_pq = sq + NAQ;
    double* s_qd = sq + 2 * NAQ;
#pragma unroll
    for (int r = 0; r < RAQ; ++r) {
      const int e = lane + 32 * r;
      if (e < NAQ) { s_c[e] = cq_[r]; s_pq[e] = pq_[r]; s_qd[e] = qd_[r]; }
    }
    __syncwarp();
    // 2 x 2 register tiles of S: one lane per tile, four independent accumulation chains, half the operand loads
    constexpr int NT = NN / 2;
    static_assert(NN % 2 == 0 && NT * NT <= 32, "one lane per 2x2 tile of S");
    if (lane < NT * NT) {
      const int a0 = 2 * (lane / NT), b0 = 2 * (lane % NT);
      double acc[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
#pragma unroll
      for (int q = 0; q < NQ; ++q) {
        const double pa[2] = {s_pq[a0 * NQ + q], s_pq[(a0 + 1) * NQ + q]};
        const double qa[2] = {s_qd[a0 * NQ + q], s_qd[(a0 + 1) * NQ + q]};
        const double cb[2] = {s_c[b0 * NQ + q], s_c[(b0 + 1) * NQ + q]};
        const double fb[2] = {T.phi[q][b0], T.phi[q][b0 + 1]};
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
          for (int j = 0; j < 2; ++j) acc[i][j] += pa[i] * cb[j] + qa[i] * fb[j];
      }
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const int a = a0 + i, b = b0 + j;
          const int ia0 = T.idx[a][0], ia1 = T.idx[a][1], ib0 = T.idx[b][0], ib1 = T.idx[b][1];
          const double trG = T.Khat[a][b][0][0] * su[ia0 * NV + ib0] + T.Khat[a][b][0][1] * su[ia0 * NV + ib1] +
                             T.Khat[a][b][1][0] * su[ia1 * NV + ib0] + T.Khat[a][b][1][1] * su[ia1 * NV + ib1];
          co[CL::S + a * NN + b] = absJ * (T.Mhat[a][b] * P.inv_dt + P.theta * P.nu * trG) + acc[i][j];
        }
    }
    if (lane < NN) {
      double t = 0.0;
#pragma unroll
      for (int q = 0; q < NQ; ++q) t += s_qd[lane * NQ + q];
      co[CL::CA + lane] = t * P.dt;
    }
  }
  __syncwarp();
  }   // cell loop
}

// ------------------------------------------------------------------------------------
// pass 2
// ------------------------------------------------------------------------------------
struct RowOut {
  double* vals;            // CSR values of A (local rows, scalar-CSR order)
  double* rhs;             // [n_own]
  double* dinv;            // [nn_own][DIM*DIM]  inverse of the node-diagonal velocity block (preconditioner)
};

template <int DIM, bool NEWTON>
__global__ void __launch_bounds__(ASM_WARPS * 32, NEWTON ? 2 : NSB_ASM_MIN_CTAS)
k_node_rows(DevMesh M, AsmParams P, const double* __restrict__ ctx, const double* __restrict__ cell_rhs,
            const unsigned char* __restrict__ cflag, const double* __restrict__ cval, RowOut out,
            const int* __restrict__ tile_ptr, const FeTables* __restrict__ gT) {
  constexpr int NV = DIM + 1, NN = Fe<DIM>::NN, NQ = Fe<DIM>::NQ, DPC = Fe<DIM>::DPC;
  using C = Ctx<DIM>;
  using CL = CtxL<DIM>;
  constexpr int CTXN = NEWTON ? C::N_NEWTON : CL::N;
  constexpr int PUBN = NEWTON ? C::N_NEWTON : CL::HDR;     // context words every lane needs (published in shared memory)
  constexpr int NACT = NN * DIM;                     // active lanes (b,d)
  extern __shared__ double dyn[];
  __shared__ double s_ctx[ASM_WARPS][PUBN];
  __shared__ int s_next;
  __shared__ int s_off[65];
  __shared__ FeTables sT;
  load_tables_to_smem(&sT, gT);
  const FeTables& T = sT;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int n0 = tile_ptr[blockIdx.x], n1 = tile_ptr[blockIdx.x + 1];
  // shared-memory offsets of the tile's nodes (tile has at most 64 nodes)
  if (wid == 0) {
    int need[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int A = n0 + lane + 32 * r;
      need[r] = 0;
      if (A < n1) {
        const int len = DIM * (int)(M.nbr_ptr[A + 1] - M.nbr_ptr[A]) + (int)(M.pnbr_ptr[A + 1] - M.pnbr_ptr[A]);
        need[r] = (DIM + (M.node_pid[A] >= 0 ? 1 : 0)) * len;
      }
    }
    // exclusive scan over 64 entries
    int v0 = need[0], v1 = need[1];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t0 = __shfl_up_sync(NSB_FULL, v0, o), t1 = __shfl_up_sync(NSB_FULL, v1, o);
      if (lane >= o) { v0 += t0; v1 += t1; }
    }
    const int tot0 = __shfl_sync(NSB_FULL, v0, 31);
    s_off[lane] = v0 - need[0];
    s_off[32 + lane] = tot0 + v1 - need[1];
    if (lane == 0) s_next = 0;
  }
  __syncthreads();

  // lane roles
  const int b = (lane < NACT) ? lane / DIM : NN - 1;
  const int d = (lane < NACT) ? lane % DIM : 0;
  const bool act = lane < NACT;
  const int ib0 = T.idx[b][0], ib1 = T.idx[b][1];
  const int grp = (lane / DIM) * DIM;                // first lane of this lane's b-group
  double* sc = s_ctx[wid];
  // b-side reference values at this lane's quadrature points q = d, d+DIM, ... (lane-constant)
  constexpr int QPL = NEWTON ? (NQ + DIM - 1) / DIM : 1;
  double phb[QPL], db0[QPL], db1[QPL];
#pragma unroll
  for (int t = 0; t < QPL; ++t) {
    const int q = d + DIM * t;
    phb[t] = (NEWTON && q < NQ) ? T.phi[q][b] : 0.0;
    db0[t] = (NEWTON && q < NQ) ? T.dco[b][0][q] : 0.0;
    db1[t] = (NEWTON && q < NQ) ? T.dco[b][1][q] : 0.0;
  }

  for (;;) {
    int slot = 0;
    if (lane == 0) slot = atomicAdd(&s_next, 1);
    slot = __shfl_sync(NSB_FULL, slot, 0);
    const int A = n0 + slot;
    if (A >= n1) break;
    const int nb = (int)(M.nbr_ptr[A + 1] - M.nbr_ptr[A]);
    const int np = (int)(M.pnbr_ptr[A + 1] - M.pnbr_ptr[A]);
    const int len = DIM * nb + np;
    const int pid = M.node_pid[A];
    const bool isv = pid >= 0;
    const int rows = DIM + (isv ? 1 : 0);
    double* acc = dyn + s_off[slot];
    for (int k = lane; k < rows * len; k += 32) acc[k] = 0.0;
    const int xA = DIM * A;                                    // owned node: x-offset of (A,0)
    const int xP = isv ? DIM * M.nn_own + pid : 0;
    bool crow[DIM + 1];
    bool anyc = false;
#pragma unroll
    for (int c = 0; c < DIM; ++c) { crow[c] = cflag[xA + c] != 0; anyc |= crow[c]; }
    crow[DIM] = isv ? (cflag[xP] != 0) : false;
    anyc |= crow[DIM];
    double dacc[DIM + 1];
#pragma unroll
    for (int c = 0; c <= DIM; ++c) dacc[c] = 0.0;
    double racc = 0.0;                                         // lane c < rows accumulates rhs row c
    __syncwarp();

    // The node's (cell, local index) list is read with one coalesced load per 32 cells; the global
    // data of cell i+1 (context, neighbour ranks, rhs entry) is fetched into registers while cell i is
    // being processed, so no global-memory latency sits on the dependent chain of the cell loop.
    constexpr int NCW = (PUBN + 31) / 32;                  // published context words per lane
    const long long kc0 = M.n2c_ptr[A];
    const int ncell = (int)(M.n2c_ptr[A + 1] - kc0);
    uint32_t pk_lane = 0;
    double nctx[NCW];
    double nS = 0.0, nCa = 0.0;                            // linearised: this lane's S_ab, CA_a of the next cell
    int nrb = 0, nrp = 0;
    double nrh = 0.0;
    auto fetch = [&](uint32_t pk) {
      const int cell_ = (int)(pk >> 4), a_ = (int)(pk & 15u);
      const double* cg = ctx + (size_t)cell_ * CTXN;
#pragma unroll
      for (int w = 0; w < NCW; ++w) nctx[w] = (lane + 32 * w < PUBN) ? __ldg(cg + lane + 32 * w) : 0.0;
      if (!NEWTON) {
        nS = __ldg(cg + CL::S + a_ * NN + b);
        nCa = __ldg(cg + CL::CA + a_);
      }
      nrb = __ldg(M.rank_uu + ((size_t)cell_ * NN + a_) * NN + b);
      nrp = (lane < DIM * NV) ? (int)__ldg(M.rank_up + ((size_t)cell_ * NN + a_) * NV + lane / DIM) : 0;
      nrh = 0.0;
      if (lane < rows) {
        const int li = (lane < DIM) ? a_ * DIM + lane : NN * DIM + a_;
        nrh = __ldg(cell_rhs + (size_t)cell_ * DPC + li);
      }
    };
    if (ncell > 0) {
      pk_lane = (lane < ncell) ? __ldg(M.n2c + kc0 + lane) : 0u;
      fetch(__shfl_sync(NSB_FULL, pk_lane, 0));
    }
    for (int ic = 0; ic < ncell; ++ic) {
      if (ic > 0 && (ic & 31) == 0) pk_lane = (ic + lane < ncell) ? __ldg(M.n2c + kc0 + ic + lane) : 0u;
      const uint32_t pk = __shfl_sync(NSB_FULL, pk_lane, ic & 31);
      const int a = (int)(pk & 15u);
      // publish the prefetched data of this cell, then start fetching the next one
#pragma unroll
      for (int w = 0; w < NCW; ++w) if (lane + 32 * w < PUBN) sc[lane + 32 * w] = nctx[w];
      const int rb = nrb, rp = nrp;
      const double Slin = nS, Calin = nCa;
      racc += nrh;
      if (ic + 1 < ncell) {
        uint32_t pkn;
        if (((ic + 1) & 31) == 0) pkn = __ldg(M.n2c + kc0 + ic + 1);
        else pkn = __shfl_sync(NSB_FULL, pk_lane, (ic + 1) & 31);
        fetch(pkn);
      }
      __syncwarp();
      const double absJ = sc[C::ABSJ];
      const int ia0 = T.idx[a][0], ia1 = T.idx[a][1];
      // ---- S_ab (delta_cd part) and CA_a: finished per cell by pass 1 for the linearised system; for Newton the
      // quadrature sum is split over the DIM lanes of a b-group and recombined in fixed order
      double Svar = 0.0, Ca = Calin;
      if (NEWTON) {
        double part = 0.0, capart = 0.0;
#pragma unroll
        for (int t = 0; t < QPL; ++t) {
          const int q = d + DIM * t;
          if (q < NQ) {
            const double* s = sc + C::S + q * NV;
            const double tw = sc[C::TW + q];
            const double pha = T.phi[q][a];
            const double ca = T.dco[a][0][q] * s[ia0] + T.dco[a][1][q] * s[ia1];
            const double cb = db0[t] * s[ib0] + db1[t] * s[ib1];
            const double Pa = T.w[q] * absJ * P.theta * pha;
            const double Qa = tw * ca;
            part += Pa * cb + Qa * (phb[t] * P.inv_dt + cb);
            capart += Qa;
          }
        }
        Ca = 0.0;
#pragma unroll
        for (int k = 0; k < DIM; ++k) { Svar += shfl_d(part, grp + k); Ca += shfl_d(capart, grp + k); }
      }
      // ---- G^{cd}_ab for this lane's column d, all rows c
      const double gb0 = sc[C::GL + ib0 * DIM + d], gb1 = sc[C::GL + ib1 * DIM + d];
      const double t0 = T.Khat[a][b][0][0] * gb0 + T.Khat[a][b][0][1] * gb1;
      const double t1 = T.Khat[a][b][1][0] * gb0 + T.Khat[a][b][1][1] * gb1;
      double G[DIM];
#pragma unroll
      for (int c = 0; c < DIM; ++c) G[c] = absJ * (sc[C::GL + ia0 * DIM + c] * t0 + sc[C::GL + ia1 * DIM + c] * t1);
      double Sab = Slin;
      if (NEWTON) {
        double Gdd = 0.0;
#pragma unroll
        for (int c = 0; c < DIM; ++c) if (c == d) Gdd = G[c];
        double trG = 0.0;
#pragma unroll
        for (int k = 0; k < DIM; ++k) trG += shfl_d(Gdd, grp + k);
        Sab = absJ * T.Mhat[a][b] * P.inv_dt + P.theta * P.nu * trG + Svar;
      }
      double val[DIM];
#pragma unroll
      for (int c = 0; c < DIM; ++c) val[c] = P.gamma * G[c] + ((c == d) ? Sab : 0.0);
      if (NEWTON) {
        // T^{cd}_ab = sum_q (Pa + Qa) phi_b  d_d u^k_c      (cpp:428-429, 456)
        for (int q = 0; q < NQ; ++q) {
          const double* s = sc + C::S + q * NV;
          const double ca = T.dco[a][0][q] * s[ia0] + T.dco[a][1][q] * s[ia1];
          const double e = (T.w[q] * absJ * P.theta * T.phi[q][a] + sc[C::TW + q] * ca) * T.phi[q][b];
#pragma unroll
          for (int c = 0; c < DIM; ++c) val[c] += e * sc[C::H + q * DIM * DIM + c * DIM + d];
        }
      }
      // ---- constrained rows: remember |local diagonal| (or the cell's average)  (A.5)
      if (anyc) {
        const double avg = sc[C::AVG];
#pragma unroll
        for (int c = 0; c < DIM; ++c) {
          const double dg = shfl_d(val[c], a * DIM + c);
          if (crow[c]) dacc[c] += (dg != 0.0) ? fabs(dg) : avg;
        }
        if (crow[DIM]) dacc[DIM] += avg;                          // p-p local diagonal is identically 0
      }
      // ---- accumulate
      if (act) {
#pragma unroll
        for (int c = 0; c < DIM; ++c) acc[c * len + DIM * rb + d] += val[c];
        if (isv) {
          // pressure row of vertex a:  -(psi_a, div phi_(b,d))     (cpp:435, 763)
          const double pr = -absJ * (T.Bhat[b][a][0] * gb0 + T.Bhat[b][a][1] * gb1);
          acc[DIM * len + DIM * rb + d] += pr;
        }
      }
      if (lane < DIM * NV) {
        // velocity row (a,c), pressure column of vertex j: -(psi_j, div phi_i) + tau (u*.grad phi_a) d_c psi_j
        const int j = lane / DIM, c = lane % DIM;
        const double up = -absJ * (T.Bhat[a][j][0] * sc[C::GL + ia0 * DIM + c] + T.Bhat[a][j][1] * sc[C::GL + ia1 * DIM + c]) +
                          Ca * sc[C::GL + j * DIM + c];
        acc[c * len + DIM * nb + rp] += up;
      }
      __syncwarp();
    }

    // ---- finalize: Dirichlet elimination, rhs, store each value once
    const long long* nptr = M.nbr_ptr + A;
    const int* nx = M.nbr_xoff + nptr[0];
    const int* px = M.pnbr_xoff + M.pnbr_ptr[A];
    const int selfk = DIM * M.selfrank[A];
    double corr[DIM + 1];
#pragma unroll
    for (int c = 0; c <= DIM; ++c) corr[c] = 0.0;
    for (int k = lane; k < len; k += 32) {
      const int xo = (k < DIM * nb) ? (__ldg(nx + k / DIM) + k % DIM) : __ldg(px + (k - DIM * nb));
      const bool ccol = cflag[xo] != 0;
      const double g = ccol ? cval[xo] : 0.0;
#pragma unroll
      for (int c = 0; c < DIM; ++c) {
        double v = acc[c * len + k];
        if (ccol) { corr[c] += v * g; v = 0.0; }
        if (crow[c]) v = (k == selfk + c) ? dacc[c] : 0.0;
        acc[c * len + k] = v;
        out.vals[M.rowbase[A] + (long long)c * len + k] = v;
      }
      if (isv) {
        double v = acc[DIM * len + k];
        if (ccol) { corr[DIM] += v * g; v = 0.0; }
        if (crow[DIM]) v = (k == DIM * nb + M.pselfrank[pid]) ? dacc[DIM] : 0.0;
        out.vals[M.prowbase[pid] + k] = v;
      }
    }
#pragma unroll
    for (int c = 0; c <= DIM; ++c) corr[c] = warp_sum_fixed(corr[c]);
    // rhs rows: lane c holds the cell sum of row c
#pragma unroll
    for (int c = 0; c < DIM; ++c)
      if (lane == c) out.rhs[xA + c] = crow[c] ? 0.0 : (racc - corr[c]);
    if (isv && lane == DIM) out.rhs[xP] = crow[DIM] ? 0.0 : (racc - corr[DIM]);
    __syncwarp();
    // inverse of the node-diagonal block (block-Jacobi smoother of the velocity preconditioner)
    if (lane == 0) {
      double Dm[DIM][DIM];
#pragma unroll
      for (int c = 0; c < DIM; ++c)
#pragma unroll
        for (int e = 0; e < DIM; ++e) Dm[c][e] = acc[c * len + selfk + e];
      double* o = out.dinv + (size_t)A * DIM * DIM;
      if (DIM == 2) {
        const double id = 1.0 / (Dm[0][0] * Dm[1][1] - Dm[0][1] * Dm[1][0]);
        o[0] = Dm[1][1] * id; o[1] = -Dm[0][1] * id; o[2] = -Dm[1][0] * id; o[3] = Dm[0][0] * id;
      } else {
        const double c00 = Dm[1][1] * Dm[2][2] - Dm[1][2] * Dm[2][1];
        const double c01 = Dm[1][2] * Dm[2][0] - Dm[1][0] * Dm[2][2];
        const double c02 = Dm[1][0] * Dm[2][1] - Dm[1][1] * Dm[2][0];
        const double id = 1.0 / (Dm[0][0] * c00 + Dm[0][1] * c01 + Dm[0][2] * c02);
        o[0] = c00 * id;
        o[1] = (Dm[0][2] * Dm[2][1] - Dm[0][1] * Dm[2][2]) * id;
        o[2] = (Dm[0][1] * Dm[1][2] - Dm[0][2] * Dm[1][1]) * id;
        o[3] = c01 * id;
        o[4] = (Dm[0][0] * Dm[2][2] - Dm[0][2] * Dm[2][0]) * id;
        o[5] = (Dm[0][2] * Dm[1][0] - Dm[0][0] * Dm[1][2]) * id;
        o[6] = c02 * id;
        o[7] = (Dm[0][1] * Dm[2][0] - Dm[0][0] * Dm[2][1]) * id;
        o[8] = (Dm[0][0] * Dm[1][1] - Dm[0][1] * Dm[1][0]) * id;
      }
    }
    __syncwarp();
  }
}

}  // namespace nsb
