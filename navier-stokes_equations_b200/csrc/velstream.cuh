// Velocity-block operator of the polynomial preconditioner as a Blackwell-native stream.
//
// Replaces, together with its polynomial driver in nsb200.cu, the Ifpack ILU(1) application on F of the reference
// (reference src/classes/NavierStokes.hpp:302-304, 325).  The operator applied is B = Dinv F, the node-block-Jacobi
// scaled velocity block, kept in a PRIVATE packed copy (fp32 or fp16 values, products and sums in fp64, so every
// application is the same fixed linear operator and the outer iteration stays plain GMRES):
//
//   * the owned nodes are cut into tiles (structure.cpp: build_tile_plan / build_vel_stream); the dim x dim blocks of a
//     node are grouped in quads of four (lists padded with zero blocks), and a tile is stored plane by plane, `NQ` (quads
//     rounded up to 32) x 4 values per plane, so the whole tile is ONE contiguous chunk and lane q of a warp reads the four
//     values of quad q of a plane with one conflict-free 128-bit (fp32) / 64-bit (fp16) shared-memory load.  One lane per
//     quad instead of one per block cuts the warp shuffles of the reduction (they share the LSU pipe with the shared-memory
//     loads, which is what bounded the one-lane-per-block form) by four;
//   * one persistent CTA per SM.  Warp 0 is the producer: per tile and pipeline stage it issues three TMA bulk copies
//     (cp.async.bulk global -> shared, completion on an mbarrier: header, values, block metadata) and gathers the x values
//     of the tile's unique neighbour nodes with cp.async, arriving on the same mbarrier.  The other warps are consumers:
//     lane-per-quad products out of shared memory, a segmented warp scan over the quads of one node, sums carried across
//     the steps of a warp in a fixed order (bit-reproducible, no atomics); the warps of a tile own disjoint node ranges,
//     so each finishes its rows alone (no CTA-wide barrier) with the fused epilogue:
//         MODE 2:  y = B x                                       (Arnoldi on the scaled block)
//         MODE 3:  y = cu*u + ct*(B x) ; poly += cpu*u + cpy*y   (one root of the polynomial in product form)
//         MODE 4:  y = cu*u + ct*(B x)                           (scaled residual ahead of the smoother)
//   * stages are recycled through a second mbarrier per stage (consumers -> producer); the consumer warps form two groups
//     that take alternate tiles, so one group's block loop overlaps the other's waits and epilogue.
//
// DRAM traffic per application = the packed values + 4 B of metadata per block + the vectors of the epilogue; nothing is
// read twice from HBM (x comes through L2, once per tile that references it).
#pragma once
#include <cuda_fp16.h>

#include "device.cuh"
#include "linalg.cuh"
#include "structure.hpp"

namespace nsb {

constexpr int VS_GROUPS = 2;                       // consumer groups: consecutive tiles of a CTA go to alternating groups
constexpr int VS_THREADS = (VS_GROUPS * VS_CONSUMERS + 1) * 32;
constexpr int VS_MAX_UNIQ = TILE_MAX_UNIQ;

template <int DIM, typename VT> struct VsLayout {
  static constexpr int PL = DIM * DIM;
  static constexpr int VAL_BYTES = PL * VS_MAX_BLOCKS * (int)sizeof(VT);
  static constexpr int META_BYTES = VS_MAX_QUADS * 16;
  static constexpr int XS_BYTES = VS_MAX_UNIQ * DIM * 8;
  static constexpr int YS_BYTES = TILE_MAX_NODES * DIM * 8;
  static constexpr int HDR_BYTES = 64;
  static constexpr int OFF_VAL = 0;
  static constexpr int OFF_META = OFF_VAL + VAL_BYTES;
  static constexpr int OFF_XS = OFF_META + META_BYTES;
  static constexpr int OFF_YS = OFF_XS + XS_BYTES;
  static constexpr int OFF_HDR = OFF_YS + YS_BYTES;
  static constexpr int STAGE_BYTES = ((OFF_HDR + HDR_BYTES + 127) / 128) * 128;
  // as many stages as fit next to the barriers (2 for fp32, 3 for fp16 in 3-D)
  static constexpr int STAGES = (227 * 1024 - 256) / STAGE_BYTES >= 3 ? 3 : 2;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 256;
};

// ---- PTX wrappers (mbarrier, TMA bulk copy, cp.async) -------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// TMA bulk copy global -> shared of `bytes` (multiple of 16, both sides 16-byte aligned), completes on `bar`
__device__ __forceinline__ void tma_bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void cp_async_8(void* dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
// this thread's outstanding cp.async copies arrive on `bar` when they have landed (the barrier's count includes them)
__device__ __forceinline__ void cp_async_arrive_noinc(uint64_t* bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// what the producer reads of a tile's global header: the tile, its value / metadata chunk and its unique neighbour list
struct VsHead {
  int t, NQ, nq_off, u0, nuq;
};

// the four values of one quad of one plane
__device__ __forceinline__ void vs_load4(const float* p, double (&v)[4]) {
  const float4 f = *reinterpret_cast<const float4*>(p);
  v[0] = (double)f.x; v[1] = (double)f.y; v[2] = (double)f.z; v[3] = (double)f.w;
}
__device__ __forceinline__ void vs_load4(const __half* p, double (&v)[4]) {
  const uint2 r = *reinterpret_cast<const uint2*>(p);
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&r.x)), b = __half22float2(*reinterpret_cast<const __half2*>(&r.y));
  v[0] = (double)a.x; v[1] = (double)a.y; v[2] = (double)b.x; v[3] = (double)b.y;
}

// n_tiles comes last so that the pointer pairs and pc sit 16-byte aligned in the parameter bank: the epilogue then reads
// them with 128-bit uniform loads
template <int DIM, typename VT, int MODE>
__global__ void __launch_bounds__(VS_THREADS, 1)
k_vel_stream(const VsTile* __restrict__ tiles, const VT* __restrict__ vals, const uint32_t* __restrict__ meta,
             const int* __restrict__ uniq_xoff, const double* __restrict__ x, double* __restrict__ y,
             const double* __restrict__ u, double* __restrict__ poly, PolyCoef pc, int n_tiles) {
  using L = VsLayout<DIM, VT>;
  constexpr int PL = L::PL;
  constexpr int S = L::STAGES;
  extern __shared__ __align__(128) unsigned char vs_smem[];
  uint64_t* full = reinterpret_cast<uint64_t*>(vs_smem + S * L::STAGE_BYTES);
  uint64_t* empty = full + S;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(full + s, 1 + 32);               // expect_tx arrival of lane 0 + the 32 cp.async arrivals of the producer warp
      mbar_init(empty + s, VS_CONSUMERS);        // one arrival per consumer warp
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const int my_tiles = (n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;      // static round-robin

  if (warp == 0) {
    // ------------------------------------------------------------------ producer
    // Software-pipelined so that no global round trip sits between "stage free" and "stage refilling": the headers of this
    // CTA's tiles are loaded a batch of 32 ahead (lane j holds tile b + j) and read by shuffle, and the neighbour offsets of
    // tile it + 1 are loaded as soon as the copies of tile it are issued, so they land while the producer waits for the next
    // stage.  Between the wait on a stage and its copies there is nothing but shuffles.
    constexpr int PER_LANE = VS_MAX_UNIQ / 32;
    const int k0 = (int)blockIdx.x, dk = (int)gridDim.x;          // the it-th tile of this CTA is k0 + it * dk
    auto fetch = [&](int b, VsHead& h) {
      const int it = b + lane;
      h = VsHead{0, 0, 0, 0, 0};
      if (it < my_tiles) {
        h.t = k0 + it * dk;
        const VsTile* hd = tiles + h.t;
        h.NQ = __ldg(&hd->NQ); h.nq_off = __ldg(&hd->nq_off); h.u0 = __ldg(&hd->u0); h.nuq = __ldg(&hd->nuq);
      }
    };
    // offsets of the unique neighbour nodes of tile `it` (-1: none), lane + 32 q
    auto offsets = [&](int it, int u0, int nuq, int (&xo)[PER_LANE]) {
#pragma unroll
      for (int q = 0; q < PER_LANE; ++q) {
        const int i = lane + 32 * q;
        xo[q] = it < my_tiles && i < nuq ? __ldg(uniq_xoff + u0 + i) : -1;
      }
    };
    VsHead cur, nxt;                               // headers of tiles [b, b + 32) and [b + 32, b + 64)
    fetch(0, cur);
    fetch(32, nxt);
    int xo[PER_LANE];
    offsets(0, __shfl_sync(NSB_FULL, cur.u0, 0), __shfl_sync(NSB_FULL, cur.nuq, 0), xo);
    for (int it = 0; it < my_tiles; ++it) {
      const int s = it % S;
      const uint32_t ph = (uint32_t)(it / S) & 1u;
      if (it > 0 && (it & 31) == 0) {
        cur = nxt;
        fetch(it + 32, nxt);
      }
      const int t = __shfl_sync(NSB_FULL, cur.t, it & 31);
      const int NQ = __shfl_sync(NSB_FULL, cur.NQ, it & 31), nq_off = __shfl_sync(NSB_FULL, cur.nq_off, it & 31);
      if (it >= S) mbar_wait(empty + s, ph ^ 1u);                       // consumers released the stage's previous tile
      unsigned char* st = vs_smem + s * L::STAGE_BYTES;
      if (lane == 0) {
        const uint32_t vb = (uint32_t)(PL * 4 * NQ * (int)sizeof(VT)), mb = (uint32_t)(NQ * 16);
        mbar_expect_tx(full + s, vb + mb + (uint32_t)L::HDR_BYTES);
        tma_bulk_g2s(st + L::OFF_HDR, tiles + t, L::HDR_BYTES, full + s);
        tma_bulk_g2s(st + L::OFF_VAL, vals + (long long)PL * 4 * nq_off, vb, full + s);
        tma_bulk_g2s(st + L::OFF_META, meta + (long long)4 * nq_off, mb, full + s);
      }
      // x values of the tile's unique neighbour nodes
      double* xs = reinterpret_cast<double*>(st + L::OFF_XS);
#pragma unroll
      for (int q = 0; q < PER_LANE; ++q) {
        if (xo[q] >= 0) {
          const int i = lane + 32 * q;
#pragma unroll
          for (int c = 0; c < DIM; ++c) cp_async_8(xs + i * DIM + c, x + xo[q] + c);
        }
      }
      cp_async_arrive_noinc(full + s);
      // offsets of tile it + 1, whose header is in this batch or the next one
      const bool in_cur = (it & 31) != 31;
      const int u0 = __shfl_sync(NSB_FULL, in_cur ? cur.u0 : nxt.u0, (it + 1) & 31);
      const int nuq = __shfl_sync(NSB_FULL, in_cur ? cur.nuq : nxt.nuq, (it + 1) & 31);
      offsets(it + 1, u0, nuq, xo);
    }
    return;
  }

  // -------------------------------------------------------------------- consumers
  const int grp = (warp - 1) / VS_CONSUMERS;      // consumer group of this warp
  const int cw = (warp - 1) % VS_CONSUMERS;       // its index inside the group = its share of the tile
  for (int it = grp; it < my_tiles; it += VS_GROUPS) {
    const int s = it % S;
    const uint32_t ph = (uint32_t)(it / S) & 1u;
    mbar_wait(full + s, ph);
    unsigned char* st = vs_smem + s * L::STAGE_BYTES;
    const VsTile* hd = reinterpret_cast<const VsTile*>(st + L::OFF_HDR);
    const VT* sv = reinterpret_cast<const VT*>(st + L::OFF_VAL);
    const uint4* sm = reinterpret_cast<const uint4*>(st + L::OFF_META);
    const double* xs = reinterpret_cast<const double*>(st + L::OFF_XS);
    double* ys = reinterpret_cast<double*>(st + L::OFF_YS);
    const int NQ = hd->NQ, nn = hd->nn, n0 = hd->n0, nquad = hd->nquad;
    const int b0 = hd->split[cw], b1 = hd->split[cw + 1];      // node-aligned quad range of this warp
    // rows of this warp's nodes: [r0, r1) within the tile; the warp finishes them alone (no CTA-wide barrier), and the
    // operands of the fused epilogue are fetched now so that their latency overlaps the quad loop
    const int na = b0 < b1 ? (int)sm[b0].z : 0;
    const int nb_ = b0 < b1 ? (b1 < nquad ? (int)sm[b1].z : nn) : 0;
    const int r0 = DIM * na, r1 = DIM * nb_;
    const long long rowg0 = (long long)DIM * n0;
    double pu[2], pp[2];
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int i = r0 + lane + 32 * q;
      pu[q] = 0.0; pp[q] = 0.0;
      if (MODE >= 3 && i < r1) { pu[q] = u[rowg0 + i]; if (MODE == 3) pp[q] = poly[rowg0 + i]; }
    }
    int carry_row = -1;
    double carry[DIM];
#pragma unroll
    for (int r = 0; r < DIM; ++r) carry[r] = 0.0;
    for (int base = b0; base < b1; base += 32) {
      const int j = base + lane;
      const bool ok = j < b1;
      double acc[DIM];
#pragma unroll
      for (int r = 0; r < DIM; ++r) acc[r] = 0.0;
      int row = 0xffff;
      if (ok) {
        const uint4 m = sm[j];
        row = (int)m.z;
        double xv[4][DIM];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int loc = (int)(((e < 2 ? m.x : m.y) >> (16 * (e & 1))) & 0xffffu);
#pragma unroll
          for (int c = 0; c < DIM; ++c) xv[e][c] = xs[loc * DIM + c];
        }
#pragma unroll
        for (int r = 0; r < DIM; ++r)
#pragma unroll
          for (int c = 0; c < DIM; ++c) {
            double v[4];
            vs_load4(sv + ((size_t)(r * DIM + c) * NQ + j) * 4, v);
#pragma unroll
            for (int e = 0; e < 4; ++e) acc[r] += v[e] * xv[e][c];
          }
      }
      // the sum carried over from the previous step belongs to lane 0's node, or that node is complete
      const int row0 = __shfl_sync(NSB_FULL, row, 0);
      if (lane == 0 && carry_row >= 0) {
        if (carry_row == row0) {
#pragma unroll
          for (int r = 0; r < DIM; ++r) acc[r] += carry[r];
        } else {
#pragma unroll
          for (int r = 0; r < DIM; ++r) ys[carry_row * DIM + r] = carry[r];
        }
      }
      // segmented inclusive scan over the lanes of one node (the quads of a node are consecutive)
      const int prev = __shfl_up_sync(NSB_FULL, row, 1);
      const unsigned heads = __ballot_sync(NSB_FULL, lane == 0 || prev != row);
      const int pos = lane - (31 - __clz(heads & (0xffffffffu >> (31 - lane))));
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
#pragma unroll
        for (int r = 0; r < DIM; ++r) {
          const double o = __shfl_up_sync(NSB_FULL, acc[r], d);
          if (pos >= d) acc[r] += o;
        }
      }
      const bool last_of_seg = (lane == 31) || ((heads >> (lane + 1)) & 1u);
      if (last_of_seg && lane < 31 && row < nn) {
#pragma unroll
        for (int r = 0; r < DIM; ++r) ys[row * DIM + r] = acc[r];
      }
      carry_row = __shfl_sync(NSB_FULL, row, 31);
      if (carry_row >= nn) carry_row = -1;
#pragma unroll
      for (int r = 0; r < DIM; ++r) carry[r] = __shfl_sync(NSB_FULL, acc[r], 31);
    }
    if (lane == 0 && carry_row >= 0) {
#pragma unroll
      for (int r = 0; r < DIM; ++r) ys[carry_row * DIM + r] = carry[r];
    }
    __syncwarp();                                 // this warp's node sums are in ys
    // ---- fused epilogue over this warp's rows (contiguous in memory)
    for (int i = r0 + lane, q = 0; i < r1; i += 32, ++q) {
      const double t = ys[i];
      if (MODE == 2) {
        y[rowg0 + i] = t;
      } else {
        const double uv = q == 0 ? pu[0] : q == 1 ? pu[1] : u[rowg0 + i];
        const double pv = MODE != 3 ? 0.0 : q == 0 ? pp[0] : q == 1 ? pp[1] : poly[rowg0 + i];
        const double yv = pc.cu * uv + pc.ct * t;
        y[rowg0 + i] = yv;
        if (MODE == 3) poly[rowg0 + i] = pv + pc.cpu * uv + pc.cpy * yv;
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(empty + s);        // this warp is done with the stage (values, x, sums)
  }
}

// Packs B = Dinv F of the assembled system into the tile-planar layout (one CTA per tile).
template <int DIM, typename VT> __device__ __forceinline__ VT vs_from_double(double v);
template <> __device__ __forceinline__ float vs_from_double<2, float>(double v) { return (float)v; }
template <> __device__ __forceinline__ float vs_from_double<3, float>(double v) { return (float)v; }
template <> __device__ __forceinline__ __half vs_from_double<2, __half>(double v) { return __float2half_rn((float)v); }
template <> __device__ __forceinline__ __half vs_from_double<3, __half>(double v) { return __float2half_rn((float)v); }

template <int DIM, typename VT>
__global__ void __launch_bounds__(256)
k_vel_pack(DevMesh M, const VsTile* __restrict__ tiles, const uint32_t* __restrict__ meta, const double* __restrict__ vals,
           const double* __restrict__ dinv, VT* __restrict__ out) {
  constexpr int PL = DIM * DIM;
  const VsTile hd = tiles[blockIdx.x];
  VT* o = out + (long long)PL * 4 * hd.nq_off;
  const uint4* mt = reinterpret_cast<const uint4*>(meta) + hd.nq_off;
  // one thread per block (4 * NQ of them, padding included)
  for (int jb = threadIdx.x; jb < 4 * hd.NQ; jb += blockDim.x) {
    const int q = jb >> 2, e = jb & 3;
    double b[DIM][DIM];
#pragma unroll
    for (int r = 0; r < DIM; ++r)
#pragma unroll
      for (int c = 0; c < DIM; ++c) b[r][c] = 0.0;
    const uint4 m = __ldg(mt + q);
    if (m.z != 0xffffu && e < (int)(m.w >> 16)) {
      const int A = hd.n0 + (int)m.z;
      const NodeDesc d = load_desc(M.nd + A);
      const int k = (int)(m.w & 0xffffu) + e, len = DIM * d.nb + d.np;
      double f[DIM][DIM], di[DIM][DIM];
#pragma unroll
      for (int r = 0; r < DIM; ++r)
#pragma unroll
        for (int c = 0; c < DIM; ++c) {
          f[r][c] = __ldcs(vals + d.rowbase + (long long)r * len + DIM * k + c);
          di[r][c] = __ldg(dinv + (size_t)A * PL + r * DIM + c);
        }
#pragma unroll
      for (int r = 0; r < DIM; ++r)
#pragma unroll
        for (int c = 0; c < DIM; ++c)
#pragma unroll
          for (int ee = 0; ee < DIM; ++ee) b[r][c] += di[r][ee] * f[ee][c];
    }
#pragma unroll
    for (int r = 0; r < DIM; ++r)
#pragma unroll
      for (int c = 0; c < DIM; ++c) o[((size_t)(r * DIM + c) * hd.NQ + q) * 4 + e] = vs_from_double<DIM, VT>(b[r][c]);
  }
}

}  // namespace nsb
