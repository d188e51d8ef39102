// C-ABI implementation (include/nsb200.h): device context, uploads, the two assembly
// passes, the block-triangular preconditioner and restarted GMRES.  sm_100a only; there is
// no CPU fallback -- every entry point fails loudly when no CUDA device is usable.
#include "../../include/nsb200.h"

#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>   // types only: the library is resolved at run time (see NcclApi)
#include <nvrtc.h>  // types only: the library is resolved at run time (see NvrtcApi)

#include <algorithm>
#include <cerrno>
#include <climits>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "amg.hpp"
#include "small_eig.hpp"
#include "assemble.cuh"
#include "device.cuh"
#include "linalg.cuh"
#include "structure.hpp"
#include "twolevel.cuh"
#include "velstream.cuh"

using namespace nsb;

namespace {

struct CudaErr {
  std::string msg;
};
#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess)                                                                         \
      throw CudaErr{std::string(#call) + " failed: " + cudaGetErrorString(e_) + " (" __FILE__ ":" + \
                    std::to_string(__LINE__) + ")"};                                               \
  } while (0)
#define CKN(call)                                                                        \
  do {                                                                                   \
    ncclResult_t r_ = (call);                                                            \
    if (r_ != ncclSuccess)                                                               \
      throw CudaErr{std::string(#call) + " failed: " + g_nccl.GetErrorString(r_)};       \
  } while (0)

// NCCL is bound lazily with dlopen so that libnsb200.so has no link-time dependency on a
// particular libnccl.so.2: inside a PyTorch process the already-loaded (newer) NCCL is reused,
// in a plain C++ program the system one is loaded.  Only needed with more than one rank.
struct NcclApi {
  void* handle = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  bool load(std::string& err) {
    if (handle) return true;
    for (const char* name : {"libnccl.so.2", "libnccl.so"}) {
      handle = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
      if (handle) break;
    }
    if (!handle) { err = std::string("cannot load NCCL: ") + dlerror(); return false; }
    auto sym = [&](const char* n) { void* p = dlsym(handle, n); if (!p) err = std::string("NCCL symbol missing: ") + n; return p; };
    GetUniqueId = (decltype(GetUniqueId))sym("ncclGetUniqueId");
    CommInitRank = (decltype(CommInitRank))sym("ncclCommInitRank");
    CommDestroy = (decltype(CommDestroy))sym("ncclCommDestroy");
    AllReduce = (decltype(AllReduce))sym("ncclAllReduce");
    AllGather = (decltype(AllGather))sym("ncclAllGather");
    Send = (decltype(Send))sym("ncclSend");
    Recv = (decltype(Recv))sym("ncclRecv");
    GroupStart = (decltype(GroupStart))sym("ncclGroupStart");
    GroupEnd = (decltype(GroupEnd))sym("ncclGroupEnd");
    GetErrorString = (decltype(GetErrorString))sym("ncclGetErrorString");
    return GetUniqueId && CommInitRank && CommDestroy && AllReduce && AllGather && Send && Recv && GroupStart && GroupEnd && GetErrorString;
  }
};
NcclApi g_nccl;

// NVRTC compiles a user's device-side forcing term (nsb_set_forcing_source).  Bound lazily like NCCL: libnsb200.so has no
// link-time dependency on it, and inside a PyTorch process the NVRTC torch already loaded may be the one found (any 12.8+
// compiles for sm_100a; nsb_forcing_info reports the version).  Only the forcing-source entries need it.
struct NvrtcApi {
  void* handle = nullptr;
  std::string err;
  int major = 0, minor = 0;
  const char* (*GetErrorString)(nvrtcResult) = nullptr;
  nvrtcResult (*Version)(int*, int*) = nullptr;
  nvrtcResult (*CreateProgram)(nvrtcProgram*, const char*, const char*, int, const char* const*, const char* const*) = nullptr;
  nvrtcResult (*CompileProgram)(nvrtcProgram, int, const char* const*) = nullptr;
  nvrtcResult (*GetProgramLogSize)(nvrtcProgram, size_t*) = nullptr;
  nvrtcResult (*GetProgramLog)(nvrtcProgram, char*) = nullptr;
  nvrtcResult (*GetCUBINSize)(nvrtcProgram, size_t*) = nullptr;
  nvrtcResult (*GetCUBIN)(nvrtcProgram, char*) = nullptr;
  nvrtcResult (*DestroyProgram)(nvrtcProgram*) = nullptr;
  bool load() {
    if (handle) return true;
    if (!err.empty()) return false;
    for (const char* name : {"libnvrtc.so.12", "libnvrtc.so"}) {
      handle = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
      if (handle) break;
    }
    if (!handle) { err = std::string("cannot load NVRTC (libnvrtc.so.12), needed to compile a forcing source: ") + dlerror(); return false; }
    auto sym = [&](const char* n) { void* p = dlsym(handle, n); if (!p) err = std::string("NVRTC symbol missing: ") + n; return p; };
    GetErrorString = (decltype(GetErrorString))sym("nvrtcGetErrorString");
    Version = (decltype(Version))sym("nvrtcVersion");
    CreateProgram = (decltype(CreateProgram))sym("nvrtcCreateProgram");
    CompileProgram = (decltype(CompileProgram))sym("nvrtcCompileProgram");
    GetProgramLogSize = (decltype(GetProgramLogSize))sym("nvrtcGetProgramLogSize");
    GetProgramLog = (decltype(GetProgramLog))sym("nvrtcGetProgramLog");
    GetCUBINSize = (decltype(GetCUBINSize))sym("nvrtcGetCUBINSize");
    GetCUBIN = (decltype(GetCUBIN))sym("nvrtcGetCUBIN");
    DestroyProgram = (decltype(DestroyProgram))sym("nvrtcDestroyProgram");
    if (!err.empty()) { dlclose(handle); handle = nullptr; return false; }
    Version(&major, &minor);
    return true;
  }
};
NvrtcApi g_nvrtc;

// csrc/forcing_eval.cuh as text (the Makefile wraps it in a raw string literal)
const char kForcingEvalSrc[] =
#include "../forcing_eval_src.inc"
    ;

constexpr int kForcingMaxParams = 16;
constexpr int kForcingBlock = 256;

// The NVRTC program for a forcing source: NSB_DIM / NSB_NQ, the user's text, the evaluation kernel.  The #line directives
// make the compiler's messages name the user's lines as they wrote them.
std::string forcing_program(int dim, const char* src, const std::string& opts) {
  std::string p = "// device-side forcing term of nsb200, compiled with NVRTC: " + opts + "\n";
  p += "#define NSB_DIM " + std::to_string(dim) + "\n#define NSB_NQ " + std::to_string(dim == 2 ? Fe<2>::NQ : Fe<3>::NQ) + "\n";
  p += "#line 1 \"nsb_forcing.cu\"\n";
  p += src;
  p += "\n#line 1 \"forcing_eval.cuh\"\n";
  p += kForcingEvalSrc;
  return p;
}

// Compiles the forcing program for `arch` (e.g. "sm_100a").  Returns "" and the cubin, or the error with NVRTC's log.
std::string compile_forcing(int dim, const char* src, const std::string& arch, std::vector<char>& cubin) {
  if (!g_nvrtc.load()) return g_nvrtc.err;
  const std::string o_arch = "--gpu-architecture=" + arch, o_std = "-std=c++17";
  const char* opts[] = {o_arch.c_str(), o_std.c_str()};
  const std::string text = forcing_program(dim, src, o_arch + " " + o_std);
  nvrtcProgram prog;
  nvrtcResult r = g_nvrtc.CreateProgram(&prog, text.c_str(), "nsb_forcing.cu", 0, nullptr, nullptr);
  if (r != NVRTC_SUCCESS) return std::string("nvrtcCreateProgram failed: ") + g_nvrtc.GetErrorString(r);
  r = g_nvrtc.CompileProgram(prog, 2, opts);
  std::string msg;
  if (r != NVRTC_SUCCESS) {
    size_t n = 0;
    g_nvrtc.GetProgramLogSize(prog, &n);
    std::string log(n, '\0');
    if (n) g_nvrtc.GetProgramLog(prog, &log[0]);
    while (!log.empty() && (log.back() == '\0' || log.back() == '\n')) log.pop_back();
    msg = std::string("forcing source does not compile (") + g_nvrtc.GetErrorString(r) + ", NVRTC " + std::to_string(g_nvrtc.major) +
          "." + std::to_string(g_nvrtc.minor) + ", " + arch + "):\n" + log;
  } else {
    size_t n = 0;
    r = g_nvrtc.GetCUBINSize(prog, &n);
    if (r == NVRTC_SUCCESS) {
      cubin.resize(n);
      r = g_nvrtc.GetCUBIN(prog, cubin.data());
    }
    if (r != NVRTC_SUCCESS) msg = std::string("nvrtcGetCUBIN failed: ") + g_nvrtc.GetErrorString(r);
  }
  g_nvrtc.DestroyProgram(&prog);
  return msg;
}

template <typename T> struct DBuf {
  T* p = nullptr;
  size_t n = 0;
  bool owned = true;
  DBuf() = default;
  DBuf(const DBuf&) = delete;
  DBuf& operator=(const DBuf&) = delete;
  ~DBuf() { if (p && owned) cudaFree(p); }
  void alloc(size_t count) {
    if (p && owned) cudaFree(p);
    p = nullptr; owned = true;
    n = count;
    if (count) CK(cudaMalloc(&p, count * sizeof(T)));
  }
  // non-owning view of `count` elements at `ptr` (a slot of the symmetric halo arena)
  void view(T* ptr, size_t count) {
    if (p && owned) cudaFree(p);
    p = ptr; n = count; owned = false;
  }
  void zero(cudaStream_t s) { if (n) CK(cudaMemsetAsync(p, 0, n * sizeof(T), s)); }
  void upload(const std::vector<T>& v, cudaStream_t s) {
    alloc(v.size());
    if (n) CK(cudaMemcpyAsync(p, v.data(), n * sizeof(T), cudaMemcpyHostToDevice, s));
  }
};

enum ProfCat { PC_ASM_CTX = 0, PC_ASM_ROWS, PC_SPMV, PC_SPMV_VEL, PC_SCHUR, PC_AMG, PC_ORTH, PC_OTHER, PC_ASM_PACK, PC_COARSE, PC_ASM_COARSE, PC_FORCING, PC_N };
const char* kProfNames[PC_N] = {"asm_context", "asm_rows", "spmv", "spmv_vel", "schur", "amg", "orth", "other", "asm_pack", "coarse", "asm_coarse", "forcing"};

struct Prof {
  bool on = false;
  std::vector<cudaEvent_t> pool;
  size_t used = 0;
  struct Rec { int cat; size_t e0, e1; };
  std::vector<Rec> recs;
  double ms[PC_N] = {0};
  int64_t cnt[PC_N] = {0};
  cudaEvent_t get() {
    if (used == pool.size()) { cudaEvent_t e; cudaEventCreate(&e); pool.push_back(e); }
    return pool[used++];
  }
  size_t begin(int cat, cudaStream_t s) {
    if (!on) return 0;
    Rec r{cat, used, 0};
    cudaEventRecord(get(), s);
    recs.push_back(r);
    return recs.size() - 1;
  }
  void end(size_t id, cudaStream_t s) {
    if (!on) return;
    recs[id].e1 = used;
    cudaEventRecord(get(), s);
  }
  void collect(cudaStream_t s) {
    if (recs.empty()) return;
    cudaStreamSynchronize(s);
    for (auto& r : recs) {
      float t = 0;
      cudaEventElapsedTime(&t, pool[r.e0], pool[r.e1]);
      ms[r.cat] += t;
      cnt[r.cat]++;
    }
    recs.clear();
    used = 0;
  }
  void reset() { for (int i = 0; i < PC_N; ++i) { ms[i] = 0; cnt[i] = 0; } recs.clear(); used = 0; }
  ~Prof() { for (auto e : pool) cudaEventDestroy(e); }
};

struct DevLevel {
  DevCsr A, P, R;
  DBuf<int> Aptr, Acol, Pptr, Pcol, Rptr, Rcol;
  DBuf<double> Aval, Pval, Rval, dinv;
  DBuf<double> x, x2, b, d, r;
  double lmax = 1.0;
  int n = 0;
};

struct HaloBuf {
  DBuf<double> u, p;
  DBuf<int> uoff, poff;
};

void upload_csr(const HostCsr& H, DBuf<int>& ptr, DBuf<int>& col, DBuf<double>& val, DevCsr& D, cudaStream_t s) {
  ptr.upload(H.ptr, s); col.upload(H.col, s); val.upload(H.val, s);
  D.n = H.n; D.m = H.m; D.ptr = ptr.p; D.col = col.p; D.val = val.p;
}

// Halo exchange by direct peer stores over NVLink (no NCCL on the data path).  Every vector that is ever exchanged lives in
// one arena per rank, at the SAME offset on every rank (slots of a common stride), exported once per mesh with
// cudaIpcGetMemHandle; a rank therefore knows the address of "the same vector" inside each peer.  An exchange is one
// kernel that writes the boundary values straight into the peers' ghost tails and then raises a sequence flag in each
// peer, and one single-warp kernel that waits for the peers' flags; both are ordinary stream work.
struct PeerHalo {
  bool on = false;
  DBuf<double> arena;
  size_t stride_f = 0, stride_c = 0, coarse_base = 0;
  int slots_f = 0, slots_c = 0;
  DBuf<unsigned long long> flags;          // [2*nranks]: data sequence numbers, then consumed ("ack") sequence numbers
  DBuf<unsigned int> counter;
  std::vector<void*> opened;               // IPC mappings to close
  std::vector<double*> peer_arena;         // per peer index (order of Structure::peer)
  std::vector<unsigned long long*> peer_flags;
  // device tables; segment s < npeers: velocity block for peer s, s >= npeers: pressure block for peer s - npeers
  DBuf<double*> d_peer_arena;
  DBuf<unsigned long long*> d_peer_flags;
  DBuf<int> d_peer_rank;
  DBuf<int> seg_ptr_f, src_f, seg_ptr_c, src_c;        // fine: 2*npeers segments; coarse: npeers segments
  DBuf<long long> land_f, land_c;                      // landing offset of each segment inside the peer's vector
  unsigned long long seq = 0;
  const double* last_vec = nullptr;
  int total_f_vel = 0, total_f_all = 0, total_c = 0;
};

// device view of one streamed operator (velstream.cuh)
struct VsDev {
  const VsTile* tiles;
  const uint32_t* meta;
  const int* uniq_xoff;
  const unsigned char* vals;
  int n_tiles;
};

// one level of the velocity preconditioner: sizes, work vectors, spectrum estimate and polynomial roots
struct PolyLevel {
  bool coarse = false;
  int nn = 0;                          // owned nodes
  long long n = 0, n_tot = 0;          // owned entries (dim * nn), entries including ghosts
  const double* dinv = nullptr;        // inverse node-diagonal blocks
  const int64_t* gid = nullptr;        // global node ids (probe vector)
  double *z0 = nullptr, *z1 = nullptr, *zd = nullptr, *poly = nullptr, *pin = nullptr;
  DBuf<double> probe;
  bool probe_init = false;
  std::vector<double> wr, wi;          // harmonic Ritz values of the last Arnoldi run
  double ritz_lo = 0, ritz_hi = 0, ritz_im = 0, ritz_top = 0, probe_res = 1.0;   // harmonic Ritz range, largest standard Ritz value
  std::vector<std::pair<double, double>> roots;   // (re, im >= 0), Leja ordered
};

// coarse P1 level of the two-level cycle (twolevel.cuh)
struct Coarse {
  DBuf<VsTile> tiles;
  DBuf<uint32_t> meta;
  DBuf<int> uniq_xoff;
  DBuf<unsigned char> vals;            // packed Dinv_c F_c
  int n_tiles = 0;
  int64_t total_nq = 0;
  DBuf<long long> nbr_ptr, vedge_ptr;
  DBuf<int> nbr_vxoff, vedge_xoff, ends_xoff, send_xoff;
  DBuf<double> cvals, dinv, rc, z0, z1, zd, poly, pin, send_buf;
  std::vector<int64_t> gid, h_nbr_ptr, h_nbr_gid;     // host copies: global vertex ids of the owned rows / of the neighbours
  bool built = false, valid = false;   // structures uploaded / operator matches the assembled system
};

}  // namespace

struct nsb_ctx {
  int dim = 0, device = 0;
  int rank = 0, nranks = 1;
  ncclComm_t comm = nullptr;
  cudaStream_t stream = nullptr;
  std::string err;
  bool have_mesh = false, have_matrix = false, have_pressure = false;
  int64_t launches = 0;
  Prof prof;
  cudaEvent_t t0 = nullptr, t1 = nullptr;

  // global mesh copies needed later on the host (pressure matrices)
  int64_t n_vertices = 0, n_cells = 0, n_u = 0, n_p = 0;
  std::vector<double> coords;
  std::vector<uint32_t> cell_vertices;
  std::vector<int> g_cell_pid;      // [C][NV] global pressure ids
  Structure S;
  DevMesh M{};
  // device copies of the structure
  DBuf<int> d_cell_xoff, d_cell_poff, d_nbr_xoff, d_pnbr_xoff, d_selfrank, d_node_pid, d_pid_node, d_pselfrank, d_tile_ptr;
  DBuf<double> d_cell_geom;
  DBuf<uint16_t> d_rank_uu, d_rank_up;
  DBuf<long long> d_nbr_ptr, d_pnbr_ptr, d_rowbase, d_prowbase, d_n2c_ptr;
  DBuf<uint32_t> d_n2c;
  DBuf<NodeDesc> d_nd;
  DBuf<FeTables> d_fe;              // L2-resident copy of the FE tables (kernels stage it in shared memory)
  int num_sms = 148;
  int n_tiles = 0, tile_smem_bytes = 0;
  DBuf<int> d_stile_ptr, d_suniq_ptr, d_suniq_xoff, d_spuniq_ptr, d_spuniq_xoff;   // SpMV tiles (see linalg.cuh)
  DBuf<unsigned short> d_nbr_loc, d_pnbr_loc;
  SpmvTiles stiles{};
  int n_stiles = 0;
  // global dof -> local vector offset (or -1)
  std::vector<int> g2x;
  DBuf<int> d_pid_gid;              // [np_own] global pressure id of each owned pressure DoF (multi-GPU)
  DBuf<int> d_own_gdof;             // [n_own] global DoF of each owned local entry (multi-GPU gathers)
  DBuf<double> w_tg, w_gather;      // replicated global pressure vector / full global vector
  // vectors, all in local layout [u_own | p_own | u_ghost | p_ghost]
  DBuf<double> v_old, v_oldold, v_cur, v_sol, v_rhs;
  DBuf<unsigned char> cflag;
  DBuf<double> cval;
  DBuf<int> c_idx;                  // local offsets of the current constraint set
  DBuf<double> c_val;
  int n_con = 0;
  // system
  nsb_params par{};
  nsb_solver_opts opt{};
  DBuf<double> vals, dinv, ctx, cell_rhs;
  // forcing per (local cell, quadrature point, component) at t and t - dt (nsb_set_forcing): both allocated while either
  // slot is non-zero, both freed when both are cleared; forcing_set[k] = slot k holds non-zero values
  DBuf<double> forcing[2];
  bool forcing_set[2] = {false, false};
  // device-evaluated forcing (nsb_set_forcing_source): the loaded evaluation kernel and the source it was compiled from,
  // its parameters, and what it maps the quadrature points from -- the coordinates of the vertices of the local cells and
  // a local cell -> vertex table (uploaded on first use, freed with the mesh)
  cudaLibrary_t fsrc_lib = nullptr;
  cudaKernel_t fsrc_kernel = nullptr;
  std::string fsrc_text;
  DBuf<double> fsrc_prm, fsrc_coords;
  DBuf<int> fsrc_cells;
  DBuf<unsigned int> fsrc_flag;
  bool fsrc_geom = false;
  int64_t fsrc_compiles = 0, fsrc_evals = 0;
  // streamed velocity operator (velstream.cuh): packed copy of Dinv F in fp32 / fp16, tile headers, block metadata
  DBuf<unsigned char> vs_vals;
  DBuf<VsTile> d_vs_tiles;
  DBuf<uint32_t> d_vs_meta;
  int64_t vs_total_nq = 0;
  bool vs_valid = false;            // vs_vals describe the currently assembled system
  int ctx_stride = 0;
  // pressure matrices (global, replicated)
  HostCsr h_Mp, h_Kp;
  DevCsr Mp{};
  DBuf<int> Mp_ptr, Mp_col;
  DBuf<double> Mp_val, Mp_dinv;
  double Mp_lmax = 1.0;
  std::vector<std::unique_ptr<DevLevel>> amg;
  std::vector<std::unique_ptr<HaloBuf>> halo;
  int vs_ctas = 0;                  // NSB200_VS_CTAS: at most this many CTAs per streamed-operator launch (0: one per SM)
  double* pin = nullptr;           // pinned staging buffer for host <-> device vector traffic (n_tot doubles)
  DBuf<double> coarse_inv;
  int coarse_n = 0;
  // preconditioner / Krylov workspace
  DBuf<double> w_z0, w_z1, w_d, w_t, w_y1, w_m0, w_m1, w_md, w_in, w_tmp, w_pin, w_poly, w_y0, w_u;
  Coarse cg;
  PeerHalo ph;
  PolyLevel lvF, lvC;
  bool two_level = false;           // the last setup chose the two-level cycle
  bool cycle_disabled = false;      // the cycle stalled on this mesh / flow regime: single-level polynomial from now on (reset by a new mesh or new options)
  DBuf<double> V;                   // Krylov basis, (m+1) vectors of n_own
  int V_cap = 0;
  DBuf<double> partial, d_h, d_nrm;
  int solves = 0;

  void launch_check() {
    ++launches;
#ifdef NSB_DEBUG_SYNC
    CK(cudaStreamSynchronize(stream));
#endif
    CK(cudaGetLastError());
  }
};

namespace {

int fail(nsb_ctx* c, const std::string& m, int code = -1) {
  if (c) c->err = m;
  return code;
}

#define NSB_TRY try {
#define NSB_CATCH(c)                                               \
  }                                                                \
  catch (const CudaErr& e) { return fail(c, e.msg); }              \
  catch (const std::exception& e) { return fail(c, e.what()); }

inline int nblk(long long n, int t) { return (int)((n + t - 1) / t); }

#ifndef NSB_DEFAULT_PRECOND_PRECISION
#define NSB_DEFAULT_PRECOND_PRECISION 16
#endif

// bytes of the packed copy of Dinv F (none when the polynomial runs on the fp64 values themselves)
size_t vs_vals_bytes(const nsb_ctx* c) {
  if (c->opt.precond_precision == 64) return 0;
  return (size_t)c->vs_total_nq * 4 * c->dim * c->dim * (c->opt.precond_precision == 16 ? 2 : 4);
}

// ---- halo exchange of one local vector (ghost tail refreshed from the owners) -----------
// one exchange by peer stores: optional consumed-handshake (when the same buffer is exchanged twice in a row the peers
// might still be reading its ghosts), push + flag, wait
void peer_wait(nsb_ctx* c) {
  PeerHalo& H = c->ph;
  const int np = (int)c->S.peer.size();
  if (np == 0) return;
  k_halo_wait<<<1, 32, 0, c->stream>>>(np, H.d_peer_rank.p, H.flags.p, H.seq);
  c->launch_check();
}

void peer_exchange(nsb_ctx* c, const double* v, int nseg, const DBuf<int>& seg_ptr, const DBuf<int>& src, const DBuf<long long>& land,
                   int total_entries) {
  PeerHalo& H = c->ph;
  const int np = (int)c->S.peer.size();
  if (np == 0) return;
  const long long vec_off = v - H.arena.p;
  if (vec_off < 0 || (size_t)vec_off >= H.arena.n) throw CudaErr{"halo exchange of a vector outside the symmetric arena"};
  if (v == H.last_vec) {
    k_halo_ack<<<1, 32, 0, c->stream>>>(np, H.d_peer_flags.p, c->nranks, c->rank, H.seq);
    c->launch_check();
    k_halo_wait<<<1, 32, 0, c->stream>>>(np, H.d_peer_rank.p, H.flags.p + c->nranks, H.seq);
    c->launch_check();
  }
  H.last_vec = v;
  ++H.seq;
  const int grid = std::max(1, std::min(nblk(total_entries, 256), 64));
  k_halo_push<<<grid, 256, 0, c->stream>>>(nseg, np, seg_ptr.p, src.p, land.p, H.d_peer_arena.p, vec_off, v, H.d_peer_flags.p, c->rank,
                                            H.seq, H.counter.p);
  c->launch_check();
  peer_wait(c);
}

void halo_exchange(nsb_ctx* c, double* v, bool with_pressure = true) {
  if (c->nranks == 1) return;
  const Structure& S = c->S;
  if (c->ph.on) {
    const int np = (int)S.peer.size();
    const int nseg = with_pressure ? 2 * np : np;
    peer_exchange(c, v, nseg, c->ph.seg_ptr_f, c->ph.src_f, c->ph.land_f, with_pressure ? c->ph.total_f_all : c->ph.total_f_vel);
    return;
  }
  // One pack kernel for all peers (+ one for the pressure DoFs), then a grouped send/recv: ghosts are stored per
  // owner contiguously, so receives land in place.  The velocity polynomial only needs velocity ghosts.
  auto& B = c->halo;
  if (B.empty()) {
    auto b = std::make_unique<HaloBuf>();
    std::vector<int> uo, po;
    for (size_t k = 0; k < S.peer.size(); ++k) {
      for (int n : S.send_nodes[k]) uo.push_back((int)S.node_xoff(n));
      for (int q : S.send_pids[k]) po.push_back((int)S.pid_xoff(q));
    }
    b->uoff.upload(uo, c->stream); b->poff.upload(po, c->stream);
    CK(cudaStreamSynchronize(c->stream));
    b->u.alloc(uo.size() * S.dim); b->p.alloc(po.size());
    B.push_back(std::move(b));
  }
  HaloBuf& H = *B[0];
  const long long tu = (long long)H.uoff.n, tp = (long long)H.poff.n;
  if (tu) { k_gather_nodes<<<nblk(tu * S.dim, 256), 256, 0, c->stream>>>((int)tu, S.dim, H.uoff.p, v, H.u.p); c->launch_check(); }
  if (with_pressure && tp) { k_gather<<<nblk(tp, 256), 256, 0, c->stream>>>((int)tp, H.poff.p, v, H.p.p); c->launch_check(); }
  CKN(g_nccl.GroupStart());
  long long uoff = S.n_own_dofs(), poff = S.n_own_dofs() + (long long)S.dim * S.nn_ghost;
  size_t su = 0, sp = 0;
  for (size_t k = 0; k < S.peer.size(); ++k) {
    const int peer = S.peer[k];
    const size_t nu = S.send_nodes[k].size() * S.dim, np = S.send_pids[k].size();
    if (nu) CKN(g_nccl.Send(H.u.p + su, nu, ncclDouble, peer, c->comm, c->stream));
    if (with_pressure && np) CKN(g_nccl.Send(H.p.p + sp, np, ncclDouble, peer, c->comm, c->stream));
    const size_t ru = (size_t)S.recv_node_count[k] * S.dim, rp = (size_t)S.recv_pid_count[k];
    if (ru) CKN(g_nccl.Recv(v + uoff, ru, ncclDouble, peer, c->comm, c->stream));
    if (with_pressure && rp) CKN(g_nccl.Recv(v + poff, rp, ncclDouble, peer, c->comm, c->stream));
    uoff += ru; poff += rp;
    su += nu; sp += np;
  }
  CKN(g_nccl.GroupEnd());
}

void allreduce_sum(nsb_ctx* c, double* dbuf, int n) {
  if (c->nranks == 1) return;
  CKN(g_nccl.AllReduce(dbuf, dbuf, n, ncclDouble, ncclSum, c->comm, c->stream));
}

// ---- templated launch helpers --------------------------------------------------------
template <int DIM> void launch_coarse_assemble(nsb_ctx* c);

template <int DIM> void launch_assemble(nsb_ctx* c, bool newton) {
  AsmParams P;
  P.dt = c->par.dt; P.inv_dt = 1.0 / c->par.dt; P.theta = c->par.theta; P.nu = c->par.nu; P.rho = c->par.rho;
  P.use_supg = c->par.use_supg;
  P.gamma = c->par.use_supg ? c->par.gamma : 0.0;
  P.first_order_ustar = c->par.first_order_ustar;
  const int stride = newton ? Ctx<DIM>::N_NEWTON : CtxL<DIM>::N;
  if ((int)c->ctx_stride < stride) {
    c->ctx.alloc((size_t)c->S.nc * stride);
    c->ctx_stride = stride;
  }
  const double* vecA = newton ? c->v_cur.p : c->v_old.p;
  const double* vecB = newton ? c->v_old.p : c->v_oldold.p;
  size_t id = c->prof.begin(PC_ASM_CTX, c->stream);
  const int cgrid = std::min(nblk(c->S.nc, ASM_WARPS), c->num_sms * 8);     // persistent: CTAs stride over the cells
  const double *fn = c->forcing[NSB_FORCING_NEW].p, *fo = c->forcing[NSB_FORCING_OLD].p;
  const bool forced = fn != nullptr;          // both slots are allocated together, and only while one is non-zero
  if (newton && forced)
    k_cell_context<DIM, true, true><<<cgrid, ASM_WARPS * 32, 0, c->stream>>>(c->M, P, c->d_fe.p, vecA, vecB, c->ctx.p, c->cell_rhs.p, fn, fo);
  else if (newton)
    k_cell_context<DIM, true, false><<<cgrid, ASM_WARPS * 32, 0, c->stream>>>(c->M, P, c->d_fe.p, vecA, vecB, c->ctx.p, c->cell_rhs.p, nullptr, nullptr);
  else if (forced)
    k_cell_context<DIM, false, true><<<cgrid, ASM_WARPS * 32, 0, c->stream>>>(c->M, P, c->d_fe.p, vecA, vecB, c->ctx.p, c->cell_rhs.p, fn, fo);
  else
    k_cell_context<DIM, false, false><<<cgrid, ASM_WARPS * 32, 0, c->stream>>>(c->M, P, c->d_fe.p, vecA, vecB, c->ctx.p, c->cell_rhs.p, nullptr, nullptr);
  c->launch_check();
  c->prof.end(id, c->stream);
  RowOut out{c->vals.p, c->v_rhs.p, c->dinv.p};
  id = c->prof.begin(PC_ASM_ROWS, c->stream);
  if (newton)
    k_node_rows<DIM, true><<<c->n_tiles, ASM_WARPS * 32, c->tile_smem_bytes, c->stream>>>(c->M, P, c->ctx.p, c->cell_rhs.p, c->cflag.p, c->cval.p, out, c->d_tile_ptr.p, c->d_fe.p);
  else
    k_node_rows<DIM, false><<<c->n_tiles, ASM_WARPS * 32, c->tile_smem_bytes, c->stream>>>(c->M, P, c->ctx.p, c->cell_rhs.p, c->cflag.p, c->cval.p, out, c->d_tile_ptr.p, c->d_fe.p);
  c->launch_check();
  c->prof.end(id, c->stream);
  // packed copy of Dinv F for the streamed velocity operator
  c->vs_valid = false;
  if (c->vs_vals.p) {
    id = c->prof.begin(PC_ASM_PACK, c->stream);
    if (c->opt.precond_precision == 16)
      k_vel_pack<DIM, __half><<<c->n_stiles, 256, 0, c->stream>>>(c->M, c->d_vs_tiles.p, c->d_vs_meta.p, c->vals.p, c->dinv.p, reinterpret_cast<__half*>(c->vs_vals.p));
    else
      k_vel_pack<DIM, float><<<c->n_stiles, 256, 0, c->stream>>>(c->M, c->d_vs_tiles.p, c->d_vs_meta.p, c->vals.p, c->dinv.p, reinterpret_cast<float*>(c->vs_vals.p));
    c->launch_check();
    c->prof.end(id, c->stream);
    c->vs_valid = true;
  }
  // Galerkin coarse operator of the two-level cycle (linearised systems: their cell context holds S_ab)
  c->cg.valid = false;
  if (!newton && c->vs_valid && c->cg.built && c->opt.velocity_cycle != 1) launch_coarse_assemble<DIM>(c);
}

template <int DIM> void set_smem_attr(int bytes) {
  CK(cudaFuncSetAttribute(k_node_rows<DIM, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  CK(cudaFuncSetAttribute(k_node_rows<DIM, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
}

template <int DIM, typename VT> void set_vs_attr() {
  const int bytes = VsLayout<DIM, VT>::SMEM_BYTES;
  CK(cudaFuncSetAttribute(k_vel_stream<DIM, VT, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  CK(cudaFuncSetAttribute(k_vel_stream<DIM, VT, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  CK(cudaFuncSetAttribute(k_vel_stream<DIM, VT, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
}

// one application of the streamed operator over all tiles of D
template <int DIM, typename VT, int MODE>
void launch_vel_stream(nsb_ctx* c, const VsDev& D, const double* x, double* y, const double* u, double* poly, PolyCoef pc) {
  if (D.n_tiles <= 0) return;
  const int grid = std::min(std::min(D.n_tiles, c->num_sms), c->vs_ctas > 0 ? c->vs_ctas : D.n_tiles);
  k_vel_stream<DIM, VT, MODE><<<grid, VS_THREADS, VsLayout<DIM, VT>::SMEM_BYTES, c->stream>>>(
      D.tiles, reinterpret_cast<const VT*>(D.vals), D.meta, D.uniq_xoff, x, y, u, poly, pc, D.n_tiles);
  c->launch_check();
}
template <int MODE>
void vel_stream(nsb_ctx* c, const VsDev& D, const double* x, double* y, const double* u, double* poly, PolyCoef pc) {
  const bool h = c->opt.precond_precision == 16;
  if (c->dim == 2) {
    if (h) launch_vel_stream<2, __half, MODE>(c, D, x, y, u, poly, pc);
    else launch_vel_stream<2, float, MODE>(c, D, x, y, u, poly, pc);
  } else {
    if (h) launch_vel_stream<3, __half, MODE>(c, D, x, y, u, poly, pc);
    else launch_vel_stream<3, float, MODE>(c, D, x, y, u, poly, pc);
  }
}
VsDev fine_dev(const nsb_ctx* c);

// y(owned) = A x ; x must have a valid ghost tail
void spmv_full(nsb_ctx* c, const double* x, double* y) {
  size_t id = c->prof.begin(PC_SPMV, c->stream);
  if (c->dim == 2) k_spmv_full<2, double><<<c->n_stiles, SPMV_WARPS * 32, 0, c->stream>>>(c->M, c->stiles, c->vals.p, x, y);
  else k_spmv_full<3, double><<<c->n_stiles, SPMV_WARPS * 32, 0, c->stream>>>(c->M, c->stiles, c->vals.p, x, y);
  c->launch_check();
  c->prof.end(id, c->stream);
}

template <int MODE>
void spmv_vel(nsb_ctx* c, const double* x, double* y, const double* u, double* poly, PolyCoef pc) {
  size_t id = c->prof.begin(PC_SPMV_VEL, c->stream);
  const int g = c->n_stiles;
  if (c->vs_valid && MODE != 0) {
    vel_stream<MODE == 0 ? 2 : MODE>(c, fine_dev(c), x, y, u, poly, pc);
  } else {
    if (c->dim == 2) k_spmv_vel<2, MODE, double><<<g, SPMV_WARPS * 32, 0, c->stream>>>(c->M, c->stiles, c->vals.p, x, y, u, poly, c->dinv.p, pc);
    else k_spmv_vel<3, MODE, double><<<g, SPMV_WARPS * 32, 0, c->stream>>>(c->M, c->stiles, c->vals.p, x, y, u, poly, c->dinv.p, pc);
    c->launch_check();
  }
  c->prof.end(id, c->stream);
}

void block_scale(nsb_ctx* c, const double* x, double* y) {
  if (c->dim == 2) k_block_scale<2><<<nblk(c->S.nn_own, 256), 256, 0, c->stream>>>(c->S.nn_own, c->dinv.p, x, y);
  else k_block_scale<3><<<nblk(c->S.nn_own, 256), 256, 0, c->stream>>>(c->S.nn_own, c->dinv.p, x, y);
  c->launch_check();
}

double device_norm2(nsb_ctx* c, const double* x, long long n) {
  const int nb = nblk(n, RED_CHUNK);
  k_norm2_partial<<<nb, RED_THREADS, 0, c->stream>>>(x, n, c->partial.p);
  c->launch_check();
  k_reduce_partials<<<1, RED_THREADS, 0, c->stream>>>(nb, c->partial.p, c->d_nrm.p, 0);
  c->launch_check();
  allreduce_sum(c, c->d_nrm.p, 1);
  double v = 0;
  CK(cudaMemcpyAsync(&v, c->d_nrm.p, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return std::sqrt(v);
}

// ---- Chebyshev coefficients ------------------------------------------------------------
struct Cheb {
  double theta, delta, sigma, rho;
  Cheb(double lmax, double lmin) : theta(0.5 * (lmax + lmin)), delta(0.5 * (lmax - lmin)) {
    sigma = theta / delta;
    rho = 1.0 / sigma;
  }
  // returns (c1, c2) of  d <- c1 d + c2 Dinv r  for step k >= 1 and advances rho
  void next(double& c1, double& c2) {
    const double rho_new = 1.0 / (2.0 * sigma - rho);
    c1 = rho_new * rho;
    c2 = 2.0 * rho_new / delta;
    rho = rho_new;
  }
};

// ---- velocity-block preconditioner ---------------------------------------------------------
// Everything here works on B = Dinv F, the node-block-Jacobi scaled velocity block, on one of two levels: the fine (P2)
// level and, for linearised systems, the coarse P1 level of the two-level cycle (twolevel.cuh).  A level's operator is applied
// by the streamed kernel (velstream.cuh) -- the fine level falls back to the generic fp64 row kernel when no packed copy
// is kept.  Polynomials are FIXED linear operators between rebuilds, so the outer iteration stays plain (non-flexible)
// left-preconditioned GMRES like the reference's.

VsDev fine_dev(const nsb_ctx* c) {
  return VsDev{c->d_vs_tiles.p, c->d_vs_meta.p, c->d_suniq_xoff.p, c->vs_vals.p, c->n_stiles};
}
VsDev coarse_dev(const nsb_ctx* c) {
  return VsDev{c->cg.tiles.p, c->cg.meta.p, c->cg.uniq_xoff.p, c->cg.vals.p, c->cg.n_tiles};
}

// halo of a coarse vector (layout [dim*np_own | dim*np_ghost]): the pressure halo plan with dim components per vertex
void halo_exchange_coarse(nsb_ctx* c, double* v) {
  if (c->nranks == 1) return;
  const Structure& S = c->S;
  if (c->ph.on) {
    peer_exchange(c, v, (int)S.peer.size(), c->ph.seg_ptr_c, c->ph.src_c, c->ph.land_c, c->ph.total_c);
    return;
  }
  Coarse& G = c->cg;
  const int dim = c->dim;
  const long long tp = (long long)G.send_xoff.n;
  if (tp) { k_gather_nodes<<<nblk(tp * dim, 256), 256, 0, c->stream>>>((int)tp, dim, G.send_xoff.p, v, G.send_buf.p); c->launch_check(); }
  CKN(g_nccl.GroupStart());
  long long roff = (long long)dim * S.np_own;
  size_t so = 0;
  for (size_t k = 0; k < S.peer.size(); ++k) {
    const int peer = S.peer[k];
    const size_t ns = S.send_pids[k].size() * dim, nr = (size_t)S.recv_pid_count[k] * dim;
    if (ns) CKN(g_nccl.Send(G.send_buf.p + so, ns, ncclDouble, peer, c->comm, c->stream));
    if (nr) CKN(g_nccl.Recv(v + roff, nr, ncclDouble, peer, c->comm, c->stream));
    so += ns; roff += nr;
  }
  CKN(g_nccl.GroupEnd());
}

void level_halo(nsb_ctx* c, PolyLevel& lv, double* v) {
  if (lv.coarse) halo_exchange_coarse(c, v);
  else halo_exchange(c, v, false);
}

// y = op(B x) with the fused epilogue MODE (2, 3 or 4); x must have valid ghosts
template <int MODE>
void level_apply(nsb_ctx* c, PolyLevel& lv, const double* x, double* y, const double* u, double* poly, PolyCoef pc) {
  if (!lv.coarse) { spmv_vel<MODE>(c, x, y, u, poly, pc); return; }
  size_t id = c->prof.begin(PC_COARSE, c->stream);
  vel_stream<MODE>(c, coarse_dev(c), x, y, u, poly, pc);
  c->prof.end(id, c->stream);
}

// one root of a product-form polynomial on a vector whose ghosts are stale
void level_root(nsb_ctx* c, PolyLevel& lv, double* x, double* y, const double* u, double* poly, PolyCoef pc) {
  level_halo(c, lv, x);
  level_apply<3>(c, lv, x, y, u, poly, pc);
}

void level_block_scale(nsb_ctx* c, PolyLevel& lv, const double* x, double* y) {
  if (c->dim == 2) k_block_scale<2><<<nblk(lv.nn, 256), 256, 0, c->stream>>>(lv.nn, lv.dinv, x, y);
  else k_block_scale<3><<<nblk(lv.nn, 256), 256, 0, c->stream>>>(lv.nn, lv.dinv, x, y);
  c->launch_check();
}

// d Arnoldi steps on B from a fixed pseudo-random probe (a hash of the GLOBAL DoF index, so everything derived from it is
// partition-independent); stops early once the GMRES residual of the probe drops below `target` (target <= 0: never).
// Leaves the harmonic Ritz values in lv.wr / lv.wi and the probe's residual reduction in lv.probe_res.
void level_arnoldi(nsb_ctx* c, PolyLevel& lv, int dmax, double target) {
  const long long nl = lv.n;
  const long long ld = c->S.n_own_dofs();          // stride of the Krylov basis (shared with GMRES, always >= nl)
  int d = std::max(1, std::min(dmax, 64));
  if (c->V_cap < d + 1) { c->V.alloc((size_t)(std::max(d + 1, c->V_cap)) * ld); c->V_cap = std::max(d + 1, c->V_cap); }
  const int nb = nblk(nl, RED_CHUNK);
  if (c->partial.n < (size_t)nb * (d + 2)) c->partial.alloc((size_t)nb * (d + 2));
  if (c->d_h.n < (size_t)2 * (d + 2)) c->d_h.alloc(2 * (d + 2));
  if (!lv.probe_init) {
    std::vector<double> h(nl);
    for (int A = 0; A < lv.nn; ++A)
      for (int k = 0; k < c->dim; ++k) {
        uint64_t z = (uint64_t)(lv.gid[A] * c->dim + k) + 0x9E3779B97F4A7C15ull;
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        z ^= z >> 31;
        h[(size_t)c->dim * A + k] = (double)(z >> 11) / 9007199254740992.0 - 0.5;
      }
    lv.probe.upload(h, c->stream);
    CK(cudaStreamSynchronize(c->stream));
    lv.probe_init = true;
  }
  const int ldh = d;
  std::vector<double> H((size_t)(d + 1) * d, 0.0), hh(2 * (d + 2)), gcs(d + 1), gsn(d + 1);
  double gres = 1.0;
  double beta = device_norm2(c, lv.probe.p, nl);
  k_axpby<<<nblk(nl, 256), 256, 0, c->stream>>>(nl, 1.0 / beta, lv.probe.p, 0.0, c->V.p);
  c->launch_check();
  int dd = d;
  for (int k = 0; k < d; ++k) {
    double* vk = c->V.p + (size_t)k * ld;
    double* w = c->V.p + (size_t)(k + 1) * ld;
    const double* xin = vk;
    if (c->nranks > 1) {
      double* buf = (k & 1) ? lv.z1 : lv.pin;       // never the same buffer twice in a row (peer-store halo)
      CK(cudaMemcpyAsync(buf, vk, nl * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
      level_halo(c, lv, buf);
      xin = buf;
    }
    level_apply<2>(c, lv, xin, w, nullptr, nullptr, PolyCoef{});
    for (int pass = 0; pass < 2; ++pass) {
      k_multi_dot<<<nb, RED_THREADS, 0, c->stream>>>(k + 1, c->V.p, ld, w, nl, c->partial.p);
      c->launch_check();
      double* hp = c->d_h.p + pass * (d + 2);
      k_reduce_partials<<<k + 1, RED_THREADS, 0, c->stream>>>(nb, c->partial.p, hp, 0);
      c->launch_check();
      allreduce_sum(c, hp, k + 1);
      k_multi_axpy<<<nb, RED_THREADS, 0, c->stream>>>(k + 1, c->V.p, ld, hp, -1.0, w, nl, pass == 1 ? c->partial.p : nullptr);
      c->launch_check();
    }
    k_reduce_partials<<<1, RED_THREADS, 0, c->stream>>>(nb, c->partial.p, c->d_nrm.p, 0);
    c->launch_check();
    allreduce_sum(c, c->d_nrm.p, 1);
    k_scale_by_inv_norm<<<nblk(nl, 256), 256, 0, c->stream>>>(nl, w, c->d_nrm.p, w);
    c->launch_check();
    double nrm2 = 0;
    CK(cudaMemcpyAsync(hh.data(), c->d_h.p, sizeof(double) * 2 * (d + 2), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(&nrm2, c->d_nrm.p, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    for (int i = 0; i <= k; ++i) H[(size_t)i * ldh + k] = hh[i] + hh[(d + 2) + i];
    H[(size_t)(k + 1) * ldh + k] = std::sqrt(nrm2);
    if (!(nrm2 > 1e-28)) { dd = k + 1; break; }
    // GMRES residual of the probe vector after k+1 steps (Givens on a copy of column k)
    {
      std::vector<double> col(k + 2);
      for (int i = 0; i <= k + 1; ++i) col[i] = H[(size_t)i * ldh + k];
      for (int i = 0; i < k; ++i) {
        const double t = gcs[i] * col[i] + gsn[i] * col[i + 1];
        col[i + 1] = -gsn[i] * col[i] + gcs[i] * col[i + 1];
        col[i] = t;
      }
      const double r = std::hypot(col[k], col[k + 1]);
      gcs[k] = col[k] / r; gsn[k] = col[k + 1] / r;
      gres *= std::fabs(gsn[k]);
      if (target > 0 && gres <= target && k + 1 >= 2) { dd = k + 1; break; }
    }
  }
  lv.probe_res = gres;
  // harmonic Ritz values: eig(Hd + h_{d+1,d}^2 f e_d^T),  Hd^T f = e_d
  d = dd;
  std::vector<double> Hd((size_t)d * d), At((size_t)d * d), f(d, 0.0);
  for (int i = 0; i < d; ++i)
    for (int j = 0; j < d; ++j) { Hd[(size_t)i * d + j] = H[(size_t)i * ldh + j]; At[(size_t)j * d + i] = H[(size_t)i * ldh + j]; }
  f[d - 1] = 1.0;
  {  // Gaussian elimination with partial pivoting on At f = e_d
    for (int col = 0; col < d; ++col) {
      int p = col;
      for (int r = col + 1; r < d; ++r) if (std::fabs(At[(size_t)r * d + col]) > std::fabs(At[(size_t)p * d + col])) p = r;
      if (p != col) { for (int k = 0; k < d; ++k) std::swap(At[(size_t)col * d + k], At[(size_t)p * d + k]); std::swap(f[col], f[p]); }
      const double dg = At[(size_t)col * d + col];
      for (int r = col + 1; r < d; ++r) {
        const double m = At[(size_t)r * d + col] / dg;
        if (m == 0.0) continue;
        for (int k = col; k < d; ++k) At[(size_t)r * d + k] -= m * At[(size_t)col * d + k];
        f[r] -= m * f[col];
      }
    }
    for (int r = d - 1; r >= 0; --r) {
      double sum = f[r];
      for (int k = r + 1; k < d; ++k) sum -= At[(size_t)r * d + k] * f[k];
      f[r] = sum / At[(size_t)r * d + r];
    }
  }
  const double hl = H[(size_t)d * ldh + (d - 1)];
  for (int i = 0; i < d; ++i) Hd[(size_t)i * d + (d - 1)] += hl * hl * f[i];
  // standard Ritz values (eigenvalues of H_d itself): they approach the outer end of the spectrum faster than the
  // harmonic ones, which is what the smoother's upper bound needs
  std::vector<double> H0((size_t)d * d), sr, si;
  for (int i = 0; i < d; ++i)
    for (int j = 0; j < d; ++j) H0[(size_t)i * d + j] = H[(size_t)i * ldh + j];
  if (!hessenberg_eigs(d, Hd, lv.wr, lv.wi)) throw CudaErr{"harmonic Ritz eigenvalue iteration did not converge"};
  if (!hessenberg_eigs(d, H0, sr, si)) throw CudaErr{"Ritz eigenvalue iteration did not converge"};
  lv.ritz_lo = 1e300; lv.ritz_hi = -1e300; lv.ritz_im = 0; lv.ritz_top = -1e300;
  for (int i = 0; i < d; ++i) {
    lv.ritz_lo = std::min(lv.ritz_lo, lv.wr[i]); lv.ritz_hi = std::max(lv.ritz_hi, lv.wr[i]);
    lv.ritz_im = std::max(lv.ritz_im, std::fabs(lv.wi[i]));
    lv.ritz_top = std::max(lv.ritz_top, std::hypot(sr[i], si[i]));
  }
  lv.ritz_top = std::max(lv.ritz_top, lv.ritz_hi);
}

bool level_spectrum_is_real(const PolyLevel& lv, double tol = 0.05) { return lv.ritz_lo > 0 && lv.ritz_im < tol * lv.ritz_hi; }

// roots of the degree-d Chebyshev polynomial on [lo, hi], Leja ordered
void set_roots(PolyLevel& lv, std::vector<double> wr, std::vector<double> wi) {
  const int d = (int)wr.size();
  std::vector<std::pair<double, double>> th, out;
  for (int i = 0; i < d; ++i) if (wi[i] >= 0) th.emplace_back(wr[i], wi[i]);
  auto mag = [](const std::pair<double, double>& z) { return std::hypot(z.first, z.second); };
  // Leja ordering, complex conjugates kept adjacent (positive imaginary part first)
  while (!th.empty()) {
    size_t best = 0;
    double bv = -1e300;
    for (size_t i = 0; i < th.size(); ++i) {
      double v;
      if (out.empty()) v = mag(th[i]);
      else {
        v = 0;
        for (auto& o : out) {
          v += std::log(std::hypot(th[i].first - o.first, th[i].second - o.second) + 1e-300);
          if (o.second != 0) v += std::log(std::hypot(th[i].first - o.first, th[i].second + o.second) + 1e-300);
        }
      }
      if (v > bv) { bv = v; best = i; }
    }
    out.push_back(th[best]);
    th.erase(th.begin() + best);
  }
  lv.roots = out;
}
void set_chebyshev_roots(PolyLevel& lv, int d, double lo, double hi) {
  std::vector<double> wr(d), wi(d, 0.0);
  for (int j = 1; j <= d; ++j) wr[j - 1] = 0.5 * (hi + lo) + 0.5 * (hi - lo) * std::cos(M_PI * (2 * j - 1) / (2.0 * d));
  set_roots(lv, wr, wi);
}

// poly = p(B) z0 with p ~ B^-1 given by lv.roots in product form (Leja ordered, real arithmetic for conjugate pairs);
// lv.z0 holds the (already Dinv-scaled) right-hand side and is destroyed; every root but the last is one fused operator
// application.
void apply_poly(nsb_ctx* c, PolyLevel& lv) {
  double* prod = lv.z0;
  double* other = lv.z1;
  double* tmp = lv.zd;
  double* poly = lv.poly;
  CK(cudaMemsetAsync(poly, 0, lv.n * sizeof(double), c->stream));
  const auto& R = lv.roots;
  for (size_t k = 0; k < R.size(); ++k) {
    const bool last = (k + 1 == R.size());
    const double a = R[k].first, b = R[k].second;
    if (b == 0.0) {
      if (last) {
        k_axpby<<<nblk(lv.n, 256), 256, 0, c->stream>>>(lv.n, 1.0 / a, prod, 1.0, poly);
        c->launch_check();
      } else {
        // poly += prod/theta ; prod <- prod - B prod / theta
        level_root(c, lv, prod, other, prod, poly, PolyCoef{1.0, -1.0 / a, 1.0 / a, 0.0});
        std::swap(prod, other);
      }
    } else {
      const double m2 = a * a + b * b;
      // tmp = 2a prod - B prod ; poly += tmp/m2 ; prod <- prod - B tmp / m2
      level_root(c, lv, prod, tmp, prod, poly, PolyCoef{2.0 * a, -1.0, 0.0, 1.0 / m2});
      if (!last) {
        level_root(c, lv, tmp, other, prod, poly, PolyCoef{1.0, -1.0 / m2, 0.0, 0.0});
        std::swap(prod, other);
      }
    }
  }
}

template <int DIM> void launch_coarse_assemble(nsb_ctx* c) {
  Coarse& G = c->cg;
  FeTables T;
  fill_tables(DIM, T);
  double wsum = 0;
  for (int q = 0; q < T.nq; ++q) wsum += T.w[q];
  const double gamma = c->par.use_supg ? c->par.gamma : 0.0;
  size_t id = c->prof.begin(PC_ASM_COARSE, c->stream);
  k_coarse_rows<DIM><<<nblk(c->S.np_own, CG_WARPS), CG_WARPS * 32, 0, c->stream>>>(c->M, c->ctx.p, gamma, wsum, G.nbr_ptr.p, G.nbr_vxoff.p,
                                                                                     c->cflag.p, G.cvals.p, G.dinv.p);
  c->launch_check();
  if (c->opt.precond_precision == 16)
    k_coarse_pack<DIM, __half><<<G.n_tiles, 256, 0, c->stream>>>(G.tiles.p, G.meta.p, G.nbr_ptr.p, G.cvals.p, G.dinv.p, reinterpret_cast<__half*>(G.vals.p));
  else
    k_coarse_pack<DIM, float><<<G.n_tiles, 256, 0, c->stream>>>(G.tiles.p, G.meta.p, G.nbr_ptr.p, G.cvals.p, G.dinv.p, reinterpret_cast<float*>(G.vals.p));
  c->launch_check();
  c->prof.end(id, c->stream);
  G.valid = true;
}

// Rebuilds the velocity preconditioner for the currently assembled system (once per solve, or every poly_refresh-th).
void setup_velocity_pc(nsb_ctx* c) {
  PolyLevel& F = c->lvF;
  bool two = c->opt.velocity_cycle != 1 && c->cg.valid && c->vs_valid && !c->cycle_disabled;
  if (two) {
    // fine level: the upper end of the spectrum of B for the smoother, and enough Arnoldi steps to see whether the
    // spectrum leaves the real axis (convection-dominated 2-D flows: the Chebyshev smoother would amplify those modes)
    level_arnoldi(c, F, 24, 0.0);
    two = level_spectrum_is_real(F, 0.02);
  }
  c->two_level = two;
  if (!two) {
    // single level: polynomial of the degree that reduces the probe's residual below poly_target.  Real spectrum
    // (grad-div dominated 3-D case): Chebyshev roots on the interval spanned by the harmonic Ritz values (minimax
    // instead of probe-optimal); otherwise (convection-dominated 2-D case, Im up to 2) the harmonic Ritz values
    // themselves -- the GMRES polynomial of Loe & Morgan -- where Chebyshev on a real interval diverges.
    level_arnoldi(c, F, c->opt.poly_degree_F, c->opt.poly_target);
    if (c->opt.poly_kind == 1 && level_spectrum_is_real(F)) set_chebyshev_roots(F, (int)F.wr.size(), 0.9 * F.ritz_lo, 1.05 * F.ritz_hi);
    else set_roots(F, F.wr, F.wi);
    return;
  }
  const double hi = c->opt.smoother_hi_factor * F.ritz_top;
  set_chebyshev_roots(F, std::max(1, c->opt.smoother_degree), c->opt.smoother_lo_frac * hi, hi);
  PolyLevel& C = c->lvC;
  level_arnoldi(c, C, std::max(4, std::min(64, c->opt.coarse_degree + 5)), 0.05);
  if (level_spectrum_is_real(C)) set_chebyshev_roots(C, std::max(1, c->opt.coarse_degree), 0.9 * C.ritz_lo, c->opt.smoother_hi_factor * C.ritz_top);
  else set_roots(C, C.wr, C.wi);
}

// y_u ~ F^-1 x_u ; result left in c->w_poly
void apply_velocity_pc(nsb_ctx* c, const double* x) {
  PolyLevel& F = c->lvF;
  const long long nu = F.n;
  if (!c->two_level) {
    level_block_scale(c, F, x, F.z0);
    apply_poly(c, F);
    return;
  }
  // ---- coarse correction  y0 = P p_c(B_c) Dinv_c P^T x
  PolyLevel& C = c->lvC;
  Coarse& G = c->cg;
  const double* xr = x;
  if (c->nranks > 1) {
    CK(cudaMemcpyAsync(c->w_u.p, x, nu * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));      // (w_u is rewritten below)
    halo_exchange(c, c->w_u.p, false);
    xr = c->w_u.p;
  }
  size_t id = c->prof.begin(PC_COARSE, c->stream);
  if (c->dim == 2) k_restrict<2><<<nblk(c->S.np_own, 128), 128, 0, c->stream>>>(c->S.np_own, c->M.pid_node, G.vedge_ptr.p, G.vedge_xoff.p, c->cflag.p, xr, G.rc.p);
  else k_restrict<3><<<nblk(c->S.np_own, 128), 128, 0, c->stream>>>(c->S.np_own, c->M.pid_node, G.vedge_ptr.p, G.vedge_xoff.p, c->cflag.p, xr, G.rc.p);
  c->launch_check();
  c->prof.end(id, c->stream);
  level_block_scale(c, C, G.rc.p, C.z0);
  apply_poly(c, C);
  halo_exchange_coarse(c, C.poly);
  double* y0 = c->w_y0.p;
  id = c->prof.begin(PC_COARSE, c->stream);
  if (c->dim == 2) k_prolong<2><<<nblk(nu, 256), 256, 0, c->stream>>>(c->S.nn_own, G.ends_xoff.p, c->cflag.p, C.poly, y0);
  else k_prolong<3><<<nblk(nu, 256), 256, 0, c->stream>>>(c->S.nn_own, G.ends_xoff.p, c->cflag.p, C.poly, y0);
  c->launch_check();
  c->prof.end(id, c->stream);
  // ---- smoothing from y0:  y = y0 + q(B) (Dinv x - B y0)
  level_block_scale(c, F, x, c->w_u.p);
  halo_exchange(c, y0, false);
  level_apply<4>(c, F, y0, F.z0, c->w_u.p, nullptr, PolyCoef{1.0, -1.0, 0.0, 0.0});
  apply_poly(c, F);
  k_axpby<<<nblk(nu, 256), 256, 0, c->stream>>>(nu, 1.0, y0, 1.0, F.poly);
  c->launch_check();
}

// ---- pressure-space pieces (global, replicated vectors of length n_p) -------------------
void csr_cheb(nsb_ctx* c, const DevCsr& A, const double* dinv, double lmax, double ratio, int degree,
              const double* b, double* x, double* x2, double* d, bool zero_guess, double** result) {
  // Jacobi-Chebyshev on A e = b (zero_guess) or continuing from x.  Ping-pongs x/x2.
  Cheb ch(1.1 * lmax, 1.1 * lmax / ratio);
  double* cur = x;
  double* oth = x2;
  int k0 = 0;
  const int g8 = nblk((long long)A.n * 8, 256);
  if (zero_guess) {
    k_cheb_first<<<nblk(A.n, 256), 256, 0, c->stream>>>(A.n, dinv, b, d, cur, 1.0 / ch.theta);
    c->launch_check();
    k0 = 1;
  }
  for (int k = k0; k < degree; ++k) {
    double c1, c2;
    if (k == 0) { c1 = 0.0; c2 = 1.0 / ch.theta; }
    else ch.next(c1, c2);
    k_csr<3><<<g8, 256, 0, c->stream>>>(A, cur, oth, b, d, dinv, c1, c2);
    c->launch_check();
    std::swap(cur, oth);
  }
  *result = cur;
}

void amg_vcycle(nsb_ctx* c, int lev) {
  // solves A_lev x = b_lev approximately; input levels[lev]->b, output pointer in levels[lev]->x (may swap with x2)
  DevLevel& L = *c->amg[lev];
  const int deg = c->opt.amg_smoother_degree;
  if (lev + 1 == (int)c->amg.size()) {
    if (c->coarse_n > 0) {
      k_dense_mv<<<nblk((long long)L.n * 32, 256), 256, 0, c->stream>>>(L.n, c->coarse_inv.p, L.b.p, L.x.p);
      c->launch_check();
    } else {
      double* res;
      csr_cheb(c, L.A, L.dinv.p, L.lmax, 30.0, 12, L.b.p, L.x.p, L.x2.p, L.d.p, true, &res);
      if (res != L.x.p) std::swap(L.x.p, L.x2.p);
    }
    return;
  }
  double* res;
  csr_cheb(c, L.A, L.dinv.p, L.lmax, 20.0, deg, L.b.p, L.x.p, L.x2.p, L.d.p, true, &res);
  if (res != L.x.p) std::swap(L.x.p, L.x2.p);
  const int g8 = nblk((long long)L.n * 8, 256);
  k_csr<1><<<g8, 256, 0, c->stream>>>(L.A, L.x.p, L.r.p, L.b.p, nullptr, nullptr, 0, 0);
  c->launch_check();
  DevLevel& N = *c->amg[lev + 1];
  k_csr<0><<<nblk((long long)N.n * 8, 256), 256, 0, c->stream>>>(L.R, L.r.p, N.b.p, nullptr, nullptr, nullptr, 0, 0);
  c->launch_check();
  amg_vcycle(c, lev + 1);
  k_csr<2><<<g8, 256, 0, c->stream>>>(L.P, N.x.p, L.x.p, nullptr, nullptr, nullptr, 0, 0);
  c->launch_check();
  csr_cheb(c, L.A, L.dinv.p, L.lmax, 20.0, deg, L.b.p, L.x.p, L.x2.p, L.d.p, false, &res);
  if (res != L.x.p) std::swap(L.x.p, L.x2.p);
}

// ---- the block-triangular preconditioner (reference NavierStokes.hpp:320-344) -----------
//   y0 = F~^-1 x0 ;  t = x1 - B y0 ;  y1 = -(rho/dt) Kp~^-1 t - cm Mp~^-1 t
double schur_mass_coeff(const nsb_ctx* c) {
  const double cm = c->opt.schur_mass_coeff;
  return cm >= 0 ? cm : c->par.theta * c->par.nu + (c->par.use_supg ? c->par.gamma : 0.0);
}

void precond_apply(nsb_ctx* c, const double* x, double* y) {
  const Structure& S = c->S;
  const int dim = c->dim;
  const long long nu = (long long)dim * S.nn_own;
  // --- step 1: y0 = F~^-1 x0 (two-level cycle or polynomial)
  apply_velocity_pc(c, x);
  double* z = c->w_poly.p;
  CK(cudaMemcpyAsync(y, z, nu * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
  // --- step 2: t = x1 - B y0
  halo_exchange(c, z);
  size_t id = c->prof.begin(PC_SCHUR, c->stream);
  if (dim == 2) k_schur_rhs<2, double><<<nblk(S.np_own, SPMV_WARPS), SPMV_WARPS * 32, 0, c->stream>>>(c->M, c->vals.p, z, x, c->w_t.p);
  else k_schur_rhs<3, double><<<nblk(S.np_own, SPMV_WARPS), SPMV_WARPS * 32, 0, c->stream>>>(c->M, c->vals.p, z, x, c->w_t.p);
  c->launch_check();
  c->prof.end(id, c->stream);
  // --- step 3: Cahouet-Chabard Schur complement on the (replicated) pressure space
  const double* tg = c->w_t.p;     // one rank: local pressure ids == global ids
  if (c->nranks > 1) {
    // replicate the pressure-space vector: zero-padded all-reduce of the owned entries (exact: one
    // non-zero summand per entry), so every GPU applies the same global multigrid cycle
    CK(cudaMemsetAsync(c->w_tg.p, 0, (size_t)c->n_p * sizeof(double), c->stream));
    k_scatter_vals<<<nblk(S.np_own, 256), 256, 0, c->stream>>>(S.np_own, c->d_pid_gid.p, c->w_t.p, c->w_tg.p);
    c->launch_check();
    allreduce_sum(c, c->w_tg.p, (int)c->n_p);
    tg = c->w_tg.p;
  }
  id = c->prof.begin(PC_AMG, c->stream);
  DevLevel& L0 = *c->amg[0];
  CK(cudaMemcpyAsync(L0.b.p, tg, (size_t)L0.n * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
  amg_vcycle(c, 0);
  double* mres;
  csr_cheb(c, c->Mp, c->Mp_dinv.p, c->Mp_lmax, 6.0, c->opt.cheb_degree_Mp, tg, c->w_m0.p, c->w_m1.p, c->w_md.p, true, &mres);
  const double cm = schur_mass_coeff(c);
  if (c->nranks > 1)
    k_lincomb_gather<<<nblk(S.np_own, 256), 256, 0, c->stream>>>(S.np_own, c->d_pid_gid.p, -(c->par.rho / c->par.dt), L0.x.p, -cm, mres, y + nu);
  else
    k_lincomb<<<nblk(S.np_own, 256), 256, 0, c->stream>>>(S.np_own, -(c->par.rho / c->par.dt), L0.x.p, -cm, mres, y + nu);
  c->launch_check();
  c->prof.end(id, c->stream);
}

// ---- GMRES (SolverGMRES semantics, SURVEY.md A.6) ---------------------------------------
int gmres(nsb_ctx* c, int max_it, double tol_abs, int n_tmp, int* iterations, double* residual) {
  const Structure& S = c->S;
  const long long n = S.n_own_dofs();
  const int m = std::max(1, n_tmp - 2);
  if (c->V_cap < m + 1) {
    c->V.alloc((size_t)(m + 1) * n);
    c->V_cap = m + 1;
  }
  const int nb = nblk(n, RED_CHUNK);
  if (c->partial.n < (size_t)nb * (m + 2)) c->partial.alloc((size_t)nb * (m + 2));
  if (c->d_h.n < (size_t)2 * (m + 2)) c->d_h.alloc(2 * (m + 2));
  double* x = c->v_sol.p;
  CK(cudaMemsetAsync(x, 0, S.n_tot_dofs() * sizeof(double), c->stream));
  std::vector<double> H((size_t)(m + 1) * m, 0.0), cs(m), sn(m), g(m + 1), hcol(2 * (m + 2));
  int it = 0;
  double res = 0;
  bool first = true;
  for (;;) {
    double* V0 = c->V.p;
    if (first) {
      precond_apply(c, c->v_rhs.p, c->w_in.p);
    } else {
      halo_exchange(c, x);
      spmv_full(c, x, c->w_tmp.p);
      k_lincomb<<<nblk(n, 256), 256, 0, c->stream>>>(n, 1.0, c->v_rhs.p, -1.0, c->w_tmp.p, c->w_tmp.p);
      c->launch_check();
      precond_apply(c, c->w_tmp.p, c->w_in.p);
    }
    const double beta = device_norm2(c, c->w_in.p, n);
    res = beta;
    if (first && beta <= tol_abs) { *iterations = 0; *residual = beta; return 0; }
    first = false;
    if (!(beta > 0)) { *iterations = it; *residual = beta; return 0; }
    k_axpby<<<nblk(n, 256), 256, 0, c->stream>>>(n, 1.0 / beta, c->w_in.p, 0.0, V0);
    c->launch_check();
    std::fill(g.begin(), g.end(), 0.0);
    g[0] = beta;
    int kused = 0;
    bool converged = false;
    for (int k = 0; k < m; ++k) {
      double* vk = c->V.p + (size_t)k * n;
      double* w = c->V.p + (size_t)(k + 1) * n;
      // w = P^-1 A v_k
      const double* xin = vk;
      if (c->nranks > 1) {
        CK(cudaMemcpyAsync(c->w_pin.p, vk, n * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
        halo_exchange(c, c->w_pin.p);
        xin = c->w_pin.p;
      }
      spmv_full(c, xin, c->w_tmp.p);
      precond_apply(c, c->w_tmp.p, w);
      // classical Gram-Schmidt, h = V^T w ; w -= V h, with a second pass when the first one cancelled more than half of w
      // (the DGKS criterion; reorthogonalize = 2 forces the second pass always, < 0 never).  The first dot pass also
      // returns ||w||^2: w is stored right behind the basis, so it is simply the (k+2)-th vector.
      size_t id = c->prof.begin(PC_ORTH, c->stream);
      const int mode = c->opt.reorthogonalize;
      int passes = 1;
      double nrm2 = 0, nrm2_before = 0;
      for (int pass = 0; pass < 2; ++pass) {
        const int nv = k + 1 + (pass == 0 ? 1 : 0);
        k_multi_dot<<<nb, RED_THREADS, 0, c->stream>>>(nv, c->V.p, n, w, n, c->partial.p);
        c->launch_check();
        double* hp = c->d_h.p + pass * (m + 2);
        k_reduce_partials<<<nv, RED_THREADS, 0, c->stream>>>(nb, c->partial.p, hp, 0);
        c->launch_check();
        allreduce_sum(c, hp, nv);
        k_multi_axpy<<<nb, RED_THREADS, 0, c->stream>>>(k + 1, c->V.p, n, hp, -1.0, w, n, c->partial.p);
        c->launch_check();
        k_reduce_partials<<<1, RED_THREADS, 0, c->stream>>>(nb, c->partial.p, c->d_nrm.p, 0);
        c->launch_check();
        allreduce_sum(c, c->d_nrm.p, 1);
        passes = pass + 1;
        if (pass == 1 || mode < 0) break;
        if (mode != 2) {
          CK(cudaMemcpyAsync(&nrm2_before, hp + k + 1, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
          CK(cudaMemcpyAsync(&nrm2, c->d_nrm.p, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
          CK(cudaStreamSynchronize(c->stream));
          if (nrm2 > 0.5 * nrm2_before) break;
        }
      }
      k_scale_by_inv_norm<<<nblk(n, 256), 256, 0, c->stream>>>(n, w, c->d_nrm.p, w);
      c->launch_check();
      c->prof.end(id, c->stream);
      CK(cudaMemcpyAsync(hcol.data(), c->d_h.p, sizeof(double) * 2 * (m + 2), cudaMemcpyDeviceToHost, c->stream));
      CK(cudaMemcpyAsync(&nrm2, c->d_nrm.p, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
      CK(cudaStreamSynchronize(c->stream));
      for (int i = 0; i <= k; ++i) H[(size_t)i * m + k] = hcol[i] + (passes == 2 ? hcol[(m + 2) + i] : 0.0);
      H[(size_t)(k + 1) * m + k] = std::sqrt(nrm2);
      // Givens
      for (int i = 0; i < k; ++i) {
        const double t = cs[i] * H[(size_t)i * m + k] + sn[i] * H[(size_t)(i + 1) * m + k];
        H[(size_t)(i + 1) * m + k] = -sn[i] * H[(size_t)i * m + k] + cs[i] * H[(size_t)(i + 1) * m + k];
        H[(size_t)i * m + k] = t;
      }
      const double a = H[(size_t)k * m + k], b = H[(size_t)(k + 1) * m + k];
      const double dd = std::hypot(a, b);
      cs[k] = a / dd; sn[k] = b / dd;
      H[(size_t)k * m + k] = dd;
      H[(size_t)(k + 1) * m + k] = 0.0;
      g[k + 1] = -sn[k] * g[k];
      g[k] = cs[k] * g[k];
      res = std::fabs(g[k + 1]);
      ++it;
      kused = k + 1;
      if (res <= tol_abs) { converged = true; break; }
      if (it >= max_it) break;
      if (!(nrm2 > 0)) break;       // lucky breakdown
    }
    // x += V y
    std::vector<double> yv(kused);
    for (int i = kused - 1; i >= 0; --i) {
      double s = g[i];
      for (int j = i + 1; j < kused; ++j) s -= H[(size_t)i * m + j] * yv[j];
      yv[i] = s / H[(size_t)i * m + i];
    }
    CK(cudaMemcpyAsync(c->d_h.p, yv.data(), sizeof(double) * kused, cudaMemcpyHostToDevice, c->stream));
    k_multi_axpy<<<nb, RED_THREADS, 0, c->stream>>>(kused, c->V.p, n, c->d_h.p, 1.0, x, n, nullptr);
    c->launch_check();
    CK(cudaStreamSynchronize(c->stream));
    if (converged || it >= max_it) {
      *iterations = it;
      *residual = res;
      return converged ? 0 : 1;
    }
  }
}

void build_tiles(nsb_ctx* c) {
  const Structure& S = c->S;
  int dev_max = 0;
  CK(cudaDeviceGetAttribute(&dev_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, c->device));
  const int stat = 24 * 1024;      // static shared memory of k_node_rows (upper bound: context staging + FE tables)
  int budget = std::max(S.max_node_smem_doubles, 5 * 1024);      // doubles: >= 40 KB
  if ((long long)budget * 8 + stat > dev_max)
    throw CudaErr{"a node's rows do not fit in shared memory (valence too high)"};
  std::vector<int> tp;
  tp.push_back(0);
  int sum = 0, cnt = 0;
  for (int A = 0; A < S.nn_own; ++A) {
    const int need = (S.dim + (S.node_pid[A] >= 0 ? 1 : 0)) * S.row_len(A);
    if (cnt > 0 && (sum + need > budget || cnt >= 64)) { tp.push_back(A); sum = 0; cnt = 0; }
    sum += need; ++cnt;
  }
  tp.push_back(S.nn_own);
  c->n_tiles = (int)tp.size() - 1;
  c->tile_smem_bytes = budget * 8;
  c->d_tile_ptr.upload(tp, c->stream);
  // SpMV tiles (plan built and checked on the host: structure.cpp build_tile_plan / verify_tile_plan) and the streamed
  // velocity operator's headers / metadata on top of them (build_vel_stream)
  {
    TilePlan P;
    const TileLimits L{TILE_MAX_NODES, TILE_MAX_IDX, TILE_MAX_UNIQ, TILE_MAX_PUNIQ, VS_MAX_BLOCKS};
    const std::string err = build_tile_plan(S, L, P);
    if (!err.empty()) throw CudaErr{err};
    VsPlan V;
    const std::string err2 = build_vel_stream(S, P, V);
    if (!err2.empty()) throw CudaErr{err2};
    c->n_stiles = P.n_tiles();
    c->d_stile_ptr.upload(P.node_ptr, c->stream);
    c->d_suniq_ptr.upload(P.uniq_ptr, c->stream); c->d_suniq_xoff.upload(P.uniq_xoff, c->stream);
    c->d_spuniq_ptr.upload(P.puniq_ptr, c->stream); c->d_spuniq_xoff.upload(P.puniq_xoff, c->stream);
    c->d_nbr_loc.upload(P.nbr_loc, c->stream); c->d_pnbr_loc.upload(P.pnbr_loc, c->stream);
    c->d_vs_tiles.upload(V.tiles, c->stream); c->d_vs_meta.upload(V.meta, c->stream);
    c->vs_total_nq = V.total_nq;
    CK(cudaStreamSynchronize(c->stream));       // the plans' host vectors die with this scope
    c->stiles.node_ptr = c->d_stile_ptr.p;
    c->stiles.uniq_ptr = c->d_suniq_ptr.p; c->stiles.uniq_xoff = c->d_suniq_xoff.p;
    c->stiles.puniq_ptr = c->d_spuniq_ptr.p; c->stiles.puniq_xoff = c->d_spuniq_xoff.p;
    c->stiles.nbr_loc = c->d_nbr_loc.p; c->stiles.pnbr_loc = c->d_pnbr_loc.p;
  }
  c->vs_vals.alloc(vs_vals_bytes(c));
  c->vs_valid = false;
  CK(cudaStreamSynchronize(c->stream));
  if (c->dim == 2) { set_smem_attr<2>(c->tile_smem_bytes); set_vs_attr<2, float>(); set_vs_attr<2, __half>(); }
  else { set_smem_attr<3>(c->tile_smem_bytes); set_vs_attr<3, float>(); set_vs_attr<3, __half>(); }
}

void close_peer_halo(nsb_ctx* c) {
  PeerHalo& H = c->ph;
  for (void* q : H.opened) cudaIpcCloseMemHandle(q);
  H.opened.clear(); H.peer_arena.clear(); H.peer_flags.clear();
  H.on = false;
}

void nccl_barrier(nsb_ctx* c) {
  if (c->nranks == 1 || !c->comm) return;
  CKN(g_nccl.AllReduce(c->d_nrm.p + 2, c->d_nrm.p + 2, 1, ncclDouble, ncclSum, c->comm, c->stream));
  CK(cudaStreamSynchronize(c->stream));
}

// All vectors that take part in halo exchanges as views into one symmetric arena (see PeerHalo); called from
// nsb_upload_mesh on several ranks, before the vectors are used.  `fine` / `coarse` = the buffers to place.
void setup_peer_halo(nsb_ctx* c, std::vector<DBuf<double>*> fine, std::vector<DBuf<double>*> coarse, size_t nt, size_t nct) {
  PeerHalo& H = c->ph;
  const Structure& S = c->S;
  const int R = c->nranks, dim = c->dim, np = (int)S.peer.size();
  cudaStream_t st = c->stream;
  close_peer_halo(c);
  nccl_barrier(c);                                   // nobody still maps the arena that is about to be freed
  // common strides
  long long hs[2] = {(long long)nt, (long long)nct};
  DBuf<long long> ds;
  ds.alloc(2);
  CK(cudaMemcpyAsync(ds.p, hs, sizeof(hs), cudaMemcpyHostToDevice, st));
  CKN(g_nccl.AllReduce(ds.p, ds.p, 2, ncclInt64, ncclMax, c->comm, st));
  CK(cudaMemcpyAsync(hs, ds.p, sizeof(hs), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  H.stride_f = ((size_t)hs[0] + 31) / 32 * 32;
  H.stride_c = ((size_t)hs[1] + 31) / 32 * 32;
  H.slots_f = (int)fine.size(); H.slots_c = (int)coarse.size();
  H.coarse_base = H.stride_f * H.slots_f;
  H.arena.alloc(H.coarse_base + H.stride_c * H.slots_c);
  H.arena.zero(st);
  for (size_t i = 0; i < fine.size(); ++i) fine[i]->view(H.arena.p + i * H.stride_f, nt);
  for (size_t i = 0; i < coarse.size(); ++i) coarse[i]->view(H.arena.p + H.coarse_base + i * H.stride_c, nct);
  H.flags.alloc(2 * (size_t)R); H.flags.zero(st);
  H.counter.alloc(1); H.counter.zero(st);
  H.seq = 0; H.last_vec = nullptr;
  const char* mode = std::getenv("NSB200_HALO");
  const bool want = !(mode && std::string(mode) == "nccl");
  // where each peer's data lands in MY vectors: [r][0] velocity, [r][1] pressure, [r][2] coarse; gathered so that every
  // sender can look up its landing offsets in the receivers' tables
  std::vector<long long> mine((size_t)R * 3, -1), all((size_t)R * R * 3, -1);
  {
    long long uoff = S.n_own_dofs(), poff = S.n_own_dofs() + (long long)dim * S.nn_ghost, coff = (long long)dim * S.np_own;
    for (int k = 0; k < np; ++k) {
      mine[(size_t)S.peer[k] * 3 + 0] = uoff; mine[(size_t)S.peer[k] * 3 + 1] = poff; mine[(size_t)S.peer[k] * 3 + 2] = coff;
      uoff += (long long)S.recv_node_count[k] * dim; poff += S.recv_pid_count[k]; coff += (long long)S.recv_pid_count[k] * dim;
    }
  }
  struct Handles { cudaIpcMemHandle_t arena, flags; };
  Handles hm;
  std::vector<Handles> hall(R);
  bool ok = want;
  if (ok) ok = cudaIpcGetMemHandle(&hm.arena, H.arena.p) == cudaSuccess && cudaIpcGetMemHandle(&hm.flags, H.flags.p) == cudaSuccess;
  if (!ok) { std::memset(&hm, 0, sizeof(hm)); cudaGetLastError(); }
  {
    DBuf<unsigned char> g0, g1;
    DBuf<long long> t0, t1;
    g0.alloc(sizeof(Handles) + 8); g1.alloc((sizeof(Handles) + 8) * R);
    t0.alloc(mine.size()); t1.alloc(all.size());
    unsigned char pack[sizeof(Handles) + 8] = {0};
    std::memcpy(pack, &hm, sizeof(hm));
    pack[sizeof(Handles)] = ok ? 1 : 0;
    CK(cudaMemcpyAsync(g0.p, pack, sizeof(pack), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(t0.p, mine.data(), mine.size() * sizeof(long long), cudaMemcpyHostToDevice, st));
    CKN(g_nccl.AllGather(g0.p, g1.p, sizeof(pack), ncclChar, c->comm, st));
    CKN(g_nccl.AllGather(t0.p, t1.p, mine.size(), ncclInt64, c->comm, st));
    std::vector<unsigned char> back((sizeof(Handles) + 8) * R);
    CK(cudaMemcpyAsync(back.data(), g1.p, back.size(), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(all.data(), t1.p, all.size() * sizeof(long long), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    for (int r = 0; r < R; ++r) {
      std::memcpy(&hall[r], back.data() + (sizeof(Handles) + 8) * r, sizeof(Handles));
      ok = ok && back[(sizeof(Handles) + 8) * r + sizeof(Handles)] == 1;      // every rank must be able to export
    }
  }
  if (ok) {
    for (int k = 0; k < np && ok; ++k) {
      void *pa = nullptr, *pf = nullptr;
      ok = cudaIpcOpenMemHandle(&pa, hall[S.peer[k]].arena, cudaIpcMemLazyEnablePeerAccess) == cudaSuccess;
      if (ok) { H.opened.push_back(pa); ok = cudaIpcOpenMemHandle(&pf, hall[S.peer[k]].flags, cudaIpcMemLazyEnablePeerAccess) == cudaSuccess; }
      if (ok) H.opened.push_back(pf);
      H.peer_arena.push_back((double*)pa); H.peer_flags.push_back((unsigned long long*)pf);
    }
    if (!ok) cudaGetLastError();
  }
  // the decision must be unanimous: one more reduction over "all my mappings opened"
  {
    DBuf<long long> d;
    d.alloc(1);
    long long v = ok ? 1 : 0;
    CK(cudaMemcpyAsync(d.p, &v, sizeof(v), cudaMemcpyHostToDevice, st));
    CKN(g_nccl.AllReduce(d.p, d.p, 1, ncclInt64, ncclMin, c->comm, st));
    CK(cudaMemcpyAsync(&v, d.p, sizeof(v), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    ok = v == 1;
  }
  if (!ok) {
    if (want && c->rank == 0) std::fprintf(stderr, "nsb200: peer-store halo unavailable (CUDA IPC), using NCCL send/recv\n");
    close_peer_halo(c);
    return;
  }
  // segments
  std::vector<int> sp(1, 0), src, spc(1, 0), srcc, pr(np);
  std::vector<long long> land(2 * (size_t)np), landc(np);
  for (int k = 0; k < np; ++k) {
    pr[k] = S.peer[k];
    for (int n : S.send_nodes[k]) for (int cc = 0; cc < dim; ++cc) src.push_back((int)S.node_xoff(n) + cc);
    sp.push_back((int)src.size());
    land[k] = all[((size_t)S.peer[k] * R + c->rank) * 3 + 0];
  }
  H.total_f_vel = (int)src.size();
  for (int k = 0; k < np; ++k) {
    for (int q : S.send_pids[k]) src.push_back((int)S.pid_xoff(q));
    sp.push_back((int)src.size());
    land[np + k] = all[((size_t)S.peer[k] * R + c->rank) * 3 + 1];
    for (int q : S.send_pids[k]) for (int cc = 0; cc < dim; ++cc) srcc.push_back(dim * q + cc);
    spc.push_back((int)srcc.size());
    landc[k] = all[((size_t)S.peer[k] * R + c->rank) * 3 + 2];
  }
  H.total_f_all = (int)src.size(); H.total_c = (int)srcc.size();
  for (int k = 0; k < np; ++k)
    if (land[k] < 0 || land[np + k] < 0 || landc[k] < 0) throw CudaErr{"halo plan mismatch: a peer does not expect data from this rank"};
  H.seg_ptr_f.upload(sp, st); H.src_f.upload(src, st); H.land_f.upload(land, st);
  H.seg_ptr_c.upload(spc, st); H.src_c.upload(srcc, st); H.land_c.upload(landc, st);
  H.d_peer_arena.upload(H.peer_arena, st); H.d_peer_flags.upload(H.peer_flags, st); H.d_peer_rank.upload(pr, st);
  CK(cudaStreamSynchronize(st));
  nccl_barrier(c);                                   // every rank's flags are zeroed before anybody pushes
  H.on = true;
}

// Coarse P1 level of the two-level velocity cycle: graph, tile / stream plans (the same builders as the fine level),
// transfer lists, storage.  Called once per mesh, after build_tiles.
void build_coarse_level(nsb_ctx* c) {
  const Structure& S = c->S;
  Coarse& G = c->cg;
  G.built = false; G.valid = false;
  CoarseLevel CL;
  const std::string e = build_coarse(S, CL);
  if (!e.empty()) throw CudaErr{e};
  const Structure& Sc = CL.Sc;
  for (int P = 0; P < S.np_own; ++P)
    if (Sc.nbr_ptr[P + 1] - Sc.nbr_ptr[P] > CG_MAX_NB) throw CudaErr{"a vertex has more P1 neighbours than the coarse row kernel can accumulate"};
  TilePlan P;
  const TileLimits L{TILE_MAX_NODES, TILE_MAX_IDX, TILE_MAX_UNIQ, TILE_MAX_PUNIQ, VS_MAX_BLOCKS};
  const std::string e1 = build_tile_plan(Sc, L, P);
  if (!e1.empty()) throw CudaErr{e1};
  VsPlan V;
  const std::string e2 = build_vel_stream(Sc, P, V);
  if (!e2.empty()) throw CudaErr{e2};
  cudaStream_t st = c->stream;
  const int dim = c->dim;
  G.n_tiles = P.n_tiles();
  G.total_nq = V.total_nq;
  G.tiles.upload(V.tiles, st); G.meta.upload(V.meta, st); G.uniq_xoff.upload(P.uniq_xoff, st);
  std::vector<long long> t64(Sc.nbr_ptr.begin(), Sc.nbr_ptr.end()), v64(CL.vedge_ptr.begin(), CL.vedge_ptr.end());
  G.nbr_ptr.upload(t64, st); G.vedge_ptr.upload(v64, st);
  std::vector<int> vx(Sc.nbr.size()), ex(CL.vedge.size()), en(CL.node_ends.size()), sx;
  for (size_t i = 0; i < vx.size(); ++i) vx[i] = (int)S.node_xoff(S.pid_node[Sc.nbr[i]]);
  for (size_t i = 0; i < ex.size(); ++i) ex[i] = (int)S.node_xoff(CL.vedge[i]);
  for (size_t i = 0; i < en.size(); ++i) en[i] = (int)Sc.node_xoff(CL.node_ends[i]);
  for (size_t k = 0; k < S.peer.size(); ++k)
    for (int q : S.send_pids[k]) sx.push_back((int)Sc.node_xoff(q));
  G.nbr_vxoff.upload(vx, st); G.vedge_xoff.upload(ex, st); G.ends_xoff.upload(en, st); G.send_xoff.upload(sx, st);
  G.send_buf.alloc(sx.size() * dim);
  G.gid.assign(S.pid_gid.begin(), S.pid_gid.begin() + S.np_own);
  G.h_nbr_ptr.assign(Sc.nbr_ptr.begin(), Sc.nbr_ptr.end());
  G.h_nbr_gid.resize(Sc.nbr.size());
  for (size_t i = 0; i < Sc.nbr.size(); ++i) G.h_nbr_gid[i] = S.pid_gid[Sc.nbr[i]];
  CK(cudaStreamSynchronize(st));
  const size_t nct = (size_t)Sc.n_tot_dofs();
  G.cvals.alloc(Sc.nbr.size() * dim * dim);
  G.dinv.alloc((size_t)S.np_own * dim * dim);
  if (c->nranks == 1) {
    for (DBuf<double>* v : {&G.rc, &G.z0, &G.z1, &G.zd, &G.poly, &G.pin}) { v->alloc(nct); v->zero(st); }
  } else {
    setup_peer_halo(c, {&c->v_old, &c->v_oldold, &c->v_cur, &c->v_sol, &c->v_rhs, &c->cval, &c->w_z0, &c->w_z1, &c->w_d, &c->w_in, &c->w_tmp,
                        &c->w_pin, &c->w_poly, &c->w_y0, &c->w_u},
                    {&G.rc, &G.z0, &G.z1, &G.zd, &G.poly, &G.pin}, (size_t)S.n_tot_dofs(), nct);
  }
  CK(cudaStreamSynchronize(st));
  PolyLevel& C = c->lvC;
  C.coarse = true; C.nn = S.np_own; C.n = (long long)dim * S.np_own; C.n_tot = (long long)nct;
  C.dinv = G.dinv.p; C.gid = G.gid.data();
  C.z0 = G.z0.p; C.z1 = G.z1.p; C.zd = G.zd.p; C.poly = G.poly.p; C.pin = G.pin.p;
  C.probe_init = false; C.roots.clear();
  G.built = true;
}

size_t coarse_vals_bytes(const nsb_ctx* c) {
  if (c->opt.precond_precision == 64) return 0;
  return (size_t)c->cg.total_nq * 4 * c->dim * c->dim * (c->opt.precond_precision == 16 ? 2 : 4);
}

// (re)binds the fine level of the velocity preconditioner to the context's buffers
void bind_fine_level(nsb_ctx* c) {
  PolyLevel& F = c->lvF;
  F.coarse = false; F.nn = c->S.nn_own; F.n = (long long)c->dim * c->S.nn_own; F.n_tot = c->S.n_tot_dofs();
  F.dinv = c->dinv.p; F.gid = c->S.node_gid.data();
  F.z0 = c->w_z0.p; F.z1 = c->w_z1.p; F.zd = c->w_d.p; F.poly = c->w_poly.p; F.pin = c->w_pin.p;
}

// one-time M_p, K_p on the host over the GLOBAL P1 graph (reference cpp:798-803, 812-829)
void host_pressure_matrices(nsb_ctx* c, const std::vector<unsigned char>& pflag) {
  const int dim = c->dim, NV = dim + 1;
  const int64_t np = c->n_p, C = c->n_cells;
  FeTables T;
  fill_tables(dim, T);
  double wsum = 0;
  for (int q = 0; q < T.nq; ++q) wsum += T.w[q];
  // P1 graph
  std::vector<std::vector<int>> adj(np);
  for (int64_t cc = 0; cc < C; ++cc)
    for (int i = 0; i < NV; ++i)
      for (int j = 0; j < NV; ++j) adj[c->g_cell_pid[cc * NV + i]].push_back(c->g_cell_pid[cc * NV + j]);
  HostCsr Mp, Kp;
  Mp.n = Mp.m = (int)np;
  Mp.ptr.assign(np + 1, 0);
  for (int64_t i = 0; i < np; ++i) {
    auto& a = adj[i];
    std::sort(a.begin(), a.end());
    a.erase(std::unique(a.begin(), a.end()), a.end());
    Mp.ptr[i + 1] = Mp.ptr[i] + (int)a.size();
  }
  Mp.col.resize(Mp.ptr[np]);
  for (int64_t i = 0; i < np; ++i) std::copy(adj[i].begin(), adj[i].end(), Mp.col.begin() + Mp.ptr[i]);
  Mp.val.assign(Mp.col.size(), 0.0);
  Kp = Mp;
  auto find = [&](int r, int col) {
    const int* b = Mp.col.data() + Mp.ptr[r];
    const int* e = Mp.col.data() + Mp.ptr[r + 1];
    return (int)(std::lower_bound(b, e, col) - Mp.col.data());
  };
  for (int64_t cc = 0; cc < C; ++cc) {
    const uint32_t* cv = c->cell_vertices.data() + cc * NV;
    double X[4][3] = {{0}};
    for (int v = 0; v < NV; ++v)
      for (int k = 0; k < dim; ++k) X[v][k] = c->coords[(size_t)cv[v] * dim + k];
    double gl[4][3] = {{0}}, det;
    if (dim == 2) {
      const double a = X[1][0] - X[0][0], b = X[2][0] - X[0][0], cq = X[1][1] - X[0][1], d = X[2][1] - X[0][1];
      det = a * d - b * cq;
      gl[1][0] = d / det; gl[1][1] = -b / det; gl[2][0] = -cq / det; gl[2][1] = a / det;
      for (int k = 0; k < 2; ++k) gl[0][k] = -(gl[1][k] + gl[2][k]);
    } else {
      double J[3][3];
      for (int r = 0; r < 3; ++r)
        for (int k = 0; k < 3; ++k) J[r][k] = X[k + 1][r] - X[0][r];
      const double c00 = J[1][1] * J[2][2] - J[1][2] * J[2][1], c01 = J[1][2] * J[2][0] - J[1][0] * J[2][2],
                   c02 = J[1][0] * J[2][1] - J[1][1] * J[2][0];
      det = J[0][0] * c00 + J[0][1] * c01 + J[0][2] * c02;
      const double id = 1.0 / det;
      gl[1][0] = c00 * id; gl[1][1] = (J[0][2] * J[2][1] - J[0][1] * J[2][2]) * id; gl[1][2] = (J[0][1] * J[1][2] - J[0][2] * J[1][1]) * id;
      gl[2][0] = c01 * id; gl[2][1] = (J[0][0] * J[2][2] - J[0][2] * J[2][0]) * id; gl[2][2] = (J[0][2] * J[1][0] - J[0][0] * J[1][2]) * id;
      gl[3][0] = c02 * id; gl[3][1] = (J[0][1] * J[2][0] - J[0][0] * J[2][1]) * id; gl[3][2] = (J[0][0] * J[1][1] - J[0][1] * J[1][0]) * id;
      for (int k = 0; k < 3; ++k) gl[0][k] = -((gl[1][k] + gl[2][k]) + gl[3][k]);
    }
    const double absJ = std::fabs(det);
    const int* pid = c->g_cell_pid.data() + cc * NV;
    for (int i = 0; i < NV; ++i) {
      const bool ci = pflag[pid[i]] != 0;
      for (int j = 0; j < NV; ++j) {
        const bool cj = pflag[pid[j]] != 0;
        double gg = 0;
        for (int k = 0; k < dim; ++k) gg += gl[i][k] * gl[j][k];
        double m = absJ * T.MPhat[i][j], kk = absJ * wsum * gg;
        if (ci || cj) {
          if (i == j) { m = std::fabs(m); kk = std::fabs(kk); }    // constrained diagonal: |m_cc| (A.5)
          else { m = 0; kk = 0; }
        }
        const int p = find(pid[i], pid[j]);
        Mp.val[p] += m;
        Kp.val[p] += kk;
      }
    }
  }
  for (size_t k = 0; k < Kp.val.size(); ++k) Kp.val[k] += 1e-6 * Mp.val[k];     // cpp:536, 828
  c->h_Mp = std::move(Mp);
  c->h_Kp = std::move(Kp);
}

double* vec_ptr(nsb_ctx* c, int which) {
  switch (which) {
    case NSB_SOLUTION_OLD: return c->v_old.p;
    case NSB_SOLUTION_OLD_OLD: return c->v_oldold.p;
    case NSB_CURRENT_SOLUTION: return c->v_cur.p;
    case NSB_SOLUTION: return c->v_sol.p;
    case NSB_RHS: return c->v_rhs.p;
  }
  return nullptr;
}

// ---- inspection of the velocity preconditioner's operators (parity tests) ------------------------------------------
// Vectors of a level in its own global numbering: level 0 = velocity DoFs (dim * node + component), level 1 = the coarse
// P1 level (dim * vertex + component, vertex = pressure DoF - n_u).  Level 1 is only mapped on one GPU (no ghost vertices).
PolyLevel& level_of(nsb_ctx* c, int level) { return level == 0 ? c->lvF : c->lvC; }

void level_upload(nsb_ctx* c, int level, const double* g, double* d) {
  const Structure& S = c->S;
  const int dim = c->dim;
  const int nn = level == 0 ? S.nn_own + S.nn_ghost : S.np_own;
  std::vector<double> loc(level == 0 ? (size_t)S.n_tot_dofs() : (size_t)dim * nn, 0.0);
  for (int A = 0; A < nn; ++A) {
    const int64_t off = level == 0 ? S.node_xoff(A) : (int64_t)dim * A;
    const int64_t gid = level == 0 ? S.node_gid[A] : S.pid_gid[A];
    for (int k = 0; k < dim; ++k) loc[off + k] = g[gid * dim + k];
  }
  CK(cudaMemcpyAsync(d, loc.data(), loc.size() * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  CK(cudaStreamSynchronize(c->stream));
}

void level_download(nsb_ctx* c, int level, const double* d, double* g) {
  const Structure& S = c->S;
  const int dim = c->dim;
  const int nn = level == 0 ? S.nn_own : S.np_own;
  std::vector<double> out((size_t)dim * nn);
  CK(cudaMemcpyAsync(out.data(), d, out.size() * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  for (int A = 0; A < nn; ++A) {
    const int64_t gid = level == 0 ? S.node_gid[A] : S.pid_gid[A];
    for (int k = 0; k < dim; ++k) g[gid * dim + k] = out[(size_t)dim * A + k];
  }
}

// one level_apply<mode> on host vectors of the level's global numbering (u read for modes 3 / 4, poly read and written for 3)
void velocity_operator_apply(nsb_ctx* c, int level, int mode, const double* coef, const double* xg, const double* ug, double* yg,
                             double* pg) {
  PolyLevel& lv = level_of(c, level);
  double* x = level == 0 ? c->w_pin.p : c->cg.pin.p;
  double* u = level == 0 ? c->w_u.p : c->cg.z0.p;
  double* y = level == 0 ? c->w_tmp.p : c->cg.z1.p;
  double* p = level == 0 ? c->w_poly.p : c->cg.poly.p;
  level_upload(c, level, xg, x);
  if (mode >= 3) level_upload(c, level, ug, u);
  if (mode == 3) level_upload(c, level, pg, p);
  const PolyCoef pc = coef ? PolyCoef{coef[0], coef[1], coef[2], coef[3]} : PolyCoef{};
  if (mode == 2) level_apply<2>(c, lv, x, y, nullptr, nullptr, pc);
  else if (mode == 3) level_apply<3>(c, lv, x, y, u, p, pc);
  else level_apply<4>(c, lv, x, y, u, nullptr, pc);
  level_download(c, level, y, yg);
  if (mode == 3) level_download(c, level, p, pg);
}

// The packed copy of a level's B = Dinv F unpacked into (node, neighbour, dim*dim values) in stream order, from the tile
// headers, the quad metadata and the unique-neighbour lists exactly as the streamed kernel reads them.
template <typename VT>
void unpack_level(nsb_ctx* c, const VsDev& D, int64_t total_nq, size_t n_uniq, std::vector<int>& node, std::vector<int>& nbr,
                  std::vector<double>& val) {
  const int dim = c->dim, PL = dim * dim;
  std::vector<VsTile> tiles(D.n_tiles);
  std::vector<uint32_t> meta((size_t)total_nq * 4);
  std::vector<int> uniq(n_uniq);
  std::vector<VT> v((size_t)total_nq * 4 * PL);
  CK(cudaMemcpyAsync(tiles.data(), D.tiles, tiles.size() * sizeof(VsTile), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemcpyAsync(meta.data(), D.meta, meta.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemcpyAsync(uniq.data(), D.uniq_xoff, uniq.size() * sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemcpyAsync(v.data(), D.vals, v.size() * sizeof(VT), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  for (const VsTile& T : tiles) {
    const uint32_t* m = meta.data() + (size_t)T.nq_off * 4;
    const VT* tv = v.data() + (size_t)T.nq_off * 4 * PL;
    for (int q = 0; q < T.nquad; ++q) {
      const uint32_t* mq = m + 4 * q;
      if (mq[2] == 0xffffu) continue;
      const int cnt = (int)(mq[3] >> 16);
      for (int e = 0; e < cnt; ++e) {
        const int loc = (int)(((e < 2 ? mq[0] : mq[1]) >> (16 * (e & 1))) & 0xffffu);
        node.push_back(T.n0 + (int)mq[2]);
        nbr.push_back(uniq[T.u0 + loc] / dim);
        for (int rc = 0; rc < PL; ++rc) val.push_back((double)(float)tv[((size_t)rc * T.NQ + q) * 4 + e]);
      }
    }
  }
}

size_t forcing_len(const nsb_ctx* c) { return (size_t)c->S.nc * (c->dim == 2 ? Fe<2>::NQ : Fe<3>::NQ) * c->dim; }

// Both forcing slots are allocated (zeroed) together, the first time one of them receives values.
void forcing_alloc(nsb_ctx* c) {
  if (c->forcing[0].p) return;
  for (auto& b : c->forcing) { b.alloc(forcing_len(c)); b.zero(c->stream); }
}

// Slot `which` now holds non-zero values or not.  A slot that is not set holds zeros while the other one is set (`written`:
// its values were just overwritten, so they are zeroed even if it was clear before); both clear = both freed, and the
// kernels read nothing.
void forcing_commit(nsb_ctx* c, int which, bool nonzero, bool written) {
  if (!nonzero && c->forcing_set[1 - which] && (written || c->forcing_set[which])) c->forcing[which].zero(c->stream);
  c->forcing_set[which] = nonzero;
  if (!c->forcing_set[0] && !c->forcing_set[1] && c->forcing[0].p) {
    CK(cudaStreamSynchronize(c->stream));       // an assembly may still read them
    for (auto& b : c->forcing) b.alloc(0);
  }
}

// The vertices of the local cells (owned + ghost layer) and the local cell -> vertex table the evaluation kernel reads.
void forcing_geometry(nsb_ctx* c) {
  if (c->fsrc_geom) return;
  const Structure& S = c->S;
  const int dim = c->dim, NV = dim + 1;
  std::vector<int> g2l(c->n_vertices, -1), cells((size_t)S.nc * NV);
  std::vector<double> X;
  for (int cl = 0; cl < S.nc; ++cl)
    for (int v = 0; v < NV; ++v) {
      const uint32_t g = c->cell_vertices[(size_t)S.cell_gid[cl] * NV + v];
      if (g2l[g] < 0) {
        g2l[g] = (int)(X.size() / dim);
        X.insert(X.end(), c->coords.begin() + (size_t)g * dim, c->coords.begin() + (size_t)(g + 1) * dim);
      }
      cells[(size_t)cl * NV + v] = g2l[g];
    }
  c->fsrc_coords.upload(X, c->stream);
  c->fsrc_cells.upload(cells, c->stream);
  CK(cudaStreamSynchronize(c->stream));
  c->fsrc_geom = true;
}

void forcing_unload(nsb_ctx* c) {
  if (c->fsrc_lib) {
    CK(cudaStreamSynchronize(c->stream));       // an evaluation may still run
    CK(cudaLibraryUnload(c->fsrc_lib));
  }
  c->fsrc_lib = nullptr;
  c->fsrc_kernel = nullptr;
  c->fsrc_text.clear();
}

}  // namespace

// =====================================================================================
extern "C" {

int nsb_create(int dim, int device, nsb_handle* out) {
  if (!out) return -1;
  *out = nullptr;
  if (dim != 2 && dim != 3) return -1;
  nsb_ctx* c = new nsb_ctx();
  c->dim = dim; c->device = device;
  *out = c;
  NSB_TRY
  // NSB200_VS_CTAS=n caps the grid of the streamed velocity operator at n CTAs, so that every CTA walks its ring of stages
  // through many tiles; the result does not depend on it (a tile is reduced by one consumer group in a fixed order)
  if (const char* cap = std::getenv("NSB200_VS_CTAS")) {
    char* end = nullptr;
    errno = 0;
    const long v = std::strtol(cap, &end, 10);
    if (end == cap || *end != '\0' || errno == ERANGE || v < 1 || v > INT_MAX)
      throw CudaErr{std::string("NSB200_VS_CTAS must be a positive integer, got \"") + cap + "\""};
    c->vs_ctas = (int)v;
  }
  int ndev = 0;
  CK(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) throw CudaErr{"no such CUDA device (the product path has no CPU fallback)"};
  CK(cudaSetDevice(device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) throw CudaErr{"nsb200 is built for sm_100a (B200) only"};
  CK(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  CK(cudaEventCreate(&c->t0));
  CK(cudaEventCreate(&c->t1));
  FeTables T2, T3;
  fill_tables(2, T2);
  fill_tables(3, T3);
  {
    std::vector<FeTables> tv(1, dim == 2 ? T2 : T3);
    c->d_fe.upload(tv, c->stream);
    CK(cudaStreamSynchronize(c->stream));
  }
  CK(cudaDeviceGetAttribute(&c->num_sms, cudaDevAttrMultiProcessorCount, device));
  c->opt.poly_degree_F = 64; c->opt.poly_refresh = 1; c->opt.poly_target = 0.08; c->opt.poly_kind = 1; c->opt.cheb_degree_Mp = 3;
  c->opt.amg_smoother_degree = 2; c->opt.schur_mass_coeff = -1.0; c->opt.reorthogonalize = 1;
  c->opt.precond_precision = NSB_DEFAULT_PRECOND_PRECISION;
  c->opt.precond_operator = 1;
  c->opt.velocity_cycle = 2; c->opt.smoother_degree = 14; c->opt.smoother_lo_frac = 0.012; c->opt.coarse_degree = 15; c->opt.smoother_hi_factor = 1.1;
  c->par.dt = 0.01; c->par.theta = 1.0; c->par.nu = 1e-3; c->par.rho = 1.0; c->par.gamma = 0.1;
  c->d_nrm.alloc(4);
  return 0;
  NSB_CATCH(c)
}

int nsb_destroy(nsb_handle c) {
  if (!c) return 0;
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  if (c->ph.on) {
    // peers may still map this rank's arena: close our mappings, then rendezvous before anything is freed
    try { close_peer_halo(c); nccl_barrier(c); } catch (...) {}
  }
  if (c->pin) cudaFreeHost(c->pin);
  if (c->fsrc_lib) cudaLibraryUnload(c->fsrc_lib);
  if (c->comm) g_nccl.CommDestroy(c->comm);
  if (c->t0) cudaEventDestroy(c->t0);
  if (c->t1) cudaEventDestroy(c->t1);
  cudaStream_t s = c->stream;
  delete c;
  if (s) cudaStreamDestroy(s);
  return 0;
}

const char* nsb_last_error(nsb_handle c) { return c ? c->err.c_str() : "null handle"; }

int nsb_comm_unique_id(void* out128) {
  ncclUniqueId id;
  std::string err;
  if (!g_nccl.load(err)) { std::fprintf(stderr, "nsb200: %s\n", err.c_str()); return -1; }
  if (g_nccl.GetUniqueId(&id) != ncclSuccess) return -1;
  std::memcpy(out128, &id, sizeof(id));
  return 0;
}

int nsb_comm_init(nsb_handle c, int rank, int nranks, const void* uid) {
  if (!c) return -1;
  NSB_TRY
  CK(cudaSetDevice(c->device));
  if (c->have_mesh) throw CudaErr{"nsb_comm_init must precede nsb_upload_mesh"};
  if (nranks > 1) {
    std::string err;
    if (!g_nccl.load(err)) throw CudaErr{err};
    if (!uid) throw CudaErr{"nccl_unique_id is required with more than one rank"};
    ncclUniqueId id;
    std::memcpy(&id, uid, sizeof(id));
    CKN(g_nccl.CommInitRank(&c->comm, nranks, id, rank));
  }
  c->rank = rank; c->nranks = nranks;
  return 0;
  NSB_CATCH(c)
}

int nsb_upload_mesh(nsb_handle c, int64_t n_vertices, const double* coords, int64_t n_cells,
                    const uint32_t* cell_vertices, const uint32_t* cell_dofs, int64_t n_u, int64_t n_p,
                    const int32_t* cell_part) {
  if (!c) return -1;
  NSB_TRY
  CK(cudaSetDevice(c->device));
  for (auto& b : c->forcing) b.alloc(0);    // forcing values belong to the previous mesh's local cells
  c->forcing_set[0] = c->forcing_set[1] = false;
  c->fsrc_coords.alloc(0); c->fsrc_cells.alloc(0);   // so does the geometry of a forcing source (the source itself stays)
  c->fsrc_geom = false;
  const int dim = c->dim, NV = dim + 1;
  std::string e = build_structure(dim, n_vertices, coords, n_cells, cell_vertices, cell_dofs, n_u, n_p,
                                  c->nranks > 1 ? cell_part : nullptr, c->rank, c->nranks, c->S);
  if (!e.empty()) return fail(c, e);
  if (c->nranks > 1 && !cell_part) return fail(c, "cell_part is required with more than one rank");
  Structure& S = c->S;
  c->n_vertices = n_vertices; c->n_cells = n_cells; c->n_u = n_u; c->n_p = n_p;
  c->coords.assign(coords, coords + n_vertices * dim);
  c->cell_vertices.assign(cell_vertices, cell_vertices + n_cells * NV);
  c->g_cell_pid.resize(n_cells * NV);
  const int DPC = S.DPC;
  for (int64_t cc = 0; cc < n_cells; ++cc)
    for (int v = 0; v < NV; ++v) c->g_cell_pid[cc * NV + v] = (int)(cell_dofs[cc * DPC + v * (dim + 1) + dim] - n_u);
  if (S.n_tot_dofs() >= (int64_t)INT32_MAX) return fail(c, "local vector too long for 32-bit offsets");
  // global dof -> local offset
  c->g2x.assign(n_u + n_p, -1);
  for (int A = 0; A < S.nn_own + S.nn_ghost; ++A)
    for (int k = 0; k < dim; ++k) c->g2x[S.node_gid[A] * dim + k] = (int)S.node_xoff(A) + k;
  for (int P = 0; P < S.np_own + S.np_ghost; ++P) c->g2x[n_u + S.pid_gid[P]] = (int)S.pid_xoff(P);
  // ---- device copies
  cudaStream_t st = c->stream;
  std::vector<int> cx(S.cell_nodes.size()), cp(S.cell_pids.size());
  for (size_t i = 0; i < cx.size(); ++i) cx[i] = (int)S.node_xoff(S.cell_nodes[i]);
  for (size_t i = 0; i < cp.size(); ++i) cp[i] = (int)S.pid_xoff(S.cell_pids[i]);
  c->d_cell_xoff.upload(cx, st); c->d_cell_poff.upload(cp, st);
  c->d_cell_geom.upload(S.cell_geom, st);
  c->d_rank_uu.upload(S.rank_uu, st); c->d_rank_up.upload(S.rank_up, st);
  std::vector<int> nx(S.nbr.size()), px(S.pnbr.size());
  for (size_t i = 0; i < nx.size(); ++i) nx[i] = (int)S.node_xoff(S.nbr[i]);
  for (size_t i = 0; i < px.size(); ++i) px[i] = (int)S.pid_xoff(S.pnbr[i]);
  c->d_nbr_xoff.upload(nx, st); c->d_pnbr_xoff.upload(px, st);
  std::vector<long long> t64;
  auto up64 = [&](const std::vector<int64_t>& v, DBuf<long long>& d) {
    t64.assign(v.begin(), v.end());
    d.upload(t64, st);
    CK(cudaStreamSynchronize(st));
  };
  up64(S.nbr_ptr, c->d_nbr_ptr); up64(S.pnbr_ptr, c->d_pnbr_ptr);
  up64(S.rowbase, c->d_rowbase); up64(S.prowbase, c->d_prowbase); up64(S.n2c_ptr, c->d_n2c_ptr);
  c->d_selfrank.upload(S.selfrank, st);
  std::vector<int> npid(S.node_pid.begin(), S.node_pid.begin() + S.nn_own);
  c->d_node_pid.upload(npid, st);
  std::vector<int> pnode(S.pid_node.begin(), S.pid_node.begin() + S.np_own);
  c->d_pid_node.upload(pnode, st);
  c->d_pselfrank.upload(S.pselfrank, st);
  c->d_n2c.upload(S.n2c, st);
  if (S.nbr.size() >= (size_t)INT32_MAX) return fail(c, "neighbour lists too long for 32-bit offsets");
  std::vector<NodeDesc> nd(S.nn_own);
  for (int A = 0; A < S.nn_own; ++A) {
    NodeDesc& d = nd[A];
    d.rowbase = S.rowbase[A];
    d.pid = S.node_pid[A];
    d.prowbase = d.pid >= 0 ? S.prowbase[d.pid] : 0;
    d.nbr0 = (int)S.nbr_ptr[A];
    d.pnbr0 = (int)S.pnbr_ptr[A];
    d.nb = (unsigned short)(S.nbr_ptr[A + 1] - S.nbr_ptr[A]);
    d.np = (unsigned short)(S.pnbr_ptr[A + 1] - S.pnbr_ptr[A]);
  }
  c->d_nd.upload(nd, st);
  CK(cudaStreamSynchronize(st));
  DevMesh& M = c->M;
  M.nd = c->d_nd.p;
  M.dim = dim; M.nn_own = S.nn_own; M.nn_tot = S.nn_own + S.nn_ghost; M.np_own = S.np_own;
  M.np_tot = S.np_own + S.np_ghost; M.nc = S.nc; M.n_own = S.n_own_dofs(); M.n_tot = S.n_tot_dofs();
  M.cell_xoff = c->d_cell_xoff.p; M.cell_poff = c->d_cell_poff.p; M.cell_geom = c->d_cell_geom.p;
  M.rank_uu = c->d_rank_uu.p; M.rank_up = c->d_rank_up.p;
  M.nbr_ptr = c->d_nbr_ptr.p; M.nbr_xoff = c->d_nbr_xoff.p; M.pnbr_ptr = c->d_pnbr_ptr.p; M.pnbr_xoff = c->d_pnbr_xoff.p;
  M.selfrank = c->d_selfrank.p; M.node_pid = c->d_node_pid.p; M.pid_node = c->d_pid_node.p; M.pselfrank = c->d_pselfrank.p;
  M.rowbase = c->d_rowbase.p; M.prowbase = c->d_prowbase.p; M.n2c_ptr = c->d_n2c_ptr.p; M.n2c = c->d_n2c.p;
  build_tiles(c);
  if (c->nranks > 1) {
    std::vector<int> pg(S.np_own), og(S.n_own_dofs());
    for (int P = 0; P < S.np_own; ++P) pg[P] = (int)S.pid_gid[P];
    for (int A = 0; A < S.nn_own; ++A)
      for (int k = 0; k < dim; ++k) og[(size_t)dim * A + k] = (int)(S.node_gid[A] * dim + k);
    for (int P = 0; P < S.np_own; ++P) og[(size_t)dim * S.nn_own + P] = (int)(n_u + S.pid_gid[P]);
    c->d_pid_gid.upload(pg, st);
    c->d_own_gdof.upload(og, st);
    c->w_tg.alloc((size_t)n_p);
    c->w_gather.alloc((size_t)(n_u + n_p));
    CK(cudaStreamSynchronize(st));
  }
  // vectors and system storage (several ranks: build_coarse_level places all exchanged vectors in the symmetric arena)
  const size_t nt = (size_t)S.n_tot_dofs();
  build_coarse_level(c);
  if (c->nranks == 1) {
    for (DBuf<double>* v : {&c->v_old, &c->v_oldold, &c->v_cur, &c->v_sol, &c->v_rhs, &c->cval, &c->w_z0, &c->w_z1, &c->w_d,
                            &c->w_in, &c->w_tmp, &c->w_pin, &c->w_poly, &c->w_y0, &c->w_u}) {
      v->alloc(nt);
      v->zero(st);
    }
  }
  if (c->pin) { cudaFreeHost(c->pin); c->pin = nullptr; }
  CK(cudaMallocHost(&c->pin, nt * sizeof(double)));
  c->cflag.alloc(nt); c->cflag.zero(st);
  c->vals.alloc((size_t)S.nnz_local);
  c->cg.vals.alloc(coarse_vals_bytes(c));
  c->dinv.alloc((size_t)S.nn_own * dim * dim);
  c->cell_rhs.alloc((size_t)S.nc * S.DPC);
  c->ctx_stride = 0;
  c->partial.alloc((size_t)nblk(S.n_own_dofs(), RED_CHUNK) * 4);
  CK(cudaStreamSynchronize(st));
  c->have_mesh = true; c->have_matrix = false; c->have_pressure = false;
  bind_fine_level(c);
  c->lvF.probe_init = false; c->lvF.roots.clear(); c->solves = 0; c->V_cap = 0; c->two_level = false; c->cycle_disabled = false;
  c->halo.clear();                 // pack lists of the previous mesh
  return 0;
  NSB_CATCH(c)
}

int nsb_get_sizes(nsb_handle c, int64_t* nrows, int64_t* nnz, int64_t* ncl) {
  if (!c || !c->have_mesh) return fail(c, "no mesh uploaded");
  if (nrows) *nrows = c->S.n_own_dofs();
  if (nnz) *nnz = c->S.nnz_local;
  if (ncl) *ncl = c->S.nc;
  return 0;
}

int nsb_get_block_nnz(nsb_handle c, int64_t* uu, int64_t* up, int64_t* pu, int64_t* pp) {
  if (!c || !c->have_mesh) return fail(c, "no mesh uploaded");
  const Structure& S = c->S;
  int64_t a = 0, b = 0, d = 0, e = 0;
  for (int A = 0; A < S.nn_own; ++A) {
    const int64_t nb = S.nbr_ptr[A + 1] - S.nbr_ptr[A], np = S.pnbr_ptr[A + 1] - S.pnbr_ptr[A];
    a += (int64_t)S.dim * S.dim * nb;
    b += (int64_t)S.dim * np;
    if (S.node_pid[A] >= 0) { d += (int64_t)S.dim * nb; e += np; }
  }
  if (uu) *uu = a;
  if (up) *up = b;
  if (pu) *pu = d;
  if (pp) *pp = e;
  return 0;
}

int nsb_get_pattern(nsb_handle c, int64_t* rowptr, uint32_t* col) {
  if (!c || !c->have_mesh) return fail(c, "no mesh uploaded");
  std::vector<int64_t> rp;
  std::vector<uint32_t> cl;
  export_pattern(c->S, rp, cl);
  std::copy(rp.begin(), rp.end(), rowptr);
  std::copy(cl.begin(), cl.end(), col);
  return 0;
}

int nsb_get_row_gids(nsb_handle c, int64_t* gid) {
  if (!c || !c->have_mesh) return fail(c, "no mesh uploaded");
  std::vector<int64_t> g;
  export_row_gids(c->S, g);
  std::copy(g.begin(), g.end(), gid);
  return 0;
}

int nsb_set_constraints(nsb_handle c, int64_t n, const uint32_t* dof, const double* val) {
  if (!c || !c->have_mesh) return fail(c, "no mesh uploaded");
  NSB_TRY
  CK(cudaSetDevice(c->device));
  cudaStream_t st = c->stream;
  // clear the previous set
  if (c->n_con) {
    k_scatter_flags<<<nblk(c->n_con, 256), 256, 0, st>>>(c->n_con, c->c_idx.p, c->cflag.p, 0);
    c->launch_check();
  }
  std::vector<int> idx;
  std::vector<double> v;
  idx.reserve(n); v.reserve(n);
  const int64_t N = c->n_u + c->n_p;
  for (int64_t i = 0; i < n; ++i) {
    if (dof[i] >= N) return fail(c, "constraint DoF out of range");
    const int x = c->g2x[dof[i]];
    if (x >= 0) { idx.push_back(x); v.push_back(val[i]); }
  }
  c->n_con = (int)idx.size();
  CK(cudaStreamSynchronize(st));
  c->c_idx.upload(idx, st);
  c->c_val.upload(v, st);
  if (c->n_con) {
    k_scatter_flags<<<nblk(c->n_con, 256), 256, 0, st>>>(c->n_con, c->c_idx.p, c->cflag.p, 1);
    c->launch_check();
    k_scatter_vals<<<nblk(c->n_con, 256), 256, 0, st>>>(c->n_con, c->c_idx.p, c->c_val.p, c->cval.p);
    c->launch_check();
  }
  CK(cudaStreamSynchronize(st));
  return 0;
  NSB_CATCH(c)
}

int nsb_set_params(nsb_handle c, const nsb_params* p) {
  if (!c || !p) return -1;
  if (!(p->dt > 0)) return fail(c, "dt must be positive");
  c->par = *p;
  return 0;
}

int nsb_set_solver_opts(nsb_handle c, const nsb_solver_opts* o) {
  if (!c || !o) return -1;
  nsb_solver_opts n = *o;
  if (n.poly_degree_F <= 0) n.poly_degree_F = 64;
  if (!(n.poly_target > 0)) n.poly_target = 0.08;
  if (n.poly_kind == 0) n.poly_kind = 1;          // 0 = default (Chebyshev roots when the spectrum is real)
  else if (n.poly_kind < 0) n.poly_kind = 0;      // negative = force the harmonic-Ritz (GMRES) polynomial
  if (n.poly_refresh <= 0) n.poly_refresh = 1;
  if (n.cheb_degree_Mp <= 0) n.cheb_degree_Mp = 3;
  if (n.amg_smoother_degree <= 0) n.amg_smoother_degree = 2;
  if (n.schur_mass_coeff == 0.0) n.schur_mass_coeff = -1.0;
  if (n.reorthogonalize == 0) n.reorthogonalize = 1;   // 0 = default; see nsb200.h
  if (n.precond_precision != 64 && n.precond_precision != 16 && n.precond_precision != 32) n.precond_precision = NSB_DEFAULT_PRECOND_PRECISION;
  n.precond_operator = 1;                         // the element-wise operator of round 1 is gone (slower than the packed copy)
  if (n.velocity_cycle != 1 && n.velocity_cycle != 2) n.velocity_cycle = 2;
  if (n.smoother_degree <= 0) n.smoother_degree = 14;
  if (!(n.smoother_lo_frac > 0 && n.smoother_lo_frac < 1)) n.smoother_lo_frac = 0.012;
  if (n.coarse_degree <= 0) n.coarse_degree = 15;
  if (!(n.smoother_hi_factor >= 1.0)) n.smoother_hi_factor = 1.1;
  const bool changed = n.precond_precision != c->opt.precond_precision;
  c->opt = n;
  c->cycle_disabled = false;
  if (c->have_mesh && changed) {
    // (de)allocate the packed operator copy of the velocity polynomial; it is refilled by the next assembly
    try {
      cudaSetDevice(c->device);
      c->vs_vals.alloc(vs_vals_bytes(c));
      c->cg.vals.alloc(coarse_vals_bytes(c));
      c->vs_valid = false; c->cg.valid = false;
    } catch (const CudaErr& e) { return fail(c, e.msg); }
    c->have_matrix = false;
    c->lvF.roots.clear();
  }
  return 0;
}

int nsb_set_vector(nsb_handle c, int which, const double* vg) {
  if (!c || !c->have_mesh) return fail(c, "no mesh uploaded");
  NSB_TRY
  CK(cudaSetDevice(c->device));
  double* d = vec_ptr(c, which);
  if (!d) return fail(c, "bad vector id");
  const Structure& S = c->S;
  double* loc = c->pin;
  const int dim = c->dim;
  if (c->nranks == 1) {
    std::memcpy(loc, vg, (size_t)S.n_own_dofs() * sizeof(double));     // local layout == global numbering
  } else {
#pragma omp parallel for schedule(static)
    for (int A = 0; A < S.nn_own + S.nn_ghost; ++A)
      for (int k = 0; k < dim; ++k) loc[S.node_xoff(A) + k] = vg[S.node_gid[A] * dim + k];
#pragma omp parallel for schedule(static)
    for (int P = 0; P < S.np_own + S.np_ghost; ++P) loc[S.pid_xoff(P)] = vg[c->n_u + S.pid_gid[P]];
  }
  CK(cudaMemcpyAsync(d, loc, (size_t)S.n_tot_dofs() * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return 0;
  NSB_CATCH(c)
}

int nsb_get_quadrature_points(nsb_handle c, int* n_q, double* pts) {
  if (!c || !c->have_mesh) return fail(c, "nsb_get_quadrature_points: no mesh uploaded");
  NSB_TRY
  const Structure& S = c->S;
  const int dim = c->dim, NV = dim + 1;
  FeTables T;
  fill_tables(dim, T);
  if (n_q) *n_q = T.nq;
  if (!pts) return 0;
  const int nq = T.nq;
#pragma omp parallel for schedule(static)
  for (int cl = 0; cl < S.nc; ++cl) {
    const uint32_t* cv = c->cell_vertices.data() + (size_t)S.cell_gid[cl] * NV;
    for (int q = 0; q < nq; ++q)
      for (int k = 0; k < dim; ++k) {
        double x = 0.0;
        for (int v = 0; v < NV; ++v) x += T.lam[q][v] * c->coords[(size_t)cv[v] * dim + k];
        pts[((size_t)cl * nq + q) * dim + k] = x;
      }
  }
  return 0;
  NSB_CATCH(c)
}

int nsb_set_forcing(nsb_handle c, int which, const double* f) {
  if (!c || !c->have_mesh) return fail(c, "nsb_set_forcing: no mesh uploaded");
  if (which != NSB_FORCING_NEW && which != NSB_FORCING_OLD)
    return fail(c, "nsb_set_forcing: which must be NSB_FORCING_NEW (0) or NSB_FORCING_OLD (1)");
  NSB_TRY
  CK(cudaSetDevice(c->device));
  const size_t n = forcing_len(c);
  bool nonzero = false;
  if (f)
    for (size_t i = 0; i < n && !nonzero; ++i) nonzero = f[i] != 0.0;
  if (nonzero) {
    forcing_alloc(c);
    CK(cudaMemcpyAsync(c->forcing[which].p, f, n * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    CK(cudaStreamSynchronize(c->stream));       // f is the caller's pageable buffer
  }
  forcing_commit(c, which, nonzero, false);
  return 0;
  NSB_CATCH(c)
}

int nsb_set_forcing_source(nsb_handle c, const char* src, const double* prm, int n_prm) {
  if (!c || !c->have_mesh) return fail(c, "nsb_set_forcing_source: no mesh uploaded");
  if (n_prm < 0 || n_prm > kForcingMaxParams)
    return fail(c, "nsb_set_forcing_source: n_prm must be in 0.." + std::to_string(kForcingMaxParams) + ", got " + std::to_string(n_prm));
  if (!prm && n_prm > 0) return fail(c, "nsb_set_forcing_source: prm is NULL but n_prm > 0");
  NSB_TRY
  CK(cudaSetDevice(c->device));
  if (!src) {
    forcing_unload(c);
    forcing_commit(c, NSB_FORCING_NEW, false, false);
    forcing_commit(c, NSB_FORCING_OLD, false, false);
    c->fsrc_coords.alloc(0); c->fsrc_cells.alloc(0);
    c->fsrc_geom = false;
    return 0;
  }
  if (!c->fsrc_lib || c->fsrc_text != src) {
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, c->device));
    std::vector<char> cubin;
    const std::string e = compile_forcing(c->dim, src, "sm_" + std::to_string(prop.major) + std::to_string(prop.minor) + "a", cubin);
    if (!e.empty()) return fail(c, e);
    forcing_unload(c);
    CK(cudaLibraryLoadData(&c->fsrc_lib, cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0));
    CK(cudaLibraryGetKernel(&c->fsrc_kernel, c->fsrc_lib, "nsb_forcing_eval"));
    c->fsrc_text = src;
    ++c->fsrc_compiles;
  }
  std::vector<double> p(kForcingMaxParams, 0.0);
  std::copy(prm, prm + n_prm, p.begin());
  c->fsrc_prm.upload(p, c->stream);
  if (!c->fsrc_flag.p) c->fsrc_flag.alloc(1);
  forcing_geometry(c);                          // synchronises: p may go out of scope
  return 0;
  NSB_CATCH(c)
}

int nsb_eval_forcing(nsb_handle c, int which, double t) {
  if (!c || !c->have_mesh) return fail(c, "nsb_eval_forcing: no mesh uploaded");
  if (which != NSB_FORCING_NEW && which != NSB_FORCING_OLD)
    return fail(c, "nsb_eval_forcing: which must be NSB_FORCING_NEW (0) or NSB_FORCING_OLD (1)");
  if (!c->fsrc_lib) return fail(c, "nsb_eval_forcing: no forcing source set (nsb_set_forcing_source)");
  NSB_TRY
  CK(cudaSetDevice(c->device));
  forcing_geometry(c);
  forcing_alloc(c);
  const int dim = c->dim, nq = dim == 2 ? Fe<2>::NQ : Fe<3>::NQ;
  FeTables T;
  fill_tables(dim, T);
  double lam[Fe<3>::NQ * 4];                    // passed by value: [nq][dim + 1], the kernel's nsb_lambda
  for (int q = 0; q < nq; ++q)
    for (int v = 0; v <= dim; ++v) lam[q * (dim + 1) + v] = T.lam[q][v];
  long long n_points = (long long)c->S.nc * nq;
  const double* coords = c->fsrc_coords.p;
  const int* cells = c->fsrc_cells.p;
  const double* prm = c->fsrc_prm.p;
  double* f = c->forcing[which].p;
  unsigned int* flag = c->fsrc_flag.p;
  void* args[] = {&coords, &cells, lam, &n_points, &t, &prm, &f, &flag};
  CK(cudaMemsetAsync(flag, 0, sizeof(unsigned int), c->stream));
  if (n_points > 0) {
    const size_t id = c->prof.begin(PC_FORCING, c->stream);
    CK(cudaLaunchKernel((const void*)c->fsrc_kernel, dim3(nblk(n_points, kForcingBlock)), dim3(kForcingBlock), args, 0, c->stream));
    c->launch_check();
    c->prof.end(id, c->stream);
  }
  unsigned int nonzero = 0;
  CK(cudaMemcpyAsync(&nonzero, flag, sizeof(unsigned int), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  ++c->fsrc_evals;
  forcing_commit(c, which, nonzero != 0, true);
  return 0;
  NSB_CATCH(c)
}

int nsb_get_forcing(nsb_handle c, int which, double* f) {
  if (!c || !c->have_mesh) return fail(c, "nsb_get_forcing: no mesh uploaded");
  if (which != NSB_FORCING_NEW && which != NSB_FORCING_OLD)
    return fail(c, "nsb_get_forcing: which must be NSB_FORCING_NEW (0) or NSB_FORCING_OLD (1)");
  if (!f) return fail(c, "nsb_get_forcing: f is NULL");
  NSB_TRY
  CK(cudaSetDevice(c->device));
  const size_t n = forcing_len(c);
  if (!c->forcing_set[which]) {
    std::fill(f, f + n, 0.0);
    return 1;
  }
  CK(cudaMemcpyAsync(f, c->forcing[which].p, n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return 0;
  NSB_CATCH(c)
}

int nsb_forcing_info(nsb_handle c, int* has_source, int64_t* compiles, int64_t* evaluations, int* nvrtc_major, int* nvrtc_minor) {
  if (!c) return -1;
  g_nvrtc.load();
  if (has_source) *has_source = c->fsrc_lib != nullptr;
  if (compiles) *compiles = c->fsrc_compiles;
  if (evaluations) *evaluations = c->fsrc_evals;
  if (nvrtc_major) *nvrtc_major = g_nvrtc.major;
  if (nvrtc_minor) *nvrtc_minor = g_nvrtc.minor;
  return 0;
}

int nsb_check_forcing_source(int dim, const char* src, char* log, size_t log_size) {
  std::string e;
  std::vector<char> cubin;
  if (dim != 2 && dim != 3) e = "nsb_check_forcing_source: dim must be 2 or 3";
  else if (!src) e = "nsb_check_forcing_source: src is NULL";
  else e = compile_forcing(dim, src, "sm_100a", cubin);
  if (log && log_size) {
    const size_t n = std::min(e.size(), log_size - 1);
    std::memcpy(log, e.data(), n);
    log[n] = '\0';
  }
  return e.empty() ? 0 : -1;
}

int nsb_get_vector(nsb_handle c, int which, double* vg) {
  if (!c || !c->have_mesh) return fail(c, "no mesh uploaded");
  NSB_TRY
  CK(cudaSetDevice(c->device));
  double* d = vec_ptr(c, which);
  if (!d) return fail(c, "bad vector id");
  const Structure& S = c->S;
  if (c->nranks == 1) {
    CK(cudaMemcpyAsync(c->pin, d, (size_t)S.n_own_dofs() * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    std::memcpy(vg, c->pin, (size_t)S.n_own_dofs() * sizeof(double));
  } else {
    // collective: every rank receives the full vector (owned entries scattered to their global
    // positions, zero elsewhere, summed over the ranks)
    const size_t N = (size_t)(c->n_u + c->n_p);
    CK(cudaMemsetAsync(c->w_gather.p, 0, N * sizeof(double), c->stream));
    const int n = (int)S.n_own_dofs();
    k_scatter_vals<<<nblk(n, 256), 256, 0, c->stream>>>(n, c->d_own_gdof.p, d, c->w_gather.p);
    c->launch_check();
    CKN(g_nccl.AllReduce(c->w_gather.p, c->w_gather.p, N, ncclDouble, ncclSum, c->comm, c->stream));
    CK(cudaMemcpyAsync(vg, c->w_gather.p, N * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
  }
  return 0;
  NSB_CATCH(c)
}

int nsb_copy_vector(nsb_handle c, int dst, int src) {
  if (!c || !c->have_mesh) return fail(c, "no mesh uploaded");
  NSB_TRY
  CK(cudaSetDevice(c->device));
  double *d = vec_ptr(c, dst), *s = vec_ptr(c, src);
  if (!d || !s) return fail(c, "bad vector id");
  CK(cudaMemcpyAsync(d, s, c->S.n_own_dofs() * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
  halo_exchange(c, d);
  return 0;
  NSB_CATCH(c)
}

int nsb_axpy_vector(nsb_handle c, int dst, double alpha, int src) {
  if (!c || !c->have_mesh) return fail(c, "no mesh uploaded");
  NSB_TRY
  CK(cudaSetDevice(c->device));
  double *d = vec_ptr(c, dst), *s = vec_ptr(c, src);
  if (!d || !s) return fail(c, "bad vector id");
  const long long n = c->S.n_own_dofs();
  k_axpby<<<nblk(n, 256), 256, 0, c->stream>>>(n, alpha, s, 1.0, d);
  c->launch_check();
  halo_exchange(c, d);
  return 0;
  NSB_CATCH(c)
}

static int assemble_common(nsb_handle c, bool newton) {
  if (!c || !c->have_mesh) return fail(c, "no mesh uploaded");
  NSB_TRY
  CK(cudaSetDevice(c->device));
  if (c->dim == 2) launch_assemble<2>(c, newton);
  else launch_assemble<3>(c, newton);
  c->have_matrix = true;
  return 0;
  NSB_CATCH(c)
}

int nsb_assemble_linearized(nsb_handle c) { return assemble_common(c, false); }
int nsb_assemble_newton(nsb_handle c) { return assemble_common(c, true); }

int nsb_assemble_pressure_matrices(nsb_handle c) {
  if (!c || !c->have_mesh) return fail(c, "no mesh uploaded");
  NSB_TRY
  CK(cudaSetDevice(c->device));
  cudaStream_t st = c->stream;
  // pressure constraint flags in GLOBAL pressure numbering, from the current constraint set
  std::vector<unsigned char> pflag(c->n_p, 0);
  {
    std::vector<unsigned char> lf(c->S.n_tot_dofs());
    CK(cudaMemcpyAsync(lf.data(), c->cflag.p, lf.size(), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    for (int P = 0; P < c->S.np_own + c->S.np_ghost; ++P) pflag[c->S.pid_gid[P]] = lf[c->S.pid_xoff(P)];
    if (c->nranks > 1) {
      // merge flags across ranks (max) through a small device buffer
      DBuf<double> tmp;
      std::vector<double> f(pflag.begin(), pflag.end());
      tmp.upload(f, st);
      CKN(g_nccl.AllReduce(tmp.p, tmp.p, f.size(), ncclDouble, ncclMax, c->comm, st));
      CK(cudaMemcpyAsync(f.data(), tmp.p, f.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
      CK(cudaStreamSynchronize(st));
      for (size_t i = 0; i < f.size(); ++i) pflag[i] = f[i] != 0.0;
    }
  }
  host_pressure_matrices(c, pflag);
  // M_p on the device + Jacobi data
  upload_csr(c->h_Mp, c->Mp_ptr, c->Mp_col, c->Mp_val, c->Mp, st);
  std::vector<double> md(c->h_Mp.n);
  for (int i = 0; i < c->h_Mp.n; ++i)
    for (int k = c->h_Mp.ptr[i]; k < c->h_Mp.ptr[i + 1]; ++k)
      if (c->h_Mp.col[k] == i) md[i] = 1.0 / c->h_Mp.val[k];
  c->Mp_lmax = power_lmax_jacobi(c->h_Mp, md);
  c->Mp_dinv.upload(md, st);
  // multigrid hierarchy of K_p
  AmgHierarchy H;
  amg_setup(c->h_Kp, H);
  c->amg.clear();
  for (auto& L : H.levels) {
    auto D = std::make_unique<DevLevel>();
    D->n = L.A.n;
    D->lmax = L.lmax;
    upload_csr(L.A, D->Aptr, D->Acol, D->Aval, D->A, st);
    if (L.P.n) {
      upload_csr(L.P, D->Pptr, D->Pcol, D->Pval, D->P, st);
      upload_csr(L.R, D->Rptr, D->Rcol, D->Rval, D->R, st);
    }
    D->dinv.upload(L.dinv, st);
    for (DBuf<double>* v : {&D->x, &D->x2, &D->b, &D->d, &D->r}) { v->alloc(L.A.n); v->zero(st); }
    c->amg.push_back(std::move(D));
  }
  c->coarse_n = 0;
  if (!H.coarse_inv.empty()) {
    c->coarse_inv.upload(H.coarse_inv, st);
    c->coarse_n = H.levels.back().A.n;
  }
  const size_t np = (size_t)c->n_p;
  for (DBuf<double>* v : {&c->w_t, &c->w_y1, &c->w_m0, &c->w_m1, &c->w_md}) { v->alloc(np); v->zero(st); }
  CK(cudaStreamSynchronize(st));
  c->have_pressure = true;
  return 0;
  NSB_CATCH(c)
}

int nsb_rhs_norm(nsb_handle c, double* norm) {
  if (!c || !c->have_matrix) return fail(c, "no assembled system");
  NSB_TRY
  CK(cudaSetDevice(c->device));
  *norm = device_norm2(c, c->v_rhs.p, c->S.n_own_dofs());
  return 0;
  NSB_CATCH(c)
}

int nsb_solve(nsb_handle c, int max_it, double tol_rel, int n_tmp, int* iterations, double* residual) {
  if (!c || !c->have_matrix) return fail(c, "no assembled system");
  if (!c->have_pressure) return fail(c, "nsb_assemble_pressure_matrices has not been called");
  NSB_TRY
  CK(cudaSetDevice(c->device));
  int it = 0;
  double res = 0;
  if (c->lvF.roots.empty() || c->solves % c->opt.poly_refresh == 0) setup_velocity_pc(c);
  const double bnorm = device_norm2(c, c->v_rhs.p, c->S.n_own_dofs());
  int rc = gmres(c, max_it, tol_rel * bnorm, n_tmp > 2 ? n_tmp : 150, &it, &res);
  if (c->two_level && (rc == 1 || it > 100)) {
    // The two-level cycle is only a good preconditioner while the scaled velocity spectrum stays near the real axis; when
    // it stalls (developing convection in the 2-D cases) the robust single-level polynomial takes over for the rest of the
    // run -- and a solve the cycle failed on is repeated with it before non-convergence is reported to the caller, so
    // that the reference's fallback branches (cpp:1241-1286) only fire for reasons the reference would have too.
    c->cycle_disabled = true;
    if (rc == 1) {
      setup_velocity_pc(c);
      int it2 = 0;
      rc = gmres(c, max_it, tol_rel * bnorm, n_tmp > 2 ? n_tmp : 150, &it2, &res);
      it = it2;
    }
  }
  // constraints.distribute(x)   (cpp:566, 862)
  if (c->n_con) {
    k_scatter_vals<<<nblk(c->n_con, 256), 256, 0, c->stream>>>(c->n_con, c->c_idx.p, c->c_val.p, c->v_sol.p);
    c->launch_check();
  }
  halo_exchange(c, c->v_sol.p);
  CK(cudaStreamSynchronize(c->stream));
  ++c->solves;
  if (iterations) *iterations = it;
  if (residual) *residual = res;
  return rc;
  NSB_CATCH(c)
}

int nsb_get_matrix_values(nsb_handle c, double* vals) {
  if (!c || !c->have_matrix) return fail(c, "no assembled system");
  NSB_TRY
  CK(cudaSetDevice(c->device));
  CK(cudaMemcpyAsync(vals, c->vals.p, (size_t)c->S.nnz_local * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return 0;
  NSB_CATCH(c)
}

int nsb_get_pressure_matrix(nsb_handle c, int which, int64_t* n, int64_t* nnz, int32_t* rowptr, int32_t* col, double* val) {
  if (!c || !c->have_pressure) return fail(c, "pressure matrices not assembled");
  const HostCsr& A = which == 0 ? c->h_Mp : c->h_Kp;
  if (n) *n = A.n;
  if (nnz) *nnz = A.nnz();
  if (rowptr) std::copy(A.ptr.begin(), A.ptr.end(), rowptr);
  if (col) std::copy(A.col.begin(), A.col.end(), col);
  if (val) std::copy(A.val.begin(), A.val.end(), val);
  return 0;
}

int nsb_spmv(nsb_handle c, const double* xg, double* yg) {
  if (!c || !c->have_matrix) return fail(c, "no assembled system");
  NSB_TRY
  CK(cudaSetDevice(c->device));
  const Structure& S = c->S;
  std::vector<double> loc(S.n_tot_dofs());
  const int dim = c->dim;
  for (int A = 0; A < S.nn_own + S.nn_ghost; ++A)
    for (int k = 0; k < dim; ++k) loc[S.node_xoff(A) + k] = xg[S.node_gid[A] * dim + k];
  for (int P = 0; P < S.np_own + S.np_ghost; ++P) loc[S.pid_xoff(P)] = xg[c->n_u + S.pid_gid[P]];
  CK(cudaMemcpyAsync(c->w_pin.p, loc.data(), loc.size() * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  spmv_full(c, c->w_pin.p, c->w_tmp.p);
  std::vector<double> out(S.n_own_dofs());
  CK(cudaMemcpyAsync(out.data(), c->w_tmp.p, out.size() * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  for (int A = 0; A < S.nn_own; ++A)
    for (int k = 0; k < dim; ++k) yg[S.node_gid[A] * dim + k] = out[(size_t)dim * A + k];
  for (int P = 0; P < S.np_own; ++P) yg[c->n_u + S.pid_gid[P]] = out[(size_t)dim * S.nn_own + P];
  return 0;
  NSB_CATCH(c)
}

int nsb_apply_velocity_block(nsb_handle c, const double* xg, double* yg) {
  if (!c || !c->have_matrix) return fail(c, "no assembled system");
  NSB_TRY
  CK(cudaSetDevice(c->device));
  velocity_operator_apply(c, 0, 2, nullptr, xg, nullptr, yg, nullptr);     // the velocity block leads the global numbering
  return 0;
  NSB_CATCH(c)
}

// the checks shared by the inspection entries of one level
static int level_entry_check(nsb_handle c, int level, const char* what) {
  if (!c || !c->have_matrix) return fail(c, "no assembled system");
  if (c->nranks > 1) return fail(c, std::string(what) + ": single GPU only (global numbering of one rank's vectors)");
  if (level != 0 && level != 1) return fail(c, std::string(what) + ": level must be 0 (fine) or 1 (coarse)");
  return 0;
}

int nsb_get_velocity_operator(nsb_handle c, int level, int* precision, int64_t* tiles, int64_t* n_rows, int64_t* n_blocks,
                              int64_t* row_gid, int64_t* rowptr, int64_t* col_gid, double* vals) {
  if (int rc = level_entry_check(c, level, "nsb_get_velocity_operator")) return rc;
  NSB_TRY
  CK(cudaSetDevice(c->device));
  const Structure& S = c->S;
  const int prec = c->opt.precond_precision, PL = c->dim * c->dim;
  const int nn = level == 0 ? S.nn_own : S.np_own;
  if (precision) *precision = prec;
  if (tiles) *tiles = level == 0 ? c->n_stiles : c->cg.n_tiles;
  if (n_rows) *n_rows = nn;
  if (row_gid) for (int A = 0; A < nn; ++A) row_gid[A] = level == 0 ? S.node_gid[A] : S.pid_gid[A];
  std::vector<int> node, nbr;
  std::vector<double> v;
  if (prec != 64) {
    if (level == 0 && !c->vs_valid) return fail(c, "the packed velocity operator does not match the assembled system");
    if (level == 1 && !c->cg.valid) return fail(c, "the coarse operator has not been assembled (linearised systems with velocity_cycle = 2 only)");
    const VsDev D = level == 0 ? fine_dev(c) : coarse_dev(c);
    const int64_t nq = level == 0 ? c->vs_total_nq : c->cg.total_nq;
    const size_t nuq = level == 0 ? c->d_suniq_xoff.n : c->cg.uniq_xoff.n;
    if (prec == 16) unpack_level<__half>(c, D, nq, nuq, node, nbr, v);
    else unpack_level<float>(c, D, nq, nuq, node, nbr, v);
  }
  if (n_blocks) *n_blocks = (int64_t)node.size();
  std::vector<int64_t> rp(nn + 1, 0);
  for (int a : node) ++rp[a + 1];
  for (int A = 0; A < nn; ++A) rp[A + 1] += rp[A];
  if (rowptr) std::copy(rp.begin(), rp.end(), rowptr);
  std::vector<int64_t> cur(rp.begin(), rp.end() - 1);
  for (size_t i = 0; i < node.size(); ++i) {
    const int64_t k = cur[node[i]]++;
    if (col_gid) col_gid[k] = level == 0 ? S.node_gid[nbr[i]] : S.pid_gid[nbr[i]];
    if (vals) std::copy(v.begin() + i * PL, v.begin() + (i + 1) * PL, vals + k * PL);
  }
  return 0;
  NSB_CATCH(c)
}

int nsb_apply_velocity_operator(nsb_handle c, int level, int mode, const double coef[4], const double* x, const double* u, double* y,
                                double* poly) {
  if (int rc = level_entry_check(c, level, "nsb_apply_velocity_operator")) return rc;
  if (mode < 2 || mode > 4) return fail(c, "nsb_apply_velocity_operator: mode must be 2, 3 or 4");
  if (mode >= 3 && (!coef || !u || (mode == 3 && !poly))) return fail(c, "nsb_apply_velocity_operator: missing coefficients or vectors");
  if (level == 1 && !c->cg.valid) return fail(c, "the coarse operator has not been assembled (linearised systems with velocity_cycle = 2 only)");
  NSB_TRY
  CK(cudaSetDevice(c->device));
  velocity_operator_apply(c, level, mode, coef, x, u, y, poly);
  return 0;
  NSB_CATCH(c)
}

int nsb_get_velocity_pc_roots(nsb_handle c, int level, int* n, double* re, double* im) {
  if (int rc = level_entry_check(c, level, "nsb_get_velocity_pc_roots")) return rc;
  const auto& R = level_of(c, level).roots;
  const size_t k = (level == 1 && !c->two_level) ? 0 : R.size();
  if (n) *n = (int)k;
  for (size_t i = 0; i < k; ++i) {
    if (re) re[i] = R[i].first;
    if (im) im[i] = R[i].second;
  }
  return 0;
}

// the preconditioner as set up by the last solve: it exists, and the two-level cycle's coarse operator is the current one
static int pc_entry_check(nsb_handle c, const char* what) {
  if (int rc = level_entry_check(c, 0, what)) return rc;
  if (!c->have_pressure) return fail(c, "nsb_assemble_pressure_matrices has not been called");
  if (c->lvF.roots.empty()) return fail(c, std::string(what) + ": no preconditioner has been set up (call nsb_solve first)");
  if (c->two_level && !c->cg.valid) return fail(c, std::string(what) + ": the two-level cycle's coarse operator no longer matches the assembled system");
  return 0;
}

int nsb_apply_velocity_pc(nsb_handle c, const double* xg, double* yg) {
  if (int rc = pc_entry_check(c, "nsb_apply_velocity_pc")) return rc;
  NSB_TRY
  CK(cudaSetDevice(c->device));
  const size_t n = (size_t)c->S.n_own_dofs(), nu = (size_t)c->dim * c->S.nn_own;      // one GPU: local layout == global numbering
  CK(cudaMemcpyAsync(c->w_tmp.p, xg, n * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  apply_velocity_pc(c, c->w_tmp.p);
  CK(cudaMemcpyAsync(yg, c->w_poly.p, nu * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return 0;
  NSB_CATCH(c)
}

int nsb_apply_preconditioner(nsb_handle c, const double* xg, double* yg) {
  if (int rc = pc_entry_check(c, "nsb_apply_preconditioner")) return rc;
  NSB_TRY
  CK(cudaSetDevice(c->device));
  const size_t n = (size_t)c->S.n_own_dofs();
  CK(cudaMemcpyAsync(c->w_tmp.p, xg, n * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  precond_apply(c, c->w_tmp.p, c->w_in.p);
  CK(cudaMemcpyAsync(yg, c->w_in.p, n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return 0;
  NSB_CATCH(c)
}

int nsb_pressure_pc_info(nsb_handle c, double* mp_lambda_max, double* mass_coeff) {
  if (!c || !c->have_pressure) return fail(c, "pressure matrices not assembled");
  if (mp_lambda_max) *mp_lambda_max = c->Mp_lmax;
  if (mass_coeff) *mass_coeff = schur_mass_coeff(c);
  return 0;
}

int nsb_timer_start(nsb_handle c) {
  if (!c) return -1;
  cudaSetDevice(c->device);
  return cudaEventRecord(c->t0, c->stream) == cudaSuccess ? 0 : -1;
}
int nsb_timer_stop(nsb_handle c, double* ms) {
  if (!c) return -1;
  cudaSetDevice(c->device);
  cudaEventRecord(c->t1, c->stream);
  cudaEventSynchronize(c->t1);
  float t = 0;
  cudaEventElapsedTime(&t, c->t0, c->t1);
  if (ms) *ms = t;
  return 0;
}
int nsb_synchronize(nsb_handle c) {
  if (!c) return -1;
  cudaSetDevice(c->device);
  return cudaStreamSynchronize(c->stream) == cudaSuccess ? 0 : fail(c, "stream synchronize failed");
}
int nsb_profile_enable(nsb_handle c, int on) {
  if (!c) return -1;
  c->prof.collect(c->stream);
  c->prof.on = on != 0;
  return 0;
}
int nsb_profile_reset(nsb_handle c) {
  if (!c) return -1;
  c->prof.collect(c->stream);
  c->prof.reset();
  return 0;
}
int nsb_profile_get(nsb_handle c, const char* name, double* total_ms, int64_t* launches) {
  if (!c) return -1;
  c->prof.collect(c->stream);
  for (int i = 0; i < PC_N; ++i)
    if (std::strcmp(name, kProfNames[i]) == 0) {
      if (total_ms) *total_ms = c->prof.ms[i];
      if (launches) *launches = c->prof.cnt[i];
      return 0;
    }
  return fail(c, "unknown profile class");
}
/* host-only helpers exported for the CPU test-suite (no CUDA calls) ------------------------- */
/* builds the node-block structure of `rank`/`nranks` and exports the owned rows as scalar CSR
 * with global columns, the global row ids and the halo plan sizes.  Pass NULL arrays to query sizes. */
int nsb_test_build_pattern(int dim, int64_t n_vertices, const double* coords, int64_t n_cells,
                           const uint32_t* cell_vertices, const uint32_t* cell_dofs, int64_t n_u, int64_t n_p,
                           const int32_t* cell_part, int rank, int nranks, int64_t* n_rows, int64_t* nnz,
                           int64_t* rowptr, uint32_t* col, int64_t* row_gids, int64_t* n_ghost_dofs,
                           int64_t* n_send_dofs, int64_t* n_local_cells) {
  Structure S;
  const std::string e = build_structure(dim, n_vertices, coords, n_cells, cell_vertices, cell_dofs, n_u, n_p, cell_part, rank, nranks, S);
  if (!e.empty()) { std::fprintf(stderr, "nsb_test_build_pattern: %s\n", e.c_str()); return -1; }
  if (n_rows) *n_rows = S.n_own_dofs();
  if (nnz) *nnz = S.nnz_local;
  if (n_ghost_dofs) *n_ghost_dofs = S.n_tot_dofs() - S.n_own_dofs();
  if (n_local_cells) *n_local_cells = S.nc;
  if (n_send_dofs) {
    int64_t t = 0;
    for (size_t k = 0; k < S.peer.size(); ++k) t += (int64_t)S.send_nodes[k].size() * dim + (int64_t)S.send_pids[k].size();
    *n_send_dofs = t;
  }
  if (rowptr && col) {
    std::vector<int64_t> rp;
    std::vector<uint32_t> cl;
    export_pattern(S, rp, cl);
    std::copy(rp.begin(), rp.end(), rowptr);
    std::copy(cl.begin(), cl.end(), col);
  }
  if (row_gids) {
    std::vector<int64_t> g;
    export_row_gids(S, g);
    std::copy(g.begin(), g.end(), row_gids);
  }
  return 0;
}

/* halo plan of `rank`/`nranks` in GLOBAL DoF ids (two calls: first with NULL arrays for the sizes).
 * ghost_gdof: global DoF of every ghost entry in local vector order [u_ghost | p_ghost];
 * per peer k: send_u (velocity DoFs, node-major) / send_p (pressure DoFs) lists concatenated in peer order with
 * prefix arrays send_u_ptr / send_p_ptr [n_peers+1]; recv_u_count / recv_p_count = entries received from peer k,
 * which land contiguously, in peer order, in the u-ghost resp. p-ghost range. */
int nsb_test_halo_plan(int dim, int64_t n_vertices, const double* coords, int64_t n_cells, const uint32_t* cell_vertices,
                       const uint32_t* cell_dofs, int64_t n_u, int64_t n_p, const int32_t* cell_part, int rank, int nranks,
                       int64_t* n_ghost, int64_t* ghost_gdof, int32_t* n_peers, int32_t* peers, int64_t* send_u_ptr,
                       int64_t* send_u_gdof, int64_t* send_p_ptr, int64_t* send_p_gdof, int64_t* recv_u_count,
                       int64_t* recv_p_count) {
  Structure S;
  const std::string e = build_structure(dim, n_vertices, coords, n_cells, cell_vertices, cell_dofs, n_u, n_p, cell_part, rank, nranks, S);
  if (!e.empty()) { std::fprintf(stderr, "nsb_test_halo_plan: %s\n", e.c_str()); return -1; }
  if (n_ghost) *n_ghost = S.n_tot_dofs() - S.n_own_dofs();
  if (n_peers) *n_peers = (int32_t)S.peer.size();
  if (ghost_gdof) {
    int64_t k = 0;
    for (int A = S.nn_own; A < S.nn_own + S.nn_ghost; ++A)
      for (int c = 0; c < dim; ++c) ghost_gdof[k++] = S.node_gid[A] * dim + c;
    for (int P = S.np_own; P < S.np_own + S.np_ghost; ++P) ghost_gdof[k++] = n_u + S.pid_gid[P];
  }
  int64_t su = 0, sp = 0;
  for (size_t k = 0; k < S.peer.size(); ++k) {
    if (peers) peers[k] = S.peer[k];
    if (send_u_ptr) send_u_ptr[k] = su;
    if (send_p_ptr) send_p_ptr[k] = sp;
    for (int A : S.send_nodes[k])
      for (int c = 0; c < dim; ++c) { if (send_u_gdof) send_u_gdof[su] = S.node_gid[A] * dim + c; ++su; }
    for (int P : S.send_pids[k]) { if (send_p_gdof) send_p_gdof[sp] = n_u + S.pid_gid[P]; ++sp; }
    if (recv_u_count) recv_u_count[k] = (int64_t)S.recv_node_count[k] * dim;
    if (recv_p_count) recv_p_count[k] = S.recv_pid_count[k];
  }
  if (send_u_ptr) send_u_ptr[S.peer.size()] = su;
  if (send_p_ptr) send_p_ptr[S.peer.size()] = sp;
  return 0;
}

/* eigenvalues of an upper-Hessenberg matrix */
// host-only: builds rank's structure, its SpMV tile plan and the streamed-operator plan on top of it and checks every
// invariant the kernels rely on; out = {tiles, interior tiles, boundary tiles, padded velocity blocks, violations}
int nsb_test_tile_plan(int dim, int64_t n_vertices, const double* coords, int64_t n_cells, const uint32_t* cell_vertices,
                       const uint32_t* cell_dofs, int64_t n_u, int64_t n_p, const int32_t* cell_part, int rank, int nranks,
                       int64_t* out5) {
  Structure S;
  const std::string e = build_structure(dim, n_vertices, coords, n_cells, cell_vertices, cell_dofs, n_u, n_p,
                                        nranks > 1 ? cell_part : nullptr, rank, nranks, S);
  if (!e.empty()) { std::fprintf(stderr, "nsb_test_tile_plan: %s\n", e.c_str()); return -1; }
  TilePlan P;
  const TileLimits L{TILE_MAX_NODES, TILE_MAX_IDX, TILE_MAX_UNIQ, TILE_MAX_PUNIQ, VS_MAX_BLOCKS};
  const std::string e2 = build_tile_plan(S, L, P);
  if (!e2.empty()) { std::fprintf(stderr, "nsb_test_tile_plan: %s\n", e2.c_str()); return -1; }
  VsPlan V;
  const std::string e3 = build_vel_stream(S, P, V);
  if (!e3.empty()) { std::fprintf(stderr, "nsb_test_tile_plan: %s\n", e3.c_str()); return -1; }
  out5[0] = P.n_tiles(); out5[1] = (int64_t)P.tiles_int.size(); out5[2] = (int64_t)P.tiles_bnd.size();
  out5[3] = 4 * V.total_nq; out5[4] = verify_tile_plan(S, L, P) + verify_vel_stream(S, P, V);
  return 0;
}

// host-only: the coarse P1 level of rank `rank` (structure.cpp build_coarse) in GLOBAL ids, for the CPU tests.
// Two calls: NULL arrays for the sizes.  ends_gid[nn_own][2] = global pressure ids of the end vertices of every owned node,
// node_gid[nn_own]; vedge pairs (global pressure id of an owned vertex, global node id of a line node ending there);
// coarse neighbour lists of the owned vertices as (rowptr[np_own+1], global pressure ids), rows = vertex_gid[np_own].
int nsb_test_coarse_level(int dim, int64_t n_vertices, const double* coords, int64_t n_cells, const uint32_t* cell_vertices,
                          const uint32_t* cell_dofs, int64_t n_u, int64_t n_p, const int32_t* cell_part, int rank, int nranks,
                          int64_t* sizes4, int64_t* node_gid, int64_t* ends_gid, int64_t* vedge_pairs, int64_t* vertex_gid,
                          int64_t* cnbr_ptr, int64_t* cnbr_gid) {
  Structure S;
  const std::string e = build_structure(dim, n_vertices, coords, n_cells, cell_vertices, cell_dofs, n_u, n_p,
                                        nranks > 1 ? cell_part : nullptr, rank, nranks, S);
  if (!e.empty()) { std::fprintf(stderr, "nsb_test_coarse_level: %s\n", e.c_str()); return -1; }
  CoarseLevel C;
  const std::string e2 = build_coarse(S, C);
  if (!e2.empty()) { std::fprintf(stderr, "nsb_test_coarse_level: %s\n", e2.c_str()); return -1; }
  sizes4[0] = S.nn_own; sizes4[1] = (int64_t)C.vedge.size(); sizes4[2] = S.np_own; sizes4[3] = (int64_t)C.Sc.nbr.size();
  if (node_gid) for (int A = 0; A < S.nn_own; ++A) node_gid[A] = S.node_gid[A];
  if (ends_gid) for (size_t i = 0; i < C.node_ends.size(); ++i) ends_gid[i] = S.pid_gid[C.node_ends[i]];
  if (vedge_pairs)
    for (int P = 0; P < S.np_own; ++P)
      for (int64_t k = C.vedge_ptr[P]; k < C.vedge_ptr[P + 1]; ++k) { vedge_pairs[2 * k] = S.pid_gid[P]; vedge_pairs[2 * k + 1] = S.node_gid[C.vedge[k]]; }
  if (vertex_gid) for (int P = 0; P < S.np_own; ++P) vertex_gid[P] = S.pid_gid[P];
  if (cnbr_ptr) std::copy(C.Sc.nbr_ptr.begin(), C.Sc.nbr_ptr.end(), cnbr_ptr);
  if (cnbr_gid) for (size_t i = 0; i < C.Sc.nbr.size(); ++i) cnbr_gid[i] = S.pid_gid[C.Sc.nbr[i]];
  return 0;
}

int nsb_test_hessenberg_eigs(int n, const double* a, double* wr, double* wi) {
  std::vector<double> A(a, a + (size_t)n * n), r, i;
  if (!hessenberg_eigs(n, A, r, i)) return 1;
  std::copy(r.begin(), r.end(), wr);
  std::copy(i.begin(), i.end(), wi);
  return 0;
}

int nsb_solver_info(nsb_handle c, int* poly_degree, double* poly_probe_residual, int* amg_levels) {
  if (!c) return -1;
  if (poly_degree) {
    int d = 0;
    for (auto& r : c->lvF.roots) d += (r.second != 0.0) ? 2 : 1;
    *poly_degree = d;
  }
  if (poly_probe_residual) *poly_probe_residual = c->lvF.probe_res;
  if (amg_levels) *amg_levels = (int)c->amg.size();
  return 0;
}

int nsb_velocity_operator_info(nsb_handle c, int* precision, int64_t* value_bytes, int64_t* index_bytes, int64_t* tiles,
                               int64_t* blocks) {
  if (!c || !c->have_mesh) return fail(c, "no mesh uploaded");
  if (precision) *precision = c->opt.precond_precision;
  if (value_bytes) *value_bytes = (int64_t)vs_vals_bytes(c);
  if (index_bytes) *index_bytes = 16 * c->vs_total_nq + 64 * (int64_t)c->n_stiles + 4 * (int64_t)c->d_suniq_xoff.n;
  if (tiles) *tiles = c->n_stiles;
  if (blocks) *blocks = (int64_t)c->S.nbr.size();
  return 0;
}

int nsb_comm_info(nsb_handle c, int* nranks, int* halo_mode, int64_t* halo_doubles_per_exchange) {
  if (!c) return -1;
  if (nranks) *nranks = c->nranks;
  if (halo_mode) *halo_mode = c->nranks == 1 ? 0 : !c->ph.on ? 1 : 2;
  if (halo_doubles_per_exchange) {
    int64_t t = 0;
    for (size_t k = 0; k < c->S.peer.size(); ++k) t += (int64_t)c->S.send_nodes[k].size() * c->dim;
    *halo_doubles_per_exchange = t;
  }
  return 0;
}

int nsb_get_coarse_operator(nsb_handle c, int64_t* n_rows, int64_t* n_blocks, int64_t* row_gid, int64_t* rowptr, int64_t* col_gid,
                            double* vals) {
  if (!c || !c->have_mesh || !c->cg.built) return fail(c, "no coarse level");
  NSB_TRY
  CK(cudaSetDevice(c->device));
  const Coarse& G = c->cg;
  if (n_rows) *n_rows = (int64_t)G.gid.size();
  if (n_blocks) *n_blocks = (int64_t)G.h_nbr_gid.size();
  if (row_gid) std::copy(G.gid.begin(), G.gid.end(), row_gid);
  if (rowptr) std::copy(G.h_nbr_ptr.begin(), G.h_nbr_ptr.end(), rowptr);
  if (col_gid) std::copy(G.h_nbr_gid.begin(), G.h_nbr_gid.end(), col_gid);
  if (vals) {
    if (!G.valid) return fail(c, "the coarse operator has not been assembled (linearised systems with velocity_cycle = 2 only)");
    CK(cudaMemcpyAsync(vals, G.cvals.p, G.cvals.n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
  }
  return 0;
  NSB_CATCH(c)
}

int nsb_velocity_pc_info(nsb_handle c, int* two_level, int* smoother_degree, int* coarse_degree, int64_t* coarse_rows,
                         int64_t* coarse_value_bytes, double* fine_lambda_max) {
  if (!c) return -1;
  if (two_level) *two_level = c->two_level ? 1 : 0;
  if (smoother_degree) *smoother_degree = (int)c->lvF.roots.size();
  if (coarse_degree) *coarse_degree = c->two_level ? (int)c->lvC.roots.size() : 0;
  if (coarse_rows) *coarse_rows = c->lvC.n;
  if (coarse_value_bytes) *coarse_value_bytes = (int64_t)coarse_vals_bytes(c);
  if (fine_lambda_max) *fine_lambda_max = c->lvF.ritz_top;
  return 0;
}

int nsb_get_solver_opts(nsb_handle c, nsb_solver_opts* o) {
  if (!c || !o) return -1;
  *o = c->opt;
  return 0;
}

int nsb_get_run_state(nsb_handle c, int32_t* cycle_disabled) {
  if (!c || !cycle_disabled) return -1;
  if (!c->have_mesh) return fail(c, "nsb_get_run_state: no mesh uploaded");
  *cycle_disabled = c->cycle_disabled ? 1 : 0;
  return 0;
}

int nsb_set_run_state(nsb_handle c, int32_t cycle_disabled) {
  if (!c) return -1;
  if (!c->have_mesh) return fail(c, "nsb_set_run_state: no mesh uploaded (order: solver options, mesh, run state)");
  c->cycle_disabled = cycle_disabled != 0;
  return 0;
}

int nsb_launch_count(nsb_handle c, int64_t* n) {
  if (!c) return -1;
  *n = c->launches;
  return 0;
}

}  // extern "C"
