// mpas_b200.cu -- C ABI of libmpas_b200.so (include/mpas_b200.h): device mirror management,
// space-filling-curve renumbering, the task entry points and the atm_srk3 driver.
//
// Reference interfaces replaced (alexaiken/mpas-regent): the bodies of the leaf tasks in
// dynamics/dynamics_tasks.rg and of atm_srk3/atm_timestep in dynamics/rk_timestep.rg:361-519.
// There is no host compute path in this file: every task entry launches kernels (kernels.cuh).
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstddef>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <numeric>
#include <string>
#include <vector>

#include "kernels.cuh"
#ifdef MPASB200_LAB
#include "kernels_tiles.cuh"     // tile-staged k_dt_edge (TMA, de-duplicated columns): bit-identical, measured slower (profiles/r2_edge_tiles.md)
#endif
#include "kernels_init.cuh"
#include "kernels_jw.cuh"
#ifdef MPASB200_LAB
#include "kernels_staged.cuh"     // cp.async-staged gather kernels: measured slower than the plain ones (profiles/r2_staged_gathers.md)
#include "kernels_lab.cuh"
#endif

namespace {

struct FieldInfo { const char* name; int entity; int slots; };
const FieldInfo kFields[] = {
#define MPASB200_FIELD(name, entity, slots) {#name, MPASB200_##entity, slots},
#define MPASB200_VFIELD(name) {#name, MPASB200_VERTICAL, 1},
#include "../../include/mpas_b200_fields.def"
#undef MPASB200_FIELD
#undef MPASB200_VFIELD
};
const char* kTaskNames[MPASB200_T_COUNT] = {
    "rk_integration_setup", "compute_moist_coefficients", "compute_vert_imp_coefs", "compute_dyn_tend",
    "set_smlstep_pert_variables", "advance_acoustic_step", "divergence_damping_3d", "recover_large_step_variables",
    "compute_solve_diagnostics", "rk_dynamics_substep_finish", "advance_scalars"};

std::string g_create_error;

struct HaloList { int entity; int n; int* d_idx; };
struct Weights { int entity; int n; double* d_w; };      // mpasb200_register_weights, caller's numbering

}  // namespace

struct mpasb200 {
  MpasDims d; MpasConfig c;
  int device = 0;
  int nCells, nEdges, nVertices, L, LP, L1, CPB;
  int num_sms = 148;
  int dd_blocks_per_sm = 0;      // resident blocks of k_divdamp per SM (occupancy query, first launch)
  int max_smem_optin = 48 * 1024;
  View V;                               // device pointers
  std::vector<void*> allocs;            // everything cudaMalloc'ed
  int64_t bytes = 0;
  bool mesh_ok = false, mesh_started = false;
  std::map<std::string, std::vector<char>> mesh_stage;      // mpasb200_mesh_member: dense host copies of strided region members
  // renumbering: newOf[entity][old] = internal index (size n+1, pad -> pad)
  std::vector<int> newOf[3];
  // launch classes (MpasMeshPtrs.cellClass / edgeClass): internal numbering is class-major, classBegin[ent][c] .. classBegin[ent][c+1]
  int classBegin[3][5] = {{0, 0, 0, 0, 0}, {0, 0, 0, 0, 0}, {0, 0, 0, 0, 0}};
  int rangeB[3] = {0, 0, 0}, rangeE[3] = {0, 0, 0}; bool rangeSet[3] = {false, false, false};     // mpasb200_set_range
  int* d_newOf[3] = {nullptr, nullptr, nullptr};
  // staging
  double* d_stage = nullptr; size_t stage_elems = 0;
  double* h_stage = nullptr; size_t h_stage_elems = 0;
  // streams / timing
  cudaStream_t own_stream = nullptr, stream = nullptr;
  bool timing = false;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  // pipelined transfers: one staging buffer per field and direction, copies on their own streams
  cudaStream_t up_stream = nullptr, dn_stream = nullptr;
  struct Pipe { double* up = nullptr; double* dn = nullptr; cudaEvent_t up_copied = nullptr, up_scattered = nullptr, dn_gathered = nullptr,
                dn_copied = nullptr; bool up_used = false, dn_used = false; };
  std::vector<Pipe> pipe;
  double task_ms[MPASB200_T_COUNT] = {0}; int64_t task_calls[MPASB200_T_COUNT] = {0};
  int64_t launches = 0;
  bool capturing = false;
  // per-kernel CUDA-event timing (bench / profiling aid): event pairs recorded around every launch
  bool ktiming = false;
  std::vector<cudaEvent_t> ev_pool; size_t ev_used = 0;
  struct Pending { int stat; cudaEvent_t a, b; bool comm; };
  // timeline mode (mpasb200_enable_kernel_timing(h, 2)): start / end of every launch in ms since the mode was switched on, with its stream
  bool ktimeline = false; cudaEvent_t ktl_base = nullptr;
  struct TlEntry { int stat; float t0, t1; bool comm; };
  std::vector<TlEntry> timeline;
  std::vector<Pending> pending;
  struct KStat { std::string name; double ms; int64_t n; };
  std::vector<KStat> kstats;
  std::map<double, std::pair<cudaGraphExec_t, int64_t>> graphs;   // dt -> (exec, kernel launches per replay)
  std::vector<HaloList> lists;
  int* d_gid[3] = {nullptr, nullptr, nullptr}; int n_gid[3] = {0, 0, 0};   // mpasb200_set_global_ids
  SumAcc* d_acc = nullptr;
  std::vector<Weights> weights; IntAcc* d_iacc = nullptr; double* d_wv = nullptr;   // mpasb200_integrate
  double* d_iso = nullptr; size_t iso_elems = 0;      // mpasb200_isobaric_diagnostics output, grown on demand
  // distributed step (mpasb200_dist_*): NCCL communicator, halo lists, packed buffers, communication stream
  void* comm = nullptr; int rank = 0, world = 1;
  struct Halo { std::vector<int> peers_s, off_s, peers_r, off_r; int* d_s = nullptr; int* d_r = nullptr; int ns = 0, nr = 0; bool set = false; } halo[3];
  struct ExPart { int ent; std::vector<int> fields; int entries; double* sbuf = nullptr; double* rbuf = nullptr; };
  std::vector<ExPart> xplan[MPASB200_X_COUNT]; bool xplan_built = false;
  cudaStream_t comm_stream = nullptr; cudaEvent_t ev_ready = nullptr, ev_done = nullptr, ev_side = nullptr; bool x_pending = false; bool has_classes = false;
  EdgeTiles et = {nullptr, nullptr, nullptr, 0, 0, 0}; size_t et_smem = 0; int et_minb = 0, et_abl = 0;     // k_dt_edge_tile (MpasConfig.edge_tiles; laboratory builds), built by upload_mesh
  double* d_sflux = nullptr;            // horiz_flux_arr of atm_advance_scalars: [nScalars][(nEdges+1)][LP], allocated on first use
  std::string err;
  std::mutex mu;
};

namespace {

#define CK(call)                                                                                       \
  do {                                                                                                 \
    cudaError_t e_ = (call);                                                                           \
    if (e_ != cudaSuccess) {                                                                           \
      h->err = std::string(#call) + ": " + cudaGetErrorString(e_);                                     \
      return MPASB200_ECUDA;                                                                           \
    }                                                                                                  \
  } while (0)

int fail(mpasb200_t* h, int code, const std::string& msg) { if (h) h->err = msg; else g_create_error = msg; return code; }

template <class T> int dev_alloc(mpasb200_t* h, T** p, size_t n) {
  void* q = nullptr;
  size_t b = std::max<size_t>(n, 1) * sizeof(T);
  cudaError_t e = cudaMalloc(&q, b);
  if (e != cudaSuccess) { h->err = std::string("cudaMalloc: ") + cudaGetErrorString(e); return MPASB200_ENOMEM; }
  e = cudaMemsetAsync(q, 0, b, h->stream);
  if (e != cudaSuccess) { h->err = std::string("cudaMemset: ") + cudaGetErrorString(e); return MPASB200_ECUDA; }
  h->allocs.push_back(q); h->bytes += (int64_t)b; *p = (T*)q;
  return 0;
}
template <class T> int dev_upload(mpasb200_t* h, const T** dst, const std::vector<T>& src) {
  T* p = nullptr;
  int rc = dev_alloc(h, &p, src.size());
  if (rc) return rc;
  if (!src.empty()) CK(cudaMemcpyAsync(p, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));      // src is a temporary
  *dst = p;
  return 0;
}

int entity_count(const mpasb200_t* h, int ent) {
  return ent == MPASB200_CELL ? h->nCells : ent == MPASB200_EDGE ? h->nEdges : ent == MPASB200_VERTEX ? h->nVertices : 1;
}

// ---- space-filling curve -------------------------------------------------------------------------
inline uint64_t spread21(uint64_t v) {            // 21 bits -> every third bit
  v &= 0x1fffffULL;
  v = (v | v << 32) & 0x1f00000000ffffULL;
  v = (v | v << 16) & 0x1f0000ff0000ffULL;
  v = (v | v << 8) & 0x100f00f00f00f00fULL;
  v = (v | v << 4) & 0x10c30c30c30c30c3ULL;
  v = (v | v << 2) & 0x1249249249249249ULL;
  return v;
}
// Hilbert index of a 3-D lattice point (Skilling's transpose algorithm, 21 bits per axis), then
// interleaved to one 63-bit key.  Cells that are close on the sphere get close keys.
uint64_t hilbert3(uint32_t X0, uint32_t X1, uint32_t X2) {
  const int bits = 21;
  uint32_t X[3] = {X0, X1, X2};
  uint32_t M = 1u << (bits - 1), P, Q, t;
  for (Q = M; Q > 1; Q >>= 1) {
    P = Q - 1;
    for (int i = 0; i < 3; ++i) {
      if (X[i] & Q) X[0] ^= P;
      else { t = (X[0] ^ X[i]) & P; X[0] ^= t; X[i] ^= t; }
    }
  }
  for (int i = 1; i < 3; ++i) X[i] ^= X[i - 1];
  t = 0;
  for (Q = M; Q > 1; Q >>= 1) if (X[2] & Q) t ^= Q - 1;
  for (int i = 0; i < 3; ++i) X[i] ^= t;
  return (spread21(X[0]) << 2) | (spread21(X[1]) << 1) | spread21(X[2]);
}

// resolve a stored id to an (old-numbering) index with pad = n
inline int resolve(int id, int n, int policy) {
  long idx = (policy == MPASB200_INDEX_LITERAL) ? (long)id : (long)id - 1;
  if (idx < 0 || idx > n) idx = n;
  return (int)idx;
}

// out[new][w] = remap(resolve(src[old][w])); pad row -> all pads.  src null: ids are all 0 (rule M1).
std::vector<int> build_ids(const int32_t* src, int n, int w, const std::vector<int>& rowNew, int targetN,
                           const std::vector<int>& targetNew, int policy) {
  std::vector<int> out((size_t)(n + 1) * w, targetN);
  for (int o = 0; o < n; ++o) {
    const int r = rowNew[o];
    for (int j = 0; j < w; ++j) {
      const int id = src ? src[(size_t)o * w + j] : 0;
      out[(size_t)r * w + j] = targetNew[resolve(id, targetN, policy)];
    }
  }
  return out;
}
template <class T, class S> std::vector<T> build_vals(const S* src, int n, int w, const std::vector<int>& rowNew) {
  std::vector<T> out((size_t)(n + 1) * w, T(0));
  if (src)
    for (int o = 0; o < n; ++o) {
      const int r = rowNew[o];
      for (int j = 0; j < w; ++j) out[(size_t)r * w + j] = (T)src[(size_t)o * w + j];
    }
  return out;
}

// ---- launch helpers --------------------------------------------------------------------------------
struct Cfg { dim3 grid, block; };
// one thread per level PAIR: block = (LP/2, CPB) with CPB whole columns
Cfg cfg_for(const mpasb200_t* h, int n) { return Cfg{dim3((unsigned)((n + h->CPB - 1) / h->CPB)), dim3((unsigned)(h->LP / 2), (unsigned)h->CPB)}; }

cudaEvent_t pool_event(mpasb200_t* h) {
  if (h->ev_used == h->ev_pool.size()) { cudaEvent_t e; cudaEventCreate(&e); h->ev_pool.push_back(e); }
  return h->ev_pool[h->ev_used++];
}
int kstat_id(mpasb200_t* h, const char* name) {
  for (size_t i = 0; i < h->kstats.size(); ++i) if (h->kstats[i].name == name) return (int)i;
  h->kstats.push_back({name, 0.0, 0});
  return (int)h->kstats.size() - 1;
}
struct KTimer {      // brackets one launch with an event pair when kernel timing is on
  mpasb200_t* h; cudaEvent_t a = nullptr; int id = -1;
  KTimer(mpasb200_t* h_, const char* name) : h(h_) {
    if (h->ktiming && !h->capturing) { id = kstat_id(h, name); a = pool_event(h); cudaEventRecord(a, h->stream); }
  }
  ~KTimer() {
    if (a) { cudaEvent_t b = pool_event(h); cudaEventRecord(b, h->stream); h->pending.push_back({id, a, b, h->comm_stream && h->stream == h->comm_stream}); }   // same stream as `a`: one LAUNCH
  }
};
void drain_kernel_times(mpasb200_t* h) {
  if (h->pending.empty()) return;
  // events may sit on any stream the handle was pointed at (mpasb200_set_stream): wait for each pair itself
  for (auto& p : h->pending) {
    float ms = 0;
    if (cudaEventSynchronize(p.b) != cudaSuccess || cudaEventElapsedTime(&ms, p.a, p.b) != cudaSuccess) { cudaGetLastError(); continue; }
    h->kstats[p.stat].ms += ms; h->kstats[p.stat].n++;
    if (h->ktimeline && h->ktl_base) {
      float t0 = 0, t1 = 0;
      if (cudaEventElapsedTime(&t0, h->ktl_base, p.a) == cudaSuccess && cudaEventElapsedTime(&t1, h->ktl_base, p.b) == cudaSuccess) h->timeline.push_back({p.stat, t0, t1, p.comm});
      else cudaGetLastError();
    }
  }
  h->pending.clear(); h->ev_used = 0;
}

#define LAUNCH(kernel, n, smem, ...)                                                        \
  do {                                                                                      \
    if ((n) > 0) {                                                                          \
      Cfg cf_ = cfg_for(h, (n));                                                            \
      KTimer kt_(h, #kernel);                                                               \
      kernel<<<cf_.grid, cf_.block, (smem), h->stream>>>(__VA_ARGS__);                      \
      h->launches++;                                                                        \
    }                                                                                       \
  } while (0)

// staged gather kernels (kernels_staged.cuh): `slots` 16-byte shared-memory slots per thread + `tiles` column tiles
enum { GS_DT_EDGE = 1, GS_AC_GATHER = 2, GS_THETA_FLUX = 4, GS_CELLC = 8, GS_DIVDAMP = 16, GS_SMLSTEP = 32, GS_DIAG = 64 };
size_t staged_bytes(const mpasb200_t* h, int slots, int tiles) {
  const size_t tile = (((size_t)tiles * h->CPB * (h->LP + 2) + 1) & ~(size_t)1) * sizeof(double);
  return tile + (size_t)slots * 16 * (size_t)(h->LP / 2) * h->CPB;
}
#ifdef MPASB200_LAB
bool staged_on(const mpasb200_t* h, int bit, size_t smem) { return (h->c.gather_stage & bit) && smem <= (size_t)h->max_smem_optin && h->LP / 2 * h->CPB <= 224; }
#else
// the staged kernels exist in -DMPASB200_LAB builds only; the shipped library always takes the plain kernels
#define staged_on(h, bit, smem) false
#define LAUNCH_STAGED(kernel, n, smem, ...) do { } while (0)
#endif
#ifdef MPASB200_LAB
#define LAUNCH_STAGED(kernel, n, smem, ...)                                                 \
  do {                                                                                      \
    if ((n) > 0) {                                                                          \
      static bool attr_ = false;                                                            \
      if (!attr_) { cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, h->max_smem_optin); attr_ = true; } \
      Cfg cf_ = cfg_for(h, (n));                                                            \
      KTimer kt_(h, #kernel);                                                               \
      kernel<<<cf_.grid, cf_.block, (smem), h->stream>>>(__VA_ARGS__);                      \
      h->launches++;                                                                        \
    }                                                                                       \
  } while (0)
#endif
size_t tile_bytes(const mpasb200_t* h, int tiles) { return (size_t)tiles * h->CPB * (h->LP + 2) * sizeof(double); }
// dynamic shared memory of k_dt_theta_flux: the advection row of each column's edge (ids + coefficient pairs)
#define TF_SMEM(h) ((size_t)(h)->CPB * (h)->V.NAE * (sizeof(double2) + sizeof(int)))

#ifdef MPASB200_LAB
// k_dt_edge_tile (kernels_tiles.cuh): compiled for at most ET_MAXT threads per block, ET_MINB resident blocks
enum { ET_MAXT16 = 448, ET_MINB16 = 3, ET_MAXT8 = 224, ET_MINB8 = 5 };
void launch_dt_edge(mpasb200_t* h, const DynTendParams& P) {
  if (h->et.TE == 0) return;
  const int nT = (h->nEdges + h->et.TE - 1) / h->et.TE;
  const dim3 block((unsigned)(h->LP / 2), (unsigned)h->et.TE);
  KTimer kt_(h, "k_dt_edge_tile");
#define ET_GO(TE_, MT_, MB_) k_dt_edge_tile<TE_, MT_, MB_><<<nT, block, h->et_smem, h->stream>>>(h->V, P, h->et)
#ifdef MPASB200_LAB
  if (h->et_abl && h->et.TE == 16) { if (h->et_abl == 1) k_dt_edge_tile<16, ET_MAXT16, 2, 1><<<nT, block, h->et_smem, h->stream>>>(h->V, P, h->et); else k_dt_edge_tile<16, ET_MAXT16, 2, 2><<<nT, block, h->et_smem, h->stream>>>(h->V, P, h->et); }
  else if (h->et_abl) { if (h->et_abl == 1) k_dt_edge_tile<8, ET_MAXT8, ET_MINB8, 1><<<nT, block, h->et_smem, h->stream>>>(h->V, P, h->et); else k_dt_edge_tile<8, ET_MAXT8, ET_MINB8, 2><<<nT, block, h->et_smem, h->stream>>>(h->V, P, h->et); }
  else
#endif
  if (h->et.TE == 16 && h->et_minb == 2) ET_GO(16, ET_MAXT16, 2);
  else if (h->et.TE == 16) ET_GO(16, ET_MAXT16, ET_MINB16);
  else if (h->et_minb == 4) ET_GO(8, ET_MAXT8, 4);
  else ET_GO(8, ET_MAXT8, ET_MINB8);
#undef ET_GO
  h->launches++;
}
#define ET_ON(h) ((h)->et.TE != 0)
#else
#define ET_ON(h) false
#define launch_dt_edge(h, P) do { } while (0)
#endif

int post_launch(mpasb200_t* h) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { h->err = std::string("kernel launch: ") + cudaGetErrorString(e); return MPASB200_ECUDA; }
  return 0;
}

// ---- the tasks (internal: no locking, no timing) -------------------------------------------------------
int t_setup(mpasb200_t* h) {
  LAUNCH(k_setup_cell, h->nCells, 0, h->V);
  LAUNCH(k_setup_edge, h->nEdges, 0, h->V);
  if (h->c.config_scalar_advection && h->nCells > 0) {             // MPAS: scalars_2 = scalars_1
    Cfg cf = cfg_for(h, h->nCells); cf.grid.y = kFields[MPASB200_F_scalars].slots;
    KTimer kt_(h, "k_setup_scalars");
    k_setup_scalars<<<cf.grid, cf.block, 0, h->stream>>>(h->V);
    h->launches++;
  }
  return post_launch(h);
}
int ensure_sflux(mpasb200_t* h) {      // horiz_flux_arr scratch of atm_advance_scalars, allocated on first use
  if (h->d_sflux) return 0;
  if (h->capturing) return fail(h, MPASB200_ESTATE, "scalar flux scratch must exist before a graph capture");
  const size_t n = (size_t)(h->nEdges + 1) * h->LP * kFields[MPASB200_F_scalars].slots;
  cudaError_t e = cudaMalloc((void**)&h->d_sflux, n * sizeof(double));
  if (e != cudaSuccess) { h->err = std::string("cudaMalloc(scalar flux scratch): ") + cudaGetErrorString(e); return MPASB200_ENOMEM; }
  cudaMemsetAsync(h->d_sflux, 0, n * sizeof(double), h->stream);
  h->bytes += (int64_t)(n * sizeof(double));
  return 0;
}
// init chain on the device: atm_init_coupled_diagnostics (:651-725), mpas_reconstruct_2d (:1894-1948)
int t_init_coupled(mpasb200_t* h) {
  const double rcv = h->c.rgas / (h->c.cp - h->c.rgas);
  LAUNCH(k_icd_cell1, h->nCells, 0, h->V);
  LAUNCH(k_icd_edge, h->nEdges, 0, h->V);
  LAUNCH(k_icd_cell2, h->nCells, 0, h->V, h->c.rgas, rcv);
  return post_launch(h);
}
int t_reconstruct(mpasb200_t* h, int on_a_sphere) { LAUNCH(k_reconstruct, h->nCells, 0, h->V, on_a_sphere); return post_launch(h); }
// atm_advance_scalars (mpas_b200.h): per-edge horizontal fluxes into scratch, then the cell update
int t_scalars(mpasb200_t* h, double dt, int rk_step) {
  (void)rk_step;
  constexpr int NS = 8;
  static_assert(NS == 8, "nScalars");
  if (kFields[MPASB200_F_scalars].slots != NS) return fail(h, MPASB200_EINVAL, "advance_scalars is compiled for nScalars = 8 (constants.rg:42)");
  const size_t edgeSlot = (size_t)(h->nEdges + 1) * h->LP;
  if (int rc = ensure_sflux(h)) return rc;
  LAUNCH(k_scalar_flux<NS>, h->nEdges, 0, h->V, h->d_sflux, edgeSlot);
  LAUNCH(k_scalar_update<NS>, h->nCells, 0, h->V, h->d_sflux, edgeSlot, dt, h->c.config_coef_3rd_order);
  return post_launch(h);
}
int t_moist(mpasb200_t* h) { LAUNCH(k_moist, h->nCells, 0, h->V); return post_launch(h); }
int t_vert_imp(mpasb200_t* h, double dts) {
  const MpasConfig& C = h->c;
  const double dtseps = .5 * dts * (1.0 + C.config_epssm);
  const double rcv = C.rgas / (C.cp - C.rgas), c2 = C.cp * rcv;
  LAUNCH(k_vert_imp, h->nCells, tile_bytes(h, 2), h->V, dtseps, c2, rcv, C.gravity);
  return post_launch(h);
}
int t_diag(mpasb200_t* h, int hollingsworth, int rk_step) {
  LAUNCH(k_diag_vertex, h->nVertices, 0, h->V);
  LAUNCH(k_diag_cell, h->nCells, 0, h->V);
  const bool recon = !(rk_step != -1 && rk_step != 2);
  if (recon) LAUNCH(k_diag_edge<true>, h->nEdges, 0, h->V); else LAUNCH(k_diag_edge<false>, h->nEdges, 0, h->V);
  if (hollingsworth) {
    LAUNCH(k_diag_ke_vertex, h->nVertices, 0, h->V);
    LAUNCH(k_diag_ke_holl, h->nCells, 0, h->V);
  }
  return post_launch(h);
}
int t_dyn_tend(mpasb200_t* h, int rk_step, double dt, int mixing, double cam_coef, int mix_full, int rayleigh_u) {
  const MpasConfig& C = h->c;
  DynTendParams P;
  std::memset(&P, 0, sizeof(P));
  P.rk_step = rk_step; P.mixing = mixing; P.mix_full = mix_full; P.rayleigh_u = rayleigh_u;
  double h_mom4 = C.config_h_mom_eddy_visc4, h_th4 = C.config_h_theta_eddy_visc4;
  if (rk_step == 0 && mixing == MPASB200_MIX_2D_SMAGORINSKY) {
    h_mom4 = C.config_visc4_2dsmag * pow(C.config_len_disp, 3.0);        // :889-890
    h_th4 = h_mom4;
  }
  P.h_mom_eddy_visc4 = h_mom4; P.h_theta_eddy_visc4 = h_th4;
  // the reference tests h_mom_eddy_visc4 for the u and w filters and h_theta_eddy_visc4 for theta; with the
  // shipped constants both switch together.  Mixed settings are refused rather than silently merged.
  if ((h_mom4 > 0.0) != (h_th4 > 0.0)) return fail(h, MPASB200_EINVAL, "h_mom_eddy_visc4 and h_theta_eddy_visc4 must be enabled together");
  P.visc4_on = h_mom4 > 0.0;
  P.cam_on = cam_coef > 0.0;
  P.v_mom_eddy_visc2 = C.config_v_mom_eddy_visc2; P.v_theta_eddy_visc2 = C.config_v_theta_eddy_visc2;
  P.vmix_u_on = P.v_mom_eddy_visc2 > 0.0; P.vmix_t_on = P.v_theta_eddy_visc2 > 0.0;
  P.kdiff_scale = pow(C.config_smagorinsky_coef * C.config_len_disp, 2.0);
  P.kdiff_cap = (0.01 * pow(C.config_len_disp, 2.0)) * (1.0 / dt);
  P.prandtl_inv = 1.0 / C.prandtl; P.r_earth = C.sphere_radius; P.inv_r_earth = 1.0 / C.sphere_radius;
  P.omega2 = 2.0 * C.omega; P.gravity = C.gravity; P.del4u_div_factor = C.config_del4u_div_factor;
  P.rayleigh_levels = C.config_number_rayleigh_damp_u_levels;
  P.rayleigh_coef_inverse = 1.0 / ((double)(C.config_number_rayleigh_damp_u_levels) * (C.config_rayleigh_damp_u_timescale_days * 86400.0));
  // two column tiles + the static rows of the theta loops (k_dt_cellC<false> stages them; the <true> form leaves the space unused)
  const size_t sm2 = tile_bytes(h, 2) + (size_t)h->CPB * h->d.maxEdges * (2 * sizeof(double) + 3 * sizeof(int));
  const size_t sm_edge = staged_bytes(h, 20, 1), sm_flux = staged_bytes(h, 10, 0);
  if (rk_step == 0) {
    LAUNCH(k_dt_cell0<true>, h->nCells, 0, h->V, P, C.config_len_disp, cam_coef);
    LAUNCH(k_dt_edge_delsq, h->nEdges, 0, h->V);
    if (P.visc4_on) {
      LAUNCH(k_dt_vertex_delsq, h->nVertices, 0, h->V);
      LAUNCH(k_dt_cell_delsq, h->nCells, 0, h->V);
    }
    LAUNCH(k_dt_edge_euler, h->nEdges, tile_bytes(h, 1), h->V, P);
    if (staged_on(h, GS_DT_EDGE, sm_edge)) LAUNCH_STAGED(k_dt_edge_s<10>, h->nEdges, sm_edge, h->V, P);
    else if (ET_ON(h)) launch_dt_edge(h, P);
    else LAUNCH(k_dt_edge, h->nEdges, tile_bytes(h, 1), h->V, P);
    LAUNCH(k_dt_cellA, h->nCells, 0, h->V, P);
    LAUNCH(k_dt_cellB, h->nCells, 0, h->V, P);
    if (staged_on(h, GS_THETA_FLUX, sm_flux)) LAUNCH_STAGED(k_dt_theta_flux_s<10>, h->nEdges, sm_flux, h->V);
    else LAUNCH(k_dt_theta_flux, h->nEdges, TF_SMEM(h), h->V);
    if (h->c.kernel_forms & 1) { LAUNCH((k_dt_cellC<true, 1>), h->nCells, sm2, h->V, P); LAUNCH((k_dt_cellC<true, 2>), h->nCells, sm2, h->V, P); }
    else LAUNCH(k_dt_cellC<true>, h->nCells, sm2, h->V, P);
  } else {
    LAUNCH(k_dt_cell0<false>, h->nCells, 0, h->V, P, C.config_len_disp, cam_coef);
    if (staged_on(h, GS_DT_EDGE, sm_edge)) LAUNCH_STAGED(k_dt_edge_s<10>, h->nEdges, sm_edge, h->V, P);
    else if (ET_ON(h)) launch_dt_edge(h, P);
    else LAUNCH(k_dt_edge, h->nEdges, tile_bytes(h, 1), h->V, P);
    if (staged_on(h, GS_THETA_FLUX, sm_flux)) LAUNCH_STAGED(k_dt_theta_flux_s<10>, h->nEdges, sm_flux, h->V);
    else LAUNCH(k_dt_theta_flux, h->nEdges, TF_SMEM(h), h->V);
    if (h->c.kernel_forms & 1) { LAUNCH((k_dt_cellC<false, 1>), h->nCells, sm2, h->V, P); LAUNCH((k_dt_cellC<false, 2>), h->nCells, sm2, h->V, P); }
    else LAUNCH(k_dt_cellC<false>, h->nCells, sm2, h->V, P);
  }
  return post_launch(h);
}
// mpasb200_set_range: the acoustic step and the divergence damping run on [begin, end) of the cells / edges
struct Range { int b, e, n; bool whole; };
Range range_of(const mpasb200_t* h, int ent, int n) {
  if (!h->rangeSet[ent]) return Range{0, n, n, true};
  const int b = std::min(h->rangeB[ent], n), e = std::min(h->rangeE[ent], n);
  return Range{b, e, std::max(0, e - b), b == 0 && e == n};
}
View ranged(const mpasb200_t* h, const Range& r) { View v = h->V; v.xoff = r.b; v.xend = r.e; return v; }
int t_smlstep(mpasb200_t* h) { LAUNCH(k_smlstep, h->nCells, 0, h->V, h->c.nRelaxZone); return post_launch(h); }
int t_acoustic(mpasb200_t* h, double dts, int small_step) {
  const double epssm = h->c.config_epssm;
  const double resm = (1.0 - epssm) / (1.0 + epssm);
  const Range rc_ = range_of(h, MPASB200_CELL, h->nCells), re_ = range_of(h, MPASB200_EDGE, h->nEdges);
  const View Vc = ranged(h, rc_), Ve = ranged(h, re_);
  const size_t sm_gather = staged_bytes(h, 12, 0);
  if (h->c.physics_mode == MPASB200_PHYSICS_CORRECTED) {        // edge update, flux gather, column solve with back-substitution
    const double rcv = h->c.rgas / (h->c.cp - h->c.rgas), c2 = h->c.cp * rcv;
    if (small_step == 0) LAUNCH(k_acoustic_u<true>, re_.n, 0, Ve, dts, c2, h->c.gravity);
    else LAUNCH(k_acoustic_u<false>, re_.n, 0, Ve, dts, c2, h->c.gravity);
    if (staged_on(h, GS_AC_GATHER, sm_gather)) LAUNCH_STAGED(k_acoustic_gather_s<6>, rc_.n, sm_gather, Vc, dts);
    else LAUNCH(k_acoustic_gather, rc_.n, 0, Vc, dts);
    if (small_step == 0) LAUNCH(k_acoustic_col<true>, rc_.n, tile_bytes(h, 6), Vc, dts, epssm, resm);
    else LAUNCH(k_acoustic_col<false>, rc_.n, tile_bytes(h, 6), Vc, dts, epssm, resm);
    return post_launch(h);
  }
  // acoustic_tma = 3 (default): lean gather kernel + the column-per-lane exact pipeline (k_acoustic_lane)
  {
    const size_t smem_lane = ((size_t)2 * (AF_COUNT + 2) * AL_COLS * AL_KC + (size_t)2 * AL_NOUT * AL_COLS * AL_KC + (size_t)4 * h->LP) * sizeof(double) + 64;
    if (!h->c.acoustic_exact && h->c.acoustic_tma == 3 && smem_lane <= (size_t)h->max_smem_optin) {
      if (rc_.n == 0) return 0;
      const View& V = Vc;
      AcPtrs F;
#define AF(n) F.p[AF_##n] = V.f[MPASB200_F_##n]
      AF(tend_rho); AF(theta_m); AF(w); AF(coftz); AF(cofwz); AF(cofwr); AF(cofwt); AF(a_tri); AF(alpha_tri); AF(zz); AF(rw_save); AF(rw);
      AF(dss); AF(rho_zz); AF(rho_pp); AF(rtheta_pp); AF(rw_p); AF(wwAvg);
#undef AF
      F.p[AF_rs] = V.scr_rs; F.p[AF_ts] = V.scr_ts;
      LAUNCH(k_acoustic_gather, rc_.n, 0, Vc, dts);
      static bool attr_ = false;
      if (!attr_) {
        cudaFuncSetAttribute(k_acoustic_lane<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->max_smem_optin);
        cudaFuncSetAttribute(k_acoustic_lane<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->max_smem_optin);
        attr_ = true;
      }
      const size_t smem0 = ((size_t)2 * ((int)AF_rho_pp + 1) * AL_COLS * AL_KC + (size_t)2 * AL_NOUT * AL_COLS * AL_KC + (size_t)4 * h->LP) * sizeof(double) + 64;
      const int tiles = (rc_.n + AL_COLS - 1) / AL_COLS;
      const dim3 grid(std::min(tiles, 2 * h->num_sms)), block(32 + AL_NMOV);      // persistent: two resident blocks per SM walk the tiles
      {
        KTimer kt_(h, small_step == 0 ? "k_acoustic_lane<true>" : "k_acoustic_lane<false>");
        if (small_step == 0) k_acoustic_lane<true><<<grid, block, smem0, h->stream>>>(V, F, dts, epssm, resm);
        else k_acoustic_lane<false><<<grid, block, smem_lane, h->stream>>>(V, F, dts, epssm, resm);
      }
      h->launches++;
      return post_launch(h);
    }
  }
  const bool tma_fits = ((size_t)AF_COUNT * h->LP + (size_t)4 * (h->LP + 2)) * sizeof(double) + 16 <= 48 * 1024 && h->LP / 2 <= 128;
  if (!h->c.acoustic_exact && h->c.acoustic_tma && h->nCells > 0 && tma_fits) {
    if (rc_.n == 0) return 0;
    const View& V = Vc;
    AcPtrs F;
#define AF(n) F.p[AF_##n] = V.f[MPASB200_F_##n]
    AF(tend_rho); AF(theta_m); AF(w); AF(coftz); AF(cofwz); AF(cofwr); AF(cofwt); AF(a_tri); AF(alpha_tri); AF(zz); AF(rw_save); AF(rw);
    AF(dss); AF(rho_zz); AF(rho_pp); AF(rtheta_pp); AF(rw_p); AF(wwAvg);
#undef AF
    F.p[AF_rs] = V.scr_rs; F.p[AF_ts] = V.scr_ts;
    const int split = h->c.acoustic_tma == 2;
    if (split) {
      if (staged_on(h, GS_AC_GATHER, sm_gather)) LAUNCH_STAGED(k_acoustic_gather_s<6>, rc_.n, sm_gather, Vc, dts);
      else LAUNCH(k_acoustic_gather, rc_.n, 0, Vc, dts);
    }
    const int T = h->LP / 2, NF = small_step == 0 ? (int)AF_rho_pp : (int)AF_COUNT;
    int C = 4;                               // columns per block: as many as fit the default 48 KB of dynamic shared memory
    auto smem_for = [&](int c) { return ((size_t)NF * c * h->LP + (size_t)4 * c * (h->LP + 2)) * sizeof(double) + 16; };
    while (C > 1 && (smem_for(C) > 48 * 1024 || C * T > 128)) C /= 2;
    const size_t smem = smem_for(C);
    dim3 block(T, C), grid((rc_.n + C - 1) / C);
    {
      KTimer kt_(h, small_step == 0 ? "k_acoustic_tma<true>" : "k_acoustic_tma<false>");
      if (small_step == 0) { if (split) k_acoustic_tma<true, 8><<<grid, block, smem, h->stream>>>(V, F, dts, epssm, resm);
                             else k_acoustic_tma<true, 0><<<grid, block, smem, h->stream>>>(V, F, dts, epssm, resm); }
      else { if (split) k_acoustic_tma<false, 8><<<grid, block, smem, h->stream>>>(V, F, dts, epssm, resm);
             else k_acoustic_tma<false, 0><<<grid, block, smem, h->stream>>>(V, F, dts, epssm, resm); }
    }
    h->launches++;
    return post_launch(h);
  }
  if (!h->c.acoustic_exact) {
    if (small_step == 0) LAUNCH(k_acoustic<true>, rc_.n, tile_bytes(h, 4), Vc, dts, epssm, resm);
    else LAUNCH(k_acoustic<false>, rc_.n, tile_bytes(h, 4), Vc, dts, epssm, resm);
    return post_launch(h);
  }
  if (!rc_.whole) return fail(h, MPASB200_ESTATE, "acoustic_exact does not support mpasb200_set_range");
  if (h->nCells > 0) {
    const int rows = std::max(1, 128 / h->LP);      // two-kernel exact mode: one thread per level
    KTimer kt_(h, "k_acoustic_flux");
    k_acoustic_flux<<<(h->nCells + rows - 1) / rows, dim3(h->LP, rows), 0, h->stream>>>(h->V, dts, small_step);
    h->launches++;
  }
  if (h->nCells > 0) {
    const int tb = 64;
    KTimer kt_(h, "k_acoustic_column");
    k_acoustic_column<<<(h->nCells + tb - 1) / tb, tb, 0, h->stream>>>(h->V, dts, small_step, epssm, resm);
    h->launches++;
  }
  return post_launch(h);
}
int t_divdamp(mpasb200_t* h, double dts) {
  const double rdts = 1.0 / dts;
  const double coef_divdamp = 2.0 * h->c.config_smdiv * h->c.config_len_disp * rdts;
  const Range re_ = range_of(h, MPASB200_EDGE, h->nEdges);
  if (re_.n > 0) {            // persistent: the resident blocks loop over the edge tiles
    const int tiles = (re_.n + h->CPB - 1) / h->CPB;
    KTimer kt_(h, "k_divdamp");
    // persistent: exactly the blocks that are resident at once walk the tiles (the 9 per SM of round 1 ran as two waves at 56 registers:
    // 1.084 -> 0.995 ms per step on x1.163842)
    if (h->dd_blocks_per_sm == 0) {
      int nb = 0;
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_divdamp, (h->LP / 2) * h->CPB, 0) != cudaSuccess || nb < 1) { cudaGetLastError(); nb = 5; }
      h->dd_blocks_per_sm = nb;
    }
    k_divdamp<<<std::min(tiles, h->num_sms * h->dd_blocks_per_sm), dim3(h->LP / 2, h->CPB), 0, h->stream>>>(ranged(h, re_), coef_divdamp);
    h->launches++;
  }
  return post_launch(h);
}
int t_recover(mpasb200_t* h, int ns, int rk_step, double dt) {
  const MpasConfig& C = h->c;
  const double invNs = 1 / (double)(ns);
  const double rcv = C.rgas / (C.cp - C.rgas);
  k_rec_pad<<<1, h->LP, 0, h->stream>>>(h->V); h->launches++;
  const int fix = C.physics_mode == MPASB200_PHYSICS_CORRECTED;
  LAUNCH(k_rec_cell1, h->nCells, 0, h->V, invNs, rk_step, dt, C.rgas, rcv, fix);
  LAUNCH(k_rec_edge, h->nEdges, 0, h->V, invNs, fix);
  LAUNCH(k_rec_cell2, h->nCells, (size_t)h->CPB * 34 * sizeof(double), h->V, C.nRelaxZone, fix);
  return post_launch(h);
}
int t_finish(mpasb200_t* h, int substep, int split) {
  const double inv = 1.0 / (double)(split);
  const int lt = substep < split, first = substep == 1, last = substep == split;
  LAUNCH(k_finish_cell, h->nCells, 0, h->V, lt, first, last, inv);
  LAUNCH(k_finish_edge, h->nEdges, 0, h->V, lt, first, last, inv);
  return post_launch(h);
}

// atm_srk3  rk_timestep.rg:361-500
int t_srk3(mpasb200_t* h, double dt) {
  const MpasConfig& C = h->c;
  const int number_of_sub_steps = C.number_of_sub_steps;
  const int dynamics_split = C.config_dynamics_split_steps;
  const double dt_dynamics = dt;
  const double rk_timestep[3] = {dt_dynamics / 3, dt_dynamics / 2, dt_dynamics};                         // :386-389
  const double rk_sub_timestep[3] = {dt_dynamics / 3, dt_dynamics / number_of_sub_steps, dt_dynamics / number_of_sub_steps};
  const int number_sub_steps[3] = {std::max(1, number_of_sub_steps / 2), std::max(1, number_of_sub_steps / 2), number_of_sub_steps};
  int rc;
  // per-task CUDA-event timing inside the driver (off while a graph is being captured)
  const bool tm = h->timing && !h->capturing;
#define T(task, call)                                                                   \
  do {                                                                                  \
    if (tm) cudaEventRecord(h->ev0, h->stream);                                         \
    rc = (call);                                                                        \
    if (tm) {                                                                           \
      cudaEventRecord(h->ev1, h->stream); cudaEventSynchronize(h->ev1);                 \
      float ms_ = 0; cudaEventElapsedTime(&ms_, h->ev0, h->ev1);                        \
      h->task_ms[task] += ms_; h->task_calls[task]++;                                   \
    }                                                                                   \
    if (rc) return rc;                                                                  \
  } while (0)
  T(MPASB200_T_SETUP, t_setup(h));                                         // :404
  T(MPASB200_T_MOIST, t_moist(h));                                         // :408
  T(MPASB200_T_VERT_IMP, t_vert_imp(h, rk_sub_timestep[0]));               // :417
  for (int rk_step = 0; rk_step < 3; ++rk_step) {                          // :426
    if (rk_step == 1) T(MPASB200_T_VERT_IMP, t_vert_imp(h, rk_sub_timestep[rk_step]));   // :429-434
    const int rk_arg = (C.rkarg_policy == MPASB200_RKARG_SUBSTEP_TRUNC) ? (int)rk_sub_timestep[rk_step] : rk_step;   // :437 (Q3)
    T(MPASB200_T_DYN_TEND, t_dyn_tend(h, rk_arg, dt, C.config_horiz_mixing, C.config_mpas_cam_coef, C.config_mix_full, C.config_rayleigh_damp_u));
    T(MPASB200_T_SMLSTEP, t_smlstep(h));                                   // :441
    for (int small_step = 0; small_step < number_sub_steps[rk_step] + 1; ++small_step) {   // :450 (Q4)
      T(MPASB200_T_ACOUSTIC, t_acoustic(h, rk_sub_timestep[rk_step], small_step));
      T(MPASB200_T_DIVDAMP, t_divdamp(h, rk_sub_timestep[rk_step]));
    }
    // :459-460 atm_recover_large_step_variables is commented out in the reference (Q5); CORRECTED calls it as commented
    if (C.physics_mode == MPASB200_PHYSICS_CORRECTED) T(MPASB200_T_RECOVER, t_recover(h, number_sub_steps[rk_step], rk_step, dt));
    // :465 "SKIPPING if (config_scalar_advection ...)": the call MPAS makes here, with rk_timestep[rk_step] (:386-389)
    if (C.config_scalar_advection) T(MPASB200_T_SCALARS, t_scalars(h, rk_timestep[rk_step], rk_step));
    T(MPASB200_T_DIAG, t_diag(h, 0, rk_step));                             // :467
  }
  T(MPASB200_T_FINISH, t_finish(h, 1, dynamics_split));                    // :481
#undef T
  return 0;
}

// ---- entry wrapper: lock, device, optional event timing ---------------------------------------------------
struct Entry {
  mpasb200_t* h; int task; bool timed; std::unique_lock<std::mutex> lk;
  Entry(mpasb200_t* h_, int task_) : h(h_), task(task_), timed(false), lk(h_->mu) {
    cudaSetDevice(h->device);
    if (h->timing && task >= 0 && !h->capturing) { cudaEventRecord(h->ev0, h->stream); timed = true; }
  }
  int done(int rc) {
    if (timed) {
      cudaEventRecord(h->ev1, h->stream);
      cudaEventSynchronize(h->ev1);
      float ms = 0; cudaEventElapsedTime(&ms, h->ev0, h->ev1);
      h->task_ms[task] += ms; h->task_calls[task]++;
    }
    return rc;
  }
};
#define REQUIRE_MESH() if (!h) return MPASB200_EINVAL; if (!h->mesh_ok) return fail(h, MPASB200_ESTATE, "upload_mesh has not been called")

int ensure_stage(mpasb200_t* h, size_t elems) {
  if (h->stage_elems >= elems) return 0;
  double* p = nullptr;
  cudaError_t e = cudaMalloc((void**)&p, elems * sizeof(double));
  if (e != cudaSuccess) { h->err = std::string("cudaMalloc(staging): ") + cudaGetErrorString(e); return MPASB200_ENOMEM; }
  if (h->d_stage) cudaFree(h->d_stage);
  h->d_stage = p; h->stage_elems = elems;
  return 0;
}
int ensure_hstage(mpasb200_t* h, size_t elems) {
  if (h->h_stage_elems >= elems) return 0;
  double* p = nullptr;
  cudaError_t e = cudaMallocHost((void**)&p, elems * sizeof(double));
  if (e != cudaSuccess) { h->err = std::string("cudaMallocHost: ") + cudaGetErrorString(e); return MPASB200_ENOMEM; }
  if (h->h_stage) cudaFreeHost(h->h_stage);
  h->h_stage = p; h->h_stage_elems = elems;
  return 0;
}


// ---- NCCL, loaded on first use (dlopen): the single-GPU library has no NCCL dependency ---------------------------------------
struct NcclId128 { char b[128]; };        // ncclUniqueId (passed BY VALUE to ncclCommInitRank)
struct NcclApi {
  void* lib = nullptr; bool tried = false; std::string err;
  int (*GetUniqueId)(void*) = nullptr;
  int (*CommInitRank)(void**, int, NcclId128, int) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  int (*GroupStart)() = nullptr; int (*GroupEnd)() = nullptr;
  int (*Send)(const void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*Recv)(void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
NcclApi g_nccl;
std::mutex g_nccl_mu;
bool nccl_load() {
  std::unique_lock<std::mutex> lk(g_nccl_mu);
  if (g_nccl.tried) return g_nccl.lib != nullptr;
  g_nccl.tried = true;
  void* lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!lib) { g_nccl.err = std::string("dlopen(libnccl.so.2): ") + dlerror(); return false; }
#define SYM(member, name) *(void**)(&g_nccl.member) = dlsym(lib, name); if (!g_nccl.member) { g_nccl.err = std::string("dlsym ") + name; return false; }
  SYM(GetUniqueId, "ncclGetUniqueId"); SYM(CommInitRank, "ncclCommInitRank"); SYM(CommDestroy, "ncclCommDestroy");
  SYM(GroupStart, "ncclGroupStart"); SYM(GroupEnd, "ncclGroupEnd"); SYM(Send, "ncclSend"); SYM(Recv, "ncclRecv");
  SYM(GetErrorString, "ncclGetErrorString");
#undef SYM
  g_nccl.lib = lib;
  return true;
}
#define NCK(call)                                                                                      \
  do {                                                                                                 \
    int r_ = (call);                                                                                   \
    if (r_ != 0) { h->err = std::string(#call) + ": " + g_nccl.GetErrorString(r_); return MPASB200_ECUDA; } \
  } while (0)
enum { NCCL_F64 = 8 };

void dist_release(mpasb200_t* h) {
  for (int k = 0; k < MPASB200_X_COUNT; ++k) { for (auto& p : h->xplan[k]) { if (p.sbuf) cudaFree(p.sbuf); if (p.rbuf) cudaFree(p.rbuf); } h->xplan[k].clear(); }
  for (int e = 0; e < 3; ++e) { if (h->halo[e].d_s) cudaFree(h->halo[e].d_s); if (h->halo[e].d_r) cudaFree(h->halo[e].d_r); h->halo[e].d_s = h->halo[e].d_r = nullptr; }
  if (h->comm && g_nccl.CommDestroy) { g_nccl.CommDestroy(h->comm); h->comm = nullptr; }
  if (h->ev_ready) { cudaEventDestroy(h->ev_ready); h->ev_ready = nullptr; }
  if (h->ev_done) { cudaEventDestroy(h->ev_done); h->ev_done = nullptr; }
  if (h->ev_side) { cudaEventDestroy(h->ev_side); h->ev_side = nullptr; }
  if (h->comm_stream) { cudaStreamDestroy(h->comm_stream); h->comm_stream = nullptr; }
}

// which fields travel at which point of the step (mirrors parallel.EXCHANGES / EXCHANGES_CORRECTED; SURVEY.md 8e, Appendix B)
int dist_build_plans(mpasb200_t* h) {
  if (h->xplan_built) return 0;
  const bool corr = h->c.physics_mode == MPASB200_PHYSICS_CORRECTED;
  auto F = [](std::initializer_list<int> l) { return std::vector<int>(l); };
  std::vector<std::pair<int, std::vector<int>>> spec[MPASB200_X_COUNT];
  spec[MPASB200_X_ACOUSTIC_FIRST] = {{MPASB200_CELL, corr ? F({MPASB200_F_w, MPASB200_F_rtheta_pp, MPASB200_F_rtheta_pp_old, MPASB200_F_rho_pp, MPASB200_F_rw_p, MPASB200_F_wwAvg})
                                                          : F({MPASB200_F_w, MPASB200_F_rtheta_pp, MPASB200_F_rtheta_pp_old})}};
  spec[MPASB200_X_ACOUSTIC] = {{MPASB200_CELL, corr ? F({MPASB200_F_rtheta_pp, MPASB200_F_rtheta_pp_old, MPASB200_F_rho_pp, MPASB200_F_rw_p, MPASB200_F_wwAvg})
                                                    : F({MPASB200_F_rtheta_pp, MPASB200_F_rtheta_pp_old})}};
  spec[MPASB200_X_DIAG] = {{MPASB200_CELL, F({MPASB200_F_ke, MPASB200_F_divergence})}, {MPASB200_EDGE, F({MPASB200_F_pv_edge, MPASB200_F_v})},
                           {MPASB200_VERTEX, F({MPASB200_F_vorticity})}};
  spec[MPASB200_X_RECOVER] = {{MPASB200_CELL, F({MPASB200_F_w})}, {MPASB200_EDGE, F({MPASB200_F_u, MPASB200_F_ru, MPASB200_F_ruAvg})}};
  spec[MPASB200_X_SCALARS] = {{MPASB200_CELL, F({MPASB200_F_scalars})}};
  for (int k = 0; k < MPASB200_X_COUNT; ++k)
    for (auto& sp : spec[k]) {
      mpasb200_t::ExPart p; p.ent = sp.first; p.fields = sp.second; p.entries = 0;
      for (int f : p.fields) p.entries += kFields[f].slots;
      const mpasb200_t::Halo& H = h->halo[p.ent];
      const size_t row = (size_t)p.entries * h->L1;
      CK(cudaMalloc((void**)&p.sbuf, std::max<size_t>(1, (size_t)H.ns * row) * sizeof(double)));
      CK(cudaMalloc((void**)&p.rbuf, std::max<size_t>(1, (size_t)H.nr * row) * sizeof(double)));
      h->bytes += (int64_t)(((size_t)H.ns + H.nr) * row * sizeof(double));
      h->xplan[k].push_back(p);
    }
  h->xplan_built = true;
  return 0;
}
int dist_pack_unpack(mpasb200_t* h, const mpasb200_t::ExPart& p, bool pack) {
  const mpasb200_t::Halo& H = h->halo[p.ent];
  const int n = pack ? H.ns : H.nr;
  if (n == 0) return 0;
  PackArgs A; A.nf = 0;
  const size_t slotStride = (size_t)(entity_count(h, p.ent) + 1) * h->LP;
  for (int f : p.fields) for (int sl = 0; sl < kFields[f].slots; ++sl) A.f[A.nf++] = h->V.f[f] + sl * slotStride;
  const int rows = std::max(1, 128 / h->LP);
  dim3 block(h->LP, rows), grid((n + rows - 1) / rows, A.nf);
  KTimer kt_(h, pack ? "k_pack" : "k_unpack");
  if (pack) k_pack<<<grid, block, 0, h->stream>>>(A, H.d_s, n, h->L1, h->LP, p.sbuf);
  else k_unpack<<<grid, block, 0, h->stream>>>(A, H.d_r, n, h->L1, h->LP, p.rbuf);
  h->launches++;
  return 0;
}
// pack -> one NCCL group -> unpack, all on the communication stream; the compute stream continues at once
// the communication stream joins the compute stream's order here (everything enqueued on compute so far is visible to it)
int dist_fork(mpasb200_t* h) {
  CK(cudaEventRecord(h->ev_ready, h->stream));
  CK(cudaStreamWaitEvent(h->comm_stream, h->ev_ready, 0));
  return 0;
}
int dist_start(mpasb200_t* h, int kind, bool forked = false) {
  if (!h->comm) return fail(h, MPASB200_ESTATE, "mpasb200_dist_init has not been called");
  if (int rc = dist_build_plans(h)) return rc;
  if (h->x_pending) return fail(h, MPASB200_ESTATE, "an exchange is still travelling (dist_flush first)");
  if (!forked) { if (int rc = dist_fork(h)) return rc; }
  cudaStream_t compute = h->stream;
  h->stream = h->comm_stream;
  int rc = 0;
  for (auto& p : h->xplan[kind]) if ((rc = dist_pack_unpack(h, p, true))) break;
  if (!rc) {
    KTimer kt_(h, "nccl_send_recv");
    int nrc = g_nccl.GroupStart();
    for (auto& p : h->xplan[kind]) {
      const mpasb200_t::Halo& H = h->halo[p.ent];
      const size_t row = (size_t)p.entries * h->L1;
      for (size_t i = 0; i < H.peers_s.size() && !nrc; ++i)
        if (H.off_s[i + 1] > H.off_s[i]) nrc = g_nccl.Send(p.sbuf + (size_t)H.off_s[i] * row, (size_t)(H.off_s[i + 1] - H.off_s[i]) * row, NCCL_F64, H.peers_s[i], h->comm, h->comm_stream);
      for (size_t i = 0; i < H.peers_r.size() && !nrc; ++i)
        if (H.off_r[i + 1] > H.off_r[i]) nrc = g_nccl.Recv(p.rbuf + (size_t)H.off_r[i] * row, (size_t)(H.off_r[i + 1] - H.off_r[i]) * row, NCCL_F64, H.peers_r[i], h->comm, h->comm_stream);
    }
    const int erc = g_nccl.GroupEnd();
    if (nrc || erc) { h->err = std::string("NCCL send/recv: ") + g_nccl.GetErrorString(nrc ? nrc : erc); rc = MPASB200_ECUDA; }
  }
  if (!rc) for (auto& p : h->xplan[kind]) if ((rc = dist_pack_unpack(h, p, false))) break;
  h->stream = compute;
  if (rc) return rc;
  CK(cudaEventRecord(h->ev_done, h->comm_stream));
  h->x_pending = true;
  return post_launch(h);
}
int dist_finish(mpasb200_t* h) {
  if (!h->x_pending) return 0;
  CK(cudaStreamWaitEvent(h->stream, h->ev_done, 0));
  h->x_pending = false;
  return 0;
}
int dist_exchange(mpasb200_t* h, int kind) { if (int rc = dist_start(h, kind)) return rc; return dist_finish(h); }

void set_ranges(mpasb200_t* h, int ent, int cls) {      // launch class -> range of mpasb200_set_range (cls < 0: everything)
  if (cls < 0) { h->rangeSet[ent] = false; return; }
  h->rangeB[ent] = h->classBegin[ent][cls]; h->rangeE[ent] = h->classBegin[ent][cls + 1]; h->rangeSet[ent] = true;
}
void set_empty(mpasb200_t* h, int ent) { h->rangeB[ent] = h->rangeE[ent] = 0; h->rangeSet[ent] = true; }

// atm_srk3 (rk_timestep.rg:361-500) on one rank of an N-rank run
int t_srk3_dist(mpasb200_t* h, double dt) {
  const MpasConfig& C = h->c;
  const int number_of_sub_steps = C.number_of_sub_steps, dynamics_split = C.config_dynamics_split_steps;
  const double rk_timestep[3] = {dt / 3, dt / 2, dt};
  const double rk_sub_timestep[3] = {dt / 3, dt / number_of_sub_steps, dt / number_of_sub_steps};
  const int number_sub_steps[3] = {std::max(1, number_of_sub_steps / 2), std::max(1, number_of_sub_steps / 2), number_of_sub_steps};
  const bool corr = C.physics_mode == MPASB200_PHYSICS_CORRECTED;
  const bool overlap = h->has_classes;
  const bool saved[2] = {h->rangeSet[MPASB200_CELL], h->rangeSet[MPASB200_EDGE]};
  if (saved[0] || saved[1]) return fail(h, MPASB200_ESTATE, "mpasb200_srk3_dist manages the launch ranges itself: clear mpasb200_set_range first");
  int rc;
#define R(call) do { if ((rc = (call))) { h->rangeSet[MPASB200_CELL] = h->rangeSet[MPASB200_EDGE] = false; return rc; } } while (0)
  R(t_setup(h)); R(t_moist(h));
  R(t_vert_imp(h, rk_sub_timestep[0]));
  R(dist_finish(h));                         // the diagnostics exchange of the previous step's last stage travelled under setup/moist/vert_imp
  for (int rk_step = 0; rk_step < 3; ++rk_step) {
    if (rk_step == 1) { R(t_vert_imp(h, rk_sub_timestep[rk_step])); R(dist_finish(h)); }
    const int rk_arg = (C.rkarg_policy == MPASB200_RKARG_SUBSTEP_TRUNC) ? (int)rk_sub_timestep[rk_step] : rk_step;
    R(t_dyn_tend(h, rk_arg, dt, C.config_horiz_mixing, C.config_mpas_cam_coef, C.config_mix_full, C.config_rayleigh_damp_u));
    R(t_smlstep(h));
    for (int small_step = 0; small_step < number_sub_steps[rk_step] + 1; ++small_step) {
      const double dts = rk_sub_timestep[rk_step];
      const int kind = small_step == 0 ? MPASB200_X_ACOUSTIC_FIRST : MPASB200_X_ACOUSTIC;
      if (!overlap) {
        R(t_acoustic(h, dts, small_step)); R(dist_exchange(h, kind)); R(t_divdamp(h, dts));
        continue;
      }
      if (corr) {                            // the edge update belongs to the task call: all edges once, before any cell
        set_empty(h, MPASB200_CELL); set_ranges(h, MPASB200_EDGE, -1);
        R(t_acoustic(h, dts, small_step));
        set_empty(h, MPASB200_EDGE);
      }
      // the owned cells some rank reads (a small launch) are advanced ON THE COMMUNICATION STREAM, at its high priority and
      // concurrently with the interior cells on the compute stream: the small launch does not leave the GPU half empty, and the
      // exchange starts as soon as those cells are done
      R(dist_fork(h));
      {
        cudaStream_t compute = h->stream;
        h->stream = h->comm_stream;
        set_ranges(h, MPASB200_CELL, 1);
        rc = t_acoustic(h, dts, small_step);
        h->stream = compute;
        if (rc) { h->rangeSet[MPASB200_CELL] = h->rangeSet[MPASB200_EDGE] = false; return rc; }
        CK(cudaEventRecord(h->ev_side, h->comm_stream));
      }
      R(dist_start(h, kind, true));                                                // ... they travel
      set_ranges(h, MPASB200_CELL, 0); R(t_acoustic(h, dts, small_step));          // ... under the interior cells
      CK(cudaStreamWaitEvent(h->stream, h->ev_side, 0));                           // interior edges touch sent cells too
      set_ranges(h, MPASB200_EDGE, 0); R(t_divdamp(h, dts));                       // ... and the interior edges
      R(dist_finish(h));
      set_ranges(h, MPASB200_EDGE, 1); R(t_divdamp(h, dts));                       // edges next to ghosts
      set_ranges(h, MPASB200_CELL, -1); set_ranges(h, MPASB200_EDGE, -1);
    }
    if (corr) { R(t_recover(h, number_sub_steps[rk_step], rk_step, dt)); R(dist_exchange(h, MPASB200_X_RECOVER)); }
    if (C.config_scalar_advection) { R(t_scalars(h, rk_timestep[rk_step], rk_step)); R(dist_exchange(h, MPASB200_X_SCALARS)); }
    R(t_diag(h, 0, rk_step));
    // read next by atm_compute_dyn_tend only: stages 0 and 2 let it travel under the column work in between
    if (overlap && rk_step != 1) R(dist_start(h, MPASB200_X_DIAG)); else R(dist_exchange(h, MPASB200_X_DIAG));
  }
  R(t_finish(h, 1, dynamics_split));
#undef R
  return 0;
}
}  // namespace

// =====================================================================================================
extern "C" {

void mpasb200_default_config(MpasConfig* c) {
  if (!c) return;
  std::memset(c, 0, sizeof(*c));
  c->rgas = 287.0; c->cp = 7.0 * c->rgas / 2.0; c->cv = c->cp - c->rgas;                // constants.rg:33-35
  c->gravity = 9.80616; c->omega = 7.29212E-5; c->sphere_radius = 6371229.0; c->prandtl = 1.0;
  c->config_epssm = 0.1; c->config_smdiv = 0.1; c->config_len_disp = 120000.0;
  c->config_smagorinsky_coef = 0.125; c->config_visc4_2dsmag = 0.05; c->config_del4u_div_factor = 10.0;
  c->config_rayleigh_damp_u_timescale_days = 5.0; c->config_mpas_cam_coef = 0.0;
  c->config_number_rayleigh_damp_u_levels = 6;
  c->config_horiz_mixing = MPASB200_MIX_2D_SMAGORINSKY;
  c->nRelaxZone = 5; c->number_of_sub_steps = 2; c->config_dynamics_split_steps = 1;
  c->index_policy = MPASB200_INDEX_CORRECTED; c->rkarg_policy = MPASB200_RKARG_SUBSTEP_TRUNC;
  c->sfc_renumber = 1; c->device = -1; c->use_graph = 0; c->acoustic_exact = 0; c->acoustic_tma = 3;
  c->physics_mode = MPASB200_PHYSICS_LITERAL;
  c->gather_stage = 0;
  c->config_scalar_advection = 0; c->config_coef_3rd_order = 0.25;        // constants.rg:59
  c->edge_tiles = 0; c->kernel_forms = 0; c->reserved0 = 0;
}

const char* mpasb200_last_error(const mpasb200_t* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int mpasb200_create(const MpasDims* dims, const MpasConfig* cfg, mpasb200_t** out) {
  if (!dims || !cfg || !out) return fail(nullptr, MPASB200_EINVAL, "null argument");
  if (dims->nCells < 0 || dims->nEdges < 0 || dims->nVertices < 0 || dims->nVertLevels < 3)
    return fail(nullptr, MPASB200_EINVAL, "bad dimensions (nVertLevels must be >= 3)");
  if (dims->maxEdges < 1 || dims->maxEdges > 16 || dims->nAdvCells < 1 || dims->vertexDegree != 3)
    return fail(nullptr, MPASB200_EINVAL, "unsupported maxEdges / nAdvCells / vertexDegree");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(nullptr, MPASB200_ENODEVICE, std::string("no CUDA device (") + cudaGetErrorString(e) + "); libmpas_b200 has no host path");
  mpasb200_t* h = new mpasb200();
  h->d = *dims; h->c = *cfg;
  if (cfg->device >= 0) h->device = cfg->device; else cudaGetDevice(&h->device);
  if ((e = cudaSetDevice(h->device)) != cudaSuccess) { g_create_error = std::string("cudaSetDevice: ") + cudaGetErrorString(e); delete h; return MPASB200_ECUDA; }
  h->nCells = dims->nCells; h->nEdges = dims->nEdges; h->nVertices = dims->nVertices;
  h->L = dims->nVertLevels; h->L1 = h->L + 1; h->LP = (h->L1 + 3) / 4 * 4;
  { const int T = h->LP / 2; int g = T, b = 32; while (b) { int t = g % b; g = b; b = t; } h->CPB = 32 / g; while (h->CPB * T < 128) h->CPB *= 2;
    while (h->CPB * T > 256 && h->CPB > 1) h->CPB /= 2; }      // several kernels are compiled for <= 256 threads per block
  if (h->LP / 2 * h->CPB > 256) { g_create_error = "nVertLevels too large for one block per column group"; delete h; return MPASB200_EINVAL; }
  cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, h->device);
  cudaDeviceGetAttribute(&h->max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, h->device);
  cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking);
  h->stream = h->own_stream;
  cudaEventCreate(&h->ev0); cudaEventCreate(&h->ev1);
  View& V = h->V;
  std::memset(&V, 0, sizeof(V));
  V.nCells = h->nCells; V.nEdges = h->nEdges; V.nVertices = h->nVertices; V.L = h->L; V.LP = h->LP;
  V.xoff = 0; V.xend = 0;      // set per launch by ranged() for the kernels that use PAIR_THREAD_R
  V.maxEdges = dims->maxEdges; V.maxEdges2 = dims->maxEdges2; V.vertexDegree = dims->vertexDegree; V.nAdv = dims->nAdvCells;
  V.cellSlot = (size_t)(h->nCells + 1) * h->LP;
  // one arena for every field (zero-filled: memory-model rule M1)
  size_t total = 0;
  std::vector<size_t> off(MPASB200_F_COUNT);
  for (int id = 0; id < MPASB200_F_COUNT; ++id) {
    size_t n = (kFields[id].entity == MPASB200_VERTICAL) ? (size_t)h->LP
                                                         : (size_t)(entity_count(h, kFields[id].entity) + 1) * h->LP * kFields[id].slots;
    n = (n + 15) / 16 * 16;     // keep every field 128-byte aligned
    off[id] = total; total += n;
  }
  const size_t scr = ((size_t)(h->nCells + 1) * h->LP + 15) / 16 * 16;
  double* arena = nullptr;
  const size_t scr_e = ((size_t)(h->nEdges + 1) * h->LP + 15) / 16 * 16;
  int rc = dev_alloc(h, &arena, total + 2 * scr + scr_e + (size_t)16 * h->LP);   // + slack: bulk strips of a last, partial tile
  if (rc) { g_create_error = h->err; mpasb200_destroy(h); return rc; }
  for (int id = 0; id < MPASB200_F_COUNT; ++id) V.f[id] = arena + off[id];
  V.scr_rs = arena + total; V.scr_ts = arena + total + scr; V.scr_flux = arena + total + 2 * scr;
  if (cudaStreamSynchronize(h->stream) != cudaSuccess) { g_create_error = "arena memset failed"; mpasb200_destroy(h); return MPASB200_ECUDA; }
  *out = h;
  return 0;
}

int mpasb200_destroy(mpasb200_t* h) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  for (auto& g : h->graphs) cudaGraphExecDestroy(g.second.first);
  for (auto e : h->ev_pool) cudaEventDestroy(e);
  for (void* p : h->allocs) cudaFree(p);
  for (auto& l : h->lists) if (l.d_idx) cudaFree(l.d_idx);
  if (h->d_stage) cudaFree(h->d_stage);
  if (h->h_stage) cudaFreeHost(h->h_stage);
  for (int e = 0; e < 3; ++e) if (h->d_gid[e]) cudaFree(h->d_gid[e]);
  if (h->d_acc) cudaFree(h->d_acc);
  for (auto& w : h->weights) if (w.d_w) cudaFree(w.d_w);
  if (h->d_iacc) cudaFree(h->d_iacc);
  if (h->d_wv) cudaFree(h->d_wv);
  if (h->d_iso) cudaFree(h->d_iso);
  if (h->d_sflux) cudaFree(h->d_sflux);
  dist_release(h);
  for (auto& pp : h->pipe) {
    if (pp.up) cudaFree(pp.up);
    if (pp.dn) cudaFree(pp.dn);
    for (cudaEvent_t e : {pp.up_copied, pp.up_scattered, pp.dn_gathered, pp.dn_copied}) if (e) cudaEventDestroy(e);
  }
  if (h->up_stream) cudaStreamDestroy(h->up_stream);
  if (h->dn_stream) cudaStreamDestroy(h->dn_stream);
  if (h->ktl_base) cudaEventDestroy(h->ktl_base);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  delete h;
  return 0;
}

#ifdef MPASB200_LAB
// ---- tile lists of k_dt_edge_tile (kernels_tiles.cuh): per tile of TE consecutive internal edges the distinct columns to stage
// (own edges first, then edgesOnEdge neighbours in first-use order, at most `cap`), per edge the staged slot of every neighbour.
namespace {
int build_edge_tiles(mpasb200_t* h, const std::vector<int>& eoe, const std::vector<int>& nEoE) {
  const int TE = h->c.edge_tiles % 100, minb_over = h->c.edge_tiles / 100 % 10, nE = h->nEdges, ME2 = h->d.maxEdges2, LP = h->LP;
  if (TE == 0 || nE == 0) return 0;
  if (TE != 8 && TE != 16) return fail(h, MPASB200_EINVAL, "edge_tiles must be 0, 8 or 16");
  const int maxt = TE == 16 ? ET_MAXT16 : ET_MAXT8, minb = (TE == 16 && minb_over == 2) ? 2 : (TE == 8 && minb_over == 4) ? 4 : (TE == 16 ? ET_MINB16 : ET_MINB8);
  h->et_minb = minb; h->et_abl = h->c.edge_tiles / 1000;      // ablations: laboratory build only
  if ((ME2 & 1) || LP / 2 * TE > maxt) { h->c.edge_tiles = 0; return 0; }      // shapes the tile kernel is not compiled for: plain kernel
  int smem_sm = 0;
  cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, h->device);
  const size_t fixed = ((size_t)TE * ME2 + (size_t)TE * (LP + 2)) * sizeof(double) + 16;
  const size_t per_block = std::min<size_t>((size_t)smem_sm / minb - 1024, (size_t)h->max_smem_optin);
  if (per_block < fixed + (size_t)TE * 2 * LP * sizeof(double)) { h->c.edge_tiles = 0; return 0; }
  int cap = (int)((per_block - fixed) / ((size_t)2 * LP * sizeof(double)));
  cap = std::min(cap, std::min(254, TE * (ME2 + 1)));
  const int SP = (ME2 + 15) / 16 * 16;
  const int nT = (nE + TE - 1) / TE;
  std::vector<int> cols((size_t)nT * cap, nE), ncols(nT, 0);
  std::vector<unsigned char> slot((size_t)(nE + 1) * SP, 255);
  std::vector<int> slotOf((size_t)nE + 1, -1);
  for (int t = 0; t < nT; ++t) {
    int* cl = cols.data() + (size_t)t * cap;
    int nc = TE;                                        // own edges: slot = local index (entries past nEdges stay the pad column)
    for (int i = 0; i < TE; ++i) { const int e = t * TE + i; if (e < nE) { cl[i] = e; slotOf[e] = i; } }
    for (int i = 0; i < TE; ++i) {
      const int e = t * TE + i;
      if (e >= nE) break;
      const int n = std::min(nEoE[e], ME2);
      for (int j = 0; j < n; ++j) {
        const int id = eoe[(size_t)e * ME2 + j];
        if (slotOf[id] < 0 && nc < cap) { slotOf[id] = nc; cl[nc++] = id; }
        if (slotOf[id] >= 0) slot[(size_t)e * SP + j] = (unsigned char)slotOf[id];
      }
    }
    ncols[t] = nc;
    for (int i = 0; i < nc; ++i) slotOf[cl[i]] = -1;
  }
  int rc;
  if ((rc = dev_upload<int>(h, &h->et.cols, cols))) return rc;
  if ((rc = dev_upload<int>(h, &h->et.ncols, ncols))) return rc;
  if ((rc = dev_upload<unsigned char>(h, &h->et.slot, slot))) return rc;
  h->et.cap = cap; h->et.SP = SP; h->et.TE = TE;
  h->et_smem = fixed + (size_t)cap * 2 * LP * sizeof(double);
#define ET_ATTR(TE_, MT_, MB_) cudaFuncSetAttribute(k_dt_edge_tile<TE_, MT_, MB_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->et_smem)
  cudaError_t e = (TE == 16 && minb == 2) ? ET_ATTR(16, ET_MAXT16, 2) : (TE == 16) ? ET_ATTR(16, ET_MAXT16, ET_MINB16)
                  : (minb == 4) ? ET_ATTR(8, ET_MAXT8, 4) : ET_ATTR(8, ET_MAXT8, ET_MINB8);
#undef ET_ATTR
#ifdef MPASB200_LAB
  cudaFuncSetAttribute(k_dt_edge_tile<16, ET_MAXT16, 2, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->et_smem);
  cudaFuncSetAttribute(k_dt_edge_tile<16, ET_MAXT16, 2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->et_smem);
  cudaFuncSetAttribute(k_dt_edge_tile<8, ET_MAXT8, ET_MINB8, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->et_smem);
  cudaFuncSetAttribute(k_dt_edge_tile<8, ET_MAXT8, ET_MINB8, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->et_smem);
#endif
  if (e != cudaSuccess) return fail(h, MPASB200_ECUDA, std::string("k_dt_edge_tile shared memory: ") + cudaGetErrorString(e));
  return 0;
}
}  // namespace
#endif

int mpasb200_upload_mesh(mpasb200_t* h, const MpasMeshPtrs* m) {
  if (!h || !m) return MPASB200_EINVAL;
  std::unique_lock<std::mutex> lk(h->mu);
  cudaSetDevice(h->device);
  if (h->mesh_ok) return fail(h, MPASB200_ESTATE, "upload_mesh may be called once per handle");
  // a failed upload leaves a half-built mirror (its allocations are released by mpasb200_destroy): the handle is unusable
  if (h->mesh_started) return fail(h, MPASB200_ESTATE, "a previous upload_mesh failed on this handle; destroy it and create a new one");
  h->mesh_started = true;
  if (!m->nEdgesOnCell || !m->edgesOnCell || !m->cellsOnEdge || !m->verticesOnEdge || !m->edgesOnVertex)
    return fail(h, MPASB200_EINVAL, "nEdgesOnCell, edgesOnCell, cellsOnEdge, verticesOnEdge, edgesOnVertex are required");
  const int nC = h->nCells, nE = h->nEdges, nV = h->nVertices, pol = h->c.index_policy;
  const int ME = h->d.maxEdges, ME2 = h->d.maxEdges2, VD = h->d.vertexDegree, NA = h->d.nAdvCells;
  for (int c = 0; c < nC; ++c)
    if (m->nEdgesOnCell[c] < 0 || m->nEdgesOnCell[c] > ME) return fail(h, MPASB200_EINVAL, "nEdgesOnCell out of range");
  if (m->nEdgesOnEdge) for (int e = 0; e < nE; ++e)
    if (m->nEdgesOnEdge[e] < 0 || m->nEdgesOnEdge[e] > ME2) return fail(h, MPASB200_EINVAL, "nEdgesOnEdge out of range");
  if (m->nAdvCellsForEdge) for (int e = 0; e < nE; ++e)
    if (m->nAdvCellsForEdge[e] < 0 || m->nAdvCellsForEdge[e] > NA) return fail(h, MPASB200_EINVAL, "nAdvCellsForEdge out of range");
  if (m->kiteForCell) for (size_t i = 0; i < (size_t)nC * ME; ++i)
    if (m->kiteForCell[i] < 0 || m->kiteForCell[i] >= VD) return fail(h, MPASB200_EINVAL, "kiteForCell out of range");

  // ---- renumbering: cells along a Hilbert curve, edges and vertices by the cells they touch
  std::vector<int>& cNew = h->newOf[MPASB200_CELL]; std::vector<int>& eNew = h->newOf[MPASB200_EDGE]; std::vector<int>& vNew = h->newOf[MPASB200_VERTEX];
  cNew.resize(nC + 1); eNew.resize(nE + 1); vNew.resize(nV + 1);
  std::iota(cNew.begin(), cNew.end(), 0); std::iota(eNew.begin(), eNew.end(), 0); std::iota(vNew.begin(), vNew.end(), 0);
  const bool sfc = h->c.sfc_renumber && m->xCell && m->yCell && m->zCell && nC > 0;
  const int nEnt[3] = {nC, nE, nV};
  for (int ent = 0; ent < 3; ++ent) { for (int c = 0; c < 5; ++c) h->classBegin[ent][c] = c ? nEnt[ent] : 0; h->rangeB[ent] = h->rangeE[ent] = 0; h->rangeSet[ent] = false; }
  if (sfc || m->cellClass || m->edgeClass) {
    // cells: class-major (if classes are given), then along the Hilbert curve (or in the caller's order)
    typedef std::pair<std::pair<int, uint64_t>, int> Key;
    std::vector<Key> key(nC);
    for (int c = 0; c < nC; ++c) {
      uint64_t hk = (uint64_t)c;
      if (sfc) {
        const double x = m->xCell[c], y = m->yCell[c], z = m->zCell[c];
        double r = std::sqrt(x * x + y * y + z * z); if (!(r > 0)) r = 1;
        auto q = [&](double t) { double u = (t / r + 1.0) * 0.5; u = std::min(std::max(u, 0.0), 1.0); return (uint32_t)(u * 2097151.0); };
        hk = hilbert3(q(x), q(y), q(z));
      }
      const int cls = m->cellClass ? m->cellClass[c] : 0;
      if (cls < 0 || cls > 3) return fail(h, MPASB200_EINVAL, "cellClass must be 0..3");
      key[c] = {{cls, hk}, c};
    }
    std::sort(key.begin(), key.end());
    for (int r = 0; r < nC; ++r) cNew[key[r].second] = r;
    if (m->cellClass) for (int c = 1; c < 5; ++c) {
      int cnt = 0; for (int i = 0; i < nC; ++i) cnt += (m->cellClass[i] < c);
      h->classBegin[MPASB200_CELL][c] = cnt;
    }
    std::vector<Key> ek(nE);
    for (int e = 0; e < nE; ++e) {
      const uint64_t a = cNew[resolve(m->cellsOnEdge[e * 2], nC, pol)], b = cNew[resolve(m->cellsOnEdge[e * 2 + 1], nC, pol)];
      const int cls = m->edgeClass ? m->edgeClass[e] : 0;
      if (cls < 0 || cls > 3) return fail(h, MPASB200_EINVAL, "edgeClass must be 0..3");
      ek[e] = {{cls, sfc ? ((std::min(a, b) << 32) | std::max(a, b)) : (uint64_t)e}, e};
    }
    std::sort(ek.begin(), ek.end());
    for (int r = 0; r < nE; ++r) eNew[ek[r].second] = r;
    if (m->edgeClass) for (int c = 1; c < 5; ++c) {
      int cnt = 0; for (int i = 0; i < nE; ++i) cnt += (m->edgeClass[i] < c);
      h->classBegin[MPASB200_EDGE][c] = cnt;
    }
  }
  if (sfc) {
    std::vector<std::pair<uint64_t, int>> vk(nV);
    for (int v = 0; v < nV; ++v) {
      uint64_t best = ~0ULL;
      for (int j = 0; j < VD; ++j) best = std::min<uint64_t>(best, (uint64_t)eNew[resolve(m->edgesOnVertex[v * VD + j], nE, pol)]);
      vk[v] = {best, v};
    }
    std::sort(vk.begin(), vk.end());
    for (int r = 0; r < nV; ++r) vNew[vk[r].second] = r;
  }
  int rc;
  for (int ent = 0; ent < 3; ++ent) {
    const int* p = nullptr;
    if ((rc = dev_upload<int>(h, &p, h->newOf[ent]))) return rc;
    h->d_newOf[ent] = const_cast<int*>(p);
  }
  View& V = h->V;
#define UP_IDS(member, src, n, w, rowNew, tN, tNew) if ((rc = dev_upload<int>(h, &V.member, build_ids(src, n, w, rowNew, tN, tNew, pol)))) return rc
#define UP_INT(member, src, n, w, rowNew) if ((rc = dev_upload<int>(h, &V.member, build_vals<int, int32_t>(src, n, w, rowNew)))) return rc
#define UP_DBL(member, src, n, w, rowNew) if ((rc = dev_upload<double>(h, &V.member, build_vals<double, double>(src, n, w, rowNew)))) return rc
  UP_INT(nEdgesOnCell, m->nEdgesOnCell, nC, 1, cNew);
  const int MEP = (ME + 3) / 4 * 4;
  V.MEP = MEP;
  {
    // edgesOnCell with a 16-byte-aligned row pitch, plus per-(cell, slot) copies of what a cell kernel needs
    // from its slot-i edge (cellsOnEdge, dvEdge, invDcEdge, meshScalingDel2/4, advection list): exact copies,
    // so the arithmetic is unchanged; they remove the second level of dependent index loads.
    const std::vector<int> eocC = build_ids(m->edgesOnCell, nC, ME, cNew, nE, eNew, pol);       // [new cell][ME] -> new edge
    const std::vector<int> coe = build_ids(m->cellsOnEdge, nE, 2, eNew, nC, cNew, pol);          // [new edge][2] -> new cell
    const std::vector<double> dvE = build_vals<double, double>(m->dvEdge, nE, 1, eNew), idcE = build_vals<double, double>(m->invDcEdge, nE, 1, eNew);
    const std::vector<double> ms2E = build_vals<double, double>(m->meshScalingDel2, nE, 1, eNew), ms4E = build_vals<double, double>(m->meshScalingDel4, nE, 1, eNew);
    const std::vector<int> nAdvE = build_vals<int, int32_t>(m->nAdvCellsForEdge, nE, 1, eNew);
    const std::vector<int> advE = build_ids(m->advCellsForEdge, nE, NA, eNew, nC, cNew, pol);
    const std::vector<double> acE = build_vals<double, double>(m->adv_coefs, nE, NA, eNew), a3E = build_vals<double, double>(m->adv_coefs_3rd, nE, NA, eNew);
    int nap = 2;
    for (int e = 0; e < nE; ++e) nap = std::max(nap, nAdvE[e]);
    nap = (nap + 1) / 2 * 2;
    V.NAP = nap;
    std::vector<int> eoc((size_t)(nC + 1) * MEP, nE), c1((size_t)(nC + 1) * MEP, nC), c2((size_t)(nC + 1) * MEP, nC);
    std::vector<double> dvS((size_t)(nC + 1) * ME, 0.0), idcS((size_t)(nC + 1) * ME, 0.0), ms2S((size_t)(nC + 1) * ME, 0.0), ms4S((size_t)(nC + 1) * ME, 0.0);
    std::vector<int> nAdvS((size_t)(nC + 1) * ME, 0), advS((size_t)(nC + 1) * ME * nap, nC);
    std::vector<double> acS((size_t)(nC + 1) * ME * nap, 0.0), a3S((size_t)(nC + 1) * ME * nap, 0.0);
    for (int c = 0; c <= nC; ++c)
      for (int i = 0; i < ME; ++i) {
        const int e = eocC[(size_t)c * ME + i];
        eoc[(size_t)c * MEP + i] = e;
        c1[(size_t)c * MEP + i] = coe[(size_t)e * 2]; c2[(size_t)c * MEP + i] = coe[(size_t)e * 2 + 1];
        dvS[(size_t)c * ME + i] = dvE[e]; idcS[(size_t)c * ME + i] = idcE[e]; ms2S[(size_t)c * ME + i] = ms2E[e]; ms4S[(size_t)c * ME + i] = ms4E[e];
        nAdvS[(size_t)c * ME + i] = nAdvE[e];
        for (int j = 0; j < nAdvE[e] && j < nap; ++j) {
          const size_t d = ((size_t)c * ME + i) * nap + j;
          advS[d] = advE[(size_t)e * NA + j]; acS[d] = acE[(size_t)e * NA + j]; a3S[d] = a3E[(size_t)e * NA + j];
        }
      }
    {   // per-edge advection rows with a 16-byte pitch (k_dt_theta_flux)
      const int nae = (NA + 3) / 4 * 4;
      V.NAE = nae;
      std::vector<int> idE((size_t)(nE + 1) * nae, nC);
      std::vector<double2> cfE((size_t)(nE + 1) * nae, make_double2(0.0, 0.0));
      for (int e = 0; e <= nE; ++e)
        for (int j = 0; j < NA; ++j) {
          idE[(size_t)e * nae + j] = advE[(size_t)e * NA + j];
          cfE[(size_t)e * nae + j] = make_double2(acE[(size_t)e * NA + j], a3E[(size_t)e * NA + j]);
        }
      if ((rc = dev_upload<int>(h, &V.advCellE, idE))) return rc;
      if ((rc = dev_upload<double2>(h, &V.advCoefE, cfE))) return rc;
    }
    if ((rc = dev_upload<int>(h, &V.edgesOnCell, eoc))) return rc;
    if ((rc = dev_upload<int>(h, &V.c1OnCell, c1))) return rc;
    if ((rc = dev_upload<int>(h, &V.c2OnCell, c2))) return rc;
    if ((rc = dev_upload<double>(h, &V.dvOnCell, dvS))) return rc;
    {   // dcEdge of the slot-i edge (k_diag_cell: one dependent scalar load less)
      const std::vector<double> dcE2 = build_vals<double, double>(m->dcEdge, nE, 1, eNew);
      std::vector<double> dcS((size_t)(nC + 1) * ME, 0.0);
      for (int c = 0; c <= nC; ++c)
        for (int i = 0; i < ME; ++i) dcS[(size_t)c * ME + i] = dcE2[eocC[(size_t)c * ME + i]];
      if ((rc = dev_upload<double>(h, &V.dcOnCell, dcS))) return rc;
    }
    if ((rc = dev_upload<double>(h, &V.invDcOnCell, idcS))) return rc;
    if ((rc = dev_upload<double>(h, &V.ms2OnCell, ms2S))) return rc;
    if ((rc = dev_upload<double>(h, &V.ms4OnCell, ms4S))) return rc;
    if ((rc = dev_upload<int>(h, &V.nAdvOnCell, nAdvS))) return rc;
    if ((rc = dev_upload<int>(h, &V.advCellOnCell, advS))) return rc;
    if ((rc = dev_upload<double>(h, &V.advCoefOnCell, acS))) return rc;
    if ((rc = dev_upload<double>(h, &V.adv3OnCell, a3S))) return rc;
    {   // w_adv_curv multiplies every coefficient by an exact 0.0 (the reference's flux of a zeroed w): with finite coefficients the sum
        // is +0.0 whatever they are, and the kernel may leave the loads out
      bool fin = true;
      for (size_t i = 0; i < acS.size() && fin; ++i) fin = std::fabs(acS[i]) <= 1e150 && std::fabs(a3S[i]) <= 1e150;   // false for NaN / Inf
      V.advFinite = fin ? 1 : 0;
    }
    // per-edge {cell1, cell2, vertex1, vertex2} in one 16-byte word, and the divergence-damping skip flag
    const std::vector<int> voe = build_ids(m->verticesOnEdge, nE, 2, eNew, nV, vNew, pol);
    const std::vector<unsigned char> shr = build_vals<unsigned char, uint8_t>(m->isShared, nC, 1, cNew);
    std::vector<int4> ecv((size_t)nE + 1);
    std::vector<unsigned char> skip((size_t)nE + 1, 0);
    for (int e = 0; e <= nE; ++e) {
      ecv[e] = make_int4(coe[(size_t)e * 2], coe[(size_t)e * 2 + 1], voe[(size_t)e * 2], voe[(size_t)e * 2 + 1]);
      skip[e] = (shr[coe[(size_t)e * 2]] && shr[coe[(size_t)e * 2 + 1]]) ? 1 : 0;
    }
    if ((rc = dev_upload<int4>(h, &V.ecv, ecv))) return rc;
    if ((rc = dev_upload<unsigned char>(h, &V.divdampSkip, skip))) return rc;
    // dcEdge of each vertex's three edges
    const std::vector<int> eov = build_ids(m->edgesOnVertex, nV, VD, vNew, nE, eNew, pol);
    const std::vector<double> dcE = build_vals<double, double>(m->dcEdge, nE, 1, eNew);
    std::vector<double> dcV((size_t)(nV + 1) * VD, 0.0);
    for (size_t i = 0; i < dcV.size(); ++i) dcV[i] = dcE[eov[i]];
    if ((rc = dev_upload<double>(h, &V.dcOnVertex, dcV))) return rc;
  }
  UP_IDS(verticesOnCell, m->verticesOnCell, nC, ME, cNew, nV, vNew);
  UP_INT(kiteForCell, m->kiteForCell, nC, ME, cNew);
  UP_DBL(edgesOnCellSign, m->edgesOnCellSign, nC, ME, cNew);
  UP_DBL(edgesOnCell_sign, m->edgesOnCell_sign, nC, ME, cNew);
  UP_DBL(invAreaCell, m->invAreaCell, nC, 1, cNew);
  UP_DBL(defc_a, m->defc_a, nC, ME, cNew);
  UP_DBL(defc_b, m->defc_b, nC, ME, cNew);
  UP_INT(bdyMaskCell, m->bdyMaskCell, nC, 1, cNew);
  UP_DBL(specZoneMaskCell, m->specZoneMaskCell, nC, 1, cNew);
  UP_DBL(coeffsRecon, m->coeffs_reconstruct, nC, ME * 3, cNew);
  {
    std::vector<double> cl((size_t)nC + 1, 1.0);        // cos(0) for the pad
    for (int c = 0; c < nC; ++c) cl[cNew[c]] = std::cos(m->latCell ? m->latCell[c] : 0.0);
    if ((rc = dev_upload<double>(h, &V.cosLatCell, cl))) return rc;
    std::vector<double> sl((size_t)nC + 1, 0.0), clo((size_t)nC + 1, 1.0), slo((size_t)nC + 1, 0.0);
    for (int c = 0; c < nC; ++c) {
      sl[cNew[c]] = std::sin(m->latCell ? m->latCell[c] : 0.0);
      clo[cNew[c]] = std::cos(m->lonCell ? m->lonCell[c] : 0.0); slo[cNew[c]] = std::sin(m->lonCell ? m->lonCell[c] : 0.0);
    }
    if ((rc = dev_upload<double>(h, &V.sinLatCell, sl))) return rc;
    if ((rc = dev_upload<double>(h, &V.cosLonCell, clo))) return rc;
    if ((rc = dev_upload<double>(h, &V.sinLonCell, slo))) return rc;
    std::vector<unsigned char> sh = build_vals<unsigned char, uint8_t>(m->isShared, nC, 1, cNew);
    std::vector<unsigned char> cp((size_t)nC + 1, 1); cp[nC] = 0;
    if (m->inCpr) for (int c = 0; c < nC; ++c) cp[cNew[c]] = m->inCpr[c];
    if ((rc = dev_upload<unsigned char>(h, &V.isShared, sh))) return rc;
    if ((rc = dev_upload<unsigned char>(h, &V.inCpr, cp))) return rc;
  }
  UP_IDS(cellsOnEdge, m->cellsOnEdge, nE, 2, eNew, nC, cNew);
  UP_IDS(verticesOnEdge, m->verticesOnEdge, nE, 2, eNew, nV, vNew);
  UP_INT(nEdgesOnEdge, m->nEdgesOnEdge, nE, 1, eNew);
  UP_IDS(edgesOnEdge_ECP, m->edgesOnEdge_ECP, nE, ME2, eNew, nE, eNew);
  UP_IDS(edgesOnEdge, m->edgesOnEdge, nE, ME2, eNew, nE, eNew);
#ifdef MPASB200_LAB
  if (h->c.edge_tiles) {
    if ((rc = build_edge_tiles(h, build_ids(m->edgesOnEdge, nE, ME2, eNew, nE, eNew, pol), build_vals<int, int32_t>(m->nEdgesOnEdge, nE, 1, eNew)))) return rc;
  }
#endif
  UP_DBL(weightsOnEdge, m->weightsOnEdge, nE, ME2, eNew);
  UP_DBL(dcEdge, m->dcEdge, nE, 1, eNew);
  UP_DBL(dvEdge, m->dvEdge, nE, 1, eNew);
  UP_DBL(invDcEdge, m->invDcEdge, nE, 1, eNew);
  UP_DBL(invDvEdge, m->invDvEdge, nE, 1, eNew);
  {
    std::vector<double> ca((size_t)nE + 1, 1.0), sa((size_t)nE + 1, 0.0), cl((size_t)nE + 1, 1.0);
    for (int e = 0; e < nE; ++e) {
      const double a = m->angleEdge ? m->angleEdge[e] : 0.0;
      ca[eNew[e]] = std::cos(a); sa[eNew[e]] = std::sin(a); cl[eNew[e]] = std::cos(m->latEdge ? m->latEdge[e] : 0.0);
    }
    if ((rc = dev_upload<double>(h, &V.cosAngleEdge, ca))) return rc;
    if ((rc = dev_upload<double>(h, &V.sinAngleEdge, sa))) return rc;
    if ((rc = dev_upload<double>(h, &V.cosLatEdge, cl))) return rc;
  }
  UP_INT(nAdvCellsForEdge, m->nAdvCellsForEdge, nE, 1, eNew);
  UP_IDS(advCellsForEdge, m->advCellsForEdge, nE, NA, eNew, nC, cNew);
  UP_DBL(adv_coefs, m->adv_coefs, nE, NA, eNew);
  UP_DBL(adv_coefs_3rd, m->adv_coefs_3rd, nE, NA, eNew);
  UP_DBL(meshScalingDel2, m->meshScalingDel2, nE, 1, eNew);
  UP_DBL(meshScalingDel4, m->meshScalingDel4, nE, 1, eNew);
  UP_DBL(specZoneMaskEdge, m->specZoneMaskEdge, nE, 1, eNew);
  UP_IDS(edgesOnVertex, m->edgesOnVertex, nV, VD, vNew, nE, eNew);
  UP_DBL(edgesOnVertexSign, m->edgesOnVertexSign, nV, VD, vNew);
  UP_DBL(edgesOnVertex_sign, m->edgesOnVertex_sign, nV, VD, vNew);
  UP_DBL(kiteAreasOnVertex, m->kiteAreasOnVertex, nV, VD, vNew);
  UP_DBL(fVertex, m->fVertex, nV, 1, vNew);
  UP_DBL(invAreaTriangle, m->invAreaTriangle, nV, 1, vNew);
#undef UP_IDS
#undef UP_INT
#undef UP_DBL
  h->has_classes = m->cellClass && m->edgeClass;
  h->mesh_ok = true;
  return 0;
}

// ---- strided members of the static region data (mpas_b200.h) -----------------------------------------------------------------
namespace {
struct MemberInfo { const char* name; size_t offset; int elem; int entity; int wkind; };   // wkind: 1, 2, -1 maxEdges, -2 maxEdges2, -3 vertexDegree, -4 nAdvCells
#define MM(name, T, ent, w) {#name, offsetof(MpasMeshPtrs, name), (int)sizeof(T), MPASB200_##ent, w}
const MemberInfo kMembers[] = {
    MM(nEdgesOnCell, int32_t, CELL, 1), MM(edgesOnCell, int32_t, CELL, -1), MM(verticesOnCell, int32_t, CELL, -1), MM(kiteForCell, int32_t, CELL, -1),
    MM(edgesOnCellSign, double, CELL, -1), MM(edgesOnCell_sign, double, CELL, -1), MM(invAreaCell, double, CELL, 1), MM(latCell, double, CELL, 1),
    MM(defc_a, double, CELL, -1), MM(defc_b, double, CELL, -1), MM(bdyMaskCell, int32_t, CELL, 1), MM(specZoneMaskCell, double, CELL, 1),
    MM(isShared, uint8_t, CELL, 1), MM(inCpr, uint8_t, CELL, 1),
    MM(cellsOnEdge, int32_t, EDGE, 2), MM(verticesOnEdge, int32_t, EDGE, 2), MM(nEdgesOnEdge, int32_t, EDGE, 1), MM(edgesOnEdge_ECP, int32_t, EDGE, -2),
    MM(edgesOnEdge, int32_t, EDGE, -2), MM(weightsOnEdge, double, EDGE, -2), MM(dcEdge, double, EDGE, 1), MM(dvEdge, double, EDGE, 1),
    MM(invDcEdge, double, EDGE, 1), MM(invDvEdge, double, EDGE, 1), MM(angleEdge, double, EDGE, 1), MM(latEdge, double, EDGE, 1),
    MM(nAdvCellsForEdge, int32_t, EDGE, 1), MM(advCellsForEdge, int32_t, EDGE, -4), MM(adv_coefs, double, EDGE, -4), MM(adv_coefs_3rd, double, EDGE, -4),
    MM(meshScalingDel2, double, EDGE, 1), MM(meshScalingDel4, double, EDGE, 1), MM(specZoneMaskEdge, double, EDGE, 1),
    MM(edgesOnVertex, int32_t, VERTEX, -3), MM(edgesOnVertexSign, double, VERTEX, -3), MM(edgesOnVertex_sign, double, VERTEX, -3),
    MM(kiteAreasOnVertex, double, VERTEX, -3), MM(fVertex, double, VERTEX, 1), MM(invAreaTriangle, double, VERTEX, 1),
    MM(xCell, double, CELL, 1), MM(yCell, double, CELL, 1), MM(zCell, double, CELL, 1), MM(cellClass, uint8_t, CELL, 1), MM(edgeClass, uint8_t, EDGE, 1),
    MM(lonCell, double, CELL, 1), MM(coeffs_reconstruct, double, CELL, -5),
};
#undef MM
int member_width(const mpasb200_t* h, int wkind) {
  switch (wkind) { case -1: return h->d.maxEdges; case -2: return h->d.maxEdges2; case -3: return h->d.vertexDegree; case -4: return h->d.nAdvCells; case -5: return 3 * h->d.maxEdges; default: return wkind; }
}
}  // namespace
int mpasb200_mesh_member(mpasb200_t* h, const char* member, const void* base, int64_t stride_x) {
  if (!h || !member || !base) return MPASB200_EINVAL;
  std::unique_lock<std::mutex> lk(h->mu);
  if (h->mesh_ok) return fail(h, MPASB200_ESTATE, "mesh_member after upload_mesh");
  for (const MemberInfo& mi : kMembers)
    if (!std::strcmp(mi.name, member)) {
      const int n = entity_count(h, mi.entity), w = member_width(h, mi.wkind);
      const size_t row = (size_t)w * mi.elem;
      if (stride_x == 0) stride_x = (int64_t)row;
      if (stride_x > 0 && (size_t)stride_x < row) return fail(h, MPASB200_EINVAL, "mesh_member: stride smaller than one element row");
      std::vector<char>& v = h->mesh_stage[member];
      v.resize((size_t)n * row);
      for (int x = 0; x < n; ++x) std::memcpy(v.data() + (size_t)x * row, (const char*)base + (int64_t)x * stride_x, row);
      return 0;
    }
  return fail(h, MPASB200_EINVAL, std::string("mesh_member: unknown member ") + member);
}
int mpasb200_upload_mesh_staged(mpasb200_t* h) {
  if (!h) return MPASB200_EINVAL;
  MpasMeshPtrs m;
  std::memset(&m, 0, sizeof(m));
  {
    std::unique_lock<std::mutex> lk(h->mu);
    for (const MemberInfo& mi : kMembers) {
      auto it = h->mesh_stage.find(mi.name);
      if (it != h->mesh_stage.end()) *(const void**)((char*)&m + mi.offset) = it->second.data();
    }
  }
  const int rc = mpasb200_upload_mesh(h, &m);
  if (rc == 0) { std::unique_lock<std::mutex> lk(h->mu); h->mesh_stage.clear(); }
  return rc;
}

// ---- field transfers ---------------------------------------------------------------------------------
static int field_xfer(mpasb200_t* h, int field, void* base, int64_t stride_x, int64_t stride_k, bool up) {
  if (!h || !base) return MPASB200_EINVAL;
  std::unique_lock<std::mutex> lk(h->mu);
  cudaSetDevice(h->device);
  if (field < 0 || field >= MPASB200_F_COUNT) return fail(h, MPASB200_EINVAL, "field id out of range");
  const FieldInfo& fi = kFields[field];
  const int L1 = h->L1, S = fi.slots;
  char* b = (char*)base;
  if (fi.entity == MPASB200_VERTICAL) {
    if (stride_k == 0) stride_k = 8;
    std::vector<double> tmp(L1);
    if (up) {
      for (int k = 0; k < L1; ++k) tmp[k] = *(const double*)(b + (int64_t)k * stride_k);
      CK(cudaMemcpyAsync(h->V.f[field], tmp.data(), sizeof(double) * L1, cudaMemcpyHostToDevice, h->stream));
      CK(cudaStreamSynchronize(h->stream));
    } else {
      CK(cudaMemcpyAsync(tmp.data(), h->V.f[field], sizeof(double) * L1, cudaMemcpyDeviceToHost, h->stream));
      CK(cudaStreamSynchronize(h->stream));
      for (int k = 0; k < L1; ++k) *(double*)(b + (int64_t)k * stride_k) = tmp[k];
    }
    return 0;
  }
  if (!h->mesh_ok) return fail(h, MPASB200_ESTATE, "upload_mesh must precede field transfers (it fixes the renumbering)");
  const int n = entity_count(h, fi.entity);
  if (n == 0) return 0;
  const size_t rowElems = (size_t)L1 * S;
  const bool contiguous = (stride_k == (int64_t)(8 * S)) && (stride_x == (int64_t)(8 * rowElems));
  const size_t chunkRows = std::max<size_t>(1, std::min<size_t>((size_t)n, ((size_t)32 << 20) / rowElems));   // <= 256 MB of doubles per chunk
  int rc;
  if ((rc = ensure_stage(h, chunkRows * rowElems))) return rc;
  if (!contiguous && (rc = ensure_hstage(h, chunkRows * rowElems))) return rc;
  const size_t slotStride = (size_t)(n + 1) * h->LP;
  const int* map = h->d_newOf[fi.entity];
  for (size_t r0 = 0; r0 < (size_t)n; r0 += chunkRows) {
    const size_t rows = std::min(chunkRows, (size_t)n - r0);
    const size_t elems = rows * rowElems;
    const unsigned blocks = (unsigned)((elems + 255) / 256);
    if (up) {
      const double* src;
      if (contiguous) src = (const double*)(b + (int64_t)r0 * stride_x);
      else {
        for (size_t r = 0; r < rows; ++r)
          for (int k = 0; k < L1; ++k)
            std::memcpy(h->h_stage + (r * L1 + k) * S, b + (int64_t)(r0 + r) * stride_x + (int64_t)k * stride_k, sizeof(double) * S);
        src = h->h_stage;
      }
      CK(cudaMemcpyAsync(h->d_stage, src, elems * sizeof(double), cudaMemcpyHostToDevice, h->stream));
      k_stage_to_field<<<blocks, 256, 0, h->stream>>>(h->V.f[field], h->d_stage, map + r0, (int)rows, L1, h->LP, S, slotStride);
      h->launches++;
      CK(cudaGetLastError());
      CK(cudaStreamSynchronize(h->stream));
    } else {
      k_field_to_stage<<<blocks, 256, 0, h->stream>>>(h->V.f[field], h->d_stage, map + r0, (int)rows, L1, h->LP, S, slotStride);
      h->launches++;
      CK(cudaGetLastError());
      double* dst = contiguous ? (double*)(b + (int64_t)r0 * stride_x) : h->h_stage;
      CK(cudaMemcpyAsync(dst, h->d_stage, elems * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
      CK(cudaStreamSynchronize(h->stream));
      if (!contiguous)
        for (size_t r = 0; r < rows; ++r)
          for (int k = 0; k < L1; ++k)
            std::memcpy(b + (int64_t)(r0 + r) * stride_x + (int64_t)k * stride_k, h->h_stage + (r * L1 + k) * S, sizeof(double) * S);
    }
  }
  return 0;
}
int mpasb200_upload_field(mpasb200_t* h, int field, const void* base, int64_t stride_x, int64_t stride_k) {
  return field_xfer(h, field, const_cast<void*>(base), stride_x, stride_k, true);
}
int mpasb200_download_field(mpasb200_t* h, int field, void* base, int64_t stride_x, int64_t stride_k) {
  return field_xfer(h, field, base, stride_x, stride_k, false);
}
// Pipelined transfers.  Contiguous page-locked host arrays only.  Upload: H2D copy on the upload stream into the field's
// own staging buffer, renumbering scatter on the compute stream (ordered before every later task).  Download: gather on the
// compute stream (ordered after every earlier task), D2H copy on the download stream.  The two copy directions and the
// compute stream overlap; a staging buffer is reused only after the event that frees it.
static int field_xfer_async(mpasb200_t* h, int field, void* base, bool up) {
  if (!h || !base) return MPASB200_EINVAL;
  std::unique_lock<std::mutex> lk(h->mu);
  cudaSetDevice(h->device);
  if (field < 0 || field >= MPASB200_F_COUNT) return fail(h, MPASB200_EINVAL, "field id out of range");
  const FieldInfo& fi = kFields[field];
  if (fi.entity == MPASB200_VERTICAL) return fail(h, MPASB200_EINVAL, "vertical fields have no asynchronous transfer");
  if (!h->mesh_ok) return fail(h, MPASB200_ESTATE, "upload_mesh must precede field transfers (it fixes the renumbering)");
  if (h->capturing) return fail(h, MPASB200_ESTATE, "transfer during graph capture");
  const int n = entity_count(h, fi.entity);
  if (n == 0) return 0;
  const int L1 = h->L1, S = fi.slots;
  const size_t elems = (size_t)n * L1 * S, bytes = elems * sizeof(double);
  if (!h->up_stream) {
    CK(cudaStreamCreateWithFlags(&h->up_stream, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&h->dn_stream, cudaStreamNonBlocking));
    h->pipe.resize(MPASB200_F_COUNT);
  }
  mpasb200_t::Pipe& pp = h->pipe[field];
  if (!pp.up_copied) {
    for (cudaEvent_t* e : {&pp.up_copied, &pp.up_scattered, &pp.dn_gathered, &pp.dn_copied}) CK(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
  }
  double*& stage = up ? pp.up : pp.dn;
  if (!stage) {
    cudaError_t e = cudaMalloc((void**)&stage, bytes);
    if (e != cudaSuccess) { h->err = std::string("cudaMalloc(pipeline staging): ") + cudaGetErrorString(e); stage = nullptr; return MPASB200_ENOMEM; }
    h->bytes += bytes;
  }
  const size_t slotStride = (size_t)(n + 1) * h->LP;
  const int* map = h->d_newOf[fi.entity];
  const unsigned blocks = (unsigned)((elems + 255) / 256);
  if (up) {
    if (pp.up_used) CK(cudaStreamWaitEvent(h->up_stream, pp.up_scattered, 0));        // staging free again
    CK(cudaMemcpyAsync(pp.up, base, bytes, cudaMemcpyHostToDevice, h->up_stream));
    CK(cudaEventRecord(pp.up_copied, h->up_stream));
    CK(cudaStreamWaitEvent(h->stream, pp.up_copied, 0));
    k_stage_to_field<<<blocks, 256, 0, h->stream>>>(h->V.f[field], pp.up, map, n, L1, h->LP, S, slotStride);
    h->launches++;
    CK(cudaGetLastError());
    CK(cudaEventRecord(pp.up_scattered, h->stream));
    pp.up_used = true;
  } else {
    if (pp.dn_used) CK(cudaStreamWaitEvent(h->stream, pp.dn_copied, 0));              // staging free again
    k_field_to_stage<<<blocks, 256, 0, h->stream>>>(h->V.f[field], pp.dn, map, n, L1, h->LP, S, slotStride);
    h->launches++;
    CK(cudaGetLastError());
    CK(cudaEventRecord(pp.dn_gathered, h->stream));
    CK(cudaStreamWaitEvent(h->dn_stream, pp.dn_gathered, 0));
    CK(cudaMemcpyAsync(base, pp.dn, bytes, cudaMemcpyDeviceToHost, h->dn_stream));
    CK(cudaEventRecord(pp.dn_copied, h->dn_stream));
    pp.dn_used = true;
  }
  return 0;
}
int mpasb200_upload_field_async(mpasb200_t* h, int field, const void* base) { return field_xfer_async(h, field, const_cast<void*>(base), true); }
int mpasb200_download_field_async(mpasb200_t* h, int field, void* base) { return field_xfer_async(h, field, base, false); }
int mpasb200_transfer_wait(mpasb200_t* h) {
  if (!h) return MPASB200_EINVAL;
  std::unique_lock<std::mutex> lk(h->mu);
  cudaSetDevice(h->device);
  if (h->up_stream) { CK(cudaStreamSynchronize(h->up_stream)); }
  CK(cudaStreamSynchronize(h->stream));
  if (h->dn_stream) { CK(cudaStreamSynchronize(h->dn_stream)); }
  return 0;
}
int mpasb200_zero_field(mpasb200_t* h, int field) {
  if (!h || field < 0 || field >= MPASB200_F_COUNT) return MPASB200_EINVAL;
  std::unique_lock<std::mutex> lk(h->mu);
  cudaSetDevice(h->device);
  const FieldInfo& fi = kFields[field];
  const size_t n = (fi.entity == MPASB200_VERTICAL) ? (size_t)h->LP : (size_t)(entity_count(h, fi.entity) + 1) * h->LP * fi.slots;
  CK(cudaMemsetAsync(h->V.f[field], 0, n * sizeof(double), h->stream));
  return 0;
}
int mpasb200_sync(mpasb200_t* h) {
  if (!h) return MPASB200_EINVAL;
  std::unique_lock<std::mutex> lk(h->mu);
  cudaSetDevice(h->device);
  CK(cudaStreamSynchronize(h->stream));
  return 0;
}
int mpasb200_class_range(mpasb200_t* h, int entity, int cls, int32_t* begin, int32_t* end) {
  if (!h || entity < 0 || entity > 2 || cls < 0 || cls > 3 || !begin || !end) return MPASB200_EINVAL;
  std::unique_lock<std::mutex> lk(h->mu);
  if (!h->mesh_ok) return fail(h, MPASB200_ESTATE, "upload_mesh has not been called");
  *begin = h->classBegin[entity][cls]; *end = h->classBegin[entity][cls + 1];
  return 0;
}
int mpasb200_set_range(mpasb200_t* h, int entity, int32_t begin, int32_t end) {
  if (!h || entity < 0 || entity > 2) return MPASB200_EINVAL;
  std::unique_lock<std::mutex> lk(h->mu);
  if (end >= 0 && begin >= 0 && end < begin) return fail(h, MPASB200_EINVAL, "set_range: end < begin");
  // a captured atm_srk3 graph has the launch ranges baked in: drop the cache whenever a range changes
  for (auto& g : h->graphs) cudaGraphExecDestroy(g.second.first);
  h->graphs.clear();
  if (begin < 0 || end < 0) { h->rangeSet[entity] = false; return 0; }
  h->rangeB[entity] = begin; h->rangeE[entity] = end; h->rangeSet[entity] = true;
  return 0;
}
int mpasb200_set_stream(mpasb200_t* h, void* s) {
  if (!h) return MPASB200_EINVAL;
  std::unique_lock<std::mutex> lk(h->mu);
  h->stream = s ? (cudaStream_t)s : h->own_stream;
  return 0;
}

int mpasb200_set_use_graph(mpasb200_t* h, int on) {
  if (!h) return MPASB200_EINVAL;
  std::unique_lock<std::mutex> lk(h->mu);
  h->c.use_graph = on != 0;
  return 0;
}

// ---- tasks ------------------------------------------------------------------------------------------------
int mpasb200_rk_integration_setup(mpasb200_t* h) { REQUIRE_MESH(); Entry en(h, MPASB200_T_SETUP); return en.done(t_setup(h)); }
int mpasb200_compute_moist_coefficients(mpasb200_t* h) { REQUIRE_MESH(); Entry en(h, MPASB200_T_MOIST); return en.done(t_moist(h)); }
int mpasb200_compute_vert_imp_coefs(mpasb200_t* h, double dts) { REQUIRE_MESH(); Entry en(h, MPASB200_T_VERT_IMP); return en.done(t_vert_imp(h, dts)); }
int mpasb200_compute_dyn_tend(mpasb200_t* h, int rk_step, double dt, int mixing, double cam_coef, int mix_full, int rayleigh_u) {
  REQUIRE_MESH();
  if (mixing < 0 || mixing > MPASB200_MIX_OTHER) return fail(h, MPASB200_EINVAL, "config_horiz_mixing: unknown enum value");
  Entry en(h, MPASB200_T_DYN_TEND);
  return en.done(t_dyn_tend(h, rk_step, dt, mixing, cam_coef, mix_full, rayleigh_u));
}
int mpasb200_set_smlstep_pert_variables(mpasb200_t* h) { REQUIRE_MESH(); Entry en(h, MPASB200_T_SMLSTEP); return en.done(t_smlstep(h)); }
int mpasb200_advance_acoustic_step(mpasb200_t* h, double dts, int small_step) { REQUIRE_MESH(); Entry en(h, MPASB200_T_ACOUSTIC); return en.done(t_acoustic(h, dts, small_step)); }
int mpasb200_divergence_damping_3d(mpasb200_t* h, double dts) { REQUIRE_MESH(); Entry en(h, MPASB200_T_DIVDAMP); return en.done(t_divdamp(h, dts)); }
int mpasb200_recover_large_step_variables(mpasb200_t* h, int ns, int rk_step, double dt) { REQUIRE_MESH(); Entry en(h, MPASB200_T_RECOVER); return en.done(t_recover(h, ns, rk_step, dt)); }
int mpasb200_compute_solve_diagnostics(mpasb200_t* h, int hollingsworth, int rk_step) { REQUIRE_MESH(); Entry en(h, MPASB200_T_DIAG); return en.done(t_diag(h, hollingsworth, rk_step)); }
int mpasb200_advance_scalars(mpasb200_t* h, double dt, int rk_step) { REQUIRE_MESH(); Entry en(h, MPASB200_T_SCALARS); return en.done(t_scalars(h, dt, rk_step)); }
int mpasb200_init_coupled_diagnostics(mpasb200_t* h) { REQUIRE_MESH(); Entry en(h, -1); return t_init_coupled(h); }
int mpasb200_reconstruct_2d(mpasb200_t* h, int includeHalos, int on_a_sphere) { (void)includeHalos; REQUIRE_MESH(); Entry en(h, -1); return t_reconstruct(h, on_a_sphere); }
}  // extern "C"
// ---- the mesh-only producers of atm_core_init on the device (kernels_init.cuh) ---------------------------------------------------
namespace {
struct TempDev {                       // device scratch of one call, released on return
  std::vector<void*> p;
  ~TempDev() { for (void* q : p) cudaFree(q); }
  template <class T> T* up(const T* src, size_t n, cudaStream_t st, cudaError_t* err) {
    if (!src || n == 0) return nullptr;
    T* d = nullptr;
    if ((*err = cudaMalloc(&d, n * sizeof(T))) != cudaSuccess) return nullptr;
    p.push_back(d);
    *err = cudaMemcpyAsync(d, src, n * sizeof(T), cudaMemcpyHostToDevice, st);
    return d;
  }
  template <class T> T* out(size_t n, cudaError_t* err) {
    T* d = nullptr;
    if ((*err = cudaMalloc(&d, std::max<size_t>(n, 1) * sizeof(T))) != cudaSuccess) return nullptr;
    p.push_back(d);
    return d;
  }
};
#define TD(expr) do { expr; if (err != cudaSuccess) return fail(h, MPASB200_ECUDA, std::string("init producers: ") + cudaGetErrorString(err)); } while (0)
int init_mesh_dev(mpasb200_t* h, const MpasInitMesh* m, TempDev& t, InitMeshDev& M) {
  const size_t nC = h->nCells, nE = h->nEdges, nV = h->nVertices, ME = h->d.maxEdges, VD = h->d.vertexDegree, NA = h->d.nAdvCells;
  cudaError_t err = cudaSuccess;
  std::memset(&M, 0, sizeof(M));
  M.nC = (int)nC; M.nE = (int)nE; M.nV = (int)nV; M.ME = (int)ME; M.VD = (int)VD; M.NA = (int)NA; M.pol = h->c.index_policy;
  TD(M.nEdgesOnCell = t.up<int>(m->nEdgesOnCell, nC, h->stream, &err));
  TD(M.edgesOnCell = t.up<int>(m->edgesOnCell, nC * ME, h->stream, &err));
  TD(M.verticesOnCell = t.up<int>(m->verticesOnCell, nC * ME, h->stream, &err));
  TD(M.cellsOnCell = t.up<int>(m->cellsOnCell, nC * ME, h->stream, &err));
  TD(M.cellsOnEdge = t.up<int>(m->cellsOnEdge, nE * 2, h->stream, &err));
  TD(M.verticesOnEdge = t.up<int>(m->verticesOnEdge, nE * 2, h->stream, &err));
  TD(M.cellsOnVertex = t.up<int>(m->cellsOnVertex, nV * VD, h->stream, &err));
  TD(M.edgesOnVertex = t.up<int>(m->edgesOnVertex, nV * VD, h->stream, &err));
  TD(M.dcEdge = t.up<double>(m->dcEdge, nE, h->stream, &err));
  TD(M.dvEdge = t.up<double>(m->dvEdge, nE, h->stream, &err));
  TD(M.deriv_two = t.up<double>(m->deriv_two, nE * 2 * NA, h->stream, &err));
  return 0;
}
template <class T> int fetch(mpasb200_t* h, T* host, const T* dev, size_t n) {
  if (!host || n == 0) return 0;
  CK(cudaMemcpyAsync(host, dev, n * sizeof(T), cudaMemcpyDeviceToHost, h->stream));
  return 0;
}
}  // namespace

extern "C" {
int mpasb200_compute_signs(mpasb200_t* h, const MpasInitMesh* m, double* edgesOnVertexSign, double* edgesOnCellSign, int32_t* kiteForCell) {
  if (!h || !m) return MPASB200_EINVAL;
  std::unique_lock<std::mutex> lk(h->mu);
  cudaSetDevice(h->device);
  if (!m->nEdgesOnCell || !m->edgesOnCell || !m->verticesOnCell || !m->cellsOnEdge || !m->verticesOnEdge || !m->cellsOnVertex || !m->edgesOnVertex)
    return fail(h, MPASB200_EINVAL, "compute_signs: nEdgesOnCell, edgesOnCell, verticesOnCell, cellsOnEdge, verticesOnEdge, cellsOnVertex, edgesOnVertex are required");
  TempDev t; InitMeshDev M;
  if (int rc = init_mesh_dev(h, m, t, M)) return rc;
  cudaError_t err = cudaSuccess;
  const size_t nC = h->nCells, nV = h->nVertices, ME = h->d.maxEdges, VD = h->d.vertexDegree;
  double* d_eov = nullptr; double* d_eoc = nullptr; int* d_kite = nullptr;
  TD(d_eov = t.out<double>(nV * VD, &err)); TD(d_eoc = t.out<double>(nC * ME, &err)); TD(d_kite = t.out<int>(nC * ME, &err));
  if (nV) { KTimer kt_(h, "k_signs_vertex"); k_signs_vertex<<<(unsigned)((nV + 127) / 128), 128, 0, h->stream>>>(M, d_eov); h->launches++; }
  if (nC) { KTimer kt_(h, "k_signs_cell"); k_signs_cell<<<(unsigned)((nC + 127) / 128), 128, 0, h->stream>>>(M, d_eoc, d_kite); h->launches++; }
  if (int rc = post_launch(h)) return rc;
  if (int rc = fetch(h, edgesOnVertexSign, d_eov, nV * VD)) return rc;
  if (int rc = fetch(h, edgesOnCellSign, d_eoc, nC * ME)) return rc;
  if (int rc = fetch(h, (int*)kiteForCell, d_kite, nC * ME)) return rc;
  CK(cudaStreamSynchronize(h->stream));
  return 0;
}

int mpasb200_adv_coef_compression(mpasb200_t* h, const MpasInitMesh* m, int32_t* nAdvCellsForEdge, int32_t* advCellsForEdge,
                                  double* adv_coefs, double* adv_coefs_3rd) {
  if (!h || !m) return MPASB200_EINVAL;
  std::unique_lock<std::mutex> lk(h->mu);
  cudaSetDevice(h->device);
  if (!m->nEdgesOnCell || !m->cellsOnCell || !m->cellsOnEdge || !m->dcEdge || !m->dvEdge)
    return fail(h, MPASB200_EINVAL, "adv_coef_compression: nEdgesOnCell, cellsOnCell, cellsOnEdge, dcEdge, dvEdge are required");
  if (!nAdvCellsForEdge || !advCellsForEdge || !adv_coefs || !adv_coefs_3rd) return fail(h, MPASB200_EINVAL, "adv_coef_compression: null output");
  enum { WMAX = 34 };                                   // 2 + 2*maxEdges, maxEdges <= 16 (mpasb200_create)
  if (2 + 2 * h->d.maxEdges > WMAX) return fail(h, MPASB200_EINVAL, "adv_coef_compression: maxEdges too large");
  TempDev t; InitMeshDev M;
  if (int rc = init_mesh_dev(h, m, t, M)) return rc;
  cudaError_t err = cudaSuccess;
  const size_t nE = h->nEdges, NA = h->d.nAdvCells;
  int* d_n = nullptr; int* d_adv = nullptr; double* d_a = nullptr; double* d_a3 = nullptr;
  TD(d_n = t.out<int>(nE, &err)); TD(d_adv = t.out<int>(nE * NA, &err)); TD(d_a = t.out<double>(nE * NA, &err)); TD(d_a3 = t.out<double>(nE * NA, &err));
  if (nE) { KTimer kt_(h, "k_adv_coef"); k_adv_coef<WMAX><<<(unsigned)((nE + 127) / 128), 128, 0, h->stream>>>(M, d_n, d_adv, d_a, d_a3); h->launches++; }
  if (int rc = post_launch(h)) return rc;
  if (int rc = fetch(h, (int*)nAdvCellsForEdge, d_n, nE)) return rc;
  if (int rc = fetch(h, (int*)advCellsForEdge, d_adv, nE * NA)) return rc;
  if (int rc = fetch(h, adv_coefs, d_a, nE * NA)) return rc;
  if (int rc = fetch(h, adv_coefs_3rd, d_a3, nE * NA)) return rc;
  CK(cudaStreamSynchronize(h->stream));
  return 0;
}

int mpasb200_compute_mesh_scaling(mpasb200_t* h, const MpasInitMesh* m, const double* meshDensity, int scale_with_mesh, double* del2, double* del4) {
  if (!h || !m) return MPASB200_EINVAL;
  std::unique_lock<std::mutex> lk(h->mu);
  cudaSetDevice(h->device);
  if (!m->cellsOnEdge || !del2 || !del4 || (scale_with_mesh && !meshDensity)) return fail(h, MPASB200_EINVAL, "compute_mesh_scaling: cellsOnEdge, meshDensity and both outputs are required");
  TempDev t; InitMeshDev M;
  MpasInitMesh only; std::memset(&only, 0, sizeof(only)); only.cellsOnEdge = m->cellsOnEdge;
  if (int rc = init_mesh_dev(h, &only, t, M)) return rc;
  cudaError_t err = cudaSuccess;
  const size_t nE = h->nEdges, nC = h->nCells;
  double* d_md = nullptr; double* d2 = nullptr; double* d4 = nullptr;
  TD(d_md = t.up<double>(meshDensity, nC, h->stream, &err)); TD(d2 = t.out<double>(nE, &err)); TD(d4 = t.out<double>(nE, &err));
  if (nE) { KTimer kt_(h, "k_mesh_scaling"); k_mesh_scaling<<<(unsigned)((nE + 127) / 128), 128, 0, h->stream>>>(M, d_md, scale_with_mesh, d2, d4); h->launches++; }
  if (int rc = post_launch(h)) return rc;
  if (int rc = fetch(h, del2, d2, nE)) return rc;
  if (int rc = fetch(h, del4, d4, nE)) return rc;
  CK(cudaStreamSynchronize(h->stream));
  return 0;
}

int mpasb200_compute_damping_coefs(mpasb200_t* h, const double* meshDensity, double config_zd, double config_xnutr) {
  REQUIRE_MESH();
  if (!meshDensity) return fail(h, MPASB200_EINVAL, "compute_damping_coefs: meshDensity is required");
  Entry en(h, -1);
  TempDev t;
  cudaError_t err = cudaSuccess;
  std::vector<double> md((size_t)h->nCells + 1, 1.0);
  for (int c = 0; c < h->nCells; ++c) md[h->newOf[MPASB200_CELL][c]] = meshDensity[c];
  double* d_md = nullptr;
  TD(d_md = t.up<double>(md.data(), md.size(), h->stream, &err));
  LAUNCH(k_damping_coefs, h->nCells, 0, h->V, d_md, config_zd, config_xnutr);
  if (int rc = post_launch(h)) return rc;
  CK(cudaStreamSynchronize(h->stream));
  return 0;
}

int mpasb200_compute_zb_cell(mpasb200_t* h) {
  REQUIRE_MESH();
  Entry en(h, -1);
  LAUNCH(k_zb_cell, h->nCells, 0, h->V);
  return post_launch(h);
}

int mpasb200_couple_coef_3rd_order(mpasb200_t* h, double coef, double* adv_coefs_3rd) {
  if (!h) return MPASB200_EINVAL;
  std::unique_lock<std::mutex> lk(h->mu);
  cudaSetDevice(h->device);
  TempDev t;
  cudaError_t err = cudaSuccess;
  const size_t n = (size_t)h->nEdges * h->d.nAdvCells;
  if (adv_coefs_3rd && n) {
    double* d = nullptr;
    TD(d = t.up<double>(adv_coefs_3rd, n, h->stream, &err));
    { KTimer kt_(h, "k_scale"); k_scale<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(d, n, coef); h->launches++; }
    if (int rc = fetch(h, adv_coefs_3rd, d, n)) return rc;
  }
  if (h->mesh_ok && h->nCells) { KTimer kt_(h, "k_zb3_level0"); k_zb3_level0<<<(unsigned)((h->nCells + 127) / 128), 128, 0, h->stream>>>(h->V, coef); h->launches++; }
  if (int rc = post_launch(h)) return rc;
  CK(cudaStreamSynchronize(h->stream));
  return 0;
}
#undef TD

// init_atm_case_jw on the device (kernels_jw.cuh)
int mpasb200_init_atm_case_jw(mpasb200_t* h, const MpasJwGeometry* g) {
  REQUIRE_MESH();
  if (!g || !g->latCell || !g->areaCell || !g->latVertex) return fail(h, MPASB200_EINVAL, "init_atm_case_jw: latCell, areaCell, latVertex are required");
  Entry en(h, -1);
  const int L = h->L, L1 = h->L1, nC = h->nCells, nV = h->nVertices;
  if (L < 3) return fail(h, MPASB200_EINVAL, "init_atm_case_jw: nVertLevels >= 3");
  // ---- vertical grid (init_atm_cases.rg:165-237, corrected indexing: zw[k] = k*dz), on the host: L+1 numbers per array
  const double zt = 45000.0, strf = 1.5, pii = 3.141592653589793;
  std::vector<double> zw(L1), sh(L1), ah(L1), dzw(L1, 0.0), dzu(L1, 0.0), rdzw(L1, 0.0), rdzu(L1, 0.0), fzm(L1, 0.0), fzp(L1, 0.0), cf1(L1, 0.0), cf2(L1, 0.0), cf3(L1, 0.0);
  const double dz = zt / L;
  for (int k = 0; k <= L; ++k) { zw[k] = k * dz; sh[k] = std::pow(k * dz / zt, strf); ah[k] = 1.0 - std::pow(std::cos(0.5 * pii * k * dz / zt), 6.0); }
  for (int k = 0; k < L; ++k) { dzw[k] = zw[k + 1] - zw[k]; rdzw[k] = 1.0 / dzw[k]; }
  for (int k = 1; k < L; ++k) { dzu[k] = 0.5 * (dzw[k] + dzw[k - 1]); rdzu[k] = 1.0 / dzu[k]; fzp[k] = 0.5 * dzw[k] / dzu[k]; fzm[k] = 0.5 * dzw[k - 1] / dzu[k]; }
  { const double cof1 = (2.0 * dzu[1] + dzu[2]) / (dzu[1] + dzu[2]) * dzw[0] / dzu[1], cof2 = dzu[1] / (dzu[1] + dzu[2]) * dzw[0] / dzu[2];
    cf1[0] = fzp[1] + cof1; cf2[0] = fzm[1] - cof1 - cof2; cf3[0] = cof2; }
  auto putv = [&](int id, const std::vector<double>& v) { return cudaMemcpyAsync(h->V.f[id], v.data(), sizeof(double) * L1, cudaMemcpyHostToDevice, h->stream); };
  CK(putv(MPASB200_F_rdzw, rdzw)); CK(putv(MPASB200_F_rdzu, rdzu)); CK(putv(MPASB200_F_fzm, fzm)); CK(putv(MPASB200_F_fzp, fzp));
  CK(putv(MPASB200_F_cf1, cf1)); CK(putv(MPASB200_F_cf2, cf2)); CK(putv(MPASB200_F_cf3, cf3));
  // ---- device scratch: vertical helpers, geometry in internal numbering, the (z, lat) section
  TempDev t;
  cudaError_t err = cudaSuccess;
#define TDJ(expr) do { expr; if (err != cudaSuccess) return fail(h, MPASB200_ECUDA, std::string("init_atm_case_jw: ") + cudaGetErrorString(err)); } while (0)
  JwParams J;
  std::memset(&J, 0, sizeof(J));
  J.nlat = g->n_lat_table > 1 ? g->n_lat_table : 4097;
  J.u0 = 35.0; J.t0 = 288.0; J.t0b = 250.0; J.dtdz = 0.005; J.eta_t = 0.2; J.delta_t = 4.8e5; J.etavs0 = (1.0 - 0.252) * pii / 2.0; J.p0 = 1.0e5; J.zt = zt;
  J.r_earth = h->c.sphere_radius; J.omega = h->c.omega; J.rgas = h->c.rgas; J.cp = h->c.cp; J.gravity = h->c.gravity; J.pii = pii;
  TDJ(J.sh = t.up<double>(sh.data(), L1, h->stream, &err)); TDJ(J.ah = t.up<double>(ah.data(), L1, h->stream, &err));
  TDJ(J.dzw = t.up<double>(dzw.data(), L1, h->stream, &err)); TDJ(J.dzu = t.up<double>(dzu.data(), L1, h->stream, &err));
  std::vector<double> latC((size_t)nC + 1, 0.0), areaC((size_t)nC + 1, 1.0), latV((size_t)nV + 1, 0.0);
  for (int c = 0; c < nC; ++c) { latC[h->newOf[MPASB200_CELL][c]] = g->latCell[c]; areaC[h->newOf[MPASB200_CELL][c]] = g->areaCell[c]; }
  for (int v = 0; v < nV; ++v) latV[h->newOf[MPASB200_VERTEX][v]] = g->latVertex[v];
  TDJ(J.latCell = t.up<double>(latC.data(), latC.size(), h->stream, &err)); TDJ(J.areaCell = t.up<double>(areaC.data(), areaC.size(), h->stream, &err));
  TDJ(J.latVertex = t.up<double>(latV.data(), latV.size(), h->stream, &err));
  const size_t plane = (size_t)J.nlat * L;
  double* wk = nullptr;
  TDJ(J.pp_t = t.out<double>(plane, &err)); TDJ(J.tt_t = t.out<double>(plane, &err)); TDJ(wk = t.out<double>(4 * plane, &err));
#undef TDJ
  { KTimer kt_(h, "k_jw_table"); k_jw_table<<<(unsigned)((J.nlat + 63) / 64), 64, 0, h->stream>>>(J, h->V, wk); h->launches++; }
  { Cfg cf_ = cfg_for(h, nC); KTimer kt_(h, "k_jw_cell"); k_jw_cell<<<cf_.grid, cf_.block, 0, h->stream>>>(J, h->V); h->launches++; }
  if (h->nEdges) { Cfg cf_ = cfg_for(h, h->nEdges); KTimer kt_(h, "k_jw_edge"); k_jw_edge<<<cf_.grid, cf_.block, 0, h->stream>>>(J, h->V); h->launches++; }
  LAUNCH(k_jw_rw, nC, 0, h->V);
  if (int rc = post_launch(h)) return rc;
  CK(cudaStreamSynchronize(h->stream));        // the scratch goes away with `t`
  return 0;
}

int mpasb200_rk_dynamics_substep_finish(mpasb200_t* h, int substep, int split) {
  REQUIRE_MESH();
  if (split < 1) return fail(h, MPASB200_EINVAL, "dynamics_split must be >= 1");
  Entry en(h, MPASB200_T_FINISH);
  return en.done(t_finish(h, substep, split));
}

int mpasb200_srk3(mpasb200_t* h, double dt) {
  REQUIRE_MESH();
  Entry en(h, -1);
  if (h->c.config_scalar_advection) { if (int rc = ensure_sflux(h)) return rc; }
  if (!h->c.use_graph) return t_srk3(h, dt);
  auto it = h->graphs.find(dt);
  if (it == h->graphs.end()) {
    // capture the whole step once per dt: ~60 launch-bound kernels become one graph launch
    cudaGraph_t g = nullptr; cudaGraphExec_t ex = nullptr;
    const int64_t before = h->launches;
    CK(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
    h->capturing = true;
    int rc = t_srk3(h, dt);
    h->capturing = false;
    cudaError_t e = cudaStreamEndCapture(h->stream, &g);
    const int64_t per = h->launches - before;
    h->launches = before;
    if (rc) { if (g) cudaGraphDestroy(g); return rc; }
    if (e != cudaSuccess) { h->err = std::string("cudaStreamEndCapture: ") + cudaGetErrorString(e); return MPASB200_ECUDA; }
    CK(cudaGraphInstantiate(&ex, g, 0));
    cudaGraphDestroy(g);
    it = h->graphs.emplace(dt, std::make_pair(ex, per)).first;
  }
  CK(cudaGraphLaunch(it->second.first, h->stream));
  h->launches += it->second.second;
  return 0;
}
int mpasb200_timestep(mpasb200_t* h, double dt) { return mpasb200_srk3(h, dt); }   // rk_timestep.rg:503-519

// ---- halo building blocks -----------------------------------------------------------------------------------
int mpasb200_register_list(mpasb200_t* h, int entity, const int32_t* idx, int32_t n, int32_t* list_id) {
  REQUIRE_MESH();
  if (entity < 0 || entity > MPASB200_VERTEX || n < 0 || (!idx && n > 0) || !list_id) return fail(h, MPASB200_EINVAL, "register_list: bad argument");
  std::unique_lock<std::mutex> lk(h->mu);
  cudaSetDevice(h->device);
  const int cnt = entity_count(h, entity);
  std::vector<int> tmp(n);
  for (int i = 0; i < n; ++i) {
    if (idx[i] < 0 || idx[i] >= cnt) return fail(h, MPASB200_EINVAL, "register_list: index out of range");
    tmp[i] = h->newOf[entity][idx[i]];
  }
  HaloList l{entity, n, nullptr};
  if (n > 0) {
    CK(cudaMalloc((void**)&l.d_idx, sizeof(int) * n));
    CK(cudaMemcpy(l.d_idx, tmp.data(), sizeof(int) * n, cudaMemcpyHostToDevice));
  }
  h->lists.push_back(l);
  *list_id = (int32_t)h->lists.size() - 1;
  return 0;
}
static int pack_unpack(mpasb200_t* h, int list_id, const int32_t* fields, int32_t nfields, void* d_buf, bool pack) {
  REQUIRE_MESH();
  std::unique_lock<std::mutex> lk(h->mu);
  cudaSetDevice(h->device);
  if (list_id < 0 || list_id >= (int)h->lists.size() || !fields || nfields < 1 || nfields > 32 || !d_buf) return fail(h, MPASB200_EINVAL, "pack/unpack: bad argument");
  const HaloList& l = h->lists[list_id];
  if (l.n == 0) return 0;
  // an array-typed field (scalars : double[8]) travels as one buffer entry per slot, slots in order
  PackArgs A; A.nf = 0;
  const size_t slotStride = (size_t)(entity_count(h, l.entity) + 1) * h->LP;
  for (int i = 0; i < nfields; ++i) {
    if (fields[i] < 0 || fields[i] >= MPASB200_F_COUNT || kFields[fields[i]].entity != l.entity)
      return fail(h, MPASB200_EINVAL, "pack/unpack: field does not live on the list's entity type");
    for (int sl = 0; sl < kFields[fields[i]].slots; ++sl) {
      if (A.nf >= 32) return fail(h, MPASB200_EINVAL, "pack/unpack: more than 32 buffer entries (fields x slots)");
      A.f[A.nf++] = h->V.f[fields[i]] + sl * slotStride;
    }
  }
  const int rows = std::max(1, 128 / h->LP);
  dim3 block(h->LP, rows), grid((l.n + rows - 1) / rows, A.nf);
  if (pack) k_pack<<<grid, block, 0, h->stream>>>(A, l.d_idx, l.n, h->L1, h->LP, (double*)d_buf);
  else k_unpack<<<grid, block, 0, h->stream>>>(A, l.d_idx, l.n, h->L1, h->LP, (const double*)d_buf);
  h->launches++;
  return post_launch(h);
}
int mpasb200_pack(mpasb200_t* h, int list_id, const int32_t* fields, int32_t nfields, void* d_buf) { return pack_unpack(h, list_id, fields, nfields, d_buf, true); }
int mpasb200_unpack(mpasb200_t* h, int list_id, const int32_t* fields, int32_t nfields, const void* d_buf) { return pack_unpack(h, list_id, fields, nfields, const_cast<void*>(d_buf), false); }

// ---- summarize_timestep (rk_timestep.rg:29-359) as a device scan ------------------------------------------------------
int mpasb200_set_global_ids(mpasb200_t* h, int entity, const int32_t* gid, int32_t n) {
  REQUIRE_MESH();
  if (entity < 0 || entity > MPASB200_VERTEX) return fail(h, MPASB200_EINVAL, "set_global_ids: bad entity");
  std::unique_lock<std::mutex> lk(h->mu);
  cudaSetDevice(h->device);
  if (h->d_gid[entity]) { cudaFree(h->d_gid[entity]); h->d_gid[entity] = nullptr; h->n_gid[entity] = 0; }
  if (!gid) return 0;
  if (n < 0 || n > entity_count(h, entity)) return fail(h, MPASB200_EINVAL, "set_global_ids: n out of range");
  for (int i = 0; i < n; ++i) if (gid[i] < 0) return fail(h, MPASB200_EINVAL, "set_global_ids: negative id");
  if (n > 0) {
    CK(cudaMalloc((void**)&h->d_gid[entity], sizeof(int) * n));
    CK(cudaMemcpy(h->d_gid[entity], gid, sizeof(int) * n, cudaMemcpyHostToDevice));
  }
  h->n_gid[entity] = n;
  return 0;
}
int mpasb200_summarize_field(mpasb200_t* h, int field, int32_t n_first, int32_t nlevels, MpasFieldSummary* out) {
  REQUIRE_MESH();
  if (!out || field < 0 || field >= MPASB200_F_COUNT) return fail(h, MPASB200_EINVAL, "summarize_field: bad argument");
  const FieldInfo& fi = kFields[field];
  if (fi.entity == MPASB200_VERTICAL || fi.slots != 1) return fail(h, MPASB200_EINVAL, "summarize_field: scalar 3-D fields only");
  std::unique_lock<std::mutex> lk(h->mu);
  cudaSetDevice(h->device);
  if (h->capturing) return fail(h, MPASB200_ESTATE, "summarize_field during graph capture");
  const int n = entity_count(h, fi.entity);
  if (n_first < 0 || n_first > n || nlevels < 1 || nlevels > h->L1) return fail(h, MPASB200_EINVAL, "summarize_field: range");
  const int* gid = h->d_gid[fi.entity];
  if (gid && h->n_gid[fi.entity] < n_first) return fail(h, MPASB200_EINVAL, "summarize_field: fewer global ids than entities scanned");
  if (!h->d_acc) CK(cudaMalloc((void**)&h->d_acc, sizeof(SumAcc)));
  SumAcc a; a.kmin = ~0ULL; a.kmax = 0ULL; a.n_nan = a.n_inf = a.checksum = 0ULL; a.loc_min = a.loc_max = ~0ULL;
  CK(cudaMemcpyAsync(h->d_acc, &a, sizeof(a), cudaMemcpyHostToDevice, h->stream));
  const size_t total = (size_t)n_first * nlevels;
  if (total > 0) {
    const int blocks = (int)std::min<size_t>((total + 255) / 256, (size_t)h->num_sms * 16);
    { KTimer kt_(h, "k_summarize"); k_summarize<<<blocks, 256, 0, h->stream>>>(h->V.f[field], h->d_newOf[fi.entity], gid, n_first, nlevels, h->LP, h->d_acc); h->launches++; }
    { KTimer kt_(h, "k_summarize_loc"); k_summarize_loc<<<blocks, 256, 0, h->stream>>>(h->V.f[field], h->d_newOf[fi.entity], gid, n_first, nlevels, h->LP, h->d_acc); h->launches++; }
    CK(cudaGetLastError());
  }
  CK(cudaMemcpyAsync(&a, h->d_acc, sizeof(a), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  auto unkey = [](unsigned long long k) { unsigned long long b = (k & 0x8000000000000000ULL) ? (k & 0x7fffffffffffffffULL) : ~k; double v; std::memcpy(&v, &b, 8); return v; };
  const bool any = a.kmin <= a.kmax;
  out->min = any ? unkey(a.kmin) : INFINITY; out->max = any ? unkey(a.kmax) : -INFINITY;
  out->min_index = any ? (int64_t)(a.loc_min / (unsigned long long)nlevels) : -1; out->min_level = any ? (int32_t)(a.loc_min % (unsigned long long)nlevels) : -1;
  out->max_index = any ? (int64_t)(a.loc_max / (unsigned long long)nlevels) : -1; out->max_level = any ? (int32_t)(a.loc_max % (unsigned long long)nlevels) : -1;
  out->n_nan = (int64_t)a.n_nan; out->n_inf = (int64_t)a.n_inf; out->count = (int64_t)total; out->checksum = a.checksum;
  return 0;
}

// ---- surface pressure and pressure-level diagnostics (k_isobaric) ---------------------------------------------------------------
int mpasb200_isobaric_diagnostics(mpasb200_t* h, const double* plev, int32_t nplev, int32_t n_first, double* out) {
  REQUIRE_MESH();
  if (!out || !plev) return fail(h, MPASB200_EINVAL, "isobaric_diagnostics: null out or plev");
  if (nplev < 1 || nplev > MPASB200_ISOBARIC_MAX_LEVELS) return fail(h, MPASB200_EINVAL, "isobaric_diagnostics: nplev outside [1, 32]");
  IsoLevels P{};
  P.n = nplev;
  for (int j = 0; j < nplev; ++j) {
    if (!std::isfinite(plev[j]) || !(plev[j] > 0.0)) return fail(h, MPASB200_EINVAL, "isobaric_diagnostics: a plev entry is not finite and > 0");
    P.p[j] = plev[j];
  }
  if (n_first < 0 || n_first > h->nCells) return fail(h, MPASB200_EINVAL, "isobaric_diagnostics: n_first outside [0, nCells]");
  std::unique_lock<std::mutex> lk(h->mu);
  cudaSetDevice(h->device);
  if (h->capturing) return fail(h, MPASB200_ESTATE, "isobaric_diagnostics during graph capture");
  const size_t elems = (size_t)n_first * (1 + 6 * nplev);
  if (elems == 0) return 0;
  if (h->iso_elems < elems) {
    if (h->d_iso) { CK(cudaFree(h->d_iso)); h->d_iso = nullptr; h->iso_elems = 0; }
    CK(cudaMalloc((void**)&h->d_iso, sizeof(double) * elems));
    h->iso_elems = elems;
  }
  {
    KTimer kt_(h, "k_isobaric");
    k_isobaric<<<(n_first + ISO_WARPS - 1) / ISO_WARPS, 32 * ISO_WARPS, 0, h->stream>>>(h->V, h->d_newOf[MPASB200_CELL], P, n_first, h->d_iso);
    h->launches++;
  }
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out, h->d_iso, sizeof(double) * elems, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  return 0;
}

// ---- exact global integrals (k_integrate) ------------------------------------------------------------------------------------------
static_assert(IACC_LIMBS == MPASB200_INTEGRAL_LIMBS && IACC_BIAS == MPASB200_INTEGRAL_BIAS, "k_integrate and mpas_b200.h disagree");
int mpasb200_register_weights(mpasb200_t* h, int entity, const double* w, int32_t n, int32_t* weight_id) {
  REQUIRE_MESH();
  if (entity < 0 || entity > MPASB200_VERTEX || !w || !weight_id) return fail(h, MPASB200_EINVAL, "register_weights: bad argument");
  std::unique_lock<std::mutex> lk(h->mu);
  cudaSetDevice(h->device);
  if (n != entity_count(h, entity)) return fail(h, MPASB200_EINVAL, "register_weights: n is not the entity count");
  Weights x{entity, n, nullptr};
  CK(cudaMalloc((void**)&x.d_w, sizeof(double) * std::max(n, 1)));
  h->weights.push_back(x);                    // before the copy, so that destroy frees it whatever happens next
  if (n > 0) CK(cudaMemcpy(x.d_w, w, sizeof(double) * n, cudaMemcpyHostToDevice));
  *weight_id = (int32_t)h->weights.size() - 1;
  return 0;
}
int mpasb200_integrate(mpasb200_t* h, int field_a, int slot_a, int field_b, int slot_b, int weight_id, const double* wv,
                       int32_t n_first, int32_t nlevels, MpasIntegral* out) {
  REQUIRE_MESH();
  if (!out || field_a < 0 || field_a >= MPASB200_F_COUNT || field_b < -1 || field_b >= MPASB200_F_COUNT)
    return fail(h, MPASB200_EINVAL, "integrate: bad argument");
  const FieldInfo& fa = kFields[field_a];
  if (fa.entity == MPASB200_VERTICAL) return fail(h, MPASB200_EINVAL, "integrate: a vertical field");
  if (slot_a < 0 || slot_a >= fa.slots) return fail(h, MPASB200_EINVAL, "integrate: slot_a out of range");
  if (field_b >= 0) {
    if (kFields[field_b].entity != fa.entity) return fail(h, MPASB200_EINVAL, "integrate: field_b lives on another entity type");
    if (slot_b < 0 || slot_b >= kFields[field_b].slots) return fail(h, MPASB200_EINVAL, "integrate: slot_b out of range");
  }
  std::unique_lock<std::mutex> lk(h->mu);
  cudaSetDevice(h->device);
  if (h->capturing) return fail(h, MPASB200_ESTATE, "integrate during graph capture");
  if (weight_id < -1 || weight_id >= (int)h->weights.size()) return fail(h, MPASB200_EINVAL, "integrate: unknown weight_id");
  if (weight_id >= 0 && h->weights[weight_id].entity != fa.entity) return fail(h, MPASB200_EINVAL, "integrate: weights on another entity type");
  const int n = entity_count(h, fa.entity);
  if (n_first < 0 || n_first > n || nlevels < 1 || nlevels > h->L1) return fail(h, MPASB200_EINVAL, "integrate: range");
  const size_t slotStride = (size_t)(n + 1) * h->LP;          // array-typed fields: slots one after the other (as pack)
  const double* pa = h->V.f[field_a] + slot_a * slotStride;
  const double* pb = field_b >= 0 ? h->V.f[field_b] + slot_b * slotStride : nullptr;
  const double* pw = weight_id >= 0 ? h->weights[weight_id].d_w : nullptr;
  if (!h->d_iacc) CK(cudaMalloc((void**)&h->d_iacc, sizeof(IntAcc)));
  if (wv && !h->d_wv) CK(cudaMalloc((void**)&h->d_wv, sizeof(double) * h->L1));
  if (wv) CK(cudaMemcpyAsync(h->d_wv, wv, sizeof(double) * nlevels, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemsetAsync(h->d_iacc, 0, sizeof(IntAcc), h->stream));
  const size_t total = (size_t)n_first * nlevels;
  if (total > 0) {
    const int tpb = 32 * IACC_WARPS;
    const int blocks = (int)std::min<size_t>((total + tpb - 1) / tpb, (size_t)h->num_sms * 8);
    KTimer kt_(h, "k_integrate");
    k_integrate<<<blocks, tpb, 0, h->stream>>>(pa, pb, h->d_newOf[fa.entity], pw, wv ? h->d_wv : nullptr, n_first, nlevels, h->LP, h->d_iacc);
    h->launches++;
    CK(cudaGetLastError());
  }
  IntAcc a;
  CK(cudaMemcpyAsync(&a, h->d_iacc, sizeof(a), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));                        // also keeps wv borrowed for the call only
  MpasIntegral r{};
  for (int j = 0; j < IACC_LIMBS; ++j) r.limb[j] = a.limb[j];
  r.count = (int64_t)total; r.n_nan = (int64_t)a.n_nan; r.n_pinf = (int64_t)a.n_pinf; r.n_ninf = (int64_t)a.n_ninf;
  *out = MpasIntegral{};
  return mpasb200_integral_merge(out, &r);                     // the canonical form
}

namespace {
// exact canonical form of sum_j t[j] * 2^(32 j - BIAS): limbs 0..66 in [0, 2^32), the rest (signed) returned as the top
__int128 integral_canon(const __int128* t, int64_t* limb) {
  __int128 c = 0;
  for (int j = 0; j < MPASB200_INTEGRAL_LIMBS - 1; ++j) {
    const __int128 v = t[j] + c;
    limb[j] = (int64_t)(v & 0xffffffff);
    c = (v - limb[j]) / ((__int128)1 << 32);                    // exact: v - limb[j] is a multiple of 2^32
  }
  return t[MPASB200_INTEGRAL_LIMBS - 1] + c;
}
}  // namespace

int mpasb200_integral_merge(MpasIntegral* acc, const MpasIntegral* x) {
  if (!acc || !x) return MPASB200_EINVAL;
  __int128 t[MPASB200_INTEGRAL_LIMBS];
  for (int j = 0; j < MPASB200_INTEGRAL_LIMBS; ++j) t[j] = (__int128)acc->limb[j] + x->limb[j];
  int64_t limb[MPASB200_INTEGRAL_LIMBS];
  const __int128 top = integral_canon(t, limb);
  if (top > INT64_MAX || top < INT64_MIN) return MPASB200_EINVAL;    // |sum| >= 2^1119 (no library result gets near): acc unchanged
  limb[MPASB200_INTEGRAL_LIMBS - 1] = (int64_t)top;
  std::memcpy(acc->limb, limb, sizeof(limb));
  acc->count += x->count; acc->n_nan += x->n_nan; acc->n_pinf += x->n_pinf; acc->n_ninf += x->n_ninf;
  return 0;
}

double mpasb200_integral_value(const MpasIntegral* x) {
  constexpr int NL = MPASB200_INTEGRAL_LIMBS;
  if (!x || x->n_nan || (x->n_pinf && x->n_ninf)) return NAN;
  if (x->n_pinf) return INFINITY;
  if (x->n_ninf) return -INFINITY;
  __int128 t[NL];
  int64_t limb[NL];
  for (int j = 0; j < NL; ++j) t[j] = x->limb[j];
  __int128 top = integral_canon(t, limb);
  const bool neg = top < 0;
  if (neg) {                                                     // the magnitude: negate limb by limb, then canonicalise again
    for (int j = 0; j < NL - 1; ++j) t[j] = -(__int128)limb[j];
    t[NL - 1] = -top;
    top = integral_canon(t, limb);                              // now >= 0
  }
  // the magnitude as base-2^32 digits: limbs 0..66, then the 128-bit top in four digits
  uint32_t d[NL + 3];
  for (int j = 0; j < NL - 1; ++j) d[j] = (uint32_t)limb[j];
  for (int j = 0; j < 4; ++j) d[NL - 1 + j] = (uint32_t)((unsigned __int128)top >> (32 * j));
  int hi = NL + 2;
  while (hi >= 0 && d[hi] == 0) --hi;
  if (hi < 0) return 0.0;                                        // an exact zero is +0
  auto bit = [&](int b) { return (d[b >> 5] >> (b & 31)) & 1u; };
  const int msb = 32 * hi + 31 - __builtin_clz(d[hi]);            // bit index of the leading one
  const int e_msb = msb - MPASB200_INTEGRAL_BIAS;
  if (e_msb > 1023) return neg ? -INFINITY : INFINITY;
  const int lsb = std::max(e_msb - 52, -1074);                  // weight of the last bit a double keeps (subnormals: 2^-1074)
  const int q = lsb + MPASB200_INTEGRAL_BIAS;                    // >= 14
  uint64_t m = 0;
  for (int b = msb; b >= q; --b) m = (m << 1) | bit(b);
  bool sticky = false;                                          // any one below the rounding bit q - 1
  for (int j = 0; j < ((q - 1) >> 5) && !sticky; ++j) sticky = d[j] != 0;
  sticky = sticky || (d[(q - 1) >> 5] & ((1u << ((q - 1) & 31)) - 1u)) != 0;
  if (bit(q - 1) && (sticky || (m & 1))) ++m;                    // to nearest, ties to even
  const double r = std::ldexp((double)m, lsb);                  // exact, or +inf when rounding reached 2^1024
  return neg ? -r : r;
}

// ---- the distributed step ----------------------------------------------------------------------------------------------------
int mpasb200_dist_unique_id(void* id128) {
  if (!id128) return MPASB200_EINVAL;
  if (!nccl_load()) { g_create_error = g_nccl.err; return MPASB200_ESTATE; }
  return g_nccl.GetUniqueId(id128) == 0 ? 0 : MPASB200_ECUDA;
}
int mpasb200_dist_init(mpasb200_t* h, int rank, int world, const void* id128) {
  if (!h || !id128 || world < 1 || rank < 0 || rank >= world) return MPASB200_EINVAL;
  std::unique_lock<std::mutex> lk(h->mu);
  cudaSetDevice(h->device);
  if (h->comm) return fail(h, MPASB200_ESTATE, "dist_init may be called once per handle");
  if (!nccl_load()) return fail(h, MPASB200_ESTATE, g_nccl.err);
  NcclId128 id; std::memcpy(id.b, id128, 128);
  NCK(g_nccl.CommInitRank(&h->comm, world, id, rank));
  h->rank = rank; h->world = world;
  // highest priority: when the compute stream fills the GPU, the blocks of k_pack / the NCCL kernels / k_unpack are scheduled
  // ahead of the interior compute's pending blocks, so an exchange starts as soon as SMs drain instead of behind the whole kernel
  int prio_lo = 0, prio_hi = 0;
  cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
  CK(cudaStreamCreateWithPriority(&h->comm_stream, cudaStreamNonBlocking, prio_hi));
  CK(cudaEventCreateWithFlags(&h->ev_ready, cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&h->ev_done, cudaEventDisableTiming));
  CK(cudaEventCreateWithFlags(&h->ev_side, cudaEventDisableTiming));
  return 0;
}
int mpasb200_dist_set_halo(mpasb200_t* h, int entity, int32_t nsp, const int32_t* sp, const int32_t* so, const int32_t* si,
                           int32_t nrp, const int32_t* rp, const int32_t* ro, const int32_t* ri) {
  REQUIRE_MESH();
  if (entity < 0 || entity > MPASB200_VERTEX || nsp < 0 || nrp < 0) return fail(h, MPASB200_EINVAL, "dist_set_halo: bad argument");
  if ((nsp && (!sp || !so || !si)) || (nrp && (!rp || !ro || !ri))) return fail(h, MPASB200_EINVAL, "dist_set_halo: null list");
  std::unique_lock<std::mutex> lk(h->mu);
  cudaSetDevice(h->device);
  if (h->xplan_built) return fail(h, MPASB200_ESTATE, "dist_set_halo after the first exchange");
  mpasb200_t::Halo& H = h->halo[entity];
  const int cnt = entity_count(h, entity);
  auto load = [&](int np, const int32_t* peers, const int32_t* off, const int32_t* idx, std::vector<int>& P, std::vector<int>& O, int** d, int* n) -> int {
    P.assign(peers, peers + np); O.assign(1, 0);
    if (np) O.assign(off, off + np + 1);
    *n = np ? O[np] : 0;
    for (int i = 0; i < np; ++i) if (P[i] < 0 || P[i] >= h->world || P[i] == h->rank || O[i + 1] < O[i]) return fail(h, MPASB200_EINVAL, "dist_set_halo: bad peer / offsets");
    std::vector<int> tmp(*n);
    for (int i = 0; i < *n; ++i) { if (idx[i] < 0 || idx[i] >= cnt) return fail(h, MPASB200_EINVAL, "dist_set_halo: index out of range"); tmp[i] = h->newOf[entity][idx[i]]; }
    if (*d) { cudaFree(*d); *d = nullptr; }
    if (*n) { CK(cudaMalloc((void**)d, sizeof(int) * *n)); CK(cudaMemcpy(*d, tmp.data(), sizeof(int) * *n, cudaMemcpyHostToDevice)); }
    return 0;
  };
  int rc;
  if ((rc = load(nsp, sp, so, si, H.peers_s, H.off_s, &H.d_s, &H.ns))) return rc;
  if ((rc = load(nrp, rp, ro, ri, H.peers_r, H.off_r, &H.d_r, &H.nr))) return rc;
  H.set = true;
  return 0;
}
int mpasb200_dist_exchange(mpasb200_t* h, int kind) {
  REQUIRE_MESH();
  if (kind < 0 || kind >= MPASB200_X_COUNT) return fail(h, MPASB200_EINVAL, "dist_exchange: unknown kind");
  Entry en(h, -1);
  if (int rc = dist_finish(h)) return rc;
  return dist_exchange(h, kind);
}
int mpasb200_dist_flush(mpasb200_t* h) { REQUIRE_MESH(); Entry en(h, -1); return dist_finish(h); }
int mpasb200_srk3_dist(mpasb200_t* h, double dt) {
  REQUIRE_MESH();
  Entry en(h, -1);
  if (!h->comm) return fail(h, MPASB200_ESTATE, "mpasb200_dist_init has not been called");
  if (h->c.config_scalar_advection) { if (int rc = ensure_sflux(h)) return rc; }
  return t_srk3_dist(h, dt);
}

// ---- introspection ------------------------------------------------------------------------------------------------
int64_t mpasb200_launch_count(const mpasb200_t* h) { return h ? h->launches : 0; }
int64_t mpasb200_device_bytes(const mpasb200_t* h) { return h ? h->bytes : 0; }
int mpasb200_field_info(int field, int* entity, int* slots, const char** name) {
  if (field < 0 || field >= MPASB200_F_COUNT) return MPASB200_EINVAL;
  if (entity) *entity = kFields[field].entity;
  if (slots) *slots = kFields[field].slots;
  if (name) *name = kFields[field].name;
  return 0;
}
int mpasb200_field_by_name(const char* name) {
  if (!name) return -1;
  for (int i = 0; i < MPASB200_F_COUNT; ++i) if (!std::strcmp(name, kFields[i].name)) return i;
  return -1;
}
int mpasb200_restart_fields(const MpasConfig* cfg, int32_t* ids, int32_t cap) {
  if (!cfg) return MPASB200_EINVAL;
  const bool ALWAYS = true, CORRECTED = cfg->physics_mode == MPASB200_PHYSICS_CORRECTED, SCALARS = cfg->config_scalar_advection != 0;
  (void)CORRECTED;
  int32_t n = 0;
#define MPASB200_RESTART(name, when) \
  if (when) { if (ids && n < cap) ids[n] = MPASB200_F_##name; ++n; }
#include "../../include/mpas_b200_restart.def"
#undef MPASB200_RESTART
  return n;
}
#ifdef MPASB200_LAB
// Experimental launch variants of the divergence-damping kernel (not part of the public header): used by
// profiles/ scripts to measure latency-hiding structures.  variant 0 = production kernel.
int mpasb200_debug_divdamp(mpasb200_t* h, int variant, double dts, int arg) {
  REQUIRE_MESH();
  Entry en(h, -1);
  const double coef = 2.0 * h->c.config_smdiv * h->c.config_len_disp * (1.0 / dts);
  const int nE = h->nEdges, T = h->LP / 2, C = h->CPB;
  switch (variant) {
    case 0: { KTimer kt(h, "k_divdamp"); k_divdamp<<<h->num_sms * 9, dim3(T, C), 0, h->stream>>>(ranged(h, range_of(h, MPASB200_EDGE, nE)), coef); h->launches++; } break;
    case 1: LAUNCH(k_divdamp_v1, nE, 0, h->V, coef); break;
    case 2: LAUNCH(k_divdamp_v2, nE, 0, h->V, coef, arg); break;
    case 3: { KTimer kt(h, "k_divdamp_v3"); const int half = (nE + 1) / 2;
              k_divdamp_v3<<<(half + C - 1) / C, dim3(T, C), 0, h->stream>>>(h->V, coef); h->launches++; } break;
    case 4: { KTimer kt(h, "k_divdamp_v4"); k_divdamp_v4<<<arg, dim3(T, C), 0, h->stream>>>(h->V, coef); h->launches++; } break;
    case 5: { KTimer kt(h, "k_divdamp_v5"); const int T4 = h->LP / 4, C4 = 256 / T4;
              k_divdamp_v5<<<(nE + C4 - 1) / C4, dim3(T4, C4), 0, h->stream>>>(h->V, coef); h->launches++; } break;
    case 6: LAUNCH(k_divdamp_v6, nE, 0, h->V, coef, arg); break;
    case 7: { KTimer kt(h, "k_divdamp_v7"); const int T4 = h->LP / 4, C4 = 256 / T4;
              k_divdamp_v7<<<arg, dim3(T4, C4), 0, h->stream>>>(h->V, coef); h->launches++; } break;
    case 8: { KTimer kt(h, "k_divdamp_v8"); k_divdamp_v8<<<arg, dim3(T, C), 0, h->stream>>>(h->V, coef); h->launches++; } break;
    default: return fail(h, MPASB200_EINVAL, "unknown variant");
  }
  return post_launch(h);
}
// Ablation launches of the TMA acoustic kernel (profiling only; results are NOT the task's results).
int mpasb200_debug_acoustic(mpasb200_t* h, int abl, double dts) {
  REQUIRE_MESH();
  Entry en(h, -1);
  const View V = ranged(h, range_of(h, MPASB200_CELL, h->nCells));
  AcPtrs F;
#define AF(n) F.p[AF_##n] = V.f[MPASB200_F_##n]
  AF(tend_rho); AF(theta_m); AF(w); AF(coftz); AF(cofwz); AF(cofwr); AF(cofwt); AF(a_tri); AF(alpha_tri); AF(zz); AF(rw_save); AF(rw);
  AF(dss); AF(rho_zz); AF(rho_pp); AF(rtheta_pp); AF(rw_p); AF(wwAvg);
#undef AF
  F.p[AF_rs] = V.scr_rs; F.p[AF_ts] = V.scr_ts;
  const double epssm = h->c.config_epssm, resm = (1.0 - epssm) / (1.0 + epssm);
  const int C = 4, T = h->LP / 2, NF = (int)AF_COUNT;
  const size_t smem = ((size_t)NF * C * h->LP + (size_t)4 * C * (h->LP + 2)) * sizeof(double) + 16;
  dim3 block(T, C), grid((h->nCells + C - 1) / C);
  KTimer kt_(h, "k_acoustic_tma_abl");
  switch (abl) {
    case 0: k_acoustic_tma<false, 0><<<grid, block, smem, h->stream>>>(V, F, dts, epssm, resm); break;
    case 1: k_acoustic_tma<false, 1><<<grid, block, smem, h->stream>>>(V, F, dts, epssm, resm); break;
    case 2: k_acoustic_tma<false, 2><<<grid, block, smem, h->stream>>>(V, F, dts, epssm, resm); break;
    case 3: k_acoustic_tma<false, 3><<<grid, block, smem, h->stream>>>(V, F, dts, epssm, resm); break;
    case 4: k_acoustic_tma<false, 4><<<grid, block, smem, h->stream>>>(V, F, dts, epssm, resm); break;
    case 7: k_acoustic_tma<false, 7><<<grid, block, smem, h->stream>>>(V, F, dts, epssm, resm); break;
    default: return fail(h, MPASB200_EINVAL, "unknown ablation");
  }
  h->launches++;
  return post_launch(h);
}
#endif  // MPASB200_LAB
int mpasb200_enable_kernel_timing(mpasb200_t* h, int on) {
  if (!h) return MPASB200_EINVAL;
  std::unique_lock<std::mutex> lk(h->mu);
  cudaSetDevice(h->device);
  drain_kernel_times(h);
  h->ktiming = on != 0;
  h->ktimeline = on == 2;
  if (h->ktimeline) {          // the time origin of the timeline: now, on the compute stream
    if (!h->ktl_base) cudaEventCreate(&h->ktl_base);
    h->timeline.clear();
    cudaEventRecord(h->ktl_base, h->stream);
  }
  return 0;
}
// timeline mode: entry idx (launch order per drain) -> kernel name, start / end in ms since mode 2 was switched on, stream (0 = compute,
// 1 = the handle's communication stream).  MPASB200_EINVAL past the end.
int mpasb200_timeline_entry(mpasb200_t* h, int idx, const char** name, double* t0_ms, double* t1_ms, int* stream) {
  if (!h) return MPASB200_EINVAL;
  std::unique_lock<std::mutex> lk(h->mu);
  cudaSetDevice(h->device);
  drain_kernel_times(h);
  if (idx < 0 || idx >= (int)h->timeline.size()) return MPASB200_EINVAL;
  const auto& e = h->timeline[idx];
  if (name) *name = h->kstats[e.stat].name.c_str();
  if (t0_ms) *t0_ms = e.t0;
  if (t1_ms) *t1_ms = e.t1;
  if (stream) *stream = e.comm ? 1 : 0;
  return 0;
}
int mpasb200_reset_kernel_timing(mpasb200_t* h) {
  if (!h) return MPASB200_EINVAL;
  std::unique_lock<std::mutex> lk(h->mu);
  cudaSetDevice(h->device);
  drain_kernel_times(h);
  h->kstats.clear();
  return 0;
}
int mpasb200_kernel_time(mpasb200_t* h, int idx, const char** name, double* ms, int64_t* launches) {
  if (!h) return MPASB200_EINVAL;
  std::unique_lock<std::mutex> lk(h->mu);
  cudaSetDevice(h->device);
  drain_kernel_times(h);
  if (idx < 0 || idx >= (int)h->kstats.size()) return MPASB200_EINVAL;
  if (name) *name = h->kstats[idx].name.c_str();
  if (ms) *ms = h->kstats[idx].ms;
  if (launches) *launches = h->kstats[idx].n;
  return 0;
}
int mpasb200_enable_timing(mpasb200_t* h, int on) { if (!h) return MPASB200_EINVAL; std::unique_lock<std::mutex> lk(h->mu); h->timing = on != 0; return 0; }
int mpasb200_reset_timing(mpasb200_t* h) {
  if (!h) return MPASB200_EINVAL;
  std::unique_lock<std::mutex> lk(h->mu);
  for (int i = 0; i < MPASB200_T_COUNT; ++i) { h->task_ms[i] = 0; h->task_calls[i] = 0; }
  return 0;
}
int mpasb200_task_time(mpasb200_t* h, int task, double* ms, int64_t* calls, const char** name) {
  if (!h || task < 0 || task >= MPASB200_T_COUNT) return MPASB200_EINVAL;
  std::unique_lock<std::mutex> lk(h->mu);
  if (ms) *ms = h->task_ms[task];
  if (calls) *calls = h->task_calls[task];
  if (name) *name = kTaskNames[task];
  return 0;
}

}  // extern "C"
