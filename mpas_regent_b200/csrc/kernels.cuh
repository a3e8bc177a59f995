// kernels.cuh -- hand-written sm_100a kernels for the RK3 dynamics hot path.
//
// Thread mapping (all stencil kernels): blockDim = (LP/2, CPB).  threadIdx.x owns the level PAIR
// (2*tx, 2*tx+1) of one column -- levels are contiguous in memory and LP is a multiple of 4, so
// every access to a 3-D field is one aligned 128-bit load/store and a column is a run of
// consecutive 16-byte words across the lanes; threadIdx.y = column within the block, CPB chosen so
// the block is a multiple of 32 threads.  A block owns CPB whole columns, so column neighbours
// (k-2..k+1) produced inside a kernel are exchanged through shared memory; neighbour columns
// (edgesOnCell, cellsOnEdge, advCellsForEdge ...) are gathered from L2/HBM as contiguous level strips
// after ONE level of index loads (per-(cell,slot) copies of the edge statics, view.h).  Flux
// divergences are cell-centric gathers over edgesOnCell in slot order: no atomics, bit-reproducible.
// Every kernel is HBM-bound (fp64, ~0.3 flop/B); the design goal is bytes in flight per thread.
//
// Arithmetic follows the reference's expression order (compiled with --fmad=false) so that
// results agree with the CPU oracle to the last bit wherever no libm call is involved.
// Each kernel cites the reference lines it implements (dynamics/dynamics_tasks.rg).
#pragma once
#include "view.h"

#define DI __device__ __forceinline__
// minimum resident blocks per SM requested from ptxas (register caps); tuned by measurement, see profiles/
#ifndef LB_EDGE
#define LB_EDGE 1
#endif
#ifndef LB_CELLC
#define LB_CELLC 4
#endif
#ifndef LB_CELLC_SPLIT
#define LB_CELLC_SPLIT 5
#endif
#ifndef LB_AC
#define LB_AC 3
#endif
#ifndef KDE_PREFETCH
#define KDE_PREFETCH 1       /* measured: k_dt_edge 2.208 -> 2.135 ms/step on x1.163842 (profiles/r2_small_experiments.md) */
#endif
#ifndef LB_MISC
#define LB_MISC 1
#endif
// Stall-guided forms (profiles/r2_stall_profiles.md, GPU calls 18-23; x1.163842 x 55, ms per step, all bit-identical).  Adopted:
//  * HOIST: loads whose latency sat in front of a barrier or at the head of a dependent chain -- the one-lane level-L reads of
//    k_dt_edge / k_dt_cellC / k_vert_imp, the length of the edgesOnEdge row -- are requested at the top of the kernel and consumed
//    where they were read before (k_dt_edge 2.139 -> 1.874 at the same 56 registers, k_dt_cellC<false> 1.259 -> 1.234, <true>
//    0.614 -> 0.590, k_vert_imp 0.626 -> 0.584);
//  * w_adv_curv leaves out the advection-coefficient loads whose values are multiplied by an exact 0.0 (k_dt_cellC<false>
//    1.362 -> 1.259, k_dt_cellA 0.357 -> 0.322); slot 0 of k_diag_cell peeled, dcEdge from a per-(cell, slot) copy (0.411 -> 0.384);
//  * cross-block prefetch of the index WORDS / ROWS of the block about one wave later (XPF_*): k_acoustic_gather 1.146 -> 1.102,
//    k_dt_edge 1.868 -> 1.830, k_diag_cell, k_diag_edge, k_dt_edge_euler, k_dt_cellA/B -1 .. -4 %; k_dt_cellC and k_dt_theta_flux
//    got slower with it (+0.6 %) and go without;
//  * static rows staged in shared memory by lane-distributed loads where a slot loop read several statics per slot: the advection
//    row of k_dt_theta_flux (ids + coefficient pairs; 0.756 -> 0.615) and the theta-loop rows of k_dt_cellC<false> (1.236 -> 1.205);
//    k_smlstep requests its two masks and the row length together (0.820 -> 0.799).
// Measured and removed: the neighbour columns of 2..6 slots of a gather loop requested together (ptxas issues slot j+1's gathers
// after slot j's arithmetic) -- k_dt_edge 2.11 .. 2.64, k_acoustic_gather 1.29 .. 1.96 against 1.148, k_dt_theta_flux 1.01 against
// 0.756, k_diag_cell 0.46 .. 0.60 against 0.411: resident warps, not loads in flight per thread, carry these kernels; slot 0's statics
// and columns peeled in front of the row length (k_acoustic_gather +4 %, k_dt_theta_flux +27 %, k_dt_edge +8 %); a last-edge static
// for w_adv_curv (+1 %); prefetch.global.L1 instead of .L2 (no change); in-thread L2 prefetch of the columns a slot loop will
// gather, lanes spread over slot x line (k_dt_edge +11 %, k_dt_theta_flux +9 %, k_acoustic_gather -0.8 %); the same row staging in
// k_dt_edge (Coriolis row, +12 %), k_acoustic_gather (+10 %) and k_dt_cellC<true> (+8 %); an L2 prefetch of k_smlstep's own strips (+10 %);
// register caps that buy a resident block (k_acoustic_gather 48 / 40 registers: +3 % / +9 %, k_divdamp 48: +2 %).
#ifndef KDE_MAXREG
#define KDE_MAXREG 56        /* the hoisted values would cost k_dt_edge a resident block (60 registers): capped, 8 bytes of spills */
#endif
// cross-block row prefetch of a cell kernel / an edge kernel (statics of the block about one wave later)
#define XPF_CELL_ROWS() do { if (threadIdx.y < 2) prefetch_cell_rows(V, (long)x + (long)(PF_AHEAD + threadIdx.y * 4) * blockDim.y, threadIdx.x); } while (0)
#define XPF_EDGE_WORDS() do { if (threadIdx.y == 0 && threadIdx.x < 3) { const long xa_ = (long)x + (long)PF_AHEAD * blockDim.y; \
    if (xa_ < V.nEdges) { if (threadIdx.x == 0) prefetch_l2(V.ecv + xa_); if (threadIdx.x == 1) prefetch_l2(V.invDcEdge + xa_); if (threadIdx.x == 2) prefetch_l2(V.invDvEdge + xa_); } } } while (0)
typedef double2 D2;

DI D2 mk(double a, double b) { return make_double2(a, b); }
DI D2 bc(double a) { return make_double2(a, a); }
DI D2 operator+(D2 a, D2 b) { return mk(a.x + b.x, a.y + b.y); }
DI D2 operator-(D2 a, D2 b) { return mk(a.x - b.x, a.y - b.y); }
DI D2 operator*(D2 a, D2 b) { return mk(a.x * b.x, a.y * b.y); }
DI D2 operator/(D2 a, D2 b) { return mk(a.x / b.x, a.y / b.y); }
DI D2 operator+(D2 a, double b) { return mk(a.x + b, a.y + b); }
DI D2 operator-(D2 a, double b) { return mk(a.x - b, a.y - b); }
DI D2 operator*(D2 a, double b) { return mk(a.x * b, a.y * b); }
DI D2 operator/(D2 a, double b) { return mk(a.x / b, a.y / b); }
DI D2 operator+(double a, D2 b) { return mk(a + b.x, a + b.y); }
DI D2 operator-(double a, D2 b) { return mk(a - b.x, a - b.y); }
DI D2 operator*(double a, D2 b) { return mk(a * b.x, a * b.y); }
DI D2 operator/(double a, D2 b) { return mk(a / b.x, a / b.y); }
DI D2 operator-(D2 a) { return mk(-a.x, -a.y); }
DI D2& operator+=(D2& a, D2 b) { a.x += b.x; a.y += b.y; return a; }
DI D2& operator-=(D2& a, D2 b) { a.x -= b.x; a.y -= b.y; return a; }
DI D2& operator*=(D2& a, D2 b) { a.x *= b.x; a.y *= b.y; return a; }
DI D2& operator*=(D2& a, double b) { a.x *= b; a.y *= b; return a; }
DI D2& operator/=(D2& a, D2 b) { a.x /= b.x; a.y /= b.y; return a; }
DI D2 sgn1(D2 v) { return mk(copysign(1.0, v.x), copysign(1.0, v.y)); }
DI double dmin(double a, double b) { return (b < a) ? b : a; }     // std::min
DI double dmax(double a, double b) { return (a < b) ? b : a; }     // std::max
DI D2 sel(bool c0, bool c1, D2 a, D2 b) { return mk(c0 ? a.x : b.x, c1 ? a.y : b.y); }
DI D2 ld2(const double* p, size_t i) { return *reinterpret_cast<const D2*>(p + i); }
DI void st2(double* p, size_t i, D2 v) { *reinterpret_cast<D2*>(p + i) = v; }
// streaming forms for strips nobody reads again in this kernel: evict-first loads / stores leave L1 and L2 to the gathered columns
DI D2 ld2s(const double* p, size_t i) { return __ldcs(reinterpret_cast<const D2*>(p + i)); }
DI void st2s(double* p, size_t i, D2 v) { __stcs(reinterpret_cast<D2*>(p + i), v); }
DI void st2ms(double* p, size_t i, D2 v, bool m0, bool m1) {
  if (m0 && m1) st2s(p, i, v);
  else { if (m0) __stcs(p + i, v.x); if (m1) __stcs(p + i + 1, v.y); }
}
// store the components whose mask is set (a pair that straddles the top level stores one double)
DI void st2m(double* p, size_t i, D2 v, bool m0, bool m1) {
  if (m0 && m1) st2(p, i, v);
  else { if (m0) p[i] = v.x; if (m1) p[i + 1] = v.y; }
}

DI void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
// Blocks are short-lived (8 columns each), so the index loads at the top of a block are an exposed DRAM round
// trip.  Every block therefore prefetches into L2 the static index rows of the block that will run about one
// wave later (profiles/r1_divdamp_variants.md: +11 % on a light gather kernel for three instructions).
#define PF_AHEAD 1400    /* ~ resident blocks on 148 SMs */
DI void prefetch_cell_rows(const View& V, long xa, int lane) {
  if (xa >= V.nCells) return;
  const int ME = V.maxEdges;
  switch (lane) {
    case 0: prefetch_l2(V.edgesOnCell + xa * V.MEP); prefetch_l2(V.nEdgesOnCell + xa); break;
    case 1: prefetch_l2(V.c1OnCell + xa * V.MEP); break;
    case 2: prefetch_l2(V.c2OnCell + xa * V.MEP); break;
    case 3: prefetch_l2(V.edgesOnCell_sign + xa * ME); break;
    case 4: prefetch_l2(V.edgesOnCellSign + xa * ME); break;
    case 5: prefetch_l2(V.dvOnCell + xa * ME); break;
    case 6: prefetch_l2(V.invDcOnCell + xa * ME); prefetch_l2(V.invAreaCell + xa); break;
    case 7: prefetch_l2(V.ms2OnCell + xa * ME); prefetch_l2(V.ms4OnCell + xa * ME); break;
    default: break;
  }
}
DI void prefetch_edge_rows(const View& V, long xa, int lane, const int* eoe) {
  if (xa >= V.nEdges) return;
  switch (lane) {
    case 0: prefetch_l2(V.ecv + xa); break;
    case 1: prefetch_l2(V.invDcEdge + xa); prefetch_l2(V.invDvEdge + xa); break;
    case 2: if (eoe) { prefetch_l2(eoe + xa * V.maxEdges2); prefetch_l2(eoe + xa * V.maxEdges2 + 16); } break;
    case 3: if (eoe) { prefetch_l2(V.weightsOnEdge + xa * V.maxEdges2); prefetch_l2(V.weightsOnEdge + xa * V.maxEdges2 + 16); } break;
    default: break;
  }
}
#define PF_CELLS() prefetch_cell_rows(V, (long)x + (long)PF_AHEAD * blockDim.y, threadIdx.x)
#define PF_EDGES(eoe) prefetch_edge_rows(V, (long)x + (long)PF_AHEAD * blockDim.y, threadIdx.x, (eoe))

#define FLD(name) (V.f[MPASB200_F_##name])
#define PAIR_THREAD(n)                                          \
  const int k0 = 2 * (int)threadIdx.x, k1 = k0 + 1;             \
  const int x = blockIdx.x * blockDim.y + threadIdx.y;          \
  const bool inx = x < (n);                                     \
  const int LP = V.LP; const int L = V.L;                       \
  const size_t ix = (size_t)(inx ? x : 0) * LP + k0;            \
  const bool m0 = inx && k0 < L, m1 = inx && k1 < L;            \
  (void)ix; (void)m1; (void)k1;
// the same for the kernels that honour mpasb200_set_range: internal indices [V.xoff, V.xend), xend <= n set by the host
#define PAIR_THREAD_R()                                         \
  const int k0 = 2 * (int)threadIdx.x, k1 = k0 + 1;             \
  const int x = V.xoff + blockIdx.x * blockDim.y + threadIdx.y; \
  const bool inx = x < V.xend;                                  \
  const int LP = V.LP; const int L = V.L;                       \
  const size_t ix = (size_t)(inx ? x : 0) * LP + k0;            \
  const bool m0 = inx && k0 < L, m1 = inx && k1 < L;            \
  (void)ix; (void)m1; (void)k1;
#define G2(p, e) ld2((p), (size_t)(e) * LP + k0)                 /* the level pair of neighbour column e */
#define G1(p, e, k_) ((p)[(size_t)(e) * LP + (k_)])
// (Measured and removed, profiles/r2_small_experiments.md: taking the cell's OWN level pair from a register instead of gathering it
// again in the edgesOnCell loops -- one of the two cells of every slot is the cell itself -- saves a third of those gathers and is
// SLOWER: k_acoustic_gather 1.147 -> 1.237 ms/step, k_dt_cellA 0.357 -> 0.440, k_dt_cellB 0.267 -> 0.332 on x1.163842.  So is packing
// the per-slot statics of k_acoustic_gather into one 16-byte id word + one sign*dvEdge double: 1.151 -> 1.256.)
#ifndef CELLC_PREFETCH
#define CELLC_PREFETCH 1     /* measured: k_dt_cellC<false> 1.392 -> 1.363 ms/step on x1.163842 (profiles/r2_small_experiments.md) */
#endif
// values one level below / above the pair: (f[k0-1], f[k0]) and (f[k1], f[k1+1])
DI D2 below(const double* p, size_t ix, int k0, D2 cur) { return mk(k0 > 0 ? p[ix - 1] : 0.0, cur.x); }
DI D2 above(const double* p, size_t ix, int k0, int L, D2 cur) { return mk(cur.y, (k0 + 2 <= L) ? p[ix + 2] : 0.0); }

DI double flux4(double q_im2, double q_im1, double q_i, double q_ip1, double ua) {
  return ua * (7. * (q_i + q_im1) - (q_ip1 + q_im2)) / 12.0;                       // :781-783
}
DI double flux3(double q_im2, double q_im1, double q_i, double q_ip1, double ua, double coef3) {
  return flux4(q_im2, q_im1, q_i, q_ip1, ua) + coef3 * fabs(ua) * ((q_ip1 - q_im2) - 3. * (q_i - q_im1)) / 12.0;   // :786-789
}

// ============================================================================================
// atm_rk_integration_setup  :747-778
__global__ void k_setup_cell(const View V) {
  PAIR_THREAD(V.nCells)
  if (!m0) return;
  st2m(FLD(rw_save), ix, ld2(FLD(rw), ix), m0, m1);
  st2m(FLD(rtheta_p_save), ix, ld2(FLD(rtheta_p), ix), m0, m1);
  st2m(FLD(rho_p_save), ix, ld2(FLD(rho_p), ix), m0, m1);
  st2m(FLD(w_2), ix, ld2(FLD(w), ix), m0, m1);
  st2m(FLD(theta_m_2), ix, ld2(FLD(theta_m), ix), m0, m1);
  const D2 r = ld2(FLD(rho_zz), ix);
  st2m(FLD(rho_zz_2), ix, r, m0, m1);
  st2m(FLD(rho_zz_old_split), ix, r, m0, m1);
}
__global__ void k_setup_edge(const View V) {
  PAIR_THREAD(V.nEdges)
  if (!m0) return;
  st2m(FLD(ru_save), ix, ld2(FLD(ru), ix), m0, m1);
  st2m(FLD(u_2), ix, ld2(FLD(u), ix), m0, m1);
}

// atm_compute_moist_coefficients  :460-502   (qtot = 0; cqw from it for k > 0; cqu never written)
__global__ void k_moist(const View V) {
  PAIR_THREAD(V.nCells)
  if (!m0) return;
  const double qz = 0.0;
  st2m(FLD(qtot), ix, bc(qz), m0, m1);
  const double qtotal = 0.5 * (qz + qz);
  st2m(FLD(cqw), ix, bc(1.0 / (1.0 + qtotal)), m0 && k0 > 0, m1);
}

// atm_compute_vert_imp_coefs  :513-592
// One block owns whole columns: everything read from the previous call (gamma_tri[k-1]) is read
// before the barrier, everything this call produces for neighbours (coftz, cofwt) goes through smem.
__global__ void k_vert_imp(const View V, double dtseps, double c2, double rcv, double gravity) {
  extern __shared__ double sm[];
  PAIR_THREAD(V.nCells)
  const int TS = LP + 2;
  double* s_coftz = sm + (size_t)threadIdx.y * TS;
  double* s_cofwt = sm + (size_t)(blockDim.y + threadIdx.y) * TS;
  if (blockIdx.x == 0 && threadIdx.y == 0) {                                                         // :537-539
    if (k0 < L) FLD(cofrz)[k0] = dtseps * FLD(rdzw)[k0];
    if (k1 < L) FLD(cofrz)[k1] = dtseps * FLD(rdzw)[k1];
  }
  D2 zz = bc(0), zzm = bc(0), coftz = bc(0), cofwt = bc(0), cofwr = bc(0), cofwz = bc(0), gprev = bc(0);
  D2 rdzw2 = bc(0), rdzwm = bc(0);
  double coftz_L = 0.0;                  // level L is never written: whatever the mirror holds (requested first, stored in front of the barrier)
  if (inx && k0 == L) coftz_L = FLD(coftz)[ix];
  if (inx && k1 == L) coftz_L = FLD(coftz)[ix + 1];
  if (m0) {
    const D2 fzm = ld2(FLD(fzm), k0), fzp = ld2(FLD(fzp), k0), rdzu = ld2(FLD(rdzu), k0);
    rdzw2 = ld2(FLD(rdzw), k0); rdzwm = below(FLD(rdzw), k0, k0, rdzw2);
    zz = ld2(FLD(zz), ix); zzm = below(FLD(zz), ix, k0, zz);
    const D2 ex = ld2(FLD(exner), ix), exm = below(FLD(exner), ix, k0, ex);
    const D2 th = ld2(FLD(theta_m), ix), thm = below(FLD(theta_m), ix, k0, th);
    const D2 zf = fzm * zz + fzp * zzm;
    cofwr = .5 * dtseps * gravity * zf;                                                               // :552
    cofwz = dtseps * c2 * zf * rdzu * ld2(FLD(cqw), ix) * (fzm * ex + fzp * exm);                     // :557
    coftz = dtseps * (fzm * th + fzp * thm);                                                          // :558
    if (k0 == 0) coftz.x = 0.0;                                                                       // :555
    const D2 g = ld2(FLD(gamma_tri), ix);                      // previous call's gamma (:583)
    gprev = mk(k0 > 1 ? FLD(gamma_tri)[ix - 1] : 0.0, k0 > 0 ? g.x : 0.0);                            // gamma(0) = 0 (:545)
    const D2 qtotal = ld2(FLD(qtot), ix);
    cofwt = .5 * dtseps * rcv * zz * gravity * ld2(FLD(rho_base), ix) / (1.0 + qtotal) * ex
            / ((ld2(FLD(rtheta_base), ix) + ld2(FLD(rtheta_p), ix)) * ld2(FLD(exner_base), ix));      // :563
    s_coftz[k0] = coftz.x; s_cofwt[k0] = cofwt.x;
    if (m1) { s_coftz[k1] = coftz.y; s_cofwt[k1] = cofwt.y; }
  }
  // level L is never written: whatever the mirror holds
  if (inx && (k0 == L || k1 == L)) s_coftz[L] = coftz_L;
  __syncthreads();
  if (!m0) return;
  st2m(FLD(coftz), ix, coftz, m0, m1); st2m(FLD(cofwt), ix, cofwt, m0, m1);
  const bool w0 = k0 > 0, w1 = m1;
  st2m(FLD(cofwr), ix, cofwr, w0, w1); st2m(FLD(cofwz), ix, cofwz, w0, w1);
  const D2 coftz_m = mk(k0 > 0 ? s_coftz[k0 - 1] : 0.0, coftz.x);
  const D2 coftz_p = mk(m1 ? s_coftz[k1] : s_coftz[L], m1 ? s_coftz[k1 + 1] : 0.0);
  const D2 cofwt_m = mk(k0 > 0 ? s_cofwt[k0 - 1] : 0.0, cofwt.x);
  const D2 cofrz = dtseps * rdzw2, cofrz_m = dtseps * rdzwm;
  const D2 a = -1.0 * cofwz * coftz_m * rdzwm * zzm + cofwr * cofrz_m - cofwt_m * coftz_m * rdzwm;    // :568-569
  const D2 b = 1.0 + cofwz * (coftz * rdzw2 * zz + coftz * rdzwm * zzm)
               - coftz * (cofwt * rdzw2 - cofwt * rdzwm) + cofwr * ((cofrz - cofrz_m));               // :571-573
  const D2 c = -1.0 * cofwz * coftz_p * rdzw2 * zz - cofwr * cofrz + cofwt * coftz_p * rdzw2;          // :575-576
  const D2 alpha = 1.0 / (b - a * gprev);                                                             // :583
  st2m(FLD(a_tri), ix, a, w0, w1); st2m(FLD(b_tri), ix, b, w0, w1); st2m(FLD(c_tri), ix, c, w0, w1);
  st2m(FLD(alpha_tri), ix, alpha, w0, w1);
  D2 gam = c * alpha;                                                                                 // :589
  if (k0 == 0) gam.x = 0.0;                                                                           // :545
  st2m(FLD(gamma_tri), ix, gam, m0, m1);
}

// ============================================================================================
// atm_compute_solve_diagnostics  :328-454
__global__ void k_diag_vertex(const View V) {      // vorticity :356-366, pv_vertex :443-445
  PAIR_THREAD(V.nVertices)
  if (!m0) return;
  const double* u = FLD(u);
  const int e0 = V.edgesOnVertex[x * 3], e1 = V.edgesOnVertex[x * 3 + 1], e2 = V.edgesOnVertex[x * 3 + 2];
  const D2 u0 = G2(u, e0), u1 = G2(u, e1), u2 = G2(u, e2);
  D2 vort = bc(0.0);
  vort += (V.edgesOnVertexSign[x * 3] * V.dcOnVertex[x * 3]) * u0;
  vort += (V.edgesOnVertexSign[x * 3 + 1] * V.dcOnVertex[x * 3 + 1]) * u1;
  vort += (V.edgesOnVertexSign[x * 3 + 2] * V.dcOnVertex[x * 3 + 2]) * u2;
  vort *= V.invAreaTriangle[x];
  st2m(FLD(vorticity), ix, vort, m0, m1);
  st2m(FLD(pv_vertex), ix, V.fVertex[x] + vort, m0, m1);
}
__global__ void k_diag_cell(const View V) {        // divergence :369-379 (s + u), ke :382-390
  PAIR_THREAD(V.nCells)
  XPF_CELL_ROWS();
  if (!m0) return;
  const int ME = V.maxEdges, n = V.nEdgesOnCell[x];
  const double* u = FLD(u);
  D2 div = bc(0.0), kec = bc(0.0);
  // slot 0's statics and column are requested together with the row length; dcEdge comes from the per-(cell, slot) copy
  const double r = V.invAreaCell[x];
  {
    const int e = V.edgesOnCell[x * V.MEP];
    const double dv = V.dvOnCell[x * ME], sg = V.edgesOnCellSign[x * ME], dc = V.dcOnCell[x * ME];
    const D2 ue = G2(u, e);
    if (n > 0) {
      const double s = sg * dv;
      div += s + ue;
      const double efac = dc * dv;
      kec += 0.25 * (efac * (ue * ue));
    }
  }
#pragma unroll 2
  for (int i = 1; i < n; ++i) {
    const int e = V.edgesOnCell[x * V.MEP + i];
    const double dv = V.dvOnCell[x * ME + i];
    const double s = V.edgesOnCellSign[x * ME + i] * dv;
    const D2 ue = G2(u, e);
    div += s + ue;
    const double efac = V.dcOnCell[x * ME + i] * dv;
    kec += 0.25 * (efac * (ue * ue));               // ke_edge recomputed from u: same value as the stored field
  }
  st2m(FLD(divergence), ix, div * r, m0, m1);
  st2m(FLD(ke), ix, kec * r, m0, m1);
}
template <bool RECON_V>
__global__ void k_diag_edge(const View V) {        // h_edge, ke_edge :346-353; v :431-438; pv_edge :449-451
  PAIR_THREAD(V.nEdges)
  XPF_EDGE_WORDS();
  if (!m0) return;
  const int4 cv = V.ecv[x];
  const double* u = FLD(u); const double* h = FLD(h); const double* pvv = FLD(pv_vertex);
  const D2 h1 = G2(h, cv.x), h2 = G2(h, cv.y), p1 = G2(pvv, cv.z), p2 = G2(pvv, cv.w);
  const D2 ue = ld2(u, ix);
  st2m(FLD(h_edge), ix, 0.5 * (h1 + h2), m0, m1);
  const double efac = V.dcEdge[x] * V.dvEdge[x];
  st2m(FLD(ke_edge), ix, efac * (ue * ue), m0, m1);
  if (RECON_V) {
    const int ME2 = V.maxEdges2, n = V.nEdgesOnEdge[x];
    D2 vv = bc(0.0);
#pragma unroll 2
    for (int i = 1; i < n; ++i) {                   // starts at 1 (Q7)
      const int eoe = V.edgesOnEdge_ECP[x * ME2 + i];
      vv += V.weightsOnEdge[x * ME2 + i] * G2(u, eoe);
    }
    st2m(FLD(v), ix, vv, m0, m1);
  }
  st2m(FLD(pv_edge), ix, 0.5 * (p1 + p2), m0, m1);
}
__global__ void k_diag_ke_vertex(const View V) {   // hollingsworth part 1 :395-400
  PAIR_THREAD(V.nVertices)
  if (!m0) return;
  const double* ke_edge = FLD(ke_edge);
  const double r = 0.25 * V.invAreaTriangle[x];
  st2m(FLD(ke_vertex), ix, (G2(ke_edge, V.edgesOnVertex[x * 3]) + G2(ke_edge, V.edgesOnVertex[x * 3 + 1])
                            + G2(ke_edge, V.edgesOnVertex[x * 3 + 2])) * r, m0, m1);
}
__global__ void k_diag_ke_holl(const View V) {     // hollingsworth part 2 :403-417
  PAIR_THREAD(V.nCells)
  if (!m0) return;
  const int ME = V.maxEdges, n = V.nEdgesOnCell[x];
  const double ke_fact = 1.0 - 0.375;
  const double* kev = FLD(ke_vertex);
  D2 kec = ld2(FLD(ke), ix) * ke_fact;
  const double r = V.invAreaCell[x];
  for (int i = 0; i < n; ++i) {
    const int iv = V.verticesOnCell[x * ME + i];
    const int j = V.kiteForCell[x * ME + i];
    kec += (1.0 - ke_fact) * V.kiteAreasOnVertex[iv * 3 + j] * G2(kev, iv) * r;
  }
  st2m(FLD(ke), ix, kec, m0, m1);
}

// ============================================================================================
// atm_compute_dyn_tend_work  :814-1480
// cell pre-pass: kdiff (:858-917), h_divergence (:924-938), tend_rho + dpdz (:942-951)
template <bool RK0>
__global__ void k_dt_cell0(const View V, const DynTendParams P, double len_disp, double cam_coef) {
  PAIR_THREAD(V.nCells)
  if (!m0) return;
  const int ME = V.maxEdges, n = V.nEdgesOnCell[x];
  const double* ru = FLD(ru);
  D2 hdiv = bc(0.0);
  const bool smag = RK0 && P.mixing == MPASB200_MIX_2D_SMAGORINSKY;
  if (smag) {
    const double* u = FLD(u); const double* v = FLD(v);
    D2 d_diag = bc(0.0), d_off = bc(0.0);
#pragma unroll 2
    for (int i = 0; i < n; ++i) {
      const int e = V.edgesOnCell[x * V.MEP + i];
      const double a = V.defc_a[x * ME + i], b = V.defc_b[x * ME + i];
      const D2 ue = G2(u, e), ve = G2(v, e), rue = G2(ru, e);
      d_diag += a * ue - b * ve;
      d_off += b * ue + a * ve;
      hdiv += (V.edgesOnCell_sign[x * ME + i] * V.dvOnCell[x * ME + i]) * rue;
    }
    const D2 mag = d_diag * d_diag + d_off * d_off;
    D2 kd = mk(dmin(P.kdiff_scale * sqrt(mag.x), P.kdiff_cap), dmin(P.kdiff_scale * sqrt(mag.y), P.kdiff_cap));   // :884-886
    if (P.cam_on) {                                                                                                // :911-914
      if (k0 >= L - 2) kd.x = dmax(kd.x, pow(2.0, (double)(k0 - (L - 2))) * 2.0833 * len_disp * cam_coef);
      if (k1 >= L - 2) kd.y = dmax(kd.y, pow(2.0, (double)(k1 - (L - 2))) * 2.0833 * len_disp * cam_coef);
    }
    st2m(FLD(kdiff), ix, kd, m0, m1);
  } else {
#pragma unroll 2
    for (int i = 0; i < n; ++i) {
      const int e = V.edgesOnCell[x * V.MEP + i];
      hdiv += (V.edgesOnCell_sign[x * ME + i] * V.dvOnCell[x * ME + i]) * G2(ru, e);
    }
    if (RK0 && (P.mixing == MPASB200_MIX_2D_FIXED || P.cam_on)) {
      D2 kd = (P.mixing == MPASB200_MIX_2D_FIXED) ? bc(0.0) : ld2(FLD(kdiff), ix);
      if (P.cam_on) {
        if (k0 >= L - 2) kd.x = dmax(kd.x, pow(2.0, (double)(k0 - (L - 2))) * 2.0833 * len_disp * cam_coef);
        if (k1 >= L - 2) kd.y = dmax(kd.y, pow(2.0, (double)(k1 - (L - 2))) * 2.0833 * len_disp * cam_coef);
      }
      st2m(FLD(kdiff), ix, kd, m0, m1);
    }
  }
  hdiv *= V.invAreaCell[x];
  st2m(FLD(h_divergence), ix, hdiv, m0, m1);
  if (RK0) {
    const double* rw = FLD(rw);
    const D2 rw2 = ld2(rw, ix), rwp = above(rw, ix, k0, L, rw2);
    const D2 qt = ld2(FLD(qtot), ix);
    st2m(FLD(tend_rho), ix, -hdiv - ld2(FLD(rdzw), k0) * (rwp - rw2 + ld2(FLD(tend_rho_physics), ix)), m0, m1);   // :947
    st2m(FLD(dpdz), ix, -P.gravity * (ld2(FLD(rho_base), ix) * (qt) + ld2(FLD(rho_p_save), ix) * (1.0 + qt)), m0, m1);   // :949
  }
}

// first del^2 of u  :1030-1043  (only delsq_u; the tend_u_euler contribution is added in k_dt_edge)
DI D2 u_diffusion2(const View& V, int x, int4 cv, int k0, int LP) {
  const double* dv = FLD(divergence); const double* vo = FLD(vorticity);
  const double r_dc = V.invDcEdge[x];
  const double r_dv = dmin(V.invDvEdge[x], 4 * r_dc);
  const D2 d2 = G2(dv, cv.y), d1 = G2(dv, cv.x), o2 = G2(vo, cv.w), o1 = G2(vo, cv.z);
  return (d2 - d1) * r_dc - (o2 - o1) * r_dv;                                                         // :1041-1042
}
__global__ void k_dt_edge_delsq(const View V) {
  PAIR_THREAD(V.nEdges)
  if (!m0) return;
  st2m(FLD(delsq_u), ix, 0.0 + u_diffusion2(V, x, V.ecv[x], k0, LP), m0, m1);
}
__global__ void k_dt_vertex_delsq(const View V) {   // delsq_vorticity :1052-1060
  PAIR_THREAD(V.nVertices)
  if (!m0) return;
  const double* dsu = FLD(delsq_u);
  const D2 a0 = G2(dsu, V.edgesOnVertex[x * 3]), a1 = G2(dsu, V.edgesOnVertex[x * 3 + 1]), a2 = G2(dsu, V.edgesOnVertex[x * 3 + 2]);
  const double iat = V.invAreaTriangle[x];
  D2 acc = bc(0.0);
  acc += (iat * V.dcOnVertex[x * 3] * V.edgesOnVertex_sign[x * 3]) * a0;
  acc += (iat * V.dcOnVertex[x * 3 + 1] * V.edgesOnVertex_sign[x * 3 + 1]) * a1;
  acc += (iat * V.dcOnVertex[x * 3 + 2] * V.edgesOnVertex_sign[x * 3 + 2]) * a2;
  st2m(FLD(delsq_vorticity), ix, acc, m0, m1);
}
__global__ void k_dt_cell_delsq(const View V) {     // delsq_divergence :1062-1070
  PAIR_THREAD(V.nCells)
  if (!m0) return;
  const int ME = V.maxEdges, n = V.nEdgesOnCell[x];
  const double* dsu = FLD(delsq_u);
  const double r = V.invAreaCell[x];
  D2 acc = bc(0.0);
#pragma unroll 2
  for (int i = 0; i < n; ++i) {
    const int e = V.edgesOnCell[x * V.MEP + i];
    const double edge_sign = r * V.dvOnCell[x * ME + i] * V.edgesOnCell_sign[x * ME + i];
    acc += edge_sign * G2(dsu, e);
  }
  st2m(FLD(delsq_divergence), ix, acc, m0, m1);
}

// vertical transport of u at one level  :973-980
DI double wduz_at(int k, int L, double rwavg, double fzm, double fzp, double um2, double um1, double u0, double up1) {
  double r = 0.0;
  if (k == 1 || k == L - 1) r = rwavg * (fzm * u0 + fzp * um1);
  if (k > 1 && k < L - 1) r = flux3(um2, um1, u0, up1, rwavg, 1.0);
  return r;
}
DI double vmix_u_at(double rho_e, double visc, double up, double uc, double um, double z1, double z2, double z3, double z4) {
  const double zm = 0.5 * (z1 + z2), z0 = 0.5 * (z2 + z3), zp = 0.5 * (z3 + z4);
  return rho_e * visc * ((up - uc) / (zp - z0) - (uc - um) / (z0 - zm)) / (0.5 * (zp - zm));
}

// tend_u_euler at rk_step == 0: pressure gradient (:964-970), 2nd-order Smagorinsky mixing (:1044-1047), the second del^2
// of the 4th-order filter (:1072-1090) and the optional vertical mixing (:1094-1146).  A lean gather kernel of its own:
// k_dt_edge then is the same kernel for every stage and just reads tend_u_euler.
__global__ void k_dt_edge_euler(const View V, const DynTendParams P) {
  extern __shared__ double sm[];
  PAIR_THREAD(V.nEdges)
  XPF_EDGE_WORDS();
  const int TS = LP + 2;
  double* s_um = sm + (size_t)threadIdx.y * TS;      // u_mix (vertical mixing of the perturbation from the initial state)
  const double* u = FLD(u);
  const bool vmix_pert = P.vmix_u_on && !P.mix_full;
  int4 cv = make_int4(0, 0, 0, 0);
  D2 rho_e = bc(0.0), tue = bc(0.0);
  if (m0) {
    cv = V.ecv[x];
    rho_e = ld2(FLD(rho_edge), ix);
    const double invDc = V.invDcEdge[x];
    const double* pp = FLD(pressure_p); const double* zz = FLD(zz); const double* dpdz = FLD(dpdz);
    tue = -ld2(FLD(cqu), ix) * ((G2(pp, cv.y) - G2(pp, cv.x)) * invDc / (0.5 * (G2(zz, cv.y) + G2(zz, cv.x)))
                                - 0.5 * ld2(FLD(zxu), ix) * (G2(dpdz, cv.x) + G2(dpdz, cv.y)));      // :967-969
    const double* kd = FLD(kdiff);
    const D2 u_diffusion = u_diffusion2(V, x, cv, k0, LP);
    const D2 kdiffu = 0.5 * (G2(kd, cv.x) + G2(kd, cv.y));
    tue += rho_e * kdiffu * u_diffusion * V.meshScalingDel2[x];                                     // :1046-1047
    if (P.visc4_on) {                                                                               // :1072-1090
      const double* dd = FLD(delsq_divergence); const double* dvo = FLD(delsq_vorticity);
      const double u_mix_scale = V.meshScalingDel4[x] * P.h_mom_eddy_visc4;
      const double r_dc4 = u_mix_scale * P.del4u_div_factor * invDc;
      const double r_dv4 = u_mix_scale * dmin(V.invDvEdge[x], 4 * invDc);
      const D2 ud4 = rho_e * ((G2(dd, cv.y) - G2(dd, cv.x)) * r_dc4 - (G2(dvo, cv.w) - G2(dvo, cv.z)) * r_dv4);
      tue -= ud4;
    }
    if (vmix_pert) {                                                                                // :1120-1123
      const D2 umix = ld2(u, ix) - ld2(FLD(u_init), k0) * V.cosAngleEdge[x] - ld2(FLD(v_init), k0) * V.sinAngleEdge[x];
      s_um[k0] = umix.x; if (m1) s_um[k1] = umix.y;
      st2m(FLD(u_mix), ix, umix, m0, m1);
    }
  }
  if (vmix_pert) __syncthreads();          // uniform: P is a kernel argument
  if (!m0) return;
  if (P.vmix_u_on) {                                                                                // :1094-1146
    const double* zg = FLD(zgrid);
    for (int c = 0; c < 2; ++c) {
      const int k = k0 + c;
      if (!(k > 0 && k < L - 1)) continue;
      const double z1 = 0.5 * (G1(zg, cv.x, k - 1) + G1(zg, cv.y, k - 1)), z2 = 0.5 * (G1(zg, cv.x, k) + G1(zg, cv.y, k));
      const double z3 = 0.5 * (G1(zg, cv.x, k + 1) + G1(zg, cv.y, k + 1)), z4 = 0.5 * (G1(zg, cv.x, k + 2) + G1(zg, cv.y, k + 2));
      double up, uc, um;
      if (P.mix_full) { up = G1(u, x, k + 1); uc = G1(u, x, k); um = G1(u, x, k - 1); }
      else { up = s_um[k + 1]; uc = s_um[k]; um = s_um[k - 1]; }
      const double add = vmix_u_at(c ? rho_e.y : rho_e.x, P.v_mom_eddy_visc2, up, uc, um, z1, z2, z3, z4);
      if (c) tue.y += add; else tue.x += add;
    }
  }
  st2m(FLD(tend_u_euler), ix, tue, m0, m1);
}

// u tendency  :958-1163 (tend_u_euler comes from k_dt_edge_euler at rk_step 0, from the previous stages otherwise)
#if KDE_MAXREG
#define KDE_REGCAP __maxnreg__(KDE_MAXREG)
#else
#define KDE_REGCAP
#endif
// read-once strips and outputs go through evict-first loads / stores (k_dt_edge 1.834 -> 1.816 ms per step on x1.163842)
#define KDE_LD ld2s
#define KDE_ST st2ms
__global__ void KDE_REGCAP k_dt_edge(const View V, const DynTendParams P) {
  extern __shared__ double sm[];
  PAIR_THREAD(V.nEdges)
  const int TS = LP + 2;
  double* s_wduz = sm + (size_t)threadIdx.y * TS;
  const double* u = FLD(u);
  int4 cv = make_int4(0, 0, 0, 0);
  D2 u2 = bc(0.0), wduz = bc(0.0);
  // requested first, consumed behind the barrier: level L of wduz (one lane; 6 % of the kernel's stall samples sat on this load in
  // front of the barrier) and the length of the edgesOnEdge row; the row itself and its weights are asked into L2
  double wduz_L = 0.0; int n_eoe = 0;
  if (inx && k0 == L) wduz_L = FLD(wduz)[ix];
  if (inx && k1 == L) wduz_L = FLD(wduz)[ix + 1];
  if (threadIdx.y == 0 && threadIdx.x < 3) {       // the 16-byte words / row lengths of the block about one wave later: one line each
    const long xa = (long)x + (long)PF_AHEAD * blockDim.y;
    if (xa < V.nEdges) {
      if (threadIdx.x == 0) prefetch_l2(V.ecv + xa);
      if (threadIdx.x == 1) prefetch_l2(V.nEdgesOnEdge + xa);
      if (threadIdx.x == 2) prefetch_l2(V.invDcEdge + xa);
    }
  }
  if (m0) {
    n_eoe = V.nEdgesOnEdge[x];
    if (threadIdx.x == 1) { prefetch_l2(V.edgesOnEdge + (size_t)x * V.maxEdges2); prefetch_l2(V.edgesOnEdge + (size_t)x * V.maxEdges2 + V.maxEdges2 - 1); }
    if (threadIdx.x == 2) { prefetch_l2(V.weightsOnEdge + (size_t)x * V.maxEdges2); prefetch_l2(V.weightsOnEdge + (size_t)x * V.maxEdges2 + V.maxEdges2 - 1); }
  }
  if (m0) {
    cv = V.ecv[x];
#if KDE_PREFETCH
    // the loads of the kernel's tail -- own-column strips and the cell columns that depend only on `cv` -- are
    // requested into L2 now, one request per 128-byte line, so that they later cost an L2 round trip instead of a DRAM one
    if ((threadIdx.x & 7) == 0) {
      prefetch_l2(FLD(rho_edge) + ix); prefetch_l2(FLD(tend_u_euler) + ix); prefetch_l2(FLD(tend_ru_physics) + ix); prefetch_l2(FLD(pv_edge) + ix);
      const size_t a = (size_t)cv.x * LP + k0, b = (size_t)cv.y * LP + k0;
      prefetch_l2(FLD(ke) + a); prefetch_l2(FLD(ke) + b); prefetch_l2(FLD(h_divergence) + a); prefetch_l2(FLD(h_divergence) + b);
      prefetch_l2(FLD(w) + a); prefetch_l2(FLD(w) + b);
    }
#endif
    u2 = ld2(u, ix);
    const double* rw = FLD(rw);
    const D2 rw_a = G2(rw, cv.x), rw_b = G2(rw, cv.y);
    const D2 rwavg = 0.5 * (rw_a + rw_b);
    const D2 fzm = ld2(FLD(fzm), k0), fzp = ld2(FLD(fzp), k0);
    const D2 um = (k0 >= 2) ? ld2(u, ix - 2) : bc(0.0);            // (u[k0-2], u[k0-1])
    const double up = (k0 + 2 <= L) ? u[ix + 2] : 0.0;             // u[k1+1]
    wduz.x = wduz_at(k0, L, rwavg.x, fzm.x, fzp.x, um.x, um.y, u2.x, u2.y);
    if (m1) wduz.y = wduz_at(k1, L, rwavg.y, fzm.y, fzp.y, um.y, u2.x, u2.y, up);
    s_wduz[k0] = wduz.x; if (m1) s_wduz[k1] = wduz.y;
    KDE_ST(FLD(wduz), ix, wduz, m0, m1);
  }
  if (inx && (k0 == L || k1 == L)) s_wduz[L] = wduz_L;    // level L: never written, read as stored
  __syncthreads();
  if (!m0) return;
  const D2 rho_e = KDE_LD(FLD(rho_edge), ix);
  const double invDc = V.invDcEdge[x];
  const D2 wduz_p = mk(s_wduz[k1], m1 ? s_wduz[k1 + 1] : 0.0);
  D2 tend_u = -ld2(FLD(rdzw), k0) * (wduz_p - wduz);                                                // :987
  // nonlinear Coriolis term :991-1001.  The reference adds each term nVertLevels times in a row
  // (Q14); here it is added once, multiplied by nVertLevels (same value to O(L) ulp, see DESIGN.md).
  D2 q = bc(0.0);
  {
    const int ME2 = V.maxEdges2, n = n_eoe;
    const double* pv = FLD(pv_edge);
    const D2 pv_k = ld2(pv, ix);
    const double Ld = (double)L;
    // (reading the static rows two slots at a time -- int2 ids, double2 weights -- was measured: 64 registers instead of 56,
    // 28 resident warps instead of 35, 2.94 -> 3.52 ms per launch on x1.655362; profiles/r2_ncu_gather_kernels.md)
#pragma unroll 2
    for (int j = 0; j < n; ++j) {
      const int eoe = V.edgesOnEdge[x * ME2 + j];
      const D2 workpv = 0.5 * (pv_k + G2(pv, eoe));
      q += Ld * (V.weightsOnEdge[x * ME2 + j] * G2(u, eoe) * workpv);
    }
  }
  KDE_ST(FLD(q), ix, q, m0, m1);
  const double* ke = FLD(ke); const double* hd = FLD(h_divergence); const double* w = FLD(w);
  tend_u += rho_e * (q - (G2(ke, cv.y) - G2(ke, cv.x)) * invDc) - u2 * 0.5 * (G2(hd, cv.x) + G2(hd, cv.y));   // :1005-1007
  {
    const D2 w1 = G2(w, cv.x), w2 = G2(w, cv.y);
    const D2 w1p = mk(w1.y, m1 ? G1(w, cv.x, k0 + 2) : 0.0), w2p = mk(w2.y, m1 ? G1(w, cv.y, k0 + 2) : 0.0);
    const D2 wsum = w1 + w1p + w2 + w2p;
    tend_u -= (P.omega2 * V.cosAngleEdge[x] * V.cosLatEdge[x] * rho_e * 0.25 * wsum)
              - (u2 * 0.25 * wsum * rho_e * P.inv_r_earth);                                        // :1011-1017
  }
  const D2 tue = KDE_LD(FLD(tend_u_euler), ix);
  if (P.rayleigh_u) {                                                                               // :1152-1159
    const int lim = L - P.rayleigh_levels + 1;
    if (k0 > lim) tend_u.x -= rho_e.x * u2.x * ((double)((double)k0 - (L - P.rayleigh_levels)) * P.rayleigh_coef_inverse);
    if (k1 > lim) tend_u.y -= rho_e.y * u2.y * ((double)((double)k1 - (L - P.rayleigh_levels)) * P.rayleigh_coef_inverse);
  }
  tend_u += tue + KDE_LD(FLD(tend_ru_physics), ix);                                                   // :1162
  KDE_ST(FLD(tend_u), ix, tend_u, m0, m1);
}

// horizontal advection + curvature part of the w tendency  :1170-1218  (value of cr.w before mixing);
// level 0 stays 0.  Also writes ru_edge_w for levels > 0.
DI D2 w_adv_curv(const View& V, const DynTendParams& P, int x, int k0, size_t ix, int LP, bool m0, bool m1) {
  const int ME = V.maxEdges, n = V.nEdgesOnCell[x];
  const D2 fm = ld2(FLD(fzm), k0), fp = ld2(FLD(fzp), k0);
  D2 wv = bc(0.0);
  if (n > 0) {
    // ru_edge_w / flux_arr are per-point fields overwritten for every edge (Q18): only the LAST
    // edge's values survive, and the second loop multiplies them by every edge's sign.
    const double* ru = FLD(ru);
    const int e = V.edgesOnCell[x * V.MEP + (n - 1)];
    const D2 ru2 = G2(ru, e);
    const D2 rew = fm * ru2 + fp * below(ru, (size_t)e * LP + k0, k0, ru2);
    D2 fa = bc(0.0);
    // every term is (coefficient) * 0.0: with finite coefficients (checked once at upload_mesh) the sum is +0.0 exactly and the
    // na coefficient loads -- 6 % of k_dt_cellC<false>'s stall samples -- are left out; a NaN / Inf coefficient takes the literal loop
    if (!V.advFinite) {
      const int na = V.nAdvOnCell[x * ME + (n - 1)];
      const size_t ab = ((size_t)x * ME + (n - 1)) * V.NAP;
      for (int j = 0; j < na; ++j) {
        const D2 sw = V.advCoefOnCell[ab + j] + sgn1(rew) * V.adv3OnCell[ab + j];
        fa += sw * 0.0;          // cr.w was zeroed on levels < L just before (:1170-1172); the pad cell is zero too
      }
    }
    st2m(FLD(ru_edge_w), ix, rew, m0 && k0 > 0, m1);
    for (int i = 0; i < n; ++i) wv -= V.edgesOnCell_sign[x * ME + i] * rew * fa;                    // :1202
  }
  const double* rz = FLD(rho_zz); const double* uz = FLD(uReconstructZonal); const double* um = FLD(uReconstructMeridional);
  const D2 rz2 = ld2(rz, ix), uz2 = ld2(uz, ix), um2 = ld2(um, ix);
  const D2 rzf = rz2 * fm + below(rz, ix, k0, rz2) * fp;
  const D2 uzf = fm * uz2 + fp * below(uz, ix, k0, uz2);
  const D2 umf = fm * um2 + fp * below(um, ix, k0, um2);
  wv += rzf * (uzf * uzf + umf * umf) / P.r_earth + P.omega2 * V.cosLatCell[x] * uzf * rzf;         // :1210-1216
  if (k0 == 0) wv.x = 0.0;
  return wv;
}

// rk_step == 0, cell pass A: w after advection+curvature (:1170-1218) and the first del^2 of theta (:1365-1382)
__global__ void k_dt_cellA(const View V, const DynTendParams P) {
  PAIR_THREAD(V.nCells)
  XPF_CELL_ROWS();
  if (!m0) return;
  st2m(FLD(w), ix, w_adv_curv(V, P, x, k0, ix, LP, m0, m1), m0, m1);
  const int ME = V.maxEdges, n = V.nEdgesOnCell[x];
  const double* tm = FLD(theta_m); const double* kd = FLD(kdiff); const double* re = FLD(rho_edge);
  const double r_areaCell = V.invAreaCell[x];
  D2 dsq = bc(0.0), tte = bc(0.0);
#pragma unroll 2
  for (int i = 0; i < n; ++i) {
    const int e = V.edgesOnCell[x * V.MEP + i];
    const int c1 = V.c1OnCell[x * V.MEP + i], c2 = V.c2OnCell[x * V.MEP + i];
    const double edge_sign = r_areaCell * V.edgesOnCell_sign[x * ME + i] * V.dvOnCell[x * ME + i] * V.invDcOnCell[x * ME + i];
    const double pr_scale = P.prandtl_inv * V.ms2OnCell[x * ME + i];
    D2 flux = edge_sign * (G2(tm, c2) - G2(tm, c1)) * G2(re, e);
    dsq += flux;
    flux *= 0.5 * (G2(kd, c1) + G2(kd, c2)) * pr_scale;
    tte += flux;
  }
  st2m(FLD(delsq_theta), ix, dsq, m0, m1);
  st2m(FLD(tend_theta_euler), ix, tte, m0, m1);
}
// rk_step == 0, cell pass B: first del^2 of w  :1231-1254  (needs pass A's w on neighbour cells)
__global__ void k_dt_cellB(const View V, const DynTendParams P) {
  PAIR_THREAD(V.nCells)
  XPF_CELL_ROWS();
  if (!m0) return;
  const int ME = V.maxEdges, n = V.nEdgesOnCell[x];
  const double* w = FLD(w); const double* kd = FLD(kdiff); const double* re = FLD(rho_edge);
  const double r_areaCell = V.invAreaCell[x];
  D2 dsq = bc(0.0), twe = bc(0.0);
#pragma unroll 2
  for (int i = 0; i < n; ++i) {
    const int e = V.edgesOnCell[x * V.MEP + i];
    const int c1 = V.c1OnCell[x * V.MEP + i], c2 = V.c2OnCell[x * V.MEP + i];
    const double edge_sign = 0.5 * r_areaCell * V.edgesOnCell_sign[x * ME + i] * V.dvOnCell[x * ME + i] * V.invDcOnCell[x * ME + i];
    const D2 re2 = G2(re, e), k1v = G2(kd, c1), k2v = G2(kd, c2);
    const D2 rem = below(re, (size_t)e * LP + k0, k0, re2);
    const D2 k1m = below(kd, (size_t)c1 * LP + k0, k0, k1v), k2m = below(kd, (size_t)c2 * LP + k0, k0, k2v);
    D2 flux = edge_sign * (re2 + rem) * (G2(w, c2) - G2(w, c1));
    dsq += flux;
    flux *= V.ms2OnCell[x * ME + i] * 0.25 * (k1v + k2v + k1m + k2m);
    twe += flux;
  }
  if (k0 == 0) { dsq.x = 0.0; twe.x = 0.0; }           // only k > 0 accumulates (:1244)
  st2m(FLD(delsq_w), ix, dsq, m0, m1);
  st2m(FLD(tend_w_euler), ix, twe, m0, m1);
}

// horizontal theta flux through each edge, evaluated ONCE per edge  (:1333-1340).  The reference evaluates
// flux_arr for edge e inside the loop of each of e's two cells; the value depends only on (e, level), so it is
// computed here per edge into library scratch and the cell pass sums it in slot order -- same bits, half the
// 2-ring gathers, and the gather lives in a kernel with a single level of index loads.
__global__ void k_dt_theta_flux(const View V) {
  PAIR_THREAD(V.nEdges)
  // the advection row of the column's edge -- ids and {adv_coefs, adv_coefs_3rd} pairs -- goes to shared memory, one entry per lane;
  // the stencil loop reads them with broadcast LDS
  extern __shared__ double sm[];
  const int NAE = V.NAE;
  double2* s_c = reinterpret_cast<double2*>(sm) + (size_t)threadIdx.y * NAE;
  int* s_i = reinterpret_cast<int*>(reinterpret_cast<double2*>(sm) + (size_t)blockDim.y * NAE) + (size_t)threadIdx.y * NAE;
  int na = 0; D2 ru2 = bc(0.0);
  if (inx) {
    na = V.nAdvCellsForEdge[x];
    for (int j = threadIdx.x; j < NAE; j += blockDim.x) { s_i[j] = V.advCellE[(size_t)x * NAE + j]; s_c[j] = V.advCoefE[(size_t)x * NAE + j]; }
  }
  if (m0) ru2 = ld2(FLD(ru), ix);
  __syncthreads();
  if (!m0) return;
  const double* tm = FLD(theta_m);
  const D2 sg = sgn1(ru2);
  D2 fa = bc(0.0);
#pragma unroll 2
  for (int j = 0; j < na; ++j) {
    const double2 c = s_c[j];
    const D2 sw = c.x + sg * c.y;
    fa += sw * G2(tm, s_i[j]);
  }
  st2m(V.scr_flux, ix, fa, m0, m1);
}

DI double wdwz_at(int k, int L, double rw_k, double rw_m, const double* s) {      // :1277-1287, s = w of the column in smem
  double r = 0.0;
  if (k == 1 || k == L - 1) r = 0.25 * (rw_k + rw_m) * (s[k] + s[k - 1]);
  if (k > 1 && k < L - 1) r = flux3(s[k - 2], s[k - 1], s[k], s[k + 1], 0.5 * (rw_k + rw_m), 1.0);
  return r;
}
DI double wdtz_at(int k, int L, double rws, double rw, double fzm, double fzp, double tms_k, double tms_m, double tm_k, double tm_m) {
  double r = 0.0;                                                                 // :1406-1420
  if (k > 0 && k < L - 1) r = ((rws - rw) * (fzm * tms_k + fzp * tms_m));
  if (k == 1) r += rw * (fzm * tm_k + fzp * tm_m);
  if (k == L - 1) r = rws * (fzm * tms_k + fzp * tms_m);
  return r;
}

// final cell pass: w (:1256-1322) and theta (:1328-1479)
// PART 0: both passes in one launch; 1: the w pass alone; 2: the theta pass alone.  The two passes share only `rw` (one unit re-read):
// launched separately each needs fewer registers and fewer barriers than the fused kernel (64 registers with 80-96 B of spills).
// read-once strips and outputs go through evict-first loads / stores (k_dt_cellC<false> 1.201 -> 1.179, <true> 0.591 -> 0.583)
#define CC_LD ld2s
#define CC_ST st2ms
template <bool RK0, int PART = 0>
__global__ void __launch_bounds__(256, PART == 0 ? LB_CELLC : LB_CELLC_SPLIT) k_dt_cellC(const View V, const DynTendParams P) {
  extern __shared__ double sm[];
  PAIR_THREAD(V.nCells)
  const int TS = LP + 2;
  double* s_a = sm + (size_t)threadIdx.y * TS;                       // w, later wdtz
  double* s_b = sm + (size_t)(blockDim.y + threadIdx.y) * TS;        // wdwz, later post-multiply w
  const int ME = V.maxEdges;
  const int n = inx ? V.nEdgesOnCell[x] : 0;
  // the static rows of the theta loops -- ids {e, c1, c2}, edgesOnCell_sign, dvOnCell -- go to shared memory at the top, one slot per
  // lane; the w pass's barriers make them visible and the loops read them with broadcast LDS (k_dt_cellC<false> 1.236 -> 1.205 ms per
  // step on x1.163842; the rk_step == 0 form got slower with it, 0.591 -> 0.637, and keeps its global rows)
  constexpr bool SROW = !RK0;
  double* s_sg = sm + (size_t)2 * blockDim.y * TS + (size_t)threadIdx.y * 2 * ME; double* s_dv = s_sg + ME;
  int* s_e = reinterpret_cast<int*>(sm + (size_t)2 * blockDim.y * (TS + ME)) + (size_t)threadIdx.y * 3 * ME;
  if (SROW) {
    if (inx && PART != 1)
      for (int i = threadIdx.x; i < ME; i += blockDim.x) {
        s_e[3 * i] = V.edgesOnCell[x * V.MEP + i]; s_e[3 * i + 1] = V.c1OnCell[x * V.MEP + i]; s_e[3 * i + 2] = V.c2OnCell[x * V.MEP + i];
        s_sg[i] = V.edgesOnCell_sign[x * ME + i]; s_dv[i] = V.dvOnCell[x * ME + i];
      }
    if (PART == 2) __syncthreads();
  }
  const double* rw = FLD(rw);
  D2 w2 = bc(0.0), twe = bc(0.0), fzm = bc(0.0), fzp = bc(0.0), rdzu = bc(0.0), rdzw = bc(0.0), rw2 = bc(0.0), rwm = bc(0.0);
  // level L of w / wdwz / wdtz (one lane per column) requested first, consumed in front of the barriers
  double wL = 0.0, wdwzL = 0.0, wdtzL = 0.0;
  if (inx && (k0 == L || k1 == L)) {
    const size_t iL = ix + (k0 == L ? 0 : 1);
    if (PART != 2) { wL = FLD(w)[iL]; wdwzL = FLD(wdwz)[iL]; }
    if (PART != 1) wdtzL = FLD(wdtz)[iL];
  }
  if (m0) {
#if CELLC_PREFETCH
    // own-column strips this kernel reads late (behind its barriers): requested into L2 now, one request per 128-byte line
    if ((threadIdx.x & 7) == 0) {
      if (PART != 1) {
        prefetch_l2(FLD(theta_m) + ix); prefetch_l2(FLD(theta_m_save) + ix); prefetch_l2(FLD(rw_save) + ix); prefetch_l2(FLD(rho_zz) + ix);
        prefetch_l2(FLD(rt_diabatic_tend) + ix); prefetch_l2(FLD(tend_theta_euler) + ix); prefetch_l2(FLD(tend_rtheta_physics) + ix);
      }
      if (PART != 2 && !RK0) prefetch_l2(FLD(tend_w_euler) + ix);
    }
#endif
    fzm = ld2(FLD(fzm), k0); fzp = ld2(FLD(fzp), k0); rdzu = ld2(FLD(rdzu), k0); rdzw = ld2(FLD(rdzw), k0);
    rw2 = ld2(rw, ix); rwm = below(rw, ix, k0, rw2);
    if (PART != 2) {
    if (RK0) {
      w2 = ld2(FLD(w), ix);
      twe = ld2(FLD(tend_w_euler), ix);
      if (P.visc4_on) {                                                                             // :1256-1272
        const double* dsw = FLD(delsq_w);
        const double r_areaCell = P.h_mom_eddy_visc4 * V.invAreaCell[x];
        D2 acc = twe;
#pragma unroll 2
        for (int i = 0; i < n; ++i) {
          const int c1 = V.c1OnCell[x * V.MEP + i], c2 = V.c2OnCell[x * V.MEP + i];
          const double edge_sign = V.ms4OnCell[x * ME + i] * r_areaCell * V.dvOnCell[x * ME + i] * V.edgesOnCell_sign[x * ME + i] * V.invDcOnCell[x * ME + i];
          acc -= edge_sign * (G2(dsw, c2) - G2(dsw, c1));
        }
        twe = mk(k0 > 0 ? acc.x : twe.x, acc.y);
      }
    } else {
      w2 = w_adv_curv(V, P, x, k0, ix, LP, m0, m1);
    }
    s_a[k0] = w2.x; if (m1) s_a[k1] = w2.y;
    }
  }
  if (PART != 2) {
  if (inx && (k0 == L || k1 == L)) { s_a[L] = wL; s_b[L] = wdwzL; }             // level L keeps its stored value
  __syncthreads();
  D2 wdwz = bc(0.0);
  if (m0) {
    wdwz.x = wdwz_at(k0, L, rw2.x, rwm.x, s_a);
    if (m1) wdwz.y = wdwz_at(k1, L, rw2.y, rwm.y, s_a);
    s_b[k0] = wdwz.x; if (m1) s_b[k1] = wdwz.y;
    CC_ST(FLD(wdwz), ix, wdwz, m0, m1);
  }
  __syncthreads();
  D2 wdwz_p = bc(0.0);
  if (m0) wdwz_p = mk(s_b[k1], m1 ? s_b[k1 + 1] : 0.0);
  __syncthreads();
  if (m0) {
    const D2 wmul = w2 * (V.invAreaCell[x] - rdzu * (wdwz_p - wdwz));                                // :1292
    w2 = mk(k0 > 0 ? wmul.x : w2.x, wmul.y);
    if (RK0) {                                                                                       // :1297-1299
      const double* pp = FLD(pressure_p); const double* dpdz = FLD(dpdz);
      const D2 pp2 = ld2(pp, ix), dp2 = ld2(dpdz, ix);
      const D2 t = twe - ld2(FLD(cqw), ix) * (rdzu * (pp2 - below(pp, ix, k0, pp2)) - (fzm * dp2 + fzp * below(dpdz, ix, k0, dp2)));
      twe = mk(k0 > 0 ? t.x : twe.x, t.y);
    }
    s_b[k0] = w2.x; if (m1) s_b[k1] = w2.y;                         // post-multiply w, for the vertical mixing of w
  }
  if (inx && (k0 == L || k1 == L)) s_b[L] = s_a[L];
  __syncthreads();
  if (m0) {
    if (RK0 && P.vmix_u_on) {                                                                        // :1304-1314
      const double* rz = FLD(rho_zz);
      const double* rdzw_ = FLD(rdzw);
      for (int c = 0; c < 2; ++c) {
        const int k = k0 + c;
        if (k == 0 || k >= L) continue;
        const double add = P.v_mom_eddy_visc2 * (rz[ix + c] + rz[ix + c - 1]) * 0.5
                           * ((s_b[k + 1] - s_b[k]) * rdzw_[k] - (s_b[k] - s_b[k - 1]) * rdzw_[k - 1]) * (c ? rdzu.y : rdzu.x);
        if (c) twe.y += add; else twe.x += add;
      }
    }
    if (!RK0) { const D2 t = ld2(FLD(tend_w_euler), ix); twe = mk(k0 > 0 ? t.x : 0.0, t.y); }
    if (RK0) CC_ST(FLD(tend_w_euler), ix, twe, m0, m1);
    w2 = mk(k0 > 0 ? w2.x + twe.x : w2.x, w2.y + twe.y);                                            // :1320
    CC_ST(FLD(w), ix, w2, m0, m1);
  }
  }
  if (PART == 1) return;
  // ---------------- theta ----------------
  const double* tm = FLD(theta_m); const double* tms = FLD(theta_m_save);
  D2 tt = bc(0.0), wdtz = bc(0.0);
  if (m0) {
    const double* ru = FLD(ru);
    D2 fa_last = bc(0.0);
#pragma unroll 2
    for (int i = 0; i < n; ++i) {                                                                     // :1328-1344
      const int e = SROW ? s_e[3 * i] : V.edgesOnCell[x * V.MEP + i];
      const double sg_i = SROW ? s_sg[i] : V.edgesOnCell_sign[x * ME + i];
      const D2 ru_e = G2(ru, e);
      const D2 fa = G2(V.scr_flux, e);              // flux_arr of this edge (k_dt_theta_flux)
      tt -= sg_i * ru_e * fa;
      fa_last = fa;
    }
    if (n > 0) CC_ST(FLD(flux_arr), ix, fa_last, m0, m1);
    if (P.rk_step > 0) {                                                                              // :1347-1360
      const double* rus = FLD(ru_save);
#pragma unroll 2
      for (int i = 0; i < n; ++i) {
        const int e = SROW ? s_e[3 * i] : V.edgesOnCell[x * V.MEP + i];
        const int c1 = SROW ? s_e[3 * i + 1] : V.c1OnCell[x * V.MEP + i], c2 = SROW ? s_e[3 * i + 2] : V.c2OnCell[x * V.MEP + i];
        const double sd_i = SROW ? s_sg[i] * s_dv[i] : V.edgesOnCell_sign[x * ME + i] * V.dvOnCell[x * ME + i];
        const D2 flux = sd_i * (G2(rus, e) - G2(ru, e)) * 0.5 * (G2(tms, c2) + G2(tms, c1));
        tt -= flux;
      }
    }
    const D2 tm2 = ld2(tm, ix), tms2 = ld2(tms, ix), rws2 = CC_LD(FLD(rw_save), ix);
    const D2 tmm = below(tm, ix, k0, tm2), tmsm = below(tms, ix, k0, tms2);
    wdtz.x = wdtz_at(k0, L, rws2.x, rw2.x, fzm.x, fzp.x, tms2.x, tmsm.x, tm2.x, tmm.x);
    if (m1) wdtz.y = wdtz_at(k1, L, rws2.y, rw2.y, fzm.y, fzp.y, tms2.y, tmsm.y, tm2.y, tmm.y);
    s_a[k0] = wdtz.x; if (m1) s_a[k1] = wdtz.y;
    CC_ST(FLD(wdtz), ix, wdtz, m0, m1);
  }
  if (inx && (k0 == L || k1 == L)) s_a[L] = wdtzL;
  __syncthreads();
  if (!m0) return;
  const D2 rz = ld2(FLD(rho_zz), ix);
  const D2 wdtz_p = mk(s_a[k1], m1 ? s_a[k1 + 1] : 0.0);
  tt *= V.invAreaCell[x] - rdzw * (wdtz_p - wdtz);                                                   // :1423
  CC_ST(FLD(tend_rtheta_adv), ix, tt, m0, m1);
  CC_ST(FLD(rthdynten), ix, tt / rz, m0, m1);
  tt += rz * CC_LD(FLD(rt_diabatic_tend), ix);
  D2 tte = ld2(FLD(tend_theta_euler), ix);
  if (RK0) {
    if (P.visc4_on) {                                                                                 // :1384-1399
      const double* dst = FLD(delsq_theta);
      const double r_areaCell = P.h_theta_eddy_visc4 * P.prandtl_inv * V.invAreaCell[x];
#pragma unroll 2
      for (int i = 0; i < n; ++i) {
        const int c1 = V.c1OnCell[x * V.MEP + i], c2 = V.c2OnCell[x * V.MEP + i];
        const double edge_sign = V.ms4OnCell[x * ME + i] * r_areaCell * V.dvOnCell[x * ME + i] * V.edgesOnCell_sign[x * ME + i] * V.invDcOnCell[x * ME + i];
        tte -= edge_sign * (G2(dst, c2) - G2(dst, c1));
      }
    }
    if (P.vmix_t_on) {                                                                                // :1432-1473
      const double* zg = FLD(zgrid); const double* ti = FLD(t_init);
      for (int c = 0; c < 2; ++c) {
        const int k = k0 + c;
        if (!(k > 0 && k < L - 1)) continue;
        const size_t i_ = ix + c;
        const double z1 = zg[i_ - 1], z2 = zg[i_], z3 = zg[i_ + 1], z4 = zg[i_ + 2];
        const double zm = 0.5 * (z1 + z2), z0 = 0.5 * (z2 + z3), zp = 0.5 * (z3 + z4);
        const double rzc = c ? rz.y : rz.x;
        double add;
        if (P.mix_full)
          add = P.v_theta_eddy_visc2 * P.prandtl_inv * rzc * ((tm[i_ + 1] - tm[i_]) / (zp - z0) - (tm[i_] - tm[i_ - 1]) / (z0 - zm)) / (0.5 * (zp - zm));
        else
          add = P.v_theta_eddy_visc2 * P.prandtl_inv * rzc
                * (((tm[i_ + 1] - ti[i_ + 1]) - (tm[i_] - ti[i_])) / (zp - z0) - ((tm[i_] - ti[i_]) - (tm[i_ - 1] - ti[i_ - 1])) / (z0 - zm)) / (0.5 * (zp - zm));
        if (c) tte.y += add; else tte.x += add;
      }
    }
    CC_ST(FLD(tend_theta_euler), ix, tte, m0, m1);
  }
  tt += tte + CC_LD(FLD(tend_rtheta_physics), ix);                                                      // :1478
  CC_ST(FLD(tend_theta), ix, tt, m0, m1);
}

// ============================================================================================
// atm_set_smlstep_pert_variables_work  :1503-1528.  `for iCell in cpr` (:1516) visits EVERY point of the region, so the
// levels are 0..L inclusive (regions hold L+1 levels, main.rg:21-24); level -1 reads 0 (M3), level L uses whatever the
// mirror holds there for fzm/fzp/zz/zb_cell/u_tend (zero until uploaded, M1).
__global__ void k_smlstep(const View V, int nRelaxZone) {
  PAIR_THREAD(V.nCells)
  const bool a0 = inx && k0 <= L, a1 = inx && k1 <= L;        // level L included
  (void)m0;
  if (!a0) return;
  // the two masks and the row length are requested together (they were three dependent round trips: || and the early return)
  const unsigned char in_cpr = V.inCpr[x]; const int bdy = V.bdyMaskCell[x];
  const int ME = V.maxEdges, n = V.nEdgesOnCell[x];
  if (!in_cpr || bdy > nRelaxZone) return;
  const double* ut = FLD(u_tend); const double* zb = FLD(zb_cell); const double* zb3 = FLD(zb3_cell);
  const D2 fm = ld2(FLD(fzm), k0), fp = ld2(FLD(fzp), k0);
  D2 wv = ld2(FLD(w), ix);
#pragma unroll 2
  for (int i = 0; i < n; ++i) {
    const int e = V.edgesOnCell[x * V.MEP + i];
    const D2 ut_k = G2(ut, e);
    const D2 ut_m = below(ut, (size_t)e * LP + k0, k0, ut_k);
    const D2 flux = V.edgesOnCell_sign[x * ME + i] * (fm * ut_k + fp * ut_m);
    wv -= (ld2(zb, i * V.cellSlot + ix) + sgn1(ut_k) * ld2(zb3, i * V.cellSlot + ix)) * flux;
  }
  const D2 zz2 = ld2(FLD(zz), ix);
  wv *= (fm * zz2 + fp * below(FLD(zz), ix, k0, zz2));
  st2m(FLD(w), ix, wv, a0, a1);
}

// ============================================================================================
// atm_advance_acoustic_step_work  :1546-1705
// Fused single-kernel form of the acoustic step (default).  A block owns whole columns.
// Everything except the dependence of rw_p(k) on the freshly updated level k-1 is evaluated in
// parallel exactly as written in the reference.  That dependence is affine: with x = rw_p_new,
//     rho_pp_new(k-1)    = rp0 + rp1 * x(k-1)          (:1694)
//     rtheta_pp_new(k-1) = rt0 + rt1 * x(k-1)          (:1695-1696)
//     x(k) = P(k) + Q(k) * x(k-1)                      (:1662-1686 collected in x(k-1))
// so every thread computes its (P, Q) and ONE thread per column runs the 1-multiply-add-per-level
// sweep out of shared memory; rho_pp / rtheta_pp / wwAvg then follow in parallel from x with the
// reference's own expressions.  rs[k-1] and ts[k-1] are always 0 (the reference re-zeroes both arrays
// at every point, Q25); the back-substitution is absent (Q28); cr.theta_m stands in for tend_rt and
// cr.w for tend_rw (Q27).  Differs from the literal left-to-right evaluation only by the regrouping
// of terms inside one level (a few ulp; checked against the oracle at 1e-12).
// Per-level pieces of the affine form.  Everything is local to the level except (rp0m, rt0m), the
// constant parts of level k-1's new rho_pp / rtheta_pp.
struct AcTerms { double A0, A1, A2, al, r1, r2, r3, Q; };
DI AcTerms ac_terms(double dts, double resm, double rw_old_k, double w_k, double ts, double rs, double rt_old, double rho_old,
                    double zz_k, double zz_m, double cofwt_k, double cofwt_m, double rz_k, double rz_m, double cofwz_k, double cofwr_k,
                    double fm, double fp, double dsk, double rws_k, double rw_k, double rp1m, double rt1m, double a_k, double al_k) {
  AcTerms o;
  o.r3 = rws_k - rw_k;
  o.r1 = o.r3 - dts * dsk * (fm * zz_k + fp * zz_m) * (fm * rz_k + fp * rz_m) * w_k;                 // :1682-1684
  o.r2 = 1.0 + dts * dsk;                                                                           // :1685
  // terms of :1662-1667 that do not involve level k-1's new values
  o.A0 = rw_old_k + (dts * w_k - cofwz_k * ((zz_k * ts - zz_m * 0.0) + resm * (zz_k * rt_old))
                     - cofwr_k * ((rs + 0.0) + resm * rho_old) + cofwt_k * (ts + resm * rt_old));
  o.A1 = resm * (cofwz_k * zz_m + cofwt_m);        // coefficient of rtheta_pp_new(k-1)
  o.A2 = resm * cofwr_k;                           // coefficient of -rho_pp_new(k-1)
  o.al = al_k;                                                                                      // :1671
  o.Q = (o.A1 * rt1m - o.A2 * rp1m - a_k) * al_k / o.r2;                                            // :1670
  return o;
}
DI double ac_P(const AcTerms& t, double rp0m, double rt0m) {
  return ((t.A0 + t.A1 * rt0m - t.A2 * rp0m) * t.al + t.r1) / t.r2 - t.r3;                          // :1682-1686
}
template <bool S0>
__global__ void __launch_bounds__(256, S0 ? LB_AC + 1 : LB_AC) k_acoustic(const View V, double dts, double epssm, double resm) {
  extern __shared__ double sm[];
  PAIR_THREAD_R()
  const int TS = LP + 2;
  double* s_rp0 = sm + (size_t)threadIdx.y * TS;
  double* s_rt0 = sm + (size_t)(blockDim.y + threadIdx.y) * TS;
  double* s_P = sm + (size_t)(2 * blockDim.y + threadIdx.y) * TS;
  double* s_Q = sm + (size_t)(3 * blockDim.y + threadIdx.y) * TS;
  const bool spec = inx ? (V.specZoneMaskCell[x] != 0.0) : false;
  if (S0 && inx) {                                                                                    // :1625-1630, level L
    if (k0 == L) { FLD(wwAvg)[ix] = 0; FLD(rw_p)[ix] = 0; }
    if (k1 == L) { FLD(wwAvg)[ix + 1] = 0; FLD(rw_p)[ix + 1] = 0; }
  }
  D2 rs = bc(0), ts = bc(0), rw_old = bc(0);
  double rw_oldp_y = 0.0;
  AcTerms t0;                      // level k0's terms wait for level k0-1 (another thread) behind the barrier
  t0.A0 = t0.A1 = t0.A2 = t0.al = t0.r1 = t0.r3 = t0.Q = 0.0; t0.r2 = 1.0;
  if (m0) {
    const double* tm = FLD(theta_m);
    const D2 cofrz = ld2(FLD(cofrz), k0), rdzw = ld2(FLD(rdzw), k0);
    D2 rho_old = bc(0), rt_old = bc(0), rw_oldp = bc(0);
    if (!S0) {
      rw_old = ld2(FLD(rw_p), ix); rw_oldp = above(FLD(rw_p), ix, k0, L, rw_old);
      rho_old = ld2(FLD(rho_pp), ix); rt_old = ld2(FLD(rtheta_pp), ix);
    }
    rw_oldp_y = rw_oldp.y;
    st2m(FLD(rtheta_pp_old), ix, S0 ? bc(0.0) : rt_old, m0, m1);                                      // :1615-1623
    if (!spec) {
      const D2 w2 = ld2(FLD(w), ix), tr = ld2(FLD(tend_rho), ix), tm2 = ld2(tm, ix);
      const int ME = V.maxEdges, n = V.nEdgesOnCell[x];
      const double* ru_p = FLD(ru_p);
      const double inva = V.invAreaCell[x];
#pragma unroll 2
      for (int i = 0; i < n; ++i) {                                                                   // :1644-1652
        const int e = V.edgesOnCell[x * V.MEP + i];
        const int c1 = V.c1OnCell[x * V.MEP + i], c2 = V.c2OnCell[x * V.MEP + i];
        const D2 flux = V.edgesOnCellSign[x * ME + i] * dts * V.dvOnCell[x * ME + i] * G2(ru_p, e) * inva;
        rs -= flux;
        ts -= flux * 0.5 * (G2(tm, c2) + G2(tm, c1));
      }
      const D2 coftz = ld2(FLD(coftz), ix), coftz_p = above(FLD(coftz), ix, k0, L, coftz);
      rs = rho_old + dts * tr + rs - cofrz * resm * (rw_oldp - rw_old);                               // :1657
      ts = rt_old + dts * tm2 + ts - resm * rdzw * (coftz_p * rw_oldp - coftz * rw_old);              // :1658
      // new rho_pp / rtheta_pp of a level as affine functions of x(k):  rp0 + cofrz*x,  rt0 + rdzw*coftz*x
      const D2 rp0 = rs - cofrz * rw_oldp, rt0 = ts - rdzw * (coftz_p * rw_oldp);
      const D2 zz = ld2(FLD(zz), ix), zzm = below(FLD(zz), ix, k0, zz);
      const D2 cwt = ld2(FLD(cofwt), ix), cwtm = below(FLD(cofwt), ix, k0, cwt);
      const D2 rz = ld2(FLD(rho_zz), ix), rzm = below(FLD(rho_zz), ix, k0, rz);
      const D2 cwz = ld2(FLD(cofwz), ix), cwr = ld2(FLD(cofwr), ix);
      const D2 fm = ld2(FLD(fzm), k0), fp = ld2(FLD(fzp), k0);
      const D2 ds = ld2(FLD(dss), ix), rws = ld2(FLD(rw_save), ix), rwv = ld2(FLD(rw), ix);
      const D2 at = ld2(FLD(a_tri), ix), al = ld2(FLD(alpha_tri), ix);
      if (k0 > 0) {
        const double cofrz_m = FLD(cofrz)[k0 - 1], rdzw_m = FLD(rdzw)[k0 - 1], coftz_m = FLD(coftz)[ix - 1];
        t0 = ac_terms(dts, resm, rw_old.x, w2.x, ts.x, rs.x, rt_old.x, rho_old.x, zz.x, zzm.x, cwt.x, cwtm.x, rz.x, rzm.x, cwz.x, cwr.x,
                      fm.x, fp.x, ds.x, rws.x, rwv.x, cofrz_m, rdzw_m * coftz_m, at.x, al.x);
        s_Q[k0] = t0.Q;
      } else { s_P[0] = rw_old.x; s_Q[0] = 0.0; }
      if (m1) {                     // level k1's partner is this thread's own level k0
        const AcTerms t1 = ac_terms(dts, resm, rw_old.y, w2.y, ts.y, rs.y, rt_old.y, rho_old.y, zz.y, zzm.y, cwt.y, cwtm.y, rz.y, rzm.y,
                                    cwz.y, cwr.y, fm.y, fp.y, ds.y, rws.y, rwv.y, cofrz.x, rdzw.x * coftz.x, at.y, al.y);
        s_P[k1] = ac_P(t1, rp0.x, rt0.x); s_Q[k1] = t1.Q;
        s_rp0[k1] = rp0.y; s_rt0[k1] = rt0.y;
      }
    }
  }
  __syncthreads();
  if (m0 && !spec && k0 > 0) s_P[k0] = ac_P(t0, s_rp0[k0 - 1], s_rt0[k0 - 1]);
  __syncthreads();
  if (inx && !spec && k0 == 0) {            // the sweep: one fused multiply-add per level, levels ascending (M4)
    double xv = s_P[0];
#pragma unroll 4
    for (int kk = 1; kk < L; ++kk) { xv = __fma_rn(s_Q[kk], xv, s_P[kk]); s_P[kk] = xv; }
  }
  __syncthreads();
  if (!m0) return;
  const D2 ww_old = S0 ? bc(0.0) : ld2(FLD(wwAvg), ix);
  D2 rw_new, rho_new, rt_new, ww_new;
  if (!spec) {
    const D2 cofrz = ld2(FLD(cofrz), k0), rdzw = ld2(FLD(rdzw), k0);
    const D2 coftz = ld2(FLD(coftz), ix), coftz_p = above(FLD(coftz), ix, k0, L, coftz);
    const D2 rw_oldp = mk(rw_old.y, rw_oldp_y);
    rw_new = mk(s_P[k0], m1 ? s_P[k1] : 0.0);
    const D2 wa = ww_old + 0.5 * (1.0 - epssm) * rw_old;                                              // :1661
    const D2 wb = wa + 0.5 * (1.0 + epssm) * rw_new;                                                  // :1689
    ww_new = mk(k0 > 0 ? wb.x : ww_old.x, wb.y);
    rho_new = rs - cofrz * (rw_oldp - rw_new);                                                        // :1694
    rt_new = ts - rdzw * (coftz_p * rw_oldp - coftz * rw_new);                                        // :1695-1696
  } else {                                                                                            // :1698-1703
    const D2 rho_old = S0 ? bc(0.0) : ld2(FLD(rho_pp), ix), rt_old = S0 ? bc(0.0) : ld2(FLD(rtheta_pp), ix);
    rho_new = rho_old + dts * ld2(FLD(tend_rho), ix);
    rt_new = rt_old + dts * ld2(FLD(theta_m), ix);
    rw_new = rw_old + dts * ld2(FLD(w), ix);
    ww_new = ww_old + 0.5 * (1.0 + epssm) * rw_new;
  }
  st2m(FLD(rho_pp), ix, rho_new, m0, m1); st2m(FLD(rtheta_pp), ix, rt_new, m0, m1);
  const bool wr0 = S0 || spec || k0 > 0;
  st2m(FLD(rw_p), ix, rw_new, wr0, m1); st2m(FLD(wwAvg), ix, ww_new, wr0, m1);
}

// Split form of the acoustic step, phase 1 (lean, register-light): the edgesOnCell gathers only  (:1644-1652).
// rs_h / ts_h go to library scratch and are streamed by phase 2 as two more strips.
__global__ void k_acoustic_gather(const View V, double dts) {
  PAIR_THREAD_R()
  XPF_CELL_ROWS();                                  // rows of 8 cells span 2 lines
  if (!m0) return;
  if (V.specZoneMaskCell[x] != 0.0) return;
  const int ME = V.maxEdges, n = V.nEdgesOnCell[x];
  const double inva = V.invAreaCell[x];
  const double* ru_p = FLD(ru_p); const double* tm = FLD(theta_m);
  D2 rs = bc(0), ts = bc(0);
#pragma unroll 2
  for (int i = 0; i < n; ++i) {
    const int e = V.edgesOnCell[x * V.MEP + i];
    const int c1 = V.c1OnCell[x * V.MEP + i], c2 = V.c2OnCell[x * V.MEP + i];
    const D2 flux = V.edgesOnCellSign[x * ME + i] * dts * V.dvOnCell[x * ME + i] * G2(ru_p, e) * inva;
    rs -= flux;
    ts -= flux * 0.5 * (G2(tm, c2) + G2(tm, c1));
  }
  st2m(V.scr_rs, ix, rs, m0, m1); st2m(V.scr_ts, ix, ts, m0, m1);
}

// ---- MPASB200_PHYSICS_CORRECTED (mpas_b200.h): the acoustic step with its three disabled pieces enabled ------------
// Edge update :1581-1613, exactly the commented lines; every edge (the nCellsSolve test stays out).
template <bool S0>
__global__ void k_acoustic_u(const View V, double dts, double c2, double gravity) {
  PAIR_THREAD_R()
  if (!m0) return;
  const D2 tru = ld2(FLD(tend_ru), ix);
  if (S0) {                                                                                           // :1601-1613
    const D2 r = dts * tru;
    st2m(FLD(ru_p), ix, r, m0, m1); st2m(FLD(ruAvg), ix, r, m0, m1);
    return;
  }
  const int4 cv = V.ecv[x];
  const double* rpp = FLD(rtheta_pp); const double* zz = FLD(zz); const double* ex = FLD(exner); const double* rho = FLD(rho_pp);
  D2 pgrad = ((G2(rpp, cv.y) - G2(rpp, cv.x)) * V.invDcEdge[x]) / (0.5 * (G2(zz, cv.y) + G2(zz, cv.x)));      // :1591
  pgrad = pgrad * (ld2(FLD(cqu), ix) * 0.5 * c2 * (G2(ex, cv.x) + G2(ex, cv.y)));                          // :1592
  pgrad = pgrad + 0.5 * ld2(FLD(zxu), ix) * gravity * (G2(rho, cv.x) + G2(rho, cv.y));                     // :1593
  const D2 r = ld2(FLD(ru_p), ix) + dts * (tru - (1.0 - V.specZoneMaskEdge[x]) * pgrad);                   // :1594
  st2m(FLD(ru_p), ix, r, m0, m1);
  st2m(FLD(ruAvg), ix, ld2(FLD(ruAvg), ix) + r, m0, m1);                                                   // :1597
}

// Cell part :1615-1704, column by column as in MPAS: rs/ts for the whole column, right-hand side, forward elimination
// (:1670-1671), back-substitution (:1674-1677), Rayleigh damping (:1681-1690), rho_pp / rtheta_pp (:1694-1696).
// The horizontal flux sums come from k_acoustic_gather (scratch).  One thread per level pair; the two sweeps are run
// strictly in order by one thread per column out of shared memory, so the result is bit-identical to the oracle.
template <bool S0>
__global__ void __launch_bounds__(256) k_acoustic_col(const View V, double dts, double epssm, double resm) {
  extern __shared__ double sm[];
  PAIR_THREAD_R()
  const int TS = LP + 2, CB = blockDim.y, ty = threadIdx.y;
  double* s_rs = sm + (size_t)(0 * CB + ty) * TS;
  double* s_ts = sm + (size_t)(1 * CB + ty) * TS;
  double* s_x = sm + (size_t)(2 * CB + ty) * TS;
  double* s_a = sm + (size_t)(3 * CB + ty) * TS;
  double* s_al = sm + (size_t)(4 * CB + ty) * TS;
  double* s_g = sm + (size_t)(5 * CB + ty) * TS;
  const bool spec = inx ? (V.specZoneMaskCell[x] != 0.0) : false;
  const bool act = m0 && !spec;
  if (S0 && inx) {                                                                                    // :1625-1630, level L
    if (k0 == L) { FLD(wwAvg)[ix] = 0; FLD(rw_p)[ix] = 0; }
    if (k1 == L) { FLD(wwAvg)[ix + 1] = 0; FLD(rw_p)[ix + 1] = 0; }
  }
  D2 rs = bc(0), ts = bc(0), rw_old = bc(0), rw_oldp = bc(0), rho_old = bc(0), rt_old = bc(0);
  D2 zz = bc(0), zzm = bc(0), w2 = bc(0);
  if (m0) {
    if (!S0) {
      rw_old = ld2(FLD(rw_p), ix); rw_oldp = above(FLD(rw_p), ix, k0, L, rw_old);
      rho_old = ld2(FLD(rho_pp), ix); rt_old = ld2(FLD(rtheta_pp), ix);
    }
    st2m(FLD(rtheta_pp_old), ix, S0 ? bc(0.0) : rt_old, m0, m1);                                      // :1615-1623
  }
  if (act) {
    const D2 cofrz = ld2(FLD(cofrz), k0), rdzw = ld2(FLD(rdzw), k0);
    const D2 coftz = ld2(FLD(coftz), ix), coftz_p = above(FLD(coftz), ix, k0, L, coftz);
    rs = rho_old + dts * ld2(FLD(tend_rho), ix) + ld2(V.scr_rs, ix) - cofrz * resm * (rw_oldp - rw_old);                // :1657
    ts = rt_old + dts * ld2(FLD(theta_m), ix) + ld2(V.scr_ts, ix) - resm * rdzw * (coftz_p * rw_oldp - coftz * rw_old);   // :1658
    s_rs[k0] = rs.x; s_ts[k0] = ts.x;
    if (m1) { s_rs[k1] = rs.y; s_ts[k1] = ts.y; }
  }
  __syncthreads();
  if (act) {
    zz = ld2(FLD(zz), ix); zzm = below(FLD(zz), ix, k0, zz); w2 = ld2(FLD(w), ix);
    const D2 rsm = mk(k0 > 0 ? s_rs[k0 - 1] : 0.0, rs.x), tsm = mk(k0 > 0 ? s_ts[k0 - 1] : 0.0, ts.x);
    const D2 rtm = S0 ? bc(0.0) : below(FLD(rtheta_pp), ix, k0, rt_old), rhm = S0 ? bc(0.0) : below(FLD(rho_pp), ix, k0, rho_old);
    const D2 cwt = ld2(FLD(cofwt), ix), cwtm = below(FLD(cofwt), ix, k0, cwt);
    const D2 cwz = ld2(FLD(cofwz), ix), cwr = ld2(FLD(cofwr), ix);
    const D2 xr = rw_old + (dts * w2 - cwz * ((zz * ts - zzm * tsm) + resm * (zz * rt_old - zzm * rtm))             // :1662-1667
                            - cwr * ((rs + rsm) + resm * (rho_old + rhm))
                            + cwt * (ts + resm * rt_old)
                            + cwtm * (tsm + resm * rtm));
    const D2 at = ld2(FLD(a_tri), ix), al = ld2(FLD(alpha_tri), ix), gt = ld2(FLD(gamma_tri), ix);
    s_x[k0] = k0 > 0 ? xr.x : rw_old.x; s_a[k0] = at.x; s_al[k0] = al.x; s_g[k0] = gt.x;
    if (m1) { s_x[k1] = xr.y; s_a[k1] = at.y; s_al[k1] = al.y; s_g[k1] = gt.y; }
    if (k0 == 0) s_x[L] = S0 ? 0.0 : FLD(rw_p)[(size_t)x * LP + L];
  }
  if (threadIdx.x == 0) s_al[L + 1] = act ? 1.0 : 0.0;
  __syncthreads();
  {   // the two sweeps, strictly in order: one lane per column, all in the block's first warp
    const int lin = ty * blockDim.x + threadIdx.x;
    if (lin < CB && sm[(size_t)(4 * CB + lin) * TS + L + 1] != 0.0) {
      double* cx = sm + (size_t)(2 * CB + lin) * TS; const double* ca = sm + (size_t)(3 * CB + lin) * TS;
      const double* cal = sm + (size_t)(4 * CB + lin) * TS; const double* cg = sm + (size_t)(5 * CB + lin) * TS;
      double xv = cx[0];
#pragma unroll 4
      for (int kk = 1; kk < L; ++kk) { xv = (cx[kk] - ca[kk] * xv) * cal[kk]; cx[kk] = xv; }         // :1670-1671
      xv = cx[L];
#pragma unroll 4
      for (int kk = L - 1; kk >= 0; --kk) { xv = cx[kk] - cg[kk] * xv; cx[kk] = xv; }                 // :1674-1677
    }
  }
  __syncthreads();
  D2 xn = bc(0), ww_new = bc(0);
  if (act) {
    xn = mk(s_x[k0], m1 ? s_x[k1] : 0.0);
    const D2 ww_old = S0 ? bc(0.0) : ld2(FLD(wwAvg), ix);
    const D2 rz = ld2(FLD(rho_zz), ix), rzm = below(FLD(rho_zz), ix, k0, rz);
    const D2 fm = ld2(FLD(fzm), k0), fp = ld2(FLD(fzp), k0);
    const D2 ds = ld2(FLD(dss), ix), d3 = ld2(FLD(rw_save), ix) - ld2(FLD(rw), ix);
    D2 xd = xn + (d3 - dts * ds * (fm * zz + fp * zzm) * (fm * rz + fp * rzm) * w2);                  // :1682-1684
    xd = xd / (1.0 + dts * ds);                                                                       // :1685
    xd = xd - d3;                                                                                     // :1686
    const D2 wb = (ww_old + 0.5 * (1.0 - epssm) * rw_old) + 0.5 * (1.0 + epssm) * xd;                 // :1661, :1689
    if (k0 > 0) { xn.x = xd.x; ww_new.x = wb.x; } else ww_new.x = ww_old.x;
    xn.y = xd.y; ww_new.y = wb.y;
    s_a[k0] = xn.x;                                                     // s_a is free now: the final rw_p of the column
    if (m1) s_a[k1] = xn.y;
    if (k0 == 0) s_a[L] = s_x[L];
  }
  __syncthreads();
  if (!m0) return;
  if (act) {
    const D2 cofrz = ld2(FLD(cofrz), k0), rdzw = ld2(FLD(rdzw), k0);
    const D2 coftz = ld2(FLD(coftz), ix), coftz_p = above(FLD(coftz), ix, k0, L, coftz);
    const D2 xp = mk(s_a[k1], k1 + 1 <= L ? s_a[k1 + 1] : 0.0);
    st2m(FLD(rho_pp), ix, rs - cofrz * (xp - xn), m0, m1);                                            // :1694
    st2m(FLD(rtheta_pp), ix, ts - rdzw * (coftz_p * xp - coftz * xn), m0, m1);                        // :1695-1696
    st2m(FLD(rw_p), ix, xn, m0, m1); st2m(FLD(wwAvg), ix, ww_new, m0, m1);
  } else {                                                                                            // :1698-1703
    const D2 ww_old = S0 ? bc(0.0) : ld2(FLD(wwAvg), ix);
    const D2 rw_new = rw_old + dts * ld2(FLD(w), ix);
    st2m(FLD(rho_pp), ix, rho_old + dts * ld2(FLD(tend_rho), ix), m0, m1);
    st2m(FLD(rtheta_pp), ix, rt_old + dts * ld2(FLD(theta_m), ix), m0, m1);
    st2m(FLD(rw_p), ix, rw_new, m0, m1); st2m(FLD(wwAvg), ix, ww_new = ww_old + 0.5 * (1.0 + epssm) * rw_new, m0, m1);
  }
}

// ---- TMA (bulk async copy) helpers: global -> shared strips whose bytes in flight cost no registers -----------------
DI uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
DI void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%1], %0;" ::"r"(count), "r"(smem_u32(bar)));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
DI void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%1], %0;" ::"r"(bytes), "r"(smem_u32(bar)) : "memory");
}
DI void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
DI void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok = 0;
  for (int spin = 0; spin < (1 << 28); ++spin) {
    asm volatile("{\n\t.reg .pred P1;\n\tmbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\tselp.u32 %0, 1, 0, P1;\n\t}"
                 : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    if (ok) return;
  }
  __trap();      // a lost transaction must fail loudly, never hang the GPU
}

// TMA form of the fused acoustic kernel (MpasConfig.acoustic_tma = 1).  A block owns C whole columns; for a tile
// of C consecutive columns every own-column input field is ONE contiguous strip of C*LP doubles, fetched with one
// cp.async.bulk per field into shared memory (14 or 18 strips per block, issued up front by 18 threads; completion on
// an mbarrier).  While the strips are in flight the threads do the index loads and the edgesOnCell gathers.  All
// column arithmetic then reads shared memory.  Same arithmetic as k_acoustic.
enum { AF_tend_rho, AF_theta_m, AF_w, AF_coftz, AF_cofwz, AF_cofwr, AF_cofwt, AF_a_tri, AF_alpha_tri, AF_zz, AF_rw_save, AF_rw,
       AF_dss, AF_rho_zz, AF_rs, AF_ts, AF_rho_pp, AF_rtheta_pp, AF_rw_p, AF_wwAvg, AF_COUNT };
struct AcPtrs { const double* p[AF_COUNT]; };
template <bool S0, int ABL = 0>     // ABL: ablation switches for profiling only (1 = no gathers, 2 = no sweep, 4 = no stores)
__global__ void __launch_bounds__(128, 5) k_acoustic_tma(const View V, const AcPtrs F, double dts, double epssm, double resm) {
  extern __shared__ __align__(128) unsigned char smraw[];
  PAIR_THREAD_R()
  const int C = blockDim.y, TS = LP + 2, NF = S0 ? (int)AF_rho_pp : (int)AF_COUNT;
  const int CL = C * LP;
  double* in = reinterpret_cast<double*>(smraw);                 // [NF][C*LP]
  double* s_rp0 = in + (size_t)NF * CL + (size_t)threadIdx.y * TS;
  double* s_rt0 = s_rp0 + (size_t)C * TS;
  double* s_P = s_rt0 + (size_t)C * TS;
  double* s_Q = s_P + (size_t)C * TS;
  uint64_t* bar = reinterpret_cast<uint64_t*>(in + (size_t)NF * CL + (size_t)4 * C * TS);
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  if (tid == 0) mbar_init(bar, 1);
  __syncthreads();
  const size_t tile0 = ((size_t)V.xoff + (size_t)blockIdx.x * C) * LP;
  if (tid == 0) mbar_expect_tx(bar, (uint32_t)(NF * CL * sizeof(double)));
  for (int f = tid; f < NF; f += blockDim.x * blockDim.y)         // one strip per thread (blocks can be smaller than NF)
    bulk_g2s(in + (size_t)f * CL, F.p[f] + tile0, (uint32_t)(CL * sizeof(double)), bar);
  const size_t cl = (size_t)threadIdx.y * LP + k0;                 // this thread's level pair inside a strip
#define SIN(f) (in + (size_t)(f) * CL)
  const bool spec = inx ? (V.specZoneMaskCell[x] != 0.0) : false;
  if (S0 && inx) {                                                                                    // :1625-1630, level L
    if (k0 == L) { FLD(wwAvg)[ix] = 0; FLD(rw_p)[ix] = 0; }
    if (k1 == L) { FLD(wwAvg)[ix + 1] = 0; FLD(rw_p)[ix + 1] = 0; }
  }
  D2 rs = bc(0), ts = bc(0);
  if (m0 && !spec && !(ABL & 8)) {                                 // gathers overlap with the bulk copies
    const double* tm = FLD(theta_m);
    const int ME = V.maxEdges, n = (ABL & 1) ? 0 : V.nEdgesOnCell[x];
    const double* ru_p = FLD(ru_p);
    const double inva = V.invAreaCell[x];
#pragma unroll 2
    for (int i = 0; i < n; ++i) {                                                                     // :1644-1652
      const int e = V.edgesOnCell[x * V.MEP + i];
      const int c1 = V.c1OnCell[x * V.MEP + i], c2 = V.c2OnCell[x * V.MEP + i];
      const D2 flux = V.edgesOnCellSign[x * ME + i] * dts * V.dvOnCell[x * ME + i] * G2(ru_p, e) * inva;
      rs -= flux;
      ts -= flux * 0.5 * (G2(tm, c2) + G2(tm, c1));
    }
  }
  mbar_wait(bar, 0);
  D2 rw_old = bc(0), rw_oldp = bc(0), rho_old = bc(0), rt_old = bc(0);
  D2 cofrz = bc(0), rdzw = bc(0), coftz = bc(0), coftz_p = bc(0);
  AcTerms t0;
  t0.A0 = t0.A1 = t0.A2 = t0.al = t0.r1 = t0.r3 = t0.Q = 0.0; t0.r2 = 1.0;
  double P0 = 0.0, Q0 = 0.0, P1 = 0.0, Q1 = 1.0;
  if (m0) {
    cofrz = ld2(FLD(cofrz), k0); rdzw = ld2(FLD(rdzw), k0);
    if (!S0) {
      rw_old = ld2(SIN(AF_rw_p), cl); rw_oldp = above(SIN(AF_rw_p), cl, k0, L, rw_old);
      rho_old = ld2(SIN(AF_rho_pp), cl); rt_old = ld2(SIN(AF_rtheta_pp), cl);
    }
    st2m(FLD(rtheta_pp_old), ix, S0 ? bc(0.0) : rt_old, m0, m1);                                      // :1615-1623
    if (!spec) {
      const D2 w2 = ld2(SIN(AF_w), cl), tr = ld2(SIN(AF_tend_rho), cl), tm2 = ld2(SIN(AF_theta_m), cl);
      coftz = ld2(SIN(AF_coftz), cl); coftz_p = above(SIN(AF_coftz), cl, k0, L, coftz);
      if (ABL & 8) { rs = ld2(SIN(AF_rs), cl); ts = ld2(SIN(AF_ts), cl); }      // phase 1 of the split form (k_acoustic_gather)
      rs = rho_old + dts * tr + rs - cofrz * resm * (rw_oldp - rw_old);                               // :1657
      ts = rt_old + dts * tm2 + ts - resm * rdzw * (coftz_p * rw_oldp - coftz * rw_old);              // :1658
      const D2 rp0 = rs - cofrz * rw_oldp, rt0 = ts - rdzw * (coftz_p * rw_oldp);
      const D2 zz = ld2(SIN(AF_zz), cl), zzm = below(SIN(AF_zz), cl, k0, zz);
      const D2 cwt = ld2(SIN(AF_cofwt), cl), cwtm = below(SIN(AF_cofwt), cl, k0, cwt);
      const D2 rz = ld2(SIN(AF_rho_zz), cl), rzm = below(SIN(AF_rho_zz), cl, k0, rz);
      const D2 cwz = ld2(SIN(AF_cofwz), cl), cwr = ld2(SIN(AF_cofwr), cl);
      const D2 fm = ld2(FLD(fzm), k0), fp = ld2(FLD(fzp), k0);
      const D2 ds = ld2(SIN(AF_dss), cl), rws = ld2(SIN(AF_rw_save), cl), rwv = ld2(SIN(AF_rw), cl);
      const D2 at = ld2(SIN(AF_a_tri), cl), al = ld2(SIN(AF_alpha_tri), cl);
      if (k0 > 0) {
        const double cofrz_m = FLD(cofrz)[k0 - 1], rdzw_m = FLD(rdzw)[k0 - 1], coftz_m = SIN(AF_coftz)[cl - 1];
        t0 = ac_terms(dts, resm, rw_old.x, w2.x, ts.x, rs.x, rt_old.x, rho_old.x, zz.x, zzm.x, cwt.x, cwtm.x, rz.x, rzm.x, cwz.x, cwr.x,
                      fm.x, fp.x, ds.x, rws.x, rwv.x, cofrz_m, rdzw_m * coftz_m, at.x, al.x);
        Q0 = t0.Q;
      } else { P0 = rw_old.x; Q0 = 0.0; }
      if (m1) {
        const AcTerms t1 = ac_terms(dts, resm, rw_old.y, w2.y, ts.y, rs.y, rt_old.y, rho_old.y, zz.y, zzm.y, cwt.y, cwtm.y, rz.y, rzm.y,
                                    cwz.y, cwr.y, fm.y, fp.y, ds.y, rws.y, rwv.y, cofrz.x, rdzw.x * coftz.x, at.y, al.y);
        P1 = ac_P(t1, rp0.x, rt0.x); Q1 = t1.Q;
        s_rp0[k1] = rp0.y; s_rt0[k1] = rt0.y;
      }
    }
  }
  __syncthreads();
  // Two-level sweep: every thread folds its two levels into one affine map, ONE thread per column runs the
  // recurrence over the 28 pair maps (half the serial length), every thread then finishes its own two levels.
  const int pr = threadIdx.x;
  if (m0 && !spec) {
    if (k0 > 0) P0 = ac_P(t0, s_rp0[k0 - 1], s_rt0[k0 - 1]);
    s_P[pr] = __fma_rn(Q1, P0, P1); s_Q[pr] = Q1 * Q0;          // level k1 is the identity map (P1 = 0, Q1 = 1) when it is inactive
  }
  __syncthreads();
  if (inx && !spec && k0 == 0 && !(ABL & 2)) {
    const int np = (L + 1) / 2;
    double xe = s_P[0];
#pragma unroll 4
    for (int p = 1; p < np; ++p) { xe = __fma_rn(s_Q[p], xe, s_P[p]); s_P[p] = xe; }
  }
  __syncthreads();
  if (!m0) return;
  const D2 ww_old = S0 ? bc(0.0) : ld2(SIN(AF_wwAvg), cl);
  D2 rw_new, rho_new, rt_new, ww_new;
  if (!spec) {
    const double xprev = pr > 0 ? s_P[pr - 1] : 0.0;           // rw_p_new of the level below this pair
    const double x0 = __fma_rn(Q0, xprev, P0);
    rw_new = mk(x0, m1 ? __fma_rn(Q1, x0, P1) : 0.0);
    const D2 wa = ww_old + 0.5 * (1.0 - epssm) * rw_old;                                              // :1661
    const D2 wb = wa + 0.5 * (1.0 + epssm) * rw_new;                                                  // :1689
    ww_new = mk(k0 > 0 ? wb.x : ww_old.x, wb.y);
    rho_new = rs - cofrz * (rw_oldp - rw_new);                                                        // :1694
    rt_new = ts - rdzw * (coftz_p * rw_oldp - coftz * rw_new);                                        // :1695-1696
  } else {                                                                                            // :1698-1703
    rho_new = rho_old + dts * ld2(SIN(AF_tend_rho), cl);
    rt_new = rt_old + dts * ld2(SIN(AF_theta_m), cl);
    rw_new = rw_old + dts * ld2(SIN(AF_w), cl);
    ww_new = ww_old + 0.5 * (1.0 + epssm) * rw_new;
  }
  if ((ABL & 4) && rho_new.x != 1.2345e300) return;       // profiling only: keep the math, drop the stores
  st2m(FLD(rho_pp), ix, rho_new, m0, m1); st2m(FLD(rtheta_pp), ix, rt_new, m0, m1);
  const bool wr0 = S0 || spec || k0 > 0;
  st2m(FLD(rw_p), ix, rw_new, wr0, m1); st2m(FLD(wwAvg), ix, ww_new, wr0, m1);
#undef SIN
}

// ---- EXACT, column-per-lane streaming form (MpasConfig.acoustic_tma = 3, the default) ----------------------------------------
// Why exact is the default: the affine regrouping of k_acoustic_tma changes rw_p by a few ulp of its LARGEST term, which the
// differences taken by atm_divergence_damping_3d amplify -- at BASELINE config 2 (x1.40962 x 41, dt = 180 s) ru_p then misses
// the 1e-12 bound after ONE step (3.7e-12; profiles/r2_acoustic_exact.md).  With this kernel every field of the step except
// q / tend_u (Q14) is bit-identical to the oracle, at the affine kernel's speed.
// "The vertical implicit acoustic solve runs one thread per column" (north_star), at streaming speed: a block is a
// warp-specialised pipeline over a tile of 32 consecutive columns.
//   * warp 0, the SWEEPER: lane = column.  It walks the levels strictly in the reference's order (the body of
//     k_acoustic_column, bit-identical to the oracle) with the recurrence state in registers, reading its inputs two
//     levels at a time (one 128-bit shared-memory load per field) and writing its five outputs the same way.
//   * warps 1..5, the MOVERS (AL_NMOV threads): stream the 20 (16 at small_step 0) input fields of the tile, chunk by chunk of 8 levels, from
//     global memory into a two-stage shared-memory ring with cp.async (16 bytes per lane, 64 contiguous bytes per column
//     and field; the two fields read one level ahead -- coftz(k+1), rw_p(k+1) -- come as 8-byte copies of the shifted
//     strip), and write the finished chunks back with 128-bit stores.
//   * stages are handed over with mbarriers (full/empty for inputs, ofull/oempty for outputs); a stage is laid out
//     [field][column][8 levels] with the 16-byte pieces of a row XOR-swizzled by the column so that the sweeper's
//     128-bit loads and the movers' 128-bit loads/stores are all bank-conflict free.
// 32 recurrences advance per sweeper instruction, two blocks are resident per SM, and while the
// sweeper works on chunk j the copies of chunk j+1 are in flight: the kernel is bound by the strips, not by the chain.
#ifndef AL_NMOV
#define AL_NMOV 160           /* mover threads: 5 warps (3 -> 5: k_acoustic_lane<false> 1.610 -> 1.586, <true> 1.133 -> 1.093 ms/step on x1.163842; 2 warps: 1.837 / 1.233) */
#endif
enum { AL_KC = 8, AL_COLS = 32, AL_NOUT = 5 };
DI void mbar_arrive(uint64_t* bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory"); }
DI void cp_async_arrive_noinc(uint64_t* bar) { asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory"); }
DI void cp_async_16(void* dst, const void* src) { asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory"); }
DI void cp_async_8(void* dst, const void* src) { asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(dst)), "l"(src) : "memory"); }
DI int al_off(int c, int p) { return c * AL_KC + (((p ^ (c >> 1)) & 3) << 1); }      // doubles: row c, swizzled 16-byte piece p
struct AcCarry { double rw_prev, rho_prev, rt_prev, zz_m, cofwt_m, rz_m; };
// one level of :1657-1703, exactly the body of k_acoustic_column
DI void ac_level(int k, bool spec, bool S0, double dts, double epssm, double resm, double cofrz_k, double rdzw_k, double fzm_k, double fzp_k,
                 double tend_rho_k, double theta_m_k, double w_k, double coftz_k, double coftz_p, double cofwz_k, double cofwr_k,
                 double cofwt_k, double a_k, double al_k, double zz_k, double rws_k, double rwv_k, double dsk, double rz_k, double srs_k,
                 double sts_k, double rho_old, double rt_old, double rw_old_k, double rw_old_p, double ww_old, AcCarry& c,
                 double& rho_new, double& rt_new, double& rw_new, double& ww_new) {
  ww_new = ww_old;
  if (!spec) {
    const double rs = rho_old + dts * tend_rho_k + srs_k - cofrz_k * resm * (rw_old_p - rw_old_k);                       // :1657
    const double ts = rt_old + dts * theta_m_k + sts_k - resm * rdzw_k * (coftz_p * rw_old_p - coftz_k * rw_old_k);       // :1658
    rw_new = rw_old_k;
    if (k > 0) {
      ww_new += 0.5 * (1.0 - epssm) * rw_old_k;                                                                          // :1661
      rw_new += dts * w_k - cofwz_k * ((zz_k * ts - c.zz_m * 0.0) + resm * (zz_k * rt_old - c.zz_m * c.rt_prev))
                - cofwr_k * ((rs + 0.0) + resm * (rho_old + c.rho_prev))
                + cofwt_k * (ts + resm * rt_old)
                + c.cofwt_m * (0.0 + resm * c.rt_prev);                                                                   // :1662-1667
      rw_new -= a_k * c.rw_prev;                                                                                         // :1670
      rw_new *= al_k;                                                                                                    // :1671
      const double r3 = rws_k - rwv_k;
      rw_new += r3 - dts * dsk * (fzm_k * zz_k + fzp_k * c.zz_m) * (fzm_k * rz_k + fzp_k * c.rz_m) * w_k;                 // :1682-1684
      const double r2 = 1.0 + dts * dsk;
      if (r2 != 1.0) rw_new /= r2;                                     // x / 1.0 == x exactly: skip the division where dss = 0  :1685
      rw_new -= r3;                                                                                                      // :1686
      ww_new += 0.5 * (1.0 + epssm) * rw_new;                                                                            // :1689
    }
    rho_new = rs - cofrz_k * (rw_old_p - rw_new);                                                                        // :1694
    rt_new = ts - rdzw_k * (coftz_p * rw_old_p - coftz_k * rw_new);                                                      // :1695-1696
  } else {                                                                                                               // :1698-1703
    rho_new = rho_old + dts * tend_rho_k;
    rt_new = rt_old + dts * theta_m_k;
    rw_new = rw_old_k + dts * w_k;
    ww_new = ww_old + 0.5 * (1.0 + epssm) * rw_new;
  }
  c.rw_prev = rw_new; c.rho_prev = rho_new; c.rt_prev = rt_new; c.zz_m = zz_k; c.cofwt_m = cofwt_k; c.rz_m = rz_k;
  (void)S0;
}
template <bool S0>
__global__ void __launch_bounds__(32 + AL_NMOV, 2) k_acoustic_lane(const View V, const AcPtrs F, double dts, double epssm, double resm) {
  extern __shared__ __align__(128) unsigned char smraw[];
  constexpr int NS16 = S0 ? (int)AF_rho_pp : (int)AF_COUNT;      // fields copied 16 bytes at a time (AF_* order)
  constexpr int NS8 = S0 ? 1 : 2;                                // shifted strips: coftz(k+1) [, rw_p(k+1)]
  constexpr int NSTR = NS16 + NS8;
  constexpr int STRIP = AL_COLS * AL_KC;                         // doubles per field per stage
  double* in = reinterpret_cast<double*>(smraw);                 // [2][NSTR][STRIP]
  double* out = in + (size_t)2 * NSTR * STRIP;                   // [2][AL_NOUT][STRIP]
  double* s_v = out + (size_t)2 * AL_NOUT * STRIP;               // cofrz, rdzw, fzm, fzp  [4][LP]
  const int L = V.L, LP = V.LP;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_v + (size_t)4 * LP);
  uint64_t* full = bars; uint64_t* empty = bars + 2; uint64_t* ofull = bars + 4; uint64_t* oempty = bars + 6;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int nch = (L + AL_KC - 1) / AL_KC;
  // persistent: a block walks the tiles blockIdx.x, + gridDim.x, ... as ONE stream of chunks, so the ring never drains between tiles
  const int ntile = (V.xend - V.xoff + AL_COLS - 1) / AL_COLS;
  const int my_tiles = ((int)blockIdx.x < ntile) ? (ntile - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
  const int ng = my_tiles * nch;                                 // chunks this block streams
  if (tid == 0) {
    for (int s = 0; s < 2; ++s) { mbar_init(full + s, AL_NMOV); mbar_init(empty + s, 32); mbar_init(ofull + s, 32); mbar_init(oempty + s, AL_NMOV); }
  }
  for (int i = tid; i < LP; i += blockDim.x) {
    s_v[i] = FLD(cofrz)[i]; s_v[LP + i] = FLD(rdzw)[i]; s_v[2 * LP + i] = FLD(fzm)[i]; s_v[3 * LP + i] = FLD(fzp)[i];
  }
  __syncthreads();
  if (warp == 0) {
    // ------------------------------------------------ sweeper: lane = column ------------------------------------------------
    const int c = lane;
    int x = 0; bool on = false, spec = false;
    AcCarry cr; cr.rw_prev = cr.rho_prev = cr.rt_prev = cr.zz_m = cr.cofwt_m = cr.rz_m = 0.0;
    for (int g = 0; g < ng; ++g) {
      const int j = g % nch;
      if (j == 0) {                                              // next tile: new columns, recurrence state back to level -1
        x = V.xoff + ((int)blockIdx.x + (g / nch) * (int)gridDim.x) * AL_COLS + c;
        on = x < V.xend;
        spec = on ? (V.specZoneMaskCell[x] != 0.0) : false;
        cr.rw_prev = cr.rho_prev = cr.rt_prev = cr.zz_m = cr.cofwt_m = cr.rz_m = 0.0;
      }
      const int s = g & 1, u = g >> 1;
      mbar_wait(full + s, u & 1);
      if (g >= 2) mbar_wait(oempty + s, (u - 1) & 1);
      const double* __restrict__ si = in + (size_t)s * NSTR * STRIP;
      double* __restrict__ so = out + (size_t)s * AL_NOUT * STRIP;
#pragma unroll
      for (int p = 0; p < AL_KC / 2; ++p) {
        const int k0 = j * AL_KC + 2 * p;
        const int o = al_off(c, p);
#define LDP(f) (*reinterpret_cast<const D2*>(si + (size_t)(f) * STRIP + o))
        const D2 tr = LDP(AF_tend_rho), tm = LDP(AF_theta_m), w2 = LDP(AF_w), cz = LDP(AF_coftz), cwz = LDP(AF_cofwz), cwr = LDP(AF_cofwr),
                 cwt = LDP(AF_cofwt), at = LDP(AF_a_tri), al = LDP(AF_alpha_tri), zz = LDP(AF_zz), rws = LDP(AF_rw_save), rwv = LDP(AF_rw),
                 ds = LDP(AF_dss), rz = LDP(AF_rho_zz), rsh = LDP(AF_rs), tsh = LDP(AF_ts);
        const D2 czn = LDP(NS16);                                          // coftz(k+1)
        D2 rho_o = bc(0.0), rt_o = bc(0.0), rwp = bc(0.0), wwo = bc(0.0), rwpn = bc(0.0);
        if (!S0) { rho_o = LDP(AF_rho_pp); rt_o = LDP(AF_rtheta_pp); rwp = LDP(AF_rw_p); wwo = LDP(AF_wwAvg); rwpn = LDP(NS16 + 1); }
#undef LDP
        D2 rho_n = bc(0.0), rt_n = bc(0.0), rw_n = bc(0.0), ww_n = bc(0.0);
#ifdef AL_ABLATE_SWEEP      /* measurement only: the sweeper moves data but skips the arithmetic (results are wrong) */
        if (false)
#else
        if (on && k0 < L)
#endif
          ac_level(k0, spec, S0, dts, epssm, resm, s_v[k0], s_v[LP + k0], s_v[2 * LP + k0], s_v[3 * LP + k0], tr.x, tm.x, w2.x, cz.x, czn.x,
                   cwz.x, cwr.x, cwt.x, at.x, al.x, zz.x, rws.x, rwv.x, ds.x, rz.x, rsh.x, tsh.x, rho_o.x, rt_o.x, rwp.x, rwpn.x, wwo.x, cr,
                   rho_n.x, rt_n.x, rw_n.x, ww_n.x);
#ifdef AL_ABLATE_SWEEP
        if (false)
#else
        if (on && k0 + 1 < L)
#endif
          ac_level(k0 + 1, spec, S0, dts, epssm, resm, s_v[k0 + 1], s_v[LP + k0 + 1], s_v[2 * LP + k0 + 1], s_v[3 * LP + k0 + 1], tr.y, tm.y, w2.y,
                   cz.y, czn.y, cwz.y, cwr.y, cwt.y, at.y, al.y, zz.y, rws.y, rwv.y, ds.y, rz.y, rsh.y, tsh.y, rho_o.y, rt_o.y, rwp.y, rwpn.y,
                   wwo.y, cr, rho_n.y, rt_n.y, rw_n.y, ww_n.y);
        *reinterpret_cast<D2*>(so + (size_t)0 * STRIP + o) = rho_n;
        *reinterpret_cast<D2*>(so + (size_t)1 * STRIP + o) = rt_n;
        *reinterpret_cast<D2*>(so + (size_t)2 * STRIP + o) = rw_n;
        *reinterpret_cast<D2*>(so + (size_t)3 * STRIP + o) = ww_n;
        *reinterpret_cast<D2*>(so + (size_t)4 * STRIP + o) = rt_o;            // rtheta_pp_old  :1615-1623
      }
      mbar_arrive(empty + s);
      mbar_arrive(ofull + s);
      if (S0 && on && j == nch - 1) { FLD(wwAvg)[(size_t)x * LP + L] = 0; FLD(rw_p)[(size_t)x * LP + L] = 0; }   // :1625-1630, level L
    }
  } else {
    // ------------------------------------------------ movers ------------------------------------------------
    const int m = tid - 32;
    double* const dst_f[AL_NOUT] = {FLD(rho_pp), FLD(rtheta_pp), FLD(rw_p), FLD(wwAvg), FLD(rtheta_pp_old)};
    const int xl = V.xend - 1;                                     // columns past the range read the last valid one
    for (int g = 0; g <= ng; ++g) {
      if (g < ng) {
        const int s = g & 1, u = g >> 1;
        if (g >= 2) mbar_wait(empty + s, (u - 1) & 1);
        double* si = in + (size_t)s * NSTR * STRIP;
        const int kb = (g % nch) * AL_KC;
        const int x0 = V.xoff + ((int)blockIdx.x + (g / nch) * (int)gridDim.x) * AL_COLS;
        for (int it = m; it < NS16 * (AL_COLS * 4); it += AL_NMOV) {
          const int f = it >> 7, cp = it & 127, c = cp >> 2, p = cp & 3;
          const int xc = min(x0 + c, xl);
          cp_async_16(si + (size_t)f * STRIP + al_off(c, p), F.p[f] + (size_t)xc * LP + kb + 2 * p);
        }
        for (int it = m; it < NS8 * (AL_COLS * 8); it += AL_NMOV) {
          const int f = it >> 8, ck = it & 255, c = ck >> 3, kk = ck & 7;
          const int xc = min(x0 + c, xl);
          const double* src = (f == 0 ? F.p[AF_coftz] : F.p[AF_rw_p]) + (size_t)xc * LP + kb + kk + 1;
          cp_async_8(si + (size_t)(NS16 + f) * STRIP + al_off(c, kk >> 1) + (kk & 1), src);
        }
        cp_async_arrive_noinc(full + s);
      }
      if (g >= 1) {
        const int gg = g - 1, s = gg & 1, u = gg >> 1;
        mbar_wait(ofull + s, u & 1);
        const double* so = out + (size_t)s * AL_NOUT * STRIP;
        const int kb = (gg % nch) * AL_KC;
        const int x0 = V.xoff + ((int)blockIdx.x + (gg / nch) * (int)gridDim.x) * AL_COLS;
        for (int it = m; it < AL_NOUT * (AL_COLS * 4); it += AL_NMOV) {
          const int f = it >> 7, cp = it & 127, c = cp >> 2, p = cp & 3;
          const int x = x0 + c, k0 = kb + 2 * p;
          const D2 v = *reinterpret_cast<const D2*>(so + (size_t)f * STRIP + al_off(c, p));
          if (x < V.xend && k0 < L) st2m(dst_f[f], (size_t)x * LP + k0, v, true, k0 + 1 < L);
        }
        mbar_arrive(oempty + s);
      }
    }
  }
}

// Two-kernel, strictly left-to-right form (MpasConfig.acoustic_exact = 1).  One thread per level in
// phase 1, one thread per column in phase 2.
__global__ void k_acoustic_flux(const View V, double dts, int small_step) {
  const int k = threadIdx.x;
  const int x = blockIdx.x * blockDim.y + threadIdx.y;
  if (x >= V.nCells) return;
  const int LP = V.LP, L = V.L;
  const size_t ix = (size_t)x * LP + k;
  if (k == L && small_step == 0) { FLD(wwAvg)[ix] = 0; FLD(rw_p)[ix] = 0; }
  if (k >= L) return;
  FLD(rtheta_pp_old)[ix] = (small_step == 0) ? 0.0 : FLD(rtheta_pp)[ix];
  if (V.specZoneMaskCell[x] != 0.0) return;
  const int ME = V.maxEdges, n = V.nEdgesOnCell[x];
  const double* ru_p = FLD(ru_p); const double* tm = FLD(theta_m);
  const double inva = V.invAreaCell[x];
  double rs = 0, ts = 0;
  for (int i = 0; i < n; ++i) {
    const int e = V.edgesOnCell[x * V.MEP + i];
    const int c1 = V.c1OnCell[x * V.MEP + i], c2 = V.c2OnCell[x * V.MEP + i];
    const double flux = V.edgesOnCellSign[x * ME + i] * dts * V.dvOnCell[x * ME + i] * G1(ru_p, e, k) * inva;
    rs -= flux;
    ts -= flux * 0.5 * (G1(tm, c2, k) + G1(tm, c1, k));
  }
  V.scr_rs[ix] = rs; V.scr_ts[ix] = ts;
}
__global__ void k_acoustic_column(const View V, double dts, int small_step, double epssm, double resm) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= V.nCells) return;
  const int L = V.L, LP = V.LP;
  const size_t b = (size_t)c * LP;
  const bool S0 = small_step == 0;
  const double* cofrz = FLD(cofrz); const double* rdzw = FLD(rdzw); const double* fzm = FLD(fzm); const double* fzp = FLD(fzp);
  double* rho_pp = FLD(rho_pp) + b; double* rtheta_pp = FLD(rtheta_pp) + b; double* rw_p = FLD(rw_p) + b; double* wwAvg = FLD(wwAvg) + b;
  const double* tend_rho = FLD(tend_rho) + b; const double* theta_m = FLD(theta_m) + b; const double* w = FLD(w) + b;
  const double* coftz = FLD(coftz) + b; const double* cofwz = FLD(cofwz) + b; const double* cofwr = FLD(cofwr) + b; const double* cofwt = FLD(cofwt) + b;
  const double* a_tri = FLD(a_tri) + b; const double* alpha_tri = FLD(alpha_tri) + b; const double* zz = FLD(zz) + b;
  const double* rw_save = FLD(rw_save) + b; const double* rw = FLD(rw) + b; const double* dss = FLD(dss) + b; const double* rho_zz = FLD(rho_zz) + b;
  const double* srs = V.scr_rs + b; const double* sts = V.scr_ts + b;
  const bool spec = V.specZoneMaskCell[c] != 0.0;
  double rw_prev = 0, rho_prev = 0, rt_prev = 0;
  double rw_old_k = S0 ? 0.0 : rw_p[0];
  double zz_m = 0.0, cofwt_m = 0.0, rz_m = 0.0;
  for (int k = 0; k < L; ++k) {
    const double rw_old_p = S0 ? 0.0 : rw_p[k + 1];
    const double rho_old = S0 ? 0.0 : rho_pp[k];
    const double rt_old = S0 ? 0.0 : rtheta_pp[k];
    const double ww_old = S0 ? 0.0 : wwAvg[k];
    const double zz_k = zz[k], cofwt_k = cofwt[k], rz_k = rho_zz[k];
    double rw_new, rho_new, rt_new, ww_new = ww_old;
    if (!spec) {
      const double coftz_k = coftz[k], coftz_p = coftz[k + 1];
      const double rs = rho_old + dts * tend_rho[k] + srs[k] - cofrz[k] * resm * (rw_old_p - rw_old_k);                       // :1657
      const double ts = rt_old + dts * theta_m[k] + sts[k] - resm * rdzw[k] * (coftz_p * rw_old_p - coftz_k * rw_old_k);       // :1658
      rw_new = rw_old_k;
      if (k > 0) {
        const double w_k = w[k];
        ww_new += 0.5 * (1.0 - epssm) * rw_old_k;                                                                            // :1661
        rw_new += dts * w_k - cofwz[k] * ((zz_k * ts - zz_m * 0.0) + resm * (zz_k * rt_old - zz_m * rt_prev))
                  - cofwr[k] * ((rs + 0.0) + resm * (rho_old + rho_prev))
                  + cofwt_k * (ts + resm * rt_old)
                  + cofwt_m * (0.0 + resm * rt_prev);                                                                         // :1662-1667
        rw_new -= a_tri[k] * rw_prev;                                                                                        // :1670
        rw_new *= alpha_tri[k];                                                                                              // :1671
        const double dsk = dss[k];
        const double r3 = rw_save[k] - rw[k];
        rw_new += r3 - dts * dsk * (fzm[k] * zz_k + fzp[k] * zz_m) * (fzm[k] * rz_k + fzp[k] * rz_m) * w_k;                   // :1682-1684
        rw_new /= (1.0 + dts * dsk);                                                                                         // :1685
        rw_new -= r3;                                                                                                        // :1686
        ww_new += 0.5 * (1.0 + epssm) * rw_new;                                                                              // :1689
      }
      rho_new = rs - cofrz[k] * (rw_old_p - rw_new);                                                                         // :1694
      rt_new = ts - rdzw[k] * (coftz_p * rw_old_p - coftz_k * rw_new);                                                       // :1695-1696
    } else {                                                                                                                 // :1698-1703
      rho_new = rho_old + dts * tend_rho[k];
      rt_new = rt_old + dts * theta_m[k];
      rw_new = rw_old_k + dts * w[k];
      ww_new = ww_old + 0.5 * (1.0 + epssm) * rw_new;
    }
    rho_pp[k] = rho_new; rtheta_pp[k] = rt_new;
    if (S0 || spec || k > 0) { rw_p[k] = rw_new; wwAvg[k] = ww_new; }
    rw_prev = rw_new; rho_prev = rho_new; rt_prev = rt_new;
    rw_old_k = rw_old_p; zz_m = zz_k; cofwt_m = cofwt_k; rz_m = rz_k;
  }
}

// ============================================================================================
// atm_divergence_damping_3d  :1726-1763
// Persistent blocks loop over edge tiles; the next tile's index word, skip flag and own column are loaded
// before the current tile's gathers are consumed, so the index round trip is off the critical path
// (profiles/r1_divdamp_variants.md, variant v4: 3.37 -> 4.37 TB/s).
__global__ void k_divdamp(const View V, double coef_divdamp) {
  const int k0 = 2 * (int)threadIdx.x, k1 = k0 + 1;
  const int LP = V.LP, L = V.L;
  if (k0 >= L) return;
  const bool m1 = k1 < L;
  const int stride = gridDim.x * blockDim.y;
  const int nE = V.xend;
  int x = V.xoff + blockIdx.x * blockDim.y + threadIdx.y;
  if (x >= nE) return;
  const double* rpp = FLD(rtheta_pp); const double* rppo = FLD(rtheta_pp_old); const double* tm = FLD(theta_m);
  int4 cv = V.ecv[x]; unsigned char skip = V.divdampSkip[x]; double sz = 1.0 - V.specZoneMaskEdge[x];
  D2 r = ld2(FLD(ru_p), (size_t)x * LP + k0);
  while (true) {
    const int xn = x + stride;
    const bool more = xn < nE;
    const int xs = more ? xn : x;
    const int4 cvn = V.ecv[xs]; const unsigned char skn = V.divdampSkip[xs]; const double szn = 1.0 - V.specZoneMaskEdge[xs];
    const D2 rn = ld2(FLD(ru_p), (size_t)xs * LP + k0);
    if (!skip) {
      const D2 a1 = G2(rpp, cv.x), b1 = G2(rppo, cv.x), a2 = G2(rpp, cv.y), b2 = G2(rppo, cv.y), t1 = G2(tm, cv.x), t2 = G2(tm, cv.y);
      const D2 divCell1 = -(a1 - b1);
      const D2 divCell2 = -(a2 - b2);
      st2m(FLD(ru_p), (size_t)x * LP + k0, r + coef_divdamp * (divCell2 - divCell1) * sz / (t1 + t2), true, m1);
    }
    if (!more) break;
    x = xn; cv = cvn; skip = skn; sz = szn; r = rn;
  }
}

// ============================================================================================
// atm_recover_large_step_variables_work  :1766-1872
__global__ void k_rec_pad(const View V) {           // :1792-1794: rho_zz = 1 on the "garbage cell" = the pad cell
  const int k = threadIdx.x;
  if (k < V.L) FLD(rho_zz)[(size_t)V.nCells * V.LP + k] = 1.0;
}
// `fix` (MPASB200_PHYSICS_CORRECTED) restores four expressions: w(level 0) :1810, exner :1819, ru :1840, flux2 :1856 (mpas_b200.h).
__global__ void k_rec_cell1(const View V, double invNs, int rk_step, double dt, double rgas, double rcv, int fix) {   // :1800-1826
  PAIR_THREAD(V.nCells)
  if (!m0) return;
  const D2 rws = ld2(FLD(rw_save), ix);
  const D2 rho_p = ld2(FLD(rho_p_save), ix) + ld2(FLD(rho_pp), ix);
  const D2 rho_zz = rho_p + ld2(FLD(rho_base), ix);
  st2m(FLD(rho_p), ix, rho_p, m0, m1); st2m(FLD(rho_zz), ix, rho_zz, m0, m1);
  D2 ww = ld2(FLD(wwAvg), ix);
  ww *= invNs; ww += rws;
  st2m(FLD(wwAvg), ix, ww, m0, m1);
  const D2 rwv = rws + ld2(FLD(rw_p), ix);
  st2m(FLD(rw), ix, rwv, m0, m1);
  const D2 zz = ld2(FLD(zz), ix);
  D2 wd = rwv / (ld2(FLD(fzm), k0) * zz + ld2(FLD(fzp), k0) * below(FLD(zz), ix, k0, zz));                  // :1810
  if (fix && k0 == 0) wd.x = 0.0;                                                                      // MPAS: w(1) = 0, k = 2..nVertLevels
  st2m(FLD(w), ix, wd, m0, m1);
  const D2 rtb = ld2(FLD(rtheta_base), ix);
  if (rk_step == 2) {
    const D2 rtp = ld2(FLD(rtheta_p_save), ix) + ld2(FLD(rtheta_pp), ix) - dt * rho_zz * ld2(FLD(rt_diabatic_tend), ix);
    st2m(FLD(rtheta_p), ix, rtp, m0, m1);
    st2m(FLD(theta_m), ix, (rtp + rtb) / rho_zz, m0, m1);
    const D2 s = rtp + rtb;
    const D2 sz = zz * (rgas / 100000) * s;
    const D2 ex = fix ? mk(pow(sz.x, rcv), pow(sz.y, rcv)) : zz * (rgas / 100000) * mk(pow(s.x, rcv), pow(s.y, rcv));   // :1819
    st2m(FLD(exner), ix, ex, m0, m1);
    st2m(FLD(pressure_p), ix, zz * rgas * (ex * rtp + rtb * (ex - ld2(FLD(exner_base), ix))), m0, m1);   // :1821
  } else {
    const D2 rtp = ld2(FLD(rtheta_p_save), ix) + ld2(FLD(rtheta_pp), ix);
    st2m(FLD(rtheta_p), ix, rtp, m0, m1);
    st2m(FLD(theta_m), ix, (rtp + rtb) / rho_zz, m0, m1);
  }
}
__global__ void k_rec_edge(const View V, double invNs, int fix) {                                      // :1835-1842
  PAIR_THREAD(V.nEdges)
  if (!m0) return;
  const int4 cv = V.ecv[x];
  const double* rz = FLD(rho_zz);
  const D2 rus = ld2(FLD(ru_save), ix);
  D2 ra = ld2(FLD(ruAvg), ix);
  ra *= invNs; ra += rus;
  st2m(FLD(ruAvg), ix, ra, m0, m1);
  const D2 rup = ld2(FLD(ru_p), ix);
  const D2 ruv = fix ? rus + rup : rus * rup;                                                         // a product, as written (:1840)
  st2m(FLD(ru), ix, ruv, m0, m1);
  st2m(FLD(u), ix, 2 * ruv / (G2(rz, cv.x) + G2(rz, cv.y)), m0, m1);
}
template <int N>
DI double rec_chain(const double* c, double w0, int L) {      // passes 1..L-1 of the level-0 accumulation, terms in registers
  double t[N];
#pragma unroll
  for (int i = 0; i < N; ++i) t[i] = c[i];
  for (int kk = 1; kk < L; ++kk) {
#pragma unroll
    for (int i = 0; i < N; ++i) w0 += t[i];
  }
  return w0;
}
__global__ void k_rec_cell2(const View V, int nRelaxZone, int fix) {                                   // :1844-1871
  extern __shared__ double sm[];
  PAIR_THREAD(V.nCells)
  // per column: t1[16], t2[16], w0, n  (the level-0 chain below runs with one lane per column in the block's first warp)
  double* s_col = sm + (size_t)threadIdx.y * 34;
  const bool act = m0 && V.bdyMaskCell[x] <= nRelaxZone;
  const int ME = V.maxEdges, n = act ? V.nEdgesOnCell[x] : 0;
  const double* ru = FLD(ru); const double* zb = FLD(zb_cell); const double* zb3 = FLD(zb3_cell); const double* rz = FLD(rho_zz);
  const double cf1 = FLD(cf1)[0], cf2 = FLD(cf2)[0], cf3 = FLD(cf3)[0];
  D2 wv = bc(0.0), rz2 = bc(0.0), fm = bc(0.0), fp = bc(0.0);
  if (threadIdx.x == 0) s_col[33] = 0.0;
  if (act) {
    fm = ld2(FLD(fzm), k0); fp = ld2(FLD(fzp), k0);
    wv = ld2(FLD(w), ix);
    rz2 = ld2(rz, ix);
    // levels k0 (if > 0) and k1: w += sign*(zb + sign(flux2)*zb3)*flux2, flux2 a PRODUCT as written (:1855)
    for (int i = 0; i < n; ++i) {
      const int e = V.edgesOnCell[x * V.MEP + i];
      const D2 ru2 = G2(ru, e);
      const D2 rum = below(ru, (size_t)e * LP + k0, k0, ru2);
      const D2 flux2 = fix ? fm * ru2 + fp * rum : fm * ru2 * (fp * rum);
      const double sgn = V.edgesOnCell_sign[x * ME + i];
      const D2 z = ld2(zb, i * V.cellSlot + ix), z3 = ld2(zb3, i * V.cellSlot + ix);
      const D2 add = sgn * (z + sgn1(flux2) * z3) * flux2;
      if (k0 > 0) wv.x += add.x;
      wv.y += add.y;
      if (k0 == 0) {
        // level 0: the surface term is accumulated once per (cell, LEVEL) iteration, i.e. L times, interleaved with the
        // level-0 flux2 term on the first pass (level -1 reads 0).  The terms do not depend on the pass: form them once.
        const double flux = (cf1 * ru2.x + cf2 * ru2.y + cf3 * G1(ru, e, 2));
        s_col[i] = sgn * (z.x + copysign(1.0, flux) * z3.x) * flux;
        const double f20 = fix ? fm.x * ru2.x + fp.x * 0.0 : fm.x * ru2.x * (fp.x * 0.0);
        s_col[16 + i] = sgn * (z.x + copysign(1.0, f20) * z3.x) * f20;
      }
    }
    if (k0 == 0) { s_col[32] = wv.x; s_col[33] = (double)n; }
  }
  __syncthreads();
  {   // the L*n additions in the reference's order: one lane per column, all in the block's first warp(s)
    const int lin = threadIdx.y * blockDim.x + threadIdx.x;
    if (lin < (int)blockDim.y) {
      double* c = sm + (size_t)lin * 34;
      const int nn = (int)c[33];
      if (nn > 0) {
        double w0 = c[32];
        for (int i = 0; i < nn; ++i) { w0 += c[i]; w0 += c[16 + i]; }
        switch (nn) {                  // the common cell degrees keep their terms in registers
          case 5: w0 = rec_chain<5>(c, w0, L); break;
          case 6: w0 = rec_chain<6>(c, w0, L); break;
          case 7: w0 = rec_chain<7>(c, w0, L); break;
          default:
            for (int kk = 1; kk < L; ++kk)
              for (int i = 0; i < nn; ++i) w0 += c[i];
        }
        c[32] = w0;
      }
    }
  }
  __syncthreads();
  if (!act) return;
  if (k0 == 0) {
    wv.x = s_col[32] / (cf1 * rz2.x + cf2 * rz2.y + cf3 * rz[ix + 2]);
    wv.y = wv.y / (fm.y * rz2.y + fp.y * rz2.x);
  } else {
    const D2 rzm = below(rz, ix, k0, rz2);
    wv = wv / (fm * rz2 + fp * rzm);
  }
  st2m(FLD(w), ix, wv, m0, m1);
}

// ============================================================================================
// atm_rk_dynamics_substep_finish  :1951-2007
__global__ void k_finish_cell(const View V, int lt_split, int first, int last, double inv_split) {
  PAIR_THREAD(V.nCells)
  if (!m0) return;
  if (lt_split) {
    st2m(FLD(rw_save), ix, ld2(FLD(rw), ix), m0, m1); st2m(FLD(rtheta_p_save), ix, ld2(FLD(rtheta_p), ix), m0, m1);
    st2m(FLD(rho_p_save), ix, ld2(FLD(rho_p), ix), m0, m1);
    st2m(FLD(w), ix, ld2(FLD(w_2), ix), m0, m1); st2m(FLD(theta_m), ix, ld2(FLD(theta_m_2), ix), m0, m1);
    st2m(FLD(rho_zz), ix, ld2(FLD(rho_zz_2), ix), m0, m1);
  }
  const D2 ws = first ? ld2(FLD(wwAvg), ix) : ld2(FLD(wwAvg), ix) + ld2(FLD(wwAvg_split), ix);
  st2m(FLD(wwAvg_split), ix, ws, m0, m1);
  if (last) { st2m(FLD(wwAvg), ix, ws * inv_split, m0, m1); st2m(FLD(rho_zz), ix, ld2(FLD(rho_zz_old_split), ix), m0, m1); }
}
__global__ void k_finish_edge(const View V, int lt_split, int first, int last, double inv_split) {
  PAIR_THREAD(V.nEdges)
  if (!m0) return;
  if (lt_split) { st2m(FLD(ru_save), ix, ld2(FLD(ru), ix), m0, m1); st2m(FLD(u), ix, ld2(FLD(u_2), ix), m0, m1); }
  const D2 rs = first ? ld2(FLD(ruAvg), ix) : ld2(FLD(ruAvg), ix) + ld2(FLD(ruAvg_split), ix);
  st2m(FLD(ruAvg_split), ix, rs, m0, m1);
  if (last) st2m(FLD(ruAvg), ix, rs * inv_split, m0, m1);
}

// ============================================================================================
// atm_advance_scalars -- absent from the reference (rk_timestep.rg:465,485 skip the call; storage data_structures.rg:36).
// atm_advance_scalars_work of MPAS-Atmosphere v7.0, non-monotonic branch, no physics tendency (mpas_b200.h).  Two kernels:
// the horizontal flux of every scalar through an edge is evaluated once per edge into library scratch (as for theta),
// the cell kernel sums it over edgesOnCell in slot order (deterministic gather, no atomics), adds the vertical flux
// divergence of its own column and updates the scalars in place (a block owns whole columns: reads, barrier, writes).
template <int NS>
__global__ void k_scalar_flux(const View V, double* __restrict__ sflux, size_t edgeSlot) {
  PAIR_THREAD(V.nEdges)
  if (!m0) return;
  const int NA = V.nAdv;
  const double* sc = FLD(scalars);
  const int na = V.nAdvCellsForEdge[x];
  const D2 sg = sgn1(ld2(FLD(ruAvg), ix));
  D2 fa[NS];
#pragma unroll
  for (int s = 0; s < NS; ++s) fa[s] = bc(0.0);
  for (int j = 0; j < na; ++j) {
    const size_t ic = (size_t)V.advCellsForEdge[x * NA + j] * LP + k0;
    const D2 sw = V.adv_coefs[x * NA + j] + sg * V.adv_coefs_3rd[x * NA + j];
#pragma unroll
    for (int s = 0; s < NS; ++s) fa[s] += sw * ld2(sc + s * V.cellSlot, ic);
  }
#pragma unroll
  for (int s = 0; s < NS; ++s) st2m(sflux + s * edgeSlot, ix, fa[s], m0, m1);
}
DI double wdtn_at(int k, int L, double ww, double fm, double fp, double qm2, double qm1, double q0, double qp1, double coef3) {
  double r = 0.0;                                       // wdtn(0) = wdtn(L) = 0
  if (k == 1 || k == L - 1) r = ww * (fm * q0 + fp * qm1);
  if (k > 1 && k < L - 1) r = flux3(qm2, qm1, q0, qp1, ww, coef3);
  return r;
}
template <int NS>
__global__ void k_scalar_update(const View V, const double* __restrict__ sflux, size_t edgeSlot, double dt, double coef3) {
  PAIR_THREAD(V.nCells)
  D2 out[NS];
  if (m0) {
    const int ME = V.maxEdges, n = V.nEdgesOnCell[x];
    const double* ru = FLD(ruAvg);
    D2 tend[NS];
#pragma unroll
    for (int s = 0; s < NS; ++s) tend[s] = bc(0.0);
    for (int i = 0; i < n; ++i) {
      const int e = V.edgesOnCell[x * V.MEP + i];
      const D2 sr = V.edgesOnCellSign[x * ME + i] * G2(ru, e);
#pragma unroll
      for (int s = 0; s < NS; ++s) tend[s] -= sr * G2(sflux + s * edgeSlot, e);
    }
    const double inv = V.invAreaCell[x];
    const double* wwA = FLD(wwAvg);
    const D2 ww = ld2(wwA, ix); const double ww2 = wwA[ix + 2 < (size_t)(x + 1) * LP ? ix + 2 : ix];     // wwAvg(k1+1)
    const D2 fm = ld2(FLD(fzm), k0), fp = ld2(FLD(fzp), k0), rdzw = ld2(FLD(rdzw), k0);
    const double fm2 = k0 + 2 < LP ? FLD(fzm)[k0 + 2] : 0.0, fp2 = k0 + 2 < LP ? FLD(fzp)[k0 + 2] : 0.0;
    const D2 rz = ld2(FLD(rho_zz), ix), rzo = ld2(FLD(rho_zz_old_split), ix);
#pragma unroll
    for (int s = 0; s < NS; ++s) {
      const double* q = FLD(scalars) + s * V.cellSlot;
      const D2 qm = k0 >= 2 ? ld2(q, ix - 2) : bc(0.0), q2 = ld2(q, ix), qp = k0 + 2 < LP ? ld2(q, ix + 2) : bc(0.0);
      const double wd0 = wdtn_at(k0, L, ww.x, fm.x, fp.x, qm.x, qm.y, q2.x, q2.y, coef3);
      const double wd1 = wdtn_at(k1, L, ww.y, fm.y, fp.y, qm.y, q2.x, q2.y, qp.x, coef3);
      const double wd2 = wdtn_at(k1 + 1, L, ww2, fm2, fp2, q2.x, q2.y, qp.x, qp.y, coef3);
      const D2 old = ld2(FLD(scalars_old) + s * V.cellSlot, ix);
      const D2 t = tend[s] * inv;
      out[s] = mk((old.x * rzo.x + dt * (t.x - rdzw.x * (wd1 - wd0))) / rz.x, (old.y * rzo.y + dt * (t.y - rdzw.y * (wd2 - wd1))) / rz.y);
    }
  }
  __syncthreads();                                     // every level pair of the block's columns has read its neighbours' levels
  if (!m0) return;
#pragma unroll
  for (int s = 0; s < NS; ++s) st2m(FLD(scalars) + s * V.cellSlot, ix, out[s], m0, m1);
}
// scalars_old = scalars (MPAS: scalars_2 = scalars_1 in atm_rk_integration_setup); grid.y = slot
__global__ void k_setup_scalars(const View V) {
  PAIR_THREAD(V.nCells)
  if (!m0) return;
  const size_t o = (size_t)blockIdx.y * V.cellSlot;
  st2m(FLD(scalars_old) + o, ix, ld2(FLD(scalars) + o, ix), m0, m1);
}

// ============================================================================================
// Init chain on the device (SURVEY.md 8f rank 3).
// atm_init_coupled_diagnostics  :651-725.  Three passes with the reference's grid-wide dependencies between them:
// rho_zz /= zz on every cell (:676), ru on every edge from both cells' rho_zz (:679-683), then everything cell-local.
__global__ void k_icd_cell1(const View V) {
  PAIR_THREAD(V.nCells)
  if (!m0) return;
  st2m(FLD(rho_zz), ix, ld2(FLD(rho_zz), ix) / ld2(FLD(zz), ix), m0, m1);
}
__global__ void k_icd_edge(const View V) {
  PAIR_THREAD(V.nEdges)
  if (!m0) return;
  const int4 cv = V.ecv[x];
  const double* rz = FLD(rho_zz);
  st2m(FLD(ru), ix, 0.5 * ld2(FLD(u), ix) * (G2(rz, cv.x) + G2(rz, cv.y)), m0, m1);
}
__global__ void k_icd_cell2(const View V, double rgas, double rcv) {
  PAIR_THREAD(V.nCells)
  if (!m0) return;
  const int ME = V.maxEdges, n = V.nEdgesOnCell[x];
  const double* ru = FLD(ru); const double* zb = FLD(zb_cell); const double* zb3 = FLD(zb3_cell);
  const D2 fm = ld2(FLD(fzm), k0), fp = ld2(FLD(fzp), k0);
  const D2 rz = ld2(FLD(rho_zz), ix), rzm = below(FLD(rho_zz), ix, k0, rz);
  const D2 zz = ld2(FLD(zz), ix), zzm = below(FLD(zz), ix, k0, zz);
  const D2 zf = fp * zzm + fm * zz;
  D2 rw = ld2(FLD(w), ix) * (fp * rzm + fm * rz) * zf;                                                 // :691-694
  if (k0 == 0) rw.x = 0.0;
  for (int i = 0; i < n; ++i) {                                                                       // :698-709
    const int e = V.edgesOnCell[x * V.MEP + i];
    const D2 r2 = G2(ru, e);
    const D2 flux = fm * r2 + fp * below(ru, (size_t)e * LP + k0, k0, r2);
    const D2 t = V.edgesOnCellSign[x * ME + i] * (ld2(zb, i * V.cellSlot + ix) + sgn1(flux) * ld2(zb3, i * V.cellSlot + ix)) * flux * zf;
    if (k0 > 0) rw.x -= t.x;
    rw.y -= t.y;
  }
  st2m(FLD(rw), ix, rw, m0, m1);
  const int p0 = 100000;
  const D2 rb = ld2(FLD(rho_base), ix), tb = ld2(FLD(theta_base), ix), tm = ld2(FLD(theta_m), ix);
  const D2 rho_p = rz - rb, rtb = tb * rb;
  const D2 rtp = tm * rho_p + rb * (tm - tb);
  const D2 a = zz * (rgas / p0) * (rtp + rtb), b = zz * (rgas / p0) * (rtb);
  const D2 ex = mk(pow(a.x, rcv), pow(a.y, rcv)), exb = mk(pow(b.x, rcv), pow(b.y, rcv));
  st2m(FLD(rho_p), ix, rho_p, m0, m1); st2m(FLD(rtheta_base), ix, rtb, m0, m1); st2m(FLD(rtheta_p), ix, rtp, m0, m1);
  st2m(FLD(exner), ix, ex, m0, m1); st2m(FLD(exner_base), ix, exb, m0, m1);
  st2m(FLD(pressure_p), ix, zz * rgas * (ex * rtp + rtb * (ex - exb)), m0, m1);
  st2m(FLD(pressure_base), ix, zz * rgas * exb * rtb, m0, m1);
}
// mpas_reconstruct_2d  :1894-1948
__global__ void k_reconstruct(const View V, int on_a_sphere) {
  PAIR_THREAD(V.nCells)
  if (!m0) return;
  const int ME = V.maxEdges, n = V.nEdgesOnCell[x];
  const double* u = FLD(u);
  D2 ux = bc(0.0), uy = bc(0.0), uz = bc(0.0);
  for (int i = 0; i < n; ++i) {
    const D2 ue = G2(u, V.edgesOnCell[x * V.MEP + i]);
    const double* cf = V.coeffsRecon + ((size_t)x * ME + i) * 3;
    ux += cf[0] * ue; uy += cf[1] * ue; uz += cf[2] * ue;
  }
  st2m(FLD(uReconstructX), ix, ux, m0, m1); st2m(FLD(uReconstructY), ix, uy, m0, m1); st2m(FLD(uReconstructZ), ix, uz, m0, m1);
  if (on_a_sphere) {
    const double clat = V.cosLatCell[x], slat = V.sinLatCell[x], clon = V.cosLonCell[x], slon = V.sinLonCell[x];
    st2m(FLD(uReconstructZonal), ix, -ux * slon + uy * clon, m0, m1);
    st2m(FLD(uReconstructMeridional), ix, -(ux * clon + uy * slon) * slat + uz * clat, m0, m1);
  } else {
    st2m(FLD(uReconstructZonal), ix, ux, m0, m1); st2m(FLD(uReconstructMeridional), ix, uy, m0, m1);
  }
}

// ============================================================================================
// region <-> mirror transfers and halo pack/unpack.  `map[i]` = internal (SFC) index of caller index i.
// staging layout: [i][L1][slots] (exactly the host array of an array-typed region field).
__global__ void k_stage_to_field(double* __restrict__ field, const double* __restrict__ staging, const int* __restrict__ map,
                                 int n, int L1, int LP, int slots, size_t slotStride) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t total = (size_t)n * L1 * slots;
  if (t >= total) return;
  const int s = (int)(t % slots); const size_t r = t / slots; const int k = (int)(r % L1); const int i = (int)(r / L1);
  field[s * slotStride + (size_t)map[i] * LP + k] = staging[t];
}
__global__ void k_field_to_stage(const double* __restrict__ field, double* __restrict__ staging, const int* __restrict__ map,
                                 int n, int L1, int LP, int slots, size_t slotStride) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t total = (size_t)n * L1 * slots;
  if (t >= total) return;
  const int s = (int)(t % slots); const size_t r = t / slots; const int k = (int)(r % L1); const int i = (int)(r / L1);
  staging[t] = field[s * slotStride + (size_t)map[i] * LP + k];
}
// halo buffers: [i][field][L1] (one contiguous row per listed entity, so the rows of one peer are one contiguous
// slice of a list that concatenates all peers); idx holds internal indices
struct PackArgs { double* f[32]; int nf; };
__global__ void k_pack(const PackArgs A, const int* __restrict__ idx, int n, int L1, int LP, double* __restrict__ buf) {
  const int k = threadIdx.x; const int i = blockIdx.x * blockDim.y + threadIdx.y; const int fi = blockIdx.y;
  if (i >= n || k >= L1) return;
  buf[((size_t)i * A.nf + fi) * L1 + k] = A.f[fi][(size_t)idx[i] * LP + k];
}
__global__ void k_unpack(const PackArgs A, const int* __restrict__ idx, int n, int L1, int LP, const double* __restrict__ buf) {
  const int k = threadIdx.x; const int i = blockIdx.x * blockDim.y + threadIdx.y; const int fi = blockIdx.y;
  if (i >= n || k >= L1) return;
  A.f[fi][(size_t)idx[i] * LP + k] = buf[((size_t)i * A.nf + fi) * L1 + k];
}

// ============================================================================================
// summarize_timestep  rk_timestep.rg:29-359: global min / max of a field with the place they occur, plus what the
// reference's (disabled) NaN scan looks for, plus an order-independent 64-bit checksum of the bit patterns.
// The scan covers the first n caller-numbered entities (the owned ones of a partition) and levels [0, nlev).
// Every reduction here is commutative and exact (min, max, integer add mod 2^64), so the result does not depend
// on the block schedule, on the renumbering or on how many ranks share the mesh; atomics are therefore harmless
// (this is the checker of the step, not one of its stencils).
struct SumAcc { unsigned long long kmin, kmax, n_nan, n_inf, checksum, loc_min, loc_max; };
DI unsigned long long ord_key(double v) {            // monotone map double -> uint64 (NaN never gets here)
  const unsigned long long b = (unsigned long long)__double_as_longlong(v);
  return (b & 0x8000000000000000ULL) ? ~b : (b | 0x8000000000000000ULL);
}
DI unsigned long long mix64(unsigned long long z) {  // splitmix64 finaliser
  z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ULL; z = (z ^ (z >> 27)) * 0x94d049bb133111ebULL; return z ^ (z >> 31);
}
__global__ void k_summarize(const double* __restrict__ field, const int* __restrict__ map, const int* __restrict__ gid,
                            int n, int nlev, int LP, SumAcc* __restrict__ acc) {
  __shared__ unsigned long long s[5][8];
  unsigned long long kmin = ~0ULL, kmax = 0ULL, nn = 0, ni = 0, cs = 0;
  const size_t total = (size_t)n * nlev;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const int i = (int)(t / nlev), k = (int)(t % nlev);
    const double v = field[(size_t)map[i] * LP + k];
    unsigned long long bits = (unsigned long long)__double_as_longlong(v);
    if (v != v) { nn++; bits = 0x7ff8000000000000ULL; }      // one canonical NaN: payloads differ between CPU and GPU
    else {
      if (isinf(v)) ni++;
      const unsigned long long key = ord_key(v);
      kmin = key < kmin ? key : kmin; kmax = key > kmax ? key : kmax;
    }
    const unsigned long long id = (unsigned long long)(gid ? gid[i] : i) * (unsigned long long)nlev + (unsigned long long)k + 1ULL;
    cs += mix64(bits + 0x9e3779b97f4a7c15ULL * id);
  }
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long a = __shfl_down_sync(0xffffffffu, kmin, o), b = __shfl_down_sync(0xffffffffu, kmax, o);
    kmin = a < kmin ? a : kmin; kmax = b > kmax ? b : kmax;
    nn += __shfl_down_sync(0xffffffffu, nn, o); ni += __shfl_down_sync(0xffffffffu, ni, o); cs += __shfl_down_sync(0xffffffffu, cs, o);
  }
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  if (l == 0) { s[0][w] = kmin; s[1][w] = kmax; s[2][w] = nn; s[3][w] = ni; s[4][w] = cs; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int j = 1; j < (int)(blockDim.x >> 5); ++j) {
      kmin = s[0][j] < kmin ? s[0][j] : kmin; kmax = s[1][j] > kmax ? s[1][j] : kmax; nn += s[2][j]; ni += s[3][j]; cs += s[4][j];
    }
    atomicMin(&acc->kmin, kmin); atomicMax(&acc->kmax, kmax);
    atomicAdd(&acc->n_nan, nn); atomicAdd(&acc->n_inf, ni); atomicAdd(&acc->checksum, cs);
  }
}
// second pass: the FIRST place, in (entity id, level) order, where the extreme values occur (the reference keeps the
// first hit of a strict comparison, rk_timestep.rg:62-72)
__global__ void k_summarize_loc(const double* __restrict__ field, const int* __restrict__ map, const int* __restrict__ gid,
                                int n, int nlev, int LP, SumAcc* __restrict__ acc) {
  const unsigned long long kmin = acc->kmin, kmax = acc->kmax;
  const size_t total = (size_t)n * nlev;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const int i = (int)(t / nlev), k = (int)(t % nlev);
    const double v = field[(size_t)map[i] * LP + k];
    if (v != v) continue;
    const unsigned long long key = ord_key(v);
    const unsigned long long id = (unsigned long long)(gid ? gid[i] : i) * (unsigned long long)nlev + (unsigned long long)k;
    if (key == kmin) atomicMin(&acc->loc_min, id);
    if (key == kmax) atomicMin(&acc->loc_max, id);
  }
}

// ============================================================================================
// Exact global integrals (an extension of summarize_timestep): the exact sum over entities i < n (caller's numbering) and
// levels k < nlev of p = ((a * b) * wh[i]) * wv[k], every product one multiply rounded to nearest in that order (b, wh, wv
// absent = 1).  NaN / +Inf / -Inf products are counted and left out; every finite product enters a fixed-point
// superaccumulator whose limb j holds a signed multiple of 2^(32 j - IACC_BIAS).  A double is m * 2^e with m < 2^53 and
// e >= -1074, so it lands as three 32-bit digits in limbs j, j+1, j+2 with j = (e + IACC_BIAS) / 32 <= 64.  Integer addition
// is associative, so nothing here depends on the grid, the block schedule, the renumbering or the partition.
// Each warp owns one accumulator in shared memory.  When every product of one warp-wide iteration falls in the same two
// limb positions (the usual case: a field spans few binades), the warp sums the digits over its lanes and one lane adds
// four limbs; otherwise each lane adds its own three digits.  Either way one iteration moves a limb by less than
// 32 * 2^32 = 2^37, and the warp folds the carries of its accumulator (limbs 0..66 back into [0, 2^32)) every
// IACC_FOLD_EVERY iterations, so no int64 limb can overflow however many products one warp takes.
constexpr int IACC_LIMBS = 68;          // MPASB200_INTEGRAL_LIMBS
constexpr int IACC_BIAS = 1088;         // limb 0 weighs 2^-1088
constexpr int IACC_FOLD_EVERY = 1 << 24;
constexpr int IACC_WARPS = 8;           // blockDim.x = 32 * IACC_WARPS
struct IntAcc { long long limb[IACC_LIMBS]; unsigned long long n_nan, n_pinf, n_ninf; };

DI void iacc_fold(long long* a) {       // limbs 0..66 into [0, 2^32), the carries into limb 67 (arithmetic shifts)
  long long c = 0;
  for (int j = 0; j < IACC_LIMBS - 1; ++j) { const long long v = a[j] + c; a[j] = v & 0xffffffffLL; c = v >> 32; }
  a[IACC_LIMBS - 1] += c;
}
DI long long warp_sum_ll(long long v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
DI void iacc_add(long long* a, int j, long long v) {
  if (v) atomicAdd(reinterpret_cast<unsigned long long*>(a + j), (unsigned long long)v);   // two's complement: a signed add
}

__global__ void __launch_bounds__(32 * IACC_WARPS)
k_integrate(const double* __restrict__ fa, const double* __restrict__ fb, const int* __restrict__ map,
            const double* __restrict__ wh, const double* __restrict__ wv, int n, int nlev, int LP, IntAcc* __restrict__ out) {
  __shared__ long long acc[IACC_WARPS][IACC_LIMBS];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int j = lane; j < IACC_LIMBS; j += 32) acc[w][j] = 0;
  __syncwarp();
  unsigned long long nn = 0, np = 0, nm = 0;
  const size_t total = (size_t)n * nlev;
  int iters = 0;
  // the loop runs warp-uniformly (lanes past the end take part with no product) so that the full-mask collectives are legal
  for (size_t base = ((size_t)blockIdx.x * IACC_WARPS + w) * 32; base < total; base += (size_t)gridDim.x * blockDim.x) {
    const size_t t = base + lane;
    bool fin = false;
    int j = 0;
    long long d0 = 0, d1 = 0, d2 = 0;
    if (t < total) {
      const int i = (int)(t / nlev), k = (int)(t % nlev);
      const size_t at = (size_t)map[i] * LP + k;
      double p = fa[at];
      if (fb) p = __dmul_rn(p, fb[at]);
      if (wh) p = __dmul_rn(p, wh[i]);
      if (wv) p = __dmul_rn(p, wv[k]);
      if (p != p) nn++;
      else if (isinf(p)) { if (p > 0) np++; else nm++; }
      else if (p != 0.0) {
        const unsigned long long bits = (unsigned long long)__double_as_longlong(p);
        const int ex = (int)((bits >> 52) & 0x7ff);
        unsigned long long m = bits & 0xfffffffffffffULL;
        if (ex) m |= 1ULL << 52;
        const int s = (ex ? ex - 1075 : -1074) + IACC_BIAS;     // bit position of m's unit, >= 14
        const int r = s & 31;
        j = s >> 5;
        const unsigned long long lo = m << r, hi = r ? m >> (64 - r) : 0ULL;   // m * 2^r < 2^85
        d0 = (long long)(lo & 0xffffffffULL); d1 = (long long)(lo >> 32); d2 = (long long)hi;
        if (bits >> 63) { d0 = -d0; d1 = -d1; d2 = -d2; }
        fin = true;
      }
    }
    const unsigned jmin = __reduce_min_sync(0xffffffffu, fin ? (unsigned)j : 0xffffffffu);
    if (jmin != 0xffffffffu) {
      const unsigned jmax = __reduce_max_sync(0xffffffffu, fin ? (unsigned)j : 0u);
      if (jmax - jmin <= 1) {             // jmin + 3 <= 67
        const bool up = fin && (unsigned)j != jmin;
        long long w0 = up ? 0 : d0, w1 = up ? d0 : d1, w2 = up ? d1 : d2, w3 = up ? d2 : 0;
        w0 = warp_sum_ll(w0); w1 = warp_sum_ll(w1); w2 = warp_sum_ll(w2); w3 = warp_sum_ll(w3);
        if (lane == 0) { iacc_add(acc[w], jmin, w0); iacc_add(acc[w], jmin + 1, w1); iacc_add(acc[w], jmin + 2, w2); iacc_add(acc[w], jmin + 3, w3); }
      } else if (fin) {
        iacc_add(acc[w], j, d0); iacc_add(acc[w], j + 1, d1); iacc_add(acc[w], j + 2, d2);
      }
    }
    if (++iters == IACC_FOLD_EVERY) {
      __syncwarp();
      if (lane == 0) iacc_fold(acc[w]);
      __syncwarp();
      iters = 0;
    }
  }
  __syncwarp();
  if (lane == 0) iacc_fold(acc[w]);
  nn = warp_sum_ll((long long)nn); np = warp_sum_ll((long long)np); nm = warp_sum_ll((long long)nm);
  if (lane == 0) {
    if (nn) atomicAdd(&out->n_nan, nn);
    if (np) atomicAdd(&out->n_pinf, np);
    if (nm) atomicAdd(&out->n_ninf, nm);
  }
  __syncthreads();
  // one global add per limb and block: |sum| < IACC_WARPS * 2^32 per block (limb 67 excepted, which stays small) and the
  // grid is a few thousand blocks, so the global limbs cannot overflow; the host folds their carries
  for (int j = threadIdx.x; j < IACC_LIMBS; j += blockDim.x) {
    long long s = 0;
    for (int v = 0; v < IACC_WARPS; ++v) s += acc[v][j];
    iacc_add(out->limb, j, s);
  }
}
