/* mpas_b200.h -- C ABI of libmpas_b200.so
 *
 * Drop-in boundary for the RK3 dynamics hot path of alexaiken/mpas-regent.
 * Every Regent leaf task on the path keeps its signature, privileges and call site
 * (dynamics/rk_timestep.rg:404-481, atm_core.rg:31); its *body* becomes one call of
 * the matching entry point below, made from a Terra shim written to the only FFI
 * pattern the reference has (fortran/examples.rg:14-69: __physical/__fields ->
 * legion_accessor_array_*_raw_rect_ptr -> extern call).  INTEGRATION.md shows the shim.
 *
 * Conventions
 *   - plain C, POD structs, no C++/torch types cross this line;
 *   - every entry returns 0 on success and a negative MPASB200_E* code otherwise, the
 *     message is available from mpasb200_last_error(); nothing here exit()s or throws
 *     (the reference's own convention is "retval == 1 + printf", netcdf_tasks.rg:13-18);
 *   - state is DEVICE-RESIDENT between calls: the library owns a structure-of-arrays
 *     mirror of the hot-path fields (mpas_b200_fields.def); host regions are touched
 *     only by upload_field / download_field;
 *   - task entries enqueue work on the handle's stream and return (asynchronous);
 *     mpasb200_sync() is the host-visible point;
 *   - pointers passed in are borrowed for the duration of the call only;
 *   - there is no CPU fallback: with no usable CUDA device mpasb200_create fails.
 */
#ifndef MPAS_B200_H
#define MPAS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mpasb200 mpasb200_t;

/* ---- error codes ------------------------------------------------------------ */
enum {
  MPASB200_OK        =  0,
  MPASB200_EINVAL    = -1,  /* bad argument (null pointer, id out of range, bad enum) */
  MPASB200_ECUDA     = -2,  /* a CUDA runtime call failed; text in last_error          */
  MPASB200_ENODEVICE = -3,  /* no CUDA device: the library never computes on the host  */
  MPASB200_ESTATE    = -4,  /* call order violated (e.g. task before upload_mesh)      */
  MPASB200_ENOMEM    = -5
};

/* ---- field ids (one per line of mpas_b200_fields.def) -------------------------- */
typedef enum {
#define MPASB200_FIELD(name, entity, slots) MPASB200_F_##name,
#define MPASB200_VFIELD(name)               MPASB200_F_##name,
#include "mpas_b200_fields.def"
#undef MPASB200_FIELD
#undef MPASB200_VFIELD
  MPASB200_F_COUNT
} mpasb200_field_t;

typedef enum { MPASB200_CELL = 0, MPASB200_EDGE = 1, MPASB200_VERTEX = 2, MPASB200_VERTICAL = 3 } mpasb200_entity_t;

/* How a stored mesh id becomes an array index (SURVEY.md 8c, rule M2).
 * LITERAL   : what the reference does -- the 1-based id read from the grid file
 *             (mesh_loading.rg:228-230,268-269,294-295) is used as a 0-based index
 *             (dynamics_tasks.rg:347-350 ...); id == N addresses a zero pad entity.
 * CORRECTED : id-1; id 0 (absent neighbour) addresses the pad entity.             */
typedef enum { MPASB200_INDEX_LITERAL = 0, MPASB200_INDEX_CORRECTED = 1 } mpasb200_index_policy_t;

/* config_horiz_mixing (constants.rg:63).  An enum, because the reference compares
 * rawstring *pointers* (dynamics_tasks.rg:861,892), which is toolchain-dependent.     */
typedef enum { MPASB200_MIX_2D_SMAGORINSKY = 0, MPASB200_MIX_2D_FIXED = 1, MPASB200_MIX_OTHER = 2 } mpasb200_horiz_mixing_t;

/* What atm_srk3 passes as atm_compute_dyn_tend's `rk_step : int`.
 * SUBSTEP_TRUNC : literal -- rk_timestep.rg:437 passes rk_sub_timestep[rk_step] (a
 *                 double) which narrows to int, so the rk_step==0 branches run only
 *                 when the sub-timestep truncates to 0.
 * STAGE_INDEX   : the RK stage index 0,1,2 (what MPAS does).                          */
typedef enum { MPASB200_RKARG_SUBSTEP_TRUNC = 0, MPASB200_RKARG_STAGE_INDEX = 1 } mpasb200_rkarg_policy_t;

/* Which text of the acoustic loop runs (SURVEY.md 8f rank 1).
 * LITERAL   : the reference as it executes: the ru_p / ruAvg edge update is commented out
 *             (dynamics_tasks.rg:1585-1613), so is the tridiagonal back-substitution (:1674-1677), and
 *             atm_srk3 never calls atm_recover_large_step_variables (rk_timestep.rg:459-460).
 * CORRECTED : those three pieces enabled with the semantics of the MPAS-A routines they were transcribed from
 *             (atm_advance_acoustic_step_work, atm_recover_large_step_variables_work of MPAS v7): the edge update
 *             as written in the commented lines; the cell part evaluated column by column (rs/ts kept for the
 *             whole column, forward elimination, then back-substitution with gamma_tri, then Rayleigh damping,
 *             then rho_pp / rtheta_pp); recover called after the acoustic loop of every RK stage with
 *             (number_sub_steps[rk_step], rk_step, dt), with four of its expressions restored
 *             (w(level 0) = 0 before the flux sums instead of rw/0, :1810; exner = (zz*(rgas/p0)*
 *             (rtheta_p+rtheta_base))^rcv, :1819; ru = ru_save + ru_p, :1840; flux = fzm*ru(k) + fzp*ru(k-1), :1856).  Everything else, including the reference's field bindings
 *             (cr.w for tend_rw, cr.theta_m for tend_rt, er.tend_ru), stays literal.  Parity for this mode is against
 *             the oracle's restatement of exactly this text; the reference cannot run it.                     */
typedef enum { MPASB200_PHYSICS_LITERAL = 0, MPASB200_PHYSICS_CORRECTED = 1 } mpasb200_physics_mode_t;

/* ---- dimensions (constants.rg:18-26) ------------------------------------------- */
typedef struct {
  int32_t nCells, nEdges, nVertices;  /* entities in the regions handed to the tasks  */
  int32_t nVertLevels;                /* regions hold nVertLevels+1 levels (main.rg:21-24) */
  int32_t maxEdges;                   /* 10 */
  int32_t maxEdges2;                  /* 20 */
  int32_t vertexDegree;               /* 3  */
  int32_t nAdvCells;                  /* FIFTEEN = 15 */
} MpasDims;

/* ---- configuration (constants.rg:27-69,99-104; rk_timestep.rg:378-382) ----------- */
typedef struct {
  double gravity, rgas, cp, cv, omega, sphere_radius, prandtl;
  double config_epssm, config_smdiv, config_len_disp;
  double config_smagorinsky_coef, config_visc4_2dsmag, config_del4u_div_factor;
  double config_v_mom_eddy_visc2, config_v_theta_eddy_visc2;
  double config_h_mom_eddy_visc4, config_h_theta_eddy_visc4;
  double config_rayleigh_damp_u_timescale_days;
  double config_mpas_cam_coef;
  int32_t config_number_rayleigh_damp_u_levels;
  int32_t config_horiz_mixing;        /* mpasb200_horiz_mixing_t */
  int32_t config_mix_full, config_rayleigh_damp_u;
  int32_t nRelaxZone;
  int32_t number_of_sub_steps;        /* 2, rk_timestep.rg:378 */
  int32_t config_dynamics_split_steps;/* 1, constants.rg:60    */
  int32_t index_policy;               /* mpasb200_index_policy_t */
  int32_t rkarg_policy;               /* mpasb200_rkarg_policy_t */
  int32_t sfc_renumber;               /* 1: renumber cells/edges/vertices along a space-filling curve on the device */
  int32_t device;                     /* CUDA ordinal; -1 = the calling thread's current device */
  int32_t use_graph;                  /* 1: mpasb200_srk3 replays a captured CUDA graph */
  int32_t acoustic_exact;             /* 1: evaluate the acoustic column sweep strictly left-to-right (two kernels, one
                                         thread per column); 0 (default): fused kernel, affine sweep (a few ulp apart) */
  int32_t acoustic_tma;               /* acoustic step form: 3 (default) = lean gather kernel + k_acoustic_lane, a warp-specialised streaming
                                         pipeline whose column sweep runs one column per lane strictly in the reference's order
                                         (bit-identical to the CPU restatement); 2 = gather kernel + cp.async.bulk strips with the affine
                                         two-level sweep (a few ulp of the largest term apart); 1 = one fused kernel, bulk strips, affine
                                         sweep; 0 = fused, plain loads */
  int32_t physics_mode;               /* mpasb200_physics_mode_t; default LITERAL */
  int32_t gather_stage;               /* LABORATORY builds (-DMPASB200_LAB) only, ignored by the shipped library: bit mask selecting the
                                         cp.async-staged forms of k_dt_edge (1), k_acoustic_gather (2), k_dt_theta_flux (4).  Measured
                                         slower than the plain kernels on B200 (profiles/r2_staged_gathers.md); bit-identical results. */
  int32_t config_scalar_advection;    /* 0 (default): atm_srk3 skips scalar transport exactly like the reference (rk_timestep.rg:465);
                                         1: atm_rk_integration_setup saves scalars_old and every RK stage calls atm_advance_scalars
                                         with rk_timestep[rk_step] = dt/3, dt/2, dt (rk_timestep.rg:386-389)              */
  int32_t edge_tiles;                 /* LABORATORY builds (-DMPASB200_LAB) only, ignored by the shipped library: 8 / 16 = k_dt_edge as a
                                         tile kernel (a block owns 8 / 16 consecutive edges and stages the DISTINCT edgesOnEdge columns of
                                         the tile once in shared memory with cp.async.bulk, lists built at upload_mesh).  Bit-identical
                                         results, measured slower than the plain kernel on B200 (profiles/r2_edge_tiles.md). */
  int32_t kernel_forms;               /* bit mask of alternative launch forms with bit-identical results: 1 = k_dt_cellC as two launches
                                         (the w pass, then the theta pass) instead of one fused kernel */
  int32_t reserved0;
  double  config_coef_3rd_order;      /* 0.25, constants.rg:59 */
} MpasConfig;

/* ---- level-0 ("static") region data -------------------------------------------- *
 * Host pointers, each array row-major [entity][slot] exactly like the array-typed
 * region fields (int[maxEdges] ...).  Ids are the RAW stored values; index_policy says
 * how to resolve them.  A null pointer means "never written": the field is all zero
 * (memory-model rule M1 of SURVEY.md 8c).                                           */
typedef struct {
  /* cell_fs */
  const int32_t *nEdgesOnCell;      /* [nCells]                                      */
  const int32_t *edgesOnCell;       /* [nCells][maxEdges]                            */
  const int32_t *verticesOnCell;    /* [nCells][maxEdges]                            */
  const int32_t *kiteForCell;       /* [nCells][maxEdges]   (atm_compute_signs)      */
  const double  *edgesOnCellSign;   /* [nCells][maxEdges]   (atm_compute_signs)      */
  const double  *edgesOnCell_sign;  /* [nCells][maxEdges]   never written upstream   */
  const double  *invAreaCell;       /* [nCells]             never written upstream   */
  const double  *latCell;           /* [nCells]                                      */
  const double  *defc_a, *defc_b;   /* [nCells][maxEdges]   never written upstream   */
  const int32_t *bdyMaskCell;       /* [nCells]             never written upstream   */
  const double  *specZoneMaskCell;  /* [nCells]             never written upstream   */
  const uint8_t *isShared;          /* [nCells]  mark_shared_cells, main.rg:48-52    */
  const uint8_t *inCpr;             /* [nCells]  1 if the cell belongs to `cpr` (private_1[i], main.rg:57-66); null = all */
  /* edge_fs */
  const int32_t *cellsOnEdge;       /* [nEdges][2]  (also cellOne/cellTwo .lo.x)     */
  const int32_t *verticesOnEdge;    /* [nEdges][2]                                   */
  const int32_t *nEdgesOnEdge;      /* [nEdges]                                      */
  const int32_t *edgesOnEdge_ECP;   /* [nEdges][maxEdges2]  the field load_mesh fills */
  const int32_t *edgesOnEdge;       /* [nEdges][maxEdges2]  never written upstream   */
  const double  *weightsOnEdge;     /* [nEdges][maxEdges2]                           */
  const double  *dcEdge, *dvEdge;   /* [nEdges]                                      */
  const double  *invDcEdge, *invDvEdge; /* [nEdges]         never written upstream   */
  const double  *angleEdge, *latEdge;   /* [nEdges]                                  */
  const int32_t *nAdvCellsForEdge;  /* [nEdges]             atm_adv_coef_compression */
  const int32_t *advCellsForEdge;   /* [nEdges][nAdvCells]                           */
  const double  *adv_coefs, *adv_coefs_3rd; /* [nEdges][nAdvCells]                   */
  const double  *meshScalingDel2, *meshScalingDel4; /* [nEdges]                      */
  const double  *specZoneMaskEdge;  /* [nEdges]             never written upstream   */
  /* vertex_fs */
  const int32_t *edgesOnVertex;     /* [nVertices][vertexDegree]                     */
  const double  *edgesOnVertexSign; /* [nVertices][vertexDegree] (atm_compute_signs) */
  const double  *edgesOnVertex_sign;/* [nVertices][vertexDegree] never written upstream */
  const double  *kiteAreasOnVertex; /* [nVertices][vertexDegree]                     */
  const double  *fVertex;           /* [nVertices]                                   */
  const double  *invAreaTriangle;   /* [nVertices]          never written upstream   */
  /* coordinates used only to build the space-filling-curve order (may be null: no renumbering) */
  const double  *xCell, *yCell, *zCell;
  /* launch classes 0..3 (may be null: one class).  Inside the library entities are numbered class by class (then
   * along the curve), so a class is one contiguous range for mpasb200_set_range.  The multi-GPU driver uses
   * cells: 0 = owned, not sent to any rank; 1 = owned, sent; 2 = ghost.  edges: 0 = both cells owned; 1 = the rest. */
  const uint8_t *cellClass;         /* [nCells] */
  const uint8_t *edgeClass;         /* [nEdges] */
  /* init chain on the device (mpasb200_reconstruct_2d); may be null */
  const double  *lonCell;           /* [nCells]                                      */
  const double  *coeffs_reconstruct;/* [nCells][maxEdges][3]  (data_structures.rg: coeffs_reconstruct : double[maxEdges][3]) */
} MpasMeshPtrs;

/* ---- lifecycle ------------------------------------------------------------------ */
void mpasb200_default_config(MpasConfig *cfg);   /* the values of constants.rg */
int  mpasb200_create(const MpasDims *dims, const MpasConfig *cfg, mpasb200_t **out);
int  mpasb200_destroy(mpasb200_t *h);
const char *mpasb200_last_error(const mpasb200_t *h);   /* h may be null: last create error */
int  mpasb200_upload_mesh(mpasb200_t *h, const MpasMeshPtrs *mesh);

/* Strided form for a Legion caller: the static data of the reference sits at level 0 of the 2-D regions (cr[{iCell, 0}].edgesOnCell,
 * mesh_loading.rg:228-344), i.e. one element (or one int[w] / double[w] array, elements contiguous) per x with a BYTE stride
 * between consecutive x -- offsets[0] of legion_accessor_array_2d_raw_rect_ptr.  mpasb200_mesh_member copies one member of
 * MpasMeshPtrs (by its name, e.g. "edgesOnCell") out of such an instance into a dense staging copy owned by the handle;
 * mpasb200_upload_mesh_staged then does what mpasb200_upload_mesh does with the staged members (members never staged are null =
 * "never written").  `base` addresses the element of x = 0, level 0.  isShared / inCpr / cellClass / edgeClass are uint8_t (a
 * Regent bool is one byte).                                                                                                */
int  mpasb200_mesh_member(mpasb200_t *h, const char *member, const void *base, int64_t stride_x);
int  mpasb200_upload_mesh_staged(mpasb200_t *h);

/* ---- region <-> device mirror ---------------------------------------------------- *
 * `base` addresses element (x=0, level=0, slot=0) of the field instance; stride_x /
 * stride_k are BYTE strides in x and level exactly as legion_accessor_array_2d_raw_rect_ptr
 * reports them in offsets[0..1]; array-typed fields have their slots contiguous.
 * Levels 0..nVertLevels are transferred.  Vertical fields use stride_k only.
 * Both calls are synchronous with respect to the host buffer.                          */
int  mpasb200_upload_field(mpasb200_t *h, int field, const void *base, int64_t stride_x, int64_t stride_k);
int  mpasb200_download_field(mpasb200_t *h, int field, void *base, int64_t stride_x, int64_t stride_k);
int  mpasb200_zero_field(mpasb200_t *h, int field);
int  mpasb200_sync(mpasb200_t *h);
/* Pipelined variants for contiguous, page-locked host arrays ([n][nVertLevels+1][slots]): the H2D / D2H copies run on the
 * library's own copy streams (both PCIe directions and the compute stream overlap), ordered against the tasks by events:
 * an upload is visible to every task enqueued after it, a download sees every task enqueued before it.  The host array
 * may be reused (upload) or read (download) after mpasb200_transfer_wait().  Each field gets its own device staging
 * buffer per direction on first use (counted in mpasb200_device_bytes).                                            */
int  mpasb200_upload_field_async(mpasb200_t *h, int field, const void *base);
int  mpasb200_download_field_async(mpasb200_t *h, int field, void *base);
int  mpasb200_transfer_wait(mpasb200_t *h);

/* ---- one entry per hot-path task: scalars only -------------------------------------- */
/* atm_rk_integration_setup            dynamics_tasks.rg:747-778   */
int  mpasb200_rk_integration_setup(mpasb200_t *h);
/* atm_compute_moist_coefficients      dynamics_tasks.rg:460-502   */
int  mpasb200_compute_moist_coefficients(mpasb200_t *h);
/* atm_compute_vert_imp_coefs          dynamics_tasks.rg:513-592   */
int  mpasb200_compute_vert_imp_coefs(mpasb200_t *h, double dts);
/* atm_compute_dyn_tend(_work)         dynamics_tasks.rg:814-1500  */
int  mpasb200_compute_dyn_tend(mpasb200_t *h, int rk_step, double dt, int config_horiz_mixing,
                               double config_mpas_cam_coef, int config_mix_full, int config_rayleigh_damp_u);
/* atm_set_smlstep_pert_variables      dynamics_tasks.rg:1503-1538 */
int  mpasb200_set_smlstep_pert_variables(mpasb200_t *h);
/* atm_advance_acoustic_step           dynamics_tasks.rg:1546-1719 */
int  mpasb200_advance_acoustic_step(mpasb200_t *h, double dts, int small_step);
/* atm_divergence_damping_3d           dynamics_tasks.rg:1726-1763 */
int  mpasb200_divergence_damping_3d(mpasb200_t *h, double dts);
/* atm_recover_large_step_variables    dynamics_tasks.rg:1766-1887 (call commented out at rk_timestep.rg:460) */
int  mpasb200_recover_large_step_variables(mpasb200_t *h, int ns, int rk_step, double dt);
/* atm_compute_solve_diagnostics       dynamics_tasks.rg:328-454   */
int  mpasb200_compute_solve_diagnostics(mpasb200_t *h, int hollingsworth, int rk_step);
/* atm_advance_scalars: NOT in the reference (its call sites are "SKIPPING" comments, rk_timestep.rg:465,485; the storage is
 * cell_fs.scalars, data_structures.rg:36).  Implements atm_advance_scalars_work of MPAS-Atmosphere v7.0 (non-monotonic
 * transport, no physics tendency): horizontal flux of every scalar through every edge with the advection stencil of
 * atm_adv_coef_compression and the time-averaged mass flux ruAvg, cell-centric flux divergence over edgesOnCell with
 * edgesOnCellSign, 3rd-order vertical flux with wwAvg (flux3, dynamics_tasks.rg:786-789; 2nd order at the two end levels),
 * scalars = (scalars_old * rho_zz_old_split + dt * (tend - rdzw * d(wdtn))) / rho_zz.  Parity is against the oracle's
 * restatement of that routine (unpinned: the reference cannot run it).                                                    */
int  mpasb200_advance_scalars(mpasb200_t *h, double dt, int rk_step);
/* atm_rk_dynamics_substep_finish      dynamics_tasks.rg:1951-2007 */
int  mpasb200_rk_dynamics_substep_finish(mpasb200_t *h, int dynamics_substep, int dynamics_split);

/* ---- init chain on the device (SURVEY.md 8f rank 3): the two one-time tasks of atm_core_init that are stencils over 3-D fields ---- */
/* atm_init_coupled_diagnostics        dynamics_tasks.rg:651-725  (rho_zz /= zz; ru; rw from w and ru; rho_p, rtheta_base, rtheta_p,
 *                                     exner, exner_base, pressure_p, pressure_base; levels 0..nVertLevels-1)                        */
int  mpasb200_init_coupled_diagnostics(mpasb200_t *h);
/* mpas_reconstruct_2d                 dynamics_tasks.rg:1894-1948 (uReconstructX/Y/Z from u with coeffs_reconstruct, then
 *                                     uReconstructZonal / uReconstructMeridional; also MPAS's end-of-step call, rk_timestep.rg:487) */
int  mpasb200_reconstruct_2d(mpasb200_t *h, int includeHalos, int on_a_sphere);

/* ---- the mesh-only producers of atm_core_init on the device (SURVEY.md 8f rank 3) ------------------------------------------- *
 * atm_compute_signs (dynamics_tasks.rg:46-130), atm_adv_coef_compression (:133-269) and atm_couple_coef_3rd_order (:303-325) run
 * once, before the first step, on connectivity alone.  Their inputs are the RAW stored ids of the static region fields in the
 * caller's numbering (host pointers, row-major [entity][slot] like MpasMeshPtrs; index_policy of the handle resolves them), their
 * outputs are exactly the MpasMeshPtrs members / 3-D fields the hot path consumes.  The two list builders may be called before
 * mpasb200_upload_mesh (their outputs feed it); the 3-D part of atm_compute_signs (zb_cell, zb3_cell from the edge fields zb, zb3)
 * works on the device mirror and therefore comes after mpasb200_upload_mesh + the upload of zb, zb3.                             */
typedef struct {
  const int32_t *nEdgesOnCell;      /* [nCells]                    */
  const int32_t *edgesOnCell;       /* [nCells][maxEdges]          */
  const int32_t *verticesOnCell;    /* [nCells][maxEdges]          */
  const int32_t *cellsOnCell;       /* [nCells][maxEdges]          */
  const int32_t *cellsOnEdge;       /* [nEdges][2]                 */
  const int32_t *verticesOnEdge;    /* [nEdges][2]                 */
  const int32_t *cellsOnVertex;     /* [nVertices][vertexDegree]   */
  const int32_t *edgesOnVertex;     /* [nVertices][vertexDegree]   */
  const double  *dcEdge, *dvEdge;   /* [nEdges]                    */
  const double  *deriv_two;         /* [nEdges][2*FIFTEEN]; null = never written upstream = all zero (rule M1) */
} MpasInitMesh;
/* atm_compute_signs, level-0 part     dynamics_tasks.rg:60-86, 113-129: edgesOnVertexSign [nVertices][vertexDegree],
 *                                     edgesOnCellSign [nCells][maxEdges], kiteForCell [nCells][maxEdges] (host, caller's numbering) */
int  mpasb200_compute_signs(mpasb200_t *h, const MpasInitMesh *m, double *edgesOnVertexSign, double *edgesOnCellSign, int32_t *kiteForCell);
/* atm_compute_signs, 3-D part         dynamics_tasks.rg:88-110: zb_cell, zb3_cell from zb, zb3 (levels 0..nVertLevels) */
int  mpasb200_compute_zb_cell(mpasb200_t *h);
/* atm_adv_coef_compression            dynamics_tasks.rg:133-269: nAdvCellsForEdge [nEdges], advCellsForEdge (raw ids) / adv_coefs /
 *                                     adv_coefs_3rd [nEdges][FIFTEEN]; quirks kept (the list index n, the cap at maxEdges-1)       */
int  mpasb200_adv_coef_compression(mpasb200_t *h, const MpasInitMesh *m, int32_t *nAdvCellsForEdge, int32_t *advCellsForEdge,
                                   double *adv_coefs, double *adv_coefs_3rd);
/* atm_couple_coef_3rd_order           dynamics_tasks.rg:303-325: adv_coefs_3rd [nEdges][FIFTEEN] (host array, scaled on the device,
 *                                     may be null) *= coef; zb3_cell *= coef at LEVEL 0 only (the device field; skipped before
 *                                     mpasb200_upload_mesh)                                                                        */
int  mpasb200_couple_coef_3rd_order(mpasb200_t *h, double config_coef_3rd_order, double *adv_coefs_3rd);

/* atm_compute_mesh_scaling            dynamics_tasks.rg:595-646: meshScalingDel2 / meshScalingDel4 [nEdges] (host arrays, caller's numbering)
 *                                     from meshDensity [nCells] read through cellsOnEdge (m->cellsOnEdge, raw ids); 1.0 when
 *                                     config_h_ScaleWithMesh is false.  The regional-relaxation factors are not on the hot path.   */
int  mpasb200_compute_mesh_scaling(mpasb200_t *h, const MpasInitMesh *m, const double *meshDensity, int config_h_ScaleWithMesh,
                                   double *meshScalingDel2, double *meshScalingDel4);
/* atm_compute_damping_coefs           dynamics_tasks.rg:274-300: dss from zgrid (device fields) and meshDensity [nCells] (host, caller's
 *                                     numbering); levels 0..nVertLevels-1; after mpasb200_upload_mesh.                                */
int  mpasb200_compute_damping_coefs(mpasb200_t *h, const double *meshDensity, double config_zd, double config_xnutr);
/* init_atm_case_jw                    vertical_init/init_atm_cases.rg:24-743 -- the Jablonowski-Williamson baroclinic-wave initial
 * state on the device, CORRECTED reading (the reference text indexes regions with swapped, out-of-range (level, cell) pairs and cannot
 * be restated literally; this is the formula-by-formula equivalent of the host generator mpas_regent_b200/init_jw.py, dry case, parity
 * against it at 1e-12).  After mpasb200_upload_mesh.  Inputs: host arrays in the caller's numbering, geometry already scaled to the
 * sphere (init_atm_cases.rg:87-111).  Writes the vertical fields rdzw, rdzu, fzm, fzp, cf1, cf2, cf3 and the 3-D fields zgrid, zz,
 * zxu, rho_base, theta_base, pressure_p, rho_p, exner, theta_m, rtheta_p, rho_zz, u, ru, zb, zb3 (= 0), rw, w.                       */
typedef struct {
  const double *latCell, *areaCell;   /* [nCells]    */
  const double *latVertex;            /* [nVertices] */
  int32_t n_lat_table;                /* rows of the (z, lat) section the columns are balanced on; 0 = 4097 */
} MpasJwGeometry;
int  mpasb200_init_atm_case_jw(mpasb200_t *h, const MpasJwGeometry *g);

/* ---- the driver: atm_srk3 / atm_timestep  rk_timestep.rg:361-519 ------------------------- *
 * Replays the reference's call sequence on the device (control flow + scalars only).    */
int  mpasb200_srk3(mpasb200_t *h, double dt);
int  mpasb200_timestep(mpasb200_t *h, double dt);

/* ---- summarize_timestep  rk_timestep.rg:29-359 --------------------------------------------------- *
 * The reference's per-step sanity scan (global min / max of a field with the place they occur, NaN scan; every branch
 * is disabled by configuration there) as a device reduction, extended by an order-independent 64-bit checksum of the
 * bit patterns so that runs on 1 and N GPUs can be compared bit for bit without moving the fields.
 * The scan covers entities [0, n_first) of the caller's numbering (the owned entities of a partition come first) and
 * levels [0, nlevels).  min / max ignore NaN (a comparison with NaN is false, :64); the place is the first one in
 * (id, level) order, id = global id if mpasb200_set_global_ids was called for the entity type, else the caller's index.
 * checksum = sum mod 2^64 over the scanned points of mix64(bits(v) + 0x9e3779b97f4a7c15 * (id * nlevels + level + 1)),
 * mix64 = the splitmix64 finaliser, every NaN counted as 0x7ff8000000000000.  Synchronous (host-visible point).       */
typedef struct {
  double   min, max;                 /* +inf / -inf when nothing compares */
  int64_t  min_index, max_index;     /* -1 when nothing compares */
  int32_t  min_level, max_level;
  int64_t  n_nan, n_inf, count;
  uint64_t checksum;
} MpasFieldSummary;
int  mpasb200_set_global_ids(mpasb200_t *h, int entity, const int32_t *global_id, int32_t n);   /* null: back to identity */
int  mpasb200_summarize_field(mpasb200_t *h, int field, int32_t n_first, int32_t nlevels, MpasFieldSummary *out);

/* ---- exact global integrals (summarize_timestep's scan extended by a sum) ------------------------------------------ *
 * I = the EXACT sum over entities i < n_first of the caller's numbering and levels k < nlevels of
 *       p(i,k) = ((a[i,k] * b[i,k]) * wh[i]) * wv[k]
 * where every product is one IEEE multiply rounded to nearest, in exactly that order; b (field_b = -1), wh (weight_id = -1)
 * and wv (null) default to 1.  NaN, +Inf and -Inf products are counted and left out of the sum.  The finite products are
 * added into a fixed-point accumulator without rounding, so the result does not depend on the block schedule, the
 * renumbering or the partition: the integrals of the owned entities of N ranks, merged with mpasb200_integral_merge, have
 * the same bits at every N, and a Legion caller may use the merge as a reduction operator over partitions.
 *
 * Representation of MpasIntegral: the sum is   sum_{j=0}^{67} limb[j] * 2^(32*j - 1088)   exactly, as integers.  That
 * covers 2^-1088 .. 2^1088, enough for any sum of up to 2^40 doubles, subnormals included (a double is a multiple of
 * 2^-1074 below 2^1024).  Any int64 limbs form a valid accumulator.  Every result of the library is in canonical form:
 * limbs 0..66 in [0, 2^32) and limb 67 signed, so two equal sums have equal limbs.  count = the products taken
 * (n_first * nlevels, non-finite ones included); n_nan, n_pinf, n_ninf = the products left out.
 *
 * register_weights uploads wh once: w[n] in the caller's numbering, n = the entity count of the handle.
 * integrate is synchronous (host-visible point) and refused during graph capture.  wv is a host array [nlevels].  It
 * returns MPASB200_EINVAL for an unknown field, slot or weight id, a vertical field, field_b or the weights on another
 * entity type than field_a, and n_first outside [0, count] or nlevels outside [1, nVertLevels+1].
 * integral_merge and integral_value need no handle and no GPU.  merge: acc += x, exact, associative and commutative
 * (MPASB200_EINVAL only if the sum leaves the range above).  value: the sum rounded once, to nearest with ties to even;
 * +-Inf on overflow, +0.0 for an exact zero.  Any NaN, or both signs of infinity, gives NaN; one sign of infinity alone
 * gives that infinity.                                                                                                  */
#define MPASB200_INTEGRAL_LIMBS 68
#define MPASB200_INTEGRAL_BIAS  1088
typedef struct {
  int64_t limb[MPASB200_INTEGRAL_LIMBS];
  int64_t count, n_nan, n_pinf, n_ninf;
} MpasIntegral;
int  mpasb200_register_weights(mpasb200_t *h, int entity, const double *w, int32_t n, int32_t *weight_id);
int  mpasb200_integrate(mpasb200_t *h, int field_a, int slot_a, int field_b, int slot_b, int weight_id, const double *wv,
                        int32_t n_first, int32_t nlevels, MpasIntegral *out);
int  mpasb200_integral_merge(MpasIntegral *acc, const MpasIntegral *x);
double mpasb200_integral_value(const MpasIntegral *x);

/* ---- halo exchange building blocks (one process per GPU; the wire is the host's job) ------ *
 * Lists are LOCAL entity indices in the caller's (un-renumbered) numbering.  pack gathers
 * `n` columns x `nfields` fields x (nVertLevels+1) levels into the contiguous device
 * buffer `d_buf` laid out [i][field][level] (one contiguous row per listed entity, so a list that
 * concatenates several peers yields one contiguous slice per peer); unpack scatters the same layout back.  An array-typed
 * field (scalars : double[8]) occupies one `field` entry per slot, in slot order.
 * A list is registered once and referred to by the returned id.                         */
int  mpasb200_register_list(mpasb200_t *h, int entity, const int32_t *idx, int32_t n, int32_t *list_id);
int  mpasb200_pack(mpasb200_t *h, int list_id, const int32_t *fields, int32_t nfields, void *d_buf);
int  mpasb200_unpack(mpasb200_t *h, int list_id, const int32_t *fields, int32_t nfields, const void *d_buf);
/* Restrict compute to a sub-range of entities (interior / boundary split, so a halo exchange can overlap interior
 * compute): mpasb200_advance_acoustic_step runs on cells [begin,end) and mpasb200_divergence_damping_3d on edges
 * [begin,end) of the library's internal order (with physics_mode CORRECTED the acoustic edge update follows the edge range);
 * mpasb200_class_range gives the range of a launch class of MpasMeshPtrs.  begin < 0 restores the whole entity.  All
 * other tasks always run on everything.                                                                              */
int  mpasb200_class_range(mpasb200_t *h, int entity, int cls, int32_t *begin, int32_t *end);
int  mpasb200_set_range(mpasb200_t *h, int entity, int32_t begin, int32_t end);
int  mpasb200_set_stream(mpasb200_t *h, void *cuda_stream);  /* null = the handle's own stream */
int  mpasb200_set_use_graph(mpasb200_t *h, int on);          /* MpasConfig.use_graph after creation */

/* ---- the distributed step: one process (or thread) per GPU, the whole exchange schedule inside the library ---------------- *
 * Replaces what the reference computes but never runs: partition_regions (mesh_loading.rg:399-483) hands every rank its
 * [owned | ghost ring 1 | ghost ring 2] cells; mpasb200_srk3_dist is atm_srk3 (rk_timestep.rg:361-500) on that local mesh
 * with the halo exchanges the stencils need, issued by the library itself: k_pack -> ncclSend/ncclRecv (one ncclGroup per
 * exchange, NVLink) -> k_unpack on a communication stream owned by the handle, ordered against the compute stream by events.
 * When the mesh was uploaded with launch classes (MpasMeshPtrs.cellClass/edgeClass) every acoustic-loop exchange is hidden
 * under interior compute (sent cells first, interior cells and interior edges under the exchange, edges next to ghosts after
 * it; ghost cells are never advanced) and the exchanges after atm_compute_solve_diagnostics of stages 0 and 2 travel under the
 * column work that follows.  Owned results are bit-identical to the single-partition run.
 *   unique_id : 128 bytes from mpasb200_dist_unique_id on ONE rank, distributed by the host's own channel (Legion future,
 *               MPI_Bcast, torch.distributed ...).  NCCL is dlopen'ed ("libnccl.so.2") on first use: single-GPU users need none.
 *   halo      : per entity type, peers in any order; lists are LOCAL indices in the caller's numbering; for a pair of ranks
 *               both sides list the same global entities in the same order (partition.build_halo_lists).                    */
enum { MPASB200_X_ACOUSTIC_FIRST = 0, MPASB200_X_ACOUSTIC, MPASB200_X_DIAG, MPASB200_X_RECOVER, MPASB200_X_SCALARS, MPASB200_X_COUNT };
int  mpasb200_dist_unique_id(void *id128);
int  mpasb200_dist_init(mpasb200_t *h, int rank, int world, const void *id128);
int  mpasb200_dist_set_halo(mpasb200_t *h, int entity,
                            int32_t n_send_peers, const int32_t *send_peers, const int32_t *send_off /*[n+1]*/, const int32_t *send_idx,
                            int32_t n_recv_peers, const int32_t *recv_peers, const int32_t *recv_off /*[n+1]*/, const int32_t *recv_idx);
int  mpasb200_dist_exchange(mpasb200_t *h, int kind);     /* one exchange, complete on return of the stream order (init, tests) */
int  mpasb200_srk3_dist(mpasb200_t *h, double dt);
int  mpasb200_dist_flush(mpasb200_t *h);                  /* joins an exchange still travelling on the communication stream   */

/* ---- introspection --------------------------------------------------------------------- */
int64_t mpasb200_launch_count(const mpasb200_t *h);   /* kernels launched so far by this handle */
int64_t mpasb200_device_bytes(const mpasb200_t *h);   /* bytes of HBM held by the mirror */
int  mpasb200_field_info(int field, int *entity, int *slots, const char **name);
int  mpasb200_field_by_name(const char *name);        /* -1 if unknown */
/* Per-task CUDA-event timing: when enabled every task entry is bracketed by events on the
 * handle's stream; task_ms returns the accumulated milliseconds and call count per entry. */
int  mpasb200_enable_timing(mpasb200_t *h, int on);
int  mpasb200_task_time(mpasb200_t *h, int task, double *ms, int64_t *calls, const char **name);
int  mpasb200_reset_timing(mpasb200_t *h);
/* Per-KERNEL CUDA-event timing: every launch is bracketed by an event pair on the handle's stream.
 * kernel_time(idx) walks the table (returns MPASB200_EINVAL past the end).                       */
int  mpasb200_enable_kernel_timing(mpasb200_t *h, int on);
int  mpasb200_reset_kernel_timing(mpasb200_t *h);
int  mpasb200_kernel_time(mpasb200_t *h, int idx, const char **name, double *ms, int64_t *launches);
/* enable_kernel_timing(h, 2) additionally keeps a TIMELINE: start and end of every launch (and of every NCCL send/recv group) in ms since
 * the call, with the stream it ran on (0 = compute, 1 = the handle's communication stream) -- what shows the exchanges travelling
 * under interior compute (profiles/r2_timeline_2gpu.md).  timeline_entry(idx) walks it (MPASB200_EINVAL past the end).          */
int  mpasb200_timeline_entry(mpasb200_t *h, int idx, const char **name, double *t0_ms, double *t1_ms, int *stream);
enum { MPASB200_T_SETUP = 0, MPASB200_T_MOIST, MPASB200_T_VERT_IMP, MPASB200_T_DYN_TEND, MPASB200_T_SMLSTEP,
       MPASB200_T_ACOUSTIC, MPASB200_T_DIVDAMP, MPASB200_T_RECOVER, MPASB200_T_DIAG, MPASB200_T_FINISH, MPASB200_T_SCALARS, MPASB200_T_COUNT };

#ifdef __cplusplus
}
#endif
#endif /* MPAS_B200_H */
