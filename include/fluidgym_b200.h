/*
 * fluidgym_b200 -- C ABI of the batched B200 (sm_100a) PISO solver step.
 *
 * This is the drop-in boundary for the fluid-solver step of FluidGym.  Each entry point names the
 * reference interface it replaces (paths relative to /root/reference/src/fluidgym/):
 *   BIND.cpp  = simulation/extensions/PISOtorch.cpp        (pybind11 module `PISOtorch`)
 *   K.cu      = simulation/extensions/PISO_multiblock_cuda_kernel.cu
 *   SIM.py    = simulation/pict/PISOtorch_simulation.py
 *   DIFF.py   = simulation/pict/PISOtorch_diff.py          (autograd Functions, linear-solve wrapper)
 *   FGSIM.py  = simulation/simulation.py                   (FluidGym's Simulation subclass: single_step)
 *   DS.cpp    = simulation/extensions/domain_structs.cpp   (Domain / Block / boundaries)
 *   CG.cu     = simulation/extensions/cg_solver_kernel.cu,  BICG.cu = simulation/extensions/bicgstab_solver_kernel.cu
 *   CYL.py    = envs/cylinder/cylinder_env_base.py
 *
 * Differences by design: the reference ops work on ONE mutable Domain object (batch size 1,
 * DS.cpp:1136) and synchronise the device around every launch; here every op advances B independent
 * environments that share one geometry, takes raw device pointers + a CUDA stream, never synchronises
 * and never allocates.  All arrays are float32 / int32, structure-of-arrays, environment-major:
 *   u    [B][2][N]    cell velocity            (Block.velocity, all blocks concatenated)
 *   p    [B][N]       cell pressure            (Block.pressure == Domain.pressureResult)
 *   bvel [B][2][NB]   Dirichlet boundary velocity of every fixed-boundary face (FixedBoundary.velocity)
 * plus per-environment scalars dt[B] (float) and active[B] (int32: 0 = skip this environment).
 *
 * Error handling: every function returns 0 on success, a negative FGB_E_* code otherwise;
 * fgb_last_error() returns a static message for the calling thread.  No exceptions cross the ABI.
 * There is NO CPU fallback: without a CUDA device every launch returns FGB_E_CUDA.
 */
#ifndef FLUIDGYM_B200_H
#define FLUIDGYM_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FGB_OK 0
#define FGB_E_ARG -1
#define FGB_E_CUDA -2
#define FGB_E_WORKSPACE -3

typedef void *fgb_stream_t; /* cudaStream_t */

/* Geometry tables of one domain, produced on the host by fluidgym_b200.domain.CompiledDomain and
 * uploaded by the caller.  ALL pointers are DEVICE pointers owned by the caller and must outlive the
 * handle.  Replaces the packed DomainGPU/BlockGPU/BoundaryGPU atlas (DSG.h:160-397, DS.cpp:3055-3282). */
typedef struct fgb_tables {
    int32_t N, NB, K_no, K_nob;
    float viscosity;
    const int32_t *nbr;     /* [4][N]   neighbour cell across face f, or -1-j for boundary face j      */
    const int8_t *fl_comp;  /* [4][N]   bit0: contravariant component of the neighbour, bit1: negate   */
    const float *minv;      /* [4][N]   M^-1 row-major                                                  */
    const float *det;       /* [N]                                                                      */
    const float *Cd;        /* [5][N]   constant (diffusive + non-orthogonal) part of C, before /det    */
    const float *Wp;        /* [25][N]  P_e = sum_j Wp[5e+j] * (1/A)_j, j=0 self, 1..4 face neighbours  */
    const int32_t *no_idx;  /* [K_no][N] deferred non-orthogonal terms: cell index                      */
    const int8_t *no_face;  /* [K_no][N] face whose neighbour 1/A enters the pressure weight           */
    const float *no_gP;     /* [K_no][N]                                                                */
    const float *no_gN;     /* [K_no][N] pressure weight = gP*(1/A)_P + gN*(1/A)_nbr(face)              */
    const float *no_wv;     /* [K_no][N] velocity weight (viscosity folded in)                          */
    const int32_t *nob_idx; /* [K_nob][N] boundary-face index                                           */
    const float *nob_w;     /* [K_nob][N] weight of that boundary velocity in the velocity correction  */
    const float *b_minv;    /* [4][NB]  boundary-face M^-1                                              */
    const float *b_det;     /* [NB]                                                                     */
    const float *b_alpha;   /* [NB]     det*|M^-1 row(axis)|^2 of the boundary face                     */
    const int32_t *b_cell;  /* [NB]     cell adjacent to the boundary face                              */
    const int8_t *b_face;   /* [NB]     face direction 0..3                                             */
    const int8_t *b_out;    /* [NB]     1 = advective-outflow face (SIM.py:228-393), may be NULL        */
    /* passive scalar (temperature) transport, NULL / 0 when the domain has none */
    float scalar_viscosity; /*          scalar diffusivity (Domain.setScalarViscosity)                     */
    const float *Cd_s;      /* [5][N]   constant part of the scalar transport matrix, before /det          */
    const int8_t *sb_neumann; /* [NB]   scalar boundary condition type: 0 Dirichlet, 1 Neumann             */
    const int8_t *rev;      /* [4][N]   face of the neighbour nbr[f] that points back to this cell (adjoint /
                                        transposed solves), -1 on boundary faces                        */
    /* optional halo plan of the on-chip Krylov kernels (cg_impl 6), built for ONE cluster size cg_cs by
     * fluidgym_b200/solver.py::halo_plan: every CTA of a cluster owns ceil(N/cg_cs) consecutive cells, keeps the
     * exposed vector of its own cells in shared-memory slots [0, cells) and receives the remote cells its stencils
     * touch into slots [pad, pad + n_halo).  NULL = not available (kernels gather through DSMEM instead). */
    const int32_t *cg_slot; /* [4][N]   shared-memory slot (in floats) holding the neighbour across face f      */
    const int32_t *cg_exp;  /* [cg_cs][cg_emax][2]  export list of each CTA: {own slot | dest rank << 24, dest slot} */
    const int32_t *cg_cnt;  /* [cg_cs][2]  {exports, halo cells} of each CTA                                     */
    int32_t cg_cs, cg_emax, cg_hmax, cg_pad;
    /* optional strip plan of the register-blocked on-chip CG (cg_impl 11), built by fluidgym_b200/strip_plan.py for ONE
     * cluster size st_cs: the cells of every CTA are laid out as padded 2-D arrays so that the stencil neighbours of
     * shared-memory slot s are s-1, s+1, s-S, s+S; a thread owns st_cpt consecutive rows of one column; cells that are
     * not array-adjacent (block connections, periodic wrap, cuts between CTAs) are GHOST slots: replicas that receive the
     * residual of the mirrored cell every iteration (owner in another CTA) or mirror slots the owner writes itself (same
     * CTA).  NULL = not available. */
    const int32_t *st_thread; /* [st_cs][st_T][8]  {first slot, row stride S, face map (2 bits per W,E,S,N), remote exports
                                 (offset | count << 16), 0, first index in the receive buffer, remote ghost rows (bit k),
                                 local ghost rows (bit k)}                                               */
    const int32_t *st_cell;   /* [st_cs][st_T][st_cpt]  cell id of the thread's k-th row, -1 dead, -2-g ghost of cell g      */
    const int32_t *st_rexp;   /* [st_cs][st_remax][2]  {k | destination rank << 8, index in the destination's receive buffer} */
    const int32_t *st_lexp;   /* [st_cs][st_lemax][2]  {owner's slot, mirror slot} copy list of the local ghosts              */
    const int32_t *st_cnt;    /* [st_cs][4]  {remote ghosts, remote exports, local exports, 0} of each CTA                    */
    int32_t st_cs, st_T, st_cpt, st_slots, st_remax, st_lemax, st_gmax;
} fgb_tables;

/* Passive scalar + buoyancy coupling of one batch (RBC: temperature; rbc_env_base.py:190-304).  With the
 * reference's ordering: the scalar is advected first with the old velocity (SIM.py:1471-1644), then
 * the velocity source (0, beta*T_new) is built ("PRE_VELOCITY_SETUP" hook) and used by the predictor / HbyA. */
typedef struct fgb_scalar {
    float *T;             /* [B][N]   scalar field, updated in place                                   */
    const float *sbval;   /* [B][NB]  boundary values (FixedBoundary.passiveScalar)                    */
    float beta;           /*          buoyancy factor                                                    */
    float *src;           /* [B][2][N] velocity-source buffer written by the step                       */
} fgb_scalar;

typedef struct fgb_batch fgb_batch; /* opaque: tables + workspace carving for B environments */

/* Solver options (Simulation ctor arguments, SIM.py:489-1037; defaults of CylinderEnvBase, CYL.py:303-332) */
typedef struct fgb_options {
    int32_t corrector_steps;        /* 2 */
    int32_t adv_nonortho_steps;     /* 1 */
    int32_t p_nonortho_steps;       /* 1 */
    int32_t nonortho;               /* 1: flags CENTER_MATRIX|DIRECT_MATRIX|DIAGONAL_RHS, 0: orthogonal */
    float adv_tol, p_tol;           /* 1e-5, 1e-5 : ||r||_2/sqrt(N) absolute (SIM.py:1096-1098)          */
    int32_t max_iter;               /* 5000 */
    int32_t cg_impl;                /* pressure CG (and whether the advection BiCGStab runs on chip: 0 = never).
                                       Every on-chip variant takes the smallest cluster that holds the grid and falls
                                       through to 0 when none does (the pressure solve; BiCGStab likewise), except:
                                       11 / 13 fail (FGB_E_ARG) on a grid smaller than the best-iterate scratch
                                       (cluster x threads x rows per thread > 12 N), 12 fails on a strip plan it
                                       has no instantiation for (1 or 16 CTAs).
                                       0: one CTA per environment, vectors in global memory
                                       1: thread-block cluster per environment, vectors on chip,
                                          textbook recurrence (3 cluster barriers / iteration)
                                       2: as 1 with A*p from the recurrence Ap <- A*r + beta*Ap
                                          (mathematically identical, 2 cluster barriers / iteration)
                                       3: as 1 without cluster barriers: st.async + mbarrier transactions
                                          for the reductions, remote mbarrier arrive for the p hand-shake
                                       4: as 3 with x/r/p/neighbour table in shared memory, 2x cells per CTA
                                       5: as 4 with two co-resident CTAs per SM
                                       6: as 3 with PUSHED halos (tables.cg_slot/cg_exp): after updating the
                                          search direction every CTA st.async-es the cells its neighbours need into
                                          their shared memory, all stencil gathers become plain ld.shared
                                          (default of BatchedPISO, RBC2D and Airfoil2D)
                                       7: as 6 with 256-thread CTAs and twice the cells per thread
                                       8: as 6 with 256-thread CTAs of 1792 cells, two co-resident CTAs per SM
                                       11: register-blocked strip layout (tables.st_*): TWO cross-CTA exchanges per
                                          iteration instead of three (the residual of the ghost cells travels with the
                                          partial sums of <r,r>, ghost replicas update p and x themselves), no per-cell
                                          neighbour addresses, north/south neighbours in registers (default of the
                                          cylinder environments; 6 where the domain has no strip plan)
                                       12: as 11 with two environments per cluster (k_cg_strip2, 2 / 4 / 8-CTA plans
                                          only; any other plan is an error)
                                       13: as 11 with the eager bookkeeping order (bit-identical to 11)          */
} fgb_options;

/* message of the last failed fgb_* call of the calling thread (the analogue of the reference's TORCH_CHECK text, BIND.cpp) */
const char *fgb_last_error(void);
/* ABI version of this header (1) */
int fgb_version(void);

/* bytes of device workspace fgb_batch_create needs for B environments */
size_t fgb_workspace_bytes(const fgb_tables *t, int32_t B);
/* workspace: device memory (>= fgb_workspace_bytes, 256-byte aligned) owned by the caller */
int fgb_batch_create(const fgb_tables *t, int32_t B, void *workspace, size_t workspace_bytes,
                     const fgb_options *opt, fgb_batch **out);
void fgb_batch_destroy(fgb_batch *b);
int fgb_batch_set_options(fgb_batch *b, const fgb_options *opt);
/* Environment groups, 1 (default) .. 8: fgb_piso_substep / fgb_sim_step run contiguous groups of the batch on streams of their
 * own (forked from and joined with the caller's stream), so that one group's assembly kernels and the ragged end of its Krylov
 * launches overlap the other groups' solves.  Results are bit-identical to groups = 1: environments are independent
 * (the reference runs one OS process per environment, envs/parallel_env.py:162-175).  Also settable with FGB_GROUPS. */
int fgb_batch_set_groups(fgb_batch *b, int32_t groups);

/* Device pointer of a named intermediate inside the workspace (for parity tests and autograd glue):
 * "Coff"[B][4][N] "A"[B][N] "rhs"[B][2][N] "ures"[B][2][N] "Poff"[B][4][N] "Pdiag"[B][N]
 * "hbya"[B][2][N] "div"[B][N] "pres"[B][N] "iters"[B][8] int32 "resid"[B][8] "dt"[B] "active"[B] int32
 * "iter_total"[B][2] uint64 (cg, bicgstab) "remaining"[B] double "nsub"[B] int32 "maxvel"[B] "fluxbal"[B] */
void *fgb_batch_buffer(fgb_batch *b, const char *name);

/* ---- individual native ops (each replaces one PISOtorch free function) ------------------------- */
/* SetupAdvectionMatrix + SetupAdvectionVelocity (BIND.cpp:518-579, K.cu:3617-3880, 4296-4400):
 * C off-diagonals, A = diag(C), predictor right-hand side.  ures = velocity used in the deferred
 * non-orthogonal term (u itself on the first non-orthogonal step). */
int fgb_setup_advection(fgb_batch *b, const float *u, const float *ures, const float *bvel, const float *src,
                        const float *dt, const int32_t *active, fgb_stream_t s);
/* SolveLinear(C, velocityRHS, BiCG) (K.cu:7085-7118, BICG.cu:64-411) for both components; x=ures */
int fgb_solve_advection(fgb_batch *b, int zero_init, const int32_t *active, fgb_stream_t s);
/* SetupPressureMatrix (K.cu:4812-4978) */
int fgb_setup_pressure_matrix(fgb_batch *b, const int32_t *active, fgb_stream_t s);
/* SetupPressureRHS / SetupPressureRHSdiv (K.cu:5136-5255, 5389-5492); p_prev = pressureResult used
 * by the deferred non-orthogonal correction; with_hbya=0 rebuilds only the divergence */
int fgb_setup_pressure_rhs(fgb_batch *b, const float *u, const float *bvel, const float *src, const float *p_prev,
                           const float *dt, int with_hbya, const int32_t *active, fgb_stream_t s);
/* SolveLinear(P, pressureRHSdiv, CG, residual reset 100, best result) + mean removal (CG.cu:130-471,
 * SIM.py:1908-1925). p_out may alias p_prev. */
int fgb_solve_pressure(fgb_batch *b, float *p_out, int zero_init, int reset_steps, int max_iter,
                       const int32_t *active, fgb_stream_t s);
/* CorrectVelocity version 1 "FD" (K.cu:816-849, 5962-5995): u_out = HbyA - 1/A * M^-T grad p */
int fgb_correct_velocity(fgb_batch *b, const float *p, float *u_out, const int32_t *active, fgb_stream_t s);

/* ---- fused driver level (replaces the python loops of SIM.py) ----------------------------------- */
/* Simulation._PISO_split_step(iterations=1) (SIM.py:1431-2002): one PISO substep of dt[e] for every
 * active environment; u, p updated in place. */
int fgb_piso_substep(fgb_batch *b, float *u, float *p, const float *bvel, const float *src, const float *dt,
                     const int32_t *active, const fgb_scalar *sc /* may be NULL */, fgb_stream_t s);
/* Simulation.make_divergence_free (SIM.py:1320-1429): A=1, dt=1 projection of u (max_iter 1000). */
int fgb_make_divergence_free(fgb_batch *b, float *u, float *p, const float *bvel, int max_iter, fgb_stream_t s);
/* Simulation.single_step with substeps="ADAPTIVE" (FGSIM.py:210-280, SIM.py:2004-2064) including the
 * advective-outflow "PRE" hook of the cylinder / airfoil environments (CYL.py:289-295, SIM.py:228-393)
 * when the tables carry b_out and char_vel (HOST pointer, 2 floats) is given.  Returns in *substeps_max the largest number of substeps any
 * environment needed (one small device->host read per substep round). */
int fgb_sim_step(fgb_batch *b, float *u, float *p, float *bvel, const float *src, float dt_target, float cfl,
                 const float *char_vel, float bc_tol, const fgb_scalar *sc /* may be NULL */, int32_t *substeps_max,
                 fgb_stream_t s);

/* update_advective_boundaries + balance_boundary_fluxes (SIM.py:188-224, 228-393) for the faces marked in
 * tables.b_out, with the per-environment time step dt[B] (device).  char_vel: HOST pointer to the two
 * components of the characteristic velocity (CYL.py:279-295). */
int fgb_update_outflow(fgb_batch *b, const float *u, float *bvel, const float *dt, const float *char_vel, float bc_tol,
                       fgb_stream_t s);
/* Domain.GetBoundaryFluxBalance (DS.cpp:2476-2510): signed sum of boundary fluxes per environment */
int fgb_flux_balance(fgb_batch *b, const float *bvel, float *out, fgb_stream_t s);
/* balance_boundary_fluxes(domain, free_bounds) (SIM.py:188-224) for an explicit set of free faces
 * (free_mask[NB], device, int8): their velocities are scaled so that the net boundary flux vanishes.  Used
 * by the airfoil actuation, whose free set is outflow + jet wall (airfoil_env_base.py:709-718). */
int fgb_balance_fluxes(fgb_batch *b, float *bvel, const int8_t *free_mask, float bc_tol, fgb_stream_t s);
/* PISOtorch.ComputeSpatialVelocityGradients (PISO_multiblock_cuda_kernel.cu:2997-3043, 6460-6550; used for the vorticity of
 * envs/fluid_env.py:577-656): grad_out [B][2 component c][2 direction d][N] = d u_c / d x_d */
int fgb_velocity_gradients(fgb_batch *b, const float *u, const float *bvel, float *grad_out, fgb_stream_t s);
/* Domain.getMaxVelocity(True, True) (DS.cpp:1580-1611, 2403-2411) */
int fgb_max_velocity(fgb_batch *b, const float *u, const float *bvel, float *out, fgb_stream_t s);

/* ---- environment glue ---------------------------------------------------------------------------- */
/* jet actuation (CYL.py:748-753, jet_cylinder_env_2d.py:185-188): control = last + smoothing*(action-last);
 * bvel[:, faces] = template * control.  faces/template are device arrays of n_faces entries. */
int fgb_apply_jet_action(fgb_batch *b, float *bvel, float *last_control, const float *action, float smoothing,
                         const int32_t *faces, const float *templ /*[2][n_faces]*/, int32_t n_faces, fgb_stream_t s);
/* wall forces (CYL.py:657-698, forces.py:193-275): drag/lift coefficients of one sim step accumulated
 * into acc[B][2].  Ring tables have n_wall entries (ordered around the body). */
typedef struct fgb_wall {
    int32_t n_wall;
    const int32_t *cell;   /* [n] wall-adjacent cell   */
    const int32_t *bface;  /* [n] boundary face index  */
    const float *normal;   /* [2][n] into the fluid    */
    const float *dist;     /* [n] wall distance        */
    const float *tlen;     /* [n] tangent length       */
    const float *flen;     /* [n] wall face length     */
    float scale;           /* 1 / (0.5 U^2 D)          */
} fgb_wall;
/* compute_forces (forces.py:193-275) over the ring w + the drag / lift coefficients of CYL.py:657-698, added to acc[B][2] */
int fgb_wall_forces(fgb_batch *b, const fgb_wall *w, const float *u, const float *p, const float *bvel,
                    float *acc, fgb_stream_t s);
/* column sums over y of fa*fb*det and of det for a single structured nx x ny block (Nusselt number,
 * rbc_env_base.py:491-539; local rewards rbc_env_2d.py:328-357): out[B][2][nx] */
int fgb_column_sums(fgb_batch *b, const float *fa, const float *fb, int32_t nx, int32_t ny, float *out, fgb_stream_t s);
/* sensor sampling (obs_extraction.py:10-57 -> resampling.cu:296-364): out[B][C][n_s] =
 * sum_k w[k][s] * field[B][C][idx[k][s]] (the static splat+normalise+fill map evaluated at the sensors) */
int fgb_sample_sensors(fgb_batch *b, const float *field, int32_t channels, const int32_t *idx, const float *w,
                       int32_t K, int32_t n_sensors, float *out, fgb_stream_t s);
/* the same map without a solver handle: field [B][channels][N] (3-D environments: rendered-voxel sensors of RBC3D,
 * rbc_env_3d.py:183-203, 285-321) */
int fgb_sample_sensors_n(const float *field, int32_t B, int32_t channels, int32_t N, const int32_t *idx, const float *w, int32_t K,
                         int32_t n_sensors, float *out, fgb_stream_t s);

/* ---- rendering (fluidgym_b200/render.py; no solver handle) --------------------------------------------------------------- */
#define FGB_RENDER_IDENTITY 0   /* img = the resampled channel (channels = 1)                    */
#define FGB_RENDER_NORM 1       /* img = |resampled vector| over 2 or 3 channels                  */
/* env.render / render_field (fluid_env.py:577-606 -> resample.py:300-358, resampling.cu:191-364): img[B][P] float32 = the CSR
 * render map (rowptr [P+1], col, w; splat + normalise + fill sweeps, rows in image order) applied to channel c of environment b at
 * field + b * env_stride + c * chan_stride, combined by ``mode``.  range (optional) [B][2] receives order-preserving uint32 keys
 * of each environment's min and max for fgb_render_colour; it is initialised by this call.  No host synchronisation. */
int fgb_render_gather(const float *field, int32_t B, int32_t channels, int32_t N, int64_t chan_stride, int64_t env_stride,
                      int32_t mode, const int32_t *rowptr, const int32_t *col, const float *w, int32_t P, float *img,
                      uint32_t *range, fgb_stream_t s);
/* the colour step of env.render: rgb[B][P][3] uint8 = lut[256][3] at bin floor(256 (v - lo) / (hi - lo)) clamped to [0, 255] (128
 * when hi <= lo); [lo, hi] = the environment's range from fgb_render_gather, or [vmin, vmax] for the whole batch when range is
 * NULL; symmetric != 0 widens it to [-m, m], m = max(|lo|, |hi|).  img 16-byte, rgb 4-byte aligned. */
int fgb_render_colour(const float *img, int32_t B, int32_t P, const uint32_t *range, float vmin, float vmax, int32_t symmetric,
                      const uint8_t *lut, uint8_t *rgb, fgb_stream_t s);

/* ---- differentiability (torch.autograd is layered on top in fluidgym_b200/autograd.py) ----------------- */
/* Tape of one substep: device buffers owned by the caller, filled by fgb_piso_substep_record.  Replaces the
 * tensors the reference's autograd.Functions save per native op (DIFF.py:624-1808). */
typedef struct fgb_tape {      /* C = corrector_steps, n_adv / n_p = advect / pressure non-orthogonal iterations (fgb_options) */
    float *u_in;     /* [B][2][N]   */
    float *p_in;     /* [B][N]      */
    float *bvel_in;  /* [B][2][NB]  */
    float *dt;       /* [B]         */
    float *Coff;     /* [B][4][N]   */
    float *A;        /* [B][N]      */
    float *ustar;    /* [n_adv][B][2][N]  predictor iterates (the last one is the predictor result) */
    float *hb;       /* [C][B][2][N]      HbyA of every corrector */
    float *p;        /* [C*n_p][B][N]     pressure after every solve (mean removed) */
    float *pmean;    /* [C*n_p][B]        the removed means */
    float *u1;       /* [max(C-1,1)][B][2][N]  velocity after every corrector but the last */
    const int32_t *active; /* [B] (0 = skip this environment) or NULL = every environment active.  Read by the recording and the
                              backward call: a skipped environment is the identity (its outputs equal its inputs bit for bit, its
                              cotangents are u_bar = u_out_bar, p_prev_bar = p_out_bar, T_bar = T_out_bar, bvel_bar = sbval_bar = 0)
                              and its tape rows are neither written meaningfully nor read. */
} fgb_tape;
/* forward substep (non-orthogonal path, no passive scalar, the environments of tape->active, C * n_p <= 8) + tape */
int fgb_piso_substep_record(fgb_batch *b, float *u, float *p, const float *bvel, const float *dt, const fgb_tape *tape,
                            fgb_stream_t s);
/* bytes of scratch fgb_piso_substep_backward[_scalar] needs */
size_t fgb_adjoint_workspace_bytes(const fgb_tables *t, int32_t B);
/* vector-Jacobian product of that substep: (u_out_bar, p_out_bar) -> (u_bar, p_prev_bar, bvel_bar), all overwritten.
 * Linear-solve adjoints are solves with the transposed operator (DIFF.py:572-590) by the same on-chip kernels;
 * replaces SetupAdvectionMatrixGrad ... CorrectVelocityGrad (BIND.cpp:582-608). */
int fgb_piso_substep_backward(fgb_batch *b, const fgb_tape *tape, const float *u_out_bar, const float *p_out_bar,
                              float *u_bar, float *p_prev_bar, float *bvel_bar, void *workspace, size_t workspace_bytes,
                              fgb_stream_t s);

/* Passive scalar + buoyancy (RBC environments; the reference differentiates them through the same per-op
 * autograd.Functions, DIFF.py:624-1808, with SetupAdvectionScalarGrad / SetupAdvectionMatrixGrad(forPassiveScalar),
 * BIND.cpp:582-608).  Works on the orthogonal path (fgb_options.nonortho = 0: one predictor solve started from the
 * previous result, one pressure solve per corrector) as well as on the non-orthogonal one. */
typedef struct fgb_tape_scalar {
    float *T_in;      /* [B][N]   temperature entering the substep                  */
    float *T_out;     /* [B][N]   temperature after the scalar solve                */
    float *sbval_in;  /* [B][NB]  boundary temperatures (heaters)                   */
} fgb_tape_scalar;
/* forward substep with scalar transport and buoyancy source (as fgb_piso_substep with sc != NULL) + tapes */
int fgb_piso_substep_record_scalar(fgb_batch *b, float *u, float *p, const float *bvel, const float *dt, const fgb_scalar *sc,
                                   const fgb_tape *tape, const fgb_tape_scalar *stape, fgb_stream_t s);
/* (u_out_bar, p_out_bar, T_out_bar) -> (u_bar, p_prev_bar, bvel_bar, T_bar, sbval_bar), all overwritten.  beta = buoyancy factor
 * of the forward call; workspace as fgb_piso_substep_backward. */
int fgb_piso_substep_backward_scalar(fgb_batch *b, const fgb_tape *tape, const fgb_tape_scalar *stape, float beta,
                                     const float *u_out_bar, const float *p_out_bar, const float *T_out_bar, float *u_bar,
                                     float *p_prev_bar, float *bvel_bar, float *T_bar, float *sbval_bar, void *workspace,
                                     size_t workspace_bytes, fgb_stream_t s);

/* ---- D = 3, orthogonal grids (turbulent channel flow; the same K.cu kernels with DIMS = 3) ------------------ */
/* Geometry tables of a 3-D domain whose metric tensors are diagonal (rectilinear blocks).  Fields are
 * component-major [B][3][N]; faces 0..5 = -x,+x,-y,+y,-z,+z; prescribed (Dirichlet) faces are numbered 0..NB-1
 * and carry boundary velocities bvel [B][3][NB].  On such grids every non-orthogonal coefficient is exactly zero, so
 * one predictor solve and one pressure solve per corrector reproduce the reference's non-orthogonal code path. */
typedef struct fgb_ortho3_tables {
    int32_t N, NB;
    float viscosity;
    const int32_t *nbr;   /* [6][N]  neighbour cell across face f, or -1-j for prescribed face j                 */
    const float *minv;    /* [3][N]  diagonal of M^-1                                                            */
    const float *det;     /* [N]                                                                                 */
    const float *b_minv;  /* [3][NB] diagonal of the boundary-face M^-1 (FixedBoundary.transform)                */
    const float *b_det;   /* [NB]                                                                                */
    /* slab decomposition (0 = single GPU): per-cell arrays are strided by NS = N + 2 * plane cells -- owned cells [0, N),
     * lower halo plane [N, N + plane), upper halo plane [N + plane, NS); N_global = cells of the whole domain (norms) */
    int32_t NS, N_global, plane;
    /* structured box (0 = unknown: the kernels read nbr): cells are ordered (z, y, x) with nx * ny * nz = N owned cells and
     * `closed` has bit d set where direction d ends in prescribed faces (periodic otherwise), boff[f] = index of the first
     * prescribed face of cell face f in the [NB] arrays (faces of a layer in (z,y) / (z,x) / (y,x) order).  The kernels then compute
     * the neighbour indices instead of loading them (24 bytes per cell less, one dependent load less per gather). */
    int32_t nx, ny, nz, closed;
    int32_t boff[6];
    /* z-extruded multi-block grids (nx = 0, nbr = the 6-face table of the extruded domain): rev [4][plane] = the in-plane face of
     * neighbour nbr[f] that points back (tables.rev of the 2-D plane), plane = cells per plane; NULL: the opposite face.  Only the
     * transposed Krylov solves of the reverse mode read it. */
    const int8_t *rev;
} fgb_ortho3_tables;
typedef struct fgb_ortho3 fgb_ortho3;
/* D = 3 handle over caller-owned device memory, as fgb_workspace_bytes / fgb_batch_create / fgb_batch_destroy / fgb_batch_set_options
 * (stands for the reference's Domain + PISOtorch block set-up of a box grid, domain_structs.cpp, envs/tcf/grid.py) */
size_t fgb_ortho3_workspace_bytes(const fgb_ortho3_tables *t, int32_t B);
int fgb_ortho3_create(const fgb_ortho3_tables *t, int32_t B, void *workspace, size_t workspace_bytes, const fgb_options *opt,
                      fgb_ortho3 **out);
void fgb_ortho3_destroy(fgb_ortho3 *b);
int fgb_ortho3_set_options(fgb_ortho3 *b, const fgb_options *opt);
/* named workspace buffers: "Coff" [B][6][N], "A", "rhs" [B][3][N], "ures", "Poff", "Pdiag", "hbya", "div", "iters" [B][8]
 * (0..2 BiCGStab per component, 3.. CG per corrector), "resid", "dt", "active", "nsub", "maxvel", "src" [B][4], "rowmean" [B][4] */
void *fgb_ortho3_buffer(fgb_ortho3 *b, const char *name);
/* number of kernel launches issued through this handle since creation */
long long fgb_ortho3_launch_count(fgb_ortho3 *b);
/* per-op entry points (SetupAdvectionMatrix + SetupAdvectionVelocity | SolveLinear(BiCGStab) | SetupPressureMatrix +
 * SetupPressureRHS + SetupPressureRHSdiv | SolveLinear(CG) + mean removal | CorrectVelocity), cf. the 2-D table above.
 * src: optional per-environment static velocity source [B][4] (Block.setVelocitySource, 3 used). */
int fgb_ortho3_setup_advection(fgb_ortho3 *b, const float *u, const float *bvel, const float *src, const float *dt,
                               const int32_t *active, fgb_stream_t s);
int fgb_ortho3_solve_advection(fgb_ortho3 *b, int zero_init, const int32_t *active, fgb_stream_t s);
int fgb_ortho3_setup_pressure(fgb_ortho3 *b, const float *u, const float *bvel, const float *src, const float *dt, int with_matrix,
                              const int32_t *active, fgb_stream_t s);
int fgb_ortho3_solve_pressure(fgb_ortho3 *b, float *p_out, int zero_init, int reset_steps, int max_iter, int slot,
                              const int32_t *active, fgb_stream_t s);
int fgb_ortho3_correct_velocity(fgb_ortho3 *b, const float *p, float *u_out, const int32_t *active, fgb_stream_t s);
/* fused: Simulation._PISO_split_step / make_divergence_free / single_step (adaptive CFL) for D = 3 */
int fgb_ortho3_piso_substep(fgb_ortho3 *b, float *u, float *p, const float *bvel, const float *src, const float *dt,
                            const int32_t *active, fgb_stream_t s);
/* Passive scalar + buoyancy on a 3-D box (RBC3D: rbc_env_base.py:190-304 with ndims = 3).  Buffers are caller-owned device memory. */
typedef struct fgb_ortho3_scalar {
    float *T;             /* [B][NS]  scalar field, updated in place by the substep                        */
    const float *sbval;   /* [B][NB]  Dirichlet values on the prescribed faces (FixedBoundary.passiveScalar) */
    float kappa;          /*          scalar diffusivity (Domain.setScalarViscosity)                        */
    float beta;           /*          buoyancy factor: velocity source (0, beta T, 0)                       */
} fgb_ortho3_scalar;
/* attach (or with NULL detach) the scalar: fgb_ortho3_piso_substep / _sim_step then run the scalar transport first */
int fgb_ortho3_set_scalar(fgb_ortho3 *b, const fgb_ortho3_scalar *sc);
/* SetupAdvectionMatrix(forPassiveScalar) + SetupAdvectionScalar + SolveLinear(BiCGStab, zero start): T <- C_s(u)^-1 rhs_s(T) */
int fgb_ortho3_advect_scalar(fgb_ortho3 *b, const float *u, const float *bvel, const float *dt, const int32_t *active, fgb_stream_t s);
/* Smagorinsky sub-grid viscosity (PISOtorch.SGSviscosityIncompressibleSmagorinsky, PISO_multiblock_cuda_kernel.cu:6913-7035, as
 * used by the channel-flow "PRE" prep function, envs/tcf/tcf_env.py:441-472): nu_cell = nu + coefficient * delta * |S| * damping,
 * delta = squared longest cell edge, |S| = sqrt(2 S_ij S_ij).  coefficient 0 switches the model off.  damping: [N] device floats
 * (squared van Driest factor, envs/tcf/grid.py:101-125) or NULL; kept by pointer.  With a model set, fgb_ortho3_piso_substep /
 * _sim_step refresh the per-cell viscosity (buffer "visc") from the incoming velocity before every substep. */
int fgb_ortho3_set_sgs(fgb_ortho3 *b, float coefficient, const float *damping);
int fgb_ortho3_sgs_viscosity(fgb_ortho3 *b, const float *u, const float *bvel, const int32_t *active, fgb_stream_t s);
/* PISOtorch.ComputeSpatialVelocityGradients (PISO_multiblock_cuda_kernel.cu:6460-6550; Q criterion tcf_env.py:586-644, vorticity
 * fluid_env.py:577-656): grad_out [B][3 component c][3 direction d][NS] = d u_c / d x_d -- the reference's list index is the
 * component and the tensor channel the direction (its kernel, K.cu:6470-6480), the layout kept here */
int fgb_ortho3_velocity_gradients(fgb_ortho3 *b, const float *u, const float *bvel, float *grad_out, fgb_stream_t s);
/* Reverse mode of the D = 3 substep (single GPU, structured box, no scalar / SGS): tape filled by the recording forward call,
 * vector-Jacobian product by hand-written adjoint kernels + the Krylov solves with the transposed operator.  Replaces the
 * dimension-generic _GRAD kernels the reference differentiates these grids with (PISO_multiblock_cuda_kernel.cu:3884-4090,
 * 4403-4491, 6265-6309; PISOtorch_diff.py:624-1808).  As in the reference's differentiable backend every recorded solve starts
 * from zero and the CG does not reset its residual.  C = corrector_steps. */
typedef struct fgb_ortho3_tape {
    float *u_in;     /* [B][3][N]  */
    float *bvel_in;  /* [B][3][NB] */
    float *dt;       /* [B]        */
    float *Coff;     /* [B][6][N]  */
    float *A;        /* [B][N]     */
    float *ustar;    /* [B][3][N]       predictor result */
    float *hb;       /* [C][B][3][N]    HbyA of every corrector */
    float *p;        /* [C][B][N]       pressure of every corrector (mean removed) */
    float *u1;       /* [max(C-1,1)][B][3][N]  velocity after every corrector but the last */
    float *visc;     /* [B][N] per-cell viscosity of the substep when a sub-grid model is set (fgb_ortho3_set_sgs), else NULL: a constant of
                      * the graph, as in the reference, whose Smagorinsky op has no autograd wrapper */
    const int32_t *active; /* [B] (0 = skip this environment) or NULL = every environment active; as fgb_tape.active (identity
                              cotangents u_bar = u_out_bar, T_bar = T_out_bar, bvel_bar = sbval_bar = 0) */
} fgb_ortho3_tape;
/* forward substep of the D = 3 box (as fgb_ortho3_piso_substep for the environments of tape->active) that also fills the tape (the forward() of the reference's autograd
 * Functions, PISOtorch_diff.py:624-1808) + bytes of scratch the backward needs */
int fgb_ortho3_piso_substep_record(fgb_ortho3 *b, float *u, float *p, const float *bvel, const float *src, const float *dt,
                                   const fgb_ortho3_tape *tape, fgb_stream_t s);
size_t fgb_ortho3_adjoint_workspace_bytes(const fgb_ortho3_tables *t, int32_t B);
/* (u_out_bar, p_out_bar) -> (u_bar, bvel_bar), both overwritten; the previous pressure and the source do not receive gradients
 * (zero-started solves on an orthogonal grid; the channel forcing is detached in the reference, envs/tcf/grid.py:147-161) */
int fgb_ortho3_piso_substep_backward(fgb_ortho3 *b, const fgb_ortho3_tape *tape, const float *u_out_bar, const float *p_out_bar,
                                     float *u_bar, float *bvel_bar, void *workspace, size_t workspace_bytes, fgb_stream_t s);
/* the same with an attached passive scalar + buoyancy (RBC3D; fgb_ortho3_set_scalar): the scalar buffer is advanced in place by the
 * forward call; additional gradients: temperature field and boundary temperatures (heaters).  fgb_tape_scalar as in 2-D. */
int fgb_ortho3_piso_substep_record_scalar(fgb_ortho3 *b, float *u, float *p, const float *bvel, const float *src, const float *dt,
                                          const fgb_ortho3_tape *tape, const fgb_tape_scalar *stape, fgb_stream_t s);
int fgb_ortho3_piso_substep_backward_scalar(fgb_ortho3 *b, const fgb_ortho3_tape *tape, const fgb_tape_scalar *stape, const float *u_out_bar,
                                            const float *p_out_bar, const float *T_out_bar, float *u_bar, float *bvel_bar, float *T_bar,
                                            float *sbval_bar, void *workspace, size_t workspace_bytes, fgb_stream_t s);
/* Simulation.make_divergence_free (SIM.py:1320-1429) on the box: A = 1, dt = 1 projection of u; p receives the projection pressure */
int fgb_ortho3_make_divergence_free(fgb_ortho3 *b, float *u, float *p, const float *bvel, int max_iter, fgb_stream_t s);
/* Simulation.single_step with adaptive CFL substeps (FGSIM.py:210-280, SIM.py:2004-2064) for D = 3.
 * rows: [2][n_row] cells of the first / last wall-normal layer; d_lo, d_hi their wall distances.  With rows != NULL the
 * channel forcing G_x = nu/2 (<u>_lo/d_lo + <u>_hi/d_hi) (envs/tcf/grid.py:128-163) is refreshed before every substep. */
int fgb_ortho3_sim_step(fgb_ortho3 *b, float *u, float *p, const float *bvel, float dt_target, float cfl, const int32_t *rows,
                        int n_row, float d_lo, float d_hi, int32_t *substeps_max, fgb_stream_t s);
/* wall shear stresses tau = nu <u>_row / d (tcf_env.py:564-584) into "rowmean"; set_forcing: also write "src";
 * acc [B][2] (optional): += (tau_lo, tau_hi) */
int fgb_ortho3_wall_rows(fgb_ortho3 *b, const float *u, const int32_t *rows, int n_row, float d_lo, float d_hi, int set_forcing,
                         float *acc, fgb_stream_t s);

/* Adaptive CFL plan of one round (SIM.py:2004-2031, the arithmetic of fgb_sim_step's planner), one thread per environment, no solver
 * handle: for every environment with time left (remaining > 0 and |remaining| > 1e-8) dt = the next substep size from maxvel and cfl,
 * remaining -= dt, nsub += 1, active = 1 and counter[0] += 1; finished environments get dt = 0, active = 0.  maxvel [B] float, remaining
 * [B] double, dt [B] float, active / nsub [B] int32, counter [1] int32 (not cleared by this call): all device pointers.  Lets a caller
 * drive per-environment substeps of its own (differentiable rollouts: fluidgym_b200/solver.py::cfl_substeps_per_env). */
int fgb_plan_substep(int32_t B, const float *maxvel, double *remaining, float cfl, float *dt, int32_t *active, int32_t *nsub,
                     int32_t *counter, fgb_stream_t s);

/* ---- slab decomposition of one large 3-D domain over the GPUs of a node (one process per GPU) -------------------------
 * Every rank owns nz/world z-planes.  All device memory the solver touches lives in ONE symmetric allocation per rank
 * (fgb_ipc_alloc) that every peer maps with CUDA IPC (fgb_ipc_open): halo planes and reduction partials are written
 * straight into the peer's memory over NVLink from inside the persistent Krylov kernels, sequence-numbered flags replace
 * collectives (no NCCL call on the solver path).  The first 4 KiB of the region are reserved for the flag pad. */
/* symmetric allocation of one rank + its CUDA IPC handle / map, unmap a peer's / release the own one (no reference counterpart: the
 * reference runs one domain on one GPU) */
int fgb_ipc_alloc(size_t bytes, void **ptr, unsigned char *handle_out /* [64] */);
int fgb_ipc_open(const unsigned char *handle /* [64] */, void **peer_ptr);
int fgb_ipc_close(void *peer_ptr);
int fgb_ipc_free(void *ptr);
/* bind a handle created on the rank's slab tables (NS, N_global, plane) to its place among the peers' mapped regions */
int fgb_ortho3_set_slab(fgb_ortho3 *b, int32_t rank, int32_t world, void *local_base, void *const *peer_bases);
/* non-zero in *out when a wait on a peer timed out (results invalid) */
int fgb_ortho3_slab_error(fgb_ortho3 *b, int32_t *out);

/* ---- measurement hooks (bench.py) ------------------------------------------------------------------ */
/* Record CUDA events around the solver launches on their own stream.  fgb_profile_read synchronises the
 * device and returns accumulated milliseconds / launch counts per class {0: pressure CG, 1: BiCGStab,
 * 2: assembly kernels, 3: other}. */
int fgb_profile_enable(fgb_batch *b, int on);
int fgb_profile_read(fgb_batch *b, double *ms_out /*[4]*/, int64_t *count_out /*[4]*/, int reset);
/* number of kernel launches issued through this handle since creation */
long long fgb_launch_count(fgb_batch *b);

/* ---- D = 3, z-extruded multi-block domains (CylinderJet3D, Airfoil3D: envs/cylinder/grid.py:298, shapes.py:641-676) ----------
 * The 2-D tables of the compiled plane + nz uniform periodic planes of spacing hz.  Fields [B][3][nz*N], cell = plane * N + g;
 * boundary velocities [B][3][nz][NB].  The handle is an fgb_ortho3 created on the 6-face neighbour table of the extruded domain
 * (faces 0..3 in plane, 4 = -z, 5 = +z), whose cooperative Krylov kernels solve the ELL(7) systems.  Operator arithmetic is
 * verified on the CPU against a trace of the reference (tests/test_extruded_host.py, tests/test_cylinder3d_cpu.py run the same
 * cell code) and on a B200 against the reference's env.step and gradients (tests/test_gpu_extruded.py). */
typedef struct fgb_extruded3_tables {
    fgb_tables plane;
    int32_t nz;
    float hz;
} fgb_extruded3_tables;
/* Simulation._PISO_split_step (SIM.py:1431-2002, non-orthogonal path; pressure_non_ortho_steps = 4 in 3-D, cylinder_env_base.py:317) */
int fgb_extruded3_piso_substep(fgb_ortho3 *b, const fgb_extruded3_tables *x, float *u, float *p, const float *bvel, const float *dt,
                               fgb_stream_t s);
/* Reverse mode of the extruded substep (CylinderJet3D / Airfoil3D, differentiable=True): as fgb_piso_substep_record / _backward with three
 * velocity components -- tape fields u_in / ustar / hb / u1 [..][B][3][N3], Coff [B][6][N3], A / p_in / p [..][B][N3], bvel_in
 * [B][3][nz][NB2], pmean [C*n_p][B].  The handle's tables need rev (in-plane reverse faces) and plane = N2 for the transposed solves.
 * Replaces the dimension-generic _GRAD kernels of the reference on these grids (PISO_multiblock_cuda_kernel.cu:3884-4090, 4403-4491). */
int fgb_extruded3_piso_substep_record(fgb_ortho3 *b, const fgb_extruded3_tables *x, float *u, float *p, const float *bvel, const float *dt,
                                      const fgb_tape *tape, fgb_stream_t s);
size_t fgb_extruded3_adjoint_workspace_bytes(const fgb_extruded3_tables *x, int32_t B);
int fgb_extruded3_piso_substep_backward(fgb_ortho3 *b, const fgb_extruded3_tables *x, const fgb_tape *tape, const float *u_out_bar,
                                        const float *p_out_bar, float *u_bar, float *p_prev_bar, float *bvel_bar, void *workspace,
                                        size_t workspace_bytes, fgb_stream_t s);
/* Simulation.make_divergence_free (SIM.py:1320-1430) on an extruded domain: projection with A = 1, p_nonortho_steps deferred
 * corrections; max_iter <= 0 takes the handle's option.  The outflow update of its "PRE" hook is the caller's. */
int fgb_extruded3_make_divergence_free(fgb_ortho3 *b, const fgb_extruded3_tables *x, float *u, float *p, const float *bvel, int max_iter,
                                       fgb_stream_t s);
/* Boundary hooks of the extruded environments (opt-in, FGB_X3_HOOKS=cuda; default: the torch expressions of extruded3d.py):
 * balance_boundary_fluxes (SIM.py:188-224) with an explicit set of free faces (all planes), update_advective_boundaries
 * (SIM.py:228-393) of the outflow faces followed by their balance, Domain.getMaxVelocity(True, True) (DS.cpp:1580-1612).
 * fw [2][NB]: signed in-plane flux weights per unit plane spacing; out_face / out_cell / out_adv [n_out]: outflow faces of the plane,
 * their adjacent cells and advective speeds M^-1 . u_char. */
int fgb_extruded3_balance_fluxes(const fgb_extruded3_tables *x, int32_t B, float *bvel, const float *fw, const int8_t *free_mask, float tol,
                                 fgb_stream_t s);
int fgb_extruded3_update_outflow(const fgb_extruded3_tables *x, int32_t B, const float *u, float *bvel, const float *dt, const float *fw,
                                 const int8_t *out_mask, int32_t n_out, const int32_t *out_face, const int32_t *out_cell, const float *out_adv,
                                 float tol, fgb_stream_t s);
int fgb_extruded3_max_velocity(const fgb_extruded3_tables *x, int32_t B, const float *u, const float *bvel, float *maxvel, fgb_stream_t s);
/* actuation: bvel[0..1][plane k][jet_face q] = sum_j amp[b][k][j] * templ[j][0..1][q] (amp [B][nz][J], templ [J][2][nf]), spanwise component 0,
 * then the flux balance over free_mask (jet_cylinder_env_3d.py:399-424, airfoil_env_3d.py:383-407) */
int fgb_extruded3_apply_jets(const fgb_extruded3_tables *x, int32_t B, float *bvel, const float *amp, int32_t J, const int32_t *jet_face,
                             const float *templ, int32_t nf, const float *fw, const int8_t *free_mask, float tol, fgb_stream_t s);
/* per-plane drag / lift coefficient contributions out[B][nz][2] (forces.py:278-377: 2-D wall traction x plane spacing) */
int fgb_extruded3_wall_forces(const fgb_extruded3_tables *x, int32_t B, const fgb_wall *w, const float *u, const float *p, const float *bvel,
                              float *out, fgb_stream_t s);

#ifdef __cplusplus
}
#endif
#endif
