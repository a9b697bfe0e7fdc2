// D = 3 instantiation of the PISO substep for ORTHOGONAL grids (turbulent channel flow, SURVEY.md section 8 config 5;
// reference: the same K.cu kernels with DIMS = 3).  Included at the end of piso_b200.cu (one translation unit, shared
// error handling / reductions).  On a rectilinear grid every off-diagonal metric coefficient is exactly zero, so the
// deferred non-orthogonal corrections of the 2-D path vanish (`if (alpha != 0)`, K.cu:3772) and the matrices are
// plain ELL(7) on a 6-face neighbour table.  Specification: oracle/box3d_eval.py (validated against a trace of the
// reference on a 32 x 32 x 32 channel to 1e-7 per operator).
//
// Large single environments do not fit a thread-block cluster, so the Krylov solvers here are persistent
// COOPERATIVE kernels: the whole GPU works on one system, vectors stay in L2 (266 k cells x 5 vectors = 5 MB of
// the 126 MB L2), grid-wide reductions are a fixed-order two-stage sum (deterministic) separated by grid.sync().

typedef fgb_ortho3_tables T3;

// ---- slab decomposition (one process per GPU, z-slabs, halos pushed over NVLink into the peer's memory) ----------
// Every rank allocates ONE symmetric region with identical layout (fgb_ipc_alloc) and maps the peers' regions
// (cudaIpcOpenMemHandle): the address of any buffer on rank q is peer_base[q] + (local address - local_base).
// Cells: owned [0, N), lower halo plane [N, N + P), upper halo plane [N + P, N + 2P); arrays are strided by NS = N + 2P.
static constexpr int O3_MAXR = 8;
struct O3Pad {                                      // first bytes of the symmetric region of every rank
    unsigned long long ar_seq[2][O3_MAXR];          // all-reduce arrival flags (parity double-buffered), per source rank
    double ar_val[2][O3_MAXR][8];                   // all-reduce payloads
    unsigned long long halo_seq[O3_MAXR];           // "my halo planes are in your memory" flags, per source rank
    unsigned long long bar_seq[O3_MAXR];            // stream-level barrier flags, per source rank
    int error;                                      // set when a wait timed out (a peer died): results are invalid
};
struct O3Slab {
    int rank, world, lower, upper;                  // neighbours along z (periodic)
    int on;                                         // slab protocol active (world == 1 exchanges with itself: periodic wrap)
    char *local_base;
    char *peer_base[O3_MAXR];
    unsigned long long *ctr;                        // [3] local sequence counters: all-reduce, halo, barrier
};
template <typename T>
__device__ __forceinline__ T *o3_peer(const O3Slab &sl, T *p, int q) { return (T *)(sl.peer_base[q] + ((char *)p - sl.local_base)); }
__device__ __forceinline__ O3Pad *o3_pad(const O3Slab &sl, int q) { return (O3Pad *)sl.peer_base[q]; }
__device__ __forceinline__ void o3_wait_ge(volatile unsigned long long *flag, unsigned long long s, O3Pad *mine) {
    const long long t0 = clock64();
    while (*flag < s) {
        if (clock64() - t0 > 6000000000LL) { mine->error = 1; break; }      // ~3 s: a peer is gone, do not hang the GPU
    }
}

// owned boundary planes -> the z-neighbours' halo planes (direct stores into peer memory over NVLink)
// `dirty` records that this thread has peer stores in flight: only such threads need the (expensive) system-scope fence
// before the next grid barrier; cumulativity carries their stores in front of the flag that CTA 0 writes after it.
__device__ __forceinline__ void o3_push(const O3Slab &sl, const T3 &t, float *vec, int g, float val, bool &dirty) {
    if (sl.on) {
        const int P = t.plane, N = t.N;
        if (g < P) { o3_peer(sl, vec, sl.lower)[N + P + g] = val; dirty = true; }               // my lowest plane = the lower neighbour's UPPER halo
        if (g >= N - P) { o3_peer(sl, vec, sl.upper)[N + (g - (N - P))] = val; dirty = true; }  // my highest plane = the upper neighbour's LOWER halo
    }
}

struct fgb_ortho3 {
    T3 t;
    O3Slab slab;
    int B;
    fgb_options opt;
    float *Coff, *A, *rhs, *ures, *Poff, *Pdiag, *hbya, *div, *kry, *part;
    int32_t *iters; float *resid; float *dt; int32_t *active; double *remaining; int32_t *nsub; float *maxvel;
    int32_t *counters; int32_t *h_counters; float *src; float *rowmean;
    float *pmean;                     // [B][8] mean removed from the pressure of solve slot q (the adjoint needs the raw iterate p + mean)
    unsigned long long *iter_total;
    unsigned long long *slab_ctr;     // [4] device-side sequence counters of the slab protocol
    fgb_ortho3_scalar sc;             // passive scalar + buoyancy (RBC3D); sc.T == nullptr: none
    int grid_blocks;
    float *visc;                      // [B][NS] per-cell viscosity nu + nu_sgs (fgb_ortho3_set_sgs), refreshed before every substep
    float sgs_coef; const float *sgs_damp;
    int bicg_fused;                   // k3_bicgstab<.,1>: search-direction update folded into the product (4 instead of 5 exchanges per iteration); opt-in
    int cg_fused;                     // k3_cg_fused (2 grid.sync per CG iteration, bit-identical to k3_cg) on a single GPU; default 1,
                                      // FGB_K3_CG_FUSED=0 selects k3_cg
    long long launches;
};

static constexpr int O3_T = 256;          // threads per CTA of the one-thread-per-cell kernels
static constexpr int O3_CT = 1024;        // threads per CTA of the cooperative Krylov kernels (one CTA per SM: a grid.sync over
                                          // 148 CTAs costs ~2 us, over 592 CTAs ~5 us, and there are 3-7 of them per iteration)
static constexpr int O3_KRY = 21;         // Krylov work vectors per environment (BiCGStab: 7 per component -- r, r^, p, v, t and the second
                                          // copies of p and v of the fused search-direction update)
static constexpr int O3_PART = 8;         // floats per CTA per reduction slot

extern "C" size_t fgb_ortho3_workspace_bytes(const fgb_ortho3_tables *t, int32_t B) {
    const size_t BN = (size_t)B * (t->NS > 0 ? t->NS : t->N);
    size_t n = 0;
    n += align_up(6 * BN * 4) * 2 + align_up(BN * 4) * 4 + align_up(3 * BN * 4) * 3 + align_up((size_t)O3_KRY * BN * 4);
    n += align_up((size_t)2 * 4096 * O3_PART * 4);
    n += align_up((size_t)B * 64) * 16 + 8192;        // per-environment scalars (iteration counters, dt, flags, forcing ...)
    return n;
}

extern "C" int fgb_ortho3_create(const fgb_ortho3_tables *t, int32_t B, void *workspace, size_t workspace_bytes, const fgb_options *opt,
                                 fgb_ortho3 **out) {
    if (!t || !out || B <= 0 || t->N <= 0 || !t->nbr || !t->minv || !t->det) return set_err(FGB_E_ARG, "fgb_ortho3_create: bad argument");
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0) return set_err(FGB_E_CUDA, "fgb_ortho3_create: no CUDA device (there is no CPU fallback)", ce);
    if (!workspace || workspace_bytes < fgb_ortho3_workspace_bytes(t, B)) return set_err(FGB_E_WORKSPACE, "fgb_ortho3_create: workspace too small");
    fgb_ortho3 *b = new (std::nothrow) fgb_ortho3();
    if (!b) return set_err(FGB_E_ARG, "fgb_ortho3_create: out of host memory");
    b->t = *t; b->B = B; b->launches = 0;
    if (opt) b->opt = *opt; else { b->opt.corrector_steps = 2; b->opt.adv_nonortho_steps = 1; b->opt.p_nonortho_steps = 1; b->opt.nonortho = 1;
                                   b->opt.adv_tol = 1e-6f; b->opt.p_tol = 1e-6f; b->opt.max_iter = 5000; b->opt.cg_impl = 0; }
    if (b->t.NS <= 0) b->t.NS = b->t.N;
    if (b->t.N_global <= 0) b->t.N_global = b->t.N;
    memset(&b->slab, 0, sizeof(b->slab)); b->slab.world = 1;
    memset(&b->sc, 0, sizeof(b->sc));
    b->sgs_coef = 0.f; b->sgs_damp = nullptr;
    const size_t BN = (size_t)B * b->t.NS;
    Carver c{(char *)workspace, 0};
    b->Coff = c.take<float>(6 * BN); b->Poff = c.take<float>(6 * BN);
    b->A = c.take<float>(BN); b->Pdiag = c.take<float>(BN); b->div = c.take<float>(BN);
    b->visc = c.take<float>(BN);
    b->rhs = c.take<float>(3 * BN); b->ures = c.take<float>(3 * BN); b->hbya = c.take<float>(3 * BN);
    b->kry = c.take<float>((size_t)O3_KRY * BN);
    b->part = c.take<float>((size_t)2 * 4096 * O3_PART);
    b->iters = c.take<int32_t>((size_t)B * 8); b->resid = c.take<float>((size_t)B * 8);
    b->remaining = c.take<double>(B); b->iter_total = c.take<unsigned long long>((size_t)B * 2);
    (void)c.take<double>(B);
    b->dt = c.take<float>(B); b->active = c.take<int32_t>(B); b->nsub = c.take<int32_t>(B); b->maxvel = c.take<float>(B);
    b->counters = c.take<int32_t>(4); (void)c.take<float>(B);
    b->src = c.take<float>((size_t)B * 4); b->rowmean = c.take<float>((size_t)B * 4);
    b->slab_ctr = c.take<unsigned long long>(4);
    b->pmean = c.take<float>((size_t)B * 8);
    ce = cudaMallocHost((void **)&b->h_counters, 16);
    if (ce != cudaSuccess) { delete b; return set_err(FGB_E_CUDA, "cudaMallocHost", ce); }
    ce = cudaMemset(workspace, 0, fgb_ortho3_workspace_bytes(t, B));
    if (ce != cudaSuccess) { cudaFreeHost(b->h_counters); delete b; return set_err(FGB_E_CUDA, "cudaMemset workspace", ce); }
    b->grid_blocks = 0;
    b->cg_fused = 1;                  // measured on a B200 (profiles/r02_k3_cg_fused_ab.txt): CylinderJet3D res 24 26.5 -> 21.2 ms / substep
    if (const char *ev = getenv("FGB_K3_CG_FUSED")) b->cg_fused = atoi(ev) != 0;
    b->bicg_fused = 0;                // opt-in (FGB_K3_BICG_FUSED=1): bit-identical, one exchange less per iteration, but measured SLOWER on one GPU (TCFLarge 1.11 vs
                                      // 1.04 ms / substep: 21 instead of 7 gathers per cell and 600 bytes of spills at the 64-register cap), profiles/r02_k3_kernels.md
    if (const char *ev = getenv("FGB_K3_BICG_FUSED")) b->bicg_fused = atoi(ev) != 0;
    *out = b;
    return FGB_OK;
}
extern "C" void fgb_ortho3_destroy(fgb_ortho3 *b) {
    if (!b) return;
    if (b->h_counters) cudaFreeHost(b->h_counters);
    delete b;
}
extern "C" int fgb_ortho3_set_options(fgb_ortho3 *b, const fgb_options *opt) {
    if (!b || !opt) return set_err(FGB_E_ARG, "fgb_ortho3_set_options: bad argument");
    b->opt = *opt;
    return FGB_OK;
}
extern "C" void *fgb_ortho3_buffer(fgb_ortho3 *b, const char *name) {
    if (!b || !name) return nullptr;
    struct { const char *n; void *p; } tab[] = {
        {"Coff", b->Coff}, {"A", b->A}, {"rhs", b->rhs}, {"ures", b->ures}, {"Poff", b->Poff}, {"Pdiag", b->Pdiag}, {"hbya", b->hbya},
        {"div", b->div}, {"visc", b->visc}, {"iters", b->iters}, {"resid", b->resid}, {"dt", b->dt}, {"active", b->active}, {"nsub", b->nsub},
        {"maxvel", b->maxvel}, {"pmean", b->pmean}, {"src", b->src}, {"rowmean", b->rowmean}, {"iter_total", b->iter_total}, {"remaining", b->remaining}};
    for (auto &e : tab) if (!strcmp(e.n, name)) return e.p;
    return nullptr;
}
extern "C" long long fgb_ortho3_launch_count(fgb_ortho3 *b) { return b ? b->launches : 0; }

// ------------------------------------------------------------------------------------------------
// one thread per (cell, environment): blockIdx.y = environment
// ------------------------------------------------------------------------------------------------
static inline dim3 o3_grid(const fgb_ortho3 *b) { return dim3((unsigned)((b->t.N + O3_T - 1) / O3_T), (unsigned)b->B); }

// neighbour cells of g across the six faces, or -1 - j for the prescribed face j, exactly as tables.nbr holds them.  Structured boxes
// (t.nx > 0): index arithmetic on the (z, y, x) ordering -- periodic wrap, closed ends (boundary faces of face f are numbered
// boff[f] + the flattened position in the face layer), slab halo planes [N, N + P) / [N + P, NS) -- instead of six table loads that
// every gather would depend on.
__device__ __forceinline__ void o3_nbrs(const T3 &t, int g, int (&n)[6]) {
    if (t.nx > 0) {
        const int nx = t.nx, ny = t.ny, P = nx * ny;
        const int q = g / nx, i = g - q * nx, k = q / ny, j = q - k * ny;
        const bool cx = t.closed & 1, cy = t.closed & 2, cz = t.closed & 4, halo = t.NS > t.N;
        n[0] = i > 0 ? g - 1 : (cx ? -1 - (t.boff[0] + q) : g + (nx - 1));
        n[1] = i < nx - 1 ? g + 1 : (cx ? -1 - (t.boff[1] + q) : g - (nx - 1));
        n[2] = j > 0 ? g - nx : (cy ? -1 - (t.boff[2] + k * nx + i) : g + (ny - 1) * nx);
        n[3] = j < ny - 1 ? g + nx : (cy ? -1 - (t.boff[3] + k * nx + i) : g - (ny - 1) * nx);
        n[4] = k > 0 ? g - P : (halo ? t.N + (g - k * P) : (cz ? -1 - (t.boff[4] + g - k * P) : g + (t.nz - 1) * P));
        n[5] = k < t.nz - 1 ? g + P : (halo ? t.N + P + (g - k * P) : (cz ? -1 - (t.boff[5] + g - k * P) : g - (t.nz - 1) * P));
    } else {
#pragma unroll
        for (int f = 0; f < 6; ++f) n[f] = t.nbr[f * t.NS + g];
    }
}
__device__ __forceinline__ float o3_bflux(const T3 &t, int j, int d, const float *bv /* [3][NB] of this env */) {
    return t.b_det[j] * t.b_minv[d * t.NB + j] * bv[d * t.NB + j];
}

// C = (det/dt I + convection + diffusion)/det as ELL(7), A = diag(C), predictor RHS (K.cu:3617-3880, 4296-4400)
__global__ void __launch_bounds__(O3_T) k3_setup_advection(T3 t, O3Slab sl, const float *__restrict__ U, const float *__restrict__ Bvel,
                                                           const float *__restrict__ Src /* [B][4] or null */, const float *__restrict__ dtv,
                                                           const int32_t *__restrict__ active, float *__restrict__ Coff, float *__restrict__ A,
                                                           float *__restrict__ Rhs, const float *__restrict__ Tbuoy /* [B][NS] or null */, float beta,
                                                           const float *__restrict__ Visc /* [B][NS] per-cell viscosity (SGS) or null */) {
    const int b = blockIdx.y, g = blockIdx.x * blockDim.x + threadIdx.x, N = t.N, NS = t.NS, NB = t.NB;
    if (g >= N || (active && !active[b])) return;
    const float *u = U + (size_t)b * 3 * NS, *bv = Bvel + (size_t)b * 3 * NB, *vv = Visc ? Visc + (size_t)b * NS : nullptr;
    const float dt = dtv[b], det = t.det[g], visc = vv ? vv[g] : t.viscosity;
    float uo[3], mi[3], al[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) { uo[d] = u[d * NS + g]; mi[d] = t.minv[d * NS + g]; al[d] = det * mi[d] * mi[d]; }
    float diag = det / dt, Sb[3] = {0.f, 0.f, 0.f};
    int nb6[6];
    o3_nbrs(t, g, nb6);
#pragma unroll
    for (int f = 0; f < 6; ++f) {
        const int d = f >> 1, n = nb6[f];
        const float sig = (f & 1) ? 1.f : -1.f;
        float off = 0.f;
        if (n >= 0) {
            const float dn = t.det[n], mn = t.minv[d * NS + n];
            const float fl = 0.5f * (det * mi[d] * uo[d] + dn * mn * u[d * NS + n]);
            const float vc = (al[d] * visc + (dn * mn * mn) * (vv ? vv[n] : visc)) * 0.5f;   // K.cu:3741-3750
            const float ff = sig * 0.5f * fl;
            diag += ff + vc;
            off = (ff - vc) / det;
        } else {
            const int j = -1 - n;
            diag += 2.f * visc * al[d];
            const float bm = t.b_minv[d * NB + j];
            const float k = -(sig * o3_bflux(t, j, d, bv)) + 2.f * visc * (t.b_det[j] * bm * bm);
#pragma unroll
            for (int c = 0; c < 3; ++c) Sb[c] += bv[c * NB + j] * k;
        }
        Coff[((size_t)b * 6 + f) * NS + g] = off;
    }
    const float Ag = diag / det;
    A[(size_t)b * NS + g] = Ag;
#pragma unroll
    for (int c = 0; c < 3; ++c)
        Rhs[((size_t)b * 3 + c) * NS + g] = (det * uo[c] / dt + Sb[c]) / det + (Src ? Src[b * 4 + c] : 0.f) +
                                            ((Tbuoy && c == 1) ? Tbuoy[(size_t)b * NS + g] * beta : 0.f);   // rbc_env_base.py:280-304
    bool dirty = false;
    o3_push(sl, t, A, g, Ag, dirty);          // (slabs: B == 1) consumed after the predictor solve, whose reductions order it
    if (dirty) __threadfence_system();
}

// Passive-scalar transport (SetupAdvectionMatrix(forPassiveScalar) + SetupAdvectionScalar, K.cu:3617-3880, 4094-4198):
// the same convection with the scalar diffusivity kappa; Dirichlet boundary values sb on the prescribed faces.
__global__ void __launch_bounds__(O3_T) k3_setup_scalar(T3 t, const float *__restrict__ U, const float *__restrict__ Tin, const float *__restrict__ Bvel,
                                                        const float *__restrict__ Sbval, float kappa, const float *__restrict__ dtv,
                                                        const int32_t *__restrict__ active, float *__restrict__ Coff, float *__restrict__ A,
                                                        float *__restrict__ Rhs /* [B][NS] */) {
    const int b = blockIdx.y, g = blockIdx.x * blockDim.x + threadIdx.x, N = t.N, NS = t.NS, NB = t.NB;
    if (g >= N || (active && !active[b])) return;
    const float *u = U + (size_t)b * 3 * NS, *bv = Bvel + (size_t)b * 3 * NB, *sb = Sbval + (size_t)b * NB;
    const float dt = dtv[b], det = t.det[g];
    float diag = det / dt, r = det * Tin[(size_t)b * NS + g] / dt;
    int nb6[6];
    o3_nbrs(t, g, nb6);
#pragma unroll
    for (int f = 0; f < 6; ++f) {
        const int d = f >> 1, n = nb6[f];
        const float sig = (f & 1) ? 1.f : -1.f;
        const float mi = t.minv[d * NS + g], al = det * mi * mi;
        float off = 0.f;
        if (n >= 0) {
            const float dn = t.det[n], mn = t.minv[d * NS + n];
            const float fl = 0.5f * (det * mi * u[d * NS + g] + dn * mn * u[d * NS + n]);
            const float vc = (al * kappa + (dn * mn * mn) * kappa) * 0.5f;
            const float ff = sig * 0.5f * fl;
            diag += ff + vc;
            off = (ff - vc) / det;
        } else {
            const int j = -1 - n;
            diag += 2.f * kappa * al;
            const float bm = t.b_minv[d * NB + j];
            r += sb[j] * (-(sig * o3_bflux(t, j, d, bv)) + 2.f * kappa * (t.b_det[j] * bm * bm));
        }
        Coff[((size_t)b * 6 + f) * NS + g] = off;
    }
    A[(size_t)b * NS + g] = diag / det;
    Rhs[(size_t)b * NS + g] = r / det;
}

// Cell-centred velocity gradients (getBlockDataGradient, K.cu:2997-3043): central differences in computational space -- one-sided
// with distance 1.5 against a prescribed (Dirichlet) face, whose value sits half a cell away -- times the diagonal inverse metric.
// G[c][d] = d u_c / d x_d
__device__ __forceinline__ void o3_velocity_gradient(const T3 &t, const float *__restrict__ u, const float *__restrict__ bv, int g, float G[3][3]) {
    const int NS = t.NS, NB = t.NB;
    int nb6[6];
    o3_nbrs(t, g, nb6);
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        const int nl = nb6[2 * d], nh = nb6[2 * d + 1];
        const float dist = 2.0f - (nl < 0 ? 0.5f : 0.f) - (nh < 0 ? 0.5f : 0.f), mi = t.minv[d * NS + g];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float lo = nl >= 0 ? u[c * NS + nl] : bv[c * NB + (-1 - nl)];
            const float hi = nh >= 0 ? u[c * NS + nh] : bv[c * NB + (-1 - nh)];
            G[c][d] = ((hi - lo) / dist) * mi;
        }
    }
}
// ComputeSpatialVelocityGradients (K.cu:6460-6550): Gout[b][c][d][NS] = d u_c / d x_d -- the reference returns one NCDHW tensor per
// velocity COMPONENT c whose channel is the DIRECTION d (its Python callers name them d_dx, d_dy, d_dz, i.e. read them transposed)
__global__ void __launch_bounds__(O3_T) k3_velocity_gradients(T3 t, const float *__restrict__ U, const float *__restrict__ Bvel, float *__restrict__ Gout) {
    const int b = blockIdx.y, g = blockIdx.x * blockDim.x + threadIdx.x, NS = t.NS;
    if (g >= t.N) return;
    float G[3][3];
    o3_velocity_gradient(t, U + (size_t)b * 3 * NS, Bvel + (size_t)b * 3 * t.NB, g, G);
#pragma unroll
    for (int d = 0; d < 3; ++d)
#pragma unroll
        for (int c = 0; c < 3; ++c) Gout[(((size_t)b * 3 + c) * 3 + d) * NS + g] = G[c][d];
}
// Smagorinsky sub-grid viscosity (k_SGSviscosityIncompressibleSmagorinsky, K.cu:6913-6966) + the environment's prep function
// (tcf_env.py:441-472): Visc = nu + C delta |S| f_vd^2, |S| = sqrt(2 S_ij S_ij), delta = max_d h_d^2 (the squared longest cell edge),
// f_vd^2 the squared van Driest damping (envs/tcf/grid.py:101-125) or 1.
__global__ void __launch_bounds__(O3_T) k3_sgs_viscosity(T3 t, O3Slab sl, const float *__restrict__ U, const float *__restrict__ Bvel, float coef,
                                                         const float *__restrict__ damp /* [N] or null */, const int32_t *__restrict__ active,
                                                         float *__restrict__ Visc) {
    const int b = blockIdx.y, g = blockIdx.x * blockDim.x + threadIdx.x, NS = t.NS;
    if (g >= t.N || (active && !active[b])) return;
    float G[3][3];
    o3_velocity_gradient(t, U + (size_t)b * 3 * NS, Bvel + (size_t)b * 3 * t.NB, g, G);
    float dsum = 0.f, delta = 0.f;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
#pragma unroll
        for (int j = i; j < 3; ++j) {
            float sij = 0.5f * (G[i][j] + G[j][i]);
            sij *= sij;
            dsum += (i != j) ? 2.f * sij : sij;
        }
        const float h = 1.0f / t.minv[i * NS + g];
        delta = fmaxf(delta, h * h);
    }
    float v = coef * delta * sqrtf(2.f * dsum);
    if (damp) v *= damp[g];
    v += t.viscosity;
    Visc[(size_t)b * NS + g] = v;
    bool dirty = false;
    o3_push(sl, t, Visc, g, v, dirty);            // slabs (B == 1): the assembly reads the z-neighbours' viscosity
    if (dirty) __threadfence_system();
}

// P: off = 1/2 (alpha_P / A_P + alpha_N / A_N), diag = -sum (K.cu:4812-4978)
__global__ void __launch_bounds__(O3_T) k3_pressure_matrix(T3 t, const float *__restrict__ A, const int32_t *__restrict__ active,
                                                           float *__restrict__ Poff, float *__restrict__ Pdiag) {
    const int b = blockIdx.y, g = blockIdx.x * blockDim.x + threadIdx.x, N = t.N, NS = t.NS;
    if (g >= N || (active && !active[b])) return;
    const float *a = A + (size_t)b * NS;
    const float det = t.det[g], rA = 1.0f / a[g];
    float diag = 0.f;
    int nb6[6];
    o3_nbrs(t, g, nb6);
#pragma unroll
    for (int f = 0; f < 6; ++f) {
        const int d = f >> 1, n = nb6[f];
        float c = 0.f;
        if (n >= 0) {
            const float mi = t.minv[d * NS + g], mn = t.minv[d * NS + n];
            c = 0.5f * ((det * mi * mi) * rA + (t.det[n] * mn * mn) * (1.0f / a[n]));
        }
        Poff[((size_t)b * 6 + f) * NS + g] = c;
        diag -= c;
    }
    Pdiag[(size_t)b * NS + g] = diag;
}

// HbyA = (u/dt - H(u_prev) + S_b/det + source) / A (K.cu:5136-5255)
__global__ void __launch_bounds__(O3_T) k3_hbya(T3 t, O3Slab sl, const float *__restrict__ U, const float *__restrict__ Uprev, const float *__restrict__ Bvel,
                                                const float *__restrict__ Src, const float *__restrict__ dtv, const int32_t *__restrict__ active,
                                                const float *__restrict__ Coff, const float *__restrict__ A, float *__restrict__ Hb,
                                                const float *__restrict__ Tbuoy /* [B][NS] or null */, float beta,
                                                const float *__restrict__ Visc /* [B][NS] or null */,
                                                float *__restrict__ Poff /* with Pdiag: also assemble the pressure matrix (first corrector), or null */,
                                                float *__restrict__ Pdiag) {
    const int b = blockIdx.y, g = blockIdx.x * blockDim.x + threadIdx.x, N = t.N, NS = t.NS, NB = t.NB;
    if (g >= N || (active && !active[b])) return;
    const float *u = U + (size_t)b * 3 * NS, *up = Uprev + (size_t)b * 3 * NS, *bv = Bvel + (size_t)b * 3 * NB;
    const float dt = dtv[b], det = t.det[g], visc = Visc ? Visc[(size_t)b * NS + g] : t.viscosity, Ag = A[(size_t)b * NS + g];
    float H[3] = {0.f, 0.f, 0.f}, Sb[3] = {0.f, 0.f, 0.f};
    int nb6[6];
    o3_nbrs(t, g, nb6);
#pragma unroll
    for (int f = 0; f < 6; ++f) {
        const int d = f >> 1, n = nb6[f];
        if (n >= 0) {
            const float c = Coff[((size_t)b * 6 + f) * NS + g];
#pragma unroll
            for (int k = 0; k < 3; ++k) H[k] += c * up[k * NS + n];
        } else {
            const int j = -1 - n;
            const float sig = (f & 1) ? 1.f : -1.f, bm = t.b_minv[d * NB + j];
            const float k = -(sig * o3_bflux(t, j, d, bv)) + 2.f * visc * (t.b_det[j] * bm * bm);
#pragma unroll
            for (int c = 0; c < 3; ++c) Sb[c] += bv[c * NB + j] * k;
        }
    }
    if (Poff) {                                 // k3_pressure_matrix for this cell (same expressions, same order: bit-identical)
        const float *a = A + (size_t)b * NS;
        const float rA = 1.0f / Ag;
        float pdiag = 0.f;
#pragma unroll
        for (int f = 0; f < 6; ++f) {
            const int d = f >> 1, n = nb6[f];
            float c = 0.f;
            if (n >= 0) {
                const float mi = t.minv[d * NS + g], mn = t.minv[d * NS + n];
                c = 0.5f * ((det * mi * mi) * rA + (t.det[n] * mn * mn) * (1.0f / a[n]));
            }
            Poff[((size_t)b * 6 + f) * NS + g] = c;
            pdiag -= c;
        }
        Pdiag[(size_t)b * NS + g] = pdiag;
    }
    bool dirty = false;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float srcv = (Src ? Src[b * 4 + c] : 0.f) + ((Tbuoy && c == 1) ? Tbuoy[(size_t)b * NS + g] * beta : 0.f);
        const float hv = (u[c * NS + g] / dt - H[c] + Sb[c] / det + srcv) / Ag;
        Hb[((size_t)b * 3 + c) * NS + g] = hv;
        o3_push(sl, t, Hb + (size_t)c * NS, g, hv, dirty);
    }
    if (dirty) __threadfence_system();
}

// divergence of the contravariant face fluxes of a cell-centred field (K.cu:1567-1645, 5389-5434)
__global__ void __launch_bounds__(O3_T) k3_divergence(T3 t, const float *__restrict__ V, const float *__restrict__ Bvel,
                                                      const int32_t *__restrict__ active, float *__restrict__ Div) {
    const int b = blockIdx.y, g = blockIdx.x * blockDim.x + threadIdx.x, N = t.N, NS = t.NS, NB = t.NB;
    if (g >= N || (active && !active[b])) return;
    const float *v = V + (size_t)b * 3 * NS, *bv = Bvel + (size_t)b * 3 * NB;
    const float det = t.det[g];
    float fl[6];
    int nb6[6];
    o3_nbrs(t, g, nb6);
#pragma unroll
    for (int f = 0; f < 6; ++f) {
        const int d = f >> 1, n = nb6[f];
        if (n >= 0) fl[f] = 0.5f * (det * t.minv[d * NS + g] * v[d * NS + g] + t.det[n] * t.minv[d * NS + n] * v[d * NS + n]);
        else fl[f] = o3_bflux(t, -1 - n, d, bv);
    }
    Div[(size_t)b * NS + g] = (fl[1] - fl[0]) + (fl[3] - fl[2]) + (fl[5] - fl[4]);
}

// u = HbyA - (1/A) M^-T grad(p), central differences, one-sided at prescribed boundaries (K.cu:816-849, 5962-5995)
__global__ void __launch_bounds__(O3_T) k3_correct(T3 t, O3Slab sl, const float *__restrict__ Hb, const float *__restrict__ P, const float *__restrict__ A,
                                                   const int32_t *__restrict__ active, float *__restrict__ Uout,
                                                   float *__restrict__ Uout2 /* second destination (the state buffer after the last corrector) or null */) {
    const int b = blockIdx.y, g = blockIdx.x * blockDim.x + threadIdx.x, N = t.N, NS = t.NS;
    if (g >= N || (active && !active[b])) return;
    const float *p = P + (size_t)b * NS;
    const float pc = p[g], rA = 1.0f / A[(size_t)b * NS + g];
    bool dirty = false;
    int nb6[6];
    o3_nbrs(t, g, nb6);
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        const int nl = nb6[2 * d], nu = nb6[2 * d + 1];
        const float fac = (nl < 0 || nu < 0) ? 1.0f : 0.5f;
        const float pg = ((nu >= 0 ? p[nu] : pc) - (nl >= 0 ? p[nl] : pc)) * fac;
        const float uv = Hb[((size_t)b * 3 + d) * NS + g] - pg * t.minv[d * NS + g] * rA;
        Uout[((size_t)b * 3 + d) * NS + g] = uv;
        o3_push(sl, t, Uout + (size_t)d * NS, g, uv, dirty);
        if (Uout2) { Uout2[((size_t)b * 3 + d) * NS + g] = uv; o3_push(sl, t, Uout2 + (size_t)d * NS, g, uv, dirty); }
    }
    if (dirty) __threadfence_system();
}

__global__ void k3_copy_active(const float *__restrict__ src, float *__restrict__ dst, size_t n, const int32_t *__restrict__ active) {
    const int b = blockIdx.y;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || (active && !active[b])) return;
    dst[(size_t)b * n + i] = src[(size_t)b * n + i];
}

// ------------------------------------------------------------------------------------------------
// cooperative Krylov kernels
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float o3_row(const T3 &t, int g, const float *__restrict__ off, const float *__restrict__ dg, const float *x) {
    const int NS = t.NS;
    int n[6];
    o3_nbrs(t, g, n);
    float s = dg[g] * x[g];
#pragma unroll
    for (int f = 0; f < 6; ++f) if (n[f] >= 0) s += off[f * NS + g] * __ldcg(&x[n[f]]);
    return s;
}
// row g of the TRANSPOSED operator: the entry (n, g) is the coefficient of neighbour n's opposite face (adjoint solves, single GPU)
__device__ __forceinline__ float o3_row_t(const T3 &t, int g, const float *__restrict__ off, const float *__restrict__ dg, const float *x) {
    const int NS = t.NS;
    int n[6];
    o3_nbrs(t, g, n);
    float s = dg[g] * x[g];
#pragma unroll
    for (int f = 0; f < 6; ++f)
        if (n[f] >= 0) {
            // extruded multi-block grids: the in-plane reverse face comes from the plane's table (block connections may flip axes)
            const int rf = (t.rev && f < 4) ? (int)t.rev[f * t.plane + (g % t.plane)] : (f ^ 1);
            s += off[rf * NS + n[f]] * __ldcg(&x[n[f]]);
        }
    return s;
}

// (measured: batching four rows per thread to get more loads in flight made these kernels SLOWER -- 1.12 vs 1.01 ms per
//  substep on 1 M cells -- because the 64-register cap of 1024-thread CTAs turns the batch into local-memory spills)
// deterministic grid-wide sum of K values: block sums -> part[slot][cta][k] -> grid.sync -> fixed-order sum in every CTA;
// with slabs the per-GPU totals are then exchanged through the peers' pads (every rank adds them in rank order, so all
// ranks hold bit-identical results and take identical branches).  Because every thread fences at system scope before
// the grid.sync and the flag is written after it, a completed all-reduce also implies that all halo pushes issued
// before it have landed: it doubles as the halo hand-shake.
template <int K>
__device__ __forceinline__ void o3_grid_sum(cg::grid_group &grid, const O3Slab &sl, float (&v)[K], float *part, unsigned &rcount,
                                            unsigned long long &arc, bool &dirty, double *sm) {
    static_assert(K <= O3_PART, "partials per CTA");
    block_reduce_sum<K>(v, sm);
    float *slot = part + (size_t)(rcount & 1u) * 4096 * O3_PART;
#pragma unroll
    for (int k = 0; k < K; ++k) if (threadIdx.x == k) slot[blockIdx.x * O3_PART + k] = v[k];
    if (dirty) { __threadfence_system(); dirty = false; } else __threadfence();
    grid.sync();
    const int nb = gridDim.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (warp < K) {
        double s = 0.0;
        for (int i = lane; i < nb; i += 32) s += (double)__ldcg(&slot[i * O3_PART + warp]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) sm[warp] = s;
    }
    __syncthreads();
    if (sl.on) {
        const unsigned long long sq = ++arc;
        const int par = (int)(sq & 1ull);
        O3Pad *mine = (O3Pad *)sl.local_base;
        if (blockIdx.x == 0 && threadIdx.x < sl.world) {
            O3Pad *dst = o3_pad(sl, threadIdx.x);
            for (int k = 0; k < K; ++k) ((volatile double *)dst->ar_val[par][sl.rank])[k] = sm[k];
            __threadfence_system();
            ((volatile unsigned long long *)dst->ar_seq[par])[sl.rank] = sq;
        }
        if (threadIdx.x < sl.world) { o3_wait_ge(&mine->ar_seq[par][threadIdx.x], sq, mine); __threadfence_system(); }
        __syncthreads();
        double tot = 0.0;
        if (threadIdx.x < K) for (int q = 0; q < sl.world; ++q) tot += ((volatile double *)mine->ar_val[par][q])[threadIdx.x];
        __syncthreads();
        if (threadIdx.x < K) sm[threadIdx.x] = tot;
        __syncthreads();
    }
#pragma unroll
    for (int k = 0; k < K; ++k) v[k] = (float)sm[k];
    __syncthreads();
    ++rcount;
}
// "the vector I just updated is complete everywhere": grid barrier + (slabs) flags to / from both z-neighbours
__device__ __forceinline__ void o3_halo_sync(cg::grid_group &grid, const O3Slab &sl, unsigned long long &hc, bool &dirty) {
    if (dirty) { __threadfence_system(); dirty = false; } else __threadfence();
    grid.sync();
    if (sl.on) {
        const unsigned long long sq = ++hc;
        O3Pad *mine = (O3Pad *)sl.local_base;
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            ((volatile unsigned long long *)o3_pad(sl, sl.lower)->halo_seq)[sl.rank] = sq;
            ((volatile unsigned long long *)o3_pad(sl, sl.upper)->halo_seq)[sl.rank] = sq;
        }
        if (threadIdx.x == 0) { o3_wait_ge(&mine->halo_seq[sl.lower], sq, mine); o3_wait_ge(&mine->halo_seq[sl.upper], sq, mine); __threadfence_system(); }
        __syncthreads();
    }
}

// new BiCGStab search direction of cell i from (r, p_old, v_old): one expression for the separate update pass and for the fused product
__device__ __forceinline__ float o3_bpnew(const float *r, const float *p, const float *v, float beta, float omega, int i) {
    return fmaf(beta, fmaf(-omega, __ldcg(&v[i]), __ldcg(&p[i])), __ldcg(&r[i]));
}
// BiCGStab for NC right-hand sides in lock step (3 velocity components, or 1 passive scalar) (BICG.cu:237-376; same
// operation order as k_bicgstab)
template <int NC, int FUSED>
__global__ void __launch_bounds__(O3_CT) k3_bicgstab(T3 t, O3Slab sl, int B, const float *__restrict__ Coff, const float *__restrict__ Adiag,
                                                    const float *__restrict__ Rhs, float *X, float *work, float *part, int maxit, float tol,
                                                    int zero_init, const int32_t *__restrict__ active, int32_t *__restrict__ iters,
                                                    float *__restrict__ resid, unsigned long long *__restrict__ iter_total, int mode /* bit 0: transposed operator */) {
    cg::grid_group grid = cg::this_grid();
    __shared__ double red[32 * 6 + 8];
    const int transposed = mode & 1;
    constexpr bool fused = FUSED != 0;            // search-direction update folded into the product (4 exchanges per iteration)
    const int N = t.N, NS = t.NS;
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
    const float norm = 1.0f / sqrtf((float)t.N_global);
    unsigned rcount = 0;
    unsigned long long arc = sl.on ? sl.ctr[0] : 0ull, hc = sl.on ? sl.ctr[1] : 0ull;
    bool dirty = false;
    for (int b = 0; b < B; ++b) {
        if (active && !active[b]) continue;
        const float *off = Coff + (size_t)b * 6 * NS, *dg = Adiag + (size_t)b * NS;
        float *wb = work + (size_t)b * O3_KRY * NS;
        float *r[3], *rw[3], *p[3], *v[3], *tt[3], *x[3], *p2[3], *v2[3];
        const float *f[3];
        for (int c = 0; c < NC; ++c) {
            r[c] = wb + (size_t)(7 * c) * NS; rw[c] = r[c] + NS; p[c] = r[c] + 2 * (size_t)NS; v[c] = r[c] + 3 * (size_t)NS; tt[c] = r[c] + 4 * (size_t)NS;
            p2[c] = r[c] + 5 * (size_t)NS; v2[c] = r[c] + 6 * (size_t)NS;
            x[c] = X + ((size_t)b * NC + c) * NS; f[c] = Rhs + ((size_t)b * NC + c) * NS;
        }
        if (zero_init) { for (int c = 0; c < NC; ++c) for (int g = tid; g < N; g += nth) x[c][g] = 0.f; }
        else grid.sync();
        float acc[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        for (int c = 0; c < NC; ++c)
            for (int g = tid; g < N; g += nth) {
                const float rr = f[c][g] - (zero_init ? 0.f : (transposed ? o3_row_t(t, g, off, dg, x[c]) : o3_row(t, g, off, dg, x[c])));
                r[c][g] = rr; rw[c][g] = rr; p[c][g] = rr;
                o3_push(sl, t, p[c], g, rr, dirty);
                acc[c] += rr * rr;
            }
        o3_grid_sum<6>(grid, sl, acc, part, rcount, arc, dirty, red);
        bool done[3] = {true, true, true}; int used[3] = {-1, -1, -1}; float fin[3] = {0.f, 0.f, 0.f}, rho[3] = {1.f, 1.f, 1.f}, alpha[3] = {1.f, 1.f, 1.f}, omega[3] = {1.f, 1.f, 1.f};
        for (int c = 0; c < NC; ++c) { fin[c] = sqrtf(acc[c]) * norm; used[c] = -1; done[c] = fin[c] < tol; }
        // rho_0 = <r^, r> = <r, r> (r^ = r at the start: the same products in the same order as the sum above); later rho is reduced
        // together with the residual norm that closes the previous iteration (same operands): 5 grid-wide exchanges per iteration
        float rho_next[3] = {acc[0], acc[1], acc[2]};
        for (int i = 0; i < maxit && !(done[0] && done[1] && done[2]); ++i) {
            float beta[3] = {0.f, 0.f, 0.f};
            for (int c = 0; c < NC; ++c) if (!done[c]) {
                const float rhop = rho[c]; rho[c] = rho_next[c];
                if (i > 0) beta[c] = (rho[c] / rhop) * (alpha[c] / omega[c]);
            }
            for (int k = 0; k < 6; ++k) acc[k] = 0.f;
            if (FUSED && i > 0) {
                // p = r + beta (p - omega v) folded into the product: every thread forms the new direction of its cell AND of the six
                // neighbours from (r, p_old, v_old) -- the same fp32 expression, so the same bits -- and writes p, v = C p into the second
                // copies; the separate pass over (r, p, v) and its grid-wide "p is complete" hand-shake are gone (4 exchanges per iteration)
                for (int c = 0; c < NC; ++c) if (!done[c]) {
                    const float bt = beta[c], om = omega[c];
                    const float *rc = r[c], *pc = p[c], *vc = v[c];
                    for (int g = tid; g < N; g += nth) {
                        int nb6[6];
                        o3_nbrs(t, g, nb6);
                        const float pg = o3_bpnew(rc, pc, vc, bt, om, g);
                        float vv = dg[g] * pg;
#pragma unroll
                        for (int fc = 0; fc < 6; ++fc)
                            if (nb6[fc] >= 0) {
                                const int n = nb6[fc];
                                const float cf = transposed ? off[((t.rev && fc < 4) ? (int)t.rev[fc * t.plane + (g % t.plane)] : (fc ^ 1)) * NS + n] : off[fc * NS + g];
                                vv += cf * o3_bpnew(rc, pc, vc, bt, om, n);
                            }
                        p2[c][g] = pg; v2[c][g] = vv; acc[c] += rw[c][g] * vv;
                        o3_push(sl, t, p2[c], g, pg, dirty); o3_push(sl, t, v2[c], g, vv, dirty);
                    }
                    float *tp_ = p[c]; p[c] = p2[c]; p2[c] = tp_;
                    float *tv_ = v[c]; v[c] = v2[c]; v2[c] = tv_;
                }
            } else {
                if (i > 0) {
                    for (int c = 0; c < NC; ++c) if (!done[c])
                        for (int g = tid; g < N; g += nth) { const float pn = o3_bpnew(r[c], p[c], v[c], beta[c], omega[c], g); p[c][g] = pn; o3_push(sl, t, p[c], g, pn, dirty); }
                }
                o3_halo_sync(grid, sl, hc, dirty);
                for (int c = 0; c < NC; ++c) if (!done[c])
                    for (int g = tid; g < N; g += nth) {
                        const float vv = transposed ? o3_row_t(t, g, off, dg, p[c]) : o3_row(t, g, off, dg, p[c]);
                        v[c][g] = vv; acc[c] += rw[c][g] * vv;
                        if (fused) o3_push(sl, t, v[c], g, vv, dirty);        // the next iteration's fused product reads the neighbours' v
                    }
            }
            o3_grid_sum<6>(grid, sl, acc, part, rcount, arc, dirty, red);
            float acc2[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
            for (int c = 0; c < NC; ++c) if (!done[c]) {
                alpha[c] = rho[c] / acc[c];
                for (int g = tid; g < N; g += nth) {
                    const float rr = r[c][g] - alpha[c] * v[c][g];
                    r[c][g] = rr; x[c][g] += alpha[c] * p[c][g];
                    o3_push(sl, t, r[c], g, rr, dirty);
                    acc2[c] += rr * rr;
                }
            }
            o3_grid_sum<6>(grid, sl, acc2, part, rcount, arc, dirty, red);     // (its grid.sync also publishes r for the next product)
            for (int c = 0; c < NC; ++c) if (!done[c]) {
                const float nr = sqrtf(acc2[c]) * norm;
                used[c] = i; fin[c] = nr;
                if (!isfinite(nr) || nr < tol) done[c] = true;
            }
            for (int k = 0; k < 6; ++k) acc[k] = 0.f;
            for (int c = 0; c < NC; ++c) if (!done[c])
                for (int g = tid; g < N; g += nth) {
                    const float tv = transposed ? o3_row_t(t, g, off, dg, r[c]) : o3_row(t, g, off, dg, r[c]); tt[c][g] = tv;
                    acc[c] += tv * r[c][g]; acc[3 + c] += tv * tv;
                }
            o3_grid_sum<6>(grid, sl, acc, part, rcount, arc, dirty, red);      // every row of t = C r is complete before r is overwritten
            for (int k = 0; k < 6; ++k) acc2[k] = 0.f;
            for (int c = 0; c < NC; ++c) if (!done[c]) {
                omega[c] = acc[c] / acc[3 + c];
                for (int g = tid; g < N; g += nth) {
                    const float rg = r[c][g];
                    x[c][g] += omega[c] * rg;
                    const float rr = rg - omega[c] * tt[c][g];
                    acc2[c] += rr * rr;
                    acc2[3 + c] += rw[c][g] * rr;
                    r[c][g] = rr;
                    if (fused) o3_push(sl, t, r[c], g, rr, dirty);          // the fused product forms the neighbours' new direction from r
                }
            }
            o3_grid_sum<6>(grid, sl, acc2, part, rcount, arc, dirty, red);
            for (int c = 0; c < NC; ++c) if (!done[c]) {
                const float nr = sqrtf(acc2[c]) * norm;
                rho_next[c] = acc2[3 + c];
                fin[c] = nr;
                if (nr < tol) { done[c] = true; used[c] = i + 1; }
            }
        }
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            unsigned long long tot = 0;
            const int slot0 = NC == 1 ? 7 : 0;       // the scalar solve reports in slot 7, like the 2-D path
            for (int c = 0; c < NC; ++c) { iters[b * 8 + slot0 + c] = used[c]; resid[b * 8 + slot0 + c] = fin[c]; tot += (unsigned long long)(used[c] + 1); }
            iter_total[b * 2 + 1] += tot;
        }
        if (sl.on) for (int c = 0; c < NC; ++c) for (int g = tid; g < N; g += nth) o3_push(sl, t, x[c], g, x[c][g], dirty);
        o3_halo_sync(grid, sl, hc, dirty);       // the solution incl. the neighbours' halo planes is complete when the kernel ends
    }
    if (sl.on && blockIdx.x == 0 && threadIdx.x == 0) { sl.ctr[0] = arc; sl.ctr[1] = hc; }
}

// CG with residual reset, best-iterate tracking, 100-rising-steps cut-off and mean removal (CG.cu:225-446, SIM.py:1908-1925)
template <int TR>      // TR = 1: the transposed operator (adjoint solves; single GPU)
__global__ void __launch_bounds__(O3_CT) k3_cg(T3 t, O3Slab sl, int B, const float *__restrict__ Poff, const float *__restrict__ Pdiag,
                                              const float *__restrict__ Rhs, float *Xout, float *work, float *part, int maxit, float tol,
                                              int zero_init, int reset_steps, int slot, const int32_t *__restrict__ active,
                                              int32_t *__restrict__ iters, float *__restrict__ resid, unsigned long long *__restrict__ iter_total,
                                              float *__restrict__ pmean) {
    cg::grid_group grid = cg::this_grid();
    __shared__ double red[32 * 2 + 8];
    const int N = t.N, NS = t.NS;
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
    const float norm = 1.0f / sqrtf((float)t.N_global);
    unsigned rcount = 0;
    unsigned long long arc = sl.on ? sl.ctr[0] : 0ull, hc = sl.on ? sl.ctr[1] : 0ull;
    bool dirty = false;
    for (int b = 0; b < B; ++b) {
        if (active && !active[b]) continue;
        const float *off = Poff + (size_t)b * 6 * NS, *dg = Pdiag + (size_t)b * NS, *f = Rhs + (size_t)b * NS;
        float *wb = work + (size_t)b * O3_KRY * NS;
        float *r = wb, *p = wb + NS, *ap = wb + 2 * (size_t)NS, *best = wb + 3 * (size_t)NS, *x = wb + 4 * (size_t)NS;
        float *xo = Xout + (size_t)b * NS;
        float acc[2] = {0.f, 0.f};
        for (int g = tid; g < N; g += nth) { x[g] = zero_init ? 0.f : xo[g]; acc[1] += (f[g] != 0.f) ? 1.f : 0.f; }
        o3_grid_sum<2>(grid, sl, acc, part, rcount, arc, dirty, red);
        int used = -1; float fin = 0.f;
        if (!(acc[1] > 0.f)) {            // all-zero right-hand side -> zero result (DIFF.py:392, 489-490)
            for (int g = tid; g < N; g += nth) x[g] = 0.f;
        } else {
            acc[0] = acc[1] = 0.f;
            for (int g = tid; g < N; g += nth) {
                const float rr = f[g] - (zero_init ? 0.f : (TR ? o3_row_t(t, g, off, dg, x) : o3_row(t, g, off, dg, x)));
                r[g] = rr; p[g] = rr; acc[0] += rr * rr;
                o3_push(sl, t, p, g, rr, dirty);
            }
            o3_grid_sum<2>(grid, sl, acc, part, rcount, arc, dirty, red);
            float rho = acc[0], bestc = 0.f, lastc = 0.f; int best_it = -1, rising = 0;
            int until_reset = reset_steps > 0 ? reset_steps - 1 : -1;
            for (int i = 0; i < maxit; ++i) {
                const bool do_reset = until_reset == 0;
                if (until_reset >= 0) until_reset = do_reset ? reset_steps - 1 : until_reset - 1;
                if (do_reset) {
                    if (sl.on) for (int g = tid; g < N; g += nth) o3_push(sl, t, x, g, x[g], dirty);
                    o3_halo_sync(grid, sl, hc, dirty);
                    acc[0] = acc[1] = 0.f;
                    for (int g = tid; g < N; g += nth) { const float rr = f[g] - (TR ? o3_row_t(t, g, off, dg, x) : o3_row(t, g, off, dg, x)); r[g] = rr; acc[0] += rr * rr; }
                    o3_halo_sync(grid, sl, hc, dirty);              // every row has read the old p halos before p is overwritten
                    for (int g = tid; g < N; g += nth) { const float rr = r[g]; p[g] = rr; o3_push(sl, t, p, g, rr, dirty); }
                    o3_grid_sum<2>(grid, sl, acc, part, rcount, arc, dirty, red);
                    rho = acc[0];
                }
                acc[0] = acc[1] = 0.f;
                for (int g = tid; g < N; g += nth) { const float a = (TR ? o3_row_t(t, g, off, dg, p) : o3_row(t, g, off, dg, p)); ap[g] = a; acc[0] += p[g] * a; }
                o3_grid_sum<2>(grid, sl, acc, part, rcount, arc, dirty, red);
                const float alpha = rho / acc[0];
                acc[0] = acc[1] = 0.f;
                for (int g = tid; g < N; g += nth) {
                    x[g] += alpha * p[g];
                    const float rr = r[g] - alpha * ap[g];
                    r[g] = rr; acc[0] += rr * rr;
                }
                o3_grid_sum<2>(grid, sl, acc, part, rcount, arc, dirty, red);
                const float crit = sqrtf(acc[0]) * norm;
                if (!isfinite(crit)) { used = i; fin = crit; break; }
                if (i == 0 || crit < bestc) {
                    bestc = crit; best_it = i;
                    for (int g = tid; g < N; g += nth) best[g] = x[g];
                }
                if (i > 0 && crit >= lastc) ++rising; else rising = 0;
                lastc = crit; used = i; fin = crit;
                if (crit < tol) break;
                if (i == maxit - 1 || rising >= 100) {
                    for (int g = tid; g < N; g += nth) x[g] = best[g];
                    used = best_it; fin = bestc;
                    break;
                }
                const float rhop = rho; rho = acc[0];
                const float beta = rho / rhop;
                for (int g = tid; g < N; g += nth) { const float pn = r[g] + beta * p[g]; p[g] = pn; o3_push(sl, t, p, g, pn, dirty); }
                o3_halo_sync(grid, sl, hc, dirty);          // p complete (incl. the neighbours' halo planes) before the next product gathers it
            }
        }
        acc[0] = acc[1] = 0.f;
        for (int g = tid; g < N; g += nth) acc[0] += x[g];
        o3_grid_sum<2>(grid, sl, acc, part, rcount, arc, dirty, red);
        // (adjoint solves keep the raw iterate: with a non-symmetric singular operator the constant vector is not in the null space of
        //  its transpose, removing the mean would change P^T lam)
        const float mean = TR ? 0.f : acc[0] / (float)t.N_global;
        for (int g = tid; g < N; g += nth) { const float xv = x[g] - mean; xo[g] = xv; o3_push(sl, t, xo, g, xv, dirty); }
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            pmean[b * 8 + 3 + slot] = mean;
            iters[b * 8 + 3 + slot] = used; resid[b * 8 + 3 + slot] = fin; iter_total[b * 2] += (unsigned long long)(used + 1);
        }
        o3_halo_sync(grid, sl, hc, dirty);
    }
    if (sl.on && blockIdx.x == 0 && threadIdx.x == 0) { sl.ctr[0] = arc; sl.ctr[1] = hc; }
}

// Default variant of k3_cg on a single GPU (FGB_K3_CG_FUSED=0 switches it off): the search-direction update p <- r + beta p is
// folded into the next matrix-vector product.  Every row forms r[n] + beta * p_old[n] for itself and its six neighbours on the fly and
// stores its own new value into a second buffer, so the grid-wide synchronisation that separated the update from the product
// disappears: 2 instead of 3 grid.sync per iteration -- the solves of the extruded environments (1 000 - 2 000 iterations on 10^4 -
// 10^5 cells) are bound by exactly these synchronisations.  The expression and the summation order of every value are those of
// k3_cg, so iterates, iteration counts and results are BIT-IDENTICAL (tests/zz_first_run_worker.py cg_fused, green on a B200).
__device__ __forceinline__ float o3_pnew(const float *r, const float *pold, float beta, int i) { return __ldcg(&r[i]) + beta * __ldcg(&pold[i]); }
__global__ void __launch_bounds__(O3_CT) k3_cg_fused(T3 t, O3Slab sl, int B, const float *__restrict__ Poff, const float *__restrict__ Pdiag,
                                                    const float *__restrict__ Rhs, float *Xout, float *work, float *part, int maxit, float tol,
                                                    int zero_init, int reset_steps, int slot, const int32_t *__restrict__ active,
                                                    int32_t *__restrict__ iters, float *__restrict__ resid, unsigned long long *__restrict__ iter_total,
                                                    float *__restrict__ pmean) {
    cg::grid_group grid = cg::this_grid();
    __shared__ double red[32 * 2 + 8];
    const int N = t.N, NS = t.NS;
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
    const float norm = 1.0f / sqrtf((float)t.N_global);
    unsigned rcount = 0;
    unsigned long long arc = 0ull;
    bool dirty = false;
    for (int b = 0; b < B; ++b) {
        if (active && !active[b]) continue;
        const float *off = Poff + (size_t)b * 6 * NS, *dg = Pdiag + (size_t)b * NS, *f = Rhs + (size_t)b * NS;
        float *wb = work + (size_t)b * O3_KRY * NS;
        float *r = wb, *p = wb + NS, *ap = wb + 2 * (size_t)NS, *best = wb + 3 * (size_t)NS, *x = wb + 4 * (size_t)NS, *p2 = wb + 5 * (size_t)NS;
        float *xo = Xout + (size_t)b * NS;
        float acc[2] = {0.f, 0.f};
        for (int g = tid; g < N; g += nth) { x[g] = zero_init ? 0.f : xo[g]; acc[1] += (f[g] != 0.f) ? 1.f : 0.f; }
        o3_grid_sum<2>(grid, sl, acc, part, rcount, arc, dirty, red);
        int used = -1; float fin = 0.f;
        if (!(acc[1] > 0.f)) {
            for (int g = tid; g < N; g += nth) x[g] = 0.f;
        } else {
            acc[0] = acc[1] = 0.f;
            for (int g = tid; g < N; g += nth) {
                const float rr = f[g] - (zero_init ? 0.f : o3_row(t, g, off, dg, x));
                r[g] = rr; p[g] = rr; acc[0] += rr * rr;
            }
            o3_grid_sum<2>(grid, sl, acc, part, rcount, arc, dirty, red);
            float rho = acc[0], bestc = 0.f, lastc = 0.f, beta = 0.f; int best_it = -1, rising = 0;
            bool fresh = true;                       // p holds the search direction itself (first iteration, after a residual reset)
            int until_reset = reset_steps > 0 ? reset_steps - 1 : -1;
            for (int i = 0; i < maxit; ++i) {
                const bool do_reset = until_reset == 0;
                if (until_reset >= 0) until_reset = do_reset ? reset_steps - 1 : until_reset - 1;
                if (do_reset) {
                    __threadfence(); grid.sync();                                    // x of the previous iteration is complete
                    acc[0] = acc[1] = 0.f;
                    for (int g = tid; g < N; g += nth) { const float rr = f[g] - o3_row(t, g, off, dg, x); r[g] = rr; p[g] = rr; acc[0] += rr * rr; }
                    o3_grid_sum<2>(grid, sl, acc, part, rcount, arc, dirty, red);
                    rho = acc[0];
                    fresh = true;
                }
                acc[0] = acc[1] = 0.f;
                float *pc = p;                                                        // buffer that holds this iteration's direction
                if (fresh) {
                    for (int g = tid; g < N; g += nth) { const float a = o3_row(t, g, off, dg, p); ap[g] = a; acc[0] += p[g] * a; }
                } else {
                    for (int g = tid; g < N; g += nth) {
                        const float pg = o3_pnew(r, p, beta, g);
                        float a = dg[g] * pg;
                        int nb6[6];
                        o3_nbrs(t, g, nb6);
#pragma unroll
                        for (int fc = 0; fc < 6; ++fc) if (nb6[fc] >= 0) a += off[fc * NS + g] * o3_pnew(r, p, beta, nb6[fc]);
                        p2[g] = pg; ap[g] = a; acc[0] += pg * a;
                    }
                    pc = p2;
                }
                o3_grid_sum<2>(grid, sl, acc, part, rcount, arc, dirty, red);
                const float alpha = rho / acc[0];
                acc[0] = acc[1] = 0.f;
                for (int g = tid; g < N; g += nth) {
                    x[g] += alpha * pc[g];
                    const float rr = r[g] - alpha * ap[g];
                    r[g] = rr; acc[0] += rr * rr;
                }
                o3_grid_sum<2>(grid, sl, acc, part, rcount, arc, dirty, red);
                if (!fresh) { float *tmp = p; p = p2; p2 = tmp; }                   // the new direction becomes "p old" of the next iteration
                fresh = false;
                const float crit = sqrtf(acc[0]) * norm;
                if (!isfinite(crit)) { used = i; fin = crit; break; }
                if (i == 0 || crit < bestc) {
                    bestc = crit; best_it = i;
                    for (int g = tid; g < N; g += nth) best[g] = x[g];
                }
                if (i > 0 && crit >= lastc) ++rising; else rising = 0;
                lastc = crit; used = i; fin = crit;
                if (crit < tol) break;
                if (i == maxit - 1 || rising >= 100) {
                    for (int g = tid; g < N; g += nth) x[g] = best[g];
                    used = best_it; fin = bestc;
                    break;
                }
                const float rhop = rho; rho = acc[0];
                beta = rho / rhop;
            }
        }
        acc[0] = acc[1] = 0.f;
        for (int g = tid; g < N; g += nth) acc[0] += x[g];
        o3_grid_sum<2>(grid, sl, acc, part, rcount, arc, dirty, red);
        const float mean = acc[0] / (float)t.N_global;
        for (int g = tid; g < N; g += nth) { const float xv = x[g] - mean; xo[g] = xv; }
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            pmean[b * 8 + 3 + slot] = mean;
            iters[b * 8 + 3 + slot] = used; resid[b * 8 + 3 + slot] = fin; iter_total[b * 2] += (unsigned long long)(used + 1);
        }
        __threadfence(); grid.sync();
    }
}

// ---- stream-level slab helpers ---------------------------------------------------------------------------------------
// copy the two owned boundary planes of `ncomp` components of a field into the z-neighbours' halo planes
__global__ void __launch_bounds__(256) k3_halo_push(O3Slab sl, T3 t, float *field, int ncomp) {
    const int P = t.plane, N = t.N, NS = t.NS;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 2 * P * ncomp) return;
    const int c = i / (2 * P), r = i - c * 2 * P;
    float *f = field + (size_t)c * NS;
    if (r < P) o3_peer(sl, f, sl.lower)[N + P + r] = f[r];
    else o3_peer(sl, f, sl.upper)[N + (r - P)] = f[N - P + (r - P)];
}
// all ranks reach this point of their streams; what every rank wrote before it is visible to all after it
__global__ void k3_rank_barrier(O3Slab sl) {
    O3Pad *mine = (O3Pad *)sl.local_base;
    const unsigned long long sq = sl.ctr[2] + 1;
    __threadfence_system();
    if ((int)threadIdx.x < sl.world) {
        ((volatile unsigned long long *)o3_pad(sl, threadIdx.x)->bar_seq)[sl.rank] = sq;
        o3_wait_ge(&mine->bar_seq[threadIdx.x], sq, mine);
    }
    __syncthreads();
    __threadfence_system();
    if (threadIdx.x == 0) sl.ctr[2] = sq;
}
// all-reduce of n <= 8 floats across ranks in place (op 0: sum, 1: max), fixed rank order
__global__ void k3_rank_allreduce(O3Slab sl, float *buf, int n, int op) {
    __shared__ double res[8];
    O3Pad *mine = (O3Pad *)sl.local_base;
    const unsigned long long sq = sl.ctr[0] + 1;
    const int par = (int)(sq & 1ull);
    if ((int)threadIdx.x < sl.world) {
        O3Pad *dst = o3_pad(sl, threadIdx.x);
        for (int k = 0; k < n; ++k) ((volatile double *)dst->ar_val[par][sl.rank])[k] = (double)buf[k];
        __threadfence_system();
        ((volatile unsigned long long *)dst->ar_seq[par])[sl.rank] = sq;
        o3_wait_ge(&mine->ar_seq[par][threadIdx.x], sq, mine);
    }
    __syncthreads();
    __threadfence_system();
    if ((int)threadIdx.x < n) {
        double a = ((volatile double *)mine->ar_val[par][0])[threadIdx.x];
        for (int q = 1; q < sl.world; ++q) { const double v = ((volatile double *)mine->ar_val[par][q])[threadIdx.x]; a = op ? fmax(a, v) : a + v; }
        res[threadIdx.x] = a;
    }
    __syncthreads();
    if ((int)threadIdx.x < n) buf[threadIdx.x] = (float)res[threadIdx.x];
    if (threadIdx.x == 0) sl.ctr[0] = sq;
}
static int o3_exchange(fgb_ortho3 *b, float *field, int ncomp, cudaStream_t st) {
    if (!b->slab.on) return FGB_OK;
    const int n = 2 * b->t.plane * ncomp;
    b->launches += 2;
    k3_halo_push<<<(n + 255) / 256, 256, 0, st>>>(b->slab, b->t, field, ncomp);
    LAUNCH_CHECK("k3_halo_push");
    k3_rank_barrier<<<1, 32, 0, st>>>(b->slab);
    LAUNCH_CHECK("k3_rank_barrier");
    return FGB_OK;
}
static int o3_barrier(fgb_ortho3 *b, cudaStream_t st) {     // after a kernel that pushed its own output planes
    if (!b->slab.on) return FGB_OK;
    b->launches++;
    k3_rank_barrier<<<1, 32, 0, st>>>(b->slab);
    LAUNCH_CHECK("k3_rank_barrier");
    return FGB_OK;
}
static int o3_allreduce(fgb_ortho3 *b, float *buf, int n, int op, cudaStream_t st) {
    if (!b->slab.on || b->slab.world <= 1) return FGB_OK;
    b->launches++;
    k3_rank_allreduce<<<1, 32, 0, st>>>(b->slab, buf, n, op);
    LAUNCH_CHECK("k3_rank_allreduce");
    return FGB_OK;
}

// Slab decomposition: this handle owns z-slab `rank` of `world`; local_base / peer_bases = the symmetric regions (see O3Slab).
// The tables must describe the slab (NS = N + 2 plane, halo neighbours), every field buffer passed to the fgb_ortho3_* calls
// and the workspace must live inside the symmetric region, B must be 1.
extern "C" int fgb_ortho3_set_slab(fgb_ortho3 *b, int32_t rank, int32_t world, void *local_base, void *const *peer_bases) {
    if (!b || world < 1 || world > O3_MAXR || rank < 0 || rank >= world || !local_base || !peer_bases)
        return set_err(FGB_E_ARG, "fgb_ortho3_set_slab: bad argument");
    if (b->B != 1 || b->t.plane <= 0 || b->t.NS != b->t.N + 2 * b->t.plane)
        return set_err(FGB_E_ARG, "fgb_ortho3_set_slab: slab tables need B == 1 and NS == N + 2 * plane");
    b->slab.rank = rank; b->slab.world = world; b->slab.on = 1;
    b->slab.lower = (rank + world - 1) % world; b->slab.upper = (rank + 1) % world;
    b->slab.local_base = (char *)local_base;
    for (int q = 0; q < world; ++q) b->slab.peer_base[q] = (char *)peer_bases[q];
    b->slab.peer_base[rank] = (char *)local_base;
    b->slab.ctr = (unsigned long long *)b->slab_ctr;
    return FGB_OK;
}
extern "C" int fgb_ortho3_slab_error(fgb_ortho3 *b, int32_t *out) {
    if (!b || !out) return set_err(FGB_E_ARG, "fgb_ortho3_slab_error: null argument");
    *out = 0;
    if (!b->slab.on) return FGB_OK;
    cudaError_t ce = cudaMemcpy(out, &((O3Pad *)b->slab.local_base)->error, sizeof(int), cudaMemcpyDeviceToHost);
    return ce == cudaSuccess ? FGB_OK : set_err(FGB_E_CUDA, "fgb_ortho3_slab_error", ce);
}

// ---- symmetric memory over CUDA IPC (one allocation per rank, mapped into every peer) -------------------------------
extern "C" int fgb_ipc_alloc(size_t bytes, void **ptr, unsigned char *handle_out /*[64]*/) {
    if (!ptr || !handle_out || bytes == 0) return set_err(FGB_E_ARG, "fgb_ipc_alloc: bad argument");
    cudaError_t ce = cudaMalloc(ptr, bytes);
    if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "fgb_ipc_alloc: cudaMalloc", ce);
    ce = cudaMemset(*ptr, 0, bytes);
    if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "fgb_ipc_alloc: cudaMemset", ce);
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    ce = cudaIpcGetMemHandle((cudaIpcMemHandle_t *)handle_out, *ptr);
    if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "fgb_ipc_alloc: cudaIpcGetMemHandle", ce);
    return FGB_OK;
}
extern "C" int fgb_ipc_open(const unsigned char *handle /*[64]*/, void **peer_ptr) {
    if (!handle || !peer_ptr) return set_err(FGB_E_ARG, "fgb_ipc_open: bad argument");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    cudaError_t ce = cudaIpcOpenMemHandle(peer_ptr, h, cudaIpcMemLazyEnablePeerAccess);
    return ce == cudaSuccess ? FGB_OK : set_err(FGB_E_CUDA, "fgb_ipc_open: cudaIpcOpenMemHandle", ce);
}
extern "C" int fgb_ipc_close(void *peer_ptr) {
    cudaError_t ce = cudaIpcCloseMemHandle(peer_ptr);
    return ce == cudaSuccess ? FGB_OK : set_err(FGB_E_CUDA, "fgb_ipc_close", ce);
}
extern "C" int fgb_ipc_free(void *ptr) {
    cudaError_t ce = cudaFree(ptr);
    return ce == cudaSuccess ? FGB_OK : set_err(FGB_E_CUDA, "fgb_ipc_free", ce);
}

static int o3_coop_blocks(fgb_ortho3 *b) {
    if (b->grid_blocks > 0) return b->grid_blocks;
    int dev = 0, sms = 0, per_a = 0, per_b = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_a, k3_cg<0>, O3_CT, 0);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_b, k3_bicgstab<3, 0>, O3_CT, 0);
    if (b->cg_fused) { int per_c = 0; cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_c, k3_cg_fused, O3_CT, 0); if (per_c < per_a) per_a = per_c; }
    int blocks = (per_a > 0 && per_b > 0) ? sms : 1;     // one CTA per SM (co-residency is what a cooperative launch needs)
    const int need = (b->t.N + O3_CT - 1) / O3_CT;
    if (blocks > need) blocks = need;
    if (blocks > 4096) blocks = 4096;
    if (blocks < 1) blocks = 1;
    b->grid_blocks = blocks;
    return blocks;
}

// Smagorinsky model on / off (coefficient 0 = off).  `damping`: [N] device floats (squared van Driest factor per owned cell) or NULL;
// the pointer is kept, not copied.  tcf_env.py:441-472.
extern "C" int fgb_ortho3_set_sgs(fgb_ortho3 *b, float coefficient, const float *damping) {
    if (!b) return set_err(FGB_E_ARG, "fgb_ortho3_set_sgs: null argument");
    b->sgs_coef = coefficient; b->sgs_damp = coefficient != 0.f ? damping : nullptr;
    return FGB_OK;
}
// Refresh the per-cell viscosity from the velocity (the reference's "PRE" prep function); u's halo planes must be current on slabs.
extern "C" int fgb_ortho3_sgs_viscosity(fgb_ortho3 *b, const float *u, const float *bvel, const int32_t *active, fgb_stream_t s) {
    if (!b || !u || !bvel) return set_err(FGB_E_ARG, "fgb_ortho3_sgs_viscosity: null argument");
    if (b->sgs_coef == 0.f) return set_err(FGB_E_ARG, "fgb_ortho3_sgs_viscosity: no model set (fgb_ortho3_set_sgs)");
    b->launches++;
    k3_sgs_viscosity<<<o3_grid(b), O3_T, 0, STREAM(s)>>>(b->t, b->slab, u, bvel, b->sgs_coef, b->sgs_damp, active, b->visc);
    LAUNCH_CHECK("k3_sgs_viscosity");
    return o3_barrier(b, STREAM(s));
}
// PISOtorch.ComputeSpatialVelocityGradients (K.cu:6460-6550): grad_out[B][3 (component c)][3 (direction d)][NS] = d u_c / d x_d
extern "C" int fgb_ortho3_velocity_gradients(fgb_ortho3 *b, const float *u, const float *bvel, float *grad_out, fgb_stream_t s) {
    if (!b || !u || !bvel || !grad_out) return set_err(FGB_E_ARG, "fgb_ortho3_velocity_gradients: null argument");
    b->launches++;
    k3_velocity_gradients<<<o3_grid(b), O3_T, 0, STREAM(s)>>>(b->t, u, bvel, grad_out);
    LAUNCH_CHECK("k3_velocity_gradients");
    return FGB_OK;
}

extern "C" int fgb_ortho3_setup_advection(fgb_ortho3 *b, const float *u, const float *bvel, const float *src, const float *dt,
                                          const int32_t *active, fgb_stream_t s) {
    if (!b || !u || !bvel || !dt) return set_err(FGB_E_ARG, "fgb_ortho3_setup_advection: null argument");
    b->launches++;
    k3_setup_advection<<<o3_grid(b), O3_T, 0, STREAM(s)>>>(b->t, b->slab, u, bvel, src, dt, active, b->Coff, b->A, b->rhs, b->sc.T, b->sc.beta, b->sgs_coef != 0.f ? b->visc : nullptr);
    LAUNCH_CHECK("k3_setup_advection");
    return FGB_OK;
}

extern "C" int fgb_ortho3_solve_advection(fgb_ortho3 *b, int zero_init, const int32_t *active, fgb_stream_t s) {
    if (!b) return set_err(FGB_E_ARG, "fgb_ortho3_solve_advection: null argument");
    T3 t = b->t; O3Slab sl = b->slab; int B = b->B; const float *coff = b->Coff, *a = b->A, *rhs = b->rhs; float *x = b->ures, *work = b->kry, *part = b->part;
    int maxit = b->opt.max_iter; float tol = b->opt.adv_tol;
    int32_t *iters = b->iters; float *resid = b->resid; unsigned long long *itot = b->iter_total;
    int transposed = 0;
    void *args[] = {&t, &sl, &B, &coff, &a, &rhs, &x, &work, &part, &maxit, &tol, &zero_init, &active, &iters, &resid, &itot, &transposed};
    b->launches++;
    cudaError_t ce = cudaLaunchCooperativeKernel((b->bicg_fused ? (void *)k3_bicgstab<3, 1> : (void *)k3_bicgstab<3, 0>), dim3(o3_coop_blocks(b)), dim3(O3_CT), args, 0, STREAM(s));
    if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "cudaLaunchCooperativeKernel(k3_bicgstab)", ce);
    return FGB_OK;
}

// Passive scalar of a 3-D box (RBC3D): attach / detach the description; the substep then transports the scalar with the
// incoming velocity first and adds the buoyancy source (0, beta T, 0) to the predictor and to HbyA (SIM.py:1471-1657).
extern "C" int fgb_ortho3_set_scalar(fgb_ortho3 *b, const fgb_ortho3_scalar *sc) {
    if (!b) return set_err(FGB_E_ARG, "fgb_ortho3_set_scalar: null argument");
    if (!sc) { memset(&b->sc, 0, sizeof(b->sc)); return FGB_OK; }
    if (!sc->T || !sc->sbval) return set_err(FGB_E_ARG, "fgb_ortho3_set_scalar: T and sbval are required");
    b->sc = *sc;
    return FGB_OK;
}
// SetupAdvectionMatrix(forPassiveScalar) + SetupAdvectionScalar + SolveLinear: T <- C_s(u)^-1 rhs_s(T) (zero start)
extern "C" int fgb_ortho3_advect_scalar(fgb_ortho3 *b, const float *u, const float *bvel, const float *dt, const int32_t *active,
                                        fgb_stream_t s) {
    if (!b || !u || !bvel || !dt) return set_err(FGB_E_ARG, "fgb_ortho3_advect_scalar: null argument");
    if (!b->sc.T) return set_err(FGB_E_ARG, "fgb_ortho3_advect_scalar: no scalar attached (fgb_ortho3_set_scalar)");
    b->launches += 2;
    k3_setup_scalar<<<o3_grid(b), O3_T, 0, STREAM(s)>>>(b->t, u, b->sc.T, bvel, b->sc.sbval, b->sc.kappa, dt, active, b->Coff, b->A, b->rhs);
    LAUNCH_CHECK("k3_setup_scalar");
    T3 t = b->t; O3Slab sl = b->slab; int B = b->B; const float *coff = b->Coff, *a = b->A, *rhs = b->rhs; float *x = b->sc.T, *work = b->kry, *part = b->part;
    int maxit = b->opt.max_iter, zero_init = 1; float tol = b->opt.adv_tol;
    int32_t *iters = b->iters; float *resid = b->resid; unsigned long long *itot = b->iter_total;
    int transposed = 0;
    void *args[] = {&t, &sl, &B, &coff, &a, &rhs, &x, &work, &part, &maxit, &tol, &zero_init, &active, &iters, &resid, &itot, &transposed};
    cudaError_t ce = cudaLaunchCooperativeKernel((b->bicg_fused ? (void *)k3_bicgstab<1, 1> : (void *)k3_bicgstab<1, 0>), dim3(o3_coop_blocks(b)), dim3(O3_CT), args, 0, STREAM(s));
    if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "cudaLaunchCooperativeKernel(k3_bicgstab<1>)", ce);
    return FGB_OK;
}

extern "C" int fgb_ortho3_setup_pressure(fgb_ortho3 *b, const float *u, const float *bvel, const float *src, const float *dt,
                                         int with_matrix, const int32_t *active, fgb_stream_t s) {
    if (!b || !u || !bvel || !dt) return set_err(FGB_E_ARG, "fgb_ortho3_setup_pressure: null argument");
    cudaStream_t st = STREAM(s);
    b->launches += 2;           // (the pressure matrix of the first corrector is assembled by k3_hbya: one launch and one pass over the metrics less)
    k3_hbya<<<o3_grid(b), O3_T, 0, st>>>(b->t, b->slab, u, b->ures, bvel, src, dt, active, b->Coff, b->A, b->hbya, b->sc.T, b->sc.beta, b->sgs_coef != 0.f ? b->visc : nullptr,
                                         with_matrix ? b->Poff : nullptr, with_matrix ? b->Pdiag : nullptr);
    LAUNCH_CHECK("k3_hbya");
    { int rc = o3_barrier(b, st); if (rc) return rc; }          // k3_hbya pushed its boundary planes itself
    k3_divergence<<<o3_grid(b), O3_T, 0, st>>>(b->t, b->hbya, bvel, active, b->div);
    LAUNCH_CHECK("k3_divergence");
    return FGB_OK;
}

extern "C" int fgb_ortho3_solve_pressure(fgb_ortho3 *b, float *p_out, int zero_init, int reset_steps, int max_iter, int slot,
                                         const int32_t *active, fgb_stream_t s) {
    if (!b || !p_out) return set_err(FGB_E_ARG, "fgb_ortho3_solve_pressure: null argument");
    if (slot < 0 || slot > 4) slot = 4;
    T3 t = b->t; O3Slab sl = b->slab; int B = b->B; const float *poff = b->Poff, *pd = b->Pdiag, *rhs = b->div; float *work = b->kry, *part = b->part;
    float tol = b->opt.p_tol;
    int32_t *iters = b->iters; float *resid = b->resid; unsigned long long *itot = b->iter_total;
    float *pmean = b->pmean;
    void *args[] = {&t, &sl, &B, &poff, &pd, &rhs, &p_out, &work, &part, &max_iter, &tol, &zero_init, &reset_steps, &slot, &active, &iters, &resid, &itot, &pmean};
    b->launches++;
    const bool fused = b->cg_fused && !b->slab.on;
    cudaError_t ce = cudaLaunchCooperativeKernel(fused ? (void *)k3_cg_fused : (void *)k3_cg<0>, dim3(o3_coop_blocks(b)), dim3(O3_CT), args, 0, STREAM(s));
    if (ce != cudaSuccess) return set_err(FGB_E_CUDA, fused ? "cudaLaunchCooperativeKernel(k3_cg_fused)" : "cudaLaunchCooperativeKernel(k3_cg)", ce);
    return FGB_OK;
}

extern "C" int fgb_ortho3_correct_velocity(fgb_ortho3 *b, const float *p, float *u_out, const int32_t *active, fgb_stream_t s) {
    if (!b || !p || !u_out) return set_err(FGB_E_ARG, "fgb_ortho3_correct_velocity: null argument");
    b->launches++;
    k3_correct<<<o3_grid(b), O3_T, 0, STREAM(s)>>>(b->t, b->slab, b->hbya, p, b->A, active, u_out, nullptr);
    LAUNCH_CHECK("k3_correct");
    return FGB_OK;
}

// Simulation._PISO_split_step for D = 3 (SIM.py:1431-2002; orthogonal grid: one predictor and one pressure solve per corrector).
// With slabs every field a stencil reads across the slab boundary is pushed into the neighbours' halo planes first.
extern "C" int fgb_ortho3_piso_substep(fgb_ortho3 *b, float *u, float *p, const float *bvel, const float *src, const float *dt,
                                       const int32_t *active, fgb_stream_t s) {
    if (!b || !u || !p || !bvel || !dt) return set_err(FGB_E_ARG, "fgb_ortho3_piso_substep: null argument");
    cudaStream_t st = STREAM(s);
    int rc;
    // slabs: u is exchanged explicitly (the caller may have changed it); every later field is pushed by the kernel that
    // produces it -- A by the assembly (ordered by the predictor's reductions), u* and p by the Krylov kernels (hand-shake at
    // their end), HbyA and the corrected velocity by their kernels followed by a flag-only barrier.
    if ((rc = o3_exchange(b, u, 3, st))) return rc;
    if (b->sc.T && (rc = fgb_ortho3_advect_scalar(b, u, bvel, dt, active, s))) return rc;
    if (b->sgs_coef != 0.f && (rc = fgb_ortho3_sgs_viscosity(b, u, bvel, active, s))) return rc;
    if ((rc = fgb_ortho3_setup_advection(b, u, bvel, src, dt, active, s))) return rc;
    // non-orthogonal code path (TCF): zero start; orthogonal path (RBC, non_orthogonal=False): previous velocityResult ("ures")
    if ((rc = fgb_ortho3_solve_advection(b, b->opt.nonortho ? 1 : 0, active, s))) return rc;
    for (int cs = 0; cs < b->opt.corrector_steps; ++cs) {
        if ((rc = fgb_ortho3_setup_pressure(b, u, bvel, src, dt, cs == 0, active, s))) return rc;
        if ((rc = fgb_ortho3_solve_pressure(b, p, 1, b->opt.nonortho ? 100 : 0, b->opt.max_iter, cs, active, s))) return rc;
        // the last corrector writes the new velocity into the result buffer AND into the state (both incl. the neighbours' halo planes):
        // no separate copy kernel
        b->launches++;
        k3_correct<<<o3_grid(b), O3_T, 0, st>>>(b->t, b->slab, b->hbya, p, b->A, active, b->ures, cs + 1 == b->opt.corrector_steps ? u : nullptr);
        LAUNCH_CHECK("k3_correct");
        if ((rc = o3_barrier(b, st))) return rc;
    }
    return FGB_OK;
}


// ------------------------------------------------------------------------------------------------
// Reverse mode of the D = 3 substep (single GPU, structured box, no passive scalar / SGS).  Same construction as the 2-D adjoint
// (piso_b200.cu: k_adj_*): the forward call records a tape, the backward call runs hand-written adjoint kernels and the two
// Krylov solves with the transposed operator; the reference differentiates these grids through the same dimension-generic
// _GRAD kernels as 2-D (K.cu:3884-4090, 4403-4491, 6265-6309).  As in its differentiable backend every recorded solve starts
// from zero and the CG never resets its residual (DIFF.py:527-545, SIM.py:1436-1440).  On these orthogonal grids the previous
// pressure does not enter a substep (no deferred non-orthogonal term), so its gradient is zero.  One thread per (cell, env).
// ------------------------------------------------------------------------------------------------
// scatter of a flux-divergence adjoint: flb[f] = adjoint of face flux f of cell g;  flux_f = 1/2 (det mi_d v_d |g + det mi_d v_d |n)
__device__ __forceinline__ void o3_fluxes_adjoint(const T3 &t, int g, const int (&nb)[6], const float (&flb)[6], float *__restrict__ vb /*[3][NS]*/,
                                                  float *__restrict__ Fbb /*[NB] or null*/) {
    const int NS = t.NS;
    const float det = t.det[g];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        float own = 0.f;
#pragma unroll
        for (int s = 0; s < 2; ++s) {
            const int f = 2 * d + s, n = nb[f];
            if (n >= 0) {
                const float gq = 0.5f * flb[f];
                own += gq;
                atomicAdd(&vb[d * NS + n], gq * t.det[n] * t.minv[d * NS + n]);
            } else if (Fbb) atomicAdd(&Fbb[-1 - n], flb[f]);
        }
        atomicAdd(&vb[d * NS + g], own * det * t.minv[d * NS + g]);
    }
}
// adjoint of the corrector u_next = hb - rA * minv_d * dp_d:  hbb = unb ; rAb -= sum_d dp_d minv_d unb_d ; pb += D^T(-rA minv_d unb_d)
__global__ void __launch_bounds__(O3_T) k3_adj_correct(T3 t, const float *__restrict__ Unb, const float *__restrict__ P, const float *__restrict__ A,
                                                       float *__restrict__ Hbb, float *__restrict__ rAb, float *__restrict__ Pb, const int32_t *__restrict__ active) {
    const int b = blockIdx.y, g = blockIdx.x * blockDim.x + threadIdx.x, NS = t.NS;
    if (g >= t.N || (active && !active[b])) return;
    const float *p = P + (size_t)b * NS;
    float *pb = Pb + (size_t)b * NS;
    const float pc = p[g], rA = 1.0f / A[(size_t)b * NS + g];
    int nb6[6];
    o3_nbrs(t, g, nb6);
    float accr = 0.f;
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        const float ub = Unb[((size_t)b * 3 + d) * NS + g];
        Hbb[((size_t)b * 3 + d) * NS + g] = ub;
        const int nl = nb6[2 * d], nu = nb6[2 * d + 1];
        const float fac = (nl < 0 || nu < 0) ? 1.0f : 0.5f, mi = t.minv[d * NS + g];
        const float pg = ((nu >= 0 ? p[nu] : pc) - (nl >= 0 ? p[nl] : pc)) * fac;
        accr -= pg * mi * ub;
        const float w = -rA * mi * ub * fac;
        atomicAdd(&pb[nu >= 0 ? nu : g], w);
        atomicAdd(&pb[nl >= 0 ? nl : g], -w);
    }
    atomicAdd(&rAb[(size_t)b * NS + g], accr);
}
// x_bar = p_bar - mean(p_bar)   (adjoint of the mean removal), one CTA per environment
__global__ void __launch_bounds__(1024) k3_adj_remove_mean(int N, int NS, const float *__restrict__ Pb, float *__restrict__ Xb, const int32_t *__restrict__ active) {
    __shared__ double red[32 * 2 + 2];
    const int b = blockIdx.x;
    if (active && !active[b]) return;
    float acc[2] = {0.f, 0.f};
    for (int g = threadIdx.x; g < N; g += 1024) acc[0] += Pb[(size_t)b * NS + g];
    block_reduce_sum<2>(acc, red);
    const float m = acc[0] / (float)N;
    for (int g = threadIdx.x; g < N; g += 1024) Xb[(size_t)b * NS + g] = Pb[(size_t)b * NS + g] - m;
}
// adjoint of  div = fluxdiv(hb)  and of  x = P^-1 div  w.r.t. P(rA):  given lam = P^-1 x_bar (P is symmetric on these grids)
//   P_ij = 1/2 (alpha_i rA_i + alpha_j rA_j) across face (i, j), P_ii = - sum_j P_ij,  P_bar_ij = -lam_i x_j
__global__ void __launch_bounds__(O3_T) k3_adj_pressure_rhs(T3 t, const float *__restrict__ Lam, const float *__restrict__ X, float *__restrict__ Hbb,
                                                            float *__restrict__ Fbb, float *__restrict__ rAb, const int32_t *__restrict__ active) {
    const int b = blockIdx.y, g = blockIdx.x * blockDim.x + threadIdx.x, NS = t.NS;
    if (g >= t.N || (active && !active[b])) return;
    const float lam = Lam[(size_t)b * NS + g];
    const float *x = X + (size_t)b * NS;
    float *ra = rAb + (size_t)b * NS;
    int nb6[6];
    o3_nbrs(t, g, nb6);
    const float det = t.det[g], xg = x[g];
    float own = 0.f, flb[6];
#pragma unroll
    for (int f = 0; f < 6; ++f) {
        const int d = f >> 1, n = nb6[f];
        flb[f] = (f & 1) ? lam : -lam;
        if (n >= 0) {
            const float w = 0.5f * (-lam) * (x[n] - xg);                 // P_bar_f - P_bar_diag
            const float mi = t.minv[d * NS + g], mn = t.minv[d * NS + n];
            own += w * (det * mi * mi);
            atomicAdd(&ra[n], w * (t.det[n] * mn * mn));
        }
    }
    atomicAdd(&ra[g], own);
    o3_fluxes_adjoint(t, g, nb6, flb, Hbb + (size_t)b * 3 * NS, Fbb + (size_t)b * t.NB);
}
// adjoint of  hb = rA * (u/dt - H + Sb/det + src),  H_c = sum_f Coff_f * uprev_c[nb_f]
__global__ void __launch_bounds__(O3_T) k3_adj_hbya(T3 t, const float *__restrict__ Hbb, const float *__restrict__ Hb /*saved hb*/,
                                                    const float *__restrict__ A, const float *__restrict__ Coff, const float *__restrict__ Uprev,
                                                    const float *__restrict__ dtv, float *__restrict__ rAb, float *__restrict__ Ub,
                                                    float *__restrict__ Sbb, float *__restrict__ Coffb, float *__restrict__ Uprevb, const int32_t *__restrict__ active) {
    const int b = blockIdx.y, g = blockIdx.x * blockDim.x + threadIdx.x, NS = t.NS;
    if (g >= t.N || (active && !active[b])) return;
    const float dt = dtv[b], Ag = A[(size_t)b * NS + g], rA = 1.0f / Ag, det = t.det[g];
    int nb6[6];
    o3_nbrs(t, g, nb6);
    float accr = 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const size_t o = ((size_t)b * 3 + c) * NS;
        const float hbb = Hbb[o + g];
        accr += hbb * (Hb[o + g] * Ag);
        const float ib = rA * hbb;
        atomicAdd(&Ub[o + g], ib / dt);
        Sbb[o + g] += ib / det;
#pragma unroll
        for (int f = 0; f < 6; ++f) {
            const int n = nb6[f];
            if (n >= 0) {
                Coffb[((size_t)b * 6 + f) * NS + g] += -ib * Uprev[o + n];
                atomicAdd(&Uprevb[o + n], -ib * Coff[((size_t)b * 6 + f) * NS + g]);
            }
        }
    }
    atomicAdd(&rAb[(size_t)b * NS + g], accr);
}
// adjoint of the predictor  C ustar = rhs,  rhs = u/dt + Sb/det + src,  C = A I + Coff:  given mu = C^-T ustar_bar
__global__ void __launch_bounds__(O3_T) k3_adj_advection(T3 t, const float *__restrict__ Mu, const float *__restrict__ Ustar, const float *__restrict__ rAb,
                                                         const float *__restrict__ A, const float *__restrict__ dtv, float *__restrict__ Ab,
                                                         float *__restrict__ Coffb, float *__restrict__ Ub, float *__restrict__ Sbb, const int32_t *__restrict__ active) {
    const int b = blockIdx.y, g = blockIdx.x * blockDim.x + threadIdx.x, NS = t.NS;
    if (g >= t.N || (active && !active[b])) return;
    const float dt = dtv[b], det = t.det[g], Ag = A[(size_t)b * NS + g];
    int nb6[6];
    o3_nbrs(t, g, nb6);
    float ab = -rAb[(size_t)b * NS + g] / (Ag * Ag);                      // A_bar from rA_bar (rA = 1 / A)
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const size_t o = ((size_t)b * 3 + c) * NS;
        const float mu = Mu[o + g];
        ab += -mu * Ustar[o + g];
#pragma unroll
        for (int f = 0; f < 6; ++f) if (nb6[f] >= 0) Coffb[((size_t)b * 6 + f) * NS + g] += -mu * Ustar[o + nb6[f]];
        atomicAdd(&Ub[o + g], mu / dt);
        Sbb[o + g] += mu / det;
    }
    Ab[(size_t)b * NS + g] = ab;
}
// adjoint of the assembly (A, Coff from the face fluxes; constant viscosity) and of the boundary sources Sb
__global__ void __launch_bounds__(O3_T) k3_adj_assemble(T3 t, const float *__restrict__ Ab, const float *__restrict__ Coffb, const float *__restrict__ Sbb,
                                                        const float *__restrict__ Bvel, float *__restrict__ Ub, float *__restrict__ Bvb, float *__restrict__ Fbb,
                                                        const float *__restrict__ Visc /* [B][NS] taped per-cell viscosity or null */, const int32_t *__restrict__ active) {
    const int b = blockIdx.y, g = blockIdx.x * blockDim.x + threadIdx.x, NS = t.NS, NB = t.NB;
    if (g >= t.N || (active && !active[b])) return;
    const float det = t.det[g], diagb = Ab[(size_t)b * NS + g] / det;
    const float *bv = Bvel + (size_t)b * 3 * NB;
    int nb6[6];
    o3_nbrs(t, g, nb6);
    float flb[6];
#pragma unroll
    for (int f = 0; f < 6; ++f) {
        const float sig = (f & 1) ? 1.f : -1.f;
        flb[f] = 0.f;
        if (nb6[f] >= 0) flb[f] = 0.5f * sig * (Coffb[((size_t)b * 6 + f) * NS + g] / det + diagb);
        else {
            const int j = -1 - nb6[f], d = f >> 1;
            const float bm = t.b_minv[d * NB + j];
            const float k = -(sig * o3_bflux(t, j, d, bv)) + 2.f * (Visc ? Visc[(size_t)b * NS + g] : t.viscosity) * (t.b_det[j] * bm * bm);
            float dot = 0.f;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float sb = Sbb[((size_t)b * 3 + c) * NS + g];
                atomicAdd(&Bvb[((size_t)b * 3 + c) * NB + j], sb * k);
                dot += sb * bv[c * NB + j];
            }
            atomicAdd(&Fbb[(size_t)b * NB + j], -dot * sig);
        }
    }
    o3_fluxes_adjoint(t, g, nb6, flb, Ub + (size_t)b * 3 * NS, nullptr);
}
// Passive scalar + buoyancy (RBC3D).  The source (0, beta T_new, 0) enters the predictor right-hand side and HbyA next to S_b / det, so
// its adjoint is det * S_b_bar:  T_new_bar = T_out_bar + beta * det * S_b_bar[1]
__global__ void __launch_bounds__(O3_T) k3_adj_buoyancy(T3 t, const float *__restrict__ Sbb, const float *__restrict__ Toutb, float beta, float *__restrict__ Tnb, const int32_t *__restrict__ active) {
    const int b = blockIdx.y, g = blockIdx.x * blockDim.x + threadIdx.x, NS = t.NS;
    if (g >= t.N || (active && !active[b])) return;
    Tnb[(size_t)b * NS + g] = Toutb[(size_t)b * NS + g] + beta * t.det[g] * Sbb[((size_t)b * 3 + 1) * NS + g];
}
// adjoint of k3_setup_scalar + the scalar solve, given lam = C_s^-T T_new_bar:  A_s_bar = -lam T_new, Coff_s_bar[f] = -lam T_new[nb_f];
// rhs_s = r / det with r = det T_in / dt + sum_{prescribed f} sb (-(sig F_b) + 2 kappa alpha_b)
__global__ void __launch_bounds__(O3_T) k3_adj_scalar(T3 t, const float *__restrict__ Lam, const float *__restrict__ Tnew, const float *__restrict__ Bvel,
                                                      const float *__restrict__ Sbval, float kappa, const float *__restrict__ dtv,
                                                      float *__restrict__ Tinb, float *__restrict__ Sbvalb, float *__restrict__ Fbb, float *__restrict__ Ub, const int32_t *__restrict__ active) {
    const int b = blockIdx.y, g = blockIdx.x * blockDim.x + threadIdx.x, NS = t.NS, NB = t.NB;
    if (g >= t.N || (active && !active[b])) return;
    const float *tn = Tnew + (size_t)b * NS, *bv = Bvel + (size_t)b * 3 * NB, *sb = Sbval + (size_t)b * NB;
    const float lam = Lam[(size_t)b * NS + g], det = t.det[g], rb = lam / det;
    Tinb[(size_t)b * NS + g] = lam / dtv[b];
    const float diagb = -lam * tn[g] / det;                   // A_s = diag / det
    int nb6[6];
    o3_nbrs(t, g, nb6);
    float flb[6];
#pragma unroll
    for (int f = 0; f < 6; ++f) {
        const float sig = (f & 1) ? 1.f : -1.f;
        flb[f] = 0.f;
        if (nb6[f] >= 0) flb[f] = 0.5f * sig * (-lam * tn[nb6[f]] / det + diagb);
        else {
            const int j = -1 - nb6[f], d = f >> 1;
            const float bm = t.b_minv[d * NB + j];
            atomicAdd(&Sbvalb[(size_t)b * NB + j], rb * (-(sig * o3_bflux(t, j, d, bv)) + 2.f * kappa * (t.b_det[j] * bm * bm)));
            atomicAdd(&Fbb[(size_t)b * NB + j], -rb * sb[j] * sig);
        }
    }
    o3_fluxes_adjoint(t, g, nb6, flb, Ub + (size_t)b * 3 * NS, nullptr);
}
// adjoint of the boundary flux Fb_j = b_det minv_d bv_d (d = axis of the face): one thread per (boundary face, environment)
__global__ void k3_adj_bflux(T3 t, const float *__restrict__ Fbb, float *__restrict__ Bvb, const int32_t *__restrict__ active) {
    const int b = blockIdx.y, j = blockIdx.x * blockDim.x + threadIdx.x, NB = t.NB;
    if (j >= NB || (active && !active[b])) return;
    const int cnt[3] = {t.ny * t.nz, t.nx * t.nz, t.nx * t.ny};
    int d = -1;
#pragma unroll
    for (int f = 0; f < 6; ++f) if ((t.closed >> (f >> 1)) & 1) { if (j >= t.boff[f] && j < t.boff[f] + cnt[f >> 1]) d = f >> 1; }
    if (d < 0) return;
    Bvb[((size_t)b * 3 + d) * NB + j] += Fbb[(size_t)b * NB + j] * t.b_det[j] * t.b_minv[d * NB + j];
}

static int o3_copy(void *dst, const void *src, size_t bytes, cudaStream_t st) {
    cudaError_t ce = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, st);
    return ce == cudaSuccess ? FGB_OK : set_err(FGB_E_CUDA, "cudaMemcpyAsync (D = 3 tape)", ce);
}
// dst <- src ([B][n / B] floats) for the environments of active (NULL: a plain copy of everything)
static int o3_copy_active(fgb_ortho3 *b, float *dst, const float *src, size_t n, const int32_t *active, cudaStream_t st) {
    if (!active) return o3_copy(dst, src, n * 4, st);
    b->launches++;
    k3_copy_active<<<dim3((unsigned)((n / b->B + 255) / 256), (unsigned)b->B), 256, 0, st>>>(src, dst, n / b->B, active);
    LAUNCH_CHECK("k3_copy_active");
    return FGB_OK;
}
static int o3_adjoint_supported(const fgb_ortho3 *b, bool with_scalar) {
    if (b->slab.on || b->t.NS != b->t.N) return set_err(FGB_E_ARG, "D = 3 reverse mode: single GPU only (no slabs)");
    if (b->t.nx <= 0) return set_err(FGB_E_ARG, "D = 3 reverse mode: needs the structured-box description (tables.nx/ny/nz/closed/boff)");
    if (with_scalar != (b->sc.T != nullptr))
        return set_err(FGB_E_ARG, with_scalar ? "D = 3 reverse mode (scalar): no scalar attached (fgb_ortho3_set_scalar)"
                                              : "D = 3 reverse mode: a scalar is attached, use the _scalar entry points");
    if (b->opt.corrector_steps < 1 || b->opt.corrector_steps > 8) return set_err(FGB_E_ARG, "D = 3 reverse mode: 1..8 corrector steps");
    return FGB_OK;
}
// fgb_ortho3_piso_substep for the environments of tp->active (NULL: all) that additionally records the tape of the backward pass; a
// skipped environment keeps u, p (and T) bit for bit (every kernel and solve skips it, the final u <- ures copy is masked)
static int o3_record_impl(fgb_ortho3 *b, float *u, float *p, const float *bvel, const float *src, const float *dt,
                          const fgb_ortho3_tape *tp, const fgb_tape_scalar *stp, fgb_stream_t s) {
    if (!b || !u || !p || !bvel || !dt || !tp) return set_err(FGB_E_ARG, "fgb_ortho3_piso_substep_record: null argument");
    int rc;
    if ((rc = o3_adjoint_supported(b, stp != nullptr))) return rc;
    if (stp && (!stp->T_in || !stp->T_out || !stp->sbval_in)) return set_err(FGB_E_ARG, "fgb_ortho3_piso_substep_record_scalar: incomplete scalar tape");
    cudaStream_t st = STREAM(s);
    const size_t BN = (size_t)b->B * b->t.NS, BNB = (size_t)b->B * (b->t.NB > 0 ? b->t.NB : 1);
    const int C = b->opt.corrector_steps;
    const int32_t *act = tp->active;
    if ((rc = o3_copy(tp->u_in, u, 3 * BN * 4, st))) return rc;
    if ((rc = o3_copy(tp->bvel_in, bvel, 3 * BNB * 4, st))) return rc;
    if ((rc = o3_copy(tp->dt, dt, (size_t)b->B * 4, st))) return rc;
    if (stp) {      // scalar transport with the incoming velocity first; the predictor / HbyA then read the new temperature (buoyancy)
        if ((rc = o3_copy(stp->T_in, b->sc.T, BN * 4, st))) return rc;
        if ((rc = o3_copy(stp->sbval_in, b->sc.sbval, BNB * 4, st))) return rc;
        if ((rc = fgb_ortho3_advect_scalar(b, u, bvel, dt, act, s))) return rc;
        if ((rc = o3_copy(stp->T_out, b->sc.T, BN * 4, st))) return rc;
    }
    if (b->sgs_coef != 0.f) {     // per-cell viscosity of this substep: a CONSTANT of the graph, as in the reference (its Smagorinsky op has no
                                  // autograd wrapper: tcf_env.py:456-470 sets the block viscosity from a raw extension call)
        if (!tp->visc) return set_err(FGB_E_ARG, "fgb_ortho3_piso_substep_record: sub-grid model set, the tape needs a visc buffer");
        if ((rc = fgb_ortho3_sgs_viscosity(b, u, bvel, act, s))) return rc;
        if ((rc = o3_copy(tp->visc, b->visc, BN * 4, st))) return rc;
    }
    if ((rc = fgb_ortho3_setup_advection(b, u, bvel, src, dt, act, s))) return rc;
    if ((rc = fgb_ortho3_solve_advection(b, 1, act, s))) return rc;
    if ((rc = o3_copy(tp->ustar, b->ures, 3 * BN * 4, st))) return rc;
    if ((rc = o3_copy(tp->Coff, b->Coff, 6 * BN * 4, st))) return rc;
    if ((rc = o3_copy(tp->A, b->A, BN * 4, st))) return rc;
    for (int cs = 0; cs < C; ++cs) {
        if ((rc = fgb_ortho3_setup_pressure(b, u, bvel, src, dt, cs == 0, act, s))) return rc;
        if ((rc = o3_copy(tp->hb + (size_t)cs * 3 * BN, b->hbya, 3 * BN * 4, st))) return rc;
        if ((rc = fgb_ortho3_solve_pressure(b, p, 1, 0, b->opt.max_iter, cs, act, s))) return rc;      // zero start, no residual reset
        if ((rc = o3_copy(tp->p + (size_t)cs * BN, p, BN * 4, st))) return rc;
        if ((rc = fgb_ortho3_correct_velocity(b, p, b->ures, act, s))) return rc;
        if (cs + 1 < C && (rc = o3_copy(tp->u1 + (size_t)cs * 3 * BN, b->ures, 3 * BN * 4, st))) return rc;
    }
    return o3_copy_active(b, u, b->ures, 3 * BN, act, st);
}
extern "C" int fgb_ortho3_piso_substep_record(fgb_ortho3 *b, float *u, float *p, const float *bvel, const float *src, const float *dt,
                                              const fgb_ortho3_tape *tp, fgb_stream_t s) {
    return o3_record_impl(b, u, p, bvel, src, dt, tp, nullptr, s);
}
// with an attached scalar (RBC3D): the scalar buffer (fgb_ortho3_scalar.T) is advanced in place, as in fgb_ortho3_piso_substep
extern "C" int fgb_ortho3_piso_substep_record_scalar(fgb_ortho3 *b, float *u, float *p, const float *bvel, const float *src, const float *dt,
                                                     const fgb_ortho3_tape *tp, const fgb_tape_scalar *stp, fgb_stream_t s) {
    if (!stp) return set_err(FGB_E_ARG, "fgb_ortho3_piso_substep_record_scalar: null scalar tape");
    return o3_record_impl(b, u, p, bvel, src, dt, tp, stp, s);
}
extern "C" size_t fgb_ortho3_adjoint_workspace_bytes(const fgb_ortho3_tables *t, int32_t B) {
    const size_t BN = (size_t)B * (t->NS > 0 ? t->NS : t->N), BNB = (size_t)B * (t->NB > 0 ? t->NB : 1);
    return (size_t)(3 + 3 + 1 + 6 + 3 + 1 + 1 + 1 + 3 + 1 + 3) * align_up(BN * 4) + align_up(BNB * 4) + 8192;
}
// vector-Jacobian product of that substep: (u_out_bar, p_out_bar) -> (u_bar, bvel_bar), both overwritten; environments tp->active skips
// are skipped by every adjoint kernel and transposed solve and get the identity cotangents (k_adj_inactive)
static int o3_backward_impl(fgb_ortho3 *b, const fgb_ortho3_tape *tp, const fgb_tape_scalar *stp, const float *u_out_bar, const float *p_out_bar,
                            const float *T_out_bar, float *u_bar, float *bvel_bar, float *T_bar, float *sbval_bar, void *ws, size_t ws_bytes,
                            fgb_stream_t s) {
    if (!b || !tp || !u_out_bar || !p_out_bar || !u_bar || !bvel_bar || !ws) return set_err(FGB_E_ARG, "fgb_ortho3_piso_substep_backward: null argument");
    int rc;
    if ((rc = o3_adjoint_supported(b, stp != nullptr))) return rc;
    if (stp && (!T_out_bar || !T_bar || !sbval_bar || !stp->T_in || !stp->T_out || !stp->sbval_in))
        return set_err(FGB_E_ARG, "fgb_ortho3_piso_substep_backward_scalar: incomplete scalar arguments");
    if (ws_bytes < fgb_ortho3_adjoint_workspace_bytes(&b->t, b->B)) return set_err(FGB_E_WORKSPACE, "fgb_ortho3_piso_substep_backward: workspace too small");
    if (b->sgs_coef != 0.f && !tp->visc) return set_err(FGB_E_ARG, "fgb_ortho3_piso_substep_backward: sub-grid model set, the tape needs its visc buffer");
    cudaStream_t st = STREAM(s);
    const size_t B = b->B, NB = b->t.NB > 0 ? b->t.NB : 1, BN = B * b->t.NS;
    const int32_t *act = tp->active;
    Carver c{(char *)ws, 0};
    float *unb = c.take<float>(3 * BN), *hbb = c.take<float>(3 * BN), *rAb = c.take<float>(BN), *Coffb = c.take<float>(6 * BN);
    float *Sbb = c.take<float>(3 * BN), *pb = c.take<float>(BN), *xb = c.take<float>(BN), *lam = c.take<float>(BN);
    float *uprevb = c.take<float>(3 * BN), *Ab = c.take<float>(BN), *mu = c.take<float>(3 * BN), *Fbb = c.take<float>(B * NB);
    const int C = b->opt.corrector_steps;
    const dim3 grid = o3_grid(b);
    cudaError_t ce;
#define ZERO3(ptr, n) do { ce = cudaMemsetAsync(ptr, 0, (n) * sizeof(float), st); if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "memset", ce); } while (0)
    ZERO3(rAb, BN); ZERO3(Coffb, 6 * BN); ZERO3(Sbb, 3 * BN); ZERO3(Fbb, B * NB); ZERO3(u_bar, 3 * BN); ZERO3(bvel_bar, 3 * B * NB);
    if ((rc = o3_copy(unb, u_out_bar, 3 * BN * 4, st))) return rc;
    if ((rc = o3_copy(pb, p_out_bar, BN * 4, st))) return rc;
    b->launches++;
    k3_pressure_matrix<<<grid, O3_T, 0, st>>>(b->t, tp->A, act, b->Poff, b->Pdiag);      // the pressure matrix of this substep (function of A only)
    LAUNCH_CHECK("k3_pressure_matrix (backward)");
    for (int cs = C - 1; cs >= 0; --cs) {
        const float *hb_c = tp->hb + (size_t)cs * 3 * BN, *p_c = tp->p + (size_t)cs * BN;
        const float *uprev = cs == 0 ? tp->ustar : tp->u1 + (size_t)(cs - 1) * 3 * BN;
        b->launches += 4;
        k3_adj_correct<<<grid, O3_T, 0, st>>>(b->t, unb, p_c, tp->A, hbb, rAb, pb, act);
        LAUNCH_CHECK("k3_adj_correct");
        k3_adj_remove_mean<<<b->B, 1024, 0, st>>>(b->t.N, b->t.NS, pb, xb, act);
        LAUNCH_CHECK("k3_adj_remove_mean");
        {   // lam = P^-1 x_bar (P symmetric): the forward CG kernel, zero start, no residual reset, right-hand side xb
            T3 t = b->t; O3Slab sl = b->slab; int Bi = b->B; const float *poff = b->Poff, *pd = b->Pdiag, *rhs = xb; float *work = b->kry, *part = b->part;
            float tol = b->opt.p_tol; int max_iter = b->opt.max_iter, zero_init = 1, reset_steps = 0, slot = 4; const int32_t *active = act;
            int32_t *iters = b->iters; float *resid = b->resid; unsigned long long *itot = b->iter_total; float *out = lam;
            float *pmean = b->pmean;
            void *args[] = {&t, &sl, &Bi, &poff, &pd, &rhs, &out, &work, &part, &max_iter, &tol, &zero_init, &reset_steps, &slot, &active, &iters, &resid, &itot, &pmean};
            ce = cudaLaunchCooperativeKernel(b->cg_fused ? (void *)k3_cg_fused : (void *)k3_cg<0>, dim3(o3_coop_blocks(b)), dim3(O3_CT), args, 0, st);
            if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "cudaLaunchCooperativeKernel(k3_cg, backward)", ce);
        }
        k3_adj_pressure_rhs<<<grid, O3_T, 0, st>>>(b->t, lam, p_c, hbb, Fbb, rAb, act);
        LAUNCH_CHECK("k3_adj_pressure_rhs");
        ZERO3(pb, BN);                         // the previous pressure does not enter this corrector (zero-started solve, orthogonal grid)
        ZERO3(uprevb, 3 * BN);
        b->launches++;
        k3_adj_hbya<<<grid, O3_T, 0, st>>>(b->t, hbb, hb_c, tp->A, tp->Coff, uprev, tp->dt, rAb, u_bar, Sbb, Coffb, uprevb, act);
        LAUNCH_CHECK("k3_adj_hbya");
        float *tmp = unb; unb = uprevb; uprevb = tmp;       // gradient w.r.t. the velocity entering this corrector
    }
    {   // mu = C^-T ustar_bar
        T3 t = b->t; O3Slab sl = b->slab; int Bi = b->B; const float *coff = tp->Coff, *a = tp->A, *rhs = unb; float *x = mu, *work = b->kry, *part = b->part;
        int maxit = b->opt.max_iter, zero_init = 1, transposed = 1; float tol = b->opt.adv_tol; const int32_t *active = act;
        int32_t *iters = b->iters; float *resid = b->resid; unsigned long long *itot = b->iter_total;
        void *args[] = {&t, &sl, &Bi, &coff, &a, &rhs, &x, &work, &part, &maxit, &tol, &zero_init, &active, &iters, &resid, &itot, &transposed};
        b->launches++;
        ce = cudaLaunchCooperativeKernel((b->bicg_fused ? (void *)k3_bicgstab<3, 1> : (void *)k3_bicgstab<3, 0>), dim3(o3_coop_blocks(b)), dim3(O3_CT), args, 0, st);
        if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "cudaLaunchCooperativeKernel(k3_bicgstab, transposed)", ce);
    }
    b->launches += 3;
    k3_adj_advection<<<grid, O3_T, 0, st>>>(b->t, mu, tp->ustar, rAb, tp->A, tp->dt, Ab, Coffb, u_bar, Sbb, act);
    LAUNCH_CHECK("k3_adj_advection");
    k3_adj_assemble<<<grid, O3_T, 0, st>>>(b->t, Ab, Coffb, Sbb, tp->bvel_in, u_bar, bvel_bar, Fbb, b->sgs_coef != 0.f ? tp->visc : nullptr, act);
    LAUNCH_CHECK("k3_adj_assemble");
    if (stp) {
        // buoyancy + scalar transport (they ran BEFORE the predictor): T_new_bar from the source adjoint, one transposed scalar solve,
        // then the adjoint of the scalar assembly.  xb / lam are free again; the scalar matrix is rebuilt from the taped inputs into
        // the forward workspace (Coff / A / rhs are not read by this pass any more).
        float *Tnb = xb;
        b->launches += 4;
        k3_adj_buoyancy<<<grid, O3_T, 0, st>>>(b->t, Sbb, T_out_bar, b->sc.beta, Tnb, act);
        LAUNCH_CHECK("k3_adj_buoyancy");
        k3_setup_scalar<<<grid, O3_T, 0, st>>>(b->t, tp->u_in, stp->T_in, tp->bvel_in, stp->sbval_in, b->sc.kappa, tp->dt, act, b->Coff, b->A, b->rhs);
        LAUNCH_CHECK("k3_setup_scalar (backward)");
        {   // lam = C_s^-T T_new_bar
            T3 t = b->t; O3Slab sl = b->slab; int Bi = b->B; const float *coff = b->Coff, *a = b->A, *rhs = Tnb; float *x = lam, *work = b->kry, *part = b->part;
            int maxit = b->opt.max_iter, zero_init = 1, transposed = 1; float tol = b->opt.adv_tol; const int32_t *active = act;
            int32_t *iters = b->iters; float *resid = b->resid; unsigned long long *itot = b->iter_total;
            void *args[] = {&t, &sl, &Bi, &coff, &a, &rhs, &x, &work, &part, &maxit, &tol, &zero_init, &active, &iters, &resid, &itot, &transposed};
            ce = cudaLaunchCooperativeKernel((b->bicg_fused ? (void *)k3_bicgstab<1, 1> : (void *)k3_bicgstab<1, 0>), dim3(o3_coop_blocks(b)), dim3(O3_CT), args, 0, st);
            if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "cudaLaunchCooperativeKernel(k3_bicgstab<1>, transposed)", ce);
        }
        ZERO3(sbval_bar, B * NB);
        k3_adj_scalar<<<grid, O3_T, 0, st>>>(b->t, lam, stp->T_out, tp->bvel_in, stp->sbval_in, b->sc.kappa, tp->dt, T_bar, sbval_bar, Fbb, u_bar, act);
        LAUNCH_CHECK("k3_adj_scalar");
    }
    if (b->t.NB > 0) {
        k3_adj_bflux<<<dim3((unsigned)((b->t.NB + 127) / 128), b->B), 128, 0, st>>>(b->t, Fbb, bvel_bar, act);
        LAUNCH_CHECK("k3_adj_bflux");
    }
#undef ZERO3
    if (act) b->launches++;
    return launch_adj_inactive(act, b->B, 3, b->t.NS, u_out_bar, u_bar, nullptr, nullptr, stp ? T_out_bar : nullptr, stp ? T_bar : nullptr,
                               (int)(3 * NB), bvel_bar, stp ? (int)NB : 0, stp ? sbval_bar : nullptr, st);
}
extern "C" int fgb_ortho3_piso_substep_backward(fgb_ortho3 *b, const fgb_ortho3_tape *tp, const float *u_out_bar, const float *p_out_bar,
                                                float *u_bar, float *bvel_bar, void *ws, size_t ws_bytes, fgb_stream_t s) {
    return o3_backward_impl(b, tp, nullptr, u_out_bar, p_out_bar, nullptr, u_bar, bvel_bar, nullptr, nullptr, ws, ws_bytes, s);
}
// (u_out_bar, p_out_bar, T_out_bar) -> (u_bar, bvel_bar, T_bar, sbval_bar), all overwritten
extern "C" int fgb_ortho3_piso_substep_backward_scalar(fgb_ortho3 *b, const fgb_ortho3_tape *tp, const fgb_tape_scalar *stp, const float *u_out_bar,
                                                       const float *p_out_bar, const float *T_out_bar, float *u_bar, float *bvel_bar, float *T_bar,
                                                       float *sbval_bar, void *ws, size_t ws_bytes, fgb_stream_t s) {
    if (!stp) return set_err(FGB_E_ARG, "fgb_ortho3_piso_substep_backward_scalar: null scalar tape");
    return o3_backward_impl(b, tp, stp, u_out_bar, p_out_bar, T_out_bar, u_bar, bvel_bar, T_bar, sbval_bar, ws, ws_bytes, s);
}

// make_divergence_free (SIM.py:1320-1429): A = 1, one projection of the current velocity
extern "C" int fgb_ortho3_make_divergence_free(fgb_ortho3 *b, float *u, float *p, const float *bvel, int max_iter, fgb_stream_t s) {
    if (!b || !u || !p || !bvel) return set_err(FGB_E_ARG, "fgb_ortho3_make_divergence_free: null argument");
    cudaStream_t st = STREAM(s);
    const size_t BN = (size_t)b->B * b->t.NS;
    int rc;
    b->launches += 3;
    k_fill<<<(unsigned)((BN + 255) / 256), 256, 0, st>>>(b->A, 1.0f, BN);
    LAUNCH_CHECK("k_fill");
    if ((rc = o3_exchange(b, u, 3, st))) return rc;
    cudaError_t ce = cudaMemcpyAsync(b->hbya, u, 3 * BN * sizeof(float), cudaMemcpyDeviceToDevice, st);
    if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "memcpy hbya", ce);
    k3_pressure_matrix<<<o3_grid(b), O3_T, 0, st>>>(b->t, b->A, nullptr, b->Poff, b->Pdiag);
    LAUNCH_CHECK("k3_pressure_matrix");
    k3_divergence<<<o3_grid(b), O3_T, 0, st>>>(b->t, b->hbya, bvel, nullptr, b->div);
    LAUNCH_CHECK("k3_divergence");
    if ((rc = fgb_ortho3_solve_pressure(b, p, 1, 0, max_iter, 0, nullptr, s))) return rc;
    if ((rc = fgb_ortho3_correct_velocity(b, p, u, nullptr, s))) return rc;
    return o3_barrier(b, st);
}

// ------------------------------------------------------------------------------------------------
// stepping glue: CFL plan, channel forcing / wall shear (one CTA per environment)
// ------------------------------------------------------------------------------------------------
// Domain.getMaxVelocity(True, True): max |(M^-1 u)_d| over cells and prescribed faces (many CTAs per environment,
// combined with an integer atomicMax on the bit pattern of the non-negative float), then the adaptive plan of
// SIM.py:2004-2031 (same arithmetic as k_plan_substep) by one thread per environment.
__global__ void __launch_bounds__(256) k3_max_velocity(T3 t, const float *__restrict__ U, const float *__restrict__ Bvel, float *__restrict__ maxvel) {
    __shared__ float smf[33];
    const int b = blockIdx.y, N = t.N, NS = t.NS, NB = t.NB;
    const float *u = U + (size_t)b * 3 * NS, *bv = Bvel + (size_t)b * 3 * NB;
    float m = 0.f;
    for (int g = blockIdx.x * blockDim.x + threadIdx.x; g < N; g += gridDim.x * blockDim.x)
#pragma unroll
        for (int d = 0; d < 3; ++d) m = fmaxf(m, fabsf(t.minv[d * NS + g] * u[d * NS + g]));
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < NB; j += gridDim.x * blockDim.x)
#pragma unroll
        for (int d = 0; d < 3; ++d) m = fmaxf(m, fabsf(t.b_minv[d * NB + j] * bv[d * NB + j]));
    const float mv = block_reduce_max(m, smf);
    if (threadIdx.x == 0) atomicMax((int *)&maxvel[b], __float_as_int(mv));
}
__global__ void k3_plan_substep(int B, double *__restrict__ remaining, float *__restrict__ dtv, int32_t *__restrict__ active,
                                int32_t *__restrict__ nsub, const float *__restrict__ maxvel, int32_t *__restrict__ counters, float cfl) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const float mv = maxvel[b];
    double rem = remaining[b];
    const int act = (rem > 0.0) && !(fabs(rem) <= 1e-8);
    float dt = 0.f;
    if (act) {
        double ts;
        if (fabsf(mv) <= 1e-8f) ts = rem;
        else {
            const float mts = cfl / mv;
            if ((double)mts >= rem) ts = rem;
            else { const int k = (int)ceilf((float)rem / mts); ts = rem / (double)k; }
        }
        rem -= ts;
        dt = (float)ts;
        remaining[b] = rem;
        nsub[b] += 1;
        atomicAdd(&counters[0], 1);
    }
    dtv[b] = dt; active[b] = act;
}

// the planner of one round without a handle (differentiable rollouts plan per environment on the host's behalf: solver.py::cfl_substeps_per_env)
extern "C" int fgb_plan_substep(int32_t B, const float *maxvel, double *remaining, float cfl, float *dt, int32_t *active, int32_t *nsub,
                                int32_t *counter, fgb_stream_t s) {
    if (B < 1 || !maxvel || !remaining || !dt || !active || !nsub || !counter) return set_err(FGB_E_ARG, "fgb_plan_substep: bad argument");
    k3_plan_substep<<<(B + 127) / 128, 128, 0, STREAM(s)>>>(B, remaining, dt, active, nsub, maxvel, counter, cfl);
    LAUNCH_CHECK("k3_plan_substep");
    return FGB_OK;
}

// mean streamwise velocity of the first and last wall-normal cell layers -> wall shear stresses and the dynamic
// forcing G_x = nu/2 (u_lo/d_lo + u_hi/d_hi) (envs/tcf/grid.py:128-163, tcf_env.py:564-584).  rows: [2][n_row] cell lists.
// (two stages, both in fixed order: a single CTA per environment walking 2 x 16 384 indexed cells took 37 us on the 1 M-cell channel)
__global__ void __launch_bounds__(512) k3_wall_rows_sum(T3 t, const float *__restrict__ U, const int32_t *__restrict__ rows, int n_row,
                                                        float *__restrict__ part /* [B][gridDim.x][2] */) {
    __shared__ double red[32 * 2 + 2];
    const int b = blockIdx.y, NS = t.NS;
    const float *u = U + (size_t)b * 3 * NS;
    float a[2] = {0.f, 0.f};
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_row; i += gridDim.x * blockDim.x) { a[0] += u[rows[i]]; a[1] += u[rows[n_row + i]]; }
    block_reduce_sum<2>(a, red);
    if (threadIdx.x == 0) { part[((size_t)b * gridDim.x + blockIdx.x) * 2 + 0] = a[0]; part[((size_t)b * gridDim.x + blockIdx.x) * 2 + 1] = a[1]; }
}
__global__ void k3_wall_rows_collect(int B, int nchunk, const float *__restrict__ part, float *__restrict__ rowmean /* [B][4]: [0..1] = sums over this rank's rows */) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    double s0 = 0.0, s1 = 0.0;
    for (int c = 0; c < nchunk; ++c) { s0 += (double)part[((size_t)b * nchunk + c) * 2]; s1 += (double)part[((size_t)b * nchunk + c) * 2 + 1]; }
    rowmean[b * 4 + 0] = (float)s0; rowmean[b * 4 + 1] = (float)s1;
}
__global__ void k3_wall_rows_finish(int B, float visc, int n_row_global, float d_lo, float d_hi, float *__restrict__ rowmean,
                                    float *__restrict__ src /* [B][4] or null */, float *__restrict__ acc /* [B][2] += tau, or null */) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const float mlo = rowmean[b * 4 + 0] / (float)n_row_global, mhi = rowmean[b * 4 + 1] / (float)n_row_global;
    const float tlo = visc * mlo / d_lo, thi = visc * mhi / d_hi;
    rowmean[b * 4 + 0] = mlo; rowmean[b * 4 + 1] = mhi; rowmean[b * 4 + 2] = tlo; rowmean[b * 4 + 3] = thi;
    if (src) { src[b * 4 + 0] = (tlo + thi) * 0.5f; src[b * 4 + 1] = 0.f; src[b * 4 + 2] = 0.f; src[b * 4 + 3] = 0.f; }
    if (acc) { acc[b * 2 + 0] += tlo; acc[b * 2 + 1] += thi; }
}

extern "C" int fgb_ortho3_wall_rows(fgb_ortho3 *b, const float *u, const int32_t *rows, int n_row, float d_lo, float d_hi, int set_forcing,
                                    float *acc, fgb_stream_t s) {
    if (!b || !u || !rows || n_row <= 0) return set_err(FGB_E_ARG, "fgb_ortho3_wall_rows: bad argument");
    cudaStream_t st = STREAM(s);
    int rc;
    b->launches += 3;
    int nchunk = (n_row + 511) / 512;
    if (nchunk > 64) nchunk = 64;
    while (nchunk > 1 && (size_t)b->B * nchunk * 2 > (size_t)2 * 4096 * O3_PART) nchunk >>= 1;     // partials live in the reduction scratch
    if ((size_t)b->B * nchunk * 2 > (size_t)2 * 4096 * O3_PART) return set_err(FGB_E_ARG, "fgb_ortho3_wall_rows: too many environments");
    k3_wall_rows_sum<<<dim3((unsigned)nchunk, (unsigned)b->B), 512, 0, st>>>(b->t, u, rows, n_row, b->part);
    LAUNCH_CHECK("k3_wall_rows_sum");
    k3_wall_rows_collect<<<(b->B + 127) / 128, 128, 0, st>>>(b->B, nchunk, b->part, b->rowmean);
    LAUNCH_CHECK("k3_wall_rows_collect");
    if ((rc = o3_allreduce(b, b->rowmean, 2, 0, st))) return rc;       // slabs: every rank holds a part of both wall layers
    k3_wall_rows_finish<<<(b->B + 127) / 128, 128, 0, st>>>(b->B, b->t.viscosity, n_row * b->slab.world, d_lo, d_hi, b->rowmean,
                                                           set_forcing ? b->src : nullptr, acc);
    LAUNCH_CHECK("k3_wall_rows_finish");
    return FGB_OK;
}

// Simulation.single_step with adaptive CFL sub-stepping; channel forcing (if rows != NULL) is refreshed before every
// substep like the reference's "PRE" prep function.  Returns the number of substep rounds in *substeps_max.
extern "C" int fgb_ortho3_sim_step(fgb_ortho3 *b, float *u, float *p, const float *bvel, float dt_target, float cfl, const int32_t *rows,
                                   int n_row, float d_lo, float d_hi, int32_t *substeps_max, fgb_stream_t s) {
    if (!b || !u || !p || !bvel) return set_err(FGB_E_ARG, "fgb_ortho3_sim_step: null argument");
    cudaStream_t st = STREAM(s);
    b->launches++;
    k_set_remaining<<<(b->B + 255) / 256, 256, 0, st>>>(b->remaining, b->nsub, b->counters, (double)dt_target, b->B);
    LAUNCH_CHECK("k_set_remaining");
    int rounds = 0, rc;
    for (;; ++rounds) {
        if (rounds > 1000) return set_err(FGB_E_ARG, "fgb_ortho3_sim_step: more than 1000 adaptive substeps");
        b->launches += 3;
        k_zero_counter<<<1, 1, 0, st>>>(b->counters);
        cudaError_t ce0 = cudaMemsetAsync(b->maxvel, 0, (size_t)b->B * sizeof(float), st);
        if (ce0 != cudaSuccess) return set_err(FGB_E_CUDA, "memset maxvel", ce0);
        const int mv_blocks = (b->t.N + 256 * 8 - 1) / (256 * 8);
        k3_max_velocity<<<dim3((unsigned)(mv_blocks < 1 ? 1 : mv_blocks), (unsigned)b->B), 256, 0, st>>>(b->t, u, bvel, b->maxvel);
        LAUNCH_CHECK("k3_max_velocity");
        if ((rc = o3_allreduce(b, b->maxvel, 1, 1, st))) return rc;
        k3_plan_substep<<<(b->B + 127) / 128, 128, 0, st>>>(b->B, b->remaining, b->dt, b->active, b->nsub, b->maxvel, b->counters, cfl);
        LAUNCH_CHECK("k3_plan_substep");
        cudaError_t ce = cudaMemcpyAsync(b->h_counters, b->counters, sizeof(int32_t), cudaMemcpyDeviceToHost, st);
        if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "memcpy counters", ce);
        ce = cudaStreamSynchronize(st);
        if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "fgb_ortho3_sim_step: sync", ce);
        if (b->h_counters[0] == 0) break;
        if (rows && (rc = fgb_ortho3_wall_rows(b, u, rows, n_row, d_lo, d_hi, 1, nullptr, s))) return rc;
        if ((rc = fgb_ortho3_piso_substep(b, u, p, bvel, rows ? b->src : nullptr, b->dt, b->active, s))) return rc;
    }
    if (substeps_max) *substeps_max = rounds;
    return FGB_OK;
}
