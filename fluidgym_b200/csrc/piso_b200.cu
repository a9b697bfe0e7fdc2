// fluidgym_b200 -- batched PISO solver step for B200 (sm_100a).  See include/fluidgym_b200.h for the ABI
// and DESIGN.md for the data layout and the per-kernel rooflines.
//
// All kernels are table driven: the multi-block / curvilinear / boundary-condition logic the reference
// re-derives per cell at run time (K.cu = extensions/PISO_multiblock_cuda_kernel.cu) is resolved once on
// the host (fluidgym_b200/domain.py) into neighbour and coefficient tables shared by every environment
// of the batch.  Fields are [B][C][N] float32 with the cell index contiguous, so every access that is
// not a neighbour gather is fully coalesced; the shared tables stay L2 resident across environments.
#include <cuda_runtime.h>
#include <cooperative_groups.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <math.h>
#include <new>
#include <type_traits>

#include "fluidgym_b200.h"

namespace cg = cooperative_groups;

// ------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
static int set_err(int code, const char *msg, cudaError_t ce = cudaSuccess) {
    if (ce != cudaSuccess) snprintf(g_err, sizeof(g_err), "%s: %s", msg, cudaGetErrorString(ce));
    else snprintf(g_err, sizeof(g_err), "%s", msg);
    return code;
}
extern "C" const char *fgb_last_error(void) { return g_err; }
extern "C" int fgb_version(void) { return 1; }

#define LAUNCH_CHECK(name)                                                       \
    do {                                                                         \
        cudaError_t e_ = cudaGetLastError();                                     \
        if (e_ != cudaSuccess) return set_err(FGB_E_CUDA, name, e_);             \
    } while (0)

typedef fgb_tables Tab;

struct fgb_batch {
    Tab t;
    int B;
    fgb_options opt;
    char *ws;
    size_t ws_bytes;
    // carved buffers
    float *Coff, *A, *rhs, *ures, *Poff, *Pdiag, *hbya, *div, *pres, *kry;
    float *resid, *dt, *maxvel, *fluxbal, *pmean;
    double *remaining;
    int32_t *iters, *active, *nsub, *counters;
    int32_t *h_counters;  // pinned host mirror
    unsigned long long *iter_total;   // [B][2] accumulated Krylov iterations (cg, bicgstab)
    long long launches;               // kernels launched through this handle
    int asm_envs;                     // environments per thread in the table-heavy assembly kernels (FGB_ASM_ENVS; 1 = default kernels)
    // optional CUDA-event profiling of the solver launches (bench.py roofline)
    int prof_on;
    static const int PROF_MAX = 8192;
    cudaEvent_t *prof_ev;             // [PROF_MAX][2]
    int *prof_cls;                    // class of each recorded pair
    int prof_n;
    // environment groups (fgb_batch_set_groups / FGB_GROUPS): fgb_piso_substep runs the groups on their own streams, so that the
    // ragged end of one group's Krylov launch (environments need different iteration counts; a launch only ends with its
    // slowest environment) is filled by the other groups' kernels and the HBM-bound assembly kernels overlap the
    // latency-bound solves.  A group is a VIEW of the batch: same tables and options, per-environment pointers advanced.
    static const int MAX_GROUPS = 8;
    int groups;
    fgb_batch *parent;                // view -> the batch that owns the profiling state
    int pmean_stride;                 // row stride of pmean (= B of the owning batch)
    cudaStream_t gstream[MAX_GROUPS];
    cudaEvent_t gfork, gjoin[MAX_GROUPS];
};
enum { CLS_CG = 0, CLS_BICG = 1, CLS_ASM = 2, CLS_OTHER = 3 };
struct ProfScope {
    fgb_batch *b; cudaStream_t st; int idx;
    ProfScope(fgb_batch *b_, int cls, cudaStream_t st_) : b(b_->parent ? b_->parent : b_), st(st_), idx(-1) {
        b_->launches++;
        if (b->prof_on && b->prof_n < fgb_batch::PROF_MAX) {
            idx = b->prof_n++;
            b->prof_cls[idx] = cls;
            cudaEventRecord(b->prof_ev[2 * idx], st);
        }
    }
    ~ProfScope() { if (idx >= 0) cudaEventRecord(b->prof_ev[2 * idx + 1], st); }
};

static size_t align_up(size_t x) { return (x + 255) & ~(size_t)255; }

struct Carver {
    char *base; size_t off;
    template <typename T> T *take(size_t n) { T *p = (T *)(base + off); off = align_up(off + n * sizeof(T)); return p; }
};
static const int KRY_VECS = 12;

static void carve(fgb_batch *b, char *base, size_t *total) {
    Carver c{base, 0};
    size_t BN = (size_t)b->B * b->t.N;
    b->Coff = c.take<float>(4 * BN); b->A = c.take<float>(BN); b->rhs = c.take<float>(2 * BN);
    b->ures = c.take<float>(2 * BN); b->Poff = c.take<float>(4 * BN); b->Pdiag = c.take<float>(BN);
    b->hbya = c.take<float>(2 * BN); b->div = c.take<float>(BN); b->pres = c.take<float>(BN);
    b->kry = c.take<float>(KRY_VECS * BN);
    b->resid = c.take<float>(8 * (size_t)b->B); b->dt = c.take<float>(b->B); b->maxvel = c.take<float>(b->B);
    b->fluxbal = c.take<float>(b->B); b->pmean = c.take<float>(8 * (size_t)b->B); b->remaining = c.take<double>(b->B);
    b->iters = c.take<int32_t>(8 * (size_t)b->B); b->active = c.take<int32_t>(b->B); b->nsub = c.take<int32_t>(b->B);
    b->counters = c.take<int32_t>(64);
    b->iter_total = c.take<unsigned long long>(2 * (size_t)b->B);
    *total = c.off;
}

extern "C" size_t fgb_workspace_bytes(const fgb_tables *t, int32_t B) {
    fgb_batch tmp; memset(&tmp, 0, sizeof(tmp)); tmp.t = *t; tmp.B = B;
    size_t total = 0; carve(&tmp, nullptr, &total);
    return total;
}

static fgb_options default_options() {
    fgb_options o; o.corrector_steps = 2; o.adv_nonortho_steps = 1; o.p_nonortho_steps = 1; o.nonortho = 1;
    o.adv_tol = 1e-5f; o.p_tol = 1e-5f; o.max_iter = 5000; o.cg_impl = 0; return o;
}

extern "C" int fgb_batch_create(const fgb_tables *t, int32_t B, void *workspace, size_t workspace_bytes,
                                const fgb_options *opt, fgb_batch **out) {
    if (!t || !out || B <= 0 || t->N <= 0) return set_err(FGB_E_ARG, "fgb_batch_create: bad argument");
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0) return set_err(FGB_E_CUDA, "fgb_batch_create: no CUDA device (there is no CPU fallback)", ce);
    size_t need = fgb_workspace_bytes(t, B);
    if (!workspace || workspace_bytes < need) return set_err(FGB_E_WORKSPACE, "fgb_batch_create: workspace too small");
    fgb_batch *b = new (std::nothrow) fgb_batch();
    if (!b) return set_err(FGB_E_ARG, "fgb_batch_create: out of host memory");
    memset(b, 0, sizeof(*b));
    b->t = *t; b->B = B; b->opt = opt ? *opt : default_options();
    b->ws = (char *)workspace; b->ws_bytes = workspace_bytes;
    b->asm_envs = 1;
    if (const char *ev = getenv("FGB_ASM_ENVS")) { const int v = atoi(ev); if (v == 2 || v == 4 || v == 8) b->asm_envs = v; }
    b->groups = 1; b->pmean_stride = B;
    if (const char *ev = getenv("FGB_GROUPS")) { const int v = atoi(ev); if (v >= 1 && v <= fgb_batch::MAX_GROUPS) b->groups = v; }
    size_t total; carve(b, b->ws, &total);
    ce = cudaMallocHost(&b->h_counters, 64 * sizeof(int32_t));
    if (ce != cudaSuccess) { delete b; return set_err(FGB_E_CUDA, "cudaMallocHost", ce); }
    ce = cudaMemset(b->ws, 0, need);
    if (ce != cudaSuccess) { cudaFreeHost(b->h_counters); delete b; return set_err(FGB_E_CUDA, "cudaMemset workspace", ce); }
    *out = b;
    return FGB_OK;
}
extern "C" int fgb_batch_set_groups(fgb_batch *b, int32_t groups) {
    if (!b || groups < 1 || groups > fgb_batch::MAX_GROUPS) return set_err(FGB_E_ARG, "fgb_batch_set_groups: 1 <= groups <= 8");
    b->groups = groups;
    return FGB_OK;
}
extern "C" void fgb_batch_destroy(fgb_batch *b) {
    if (!b) return;
    if (b->gfork) {
        cudaEventDestroy(b->gfork);
        for (int g = 0; g < fgb_batch::MAX_GROUPS; ++g) { cudaEventDestroy(b->gjoin[g]); cudaStreamDestroy(b->gstream[g]); }
    }
    if (b->h_counters) cudaFreeHost(b->h_counters);
    if (b->prof_ev) { for (int i = 0; i < 2 * fgb_batch::PROF_MAX; ++i) cudaEventDestroy(b->prof_ev[i]); delete[] b->prof_ev; delete[] b->prof_cls; }
    delete b;
}
extern "C" int fgb_profile_enable(fgb_batch *b, int on) {
    if (!b) return set_err(FGB_E_ARG, "fgb_profile_enable: null argument");
    if (on && !b->prof_ev) {
        b->prof_ev = new cudaEvent_t[2 * fgb_batch::PROF_MAX];
        b->prof_cls = new int[fgb_batch::PROF_MAX];
        for (int i = 0; i < 2 * fgb_batch::PROF_MAX; ++i) {
            cudaError_t ce = cudaEventCreate(&b->prof_ev[i]);
            if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "cudaEventCreate", ce);
        }
    }
    b->prof_on = on; b->prof_n = 0;
    return FGB_OK;
}
extern "C" int fgb_profile_read(fgb_batch *b, double *ms_out, int64_t *count_out, int reset) {
    if (!b || !ms_out || !count_out) return set_err(FGB_E_ARG, "fgb_profile_read: null argument");
    for (int k = 0; k < 4; ++k) { ms_out[k] = 0.0; count_out[k] = 0; }
    cudaError_t ce = cudaDeviceSynchronize();
    if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "fgb_profile_read: sync", ce);
    for (int i = 0; i < b->prof_n; ++i) {
        float ms = 0.f;
        ce = cudaEventElapsedTime(&ms, b->prof_ev[2 * i], b->prof_ev[2 * i + 1]);
        if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "cudaEventElapsedTime", ce);
        ms_out[b->prof_cls[i]] += ms; count_out[b->prof_cls[i]] += 1;
    }
    if (reset) b->prof_n = 0;
    return FGB_OK;
}
extern "C" long long fgb_launch_count(fgb_batch *b) { return b ? b->launches : 0; }
extern "C" int fgb_batch_set_options(fgb_batch *b, const fgb_options *opt) {
    if (!b || !opt) return set_err(FGB_E_ARG, "fgb_batch_set_options: bad argument");
    b->opt = *opt; return FGB_OK;
}
extern "C" void *fgb_batch_buffer(fgb_batch *b, const char *name) {
    if (!b || !name) return nullptr;
#define BUF(n) if (!strcmp(name, #n)) return (void *)b->n;
    BUF(Coff) BUF(A) BUF(rhs) BUF(ures) BUF(Poff) BUF(Pdiag) BUF(hbya) BUF(div) BUF(pres) BUF(kry)
    BUF(pmean) BUF(iter_total) BUF(iters) BUF(resid) BUF(dt) BUF(active) BUF(remaining) BUF(nsub) BUF(maxvel) BUF(fluxbal) BUF(counters)
#undef BUF
    return nullptr;
}

// ------------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float contra_cell(const Tab &t, int k, int g, float u, float v) {
    // det * (Minv[k] . vel)   (K.cu:495-510)
    const int N = t.N;
    return t.det[g] * (t.minv[(2 * k) * N + g] * u + t.minv[(2 * k + 1) * N + g] * v);
}
__device__ __forceinline__ float bflux(const Tab &t, int j, int ax, float bu, float bv) {
    const int NB = t.NB;
    return t.b_det[j] * (t.b_minv[(2 * ax) * NB + j] * bu + t.b_minv[(2 * ax + 1) * NB + j] * bv);
}

// face fluxes of a cell-centred vector field (K.cu:1567-1645): F_f = 1/2 (U_P + +-U_N), boundary: U_b
__device__ __forceinline__ void face_fluxes(const Tab &t, int g, const float *__restrict__ vel, const float *__restrict__ bv,
                                            const int nb[4], float fl[4]) {
    const int N = t.N, NB = t.NB;
    const float ux = vel[g], uy = vel[N + g];
    const float Uc[2] = {contra_cell(t, 0, g, ux, uy), contra_cell(t, 1, g, ux, uy)};
#pragma unroll
    for (int f = 0; f < 4; ++f) {
        if (nb[f] >= 0) {
            const int fc = t.fl_comp[f * N + g];
            float velN = contra_cell(t, fc & 1, nb[f], vel[nb[f]], vel[N + nb[f]]);
            if (fc & 2) velN = -velN;
            fl[f] = (velN + Uc[f >> 1]) * 0.5f;
        } else {
            const int j = -1 - nb[f];
            fl[f] = bflux(t, j, f >> 1, bv[j], bv[NB + j]);
        }
    }
}

// Dirichlet boundary advection + diffusion sources of a cell (K.cu:4321-4380), before the division by det
__device__ __forceinline__ void boundary_source(const Tab &t, const float *__restrict__ bv, const int nb[4], float S[2]) {
    const int NB = t.NB;
    S[0] = 0.f; S[1] = 0.f;
#pragma unroll
    for (int f = 0; f < 4; ++f) {
        if (nb[f] < 0) {
            const int j = -1 - nb[f];
            const float bu = bv[j], bw = bv[NB + j];
            const float flux = bflux(t, j, f >> 1, bu, bw) * ((f & 1) ? 1.f : -1.f);
            const float visc2a = t.viscosity * 2.f * t.b_alpha[j];
            S[0] -= bu * flux; S[0] += bu * visc2a;
            S[1] -= bw * flux; S[1] += bw * visc2a;
        }
    }
}

template <int K>
__device__ __forceinline__ void block_reduce_sum(float (&v)[K], double *sm /* [32*K + K] */) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        float x = v[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
        if (lane == 0) sm[warp * K + k] = (double)x;
    }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
        for (int k = 0; k < K; ++k) {
            double x = lane < nw ? sm[lane * K + k] : 0.0;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
            if (lane == 0) sm[32 * K + k] = x;
        }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < K; ++k) v[k] = (float)sm[32 * K + k];
    __syncthreads();
}
__device__ __forceinline__ float block_reduce_max(float v, float *sm /*[33]*/) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    if (lane == 0) sm[warp] = v;
    __syncthreads();
    if (warp == 0) {
        float x = lane < nw ? sm[lane] : 0.f;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) x = fmaxf(x, __shfl_xor_sync(0xffffffffu, x, o));
        if (lane == 0) sm[32] = x;
    }
    __syncthreads();
    float r = sm[32];
    __syncthreads();
    return r;
}

// ------------------------------------------------------------------------------------------------
// assembly kernels: one thread per (cell, environment), grid = (ceil(N/256), B)
// ------------------------------------------------------------------------------------------------
// SetupAdvectionMatrix + SetupAdvectionVelocity fused (K.cu:3617-3880, 4296-4400).
__global__ void __launch_bounds__(256) k_setup_advection(Tab t, const float *__restrict__ U, const float *__restrict__ Ures,
                                                          const float *__restrict__ Bvel, const float *__restrict__ Src,
                                                          const float *__restrict__ dtv, const int32_t *__restrict__ active,
                                                          float *__restrict__ Coff, float *__restrict__ A, float *__restrict__ Rhs,
                                                          int with_matrix) {
    const int b = blockIdx.y;
    if (active && !active[b]) return;
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    const int N = t.N, NB = t.NB;
    if (g >= N) return;
    const float *u = U + (size_t)b * 2 * N, *ur = Ures + (size_t)b * 2 * N, *bv = Bvel + (size_t)b * 2 * NB;
    const float dt = dtv[b];
    const float det = t.det[g];
    int nb[4];
#pragma unroll
    for (int f = 0; f < 4; ++f) nb[f] = t.nbr[f * N + g];
    if (with_matrix) {
        float fl[4];
        face_fluxes(t, g, u, bv, nb, fl);
        float diag = det / dt + t.Cd[g];
        float *co = Coff + (size_t)b * 4 * N;
#pragma unroll
        for (int f = 0; f < 4; ++f) {
            float o = 0.f;
            if (nb[f] >= 0) {
                const float ff = ((f & 1) ? 0.5f : -0.5f) * fl[f];
                diag += ff;
                o = (ff + t.Cd[(f + 1) * N + g]) / det;
            }
            co[f * N + g] = o;
        }
        A[(size_t)b * N + g] = diag / det;
    }
    float S[2];
    boundary_source(t, bv, nb, S);
    float no0 = 0.f, no1 = 0.f;
    for (int k = 0; k < t.K_no; ++k) {
        const float w = t.no_wv[k * N + g];
        if (w != 0.f) { const int j = t.no_idx[k * N + g]; no0 += w * ur[j]; no1 += w * ur[N + j]; }
    }
    for (int k = 0; k < t.K_nob; ++k) {
        const float w = t.nob_w[k * N + g];
        if (w != 0.f) { const int j = t.nob_idx[k * N + g]; no0 += w * bv[j]; no1 += w * bv[NB + j]; }
    }
    float r0 = (det * u[g] / dt + S[0] - no0) / det;
    float r1 = (det * u[N + g] / dt + S[1] - no1) / det;
    if (Src) { r0 += Src[(size_t)b * 2 * N + g]; r1 += Src[(size_t)b * 2 * N + N + g]; }
    Rhs[(size_t)b * 2 * N + g] = r0;
    Rhs[(size_t)b * 2 * N + N + g] = r1;
}

// SetupPressureMatrix (K.cu:4812-4978): P_e = sum_j Wp[e][j] * (1/A)_j
__global__ void __launch_bounds__(256) k_setup_pressure_matrix(Tab t, const float *__restrict__ A, const int32_t *__restrict__ active,
                                                                float *__restrict__ Poff, float *__restrict__ Pdiag) {
    const int b = blockIdx.y;
    if (active && !active[b]) return;
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    const int N = t.N;
    if (g >= N) return;
    const float *a = A + (size_t)b * N;
    float rA[5];
    rA[0] = 1.0f / a[g];
#pragma unroll
    for (int f = 0; f < 4; ++f) { const int nb = t.nbr[f * N + g]; rA[f + 1] = nb >= 0 ? 1.0f / a[nb] : rA[0]; }
    float P[5];
#pragma unroll
    for (int e = 0; e < 5; ++e) {
        float s = 0.f;
#pragma unroll
        for (int j = 0; j < 5; ++j) s += t.Wp[(5 * e + j) * N + g] * rA[j];
        P[e] = s;
    }
    Pdiag[(size_t)b * N + g] = P[0];
#pragma unroll
    for (int f = 0; f < 4; ++f) Poff[(size_t)b * 4 * N + f * N + g] = P[f + 1];
}

// PISO_build_pressure_rhs (K.cu:5136-5255): HbyA = (u^n/dt - sum_nb C_nb u*_nb + S_bnd/det + src) / A
__global__ void __launch_bounds__(256) k_hbya(Tab t, const float *__restrict__ U, const float *__restrict__ Ures,
                                               const float *__restrict__ Bvel, const float *__restrict__ Src,
                                               const float *__restrict__ Coff, const float *__restrict__ A,
                                               const float *__restrict__ dtv, const int32_t *__restrict__ active,
                                               float *__restrict__ Hbya) {
    const int b = blockIdx.y;
    if (active && !active[b]) return;
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    const int N = t.N, NB = t.NB;
    if (g >= N) return;
    const float *u = U + (size_t)b * 2 * N, *ur = Ures + (size_t)b * 2 * N, *bv = Bvel + (size_t)b * 2 * NB;
    const float *co = Coff + (size_t)b * 4 * N;
    const float dt = dtv[b];
    int nb[4];
#pragma unroll
    for (int f = 0; f < 4; ++f) nb[f] = t.nbr[f * N + g];
    float H0 = 0.f, H1 = 0.f;
#pragma unroll
    for (int f = 0; f < 4; ++f)
        if (nb[f] >= 0) { const float c = co[f * N + g]; H0 += c * ur[nb[f]]; H1 += c * ur[N + nb[f]]; }
    float S[2];
    boundary_source(t, bv, nb, S);
    const float det = t.det[g];
    float s0 = S[0] / det, s1 = S[1] / det;
    if (Src) { s0 += Src[(size_t)b * 2 * N + g]; s1 += Src[(size_t)b * 2 * N + N + g]; }
    const float rD = 1.0f / A[(size_t)b * N + g];
    Hbya[(size_t)b * 2 * N + g] = rD * (u[g] / dt - H0 + s0);
    Hbya[(size_t)b * 2 * N + N + g] = rD * (u[N + g] / dt - H1 + s1);
}

// k_computePressureRHSdivergenceFromFlux + k_pressureRHSaddNonOrthoComponents (K.cu:5389-5492)
__global__ void __launch_bounds__(256) k_pressure_div(Tab t, const float *__restrict__ Hbya, const float *__restrict__ Bvel,
                                                       const float *__restrict__ Pprev, const float *__restrict__ A,
                                                       const int32_t *__restrict__ active, int nonortho, float *__restrict__ Div) {
    const int b = blockIdx.y;
    if (active && !active[b]) return;
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    const int N = t.N, NB = t.NB;
    if (g >= N) return;
    const float *h = Hbya + (size_t)b * 2 * N, *bv = Bvel + (size_t)b * 2 * NB;
    int nb[4];
#pragma unroll
    for (int f = 0; f < 4; ++f) nb[f] = t.nbr[f * N + g];
    float fl[4];
    face_fluxes(t, g, h, bv, nb, fl);
    float d = (fl[1] - fl[0]) + (fl[3] - fl[2]);
    if (nonortho) {
        const float *a = A + (size_t)b * N, *pp = Pprev + (size_t)b * N;
        float rA[5];
        rA[0] = 1.0f / a[g];
#pragma unroll
        for (int f = 0; f < 4; ++f) rA[f + 1] = nb[f] >= 0 ? 1.0f / a[nb[f]] : rA[0];
        float S = 0.f;
        for (int k = 0; k < t.K_no; ++k) {
            const float gP = t.no_gP[k * N + g], gN = t.no_gN[k * N + g];
            if (gP != 0.f || gN != 0.f) {
                const int fc = t.no_face[k * N + g];
                const float rn = fc == 0 ? rA[1] : fc == 1 ? rA[2] : fc == 2 ? rA[3] : rA[4];
                S += (gP * rA[0] + gN * rn) * pp[t.no_idx[k * N + g]];
            }
        }
        d += S;
    }
    Div[(size_t)b * N + g] = d;
}

// ------------------------------------------------------------------------------------------------
// OPT-IN variants (FGB_ASM_ENVS = 2 / 4 / 8, default 1 = the kernels above): one thread handles the same cell of E
// consecutive environments.  The geometry tables are shared by all environments, and the two kernels below read 29 / 45
// table values per cell for 6 / 5 values of per-environment state (profiles/r01_assembly_kernel_roofline_cylinder_B256.md),
// i.e. they are bound by re-reading the tables from L2 once per environment.  Here every table value is loaded once per
// thread (all loads precede the first store; the deferred-correction loop runs over the table entries outside and the
// environments inside) and the per-environment arithmetic is the same expression, statement by statement, as in
// k_setup_pressure_matrix / k_pressure_div, so results are bit-identical (tests/test_gpu_extruded.py::test_opt_in_kernels[asm2|asm4|asm8] on a B200).  Selected only
// when the environment variable FGB_ASM_ENVS is set: measured without gain on the headline batch (DESIGN.md section 6).
template <int E>
__global__ void __launch_bounds__(256) k_setup_pressure_matrix_multi(Tab t, int B, const float *__restrict__ A,
                                                                      const int32_t *__restrict__ active, float *__restrict__ Poff,
                                                                      float *__restrict__ Pdiag) {
    const int b0 = blockIdx.y * E;
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    const int N = t.N;
    if (g >= N) return;
    int nb[4];
#pragma unroll
    for (int f = 0; f < 4; ++f) nb[f] = t.nbr[f * N + g];
    float W[25];
#pragma unroll
    for (int q = 0; q < 25; ++q) W[q] = t.Wp[q * N + g];
    float P[E][5];
    bool on[E];
#pragma unroll
    for (int e = 0; e < E; ++e) {
        const int b = b0 + e;
        on[e] = b < B && !(active && !active[b]);
        if (!on[e]) continue;
        const float *a = A + (size_t)b * N;
        float rA[5];
        rA[0] = 1.0f / a[g];
#pragma unroll
        for (int f = 0; f < 4; ++f) rA[f + 1] = nb[f] >= 0 ? 1.0f / a[nb[f]] : rA[0];
#pragma unroll
        for (int q = 0; q < 5; ++q) {
            float sacc = 0.f;
#pragma unroll
            for (int j = 0; j < 5; ++j) sacc += W[5 * q + j] * rA[j];
            P[e][q] = sacc;
        }
    }
#pragma unroll
    for (int e = 0; e < E; ++e) {
        if (!on[e]) continue;
        const int b = b0 + e;
        Pdiag[(size_t)b * N + g] = P[e][0];
#pragma unroll
        for (int f = 0; f < 4; ++f) Poff[(size_t)b * 4 * N + f * N + g] = P[e][f + 1];
    }
}

template <int E>
__global__ void __launch_bounds__(256) k_pressure_div_multi(Tab t, int B, const float *__restrict__ Hbya, const float *__restrict__ Bvel,
                                                             const float *__restrict__ Pprev, const float *__restrict__ A,
                                                             const int32_t *__restrict__ active, int nonortho, float *__restrict__ Div) {
    const int b0 = blockIdx.y * E;
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    const int N = t.N, NB = t.NB;
    if (g >= N) return;
    // tables of this cell, loaded once for all E environments (the arithmetic below is face_fluxes / contra_cell / bflux verbatim)
    int nb[4], src[4], fcm[4];
    float fdet[4], fma[4], fmb[4];
    const float det_g = t.det[g], m0 = t.minv[g], m1 = t.minv[N + g], m2 = t.minv[2 * N + g], m3 = t.minv[3 * N + g];
#pragma unroll
    for (int f = 0; f < 4; ++f) {
        nb[f] = t.nbr[f * N + g];
        if (nb[f] >= 0) {
            const int fc = t.fl_comp[f * N + g], k = fc & 1, n = nb[f];
            fcm[f] = fc; src[f] = n;
            fdet[f] = t.det[n]; fma[f] = t.minv[(2 * k) * N + n]; fmb[f] = t.minv[(2 * k + 1) * N + n];
        } else {
            const int j = -1 - nb[f], ax = f >> 1;
            fcm[f] = 0; src[f] = j;
            fdet[f] = t.b_det[j]; fma[f] = t.b_minv[(2 * ax) * NB + j]; fmb[f] = t.b_minv[(2 * ax + 1) * NB + j];
        }
    }
    float d[E], rA[E][5];
    bool on[E];
#pragma unroll
    for (int e = 0; e < E; ++e) {
        const int b = b0 + e;
        on[e] = b < B && !(active && !active[b]);
        d[e] = 0.f;
        if (!on[e]) continue;
        const float *vel = Hbya + (size_t)b * 2 * N, *bv = Bvel + (size_t)b * 2 * NB;
        const float ux = vel[g], uy = vel[N + g];
        const float Uc[2] = {det_g * (m0 * ux + m1 * uy), det_g * (m2 * ux + m3 * uy)};
        float fl[4];
#pragma unroll
        for (int f = 0; f < 4; ++f) {
            if (nb[f] >= 0) {
                float velN = fdet[f] * (fma[f] * vel[src[f]] + fmb[f] * vel[N + src[f]]);
                if (fcm[f] & 2) velN = -velN;
                fl[f] = (velN + Uc[f >> 1]) * 0.5f;
            } else {
                fl[f] = fdet[f] * (fma[f] * bv[src[f]] + fmb[f] * bv[NB + src[f]]);
            }
        }
        d[e] = (fl[1] - fl[0]) + (fl[3] - fl[2]);
        if (nonortho) {
            const float *a = A + (size_t)b * N;
            rA[e][0] = 1.0f / a[g];
#pragma unroll
            for (int f = 0; f < 4; ++f) rA[e][f + 1] = nb[f] >= 0 ? 1.0f / a[nb[f]] : rA[e][0];
        }
    }
    if (nonortho) {
        float S[E];
#pragma unroll
        for (int e = 0; e < E; ++e) S[e] = 0.f;
        for (int k = 0; k < t.K_no; ++k) {
            const float gP = t.no_gP[k * N + g], gN = t.no_gN[k * N + g];
            if (gP != 0.f || gN != 0.f) {
                const int fc = t.no_face[k * N + g];
                const int j = t.no_idx[k * N + g];
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    if (!on[e]) continue;
                    const float rn = fc == 0 ? rA[e][1] : fc == 1 ? rA[e][2] : fc == 2 ? rA[e][3] : rA[e][4];
                    S[e] += (gP * rA[e][0] + gN * rn) * Pprev[(size_t)(b0 + e) * N + j];
                }
            }
        }
#pragma unroll
        for (int e = 0; e < E; ++e) d[e] += S[e];
    }
#pragma unroll
    for (int e = 0; e < E; ++e)
        if (on[e]) Div[(size_t)(b0 + e) * N + g] = d[e];
}

// k_setup_advection for E environments per thread (opt-in, see above): 30 table values per cell for 9 values of state.
template <int E>
__global__ void __launch_bounds__(256) k_setup_advection_multi(Tab t, int B, const float *__restrict__ U, const float *__restrict__ Ures,
                                                                const float *__restrict__ Bvel, const float *__restrict__ Src,
                                                                const float *__restrict__ dtv, const int32_t *__restrict__ active,
                                                                float *__restrict__ Coff, float *__restrict__ A, float *__restrict__ Rhs,
                                                                int with_matrix) {
    const int b0 = blockIdx.y * E;
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    const int N = t.N, NB = t.NB;
    if (g >= N) return;
    int nb[4], src[4], fcm[4];
    float fdet[4], fma[4], fmb[4], falpha[4], cd[5];
    const float det = t.det[g], m0 = t.minv[g], m1 = t.minv[N + g], m2 = t.minv[2 * N + g], m3 = t.minv[3 * N + g];
#pragma unroll
    for (int q = 0; q < 5; ++q) cd[q] = with_matrix ? t.Cd[q * N + g] : 0.f;
#pragma unroll
    for (int f = 0; f < 4; ++f) {
        nb[f] = t.nbr[f * N + g];
        falpha[f] = 0.f;
        if (nb[f] >= 0) {
            const int fc = with_matrix ? t.fl_comp[f * N + g] : 0, k = fc & 1, n = nb[f];
            fcm[f] = fc; src[f] = n;
            fdet[f] = with_matrix ? t.det[n] : 0.f;
            fma[f] = with_matrix ? t.minv[(2 * k) * N + n] : 0.f; fmb[f] = with_matrix ? t.minv[(2 * k + 1) * N + n] : 0.f;
        } else {
            const int j = -1 - nb[f], ax = f >> 1;
            fcm[f] = 0; src[f] = j;
            fdet[f] = t.b_det[j]; fma[f] = t.b_minv[(2 * ax) * NB + j]; fmb[f] = t.b_minv[(2 * ax + 1) * NB + j];
            falpha[f] = t.b_alpha[j];
        }
    }
    bool on[E];
    float dt[E], S0[E], S1[E], no0[E], no1[E];
#pragma unroll
    for (int e = 0; e < E; ++e) {
        const int b = b0 + e;
        on[e] = b < B && !(active && !active[b]);
        no0[e] = 0.f; no1[e] = 0.f; S0[e] = 0.f; S1[e] = 0.f; dt[e] = 1.f;
        if (!on[e]) continue;
        const float *u = U + (size_t)b * 2 * N, *bv = Bvel + (size_t)b * 2 * NB;
        dt[e] = dtv[b];
        if (with_matrix) {                                                             // face_fluxes + matrix rows, verbatim
            const float ux = u[g], uy = u[N + g];
            const float Uc[2] = {det * (m0 * ux + m1 * uy), det * (m2 * ux + m3 * uy)};
            float diag = det / dt[e] + cd[0];
            float *co = Coff + (size_t)b * 4 * N;
#pragma unroll
            for (int f = 0; f < 4; ++f) {
                float o = 0.f;
                if (nb[f] >= 0) {
                    float velN = fdet[f] * (fma[f] * u[src[f]] + fmb[f] * u[N + src[f]]);
                    if (fcm[f] & 2) velN = -velN;
                    const float flf = (velN + Uc[f >> 1]) * 0.5f;
                    const float ff = ((f & 1) ? 0.5f : -0.5f) * flf;
                    diag += ff;
                    o = (ff + cd[f + 1]) / det;
                }
                co[f * N + g] = o;
            }
            A[(size_t)b * N + g] = diag / det;
        }
#pragma unroll
        for (int f = 0; f < 4; ++f) {                                                  // boundary_source, verbatim
            if (nb[f] < 0) {
                const float bu = bv[src[f]], bw = bv[NB + src[f]];
                const float flux = fdet[f] * (fma[f] * bu + fmb[f] * bw) * ((f & 1) ? 1.f : -1.f);
                const float visc2a = t.viscosity * 2.f * falpha[f];
                S0[e] -= bu * flux; S0[e] += bu * visc2a;
                S1[e] -= bw * flux; S1[e] += bw * visc2a;
            }
        }
    }
    for (int k = 0; k < t.K_no; ++k) {
        const float w = t.no_wv[k * N + g];
        if (w != 0.f) {
            const int j = t.no_idx[k * N + g];
#pragma unroll
            for (int e = 0; e < E; ++e)
                if (on[e]) { const float *ur = Ures + (size_t)(b0 + e) * 2 * N; no0[e] += w * ur[j]; no1[e] += w * ur[N + j]; }
        }
    }
    for (int k = 0; k < t.K_nob; ++k) {
        const float w = t.nob_w[k * N + g];
        if (w != 0.f) {
            const int j = t.nob_idx[k * N + g];
#pragma unroll
            for (int e = 0; e < E; ++e)
                if (on[e]) { const float *bv = Bvel + (size_t)(b0 + e) * 2 * NB; no0[e] += w * bv[j]; no1[e] += w * bv[NB + j]; }
        }
    }
#pragma unroll
    for (int e = 0; e < E; ++e) {
        if (!on[e]) continue;
        const int b = b0 + e;
        const float *u = U + (size_t)b * 2 * N;
        float r0 = (det * u[g] / dt[e] + S0[e] - no0[e]) / det;
        float r1 = (det * u[N + g] / dt[e] + S1[e] - no1[e]) / det;
        if (Src) { r0 += Src[(size_t)b * 2 * N + g]; r1 += Src[(size_t)b * 2 * N + N + g]; }
        Rhs[(size_t)b * 2 * N + g] = r0;
        Rhs[(size_t)b * 2 * N + N + g] = r1;
    }
}

// PISO_update_velocity (K.cu:816-849, 5962-5995)
__global__ void __launch_bounds__(256) k_correct_velocity(Tab t, const float *__restrict__ Hbya, const float *__restrict__ P,
                                                           const float *__restrict__ A, const int32_t *__restrict__ active,
                                                           float *__restrict__ Uout) {
    const int b = blockIdx.y;
    if (active && !active[b]) return;
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    const int N = t.N;
    if (g >= N) return;
    const float *p = P + (size_t)b * N;
    const float pc = p[g];
    float pg[2];
#pragma unroll
    for (int d = 0; d < 2; ++d) {
        const int nl = t.nbr[(2 * d) * N + g], nu = t.nbr[(2 * d + 1) * N + g];
        const float fac = (nl < 0 || nu < 0) ? 1.0f : 0.5f;
        const float vl = nl >= 0 ? p[nl] : pc, vu = nu >= 0 ? p[nu] : pc;
        pg[d] = (vu - vl) * fac;
    }
    const float gx = pg[0] * t.minv[g] + pg[1] * t.minv[2 * N + g];
    const float gy = pg[0] * t.minv[N + g] + pg[1] * t.minv[3 * N + g];
    const float rD = 1.0f / A[(size_t)b * N + g];
    Uout[(size_t)b * 2 * N + g] = -rD * gx + Hbya[(size_t)b * 2 * N + g];
    Uout[(size_t)b * 2 * N + N + g] = -rD * gy + Hbya[(size_t)b * 2 * N + N + g];
}

// Passive-scalar transport: SetupAdvectionMatrix(forPassiveScalar) + SetupAdvectionScalar fused
// (K.cu:3617-3880 with the scalar diffusivity, K.cu:4094-4198), orthogonal path.
__global__ void __launch_bounds__(256) k_setup_scalar(Tab t, const float *__restrict__ U, const float *__restrict__ Tin,
                                                       const float *__restrict__ Bvel, const float *__restrict__ Sbval,
                                                       const float *__restrict__ dtv, const int32_t *__restrict__ active,
                                                       float *__restrict__ Coff, float *__restrict__ A, float *__restrict__ Rhs) {
    const int b = blockIdx.y;
    if (active && !active[b]) return;
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    const int N = t.N, NB = t.NB;
    if (g >= N) return;
    const float *u = U + (size_t)b * 2 * N, *bv = Bvel + (size_t)b * 2 * NB, *sb = Sbval + (size_t)b * NB;
    const float dt = dtv[b];
    const float det = t.det[g];
    int nb[4];
#pragma unroll
    for (int f = 0; f < 4; ++f) nb[f] = t.nbr[f * N + g];
    float fl[4];
    face_fluxes(t, g, u, bv, nb, fl);
    float diag = det / dt + t.Cd_s[g];
    float r = det * Tin[(size_t)b * N + g] / dt;
    float *co = Coff + (size_t)b * 4 * N;
#pragma unroll
    for (int f = 0; f < 4; ++f) {
        float o = 0.f;
        if (nb[f] >= 0) {
            const float ff = ((f & 1) ? 0.5f : -0.5f) * fl[f];
            diag += ff;
            o = (ff + t.Cd_s[(f + 1) * N + g]) / det;
        } else {
            const int j = -1 - nb[f];
            const float sc = sb[j];
            const float flux = fl[f] * ((f & 1) ? 1.f : -1.f);   // fl[f] is the boundary flux on prescribed faces
            r -= sc * flux;
            if (t.sb_neumann[j] == 0) r += sc * t.scalar_viscosity * 2.f * t.b_alpha[j];
            else r += sc * t.scalar_viscosity;
        }
        co[f * N + g] = o;
    }
    A[(size_t)b * N + g] = diag / det;
    Rhs[(size_t)b * N + g] = r / det;
}

// buoyancy hook of the RBC environments (rbc_env_base.py:280-304): velocity source = (0, beta * T)
__global__ void k_buoyancy(const float *__restrict__ Tin, float beta, int N, const int32_t *__restrict__ active, float *__restrict__ src) {
    const int b = blockIdx.y;
    if (active && !active[b]) return;
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= N) return;
    src[(size_t)b * 2 * N + g] = 0.f;
    src[(size_t)b * 2 * N + N + g] = Tin[(size_t)b * N + g] * beta;
}

// column sums of a * b * det and of det over a single structured block of nx x ny cells (Nusselt number,
// rbc_env_base.py:491-539, rbc_env_2d.py:328-357): out[b][0][x] = sum_y a*b*det, out[b][1][x] = sum_y det
__global__ void k_column_sums(Tab t, const float *__restrict__ Afield, const float *__restrict__ Bfield, int nx, int ny,
                              float *__restrict__ out) {
    const int b = blockIdx.y;
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= nx) return;
    const int N = t.N;
    float s = 0.f, v = 0.f;
    for (int y = 0; y < ny; ++y) {
        const int g = x + nx * y;
        const float d = t.det[g];
        s += Afield[(size_t)b * N + g] * Bfield[(size_t)b * N + g] * d;
        v += d;
    }
    out[(size_t)b * 2 * nx + x] = s;
    out[(size_t)b * 2 * nx + nx + x] = v;
}

__global__ void k_fill(float *p, float v, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}
__global__ void k_copy_active(const float *__restrict__ src, float *__restrict__ dst, int per_env, const int32_t *__restrict__ active) {
    const int b = blockIdx.y;
    if (active && !active[b]) return;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < per_env) dst[(size_t)b * per_env + i] = src[(size_t)b * per_env + i];
}

// ------------------------------------------------------------------------------------------------
// Krylov solvers, implementation 0: one CTA per environment, vectors in global memory (L2 resident)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float ell_row(const Tab &t, int g, const float *__restrict__ off, const float *__restrict__ diag,
                                         const float *__restrict__ x) {
    const int N = t.N;
    float s = diag[g] * x[g];
#pragma unroll
    for (int f = 0; f < 4; ++f) { const int nb = t.nbr[f * N + g]; if (nb >= 0) s += off[f * N + g] * x[nb]; }
    return s;
}

// BiCGStab without preconditioner (BICG.cu:237-376); NC right-hand sides (velocity components) in lock step.
template <int T, int NC>
__global__ void __launch_bounds__(T) k_bicgstab(Tab t, const float *__restrict__ Coff, const float *__restrict__ Adiag,
                                                 const float *__restrict__ Rhs, float *__restrict__ X, float *__restrict__ work,
                                                 int maxit, float tol, int zero_init, const int32_t *__restrict__ active,
                                                 int32_t *__restrict__ iters, float *__restrict__ resid,
                                                 unsigned long long *__restrict__ iter_total) {
    const int b = blockIdx.x;
    if (active && !active[b]) return;
    __shared__ double red[32 * 4 + 4];
    const int N = t.N;
    const float *off = Coff + (size_t)b * 4 * N, *dg = Adiag + (size_t)b * N;
    const float norm = 1.0f / sqrtf((float)N);
    float *wb = work + (size_t)b * KRY_VECS * N;
    // per component c: r, rw, p, v, tt
    float *r[2] = {wb, wb + 5 * (size_t)N}, *rw[2] = {wb + N, wb + 6 * (size_t)N}, *p[2] = {wb + 2 * (size_t)N, wb + 7 * (size_t)N};
    float *v[2] = {wb + 3 * (size_t)N, wb + 8 * (size_t)N}, *tt[2] = {wb + 4 * (size_t)N, wb + 9 * (size_t)N};
    float *x[2] = {X + (size_t)b * NC * N, X + (size_t)b * NC * N + (NC - 1) * N};
    const float *f[2] = {Rhs + (size_t)b * NC * N, Rhs + (size_t)b * NC * N + (NC - 1) * N};

    if (zero_init) { for (int c = 0; c < NC; ++c) for (int g = threadIdx.x; g < N; g += T) x[c][g] = 0.f; }
    __syncthreads();
    float acc[4];
    acc[0] = acc[1] = acc[2] = acc[3] = 0.f;
    for (int c = 0; c < NC; ++c)
        for (int g = threadIdx.x; g < N; g += T) {
            const float rr = f[c][g] - (zero_init ? 0.f : ell_row(t, g, off, dg, x[c]));
            r[c][g] = rr; rw[c][g] = rr; p[c][g] = rr;
            acc[c] += rr * rr;
        }
    block_reduce_sum<4>(acc, red);
    bool done[2] = {true, true}; int used[2] = {-1, -1}; float fin[2] = {0.f, 0.f};
    float rho[2] = {1.f, 1.f}, alpha[2] = {1.f, 1.f}, omega[2] = {1.f, 1.f};
    for (int c = 0; c < NC; ++c) {
        fin[c] = sqrtf(acc[c]) * norm; used[c] = -1; done[c] = fin[c] < tol;
    }
    for (int i = 0; i < maxit && !(done[0] && done[NC - 1]); ++i) {
        // rho = <rw, r>
        acc[0] = acc[1] = acc[2] = acc[3] = 0.f;
        for (int c = 0; c < NC; ++c) if (!done[c])
            for (int g = threadIdx.x; g < N; g += T) acc[c] += rw[c][g] * r[c][g];
        block_reduce_sum<4>(acc, red);
        for (int c = 0; c < NC; ++c) if (!done[c]) {
            const float rhop = rho[c]; rho[c] = acc[c];
            if (i > 0) {
                const float beta = (rho[c] / rhop) * (alpha[c] / omega[c]);
                for (int g = threadIdx.x; g < N; g += T) p[c][g] = r[c][g] + beta * (p[c][g] - omega[c] * v[c][g]);
            }
        }
        __syncthreads();
        acc[0] = acc[1] = acc[2] = acc[3] = 0.f;
        for (int c = 0; c < NC; ++c) if (!done[c])
            for (int g = threadIdx.x; g < N; g += T) { const float vv = ell_row(t, g, off, dg, p[c]); v[c][g] = vv; acc[c] += rw[c][g] * vv; }
        block_reduce_sum<4>(acc, red);
        float acc2[4] = {0.f, 0.f, 0.f, 0.f};
        for (int c = 0; c < NC; ++c) if (!done[c]) {
            alpha[c] = rho[c] / acc[c];
            for (int g = threadIdx.x; g < N; g += T) {
                const float rr = r[c][g] - alpha[c] * v[c][g];
                r[c][g] = rr; x[c][g] += alpha[c] * p[c][g];
                acc2[c] += rr * rr;
            }
        }
        block_reduce_sum<4>(acc2, red);
        for (int c = 0; c < NC; ++c) if (!done[c]) {
            const float nr = sqrtf(acc2[c]) * norm;
            used[c] = i; fin[c] = nr;
            if (!isfinite(nr) || nr < tol) done[c] = true;
        }
        // t = C r (s = r)
        acc[0] = acc[1] = acc[2] = acc[3] = 0.f;
        for (int c = 0; c < NC; ++c) if (!done[c])
            for (int g = threadIdx.x; g < N; g += T) {
                const float tv = ell_row(t, g, off, dg, r[c]); tt[c][g] = tv;
                acc[c] += tv * r[c][g]; acc[2 + c] += tv * tv;
            }
        block_reduce_sum<4>(acc, red);
        acc2[0] = acc2[1] = acc2[2] = acc2[3] = 0.f;
        for (int c = 0; c < NC; ++c) if (!done[c]) {
            omega[c] = acc[c] / acc[2 + c];
            for (int g = threadIdx.x; g < N; g += T) {
                const float rg = r[c][g];
                x[c][g] += omega[c] * rg;
                const float rr = rg - omega[c] * tt[c][g];
                acc2[c] += rr * rr;
                r[c][g] = rr;   // all rows of t = C r are complete (the reduction above synchronised the block)
            }
        }
        block_reduce_sum<4>(acc2, red);
        for (int c = 0; c < NC; ++c) if (!done[c]) {
            const float nr = sqrtf(acc2[c]) * norm;
            fin[c] = nr;
            if (nr < tol) { done[c] = true; used[c] = i + 1; }
        }
    }
    if (threadIdx.x == 0) {
        if (NC == 2) {
            iters[b * 8 + 0] = used[0]; iters[b * 8 + 1] = used[1];
            resid[b * 8 + 0] = fin[0]; resid[b * 8 + 1] = fin[1];
            iter_total[b * 2 + 1] += (unsigned long long)(used[0] + 1 + used[1] + 1);
        } else {
            iters[b * 8 + 7] = used[0]; resid[b * 8 + 7] = fin[0];
            iter_total[b * 2 + 1] += (unsigned long long)(used[0] + 1);
        }
    }
}

// Conjugate gradients (CG.cu:225-446) with residual reset, best-iterate tracking and mean removal.
template <int T>
__global__ void __launch_bounds__(T) k_cg(Tab t, const float *__restrict__ Poff, const float *__restrict__ Pdiag,
                                           const float *__restrict__ Rhs, float *__restrict__ Xout, float *__restrict__ work,
                                           int maxit, float tol, int zero_init, int reset_steps, int slot,
                                           const int32_t *__restrict__ active, int32_t *__restrict__ iters, float *__restrict__ resid,
                                           unsigned long long *__restrict__ iter_total) {
    const int b = blockIdx.x;
    if (active && !active[b]) return;
    __shared__ double red[32 * 2 + 2];
    const int N = t.N;
    const float *off = Poff + (size_t)b * 4 * N, *dg = Pdiag + (size_t)b * N, *f = Rhs + (size_t)b * N;
    float *wb = work + (size_t)b * KRY_VECS * N;
    float *r = wb, *p = wb + N, *ap = wb + 2 * (size_t)N, *best = wb + 3 * (size_t)N, *x = wb + 4 * (size_t)N;
    float *xo = Xout + (size_t)b * N;
    const float norm = 1.0f / sqrtf((float)N);
    float acc[2] = {0.f, 0.f};
    int allzero_local = 1;
    for (int g = threadIdx.x; g < N; g += T) {
        const float x0 = zero_init ? 0.f : xo[g];
        x[g] = x0;
        if (f[g] != 0.f) allzero_local = 0;
    }
    __syncthreads();
    const int nonzero = __syncthreads_or(!allzero_local);
    int used = -1; float fin = 0.f;
    if (!nonzero) {   // all-zero right-hand side -> zero result (DIFF.py:392, 489-490)
        for (int g = threadIdx.x; g < N; g += T) x[g] = 0.f;
    } else {
        for (int g = threadIdx.x; g < N; g += T) {
            const float rr = f[g] - (zero_init ? 0.f : ell_row(t, g, off, dg, x));
            r[g] = rr; p[g] = rr; acc[0] += rr * rr;
        }
        block_reduce_sum<2>(acc, red);
        float rho = acc[0];
        float bestc = 0.f, lastc = 0.f; int best_it = -1, rising = 0;
        int until_reset = reset_steps > 0 ? reset_steps - 1 : -1;     // (i + 1) % reset_steps == 0 without the division
        for (int i = 0; i < maxit; ++i) {
            const bool do_reset = until_reset == 0;
            if (until_reset >= 0) until_reset = do_reset ? reset_steps - 1 : until_reset - 1;
            if (do_reset) {
                __syncthreads();
                acc[0] = 0.f;
                for (int g = threadIdx.x; g < N; g += T) {
                    const float rr = f[g] - ell_row(t, g, off, dg, x);
                    r[g] = rr; acc[0] += rr * rr;
                }
                __syncthreads();
                for (int g = threadIdx.x; g < N; g += T) p[g] = r[g];
                acc[1] = 0.f;
                block_reduce_sum<2>(acc, red);
                rho = acc[0];
            }
            __syncthreads();
            acc[0] = acc[1] = 0.f;
            for (int g = threadIdx.x; g < N; g += T) { const float a = ell_row(t, g, off, dg, p); ap[g] = a; acc[0] += p[g] * a; }
            block_reduce_sum<2>(acc, red);
            const float alpha = rho / acc[0];
            acc[0] = acc[1] = 0.f;
            for (int g = threadIdx.x; g < N; g += T) {
                x[g] += alpha * p[g];
                const float rr = r[g] - alpha * ap[g];
                r[g] = rr; acc[0] += rr * rr;
            }
            block_reduce_sum<2>(acc, red);
            const float crit = sqrtf(acc[0]) * norm;
            if (!isfinite(crit)) { used = i; fin = crit; break; }
            if (i == 0 || crit < bestc) {
                bestc = crit; best_it = i;
                for (int g = threadIdx.x; g < N; g += T) best[g] = x[g];
            }
            if (i > 0 && crit >= lastc) ++rising; else rising = 0;
            lastc = crit;
            used = i; fin = crit;
            if (crit < tol) break;
            if (i == maxit - 1 || rising >= 100) {
                __syncthreads();
                for (int g = threadIdx.x; g < N; g += T) x[g] = best[g];
                used = best_it; fin = bestc;
                break;
            }
            const float rhop = rho; rho = acc[0];
            const float beta = rho / rhop;
            for (int g = threadIdx.x; g < N; g += T) p[g] = r[g] + beta * p[g];
        }
    }
    __syncthreads();
    // mean removal (SIM.py:1922-1925)
    acc[0] = acc[1] = 0.f;
    for (int g = threadIdx.x; g < N; g += T) acc[0] += x[g];
    block_reduce_sum<2>(acc, red);
    const float mean = acc[0] / (float)N;
    for (int g = threadIdx.x; g < N; g += T) xo[g] = x[g] - mean;
    if (threadIdx.x == 0) { iters[b * 8 + 2 + slot] = used; resid[b * 8 + 2 + slot] = fin; iter_total[b * 2] += (unsigned long long)(used + 1); }
}

// ------------------------------------------------------------------------------------------------
// Krylov solvers, implementation 1: one thread-block cluster per environment, everything on chip.
// Each CTA of the cluster owns a contiguous range of cells; the search direction p lives in shared
// memory (neighbour gathers hit local smem or a peer CTA's smem through DSMEM), x / r / best and the
// five stencil coefficients of the owned cells live in registers; the two dot products per iteration
// are reduced inside the cluster through DSMEM + one cluster barrier each.  HBM traffic per solve is
// one read of P, rhs and one write of p.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ float ld_dsmem_f32(uint32_t addr) {
    float v;
    asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void st_dsmem_f64x2(uint32_t addr, double a, double b) {
    asm volatile("st.shared::cluster.v2.f64 [%0], {%1, %2};" ::"r"(addr), "d"(a), "d"(b) : "memory");
}

__device__ __forceinline__ void st_dsmem_f32x2(uint32_t addr, float a, float b) {
    asm volatile("st.shared::cluster.v2.f32 [%0], {%1, %2};" ::"r"(addr), "f"(a), "f"(b) : "memory");
}
__device__ __forceinline__ void cluster_arrive_release() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait_acquire() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_sync_all() { cluster_arrive_release(); cluster_wait_acquire(); }

// VARIANT: 0 = textbook recurrence of the reference (A*p applied to the search direction, 3 cluster
// barriers per iteration); 1 = A*p obtained from the recurrence Ap <- A*r + beta*Ap (mathematically
// identical, 2 cluster barriers per iteration, p and Ap never leave registers).
// Cells are padded to T*CPT per CTA: padding cells carry zero coefficients / zero data so the inner loops
// need no bounds predicates.
template <int T, int CPT, int CS, int VARIANT>
__global__ void __launch_bounds__(T, 1) k_cg_cluster(Tab t, const float *__restrict__ Poff, const float *__restrict__ Pdiag,
                                                      const float *__restrict__ Rhs, float *__restrict__ Xout,
                                                      int maxit, float tol, int zero_init, int reset_steps, int slot,
                                                      const int32_t *__restrict__ active, int32_t *__restrict__ iters,
                                                      float *__restrict__ resid, unsigned long long *__restrict__ iter_total) {
    constexpr int NW = T / 32;                  // warps per CTA
    constexpr int NP = NW * CS;                 // warp partials per cluster-wide reduction
    constexpr int PAD = T * CPT;                // padded cells per CTA
    static_assert(NP <= 64, "final reduction reads two partials per lane");
    const int b = blockIdx.x / CS;
    uint32_t rank;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
    if (active && !active[b]) return;  // uniform over the cluster
    extern __shared__ __align__(16) float smem[];
    const int N = t.N;
    const int per = (N + CS - 1) / CS;          // cells owned per CTA
    const int start = (int)rank * per;
    const int cnt = max(0, min(per, N - start));
    float *vs = smem;                            // [PAD] vector exposed to the neighbours (p, or r in variant 1)
    float *bs = smem + PAD;                      // [PAD] best iterate of the owned cells
    float *red = smem + 2 * PAD;                 // [2 parity][NP] warp partials written by every warp of the cluster
    const float *off = Poff + (size_t)b * 4 * N, *dg = Pdiag + (size_t)b * N, *f = Rhs + (size_t)b * N;
    float *xo = Xout + (size_t)b * N;
    const float norm = 1.0f / sqrtf((float)N);
    const uint32_t vs_addr = smem_u32(vs), red_addr = smem_u32(red);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    // registers: stencil coefficients, cluster-shared addresses of the 4 neighbours, x, r
    float cd[CPT], co[CPT][4], xr[CPT], rr[CPT];
    uint32_t na[CPT][4];
#pragma unroll
    for (int k = 0; k < CPT; ++k) {
        const int l = threadIdx.x + k * T;
        const int g = start + l;
        const bool ok = l < cnt;
        cd[k] = ok ? dg[g] : 0.f;
        xr[k] = (ok && !zero_init) ? xo[g] : 0.f;
        vs[l] = 0.f; bs[l] = 0.f;
#pragma unroll
        for (int ff = 0; ff < 4; ++ff) {
            const int nb = ok ? t.nbr[ff * N + g] : -1;
            co[k][ff] = (ok && nb >= 0) ? off[ff * N + g] : 0.f;
            const int gi = nb >= 0 ? nb : (ok ? g : start);   // coefficient is 0 for absent neighbours
            const int c = gi / per;
            na[k][ff] = mapa_u32(vs_addr + 4u * (uint32_t)(gi - c * per), (uint32_t)c);
        }
    }
    int parity = 0;
    // Cluster-wide sum with ONE cluster barrier and no block barrier: every warp pushes its partial into
    // the reduction slots of all CTAs through DSMEM; after the barrier every warp folds the NP partials
    // with the same butterfly, so all threads of the cluster obtain bit-identical totals.
    auto cluster_sum = [&](float a0) -> float {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) a0 += __shfl_xor_sync(0xffffffffu, a0, o);
        if (lane < CS) {
            const uint32_t ra = mapa_u32(red_addr + 4u * (uint32_t)(parity * NP + (int)rank * NW + warp), (uint32_t)lane);
            asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(ra), "f"(a0) : "memory");
        }
        cluster_sync_all();
        const float *rp = red + parity * NP;
        float s0 = lane < NP ? rp[lane] : 0.f;
        if (NP > 32) s0 += (lane + 32 < NP) ? rp[lane + 32] : 0.f;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s0 += __shfl_xor_sync(0xffffffffu, s0, o);
        parity ^= 1;
        return s0;
    };
    auto apply = [&](int k) -> float {   // row k of P times the vector currently exposed in vs (cluster wide)
        float s = cd[k] * vs[threadIdx.x + k * T];
#pragma unroll
        for (int ff = 0; ff < 4; ++ff) s += co[k][ff] * ld_dsmem_f32(na[k][ff]);
        return s;
    };
    auto load_f = [&](int k) -> float { const int l = threadIdx.x + k * T; return l < cnt ? f[start + l] : 0.f; };

    // all-zero right-hand side -> result zero (DIFF.py:392, 489-490)
    float nz = 0.f;
#pragma unroll
    for (int k = 0; k < CPT; ++k) nz += (load_f(k) != 0.f) ? 1.f : 0.f;
    const float nzt = cluster_sum(nz);           // the barrier also orders the zero-fill of vs/bs
    int used = -1; float fin = 0.f;
    if (!(nzt > 0.f)) {
#pragma unroll
        for (int k = 0; k < CPT; ++k) xr[k] = 0.f;
    } else {
        // r0 = f - P x0
        if (!zero_init) {
#pragma unroll
            for (int k = 0; k < CPT; ++k) vs[threadIdx.x + k * T] = xr[k];
            cluster_sync_all();
#pragma unroll
            for (int k = 0; k < CPT; ++k) rr[k] = load_f(k) - apply(k);
            cluster_sync_all();
        } else {
#pragma unroll
            for (int k = 0; k < CPT; ++k) rr[k] = load_f(k);
        }
        float a0 = 0.f;
#pragma unroll
        for (int k = 0; k < CPT; ++k) { const int l = threadIdx.x + k * T; vs[l] = rr[k]; bs[l] = xr[k]; a0 += rr[k] * rr[k]; }
        float rho = cluster_sum(a0);             // the barrier inside also publishes vs (= r0 = p0)
        float bestc = 0.f, lastc = 0.f; int best_it = -1, rising = 0;
        float pk[CPT], apk[CPT];                 // search direction and A*p of the owned cells
        float beta = 0.f;
#pragma unroll
        for (int k = 0; k < CPT; ++k) { pk[k] = 0.f; apk[k] = 0.f; }
        for (int i = 0; i < maxit; ++i) {
            if (reset_steps > 0 && (i + 1) % reset_steps == 0) {
                // r = f - P x ; p = r ; rho = <r,r>   (CG.cu:281-302)
                cluster_sync_all();              // everyone is done reading vs
#pragma unroll
                for (int k = 0; k < CPT; ++k) vs[threadIdx.x + k * T] = xr[k];
                cluster_sync_all();
#pragma unroll
                for (int k = 0; k < CPT; ++k) rr[k] = load_f(k) - apply(k);
                cluster_sync_all();
                a0 = 0.f;
#pragma unroll
                for (int k = 0; k < CPT; ++k) { vs[threadIdx.x + k * T] = rr[k]; a0 += rr[k] * rr[k]; }
                rho = cluster_sum(a0);
                beta = 0.f;
            }
            a0 = 0.f;
            if (VARIANT == 0) {
#pragma unroll
                for (int k = 0; k < CPT; ++k) {
                    apk[k] = apply(k);
                    pk[k] = vs[threadIdx.x + k * T];
                    a0 += pk[k] * apk[k];
                }
            } else {
                // vs holds r:  Ap <- A r + beta Ap ,  p <- r + beta p   (beta = 0 right after (re)starts)
#pragma unroll
                for (int k = 0; k < CPT; ++k) {
                    apk[k] = apply(k) + beta * apk[k];
                    pk[k] = rr[k] + beta * pk[k];
                    a0 += pk[k] * apk[k];
                }
            }
            const float pap = cluster_sum(a0);   // after this barrier every CTA has finished reading vs
            const float alpha = rho / pap;
            a0 = 0.f;
#pragma unroll
            for (int k = 0; k < CPT; ++k) {
                xr[k] += alpha * pk[k];
                rr[k] -= alpha * apk[k];
                a0 += rr[k] * rr[k];
                if (VARIANT == 1) vs[threadIdx.x + k * T] = rr[k];   // published by the barrier of the next reduction
            }
            const float rr2 = cluster_sum(a0);
            const float crit = sqrtf(rr2) * norm;
            if (!isfinite(crit)) { used = i; fin = crit; break; }
            if (i == 0 || crit < bestc) {
                bestc = crit; best_it = i;
#pragma unroll
                for (int k = 0; k < CPT; ++k) bs[threadIdx.x + k * T] = xr[k];
            }
            if (i > 0 && crit >= lastc) ++rising; else rising = 0;
            lastc = crit; used = i; fin = crit;
            if (crit < tol) break;
            if (i == maxit - 1 || rising >= 100) {
#pragma unroll
                for (int k = 0; k < CPT; ++k) xr[k] = bs[threadIdx.x + k * T];
                used = best_it; fin = bestc;
                break;
            }
            beta = rr2 / rho;
            rho = rr2;
            if (VARIANT == 0) {
#pragma unroll
                for (int k = 0; k < CPT; ++k) vs[threadIdx.x + k * T] = rr[k] + beta * pk[k];
                cluster_sync_all();   // new p visible cluster wide
            }
        }
    }
    // mean removal
    float sx = 0.f;
#pragma unroll
    for (int k = 0; k < CPT; ++k) sx += xr[k];
    const float mean = cluster_sum(sx) / (float)N;
#pragma unroll
    for (int k = 0; k < CPT; ++k) { const int l = threadIdx.x + k * T; if (l < cnt) xo[start + l] = xr[k] - mean; }
    if (threadIdx.x == 0 && rank == 0) { iters[b * 8 + 2 + slot] = used; resid[b * 8 + 2 + slot] = fin; iter_total[b * 2] += (unsigned long long)(used + 1); }
    cluster_sync_all();   // keep peer shared memory alive until everyone is done
}

// ------------------------------------------------------------------------------------------------
// Krylov solvers, implementation 3: as implementation 1 (cluster per environment, textbook CG
// recurrence) but WITHOUT cluster-wide barriers in the iteration.  All cross-CTA synchronisation is
// point-to-point through shared-memory mbarriers:
//   * reductions: every warp pushes its partial into every CTA's slot array with
//     st.async ... mbarrier::complete_tx (data and completion signal travel together, no fence);
//     consumers wait on their local transaction barrier;
//   * search-direction visibility: after a CTA has rewritten its part of p, one thread arrives
//     (release.cluster) on every peer's "p ready" mbarrier; consumers acquire it before the gathers.
// Write-after-read safety of p and of the slot arrays follows from the data flow: a reduction can only
// complete once every warp of every CTA has contributed, i.e. has finished the preceding phase.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t a, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(a), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t a, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(a), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive_remote_release(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// CTA-scope acquire (the default): everything exchanged here lives in shared memory (st.async payloads, or
// st.shared data published with a release.cluster arrive and read back with ld.shared::cluster), which is
// never cached in L1, so the cluster-scope acquire -- a CCTL.IVALL L1 invalidation per waiting warp, 10 % of
// all stall samples in profiles/r01_ncu_cg_cluster_impl3.txt -- buys nothing.
__device__ __forceinline__ bool mbar_try_wait(uint32_t a, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred P1;\n\t"
                 "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
                 "selp.b32 %0, 1, 0, P1;\n\t}"
                 : "=r"(ok) : "r"(a), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t a, uint32_t parity) { while (!mbar_try_wait(a, parity)) {} }
// as mbar_wait, with a suspend-time hint: the warp sleeps in hardware until the phase completes (or ~1 us passes) instead
// of re-issuing the test -- spinning warps otherwise take issue slots and shared-memory pipe cycles from the working ones
__device__ __forceinline__ void mbar_wait_sleep(uint32_t a, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile("{\n\t.reg .pred P1;\n\t"
                     "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2, %3;\n\t"
                     "selp.b32 %0, 1, 0, P1;\n\t}"
                     : "=r"(ok) : "r"(a), "r"(parity), "r"(1000u) : "memory");
    } while (!ok);
}
__device__ __forceinline__ void st_async_f32(uint32_t cluster_addr, float v, uint32_t cluster_mbar) {
    asm volatile("st.async.shared::cluster.mbarrier::complete_tx::bytes.u32 [%0], %1, [%2];"
                 ::"r"(cluster_addr), "r"(__float_as_uint(v)), "r"(cluster_mbar) : "memory");
}

__device__ __forceinline__ float ld_shared_f32(uint32_t addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
    return v;
}

// PUSH = false: neighbours are gathered from the owning CTA's shared memory through the cluster window (DSMEM).
// PUSH = true : halo plan of tables.cg_* -- after every update of the exposed vector each CTA pushes the cells its
//               neighbours need into THEIR shared memory (st.async, completing the receiver's mbarrier transaction
//               count), so every stencil gather is a plain ld.shared and the hand-shake carries the data itself
//               (no release fence, no remote arrive).  ncu on the PUSH=false kernel: each DSMEM gather costs an
//               LD.E on a generic address plus two MOVs to assemble it, 84 of 391 instructions per iteration.
template <int T, int CPT, int CS, bool PUSH, int MINB = 1>
__global__ void __launch_bounds__(T, MINB) k_cg_cluster_mb(Tab t, const float *__restrict__ Poff, const float *__restrict__ Pdiag,
                                                         const float *__restrict__ Rhs, float *__restrict__ Xout,
                                                         int maxit, float tol, int zero_init, int reset_steps, int slot,
                                                         const int32_t *__restrict__ active, int32_t *__restrict__ iters,
                                                         float *__restrict__ resid, unsigned long long *__restrict__ iter_total,
                                                         int flags, float *__restrict__ mean_out) {
    // flags bit 0: apply the TRANSPOSED operator (adjoint solve, DIFF.py:572-590): the coefficient of neighbour
    //              j in row i is the one stored in row j for the face that points back to i (tables.rev)
    //       bit 1: do not remove the mean of the result
    constexpr int NW = T / 32;
    constexpr int NP = NW * CS;
    constexpr int PAD = T * CPT;
    const int b = blockIdx.x / CS;
    uint32_t rank;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
    if (active && !active[b]) return;
    extern __shared__ __align__(16) float smem[];
    const int N = t.N;
    const int per = (N + CS - 1) / CS;
    const int start = (int)rank * per;
    const int cnt = max(0, min(per, N - start));
    float *vs = smem;                            // [PAD] search direction of the owned cells
    const int HM = PUSH ? t.cg_hmax : 0;         // halo slots follow the owned cells: vs[PAD .. PAD + HM)
    float *bs = smem + PAD + HM;                 // [PAD] best iterate
    float *red = bs + PAD;                       // [2][NP] reduction slots (alternating)
    unsigned long long *mb = (unsigned long long *)(red + 2 * NP);   // [0],[1]: reductions, [2]: p ready
    uint2 *exps = (uint2 *)(mb + 4);             // [cg_emax] export list (PUSH)
    const float *off = Poff + (size_t)b * 4 * N, *dg = Pdiag + (size_t)b * N, *f = Rhs + (size_t)b * N;
    float *xo = Xout + (size_t)b * N;
    const float norm = 1.0f / sqrtf((float)N);
    const uint32_t vs_addr = smem_u32(vs), red_addr = smem_u32(red), mb_addr = smem_u32(mb);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    const int n_exp = PUSH ? t.cg_cnt[2 * rank] : 0;
    const uint32_t halo_bytes = PUSH ? 4u * (uint32_t)t.cg_cnt[2 * rank + 1] : 0u;
    if (threadIdx.x == 0) {
        mbar_init(mb_addr, 1); mbar_init(mb_addr + 8, 1); mbar_init(mb_addr + 16, PUSH ? 1 : CS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        mbar_arrive_expect_tx(mb_addr, NP * 4);          // arm both reduction barriers for their first use
        mbar_arrive_expect_tx(mb_addr + 8, NP * 4);
        if (PUSH) mbar_arrive_expect_tx(mb_addr + 16, halo_bytes);
    }
    if (PUSH) {
        for (int e = threadIdx.x; e < n_exp; e += T) {
            const int32_t a = t.cg_exp[((size_t)rank * t.cg_emax + e) * 2], d = t.cg_exp[((size_t)rank * t.cg_emax + e) * 2 + 1];
            const uint32_t dst_rank = (uint32_t)a >> 24;
            // x: byte offset of the own slot in vs | dest rank << 24 ; y: cluster address of the destination slot
            // (a shared::cta address carries the CTA's position in the cluster window in its high bits, so the
            //  byte OFFSET is packed, not the address)
            exps[e] = make_uint2((4u * ((uint32_t)a & 0xffffffu)) | (dst_rank << 24), mapa_u32(vs_addr + 4u * (uint32_t)d, dst_rank));
        }
        for (int h = threadIdx.x; h < HM; h += T) vs[PAD + h] = 0.f;
    }
    float cd[CPT], co[CPT][4], xr[CPT], rr[CPT];
    uint32_t na[CPT][4];
#pragma unroll
    for (int k = 0; k < CPT; ++k) {
        const int l = threadIdx.x + k * T;
        const int g = start + l;
        const bool ok = l < cnt;
        cd[k] = ok ? dg[g] : 0.f;
        xr[k] = (ok && !zero_init) ? xo[g] : 0.f;
        vs[l] = 0.f; bs[l] = 0.f;
#pragma unroll
        for (int ff = 0; ff < 4; ++ff) {
            const int nb = ok ? t.nbr[ff * N + g] : -1;
            if (flags & 1) co[k][ff] = (ok && nb >= 0) ? off[(int)t.rev[ff * N + g] * N + nb] : 0.f;
            else co[k][ff] = (ok && nb >= 0) ? off[ff * N + g] : 0.f;
            const int gi = nb >= 0 ? nb : (ok ? g : start);
            const int c = gi / per;
            // (measured: splitting local neighbours onto plain ld.shared with a per-gather predicate is SLOWER,
            //  10.8 vs 8.3 ms per substep -- the cluster-window load of an own-CTA address is not the bottleneck)
            if (PUSH) na[k][ff] = vs_addr + 4u * (uint32_t)(ok ? t.cg_slot[ff * N + g] : 0);
            else na[k][ff] = mapa_u32(vs_addr + 4u * (uint32_t)(gi - c * per), (uint32_t)c);
        }
    }
    // addresses this lane pushes partials to (lane < CS): slot array and barriers of CTA `lane`
    const uint32_t peer_red = mapa_u32(red_addr, (uint32_t)(lane < CS ? lane : 0));
    const uint32_t peer_mb = mapa_u32(mb_addr, (uint32_t)(lane < CS ? lane : 0));
    cluster_sync_all();                          // barriers initialised and vs/bs zero-filled everywhere

    uint32_t rcount = 0;                         // reductions issued so far (slot array / barrier = rcount & 1)
    uint32_t pphase = 0;                         // phase parity of the "p ready" barrier
    auto cluster_sum = [&](float a0) -> float {
        const uint32_t w = rcount & 1u, par = (rcount >> 1) & 1u;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) a0 += __shfl_xor_sync(0xffffffffu, a0, o);
        if (lane < CS) st_async_f32(peer_red + 4u * (w * NP + rank * NW + (uint32_t)warp), a0, peer_mb + 8u * w);
        mbar_wait(mb_addr + 8u * w, par);
        const float *rp = red + w * NP;
        float s0 = 0.f;
#pragma unroll
        for (int q = 0; q < (NP + 31) / 32; ++q) s0 += (lane + 32 * q < NP) ? rp[lane + 32 * q] : 0.f;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s0 += __shfl_xor_sync(0xffffffffu, s0, o);
        // re-arm this barrier for its next use (two reductions from now); every warp of this CTA has to be
        // past the wait first, which the CTA-wide barrier of the following publish()/sync guarantees only
        // loosely -- the arm may trail the first complete_tx of the next phase, which mbarrier semantics allow
        // (the phase cannot complete before the pending arrival of the arm itself).
        if (threadIdx.x == 0) mbar_arrive_expect_tx(mb_addr + 8u * w, NP * 4);
        ++rcount;
        return s0;
    };
    auto publish = [&]() {                       // my part of vs is written: tell every CTA of the cluster
        __syncthreads();
        if (PUSH) {
            for (int e = threadIdx.x; e < n_exp; e += T) {
                const uint2 ex = exps[e];
                st_async_f32(ex.y, ld_shared_f32(vs_addr + (ex.x & 0xffffffu)), mapa_u32(mb_addr + 16, ex.x >> 24));
            }
        } else if (threadIdx.x < CS) mbar_arrive_remote_release(mapa_u32(mb_addr + 16, threadIdx.x));
    };
    auto acquire_p = [&]() {
        mbar_wait(mb_addr + 16, pphase); pphase ^= 1u;
        // PUSH: re-arm for the next hand-shake.  Its data cannot complete the phase before this arrival, and no
        // sender can start the next push before every warp of this CTA has passed the wait above (the senders
        // first need this CTA's partials of the following reduction).
        if (PUSH && threadIdx.x == 0) mbar_arrive_expect_tx(mb_addr + 16, halo_bytes);
    };
    auto apply = [&](int k) -> float {
        float s = cd[k] * vs[threadIdx.x + k * T];
#pragma unroll
        for (int ff = 0; ff < 4; ++ff) s += co[k][ff] * (PUSH ? ld_shared_f32(na[k][ff]) : ld_dsmem_f32(na[k][ff]));
        return s;
    };
    auto load_f = [&](int k) -> float { const int l = threadIdx.x + k * T; return l < cnt ? f[start + l] : 0.f; };

    float nz = 0.f;
#pragma unroll
    for (int k = 0; k < CPT; ++k) nz += (load_f(k) != 0.f) ? 1.f : 0.f;
    const float nzt = cluster_sum(nz);
    int used = -1; float fin = 0.f;
    if (!(nzt > 0.f)) {
#pragma unroll
        for (int k = 0; k < CPT; ++k) xr[k] = 0.f;
    } else {
        if (!zero_init) {
#pragma unroll
            for (int k = 0; k < CPT; ++k) vs[threadIdx.x + k * T] = xr[k];
            publish(); acquire_p();
#pragma unroll
            for (int k = 0; k < CPT; ++k) rr[k] = load_f(k) - apply(k);
            (void)cluster_sum(0.f);              // everyone is done reading vs (= x)
        } else {
#pragma unroll
            for (int k = 0; k < CPT; ++k) rr[k] = load_f(k);
        }
        float a0 = 0.f;
#pragma unroll
        for (int k = 0; k < CPT; ++k) { const int l = threadIdx.x + k * T; vs[l] = rr[k]; bs[l] = xr[k]; a0 += rr[k] * rr[k]; }
        publish();
        float rho = cluster_sum(a0);
        float bestc = 0.f, lastc = 0.f; int best_it = -1, rising = 0;
        bool take_best = false;
        float pk[CPT], apk[CPT];
        for (int i = 0; i < maxit; ++i) {
            if (reset_steps > 0 && (i + 1) % reset_steps == 0) {
                // r = f - P x ; p = r ; rho = <r,r>   (CG.cu:281-302).  The pending "p ready" phase is consumed
                // first so that the barrier phases stay aligned.
                acquire_p();
                (void)cluster_sum(0.f);          // nobody reads vs any more
#pragma unroll
                for (int k = 0; k < CPT; ++k) vs[threadIdx.x + k * T] = xr[k];
                publish(); acquire_p();
#pragma unroll
                for (int k = 0; k < CPT; ++k) rr[k] = load_f(k) - apply(k);
                (void)cluster_sum(0.f);
                a0 = 0.f;
#pragma unroll
                for (int k = 0; k < CPT; ++k) { vs[threadIdx.x + k * T] = rr[k]; a0 += rr[k] * rr[k]; }
                publish();
                rho = cluster_sum(a0);
            }
            acquire_p();                         // p of every CTA is visible
            a0 = 0.f;
#pragma unroll
            for (int k = 0; k < CPT; ++k) {
                apk[k] = apply(k);
                pk[k] = vs[threadIdx.x + k * T];
                a0 += pk[k] * apk[k];
            }
            const float pap = cluster_sum(a0);   // completes only after every warp of the cluster finished its gathers
            const float alpha = rho / pap;
            a0 = 0.f;
#pragma unroll
            for (int k = 0; k < CPT; ++k) {
                xr[k] += alpha * pk[k];
                rr[k] -= alpha * apk[k];
                a0 += rr[k] * rr[k];
            }
            const float rr2 = cluster_sum(a0);
            const float crit = sqrtf(rr2) * norm;
            // ONE loop exit (see k_cg_strip: several `break`s made the compiler copy the iterate's registers before every test)
            int stop = isfinite(crit) ? 0 : 1;   // 1: leave with the current iterate, 2: leave with the best one
            used = i; fin = crit;
            if (!stop) {
                if (i == 0 || crit < bestc) {
                    bestc = crit; best_it = i;
#pragma unroll
                    for (int k = 0; k < CPT; ++k) bs[threadIdx.x + k * T] = xr[k];
                }
                if (i > 0 && crit >= lastc) ++rising; else rising = 0;
                lastc = crit;
                if (crit < tol) stop = 1;
                else if (i == maxit - 1 || rising >= 100) stop = 2;
            }
            asm volatile("" : "+r"(stop));             // opaque: keeps the compiler from threading the exits apart again
            if (stop) { take_best = stop == 2; break; }
            const float beta = rr2 / rho;
            rho = rr2;
#pragma unroll
            for (int k = 0; k < CPT; ++k) vs[threadIdx.x + k * T] = rr[k] + beta * pk[k];
            publish();
        }
        if (take_best) {
#pragma unroll
            for (int k = 0; k < CPT; ++k) xr[k] = bs[threadIdx.x + k * T];
            used = best_it; fin = bestc;
        }
    }
    float sx = 0.f;
#pragma unroll
    for (int k = 0; k < CPT; ++k) sx += xr[k];
    const float mean = (flags & 2) ? 0.f : cluster_sum(sx) / (float)N;
    if (mean_out && threadIdx.x == 0 && rank == 0) mean_out[b] = mean;
#pragma unroll
    for (int k = 0; k < CPT; ++k) { const int l = threadIdx.x + k * T; if (l < cnt) xo[start + l] = xr[k] - mean; }
    if (threadIdx.x == 0 && rank == 0) { iters[b * 8 + 2 + slot] = used; resid[b * 8 + 2 + slot] = fin; iter_total[b * 2] += (unsigned long long)(used + 1); }
    cluster_sync_all();   // keep peer shared memory (and in-flight st.async targets) alive until everyone is done
}

// ------------------------------------------------------------------------------------------------
// Krylov solvers, implementation 11: register-blocked strip layout (fluidgym_b200/strip_plan.py, tables.st_*).
// Same recurrence and stopping rules as above (CG.cu:225-446), different data layout and hand-shakes:
//   * the cells of a CTA are padded 2-D arrays in shared memory, the stencil neighbours of slot s are s-1, s+1,
//     s-S, s+S: no per-cell neighbour addresses (k_cg_cluster_mb keeps 4 address registers per cell);
//   * a thread owns CPT = 9 consecutive rows of one column, so the south / north neighbours of its cells are its own
//     registers: per cell and iteration 2 + 2/CPT shared-memory loads of the search direction instead of 5, all of
//     them conflict free (S is a multiple of 4, so a warp that runs from one band of rows into the next continues
//     on the next bank);
//   * x, r, p, A p live in registers, the five stencil coefficients in shared memory (thread-major, one LDS.128 + one
//     LDS.32 per row): 72 registers per thread, 896 threads per CTA, 8 064 cells per CTA -- HALF the cluster size of
//     k_cg_cluster_mb for every domain (cylinder-24: 2 CTAs instead of 4, RBC: 1 instead of 2, airfoil: 8 instead of
//     16), so twice the environments are in flight and a 2-CTA cluster packs onto all 148 SMs;
//   * cells that are not array-adjacent are GHOST slots.  Remote ghosts (owner in another CTA) are replicas that run
//     the same x / p updates with the same scalars as their owner (bit-identical by construction); the only vector
//     data exchanged per iteration is the residual of the mirrored cells, pushed (st.async) by the owning thread onto
//     the SAME transaction barrier as the partial sums of <r,r>: an iteration has TWO cross-CTA exchanges (<p,Ap>;
//     <r,r> + ghost residuals), the separate "search direction published" hand-shake of k_cg_cluster_mb is gone.
//     Local ghosts (owner in the same CTA: block connections, periodic wrap) are mirror slots the owner stores its new
//     search direction into before the CTA barrier that publishes the direction anyway.
// Barrier A (mb[0]) collects NP partials, barrier B (mb[1]) NP partials + the ghost residuals of this CTA; they are
// used strictly alternately (a reset iteration inserts an empty A), which is what makes the single-buffered slot
// arrays safe: a CTA can only start exchange n+1 after every warp of every CTA has contributed to exchange n, i.e.
// has consumed exchange n-1.  The best iterate (CG.cu:335-352) is kept in global scratch (written, never read, unless
// the solve fails), thread-major and coalesced.
// LAZY (cg_impl 11; false = cg_impl 13, the eager order) moves the bookkeeping that does not feed the recurrence off the
// chain between the two exchanges, with the same floating-point operations on the same values (bit-identical results):
//   * x += alpha p is deferred into the next direction update, which loads p_old for p = r + beta p anyway; between
//     exchanges A and B only r is updated.  Every exit that leaves with the current iterate applies the update first;
//   * the best iterate is stored only when it is about to be lost: on the first non-improving iteration after an
//     improving run the registers (not yet advanced) still hold it.  A failed solve whose last iteration improved takes
//     it from the registers.
// ------------------------------------------------------------------------------------------------
template <int T, int CPT, int CS, int MINB, bool LAZY>
__global__ void __launch_bounds__(T, MINB) k_cg_strip(Tab t, const float *__restrict__ Poff, const float *__restrict__ Pdiag,
                                                    const float *__restrict__ Rhs, float *__restrict__ Xout,
                                                    int maxit, float tol, int zero_init, int reset_steps, int slot,
                                                    const int32_t *__restrict__ active, int32_t *__restrict__ iters,
                                                    float *__restrict__ resid, unsigned long long *__restrict__ iter_total,
                                                    int flags, float *__restrict__ mean_out, float *__restrict__ best) {
    static_assert(T % 32 == 0, "whole warps only: every warp contributes exactly one partial sum per exchange");
    constexpr int NW = T / 32;
    const int b = blockIdx.x / CS;
    uint32_t rank;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
    if (active && !active[b]) return;
    extern __shared__ __align__(16) float smem[];
    const int N = t.N, SL = t.st_slots, G = t.st_gmax;
    float4 *co4 = reinterpret_cast<float4 *>(smem);    // [CPT][T] off-diagonal coefficients (W, E, S, N)
    float *cdg = smem + 4 * CPT * T;                   // [CPT][T] diagonal
    float *vs = cdg + CPT * T;                         // [SL] exposed vector (search direction; x at residual resets)
    float *rs = vs + SL;                               // [G] residuals received for the remote ghost rows
    float *red = rs + G;                               // [2][CS] totals of every CTA: A, B ; then [2][NW] warp partials of this CTA
    float *wpart = red + 2 * CS + (2 * CS & 1 ? 1 : 0);
    unsigned long long *mb = (unsigned long long *)(wpart + 2 * NW + (2 * NW & 1 ? 1 : 0));   // [0]: A, [1]: B, [2]: A local, [3]: B local
    uint2 *rex = (uint2 *)(mb + 4);                    // [st_remax] {k | dest rank << 8, cluster address of the destination in rs}
    uint2 *lex = rex + t.st_remax;                     // [st_lemax] {owner's slot, mirror slot} in vs
    const float *off = Poff + (size_t)b * 4 * N, *dg = Pdiag + (size_t)b * N, *f = Rhs + (size_t)b * N;
    float *xo = Xout + (size_t)b * N;
    const float norm = 1.0f / sqrtf((float)N);
    const uint32_t red_addr = smem_u32(red), mb_addr = smem_u32(mb), rs_addr = smem_u32(rs);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    const int4 th0 = reinterpret_cast<const int4 *>(t.st_thread)[((size_t)rank * T + tid) * 2];
    const int4 th1 = reinterpret_cast<const int4 *>(t.st_thread)[((size_t)rank * T + tid) * 2 + 1];
    const int S = th0.y;
    float *vp = vs + th0.x;                            // slot of row 0 of this thread
    const int re_off = th0.w & 0xffff, re_cnt = (th0.w >> 16) & 0xff;
    const int n_lex = t.st_cnt[4 * rank + 2];
    const float *rgp = rs + th1.y;                     // first remote ghost row of this thread in the receive buffer
    const uint32_t rm = (uint32_t)th1.z;               // remote ghost rows of this thread (bit k)
    const int32_t *cellp = t.st_cell + ((size_t)rank * T + tid) * CPT;
    // LAZY: volatile, or the compiler forwards the stored best iterate to the reload at the failure exit in CPT registers
    // that stay live across the whole loop (and push the iteration into spills)
    typename std::conditional<LAZY, volatile float, float>::type *bestp = best + ((size_t)b * CS + rank) * T * CPT + tid;
    const uint32_t bytesA = CS * 4u, bytesB = CS * 4u + 4u * (uint32_t)t.st_cnt[4 * rank];
    if (tid == 0) {
        mbar_init(mb_addr, 1); mbar_init(mb_addr + 8, 1);
        mbar_init(mb_addr + 16, NW); mbar_init(mb_addr + 24, NW);   // "warp partials of this CTA are in shared memory"
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        mbar_arrive_expect_tx(mb_addr, bytesA);
        mbar_arrive_expect_tx(mb_addr + 8, bytesB);
    }
    for (int e = tid; e < t.st_cnt[4 * rank + 1]; e += T) {
        const int32_t a = t.st_rexp[((size_t)rank * t.st_remax + e) * 2], d = t.st_rexp[((size_t)rank * t.st_remax + e) * 2 + 1];
        rex[e] = make_uint2((uint32_t)a, mapa_u32(rs_addr + 4u * (uint32_t)d, (uint32_t)a >> 8));
    }
    for (int e = tid; e < n_lex; e += T)
        lex[e] = make_uint2((uint32_t)t.st_lexp[((size_t)rank * t.st_lemax + e) * 2], (uint32_t)t.st_lexp[((size_t)rank * t.st_lemax + e) * 2 + 1]);
    for (int i = tid; i < SL + G; i += T) vs[i] = 0.f;   // vs and rs (pads, dead slots)

    float x[CPT], r[CPT], ap[CPT];                     // the search direction itself lives in vs only
#pragma unroll
    for (int k = 0; k < CPT; ++k) {
        const int c = cellp[k];
        const bool real = c >= 0;
        const int g = real ? c : (c <= -2 ? -2 - c : 0);
        float co[4];
#pragma unroll
        for (int d = 0; d < 4; ++d) {
            const int ff = (th0.z >> (2 * d)) & 3;
            const int nb = real ? t.nbr[ff * N + g] : -1;
            if (flags & 1) co[d] = nb >= 0 ? off[(int)t.rev[ff * N + g] * N + nb] : 0.f;
            else co[d] = nb >= 0 ? off[ff * N + g] : 0.f;
        }
        co4[k * T + tid] = make_float4(co[0], co[1], co[2], co[3]);
        cdg[k * T + tid] = real ? dg[g] : 0.f;
        x[k] = (c != -1 && !zero_init) ? xo[g] : 0.f;  // ghost replicas start from their owner's value
        r[k] = real ? f[g] : 0.f;
        ap[k] = 0.f;
    }
    const uint32_t peer_red = mapa_u32(red_addr, (uint32_t)(lane < CS ? lane : 0));
    const uint32_t peer_mb = mapa_u32(mb_addr, (uint32_t)(lane < CS ? lane : 0));
    cluster_sync_all();                                // barriers initialised, shared memory filled everywhere

    // Two-level sum over the cluster: warp shuffle -> one partial per warp in this CTA's shared memory -> warp 0 adds them in
    // fixed order and pushes ONE value to every CTA of the cluster (CS st.async per CTA and exchange instead of NW * CS:
    // the transaction-count updates of the receiving barrier serialise) -> every thread adds the CS totals in rank order.
    uint32_t parA = 0, parB = 0;
    auto exchange = [&](float a0, const uint32_t which, uint32_t &par, const uint32_t bytes) -> float {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) a0 += __shfl_xor_sync(0xffffffffu, a0, o);
        if (lane == 0) {
            wpart[which * NW + warp] = a0;
            asm volatile("mbarrier.arrive.release.cta.shared::cta.b64 _, [%0];" ::"r"(mb_addr + 16u + 8u * which) : "memory");
        }
        if (warp == 0) {
            mbar_wait_sleep(mb_addr + 16u + 8u * which, par);
            float s1 = lane < NW ? wpart[which * NW + lane] : 0.f;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s1 += __shfl_xor_sync(0xffffffffu, s1, o);
            if (lane < CS) st_async_f32(peer_red + 4u * (which * CS + rank), s1, peer_mb + 8u * which);
        }
        mbar_wait_sleep(mb_addr + 8u * which, par); par ^= 1u;
        float s0 = 0.f;
#pragma unroll
        for (int q = 0; q < CS; ++q) s0 += red[which * CS + q];
        if (tid == 0) mbar_arrive_expect_tx(mb_addr + 8u * which, bytes);   // re-arm (see k_cg_cluster_mb)
        return s0;
    };
    auto row_of = [&](const float (&v)[CPT], int kk) -> float {
        float s = v[0];
#pragma unroll
        for (int k = 1; k < CPT; ++k) s = (kk == k) ? v[k] : s;
        return s;
    };
    // ap = P v for the vector v published in vs (own column: a sliding window of CPT + 2 loads, east / west: 2 per row);
    // returns this thread's part of <v, P v>
    auto spmv = [&]() -> float {
        float a0 = 0.f, a1 = 0.f;                      // two chains: the sum is on the critical path of the iteration
        float vsouth = vp[-S], vc = vp[0];
#pragma unroll
        for (int k = 0; k < CPT; ++k) {
            const float *row = vp + k * S;
            const float vnorth = row[S];
            const float4 o = co4[k * T + tid];
            float s = cdg[k * T + tid] * vc;
            s = fmaf(o.x, row[-1], s);
            s = fmaf(o.y, row[1], s);
            s = fmaf(o.z, vsouth, s);
            s = fmaf(o.w, vnorth, s);
            ap[k] = s;
            if (k & 1) a1 = fmaf(vc, s, a1); else a0 = fmaf(vc, s, a0);
            vsouth = vc; vc = vnorth;
        }
        return a0 + a1;
    };
    auto mirror_local_ghosts = [&]() {                 // after the vector has been stored: owners' values -> local ghost slots
        __syncthreads();
        if (n_lex) {                                   // (uniform over the CTA)
            for (int e = tid; e < n_lex; e += T) { const uint2 ex = lex[e]; vs[ex.y] = vs[ex.x]; }
            __syncthreads();
        }
    };
    auto publish_x = [&]() {
#pragma unroll
        for (int k = 0; k < CPT; ++k) vp[k * S] = x[k];
        mirror_local_ghosts();
    };
    // p = r + beta p in place in vs; remote ghost rows use the residual they received.  advance_x: also the deferred
    // x += alpha p of the LAZY order, from the same load of p_old (ghost replicas too, so they stay equal to their owners)
    auto new_direction = [&](float beta, float alpha, bool advance_x) {
        if (rm) {                                      // (r of a ghost row is zero otherwise: its coefficients are)
            int n = 0;
#pragma unroll
            for (int k = 0; k < CPT; ++k) if (rm & (1u << k)) r[k] = rgp[n++];
        }
#pragma unroll
        for (int k = 0; k < CPT; ++k) ap[k] = vp[k * S];   // (loads first: the stores below would otherwise serialise them; A p is dead here)
#pragma unroll
        for (int k = 0; k < CPT; ++k) vp[k * S] = fmaf(beta, ap[k], r[k]);
        if (advance_x) {
#pragma unroll
            for (int k = 0; k < CPT; ++k) x[k] = fmaf(alpha, ap[k], x[k]);
        }
        if (rm) {
#pragma unroll
            for (int k = 0; k < CPT; ++k) if (rm & (1u << k)) r[k] = 0.f;
        }
        mirror_local_ghosts();
    };
    auto residual_norm2 = [&]() -> float {             // exchange B: <r,r> + residuals of the remotely mirrored rows
        for (int j = 0; j < re_cnt; ++j) {
            const uint2 ex = rex[re_off + j];
            st_async_f32(ex.y, row_of(r, (int)(ex.x & 0xff)), mapa_u32(mb_addr + 8, ex.x >> 8));
        }
        float a0 = 0.f, a1 = 0.f;
#pragma unroll
        for (int k = 0; k < CPT; k += 2) { a0 = fmaf(r[k], r[k], a0); if (k + 1 < CPT) a1 = fmaf(r[k + 1], r[k + 1], a1); }
        return exchange(a0 + a1, 1u, parB, bytesB);
    };

    float nz = 0.f;
#pragma unroll
    for (int k = 0; k < CPT; ++k) nz += (r[k] != 0.f) ? 1.f : 0.f;
    const float nzt = exchange(nz, 0u, parA, bytesA);
    int used = -1; float fin = 0.f;
    bool solved = false;
    if (!(nzt > 0.f)) {
#pragma unroll
        for (int k = 0; k < CPT; ++k) x[k] = 0.f;
    } else {
        solved = true;
        if (!zero_init) {                              // r = f - P x0
            publish_x();
            (void)spmv();
#pragma unroll
            for (int k = 0; k < CPT; ++k) r[k] -= ap[k];
            __syncthreads();                           // everyone is done reading vs (= x) before it becomes p
        }
#pragma unroll
        for (int k = 0; k < CPT; ++k) bestp[k * T] = x[k];
        float rho = residual_norm2();
        new_direction(0.f, 0.f, false);                // p = r (vs holds zeros or x0: 0 * finite + r)
        float bestc = 0.f, lastc = 0.f; int best_it = -1, rising = 0;
        bool take_best = false;
        bool pending = false;                          // LAZY: the best iterate is x + alpha p of this iteration, not stored yet
        bool advance = false;                          // LAZY: the loop left with the current iterate, x += alpha p is still due
        float alpha = 0.f;
        int until_reset = reset_steps > 0 ? reset_steps - 1 : -1;   // iterations left before the next residual reset
        for (int i = 0; i < maxit; ++i) {
            if (until_reset == 0) {
                // r = f - P x ; p = r ; rho = <r,r>   (CG.cu:281-302).  x of the ghost rows is already there.
                until_reset = reset_steps;
                (void)exchange(0.f, 0u, parA, bytesA);  // keeps A / B alternating
                publish_x();
                (void)spmv();
#pragma unroll
                for (int k = 0; k < CPT; ++k) { const int c = cellp[k]; r[k] = (c >= 0 ? f[c] : 0.f) - ap[k]; }
                __syncthreads();
                rho = residual_norm2();
                new_direction(0.f, 0.f, false);
            }
            --until_reset;
            const float pap = exchange(spmv(), 0u, parA, bytesA);
            alpha = rho / pap;
#pragma unroll
            for (int k = 0; k < CPT; ++k) {
                if (!LAZY) x[k] = fmaf(alpha, vp[k * S], x[k]);
                r[k] = fmaf(-alpha, ap[k], r[k]);
            }
            const float rr2 = residual_norm2();
            const float crit = sqrtf(rr2) * norm;
            // ONE loop exit: with several `break`s (each with its own live iterate) the compiler copied all CPT registers of x in front
            // of every test, 70 of the 625 instructions of an iteration (profiles/r02_cg_strip_development.md)
            int stop = isfinite(crit) ? 0 : 1;         // 1: leave with the current iterate, 2: leave with the best one
            used = i; fin = crit;
            if (!stop) {
                if (i == 0 || crit < bestc) {
                    bestc = crit; best_it = i;
                    if (LAZY) pending = true;
                    else {
#pragma unroll
                        for (int k = 0; k < CPT; ++k) bestp[k * T] = x[k];
                    }
                } else if (LAZY && pending) {          // x is not advanced yet: it is the iterate of best_it
                    pending = false;
#pragma unroll
                    for (int k = 0; k < CPT; ++k) bestp[k * T] = x[k];
                }
                if (i > 0 && crit >= lastc) ++rising; else rising = 0;
                lastc = crit;
                if (crit < tol) stop = 1;
                else if (i == maxit - 1 || rising >= 100) stop = 2;
            }
            asm volatile("" : "+r"(stop));             // opaque: keeps the compiler from threading the exits apart again
            if (stop) {
                take_best = stop == 2 && !pending;     // (pending: this iteration improved, best_it == i, bestc == crit)
                advance = LAZY && !take_best;
                break;
            }
            const float beta = rr2 / rho;
            rho = rr2;
            new_direction(beta, alpha, LAZY);
        }
        if (take_best) {
#pragma unroll
            for (int k = 0; k < CPT; ++k) x[k] = bestp[k * T];
            used = best_it; fin = bestc;
        } else if (advance) {
#pragma unroll
            for (int k = 0; k < CPT; ++k) x[k] = fmaf(alpha, vp[k * S], x[k]);
        }
    }
    float mean = 0.f;
    if (solved && !(flags & 2)) {
        float sx = 0.f;
#pragma unroll
        for (int k = 0; k < CPT; ++k) sx += (cellp[k] >= 0) ? x[k] : 0.f;
        mean = exchange(sx, 0u, parA, bytesA) / (float)N;
    }
    if (mean_out && tid == 0 && rank == 0) mean_out[b] = mean;
#pragma unroll
    for (int k = 0; k < CPT; ++k) { const int c = cellp[k]; if (c >= 0) xo[c] = x[k] - mean; }
    if (tid == 0 && rank == 0) { iters[b * 8 + 2 + slot] = used; resid[b * 8 + 2 + slot] = fin; iter_total[b * 2] += (unsigned long long)(used + 1); }
    cluster_sync_all();   // keep peer shared memory (and in-flight st.async targets) alive until everyone is done
}

// ------------------------------------------------------------------------------------------------
// Krylov solvers, implementation 12: the strip kernel with TWO environments per cluster, software-interleaved.
// k_cg_strip is one dependent chain per iteration (SpMV -> all-reduce -> update -> all-reduce -> direction): while a CTA waits
// for a cluster exchange (~850 cycles, twice per iteration) its SM idles, and co-resident CTAs do not fix that (their compute
// phases collide as often as they interleave, profiles/r02_cg_strip_development.md).  Here every CTA holds the strips of two
// independent systems (half the rows per thread each, so a cluster spans twice the CTAs) and runs them in a fixed order:
//     SpMV(e0) -> start <p,Ap>(e0) -> SpMV(e1) -> start <p,Ap>(e1) -> finish(e0), x/r update, start <r,r>(e0) -> finish(e1), ...
// An exchange is split in a non-blocking start (warp partials -> the LAST arriving warp of the CTA adds them in fixed order and
// pushes one value to every CTA of the cluster) and a finish (wait on the transaction barrier, add the CS totals in rank
// order), so the flight time of one system's reduction is covered by the other system's arithmetic.  Arithmetic, operation
// order and stopping rules per system are those of k_cg_strip with the eager bookkeeping order; results are NOT bit-identical to
// cg_impl 11, whose layout (17 rows per thread, half the CTAs) sums the dot products in another order.  The two systems converge independently,
// the faster one idles until both are done.  Same tables (strip_plan.py) with the shape (T, CPT) of this kernel.
// ------------------------------------------------------------------------------------------------
template <int E> struct EnvTag { static constexpr int value = E; };

template <int T, int CPT, int CS>
__global__ void __launch_bounds__(T, 1) k_cg_strip2(Tab t, const float *__restrict__ Poff, const float *__restrict__ Pdiag,
                                                    const float *__restrict__ Rhs, float *__restrict__ Xout, int B,
                                                    int maxit, float tol, int zero_init, int reset_steps, int slot,
                                                    const int32_t *__restrict__ active, int32_t *__restrict__ iters,
                                                    float *__restrict__ resid, unsigned long long *__restrict__ iter_total,
                                                    int flags, float *__restrict__ mean_out, float *__restrict__ best) {
    static_assert(T % 32 == 0, "whole warps only");
    constexpr int NW = T / 32;
    constexpr uint32_t FULL = 0xffffffffu;
    const int b0 = 2 * (int)(blockIdx.x / CS);
    uint32_t rank;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
    bool on[2];
    on[0] = !active || active[b0];
    on[1] = b0 + 1 < B && (!active || active[b0 + 1]);
    if (!on[0] && !on[1]) return;                      // (uniform over the cluster)
    extern __shared__ __align__(16) float smem[];
    const int N = t.N, SL = t.st_slots, G = t.st_gmax;
    // per environment: co4 [CPT][T] float4 | cdg [CPT][T] | vs [SL] | rs [G] | red [2][CS] | wpart [2][NW]   (ENVF floats, multiple of 4)
    const int ENVF = (5 * CPT * T + SL + G + 2 * CS + 2 * NW + 3) & ~3;
    unsigned long long *mb = (unsigned long long *)(smem + 2 * ENVF);      // [e][which]: cluster transaction barriers
    unsigned int *cnt = (unsigned int *)(mb + 4);                          // [e][which]: warps of this CTA that have delivered their partial
    uint2 *rex = (uint2 *)(cnt + 4);                   // [st_remax] {k | dest rank << 8, cluster address of the destination in rs of environment 0}
    uint2 *lex = rex + t.st_remax;                     // [st_lemax] {owner's slot, mirror slot} in vs
    const float norm = 1.0f / sqrtf((float)N);
    const uint32_t mb_addr = smem_u32(mb);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    const int4 th0 = reinterpret_cast<const int4 *>(t.st_thread)[((size_t)rank * T + tid) * 2];
    const int4 th1 = reinterpret_cast<const int4 *>(t.st_thread)[((size_t)rank * T + tid) * 2 + 1];
    const int S = th0.y;
    const int vp_off = 5 * CPT * T + th0.x;            // slot of row 0 of this thread, relative to the environment's base
    const int re_off = th0.w & 0xffff, re_cnt = (th0.w >> 16) & 0xff;
    const int n_lex = t.st_cnt[4 * rank + 2];
    const int rg_off = 5 * CPT * T + SL + th1.y;       // first remote ghost row of this thread in the receive buffer
    const uint32_t rm = (uint32_t)th1.z;               // remote ghost rows of this thread (bit k)
    const int32_t *cellp = t.st_cell + ((size_t)rank * T + tid) * CPT;
    const uint32_t bytesA = CS * 4u, bytesB = CS * 4u + 4u * (uint32_t)t.st_cnt[4 * rank];
    if (tid == 0) {
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            mbar_init(mb_addr + 16u * e, 1); mbar_init(mb_addr + 16u * e + 8u, 1);
            cnt[2 * e] = 0u; cnt[2 * e + 1] = 0u;
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
#pragma unroll
        for (int e = 0; e < 2; ++e) { mbar_arrive_expect_tx(mb_addr + 16u * e, bytesA); mbar_arrive_expect_tx(mb_addr + 16u * e + 8u, bytesB); }
    }
    {
        const uint32_t rs_addr = smem_u32(smem + 5 * CPT * T + SL);
        for (int e = tid; e < t.st_cnt[4 * rank + 1]; e += T) {
            const int32_t a = t.st_rexp[((size_t)rank * t.st_remax + e) * 2], d = t.st_rexp[((size_t)rank * t.st_remax + e) * 2 + 1];
            rex[e] = make_uint2((uint32_t)a, mapa_u32(rs_addr + 4u * (uint32_t)d, (uint32_t)a >> 8));
        }
    }
    for (int e = tid; e < n_lex; e += T)
        lex[e] = make_uint2((uint32_t)t.st_lexp[((size_t)rank * t.st_lemax + e) * 2], (uint32_t)t.st_lexp[((size_t)rank * t.st_lemax + e) * 2 + 1]);
#pragma unroll
    for (int e = 0; e < 2; ++e)
        for (int i = tid; i < SL + G; i += T) smem[e * ENVF + 5 * CPT * T + i] = 0.f;   // vs and rs (pads, dead slots)

    float x[2][CPT], r[2][CPT], ap[2][CPT];            // the search directions live in vs only
    uint32_t par[2][2] = {{0u, 0u}, {0u, 0u}};
    auto load_env = [&](auto E) {
        constexpr int e = decltype(E)::value;
        const int b = b0 + e;
        const float *off = Poff + (size_t)b * 4 * N, *dg = Pdiag + (size_t)b * N, *f = Rhs + (size_t)b * N;
        const float *xo = Xout + (size_t)b * N;
        float4 *co4 = reinterpret_cast<float4 *>(smem + e * ENVF);
        float *cdg = smem + e * ENVF + 4 * CPT * T;
#pragma unroll
        for (int k = 0; k < CPT; ++k) {
            const int c = cellp[k];
            const bool real = c >= 0;
            const int g = real ? c : (c <= -2 ? -2 - c : 0);
            float co[4];
#pragma unroll
            for (int d = 0; d < 4; ++d) {
                const int ff = (th0.z >> (2 * d)) & 3;
                const int nb = real ? t.nbr[ff * N + g] : -1;
                if (flags & 1) co[d] = nb >= 0 ? off[(int)t.rev[ff * N + g] * N + nb] : 0.f;
                else co[d] = nb >= 0 ? off[ff * N + g] : 0.f;
            }
            co4[k * T + tid] = make_float4(co[0], co[1], co[2], co[3]);
            cdg[k * T + tid] = real ? dg[g] : 0.f;
            x[e][k] = (c != -1 && !zero_init) ? xo[g] : 0.f;   // ghost replicas start from their owner's value
            r[e][k] = real ? f[g] : 0.f;
            ap[e][k] = 0.f;
        }
    };
#pragma unroll
    for (int k = 0; k < CPT; ++k) { x[0][k] = r[0][k] = ap[0][k] = 0.f; x[1][k] = r[1][k] = ap[1][k] = 0.f; }
    if (on[0]) load_env(EnvTag<0>{});
    if (on[1]) load_env(EnvTag<1>{});
    const uint32_t peer_smem = mapa_u32(smem_u32(smem), (uint32_t)(lane < CS ? lane : 0));
    const uint32_t peer_mb = mapa_u32(mb_addr, (uint32_t)(lane < CS ? lane : 0));
    cluster_sync_all();                                // barriers initialised, shared memory filled everywhere

    // ---- exchange, split.  which: 0 = A (<p,Ap>, also non-zero count, mean), 1 = B (<r,r> + ghost residuals) ----------------------
    auto xstart = [&](auto E, auto W, float a0) {
        constexpr int e = decltype(E)::value;
        constexpr uint32_t which = decltype(W)::value;
        float *red = smem + e * ENVF + 5 * CPT * T + SL + G;
        volatile float *wpart = red + 2 * CS;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) a0 += __shfl_xor_sync(FULL, a0, o);
        unsigned int last = 0u;
        if (lane == 0) {
            wpart[which * NW + warp] = a0;
            __threadfence_block();
            last = atomicInc(&cnt[2 * e + which], (unsigned int)(NW - 1)) == (unsigned int)(NW - 1);
        }
        last = __shfl_sync(FULL, last, 0);
        if (last) {                                    // every warp of this CTA has delivered: add in fixed order, one value to every CTA
            __threadfence_block();
            float s1 = lane < NW ? wpart[which * NW + lane] : 0.f;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s1 += __shfl_xor_sync(FULL, s1, o);
            if (lane < CS)
                st_async_f32(peer_smem + 4u * (uint32_t)(e * ENVF + 5 * CPT * T + SL + G + which * CS + rank), s1, peer_mb + 16u * e + 8u * which);
        }
    };
    auto xfinish = [&](auto E, auto W) -> float {
        constexpr int e = decltype(E)::value;
        constexpr uint32_t which = decltype(W)::value;
        const float *red = smem + e * ENVF + 5 * CPT * T + SL + G;
        mbar_wait_sleep(mb_addr + 16u * e + 8u * which, par[e][which]); par[e][which] ^= 1u;
        float s0 = 0.f;
#pragma unroll
        for (int q = 0; q < CS; ++q) s0 += red[which * CS + q];
        if (tid == 0) mbar_arrive_expect_tx(mb_addr + 16u * e + 8u * which, which ? bytesB : bytesA);   // re-arm (see k_cg_cluster_mb)
        return s0;
    };
    auto spmv = [&](auto E) -> float {                 // ap = P v for the vector published in vs; returns this thread's part of <v, P v>
        constexpr int e = decltype(E)::value;
        const float4 *co4 = reinterpret_cast<const float4 *>(smem + e * ENVF);
        const float *cdg = smem + e * ENVF + 4 * CPT * T, *vp = smem + e * ENVF + vp_off;
        float a0 = 0.f, a1 = 0.f;
        float vsouth = vp[-S], vc = vp[0];
#pragma unroll
        for (int k = 0; k < CPT; ++k) {
            const float *row = vp + k * S;
            const float vnorth = row[S];
            const float4 o = co4[k * T + tid];
            float s = cdg[k * T + tid] * vc;
            s = fmaf(o.x, row[-1], s);
            s = fmaf(o.y, row[1], s);
            s = fmaf(o.z, vsouth, s);
            s = fmaf(o.w, vnorth, s);
            ap[e][k] = s;
            if (k & 1) a1 = fmaf(vc, s, a1); else a0 = fmaf(vc, s, a0);
            vsouth = vc; vc = vnorth;
        }
        return a0 + a1;
    };
    auto mirror = [&]() {                              // after vectors have been stored: owners' values -> local ghost slots, both environments
        __syncthreads();
        if (n_lex) {                                   // (uniform over the CTA)
            for (int i = tid; i < n_lex; i += T) {
                const uint2 ex = lex[i];
                float *v0 = smem + 5 * CPT * T, *v1 = v0 + ENVF;
                v0[ex.y] = v0[ex.x]; v1[ex.y] = v1[ex.x];
            }
            __syncthreads();
        }
    };
    auto store_x = [&](auto E) {
        constexpr int e = decltype(E)::value;
        float *vp = smem + e * ENVF + vp_off;
#pragma unroll
        for (int k = 0; k < CPT; ++k) vp[k * S] = x[e][k];
    };
    auto store_direction = [&](auto E, float beta) {   // p = r + beta p in place in vs; remote ghost rows use the residual they received
        constexpr int e = decltype(E)::value;
        float *vp = smem + e * ENVF + vp_off;
        if (rm) {
            const float *rgp = smem + e * ENVF + rg_off;
            int n = 0;
#pragma unroll
            for (int k = 0; k < CPT; ++k) if (rm & (1u << k)) r[e][k] = rgp[n++];
        }
#pragma unroll
        for (int k = 0; k < CPT; ++k) ap[e][k] = vp[k * S];      // (loads first; A p is dead here)
#pragma unroll
        for (int k = 0; k < CPT; ++k) vp[k * S] = fmaf(beta, ap[e][k], r[e][k]);
        if (rm) {
#pragma unroll
            for (int k = 0; k < CPT; ++k) if (rm & (1u << k)) r[e][k] = 0.f;
        }
    };
    auto residual_start = [&](auto E) {                // exchange B: <r,r> + residuals of the remotely mirrored rows
        constexpr int e = decltype(E)::value;
        if (re_cnt) {                                  // the export list of a thread is sorted by row: rows stay compile-time indices (registers)
            int j = 0;
            uint2 ex = rex[re_off];
#pragma unroll
            for (int k = 0; k < CPT; ++k) {
                while (j < re_cnt && (int)(ex.x & 0xff) == k) {
                    st_async_f32(ex.y + 4u * (uint32_t)(e * ENVF), r[e][k], mapa_u32(mb_addr + 16u * e + 8u, ex.x >> 8));
                    if (++j < re_cnt) ex = rex[re_off + j];
                }
            }
        }
        float a0 = 0.f, a1 = 0.f;
#pragma unroll
        for (int k = 0; k < CPT; k += 2) { a0 = fmaf(r[e][k], r[e][k], a0); if (k + 1 < CPT) a1 = fmaf(r[e][k + 1], r[e][k + 1], a1); }
        xstart(E, EnvTag<1>{}, a0 + a1);
    };

    bool run[2] = {false, false}, solved[2] = {false, false};
    int used[2] = {-1, -1}, it[2] = {0, 0}, best_it[2] = {-1, -1}, rising[2] = {0, 0}, until_reset[2];
    float fin[2] = {0.f, 0.f}, rho[2] = {0.f, 0.f}, bestc[2] = {0.f, 0.f}, lastc[2] = {0.f, 0.f};
    until_reset[0] = until_reset[1] = reset_steps > 0 ? reset_steps - 1 : -1;   // iterations left before the next residual reset

    auto count_start = [&](auto E) {
        constexpr int e = decltype(E)::value;
        float nz = 0.f;
#pragma unroll
        for (int k = 0; k < CPT; ++k) nz += (r[e][k] != 0.f) ? 1.f : 0.f;
        xstart(E, EnvTag<0>{}, nz);
    };
    auto count_finish = [&](auto E) {
        constexpr int e = decltype(E)::value;
        const float nzt = xfinish(E, EnvTag<0>{});
        run[e] = solved[e] = nzt > 0.f;
        if (!run[e]) {
#pragma unroll
            for (int k = 0; k < CPT; ++k) x[e][k] = 0.f;
        }
    };
    if (on[0]) count_start(EnvTag<0>{});
    if (on[1]) count_start(EnvTag<1>{});
    if (on[0]) count_finish(EnvTag<0>{});
    if (on[1]) count_finish(EnvTag<1>{});

    auto initial_residual = [&](auto E) {              // r = f - P x0 (x0 published in vs)
        constexpr int e = decltype(E)::value;
        (void)spmv(E);
#pragma unroll
        for (int k = 0; k < CPT; ++k) r[e][k] -= ap[e][k];
    };
    auto save_best = [&](auto E) {
        constexpr int e = decltype(E)::value;
        float *bestp = best + ((size_t)(b0 + e) * CS + rank) * T * CPT + tid;
#pragma unroll
        for (int k = 0; k < CPT; ++k) bestp[k * T] = x[e][k];
    };
    if (run[0] || run[1]) {
        if (!zero_init) {
            if (run[0]) store_x(EnvTag<0>{});
            if (run[1]) store_x(EnvTag<1>{});
            mirror();
            if (run[0]) initial_residual(EnvTag<0>{});
            if (run[1]) initial_residual(EnvTag<1>{});
            __syncthreads();                           // everyone is done reading vs (= x) before it becomes p
        }
        if (run[0]) { save_best(EnvTag<0>{}); residual_start(EnvTag<0>{}); }
        if (run[1]) { save_best(EnvTag<1>{}); residual_start(EnvTag<1>{}); }
        if (run[0]) { rho[0] = xfinish(EnvTag<0>{}, EnvTag<1>{}); store_direction(EnvTag<0>{}, 0.f); }   // p = r (vs holds zeros or x0: 0 * finite + r)
        if (run[1]) { rho[1] = xfinish(EnvTag<1>{}, EnvTag<1>{}); store_direction(EnvTag<1>{}, 0.f); }
        mirror();
    }

    // one system's share of the three phases of an iteration
    auto phase1 = [&](auto E) { xstart(E, EnvTag<0>{}, spmv(E)); };
    auto phase2 = [&](auto E) {
        constexpr int e = decltype(E)::value;
        const float pap = xfinish(E, EnvTag<0>{});
        const float alpha = rho[e] / pap;
        const float *vp = smem + e * ENVF + vp_off;
#pragma unroll
        for (int k = 0; k < CPT; ++k) {
            x[e][k] = fmaf(alpha, vp[k * S], x[e][k]);
            r[e][k] = fmaf(-alpha, ap[e][k], r[e][k]);
        }
        residual_start(E);
    };
    auto phase3 = [&](auto E) {
        constexpr int e = decltype(E)::value;
        const float rr2 = xfinish(E, EnvTag<1>{});
        const float crit = sqrtf(rr2) * norm;
        const int i = it[e];
        if (!isfinite(crit)) { used[e] = i; fin[e] = crit; run[e] = false; return; }
        if (i == 0 || crit < bestc[e]) { bestc[e] = crit; best_it[e] = i; save_best(E); }
        if (i > 0 && crit >= lastc[e]) ++rising[e]; else rising[e] = 0;
        lastc[e] = crit; used[e] = i; fin[e] = crit;
        if (crit < tol) { run[e] = false; return; }
        if (i == maxit - 1 || rising[e] >= 100) {
            const float *bestp = best + ((size_t)(b0 + e) * CS + rank) * T * CPT + tid;
#pragma unroll
            for (int k = 0; k < CPT; ++k) x[e][k] = bestp[k * T];
            used[e] = best_it[e]; fin[e] = bestc[e];
            run[e] = false; return;
        }
        const float beta = rr2 / rho[e];
        rho[e] = rr2;
        store_direction(E, beta);
        it[e] = i + 1;
    };
    auto reset_a = [&](auto E) { constexpr int e = decltype(E)::value; until_reset[e] = reset_steps; xstart(E, EnvTag<0>{}, 0.f); };   // keeps A / B alternating
    auto reset_b = [&](auto E) { (void)xfinish(E, EnvTag<0>{}); store_x(E); };
    auto reset_c = [&](auto E) {                       // r = f - P x ; rho = <r,r>   (CG.cu:281-302).  x of the ghost rows is already there.
        constexpr int e = decltype(E)::value;
        const float *f = Rhs + (size_t)(b0 + e) * N;
        (void)spmv(E);
#pragma unroll
        for (int k = 0; k < CPT; ++k) { const int c = cellp[k]; r[e][k] = (c >= 0 ? f[c] : 0.f) - ap[e][k]; }
    };
    auto reset_d = [&](auto E) { constexpr int e = decltype(E)::value; rho[e] = xfinish(E, EnvTag<1>{}); store_direction(E, 0.f); };

    if (maxit <= 0) run[0] = run[1] = false;
    while (run[0] || run[1]) {
        const bool rs0 = run[0] && until_reset[0] == 0, rs1 = run[1] && until_reset[1] == 0;
        if (rs0 || rs1) {
            if (rs0) reset_a(EnvTag<0>{});
            if (rs1) reset_a(EnvTag<1>{});
            if (rs0) reset_b(EnvTag<0>{});
            if (rs1) reset_b(EnvTag<1>{});
            mirror();
            if (rs0) reset_c(EnvTag<0>{});
            if (rs1) reset_c(EnvTag<1>{});
            __syncthreads();
            if (rs0) residual_start(EnvTag<0>{});
            if (rs1) residual_start(EnvTag<1>{});
            if (rs0) reset_d(EnvTag<0>{});
            if (rs1) reset_d(EnvTag<1>{});
            mirror();
        }
        if (run[0]) --until_reset[0];
        if (run[1]) --until_reset[1];
        if (run[0]) phase1(EnvTag<0>{});
        if (run[1]) phase1(EnvTag<1>{});
        const bool r0 = run[0], r1 = run[1];
        if (r0) phase2(EnvTag<0>{});
        if (r1) phase2(EnvTag<1>{});
        if (r0) phase3(EnvTag<0>{});
        if (r1) phase3(EnvTag<1>{});
        if (run[0] || run[1]) mirror();
    }

    auto mean_start = [&](auto E) {
        constexpr int e = decltype(E)::value;
        float sx = 0.f;
#pragma unroll
        for (int k = 0; k < CPT; ++k) sx += (cellp[k] >= 0) ? x[e][k] : 0.f;
        xstart(E, EnvTag<0>{}, sx);
    };
    auto finish_env = [&](auto E, bool with_mean) {
        constexpr int e = decltype(E)::value;
        const int b = b0 + e;
        float mean = 0.f;
        if (with_mean) mean = xfinish(E, EnvTag<0>{}) / (float)N;
        if (mean_out && tid == 0 && rank == 0) mean_out[b] = mean;
        float *xo = Xout + (size_t)b * N;
#pragma unroll
        for (int k = 0; k < CPT; ++k) { const int c = cellp[k]; if (c >= 0) xo[c] = x[e][k] - mean; }
        if (tid == 0 && rank == 0) { iters[b * 8 + 2 + slot] = used[e]; resid[b * 8 + 2 + slot] = fin[e]; iter_total[b * 2] += (unsigned long long)(used[e] + 1); }
    };
    const bool m0 = on[0] && solved[0] && !(flags & 2), m1 = on[1] && solved[1] && !(flags & 2);
    if (m0) mean_start(EnvTag<0>{});
    if (m1) mean_start(EnvTag<1>{});
    if (on[0]) finish_env(EnvTag<0>{}, m0);
    if (on[1]) finish_env(EnvTag<1>{}, m1);
    cluster_sync_all();   // keep peer shared memory (and in-flight st.async targets) alive until everyone is done
}

// ------------------------------------------------------------------------------------------------
// BiCGStab on chip: one cluster per environment, same mbarrier protocol as the CG above.  r, p, x and the
// shadow residual live in shared memory (r and p are the two vectors the neighbours gather), v, t and the
// stencil in registers.  Operation order follows BICG.cu:276-366; rho of the next iteration is reduced
// together with the residual norm of the second half step (same operands, one reduction less).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void st_async_f32x4(uint32_t cluster_addr, float a, float b, float c, float d, uint32_t cluster_mbar) {
    asm volatile("st.async.shared::cluster.mbarrier::complete_tx::bytes.v4.f32 [%0], {%1, %2, %3, %4}, [%5];"
                 ::"r"(cluster_addr), "f"(a), "f"(b), "f"(c), "f"(d), "r"(cluster_mbar) : "memory");
}

template <int T, int CPT, int CS, int NC>
__global__ void __launch_bounds__(T, 1) k_bicgstab_cluster(Tab t, const float *__restrict__ Coff, const float *__restrict__ Adiag,
                                                            const float *__restrict__ Rhs, float *__restrict__ X,
                                                            int maxit, float tol, int zero_init, const int32_t *__restrict__ active,
                                                            int32_t *__restrict__ iters, float *__restrict__ resid,
                                                            unsigned long long *__restrict__ iter_total, int transposed) {
    constexpr int NW = T / 32;
    constexpr int NP = NW * CS;
    constexpr int PAD = T * CPT;
    const int b = blockIdx.x / CS;
    uint32_t rank;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
    if (active && !active[b]) return;
    extern __shared__ __align__(16) float smem[];
    const int N = t.N;
    const int per = (N + CS - 1) / CS;
    const int start = (int)rank * per;
    const int cnt = max(0, min(per, N - start));
    float *rs = smem;                            // [NC][PAD] residual            (exposed to the neighbours)
    float *ps = smem + NC * PAD;                 // [NC][PAD] search direction    (exposed)
    float *ws = smem + 2 * NC * PAD;             // [NC][PAD] shadow residual r^_0
    float *xs = smem + 3 * NC * PAD;             // [NC][PAD] iterate
    float4 *red = (float4 *)(smem + 4 * NC * PAD);       // [2][NP] partials
    unsigned long long *mb = (unsigned long long *)(smem + 4 * NC * PAD + 2 * NP * 4);
    const float *off = Coff + (size_t)b * 4 * N, *dg = Adiag + (size_t)b * N;
    const float norm = 1.0f / sqrtf((float)N);
    const uint32_t rs_addr = smem_u32(rs), red_addr = smem_u32(red), mb_addr = smem_u32(mb);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    if (threadIdx.x == 0) {
        mbar_init(mb_addr, 1); mbar_init(mb_addr + 8, 1); mbar_init(mb_addr + 16, CS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        mbar_arrive_expect_tx(mb_addr, NP * 16);
        mbar_arrive_expect_tx(mb_addr + 8, NP * 16);
    }
    float cd[CPT], co[CPT][4], vv[NC][CPT], tt[NC][CPT];
    uint32_t na[CPT][4];                          // cluster address of the neighbour's slot in rs, component 0
#pragma unroll
    for (int k = 0; k < CPT; ++k) {
        const int l = threadIdx.x + k * T;
        const int g = start + l;
        const bool ok = l < cnt;
        cd[k] = ok ? dg[g] : 0.f;
#pragma unroll
        for (int ff = 0; ff < 4; ++ff) {
            const int nb = ok ? t.nbr[ff * N + g] : -1;
            if (transposed) co[k][ff] = (ok && nb >= 0) ? off[(int)t.rev[ff * N + g] * N + nb] : 0.f;
            else co[k][ff] = (ok && nb >= 0) ? off[ff * N + g] : 0.f;
            const int gi = nb >= 0 ? nb : (ok ? g : start);
            const int c = gi / per;
            na[k][ff] = mapa_u32(rs_addr + 4u * (uint32_t)(gi - c * per), (uint32_t)c);
        }
#pragma unroll
        for (int c = 0; c < NC; ++c) {
            xs[c * PAD + l] = (ok && !zero_init) ? X[(size_t)b * NC * N + (size_t)c * N + g] : 0.f;
            rs[c * PAD + l] = 0.f; ps[c * PAD + l] = 0.f; ws[c * PAD + l] = 0.f;
            vv[c][k] = 0.f; tt[c][k] = 0.f;
        }
    }
    const uint32_t peer_red = mapa_u32(red_addr, (uint32_t)(lane < CS ? lane : 0));
    const uint32_t peer_mb = mapa_u32(mb_addr, (uint32_t)(lane < CS ? lane : 0));
    cluster_sync_all();

    uint32_t rcount = 0, pphase = 0;
    auto cluster_sum4 = [&](float (&a)[4]) {
        const uint32_t w = rcount & 1u, par = (rcount >> 1) & 1u;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) a[q] += __shfl_xor_sync(0xffffffffu, a[q], o);
        }
        if (lane < CS) st_async_f32x4(peer_red + 16u * (w * NP + rank * NW + (uint32_t)warp), a[0], a[1], a[2], a[3], peer_mb + 8u * w);
        mbar_wait(mb_addr + 8u * w, par);
        const float4 *rp = red + w * NP;
        float4 s0 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int q = 0; q < (NP + 31) / 32; ++q)
            if (lane + 32 * q < NP) { const float4 v = rp[lane + 32 * q]; s0.x += v.x; s0.y += v.y; s0.z += v.z; s0.w += v.w; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            s0.x += __shfl_xor_sync(0xffffffffu, s0.x, o); s0.y += __shfl_xor_sync(0xffffffffu, s0.y, o);
            s0.z += __shfl_xor_sync(0xffffffffu, s0.z, o); s0.w += __shfl_xor_sync(0xffffffffu, s0.w, o);
        }
        if (threadIdx.x == 0) mbar_arrive_expect_tx(mb_addr + 8u * w, NP * 16);
        ++rcount;
        a[0] = s0.x; a[1] = s0.y; a[2] = s0.z; a[3] = s0.w;
    };
    auto publish = [&]() {
        __syncthreads();
        if (threadIdx.x < CS) mbar_arrive_remote_release(mapa_u32(mb_addr + 16, threadIdx.x));
    };
    auto acquire = [&]() { mbar_wait(mb_addr + 16, pphase); pphase ^= 1u; };
    // row k of C times an exposed array: `arr` = local base of the array, aoff = its byte offset from rs
    auto apply = [&](int k, const float *arr, uint32_t aoff) -> float {
        float s = cd[k] * arr[threadIdx.x + k * T];
#pragma unroll
        for (int ff = 0; ff < 4; ++ff) s += co[k][ff] * ld_dsmem_f32(na[k][ff] + aoff);
        return s;
    };
    auto load_f = [&](int c, int k) -> float { const int l = threadIdx.x + k * T; return l < cnt ? Rhs[(size_t)b * NC * N + (size_t)c * N + start + l] : 0.f; };

    float acc[4];
    // r0 = f - C x0 ; shadow = r0 ; p = r0
    if (!zero_init) {
#pragma unroll
        for (int c = 0; c < NC; ++c)
#pragma unroll
            for (int k = 0; k < CPT; ++k) ps[c * PAD + threadIdx.x + k * T] = xs[c * PAD + threadIdx.x + k * T];
        publish(); acquire();
#pragma unroll
        for (int c = 0; c < NC; ++c)
#pragma unroll
            for (int k = 0; k < CPT; ++k) tt[c][k] = load_f(c, k) - apply(k, ps + c * PAD, (uint32_t)((NC + c) * PAD * 4));
        acc[0] = acc[1] = acc[2] = acc[3] = 0.f;
        cluster_sum4(acc);                       // everyone is done reading ps (= x)
    } else {
#pragma unroll
        for (int c = 0; c < NC; ++c)
#pragma unroll
            for (int k = 0; k < CPT; ++k) tt[c][k] = load_f(c, k);
    }
    acc[0] = acc[1] = acc[2] = acc[3] = 0.f;
#pragma unroll
    for (int c = 0; c < NC; ++c)
#pragma unroll
        for (int k = 0; k < CPT; ++k) {
            const int l = c * PAD + threadIdx.x + k * T;
            rs[l] = tt[c][k]; ws[l] = tt[c][k]; ps[l] = tt[c][k];
            acc[c] += tt[c][k] * tt[c][k];
        }
    publish();                                   // p0 (= r0) exposed
    cluster_sum4(acc);                           // ||r0||^2 = <shadow, r0> = rho of the first iteration
    bool done[2] = {true, true}; int used[2] = {-1, -1}; float fin[2] = {0.f, 0.f};
    float rho[2] = {1.f, 1.f}, rho_next[2] = {1.f, 1.f}, alpha[2] = {1.f, 1.f}, omega[2] = {1.f, 1.f};
#pragma unroll
    for (int c = 0; c < NC; ++c) { fin[c] = sqrtf(acc[c]) * norm; done[c] = fin[c] < tol; rho_next[c] = acc[c]; }
    for (int i = 0; i < maxit && !(done[0] && done[NC - 1]); ++i) {
        // rho = <shadow, r> ; p = r + beta (p - omega v)      (ps already holds p - omega v from the last half step)
        if (i > 0) {
#pragma unroll
            for (int c = 0; c < NC; ++c) if (!done[c]) {
                const float beta = (rho_next[c] / rho[c]) * (alpha[c] / omega[c]);
#pragma unroll
                for (int k = 0; k < CPT; ++k) { const int l = c * PAD + threadIdx.x + k * T; ps[l] = rs[l] + beta * ps[l]; }
            }
            publish();
        }
#pragma unroll
        for (int c = 0; c < NC; ++c) if (!done[c]) rho[c] = rho_next[c];
        acquire();                               // p of every CTA visible
        // v = C p ; alpha = rho / <shadow, v>
        acc[0] = acc[1] = acc[2] = acc[3] = 0.f;
#pragma unroll
        for (int c = 0; c < NC; ++c) if (!done[c])
#pragma unroll
            for (int k = 0; k < CPT; ++k) {
                vv[c][k] = apply(k, ps + c * PAD, (uint32_t)((NC + c) * PAD * 4));
                acc[c] += ws[c * PAD + threadIdx.x + k * T] * vv[c][k];
            }
        cluster_sum4(acc);                       // completes only when every warp has finished gathering p
        float acc2[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int c = 0; c < NC; ++c) if (!done[c]) {
            alpha[c] = rho[c] / acc[c];
#pragma unroll
            for (int k = 0; k < CPT; ++k) {
                const int l = c * PAD + threadIdx.x + k * T;
                const float rn = rs[l] - alpha[c] * vv[c][k];
                rs[l] = rn; xs[l] += alpha[c] * ps[l];
                acc2[c] += rn * rn;
            }
        }
        publish();                               // r exposed for t = C r; the hand-shake overlaps the reduction
        cluster_sum4(acc2);
#pragma unroll
        for (int c = 0; c < NC; ++c) if (!done[c]) {
            const float nr = sqrtf(acc2[c]) * norm;
            used[c] = i; fin[c] = nr;
            if (!isfinite(nr) || nr < tol) done[c] = true;
        }
        acquire();
        // t = C r ; omega = <t,r>/<t,t>
        acc[0] = acc[1] = acc[2] = acc[3] = 0.f;
#pragma unroll
        for (int c = 0; c < NC; ++c) if (!done[c])
#pragma unroll
            for (int k = 0; k < CPT; ++k) {
                tt[c][k] = apply(k, rs + c * PAD, (uint32_t)(c * PAD * 4));
                const float rv = rs[c * PAD + threadIdx.x + k * T];
                acc[c] += tt[c][k] * rv; acc[2 + c] += tt[c][k] * tt[c][k];
            }
        cluster_sum4(acc);                       // every warp has finished gathering r
        acc2[0] = acc2[1] = acc2[2] = acc2[3] = 0.f;
#pragma unroll
        for (int c = 0; c < NC; ++c) if (!done[c]) {
            omega[c] = acc[c] / acc[2 + c];
#pragma unroll
            for (int k = 0; k < CPT; ++k) {
                const int l = c * PAD + threadIdx.x + k * T;
                const float rg = rs[l];
                xs[l] += omega[c] * rg;
                const float rn = rg - omega[c] * tt[c][k];
                rs[l] = rn;
                ps[l] = ps[l] - omega[c] * vv[c][k];          // p - omega v, finished into the new p at the top of the loop
                acc2[c] += rn * rn; acc2[2 + c] += ws[l] * rn;  // ||r||^2 and rho of the next iteration
            }
        }
        cluster_sum4(acc2);
#pragma unroll
        for (int c = 0; c < NC; ++c) if (!done[c]) {
            const float nr = sqrtf(acc2[c]) * norm;
            fin[c] = nr; rho_next[c] = acc2[2 + c];
            if (nr < tol) { done[c] = true; used[c] = i + 1; }
        }
    }
#pragma unroll
    for (int c = 0; c < NC; ++c)
#pragma unroll
        for (int k = 0; k < CPT; ++k) { const int l = threadIdx.x + k * T; if (l < cnt) X[(size_t)b * NC * N + (size_t)c * N + start + l] = xs[c * PAD + l]; }
    if (threadIdx.x == 0 && rank == 0) {
        if (NC == 2) {
            iters[b * 8 + 0] = used[0]; iters[b * 8 + 1] = used[1];
            resid[b * 8 + 0] = fin[0]; resid[b * 8 + 1] = fin[1];
            iter_total[b * 2 + 1] += (unsigned long long)(used[0] + 1 + used[1] + 1);
        } else {
            iters[b * 8 + 7] = used[0]; resid[b * 8 + 7] = fin[0];
            iter_total[b * 2 + 1] += (unsigned long long)(used[0] + 1);
        }
    }
    cluster_sync_all();
}

template <int CS, int CPT, int NC>
static int launch_bicgstab_cluster(fgb_batch *b, const float *coff, const float *adiag, const float *rhs, float *x, int zero_init,
                                   const int32_t *active, int transposed, cudaStream_t st) {
    constexpr int T = 512;
    const int N = b->t.N;
    const int per = (N + CS - 1) / CS;
    if (per > T * CPT) return 1;
    const size_t smem = ((size_t)4 * NC * T * CPT + (size_t)2 * (T / 32) * CS * 4) * sizeof(float) + 3 * 8 + 16;
    if (smem > 227 * 1024) return 1;
    auto kern = k_bicgstab_cluster<T, CPT, CS, NC>;
    cudaError_t ce = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "cudaFuncSetAttribute(k_bicgstab_cluster)", ce);
    if (CS > 8) {   // 16-CTA clusters are a non-portable size: opt in (one cluster then occupies most of a GPC)
        ce = cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
        if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "cudaFuncSetAttribute(k_bicgstab_cluster, non-portable cluster)", ce);
    }
    cudaLaunchConfig_t cfg; memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(b->B * CS); cfg.blockDim = dim3(T); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CS; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    ce = cudaLaunchKernelEx(&cfg, kern, b->t, coff, adiag, rhs, x, b->opt.max_iter, b->opt.adv_tol,
                            zero_init, active, b->iters, b->resid, b->iter_total, transposed);
    if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "cudaLaunchKernelEx(k_bicgstab_cluster)", ce);
    return FGB_OK;
}
// smallest cluster that holds the grid on chip: 2 x 3072, 4 x 3584, 8 x 3584 or 16 x 3072 cells (returns 1 if none does)
template <int NC>
static int bicgstab_cluster_any(fgb_batch *b, const float *coff, const float *adiag, const float *rhs, float *x, int zero_init,
                                const int32_t *active, int transposed, cudaStream_t st) {
    int rc = launch_bicgstab_cluster<2, 6, NC>(b, coff, adiag, rhs, x, zero_init, active, transposed, st);
    if (rc == 1) rc = launch_bicgstab_cluster<4, 7, NC>(b, coff, adiag, rhs, x, zero_init, active, transposed, st);
    if (rc == 1) rc = launch_bicgstab_cluster<8, 7, NC>(b, coff, adiag, rhs, x, zero_init, active, transposed, st);
    if (rc == 1) rc = launch_bicgstab_cluster<16, 6, NC>(b, coff, adiag, rhs, x, zero_init, active, transposed, st);
    return rc;
}
// BiCGStab dispatcher: on-chip cluster kernel when the grid fits, else one CTA per environment in global memory
template <int NC>
static int run_bicgstab(fgb_batch *b, const float *rhs, float *x, int zero_init, const int32_t *active, cudaStream_t st) {
    if (b->opt.cg_impl >= 1) {
        int rc = bicgstab_cluster_any<NC>(b, b->Coff, b->A, rhs, x, zero_init, active, 0, st);
        if (rc <= 0) return rc;
    }
    k_bicgstab<1024, NC><<<b->B, 1024, 0, st>>>(b->t, b->Coff, b->A, rhs, x, b->kry, b->opt.max_iter, b->opt.adv_tol, zero_init, active,
                                                 b->iters, b->resid, b->iter_total);
    LAUNCH_CHECK("k_bicgstab");
    return FGB_OK;
}

// ------------------------------------------------------------------------------------------------
// Krylov solvers, implementation 4: "fat CTA" variant of implementation 3.  Twice the cells per CTA
// (cluster of 2 for the 14k-cell cylinder grid -> every SM of the chip is usable, 74 environments in
// flight) so that the cross-CTA latency of the two reductions and of the p hand-shake is amortised over
// twice the work.  To fit, only the stencil coefficients, A*p and p of the owned cells stay in
// registers; x, r, the best iterate, p and the neighbour table (16 bit: 3 bits CTA rank, 13 bits slot)
// live in shared memory (172 KB per CTA).  Same textbook recurrence, same mbarrier protocol.
// ------------------------------------------------------------------------------------------------
template <int T, int CPT, int CS, int MINB>
__global__ void __launch_bounds__(T, MINB) k_cg_smem(Tab t, const float *__restrict__ Poff, const float *__restrict__ Pdiag,
                                                   const float *__restrict__ Rhs, float *__restrict__ Xout,
                                                   int maxit, float tol, int zero_init, int reset_steps, int slot,
                                                   const int32_t *__restrict__ active, int32_t *__restrict__ iters,
                                                   float *__restrict__ resid, unsigned long long *__restrict__ iter_total) {
    constexpr int NW = T / 32;
    constexpr int NP = NW * CS;
    constexpr int PAD = T * CPT;
    static_assert(PAD <= 8192, "13-bit slot index");
    const int b = blockIdx.x / CS;
    uint32_t rank;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
    if (active && !active[b]) return;
    extern __shared__ __align__(16) float smem[];
    const int N = t.N;
    const int per = (N + CS - 1) / CS;
    const int start = (int)rank * per;
    const int cnt = max(0, min(per, N - start));
    float *ps = smem;                            // [PAD] search direction
    float *xs = smem + PAD;                      // [PAD] iterate
    float *rs = smem + 2 * PAD;                  // [PAD] residual
    float *bs = smem + 3 * PAD;                  // [PAD] best iterate
    uint2 *nbs = (uint2 *)(smem + 4 * PAD);      // [PAD] 4 x 16-bit neighbour codes
    float *red = smem + 6 * PAD;                 // [2][NP]
    unsigned long long *mb = (unsigned long long *)(smem + 6 * PAD + 2 * NP);
    const float *off = Poff + (size_t)b * 4 * N, *dg = Pdiag + (size_t)b * N, *f = Rhs + (size_t)b * N;
    float *xo = Xout + (size_t)b * N;
    const float norm = 1.0f / sqrtf((float)N);
    const uint32_t ps_addr = smem_u32(ps), red_addr = smem_u32(red), mb_addr = smem_u32(mb);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

    if (threadIdx.x == 0) {
        mbar_init(mb_addr, 1); mbar_init(mb_addr + 8, 1); mbar_init(mb_addr + 16, CS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        mbar_arrive_expect_tx(mb_addr, NP * 4);
        mbar_arrive_expect_tx(mb_addr + 8, NP * 4);
    }
    float cd[CPT], co[CPT][4];
#pragma unroll
    for (int k = 0; k < CPT; ++k) {
        const int l = threadIdx.x + k * T;
        const int g = start + l;
        const bool ok = l < cnt;
        cd[k] = ok ? dg[g] : 0.f;
        xs[l] = (ok && !zero_init) ? xo[g] : 0.f;
        ps[l] = 0.f; bs[l] = 0.f; rs[l] = 0.f;
        uint32_t code[4];
#pragma unroll
        for (int ff = 0; ff < 4; ++ff) {
            const int nb = ok ? t.nbr[ff * N + g] : -1;
            co[k][ff] = (ok && nb >= 0) ? off[ff * N + g] : 0.f;
            const int gi = nb >= 0 ? nb : (ok ? g : start);
            const int c = gi / per;
            code[ff] = ((uint32_t)c << 13) | (uint32_t)(gi - c * per);
        }
        nbs[l] = make_uint2(code[0] | (code[1] << 16), code[2] | (code[3] << 16));
    }
    const uint32_t peer_red = mapa_u32(red_addr, (uint32_t)(lane < CS ? lane : 0));
    const uint32_t peer_mb = mapa_u32(mb_addr, (uint32_t)(lane < CS ? lane : 0));
    cluster_sync_all();

    uint32_t rcount = 0, pphase = 0;
    auto cluster_sum = [&](float a0) -> float {
        const uint32_t w = rcount & 1u, par = (rcount >> 1) & 1u;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) a0 += __shfl_xor_sync(0xffffffffu, a0, o);
        if (lane < CS) st_async_f32(peer_red + 4u * (w * NP + rank * NW + (uint32_t)warp), a0, peer_mb + 8u * w);
        mbar_wait(mb_addr + 8u * w, par);
        const float *rp = red + w * NP;
        float s0 = 0.f;
#pragma unroll
        for (int q = 0; q < (NP + 31) / 32; ++q) s0 += (lane + 32 * q < NP) ? rp[lane + 32 * q] : 0.f;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s0 += __shfl_xor_sync(0xffffffffu, s0, o);
        if (threadIdx.x == 0) mbar_arrive_expect_tx(mb_addr + 8u * w, NP * 4);
        ++rcount;
        return s0;
    };
    auto publish = [&]() {
        __syncthreads();
        if (threadIdx.x < CS) mbar_arrive_remote_release(mapa_u32(mb_addr + 16, threadIdx.x));
    };
    auto acquire_p = [&]() { mbar_wait(mb_addr + 16, pphase); pphase ^= 1u; };
    auto gather = [&](uint32_t code) -> float {
        return ld_dsmem_f32(mapa_u32(ps_addr + ((code & 0x1fffu) << 2), (code >> 13) & 7u));
    };
    auto apply = [&](int k, float &own) -> float {   // row k of P times the vector exposed in ps
        const int l = threadIdx.x + k * T;
        const uint2 nb = nbs[l];
        own = ps[l];
        float s = cd[k] * own;
        s += co[k][0] * gather(nb.x & 0xffffu);
        s += co[k][1] * gather(nb.x >> 16);
        s += co[k][2] * gather(nb.y & 0xffffu);
        s += co[k][3] * gather(nb.y >> 16);
        return s;
    };
    auto load_f = [&](int k) -> float { const int l = threadIdx.x + k * T; return l < cnt ? f[start + l] : 0.f; };

    float nz = 0.f;
#pragma unroll
    for (int k = 0; k < CPT; ++k) nz += (load_f(k) != 0.f) ? 1.f : 0.f;
    const float nzt = cluster_sum(nz);
    int used = -1; float fin = 0.f;
    bool result_in_best = false;
    if (!(nzt > 0.f)) {
#pragma unroll
        for (int k = 0; k < CPT; ++k) xs[threadIdx.x + k * T] = 0.f;
    } else {
        float a0 = 0.f, own;
        if (!zero_init) {
#pragma unroll
            for (int k = 0; k < CPT; ++k) ps[threadIdx.x + k * T] = xs[threadIdx.x + k * T];
            publish(); acquire_p();
            float tmp[CPT];
#pragma unroll
            for (int k = 0; k < CPT; ++k) tmp[k] = load_f(k) - apply(k, own);
            (void)cluster_sum(0.f);
#pragma unroll
            for (int k = 0; k < CPT; ++k) { const int l = threadIdx.x + k * T; rs[l] = tmp[k]; ps[l] = tmp[k]; a0 += tmp[k] * tmp[k]; }
        } else {
#pragma unroll
            for (int k = 0; k < CPT; ++k) { const int l = threadIdx.x + k * T; const float r0 = load_f(k); rs[l] = r0; ps[l] = r0; a0 += r0 * r0; }
        }
        publish();
        float rho = cluster_sum(a0);
        float bestc = 0.f, lastc = 0.f; int best_it = -1, rising = 0;
        bool copy_best = false;                  // x of the previous iteration still has to be saved into bs
        float pk[CPT], apk[CPT];
        for (int i = 0; i < maxit; ++i) {
            if (reset_steps > 0 && (i + 1) % reset_steps == 0) {
                acquire_p();
                (void)cluster_sum(0.f);
                if (copy_best) {
#pragma unroll
                    for (int k = 0; k < CPT; ++k) bs[threadIdx.x + k * T] = xs[threadIdx.x + k * T];
                    copy_best = false;
                }
#pragma unroll
                for (int k = 0; k < CPT; ++k) ps[threadIdx.x + k * T] = xs[threadIdx.x + k * T];
                publish(); acquire_p();
                float tmp[CPT];
#pragma unroll
                for (int k = 0; k < CPT; ++k) tmp[k] = load_f(k) - apply(k, own);
                (void)cluster_sum(0.f);
                a0 = 0.f;
#pragma unroll
                for (int k = 0; k < CPT; ++k) { const int l = threadIdx.x + k * T; rs[l] = tmp[k]; ps[l] = tmp[k]; a0 += tmp[k] * tmp[k]; }
                publish();
                rho = cluster_sum(a0);
            }
            acquire_p();
            a0 = 0.f;
#pragma unroll
            for (int k = 0; k < CPT; ++k) {
                apk[k] = apply(k, pk[k]);
                a0 += pk[k] * apk[k];
            }
            const float pap = cluster_sum(a0);
            const float alpha = rho / pap;
            a0 = 0.f;
#pragma unroll
            for (int k = 0; k < CPT; ++k) {
                const int l = threadIdx.x + k * T;
                const float xo_ = xs[l];
                if (copy_best) bs[l] = xo_;      // deferred copy of the previous (best so far) iterate
                xs[l] = xo_ + alpha * pk[k];
                const float rn = rs[l] - alpha * apk[k];
                rs[l] = rn;
                a0 += rn * rn;
            }
            copy_best = false;
            const float rr2 = cluster_sum(a0);
            const float crit = sqrtf(rr2) * norm;
            if (!isfinite(crit)) { used = i; fin = crit; break; }
            if (i == 0 || crit < bestc) { bestc = crit; best_it = i; copy_best = true; }
            if (i > 0 && crit >= lastc) ++rising; else rising = 0;
            lastc = crit; used = i; fin = crit;
            if (crit < tol) break;
            if (i == maxit - 1 || rising >= 100) {
                // the best iterate is the current x if it was flagged this very iteration, else what bs holds
                result_in_best = !copy_best;
                used = best_it; fin = bestc;
                break;
            }
            const float beta = rr2 / rho;
            rho = rr2;
#pragma unroll
            for (int k = 0; k < CPT; ++k) { const int l = threadIdx.x + k * T; ps[l] = rs[l] + beta * pk[k]; }
            publish();
        }
    }
    const float *res = result_in_best ? bs : xs;
    float sx = 0.f;
#pragma unroll
    for (int k = 0; k < CPT; ++k) sx += res[threadIdx.x + k * T];
    const float mean = cluster_sum(sx) / (float)N;
#pragma unroll
    for (int k = 0; k < CPT; ++k) { const int l = threadIdx.x + k * T; if (l < cnt) xo[start + l] = res[l] - mean; }
    if (threadIdx.x == 0 && rank == 0) { iters[b * 8 + 2 + slot] = used; resid[b * 8 + 2 + slot] = fin; iter_total[b * 2] += (unsigned long long)(used + 1); }
    cluster_sync_all();
}

// ------------------------------------------------------------------------------------------------
// boundary / stepping kernels: one CTA per environment
// ------------------------------------------------------------------------------------------------
// Domain.getMaxVelocity(True, True) (DS.cpp:1360-1367, 1580-1611): max |M^-1 u| over cells and fixed faces
template <int T>
__device__ float env_max_velocity(const Tab &t, const float *u, const float *bv, float *sm) {
    const int N = t.N, NB = t.NB;
    float m = 0.f;
    for (int g = threadIdx.x; g < N; g += T) {
        const float a = u[g], c = u[N + g];
        m = fmaxf(m, fabsf(t.minv[g] * a + t.minv[N + g] * c));
        m = fmaxf(m, fabsf(t.minv[2 * N + g] * a + t.minv[3 * N + g] * c));
    }
    for (int j = threadIdx.x; j < NB; j += T) {
        const float a = bv[j], c = bv[NB + j];
        m = fmaxf(m, fabsf(t.b_minv[j] * a + t.b_minv[NB + j] * c));
        m = fmaxf(m, fabsf(t.b_minv[2 * NB + j] * a + t.b_minv[3 * NB + j] * c));
    }
    return block_reduce_max(m, sm);
}
template <int T>
__global__ void __launch_bounds__(T) k_max_velocity(Tab t, const float *__restrict__ U, const float *__restrict__ Bvel, float *__restrict__ out) {
    __shared__ float sm[33];
    const int b = blockIdx.x;
    const float m = env_max_velocity<T>(t, U + (size_t)b * 2 * t.N, Bvel + (size_t)b * 2 * t.NB, sm);
    if (threadIdx.x == 0) out[b] = m;
}

// signed boundary flux sums; which: 0 = faces with b_out==0, 1 = faces with b_out==1, 2 = all
template <int T>
__device__ void env_flux_sums(const Tab &t, const float *bv, float &fixed, float &var, double *red, const int8_t *mask = nullptr) {
    if (!mask) mask = t.b_out;
    const int NB = t.NB;
    float acc[2] = {0.f, 0.f};
    for (int j = threadIdx.x; j < NB; j += T) {
        const int f = t.b_face[j];
        float fl = bflux(t, j, f >> 1, bv[j], bv[NB + j]);
        if (!(f & 1)) fl = -fl;
        if (mask && mask[j]) acc[1] += fl; else acc[0] += fl;
    }
    block_reduce_sum<2>(acc, red);
    fixed = acc[0]; var = acc[1];
}
template <int T>
__global__ void __launch_bounds__(T) k_flux_balance(Tab t, const float *__restrict__ Bvel, float *__restrict__ out) {
    __shared__ double red[32 * 2 + 2];
    const int b = blockIdx.x;
    float fx, vr;
    env_flux_sums<T>(t, Bvel + (size_t)b * 2 * t.NB, fx, vr, red);
    if (threadIdx.x == 0) out[b] = fx + vr;
}

// advective outflow boundary relaxation and global flux rescale (SIM.py:188-224, 282-393)
template <int T>
__device__ void env_update_outflow(const Tab &t, const float *u, float *bv, float dt, float cvx, float cvy, float bc_tol, double *red) {
    const int N = t.N, NB = t.NB;
    for (int j = threadIdx.x; j < NB; j += T) {
        if (t.b_out[j]) {
            const int ax = t.b_face[j] >> 1;
            const float adv = t.b_minv[(2 * ax) * NB + j] * cvx + t.b_minv[(2 * ax + 1) * NB + j] * cvy;
            const float al = dt * 2.f * adv;
            const float w = 1.f - 1.f / (1.f + al);
            const int c = t.b_cell[j];
            const float b0 = bv[j], b1 = bv[NB + j];
            bv[j] = b0 - w * (b0 - u[c]);
            bv[NB + j] = b1 - w * (b1 - u[N + c]);
        }
    }
    __syncthreads();
    float fx, vr;
    env_flux_sums<T>(t, bv, fx, vr, red);
    if (!(fabsf(fx + vr) <= bc_tol * 0.01f)) {
        const float sc = -fx / vr;
        for (int j = threadIdx.x; j < NB; j += T)
            if (t.b_out[j]) { bv[j] *= sc; bv[NB + j] *= sc; }
    }
    __syncthreads();
}

// Adaptive sub-stepping plan (SIM.py:2004-2031) + advective outflow boundary update and global flux
// balancing (SIM.py:188-224, 228-393), fused: one CTA per environment.
template <int T>
__global__ void __launch_bounds__(T) k_plan_substep(Tab t, const float *__restrict__ U, float *__restrict__ Bvel,
                                                     double *__restrict__ remaining, float *__restrict__ dtv,
                                                     int32_t *__restrict__ active, int32_t *__restrict__ nsub,
                                                     float *__restrict__ maxvel, int32_t *__restrict__ counters,
                                                     float cfl, float cvx, float cvy, float bc_tol, int do_outflow) {
    __shared__ float smf[33];
    __shared__ double red[32 * 2 + 2];
    __shared__ float s_dt; __shared__ int s_active;
    const int b = blockIdx.x;
    const int N = t.N, NB = t.NB;
    const float *u = U + (size_t)b * 2 * N;
    float *bv = Bvel + (size_t)b * 2 * NB;
    const float mv = env_max_velocity<T>(t, u, bv, smf);
    if (threadIdx.x == 0) {
        double rem = remaining[b];
        int act = (rem > 0.0) && !(fabs(rem) <= 1e-8);
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
        dtv[b] = dt; active[b] = act; maxvel[b] = mv;
        s_dt = dt; s_active = act;
    }
    __syncthreads();
    if (!s_active || !do_outflow || !t.b_out) return;
    env_update_outflow<T>(t, u, bv, s_dt, cvx, cvy, bc_tol, red);
}
template <int T>
__global__ void __launch_bounds__(T) k_update_outflow(Tab t, const float *__restrict__ U, float *__restrict__ Bvel,
                                                       const float *__restrict__ dtv, float cvx, float cvy, float bc_tol) {
    __shared__ double red[32 * 2 + 2];
    const int b = blockIdx.x;
    env_update_outflow<T>(t, U + (size_t)b * 2 * t.N, Bvel + (size_t)b * 2 * t.NB, dtv[b], cvx, cvy, bc_tol, red);
}
// balance_boundary_fluxes (SIM.py:188-224) with an explicit set of free faces: all their velocities are scaled by
// -(flux through the other prescribed faces) / (flux through the free faces)
template <int T>
__global__ void __launch_bounds__(T) k_balance_fluxes(Tab t, float *__restrict__ Bvel, const int8_t *__restrict__ free_mask, float bc_tol) {
    __shared__ double red[32 * 2 + 2];
    const int b = blockIdx.x, NB = t.NB;
    float *bv = Bvel + (size_t)b * 2 * NB;
    float fx, vr;
    env_flux_sums<T>(t, bv, fx, vr, red, free_mask);
    if (!(fabsf(fx + vr) <= bc_tol * 0.01f)) {
        const float sc = -fx / vr;
        for (int j = threadIdx.x; j < NB; j += T)
            if (free_mask[j]) { bv[j] *= sc; bv[NB + j] *= sc; }
    }
}
__global__ void k_set_remaining(double *remaining, int32_t *nsub, int32_t *counters, double v, int B) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < B) { remaining[i] = v; nsub[i] = 0; }
    if (i == 0) counters[0] = 0;
}
__global__ void k_zero_counter(int32_t *counters) { counters[0] = 0; }

// jet actuation
__global__ void k_apply_jet(float *__restrict__ Bvel, float *__restrict__ last, const float *__restrict__ action, float smoothing,
                            const int32_t *__restrict__ faces, const float *__restrict__ templ, int nf, int NB, int B) {
    const int b = blockIdx.x;
    const float l = last[b];
    const float c = l + smoothing * (action[b] - l);
    for (int k = threadIdx.x; k < nf; k += blockDim.x) {
        const int j = faces[k];
        Bvel[(size_t)b * 2 * NB + j] = templ[k] * c;
        Bvel[(size_t)b * 2 * NB + NB + j] = templ[nf + k] * c;
    }
    __syncthreads();
    if (threadIdx.x == 0) last[b] = c;
}

// wall forces (forces.py:193-275)
__global__ void __launch_bounds__(128) k_wall_forces(fgb_wall w, float visc, int N, int NB, const float *__restrict__ U,
                                                      const float *__restrict__ P, const float *__restrict__ Bvel, float *__restrict__ acc) {
    __shared__ double red[32 * 2 + 2];
    const int b = blockIdx.x;
    const float *u = U + (size_t)b * 2 * N, *p = P + (size_t)b * N, *bv = Bvel + (size_t)b * 2 * NB;
    const int n = w.n_wall;
    float f[2] = {0.f, 0.f};
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int c = w.cell[i], j = w.bface[i];
        const int il = w.cell[(i + 1) % n], ir = w.cell[(i + n - 1) % n];   // roll(-1) / roll(+1)
        const float nx = w.normal[i], ny = w.normal[n + i];
        const float tx = ny, ty = -nx;
        const float du_dn = (u[c] - bv[j]) / w.dist[i], dv_dn = (u[N + c] - bv[NB + j]) / w.dist[i];
        const float du_dt = (u[ir] - u[il]) / (2.f * w.tlen[i]), dv_dt = (u[N + ir] - u[N + il]) / (2.f * w.tlen[i]);
        const float du_dx = du_dn * nx + du_dt * tx, du_dy = du_dn * ny + du_dt * ty;
        const float dv_dx = dv_dn * nx + dv_dt * tx, dv_dy = dv_dn * ny + dv_dt * ty;
        const float sxx = 2.f * visc * du_dx - p[c], syy = 2.f * visc * dv_dy - p[c];
        const float sxy = 2.f * visc * (0.5f * (du_dy + dv_dx));
        f[0] += (sxx * nx + sxy * ny) * w.flen[i];
        f[1] += (sxy * nx + syy * ny) * w.flen[i];
    }
    block_reduce_sum<2>(f, red);
    if (threadIdx.x == 0) { acc[b * 2] += f[0] * w.scale; acc[b * 2 + 1] += f[1] * w.scale; }
}

// sensors: out[b][c][s] = sum_k w[k][s] * field[b][c][idx[k][s]]
__global__ void k_sample_sensors(const float *__restrict__ field, int C, int N, const int32_t *__restrict__ idx,
                                 const float *__restrict__ w, int K, int ns, float *__restrict__ out) {
    const int b = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= C * ns) return;
    const int c = i / ns, s = i - c * ns;
    const float *fl = field + ((size_t)b * C + c) * N;
    float v = 0.f;
    for (int k = 0; k < K; ++k) { const float ww = w[k * ns + s]; if (ww != 0.f) v += ww * fl[idx[k * ns + s]]; }
    out[((size_t)b * C + c) * ns + s] = v;
}

// rendering (fluidgym_b200/render.py): the full static render map as CSR, rows in image order.  One thread per (pixel,
// environment), the environment in blockIdx.y so that the tables are read by the whole batch from L2.
#define RENDER_THREADS 256
// order-preserving float -> uint32 key (a < b <=> key(a) < key(b)); the range slots hold min key(v) and min ~key(v) so that a
// single 0xff memset initialises both and both are atomicMin
__device__ __forceinline__ unsigned int render_key(float v) {
    const unsigned int u = __float_as_uint(v);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float render_unkey(unsigned int k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

__global__ void __launch_bounds__(RENDER_THREADS) k_render_gather(const float *__restrict__ field, int C, long long chan_stride,
                                                                  long long env_stride, int mode, const int32_t *__restrict__ rowptr,
                                                                  const int32_t *__restrict__ col, const float *__restrict__ w, int P,
                                                                  float *__restrict__ img, unsigned int *__restrict__ range) {
    const int b = blockIdx.y;
    const int p = blockIdx.x * RENDER_THREADS + threadIdx.x;
    float v = 0.f;
    if (p < P) {
        const float *f = field + (size_t)b * env_stride;
        float a[3] = {0.f, 0.f, 0.f};
        const int k1 = rowptr[p + 1];
        for (int k = rowptr[p]; k < k1; ++k) {
            const long long c0 = col[k];
            const float ww = w[k];
#pragma unroll
            for (int c = 0; c < 3; ++c)
                if (c < C) a[c] += ww * f[c * chan_stride + c0];
        }
        v = (mode == FGB_RENDER_NORM) ? sqrtf(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]) : a[0];
        img[(size_t)b * P + p] = v;
    }
    if (!range) return;                                          // uniform over the grid
    unsigned int lo = 0xffffffffu, hi = 0xffffffffu;
    if (p < P) { lo = render_key(v); hi = ~lo; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = min(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    __shared__ unsigned int red[2][RENDER_THREADS / 32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { red[0][warp] = lo; red[1][warp] = hi; }
    __syncthreads();
    if (warp == 0) {
        lo = lane < RENDER_THREADS / 32 ? red[0][lane] : 0xffffffffu;
        hi = lane < RENDER_THREADS / 32 ? red[1][lane] : 0xffffffffu;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
            hi = min(hi, __shfl_xor_sync(0xffffffffu, hi, o));
        }
        if (lane == 0) { atomicMin(&range[2 * b], lo); atomicMin(&range[2 * b + 1], hi); }
    }
}

// LUT bin of v in [lo, hi]: floor(256 (v - lo) / (hi - lo)) clamped to [0, 255] (NaN -> 0), 128 for an empty range
__device__ __forceinline__ int render_bin(float v, float lo, float hi) {
    const float t = hi > lo ? (v - lo) / (hi - lo) : 0.5f;
    return (int)fminf(fmaxf(t * 256.f, 0.f), 255.f);
}

// rgb[B*P][3] uint8 from img[B*P] through a 256-entry LUT in shared memory; one thread per 4 consecutive pixels of the flattened
// batch, whose 12 bytes go out as 3 aligned uint32 stores
__global__ void __launch_bounds__(RENDER_THREADS) k_render_colour(const float *__restrict__ img, int P, long long total,
                                                                  const unsigned int *__restrict__ range, float vmin, float vmax,
                                                                  int symmetric, const uint8_t *__restrict__ lut,
                                                                  uint8_t *__restrict__ rgb) {
    __shared__ unsigned int s_lut[256];
    for (int i = threadIdx.x; i < 256; i += RENDER_THREADS)
        s_lut[i] = (unsigned int)lut[3 * i] | ((unsigned int)lut[3 * i + 1] << 8) | ((unsigned int)lut[3 * i + 2] << 16);
    __syncthreads();
    const long long i0 = 4 * ((long long)blockIdx.x * RENDER_THREADS + threadIdx.x);
    if (i0 >= total) return;
    const bool full = i0 + 4 <= total;
    float v[4];
    if (full) {
        const float4 q = *reinterpret_cast<const float4 *>(img + i0);
        v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
    } else {
        for (int j = 0; j < 4; ++j) v[j] = i0 + j < total ? img[i0 + j] : 0.f;
    }
    unsigned int c[4];
    int bprev = -1;
    float lo = vmin, hi = vmax;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        c[j] = 0u;
        if (i0 + j >= total) continue;
        const int b = (int)((i0 + j) / P);
        if (b != bprev) {
            bprev = b;
            if (range) { lo = render_unkey(range[2 * b]); hi = render_unkey(~range[2 * b + 1]); }
            else { lo = vmin; hi = vmax; }
            if (symmetric) { hi = fmaxf(fabsf(lo), fabsf(hi)); lo = -hi; }
        }
        c[j] = s_lut[render_bin(v[j], lo, hi)];
    }
    if (full) {
        unsigned int *o = reinterpret_cast<unsigned int *>(rgb + 3 * i0);
        o[0] = c[0] | (c[1] << 24);
        o[1] = (c[1] >> 8) | (c[2] << 16);
        o[2] = (c[2] >> 16) | (c[3] << 8);
    } else {
        for (int j = 0; i0 + j < total; ++j)
            for (int k = 0; k < 3; ++k) rgb[3 * (i0 + j) + k] = (uint8_t)(c[j] >> (8 * k));
    }
}

// ------------------------------------------------------------------------------------------------
// Reverse-mode adjoint of one PISO substep (replaces the *_GRAD kernels K.cu:3884-4090, 4403-4491,
// 4982-5130, 5258-5385, 5438-5509, 6265-6309 and the python glue DIFF.py:516-1808).  Specification:
// oracle/adjoint_eval.py (float64 numpy, validated against finite differences).  Every forward gather
// y_i += w * x[j] becomes the scatter xbar[j] += w * ybar_i with red.global.add.f32; the two linear solves
// become solves with the transposed operator by the same on-chip Krylov kernels.
// All kernels: one thread per (cell, environment).
// ------------------------------------------------------------------------------------------------
// scatter of a flux-divergence adjoint: flb[f] = adjoint of face flux f of this cell
__device__ __forceinline__ void fluxes_adjoint(const Tab &t, int g, const int nb[4], const float flb[4], float *__restrict__ vb /*[2][N]*/,
                                               float *__restrict__ Fbb /*[NB]*/) {
    const int N = t.N;
    float Ub[2] = {0.f, 0.f};
#pragma unroll
    for (int f = 0; f < 4; ++f) {
        if (nb[f] >= 0) {
            const float gq = 0.5f * flb[f];
            Ub[f >> 1] += gq;
            const int fc = t.fl_comp[f * N + g];
            const int cn = fc & 1, n = nb[f];
            const float w = ((fc & 2) ? -gq : gq) * t.det[n];
            atomicAdd(&vb[n], w * t.minv[(2 * cn) * N + n]);
            atomicAdd(&vb[N + n], w * t.minv[(2 * cn + 1) * N + n]);
        } else if (Fbb) {
            atomicAdd(&Fbb[-1 - nb[f]], flb[f]);
        }
    }
    const float d = t.det[g];
    atomicAdd(&vb[g], d * (t.minv[g] * Ub[0] + t.minv[2 * N + g] * Ub[1]));
    atomicAdd(&vb[N + g], d * (t.minv[N + g] * Ub[0] + t.minv[3 * N + g] * Ub[1]));
}

// adjoint of the corrector u_next = hb - rA * Minv^T grad(p):  hbb += unb ; rAb += -(g . unb) ; pb += grad^T(...)
__global__ void __launch_bounds__(256) k_adj_correct(Tab t, const float *__restrict__ Unb, const float *__restrict__ P, const float *__restrict__ A,
                                                      float *__restrict__ Hbb, float *__restrict__ rAb, float *__restrict__ Pb,
                                                      const int32_t *__restrict__ active) {
    const int b = blockIdx.y;
    if (active && !active[b]) return;   // skipped environment: identity cotangents from k_adj_inactive
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    const int N = t.N;
    if (g >= N) return;
    const float *p = P + (size_t)b * N;
    const float ub0 = Unb[(size_t)b * 2 * N + g], ub1 = Unb[(size_t)b * 2 * N + N + g];
    Hbb[(size_t)b * 2 * N + g] = ub0; Hbb[(size_t)b * 2 * N + N + g] = ub1;
    const float rA = 1.0f / A[(size_t)b * N + g];
    const float pc = p[g];
    float pg[2]; int nl[2], nu[2]; float fac[2];
#pragma unroll
    for (int d = 0; d < 2; ++d) {
        nl[d] = t.nbr[(2 * d) * N + g]; nu[d] = t.nbr[(2 * d + 1) * N + g];
        fac[d] = (nl[d] < 0 || nu[d] < 0) ? 1.0f : 0.5f;
        pg[d] = ((nu[d] >= 0 ? p[nu[d]] : pc) - (nl[d] >= 0 ? p[nl[d]] : pc)) * fac[d];
    }
    const float m00 = t.minv[g], m01 = t.minv[N + g], m10 = t.minv[2 * N + g], m11 = t.minv[3 * N + g];
    const float gx = pg[0] * m00 + pg[1] * m10, gy = pg[0] * m01 + pg[1] * m11;
    atomicAdd(&rAb[(size_t)b * N + g], -(gx * ub0 + gy * ub1));
    const float gb0 = -rA * ub0, gb1 = -rA * ub1;
    const float pgb[2] = {gb0 * m00 + gb1 * m01, gb0 * m10 + gb1 * m11};
    float *pb = Pb + (size_t)b * N;
#pragma unroll
    for (int d = 0; d < 2; ++d) {
        const float w = pgb[d] * fac[d];
        atomicAdd(&pb[nu[d] >= 0 ? nu[d] : g], w);
        atomicAdd(&pb[nl[d] >= 0 ? nl[d] : g], -w);
    }
}

// x_bar = p_bar - mean(p_bar)   (adjoint of the mean removal), one CTA per environment
template <int T>
__global__ void __launch_bounds__(T) k_adj_remove_mean(int N, const float *__restrict__ Pb, float *__restrict__ Xb,
                                                        const int32_t *__restrict__ active) {
    __shared__ double red[32 * 2 + 2];
    const int b = blockIdx.x;
    if (active && !active[b]) return;   // skipped environment: identity cotangents from k_adj_inactive
    float acc[2] = {0.f, 0.f};
    for (int g = threadIdx.x; g < N; g += T) acc[0] += Pb[(size_t)b * N + g];
    block_reduce_sum<2>(acc, red);
    const float m = acc[0] / (float)N;
    for (int g = threadIdx.x; g < N; g += T) Xb[(size_t)b * N + g] = Pb[(size_t)b * N + g] - m;
}

// adjoint of  div = fluxdiv(hb) + NOp(p_prev, rA)  and of  x = P^-1 div  w.r.t. P:   given lam = P^-T x_bar
__global__ void __launch_bounds__(256) k_adj_pressure_rhs(Tab t, const float *__restrict__ Lam, const float *__restrict__ Pm /*p of this corrector*/,
                                                           const float *__restrict__ Pmean, const float *__restrict__ Pprev,
                                                           const float *__restrict__ A, float *__restrict__ Hbb, float *__restrict__ Fbb,
                                                           float *__restrict__ rAb, float *__restrict__ Pprevb, const int32_t *__restrict__ active) {
    const int b = blockIdx.y;
    if (active && !active[b]) return;   // skipped environment: identity cotangents from k_adj_inactive
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    const int N = t.N, NB = t.NB;
    if (g >= N) return;
    const float lam = Lam[(size_t)b * N + g];
    const float *px = Pm + (size_t)b * N;
    const float mean = Pmean[b];
    int nb[4];
#pragma unroll
    for (int f = 0; f < 4; ++f) nb[f] = t.nbr[f * N + g];
    // P_bar_e = -lam_i * x_j on the pattern (x = p + mean); rA_bar_j += Wp[e][j] * P_bar_e
    float Pb[5];
    Pb[0] = -lam * (px[g] + mean);
#pragma unroll
    for (int f = 0; f < 4; ++f) Pb[f + 1] = nb[f] >= 0 ? -lam * (px[nb[f]] + mean) : 0.f;
    float rb[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int e = 0; e < 5; ++e)
#pragma unroll
        for (int j = 0; j < 5; ++j) rb[j] += t.Wp[(5 * e + j) * N + g] * Pb[e];
    // deferred non-orthogonal pressure term: div += sum_k (gP rA_P + gN rA_nbr(face)) * pprev[idx]
    const float *a = A + (size_t)b * N, *pp = Pprev + (size_t)b * N;
    float rA[5];
    rA[0] = 1.0f / a[g];
#pragma unroll
    for (int f = 0; f < 4; ++f) rA[f + 1] = nb[f] >= 0 ? 1.0f / a[nb[f]] : rA[0];
    for (int k = 0; k < t.K_no; ++k) {
        const float gP = t.no_gP[k * N + g], gN = t.no_gN[k * N + g];
        if (gP != 0.f || gN != 0.f) {
            const int fc = t.no_face[k * N + g], j = t.no_idx[k * N + g];
            const float wb = lam * pp[j];
            rb[0] += gP * wb; rb[1 + fc] += gN * wb;
            atomicAdd(&Pprevb[(size_t)b * N + j], (gP * rA[0] + gN * rA[1 + fc]) * lam);
        }
    }
    float *ra = rAb + (size_t)b * N;
    atomicAdd(&ra[g], rb[0]);
#pragma unroll
    for (int f = 0; f < 4; ++f) atomicAdd(&ra[nb[f] >= 0 ? nb[f] : g], rb[f + 1]);
    const float flb[4] = {-lam, lam, -lam, lam};
    fluxes_adjoint(t, g, nb, flb, Hbb + (size_t)b * 2 * N, Fbb + (size_t)b * NB);
}

// adjoint of  hb = rA * (u/dt - H + Sb/det),  H_c = sum_f Coff_f * uprev_c[nb_f]
__global__ void __launch_bounds__(256) k_adj_hbya(Tab t, const float *__restrict__ Hbb, const float *__restrict__ Hb /*saved hb*/,
                                                   const float *__restrict__ A, const float *__restrict__ Coff, const float *__restrict__ Uprev,
                                                   const float *__restrict__ dtv, float *__restrict__ rAb, float *__restrict__ Ub,
                                                   float *__restrict__ Sbb, float *__restrict__ Coffb, float *__restrict__ Uprevb,
                                                   const int32_t *__restrict__ active) {
    const int b = blockIdx.y;
    if (active && !active[b]) return;   // skipped environment: identity cotangents from k_adj_inactive
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    const int N = t.N;
    if (g >= N) return;
    const float dt = dtv[b];
    const float Ag = A[(size_t)b * N + g];
    const float rA = 1.0f / Ag;
    const float det = t.det[g];
    float accr = 0.f;
#pragma unroll
    for (int c = 0; c < 2; ++c) {
        const size_t o = (size_t)b * 2 * N + (size_t)c * N;
        const float hbb = Hbb[o + g];
        accr += hbb * (Hb[o + g] * Ag);
        const float ib = rA * hbb;
        Ub[o + g] += ib / dt;
        Sbb[o + g] += ib / det;
#pragma unroll
        for (int f = 0; f < 4; ++f) {
            const int nb = t.nbr[f * N + g];
            if (nb >= 0) {
                Coffb[(size_t)b * 4 * N + f * N + g] += -ib * Uprev[o + nb];
                atomicAdd(&Uprevb[o + nb], -ib * Coff[(size_t)b * 4 * N + f * N + g]);
            }
        }
    }
    atomicAdd(&rAb[(size_t)b * N + g], accr);
}

// adjoint of the predictor: given mu = C^-T ustar_bar
__global__ void __launch_bounds__(256) k_adj_advection(Tab t, const float *__restrict__ Mu, const float *__restrict__ Ustar, const float *__restrict__ rAb,
                                                        const float *__restrict__ A, const float *__restrict__ dtv, float *__restrict__ Ab,
                                                        float *__restrict__ Coffb, float *__restrict__ Ub, float *__restrict__ Sbb, float *__restrict__ Bvb,
                                                        float *__restrict__ NoTarget /* adjoint of the field the deferred term read: u_bar (first
                                                        iteration) or the previous iterate's bar */, int first /* initialise A_bar from rA_bar */,
                                                        const int32_t *__restrict__ active) {
    const int b = blockIdx.y;
    if (active && !active[b]) return;   // skipped environment: identity cotangents from k_adj_inactive
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    const int N = t.N, NB = t.NB;
    if (g >= N) return;
    const float dt = dtv[b];
    const float det = t.det[g];
    const float Ag = A[(size_t)b * N + g];
    float ab = first ? -rAb[(size_t)b * N + g] / (Ag * Ag) : Ab[(size_t)b * N + g];   // A_bar from rA_bar (rA = 1/A)
#pragma unroll
    for (int c = 0; c < 2; ++c) {
        const size_t o = (size_t)b * 2 * N + (size_t)c * N;
        const float mu = Mu[o + g];
        ab += -mu * Ustar[o + g];
#pragma unroll
        for (int f = 0; f < 4; ++f) {
            const int nb = t.nbr[f * N + g];
            if (nb >= 0) Coffb[(size_t)b * 4 * N + f * N + g] += -mu * Ustar[o + nb];
        }
        atomicAdd(&Ub[o + g], mu / dt);  // rhs = (det u/dt + Sb - NOv)/det  (other threads scatter into Ub in this kernel)
        Sbb[o + g] += mu / det;
        const float nob = -mu / det;
        for (int k = 0; k < t.K_no; ++k) { const float w = t.no_wv[k * N + g]; if (w != 0.f) atomicAdd(&NoTarget[o + t.no_idx[k * N + g]], w * nob); }
        for (int k = 0; k < t.K_nob; ++k) {
            const float w = t.nob_w[k * N + g];
            if (w != 0.f) atomicAdd(&Bvb[(size_t)b * 2 * NB + (size_t)c * NB + t.nob_idx[k * N + g]], w * nob);
        }
    }
    Ab[(size_t)b * N + g] = ab;
}

// adjoint of the assembly (A, Coff from the face fluxes) and of the boundary sources
__global__ void __launch_bounds__(256) k_adj_assemble(Tab t, const float *__restrict__ Ab, const float *__restrict__ Coffb, const float *__restrict__ Sbb,
                                                       const float *__restrict__ Bvel, float *__restrict__ Ub, float *__restrict__ Bvb, float *__restrict__ Fbb,
                                                       const int32_t *__restrict__ active) {
    const int b = blockIdx.y;
    if (active && !active[b]) return;   // skipped environment: identity cotangents from k_adj_inactive
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    const int N = t.N, NB = t.NB;
    if (g >= N) return;
    const float det = t.det[g];
    const float diagb = Ab[(size_t)b * N + g] / det;
    const float *bv = Bvel + (size_t)b * 2 * NB;
    int nb[4]; float flb[4];
#pragma unroll
    for (int f = 0; f < 4; ++f) {
        nb[f] = t.nbr[f * N + g];
        const float sig = (f & 1) ? 1.f : -1.f;
        flb[f] = 0.f;
        if (nb[f] >= 0) flb[f] = 0.5f * sig * (Coffb[(size_t)b * 4 * N + f * N + g] / det + diagb);
        else {
            const int j = -1 - nb[f];
            const float Fb = bflux(t, j, f >> 1, bv[j], bv[NB + j]);
            const float s0 = Sbb[(size_t)b * 2 * N + g], s1 = Sbb[(size_t)b * 2 * N + N + g];
            const float k = -(sig * Fb) + 2.f * t.viscosity * t.b_alpha[j];
            atomicAdd(&Bvb[(size_t)b * 2 * NB + j], s0 * k);
            atomicAdd(&Bvb[(size_t)b * 2 * NB + NB + j], s1 * k);
            atomicAdd(&Fbb[(size_t)b * NB + j], -(s0 * bv[j] + s1 * bv[NB + j]) * sig);
        }
    }
    fluxes_adjoint(t, g, nb, flb, Ub + (size_t)b * 2 * N, nullptr);
}

// adjoint of Fb(bvel): one thread per (boundary face, environment)
__global__ void k_adj_bflux(Tab t, const float *__restrict__ Fbb, float *__restrict__ Bvb, const int32_t *__restrict__ active) {
    const int b = blockIdx.y;
    if (active && !active[b]) return;   // skipped environment: identity cotangents from k_adj_inactive
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const int NB = t.NB;
    if (j >= NB) return;
    const int ax = t.b_face[j] >> 1;
    const float f = Fbb[(size_t)b * NB + j] * t.b_det[j];
    Bvb[(size_t)b * 2 * NB + j] += f * t.b_minv[(2 * ax) * NB + j];
    Bvb[(size_t)b * 2 * NB + NB + j] += f * t.b_minv[(2 * ax + 1) * NB + j];
}

// Passive scalar + buoyancy (RBC substep).  The velocity source enters the predictor right-hand side and HbyA next to
// S_b / det, so its adjoint is det * S_b_bar; with src = (0, beta * T_new):
//   T_new_bar = T_out_bar + beta * det * S_b_bar[1]
__global__ void __launch_bounds__(256) k_adj_buoyancy(Tab t, const float *__restrict__ Sbb, const float *__restrict__ Toutb, float beta,
                                                       float *__restrict__ Tnb, const int32_t *__restrict__ active) {
    const int b = blockIdx.y;
    if (active && !active[b]) return;   // skipped environment: identity cotangents from k_adj_inactive
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    const int N = t.N;
    if (g >= N) return;
    Tnb[(size_t)b * N + g] = Toutb[(size_t)b * N + g] + beta * t.det[g] * Sbb[(size_t)b * 2 * N + N + g];
}

// adjoint of k_setup_scalar + the scalar solve, given lam = C_s^-T T_new_bar:
//   A_s_bar = -lam * T_new, Coff_s_bar[f] = -lam * T_new[nb_f]; rhs_s = r / det with
//   r = det * T_in / dt + sum_{prescribed f} sb * (-(sig F_b) + kappa * (2 alpha_b | 1))
__global__ void __launch_bounds__(256) k_adj_scalar(Tab t, const float *__restrict__ Lam, const float *__restrict__ Tnew,
                                                     const float *__restrict__ Bvel, const float *__restrict__ Sbval,
                                                     const float *__restrict__ dtv, float *__restrict__ Tinb, float *__restrict__ Sbvalb,
                                                     float *__restrict__ Fbb, float *__restrict__ Ub, const int32_t *__restrict__ active) {
    const int b = blockIdx.y;
    if (active && !active[b]) return;   // skipped environment: identity cotangents from k_adj_inactive
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    const int N = t.N, NB = t.NB;
    if (g >= N) return;
    const float *tn = Tnew + (size_t)b * N, *bv = Bvel + (size_t)b * 2 * NB, *sb = Sbval + (size_t)b * NB;
    const float lam = Lam[(size_t)b * N + g];
    const float det = t.det[g];
    const float rb = lam / det;
    Tinb[(size_t)b * N + g] = lam / dtv[b];
    const float diagb = -lam * tn[g] / det;                 // A_s = diag / det
    int nb[4]; float flb[4];
#pragma unroll
    for (int f = 0; f < 4; ++f) {
        nb[f] = t.nbr[f * N + g];
        const float sig = (f & 1) ? 1.f : -1.f;
        flb[f] = 0.f;
        if (nb[f] >= 0) flb[f] = 0.5f * sig * (-lam * tn[nb[f]] / det + diagb);
        else {
            const int j = -1 - nb[f];
            const float Fb = bflux(t, j, f >> 1, bv[j], bv[NB + j]);
            const float dif = t.scalar_viscosity * (t.sb_neumann[j] == 0 ? 2.f * t.b_alpha[j] : 1.f);
            atomicAdd(&Sbvalb[(size_t)b * NB + j], rb * (-(sig * Fb) + dif));
            atomicAdd(&Fbb[(size_t)b * NB + j], -rb * sb[j] * sig);
        }
    }
    fluxes_adjoint(t, g, nb, flb, Ub + (size_t)b * 2 * N, nullptr);
}

// Cotangents of the environments a masked substep skipped (fgb_tape.active == 0): the substep is the identity there, so
// u_bar = u_out_bar, p_prev_bar = p_out_bar, T_bar = T_out_bar, bvel_bar = 0, sbval_bar = 0.  Shared by the 2-D, box and extruded
// reverse passes: nc velocity components and n cells per environment (p / T arrays optional), nbv boundary-velocity and nsb
// boundary-scalar values per environment.  One thread per (index, environment) over max(nc * n, nbv, nsb).
__global__ void k_adj_inactive(const int32_t *__restrict__ active, int nc, int n, const float *__restrict__ Uob, float *__restrict__ Ub,
                               const float *__restrict__ Pob, float *__restrict__ Pb, const float *__restrict__ Tob, float *__restrict__ Tb,
                               int nbv, float *__restrict__ Bvb, int nsb, float *__restrict__ Sbb) {
    const int b = blockIdx.y;
    if (active[b]) return;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const size_t nu = (size_t)nc * n;
    if ((size_t)i < nu) Ub[b * nu + i] = Uob[b * nu + i];
    if (i < n) {
        if (Pb) Pb[(size_t)b * n + i] = Pob[(size_t)b * n + i];
        if (Tb) Tb[(size_t)b * n + i] = Tob[(size_t)b * n + i];
    }
    if (i < nbv) Bvb[(size_t)b * nbv + i] = 0.f;
    if (Sbb && i < nsb) Sbb[(size_t)b * nsb + i] = 0.f;
}
static int launch_adj_inactive(const int32_t *active, int B, int nc, int n, const float *uob, float *ub, const float *pob, float *pb,
                               const float *tob, float *tb, int nbv, float *bvb, int nsb, float *sbb, cudaStream_t st) {
    if (!active) return 0;
    int m = nc * n;
    if (nbv > m) m = nbv;
    if (nsb > m) m = nsb;
    k_adj_inactive<<<dim3((unsigned)((m + 255) / 256), (unsigned)B), 256, 0, st>>>(active, nc, n, uob, ub, pob, pb, tob, tb, nbv, bvb, nsb, sbb);
    const cudaError_t ce = cudaGetLastError();
    return ce == cudaSuccess ? 0 : set_err(FGB_E_CUDA, "k_adj_inactive launch", ce);
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static inline dim3 cell_grid(const fgb_batch *b) { return dim3((b->t.N + 255) / 256, b->B); }
#define STREAM(s) ((cudaStream_t)(s))

static inline void launch_setup_advection(fgb_batch *b, cudaStream_t st, const float *u, const float *ures, const float *bvel, const float *src,
                                          const float *dt, const int32_t *active, int with_matrix) {
    const int ae = b->asm_envs > 1 ? b->asm_envs : 1;
    const dim3 gm((b->t.N + 255) / 256, (b->B + ae - 1) / ae);
    if (ae == 8) k_setup_advection_multi<8><<<gm, 256, 0, st>>>(b->t, b->B, u, ures, bvel, src, dt, active, b->Coff, b->A, b->rhs, with_matrix);
    else if (ae == 4) k_setup_advection_multi<4><<<gm, 256, 0, st>>>(b->t, b->B, u, ures, bvel, src, dt, active, b->Coff, b->A, b->rhs, with_matrix);
    else if (ae == 2) k_setup_advection_multi<2><<<gm, 256, 0, st>>>(b->t, b->B, u, ures, bvel, src, dt, active, b->Coff, b->A, b->rhs, with_matrix);
    else k_setup_advection<<<cell_grid(b), 256, 0, st>>>(b->t, u, ures, bvel, src, dt, active, b->Coff, b->A, b->rhs, with_matrix);
}

extern "C" int fgb_setup_advection(fgb_batch *b, const float *u, const float *ures, const float *bvel, const float *src,
                                   const float *dt, const int32_t *active, fgb_stream_t s) {
    if (!b || !u || !bvel || !dt) return set_err(FGB_E_ARG, "fgb_setup_advection: null argument");
    ProfScope ps(b, CLS_ASM, STREAM(s));
    launch_setup_advection(b, STREAM(s), u, ures ? ures : u, bvel, src, dt, active, 1);
    LAUNCH_CHECK("k_setup_advection");
    return FGB_OK;
}
extern "C" int fgb_solve_advection(fgb_batch *b, int zero_init, const int32_t *active, fgb_stream_t s) {
    if (!b) return set_err(FGB_E_ARG, "fgb_solve_advection: null argument");
    ProfScope ps(b, CLS_BICG, STREAM(s));
    return run_bicgstab<2>(b, b->rhs, b->ures, zero_init, active, STREAM(s));
}
extern "C" int fgb_setup_pressure_matrix(fgb_batch *b, const int32_t *active, fgb_stream_t s) {
    if (!b) return set_err(FGB_E_ARG, "fgb_setup_pressure_matrix: null argument");
    ProfScope ps(b, CLS_ASM, STREAM(s));
    const int ae = b->asm_envs > 1 ? b->asm_envs : 1;
    const dim3 gm((b->t.N + 255) / 256, (b->B + ae - 1) / ae);
    if (ae == 8) k_setup_pressure_matrix_multi<8><<<gm, 256, 0, STREAM(s)>>>(b->t, b->B, b->A, active, b->Poff, b->Pdiag);
    else if (ae == 4) k_setup_pressure_matrix_multi<4><<<gm, 256, 0, STREAM(s)>>>(b->t, b->B, b->A, active, b->Poff, b->Pdiag);
    else if (ae == 2) k_setup_pressure_matrix_multi<2><<<gm, 256, 0, STREAM(s)>>>(b->t, b->B, b->A, active, b->Poff, b->Pdiag);
    else k_setup_pressure_matrix<<<cell_grid(b), 256, 0, STREAM(s)>>>(b->t, b->A, active, b->Poff, b->Pdiag);
    LAUNCH_CHECK("k_setup_pressure_matrix");
    return FGB_OK;
}
extern "C" int fgb_setup_pressure_rhs(fgb_batch *b, const float *u, const float *bvel, const float *src, const float *p_prev,
                                      const float *dt, int with_hbya, const int32_t *active, fgb_stream_t s) {
    if (!b || !bvel) return set_err(FGB_E_ARG, "fgb_setup_pressure_rhs: null argument");
    ProfScope ps(b, CLS_ASM, STREAM(s));
    if (with_hbya) {
        if (!u || !dt) return set_err(FGB_E_ARG, "fgb_setup_pressure_rhs: u/dt required with_hbya");
        b->launches++;
        k_hbya<<<cell_grid(b), 256, 0, STREAM(s)>>>(b->t, u, b->ures, bvel, src, b->Coff, b->A, dt, active, b->hbya);
        LAUNCH_CHECK("k_hbya");
    }
    const int no = b->opt.nonortho && p_prev;
    const int ae = b->asm_envs > 1 ? b->asm_envs : 1;
    const dim3 gm((b->t.N + 255) / 256, (b->B + ae - 1) / ae);
    if (ae == 8) k_pressure_div_multi<8><<<gm, 256, 0, STREAM(s)>>>(b->t, b->B, b->hbya, bvel, p_prev, b->A, active, no, b->div);
    else if (ae == 4) k_pressure_div_multi<4><<<gm, 256, 0, STREAM(s)>>>(b->t, b->B, b->hbya, bvel, p_prev, b->A, active, no, b->div);
    else if (ae == 2) k_pressure_div_multi<2><<<gm, 256, 0, STREAM(s)>>>(b->t, b->B, b->hbya, bvel, p_prev, b->A, active, no, b->div);
    else k_pressure_div<<<cell_grid(b), 256, 0, STREAM(s)>>>(b->t, b->hbya, bvel, p_prev, b->A, active, no, b->div);
    LAUNCH_CHECK("k_pressure_div");
    return FGB_OK;
}

template <int CS, int CPT, int VARIANT>
static int launch_cg_cluster(fgb_batch *b, float *p_out, int zero_init, int reset_steps, int max_iter, int slot,
                             const int32_t *active, cudaStream_t st) {
    constexpr int T = 512;
    const int N = b->t.N;
    const int per = (N + CS - 1) / CS;
    if (per > T * CPT) return 1;  // does not fit this instantiation
    const size_t smem = ((size_t)2 * T * CPT + (size_t)2 * (T / 32) * CS) * sizeof(float) + 16;
    auto kern = k_cg_cluster<T, CPT, CS, VARIANT>;
    cudaError_t ce = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "cudaFuncSetAttribute(k_cg_cluster)", ce);
    cudaLaunchConfig_t cfg; memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(b->B * CS); cfg.blockDim = dim3(T); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CS; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    ce = cudaLaunchKernelEx(&cfg, kern, b->t, (const float *)b->Poff, (const float *)b->Pdiag, (const float *)b->div, p_out,
                            max_iter, b->opt.p_tol, zero_init, reset_steps, slot, active, b->iters, b->resid, b->iter_total);
    if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "cudaLaunchKernelEx(k_cg_cluster)", ce);
    return FGB_OK;
}

template <int CS, int CPT, bool PUSH = false, int T = 512, int MINB = 1>
static int launch_cg_cluster_mb(fgb_batch *b, const float *poff, const float *pdiag, const float *rhs, float *p_out, int zero_init,
                                int reset_steps, int max_iter, int slot, const int32_t *active, int flags, float *mean_out,
                                cudaStream_t st) {
    const int N = b->t.N;
    const int per = (N + CS - 1) / CS;
    if (per > T * CPT) return 1;
    if (PUSH && (!b->t.cg_slot || !b->t.cg_exp || !b->t.cg_cnt || b->t.cg_cs != CS || b->t.cg_pad != T * CPT))
        return set_err(FGB_E_ARG, "cg_impl 6: tables.cg_* (halo plan) missing or built for another cluster size");
    const size_t smem = ((size_t)2 * T * CPT + (size_t)2 * (T / 32) * CS + (PUSH ? (size_t)b->t.cg_hmax : 0)) * sizeof(float) + 4 * 8 + 16 +
                        (PUSH ? (size_t)b->t.cg_emax * 8 : 0);
    if (smem > 227 * 1024) return set_err(FGB_E_ARG, "cg_impl 6: halo plan does not fit in shared memory");
    auto kern = k_cg_cluster_mb<T, CPT, CS, PUSH, MINB>;
    cudaError_t ce = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "cudaFuncSetAttribute(k_cg_cluster_mb)", ce);
    if (CS > 8) {   // 16-CTA clusters are a non-portable size: opt in (one cluster then occupies most of a GPC)
        ce = cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
        if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "cudaFuncSetAttribute(k_cg_cluster_mb, non-portable cluster)", ce);
    }
    cudaLaunchConfig_t cfg; memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(b->B * CS); cfg.blockDim = dim3(T); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CS; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    ce = cudaLaunchKernelEx(&cfg, kern, b->t, poff, pdiag, rhs, p_out, max_iter, b->opt.p_tol, zero_init, reset_steps, slot, active,
                            b->iters, b->resid, b->iter_total, flags, mean_out);
    if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "cudaLaunchKernelEx(k_cg_cluster_mb)", ce);
    return FGB_OK;
}

template <int T, int CPT, int CS, int MINB, bool LAZY>
static int launch_cg_strip(fgb_batch *b, const float *poff, const float *pdiag, const float *rhs, float *p_out, int zero_init,
                           int reset_steps, int max_iter, int slot, const int32_t *active, int flags, float *mean_out,
                           cudaStream_t st) {
    if (b->t.st_cs != CS || b->t.st_T != T || b->t.st_cpt != CPT) return 1;
    if ((size_t)CS * T * CPT > (size_t)KRY_VECS * b->t.N)
        return set_err(FGB_E_ARG, "cg_impl 11/13: domain too small for the best-iterate scratch (use cg_impl 6)");
    const size_t smem = ((size_t)5 * CPT * T + (size_t)b->t.st_slots + (size_t)b->t.st_gmax + (size_t)2 * CS + 2 * (T / 32) + 2) * sizeof(float) + 4 * 8 +
                        ((size_t)b->t.st_remax + (size_t)b->t.st_lemax) * 8;
    if (smem > 227 * 1024 || (b->t.st_slots & 3) || (b->t.st_gmax & 1))
        return set_err(FGB_E_ARG, "cg_impl 11/13: strip plan does not fit in shared memory");
    auto kern = k_cg_strip<T, CPT, CS, MINB, LAZY>;
    cudaError_t ce = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "cudaFuncSetAttribute(k_cg_strip)", ce);
    if (CS > 8) {
        ce = cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
        if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "cudaFuncSetAttribute(k_cg_strip, non-portable cluster)", ce);
    }
    cudaLaunchConfig_t cfg; memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(b->B * CS); cfg.blockDim = dim3(T); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CS; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    ce = cudaLaunchKernelEx(&cfg, kern, b->t, poff, pdiag, rhs, p_out, max_iter, b->opt.p_tol, zero_init, reset_steps, slot, active,
                            b->iters, b->resid, b->iter_total, flags, mean_out, b->kry);
    if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "cudaLaunchKernelEx(k_cg_strip)", ce);
    return FGB_OK;
}

template <int T, int CPT, int MINB, bool LAZY>
static int cg_strip_cs(fgb_batch *b, const float *poff, const float *pdiag, const float *rhs, float *p_out, int zero_init,
                       int reset_steps, int max_iter, int slot, const int32_t *active, int flags, float *mean_out, cudaStream_t st) {
    int rc = launch_cg_strip<T, CPT, 1, MINB, LAZY>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
    if (rc == 1) rc = launch_cg_strip<T, CPT, 2, MINB, LAZY>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
    if (rc == 1) rc = launch_cg_strip<T, CPT, 4, MINB, LAZY>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
    if (rc == 1) rc = launch_cg_strip<T, CPT, 8, MINB, LAZY>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
    if (rc == 1) rc = launch_cg_strip<T, CPT, 16, MINB, LAZY>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
    return rc;
}
// instantiated shapes = fluidgym_b200/strip_plan.py::SHAPES: 4 / 2 / 1 co-resident CTAs per SM, 8 320 cells per SM in every case
template <bool LAZY>
static int cg_strip_any(fgb_batch *b, const float *poff, const float *pdiag, const float *rhs, float *p_out, int zero_init,
                        int reset_steps, int max_iter, int slot, const int32_t *active, int flags, float *mean_out, cudaStream_t st) {
    int rc = cg_strip_cs<480, 17, 1, LAZY>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
    if (rc == 1) rc = cg_strip_cs<256, 17, 2, LAZY>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
    if (rc == 1) rc = cg_strip_cs<896, 9, 1, LAZY>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
    if (rc == 1) rc = cg_strip_cs<640, 13, 1, LAZY>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
    if (rc == 1) rc = cg_strip_cs<320, 13, 2, LAZY>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
    return rc;
}


// cg_impl 12: two environments per cluster (k_cg_strip2); rc 1 = this instantiation does not match the plan
template <int T, int CPT, int CS>
static int launch_cg_strip2(fgb_batch *b, const float *poff, const float *pdiag, const float *rhs, float *p_out, int zero_init,
                            int reset_steps, int max_iter, int slot, const int32_t *active, int flags, float *mean_out,
                            cudaStream_t st) {
    if (b->t.st_cs != CS || b->t.st_T != T || b->t.st_cpt != CPT) return 1;
    if ((size_t)CS * T * CPT > (size_t)KRY_VECS * b->t.N)
        return set_err(FGB_E_ARG, "cg_impl 12: domain too small for the best-iterate scratch (use cg_impl 6)");
    const size_t envf = ((size_t)5 * CPT * T + (size_t)b->t.st_slots + (size_t)b->t.st_gmax + (size_t)2 * CS + 2 * (T / 32) + 3) & ~(size_t)3;
    const size_t smem = 2 * envf * sizeof(float) + 4 * 8 + 4 * 4 + ((size_t)b->t.st_remax + (size_t)b->t.st_lemax) * 8;
    if (smem > 227 * 1024 || (b->t.st_slots & 3) || (b->t.st_gmax & 1))
        return set_err(FGB_E_ARG, "cg_impl 12: strip plan does not fit in shared memory");
    auto kern = k_cg_strip2<T, CPT, CS>;
    cudaError_t ce = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "cudaFuncSetAttribute(k_cg_strip2)", ce);
    if (CS > 8) {
        ce = cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
        if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "cudaFuncSetAttribute(k_cg_strip2, non-portable cluster)", ce);
    }
    cudaLaunchConfig_t cfg; memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(((b->B + 1) / 2) * CS); cfg.blockDim = dim3(T); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CS; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    ce = cudaLaunchKernelEx(&cfg, kern, b->t, poff, pdiag, rhs, p_out, b->B, max_iter, b->opt.p_tol, zero_init, reset_steps, slot, active,
                            b->iters, b->resid, b->iter_total, flags, mean_out, b->kry);
    if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "cudaLaunchKernelEx(k_cg_strip2)", ce);
    return FGB_OK;
}
// instantiated: the shape of fluidgym_b200/strip_plan.py::SHAPES2 for 2 / 4 / 8-CTA clusters (an opt-in kernel kept for the measured
// comparison of profiles/r02_cg_strip_development.md: slower than k_cg_strip, see there)
static int cg_strip2_any(fgb_batch *b, const float *poff, const float *pdiag, const float *rhs, float *p_out, int zero_init,
                         int reset_steps, int max_iter, int slot, const int32_t *active, int flags, float *mean_out, cudaStream_t st) {
    int rc = launch_cg_strip2<480, 9, 2>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
    if (rc == 1) rc = launch_cg_strip2<480, 9, 4>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
    if (rc == 1) rc = launch_cg_strip2<480, 9, 8>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
    return rc;
}

static inline bool uses_halo_plan(int cg_impl) { return cg_impl == 6 || cg_impl == 11 || cg_impl == 12 || cg_impl == 13; }

static int cg_cluster_mb_any(fgb_batch *b, const float *poff, const float *pdiag, const float *rhs, float *p_out, int zero_init,
                             int reset_steps, int max_iter, int slot, const int32_t *active, int flags, float *mean_out, cudaStream_t st) {
    if (b->opt.cg_impl == 12 && b->t.st_thread && b->t.st_cell && b->t.st_rexp && b->t.st_lexp && b->t.st_cnt) {
        const int rc = cg_strip2_any(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
        if (rc == 1) return set_err(FGB_E_ARG, "cg_impl 12: no k_cg_strip2 instantiation for the shape (st_T, st_cpt, st_cs) of this strip plan");
        return rc;
    }
    // 11: k_cg_strip with the iterate update deferred and the best iterate stored lazily; 13: the same kernel with the eager
    // bookkeeping order (bit-identical results, kept for A/B measurements and as the in-tree reference of the reorder)
    if ((b->opt.cg_impl == 11 || b->opt.cg_impl == 13) && b->t.st_thread && b->t.st_cell && b->t.st_rexp && b->t.st_lexp && b->t.st_cnt) {
        const int rc = b->opt.cg_impl == 11
            ? cg_strip_any<true>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st)
            : cg_strip_any<false>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
        if (rc == 1) return set_err(FGB_E_ARG, "cg_impl 11/13: no k_cg_strip instantiation for the shape (st_T, st_cpt, st_cs) of this strip plan");
        return rc;
    }
    if (b->opt.cg_impl == 8) {       // as 6 with 256-thread CTAs of 1792 cells, TWO co-resident CTAs per SM (of different environments):
                                     // while one waits for a cluster hand-shake the other one computes
        int rc = launch_cg_cluster_mb<2, 7, true, 256, 2>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
        if (rc == 1) rc = launch_cg_cluster_mb<4, 7, true, 256, 2>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
        if (rc == 1) rc = launch_cg_cluster_mb<8, 7, true, 256, 2>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
        if (rc == 1) rc = launch_cg_cluster_mb<16, 7, true, 256, 2>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
        return rc;
    }
    if (b->opt.cg_impl == 7) {       // as 6 with half the threads and twice the cells per thread (same padding per CTA)
        int rc = launch_cg_cluster_mb<2, 12, true, 256>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
        if (rc == 1) rc = launch_cg_cluster_mb<4, 14, true, 256>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
        if (rc == 1) rc = launch_cg_cluster_mb<8, 14, true, 256>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
        if (rc == 1) rc = launch_cg_cluster_mb<16, 12, true, 256>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
        return rc;
    }
    if (uses_halo_plan(b->opt.cg_impl)) {   // pushed halos: same cluster-size rule, gathers from local shared memory (11 / 13 without a strip plan = 6)
        int rc = launch_cg_cluster_mb<2, 6, true>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
        if (rc == 1) rc = launch_cg_cluster_mb<4, 7, true>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
        if (rc == 1) rc = launch_cg_cluster_mb<8, 7, true>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
        if (rc == 1) rc = launch_cg_cluster_mb<16, 6, true>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
        return rc;
    }
    int rc = launch_cg_cluster_mb<2, 6>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
    if (rc == 1) rc = launch_cg_cluster_mb<4, 7>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
    if (rc == 1) rc = launch_cg_cluster_mb<8, 7>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
    if (rc == 1) rc = launch_cg_cluster_mb<16, 6>(b, poff, pdiag, rhs, p_out, zero_init, reset_steps, max_iter, slot, active, flags, mean_out, st);
    return rc;
}

template <int CS, int CPT, int MINB>
static int launch_cg_smem(fgb_batch *b, float *p_out, int zero_init, int reset_steps, int max_iter, int slot,
                          const int32_t *active, cudaStream_t st) {
    constexpr int T = 512;
    const int N = b->t.N;
    const int per = (N + CS - 1) / CS;
    if (per > T * CPT) return 1;
    const size_t smem = ((size_t)6 * T * CPT + (size_t)2 * (T / 32) * CS) * sizeof(float) + 3 * 8 + 16;
    auto kern = k_cg_smem<T, CPT, CS, MINB>;
    cudaError_t ce = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "cudaFuncSetAttribute(k_cg_smem)", ce);
    cudaLaunchConfig_t cfg; memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(b->B * CS); cfg.blockDim = dim3(T); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CS; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    ce = cudaLaunchKernelEx(&cfg, kern, b->t, (const float *)b->Poff, (const float *)b->Pdiag, (const float *)b->div, p_out,
                            max_iter, b->opt.p_tol, zero_init, reset_steps, slot, active, b->iters, b->resid, b->iter_total);
    if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "cudaLaunchKernelEx(k_cg_smem)", ce);
    return FGB_OK;
}

static int solve_pressure_slot(fgb_batch *b, float *p_out, int zero_init, int reset_steps, int max_iter, int slot,
                               const int32_t *active, fgb_stream_t s) {
    if (!b || !p_out) return set_err(FGB_E_ARG, "fgb_solve_pressure: null argument");
    const int mean_slot = slot < 0 ? 7 : (slot > 7 ? 7 : slot);      // pmean has 8 rows; iteration counters only 6
    if (slot < 0 || slot > 5) slot = 5;
    ProfScope ps(b, CLS_CG, STREAM(s));
    if (b->opt.cg_impl == 4) {
        int rc = launch_cg_smem<1, 12, 1>(b, p_out, zero_init, reset_steps, max_iter, slot, active, STREAM(s));
        if (rc == 1) rc = launch_cg_smem<2, 14, 1>(b, p_out, zero_init, reset_steps, max_iter, slot, active, STREAM(s));
        if (rc == 1) rc = launch_cg_smem<4, 12, 1>(b, p_out, zero_init, reset_steps, max_iter, slot, active, STREAM(s));
        if (rc <= 0) return rc;
    }
    if (b->opt.cg_impl == 5) {   // two co-resident CTAs per SM (64 registers per thread): twice the environments in flight
        int rc = launch_cg_smem<2, 6, 2>(b, p_out, zero_init, reset_steps, max_iter, slot, active, STREAM(s));
        if (rc == 1) rc = launch_cg_smem<4, 7, 2>(b, p_out, zero_init, reset_steps, max_iter, slot, active, STREAM(s));
        if (rc == 1) rc = launch_cg_smem<8, 7, 2>(b, p_out, zero_init, reset_steps, max_iter, slot, active, STREAM(s));
        if (rc <= 0) return rc;
    }
    if (b->opt.cg_impl == 3 || uses_halo_plan(b->opt.cg_impl) || b->opt.cg_impl == 7 || b->opt.cg_impl == 8) {
        int rc = cg_cluster_mb_any(b, b->Poff, b->Pdiag, b->div, p_out, zero_init, reset_steps, max_iter, slot, active, 0,
                                   b->pmean + (size_t)mean_slot * b->pmean_stride, STREAM(s));
        if (rc <= 0) return rc;
    }
    if (b->opt.cg_impl == 1 || b->opt.cg_impl == 2) {
        int rc;
        if (b->opt.cg_impl == 1) {
            rc = launch_cg_cluster<2, 6, 0>(b, p_out, zero_init, reset_steps, max_iter, slot, active, STREAM(s));
            if (rc == 1) rc = launch_cg_cluster<4, 7, 0>(b, p_out, zero_init, reset_steps, max_iter, slot, active, STREAM(s));
        } else {
            rc = launch_cg_cluster<2, 6, 1>(b, p_out, zero_init, reset_steps, max_iter, slot, active, STREAM(s));
            if (rc == 1) rc = launch_cg_cluster<4, 7, 1>(b, p_out, zero_init, reset_steps, max_iter, slot, active, STREAM(s));
        }
        if (rc <= 0) return rc;
        // too large for the on-chip variants: fall through to the global-memory kernel
    }
    k_cg<1024><<<b->B, 1024, 0, STREAM(s)>>>(b->t, b->Poff, b->Pdiag, b->div, p_out, b->kry, max_iter, b->opt.p_tol, zero_init,
                                             reset_steps, slot, active, b->iters, b->resid, b->iter_total);
    LAUNCH_CHECK("k_cg");
    return FGB_OK;
}
extern "C" int fgb_solve_pressure(fgb_batch *b, float *p_out, int zero_init, int reset_steps, int max_iter,
                                  const int32_t *active, fgb_stream_t s) {
    return solve_pressure_slot(b, p_out, zero_init, reset_steps, max_iter, 0, active, s);
}
extern "C" int fgb_correct_velocity(fgb_batch *b, const float *p, float *u_out, const int32_t *active, fgb_stream_t s) {
    if (!b || !p || !u_out) return set_err(FGB_E_ARG, "fgb_correct_velocity: null argument");
    ProfScope ps(b, CLS_ASM, STREAM(s));
    k_correct_velocity<<<cell_grid(b), 256, 0, STREAM(s)>>>(b->t, b->hbya, p, b->A, active, u_out);
    LAUNCH_CHECK("k_correct_velocity");
    return FGB_OK;
}

static int piso_substep_impl(fgb_batch *b, float *u, float *p, const float *bvel, const float *src, const float *dt,
                             const int32_t *active, const fgb_scalar *sc, fgb_stream_t s);

// view of environments [g0, g0 + cnt) of a batch
static fgb_batch group_view(fgb_batch *b, int g0, int cnt) {
    fgb_batch v = *b;
    const size_t N = b->t.N, o = (size_t)g0;
    v.B = cnt; v.groups = 1; v.parent = b->parent ? b->parent : b; v.launches = 0;
    v.Coff += 4 * o * N; v.A += o * N; v.rhs += 2 * o * N; v.ures += 2 * o * N; v.Poff += 4 * o * N; v.Pdiag += o * N;
    v.hbya += 2 * o * N; v.div += o * N; v.pres += o * N; v.kry += (size_t)KRY_VECS * o * N;
    v.resid += 8 * o; v.dt += o; v.maxvel += o; v.fluxbal += o; v.pmean += o; v.remaining += o;
    v.iters += 8 * o; v.active += o; v.nsub += o; v.iter_total += 2 * o;
    return v;
}

extern "C" int fgb_piso_substep(fgb_batch *b, float *u, float *p, const float *bvel, const float *src, const float *dt,
                                const int32_t *active, const fgb_scalar *sc, fgb_stream_t s) {
    if (!b || !u || !p || !bvel || !dt) return set_err(FGB_E_ARG, "fgb_piso_substep: null argument");
    const int G = b->groups;
    if (G <= 1 || b->B < 2 * G) return piso_substep_impl(b, u, p, bvel, src, dt, active, sc, s);
    cudaStream_t st = STREAM(s);
    cudaError_t ce;
    if (!b->gfork) {
        if ((ce = cudaEventCreateWithFlags(&b->gfork, cudaEventDisableTiming)) != cudaSuccess) return set_err(FGB_E_CUDA, "group event", ce);
        for (int g = 0; g < fgb_batch::MAX_GROUPS; ++g) {
            if ((ce = cudaEventCreateWithFlags(&b->gjoin[g], cudaEventDisableTiming)) != cudaSuccess) return set_err(FGB_E_CUDA, "group event", ce);
            if ((ce = cudaStreamCreateWithFlags(&b->gstream[g], cudaStreamNonBlocking)) != cudaSuccess) return set_err(FGB_E_CUDA, "group stream", ce);
        }
    }
    const size_t N = b->t.N, NB = b->t.NB;
    if ((ce = cudaEventRecord(b->gfork, st)) != cudaSuccess) return set_err(FGB_E_CUDA, "group fork", ce);
    for (int g = 0; g < G; ++g) {
        const int g0 = (int)(((long long)b->B * g) / G), g1 = (int)(((long long)b->B * (g + 1)) / G);
        fgb_batch v = group_view(b, g0, g1 - g0);
        fgb_scalar scv;
        if (sc) { scv = *sc; scv.T += (size_t)g0 * N; scv.sbval += (size_t)g0 * NB; scv.src += 2 * (size_t)g0 * N; }
        cudaStreamWaitEvent(b->gstream[g], b->gfork, 0);
        const int rc = piso_substep_impl(&v, u + 2 * (size_t)g0 * N, p + (size_t)g0 * N, bvel + 2 * (size_t)g0 * NB,
                                         src ? src + 2 * (size_t)g0 * N : nullptr, dt + g0, active ? active + g0 : nullptr,
                                         sc ? &scv : nullptr, (fgb_stream_t)b->gstream[g]);
        b->launches += v.launches;
        // the join is recorded even after an error so that the caller's stream never runs ahead of a group
        cudaEventRecord(b->gjoin[g], b->gstream[g]);
        cudaStreamWaitEvent(st, b->gjoin[g], 0);
        if (rc) return rc;
    }
    return FGB_OK;
}

static int piso_substep_impl(fgb_batch *b, float *u, float *p, const float *bvel, const float *src, const float *dt,
                             const int32_t *active, const fgb_scalar *sc, fgb_stream_t s) {
    int rc;
    const fgb_options &o = b->opt;
    cudaStream_t st = STREAM(s);
    const int N = b->t.N;
    // passive scalar first, with the velocity of the previous step (SIM.py:1471-1644), then the buoyancy hook
    if (sc) {
        if (!sc->T || !sc->sbval || !sc->src || !b->t.Cd_s || !b->t.sb_neumann)
            return set_err(FGB_E_ARG, "fgb_piso_substep: incomplete scalar description / tables");
        {
            ProfScope ps(b, CLS_ASM, st);
            k_setup_scalar<<<cell_grid(b), 256, 0, st>>>(b->t, u, sc->T, bvel, sc->sbval, dt, active, b->Coff, b->A, b->rhs);
            LAUNCH_CHECK("k_setup_scalar");
        }
        {
            ProfScope ps(b, CLS_BICG, st);
            if ((rc = run_bicgstab<1>(b, b->rhs, sc->T, 1, active, st))) return rc;
        }
        b->launches++;
        k_buoyancy<<<cell_grid(b), 256, 0, st>>>(sc->T, sc->beta, N, active, sc->src);
        LAUNCH_CHECK("k_buoyancy");
        src = sc->src;
    }
    // predictor (SIM.py:1662-1757).  Orthogonal path: one solve started from the previous velocityResult
    // (which is kept in the workspace buffer "ures"); non-orthogonal path: zero start, deferred corrections.
    const int n_adv = o.nonortho ? o.adv_nonortho_steps : 1;
    for (int ns = 0; ns < n_adv; ++ns) {
        b->launches++;
        launch_setup_advection(b, st, u, ns == 0 ? u : b->ures, bvel, src, dt, active, ns == 0);
        LAUNCH_CHECK("k_setup_advection");
        if ((rc = fgb_solve_advection(b, o.nonortho ? (ns == 0) : 0, active, s))) return rc;
    }
    // correctors (SIM.py:1777-1972)
    int slot = 0;
    const int n_p = o.nonortho ? o.p_nonortho_steps : 1;
    const int reset = o.nonortho ? 100 : 0;
    for (int cs = 0; cs < o.corrector_steps; ++cs) {
        if (cs == 0) { if ((rc = fgb_setup_pressure_matrix(b, active, s))) return rc; }   // A is unchanged between correctors
        for (int ps = 0; ps < n_p; ++ps) {
            if ((rc = fgb_setup_pressure_rhs(b, u, bvel, src, p, dt, ps == 0, active, s))) return rc;
            if ((rc = solve_pressure_slot(b, p, ps == 0, reset, o.max_iter, slot++, active, s))) return rc;
        }
        if ((rc = fgb_correct_velocity(b, p, b->ures, active, s))) return rc;
    }
    // CopyVelocityResultToBlocks (SIM.py:1974): "ures" keeps domain.velocityResult for the next predictor
    b->launches++;
    k_copy_active<<<dim3((2 * N + 255) / 256, b->B), 256, 0, st>>>(b->ures, u, 2 * N, active);
    LAUNCH_CHECK("k_copy_active");
    return FGB_OK;
}

static int copy_async(void *dst, const void *src, size_t bytes, cudaStream_t st) {
    cudaError_t ce = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, st);
    return ce == cudaSuccess ? FGB_OK : set_err(FGB_E_CUDA, "cudaMemcpyAsync (tape)", ce);
}

// fgb_piso_substep that additionally records the tape the backward pass needs, for the environments of tp->active (NULL: all).
// C = corrector_steps, n_adv / n_p = advect / pressure non-orthogonal iterations (1 / 1 on the orthogonal path).
// sc / stp: passive scalar + buoyancy (RBC), both or neither.  A skipped environment is the identity: every kernel and solve
// leaves its u, p (and T) alone, the final u <- ures copy is masked; its tape rows hold whatever the copies found and are never read.
static int record_impl(fgb_batch *b, float *u, float *p, const float *bvel, const float *dt, const fgb_tape *tp,
                       const fgb_scalar *sc, const fgb_tape_scalar *stp, fgb_stream_t s) {
    const fgb_options &o = b->opt;
    const int C = o.corrector_steps, n_adv = o.nonortho ? o.adv_nonortho_steps : 1, n_p = o.nonortho ? o.p_nonortho_steps : 1;
    // no residual reset in the differentiable backend: its LinearSolveFunction passes residualResetSteps = 0 in both directions
    // (DIFF.py:527-545, 574-590), unlike the plain backend's 100 (SIM.py:1908); on the singular pressure system the fp32 recurrence
    // residual then drifts and many solves end with "residual rising for 100 iterations -> best iterate", in the reference and here
    const int reset = 0;
    if ((o.cg_impl != 3 && !uses_halo_plan(o.cg_impl) && o.cg_impl != 7 && o.cg_impl != 8) || C < 1 || n_adv < 1 || n_p < 1 || C * n_p > 8)
        return set_err(FGB_E_ARG, "fgb_piso_substep_record: needs cg_impl 3 or 6 and correctors x pressure iterations <= 8");
    cudaStream_t st = STREAM(s);
    const size_t B = b->B, N = b->t.N, NB = b->t.NB;
    const int32_t *act = tp->active;
    int rc;
    if ((rc = copy_async(tp->u_in, u, 2 * B * N * 4, st))) return rc;
    if ((rc = copy_async(tp->p_in, p, B * N * 4, st))) return rc;
    if ((rc = copy_async(tp->bvel_in, bvel, 2 * B * NB * 4, st))) return rc;
    if ((rc = copy_async(tp->dt, dt, B * 4, st))) return rc;
    const float *src = nullptr;
    if (sc) {   // scalar transport with the incoming velocity, then the buoyancy source from the new temperature (SIM.py:1471-1657)
        if (!sc->T || !sc->sbval || !sc->src || !stp->T_in || !stp->T_out || !stp->sbval_in || !b->t.Cd_s || !b->t.sb_neumann)
            return set_err(FGB_E_ARG, "fgb_piso_substep_record_scalar: incomplete scalar description / tables");
        if ((rc = copy_async(stp->T_in, sc->T, B * N * 4, st))) return rc;
        if ((rc = copy_async(stp->sbval_in, sc->sbval, B * NB * 4, st))) return rc;
        {
            ProfScope ps(b, CLS_ASM, st);
            k_setup_scalar<<<cell_grid(b), 256, 0, st>>>(b->t, u, sc->T, bvel, sc->sbval, dt, act, b->Coff, b->A, b->rhs);
            LAUNCH_CHECK("k_setup_scalar");
        }
        {
            ProfScope ps(b, CLS_BICG, st);
            if ((rc = run_bicgstab<1>(b, b->rhs, sc->T, 1, act, st))) return rc;
        }
        if ((rc = copy_async(stp->T_out, sc->T, B * N * 4, st))) return rc;
        b->launches++;
        k_buoyancy<<<cell_grid(b), 256, 0, st>>>(sc->T, sc->beta, (int)N, act, sc->src);
        LAUNCH_CHECK("k_buoyancy");
        src = sc->src;
    }
    // The reference's differentiable mode starts EVERY linear solve from zero (advect_use_prev_result, advect_non_ortho_reuse_result and
    // pressure_reuse_result are all "True and not self.differentiable", SIM.py:1436-1440): the recorded forward pass does the same,
    // so that env.step(differentiable=True) reproduces the reference's differentiable run, which on the airfoil differs visibly from
    // its plain run (the deferred-correction pressure solves restart from zero and stop at residual ~4e-4).
    for (int k = 0; k < n_adv; ++k) {
        if ((rc = fgb_setup_advection(b, u, k == 0 ? u : b->ures, bvel, src, dt, act, s))) return rc;
        if ((rc = fgb_solve_advection(b, 1, act, s))) return rc;
        if ((rc = copy_async(tp->ustar + (size_t)k * 2 * B * N, b->ures, 2 * B * N * 4, st))) return rc;
    }
    if ((rc = copy_async(tp->Coff, b->Coff, 4 * B * N * 4, st))) return rc;
    if ((rc = copy_async(tp->A, b->A, B * N * 4, st))) return rc;
    if ((rc = fgb_setup_pressure_matrix(b, act, s))) return rc;
    for (int cs = 0; cs < C; ++cs) {
        for (int ps = 0; ps < n_p; ++ps) {
            const int q = cs * n_p + ps;
            if ((rc = fgb_setup_pressure_rhs(b, u, bvel, src, p, dt, ps == 0, act, s))) return rc;
            if ((rc = solve_pressure_slot(b, p, 1, reset, o.max_iter, q, act, s))) return rc;
            if ((rc = copy_async(tp->p + (size_t)q * B * N, p, B * N * 4, st))) return rc;
            if ((rc = copy_async(tp->pmean + (size_t)q * B, b->pmean + (size_t)q * B, B * 4, st))) return rc;
        }
        if ((rc = copy_async(tp->hb + (size_t)cs * 2 * B * N, b->hbya, 2 * B * N * 4, st))) return rc;
        if ((rc = fgb_correct_velocity(b, p, b->ures, act, s))) return rc;
        if (cs + 1 < C && (rc = copy_async(tp->u1 + (size_t)cs * 2 * B * N, b->ures, 2 * B * N * 4, st))) return rc;
    }
    if (!act) return copy_async(u, b->ures, 2 * B * N * 4, st);
    b->launches++;
    k_copy_active<<<dim3((unsigned)((2 * N + 255) / 256), b->B), 256, 0, st>>>(b->ures, u, (int)(2 * N), act);
    LAUNCH_CHECK("k_copy_active (record)");
    return FGB_OK;
}
extern "C" int fgb_piso_substep_record(fgb_batch *b, float *u, float *p, const float *bvel, const float *dt, const fgb_tape *tp,
                                       fgb_stream_t s) {
    if (!b || !u || !p || !bvel || !dt || !tp) return set_err(FGB_E_ARG, "fgb_piso_substep_record: null argument");
    if (!b->opt.nonortho) return set_err(FGB_E_ARG, "fgb_piso_substep_record: needs the non-orthogonal path (use fgb_piso_substep_record_scalar for the orthogonal scalar path)");
    return record_impl(b, u, p, bvel, dt, tp, nullptr, nullptr, s);
}
extern "C" int fgb_piso_substep_record_scalar(fgb_batch *b, float *u, float *p, const float *bvel, const float *dt, const fgb_scalar *sc,
                                              const fgb_tape *tp, const fgb_tape_scalar *stp, fgb_stream_t s) {
    if (!b || !u || !p || !bvel || !dt || !tp || !sc || !stp) return set_err(FGB_E_ARG, "fgb_piso_substep_record_scalar: null argument");
    return record_impl(b, u, p, bvel, dt, tp, sc, stp, s);
}

extern "C" size_t fgb_adjoint_workspace_bytes(const fgb_tables *t, int32_t B) {
    const size_t BN = (size_t)B * t->N, BNB = (size_t)B * (t->NB > 0 ? t->NB : 1);
    return (size_t)(2 + 2 + 1 + 4 + 2 + 1 + 1 + 1 + 2 + 1 + 2 + 1 + 2) * align_up(BN * 4) + align_up(BNB * 4) + 8192;
}

// Reverse pass of fgb_piso_substep_record.  u_out_bar / p_out_bar: incoming gradients; u_bar, p_prev_bar, bvel_bar
// are OVERWRITTEN with the gradients w.r.t. the inputs of the substep.  ws: >= fgb_adjoint_workspace_bytes.  Environments that
// tp->active skips are skipped by every adjoint kernel and transposed solve and get the identity cotangents (k_adj_inactive).
static int backward_impl(fgb_batch *b, const fgb_tape *tp, const fgb_tape_scalar *stp, float beta, const float *u_out_bar,
                         const float *p_out_bar, const float *T_out_bar, float *u_bar, float *p_prev_bar, float *bvel_bar,
                         float *T_bar, float *sbval_bar, void *ws, size_t ws_bytes, fgb_stream_t s) {
    if (!b || !tp || !u_out_bar || !p_out_bar || !u_bar || !p_prev_bar || !bvel_bar || !ws)
        return set_err(FGB_E_ARG, "fgb_piso_substep_backward: null argument");
    if (stp && (!T_out_bar || !T_bar || !sbval_bar || !stp->T_in || !stp->T_out || !stp->sbval_in || !b->t.Cd_s || !b->t.sb_neumann))
        return set_err(FGB_E_ARG, "fgb_piso_substep_backward_scalar: incomplete scalar tape / tables");
    if (ws_bytes < fgb_adjoint_workspace_bytes(&b->t, b->B)) return set_err(FGB_E_WORKSPACE, "fgb_piso_substep_backward: workspace too small");
    if (!b->t.rev) return set_err(FGB_E_ARG, "fgb_piso_substep_backward: tables.rev missing");
    cudaStream_t st = STREAM(s);
    const size_t B = b->B, N = b->t.N, NB = b->t.NB, BN = B * N;
    const int32_t *act = tp->active;
    Carver c{(char *)ws, 0};
    float *unb = c.take<float>(2 * BN), *hbb = c.take<float>(2 * BN), *rAb = c.take<float>(BN), *Coffb = c.take<float>(4 * BN);
    float *Sbb = c.take<float>(2 * BN), *pb = c.take<float>(BN), *xb = c.take<float>(BN), *lam = c.take<float>(BN);
    float *uprevb = c.take<float>(2 * BN), *Ab = c.take<float>(BN), *mu = c.take<float>(2 * BN), *Fbb = c.take<float>(B * NB);
    float *pb2 = c.take<float>(BN), *xkb = c.take<float>(2 * BN);
    const fgb_options &o = b->opt;
    const int C = o.corrector_steps, n_adv = o.nonortho ? o.adv_nonortho_steps : 1, n_p = o.nonortho ? o.p_nonortho_steps : 1;
    if (C < 1 || n_adv < 1 || n_p < 1 || C * n_p > 8) return set_err(FGB_E_ARG, "fgb_piso_substep_backward: unsupported iteration counts");
    const dim3 grid = cell_grid(b);
    cudaError_t ce;
#define ZERO(ptr, n) do { ce = cudaMemsetAsync(ptr, 0, (n) * sizeof(float), st); if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "memset", ce); } while (0)
    ZERO(rAb, BN); ZERO(Coffb, 4 * BN); ZERO(Sbb, 2 * BN); ZERO(Fbb, B * NB); ZERO(u_bar, 2 * BN); ZERO(bvel_bar, 2 * B * NB);
    int rc;
    if ((rc = copy_async(unb, u_out_bar, 2 * BN * 4, st))) return rc;
    if ((rc = copy_async(pb, p_out_bar, BN * 4, st))) return rc;
    // the pressure matrix of this substep (function of A only)
    b->launches++;
    k_setup_pressure_matrix<<<grid, 256, 0, st>>>(b->t, tp->A, act, b->Poff, b->Pdiag);
    LAUNCH_CHECK("k_setup_pressure_matrix (backward)");
    for (int cs = C - 1; cs >= 0; --cs) {
        const float *hb_c = tp->hb + (size_t)cs * 2 * BN;
        const float *uprev = cs == 0 ? tp->ustar + (size_t)(n_adv - 1) * 2 * BN : tp->u1 + (size_t)(cs - 1) * 2 * BN;
        b->launches++;
        // u_next = hb - rA grad(p of the last pressure iteration): hbb = unb, rAb +=, pb += grad^T
        k_adj_correct<<<grid, 256, 0, st>>>(b->t, unb, tp->p + (size_t)(cs * n_p + n_p - 1) * BN, tp->A, hbb, rAb, pb, act);
        LAUNCH_CHECK("k_adj_correct");
        for (int ps = n_p - 1; ps >= 0; --ps) {
            const int q = cs * n_p + ps;
            // the pressure the deferred term of this solve read: previous iteration, previous corrector, or the input
            const float *pprev = q == 0 ? tp->p_in : tp->p + (size_t)(q - 1) * BN;
            b->launches++;
            k_adj_remove_mean<256><<<b->B, 256, 0, st>>>((int)N, pb, xb, act);
            LAUNCH_CHECK("k_adj_remove_mean");
            {   // lam = P^-T x_bar
                ProfScope psc(b, CLS_CG, st);
                rc = cg_cluster_mb_any(b, b->Poff, b->Pdiag, xb, lam, 1, 0, b->opt.max_iter, 5, act, 1 | 2, nullptr, st);
                if (rc == 1) return set_err(FGB_E_ARG, "fgb_piso_substep_backward: grid too large for the on-chip transposed solve");
                if (rc) return rc;
            }
            ZERO(pb2, BN);                 // becomes the gradient w.r.t. pprev
            b->launches++;
            k_adj_pressure_rhs<<<grid, 256, 0, st>>>(b->t, lam, tp->p + (size_t)q * BN, tp->pmean + (size_t)q * B, pprev, tp->A, hbb, Fbb, rAb, pb2, act);
            LAUNCH_CHECK("k_adj_pressure_rhs");
            float *tmp = pb; pb = pb2; pb2 = tmp;      // the previous iterate enters only through that deferred term
        }
        ZERO(uprevb, 2 * BN);
        b->launches++;
        k_adj_hbya<<<grid, 256, 0, st>>>(b->t, hbb, hb_c, tp->A, tp->Coff, uprev, tp->dt, rAb, u_bar, Sbb, Coffb, uprevb, act);
        LAUNCH_CHECK("k_adj_hbya");
        float *tmp = unb; unb = uprevb; uprevb = tmp;   // gradient w.r.t. the velocity entering this corrector
    }
    if ((rc = copy_async(p_prev_bar, pb, BN * 4, st))) return rc;
    // predictor iterations x_k = C^-1 rhs(u, x_{k-1}), x_{-1} = u, in reverse; unb holds the gradient w.r.t. the last one
    float *xb_cur = unb, *xb_prev = xkb;
    for (int k = n_adv - 1; k >= 0; --k) {
        {   // mu = C^-T x_k_bar
            ProfScope psc(b, CLS_BICG, st);
            rc = bicgstab_cluster_any<2>(b, tp->Coff, tp->A, xb_cur, mu, 1, act, 1, st);
            if (rc == 1) return set_err(FGB_E_ARG, "fgb_piso_substep_backward: grid too large for the on-chip transposed solve");
            if (rc) return rc;
        }
        if (k > 0) ZERO(xb_prev, 2 * BN);
        b->launches++;
        k_adj_advection<<<grid, 256, 0, st>>>(b->t, mu, tp->ustar + (size_t)k * 2 * BN, rAb, tp->A, tp->dt, Ab, Coffb, u_bar, Sbb, bvel_bar,
                                              k > 0 ? xb_prev : u_bar, k == n_adv - 1, act);
        LAUNCH_CHECK("k_adj_advection");
        float *tmp = xb_cur; xb_cur = xb_prev; xb_prev = tmp;
    }
    b->launches += 2;
    k_adj_assemble<<<grid, 256, 0, st>>>(b->t, Ab, Coffb, Sbb, tp->bvel_in, u_bar, bvel_bar, Fbb, act);
    LAUNCH_CHECK("k_adj_assemble");
    if (stp) {
        // buoyancy + scalar transport (they ran BEFORE the predictor): T_new_bar from the source adjoint, one transposed
        // scalar solve, then the assembly adjoint.  xb / lam (pressure temporaries) are free again; the scalar matrix is
        // rebuilt from the taped inputs into the forward workspace (Coff / A / rhs are not read by this pass).
        float *Tnb = xb;
        b->launches += 3;
        k_adj_buoyancy<<<grid, 256, 0, st>>>(b->t, Sbb, T_out_bar, beta, Tnb, act);
        LAUNCH_CHECK("k_adj_buoyancy");
        k_setup_scalar<<<grid, 256, 0, st>>>(b->t, tp->u_in, stp->T_in, tp->bvel_in, stp->sbval_in, tp->dt, act, b->Coff, b->A, b->rhs);
        LAUNCH_CHECK("k_setup_scalar (backward)");
        {
            ProfScope psc(b, CLS_BICG, st);
            rc = bicgstab_cluster_any<1>(b, b->Coff, b->A, Tnb, lam, 1, act, 1, st);
            if (rc == 1) return set_err(FGB_E_ARG, "fgb_piso_substep_backward_scalar: grid too large for the on-chip transposed solve");
            if (rc) return rc;
        }
        ZERO(sbval_bar, B * NB);
        k_adj_scalar<<<grid, 256, 0, st>>>(b->t, lam, stp->T_out, tp->bvel_in, stp->sbval_in, tp->dt, T_bar, sbval_bar, Fbb, u_bar, act);
        LAUNCH_CHECK("k_adj_scalar");
    }
    k_adj_bflux<<<dim3((unsigned)((NB + 127) / 128), b->B), 128, 0, st>>>(b->t, Fbb, bvel_bar, act);
    LAUNCH_CHECK("k_adj_bflux");
#undef ZERO
    if (act) b->launches++;
    return launch_adj_inactive(act, b->B, 2, (int)N, u_out_bar, u_bar, p_out_bar, p_prev_bar, stp ? T_out_bar : nullptr, stp ? T_bar : nullptr,
                               (int)(2 * NB), bvel_bar, stp ? (int)NB : 0, stp ? sbval_bar : nullptr, st);
}
extern "C" int fgb_piso_substep_backward(fgb_batch *b, const fgb_tape *tp, const float *u_out_bar, const float *p_out_bar,
                                         float *u_bar, float *p_prev_bar, float *bvel_bar, void *ws, size_t ws_bytes, fgb_stream_t s) {
    return backward_impl(b, tp, nullptr, 0.f, u_out_bar, p_out_bar, nullptr, u_bar, p_prev_bar, bvel_bar, nullptr, nullptr, ws, ws_bytes, s);
}
extern "C" int fgb_piso_substep_backward_scalar(fgb_batch *b, const fgb_tape *tp, const fgb_tape_scalar *stp, float beta,
                                                const float *u_out_bar, const float *p_out_bar, const float *T_out_bar, float *u_bar,
                                                float *p_prev_bar, float *bvel_bar, float *T_bar, float *sbval_bar, void *ws,
                                                size_t ws_bytes, fgb_stream_t s) {
    if (!stp) return set_err(FGB_E_ARG, "fgb_piso_substep_backward_scalar: null scalar tape");
    return backward_impl(b, tp, stp, beta, u_out_bar, p_out_bar, T_out_bar, u_bar, p_prev_bar, bvel_bar, T_bar, sbval_bar, ws, ws_bytes, s);
}

extern "C" int fgb_make_divergence_free(fgb_batch *b, float *u, float *p, const float *bvel, int max_iter, fgb_stream_t s) {
    if (!b || !u || !p || !bvel) return set_err(FGB_E_ARG, "fgb_make_divergence_free: null argument");
    cudaStream_t st = STREAM(s);
    const size_t BN = (size_t)b->B * b->t.N;
    int rc;
    b->launches += 2;
    k_fill<<<(unsigned)((BN + 255) / 256), 256, 0, st>>>(b->A, 1.0f, BN);
    LAUNCH_CHECK("k_fill");
    cudaError_t ce = cudaMemcpyAsync(b->hbya, u, 2 * BN * sizeof(float), cudaMemcpyDeviceToDevice, st);
    if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "memcpy hbya", ce);
    if ((rc = fgb_setup_pressure_matrix(b, nullptr, s))) return rc;
    for (int ps = 0; ps < b->opt.p_nonortho_steps; ++ps) {
        if ((rc = fgb_setup_pressure_rhs(b, nullptr, bvel, nullptr, p, nullptr, 0, nullptr, s))) return rc;
        if ((rc = solve_pressure_slot(b, p, ps == 0, 0, max_iter, ps, nullptr, s))) return rc;
    }
    return fgb_correct_velocity(b, p, u, nullptr, s);
}

extern "C" int fgb_sim_step(fgb_batch *b, float *u, float *p, float *bvel, const float *src, float dt_target, float cfl,
                            const float *char_vel, float bc_tol, const fgb_scalar *sc, int32_t *substeps_max, fgb_stream_t s) {
    if (!b || !u || !p || !bvel) return set_err(FGB_E_ARG, "fgb_sim_step: null argument");
    cudaStream_t st = STREAM(s);
    b->launches++;
    k_set_remaining<<<(b->B + 255) / 256, 256, 0, st>>>(b->remaining, b->nsub, b->counters, (double)dt_target, b->B);
    LAUNCH_CHECK("k_set_remaining");
    const int do_out = (char_vel != nullptr) && (b->t.b_out != nullptr);
    int rounds = 0;
    for (;; ++rounds) {
        if (rounds > 1000) return set_err(FGB_E_ARG, "fgb_sim_step: more than 1000 adaptive substeps");
        b->launches += 2;
        k_zero_counter<<<1, 1, 0, st>>>(b->counters);
        k_plan_substep<512><<<b->B, 512, 0, st>>>(b->t, u, bvel, b->remaining, b->dt, b->active, b->nsub, b->maxvel, b->counters,
                                                  cfl, do_out ? char_vel[0] : 0.f, do_out ? char_vel[1] : 0.f, bc_tol, do_out);
        LAUNCH_CHECK("k_plan_substep");
        cudaError_t ce = cudaMemcpyAsync(b->h_counters, b->counters, sizeof(int32_t), cudaMemcpyDeviceToHost, st);
        if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "memcpy counters", ce);
        ce = cudaStreamSynchronize(st);
        if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "fgb_sim_step: stream sync", ce);
        if (b->h_counters[0] == 0) break;
        int rc = fgb_piso_substep(b, u, p, bvel, src, b->dt, b->active, sc, s);
        if (rc) return rc;
    }
    if (substeps_max) *substeps_max = rounds;
    return FGB_OK;
}

extern "C" int fgb_update_outflow(fgb_batch *b, const float *u, float *bvel, const float *dt, const float *char_vel, float bc_tol,
                                  fgb_stream_t s) {
    if (!b || !u || !bvel || !dt || !char_vel) return set_err(FGB_E_ARG, "fgb_update_outflow: null argument");
    if (!b->t.b_out) return FGB_OK;
    b->launches++;
    k_update_outflow<512><<<b->B, 512, 0, STREAM(s)>>>(b->t, u, bvel, dt, char_vel[0], char_vel[1], bc_tol);
    LAUNCH_CHECK("k_update_outflow");
    return FGB_OK;
}
extern "C" int fgb_flux_balance(fgb_batch *b, const float *bvel, float *out, fgb_stream_t s) {
    if (!b || !bvel || !out) return set_err(FGB_E_ARG, "fgb_flux_balance: null argument");
    b->launches++;
    k_flux_balance<256><<<b->B, 256, 0, STREAM(s)>>>(b->t, bvel, out);
    LAUNCH_CHECK("k_flux_balance");
    return FGB_OK;
}
extern "C" int fgb_balance_fluxes(fgb_batch *b, float *bvel, const int8_t *free_mask, float bc_tol, fgb_stream_t s) {
    if (!b || !bvel || !free_mask) return set_err(FGB_E_ARG, "fgb_balance_fluxes: null argument");
    b->launches++;
    k_balance_fluxes<256><<<b->B, 256, 0, STREAM(s)>>>(b->t, bvel, free_mask, bc_tol);
    LAUNCH_CHECK("k_balance_fluxes");
    return FGB_OK;
}

// PISOtorch.ComputeSpatialVelocityGradients on the 2-D multi-block domains (getBlockDataGradient, K.cu:2997-3043, 6460-6550; vorticity of
// envs/fluid_env.py:577-656): central differences in computational space -- against a prescribed (Dirichlet) face the face value with
// distance 1.5 -- times M^-1 (row vector x matrix).  Gout[b][c][d][N] = d u_c / d x_d: as in the reference the outer index is the velocity
// component and the inner one the direction.
__global__ void __launch_bounds__(256) k_velocity_gradients(Tab t, const float *__restrict__ U, const float *__restrict__ Bvel, float *__restrict__ Gout) {
    const int b = blockIdx.y, g = blockIdx.x * blockDim.x + threadIdx.x, N = t.N, NB = t.NB;
    if (g >= N) return;
    const float *u = U + (size_t)b * 2 * N, *bv = Bvel + (size_t)b * 2 * NB;
    int nl[2], nu[2]; float dist[2];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        nl[i] = t.nbr[(2 * i) * N + g]; nu[i] = t.nbr[(2 * i + 1) * N + g];
        dist[i] = 2.0f - (nl[i] < 0 ? 0.5f : 0.f) - (nu[i] < 0 ? 0.5f : 0.f);
    }
#pragma unroll
    for (int c = 0; c < 2; ++c) {
        float dG[2];
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const float lo = nl[i] >= 0 ? u[c * N + nl[i]] : bv[c * NB + (-1 - nl[i])];
            const float hi = nu[i] >= 0 ? u[c * N + nu[i]] : bv[c * NB + (-1 - nu[i])];
            dG[i] = (hi - lo) / dist[i];
        }
#pragma unroll
        for (int j = 0; j < 2; ++j)
            Gout[(((size_t)b * 2 + c) * 2 + j) * N + g] = dG[0] * t.minv[j * N + g] + dG[1] * t.minv[(2 + j) * N + g];
    }
}
extern "C" int fgb_velocity_gradients(fgb_batch *b, const float *u, const float *bvel, float *grad_out, fgb_stream_t s) {
    if (!b || !u || !bvel || !grad_out) return set_err(FGB_E_ARG, "fgb_velocity_gradients: null argument");
    b->launches++;
    k_velocity_gradients<<<cell_grid(b), 256, 0, STREAM(s)>>>(b->t, u, bvel, grad_out);
    LAUNCH_CHECK("k_velocity_gradients");
    return FGB_OK;
}
extern "C" int fgb_max_velocity(fgb_batch *b, const float *u, const float *bvel, float *out, fgb_stream_t s) {
    if (!b || !u || !bvel || !out) return set_err(FGB_E_ARG, "fgb_max_velocity: null argument");
    b->launches++;
    k_max_velocity<512><<<b->B, 512, 0, STREAM(s)>>>(b->t, u, bvel, out);
    LAUNCH_CHECK("k_max_velocity");
    return FGB_OK;
}
extern "C" int fgb_apply_jet_action(fgb_batch *b, float *bvel, float *last_control, const float *action, float smoothing,
                                    const int32_t *faces, const float *templ, int32_t n_faces, fgb_stream_t s) {
    if (!b || !bvel || !last_control || !action || !faces || !templ) return set_err(FGB_E_ARG, "fgb_apply_jet_action: null argument");
    b->launches++;
    k_apply_jet<<<b->B, 64, 0, STREAM(s)>>>(bvel, last_control, action, smoothing, faces, templ, n_faces, b->t.NB, b->B);
    LAUNCH_CHECK("k_apply_jet");
    return FGB_OK;
}
extern "C" int fgb_wall_forces(fgb_batch *b, const fgb_wall *w, const float *u, const float *p, const float *bvel, float *acc,
                               fgb_stream_t s) {
    if (!b || !w || !u || !p || !bvel || !acc) return set_err(FGB_E_ARG, "fgb_wall_forces: null argument");
    b->launches++;
    k_wall_forces<<<b->B, 128, 0, STREAM(s)>>>(*w, b->t.viscosity, b->t.N, b->t.NB, u, p, bvel, acc);
    LAUNCH_CHECK("k_wall_forces");
    return FGB_OK;
}
extern "C" int fgb_column_sums(fgb_batch *b, const float *fa, const float *fb, int32_t nx, int32_t ny, float *out, fgb_stream_t s) {
    if (!b || !fa || !fb || !out || nx * ny != b->t.N) return set_err(FGB_E_ARG, "fgb_column_sums: bad argument (single nx*ny block expected)");
    b->launches++;
    k_column_sums<<<dim3((nx + 63) / 64, b->B), 64, 0, STREAM(s)>>>(b->t, fa, fb, nx, ny, out);
    LAUNCH_CHECK("k_column_sums");
    return FGB_OK;
}
extern "C" int fgb_sample_sensors(fgb_batch *b, const float *field, int32_t channels, const int32_t *idx, const float *w,
                                  int32_t K, int32_t n_sensors, float *out, fgb_stream_t s) {
    if (!b || !field || !idx || !w || !out) return set_err(FGB_E_ARG, "fgb_sample_sensors: null argument");
    dim3 grid((channels * n_sensors + 127) / 128, b->B);
    b->launches++;
    k_sample_sensors<<<grid, 128, 0, STREAM(s)>>>(field, channels, b->t.N, idx, w, K, n_sensors, out);
    LAUNCH_CHECK("k_sample_sensors");
    return FGB_OK;
}

// handle-free variant (any field layout [B][channels][N]; used by the 3-D environments, whose solver handle is fgb_ortho3)
extern "C" int fgb_sample_sensors_n(const float *field, int32_t B, int32_t channels, int32_t N, const int32_t *idx, const float *w,
                                    int32_t K, int32_t n_sensors, float *out, fgb_stream_t s) {
    if (!field || !idx || !w || !out || B <= 0 || channels <= 0 || N <= 0) return set_err(FGB_E_ARG, "fgb_sample_sensors_n: bad argument");
    dim3 grid((channels * n_sensors + 127) / 128, B);
    k_sample_sensors<<<grid, 128, 0, STREAM(s)>>>(field, channels, N, idx, w, K, n_sensors, out);
    LAUNCH_CHECK("k_sample_sensors");
    return FGB_OK;
}

extern "C" int fgb_render_gather(const float *field, int32_t B, int32_t channels, int32_t N, int64_t chan_stride, int64_t env_stride,
                                 int32_t mode, const int32_t *rowptr, const int32_t *col, const float *w, int32_t P, float *img,
                                 uint32_t *range, fgb_stream_t s) {
    if (!field || !rowptr || !col || !w || !img || B <= 0 || B > 65535 || N <= 0 || P <= 0 || chan_stride < 0 || env_stride < 0)
        return set_err(FGB_E_ARG, "fgb_render_gather: bad argument");
    if (!((mode == FGB_RENDER_IDENTITY && channels == 1) || (mode == FGB_RENDER_NORM && channels >= 2 && channels <= 3)))
        return set_err(FGB_E_ARG, "fgb_render_gather: mode IDENTITY takes 1 channel, NORM 2 or 3");
    if (range) {
        cudaError_t ce = cudaMemsetAsync(range, 0xff, sizeof(uint32_t) * 2 * (size_t)B, STREAM(s));
        if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "fgb_render_gather: range initialisation", ce);
    }
    dim3 grid((P + RENDER_THREADS - 1) / RENDER_THREADS, B);
    k_render_gather<<<grid, RENDER_THREADS, 0, STREAM(s)>>>(field, channels, chan_stride, env_stride, mode, rowptr, col, w, P, img, range);
    LAUNCH_CHECK("k_render_gather");
    return FGB_OK;
}

extern "C" int fgb_render_colour(const float *img, int32_t B, int32_t P, const uint32_t *range, float vmin, float vmax,
                                 int32_t symmetric, const uint8_t *lut, uint8_t *rgb, fgb_stream_t s) {
    if (!img || !lut || !rgb || B <= 0 || P <= 0) return set_err(FGB_E_ARG, "fgb_render_colour: bad argument");
    if ((reinterpret_cast<uintptr_t>(img) & 15) || (reinterpret_cast<uintptr_t>(rgb) & 3))
        return set_err(FGB_E_ARG, "fgb_render_colour: img must be 16-byte and rgb 4-byte aligned");
    const long long total = (long long)B * P;
    const long long groups = (total + 3) / 4;
    k_render_colour<<<(unsigned int)((groups + RENDER_THREADS - 1) / RENDER_THREADS), RENDER_THREADS, 0, STREAM(s)>>>(
        img, P, total, range, vmin, vmax, symmetric, lut, rgb);
    LAUNCH_CHECK("k_render_colour");
    return FGB_OK;
}

// D = 3 orthogonal-grid path (turbulent channel flow)
#include "ortho3_b200.cuh"

// D = 3 operators on z-extruded multi-block domains (CylinderJet3D / Airfoil3D): 2-D tables + periodic z faces
#include "extruded3_b200.cuh"
