// D = 3 operators on z-EXTRUDED multi-block domains (CylinderJet3D, Airfoil3D: the 2-D multi-block grid repeated over nz
// uniform, periodic z planes; envs/cylinder/grid.py:298, shapes.py:641-676; reference: the K.cu kernels with DIMS = 3).
//
// The per-cell functions below are __host__ __device__ so that tests/test_extruded_host.py can execute exactly this code on the
// CPU (through tests/cpu_harness/extruded_host.cu) and compare it with the numpy specification oracle/extruded_eval.py, which is
// pinned to an op trace of the unmodified reference on CylinderJet3D-easy (tests/golden/cyl3d_substep*.npz).  The launch glue at
// the end of this file is verified on a B200 against the same goldens (tests/test_gpu_extruded.py, profiles/r02_extruded_check.json):
// substep u 1.7e-6 / p 5.6e-5 with the reference's iteration counts, a whole env.step inside the bars of tools/extruded_check.py.
//
// The metric tensor of an extruded cell is block diagonal, M3 = diag(M2, hz): every in-plane coefficient of a row / det3
// equals the 2-D one from the compiled tables (fgb_tables), the z faces add  -+1/4 (u_z,P + u_z,N) / hz - nu / hz^2  off
// the diagonal; all non-orthogonal (corner) terms stay in the x-y plane because alpha^{xz} = alpha^{yz} = 0.
//
// Layout: cell g3 = k * N2 + g (plane k, 2-D cell g); fields [B][3][N3]; boundary velocities [B][3][nz][NB2]; matrices
// ELL(7) on a 6-face neighbour table (faces 0..3 in plane, 4 = -z, 5 = +z) so that the cooperative Krylov kernels of
// ortho3_b200.cuh (k3_bicgstab, k3_cg) solve them unchanged.
#pragma once

#ifndef X3_HD
#define X3_HD __host__ __device__ __forceinline__
#endif

struct X3Tab {
    fgb_tables t;     // in-plane tables of the compiled 2-D domain
    int nz;           // z planes (periodic)
    float hz;         // plane spacing
};

X3_HD float x3_contra(const fgb_tables &t, int k, int g, float u, float v) {          // det2 * (Minv[k] . (u, v))   (K.cu:495-510)
    const int N = t.N;
    return t.det[g] * (t.minv[(2 * k) * N + g] * u + t.minv[(2 * k + 1) * N + g] * v);
}
X3_HD float x3_bflux(const fgb_tables &t, int j, int ax, float bu, float bv) {
    const int NB = t.NB;
    return t.b_det[j] * (t.b_minv[(2 * ax) * NB + j] * bu + t.b_minv[(2 * ax + 1) * NB + j] * bv);
}
// in-plane face fluxes / hz of plane-local fields ux, uy [N2] (K.cu:1567-1645)
X3_HD void x3_face_fluxes(const fgb_tables &t, int g, const float *ux, const float *uy, const float *bx, const float *by,
                          const int nb[4], float fl[4]) {
    const int N = t.N;
    const float Uc[2] = {x3_contra(t, 0, g, ux[g], uy[g]), x3_contra(t, 1, g, ux[g], uy[g])};
    for (int f = 0; f < 4; ++f) {
        if (nb[f] >= 0) {
            const int fc = t.fl_comp[f * N + g];
            float velN = x3_contra(t, fc & 1, nb[f], ux[nb[f]], uy[nb[f]]);
            if (fc & 2) velN = -velN;
            fl[f] = (velN + Uc[f >> 1]) * 0.5f;
        } else {
            const int j = -1 - nb[f];
            fl[f] = x3_bflux(t, j, f >> 1, bx[j], by[j]);
        }
    }
}
// Dirichlet boundary advection + diffusion source of component values bc [NB2] (K.cu:4321-4380), before / det
X3_HD float x3_boundary_source(const fgb_tables &t, const float *bx, const float *by, const float *bc, const int nb[4]) {
    float S = 0.f;
    for (int f = 0; f < 4; ++f)
        if (nb[f] < 0) {
            const int j = -1 - nb[f];
            const float flux = x3_bflux(t, j, f >> 1, bx[j], by[j]) * ((f & 1) ? 1.f : -1.f);
            S -= bc[j] * flux;
            S += bc[j] * (t.viscosity * 2.f * t.b_alpha[j]);
        }
    return S;
}

// SetupAdvectionMatrix + SetupAdvectionVelocity (K.cu:3617-3880, 4296-4400) for cell (k, g) of one environment.
// u, ures: [3][N3]; bvel: [3][nz][NB2]; outputs coff [6][N3], A [N3], rhs [3][N3]
X3_HD void x3_setup_advection_cell(const X3Tab &x, int k, int g, const float *u, const float *ures, const float *bvel, float dt,
                                   float *coff, float *A, float *rhs, int with_matrix) {
    const fgb_tables &t = x.t;
    const int N = t.N, NB = t.NB, nz = x.nz, N3 = N * nz, g3 = k * N + g;
    const float det = t.det[g], hz = x.hz;
    const float *ux = u + (size_t)k * N, *uy = u + (size_t)N3 + (size_t)k * N, *uz = u + 2 * (size_t)N3;
    const float *bx = bvel + (size_t)k * NB, *by = bvel + (size_t)nz * NB + (size_t)k * NB;
    int nb[4];
    for (int f = 0; f < 4; ++f) nb[f] = t.nbr[f * N + g];
    if (with_matrix) {
        float fl[4];
        x3_face_fluxes(t, g, ux, uy, bx, by, nb, fl);
        float diag = det / dt + t.Cd[g];
        for (int f = 0; f < 4; ++f) {
            float o = 0.f;
            if (nb[f] >= 0) {
                const float ff = ((f & 1) ? 0.5f : -0.5f) * fl[f];
                diag += ff;
                o = (ff + t.Cd[(f + 1) * N + g]) / det;
            }
            coff[(size_t)f * N3 + g3] = o;
        }
        const int kl = (k + nz - 1) % nz, ku = (k + 1) % nz;
        const float uzP = uz[g3], Fzm = 0.5f * (uzP + uz[(size_t)kl * N + g]), Fzp = 0.5f * (uzP + uz[(size_t)ku * N + g]);
        const float dz = t.viscosity / (hz * hz);
        coff[(size_t)4 * N3 + g3] = (-0.5f * Fzm) / hz - dz;
        coff[(size_t)5 * N3 + g3] = (0.5f * Fzp) / hz - dz;
        A[g3] = diag / det + 2.f * dz + 0.5f * (Fzp - Fzm) / hz;
    }
    for (int c = 0; c < 3; ++c) {
        const float *bc = bvel + ((size_t)c * nz + k) * NB;
        const float *ur = ures + (size_t)c * N3 + (size_t)k * N;
        const float S = x3_boundary_source(t, bx, by, bc, nb);
        float no = 0.f;
        for (int q = 0; q < t.K_no; ++q) {
            const float w = t.no_wv[q * N + g];
            if (w != 0.f) no += w * ur[t.no_idx[q * N + g]];
        }
        for (int q = 0; q < t.K_nob; ++q) {
            const float w = t.nob_w[q * N + g];
            if (w != 0.f) no += w * bc[t.nob_idx[q * N + g]];
        }
        rhs[(size_t)c * N3 + g3] = (det * u[(size_t)c * N3 + g3] / dt + S - no) / det;
    }
}

// SetupPressureMatrix (K.cu:4812-4978), NOT divided by det: in-plane  hz * sum_j Wp[e][j] (1/A)_j , z faces 1/2 (det2 / hz) (1/A_P + 1/A_N)
X3_HD void x3_pressure_matrix_cell(const X3Tab &x, int k, int g, const float *A, float *poff, float *pdiag) {
    const fgb_tables &t = x.t;
    const int N = t.N, nz = x.nz, N3 = N * nz, g3 = k * N + g;
    const float *a = A + (size_t)k * N;
    float rA[5];
    rA[0] = 1.0f / a[g];
    for (int f = 0; f < 4; ++f) { const int nb = t.nbr[f * N + g]; rA[f + 1] = nb >= 0 ? 1.0f / a[nb] : rA[0]; }
    float P[5];
    for (int e = 0; e < 5; ++e) {
        float s = 0.f;
        for (int j = 0; j < 5; ++j) s += t.Wp[(5 * e + j) * N + g] * rA[j];
        P[e] = s * x.hz;
    }
    const int kl = (k + nz - 1) % nz, ku = (k + 1) % nz;
    const float az = t.det[g] / x.hz;
    const float pl = 0.5f * az * (rA[0] + 1.0f / A[(size_t)kl * N + g]), pu = 0.5f * az * (rA[0] + 1.0f / A[(size_t)ku * N + g]);
    for (int f = 0; f < 4; ++f) poff[(size_t)f * N3 + g3] = P[f + 1];
    poff[(size_t)4 * N3 + g3] = pl;
    poff[(size_t)5 * N3 + g3] = pu;
    pdiag[g3] = P[0] - pl - pu;
}

// PISO_build_pressure_rhs (K.cu:5136-5255): HbyA = (u/dt - sum_nb C_nb u*_nb + S_b/det) / A for the three components
X3_HD void x3_hbya_cell(const X3Tab &x, int k, int g, const float *u, const float *ures, const float *bvel, const float *coff,
                        const float *A, float dt, float *hb) {
    const fgb_tables &t = x.t;
    const int N = t.N, NB = t.NB, nz = x.nz, N3 = N * nz, g3 = k * N + g;
    const float *bx = bvel + (size_t)k * NB, *by = bvel + (size_t)nz * NB + (size_t)k * NB;
    const int kl = (k + nz - 1) % nz, ku = (k + 1) % nz;
    int nb[4];
    for (int f = 0; f < 4; ++f) nb[f] = t.nbr[f * N + g];
    const float rD = 1.0f / A[g3], det = t.det[g];
    for (int c = 0; c < 3; ++c) {
        const float *ur = ures + (size_t)c * N3;
        float H = 0.f;
        for (int f = 0; f < 4; ++f)
            if (nb[f] >= 0) H += coff[(size_t)f * N3 + g3] * ur[(size_t)k * N + nb[f]];
        H += coff[(size_t)4 * N3 + g3] * ur[(size_t)kl * N + g] + coff[(size_t)5 * N3 + g3] * ur[(size_t)ku * N + g];
        const float S = x3_boundary_source(t, bx, by, bvel + ((size_t)c * nz + k) * NB, nb);
        hb[(size_t)c * N3 + g3] = rD * (u[(size_t)c * N3 + g3] / dt - H + S / det);
    }
}

// divergence of the face fluxes of HbyA (K.cu:5389-5434) + deferred non-orthogonal pressure term (K.cu:5470-5492)
X3_HD void x3_divergence_cell(const X3Tab &x, int k, int g, const float *hb, const float *bvel, const float *pprev /* or null */,
                              const float *A, float *div) {
    const fgb_tables &t = x.t;
    const int N = t.N, NB = t.NB, nz = x.nz, N3 = N * nz, g3 = k * N + g;
    const float *hx = hb + (size_t)k * N, *hy = hb + (size_t)N3 + (size_t)k * N, *hzc = hb + 2 * (size_t)N3;
    const float *bx = bvel + (size_t)k * NB, *by = bvel + (size_t)nz * NB + (size_t)k * NB;
    int nb[4];
    for (int f = 0; f < 4; ++f) nb[f] = t.nbr[f * N + g];
    float fl[4];
    x3_face_fluxes(t, g, hx, hy, bx, by, nb, fl);
    float d = (fl[1] - fl[0]) + (fl[3] - fl[2]);
    if (pprev) {
        const float *a = A + (size_t)k * N, *pp = pprev + (size_t)k * N;
        float rA[5];
        rA[0] = 1.0f / a[g];
        for (int f = 0; f < 4; ++f) rA[f + 1] = nb[f] >= 0 ? 1.0f / a[nb[f]] : rA[0];
        float S = 0.f;
        for (int q = 0; q < t.K_no; ++q) {
            const float gP = t.no_gP[q * N + g], gN = t.no_gN[q * N + g];
            if (gP != 0.f || gN != 0.f) S += (gP * rA[0] + gN * rA[1 + t.no_face[q * N + g]]) * pp[t.no_idx[q * N + g]];
        }
        d += S;
    }
    const int kl = (k + nz - 1) % nz, ku = (k + 1) % nz;
    const float hP = hzc[g3];
    div[g3] = d * x.hz + t.det[g] * (0.5f * (hP + hzc[(size_t)ku * N + g]) - 0.5f * (hP + hzc[(size_t)kl * N + g]));
}

// PISO_update_velocity (K.cu:816-849, 5962-5995)
X3_HD void x3_correct_cell(const X3Tab &x, int k, int g, const float *hb, const float *p, const float *A, float *uout) {
    const fgb_tables &t = x.t;
    const int N = t.N, nz = x.nz, N3 = N * nz, g3 = k * N + g;
    const float *pk = p + (size_t)k * N;
    const float pc = pk[g];
    float pg[2];
    for (int d = 0; d < 2; ++d) {
        const int nl = t.nbr[(2 * d) * N + g], nu = t.nbr[(2 * d + 1) * N + g];
        const float fac = (nl < 0 || nu < 0) ? 1.0f : 0.5f;
        pg[d] = ((nu >= 0 ? pk[nu] : pc) - (nl >= 0 ? pk[nl] : pc)) * fac;
    }
    const float gx = pg[0] * t.minv[g] + pg[1] * t.minv[2 * N + g];
    const float gy = pg[0] * t.minv[N + g] + pg[1] * t.minv[3 * N + g];
    const int kl = (k + nz - 1) % nz, ku = (k + 1) % nz;
    const float gz = 0.5f * (p[(size_t)ku * N + g] - p[(size_t)kl * N + g]) / x.hz;
    const float rD = 1.0f / A[g3];
    uout[g3] = hb[g3] - rD * gx;
    uout[(size_t)N3 + g3] = hb[(size_t)N3 + g3] - rD * gy;
    uout[2 * (size_t)N3 + g3] = hb[2 * (size_t)N3 + g3] - rD * gz;
}

#ifdef __CUDACC__
#ifndef X3_HOST_ONLY
// ------------------------------------------------------------------------------------------------------------------
// launch glue (one thread per (cell, plane, environment)); matrices / vectors live in the workspace of an fgb_ortho3
// handle created on the 6-face neighbour table of the extruded domain, so fgb_ortho3_solve_advection / _solve_pressure
// run the Krylov iterations.
// ------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) kx3_setup_advection(X3Tab x, const float *U, const float *Ures, const float *Bvel, const float *dtv,
                                                          float *Coff, float *A, float *Rhs, int with_matrix, const int32_t *active) {
    const int b = blockIdx.z, k = blockIdx.y, g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= x.t.N || (active && !active[b])) return;
    const size_t N3 = (size_t)x.t.N * x.nz;
    x3_setup_advection_cell(x, k, g, U + b * 3 * N3, Ures + b * 3 * N3, Bvel + (size_t)b * 3 * x.nz * x.t.NB, dtv[b], Coff + b * 6 * N3,
                            A + b * N3, Rhs + b * 3 * N3, with_matrix);
}
__global__ void __launch_bounds__(256) kx3_pressure_matrix(X3Tab x, const float *A, float *Poff, float *Pdiag, const int32_t *active) {
    const int b = blockIdx.z, k = blockIdx.y, g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= x.t.N || (active && !active[b])) return;
    const size_t N3 = (size_t)x.t.N * x.nz;
    x3_pressure_matrix_cell(x, k, g, A + b * N3, Poff + b * 6 * N3, Pdiag + b * N3);
}
__global__ void __launch_bounds__(256) kx3_hbya(X3Tab x, const float *U, const float *Ures, const float *Bvel, const float *Coff, const float *A,
                                               const float *dtv, float *Hb, const int32_t *active) {
    const int b = blockIdx.z, k = blockIdx.y, g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= x.t.N || (active && !active[b])) return;
    const size_t N3 = (size_t)x.t.N * x.nz;
    x3_hbya_cell(x, k, g, U + b * 3 * N3, Ures + b * 3 * N3, Bvel + (size_t)b * 3 * x.nz * x.t.NB, Coff + b * 6 * N3, A + b * N3, dtv[b], Hb + b * 3 * N3);
}
__global__ void __launch_bounds__(256) kx3_divergence(X3Tab x, const float *Hb, const float *Bvel, const float *Pprev, const float *A, float *Div, const int32_t *active) {
    const int b = blockIdx.z, k = blockIdx.y, g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= x.t.N || (active && !active[b])) return;
    const size_t N3 = (size_t)x.t.N * x.nz;
    x3_divergence_cell(x, k, g, Hb + b * 3 * N3, Bvel + (size_t)b * 3 * x.nz * x.t.NB, Pprev ? Pprev + b * N3 : nullptr, A + b * N3, Div + b * N3);
}
__global__ void __launch_bounds__(256) kx3_correct(X3Tab x, const float *Hb, const float *P, const float *A, float *Uout, const int32_t *active) {
    const int b = blockIdx.z, k = blockIdx.y, g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= x.t.N || (active && !active[b])) return;
    const size_t N3 = (size_t)x.t.N * x.nz;
    x3_correct_cell(x, k, g, Hb + b * 3 * N3, P + b * N3, A + b * N3, Uout + b * 3 * N3);
}

// Simulation._PISO_split_step on an extruded domain (SIM.py:1431-2002, non-orthogonal path): b = fgb_ortho3 handle created on
// the 6-face table (N = nz * N2); opt.adv_nonortho_steps / p_nonortho_steps deferred-correction iterations.
extern "C" int fgb_extruded3_piso_substep(fgb_ortho3 *b, const fgb_extruded3_tables *xt, float *u, float *p, const float *bvel, const float *dt,
                                          fgb_stream_t s) {
    if (!b || !xt || !u || !p || !bvel || !dt) return set_err(FGB_E_ARG, "fgb_extruded3_piso_substep: null argument");
    if (b->t.N != xt->plane.N * xt->nz || b->slab.on) return set_err(FGB_E_ARG, "fgb_extruded3_piso_substep: handle / tables mismatch");
    X3Tab x; x.t = xt->plane; x.nz = xt->nz; x.hz = xt->hz;
    cudaStream_t st = STREAM(s);
    const dim3 grid((unsigned)((x.t.N + 255) / 256), (unsigned)x.nz, (unsigned)b->B);
    const fgb_options &o = b->opt;
    int rc;
    for (int ns = 0; ns < o.adv_nonortho_steps; ++ns) {
        b->launches++;
        kx3_setup_advection<<<grid, 256, 0, st>>>(x, u, ns == 0 ? u : b->ures, bvel, dt, b->Coff, b->A, b->rhs, ns == 0, nullptr);
        LAUNCH_CHECK("kx3_setup_advection");
        if ((rc = fgb_ortho3_solve_advection(b, ns == 0, nullptr, s))) return rc;
    }
    for (int cs = 0; cs < o.corrector_steps; ++cs) {
        b->launches += 2;
        if (cs == 0) { kx3_pressure_matrix<<<grid, 256, 0, st>>>(x, b->A, b->Poff, b->Pdiag, nullptr); LAUNCH_CHECK("kx3_pressure_matrix"); }
        kx3_hbya<<<grid, 256, 0, st>>>(x, u, b->ures, bvel, b->Coff, b->A, dt, b->hbya, nullptr);
        LAUNCH_CHECK("kx3_hbya");
        for (int ps = 0; ps < o.p_nonortho_steps; ++ps) {
            b->launches++;
            kx3_divergence<<<grid, 256, 0, st>>>(x, b->hbya, bvel, p, b->A, b->div, nullptr);
            LAUNCH_CHECK("kx3_divergence");
            if ((rc = fgb_ortho3_solve_pressure(b, p, ps == 0, 100, o.max_iter, cs * o.p_nonortho_steps + ps, nullptr, s))) return rc;
        }
        b->launches++;
        kx3_correct<<<grid, 256, 0, st>>>(x, b->hbya, p, b->A, b->ures, nullptr);
        LAUNCH_CHECK("kx3_correct");
    }
    cudaError_t ce = cudaMemcpyAsync(u, b->ures, (size_t)b->B * 3 * b->t.N * sizeof(float), cudaMemcpyDeviceToDevice, st);
    if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "fgb_extruded3_piso_substep: copy", ce);
    return FGB_OK;
}


// ------------------------------------------------------------------------------------------------------------------
// Reverse mode of the extruded substep (CylinderJet3D / Airfoil3D with differentiable=True).  Same construction as the 2-D adjoint
// (piso_b200.cu: k_adj_*, whose in-plane terms these kernels repeat per plane on the same tables) plus the z faces; the transposed
// Krylov solves run in k3_bicgstab / k3_cg<1> with the plane's reverse-face table (fgb_ortho3_tables.rev).  The recorded forward pass
// follows the reference's differentiable backend: every solve starts from zero, the CG never resets its residual.
// Tape = fgb_tape with three components: u_in / ustar / hb / u1 [..][B][3][N3], Coff [B][6][N3], bvel_in [B][3][nz][NB2].
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void x3_fluxes_adjoint(const fgb_tables &t, int g, const int nb[4], const float flb[4], float *__restrict__ vbx,
                                                  float *__restrict__ vby /* plane-local [N2] */, float *__restrict__ Fbb /* plane-local [NB2] or null */) {
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
            atomicAdd(&vbx[n], w * t.minv[(2 * cn) * N + n]);
            atomicAdd(&vby[n], w * t.minv[(2 * cn + 1) * N + n]);
        } else if (Fbb) {
            atomicAdd(&Fbb[-1 - nb[f]], flb[f]);
        }
    }
    const float d = t.det[g];
    atomicAdd(&vbx[g], d * (t.minv[g] * Ub[0] + t.minv[2 * N + g] * Ub[1]));
    atomicAdd(&vby[g], d * (t.minv[N + g] * Ub[0] + t.minv[3 * N + g] * Ub[1]));
}
#define X3_ADJ_PROLOGUE \
    const int b = blockIdx.z, k = blockIdx.y, g = blockIdx.x * blockDim.x + threadIdx.x; \
    const fgb_tables &t = x.t; \
    const int N = t.N, nz = x.nz; \
    if (g >= N || (active && !active[b])) return;    /* skipped environment: identity cotangents from k_adj_inactive */ \
    const size_t N3 = (size_t)N * nz, g3 = (size_t)k * N + g; \
    const int kl = (k + nz - 1) % nz, ku = (k + 1) % nz; \
    (void)kl; (void)ku; (void)N3; (void)g3;

__global__ void __launch_bounds__(256) kx3_adj_correct(X3Tab x, const float *__restrict__ Unb, const float *__restrict__ P, const float *__restrict__ A,
                                                       float *__restrict__ Hbb, float *__restrict__ rAb, float *__restrict__ Pb,
                                                       const int32_t *__restrict__ active) {
    X3_ADJ_PROLOGUE
    const float *p = P + b * N3, *pk = p + (size_t)k * N;
    float *pb = Pb + b * N3, *pbk = pb + (size_t)k * N;
    const float ub0 = Unb[b * 3 * N3 + g3], ub1 = Unb[b * 3 * N3 + N3 + g3], ub2 = Unb[b * 3 * N3 + 2 * N3 + g3];
    Hbb[b * 3 * N3 + g3] = ub0; Hbb[b * 3 * N3 + N3 + g3] = ub1; Hbb[b * 3 * N3 + 2 * N3 + g3] = ub2;
    const float rA = 1.0f / A[b * N3 + g3], pc = pk[g];
    float pg[2], fac[2]; int nl[2], nu[2];
#pragma unroll
    for (int d = 0; d < 2; ++d) {
        nl[d] = t.nbr[(2 * d) * N + g]; nu[d] = t.nbr[(2 * d + 1) * N + g];
        fac[d] = (nl[d] < 0 || nu[d] < 0) ? 1.0f : 0.5f;
        pg[d] = ((nu[d] >= 0 ? pk[nu[d]] : pc) - (nl[d] >= 0 ? pk[nl[d]] : pc)) * fac[d];
    }
    const float m00 = t.minv[g], m01 = t.minv[N + g], m10 = t.minv[2 * N + g], m11 = t.minv[3 * N + g];
    const float gx = pg[0] * m00 + pg[1] * m10, gy = pg[0] * m01 + pg[1] * m11;
    const float gz = 0.5f * (p[(size_t)ku * N + g] - p[(size_t)kl * N + g]) / x.hz;
    atomicAdd(&rAb[b * N3 + g3], -(gx * ub0 + gy * ub1 + gz * ub2));
    const float gb0 = -rA * ub0, gb1 = -rA * ub1;
    const float pgb[2] = {gb0 * m00 + gb1 * m01, gb0 * m10 + gb1 * m11};
#pragma unroll
    for (int d = 0; d < 2; ++d) {
        const float w = pgb[d] * fac[d];
        atomicAdd(&pbk[nu[d] >= 0 ? nu[d] : g], w);
        atomicAdd(&pbk[nl[d] >= 0 ? nl[d] : g], -w);
    }
    const float wz = -rA * ub2 * 0.5f / x.hz;
    atomicAdd(&pb[(size_t)ku * N + g], wz);
    atomicAdd(&pb[(size_t)kl * N + g], -wz);
}
// adjoint of  div = hz (fluxdiv2(hb) + NOp(p_prev, rA)) + det2 D_z(hb_z)  and of  x = P^-1 div  w.r.t. P(rA):  given lam = P^-T x_bar
__global__ void __launch_bounds__(256) kx3_adj_pressure_rhs(X3Tab x, const float *__restrict__ Lam, const float *__restrict__ Pm, const float *__restrict__ Pmean,
                                                            const float *__restrict__ Pprev, const float *__restrict__ A, float *__restrict__ Hbb,
                                                            float *__restrict__ Fbb, float *__restrict__ rAb, float *__restrict__ Pprevb,
                                                            const int32_t *__restrict__ active) {
    X3_ADJ_PROLOGUE
    const int NB = t.NB;
    const float hz = x.hz, lam = Lam[b * N3 + g3], mean = Pmean[b];
    const float *px = Pm + b * N3, *pxk = px + (size_t)k * N;
    const float *a = A + b * N3, *ak = a + (size_t)k * N, *pp = Pprev + b * N3 + (size_t)k * N;
    float *ra = rAb + b * N3, *rak = ra + (size_t)k * N;
    int nb[4];
#pragma unroll
    for (int f = 0; f < 4; ++f) nb[f] = t.nbr[f * N + g];
    float Pb[5];
    Pb[0] = -lam * (pxk[g] + mean);
#pragma unroll
    for (int f = 0; f < 4; ++f) Pb[f + 1] = nb[f] >= 0 ? -lam * (pxk[nb[f]] + mean) : 0.f;
    float rb[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int e = 0; e < 5; ++e)
#pragma unroll
        for (int j = 0; j < 5; ++j) rb[j] += hz * t.Wp[(5 * e + j) * N + g] * Pb[e];
    float rA[5];
    rA[0] = 1.0f / ak[g];
#pragma unroll
    for (int f = 0; f < 4; ++f) rA[f + 1] = nb[f] >= 0 ? 1.0f / ak[nb[f]] : rA[0];
    for (int q = 0; q < t.K_no; ++q) {
        const float gP = t.no_gP[q * N + g], gN = t.no_gN[q * N + g];
        if (gP != 0.f || gN != 0.f) {
            const int fc = t.no_face[q * N + g], j = t.no_idx[q * N + g];
            const float wb = lam * hz * pp[j];
            rb[0] += gP * wb; rb[1 + fc] += gN * wb;
            atomicAdd(&Pprevb[b * N3 + (size_t)k * N + j], (gP * rA[0] + gN * rA[1 + fc]) * lam * hz);
        }
    }
    // z faces of the matrix: pl = 1/2 (det2 / hz) (rA_P + rA_lower), pdiag -= pl (same for the upper face)
    const float az = 0.5f * t.det[g] / hz;
    const float wl = (-lam * (px[(size_t)kl * N + g] + mean) - Pb[0]) * az, wu = (-lam * (px[(size_t)ku * N + g] + mean) - Pb[0]) * az;
    atomicAdd(&rak[g], rb[0] + wl + wu);
    atomicAdd(&ra[(size_t)kl * N + g], wl);
    atomicAdd(&ra[(size_t)ku * N + g], wu);
#pragma unroll
    for (int f = 0; f < 4; ++f) atomicAdd(&rak[nb[f] >= 0 ? nb[f] : g], rb[f + 1]);
    const float flb[4] = {-lam * hz, lam * hz, -lam * hz, lam * hz};
    float *hbb = Hbb + b * 3 * N3;
    x3_fluxes_adjoint(t, g, nb, flb, hbb + (size_t)k * N, hbb + N3 + (size_t)k * N, Fbb + ((size_t)b * nz + k) * NB);
    const float wzf = 0.5f * t.det[g] * lam;
    atomicAdd(&hbb[2 * N3 + (size_t)ku * N + g], wzf);
    atomicAdd(&hbb[2 * N3 + (size_t)kl * N + g], -wzf);
}
// adjoint of  hb = rA (u/dt - H + Sb/det2),  H_c = sum_f Coff_f uprev_c[nb_f]  (6 faces)
__global__ void __launch_bounds__(256) kx3_adj_hbya(X3Tab x, const float *__restrict__ Hbb, const float *__restrict__ Hb, const float *__restrict__ A,
                                                    const float *__restrict__ Coff, const float *__restrict__ Uprev, const float *__restrict__ dtv,
                                                    float *__restrict__ rAb, float *__restrict__ Ub, float *__restrict__ Sbb, float *__restrict__ Coffb,
                                                    float *__restrict__ Uprevb, const int32_t *__restrict__ active) {
    X3_ADJ_PROLOGUE
    const float dt = dtv[b], Ag = A[b * N3 + g3], rA = 1.0f / Ag, det = t.det[g];
    const float *coff = Coff + b * 6 * N3;
    float *coffb = Coffb + b * 6 * N3;
    int nb[4];
#pragma unroll
    for (int f = 0; f < 4; ++f) nb[f] = t.nbr[f * N + g];
    float accr = 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const size_t o = b * 3 * N3 + (size_t)c * N3;
        const float hbb = Hbb[o + g3];
        accr += hbb * (Hb[o + g3] * Ag);
        const float ib = rA * hbb;
        atomicAdd(&Ub[o + g3], ib / dt);
        Sbb[o + g3] += ib / det;
#pragma unroll
        for (int f = 0; f < 4; ++f)
            if (nb[f] >= 0) {
                coffb[(size_t)f * N3 + g3] += -ib * Uprev[o + (size_t)k * N + nb[f]];
                atomicAdd(&Uprevb[o + (size_t)k * N + nb[f]], -ib * coff[(size_t)f * N3 + g3]);
            }
        coffb[4 * N3 + g3] += -ib * Uprev[o + (size_t)kl * N + g];
        atomicAdd(&Uprevb[o + (size_t)kl * N + g], -ib * coff[4 * N3 + g3]);
        coffb[5 * N3 + g3] += -ib * Uprev[o + (size_t)ku * N + g];
        atomicAdd(&Uprevb[o + (size_t)ku * N + g], -ib * coff[5 * N3 + g3]);
    }
    atomicAdd(&rAb[b * N3 + g3], accr);
}
// adjoint of one predictor iteration  C x = rhs(u, x_prev):  given mu = C^-T x_bar
__global__ void __launch_bounds__(256) kx3_adj_advection(X3Tab x, const float *__restrict__ Mu, const float *__restrict__ X, const float *__restrict__ rAb,
                                                         const float *__restrict__ A, const float *__restrict__ dtv, float *__restrict__ Ab,
                                                         float *__restrict__ Coffb, float *__restrict__ Ub, float *__restrict__ Sbb, float *__restrict__ Bvb,
                                                         float *__restrict__ NoTarget, int first, const int32_t *__restrict__ active) {
    X3_ADJ_PROLOGUE
    const int NB = t.NB;
    const float dt = dtv[b], det = t.det[g], Ag = A[b * N3 + g3];
    float *coffb = Coffb + b * 6 * N3;
    int nb[4];
#pragma unroll
    for (int f = 0; f < 4; ++f) nb[f] = t.nbr[f * N + g];
    float ab = first ? -rAb[b * N3 + g3] / (Ag * Ag) : Ab[b * N3 + g3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const size_t o = b * 3 * N3 + (size_t)c * N3;
        const float mu = Mu[o + g3];
        ab += -mu * X[o + g3];
#pragma unroll
        for (int f = 0; f < 4; ++f) if (nb[f] >= 0) coffb[(size_t)f * N3 + g3] += -mu * X[o + (size_t)k * N + nb[f]];
        coffb[4 * N3 + g3] += -mu * X[o + (size_t)kl * N + g];
        coffb[5 * N3 + g3] += -mu * X[o + (size_t)ku * N + g];
        atomicAdd(&Ub[o + g3], mu / dt);
        Sbb[o + g3] += mu / det;
        const float nob = -mu / det;
        for (int q = 0; q < t.K_no; ++q) { const float w = t.no_wv[q * N + g]; if (w != 0.f) atomicAdd(&NoTarget[o + (size_t)k * N + t.no_idx[q * N + g]], w * nob); }
        for (int q = 0; q < t.K_nob; ++q) {
            const float w = t.nob_w[q * N + g];
            if (w != 0.f) atomicAdd(&Bvb[((size_t)b * 3 + c) * nz * NB + (size_t)k * NB + t.nob_idx[q * N + g]], w * nob);
        }
    }
    Ab[b * N3 + g3] = ab;
}
// adjoint of the assembly (A, Coff from the in-plane face fluxes and the z fluxes) and of the boundary sources
__global__ void __launch_bounds__(256) kx3_adj_assemble(X3Tab x, const float *__restrict__ Ab, const float *__restrict__ Coffb, const float *__restrict__ Sbb,
                                                        const float *__restrict__ Bvel, float *__restrict__ Ub, float *__restrict__ Bvb, float *__restrict__ Fbb,
                                                        const int32_t *__restrict__ active) {
    X3_ADJ_PROLOGUE
    const int NB = t.NB;
    const float det = t.det[g], ab = Ab[b * N3 + g3], diagb = ab / det, hz = x.hz;
    const float *bvel = Bvel + (size_t)b * 3 * nz * NB;
    const float *bx = bvel + (size_t)k * NB, *by = bvel + (size_t)nz * NB + (size_t)k * NB;
    const float *coffb = Coffb + b * 6 * N3;
    int nb[4]; float flb[4];
#pragma unroll
    for (int f = 0; f < 4; ++f) {
        nb[f] = t.nbr[f * N + g];
        const float sig = (f & 1) ? 1.f : -1.f;
        flb[f] = 0.f;
        if (nb[f] >= 0) flb[f] = 0.5f * sig * (coffb[(size_t)f * N3 + g3] / det + diagb);
        else {
            const int j = -1 - nb[f];
            const float kk = -(sig * x3_bflux(t, j, f >> 1, bx[j], by[j])) + 2.f * t.viscosity * t.b_alpha[j];
            float dot = 0.f;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float sb = Sbb[b * 3 * N3 + (size_t)c * N3 + g3];
                atomicAdd(&Bvb[((size_t)b * 3 + c) * nz * NB + (size_t)k * NB + j], sb * kk);
                dot += sb * bvel[((size_t)c * nz + k) * NB + j];
            }
            atomicAdd(&Fbb[((size_t)b * nz + k) * NB + j], -dot * sig);
        }
    }
    float *ub = Ub + b * 3 * N3;
    x3_fluxes_adjoint(t, g, nb, flb, ub + (size_t)k * N, ub + N3 + (size_t)k * N, nullptr);
    // z faces: coff4 = -1/2 Fzm / hz - dz, coff5 = 1/2 Fzp / hz - dz, A += 1/2 (Fzp - Fzm) / hz, Fzm = 1/2 (w_P + w_lower)
    const float fzm = (-0.5f / hz) * (coffb[4 * N3 + g3] + ab), fzp = (0.5f / hz) * (coffb[5 * N3 + g3] + ab);
    atomicAdd(&ub[2 * N3 + g3], 0.5f * (fzm + fzp));
    atomicAdd(&ub[2 * N3 + (size_t)kl * N + g], 0.5f * fzm);
    atomicAdd(&ub[2 * N3 + (size_t)ku * N + g], 0.5f * fzp);
}
// adjoint of the in-plane boundary flux Fb(bx, by): one thread per (boundary face, plane, environment)
__global__ void kx3_adj_bflux(X3Tab x, const float *__restrict__ Fbb, float *__restrict__ Bvb, const int32_t *__restrict__ active) {
    const int b = blockIdx.z, k = blockIdx.y, j = blockIdx.x * blockDim.x + threadIdx.x;
    const fgb_tables &t = x.t;
    const int NB = t.NB, nz = x.nz;
    if (j >= NB || (active && !active[b])) return;
    const int ax = t.b_face[j] >> 1;
    const float f = Fbb[((size_t)b * nz + k) * NB + j] * t.b_det[j];
    Bvb[((size_t)b * 3 + 0) * nz * NB + (size_t)k * NB + j] += f * t.b_minv[(2 * ax) * NB + j];
    Bvb[((size_t)b * 3 + 1) * nz * NB + (size_t)k * NB + j] += f * t.b_minv[(2 * ax + 1) * NB + j];
}
__global__ void kx3_take_mean(int B, const float *__restrict__ pmean8, int slot, float *__restrict__ out) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < B) out[b] = pmean8[b * 8 + 3 + slot];
}

static int x3_copy(void *dst, const void *src, size_t bytes, cudaStream_t st) {
    cudaError_t ce = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, st);
    return ce == cudaSuccess ? FGB_OK : set_err(FGB_E_CUDA, "cudaMemcpyAsync (extruded tape)", ce);
}
// fgb_extruded3_piso_substep that additionally records the tape of the backward pass (zero-started solves, no CG residual reset), for the
// environments of tp->active (NULL: all); a skipped environment keeps u and p bit for bit
extern "C" int fgb_extruded3_piso_substep_record(fgb_ortho3 *b, const fgb_extruded3_tables *xt, float *u, float *p, const float *bvel, const float *dt,
                                                 const fgb_tape *tp, fgb_stream_t s) {
    if (!b || !xt || !u || !p || !bvel || !dt || !tp) return set_err(FGB_E_ARG, "fgb_extruded3_piso_substep_record: null argument");
    if (b->t.N != xt->plane.N * xt->nz || b->slab.on) return set_err(FGB_E_ARG, "fgb_extruded3_piso_substep_record: handle / tables mismatch");
    const fgb_options &o = b->opt;
    const int C = o.corrector_steps, n_adv = o.adv_nonortho_steps, n_p = o.p_nonortho_steps;
    if (C < 1 || n_adv < 1 || n_p < 1 || C * n_p > 8) return set_err(FGB_E_ARG, "fgb_extruded3_piso_substep_record: correctors x pressure iterations <= 8");
    X3Tab x; x.t = xt->plane; x.nz = xt->nz; x.hz = xt->hz;
    cudaStream_t st = STREAM(s);
    const dim3 grid((unsigned)((x.t.N + 255) / 256), (unsigned)x.nz, (unsigned)b->B);
    const size_t B = b->B, BN = B * b->t.N, BNB = B * (size_t)x.nz * (x.t.NB > 0 ? x.t.NB : 1);
    const int32_t *act = tp->active;
    int rc;
    if ((rc = x3_copy(tp->u_in, u, 3 * BN * 4, st))) return rc;
    if ((rc = x3_copy(tp->p_in, p, BN * 4, st))) return rc;
    if ((rc = x3_copy(tp->bvel_in, bvel, 3 * BNB * 4, st))) return rc;
    if ((rc = x3_copy(tp->dt, dt, B * 4, st))) return rc;
    for (int ns = 0; ns < n_adv; ++ns) {
        b->launches++;
        kx3_setup_advection<<<grid, 256, 0, st>>>(x, u, ns == 0 ? u : b->ures, bvel, dt, b->Coff, b->A, b->rhs, ns == 0, act);
        LAUNCH_CHECK("kx3_setup_advection");
        if ((rc = fgb_ortho3_solve_advection(b, 1, act, s))) return rc;
        if ((rc = x3_copy(tp->ustar + (size_t)ns * 3 * BN, b->ures, 3 * BN * 4, st))) return rc;
    }
    if ((rc = x3_copy(tp->Coff, b->Coff, 6 * BN * 4, st))) return rc;
    if ((rc = x3_copy(tp->A, b->A, BN * 4, st))) return rc;
    b->launches++;
    kx3_pressure_matrix<<<grid, 256, 0, st>>>(x, b->A, b->Poff, b->Pdiag, act);
    LAUNCH_CHECK("kx3_pressure_matrix");
    for (int cs = 0; cs < C; ++cs) {
        b->launches++;
        kx3_hbya<<<grid, 256, 0, st>>>(x, u, b->ures, bvel, b->Coff, b->A, dt, b->hbya, act);
        LAUNCH_CHECK("kx3_hbya");
        for (int ps = 0; ps < n_p; ++ps) {
            const int q = cs * n_p + ps, slot = q > 4 ? 4 : q;
            b->launches += 2;
            kx3_divergence<<<grid, 256, 0, st>>>(x, b->hbya, bvel, p, b->A, b->div, act);
            LAUNCH_CHECK("kx3_divergence");
            if ((rc = fgb_ortho3_solve_pressure(b, p, 1, 0, o.max_iter, slot, act, s))) return rc;
            if ((rc = x3_copy(tp->p + (size_t)q * BN, p, BN * 4, st))) return rc;
            kx3_take_mean<<<(unsigned)((B + 127) / 128), 128, 0, st>>>((int)B, b->pmean, slot, tp->pmean + (size_t)q * B);
            LAUNCH_CHECK("kx3_take_mean");
        }
        if ((rc = x3_copy(tp->hb + (size_t)cs * 3 * BN, b->hbya, 3 * BN * 4, st))) return rc;
        b->launches++;
        kx3_correct<<<grid, 256, 0, st>>>(x, b->hbya, p, b->A, b->ures, act);
        LAUNCH_CHECK("kx3_correct");
        if (cs + 1 < C && (rc = x3_copy(tp->u1 + (size_t)cs * 3 * BN, b->ures, 3 * BN * 4, st))) return rc;
    }
    return o3_copy_active(b, u, b->ures, 3 * BN, act, st);
}
extern "C" size_t fgb_extruded3_adjoint_workspace_bytes(const fgb_extruded3_tables *xt, int32_t B) {
    const size_t BN = (size_t)B * xt->plane.N * xt->nz, BNB = (size_t)B * xt->nz * (xt->plane.NB > 0 ? xt->plane.NB : 1);
    return (size_t)(3 + 3 + 1 + 6 + 3 + 1 + 1 + 1 + 3 + 1 + 3 + 1 + 3) * align_up(BN * 4) + align_up(BNB * 4) + 8192;
}
// (u_out_bar, p_out_bar) -> (u_bar, p_prev_bar, bvel_bar), all overwritten; environments tp->active skips are skipped by every adjoint
// kernel and transposed solve and get the identity cotangents (k_adj_inactive)
extern "C" int fgb_extruded3_piso_substep_backward(fgb_ortho3 *b, const fgb_extruded3_tables *xt, const fgb_tape *tp, const float *u_out_bar,
                                                   const float *p_out_bar, float *u_bar, float *p_prev_bar, float *bvel_bar, void *ws, size_t ws_bytes,
                                                   fgb_stream_t s) {
    if (!b || !xt || !tp || !u_out_bar || !p_out_bar || !u_bar || !p_prev_bar || !bvel_bar || !ws)
        return set_err(FGB_E_ARG, "fgb_extruded3_piso_substep_backward: null argument");
    if (b->t.N != xt->plane.N * xt->nz || b->slab.on) return set_err(FGB_E_ARG, "fgb_extruded3_piso_substep_backward: handle / tables mismatch");
    if (!b->t.rev || b->t.plane != xt->plane.N) return set_err(FGB_E_ARG, "fgb_extruded3_piso_substep_backward: the handle's tables need rev / plane (transposed solves)");
    if (ws_bytes < fgb_extruded3_adjoint_workspace_bytes(xt, b->B)) return set_err(FGB_E_WORKSPACE, "fgb_extruded3_piso_substep_backward: workspace too small");
    const fgb_options &o = b->opt;
    const int C = o.corrector_steps, n_adv = o.adv_nonortho_steps, n_p = o.p_nonortho_steps;
    if (C < 1 || n_adv < 1 || n_p < 1 || C * n_p > 8) return set_err(FGB_E_ARG, "fgb_extruded3_piso_substep_backward: unsupported iteration counts");
    X3Tab x; x.t = xt->plane; x.nz = xt->nz; x.hz = xt->hz;
    cudaStream_t st = STREAM(s);
    const dim3 grid((unsigned)((x.t.N + 255) / 256), (unsigned)x.nz, (unsigned)b->B);
    const size_t B = b->B, NBz = (size_t)x.nz * (x.t.NB > 0 ? x.t.NB : 1), BN = B * b->t.N;
    const int32_t *act = tp->active;
    Carver c{(char *)ws, 0};
    float *unb = c.take<float>(3 * BN), *hbb = c.take<float>(3 * BN), *rAb = c.take<float>(BN), *Coffb = c.take<float>(6 * BN);
    float *Sbb = c.take<float>(3 * BN), *pb = c.take<float>(BN), *xb = c.take<float>(BN), *lam = c.take<float>(BN);
    float *uprevb = c.take<float>(3 * BN), *Ab = c.take<float>(BN), *mu = c.take<float>(3 * BN), *Fbb = c.take<float>(B * NBz);
    float *pb2 = c.take<float>(BN), *xkb = c.take<float>(3 * BN);
    cudaError_t ce;
    int rc;
#define ZEROX(ptr, n) do { ce = cudaMemsetAsync(ptr, 0, (n) * sizeof(float), st); if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "memset", ce); } while (0)
    ZEROX(rAb, BN); ZEROX(Coffb, 6 * BN); ZEROX(Sbb, 3 * BN); ZEROX(Fbb, B * NBz); ZEROX(u_bar, 3 * BN); ZEROX(bvel_bar, 3 * B * NBz);
    if ((rc = x3_copy(unb, u_out_bar, 3 * BN * 4, st))) return rc;
    if ((rc = x3_copy(pb, p_out_bar, BN * 4, st))) return rc;
    b->launches++;
    kx3_pressure_matrix<<<grid, 256, 0, st>>>(x, tp->A, b->Poff, b->Pdiag, act);
    LAUNCH_CHECK("kx3_pressure_matrix (backward)");
    for (int cs = C - 1; cs >= 0; --cs) {
        const float *hb_c = tp->hb + (size_t)cs * 3 * BN;
        const float *uprev = cs == 0 ? tp->ustar + (size_t)(n_adv - 1) * 3 * BN : tp->u1 + (size_t)(cs - 1) * 3 * BN;
        b->launches++;
        kx3_adj_correct<<<grid, 256, 0, st>>>(x, unb, tp->p + (size_t)(cs * n_p + n_p - 1) * BN, tp->A, hbb, rAb, pb, act);
        LAUNCH_CHECK("kx3_adj_correct");
        for (int ps = n_p - 1; ps >= 0; --ps) {
            const int q = cs * n_p + ps;
            const float *pprev = q == 0 ? tp->p_in : tp->p + (size_t)(q - 1) * BN;
            b->launches += 3;
            k3_adj_remove_mean<<<b->B, 1024, 0, st>>>(b->t.N, b->t.N, pb, xb, act);
            LAUNCH_CHECK("k3_adj_remove_mean");
            {   // lam = P^-T x_bar: the forward CG kernel on the transposed operator, zero start, no residual reset
                T3 t = b->t; O3Slab sl = b->slab; int Bi = b->B; const float *poff = b->Poff, *pd = b->Pdiag, *rhs = xb; float *work = b->kry, *part = b->part;
                float tol = b->opt.p_tol; int max_iter = b->opt.max_iter, zero_init = 1, reset_steps = 0, slot = 4; const int32_t *active = act;
                int32_t *iters = b->iters; float *resid = b->resid; unsigned long long *itot = b->iter_total; float *out = lam, *pmean = b->pmean;
                void *args[] = {&t, &sl, &Bi, &poff, &pd, &rhs, &out, &work, &part, &max_iter, &tol, &zero_init, &reset_steps, &slot, &active, &iters, &resid, &itot, &pmean};
                ce = cudaLaunchCooperativeKernel((void *)k3_cg<1>, dim3(o3_coop_blocks(b)), dim3(O3_CT), args, 0, st);
                if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "cudaLaunchCooperativeKernel(k3_cg<1>, backward)", ce);
            }
            ZEROX(pb2, BN);                 // becomes the gradient w.r.t. pprev
            kx3_adj_pressure_rhs<<<grid, 256, 0, st>>>(x, lam, tp->p + (size_t)q * BN, tp->pmean + (size_t)q * B, pprev, tp->A, hbb, Fbb, rAb, pb2, act);
            LAUNCH_CHECK("kx3_adj_pressure_rhs");
            float *tmp = pb; pb = pb2; pb2 = tmp;      // the previous iterate enters only through the deferred term
        }
        ZEROX(uprevb, 3 * BN);
        b->launches++;
        kx3_adj_hbya<<<grid, 256, 0, st>>>(x, hbb, hb_c, tp->A, tp->Coff, uprev, tp->dt, rAb, u_bar, Sbb, Coffb, uprevb, act);
        LAUNCH_CHECK("kx3_adj_hbya");
        float *tmp = unb; unb = uprevb; uprevb = tmp;   // gradient w.r.t. the velocity entering this corrector
    }
    if ((rc = x3_copy(p_prev_bar, pb, BN * 4, st))) return rc;
    float *xb_cur = unb, *xb_prev = xkb;
    for (int k = n_adv - 1; k >= 0; --k) {
        {   // mu = C^-T x_k_bar
            T3 t = b->t; O3Slab sl = b->slab; int Bi = b->B; const float *coff = tp->Coff, *a = tp->A, *rhs = xb_cur; float *xo = mu, *work = b->kry, *part = b->part;
            int maxit = b->opt.max_iter, zero_init = 1, transposed = 1; float tol = b->opt.adv_tol; const int32_t *active = act;
            int32_t *iters = b->iters; float *resid = b->resid; unsigned long long *itot = b->iter_total;
            void *args[] = {&t, &sl, &Bi, &coff, &a, &rhs, &xo, &work, &part, &maxit, &tol, &zero_init, &active, &iters, &resid, &itot, &transposed};
            b->launches++;
            ce = cudaLaunchCooperativeKernel((b->bicg_fused ? (void *)k3_bicgstab<3, 1> : (void *)k3_bicgstab<3, 0>), dim3(o3_coop_blocks(b)), dim3(O3_CT), args, 0, st);
            if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "cudaLaunchCooperativeKernel(k3_bicgstab, transposed)", ce);
        }
        if (k > 0) ZEROX(xb_prev, 3 * BN);
        b->launches++;
        kx3_adj_advection<<<grid, 256, 0, st>>>(x, mu, tp->ustar + (size_t)k * 3 * BN, rAb, tp->A, tp->dt, Ab, Coffb, u_bar, Sbb, bvel_bar,
                                                k > 0 ? xb_prev : u_bar, k == n_adv - 1, act);
        LAUNCH_CHECK("kx3_adj_advection");
        float *tmp = xb_cur; xb_cur = xb_prev; xb_prev = tmp;
    }
    b->launches += 2;
    kx3_adj_assemble<<<grid, 256, 0, st>>>(x, Ab, Coffb, Sbb, tp->bvel_in, u_bar, bvel_bar, Fbb, act);
    LAUNCH_CHECK("kx3_adj_assemble");
    if (x.t.NB > 0) {
        kx3_adj_bflux<<<dim3((unsigned)((x.t.NB + 127) / 128), (unsigned)x.nz, (unsigned)b->B), 128, 0, st>>>(x, Fbb, bvel_bar, act);
        LAUNCH_CHECK("kx3_adj_bflux");
    }
#undef ZEROX
    if (act) b->launches++;
    return launch_adj_inactive(act, b->B, 3, b->t.N, u_out_bar, u_bar, p_out_bar, p_prev_bar, nullptr, nullptr, (int)(3 * NBz), bvel_bar, 0, nullptr, st);
}

// Simulation.make_divergence_free on an extruded domain (SIM.py:1320-1430): A = 1, the velocity itself is the pressure right-hand
// side vector; p_nonortho_steps x [divergence + deferred non-orthogonal term of the current pressure, CG (zero start in the first
// iteration, then restarted from the previous result), mean removal], one velocity correction.  The "PRE" hook (outflow update
// with time step 1) is the caller's.
extern "C" int fgb_extruded3_make_divergence_free(fgb_ortho3 *b, const fgb_extruded3_tables *xt, float *u, float *p, const float *bvel,
                                                  int max_iter, fgb_stream_t s) {
    if (!b || !xt || !u || !p || !bvel) return set_err(FGB_E_ARG, "fgb_extruded3_make_divergence_free: null argument");
    if (b->t.N != xt->plane.N * xt->nz || b->slab.on) return set_err(FGB_E_ARG, "fgb_extruded3_make_divergence_free: handle / tables mismatch");
    X3Tab x; x.t = xt->plane; x.nz = xt->nz; x.hz = xt->hz;
    cudaStream_t st = STREAM(s);
    const dim3 grid((unsigned)((x.t.N + 255) / 256), (unsigned)x.nz, (unsigned)b->B);
    const size_t BN = (size_t)b->B * b->t.N;
    int rc;
    b->launches += 2;
    k_fill<<<(unsigned)((BN + 255) / 256), 256, 0, st>>>(b->A, 1.0f, BN);
    LAUNCH_CHECK("k_fill");
    kx3_pressure_matrix<<<grid, 256, 0, st>>>(x, b->A, b->Poff, b->Pdiag, nullptr);
    LAUNCH_CHECK("kx3_pressure_matrix");
    for (int ps = 0; ps < b->opt.p_nonortho_steps; ++ps) {
        b->launches++;
        kx3_divergence<<<grid, 256, 0, st>>>(x, u, bvel, p, b->A, b->div, nullptr);
        LAUNCH_CHECK("kx3_divergence");
        if ((rc = fgb_ortho3_solve_pressure(b, p, ps == 0, 0 /* no residual reset here, SIM.py:1387-1396 */, max_iter > 0 ? max_iter : b->opt.max_iter, ps, nullptr, s))) return rc;
    }
    b->launches++;
    kx3_correct<<<grid, 256, 0, st>>>(x, u, p, b->A, b->ures, nullptr);
    LAUNCH_CHECK("kx3_correct");
    cudaError_t ce = cudaMemcpyAsync(u, b->ures, 3 * BN * sizeof(float), cudaMemcpyDeviceToDevice, st);
    if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "fgb_extruded3_make_divergence_free: copy", ce);
    return FGB_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// Boundary hooks of the extruded environments as kernels (the default on a GPU; FGB_X3_HOOKS=torch selects the torch expressions of
// ExtrudedStepping, which are what the CPU tests pin to the reference).  Same formulas, statement by statement:
// balance_boundary_fluxes (SIM.py:188-224), update_advective_boundaries (SIM.py:228-393), Domain.getMaxVelocity (DS.cpp:1580-1612).
// One CTA per environment for the boundary kernels (a few thousand faces), flux sums accumulated in double.  Checked on a B200 against
// the torch expressions and a float64 evaluation of them (tests/zz_first_run_worker.py, profiles/r02_hooks_vs_float64.log).
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void x3_block_sum2(double &a, double &b, double *sm /* [66] */) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); }
    if (lane == 0) { sm[2 * warp] = a; sm[2 * warp + 1] = b; }
    __syncthreads();
    if (warp == 0) {
        double x = lane < nw ? sm[2 * lane] : 0.0, y = lane < nw ? sm[2 * lane + 1] : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { x += __shfl_xor_sync(0xffffffffu, x, o); y += __shfl_xor_sync(0xffffffffu, y, o); }
        if (lane == 0) { sm[64] = x; sm[65] = y; }
    }
    __syncthreads();
    a = sm[64]; b = sm[65];
    __syncthreads();
}
// scale all components of the free faces by -(flux through the other prescribed faces) / (flux through the free faces)
__device__ void x3_balance(int NB, int nz, float hz, float *bv /* [3][nz][NB] */, const float *__restrict__ fw /* [2][NB] */,
                           const int8_t *__restrict__ free_mask, float tol, double *sm) {
    const int n = nz * NB;
    double fixed = 0.0, var = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int j = i % NB;
        const float fl = (bv[i] * fw[j] + bv[n + i] * fw[NB + j]) * hz;
        if (free_mask[j]) var += (double)fl; else fixed += (double)fl;
    }
    x3_block_sum2(fixed, var, sm);
    if (!(fabs(fixed + var) <= (double)tol * 0.01)) {
        const float sc = (float)(-fixed / var);
        for (int i = threadIdx.x; i < n; i += blockDim.x)
            if (free_mask[i % NB]) { bv[i] *= sc; bv[n + i] *= sc; bv[2 * n + i] *= sc; }
    }
    __syncthreads();
}
__global__ void __launch_bounds__(512) kx3_balance_fluxes(int NB, int nz, float hz, float *Bvel, const float *__restrict__ fw,
                                                          const int8_t *__restrict__ free_mask, float tol) {
    __shared__ double sm[66];
    x3_balance(NB, nz, hz, Bvel + (size_t)blockIdx.x * 3 * nz * NB, fw, free_mask, tol, sm);
}
__global__ void __launch_bounds__(512) kx3_update_outflow(int N2, int NB, int nz, float hz, const float *__restrict__ U, float *Bvel,
                                                          const float *__restrict__ dtv, const float *__restrict__ fw,
                                                          const int8_t *__restrict__ out_mask, int n_out, const int32_t *__restrict__ out_face,
                                                          const int32_t *__restrict__ out_cell, const float *__restrict__ out_adv, float tol) {
    __shared__ double sm[66];
    const int b = blockIdx.x, n = nz * NB;
    const size_t N3 = (size_t)N2 * nz;
    const float *u = U + (size_t)b * 3 * N3;
    float *bv = Bvel + (size_t)b * 3 * n;
    const float dt = dtv[b];
    for (int i = threadIdx.x; i < nz * n_out; i += blockDim.x) {
        const int k = i / n_out, q = i % n_out, j = out_face[q], c = out_cell[q];
        const float w = 1.0f - 1.0f / (1.0f + 2.0f * dt * out_adv[q]);
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            const float bo = bv[(size_t)d * n + k * NB + j];
            bv[(size_t)d * n + k * NB + j] = bo - w * (bo - u[(size_t)d * N3 + (size_t)k * N2 + c]);
        }
    }
    __syncthreads();
    x3_balance(NB, nz, hz, bv, fw, out_mask, tol, sm);
}
__global__ void __launch_bounds__(256) kx3_max_velocity(X3Tab x, const float *__restrict__ U, const float *__restrict__ Bvel, float *__restrict__ maxvel) {
    __shared__ float smf[33];
    const int b = blockIdx.y, N2 = x.t.N, NB = x.t.NB, nz = x.nz;
    const size_t N3 = (size_t)N2 * nz;
    const float *u = U + (size_t)b * 3 * N3, *bv = Bvel + (size_t)b * 3 * nz * NB;
    float m = 0.f;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < N3; i += (size_t)gridDim.x * blockDim.x) {
        const int g = (int)(i % N2);
        const float ux = u[i], uy = u[N3 + i];
        m = fmaxf(m, fabsf(x.t.minv[g] * ux + x.t.minv[N2 + g] * uy));
        m = fmaxf(m, fabsf(x.t.minv[2 * N2 + g] * ux + x.t.minv[3 * N2 + g] * uy));
        m = fmaxf(m, fabsf(u[2 * N3 + i]) / x.hz);
    }
    const int nb = nz * NB;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nb; i += gridDim.x * blockDim.x) {
        const int j = i % NB;
        const float bx = bv[i], by = bv[nb + i];
        m = fmaxf(m, fabsf(x.t.b_minv[j] * bx + x.t.b_minv[NB + j] * by));
        m = fmaxf(m, fabsf(x.t.b_minv[2 * NB + j] * bx + x.t.b_minv[3 * NB + j] * by));
        m = fmaxf(m, fabsf(bv[2 * nb + i]) / x.hz);
    }
    const float mv = block_reduce_max(m, smf);
    if (threadIdx.x == 0) atomicMax((int *)&maxvel[b], __float_as_int(mv));
}

// per-plane wall forces (forces.py:278-377 = the 2-D wall traction of every plane times the plane spacing; same statements as
// k_wall_forces with the extruded strides): out[B][nz][2] (drag, lift coefficient contributions), overwritten
__global__ void __launch_bounds__(128) kx3_wall_forces(fgb_wall w, float visc, int N2, int NB, int nz, float hz, const float *__restrict__ U,
                                                        const float *__restrict__ P, const float *__restrict__ Bvel, float *__restrict__ out) {
    __shared__ double red[32 * 2 + 2];
    const int k = blockIdx.x, b = blockIdx.y;
    const size_t N3 = (size_t)N2 * nz, nb3 = (size_t)nz * NB;
    const float *u = U + (size_t)b * 3 * N3 + (size_t)k * N2, *p = P + (size_t)b * N3 + (size_t)k * N2;
    const float *bv = Bvel + (size_t)b * 3 * nb3 + (size_t)k * NB;
    const int n = w.n_wall;
    float f[2] = {0.f, 0.f};
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int c = w.cell[i], j = w.bface[i];
        const int il = w.cell[(i + 1) % n], ir = w.cell[(i + n - 1) % n];
        const float nx = w.normal[i], ny = w.normal[n + i];
        const float tx = ny, ty = -nx;
        const float du_dn = (u[c] - bv[j]) / w.dist[i], dv_dn = (u[N3 + c] - bv[nb3 + j]) / w.dist[i];
        const float du_dt = (u[ir] - u[il]) / (2.f * w.tlen[i]), dv_dt = (u[N3 + ir] - u[N3 + il]) / (2.f * w.tlen[i]);
        const float du_dx = du_dn * nx + du_dt * tx, du_dy = du_dn * ny + du_dt * ty;
        const float dv_dx = dv_dn * nx + dv_dt * tx, dv_dy = dv_dn * ny + dv_dt * ty;
        const float sxx = 2.f * visc * du_dx - p[c], syy = 2.f * visc * dv_dy - p[c];
        const float sxy = 2.f * visc * (0.5f * (du_dy + dv_dx));
        f[0] += (sxx * nx + sxy * ny) * w.flen[i];
        f[1] += (sxy * nx + syy * ny) * w.flen[i];
    }
    block_reduce_sum<2>(f, red);
    if (threadIdx.x == 0) { out[((size_t)b * nz + k) * 2] = f[0] * w.scale * hz; out[((size_t)b * nz + k) * 2 + 1] = f[1] * w.scale * hz; }
}
extern "C" int fgb_extruded3_wall_forces(const fgb_extruded3_tables *xt, int32_t B, const fgb_wall *w, const float *u, const float *p,
                                         const float *bvel, float *out, fgb_stream_t s) {
    if (!xt || !w || !u || !p || !bvel || !out || B <= 0) return set_err(FGB_E_ARG, "fgb_extruded3_wall_forces: bad argument");
    kx3_wall_forces<<<dim3((unsigned)xt->nz, (unsigned)B), 128, 0, STREAM(s)>>>(*w, xt->plane.viscosity, xt->plane.N, xt->plane.NB, xt->nz, xt->hz,
                                                                               u, p, bvel, out);
    LAUNCH_CHECK("kx3_wall_forces");
    return FGB_OK;
}
// actuation (jet_cylinder_env_3d.py:399-424, airfoil_env_3d.py:383-407): bvel[0..1][k][face q] = sum_j amp[b][k][j] * templ[j][0..1][q],
// spanwise component 0, then the flux balance over the free faces (jets + outflow)
__global__ void __launch_bounds__(512) kx3_apply_jets(int NB, int nz, float hz, float *Bvel, const float *__restrict__ amp, int J,
                                                      const int32_t *__restrict__ jet_face, const float *__restrict__ templ, int nf,
                                                      const float *__restrict__ fw, const int8_t *__restrict__ free_mask, float tol) {
    __shared__ double sm[66];
    const int b = blockIdx.x, n = nz * NB;
    float *bv = Bvel + (size_t)b * 3 * n;
    const float *a = amp + (size_t)b * nz * J;
    for (int i = threadIdx.x; i < nz * nf; i += blockDim.x) {
        const int k = i / nf, q = i % nf, j = jet_face[q];
        float v0 = 0.f, v1 = 0.f;
        for (int jj = 0; jj < J; ++jj) { const float am = a[k * J + jj]; v0 += am * templ[(jj * 2) * nf + q]; v1 += am * templ[(jj * 2 + 1) * nf + q]; }
        bv[k * NB + j] = v0; bv[n + k * NB + j] = v1; bv[2 * n + k * NB + j] = 0.f;
    }
    __syncthreads();
    x3_balance(NB, nz, hz, bv, fw, free_mask, tol, sm);
}
extern "C" int fgb_extruded3_apply_jets(const fgb_extruded3_tables *xt, int32_t B, float *bvel, const float *amp, int32_t J, const int32_t *jet_face,
                                        const float *templ, int32_t nf, const float *fw, const int8_t *free_mask, float tol, fgb_stream_t s) {
    if (!xt || !bvel || !amp || !jet_face || !templ || !fw || !free_mask || B <= 0 || J <= 0 || nf <= 0)
        return set_err(FGB_E_ARG, "fgb_extruded3_apply_jets: bad argument");
    kx3_apply_jets<<<B, 512, 0, STREAM(s)>>>(xt->plane.NB, xt->nz, xt->hz, bvel, amp, J, jet_face, templ, nf, fw, free_mask, tol);
    LAUNCH_CHECK("kx3_apply_jets");
    return FGB_OK;
}
extern "C" int fgb_extruded3_balance_fluxes(const fgb_extruded3_tables *xt, int32_t B, float *bvel, const float *fw, const int8_t *free_mask,
                                            float tol, fgb_stream_t s) {
    if (!xt || !bvel || !fw || !free_mask || B <= 0) return set_err(FGB_E_ARG, "fgb_extruded3_balance_fluxes: bad argument");
    kx3_balance_fluxes<<<B, 512, 0, STREAM(s)>>>(xt->plane.NB, xt->nz, xt->hz, bvel, fw, free_mask, tol);
    LAUNCH_CHECK("kx3_balance_fluxes");
    return FGB_OK;
}
extern "C" int fgb_extruded3_update_outflow(const fgb_extruded3_tables *xt, int32_t B, const float *u, float *bvel, const float *dt, const float *fw,
                                            const int8_t *out_mask, int32_t n_out, const int32_t *out_face, const int32_t *out_cell,
                                            const float *out_adv, float tol, fgb_stream_t s) {
    if (!xt || !u || !bvel || !dt || !fw || !out_mask || !out_face || !out_cell || !out_adv || B <= 0 || n_out <= 0)
        return set_err(FGB_E_ARG, "fgb_extruded3_update_outflow: bad argument");
    kx3_update_outflow<<<B, 512, 0, STREAM(s)>>>(xt->plane.N, xt->plane.NB, xt->nz, xt->hz, u, bvel, dt, fw, out_mask, n_out, out_face, out_cell,
                                                 out_adv, tol);
    LAUNCH_CHECK("kx3_update_outflow");
    return FGB_OK;
}
extern "C" int fgb_extruded3_max_velocity(const fgb_extruded3_tables *xt, int32_t B, const float *u, const float *bvel, float *maxvel,
                                          fgb_stream_t s) {
    if (!xt || !u || !bvel || !maxvel || B <= 0) return set_err(FGB_E_ARG, "fgb_extruded3_max_velocity: bad argument");
    cudaStream_t st = STREAM(s);
    cudaError_t ce = cudaMemsetAsync(maxvel, 0, (size_t)B * sizeof(float), st);
    if (ce != cudaSuccess) return set_err(FGB_E_CUDA, "fgb_extruded3_max_velocity: memset", ce);
    X3Tab x; x.t = xt->plane; x.nz = xt->nz; x.hz = xt->hz;
    const size_t N3 = (size_t)x.t.N * x.nz;
    unsigned blocks = (unsigned)((N3 + 255) / 256);
    if (blocks > 592) blocks = 592;
    kx3_max_velocity<<<dim3(blocks, (unsigned)B), 256, 0, st>>>(x, u, bvel, maxvel);
    LAUNCH_CHECK("kx3_max_velocity");
    return FGB_OK;
}
#endif  // X3_HOST_ONLY
#endif  // __CUDACC__
