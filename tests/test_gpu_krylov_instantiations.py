"""Every instantiation of the 2-D Krylov kernels (csrc/piso_b200.cu) the launchers can select, against the float64 statement of the
same recurrence (oracle/krylov_eval.py).

Case table.  Each case is a domain, a ``cg_impl`` (and a strip shape through FGB_STRIP_SHAPE) and the kernel template that must run
for it.  Domains are sized so that the launchers' capacity rules pick every cluster size (cylinder res 8 / 16 / 24 / 32 / 36 / 52
= 1 984 / 6 192 / 14 232 / 23 424 / 29 700 / 60 840 cells, five blocks with flipped axes and non-orthogonal cells; RBC2D-easy, 5 856
cells, one block with a periodic wrap) and every fall-through to the global-memory kernels.  One solve of each case runs under
torch.profiler: the demangled kernel name must carry the expected template arguments, so a dispatcher that silently falls through
fails the case that names it.  The table of (kernel, template arguments) -> cases is printed.

Contracts, on a synthetic SPD system on the domain's own stencil (symmetric through tables.rev, NaN in the slots of faces without a
neighbour) and on a non-symmetric diagonally dominant one for BiCGStab:
1. capped iterates: max_iter 1, 2, 3, 5, 8, 13, 21 x reset every 0 / 7 x zero / warm start: the returned iterate (and the removed
   mean where the kernel reports it), iteration and criterion equal the float64 recurrence at the same cap.  Tolerance: the float32
   recurrence differs from the float64 one at these caps by <= 2e-7 relative (measured with krylov_eval in float32 on these
   systems: every update is a 5-term stencil row or a sum of N products, rounded once per operation, and the shifted system has a
   condition number below 100, which bounds the growth of those errors over 21 iterations); 1e-5 leaves 50x for the kernels'
   other summation orders.  A wrong coefficient or neighbour value in one cell reaches the first iterate of a zero start only
   through alpha_0 (x_1 = alpha_0 f: O(1 / N), 1.6e-5 at N = 60 840); from the second iterate on it enters r_1 and p_1 directly,
   O(1 / sqrt(N)) >= 4e-3, which caps 2 and up see.  Where the float64 best-iterate choice is within 1e-4 of a tie, either
   candidate is accepted.  The capped loop also runs on the non-symmetric system (caps 1-8: the CG recurrence is defined for a
   few iterations of any matrix), so a kernel that applies the transposed coefficients in a forward solve fails it.
2. full synthetic solves: iteration count within 2 of the float64 recurrence; reported criterion = float64 true residual of the
   returned iterate within 2 % (the recurrence residual drifts from f - P x by float32 rounding); the error to spsolve is bounded by
   the true residual over the Gershgorin bound of the smallest eigenvalue.
3. the solver's own assembled systems (the state of a seeded environment reset on the cylinder grids, a seeded closed-box state on
   RBC2D; setup_* kernels): float64 true residual below 5 x tol, iteration count within 2 % + 2 of the C oracle on the same system,
   solution within the 5e-4 tolerance ball of cg_impl 0; BiCGStab residuals below tol.
4. edges: a zero right-hand side in one environment while the others solve, a pair of environments of which one finishes after
   a few iterations and the other runs long (scaled right-hand side: the criterion is absolute), right-hand sides non-zero in one
   cell at both sides of a CTA cut, at halo / ghost cells and at cell N - 1, identical environments give identical bits, an
   environment equals itself solved alone (B = 1, a half-empty pair for the two-environment kernel), an active mask leaves the
   inactive environment's outputs untouched bit for bit, BiCGStab components that finish at different iterations; the launchers'
   clean errors.
5. transposed solves of one backward (one corrector, one pressure iteration, one predictor iteration): lam = P^-T x_bar
   (cg_impl 6 on 2 / 4 / 8 / 16-CTA clusters, cg_impl 11 on 1 / 2 / 4 / 8-CTA strip plans) and mu = C^-T x_bar of the predictor
   (BiCGStab on 2 / 4 / 8 / 16-CTA clusters), read from the adjoint workspace.  The backward is repeated with max_iter 1 ... 21:
   the capped iterates and iteration counts equal the float64 transposed recurrences (krylov_eval flags bit 0, no convergence
   needed).  With the default cap mu converges (residual below 1.5 x tol plus the float32 rounding floor of its right-hand side,
   iteration count within 2 of the float64 recurrence);
   the transposed pressure CG reaches tol exactly when the float64 recurrence does, and then ||x_bar - P^T lam|| / sqrt(N) is
   below 5 x tol and the count within 2 % + 2 (on these states neither converges: CG on the non-symmetric P^T stalls).
"""
import re

import numpy as np
import pytest
import scipy.sparse.linalg as sla

import krylov_eval as ke
from conftest import rel_l2

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

TOL = 1e-5                     # the solvers' default pressure_tol / advection_tol
TOL_CAP = 1e-5
CAPS = (1, 2, 3, 5, 8, 13, 21)
CAPS_NONSYM = (1, 2, 3, 5, 8)

# (domain, cg_impl, FGB_STRIP_SHAPE or None, expected kernel)
CG_CASES = [
    ("cyl8", 0, None, "k_cg<1024>"),
    ("cyl8", 1, None, "k_cg_cluster<512, 6, 2, 0>"), ("cyl16", 1, None, "k_cg_cluster<512, 7, 4, 0>"), ("cyl32", 1, None, "k_cg<1024>"),
    ("cyl8", 2, None, "k_cg_cluster<512, 6, 2, 1>"), ("cyl16", 2, None, "k_cg_cluster<512, 7, 4, 1>"), ("cyl32", 2, None, "k_cg<1024>"),
    ("cyl8", 3, None, "k_cg_cluster_mb<512, 6, 2, false, 1>"), ("cyl16", 3, None, "k_cg_cluster_mb<512, 7, 4, false, 1>"),
    ("cyl32", 3, None, "k_cg_cluster_mb<512, 7, 8, false, 1>"), ("cyl36", 3, None, "k_cg_cluster_mb<512, 6, 16, false, 1>"),
    ("cyl52", 3, None, "k_cg<1024>"),
    ("cyl8", 4, None, "k_cg_smem<512, 12, 1, 1>"), ("cyl16", 4, None, "k_cg_smem<512, 14, 2, 1>"), ("cyl32", 4, None, "k_cg_smem<512, 12, 4, 1>"),
    ("cyl36", 4, None, "k_cg<1024>"),
    ("cyl8", 5, None, "k_cg_smem<512, 6, 2, 2>"), ("cyl16", 5, None, "k_cg_smem<512, 7, 4, 2>"), ("cyl32", 5, None, "k_cg_smem<512, 7, 8, 2>"),
    ("cyl36", 5, None, "k_cg<1024>"),
    ("cyl8", 6, None, "k_cg_cluster_mb<512, 6, 2, true, 1>"), ("rbc12", 6, None, "k_cg_cluster_mb<512, 6, 2, true, 1>"),
    ("cyl16", 6, None, "k_cg_cluster_mb<512, 7, 4, true, 1>"), ("cyl32", 6, None, "k_cg_cluster_mb<512, 7, 8, true, 1>"),
    ("cyl36", 6, None, "k_cg_cluster_mb<512, 6, 16, true, 1>"), ("cyl52", 6, None, "k_cg<1024>"),
    ("cyl8", 7, None, "k_cg_cluster_mb<256, 12, 2, true, 1>"), ("cyl16", 7, None, "k_cg_cluster_mb<256, 14, 4, true, 1>"),
    ("cyl32", 7, None, "k_cg_cluster_mb<256, 14, 8, true, 1>"), ("cyl36", 7, None, "k_cg_cluster_mb<256, 12, 16, true, 1>"),
    ("cyl52", 7, None, "k_cg<1024>"),
    ("cyl8", 8, None, "k_cg_cluster_mb<256, 7, 2, true, 2>"), ("cyl16", 8, None, "k_cg_cluster_mb<256, 7, 4, true, 2>"),
    ("cyl24", 8, None, "k_cg_cluster_mb<256, 7, 8, true, 2>"), ("cyl32", 8, None, "k_cg_cluster_mb<256, 7, 16, true, 2>"),
    ("cyl36", 8, None, "k_cg<1024>"),
    ("cyl8", 11, None, "k_cg_strip<480, 17, 1, 1, true>"), ("rbc12", 11, None, "k_cg_strip<480, 17, 1, 1, true>"),
    ("cyl16", 11, None, "k_cg_strip<480, 17, 2, 1, true>"), ("cyl32", 11, None, "k_cg_strip<480, 17, 4, 1, true>"),
    ("cyl36", 11, None, "k_cg_strip<480, 17, 8, 1, true>"), ("cyl52", 11, None, "k_cg_strip<480, 17, 16, 1, true>"),
    ("cyl16", 11, "256,17", "k_cg_strip<256, 17, 2, 2, true>"), ("cyl36", 11, "256,17", "k_cg_strip<256, 17, 16, 2, true>"),
    ("cyl16", 11, "896,9", "k_cg_strip<896, 9, 1, 1, true>"), ("cyl36", 11, "896,9", "k_cg_strip<896, 9, 8, 1, true>"),
    ("cyl16", 11, "640,13", "k_cg_strip<640, 13, 1, 1, true>"), ("cyl32", 11, "640,13", "k_cg_strip<640, 13, 4, 1, true>"),
    ("cyl16", 11, "320,13", "k_cg_strip<320, 13, 2, 2, true>"), ("cyl36", 11, "320,13", "k_cg_strip<320, 13, 16, 2, true>"),
    ("cyl52", 11, "256,17", "k_cg<1024>"),          # no strip plan of this shape and no halo plan (N > 16 x 3072): k_cg
    ("cyl16", 12, None, "k_cg_strip2<480, 9, 2>"), ("rbc12", 12, None, "k_cg_strip2<480, 9, 2>"),
    ("cyl24", 12, None, "k_cg_strip2<480, 9, 4>"), ("cyl32", 12, None, "k_cg_strip2<480, 9, 8>"),
    ("cyl16", 13, None, "k_cg_strip<480, 17, 2, 1, false>"), ("cyl36", 13, None, "k_cg_strip<480, 17, 8, 1, false>"),
]
# advection BiCGStab, NC = 2 (cg_impl 0 always takes the global-memory kernel)
BICG_CASES = [
    ("cyl8", 0, "k_bicgstab<1024, 2>"), ("cyl8", 6, "k_bicgstab_cluster<512, 6, 2, 2>"), ("cyl16", 6, "k_bicgstab_cluster<512, 7, 4, 2>"),
    ("cyl32", 11, "k_bicgstab_cluster<512, 7, 8, 2>"), ("cyl36", 6, "k_bicgstab_cluster<512, 6, 16, 2>"), ("cyl52", 11, "k_bicgstab<1024, 2>"),
]
# the launchers refuse these before anything runs
ERROR_CASES = [
    ("cyl8", 12, "cg_impl 12: no k_cg_strip2 instantiation"),            # one-CTA plan
    ("cyl52", 12, "cg_impl 12: no k_cg_strip2 instantiation"),           # 16-CTA plan
    ("rbc4", 11, "cg_impl 11/13: domain too small for the best-iterate scratch"),   # 1 x 480 x 17 > 12 x 640
]
# domains of contract 3.  From the state of a fresh reset the cylinder-32 system needs more than the 5 000-iteration cap (the C
# oracle does not converge either); the environments solve it from the previous step's pressure.
ASSEMBLED = ("cyl8", "rbc12", "cyl16", "cyl24")
# (domain, cg_impl, cluster size of the pressure solve, cluster size of the BiCGStab adjoint)
TRANSPOSED = [("cyl8", 6, 2, 2), ("cyl16", 6, 4, 4), ("cyl32", 6, 8, 8), ("cyl36", 6, 16, 16),
              ("cyl8", 11, 1, 2), ("cyl16", 11, 2, 4), ("cyl32", 11, 4, 8), ("cyl36", 11, 8, 16)]
DT = 0.01
# instantiations the launchers can reach that the table above does not run, with the reason
NOT_RUN = {
    "k_bicgstab_cluster<..., NC = 1>": "scalar transport of piso_substep only (RBC2D end to end against goldens, test_gpu_rbc.py); "
                                       "its transposed solve: test_gpu_rbc_autograd.py",
    "k_bicgstab<1024, 1>": "scalar transport with cg_impl 0 only (same path)",
    "k_cg_cluster_mb<..., PUSH> under cg_impl 11 / 13 without a strip plan": "the cg_impl 6 instantiations above; no domain of "
                                                                             "<= 49 152 cells lacks a strip plan",
}

_COVERED = {}


def _cid(c):
    return f"{c[0]}-impl{c[1]}" + (f"-shape{c[2].replace(',', 'x')}" if len(c) > 3 and c[2] else "")


_SPECS = {}


@pytest.fixture(scope="module")
def domains(cyl24):
    from fluidgym_b200.envs.cylinder_domain import make_cylinder_domain
    from fluidgym_b200.envs.rbc_domain import make_rbc_domain
    out = {}
    for r in (8, 16, 32, 36, 52):
        _SPECS[f"cyl{r}"] = make_cylinder_domain(r)
        out[f"cyl{r}"] = _SPECS[f"cyl{r}"].prepare()
    _SPECS["cyl24"], out["cyl24"] = cyl24
    out["rbc12"] = make_rbc_domain(n_heaters=12, heater_width=8)[0].prepare()
    out["rbc4"] = make_rbc_domain(n_heaters=4, heater_width=8)[0].prepare()
    return out


_REF = {}


def _spd(cd, name):
    """synthetic SPD system of the domain, its right-hand side / warm start and the float64 references that do not depend on the
    kernel (cached per domain)"""
    if name not in _REF:
        off, diag = ke.synthetic_spd(cd.nbr, cd.rev, seed=11)
        P = ke.ell_matrix(cd.nbr, off, diag)
        rng = np.random.default_rng(12)
        f = rng.standard_normal(cd.N).astype(np.float32)
        x0 = (0.3 * rng.standard_normal(cd.N)).astype(np.float32)
        hist = {(reset, warm): ke.cg_history(P, f, x0 if warm else None, reset, max(CAPS)) for reset in (0, 7) for warm in (False, True)}
        full = ke.cg(P, f, None, TOL, 100, 5000)
        exact = sla.spsolve(P.tocsc(), f.astype(np.float64))
        lam_min = float((diag - np.abs(np.where(np.asarray(cd.nbr) >= 0, off, 0)).sum(0)).min())   # Gershgorin
        off_n, diag_n = ke.synthetic_nonsym(cd.nbr, seed=15)
        hist_n = ke.cg_history(ke.ell_matrix(cd.nbr, off_n, diag_n), f, None, 0, max(CAPS_NONSYM))
        scaled = ke.cg(P, f * np.float32(1e-3), None, TOL, 100, 5000)
        _REF[name] = dict(off=off, diag=diag, P=P, f=f, x0=x0, hist=hist, full=full, exact=exact, lam_min=lam_min,
                          off_n=off_n, diag_n=diag_n, hist_n=hist_n, scaled=scaled)
    return _REF[name]


def _solver(cd, B, cg_impl, shape, monkeypatch, **kw):
    from fluidgym_b200.solver import BatchedPISO
    if shape:
        monkeypatch.setenv("FGB_STRIP_SHAPE", shape)
    else:
        monkeypatch.delenv("FGB_STRIP_SHAPE", raising=False)
    monkeypatch.delenv("FGB_CG_IMPL", raising=False)
    monkeypatch.delenv("FGB_GROUPS", raising=False)
    return BatchedPISO(cd, B, cg_impl=cg_impl, **kw)


def _load_p(sol, off, diag, F):
    sol.buffer("Poff").copy_(torch.from_numpy(off).cuda().unsqueeze(0).expand(sol.B, -1, -1))
    sol.buffer("Pdiag").copy_(torch.from_numpy(diag).cuda().unsqueeze(0).expand(sol.B, -1))
    sol.buffer("div").copy_(torch.from_numpy(np.ascontiguousarray(F, np.float32)).cuda())


def _krylov_kernels(prof):
    """demangled names (up to the closing '>' of the template arguments) of the Krylov kernels of a trace, in launch order"""
    out = []
    for e in prof.events():
        m = re.search(r"(k_(?:cg|bicgstab)\w*<[^>]*>)", e.name)
        if m and e.device_type == torch.autograd.DeviceType.CUDA:
            out.append((e.time_range.start, m.group(1)))
    return [n for _, n in sorted(out)]


@pytest.fixture(scope="module")
def launched(domains):
    """the kernel every case launches: one solve of each case, one after the other with a device synchronisation between them,
    all in ONE profiler session (a process that opens many sessions has been seen to get empty traces from the later ones).
    Every solve launches exactly one Krylov kernel, so the k-th kernel of the trace belongs to the k-th case."""
    from torch.profiler import ProfilerActivity, profile
    runs = []
    with pytest.MonkeyPatch.context() as mp:
        for case in CG_CASES:
            name, impl, shape, _ = case
            ref = _spd(domains[name], name)
            sol = _solver(domains[name], 1, impl, shape, mp)
            _load_p(sol, ref["off"], ref["diag"], ref["f"][None])
            runs.append((_cid(case), sol, lambda sol=sol: sol.solve_pressure(zero_init=True, max_iter=3)))
        for name, impl, _ in BICG_CASES:
            cd = domains[name]
            off, diag = ke.synthetic_nonsym(cd.nbr, seed=13)
            sol = _solver(cd, 1, impl, None, mp)
            sol.buffer("Coff").copy_(torch.from_numpy(off).cuda()[None])
            sol.buffer("A").copy_(torch.from_numpy(diag).cuda()[None])
            sol.buffer("rhs").normal_()
            sol.set_options(max_iter=3)
            runs.append((f"{name}-impl{impl}-bicg", sol, lambda sol=sol: sol.solve_advection(zero_init=True)))
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _, _, fn in runs:
                fn()
                torch.cuda.synchronize()
    names = _krylov_kernels(prof)
    assert len(names) == len(runs), (len(names), len(runs), names)
    return {cid: n for (cid, _, _), n in zip(runs, names)}


def _expect_kernel(case, expected, launched):
    ran = launched[_cid(case)]
    assert ran == expected, f"case {_cid(case)}: expected {expected}, ran {ran}"
    _COVERED.setdefault(expected, []).append(_cid(case))


def _best_shift(P, f, p):
    """the iterate p + c of the smallest float64 residual (closed form): bounds the residual of the true iterate from below"""
    one = P @ np.ones(p.size)
    res = f - P @ p
    return p + float(one @ res) / float(one @ one)


def _edge_cells(sol, kernel, N):
    """cells next to the cuts of the kernel's layout: the last cell of CTA 0 and the first of CTA 1, a cell CTA 0 exports to a halo
    slot or ghost of another CTA and one it receives (strip plan: remote ghosts of CTA 1 owned by CTA 0 and vice versa; local
    ghosts of the periodic wrap / block connections of CTA 0), and cell N - 1"""
    cells = [N - 1]
    if kernel.startswith("k_cg_strip") and sol.strip is not None:
        cell = sol.strip.cell
        owned = [set(cell[r][cell[r] >= 0].tolist()) for r in range(sol.strip.cs)]
        ghosts = [set((-2 - cell[r][cell[r] <= -2]).tolist()) for r in range(sol.strip.cs)]
        cells.append(min(ghosts[0] & owned[0]) if ghosts[0] & owned[0] else 0)          # local ghost (mirror)
        if sol.strip.cs > 1:
            cells += [min(ghosts[1] & owned[0]), min(ghosts[0] & owned[1]), max(owned[0]), min(owned[1])]
    elif kernel.startswith("k_cg_cluster_mb"):
        h = sol.halo
        per = -(-N // h["cs"])
        cells += [per - 1, per]
        if h["cnt"][0][0] > 0:
            cells.append(int(h["exp"][0][0][0]) & 0xffffff)                              # CTA 0 pushes it to a halo slot
    elif not kernel.startswith("k_cg<"):                                                 # k_cg_cluster / k_cg_smem<T, CPT, CS, ...>
        per = -(-N // int(re.search(r"<\d+, \d+, (\d+)", kernel).group(1)))
        cells += [per - 1, min(per, N - 1)]
    return sorted(set(cells))


def _writes_mean(kernel):
    return kernel.startswith(("k_cg_cluster_mb", "k_cg_strip"))


def _capped_ok(got, crit, xs, m, remove_mean):
    """iterations j < m whose float64 iterate (mean-free if remove_mean) the kernel's result equals within TOL_CAP, among the best
    iterate of the first m and those within 1e-4 of a tie with it; and the errors to every candidate"""
    j_best = int(np.argmin(crit[:m]))
    errs = {j: rel_l2(got, xs[j] - xs[j].mean() if remove_mean else xs[j]) for j in range(m) if crit[j] <= crit[j_best] * (1 + 1e-4)}
    return [j for j, e in errs.items() if e < TOL_CAP], errs


_STATES = {}


def _state(sol, name, seed):
    """cylinder grids: the state of a seeded environment reset (inflow profile, balanced outflow, divergence-free velocity);
    RBC2D: a seeded velocity with closed boundaries (zero boundary velocities).  Pressure zero."""
    if name.startswith("cyl"):
        if (name, seed) not in _STATES:
            from fluidgym_b200.envs.cylinder import CylinderJet2DEnv
            env = CylinderJet2DEnv(n_envs=1, resolution=int(name[3:]), compiled=(_SPECS[name], sol.cd))
            env.reset(seed=seed)
            _STATES[(name, seed)] = (env.solver.u[0].clone(), env.solver.bvel[0].clone())
            del env
        u, bvel = _STATES[(name, seed)]
        sol.u.copy_(u.expand_as(sol.u))
        sol.bvel.copy_(bvel.expand_as(sol.bvel))
    else:
        gen = torch.Generator(device="cuda").manual_seed(seed)
        sol.u.copy_(0.3 + 0.05 * torch.randn(sol.u.shape, device="cuda", generator=gen))
        sol.bvel.zero_()
    sol.p.zero_()


# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CG_CASES, ids=[_cid(c) for c in CG_CASES])
def test_cg_instantiation(domains, launched, case, monkeypatch):
    name, impl, shape, kernel = case
    cd = domains[name]
    N = cd.N
    ref = _spd(cd, name)
    B = 4
    sol = _solver(cd, B, impl, shape, monkeypatch)
    writes_mean = _writes_mean(kernel)
    # edges in one batch: env 0 the system, env 1 its right-hand side scaled by 1e-3 (finishes much earlier; with env 0 it forms
    # the first pair of the two-environment kernel), env 2 identical to env 0, env 3 an all-zero right-hand side
    F = np.stack([ref["f"], ref["f"] * np.float32(1e-3), ref["f"], np.zeros(N, np.float32)])
    _load_p(sol, ref["off"], ref["diag"], F)
    p = torch.empty(B, N, device="cuda")
    _expect_kernel(case, kernel, launched)
    sol.solve_pressure(p_out=p, zero_init=True, reset_steps=100, max_iter=5000)
    torch.cuda.synchronize()
    it, rs, pm = sol.buffer("iters")[:, 2].cpu().numpy(), sol.buffer("resid")[:, 2].cpu().numpy(), sol.buffer("pmean")[0].cpu().numpy()
    pc = p.cpu().numpy().astype(np.float64)
    assert np.array_equal(pc[0], pc[2]) and it[0] == it[2] and rs[0] == rs[2]
    assert not pc[3].any() and it[3] == -1 and rs[3] == 0.0 and (not writes_mean or pm[3] == 0.0)
    scaled = ref["scaled"]
    assert abs(int(it[1]) - scaled.used) <= 2 and it[1] < it[0] and rs[1] < TOL, (it[:2], scaled.used)
    # 2. full solve
    full = ref["full"]
    assert abs(int(it[0]) - full.used) <= 2, (it[0], full.used)
    x = pc[0] + pm[0] if writes_mean else _best_shift(ref["P"], ref["f"], pc[0])
    true = np.linalg.norm(ref["f"] - ref["P"] @ x) / np.sqrt(N)
    assert rs[0] < TOL and true < 1.5 * TOL
    if writes_mean:
        assert abs(rs[0] - true) <= 0.02 * true + 1e-7
    assert np.linalg.norm(x - ref["exact"]) <= 1.01 * true * np.sqrt(N) / ref["lam_min"]
    # 1. capped iterates
    x0 = torch.from_numpy(ref["x0"]).cuda()
    for reset in (0, 7):
        for warm in (False, True):
            crit, xs = ref["hist"][(reset, warm)]
            for m in CAPS:
                p.copy_(x0.expand(B, N))
                sol.solve_pressure(p_out=p, zero_init=not warm, reset_steps=reset, max_iter=m)
                torch.cuda.synchronize()
                ok, errs = _capped_ok(p[0].double().cpu().numpy(), crit, xs, m, remove_mean=True)
                where = f"{_cid(case)} reset {reset} warm {warm} cap {m}"
                assert ok, (where, errs)
                assert int(sol.buffer("iters")[0, 2]) in ok, where
                j = int(sol.buffer("iters")[0, 2])
                assert abs(float(sol.buffer("resid")[0, 2]) - crit[j]) <= TOL_CAP * crit[j] + 1e-9, where
                if writes_mean:
                    scale = np.linalg.norm(xs[j]) / np.sqrt(N)
                    assert abs(float(sol.buffer("pmean")[0, 0]) - xs[j].mean()) <= TOL_CAP * scale, where
    # 4. one-cell right-hand sides at the CTA cuts, at halo / ghost cells and at cell N - 1, against the float64 recurrence
    cells = _edge_cells(sol, kernel, N)
    for k in range(0, len(cells), B):
        F1 = np.zeros((B, N), np.float32)
        for e, g in enumerate(cells[k:k + B]):
            F1[e, g] = 1.0
        sol.buffer("div").copy_(torch.from_numpy(F1).cuda())
        sol.solve_pressure(p_out=p, zero_init=True, reset_steps=0, max_iter=5)
        torch.cuda.synchronize()
        for e, g in enumerate(cells[k:k + B]):
            r = ke.cg(ref["P"], F1[e], None, TOL, 0, 5)
            assert rel_l2(p[e].double().cpu().numpy(), r.x) < TOL_CAP, (_cid(case), "one-hot", g)
    # 1. capped iterates of the non-symmetric system (zero start, no reset)
    _load_p(sol, ref["off_n"], ref["diag_n"], np.stack([ref["f"]] * B))
    crit, xs = ref["hist_n"]
    for m in CAPS_NONSYM:
        sol.solve_pressure(p_out=p, zero_init=True, reset_steps=0, max_iter=m)
        torch.cuda.synchronize()
        ok, errs = _capped_ok(p[0].double().cpu().numpy(), crit, xs, m, remove_mean=True)
        assert ok and int(sol.buffer("iters")[0, 2]) in ok, (_cid(case), "non-symmetric cap", m, errs)
    # 4. active mask: the inactive environment keeps its sentinels bit for bit, the others equal the batch result
    _load_p(sol, ref["off"], ref["diag"], F)
    sentinels = {k: sol.buffer(k).clone().fill_(7) for k in ("iters", "resid", "iter_total")}
    for k, v in sentinels.items():
        sol.buffer(k).copy_(v)
    sol.buffer("pmean").fill_(-3.0)
    p.fill_(5.0)
    active = torch.tensor([1, 0, 1, 1], dtype=torch.int32, device="cuda")     # env 1: the partner of env 0 in a pair
    sol.solve_pressure(p_out=p, zero_init=True, reset_steps=100, max_iter=5000, active=active)
    torch.cuda.synchronize()
    assert torch.equal(p[1], torch.full_like(p[1], 5.0))
    for k in ("iters", "resid", "iter_total"):
        assert torch.equal(sol.buffer(k)[1], sentinels[k][1]), k
    assert float(sol.buffer("pmean")[0, 1]) == -3.0
    assert np.array_equal(p[0].cpu().numpy(), pc[0].astype(np.float32)) and np.array_equal(p[2].cpu().numpy(), pc[2].astype(np.float32))
    assert not p[3].any()
    # 4. the same environment solved alone
    one = _solver(cd, 1, impl, shape, monkeypatch)
    _load_p(one, ref["off"], ref["diag"], ref["f"][None])
    q = torch.empty(1, N, device="cuda")
    one.solve_pressure(p_out=q, zero_init=True, reset_steps=100, max_iter=5000)
    torch.cuda.synchronize()
    assert np.array_equal(q[0].cpu().numpy(), pc[0].astype(np.float32))
    del one, sol


_ASM = {}


def _assembled(cd, name, monkeypatch):
    """the assembled pressure and advection systems of a seeded state (cg_impl 0 builds them), the C oracle's iteration count and
    cg_impl 0's solution; cached per domain"""
    if name not in _ASM:
        from oracle import Oracle
        sol = _solver(cd, 1, 0, None, monkeypatch)
        _state(sol, name, 21)
        dt = 0.01
        sol.setup_advection(dt)
        sol.solve_advection()
        sol.setup_pressure_matrix()
        sol.setup_pressure_rhs(dt)
        sol.solve_pressure(zero_init=True)
        torch.cuda.synchronize()
        Poff, Pdiag, div = (sol.buffer(k)[0].cpu().numpy().copy() for k in ("Poff", "Pdiag", "div"))
        nbr = np.asarray(cd.nbr)
        val = np.concatenate([Pdiag[:, None], np.where(nbr >= 0, Poff, 0).T], axis=1).astype(np.float32)
        idx = np.concatenate([np.arange(cd.N)[:, None], np.where(nbr >= 0, nbr, -1).T], axis=1).astype(np.int32)
        orc = Oracle.from_compiled(cd)
        _, orc_it, _, conv = orc.cg(val, idx, div, maxit=5000, tol=TOL, reset=100)
        assert conv
        _ASM[name] = dict(Poff=Poff, Pdiag=Pdiag, div=div, P=ke.ell_matrix(nbr, Poff, Pdiag), orc_it=orc_it,
                          p0=sol.p[0].cpu().numpy().copy())
    return _ASM[name]


@pytest.mark.parametrize("case", [c for c in CG_CASES if c[0] in ASSEMBLED], ids=[_cid(c) for c in CG_CASES if c[0] in ASSEMBLED])
def test_cg_assembled_system(domains, case, monkeypatch):
    name, impl, shape, kernel = case
    cd = domains[name]
    a = _assembled(cd, name, monkeypatch)
    sol = _solver(cd, 2, impl, shape, monkeypatch)
    _load_p(sol, a["Poff"], a["Pdiag"], np.stack([a["div"], a["div"]]))
    sol.solve_pressure(zero_init=True)
    torch.cuda.synchronize()
    it = int(sol.buffer("iters")[0, 2])
    p = sol.p[0].double().cpu().numpy()
    x = p + float(sol.buffer("pmean")[0, 0]) if _writes_mean(kernel) else _best_shift(a["P"], a["div"], p)
    true = np.linalg.norm(a["div"] - a["P"] @ x) / np.sqrt(cd.N)
    assert true < 5 * TOL, (_cid(case), true)
    assert abs(it - a["orc_it"]) <= 0.02 * a["orc_it"] + 2, (_cid(case), it, a["orc_it"])
    assert rel_l2(p, a["p0"]) < 5e-4
    del sol


@pytest.mark.parametrize("case", BICG_CASES, ids=[f"{c[0]}-impl{c[1]}" for c in BICG_CASES])
def test_bicgstab_instantiation(domains, launched, case, monkeypatch):
    name, impl, kernel = case
    cd = domains[name]
    N = cd.N
    off, diag = ke.synthetic_nonsym(cd.nbr, seed=13)
    C = ke.ell_matrix(cd.nbr, off, diag)
    dominance = float((diag - np.abs(np.where(np.asarray(cd.nbr) >= 0, off, 0)).sum(0)).min())
    rng = np.random.default_rng(14)
    F = rng.standard_normal((2, N)).astype(np.float32)
    F[1] *= np.float32(1e-3)                     # absolute criterion: this component finishes after a few iterations
    B = 3
    sol = _solver(cd, B, impl, None, monkeypatch)
    sol.buffer("Coff").copy_(torch.from_numpy(off).cuda().unsqueeze(0).expand(B, -1, -1))
    sol.buffer("A").copy_(torch.from_numpy(diag).cuda().unsqueeze(0).expand(B, -1))
    rhs = np.stack([F, F, np.stack([F[1], np.zeros(N, np.float32)])])   # env 2: the early component, and an all-zero one
    sol.buffer("rhs").copy_(torch.from_numpy(rhs).cuda())
    ran = launched[f"{name}-impl{impl}-bicg"]
    assert ran == kernel, f"case {name}-impl{impl}: expected {kernel}, ran {ran}"
    _COVERED.setdefault(kernel, []).append(f"{name}-impl{impl}")
    sol.solve_advection(zero_init=True)
    torch.cuda.synchronize()
    x = sol.buffer("ures").double().cpu().numpy()
    it, rs = sol.buffer("iters")[:, :2].cpu().numpy(), sol.buffer("resid")[:, :2].cpu().numpy()
    ref = ke.bicgstab(C, F, None, TOL, 5000)
    assert np.array_equal(x[0], x[1]) and np.array_equal(it[0], it[1])
    for c in range(2):
        assert abs(int(it[0, c]) - int(ref.used[c])) <= 2, (c, it[0], ref.used)
        true = np.linalg.norm(F[c] - C @ x[0, c]) / np.sqrt(N)
        assert rs[0, c] < TOL and true < 1.5 * TOL
        # C is strictly diagonally dominant by rows: ||C^-1||_inf <= 1 / min_i (|c_ii| - sum_j |c_ij|)
        exact = sla.spsolve(C.tocsc(), F[c].astype(np.float64))
        res = F[c] - C @ x[0, c]
        assert np.abs(x[0, c] - exact).max() <= 1.01 * np.abs(res).max() / dominance
    assert it[0, 1] < it[0, 0]
    assert it[2, 1] == -1 and rs[2, 1] == 0.0 and not x[2, 1].any() and it[2, 0] == it[0, 1]
    assert rel_l2(x[2, 0], x[0, 1]) < TOL_CAP
    # capped iterates against the float64 recurrence (a capped component reports used = i of its last half step; its iterate
    # includes the full step that followed)
    for m in (1, 2, 3, 5, 8):
        sol.set_options(max_iter=m)
        sol.solve_advection(zero_init=True)
        torch.cuda.synchronize()
        r = ke.bicgstab(C, F, None, TOL, m)
        got = sol.buffer("ures")[0].double().cpu().numpy()
        for c in range(2):
            assert rel_l2(got[c], r.x[c]) < TOL_CAP, (name, impl, m, c)
            assert int(sol.buffer("iters")[0, c]) == int(r.used[c]), (name, impl, m, c)
    sol.set_options(max_iter=5000)
    # the assembled advection system of a seeded state
    _state(sol, name, 22)
    sol.setup_advection(0.01)
    sol.solve_advection()
    torch.cuda.synchronize()
    Ca = ke.ell_matrix(cd.nbr, sol.buffer("Coff")[0].cpu().numpy(), sol.buffer("A")[0].cpu().numpy())
    xa, fa = sol.buffer("ures")[0].double().cpu().numpy(), sol.buffer("rhs")[0].double().cpu().numpy()
    for c in range(2):
        assert float(sol.buffer("resid")[0, c]) < TOL
        assert np.linalg.norm(fa[c] - Ca @ xa[c]) / np.sqrt(N) < 1.5 * TOL
    del sol


@pytest.mark.parametrize("case", ERROR_CASES, ids=[f"{c[0]}-impl{c[1]}" for c in ERROR_CASES])
def test_launcher_errors(domains, case, monkeypatch):
    from fluidgym_b200.native import FGBError
    name, impl, msg = case
    cd = domains[name]
    sol = _solver(cd, 3, impl, None, monkeypatch)
    from torch.profiler import ProfilerActivity, profile
    ref = _spd(cd, name)
    _load_p(sol, ref["off"], ref["diag"], np.stack([ref["f"]] * 3))
    p = torch.full((3, cd.N), 9.0, device="cuda")
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        with pytest.raises(FGBError, match=re.escape(msg)):
            sol.solve_pressure(p_out=p, zero_init=True)
        torch.cuda.synchronize()
    assert not _krylov_kernels(prof)
    assert bool((p == 9.0).all())
    del sol


ADJ_SIZES = (2, 2, 1, 4, 2, 1, 1, 1, 2, 1, 2)   # unb, hbb, rAb, Coffb, Sbb, pb, xb, lam, uprevb, Ab, mu (in B * N floats)


def _adjoint_vector(sol, want):
    """environment 0 of vector ``want`` carved from the adjoint workspace by fgb_piso_substep_backward (each vector starts on a
    256-byte boundary), as float64 [ADJ_SIZES[want], N]"""
    ws = sol._adj_ws
    off = (-ws.data_ptr()) % 256
    for n in ADJ_SIZES[:want]:
        off += -(-n * sol.B * sol.N * 4 // 256) * 256
    n = ADJ_SIZES[want]
    return ws[off:off + n * sol.B * sol.N * 4].view(torch.float32).view(sol.B, n, sol.N)[0].double().cpu().numpy()


@pytest.mark.parametrize("case", TRANSPOSED, ids=[f"{c[0]}-impl{c[1]}-cs{c[2]}" for c in TRANSPOSED])
def test_transposed_solves(domains, case, monkeypatch):
    """lam = P^-T x_bar and mu = C^-T x_bar of one backward.  With one corrector and one pressure iteration x_bar of the pressure
    solve is the mean-free cotangent of p (xb), lam its solution; x_bar of the predictor is left in uprevb (the corrector loop swaps
    it into place), mu in mu.  P is rebuilt by the backward into Poff / Pdiag, C is the forward's advection matrix (Coff / A)."""
    from fluidgym_b200.autograd import piso_substep
    name, impl, cs, bcs = case
    cd = domains[name]
    N = cd.N
    sol = _solver(cd, 1, impl, None, monkeypatch, corrector_steps=1, pressure_non_ortho_steps=1, advect_non_ortho_steps=1)
    assert (sol.strip.cs if impl == 11 else sol.halo["cs"]) == cs
    # bicgstab_cluster_any: the smallest of 2 x 3072, 4 x 3584, 8 x 3584, 16 x 3072 cells that holds the grid
    assert next(c for c, cap in ((2, 3072), (4, 3584), (8, 3584), (16, 3072)) if -(-N // c) <= cap) == bcs
    _state(sol, name, 23)
    u = sol.u.clone().requires_grad_(True)
    u_out, p_out = piso_substep(sol, u, sol.p.clone(), sol.bvel.clone(), DT)[:2]
    torch.cuda.synchronize()
    C = ke.ell_matrix(cd.nbr, sol.buffer("Coff")[0].cpu().numpy(), sol.buffer("A")[0].cpu().numpy())
    loss = (p_out * p_out.detach()).sum() + (u_out * u_out.detach()).sum()      # smooth cotangents: the fields themselves
    full = sol.options.max_iter
    for m in CAPS + (full,):
        sol.set_options(max_iter=m)
        loss.backward(retain_graph=True)
        torch.cuda.synchronize()
        P = ke.ell_matrix(cd.nbr, sol.buffer("Poff")[0].cpu().numpy(), sol.buffer("Pdiag")[0].cpu().numpy())
        xb, lam = _adjoint_vector(sol, 6)[0], _adjoint_vector(sol, 7)[0]
        xk, mu = _adjoint_vector(sol, 8), _adjoint_vector(sol, 10)
        it, rs = int(sol.buffer("iters")[0, 7]), float(sol.buffer("resid")[0, 7])
        bit = sol.buffer("iters")[0, :2].cpu().numpy()
        where = f"{name}-impl{impl} cap {m}"
        assert np.abs(xb).max() > 0 and abs(xb.mean()) < 1e-6 * np.abs(xb).max(), where
        if m < full:
            crit, xs = ke.cg_history(P, xb, None, 0, m, flags=1)
            ok, errs = _capped_ok(lam, crit, xs, m, remove_mean=False)
            assert ok and it in ok, (where, it, errs)
            assert abs(rs - crit[it]) <= TOL_CAP * crit[it] + 1e-9, (where, rs, crit[it])
            if m <= 5:                                      # the predictor's BiCGStab converges within a few iterations
                r = ke.bicgstab(C, xk, None, TOL, m, flags=1)
                for c in range(2):
                    assert rel_l2(mu[c], r.x[c]) < TOL_CAP and bit[c] == r.used[c], (where, c, rel_l2(mu[c], r.x[c]), bit, r.used)
        else:
            # P is not symmetric at the non-orthogonal corners, and CG on P^T does not converge there, in float64 either (it
            # leaves by the 100-rising-steps rule with a criterion of 0.5 ... 240 on these grids): only the outcome is compared
            ref = ke.cg(P, xb, None, TOL, 0, full, flags=1 | 2)
            assert (rs < TOL) == (ref.fin < TOL), (where, it, rs, ref.used, ref.fin)
            if ref.fin < TOL:
                assert abs(it - ref.used) <= 0.02 * ref.used + 2, (where, it, ref.used)
                assert np.linalg.norm(xb - P.T @ lam) / np.sqrt(N) < 5 * TOL, where
            r = ke.bicgstab(C, xk, None, TOL, full, flags=1)
            for c in range(2):
                assert abs(int(bit[c]) - int(r.used[c])) <= 2, (where, c, bit, r.used)
                # the recurrence residual is below tol; the true one also carries the float32 rounding of C^T mu, which is of the
                # order of eps32 times the size of the right-hand side (large here: the cotangents are the fields themselves)
                floor = 64 * float(np.finfo(np.float32).eps) * np.linalg.norm(xk[c]) / np.sqrt(N)
                true = np.linalg.norm(xk[c] - C.T @ mu[c]) / np.sqrt(N)
                assert true < 1.5 * TOL + floor, (where, c, true, floor)
    del sol


def test_print_coverage():
    """runs last in this module: the instantiations the cases above ran, each with its cases"""
    if not _COVERED:
        pytest.skip("no case ran")
    print("\n2-D Krylov instantiations -> cases")
    for k in sorted(_COVERED):
        print(f"  {k:42s} {', '.join(_COVERED[k])}")
    for k, why in NOT_RUN.items():
        print(f"  {k:42s} not run here: {why}")
    expected = {c[3] for c in CG_CASES} | {c[2] for c in BICG_CASES}
    assert expected <= set(_COVERED), sorted(expected - set(_COVERED))
