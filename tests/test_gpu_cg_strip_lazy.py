"""k_cg_strip with the deferred iterate update and the lazily stored best iterate (cg_impl 11) against the same kernel with the
eager bookkeeping order (cg_impl 13): the two orders perform the same floating-point operations on the same values, so solution,
iteration counts, criteria, iteration totals and the removed mean must be equal under ==.  Covered: 2-CTA (cylinder-24), 1-CTA
(RBC2D) and 8-CTA (Airfoil2D) clusters; identical and distinct environments, an odd batch, an active mask, zero and warm starts,
residual resets every 100 / 7 / no iterations, iteration caps that leave with the pending and with a stored best iterate, the
transposed solve of one autograd backward, and full env.step calls.  (CPU emulation of both orders:
tests/test_cg_strip_bookkeeping_cpu.py.)"""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

CAPS = tuple(range(1, 160, 3))


def _snapshot(sol, p):
    torch.cuda.synchronize()
    return {"x": p.clone(), "iters": sol.buffer("iters").clone(), "resid": sol.buffer("resid").clone(),
            "iter_total": sol.buffer("iter_total").clone(), "mean": sol.buffer("pmean")[0].clone()}


def _solves(sol, dt):
    """the pressure system of the solver's current state, solved in every way the kernel can leave"""
    sol.setup_advection(dt)
    sol.solve_advection()
    sol.setup_pressure_matrix()
    sol.setup_pressure_rhs(dt)
    B, N = sol.B, sol.N
    gen = torch.Generator(device="cuda").manual_seed(7)
    start = torch.randn((B, N), device="cuda", generator=gen)
    out = []
    p = torch.empty((B, N), device="cuda")
    for zero_init in (True, False):
        for reset_steps in (100, 7, 0):
            p.copy_(start)
            sol.solve_pressure(p_out=p, zero_init=zero_init, reset_steps=reset_steps)
            out.append(_snapshot(sol, p))
    for m in CAPS:
        p.copy_(start)
        sol.solve_pressure(p_out=p, zero_init=(m % 2 == 0), reset_steps=(100, 7, 0)[m % 3], max_iter=m)
        out.append(_snapshot(sol, p) | {"cap": m})
    active = torch.tensor([1 if e % 3 != 1 else 0 for e in range(B)], dtype=torch.int32, device="cuda")
    p.copy_(start)
    sol.solve_pressure(p_out=p, zero_init=True, max_iter=40, active=active)
    out.append(_snapshot(sol, p))
    return out


def _assert_equal(a, b):
    assert len(a) == len(b)
    for k, (sa, sb) in enumerate(zip(a, b)):
        for key in sa:
            if key != "cap":
                assert torch.equal(sa[key], sb[key]), (k, sa.get("cap"), key)


def _cap_exits(snaps):
    """(capped solves that left with the pending iterate, capped solves that left with an older stored one)"""
    last = [int(v) for s in snaps if "cap" in s for v in (s["iters"][:, 2] == s["cap"] - 1).tolist()]
    return last.count(1), last.count(0)


def _load_cyl(sol, fx, noisy):
    for dst, src in ((sol.u, fx["u_in"]), (sol.p, fx["presres_in"]), (sol.bvel, fx["bvel_in"])):
        dst.copy_(torch.from_numpy(np.ascontiguousarray(src)).cuda().unsqueeze(0).expand_as(dst))
    gen = torch.Generator(device="cuda").manual_seed(1234)
    sol.u[noisy:] += 1e-3 * torch.randn(sol.u[noisy:].shape, device="cuda", generator=gen)


def test_cylinder_solves_bit_identical(cyl24, golden):
    from fluidgym_b200.solver import BatchedPISO
    spec, cd = cyl24
    fx = golden("cyl24_substep1.npz")
    res = {}
    for impl in (11, 13):
        sol = BatchedPISO(cd, 5, cg_impl=impl)
        assert sol.strip is not None and sol.strip.cs == 2
        _load_cyl(sol, fx, noisy=2)                   # environments 0 and 1 identical, 2..4 distinct
        res[impl] = _solves(sol, float(fx["dt"][0]))
        del sol
    _assert_equal(res[11], res[13])
    pending, stored = _cap_exits(res[11])
    assert pending > 0 and stored > 0
    s = res[11][0]
    assert torch.equal(s["x"][0], s["x"][1]) and not torch.equal(s["x"][2], s["x"][3])
    assert (s["resid"][:, 2] < 1e-5).all()


@pytest.mark.parametrize("family", ["RBC2D", "Airfoil2D"])
def test_other_cluster_sizes_bit_identical(family, airfoil):
    """RBC2D packs into one CTA, Airfoil2D-medium into an 8-CTA cluster (both default to cg_impl 6; 11 / 13 on request)"""
    res, cs = {}, {}
    for impl in (11, 13):
        if family == "RBC2D":
            import fluidgym_b200
            env = fluidgym_b200.make("RBC2D-easy-v0", n_envs=3, cg_impl=impl)
        else:
            from fluidgym_b200.envs.airfoil import Airfoil2DEnv
            env = Airfoil2DEnv(n_envs=3, compiled=airfoil, cg_impl=impl)
        env.reset(seed=5)
        obs, rew, *_ = env.step(env.sample_action())
        sol = env.solver
        cs[impl] = sol.strip.cs
        state = [sol.u.clone(), sol.p.clone(), rew.clone(), sol.buffer("iter_total").clone()]
        res[impl] = (state, _solves(sol, float(env.dt) / 4))
        del env, sol
    assert cs[11] == cs[13] == (1 if family == "RBC2D" else 8)
    for a, b in zip(res[11][0], res[13][0]):
        assert torch.equal(a, b)
    _assert_equal(res[11][1], res[13][1])


def _adjoint_vectors(sol, *sizes):
    """the first vectors carved from the adjoint workspace by fgb_piso_substep_backward (n * B * N floats each, every one
    starting on a 256-byte boundary), each as a [B, N] copy of its first B * N floats"""
    ws = sol._adj_ws
    off, out = (-ws.data_ptr()) % 256, []
    for n in sizes:
        out.append(ws[off:off + sol.B * sol.N * 4].view(torch.float32).view(sol.B, sol.N).clone())
        off += -(-n * sol.B * sol.N * 4 // 256) * 256
    return out


def test_transposed_solve_bit_identical(cyl24, golden):
    """the one transposed pressure solve of a backward with one corrector and one pressure iteration: its right-hand side x_bar is
    the mean-free cotangent of p (exact here: u_out_bar = 0, so the scattered velocity terms add only zeros); x_bar and the solution
    lam are read from the adjoint workspace (unb, hbb, rAb, Coffb, Sbb, pb, xb, lam)"""
    from fluidgym_b200.autograd import piso_substep
    from fluidgym_b200.solver import BatchedPISO
    spec, cd = cyl24
    fx = golden("cyl24_substep1.npz")
    res = {}
    for impl in (11, 13):
        sol = BatchedPISO(cd, 3, cg_impl=impl, corrector_steps=1, pressure_non_ortho_steps=1)
        _load_cyl(sol, fx, noisy=1)
        u = sol.u.clone().requires_grad_(True)
        p_out = piso_substep(sol, u, sol.p.clone(), sol.bvel.clone(), float(fx["dt"][0]))[1]
        gen = torch.Generator(device="cuda").manual_seed(3)
        w = 1.0 + torch.rand(p_out.shape, device="cuda", generator=gen)
        (p_out * w).sum().backward()
        torch.cuda.synchronize()
        xb, lam = _adjoint_vectors(sol, 2, 2, 1, 4, 2, 1, 1, 1)[-2:]
        assert torch.allclose(xb, w - w.mean(dim=1, keepdim=True), rtol=0, atol=1e-5)   # the right-hand side is where it belongs
        res[impl] = (p_out.detach().clone(), lam, sol.buffer("iters")[:, 7].clone(), sol.buffer("resid")[:, 7].clone(),
                     sol.buffer("iter_total").clone())
        del sol
    assert (res[11][2] > 10).all() and bool(res[11][1].abs().max() > 0)
    for a, b in zip(res[11], res[13]):
        assert torch.equal(a, b)


def test_env_steps_bit_identical(cyl24):
    from fluidgym_b200.envs.cylinder import CylinderJet2DEnv
    spec, cd = cyl24
    out = {}
    for impl in (11, 13):
        env = CylinderJet2DEnv(n_envs=3, compiled=(spec, cd), cg_impl=impl)
        env.reset(seed=11)
        rows = []
        for k in range(3):
            act = torch.tensor([[0.3 * k], [-0.2], [0.1 * k - 0.5]], device="cuda")
            obs, rew, *_ = env.step(act)
            rows += [obs["velocity"].clone(), obs["pressure"].clone(), rew.clone()]
        rows += [env.solver.u.clone(), env.solver.p.clone(), env.solver.buffer("iter_total").clone()]
        out[impl] = rows
        del env
    for a, b in zip(out[11], out[13]):
        assert torch.equal(a, b)
