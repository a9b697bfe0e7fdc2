"""Per-environment adaptive substeps of batched differentiable rollouts (``per_env_substeps=True``) on the GPU.

1. the device planner ``fgb_plan_substep`` (through ``solver.cfl_substeps_per_env``) equals ``solver.cfl_substep`` under ``==``;
2. every recorded substep node with an environment mask: skipped environments are the identity in both directions, the others equal
   the unmasked call (forward bit for bit, gradients up to the float atomics of the adjoint scatters);
3. an environment of a diverging batch equals the same environment run alone (``n_envs=1``, default settings): substep sizes, state,
   observations, reward and gradients -- and the shared plan of the default mode does not;
4. in plain mode the keyword changes nothing.
Small grids as in the other GPU tests.  Observed differences are printed, and written as JSON to $FGB_REPORT_DIR/diff_substeps_observed.json
when FGB_REPORT_DIR is set."""
import json
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

FAMILIES = {   # id, constructor keywords (small grids, short steps), the field whose initial value gets a gradient
    "CylinderJet2D": ("CylinderJet2D-easy-v0", dict(step_length=0.05), "u"),
    "RBC2D": ("RBC2D-easy-v0", dict(step_length=0.1), "T"),
    "TCF": ("TCFSmall3D-both-easy-v0", dict(resolution_x_z=32, resolution_y=33), "u"),
    "RBC3D": ("RBC3D-easy-v0", dict(n_heaters=4, resolution=4, step_length=0.1), "T"),
    "CylinderJet3D": ("CylinderJet3D-easy-v0", dict(resolution=8, n_jets=8, step_length=0.05), "u"),
    "Airfoil2D": ("Airfoil2D-easy-v0", dict(step_length=0.05), "u"),
}
SCALES = (1.0, 2.0, 3.0)          # velocity scale of environment b: different CFL limits
OBSERVED = {}
# Gradients are compared with a relative L2 bar of GRAD_TOL, or 10x the difference between two identical runs where that is larger.  The
# adjoints scatter with float atomics whose order varies between launches, and the transposed Krylov solves stop at their tolerance, so
# gradients of the non-orthogonal paths (cylinder, airfoil, extruded) differ between identical calls well above 1e-6; the difference of
# two identical runs is recorded next to every comparison.
GRAD_TOL = 1e-3
# State, observations and reward: kernels alone are bit-identical between a batch and a single environment; the 2-D outflow / flux
# balance hook sums boundary fluxes with float32 torch reductions whose order depends on the batch size, and the Krylov solves of the
# following substeps carry those last bits up to their tolerance.
STATE_TOL = 5e-4


def _record(name, **values):
    OBSERVED.setdefault(name, {}).update(values)
    print(name, values)
    out = os.environ.get("FGB_REPORT_DIR")
    if out:
        os.makedirs(out, exist_ok=True)
        with open(os.path.join(out, "diff_substeps_observed.json"), "w") as f:
            json.dump(OBSERVED, f, indent=1, sort_keys=True)


def _rel(a, b):
    a, b = a.detach().double().flatten(), b.detach().double().flatten()
    return float((a - b).norm() / b.norm().clamp_min(1e-300))


# ---- 1. planner ------------------------------------------------------------------------------------------------------------------
def _plan_rounds(lib, dts, cfl, velocities, dev):
    """fgb_plan_substep rounds for environments with their own initial time dts[e] and per-round maximum velocities
    velocities[e][r] (the loop of solver.cfl_substeps_per_env, which starts every environment at one dt) -> sizes per environment"""
    import ctypes as C

    from fluidgym_b200 import native
    from fluidgym_b200.solver import _ptr
    B, width = len(dts), max(len(v) for v in velocities) + 1
    vel = np.zeros((B, width), np.float32)
    for e, v in enumerate(velocities):
        vel[e, :len(v)] = np.asarray(v, np.float32)
    remaining = torch.tensor(dts, dtype=torch.float64, device=dev)
    nsub = torch.zeros(B, dtype=torch.int32, device=dev)
    count = torch.zeros(1, dtype=torch.int32, device=dev)
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    got, done = [[] for _ in range(B)], np.zeros(B, bool)
    for r in range(10 ** 6):
        mv = torch.from_numpy(vel[:, min(r, width - 1)].copy()).to(dev)
        dtv = torch.empty(B, dtype=torch.float32, device=dev)
        act = torch.empty(B, dtype=torch.int32, device=dev)
        count.zero_()
        native.check(lib.fgb_plan_substep(B, _ptr(mv), _ptr(remaining), float(cfl), _ptr(dtv), _ptr(act), _ptr(nsub), _ptr(count), stream),
                     "fgb_plan_substep")
        if int(count.item()) == 0:
            break
        d, a = dtv.cpu().numpy(), act.cpu().numpy().astype(bool)
        assert not (a & done).any() and (d[~a] == 0).all()          # finished environments stay finished, with dt = 0
        done |= ~a
        for e in np.nonzero(a)[0]:
            got[e].append(float(d[e]))
    assert nsub.cpu().tolist() == [len(g) for g in got]
    return got, r


def test_planner_equals_cfl_substep():
    """fgb_plan_substep against solver.cfl_substep (through cfl_substeps) under ==, per environment and round, on the cases of
    test_env_lifecycle_cpu.py: seeded random inputs, velocities within 3 ulps of exact multiples, vanishing velocities, remainders
    around 1e-8 and velocities that change between substeps"""
    from test_env_lifecycle_cpu import _cases, _velocities

    from fluidgym_b200 import native
    from fluidgym_b200.solver import cfl_substeps
    lib, dev = native.load_for("cuda:0"), torch.device("cuda:0")
    groups = {}
    for dt, cfl, vel in _cases():
        groups.setdefault(cfl, []).append((dt, vel))
    n_rounds = 0
    for cfl, cases in groups.items():
        want = [list(cfl_substeps(dt, cfl, _velocities(vel))) for dt, vel in cases]
        got, r = _plan_rounds(lib, [dt for dt, _ in cases], cfl, [v for _, v in cases], dev)
        n_rounds += r
        for e in range(len(cases)):
            assert got[e] == want[e], (cases[e][0], cfl, got[e][:5], want[e][:5])
    _record("planner", cases=sum(len(c) for c in groups.values()), rounds=n_rounds)


def test_cfl_substeps_per_env_equals_cfl_substeps_per_environment():
    """the generator itself (one dt for the batch) against cfl_substeps run on every environment alone"""
    from fluidgym_b200 import native
    from fluidgym_b200.solver import cfl_substeps, cfl_substeps_per_env
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(3)
    for dt, cfl in ((0.01, 0.8), (0.05, 0.1), (0.25, 0.8)):
        vel = (cfl / dt * 10.0 ** rng.uniform(-1, 1.5, size=(16, 200))).astype(np.float32)
        r = [0]

        def mv():
            r[0] += 1
            return torch.from_numpy(vel[:, r[0] - 1].copy()).to(dev)
        got = [[] for _ in range(16)]
        for dtv, act in cfl_substeps_per_env(native.load_for(dev), 16, dt, cfl, mv, dev, torch.cuda.current_stream(dev).cuda_stream):
            for e in np.nonzero(act.cpu().numpy())[0]:
                got[e].append(float(dtv[e].cpu()))
        for e in range(16):
            it = iter(vel[e])
            assert got[e] == list(cfl_substeps(dt, cfl, lambda: float(next(it)))), e


# ---- helpers: environments in diverging states ---------------------------------------------------------------------------------
def _max_velocity(env):
    """each environment's maximum velocity as the planner sees it"""
    s = env.solver
    if hasattr(s, "xtables") or type(s).__name__ == "BatchedPISO":
        return s.max_velocity()
    minv, b_minv = s._tab["minv"].reshape(1, 3, -1), s._tab["b_minv"].reshape(1, 3, -1)
    return torch.maximum((minv * s.u).abs().amax(dim=(1, 2)), (b_minv * s.bvel).abs().amax(dim=(1, 2)))


def _make(name, B, **kw):
    import fluidgym_b200 as fg
    env_id, ekw, _ = FAMILIES[name]
    env = fg.make(env_id, n_envs=B, **{**ekw, **kw})
    env.reset(seed=0)
    return env


def _diverge(env):
    """scale environment b's velocity by SCALES[b] and pick a CFL number that splits environment 0's first solver step into two substeps"""
    s = env.solver
    with torch.no_grad():
        s.u.mul_(torch.tensor(SCALES, device=s.u.device).view(-1, *[1] * (s.u.dim() - 1)))
    mv = float(_max_velocity(env)[0])
    return env.dt * mv / 1.5


_STATE = ("u", "p", "bvel", "T", "sbval")


def _leaf(env, name):
    """the differentiable initial field of the family (velocity or temperature)"""
    s = env.solver
    if hasattr(env, "mark_state_differentiable"):
        out = env.mark_state_differentiable()
        return out[1] if FAMILIES[name][2] == "T" else out
    if FAMILIES[name][2] == "T":                       # RBC2D: (u, p, T, sbval)
        T = s.T.clone().requires_grad_(True)
        env._dstate = (s.u.clone(), s.p.clone(), T, s.sbval.clone())
        return T
    u = s.u.clone().requires_grad_(True)                # cylinder / airfoil: (u, p, bvel, last_control)
    env._dstate = (u, s.p.clone(), s.bvel.clone(), env.last_control.clone())
    return u


def _rows(x, b):
    if isinstance(x, dict):
        return [t for k in sorted(x) for t in _rows(x[k], b)]
    return [x[b]]


class _Plans:
    """records the substep sizes the rollouts use: shared plans (cfl_substeps, per family module) and per-environment rounds"""

    def __init__(self, monkeypatch):
        import importlib

        from fluidgym_b200 import solver
        self.shared, self.rounds = [], []
        for mod in ("common", "rbc", "tcf", "rbc3d", "cylinder3d"):
            m = importlib.import_module(f"fluidgym_b200.envs.{mod}")
            monkeypatch.setattr(m, "cfl_substeps", self._shared(solver.cfl_substeps))
        from fluidgym_b200.envs import common
        monkeypatch.setattr(common, "cfl_substeps_per_env", self._per_env(solver.cfl_substeps_per_env))

    def _shared(self, fn):
        def wrapped(*a, **k):
            for ts in fn(*a, **k):
                self.shared.append(float(np.float32(ts)))
                yield ts
        return wrapped

    def _per_env(self, fn):
        def wrapped(*a, **k):
            for dtv, act in fn(*a, **k):
                self.rounds.append((dtv.cpu().numpy().copy(), act.cpu().numpy().copy()))
                yield dtv, act
        return wrapped

    def env_sizes(self, b):
        return [float(d[b]) for d, a in self.rounds if a[b]]


# ---- 2. masked nodes ---------------------------------------------------------------------------------------------------------------
def _node_inputs(name):
    """(apply(inputs, active) -> outputs, differentiable inputs, index of the previous pressure or None) of the family's substep node"""
    from fluidgym_b200 import autograd as ag
    env = _make(name, 3, differentiable=True)
    _diverge(env)
    s = env.solver
    dt = torch.full((3,), env.dt / 4, device="cuda")
    if name == "CylinderJet2D":
        return (lambda x, a: ag.piso_substep(s, *x, dt, active=a)), [s.u.clone(), s.p.clone(), s.bvel.clone()], 1
    if name == "RBC2D":
        return (lambda x, a: ag.piso_substep_scalar(s, *x, dt, env.buoyancy_factor, active=a)), \
            [s.u.clone(), s.p.clone(), s.bvel.clone(), s.T.clone(), s.sbval.clone()], 1
    if name == "TCF":
        src = env._forcing_torch(s.u)
        return (lambda x, a: ag.piso_substep_3d(s, *x, dt, src, active=a)), [s.u.clone(), s.p.clone(), s.bvel.clone()], None
    if name == "RBC3D":
        return (lambda x, a: ag.piso_substep_scalar_3d(s, *x, dt, active=a)), \
            [s.u.clone(), s.p.clone(), s.bvel.clone(), s.T.clone(), s.sbval.clone()], None
    return (lambda x, a: ag.piso_substep_extruded(s, *x, dt, active=a)), [s.u.clone(), s.p.clone(), s.bvel.clone()], 1


@pytest.mark.parametrize("name", ["CylinderJet2D", "RBC2D", "TCF", "RBC3D", "CylinderJet3D"])
def test_masked_node(name):
    fn, xs, p_idx = _node_inputs(name)
    active = torch.tensor([1, 0, 1], dtype=torch.int32, device="cuda")
    outs = {}
    for key, a in (("all", None), ("repeat", None), ("masked", active)):
        ins = [x.detach().clone().requires_grad_(True) for x in xs]
        y = fn(ins, a)
        g = torch.Generator(device="cuda").manual_seed(5)
        cot = [torch.randn(t.shape, device="cuda", generator=g) for t in y]
        grads = torch.autograd.grad(y, ins, grad_outputs=cot, allow_unused=True)
        torch.cuda.synchronize()
        outs[key] = ([t.detach() for t in y], grads, cot, ins)
    y_all, g_all, _, _ = outs["all"]
    y_m, g_m, cot, ins = outs["masked"]
    n_y = len(y_m)
    for k in range(n_y):                                            # forward: 0 and 2 as unmasked, 1 unchanged
        assert torch.equal(y_m[k][0], y_all[k][0]) and torch.equal(y_m[k][2], y_all[k][2]), k
    # outputs (u, p[, T]) correspond to inputs 0, 1[, 3]
    out_in = [0, 1, 3][:n_y]
    for k, i in enumerate(out_in):
        assert torch.equal(y_m[k][1], xs[i][1]), k
    # backward: identity cotangents of environment 1
    assert torch.equal(g_m[0][1], cot[0][1])                                          # u_bar = u_out_bar
    if p_idx is not None:
        assert torch.equal(g_m[1][1], cot[1][1])                                      # p_prev_bar = p_out_bar
    assert torch.count_nonzero(g_m[2][1]) == 0                                        # bvel_bar = 0
    if len(xs) == 5:
        assert torch.equal(g_m[3][1], cot[2][1])                                      # T_bar = T_out_bar
        assert torch.count_nonzero(g_m[4][1]) == 0                                    # sbval_bar = 0
    worst, noise = 0.0, 0.0
    for ga, gr, gm in zip(g_all, outs["repeat"][1], g_m):
        if ga is None:
            continue
        for b in (0, 2):
            if float(ga[b].norm()) > 0:
                worst = max(worst, _rel(gm[b], ga[b]))
                noise = max(noise, _rel(gr[b], ga[b]))
    _record("masked_node", **{name: dict(grad_rel_l2=worst, repeat_rel_l2=noise)})
    assert worst <= max(GRAD_TOL, 10 * noise), (worst, noise)


# ---- 3. batch equals alone -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(FAMILIES))
def test_batch_equals_alone(name, monkeypatch):
    plans = _Plans(monkeypatch)
    env = _make(name, 3, differentiable=True, per_env_substeps=True)
    cfl = _diverge(env)
    env.cfl = cfl
    start = {k: getattr(env.solver, k).clone() for k in _STATE if isinstance(getattr(env.solver, k, None), torch.Tensor)}
    control = env.last_control.clone() if isinstance(getattr(env, "last_control", None), torch.Tensor) else None
    g = torch.Generator(device="cuda").manual_seed(1)
    action = (torch.rand(env._zero_action.shape, device="cuda", generator=g) * 2 - 1).requires_grad_(True)
    x0 = _leaf(env, name)
    obs, reward, *_ = env.step(action)
    g_a, g_x = torch.autograd.grad(reward.sum(), [action, x0])
    torch.cuda.synchronize()
    per_env = env.last_substeps_per_env.cpu().tolist()
    assert env.per_env_substeps and len(set(per_env)) > 1, per_env
    assert env.last_substeps == len(plans.rounds)
    batch = dict(state={k: getattr(env.solver, k).clone() for k in start}, obs=obs, reward=reward.detach(), g_a=g_a, g_x=g_x)
    sizes = [plans.env_sizes(b) for b in range(3)]
    assert per_env == [len(s) for s in sizes]

    single = _make(name, 1, differentiable=True)
    single.cfl = cfl
    worst = dict(state=0.0, obs=0.0, reward=0.0, grad_action=0.0, grad_x0=0.0, grad_repeat=0.0)
    bitwise = True
    alone_sizes, first = [], None
    for b in (0, 1, 2, 0):                              # environment 0 twice: the gradient difference of two identical runs
        repeat = first is not None and b == 0
        plans.shared.clear()
        single.reset(seed=0)
        with torch.no_grad():
            for k, t in start.items():
                getattr(single.solver, k).copy_(t[b:b + 1])
        if control is not None:
            single.last_control = control[b:b + 1].clone()
        single._dstate = None
        a1 = action.detach()[b:b + 1].clone().requires_grad_(True)
        x1 = _leaf(single, name)
        obs1, r1, *_ = single.step(a1)
        h_a, h_x = torch.autograd.grad(r1.sum(), [a1, x1])
        torch.cuda.synchronize()
        if repeat:
            worst["grad_repeat"] = max(_rel(h_a[0], first[0]), _rel(h_x[0], first[1]))
            continue
        if b == 0:
            first = (h_a[0], h_x[0])
        alone_sizes.append(list(plans.shared))
        assert sizes[b] == plans.shared, (b, sizes[b][:4], plans.shared[:4])
        for k in start:
            bitwise &= torch.equal(batch["state"][k][b], getattr(single.solver, k)[0])
            worst["state"] = max(worst["state"], _rel(batch["state"][k][b], getattr(single.solver, k)[0]))
        for t_b, t_1 in zip(_rows(batch["obs"], b), _rows(obs1, 0)):
            bitwise &= torch.equal(t_b, t_1)
            worst["obs"] = max(worst["obs"], _rel(t_b, t_1))
        bitwise &= torch.equal(batch["reward"][b], r1.detach()[0])
        worst["reward"] = max(worst["reward"], _rel(batch["reward"][b], r1.detach()[0]))
        worst["grad_action"] = max(worst["grad_action"], _rel(g_a[b], h_a[0]))
        worst["grad_x0"] = max(worst["grad_x0"], _rel(g_x[b], h_x[0]))
    _record("batch_equals_alone", **{name: dict(worst, bitwise_state_obs_reward=bool(bitwise), substeps_per_env=per_env)})
    assert worst["state"] <= STATE_TOL and worst["obs"] <= STATE_TOL and worst["reward"] <= STATE_TOL, worst
    bar = max(GRAD_TOL, 10 * worst["grad_repeat"])
    assert worst["grad_action"] <= bar and worst["grad_x0"] <= bar, worst

    # non-vacuity: the shared plan of the default mode gives at least one environment other substeps than it takes alone
    shared = _make(name, 3, differentiable=True)
    shared.cfl = cfl
    with torch.no_grad():
        for k, t in start.items():
            getattr(shared.solver, k).copy_(t)
    if control is not None:
        shared.last_control = control.clone()
    shared._dstate = None
    plans.shared.clear()
    shared.step(action.detach())
    assert shared.last_substeps_per_env is None
    assert any(plans.shared != alone_sizes[b] for b in range(3))


# ---- 4. plain mode ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["CylinderJet2D", "RBC2D", "TCF", "RBC3D", "CylinderJet3D"])
def test_plain_mode_ignores_the_keyword(name):
    out = []
    for flag in (False, True):
        env = _make(name, 3, per_env_substeps=flag)
        _diverge(env)
        g = torch.Generator(device="cuda").manual_seed(2)
        obs, reward, *_ = env.step(torch.rand(env._zero_action.shape, device="cuda", generator=g) * 2 - 1)
        torch.cuda.synchronize()
        assert env.per_env_substeps is flag and env.last_substeps_per_env is None
        out.append((_rows(obs, slice(None)), reward, env.solver.u.clone(), env.last_substeps))
    for a, b in zip(out[0][0], out[1][0]):
        assert torch.equal(a, b)
    assert torch.equal(out[0][1], out[1][1]) and torch.equal(out[0][2], out[1][2]) and out[0][3] == out[1][3]
