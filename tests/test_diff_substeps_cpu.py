"""The ``per_env_substeps`` keyword of every environment family and the per-environment CFL plan generator
(``solver.cfl_substeps_per_env``) on the CPU: the generator's loop runs against a stand-in for ``fgb_plan_substep`` that applies
``solver.cfl_substep`` per environment on host memory; the device planner itself is checked in tests/test_gpu_diff_substeps.py."""
import ctypes as C
import importlib
import inspect

import numpy as np
import pytest

torch = pytest.importorskip("torch")

import fluidgym_b200  # noqa: E402
from fluidgym_b200.envs.common import EpisodeLifecycle  # noqa: E402
from fluidgym_b200.solver import cfl_substep, cfl_substeps, cfl_substeps_per_env  # noqa: E402

FAMILIES = [("cylinder", "CylinderJet2DEnv"), ("cylinder", "CylinderRot2DEnv"), ("airfoil", "Airfoil2DEnv"), ("rbc", "RBC2DEnv"),
            ("rbc3d", "RBC3DEnv"), ("tcf", "TCF3DBottomEnv"), ("tcf", "TCF3DBothEnv"), ("cylinder3d", "CylinderJet3DEnv"),
            ("airfoil3d", "Airfoil3DEnv")]


def _cls(module, name):
    return getattr(importlib.import_module(f"fluidgym_b200.envs.{module}"), name)


@pytest.mark.parametrize("module,name", FAMILIES, ids=[f[1] for f in FAMILIES])
def test_family_accepts_and_stores_the_keyword(module, name):
    cls = _cls(module, name)
    par = inspect.signature(cls.__init__).parameters["per_env_substeps"]
    assert par.default is False
    assert issubclass(cls, EpisodeLifecycle) and cls.per_env_substeps is False and cls.last_substeps_per_env is None
    # the constructor stores it before it builds anything: stopped at its first torch.device / np.zeros call (no solver on the CPU)
    env = object.__new__(cls)

    class Stop(Exception):
        pass

    def stop(*a, **k):
        raise Stop
    for flag in (True, False):
        env.__dict__.clear()
        try:
            with pytest.MonkeyPatch.context() as mp:
                mp.setattr(torch, "device", stop)
                mp.setattr(np, "zeros", stop)
                cls.__init__(env, n_envs=1, per_env_substeps=flag)
        except Exception:
            pass
        assert env.__dict__.get("per_env_substeps") is flag


def test_make_passes_the_keyword_through(monkeypatch):
    fluidgym_b200._register_defaults()
    seen = {}
    for env_id, (entry, _) in list(fluidgym_b200._REGISTRY.items()):
        def fake_init(self, n_envs=1, per_env_substeps=False, differentiable=False, _id=env_id, **kw):
            seen[_id] = (per_env_substeps, differentiable)
        monkeypatch.setattr(entry, "__init__", fake_init)
        fluidgym_b200.make(env_id, n_envs=2, differentiable=True, per_env_substeps=True)
    assert seen and all(v == (True, True) for v in seen.values())


class _PlannerStandIn:
    """fgb_plan_substep on host memory with solver.cfl_substep per environment (the kernel's contract, header fluidgym_b200.h)"""

    def __init__(self):
        self.calls = 0

    def fgb_plan_substep(self, B, maxvel, remaining, cfl, dt, active, nsub, counter, stream):
        self.calls += 1
        arr = lambda p, t: np.ctypeslib.as_array((t * B).from_address(p.value))   # noqa: E731
        mv, rem, d, act, ns = arr(maxvel, C.c_float), arr(remaining, C.c_double), arr(dt, C.c_float), arr(active, C.c_int32), arr(nsub, C.c_int32)
        cnt = np.ctypeslib.as_array((C.c_int32 * 1).from_address(counter.value))
        for e in range(B):
            r = float(rem[e])
            on = r > 0.0 and not abs(r) <= 1e-8
            d[e], act[e] = 0.0, int(on)
            if on:
                ts = cfl_substep(r, cfl, float(mv[e]))
                rem[e] = r - ts
                d[e] = np.float32(ts)
                ns[e] += 1
                cnt[0] += 1
        return 0


@pytest.mark.parametrize("dt,cfl", [(0.01, 0.8), (0.05, 0.1), (0.25, 0.8), (1e-3, 0.5)])
def test_per_env_generator_equals_cfl_substeps_alone(dt, cfl):
    rng = np.random.default_rng(11)
    B, R = 8, 400
    vel = (cfl / dt * 10.0 ** rng.uniform(-1.5, 1.5, size=(B, R))).astype(np.float32)
    vel[0] = 0.0                                                          # a vanishing velocity: one substep
    r = [0]

    def max_velocity_env():
        r[0] += 1
        return torch.from_numpy(vel[:, r[0] - 1].copy())
    lib = _PlannerStandIn()
    got = [[] for _ in range(B)]
    rounds = 0
    for dtv, act in cfl_substeps_per_env(lib, B, dt, cfl, max_velocity_env, "cpu", None):
        assert dtv.dtype == torch.float32 and act.dtype == torch.int32 and dtv.shape == act.shape == (B,)
        assert (dtv[act == 0] == 0).all()
        for e in np.nonzero(act.numpy())[0]:
            got[e].append(float(dtv[e]))
        rounds += 1
    for e in range(B):
        it = iter(vel[e])
        want = list(cfl_substeps(dt, cfl, lambda: float(next(it))))
        assert got[e] == want, e
    assert rounds == max(len(g) for g in got) and lib.calls == rounds + 1          # one planner call (and count read) per round + the last
