"""The episode lifecycle every environment family shares (envs/common.py::EpisodeLifecycle) and the adaptive CFL substep plan
(solver.py::cfl_substep / cfl_substeps), on the CPU without a solver.

The plan is compared with the arithmetic the environments carried before it was shared, kept here verbatim: sizes and counts must
be equal, not close -- a last-bit difference changes the substeps of a differentiable rollout and with them its gradients.  The
lifecycle is checked on every family class, each built with ``object.__new__`` and the few attributes the shared helpers read:
the reference's error strings (tests/env_utils/test_fluid_env.py) and the seeded action stream."""
import re

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from fluidgym_b200.solver import cfl_substep, cfl_substeps  # noqa: E402


# ---- the substep plan ------------------------------------------------------------------------------------------------------------
def _reference_plan(dt, cfl, max_velocity):
    """The loop of SIM.py:2004-2031 as envs/common.py, rbc.py, rbc3d.py, tcf.py and cylinder3d.py wrote it (the 3-D files with
    ``float(int(np.ceil(..)))``, the same value): -> sizes handed to the substep"""
    remaining, sizes = float(dt), []
    while remaining > 0.0 and not abs(remaining) <= 1e-8:
        mv = max_velocity()
        if abs(mv) <= 1e-8:
            ts = remaining
        else:
            mts = np.float32(cfl) / np.float32(mv)
            ts = remaining if float(mts) >= remaining else remaining / float(np.ceil(np.float32(remaining) / mts))
        remaining -= ts
        sizes.append(float(np.float32(ts)))
    return sizes


def _reference_extruded_size(rem, cfl, mv):
    """ExtrudedStepping.single_step's per-environment size: ``rem`` a float64 array element, ``mv`` a float32 array element"""
    if abs(mv) <= 1e-8:
        return rem
    mts = np.float32(cfl) / mv
    return rem if float(mts) >= rem else rem / float(np.ceil(np.float32(rem) / mts))


def _velocities(values):
    it = iter(values)
    return lambda: float(next(it))


def _boundary_velocities(dt, cfl):
    """float32 velocities within 3 ulps of those for which dt is an exact multiple k of the CFL step: where the float32 ratio
    and its ceiling decide the substep count"""
    out = []
    for k in range(1, 40):
        v = np.float32(cfl * k / dt)
        lo, hi = [v], [v]
        for _ in range(3):
            lo.append(np.nextafter(lo[-1], np.float32(0)))
            hi.append(np.nextafter(hi[-1], np.float32(np.inf)))
        out += lo[1:] + hi
    return out


def _cases():
    rng = np.random.default_rng(20261020)
    cases = []
    for _ in range(300):                                                # float32 velocities, as the device maxima are
        dt = float(10.0 ** rng.uniform(-4, 0))
        cfl = float(rng.choice([0.1, 0.8, rng.uniform(0.05, 1.0)]))
        mv = np.float32(cfl / dt * 10.0 ** rng.uniform(-1, 2))           # 1 to ~100 substeps
        cases.append((dt, cfl, [mv] * 1000))
    for _ in range(100):                                                # a velocity that changes between substeps
        dt = float(10.0 ** rng.uniform(-3, 0))
        cases.append((dt, 0.8, (0.8 / dt * 10.0 ** rng.uniform(-1, 1.5, size=1000)).astype(np.float32)))
    for dt, cfl in ((0.01, 0.8), (0.05, 0.8), (0.06, 0.1), (0.25, 0.8), (1e-3, 0.1)):
        cases += [(dt, cfl, [v] * 1000) for v in _boundary_velocities(dt, cfl)]
    f32 = np.float32
    cases += [
        (0.01, 0.8, [f32(0.0)]), (0.01, 0.8, [f32(1e-8)]), (0.01, 0.8, [f32(5e-9)]),            # max velocity <= 1e-8: one substep
        (0.01, 0.8, [np.nextafter(f32(1e-8), f32(1))] * 10),                                      # just above it
        (0.01, 0.8, [f32(80.0)]), (0.01, 0.8, [f32(79.99)] * 10),                                # mts >= remaining / just below
        (1.0000001e-8, 0.8, [f32(1.0)] * 10), (1e-8, 0.8, []), (9e-9, 0.8, []), (0.0, 0.8, []),  # remainders around 1e-8
        (2.5e-8, 0.8, [f32(4e7)] * 10), (3e-8, 0.8, [f32(8e7), f32(0.0)]),
        (0.01, 0.8, [f32(1e3), f32(1e-9), f32(10.0)] * 10), (0.01, 0.8, [f32(400.0), f32(7.0), f32(2e3)] * 100),
    ]
    return cases


def test_cfl_substeps_equal_the_reference_arithmetic():
    for dt, cfl, vel in _cases():
        want = _reference_plan(dt, cfl, _velocities(vel))
        got = list(cfl_substeps(dt, cfl, _velocities(vel)))
        assert len(got) == len(want) and got == want, (dt, cfl)


def test_cfl_substep_equals_the_extruded_per_environment_arithmetic():
    rng = np.random.default_rng(7)
    rem = np.concatenate([10.0 ** rng.uniform(-8, 0, size=2000), [1.0000001e-8, 2e-8, 0.01, 0.05]])
    mv = np.concatenate([(10.0 ** rng.uniform(-10, 4, size=2000)), [0.0, 1e-8, 5e-9, 80.0]]).astype(np.float32)
    for cfl in (0.1, 0.8):
        pairs = list(zip(rem, mv)) + [(np.float64(0.05), v) for v in _boundary_velocities(0.05, cfl)]
        for r, m in pairs:
            assert cfl_substep(float(r), cfl, float(m)) == _reference_extruded_size(r, cfl, m), (r, m, cfl)


# ---- the episode lifecycle of every family -----------------------------------------------------------------------------------
FAMILIES = [("cylinder", "CylinderJet2DEnv", (2, 1)), ("cylinder", "CylinderRot2DEnv", (2, 1)), ("airfoil", "Airfoil2DEnv", (2, 3)),
            ("rbc", "RBC2DEnv", (2, 12, 1)), ("rbc3d", "RBC3DEnv", (2, 64, 1)), ("tcf", "TCF3DBottomEnv", (2, 256, 1)),
            ("tcf", "TCF3DBothEnv", (2, 512, 1)), ("cylinder3d", "CylinderJet3DEnv", (2, 8, 1)), ("airfoil3d", "Airfoil3DEnv", (2, 4, 3))]


def _standin(module, name, shape):
    """the family class without its constructor, with what the lifecycle helpers read (action shape as the default configuration)"""
    import importlib
    e = object.__new__(getattr(importlib.import_module(f"fluidgym_b200.envs.{module}"), name))
    e.device = torch.device("cpu")
    e.n_envs, e.episode_length, e.dt, e.step_length = shape[0], 3, 0.05, 0.25
    e._zero_action = torch.zeros(shape)
    e.solver = object()                                                 # keeps no residual table: the solve watch has nothing to read
    return e


@pytest.mark.parametrize("module,name,shape", FAMILIES, ids=[f[1] for f in FAMILIES])
def test_lifecycle_error_strings(module, name, shape):
    e = _standin(module, name, shape)
    with pytest.raises(ValueError, match=re.escape("Seed must be provided either during reset or by calling seed().")):
        e.reset()
    with pytest.raises(RuntimeError, match=re.escape("Environment must be seeded before sampling actions")):
        e.sample_action()
    with pytest.raises(RuntimeError, match=re.escape("Environment must be reset before stepping. Call 'reset()' before'step()'.")):
        e.step(torch.zeros(shape))
    e._reset_called = True
    wrong = torch.zeros(shape[0], shape[1] + 1, *shape[2:])
    with pytest.raises(ValueError, match=re.escape(f"Action shape {wrong.shape} does not match expected shape {torch.Size(shape)}.")):
        e.step(wrong)
    e._n_steps = e.episode_length
    with pytest.raises(RuntimeError, match=re.escape("Episode has already terminated. Call 'reset()' first.")):
        e.step(torch.zeros(shape))


@pytest.mark.parametrize("module,name,shape", FAMILIES, ids=[f[1] for f in FAMILIES])
def test_lifecycle_seed_action_and_truncation(module, name, shape):
    e = _standin(module, name, shape)
    assert (e._reset_called, e._seed, e._n_steps, e.last_substeps, e._dstate) == (False, None, 0, 0, None)
    assert e.n_sim_steps == 5
    e.seed(11)
    a = e.sample_action()
    assert torch.equal(a, torch.rand(shape, generator=torch.Generator().manual_seed(11)) * 2 - 1)
    assert int(e._np_rng.integers(0, 1 << 30)) == int(np.random.default_rng(11).integers(0, 1 << 30))
    e._reset_called = True
    got = e._begin_step(a.double().tolist())
    assert got.dtype == torch.float32 and torch.equal(got, a)
    assert [e._end_step() for _ in range(e.episode_length)] == [False, False, True] and e._n_steps == e.episode_length
