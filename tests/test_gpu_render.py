"""env.render_field / env.render on the GPU (fgb_render_gather / fgb_render_colour) for every family: the resampled field equals
the host CSR map applied in float64 to the solver state, the colours equal the numpy specification, environments are
independent of the batch, and rendering leaves the run untouched (plain and differentiable mode)."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

B = 3
CASES = {"CylinderJet2D-easy-v0": {}, "CylinderRot2D-easy-v0": {}, "Airfoil2D-easy-v0": {}, "RBC2D-easy-v0": {}, "RBC3D-easy-v0": {},
         "CylinderJet3D-easy-v0": {"resolution": 8}, "Airfoil3D-easy-v0": {"res_z": 8}, "TCFSmall3D-bottom-easy-v0": {},
         "TCFSmall3D-both-easy-v0": {}}
_ENVS, _MAPS = {}, {}


def _env(env_id):
    if env_id not in _ENVS:
        import fluidgym_b200 as fg
        env = fg.make(env_id, n_envs=B, use_marl=False, **CASES[env_id])
        env.reset(seed=11)
        env.step(env.sample_action())
        _ENVS[env_id] = env
    return _ENVS[env_id]


def _host(t):
    return t.detach().double().cpu().numpy()


def _reference(env, field, plane):
    """float64 [B, H, W]: the host CSR map applied to the state pulled to the host"""
    planes = env._render_planes()
    plane = None if planes is None else (planes[1] if plane is None else plane)
    key = (id(env), plane)
    if key not in _MAPS:
        _MAPS[key] = env._build_render_map(plane)
    m = _MAPS[key]
    s = env.solver
    with torch.no_grad():
        src = {"pressure": lambda: s.p, "temperature": lambda: s.T, "vorticity": lambda: s.vorticity(), "q_criterion": lambda: s.q_criterion()}
        if field == "velocity_magnitude" or field.startswith("velocity_"):
            u = _host(s.u)
            chans = range(u.shape[1]) if field == "velocity_magnitude" else ["xyz".index(field[-1])]
            f = [u[:, c] for c in chans]
        else:
            f = [_host(src[field]()).reshape(B, -1)]
    R = m.matrix(f[0].shape[1])
    vals = [(R @ x.T).T for x in f]
    out = np.sqrt(sum(v * v for v in vals)) if field == "velocity_magnitude" else vals[0]
    return out.reshape(B, *m.shape)


@pytest.mark.parametrize("env_id", list(CASES))
def test_render_field_equals_host_map(env_id):
    env = _env(env_id)
    planes = env._render_planes()
    for k, field in enumerate(env.render_fields):
        for plane in ([None] if planes is None or k else [None, 0]):
            img = env.render_field(field, plane=plane)
            assert img.dtype == torch.float32 and img.device == env.device and img.shape[0] == B
            ref = _reference(env, field, plane)
            got = _host(img)
            assert got.shape == ref.shape
            assert np.linalg.norm(got - ref) <= 1e-6 * np.linalg.norm(ref) + 1e-30, (field, plane)
    with pytest.raises(ValueError, match="renders"):
        env.render_field("no_such_field")
    with pytest.raises(ValueError, match="plane"):
        env.render_field(plane=10 ** 6)


@pytest.mark.parametrize("env_id", list(CASES))
def test_render_equals_colour_specification(env_id):
    from fluidgym_b200.envs.common import _SIGNED_FIELDS
    from fluidgym_b200.render import DIVERGING, SEQUENTIAL, colour_bins
    env = _env(env_id)
    for field in env.render_fields:
        signed = field in _SIGNED_FIELDS
        lut = DIVERGING if signed else SEQUENTIAL
        img = _host(env.render_field(field)).astype(np.float32)
        for kw in ({}, {"vmin": -0.5, "vmax": 1.5}):
            rgb = env.render(field, **kw)
            assert rgb.dtype == torch.uint8 and rgb.device == env.device and tuple(rgb.shape) == img.shape + (3,)
            if kw:
                lo, hi = np.float32(kw["vmin"]), np.float32(kw["vmax"])
            else:
                flat = img.reshape(B, -1)
                lo, hi = flat.min(1), flat.max(1)
                if signed:
                    hi = np.maximum(np.abs(lo), np.abs(hi))
                    lo = -hi
            bins = colour_bins(img, lo, hi)
            got = rgb.cpu().numpy()
            off = ~np.all(got == lut[bins], axis=-1)
            near = np.all(got == lut[np.clip(bins + 1, 0, 255)], axis=-1) | np.all(got == lut[np.clip(bins - 1, 0, 255)], axis=-1)
            assert not (off & ~near).any(), (field, kw)                    # at most one bin, at bin edges only
            assert off.sum() <= 1e-4 * off.size, (field, kw, int(off.sum()))


@pytest.mark.parametrize("env_id", ["CylinderJet2D-easy-v0", "RBC2D-easy-v0", "RBC3D-easy-v0", "CylinderJet3D-easy-v0",
                                    "TCFSmall3D-bottom-easy-v0"])
def test_batch_independence(env_id):
    import fluidgym_b200 as fg
    env = _env(env_id)
    one = fg.make(env_id, n_envs=1, use_marl=False, **CASES[env_id])
    e = 1
    for name in ("u", "p", "bvel", "T", "sbval"):
        if hasattr(env.solver, name):
            getattr(one.solver, name).copy_(getattr(env.solver, name)[e:e + 1])
    for field in env.render_fields:
        assert torch.equal(env.render_field(field)[e], one.render_field(field)[0]), field
        assert torch.equal(env.render(field)[e], one.render(field)[0]), field


def _run(env_id, kw, with_render, differentiable):
    """reset, step, (render every field), step -> everything the second step returns, the state and the action gradient"""
    import fluidgym_b200 as fg
    env = fg.make(env_id, n_envs=2, use_marl=False, differentiable=differentiable, **kw)
    env.reset(seed=5)
    g = torch.Generator(device="cuda").manual_seed(3)
    shape = env._zero_action.shape
    a1 = (torch.rand(shape, device="cuda", generator=g) * 2 - 1).requires_grad_(differentiable)
    a2 = (torch.rand(shape, device="cuda", generator=g) * 2 - 1).requires_grad_(differentiable)
    env.step(a1)
    if with_render:
        for field in env.render_fields:
            env.render(field)
            env.render_field(field)
    obs, reward, _, _, _ = env.step(a2)
    grad = torch.autograd.grad(reward.sum(), [a1, a2], allow_unused=True) if differentiable else None
    torch.cuda.synchronize()
    return obs, reward.detach(), env.solver.u.clone(), env.solver.p.clone(), grad


@pytest.mark.parametrize("env_id,kw,differentiable", [
    ("CylinderJet2D-easy-v0", {}, False), ("TCFSmall3D-bottom-easy-v0", {"resolution_x_z": 32, "resolution_y": 33}, False),
    ("CylinderJet2D-easy-v0", {}, True), ("TCFSmall3D-bottom-easy-v0", {"resolution_x_z": 32, "resolution_y": 33}, True)])
def test_rendering_does_not_perturb_the_run(env_id, kw, differentiable):
    ref = _run(env_id, kw, False, differentiable)
    got = _run(env_id, kw, True, differentiable)
    for k in ref[0]:
        assert torch.equal(ref[0][k], got[0][k]), k
    for a, b in zip(ref[1:4], got[1:4]):
        assert torch.equal(a, b)
    if differentiable:                                  # the adjoint scatters with atomics: equal up to summation order
        assert ref[4][1] is not None
        for a, b in zip(ref[4], got[4]):
            assert (a is None) == (b is None)
            if a is not None:
                assert float((a - b).abs().max()) <= 1e-4 * float(a.abs().max())


def test_torchrl_from_pixels():
    import fluidgym_b200 as fg
    from fluidgym_b200.integration import TorchRLFluidEnv
    env = fg.make("CylinderJet2D-easy-v0", n_envs=3)
    tenv = TorchRLFluidEnv(env, from_pixels=True)
    assert tuple(tenv.observation_spec["pixels"].shape) == (3, 96, 515, 3)
    tenv.set_seed(0)
    td = tenv.reset()
    px = td["pixels"]
    assert tuple(px.shape) == (3, 96, 515, 3) and px.dtype == torch.uint8 and px.device == env.device
    out = tenv.step({"action": torch.zeros(3, 1, device=env.device)})["next"]
    assert tuple(out["pixels"].shape) == (3, 96, 515, 3) and out["pixels"].device == env.device
