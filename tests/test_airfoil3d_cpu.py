"""Airfoil3D environment (fluidgym_b200/envs/airfoil3d.py): host logic on the CPU with the solver calls stubbed out, at a reduced
number of z planes (8 instead of 96; the plane mesh is the real 46 806-cell airfoil grid).  The environment is assembled from pinned
parts (extruded solver path + spanwise machinery: tests/test_cylinder3d_cpu.py; 2-D airfoil tables: tests/test_gpu_airfoil.py,
test_airfoil_cpu.py); ENVIRONMENT-LEVEL PARITY IS UNPINNED until a golden run of the reference's Airfoil3D exists -- these tests
check the reference's formulas (airfoil_env_3d.py, cited per assertion), not its outputs."""
import os
import sys

import numpy as np
import pytest

import reference_values
from conftest import ROOT

torch = pytest.importorskip("torch")
sys.path.insert(0, os.path.join(ROOT, "tests", "cpu_harness"))


@pytest.fixture(scope="module")
def compiled():
    from fluidgym_b200.envs.airfoil_domain import make_airfoil_domain
    spec = make_airfoil_domain()
    return spec, spec.prepare()


def _env(compiled, **kw):
    from extruded_standin import HostExtrudedPISO3D
    from fluidgym_b200.envs.airfoil3d import Airfoil3DEnv
    e = Airfoil3DEnv(res_z=8, device="cpu", compiled=compiled, solver_cls=HostExtrudedPISO3D, **kw)
    e.solver.piso_substep = lambda dt: None                      # host logic only: 374 448 cells are too many for numpy Krylov solvers
    e.solver.make_divergence_free = lambda max_iter=1000: None
    return e


def test_actions_become_per_plane_jet_profiles_with_zero_net_flux(compiled):
    """airfoil_env_3d.py:383-407, airfoil_env_base.py:709-718: per agent zero-mean / clamped amplitudes times the 2-D unit-flux jet
    profiles in the agent's planes, no spanwise component, outflow + airfoil top wall rescaled to a zero net boundary flux."""
    from fluidgym_b200.envs.airfoil import Airfoil2DEnv
    env = _env(compiled, n_envs=2, n_agents=4)
    env.reset(seed=0)
    s = env.solver
    ctrl = torch.tensor([[[0.5, -0.2, 0.1], [2.0, -3.0, 0.4], [0.0, 0.0, 0.0], [1.0, 1.0, 1.0]]]).repeat(2, 1, 1)
    ctrl[1] *= -0.5
    before = s.bvel.clone()
    env._apply_action(ctrl)
    jf = env.jet_faces.long()
    for b in range(2):
        for a in range(4):
            want = Airfoil2DEnv._control_to_profile(env, ctrl[b, a][None])[0]              # [2, n_top], the 2-D formula
            for k in (2 * a, 2 * a + 1):
                got = s.bvel[b, :2, k, jf]
                scale = float((got * want).sum() / (want * want).sum()) if float(want.abs().max()) > 0 else 1.0
                assert torch.allclose(got, want * scale, atol=1e-7)                          # same shape, common flux-balance factor
                assert not s.bvel[b, 2, k, jf].any()
    fl = (s.bvel[:, 0] * s._st["fw"][0] + s.bvel[:, 1] * s._st["fw"][1]) * s.hz
    assert fl.double().sum(dim=(1, 2)).abs().max() < 1e-7
    fixed = ~env._free_jets
    assert torch.equal(s.bvel[:, :, :, fixed], before[:, :, :, fixed])                      # inflow / walls untouched
    # agents 2 (zero) and 3 (constant = zero-mean zero): no blowing
    assert float(s.bvel[0, :2, 4:8][:, :, jf].abs().max()) == 0.0


def test_sensor_layout_spaces_and_multi_agent_rewards(compiled):
    from fluidgym_b200.envs.airfoil import Airfoil2DEnv
    env = _env(compiled, n_envs=2, n_agents=4, use_marl=True, local_reward_weight=0.5, cl_cd_ref=1.5, step_length=0.05)   # one solver step
    # the (x, y) sensor columns are the 2-D environment's, repeated at 4 span positions (airfoil_env_3d.py:303-344)
    e2 = object.__new__(Airfoil2DEnv)
    e2.attack_angle_deg = 10.0
    px2 = Airfoil2DEnv._to_pixels(e2, Airfoil2DEnv.sensor_locations_physical(e2)).numpy()
    px = env.sensor_px.reshape(3, 4, -1)
    assert env.n_sensors_xy == px.shape[2] and env.n_sensors_xy <= px2.shape[1]
    assert all(np.array_equal(px[:2, k], px[:2, 0]) for k in range(4)) and len(set(px[2, :, 0].tolist())) == 4
    assert set(map(tuple, px[:2, 0].T.tolist())) <= set(map(tuple, px2.T.tolist()))
    assert not env.airfoil_mask[px[1], px[0]].any()
    zs = np.round((np.linspace(-0.7, 0.7, 5)[:-1] + 0.175 + 0.7) * 150 / 1.4).astype(int)   # :331-337 with airfoil_env_base.py:581-583
    assert px[2, :, 0].tolist() == zs.tolist()
    assert env.n_agents == 4 and env.action_space.shape == (3,)
    assert env.observation_space.spaces["velocity"].shape == (1, 1, 3, env.n_sensors_xy)
    env.seed(3)
    with pytest.raises(RuntimeError, match="must be reset"):
        env.step(env.sample_action())
    obs, _ = env.reset()
    assert obs["velocity"].shape == (2, 4, 1, 1, 3, env.n_sensors_xy) and obs["pressure"].shape == (2, 4, 1, 1, env.n_sensors_xy)
    env.solver.u[:, 0] = 0.3
    env.solver.u[:, 0] += 0.01 * torch.randn(env.solver.u[:, 0].shape, generator=torch.Generator().manual_seed(1))
    a = env.sample_action()
    assert a.shape == (2, 4, 3)
    obs, reward, term, trunc, info = env.step(a)
    cds, cls_ = env._drag_and_lift()                              # one (stubbed) solver step: the mean over the step = the final value
    cd, cl = cds.sum(1) / 1.4, cls_.sum(1) / 1.4
    assert torch.allclose(info["drag"], cd, rtol=1e-5) and torch.allclose(info["lift"], cl, rtol=1e-5)
    glob = cl / cd - 1.5                                         # airfoil_env_3d.py:420
    lcd, lcl = cds.view(2, 4, -1).sum(2) / 0.35, cls_.view(2, 4, -1).sum(2) / 0.35          # :441-448
    assert torch.allclose(info["global_reward"], glob, rtol=1e-5, atol=1e-6)
    assert reward.shape == (2, 4) and torch.allclose(reward, 0.5 * (lcl / lcd - 1.5) + 0.5 * glob[:, None], rtol=1e-4, atol=1e-5)
    sarl = _env(compiled, n_agents=2)
    assert sarl.action_space.shape == (2, 3) and sarl.observation_space.spaces["pressure"].shape == (2, 1, sarl.n_sensors_xy)


def test_constructor_checks_and_registry(compiled):
    import fluidgym_b200
    from extruded_standin import HostExtrudedPISO3D
    from fluidgym_b200.envs.airfoil3d import Airfoil3DEnv
    with pytest.raises(ValueError, match="evenly divides"):
        Airfoil3DEnv(n_agents=5, device="cpu", compiled=compiled)
    with pytest.raises(ValueError, match="Attack angle"):
        Airfoil3DEnv(attack_angle_deg=25.0, device="cpu", compiled=compiled)
    if not torch.cuda.is_available():
        from fluidgym_b200 import native
        with pytest.raises(native.FGBError, match="no CPU fallback"):        # the product path has no CPU solver
            Airfoil3DEnv(device="cpu", compiled=compiled)
    env = fluidgym_b200.make("Airfoil3D-hard-v0", res_z=8, device="cpu", compiled=compiled, solver_cls=HostExtrudedPISO3D,
                             load_domain_statistics=False)
    assert env.reynolds_number == 5e3 and env.initial_domain_id == "airfoil_3D_Re5000" and env.nz_per_agent == 2
    assert env.solver.opt["ans"] == 2 and env.solver.opt["pns"] == 4 and env.solver.opt["ptol"] == 1e-8      # airfoil_env_base.py:262-283


def test_init_from_2d_copies_the_2d_velocity_into_every_plane(compiled, tmp_path):
    """airfoil_env_3d.py:524-593: a 2-D airfoil initial domain (the reference's on-disk format, fluidgym_b200/domain_io.py) of the
    training split seeds the 3-D velocity plane by plane with a zero spanwise component; a missing file raises."""
    from fluidgym_b200.domain_io import save_domain
    spec, cd = compiled
    rng = np.random.default_rng(2)
    files = {}
    for idx in range(10):
        st = dict(u=rng.standard_normal((2, cd.N)).astype(np.float32), p=np.zeros(cd.N, np.float32), bvel=cd.bvel0[:, :cd.NB].astype(np.float32))
        d = tmp_path / "airfoil_2D_Re3000" / str(idx)
        d.mkdir(parents=True)
        save_domain(spec, st, str(d / "train"))
        files[idx] = st["u"]
    env = _env(compiled, n_envs=3, n_agents=4, init_from_2d=True, initial_domains_path=str(tmp_path))
    env.reset(seed=5)                                            # projection and solver are stubbed: the seeded field survives
    u4 = env.solver.u.view(3, 3, 8, cd.N)
    picks = []
    for e in range(3):
        match = [i for i, u in files.items() if np.array_equal(u4[e, :2, 0].numpy(), u)]
        assert len(match) == 1
        picks.append(match[0])
        assert all(torch.equal(u4[e, :2, k], u4[e, :2, 0]) for k in range(8)) and not u4[e, 2].any()
    rng2 = np.random.default_rng(5)
    assert picks == [int(rng2.integers(0, 10)) for _ in range(3)]
    missing = _env(compiled, init_from_2d=True, initial_domains_path=str(tmp_path / "nowhere"))
    with pytest.raises(FileNotFoundError, match="2D initial domain not found"):
        missing.reset(seed=1)


def _reference_stub(env):
    """an object carrying just the attributes the reference's pure-torch methods read, so that they run on the CPU"""
    from fluidgym.envs.airfoil.airfoil_env_3d import AirfoilEnv3D
    from fluidgym.envs.airfoil.airfoil_env_base import AirfoilEnvBase
    from fluidgym_b200.envs.airfoil_domain import airfoil_polyline

    class Stub:
        pass
    st = Stub()
    st.H, st.L, st.D, st.airfoil_length = env.H, env.L, env.D, env.airfoil_length
    st.render_shape, st._ndims = env.render_shape, 3
    st._n_agents, st._n_sensors_per_agent, st._n_sensors_z = env.n_span, env.n_sensors_per_agent, env.n_sensors_z
    st._n_jets, st._nz_per_agent = env.n_jets, env.nz_per_agent
    st._get_sensor_locations_2d = lambda: AirfoilEnvBase._get_sensor_locations_2d(st)
    st._get_sensor_locations_3d = lambda: AirfoilEnv3D._get_sensor_locations_3d(st)
    st._physical_locations_to_grid_coords = lambda c: AirfoilEnvBase._physical_locations_to_grid_coords(st, c)
    st._airfoil_coords = airfoil_polyline(env.attack_angle_deg)
    return st, AirfoilEnv3D, AirfoilEnvBase


def test_sensor_layout_and_action_mapping_equal_the_reference_methods(compiled):
    """The reference's own pure-torch methods -- AirfoilEnvBase._get_airfoil_mask, AirfoilEnv3D._get_sensor_locations (z-major voxel
    coordinates, columns touching the airfoil mask dropped) and AirfoilEnv3D._action_to_control (zero-mean clamped amplitudes repeated
    over the agents' planes) -- executed on the CPU from the installed reference on a stub object (their stored values elsewhere:
    tests/reference_values.py), against this environment."""
    have_ref = reference_values.module("fluidgym.envs.airfoil.airfoil_env_3d") is not None
    env = _env(compiled, n_envs=1, n_agents=4)
    st, Ref3D, RefBase = _reference_stub(env) if have_ref else (None, None, None)
    if have_ref:
        st._airfoil_mask = RefBase._get_airfoil_mask(st)
    mask = reference_values.value("airfoil3d_mask", have_ref and (lambda: st._airfoil_mask[0]), env.airfoil_mask)
    assert np.array_equal(env.airfoil_mask, mask)
    gc = reference_values.value("airfoil3d_sensor_locations", have_ref and (lambda: Ref3D._get_sensor_locations(st)),
                                env.sensor_px.reshape(3, 4, -1))
    assert tuple(gc.shape) == (3, 4, env.n_sensors_xy) and np.array_equal(env.sensor_px.reshape(3, 4, -1), np.asarray(gc))
    # action -> jet wall velocity (before the flux balance, which rescales jets and outflow by one common factor)
    nz, n_top = env.nz, env.jet_base.shape[2]
    action = torch.tensor([[0.5, -0.2, 0.1], [2.0, -3.0, 0.4], [0.0, 0.3, 0.0], [1.0, 1.0, 1.0]])
    if have_ref:
        base = torch.zeros(1, 3, nz, 1, n_top)
        base[0, :2, :, 0, :] = env.jet_base.sum(dim=0)[:, None, :]                   # the three slots do not overlap
        st._top_base_profile, st._jet_locations_top = base, [list(ab) for ab in env.jet_slots]
    env.reset(seed=0)
    env._apply_action(action[None])
    got = env.solver.bvel[0][:, :, env.jet_faces.long()]
    # stored: this environment's jet velocities, i.e. the reference's up to the common factor the assertion fits
    ref = reference_values.value("airfoil3d_action_to_control", have_ref and (lambda: Ref3D._action_to_control(st, action)[0, :, :, 0, :]),
                                 got)                                                  # [3, nz, n_top]
    scale = float((got[:2] * ref[:2]).sum() / (ref[:2] * ref[:2]).sum())
    assert 0.5 < scale < 2.0 and torch.allclose(got, ref * scale, atol=1e-7) and not got[2].any()


def test_multi_agent_reward_mix_equals_the_reference_methods(compiled):
    """AirfoilEnv3D._step_marl_impl and CylinderJetEnv3D._step_marl_impl (pure torch once the solver step is stubbed: they receive the
    per-plane coefficients from ``_step_impl``) executed from the installed reference (their stored values elsewhere:
    tests/reference_values.py), against ``SpanwiseExtrudedEnv.step``'s mix."""
    air3d = reference_values.module("fluidgym.envs.airfoil.airfoil_env_3d")
    cyl3d = reference_values.module("fluidgym.envs.cylinder.jet_cylinder_env_3d")
    g = torch.Generator().manual_seed(4)
    cds, cls_ = 1.0 + torch.rand(8, generator=g), torch.randn(8, generator=g)

    class Stub:
        pass
    from extruded_standin import HostExtrudedPISO3D
    from fluidgym_b200.envs.cylinder3d import CylinderJet3DEnv
    from fluidgym_b200.envs.cylinder_domain import make_cylinder_domain
    cspec = make_cylinder_domain(8)
    cyl = CylinderJet3DEnv(resolution=8, n_jets=8, device="cpu", compiled=(cspec, cspec.prepare()), solver_cls=HostExtrudedPISO3D, use_marl=True,
                           local_reward_weight=0.3, cd_ref=3.0, lift_penalty=0.7, step_length=0.01)
    air = _env(compiled, n_agents=4, use_marl=True, local_reward_weight=0.3, cl_cd_ref=1.5, step_length=0.05)
    for name, ref_cls, env, n_agents, D, extra, formula in (
            ("airfoil3d", air3d and air3d.AirfoilEnv3D, air, 4, 1.4, dict(_cl_cd_ref=1.5), lambda cd, cl: cl / cd - 1.5),
            ("cylinder3d", cyl3d and cyl3d.CylinderJetEnv3D, cyl, 8, 4.0, dict(_cd_ref=3.0, _lift_penalty=0.7),
             lambda cd, cl: 3.0 - cd - 0.7 * torch.abs(cl))):
        st = Stub()
        st.D, st._n_agents, st._n_jets, st._local_reward_weight = D, n_agents, n_agents, 0.3
        for k, v in extra.items():
            setattr(st, k, v)
        cd, cl = cds.sum() / D, cls_.sum() / D
        glob = formula(cd, cl)                                                       # the reference's _step_impl result (:420 / :436)
        st._step_impl = lambda a: (None, glob, False, {"drag": cd, "lift": cl, "all_cds": cds.clone(), "all_cls": cls_.clone()})
        st._get_local_obs = lambda: {}
        ref_out = ref_cls and ref_cls._step_marl_impl(st, None)
        # this repository: one (stubbed) solver step whose per-plane coefficients are the same numbers
        env.solver.piso_substep = lambda dt: None
        env.solver.make_divergence_free = lambda max_iter=1000: None
        env.reset(seed=0)
        env._drag_and_lift = lambda: (cds[None].clone(), cls_[None].clone())
        _, reward, _, _, info = env.step(torch.zeros_like(env._zero_action))
        ref_rewards = reference_values.value(f"{name}_marl_rewards", ref_out and (lambda: ref_out[1]), reward[0])
        ref_global = reference_values.value(f"{name}_marl_global_reward", ref_out and (lambda: ref_out[3]["global_reward"]),
                                            info["global_reward"][0])
        assert reward.shape == (1, n_agents) and torch.allclose(reward[0], ref_rewards, rtol=1e-6, atol=1e-6)
        assert torch.allclose(info["global_reward"][0], ref_global, rtol=1e-6) and "all_cds" not in info
        assert not ref_out or "all_cds" not in ref_out[3]
        assert torch.allclose(info["drag"][0], cd) and torch.allclose(info["lift"][0], cl)


def test_per_plane_forces_equal_the_reference_force_function(compiled):
    """Airfoil3D drag / lift per plane (airfoil_env_base.py:452-476: compute_forces_3d with face areas = wall face length x D / res_z)
    evaluated by the reference's own function on the CPU (its stored values elsewhere: tests/reference_values.py), against
    ``SpanwiseExtrudedEnv._drag_and_lift`` on a random state."""
    forces = reference_values.module("fluidgym.envs.util.forces")
    env = _env(compiled, n_envs=1, n_agents=4)
    s, tab = env.solver, env._wall_t
    g = torch.Generator().manual_seed(9)
    s.u.copy_(torch.randn(s.u.shape, generator=g))
    s.p.copy_(torch.randn(s.p.shape, generator=g))
    s.bvel.copy_(0.1 * torch.randn(s.bvel.shape, generator=g))
    nz, N2 = env.nz, s.N2
    u = s.u[0].view(3, nz, N2)
    p = s.p[0].view(nz, N2)
    bv = s.bvel[0]
    cell, bface = tab["cell"].long(), tab["bface"].long()
    cds, cls_ = env._drag_and_lift()
    scale = 1.0 / (0.5 * env.U_mean ** 2 * env.airfoil_length)
    ref = reference_values.value("airfoil3d_wall_forces", forces and (lambda: forces.compute_forces_3d(
        u[:, :, cell], bv[:, :, bface], p[:, cell], tab["normal"][:, :, None], tab["tlen"][:, None], tab["dist"][:, None],
        tab["flen"] * env.hz, torch.tensor(float(env.cd.visc)))), torch.stack([cds[0], cls_[0]]) / scale)        # [2, nz] forces
    assert float(ref.abs().max()) > 1e-3
    assert torch.allclose(cds[0], ref[0] * scale, rtol=2e-4, atol=1e-5 * float((ref * scale).abs().max()))
    assert torch.allclose(cls_[0], ref[1] * scale, rtol=2e-4, atol=1e-5 * float((ref * scale).abs().max()))
