"""z-extruded multi-block domains (CylinderJet3D / Airfoil3D, SURVEY section 8(f) rank 3): the float32 numpy specification
oracle/extruded_eval.py -- 2-D compiled tables + uniform periodic z faces -- against an op trace of the UNMODIFIED reference on
CylinderJet3D-easy-v0 with resolution 8 (tests/golden/cyl3d_substep*.npz, generated on a B200 by oracle/ref_harness.py and
tests/golden/extract_cyl3d_fixtures.py).  This pins the operator the D = 3 non-orthogonal kernels have to implement."""
import numpy as np
import pytest
import scipy.sparse as sp

import extruded_eval as ee
from conftest import rel_l2

f32 = np.float32


@pytest.fixture(scope="module")
def cyl3d():
    from fluidgym_b200.envs.cylinder_domain import make_cylinder_domain
    return make_cylinder_domain(8).prepare()


@pytest.mark.parametrize("s", [0, 1])
def test_extruded_operators_match_reference_trace(cyl3d, golden, s):
    cd = cyl3d
    fx = golden(f"cyl3d_substep{s}.npz")
    dt, hz = float(fx["dt"][0]), float(fx["hz"][0])
    u, p, bvel = fx["u_in"], fx["p_in"], fx["bvel"]
    off, offz, A = ee.assemble(cd, u, bvel, dt, hz)
    assert rel_l2(A, fx["A"]) < 5e-7
    assert rel_l2(ee.adv_rhs(cd, u, u, bvel, dt), fx["rhs"]) < 5e-7           # first deferred-correction iteration reads u itself
    hb = ee.hbya(cd, u, fx["ustar"], off, offz, A, bvel, dt)
    assert rel_l2(hb, fx["hbya0"]) < 1e-6
    # divergence incl. the deferred non-orthogonal pressure term: first iteration reads the incoming pressure, the second one
    # the (mean-free) result of the first solve -- pressure_non_ortho_steps = 4 in 3-D (cylinder_env_base.py:317)
    assert rel_l2(ee.divergence(cd, hb, bvel, hz, pres=p, A=A), fx["div0"]) < 3e-5
    x1 = fx["x1"]
    assert rel_l2(ee.divergence(cd, hb, bvel, hz, pres=x1 - x1.mean(), A=A), fx["div1"]) < 3e-5
    assert rel_l2(ee.correct(cd, hb, fx["p0"], A, hz), fx["u0"]) < 1e-6
    assert list(fx["cg_iters"].shape) == [8]                                # 2 correctors x 4 pressure iterations


def test_extruded_matrices_match_reference_csr(cyl3d, golden):
    cd = cyl3d
    fx = golden("cyl3d_substep0.npz")
    nz, N2 = fx["A"].shape
    N3 = nz * N2
    glob = fx["glob"].astype(np.int64).reshape(-1)
    off, offz, A = ee.assemble(cd, fx["u_in"], fx["bvel"], float(fx["dt"][0]), float(fx["hz"][0]))
    Poff, Poffz, Pd = ee.build_P(cd, A, float(fx["hz"][0]))
    C = sp.csr_matrix((fx["C_value"], fx["C_index"], fx["C_row"]), shape=(N3, N3))
    P = sp.csr_matrix((fx["P_value"], fx["P_index"], fx["P_row"]), shape=(N3, N3))
    assert C.nnz < 7 * N3                                                    # ELL(7) minus the prescribed-boundary faces
    rng = np.random.default_rng(0)
    for _ in range(2):
        x = rng.standard_normal((nz, N2)).astype(f32)
        xg = np.zeros(N3, f32)
        xg[glob] = x.reshape(-1)
        assert rel_l2(ee.spmv(cd, off, offz, A, x), (C @ xg)[glob].reshape(nz, N2)) < 5e-7
        assert rel_l2(ee.spmv(cd, Poff, Poffz, Pd, x), (P @ xg)[glob].reshape(nz, N2)) < 5e-7


def test_six_face_neighbour_table_reproduces_the_extruded_matvec(cyl3d):
    """fluidgym_b200.extruded3d.extruded_neighbours: the ELL(7) product the cooperative Krylov kernels form on that table (o3_row:
    diag * x + sum_f off[f] * x[nbr[f]] for nbr >= 0) equals the specification's matvec."""
    from fluidgym_b200.extruded3d import extruded_neighbours
    cd = cyl3d
    nz, hz = 8, 0.5
    rng = np.random.default_rng(3)
    u = rng.standard_normal((3, nz, cd.N)).astype(f32)
    bvel = np.zeros((3, nz, cd.NB), f32)
    bvel[:2] = cd.bvel0[:, None, :cd.NB]
    off, offz, A = ee.assemble(cd, u, bvel, 0.01, hz)
    nbr6 = extruded_neighbours(np.asarray(cd.nbr), nz)
    assert nbr6.shape == (6, nz * cd.N) and (nbr6[4:] >= 0).all()
    coff = np.concatenate([off, offz]).reshape(6, -1)
    x = rng.standard_normal(nz * cd.N).astype(f32)
    y = A.reshape(-1) * x
    for f in range(6):
        ok = nbr6[f] >= 0
        y = y + np.where(ok, coff[f] * x[np.where(ok, nbr6[f], 0)], 0)
    assert rel_l2(y.reshape(nz, cd.N), ee.spmv(cd, off, offz, A, x.reshape(nz, cd.N))) < 1e-6


def test_cylinder3d_observations_from_the_reference_state(golden):
    """CylinderJet3D observation path (extract_global_3d_obs, obs_extraction.py:60-150): rendered-voxel map of the extruded
    5-block domain (6-corner splat of the reference's 3-D kernel, 16 fill sweeps) read at 16 x 151 sensor voxels, incl. the
    reference's raw ``view`` of the [sensor, component] axes; states and observations of the unmodified reference
    (tests/golden/cyl3d_env.npz: after reset and after the first env.step)."""
    import torch
    from fluidgym_b200.envs.cylinder import CylinderJet2DEnv
    from fluidgym_b200.envs.cylinder_domain import make_cylinder_domain
    from fluidgym_b200.sensors import pixel_map_extruded
    fx = golden("cyl3d_env.npz")
    spec = make_cylinder_domain(8)
    nz, n_jets, per_agent, H, L = 8, 8, 2, 4.1, 22.0
    res = 8
    rs = (int(res * 4 / H * L), res * 4, res * 4)                       # cylinder_env_base.py:235-240
    R, level = pixel_map_extruded([b.vertex for b in spec.blocks], np.linspace(-2.0, 2.0, nz + 1, dtype=np.float32), rs, 16)
    assert (level >= 0).all()
    e = object.__new__(CylinderJet2DEnv)
    e.cylinder_diameter = 1.0
    xy = CylinderJet2DEnv.sensor_locations_physical(e)                  # [2, 151] physical sensor positions (shared with 2-D)
    from fluidgym_b200.envs.spanwise import global_obs_from_samples, spanwise_sensor_voxels
    nsz = n_jets * per_agent
    gc = spanwise_sensor_voxels(xy, nsz, H, L, rs).numpy()              # z-major sensor order
    flat = gc[0] + rs[0] * (gc[1] + rs[1] * gc[2])
    Rs = R[flat]
    for tag in ("reset", "env0"):
        u, p = fx[f"{tag}_u"].reshape(3, -1), fx[f"{tag}_p"].reshape(-1)
        us = (Rs @ u.T.astype(np.float64)).astype(np.float32)           # [sensors, 3]
        ps = (Rs @ p.astype(np.float64)).astype(np.float32)
        g = global_obs_from_samples(torch.from_numpy(us)[None], torch.from_numpy(ps)[None], n_jets, per_agent)
        ov, op = g["velocity"][0].numpy(), g["pressure"][0].numpy()
        ref_v = fx["reset_obs_velocity"] if tag == "reset" else fx["step0_obs_velocity"]
        ref_p = fx["reset_obs_pressure"] if tag == "reset" else fx["step0_obs_pressure"]
        assert ov.shape == ref_v.shape == (8, 2, 3, 151)
        assert np.abs(ov - ref_v).max() < 5e-5 * max(1.0, np.abs(ref_v).max())
        assert np.abs(op - ref_p).max() < 5e-5 * max(1.0, np.abs(ref_p).max())


def test_wall_forces_per_plane_equal_the_reference_force_function(golden):
    """The 3-D cylinder's drag / lift (jet_cylinder_env_3d.py:441-470) are the 2-D wall-traction formula applied in every z plane
    with face areas = face length x plane spacing: our torch statement of k_wall_forces (envs/common.py::_forces_torch, the
    differentiable twin of the CUDA kernel) on the reference's traced 3-D state vs the reference's own ``compute_forces_3d``
    (envs/util/forces.py:278-377, pure torch) evaluated on the CPU from the installed reference (its stored values elsewhere:
    tests/reference_values.py)."""
    import torch
    import reference_values
    forces = reference_values.module("fluidgym.envs.util.forces")
    from fluidgym_b200.envs.common import DifferentiableRollout, build_wall_tables
    from fluidgym_b200.envs.cylinder import CylinderJet2DEnv
    from fluidgym_b200.envs.cylinder_domain import make_cylinder_domain
    spec = make_cylinder_domain(8)
    cd = spec.prepare()
    env = object.__new__(CylinderJet2DEnv)
    env.spec, env.cd, env.device, env.U_mean, env.cylinder_diameter = spec, cd, torch.device("cpu"), 1.0, 1.0
    CylinderJet2DEnv._setup_wall(env)
    tab = env._wall_t
    fx = golden("cyl3d_env.npz")
    u, p, bv = torch.from_numpy(fx["env0_u"]), torch.from_numpy(fx["env0_p"]), torch.from_numpy(fx["env0_bvel"])
    nz, hz = u.shape[1], 0.5
    cell, bface = tab["cell"].long(), tab["bface"].long()
    env.wall = type("W", (), {"scale": 1.0})()
    mine = torch.stack([DifferentiableRollout._forces_torch(env, u[:, k][None], p[k][None], bv[:, k][None])[0] for k in range(nz)], dim=1) * hz
    ref = reference_values.value("cylinder3d_wall_forces", forces and (lambda: forces.compute_forces_3d(
        u[:, :, cell], bv[:, :, bface], p[:, cell], tab["normal"][:, :, None], tab["tlen"][:, None], tab["dist"][:, None],
        tab["flen"] * hz, torch.tensor(float(cd.visc)))), mine)                                                  # [2, nz]
    assert float(ref.abs().max()) > 1e-2
    assert torch.allclose(mine, ref, rtol=2e-5, atol=1e-6)


def test_cylinder3d_boundary_hooks_reproduce_the_reference_boundary_values(cyl3d, golden):
    """From the reference's reset state and its first action to the boundary velocities its first substep saw: action smoothing
    (0.1), spanwise jets from the 2-D templates, flux balance over jets + outflow, advective outflow update + outflow balance."""
    import torch
    from fluidgym_b200.envs.cylinder import CylinderJet2DEnv
    from fluidgym_b200.envs.cylinder_domain import WAKE, make_cylinder_domain
    cd = cyl3d
    spec = make_cylinder_domain(8)
    env = object.__new__(CylinderJet2DEnv)
    env.spec, env.cd, env.device, env.jet_angle = spec, cd, torch.device("cpu"), 10.0
    CylinderJet2DEnv._setup_jets(env)
    jf, jt = env.jet_faces.numpy().astype(np.int64), env.jet_templ.numpy()
    fx, s0 = golden("cyl3d_env.npz"), golden("cyl3d_substep0.npz")
    hz = float(s0["hz"][0])
    out = np.zeros(cd.NB, bool)
    o = cd.boff[WAKE, 1]
    out[o:o + spec.blocks[WAKE].ny] = True
    control = CylinderJet2DEnv.action_smoothing_alpha * fx["actions"][0].reshape(-1)          # last control = 0 after reset; one jet per plane
    assert not fx["reset_bvel"][:, :, jf].any()
    bv = ee.apply_jets(cd, fx["reset_bvel"], control, jf, jt, out, hz)
    bv = ee.update_outflow(cd, s0["u_in"], bv, float(s0["dt"][0]), out, hz)
    assert np.abs(bv[:, :, jf] - s0["bvel"][:, :, jf]).max() < 1e-7
    assert np.abs(bv - s0["bvel"]).max() < 1e-6


def test_localized_sensor_rows_equal_the_full_voxel_map():
    """sensors.sensor_tables_extruded builds only the rows of the sensor voxels (memoised recursion over the fill levels); they must
    equal the rows of the full rendered-voxel map (matrix recurrence over all 175 104 voxels) entry by entry."""
    from fluidgym_b200 import sensors as S
    from fluidgym_b200.envs.cylinder import cylinder_sensor_locations
    from fluidgym_b200.envs.cylinder_domain import make_cylinder_domain
    from fluidgym_b200.envs.spanwise import spanwise_sensor_voxels
    spec = make_cylinder_domain(8)
    rs = (171, 32, 32)
    px = spanwise_sensor_voxels(cylinder_sensor_locations(1.0), 16, 4.1, 22.0, rs).numpy()
    zv = np.linspace(-2.0, 2.0, 9, dtype=np.float32)
    vs = [b.vertex for b in spec.blocks]
    idx, w = S.sensor_tables_extruded(vs, zv, rs, px, 16)
    R, level = S.pixel_map_extruded(vs, zv, rs, 16)
    flat = px[0].astype(np.int64) + rs[0] * (px[1].astype(np.int64) + rs[1] * px[2].astype(np.int64))
    assert level[flat].max() >= 1                                    # some sensors sit in voxels that only the fill sweeps reach
    dense = np.zeros((flat.size, R.shape[1]))
    np.add.at(dense, (np.repeat(np.arange(flat.size), idx.shape[0]), idx.T.reshape(-1)), w.T.reshape(-1).astype(np.float64))
    ref = R[flat].toarray()
    assert np.abs(dense - ref).max() < 1e-7 and ((dense != 0) == (np.abs(ref) > 1e-12)).all()
