"""Render maps (fluidgym_b200/render.py) without a GPU: the full maps agree with the sensor tables at the sensor pixels and with
an independent pixel-grid evaluation of splat -> normalise -> fill sweeps; the numpy colour specification; the RL adapters'
image paths on a stand-in environment that renders."""
import numpy as np
import pytest
import torch

from fluidgym_b200 import render
from fluidgym_b200.sensors import cell_centres, pixel_map_3d, sensor_tables_3d, uniform_grid_transform
from test_integration import FakeEnv


def _env(cls, **attrs):
    """a family's host-side setup (sensor tables, render map) without constructing its solver"""
    env = cls.__new__(cls)
    env.device = torch.device("cpu")
    for k, v in attrs.items():
        setattr(env, k, v)
    env._setup_sensors()
    return env


def _cylinder(res):
    from fluidgym_b200.envs.cylinder import CylinderJet2DEnv
    from fluidgym_b200.envs.cylinder_domain import make_cylinder_domain
    return _env(CylinderJet2DEnv, resolution=res, spec=make_cylinder_domain(res))


def _airfoil():
    from fluidgym_b200.envs.airfoil import Airfoil2DEnv
    from fluidgym_b200.envs.airfoil_domain import make_airfoil_domain
    return _env(Airfoil2DEnv, attack_angle_deg=10.0, spec=make_airfoil_domain())


def _rbc2d():
    from fluidgym_b200.envs.rbc import RBC2DEnv
    from fluidgym_b200.envs.rbc_domain import make_rbc_domain
    spec, _ = make_rbc_domain(8e4, 0.7, 12, 8)
    return _env(RBC2DEnv, n_heaters=12, aspect=np.pi, spec=spec)


FAMILIES_2D = {"cylinder24": lambda: _cylinder(24), "cylinder32": lambda: _cylinder(32), "airfoil": _airfoil, "rbc2d": _rbc2d}
_CACHE = {}


def _family(name):
    if name not in _CACHE:
        env = FAMILIES_2D[name]()
        _CACHE[name] = (env, env._build_render_map(None))
    return _CACHE[name]


@pytest.mark.parametrize("name", sorted(FAMILIES_2D))
def test_full_map_rows_equal_sensor_tables(name):
    env, m = _family(name)
    W, H = env.render_shape
    assert m.shape == (H, W) and m.rowptr.dtype == np.int32 and m.col.dtype == np.int32 and m.w.dtype == np.float32
    assert m.rowptr[0] == 0 and m.rowptr[-1] == m.col.size == m.w.size and np.all(np.diff(m.rowptr) >= 0)
    N = sum(b.nx * b.ny for b in env.spec.blocks)
    R = m.matrix(N)
    x, y = env.sensor_px
    rows = R[(H - 1 - y) * W + x].toarray()                            # image row 0 = largest y
    idx, w = env.sens_idx.numpy(), env.sens_w.numpy()
    ref = np.zeros_like(rows)
    for s in range(idx.shape[1]):
        np.add.at(ref[s], idx[:, s], w[:, s].astype(np.float64))
    assert np.abs(rows - ref).max() <= 1e-7


def _numpy_render(vertex_list, out_shape, fill_max_steps, cell_values):
    """splat with np.add.at, normalise, fill sweeps on the pixel grid (float64), image order"""
    W, H = out_shape
    scale, centre, os_ = uniform_grid_transform(vertex_list, out_shape)
    c = np.concatenate([cell_centres(v).reshape(2, -1) for v in vertex_list], axis=1)
    sc = ((c - centre[:, None]) / scale + (os_ * np.float32(0.5) - np.float32(0.5))[:, None]).astype(np.float32)
    fl = np.floor(sc)
    fr = (sc - fl).astype(np.float32)
    val, wsum = np.zeros((H, W)), np.zeros((H, W))
    for dx in (0, 1):
        for dy in (0, 1):
            px, py = (np.ceil(sc[0]) if dx else fl[0]).astype(np.int64), (np.ceil(sc[1]) if dy else fl[1]).astype(np.int64)
            wt = ((fr[0] if dx else 1 - fr[0]) * (fr[1] if dy else 1 - fr[1])).astype(np.float64)
            ok = (px >= 0) & (px < W) & (py >= 0) & (py < H)
            np.add.at(val, (py[ok], px[ok]), wt[ok] * cell_values[ok])
            np.add.at(wsum, (py[ok], px[ok]), wt[ok])
    valid = wsum > 1e-8
    img = np.where(valid, val / np.where(valid, wsum, 1.0), 0.0)
    for _ in range(fill_max_steps):
        if valid.all():
            break
        acc, cnt = np.zeros((H, W)), np.zeros((H, W))
        for sl_dst, sl_src in (((slice(None), slice(1, None)), (slice(None), slice(None, -1))),
                               ((slice(None), slice(None, -1)), (slice(None), slice(1, None))),
                               ((slice(1, None), slice(None)), (slice(None, -1), slice(None))),
                               ((slice(None, -1), slice(None)), (slice(1, None), slice(None)))):
            acc[sl_dst] += np.where(valid[sl_src], img[sl_src], 0.0)
            cnt[sl_dst] += valid[sl_src]
        newly = ~valid & (cnt > 0)
        img = np.where(newly, acc / np.maximum(cnt, 1), img)
        valid = valid | newly
    return img[::-1]


@pytest.mark.parametrize("name,fill", [("cylinder24", 16), ("airfoil", 128)])
def test_full_map_equals_pixel_grid_evaluation(name, fill):
    env, m = _family(name)
    vl = [b.vertex for b in env.spec.blocks]
    N = sum(b.nx * b.ny for b in env.spec.blocks)
    if name == "airfoil":
        assert np.diff(m.rowptr).max() >= 100                          # the rows behind the airfoil's interior
    rng = np.random.default_rng(5)
    for _ in range(2):
        f = rng.standard_normal(N)
        got = (m.matrix(N) @ f).reshape(m.shape)
        ref = _numpy_render(vl, env.render_shape, fill, f)
        assert np.linalg.norm(got - ref) <= 1e-6 * np.linalg.norm(ref)


def test_rbc3d_slice_rows_equal_voxel_map():
    from fluidgym_b200.envs.rbc3d import RBC3DEnv, rbc3d_vertex_grid
    nh, hw = 2, 4
    nx = nh * hw
    ny = round(2.0 * nx / np.pi)
    env = RBC3DEnv.__new__(RBC3DEnv)
    env.n_heaters, env.aspect = nh, np.pi
    vertex = rbc3d_vertex_grid(nx, ny, np.pi, 1.0, 1.02)
    env.dom = type("Dom", (), {"vertex": vertex})()
    W, H, Z = env.render_shape
    n_planes, default = env._render_planes()
    assert (n_planes, default) == (Z, Z // 2)
    R, _ = pixel_map_3d(vertex, (W, H, Z), 16)
    for plane in (default, 0):
        m = env._build_render_map(plane)
        assert m.shape == (H, W)
        y, x = np.meshgrid(np.arange(H - 1, -1, -1), np.arange(W), indexing="ij")
        ref = R[(x + W * (y + H * plane)).ravel()].toarray()
        assert np.abs(m.matrix(R.shape[1]).toarray() - ref).max() <= 1e-7
    # and the sensor tables at the voxels of the default plane
    px = np.array([[3, 20, 37], [2, 5, H - 1], [default] * 3])
    idx, w = sensor_tables_3d(vertex, (W, H, Z), px, 16)
    rows = env._build_render_map(default).matrix(R.shape[1])[(H - 1 - px[1]) * W + px[0]].toarray()
    ref = np.zeros_like(rows)
    for s in range(3):
        np.add.at(ref[s], idx[:, s], w[:, s].astype(np.float64))
    assert np.abs(rows - ref).max() <= 1e-7


def test_cell_plane_map_is_the_identity():
    m = render.render_map_cell_plane(5, 4, 3, 2)
    f = np.arange(5 * 4 * 3, dtype=np.float64)
    assert m.shape == (3, 5)
    assert np.array_equal((m.matrix(f.size) @ f).reshape(3, 5), f.reshape(3, 4, 5)[:, 2, :])


def test_colour_specification():
    for lut in (render.DIVERGING, render.SEQUENTIAL):
        assert lut.shape == (256, 3) and lut.dtype == np.uint8
    assert render.DIVERGING[127].min() > 230 and render.DIVERGING[128].min() > 230       # white at zero
    img = np.array([[[-1.0, 0.0, 1.0, 3.0]], [[2.0, 4.0, 6.0, 10.0]]], dtype=np.float32)   # [B=2, 1, 4]
    # each environment over its own range: the ends land in the first / last bin
    b = render.colour_bins(img, img.reshape(2, -1).min(1), img.reshape(2, -1).max(1))
    assert b.tolist() == [[[0, 64, 128, 255]], [[0, 64, 128, 255]]]
    out = render.colour_reference(img, render.SEQUENTIAL)
    assert out.shape == (2, 1, 4, 3) and out.dtype == np.uint8 and np.array_equal(out[0, 0, 0], render.SEQUENTIAL[0])
    # a fixed range for the batch: values beyond the ends are clamped
    b = render.colour_bins(img, 0.0, 4.0)
    assert b.tolist() == [[[0, 0, 64, 192]], [[128, 255, 255, 255]]]
    out = render.colour_reference(img, render.DIVERGING, vmin=0.0, vmax=4.0)
    assert np.array_equal(out[1, 0, 3], render.DIVERGING[255]) and np.array_equal(out[0, 0, 0], render.DIVERGING[0])
    # symmetric: [-max|v|, max|v|] per environment, zero in the middle bin
    out = render.colour_reference(img, render.DIVERGING, symmetric=True)
    assert np.array_equal(out[0, 0, 1], render.DIVERGING[128]) and np.array_equal(out[0, 0, 3], render.DIVERGING[255])
    assert np.array_equal(out[0, 0, 0], render.DIVERGING[int(256 * (2.0 / 6.0))])
    # an empty range (a uniform field) maps to the middle bin, NaN to the first
    assert render.colour_bins(np.full((1, 3), 2.0, np.float32), 2.0, 2.0).tolist() == [[128, 128, 128]]
    assert render.colour_bins(np.array([[np.nan]], np.float32), 0.0, 1.0).tolist() == [[0]]


# ---- RL adapters on a stand-in environment that renders ----------------------------------------------------------------------
class RenderingEnv(FakeEnv):
    H, W = 6, 9

    def render(self, field=None, *, plane=None, vmin=None, vmax=None):
        env = torch.arange(self.n_envs, dtype=torch.uint8)[:, None, None, None] * 10
        return env + self.t + torch.zeros(self.H, self.W, 3, dtype=torch.uint8)


def test_gym_render():
    from fluidgym_b200.integration import GymFluidEnv
    env = GymFluidEnv(RenderingEnv(1), render_mode="rgb_array")
    env.reset(seed=0)
    img = env.render()
    assert isinstance(img, np.ndarray) and img.shape == (6, 9, 3) and img.dtype == np.uint8
    assert GymFluidEnv(RenderingEnv(1)).render() is None


def test_vec_env_images():
    from fluidgym_b200.integration import VecFluidEnv
    venv = VecFluidEnv(RenderingEnv(3, n_agents=2, use_marl=True), render_mode="rgb_array")
    venv.reset(seed=0)
    imgs = venv.get_images()
    assert len(imgs) == 6 and all(i.shape == (6, 9, 3) and i.dtype == np.uint8 for i in imgs)
    assert [int(i[0, 0, 0]) for i in imgs] == [0, 0, 10, 10, 20, 20]
    assert VecFluidEnv(RenderingEnv(3)).get_images() == [None] * 3
    with pytest.raises(ValueError):
        VecFluidEnv(RenderingEnv(3), render_mode="human")


@pytest.mark.parametrize("marl", [False, True])
def test_torchrl_pixels(marl):
    from fluidgym_b200.integration import TorchRLFluidEnv
    env = RenderingEnv(3, n_agents=2, use_marl=marl)
    tenv = TorchRLFluidEnv(env, from_pixels=True)
    lead = (3, 2) if marl else (3,)
    assert tuple(tenv.observation_spec["pixels"].shape) == (*lead, 6, 9, 3) and tenv.observation_spec["pixels"].dtype == torch.uint8
    td = tenv.reset()
    assert tuple(td["pixels"].shape) == (*lead, 6, 9, 3) and td["pixels"].dtype == torch.uint8
    out = tenv.step({"action": torch.ones(*lead, 1)})["next"]
    assert tuple(out["pixels"].shape) == (*lead, 6, 9, 3)
    assert int(out["pixels"][(2, 1) if marl else (2,)][0, 0, 0]) == 21          # environment 2 after one step; agents share it
    assert "pixels" not in TorchRLFluidEnv(env).observation_spec
