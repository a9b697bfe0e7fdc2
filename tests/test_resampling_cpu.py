"""The static sensor maps (fluidgym_b200/sensors.py) against the reference's own torch re-implementation of its resampling
kernel (simulation/pict/data/resample.py:361-549, the function its test tests/simulation/test_torch_resample.py compares the
CUDA kernel with at atol = rtol = 1e-3), run on the CPU from the installed unmodified reference (baseline/_ref); its stored values
where the reference is not installed (tests/reference_values.py).  The GPU goldens (tests/golden/*_steps.npz observations) pin the
same maps independently."""
import numpy as np
import pytest
import torch

import reference_values


@pytest.fixture(scope="module")
def resample():
    return reference_values.module("fluidgym.simulation.pict.data.resample")


def test_2d_sensor_tables_equal_the_rendered_pixels(resample):
    """RBC2D: 96 x 61 wall-refined grid -> 240 x 76 render grid, 16 fill sweeps, 48 x 8 sensor pixels."""
    from fluidgym_b200.envs.rbc_domain import make_rbc_domain
    from fluidgym_b200.sensors import sensor_tables
    spec, info = make_rbc_domain()
    vertex = spec.blocks[0].vertex                              # [2, ny+1, nx+1]
    nx, ny = 240, 76
    sx = torch.linspace(0, nx, 49)[:-1] + nx / 96
    sy = torch.linspace(0, ny, 9)[:-1] + ny / 16
    gx, gy = torch.meshgrid(sx, sy, indexing="ij")
    px = torch.stack([gx, gy], dim=-1).reshape(-1, 2).T.round().to(torch.int).numpy()
    idx, w = sensor_tables([vertex], (nx, ny), px, fill_max_steps=16)
    rng = np.random.default_rng(0)
    field = rng.standard_normal((3, info["ny"], info["nx"])).astype(np.float32)
    mine = (w[None] * field.reshape(3, -1)[:, idx]).sum(axis=1)                                   # [3, n_sensors]
    ref = reference_values.value("resample_2d_sensors", resample and (lambda: resample.sample_multi_coords_to_uniform_grid(
        [torch.from_numpy(field)[None]], [torch.from_numpy(vertex)[None]], [nx, ny], fill_max_steps=16,
        differentiable=True)[0][:, px[1], px[0]]), mine)                                    # [3, H, W] -> [3, n_sensors]
    # white-noise field of unit variance; the torch path computes the voxel coordinates in float64, the kernel (and the map) in
    # float32: observed 2.3e-5 (the reference's own bar between its two implementations is 1e-3)
    assert np.abs(mine - ref).max() < 1e-4


def test_3d_pixel_map_equals_the_trilinear_torch_path(resample, golden):
    """RBC3D fixture grid (16 x 10 x 16 cells -> 80 x 25 x 80 voxels): with all 8 corners the sparse map reproduces the
    reference's torch path at every voxel (transform, indexing, hole filling); the product uses 6 corners like the CUDA kernel."""
    from fluidgym_b200.sensors import pixel_map_3d
    vertex = golden("rbc3d_geometry.npz")["vertex"]
    W, H, Z = 80, 25, 80
    R8, level = pixel_map_3d(vertex, (W, H, Z), 16, n_corners=8)
    assert (level >= 0).all()
    rng = np.random.default_rng(1)
    field = rng.standard_normal((2, 16, 10, 16)).astype(np.float32)
    mine = (R8 @ field.reshape(2, -1).T.astype(np.float64)).T.reshape(2, Z, H, W)
    ref = resample and resample.sample_multi_coords_to_uniform_grid([torch.from_numpy(field)[None]], [torch.from_numpy(vertex)[None]],
                                                                    [W, H, Z], fill_max_steps=16, differentiable=True)[0].numpy()
    assert ref is None or np.abs(mine - ref).max() < 1e-4
    # stored: a fixed sample of 2048 voxels (all 160 000 would be 1.3 MB)
    vox = np.sort(np.random.default_rng(3).choice(Z * H * W, 2048, replace=False))
    mine_s = mine.reshape(2, -1)[:, vox].astype(np.float32)
    ref_s = reference_values.value("resample_3d_voxel_sample", ref is not None and (lambda: ref.reshape(2, -1)[:, vox]), mine_s)
    assert np.abs(mine_s - ref_s).max() < 1e-4
    R6, _ = pixel_map_3d(vertex, (W, H, Z), 16)
    assert R6.nnz < R8.nnz and abs((R6 - R8)).max() > 1e-3          # the kernel's 6-corner splat is a different map
