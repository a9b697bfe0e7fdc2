"""Moving-window extraction of the multi-agent environments: the cases of the reference's own test file
(tests/env_utils/test_obs_extraction.py: parametrisations and the property each one checks) applied to the batched
implementations, plus equality with the reference's functions on random fields (called where the unmodified reference is
installed, baseline/_ref, CPU only; their stored values elsewhere: tests/reference_values.py)."""
import pytest
import torch

import reference_values
from fluidgym_b200.envs.rbc import extract_moving_window_2d
from fluidgym_b200.envs.rbc3d import extract_moving_window_3d
from fluidgym_b200.envs.tcf import agent_window_means


@pytest.mark.parametrize("n_agents, agent_width, n_agents_per_window", [(8, 12, 1), (8, 12, 3), (8, 12, 5)])
def test_moving_window_2d(n_agents, agent_width, n_agents_per_window):
    torch.manual_seed(0)
    y, X = 10, n_agents * agent_width
    field = torch.rand(2, y, X)                                   # leading environment dimension
    half = n_agents_per_window // 2
    win = extract_moving_window_2d(field, n_agents, agent_width, n_agents_per_window)
    assert win.shape == (2, n_agents, y, n_agents_per_window * agent_width)
    cols = torch.arange(X)
    for a in range(n_agents):
        idx = (cols[: n_agents_per_window * agent_width] + (a - half) * agent_width) % X      # circular slice centred on agent a
        assert torch.equal(win[:, a], field[:, :, idx])


@pytest.mark.parametrize("n_agents, agent_width, n_agents_per_window", [(10, 1, 1), (10, 2, 3), (20, 4, 1), (20, 4, 3)])
def test_moving_window_3d(n_agents, agent_width, n_agents_per_window):
    torch.manual_seed(0)
    y, k = 10, n_agents_per_window * agent_width
    field = torch.rand(n_agents * agent_width, y, n_agents * agent_width)
    res = extract_moving_window_3d(field, n_agents, agent_width, n_agents_per_window)
    assert res.shape == (n_agents * n_agents, k, y, k)
    a = (n_agents_per_window // 2) * n_agents + (n_agents_per_window // 2)                    # the agent whose window starts at 0
    assert torch.equal(res[a], field[:k, :, :k])
    # every agent: circular slices in z and x
    pos = torch.arange(k)
    for az, ax in ((0, 0), (n_agents - 1, 1), (3, n_agents - 1)):
        iz = (pos + (az - n_agents_per_window // 2) * agent_width) % (n_agents * agent_width)
        ix = (pos + (ax - n_agents_per_window // 2) * agent_width) % (n_agents * agent_width)
        assert torch.equal(res[az * n_agents + ax], field[iz][:, :, ix])


@pytest.mark.parametrize("nax, naz, aw, wx, wz, pad_x, pad_z", [(10, 20, 2, 1, 1, 0, 0), (20, 40, 2, 5, 3, 4, 1), (10, 20, 4, 5, 5, 4, 4)])
def test_moving_window_2d_x_z(nax, naz, aw, wx, wz, pad_x, pad_z):
    """the channel's per-agent patch means (extract_moving_window_2d_x_z): the window that starts at the origin"""
    torch.manual_seed(0)
    field = torch.rand(naz * aw, nax * aw)
    field[: wz * aw, : wx * aw] = 1.0
    res = agent_window_means(field, nax, naz, aw, wx, wz, pad_x, pad_z)
    assert res.shape == (naz * nax, wz, wx)
    expected = field[: wz * aw, : wx * aw].view(wz, aw, wx, aw).mean(dim=(1, 3))
    assert torch.allclose(res[pad_x * naz + pad_z], expected)


def _positions(field, out):
    """where in ``field`` each value of ``out`` comes from: the moving windows only move values, and the values of a random field
    are distinct, so equality with ``field.flatten()[_positions(field, out)]`` is equality with ``out``"""
    flat = field.reshape(-1)
    assert flat.numel() <= 2 ** 15                                # stored as int16
    order = torch.argsort(flat)
    pos = order[torch.searchsorted(flat[order], out.reshape(-1)).clamp(max=flat.numel() - 1)]
    assert torch.equal(flat[pos], out.reshape(-1))
    return pos.reshape(out.shape).to(torch.int16)


def test_equal_to_the_reference_functions():
    ox = reference_values.module("fluidgym.envs.util.obs_extraction")
    torch.manual_seed(1)
    for n, w, k in ((8, 12, 1), (8, 12, 3), (12, 8, 11)):
        f = torch.rand(3, 10, n * w)
        mine = extract_moving_window_2d(f, n, w, k)
        for b in range(3):
            pos = reference_values.value(f"window_2d_{n}_{w}_{k}_{b}", ox and (lambda: _positions(f[b], ox.extract_moving_window_2d(
                f[b], n_agents=n, agent_width=w, n_agents_per_window=k))), _positions(f[b], mine[b]))
            assert torch.equal(mine[b], f[b].reshape(-1)[pos.long()])
    for nax, naz, aw, wx, wz, px, pz in ((10, 20, 2, 1, 1, 0, 0), (20, 40, 2, 5, 3, 4, 1), (10, 20, 4, 5, 5, 4, 4), (8, 8, 2, 3, 3, 1, 1)):
        f = torch.rand(2, naz * aw, nax * aw)
        mine = agent_window_means(f, nax, naz, aw, wx, wz, px, pz)
        for b in range(2):
            ref = reference_values.value(f"window_2d_x_z_{nax}_{naz}_{aw}_{wx}_{wz}_{px}_{pz}_{b}", ox and (lambda: ox.extract_moving_window_2d_x_z(
                field=f[b], n_agents_x=nax, n_agents_z=naz, agent_width=aw, n_agents_per_window_x=wx, n_agents_per_window_z=wz,
                pad_x=px, pad_z=pz)), mine[b])
            assert torch.allclose(mine[b], ref, atol=1e-7)
    for n, w, k in ((4, 3, 1), (4, 3, 3), (6, 2, 5), (8, 4, 3)):
        f = torch.rand(2, n * w, 7, n * w)
        mine = extract_moving_window_3d(f, n, w, k)
        for b in range(2):
            pos = reference_values.value(f"window_3d_{n}_{w}_{k}_{b}", ox and (lambda: _positions(f[b], ox.extract_moving_window_3d(
                f[b], n_agents=n, agent_width=w, n_agents_per_window=k))), _positions(f[b], mine[b]))
            assert torch.equal(mine[b], f[b].reshape(-1)[pos.long()])


def test_spanwise_local_windows_equal_the_reference():
    """transform_global_to_local_obs_3d (CylinderJet3D / Airfoil3D multi-agent observations)"""
    ox = reference_values.module("fluidgym.envs.util.obs_extraction")
    from fluidgym_b200.envs.spanwise import local_obs_windows
    torch.manual_seed(2)
    for n_agents, window in ((8, 3), (8, 1), (6, 5)):
        g = {"velocity": torch.rand(2, n_agents, 2, 3, 11), "pressure": torch.rand(2, n_agents, 2, 11)}
        mine = local_obs_windows(g, window)
        for b in range(2):
            ref = ox and ox.transform_global_to_local_obs_3d({k: v[b] for k, v in g.items()}, local_obs_window=window, n_agents=n_agents)
            for k in g:
                pos = reference_values.value(f"local_obs_{n_agents}_{window}_{b}_{k}", ref and (lambda: _positions(g[k][b], ref[k])),
                                             _positions(g[k][b], mine[k][b]))
                assert torch.equal(mine[k][b], g[k][b].reshape(-1)[pos.long()]), (n_agents, window, k)
