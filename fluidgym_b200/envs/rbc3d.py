"""Batched ``RBC3D`` (three-dimensional Rayleigh-Benard convection, bottom plate of n x n heaters) environment.

Mirrors ``envs/rbc/rbc_env_3d.py`` + ``rbc_env_base.py`` of the reference with ``ndims = 3``: the 2-D wall-refined grid
extruded uniformly in z (periodic x and z, no-slip plates at -y / +y), temperature as passive scalar with the buoyancy
source ``(0, T, 0)``, orthogonal solver path (``non_orthogonal=False``), heater actuation (zero-mean, clamped, cubic
blend applied along x and then along z, rbc_env_3d.py:205-272), Nusselt reward, sensors read from the rendered voxel grid
(``n_heaters * 4`` x 8 x ``n_heaters * 4``) and the multi-agent interface (one agent per heater, circular moving windows
in x and z, obs_extraction.py:255-330).  The solver is the D = 3 orthogonal box path (``fgb_ortho3_*`` with the scalar
attached, ``csrc/ortho3_b200.cuh``).  All tensors carry a leading environment dimension.
"""
from __future__ import annotations

import numpy as np
import torch

from .. import native
from ..box3d import BatchedPISO3D, Box3DDomain
from ..grids import wall_refined_ortho_grid
from ..sensors import sensor_tables_3d
from ..solver import _ptr, cfl_substeps
from .common import EpisodeLifecycle, InitialDomains3D, Renderable

RBC_3D_DEFAULT_CONFIG = {
    "rayleigh_number": 2e3, "prandtl_number": 0.7, "n_heaters": 8, "resolution": 8, "dt": 0.05, "adaptive_cfl": 0.8,
    "step_length": 1.0, "episode_length": 200, "local_obs_window": 3, "local_reward_weight": 0.0015, "uniform_grid": False,
    "aspect_ratio": 1.0, "use_marl": True,
}


def rbc3d_vertex_grid(nx: int, ny: int, L: float, H: float, base: float) -> np.ndarray:
    """[3, nz+1, ny+1, nx+1] float32: make_wall_refined_ortho_grid extruded with linear z weights over [0, L]
    (rbc_env_base.py:190-208, shapes.py:641-676), nz = nx."""
    g2 = wall_refined_ortho_grid(nx, ny, (0, -H / 2), (L, H / 2), ["-y", "+y"], base)
    nz = nx
    zs = np.asarray([0.0 * (1 - w) + L * w for w in (k / nz for k in range(nz + 1))], dtype=np.float32)
    out = np.zeros((3, nz + 1, ny + 1, nx + 1), dtype=np.float32)
    out[0], out[1] = g2[0][None], g2[1][None]
    out[2] = zs[:, None, None]
    return out


def extract_moving_window_3d(field: torch.Tensor, n_agents: int, agent_width: int, n_agents_per_window: int) -> torch.Tensor:
    """[..., Z, Y, X] -> [..., n_agents**2, wZ, Y, wX]: circular windows of ``n_agents_per_window`` heaters in x and z centred
    on every agent, agent index = z_agent * n_agents + x_agent (obs_extraction.py:255-330, batched)."""
    *lead, Z, Y, X = field.shape
    assert X == n_agents * agent_width and Z == n_agents * agent_width
    dev = field.device
    pad = n_agents_per_window // 2
    idx = (torch.arange(n_agents, device=dev)[:, None] + torch.arange(n_agents_per_window, device=dev)[None, :] - pad) % n_agents
    cells = (idx[:, :, None] * agent_width + torch.arange(agent_width, device=dev)[None, None, :]).reshape(n_agents, -1)   # [A, w*aw]
    fz = field[..., cells, :, :]                    # [..., Az, wZ, Y, X]
    fzx = fz[..., cells]                            # [..., Az, wZ, Y, Ax, wX]
    fzx = fzx.movedim(-2, -4)                       # [..., Az, Ax, wZ, Y, wX]
    return fzx.reshape(*lead, n_agents * n_agents, cells.shape[1], Y, cells.shape[1])


class RBC3DEnv(EpisodeLifecycle, InitialDomains3D, Renderable):
    T_cold, T_hot, heater_limit = 0.0, 1.0, 0.75
    n_sensors_y, n_sensors_per_heater = 8, 4
    buoyancy_factor = 1.0
    H = 1.0
    resolution_scale_y, grid_base = 2.0, 1.02
    metrics = ["nusselt"]
    reference_values = {"nu_ref": ("nusselt", "mean")}
    render_fields = ("temperature", "velocity_magnitude", "q_criterion", "pressure")

    def __init__(self, n_envs: int = 1, rayleigh_number=2e3, prandtl_number=0.7, n_heaters=8, resolution=8, dt=0.05,
                 adaptive_cfl=0.8, step_length=1.0, episode_length=200, local_obs_window=3, local_reward_weight=0.0015,
                 uniform_grid=False, aspect_ratio=1.0, use_marl=True, device="cuda:0", nu_ref=0.0, randomize_initial_state=False,
                 enable_actions=True, load_initial_domain=False, initial_domains_path=None, transforms=None, btransforms=None,
                 differentiable=False, per_env_substeps: bool = False):
        self.per_env_substeps = bool(per_env_substeps)
        self.n_envs = int(n_envs)
        self.differentiable = bool(differentiable)
        self.load_domain_on_reset, self.initial_domains_path = bool(load_initial_domain), initial_domains_path
        self.rayleigh_number, self.prandtl_number = rayleigh_number, prandtl_number
        self.Ra, self.Pr = float(rayleigh_number), float(prandtl_number)
        self.n_heaters, self.heater_width = int(n_heaters), int(resolution)
        self.dt, self.cfl = float(dt), float(adaptive_cfl)
        self.step_length, self.episode_length = float(step_length), int(episode_length)
        self.local_obs_window, self.local_reward_weight = int(local_obs_window), local_reward_weight
        self.use_marl, self.nu_ref = bool(use_marl), float(nu_ref)
        self.enable_actions, self.randomize_initial_state = enable_actions, randomize_initial_state
        self.device = torch.device(device)
        self.aspect = aspect_ratio * torch.pi
        self.nx = self.nz = int(resolution * n_heaters)
        self.ny = round(self.resolution_scale_y * self.nx / self.aspect)
        self.L = self.H * self.aspect
        self.nu = float(torch.tensor([(prandtl_number / rayleigh_number) ** 0.5], dtype=torch.float32)[0])
        self.kappa = float(torch.tensor([(rayleigh_number * prandtl_number) ** -0.5], dtype=torch.float32)[0])
        vertex = rbc3d_vertex_grid(self.nx, self.ny, self.L, self.H, 1.0 if uniform_grid else self.grid_base)
        self.dom = Box3DDomain(vertex, closed=(False, True, False), viscosity=self.nu, transforms=transforms, btransforms=btransforms)
        self.solver = BatchedPISO3D(self.dom, self.n_envs, device=device, corrector_steps=2, advection_tol=1e-5, pressure_tol=1e-5,
                                    non_orthogonal=False)
        self.lib = self.solver.lib
        nface = self.nx * self.nz
        self._bottom = slice(self.dom.boff[2], self.dom.boff[2] + nface)            # -y face: heaters, faces in (z, x) order
        self._top = slice(self.dom.boff[3], self.dom.boff[3] + nface)
        sb0 = np.zeros(self.dom.NB, dtype=np.float32)
        sb0[self._bottom], sb0[self._top] = self.T_hot, self.T_cold
        self._sb0 = sb0
        self.solver.attach_scalar(self.kappa, self.buoyancy_factor, sbval0=sb0)
        self.cell_size = torch.from_numpy(np.ascontiguousarray(self.dom.det, dtype=np.float32)).to(self.device)     # [nz, ny, nx]
        self._setup_sensors()
        self._zero_action = torch.zeros(self.n_envs, self.n_heaters ** 2, 1, device=self.device) if self.use_marl else \
            torch.zeros(self.n_envs, self.n_heaters, self.n_heaters, 1, device=self.device)

    # ---- static tables ---------------------------------------------------------------------------
    @property
    def render_shape(self):
        nx = self.n_heaters * 20
        return (nx, round(nx / self.aspect), nx)

    @property
    def n_sensors_x(self):
        return self.n_heaters * self.n_sensors_per_heater

    def _render_planes(self):
        Z = self.render_shape[2]
        return Z, Z // 2

    def _build_render_map(self, plane):
        from ..render import render_map_box3d
        return render_map_box3d(self.dom.vertex, self.render_shape, plane, fill_max_steps=16)

    def _setup_sensors(self):
        """rbc_env_base.py:445-470 + rbc_env_3d.py:183-203: (x, y) sensor voxels x-major, every pair repeated over z."""
        nx, ny, nz = self.render_shape
        nsx, nsy = self.n_sensors_x, self.n_sensors_y
        sx = torch.linspace(0, nx, nsx + 1)[:-1] + nx / (2 * nsx)
        sy = torch.linspace(0, ny, nsy + 1)[:-1] + ny / (2 * nsy)
        gx, gy = torch.meshgrid(sx, sy, indexing="ij")
        loc2 = torch.stack([gx, gy], dim=-1).reshape(-1, 2).T.round().to(torch.int)
        sz = (torch.linspace(0, nz, nsx + 1)[:-1] + nz / (2 * nsx)).round().to(torch.int)
        x = loc2[0].repeat_interleave(nsx)
        y = loc2[1].repeat_interleave(nsx)
        z = sz.repeat(loc2.shape[1])
        self.sensor_px = torch.stack([x, y, z]).numpy()                 # [3, nsx * nsy * nsx], order (x, y, z) with z fastest
        idx, w = sensor_tables_3d(self.dom.vertex, (nx, ny, nz), self.sensor_px, fill_max_steps=16)
        self.sens_idx = torch.from_numpy(idx).to(self.device)
        self.sens_w = torch.from_numpy(w).to(self.device)

    # ---- reference-shaped API ---------------------------------------------------------------------
    @property
    def n_agents(self):
        return self.n_heaters ** 2 if self.use_marl else 1

    @property
    def initial_domain_id(self):
        """rbc_env_base.py:606-611"""
        return f"rbc_3d_Ra{self.rayleigh_number}_Pr{self.prandtl_number}_NH{self.n_heaters}_HW{self.heater_width}"

    @property
    def observation_space(self):
        from .. import spaces
        w = self.n_sensors_per_heater * (self.local_obs_window if self.use_marl else self.n_heaters)
        shape = (w, self.n_sensors_y, w)
        inf = float("inf")
        return spaces.Dict({"temperature": spaces.Box(self.T_cold, self.T_hot + self.heater_limit, shape=shape),
                            "velocity": spaces.Box(-inf, inf, shape=(3,) + shape), "pressure": spaces.Box(-inf, inf, shape=shape)})

    @property
    def action_space(self):
        from .. import spaces
        return spaces.Box(-1.0, 1.0, shape=(1,) if self.use_marl else (self.n_heaters, self.n_heaters, 1))

    def set_state(self, u, p, T, sbval=None, ures=None):
        s = self.solver
        for dst, src in ((s.u, u), (s.p, p), (s.T, T)):
            self._copy_state(dst, src)
        if sbval is not None:
            self._copy_state(s.sbval, sbval)
        ur = s.buffer("ures")
        if ures is None:
            ur.zero_()
        else:
            self._copy_state(ur, ures)
        self._reset_called = True

    def reset(self, seed: int | None = None, randomize: bool | None = None):
        """rbc_env_base.py:190-278 with ndims = 3: linear temperature profile + 0.1 N(0,1) clamped to [T_cold, T_hot], velocity
        0.05 N(0,1); ``randomize`` adds the mirror / shift / noise / settling of rbc_env_base.py:336-393 per environment."""
        self._begin_reset(seed)
        s = self.solver
        B, nx, ny, nz = self.n_envs, self.nx, self.ny, self.nz
        randomize = self.randomize_initial_state if randomize is None else randomize
        if self.load_domain_on_reset:                      # fluid_env.py:519-551
            self._load_initial_domains_on_reset(randomize)
            s.buffer("ures").copy_(s.u)
            if randomize:
                self._randomize_domain()
            self._apply_action(self._zero_action)
            self._reset_called, self._n_steps = True, 0
            return (self._get_local_obs() if self.use_marl else self._get_global_obs()), {}
        grad = torch.linspace(self.T_hot, self.T_cold, steps=ny, device=self.device)[None, :, None].expand(nz, ny, nx)
        T0 = grad[None] + torch.randn(B, nz, ny, nx, device=self.device, generator=self._torch_rng) * 0.1 * (self.T_hot - self.T_cold)
        s.T.copy_(torch.clamp(T0, self.T_cold, self.T_hot).reshape(B, -1))
        s.u.copy_(torch.randn(B, 3, nz * ny * nx, device=self.device, generator=self._torch_rng) * 0.05)
        s.p.zero_()
        s.buffer("ures").zero_()
        s.sbval.copy_(torch.from_numpy(self._sb0).to(self.device).unsqueeze(0).expand_as(s.sbval))
        if randomize:
            self._randomize_domain()
        self._apply_action(self._zero_action)
        self._reset_called, self._n_steps = True, 0
        return (self._get_local_obs() if self.use_marl else self._get_global_obs()), {}

    def _randomize_domain(self):
        """rbc_env_base.py:336-393: mirror in x / in z with probability 1/2 each (the matching velocity component changes
        sign), periodic shifts in x and z, N(0, 0.05) noise on T (clamped) and u, 1-2 time units of settling.  Mirrors and
        shifts are drawn per environment; the settling time is common to the batch."""
        s = self.solver
        B, nx, ny, nz = self.n_envs, self.nx, self.ny, self.nz
        rng = self._np_rng
        flip = {0: rng.uniform(0.0, 1.0, size=B) > 0.5, 2: rng.uniform(0.0, 1.0, size=B) > 0.5}
        shift = {0: rng.integers(0, nx, size=B), 2: rng.integers(0, nx, size=B)}
        T = s.T.reshape(B, nz, ny, nx)
        u = s.u.reshape(B, 3, nz, ny, nx).clone()
        for comp, axis, n in ((0, 4, nx), (2, 2, nz)):          # velocity component, array axis of u [B,3,z,y,x], cells
            fl = torch.from_numpy(flip[comp]).to(self.device)
            sh = torch.from_numpy(shift[comp]).to(self.device)
            pos = torch.arange(n, device=self.device)
            src = (pos[None, :] - sh[:, None]) % n                                   # roll(mirror(field), shift)
            src = torch.where(fl[:, None], n - 1 - src, src)
            shp = [B, 1, 1, 1, 1]
            shp[axis] = n
            u = torch.gather(u, axis, src.reshape(shp).expand_as(u)).clone()
            T = torch.gather(T, axis - 1, src.reshape([B] + shp[2:]).expand_as(T))
            u[:, comp] = torch.where(fl[:, None, None, None], -u[:, comp], u[:, comp])
        T = torch.clamp(T + torch.randn(T.shape, device=self.device, generator=self._torch_rng) * 0.05, self.T_cold, self.T_hot)
        u = u + torch.randn(u.shape, device=self.device, generator=self._torch_rng) * 0.05
        s.T.copy_(T.reshape(B, -1))
        s.u.copy_(u.reshape(B, 3, -1))
        for _ in range(int(rng.uniform(1.0, 2.0) / self.dt)):
            s.single_step(self.dt, self.cfl)

    # ---- actuation ---------------------------------------------------------------------------------
    def _smooth_1d(self, T_action: torch.Tensor) -> torch.Tensor:
        """[..., n_heaters] -> [..., nx]: cubic blend between neighbouring heaters along the last axis (rbc_env_3d.py:205-247)."""
        hw = self.heater_width
        bw = round(hw * 0.1)
        T_left, T_right = torch.roll(T_action, 1, dims=-1), torch.roll(T_action, -1, dims=-1)
        x_idx = torch.arange(self.nx, device=T_action.device)
        seg, xpos = x_idx // hw, x_idx % hw
        T0, T1, T2 = T_left[..., seg], T_action[..., seg], T_right[..., seg]
        left_zone, right_zone = xpos < bw, xpos >= hw - bw
        tL = (xpos.to(torch.float32) / bw + 0.5).clamp(0.0, 1.0) if bw > 0 else torch.ones_like(xpos, dtype=torch.float32)
        tR = 1 - torch.roll(tL, shifts=hw - bw + 1, dims=-1)

        def blend(t, A, Bv):
            sm = t * t * (3 - 2 * t)
            return (1 - sm) * A + sm * Bv

        return torch.where(left_zone, blend(tL, T0, T1), torch.where(right_zone, blend(tR, T1, T2), T1))

    def _action_to_control(self, action: torch.Tensor) -> torch.Tensor:
        """[B, n, n] -> bottom-plate temperature [B, nz, nx] (rbc_env_3d.py:249-272): the 1-D profile is applied to the
        transposed array twice, i.e. first along the first heater axis, then along the second."""
        T_shifted = action - action.mean(dim=(1, 2), keepdim=True)
        T_action = T_shifted / (torch.clamp(T_shifted.abs(), min=1.0) / self.heater_limit) + self.T_hot
        smooth_x = self._smooth_1d(T_action.transpose(1, 2))            # [B, n(second), nx(first)]
        return self._smooth_1d(smooth_x.transpose(1, 2))                # [B, nx(first), nx(second)]

    def _apply_action(self, action):
        a = torch.as_tensor(action, dtype=torch.float32, device=self.device).reshape(self.n_envs, self.n_heaters, self.n_heaters)
        self.solver.sbval[:, self._bottom] = self._action_to_control(a).reshape(self.n_envs, -1)

    # ---- observations / rewards ----------------------------------------------------------------------
    def _sample(self, field, channels):
        s = self.solver
        ns, K = self.sens_idx.shape[1], self.sens_idx.shape[0]
        out = torch.empty(self.n_envs, channels, ns, device=self.device)
        native.check(self.lib.fgb_sample_sensors_n(_ptr(field), self.n_envs, channels, s.N, _ptr(self.sens_idx), _ptr(self.sens_w), K, ns,
                                                   _ptr(out), s.stream), "fgb_sample_sensors_n")
        # sensors are enumerated (x, y, z) with z fastest; the reference reshapes to [n_sx, n_sy, n_sx] and permutes to (z, y, x)
        nsx, nsy = self.n_sensors_x, self.n_sensors_y
        return out.reshape(self.n_envs, channels, nsx, nsy, nsx).permute(0, 1, 4, 3, 2).contiguous()

    def _get_global_obs(self):
        s = self.solver
        return {"temperature": self._sample(s.T, 1)[:, 0], "velocity": self._sample(s.u, 3), "pressure": self._sample(s.p, 1)[:, 0]}

    def _get_local_obs(self):
        g = self._get_global_obs()
        w = dict(n_agents=self.n_heaters, agent_width=self.n_sensors_per_heater, n_agents_per_window=self.local_obs_window)
        T = extract_moving_window_3d(g["temperature"], **w)
        u = torch.stack([extract_moving_window_3d(g["velocity"][:, c], **w) for c in range(3)], dim=2)
        p = extract_moving_window_3d(g["pressure"], **w)
        return {"temperature": T, "velocity": u, "pressure": p}

    def _fields(self):
        s = self.solver
        B = self.n_envs
        u, T = getattr(self, "_dfields", None) or (s.u, s.T)      # differentiable mode: the tensors that carry the graph
        return T.reshape(B, self.nz, self.ny, self.nx), u[:, 1].reshape(B, self.nz, self.ny, self.nx)

    def compute_global_nusselt(self):
        """rbc_env_base.py:491-539: Nu = 1 + sqrt(Ra Pr) <u_y T>_V"""
        T, uy = self._fields()
        q = (uy * T * self.cell_size).sum(dim=(1, 2, 3)) / self.cell_size.sum()
        return 1.0 + (self.Ra * self.Pr) ** 0.5 * q

    def _get_local_rewards(self):
        """rbc_env_3d.py:374-409: Nusselt number over every agent's window; as in the reference the cell volumes are those of
        the FIRST window * heater_width columns in x and z for every agent."""
        T, uy = self._fields()
        w = dict(n_agents=self.n_heaters, agent_width=self.heater_width, n_agents_per_window=self.local_obs_window)
        k = self.local_obs_window * self.heater_width
        cs = self.cell_size[:k, :, :k]
        lT, lu = extract_moving_window_3d(T, **w), extract_moving_window_3d(uy, **w)        # [B, A, k, ny, k]
        q = (lu * lT * cs).sum(dim=(2, 3, 4)) / cs.sum()
        return self.nu_ref - (1.0 + (self.Ra * self.Pr) ** 0.5 * q)

    # ---- differentiable mode: one autograd node per substep (autograd.PISOSubstepScalar3D, CUDA adjoint of the D = 3 box path); the
    # heater profile and the Nusselt integrals around it are torch expressions, as in the reference.  The CFL plan is taken from
    # detached maxima with one common substep size for the batch (the most restrictive environment decides), or with per_env_substeps
    # every environment's own plan (EpisodeLifecycle._substep_rounds).
    def mark_state_differentiable(self):
        """envs/util/diff_tools.py:8-22: (velocity, temperature) leaves of the incoming state"""
        s = self.solver
        u, T = s.u.detach().clone().requires_grad_(True), s.T.detach().clone().requires_grad_(True)
        self._dstate = (u, s.p.detach().clone(), T, s.sbval.detach().clone())
        return u, T

    def _advance_differentiable(self, action):
        from ..autograd import piso_substep_scalar_3d
        s = self.solver
        if self._dstate is None:
            self._dstate = (s.u.clone(), s.p.clone(), s.T.clone(), s.sbval.clone())
        u, p, T, sb = self._dstate
        if self.enable_actions:
            ctrl = self._action_to_control(action.reshape(self.n_envs, self.n_heaters, self.n_heaters)).reshape(self.n_envs, -1)
            sb = sb.index_copy(1, torch.arange(self._bottom.start, self._bottom.stop, device=self.device), ctrl)
        bv = s.bvel
        minv, b_minv = s._tab["minv"].reshape(1, 3, -1), s._tab["b_minv"].reshape(1, 3, -1)

        def max_velocity():
            with torch.no_grad():
                return float(torch.maximum((minv * u).abs().max(), (b_minv * bv).abs().max()))

        def max_velocity_env():
            with torch.no_grad():
                return torch.maximum((minv * u).abs().amax(dim=(1, 2)), (b_minv * bv).abs().amax(dim=(1, 2)))
        nsub = 0
        self._begin_substep_count()
        for _ in range(self.n_sim_steps):
            if self.per_env_substeps:
                for dtv, act in self._substep_rounds(max_velocity_env):
                    u, p, T = piso_substep_scalar_3d(s, u, p, bv, T, sb, dtv, active=act)
                    nsub += 1
                continue
            for ts in cfl_substeps(self.dt, self.cfl, max_velocity):                 # SIM.py:2004-2031
                u, p, T = piso_substep_scalar_3d(s, u, p, bv, T, sb, ts)
                nsub += 1
        self._dstate = (u, p, T, sb)
        with torch.no_grad():                      # keep the solver's own state in step for observations / get_state
            s.u.copy_(u); s.p.copy_(p); s.T.copy_(T); s.sbval.copy_(sb)
        self.last_substeps = nsub
        return u, T

    def step(self, action):
        action = self._begin_step(action)
        if self.differentiable:
            self._dfields = self._advance_differentiable(action)
        else:
            self._dfields = None
            if self.enable_actions:
                self._apply_action(action)
            nsub = 0
            for _ in range(self.n_sim_steps):
                nsub += self.solver.single_step(self.dt, self.cfl)
            self.last_substeps = nsub
        nu = self.compute_global_nusselt()
        reward = self.nu_ref - nu
        info = {"nusselt": nu.detach()}
        truncated = self._end_step()
        if not self.use_marl:
            return self._get_global_obs(), reward, False, truncated, info
        lw = self.local_reward_weight
        local = self._get_local_rewards() if lw > 0 else torch.zeros(self.n_envs, self.n_agents, device=self.device)
        info["global_reward"] = reward
        return self._get_local_obs(), lw * local + (1 - lw) * reward[:, None], False, truncated, info
