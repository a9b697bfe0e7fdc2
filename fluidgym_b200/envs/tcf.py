"""Batched 3-D turbulent-channel-flow environments (``TCF3DBottomEnv`` / ``TCF3DBothEnv``, envs/tcf/tcf_env.py):
wall blowing / suction actuators on a grid of ``actor_size x actor_size`` patches, reward = wall-shear-stress
reduction, observation = velocity fluctuation and pressure on the plane y+ = 15 (per-agent window means in MARL
mode).  Solver: the D = 3 orthogonal path (``fluidgym_b200/box3d.py`` -> ``fgb_ortho3_*``); the dynamic forcing and the
wall shear are device stages of it.
"""
from __future__ import annotations

import numpy as np
import torch

from ..box3d import BatchedPISO3D, Box3DDomain
from ..grids import channel_vertex_grid
from ..solver import cfl_substeps
from .common import EpisodeLifecycle, InitialDomains3D, Renderable

SMALL_TCF_3D_DEFAULT_CONFIG = {
    "resolution_y": 65, "resolution_x_z": 64, "actor_size": 2, "L": np.pi, "D": np.pi / 2, "reynolds_number_wall": 180,
    "adaptive_cfl": 0.1, "step_length": 0.6, "episode_length": 1000, "local_obs_window": 1, "local_reward_weight": 0.0,
    "use_marl": True, "C_smag": 0.0, "use_van_driest": False, "init_with_noise": False,
}
LARGE_TCF_3D_DEFAULT_CONFIG = {**SMALL_TCF_3D_DEFAULT_CONFIG, "resolution_x_z": 128, "L": 2 * np.pi, "D": np.pi}


def re_wall_to_cl(re_wall: float) -> float:
    """TCF_tools.Re_wall_to_cl"""
    return (re_wall / 0.116) ** (1 / 0.88)


def agent_window_means(field, n_agents_x, n_agents_z, agent_width, wx, wz, pad_x, pad_z):
    """[..., Z, X] -> [..., n_agents_x * n_agents_z, wz, wx]: circular windows of per-agent patch means, agents ordered x-major
    (extract_moving_window_2d_x_z, envs/util/obs_extraction.py:255-343)."""
    lead = field.shape[:-2]
    fa = field.reshape(*lead, n_agents_z, agent_width, n_agents_x, agent_width).mean(dim=(-3, -1))       # [..., naz, nax]
    fa = torch.roll(fa, shifts=(pad_z, pad_x), dims=(-2, -1))
    iz = (torch.arange(n_agents_z, device=field.device)[:, None] + torch.arange(wz, device=field.device)[None, :]) % n_agents_z
    ix = (torch.arange(n_agents_x, device=field.device)[:, None] + torch.arange(wx, device=field.device)[None, :]) % n_agents_x
    win = fa[..., iz[:, None, :, None], ix[None, :, None, :]]                                            # [..., naz, nax, wz, wx]
    win = win.transpose(-4, -3)                                                                          # x outer, z inner
    return win.reshape(*lead, n_agents_x * n_agents_z, wz, wx)


class TCF3DEnv(EpisodeLifecycle, InitialDomains3D, Renderable):
    delta, H = 1.0, 2.0
    y_obs_wall = 15.0
    metrics = ["wall_stress", "wall_stress_bottom", "wall_stress_top"]
    both_walls = False
    render_fields = ("velocity_x", "velocity_magnitude", "pressure", "q_criterion")

    def __init__(self, n_envs: int = 1, resolution_y=65, resolution_x_z=64, actor_size=2, L=np.pi, D=np.pi / 2, reynolds_number_wall=180,
                 adaptive_cfl=0.1, step_length=0.6, episode_length=1000, local_obs_window=1, local_reward_weight=0.0, use_marl=True,
                 C_smag=0.0, use_van_driest=False, init_with_noise=False, device="cuda:0", tau_ref=1.0, randomize_initial_state=False,
                 enable_actions=True, domain=None, load_initial_domain=False, initial_domains_path=None, differentiable=False,
                 per_env_substeps: bool = False):
        self.per_env_substeps = bool(per_env_substeps)
        if init_with_noise:
            raise NotImplementedError("init_with_noise needs the reference's optional simplex-noise extension; start from a state instead")
        self.n_envs = int(n_envs)
        self.differentiable = bool(differentiable)
        self.load_domain_on_reset, self.initial_domains_path = bool(load_initial_domain), initial_domains_path
        self.L, self.D = float(L), float(D)
        self.re_wall = float(reynolds_number_wall)
        self.re_center = re_wall_to_cl(self.re_wall)
        self.viscosity = float(torch.tensor([self.delta / self.re_center], dtype=torch.float32)[0])
        self.u_wall = self.re_wall / self.re_center
        self.x = self.z = int(resolution_x_z)
        self.y = int(resolution_y)
        self.actor_size = int(actor_size)
        self.local_obs_window, self.local_reward_weight = int(local_obs_window), local_reward_weight
        self.use_marl = bool(use_marl)
        self.cfl = float(adaptive_cfl)
        self.step_length = step_length * (self.viscosity / self.u_wall ** 2)            # wall units -> physical time
        self.dt = self.step_length / 10
        self.episode_length = int(episode_length)
        self.tau_ref = float(tau_ref)
        self.randomize_initial_state, self.enable_actions = randomize_initial_state, enable_actions
        self.scale_actions = True
        self.device = torch.device(device)
        strength = self.grid_refinement_strength = 2 if resolution_x_z < 64 else 1          # tcf_env.py:252
        if domain is None:
            vertex = channel_vertex_grid(self.H, self.L, self.D, self.x, self.y // 2, strength, self.z)
            domain = Box3DDomain(vertex, closed=(False, True, False), viscosity=self.viscosity)
        self.dom = domain
        self.ny = domain.ny
        self.solver = BatchedPISO3D(domain, self.n_envs, device=device, corrector_steps=2, advection_tol=1e-6, pressure_tol=1e-6)
        self.lib = self.solver.lib
        dev = self.device
        cc = torch.from_numpy(domain.cell_centres())                      # [3, nz, ny, nx]
        pos_y = torch.mean(cc[1], dim=(0, 2))
        self.d_lo, self.d_hi = float(1 + pos_y[0].numpy()), float(1 - pos_y[-1].numpy())
        cells = np.arange(domain.N).reshape(domain.shape)
        self.rows = torch.from_numpy(np.stack([cells[:, 0, :].ravel(), cells[:, -1, :].ravel()]).astype(np.int32)).to(dev)
        y_obs = -self.delta + self.y_obs_wall / ((1 / self.viscosity) * self.u_wall)
        self.y_obs_bottom_idx = int(torch.argmin(torch.abs(cc[1, 0, :, 0] - y_obs)))
        self.y_obs_top_idx = self.y - self.y_obs_bottom_idx                # tcf_env.py:1141 (uses resolution_y, as the reference)
        self.cell_size = torch.from_numpy(domain.det.copy()).to(dev)      # [nz, ny, nx]
        # Smagorinsky sub-grid viscosity with optional van Driest wall damping (tcf_env.py:441-472, envs/tcf/grid.py:75-125)
        self.C_smag, self.use_van_driest = float(C_smag), bool(use_van_driest)
        if self.C_smag != 0.0:
            damp = None
            if self.use_van_driest:
                wd_cells = (1 - torch.abs(cc[1].to(torch.float32))) * self.u_wall / torch.tensor([self.viscosity], dtype=torch.float32)
                vd = 1 - torch.exp(-wd_cells * (1.0 / 25.0))
                damp = (vd * vd).numpy()
            self.solver.set_sgs(self.C_smag, damp)
        # initial state: Reichardt mean profile (envs/tcf/grid.py:83-98)
        wd = (1 - torch.abs(cc[1, 0, :, 0])) * self.u_wall / torch.tensor([self.viscosity], dtype=torch.float32)
        k = 0.41
        prof = (1 / k) * torch.log(1 + k * wd) + 7.8 * (1 - torch.exp(-wd / 11.0) - (wd / 11.0) * torch.exp(-wd / 3))
        self.u_init = (prof * self.u_wall).to(torch.float32)              # [ny]
        self.nax, self.naz = self.x // self.actor_size, self.z // self.actor_size
        self._face_lo = slice(domain.boff[2], domain.boff[2] + self.x * self.z)
        self._face_hi = slice(domain.boff[3], domain.boff[3] + self.x * self.z)
        self._acc = torch.zeros(self.n_envs, 2, device=dev)
        shape = (self.n_agents, 1)
        self._zero_action = torch.zeros(self.n_envs, *shape, device=dev)

    # ---- reference-shaped API ---------------------------------------------------------------------
    @property
    def n_agents(self):
        return self.nax * self.naz * (2 if self.both_walls else 1)

    @property
    def initial_domain_id(self):
        """tcf_env.py:866-872"""
        return f"channel_flow3D_L{self.L:.2f}_Re{int(self.re_wall)}_Res{self.x}_Ref{self.grid_refinement_strength}"

    @property
    def observation_space(self):
        from .. import spaces
        inf, w = float("inf"), self.local_obs_window
        vs, ps = ((w, w, 2), (w, w)) if self.use_marl else ((2, self.z, self.x), (self.z, self.x))
        if self.both_walls and not self.use_marl:
            vs, ps = (2,) + vs, (2,) + ps
        return spaces.Dict({"velocity": spaces.Box(-inf, inf, shape=vs), "pressure": spaces.Box(-inf, inf, shape=ps)})

    @property
    def action_space(self):
        from .. import spaces
        return spaces.Box(-1.0, 1.0, shape=(1,) if self.use_marl else (self.n_agents, 1))

    def set_state(self, u, p, bvel=None):
        s = self.solver
        for dst, src in ((s.u, u), (s.p, p)) + (((s.bvel, bvel),) if bvel is not None else ()):
            self._copy_state(dst, src)
        self._reset_called = True

    def get_state(self):
        s = self.solver
        return dict(u=s.u.clone(), p=s.p.clone(), bvel=s.bvel.clone())

    def reset(self, seed: int | None = None, randomize: bool | None = None):
        self._begin_reset(seed)
        s = self.solver
        randomize = self.randomize_initial_state if randomize is None else randomize
        if self.load_domain_on_reset:                      # fluid_env.py:519-551
            self._load_initial_domains_on_reset(randomize)
            # the reference projects loaded domains as well: _get_simulation always ends with CopyVelocityResultFromBlocks +
            # make_divergence_free (tcf_env.py:478-511), which also replaces the stored pressure by the projection pressure
            s.make_divergence_free(max_iter=1000)
        else:
            u0 = torch.zeros(3, self.z, self.ny, self.x)
            u0[0] = self.u_init[None, :, None]
            s.u.copy_(u0.reshape(1, 3, -1).to(self.device).expand_as(s.u))
            s.p.zero_()
            s.bvel.zero_()
            s.make_divergence_free(max_iter=1000)
        if randomize:
            self._randomize_domain()
        self._apply_action(self._zero_action)
        self._reset_called, self._n_steps = True, 0
        return self._get_obs(), {}

    def _randomize_domain(self):
        """tcf_env.py:879-916"""
        max_n = int(0.01 * self.episode_length)
        n_steps = int(self._np_rng.integers(int(0.5 * max_n), max_n)) + 1
        s = self.solver
        s.u += torch.randn(s.u.shape, device=self.device, generator=self._torch_rng) * 0.01
        s.p += torch.randn(s.p.shape, device=self.device, generator=self._torch_rng) * 0.01
        for _ in range(n_steps):
            s.single_step(self.dt, self.cfl, self.rows, self.d_lo, self.d_hi)

    def _action_to_control(self, a: torch.Tensor) -> torch.Tensor:
        """[B, nax, naz] -> wall-normal velocity [B, nz*nx] (tcf_env.py:521-547): zero net mass flux, |v| <= u_wall"""
        if self.scale_actions:
            a = a - a.mean(dim=(1, 2), keepdim=True)
            a = self.u_wall * a / torch.clamp(a.abs(), min=1.0)
            a = a - a.mean(dim=(1, 2), keepdim=True)
        v = a.repeat_interleave(self.actor_size, dim=1).repeat_interleave(self.actor_size, dim=2)     # [B, x, z]
        return v.transpose(1, 2).reshape(a.shape[0], -1)                                            # [B, z*x], x fastest

    def _apply_action(self, action):
        a = torch.as_tensor(action, dtype=torch.float32, device=self.device).reshape(self.n_envs, -1)
        s = self.solver
        half = self.nax * self.naz
        s.bvel[:, 1, self._face_lo] = self._action_to_control(a[:, :half].reshape(self.n_envs, self.nax, self.naz))
        if self.both_walls:
            s.bvel[:, 1, self._face_hi] = -1 * self._action_to_control(a[:, half:].reshape(self.n_envs, self.nax, self.naz))

    def _plane(self, y_idx):
        s = self.solver
        B = self.n_envs
        u = s.u.view(B, 3, self.z, self.ny, self.x)
        p = s.p.view(B, self.z, self.ny, self.x)
        return u[:, :2, :, y_idx, :], p[:, :, y_idx, :]

    def _global_obs_at(self, y_idx):
        """tcf_env.py:646-677: velocity minus its volume-weighted mean, on one wall-parallel plane"""
        s = self.solver
        B = self.n_envs
        u = s.u.view(B, 3, self.z, self.ny, self.x)
        mean_u = (u * self.cell_size).sum(dim=(2, 3, 4), keepdim=True) / self.cell_size.sum()
        up, pp = self._plane(y_idx)
        return {"velocity": up - mean_u[:, :2, :, 0, :], "pressure": pp.clone()}

    def _local_obs_at(self, y_idx, flip):
        """tcf_env.py:918-992"""
        up, pp = self._plane(y_idx)
        up = up - up.mean(dim=(2, 3), keepdim=True)
        w = self.local_obs_window
        kw = dict(n_agents_x=self.nax, n_agents_z=self.naz, agent_width=self.actor_size, wx=w, wz=w)
        ox = agent_window_means(up[:, 0], pad_x=w - 1, pad_z=w // 2, **kw)
        oy = agent_window_means(up[:, 1], pad_x=w, pad_z=w // 2, **kw)
        op = agent_window_means(pp, pad_x=w, pad_z=w // 2, **kw)
        if flip:
            ox = torch.flip(ox, dims=[3])
            oy = torch.flip(oy, dims=[3]) * -1
            op = torch.flip(op, dims=[2])
        return {"velocity": torch.stack((ox, oy), dim=-1), "pressure": op}

    def _render_planes(self):
        return self.ny, self.y_obs_bottom_idx

    def _build_render_map(self, plane):
        """the wall-parallel cell plane y = ``plane``, shown [z, x]: x and z are uniform, so the map is the identity"""
        from ..render import render_map_cell_plane
        return render_map_cell_plane(self.x, self.ny, self.z, plane)

    def q_criterion(self):
        """_get_q_criterion (tcf_env.py:586-644) on the cell grid [B, nz, ny, nx]: Q = (|Omega|^2 - |S|^2) / 2 from
        ComputeSpatialVelocityGradients (the reference then resamples it to its rendering grid, which is out of scope here)"""
        return self.solver.q_criterion().view(self.n_envs, self.z, self.ny, self.x)

    def _get_obs(self):
        if self.use_marl:
            b = self._local_obs_at(self.y_obs_bottom_idx, False)
            if not self.both_walls:
                return b
            t = self._local_obs_at(self.y_obs_top_idx, True)
            return {k: torch.cat((b[k], t[k]), dim=1) for k in b}
        b = self._global_obs_at(self.y_obs_bottom_idx)
        if not self.both_walls:
            return b
        t = self._global_obs_at(self.y_obs_top_idx)
        return {k: torch.stack((b[k], t[k]), dim=1) for k in b}

    # ---- differentiable mode (fluidgym.make(..., differentiable=True); reverse mode of the D = 3 substep, autograd.PISOSubstep3D) -------
    def _forcing_torch(self, u):
        """set_dynamic_forcing (envs/tcf/grid.py:128-163): G_x = nu / 2 (<u>_lo / d_lo + <u>_hi / d_hi); the reference rebuilds G with
        ``torch.tensor``: no gradient flows through it"""
        with torch.no_grad():
            ux = u[:, 0].reshape(self.n_envs, self.z, self.ny, self.x)
            tlo = self.viscosity * ux[:, :, 0, :].mean(dim=(1, 2)) / self.d_lo
            thi = self.viscosity * ux[:, :, -1, :].mean(dim=(1, 2)) / self.d_hi
            src = torch.zeros(self.n_envs, 4, device=self.device)
            src[:, 0] = 0.5 * (tlo + thi)
        return src

    def _wall_stress_torch(self, u):
        """_get_wall_stress (tcf_env.py:564-584) as differentiable torch ops -> (tau_bottom, tau_top) [B]"""
        ux = u[:, 0].reshape(self.n_envs, self.z, self.ny, self.x)
        return (self.viscosity * ux[:, :, 0, :].mean(dim=(1, 2)) / self.d_lo, self.viscosity * ux[:, :, -1, :].mean(dim=(1, 2)) / self.d_hi)

    def _single_step_differentiable(self, u, p, bv):
        """Simulation.single_step with the adaptive CFL plan (SIM.py:2004-2031, k3_plan_substep); the plan is not differentiated.
        One common substep size for the batch (the most restrictive environment decides), or with ``per_env_substeps`` every
        environment's own plan."""
        from ..autograd import piso_substep_3d
        s = self.solver
        minv = s._tab["minv"].reshape(1, 3, -1)
        b_minv = s._tab["b_minv"].reshape(1, 3, -1)
        nsub = 0
        if self.per_env_substeps:
            def max_velocity_env():
                with torch.no_grad():
                    return torch.maximum((minv * u).abs().amax(dim=(1, 2)), (b_minv * bv).abs().amax(dim=(1, 2)))
            for dtv, act in self._substep_rounds(max_velocity_env):
                u, p = piso_substep_3d(s, u, p, bv, dtv, self._forcing_torch(u), active=act)
                nsub += 1
            return u, p, nsub

        def max_velocity():
            with torch.no_grad():
                return float(torch.maximum((minv * u).abs().max(), (b_minv * bv).abs().max()))
        for ts in cfl_substeps(self.dt, self.cfl, max_velocity):
            u, p = piso_substep_3d(s, u, p, bv, ts, self._forcing_torch(u))
            nsub += 1
        return u, p, nsub

    def mark_state_differentiable(self):
        """envs/util/diff_tools.py:8-22: returns the velocity leaf of the incoming state [B, 3, N]"""
        self._du = self.solver.u.detach().clone().requires_grad_(True)
        return self._du

    def detach(self):
        self._du = None

    def _advance_differentiable(self, action):
        s = self.solver
        u = self._du if getattr(self, "_du", None) is not None else s.u.detach().clone()
        p = s.p.detach().clone()
        bv = s.bvel.detach().clone()
        if self.enable_actions:
            a = action.reshape(self.n_envs, -1)
            half = self.nax * self.naz
            lo = torch.zeros(self.n_envs, 3, self.x * self.z, device=self.device)
            lo = torch.stack([lo[:, 0], self._action_to_control(a[:, :half].reshape(self.n_envs, self.nax, self.naz)), lo[:, 2]], dim=1)
            bv = torch.cat([bv[:, :, :self._face_lo.start], lo, bv[:, :, self._face_lo.stop:]], dim=2)
            if self.both_walls:
                hi = torch.zeros(self.n_envs, 3, self.x * self.z, device=self.device)
                hi = torch.stack([hi[:, 0], -1 * self._action_to_control(a[:, half:].reshape(self.n_envs, self.nax, self.naz)), hi[:, 2]], dim=1)
                bv = torch.cat([bv[:, :, :self._face_hi.start], hi, bv[:, :, self._face_hi.stop:]], dim=2)
        tb, tt, nsub = [], [], 0
        self._begin_substep_count()
        for _ in range(self.n_sim_steps):
            u, p, n = self._single_step_differentiable(u, p, bv)
            nsub += n
            lo_, hi_ = self._wall_stress_torch(u)
            tb.append(lo_); tt.append(hi_)
        self.last_substeps = nsub
        with torch.no_grad():                      # the solver buffers mirror the state (observations read them)
            s.u.copy_(u); s.p.copy_(p); s.bvel.copy_(bv)
        self._du = u
        tau_bottom, tau_top = torch.stack(tb).mean(dim=0), torch.stack(tt).mean(dim=0)
        return tau_bottom, tau_top

    def _advance(self, action):
        """-> (tau_bottom, tau_top) [B]: the wall shear stresses averaged over the solver steps"""
        if self.enable_actions:
            self._apply_action(action)
        s = self.solver
        self._acc.zero_()
        nsub = 0
        for _ in range(self.n_sim_steps):
            nsub += s.single_step(self.dt, self.cfl, self.rows, self.d_lo, self.d_hi)
            s.wall_rows(self.rows, self.d_lo, self.d_hi, set_forcing=False, acc=self._acc)
        self.last_substeps = nsub
        tau = self._acc / self.n_sim_steps
        return tau[:, 0], tau[:, 1]

    def step(self, action):
        action = self._begin_step(action)
        tau_bottom, tau_top = self._advance_differentiable(action) if self.differentiable else self._advance(action)
        tau_total = 0.5 * (tau_bottom + tau_top)
        reward = 1 - (tau_total if self.both_walls else tau_bottom) / self.tau_ref
        info = {"wall_stress": tau_total, "wall_stress_bottom": tau_bottom, "wall_stress_top": tau_top}
        truncated = self._end_step()
        obs = self._get_obs()
        if self.use_marl:
            info["global_reward"] = reward
            reward = reward[:, None] * torch.ones(self.n_envs, self.n_agents, device=self.device)
        return obs, reward, False, truncated, info


class TCF3DBottomEnv(TCF3DEnv):
    both_walls = False
    reference_values = {"tau_ref": ("wall_stress_bottom", "mean")}           # tcf_env.py:556-562


class TCF3DBothEnv(TCF3DEnv):
    both_walls = True
    reference_values = {"tau_ref": ("wall_stress", "mean")}                  # tcf_env.py:1131-1137
