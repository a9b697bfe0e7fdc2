"""Batched ``RBC2D`` (Rayleigh-Benard convection with bottom-plate heaters) environment.

Mirrors ``envs/rbc/rbc_env_base.py`` / ``rbc_env_2d.py`` of the reference: temperature as passive scalar,
buoyancy source after the scalar advection of every substep, heater actuation on the bottom plate
(zero-mean, clamped, cubic-blended profile, ``rbc_env_2d.py:210-282``), Nusselt-number reward
(``rbc_env_base.py:491-539``), 48 x 8 sensor grid on the rendered field, and the multi-agent interface
(``use_marl``: one agent per heater, circular moving observation windows ``obs_extraction.py:206-252`` and
local Nusselt rewards ``rbc_env_2d.py:328-357``).  All tensors carry a leading environment dimension.
"""
from __future__ import annotations

import numpy as np
import torch

from .. import native
from ..sensors import sensor_tables
from ..solver import BatchedPISO, _ptr, cfl_substeps
from .common import EpisodeLifecycle, InitialDomains, Renderable
from .rbc_domain import make_rbc_domain

RBC_2D_DEFAULT_CONFIG = {
    "rayleigh_number": 8e4, "prandtl_number": 0.7, "n_heaters": 12, "resolution": 8, "dt": 0.05, "adaptive_cfl": 0.8,
    "step_length": 1.0, "episode_length": 200, "local_obs_window": 11, "local_reward_weight": 0.2, "uniform_grid": False,
    "aspect_ratio": 1.0, "use_marl": False,
}


def extract_moving_window_2d(field: torch.Tensor, n_agents: int, agent_width: int, n_agents_per_window: int) -> torch.Tensor:
    """[..., Y, X] -> [..., n_agents, Y, window*agent_width] circular windows centred on each agent
    (obs_extraction.py:206-252, batched)."""
    *lead, Y, X = field.shape
    assert X == n_agents * agent_width
    fa = field.reshape(*lead, Y, n_agents, agent_width)
    pad = n_agents_per_window // 2
    idx = (torch.arange(n_agents, device=field.device)[:, None] + torch.arange(n_agents_per_window, device=field.device)[None, :] - pad) % n_agents
    win = fa[..., idx, :]                       # [..., Y, n_agents, window, agent_width]
    win = win.movedim(-3, -4)                   # [..., n_agents, Y, window, agent_width]
    return win.reshape(*lead, n_agents, Y, n_agents_per_window * agent_width)


class RBC2DEnv(EpisodeLifecycle, InitialDomains, Renderable):
    T_cold, T_hot, heater_limit = 0.0, 1.0, 0.75
    n_sensors_y, n_sensors_per_heater = 8, 4
    buoyancy_factor = 1.0
    metrics = ["nusselt"]
    reference_values = {"nu_ref": ("nusselt", "p50")}
    render_fields = ("temperature", "velocity_magnitude", "vorticity", "pressure")

    def __init__(self, n_envs: int = 1, rayleigh_number=8e4, prandtl_number=0.7, n_heaters=12, resolution=8, dt=0.05,
                 adaptive_cfl=0.8, step_length=1.0, episode_length=200, local_obs_window=11, local_reward_weight=0.2,
                 uniform_grid=False, aspect_ratio=1.0, use_marl=False, device="cuda:0", cg_impl=6, nu_ref=0.0,
                 randomize_initial_state=False, enable_actions=True, load_initial_domain=False, initial_domains_path=None,
                 differentiable=False, per_env_substeps: bool = False):
        self.per_env_substeps = bool(per_env_substeps)
        self.n_envs = int(n_envs)
        self.Ra, self.Pr = float(rayleigh_number), float(prandtl_number)
        self.n_heaters, self.heater_width = int(n_heaters), int(resolution)
        self.dt, self.cfl = float(dt), float(adaptive_cfl)
        self.step_length, self.episode_length = float(step_length), int(episode_length)
        self.local_obs_window, self.local_reward_weight = int(local_obs_window), local_reward_weight
        self.use_marl, self.nu_ref = bool(use_marl), float(nu_ref)
        self.enable_actions = enable_actions
        self.differentiable = bool(differentiable)
        self.randomize_initial_state = randomize_initial_state
        self.load_domain_on_reset, self.initial_domains_path = bool(load_initial_domain), initial_domains_path
        self.prandtl_number, self.rayleigh_number = prandtl_number, rayleigh_number
        self.device = torch.device(device)
        self.aspect = aspect_ratio * torch.pi
        spec, info = make_rbc_domain(rayleigh_number, prandtl_number, n_heaters, resolution, aspect_ratio, uniform_grid)
        self.spec, self.info = spec, info
        self.cd = spec.prepare()
        self.nx, self.ny = info["nx"], info["ny"]
        self.solver = BatchedPISO(self.cd, self.n_envs, device=device, corrector_steps=2, advect_non_ortho_steps=1,
                                  pressure_non_ortho_steps=1, non_orthogonal=False, pressure_tol=1e-5, cg_impl=cg_impl)
        self.solver.set_buoyancy(self.buoyancy_factor)
        self.lib = self.solver.lib
        self._bottom = slice(int(self.cd.boff[0, 2]), int(self.cd.boff[0, 2]) + self.nx)
        self._setup_sensors()
        self._zero_action = torch.zeros(self.n_envs, self.n_heaters, 1, device=self.device)

    # ---- static tables ---------------------------------------------------------------------------
    @property
    def render_shape(self):
        nx = self.n_heaters * 20
        return (nx, round(nx / self.aspect))

    @property
    def n_sensors_x(self):
        return self.n_heaters * self.n_sensors_per_heater

    def _build_render_map(self, plane):
        from ..render import render_map_2d
        return render_map_2d([b.vertex for b in self.spec.blocks], self.render_shape, fill_max_steps=16)

    def _setup_sensors(self):
        nx, ny = self.render_shape
        sx = torch.linspace(0, nx, self.n_sensors_x + 1)[:-1] + nx / (2 * self.n_sensors_x)
        sy = torch.linspace(0, ny, self.n_sensors_y + 1)[:-1] + ny / (2 * self.n_sensors_y)
        gx, gy = torch.meshgrid(sx, sy, indexing="ij")
        loc = torch.stack([gx, gy], dim=-1).reshape(-1, 2).T
        self.sensor_px = loc.round().to(torch.int).numpy()       # [2, n_sx * n_sy], x-major (rbc_env_base.py:445-470)
        idx, w = sensor_tables([b.vertex for b in self.spec.blocks], (nx, ny), self.sensor_px, fill_max_steps=16)
        self.sens_idx = torch.from_numpy(idx).to(self.device)
        self.sens_w = torch.from_numpy(w).to(self.device)

    # ---- reference-shaped API ---------------------------------------------------------------------
    @property
    def n_agents(self):
        return self.n_heaters if self.use_marl else 1

    @property
    def initial_domain_id(self):
        """rbc_env_base.py:606-611"""
        return f"rbc_2d_Ra{self.rayleigh_number}_Pr{self.prandtl_number}_NH{self.n_heaters}_HW{self.heater_width}"

    @property
    def observation_space(self):
        """Per-environment (per-agent in MARL mode) space, rbc_env_2d.py:131-166."""
        from .. import spaces
        width = self.n_sensors_per_heater * (self.local_obs_window if self.use_marl else self.n_heaters)
        shape = (self.n_sensors_y, width)
        inf = float("inf")
        return spaces.Dict({"temperature": spaces.Box(self.T_cold, self.T_hot + self.heater_limit, shape=shape),
                            "velocity": spaces.Box(-inf, inf, shape=(2,) + shape), "pressure": spaces.Box(-inf, inf, shape=shape)})

    @property
    def action_space(self):
        from .. import spaces
        return spaces.Box(-1.0, 1.0, shape=(1,) if self.use_marl else (self.n_heaters, 1))

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
        self._dstate = None

    def reset(self, seed: int | None = None, randomize: bool | None = None):
        """rbc_env_base.py:190-278: linear temperature profile + 0.1 N(0,1) clamped to [T_cold, T_hot],
        velocity 0.05 N(0,1) (per environment streams of one generator)."""
        self._begin_reset(seed)
        s = self.solver
        B, nx, ny = self.n_envs, self.nx, self.ny
        self._dstate = None
        randomize = self.randomize_initial_state if randomize is None else randomize
        if self.load_domain_on_reset:                      # fluid_env.py:519-539
            self._load_initial_domains_on_reset(randomize)
            s.buffer("ures").copy_(s.u)
            if randomize:
                self._randomize_domain()
            self._apply_action(self._zero_action)
            self._reset_called, self._n_steps = True, 0
            return (self._get_local_obs() if self.use_marl else self._get_global_obs()), {}
        grad = torch.linspace(self.T_hot, self.T_cold, steps=ny, device=self.device)[:, None].expand(ny, nx)
        T0 = grad[None] + torch.randn(B, ny, nx, device=self.device, generator=self._torch_rng) * 0.1 * (self.T_hot - self.T_cold)
        s.T.copy_(torch.clamp(T0, self.T_cold, self.T_hot).reshape(B, -1))
        s.u.copy_(torch.randn(B, 2, ny * nx, device=self.device, generator=self._torch_rng) * 0.05)
        s.p.zero_()
        s.buffer("ures").zero_()
        s.sbval.copy_(torch.from_numpy(self.cd.sb_val0[:self.cd.NB].copy()).to(self.device).unsqueeze(0).expand_as(s.sbval))
        if randomize:                                      # fluid_env.py:549-551: also for a freshly built domain
            self._randomize_domain()
        self._apply_action(self._zero_action)
        self._reset_called, self._n_steps = True, 0
        return (self._get_local_obs() if self.use_marl else self._get_global_obs()), {}

    def _randomize_domain(self):
        """rbc_env_base.py:336-393: mirror in x with probability 1/2 (the x velocity changes sign), periodic shift in x,
        N(0, 0.05) noise on T (clamped) and u, then 1-2 time units of settling.  Flip and shift are drawn per environment;
        the settling time is common to the batch (one launch sequence advances every environment)."""
        s = self.solver
        B, nx, ny = self.n_envs, self.nx, self.ny
        flip = torch.from_numpy(self._np_rng.uniform(0.0, 1.0, size=B) > 0.5).to(self.device)
        shift = torch.from_numpy(self._np_rng.integers(0, nx, size=B)).to(self.device)
        T = s.T.reshape(B, ny, nx)
        u = s.u.reshape(B, 2, ny, nx)
        x = torch.arange(nx, device=self.device)
        # flipped then rolled: out[x] = in_flipped[(x - shift) % nx], in_flipped[x'] = in[nx - 1 - x']
        src = (x[None, :] - shift[:, None]) % nx
        src = torch.where(flip[:, None], nx - 1 - src, src)                      # [B, nx]
        T = torch.gather(T, 2, src[:, None, :].expand(B, ny, nx))
        u = torch.gather(u, 3, src[:, None, None, :].expand(B, 2, ny, nx)).clone()
        u[:, 0] = torch.where(flip[:, None, None], -u[:, 0], u[:, 0])
        T = T + torch.randn(T.shape, device=self.device, generator=self._torch_rng) * 0.05
        T = torch.clamp(T, self.T_cold, self.T_hot)
        u = u + torch.randn(u.shape, device=self.device, generator=self._torch_rng) * 0.05
        s.T.copy_(T.reshape(B, -1))
        s.u.copy_(u.reshape(B, 2, -1))
        n_steps = int(self._np_rng.uniform(1.0, 2.0) / self.dt)
        for _ in range(n_steps):
            s.single_step(self.dt, self.cfl)

    def _action_to_control(self, action: torch.Tensor) -> torch.Tensor:
        """[B, n_heaters] -> bottom-plate temperature [B, nx] (rbc_env_2d.py:210-270)."""
        hw = self.heater_width
        T_shifted = action - action.mean(dim=1, keepdim=True)
        T_action = T_shifted / (torch.clamp(T_shifted.abs(), min=1.0) / self.heater_limit) + self.T_hot
        bw = round(hw * 0.1)
        T_left, T_right = torch.roll(T_action, 1, dims=1), torch.roll(T_action, -1, dims=1)
        x_idx = torch.arange(self.nx, device=action.device)
        seg, xpos = x_idx // hw, x_idx % hw
        T0, T1, T2 = T_left[:, seg], T_action[:, seg], T_right[:, seg]
        left_zone, right_zone = xpos < bw, xpos >= hw - bw
        tL = (xpos.to(torch.float32) / bw + 0.5).clamp(0.0, 1.0) if bw > 0 else torch.ones_like(xpos, dtype=torch.float32)
        tR = 1 - torch.roll(tL, shifts=hw - bw + 1, dims=0)

        def blend(t, A, Bv):
            sm = t * t * (3 - 2 * t)
            return (1 - sm) * A + sm * Bv

        return torch.where(left_zone, blend(tL, T0, T1), torch.where(right_zone, blend(tR, T1, T2), T1))

    def _apply_action(self, action):
        a = torch.as_tensor(action, dtype=torch.float32, device=self.device).reshape(self.n_envs, self.n_heaters)
        self.solver.sbval[:, self._bottom] = self._action_to_control(a)

    def _sample(self, field, channels):
        s = self.solver
        ns, K = self.sens_idx.shape[1], self.sens_idx.shape[0]
        out = torch.empty(self.n_envs, channels, ns, device=self.device)
        native.check(self.lib.fgb_sample_sensors(s.handle, _ptr(field), channels, _ptr(self.sens_idx), _ptr(self.sens_w), K, ns,
                                                 _ptr(out), s.stream), "fgb_sample_sensors")
        # sensors are enumerated x-major; the reference reshapes to [n_sx, n_sy] and transposes to [n_sy, n_sx]
        return out.reshape(self.n_envs, channels, self.n_sensors_x, self.n_sensors_y).transpose(-1, -2).contiguous()

    def _get_global_obs(self):
        s = self.solver
        return {"temperature": self._sample(s.T, 1)[:, 0], "velocity": self._sample(s.u, 2), "pressure": self._sample(s.p, 1)[:, 0]}

    def _get_local_obs(self):
        g = self._get_global_obs()
        w = dict(n_agents=self.n_heaters, agent_width=self.n_sensors_per_heater, n_agents_per_window=self.local_obs_window)
        T = extract_moving_window_2d(g["temperature"], **w)
        ux = extract_moving_window_2d(g["velocity"][:, 0], **w)
        uy = extract_moving_window_2d(g["velocity"][:, 1], **w)
        p = extract_moving_window_2d(g["pressure"], **w)
        return {"temperature": T, "velocity": torch.stack([ux, uy], dim=2), "pressure": p}

    def _column_sums(self):
        s = self.solver
        return s.column_sums(s.u[:, 1].contiguous(), s.T, self.nx, self.ny)     # [B, 2, nx]: sum_y u_y T dV, sum_y dV

    def compute_global_nusselt(self, cs=None):
        cs = self._column_sums() if cs is None else cs
        return 1.0 + (self.Ra * self.Pr) ** 0.5 * cs[:, 0].sum(dim=1) / cs[:, 1].sum(dim=1)

    def _get_local_rewards(self, cs=None):
        """rbc_env_2d.py:328-357: Nusselt number over each agent's moving window.  NB the reference divides by
        the cell volume of the FIRST window*heater_width columns for every agent -- reproduced."""
        cs = self._column_sums() if cs is None else cs
        w = dict(n_agents=self.n_heaters, agent_width=self.heater_width, n_agents_per_window=self.local_obs_window)
        num = extract_moving_window_2d(cs[:, 0:1], **w).sum(dim=(-1, -2))            # [B, n_agents]
        vol = cs[:, 1, : self.local_obs_window * self.heater_width].sum(dim=1, keepdim=True)
        return self.nu_ref - (1.0 + (self.Ra * self.Pr) ** 0.5 * num / vol)

    # ---- differentiable mode (fluid_env.py:154,232; examples/interfaces/gradient_based_methods.py) -----------------
    # One autograd node per substep (scalar transport + buoyancy + PISO, fluidgym_b200.autograd.PISOSubstepScalar backed by
    # the CUDA adjoint); the heater profile (rbc_env_2d.py:210-282) and the Nusselt sums (rbc_env_base.py:491-539) around it
    # are torch expressions, as in the reference.  The CFL plan is taken from detached maxima with one common substep size
    # for the batch (the most restrictive environment decides): solver.cfl_substeps; with per_env_substeps every environment
    # follows its own plan (EpisodeLifecycle._substep_rounds).
    def _advance_differentiable(self, action):
        from ..autograd import piso_substep_scalar
        s = self.solver
        if self._dstate is None:
            self._dstate = (s.u.clone(), s.p.clone(), s.T.clone(), s.sbval.clone())
        u, p, T, sb = self._dstate
        if self.enable_actions:
            ctrl = self._action_to_control(action.reshape(self.n_envs, self.n_heaters))
            sb = sb.index_copy(1, torch.arange(self._bottom.start, self._bottom.stop, device=self.device), ctrl)
        bv = s.bvel
        mvb = torch.empty(self.n_envs, device=self.device)

        def max_velocity_env():
            native.check(self.lib.fgb_max_velocity(s.handle, _ptr(u.detach().contiguous()), _ptr(bv), _ptr(mvb), s.stream), "fgb_max_velocity")
            return mvb
        nsub = 0
        self._begin_substep_count()
        for _ in range(self.n_sim_steps):
            if self.per_env_substeps:
                for dtv, act in self._substep_rounds(max_velocity_env):
                    u, p, T = piso_substep_scalar(s, u, p, bv, T, sb, dtv, self.buoyancy_factor, active=act)
                    nsub += 1
                continue
            for ts in cfl_substeps(self.dt, self.cfl, lambda: float(max_velocity_env().max())):                 # SIM.py:2004-2031
                u, p, T = piso_substep_scalar(s, u, p, bv, T, sb, ts, self.buoyancy_factor)
                nsub += 1
        self._dstate = (u, p, T, sb)
        with torch.no_grad():                      # keep the solver's own state in step for observations / get_state
            s.u.copy_(u); s.p.copy_(p); s.T.copy_(T); s.sbval.copy_(sb)
        self.last_substeps = nsub
        det = self._det_columns()
        uyT = (u[:, 1] * T).reshape(self.n_envs, self.ny, self.nx) * det
        return torch.stack([uyT.sum(dim=1), det.sum(dim=0)[None].expand(self.n_envs, self.nx)], dim=1)   # as k_column_sums

    def _det_columns(self):
        if getattr(self, "_det_t", None) is None:
            self._det_t = torch.from_numpy(np.ascontiguousarray(self.cd.det, dtype=np.float32)).to(self.device).reshape(self.ny, self.nx)
        return self._det_t

    def step(self, action):
        action = self._begin_step(action)
        if self.differentiable:
            cs = self._advance_differentiable(action)
        else:
            if self.enable_actions:
                self._apply_action(action)
            nsub = 0
            for _ in range(self.n_sim_steps):
                nsub += self.solver.single_step(self.dt, self.cfl)
            self.last_substeps = nsub
            cs = self._column_sums()
        nu = self.compute_global_nusselt(cs)
        reward = self.nu_ref - nu
        info = {"nusselt": nu.detach()}
        truncated = self._end_step()
        if not self.use_marl:
            return self._get_global_obs(), reward, False, truncated, info
        lw = self.local_reward_weight
        local = self._get_local_rewards(cs) if lw > 0 else torch.zeros(self.n_envs, self.n_heaters, device=self.device)
        info["global_reward"] = reward
        return self._get_local_obs(), lw * local + (1 - lw) * reward[:, None], False, truncated, info
