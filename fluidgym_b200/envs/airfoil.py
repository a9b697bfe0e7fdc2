"""Batched ``Airfoil2D`` environment (NACA 0012 at an angle of attack, three synthetic jets on the suction side).

Public surface mirrors ``AirfoilEnv2D`` / ``AirfoilEnvBase`` (``envs/airfoil/airfoil_env_2d.py``,
``airfoil_env_base.py``): reward = lift/drag - reference, action = 3 jet amplitudes (zero-mean, smoothed),
observation = velocity / pressure at the sensor pixels outside the body.  As for the other environments every
tensor carries a leading environment dimension.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from .. import native
from ..sensors import sensor_tables
from ..solver import BatchedPISO, _ptr
from .airfoil_domain import BOT, FRONT, JET_CENTERS, JET_WIDTH, TAIL_LOWER, TAIL_UPPER, TOP, airfoil_polyline, make_airfoil_domain
from .common import DifferentiableRollout, EpisodeLifecycle, InitialDomains, Renderable, build_wall_tables
from .cylinder_domain import jet_profile

AIRFOIL_2D_DEFAULT_CONFIG = {
    "reynolds_number": 3e3, "dt": 0.05, "step_length": 0.25, "adaptive_cfl": 0.8, "episode_length": 300,
    "attack_angle_deg": 10.0,
}


def polygon_mask(polygon_xy: np.ndarray, nx: int, ny: int) -> np.ndarray:
    """Pixels of an ``[ny, nx]`` raster whose integer coordinates lie inside the polygon (even-odd rule);
    stands for ``matplotlib.path.Path.contains_points`` in airfoil_env_base.py:174-208."""
    xs, ys = np.meshgrid(np.linspace(0, nx - 1, nx), np.linspace(0, ny - 1, ny))
    x, y = xs.ravel(), ys.ravel()
    v = np.asarray(polygon_xy, dtype=np.float64)
    inside = np.zeros(x.shape, dtype=bool)
    for i in range(len(v)):
        (x0, y0), (x1, y1) = v[i], v[(i + 1) % len(v)]
        if y0 == y1:
            continue
        crosses = (y0 > y) != (y1 > y)
        inside ^= crosses & (x < x0 + (y - y0) * (x1 - x0) / (y1 - y0))
    return inside.reshape(ny, nx)


class Airfoil2DEnv(EpisodeLifecycle, DifferentiableRollout, InitialDomains, Renderable):
    H, L, U_mean, airfoil_length = 1.4, 4.5, 0.3, 1.0
    n_jets = 3
    action_smoothing_alpha = 0.1
    render_shape = (600, 150)
    render_fields = ("vorticity", "velocity_magnitude", "velocity_x", "velocity_y", "pressure")
    metrics = ["drag", "lift"]
    reference_values = {"cl_cd_ref": ("lift", "mean", "drag", "mean")}
    use_marl = False

    def __init__(self, n_envs: int = 1, reynolds_number=3e3, dt=0.05, step_length=0.25, adaptive_cfl=0.8, episode_length=300,
                 attack_angle_deg=10.0, device="cuda:0", cg_impl=6, compiled=None, cl_cd_ref=0.0, randomize_initial_state=False,
                 enable_actions=True, use_marl=False, differentiable=False, load_initial_domain=False, initial_domains_path=None,
                 per_env_substeps: bool = False):
        self.per_env_substeps = bool(per_env_substeps)
        if attack_angle_deg < 0.0 or attack_angle_deg > 20.0:
            raise ValueError("Attack angle must be between 0 and 20 degrees.")
        if use_marl:
            raise ValueError("Airfoil2D has a single agent controlling all three jets")
        self.n_envs = int(n_envs)
        self.reynolds_number, self.attack_angle_deg = float(reynolds_number), float(attack_angle_deg)
        self.dt, self.cfl = float(dt), float(adaptive_cfl)
        self.step_length, self.episode_length = float(step_length), int(episode_length)
        self.cl_cd_ref = float(cl_cd_ref)
        self.randomize_initial_state, self.enable_actions = randomize_initial_state, enable_actions
        self.differentiable = bool(differentiable)
        self.load_domain_on_reset, self.initial_domains_path = bool(load_initial_domain), initial_domains_path
        self.device = torch.device(device)
        if compiled is None:
            spec = make_airfoil_domain(reynolds_number, self.U_mean, self.airfoil_length, self.H, self.L, attack_angle_deg)
            cd = spec.prepare()
        else:
            spec, cd = compiled
        self.spec, self.cd = spec, cd
        out_mask = np.zeros(cd.NB, dtype=np.int8)
        for blk in (TAIL_UPPER, TAIL_LOWER):
            o = cd.boff[blk, 1]
            out_mask[o:o + spec.blocks[blk].ny] = 1
        # airfoil_env_base.py:260-289
        self.solver = BatchedPISO(cd, self.n_envs, device=device, corrector_steps=2, advect_non_ortho_steps=2,
                                  pressure_non_ortho_steps=4, non_orthogonal=True, advection_tol=1e-6, pressure_tol=1e-7,
                                  cg_impl=cg_impl, out_mask=out_mask)
        self.lib = self.solver.lib
        self.char_vel = (self.U_mean, 0.0)
        ring = [(FRONT, 1, False), (TOP, 2, False), (BOT, 3, True)]
        self._wall_t, self.wall = build_wall_tables(cd, spec, ring, self.device, 1.0 / (0.5 * self.U_mean ** 2 * self.airfoil_length))
        self._setup_jets(out_mask)
        self._setup_sensors()
        B, dev = self.n_envs, self.device
        self.last_control = torch.zeros(B, self.n_jets, device=dev)
        self._acc = torch.zeros(B, 2, device=dev)
        self._zero_action = torch.zeros(B, self.n_jets, device=dev)

    # ---- static tables ---------------------------------------------------------------------------
    def _setup_jets(self, out_mask):
        """Jet slots on the suction side (grid.py:18-46) and their unit-mass-flux profiles along the local wall
        normal (airfoil_env_base.py:484-538).  NB the reference offsets the normal lookup by the VERTEX count of
        the front block's wall (22) although the concatenated normals hold one entry per CELL (21): each jet uses
        the normals of the cells one to the right of its own -- reproduced."""
        cd, spec = self.cd, self.spec
        x_surface = torch.from_numpy(spec.blocks[TOP].vertex[0, 0, :])
        self.jet_slots = []
        for c in JET_CENTERS:
            lo, hi = c - JET_WIDTH / 2, c + JET_WIDTH / 2
            self.jet_slots.append((int(torch.argmin(torch.abs(x_surface - lo))), int(torch.argmin(torch.abs(x_surface - hi)))))
        n_top = spec.blocks[TOP].nx
        normals = self._wall_t["normal"].cpu()
        offset = spec.blocks[FRONT].vertex.shape[1]
        base = torch.zeros(self.n_jets, 2, n_top)
        for i, (a, b) in enumerate(self.jet_slots):
            prof = torch.from_numpy(jet_profile(b - a + 3))[1:-1].clone()
            prof /= prof.sum()
            base[i, :, a:b + 1] = prof.unsqueeze(0) * normals[:, offset + a: offset + b + 1]
        self.jet_base = base.to(self.device)                                       # [n_jets, 2, n_top]
        o = int(cd.boff[TOP, 2])
        self.jet_faces = torch.arange(o, o + n_top, device=self.device)
        free = out_mask.copy()
        free[o:o + n_top] = 1                                                       # outflow + airfoil top wall
        self.free_mask = torch.from_numpy(free).to(self.device)

    def _to_pixels(self, xy: torch.Tensor) -> torch.Tensor:
        """airfoil_env_base.py:570-585"""
        xy = xy.clone()
        xy[0] = (xy[0] + 1.5) * (self.render_shape[0] / (self.L + 1.5))
        xy[1] = (xy[1] + self.H / 2) * (self.render_shape[1] / self.H)
        return torch.round(xy).to(torch.int32)

    def _build_render_map(self, plane):
        from ..render import render_map_2d
        return render_map_2d([b.vertex for b in self.spec.blocks], self.render_shape, fill_max_steps=128)

    def sensor_locations_physical(self) -> torch.Tensor:
        """airfoil_env_base.py:607-656: coarse wake grid, fine near wake, box around the airfoil."""
        def grid(xs, ys):
            gx, gy = torch.meshgrid(xs, ys, indexing="ij")
            return torch.stack([gx.ravel(), gy.ravel()], dim=0)
        ys = torch.linspace(-self.H / 2, self.H / 2, 10)[1:-1]
        coarse = grid(torch.arange(1.5, 2.6, step=0.125), ys)
        fine = grid(torch.arange(1.05, 1.5 - 0.05, step=0.05), ys)
        near = grid(torch.linspace(-0.125, self.airfoil_length, 10), torch.linspace(-0.5, 0.125, 8))
        return torch.cat([coarse, fine, near], dim=1)

    def _setup_sensors(self):
        nx, ny = self.render_shape
        body = self._to_pixels(airfoil_polyline(self.attack_angle_deg)).numpy()
        self.airfoil_mask = polygon_mask(body.T, nx, ny)
        px = self._to_pixels(self.sensor_locations_physical()).numpy()
        keep = [i for i in range(px.shape[1]) if not self.airfoil_mask[px[1, i], px[0, i]]]
        self.sensor_px = px[:, keep]
        idx, w = sensor_tables([b.vertex for b in self.spec.blocks], self.render_shape, self.sensor_px, fill_max_steps=128)
        self.sens_idx = torch.from_numpy(idx).to(self.device)
        self.sens_w = torch.from_numpy(w).to(self.device)

    # ---- reference-shaped API ---------------------------------------------------------------------
    @property
    def n_agents(self):
        return self.n_jets

    @property
    def initial_domain_id(self):
        """airfoil_env_base.py:829-831"""
        return f"airfoil_2D_Re{int(self.reynolds_number)}"

    @property
    def observation_space(self):
        from .. import spaces
        inf, ns = float("inf"), int(self.sens_idx.shape[1])
        return spaces.Dict({"velocity": spaces.Box(-inf, inf, shape=(ns, 2)), "pressure": spaces.Box(-inf, inf, shape=(ns,))})

    @property
    def action_space(self):
        from .. import spaces
        return spaces.Box(-1.0, 1.0, shape=(self.n_jets,))

    def set_state(self, u, p, bvel, last_control=None):
        s = self.solver
        for dst, src in ((s.u, u), (s.p, p), (s.bvel, bvel)):
            self._copy_state(dst, src)
        if last_control is not None:
            self.last_control.copy_(torch.as_tensor(last_control, device=self.device).expand_as(self.last_control))
        self._dstate = None
        self._reset_called = True

    def get_state(self):
        s = self.solver
        return dict(u=s.u.clone(), p=s.p.clone(), bvel=s.bvel.clone(), last_control=self.last_control.clone())

    def reset(self, seed: int | None = None, randomize: bool | None = None):
        self._begin_reset(seed)
        s = self.solver
        if self.load_domain_on_reset:
            self._load_initial_domains_on_reset(self.randomize_initial_state if randomize is None else randomize)
        else:
            s.u.zero_()
            s.p.zero_()
            s.bvel.copy_(torch.from_numpy(self.cd.bvel0[:, :self.cd.NB].copy()).to(self.device).unsqueeze(0).expand_as(s.bvel))
        s.update_outflow(1.0, self.char_vel, tol=1e-5)       # the "PRE" hook of make_divergence_free (SIM.py:1335-1347)
        s.make_divergence_free(max_iter=1000)
        self.last_control.zero_()
        randomize = self.randomize_initial_state if randomize is None else randomize
        if randomize:
            self._randomize_domain()
        self._apply_control(self.last_control)
        self._dstate = None
        self._reset_called, self._n_steps = True, 0
        return self._get_obs(), {}

    def _randomize_domain(self):
        """airfoil_env_base.py:302-339"""
        max_n = int(0.05 * self.episode_length)
        n_steps = int(self._np_rng.integers(int(0.5 * max_n), max_n)) + 1
        s = self.solver
        s.u += torch.randn(s.u.shape, device=self.device, generator=self._torch_rng) * 0.01
        s.p += torch.randn(s.p.shape, device=self.device, generator=self._torch_rng) * 0.01
        for _ in range(n_steps):
            s.single_step(self.dt, self.cfl, char_vel=self.char_vel, bc_tol=1e-5)

    def _control_to_profile(self, control: torch.Tensor) -> torch.Tensor:
        """airfoil_env_2d.py:165-191: zero-mean, max-abs <= 1 amplitudes times the base profiles -> [B, 2, n_top]."""
        v = control - control.mean(dim=1, keepdim=True)
        mx = v.abs().max(dim=1, keepdim=True).values
        v = torch.where(mx > 1.0, v / mx, v)
        return torch.einsum("bj,jcx->bcx", v, self.jet_base)

    def _apply_control(self, control):
        """airfoil_env_base.py:709-718: set the jet wall velocity, then rescale outflow + jet wall to zero net flux."""
        s = self.solver
        s.bvel[:, :, self.jet_faces] = self._control_to_profile(control)
        native.check(self.lib.fgb_balance_fluxes(s.handle, _ptr(s.bvel), _ptr(self.free_mask), 1e-5, s.stream), "fgb_balance_fluxes")

    def _get_obs(self):
        s = self.solver
        B, ns, K = self.n_envs, self.sens_idx.shape[1], self.sens_idx.shape[0]
        vel = torch.empty(B, 2, ns, device=self.device)
        prs = torch.empty(B, 1, ns, device=self.device)
        for field, ch, out in ((s.u, 2, vel), (s.p, 1, prs)):
            native.check(self.lib.fgb_sample_sensors(s.handle, _ptr(field), ch, _ptr(self.sens_idx), _ptr(self.sens_w), K, ns, _ptr(out),
                                                     s.stream), "fgb_sample_sensors")
        return {"velocity": vel.permute(0, 2, 1).contiguous(), "pressure": prs[:, 0]}

    def _advance(self, action):
        s = self.solver
        self._acc.zero_()
        nsub = 0
        for _ in range(self.n_sim_steps):
            # smoothing as proposed by Rabault et al. (airfoil_env_base.py:727-733)
            self.last_control = self.last_control + self.action_smoothing_alpha * (action - self.last_control)
            if self.enable_actions:
                self._apply_control(self.last_control)
            nsub += s.single_step(self.dt, self.cfl, char_vel=self.char_vel, bc_tol=1e-5)
            native.check(self.lib.fgb_wall_forces(s.handle, C.byref(self.wall), _ptr(s.u), _ptr(s.p), _ptr(s.bvel), _ptr(self._acc),
                                                  s.stream), "fgb_wall_forces")
        self.last_substeps = nsub
        return self._acc

    def _reward(self, cd, cl):
        return cl / cd - self.cl_cd_ref

    def _advance_differentiable(self, action):
        s = self.solver
        if self._dstate is None:
            self._dstate = (s.u.clone(), s.p.clone(), s.bvel.clone(), self.last_control.clone())
        u, p, bv, last = self._dstate
        acc = torch.zeros(self.n_envs, 2, device=self.device)
        nsub = 0
        free = self.free_mask.bool()
        self._begin_substep_count()
        for _ in range(self.n_sim_steps):
            last = last + self.action_smoothing_alpha * (action - last)
            if self.enable_actions:
                bv = bv.index_copy(2, self.jet_faces, self._control_to_profile(last))
                bv = self._balance_torch(bv, free, 1e-5)
            u, p, bv, k = self._single_step_differentiable(u, p, bv)
            nsub += k
            acc = acc + self._forces_torch(u, p, bv)
        self._dstate = (u, p, bv, last)
        with torch.no_grad():
            s.u.copy_(u); s.p.copy_(p); s.bvel.copy_(bv)
            self.last_control = last.detach().clone()
        self.last_substeps = nsub
        return acc
