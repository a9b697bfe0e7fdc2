"""Batched ``CylinderJet2D`` environment: B independent environments advanced by one launch sequence.

Public surface mirrors the reference's ``FluidEnv`` / ``CylinderJetEnv2D``
(``envs/fluid_env.py:749-917``, ``envs/cylinder/cylinder_env_base.py``, ``jet_cylinder_env_2d.py``):
``reset(seed, randomize)``, ``step(action)``, ``sample_action``, ``n_agents``, ``observation_space`` /
``action_space`` shapes, ``get_state/set_state``, and the error strings of
``tests/env_utils/test_fluid_env.py``.  Every tensor gains a leading environment dimension, exactly like
the reference's ``ParallelFluidEnv`` (``envs/parallel_env.py:233-287``) -- but the B environments live in
one process / one CUDA context and never leave the device.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from .. import native
from ..sensors import sensor_tables
from ..solver import BatchedPISO, _ptr
from .common import DifferentiableRollout, EpisodeLifecycle, InitialDomains, Renderable, build_wall_tables
from .cylinder_domain import BOTTOM, LEFT, RIGHT, TOP, WAKE, jet_profile, make_cylinder_domain

CYLINDER_ROT_2D_DEFAULT_CONFIG = {
    "reynolds_number": 1e2, "resolution": 24, "dt": 1e-2, "adaptive_cfl": 0.8, "step_length": 0.25,
    "episode_length": 80, "lift_penalty": 1.0,
}
CYLINDER_JET_2D_DEFAULT_CONFIG = {
    "reynolds_number": 1e2, "resolution": 24, "dt": 1e-2, "adaptive_cfl": 0.8, "step_length": 0.25,
    "episode_length": 80, "lift_penalty": 1.0,
}


def cylinder_jet_templates(spec, cd, jet_angle: float):
    """Jet velocity templates on the cylinder faces of the top / bottom blocks (jet_cylinder_env_2d.py:136-183; the 3-D
    environment repeats them in every z plane, jet_cylinder_env_3d.py:328-396) -> (face indices int32 [nf], template float32 [2, nf])."""

    def coords_to_velocities(coords_boundary, direction):
        cb = torch.from_numpy(np.ascontiguousarray(coords_boundary))
        centers = 0.5 * (cb[:, :-1] + cb[:, 1:])
        if direction == "top":
            angles = torch.pi / 2 - torch.atan2(centers[1, :], centers[0, :])
        else:
            angles = -torch.pi / 2 - torch.atan2(centers[1, :], centers[0, :])
        angles_deg = torch.rad2deg(angles)
        angles_deg_abs = torch.abs(angles_deg)
        angles_deg_abs[angles_deg_abs > jet_angle] = 0.0
        min_idx, max_idx = torch.where(angles_deg_abs > 0.0)[0][[0, -1]]
        min_idx, max_idx = int(min_idx) - 1, int(max_idx) + 1
        prof = torch.from_numpy(jet_profile(max_idx - min_idx + 1))
        vel = torch.zeros_like(centers)
        for i, um in zip(range(min_idx, max_idx + 1), prof):
            a = angles_deg[i]
            vel[0, i] = um * torch.sin(torch.deg2rad(a))
            vel[1, i] = um * torch.cos(torch.deg2rad(a))
        return vel.numpy()

    top_v = coords_to_velocities(spec.blocks[TOP].vertex[:, 0, :], "top")
    bot_v = coords_to_velocities(spec.blocks[BOTTOM].vertex[:, -1, :], "bottom")
    nx = spec.blocks[TOP].nx
    faces = np.concatenate([cd.boff[TOP, 2] + np.arange(nx), cd.boff[BOTTOM, 3] + np.arange(nx)]).astype(np.int32)
    templ = np.ascontiguousarray(np.concatenate([top_v, bot_v], axis=1).astype(np.float32))
    return faces, templ


def cylinder_sensor_locations(cylinder_diameter: float = 1.0) -> torch.Tensor:
    """[2, 151] physical sensor positions of the cylinder environments (CYL.py:457-516; shared by the 2-D and 3-D variants)"""
    x_idx = torch.arange(1.0, 5.0, step=0.5)
    y_idx = torch.arange(-1.5, 1.75, step=0.5)
    xy = torch.meshgrid(x_idx, y_idx, indexing="ij")
    loc = torch.stack([xy[0].ravel(), xy[1].ravel()], dim=0)
    x_1 = torch.arange(-0.25, 1, 0.25)
    y_1a, y_1b = torch.full_like(x_1, -1.5), torch.full_like(x_1, 1.5)
    x_2 = torch.concatenate([torch.tensor([-0.25]), torch.arange(0.25, 1.25, 0.25)])
    y_2a, y_2b = torch.full_like(x_2, cylinder_diameter), torch.full_like(x_2, -cylinder_diameter)
    x_3, y_3 = torch.tensor([0.75] * 3), torch.tensor([-0.5, 0, 0.5])
    add = torch.stack([torch.concatenate([x_1, x_1, x_2, x_2, x_3]), torch.concatenate([y_1a, y_1b, y_2a, y_2b, y_3])], dim=0)
    ang = torch.linspace(0, 2 * torch.pi, steps=36)
    r1, r2 = 2 * 0.5, 1.25 * 0.5
    c1 = torch.stack([r1 * torch.cos(ang), r1 * torch.sin(ang)], dim=0)
    c2 = torch.stack([r2 * torch.cos(ang), r2 * torch.sin(ang)], dim=0)
    return torch.concatenate([loc, c1, c2, add], dim=1)


class CylinderJet2DEnv(EpisodeLifecycle, DifferentiableRollout, InitialDomains, Renderable):
    H, L, cylinder_diameter, U_mean, cylinder_offset_y = 4.1, 22.0, 1.0, 1.0, 0.05
    n_sensors = 151
    action_smoothing_alpha = 0.1
    jet_angle = 10.0
    metrics = ["drag", "lift"]
    reference_values = {"cd_ref": ("drag", "mean")}
    render_fields = ("vorticity", "velocity_magnitude", "velocity_x", "velocity_y", "pressure")
    bc_tol = 5e-6            # flux-balance tolerance of the cylinder's outflow hook (cylinder_env_base.py:293-295: tol=5e-6, 2-D and 3-D)

    def __init__(self, n_envs: int = 1, reynolds_number=1e2, resolution=24, dt=1e-2, adaptive_cfl=0.8, step_length=0.25,
                 episode_length=80, lift_penalty=1.0, device="cuda:0", cg_impl=11, compiled=None, cd_ref=0.0,
                 randomize_initial_state=False, enable_actions=True, use_marl=False, differentiable=False, load_initial_domain=False,
                 initial_domains_path=None, per_env_substeps: bool = False):
        if use_marl:
            raise ValueError("CylinderJet2D is a single-agent environment (n_agents == 1)")
        self.per_env_substeps = bool(per_env_substeps)
        self.n_envs = int(n_envs)
        self.resolution, self.dt, self.cfl = int(resolution), float(dt), float(adaptive_cfl)
        self.step_length, self.episode_length = float(step_length), int(episode_length)
        self.lift_penalty, self.cd_ref = float(lift_penalty), float(cd_ref)
        self.randomize_initial_state = randomize_initial_state
        self.enable_actions = enable_actions
        self.differentiable = bool(differentiable)
        self.load_domain_on_reset, self.initial_domains_path = bool(load_initial_domain), initial_domains_path
        self.reynolds_number = float(reynolds_number)
        self.device = torch.device(device)
        if compiled is None:
            spec = make_cylinder_domain(resolution, reynolds_number, self.U_mean, self.H, self.L, self.cylinder_offset_y)
            cd = spec.prepare()
        else:
            spec, cd = compiled
        self.spec, self.cd = spec, cd
        out_mask = np.zeros(cd.NB, dtype=np.int8)
        o = cd.boff[WAKE, 1]
        out_mask[o:o + spec.blocks[WAKE].ny] = 1
        self.solver = BatchedPISO(cd, self.n_envs, device=device, corrector_steps=2, advect_non_ortho_steps=1,
                                  pressure_non_ortho_steps=1, non_orthogonal=True, pressure_tol=1e-5, cg_impl=cg_impl,
                                  out_mask=out_mask)
        self.lib = self.solver.lib
        self.char_vel = (self.U_mean, 0.0)
        self._setup_jets()
        self._setup_wall()
        self._setup_sensors()
        B, dev = self.n_envs, self.device
        self.last_control = torch.zeros(B, device=dev)
        self._acc = torch.zeros(B, 2, device=dev)
        self._zero_action = torch.zeros(B, 1, device=dev)

    # ---- static tables ---------------------------------------------------------------------------
    def _setup_jets(self):
        faces, templ = cylinder_jet_templates(self.spec, self.cd, self.jet_angle)
        self.jet_faces = torch.from_numpy(faces).to(self.device)
        self.jet_templ = torch.from_numpy(templ).to(self.device)

    def _setup_wall(self):
        """Ring of wall-adjacent cells around the cylinder and its geometry (CYL.py:548-655,
        forces.py:12-39, 42-107)."""
        ring = [(LEFT, 1, False), (TOP, 2, False), (RIGHT, 0, True), (BOTTOM, 3, True)]
        self._wall_t, self.wall = build_wall_tables(self.cd, self.spec, ring, self.device,
                                                    1.0 / (0.5 * self.U_mean ** 2 * self.cylinder_diameter))

    @property
    def render_shape(self):
        z = self.resolution * 4
        return (int(z / self.H * self.L), z)

    def sensor_locations_physical(self) -> torch.Tensor:
        return cylinder_sensor_locations(self.cylinder_diameter)

    def _build_render_map(self, plane):
        from ..render import render_map_2d
        return render_map_2d([b.vertex for b in self.spec.blocks], self.render_shape, fill_max_steps=16)

    def _setup_sensors(self):
        pc = self.sensor_locations_physical()
        rs = self.render_shape
        pc[0, :] += 2.0
        pc[0, :] *= (rs[0] - 1) / (self.L - 2.0)
        pc[1, :] += self.H / 2
        pc[1, :] *= (rs[1] - 1) / self.H
        self.sensor_px = torch.round(pc).to(torch.int32).numpy()
        idx, w = sensor_tables([b.vertex for b in self.spec.blocks], rs, self.sensor_px, fill_max_steps=16)
        self.sens_idx = torch.from_numpy(idx).to(self.device)
        self.sens_w = torch.from_numpy(w).to(self.device)

    # ---- reference-shaped API ---------------------------------------------------------------------
    @property
    def n_agents(self):
        return 1

    @property
    def initial_domain_id(self):
        """cylinder_env_base.py:823-828"""
        return f"cylinder_2D_Re{int(self.reynolds_number)}_Res{self.resolution}"

    use_marl = False

    @property
    def observation_space(self):
        """cylinder_env_base.py:203-233 (per environment)."""
        from .. import spaces
        inf = float("inf")
        ns = int(self.sens_idx.shape[1])
        return spaces.Dict({"velocity": spaces.Box(-inf, inf, shape=(ns, 2)), "pressure": spaces.Box(-inf, inf, shape=(ns,))})

    @property
    def action_space(self):
        from .. import spaces
        return spaces.Box(-1.0, 1.0, shape=(1,))

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
        randomize = self.randomize_initial_state if randomize is None else randomize
        if self.load_domain_on_reset:
            self._load_initial_domains_on_reset(randomize)          # fluid_env.py:519-539
        else:
            s.u.zero_()
            s.p.zero_()
            s.bvel.copy_(torch.from_numpy(self.cd.bvel0[:, :self.cd.NB].copy()).to(self.device).unsqueeze(0).expand_as(s.bvel))
        # Simulation.make_divergence_free incl. its "PRE" hook with time step 1 (SIM.py:1335-1347)
        s.update_outflow(1.0, self.char_vel, tol=self.bc_tol)
        s.make_divergence_free(max_iter=1000)
        self.last_control.zero_()
        if randomize:
            self._randomize_domain()
        self._apply_action(self._zero_action, smooth=False)
        self._dstate = None
        self._reset_called = True
        self._n_steps = 0
        return self._get_obs(), {}

    def _randomize_domain(self):
        """CYL.py:364-404 (per-environment noise, common number of settling steps)."""
        period = 1 / (0.3 * self.U_mean / self.cylinder_diameter)
        max_n = 2 * int(period / self.step_length) - 1
        n_steps = int(self._np_rng.integers(int(0.5 * max_n), max_n)) + 1
        s = self.solver
        s.u += torch.randn(s.u.shape, device=self.device, generator=self._torch_rng) * 0.025
        s.p += torch.randn(s.p.shape, device=self.device, generator=self._torch_rng) * 0.025
        for _ in range(n_steps):
            s.single_step(self.dt, self.cfl, char_vel=self.char_vel, bc_tol=self.bc_tol)

    def _apply_action(self, action, smooth=True):
        """jet_cylinder_env_2d.py:185-188 with the exponential smoothing of CYL.py:748-751."""
        a = torch.as_tensor(action, dtype=torch.float32, device=self.device).reshape(self.n_envs).contiguous()
        if not smooth:
            self.last_control.copy_(a)
        native.check(self.lib.fgb_apply_jet_action(self.solver.handle, _ptr(self.solver.bvel), _ptr(self.last_control), _ptr(a),
                                                   self.action_smoothing_alpha if smooth else 0.0, _ptr(self.jet_faces),
                                                   _ptr(self.jet_templ), int(self.jet_faces.numel()), self.solver.stream),
                     "fgb_apply_jet_action")

    def _get_obs(self):
        s = self.solver
        B, ns = self.n_envs, self.sens_idx.shape[1]
        K = self.sens_idx.shape[0]
        vel = torch.empty(B, 2, ns, device=self.device)
        prs = torch.empty(B, 1, ns, device=self.device)
        native.check(self.lib.fgb_sample_sensors(s.handle, _ptr(s.u), 2, _ptr(self.sens_idx), _ptr(self.sens_w), K, ns, _ptr(vel),
                                                 s.stream), "fgb_sample_sensors")
        native.check(self.lib.fgb_sample_sensors(s.handle, _ptr(s.p), 1, _ptr(self.sens_idx), _ptr(self.sens_w), K, ns, _ptr(prs),
                                                 s.stream), "fgb_sample_sensors")
        return {"velocity": vel.permute(0, 2, 1).contiguous(), "pressure": prs[:, 0]}

    def _advance(self, action):
        s = self.solver
        self._acc.zero_()
        nsub = 0
        for _ in range(self.n_sim_steps):
            if self.enable_actions:
                self._apply_action(action)
            nsub += s.single_step(self.dt, self.cfl, char_vel=self.char_vel, bc_tol=self.bc_tol)
            native.check(self.lib.fgb_wall_forces(s.handle, C.byref(self.wall), _ptr(s.u), _ptr(s.p), _ptr(s.bvel), _ptr(self._acc),
                                                  s.stream), "fgb_wall_forces")
        self.last_substeps = nsub
        return self._acc

    def _reward(self, cd, cl):
        """cylinder_env_base.py:769"""
        return self.cd_ref - cd - self.lift_penalty * torch.abs(cl)

    # ---- differentiable mode (fluid_env.py:154,232; examples/interfaces/gradient_based_methods.py) -----------------
    # The PISO substep is one autograd node backed by the CUDA adjoint (fluidgym_b200.autograd); the few boundary
    # and reward formulas around it are tiny torch expressions over the same static tables the kernels use, so
    # gradients flow from the reward to the action, the block velocities and the boundary values exactly as in
    # the reference, where those parts are torch code as well (SIM.py:188-393, forces.py:193-275).
    def _advance_differentiable(self, action):
        s = self.solver
        if self._dstate is None:
            self._dstate = (s.u.clone(), s.p.clone(), s.bvel.clone(), self.last_control.clone())
        u, p, bv, last = self._dstate
        a = action.reshape(self.n_envs)
        acc = torch.zeros(self.n_envs, 2, device=self.device)
        nsub = 0
        self._begin_substep_count()
        for _ in range(self.n_sim_steps):
            if self.enable_actions:
                last = last + self.action_smoothing_alpha * (a - last)
                bv = bv.index_copy(2, self.jet_faces.long(), self.jet_templ[None] * last[:, None, None])
            u, p, bv, k = self._single_step_differentiable(u, p, bv)
            nsub += k
            acc = acc + self._forces_torch(u, p, bv)
        self._dstate = (u, p, bv, last)
        with torch.no_grad():                      # keep the solver's own state in step for obs / get_state
            s.u.copy_(u); s.p.copy_(p); s.bvel.copy_(bv); self.last_control.copy_(last)
        self.last_substeps = nsub
        return acc


class CylinderRot2DEnv(CylinderJet2DEnv):
    """``CylinderRotEnv2D`` (envs/cylinder/rotating_cylinder_env_2d.py:20-182): the action is the rotation speed of
    the cylinder wall.  Same solver, forces, sensors and smoothing as the jet environment; only the boundary
    template differs -- unit tangential velocity ``(sin theta, -cos theta)`` on all four cylinder faces
    (:131-139) instead of the two jet slots, so the same ``fgb_apply_jet_action`` kernel drives it."""

    def _setup_jets(self):
        cd, spec = self.cd, self.spec
        faces, templ = [], []
        # (block, face, boundary vertex line) in the reference's order: left +x, top -y, right -x, bottom +y
        for bi, f, line in ((LEFT, 1, spec.blocks[LEFT].vertex[:, :, -1]), (TOP, 2, spec.blocks[TOP].vertex[:, 0, :]),
                            (RIGHT, 0, spec.blocks[RIGHT].vertex[:, :, 0]), (BOTTOM, 3, spec.blocks[BOTTOM].vertex[:, -1, :])):
            cb = torch.from_numpy(np.ascontiguousarray(line))
            centers = 0.5 * (cb[:, :-1] + cb[:, 1:])
            theta = torch.atan2(centers[1, :], centers[0, :])
            templ.append(torch.stack([torch.sin(theta), -torch.cos(theta)]).numpy())
            faces.append(cd.boff[bi, f] + np.arange(centers.shape[1]))
        self.jet_faces = torch.from_numpy(np.concatenate(faces).astype(np.int32)).to(self.device)
        self.jet_templ = torch.from_numpy(np.ascontiguousarray(np.concatenate(templ, axis=1).astype(np.float32))).to(self.device)
