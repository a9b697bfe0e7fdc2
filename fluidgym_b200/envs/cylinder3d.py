"""Batched ``CylinderJet3D`` environment (``envs/cylinder/jet_cylinder_env_3d.py`` + ``cylinder_env_base.py`` with ``ndims = 3``):
the 5-block cylinder grid extruded over ``resolution`` periodic z planes (span 4 D), ``n_jets`` pairs of synthetic jets lined up
along the span -- one agent per jet with ``use_marl=True`` --, drag / lift per plane, sensors read from the rendered voxel grid.

STATUS: every host-side piece of this class (jets, flux balances, outflow update, CFL plan, forces, observations, rewards,
multi-agent windows) runs on the CPU in tests/test_cylinder3d_cpu.py on top of a stand-in solver that executes the per-cell code
of the CUDA kernels on the host, and reproduces the unmodified reference's first ``env.step`` (tests/golden/cyl3d_env.npz).  The
CUDA path underneath (``ExtrudedPISO3D`` -> ``fgb_extruded3_*``) is verified on a B200 against the same goldens
(tests/test_gpu_extruded.py: substep, reset, ``env.step``; boundary hooks / forces / jets as kernels by default), and so is the
differentiable mode (reverse mode of the extruded substep against the reference's own gradients).  All tensors carry a leading
environment dimension.
"""
from __future__ import annotations

import numpy as np
import torch

from ..sensors import sensor_tables_extruded
from ..solver import cfl_substeps
from .common import DifferentiableRollout, EpisodeLifecycle, InitialDomainsExtruded, Renderable, build_wall_tables
from .cylinder import cylinder_jet_templates, cylinder_sensor_locations
from .cylinder_domain import BOTTOM, LEFT, RIGHT, TOP, WAKE, make_cylinder_domain
from .spanwise import global_obs_from_samples, local_obs_windows, spanwise_sensor_voxels

CYLINDER_JET_3D_DEFAULT_CONFIG = {
    "n_jets": 8, "reynolds_number": 1e2, "resolution": 24, "dt": 1e-2, "adaptive_cfl": 0.8, "step_length": 0.25, "lift_penalty": 1.0,
    "episode_length": 80, "local_obs_window": 3, "local_reward_weight": 0.8, "local_2d_obs": False, "use_marl": False,
}


class SpanwiseExtrudedEnv(EpisodeLifecycle, InitialDomainsExtruded, Renderable):
    """What the environments on z-extruded domains with agents lined up along the span share (CylinderJet3D, Airfoil3D): the
    reference-shaped API, reset (zero field + inflow -> projection, or an on-disk initial domain), the solver-step loop with action
    smoothing, per-plane wall forces, voxel sensors, multi-agent windows and the local / global reward mix.  A subclass provides the
    tables (``spec, cd, nz, hz, z_vertices, n_span, nz_per_agent, solver, jet_*, _wall_t, wall, sens_idx, sens_w, last_control,
    _zero_action, _bvel0``), ``_apply_action(control)``, ``_reward(cd, cl)``, ``_randomize_domain()`` and the spaces' shapes."""

    action_smoothing_alpha = 0.1
    bc_tol = 5e-6
    metrics = ["drag", "lift"]
    render_fields = ("velocity_magnitude", "velocity_x", "velocity_y", "velocity_z", "pressure")
    render_fill_steps = 16                  # the hole-filling sweeps of the family's sensors

    def _render_planes(self):
        Z = self.render_shape[2]
        return Z, Z // 2

    def _build_render_map(self, plane):
        from ..render import render_map_extruded
        return render_map_extruded([b.vertex for b in self.spec.blocks], self.z_vertices, self.render_shape, plane, self.render_fill_steps)

    @property
    def n_sensors_z(self):
        return self.n_span * self.n_sensors_per_agent

    @property
    def n_agents(self):
        return self.n_span if self.use_marl else 1

    @property
    def observation_space(self):
        """jet_cylinder_env_3d.py:205-258 (per environment, per agent with use_marl)"""
        from .. import spaces
        inf, nxy, spa = float("inf"), self.n_sensors_xy, self.n_sensors_per_agent
        if self.use_marl and self.local_2d_obs:
            vs, ps = (nxy, 2), (nxy,)
        elif self.use_marl:
            vs, ps = (self.local_obs_window, spa, 3, nxy), (self.local_obs_window, spa, nxy)
        else:
            vs, ps = (self.n_span, spa, 3, nxy), (self.n_span, spa, nxy)
        return spaces.Dict({"velocity": spaces.Box(-inf, inf, shape=vs), "pressure": spaces.Box(-inf, inf, shape=ps)})

    def set_state(self, u, p, bvel, last_control=None):
        s = self.solver
        for dst, src in ((s.u, u), (s.p, p), (s.bvel, bvel)):
            src = torch.as_tensor(src, dtype=torch.float32, device=self.device)
            self._copy_state(dst, src.reshape(dst.shape[1:]) if src.numel() == dst[0].numel() else src.reshape(dst.shape))
        if last_control is not None:
            self.last_control.copy_(torch.as_tensor(last_control, device=self.device).expand_as(self.last_control))
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
            s.bvel.zero_()
            s.bvel[:, :2] = self._bvel0[None, :, None, :]
            self._initial_velocity()
        s.make_divergence_free_with_hook(max_iter=1000, bc_tol=self.bc_tol)      # cylinder_env_base.py:325; SIM.py:1320-1430
        self.last_control.zero_()
        if randomize:
            self._randomize_domain()
        self._apply_action(torch.zeros_like(self.last_control))     # fluid_env.py:909
        self._n_steps = 0
        self._reset_called = True
        return self._get_obs(), {}

    def _initial_velocity(self):
        """hook between the zero field and the projection (Airfoil3D: ``init_from_2d``)"""

    def _drag_and_lift(self):
        """Per-plane drag / lift coefficients [B, nz] each (cylinder_env_base.py:657-700, forces.py:278-377: the 2-D wall
        traction of every plane times the plane spacing)."""
        s = self.solver
        B, nz, N2 = self.n_envs, self.nz, s.N2
        if s.u.is_cuda and getattr(s, "_cuda_hooks", lambda: False)():                           # kernel path (default; FGB_X3_HOOKS=torch: torch expressions)
            import ctypes as C
            from .. import native
            from ..solver import _ptr
            out = torch.empty(B, nz, 2, device=self.device)
            native.check(s.lib.fgb_extruded3_wall_forces(C.byref(s.xtables), B, C.byref(self.wall), _ptr(s.u), _ptr(s.p), _ptr(s.bvel), _ptr(out),
                                                         s.stream), "fgb_extruded3_wall_forces")
            return out[:, :, 0], out[:, :, 1]
        u2 = s.u.view(B, 3, nz, N2)[:, :2].permute(0, 2, 1, 3).reshape(B * nz, 2, N2)
        p2 = s.p.view(B * nz, N2)
        b2 = s.bvel[:, :2].permute(0, 2, 1, 3).reshape(B * nz, 2, -1)
        f = DifferentiableRollout._forces_torch(self, u2, p2, b2).view(B, nz, 2) * self.hz
        return f[:, :, 0], f[:, :, 1]

    def _sample(self, field: torch.Tensor) -> torch.Tensor:
        """[B, C, N3] -> [B, C, n_sensors]: the rendered-voxel map evaluated at the sensor voxels only (static ELL rows)"""
        s = self.solver
        if field.is_cuda and getattr(s, "_cuda_hooks", lambda: False)():                         # kernel path (default; FGB_X3_HOOKS=torch: torch expressions)
            from .. import native
            from ..solver import _ptr
            if not hasattr(self, "_sens_idx32"):
                self._sens_idx32 = self.sens_idx.to(torch.int32).contiguous()
            f = field.contiguous()
            K, ns = self.sens_idx.shape
            out = torch.empty(f.shape[0], f.shape[1], ns, device=f.device)
            native.check(s.lib.fgb_sample_sensors_n(_ptr(f), f.shape[0], f.shape[1], s.N, _ptr(self._sens_idx32), _ptr(self.sens_w), K, ns,
                                                    _ptr(out), s.stream), "fgb_sample_sensors_n")
            return out
        return (field[:, :, self.sens_idx] * self.sens_w).sum(dim=2)

    def _get_global_obs(self):
        s = self.solver
        us = self._sample(s.u).permute(0, 2, 1)                                                   # [B, sensors, 3]
        ps = self._sample(s.p[:, None])[:, 0]
        return global_obs_from_samples(us, ps, self.n_span, self.n_sensors_per_agent, local_2d_obs=self.local_2d_obs)

    def _get_local_obs(self):
        loc = local_obs_windows(self._get_global_obs(), self.local_obs_window)
        if self.local_2d_obs:                                                                     # window.squeeze(), :313-314
            loc = {k: v.reshape(v.shape[0], v.shape[1], *[d for d in v.shape[2:] if d != 1]) for k, v in loc.items()}
        return loc

    def _get_obs(self):
        return self._get_local_obs() if self.use_marl else self._get_global_obs()

    # ---- differentiable mode: one autograd node per substep (autograd.PISOSubstepExtruded, CUDA adjoint of the extruded path); the
    # boundary hooks, the jets and the wall forces around it are functional torch expressions with the graph cut where the reference
    # cuts it: update_advective_boundaries runs entirely under no_grad (SIM.py:232), balance_boundary_fluxes computes its scale under
    # no_grad and applies it outside (SIM.py:191-224).  One common substep size for the batch (the most restrictive environment decides), or
    # with per_env_substeps every environment's own plan (EpisodeLifecycle._substep_rounds).
    differentiable = False

    def mark_state_differentiable(self):
        """envs/util/diff_tools.py:8-22: the velocity leaf of the incoming state [B, 3, nz * N2]"""
        s = self.solver
        u = s.u.detach().clone().requires_grad_(True)
        self._dstate = (u, s.p.detach().clone(), s.bvel.detach().clone(), self.last_control.detach().clone())
        return u

    def _balance_fn(self, bv, free, tol):
        s = self.solver
        fw = s._st["fw"]
        with torch.no_grad():
            fl = (bv[:, 0] * fw[0] + bv[:, 1] * fw[1]) * s.hz                                     # [B, nz, NB2]
            var = fl[:, :, free].double().sum(dim=(1, 2))
            fixed = fl[:, :, ~free].double().sum(dim=(1, 2))
            ok = (fixed + var).abs() <= tol * 0.01
            sc = torch.where(ok, torch.ones_like(var), -fixed / torch.where(ok, torch.ones_like(var), var)).float()
            scale = torch.where(free[None, None, None, :], sc[:, None, None, None], torch.ones((), device=bv.device))
        return bv * scale

    def _outflow_fn(self, u, bv, dtv, tol):
        s = self.solver
        st = s._st
        with torch.no_grad():
            w = 1.0 - 1.0 / (1.0 + 2.0 * dtv[:, None] * st["adv"][None])                          # [B, n_out]
            u4 = u.view(self.n_envs, 3, self.nz, s.N2)
            bo = bv[:, :, :, st["out"]]
            bo = bo - w[:, None, None, :] * (bo - u4[:, :, :, st["out_cells"]])
            bo = self._balance_fn(bv.index_copy(3, st["out"], bo), st["is_out"], tol)[:, :, :, st["out"]]
        return bv.index_copy(3, st["out"], bo)

    def _single_step_differentiable(self, u, p, bv):
        from ..autograd import piso_substep_extruded
        s = self.solver
        st = s._st

        def max_velocity():
            with torch.no_grad():
                u4, mi, bm = u.view(self.n_envs, 3, self.nz, s.N2), st["minv"], st["b_minv"]
                return float(torch.stack([(mi[0] * u4[:, 0] + mi[1] * u4[:, 1]).abs().max(), (mi[2] * u4[:, 0] + mi[3] * u4[:, 1]).abs().max(),
                                          u4[:, 2].abs().max() / s.hz, (bm[0] * bv[:, 0] + bm[1] * bv[:, 1]).abs().max(),
                                          (bm[2] * bv[:, 0] + bm[3] * bv[:, 1]).abs().max(), bv[:, 2].abs().max() / s.hz]).max())

        def max_velocity_env():                     # the same maxima per environment (ExtrudedStepping.max_velocity of u, bv)
            with torch.no_grad():
                u4, mi, bm = u.view(self.n_envs, 3, self.nz, s.N2), st["minv"], st["b_minv"]
                return torch.stack([(mi[0] * u4[:, 0] + mi[1] * u4[:, 1]).abs().amax(dim=(1, 2)), (mi[2] * u4[:, 0] + mi[3] * u4[:, 1]).abs().amax(dim=(1, 2)),
                                    u4[:, 2].abs().amax(dim=(1, 2)) / s.hz, (bm[0] * bv[:, 0] + bm[1] * bv[:, 1]).abs().amax(dim=(1, 2)),
                                    (bm[2] * bv[:, 0] + bm[3] * bv[:, 1]).abs().amax(dim=(1, 2)), bv[:, 2].abs().amax(dim=(1, 2)) / s.hz]).amax(dim=0)
        nsub = 0
        if self.per_env_substeps:
            for dtv, act in self._substep_rounds(max_velocity_env):
                bv = torch.where(act.bool()[:, None, None, None], self._outflow_fn(u, bv, dtv, self.bc_tol), bv)
                u, p = piso_substep_extruded(s, u, p, bv, dtv, active=act)
                nsub += 1
            return u, p, bv, nsub
        for ts in cfl_substeps(self.dt, self.cfl, max_velocity):                                   # SIM.py:2004-2031
            dtv = torch.full((self.n_envs,), ts, device=self.device)
            bv = self._outflow_fn(u, bv, dtv, self.bc_tol)
            u, p = piso_substep_extruded(s, u, p, bv, dtv)
            nsub += 1
        return u, p, bv, nsub

    def _advance_differentiable(self, a):
        s = self.solver
        B, nz, N2 = self.n_envs, self.nz, s.N2
        if self._dstate is None:
            self._dstate = (s.u.clone(), s.p.clone(), s.bvel.clone(), self.last_control.clone())
        u, p, bv, last = self._dstate
        cds = torch.zeros(B, nz, device=self.device)
        cls_ = torch.zeros_like(cds)
        jf = self.jet_faces.long()
        nsub = 0
        self._begin_substep_count()
        for _ in range(self.n_sim_steps):
            last = last + self.action_smoothing_alpha * (a - last)
            if self.enable_actions:
                jets, tol = self._jet_profiles(last)                                              # [B, 2, nz, n_jet_faces] (no spanwise component)
                bv = bv.index_copy(3, jf, torch.cat([jets, torch.zeros_like(jets[:, :1])], dim=1))
                bv = self._balance_fn(bv, self._free_jets, tol)
            u, p, bv, k = self._single_step_differentiable(u, p, bv)
            nsub += k
            u2 = u.view(B, 3, nz, N2)[:, :2].permute(0, 2, 1, 3).reshape(B * nz, 2, N2)
            f = DifferentiableRollout._forces_torch(self, u2, p.view(B * nz, N2), bv[:, :2].permute(0, 2, 1, 3).reshape(B * nz, 2, -1))
            f = f.view(B, nz, 2) * self.hz
            cds, cls_ = cds + f[:, :, 0], cls_ + f[:, :, 1]
        self._dstate = (u, p, bv, last)
        with torch.no_grad():                      # keep the solver's own state in step for observations / get_state
            s.u.copy_(u); s.p.copy_(p); s.bvel.copy_(bv); self.last_control = last.detach().clone()
        self.last_substeps = nsub
        return cds, cls_

    def step(self, action):
        action = self._begin_step(action)
        if self.use_marl and self.local_reward_weight is None:
            raise ValueError("local_reward_weight must be set for multi-agent step.")
        s = self.solver
        a = action.reshape(self.last_control.shape)
        if self.differentiable:
            cds, cls_ = self._advance_differentiable(a)
        else:
            cds = torch.zeros(self.n_envs, self.nz, device=self.device)
            cls_ = torch.zeros_like(cds)
            nsub = 0
            for _ in range(self.n_sim_steps):                                                     # cylinder_env_base.py:741-776
                self.last_control = self.last_control + self.action_smoothing_alpha * (a - self.last_control)
                if self.enable_actions:
                    self._apply_action(self.last_control)
                nsub += s.single_step(self.dt, self.cfl, bc_tol=self.bc_tol)
                cd_k, cl_k = self._drag_and_lift()
                cds += cd_k
                cls_ += cl_k
            self.last_substeps = nsub
        all_cds, all_cls = cds / self.n_sim_steps, cls_ / self.n_sim_steps
        cd, cl = all_cds.sum(dim=1) / self.D, all_cls.sum(dim=1) / self.D                        # jet_cylinder_env_3d.py:431-452
        reward = self._reward(cd, cl)
        truncated = self._end_step()
        info = {"drag": cd, "lift": cl}
        if not self.use_marl:
            info["all_cds"], info["all_cls"] = all_cds, all_cls
            return self._get_global_obs(), reward, False, truncated, info
        per = self.D / self.n_span                                                                # :454-486
        local_cd = all_cds.view(self.n_envs, self.n_span, -1).sum(dim=2) / per
        local_cl = all_cls.view(self.n_envs, self.n_span, -1).sum(dim=2) / per
        local = self._reward(local_cd, local_cl)
        lw = float(self.local_reward_weight)
        info["global_reward"] = reward
        return self._get_local_obs(), lw * local + (1 - lw) * reward[:, None], False, truncated, info


class CylinderJet3DEnv(SpanwiseExtrudedEnv):
    H, L, D, cylinder_diameter, U_mean, cylinder_offset_y = 4.1, 22.0, 4.0, 1.0, 1.0, 0.05
    action_smoothing_alpha = 0.1
    jet_angle = 10.0
    bc_tol = 5e-6                                                       # tolerance of the outflow update's flux balance (:295)
    metrics = ["drag", "lift"]
    reference_values = {"cd_ref": ("drag", "mean")}

    def __init__(self, n_envs: int = 1, n_jets=8, reynolds_number=1e2, resolution=24, dt=1e-2, adaptive_cfl=0.8, step_length=0.25,
                 episode_length=80, lift_penalty=1.0, local_obs_window=3, use_marl=False, local_reward_weight=0.8, local_2d_obs=False,
                 device="cuda:0", cd_ref=0.0, randomize_initial_state=False, enable_actions=True, load_initial_domain=False,
                 initial_domains_path=None, compiled=None, solver_cls=None, differentiable=False, per_env_substeps: bool = False):
        self.load_domain_on_reset, self.initial_domains_path = bool(load_initial_domain), initial_domains_path
        self.differentiable = bool(differentiable)
        self.per_env_substeps = bool(per_env_substeps)
        if n_jets < 1 or resolution % n_jets != 0:
            raise ValueError("n_agents must be a positive integer that evenly dividescircle_resolution_angular.")
        if local_2d_obs and not use_marl:
            raise ValueError("Local 2D observations are only supported in multi-agent mode.")
        self.n_envs, self.n_jets = int(n_envs), int(n_jets)
        self.n_span = self.n_jets                                   # agents lined up along the span
        self.resolution, self.dt, self.cfl = int(resolution), float(dt), float(adaptive_cfl)
        self.step_length, self.episode_length = float(step_length), int(episode_length)
        self.lift_penalty, self.cd_ref = float(lift_penalty), float(cd_ref)
        self.use_marl, self.local_reward_weight, self.local_2d_obs = bool(use_marl), local_reward_weight, bool(local_2d_obs)
        self.local_obs_window = 1 if local_2d_obs else int(local_obs_window)
        self.n_sensors_per_agent = 1 if local_2d_obs else 2
        self.randomize_initial_state, self.enable_actions = randomize_initial_state, enable_actions
        self.reynolds_number = float(reynolds_number)
        self.device = torch.device(device)
        if compiled is None:
            spec = make_cylinder_domain(resolution, reynolds_number, self.U_mean, self.H, self.L, self.cylinder_offset_y)
            cd = spec.prepare()
        else:
            spec, cd = compiled
        self.spec, self.cd = spec, cd
        self.nz = self.resolution                                   # grid.py:291-298: res_z = angular resolution, z in [-2, 2]
        self.hz = self.D / self.nz
        self.z_vertices = np.linspace(-2.0, 2.0, self.nz + 1, dtype=np.float32)
        self.nz_per_agent = self.nz // self.n_jets
        if solver_cls is None:
            from ..extruded3d import ExtrudedPISO3D as solver_cls   # raises without a CUDA device: there is no CPU path
        # cylinder_env_base.py:305-323: 2 correctors, 1 + 4 deferred non-orthogonal iterations, tolerances 1e-5 / 5e-7
        self.solver = solver_cls(cd, self.nz, self.hz, self.n_envs, device=device, corrector_steps=2, advect_non_ortho_steps=1,
                                 pressure_non_ortho_steps=4, advection_tol=1e-5, pressure_tol=5e-7, max_iter=5000)
        out_mask = np.zeros(cd.NB, dtype=bool)
        o = cd.boff[WAKE, 1]
        out_mask[o:o + spec.blocks[WAKE].ny] = True
        self.solver.setup_stepping(out_mask, (self.U_mean, 0.0))
        faces, templ = cylinder_jet_templates(spec, cd, self.jet_angle)     # the 2-D templates, repeated in every plane (:328-396)
        self.jet_faces = torch.from_numpy(faces).to(self.device)
        self.jet_templ = torch.from_numpy(templ).to(self.device)
        free = out_mask.copy()
        free[self.jet_faces.cpu().numpy()] = True
        self._free_jets = torch.from_numpy(free).to(self.device)
        ring = [(LEFT, 1, False), (TOP, 2, False), (RIGHT, 0, True), (BOTTOM, 3, True)]
        self._wall_t, self.wall = build_wall_tables(cd, spec, ring, self.device, 1.0 / (0.5 * self.U_mean ** 2 * self.cylinder_diameter))
        self._setup_sensors()
        B, dev = self.n_envs, self.device
        self.last_control = torch.zeros(B, self.n_jets, device=dev)
        self._zero_action = torch.zeros(B, self.n_jets, 1, device=dev)
        self._bvel0 = torch.from_numpy(np.ascontiguousarray(cd.bvel0[:, :cd.NB])).to(dev)

    @property
    def render_shape(self):
        z = self.resolution * 4
        return (int(z / self.H * self.L), z, z)

    def _setup_sensors(self):
        xy = cylinder_sensor_locations(self.cylinder_diameter)
        self.n_sensors_xy = int(xy.shape[1])
        rs = self.render_shape
        self.sensor_px = spanwise_sensor_voxels(xy, self.n_sensors_z, self.H, self.L, rs).numpy()
        idx, w = sensor_tables_extruded([b.vertex for b in self.spec.blocks], self.z_vertices, rs, self.sensor_px, fill_max_steps=16)
        self.sens_idx = torch.from_numpy(idx.astype(np.int64)).to(self.device)
        self.sens_w = torch.from_numpy(w).to(self.device)

    @property
    def id(self):
        return f"JetCylinder3D_Re{self.reynolds_number}"

    @property
    def initial_domain_id(self):
        return f"cylinder_3D_Re{int(self.reynolds_number)}_Res{self.resolution}"

    @property
    def action_space(self):
        from .. import spaces
        return spaces.Box(-1.0, 1.0, shape=(1,) if self.use_marl else (self.n_jets, 1))

    def _randomize_domain(self):
        """cylinder_env_base.py:364-404 (per-environment noise, common number of settling steps)"""
        period = 1 / (0.3 * self.U_mean / self.cylinder_diameter)
        max_n = 2 * int(period / self.step_length) - 1
        n_steps = int(self._np_rng.integers(int(0.5 * max_n), max_n)) + 1
        s = self.solver
        s.u += torch.randn(s.u.shape, device=self.device, generator=self._torch_rng) * 0.025
        s.p += torch.randn(s.p.shape, device=self.device, generator=self._torch_rng) * 0.025
        for _ in range(n_steps):
            s.single_step(self.dt, self.cfl, bc_tol=self.bc_tol)

    def _apply_action(self, control: torch.Tensor):
        """jet_cylinder_env_3d.py:399-424: every jet drives its ``nz_per_agent`` planes with the 2-D template (no spanwise
        component), then jets and outflow are rescaled for a zero net boundary flux (tol 1e-7)."""
        s = self.solver
        per_plane = control.repeat_interleave(self.nz_per_agent, dim=1)                           # [B, nz]
        if getattr(s, "apply_jets", None) and s.apply_jets(per_plane[:, :, None], self.jet_templ[None], self.jet_faces, self._free_jets, 1e-7):
            return                                                                                # kernel path (default; FGB_X3_HOOKS=torch: torch expressions)
        jf = self.jet_faces.long()
        s.bvel[:, :2, :, jf] = self.jet_templ[None, :, None, :] * per_plane[:, None, :, None]
        s.bvel[:, 2, :, jf] = 0.0
        s.balance_fluxes(self._free_jets, 1e-7)

    def _jet_profiles(self, control):
        """functional form of _apply_action for the differentiable mode -> (in-plane jet velocities [B, 2, nz, n_faces], balance tolerance)"""
        per_plane = control.repeat_interleave(self.nz_per_agent, dim=1)                           # [B, nz]
        return self.jet_templ[None, :, None, :] * per_plane[:, None, :, None], 1e-7

    def _reward(self, cd, cl):
        """cylinder_env_base.py:769, jet_cylinder_env_3d.py:436, 470-472"""
        return self.cd_ref - cd - self.lift_penalty * torch.abs(cl)
