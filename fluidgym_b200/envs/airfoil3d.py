"""Batched ``Airfoil3D`` environment (``envs/airfoil/airfoil_env_3d.py`` + ``airfoil_env_base.py`` with ``ndims = 3``): the 6-block
airfoil grid extruded over 96 periodic z planes (span 1.4), ``n_agents`` groups of three suction-side jets lined up along the span.

STATUS: pinned on a B200 to the unmodified reference's Airfoil3D at the reduced spanwise resolution res_z = 8 -- one ``env.step`` from
the reference's own reset state (56 substeps: plane velocities 8e-4, drag 1e-3, lift 1.3e-2, observations 5e-4; ``tests/golden/
airfoil3d_env.npz``) and the reverse-mode gradients through it (state vjp 1e-4, reward gradients 6 - 8 % with the reference's capped
solves; ``tests/golden/airfoil3d_grad.npz``), both in ``tests/test_gpu_extruded.py``.  What it is assembled from is pinned separately:
the extruded solver path and the spanwise
machinery of ``envs/cylinder3d.py`` (reference trace / ``env.step`` of CylinderJet3D through the kernels' cell code on the CPU), the
2-D airfoil tables -- grid, jet slots and profiles, wall ring, sensor positions, airfoil mask -- of ``envs/airfoil.py`` (GPU parity
with the reference's Airfoil2D), and the extruded cell code on this very plane mesh (``tests/test_extruded_host.py``).  Host logic
(action -> jet profiles per plane, flux balance, sensor layout, rewards, multi-agent interface) is exercised on the CPU with the
solver calls stubbed out, and sensor layout / airfoil mask / action mapping / reward mix equal the reference's own pure-torch methods
run from the installed reference on stub objects (``tests/test_airfoil3d_cpu.py``).  One environment is 46 806 x 96 = 4.5 M cells.
"""
from __future__ import annotations

import numpy as np
import torch

from ..sensors import sensor_tables_extruded
from .airfoil import Airfoil2DEnv, polygon_mask
from .airfoil_domain import BOT, FRONT, TAIL_LOWER, TAIL_UPPER, TOP, airfoil_polyline, make_airfoil_domain
from .common import build_wall_tables
from .cylinder3d import SpanwiseExtrudedEnv

AIRFOIL_3D_DEFAULT_CONFIG = {
    "n_agents": 4, "reynolds_number": 3e3, "dt": 0.05, "adaptive_cfl": 0.8, "step_length": 0.25, "episode_length": 200,
    "attack_angle_deg": 10.0, "local_obs_window": 1, "use_marl": False, "local_reward_weight": 0.5, "local_2d_obs": False,
}


class Airfoil3DEnv(SpanwiseExtrudedEnv):
    H, L, D, U_mean, airfoil_length = 1.4, 4.5, 1.4, 0.3, 1.0
    render_fill_steps = 128
    res_z = 96                                                          # airfoil_env_base.py:69
    n_jets = 3                                                          # jets per agent (airfoil_env_base.py:68)
    action_smoothing_alpha = 0.1
    bc_tol = 1e-5                                                       # update_advective_boundaries without an explicit tolerance (:244-249)
    metrics = ["drag", "lift"]
    reference_values = {"cl_cd_ref": ("lift", "mean", "drag", "mean")}

    def __init__(self, n_envs: int = 1, n_agents=4, reynolds_number=3e3, dt=0.05, adaptive_cfl=0.8, step_length=0.25, episode_length=200,
                 attack_angle_deg=10.0, local_obs_window=1, use_marl=False, local_reward_weight=0.5, local_2d_obs=False, init_from_2d=False,
                 device="cuda:0", cl_cd_ref=0.0, randomize_initial_state=False, enable_actions=True, load_initial_domain=False,
                 initial_domains_path=None, compiled=None, solver_cls=None, res_z=None, differentiable=False, per_env_substeps: bool = False):
        self.differentiable = bool(differentiable)
        self.per_env_substeps = bool(per_env_substeps)       # reverse mode of the extruded substep (SpanwiseExtrudedEnv._advance_differentiable)
        if res_z is not None:
            self.res_z = int(res_z)                                     # tests only: the reference's value is fixed
        if n_agents < 1 or self.res_z % n_agents != 0:
            raise ValueError("n_agents must be a positive integer that evenly dividescircle_resolution_angular.")
        if local_2d_obs and not use_marl:
            raise ValueError("Local 2D observations are only supported in multi-agent mode.")
        if attack_angle_deg < 0.0 or attack_angle_deg > 20.0:
            raise ValueError("Attack angle must be between 0 and 20 degrees.")
        self.load_domain_on_reset = bool(load_initial_domain)
        self.init_from_2d, self.initial_domains_path = bool(init_from_2d), initial_domains_path
        self.n_envs, self.n_span = int(n_envs), int(n_agents)
        self.reynolds_number, self.attack_angle_deg = float(reynolds_number), float(attack_angle_deg)
        self.dt, self.cfl = float(dt), float(adaptive_cfl)
        self.step_length, self.episode_length = float(step_length), int(episode_length)
        self.cl_cd_ref = float(cl_cd_ref)
        self.use_marl, self.local_reward_weight, self.local_2d_obs = bool(use_marl), local_reward_weight, bool(local_2d_obs)
        self.local_obs_window = 1 if local_2d_obs else int(local_obs_window)
        self.n_sensors_per_agent = 1                                    # airfoil_env_3d.py:130
        self.randomize_initial_state, self.enable_actions = randomize_initial_state, enable_actions
        self.device = torch.device(device)
        if compiled is None:
            # finer outflow grid for the hard case in 3-D (airfoil_env_base.py:210-215)
            tail = 1.001 if self.reynolds_number >= 5000 else 1.01
            spec = make_airfoil_domain(reynolds_number, self.U_mean, self.airfoil_length, self.H, self.L, attack_angle_deg, tail_grow_mul=tail)
            cd = spec.prepare()
        else:
            spec, cd = compiled
        self.spec, self.cd = spec, cd
        self.nz = self.res_z
        self.hz = self.D / self.nz
        self.z_vertices = np.linspace(-self.H / 2, self.H / 2, self.nz + 1, dtype=np.float32)                 # grid.py:609-614
        self.nz_per_agent = self.nz // self.n_span
        if solver_cls is None:
            from ..extruded3d import ExtrudedPISO3D as solver_cls      # raises without a CUDA device: there is no CPU path
        # airfoil_env_base.py:262-283: advect_non_ortho_steps = 2, pressure_non_ortho_steps = 4, tolerances 1e-6 / 1e-8 in 3-D
        self.solver = solver_cls(cd, self.nz, self.hz, self.n_envs, device=device, corrector_steps=2, advect_non_ortho_steps=2,
                                 pressure_non_ortho_steps=4, advection_tol=1e-6, pressure_tol=1e-8, max_iter=5000)
        out_mask = np.zeros(cd.NB, dtype=np.int8)
        for blk in (TAIL_UPPER, TAIL_LOWER):
            o = cd.boff[blk, 1]
            out_mask[o:o + spec.blocks[blk].ny] = 1
        self.solver.setup_stepping(out_mask.astype(bool), (self.U_mean, 0.0))
        ring = [(FRONT, 1, False), (TOP, 2, False), (BOT, 3, True)]
        self._wall_t, self.wall = build_wall_tables(cd, spec, ring, self.device, 1.0 / (0.5 * self.U_mean ** 2 * self.airfoil_length))
        Airfoil2DEnv._setup_jets(self, out_mask)                        # jet slots, unit-flux profiles, free mask: the 2-D tables per plane
        self._free_jets = self.free_mask.bool()
        self._setup_sensors()
        B, dev = self.n_envs, self.device
        self.last_control = torch.zeros(B, self.n_span, self.n_jets, device=dev)
        self._zero_action = torch.zeros(B, self.n_span, self.n_jets, device=dev)
        self._bvel0 = torch.from_numpy(np.ascontiguousarray(cd.bvel0[:, :cd.NB])).to(dev)

    # ---- static tables ---------------------------------------------------------------------------------------------------
    @property
    def render_shape(self):
        return (600, 150, 150)                                          # airfoil_env_base.py:160-163

    def _to_voxels(self, xyz: torch.Tensor) -> torch.Tensor:
        """airfoil_env_base.py:570-585 (the z coordinate is scaled with render_shape[1], as in the reference)"""
        rs = self.render_shape
        c = xyz.clone()
        c[0] = (c[0] + 1.5) * (rs[0] / (self.L + 1.5))
        c[1] = (c[1] + self.H / 2) * (rs[1] / self.H)
        if c.shape[0] == 3:
            c[2] = (c[2] + self.D / 2) * (rs[1] / self.D)
        return torch.round(c).to(torch.int64)

    def _setup_sensors(self):
        """airfoil_env_3d.py:303-344: the 2-D sensor positions repeated at n_sensors_z span positions, z-major; (x, y) columns that
        touch the airfoil mask are dropped."""
        rs = self.render_shape
        xy = Airfoil2DEnv.sensor_locations_physical(self)
        nsz, n_xy = self.n_sensors_z, xy.shape[1]
        sz = torch.linspace(-self.H / 2, self.H / 2, nsz + 1)[:-1] + self.H / (2 * nsz)
        pc = torch.stack([xy[0].unsqueeze(0).expand(nsz, -1).T, xy[1].unsqueeze(0).expand(nsz, -1).T, sz.unsqueeze(1).expand(-1, n_xy).T])
        gc = self._to_voxels(pc.reshape(3, -1))
        gc = torch.stack([gc[c].reshape(-1, nsz).T for c in range(3)])                     # [3, nsz, n_xy]
        body = Airfoil2DEnv._to_pixels(self, airfoil_polyline(self.attack_angle_deg)).numpy()
        self.airfoil_mask = polygon_mask(body.T, rs[0], rs[1])
        keep = [i for i in range(n_xy) if not self.airfoil_mask[gc[1, :, i].numpy(), gc[0, :, i].numpy()].any()]
        gc = gc[:, :, keep]
        self.n_sensors_xy = len(keep)
        self.sensor_px = gc.flatten(start_dim=1).numpy()                                   # z-major
        idx, w = sensor_tables_extruded([b.vertex for b in self.spec.blocks], self.z_vertices, rs, self.sensor_px, fill_max_steps=128)
        self.sens_idx = torch.from_numpy(idx.astype(np.int64)).to(self.device)
        self.sens_w = torch.from_numpy(w).to(self.device)

    # ---- reference-shaped API --------------------------------------------------------------------------------------------
    @property
    def n_agents(self):
        return self.n_span                                              # airfoil_env_3d.py:277-279 (also without use_marl)

    @property
    def id(self):
        return f"Airfoil3D_Re{int(self.reynolds_number)}"

    @property
    def initial_domain_id(self):
        return f"airfoil_3D_Re{int(self.reynolds_number)}"

    @property
    def action_space(self):
        from .. import spaces
        return spaces.Box(-1.0, 1.0, shape=(self.n_jets,) if self.use_marl else (self.n_span, self.n_jets))

    def _initial_velocity(self):
        """``init_from_2d`` (airfoil_env_3d.py:524-593): one random 2-D initial domain of the training split (every
        environment of the batch draws its own index here), its velocity copied into every plane with a zero spanwise component;
        pressure and boundary values stay those of the fresh 3-D domain.  A file whose grid differs is skipped, as in the reference."""
        if not self.init_from_2d:
            return
        import os
        from ..domain_io import load_domain
        from .common import N_INITIAL_DOMAINS, default_initial_domains_path
        root = self.initial_domains_path or default_initial_domains_path()
        dom_id = self.initial_domain_id.replace("airfoil_3D", "airfoil_2D").replace("Re10000", "Re3000")
        u4 = self.solver.u.view(self.n_envs, 3, self.nz, self.solver.N2)
        for e in range(self.n_envs):
            idx = int(self._np_rng.integers(0, N_INITIAL_DOMAINS))
            path = os.path.join(root, dom_id, str(idx), "train")
            if not os.path.exists(path + ".json"):
                raise FileNotFoundError(f"2D initial domain not found on disk but attempting to init from 2D: {path}")
            spec2, st = load_domain(path)
            if [b.vertex.shape for b in spec2.blocks] != [b.vertex.shape for b in self.spec.blocks]:
                continue                                                # "Using 3D initial domain as fallback." (:549-556)
            u4[e, :2] = torch.from_numpy(np.ascontiguousarray(st["u"])).to(self.device)[:, None, :]
            u4[e, 2] = 0.0

    def _randomize_domain(self):
        """airfoil_env_base.py:302-339"""
        max_n = int(0.05 * self.episode_length)
        n_steps = int(self._np_rng.integers(int(0.5 * max_n), max_n)) + 1
        s = self.solver
        s.u += torch.randn(s.u.shape, device=self.device, generator=self._torch_rng) * 0.01
        s.p += torch.randn(s.p.shape, device=self.device, generator=self._torch_rng) * 0.01
        for _ in range(n_steps):
            s.single_step(self.dt, self.cfl, bc_tol=self.bc_tol)

    def _apply_action(self, control: torch.Tensor):
        """airfoil_env_3d.py:383-407 + airfoil_env_base.py:709-718: per agent zero-mean amplitudes with max |.| <= 1, every agent
        drives its nz_per_agent planes with the three unit-flux jet profiles (no spanwise component); then outflow + airfoil top wall
        are rescaled for a zero net boundary flux."""
        s = self.solver
        v = control - control.mean(dim=2, keepdim=True)                                    # [B, n_agents, n_jets]
        mx = v.abs().max(dim=2, keepdim=True).values
        v = torch.where(mx > 1.0, v / mx, v)
        per_plane = v.repeat_interleave(self.nz_per_agent, dim=1)                          # [B, nz, n_jets]
        if getattr(s, "apply_jets", None) and s.apply_jets(per_plane, self.jet_base, self.jet_faces, self._free_jets, 1e-5):
            return                                                                         # kernel path (default; FGB_X3_HOOKS=torch: torch expressions)
        prof = torch.einsum("bkj,jcx->bckx", per_plane, self.jet_base)                     # [B, 2, nz, n_top]
        jf = self.jet_faces.long()
        s.bvel[:, :2, :, jf] = prof
        s.bvel[:, 2, :, jf] = 0.0
        s.balance_fluxes(self._free_jets, 1e-5)

    def _jet_profiles(self, control):
        """functional form of _apply_action for the differentiable mode"""
        v = control - control.mean(dim=2, keepdim=True)
        mx = v.abs().max(dim=2, keepdim=True).values
        v = torch.where(mx > 1.0, v / mx, v)
        per_plane = v.repeat_interleave(self.nz_per_agent, dim=1)                          # [B, nz, n_jets]
        return torch.einsum("bkj,jcx->bckx", per_plane, self.jet_base), 1e-5

    def _reward(self, cd, cl):
        """airfoil_env_3d.py:420, 450"""
        return cl / cd - self.cl_cd_ref
