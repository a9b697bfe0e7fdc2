"""Pieces shared by the environment families: the episode lifecycle, initial domains, domain statistics, the linear-solve
watch and rendering.  For the bluff-body environments (cylinder, airfoil) also the wall-force tables and the differentiable
rollout in which the PISO substep is one autograd node backed by the CUDA adjoint (``fluidgym_b200.autograd``)
while the few boundary / reward formulas around it are tiny torch expressions over the same static tables the
kernels use -- so gradients flow from the reward to the action, the cell velocities and the boundary values as in
the reference, where those parts are torch code as well (SIM.py:188-393, forces.py:193-275)."""
from __future__ import annotations

from typing import NamedTuple

import numpy as np
import torch

from .. import native
from ..sensors import cell_centres
from ..solver import _ptr, cfl_substeps, cfl_substeps_per_env


def build_wall_tables(cd, spec, ring, device, scale: float):
    """Wall-adjacent cells of a body described by ``ring = [(block, face, flip), ...]`` walked as one closed loop
    (forces.py:12-107; cylinder_env_base.py:548-655; airfoil_env_base.py:341-441).  Returns the tensor dict and
    the ``fgb_wall`` descriptor for ``fgb_wall_forces``."""
    vc_list, cc_list, cells, bfaces = [], [], [], []
    for k, (bi, f, flip) in enumerate(ring):
        b = spec.blocks[bi]
        v = torch.from_numpy(b.vertex)
        cc = torch.from_numpy(cell_centres(b.vertex))
        if (f >> 1) == 0:
            col = -1 if (f & 1) else 0
            bc, ce = v[:, :, col], cc[:, :, col]
            idx = [cd.gidx(bi, [b.nx - 1 if (f & 1) else 0, y]) for y in range(b.ny)]
        else:
            row = -1 if (f & 1) else 0
            bc, ce = v[:, row, :], cc[:, row, :]
            idx = [cd.gidx(bi, [x, b.ny - 1 if (f & 1) else 0]) for x in range(b.nx)]
        bf = [cd.boff[bi, f] + i for i in range(len(idx))]
        if flip:
            bc, ce = torch.flip(bc, dims=[-1]), torch.flip(ce, dims=[-1])
            idx, bf = idx[::-1], bf[::-1]
        if k != len(ring) - 1:
            bc = bc[..., :-1]          # shared vertex with the next block
        vc_list.append(bc)
        cc_list.append(ce)
        cells += idx
        bfaces += bf
    vc = torch.cat(vc_list, dim=-1)
    centers = torch.cat(cc_list, dim=-1)
    left = torch.roll(centers, shifts=-1, dims=-1)
    right = torch.roll(centers, shifts=1, dims=-1)
    tlen = torch.sqrt(torch.sum((left - right) ** 2, dim=0))
    v0, v1 = vc[:, :-1], vc[:, 1:]
    e = v1 - v0
    eps = 1e-20
    t = e / (torch.linalg.norm(e, dim=0, keepdim=True) + eps)
    n = torch.stack([t[1], -t[0]], dim=0)
    m = 0.5 * (v0 + v1)
    d = torch.clamp(((centers - m) * n).sum(dim=0).abs(), min=eps)
    n = n * -1
    flen = torch.sqrt((vc[0, 1:] - vc[0, :-1]) ** 2 + (vc[1, 1:] - vc[1, :-1]) ** 2)
    tab = dict(cell=torch.tensor(cells, dtype=torch.int32, device=device), bface=torch.tensor(bfaces, dtype=torch.int32, device=device),
               normal=n.contiguous().float().to(device), dist=d.float().to(device), tlen=tlen.float().to(device),
               flen=flen.float().to(device))
    w = native.Wall()
    w.n_wall = len(cells)
    for k2 in ("cell", "bface", "normal", "dist", "tlen", "flen"):
        setattr(w, k2, tab[k2].data_ptr())
    w.scale = float(scale)
    return tab, w


class EpisodeLifecycle:
    """Mixin: the episode lifecycle of the reference's ``FluidEnv`` (fluid_env.py) with its error strings, shared by every
    family: seeding, action sampling, the checks at the start of ``reset`` and ``step``, the end of a step and ``detach``.
    Needs ``device, dt, step_length, episode_length, _zero_action`` and ``_watch_linear_solves`` (LinearSolveWatch)."""

    _reset_called = False
    _seed = None
    _n_steps = 0
    last_substeps = 0               # substep rounds launched by the last step (every environment's count in plain mode)
    last_substeps_per_env = None    # int64 [B]: each environment's substeps in the last per-environment differentiable step
    per_env_substeps = False        # differentiable mode: every environment follows its own CFL plan (see _substep_rounds)
    _dstate = None          # differentiable mode: the state tensors carried with their autograd history

    @property
    def n_sim_steps(self):
        return max(1, int(self.step_length / self.dt))

    def seed(self, seed: int):
        self._seed = seed
        self._np_rng = np.random.default_rng(seed)
        self._torch_rng = torch.Generator(device=self.device).manual_seed(seed)

    def sample_action(self):
        if self._seed is None:
            raise RuntimeError("Environment must be seeded before sampling actions")
        return torch.rand(self._zero_action.shape, device=self.device, generator=self._torch_rng) * 2 - 1

    def _begin_reset(self, seed):
        """First thing of every ``reset``: seed, or check that ``seed()`` was called."""
        if seed is None:
            if self._seed is None:
                raise ValueError("Seed must be provided either during reset or by calling seed().")
        else:
            self.seed(seed)

    def _begin_step(self, action) -> torch.Tensor:
        """First thing of every ``step``: the checks of the reference, returns the action as float32 on the device."""
        if not self._reset_called:
            raise RuntimeError("Environment must be reset before stepping. Call 'reset()' before'step()'.")
        action = torch.as_tensor(action, dtype=torch.float32, device=self.device)
        if action.shape != self._zero_action.shape:
            raise ValueError(f"Action shape {action.shape} does not match expected shape {self._zero_action.shape}.")
        if self._n_steps >= self.episode_length:
            raise RuntimeError("Episode has already terminated. Call 'reset()' first.")
        return action

    def _end_step(self) -> bool:
        """Counts the step, watches its linear solves; returns ``truncated``."""
        self._n_steps += 1
        self._watch_linear_solves()
        return self._n_steps >= self.episode_length

    def _copy_state(self, dst: torch.Tensor, src):
        """``set_state``: ``src`` is one environment's field (copied into every environment) or the whole batch's."""
        src = torch.as_tensor(src, dtype=torch.float32, device=self.device)
        dst.copy_(src if src.dim() == dst.dim() else src.unsqueeze(0).expand_as(dst))

    def detach(self):
        """fluid_env.py ``detach()``: cut the autograd graph at the current state."""
        if self._dstate is not None:
            self._dstate = tuple(t.detach() for t in self._dstate)

    def _begin_substep_count(self):
        """start of a differentiable step: ``last_substeps_per_env`` counts from zero with per-environment plans, else it is None"""
        self.last_substeps_per_env = torch.zeros(self.n_envs, dtype=torch.int64, device=self.device) if self.per_env_substeps else None

    def _substep_rounds(self, max_velocity_env):
        """The substep rounds of one solver step of a differentiable rollout with ``per_env_substeps``: every environment follows its own
        adaptive CFL plan (``solver.cfl_substeps_per_env``, the plan plain mode uses), so an environment of a batch takes the substeps it
        would take alone.  ``max_velocity_env()`` -> float32 [B] of the current state.  Yields ``(dt [B], active [B])``; environments with
        ``active == 0`` have used up their time and must pass through the round unchanged."""
        s = self.solver
        for dtv, act in cfl_substeps_per_env(s.lib, self.n_envs, self.dt, self.cfl, max_velocity_env, self.device, s.stream):
            self.last_substeps_per_env += act
            yield dtv, act


class DifferentiableRollout:
    """Mixin of the 2-D bluff-body families (cylinder, airfoil): ``env.step`` and the differentiable rollout.  Needs ``solver,
    cd, device, lib, n_envs, dt, cfl, char_vel, wall, _wall_t, _dstate`` and, for ``step``, ``_advance(action)`` /
    ``_advance_differentiable(action)`` (-> the [B, 2] drag / lift coefficients summed over the solver steps), ``_get_obs()`` and
    ``_reward(cd, cl)``."""

    def step(self, action):
        action = self._begin_step(action)
        acc = self._advance_differentiable(action) if self.differentiable else self._advance(action)
        obs = self._get_obs()
        mean = acc / self.n_sim_steps
        cd, cl = mean[:, 0], mean[:, 1]
        reward = self._reward(cd, cl)
        truncated = self._end_step()
        return obs, reward, False, truncated, {"drag": cd.detach(), "lift": cl.detach()}

    def _diff_tables(self):
        if getattr(self, "_dt_tab", None) is None:
            cd, dev = self.cd, self.device
            NB = cd.NB
            out = np.nonzero(np.asarray(self.solver._tab["b_out"].cpu()))[0]
            face = np.asarray(cd.b_face[:NB]).astype(np.int64)
            ax = face >> 1
            bminv = np.asarray(cd.b_minv)[:, :NB]
            bdet = np.asarray(cd.b_det)[:NB]
            j = np.arange(NB)
            sign = np.where(face & 1, 1.0, -1.0)
            fw = np.stack([bdet * bminv[2 * ax, j] * sign, bdet * bminv[2 * ax + 1, j] * sign]).astype(np.float32)   # signed flux weights
            adv = bminv[2 * ax[out], out] * self.char_vel[0] + bminv[2 * ax[out] + 1, out] * self.char_vel[1]
            is_out = np.zeros(NB, dtype=bool)
            is_out[out] = True

            def tt(a, dt=torch.float32):
                return torch.as_tensor(np.ascontiguousarray(a), dtype=dt, device=dev)
            self._dt_tab = dict(out=tt(out, torch.int64), out_cell=tt(np.asarray(cd.b_cell)[out], torch.int64), adv=tt(adv),
                                fw=tt(fw), is_out=tt(is_out, torch.bool))
        return self._dt_tab

    def _balance_torch(self, bv, free, bc_tol=1e-5):
        """balance_boundary_fluxes (SIM.py:188-224): ``free`` is a bool mask [NB] of the faces that are rescaled.  As in the
        reference the flux scale is computed under ``no_grad`` (SIM.py:191-211) and applied as a constant factor outside of it
        (:212-224): gradients flow through the rescaled boundary values, not through the scale."""
        tb = self._diff_tables()
        with torch.no_grad():
            fl = (bv * tb["fw"]).sum(dim=1)
            fx = (fl * (~free)).sum(dim=1)
            vr = (fl * free).sum(dim=1)
            need = ~((fx + vr).abs() <= bc_tol * 0.01)
            sc = torch.where(need, -fx / vr, torch.ones_like(fx))
            scale = torch.where(free[None, :], sc[:, None], torch.ones_like(fl))
        return bv * scale[:, None, :]

    def _outflow_torch(self, u, bv, dt, bc_tol=1e-5):
        """k_plan_substep's boundary part (SIM.py:188-224, 282-393); ``dt`` a float or a per-environment [B, 1, 1] tensor.  The reference runs update_advective_boundaries entirely
        under ``torch.no_grad()`` (SIM.py:232), including the setVelocity of the relaxed and rescaled outflow values: the outflow
        faces carry no gradient (neither to the adjacent cells nor to their previous values), all other faces keep theirs."""
        tb = self._diff_tables()
        with torch.no_grad():
            w = 1.0 - 1.0 / (1.0 + 2.0 * dt * tb["adv"])
            bo = bv[:, :, tb["out"]]
            bo = bo - w * (bo - u[:, :, tb["out_cell"]])
            bvn = self._balance_torch(bv.index_copy(2, tb["out"], bo), tb["is_out"], bc_tol)
            bo = bvn[:, :, tb["out"]]
        return bv.index_copy(2, tb["out"], bo)

    def _forces_torch(self, u, p, bv):
        """k_wall_forces (forces.py:193-275) as differentiable torch ops -> [B,2] (drag, lift coefficients)."""
        w = self._wall_t
        c, j = w["cell"].long(), w["bface"].long()
        il, ir = torch.roll(c, -1), torch.roll(c, 1)
        n = w["normal"]
        nx, ny = n[0], n[1]
        tx, ty = ny, -nx
        visc = float(self.cd.visc)
        dn = (u[:, :, c] - bv[:, :, j]) / w["dist"]
        dt_ = (u[:, :, ir] - u[:, :, il]) / (2.0 * w["tlen"])
        du_dx, du_dy = dn[:, 0] * nx + dt_[:, 0] * tx, dn[:, 0] * ny + dt_[:, 0] * ty
        dv_dx, dv_dy = dn[:, 1] * nx + dt_[:, 1] * tx, dn[:, 1] * ny + dt_[:, 1] * ty
        pc = p[:, c]
        sxx, syy = 2.0 * visc * du_dx - pc, 2.0 * visc * dv_dy - pc
        sxy = visc * (du_dy + dv_dx)
        fxx = ((sxx * nx + sxy * ny) * w["flen"]).sum(dim=1)
        fyy = ((sxy * nx + syy * ny) * w["flen"]).sum(dim=1)
        return torch.stack([fxx, fyy], dim=1) * self.wall.scale

    def _single_step_differentiable(self, u, p, bv):
        """Simulation.single_step with the adaptive CFL plan of SIM.py:2004-2031; the plan itself is not
        differentiated (the reference computes it from detached maxima as well).  One common substep size is
        used for the batch (the most restrictive environment decides), or with ``per_env_substeps`` every
        environment's own plan (environments that are done keep their state and boundary values)."""
        from ..autograd import piso_substep
        s = self.solver
        mvb = torch.empty(self.n_envs, device=self.device)
        tol = getattr(self, "bc_tol", 1e-5)

        def max_velocity_env():
            native.check(self.lib.fgb_max_velocity(s.handle, _ptr(u.detach().contiguous()), _ptr(bv.detach().contiguous()), _ptr(mvb),
                                                   s.stream), "fgb_max_velocity")
            return mvb
        nsub = 0
        if self.per_env_substeps:
            for dtv, act in self._substep_rounds(max_velocity_env):
                bv = torch.where(act.bool()[:, None, None], self._outflow_torch(u, bv, dtv[:, None, None], tol), bv)
                u, p = piso_substep(s, u, p, bv, dtv, active=act)
                nsub += 1
            return u, p, bv, nsub
        for ts in cfl_substeps(self.dt, self.cfl, lambda: float(max_velocity_env().max())):
            bv = self._outflow_torch(u, bv, ts, tol)
            u, p = piso_substep(s, u, p, bv, ts)
            nsub += 1
        return u, p, bv, nsub


_SIGNED_FIELDS = ("vorticity", "velocity_x", "velocity_y", "velocity_z", "pressure", "q_criterion")


class Renderable:
    """Mixin: batched images of the flow (the reference's ``render``, fluid_env.py:577-606, for every environment of the batch).

    ``render_field`` resamples one field onto the family's image grid with the static render map of ``fluidgym_b200.render``
    (``fgb_render_gather``); ``render`` colours it (``fgb_render_colour``): signed fields with the diverging map over a range
    symmetric about zero, magnitudes and temperature with the sequential one, each environment over its own range unless
    ``vmin`` / ``vmax`` fix one for the batch.  Both run on the solver's stream under ``no_grad`` and read the solver state
    only.  The map is built on the first call for a plane and kept by the instance.  ``vorticity`` is the physical omega
    = dv/dx - du/dy (the reference's 2-D renderer shows -omega).

    A family sets ``render_fields`` (the first is the default) and ``_build_render_map(plane)``; 3-D families also
    ``_render_planes()`` -> (number of planes, default plane).  Needs ``solver`` (u, p, optionally T / vorticity() /
    q_criterion()), ``n_envs``, ``device``."""

    render_fields: tuple = ()

    def _render_planes(self):
        return None

    def _build_render_map(self, plane):
        raise NotImplementedError

    def _render_map(self, plane):
        planes = self._render_planes()
        if planes is None:
            if plane is not None:
                raise ValueError(f"{type(self).__name__} renders its 2-D domain: plane must be None, got {plane!r}")
        else:
            n, default = planes
            plane = default if plane is None else plane
            if not isinstance(plane, (int, np.integer)) or not 0 <= plane < n:
                raise ValueError(f"plane {plane!r} out of range: valid planes of {type(self).__name__} are 0 .. {n - 1}")
            plane = int(plane)
        cache = self.__dict__.setdefault("_render_maps", {})
        if plane not in cache:
            m = self._build_render_map(plane)
            cache[plane] = (tuple(torch.from_numpy(a).to(self.device) for a in (m.rowptr, m.col, m.w)), m.shape)
        return cache[plane]

    def _render_source(self, field):
        """-> ([B, C, N] strided view of the field, fgb_render_gather mode)"""
        from ..render import IDENTITY, NORM
        if field is None:
            field = self.render_fields[0]
        if field not in self.render_fields:
            raise ValueError(f"unknown render field {field!r}: {type(self).__name__} renders {self.render_fields}")
        s = self.solver
        if field == "velocity_magnitude":
            return s.u, NORM
        if field.startswith("velocity_"):
            c = "xyz".index(field[-1])
            return s.u[:, c:c + 1], IDENTITY
        src = {"pressure": lambda: s.p, "temperature": lambda: s.T, "vorticity": lambda: s.vorticity(),
               "q_criterion": lambda: s.q_criterion()}[field]()
        return src.reshape(self.n_envs, 1, -1), IDENTITY

    def _render_gather(self, field, plane, with_range: bool):
        with torch.no_grad():
            src, mode = self._render_source(field)
            (rowptr, col, w), (H, W) = self._render_map(plane)
            B, Cn, N = src.shape
            if src.stride(2) != 1:
                src = src.contiguous()
            img = torch.empty(B, H, W, device=self.device)
            rng = torch.empty(B, 2, dtype=torch.int32, device=self.device) if with_range else None
            s = self.solver
            native.check(s.lib.fgb_render_gather(_ptr(src), B, Cn, N, src.stride(1), src.stride(0), mode, _ptr(rowptr), _ptr(col), _ptr(w),
                                                 H * W, _ptr(img), _ptr(rng), s.stream), "fgb_render_gather")
        return img, rng

    def render_field(self, field=None, *, plane=None) -> torch.Tensor:
        """float32 [B, H, W] on the environment's device: ``field`` (default ``render_fields[0]``) resampled onto the image grid;
        3-D families show the slice ``plane``."""
        return self._render_gather(field, plane, False)[0]

    def render(self, field=None, *, plane=None, vmin=None, vmax=None) -> torch.Tensor:
        """uint8 [B, H, W, 3] on the environment's device: ``render_field`` coloured (see the class documentation)."""
        from ..render import DIVERGING, SEQUENTIAL
        if (vmin is None) != (vmax is None):
            raise ValueError("render: give both vmin and vmax (a fixed range for the batch) or neither (each environment's own range)")
        fixed = vmin is not None
        img, rng = self._render_gather(field, plane, not fixed)
        signed = (field or self.render_fields[0]) in _SIGNED_FIELDS
        luts = self.__dict__.setdefault("_render_luts", {})
        if signed not in luts:
            luts[signed] = torch.from_numpy(DIVERGING if signed else SEQUENTIAL).to(self.device)
        B, H, W = img.shape
        rgb = torch.empty(B, H, W, 3, dtype=torch.uint8, device=self.device)
        s = self.solver
        native.check(s.lib.fgb_render_colour(_ptr(img), B, H * W, _ptr(rng), float(vmin) if fixed else 0.0, float(vmax) if fixed else 0.0,
                                             int(signed and not fixed), _ptr(luts[signed]), _ptr(rgb), s.stream), "fgb_render_colour")
        return rgb


N_INITIAL_DOMAINS = 10      # envs/fluid_env.py:58


def default_initial_domains_path() -> str:
    """``fluidgym.config.initial_domains_path`` (config.py:137-144: platformdirs user data dir / initial_domains); override
    with the environment variable FLUIDGYM_INITIAL_DOMAINS."""
    import os
    return os.environ.get("FLUIDGYM_INITIAL_DOMAINS", os.path.join(os.path.expanduser("~"), ".local", "share", "FluidGym", "initial_domains"))


class Stats(NamedTuple):
    """envs/fluid_env.py:33-44"""
    mean: float
    min: float
    max: float
    p5: float
    p25: float
    p50: float
    p75: float
    p95: float


STATISTICS_FILENAME = "domain_statistics.json"        # util/data_utils.py:19


class DomainStatistics:
    """Mixin: ``load_domain_statistics=True`` of the reference (envs/fluid_env.py:234-238, 1205-1221; util/data_utils.py:82-98):
    ``<initial_domains_path>/<initial_domain_id>/domain_statistics.json`` holds the Stats of the velocity magnitude, the pressure
    and every metric of the uncontrolled flow; the reward normalisers are read from it (``reference_values``).  Needs
    ``initial_domain_id`` and ``metrics``; ``initial_domains_path`` optional."""

    metrics_stats: dict = {}
    velocity_stats = None
    pressure_stats = None
    # attribute <- (metric, field) or (metric, field, metric2, field2) for a ratio; per family, as in the reference:
    # cylinder_env_base.py:271-275, rbc_env_base.py:407-416, airfoil_env_base.py:166-172, tcf_env.py:556-562, 1131-1137
    reference_values: dict = {}

    def domain_statistics_file(self) -> str:
        import os
        root = getattr(self, "initial_domains_path", None) or default_initial_domains_path()
        return os.path.join(root, self.initial_domain_id, STATISTICS_FILENAME)

    def load_domain_statistics(self) -> dict:
        import json
        with open(self.domain_statistics_file()) as f:
            stats = json.load(f)
        self.velocity_stats = Stats(**stats["velocity_magnitude"])
        self.pressure_stats = Stats(**stats["pressure"])
        self.metrics_stats = {key: Stats(**stats[key]) for key in self.metrics}
        for attr, rule in self.reference_values.items():
            if all(m in self.metrics_stats for m in rule[0::2]):
                v = getattr(self.metrics_stats[rule[0]], rule[1])
                if len(rule) == 4:
                    v = v / getattr(self.metrics_stats[rule[2]], rule[3])
                setattr(self, attr, float(v))
        return stats

    def save_domain_statistics(self, statistics: dict) -> str:
        """fluid_env.py:1191-1203"""
        import json
        import os
        path = self.domain_statistics_file()
        os.makedirs(os.path.dirname(path), exist_ok=True)
        with open(path, "w") as f:
            json.dump(statistics, f, indent=4)
        return path


class LinsolveError(RuntimeError):
    """A linear solve reported a non-finite residual (PISOtorch_diff.py: LinsolveError)."""


class LinearSolveWatch:
    """Error behaviour of ``_check_solver_return_infos`` (PISOtorch_diff.py:266-301): a non-finite residual of any
    linear solve raises ``LinsolveError``.  (Its fp64 / preconditioned retries, :418-476, fire on the same condition
    only, because the environments solve with return_best_result; they are not built -- DESIGN.md §8.)

    The reference inspects the solver infos on the host after every solve.  Here the final residuals of the last
    substep stay in the solver's ``resid`` table [B, 8]; every ``env.step`` ends with a non-blocking copy of that table
    into pinned memory and the table of step k is examined when step k+1 ends (or on ``check_linear_solves()``), when
    the copy has long landed -- no stall.  A state that went non-finite stays so, hence the one-step delay loses nothing
    but promptness.  ``check_solves = False`` switches the watch off.  Needs ``solver`` with ``buffer("resid")``."""

    check_solves = True
    _ls_pending = False

    def _watch_linear_solves(self):
        if not self.check_solves or not hasattr(self.solver, "buffer"):    # (host stand-ins of the CPU tests keep no residual table)
            return
        self.check_linear_solves()
        resid = self.solver.buffer("resid")
        if getattr(self, "_ls_host", None) is None or self._ls_host.shape != resid.shape:
            self._ls_host = torch.empty(resid.shape, dtype=resid.dtype, pin_memory=resid.is_cuda)
            self._ls_event = torch.cuda.Event() if resid.is_cuda else None
        self._ls_host.copy_(resid, non_blocking=True)
        if self._ls_event is not None:
            self._ls_event.record()
        self._ls_pending, self._ls_step = True, getattr(self, "_n_steps", 0)

    def check_linear_solves(self):
        """Raise LinsolveError if the last watched step left a non-finite residual; returns the residual table otherwise."""
        if not self._ls_pending:
            return None
        if self._ls_event is not None:
            self._ls_event.synchronize()
        self._ls_pending = False
        table = self._ls_host.numpy()
        bad = ~np.isfinite(table)
        if bad.any():
            envs = np.nonzero(bad.any(axis=-1))[0].tolist()
            raise LinsolveError("Linear solve reported non-finite residual in env.step %d for environment(s) %s of %d "
                                "(residual slots %s)." % (self._ls_step, envs[:16], table.shape[0],
                                                         np.nonzero(bad.any(axis=0))[0].tolist()))
        return table


class InitialDomains(LinearSolveWatch, DomainStatistics):
    """Mixin: the published initial-domain splits (``initial_domains/<initial_domain_id>/<idx>/<mode>.{json,npz}``,
    envs/fluid_env.py:507-551, 1040-1112) for batched environments.  Files are read once into a device-resident pool; every
    environment of the batch draws its own index on ``reset`` (the reference draws one per process).
    Needs ``spec, cd, solver, device, n_envs, initial_domain_id``."""

    mode = "train"

    def train(self):
        self.mode = "train"

    def val(self):
        self.mode = "val"

    def test(self):
        self.mode = "test"

    def initial_domain_file(self, idx: int, mode: str | None = None) -> str:
        import os
        root = getattr(self, "initial_domains_path", None) or default_initial_domains_path()
        return os.path.join(root, self.initial_domain_id, str(idx), mode or self.mode)

    def _pool_entry(self, idx: int, mode: str):
        pool = self.__dict__.setdefault("_domain_pool", {})
        key = (mode, idx)
        if key not in pool:
            import os
            path = self.initial_domain_file(idx, mode)
            if not os.path.exists(path + ".json"):
                raise RuntimeError("Initial domain not found. Please ensure it was downloaded.")
            st = self._read_domain_file(path)
            pool[key] = {k: torch.from_numpy(np.ascontiguousarray(v)).to(self.device) for k, v in st.items() if v is not None}
        return pool[key]

    def _read_domain_file(self, path: str) -> dict:
        """2-D multi-block domains (``self.spec``); the 3-D box environments override this (InitialDomains3D)."""
        from ..domain_io import load_domain
        spec, st = load_domain(path)
        if [b.vertex.shape for b in spec.blocks] != [b.vertex.shape for b in self.spec.blocks] or any(
                not np.array_equal(a.vertex, b.vertex) for a, b in zip(spec.blocks, self.spec.blocks)):
            raise ValueError(f"{path}: the stored grid is not the grid of this environment")
        return st

    def load_initial_domain(self, idx: int, mode: str | None = None, env_index=None):
        """fluid_env.py:1065-1086; ``env_index`` (int, list or None = all) selects which environments receive the state."""
        st = self._pool_entry(int(idx), mode or self.mode)
        s = self.solver
        sel = slice(None) if env_index is None else env_index
        s.u[sel] = st["u"]
        s.p[sel] = st["p"]
        s.bvel[sel] = st["bvel"]
        if "T" in st and getattr(s, "has_scalar", False):
            s.T[sel] = st["T"]
            s.sbval[sel] = st["sbval"]
        if getattr(self, "_dstate", None) is not None:
            self._dstate = None

    def save_initial_domain(self, idx: int, mode: str | None = None, env_index: int = 0):
        """fluid_env.py:1047-1063: writes environment ``env_index`` in the reference's format."""
        import os
        path = self.initial_domain_file(idx, mode)
        os.makedirs(os.path.dirname(path), exist_ok=True)
        s = self.solver
        st = dict(u=s.u[env_index].cpu().numpy(), p=s.p[env_index].cpu().numpy(), bvel=s.bvel[env_index].cpu().numpy())
        if getattr(s, "has_scalar", False):
            st.update(T=s.T[env_index].cpu().numpy(), sbval=s.sbval[env_index].cpu().numpy())
        self._write_domain_file(st, path)
        return path

    def _write_domain_file(self, st: dict, path: str):
        from ..domain_io import save_domain
        save_domain(self.spec, st, path)

    def _load_initial_domains_on_reset(self, randomize: bool):
        """_set_initial_state with load_initial_domain=True: index 0, or one random index per environment."""
        if randomize:
            idxs = [int(self._np_rng.integers(0, N_INITIAL_DOMAINS)) for _ in range(self.n_envs)]
        else:
            idxs = [0] * self.n_envs
        for idx in sorted(set(idxs)):
            self.load_initial_domain(idx, env_index=[e for e, i in enumerate(idxs) if i == idx])
        return idxs


class InitialDomains3D(InitialDomains):
    """The same for the single-block 3-D box environments (TCF, RBC3D): needs ``dom`` (Box3DDomain) instead of ``spec``."""

    def _read_domain_file(self, path: str) -> dict:
        from ..domain_io import load_box_domain
        d = load_box_domain(path)
        if d["vertex"].shape != self.dom.vertex.shape or not np.array_equal(d["vertex"], self.dom.vertex) or d["closed"] != self.dom.closed:
            raise ValueError(f"{path}: the stored grid is not the grid of this environment")
        st = d["state"]
        if st["bvel"].shape[1] == 0:
            st["bvel"] = np.zeros((3, 1), np.float32)
        return st

    def _write_domain_file(self, st: dict, path: str):
        from ..domain_io import save_box_domain
        s = self.solver
        st = dict(st, bvel=st["bvel"][:, :self.dom.NB])
        if "sbval" in st:
            st["sbval"] = st["sbval"][:self.dom.NB]
        save_box_domain(self.dom.vertex, self.dom.closed, self.dom.visc, st, path,
                        scalar_viscosity=getattr(s, "kappa", None) if getattr(s, "has_scalar", False) else None,
                        name=type(self).__name__)


class InitialDomainsExtruded(InitialDomains):
    """The same for the z-extruded multi-block environments (CylinderJet3D, Airfoil3D): needs ``spec`` (plane), ``nz``, ``z_vertices``."""

    def _read_domain_file(self, path: str) -> dict:
        from ..domain_io import load_extruded_domain
        spec, zv, st = load_extruded_domain(path)
        if [b.vertex.shape for b in spec.blocks] != [b.vertex.shape for b in self.spec.blocks] or any(
                not np.array_equal(a.vertex, b.vertex) for a, b in zip(spec.blocks, self.spec.blocks)) or zv.size != self.nz + 1 or \
                not np.allclose(zv, self.z_vertices, atol=1e-6):
            raise ValueError(f"{path}: the stored grid is not the grid of this environment")
        return dict(u=st["u"].reshape(3, -1), p=st["p"].reshape(-1), bvel=st["bvel"])

    def _write_domain_file(self, st: dict, path: str):
        from ..domain_io import save_extruded_domain
        N2 = self.solver.N2
        save_extruded_domain(self.spec, self.z_vertices, dict(u=st["u"].reshape(3, self.nz, N2), p=st["p"].reshape(self.nz, N2), bvel=st["bvel"]), path)
