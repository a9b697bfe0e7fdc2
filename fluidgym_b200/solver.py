"""Batched PISO solver: host-side mirror of ``fluidgym.simulation.Simulation`` for B environments.

Keeps the reference's vocabulary (``single_step``, ``make_divergence_free``, ``corrector_steps``,
``pressure_tol`` ...; FGSIM.py:125-280, SIM.py:489-1037) but advances a whole batch of environments
that share one geometry with the sm_100a kernels behind ``include/fluidgym_b200.h``.  torch is used
only to own device memory and streams.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np
import torch

from . import native
from .domain import CompiledDomain

_TABLE_FIELDS = ["nbr", "fl_comp", "minv", "det", "Cd", "Wp", "no_idx", "no_face", "no_gP", "no_gN", "no_wv",
                 "nob_idx", "nob_w", "b_minv", "b_det", "b_alpha", "b_cell", "b_face", "rev"]


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def cfl_substep(remaining: float, cfl: float, max_vel: float) -> float:
    """Size of the next substep of the adaptive CFL plan (SIM.py:2004-2031), in k_plan_substep's precision: the CFL-limited
    step cfl / max_vel is formed in float32, ``remaining`` stays float64 and is split into equal parts when it is longer."""
    if abs(max_vel) <= 1e-8:
        return remaining
    mts = np.float32(cfl) / np.float32(max_vel)
    return remaining if float(mts) >= remaining else remaining / float(np.ceil(np.float32(remaining) / mts))


def cfl_substeps(dt: float, cfl: float, max_velocity):
    """The substeps of one solver step of length ``dt``: yields each size rounded to float32 (what the substep kernels take).
    ``max_velocity()`` returns the maximum velocity of the batch as a Python float and is called before every substep, so one
    common size serves the whole batch (the most restrictive environment decides).  ``cfl_substeps_per_env`` plans every
    environment on its own."""
    remaining = float(dt)
    while remaining > 0.0 and not abs(remaining) <= 1e-8:
        ts = cfl_substep(remaining, cfl, max_velocity())
        remaining -= ts
        yield float(np.float32(ts))


def cfl_substeps_per_env(lib, B: int, dt: float, cfl: float, max_velocity, device, stream):
    """The per-environment counterpart of ``cfl_substeps``: every environment follows its own adaptive CFL plan through one solver
    step of length ``dt``, as ``fgb_sim_step`` plans plain steps.  ``max_velocity()`` returns the maximum velocity of every environment
    (float32 [B] on ``device``) and is called before every round; the plan of the round comes from ``fgb_plan_substep`` (the same
    arithmetic as ``cfl_substep``, float64 remainders on the device).  Yields ``(dt, active)`` per round -- float32 [B] substep sizes,
    0 for environments whose time is used up, and the int32 [B] mask of the environments that take the substep -- until no
    environment has time left.  The only host read is the round's 4-byte count of active environments, which also ends the loop
    (``lib``: the loaded library; ``stream``: the ctypes stream handle the solver launches on)."""
    remaining = torch.full((B,), float(dt), dtype=torch.float64, device=device)
    nsub = torch.zeros(B, dtype=torch.int32, device=device)
    count = torch.zeros(1, dtype=torch.int32, device=device)
    while True:
        mv = max_velocity().to(device=device, dtype=torch.float32).contiguous()
        dtv = torch.empty(B, dtype=torch.float32, device=device)
        active = torch.empty(B, dtype=torch.int32, device=device)
        count.zero_()
        native.check(lib.fgb_plan_substep(B, _ptr(mv), _ptr(remaining), float(cfl), _ptr(dtv), _ptr(active), _ptr(nsub), _ptr(count), stream),
                     "fgb_plan_substep")
        if int(count.item()) == 0:
            return
        yield dtv, active


def cluster_shape(N: int, cg_impl: int = 6):
    """(cluster size, cells per CTA incl. padding) the on-chip Krylov launchers pick for a grid of N cells
    (cg_cluster_mb_any in csrc/piso_b200.cu): smallest cluster whose CTAs hold ceil(N/CS) cells."""
    shapes = ((2, 1792), (4, 1792), (8, 1792), (16, 1792)) if cg_impl == 8 else ((2, 3072), (4, 3584), (8, 3584), (16, 3072))
    for cs, pad in shapes:
        if -(-N // cs) <= pad:
            return cs, pad
    return None


def halo_plan(nbr: np.ndarray, N: int, cg_impl: int = 6):
    """Static communication plan of the pushed-halo CG (cg_impl 6, tables.cg_*): CTA r of the cluster owns cells
    [r*per, (r+1)*per) in slots [0, per); every remote cell one of its stencils touches gets a halo slot
    pad + h.  Returns dict(cs, pad, slot[4][N], exp[cs][emax][2], cnt[cs][2], emax, hmax) or None."""
    shape = cluster_shape(N, cg_impl)
    if shape is None:
        return None
    cs, pad = shape
    per = -(-N // cs)
    cells = np.arange(N)
    owner = cells // per
    slot = np.zeros((4, N), dtype=np.int32)
    halos = []                                    # per CTA: sorted unique remote cells
    for r in range(cs):
        mine = owner == r
        remote = []
        for f in range(4):
            n = nbr[f][mine]
            ok = n >= 0
            remote.append(n[ok][(n[ok] // per) != r])
        halos.append(np.unique(np.concatenate(remote)) if remote else np.zeros(0, dtype=np.int64))
    for f in range(4):
        n = nbr[f]
        inner = n >= 0
        nn = np.where(inner, n, cells)
        local = (nn // per) == owner
        s = np.where(local, nn - owner * per, 0)
        for r in range(cs):
            sel = (~local) & (owner == r)
            if sel.any():
                s[sel] = pad + np.searchsorted(halos[r], nn[sel])
        slot[f] = s
    exports = [[] for _ in range(cs)]
    for r in range(cs):
        for h, g in enumerate(halos[r]):
            src = int(g // per)
            exports[src].append((int(g - src * per) | (r << 24), pad + h))
    emax = max(1, max(len(e) for e in exports))
    exp = np.zeros((cs, emax, 2), dtype=np.int32)
    cnt = np.zeros((cs, 2), dtype=np.int32)
    for r in range(cs):
        if exports[r]:
            exp[r, :len(exports[r])] = np.asarray(exports[r], dtype=np.int64).astype(np.int32)
        cnt[r] = (len(exports[r]), len(halos[r]))
    hmax = int(max(len(h) for h in halos))
    hmax += hmax & 1                              # keeps the mbarriers behind the halo slots 8-byte aligned
    return dict(cs=cs, pad=pad, slot=slot, exp=exp, cnt=cnt, emax=emax, hmax=hmax)


class BatchedPISO:
    """State + solver for ``n_envs`` environments on one GPU.

    State tensors (device, float32): ``u [B,2,N]``, ``p [B,N]``, ``bvel [B,2,NB]``.
    """

    def __init__(self, cd: CompiledDomain, n_envs: int, device="cuda:0", corrector_steps=2, advect_non_ortho_steps=1,
                 pressure_non_ortho_steps=1, non_orthogonal=True, advection_tol=1e-5, pressure_tol=1e-5,
                 max_iter=5000, cg_impl=6, out_mask=None, groups=None):
        if not torch.cuda.is_available():
            raise native.FGBError("fluidgym_b200 needs a CUDA device (there is no CPU fallback)")
        if os.environ.get("FGB_CG_IMPL"):     # A/B runs: overrides the pressure-CG implementation of every solver
            cg_impl = int(os.environ["FGB_CG_IMPL"])
        self.lib = native.load_for(device)
        self.cd = cd
        self.B = int(n_envs)
        self.N, self.NB = cd.N, cd.NB
        self.device = torch.device(device)
        torch.cuda.set_device(self.device)
        dev = self.device
        self._tab = {}
        for name in _TABLE_FIELDS:
            arr = getattr(cd, name)
            if name == "b_face":
                arr = arr.astype(np.int8)
            self._tab[name] = torch.from_numpy(np.ascontiguousarray(arr)).to(dev)
        self._tab["b_out"] = torch.from_numpy(np.ascontiguousarray(out_mask, dtype=np.int8)).to(dev) if out_mask is not None else None
        self.tables = native.Tables()
        self.tables.N, self.tables.NB, self.tables.K_no, self.tables.K_nob = cd.N, cd.NB, cd.K_no, cd.K_nob
        self.tables.viscosity = float(cd.visc)
        self.has_scalar = cd.scalar_visc is not None
        if self.has_scalar:
            self._tab["Cd_s"] = torch.from_numpy(np.ascontiguousarray(cd.Cd_s)).to(dev)
            self._tab["sb_neumann"] = torch.from_numpy(np.ascontiguousarray(cd.sb_neumann[:max(cd.NB, 1)], dtype=np.int8)).to(dev)
            self.tables.scalar_viscosity = float(cd.scalar_visc)
        else:
            self._tab["Cd_s"] = self._tab["sb_neumann"] = None
        plan = halo_plan(np.asarray(cd.nbr), cd.N, 6 if cg_impl in (11, 12, 13) else cg_impl)
        self.halo = plan
        self.strip = None
        if cg_impl in (11, 12, 13):          # register-blocked strip layout of the pressure CG (strip_plan.py); 6 when it does not apply
            # 13: k_cg_strip with the eager bookkeeping order of round 2 (bit-identical to 11, kept for A/B runs)
            from .strip_plan import pair_shape, plan_for_domain
            # 12: two environments per cluster (k_cg_strip2), half the rows per thread and environment
            sp = self.strip = plan_for_domain(cd, None, *pair_shape()) if cg_impl == 12 else plan_for_domain(cd)
            if sp is not None:
                for k, arr in (("st_thread", sp.thread), ("st_cell", sp.cell), ("st_rexp", sp.rexp), ("st_lexp", sp.lexp), ("st_cnt", sp.cnt)):
                    self._tab[k] = torch.from_numpy(np.ascontiguousarray(arr, dtype=np.int32)).to(dev)
                    setattr(self.tables, k, self._tab[k].data_ptr())
                self.tables.st_cs, self.tables.st_T, self.tables.st_cpt = sp.cs, sp.T, sp.cpt
                self.tables.st_slots, self.tables.st_remax, self.tables.st_lemax = sp.slots, sp.remax, sp.lemax
                self.tables.st_gmax = sp.gmax + (sp.gmax & 1)
        if plan is not None:
            self._tab["cg_slot"] = torch.from_numpy(plan["slot"]).to(dev)
            self._tab["cg_exp"] = torch.from_numpy(plan["exp"]).to(dev)
            self._tab["cg_cnt"] = torch.from_numpy(plan["cnt"]).to(dev)
            self.tables.cg_slot, self.tables.cg_exp, self.tables.cg_cnt = (self._tab[k].data_ptr() for k in ("cg_slot", "cg_exp", "cg_cnt"))
            self.tables.cg_cs, self.tables.cg_emax, self.tables.cg_hmax, self.tables.cg_pad = plan["cs"], plan["emax"], plan["hmax"], plan["pad"]
        for name in _TABLE_FIELDS + ["b_out", "Cd_s", "sb_neumann"]:
            t = self._tab[name]
            setattr(self.tables, name, t.data_ptr() if t is not None else None)
        self.options = native.Options(corrector_steps, advect_non_ortho_steps, pressure_non_ortho_steps,
                                      int(bool(non_orthogonal)), advection_tol, pressure_tol, max_iter, cg_impl)
        nbytes = self.lib.fgb_workspace_bytes(C.byref(self.tables), self.B)
        self.workspace = torch.empty(nbytes + 256, dtype=torch.uint8, device=dev)
        self._ws_off = (-self.workspace.data_ptr()) % 256
        handle = C.c_void_p()
        native.check(self.lib.fgb_batch_create(C.byref(self.tables), self.B, C.c_void_p(self.workspace.data_ptr() + self._ws_off),
                                               nbytes, C.byref(self.options), C.byref(handle)), "fgb_batch_create")
        self.handle = handle
        B, N, NB = self.B, self.N, self.NB
        self.u = torch.zeros(B, 2, N, device=dev)
        self.p = torch.zeros(B, N, device=dev)
        self.bvel = torch.from_numpy(cd.bvel0[:, :NB].copy()).to(dev).unsqueeze(0).repeat(B, 1, 1).contiguous()
        self.src = None
        self.scalar = None           # native.Scalar when the domain carries a passive scalar
        if self.has_scalar:
            self.T = torch.zeros(B, N, device=dev)
            self.sbval = torch.from_numpy(cd.sb_val0[:NB].copy()).to(dev).unsqueeze(0).repeat(B, 1).contiguous()
            self.vsrc = torch.zeros(B, 2, N, device=dev)
            self.set_buoyancy(1.0)
        self.ones_dt = torch.ones(B, device=dev)
        # environment groups on streams of their own inside every substep (fgb_batch_set_groups): measured +8 % (cg_impl 6) / +16 %
        # (cg_impl 11) on 256 cylinder environments with 4 groups (profiles/r02_groups_ab.txt); pointless for small batches
        if groups is None and not os.environ.get("FGB_GROUPS"):
            groups = 4 if self.B >= 64 else (2 if self.B >= 16 else 1)
        self.groups = int(os.environ.get("FGB_GROUPS", 1))
        if groups is not None:
            self.set_groups(groups)

    def set_buoyancy(self, beta: float):
        self.scalar = native.Scalar(self.T.data_ptr(), self.sbval.data_ptr(), float(beta), self.vsrc.data_ptr())

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.lib.fgb_batch_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    # ------------------------------------------------------------------
    @property
    def stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def set_groups(self, groups: int):
        """Run ``groups`` contiguous groups of the batch on their own streams inside every substep (fgb_batch_set_groups)."""
        native.check(self.lib.fgb_batch_set_groups(self.handle, int(groups)), "fgb_batch_set_groups")
        self.groups = int(groups)

    def set_options(self, **kw):
        for k, v in kw.items():
            setattr(self.options, k, v)
        native.check(self.lib.fgb_batch_set_options(self.handle, C.byref(self.options)), "fgb_batch_set_options")

    def buffer(self, name: str) -> torch.Tensor:
        """Zero-copy view of a named workspace buffer (see fgb_batch_buffer)."""
        B, N = self.B, self.N
        shapes = {"Coff": ((B, 4, N), torch.float32), "A": ((B, N), torch.float32), "rhs": ((B, 2, N), torch.float32),
                  "ures": ((B, 2, N), torch.float32), "Poff": ((B, 4, N), torch.float32), "Pdiag": ((B, N), torch.float32),
                  "hbya": ((B, 2, N), torch.float32), "div": ((B, N), torch.float32), "pres": ((B, N), torch.float32),
                  "iters": ((B, 8), torch.int32), "iter_total": ((B, 2), torch.int64), "resid": ((B, 8), torch.float32), "dt": ((B,), torch.float32),
                  "active": ((B,), torch.int32), "remaining": ((B,), torch.float64), "nsub": ((B,), torch.int32),
                  "maxvel": ((B,), torch.float32), "fluxbal": ((B,), torch.float32), "pmean": ((8, B), torch.float32)}
        shape, dtype = shapes[name]
        ptr = self.lib.fgb_batch_buffer(self.handle, name.encode())
        off = ptr - self.workspace.data_ptr()
        n = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
        return self.workspace[off:off + n].view(dtype).view(shape)

    # ---- individual ops (names follow the PISOtorch free functions) --------------------------------
    def _dt(self, dt):
        if isinstance(dt, torch.Tensor):
            return dt.to(self.device, torch.float32).contiguous()
        return torch.full((self.B,), float(dt), device=self.device)

    def setup_advection(self, dt, ures=None, active=None):
        self._dtc = self._dt(dt)
        native.check(self.lib.fgb_setup_advection(self.handle, _ptr(self.u), _ptr(ures), _ptr(self.bvel), _ptr(self.src),
                                                  _ptr(self._dtc), _ptr(active), self.stream), "fgb_setup_advection")

    def solve_advection(self, zero_init=True, active=None):
        native.check(self.lib.fgb_solve_advection(self.handle, int(zero_init), _ptr(active), self.stream), "fgb_solve_advection")

    def setup_pressure_matrix(self, active=None):
        native.check(self.lib.fgb_setup_pressure_matrix(self.handle, _ptr(active), self.stream), "fgb_setup_pressure_matrix")

    def setup_pressure_rhs(self, dt, p_prev=None, with_hbya=True, active=None):
        self._dtc = self._dt(dt)
        p_prev = self.p if p_prev is None else p_prev
        native.check(self.lib.fgb_setup_pressure_rhs(self.handle, _ptr(self.u), _ptr(self.bvel), _ptr(self.src), _ptr(p_prev),
                                                     _ptr(self._dtc), int(with_hbya), _ptr(active), self.stream), "fgb_setup_pressure_rhs")

    def solve_pressure(self, p_out=None, zero_init=True, reset_steps=100, max_iter=None, active=None):
        p_out = self.p if p_out is None else p_out
        native.check(self.lib.fgb_solve_pressure(self.handle, _ptr(p_out), int(zero_init), reset_steps,
                                                 max_iter or self.options.max_iter, _ptr(active), self.stream), "fgb_solve_pressure")

    def correct_velocity(self, p=None, u_out=None, active=None):
        p = self.p if p is None else p
        u_out = self.buffer("ures") if u_out is None else u_out
        native.check(self.lib.fgb_correct_velocity(self.handle, _ptr(p), _ptr(u_out), _ptr(active), self.stream), "fgb_correct_velocity")

    # ---- fused level ------------------------------------------------------------------------------
    def piso_substep(self, dt, active=None):
        """``Simulation._PISO_split_step(iterations=1, time_step=dt)`` for every (active) environment."""
        self._dtc = self._dt(dt)
        sc = C.byref(self.scalar) if self.scalar is not None else None
        native.check(self.lib.fgb_piso_substep(self.handle, _ptr(self.u), _ptr(self.p), _ptr(self.bvel), _ptr(self.src),
                                               _ptr(self._dtc), _ptr(active), sc, self.stream), "fgb_piso_substep")

    def make_divergence_free(self, max_iter=1000):
        native.check(self.lib.fgb_make_divergence_free(self.handle, _ptr(self.u), _ptr(self.p), _ptr(self.bvel), max_iter,
                                                       self.stream), "fgb_make_divergence_free")

    def update_outflow(self, dt, char_vel, tol=1e-5):
        self._dtc = self._dt(dt)
        cv = (C.c_float * 2)(*[float(x) for x in char_vel])
        native.check(self.lib.fgb_update_outflow(self.handle, _ptr(self.u), _ptr(self.bvel), _ptr(self._dtc), cv, tol, self.stream),
                     "fgb_update_outflow")

    def single_step(self, dt, cfl=0.8, char_vel=None, bc_tol=1e-5) -> int:
        """``Simulation.single_step()`` with adaptive CFL sub-stepping; returns the substep rounds used."""
        cv = (C.c_float * 2)(*[float(x) for x in char_vel]) if char_vel is not None else None
        n = C.c_int32(0)
        sc = C.byref(self.scalar) if self.scalar is not None else None
        native.check(self.lib.fgb_sim_step(self.handle, _ptr(self.u), _ptr(self.p), _ptr(self.bvel), _ptr(self.src), float(dt),
                                           float(cfl), cv, float(bc_tol), sc, C.byref(n), self.stream), "fgb_sim_step")
        return n.value

    def flux_balance(self) -> torch.Tensor:
        out = torch.empty(self.B, device=self.device)
        native.check(self.lib.fgb_flux_balance(self.handle, _ptr(self.bvel), _ptr(out), self.stream), "fgb_flux_balance")
        return out

    def column_sums(self, fa: torch.Tensor, fb: torch.Tensor, nx: int, ny: int) -> torch.Tensor:
        out = torch.empty(self.B, 2, nx, device=self.device)
        native.check(self.lib.fgb_column_sums(self.handle, _ptr(fa), _ptr(fb), nx, ny, _ptr(out), self.stream), "fgb_column_sums")
        return out

    def velocity_gradients(self) -> torch.Tensor:
        """PISOtorch.ComputeSpatialVelocityGradients: ``[B, 2 (component c), 2 (direction d), N]`` = d u_c / d x_d (K.cu:6460-6550)"""
        out = torch.empty(self.B, 2, 2, self.N, device=self.device)
        native.check(self.lib.fgb_velocity_gradients(self.handle, _ptr(self.u), _ptr(self.bvel), _ptr(out), self.stream), "fgb_velocity_gradients")
        return out

    def vorticity(self) -> torch.Tensor:
        """omega = d v / d x - d u / d y per cell [B, N].  (The reference's renderer, fluid_env.py:577-606, unpacks the per-component
        tensors as if they were per-direction and therefore shows - omega.)"""
        g = self.velocity_gradients()
        return g[:, 1, 0] - g[:, 0, 1]

    def max_velocity(self) -> torch.Tensor:
        out = torch.empty(self.B, device=self.device)
        native.check(self.lib.fgb_max_velocity(self.handle, _ptr(self.u), _ptr(self.bvel), _ptr(out), self.stream), "fgb_max_velocity")
        return out
