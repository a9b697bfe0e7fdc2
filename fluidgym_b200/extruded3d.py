"""z-extruded multi-block domains (CylinderJet3D / Airfoil3D: the 2-D multi-block grid repeated over ``nz`` uniform periodic
planes, ``envs/cylinder/grid.py:298``, ``shapes.py:641-676``) -- host side of ``csrc/extruded3_b200.cuh``.

STATUS: the operator arithmetic is verified on the CPU against an op trace of the unmodified reference
(``tests/test_extruded_host.py``, ``tests/test_extruded_cpu.py``; ``envs/cylinder3d.py`` runs on the CPU through a stand-in that
executes the same cell code on the host, ``tests/test_cylinder3d_cpu.py``), and ``ExtrudedPISO3D`` (the launch path) on a B200
against the reference's substep, reset state, ``env.step`` and reverse-mode gradients of CylinderJet3D and Airfoil3D
(``tests/test_gpu_extruded.py``, ``tools/extruded_check.py``).
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import native
from .domain import CompiledDomain
from .solver import _TABLE_FIELDS, _ptr, cfl_substep


def extruded_neighbours(nbr2: np.ndarray, nz: int) -> np.ndarray:
    """6-face neighbour table [6][nz * N2] of the extruded domain (cell = plane * N2 + g): faces 0..3 are the in-plane
    neighbours of the compiled 2-D domain shifted into the plane (prescribed faces stay negative: no matrix entry), face 4 / 5 the
    same cell in the plane below / above (periodic)."""
    N2 = nbr2.shape[1]
    k = np.arange(nz, dtype=np.int64)[:, None]
    g = np.arange(N2, dtype=np.int64)[None, :]
    out = np.zeros((6, nz, N2), dtype=np.int64)
    for f in range(4):
        n = nbr2[f].astype(np.int64)[None, :]
        out[f] = np.where(n >= 0, n + k * N2, -1)
    out[4] = ((k - 1) % nz) * N2 + g
    out[5] = ((k + 1) % nz) * N2 + g
    return np.ascontiguousarray(out.reshape(6, nz * N2).astype(np.int32))


class ExtrudedStepping:
    """``Simulation.single_step`` around the extruded substep: the adaptive CFL plan (SIM.py:2004-2031), the "PRE" hook of the
    cylinder / airfoil environments (advective outflow relaxation + flux balance, SIM.py:188-393, cylinder_env_base.py:277-300) and
    the boundary-flux balance used by the actuators -- small torch expressions over the boundary faces ([B, 3, nz, NB2], a few
    thousand values), device agnostic so that the very same code is exercised on the CPU against the reference's boundary values
    (tests/test_cylinder3d_cpu.py).  The class that mixes this in provides ``cd, nz, hz, B, N2, NB2, device, u, p, bvel`` and
    ``piso_substep(dt)``."""

    def setup_stepping(self, out_mask: np.ndarray, char_vel=(1.0, 0.0)):
        cd, NB, dev = self.cd, self.cd.NB, self.device
        face = cd.b_face[:NB].astype(np.int64)
        ax = face >> 1
        sign = np.where(face & 1, 1.0, -1.0).astype(np.float32)
        j = np.arange(NB)
        bm, bd = np.asarray(cd.b_minv)[:, :NB], np.asarray(cd.b_det)[:NB]
        fw = np.stack([bd * bm[2 * ax, j] * sign, bd * bm[2 * ax + 1, j] * sign]).astype(np.float32)
        o = np.nonzero(np.asarray(out_mask).astype(bool))[0]
        adv = (bm[2 * ax[o], o] * np.float32(char_vel[0]) + bm[2 * ax[o] + 1, o] * np.float32(char_vel[1])).astype(np.float32)
        self._st = dict(fw=torch.from_numpy(fw).to(dev), out=torch.from_numpy(o).to(dev), adv=torch.from_numpy(adv).to(dev),
                        out_cells=torch.from_numpy(np.asarray(cd.b_cell)[:NB][o].astype(np.int64)).to(dev),
                        is_out=torch.from_numpy(np.asarray(out_mask).astype(bool)).to(dev),
                        minv=torch.from_numpy(np.ascontiguousarray(cd.minv)).to(dev),
                        b_minv=torch.from_numpy(np.ascontiguousarray(bm)).to(dev))

    def balance_fluxes(self, free: torch.Tensor, tol: float):
        """balance_boundary_fluxes (SIM.py:188-224): all components of the ``free`` faces (bool [NB2], every plane) are scaled by
        -(flux through the other prescribed faces) / (flux through the free faces) unless the imbalance is below 0.01 tol."""
        bv = self.bvel
        fw = self._st["fw"]
        fl = (bv[:, 0] * fw[0] + bv[:, 1] * fw[1]) * self.hz                                  # [B, nz, NB2]
        var = fl[:, :, free].double().sum(dim=(1, 2))
        fixed = fl[:, :, ~free].double().sum(dim=(1, 2))
        ok = (fixed + var).abs() <= tol * 0.01
        scale = torch.where(ok, torch.ones_like(var), -fixed / torch.where(ok, torch.ones_like(var), var)).float()
        bv[:, :, :, free] = bv[:, :, :, free] * scale[:, None, None, None]

    def update_outflow(self, dt: torch.Tensor, tol: float = 5e-6):
        """update_advective_boundaries (SIM.py:228-393): the outflow values relax towards the adjacent cell with weight
        1 - 1 / (1 + 2 dt U_adv), all three components; then the outflow alone is rescaled for a zero net flux."""
        st, bv = self._st, self.bvel
        w = 1.0 - 1.0 / (1.0 + 2.0 * dt.to(self.device, torch.float32)[:, None] * st["adv"][None])       # [B, n_out]
        u4 = self.u.view(self.B, 3, self.nz, self.N2)
        bo = bv[:, :, :, st["out"]]
        bv[:, :, :, st["out"]] = bo - w[:, None, None, :] * (bo - u4[:, :, :, st["out_cells"]])
        self.balance_fluxes(st["is_out"], tol)

    def max_velocity(self) -> torch.Tensor:
        """Domain.getMaxVelocity(True, True) (DS.cpp:1580-1612) -> [B]: max |computational velocity component| over cells and
        prescribed faces; the z component of an extruded cell is w / hz."""
        st = self._st
        u4, bv = self.u.view(self.B, 3, self.nz, self.N2), self.bvel
        mi, bm = st["minv"], st["b_minv"]
        m = torch.stack([(mi[0] * u4[:, 0] + mi[1] * u4[:, 1]).abs().amax(dim=(1, 2)), (mi[2] * u4[:, 0] + mi[3] * u4[:, 1]).abs().amax(dim=(1, 2)),
                         u4[:, 2].abs().amax(dim=(1, 2)) / self.hz,
                         (bm[0] * bv[:, 0] + bm[1] * bv[:, 1]).abs().amax(dim=(1, 2)), (bm[2] * bv[:, 0] + bm[3] * bv[:, 1]).abs().amax(dim=(1, 2)),
                         bv[:, 2].abs().amax(dim=(1, 2)) / self.hz])
        return m.amax(dim=0)

    def single_step(self, dt: float, cfl: float = 0.8, bc_tol: float = 5e-6) -> int:
        """One solver step of length ``dt`` for every environment, split into CFL-limited substeps per environment (same
        arithmetic as k_plan_substep); environments that are already done keep their state.  Returns the substep rounds."""
        B = self.B
        remaining = np.full(B, float(dt), dtype=np.float64)
        rounds = 0
        while True:
            act = (remaining > 0.0) & ~(np.abs(remaining) <= 1e-8)
            if not act.any():
                return rounds
            mv = self.max_velocity().detach().cpu().numpy().astype(np.float32)
            ts = np.zeros(B, dtype=np.float64)
            for b in np.nonzero(act)[0]:
                ts[b] = cfl_substep(float(remaining[b]), cfl, float(mv[b]))
                remaining[b] -= ts[b]
            keep = None
            if not act.all():                       # finished environments ride along with a dummy step and are restored afterwards
                idle = torch.from_numpy(np.nonzero(~act)[0]).to(self.device)
                keep = (idle, self.u[idle].clone(), self.p[idle].clone(), self.bvel[idle].clone())
                ts[~act] = ts[act].max()
            dtv = torch.from_numpy(ts.astype(np.float32)).to(self.device)
            self.update_outflow(dtv, bc_tol)
            self.piso_substep(dtv)
            if keep is not None:
                idle, u0, p0, b0 = keep
                self.u[idle], self.p[idle], self.bvel[idle] = u0, p0, b0
            rounds += 1

    def make_divergence_free_with_hook(self, max_iter: int = 1000, bc_tol: float = 5e-6):
        """Simulation.make_divergence_free incl. its "PRE" hook with time step 1 (SIM.py:1335-1347)."""
        self.update_outflow(torch.ones(self.B), bc_tol)
        self.make_divergence_free(max_iter)


class ExtrudedPISO3D(ExtrudedStepping):
    """State + solver for ``n_envs`` copies of an extruded domain: ``u [B,3,nz*N2]``, ``p [B,nz*N2]``, ``bvel [B,3,nz,NB2]``."""

    def __init__(self, cd: CompiledDomain, nz: int, hz: float, n_envs: int = 1, device="cuda:0", corrector_steps=2,
                 advect_non_ortho_steps=1, pressure_non_ortho_steps=4, advection_tol=1e-5, pressure_tol=5e-7, max_iter=5000):
        if not torch.cuda.is_available():
            raise native.FGBError("fluidgym_b200 needs a CUDA device (there is no CPU fallback)")
        self.lib = native.load_for(device)
        self.cd, self.nz, self.hz, self.B = cd, int(nz), float(hz), int(n_envs)
        self.N2, self.NB2, self.N = cd.N, cd.NB, cd.N * int(nz)
        self.device = torch.device(device)
        torch.cuda.set_device(self.device)
        dev = self.device
        self._tab = {}
        plane = native.Tables()
        plane.N, plane.NB, plane.K_no, plane.K_nob, plane.viscosity = cd.N, cd.NB, cd.K_no, cd.K_nob, float(cd.visc)
        for name in _TABLE_FIELDS:
            arr = getattr(cd, name)
            if name == "b_face":
                arr = arr.astype(np.int8)
            self._tab[name] = torch.from_numpy(np.ascontiguousarray(arr)).to(dev)
            setattr(plane, name, self._tab[name].data_ptr())
        self.xtables = native.Extruded3Tables(plane, self.nz, self.hz)
        # Krylov side: an fgb_ortho3 handle on the 6-face table (its metric arrays are not read by the solvers)
        self._tab["nbr6"] = torch.from_numpy(extruded_neighbours(np.asarray(cd.nbr), self.nz)).to(dev)
        self._tab["ones"] = torch.ones(3 * self.N, device=dev)
        t3 = native.Ortho3Tables(self.N, 0, float(cd.visc), self._tab["nbr6"].data_ptr(), self._tab["ones"].data_ptr(),
                                 self._tab["ones"].data_ptr(), self._tab["ones"].data_ptr(), self._tab["ones"].data_ptr(), 0, 0, 0)
        t3.plane, t3.rev = cd.N, self._tab["rev"].data_ptr()     # transposed Krylov solves of the reverse mode (o3_row_t)
        self.tables3 = t3
        self.options = native.Options(corrector_steps, advect_non_ortho_steps, pressure_non_ortho_steps, 1, advection_tol, pressure_tol,
                                      max_iter, 0)
        nbytes = self.lib.fgb_ortho3_workspace_bytes(C.byref(t3), self.B)
        self.workspace = torch.empty(nbytes + 256, dtype=torch.uint8, device=dev)
        off = (-self.workspace.data_ptr()) % 256
        h = C.c_void_p()
        native.check(self.lib.fgb_ortho3_create(C.byref(t3), self.B, C.c_void_p(self.workspace.data_ptr() + off), nbytes,
                                                C.byref(self.options), C.byref(h)), "fgb_ortho3_create")
        self.handle = h
        self.u = torch.zeros(self.B, 3, self.N, device=dev)
        self.p = torch.zeros(self.B, self.N, device=dev)
        self.bvel = torch.zeros(self.B, 3, self.nz, max(self.NB2, 1), device=dev)

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.lib.fgb_ortho3_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    @property
    def stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def buffer(self, name):
        """workspace views of the Krylov handle (as BatchedPISO3D.buffer): "iters" [B, 8], "resid" [B, 8], "iter_total" [B, 2] (CG,
        BiCGStab iterations summed since creation), "Coff", "A", "rhs", "ures", "Poff", "Pdiag", "hbya", "div"."""
        B, N = self.B, self.N
        shapes = {"Coff": ((B, 6, N), torch.float32), "A": ((B, N), torch.float32), "rhs": ((B, 3, N), torch.float32),
                  "ures": ((B, 3, N), torch.float32), "Poff": ((B, 6, N), torch.float32), "Pdiag": ((B, N), torch.float32),
                  "hbya": ((B, 3, N), torch.float32), "div": ((B, N), torch.float32), "iters": ((B, 8), torch.int32),
                  "resid": ((B, 8), torch.float32), "iter_total": ((B, 2), torch.int64)}
        shape, dtype = shapes[name]
        ptr = self.lib.fgb_ortho3_buffer(self.handle, name.encode())
        o = ptr - self.workspace.data_ptr()
        n = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
        return self.workspace[o:o + n].view(dtype).view(shape)

    def launch_count(self) -> int:
        return int(self.lib.fgb_ortho3_launch_count(self.handle))

    def piso_substep(self, dt):
        dtc = dt.to(self.device, torch.float32).contiguous() if isinstance(dt, torch.Tensor) else torch.full((self.B,), float(dt), device=self.device)
        native.check(self.lib.fgb_extruded3_piso_substep(self.handle, C.byref(self.xtables), _ptr(self.u), _ptr(self.p), _ptr(self.bvel),
                                                         _ptr(dtc), self.stream), "fgb_extruded3_piso_substep")

    def make_divergence_free(self, max_iter: int = 1000):
        native.check(self.lib.fgb_extruded3_make_divergence_free(self.handle, C.byref(self.xtables), _ptr(self.u), _ptr(self.p), _ptr(self.bvel),
                                                                 int(max_iter), self.stream), "fgb_extruded3_make_divergence_free")

    # ---- the boundary hooks as kernels (default; FGB_X3_HOOKS=torch selects the torch expressions of ExtrudedStepping) ----
    # tests/test_gpu_extruded.py compares the two paths with each other and with a float64 evaluation (green on a B200, round 2).
    def _cuda_hooks(self) -> bool:
        import os
        return os.environ.get("FGB_X3_HOOKS", "cuda") != "torch"

    def _hook_tables(self):
        if "out32" not in self._st:
            st = self._st
            st["out32"] = st["out"].to(torch.int32).contiguous()
            st["out_cells32"] = st["out_cells"].to(torch.int32).contiguous()
            st["is_out8"] = st["is_out"].to(torch.int8).contiguous()
            st["fw"] = st["fw"].contiguous()
        return self._st

    def balance_fluxes(self, free: torch.Tensor, tol: float):
        if not self._cuda_hooks():
            return ExtrudedStepping.balance_fluxes(self, free, tol)
        st = self._hook_tables()
        mask = free.to(torch.int8).contiguous()
        native.check(self.lib.fgb_extruded3_balance_fluxes(C.byref(self.xtables), self.B, _ptr(self.bvel), _ptr(st["fw"]), _ptr(mask), float(tol),
                                                           self.stream), "fgb_extruded3_balance_fluxes")

    def update_outflow(self, dt: torch.Tensor, tol: float = 5e-6):
        if not self._cuda_hooks():
            return ExtrudedStepping.update_outflow(self, dt, tol)
        st = self._hook_tables()
        dtc = dt.to(self.device, torch.float32).contiguous()
        native.check(self.lib.fgb_extruded3_update_outflow(C.byref(self.xtables), self.B, _ptr(self.u), _ptr(self.bvel), _ptr(dtc), _ptr(st["fw"]),
                                                           _ptr(st["is_out8"]), int(st["out32"].numel()), _ptr(st["out32"]), _ptr(st["out_cells32"]),
                                                           _ptr(st["adv"]), float(tol), self.stream), "fgb_extruded3_update_outflow")

    def max_velocity(self) -> torch.Tensor:
        if not self._cuda_hooks():
            return ExtrudedStepping.max_velocity(self)
        out = torch.empty(self.B, device=self.device)
        native.check(self.lib.fgb_extruded3_max_velocity(C.byref(self.xtables), self.B, _ptr(self.u), _ptr(self.bvel), _ptr(out), self.stream),
                     "fgb_extruded3_max_velocity")
        return out

    def apply_jets(self, amp: torch.Tensor, templ: torch.Tensor, jet_faces: torch.Tensor, free: torch.Tensor, tol: float) -> bool:
        """amp [B, nz, J], templ [J, 2, nf]: one launch for actuation + flux balance when the kernel hooks are on; returns False (nothing
        done) otherwise, the caller then uses its torch expressions."""
        if not self._cuda_hooks():
            return False
        st = self._hook_tables()
        a, t = amp.to(self.device, torch.float32).contiguous(), templ.to(self.device, torch.float32).contiguous()
        jf, mask = jet_faces.to(torch.int32).contiguous(), free.to(torch.int8).contiguous()
        native.check(self.lib.fgb_extruded3_apply_jets(C.byref(self.xtables), self.B, _ptr(self.bvel), _ptr(a), int(a.shape[2]), _ptr(jf), _ptr(t),
                                                       int(jf.numel()), _ptr(st["fw"]), _ptr(mask), float(tol), self.stream), "fgb_extruded3_apply_jets")
        return True
