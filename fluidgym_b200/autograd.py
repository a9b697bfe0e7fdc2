"""torch.autograd integration of the batched PISO substep.

The reference wraps every native op in its own ``torch.autograd.Function`` and re-installs saved tensors
into the shared mutable ``Domain`` for each backward call (``simulation/pict/PISOtorch_diff.py:624-1808``).
Here one ``Function`` covers a whole substep: the forward call records a compact tape on the device
(``fgb_piso_substep_record``), the backward call runs the hand-written adjoint kernels and two transposed
on-chip Krylov solves (``fgb_piso_substep_backward``).  Differentiable inputs: cell velocity ``u``, previous
pressure ``p`` (enters through the deferred non-orthogonal correction) and the Dirichlet boundary velocities
``bvel`` (jets / inflow); geometry and viscosity are constants, like the transforms in the reference.
``PISOSubstepScalar`` is the same node for domains with a passive scalar and buoyancy (RBC): additional
differentiable inputs are the temperature field and the boundary temperatures (heaters).

Every node takes an optional ``active`` mask (int32 ``[B]`` on the solver's device, 0 = skip; ``None`` = every environment): a
skipped environment is the identity in both directions -- its outputs are its inputs bit for bit, its cotangents pass through
unchanged and its boundary values get none.  Per-environment CFL plans (``solver.cfl_substeps_per_env``) use it for environments
that have already used up their time.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import native
from .solver import BatchedPISO, _ptr


def _new_tape(solver: BatchedPISO):
    B, N, NB = solver.B, solver.N, solver.NB
    f32 = dict(device=solver.device, dtype=torch.float32)
    o = solver.options
    C_ = int(o.corrector_steps)
    n_adv, n_p = (int(o.adv_nonortho_steps), int(o.p_nonortho_steps)) if int(o.nonortho) else (1, 1)
    return dict(u_in=torch.empty(B, 2, N, **f32), p_in=torch.empty(B, N, **f32), bvel_in=torch.empty(B, 2, NB, **f32),
                dt=torch.empty(B, **f32), Coff=torch.empty(B, 4, N, **f32), A=torch.empty(B, N, **f32),
                ustar=torch.empty(n_adv, B, 2, N, **f32), hb=torch.empty(C_, B, 2, N, **f32), p=torch.empty(C_ * n_p, B, N, **f32),
                pmean=torch.empty(C_ * n_p, B, **f32), u1=torch.empty(max(C_ - 1, 1), B, 2, N, **f32))


def _ctape(cls, tape: dict, active):
    """the C tape of the buffers in ``tape`` (native.Tape / native.Ortho3Tape) with the environment mask ``active`` (or None)"""
    return cls(*[tape[k].data_ptr() for k, _ in cls._fields_ if k != "active"], active.data_ptr() if active is not None else None)


def _mask(solver, active):
    if active is None:
        return None
    if active.dtype != torch.int32 or tuple(active.shape) != (solver.B,) or active.device.type != solver.device.type:
        raise ValueError(f"active must be an int32 tensor of shape ({solver.B},) on {solver.device}")
    return active.contiguous()


def _adjoint_workspace(solver: BatchedPISO):
    nbytes = solver.lib.fgb_adjoint_workspace_bytes(C.byref(solver.tables), solver.B)
    ws = getattr(solver, "_adj_ws", None)
    if ws is None or ws.numel() < nbytes + 256:
        ws = solver._adj_ws = torch.empty(nbytes + 256, dtype=torch.uint8, device=solver.device)
    return C.c_void_p(ws.data_ptr() + (-ws.data_ptr()) % 256), nbytes


class PISOSubstep(torch.autograd.Function):
    """(u [B,2,N], p [B,N], bvel [B,2,NB]) -> (u_next, p_next) for one substep of ``dt`` (tensor [B] or float)."""

    @staticmethod
    def forward(ctx, u, p, bvel, solver: BatchedPISO, dt, active=None):
        dtc = solver._dt(dt)
        active = _mask(solver, active)
        tape = _new_tape(solver)
        ct = _ctape(native.Tape, tape, active)
        u_out = u.detach().clone().contiguous()
        p_out = p.detach().clone().contiguous()
        bv = bvel.detach().contiguous()
        native.check(solver.lib.fgb_piso_substep_record(solver.handle, _ptr(u_out), _ptr(p_out), _ptr(bv), _ptr(dtc), C.byref(ct),
                                                        solver.stream), "fgb_piso_substep_record")
        ctx.solver, ctx.tape, ctx.active = solver, tape, active
        return u_out, p_out

    @staticmethod
    def backward(ctx, u_out_bar, p_out_bar):
        solver, tape = ctx.solver, ctx.tape
        B, N, NB = solver.B, solver.N, solver.NB
        f32 = dict(device=solver.device, dtype=torch.float32)
        ct = _ctape(native.Tape, tape, ctx.active)
        ub, pb, bvb = torch.empty(B, 2, N, **f32), torch.empty(B, N, **f32), torch.empty(B, 2, NB, **f32)
        ws, nbytes = _adjoint_workspace(solver)
        uo = (u_out_bar if u_out_bar is not None else torch.zeros(B, 2, N, **f32)).contiguous()
        po = (p_out_bar if p_out_bar is not None else torch.zeros(B, N, **f32)).contiguous()
        native.check(solver.lib.fgb_piso_substep_backward(solver.handle, C.byref(ct), _ptr(uo), _ptr(po), _ptr(ub), _ptr(pb), _ptr(bvb),
                                                          ws, nbytes, solver.stream), "fgb_piso_substep_backward")
        return ub, pb, bvb, None, None, None


class PISOSubstepScalar(torch.autograd.Function):
    """(u [B,2,N], p [B,N], bvel [B,2,NB], T [B,N], sbval [B,NB]) -> (u_next, p_next, T_next): scalar transport with the
    incoming velocity, buoyancy source ``(0, beta T_next)``, PISO substep (SIM.py:1471-1657, rbc_env_base.py:280-304)."""

    @staticmethod
    def forward(ctx, u, p, bvel, T, sbval, solver: BatchedPISO, dt, beta, active=None):
        dtc = solver._dt(dt)
        active = _mask(solver, active)
        tape = _new_tape(solver)
        f32 = dict(device=solver.device, dtype=torch.float32)
        stape = dict(T_in=torch.empty(solver.B, solver.N, **f32), T_out=torch.empty(solver.B, solver.N, **f32),
                     sbval_in=torch.empty(solver.B, solver.NB, **f32))
        ct = _ctape(native.Tape, tape, active)
        cs = native.ScalarTape(*[stape[k].data_ptr() for k, _ in native.ScalarTape._fields_])
        u_out, p_out, T_out = (x.detach().clone().contiguous() for x in (u, p, T))
        bv, sb = bvel.detach().contiguous(), sbval.detach().contiguous()
        src = torch.empty(solver.B, 2, solver.N, **f32)
        sc = native.Scalar(T_out.data_ptr(), sb.data_ptr(), float(beta), src.data_ptr())
        native.check(solver.lib.fgb_piso_substep_record_scalar(solver.handle, _ptr(u_out), _ptr(p_out), _ptr(bv), _ptr(dtc), C.byref(sc),
                                                               C.byref(ct), C.byref(cs), solver.stream), "fgb_piso_substep_record_scalar")
        ctx.solver, ctx.tape, ctx.stape, ctx.beta, ctx.active = solver, tape, stape, float(beta), active
        return u_out, p_out, T_out

    @staticmethod
    def backward(ctx, u_out_bar, p_out_bar, T_out_bar):
        solver, tape, stape = ctx.solver, ctx.tape, ctx.stape
        B, N, NB = solver.B, solver.N, solver.NB
        f32 = dict(device=solver.device, dtype=torch.float32)
        ct = _ctape(native.Tape, tape, ctx.active)
        cs = native.ScalarTape(*[stape[k].data_ptr() for k, _ in native.ScalarTape._fields_])
        ub, pb, bvb = torch.empty(B, 2, N, **f32), torch.empty(B, N, **f32), torch.empty(B, 2, NB, **f32)
        Tb, sbb = torch.empty(B, N, **f32), torch.empty(B, NB, **f32)
        ws, nbytes = _adjoint_workspace(solver)
        uo = (u_out_bar if u_out_bar is not None else torch.zeros(B, 2, N, **f32)).contiguous()
        po = (p_out_bar if p_out_bar is not None else torch.zeros(B, N, **f32)).contiguous()
        To = (T_out_bar if T_out_bar is not None else torch.zeros(B, N, **f32)).contiguous()
        native.check(solver.lib.fgb_piso_substep_backward_scalar(solver.handle, C.byref(ct), C.byref(cs), ctx.beta, _ptr(uo), _ptr(po),
                                                                 _ptr(To), _ptr(ub), _ptr(pb), _ptr(bvb), _ptr(Tb), _ptr(sbb), ws, nbytes,
                                                                 solver.stream), "fgb_piso_substep_backward_scalar")
        return ub, pb, bvb, Tb, sbb, None, None, None, None


def piso_substep_scalar(solver: BatchedPISO, u, p, bvel, T, sbval, dt, beta=1.0, active=None):
    """Differentiable substep of a domain with passive scalar + buoyancy (functional form); ``active``: optional int32 [B] mask."""
    return PISOSubstepScalar.apply(u, p, bvel, T, sbval, solver, dt, beta, active)


def piso_substep(solver: BatchedPISO, u, p, bvel, dt, active=None):
    """Differentiable PISO substep (functional form: inputs are not modified); ``active``: optional int32 [B] mask of the
    environments that take the substep, the others pass through unchanged."""
    return PISOSubstep.apply(u, p, bvel, solver, dt, active)


# ---- D = 3 structured boxes (turbulent channel): fgb_ortho3_piso_substep_record / _backward ------------------------------------------
def _new_tape3(solver):
    B, N, NB = solver.B, solver.N, max(solver.NB, 1)
    f32 = dict(device=solver.device, dtype=torch.float32)
    C_ = int(solver.options.corrector_steps)
    return dict(u_in=torch.empty(B, 3, N, **f32), bvel_in=torch.empty(B, 3, NB, **f32), dt=torch.empty(B, **f32),
                Coff=torch.empty(B, 6, N, **f32), A=torch.empty(B, N, **f32), ustar=torch.empty(B, 3, N, **f32),
                hb=torch.empty(C_, B, 3, N, **f32), p=torch.empty(C_, B, N, **f32), u1=torch.empty(max(C_ - 1, 1), B, 3, N, **f32),
                visc=torch.empty(B, N, **f32))          # read only when a sub-grid model is set


def _adjoint_workspace3(solver):
    nbytes = solver.lib.fgb_ortho3_adjoint_workspace_bytes(C.byref(solver.tables), solver.B)
    ws = getattr(solver, "_adj_ws", None)
    if ws is None or ws.numel() < nbytes + 256:
        ws = solver._adj_ws = torch.empty(nbytes + 256, dtype=torch.uint8, device=solver.device)
    return C.c_void_p(ws.data_ptr() + (-ws.data_ptr()) % 256), nbytes


class PISOSubstep3D(torch.autograd.Function):
    """(u [B,3,N], p [B,N], bvel [B,3,NB]) -> (u_next, p_next) for one substep of a structured 3-D box (``BatchedPISO3D``); ``src``
    [B,4] (channel forcing) is a constant of the graph, as in the reference (envs/tcf/grid.py:147-161 rebuilds it with
    ``torch.tensor``).  The previous pressure gets no gradient: every recorded solve starts from zero."""

    @staticmethod
    def forward(ctx, u, p, bvel, solver, dt, src, active=None):
        dtc = solver._dt(dt)
        active = _mask(solver, active)
        tape = _new_tape3(solver)
        ct = _ctape(native.Ortho3Tape, tape, active)
        u_out, p_out = u.detach().clone().contiguous(), p.detach().clone().contiguous()
        bv = bvel.detach().contiguous()
        srcc = None if src is None else src.detach().contiguous()
        native.check(solver.lib.fgb_ortho3_piso_substep_record(solver.handle, _ptr(u_out), _ptr(p_out), _ptr(bv), _ptr(srcc), _ptr(dtc),
                                                               C.byref(ct), solver.stream), "fgb_ortho3_piso_substep_record")
        ctx.solver, ctx.tape, ctx.active = solver, tape, active
        return u_out, p_out

    @staticmethod
    def backward(ctx, u_out_bar, p_out_bar):
        solver, tape = ctx.solver, ctx.tape
        B, N, NB = solver.B, solver.N, max(solver.NB, 1)
        f32 = dict(device=solver.device, dtype=torch.float32)
        ct = _ctape(native.Ortho3Tape, tape, ctx.active)
        ub, bvb = torch.empty(B, 3, N, **f32), torch.empty(B, 3, NB, **f32)
        ws, nbytes = _adjoint_workspace3(solver)
        uo = (u_out_bar if u_out_bar is not None else torch.zeros(B, 3, N, **f32)).contiguous()
        po = (p_out_bar if p_out_bar is not None else torch.zeros(B, N, **f32)).contiguous()
        native.check(solver.lib.fgb_ortho3_piso_substep_backward(solver.handle, C.byref(ct), _ptr(uo), _ptr(po), _ptr(ub), _ptr(bvb), ws, nbytes,
                                                                 solver.stream), "fgb_ortho3_piso_substep_backward")
        return ub, None, bvb, None, None, None, None


def piso_substep_3d(solver, u, p, bvel, dt, src=None, active=None):
    """Differentiable substep of a structured 3-D box (functional form: inputs are not modified); ``active``: optional int32 [B] mask."""
    return PISOSubstep3D.apply(u, p, bvel, solver, dt, src, active)


class PISOSubstepScalar3D(torch.autograd.Function):
    """(u [B,3,N], p [B,N], bvel [B,3,NB], T [B,N], sbval [B,NB]) -> (u_next, p_next, T_next) on a structured 3-D box with an attached
    passive scalar + buoyancy (RBC3D; ``BatchedPISO3D.attach_scalar``).  The solver's own scalar buffers are used as scratch."""

    @staticmethod
    def forward(ctx, u, p, bvel, T, sbval, solver, dt, active=None):
        dtc = solver._dt(dt)
        active = _mask(solver, active)
        tape = _new_tape3(solver)
        f32 = dict(device=solver.device, dtype=torch.float32)
        stape = dict(T_in=torch.empty(solver.B, solver.N, **f32), T_out=torch.empty(solver.B, solver.N, **f32),
                     sbval_in=torch.empty(solver.B, max(solver.NB, 1), **f32))
        ct = _ctape(native.Ortho3Tape, tape, active)
        cs = native.ScalarTape(*[stape[k].data_ptr() for k, _ in native.ScalarTape._fields_])
        u_out, p_out = u.detach().clone().contiguous(), p.detach().clone().contiguous()
        bv = bvel.detach().contiguous()
        solver.T.copy_(T.detach()); solver.sbval.copy_(sbval.detach())
        native.check(solver.lib.fgb_ortho3_piso_substep_record_scalar(solver.handle, _ptr(u_out), _ptr(p_out), _ptr(bv), None, _ptr(dtc), C.byref(ct),
                                                                      C.byref(cs), solver.stream), "fgb_ortho3_piso_substep_record_scalar")
        ctx.solver, ctx.tape, ctx.stape, ctx.active = solver, tape, stape, active
        return u_out, p_out, solver.T.clone()

    @staticmethod
    def backward(ctx, u_out_bar, p_out_bar, T_out_bar):
        solver, tape, stape = ctx.solver, ctx.tape, ctx.stape
        B, N, NB = solver.B, solver.N, max(solver.NB, 1)
        f32 = dict(device=solver.device, dtype=torch.float32)
        ct = _ctape(native.Ortho3Tape, tape, ctx.active)
        cs = native.ScalarTape(*[stape[k].data_ptr() for k, _ in native.ScalarTape._fields_])
        ub, bvb, Tb, sbb = torch.empty(B, 3, N, **f32), torch.empty(B, 3, NB, **f32), torch.empty(B, N, **f32), torch.empty(B, NB, **f32)
        ws, nbytes = _adjoint_workspace3(solver)
        uo = (u_out_bar if u_out_bar is not None else torch.zeros(B, 3, N, **f32)).contiguous()
        po = (p_out_bar if p_out_bar is not None else torch.zeros(B, N, **f32)).contiguous()
        To = (T_out_bar if T_out_bar is not None else torch.zeros(B, N, **f32)).contiguous()
        native.check(solver.lib.fgb_ortho3_piso_substep_backward_scalar(solver.handle, C.byref(ct), C.byref(cs), _ptr(uo), _ptr(po), _ptr(To), _ptr(ub),
                                                                        _ptr(bvb), _ptr(Tb), _ptr(sbb), ws, nbytes, solver.stream),
                     "fgb_ortho3_piso_substep_backward_scalar")
        return ub, None, bvb, Tb, sbb, None, None, None


def piso_substep_scalar_3d(solver, u, p, bvel, T, sbval, dt, active=None):
    """Differentiable substep of a structured 3-D box with passive scalar + buoyancy (functional form); ``active``: optional int32 [B]
    mask."""
    return PISOSubstepScalar3D.apply(u, p, bvel, T, sbval, solver, dt, active)


# ---- z-extruded multi-block grids (CylinderJet3D / Airfoil3D): fgb_extruded3_piso_substep_record / _backward -----------------------------
class PISOSubstepExtruded(torch.autograd.Function):
    """(u [B,3,N3], p [B,N3], bvel [B,3,nz,NB2]) -> (u_next, p_next) for one substep of an ``ExtrudedPISO3D`` solver"""

    @staticmethod
    def forward(ctx, u, p, bvel, solver, dt, active=None):
        B, N3, nz, NB = solver.B, solver.N, solver.nz, max(solver.NB2, 1)
        active = _mask(solver, active)
        f32 = dict(device=solver.device, dtype=torch.float32)
        o = solver.options
        C_, n_adv, n_p = int(o.corrector_steps), int(o.adv_nonortho_steps), int(o.p_nonortho_steps)
        tape = dict(u_in=torch.empty(B, 3, N3, **f32), p_in=torch.empty(B, N3, **f32), bvel_in=torch.empty(B, 3, nz, NB, **f32),
                    dt=torch.empty(B, **f32), Coff=torch.empty(B, 6, N3, **f32), A=torch.empty(B, N3, **f32),
                    ustar=torch.empty(n_adv, B, 3, N3, **f32), hb=torch.empty(C_, B, 3, N3, **f32), p=torch.empty(C_ * n_p, B, N3, **f32),
                    pmean=torch.empty(C_ * n_p, B, **f32), u1=torch.empty(max(C_ - 1, 1), B, 3, N3, **f32))
        ct = _ctape(native.Tape, tape, active)
        dtc = dt.to(solver.device, torch.float32).contiguous() if isinstance(dt, torch.Tensor) else torch.full((B,), float(dt), **f32)
        u_out, p_out = u.detach().clone().contiguous(), p.detach().clone().contiguous()
        bv = bvel.detach().contiguous()
        native.check(solver.lib.fgb_extruded3_piso_substep_record(solver.handle, C.byref(solver.xtables), _ptr(u_out), _ptr(p_out), _ptr(bv), _ptr(dtc),
                                                                  C.byref(ct), solver.stream), "fgb_extruded3_piso_substep_record")
        ctx.solver, ctx.tape, ctx.active = solver, tape, active
        return u_out, p_out

    @staticmethod
    def backward(ctx, u_out_bar, p_out_bar):
        solver, tape = ctx.solver, ctx.tape
        B, N3, nz, NB = solver.B, solver.N, solver.nz, max(solver.NB2, 1)
        f32 = dict(device=solver.device, dtype=torch.float32)
        ct = _ctape(native.Tape, tape, ctx.active)
        ub, pb, bvb = torch.empty(B, 3, N3, **f32), torch.empty(B, N3, **f32), torch.empty(B, 3, nz, NB, **f32)
        nbytes = solver.lib.fgb_extruded3_adjoint_workspace_bytes(C.byref(solver.xtables), B)
        ws = getattr(solver, "_adj_ws", None)
        if ws is None or ws.numel() < nbytes + 256:
            ws = solver._adj_ws = torch.empty(nbytes + 256, dtype=torch.uint8, device=solver.device)
        wsp = C.c_void_p(ws.data_ptr() + (-ws.data_ptr()) % 256)
        uo = (u_out_bar if u_out_bar is not None else torch.zeros(B, 3, N3, **f32)).contiguous()
        po = (p_out_bar if p_out_bar is not None else torch.zeros(B, N3, **f32)).contiguous()
        native.check(solver.lib.fgb_extruded3_piso_substep_backward(solver.handle, C.byref(solver.xtables), C.byref(ct), _ptr(uo), _ptr(po), _ptr(ub),
                                                                    _ptr(pb), _ptr(bvb), wsp, nbytes, solver.stream), "fgb_extruded3_piso_substep_backward")
        return ub, pb, bvb, None, None, None


def piso_substep_extruded(solver, u, p, bvel, dt, active=None):
    """Differentiable substep of a z-extruded multi-block grid (functional form); ``active``: optional int32 [B] mask."""
    return PISOSubstepExtruded.apply(u, p, bvel, solver, dt, active)
