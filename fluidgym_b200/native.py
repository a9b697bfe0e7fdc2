"""ctypes binding of the C ABI in include/fluidgym_b200.h (no torch types cross the boundary).

The product path has NO CPU fallback: if the shared library is missing or no CUDA device is
present, loading / creating a batch raises.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

_lib = None


class FGBError(RuntimeError):
    pass


class Tables(C.Structure):
    _fields_ = [("N", C.c_int32), ("NB", C.c_int32), ("K_no", C.c_int32), ("K_nob", C.c_int32),
                ("viscosity", C.c_float)] + [(n, C.c_void_p) for n in (
                    "nbr", "fl_comp", "minv", "det", "Cd", "Wp", "no_idx", "no_face", "no_gP", "no_gN", "no_wv",
                    "nob_idx", "nob_w", "b_minv", "b_det", "b_alpha", "b_cell", "b_face", "b_out")] + [
                    ("scalar_viscosity", C.c_float), ("Cd_s", C.c_void_p), ("sb_neumann", C.c_void_p), ("rev", C.c_void_p),
                    ("cg_slot", C.c_void_p), ("cg_exp", C.c_void_p), ("cg_cnt", C.c_void_p),
                    ("cg_cs", C.c_int32), ("cg_emax", C.c_int32), ("cg_hmax", C.c_int32), ("cg_pad", C.c_int32),
                    ("st_thread", C.c_void_p), ("st_cell", C.c_void_p), ("st_rexp", C.c_void_p), ("st_lexp", C.c_void_p),
                    ("st_cnt", C.c_void_p), ("st_cs", C.c_int32), ("st_T", C.c_int32), ("st_cpt", C.c_int32), ("st_slots", C.c_int32),
                    ("st_remax", C.c_int32), ("st_lemax", C.c_int32), ("st_gmax", C.c_int32)]


class Tape(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("u_in", "p_in", "bvel_in", "dt", "Coff", "A", "ustar", "hb", "p", "pmean", "u1", "active")]


class Ortho3Tape(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("u_in", "bvel_in", "dt", "Coff", "A", "ustar", "hb", "p", "u1", "visc", "active")]


class ScalarTape(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("T_in", "T_out", "sbval_in")]


class Scalar(C.Structure):
    _fields_ = [("T", C.c_void_p), ("sbval", C.c_void_p), ("beta", C.c_float), ("src", C.c_void_p)]


class Options(C.Structure):
    _fields_ = [("corrector_steps", C.c_int32), ("adv_nonortho_steps", C.c_int32), ("p_nonortho_steps", C.c_int32),
                ("nonortho", C.c_int32), ("adv_tol", C.c_float), ("p_tol", C.c_float), ("max_iter", C.c_int32),
                ("cg_impl", C.c_int32)]


class Ortho3Tables(C.Structure):
    _fields_ = [("N", C.c_int32), ("NB", C.c_int32), ("viscosity", C.c_float), ("nbr", C.c_void_p), ("minv", C.c_void_p),
                ("det", C.c_void_p), ("b_minv", C.c_void_p), ("b_det", C.c_void_p), ("NS", C.c_int32), ("N_global", C.c_int32),
                ("plane", C.c_int32), ("nx", C.c_int32), ("ny", C.c_int32), ("nz", C.c_int32), ("closed", C.c_int32),
                ("boff", C.c_int32 * 6), ("rev", C.c_void_p)]


class Ortho3Scalar(C.Structure):
    _fields_ = [("T", C.c_void_p), ("sbval", C.c_void_p), ("kappa", C.c_float), ("beta", C.c_float)]


class Extruded3Tables(C.Structure):
    _fields_ = [("plane", Tables), ("nz", C.c_int32), ("hz", C.c_float)]


class Wall(C.Structure):
    _fields_ = [("n_wall", C.c_int32), ("cell", C.c_void_p), ("bface", C.c_void_p), ("normal", C.c_void_p),
                ("dist", C.c_void_p), ("tlen", C.c_void_p), ("flen", C.c_void_p), ("scale", C.c_float)]


EXPORTS = ["fgb_last_error", "fgb_version", "fgb_workspace_bytes", "fgb_batch_create", "fgb_batch_destroy",
           "fgb_batch_set_options", "fgb_batch_set_groups", "fgb_batch_buffer", "fgb_setup_advection", "fgb_solve_advection",
           "fgb_setup_pressure_matrix", "fgb_setup_pressure_rhs", "fgb_solve_pressure", "fgb_correct_velocity",
           "fgb_piso_substep", "fgb_make_divergence_free", "fgb_sim_step", "fgb_update_outflow", "fgb_flux_balance", "fgb_balance_fluxes",
           "fgb_max_velocity", "fgb_apply_jet_action", "fgb_wall_forces", "fgb_column_sums", "fgb_sample_sensors",
           "fgb_profile_enable",
           "fgb_profile_read", "fgb_launch_count", "fgb_velocity_gradients", "fgb_piso_substep_record", "fgb_adjoint_workspace_bytes",
           "fgb_piso_substep_backward", "fgb_piso_substep_record_scalar", "fgb_piso_substep_backward_scalar",
           "fgb_ortho3_workspace_bytes", "fgb_ortho3_create", "fgb_ortho3_destroy", "fgb_ortho3_set_options", "fgb_ortho3_buffer",
           "fgb_ortho3_launch_count", "fgb_ortho3_setup_advection", "fgb_ortho3_solve_advection", "fgb_ortho3_setup_pressure",
           "fgb_ortho3_solve_pressure", "fgb_ortho3_correct_velocity", "fgb_ortho3_piso_substep", "fgb_ortho3_make_divergence_free",
           "fgb_ortho3_sim_step", "fgb_ortho3_wall_rows", "fgb_ipc_alloc", "fgb_ipc_open", "fgb_ipc_close", "fgb_ipc_free",
           "fgb_ortho3_set_slab", "fgb_ortho3_slab_error", "fgb_ortho3_set_scalar", "fgb_ortho3_advect_scalar", "fgb_ortho3_set_sgs", "fgb_ortho3_sgs_viscosity", "fgb_ortho3_velocity_gradients", "fgb_ortho3_piso_substep_record", "fgb_ortho3_adjoint_workspace_bytes", "fgb_ortho3_piso_substep_backward", "fgb_ortho3_piso_substep_record_scalar", "fgb_ortho3_piso_substep_backward_scalar", "fgb_extruded3_piso_substep_record", "fgb_extruded3_adjoint_workspace_bytes", "fgb_extruded3_piso_substep_backward", "fgb_sample_sensors_n", "fgb_extruded3_piso_substep", "fgb_extruded3_make_divergence_free",
           "fgb_extruded3_balance_fluxes", "fgb_extruded3_update_outflow", "fgb_extruded3_max_velocity", "fgb_extruded3_wall_forces", "fgb_extruded3_apply_jets", "fgb_render_gather", "fgb_render_colour", "fgb_plan_substep"]


def lib_path() -> str:
    return _build.LIB


class DeviceLib:
    """The loaded library bound to ONE CUDA device: every ``fgb_*`` call is issued with that device current.

    The C entry points launch on the stream they are given and allocate nothing, but a launch (and cudaEvent / IPC calls)
    needs the stream's device to be the calling thread's current device.  A solver on cuda:1 stepped from a thread whose current
    device is cuda:0 (``ParallelFluidEnv`` worker threads, or simply after constructing another solver on cuda:0) would otherwise
    launch into the wrong context.  The guard costs one ``cudaGetDevice`` when the device is already current."""

    def __init__(self, lib, device):
        import torch
        self._lib = lib
        self._torch = torch
        self._index = torch.device(device).index if torch.device(device).index is not None else torch.cuda.current_device()
        self._cache = {}

    def __getattr__(self, name):
        fn = self._cache.get(name)
        if fn is None:
            raw = getattr(self._lib, name)
            torch, index = self._torch, self._index

            def fn(*a, _raw=raw):
                if torch.cuda.current_device() == index:
                    return _raw(*a)
                with torch.cuda.device(index):
                    return _raw(*a)
            self._cache[name] = fn
        return fn


def load_for(device):
    """``load()`` bound to a device (see DeviceLib)."""
    return DeviceLib(load(), device)


def load():
    """Load libfluidgym_b200.so (built in-tree by fluidgym_b200.build / __graft_entry__.build)."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise FGBError(f"{path} is missing: run `python -m fluidgym_b200.build` (there is no CPU fallback)")
    L = C.CDLL(path)
    vp, i32, f32 = C.c_void_p, C.c_int32, C.c_float
    L.fgb_last_error.restype = C.c_char_p
    L.fgb_workspace_bytes.restype = C.c_size_t
    L.fgb_workspace_bytes.argtypes = [C.POINTER(Tables), i32]
    L.fgb_batch_create.argtypes = [C.POINTER(Tables), i32, vp, C.c_size_t, C.POINTER(Options), C.POINTER(vp)]
    L.fgb_batch_destroy.argtypes = [vp]
    L.fgb_batch_destroy.restype = None
    L.fgb_batch_set_options.argtypes = [vp, C.POINTER(Options)]
    L.fgb_batch_set_groups.argtypes = [vp, i32]
    L.fgb_batch_buffer.restype = vp
    L.fgb_batch_buffer.argtypes = [vp, C.c_char_p]
    L.fgb_setup_advection.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    L.fgb_solve_advection.argtypes = [vp, i32, vp, vp]
    L.fgb_setup_pressure_matrix.argtypes = [vp, vp, vp]
    L.fgb_setup_pressure_rhs.argtypes = [vp, vp, vp, vp, vp, vp, i32, vp, vp]
    L.fgb_solve_pressure.argtypes = [vp, vp, i32, i32, i32, vp, vp]
    L.fgb_correct_velocity.argtypes = [vp, vp, vp, vp, vp]
    L.fgb_piso_substep.argtypes = [vp, vp, vp, vp, vp, vp, vp, C.POINTER(Scalar), vp]
    L.fgb_make_divergence_free.argtypes = [vp, vp, vp, vp, i32, vp]
    L.fgb_sim_step.argtypes = [vp, vp, vp, vp, vp, f32, f32, C.POINTER(f32), f32, C.POINTER(Scalar), C.POINTER(i32), vp]
    L.fgb_column_sums.argtypes = [vp, vp, vp, i32, i32, vp, vp]
    L.fgb_update_outflow.argtypes = [vp, vp, vp, vp, C.POINTER(f32), f32, vp]
    L.fgb_flux_balance.argtypes = [vp, vp, vp, vp]
    L.fgb_balance_fluxes.argtypes = [vp, vp, vp, C.c_float, vp]
    L.fgb_max_velocity.argtypes = [vp, vp, vp, vp, vp]
    L.fgb_apply_jet_action.argtypes = [vp, vp, vp, vp, f32, vp, vp, i32, vp]
    L.fgb_wall_forces.argtypes = [vp, C.POINTER(Wall), vp, vp, vp, vp, vp]
    L.fgb_sample_sensors.argtypes = [vp, vp, i32, vp, vp, i32, i32, vp, vp]
    L.fgb_sample_sensors_n.argtypes = [vp, i32, i32, i32, vp, vp, i32, i32, vp, vp]
    L.fgb_render_gather.argtypes = [vp, i32, i32, i32, C.c_int64, C.c_int64, i32, vp, vp, vp, i32, vp, vp, vp]
    L.fgb_render_colour.argtypes = [vp, i32, i32, vp, f32, f32, i32, vp, vp, vp]
    L.fgb_profile_enable.argtypes = [vp, i32]
    L.fgb_profile_read.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_int64), i32]
    L.fgb_launch_count.argtypes = [vp]
    L.fgb_launch_count.restype = C.c_longlong
    L.fgb_velocity_gradients.argtypes = [vp, vp, vp, vp, vp]
    L.fgb_piso_substep_record.argtypes = [vp, vp, vp, vp, vp, C.POINTER(Tape), vp]
    L.fgb_adjoint_workspace_bytes.restype = C.c_size_t
    L.fgb_adjoint_workspace_bytes.argtypes = [C.POINTER(Tables), i32]
    L.fgb_piso_substep_backward.argtypes = [vp, C.POINTER(Tape), vp, vp, vp, vp, vp, vp, C.c_size_t, vp]
    L.fgb_piso_substep_record_scalar.argtypes = [vp, vp, vp, vp, vp, C.POINTER(Scalar), C.POINTER(Tape), C.POINTER(ScalarTape), vp]
    L.fgb_piso_substep_backward_scalar.argtypes = [vp, C.POINTER(Tape), C.POINTER(ScalarTape), f32, vp, vp, vp, vp, vp, vp, vp, vp, vp,
                                                   C.c_size_t, vp]
    L.fgb_ortho3_workspace_bytes.restype = C.c_size_t
    L.fgb_ortho3_workspace_bytes.argtypes = [C.POINTER(Ortho3Tables), i32]
    L.fgb_ortho3_create.argtypes = [C.POINTER(Ortho3Tables), i32, vp, C.c_size_t, C.POINTER(Options), C.POINTER(vp)]
    L.fgb_ortho3_destroy.argtypes = [vp]
    L.fgb_ortho3_destroy.restype = None
    L.fgb_ortho3_set_options.argtypes = [vp, C.POINTER(Options)]
    L.fgb_ortho3_buffer.restype = vp
    L.fgb_ortho3_buffer.argtypes = [vp, C.c_char_p]
    L.fgb_ortho3_launch_count.argtypes = [vp]
    L.fgb_ortho3_launch_count.restype = C.c_longlong
    L.fgb_ortho3_setup_advection.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    L.fgb_ortho3_solve_advection.argtypes = [vp, i32, vp, vp]
    L.fgb_ortho3_setup_pressure.argtypes = [vp, vp, vp, vp, vp, i32, vp, vp]
    L.fgb_ortho3_solve_pressure.argtypes = [vp, vp, i32, i32, i32, i32, vp, vp]
    L.fgb_ortho3_correct_velocity.argtypes = [vp, vp, vp, vp, vp]
    L.fgb_ortho3_piso_substep.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    L.fgb_ortho3_make_divergence_free.argtypes = [vp, vp, vp, vp, i32, vp]
    L.fgb_ortho3_sim_step.argtypes = [vp, vp, vp, vp, f32, f32, vp, i32, f32, f32, C.POINTER(i32), vp]
    L.fgb_ortho3_wall_rows.argtypes = [vp, vp, vp, i32, f32, f32, i32, vp, vp]
    L.fgb_ortho3_set_scalar.argtypes = [vp, C.POINTER(Ortho3Scalar)]
    L.fgb_ortho3_advect_scalar.argtypes = [vp, vp, vp, vp, vp, vp]
    L.fgb_ortho3_set_sgs.argtypes = [vp, f32, vp]
    L.fgb_ortho3_piso_substep_record.argtypes = [vp, vp, vp, vp, vp, vp, C.POINTER(Ortho3Tape), vp]
    L.fgb_ortho3_adjoint_workspace_bytes.argtypes = [C.POINTER(Ortho3Tables), i32]
    L.fgb_ortho3_adjoint_workspace_bytes.restype = C.c_size_t
    L.fgb_ortho3_piso_substep_backward.argtypes = [vp, C.POINTER(Ortho3Tape), vp, vp, vp, vp, vp, C.c_size_t, vp]
    L.fgb_ortho3_piso_substep_record_scalar.argtypes = [vp, vp, vp, vp, vp, vp, C.POINTER(Ortho3Tape), C.POINTER(ScalarTape), vp]
    L.fgb_ortho3_piso_substep_backward_scalar.argtypes = [vp, C.POINTER(Ortho3Tape), C.POINTER(ScalarTape), vp, vp, vp, vp, vp, vp, vp, vp, C.c_size_t, vp]
    L.fgb_ortho3_sgs_viscosity.argtypes = [vp, vp, vp, vp, vp]
    L.fgb_ortho3_velocity_gradients.argtypes = [vp, vp, vp, vp, vp]
    L.fgb_extruded3_piso_substep.argtypes = [vp, C.POINTER(Extruded3Tables), vp, vp, vp, vp, vp]
    L.fgb_extruded3_piso_substep_record.argtypes = [vp, C.POINTER(Extruded3Tables), vp, vp, vp, vp, C.POINTER(Tape), vp]
    L.fgb_extruded3_adjoint_workspace_bytes.argtypes = [C.POINTER(Extruded3Tables), i32]
    L.fgb_extruded3_adjoint_workspace_bytes.restype = C.c_size_t
    L.fgb_extruded3_piso_substep_backward.argtypes = [vp, C.POINTER(Extruded3Tables), C.POINTER(Tape), vp, vp, vp, vp, vp, vp, C.c_size_t, vp]
    L.fgb_extruded3_make_divergence_free.argtypes = [vp, C.POINTER(Extruded3Tables), vp, vp, vp, i32, vp]
    L.fgb_extruded3_balance_fluxes.argtypes = [C.POINTER(Extruded3Tables), i32, vp, vp, vp, f32, vp]
    L.fgb_extruded3_update_outflow.argtypes = [C.POINTER(Extruded3Tables), i32, vp, vp, vp, vp, vp, i32, vp, vp, vp, f32, vp]
    L.fgb_extruded3_max_velocity.argtypes = [C.POINTER(Extruded3Tables), i32, vp, vp, vp, vp]
    L.fgb_extruded3_apply_jets.argtypes = [C.POINTER(Extruded3Tables), i32, vp, vp, i32, vp, vp, i32, vp, vp, f32, vp]
    L.fgb_extruded3_wall_forces.argtypes = [C.POINTER(Extruded3Tables), i32, C.POINTER(Wall), vp, vp, vp, vp, vp]
    L.fgb_plan_substep.argtypes = [i32, vp, vp, f32, vp, vp, vp, vp, vp]
    L.fgb_ipc_alloc.argtypes = [C.c_size_t, C.POINTER(vp), C.c_char_p]
    L.fgb_ipc_open.argtypes = [C.c_char_p, C.POINTER(vp)]
    L.fgb_ipc_close.argtypes = [vp]
    L.fgb_ipc_free.argtypes = [vp]
    L.fgb_ortho3_set_slab.argtypes = [vp, i32, i32, vp, C.POINTER(vp)]
    L.fgb_ortho3_slab_error.argtypes = [vp, C.POINTER(i32)]
    _lib = L
    return L


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().fgb_last_error().decode()
        raise FGBError(f"{what}: error {rc}: {msg}")
