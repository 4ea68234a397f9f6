"""ctypes binding of include/mpc_b200.h.

The product loads exactly one thing: the in-tree CUDA library ``libmpc_b200.so`` built by
``__graft_entry__.build()`` for sm_100a.  There is NO CPU fallback: if the library is missing,
or there is no CUDA device, :func:`cuda_backend` raises.

(tests/ inject a :class:`Backend` built around tests/emu's host compilation of the same source
to exercise the host logic in the GPU-less build container; nothing in this package refers to it.)
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MPCB_LIB", os.path.join(_HERE, "libmpc_b200.so"))   # MPCB_LIB: another build of the same CUDA library

MPCB_MAX_NX = 10
MPCB_MAX_NU = 2
MPCB_F32, MPCB_F64 = 0, 1

STATUS_STRING = {
    1: "solved",
    2: "solved inaccurate",
    3: "primal infeasible inaccurate",
    4: "dual infeasible inaccurate",
    -2: "maximum iterations reached",
    -3: "primal infeasible",
    -4: "dual infeasible",
    -7: "problem non convex",
    -10: "unsolved",
}


class Problem(C.Structure):
    _fields_ = [("horizon", C.c_int), ("nx", C.c_int), ("nu", C.c_int), ("slack", C.c_int), ("dtype", C.c_int),
                ("time_varying", C.c_int), ("shared_model", C.c_int), ("stage_reference", C.c_int),
                ("Q", C.c_double * MPCB_MAX_NX), ("QN", C.c_double * MPCB_MAX_NX), ("R", C.c_double * MPCB_MAX_NU),
                ("W", C.c_double * MPCB_MAX_NX), ("S", C.c_double * MPCB_MAX_NX),
                ("xmin", C.c_double * MPCB_MAX_NX), ("xmax", C.c_double * MPCB_MAX_NX),
                ("umin", C.c_double * MPCB_MAX_NU), ("umax", C.c_double * MPCB_MAX_NU)]


class Settings(C.Structure):
    _fields_ = [("rho", C.c_double), ("sigma", C.c_double), ("alpha", C.c_double), ("eps_abs", C.c_double),
                ("eps_rel", C.c_double), ("eps_prim_inf", C.c_double), ("eps_dual_inf", C.c_double),
                ("max_iter", C.c_int), ("scaling", C.c_int), ("check_termination", C.c_int),
                ("warm_start", C.c_int)]


class MpcError(RuntimeError):
    pass


_VOIDP = C.c_void_p
_SIGNATURES = {
    "mpcb_last_error": (C.c_char_p, []),
    "mpcb_version": (C.c_int, []),
    "mpcb_default_settings": (None, [C.POINTER(Settings)]),
    "mpcb_create": (C.c_int, [C.POINTER(Problem), C.POINTER(Settings), C.c_int, C.POINTER(_VOIDP)]),
    "mpcb_destroy": (None, [_VOIDP]),
    "mpcb_set_settings": (C.c_int, [_VOIDP, C.POINTER(Settings)]),
    "mpcb_set_stage_bounds": (C.c_int, [_VOIDP, C.POINTER(C.c_double)]),
    "mpcb_workspace_bytes": (C.c_size_t, [_VOIDP]),
    "mpcb_num_variables": (C.c_int, [_VOIDP]),
    "mpcb_num_constraints": (C.c_int, [_VOIDP]),
    "mpcb_setup": (C.c_int, [_VOIDP, C.c_int, C.c_size_t, _VOIDP, _VOIDP, _VOIDP, _VOIDP, _VOIDP, _VOIDP]),
    "mpcb_update": (C.c_int, [_VOIDP, _VOIDP, _VOIDP]),
    "mpcb_update_bounds": (C.c_int, [_VOIDP, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double),
                                     C.POINTER(C.c_double), C.POINTER(C.c_double), _VOIDP]),
    "mpcb_solve": (C.c_int, [_VOIDP, _VOIDP]),
    "mpcb_iterate": (C.c_int, [_VOIDP, C.c_int, _VOIDP]),
    "mpcb_cold_start": (C.c_int, [_VOIDP, _VOIDP]),
    "mpcb_get_solution": (C.c_int, [_VOIDP, _VOIDP, _VOIDP, _VOIDP, _VOIDP]),
    "mpcb_get_info": (C.c_int, [_VOIDP, _VOIDP, _VOIDP, _VOIDP, _VOIDP, _VOIDP]),
    "mpcb_solve_host": (C.c_int, [_VOIDP, C.c_int, _VOIDP, _VOIDP, _VOIDP, _VOIDP, _VOIDP, _VOIDP, _VOIDP, _VOIDP, _VOIDP]),
    "mpcb_lateral_discretize": (C.c_int, [C.c_int, C.c_int, C.c_size_t, _VOIDP, C.POINTER(C.c_double), _VOIDP, _VOIDP, _VOIDP]),
    "mpcb_dynamics_linearize": (C.c_int, [C.c_int, C.c_int, C.c_size_t, _VOIDP, _VOIDP, C.POINTER(C.c_double), _VOIDP, _VOIDP, _VOIDP, _VOIDP]),
    "mpcb_kinematics_linearize": (C.c_int, [C.c_int, C.c_int, C.c_size_t, _VOIDP, _VOIDP, C.POINTER(C.c_double), _VOIDP, _VOIDP, _VOIDP, _VOIDP]),
    "mpcb_dynamics_step": (C.c_int, [C.c_int, C.c_int, C.c_size_t, _VOIDP, _VOIDP, C.POINTER(C.c_double), _VOIDP, _VOIDP, _VOIDP]),
    "mpcb_kinematics_step": (C.c_int, [C.c_int, C.c_int, C.c_size_t, _VOIDP, _VOIDP, C.POINTER(C.c_double), _VOIDP, _VOIDP]),
    "mpcb_augment_increment": (C.c_int, [C.c_int, C.c_int, C.c_size_t, C.c_int, C.c_int, C.c_int, _VOIDP, _VOIDP, _VOIDP, _VOIDP, _VOIDP, _VOIDP, _VOIDP]),
    "mpcb_plant_step": (C.c_int, [C.c_int, C.c_int, C.c_size_t, C.c_int, C.c_int, C.c_int, _VOIDP, _VOIDP, _VOIDP, _VOIDP, _VOIDP,
                                  C.c_int, _VOIDP, _VOIDP]),
    "mpcb_build_qp": (C.c_int, [_VOIDP, _VOIDP, _VOIDP, _VOIDP, _VOIDP, _VOIDP, _VOIDP]),
    "mpcb_get_scaling": (C.c_int, [_VOIDP, _VOIDP, _VOIDP, _VOIDP, _VOIDP]),
    "mpcb_qp_pattern": (C.c_int, [_VOIDP, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "mpcb_to_element_major": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_size_t, _VOIDP, _VOIDP, _VOIDP]),
    "mpcb_to_batch_major": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_size_t, _VOIDP, _VOIDP, _VOIDP]),
    "mpcb_set_option": (C.c_int, [C.c_char_p, C.c_int]),
    "mpcb_launch_count": (C.c_longlong, []),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)


class Backend:
    """A loaded libmpc_b200 plus the torch device its pointers live on."""

    def __init__(self, cdll, device):
        self.lib = cdll
        self.device = torch.device(device)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(cdll, name)
            fn.restype = res
            fn.argtypes = args

    def check(self, rc):
        if rc != 0:
            raise MpcError("mpc_b200 error %d: %s" % (rc, self.lib.mpcb_last_error().decode()))

    def stream(self):
        if self.device.type == "cuda":
            return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        return C.c_void_p(0)

    def set_option(self, name, value):
        """Process-wide tunables of the library: "tma", "retile", "retile_min_batch" (include/mpc_b200.h)."""
        self.check(self.lib.mpcb_set_option(name.encode(), int(value)))

    def launch_count(self):
        return int(self.lib.mpcb_launch_count())


_cuda = {}        # one Backend per CUDA device (the library handle is shared; device pointers and streams are per device)
_cdll = None


def cuda_backend(device=None):
    """The product backend of a CUDA device (default: torch's current device at the time of the call).  Fails loudly;
    never substitutes anything for the CUDA library."""
    global _cdll
    if not os.path.exists(LIB_PATH):
        raise MpcError("%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                       "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
    if not torch.cuda.is_available():
        raise MpcError("mpc_b200 needs a CUDA device (B200, sm_100a); none is visible and there is no CPU fallback.")
    idx = torch.cuda.current_device() if device is None else torch.device(device).index
    be = _cuda.get(idx)
    if be is None:
        if _cdll is None:
            _cdll = C.CDLL(LIB_PATH)
        be = _cuda[idx] = Backend(_cdll, torch.device("cuda", idx))
    return be


def ptr(t):
    """Device/host pointer of a tensor (or NULL)."""
    return C.c_void_p(0) if t is None else C.c_void_p(t.data_ptr())
