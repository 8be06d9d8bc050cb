"""ctypes binding of libgsb200.so (the C ABI declared in include/gsb200.h).

There is no CPU fallback: if the shared library is missing, or no CUDA device is
visible when a compute entry point is called, this module raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_int, c_longlong, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GSB200_LIB", os.path.join(_HERE, "libgsb200.so"))

GSB_OK, GSB_EINVAL, GSB_ENODEV, GSB_ECUDA, GSB_ENOMEM, GSB_ESTATE = 0, -1, -2, -3, -4, -5


class GsbError(RuntimeError):
    """A libgsb200 call failed (CUDA error, no device, out of memory)."""


class gsb_profile(ctypes.Structure):
    _fields_ = [("hmode", c_int), ("ped_p", c_double * 4), ("ped_ff", c_double * 4)]


class gsb_picard_params(ctypes.Structure):
    _fields_ = [
        ("max_iterations", c_int), ("tol", c_double), ("alpha", c_double), ("omega", c_double),
        ("method", c_int), ("require_gs_residual", c_int), ("gs_tol", c_double), ("saddle", c_int),
        ("mu0", c_double), ("z_min", c_double), ("r_min", c_double), ("r_max", c_double),
        ("seed", c_int), ("check_every", c_int), ("prof", gsb_profile), ("external_profile", c_int), ("anderson_depth", c_int),
    ]


class gsb_free_boundary_params(ctypes.Structure):
    _fields_ = [("max_outer_iter", c_int), ("tol", c_double), ("warm_j", c_int)]


class gsb_shape_params(ctypes.Structure):
    _fields_ = [("n_coils", c_int), ("coil_rz", POINTER(c_double)), ("n_points", c_int), ("points", POINTER(c_double)),
                ("alpha", c_double), ("isoflux", c_int), ("limits", POINTER(c_double))]


class gsb_probe_params(ctypes.Structure):
    _fields_ = [("n_coils", c_int), ("n_rows", c_int), ("response", POINTER(c_double)), ("sigma", POINTER(c_double)),
                ("alpha", c_double), ("limits", POINTER(c_double)), ("max_iter", c_int)]


class gsb_boundary_params(ctypes.Structure):
    _fields_ = [("n_coils", c_int), ("coil_rz", POINTER(c_double)), ("turns", POINTER(c_int)), ("n_points", c_int),
                ("points", POINTER(c_double)), ("n_limiter", c_int), ("limiter", POINTER(c_double)),
                ("has_axis", c_int), ("axis", POINTER(c_double)), ("n_xpoints", c_int), ("xpoints", POINTER(c_double)),
                ("per_sample", c_int), ("target_mode", c_int), ("nz", c_int), ("nr", c_int),
                ("r_axis", POINTER(c_double)), ("z_axis", POINTER(c_double))]


_dp = POINTER(c_double)
_ip = POINTER(c_int)

# name -> (restype, argtypes); every symbol include/gsb200.h declares
SIGNATURES = {
    # A. reference native ABI
    "create_solver": (c_void_p, [c_int, c_int, c_double, c_double, c_double, c_double]),
    "set_boundary_dirichlet": (None, [c_void_p, c_double]),
    "run_step": (None, [c_void_p, _dp, _dp, c_int, c_int]),
    "run_step_converged": (c_int, [c_void_p, _dp, _dp, c_int, c_int, c_double, c_double, _dp]),
    "destroy_solver": (None, [c_void_p]),
    "delete_solver": (None, [c_void_p]),
    # B. device API
    "gsb_abi_version": (c_int, []),
    "gsb_last_error": (c_char_p, []),
    "gsb_device_count": (c_int, []),
    "gsb_launch_count": (c_longlong, []),
    "gsb_debug_phase_cycles": (c_int, [POINTER(c_longlong), c_int]),
    "gsb_plan_levels": (c_int, [c_int, c_int, c_int, _ip, _ip, c_int]),
    "gsb_plan_level_tables": (c_int, [c_int, c_int, _dp, c_double, c_double, c_int, c_int, _dp, _dp, _dp, _dp]),
    "gsb_create": (c_int, [POINTER(c_void_p), c_int, c_int, _dp, _dp, c_double, c_double, c_int, c_int]),
    "gsb_destroy": (None, [c_void_p]),
    "gsb_smooth": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_double, c_int, c_int, c_void_p]),
    "gsb_smooth_ex": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_double, c_int, c_int, c_int, c_void_p]),
    "gsb_jacobi": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "gsb_jacobi_steps": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "gsb_residual": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "gsb_apply_operator": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "gsb_residual_norms": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "gsb_restrict_full_weight": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "gsb_prolong_bilinear": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "gsb_vcycle": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_double, c_int, c_int, c_int, c_void_p]),
    "gsb_mg_solve": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_double, c_int, c_double, c_int, c_int,
                             c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "gsb_topology": (c_int, [c_void_p, c_void_p, c_int, c_double, c_int, c_void_p, c_void_p]),
    "gsb_plasma_source": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_double, POINTER(gsb_profile),
                                  c_void_p, c_void_p, c_int, c_void_p]),
    "gsb_picard_solve": (c_int, [c_void_p, POINTER(gsb_picard_params), c_void_p, c_void_p, c_void_p, c_void_p,
                                 c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "gsb_picard_last_launched_iterations": (c_int, [c_void_p]),
    "gsb_timing": (c_int, [c_void_p, c_int, _dp, c_int]),
    "gsb_free_boundary_solve": (c_int, [c_void_p, POINTER(gsb_picard_params), POINTER(gsb_free_boundary_params), c_void_p,
                                        c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                        c_void_p]),
    "gsb_free_boundary_shape_solve": (c_int, [c_void_p, POINTER(gsb_picard_params), POINTER(gsb_free_boundary_params),
                                              POINTER(gsb_shape_params), c_void_p, _ip, c_void_p, c_void_p, c_void_p,
                                              c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                              c_void_p, c_int, c_void_p]),
    "gsb_probe_reconstruct": (c_int, [POINTER(gsb_probe_params), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                      c_void_p, c_void_p, POINTER(c_longlong), c_int, c_void_p]),
    "gsb_boundary_flux": (c_int, [POINTER(gsb_boundary_params), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_void_p, POINTER(c_longlong), c_int, c_void_p]),
    "gsb_enable_peer_access": (c_int, [c_int, c_int]),
    "gsb_ipc_alloc": (c_int, [c_int, c_longlong, POINTER(c_void_p), c_char_p]),
    "gsb_ipc_open": (c_int, [c_int, c_char_p, POINTER(c_void_p)]),
    "gsb_ipc_close": (c_int, [c_void_p]),
    "gsb_ipc_free": (c_int, [c_void_p]),
    "gsb_halo_push": (c_int, [c_void_p, c_void_p, c_longlong, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                              c_void_p, c_void_p]),
    "gsb_halo_recv": (c_int, [c_void_p, c_void_p, c_longlong, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                              c_void_p, c_void_p]),
    "gsb_gather_push": (c_int, [c_void_p, c_longlong, c_longlong, c_longlong, POINTER(c_void_p), POINTER(c_void_p), c_int, c_int,
                                c_void_p, c_void_p, c_void_p]),
    "gsb_gather_wait": (c_int, [c_void_p, c_longlong, c_void_p, c_int, c_longlong, c_void_p, c_void_p, c_void_p, c_void_p]),
    "gsb_slab_down": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int, c_double, c_int, c_void_p]),
    "gsb_slab_up": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_void_p, c_int, c_double, c_int, c_void_p]),
    "gsb_slab_single_tile": (c_int, [c_void_p, c_int]),
    "gsb_slab_smooth": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_double, c_int, c_int, c_void_p]),
    "gsb_slab_residual_restrict": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                           c_void_p]),
    "gsb_slab_prolong_add": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_int, c_void_p]),
    "gsb_slab_residual_linf": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "gsb_b_field": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "gsb_green_table": (c_int, [c_void_p, _dp, c_int, c_int, c_void_p, c_void_p]),
    "gsb_coil_flux": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_void_p]),
    "gsb_mutual_matrix": (c_int, [_dp, _ip, c_int, _dp, c_int, c_void_p, c_void_p]),
    "gsb_wall_matrix": (c_int, [c_void_p, c_double, c_void_p, c_void_p]),
    "gsb_wall_flux": (c_int, [c_void_p, c_void_p, c_void_p, c_double, c_void_p, c_int, c_void_p]),
    "gsb_wall_scatter": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
}

_lib = None


def load():
    """Load libgsb200.so and bind every declared symbol; raises if anything is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GsbError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C scpn_fusion_core_b200/csrc` (libgsb200 has no CPU fallback)"
        )
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.gsb_abi_version() != 1:
        raise GsbError("libgsb200 ABI version mismatch")
    _lib = lib
    return lib


def last_error() -> str:
    msg = load().gsb_last_error()
    return msg.decode() if msg else ""


def check(rc: int, what: str = "") -> None:
    """Map a gsb_* return code to the exception the reference raises for the same fault."""
    if rc == GSB_OK:
        return
    msg = last_error() or what
    if rc == GSB_EINVAL:
        raise ValueError(msg)
    if rc == GSB_ENOMEM:
        raise MemoryError(msg)
    raise GsbError(f"{what}: {msg}" if what else msg)


def require_device() -> int:
    n = load().gsb_device_count()
    if n <= 0:
        raise GsbError("no CUDA device visible: scpn_fusion_core_b200 has no CPU fallback")
    return n


def launch_count() -> int:
    return int(load().gsb_launch_count())
