"""GPU drop-in for the reference's ``FusionKernel`` equilibrium entry points.

Mirrors the solver surface of ``src/scpn_fusion/core/fusion_kernel.py`` (reference) and its
mixins for the Grad-Shafranov hot path: same constructor (JSON config path), same attributes
(``Psi, J_phi, R, Z, RR, ZZ, NR, NZ, dR, dZ, cfg, B_R, B_Z``), same method names, argument
meaning, result-dict keys and error behaviour.  Every numerical step runs in libgsb200 kernels
(``csrc/``); host code only marshals buffers.  A ``BatchedFusionKernel`` runs B independent
equilibria (UQ / design sweeps) through the same kernels in one launch sequence.

The free-boundary layer (coil Green's functions, shape optimisation, probe reconstruction) lives in
``free_boundary.py``.  Out of scope here (SURVEY.md 8f): ``solver_method`` in {"newton", "rust_multigrid"} raises
``NotImplementedError`` ("anderson" - SOR sweep + Anderson mixing - runs on the device since r2).
"""
from __future__ import annotations

import ctypes
import json
import logging
import math
import time
from dataclasses import dataclass, field
from pathlib import Path
from typing import Any

import numpy as np

from . import _device as D
from . import _lib
from .free_boundary import FreeBoundaryMixin
_mg = __import__("importlib").import_module(__package__ + ".multigrid_solve")  # package re-exports a same-named function

logger = logging.getLogger(__name__)

MAX_CONFIG_BYTES = 10 * 1024 * 1024
_METHODS = {"multigrid": 0, "sor": 1, "jacobi": 2, "anderson": 3}
_PED_KEYS = ("ped_top", "ped_width", "ped_height", "core_alpha")
_MU0_SI = 4e-7 * np.pi


@dataclass
class CoilSet:
    """External coil set (reference: fusion_kernel.py:60-101)."""

    positions: list = field(default_factory=list)
    currents: np.ndarray = field(default_factory=lambda: np.array([]))
    turns: list = field(default_factory=list)
    current_limits: np.ndarray | None = None
    target_flux_points: np.ndarray | None = None
    target_flux_values: np.ndarray | None = None
    x_point_target: np.ndarray | None = None
    x_point_flux_target: float | None = None
    divertor_strike_points: np.ndarray | None = None
    divertor_flux_values: np.ndarray | None = None


# ---------------------------------------------------------------------------------------------
# configuration (reference: config_schema.py:16-102; same constraints, same defaults)
# ---------------------------------------------------------------------------------------------

def _finite(x, name):
    v = float(x)
    if not math.isfinite(v):
        raise ValueError(f"{name} must be finite")
    return v


def validate_config(raw: dict[str, Any]) -> dict[str, Any]:
    """Validate a reference-style reactor config dict and fill the reference's defaults."""
    if not isinstance(raw, dict):
        raise ValueError("configuration must be a JSON object")
    cfg = json.loads(json.dumps(raw))  # deep copy, JSON types only
    cfg.setdefault("reactor_name", "Unnamed-Reactor")
    if "dimensions" not in cfg:
        raise ValueError("dimensions: field required")
    d = cfg["dimensions"]
    for k in ("R_min", "R_max", "Z_min", "Z_max"):
        if k not in d:
            raise ValueError(f"dimensions.{k}: field required")
        d[k] = _finite(d[k], f"dimensions.{k}")
    if d["R_min"] <= 0 or d["R_max"] <= 0:
        raise ValueError("dimensions.R_min / R_max must be > 0")
    if d["R_max"] <= d["R_min"]:
        raise ValueError("R_max must be greater than R_min")
    res = cfg.get("grid_resolution", (129, 129))
    if len(res) != 2:
        raise ValueError("grid_resolution must have two entries")
    res = [int(res[0]), int(res[1])]
    if res[0] < 4 or res[1] < 4:
        raise ValueError("Grid resolution must be at least 4x4")
    cfg["grid_resolution"] = res
    coils = cfg.get("coils", [])
    for i, c in enumerate(coils):
        if "r" not in c or "z" not in c:
            raise ValueError(f"coils[{i}] must define r and z")
        c.setdefault("name", "unnamed")
        c["r"] = _finite(c["r"], f"coils[{i}].r")
        c["z"] = _finite(c["z"], f"coils[{i}].z")
        c["current"] = _finite(c.get("current", 0.0), f"coils[{i}].current")
        if c["r"] <= 0:
            raise ValueError(f"coils[{i}].r must be > 0")
    cfg["coils"] = coils
    ph = cfg.setdefault("physics", {})
    ph["plasma_current_target"] = _finite(ph.get("plasma_current_target", 5.0), "plasma_current_target")
    ph["vacuum_permeability"] = _finite(ph.get("vacuum_permeability", 1.25663706e-6), "vacuum_permeability")
    if ph["vacuum_permeability"] < 0:
        raise ValueError("physics.vacuum_permeability must be >= 0")
    so = cfg.setdefault("solver", {})
    so["max_iterations"] = int(so.get("max_iterations", 1000))
    so["convergence_threshold"] = _finite(so.get("convergence_threshold", 1e-4), "convergence_threshold")
    so["relaxation_factor"] = _finite(so.get("relaxation_factor", 0.1), "relaxation_factor")
    if so["max_iterations"] <= 0:
        raise ValueError("solver.max_iterations must be > 0")
    if so["convergence_threshold"] <= 0:
        raise ValueError("solver.convergence_threshold must be > 0")
    if not (0 < so["relaxation_factor"] <= 1.0):
        raise ValueError("solver.relaxation_factor must be in (0, 1]")
    return cfg


def _measurement_rows(value, name: str, length: int) -> np.ndarray:
    """(B, length) float64 rows of a batched measurement argument; a 1-D vector is a batch of one."""
    a = np.asarray(value, dtype=np.float64)
    if a.ndim == 1:
        a = a[None, :]
    if a.ndim != 2 or a.shape[1] != length or a.shape[0] < 1:
        raise ValueError(f"{name} must have length {length}.")
    if not np.all(np.isfinite(a)):
        raise ValueError(f"{name} must contain finite values only.")
    return a


def _load_config(src) -> dict[str, Any]:
    if isinstance(src, dict):
        return validate_config(src)
    p = Path(src)
    if p.stat().st_size > MAX_CONFIG_BYTES:
        raise ValueError(f"configuration file exceeds {MAX_CONFIG_BYTES} byte limit: {p}")
    with open(p, "r", encoding="utf-8") as f:
        return validate_config(json.load(f))


def _profile_struct(hmode: bool, ped_p: dict, ped_ff: dict) -> _lib.gsb_profile:
    s = _lib.gsb_profile()
    s.hmode = 1 if hmode else 0
    for i, k in enumerate(_PED_KEYS):
        s.ped_p[i] = float(ped_p[k])
        s.ped_ff[i] = float(ped_ff[k])
    return s


class _GridMixin:
    """Grid + profile state shared by the single and the batched kernel (fusion_kernel.py:158-200)."""

    def _init_grid(self) -> None:
        dims = self.cfg["dimensions"]
        res = self.cfg["grid_resolution"]
        self.NR, self.NZ = int(res[0]), int(res[1])
        self.R = np.linspace(dims["R_min"], dims["R_max"], self.NR)
        self.Z = np.linspace(dims["Z_min"], dims["Z_max"], self.NZ)
        self.dR = float(self.R[1] - self.R[0])
        self.dZ = float(self.Z[1] - self.Z[0])
        self.RR, self.ZZ = np.meshgrid(self.R, self.Z)
        for stale in ("_green_cache", "_wall_m_cache", "_fb_ext"):  # device tables of the previous grid
            self.__dict__.pop(stale, None)
        self.profile_mode = "l-mode"
        self.ped_params_p = {"ped_top": 0.92, "ped_width": 0.05, "ped_height": 1.0, "core_alpha": 0.3}
        self.ped_params_ff = dict(self.ped_params_p)
        prof = self.cfg.get("physics", {}).get("profiles")
        if prof:
            self.profile_mode = prof.get("mode", "l-mode")
            if "p_prime" in prof:
                self.ped_params_p.update(prof["p_prime"])
            if "ff_prime" in prof:
                self.ped_params_ff.update(prof["ff_prime"])

    @property
    def _hmode(self) -> bool:
        return self.profile_mode in ("h-mode", "H-mode", "hmode")

    def _context(self, batch: int) -> D.Context:
        return D.get_context(self.NZ, self.NR, self.R, self.Z, self.dR, self.dZ, batch, self.device)

    def _picard_params(self) -> _lib.gsb_picard_params:
        so = self.cfg["solver"]
        method = so.get("solver_method", "multigrid")
        if method not in _METHODS:
            raise NotImplementedError(
                f"solver_method {method!r} is outside the B200 hot path (supported: {sorted(_METHODS)})")
        p = _lib.gsb_picard_params()
        p.max_iterations = int(so["max_iterations"])
        p.tol = float(so["convergence_threshold"])
        p.alpha = float(so.get("relaxation_factor", 0.1))
        p.omega = _mg.validate_sor_omega(so.get("sor_omega", 1.6))
        p.method = _METHODS[method]
        p.require_gs_residual = 1 if bool(so.get("require_gs_residual", False)) else 0
        p.gs_tol = float(so.get("gs_residual_threshold", p.tol))
        if p.require_gs_residual and p.gs_tol <= 0.0:
            raise ValueError("solver.gs_residual_threshold must be > 0")
        p.saddle = 1 if bool(so.get("xpoint_use_saddle_detection", False)) else 0
        p.mu0 = float(self.cfg["physics"]["vacuum_permeability"])
        d = self.cfg["dimensions"]
        p.z_min, p.r_min, p.r_max = float(d["Z_min"]), float(d["R_min"]), float(d["R_max"])
        p.seed = 1
        p.check_every = int(so.get("gpu_check_every", 8))
        p.prof = _profile_struct(self._hmode, self.ped_params_p, self.ped_params_ff)
        p.external_profile = 1 if bool(getattr(self, "external_profile_mode", False)) else 0
        p.anderson_depth = 0
        if method == "anderson":  # fusion_kernel_newton_solver.py:481; a depth below 2 never mixes (mk < 2)
            depth = int(so.get("anderson_depth", 5))
            if depth > 8:
                raise NotImplementedError("solver.anderson_depth > 8 is outside the B200 hot path")
            p.anderson_depth = max(depth, 1)
        return p

    # Green's tables are geometry-only: build once per (coil set, flavour)
    def _green_table(self, positions, si: int):
        key = (tuple((float(r), float(z)) for r, z in positions), int(si))
        cache = self.__dict__.setdefault("_green_cache", {})
        if key not in cache:
            ctx = self._context(1)
            nc = len(positions)
            rz = np.ascontiguousarray(np.asarray(positions, dtype=np.float64).reshape(nc, 2))
            g = D.empty((nc, 1 if si else 2, self.NZ, self.NR), self.device)
            _lib.check(ctx.lib.gsb_green_table(ctx.handle, D.np_ptr(rz), nc, int(si), D.ptr(g), D.stream_ptr()),
                       "gsb_green_table")
            cache[key] = g
        return cache[key]

    def _coil_flux_dev(self, positions, weights: np.ndarray, si: int):
        """psi[b] = sum_c w[b,c]*G_c on the device; weights: host (B, n_coils)."""
        w = np.ascontiguousarray(np.atleast_2d(np.asarray(weights, dtype=np.float64)))
        B, nc = w.shape
        out = D.empty((B, self.NZ, self.NR), self.device)
        if nc == 0:
            out.zero_()
            return out
        ctx = self._context(B)
        g = self._green_table(positions, si)
        wd = D.to_device(w, self.device)
        _lib.check(ctx.lib.gsb_coil_flux(ctx.handle, D.ptr(g), D.ptr(wd), nc, int(si), D.ptr(out), B, D.stream_ptr()),
                   "gsb_coil_flux")
        return out


class FusionKernel(FreeBoundaryMixin, _GridMixin):
    """Non-linear Grad-Shafranov equilibrium solver on one B200 (reference: fusion_kernel.py:104)."""

    def __init__(self, config_path, device: int | None = None) -> None:
        self._config_path = str(config_path) if not isinstance(config_path, dict) else "<dict>"
        self.device = D.current_device() if device is None else int(device)
        self.load_config(config_path)
        self.initialize_grid()
        self.external_profile_mode = False

    # -- construction ------------------------------------------------------------------
    def load_config(self, path) -> None:
        self.cfg = _load_config(path)
        logger.info("Loaded configuration for: %s", self.cfg["reactor_name"])

    def initialize_grid(self) -> None:
        self._init_grid()
        self.Psi = np.zeros((self.NZ, self.NR))
        self.J_phi = np.zeros((self.NZ, self.NR))
        self.B_R = np.zeros((self.NZ, self.NR))
        self.B_Z = np.zeros((self.NZ, self.NR))
        self.p_prime_0 = -1.0
        self.ff_prime_0 = -1.0

    # -- vacuum field (a15) ---------------------------------------------------------------
    def calculate_vacuum_field(self) -> np.ndarray:
        """fusion_kernel.py:218-251 on the device (Cephes K/E kernel)."""
        mu0 = self.cfg["physics"].get("vacuum_permeability", 1.0)
        coils = self.cfg["coils"]
        if not coils:
            return np.zeros((self.NZ, self.NR))
        pos = [(c["r"], c["z"]) for c in coils]
        w = np.array([[(mu0 * c["current"]) / (2.0 * np.pi) for c in coils]])
        return self._coil_flux_dev(pos, w, 0)[0].cpu().numpy()

    # -- topology (a10, a11) ----------------------------------------------------------------
    def _topology(self, Psi) -> np.ndarray:
        ctx = self._context(1)
        p = D.to_device(np.asarray(Psi, dtype=np.float64).reshape(1, self.NZ, self.NR), self.device)
        out = D.empty((1, 8), self.device)
        saddle = 1 if bool(self.cfg.get("solver", {}).get("xpoint_use_saddle_detection", False)) else 0
        _lib.check(ctx.lib.gsb_topology(ctx.handle, D.ptr(p), 1, float(self.cfg["dimensions"]["Z_min"]), saddle,
                                        D.ptr(out), D.stream_ptr()), "gsb_topology")
        return out.cpu().numpy()[0]

    def find_x_point(self, Psi):
        """fusion_kernel.py:255-340: ``((R_x, Z_x), Psi_x)``."""
        raw = np.asarray(Psi, dtype=np.float64)
        fin = np.isfinite(raw)
        if fin.all():
            t = self._topology(raw)
            if t[6] == 0.0:
                return (0.0, 0.0), float(t[7])
            return (float(self.R[int(t[4])]), float(self.Z[int(t[3])])), float(t[5])
        # non-finite entries (:269-273): the search runs on nan_to_num(psi); the reported flux is the raw value
        # at the chosen point when that is finite, else the sanitised one; the fallback is the finite minimum
        if not fin.any():
            return (0.0, 0.0), 0.0
        safe = np.nan_to_num(raw, nan=0.0, posinf=1e300, neginf=-1e300)
        t = self._topology(safe)
        if t[6] == 0.0:
            return (0.0, 0.0), float(np.min(raw[fin]))
        iz, ir = int(t[3]), int(t[4])
        px = float(raw[iz, ir]) if np.isfinite(raw[iz, ir]) else float(safe[iz, ir])
        return (float(self.R[ir]), float(self.Z[iz])), px

    def _find_magnetic_axis(self):
        """fusion_kernel.py:342-355: ``(iz, ir, Psi_axis)``."""
        t = self._topology(self.Psi)
        return int(t[0]), int(t[1]), float(t[2])

    # -- source (a12) ------------------------------------------------------------------------
    def update_plasma_source_nonlinear(self, Psi_axis: float, Psi_boundary: float) -> np.ndarray:
        """fusion_kernel.py:394-444."""
        ctx = self._context(1)
        p = D.to_device(self.Psi.reshape(1, self.NZ, self.NR), self.device)
        ab = D.to_device(np.array([[float(Psi_axis), float(Psi_boundary)]]), self.device)
        ip = D.to_device(np.array([float(self.cfg["physics"]["plasma_current_target"])]), self.device)
        j = D.empty((1, self.NZ, self.NR), self.device)
        prof = _profile_struct(self._hmode, self.ped_params_p, self.ped_params_ff)
        _lib.check(ctx.lib.gsb_plasma_source(ctx.handle, D.ptr(p), D.ptr(ab), D.ptr(ip),
                                             float(self.cfg["physics"]["vacuum_permeability"]), ctypes.byref(prof),
                                             ctypes.c_void_p(), D.ptr(j), 1, D.stream_ptr()), "gsb_plasma_source")
        self.J_phi = j[0].cpu().numpy()
        return self.J_phi

    # -- elliptic sub-solvers (a2, a3, a8) -----------------------------------------------------
    @staticmethod
    def _validate_sor_omega(omega: float) -> float:
        return _mg.validate_sor_omega(omega)

    def _jacobi_step(self, Psi, Source) -> np.ndarray:
        ctx = self._context(1)
        p = D.to_device(np.asarray(Psi, dtype=np.float64).reshape(1, self.NZ, self.NR), self.device)
        s = D.to_device(np.asarray(Source, dtype=np.float64).reshape(1, self.NZ, self.NR), self.device)
        out = D.empty((1, self.NZ, self.NR), self.device)
        _lib.check(ctx.lib.gsb_jacobi(ctx.handle, D.ptr(p), D.ptr(s), D.ptr(out), 1, D.stream_ptr()), "gsb_jacobi")
        return out[0].cpu().numpy()

    def _sor_step(self, Psi, Source, omega: float = 1.6) -> np.ndarray:
        omega = _mg.validate_sor_omega(omega)
        ctx = self._context(1)
        torch = D.torch_mod()
        p = D.to_device(np.asarray(Psi, dtype=np.float64).reshape(1, self.NZ, self.NR), self.device)
        s = D.to_device(np.asarray(Source, dtype=np.float64).reshape(1, self.NZ, self.NR), self.device)
        # _sanitize_numeric_array (fusion_kernel_numerics.py:19-24) before the clipped sweep
        p = torch.nan_to_num(p, nan=0.0, posinf=1e250, neginf=-1e250).clamp_(-1e250, 1e250)
        s = torch.nan_to_num(s, nan=0.0, posinf=1e250, neginf=-1e250).clamp_(-1e250, 1e250)
        _lib.check(ctx.lib.gsb_smooth(ctx.handle, D.ptr(p), D.ptr(s), 1, omega, 1, 1, D.stream_ptr()), "gsb_smooth")
        return p[0].cpu().numpy()

    _restrict_full_weight = staticmethod(_mg.restrict_full_weight)
    _prolongate_bilinear = staticmethod(_mg.prolongate_bilinear)

    def _mg_smooth(self, Psi, Source, R_grid, dR, dZ, omega, n_sweeps):
        return _mg.mg_smooth(Psi, Source, R_grid, dR, dZ, omega, n_sweeps)

    def _mg_residual(self, Psi, Source, R_grid, dR, dZ):
        return _mg.mg_residual(Psi, Source, R_grid, dR, dZ)

    def _multigrid_vcycle(self, Psi, Source, R_grid, dR, dZ, *, omega=1.6, pre_smooth=3, post_smooth=3, min_grid=5):
        return _mg.multigrid_vcycle(Psi, Source, R_grid, dR, dZ, omega=omega, pre_smooth=pre_smooth,
                                    post_smooth=post_smooth, min_grid=min_grid)

    def _apply_boundary_conditions(self, Psi, Psi_bc) -> None:
        Psi[0, :] = Psi_bc[0, :]
        Psi[-1, :] = Psi_bc[-1, :]
        Psi[:, 0] = Psi_bc[:, 0]
        Psi[:, -1] = Psi_bc[:, -1]

    def _compute_gs_residual_rms(self, Source) -> float:
        ctx = self._context(1)
        p = D.to_device(self.Psi.reshape(1, self.NZ, self.NR), self.device)
        s = D.to_device(np.asarray(Source, dtype=np.float64).reshape(1, self.NZ, self.NR), self.device)
        rms = D.empty((1,), self.device)
        _lib.check(ctx.lib.gsb_residual_norms(ctx.handle, D.ptr(p), D.ptr(s), ctypes.c_void_p(), D.ptr(rms), 1,
                                              D.stream_ptr()), "gsb_residual_norms")
        return float(rms.cpu().numpy()[0])

    # -- main solver (a13, a14) ----------------------------------------------------------------
    def _prepare_initial_flux(self, preserve_initial_state: bool, boundary_flux):
        """fusion_kernel_iterative_solver.py:412-451."""
        if boundary_flux is not None:
            bc = np.asarray(boundary_flux, dtype=np.float64)
            if bc.shape != self.Psi.shape:
                raise ValueError(f"boundary_flux shape {bc.shape} must match Psi shape {self.Psi.shape}")
            bc = bc.copy()
        elif preserve_initial_state:
            bc = self.Psi.copy()
        else:
            bc = self.calculate_vacuum_field()
        if preserve_initial_state:
            self._apply_boundary_conditions(self.Psi, bc)
        else:
            self.Psi = bc.copy()
        return bc

    def solve_equilibrium(self, preserve_initial_state: bool = False, boundary_flux=None) -> dict[str, Any]:
        """fusion_kernel_newton_solver.py:390-615 (Picard loop on the device)."""
        t0 = time.time()
        method = self.cfg["solver"].get("solver_method", "multigrid")
        params = self._picard_params()
        ip_target = float(self.cfg["physics"]["plasma_current_target"])
        if abs(ip_target) < 1e-12 and not preserve_initial_state:
            self.Psi = self.calculate_vacuum_field()
            self.J_phi = np.zeros_like(self.Psi)
            self.compute_b_field()
            return {"psi": self.Psi, "converged": True, "iterations": 0, "residual": 0.0, "residual_history": [],
                    "gs_residual": 0.0, "gs_residual_best": 0.0, "gs_residual_history": [],
                    "wall_time_s": time.time() - t0, "solver_method": method}
        bc = self._prepare_initial_flux(preserve_initial_state, boundary_flux)
        out = _picard_run(self, params, self.Psi[None], bc[None], np.array([ip_target]), None, want_history=True)
        self.Psi = out["psi"][0]
        self.J_phi = out["j_phi"][0]
        s = out["summary"][0]
        iters = int(s[0])
        if int(s[5]) == 3 and bool(self.cfg["solver"].get("fail_on_diverge", False)):
            raise RuntimeError(f"Equilibrium solver diverged at iter={iters - 1}")
        n_hist = iters - (1 if int(s[5]) == 3 else 0)
        hist = [float(v) for v in out["hist"][0][:n_hist]]
        gs_hist = [float(v) for v in out["gs_hist"][0][:n_hist]]
        self._last_topology = s[6:12].copy()
        self.compute_b_field()
        if gs_hist:
            gs_final, gs_best = gs_hist[-1], float(s[4])
        else:
            # diverged in the very first iteration: the reference reports the GS RMS of the reverted state against
            # the last source it formed (fusion_kernel_newton_solver.py:584-590, `final_source`)
            mu0 = float(self.cfg["physics"]["vacuum_permeability"])
            gs_final = gs_best = self._compute_gs_residual_rms(-mu0 * self.RR * self.J_phi)
        return {"psi": self.Psi, "converged": bool(s[1]), "iterations": iters, "residual": float(s[2]),
                "residual_history": hist,
                "gs_residual": gs_final,
                "gs_residual_best": gs_best,
                "gs_residual_history": gs_hist, "wall_time_s": time.time() - t0, "solver_method": method}

    # -- post-processing -----------------------------------------------------------------------
    def compute_b_field(self) -> None:
        """fusion_kernel.py:450-456."""
        ctx = self._context(1)
        p = D.to_device(self.Psi.reshape(1, self.NZ, self.NR), self.device)
        br = D.empty((1, self.NZ, self.NR), self.device)
        bz = D.empty((1, self.NZ, self.NR), self.device)
        _lib.check(ctx.lib.gsb_b_field(ctx.handle, D.ptr(p), D.ptr(br), D.ptr(bz), 1, D.stream_ptr()), "gsb_b_field")
        self.B_R, self.B_Z = br[0].cpu().numpy(), bz[0].cpu().numpy()

    def save_results(self, filename: str = "equilibrium_nonlinear.npz") -> None:
        np.savez(filename, R=self.R, Z=self.Z, Psi=self.Psi, J_phi=self.J_phi)

    # -- free boundary (a16, a17) ------------------------------------------------------------------
    def build_coilset_from_config(self) -> CoilSet:
        """fusion_kernel_coilset_config.py:33-156 (positions, currents, integer turns)."""
        pos, cur, turns = [], [], []
        for i, c in enumerate(self.cfg.get("coils", [])):
            r, z, cu = float(c["r"]), float(c["z"]), float(c.get("current", 0.0))
            if not (math.isfinite(r) and r > 0 and math.isfinite(z) and math.isfinite(cu)):
                raise ValueError(f"coils[{i}] must define finite r > 0, finite z, and current.")
            t = c.get("turns", 1)
            if isinstance(t, bool) or int(t) < 1 or float(int(t)) != float(t):
                raise ValueError(f"coils[{i}].turns must be a positive integer.")
            pos.append((r, z))
            cur.append(cu)
            turns.append(int(t))
        fb = self.cfg.get("free_boundary") or {}
        cs = CoilSet(positions=pos, currents=np.asarray(cur, dtype=np.float64), turns=turns)
        for k in ("current_limits", "target_flux_points", "target_flux_values", "x_point_target",
                  "divertor_strike_points", "divertor_flux_values"):
            if fb.get(k) is not None:
                setattr(cs, k, np.asarray(fb[k], dtype=np.float64))
        if fb.get("x_point_flux_target") is not None:
            cs.x_point_flux_target = float(fb["x_point_flux_target"])
        return cs

    # _compute_external_flux, _build_mutual_inductance_matrix, optimize_coil_currents, solve_free_boundary and the
    # coil diagnostics come from FreeBoundaryMixin (free_boundary.py)


def _picard_run(k: _GridMixin, params, psi0: np.ndarray, bc: np.ndarray, ip: np.ndarray, ped, *,
                want_history: bool, keep_on_device: bool = False) -> dict[str, Any]:
    """Marshal one gsb_picard_solve call: host (or device) buffers in, results out."""
    torch = D.torch_mod()
    B = int(psi0.shape[0])
    ctx = k._context(B)
    psi = D.to_device(psi0, k.device)
    bcd = psi if bc is None else D.to_device(bc, k.device)  # ring is saved before psi is touched
    ipd = D.to_device(np.asarray(ip, dtype=np.float64).reshape(B), k.device)
    pedd = None if ped is None else D.to_device(np.asarray(ped, dtype=np.float64).reshape(B, 8), k.device)
    jphi = D.empty((B, k.NZ, k.NR), k.device)
    summ = D.empty((B, 16), k.device)
    hist = gsh = None
    if want_history:
        hist = D.zeros((B, params.max_iterations), k.device)
        gsh = D.zeros((B, params.max_iterations), k.device)
    null = ctypes.c_void_p()
    _lib.check(ctx.lib.gsb_picard_solve(ctx.handle, ctypes.byref(params), D.ptr(psi), D.ptr(bcd), D.ptr(ipd),
                                        null if pedd is None else D.ptr(pedd), D.ptr(jphi), D.ptr(summ),
                                        null if hist is None else D.ptr(hist), null if gsh is None else D.ptr(gsh),
                                        B, D.stream_ptr()), "gsb_picard_solve")
    out = {"summary": summ.cpu().numpy()}
    if keep_on_device:
        out["psi"], out["j_phi"] = psi, jphi
    else:
        out["psi"], out["j_phi"] = psi.cpu().numpy(), jphi.cpu().numpy()
    if want_history:
        out["hist"], out["gs_hist"] = hist.cpu().numpy(), gsh.cpu().numpy()
    return out


def shard_range(total: int, world: int, rank: int) -> tuple[int, int]:
    """Contiguous slice [lo, hi) of `total` independent equilibria owned by `rank` (SURVEY.md 8e:
    batched equilibria shard with no cross-GPU traffic; sizes differ by at most one)."""
    if world < 1 or not (0 <= rank < world) or total < 0:
        raise ValueError("bad shard arguments")
    base, extra = divmod(total, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def solve_sharded(kernel, coil_currents, plasma_current=None, ped_p=None, ped_ff=None, *, group=None,
                  gather: bool = True) -> dict[str, Any]:
    """Solve a batch of independent equilibria sharded over the ranks of a torch.distributed group.

    Every rank passes the FULL per-sample input arrays and solves only its `shard_range` slice with
    ``kernel.solve`` (a ``BatchedFusionKernel``); no data-path collective runs during the solves.
    With ``gather`` the per-equilibrium scalars (iterations, converged, residual, axis, X-point ...)
    are all-gathered afterwards so every rank sees the summary of the whole batch; the flux maps stay
    on the rank that computed them (``res["psi"]`` holds rows [lo, hi) only).
    """
    import torch.distributed as dist
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    cc = np.asarray(coil_currents, dtype=np.float64)
    total = cc.shape[0]
    lo, hi = shard_range(total, world, rank)
    pick = lambda a: None if a is None else np.asarray(a, dtype=np.float64)[lo:hi]
    res = kernel.solve(cc[lo:hi], pick(plasma_current), pick(ped_p), pick(ped_ff)) if hi > lo else {}
    res["shard"] = (lo, hi)
    if gather and world > 1:
        scalars = {k: v for k, v in res.items() if isinstance(v, np.ndarray) and v.ndim == 1}
        parts: list = [None] * world
        dist.all_gather_object(parts, ((lo, hi), scalars), group=group)
        keys = sorted({k for _, sc in parts for k in sc})
        merged = {}
        for k in keys:
            ref = next(sc[k] for _, sc in parts if k in sc)
            out = np.zeros(total, dtype=ref.dtype)
            for (a, b), sc in parts:
                if b > a:
                    out[a:b] = sc[k]
            merged[k] = out
        res["global"] = merged
    return res


class BatchedFusionKernel(_GridMixin):
    """B independent equilibria on one geometry (UQ / reconstruction / design sweeps).

    The reference runs such sweeps as a ``multiprocessing.Pool`` over ``FusionKernel`` solves
    (``tools/parallel_gen_iter.py:73-141``); here the whole batch advances through the same
    kernels per Picard iteration.  Per-sample inputs: coil currents, plasma current target and
    (H-mode) pedestal parameters.
    """

    def __init__(self, config, device: int | None = None) -> None:
        self.device = D.current_device() if device is None else int(device)
        self.cfg = _load_config(config)
        self._init_grid()
        self._pinned: dict = {}

    def vacuum_field(self, coil_currents: np.ndarray):
        """(B, n_coils) currents -> device tensor (B, nz, nr) (fusion_kernel.py:218-251)."""
        mu0 = self.cfg["physics"].get("vacuum_permeability", 1.0)
        pos = [(c["r"], c["z"]) for c in self.cfg["coils"]]
        w = (mu0 * np.asarray(coil_currents, dtype=np.float64)) / (2.0 * np.pi)
        return self._coil_flux_dev(pos, w, 0)

    def pinned_outputs(self, batch: int, fields=("psi", "j_phi")) -> dict:
        """Pinned host tensors (B, nz, nr) for ``solve(..., out=...)`` / ``solve_free_boundary(..., out=...)``: the
        flux maps then reach the host with one asynchronous DMA each instead of a pageable staging copy."""
        torch = D.torch_mod()
        return {k: torch.empty((batch, self.NZ, self.NR), dtype=torch.float64).pin_memory() for k in fields}

    def _fields_to_host(self, res: dict, dev: dict, to_host: bool, out: dict | None) -> None:
        for name in ("psi", "j_phi"):
            if not to_host:
                res[name] = dev[name]
            elif out is not None:
                if name in out:  # fields the caller did not ask for stay on the device
                    out[name].copy_(dev[name], non_blocking=True)
                    res[name] = out[name].numpy()
                else:
                    res[name] = dev[name]
            else:
                res[name] = dev[name].cpu().numpy()
        if to_host and out is not None:
            D.torch_mod().cuda.current_stream().synchronize()

    def solve(self, coil_currents=None, plasma_current=None, ped_p=None, ped_ff=None, *, batch: int | None = None,
              to_host: bool = True, want_history: bool = False, out: dict | None = None) -> dict[str, Any]:
        """Solve the batch; returns arrays with a leading batch axis.

        coil_currents (B, n_coils) | None (config currents), plasma_current (B,) | None,
        ped_p / ped_ff (B, 4) | None: [ped_top, ped_width, ped_height, core_alpha].
        ``out`` = ``pinned_outputs(B)`` (or a subset of its keys): those fields are copied into the given pinned
        host tensors and returned as NumPy views of them; fields not in ``out`` stay on the device.
        """
        params = self._picard_params()
        base_i = np.array([c["current"] for c in self.cfg["coils"]], dtype=np.float64)
        if coil_currents is None:
            if batch is None:
                raise ValueError("give coil_currents or batch")
            coil_currents = np.tile(base_i, (batch, 1))
        cc = np.ascontiguousarray(np.asarray(coil_currents, dtype=np.float64))
        B = cc.shape[0]
        ip = np.full(B, float(self.cfg["physics"]["plasma_current_target"])) if plasma_current is None \
            else np.asarray(plasma_current, dtype=np.float64).reshape(B)
        if np.any(np.abs(ip) < 1e-12):
            raise NotImplementedError("zero plasma current samples: use FusionKernel.calculate_vacuum_field")
        ped = self._ped_rows(B, ped_p, ped_ff)
        t0 = time.time()
        mu0 = self.cfg["physics"].get("vacuum_permeability", 1.0)
        w = (mu0 * cc) / (2.0 * np.pi)
        dev = self.solve_device(D.to_device(w, self.device), D.to_device(ip, self.device),
                                None if ped is None else D.to_device(ped, self.device),
                                want_history=want_history)
        s = dev["summary"].cpu().numpy()
        res = self.unpack_summary(s)
        self._fields_to_host(res, dev, to_host, out)
        res["wall_time_s"] = time.time() - t0
        if want_history:
            res["residual_history"] = dev["hist"].cpu().numpy()
            res["gs_residual_history"] = dev["gs_hist"].cpu().numpy()
        return res

    def topology(self, psi_dev) -> np.ndarray:
        """O-/X-point of each flux map of a device batch (a10, a11): host (B, 8) rows
        [iz_ax, ir_ax, psi_ax, iz_x, ir_x, psi_x, found_x, min psi] (gsb_topology)."""
        B = int(psi_dev.shape[0])
        ctx = self._context(B)
        out = D.empty((B, 8), self.device)
        saddle = 1 if bool(self.cfg.get("solver", {}).get("xpoint_use_saddle_detection", False)) else 0
        _lib.check(ctx.lib.gsb_topology(ctx.handle, D.ptr(psi_dev), B, float(self.cfg["dimensions"]["Z_min"]), saddle,
                                        D.ptr(out), D.stream_ptr()), "gsb_topology")
        return out.cpu().numpy()

    def unpack_summary(self, s: np.ndarray) -> dict[str, Any]:
        """Decode the [B,16] summary rows of gsb_picard_solve (include/gsb200.h)."""
        return {
            "iterations": s[:, 0].astype(np.int64), "converged": s[:, 1] > 0.5, "residual": s[:, 2],
            "gs_residual": s[:, 3], "gs_residual_best": s[:, 4], "status": s[:, 5].astype(np.int64),
            "psi_axis": s[:, 6], "psi_boundary": s[:, 7],
            "axis_R": self.R[s[:, 9].astype(np.int64)], "axis_Z": self.Z[s[:, 8].astype(np.int64)],
            "xpoint_R": np.where(s[:, 13] > 0, self.R[s[:, 11].astype(np.int64)], 0.0),
            "xpoint_Z": np.where(s[:, 13] > 0, self.Z[s[:, 10].astype(np.int64)], 0.0),
        }

    # -- batched free boundary (a17 + a18) -------------------------------------------------------------
    def wall_response_matrix(self, mu0: float = _MU0_SI):
        """Lane-C von Hagenow matrix M[N_wall, N_interior] on the device (build_response_matrix,
        jax_free_boundary_predictive.py:183-211), cached per mu0: geometry only."""
        cache = self.__dict__.setdefault("_wall_m_cache", {})
        key = float(mu0)
        if key not in cache:
            ctx = self._context(1)
            n_wall = 2 * self.NR + 2 * (self.NZ - 2)
            n_int = (self.NZ - 2) * (self.NR - 2)
            m = D.empty((n_wall, n_int), self.device)
            _lib.check(ctx.lib.gsb_wall_matrix(ctx.handle, key, D.ptr(m), D.stream_ptr()), "gsb_wall_matrix")
            cache[key] = m
        return cache[key]

    def _ped_rows(self, B: int, ped_p, ped_ff):
        if ped_p is None and ped_ff is None:
            return None
        dp = np.array([self.ped_params_p[k] for k in _PED_KEYS])
        df = np.array([self.ped_params_ff[k] for k in _PED_KEYS])
        pp = np.tile(dp, (B, 1)) if ped_p is None else np.asarray(ped_p, dtype=np.float64).reshape(B, 4)
        pf = np.tile(df, (B, 1)) if ped_ff is None else np.asarray(ped_ff, dtype=np.float64).reshape(B, 4)
        return np.concatenate([pp, pf], axis=1)

    def solve_free_boundary(self, coil_currents=None, plasma_current=None, ped_p=None, ped_ff=None, *, turns=None,
                            max_outer_iter: int = 20, tol: float = 1e-4, plasma_wall: bool = False,
                            wall_mu0: float = _MU0_SI, psi0=None, batch: int | None = None, to_host: bool = True,
                            out: dict | None = None, optimize_shape: bool = False, target_points=None,
                            target_values=None, current_limits=None, tikhonov_alpha: float = 1e-4,
                            reconstruct_boundary: bool = False, limiter_points=None, axis_point=None,
                            x_points=None) -> dict[str, Any]:
        """``FusionKernel.solve_free_boundary(coils, max_outer_iter, tol, optimize_shape, tikhonov_alpha)``
        (fusion_kernel_free_boundary.py:623-739) for B independent equilibria in one device-resident outer loop.

        coil_currents (B, n_coils) | None (config currents; then give ``batch``), turns (n_coils,) | None (config
        ``turns``, default 1), plasma_current (B,) | None, ped_p / ped_ff (B, 4) | None.  ``plasma_wall=True`` adds
        the plasma's own wall flux M @ (J_phi dA) (lane C, jax_free_boundary_predictive.py:443-498) from the second
        outer iteration on, as one FP64 tensor-core GEMM over the batch per outer iteration.  ``psi0`` (B, nz, nr)
        is the starting flux (default zeros, the state of a freshly constructed kernel).  ``out`` may carry pinned
        host tensors (``pinned_outputs``) to receive the fields without a pageable staging copy (see ``solve``).
        Returns per-equilibrium arrays: outer_iterations, final_diff, inner_iterations (sum over the outer
        iterations), fb_converged, plus the keys of ``solve`` for the last inner solve.

        ``optimize_shape=True`` with ``target_points`` (P, 2) re-fits the coil currents to the shape-control points
        after every inner solve, on the device: target = ``target_values`` ((P,) or (B, P)) or, without them, the mean
        of the flux sampled at the points (isoflux); currents = argmin |M^T I - target|^2 + tikhonov_alpha |I|^2 within
        +-``current_limits`` (n_coils,).  The fit is the exact bounded minimiser, where the reference stops
        ``lsq_linear(method="trf")`` at its tolerance (currents within ~1e-7 relative; a current the reference leaves
        just inside its limit sits on it here, so ``active_current_bounds`` can be larger).  The result then also has
        ``coil_currents`` (B, n_coils) and ``shape_optimization`` with the reference's keys (the fit scalars as (B,)
        arrays, ``target_flux`` / ``achieved_flux`` (B, P)) plus ``fit_fallback`` (B,): the fit failed (non-finite
        target) and the clipped prior currents were kept, as the reference does.  Without ``target_points`` the call is
        the ``optimize_shape=False`` solve, like the reference's.

        ``reconstruct_boundary=True`` ends the call with the reference's wall-contour check (:708-739), on the device for
        the whole batch: the result gains ``boundary_reconstruction`` (``reconstruct_boundary_flux_from_coils`` on the
        wall contour with the final currents, plus ``limiter_points``, ``axis_point`` and ``x_points``, shared or per
        sample) and ``vacuum_boundary_abs_error`` (B,), its max_abs_error.  The target is the flux the loop imposed on the
        wall in each sample's last outer iteration (the reference's psi_ext there): the coil flux (of the final currents
        with ``optimize_shape``), or with ``plasma_wall`` alone the wall ring of the final psi (coil plus plasma wall
        flux, to the rounding of the last Picard under-relaxation).  Integer ``turns`` are then required.
        """
        if not reconstruct_boundary and not (limiter_points is None and axis_point is None and x_points is None):
            raise ValueError("limiter_points, axis_point and x_points need reconstruct_boundary=True.")
        if max_outer_iter < 1:
            raise ValueError("max_outer_iter must be >= 1.")
        if not np.isfinite(tol) or tol < 0.0:
            raise ValueError("tol must be finite and >= 0.")
        coils = self.cfg["coils"]
        base_i = np.array([c["current"] for c in coils], dtype=np.float64)
        if coil_currents is None:
            if batch is None:
                raise ValueError("give coil_currents or batch")
            coil_currents = np.tile(base_i, (batch, 1))
        cc = np.ascontiguousarray(np.asarray(coil_currents, dtype=np.float64))
        B = cc.shape[0]
        tr = np.array([int(c.get("turns", 1)) for c in coils], dtype=np.float64) if turns is None \
            else np.asarray(turns, dtype=np.float64).reshape(len(coils))
        ip = np.full(B, float(self.cfg["physics"]["plasma_current_target"])) if plasma_current is None \
            else np.asarray(plasma_current, dtype=np.float64).reshape(B)
        if np.any(np.abs(ip) < 1e-12):
            raise NotImplementedError("zero plasma current samples: use FusionKernel.solve_free_boundary")
        ped = self._ped_rows(B, ped_p, ped_ff)
        shape = bool(optimize_shape) and target_points is not None
        spec = self._shape_spec(B, tr, target_points, target_values, current_limits, tikhonov_alpha) if shape else None
        t0 = time.time()
        bspec = None
        if reconstruct_boundary:
            from .free_boundary import _wall_contour
            bspec = self._boundary_spec(B, tr, _wall_contour(self)[0], limiter_points, axis_point, x_points)
        psi_in = None if psi0 is None else D.to_device(np.asarray(psi0, dtype=np.float64).reshape(B, self.NZ, self.NR),
                                                       self.device)
        kw = dict(max_outer_iter=max_outer_iter, tol=tol, plasma_wall=plasma_wall, wall_mu0=wall_mu0, psi_out=psi_in,
                  warm=psi0 is not None)
        ipd = D.to_device(ip, self.device)
        pedd = None if ped is None else D.to_device(ped, self.device)
        if shape:
            dev = self.solve_free_boundary_device(None, ipd, pedd, optimize_shape=True, target_points=spec["points"],
                                                  target_values=spec["values"], current_limits=spec["limits"],
                                                  tikhonov_alpha=spec["alpha"], turns=spec["turns"],
                                                  currents=D.to_device(cc, self.device), **kw)
        else:
            w = cc * tr[None, :]  # I * turns (fusion_kernel_free_boundary.py:88-92)
            dev = self.solve_free_boundary_device(D.to_device(w, self.device), ipd, pedd, **kw)
        if bspec is not None:
            # the reference's psi_ext after its loop: the coil flux (psi_ext; with shape steps that of the final
            # currents), or with the plasma wall flux the ring the last outer iteration imposed on psi, which only the
            # Picard under-relaxation (1-a) x + a x has touched since (rounding)
            field = dev["psi"] if plasma_wall and not shape else dev["psi_ext"]
            bdev = self._boundary_call(bspec, dev["currents"] if shape else D.to_device(cc, self.device), field, 3)
            from .free_boundary import _wall_contour
            _, iz, ir = _wall_contour(self)
            idx = D.torch_mod().as_tensor(iz * self.NR + ir, device=field.device)
            ring = field.reshape(B, -1)[:, idx].cpu().numpy()
        res = self.unpack_summary(dev["summary"].cpu().numpy())
        fb = dev["fb_summary"].cpu().numpy()
        res.update({"outer_iterations": fb[:, 0].astype(np.int64), "final_diff": fb[:, 1],
                    "inner_iterations": fb[:, 2].astype(np.int64), "fb_converged": fb[:, 3] > 0.5})
        if shape:
            res["coil_currents"] = dev["currents"].cpu().numpy()
            res["shape_optimization"] = self._shape_report(spec, dev["shape_out"].cpu().numpy())
        if bspec is not None:
            br = res["boundary_reconstruction"] = self._boundary_report(bspec, bdev, ring)
            res["vacuum_boundary_abs_error"] = br["max_abs_error"]
        self._fields_to_host(res, dev, to_host, out)
        res["wall_time_s"] = time.time() - t0
        return res

    def solve_free_boundary_device(self, w_dev, ip_dev, ped_dev=None, *, max_outer_iter: int = 20, tol: float = 1e-4,
                                   plasma_wall: bool = False, wall_mu0: float = _MU0_SI, psi_out=None, jphi_out=None,
                                   warm: bool = False, events=None, optimize_shape: bool = False, target_points=None,
                                   target_values=None, current_limits=None, tikhonov_alpha: float = 1e-4,
                                   currents=None, turns=None) -> dict[str, Any]:
        """Device-resident batched free-boundary solve (gsb_free_boundary_solve): w_dev (B, n_coils) = I*turns,
        ip_dev (B,), ped_dev (B, 8) | None - CUDA float64 tensors.  ``psi_out`` is the flux buffer (its content is
        the starting flux when ``warm``, otherwise it is zeroed).  Returns device tensors psi, j_phi, psi_ext,
        summary (B, 16), fb_summary (B, 4).

        ``optimize_shape=True`` with ``target_points`` (gsb_free_boundary_shape_solve; keywords as in
        ``solve_free_boundary``, ``turns`` (n_coils,) | None = config turns): ``currents`` (B, n_coils) CUDA float64
        holds the starting currents in amperes and receives the final ones; ``w_dev`` is not used.  The result then
        also has ``currents`` and ``shape_out`` (B, 2P+4): target, achieved flux, rmse, max |residual|, active bounds,
        fallback flag of each equilibrium's last shape step."""
        params = self._picard_params()
        shape = bool(optimize_shape) and target_points is not None
        B = int((currents if shape else w_dev).shape[0])
        ctx = self._context(B)
        pos = [(c["r"], c["z"]) for c in self.cfg["coils"]]
        nc = len(pos)
        st = D.stream_ptr()
        ext = self.__dict__.get("_fb_ext")
        if ext is None or ext.shape[0] != B:
            ext = self._fb_ext = D.empty((B, self.NZ, self.NR), self.device)
        if shape:
            tr = np.array([c.get("turns", 1) for c in self.cfg["coils"]], dtype=np.float64) if turns is None \
                else np.asarray(turns, dtype=np.float64).reshape(-1)
            spec = self._shape_spec(B, tr, target_points, target_values, current_limits, tikhonov_alpha)
            if tuple(currents.shape) != (B, nc):
                raise ValueError(f"currents must have shape ({B}, {nc}).")
        elif nc:
            g = self._green_table(pos, 1)
            _lib.check(ctx.lib.gsb_coil_flux(ctx.handle, D.ptr(g), D.ptr(w_dev), nc, 1, D.ptr(ext), B, st), "gsb_coil_flux")
        else:
            ext.zero_()
        psi = psi_out if psi_out is not None else D.empty((B, self.NZ, self.NR), self.device)
        jphi = jphi_out if jphi_out is not None else D.empty((B, self.NZ, self.NR), self.device)
        if not warm:
            psi.zero_()
            jphi.zero_()
        summ = D.empty((B, 16), self.device)
        fbs = D.empty((B, 4), self.device)
        m = self.wall_response_matrix(wall_mu0) if plasma_wall else None
        fb = _lib.gsb_free_boundary_params()
        fb.max_outer_iter, fb.tol, fb.warm_j = int(max_outer_iter), float(tol), 0
        null = ctypes.c_void_p()
        if shape:
            return self._shape_solve_call(ctx, params, fb, spec, pos, currents, psi, ext, m, ip_dev, ped_dev, jphi, summ,
                                          fbs, B, st, events)
        if events is not None:
            events[0].record()
        _lib.check(ctx.lib.gsb_free_boundary_solve(ctx.handle, ctypes.byref(params), ctypes.byref(fb), D.ptr(psi), D.ptr(ext),
                                                   null if m is None else D.ptr(m), D.ptr(ip_dev),
                                                   null if ped_dev is None else D.ptr(ped_dev), D.ptr(jphi), D.ptr(summ),
                                                   D.ptr(fbs), B, st), "gsb_free_boundary_solve")
        if events is not None:
            events[1].record()
        return {"psi": psi, "j_phi": jphi, "psi_ext": ext, "summary": summ, "fb_summary": fbs}

    # -- shape-optimising outer loop --------------------------------------------------------------------
    def _shape_spec(self, B: int, turns: np.ndarray, target_points, target_values, current_limits,
                    tikhonov_alpha) -> dict[str, Any]:
        """Check the shape-fit inputs with the reference's messages (free_boundary.py) and the device's limits."""
        nc = len(self.cfg["coils"])
        if nc == 0:
            raise ValueError("CoilSet.positions must contain at least one coil.")
        if nc > 32:
            raise ValueError("optimize_shape supports at most 32 coils on the device.")
        pts = np.ascontiguousarray(target_points, dtype=np.float64)
        if pts.ndim != 2 or pts.shape[1] != 2 or pts.shape[0] == 0:
            raise ValueError("target_flux_points must have shape (n_points, 2) with n_points > 0.")
        if not np.all(np.isfinite(pts)):
            raise ValueError("target_flux_points must contain finite values only.")
        if np.any(pts[:, 0] <= 0.0):
            raise ValueError("observation radii must be positive.")
        P = pts.shape[0]
        if P > 1024:
            raise ValueError("optimize_shape supports at most 1024 target points on the device.")
        vals = None
        if target_values is not None:
            v = np.asarray(target_values, dtype=np.float64)
            if v.ndim == 1 and v.shape == (P,):
                v = np.broadcast_to(v, (B, P))
            elif v.shape != (B, P):
                raise ValueError("target_flux_values must have the same length as target_flux_points.")
            if not np.all(np.isfinite(v)):
                raise ValueError("target_flux_values must contain finite values only.")
            vals = np.ascontiguousarray(v)
        alpha = float(tikhonov_alpha)
        if not np.isfinite(alpha) or alpha < 0.0:
            raise ValueError("tikhonov_alpha must be finite and non-negative.")
        lim = None
        if current_limits is not None:
            lim = np.ascontiguousarray(current_limits, dtype=np.float64).reshape(-1)
            if lim.shape[0] != nc:
                raise ValueError("current_limits must have one entry per coil.")
            if not np.all(np.isfinite(lim)):
                raise ValueError("current_limits must contain finite values only.")
            if np.any(lim <= 0.0):
                raise ValueError("current_limits must contain finite positive values only.")
        tr = np.asarray(turns, dtype=np.float64).reshape(-1)
        if tr.shape[0] != nc or not np.all(np.isfinite(tr)) or np.any(tr < 1) or np.any(tr != np.round(tr)):
            raise ValueError("turns must be positive integers when optimize_shape is set.")
        return {"points": pts, "values": vals, "limits": lim, "alpha": alpha, "turns": tr.astype(np.int32)}

    def _shape_solve_call(self, ctx, params, fb, spec, pos, currents, psi, ext, m, ip_dev, ped_dev, jphi, summ, fbs, B,
                          st, events) -> dict[str, Any]:
        dp = ctypes.POINTER(ctypes.c_double)
        nc, P = len(pos), spec["points"].shape[0]
        rz = np.ascontiguousarray(np.asarray(pos, dtype=np.float64).reshape(nc, 2))
        sp = _lib.gsb_shape_params()
        sp.n_coils, sp.coil_rz, sp.n_points = nc, rz.ctypes.data_as(dp), P
        sp.points, sp.alpha = spec["points"].ctypes.data_as(dp), spec["alpha"]
        sp.isoflux = 1 if spec["values"] is None else 0
        sp.limits = spec["limits"].ctypes.data_as(dp) if spec["limits"] is not None else None
        turns = spec["turns"]
        tgt = None if spec["values"] is None else D.to_device(spec["values"], self.device)
        out = D.empty((B, 2 * P + 4), self.device)
        g = self._green_table(pos, 1)
        null = ctypes.c_void_p()
        if events is not None:
            events[0].record()
        _lib.check(ctx.lib.gsb_free_boundary_shape_solve(
            ctx.handle, ctypes.byref(params), ctypes.byref(fb), ctypes.byref(sp), D.ptr(g),
            turns.ctypes.data_as(ctypes.POINTER(ctypes.c_int)), D.ptr(currents), null if tgt is None else D.ptr(tgt),
            D.ptr(out), D.ptr(psi), D.ptr(ext), null if m is None else D.ptr(m), D.ptr(ip_dev),
            null if ped_dev is None else D.ptr(ped_dev), D.ptr(jphi), D.ptr(summ), D.ptr(fbs), B, st),
            "gsb_free_boundary_shape_solve")
        if events is not None:
            events[1].record()
        return {"psi": psi, "j_phi": jphi, "psi_ext": ext, "summary": summ, "fb_summary": fbs, "currents": currents,
                "shape_out": out}

    def _shape_report(self, spec, so: np.ndarray) -> dict[str, Any]:
        """The reference's ``shape_optimization`` dict (fusion_kernel_free_boundary.py:686-699) over the batch."""
        from .free_boundary import _mutual_device
        pos = [(c["r"], c["z"]) for c in self.cfg["coils"]]
        P = spec["points"].shape[0]
        resp = _mutual_device(self.device, pos, spec["turns"], spec["points"])  # geometry only
        tgt, ach = so[:, :P].copy(), so[:, P:2 * P].copy()
        rmse = so[:, 2 * P].copy()
        return {"solver_mode": "free_boundary_solver_shape_current_optimization", "target_point_count": int(P),
                "coil_count": len(pos), "response_rank": int(np.linalg.matrix_rank(resp.T)),
                "response_condition": float(np.linalg.cond(resp.T)), "flux_rmse": rmse,
                "flux_relative_rmse": rmse / np.maximum(np.sqrt(np.mean(tgt ** 2, axis=1)), 1.0),
                "max_abs_flux_residual": so[:, 2 * P + 1].copy(),
                "active_current_bounds": so[:, 2 * P + 2].astype(np.int64), "target_flux": tgt,
                "achieved_flux": ach, "fit_fallback": so[:, 2 * P + 3] > 0.5}

    # -- magnetic-probe current reconstruction -----------------------------------------------------------
    def reconstruct_coil_currents_from_magnetic_probes(self, *, flux_points=None, flux_measurements=None,
                                                       b_probe_points=None, b_probe_directions=None,
                                                       b_probe_measurements=None, measurement_sigma=None,
                                                       tikhonov_alpha: float = 1.0e-6, coil_currents=None,
                                                       current_limits=None, turns=None) -> dict[str, Any]:
        """``FusionKernel.reconstruct_coil_currents_from_magnetic_probes`` (fusion_kernel_free_boundary.py:370-488) for
        B measurement vectors of one diagnostic set, fitted on the device in one call (gsb_probe_reconstruct).

        flux_measurements (B, n_flux) and b_probe_measurements (B, n_b) (a 1-D vector is a batch of one) follow the
        rows of ``build_magnetic_probe_response_matrix``; coil_currents (B, n_coils) | (n_coils,) | None (config
        currents) is the prior of the Tikhonov term; measurement_sigma (m,) and current_limits (n_coils,) are shared
        by the batch; turns (n_coils,) | None = config turns.  Each sample gets the exact bounded minimiser of
        |w (R x - meas)|^2 + alpha |x - prior|^2 within +-current_limits, where the reference stops
        ``lsq_linear(method="trf")`` at its tolerance (a current trf leaves just inside its limit sits on it here).
        Returns the reference's keys with a leading batch axis where the value is per sample: coil_currents (B, n),
        residual / weighted_residual (B, m), residual_rms / weighted_residual_rms / active_bounds (B,); response_rank
        and response_condition of the unweighted response.  Raises ``RuntimeError`` naming the samples whose fit
        failed (non-finite right-hand side or iteration cap), as the reference raises for its one sample.
        """
        from .free_boundary import _bounds, _points, _vector, build_magnetic_probe_response_matrix
        cfg_coils = self.cfg["coils"]
        n = len(cfg_coils)
        if n > 32:
            raise ValueError("probe reconstruction supports at most 32 coils on the device.")
        tr = np.array([c.get("turns", 1) for c in cfg_coils], dtype=np.float64) if turns is None \
            else np.asarray(turns, dtype=np.float64).reshape(-1)
        if tr.shape[0] != n or not np.all(np.isfinite(tr)) or np.any(tr < 1) or np.any(tr != np.round(tr)):
            raise ValueError("turns must be positive integers.")
        coils = CoilSet(positions=[(c["r"], c["z"]) for c in cfg_coils],
                        currents=np.array([c.get("current", 0.0) for c in cfg_coils], dtype=np.float64),
                        turns=[int(t) for t in tr], current_limits=current_limits)
        resp = build_magnetic_probe_response_matrix(self, coils, flux_points=flux_points, b_probe_points=b_probe_points,
                                                    b_probe_directions=b_probe_directions)
        parts = []
        for pts, vals, pname, vname in ((flux_points, flux_measurements, "flux_points", "flux_measurements"),
                                        (b_probe_points, b_probe_measurements, "b_probe_points", "b_probe_measurements")):
            if pts is not None:
                if vals is None:
                    raise ValueError(f"{vname} must be provided with {pname}.")
                parts.append(_measurement_rows(vals, vname, _points(pts, pname).shape[0]))
            elif vals is not None:
                raise ValueError(f"{pname} must be provided with {vname}.")
        if not parts:
            raise ValueError("At least one measurement vector must be provided.")
        if len({p.shape[0] for p in parts}) > 1:
            raise ValueError("flux_measurements and b_probe_measurements must have the same batch size.")
        meas = np.ascontiguousarray(np.concatenate(parts, axis=1))
        B, m = meas.shape
        if m != resp.shape[0]:
            raise ValueError("measurement vector length must match response rows.")
        if m > 1024:
            raise ValueError("probe reconstruction supports at most 1024 measurements on the device.")
        sg = None
        if measurement_sigma is not None:
            sg = _vector(measurement_sigma, "measurement_sigma", m)
            if np.any(sg <= 0.0):
                raise ValueError("measurement_sigma must contain finite positive values only.")
        alpha = float(tikhonov_alpha)
        if not np.isfinite(alpha) or alpha < 0.0:
            raise ValueError("tikhonov_alpha must be finite and non-negative.")
        prior = coils.currents if coil_currents is None else np.asarray(coil_currents, dtype=np.float64)
        if prior.ndim == 1 and prior.shape == (n,):
            prior = np.tile(prior, (B, 1))
        if prior.shape != (B, n) or not np.all(np.isfinite(prior)):
            raise ValueError("CoilSet.currents must be finite with one entry per coil.")
        lim = None if current_limits is None else _bounds(coils, n, positive=True)[1]
        dev = self.reconstruct_coil_currents_device(resp, D.to_device(meas, self.device),
                                                    D.to_device(prior, self.device), measurement_sigma=sg,
                                                    tikhonov_alpha=alpha, current_limits=lim)
        stats = dev["stats"].cpu().numpy()
        bad = np.flatnonzero(stats[:, 3] > 0.5)
        if bad.size:
            raise RuntimeError("Magnetic probe inverse reconstruction failed: non-finite right-hand side or iteration "
                               f"cap reached in samples {bad.tolist()}")
        return {"coil_currents": dev["currents"].cpu().numpy(), "residual": dev["residual"].cpu().numpy(),
                "weighted_residual": dev["weighted_residual"].cpu().numpy(), "residual_rms": stats[:, 0].copy(),
                "weighted_residual_rms": stats[:, 1].copy(), "response_rank": int(np.linalg.matrix_rank(resp)),
                "response_condition": float(np.linalg.cond(resp)), "active_bounds": stats[:, 2].astype(np.int64)}

    def reconstruct_coil_currents_device(self, response, meas_dev, prior_dev, *, measurement_sigma=None,
                                         tikhonov_alpha: float = 1.0e-6, current_limits=None, max_iter: int = 0,
                                         events=None) -> dict[str, Any]:
        """Device-resident probe fit (gsb_probe_reconstruct): response (m, n_coils) host array, meas_dev (B, m) and
        prior_dev (B, n_coils) CUDA float64 tensors, measurement_sigma (m,) | None, current_limits (n_coils,) | None
        (positive), max_iter = cap on the free-set solves per fit (0: 3 n_coils + 10).  Returns device tensors
        currents (B, n), residual, weighted_residual (B, m) and stats (B, 4): residual rms, weighted residual rms,
        active bounds, failed."""
        lib = _lib.load()
        dp = ctypes.POINTER(ctypes.c_double)
        resp = np.ascontiguousarray(response, dtype=np.float64)
        m, n = resp.shape
        B = int(meas_dev.shape[0])
        torch = D.torch_mod()
        for t, shape, name in ((meas_dev, (B, m), "meas_dev"), (prior_dev, (B, n), "prior_dev")):
            if tuple(t.shape) != shape or t.dtype != torch.float64 or not t.is_contiguous() or not t.is_cuda:
                raise ValueError(f"{name} must be a contiguous CUDA float64 tensor of shape {shape}.")
        sg = None if measurement_sigma is None else np.ascontiguousarray(measurement_sigma, dtype=np.float64)
        lim = None if current_limits is None else np.ascontiguousarray(current_limits, dtype=np.float64)
        pp = _lib.gsb_probe_params()
        pp.n_coils, pp.n_rows, pp.response = n, m, resp.ctypes.data_as(dp)
        pp.sigma = None if sg is None else sg.ctypes.data_as(dp)
        pp.alpha, pp.max_iter = float(tikhonov_alpha), int(max_iter)
        pp.limits = None if lim is None else lim.ctypes.data_as(dp)
        null = ctypes.c_void_p()
        need = ctypes.c_longlong(0)
        _lib.check(lib.gsb_probe_reconstruct(ctypes.byref(pp), null, null, null, null, null, null, null,
                                             ctypes.byref(need), B, null), "gsb_probe_reconstruct")
        work = D.empty(((need.value + 7) // 8,), self.device)
        need.value = work.numel() * 8
        cur, stats = D.empty((B, n), self.device), D.empty((B, 4), self.device)
        res, wres = D.empty((B, m), self.device), D.empty((B, m), self.device)
        if events is not None:
            events[0].record()
        _lib.check(lib.gsb_probe_reconstruct(ctypes.byref(pp), D.ptr(meas_dev), D.ptr(prior_dev), D.ptr(cur), D.ptr(res),
                                             D.ptr(wres), D.ptr(stats), D.ptr(work), ctypes.byref(need), B,
                                             D.stream_ptr()), "gsb_probe_reconstruct")
        if events is not None:
            events[1].record()
        return {"currents": cur, "residual": res, "weighted_residual": wres, "stats": stats}

    # -- wall-contour boundary reconstruction ------------------------------------------------------------
    def _boundary_spec(self, B: int, turns, boundary_points, limiter_points, axis_point, x_points) -> dict[str, Any]:
        """Check the reconstruction inputs with the reference's messages (free_boundary.py) and the device's limits, and
        compute the host geometry once (no device work).  An axis (B, 2) or X-points (B, X, 2) make both per sample."""
        from .free_boundary import _limiter_geometry, _points, _x_pair_symmetric
        cfg_coils = self.cfg["coils"]
        n = len(cfg_coils)
        if n < 1:
            raise ValueError("CoilSet.positions must contain at least one coil.")
        tr = np.array([c.get("turns", 1) for c in cfg_coils], dtype=np.float64) if turns is None \
            else np.asarray(turns, dtype=np.float64).reshape(-1)
        if tr.shape[0] != n or not np.all(np.isfinite(tr)) or np.any(tr < 1) or np.any(tr != np.round(tr)):
            raise ValueError("turns must be positive integers.")
        obs = np.ascontiguousarray(_points(boundary_points, "boundary_points"))
        if obs.shape[0] > 4096:
            raise ValueError("boundary reconstruction supports at most 4096 boundary points on the device.")
        lim = None
        if limiter_points is not None:
            lim = np.ascontiguousarray(_points(limiter_points, "limiter_points"))
            if lim.shape[0] > 4096:
                raise ValueError("boundary reconstruction supports at most 4096 limiter points on the device.")
        per = False
        ax = None
        if axis_point is not None:
            a = np.asarray(axis_point, dtype=np.float64)
            if a.size == 2:
                ax = _points(a.reshape(1, 2), "axis_point")[0]
            elif a.shape == (B, 2):
                ax, per = _points(a, "axis_point"), True
            else:
                raise ValueError(f"axis_point must have shape (2,) or ({B}, 2).")
        xo = None
        if x_points is not None:
            x = np.asarray(x_points, dtype=np.float64)
            if x.ndim == 3:
                if x.shape[0] != B or x.shape[1] < 1 or x.shape[2] != 2:
                    raise ValueError(f"x_points must have shape (n_points, 2) or ({B}, n_points, 2).")
                _points(x.reshape(-1, 2), "x_points")
                xo, per = x, True
            else:
                xo = _points(x, "x_points")
            if xo.shape[-2] > 64:
                raise ValueError("boundary reconstruction supports at most 64 X-points on the device.")
        for p in (obs, lim, ax, xo):
            if p is not None and np.any(p[..., 0] <= 0.0):
                raise ValueError("observation radii must be positive.")
        X = 0 if xo is None else int(xo.shape[-2])
        # the C entry reads the point arrays in storage order; per sample, both the axis and the X-points are
        if ax is not None:
            ax = np.ascontiguousarray(np.broadcast_to(ax, (B, 2)) if per else ax)
        if xo is not None:
            xo = np.ascontiguousarray(np.broadcast_to(xo, (B, X, 2)) if per else xo)
        pos = [(c["r"], c["z"]) for c in cfg_coils]
        tri = np.ascontiguousarray(tr.astype(np.int32))
        geo: dict[str, Any] = {"boundary_points": obs, "point_count": int(obs.shape[0]), "coil_count": n,
                               "limiter_point_count": 0, "min_limiter_distance_m": None, "axis_point": ax,
                               "x_point_count": X, "x_point_pair_symmetry_abs_error": None}
        if lim is not None:
            geo.update(_limiter_geometry(obs, lim))
        if xo is not None:
            geo["x_points"] = xo
        sym = None
        if ax is not None and X == 2:
            ok = _x_pair_symmetric(xo if per else xo[None], ax if per else ax[None])
            if ok.any():
                sym = np.broadcast_to(ok, (B,)) if not per else ok
        return {"B": B, "per_sample": per, "coil_rz": np.ascontiguousarray(np.asarray(pos, dtype=np.float64).reshape(n, 2)),
                "turns": tri, "points": obs, "limiter": lim, "axis": ax, "xpoints": xo, "X": X, "symmetric": sym,
                "geometry": geo}

    def _boundary_call(self, spec, currents_dev, target_dev, mode: int, events=None) -> dict[str, Any]:
        """One gsb_boundary_flux launch; mode = target_mode of gsb_boundary_params.  "response" is the boundary columns
        (n_coils, N) of the M the entry built in its workspace and used."""
        lib = _lib.load()
        dp = ctypes.POINTER(ctypes.c_double)
        B, n = spec["B"], spec["coil_rz"].shape[0]
        N = spec["points"].shape[0]
        L = 0 if spec["limiter"] is None else spec["limiter"].shape[0]
        A, X = int(spec["axis"] is not None), spec["X"]
        bp = _lib.gsb_boundary_params()
        bp.n_coils, bp.coil_rz = n, spec["coil_rz"].ctypes.data_as(dp)
        bp.turns = spec["turns"].ctypes.data_as(ctypes.POINTER(ctypes.c_int))
        bp.n_points, bp.points = N, spec["points"].ctypes.data_as(dp)
        bp.n_limiter, bp.limiter = L, None if not L else spec["limiter"].ctypes.data_as(dp)
        bp.has_axis, bp.axis = A, None if not A else spec["axis"].ctypes.data_as(dp)
        bp.n_xpoints, bp.xpoints = X, None if not X else spec["xpoints"].ctypes.data_as(dp)
        bp.per_sample, bp.target_mode = int(spec["per_sample"]), int(mode)
        if mode == 3:
            bp.nz, bp.nr = self.NZ, self.NR
            r_ax, z_ax = np.ascontiguousarray(self.R, dtype=np.float64), np.ascontiguousarray(self.Z, dtype=np.float64)
            bp.r_axis, bp.z_axis = r_ax.ctypes.data_as(dp), z_ax.ctypes.data_as(dp)
        null = ctypes.c_void_p()
        need = ctypes.c_longlong(0)
        _lib.check(lib.gsb_boundary_flux(ctypes.byref(bp), null, null, null, null, null, null, ctypes.byref(need), B,
                                         null), "gsb_boundary_flux")
        work = D.empty(((need.value + 7) // 8,), self.device)
        need.value = work.numel() * 8
        flux, stats = D.empty((B, N + L + A + X), self.device), D.empty((B, 5), self.device)
        res = D.empty((B, N), self.device) if mode else None
        if events is not None:
            events[0].record()
        _lib.check(lib.gsb_boundary_flux(ctypes.byref(bp), D.ptr(currents_dev), null if not mode else D.ptr(target_dev),
                                         D.ptr(flux), null if res is None else D.ptr(res), D.ptr(stats), D.ptr(work),
                                         ctypes.byref(need), B, D.stream_ptr()), "gsb_boundary_flux")
        if events is not None:
            events[1].record()
        ncol = N + L + (B if spec["per_sample"] else 1) * (A + X)
        return {"flux": flux, "residual": res, "stats": stats, "response": work[:n * ncol].view(n, ncol)[:, :N]}

    def _boundary_report(self, spec, dev, target) -> dict[str, Any]:
        """The reference's reconstruct_boundary_flux_from_coils dict over the batch; raises ValueError naming the samples
        with non-finite boundary flux or target."""
        flux, st = dev["flux"].cpu().numpy(), dev["stats"].cpu().numpy()
        flags = st[:, 4].astype(np.int64)
        bad = np.flatnonzero(flags & 1)
        if bad.size:
            raise ValueError(f"reconstructed boundary flux contains non-finite values in samples {bad.tolist()}")
        bad = np.flatnonzero(flags & 2)
        if bad.size:
            raise ValueError(f"target_flux must contain finite values only: samples {bad.tolist()}")
        N = spec["points"].shape[0]
        L = 0 if spec["limiter"] is None else spec["limiter"].shape[0]
        A, X = int(spec["axis"] is not None), spec["X"]
        d = dict(spec["geometry"])
        resp = d["response_matrix"] = dev["response"].cpu().numpy()
        d["response_rank"] = int(np.linalg.matrix_rank(resp))
        d.update({"reconstructed_flux": flux[:, :N], "limiter_flux": flux[:, N:N + L], "axis_flux": None,
                  "x_point_flux": flux[:, N + L + A:], "x_point_flux_span": None})
        if A:
            d["axis_flux"] = flux[:, N + L]
        if X:
            d["x_point_flux_span"] = st[:, 2].copy()
        if spec["symmetric"] is not None:
            d["x_point_pair_symmetry_abs_error"] = np.where(spec["symmetric"], st[:, 3], np.nan)
        if target is not None:
            d.update({"target_flux": target, "residual": dev["residual"].cpu().numpy(), "rmse": st[:, 0].copy(),
                      "max_abs_error": st[:, 1].copy()})
        return d

    def reconstruct_boundary_flux_from_coils(self, coil_currents=None, *, boundary_points, limiter_points=None,
                                             axis_point=None, x_points=None, target_flux=None,
                                             turns=None) -> dict[str, Any]:
        """``FusionKernel.reconstruct_boundary_flux_from_coils`` (fusion_kernel_free_boundary.py:162-267) for B coil-current
        vectors in one device call (gsb_boundary_flux).

        coil_currents (B, n_coils) | (n_coils,) (a batch of one) | None (config currents) in amperes; turns (n_coils,) |
        None = config turns; axis_point (2,) or (B, 2) and x_points (X, 2) or (B, X, 2): shared or per sample;
        target_flux (N,) or (B, N).  Returns the reference's keys.  Per-sample values have a leading batch axis:
        reconstructed_flux (B, N), limiter_flux (B, L), axis_flux (B,), x_point_flux (B, X), x_point_flux_span (B,),
        residual (B, N), rmse and max_abs_error (B,).  The geometry-only values are computed once on the host.
        x_point_pair_symmetry_abs_error is None where the reference gives None for every sample, otherwise (B,) with NaN
        for the samples whose X-point pair is not mirrored about their axis.  Each flux is sum_c M[c][p] I_c in coil
        order, so a sample's values do not depend on the batch.  Raises ValueError naming the samples whose boundary
        flux is not finite.
        """
        from .free_boundary import _points, _vector
        n = len(self.cfg["coils"])
        cur = np.array([[c.get("current", 0.0) for c in self.cfg["coils"]]], dtype=np.float64) if coil_currents is None \
            else np.asarray(coil_currents, dtype=np.float64)
        if cur.ndim == 1:
            cur = cur[None, :]
        if cur.ndim != 2 or cur.shape[0] < 1 or cur.shape[1] != n:
            raise ValueError(f"currents must have length {n}.")
        if not np.all(np.isfinite(cur)):
            raise ValueError("currents must contain finite values only.")
        B = cur.shape[0]
        N = _points(boundary_points, "boundary_points").shape[0]
        t = None
        if target_flux is not None:
            t = np.asarray(target_flux, dtype=np.float64)
            if t.ndim <= 1:
                t = _vector(t, "target_flux", N)
            elif t.shape != (B, N):
                raise ValueError(f"target_flux must have length {N}.")
            elif not np.all(np.isfinite(t)):
                raise ValueError("target_flux must contain finite values only.")
        spec = self._boundary_spec(B, turns, boundary_points, limiter_points, axis_point, x_points)
        dev = self._boundary_call(spec, D.to_device(cur, self.device), None if t is None else D.to_device(t, self.device),
                                  0 if t is None else (1 if t.ndim == 1 else 2))
        return self._boundary_report(spec, dev, t)

    def reconstruct_boundary_flux_device(self, currents_dev, *, boundary_points, limiter_points=None, axis_point=None,
                                         x_points=None, target_dev=None, target_field=None, turns=None,
                                         events=None) -> dict[str, Any]:
        """Device-resident boundary reconstruction (gsb_boundary_flux): currents_dev (B, n_coils) CUDA float64 in amperes;
        the target is target_dev (N,) | (B, N), or the wall contour of target_field (B, nz, nr) (boundary_points must then
        be that contour, ``_wall_contour``), or none; other keywords as ``reconstruct_boundary_flux_from_coils``.
        Returns device tensors flux (B, N + L + A + X) (boundary, limiter, axis, X-point flux in that order), residual
        (B, N) (None without a target), response (n_coils, N) (the boundary columns of the M the flux was summed over, a
        view of the call's workspace) and stats (B, 5): rmse, max |residual|, X-point flux span, |xf0 - xf1|, flags
        (1: a boundary flux is not finite, 2: a target value is not finite); NaN where a value does not apply."""
        from .free_boundary import _points, _wall_contour
        torch = D.torch_mod()
        B, n = int(currents_dev.shape[0]), len(self.cfg["coils"])
        obs = _points(boundary_points, "boundary_points")
        N = obs.shape[0]
        if target_dev is not None and target_field is not None:
            raise ValueError("give target_dev or target_field, not both.")
        checks = [(currents_dev, [(B, n)], "currents_dev")]
        mode, tgt = 0, None
        if target_dev is not None:
            checks.append((target_dev, [(N,), (B, N)], "target_dev"))
            mode, tgt = (1 if target_dev.ndim == 1 else 2), target_dev
        elif target_field is not None:
            checks.append((target_field, [(B, self.NZ, self.NR)], "target_field"))
            if not np.array_equal(obs, _wall_contour(self)[0]):
                raise ValueError("the wall-contour target needs the wall contour of the grid as boundary points.")
            mode, tgt = 3, target_field
        for t, shapes, name in checks:
            if tuple(t.shape) not in shapes or t.dtype != torch.float64 or not t.is_contiguous() or not t.is_cuda:
                raise ValueError(f"{name} must be a contiguous CUDA float64 tensor of shape {' or '.join(map(str, shapes))}.")
        spec = self._boundary_spec(B, turns, boundary_points, limiter_points, axis_point, x_points)
        return self._boundary_call(spec, currents_dev, tgt, mode, events)

    def solve_device(self, w_dev, ip_dev, ped_dev=None, *, want_history: bool = False, psi_out=None,
                     jphi_out=None, events=None) -> dict[str, Any]:
        """Device-resident batch solve: no host<->device traffic except the active-count poll.

        w_dev (B, n_coils) = (mu0*I)/(2 pi) per coil, ip_dev (B,), ped_dev (B, 8) or None; all CUDA
        float64 tensors.  Returns device tensors psi, j_phi, summary (B,16) [, hist, gs_hist].
        """
        params = self._picard_params()
        B = int(w_dev.shape[0])
        ctx = self._context(B)
        pos = [(c["r"], c["z"]) for c in self.cfg["coils"]]
        nc = len(pos)
        g = self._green_table(pos, 0)
        psi = psi_out if psi_out is not None else D.empty((B, self.NZ, self.NR), self.device)
        st = D.stream_ptr()
        _lib.check(ctx.lib.gsb_coil_flux(ctx.handle, D.ptr(g), D.ptr(w_dev), nc, 0, D.ptr(psi), B, st), "gsb_coil_flux")
        bc = psi  # boundary map == vacuum field; its wall ring is saved before psi is touched
        jphi = jphi_out if jphi_out is not None else D.empty((B, self.NZ, self.NR), self.device)
        summ = D.empty((B, 16), self.device)
        hist = gsh = None
        if want_history:
            hist = D.zeros((B, params.max_iterations), self.device)
            gsh = D.zeros((B, params.max_iterations), self.device)
        null = ctypes.c_void_p()
        if events is not None:  # (start, stop) CUDA events bracketing the Picard launch (bench.py roofline)
            events[0].record()
        _lib.check(ctx.lib.gsb_picard_solve(ctx.handle, ctypes.byref(params), D.ptr(psi), D.ptr(bc), D.ptr(ip_dev),
                                            null if ped_dev is None else D.ptr(ped_dev), D.ptr(jphi), D.ptr(summ),
                                            null if hist is None else D.ptr(hist), null if gsh is None else D.ptr(gsh),
                                            B, st), "gsb_picard_solve")
        if events is not None:
            events[1].record()
        out = {"psi": psi, "j_phi": jphi, "summary": summ}
        if want_history:
            out["hist"], out["gs_hist"] = hist, gsh
        return out
