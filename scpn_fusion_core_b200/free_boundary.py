"""Free-boundary layer on top of the device Green's-function and Picard kernels.

Mirrors ``src/scpn_fusion/core/fusion_kernel_free_boundary.py`` (reference): the same function names,
``(kernel, coils, ...)`` argument order, result-dict keys and ``ValueError`` behaviour; ``FusionKernel``
binds them as methods exactly as the reference's ``fusion_kernel_free_boundary_mixin.py`` does.

Every Green's-function value (coil -> grid, coil -> control/probe/contour point) is evaluated by
libgsb200 (``gsb_green_table`` / ``gsb_coil_flux`` / ``gsb_mutual_matrix``) and the inner equilibrium is
the device Picard solve.  What stays on the host is what the reference also hands to a third-party
routine or does on a handful of scalars: the bounded least-squares fit (``scipy.optimize.lsq_linear``,
n_coils unknowns), rank/condition diagnostics and the four-point flux interpolation.
"""
from __future__ import annotations

import ctypes
import logging
from typing import Any

import numpy as np

from . import _device as D
from . import _lib

logger = logging.getLogger(__name__)


# -- argument checks (reference :95-110) -----------------------------------------------------------

def _vector(value, name: str, length: int | None = None) -> np.ndarray:
    a = np.asarray(value, dtype=np.float64).reshape(-1)
    if length is not None and a.shape != (length,):
        raise ValueError(f"{name} must have length {length}.")
    if not np.all(np.isfinite(a)):
        raise ValueError(f"{name} must contain finite values only.")
    return a


def _points(value, name: str) -> np.ndarray:
    a = np.asarray(value, dtype=np.float64)
    if a.ndim != 2 or a.shape[1] != 2 or a.shape[0] < 1:
        raise ValueError(f"{name} must have shape (n_points, 2) with n_points > 0.")
    if not np.all(np.isfinite(a)):
        raise ValueError(f"{name} must contain finite values only.")
    return a


def _turns(coils, n: int) -> np.ndarray:
    return np.ascontiguousarray([coils.turns[k] if k < len(coils.turns) else 1 for k in range(n)], dtype=np.int32)


def _bounds(coils, n: int, *, positive: bool):
    if coils.current_limits is None:
        return np.full(n, -np.inf), np.full(n, np.inf)
    lim = np.asarray(coils.current_limits, dtype=np.float64).reshape(-1)
    if lim.shape[0] != n:
        raise ValueError("current_limits must have one entry per coil." if not positive
                         else f"current_limits must have length {n}.")
    if not np.all(np.isfinite(lim)):
        raise ValueError("current_limits must contain finite values only.")
    if positive and np.any(lim <= 0.0):
        raise ValueError("current_limits must contain finite positive values only.")
    return -np.abs(lim), np.abs(lim)


# -- Green's function on the device ------------------------------------------------------------------

def _mutual_device(device: int, positions, turns: np.ndarray, obs: np.ndarray) -> np.ndarray:
    """M[coil, point] = turns * G_SI(coil -> point), one gsb_mutual_matrix launch."""
    lib = _lib.load()
    nc = len(positions)
    rz = np.ascontiguousarray(np.asarray(positions, dtype=np.float64).reshape(nc, 2))
    if not np.all(np.isfinite(rz)) or np.any(rz[:, 0] <= 0.0):
        raise ValueError("source coil coordinates must be finite with R_src > 0.")
    obs = np.ascontiguousarray(obs, dtype=np.float64)
    if not np.all(np.isfinite(obs)):
        raise ValueError("observation coordinates must be finite.")
    if np.any(obs[:, 0] <= 0.0):
        raise ValueError("observation radii must be positive.")
    m = D.empty((nc, obs.shape[0]), device)
    _lib.check(lib.gsb_mutual_matrix(D.np_ptr(rz), turns.ctypes.data_as(ctypes.POINTER(ctypes.c_int)), nc, D.np_ptr(obs),
                                     obs.shape[0], D.ptr(m), D.stream_ptr()), "gsb_mutual_matrix")
    return m.cpu().numpy()


def _device_of(kernel) -> int:
    dev = getattr(kernel, "device", None)
    return D.current_device() if dev is None else int(dev)


def green_function(R_src: float, Z_src: float, R_obs: float, Z_obs: float, *, device: int | None = None) -> float:
    """Reference :31-56 - flux per ampere-turn of a circular filament; the self point is 0."""
    v = np.asarray([R_src, Z_src, R_obs, Z_obs], dtype=np.float64)
    if not np.all(np.isfinite(v)):
        raise ValueError("Green's-function coordinates must be finite.")
    if R_src <= 0.0 or R_obs <= 0.0:
        raise ValueError("Green's-function radii must be positive.")
    dev = D.current_device() if device is None else device
    return float(_mutual_device(dev, [(float(R_src), float(Z_src))], np.ones(1, dtype=np.int32),
                                np.array([[R_obs, Z_obs]]))[0, 0])


def compute_external_flux(kernel: Any, coils) -> np.ndarray:
    """Reference :83-93 - sum_c I_c*turns_c*G_c on the (Z, R) grid (SI mu0), device table + contraction."""
    w = [cur * (coils.turns[i] if i < len(coils.turns) else 1) for i, cur in enumerate(coils.currents)]
    if not w:
        return np.zeros((kernel.NZ, kernel.NR))
    return kernel._coil_flux_dev(list(coils.positions), np.array([w]), 1)[0].cpu().numpy()


def build_mutual_inductance_matrix(kernel: Any, coils, obs_points) -> np.ndarray:
    """Reference :137-153 - M[coil, point]."""
    obs = np.asarray(obs_points, dtype=np.float64)
    n = len(coils.positions)
    if n == 0 or obs.shape[0] == 0:
        return np.zeros((n, obs.shape[0]))
    return _mutual_device(_device_of(kernel), coils.positions, _turns(coils, n), obs)


# -- flux-map sampling (:156-159, :562-581) ------------------------------------------------------------

def interp_psi(kernel: Any, R_pt: float, Z_pt: float) -> float:
    ir = min(max(int(np.searchsorted(kernel.R, R_pt)) - 1, 0), kernel.NR - 2)
    iz = min(max(int(np.searchsorted(kernel.Z, Z_pt)) - 1, 0), kernel.NZ - 2)
    tr = min(max((R_pt - kernel.R[ir]) / kernel.dR, 0.0), 1.0)
    tz = min(max((Z_pt - kernel.Z[iz]) / kernel.dZ, 0.0), 1.0)
    p = kernel.Psi
    return float((1 - tr) * (1 - tz) * p[iz, ir] + tr * (1 - tz) * p[iz, ir + 1]
                 + (1 - tr) * tz * p[iz + 1, ir] + tr * tz * p[iz + 1, ir + 1])


def sample_flux_at_points(kernel: Any, points) -> np.ndarray:
    return np.asarray([interp_psi(kernel, float(r), float(z)) for r, z in _points(points, "points")], dtype=np.float64)


def resolve_shape_target_flux(kernel: Any, coils) -> np.ndarray:
    """Reference :584-605 - explicit target values, else the isoflux level = mean sampled flux."""
    if coils.target_flux_points is None:
        raise ValueError("CoilSet.target_flux_points must be set for shape optimisation.")
    obs = np.asarray(coils.target_flux_points, dtype=np.float64)
    if obs.ndim != 2 or obs.shape[1] != 2 or obs.shape[0] == 0:
        raise ValueError("target_flux_points must have shape (n_points, 2) with n_points > 0.")
    if coils.target_flux_values is not None:
        t = np.asarray(coils.target_flux_values, dtype=np.float64).reshape(-1)
        if t.shape[0] != obs.shape[0]:
            raise ValueError("target_flux_values must have the same length as target_flux_points.")
        if not np.all(np.isfinite(t)):
            raise ValueError("target_flux_values must contain finite values only.")
        return t
    samples = np.array([interp_psi(kernel, r, z) for r, z in obs], dtype=np.float64)
    return np.full(obs.shape[0], float(np.mean(samples)), dtype=np.float64)


# -- bounded current fits --------------------------------------------------------------------------------

def optimize_coil_currents(kernel: Any, coils, target_flux, tikhonov_alpha: float = 1e-4) -> np.ndarray:
    """Reference :491-559 - min |M^T I - target|^2 + alpha |I|^2 within +-current_limits."""
    from scipy.optimize import lsq_linear

    if coils.target_flux_points is None:
        raise ValueError("CoilSet.target_flux_points must be set for optimisation.")
    if len(coils.positions) == 0:
        raise ValueError("CoilSet.positions must contain at least one coil.")
    if len(coils.currents) != len(coils.positions):
        raise ValueError("CoilSet.currents length must match number of coil positions.")
    if not np.isfinite(tikhonov_alpha) or tikhonov_alpha < 0.0:
        raise ValueError("tikhonov_alpha must be finite and non-negative.")
    obs = np.asarray(coils.target_flux_points, dtype=np.float64)
    if obs.ndim != 2 or obs.shape[1] != 2 or obs.shape[0] == 0:
        raise ValueError("target_flux_points must have shape (n_points, 2) with n_points > 0.")
    if not np.all(np.isfinite(obs)):
        raise ValueError("target_flux_points must contain finite values only.")
    target = np.asarray(target_flux, dtype=np.float64).reshape(-1)
    if target.shape[0] != obs.shape[0]:
        raise ValueError("target_flux must have the same length as target_flux_points.")
    if not np.all(np.isfinite(target)):
        raise ValueError("target_flux must contain finite values only.")
    M = build_mutual_inductance_matrix(kernel, coils, obs)
    if not np.all(np.isfinite(M)):
        raise ValueError("Mutual inductance matrix contains non-finite entries.")
    n = M.shape[0]
    A = np.vstack([M.T, np.sqrt(tikhonov_alpha) * np.eye(n)])
    b = np.concatenate([target, np.zeros(n)])
    lb, ub = _bounds(coils, n, positive=False)
    fit = lsq_linear(A, b, bounds=(lb, ub), method="trf")
    if not bool(getattr(fit, "success", False)) or not np.all(np.isfinite(fit.x)):
        logger.warning("Coil optimisation failed (status=%s): %s. Falling back to prior currents.",
                       getattr(fit, "status", "unknown"), getattr(fit, "message", "no message"))
        return np.clip(np.asarray(coils.currents, dtype=np.float64).copy(), lb, ub).astype(np.float64)
    return np.asarray(fit.x, dtype=np.float64)


def _probe_directions(directions, length: int) -> list[str]:
    if len(directions) != length:
        raise ValueError("b_probe_directions must have one entry per b_probe_point.")
    out = [str(d).upper() for d in directions]
    if any(d not in ("R", "Z") for d in out):
        raise ValueError("b_probe_directions entries must be 'R' or 'Z'.")
    return out


def build_magnetic_probe_response_matrix(kernel: Any, coils, *, flux_points=None, b_probe_points=None,
                                         b_probe_directions=None) -> np.ndarray:
    """Reference :282-367 - rows = flux loops then B probes; columns = coils.

    All 2*n_probe displaced points and the flux-loop points go through ONE mutual-matrix launch; the
    centred differences B_R = -(dpsi/dZ)/R, B_Z = (dpsi/dR)/R are formed from it with the reference's
    steps eps_r = max(1e-5, 1e-5|R|), eps_z = max(1e-5, 1e-5(1+|Z|)) and R clamped to >= eps_r.
    """
    if len(coils.positions) < 1:
        raise ValueError("CoilSet.positions must contain at least one coil.")
    if len(coils.currents) != len(coils.positions):
        raise ValueError("CoilSet.currents length must match number of coil positions.")
    fl = None if flux_points is None else _points(flux_points, "flux_points")
    bp = None if b_probe_points is None else _points(b_probe_points, "b_probe_points")
    if fl is None and bp is None:
        raise ValueError("At least one flux point or B probe point must be provided.")
    dirs: list[str] = []
    if bp is not None:
        if b_probe_directions is None:
            raise ValueError("b_probe_directions must be provided with b_probe_points.")
        dirs = _probe_directions(b_probe_directions, int(bp.shape[0]))
    nf = 0 if fl is None else int(fl.shape[0])
    nb = 0 if bp is None else int(bp.shape[0])
    pts = np.empty((nf + 2 * nb, 2))
    if nf:
        pts[:nf] = fl
    scale = np.empty(nb)
    for i in range(nb):
        r, z = float(bp[i, 0]), float(bp[i, 1])
        er, ez = max(1.0e-5, 1.0e-5 * abs(r)), max(1.0e-5, 1.0e-5 * (1.0 + abs(z)))
        rs = max(r, er)
        if dirs[i] == "R":
            pts[nf + 2 * i], pts[nf + 2 * i + 1] = (rs, z + ez), (rs, z - ez)
            scale[i] = -(2.0 * ez * rs)
        else:
            pts[nf + 2 * i], pts[nf + 2 * i + 1] = (rs + er, z), (rs - er, z)
            scale[i] = 2.0 * er * rs
    if np.any(pts[:, 0] <= 0.0):
        raise ValueError("Green's-function radii must be positive.")
    n = len(coils.positions)
    G = _mutual_device(_device_of(kernel), coils.positions, _turns(coils, n), pts)  # (n_coils, nf + 2 nb)
    out = np.zeros((nf + nb, n))
    out[:nf] = G[:, :nf].T
    if nb:
        out[nf:] = (G[:, nf::2].T - G[:, nf + 1::2].T) / scale[:, None]  # -(d)/s == d/(-s) exactly
    if not np.all(np.isfinite(out)):
        raise ValueError("Magnetic probe response matrix contains non-finite entries.")
    return out


def reconstruct_coil_currents_from_magnetic_probes(kernel: Any, coils, *, flux_points=None, flux_measurements=None,
                                                   b_probe_points=None, b_probe_directions=None,
                                                   b_probe_measurements=None, measurement_sigma=None,
                                                   tikhonov_alpha: float = 1.0e-6) -> dict[str, Any]:
    """Reference :370-488 - weighted Tikhonov fit around the prior currents, bounded by current_limits."""
    from scipy.optimize import lsq_linear

    resp = build_magnetic_probe_response_matrix(kernel, coils, flux_points=flux_points, b_probe_points=b_probe_points,
                                                b_probe_directions=b_probe_directions)
    parts = []
    if flux_points is not None:
        if flux_measurements is None:
            raise ValueError("flux_measurements must be provided with flux_points.")
        parts.append(_vector(flux_measurements, "flux_measurements", _points(flux_points, "flux_points").shape[0]))
    elif flux_measurements is not None:
        raise ValueError("flux_points must be provided with flux_measurements.")
    if b_probe_points is not None:
        if b_probe_measurements is None:
            raise ValueError("b_probe_measurements must be provided with b_probe_points.")
        parts.append(_vector(b_probe_measurements, "b_probe_measurements",
                             _points(b_probe_points, "b_probe_points").shape[0]))
    elif b_probe_measurements is not None:
        raise ValueError("b_probe_points must be provided with b_probe_measurements.")
    if not parts:
        raise ValueError("At least one measurement vector must be provided.")
    target = np.concatenate(parts).astype(np.float64, copy=False)
    if target.shape != (resp.shape[0],):
        raise ValueError("measurement vector length must match response rows.")
    w = np.ones(resp.shape[0])
    if measurement_sigma is not None:
        sg = _vector(measurement_sigma, "measurement_sigma", resp.shape[0])
        if np.any(sg <= 0.0):
            raise ValueError("measurement_sigma must contain finite positive values only.")
        w = 1.0 / sg
    alpha = float(tikhonov_alpha)
    if not np.isfinite(alpha) or alpha < 0.0:
        raise ValueError("tikhonov_alpha must be finite and non-negative.")
    n = len(coils.positions)
    prior = np.asarray(coils.currents, dtype=np.float64).reshape(-1)
    if prior.shape != (n,) or not np.all(np.isfinite(prior)):
        raise ValueError("CoilSet.currents must be finite with one entry per coil.")
    A, b = resp * w[:, None], target * w
    if alpha > 0.0:
        A = np.vstack([A, np.sqrt(alpha) * np.eye(n)])
        b = np.concatenate([b, np.sqrt(alpha) * prior])
    lb, ub = _bounds(coils, n, positive=True)
    fit = lsq_linear(A, b, bounds=(lb, ub), method="trf")
    if not bool(getattr(fit, "success", False)) or not np.all(np.isfinite(fit.x)):
        raise RuntimeError(f"Magnetic probe inverse reconstruction failed: {getattr(fit, 'message', '')}")
    cur = np.asarray(fit.x, dtype=np.float64)
    res = resp @ cur - target
    wres = res * w
    return {"coil_currents": cur, "residual": res, "weighted_residual": wres,
            "residual_rms": float(np.sqrt(np.mean(res ** 2))) if res.size else 0.0,
            "weighted_residual_rms": float(np.sqrt(np.mean(wres ** 2))) if wres.size else 0.0,
            "response_rank": int(np.linalg.matrix_rank(resp)),
            "response_condition": float(np.linalg.cond(resp)) if resp.size else float("inf"),
            "active_bounds": int(np.count_nonzero(np.isclose(cur, lb) | np.isclose(cur, ub)))}


# -- contour diagnostics (:113-134, :162-267, :608-620) ----------------------------------------------------

def _points_inside_polygon(points, polygon) -> np.ndarray:
    pts, poly = _points(points, "points"), _points(polygon, "polygon")
    if poly.shape[0] < 3:
        raise ValueError("polygon must contain at least three points.")
    x, y = pts[:, 0], pts[:, 1]
    nxt = np.roll(poly, -1, axis=0)
    inside = np.zeros(pts.shape[0], dtype=bool)
    for (xa, ya), (xb, yb) in zip(poly, nxt):
        crosses = (ya > y) != (yb > y)
        inside ^= crosses & (x < (xb - xa) * (y - ya) / max(abs(yb - ya), 1.0e-300) + xa)
    return inside


def _wall_contour(kernel: Any):
    """Wall points counter-clockwise from (R_min, Z_min) and the (iz, ir) that visit a field in that order."""
    r, z = np.asarray(kernel.R, dtype=np.float64), np.asarray(kernel.Z, dtype=np.float64)
    if r.ndim != 1 or z.ndim != 1 or r.size < 2 or z.size < 2:
        raise ValueError("kernel R/Z axes must be one-dimensional with at least two points.")
    if not np.all(np.isfinite(r)) or not np.all(np.isfinite(z)):
        raise ValueError("kernel R/Z axes must contain finite values only.")
    nr, nz = r.size, z.size
    ir = np.concatenate([np.arange(nr), np.full(nz - 1, nr - 1), np.arange(nr - 2, -1, -1), np.zeros(nz - 2, dtype=int)])
    iz = np.concatenate([np.zeros(nr, dtype=int), np.arange(1, nz), np.full(nr - 1, nz - 1), np.arange(nz - 2, 0, -1)])
    return np.column_stack([r[ir], z[iz]]), iz, ir


def _limiter_geometry(obs: np.ndarray, lim: np.ndarray) -> dict[str, Any]:
    """The geometry-only limiter keys of reconstruct_boundary_flux_from_coils (:162-267), in its expressions."""
    frac = float(np.mean(_points_inside_polygon(obs, lim)))
    return {"limiter_points": lim, "limiter_point_count": int(lim.shape[0]),
            "min_limiter_distance_m": float(np.min(np.linalg.norm(lim[:, None, :] - obs[None, :, :], axis=2))),
            "boundary_containment_fraction": frac, "boundary_containment_pass": bool(frac >= 1.0)}


def _x_pair_symmetric(x_points: np.ndarray, axis: np.ndarray) -> np.ndarray:
    """Per sample, the reference's condition for x_point_pair_symmetry_abs_error: two X-points at one R, mirrored about
    the axis height.  x_points (B, 2, 2), axis (B, 2) -> (B,) bool."""
    return ((np.abs(x_points[:, 0, 0] - x_points[:, 1, 0]) <= 1.0e-9)
            & (np.abs(x_points[:, 0, 1] + x_points[:, 1, 1] - 2.0 * axis[:, 1]) <= 1.0e-9))


def _kernel_boundary_points(kernel: Any) -> np.ndarray:
    return _wall_contour(kernel)[0]


def reconstruct_boundary_flux_from_coils(kernel: Any, coils, *, boundary_points, limiter_points=None, axis_point=None,
                                         x_points=None, target_flux=None) -> dict[str, Any]:
    obs = _points(boundary_points, "boundary_points")
    if len(coils.positions) < 1:
        raise ValueError("CoilSet.positions must contain at least one coil.")
    cur = _vector(coils.currents, "currents", len(coils.positions))
    # one launch for every requested point family
    fam = [("b", obs)]
    if limiter_points is not None:
        fam.append(("l", _points(limiter_points, "limiter_points")))
    if axis_point is not None:
        fam.append(("a", _points(np.asarray(axis_point, dtype=np.float64).reshape(1, 2), "axis_point")))
    if x_points is not None:
        fam.append(("x", _points(x_points, "x_points")))
    M = build_mutual_inductance_matrix(kernel, coils, np.vstack([p for _, p in fam]))
    off, resp = 0, {}
    for tag, p in fam:
        resp[tag] = np.ascontiguousarray(M[:, off:off + p.shape[0]])
        off += p.shape[0]
    rec = resp["b"].T @ cur
    if not np.all(np.isfinite(rec)):
        raise ValueError("reconstructed boundary flux contains non-finite values.")
    d: dict[str, Any] = {
        "boundary_points": obs, "reconstructed_flux": rec, "response_matrix": resp["b"],
        "response_rank": int(np.linalg.matrix_rank(resp["b"])), "point_count": int(obs.shape[0]),
        "coil_count": int(len(coils.positions)), "limiter_point_count": 0, "limiter_flux": np.array([], dtype=np.float64),
        "min_limiter_distance_m": None, "axis_point": None, "axis_flux": None, "x_point_count": 0,
        "x_point_flux": np.array([], dtype=np.float64), "x_point_flux_span": None,
        "x_point_pair_symmetry_abs_error": None}
    fams = dict(fam)
    if "l" in fams:
        lim = fams["l"]
        frac = float(np.mean(_points_inside_polygon(obs, lim)))
        d.update({"limiter_points": lim, "limiter_flux": resp["l"].T @ cur, "limiter_point_count": int(lim.shape[0]),
                  "min_limiter_distance_m": float(np.min(np.linalg.norm(lim[:, None, :] - obs[None, :, :], axis=2))),
                  "boundary_containment_fraction": frac, "boundary_containment_pass": bool(frac >= 1.0)})
    if "a" in fams:
        d.update({"axis_point": fams["a"][0], "axis_flux": float((resp["a"].T @ cur)[0])})
    if "x" in fams:
        xo, xf = fams["x"], resp["x"].T @ cur
        sym = None
        ax = d.get("axis_point")
        if ax is not None and xo.shape[0] == 2:
            if abs(float(xo[0, 0] - xo[1, 0])) <= 1.0e-9 and abs(float(xo[0, 1] + xo[1, 1] - 2.0 * ax[1])) <= 1.0e-9:
                sym = float(abs(xf[0] - xf[1]))
        d.update({"x_points": xo, "x_point_flux": xf, "x_point_count": int(xo.shape[0]),
                  "x_point_flux_span": float(np.max(xf) - np.min(xf)) if xf.size else None,
                  "x_point_pair_symmetry_abs_error": sym})
    if target_flux is not None:
        t = _vector(target_flux, "target_flux", int(obs.shape[0]))
        r = rec - t
        d.update({"target_flux": t, "residual": r, "rmse": float(np.sqrt(np.mean(r ** 2))) if r.size else 0.0,
                  "max_abs_error": float(np.max(np.abs(r))) if r.size else 0.0})
    return d


# -- outer loop (:623-739) ---------------------------------------------------------------------------------

def solve_free_boundary(kernel: Any, coils, max_outer_iter: int = 20, tol: float = 1e-4, optimize_shape: bool = False,
                        tikhonov_alpha: float = 1e-4, limiter_points=None, axis_point=None, x_points=None) -> dict[str, Any]:
    """Coil flux on the wall -> warm-started device Picard solve -> optional bounded re-fit of the coil
    currents to the shape-control points -> repeat until max|dPsi| < tol; then the wall-contour check."""
    if max_outer_iter < 1:
        raise ValueError("max_outer_iter must be >= 1.")
    if not np.isfinite(tol) or tol < 0.0:
        raise ValueError("tol must be finite and >= 0.")
    psi_ext = compute_external_flux(kernel, coils)
    diff = float("inf")
    shape: dict[str, Any] | None = None
    outer = 0
    for outer in range(max_outer_iter):
        kernel._apply_boundary_conditions(kernel.Psi, psi_ext)
        psi_old = kernel.Psi.copy()
        kernel.solve_equilibrium(preserve_initial_state=True, boundary_flux=psi_ext)
        if optimize_shape and coils.target_flux_points is not None:
            target = resolve_shape_target_flux(kernel, coils)
            resp = build_mutual_inductance_matrix(kernel, coils, coils.target_flux_points)
            # through the kernel method, so a subclass / monkeypatched optimiser is honoured (reference :666-671)
            new = np.asarray(kernel.optimize_coil_currents(coils, target, tikhonov_alpha=tikhonov_alpha),
                             dtype=np.float64).reshape(-1)
            if new.shape != (len(coils.positions),):
                raise ValueError("optimised coil current vector length must match coil count.")
            if not np.all(np.isfinite(new)):
                raise ValueError("optimised coil currents must contain finite values only.")
            achieved = resp.T @ new
            r = achieved - target
            rmse = float(np.sqrt(np.mean(r ** 2)))
            active = 0
            if coils.current_limits is not None:
                lim = _vector(coils.current_limits, "current_limits", len(coils.positions))
                active = int(np.count_nonzero(np.isclose(np.abs(new), lim, rtol=0.0)))
            shape = {"solver_mode": "free_boundary_solver_shape_current_optimization",
                     "target_point_count": int(target.shape[0]), "coil_count": int(len(coils.positions)),
                     "response_rank": int(np.linalg.matrix_rank(resp.T)), "response_condition": float(np.linalg.cond(resp.T)),
                     "flux_rmse": rmse, "flux_relative_rmse": float(rmse / max(float(np.sqrt(np.mean(target ** 2))), 1.0)),
                     "max_abs_flux_residual": float(np.max(np.abs(r))), "active_current_bounds": active,
                     "target_flux": target.copy(), "achieved_flux": achieved.astype(np.float64, copy=False)}
            coils.currents = new
            psi_ext = compute_external_flux(kernel, coils)
        diff = float(np.max(np.abs(kernel.Psi - psi_old)))
        if diff < tol:
            logger.info("Free-boundary converged at outer iter %d (diff=%.2e)", outer, diff)
            break
    pts, iz, ir = _wall_contour(kernel)
    recon = reconstruct_boundary_flux_from_coils(kernel, coils, boundary_points=pts, limiter_points=limiter_points,
                                                 axis_point=axis_point, x_points=x_points, target_flux=psi_ext[iz, ir])
    return {"outer_iterations": outer + 1, "final_diff": diff, "coil_currents": np.asarray(coils.currents).copy(),
            "vacuum_boundary_abs_error": recon["max_abs_error"], "boundary_reconstruction": recon,
            "shape_optimization": shape}


class FreeBoundaryMixin:
    """Binds the functions above as ``FusionKernel`` methods (reference: fusion_kernel_free_boundary_mixin.py)."""

    def _green_function(self, R_src: float, Z_src: float, R_obs: float, Z_obs: float) -> float:
        return green_function(R_src, Z_src, R_obs, Z_obs, device=_device_of(self))

    def _compute_external_flux(self, coils) -> np.ndarray:
        return compute_external_flux(self, coils)

    def _build_mutual_inductance_matrix(self, coils, obs_points) -> np.ndarray:
        return build_mutual_inductance_matrix(self, coils, obs_points)

    def _build_magnetic_probe_response_matrix(self, coils, **kw) -> np.ndarray:
        return build_magnetic_probe_response_matrix(self, coils, **kw)

    def reconstruct_coil_currents_from_magnetic_probes(self, coils, **kw) -> dict[str, Any]:
        return reconstruct_coil_currents_from_magnetic_probes(self, coils, **kw)

    def reconstruct_boundary_flux_from_coils(self, coils, **kw) -> dict[str, Any]:
        return reconstruct_boundary_flux_from_coils(self, coils, **kw)

    def optimize_coil_currents(self, coils, target_flux, tikhonov_alpha: float = 1e-4) -> np.ndarray:
        return optimize_coil_currents(self, coils, target_flux, tikhonov_alpha=tikhonov_alpha)

    def _resolve_shape_target_flux(self, coils) -> np.ndarray:
        return resolve_shape_target_flux(self, coils)

    def _interp_psi(self, R_pt: float, Z_pt: float) -> float:
        return interp_psi(self, R_pt, Z_pt)

    def _sample_flux_at_points(self, points) -> np.ndarray:
        return sample_flux_at_points(self, points)

    def solve_free_boundary(self, coils, max_outer_iter: int = 20, tol: float = 1e-4, optimize_shape: bool = False,
                            tikhonov_alpha: float = 1e-4, limiter_points=None, axis_point=None, x_points=None):
        return solve_free_boundary(self, coils, max_outer_iter=max_outer_iter, tol=tol, optimize_shape=optimize_shape,
                                   tikhonov_alpha=tikhonov_alpha, limiter_points=limiter_points, axis_point=axis_point,
                                   x_points=x_points)
