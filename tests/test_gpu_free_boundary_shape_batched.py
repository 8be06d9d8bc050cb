"""GPU parity of the batched shape-optimising free-boundary loop (gsb_free_boundary_shape_solve;
BatchedFusionKernel.solve_free_boundary(optimize_shape=True)).

Every outer iteration re-fits the coil currents to the shape-control points (fusion_kernel_free_boundary.py:664-701).
The device computes the EXACT bounded minimiser of |M^T x - t|^2 + alpha |x|^2 (bounded-variable least squares on the
QR factor of [M^T; sqrt(alpha) I]), while the reference stops scipy's interior-point lsq_linear(method="trf") at its
tolerance.  On the reference fixture the two differ by at most 5.2e-11 relative in the currents, but trf leaves two
currents 2.1e-5 A and 4e-8 A inside their 6e6 A limits, so the reference reports active_current_bounds = 0 where the
exact solution has 2 currents on their limits.  Hence: currents and psi are compared with the fixture and with the
default (trf) oracle at rtol 1e-7, and tightly with the oracle whose fit is lsq_linear(method="bvls") (the exact
minimiser, `exact_fit` below); active_current_bounds is compared with the exact solution only.
"""
from __future__ import annotations

import json
import os

import numpy as np
import pytest

import gs_oracle as G
from conftest import golden, golden_cfg, rel_l2

pytestmark = pytest.mark.gpu

PSI_TOL = 1e-9
LIMITS_UQ = np.array([6.0e6, 20e6, 20e6, 20e6, 20e6, 20e6, 20e6])  # PF1 ends on its limit in some UQ samples only
ALPHA_UQ = 1e-12


@pytest.fixture(scope="module")
def pkg():
    import scpn_fusion_core_b200 as p
    return p


def _bvls_fit(positions, turns, currents, points, target, *, limits=None, alpha=1e-4):
    """gs_oracle.optimize_coil_currents with the exact bounded minimiser (lsq_linear method="bvls")."""
    from scipy.optimize import lsq_linear
    M = G.mutual_matrix(positions, turns, points)
    n = M.shape[0]
    A = np.vstack([M.T, np.sqrt(alpha) * np.eye(n)])
    b = np.concatenate([np.asarray(target, dtype=np.float64).reshape(-1), np.zeros(n)])
    lb, ub = G._current_bounds(limits, n)
    res = lsq_linear(A, b, bounds=(lb, ub), method="bvls")
    if not bool(getattr(res, "success", False)) or not np.all(np.isfinite(res.x)):
        return np.clip(np.asarray(currents, dtype=np.float64).copy(), lb, ub)
    return np.asarray(res.x, dtype=np.float64)


@pytest.fixture
def exact_fit(monkeypatch):
    """The oracle's outer loop with the exact current fit in place of trf."""
    monkeypatch.setattr(G, "optimize_coil_currents", _bvls_fit)


def _uq(cfg, B, seed0=2026, coil_scale=1.0e6):
    base = np.array([c["current"] for c in cfg["coils"]]) * coil_scale
    cc, ip, ped = [], [], []
    for ks in range(B):
        rng = np.random.default_rng(seed0 + ks)
        cc.append(base * rng.uniform(0.85, 1.15, size=len(base)))
        ip.append(cfg["physics"]["plasma_current_target"] * rng.uniform(0.8, 1.2))
        ped.append([0.92 * rng.uniform(0.97, 1.03), 0.05 * rng.uniform(0.9, 1.1), 1.0 * rng.uniform(0.9, 1.1),
                    0.3 * rng.uniform(0.9, 1.1)])
    return np.array(cc), np.array(ip), np.array(ped)


def _oracle(cfg, cc, ip, ped, **kw):
    c = json.loads(json.dumps(cfg))
    for coil, cur in zip(c["coils"], cc):
        coil["current"] = float(cur)
    c["physics"]["plasma_current_target"] = float(ip)
    if ped is not None:
        pd = dict(zip(("ped_top", "ped_width", "ped_height", "core_alpha"), (float(v) for v in ped)))
        c["physics"]["profiles"] = {"mode": "h-mode", "p_prime": pd, "ff_prime": dict(pd)}
    prob = G.PicardProblem(c)
    pos = [(q["r"], q["z"]) for q in c["coils"]]
    pw = kw.pop("plasma_wall_mu0", None)
    if pw is not None:
        kw["plasma_wall"] = G.wall_response_matrix(prob.R, prob.Z, pw)
    r = G.free_boundary_solve(prob, pos, [float(v) for v in cc], [1] * len(pos), optimize_shape=True, **kw)
    return prob, r


def _uq_cfg(n):
    cfg = golden_cfg(golden("solves"), "iter129")
    cfg["grid_resolution"] = [n, n]
    cfg["physics"]["profiles"] = {"mode": "h-mode"}
    return cfg


def test_reference_fixture_isoflux_bounded(pkg):
    """Case (i) of free_boundary_shape.npz (the reference's own run: 33^2, alpha 1e-13, isoflux target, bounded
    currents, three outer iterations), replicated five times in one batch."""
    z = golden("free_boundary_shape")
    bk = pkg.BatchedFusionKernel(json.loads(str(z["cfg"])))
    cc = np.tile(z["currents0"], (5, 1))
    r = bk.solve_free_boundary(cc, max_outer_iter=3, tol=1e-4, optimize_shape=True, target_points=z["pts"],
                               current_limits=z["limits"], tikhonov_alpha=float(z["alpha"]))
    so, sc = r["shape_optimization"], z["so_scalars"]
    for b in range(5):
        assert int(r["outer_iterations"][b]) == int(z["meta"][0])
        assert rel_l2(r["psi"][b], z["psi"]) <= PSI_TOL
        np.testing.assert_allclose(r["coil_currents"][b], z["currents"], rtol=1e-7, atol=0)
        assert abs(r["final_diff"][b] - z["meta"][1]) <= 1e-6 * abs(z["meta"][1])
        np.testing.assert_allclose(so["target_flux"][b], z["so_target"], rtol=1e-8)
        np.testing.assert_allclose(so["achieved_flux"][b], z["so_achieved"], rtol=1e-7, atol=1e-10)
        np.testing.assert_allclose([so["flux_rmse"][b], so["flux_relative_rmse"][b], so["max_abs_flux_residual"][b]],
                                   sc[4:7], rtol=1e-7)
        assert int(so["active_current_bounds"][b]) == 2  # the exact solution; trf stops inside both limits (0)
        assert not so["fit_fallback"][b]
    assert (so["target_point_count"], so["coil_count"], so["response_rank"]) == (int(sc[0]), int(sc[1]), int(sc[2]))
    assert abs(so["response_condition"] - sc[3]) <= 1e-9 * sc[3]
    assert so["solver_mode"] == "free_boundary_solver_shape_current_optimization"
    for b in range(1, 5):
        np.testing.assert_array_equal(r["psi"][b], r["psi"][0])
        np.testing.assert_array_equal(r["coil_currents"][b], r["coil_currents"][0])


def test_reference_fixture_explicit_targets(pkg):
    """Case (ii): one outer iteration, explicit targets, alpha 1e-6, unbounded."""
    z = golden("free_boundary_shape")
    bk = pkg.BatchedFusionKernel(json.loads(str(z["cfg"])))
    cc = np.tile(z["currents0"], (2, 1))
    r = bk.solve_free_boundary(cc, max_outer_iter=1, tol=0.0, optimize_shape=True, target_points=z["pts"],
                               target_values=z["explicit_targets"], tikhonov_alpha=1e-6)
    for b in range(2):
        assert rel_l2(r["psi"][b], z["explicit_psi"]) <= PSI_TOL
        np.testing.assert_allclose(r["coil_currents"][b], z["explicit_currents"], rtol=1e-7, atol=0)
        np.testing.assert_array_equal(r["shape_optimization"]["target_flux"][b], z["explicit_targets"])
    assert (r["shape_optimization"]["active_current_bounds"] == 0).all()


@pytest.mark.parametrize("n,B,streaming,isoflux,check", [(33, 5, False, True, (0, 1, 4)),
                                                          (65, 3, False, False, (0, 2)),
                                                          (65, 2, True, True, (1,))])
def test_uq_samples_vs_exact_fit_oracle(pkg, exact_fit, n, B, streaming, isoflux, check):
    """H-mode UQ batches sample by sample against the oracle with the exact fit: resident Picard kernel at 33^2 and
    65^2, and 65^2 forced onto the streaming loop, eight outer iterations.  Isoflux and per-sample explicit targets; at
    33^2 the 6 MA limit of PF1 holds the last fit of samples 1 and 2 and leaves samples 0, 3 and 4 free."""
    cfg = _uq_cfg(n)
    cc, ip, ped = _uq(cfg, B)
    z = golden("free_boundary_shape")
    pts = z["pts"]
    tv = None if isoflux else np.linspace(5.0, 6.5, B)[:, None] + 0.05 * np.arange(len(pts))[None, :]
    bk = pkg.BatchedFusionKernel(cfg)
    if streaming:
        os.environ["GSB_PICARD_STREAMING"] = "1"
    try:
        r = bk.solve_free_boundary(cc, ip, ped, ped, max_outer_iter=8, tol=1e-4, optimize_shape=True,
                                   target_points=pts, target_values=tv, current_limits=LIMITS_UQ,
                                   tikhonov_alpha=ALPHA_UQ)
    finally:
        os.environ.pop("GSB_PICARD_STREAMING", None)
    so = r["shape_optimization"]
    for b in check:
        _, ro = _oracle(cfg, cc[b], ip[b], ped[b], max_outer_iter=8, tol=1e-4, tikhonov_alpha=ALPHA_UQ,
                        target_points=pts, target_values=None if tv is None else tv[b], current_limits=LIMITS_UQ)
        assert int(r["outer_iterations"][b]) == ro["outer_iterations"]
        assert rel_l2(r["psi"][b], ro["psi"]) <= PSI_TOL
        np.testing.assert_allclose(r["coil_currents"][b], ro["coil_currents"], rtol=1e-9, atol=0)
        assert int(so["active_current_bounds"][b]) == ro["shape_optimization"]["active_current_bounds"]
        np.testing.assert_allclose(so["target_flux"][b], ro["shape_optimization"]["target_flux"], rtol=1e-9)
    if n == 33:
        assert so["active_current_bounds"].tolist() == [0, 1, 1, 0, 0]
    assert not so["fit_fallback"].any()


def test_uq_sample_vs_default_trf_oracle(pkg):
    """Against the unmodified oracle (trf fit, as the reference): currents within 1e-7.  Sample 1 ends with PF1 on its
    limit in the exact fit, where trf stops inside it."""
    cfg = _uq_cfg(33)
    cc, ip, ped = _uq(cfg, 2)
    z = golden("free_boundary_shape")
    bk = pkg.BatchedFusionKernel(cfg)
    r = bk.solve_free_boundary(cc, ip, ped, ped, max_outer_iter=8, tol=1e-4, optimize_shape=True,
                               target_points=z["pts"], current_limits=LIMITS_UQ, tikhonov_alpha=ALPHA_UQ)
    _, ro = _oracle(cfg, cc[1], ip[1], ped[1], max_outer_iter=8, tol=1e-4, tikhonov_alpha=ALPHA_UQ,
                    target_points=z["pts"], current_limits=LIMITS_UQ)
    assert int(r["outer_iterations"][1]) == ro["outer_iterations"]
    np.testing.assert_allclose(r["coil_currents"][1], ro["coil_currents"], rtol=1e-7, atol=0)


def test_fit_kernels_on_the_device_output(pkg):
    """The shape step in isolation, on the device's own final flux: the isoflux target equals the oracle's
    shape_target_flux bit for bit, the currents are lsq_linear(method="bvls")'s on that target and satisfy the KKT sign
    conditions, and achieved_flux = M^T x."""
    from scipy.optimize import lsq_linear
    cfg = _uq_cfg(33)
    cc, ip, ped = _uq(cfg, 6)
    z = golden("free_boundary_shape")
    pts = z["pts"]
    bk = pkg.BatchedFusionKernel(cfg)
    r = bk.solve_free_boundary(cc, ip, ped, ped, max_outer_iter=3, tol=1e-4, optimize_shape=True, target_points=pts,
                               current_limits=LIMITS_UQ, tikhonov_alpha=ALPHA_UQ)
    so = r["shape_optimization"]
    pos = [(c["r"], c["z"]) for c in cfg["coils"]]
    M = G.mutual_matrix(pos, [1] * len(pos), pts)
    A = np.vstack([M.T, np.sqrt(ALPHA_UQ) * np.eye(len(pos))])
    R, Z = bk.R, bk.Z
    bound_seen = False
    for b in range(6):
        t = G.shape_target_flux(r["psi"][b], R, Z, bk.dR, bk.dZ, pts)
        np.testing.assert_array_equal(so["target_flux"][b], t)
        x = r["coil_currents"][b]
        ref = lsq_linear(A, np.concatenate([t, np.zeros(len(pos))]), bounds=(-LIMITS_UQ, LIMITS_UQ), method="bvls").x
        np.testing.assert_allclose(x, ref, rtol=1e-10, atol=1e-10 * np.max(np.abs(ref)))
        g = A.T @ (A @ x - np.concatenate([t, np.zeros(len(pos))]))
        gs = 1e-9 * np.max(np.abs(A.T @ np.concatenate([t, np.zeros(len(pos))])))
        at_lo, at_hi = x <= -LIMITS_UQ, x >= LIMITS_UQ
        assert np.all(g[at_lo] >= -gs) and np.all(g[at_hi] <= gs) and np.all(np.abs(g[~at_lo & ~at_hi]) <= gs)
        bound_seen = bound_seen or bool((at_lo | at_hi).any())
        np.testing.assert_allclose(so["achieved_flux"][b], M.T @ x, rtol=1e-12, atol=1e-12 * np.max(np.abs(M.T @ x)))
        rr = so["achieved_flux"][b] - t
        np.testing.assert_allclose([so["flux_rmse"][b], so["max_abs_flux_residual"][b]],
                                   [np.sqrt(np.mean(rr ** 2)), np.max(np.abs(rr))], rtol=1e-12)
    assert bound_seen


def test_tight_limits_on_many_coils_random_targets(pkg):
    """The bounded fit where many currents sit on their limits, some of them on the limit of the opposite sign to where
    the active-set search first puts them: 12 coils, 16 points, alpha 1e-13, limits of 4 MA and 6 MA, and 512 random
    explicit targets (flux of currents up to 3 x the limits, either sign) in one batch.  Every row must be
    lsq_linear(method="bvls")'s minimiser and satisfy the KKT sign conditions."""
    from scipy.optimize import lsq_linear
    z = golden("free_boundary_shape")
    cfg = json.loads(str(z["cfg"]))
    extra = [(11.0, 5.0), (11.5, -5.5), (2.6, 6.8), (2.6, -6.8), (1.4, 3.2)]
    cfg["coils"] += [{"name": f"X{i}", "r": r, "z": zz, "current": 0.0} for i, (r, zz) in enumerate(extra)]
    pos = [(c["r"], c["z"]) for c in cfg["coils"]]
    n = len(pos)
    th = np.linspace(0.0, 2.0 * np.pi, 17)[:-1] + 0.1
    pts = np.column_stack([6.2 + 2.1 * np.cos(th), 3.2 * np.sin(th)])
    lim = np.full(n, 6e6)
    lim[::3] = 4e6
    alpha = 1e-13
    M = G.mutual_matrix(pos, [1] * n, pts)
    rng = np.random.default_rng(7)
    B = 512
    T = (rng.uniform(-3.0, 3.0, (B, n)) * lim) @ M
    cc = np.tile(np.r_[z["currents0"], np.zeros(len(extra))], (B, 1))
    bk = pkg.BatchedFusionKernel(cfg)
    r = bk.solve_free_boundary(cc, max_outer_iter=1, tol=0.0, optimize_shape=True, target_points=pts, target_values=T,
                               current_limits=lim, tikhonov_alpha=alpha)
    so = r["shape_optimization"]
    assert not so["fit_fallback"].any()
    A = np.vstack([M.T, np.sqrt(alpha) * np.eye(n)])
    both_signs = 0
    for b in range(B):
        rhs = np.concatenate([T[b], np.zeros(n)])
        x = r["coil_currents"][b]
        ref = lsq_linear(A, rhs, bounds=(-lim, lim), method="bvls").x
        np.testing.assert_allclose(x, ref, rtol=0, atol=1e-10 * np.max(np.abs(ref)), err_msg=f"row {b}")
        g = A.T @ (A @ x - rhs)
        gs = 1e-9 * np.max(np.abs(A.T @ rhs))
        at_lo, at_hi = x <= -lim, x >= lim
        assert np.all(g[at_lo] >= -gs) and np.all(g[at_hi] <= gs) and np.all(np.abs(g[~at_lo & ~at_hi]) <= gs), b
        assert int(so["active_current_bounds"][b]) == int(np.count_nonzero(at_lo | at_hi))
        both_signs += bool(at_lo.any() and at_hi.any())
    assert both_signs >= 100  # about 200 rows hold currents on limits of both signs


def test_per_equilibrium_independence(pkg):
    """A sample solved alone equals the same sample inside a batch, bit for bit; with max_outer_iter=1 nobody retires
    early and every equilibrium gets exactly one fit."""
    cfg = _uq_cfg(33)
    cc, ip, _ = _uq(cfg, 5)
    z = golden("free_boundary_shape")
    bk = pkg.BatchedFusionKernel(cfg)
    kw = dict(optimize_shape=True, target_points=z["pts"], current_limits=LIMITS_UQ, tikhonov_alpha=ALPHA_UQ)
    full = bk.solve_free_boundary(cc, ip, max_outer_iter=20, tol=1e-4, **kw)
    one = bk.solve_free_boundary(cc[3:4], ip[3:4], max_outer_iter=20, tol=1e-4, **kw)
    np.testing.assert_array_equal(full["psi"][3], one["psi"][0])
    np.testing.assert_array_equal(full["coil_currents"][3], one["coil_currents"][0])
    np.testing.assert_array_equal(full["shape_optimization"]["achieved_flux"][3],
                                  one["shape_optimization"]["achieved_flux"][0])
    assert int(full["outer_iterations"][3]) == int(one["outer_iterations"][0])
    capped = bk.solve_free_boundary(cc, ip, max_outer_iter=1, tol=1e-4, **kw)
    assert (capped["outer_iterations"] == 1).all() and not capped["fb_converged"].any()
    assert not np.array_equal(capped["coil_currents"], cc)


def test_no_points_is_the_plain_solve_and_plasma_wall(pkg, exact_fit):
    """optimize_shape=True without target points is the optimize_shape=False call, bit for bit (as the reference);
    plasma_wall=True with shape optimisation against the oracle's NumPy restatement at 33^2 (parity unpinned, as for
    plasma_wall alone)."""
    cfg = _uq_cfg(33)
    cc, ip, ped = _uq(cfg, 3)
    bk = pkg.BatchedFusionKernel(cfg)
    a = bk.solve_free_boundary(cc, ip, ped, ped, max_outer_iter=5, tol=1e-4)
    b = bk.solve_free_boundary(cc, ip, ped, ped, max_outer_iter=5, tol=1e-4, optimize_shape=True)
    assert set(a) == set(b) and "shape_optimization" not in b
    np.testing.assert_array_equal(a["psi"], b["psi"])
    np.testing.assert_array_equal(a["final_diff"], b["final_diff"])
    z = golden("free_boundary_shape")
    r = bk.solve_free_boundary(cc, ip, ped, ped, max_outer_iter=4, tol=1e-6, plasma_wall=True, wall_mu0=G.MU0_SI,
                               optimize_shape=True, target_points=z["pts"], current_limits=LIMITS_UQ,
                               tikhonov_alpha=ALPHA_UQ)
    _, ro = _oracle(cfg, cc[2], ip[2], ped[2], max_outer_iter=4, tol=1e-6, tikhonov_alpha=ALPHA_UQ,
                    target_points=z["pts"], current_limits=LIMITS_UQ, plasma_wall_mu0=G.MU0_SI)
    assert int(r["outer_iterations"][2]) == ro["outer_iterations"]
    assert rel_l2(r["psi"][2], ro["psi"]) <= PSI_TOL
    np.testing.assert_allclose(r["coil_currents"][2], ro["coil_currents"], rtol=1e-9, atol=0)


def test_argument_errors(pkg):
    z = golden("free_boundary_shape")
    cfg = json.loads(str(z["cfg"]))
    bk = pkg.BatchedFusionKernel(cfg)
    cc = np.tile(z["currents0"], (2, 1))
    pts = z["pts"]
    ok = dict(optimize_shape=True, target_points=pts, max_outer_iter=1)
    cases = [(dict(tikhonov_alpha=-1.0), "tikhonov_alpha must be finite and non-negative"),
             (dict(tikhonov_alpha=float("nan")), "tikhonov_alpha must be finite and non-negative"),
             (dict(current_limits=z["limits"][:-1]), "current_limits must have one entry per coil"),
             (dict(current_limits=np.r_[z["limits"][:-1], 0.0]), "current_limits must contain finite positive values"),
             (dict(current_limits=-z["limits"]), "current_limits must contain finite positive values"),
             (dict(target_values=z["explicit_targets"][:-1]), "target_flux_values must have the same length"),
             (dict(target_values=np.full((3, len(pts)), 1.0)), "target_flux_values must have the same length"),
             (dict(target_values=np.r_[z["explicit_targets"][:-1], np.nan]), "target_flux_values must contain finite"),
             (dict(target_points=pts[:, :1]), "target_flux_points must have shape"),
             (dict(target_points=np.r_[pts, [[np.inf, 0.0]]]), "target_flux_points must contain finite"),
             (dict(turns=[1.5] + [1] * 6), "turns must be positive integers")]
    for kw, msg in cases:
        with pytest.raises(ValueError, match=msg):
            bk.solve_free_boundary(cc, **{**ok, **kw})
    # alpha = 0 with fewer points than coils: [M^T; 0] is rank deficient
    with pytest.raises(ValueError, match="rank deficient"):
        bk.solve_free_boundary(cc, optimize_shape=True, target_points=pts[:3], tikhonov_alpha=0.0, max_outer_iter=1)
    many = json.loads(json.dumps(cfg))
    many["coils"] = [{"r": 11.0 + 0.01 * i, "z": 0.1 * i - 1.6, "current": 0.0} for i in range(33)]
    with pytest.raises(ValueError, match="at most 32 coils"):
        pkg.BatchedFusionKernel(many).solve_free_boundary(np.zeros((1, 33)), **ok)
