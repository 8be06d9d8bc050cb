"""GPU parity of the batched magnetic-probe current reconstruction (gsb_probe_reconstruct;
BatchedFusionKernel.reconstruct_coil_currents_from_magnetic_probes).

The device computes the EXACT bounded minimiser of |w (R x - meas)|^2 + alpha |x - prior|^2 (bounded-variable least
squares on the QR factor of [diag(w) R; sqrt(alpha) I]), while the reference stops scipy's interior-point
lsq_linear(method="trf") at its tolerance.  On the fixture's probe problem the optimum is interior and trf, bvls and the
unbounded solution agree bit for bit (test_probe_fit_cpu), so the device matches the fixture to the accuracy of its own
response matrix.  With active limits the currents are compared tightly with the oracle whose fit is
lsq_linear(method="bvls") (`exact_lsq` below) and loosely with the default trf oracle.  The residual is a BLAS matmul
in the reference (unspecified summation order), so it is compared at rounding level.
"""
from __future__ import annotations

import json

import numpy as np
import pytest

import gs_oracle as G
from conftest import golden

pytestmark = pytest.mark.gpu

EXTRA_COILS = [(11.0, 5.0), (11.5, -5.5), (2.6, 6.8), (2.6, -6.8), (1.4, 3.2)]


@pytest.fixture(scope="module")
def pkg():
    import scpn_fusion_core_b200 as p
    return p


@pytest.fixture
def exact_lsq(monkeypatch):
    """The oracle with lsq_linear(method="bvls") in place of trf."""
    import scipy.optimize as so
    orig = so.lsq_linear
    monkeypatch.setattr(so, "lsq_linear", lambda A, b, bounds, method="trf": orig(A, b, bounds=bounds, method="bvls"))


def _fixture(pkg):
    z = golden("free_boundary_shape")
    return z, pkg.BatchedFusionKernel(json.loads(str(z["cfg"])))


def _device_response(pkg, bk, **kw):
    """The response matrix the method builds (device Green's function, host differencing)."""
    from scpn_fusion_core_b200.free_boundary import build_magnetic_probe_response_matrix
    coils = pkg.CoilSet(positions=[(c["r"], c["z"]) for c in bk.cfg["coils"]],
                        currents=np.array([c["current"] for c in bk.cfg["coils"]]), turns=[1] * len(bk.cfg["coils"]))
    return build_magnetic_probe_response_matrix(bk, coils, **kw)


def _diagnostics():
    """10 flux loops and 12 B probes (alternating R and Z) on two ellipses outside the plasma."""
    th = np.linspace(0.0, 2.0 * np.pi, 11)[:-1] + 0.05
    fl = np.column_stack([6.2 + 3.6 * np.cos(th), 5.0 * np.sin(th)])
    tb = np.linspace(0.0, 2.0 * np.pi, 13)[:-1] + 0.2
    bp = np.column_stack([6.2 + 3.3 * np.cos(tb), 4.7 * np.sin(tb)])
    return fl, bp, ["R" if i % 2 == 0 else "Z" for i in range(len(tb))]


def _tight_problem(pkg, B, seed=11):
    """12 coils with 4 MA and 6 MA limits, noisy measurements of currents up to 2 x the limits, priors inside and
    outside the limits."""
    z = golden("free_boundary_shape")
    cfg = json.loads(str(z["cfg"]))
    cfg["coils"] += [{"name": f"X{i}", "r": r, "z": zz, "current": 0.0} for i, (r, zz) in enumerate(EXTRA_COILS)]
    bk = pkg.BatchedFusionKernel(cfg)
    fl, bp, dirs = _diagnostics()
    geo = dict(flux_points=fl, b_probe_points=bp, b_probe_directions=dirs)
    R = _device_response(pkg, bk, **geo)
    n, nf = R.shape[1], len(fl)
    lim = np.full(n, 6e6)
    lim[::3] = 4e6
    sg = np.r_[np.full(nf, 2e-3), np.full(len(bp), 1e-4)]
    rng = np.random.default_rng(seed)
    meas = (rng.uniform(-2.0, 2.0, (B, n)) * lim) @ R.T + rng.normal(size=(B, R.shape[0])) * sg
    prior = rng.uniform(-2.0, 2.0, (B, n)) * lim
    kw = dict(geo, flux_measurements=meas[:, :nf], b_probe_measurements=meas[:, nf:], measurement_sigma=sg,
              current_limits=lim, coil_currents=prior, tikhonov_alpha=1e-13)
    return bk, R, meas, prior, sg, lim, kw


def _kkt(R, w, alpha, meas, prior, x, lim):
    A = np.vstack([R * w[:, None], np.sqrt(alpha) * np.eye(len(x))])
    rhs = np.concatenate([meas * w, np.sqrt(alpha) * prior])
    g = A.T @ (A @ x - rhs)
    gs = 1e-9 * np.max(np.abs(A.T @ rhs))
    at_lo, at_hi = x <= -lim, x >= lim
    assert np.all(g[at_lo] >= -gs) and np.all(g[at_hi] <= gs) and np.all(np.abs(g[~at_lo & ~at_hi]) <= gs)
    return at_lo, at_hi


def test_reference_fixture_inside_a_batch(pkg):
    """The fixture's probe problem as sample 2 of a batch of 5 (the others carry perturbed measurements)."""
    z, bk = _fixture(pkg)
    fl, bp, dirs = z["probe_flux_pts"], z["probe_b_pts"], [str(d) for d in z["probe_dirs"]]
    meas, nf = z["probe_meas"], len(fl)
    rng = np.random.default_rng(3)
    mb = meas * (1.0 + 0.01 * rng.standard_normal((5, meas.size)))
    mb[2] = meas
    r = bk.reconstruct_coil_currents_from_magnetic_probes(
        flux_points=fl, flux_measurements=mb[:, :nf], b_probe_points=bp, b_probe_directions=dirs,
        b_probe_measurements=mb[:, nf:], measurement_sigma=z["probe_sigma"], tikhonov_alpha=1e-6,
        coil_currents=z["currents0"], current_limits=z["limits"])
    ps = z["probe_scalars"]
    # the device's B-probe rows differ from the fixture's at ~1e-8 (centred differences of G, test_gpu_free_boundary)
    np.testing.assert_allclose(r["coil_currents"][2], z["probe_currents"], rtol=1e-8, atol=1e-3)
    np.testing.assert_allclose(r["residual"][2], z["probe_residual"], rtol=0, atol=1e-6 * np.max(np.abs(meas)))
    np.testing.assert_allclose([r["residual_rms"][2], r["weighted_residual_rms"][2]], ps[:2], rtol=1e-5)
    assert r["response_rank"] == int(ps[2]) and int(r["active_bounds"][2]) == int(ps[4]) == 0
    np.testing.assert_allclose(r["response_condition"], ps[3], rtol=1e-5)
    # against the oracle on the device's own response matrix: trf = bvls = the interior optimum
    R = _device_response(pkg, bk, flux_points=fl, b_probe_points=bp, b_probe_directions=dirs)
    for b in range(5):
        ro = G.reconstruct_currents_from_probes(R, mb[b], z["currents0"], sigma=z["probe_sigma"], limits=z["limits"],
                                                alpha=1e-6)
        np.testing.assert_allclose(r["coil_currents"][b], ro["coil_currents"], rtol=1e-10, atol=1e-10 * 2e7)
        scale = np.max(np.abs(R @ ro["coil_currents"])) + np.max(np.abs(mb[b]))
        np.testing.assert_allclose(r["residual"][b], ro["residual"], rtol=0, atol=1e-9 * scale)
        np.testing.assert_array_equal(r["weighted_residual"][b], r["residual"][b] * (1.0 / z["probe_sigma"]))
        np.testing.assert_allclose([r["residual_rms"][b], r["weighted_residual_rms"][b]],
                                   [ro["residual_rms"], ro["weighted_residual_rms"]], rtol=1e-7)
        assert int(r["active_bounds"][b]) == ro["active_bounds"]


def test_tight_limits_random_batch_vs_exact_oracle(pkg, exact_lsq):
    """4096 samples, 12 coils, 4-6 MA limits, 10 flux loops and 12 R/Z probes: every sample is the oracle's with the
    exact (bvls) fit, satisfies the KKT sign conditions, and counts its active bounds with np.isclose."""
    B = 4096
    bk, R, meas, prior, sg, lim, kw = _tight_problem(pkg, B)
    r = bk.reconstruct_coil_currents_from_magnetic_probes(**kw)
    assert r["coil_currents"].shape == (B, 12) and r["residual"].shape == (B, 22)
    w = 1.0 / sg
    both = free = 0
    for b in range(B):
        x = r["coil_currents"][b]
        ro = G.reconstruct_currents_from_probes(R, meas[b], prior[b], sigma=sg, limits=lim, alpha=1e-13)
        ref = ro["coil_currents"]
        np.testing.assert_allclose(x, ref, rtol=0, atol=1e-10 * np.max(np.abs(ref)), err_msg=f"sample {b}")
        at_lo, at_hi = _kkt(R, w, 1e-13, meas[b], prior[b], x, lim)
        close = np.isclose(x, -lim) | np.isclose(x, lim)
        assert not np.any((at_lo | at_hi) & ~close) and int(r["active_bounds"][b]) == int(np.count_nonzero(close)), b
        both += bool(at_lo.any() and at_hi.any())
        free += int(np.count_nonzero(~at_lo & ~at_hi))
        res = R @ x - meas[b]
        np.testing.assert_allclose(r["residual"][b], res, rtol=0, atol=1e-12 * np.max(np.abs(meas[b])))
        np.testing.assert_allclose([r["residual_rms"][b], r["weighted_residual_rms"][b]],
                                   [np.sqrt(np.mean(res ** 2)), np.sqrt(np.mean((res * w) ** 2))], rtol=1e-9)
    assert both >= B // 2 and free >= B
    inside = np.all(np.abs(prior) <= lim, axis=1)
    assert inside.any() and not inside.all()


def test_random_samples_vs_default_trf_oracle(pkg):
    """The unmodified oracle (trf, as the reference): trf stops within ~1e-8 of the limits' scale."""
    bk, R, meas, prior, sg, lim, kw = _tight_problem(pkg, 16)
    r = bk.reconstruct_coil_currents_from_magnetic_probes(**kw)
    for b in range(16):
        ro = G.reconstruct_currents_from_probes(R, meas[b], prior[b], sigma=sg, limits=lim, alpha=1e-13)
        np.testing.assert_allclose(r["coil_currents"][b], ro["coil_currents"], rtol=0, atol=1e-7 * np.max(lim))


def test_alpha_zero_and_unbounded(pkg, exact_lsq):
    """alpha = 0 with full rank drops the prior rows (as the reference); no limits is np.linalg.lstsq of the weighted
    system."""
    bk, R, meas, prior, sg, lim, kw = _tight_problem(pkg, 64, seed=5)
    w = 1.0 / sg
    r0 = bk.reconstruct_coil_currents_from_magnetic_probes(**{**kw, "tikhonov_alpha": 0.0})
    r0b = bk.reconstruct_coil_currents_from_magnetic_probes(**{**kw, "tikhonov_alpha": 0.0, "coil_currents": None})
    np.testing.assert_array_equal(r0["coil_currents"], r0b["coil_currents"])  # the prior is not used
    for b in range(0, 64, 7):
        ro = G.reconstruct_currents_from_probes(R, meas[b], prior[b], sigma=sg, limits=lim, alpha=0.0)
        np.testing.assert_allclose(r0["coil_currents"][b], ro["coil_currents"], rtol=0,
                                   atol=1e-10 * np.max(np.abs(ro["coil_currents"])))
        _kkt(R, w, 0.0, meas[b], prior[b], r0["coil_currents"][b], lim)
    ru = bk.reconstruct_coil_currents_from_magnetic_probes(**{**kw, "current_limits": None})
    assert (ru["active_bounds"] == 0).all()
    A = np.vstack([R * w[:, None], np.sqrt(1e-13) * np.eye(12)])
    for b in range(0, 64, 5):
        x = np.linalg.lstsq(A, np.concatenate([meas[b] * w, np.sqrt(1e-13) * prior[b]]), rcond=None)[0]
        np.testing.assert_allclose(ru["coil_currents"][b], x, rtol=0, atol=1e-9 * np.max(np.abs(x)))


def test_rank_deficient_alpha_zero_is_refused_before_the_fit(pkg):
    """alpha = 0 with 4 flux loops for 7 coils: [diag(w) R; 0] is rank deficient.  ValueError after the mutual-matrix
    launch of the response and the factor launch, and no fit launch."""
    from scpn_fusion_core_b200 import _lib
    z, bk = _fixture(pkg)
    fl = z["probe_flux_pts"][:4]
    n0 = _lib.launch_count()
    with pytest.raises(ValueError, match="rank deficient"):
        bk.reconstruct_coil_currents_from_magnetic_probes(flux_points=fl, flux_measurements=z["probe_meas"][:4],
                                                          tikhonov_alpha=0.0)
    assert _lib.launch_count() - n0 == 2
    r = bk.reconstruct_coil_currents_from_magnetic_probes(flux_points=fl, flux_measurements=z["probe_meas"][:4],
                                                          tikhonov_alpha=1e-6)
    assert r["response_rank"] == 4


def test_batch_independence(pkg):
    """Permuting the batch permutes the results bit for bit; a batch of one equals its row in a batch of 4096."""
    bk, R, meas, prior, sg, lim, kw = _tight_problem(pkg, 4096, seed=21)
    full = bk.reconstruct_coil_currents_from_magnetic_probes(**kw)
    perm = np.random.default_rng(1).permutation(4096)
    pk = dict(kw, flux_measurements=kw["flux_measurements"][perm], b_probe_measurements=kw["b_probe_measurements"][perm],
              coil_currents=prior[perm])
    pr = bk.reconstruct_coil_currents_from_magnetic_probes(**pk)
    for key in ("coil_currents", "residual", "weighted_residual", "residual_rms", "weighted_residual_rms",
                "active_bounds"):
        np.testing.assert_array_equal(pr[key], full[key][perm], err_msg=key)
    for b in (0, 1234, 4095):
        one = bk.reconstruct_coil_currents_from_magnetic_probes(
            **dict(kw, flux_measurements=kw["flux_measurements"][b], b_probe_measurements=kw["b_probe_measurements"][b],
                   coil_currents=prior[b]))
        for key in ("coil_currents", "residual", "weighted_residual", "residual_rms", "active_bounds"):
            np.testing.assert_array_equal(one[key][0], full[key][b], err_msg=key)


def test_failure_flag_and_runtime_error(pkg):
    """max_iter=1 through the C entry flags the samples that need more free-set solves and leaves their clipped prior;
    a sample whose weighted measurements overflow makes the public method raise, naming it."""
    from scpn_fusion_core_b200 import _device as D
    bk, R, meas, prior, sg, lim, kw = _tight_problem(pkg, 256)
    dev = bk.reconstruct_coil_currents_device(R, D.to_device(meas, bk.device), D.to_device(prior, bk.device),
                                              measurement_sigma=sg, tikhonov_alpha=1e-13, current_limits=lim,
                                              max_iter=1)
    st, cur = dev["stats"].cpu().numpy(), dev["currents"].cpu().numpy()
    failed = st[:, 3] > 0.5
    assert failed.any() and not failed.all()
    np.testing.assert_array_equal(cur[failed], np.clip(prior[failed], -lim, lim))
    ok = bk.reconstruct_coil_currents_from_magnetic_probes(**kw)
    np.testing.assert_array_equal(cur[~failed], ok["coil_currents"][~failed])
    fm = kw["flux_measurements"][:8].copy()
    fm[5, 0] = 1e306  # x 1/sigma = 500 overflows
    with pytest.raises(RuntimeError, match=r"Magnetic probe inverse reconstruction failed: .*samples \[5\]"):
        bk.reconstruct_coil_currents_from_magnetic_probes(**dict(kw, flux_measurements=fm,
                                                                 b_probe_measurements=kw["b_probe_measurements"][:8],
                                                                 coil_currents=prior[:8]))


def test_argument_errors(pkg):
    z, bk = _fixture(pkg)
    fl, bp, dirs = z["probe_flux_pts"], z["probe_b_pts"], [str(d) for d in z["probe_dirs"]]
    meas, nf = z["probe_meas"], len(fl)
    ok = dict(flux_points=fl, flux_measurements=meas[:nf], b_probe_points=bp, b_probe_directions=dirs,
              b_probe_measurements=meas[nf:], measurement_sigma=z["probe_sigma"], current_limits=z["limits"])
    cases = [(dict(flux_points=None, b_probe_points=None, flux_measurements=None, b_probe_measurements=None),
              "At least one flux point or B probe point must be provided"),
             (dict(flux_measurements=None), "flux_measurements must be provided with flux_points"),
             (dict(flux_points=None, measurement_sigma=None), "flux_points must be provided with flux_measurements"),
             (dict(b_probe_measurements=None), "b_probe_measurements must be provided with b_probe_points"),
             (dict(b_probe_directions=None), "b_probe_directions must be provided with b_probe_points"),
             (dict(b_probe_directions=dirs[:-1]), "b_probe_directions must have one entry per b_probe_point"),
             (dict(b_probe_directions=["Q"] + dirs[1:]), "b_probe_directions entries must be 'R' or 'Z'"),
             (dict(flux_points=fl[:, :1]), "flux_points must have shape"),
             (dict(flux_measurements=meas[:nf - 1]), f"flux_measurements must have length {nf}"),
             (dict(flux_measurements=np.r_[meas[:nf - 1], np.nan]), "flux_measurements must contain finite values"),
             (dict(b_probe_measurements=np.zeros((2, 3, 2))), "b_probe_measurements must have length"),
             (dict(flux_measurements=np.tile(meas[:nf], (3, 1)), b_probe_measurements=np.tile(meas[nf:], (2, 1))),
              "must have the same batch size"),
             (dict(measurement_sigma=z["probe_sigma"][:-1]), "measurement_sigma must have length"),
             (dict(measurement_sigma=-z["probe_sigma"]), "measurement_sigma must contain finite positive values"),
             (dict(tikhonov_alpha=-1.0), "tikhonov_alpha must be finite and non-negative"),
             (dict(tikhonov_alpha=float("inf")), "tikhonov_alpha must be finite and non-negative"),
             (dict(coil_currents=np.zeros(6)), "CoilSet.currents must be finite with one entry per coil"),
             (dict(coil_currents=np.full(7, np.nan)), "CoilSet.currents must be finite with one entry per coil"),
             (dict(current_limits=z["limits"][:-1]), "current_limits must have length 7"),
             (dict(current_limits=np.r_[z["limits"][:-1], np.inf]), "current_limits must contain finite values only"),
             (dict(current_limits=-z["limits"]), "current_limits must contain finite positive values only"),
             (dict(turns=[1.5] + [1] * 6), "turns must be positive integers"),
             (dict(turns=[1] * 6), "turns must be positive integers")]
    for kw, msg in cases:
        with pytest.raises(ValueError, match=msg):
            bk.reconstruct_coil_currents_from_magnetic_probes(**{**ok, **kw})
    many = json.loads(str(z["cfg"]))
    many["coils"] = [{"r": 11.0 + 0.01 * i, "z": 0.1 * i - 1.6, "current": 0.0} for i in range(33)]
    with pytest.raises(ValueError, match="at most 32 coils"):
        pkg.BatchedFusionKernel(many).reconstruct_coil_currents_from_magnetic_probes(**ok)
    th = np.linspace(0.0, 2.0 * np.pi, 1026)[:-1]
    far = np.column_stack([6.2 + 4.0 * np.cos(th), 5.5 * np.sin(th)])
    with pytest.raises(ValueError, match="at most 1024 measurements"):
        bk.reconstruct_coil_currents_from_magnetic_probes(flux_points=far, flux_measurements=np.zeros(1025))
