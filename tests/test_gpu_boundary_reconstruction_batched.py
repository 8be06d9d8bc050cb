"""GPU parity of the batched wall-contour boundary reconstruction (gsb_boundary_flux;
BatchedFusionKernel.reconstruct_boundary_flux_from_coils and solve_free_boundary(reconstruct_boundary=True)).

Every flux is sum_c M[c][p] I_c accumulated in coil order from 0.0 without contraction, with M the returned
response_matrix (the device Green's function), so it is restated bit for bit by the NumPy loop `_coil_order`; rmse,
max_abs_error and the X-point span are restated bit for bit from the returned arrays.  The reference's flux is a BLAS
matmul (unspecified order) on its own Green's function, so it is compared at rounding level (1e-12 of the flux scale),
and the shape case at the currents' 1e-7 (the device fit is the exact minimiser, the reference's stops trf).
"""
from __future__ import annotations

import json

import numpy as np
import pytest

import gs_oracle as G
from conftest import golden, golden_cfg, rel_l2

pytestmark = pytest.mark.gpu

LIMITER = np.array([[3.9, -4.6], [8.6, -4.6], [8.6, 4.6], [3.9, 4.6]])
AXIS = np.array([6.2, 0.0])
XPTS = np.array([[5.0, -3.4], [5.0, 3.4]])
GEO = dict(limiter_points=LIMITER, axis_point=AXIS, x_points=XPTS)


@pytest.fixture(scope="module")
def pkg():
    import scpn_fusion_core_b200 as p
    return p


def _coil_order(resp, cur):
    acc = np.zeros(resp.shape[1])
    for c in range(resp.shape[0]):
        acc = acc + resp[c] * cur[c]
    return acc


def _mutual(bk, pts):
    from scpn_fusion_core_b200.free_boundary import _mutual_device
    pos = [(c["r"], c["z"]) for c in bk.cfg["coils"]]
    return _mutual_device(bk.device, pos, np.ones(len(pos), dtype=np.int32), np.asarray(pts, dtype=np.float64))


def _restatements(bk, br, cur, b):
    """Bit-exact NumPy restatements of sample b of a batched result."""
    np.testing.assert_array_equal(br["reconstructed_flux"][b], _coil_order(br["response_matrix"], cur))
    if "limiter_points" in br:
        np.testing.assert_array_equal(br["limiter_flux"][b], _coil_order(_mutual(bk, br["limiter_points"]), cur))
    if br["x_point_count"]:
        xo = br["x_points"] if br["x_points"].ndim == 2 else br["x_points"][b]
        xf = br["x_point_flux"][b]
        np.testing.assert_array_equal(xf, _coil_order(_mutual(bk, xo), cur))
        assert br["x_point_flux_span"][b] == np.max(xf) - np.min(xf)
    if "residual" in br:
        res = br["residual"][b]
        t = br["target_flux"] if br["target_flux"].ndim == 1 else br["target_flux"][b]
        np.testing.assert_array_equal(res, br["reconstructed_flux"][b] - t)
        assert br["rmse"][b] == np.sqrt(np.mean(res ** 2)) and br["max_abs_error"][b] == np.max(np.abs(res))


def _uq_cfg(n):
    cfg = golden_cfg(golden("solves"), "iter129")
    cfg["grid_resolution"] = [n, n]
    cfg["physics"]["profiles"] = {"mode": "h-mode"}
    return cfg


def _uq(cfg, B, seed0=2026):
    base = np.array([c["current"] for c in cfg["coils"]]) * 1.0e6
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
    pd = dict(zip(("ped_top", "ped_width", "ped_height", "core_alpha"), (float(v) for v in ped)))
    c["physics"]["profiles"] = {"mode": "h-mode", "p_prime": pd, "ff_prime": dict(pd)}
    prob = G.PicardProblem(c)
    pos = [(q["r"], q["z"]) for q in c["coils"]]
    pw = kw.pop("plasma_wall_mu0", None)
    if pw is not None:
        kw["plasma_wall"] = G.wall_response_matrix(prob.R, prob.Z, pw)
    return G.free_boundary_solve(prob, pos, [float(v) for v in cc], [1] * len(pos), **kw)


def _close_to_oracle(br, ro, b, rtol):
    scale = float(np.max(np.abs(ro["reconstructed_flux"])))
    np.testing.assert_allclose(br["reconstructed_flux"][b], ro["reconstructed_flux"], rtol=0, atol=rtol * scale)
    np.testing.assert_allclose(br["limiter_flux"][b], ro["limiter_flux"], rtol=0, atol=rtol * scale)
    np.testing.assert_allclose(br["x_point_flux"][b], ro["x_point_flux"], rtol=0, atol=rtol * scale)
    assert abs(br["axis_flux"][b] - ro["axis_flux"]) <= rtol * scale
    assert abs(br["x_point_flux_span"][b] - ro["x_point_flux_span"]) <= rtol * scale
    for key in ("response_rank", "point_count", "coil_count", "limiter_point_count", "x_point_count",
                "min_limiter_distance_m", "boundary_containment_fraction", "boundary_containment_pass"):
        assert br[key] == ro[key], key
    np.testing.assert_array_equal(br["boundary_points"], ro["boundary_points"])


def test_reference_fixture_shape_case_inside_a_batch(pkg):
    """The fixture's shape case as sample 1 of a batch of 4 (the others start from perturbed currents): the fixture's
    br_* arrays and br_scalars at the tolerances of the one-sample test (test_gpu_free_boundary)."""
    z = golden("free_boundary_shape")
    bk = pkg.BatchedFusionKernel(json.loads(str(z["cfg"])))
    rng = np.random.default_rng(5)
    cc = z["currents0"][None, :] * rng.uniform(0.9, 1.1, (4, 7))
    cc[1] = z["currents0"]
    r = bk.solve_free_boundary(cc, max_outer_iter=3, tol=1e-4, optimize_shape=True, target_points=z["pts"],
                               current_limits=z["limits"], tikhonov_alpha=float(z["alpha"]), reconstruct_boundary=True,
                               **GEO)
    br, bs = r["boundary_reconstruction"], z["br_scalars"]
    assert int(r["outer_iterations"][1]) == int(z["meta"][0])
    np.testing.assert_allclose(r["coil_currents"][1], z["currents"], rtol=1e-7, atol=0)
    np.testing.assert_array_equal(br["boundary_points"], z["br_points"])
    np.testing.assert_allclose(br["reconstructed_flux"][1], z["br_flux"], rtol=1e-7, atol=1e-10)
    assert (br["response_rank"], br["point_count"], br["coil_count"], br["limiter_point_count"], br["x_point_count"]) == \
        (int(bs[0]), int(bs[1]), int(bs[2]), int(bs[3]), int(bs[8]))
    assert br["min_limiter_distance_m"] == bs[4] and br["boundary_containment_fraction"] == bs[5]
    assert float(br["boundary_containment_pass"]) == bs[6]
    np.testing.assert_allclose([br["axis_flux"][1], br["x_point_flux_span"][1]], [bs[7], bs[9]], rtol=1e-7)
    np.testing.assert_allclose(br["x_point_pair_symmetry_abs_error"][1], bs[10], rtol=1e-6)
    assert r["vacuum_boundary_abs_error"].shape == (4,)
    assert np.all(r["vacuum_boundary_abs_error"] <= 1e-9 * max(1.0, float(np.max(np.abs(z["br_flux"])))))
    np.testing.assert_array_equal(r["vacuum_boundary_abs_error"], br["max_abs_error"])
    np.testing.assert_allclose(br["limiter_flux"][1], z["br_limiter_flux"], rtol=1e-7)
    np.testing.assert_allclose(br["x_point_flux"][1], z["br_x_flux"], rtol=1e-7)
    # the currents read back from br_flux through the (exact) least-squares solve of the fixture's response
    back = np.linalg.lstsq(br["response_matrix"].T, z["br_flux"], rcond=None)[0]
    np.testing.assert_allclose(back, r["coil_currents"][1], rtol=1e-7)
    for b in range(4):
        _restatements(bk, br, r["coil_currents"][b], b)
    # the target is the coil flux of the final currents on the wall contour
    _, iz, ir = G.wall_contour(bk.R, bk.Z)
    ext = G.external_flux(bk.R, bk.Z, [(c["r"], c["z"]) for c in bk.cfg["coils"]], r["coil_currents"][1], [1] * 7)
    np.testing.assert_allclose(br["target_flux"][1], ext[iz, ir], rtol=0, atol=1e-12 * np.max(np.abs(ext)))


@pytest.mark.parametrize("mode", ["plain", "shape", "plasma_wall"])
def test_free_boundary_against_the_oracle(pkg, mode):
    """solve_free_boundary(reconstruct_boundary=True) sample by sample against the oracle's free_boundary_solve at 33^2.
    Without plasma_wall the imposed wall flux is the coil flux, so vacuum_boundary_abs_error is rounding; with it, the
    error is the size of the plasma wall term of the last outer iteration."""
    cfg = _uq_cfg(33)
    B = 3
    cc, ip, ped = _uq(cfg, B)
    bk = pkg.BatchedFusionKernel(cfg)
    z = golden("free_boundary_shape")
    kw = dict(max_outer_iter=4, tol=1e-6)
    okw = {}
    if mode == "shape":
        kw.update(optimize_shape=True, target_points=z["pts"], tikhonov_alpha=1e-10)
        okw.update(optimize_shape=True, target_points=z["pts"], tikhonov_alpha=1e-10)
    if mode == "plasma_wall":
        kw.update(plasma_wall=True, wall_mu0=G.MU0_SI)
        okw.update(plasma_wall_mu0=G.MU0_SI)
    r = bk.solve_free_boundary(cc, ip, ped, ped, reconstruct_boundary=True, **GEO, **kw)
    br = r["boundary_reconstruction"]
    for b in range(B):
        ro = _oracle(cfg, cc[b], ip[b], ped[b], max_outer_iter=4, tol=1e-6, **GEO, **okw)
        rb = ro["boundary_reconstruction"]
        assert int(r["outer_iterations"][b]) == ro["outer_iterations"]
        assert rel_l2(r["psi"][b], ro["psi"]) <= 1e-9
        _close_to_oracle(br, rb, b, 1e-7 if mode == "shape" else 1e-12)
        _restatements(bk, br, r["coil_currents"][b] if mode == "shape" else cc[b], b)
        scale = float(np.max(np.abs(rb["reconstructed_flux"])))
        if mode == "plasma_wall":
            wall = float(np.max(np.abs(rb["residual"])))
            assert wall > 1e-9 * scale  # the plasma wall term, a million times rounding
            np.testing.assert_allclose(br["residual"][b], rb["residual"], rtol=0, atol=1e-6 * wall)
            np.testing.assert_allclose([r["vacuum_boundary_abs_error"][b], br["rmse"][b]],
                                       [ro["vacuum_boundary_abs_error"], rb["rmse"]], rtol=1e-6)
        else:
            assert r["vacuum_boundary_abs_error"][b] <= 1e-12 * scale
            assert ro["vacuum_boundary_abs_error"] <= 1e-12 * scale
    if mode == "plain":
        # the target is the coil-flux ring bit for bit; psi's ring holds it up to the rounding of the Picard
        # under-relaxation (1-a) x + a x, which the reference's psi (and not its target) carries too
        from scpn_fusion_core_b200 import _device as D
        tr = np.ones(7)
        dev = bk.solve_free_boundary_device(D.to_device(cc * tr, bk.device), D.to_device(ip, bk.device),
                                            D.to_device(np.concatenate([ped, ped], axis=1), bk.device), **kw)
        _, iz, ir = G.wall_contour(bk.R, bk.Z)
        ext = dev["psi_ext"].cpu().numpy()
        for b in range(B):
            np.testing.assert_array_equal(br["target_flux"][b], ext[b][iz, ir])
            np.testing.assert_allclose(r["psi"][b][iz, ir], br["target_flux"][b], rtol=0,
                                       atol=4e-16 * np.max(np.abs(ext[b])))


def _standalone(B, seed):
    rng = np.random.default_rng(seed)
    th = np.linspace(0.0, 2.0 * np.pi, 51)[:-1]
    pts = np.column_stack([6.2 + 2.9 * np.cos(th), 4.1 * np.sin(th)])
    z = golden("free_boundary_shape")
    cur = z["currents0"][None, :] * rng.uniform(0.5, 1.5, (B, 7))
    tgt = rng.normal(size=(B, len(pts))) * 3.0 + 10.0
    ax = np.column_stack([rng.uniform(5.8, 6.6, B), rng.uniform(-0.3, 0.3, B)])
    xr = rng.uniform(4.8, 5.4, B)
    xz = rng.uniform(3.0, 3.6, B)
    xp = np.stack([np.column_stack([xr, ax[:, 1] - xz]), np.column_stack([xr, ax[:, 1] + xz])], axis=1)
    xp[::3, 1, 0] += 0.05  # every third pair is not mirrored about its axis
    return z, pts, cur, tgt, ax, xp


@pytest.mark.parametrize("per_sample", [False, True])
def test_standalone_against_the_oracle(pkg, per_sample):
    """reconstruct_boundary_flux_from_coils over 9 current vectors with per-sample targets, against the oracle's
    reconstruct_boundary_flux, with shared or per-sample axis and X-points."""
    B = 9
    z, pts, cur, tgt, ax, xp = _standalone(B, 4)
    bk = pkg.BatchedFusionKernel(json.loads(str(z["cfg"])))
    geo = dict(limiter_points=LIMITER, axis_point=ax if per_sample else AXIS, x_points=xp if per_sample else XPTS)
    br = bk.reconstruct_boundary_flux_from_coils(cur, boundary_points=pts, target_flux=tgt, **geo)
    pos = [(c["r"], c["z"]) for c in bk.cfg["coils"]]
    sym = br["x_point_pair_symmetry_abs_error"]
    assert sym.shape == (B,)
    for b in range(B):
        ro = G.reconstruct_boundary_flux(pos, [1] * 7, cur[b], pts, limiter_points=LIMITER,
                                         axis_point=ax[b] if per_sample else AXIS,
                                         x_points=xp[b] if per_sample else XPTS, target_flux=tgt[b])
        _close_to_oracle(br, ro, b, 1e-12)
        _restatements(bk, br, cur[b], b)
        np.testing.assert_allclose(br["residual"][b], ro["residual"], rtol=0, atol=1e-12 * np.max(np.abs(tgt)))
        np.testing.assert_allclose([br["rmse"][b], br["max_abs_error"][b]], [ro["rmse"], ro["max_abs_error"]], rtol=1e-10)
        if ro["x_point_pair_symmetry_abs_error"] is None:
            assert np.isnan(sym[b])
        else:
            assert abs(sym[b] - ro["x_point_pair_symmetry_abs_error"]) <= 1e-12 * float(np.max(np.abs(br["x_point_flux"][b])))
            assert sym[b] == abs(br["x_point_flux"][b][0] - br["x_point_flux"][b][1])
    if per_sample:
        assert np.isnan(sym[::3]).all() and not np.isnan(sym[1::3]).any()
    # no axis: None as in the reference; a shared pair that is not mirrored: None for every sample
    r2 = bk.reconstruct_boundary_flux_from_coils(cur, boundary_points=pts, x_points=XPTS)
    assert r2["x_point_pair_symmetry_abs_error"] is None and r2["axis_flux"] is None and "residual" not in r2
    r3 = bk.reconstruct_boundary_flux_from_coils(cur, boundary_points=pts, axis_point=[6.2, 0.5], x_points=XPTS)
    assert r3["x_point_pair_symmetry_abs_error"] is None
    # one current vector, config currents, shared (N,) target
    one = bk.reconstruct_boundary_flux_from_coils(cur[2], boundary_points=pts, target_flux=tgt[2])
    np.testing.assert_array_equal(one["reconstructed_flux"][0], br["reconstructed_flux"][2])
    np.testing.assert_array_equal(one["residual"][0], br["residual"][2])
    cfgc = bk.reconstruct_boundary_flux_from_coils(boundary_points=pts)
    np.testing.assert_array_equal(cfgc["reconstructed_flux"][0],
                                  _coil_order(cfgc["response_matrix"], [c["current"] for c in bk.cfg["coils"]]))


def test_off_means_off(pkg):
    """reconstruct_boundary=False: no extra launch, and the flag changes none of the solve's outputs.  With it the call
    adds two launches: the entry's mutual matrix (which is also the returned response_matrix) and k_boundary_flux."""
    from scpn_fusion_core_b200 import _lib
    cfg = _uq_cfg(33)
    cc, ip, ped = _uq(cfg, 3)
    bk = pkg.BatchedFusionKernel(cfg)
    kw = dict(max_outer_iter=4, tol=1e-4, plasma_wall=True)
    bk.solve_free_boundary(cc, ip, ped, ped, **kw)  # warm-up: context, tables
    n0 = _lib.launch_count()
    off = bk.solve_free_boundary(cc, ip, ped, ped, **kw)
    n1 = _lib.launch_count()
    on = bk.solve_free_boundary(cc, ip, ped, ped, reconstruct_boundary=True, **kw)
    n2 = _lib.launch_count()
    off2 = bk.solve_free_boundary(cc, ip, ped, ped, **kw)
    n3 = _lib.launch_count()
    assert n3 - n2 == n1 - n0 and (n2 - n1) - (n1 - n0) == 2
    assert set(on) - set(off) == {"boundary_reconstruction", "vacuum_boundary_abs_error"} and set(off2) == set(off)
    for key in off:
        if key != "wall_time_s":
            np.testing.assert_array_equal(on[key], off[key], err_msg=key)
            np.testing.assert_array_equal(off2[key], off[key], err_msg=key)


def test_batch_independence(pkg):
    """Permuting the batch permutes every per-sample output bit for bit; a batch of one equals its row."""
    B = 64
    z, pts, cur, tgt, ax, xp = _standalone(B, 9)
    bk = pkg.BatchedFusionKernel(json.loads(str(z["cfg"])))
    kw = dict(boundary_points=pts, limiter_points=LIMITER)
    full = bk.reconstruct_boundary_flux_from_coils(cur, target_flux=tgt, axis_point=ax, x_points=xp, **kw)
    perm = np.random.default_rng(2).permutation(B)
    pr = bk.reconstruct_boundary_flux_from_coils(cur[perm], target_flux=tgt[perm], axis_point=ax[perm],
                                                 x_points=xp[perm], **kw)
    keys = ("reconstructed_flux", "limiter_flux", "axis_flux", "x_point_flux", "x_point_flux_span",
            "x_point_pair_symmetry_abs_error", "residual", "rmse", "max_abs_error")
    for key in keys:
        np.testing.assert_array_equal(pr[key], full[key][perm], err_msg=key)
    for b in (0, 17, 63):
        one = bk.reconstruct_boundary_flux_from_coils(cur[b:b + 1], target_flux=tgt[b:b + 1], axis_point=ax[b:b + 1],
                                                      x_points=xp[b:b + 1], **kw)
        for key in keys:
            if one[key] is None:  # a lone sample whose X-point pair is not mirrored: None, as in the reference
                assert key == "x_point_pair_symmetry_abs_error" and np.isnan(full[key][b])
            else:
                np.testing.assert_array_equal(one[key][0], full[key][b], err_msg=key)
    # the solve path: a sample alone equals its row in a batch
    cfg = _uq_cfg(33)
    cc, ip, ped = _uq(cfg, 4)
    bs = pkg.BatchedFusionKernel(cfg)
    a = bs.solve_free_boundary(cc, ip, ped, ped, max_outer_iter=6, tol=1e-4, reconstruct_boundary=True, **GEO)
    o = bs.solve_free_boundary(cc[2:3], ip[2:3], ped[2:3], ped[2:3], max_outer_iter=6, tol=1e-4,
                               reconstruct_boundary=True, **GEO)
    for key in ("reconstructed_flux", "residual", "rmse", "max_abs_error", "axis_flux", "x_point_flux"):
        np.testing.assert_array_equal(o["boundary_reconstruction"][key][0], a["boundary_reconstruction"][key][2])


def test_point_arrays_in_any_memory_layout(pkg):
    """Fortran-ordered, transposed and strided point arrays (boundary, limiter, shared axis and X-points; per-sample axis
    and X-points) give the bits of the C-contiguous call: the entry reads every point array in storage order."""
    B = 5
    z, pts, cur, tgt, ax, xp = _standalone(B, 13)
    bk = pkg.BatchedFusionKernel(json.loads(str(z["cfg"])))
    keys = ("reconstructed_flux", "limiter_flux", "axis_flux", "x_point_flux", "x_point_flux_span",
            "x_point_pair_symmetry_abs_error", "residual", "rmse", "max_abs_error", "response_matrix")
    xs = np.array([[5.0, 5.0], [-3.4, 3.4]]).T  # transposed: XPTS, not C-contiguous
    axs = np.array([[6.2, 1.0], [0.0, 2.0]])[:, 0]  # strided column: (6.2, 0.0)
    assert not xs.flags.c_contiguous and not axs.flags.c_contiguous
    np.testing.assert_array_equal(xs, XPTS)
    np.testing.assert_array_equal(axs, AXIS)
    for geo, odd in ((dict(axis_point=AXIS, x_points=XPTS), dict(axis_point=axs, x_points=xs)),
                     (dict(axis_point=ax, x_points=xp), dict(axis_point=np.asfortranarray(ax), x_points=np.asfortranarray(xp)))):
        ref = bk.reconstruct_boundary_flux_from_coils(cur, boundary_points=pts, target_flux=tgt, limiter_points=LIMITER,
                                                      **geo)
        got = bk.reconstruct_boundary_flux_from_coils(cur, boundary_points=np.asfortranarray(pts), target_flux=tgt,
                                                      limiter_points=np.asfortranarray(LIMITER), **odd)
        for key in keys:
            np.testing.assert_array_equal(got[key], ref[key], err_msg=key)
        np.testing.assert_array_equal(got["axis_point"], ref["axis_point"])
        np.testing.assert_array_equal(got["x_points"], ref["x_points"])
    # the axis and X-points are the reference's: the X-point flux is that of XPTS, not of the storage-order pairs
    ro = G.reconstruct_boundary_flux([(c["r"], c["z"]) for c in bk.cfg["coils"]], [1] * 7, cur[0], pts, axis_point=AXIS,
                                     x_points=XPTS)
    scale = float(np.max(np.abs(ro["reconstructed_flux"])))
    odd_shared = bk.reconstruct_boundary_flux_from_coils(cur, boundary_points=pts, axis_point=axs, x_points=xs)
    np.testing.assert_allclose(odd_shared["x_point_flux"][0], ro["x_point_flux"], rtol=0, atol=1e-12 * scale)
    assert abs(odd_shared["axis_flux"][0] - ro["axis_flux"]) <= 1e-12 * scale


def test_non_finite_flux_and_target(pkg):
    """A sample whose flux overflows makes the method raise, naming it; a non-finite device target sets flag 2."""
    from scpn_fusion_core_b200 import _device as D
    z, pts, cur, tgt, ax, xp = _standalone(4, 1)
    bk = pkg.BatchedFusionKernel(json.loads(str(z["cfg"])))
    big = cur.copy()
    big[1] = 1e306
    with pytest.raises(ValueError, match=r"reconstructed boundary flux contains non-finite values in samples \[1\]"):
        bk.reconstruct_boundary_flux_from_coils(big, boundary_points=pts, turns=[2_000_000_000] * 7)
    t = tgt.copy()
    t[3, 7] = np.nan
    dev = bk.reconstruct_boundary_flux_device(D.to_device(cur, bk.device), boundary_points=pts,
                                              target_dev=D.to_device(t, bk.device))
    st = dev["stats"].cpu().numpy()
    assert st[:, 4].tolist() == [0.0, 0.0, 0.0, 2.0] and np.isnan(st[3, 0]) and np.isnan(st[3, 1])
    assert np.isnan(st[:, 2]).all() and np.isnan(st[:, 3]).all()  # no X-points


def test_argument_errors(pkg):
    """Every argument error raises ValueError with the reference's (or the device limit's) message before any launch."""
    from scpn_fusion_core_b200 import _device as D
    from scpn_fusion_core_b200 import _lib
    z, pts, cur, tgt, ax, xp = _standalone(3, 2)
    bk = pkg.BatchedFusionKernel(json.loads(str(z["cfg"])))
    ok = dict(boundary_points=pts, target_flux=tgt, limiter_points=LIMITER, axis_point=ax, x_points=xp)
    th = np.linspace(0.0, 2.0 * np.pi, 4098)[:-1]
    many = np.column_stack([6.2 + 2.0 * np.cos(th), 3.0 * np.sin(th)])
    cases = [(dict(boundary_points=pts[:, :1]), "boundary_points must have shape"),
             (dict(boundary_points=np.r_[pts[:-1], [[np.nan, 0.0]]]), "boundary_points must contain finite values"),
             (dict(boundary_points=many, target_flux=None), "at most 4096 boundary points"),
             (dict(boundary_points=np.r_[pts[:-1], [[0.0, 0.0]]]), "observation radii must be positive"),
             (dict(limiter_points=LIMITER[:, :1]), "limiter_points must have shape"),
             (dict(limiter_points=LIMITER[:2]), "polygon must contain at least three points"),
             (dict(limiter_points=many), "at most 4096 limiter points"),
             (dict(axis_point=[6.2, 0.0, 1.0]), r"axis_point must have shape \(2,\) or \(3, 2\)"),
             (dict(axis_point=[np.inf, 0.0]), "axis_point must contain finite values"),
             (dict(x_points=xp[:2]), r"x_points must have shape \(n_points, 2\) or \(3, n_points, 2\)"),
             (dict(x_points=XPTS[:, :1]), "x_points must have shape"),
             (dict(x_points=np.r_[XPTS, [[np.nan, 1.0]]]), "x_points must contain finite values"),
             (dict(x_points=np.tile(XPTS, (33, 1))), "at most 64 X-points"),
             (dict(target_flux=tgt[:, :-1]), f"target_flux must have length {len(pts)}"),
             (dict(target_flux=tgt[0, :-1]), f"target_flux must have length {len(pts)}"),
             (dict(target_flux=np.r_[tgt[0, :-1], np.nan]), "target_flux must contain finite values"),
             (dict(coil_currents=cur[:, :-1]), "currents must have length 7"),
             (dict(coil_currents=np.full((3, 7), np.nan)), "currents must contain finite values"),
             (dict(turns=[1.5] + [1] * 6), "turns must be positive integers"),
             (dict(turns=[1] * 6), "turns must be positive integers")]
    n0 = _lib.launch_count()
    for kw, msg in cases:
        args = {**ok, **kw}
        with pytest.raises(ValueError, match=msg):
            bk.reconstruct_boundary_flux_from_coils(args.pop("coil_currents", cur), **args)
    cc = np.tile(z["currents0"], (2, 1))
    for kw in (dict(limiter_points=LIMITER), dict(axis_point=AXIS), dict(x_points=XPTS)):
        with pytest.raises(ValueError, match="need reconstruct_boundary=True"):
            bk.solve_free_boundary(cc, max_outer_iter=1, **kw)
    with pytest.raises(ValueError, match="turns must be positive integers"):
        bk.solve_free_boundary(cc, max_outer_iter=1, turns=[1.5] + [1] * 6, reconstruct_boundary=True)
    assert _lib.launch_count() == n0
    cd = D.to_device(cur, bk.device)
    n0 = _lib.launch_count()
    with pytest.raises(ValueError, match="wall contour of the grid"):
        bk.reconstruct_boundary_flux_device(cd, boundary_points=pts, target_field=D.zeros((3, bk.NZ, bk.NR), bk.device))
    with pytest.raises(ValueError, match="currents_dev must be a contiguous CUDA float64 tensor"):
        bk.reconstruct_boundary_flux_device(cd[:, :6].contiguous(), boundary_points=pts)
    with pytest.raises(ValueError, match="target_dev must be a contiguous CUDA float64 tensor"):
        bk.reconstruct_boundary_flux_device(cd, boundary_points=pts, target_dev=D.zeros((2, len(pts)), bk.device))
    assert _lib.launch_count() == n0
    # the C entry's own checks, before its first launch
    lib = _lib.load()
    pos = np.ascontiguousarray([(c["r"], c["z"]) for c in bk.cfg["coils"]], dtype=np.float64)
    turns = np.ones(7, dtype=np.int32)
    wall = np.ascontiguousarray(G.wall_contour(bk.R, bk.Z)[0])
    import ctypes
    dp = ctypes.POINTER(ctypes.c_double)

    def call(**over):
        bp = _lib.gsb_boundary_params()
        bp.n_coils, bp.coil_rz, bp.turns = 7, pos.ctypes.data_as(dp), turns.ctypes.data_as(ctypes.POINTER(ctypes.c_int))
        bp.n_points, bp.points = len(wall), wall.ctypes.data_as(dp)
        bp.target_mode, bp.nz, bp.nr = 3, bk.NZ, bk.NR
        r_ax, z_ax = np.ascontiguousarray(bk.R), np.ascontiguousarray(bk.Z)
        bp.r_axis, bp.z_axis = r_ax.ctypes.data_as(dp), z_ax.ctypes.data_as(dp)
        for k, v in over.items():
            setattr(bp, k, v)
        need = ctypes.c_longlong(0)
        null = ctypes.c_void_p()
        rc = lib.gsb_boundary_flux(ctypes.byref(bp), null, null, null, null, null, null, ctypes.byref(need), 2, null)
        if rc == 0:
            work = D.empty(((need.value + 7) // 8,), bk.device)
            f, s = D.empty((2, len(wall)), bk.device), D.empty((2, 5), bk.device)
            res, fld = D.empty((2, len(wall)), bk.device), D.zeros((2, bk.NZ, bk.NR), bk.device)
            rc = lib.gsb_boundary_flux(ctypes.byref(bp), D.ptr(cd[:2].contiguous()), D.ptr(fld), D.ptr(f), D.ptr(res),
                                       D.ptr(s), D.ptr(work), ctypes.byref(need), 2, D.stream_ptr())
        return rc, _lib.last_error()

    n0 = _lib.launch_count()
    assert call(n_points=0)[1].startswith("boundary reconstruction supports 1 to 4096 boundary points")
    assert call(n_xpoints=65)[1].startswith("boundary reconstruction supports at most 64 X-points")
    assert call(target_mode=4)[1].startswith("gsb_boundary_flux: target_mode")
    assert "N = 2 nr + 2 nz - 4" in call(n_points=len(wall) - 1)[1]
    wall[5, 1] += 1e-9
    assert "wall contour of the grid" in call()[1]
    wall[5, 1] -= 1e-9
    assert _lib.launch_count() == n0
    rc, _ = call()
    assert rc == 0 and _lib.launch_count() == n0 + 2
