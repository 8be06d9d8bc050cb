"""GPU parity of the batched, device-resident free-boundary outer loop (gsb_free_boundary_solve;
BatchedFusionKernel.solve_free_boundary) - the north_star workload: B independent free-boundary equilibria.

Lane A (wall = coil Green's-function flux, fusion_kernel_free_boundary.py:623-739): pinned against the fixture the
unmodified reference produced (tests/golden/free_boundary.npz) and, sample by sample, against the oracle restatement
`gs_oracle.free_boundary_solve` (itself pinned by tests/test_oracle_vs_golden.py).  Tolerances: relative L2 of psi
<= 1e-9, outer iteration counts equal, Picard iteration totals within +-1 per inner solve.

plasma_wall=True (lane-C wall term M @ (J dA), jax_free_boundary_predictive.py:443-498, on the FP64 tensor pipe inside
the loop): PARITY UNPINNED - jax is absent, no reference run exists; the checker is the oracle's NumPy restatement only.
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


@pytest.fixture(scope="module")
def pkg():
    import scpn_fusion_core_b200 as p
    return p


def _uq(cfg, B, seed0=2026, coil_scale=1.0e6):
    """bench.py's free-boundary inputs: SURVEY.md 8d config 3 recipe, coil currents in SI amperes (x 1e6, as the
    reference-generated fixture does) so that the SI-mu0 wall flux is O(1)."""
    base = np.array([c["current"] for c in cfg["coils"]]) * coil_scale
    cc, ip, ped = [], [], []
    for ks in range(B):
        rng = np.random.default_rng(seed0 + ks)
        cc.append(base * rng.uniform(0.85, 1.15, size=len(base)))
        ip.append(cfg["physics"]["plasma_current_target"] * rng.uniform(0.8, 1.2))
        ped.append([0.92 * rng.uniform(0.97, 1.03), 0.05 * rng.uniform(0.9, 1.1), 1.0 * rng.uniform(0.9, 1.1),
                    0.3 * rng.uniform(0.9, 1.1)])
    return np.array(cc), np.array(ip), np.array(ped)


def _oracle(cfg, cc, ip, ped, *, max_outer_iter, tol, plasma_wall_mu0=None):
    c = json.loads(json.dumps(cfg))
    for coil, cur in zip(c["coils"], cc):
        coil["current"] = float(cur)
    c["physics"]["plasma_current_target"] = float(ip)
    if ped is not None:
        pd = dict(zip(("ped_top", "ped_width", "ped_height", "core_alpha"), (float(v) for v in ped)))
        c["physics"]["profiles"] = {"mode": "h-mode", "p_prime": pd, "ff_prime": dict(pd)}
    prob = G.PicardProblem(c)
    pos = [(q["r"], q["z"]) for q in c["coils"]]
    pw = None if plasma_wall_mu0 is None else G.wall_response_matrix(prob.R, prob.Z, plasma_wall_mu0)
    r = G.free_boundary_solve(prob, pos, [float(v) for v in cc], [1] * len(pos), max_outer_iter=max_outer_iter, tol=tol,
                              plasma_wall=pw)
    return prob, r


def test_lane_a_matches_the_reference_fixture(pkg):
    """The reference's own solve_free_boundary result (free_boundary.npz), replicated 3x in one batch."""
    z = golden("free_boundary")
    cfg = json.loads(str(z["cfg"]))
    bk = pkg.BatchedFusionKernel(cfg)
    cc = np.tile(z["currents"], (3, 1))
    r = bk.solve_free_boundary(cc, max_outer_iter=4, tol=1e-4)
    for b in range(3):
        assert int(r["outer_iterations"][b]) == int(z["meta"][0])
        assert rel_l2(r["psi"][b], z["psi"]) <= PSI_TOL
        assert abs(r["final_diff"][b] - z["meta"][1]) <= 1e-7 * abs(z["meta"][1])
    np.testing.assert_array_equal(r["psi"][0], r["psi"][1])
    with pytest.raises(ValueError):
        bk.solve_free_boundary(cc, max_outer_iter=0)
    with pytest.raises(ValueError):
        bk.solve_free_boundary(cc, tol=float("nan"))


@pytest.mark.parametrize("n,B,streaming", [(65, 4, False), (129, 3, False), (65, 2, True), (257, 2, True)])
def test_lane_a_uq_samples_vs_oracle(pkg, n, B, streaming):
    """bench.py's headline workload (H-mode UQ sweep, free boundary), sample by sample against the oracle: on the
    resident kernel (<= 129^2), forced onto the streaming Picard loop, and at 257^2 (BASELINE configs[1] shape)."""
    cfg = golden_cfg(golden("solves"), "iter129")
    cfg["grid_resolution"] = [n, n]
    cfg["physics"]["profiles"] = {"mode": "h-mode"}
    cc, ip, ped = _uq(cfg, B)
    bk = pkg.BatchedFusionKernel(cfg)
    if streaming and n <= 129:
        os.environ["GSB_PICARD_STREAMING"] = "1"
    try:
        r = bk.solve_free_boundary(cc, ip, ped, ped, max_outer_iter=20, tol=1e-4)
    finally:
        os.environ.pop("GSB_PICARD_STREAMING", None)
    for b in range(B):
        prob, ro = _oracle(cfg, cc[b], ip[b], ped[b], max_outer_iter=20, tol=1e-4)
        assert int(r["outer_iterations"][b]) == ro["outer_iterations"]
        assert abs(int(r["inner_iterations"][b]) - sum(ro["inner_iterations"])) <= ro["outer_iterations"]
        assert abs(int(r["iterations"][b]) - ro["inner_iterations"][-1]) <= 1
        assert bool(r["fb_converged"][b]) == (ro["final_diff"] < 1e-4)
        assert rel_l2(r["psi"][b], ro["psi"]) <= PSI_TOL
        assert rel_l2(r["j_phi"][b], prob.J_phi) <= 1e-8
        assert abs(r["final_diff"][b] - ro["final_diff"]) <= 1e-6 * max(abs(ro["final_diff"]), 1e-12) + 1e-13


def test_outer_loop_masks_are_per_equilibrium(pkg):
    """Equilibria converge in different outer iterations; one that has stopped must not be touched again, and a
    result must not depend on the rest of the batch (compacted work list, per-equilibrium masks)."""
    cfg = golden_cfg(golden("solves"), "iter65")
    cc, ip, _ = _uq(cfg, 6)
    bk = pkg.BatchedFusionKernel(cfg)
    # a tight outer cap for everybody, then the full run: samples that stopped early are identical in both
    full = bk.solve_free_boundary(cc, ip, max_outer_iter=20, tol=1e-4)
    one = bk.solve_free_boundary(cc[2:3], ip[2:3], max_outer_iter=20, tol=1e-4)
    np.testing.assert_array_equal(full["psi"][2], one["psi"][0])
    assert int(full["outer_iterations"][2]) == int(one["outer_iterations"][0])
    # a tolerance inside the spread of the second-iteration diffs (4.6e-4 .. 7.9e-4): some samples stop after two
    # outer iterations while the others go on to a third
    loose = bk.solve_free_boundary(cc, ip, max_outer_iter=20, tol=6.3e-4)
    for b in range(6):
        _, ro = _oracle(cfg, cc[b], ip[b], None, max_outer_iter=20, tol=6.3e-4)
        assert int(loose["outer_iterations"][b]) == ro["outer_iterations"]
        assert rel_l2(loose["psi"][b], ro["psi"]) <= PSI_TOL
    assert set(loose["outer_iterations"].tolist()) == {2, 3}
    capped = bk.solve_free_boundary(cc, ip, max_outer_iter=1, tol=1e-4)
    assert (capped["outer_iterations"] == 1).all() and not capped["fb_converged"].any()


@pytest.mark.parametrize("n,wall_mu0", [(33, G.MU0_SI), (65, G.MU0_SI), (33, 2.0e-3)])
def test_plasma_wall_option_vs_numpy_restatement(pkg, n, wall_mu0):
    """plasma_wall=True: wall = coil flux + M @ (J dA) through gsb_wall_matrix + the DMMA GEMM (gsb_wall_flux) inside the
    device loop.  Parity unpinned (see module docstring): compared with the oracle's NumPy restatement.  The third case
    scales the wall coupling up (mu0 2e-3) so that the plasma term visibly moves the solution."""
    cfg = golden_cfg(golden("solves"), "iter65")
    cfg["grid_resolution"] = [n, n]
    cfg["physics"]["profiles"] = {"mode": "h-mode"}
    B = 130 if n == 33 else 3  # k_wall_gemm_sk tiles the batch by 128: two tiles (the second ragged) or one ragged tile
    cc, ip, ped = _uq(cfg, B)
    bk = pkg.BatchedFusionKernel(cfg)
    r = bk.solve_free_boundary(cc, ip, ped, ped, max_outer_iter=4, tol=1e-6, plasma_wall=True, wall_mu0=wall_mu0)
    lane_a = bk.solve_free_boundary(cc[:3], ip[:3], ped[:3], ped[:3], max_outer_iter=4, tol=1e-6)
    for b in (0, 1, 2) if n == 65 else (0, 64, 129):
        prob, ro = _oracle(cfg, cc[b], ip[b], ped[b], max_outer_iter=4, tol=1e-6, plasma_wall_mu0=wall_mu0)
        assert int(r["outer_iterations"][b]) == ro["outer_iterations"]
        assert rel_l2(r["psi"][b], ro["psi"]) <= PSI_TOL
    if wall_mu0 > 1e-4:
        assert rel_l2(r["psi"][0], lane_a["psi"][0]) > 1e-6  # the plasma term is really on the wall
