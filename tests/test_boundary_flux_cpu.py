"""CPU checks of the batched wall-contour boundary reconstruction: the gsb_boundary_params ABI layout, and the host-side
geometry (limiter distance, containment) and X-point symmetry condition against the oracle on the reference fixture's
points (see test_gpu_boundary_reconstruction_batched)."""
from __future__ import annotations

import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

import gs_oracle as G
from conftest import ROOT, golden
from scpn_fusion_core_b200 import _lib
from scpn_fusion_core_b200.free_boundary import _limiter_geometry, _wall_contour, _x_pair_symmetric

LIMITER = np.array([[3.9, -4.6], [8.6, -4.6], [8.6, 4.6], [3.9, 4.6]])


def test_boundary_params_layout_matches_the_c_header(tmp_path):
    if shutil.which("gcc") is None:
        pytest.skip("no C compiler")
    cls = _lib.gsb_boundary_params
    lines = ['printf("size %zu\\n", sizeof(gsb_boundary_params));']
    lines += [f'printf("{f} %zu\\n", offsetof(gsb_boundary_params, {f}));' for f, _ in cls._fields_]
    src = tmp_path / "boundary.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "gsb200.h"\nint main(void) {\n' + "\n".join(lines)
                   + "\nreturn 0;\n}\n")
    exe = tmp_path / "boundary"
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = dict((k, int(v)) for k, v in (ln.split() for ln in subprocess.check_output([str(exe)], text=True).splitlines()))
    assert got["size"] == ctypes.sizeof(cls)
    for f, _ in cls._fields_:
        assert got[f] == getattr(cls, f).offset, f


def _fixture_kernel_axes(z):
    import json
    cfg = json.loads(str(z["cfg"]))
    d, (nr, nz) = cfg["dimensions"], cfg["grid_resolution"]

    class Axes:
        R = np.linspace(d["R_min"], d["R_max"], nr)
        Z = np.linspace(d["Z_min"], d["Z_max"], nz)
    return Axes, cfg


def test_limiter_geometry_on_the_fixture_contour():
    """The fixture's wall contour (33^2) and limiter: the host values equal the oracle's and the fixture's exactly."""
    z = golden("free_boundary_shape")
    axes, cfg = _fixture_kernel_axes(z)
    pts = _wall_contour(axes)[0]
    np.testing.assert_array_equal(pts, z["br_points"])
    np.testing.assert_array_equal(pts, G.wall_contour(axes.R, axes.Z)[0])
    geo = _limiter_geometry(pts, LIMITER)
    pos = [(c["r"], c["z"]) for c in cfg["coils"]]
    ro = G.reconstruct_boundary_flux(pos, [1] * len(pos), z["currents"], pts, limiter_points=LIMITER)
    for key in ("limiter_point_count", "min_limiter_distance_m", "boundary_containment_fraction",
                "boundary_containment_pass"):
        assert geo[key] == ro[key], key
    bs = z["br_scalars"]
    assert (geo["limiter_point_count"], geo["min_limiter_distance_m"], geo["boundary_containment_fraction"],
            float(geo["boundary_containment_pass"])) == (int(bs[3]), bs[4], bs[5], bs[6])
    # a limiter that holds part of the contour
    part = _limiter_geometry(pts, np.array([[1.0, -5.0], [7.0, -5.0], [7.0, 5.0], [1.0, 5.0]]))
    assert 0.0 < part["boundary_containment_fraction"] < 1.0 and not part["boundary_containment_pass"]


def test_x_pair_symmetry_condition_against_the_oracle():
    """Per sample, the condition under which the reference reports x_point_pair_symmetry_abs_error (else None)."""
    z = golden("free_boundary_shape")
    _, cfg = _fixture_kernel_axes(z)
    pos = [(c["r"], c["z"]) for c in cfg["coils"]]
    base = np.array([[5.0, -3.4], [5.0, 3.4]])
    xs = np.array([base, base + [[0.0, 0.1], [0.0, 0.1]], base + [[2e-10, 0.0], [0.0, 0.0]], base + [[1e-8, 0], [0, 0]],
                   base + [[0.0, 0.0], [0.0, 5e-10]], [[5.0, -3.0], [5.0, 3.4]]])
    ax = np.array([[6.2, 0.0], [6.2, 0.1], [6.2, 0.0], [6.2, 0.0], [6.2, 0.0], [6.2, 0.2]])
    ok = _x_pair_symmetric(xs, ax)
    for b in range(len(xs)):
        ro = G.reconstruct_boundary_flux(pos, [1] * len(pos), z["currents"], z["br_points"], axis_point=ax[b],
                                         x_points=xs[b])
        assert bool(ok[b]) == (ro["x_point_pair_symmetry_abs_error"] is not None), b
    assert ok.tolist() == [True, True, True, False, True, True]


def test_point_arrays_reach_the_entry_c_contiguous():
    """The C entry reads every point array in storage order: transposed, strided and Fortran-ordered inputs (shared and
    per-sample) are handed over C-contiguous with the caller's values.  The spec does no device work."""
    import json

    import scpn_fusion_core_b200 as pkg
    z = golden("free_boundary_shape")
    bk = pkg.BatchedFusionKernel(json.loads(str(z["cfg"])), device=0)
    xs = np.array([[5.0, 5.0], [-3.4, 3.4]]).T
    axs = np.array([[6.2, 1.0], [0.0, 2.0]])[:, 0]
    pts, lim = np.asfortranarray(z["br_points"]), np.asfortranarray(LIMITER)
    for ax, xp, want_ax, want_x in ((axs, xs, [6.2, 0.0], [[5.0, -3.4], [5.0, 3.4]]),
                                    (np.asfortranarray(np.tile([6.2, 0.0], (3, 1))), xs, np.tile([6.2, 0.0], (3, 1)),
                                     np.tile([[5.0, -3.4], [5.0, 3.4]], (3, 1, 1))),
                                    (axs, np.asfortranarray(np.tile(xs, (3, 1, 1))), np.tile([6.2, 0.0], (3, 1)),
                                     np.tile([[5.0, -3.4], [5.0, 3.4]], (3, 1, 1)))):
        sp = bk._boundary_spec(3, None, pts, lim, ax, xp)
        for key, want in (("points", z["br_points"]), ("limiter", LIMITER), ("axis", want_ax), ("xpoints", want_x)):
            assert sp[key].flags.c_contiguous and sp[key].dtype == np.float64, key
            np.testing.assert_array_equal(np.frombuffer(sp[key].tobytes(order="A")), np.ravel(want), err_msg=key)
