"""CPU checks of the shape-optimising free-boundary loop: the gsb_shape_params ABI layout, and the exact bounded fit the
device computes against the reference's trf fit on the reference fixture (see test_gpu_free_boundary_shape_batched)."""
from __future__ import annotations

import ctypes
import json
import os
import shutil
import subprocess

import numpy as np
import pytest

import gs_oracle as G
from conftest import ROOT, golden
from scpn_fusion_core_b200 import _lib


def test_shape_params_layout_matches_the_c_header(tmp_path):
    if shutil.which("gcc") is None:
        pytest.skip("no C compiler")
    cls = _lib.gsb_shape_params
    lines = ['printf("size %zu\\n", sizeof(gsb_shape_params));']
    lines += [f'printf("{f} %zu\\n", offsetof(gsb_shape_params, {f}));' for f, _ in cls._fields_]
    src = tmp_path / "probe.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "gsb200.h"\nint main(void) {\n' + "\n".join(lines)
                   + "\nreturn 0;\n}\n")
    exe = tmp_path / "probe"
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = dict((k, int(v)) for k, v in (ln.split() for ln in subprocess.check_output([str(exe)], text=True).splitlines()))
    assert got["size"] == ctypes.sizeof(cls)
    for f, _ in cls._fields_:
        assert got[f] == getattr(cls, f).offset, f


def test_exact_fit_on_the_fixture_problem():
    """The last fit of the reference fixture (7 coils, 8 isoflux points, alpha 1e-13, 6e6 A limits): the exact
    minimiser (lsq_linear method="bvls") is within 1e-7 relative of trf's currents (which the fixture holds bit for
    bit), and has two currents exactly on their limits where trf stops inside both (active_current_bounds 2 vs 0)."""
    from scipy.optimize import lsq_linear
    z = golden("free_boundary_shape")
    pos = [(c["r"], c["z"]) for c in json.loads(str(z["cfg"]))["coils"]]
    M = G.mutual_matrix(pos, [1] * len(pos), z["pts"])
    A = np.vstack([M.T, np.sqrt(float(z["alpha"])) * np.eye(len(pos))])
    b = np.concatenate([z["so_target"], np.zeros(len(pos))])
    lim = z["limits"]
    trf = lsq_linear(A, b, bounds=(-lim, lim), method="trf").x
    exact = lsq_linear(A, b, bounds=(-lim, lim), method="bvls").x
    np.testing.assert_array_equal(trf, z["currents"])
    np.testing.assert_allclose(exact, trf, rtol=1e-7, atol=0)
    assert np.count_nonzero(np.isclose(np.abs(exact), lim, rtol=0.0)) == 2
    assert np.count_nonzero(np.isclose(np.abs(trf), lim, rtol=0.0)) == int(z["so_scalars"][7]) == 0
