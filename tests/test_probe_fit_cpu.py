"""CPU checks of the batched magnetic-probe reconstruction: the gsb_probe_params ABI layout, and the exact bounded fit
the device computes against the reference's trf fit on the reference fixture's probe problem (see
test_gpu_probe_reconstruction_batched)."""
from __future__ import annotations

import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import ROOT, golden
from scpn_fusion_core_b200 import _lib


def test_probe_params_layout_matches_the_c_header(tmp_path):
    if shutil.which("gcc") is None:
        pytest.skip("no C compiler")
    cls = _lib.gsb_probe_params
    lines = ['printf("size %zu\\n", sizeof(gsb_probe_params));']
    lines += [f'printf("{f} %zu\\n", offsetof(gsb_probe_params, {f}));' for f, _ in cls._fields_]
    src = tmp_path / "probe.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "gsb200.h"\nint main(void) {\n' + "\n".join(lines)
                   + "\nreturn 0;\n}\n")
    exe = tmp_path / "probe"
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = dict((k, int(v)) for k, v in (ln.split() for ln in subprocess.check_output([str(exe)], text=True).splitlines()))
    assert got["size"] == ctypes.sizeof(cls)
    for f, _ in cls._fields_:
        assert got[f] == getattr(cls, f).offset, f


def test_exact_fit_on_the_fixture_probe_problem():
    """The fixture's probe problem (7 coils, 6 flux loops, 6 B probes, sigma, alpha 1e-6, limits, prior currents0) has
    an interior bounded optimum: the exact minimiser (lsq_linear method="bvls"), trf (which the fixture holds) and the
    unbounded least-squares solution are the same currents, and no current is on a limit."""
    from scipy.optimize import lsq_linear
    z = golden("free_boundary_shape")
    resp, w, lim = z["probe_response"], 1.0 / z["probe_sigma"], z["limits"]
    n = resp.shape[1]
    A = np.vstack([resp * w[:, None], np.sqrt(1e-6) * np.eye(n)])
    b = np.concatenate([z["probe_meas"] * w, np.sqrt(1e-6) * z["currents0"]])
    trf = lsq_linear(A, b, bounds=(-lim, lim), method="trf").x
    exact = lsq_linear(A, b, bounds=(-lim, lim), method="bvls").x
    np.testing.assert_array_equal(trf, z["probe_currents"])
    np.testing.assert_allclose(exact, trf, rtol=1e-12, atol=0)
    np.testing.assert_allclose(np.linalg.lstsq(A, b, rcond=None)[0], trf, rtol=1e-12, atol=0)
    assert np.all(np.abs(exact) < lim)
    assert int(z["probe_scalars"][4]) == 0
