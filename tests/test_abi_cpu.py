"""CPU-only checks of the C ABI and the host logic (no compute calls without a GPU)."""
from __future__ import annotations

import ctypes
import hashlib
import os
import re

import numpy as np
import pytest

import gs_oracle as G
from conftest import ROOT
from scpn_fusion_core_b200 import _lib


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "gsb200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    names = re.findall(r"\b([a-z_][a-z0-9_]*)\s*\(", text)
    return sorted({n for n in names if n.startswith("gsb_") or n in (
        "create_solver", "set_boundary_dirichlet", "run_step", "run_step_converged", "destroy_solver",
        "delete_solver")})


def test_library_loads_and_exports_every_declared_symbol():
    lib = _lib.load()
    declared = _declared_symbols()
    assert len(declared) >= 30
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/gsb200.h but not exported"
    assert set(declared) == set(_lib.SIGNATURES), "ctypes signature table out of sync with the header"
    assert lib.gsb_abi_version() == 1


def test_reference_abi_symbols_match_hpc_bridge_contract():
    """The six names hpc_bridge.py:190-250 binds (destroy_solver or delete_solver accepted)."""
    lib = _lib.load()
    for name in ("create_solver", "run_step", "destroy_solver", "delete_solver", "set_boundary_dirichlet",
                 "run_step_converged"):
        assert hasattr(lib, name)
    # invalid geometry -> NULL, like solver.cpp:209-210
    assert lib.create_solver(1, 10, 1.0, 2.0, 0.0, 1.0) is None
    assert lib.create_solver(10, 10, 2.0, 1.0, 0.0, 1.0) is None
    # NULL handle / bad input are silent no-ops or 0 (solver.cpp:249-257,282-296)
    lib.set_boundary_dirichlet(None, 1.0)
    lib.run_step(None, None, None, 0, 1)
    d = ctypes.c_double(5.0)
    assert lib.run_step_converged(None, None, None, 0, 1, 1.5, 1e-6, ctypes.byref(d)) == 0
    assert d.value == 0.0
    lib.destroy_solver(None)


def test_sha256_sidecar_matches_the_library():
    """hpc_bridge.py loads a native solver only when <lib>.sha256 holds the file's digest (the Makefile writes it)."""
    with open(_lib.LIB_PATH, "rb") as f:
        digest = hashlib.sha256(f.read()).hexdigest()
    with open(_lib.LIB_PATH + ".sha256") as f:
        assert f.read().strip() == digest


@pytest.mark.parametrize("shape,expect", [
    ((129, 129), [129, 65, 33, 17, 9, 5]), ((128, 128), [128, 64, 32, 16, 8, 4]),
    ((257, 257), [257, 129, 65, 33, 17, 9, 5]), ((5, 5), [5]), ((4, 9), [4])])
def test_plan_levels(shape, expect):
    lib = _lib.load()
    nz = (ctypes.c_int * 32)()
    nr = (ctypes.c_int * 32)()
    n = lib.gsb_plan_levels(shape[0], shape[1], 5, nz, nr, 32)
    assert list(nz)[:n] == expect


def test_level_tables_bit_exact_vs_oracle():
    """Per-level R rows and a_e/a_w columns equal the oracle's restricted meshgrid coefficients."""
    lib = _lib.load()
    dp = ctypes.POINTER(ctypes.c_double)
    for nz, nr, rmin, rmax in [(129, 129, 2.0, 10.0), (128, 128, 2.0, 10.0), (48, 80, 0.8, 2.6), (33, 41, 1.2, 2.2)]:
        R = np.linspace(rmin, rmax, nr)
        Z = np.linspace(-4, 4, nz)
        dr, dz = float(R[1] - R[0]), float(Z[1] - Z[0])
        rg, _ = np.meshgrid(R, Z)
        lev = 0
        while True:
            r, ae, aw, sc = np.zeros(nr), np.zeros(nr), np.zeros(nr), np.zeros(4)
            n = lib.gsb_plan_level_tables(nz, nr, R.ctypes.data_as(dp), dr, dz, 5, lev, r.ctypes.data_as(dp),
                                          ae.ctypes.data_as(dp), aw.ctypes.data_as(dp), sc.ctypes.data_as(dp))
            assert n == rg.shape[1]
            a_e, a_w, a_ns, a_c = G._stencil_coeffs(rg, dr * 2.0 ** lev, dz * 2.0 ** lev)
            np.testing.assert_array_equal(r[1:n - 1], rg[1, 1:-1])
            np.testing.assert_array_equal(ae[1:n - 1], a_e[0])
            np.testing.assert_array_equal(aw[1:n - 1], a_w[0])
            assert (sc[2], sc[3]) == (a_ns, a_c)
            if 5 >= rg.shape[0] or 5 >= rg.shape[1]:
                break
            rg = G.restrict_full_weight(rg)
            lev += 1


def test_no_gpu_means_loud_failure(has_cuda):
    """Without a CUDA device the product path must fail loudly (no CPU fallback)."""
    if has_cuda:
        pytest.skip("a GPU is present")
    lib = _lib.load()
    assert lib.gsb_device_count() == 0
    assert lib.create_solver(16, 16, 1.0, 2.0, -1.0, 1.0) is None
    h = ctypes.c_void_p()
    r = np.linspace(1, 2, 16)
    rc = lib.gsb_create(ctypes.byref(h), 16, 16, r.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), None, 0.1, 0.1, 1, 0)
    assert rc == _lib.GSB_ENODEV
    assert "no usable CUDA device" in _lib.last_error()
    import scpn_fusion_core_b200 as pkg
    with pytest.raises(_lib.GsbError):
        pkg.mg_smooth(np.zeros((9, 9)), np.zeros((9, 9)), np.ones((9, 9)), 0.1, 0.1, 1.0, 1)
    with pytest.raises(_lib.GsbError):
        pkg.FusionKernel({"dimensions": {"R_min": 1, "R_max": 2, "Z_min": -1, "Z_max": 1}})


def test_product_does_not_import_the_oracle():
    """Nothing under scpn_fusion_core_b200/ may reference oracle/ (SURVEY 8c rule)."""
    pkg = os.path.join(ROOT, "scpn_fusion_core_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f), encoding="utf-8").read()
                assert "gs_oracle" not in text and "oracle/" not in text, f


def test_config_validation_matches_reference_schema():
    from scpn_fusion_core_b200 import validate_config

    base = {"dimensions": {"R_min": 2.0, "R_max": 10.0, "Z_min": -4.0, "Z_max": 4.0}}
    cfg = validate_config(base)
    assert cfg["grid_resolution"] == [129, 129]
    assert cfg["solver"] == {"max_iterations": 1000, "convergence_threshold": 1e-4, "relaxation_factor": 0.1}
    assert cfg["physics"]["vacuum_permeability"] == 1.25663706e-6
    for bad in (
        {"dimensions": {"R_min": 2.0, "R_max": 1.0, "Z_min": -4.0, "Z_max": 4.0}},
        {"dimensions": {"R_min": -1.0, "R_max": 1.0, "Z_min": -4.0, "Z_max": 4.0}},
        {**base, "grid_resolution": [3, 129]},
        {**base, "solver": {"relaxation_factor": 1.5}},
        {**base, "solver": {"max_iterations": 0}},
        {**base, "coils": [{"r": -1.0, "z": 0.0}]},
        {},
    ):
        with pytest.raises(ValueError):
            validate_config(bad)


def _header_prototypes():
    """name -> (return type, [parameter type strings]) parsed from include/gsb200.h."""
    text = open(os.path.join(ROOT, "include", "gsb200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    text = re.sub(r"typedef struct[^{;]*\{.*?\}\s*\w+\s*;", "", text, flags=re.S)
    protos = {}
    for ret, name, args in re.findall(r"\b((?:const\s+)?(?:unsigned\s+)?[a-z_][a-z0-9_ ]*?\s*\**)\s*\b([a-z_][a-z0-9_]*)\s*\(([^()]*)\)\s*;",
                                      text, flags=re.S):
        params = [a.strip() for a in args.replace("\n", " ").split(",")] if args.strip() not in ("", "void") else []
        protos[name] = (" ".join(ret.split()), [" ".join(p.split()) for p in params])
    return protos


def _c_kind(decl: str) -> str:
    """'ptr', 'double', 'int' or 'longlong' for a C parameter / return declaration."""
    if "*" in decl:
        return "ptr"
    words = [w for w in re.split(r"\W+", decl) if w and w != "const"]
    if "double" in words:
        return "double"
    if words[:2] == ["long", "long"]:
        return "longlong"
    if "void" in words:
        return "void"
    return "int"


def _ctypes_kind(t) -> str:
    if t is None:
        return "void"
    if t in (ctypes.c_void_p, ctypes.c_char_p) or hasattr(t, "_type_") and isinstance(getattr(t, "_type_", None), type):
        return "ptr"
    return {ctypes.c_double: "double", ctypes.c_int: "int", ctypes.c_longlong: "longlong"}.get(t, "ptr")


def test_ctypes_signatures_agree_with_the_header_prototypes():
    """A ctypes table that drifts from the header corrupts arguments silently: arity and the kind of every
    parameter (pointer / double / int / long long) and of the return value must match include/gsb200.h."""
    protos = _header_prototypes()
    assert set(_lib.SIGNATURES) <= set(protos), sorted(set(_lib.SIGNATURES) - set(protos))
    for name, (restype, argtypes) in _lib.SIGNATURES.items():
        ret, params = protos[name]
        assert len(argtypes) == len(params), f"{name}: {len(argtypes)} ctypes arguments vs {len(params)} in the header"
        assert _ctypes_kind(restype) == _c_kind(ret), f"{name}: return type {restype} vs '{ret}'"
        for i, (t, decl) in enumerate(zip(argtypes, params)):
            assert _ctypes_kind(t) == _c_kind(decl), f"{name} argument {i}: {t} vs '{decl}'"


def test_ctypes_struct_layouts_match_the_c_header(tmp_path):
    """sizeof / offsetof of every struct that crosses the ABI, from a C program compiled against
    include/gsb200.h with the system gcc, against the ctypes mirrors."""
    import shutil
    import subprocess
    from scpn_fusion_core_b200 import slab
    if shutil.which("gcc") is None:
        pytest.skip("no C compiler")
    mirrors = {"gsb_profile": _lib.gsb_profile, "gsb_picard_params": _lib.gsb_picard_params,
               "gsb_free_boundary_params": _lib.gsb_free_boundary_params,
               "gsb_slab_level_desc": slab._LevelDesc, "gsb_slab_halo_desc": slab._HaloDesc}
    lines = []
    for cname, cls in mirrors.items():
        lines.append(f'printf("{cname} size %zu\\n", sizeof({cname}));')
        for fname, _ in cls._fields_:
            lines.append(f'printf("{cname} {fname} %zu\\n", offsetof({cname}, {fname}));')
    src = tmp_path / "probe.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "gsb200.h"\nint main(void) {\n' + "\n".join(lines)
                   + "\nreturn 0;\n}\n")
    exe = tmp_path / "probe"
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = {}
    for ln in subprocess.check_output([str(exe)], text=True).splitlines():
        cname, key, val = ln.split()
        got[(cname, key)] = int(val)
    for cname, cls in mirrors.items():
        assert got[(cname, "size")] == ctypes.sizeof(cls), cname
        for fname, _ in cls._fields_:
            assert got[(cname, fname)] == getattr(cls, fname).offset, f"{cname}.{fname}"
