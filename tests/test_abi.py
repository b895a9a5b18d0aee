"""The C-ABI library loads on a CPU-only box and exports every symbol include/platymatch_b200.h declares."""
import ctypes
import os
import re
import shutil
import subprocess

import pytest

from conftest import ROOT


def _declared():
    text = open(os.path.join(ROOT, "include", "platymatch_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(pm_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_exported_and_bound():
    from platymatch_b200 import _lib
    lib = _lib.load()
    names = _declared()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), "missing export " + n
        assert n in _lib.SIGNATURES, "no ctypes signature for " + n
    assert set(_lib.SIGNATURES) == set(names)
    # and the library exports nothing else: a definition left behind by a removed declaration shows up here
    nm = shutil.which("nm")
    if nm:
        out = subprocess.run([nm, "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
        exported = {f[-1] for f in (line.split() for line in out.splitlines()) if f and f[-1].startswith("pm_")}
        assert exported == set(names), (sorted(exported - set(names)), sorted(set(names) - exported))


def test_ctypes_signatures_match_header_arity():
    """Every ctypes signature has as many arguments as the header's prototype (ABI drift shows up here, on the CPU)."""
    from platymatch_b200 import _lib
    text = open(os.path.join(ROOT, "include", "platymatch_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    protos = dict(re.findall(r"\b(pm_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", text, flags=re.S))
    assert set(protos) == set(_lib.SIGNATURES)
    for name, params in protos.items():
        params = " ".join(params.split())
        n = 0 if params in ("", "void") else params.count(",") + 1
        assert n == len(_lib.SIGNATURES[name][1]), (name, n, len(_lib.SIGNATURES[name][1]))


def test_version_and_workspace_sizes_without_gpu():
    from platymatch_b200 import _lib
    lib = _lib.load()
    assert lib.pm_version() == 200
    assert lib.pm_mean_distance_workspace_bytes(8000) == 32 * 32 * 8
    assert lib.pm_lap_workspace_bytes(4, 7200, 8000) > 4 * (7200 + 8000) * 8
    assert lib.pm_ransac_workspace_bytes(8000) >= 8000 * 13 * 8
    assert lib.pm_icp_workspace_bytes2(7200, 8000) >= 7200 * 24 + 8000 * 24
    assert isinstance(lib.pm_last_error_string(), bytes)


def test_argument_validation_is_host_side():
    """Bad arguments are rejected before any CUDA call (works without a device)."""
    from platymatch_b200 import _lib
    lib = _lib.load()
    assert lib.pm_cloud_stats(None, 10, None, None) == -1
    assert b"null pointer" in lib.pm_last_error_string()
    assert lib.pm_lap_solve(None, 1, 4, 4, 4, 0, 0, None, None, None, None, 0, None) == -1
    # more than 24 x 1024 columns: refused before any CUDA call (the pointers, 16-byte aligned and never read, stand
    # in for device buffers)
    p = ctypes.c_void_p(1 << 12)
    for nr in (1, 24577):
        assert lib.pm_lap_solve(p, 1, nr, 24577, 24580, 2048, 0, p, p, None, p, 1 << 40, None) == -5
        assert b"nc = 24577 > 24576 columns not supported" in lib.pm_last_error_string()
    with pytest.raises(ValueError):
        _lib.check(-1, "x")


def test_lap_path_bits_match_header():
    """The Python names of the assignment's path bits are the header's PM_LAP_PATH_* values."""
    from platymatch_b200 import _lib
    text = open(os.path.join(ROOT, "include", "platymatch_b200.h")).read()
    declared = {k: int(v) for k, v in re.findall(r"#define PM_LAP_PATH_([A-Z0-9_]+) (\d+)", text)}
    assert declared == _lib.LAP_PATH
    assert re.search(r"#define PM_LAP_STAT_PATH 13\b", text)
    assert sorted(declared.values()) == [1 << k for k in range(len(declared))]


def test_no_cpu_fallback_without_device():
    """Without a CUDA device the product API raises instead of computing on the host."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import numpy as np
    from platymatch_b200 import PlatyMatchError
    from platymatch_b200.utils.utils import get_mean_distance
    from platymatch_b200.lap import linear_sum_assignment
    with pytest.raises(PlatyMatchError):
        get_mean_distance(np.random.rand(3, 10), transposed=False)
    with pytest.raises(PlatyMatchError):
        linear_sum_assignment(np.random.rand(4, 5))


def test_product_never_imports_oracle():
    """The shipped package never imports, links or executes the CPU oracle, nor scipy / sklearn (comments that
    cite the reference's third-party calls are fine)."""
    import re
    bad = re.compile(r"^\s*(import|from)\s+(oracle|scipy|sklearn)\b", re.M)
    for dirpath, _, files in os.walk(os.path.join(ROOT, "platymatch_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "pm_oracle" not in src and "libpm_oracle" not in src, os.path.join(dirpath, f)
                if f.endswith(".py"):
                    assert not bad.search(src), os.path.join(dirpath, f)

