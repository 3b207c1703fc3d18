"""CPU: the C-ABI library loads, exports every symbol include/wr_gpu.h declares, parses STL on the
host, and fails loudly (no CPU fallback) when there is no CUDA device."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from test_oracle_golden import stl_bytes


@pytest.fixture(scope="module")
def L():
    from welding_robot_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    return _lib.lib()


def declared_symbols():
    hdr = open(os.path.join(ROOT, "include", "wr_gpu.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(wr_[a-z0-9_]+)\s*\(", hdr)))


def test_every_declared_symbol_is_exported(L):
    from welding_robot_b200 import _lib
    syms = declared_symbols()
    assert len(syms) >= 40
    for s in syms:
        assert hasattr(L, s), "libwrgpu.so does not export %s" % s
    assert sorted(_lib.SYMBOLS) == syms   # the Python binding covers the whole header


def test_no_torch_types_in_signatures():
    hdr = open(os.path.join(ROOT, "include", "wr_gpu.h")).read()
    code = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)   # comments may mention the host plumbing
    assert "torch" not in code.lower() and "at::" not in code and "#include <cuda" not in code and "Tensor" not in code


def test_stl_parse_on_host(L, meshes):
    from welding_robot_b200 import STLReader, WrError
    r = STLReader()
    for name in ("cubic", "simplified_piece"):
        assert r.readBuffer(stl_bytes(meshes[name]))
        assert r.NumTri() == len(meshes[name])
        assert np.array_equal(r.TriangleList().view(np.uint32), meshes[name].view(np.uint32))
    with pytest.raises(WrError):
        r.readBuffer(b"solid ascii".ljust(200, b" "))        # ASCII branch unsupported (read_STL.hpp:65)
    with pytest.raises(WrError):
        r.readBuffer(stl_bytes(meshes["cubic"])[:300])          # truncated


def test_default_params_are_the_reference_literals(L):
    from welding_robot_b200 import AcsParams
    p = AcsParams()
    assert L.wr_acs_default_params(C.byref(p)) == 0
    assert (p.alpha, p.K, p.fixed_colony) == (1, 6, 0)
    assert (np.float32(p.beta), np.float32(p.rho), np.float32(p.tau0)) == (np.float32(0.6), np.float32(0.8), np.float32(1.0))


def test_fails_loudly_without_a_gpu(L):
    """In a process that sees no CUDA device (none installed, or all hidden) the hot path raises WR_ERR_CUDA."""
    code = ("import numpy as np, welding_robot_b200 as wr\n"
            "tris = np.load(%r)['cubic']\n"
            "try:\n"
            "    wr.GridMap().creatGridMap(tris, 0.005, 10)\n"
            "except wr.WrError as e:\n"
            "    print('status', e.status)\n") % os.path.join(ROOT, "tests", "golden", "meshes.npz")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True, text=True)
    assert "status -2" in r.stdout.splitlines(), r.stdout + r.stderr     # WR_ERR_CUDA: no silent CPU path


def test_product_does_not_import_the_oracle():
    pkg = os.path.join(ROOT, "welding_robot_b200")
    for d, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp", ".cpp")):
                src = open(os.path.join(d, f), errors="replace").read()
                for line in src.splitlines():
                    if re.search(r"(import|include|from|dlopen|CDLL).*oracle", line):
                        raise AssertionError("product file %s references oracle/: %s" % (os.path.join(d, f), line))


def test_unknown_search_parameter_raises(L):
    import welding_robot_b200 as wr
    with pytest.raises(TypeError):
        wr.ACS_Rank(step_caps=600)         # a typo must not silently run with defaults
    a = wr.ACS_Rank(step_cap=600, max_iteration=7, alpha=2)
    assert (a.params.step_cap, a.max_iteration, a.params.alpha) == (600, 7, 2)
