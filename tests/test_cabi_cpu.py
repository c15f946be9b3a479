"""No-GPU checks of the boundary: the shared library loads, exports every
symbol include/egnn_b200.h declares, argument errors come back as status codes
(not crashes), and the host API refuses to run without a device."""
import os
import re

import numpy as np
import pytest
import torch

import efficient_gnn_b200 as egnn
from efficient_gnn_b200 import _cabi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "egnn_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(egnn_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = _cabi.load()
    names = declared_symbols()
    assert len(names) >= 9
    for name in names:
        assert hasattr(lib, name), f"{name} declared in include/egnn_b200.h but not exported"
    assert sorted(_cabi.SYMBOLS) == names, "ctypes binding table and header disagree"
    assert lib.egnn_abi_version() == _cabi.ABI_VERSION


def test_invalid_arguments_return_status_not_crash():
    lib = _cabi.load()
    rc = lib.egnn_cheb_wavelet(None, None, None, None, None, None, 4, 4, 1, 3, 1, None, 1.0, -1.0,
                               None, None, 1, None, None, None, 0, None, 0, None, None, None, None, None, 0,
                               None, None, 0)
    assert rc == -1
    assert b"null pointer" in lib.egnn_last_error()
    with pytest.raises(_cabi.EgnnError):
        _cabi.check(rc, "egnn_cheb_wavelet")
    assert lib.egnn_cheb_workspace_bytes(1000, 1) >= 4 * 4000
    assert lib.egnn_cheb_workspace_bytes(1000, 64) >= 2 * 4 * 64000


def test_misaligned_vector_buffers_are_refused_before_any_launch():
    """At F % 4 == 0 the kernels access the caller's signal, outputs and upstream gradients with
    16-byte vector loads: a contiguous view at an odd element offset would fault the GPU.  The
    entry points refuse such pointers before the workspace check, so a NULL workspace still
    yields the alignment error and nothing runs (the pointers here are never dereferenced)."""
    lib = _cabi.load()
    base = 1 << 20
    ok = lambda i: base + 4096 * i                        # noqa: E731  16-byte aligned fakes
    bad = lambda i: base + 4096 * i + 4                   # noqa: E731  one float past a boundary
    coeffs = np.ones(8, dtype=np.float32)
    cptr = coeffs.ctypes.data
    for x0, out, t_all in ((bad(5), ok(6), None), (ok(5), bad(6), None), (ok(5), ok(6), bad(7))):
        rc = lib.egnn_cheb_wavelet(ok(1), ok(2), None, ok(3), ok(4), x0, 4, 4, 4, 3, 1, cptr, 1.0, -1.0,
                                   out, t_all, 0, None, None, None, 0, None, 0, None, None, None, None, None, 0,
                                   None, None, 0)
        assert rc == -1, rc
        assert b"aligned" in lib.egnn_last_error()
    for cbar, tbar, xbar in ((bad(5), None, ok(6)), (ok(5), bad(7), ok(6)), (ok(5), ok(7), bad(6))):
        rc = lib.egnn_cheb_adjoint(ok(1), ok(2), None, ok(3), ok(4), 4, 4, 8, 3, 1, cptr, 1.0, -1.0,
                                   cbar, tbar, xbar, None, None, None, 0, None, 0, None, None, None)
        assert rc == -1, rc
        assert b"aligned" in lib.egnn_last_error()
    # F % 4 != 0 reads per element: the same offsets pass the check and reach the workspace check
    rc = lib.egnn_cheb_adjoint(ok(1), ok(2), None, ok(3), ok(4), 4, 4, 3, 3, 1, cptr, 1.0, -1.0,
                               bad(5), bad(7), bad(6), None, None, None, 0, None, 0, None, None, None)
    assert rc == -4 and b"workspace" in lib.egnn_last_error()
    rc = lib.egnn_cheb_wavelet(ok(1), ok(2), None, ok(3), ok(4), bad(5), 4, 4, 5, 3, 1, cptr, 1.0, -1.0,
                               bad(6), None, 0, None, None, None, 0, None, 0, None, None, None, None, None, 0,
                               None, None, 0)
    assert rc == -4 and b"workspace" in lib.egnn_last_error()


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-device failure mode")
def test_no_cpu_fallback():
    with pytest.raises(egnn.EgnnError):
        egnn.graph_wavelet_features(np.eye(4, dtype=np.float32))
    with pytest.raises(egnn.EgnnError):
        egnn.compute_normalized_laplacian(torch.eye(4))
    base = torch.nn.Linear(2, 2)
    with pytest.raises(egnn.EgnnError):
        egnn.WATS(base, torch.zeros(4, 2), torch.zeros(4, dtype=torch.long), torch.eye(4),
                  torch.ones(4, dtype=torch.bool))


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "efficient-gnn_b200")
    for dirpath, _dirs, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("oracle side", ""), f"{f} mentions the oracle"


def test_heat_coefficients_match_reference_defaults():
    c = egnn.heat_coefficients(3, 0.8)
    np.testing.assert_allclose(c[0], [1.0, 0.449329, 0.201897, 0.090718], atol=1e-6)
    assert egnn.heat_coefficients(2, [0.4, 0.8]).shape == (2, 3)


def test_shared_library_is_not_older_than_its_sources():
    """A stale build (sources edited, library not rebuilt) corrupts arguments silently when a
    signature changed; catch it here, on the CPU box, before the snapshot travels."""
    import glob
    from efficient_gnn_b200 import _cabi
    src = glob.glob(os.path.join(os.path.dirname(_cabi.LIB_PATH), "..", "csrc", "*.cu*")) + \
        [os.path.join(ROOT, "include", "egnn_b200.h")]
    newest = max(os.path.getmtime(f) for f in src)
    assert os.path.getmtime(_cabi.LIB_PATH) >= newest, "rebuild: efficient-gnn_b200/csrc/build.sh"
