"""CPU: the C-ABI library builds, loads and exports every symbol include/sdb200.h declares; the
product fails loudly (no fallback) when handed CPU tensors or when the library is missing."""
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "sdb200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(sdb_[a-z0-9_]+)\s*\(", src)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from sdb200 import _lib
    return _lib.load()


def test_header_symbols_exported(lib):
    from sdb200 import _lib
    names = _declared()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), "symbol %s declared in sdb200.h is not exported" % n
        assert n in _lib.SIGNATURES, "symbol %s has no ctypes signature" % n
    assert set(_lib.SIGNATURES) == set(names)


def test_version_and_error_string(lib):
    assert lib.sdb_version() >= 100
    assert isinstance(lib.sdb_last_error_string(), bytes)


def test_no_cpu_fallback(lib):
    from sdb200 import _lib, ops
    x = torch.zeros(1, 2, 2, 32)
    with pytest.raises(_lib.SdbError):
        ops.groupnorm(x, torch.ones(32), torch.zeros(32), 1e-5)
    with pytest.raises(_lib.SdbError):
        ops.ddim_step(torch.zeros(4), torch.zeros(4), 0.5, 0.6, 0.3, 0.0, 0.7)


def test_missing_library_is_loud(tmp_path):
    from sdb200 import _lib
    with pytest.raises(_lib.SdbError):
        _lib.load(str(tmp_path / "nope.so"))


def test_argument_validation_without_gpu(lib):
    """Bad arguments are rejected on the host before any launch (safe without a GPU)."""
    import ctypes as C
    assert lib.sdb_groupnorm_ws_bytes(1, 16, 30, 32) == -1          # C % 4 != 0
    assert lib.sdb_groupnorm_ws_bytes(2, 4096, 320, 32) > 0
    rc = lib.sdb_layernorm(None, 4, 320, 1e-5, None, None, None, 0, None)
    assert rc == -1 and b"null" in lib.sdb_last_error_string()
    rc = lib.sdb_ddim_step(None, None, None, 1.0, None, 0.5, 0.6, 0.3, 0.0, 0.7, 1.0, None, None, 0, None)
    assert rc == -1


# fake device addresses, 4 KB apart: never dereferenced, the checks reject the call first
X, E, U, NZ, XP, P0 = (0x100000 + 0x1000 * k for k in range(6))
N = 16


def _ddim_step(lib, x=X, e=E, u=U, noise=NZ, xp=XP, p0=P0):
    return lib.sdb_ddim_step(x, e, u, 7.5, noise, 0.9, 0.95, 0.3, 0.5, 0.4, 1.0, xp, p0, N, None)


def _ddim_xprev(lib, p0=P0, e=E, u=U, noise=NZ, xp=XP):
    return lib.sdb_ddim_xprev(p0, e, u, 7.5, noise, 0.95, 0.3, 0.5, 1.0, xp, N, None)


@pytest.mark.parametrize("entry, call, case", [
    *[("ddim_step", _ddim_step, c) for c in (
        dict(xp=X), dict(p0=E), dict(xp=U), dict(p0=NZ),                              # output == input
        dict(xp=X + 4 * (N - 1)), dict(p0=NZ - 4 * (N - 1)),                          # output overlaps an input
        dict(p0=XP), dict(p0=XP + 8))],                                               # the two outputs overlap
    *[("ddim_xprev", _ddim_xprev, c) for c in (
        dict(xp=P0), dict(xp=E), dict(xp=U), dict(xp=NZ),                             # output == input
        dict(xp=P0 + 4 * (N - 1)), dict(xp=E - 4 * (N - 1)))],                        # output overlaps an input
])
def test_ddim_outputs_must_not_overlap(lib, entry, call, case):
    assert call(lib, **case) == -1, case
    err = lib.sdb_last_error_string()
    assert err.startswith(entry.encode() + b": ") and b"overlap" in err, (case, err)   # rejected by the check, not by a launch
