"""The C-ABI library: loads on a CPU box, exports every symbol include/priblast_acc.h declares, refuses
to run without CUDA (no fallback), and its host-only record writer reproduces the reference bytes."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import GOLDEN, ROOT


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "priblast_acc.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(prib_[a-z_0-9]+)\s*\(", src)))


def test_header_symbols_are_exported():
    from priblast_b200 import _capi
    lib = _capi.load()
    names = _declared_symbols()
    assert len(names) >= 14
    for n in names:
        assert hasattr(lib, n), f"{n} declared in priblast_acc.h but not exported"
    assert sorted(_capi.SIGNATURES) == names, "ctypes binding and header out of sync"


def test_invalid_arguments_are_status_codes_not_exit():
    from priblast_b200 import _capi
    lib = _capi.load()
    ctx = ctypes.c_void_p()
    prm = _capi.AccParams(70, 1, 0, 0, 0)  # delta <= 1: reference exits (raccess.hpp:47-50)
    rc = lib.prib_acc_create(ctypes.byref(ctx), ctypes.byref(prm))
    assert rc == -1 and b"-d option must be greater than 1" in lib.prib_last_error()
    prm = _capi.AccParams(100000, 5, 0, 0, 0)
    assert lib.prib_acc_create(ctypes.byref(ctx), ctypes.byref(prm)) == -1


def test_no_cpu_fallback_without_gpu():
    """In a process that sees no CUDA device (any GPU of the machine hidden), creating a context fails."""
    code = ("import sys\n"
            "sys.path.insert(0, sys.argv[1])\n"
            "from priblast_b200 import Raccess, _capi\n"
            "try:\n"
            "    Raccess(70, 5)\n"
            "except _capi.PribError as e:\n"
            "    sys.exit(0 if e.code == -2 else 3)\n"  # -2: PRIB_ECUDA
            "sys.exit(4)\n")
    p = subprocess.run([sys.executable, "-c", code, ROOT], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True)
    assert p.returncode == 0, p.stderr


def test_mirror_argument_errors():
    from priblast_b200 import Raccess
    with pytest.raises(ValueError):
        Raccess(70, 1)
    with pytest.raises(ValueError):
        Raccess("", 70, 5, "")


def test_record_writer_matches_reference_layout():
    from priblast_b200 import _capi
    lib = _capi.load()
    case = next(c for c in GOLDEN if c["name"] == "rand_L100_W70_d5")
    L, delta = 100, 5
    n = lib.prib_acc_record_bytes(L, delta)
    assert n == 8 + 4 * (2 * L - delta + 1)
    buf = ctypes.create_string_buffer(int(n))
    acc = np.ascontiguousarray(case["acc"])
    cond = np.ascontiguousarray(case["cond"])
    f32p = ctypes.POINTER(ctypes.c_float)
    assert lib.prib_acc_write_record(acc.ctypes.data_as(f32p), cond.ctypes.data_as(f32p), L, delta, buf) == n
    want = (np.int32(L - delta + 1).tobytes() + acc[:L - delta + 1].tobytes() + np.int32(L).tobytes()
            + cond.tobytes())
    assert buf.raw == want
    assert lib.prib_acc_record_bytes(3, 5) < 0  # L < delta: reference writes a negative count; rejected here
