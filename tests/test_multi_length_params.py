"""Several minimum accessible lengths from one context, on the CPU: argument checks of prib_acc_create_lengths, of
Raccess with a list of lengths and of `db -d 5,8,...`, all before any CUDA call."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

FRONT = os.path.join(ROOT, "priblast_b200", "pRIblast_b200")


def _create(lengths, n=None, W=70, null_lengths=False):
    from priblast_b200 import _capi
    lib = _capi.load()
    ctx = ctypes.c_void_p()
    prm = _capi.AccParams(W, 0, 0, 0, 0)  # min_accessible_length is not read
    arr = np.asarray(lengths if len(lengths) else [0], dtype=np.int32)
    ptr = ctypes.cast(None, _capi.c_i32p) if null_lengths else arr.ctypes.data_as(_capi.c_i32p)
    rc = lib.prib_acc_create_lengths(ctypes.byref(ctx), ctypes.byref(prm), len(lengths) if n is None else n, ptr)
    return rc, lib.prib_last_error()


@pytest.mark.parametrize("lengths,n,msg", [
    ([5, 5], None, b"lengths[1] = 5: minimum accessible lengths must be strictly increasing"),
    ([5, 8, 7], None, b"lengths[2] = 7: minimum accessible lengths must be strictly increasing"),
    ([5, 1], None, b"lengths[1] = 1: Error: -d option must be greater than 1"),
    ([1, 5], None, b"lengths[0] = 1: Error: -d option must be greater than 1"),
    ([5, 1001], None, b"lengths[1] = 1001: minimum accessible length must be in 2..1000"),
    ([1], None, b"Error: -d option must be greater than 1"),
    ([1001], None, b"minimum accessible length must be in 2..1000"),
    ([], 0, b"number of minimum accessible lengths must be in 1..32"),
    (list(range(2, 35)), None, b"number of minimum accessible lengths must be in 1..32"),
])
def test_bad_length_lists_are_argument_errors(lengths, n, msg):
    rc, err = _create(lengths, n)
    assert rc == -1, err
    assert err == msg


def test_null_arguments():
    from priblast_b200 import _capi
    lib = _capi.load()
    rc, err = _create([5, 8], null_lengths=True)
    assert rc == -1 and err == b"null argument"
    lengths = np.asarray([5, 8], dtype=np.int32)
    prm = _capi.AccParams(70, 0, 0, 0, 0)
    assert lib.prib_acc_create_lengths(None, ctypes.byref(prm), 2, lengths.ctypes.data_as(_capi.c_i32p)) == -1
    ctx = ctypes.c_void_p()
    assert lib.prib_acc_create_lengths(ctypes.byref(ctx), None, 2, lengths.ctypes.data_as(_capi.c_i32p)) == -1


def test_span_is_still_checked():
    rc, err = _create([5, 8], W=1001)
    assert rc == -1 and err == b"maximal span must be in 1..1000"


def test_valid_list_reaches_the_device_check():
    """A valid list passes every argument check; without a visible device the call fails with PRIB_ECUDA."""
    code = ("import sys, ctypes\n"
            "import numpy as np\n"
            "sys.path.insert(0, sys.argv[1])\n"
            "from priblast_b200 import _capi, Raccess\n"
            "lib = _capi.load()\n"
            "ctx = ctypes.c_void_p()\n"
            "prm = _capi.AccParams(70, 0, 0, 0, 0)\n"
            "for L in ([2, 5, 8, 31], [5], list(range(2, 34)), [40, 1000]):\n"
            "    a = np.asarray(L, dtype=np.int32)\n"
            "    rc = lib.prib_acc_create_lengths(ctypes.byref(ctx), ctypes.byref(prm), len(a), a.ctypes.data_as(_capi.c_i32p))\n"
            "    if rc != -2: sys.exit(3)\n"
            "try:\n"
            "    Raccess(70, [5, 8])\n"
            "except _capi.PribError as e:\n"
            "    sys.exit(0 if e.code == -2 else 4)\n"
            "sys.exit(5)\n")
    p = subprocess.run([sys.executable, "-c", code, ROOT], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True)
    assert p.returncode == 0, p.stderr


def test_raccess_list_argument_errors():
    from priblast_b200 import Raccess, _capi
    with pytest.raises(ValueError):
        Raccess(70, [5, 1])
    with pytest.raises(_capi.PribError) as e:
        Raccess(70, [8, 5])
    assert e.value.code == -1 and "strictly increasing" in str(e.value)


def _fasta(path, lens=(40, 120, 75)):
    rng = np.random.default_rng(1)
    with open(path, "w") as f:
        for k, L in enumerate(lens):
            f.write(f">s{k}\n" + "".join("ACGU"[i] for i in rng.integers(0, 4, L)) + "\n")


def _run_front(*args, env_extra=None):
    subprocess.run(["make", "-C", os.path.join(ROOT, "priblast_b200", "csrc", "host")], check=True,
                   stdout=subprocess.DEVNULL)
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", **(env_extra or {}))
    return subprocess.run([FRONT, "db", *args], env=env, capture_output=True, text=True)


@pytest.mark.parametrize("d,msg", [
    ("5,5", "Error: the -d values must be strictly increasing"),
    ("8,5", "Error: the -d values must be strictly increasing"),
    ("5,x", "Error: -d must be an integer or a comma-separated list of integers, not '5,x'"),
    ("5,", "Error: -d must be an integer or a comma-separated list of integers, not '5,'"),
    ("1,5", "Error: -d option must be greater than 1"),
    (",".join(str(d) for d in range(2, 35)), "Error: -d takes at most 32 values"),
    ("5,100", "Error: sequence s0 is shorter than the minimum accessible length (-d)"),
])
def test_front_end_rejects_bad_lists_before_cuda(tmp_path, d, msg):
    fa = str(tmp_path / "in.fa")
    _fasta(fa)
    p = _run_front("-i", fa, "-o", str(tmp_path / "x"), "-d", d)
    assert p.returncode == 1 and p.stderr.startswith(msg), p.stderr
    assert not any(n.startswith("x") for n in os.listdir(tmp_path))


def test_front_end_list_writes_one_database_per_length(tmp_path):
    """Without the .acc step (test switch), `-d 5,9` writes <o>_d5 and <o>_d9 with the .seq/.ind/.nam/.bas of the
    single-length runs."""
    fa = str(tmp_path / "in.fa")
    _fasta(fa)
    env = {"PRIB_DB_FORMATS_ONLY": "1"}
    for args in (["-o", str(tmp_path / "m"), "-d", "5,9"], ["-o", str(tmp_path / "s5"), "-d", "5"],
                 ["-o", str(tmp_path / "s9"), "-d", "9"]):
        p = _run_front("-i", fa, "-w", "30", "-c", "2", *args, env_extra=env)
        assert p.returncode == 0, p.stderr
    for d in (5, 9):
        for ext in (".seq", ".ind", ".nam", ".bas"):
            a = open(str(tmp_path / f"m_d{d}") + ext, "rb").read()
            b = open(str(tmp_path / f"s{d}") + ext, "rb").read()
            assert a == b, (d, ext)
    assert not os.path.exists(str(tmp_path / "m.bas"))
