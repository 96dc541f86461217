"""Spans above 200 and minimum accessible lengths above 30 on the CPU: the wide-span engine's formulation (the cell
functions of acc_core.h with tables of 1,000 spans and the engine's span scaling, run by tests/hostemu/hostemu_wide.cpp)
against the plain-C oracle, and the argument limits of prib_acc_create."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ATOL_VS_REF, ROOT, RTOL_VS_REF, assert_close_kcal

_f32p = ctypes.POINTER(ctypes.c_float)
_i32p = ctypes.POINTER(ctypes.c_int32)
_i64p = ctypes.POINTER(ctypes.c_int64)


@pytest.fixture(scope="session")
def wide_emu(tmp_path_factory):
    d = tmp_path_factory.mktemp("hostemu_wide")
    cs = os.path.join(ROOT, "priblast_b200", "csrc")
    blob = os.path.join(ROOT, "priblast_b200", "data", "turner99.bin")
    subprocess.run(["gcc", "-O2", "-fPIC", "-c", os.path.join(cs, "turner_blob.c"), f'-DPRIB_TURNER_BIN="{blob}"',
                    "-o", str(d / "turner_blob.o")], check=True)
    lib = str(d / "libhostemu_wide.so")
    subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", "-Wno-unknown-pragmas",
                    os.path.join(ROOT, "tests", "hostemu", "hostemu_wide.cpp"), os.path.join(cs, "acc_tables.cpp"),
                    str(d / "turner_blob.o"), "-o", lib], check=True)
    return ctypes.CDLL(lib)


def _emu_batch(lib, seqs, W, delta):
    from oracle_py import acc_layout
    bs = [s.encode() for s in seqs]
    lens = np.array([len(b) for b in bs], np.int32)
    ao, co, tot = acc_layout(lens)
    out = np.zeros(max(tot, 1), np.float32)
    arr = (ctypes.c_char_p * len(bs))(*bs)
    assert lib.hostemu_wide_run_batch(len(bs), arr, lens.ctypes.data_as(_i32p), W, delta, out.ctypes.data_as(_f32p),
                                      ao.ctypes.data_as(_i64p), co.ctypes.data_as(_i64p)) == 1
    return [(out[a:a + l], out[c:c + l]) for a, c, l in zip(ao, co, lens)]


def _sequences():
    """300-900 nt, uniform bases, one of them in lower case with runs of N."""
    rng = np.random.default_rng(250)
    seqs = ["".join("ACGU"[k] for k in rng.integers(0, 4, L)) for L in (300, 560, 900)]
    mixed = list(seqs[1].lower())
    for p in (40, 41, 42, 300, 301):
        mixed[p] = "n"
    seqs[1] = "".join(mixed)
    return seqs


@pytest.mark.parametrize("W", [250, 400])
@pytest.mark.parametrize("delta", [5, 31, 45])
def test_wide_formulation_vs_oracle(wide_emu, oracle_lib, W, delta):
    seqs = _sequences()
    got = _emu_batch(wide_emu, seqs, W, delta)
    want, _ = oracle_lib.run_batch(seqs, W, delta)
    for k, ((a, c), (oa, oc)) in enumerate(zip(got, want)):
        assert_close_kcal(a, oa, ATOL_VS_REF, RTOL_VS_REF, f"acc seq {k} W={W} delta={delta}")
        assert_close_kcal(c, oc, ATOL_VS_REF, RTOL_VS_REF, f"cond seq {k} W={W} delta={delta}")
        assert np.all(c[:delta] == 0) and np.all(a[len(a) - delta + 1:] == 0)


def test_delta_above_span_vs_oracle(wide_emu, oracle_lib):
    """delta = 40 at W = 20: the window is wider than any base pair, so only the exterior-loop term remains."""
    seqs = _sequences()[:2]
    got = _emu_batch(wide_emu, seqs, 20, 40)
    want, _ = oracle_lib.run_batch(seqs, 20, 40)
    for (a, c), (oa, oc) in zip(got, want):
        assert_close_kcal(a, oa, ATOL_VS_REF, RTOL_VS_REF, "acc")
        assert_close_kcal(c, oc, ATOL_VS_REF, RTOL_VS_REF, "cond")


def test_widest_parameters_reach_the_device_check():
    """W = 1,000 and delta = 40 are valid arguments: without a device the create call fails for want of CUDA."""
    code = ("import sys, ctypes\n"
            "sys.path.insert(0, sys.argv[1])\n"
            "from priblast_b200 import _capi\n"
            "lib = _capi.load()\n"
            "ctx = ctypes.c_void_p()\n"
            "prm = _capi.AccParams(1000, 40, 0, 0, 0)\n"
            "sys.exit(0 if lib.prib_acc_create(ctypes.byref(ctx), ctypes.byref(prm)) == -2 else 3)\n")
    p = subprocess.run([sys.executable, "-c", code, ROOT], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True)
    assert p.returncode == 0, p.stderr


@pytest.mark.parametrize("W,delta,msg", [(1001, 5, b"maximal span must be in 1..1000"),
                                         (70, 1001, b"minimum accessible length must be in 2..1000"),
                                         (0, 5, b"maximal span must be in 1..1000")])
def test_out_of_range_parameters_are_argument_errors(W, delta, msg):
    from priblast_b200 import _capi
    lib = _capi.load()
    ctx = ctypes.c_void_p()
    prm = _capi.AccParams(W, delta, 0, 0, 0)
    assert lib.prib_acc_create(ctypes.byref(ctx), ctypes.byref(prm)) == -1
    assert msg in lib.prib_last_error()
