"""CPU check of the restructured mathematics: the per-thread bodies of the CUDA kernels
(priblast_b200/csrc/acc_core.h), run in plain loops by tests/hostemu, against the golden fixtures.
This validates the formulation where no GPU exists; the `-m gpu` tests validate the real kernels."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import ATOL_VS_EXACT, ATOL_VS_REF, GOLDEN, ROOT, RTOL_VS_EXACT, RTOL_VS_REF, assert_close_kcal

_f32p = ctypes.POINTER(ctypes.c_float)


@pytest.fixture(scope="session")
def emu():
    d = os.path.join(ROOT, "tests", "hostemu")
    subprocess.run(["make", "-C", d], check=True, stdout=subprocess.DEVNULL)
    lib = ctypes.CDLL(os.path.join(d, "libhostemu.so"))
    lib.hostemu_run.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, _f32p, _f32p]
    def run(seq, W, delta):
        L = len(seq)
        a = np.zeros(max(L, 1), np.float32)
        c = np.zeros(max(L, 1), np.float32)
        assert lib.hostemu_run(seq.encode(), L, W, delta, a.ctypes.data_as(_f32p), c.ctypes.data_as(_f32p)) == 0
        return a[:L], c[:L]

    run.lib = lib
    return run


@pytest.mark.parametrize("case", [c for c in GOLDEN if len(c["seq"]) <= 1600], ids=lambda c: c["name"])
def test_formulation_vs_reference(emu, case):
    acc, cond = emu(case["seq"], case["W"], case["delta"])
    assert_close_kcal(acc, case["acc"], ATOL_VS_REF, RTOL_VS_REF, "acc")
    assert_close_kcal(cond, case["cond"], ATOL_VS_REF, RTOL_VS_REF, "cond")
    d = case["delta"]
    assert np.all(cond[:d] == 0) and np.all(acc[len(acc) - d + 1:] == 0)


@pytest.mark.parametrize("name", ["rand_L500_W70_d5", "rand_L300_W150_d2", "gcstem_polyA_L576",
                                  "perfect_hairpin_L150_W150", "mixed_case_N_L300"])
def test_formulation_vs_exact_math(emu, oracle_lib, name):
    """Against the exact-libm twin the fast formulation is at float-rounding level."""
    case = next(c for c in GOLDEN if c["name"] == name)
    ea, ec = oracle_lib.run_exact(case["seq"], case["W"], case["delta"])
    acc, cond = emu(case["seq"], case["W"], case["delta"])
    assert_close_kcal(acc, ea, ATOL_VS_EXACT, RTOL_VS_EXACT, "acc")
    assert_close_kcal(cond, ec, ATOL_VS_EXACT, RTOL_VS_EXACT, "cond")


@pytest.mark.parametrize("W,delta", [(130, 3), (175, 5), (200, 5), (200, 31)])
def test_fp64_tile_march_at_the_device_width_vs_exact_math(emu, oracle_lib, W, delta):
    """The FP64 engine's tile on the device (TC = 288 columns: 87 owned under a 201-column halo at W = 200) on random
    sequences against the exact-libm twin.  The gate is twice the exact-math one: the finalize step takes the
    reference's table log where the twin takes libm's, which alone moves some values by up to 1.5x ATOL_VS_EXACT at
    these spans (with libm's log there the formulation stays within 0.62x)."""
    rng = np.random.default_rng(100 * W + delta)
    seqs = ["".join("ACGU"[k] for k in rng.integers(0, 4, L)) for L in (W + 1, 500)]
    seqs.append("".join("ACGUNacgun"[k] for k in rng.integers(0, 10, 300)))
    out, _, lens = _tiled(emu.lib, seqs, W, delta, 288)
    off = 0
    for s, L in zip(seqs, lens):
        L = int(L)
        ea, ec = oracle_lib.run_exact(s, W, delta)
        assert_close_kcal(out[off:off + L], ea, 2 * ATOL_VS_EXACT, 2 * RTOL_VS_EXACT, f"L={L} acc")
        assert_close_kcal(out[off + L:off + 2 * L], ec, 2 * ATOL_VS_EXACT, 2 * RTOL_VS_EXACT, f"L={L} cond")
        off += 2 * L


def _tiled(lib, seqs, W, delta, TC, scale=(0.0, 0.0, 0.0), f32=False):
    from oracle_py import acc_layout
    i32p, i64p = ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int64)
    bs = [s.encode() if isinstance(s, str) else bytes(s) for s in seqs]
    n = len(bs)
    lens = np.array([len(b) for b in bs], np.int32)
    ao, co, tot = acc_layout(lens)
    out = np.zeros(max(tot, 1), np.float32)
    flags = np.zeros(n, np.int32)
    arr = (ctypes.c_char_p * n)(*bs)
    args = [n, arr, lens.ctypes.data_as(i32p), W, delta, out.ctypes.data_as(_f32p), ao.ctypes.data_as(i64p),
            co.ctypes.data_as(i64p)]
    if TC is None:
        assert lib.hostemu_run_batch(*args, 1) == 1
    elif f32:
        assert lib.hostemu_run_batch_tiled_f32(*args, TC, *[ctypes.c_double(x) for x in scale],
                                               flags.ctypes.data_as(i32p)) == 1
    else:
        assert lib.hostemu_run_batch_tiled(*args, TC, *[ctypes.c_double(x) for x in scale]) == 1
    return out, flags, lens


_MIX_NAMES = ["rand_L500_W70_d5", "rand_L300_W70_d2", "gcstem_polyA_L576", "mixed_case_N_L300", "tiny_L9",
              "rand_L72_W70_d5", "perfect_hairpin_L70"]
_MIX = [next(c["seq"] for c in GOLDEN if c["name"] == n) for n in _MIX_NAMES]


@pytest.mark.parametrize("W,TC", [(70, 352), (70, 104), (20, 64), (150, 352)])
def test_tile_march_is_bit_identical_to_per_span_formulation(emu, W, TC):
    """Halo recomputation + ring buffers (acc_tile.h) must not change a single bit versus the
    one-cell-at-a-time formulation (acc_core.h), for any tile width."""
    ref, _, _ = _tiled(emu.lib, _MIX, W, 5, None)
    got, _, _ = _tiled(emu.lib, _MIX, W, 5, TC)
    assert np.array_equal(ref.view(np.uint32), got.view(np.uint32))


def test_span_scaling_is_transparent_in_double(emu):
    ref, _, _ = _tiled(emu.lib, _MIX, 70, 5, None)
    got, _, _ = _tiled(emu.lib, _MIX, 70, 5, 352, scale=(0.3, 4.0, 16.0))
    assert np.abs(ref - got).max() < 2e-6


def test_fp32_engine_emulation_flags_out_of_range_sequences(emu):
    ref, _, lens = _tiled(emu.lib, _MIX, 70, 5, None)
    got, flags, _ = _tiled(emu.lib, _MIX, 70, 5, 704, scale=(0.3, 4.0, 16.0), f32=True)
    off = 0
    for k, L in enumerate(lens):
        seg = slice(off, off + 2 * int(L))
        off += 2 * int(L)
        if not flags[k]:
            assert np.abs(ref[seg] - got[seg]).max() < 6e-6, k
    assert flags[len(_MIX) - 1] == 1      # perfect 33-bp GC hairpin overflows float: must be flagged
    assert flags[0] == 0 and flags[1] == 0  # random sequences stay in range


@pytest.mark.parametrize("name", ["rand_L300_W70_d2", "rand_L300_W70_d10", "rand_L100_W20_d2", "rand_L500_W150_d2",
                                  "rand_L500_W70_d5", "gcstem_polyA_L576", "mixed_case_N_L300"])
def test_tiled_formulation_vs_reference(emu, name):
    """Tile march + tiled interior-loop strand weights (incl. the delta == 2 special loops) vs the fixtures."""
    case = next(c for c in GOLDEN if c["name"] == name)
    out, _, lens = _tiled(emu.lib, [case["seq"]], case["W"], case["delta"], 352 if case["W"] > 100 else 256)
    L = int(lens[0])
    assert_close_kcal(out[:L], case["acc"], ATOL_VS_REF, RTOL_VS_REF, "acc")
    assert_close_kcal(out[L:2 * L], case["cond"], ATOL_VS_REF, RTOL_VS_REF, "cond")


@pytest.mark.parametrize("W,TC,delta", [(70, 352, 5), (20, 64, 2), (150, 352, 10)])
def test_no_kernel_reads_a_cell_it_did_not_write(emu, W, TC, delta):
    """The device does not clear its DP state between batches: with every array poisoned with NaN the tile
    path must still give the same bits (every read is of a cell written earlier in the same batch)."""
    ref, _, _ = _tiled(emu.lib, _MIX, W, delta, TC)
    emu.lib.hostemu_set_poison(1)
    try:
        got, _, _ = _tiled(emu.lib, _MIX, W, delta, TC)
        got32, flags, _ = _tiled(emu.lib, _MIX, W, delta, TC, scale=(0.3, 4.0, 16.0), f32=True)
    finally:
        emu.lib.hostemu_set_poison(0)
    assert np.all(np.isfinite(got))
    assert np.array_equal(ref.view(np.uint32), got.view(np.uint32))
    assert np.all(np.isfinite(got32))


@pytest.fixture
def chain_mode(emu):
    emu.lib.hostemu_set_chain(1)
    yield emu
    emu.lib.hostemu_set_chain(0)


@pytest.mark.parametrize("W,TC,delta", [(70, 352, 5), (70, 512, 5), (20, 64, 2), (21, 96, 5), (150, 352, 10), (71, 256, 5)])
def test_centre_line_chain_matches_direct_sums(emu, chain_mode, W, TC, delta):
    """The chain formulation of the generic interior-loop sums (acc_tile.h, "Centre-line chain": H_{s+2} of the cell
    grown by one base on both sides = H_s + two end elements) evaluates the same terms as the time-tiled direct sums
    in another order: in double the float outputs agree to rounding; W = 21 / 71 exercise odd group starts."""
    got, _, _ = _tiled(emu.lib, _MIX, W, delta, TC)
    emu.lib.hostemu_set_chain(0)
    ref, _, _ = _tiled(emu.lib, _MIX, W, delta, TC)
    assert np.all(np.isfinite(got))
    assert np.abs(ref - got).max() < 1e-6
    ulp = np.abs(ref.view(np.int32).astype(np.int64) - got.view(np.int32).astype(np.int64))
    assert ulp.max() <= 2 and (ulp > 0).mean() < 0.01, (ulp.max(), (ulp > 0).mean())


def test_centre_line_chain_fp32_and_poison(emu, chain_mode):
    """FP32 span-scaled arithmetic with the chain (the device's fast engine), on NaN-poisoned state."""
    emu.lib.hostemu_set_chain(0)
    ref, _, lens = _tiled(emu.lib, _MIX, 70, 5, None)
    emu.lib.hostemu_set_chain(1)
    emu.lib.hostemu_set_poison(1)
    try:
        got, flags, _ = _tiled(emu.lib, _MIX, 70, 5, 512, scale=(0.3, 4.0, 16.0), f32=True)
    finally:
        emu.lib.hostemu_set_poison(0)
    off = 0
    for k, L in enumerate(lens):
        seg = slice(off, off + 2 * int(L))
        off += 2 * int(L)
        if not flags[k]:
            assert np.abs(ref[seg] - got[seg]).max() < 6e-6, k
    assert flags[len(_MIX) - 1] == 1 and flags[0] == 0 and flags[1] == 0


def test_tf32_split_stencil_keeps_parity(emu):
    """The generic-loop stencil products in the 3-product TF32 split of a tensor-core formulation
    (profiles/tc_probe.cu, profiles/tc_parity.py): the FP32 engine stays inside the reference gate."""
    emu.lib.hostemu_set_tf32_split(1)
    try:
        for name in ("rand_L500_W70_d5", "rand_L300_W70_d2"):
            case = next(c for c in GOLDEN if c["name"] == name)
            out, flags, lens = _tiled(emu.lib, [case["seq"]], case["W"], case["delta"], 256, (0.45, 4.0, 16.0), f32=True)
            L = int(lens[0])
            assert flags[0] == 0
            assert_close_kcal(out[:L], case["acc"], ATOL_VS_REF, RTOL_VS_REF, "acc")
            assert_close_kcal(out[L:2 * L], case["cond"], ATOL_VS_REF, RTOL_VS_REF, "cond")
    finally:
        emu.lib.hostemu_set_tf32_split(0)
