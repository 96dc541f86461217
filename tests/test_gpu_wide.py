"""Spans above 200 and minimum accessible lengths above 30 on the GPU: the exact engine bit for bit against the oracle,
the wide-span FP64 engine (modes 0 and 1 at W > 200) within the repository tolerance of the reference arithmetic, its
exact re-run of out-of-range sequences, batching invariance, the FP32 tile path at delta > 30, and the `db` front-end
at -w 300 -d 40."""
import os
import subprocess

import numpy as np
import pytest

from conftest import (ATOL_VS_EXACT, ATOL_VS_REF, MEAN_VS_REF, ROOT, RTOL_VS_EXACT, RTOL_VS_REF, assert_close_kcal,
                      parity_stats)

pytestmark = pytest.mark.gpu

FRONT = os.path.join(ROOT, "priblast_b200", "pRIblast_b200")


def _rand(rng, L):
    return "".join("ACGU"[k] for k in rng.integers(0, 4, int(L)))


def _run(seqs, W, delta, mode=0, budget=16 << 30, calls=1):
    from priblast_b200 import Raccess
    out = []
    with Raccess(W, delta, max_batch_bytes=budget, mode=mode) as r:
        step = -(-len(seqs) // calls)
        for k in range(0, len(seqs), step):
            out += [(np.array(a), np.array(c)) for a, c in r.run_batch(seqs[k:k + step])]
        cnt = r.counters()
    return out, cnt


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _assert_bits(got, want, what):
    for k, ((a, c), (oa, oc)) in enumerate(zip(got, want)):
        for g, w, name in ((a, oa, "acc"), (c, oc, "cond")):
            bad = np.nonzero(_bits(g) != _bits(w))[0]
            assert bad.size == 0, f"{what} seq {k} {name}: {bad.size} floats differ, first at {bad[0]}"


def _gate(got, want, what, k=1.0):
    """Every value within k times the repository tolerance (1e-4 + 1e-6 |x| kcal/mol), and the mean deviation gated."""
    st = parity_stats(got, want)
    print(f"{what}: n={st['n']} max|d|={st['max_abs']:.3e} mean|d|={st['mean_abs']:.3e} kcal/mol")
    for (a, c), (oa, oc) in zip(got, want):
        assert_close_kcal(a, oa, k * ATOL_VS_REF, k * RTOL_VS_REF, f"{what} acc")
        assert_close_kcal(c, oc, k * ATOL_VS_REF, k * RTOL_VS_REF, f"{what} cond")
    assert st["mean_abs"] <= MEAN_VS_REF, (what, st)


@pytest.mark.parametrize("W,delta", [(201, 31), (250, 5), (400, 40), (1000, 31)])
def test_exact_engine_bitwise_vs_oracle(oracle_lib, W, delta):
    """Mode 2 at wide spans: every float equal to the oracle's, including a sequence shorter than W."""
    rng = np.random.default_rng(W + delta)
    seqs = [_rand(rng, W // 2), _rand(rng, W + 150), _rand(rng, 700)]
    seqs[2] = seqs[2][:200].lower() + "NNN" + seqs[2][203:]
    got, _ = _run(seqs, W, delta, mode=2)
    want, _ = oracle_lib.run_batch(seqs, W, delta)
    _assert_bits(got, want, f"exact W={W} delta={delta}")


# The reference's float-table log-sums drift from exact math with the number of terms per sum, which grows with W: at
# W = 400 and L = 3 kb the reference arithmetic alone differs from exact libm math by up to 8.2e-5 kcal/mol (three
# sequences of this set), while the wide-span formulation stays within 1e-6 of exact math.  At W = 400 the comparison
# with the reference's arithmetic therefore allows twice the repository tolerance (one value of 321,434 is 1.01e-4
# off at |x| = 1.09); the engine's own error is pinned against exact math in the next test.
@pytest.mark.parametrize("W,k", [(201, 1.0), (250, 1.0), (400, 2.0)])
def test_wide_engine_vs_reference_arithmetic(W, k):
    """Modes 0 and 1 (the wide-span engine) on 100 random 300-3,000 nt sequences against the exact engine (the
    reference's arithmetic, pinned bit for bit to the oracle above)."""
    rng = np.random.default_rng(1000 + W)
    seqs = [_rand(rng, L) for L in rng.integers(300, 3001, 100)]
    exact, _ = _run(seqs, W, 5, mode=2)
    auto, cnt0 = _run(seqs, W, 5, mode=0)
    fp64, _ = _run(seqs, W, 5, mode=1)
    _assert_bits(auto, fp64, f"mode 0 vs mode 1 W={W}")
    print(f"W={W}: exact re-runs {cnt0['exact_rerun_sequences']} of 100")
    _gate(auto, exact, f"wide engine W={W} vs reference arithmetic", k)


def test_wide_engine_vs_exact_math(oracle_lib):
    """W = 400: the wide-span engine against the oracle's exact-libm twin, at float-rounding level."""
    rng = np.random.default_rng(401)
    seqs = [_rand(rng, 1500), _rand(rng, 1200)]
    got, _ = _run(seqs, 400, 5)
    for s, (a, c) in zip(seqs, got):
        ea, ec = oracle_lib.run_exact(s, 400, 5)
        assert_close_kcal(a, ea, ATOL_VS_EXACT, RTOL_VS_EXACT, "acc")
        assert_close_kcal(c, ec, ATOL_VS_EXACT, RTOL_VS_EXACT, "cond")


@pytest.mark.parametrize("delta", [31, 60])
def test_fp32_tile_path_above_delta_30(oracle_lib, delta):
    """delta > 30 at W = 70: the FP32 tile kernels (no interior-loop strand terms remain) against the oracle."""
    rng = np.random.default_rng(delta)
    seqs = [_rand(rng, L) for L in rng.integers(100, 1500, 40)]
    got, _ = _run(seqs, 70, delta, mode=0)
    want, _ = oracle_lib.run_batch(seqs, 70, delta)
    _gate(got, want, f"FP32 tiles W=70 delta={delta} vs oracle")


def test_out_of_range_sequence_is_rerun_exactly(oracle_lib):
    """A perfect GC helix of W/2 pairs behind 2 kb at W = 600 leaves the FP64 range: the wide engine flags it and the
    exact engine recomputes it, bit for bit the oracle's values; the other sequences stay in the wide engine."""
    W = 600
    rng = np.random.default_rng(600)
    helix = _rand(rng, 2000) + "G" * (W // 2) + "AAAA" + "C" * (W // 2) + _rand(rng, 50)
    plain = [_rand(rng, 900), _rand(rng, 1300)]
    got, cnt = _run([plain[0], helix, plain[1]], W, 5, mode=0)
    assert cnt["exact_rerun_sequences"] >= 1
    want, _ = oracle_lib.run_batch([helix], W, 5)
    _assert_bits([got[1]], want, "re-run helix")
    want_plain, _ = oracle_lib.run_batch(plain, W, 5)
    for (a, c), (oa, oc) in zip([got[0], got[2]], want_plain):
        assert_close_kcal(a, oa, ATOL_VS_REF, RTOL_VS_REF, "acc")
        assert_close_kcal(c, oc, ATOL_VS_REF, RTOL_VS_REF, "cond")


def test_wide_engine_batching_invariance():
    """W = 300: one call, several calls and a small DP budget (several device batches) give the same bits."""
    rng = np.random.default_rng(300)
    seqs = [_rand(rng, L) for L in rng.integers(200, 1500, 24)]
    one, _ = _run(seqs, 300, 5)
    split, _ = _run(seqs, 300, 5, calls=3)
    small, cnt = _run(seqs, 300, 5, budget=150 << 20)
    assert cnt["batches"] > 1
    _assert_bits(split, one, "three calls")
    _assert_bits(small, one, "small budget")


def _write(path, seqs):
    with open(path, "w") as f:
        for k, s in enumerate(seqs):
            f.write(f">t{k}\n")
            for p in range(0, len(s), 60):
                f.write(s[p:p + 60] + "\n")


def _read_acc(path):
    raw, out, p = open(path, "rb").read(), [], 0
    while p < len(raw):
        n1 = int(np.frombuffer(raw[p:p + 4], np.int32)[0])
        start = p
        p += 4 + 4 * n1
        L = int(np.frombuffer(raw[p:p + 4], np.int32)[0])
        p += 4 + 4 * L
        out.append((L, raw[start:p]))
    return out


def _record(lib, acc, cond, delta):
    import ctypes
    L = len(acc)
    buf = ctypes.create_string_buffer(int(lib.prib_acc_record_bytes(L, delta)))
    a, c = np.ascontiguousarray(acc, np.float32), np.ascontiguousarray(cond, np.float32)
    f32p = ctypes.POINTER(ctypes.c_float)
    assert lib.prib_acc_write_record(a.ctypes.data_as(f32p), c.ctypes.data_as(f32p), L, delta, buf) == len(buf.raw)
    return buf.raw


def test_db_front_end_wide_span(tmp_path, oracle_lib):
    from priblast_b200 import _capi
    subprocess.run(["make", "-C", os.path.join(ROOT, "priblast_b200", "csrc", "host")], check=True,
                   stdout=subprocess.DEVNULL)
    rng = np.random.default_rng(340)
    lens = sorted({int(L) for L in rng.integers(60, 900, 14)})  # distinct lengths: records are matched by length
    seqs = [_rand(rng, L) for L in lens]
    fa = str(tmp_path / "db.fa")
    _write(fa, seqs)
    for name, extra in (("w70", ["-w", "70"]), ("fast", ["-w", "300", "-d", "40"]),
                        ("exact", ["-w", "300", "-d", "40", "-m", "exact"])):
        subprocess.run([FRONT, "db", "-i", fa, "-o", str(tmp_path / name), *extra], check=True)
    for name in ("fast", "exact"):
        assert np.array_equal(np.fromfile(str(tmp_path / name) + ".bas", np.int32), [8, 0, 300, 40])
        for ext in (".seq", ".ind", ".nam"):
            assert open(str(tmp_path / name) + ext, "rb").read() == open(str(tmp_path / "w70") + ext, "rb").read(), ext
    want, _ = oracle_lib.run_batch(seqs, 300, 40)
    lib = _capi.load()
    want_rec = {len(s): _record(lib, a, c, 40) for s, (a, c) in zip(seqs, want)}
    exact = _read_acc(str(tmp_path / "exact") + ".acc")
    fast = _read_acc(str(tmp_path / "fast") + ".acc")
    assert sorted(L for L, _ in exact) == lens and sorted(L for L, _ in fast) == lens
    for L, rec in exact:
        assert rec == want_rec[L], f"exact .acc record of length {L} differs"
    for L, rec in fast:
        got = np.frombuffer(rec, np.float32)
        ref = np.frombuffer(want_rec[L], np.float32)
        assert got.size == ref.size and np.array_equal(got[[0, L - 40 + 2]].view(np.int32), ref[[0, L - 40 + 2]].view(np.int32))
        assert_close_kcal(got, ref, ATOL_VS_REF, RTOL_VS_REF, f"fast .acc record of length {L}")
