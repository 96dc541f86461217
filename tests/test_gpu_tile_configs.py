"""Every kernel configuration of the FP32 (mode 0) and FP64 (mode 1) tile engines, against the oracle, and the
properties that must not depend on the configuration.

The engines do not run one configuration: they pick one per context from the span W and the precision
(setup_engine and run_batch in acc_kernels.cu).
  * Strand-weight tile width TXb: 256, stepped down by 32 until the tile and its span lists fit the opt-in shared
    memory (232,448 bytes on sm_100).  256, 192 and 128 have their row stride compiled in; every other width runs the
    generic instantiation (run-time row stride, one CTA per SM).  PRIB_TXB forces a width from 32 to 512.
  * Inside/outside tiles: TC = 640 (FP32) or 288 (FP64) columns per CTA, TX = TC - (W + 1) of them owned and W + 1
    halo.  Tile boundaries fall at multiples of TX of the batch's columns.
  * The time-tiled span groups start at Tile::first_group(W) = (W + 2) mod 4, whose parity (that of W) selects the
    inside kernel's instantiation.

W ranges per TXb on sm_100 (strand_tile_width below):
    FP32: 1-167 -> 256, 168-187 -> 224 (generic), 188-200 -> 192
    FP64: 1-94 -> 256, 95-105 -> 224 (generic), 106-119 -> 192, 120-138 -> 160 (generic), 139-165 -> 128,
          166-200 -> 96 (generic)
The FP64 engine also re-runs, inside a mode-0 call, the sequences the FP32 engine flags.

`pytest -s` prints the measured deviations of every case."""
import numpy as np
import pytest

from conftest import (ATOL_VS_EXACT, ATOL_VS_REF, MEAN_VS_REF, RTOL_VS_EXACT, RTOL_VS_REF, assert_close_kcal,
                      parity_stats)

pytestmark = pytest.mark.gpu

BUDGET = 4 << 30        # DP budget per context: the GPUs are shared, and every batch here is far smaller
SMEM_OPTIN_SM100 = 232448
# The FP64 engine against the exact-libm twin.  The finalize step takes the reference's table log (fmath_logf, as the
# reference does) where the twin takes libm's: with libm's log there the FP64 formulation (host emulation, no tiles)
# stays within 0.62 of ATOL_VS_EXACT on random sequences at W = 100..200, with the table log it reaches 1.5.  Twice the
# exact-math gate is still 8x tighter than the reference gate.
ATOL_FP64_VS_EXACT = 2 * ATOL_VS_EXACT
RTOL_FP64_VS_EXACT = 2 * RTOL_VS_EXACT
TILE_COLS = {0: 640, 1: 288}  # TC of the inside/outside tiles: PRIB_TC32 / PRIB_TC64 of acc_kernels.cu
KPAD = 32                     # first column of a batch (kPad of acc_core.h)


def strand_tile_width(W, real_bytes, smem=SMEM_OPTIN_SM100):
    """TXb as setup_engine chooses it (bi_bytes: band tile + uint8 span lists + halo limits + barrier)."""
    rows, txb = max(W - 5, 0), 256
    while txb > 32 and rows * (txb + 36) * real_bytes + (W + 1) * txb + 32 * 4 + 64 > smem:
        txb -= 32
    return txb


def layout_columns(L):
    """Columns one sequence takes in a batch (acc_tables.h)."""
    return (L + 1 + KPAD + 31) // 32 * 32


def _geometry(W, mode):
    real_bytes = 4 if mode == 0 else 8
    return (f"TXb {strand_tile_width(W, real_bytes)}, TX {TILE_COLS[mode] - (W + 1)}, "
            f"first group {(W + 2) % 4}")


def _rand(rng, L, alpha="ACGU"):
    return "".join(alpha[k] for k in rng.integers(0, len(alpha), int(L)))


def _helix(W):
    """A perfect GC helix of W / 2 - 4 pairs: Boltzmann weights far outside the FP32 engine's safe range."""
    pairs = W // 2 - 4
    return "G" * pairs + "AAAA" + "C" * pairs


def _run(seqs, W, delta, mode):
    from priblast_b200 import Raccess
    with Raccess(W, delta, mode=mode, max_batch_bytes=BUDGET) as r:
        got = [(np.array(a), np.array(c)) for a, c in r.run_batch(seqs)]
        return got, r.counters()


def _assert_bits(got, want, what):
    assert len(got) == len(want), what
    for k, ((a, c), (wa, wc)) in enumerate(zip(got, want)):
        for g, w, name in ((a, wa, "acc"), (c, wc, "cond")):
            g, w = g.view(np.uint32), w.view(np.uint32)
            assert g.shape == w.shape, f"{what}: sequence {k} {name} shape"
            bad = np.flatnonzero(g != w)
            assert bad.size == 0, f"{what}: sequence {k} {name}: {bad.size} floats differ, first at {bad[0]}"


def _check_vs(got, want, atol, rtol, what):
    """Per-value gate of every sequence; returns (max |d|, mean |d|, largest |d| / limit) over all of them."""
    worst = 0.0
    for k, ((a, c), (wa, wc)) in enumerate(zip(got, want)):
        for g, w, name in ((a, wa, "acc"), (c, wc, "cond")):
            assert_close_kcal(g, w, atol, rtol, f"{what}: sequence {k} {name}")
            w64 = np.asarray(w, np.float64)
            if w64.size:
                worst = max(worst, float((np.abs(np.asarray(g, np.float64) - w64) / (atol + rtol * np.abs(w64))).max()))
    st = parity_stats(got, want)
    return st["max_abs"], st["mean_abs"], worst


def test_the_sweep_reaches_every_strand_weight_width_on_this_device():
    """The span sweep below is chosen for sm_100's opt-in shared memory; on another value its W would no longer cover
    every width (and both ends of each generic range)."""
    import torch
    optin = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    assert optin == SMEM_OPTIN_SM100, optin
    assert {strand_tile_width(W, 4) for W, _ in SWEEP} == {256, 224, 192}
    assert {strand_tile_width(W, 8) for W, _ in SWEEP} == {256, 224, 192, 160, 128, 96}
    for lo, hi, real_bytes in ((168, 187, 4), (95, 105, 8), (120, 138, 8), (166, 200, 8)):  # the generic ranges
        assert strand_tile_width(lo - 1, real_bytes) != strand_tile_width(lo, real_bytes)
        assert hi == 200 or strand_tile_width(hi + 1, real_bytes) != strand_tile_width(hi, real_bytes)
        assert {lo, hi} <= {W for W, _ in SWEEP}


# (W, delta): every TXb of both precisions, both ends of each generic range, odd and even W (first-group parity),
# delta 2..4 (strand kernels with ULO = 2) and >= 5 (ULO = 5), and one delta above 30.
#   W    FP32 TXb  FP64 TXb
#   70   256       256
#   94   256       256   (last FP64 256)
#   95   256       224   (first FP64 generic 224)
#   105  256       224   (last)
#   119  256       192
#   120  256       160   (first FP64 generic 160)
#   138  256       160   (last)
#   165  256       128
#   166  256       96    (first FP64 generic 96; last FP32 256 is 167)
#   168  224       96    (first FP32 generic 224)
#   175  224       96
#   187  224       96    (last FP32 generic 224)
#   188  192       96
#   200  192       96
SWEEP = [(70, 2), (94, 5), (95, 3), (105, 5), (119, 4), (120, 5), (138, 2), (165, 7), (166, 3), (168, 5), (175, 2),
         (187, 5), (188, 3), (200, 5), (200, 31)]

_ORACLE = {}  # (W, delta, exact) -> [(acc, cond)]: the CPU references are shared by both modes


def _sweep_inputs(W, delta):
    rng = np.random.default_rng(7919 * W + delta)
    return [_rand(rng, W), _rand(rng, W + 1), _rand(rng, 500), _rand(rng, 300, "ACGUNacgun")]


def _oracle(oracle_lib, W, delta, exact):
    key = (W, delta, exact)
    if key not in _ORACLE:
        seqs = _sweep_inputs(W, delta)
        if exact:
            _ORACLE[key] = [oracle_lib.run_exact(s, W, delta) for s in seqs]
        else:
            _ORACLE[key] = [(np.array(a), np.array(c)) for a, c in oracle_lib.run_batch(seqs, W, delta)[0]]
    return _ORACLE[key]


@pytest.mark.parametrize("W,delta", SWEEP, ids=[f"W{W}_d{d}" for W, d in SWEEP])
@pytest.mark.parametrize("mode", [0, 1])
def test_span_sweep_vs_restatement_and_exact_twin(oracle_lib, mode, W, delta):
    """Random ACGU sequences of length W, W + 1 and 500, and one with unknown bases and lower case, against the
    restatement of the reference (oracle/raccess_oracle.c) at the reference gate, max and mean.  The FP64 engine must
    also match the exact-libm twin at ATOL_FP64_VS_EXACT, 8x tighter: that is the gate a missing small term fails."""
    seqs = _sweep_inputs(W, delta)
    got, cnt = _run(seqs, W, delta, mode)
    for s, (a, c) in zip(seqs, got):
        assert np.all(c[:delta] == 0) and np.all(a[len(s) - delta + 1:] == 0), f"L={len(s)}"
    what = f"mode {mode} W={W} delta={delta} ({_geometry(W, mode)})"
    mx, mean, ratio = _check_vs(got, _oracle(oracle_lib, W, delta, False), ATOL_VS_REF, RTOL_VS_REF,
                                f"{what} vs restatement")
    ex = _oracle(oracle_lib, W, delta, True)
    st = parity_stats(got, ex)
    print(f"{what}, {cnt['fp64_rerun_sequences']} FP64 re-runs: vs restatement max|d|={mx:.2e} mean|d|={mean:.2e} "
          f"(max {ratio:.2f} of the limit); vs exact twin max|d|={st['max_abs']:.2e} mean|d|={st['mean_abs']:.2e}")
    assert mean <= MEAN_VS_REF, (what, mean)
    if mode == 1:
        _, _, ratio_ex = _check_vs(got, ex, ATOL_FP64_VS_EXACT, RTOL_FP64_VS_EXACT, f"{what} vs exact twin")
        print(f"    vs exact twin: max {ratio_ex:.2f} of ATOL_FP64_VS_EXACT")


@pytest.mark.parametrize("W", [100, 130, 175])
def test_fp64_rerun_at_the_generic_fp64_widths(oracle_lib, W):
    """A perfect GC helix the FP32 engine must flag, at spans whose FP64 strand-weight width is a generic one
    (TXb 224 / 160 / 96): the re-run in FP64 inside the mode-0 call must match the restatement.  (The exact-libm twin
    is no reference here: on a perfect helix the reference's own clamp puts it kcal/mol away from exact math.)"""
    rng = np.random.default_rng(W)
    seqs = [_rand(rng, 500), _rand(rng, 40) + _helix(W) + _rand(rng, 40), _rand(rng, W + 1)]
    got, cnt = _run(seqs, W, 5, 0)
    assert cnt["fp64_rerun_sequences"] >= 1, cnt["fp64_rerun_sequences"]
    mx, mean, ratio = _check_vs(got, oracle_lib.run_batch(seqs, W, 5)[0], ATOL_VS_REF, RTOL_VS_REF,
                                f"W={W} mode 0 with FP64 re-run")
    print(f"W={W} ({_geometry(W, 1)} for the re-run): {cnt['fp64_rerun_sequences']} FP64 re-runs, vs restatement "
          f"max|d|={mx:.2e} mean|d|={mean:.2e} (max {ratio:.2f} of the limit)")
    assert mean <= MEAN_VS_REF, mean


@pytest.mark.parametrize("W,delta,mode", [(70, 2, 0), (70, 5, 0), (70, 2, 1), (70, 5, 1), (175, 5, 0)])
def test_forced_strand_weight_widths_are_bit_identical(monkeypatch, W, delta, mode):
    """Each strand-weight thread owns one column and sums over its own list of spans, so the CTA width must not change
    a single output bit.  Every multiple of 32 from 32 to 512 is forced through PRIB_TXB (read when a context is
    created); widths that do not fit the shared memory step down as they would by default.  In mode 0 the helix is
    re-run by the FP64 engine at the forced width too."""
    rng = np.random.default_rng(100 * W + delta)
    seqs = [_rand(rng, 1500), _rand(rng, 700), _rand(rng, 300, "ACGUNacgun"), _helix(W), _rand(rng, W + 1)]
    monkeypatch.delenv("PRIB_TXB", raising=False)
    want, cnt = _run(seqs, W, delta, mode)
    if mode == 0:
        assert cnt["fp64_rerun_sequences"] >= 1
    for txb in range(32, 513, 32):
        monkeypatch.setenv("PRIB_TXB", str(txb))
        got, c = _run(seqs, W, delta, mode)
        assert c["fp64_rerun_sequences"] == cnt["fp64_rerun_sequences"], txb
        _assert_bits(got, want, f"W={W} delta={delta} mode {mode} PRIB_TXB={txb}")


# Tile boundaries at chosen columns of a probe.  The engine sorts a batch longest first (stable), places the first
# sequence at column 32 and gives each sequence layout_columns(L) = 32 * ceil((L + 33) / 32) columns.  So behind one
# filler of length F >= P the probe starts at S = 32 + layout_columns(F), and its column x lies on a tile boundary when
# S + x is a multiple of TX.  With W even, TX = TC - W - 1 is odd, so such an F exists for every x.
# Columns x: -W (the outside pass's halo reaches W + 1 columns left), 0, 1, W, W + 1, P - W - 1, P - 1 and P (the column
# holding log Z).  Example, mode 1, W = 200, x = 0: F = 2719, S = 32 + 2752 = 2784 = 32 * 87.
PROBE_LEN = 520
EDGE_FILLERS = {  # (mode, W): (TX, filler length per column x in the order above)
    (0, 20): (619, [2431, 19743, 1791, 17247, 19103, 14911, 12415, 14271]),
    (0, 70): (569, [5695, 18143, 5055, 12383, 17503, 4607, 17055, 3967]),
    (0, 200): (439, [3647, 13983, 3007, 10271, 13343, 10591, 6879, 9951]),
    (1, 70): (217, [2175, 6879, 1887, 4639, 6591, 1439, 6143, 1151]),
    (1, 200): (87, [831, 2719, 543, 1823, 2431, 1791, 895, 1503]),
}


@pytest.mark.parametrize("mode,W", list(EDGE_FILLERS), ids=[f"mode{m}_W{W}" for m, W in EDGE_FILLERS])
def test_placement_at_tile_edges_is_bit_identical(mode, W):
    """Results do not depend on batching (include/priblast_acc.h): a probe whose columns 0, 1, W, ... fall on an
    inside/outside tile boundary must give the bits it gives alone.  A halo or ring mistake shows up as a value that
    changes with where the sequence sits."""
    from priblast_b200 import Raccess
    P = PROBE_LEN
    TX, fillers = EDGE_FILLERS[(mode, W)]
    assert TX == TILE_COLS[mode] - (W + 1)
    rng = np.random.default_rng(31 * W + mode)
    probe = _rand(rng, P)
    with Raccess(W, 5, mode=mode, max_batch_bytes=BUDGET) as r:
        alone = [tuple(np.array(v) for v in r.run_batch([probe])[0])]
        assert r.counters()["fp64_rerun_sequences"] == 0  # mode 0: the FP32 tiles computed the probe
        for x, F in zip([-W, 0, 1, W, W + 1, P - W - 1, P - 1, P], fillers):
            S = KPAD + layout_columns(F)
            assert F >= P and (S + x) % TX == 0, (x, F)
            res = r.run_batch([_rand(rng, F), probe])
            _assert_bits([tuple(np.array(v) for v in res[1])], alone,
                         f"mode {mode} W={W}: probe column {x} on a tile boundary (filler {F})")
