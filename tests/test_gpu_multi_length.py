"""Several minimum accessible lengths from one context (prib_acc_create_lengths / Raccess(W, [d1, d2, ...])) on the
GPU: every output float equals, bit for bit, that of a single-length context on the same inputs, in every engine
(FP32 tiles with FP64 re-run, FP64 tiles, exact, wide-span), every call form and in the `db` front-end."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, ROOT

pytestmark = pytest.mark.gpu

FRONT = os.path.join(ROOT, "priblast_b200", "pRIblast_b200")
LENGTHS = (2, 5, 8, 31)  # the delta == 2 special loops, the default, and a length above 30


def _rand(rng, L, alpha="ACGU"):
    return "".join(alpha[k] for k in rng.integers(0, len(alpha), int(L)))


def _mixed_seqs():
    """40 sequences of 50 .. 3,000 nt: N runs, lower case, and one sequence shorter than the largest length."""
    rng = np.random.default_rng(2031)
    seqs = [_rand(rng, L) for L in rng.integers(50, 3000, 34)]
    seqs += [_rand(rng, 400) + "N" * 25 + _rand(rng, 300), "NNNN" + _rand(rng, 150, "ACGUacgu") + "nnn",
             _rand(rng, 900, "acgu"), _rand(rng, 1200, "ACGTNacgtn"), _rand(rng, 20), _rand(rng, 60)]
    return seqs


SEQS = _mixed_seqs()


def _copy(res):
    return [(np.array(a), np.array(c)) for a, c in res]


def _single(seqs, W, delta, mode=0, **kw):
    from priblast_b200 import Raccess
    with Raccess(W, delta, mode=mode, **kw) as r:
        out = _copy(r.run_batch(seqs))
        return out, r.counters()


def _multi(seqs, W, lengths, mode=0, **kw):
    from priblast_b200 import Raccess
    with Raccess(W, list(lengths), mode=mode, **kw) as r:
        assert r.lengths == tuple(lengths)
        res = r.run_batch(seqs)
        assert sorted(res) == sorted(lengths)
        return {d: _copy(v) for d, v in res.items()}, r.counters()


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _assert_bits(got, want, what):
    assert len(got) == len(want), what
    for k, ((a, c), (oa, oc)) in enumerate(zip(got, want)):
        for g, w, name in ((a, oa, "acc"), (c, oc, "cond")):
            g, w = _bits(g), _bits(w)
            assert g.shape == w.shape, f"{what}: sequence {k} {name} shape"
            bad = np.flatnonzero(g != w)
            assert bad.size == 0, f"{what}: sequence {k} {name}: {bad.size} floats differ, first at {bad[0]}"


@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("W", [20, 70, 150])
def test_every_length_equals_its_single_length_context(W, mode):
    multi, cnt = _multi(SEQS, W, LENGTHS, mode=mode)
    for d in LENGTHS:
        want, single_cnt = _single(SEQS, W, d, mode=mode)
        _assert_bits(multi[d], want, f"W={W} mode={mode} delta={d}")
        assert cnt["fp64_rerun_sequences"] == single_cnt["fp64_rerun_sequences"]
    assert cnt["sequences"] == len(SEQS) and cnt["nucleotides"] == sum(map(len, SEQS))
    assert cnt["d2h_bytes"] == len(LENGTHS) * 8 * sum(map(len, SEQS))


def test_exact_engine_matches_the_oracle_at_every_length(oracle_lib):
    seqs = [s for s in SEQS if len(s) <= 700][:8]
    multi, _ = _multi(seqs, 70, LENGTHS, mode=2)
    for d in LENGTHS:
        want, _ = oracle_lib.run_batch(seqs, 70, d)
        _assert_bits(multi[d], want, f"exact engine vs oracle, delta={d}")


@pytest.mark.parametrize("mode", [0, 2])
def test_wide_spans(mode):
    rng = np.random.default_rng(250)
    seqs = [_rand(rng, L) for L in rng.integers(100, 1500, 10)] + [_rand(rng, 30)]
    multi, _ = _multi(seqs, 250, (5, 40), mode=mode)
    for d in (5, 40):
        want, _ = _single(seqs, 250, d, mode=mode)
        _assert_bits(multi[d], want, f"W=250 mode={mode} delta={d}")


def test_wide_engine_exact_rerun_counts_each_sequence_once():
    """The GC helix of test_gpu_wide.py leaves the wide engine's range at W = 600: it is re-run once, in the exact
    engine, for both lengths."""
    W = 600
    rng = np.random.default_rng(600)
    helix = _rand(rng, 2000) + "G" * (W // 2) + "AAAA" + "C" * (W // 2) + _rand(rng, 50)
    plain = [_rand(rng, 900), _rand(rng, 1300)]
    seqs = [plain[0], helix, plain[1]]
    multi, cnt = _multi(seqs, W, (5, 40))
    for d in (5, 40):
        want, single_cnt = _single(seqs, W, d)
        _assert_bits(multi[d], want, f"W=600 delta={d}")
        assert single_cnt["exact_rerun_sequences"] >= 1
        assert cnt["exact_rerun_sequences"] == single_cnt["exact_rerun_sequences"]


def test_fp64_rerun_counts_each_sequence_once():
    names = ["perfect_hairpin_L70", "rand_L500_W70_d5", "gcstem_polyA_L576", "rand_L300_W70_d5"]
    seqs = [next(c for c in GOLDEN if c["name"] == n)["seq"] for n in names]
    multi, cnt = _multi(seqs, 70, (5, 12))
    assert cnt["fp64_rerun_sequences"] >= 1
    for d in (5, 12):
        want, single_cnt = _single(seqs, 70, d)
        _assert_bits(multi[d], want, f"golden re-run cases, delta={d}")
        assert cnt["fp64_rerun_sequences"] == single_cnt["fp64_rerun_sequences"]
        assert cnt["fp32_flagged"] == single_cnt["fp32_flagged"]


def test_call_forms_give_the_same_bits():
    from priblast_b200 import Raccess, _capi
    seqs = SEQS[:24]
    lengths = (2, 5, 31)
    ref, _ = _multi(seqs, 70, lengths)
    lens = np.array([len(s) for s in seqs], dtype=np.int32)
    total = 2 * int(lens.sum())
    n, k = len(seqs), len(lengths)
    with Raccess(70, list(lengths)) as r:
        # stage / compute / fetch
        r.stage(seqs)
        r.compute()
        got = r.fetch()
        for d in lengths:
            _assert_bits(_copy(got[d]), ref[d], f"stage/compute/fetch delta={d}")
        # packed layout into page-locked memory: the device image is copied straight into the caller's buffer
        lib = r._lib
        buf = lib.prib_host_alloc(4 * k * total)
        try:
            out = np.ctypeslib.as_array(ctypes.cast(buf, _capi.c_f32p), shape=(k * total,))
            acc_off, cond_off, _ = r._layout(lens)
            bs, n2, lens2, arr = r._marshal(seqs)
            _capi.check(lib.prib_acc_run(r._ctx, n2, arr, lens2.ctypes.data_as(_capi.c_i32p), ctypes.c_void_p(buf),
                                         acc_off.ctypes.data_as(_capi.c_i64p), cond_off.ctypes.data_as(_capi.c_i64p)))
            for l, d in enumerate(lengths):
                got = [(out[acc_off[l * n + q]:acc_off[l * n + q] + lens[q]].copy(),
                        out[cond_off[l * n + q]:cond_off[l * n + q] + lens[q]].copy()) for q in range(n)]
                _assert_bits(got, ref[d], f"page-locked packed delta={d}")
        finally:
            lib.prib_host_free(buf)
        # offsets that are not packed (lengths and sequences in reverse order): the scatter path
        acc_off = np.empty(k * n, np.int64)
        cond_off = np.empty(k * n, np.int64)
        o = 0
        for l in reversed(range(k)):
            for q in reversed(range(n)):
                acc_off[l * n + q], cond_off[l * n + q] = o + lens[q], o
                o += 2 * int(lens[q])
        out = np.full(o, np.nan, np.float32)
        bs, n2, lens2, arr = r._marshal(seqs)
        _capi.check(lib.prib_acc_run(r._ctx, n2, arr, lens2.ctypes.data_as(_capi.c_i32p),
                                     out.ctypes.data_as(ctypes.c_void_p), acc_off.ctypes.data_as(_capi.c_i64p),
                                     cond_off.ctypes.data_as(_capi.c_i64p)))
        for l, d in enumerate(lengths):
            got = [(out[acc_off[l * n + q]:acc_off[l * n + q] + lens[q]], out[cond_off[l * n + q]:cond_off[l * n + q] + lens[q]])
                   for q in range(n)]
            _assert_bits(got, ref[d], f"scattered delta={d}")
    # a small DP budget: several device batches
    small, cnt = _multi(seqs, 70, lengths, max_batch_bytes=100 << 20)
    assert cnt["batches"] > 1
    for d in lengths:
        _assert_bits(small[d], ref[d], f"several batches delta={d}")


def test_one_length_list_equals_prib_acc_create():
    from priblast_b200 import _capi
    lib = _capi.load()
    seqs = SEQS[:10]
    want, want_cnt = _single(seqs, 70, 8)
    one, cnt = _multi(seqs, 70, [8])
    _assert_bits(one[8], want, "create_lengths(p, 1, &8)")
    assert cnt["kernel_launches"] == want_cnt["kernel_launches"]
    # the C ABI directly, min_accessible_length left at 0: it is not read
    ctx = ctypes.c_void_p()
    prm = _capi.AccParams(70, 0, 0, 0, 8 << 30)
    d = np.array([8], np.int32)
    _capi.check(lib.prib_acc_create_lengths(ctypes.byref(ctx), ctypes.byref(prm), 1, d.ctypes.data_as(_capi.c_i32p)))
    lib.prib_acc_destroy(ctx)


def test_phase_times_and_launches():
    from priblast_b200 import Raccess
    with Raccess(70, [5, 8, 12]) as r:
        r.run_batch(SEQS[:8])
        cnt = r.counters()
    for p in ("inside", "outside", "biloop_left", "biloop_right", "hairpin_finalize"):
        assert cnt["phase_ms"][p] > 0, cnt["phase_ms"]
    # per batch: layout, inside, scans, outside, and (left, right, finalize) per length
    assert cnt["kernel_launches"] == cnt["batches"] * (4 + 3 * 3)


def _write(path, seqs):
    with open(path, "w") as f:
        for k, s in enumerate(seqs):
            f.write(f">t{k}\n")
            for p in range(0, len(s), 60):
                f.write(s[p:p + 60] + "\n")


@pytest.mark.parametrize("extra", [[], ["-m", "exact", "-c", "5"]])
def test_db_front_end_writes_one_identical_database_per_length(tmp_path, extra):
    subprocess.run(["make", "-C", os.path.join(ROOT, "priblast_b200", "csrc", "host")], check=True,
                   stdout=subprocess.DEVNULL)
    rng = np.random.default_rng(59)
    seqs = [_rand(rng, L) for L in rng.integers(30, 1500, 14)] + [_rand(rng, 300, "ACGUNacgu")]
    fa = str(tmp_path / "in.fa")
    _write(fa, seqs)
    subprocess.run([FRONT, "db", "-i", fa, "-o", str(tmp_path / "m"), "-d", "5,9", *extra], check=True)
    for d in (5, 9):
        subprocess.run([FRONT, "db", "-i", fa, "-o", str(tmp_path / f"s{d}"), "-d", str(d), *extra], check=True)
        for ext in (".acc", ".seq", ".ind", ".nam", ".bas"):
            a = open(str(tmp_path / f"m_d{d}") + ext, "rb").read()
            b = open(str(tmp_path / f"s{d}") + ext, "rb").read()
            assert a == b, f"-d 5,9 vs -d {d}: {ext} differs"
