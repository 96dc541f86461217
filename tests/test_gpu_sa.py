"""GPU suffix array (SURVEY section 8 row f2): prib_suffix_array, the drop-in for the reference's sais() call
(db_construction.cpp:334), against the host checker on encoded database texts.  The suffix array of a
text is unique, so equality with any correct builder is equality with the reference's bytes; the e2e test
(test_gpu_db.py) additionally compares the <db>.ind file with the one the reference binary writes."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def host_sa():
    d = os.path.join(ROOT, "priblast_b200", "csrc", "host")
    subprocess.run(["make", "-C", d, os.path.join(ROOT, "priblast_b200", "libprib_dbformat.so")], check=True,
                   stdout=subprocess.DEVNULL)
    lib = ctypes.CDLL(os.path.join(ROOT, "priblast_b200", "libprib_dbformat.so"))

    def run(text):
        text = np.ascontiguousarray(text, dtype=np.uint8)
        sa = np.zeros(len(text), np.int32)
        lib.prib_suffix_array_host(text.ctypes.data_as(ctypes.c_void_p), len(text), sa.ctypes.data_as(ctypes.c_void_p))
        return sa
    return run


def _page(rng, lens, alphabet=(2, 3, 4, 5)):
    """Encoded page: sequences over the database alphabet, each followed by the sentinel 0."""
    parts = []
    for L in lens:
        parts.append(np.asarray(alphabet, np.uint8)[rng.integers(0, len(alphabet), L)])
        parts.append(np.zeros(1, np.uint8))
    return np.concatenate(parts)


@pytest.mark.parametrize("case", ["random", "tiny", "polyA", "tandem", "two_copies", "lowercase"])
def test_matches_host_builder(host_sa, case):
    from priblast_b200 import suffix_array
    rng = np.random.default_rng(11)
    if case == "random":
        text = _page(rng, rng.integers(20, 3000, 200))
    elif case == "tiny":
        for text in (np.array([0], np.uint8), np.array([3, 0], np.uint8), _page(rng, [5, 6, 7])):
            assert np.array_equal(suffix_array(text), host_sa(text))
        return
    elif case == "polyA":  # one rank class per round: the doubling has to run to the end
        text = np.concatenate([np.full(5000, 2, np.uint8), np.zeros(1, np.uint8)])
    elif case == "tandem":
        unit = np.array([2, 3, 4, 5, 5, 4, 3], np.uint8)
        text = np.concatenate([np.tile(unit, 900), np.zeros(1, np.uint8), np.tile(unit, 500), np.zeros(1, np.uint8)])
    elif case == "two_copies":  # identical sequences: ties are broken by what follows the sentinel
        s = np.asarray((2, 3, 4, 5), np.uint8)[rng.integers(0, 4, 2500)]
        text = np.concatenate([s, [0], s, [0], s[:1000], [0]]).astype(np.uint8)
    else:  # repeat_flag 1 keeps lower case as 6..9, unknown = 1 (encoder.hpp:36-78)
        text = _page(rng, rng.integers(50, 800, 60), alphabet=(1, 2, 3, 4, 5, 6, 7, 8, 9))
    got = suffix_array(text)
    assert np.array_equal(got, host_sa(text))
    assert np.array_equal(np.sort(got), np.arange(len(text), dtype=np.int32))  # a permutation


def test_rejects_symbols_outside_the_database_alphabet():
    from priblast_b200 import _capi, suffix_array
    with pytest.raises(_capi.PribError):
        suffix_array(np.array([2, 3, 200, 0], np.uint8))


def test_large_page_is_sorted():
    """2e7 symbols (about 10k transcripts): checked through the defining property on a sample of neighbours."""
    from priblast_b200 import suffix_array, workloads
    rng = np.random.default_rng(5)
    lens = workloads.cfg2_lengths(100_000)[:10_000]
    text = _page(rng, lens)
    sa = suffix_array(text)
    assert len(sa) == len(text) and sa.min() == 0 and sa.max() == len(text) - 1
    raw = text.tobytes()
    for j in rng.integers(0, len(sa) - 1, 4000):
        a, b = int(sa[j]), int(sa[j + 1])
        assert raw[a:a + 64] <= raw[b:b + 64] and (raw[a:a + 64] != raw[b:b + 64] or raw[a:] < raw[b:])


# The suffix arrays of the four texts below, as the SHA-256 of their little-endian int32 bytes and their values at 8
# positions drawn with default_rng(0) (so that a mismatch names an index).  A text has one suffix array, so this is the
# array the reference's builder (sais.cpp:656, the call of db_construction.cpp:334) returns; the values were computed
# by prefix doubling in numpy and by the host builder, which agree, not by that builder.
SAIS_GOLDEN = [
    (596048, "721c83455ac85324515314c101acbde74f896be9a63a9325302da8a14fa0c1d5",
     [230502, 508991, 344155, 209061, 402099, 178865, 93982, 475028]),
    (2103, "6dcc80542d4a67a96e2a681293a10bb1598f0b9d0ff7977113a71bde2a6c4d15",
     [1390, 672, 648, 512, 1186, 1044, 1657, 1508]),
    (11861, "8fb34bd1570bddd814d2704a3ce39d680330e57f447dc3243b623c41c66b44e6",
     [5491, 9937, 4395, 4023, 6282, 9045, 3365, 6918]),
    (2338, "108516c4ac8996df2f6b33202fb37ce056af184125594779ab8cdb0ae36957a8",
     [1059, 769, 2021, 312, 885, 1633, 1840, 1977]),
]


def test_matches_the_references_own_sais():
    """Same text in, the same `int` array out as the reference's builder."""
    import hashlib
    from priblast_b200 import suffix_array
    rng = np.random.default_rng(5)
    texts = [_page(rng, rng.integers(20, 4000, 300)), _page(rng, [700] * 3, alphabet=(2,)),
             _page(rng, rng.integers(50, 500, 40), alphabet=(2, 3, 4, 5, 6, 7, 8, 9)),
             np.tile(_page(rng, [333]), 7)]
    for text, (n, digest, sample) in zip(texts, SAIS_GOLDEN):
        text = np.ascontiguousarray(text, np.uint8)
        assert len(text) == n
        got = suffix_array(text)
        pos = np.sort(np.random.default_rng(0).choice(n, 8, replace=False))
        for p, want in zip(pos, sample):
            assert got[p] == want, f"text of {n} symbols: SA[{p}] = {got[p]}, want {want}"
        assert hashlib.sha256(got.astype("<i4").tobytes()).hexdigest() == digest, f"text of {n} symbols"
