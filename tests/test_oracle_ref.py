"""Pin the oracle's SA / sa_search / LUT restatements: to the definitions they implement (a suffix array is every suffix
in byte-wise order; on a sorted range, sa_searchb64 bisects to the suffixes that start with the pattern), to the
reference's real C library where it is built (oracle/_ref, compiled in place by oracle/Makefile from the reference's
libdivsufsort sources), and to the committed golden fixtures made from it (tests/golden/make_golden.py)."""
import bisect
import ctypes as C
import json
import os

import numpy as np
import pytest

import oracle
from tests import kat

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _texts():
    rng = np.random.default_rng(2026)
    out = {}
    out["random4k"] = np.concatenate([kat.rand_dna(rng, 4000), [ord("$")]]).astype(np.uint8)
    t = kat.rand_dna(rng, 6000); t[1000:1700] = ord("N"); t[3000:3600] = t[200:800]; t[5990:] = ord("N")
    out["nrun_dup6k"] = np.concatenate([t, [ord("$")]]).astype(np.uint8)
    out["polyA"] = np.frombuffer(b"A" * 777 + b"$", dtype=np.uint8).copy()
    out["no_terminator"] = kat.rand_dna(rng, 3000)                 # divsufsort contract without '$'
    out["bytes"] = rng.integers(0, 256, size=5000).astype(np.uint8)  # full byte alphabet
    out["abab"] = np.frombuffer(b"AB" * 500, dtype=np.uint8).copy()
    out["tiny1"] = np.frombuffer(b"$", dtype=np.uint8).copy()
    out["tiny2"] = np.frombuffer(b"A$", dtype=np.uint8).copy()
    return out


def _suffixes(t, sa, l=0, r=None):
    """The suffixes sa[l:r] points at, as bytes (quadratic memory: for the small texts of this module)."""
    b = bytes(t)
    return [b[i:] for i in sa[l:r]]


def _equal_range(suffixes, p: bytes):
    """(first index, count) of the sorted `suffixes` that start with p; for an absent p, where it would be inserted."""
    lo = bisect.bisect_left(suffixes, p)
    hi = lo
    while hi < len(suffixes) and suffixes[hi].startswith(p):
        hi += 1
    return lo, hi - lo


@pytest.mark.parametrize("name", list(_texts().keys()))
def test_sa_matches_divsufsort64(name):
    """divsufsort64 orders the suffixes byte-wise, a proper prefix first: exactly what sorting them as bytes gives. The
    reference's own divsufsort64 is compared too where oracle/_ref is built."""
    t = _texts()[name]
    sa = oracle.suffix_array(t)
    order = sorted(range(len(t)), key=lambda i: bytes(t[i:]))
    assert sa.tolist() == order
    if oracle.ref() is not None:
        sa_ref = oracle.ref_divsufsort64(t)
        assert oracle.ref_sufcheck64(t, sa_ref) == 0
        assert np.array_equal(sa, sa_ref)


def test_sa_search_matches_reference():
    """sa_searchb64 over sub-ranges of a sorted suffix array: the bisection over the suffixes themselves, and the
    reference's own function where oracle/_ref is built."""
    t = _texts()["nrun_dup6k"]
    sa = oracle.suffix_array(t)
    R, L = oracle.ref(), oracle.lib()
    rng = np.random.default_rng(5)
    pats = [bytes(t[i:i + l]) for i, l in zip(rng.integers(0, 5900, 300), rng.integers(1, 30, 300))]
    pats += [b"ACGTACGTAC", b"NNNNNNNN", b"TTTTTTTTTTTTTTTT", b"A", b"T", b"$", b"N" * 700, b"N" * 701]
    ranges = [(0, len(sa)), (10, len(sa) - 7), (100, 100), (200, 3000)]
    suffixes = {(l, r): _suffixes(t, sa, l, r) for l, r in ranges}
    for p in pats:
        pa = np.frombuffer(p, dtype=np.uint8)
        for (l, r) in ranges:
            first, c1 = _equal_range(suffixes[l, r], p)
            i2 = C.c_int64()
            c2 = L.oracle_sa_searchb(t.ctypes.data, len(t), pa.ctypes.data, len(pa), sa.ctypes.data, len(sa), C.byref(i2), l, r)
            assert c1 == c2, (p, l, r)
            if c1 > 0 or l < r:
                assert l + first == i2.value, (p, l, r, c1)
            if R is not None:
                i3 = C.c_int64()
                c3 = R.sa_searchb64(t.ctypes.data, len(t), pa.ctypes.data, len(pa), sa.ctypes.data, len(sa), C.byref(i3), l, r)
                assert c3 == c2, (p, l, r)
                if c3 > 0 or l < r:
                    assert i3.value == i2.value, (p, l, r, c3)


def test_lut_matches_reference_sa_searchb64():
    """Searcher::new (searcher.rs:99-143): every non-empty one of the 5^8 keys and a sample of the others against the
    bisection over the suffixes, and against the reference's sa_searchb64 where oracle/_ref is built."""
    t = _texts()["nrun_dup6k"]
    sa = oracle.suffix_array(t)
    keys, lo, hi = oracle.lut(t, sa)
    R = oracle.ref()
    suffixes = _suffixes(t, sa)
    rng = np.random.default_rng(0)
    nonempty = np.nonzero(hi > lo)[0]
    sample = np.concatenate([nonempty, rng.integers(0, oracle.LUT_SIZE, 3000)])
    for e in sample:
        p = int(keys[e]).to_bytes(8, "little")
        first, cnt = _equal_range(suffixes, p)
        assert (first, first + cnt) == (int(lo[e]), int(hi[e]))
        if R is not None:
            pa = np.frombuffer(p, dtype=np.uint8)
            out = C.c_int64()
            cnt = R.sa_searchb64(t.ctypes.data, len(t), pa.ctypes.data, 8, sa.ctypes.data, len(sa), C.byref(out), 0, len(sa))
            assert (out.value, out.value + cnt) == (int(lo[e]), int(hi[e]))
    # invariant of SURVEY §8c: counts over ACGT-only keys of an N-free text sum to n-7
    t2 = _texts()["random4k"]
    sa2 = oracle.suffix_array(t2)
    _, lo2, hi2 = oracle.lut(t2, sa2)
    assert int((hi2 - lo2).sum()) == (len(t2) - 1) - 7


TRIMS = "trim_search_golden.json"


def trim_cases():
    """The trimmed indexes of the literal-search test: the strand, then per trim (a, b) the suffix array of
    strand[a..b]+'$' shifted by a and the patterns looked up in it (8-mers around the cut, random substrings and random
    8-mers). tests/golden/make_trim_golden.py records the reference's answers for exactly these."""
    from tests import cases
    t = oracle.as_strand(cases.stress_text(17, n=30000, n_dups=12))
    t = np.concatenate([t, np.frombuffer(b"$", dtype=np.uint8)]) if t[-1] != ord("$") else t
    rng = np.random.default_rng(1)
    letters = np.frombuffer(b"ATGCN", dtype=np.uint8)
    out = []
    for (a, b) in [(0, len(t) - 1), (1000, 20000), (12345, 12399), (29000, len(t) - 1), (7, 8), (5000, 5009)]:
        sa = np.ascontiguousarray(oracle.trimmed_suffix_array(t, (a, b)), dtype=np.int64)
        pats = [bytes(t[i:i + 8]) for i in range(max(a, b - 40), min(b + 9, len(t) - 8))]          # around the cut
        pats += [bytes(t[i:i + l]) for i, l in zip(rng.integers(a, max(a + 1, b - 1), 400), rng.integers(1, 25, 400))]
        pats += [bytes(rng.choice(letters, size=8)) for _ in range(1500)]
        out.append((a, b, sa, [p for p in pats if b"$" not in p and len(p) > 0]))
    return t, out


def test_literal_sa_search_matches_reference_on_a_trimmed_index():
    """--trim hands sa_searchb64 the suffix array of strand[a..b]+'$' (shifted) together with the WHOLE strand
    (bin/asgart.rs:142-155): near b the array is not sorted for the text it is compared with, and only the literal
    bisection reproduces the reference. The reference's answers are stored in tests/golden/trim_search_golden.json; where
    oracle/_ref is built, its sa_searchb64 is asked as well."""
    import hashlib
    t, trims = trim_cases()
    with open(os.path.join(GOLD, TRIMS)) as f:
        gold = json.load(f)
    assert gold["text_sha256"] == hashlib.sha256(t.tobytes()).hexdigest()
    assert [(g["a"], g["b"]) for g in gold["trims"]] == [(a, b) for a, b, _, _ in trims]
    R = oracle.ref()
    differs = 0
    for (a, b, sa, pats), g in zip(trims, gold["trims"]):
        assert len(sa) == b - a + 1 and sa[0] == b
        assert len(g["first"]) == len(g["count"]) == len(pats)
        for p, first, cnt in zip(pats, g["first"], g["count"]):
            want = (first, cnt)
            pa = np.frombuffer(p, dtype=np.uint8)
            if R is not None:
                out = C.c_int64()
                c = R.sa_searchb64(t.ctypes.data, len(t), pa.ctypes.data, len(pa), sa.ctypes.data, len(sa), C.byref(out), 0, len(sa))
                assert (out.value, c) == want, (a, b, p)
            assert oracle.sa_search_literal(t, p, sa) == want, (a, b, p)
            i2 = C.c_int64()
            c2 = oracle.lib().oracle_sa_searchb(t.ctypes.data, len(t), pa.ctypes.data, len(pa), sa.ctypes.data, len(sa), C.byref(i2), 0, len(sa))
            differs += (i2.value, c2) != want
    assert differs > 0     # the plain lower/upper-bound restatement is NOT enough here: the literal one is needed


def test_effective_trim():
    """prepare_data's --trim validation (bin/asgart.rs:432-463); strand length includes the '$'."""
    assert oracle.effective_trim((5, 100), 50) == (5, 49)
    assert oracle.effective_trim((5, 49), 50) == (5, 49)
    assert oracle.effective_trim((5, 5), 50) is None and oracle.effective_trim((9, 3), 50) is None
    assert oracle.effective_trim((49, 1000), 50) is None          # stop clamps to 49 <= shift
    assert oracle.effective_trim((60, 1000), 50) is None
    assert oracle.effective_trim((0, 1), 50) == (0, 1)


def test_golden_fixtures():
    """Fixtures generated from the reference's C library (tests/golden/make_golden.py); runs without oracle/_ref."""
    with open(os.path.join(GOLD, "sa_golden.json")) as f:
        gold = json.load(f)
    assert gold["generator"].startswith("tests/golden/make_golden.py")
    for name, entry in gold["cases"].items():
        t = np.frombuffer(bytes.fromhex(entry["text_hex"]), dtype=np.uint8)
        sa = oracle.suffix_array(t)
        assert sa.tolist() == entry["sa"], name
        if "lut_nonempty" in entry:
            keys, lo, hi = oracle.lut(t, sa)
            got = {format(int(k), "016x"): [int(a), int(b)] for k, a, b in zip(keys, lo, hi) if b > a}
            assert got == entry["lut_nonempty"], name
