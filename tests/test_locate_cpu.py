"""CPU-side checks of the batched exact-match queries (asgart_b200_ctx_locate): the entry points are exported and refuse
to run without a device, the batch is laid out as the C ABI expects, and the reference answers the GPU tests compare with
(the oracle's sa_search restatement over a batch) agree with a brute force over sorted suffixes and, where oracle/_ref
is built, with the reference's own sa_searchb64."""
import ctypes as C

import numpy as np
import pytest

import asgart_b200 as ab
import oracle
from asgart_b200 import _lib
from tests import cases, kat, locate_ref
from tests.test_oracle_ref import _texts

LOCATE_SYMBOLS = ["asgart_b200_ctx_locate", "asgart_b200_hits_n_patterns", "asgart_b200_hits_first", "asgart_b200_hits_count",
                  "asgart_b200_hits_offsets", "asgart_b200_hits_positions", "asgart_b200_hits_free"]


def test_locate_symbols_exported():
    L = _lib.load()
    for s in LOCATE_SYMBOLS:
        assert s in _lib.SYMBOLS and hasattr(L, s), s
    names = [n for n, _ in _lib.Stats._fields_]
    assert names[-4:] == ["ms_locate", "locate_patterns", "locate_hits", "bytes_locate"]


def test_hits_accessors_accept_null():
    L = _lib.load()
    assert L.asgart_b200_hits_n_patterns(None) == 0
    assert not L.asgart_b200_hits_first(None) and not L.asgart_b200_hits_positions(None)
    L.asgart_b200_hits_free(None)


@pytest.mark.skipif(ab.device_count() > 0, reason="checks the no-device behaviour")
def test_locate_without_device_is_enodevice():
    L = _lib.load()
    buf = np.frombuffer(b"ACGT", dtype=np.uint8)
    off = np.array([0, 4], dtype=np.uint64)
    h = C.c_void_p()
    assert L.asgart_b200_ctx_locate(None, buf.ctypes.data, off.ctypes.data, 1, -1, C.byref(h)) == _lib.ENODEVICE
    assert not h.value


def test_pattern_batch_layout():
    buf, off = ab.api.pattern_batch(["ACG", b"", b"T\x00"])
    assert bytes(buf) == b"ACGT\x00" and off.tolist() == [0, 3, 3, 5] and off.dtype == np.uint64
    buf2, off2 = ab.api.pattern_batch((buf, off))
    assert buf2 is not None and np.array_equal(off2, off)
    b0, o0 = ab.api.pattern_batch([])
    assert len(b0) == 0 and o0.tolist() == [0]
    with pytest.raises(ab.AsgartB200Error) as e:
        ab.api.pattern_batch((buf, np.array([0, 3, 4], dtype=np.uint64)))    # last offset != byte count
    assert e.value.code == _lib.EINVAL


def _special_patterns(t: bytes, rng):
    pats = [b"", b"$", t[-1:], t[-3:], t, t + b"A", t[: len(t) // 2] + b"$", b"\x00", b"\xff", b"B", b"acgt", b"N" * 4]
    for _ in range(60):
        x = int(rng.integers(0, len(t)))
        L = int(rng.integers(1, 24))
        p = t[x:x + L]
        pats.append(p)
        if p:
            at = int(rng.integers(0, len(p)))
            pats.append(p[:at] + locate_ref.FOREIGN[int(rng.integers(0, len(locate_ref.FOREIGN)))] + p[at + 1:])
    return pats


@pytest.mark.parametrize("seed", range(6))
def test_batch_oracle_matches_brute_force_random(seed):
    rng = np.random.default_rng(seed)
    n = int(rng.integers(1, 700))
    alpha = np.frombuffer(b"ACGNT" if seed % 2 else b"ACGT", dtype=np.uint8)
    t = bytes(rng.choice(alpha, n)) + b"$"
    if seed == 3:
        t = bytes(kat.rand_dna(rng, 300)) * 2 + b"$"           # a long repeat: long equal prefixes
    pats = _special_patterns(t, rng) + locate_ref.patterns_for(np.frombuffer(t, dtype=np.uint8), seed, [0, 1, 2, 7, 8, 9, 15, 16, 33, 40])
    sa = locate_ref.sorted_suffixes(t)
    assert np.array_equal(sa, oracle.suffix_array(t))
    got = locate_ref.sa_search_batch(t, pats, sa)
    want = locate_ref.brute_force(t, pats)
    assert np.array_equal(got[1], want[1])
    assert np.array_equal(got[0], want[0])


@pytest.mark.parametrize("name", sorted(_texts()))
def test_batch_oracle_matches_brute_force_and_reference_on_fixed_texts(name):
    t = _texts()[name]
    tb = bytes(t)
    rng = np.random.default_rng(len(tb))
    pats = _special_patterns(tb, rng)
    sa = locate_ref.sorted_suffixes(tb)
    got = locate_ref.sa_search_batch(t, pats, sa)
    want = locate_ref.brute_force(tb, pats)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), name
    R = oracle.ref()
    if R is not None:
        for p, f, c in zip(pats, got[0], got[1]):
            pa = np.frombuffer(p, dtype=np.uint8) if p else np.zeros(1, dtype=np.uint8)
            out = C.c_int64()
            cnt = R.sa_searchb64(t.ctypes.data, len(t), pa.ctypes.data, len(p), sa.ctypes.data, len(sa), C.byref(out), 0, len(sa))
            assert (int(cnt), int(out.value) if cnt or p else 0) == (int(c), int(f) if c or p else 0), (name, p)


def test_batch_oracle_on_stress_text_lengths():
    """Every length 0-80 and a few long ones, hits and misses, on a text with N runs and repeats."""
    t = np.concatenate([cases.stress_text(5, n=12000, n_dups=2), np.frombuffer(b"$", dtype=np.uint8)])
    pats = locate_ref.patterns_for(t, 9, list(range(0, 81)) + [200, 1000, 4000], per_length=2)
    sa = locate_ref.sorted_suffixes(t)
    got = locate_ref.sa_search_batch(t, pats, sa)
    want = locate_ref.brute_force(t, pats)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
