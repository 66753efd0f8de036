"""Batched exact-match queries against the resident index (Context.locate / asgart_b200_ctx_locate): (first, count) bit for
bit equal to the oracle's sa_search restatement (oracle.sa_search_literal) over the CPU suffix array, positions equal to
the slice of the index, on full and --trim indexes (SURVEY Q9), at genome scale against the probe kernel."""
import numpy as np
import pytest

import asgart_b200 as ab
import oracle
from asgart_b200 import _lib
from tests import cases, locate_ref

pytestmark = pytest.mark.gpu

LENGTHS = list(range(0, 81)) + [200, 1000, 5000, 65536]


def _strand(seed, n, **kw):
    return np.concatenate([cases.stress_text(seed, n=n, **kw), np.frombuffer(b"$", dtype=np.uint8)])


def _check_full(ctx, strand, pats, sa):
    first, count = ctx.sa_search(pats)
    want_f, want_c = locate_ref.sa_search_batch(strand, pats, sa)
    bad = np.nonzero((first != want_f) | (count != want_c))[0]
    assert len(bad) == 0, [(pats[i][:40], int(first[i]), int(count[i]), int(want_f[i]), int(want_c[i])) for i in bad[:5]]
    return first, count


@pytest.mark.parametrize("bits", [32, 64])
def test_full_index_matches_oracle(bits):
    small = _strand(31, 40000, n_dups=6)
    big = _strand(32, 1_500_000, n_dups=30)
    with ab.Context(0) as ctx:
        ctx.set_index_bits(bits)
        for strand, per in ((small, 6), (big, 4)):
            ctx.load_strand(strand)
            ctx.build_index()
            sa = ctx.download_sa()
            assert np.array_equal(sa, oracle.best_suffix_array(strand))
            pats = locate_ref.patterns_for(strand, bits + len(strand), LENGTHS, per_length=per)
            first, count = _check_full(ctx, strand, pats, sa)
            assert (count > 0).sum() > len(pats) // 8 and (count == 0).sum() > len(pats) // 8
        # an uploaded index (no deep table, LUT from the array) gives the same answers
        ctx.upload_sa(sa)
        _check_full(ctx, big, pats, sa)
        st = ctx.stats()
        assert st["locate_patterns"] >= 3 * len(pats) and st["bytes_locate"] > 0 and st["ms_locate"] > 0


@pytest.mark.parametrize("bits", [32, 64])
def test_trimmed_index_matches_literal_search(bits):
    """The five trims of test_gpu_trim: the oracle's step-for-step search on the trimmed array against the whole strand."""
    strand = np.concatenate([np.frombuffer(cases.stress_text(17, n=30000, n_dups=12), dtype=np.uint8),
                             np.frombuffer(b"$", dtype=np.uint8)])
    t = bytes(strand)
    letters = np.frombuffer(b"ATGCN", dtype=np.uint8)
    differs = 0
    with ab.Context(0) as ctx:
        ctx.set_index_bits(bits)
        ctx.load_strand(strand)
        for trim in [(1000, 20000), (12345, 12399), (29000, 10 ** 9), (7, 8), (0, 30000)]:
            eff = oracle.effective_trim(trim, len(strand))
            ctx.build_index(trim=trim)
            sa = oracle.trimmed_suffix_array(strand, eff)
            pats = locate_ref.patterns_for(strand, eff[0] + bits, list(range(0, 41)) + [64, 100, 1000], per_length=2)
            for x in range(max(eff[0], eff[1] - 60), min(eff[1] + 10, len(t))):         # around the cut, where Q9 bites
                pats += [t[x:x + L] for L in (3, 8, 12, 20, 40)]
            rng = np.random.default_rng(eff[0])
            pats += [bytes(rng.choice(letters, int(L))) for L in rng.integers(6, 12, 1500)]   # random short ones: misses
            first, count = ctx.sa_search(pats)
            want_f, want_c = locate_ref.sa_search_batch(strand, pats, sa)
            assert np.array_equal(count, want_c) and np.array_equal(first, want_f), trim
            L = oracle.lib()
            for p, f, c in zip(pats, first, count):     # how often a plain lower/upper bound would have answered otherwise
                pa = np.frombuffer(p, dtype=np.uint8) if p else np.zeros(1, dtype=np.uint8)
                i2 = oracle.C.c_int64()
                c2 = L.oracle_sa_searchb(strand.ctypes.data, len(strand), pa.ctypes.data, len(p), sa.ctypes.data, len(sa),
                                         oracle.C.byref(i2), 0, len(sa))
                differs += (int(c2), int(i2.value)) != (int(c), int(f))
            hits = ctx.locate(pats, max_hits=3)
            for i in range(0, len(pats), 7):
                assert np.array_equal(hits.positions_of(i), sa[first[i]:first[i] + min(count[i], 3)])
    assert differs > 0, "no pattern shows the trimmed array's disorder: the literal path is not exercised"


def test_locate_positions_caps_and_batch_independence():
    strand = _strand(41, 200_000, n_dups=20)
    pats = locate_ref.patterns_for(strand, 5, list(range(0, 41)) + [100, 1000], per_length=6)
    pats += [b"A", b"AC", b"N", b"NNNN", b"ACGT"]          # many hits
    with ab.Context(0) as ctx:
        ctx.load_strand(strand)
        ctx.build_index()
        sa = ctx.download_sa()
        full = ctx.locate(pats)
        for cap in (-1, 0, 1, 7):
            h = ctx.locate(pats, max_hits=None if cap < 0 else cap)
            assert np.array_equal(h.count, full.count) and np.array_equal(h.first, full.first)
            for i in range(len(pats)):
                k = int(h.count[i]) if cap < 0 else min(int(h.count[i]), cap)
                assert int(h.offsets[i + 1] - h.offsets[i]) == k
                assert np.array_equal(h.positions_of(i), sa[h.first[i]:h.first[i] + k]), (cap, pats[i][:20])
        assert int(full.offsets[-1]) == int(full.count.sum())
        assert ctx.stats()["locate_hits"] >= int(full.count.sum())
        # another order and another split of the batch: the same answer per pattern
        perm = np.random.default_rng(1).permutation(len(pats))
        a = ctx.locate([pats[i] for i in perm[:len(perm) // 3]], max_hits=7)
        b = ctx.locate([pats[i] for i in perm[len(perm) // 3:]], max_hits=7)
        ref7 = ctx.locate(pats, max_hits=7)
        for part, idx in ((a, perm[:len(perm) // 3]), (b, perm[len(perm) // 3:])):
            assert np.array_equal(part.first, ref7.first[idx]) and np.array_equal(part.count, ref7.count[idx])
            for j, i in enumerate(idx):
                assert np.array_equal(part.positions_of(j), ref7.positions_of(i))
        # the (bytes, offsets) form
        buf, off = ab.api.pattern_batch(pats)
        h2 = ctx.locate((buf, off), max_hits=7)
        assert np.array_equal(h2.positions, ref7.positions) and np.array_equal(h2.offsets, ref7.offsets)


def test_genome_scale_c3_against_probe_ranges():
    """C3 at full size (249 Mbp), no CPU suffix array: counts of 10^5 probe k-mers equal the probe kernel's equal ranges,
    every reported position starts with its pattern, and `first` is the insertion point (checked on a sample)."""
    g, fr = ab.synth_genome(3)
    prep = ab.Prepared.from_memory(ab.normalise(g, False), fr, "synthC3.fa")
    strand = np.array(prep.strand)
    st = ab.RunSettings()
    k, s = st.probe_size, st.probe_size // 2
    n_probes = 100_000
    c0, clen = prep.chunks[0]
    assert clen > (n_probes + 2) * s
    with ab.Context(0) as ctx:
        ctx.load_strand(strand)
        ctx.build_index()
        lo, hi = ctx.probe_ranges(prep.chunks[0], st, n_probes)
        starts = c0 + (np.arange(n_probes, dtype=np.int64) + 1) * s
        buf = strand[(starts[:, None] + np.arange(k)[None, :]).reshape(-1)]
        off = np.arange(n_probes + 1, dtype=np.uint64) * k
        hits = ctx.locate((buf, off), max_hits=64)
        assert np.array_equal(hits.count, hi - lo)
        assert np.array_equal(hits.first[hits.count > 0], lo[hits.count > 0])
        pats = buf.reshape(n_probes, k)
        reps = np.repeat(np.arange(n_probes), np.diff(hits.offsets.astype(np.int64)))
        got = strand[(hits.positions[:, None] + np.arange(k)[None, :])]
        assert np.array_equal(got, pats[reps])
        # insertion points: random misses and hits; SA[first - 1] < P <= SA[first] as bytes
        rng = np.random.default_rng(7)
        sample = [bytes(rng.choice(list(b"ACGT"), int(L)).astype(np.uint8)) for L in rng.integers(8, 40, 300)]
        sample += [bytes(pats[i]) for i in rng.integers(0, n_probes, 100)]
        f, c = ctx.sa_search(sample)
        sa = ctx.download_sa()
        t = strand
        for p, fi, ci in zip(sample, f, c):
            if fi > 0:
                x = int(sa[fi - 1])
                assert bytes(t[x:x + len(p)]) < p
            if fi < len(sa):
                x = int(sa[fi])
                assert bytes(t[x:x + len(p)]) >= p
            if ci:
                x = int(sa[fi + ci - 1])
                assert bytes(t[x:x + len(p)]) == p


def test_edge_cases_and_errors():
    strand = _strand(51, 20000, n_dups=3)
    with ab.Context(0) as ctx:
        with pytest.raises(ab.AsgartB200Error) as e:
            ctx.locate([b"ACGT"])
        assert e.value.code == _lib.ESTATE
        ctx.load_strand(strand)
        with pytest.raises(ab.AsgartB200Error) as e:
            ctx.locate([b"ACGT"])
        assert e.value.code == _lib.ESTATE
        ctx.build_index()
        h = ctx.locate([])
        assert len(h.first) == 0 and h.offsets.tolist() == [0] and len(h.positions) == 0
        buf = np.frombuffer(b"ACGTAC", dtype=np.uint8).copy()
        with pytest.raises(ab.AsgartB200Error) as e:
            ctx.locate((buf, np.array([0, 4, 2, 6], dtype=np.uint64)))      # not non-decreasing
        assert e.value.code == _lib.EINVAL
        with pytest.raises(ab.AsgartB200Error) as e:
            ctx.locate((buf, np.array([0, 4, 5], dtype=np.uint64)))         # last offset != byte count
        assert e.value.code == _lib.EINVAL
        f, c = ctx.sa_search([b""])
        assert (int(f[0]), int(c[0])) == (0, len(strand))


def test_ingested_context_equals_loaded_one():
    rng = np.random.default_rng(3)
    seq = cases.stress_text(61, n=50000, n_dups=5).tobytes().decode()
    fasta = ">chr1 x\n" + "\n".join(seq[i:i + 60] for i in range(0, 30000, 60)) + "\n>chr2\n" + seq[30000:] + "\n"
    with ab.Context(0) as a, ab.Context(0) as b:
        a.ingest([fasta.encode()], names=["m.fa"])
        a.build_index()
        strand = a.download_strand()
        b.load_strand(strand)
        b.build_index()
        pats = locate_ref.patterns_for(strand, 11, list(range(0, 50)) + [300], per_length=4)
        ha, hb = a.locate(pats), b.locate(pats)
        for f in ("first", "count", "offsets", "positions"):
            assert np.array_equal(getattr(ha, f), getattr(hb, f)), f
        assert rng is not None
