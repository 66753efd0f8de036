"""Parity tests proper: the CUDA path (through the C ABI) against the CPU oracle on the same seeded inputs.
Bit-exact bar: suffix array, LUT, probe ranges, proto-duplicons, families after post-steps, JSON text."""
import json
import os

import numpy as np
import pytest

import asgart_b200 as ab
import oracle
from asgart_b200 import _lib
from tests import cases, kat
from tests.test_oracle_ref import _texts

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _osettings(st: ab.RunSettings):
    return oracle.make_settings(probe_size=st.probe_size, gap_size=st.gap_size, min_length=st.min_duplication_length,
                                max_cardinality=st.max_cardinality, reverse=st.reverse, complement=st.complement,
                                skip_masked=st.skip_masked)


def _rs(kw):
    kw = dict(kw)
    if "min_length" in kw:
        kw["min_duplication_length"] = kw.pop("min_length")
    return ab.RunSettings(**kw)


# ------------------------------------------------------------------------------------------------ suffix array
@pytest.mark.parametrize("bits", [32, 64])
@pytest.mark.parametrize("name", list(_texts().keys()))
def test_sa_small_texts(name, bits):
    t = _texts()[name]
    want = oracle.best_suffix_array(t)
    got = ab.r_divsufsort(t, device=0, index_bits=bits)
    assert np.array_equal(got, want)


@pytest.mark.parametrize("bits", [32, 64])
def test_sa_golden_fixtures(bits):
    """Fixtures made by the reference's own divsufsort64 (tests/golden/make_golden.py)."""
    gold = json.load(open(os.path.join(GOLD, "sa_golden.json")))
    for name, entry in gold["cases"].items():
        t = np.frombuffer(bytes.fromhex(entry["text_hex"]), dtype=np.uint8)
        assert ab.r_divsufsort(t, device=0, index_bits=bits).tolist() == entry["sa"], name


def test_sa_edge_cases():
    assert ab.r_divsufsort(b"").tolist() == []
    assert ab.r_divsufsort(b"A").tolist() == [0]
    assert ab.r_divsufsort(b"AA").tolist() == [1, 0]
    assert ab.r_divsufsort(b"$").tolist() == [0]
    a = np.zeros(70000, dtype=np.uint8)              # one symbol, every suffix ties until the end: worst case for doubling
    assert np.array_equal(ab.r_divsufsort(a), np.arange(70000)[::-1])
    b = np.tile(np.frombuffer(b"ACGTTGCA", dtype=np.uint8), 9000)   # period-8 text
    assert np.array_equal(ab.r_divsufsort(b), oracle.best_suffix_array(b))


@pytest.mark.parametrize("bits", [32, 64])
def test_sa_medium_with_repeats(bits):
    n = 1_500_000 if bits == 32 else 400_000
    text = cases.stress_text(77, n=n, n_dups=60)
    text[n // 3: n // 3 + 200_000 // (1 if bits == 32 else 4)] = ord("N")       # a long N-run: deep LCPs
    strand = np.concatenate([text, np.frombuffer(b"$", dtype=np.uint8)])
    got = ab.r_divsufsort(strand, device=0, index_bits=bits)
    if oracle.ref() is not None:
        assert oracle.ref_sufcheck64(strand, got) == 0
        assert np.array_equal(got, oracle.ref_divsufsort64(strand))
    else:
        assert np.array_equal(got, oracle.suffix_array(strand))
    assert got[0] == len(strand) - 1


@pytest.mark.parametrize("bits,scale", [(32, 3_000_000), (64, 600_000)])
def test_sa_soft_masked_genome(bits, scale):
    """C2-shaped input with -S: thousands of N-runs of assorted lengths (the run round and the large-group path of the
    doubling rounds), telomeric runs touching both ends of the strand, planted exact repeats."""
    g, fr = ab.synth_genome(2, scale_n=scale)
    strand = np.concatenate([ab.normalise(g, True), np.frombuffer(b"$", dtype=np.uint8)])
    got = ab.r_divsufsort(strand, device=0, index_bits=bits)
    assert np.array_equal(got, oracle.best_suffix_array(strand))
    # same genome without masking (upper-cased): only the long N-runs remain
    strand2 = np.concatenate([ab.normalise(g, False), np.frombuffer(b"$", dtype=np.uint8)])
    assert np.array_equal(ab.r_divsufsort(strand2, device=0, index_bits=bits), oracle.best_suffix_array(strand2))


def test_sa_runs_of_every_symbol():
    """Runs longer than the initial key of several symbols, followed by smaller and by larger symbols, and a run that
    reaches the end of the text (no terminator)."""
    rng = np.random.default_rng(9)
    parts = []
    for _ in range(300):
        x = b"ACGNT"[int(rng.integers(0, 5))]
        parts.append(np.full(int(rng.integers(1, 120)), x, dtype=np.uint8))
        parts.append(kat.rand_dna(rng, int(rng.integers(1, 40))))
    t = np.concatenate(parts + [np.full(77, ord("T"), dtype=np.uint8)])
    for bits in (32, 64):
        assert np.array_equal(ab.r_divsufsort(t, device=0, index_bits=bits), oracle.best_suffix_array(t))
    t2 = np.concatenate([t, np.frombuffer(b"$", dtype=np.uint8)])
    assert np.array_equal(ab.r_divsufsort(t2), oracle.best_suffix_array(t2))


# ------------------------------------------------------------------------------------------------ LUT + probes
def _slot_of_key(k):
    digit = {ord("A"): 0, ord("C"): 1, ord("G"): 2, ord("N"): 3, ord("T"): 4}
    s = 0
    for ch in int(k).to_bytes(8, "little"):
        s = s * 5 + digit[ch]
    return s


@pytest.mark.parametrize("source", ["upload", "build"])
@pytest.mark.parametrize("bits", [32, 64])
def test_lut_and_probe_ranges(bits, source):
    """upload: LUT from the finished SA, literal search only. build: LUT + deep table from the sorted initial keys of the
    SA build, probes go through the deep-table path and the deferred literal path."""
    text = cases.stress_text(5, n=50000)
    strand = np.concatenate([text, np.frombuffer(b"$", dtype=np.uint8)])
    sa = oracle.best_suffix_array(strand)
    with ab.Context(0) as ctx:
        ctx.set_index_bits(bits)
        ctx.load_strand(strand)
        if source == "upload":
            ctx.upload_sa(sa)
        else:
            ctx.build_index()
            assert np.array_equal(ctx.download_sa(), sa)
        assert ctx.check_sa() == 0
        lo, hi = ctx.download_lut()
        keys, olo, ohi = oracle.lut(strand, sa)
        slots = np.array([_slot_of_key(k) for k in keys])
        ne = ohi > olo
        assert np.array_equal(lo[slots[ne]], olo[ne]) and np.array_equal(hi[slots[ne]], ohi[ne])
        assert np.array_equal(lo[slots[~ne]], hi[slots[~ne]])
        # probe equal ranges == Searcher::search (unfiltered), for all four needle transforms and k = 20 / 32 / 40
        osr = oracle.OracleSearcher(strand, sa)
        comp = kat.complement
        for kw in (dict(), dict(reverse=True, complement=True), dict(reverse=True), dict(complement=True),
                   dict(probe_size=32, reverse=True, complement=True), dict(probe_size=40)):
            st = ab.RunSettings(**kw)
            chunk = (1000, 30000)
            k, s = st.probe_size, st.probe_size // 2
            nprobes = -(-(chunk[1] - k - s) // s)
            glo, ghi = ctx.probe_ranges(chunk, st, nprobes)
            needle = text[chunk[0]:chunk[0] + chunk[1]]
            if st.complement:
                needle = comp(needle)
            if st.reverse:
                needle = needle[::-1]
            for p in list(range(0, nprobes, 37)) + [nprobes - 1]:
                i = (p + 1) * s
                want = osr.search(needle[i:i + k].tobytes())
                assert ghi[p] - glo[p] == len(want), (kw, p)
                assert np.array_equal(sa[glo[p]:ghi[p]], want), (kw, p)


def test_q6_forced_less_with_deep_table():
    """Quirk Q6 on the device: the last k-1 suffixes compare Less whatever they hold (src/searcher.rs:165-166). The tail of
    this text shares its 8-mers with most probes, so most 8-mer buckets are flagged and must take the literal bisection,
    the others take the deep table; ranges and families must equal the oracle's either way."""
    rng = np.random.default_rng(3)
    unit = kat.rand_dna(rng, 11)
    text = np.concatenate([kat.rand_dna(rng, 3000), np.tile(unit, 400), kat.rand_dna(rng, 9)])
    strand = np.concatenate([text, np.frombuffer(b"$", dtype=np.uint8)])
    sa = oracle.best_suffix_array(strand)
    osr = oracle.OracleSearcher(strand, sa)
    with ab.Context(0) as ctx:
        ctx.load_strand(strand)
        ctx.build_index()
        assert np.array_equal(ctx.download_sa(), sa)
        for kw in (dict(probe_size=20, gap_size=100, min_length=200, max_cardinality=100000),
                   dict(probe_size=20, gap_size=100, min_length=200, max_cardinality=100000, reverse=True, complement=True),
                   dict(probe_size=12, gap_size=50, min_length=200, max_cardinality=100000)):
            st = _rs(kw)
            want = oracle.search(strand, sa, [(0, len(text))], _osettings(st), oracle.POST_ALL, threads=1)
            got = ctx.search([(0, len(text))], st, ab.POST_ALL)
            assert got.as_lists() == want.families.as_lists(), kw
            if not st.reverse:
                k, s = st.probe_size, st.probe_size // 2
                nprobes = -(-(len(text) - k - s) // s)
                glo, ghi = ctx.probe_ranges((0, len(text)), st, nprobes)
                for p in range(nprobes):
                    i = (p + 1) * s
                    w = osr.search(text[i:i + k].tobytes())
                    assert ghi[p] - glo[p] == len(w) and np.array_equal(sa[glo[p]:ghi[p]], w), (kw, p)


def test_check_sa_detects_corruption():
    text = cases.stress_text(21, n=30000)
    strand = np.concatenate([text, np.frombuffer(b"$", dtype=np.uint8)])
    sa = oracle.best_suffix_array(strand)
    with ab.Context(0) as ctx:
        ctx.load_strand(strand)
        ctx.upload_sa(sa)
        assert ctx.check_sa() == 0
        bad = sa.copy()
        bad[[100, 101]] = bad[[101, 100]]          # one adjacent swap: order violation
        ctx.upload_sa(bad)
        assert ctx.check_sa() > 0
        dup = sa.copy()
        dup[500] = dup[501]                        # not a permutation
        ctx.upload_sa(dup)
        assert ctx.check_sa() > 0


# ------------------------------------------------------------------------------------------------ search + automaton
@pytest.mark.parametrize("case", kat.cases(), ids=lambda c: c[0])
def test_search_kat(case):
    name, text, chunks, kw, expected = case
    strand = np.concatenate([text, np.frombuffer(b"$", dtype=np.uint8)])
    with ab.Context(0) as ctx:
        ctx.load_strand(strand)
        ctx.build_index()
        got = ctx.search(chunks, _rs(kw), ab.POST_ALL).as_lists()
    if name == "KAT-3COPIES":
        assert [sorted(f) for f in got] == [sorted(f) for f in expected]
    else:
        assert got == expected


@pytest.mark.parametrize("bits", [32, 64])
@pytest.mark.parametrize("seed", [11, 12, 13])
def test_search_stress_all_settings(seed, bits):
    text = cases.stress_text(seed)
    prep = ab.Prepared.from_memory(text, [("a", 0, 25000), ("b", 25000, len(text) - 25000)])
    strand = np.array(prep.strand)
    sa = oracle.best_suffix_array(strand)
    with ab.Context(0) as ctx:
        ctx.set_index_bits(bits)
        ctx.load_strand(strand)
        ctx.build_index()
        assert np.array_equal(ctx.download_sa(), sa)
        for label, kw in cases.settings_grid():
            st = _rs(kw)
            ctx.reset_stats()
            raw = ctx.search(prep.chunks, st, 0)
            want_raw = oracle.search(strand, sa, prep.chunks, _osettings(st), 0, threads=2)
            assert raw.as_lists() == want_raw.families.as_lists(), label
            s = ctx.stats()
            c = want_raw.counters
            assert (s["n_probes"], s["n_searched"], s["n_skipped_n"], s["n_skipped_card"], s["n_matches"], s["bytes_probe"]) == \
                   (c["probes"], c["searched"], c["skipped_n"], c["skipped_card"], c["matches"], c["alg_bytes"]), label
            full = ctx.search(prep.chunks, st, ab.POST_ALL)
            want = oracle.search(strand, sa, prep.chunks, _osettings(st), oracle.POST_ALL, threads=2)
            assert full.as_lists() == want.families.as_lists(), label
            # each post-step on its own, fed with the oracle's raw families
            for mask in (ab.POST_FILTER_NS, ab.POST_REORDER, ab.POST_REDUCE_OVERLAP, ab.POST_SORT, ab.POST_FILTER_NS | ab.POST_SORT):
                assert ctx.post_steps(raw, mask).as_lists() == oracle.post_steps(want_raw.families, strand, mask).as_lists(), (label, mask)


def test_post_steps_unit_cases():
    t = np.full(3001, ord("A"), dtype=np.uint8); t[-1] = ord("$")
    t[0:200] = ord("N"); t[1200:1401] = ord("N")
    with ab.Context(0) as ctx:
        ctx.load_strand(t)
        keep = ctx.post_steps(ab.families_from_lists([[(0, 2000, 1000, 1000)]]), ab.POST_FILTER_NS)
        drop = ctx.post_steps(ab.families_from_lists([[(0, 1100, 1000, 1000)]]), ab.POST_FILTER_NS)
        assert keep.n_families == 1 and drop.n_families == 0            # 200/1000 <= 0.2 kept, 201/1000 dropped (f32)
        merged = ctx.post_steps(ab.families_from_lists([[(100, 2000, 500, 600), (400, 2300, 500, 450), (150, 2050, 100, 100)]]),
                                ab.POST_REDUCE_OVERLAP)
        # merge() with its mixed-up lengths (Q5): lsize = max(400+500, 100+600) - 100, rsize = max(2300+500, 2000+600) - 2000
        assert [x[:4] for x in merged.as_lists()[0]] == [(100, 2000, 800, 800)]
        ro = ctx.post_steps(ab.families_from_lists([[(900, 100, 10, 20)]]), ab.POST_REORDER)
        assert [x[:4] for x in ro.as_lists()[0]] == [(100, 900, 10, 20)]          # positions only (Q4)
        fams = [[(50, 9, 1, 1), (10, 8, 1, 1), (50, 7, 1, 1), (10, 6, 1, 1)], [], [(3, 3, 3, 3)]]
        srt = ctx.post_steps(ab.families_from_lists(fams), ab.POST_SORT)
        assert [[x[:2] for x in f] for f in srt.as_lists()] == [[(10, 8), (10, 6), (50, 9), (50, 7)], [(3, 3)]]   # stable


def test_ragged_and_empty_inputs():
    text = cases.stress_text(3, n=20000)
    strand = np.concatenate([text, np.frombuffer(b"$", dtype=np.uint8)])
    sa = oracle.best_suffix_array(strand)
    with ab.Context(0) as ctx:
        ctx.load_strand(strand)
        ctx.build_index()
        st = ab.RunSettings(min_duplication_length=300)
        so = _osettings(st)
        for chunks in ([], [(0, 10)], [(0, 299)], [(0, 300)], [(5, 31), (100, 5000), (5100, 0), (6000, 14000)], [(19990, 10)], [(0, 20000)]):
            got = ctx.search(chunks, st, ab.POST_ALL).as_lists()
            want = oracle.search(strand, sa, chunks, so, oracle.POST_ALL).families.as_lists()
            assert got == want, chunks
        with pytest.raises(ab.AsgartB200Error):
            ctx.search([(19000, 2000)], st)                                   # chunk outside the strand
        with pytest.raises(ab.AsgartB200Error):
            ctx.search([(0, 20000)], ab.RunSettings(probe_size=7))            # reference needs k >= 8
        with pytest.raises(ab.AsgartB200Error):
            ctx.load_strand(np.frombuffer(b"ACGTXACGT$", dtype=np.uint8))     # not normalised
        with pytest.raises(ab.AsgartB200Error):
            ctx.load_strand(np.frombuffer(b"ACGTACGT", dtype=np.uint8))       # no '$'


@pytest.mark.parametrize("n_shards", [1, 2, 3, 8])
def test_sharded_search_equals_single(n_shards):
    """Probe-range sharding (what N GPUs do) gives the same families for every shard count."""
    text = cases.stress_text(12)
    prep = ab.Prepared.from_memory(text, [("a", 0, 25000), ("b", 25000, len(text) - 25000)])
    strand = np.array(prep.strand)
    with ab.Context(0) as ctx:
        ctx.load_strand(strand)
        ctx.build_index()
        for label, kw in cases.settings_grid()[:6]:
            st = _rs(kw)
            single = ctx.search(prep.chunks, st, ab.POST_ALL).as_lists()
            parts = [ctx.search_shard(prep.chunks, st, r, n_shards) for r in range(n_shards)]
            assert ctx.finish(prep.chunks, st, parts, ab.POST_ALL).as_lists() == single, label
            # device-resident form (what the NCCL path exchanges): blobs cloned to torch memory, as an all-gather leaves them
            import torch
            from asgart_b200.dist import _DevMem
            blobs, metas = [], []
            for r in range(n_shards):
                ptr, nbytes, meta = ctx.search_shard_dev(prep.chunks, st, r, n_shards)
                blobs.append(torch.as_tensor(_DevMem(ptr, nbytes), device="cuda:0").clone() if nbytes else
                             torch.zeros(8, dtype=torch.uint8, device="cuda:0"))
                metas.append(meta)
            torch.cuda.synchronize()
            got = ctx.finish_dev(prep.chunks, st, [b.data_ptr() for b in blobs], np.stack(metas), ab.POST_ALL)
            assert got.as_lists() == single, label


def test_run_files_json_identical_to_oracle(tmp_path):
    g, fr = ab.synth_genome(2, scale_n=800_000)
    fa = tmp_path / "synthY.fa"
    with open(fa, "w") as f:
        f.write(">synthY synthetic chrY-shaped\n")
        s = g.tobytes().decode()
        for i in range(0, len(s), 60):
            f.write(s[i:i + 60] + "\n")
    for kw in (dict(), dict(reverse=True, complement=True, skip_masked=True), dict(skip_masked=True)):
        st = ab.RunSettings(**kw)
        js = ab.search_duplications([str(fa)], st)
        want = oracle.run_files([str(fa)], _osettings(st), threads=2)
        assert js == want
        assert json.loads(js)["settings"]["max_gap_size"] == 120
    assert len(json.loads(ab.search_duplications([str(fa)], ab.RunSettings()))["families"]) > 0


# ------------------------------------------------------------------------------------------------ sharded index build
def _group_build(strand, world, bits=0):
    ctxs = [ab.Context(0) for _ in range(world)]
    for c in ctxs:
        if bits:
            c.set_index_bits(bits)
        c.load_strand(strand)
    ab.build_index_group(ctxs)
    return ctxs


@pytest.mark.parametrize("world", [2, 3, 4, 8])
@pytest.mark.parametrize("bits", [32, 64])
def test_sharded_index_equals_single(world, bits):
    """The sharded build (members = host threads, all on this GPU: key ranges, block-cyclic rank array in the members'
    slices, collectives at the phase boundaries) gives every member the suffix array, LUT and families of a lone build."""
    text = cases.stress_text(7 + world, n=300_000, n_dups=40)
    prep = ab.Prepared.from_memory(text, [("a", 0, len(text))], "g.fa")
    strand = np.array(prep.strand)
    sa_ref = oracle.best_suffix_array(strand)
    st = ab.RunSettings(min_duplication_length=500, reverse=True, complement=True)
    with ab.Context(0) as one:
        one.set_index_bits(bits)
        one.load_strand(strand)
        one.build_index()
        lut_ref = one.download_lut()
        fam_ref = one.search(prep.chunks, st, ab.POST_ALL).as_lists()
    ctxs = _group_build(strand, world, bits)
    try:
        for c in ctxs:
            assert np.array_equal(c.download_sa(), sa_ref)
            lo, hi = c.download_lut()
            ne = lut_ref[1] > lut_ref[0]
            assert np.array_equal((hi > lo), ne)
            assert np.array_equal(lo[ne], lut_ref[0][ne]) and np.array_equal(hi[ne], lut_ref[1][ne])
            assert c.check_sa() == 0
        assert ctxs[-1].search(prep.chunks, st, ab.POST_ALL).as_lists() == fam_ref
        assert len(fam_ref) > 0
    finally:
        for c in ctxs:
            c.close()


@pytest.mark.parametrize("name", ["runs", "tiny", "masked"])
def test_sharded_index_edge_texts(name):
    """Texts where the key ranges are lopsided: long single-symbol runs (one bin holds most suffixes, members with empty
    pieces), a text shorter than the member count's blocks, a soft-masked genome (15 % N)."""
    if name == "runs":
        rng = np.random.default_rng(5)
        parts = [b"A" * 40_000, bytes(rng.choice(list(b"ACGT"), 30_000).astype(np.uint8)), b"N" * 70_000, b"T" * 9_000,
                 bytes(rng.choice(list(b"ACGT"), 20_000).astype(np.uint8)), b"A" * 25_000]
        text = np.frombuffer(b"".join(parts), dtype=np.uint8)
    elif name == "tiny":
        text = np.frombuffer(b"ACGTACGTTTGACCANNNACGTACGTAC", dtype=np.uint8)
    else:
        g, fr = ab.synth_genome(2, scale_n=400_000)
        text = ab.normalise(g, True)
    strand = np.concatenate([text, np.frombuffer(b"$", dtype=np.uint8)])
    sa_ref = oracle.best_suffix_array(strand)
    for world in (2, 5):
        ctxs = _group_build(strand, world)
        try:
            for c in ctxs:
                assert np.array_equal(c.download_sa(), sa_ref)
        finally:
            for c in ctxs:
                c.close()


def test_sharded_index_full_size_c2():
    """BASELINE configs[1] at full size through a 4-member group: on-device sufcheck and the single-build families."""
    st, prep = _full_config(2)
    strand = np.array(prep.strand)
    with ab.Context(0) as one:
        one.load_strand(strand)
        one.build_index()
        fam_ref = one.search(prep.chunks, st, ab.POST_ALL).as_lists()
        lut_ref = one.download_lut()
    ctxs = _group_build(strand, 4)
    try:
        for c in (ctxs[0], ctxs[3]):
            assert c.check_sa() == 0
            lo, hi = c.download_lut()
            ne = lut_ref[1] > lut_ref[0]
            assert np.array_equal(lo[ne], lut_ref[0][ne]) and np.array_equal(hi[ne], lut_ref[1][ne])
        assert ctxs[2].search(prep.chunks, st, ab.POST_ALL).as_lists() == fam_ref
    finally:
        for c in ctxs:
            c.close()


# ------------------------------------------------------------------------------------------------ full-size configs
def _full_config(config):
    flags = {1: dict(), 2: dict(reverse=True, complement=True, skip_masked=True),
             3: dict(reverse=True, complement=True, max_cardinality=500), 4: dict(reverse=True, complement=True)}[config]
    st = ab.RunSettings(**flags)
    g, fr = ab.synth_genome(config, threads=os.cpu_count() or 8)
    prep = ab.Prepared.from_memory(ab.normalise(g, st.skip_masked), fr, f"synthC{config}.fa")
    return st, prep


def _index_properties(ctx, prep):
    """Size-independent properties of the index: on-device sufcheck, SA[0] = n, LUT buckets disjoint and inside [0, n]."""
    assert ctx.check_sa() == 0
    lo, hi = ctx.download_lut()
    ne = hi > lo
    assert (lo[ne] >= 1).all() and (hi[ne] <= len(prep.strand)).all()
    order = np.argsort(lo[ne], kind="stable")
    assert (hi[ne][order][:-1] <= lo[ne][order][1:]).all()      # slots are in suffix order and do not overlap
    return int((hi[ne] - lo[ne]).sum())


def test_full_size_c2_equals_oracle():
    """BASELINE configs[1] at full size (57 Mbp, -RC -S): families identical to the CPU oracle's (reference libdivsufsort
    SA when oracle/_ref is present), plus the index properties."""
    st, prep = _full_config(2)
    strand = np.array(prep.strand)
    with ab.Context(0) as ctx:
        ctx.load_strand(strand)
        ctx.build_index()
        in_lut = _index_properties(ctx, prep)
        assert in_lut <= len(strand) - 8
        got = ctx.search(prep.chunks, st, ab.POST_ALL)
        sa = oracle.best_suffix_array(strand)
        assert np.array_equal(ctx.download_sa(), sa)
        want = oracle.search(strand, sa, prep.chunks, _osettings(st), oracle.POST_ALL, threads=os.cpu_count() or 8)
        assert got.as_lists() == want.families.as_lists()
        assert got.n_families > 50
        # the direct pass over the same index finds the direct plants and none of the RC ones
        st_d = ab.RunSettings(skip_masked=True)
        got_d = ctx.search(prep.chunks, st_d, ab.POST_ALL)
        want_d = oracle.search(strand, sa, prep.chunks, _osettings(st_d), oracle.POST_ALL, threads=os.cpu_count() or 8)
        assert got_d.as_lists() == want_d.families.as_lists()


@pytest.mark.parametrize("config", [1, 3] + ([4] if os.environ.get("ASGART_B200_BIG") else []))
def test_full_size_properties(config):
    """Full-size C1 / C3 (and C4 = 3.1 Gbp with ASGART_B200_BIG=1): on-device sufcheck, and a search whose result does not
    depend on how the probe range is sharded (1 vs 3 shards)."""
    st, prep = _full_config(config)
    with ab.Context(0) as ctx:
        ctx.load_strand(np.array(prep.strand))
        ctx.build_index()
        _index_properties(ctx, prep)
        whole = ctx.search(prep.chunks, st, ab.POST_ALL)
        parts = [ctx.search_shard(prep.chunks, st, r, 3) for r in range(3)]
        sharded = ctx.finish(prep.chunks, st, parts, ab.POST_ALL)
        assert whole.as_lists() == sharded.as_lists()
        assert whole.n_families > 10
        for fam in whole.as_lists():
            for (l, r, ll, rl, rev, comp) in fam:
                assert l < r and ll >= 1 and rl >= st.min_duplication_length
                assert rev == st.reverse and comp == st.complement


_SORT_BACK_SCRIPT = r"""
import sys
import numpy as np
sys.path.insert(0, {root!r})
import asgart_b200 as ab
import oracle
from tests import cases
rng = np.random.default_rng(5)
texts = [rng.choice(np.frombuffer(b"ACGT", dtype=np.uint8), size=n) for n in (10, 65535, 65536, 65537, 200003, 1 << 20)]
texts.append(np.frombuffer(cases.stress_text(21, n=700_000, n_dups=40), dtype=np.uint8))
g, fr = ab.synth_genome(2, scale_n=3_000_000)
texts.append(np.array(ab.Prepared.from_memory(ab.normalise(g, True), fr, "x.fa").strand))
for t in texts:
    got = ab.r_divsufsort(t, device=0, index_bits=32)
    assert np.array_equal(got, oracle.best_suffix_array(t)), len(t)
print("sort-back ok", len(texts))
"""


def test_sa_sort_back_inverse_scatter(tmp_path):
    """The sort-back inverse scatter (scatter.cuh: two radix partition passes + per-bucket shared-memory scatter) only
    engages above 72 M suffixes; ASGART_B200_PERM_SCATTER_MIN=0 forces it for small texts, including bucket-edge sizes."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, ASGART_B200_PERM_SCATTER_MIN="0")
    r = subprocess.run([sys.executable, "-c", _SORT_BACK_SCRIPT.format(root=root)], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "sort-back ok" in r.stdout, r.stdout + r.stderr


_MSD_SCRIPT = r"""
import sys
import numpy as np
sys.path.insert(0, {root!r})
import asgart_b200 as ab
import oracle
from tests import cases
rng = np.random.default_rng(9)
acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
texts = [rng.choice(acgt, size=n) for n in (300, 4095, 4096, 4097, 6143, 6144, 6145, 70001, 1 << 20)]
texts.append(np.frombuffer(cases.stress_text(31, n=900_000, n_dups=50), dtype=np.uint8))
g, fr = ab.synth_genome(2, scale_n=3_000_000)
soft = np.array(ab.Prepared.from_memory(ab.normalise(g, True), fr, "x.fa").strand)
texts.append(soft)
texts.append(np.full(50_000, ord("A"), dtype=np.uint8))                       # one symbol: every level keeps one giant bucket
texts.append(np.tile(np.frombuffer(b"ACGTTGCA", dtype=np.uint8), 40_000))     # period 8: a handful of huge equal-key buckets
low = rng.choice(acgt, size=400_000); low[50_000:250_000] = np.tile(np.frombuffer(b"AC", dtype=np.uint8), 100_000)
low[300_000:390_000] = ord("N")
texts.append(low)
n_checked = 0
for t in texts:
    t = np.concatenate([t, np.frombuffer(b"$", dtype=np.uint8)])
    want = oracle.best_suffix_array(t)
    for bits in (32, 64):
        got = ab.r_divsufsort(t, device=0, index_bits=bits)
        assert np.array_equal(got, want), (len(t), bits)
        n_checked += 1
# the sharded build takes the same path with every member's own range of level-0 bins
ctxs = [ab.Context(0) for _ in range(3)]
for c in ctxs:
    c.load_strand(soft)
ab.build_index_group(ctxs)
want = oracle.best_suffix_array(soft)
for c in ctxs:
    assert c.stats()["msd_levels"] >= 2
    assert np.array_equal(c.download_sa(), want)
    c.close()
# and a whole search on top of it
prep = ab.Prepared.from_memory(ab.normalise(g, True), fr, "x.fa")
with ab.Context(0) as ctx:
    ctx.load_strand(soft)
    ctx.build_index()
    assert ctx.stats()["msd_levels"] >= 2
    st = ab.RunSettings(reverse=True, complement=True, skip_masked=True)
    got = ctx.search(prep.chunks, st, ab.POST_ALL)
    so = oracle.make_settings(reverse=True, complement=True, skip_masked=True)
    assert got.as_lists() == oracle.search(soft, want, prep.chunks, so, oracle.POST_ALL, threads=4).families.as_lists()
print("msd ok", n_checked)
"""


def test_sa_msd_initial_sort(tmp_path):
    """The MSD form of the initial sort (msd_sort.cuh) only engages above 2 M suffixes; ASGART_B200_MSD_MIN=0 forces it for
    small texts: tile- and window-edge sizes, soft-masked N-runs, one-symbol and periodic texts (giant equal-key buckets on
    every level, the slow path of the local sort), u32 and u64 indices, a 3-member sharded build and a full search."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, ASGART_B200_MSD_MIN="0")
    r = subprocess.run([sys.executable, "-c", _MSD_SCRIPT.format(root=root)], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "msd ok" in r.stdout, r.stdout + r.stderr
