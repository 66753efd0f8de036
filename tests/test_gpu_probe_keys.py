"""Probe search from the sorted initial keys: a single-device build_index keeps the keys of its initial sort with the index,
and probe_search_kernel compares deep buckets in them instead of in suffix-array entries and text windows. Probe ranges
and families must equal the oracle's on both paths; the n_probe_keys counter tells which path ran."""
import os
import subprocess
import sys

import numpy as np
import pytest

import asgart_b200 as ab
import oracle
from tests import cases, kat

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TRANSFORMS = (dict(), dict(complement=True), dict(reverse=True), dict(reverse=True, complement=True))


def _strand(text):
    return np.concatenate([np.asarray(text, dtype=np.uint8), np.frombuffer(b"$", dtype=np.uint8)])


def keys_used(ctx, fn):
    before = ctx.stats()["n_probe_keys"]
    out = fn()
    return out, ctx.stats()["n_probe_keys"] - before


def check_ranges(ctx, strand, sa, osr, st, chunk, every=1):
    """ctx.probe_ranges over one chunk against Searcher::search; returns the probes answered from the keys"""
    k, s = st.probe_size, st.probe_size // 2
    nprobes = -(-(chunk[1] - k - s) // s)
    (glo, ghi), used = keys_used(ctx, lambda: ctx.probe_ranges(chunk, st, nprobes))
    needle = strand[chunk[0]:chunk[0] + chunk[1]]
    if st.complement:
        needle = kat.complement(needle)
    if st.reverse:
        needle = needle[::-1]
    for p in sorted(set(range(0, nprobes, every)) | {nprobes - 1}):
        i = (p + 1) * s
        want = osr.search(needle[i:i + k].tobytes())
        assert ghi[p] - glo[p] == len(want) and np.array_equal(sa[glo[p]:ghi[p]], want), (st, p)
    return used


def check_families(ctx, strand, sa, st, chunks):
    """ctx.search with every post-step against the oracle's search; returns the probes answered from the keys"""
    so = oracle.make_settings(probe_size=st.probe_size, gap_size=st.gap_size, min_length=st.min_duplication_length,
                              max_cardinality=st.max_cardinality, reverse=st.reverse, complement=st.complement,
                              skip_masked=st.skip_masked)
    got, used = keys_used(ctx, lambda: ctx.search(chunks, st, ab.POST_ALL))
    want = oracle.search(strand, sa, chunks, so, oracle.POST_ALL, threads=4)
    assert got.as_lists() == want.families.as_lists(), st
    return used


def run_text(strand, bits, ks, expect_keys, chunk=None, every=1, families=True, transforms=TRANSFORMS):
    """build_index on one device, then ranges (and families) for every k and needle transform; expect_keys(st) -> bool"""
    sa = oracle.best_suffix_array(strand)
    osr = oracle.OracleSearcher(strand, sa)
    n = len(strand) - 1
    chunk = chunk or (0, n)
    with ab.Context(0) as ctx:
        ctx.set_index_bits(bits)
        ctx.load_strand(strand)
        ctx.build_index()
        assert np.array_equal(ctx.download_sa(), sa)
        for k in ks:
            for tr in transforms:
                st = ab.RunSettings(probe_size=k, gap_size=100, min_duplication_length=300, max_cardinality=100000, **tr)
                used = check_ranges(ctx, strand, sa, osr, st, chunk, every)
                if families:
                    used2 = check_families(ctx, strand, sa, st, [chunk])
                    assert (used2 > 0) == (used > 0), (k, tr)
                assert (used > 0) == expect_keys(st), (k, tr, used)
        return ctx.stats()


@pytest.mark.parametrize("bits", [32, 64])
def test_lsd_sized_text_all_transforms(bits):
    """LSD initial sort (p0 = 13, deep depth 7): k = 12 compares keys only, k = 20 / 32 / 40 also the text after equal keys.
    The text carries tandem repeats and a 40-copy element, so some deep buckets exceed LINEAR and are bisected."""
    strand = _strand(cases.stress_text(5, n=50_000))
    run_text(strand, bits, (12, 20, 32, 40), lambda st: True, chunk=(1000, 30_000), every=3)


@pytest.mark.parametrize("bits", [32, 64])
def test_dense_codes_differ_from_strand_codes(bits):
    """Without N the key code of T is 5 and its strand code 6; a soft-masked text under -S has long N runs."""
    no_n = _strand(cases.stress_text(7, n=40_000, with_n=False))
    run_text(no_n, bits, (20,), lambda st: True, every=2)
    g, fr = ab.synth_genome(2, scale_n=400_000)
    prep = ab.Prepared.from_memory(ab.normalise(g, True), fr, "x.fa")
    soft = np.array(prep.strand)   # prep.strand views memory that prep owns: copy it while prep is alive
    del prep
    assert (soft == ord("N")).sum() > 1000
    run_text(soft, bits, (20,), lambda st: True, chunk=(0, 200_000), every=5, families=False,
             transforms=(dict(reverse=True, complement=True, skip_masked=True),))


def test_text_without_t_searched_with_complement():
    """A strand with A but no T has no key code for T, which the complement needle holds: those searches take the text
    path (counter stays 0) and still give the reference's answers; the direct and reversed ones use the keys."""
    rng = np.random.default_rng(11)
    t = rng.choice(np.frombuffer(b"ACG", dtype=np.uint8), size=30_000)
    t[5000:5000 + 400] = t[20_000:20_000 + 400]
    run_text(_strand(t), 32, (20,), lambda st: not st.complement, every=2)


def test_q6_flagged_buckets_stay_literal():
    """The tail of this text shares its 8-mers with most probes (quirk Q6): flagged buckets take the literal search, the
    others the keys; ranges and families equal the oracle's."""
    rng = np.random.default_rng(3)
    unit = kat.rand_dna(rng, 11)
    text = np.concatenate([kat.rand_dna(rng, 3000), np.tile(unit, 400), kat.rand_dna(rng, 9)])
    run_text(_strand(text), 32, (12, 20), lambda st: True, transforms=(dict(), dict(reverse=True, complement=True)))


_MSD_SCRIPT = r"""
import sys
sys.path.insert(0, {root!r})
import numpy as np
import asgart_b200 as ab
from tests import cases
from tests.test_gpu_probe_keys import _strand, run_text
strand = _strand(cases.stress_text(13, n=300_000, n_dups=20))
for bits in (32, 64):
    s = run_text(strand, bits, (20, 21, 22, 32), lambda st: True, chunk=(10_000, 120_000), every=7)
    assert s["msd_levels"] >= 1, s["msd_levels"]
print("msd keys ok")
"""


def test_msd_initial_sort_keys():
    """The MSD form of the initial sort (forced for a small text) has 21-symbol keys: k = 20 compares part of a key, 21 a
    whole one, 22 and 32 the text after equal keys."""
    env = dict(os.environ, ASGART_B200_MSD_MIN="0")
    r = subprocess.run([sys.executable, "-c", _MSD_SCRIPT.format(root=ROOT)], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "msd keys ok" in r.stdout, r.stdout + r.stderr


@pytest.mark.parametrize("bits", [32, 64])
def test_stale_keys_are_not_used(bits):
    """Keys belong to the index they were built with: after load_strand + upload_sa of another text, and after a --trim
    build, the search answers from the new index on the text path."""
    a = _strand(cases.stress_text(17, n=40_000))
    b = _strand(cases.stress_text(19, n=40_000))
    sa_b = oracle.best_suffix_array(b)
    osr_b = oracle.OracleSearcher(b, sa_b)
    st = ab.RunSettings(probe_size=20, gap_size=100, min_duplication_length=300, max_cardinality=100000,
                        reverse=True, complement=True)
    chunk = (0, len(b) - 1)
    with ab.Context(0) as ctx:
        ctx.set_index_bits(bits)
        ctx.load_strand(a)
        ctx.build_index()
        sa_a = oracle.best_suffix_array(a)
        assert check_ranges(ctx, a, sa_a, oracle.OracleSearcher(a, sa_a), st, chunk, every=5) > 0
        ctx.load_strand(b)
        ctx.upload_sa(sa_b)
        assert check_ranges(ctx, b, sa_b, osr_b, st, chunk, every=3) == 0
        assert check_families(ctx, b, sa_b, st, [chunk]) == 0
        # a full build keeps keys again; a --trim build after it drops them
        ctx.build_index()
        assert check_ranges(ctx, b, sa_b, osr_b, st, chunk, every=5) > 0
        trim = (2000, 30_000)
        ctx.build_index(trim=trim)
        so = oracle.make_settings(probe_size=20, gap_size=100, min_length=300, max_cardinality=100000, reverse=True,
                                  complement=True)
        got, used = keys_used(ctx, lambda: ctx.search([chunk], st, ab.POST_ALL))
        assert used == 0
        assert got.as_lists() == oracle.search_trim(b, trim, [chunk], so, oracle.POST_ALL, threads=4).as_lists()


_LAZY_OFF_SCRIPT = r"""
import sys
sys.path.insert(0, {root!r})
from tests import cases
from tests.test_gpu_probe_keys import _strand, run_text
strand = _strand(cases.stress_text(5, n=50_000))
for bits in (32, 64):
    run_text(strand, bits, (20, 32), lambda st: False, chunk=(1000, 30_000), every=3)
print("lazy off ok")
"""


def test_without_lazy_ranks_keys_are_scratch():
    """ASGART_B200_LAZY_RANK=0: the sort-back scatter overwrites the key buffers, so nothing is kept and the text path
    gives the same answers."""
    env = dict(os.environ, ASGART_B200_LAZY_RANK="0")
    r = subprocess.run([sys.executable, "-c", _LAZY_OFF_SCRIPT.format(root=ROOT)], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "lazy off ok" in r.stdout, r.stdout + r.stderr


def test_group_build_keeps_no_keys():
    """Members of a sharded build hold only their key range: their searches take the text path, with the families of a
    single-device build."""
    strand = _strand(cases.stress_text(23, n=60_000, n_dups=20))
    st = ab.RunSettings(probe_size=20, gap_size=100, min_duplication_length=300, max_cardinality=100000,
                        reverse=True, complement=True)
    chunks = [(0, 30_000), (30_000, 30_000)]
    with ab.Context(0) as ctx:
        ctx.load_strand(strand)
        ctx.build_index()
        single, used = keys_used(ctx, lambda: ctx.search(chunks, st, ab.POST_ALL))
        assert used > 0
    ctxs = [ab.Context(0) for _ in range(3)]
    try:
        for c in ctxs:
            c.load_strand(strand)
        ab.build_index_group(ctxs)
        for c in ctxs:
            got, used = keys_used(c, lambda: c.search(chunks, st, ab.POST_ALL))
            assert used == 0
            assert got.as_lists() == single.as_lists()
    finally:
        for c in ctxs:
            c.close()


def test_kept_keys_do_not_grow_device_memory():
    """The kept keys go back to the context's block cache at the next build, before the sort allocates: repeated
    build + search cycles hold the device memory of the second one."""
    import torch
    strand = _strand(cases.stress_text(29, n=200_000, n_dups=20))
    st = ab.RunSettings(reverse=True, complement=True)
    chunks = [(0, len(strand) - 1)]
    used = []
    with ab.Context(0) as ctx:
        ctx.load_strand(strand)
        for _ in range(3):
            ctx.build_index()
            ctx.search(chunks, st, ab.POST_ALL)
            torch.cuda.synchronize(0)
            free, total = torch.cuda.mem_get_info(0)
            used.append(total - free)
        assert ctx.stats()["n_probe_keys"] > 0
    assert used[2] == used[1], used
