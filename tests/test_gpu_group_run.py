"""In-process group runs: several contexts of one process share a run (ctx_copy_strand, build_index_group, search_group,
run_files_devices, the CLI's --devices) and give byte for byte what the one-device path gives. Every member here is on
cuda:0 unless the machine has a second GPU."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import asgart_b200 as ab
from asgart_b200 import _lib
from tests import cases

pytestmark = pytest.mark.gpu

CLI = os.path.join(os.path.dirname(ab.__file__), "asgart-b200")


def _fasta(recs, width=60) -> bytes:
    out = []
    for name, seq in recs:
        out.append(f">{name} synthetic\n")
        out.extend(seq[i:i + width] + "\n" for i in range(0, len(seq), width))
    return "".join(out).encode()


@pytest.fixture(scope="module")
def files(tmp_path_factory):
    """Two FASTA files: the C3 genome at 2 Mbp cut into five records of unequal length (so that --collapse merges some)
    and the soft-masked C2 genome at 600 kbp."""
    d = tmp_path_factory.mktemp("group_run")
    g3, _ = ab.synth_genome(3, scale_n=2_000_000)
    t3 = g3.tobytes().decode()
    cuts = [0, 900_000, 1_500_000, 1_800_000, 1_950_000, 2_000_000]
    a = d / "c3.fa"
    a.write_bytes(_fasta([(f"chr{i + 1}", t3[cuts[i]:cuts[i + 1]]) for i in range(5)]))
    g2, _ = ab.synth_genome(2, scale_n=600_000)
    b = d / "c2.fa"
    b.write_bytes(_fasta([("synthY", g2.tobytes().decode())]))
    return [str(a), str(b)]


def _run(files, passes, devices=None, slice_op=None) -> str:
    """run_files_passes / run_files_sliced_ex on cuda:0 (devices None), else run_files_devices."""
    L = _lib.load()
    arr = (_lib.Settings * len(passes))(*[p.to_c() for p in passes])
    err = C.c_char_p()
    names = "\n".join(files).encode()
    op = C.byref(slice_op) if slice_op is not None else None
    if devices is not None:
        dev = (C.c_int32 * len(devices))(*devices)
        p = L.asgart_b200_run_files_devices(names, arr, len(passes), dev, len(devices), op, C.byref(err))
    elif slice_op is not None:
        p = L.asgart_b200_run_files_sliced_ex(names, arr, len(passes), 0, op, C.byref(err))
    else:
        p = L.asgart_b200_run_files_passes(names, arr, len(passes), 0, C.byref(err))
    if not p:
        raise ab.AsgartB200Error(-1, err.value.decode() if err.value else "run failed")
    try:
        return C.string_at(p).decode()
    finally:
        L.asgart_b200_free_string(p)


S = ab.RunSettings
RUNS = {
    "direct": ([S()], None),
    "R": ([S(reverse=True, min_duplication_length=500)], None),
    "C": ([S(complement=True, min_duplication_length=500)], None),
    "RC": ([S(reverse=True, complement=True)], None),
    "S": ([S(skip_masked=True)], None),
    "score": ([S(reverse=True, complement=True, compute_score=True)], None),
    "RC+direct": ([S(reverse=True, complement=True), S()], None),
    "low-cardinality": ([S(probe_size=12, gap_size=30, min_duplication_length=300, max_cardinality=4)], None),
    "sliced": ([S(reverse=True, complement=True), S()],
               _lib.SliceOptions(_lib.SLICE_COLLAPSE | _lib.SLICE_NO_INTRA | _lib.SLICE_MIN_LENGTH, 0, 1200, 50, None, None, None)),
    "keep-fragments": ([S()], _lib.SliceOptions(0, 0, 0, -1, b"chr1\nsynthY", None, None)),
}


@pytest.mark.parametrize("label", list(RUNS))
def test_run_files_devices_json_identical(files, label):
    passes, op = RUNS[label]
    want = _run(files, passes, slice_op=op)
    if label == "RC+direct":
        assert want.count('"chr_left"') > 10
    for devices in ([0], [0, 0], [0, 0, 0], [0, 0, 0, 0]):
        assert _run(files, passes, devices, op) == want, (label, devices)


def test_search_duplications_devices(files):
    st = S(reverse=True, complement=True, skip_masked=True)
    want = ab.search_duplications(files, st)
    assert ab.search_duplications(files, st, devices=[0, 0]) == want
    passes = [st, S(skip_masked=True)]
    assert ab.search_duplications_passes(files, passes, devices=[0, 0, 0]) == ab.search_duplications_passes(files, passes)


@pytest.mark.skipif(ab.device_count() < 2, reason="needs two GPUs")
def test_distinct_gpus_json_identical(files):
    passes, op = RUNS["RC+direct"]
    want = _run(files, passes)
    assert _run(files, passes, [0, 1]) == want
    assert _run(files, passes, [1, 0, 1]) == want
    passes, op = RUNS["sliced"]
    assert _run(files, passes, [0, 1], op) == _run(files, passes, slice_op=op)


# ------------------------------------------------------------------------------------------------ search_group
ST = S(min_duplication_length=500, reverse=True, complement=True)


@pytest.mark.parametrize("bits", [32, 64])
def test_search_group_equals_search(bits):
    text = cases.stress_text(31, n=300_000, n_dups=40)
    prep = ab.Prepared.from_memory(text, [("a", 0, 200_000), ("b", 200_000, len(text) - 200_000)], "g.fa")
    strand = np.array(prep.strand)
    # the full chunk list, one short chunk (some shards hold no probe) and a chunk with no probe at all
    chunk_lists = [prep.chunks, [(1000, 700)], [(5000, 10)]]
    settings = [ST, S(min_duplication_length=300, max_cardinality=5), S(min_duplication_length=100, compute_score=True)]
    with ab.Context(0) as one:
        one.set_index_bits(bits)
        one.load_strand(strand)
        one.build_index()
        want = {(c, s): one.search(chunk_lists[c], settings[s]).digest() for c in range(3) for s in range(3)}
    assert len(set(want.values())) >= 3
    for world in (1, 2, 3, 4):
        ctxs = [ab.Context(0) for _ in range(world)]
        try:
            for c in ctxs:
                c.set_index_bits(bits)
            ctxs[0].load_strand(strand)
            for c in ctxs[1:]:
                c.copy_strand_from(ctxs[0])
            ab.build_index_group(ctxs)
            for (ci, si), d in want.items():
                got = ab.search_group(ctxs, chunk_lists[ci], settings[si])
                assert got.digest() == d, (world, ci, si)
                assert ctxs[0].search(chunk_lists[ci], settings[si]).digest() == d, (world, ci, si)
        finally:
            for c in ctxs:
                c.close()


def test_copy_strand():
    text = cases.stress_text(5, n=200_000, n_dups=20)
    prep = ab.Prepared.from_memory(text, [("a", 0, len(text))], "g.fa")
    with ab.Context(0) as src, ab.Context(0) as dst:
        src.load_strand(np.array(prep.strand))
        src.build_index()
        dst.load_strand(np.frombuffer(b"ACGT" * 10 + b"$", dtype=np.uint8))   # replaced by the copy
        dst.build_index()
        dst.copy_strand_from(src)
        assert np.array_equal(dst.download_strand(), src.download_strand())
        with pytest.raises(ab.AsgartB200Error):   # the copy drops the index, as load_strand does
            dst.search(prep.chunks, ST)
        dst.build_index()
        assert dst.sa_fingerprint() == src.sa_fingerprint()
        assert dst.search(prep.chunks, ST).digest() == src.search(prep.chunks, ST).digest()


# ------------------------------------------------------------------------------------------------ errors
def test_group_errors_leave_contexts_usable(files):
    text = cases.stress_text(8, n=120_000, n_dups=20)
    prep = ab.Prepared.from_memory(text, [("a", 0, len(text))], "g.fa")
    strand = np.array(prep.strand)
    prep_other = ab.Prepared.from_memory(text[:100_000], [("a", 0, 100_000)], "h.fa")
    other = np.array(prep_other.strand)
    with ab.Context(0) as a, ab.Context(0) as b, ab.Context(0) as empty:
        a.load_strand(strand)
        a.build_index()
        want = a.search(prep.chunks, ST).digest()
        # copy_strand from a context without a strand
        with pytest.raises(ab.AsgartB200Error) as e:
            b.copy_strand_from(empty)
        assert e.value.code == _lib.ESTATE
        # a member without an index
        b.copy_strand_from(a)
        with pytest.raises(ab.AsgartB200Error) as e:
            ab.search_group([a, b], prep.chunks, ST)
        assert e.value.code == _lib.ESTATE and "member 1" in str(e.value)
        # members with different strands
        b.load_strand(other)
        b.build_index()
        with pytest.raises(ab.AsgartB200Error) as e:
            ab.search_group([a, b], prep.chunks, ST)
        assert e.value.code == _lib.ESTATE
        # a context given twice
        with pytest.raises(ab.AsgartB200Error):
            ab.search_group([a, a], prep.chunks, ST)
        # stage A fails on every member (a chunk outside the strand)
        b.copy_strand_from(a)
        b.build_index()
        with pytest.raises(ab.AsgartB200Error):
            ab.search_group([a, b], [(0, len(text) + 5)], ST)
        # every context still works
        assert a.search(prep.chunks, ST).digest() == want
        assert b.search(prep.chunks, ST).digest() == want
        assert ab.search_group([a, b], prep.chunks, ST).digest() == want
        empty.copy_strand_from(a)
        empty.build_index()
        assert ab.search_group([empty, a, b], prep.chunks, ST).digest() == want
    passes = [S(trim=(1000, 500_000))]
    with pytest.raises(ab.AsgartB200Error, match="--trim"):
        _run(files, passes, [0, 0])
    with pytest.raises(ab.AsgartB200Error, match="device 99"):
        _run(files, [S()], [0, 99])
    assert _run(files, [S()], [0, 0]) == _run(files, [S()])


# ------------------------------------------------------------------------------------------------ CLI
def test_cli_devices(files, tmp_path):
    one, two = tmp_path / "one.json", tmp_path / "two.json"
    r = subprocess.run([CLI, "-RC", "--with-direct", "--out", str(one), *files], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([CLI, "-RC", "--with-direct", "--devices", "0,0", "--out", str(two), *files], capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr
    assert one.read_bytes() == two.read_bytes()
    r = subprocess.run([CLI, "--device", "1", "--devices", "0", "--out", str(tmp_path / "x.json"), *files], capture_output=True,
                       text=True, timeout=60)
    assert r.returncode == 2 and "--devices" in r.stderr
    assert not (tmp_path / "x.json").exists()
    r = subprocess.run([CLI, "--devices", "0,0", "--trim", "10", "1000", "--out", str(tmp_path / "t.json"), *files],
                       capture_output=True, text=True, timeout=60)
    assert r.returncode == 1 and "--trim" in r.stderr
