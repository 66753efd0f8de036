"""Host-side mirror of the reference's interface for the duplication-search path, over the C ABI (ctypes).

Names follow the reference (delehef/asgart @ 523b07c): ``RunSettings`` (src/structs.rs:36-58), ``r_divsufsort``
(src/bin/asgart.rs:473-479), ``prepare_data`` (:273-471), ``search_duplications`` (:731-822), the Step order of
:738-747. All compute happens in libasgart_b200.so on a CUDA device; nothing here falls back to the CPU.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import _lib
from ._lib import POST_ALL, POST_COMPUTE_SCORE, POST_FILTER_NS, POST_REDUCE_OVERLAP, POST_REORDER, POST_SORT  # noqa: F401


class AsgartB200Error(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"asgart_b200 error {code}: {msg}")
        self.code = code


@dataclass
class RunSettings:
    """src/structs.rs:36-58. ``gap_size`` is the CLI value; max_gap_size = gap_size + probe_size (src/bin/asgart.rs:681)."""
    probe_size: int = 20
    gap_size: int = 100
    min_duplication_length: int = 1000
    max_cardinality: int = 500
    reverse: bool = False
    complement: bool = False
    skip_masked: bool = False
    trim: Optional[Tuple[int, int]] = None
    compute_score: bool = False   # --compute-score: the ComputeScore step (src/bin/asgart.rs:744-746) runs on the GPU

    @property
    def max_gap_size(self) -> int:
        return self.gap_size + self.probe_size

    def to_c(self) -> _lib.Settings:
        t = self.trim or (0, 0)
        return _lib.Settings(self.probe_size, self.max_gap_size, int(self.reverse), int(self.complement),
                             int(self.skip_masked), self.min_duplication_length, self.max_cardinality,
                             int(self.trim is not None), int(self.compute_score), t[0], t[1])


PROTOSD_DTYPE = np.dtype([("left", "<u8"), ("right", "<u8"), ("left_length", "<u8"), ("right_length", "<u8"),
                          ("identity", "<f4"), ("reversed", "u1"), ("complemented", "u1"), ("_pad", "u1", (2,))])
assert PROTOSD_DTYPE.itemsize == C.sizeof(_lib.ProtoSD) == 40


def families_digest(fam_offsets, fields, identity, flags) -> str:
    """sha256 over Vec<ProtoSDsFamily> in the reference's own order (chunk -> flush -> arm creation, src/bin/asgart.rs:241-253):
    family offsets as little-endian u64, then per duplicon (left, right, left_length, right_length) as u64, identity as f32
    bits, (reversed, complemented) as bytes. Equal digests <=> equal families, order included."""
    import hashlib
    h = hashlib.sha256()
    h.update(np.ascontiguousarray(fam_offsets).astype("<u8").tobytes())
    h.update(np.ascontiguousarray(fields).astype("<u8").reshape(-1, 4).tobytes())
    h.update(np.ascontiguousarray(identity).astype("<f4").tobytes())
    h.update(np.ascontiguousarray(flags).astype("u1").reshape(-1, 2).tobytes())
    return h.hexdigest()


def sa_fingerprint_host(sa: np.ndarray) -> int:
    """The order-sensitive 64-bit fingerprint Context.sa_fingerprint computes on the device, for a host array:
    sum over i of splitmix64(SA[i] + i * 0x9E3779B97F4A7C15) mod 2^64 (numpy, chunked)."""
    total = np.uint64(0)
    step = 1 << 24
    with np.errstate(over="ignore"):
        for o in range(0, len(sa), step):
            v = np.asarray(sa[o:o + step]).astype(np.uint64)
            z = v + np.arange(o, o + len(v), dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15)
            z = z + np.uint64(0x9E3779B97F4A7C15)
            z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
            z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
            z = z ^ (z >> np.uint64(31))
            total = total + z.sum(dtype=np.uint64)
    return int(total)


@dataclass
class Families:
    """Vec<ProtoSDsFamily> as CSR: family f = sds[fam_offsets[f]:fam_offsets[f+1]] (structured array, ProtoSD layout)."""
    fam_offsets: np.ndarray
    sds: np.ndarray

    def digest(self) -> str:
        s = self.sds
        fields = np.stack([s["left"], s["right"], s["left_length"], s["right_length"]], axis=1) if len(s) else np.zeros((0, 4), "<u8")
        flags = np.stack([s["reversed"], s["complemented"]], axis=1) if len(s) else np.zeros((0, 2), "u1")
        return families_digest(self.fam_offsets, fields, s["identity"], flags)

    def as_lists(self):
        out = []
        for f in range(len(self.fam_offsets) - 1):
            out.append([(int(s["left"]), int(s["right"]), int(s["left_length"]), int(s["right_length"]),
                         bool(s["reversed"]), bool(s["complemented"]))
                        for s in self.sds[int(self.fam_offsets[f]):int(self.fam_offsets[f + 1])]])
        return out

    def canonical(self):
        return sorted(sorted(f) for f in self.as_lists())

    @property
    def n_families(self) -> int:
        return len(self.fam_offsets) - 1


def _with_score(settings: "RunSettings", post_mask: int) -> int:
    """settings.compute_score pushes the ComputeScore step (src/bin/asgart.rs:744-746) onto a full pipeline."""
    return post_mask | POST_COMPUTE_SCORE if (settings.compute_score and post_mask) else post_mask


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _chunks_array(chunks: Sequence[Tuple[int, int]]) -> np.ndarray:
    return np.ascontiguousarray(np.array(list(chunks), dtype=np.uint64).reshape(-1, 2))


def _take_result(L, rh) -> Families:
    """Copy a library-owned asgart_b200_result into numpy arrays and free it."""
    try:
        nf = L.asgart_b200_result_n_families(rh)
        ns = L.asgart_b200_result_n_sds(rh)
        off = np.ctypeslib.as_array(C.cast(L.asgart_b200_result_family_offsets(rh), C.POINTER(C.c_uint64)), shape=(nf + 1,)).copy()
        if ns:
            buf = C.string_at(L.asgart_b200_result_sds(rh), ns * PROTOSD_DTYPE.itemsize)
            sds = np.frombuffer(buf, dtype=PROTOSD_DTYPE).copy()
        else:
            sds = np.zeros(0, dtype=PROTOSD_DTYPE)
        return Families(off, sds)
    finally:
        L.asgart_b200_result_free(rh)


@dataclass
class Hits:
    """Answer of Context.locate for a batch of patterns: sa_search64's (first, count) per pattern (count never capped) and
    the reported positions, pattern i's being positions[offsets[i]:offsets[i+1]] = SA[first[i] : first[i] + min(count[i],
    max_hits)], in suffix-array order."""
    first: np.ndarray      # int64[n]
    count: np.ndarray      # int64[n]
    offsets: np.ndarray    # uint64[n + 1]
    positions: np.ndarray  # int64[offsets[n]]

    def positions_of(self, i: int) -> np.ndarray:
        return self.positions[int(self.offsets[i]):int(self.offsets[i + 1])]


def pattern_batch(patterns) -> Tuple[np.ndarray, np.ndarray]:
    """(uint8 bytes, uint64 offsets[n + 1]) of a batch: a sequence of bytes / str, or such a pair already (for millions of
    patterns without a Python loop)."""
    if isinstance(patterns, tuple) and len(patterns) == 2 and isinstance(patterns[0], np.ndarray):
        buf = np.ascontiguousarray(patterns[0], dtype=np.uint8).reshape(-1)
        off = np.ascontiguousarray(patterns[1], dtype=np.uint64).reshape(-1)
        if len(off) == 0 or int(off[-1]) != len(buf):
            raise AsgartB200Error(_lib.EINVAL, "pattern offsets must have n + 1 entries, the last one the byte count")
        return buf, off
    items = [p.encode() if isinstance(p, str) else bytes(p) for p in patterns]
    off = np.zeros(len(items) + 1, dtype=np.uint64)
    if items:
        np.cumsum([len(p) for p in items], out=off[1:])
    return np.frombuffer(b"".join(items), dtype=np.uint8), off


def device_count() -> int:
    return int(_lib.load().asgart_b200_device_count())


def r_divsufsort(dna, device: Optional[int] = None, index_bits: int = 0) -> np.ndarray:
    """Suffix array of ``dna`` (any bytes) as int64 — drop-in for r_divsufsort / divsufsort64."""
    L = _lib.load()
    t = np.ascontiguousarray(np.frombuffer(bytes(dna), dtype=np.uint8) if isinstance(dna, (bytes, bytearray)) else dna,
                             dtype=np.uint8)
    sa = np.empty(len(t), dtype=np.int64)
    if device is None and index_bits == 0:
        rc = L.asgart_b200_divsufsort64(_ptr(t), _ptr(sa), len(t))
    else:
        rc = L.asgart_b200_divsufsort64_ex(_ptr(t), _ptr(sa), len(t), device or 0, index_bits)
    if rc != 0:
        raise AsgartB200Error(rc, "asgart_b200_divsufsort64 failed")
    return sa


def effective_trim(trim: Tuple[int, int], n_plus_1: int) -> Optional[Tuple[int, int]]:
    """prepare_data's --trim validation (src/bin/asgart.rs:432-463): the effective (start, stop) or None when skipped."""
    a, b = C.c_uint64(), C.c_uint64()
    ok = _lib.load().asgart_b200_effective_trim(int(trim[0]), int(trim[1]), int(n_plus_1), C.byref(a), C.byref(b))
    return (a.value, b.value) if ok else None


def dist_unique_id() -> bytes:
    """Rank 0's id for Context.dist_init (send it to the other ranks, e.g. with torch.distributed.broadcast)."""
    L = _lib.load()
    buf = np.zeros(128, dtype=np.uint8)
    n = L.asgart_b200_dist_unique_id(_ptr(buf), len(buf))
    if n <= 0:
        raise AsgartB200Error(n, "cannot create a NCCL unique id (libnccl.so.2 missing?)")
    return buf[:n].tobytes()


def build_index_group(ctxs: Sequence["Context"]):
    """Sharded index build by several contexts of this process (host threads; devices need peer access, or may all be
    the same device). Every context must have the same strand loaded; all end up with the whole index."""
    L = _lib.load()
    arr = (C.c_void_p * len(ctxs))(*[c.h for c in ctxs])
    rc = L.asgart_b200_build_index_group(arr, len(ctxs))
    if rc != 0:
        msgs = [L.asgart_b200_ctx_last_error(c.h).decode() for c in ctxs]
        raise AsgartB200Error(rc, "; ".join(m for m in msgs if m))


class Context:
    """One device context: strand + index resident in HBM, searches run against it."""

    def __init__(self, device: int = 0):
        self.L = _lib.load()
        h = C.c_void_p()
        rc = self.L.asgart_b200_ctx_create(device, C.byref(h))
        if rc != 0:
            raise AsgartB200Error(rc, "no usable CUDA device (asgart_b200 has no CPU path)" if rc == _lib.ENODEVICE
                                  else "ctx_create failed")
        self.h = h
        self.n1 = 0

    def close(self):
        if getattr(self, "h", None):
            self.L.asgart_b200_ctx_destroy(self.h)
            self.h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc: int):
        if rc != 0:
            raise AsgartB200Error(rc, self.L.asgart_b200_ctx_last_error(self.h).decode())

    # -- index
    def load_strand(self, strand_with_dollar: np.ndarray):
        t = np.ascontiguousarray(strand_with_dollar, dtype=np.uint8)
        self.n1 = len(t)
        self._check(self.L.asgart_b200_ctx_load_strand(self.h, _ptr(t), len(t)))

    def load_strand_ptr(self, ptr: int, n1: int):
        """Load from a raw host pointer (e.g. a pinned torch tensor's data_ptr())."""
        self.n1 = n1
        self._check(self.L.asgart_b200_ctx_load_strand(self.h, C.c_void_p(ptr), n1))

    # -- GPU-side FASTA ingest (prepare_data on the device, src/bin/asgart.rs:273-471)
    def ingest(self, files: Sequence, skip_masked: bool = False, names: Optional[Sequence[str]] = None) -> "Prepared":
        """read_fasta + find_chunks_to_process + '$' for FASTA files on the device. `files`: paths (str) or the files'
        raw bytes (bytes / uint8 arrays; `names` then gives the file names for the JSON). The context ends up as after
        load_strand; the returned Prepared has the fragment map and the chunks but no host copy of the strand."""
        self._check(self.L.asgart_b200_ctx_ingest_begin(self.h))
        shown = []
        for i, f in enumerate(files):
            if isinstance(f, str):
                self._check(self.L.asgart_b200_ctx_ingest_file(self.h, f.encode(), int(skip_masked)))
                shown.append(f)
            else:
                b = np.frombuffer(f, dtype=np.uint8) if isinstance(f, (bytes, bytearray)) else np.ascontiguousarray(f, dtype=np.uint8)
                self._check(self.L.asgart_b200_ctx_ingest_fasta(self.h, _ptr(b) if len(b) else None, len(b), int(skip_masked)))
                shown.append(names[i] if names else f"mem{i}.fa")
        h = C.c_void_p()
        self._check(self.L.asgart_b200_ctx_ingest_finish(self.h, "\n".join(shown).encode(), C.byref(h)))
        prep = Prepared(h.value)
        self.n1 = prep.n1
        return prep

    def download_strand(self) -> np.ndarray:
        out = np.empty(self.n1, dtype=np.uint8)
        self._check(self.L.asgart_b200_ctx_download_strand(self.h, _ptr(out), len(out)))
        return out

    def set_index_bits(self, bits: int):
        self._check(self.L.asgart_b200_ctx_set_index_bits(self.h, bits))

    def build_index(self, trim: Optional[Tuple[int, int]] = None):
        """Suffix array + LUT. `trim` = the raw --trim values: validated like prepare_data does (src/bin/asgart.rs:432-463);
        when they survive, the index covers strand[start..stop] only (src/bin/asgart.rs:142-147)."""
        self.sa_len = self.n1
        eff = effective_trim(trim, self.n1) if trim is not None else None
        if eff is None:
            self._check(self.L.asgart_b200_ctx_build_index(self.h))
        else:
            self._check(self.L.asgart_b200_ctx_build_index_trim(self.h, eff[0], eff[1]))
            self.sa_len = eff[1] - eff[0] + 1

    def dist_init(self, rank: int, world: int, unique_id: bytes):
        """Join a group of `world` processes (one per GPU): build_index becomes a collective, sharded build."""
        buf = np.frombuffer(unique_id, dtype=np.uint8).copy()
        self._check(self.L.asgart_b200_ctx_dist_init(self.h, rank, world, _ptr(buf), len(buf)))

    def dist_shutdown(self):
        self._check(self.L.asgart_b200_ctx_dist_shutdown(self.h))

    def upload_sa(self, sa: np.ndarray):
        sa = np.ascontiguousarray(sa, dtype=np.int64)
        assert len(sa) == self.n1
        self._check(self.L.asgart_b200_ctx_upload_sa(self.h, _ptr(sa)))
        self.sa_len = self.n1

    def download_sa(self) -> np.ndarray:
        sa = np.empty(getattr(self, "sa_len", self.n1) or self.n1, dtype=np.int64)
        self._check(self.L.asgart_b200_ctx_download_sa(self.h, _ptr(sa)))
        return sa

    def check_sa(self) -> int:
        """sufcheck on the device: number of violations (0 = the index is a valid suffix array of the strand)."""
        bad = C.c_int64()
        self._check(self.L.asgart_b200_ctx_check_sa(self.h, C.byref(bad)))
        return bad.value

    def sa_fingerprint(self) -> int:
        """Order-sensitive 64-bit fingerprint of the index computed on the device (== sa_fingerprint_host of the array)."""
        fp = C.c_uint64()
        self._check(self.L.asgart_b200_ctx_sa_fingerprint(self.h, C.byref(fp)))
        return fp.value

    def download_lut(self) -> Tuple[np.ndarray, np.ndarray]:
        lo = np.empty(_lib.LUT_SIZE, dtype=np.int64)
        hi = np.empty(_lib.LUT_SIZE, dtype=np.int64)
        self._check(self.L.asgart_b200_ctx_download_lut(self.h, _ptr(lo), _ptr(hi)))
        return lo, hi

    # -- search
    def _take(self, rh) -> Families:
        return _take_result(self.L, rh)

    def search(self, chunks: Sequence[Tuple[int, int]], settings: RunSettings, post_mask: int = POST_ALL) -> Families:
        ch = _chunks_array(chunks)
        st = settings.to_c()
        rh = C.c_void_p()
        self._check(self.L.asgart_b200_ctx_search(self.h, _ptr(ch), len(ch), C.byref(st), _with_score(settings, post_mask), C.byref(rh)))
        return self._take(rh)

    def probe_ranges(self, chunk: Tuple[int, int], settings: RunSettings, n_probes: int):
        ch = _chunks_array([chunk])
        st = settings.to_c()
        lo = np.empty(n_probes, dtype=np.int64)
        hi = np.empty(n_probes, dtype=np.int64)
        self._check(self.L.asgart_b200_ctx_probe_ranges(self.h, _ptr(ch), C.byref(st), _ptr(lo), _ptr(hi), n_probes))
        return lo, hi

    def locate(self, patterns, max_hits: Optional[int] = None) -> Hits:
        """Where each pattern occurs in the strand, from the resident index: libdivsufsort's sa_search64 for every pattern
        of the batch (any bytes, compared as bytes) and up to ``max_hits`` positions each (None: all, 0: counts only).
        ``patterns``: a sequence of bytes / str, or a (uint8 array, uint64 offsets[n + 1]) pair."""
        buf, off = pattern_batch(patterns)
        n = len(off) - 1
        h = C.c_void_p()
        self._check(self.L.asgart_b200_ctx_locate(self.h, _ptr(buf) if len(buf) else None, _ptr(off), n,
                                                  -1 if max_hits is None else int(max_hits), C.byref(h)))
        L = self.L
        try:
            def arr(ptr, ctype, k, dtype):
                if k == 0:
                    return np.zeros(0, dtype=dtype)
                return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(ctype)), shape=(k,)).copy()
            offsets = arr(L.asgart_b200_hits_offsets(h), C.c_uint64, n + 1, np.uint64)
            return Hits(arr(L.asgart_b200_hits_first(h), C.c_int64, n, np.int64),
                        arr(L.asgart_b200_hits_count(h), C.c_int64, n, np.int64), offsets,
                        arr(L.asgart_b200_hits_positions(h), C.c_int64, int(offsets[-1]), np.int64))
        finally:
            L.asgart_b200_hits_free(h)

    def sa_search(self, patterns) -> Tuple[np.ndarray, np.ndarray]:
        """sa_search64 for every pattern of the batch: (first int64[n], count int64[n]); see locate."""
        hits = self.locate(patterns, max_hits=0)
        return hits.first, hits.count

    def search_shard(self, chunks, settings: RunSettings, shard: int, n_shards: int) -> bytes:
        """Stage A over this rank's probe range; returns the serialised partial (to be all-gathered)."""
        ch = _chunks_array(chunks)
        st = settings.to_c()
        ph = C.c_void_p()
        self._check(self.L.asgart_b200_ctx_search_shard(self.h, _ptr(ch), len(ch), C.byref(st), shard, n_shards,
                                                        C.byref(ph)))
        try:
            n = self.L.asgart_b200_partial_size(ph)
            buf = np.empty(n, dtype=np.uint8)
            rc = self.L.asgart_b200_partial_serialize(ph, _ptr(buf), n)
            assert rc == 0
            return buf
        finally:
            self.L.asgart_b200_partial_free(ph)

    def finish(self, chunks, settings: RunSettings, partials: Sequence[np.ndarray], post_mask: int = POST_ALL) -> Families:
        ch = _chunks_array(chunks)
        st = settings.to_c()
        parts = [np.ascontiguousarray(p, dtype=np.uint8) for p in partials]
        ptrs = (C.c_void_p * len(parts))(*[p.ctypes.data for p in parts])
        sizes = (C.c_int64 * len(parts))(*[len(p) for p in parts])
        rh = C.c_void_p()
        self._check(self.L.asgart_b200_ctx_finish(self.h, _ptr(ch), len(ch), C.byref(st), ptrs, sizes, len(parts),
                                                  _with_score(settings, post_mask), C.byref(rh)))
        return self._take(rh)

    def search_shard_dev(self, chunks, settings: RunSettings, shard: int, n_shards: int):
        """Stage A over this rank's probe range, partial kept in HBM: (device pointer, bytes, meta uint64[4])."""
        ch = _chunks_array(chunks)
        st = settings.to_c()
        ptr, nbytes = C.c_void_p(), C.c_int64()
        meta = np.zeros(4, dtype=np.uint64)
        self._check(self.L.asgart_b200_ctx_search_shard_dev(self.h, _ptr(ch), len(ch), C.byref(st), shard, n_shards,
                                                            C.byref(ptr), C.byref(nbytes), _ptr(meta)))
        return ptr.value or 0, nbytes.value, meta

    def finish_dev(self, chunks, settings: RunSettings, blob_ptrs: Sequence[int], metas: np.ndarray, post_mask: int = POST_ALL) -> Families:
        ch = _chunks_array(chunks)
        st = settings.to_c()
        metas = np.ascontiguousarray(metas, dtype=np.uint64).reshape(-1, 4)
        ptrs = (C.c_void_p * len(blob_ptrs))(*blob_ptrs)
        rh = C.c_void_p()
        self._check(self.L.asgart_b200_ctx_finish_dev(self.h, _ptr(ch), len(ch), C.byref(st), ptrs, _ptr(metas), len(blob_ptrs),
                                                      _with_score(settings, post_mask), C.byref(rh)))
        return self._take(rh)

    def post_steps(self, fam: Families, post_mask: int) -> Families:
        off = np.ascontiguousarray(fam.fam_offsets, dtype=np.uint64)
        sds = np.ascontiguousarray(fam.sds, dtype=PROTOSD_DTYPE)
        rh = C.c_void_p()
        self._check(self.L.asgart_b200_ctx_post_steps(self.h, _ptr(off), len(off) - 1, _ptr(sds), post_mask, C.byref(rh)))
        return self._take(rh)

    def stats(self) -> dict:
        s = _lib.Stats()
        self._check(self.L.asgart_b200_ctx_stats(self.h, C.byref(s)))
        # n_probe_keys: probes answered from the sorted keys kept with the index (asgart_b200_ctx_probe_keys)
        return s.as_dict() | {"n_probe_keys": int(self.L.asgart_b200_ctx_probe_keys(self.h))}

    def reset_stats(self):
        self.L.asgart_b200_ctx_reset_stats(self.h)

    def timer_start(self):
        self._check(self.L.asgart_b200_ctx_timer_start(self.h))

    def timer_stop(self) -> float:
        ms = C.c_double()
        self._check(self.L.asgart_b200_ctx_timer_stop(self.h, C.byref(ms)))
        return ms.value


def families_from_lists(fams: Sequence[Sequence[Tuple[int, int, int, int]]], reverse=False, complement=False) -> Families:
    off = [0]
    rows = []
    for f in fams:
        for sd in f:
            rows.append((sd[0], sd[1], sd[2], sd[3], 0.0, int(reverse), int(complement), (0, 0)))
        off.append(len(rows))
    return Families(np.array(off, dtype=np.uint64), np.array(rows, dtype=PROTOSD_DTYPE) if rows else np.zeros(0, PROTOSD_DTYPE))


# ---------------------------------------------------------------------------------------------- host side
class Prepared:
    """prepare_data output (src/bin/asgart.rs:273-471): strand incl. '$', fragment map, chunks_to_process."""

    def __init__(self, handle):
        self.L = _lib.load()
        self.h = C.c_void_p(handle)
        n1 = C.c_int64()
        p = self.L.asgart_b200_prepared_strand(self.h, C.byref(n1))
        self.n1 = n1.value
        # view owned by the handle; None when the strand lives only on the device (Context.ingest)
        self.strand = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(n1.value,)) if p else None
        nc = C.c_int64()
        cp = self.L.asgart_b200_prepared_chunks(self.h, C.byref(nc))
        ch = np.ctypeslib.as_array(C.cast(cp, C.POINTER(C.c_uint64)), shape=(nc.value, 2)) if nc.value else np.zeros((0, 2), np.uint64)
        self.chunks = [(int(a), int(b)) for a, b in ch]
        self.map = []
        for i in range(self.L.asgart_b200_prepared_n_fragments(self.h)):
            pos, ln = C.c_uint64(), C.c_uint64()
            nm = self.L.asgart_b200_prepared_fragment(self.h, i, C.byref(pos), C.byref(ln))
            self.map.append((nm.decode(), pos.value, ln.value))

    @classmethod
    def from_files(cls, files: Sequence[str], skip_masked: bool = False) -> "Prepared":
        L = _lib.load()
        err = C.c_char_p()
        h = L.asgart_b200_prepare_files("\n".join(files).encode(), int(skip_masked), C.byref(err))
        if not h:
            raise IOError(err.value.decode() if err.value else "prepare_data failed")
        return cls(h)

    @classmethod
    def from_memory(cls, strand_no_dollar: np.ndarray, fragments: Sequence[Tuple[str, int, int]], file_names: str = "mem.fa"):
        L = _lib.load()
        t = np.ascontiguousarray(strand_no_dollar, dtype=np.uint8)
        pos = np.array([f[1] for f in fragments], dtype=np.uint64)
        ln = np.array([f[2] for f in fragments], dtype=np.uint64)
        h = L.asgart_b200_prepare_memory(file_names.encode(), _ptr(t), len(t), "\n".join(f[0] for f in fragments).encode(),
                                         _ptr(pos), _ptr(ln), len(fragments))
        if not h:
            raise ValueError("prepare_memory: bad fragment table")
        return cls(h)

    def slice(self, fam: Families, no_direct=False, no_reversed=False, no_uncomplemented=False, no_complemented=False,
              no_inter=False, no_intra=False, min_length: Optional[int] = None, max_family_members: Optional[int] = None) -> Families:
        """asgart-slice's duplicon filters (src/bin/asgart-slice.rs:126-160) on families in memory; host code only."""
        flags = (_lib.SLICE_NO_DIRECT * bool(no_direct) | _lib.SLICE_NO_REVERSED * bool(no_reversed)
                 | _lib.SLICE_NO_UNCOMPLEMENTED * bool(no_uncomplemented) | _lib.SLICE_NO_COMPLEMENTED * bool(no_complemented)
                 | _lib.SLICE_NO_INTER * bool(no_inter) | _lib.SLICE_NO_INTRA * bool(no_intra)
                 | _lib.SLICE_MIN_LENGTH * (min_length is not None))
        off = np.ascontiguousarray(fam.fam_offsets, dtype=np.uint64)
        sds = np.ascontiguousarray(fam.sds, dtype=PROTOSD_DTYPE)
        rh = C.c_void_p()
        rc = self.L.asgart_b200_slice_families(self.h, _ptr(off), len(off) - 1, _ptr(sds) if len(sds) else None, flags, int(min_length or 0),
                                               -1 if max_family_members is None else int(max_family_members), C.byref(rh))
        if rc != 0:
            raise AsgartB200Error(rc, "slice_families failed")
        return _take_result(self.L, rh)

    def slice_json(self, settings: RunSettings, fam: Families, collapse=False, no_direct=False, no_reversed=False,
                   no_uncomplemented=False, no_complemented=False, no_inter=False, no_inter_relaxed=False, no_intra=False,
                   min_length: Optional[int] = None, max_family_members: Optional[int] = None,
                   keep_fragments: Optional[Sequence[str]] = None, restrict_fragments: Optional[Sequence[str]] = None,
                   exclude_fragments: Optional[Sequence[str]] = None, regexp=False) -> str:
        """`asgart-slice` on the result of a run (src/bin/asgart-slice.rs:126-191), options applied in its order -> the JSON
        it would write. Host code only."""
        flags = (_lib.SLICE_COLLAPSE * bool(collapse) | _lib.SLICE_NO_DIRECT * bool(no_direct) | _lib.SLICE_NO_REVERSED * bool(no_reversed)
                 | _lib.SLICE_NO_UNCOMPLEMENTED * bool(no_uncomplemented) | _lib.SLICE_NO_COMPLEMENTED * bool(no_complemented)
                 | _lib.SLICE_NO_INTER * bool(no_inter) | _lib.SLICE_NO_INTER_RELAXED * bool(no_inter_relaxed)
                 | _lib.SLICE_NO_INTRA * bool(no_intra) | _lib.SLICE_MIN_LENGTH * (min_length is not None) | _lib.SLICE_REGEXP * bool(regexp))
        enc = lambda l: None if l is None else "\n".join(l).encode()   # noqa: E731
        op = _lib.SliceOptions(flags, 0, int(min_length or 0), -1 if max_family_members is None else int(max_family_members),
                               enc(keep_fragments), enc(restrict_fragments), enc(exclude_fragments))
        st = settings.to_c()
        off = np.ascontiguousarray(fam.fam_offsets, dtype=np.uint64)
        sds = np.ascontiguousarray(fam.sds, dtype=PROTOSD_DTYPE)
        rr = self.L.asgart_b200_run_result_new(self.h, C.byref(st), _ptr(off), len(off) - 1, _ptr(sds) if len(sds) else None)
        if not rr:
            raise AsgartB200Error(_lib.EINVAL, "run_result_new failed")
        try:
            rc = self.L.asgart_b200_run_result_slice(rr, C.byref(op))
            if rc != 0:
                raise AsgartB200Error(rc, self.L.asgart_b200_run_result_error(rr).decode())
            p = self.L.asgart_b200_run_result_to_json(rr)
            try:
                return C.string_at(p).decode()
            finally:
                self.L.asgart_b200_free_string(p)
        finally:
            self.L.asgart_b200_run_result_free(rr)

    def to_json(self, settings: RunSettings, fam: Families) -> str:
        st = settings.to_c()
        off = np.ascontiguousarray(fam.fam_offsets, dtype=np.uint64)
        sds = np.ascontiguousarray(fam.sds, dtype=PROTOSD_DTYPE)
        p = self.L.asgart_b200_to_json(self.h, C.byref(st), _ptr(off), len(off) - 1, _ptr(sds))
        try:
            return C.string_at(p).decode()
        finally:
            self.L.asgart_b200_free_string(p)

    def close(self):
        if getattr(self, "h", None):
            self.strand = None
            self.L.asgart_b200_prepared_free(self.h)
            self.h = None

    __del__ = close


def prepare_data(files: Sequence[str], skip_masked: bool = False) -> Prepared:
    return Prepared.from_files(files, skip_masked)


def normalise(seq: np.ndarray, skip_masked: bool) -> np.ndarray:
    """Per-base normalisation of read_fasta (src/bin/asgart.rs:291-301), vectorised for in-memory inputs."""
    # one 256-entry table: lower case -> 'N' (skip_masked) or upper case, then anything outside ATGCN -> 'N'
    table = np.full(256, ord("N"), dtype=np.uint8)
    for c in b"ATGCN":
        table[c] = c
    if not skip_masked:
        for c in b"atgcn":
            table[c] = c - 32
    seq = np.ascontiguousarray(seq, dtype=np.uint8)
    out = np.empty_like(seq)
    step = 1 << 24
    offs = range(0, len(seq), step)
    if len(offs) > 1:   # numpy drops the GIL inside take
        import os
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(max_workers=min(len(offs), os.cpu_count() or 1)) as ex:
            list(ex.map(lambda o: np.take(table, seq[o:o + step], out=out[o:o + step]), offs))
    else:
        np.take(table, seq, out=out)
    return out


def out_filename(files: Sequence[str], settings: RunSettings, prefix: str = "", out: Optional[str] = None) -> str:
    L = _lib.load()
    st = settings.to_c()
    p = L.asgart_b200_out_filename("\n".join(files).encode(), prefix.encode(), out.encode() if out else None, C.byref(st))
    try:
        return C.string_at(p).decode()
    finally:
        L.asgart_b200_free_string(p)


def search_duplications(files: Sequence[str], settings: RunSettings, device: int = 0) -> str:
    """The whole `asgart FILES...` run (src/bin/asgart.rs:731-822) -> JSON text as JSONExporter::save writes it."""
    L = _lib.load()
    st = settings.to_c()
    err = C.c_char_p()
    p = L.asgart_b200_run_files("\n".join(files).encode(), C.byref(st), device, C.byref(err))
    if not p:
        raise AsgartB200Error(-1, err.value.decode() if err.value else "run failed")
    try:
        return C.string_at(p).decode()
    finally:
        L.asgart_b200_free_string(p)


def search_duplications_passes(files: Sequence[str], passes: Sequence[RunSettings], device: int = 0) -> str:
    """Several runs (e.g. direct and -RC) over one index, combined as `asgart-slice` combines their JSON files
    (RunResult::from_files, src/structs.rs:114-141): strand and settings of the first pass, families concatenated."""
    L = _lib.load()
    arr = (_lib.Settings * len(passes))(*[p.to_c() for p in passes])
    err = C.c_char_p()
    p = L.asgart_b200_run_files_passes("\n".join(files).encode(), arr, len(passes), device, C.byref(err))
    if not p:
        raise AsgartB200Error(-1, err.value.decode() if err.value else "run failed")
    try:
        return C.string_at(p).decode()
    finally:
        L.asgart_b200_free_string(p)


# ---------------------------------------------------------------------------------------------- synthetic inputs
def synth_genome(config: int, part: int = 0, scale_n: int = 0, seed: int = 1, n_pairs: int = 0, rc_percent: int = 0,
                 threads: int = 8, out: Optional[np.ndarray] = None):
    """Deterministic synthetic genome of BASELINE config C<config> (0 = custom). Returns (bases uint8[n] with case and N,
    fragments [(name, position, length)])."""
    L = _lib.load()
    n = L.asgart_b200_synth_length(config, part, scale_n)
    if n < 0:
        raise ValueError("unknown synthetic config")
    if out is None:
        out = np.empty(n, dtype=np.uint8)
    assert out.dtype == np.uint8 and len(out) >= n
    got = L.asgart_b200_synth_fill(config, part, scale_n, seed, n_pairs, rc_percent, _ptr(out), len(out), threads)
    assert got == n
    names = C.create_string_buffer(4096)
    pos = np.zeros(64, dtype=np.uint64)
    ln = np.zeros(64, dtype=np.uint64)
    nf = L.asgart_b200_synth_fragments(config, part, scale_n, names, 4096, _ptr(pos), _ptr(ln), 64)
    nm = names.value.decode().split("\n")
    return out[:n], [(nm[i], int(pos[i]), int(ln[i])) for i in range(nf)]
