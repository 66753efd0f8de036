"""ctypes binding of libasgart_b200.so (the C ABI of include/asgart_b200.h). No torch types cross this boundary.

The library is built in-tree by ``__graft_entry__.build()`` / ``make -C asgart_b200/csrc``. Loading fails loudly when it
is missing: there is no Python or CPU fallback for any compute entry point.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libasgart_b200.so")

OK, EINVAL, ENOMEM, ECUDA, ESTATE, ENODEVICE, EPANIC = 0, -1, -2, -3, -4, -5, -6
POST_FILTER_NS, POST_REORDER, POST_REDUCE_OVERLAP, POST_SORT, POST_ALL = 1, 2, 4, 8, 15
POST_COMPUTE_SCORE = 16
LUT_SIZE = 390625
SLICE_NO_DIRECT, SLICE_NO_REVERSED, SLICE_NO_UNCOMPLEMENTED, SLICE_NO_COMPLEMENTED, SLICE_NO_INTER, SLICE_NO_INTRA, SLICE_MIN_LENGTH = 1, 2, 4, 8, 16, 32, 64
SLICE_COLLAPSE, SLICE_NO_INTER_RELAXED, SLICE_REGEXP = 128, 256, 512


class SliceOptions(C.Structure):
    _fields_ = [("flags", C.c_uint32), ("reserved", C.c_uint32), ("min_length", C.c_uint64), ("max_family_members", C.c_int64),
                ("keep_fragments", C.c_char_p), ("restrict_fragments", C.c_char_p), ("exclude_fragments", C.c_char_p)]


class Settings(C.Structure):
    """asgart_b200_settings == RunSettings (src/structs.rs:36-58); max_gap_size already includes probe_size."""
    _fields_ = [
        ("probe_size", C.c_uint64),
        ("max_gap_size", C.c_uint32),
        ("reverse", C.c_uint32),
        ("complement", C.c_uint32),
        ("skip_masked", C.c_uint32),
        ("min_duplication_length", C.c_uint64),
        ("max_cardinality", C.c_uint64),
        ("has_trim", C.c_uint32),
        ("compute_score", C.c_uint32),
        ("trim_a", C.c_uint64),
        ("trim_b", C.c_uint64),
    ]


class Chunk(C.Structure):
    _fields_ = [("start", C.c_uint64), ("length", C.c_uint64)]


class ProtoSD(C.Structure):
    _fields_ = [
        ("left", C.c_uint64),
        ("right", C.c_uint64),
        ("left_length", C.c_uint64),
        ("right_length", C.c_uint64),
        ("identity", C.c_float),
        ("reversed", C.c_uint8),
        ("complemented", C.c_uint8),
        ("_pad", C.c_uint8 * 2),
    ]


class Stats(C.Structure):
    _fields_ = (
        [(n, C.c_double) for n in ("ms_h2d", "ms_pack", "ms_sa_build", "ms_lut", "ms_search", "ms_automaton", "ms_post",
                                   "ms_d2h", "ms_sa_sort", "ms_sa_gather", "ms_sa_rank", "ms_probe", "ms_emit", "ms_sa_scatter")]
        + [(n, C.c_uint64) for n in ("launches_total", "launches_sa_sort", "launches_sa_gather", "launches_probe",
                                     "launches_sa_scatter", "bytes_sa_sort", "bytes_sa_gather", "bytes_probe",
                                     "bytes_sa_scatter", "n_probes", "n_searched",
                                     "n_skipped_n", "n_skipped_card", "n_matches", "n_events", "n_segments", "sa_rounds",
                                     "sa_index_bits", "h2d_bytes", "d2h_bytes")]
        + [("ms_sa_scatter_main", C.c_double), ("launches_sa_scatter_main", C.c_uint64), ("bytes_sa_scatter_main", C.c_uint64)]
        + [("ms_score", C.c_double), ("score_cells", C.c_uint64), ("score_pairs", C.c_uint64)]
        + [("ms_ingest", C.c_double), ("ingest_bytes", C.c_uint64), ("ingest_records", C.c_uint64)]
        + [(n, C.c_double) for n in ("ms_msd_scatter0", "ms_msd_hist", "ms_msd_local")]
        + [(n, C.c_uint64) for n in ("bytes_msd_scatter0", "bytes_msd_hist", "bytes_msd_local", "launches_msd_local", "msd_levels")]
        + [("ms_locate", C.c_double)] + [(n, C.c_uint64) for n in ("locate_patterns", "locate_hits", "bytes_locate")]
    )

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


# every symbol include/asgart_b200.h declares (tests check the library exports all of them)
SYMBOLS = [
    "asgart_b200_divsufsort64", "asgart_b200_divsufsort64_ex", "asgart_b200_version", "asgart_b200_device_count",
    "asgart_b200_ctx_create", "asgart_b200_ctx_destroy", "asgart_b200_ctx_last_error", "asgart_b200_ctx_load_strand",
    "asgart_b200_ctx_build_index", "asgart_b200_ctx_set_index_bits", "asgart_b200_ctx_upload_sa",
    "asgart_b200_ctx_download_sa", "asgart_b200_ctx_check_sa", "asgart_b200_ctx_sa_fingerprint", "asgart_b200_ctx_download_lut", "asgart_b200_ctx_search",
    "asgart_b200_ctx_probe_ranges", "asgart_b200_ctx_search_shard", "asgart_b200_partial_size",
    "asgart_b200_partial_serialize", "asgart_b200_partial_free", "asgart_b200_ctx_finish",
    "asgart_b200_ctx_search_shard_dev", "asgart_b200_ctx_finish_dev",
    "asgart_b200_result_n_families", "asgart_b200_result_n_sds", "asgart_b200_result_family_offsets",
    "asgart_b200_result_sds", "asgart_b200_result_free", "asgart_b200_ctx_post_steps", "asgart_b200_ctx_stats",
    "asgart_b200_ctx_reset_stats", "asgart_b200_ctx_probe_keys", "asgart_b200_ctx_timer_start", "asgart_b200_ctx_timer_stop", "asgart_b200_prepare_files", "asgart_b200_prepare_memory",
    "asgart_b200_prepared_strand", "asgart_b200_prepared_chunks", "asgart_b200_prepared_n_fragments",
    "asgart_b200_prepared_fragment", "asgart_b200_prepared_free", "asgart_b200_to_json", "asgart_b200_free_string",
    "asgart_b200_out_filename", "asgart_b200_run_files", "asgart_b200_synth_length", "asgart_b200_synth_fill",
    "asgart_b200_synth_fragments",
    "asgart_b200_build_index_group", "asgart_b200_dist_unique_id", "asgart_b200_ctx_dist_init", "asgart_b200_ctx_dist_shutdown",
    "asgart_b200_ctx_ingest_begin", "asgart_b200_ctx_ingest_fasta", "asgart_b200_ctx_ingest_file",
    "asgart_b200_ctx_ingest_finish", "asgart_b200_ctx_download_strand", "asgart_b200_run_files_passes",
    "asgart_b200_ctx_build_index_trim", "asgart_b200_effective_trim", "asgart_b200_slice_families",
    "asgart_b200_run_files_sliced", "asgart_b200_run_files_sliced_ex", "asgart_b200_run_result_new", "asgart_b200_run_result_slice",
    "asgart_b200_run_result_to_json", "asgart_b200_run_result_error", "asgart_b200_run_result_free",
    "asgart_b200_ctx_locate", "asgart_b200_hits_n_patterns", "asgart_b200_hits_first", "asgart_b200_hits_count",
    "asgart_b200_hits_offsets", "asgart_b200_hits_positions", "asgart_b200_hits_free",
]

_lib = None


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` or "
            "`make -C asgart_b200/csrc`. asgart_b200 has no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, u32 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32
    PS = C.POINTER(Settings)
    sig = {
        "asgart_b200_divsufsort64": (i32, [vp, vp, i64]),
        "asgart_b200_divsufsort64_ex": (i32, [vp, vp, i64, i32, i32]),
        "asgart_b200_version": (C.c_char_p, []),
        "asgart_b200_device_count": (i32, []),
        "asgart_b200_ctx_create": (i32, [i32, C.POINTER(vp)]),
        "asgart_b200_ctx_destroy": (None, [vp]),
        "asgart_b200_ctx_last_error": (C.c_char_p, [vp]),
        "asgart_b200_ctx_load_strand": (i32, [vp, vp, i64]),
        "asgart_b200_ctx_build_index": (i32, [vp]),
        "asgart_b200_ctx_set_index_bits": (i32, [vp, i32]),
        "asgart_b200_ctx_build_index_trim": (i32, [vp, C.c_uint64, C.c_uint64]),
        "asgart_b200_effective_trim": (i32, [C.c_uint64, C.c_uint64, i64, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
        "asgart_b200_build_index_group": (i32, [C.POINTER(vp), i32]),
        "asgart_b200_dist_unique_id": (i32, [vp, i64]),
        "asgart_b200_ctx_dist_init": (i32, [vp, i32, i32, vp, i64]),
        "asgart_b200_ctx_dist_shutdown": (i32, [vp]),
        "asgart_b200_ctx_ingest_begin": (i32, [vp]),
        "asgart_b200_ctx_ingest_fasta": (i32, [vp, vp, i64, i32]),
        "asgart_b200_ctx_ingest_file": (i32, [vp, C.c_char_p, i32]),
        "asgart_b200_ctx_ingest_finish": (i32, [vp, C.c_char_p, C.POINTER(vp)]),
        "asgart_b200_ctx_download_strand": (i32, [vp, vp, i64]),
        "asgart_b200_ctx_upload_sa": (i32, [vp, vp]),
        "asgart_b200_ctx_download_sa": (i32, [vp, vp]),
        "asgart_b200_ctx_check_sa": (i32, [vp, vp]),
        "asgart_b200_ctx_sa_fingerprint": (i32, [vp, vp]),
        "asgart_b200_ctx_download_lut": (i32, [vp, vp, vp]),
        "asgart_b200_ctx_search": (i32, [vp, vp, i64, PS, u32, C.POINTER(vp)]),
        "asgart_b200_ctx_probe_ranges": (i32, [vp, vp, PS, vp, vp, i64]),
        "asgart_b200_ctx_locate": (i32, [vp, vp, vp, i64, i64, C.POINTER(vp)]),
        "asgart_b200_hits_n_patterns": (i64, [vp]),
        "asgart_b200_hits_first": (vp, [vp]),
        "asgart_b200_hits_count": (vp, [vp]),
        "asgart_b200_hits_offsets": (vp, [vp]),
        "asgart_b200_hits_positions": (vp, [vp]),
        "asgart_b200_hits_free": (None, [vp]),
        "asgart_b200_ctx_search_shard": (i32, [vp, vp, i64, PS, i32, i32, C.POINTER(vp)]),
        "asgart_b200_partial_size": (i64, [vp]),
        "asgart_b200_partial_serialize": (i32, [vp, vp, i64]),
        "asgart_b200_partial_free": (None, [vp]),
        "asgart_b200_ctx_search_shard_dev": (i32, [vp, vp, i64, PS, i32, i32, C.POINTER(vp), C.POINTER(i64), vp]),
        "asgart_b200_ctx_finish_dev": (i32, [vp, vp, i64, PS, C.POINTER(vp), vp, i32, u32, C.POINTER(vp)]),
        "asgart_b200_ctx_finish": (i32, [vp, vp, i64, PS, C.POINTER(vp), C.POINTER(i64), i32, u32, C.POINTER(vp)]),
        "asgart_b200_result_n_families": (i64, [vp]),
        "asgart_b200_result_n_sds": (i64, [vp]),
        "asgart_b200_result_family_offsets": (vp, [vp]),
        "asgart_b200_result_sds": (vp, [vp]),
        "asgart_b200_result_free": (None, [vp]),
        "asgart_b200_ctx_post_steps": (i32, [vp, vp, i64, vp, u32, C.POINTER(vp)]),
        "asgart_b200_ctx_stats": (i32, [vp, C.POINTER(Stats)]),
        "asgart_b200_ctx_reset_stats": (None, [vp]),
        "asgart_b200_ctx_probe_keys": (C.c_uint64, [vp]),
        "asgart_b200_ctx_timer_start": (i32, [vp]),
        "asgart_b200_ctx_timer_stop": (i32, [vp, C.POINTER(C.c_double)]),
        "asgart_b200_prepare_files": (vp, [C.c_char_p, i32, C.POINTER(C.c_char_p)]),
        "asgart_b200_prepare_memory": (vp, [C.c_char_p, vp, i64, C.c_char_p, vp, vp, i64]),
        "asgart_b200_prepared_strand": (vp, [vp, C.POINTER(i64)]),
        "asgart_b200_prepared_chunks": (vp, [vp, C.POINTER(i64)]),
        "asgart_b200_prepared_n_fragments": (i64, [vp]),
        "asgart_b200_prepared_fragment": (C.c_char_p, [vp, i64, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
        "asgart_b200_prepared_free": (None, [vp]),
        "asgart_b200_to_json": (vp, [vp, PS, vp, i64, vp]),
        "asgart_b200_free_string": (None, [vp]),
        "asgart_b200_slice_families": (i32, [vp, vp, i64, vp, u32, C.c_uint64, i64, C.POINTER(vp)]),
        "asgart_b200_out_filename": (vp, [C.c_char_p, C.c_char_p, C.c_char_p, PS]),
        "asgart_b200_run_files": (vp, [C.c_char_p, PS, i32, C.POINTER(C.c_char_p)]),
        "asgart_b200_run_files_passes": (vp, [C.c_char_p, PS, i32, i32, C.POINTER(C.c_char_p)]),
        "asgart_b200_run_files_sliced": (vp, [C.c_char_p, PS, i32, i32, u32, C.c_uint64, i64, C.POINTER(C.c_char_p)]),
        "asgart_b200_run_files_sliced_ex": (vp, [C.c_char_p, PS, i32, i32, C.POINTER(SliceOptions), C.POINTER(C.c_char_p)]),
        "asgart_b200_run_result_new": (vp, [vp, PS, vp, i64, vp]),
        "asgart_b200_run_result_slice": (i32, [vp, C.POINTER(SliceOptions)]),
        "asgart_b200_run_result_to_json": (vp, [vp]),
        "asgart_b200_run_result_error": (C.c_char_p, [vp]),
        "asgart_b200_run_result_free": (None, [vp]),
        "asgart_b200_synth_length": (i64, [i32, i32, i64]),
        "asgart_b200_synth_fill": (i64, [i32, i32, i64, C.c_uint64, i64, i32, vp, i64, i32]),
        "asgart_b200_synth_fragments": (i64, [i32, i32, i64, vp, i64, vp, vp, i64]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L
