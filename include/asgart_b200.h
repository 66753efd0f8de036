/* asgart_b200.h — C ABI of the B200-native duplication-search hot path.
 *
 * This is the drop-in boundary for delehef/asgart (reference @ 523b07c; citations relative to its root).
 * The reference has exactly one native boundary today, `src/divsufsort.rs:8-33` (extern "C" over the
 * libdivsufsort static library that build.rs:4-16 builds); this header is what a `build.rs` + `extern "C"`
 * block would bind instead. Plain pointers and sizes only; all buffers passed in are caller-owned and are
 * not retained after the call returns; results are library-owned and freed with asgart_b200_result_free.
 *
 * Two levels:
 *   (1) asgart_b200_divsufsort64 — literal replacement for `divsufsort64` (src/divsufsort.rs:10, called from
 *       r_divsufsort, src/bin/asgart.rs:473-479).
 *   (2) a handle-based operator that replaces the *body* of SearchDuplications::run
 *       (src/bin/asgart.rs:137-258: SA build :149, Searcher::new :151, chunk fan-out :201-240, flatten :241-253)
 *       and, optionally, the FilterNs / ReOrder / ReduceOverlap / Sort steps (:33-96, :481-562). Per-probe FFI
 *       (Searcher::search, src/searcher.rs:145) is deliberately NOT exposed: the probe loop lives on the GPU.
 *
 * There is no CPU fallback: every compute entry point returns ASGART_B200_ENODEVICE when no CUDA device is usable.
 * A context is not thread-safe (one caller thread at a time); kernels run on a library-owned stream.
 */
#ifndef ASGART_B200_H
#define ASGART_B200_H 1

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ASGART_B200_API __attribute__((visibility("default")))

/* ---- status codes: 0 / -1 / -2 keep divsufsort64's meaning (libdivsufsort/lib/divsufsort.c:337-357) ---- */
#define ASGART_B200_OK          0
#define ASGART_B200_EINVAL     (-1)  /* bad arguments (NULL, negative size, strand not normalised, k out of range) */
#define ASGART_B200_ENOMEM     (-2)  /* host or device allocation failed */
#define ASGART_B200_ECUDA      (-3)  /* CUDA runtime error; see asgart_b200_ctx_last_error */
#define ASGART_B200_ESTATE     (-4)  /* call order violated (e.g. search before build_index) */
#define ASGART_B200_ENODEVICE  (-5)  /* no usable CUDA device: the product has no CPU path */
#define ASGART_B200_EPANIC     (-6)  /* the reference itself panics on this input (last_error says where) */

/* ---- (1) drop-in for divsufsort64 (src/divsufsort.rs:10) ------------------------------------------------
 * T[0..n) any bytes, SA[0..n) output, both host memory. Suffix array built on the current CUDA device by
 * prefix doubling (hand-written radix sort + rank update); bit-identical to divsufsort64's output because the
 * suffix array of a text is unique. */
ASGART_B200_API int32_t asgart_b200_divsufsort64(const uint8_t *T, int64_t *SA, int64_t n);
/* same, on an explicit device and with the index width forced (0 = auto, 32 or 64) — for tests */
ASGART_B200_API int32_t asgart_b200_divsufsort64_ex(const uint8_t *T, int64_t *SA, int64_t n, int32_t device,
                                                    int32_t index_bits);
/* replaces divsufsort64_version (src/divsufsort.rs:11) */
ASGART_B200_API const char *asgart_b200_version(void);

/* ---- (2) the search operator ---------------------------------------------------------------------------- */
typedef struct asgart_b200_ctx asgart_b200_ctx;
typedef struct asgart_b200_result asgart_b200_result;
typedef struct asgart_b200_partial asgart_b200_partial;

/* mirror of RunSettings (src/structs.rs:36-58). max_gap_size is ALREADY gap_size + probe_size
 * (src/bin/asgart.rs:681). threads_count has no meaning here; compute_score is the
 * post-step bit ASGART_B200_POST_COMPUTE_SCORE. trim holds the RAW command-line values (they go into the
 * JSON settings block as they are, src/bin/asgart.rs:691); asgart_b200_run_files builds the trimmed index from them
 * (asgart_b200_ctx_build_index_trim), ctx_search itself does not look at them. */
typedef struct asgart_b200_settings {
    uint64_t probe_size;
    uint32_t max_gap_size;
    uint32_t reverse;
    uint32_t complement;
    uint32_t skip_masked;
    uint64_t min_duplication_length;
    uint64_t max_cardinality;
    uint32_t has_trim;
    uint32_t compute_score;   /* --compute-score (src/structs.rs:57): asgart_b200_run_files adds the ComputeScore step.
                                 Sits in what used to be alignment padding: the struct keeps its 64 bytes. */
    uint64_t trim_a, trim_b;
} asgart_b200_settings;

/* one entry of chunks_to_process (src/bin/asgart.rs:115, :317-366): global start, length */
typedef struct asgart_b200_chunk {
    uint64_t start;
    uint64_t length;
} asgart_b200_chunk;

/* mirror of ProtoSD (src/structs.rs:418-429) */
typedef struct asgart_b200_protosd {
    uint64_t left;
    uint64_t right;
    uint64_t left_length;
    uint64_t right_length;
    float identity;
    uint8_t reversed;
    uint8_t complemented;
    uint8_t _pad[2];
} asgart_b200_protosd;

/* post-step selection for asgart_b200_ctx_search (applied in the reference's order, src/bin/asgart.rs:738-747) */
#define ASGART_B200_POST_FILTER_NS       1u  /* FilterNs      src/bin/asgart.rs:81-96, src/structs.rs:454-467 */
#define ASGART_B200_POST_REORDER         2u  /* ReOrder       src/bin/asgart.rs:33-51 */
#define ASGART_B200_POST_REDUCE_OVERLAP  4u  /* ReduceOverlap src/bin/asgart.rs:67-79, :481-562 */
#define ASGART_B200_POST_SORT            8u  /* Sort          src/bin/asgart.rs:53-65 */
#define ASGART_B200_POST_ALL            15u  /* the reference's default pipeline */
/* ComputeScore (--compute-score): src/bin/asgart.rs:98-111, ProtoSD::levenshtein src/structs.rs:439-452. identity =
 * 100 * (1 - levenshtein(left arm, right arm reversed then complemented per the flags) / max(left_length, right_length)),
 * arms taken as the reference takes them (inclusive ranges, length + 1 bytes), f64 arithmetic cast to f32 once.
 * Bit-parallel (Myers/Hyyro) global edit distance on the GPU, one thread block per duplicon. */
#define ASGART_B200_POST_COMPUTE_SCORE  16u

/* lifetime */
ASGART_B200_API int32_t asgart_b200_device_count(void);
ASGART_B200_API int32_t asgart_b200_ctx_create(int32_t device, asgart_b200_ctx **out);
ASGART_B200_API void asgart_b200_ctx_destroy(asgart_b200_ctx *ctx);
ASGART_B200_API const char *asgart_b200_ctx_last_error(const asgart_b200_ctx *ctx);

/* Strand = what prepare_data produces (src/bin/asgart.rs:273-471): bytes in {A,C,G,N,T} followed by one '$'
 * (n_plus_1 bytes, host memory; pinned memory makes the copy asynchronous). Copies to the device and packs it.
 * In a context that joined a group (asgart_b200_ctx_dist_init) the call is collective: every rank passes the same strand,
 * copies 1/world of it to its device and the ranks exchange the pieces over NVLink. */
ASGART_B200_API int32_t asgart_b200_ctx_load_strand(asgart_b200_ctx *ctx, const uint8_t *T, int64_t n_plus_1);
/* Suffix array (replaces r_divsufsort, :149) + 8-mer LUT (replaces Searcher::new, :151; src/searcher.rs:99-143) */
ASGART_B200_API int32_t asgart_b200_ctx_build_index(asgart_b200_ctx *ctx);
/* The index of a `--trim start stop` run (src/bin/asgart.rs:142-147): suffix array of strand[start..stop] + '$' with every
 * entry shifted by start (stop - start + 1 entries; ctx_download_sa returns that many), while the LUT and every
 * comparison of the search read the WHOLE strand, exactly as the reference does (SURVEY Q9: near `stop` the array is not
 * sorted for what it is compared with, so the LUT comes from the reference's own sa_search bisection run step for step on
 * the device, and every probe takes the literal lock-step search). Only duplications whose right arm lies inside the
 * slice are found; chunks are NOT trimmed. start < stop <= n: pass the values through asgart_b200_effective_trim first,
 * which restates prepare_data's clamping (src/bin/asgart.rs:432-463) — it returns 0 when the reference skips trimming
 * (then call ctx_build_index). One device only. */
ASGART_B200_API int32_t asgart_b200_ctx_build_index_trim(asgart_b200_ctx *ctx, uint64_t start, uint64_t stop);
ASGART_B200_API int32_t asgart_b200_effective_trim(uint64_t start, uint64_t stop, int64_t n_plus_1, uint64_t *eff_start,
                                                   uint64_t *eff_stop);
/* Sharded index build (the reference builds its suffix array on one thread, src/bin/asgart.rs:473-479, and has no
 * multi-device mode): the members of a group split the suffixes by initial-key range, keep the rank array block-cyclic
 * in each other's memory (peer stores / loads over NVLink) and end with the whole index on every member, bit-identical
 * to a single-device build. Every member must have the same strand loaded.
 *   one process, several contexts (any devices with peer access, or all on one device): build_index_group runs the
 *     members on host threads;
 *   one process per GPU: rank 0 makes a unique id (dist_unique_id, 128 bytes) and sends it to the others by any means
 *     (asgart_b200/dist.py: torch.distributed broadcast); every rank calls ctx_dist_init, after which ctx_build_index is
 *     a collective call (NCCL for the phase boundaries and the final exchange of SA pieces, CUDA IPC for the peer
 *     pointers) until ctx_dist_shutdown. */
ASGART_B200_API int32_t asgart_b200_build_index_group(asgart_b200_ctx *const *ctxs, int32_t world);
ASGART_B200_API int32_t asgart_b200_dist_unique_id(uint8_t *out, int64_t cap);   /* returns the id size (128) */
ASGART_B200_API int32_t asgart_b200_ctx_dist_init(asgart_b200_ctx *ctx, int32_t rank, int32_t world,
                                                  const uint8_t *unique_id, int64_t id_bytes);
ASGART_B200_API int32_t asgart_b200_ctx_dist_shutdown(asgart_b200_ctx *ctx);
/* force the suffix-index width of the next build_index / upload_sa: 0 = auto (32 bits when n+1 < 2^32-1), 32, 64 */
ASGART_B200_API int32_t asgart_b200_ctx_set_index_bits(asgart_b200_ctx *ctx, int32_t bits);
/* test hooks: use a suffix array built elsewhere (still builds the LUT on the device) / read the index back */
ASGART_B200_API int32_t asgart_b200_ctx_upload_sa(asgart_b200_ctx *ctx, const int64_t *SA);
ASGART_B200_API int32_t asgart_b200_ctx_download_sa(asgart_b200_ctx *ctx, int64_t *SA);
/* On-device restatement of sufcheck (libdivsufsort/lib/utils.c:159-241; the reference's only self-check,
 * examples/suftest.c:146-157): SA must be a permutation of [0, n] and every adjacent pair must be in suffix order
 * (first symbols, then the ranks of the two suffixes one symbol further on). *n_bad = number of violations (0 = valid).
 * Lets a genome-scale index be validated without a CPU-side suffix array. */
ASGART_B200_API int32_t asgart_b200_ctx_check_sa(asgart_b200_ctx *ctx, int64_t *n_bad);
/* Order-sensitive 64-bit fingerprint of the suffix array, computed on the device: sum over i of
 * splitmix64(SA[i] + i * 0x9E3779B97F4A7C15) mod 2^64. Lets a genome-scale index be compared with the output of the
 * reference's divsufsort64 (src/divsufsort.rs:10) through one number instead of a 25 GB download. */
ASGART_B200_API int32_t asgart_b200_ctx_sa_fingerprint(asgart_b200_ctx *ctx, uint64_t *fingerprint);
/* LUT as 5^8 (lo, hi) pairs indexed by the 8-mer read as a base-5 number with digits A=0,C=1,G=2,N=3,T=4 (first
 * letter most significant). Empty buckets have lo == hi (value unspecified). */
#define ASGART_B200_LUT_SIZE 390625
ASGART_B200_API int32_t asgart_b200_ctx_download_lut(asgart_b200_ctx *ctx, int64_t *lo, int64_t *hi);

/* SearchDuplications::run body + selected post-steps. Families come back in the reference's order:
 * chunk order, then flush order, then arm-creation order (src/bin/asgart.rs:241-253, src/automaton.rs:182-200). */
ASGART_B200_API int32_t asgart_b200_ctx_search(asgart_b200_ctx *ctx, const asgart_b200_chunk *chunks, int64_t n_chunks,
                                               const asgart_b200_settings *settings, uint32_t post_mask,
                                               asgart_b200_result **out);
/* Searcher::search for a batch of probes taken from the strand itself — test hook for the probe kernel:
 * probe p is the probe_size-mer the reference would cut at needle index i = (p+1)*(probe_size/2) of chunk 0 under
 * `settings` (src/automaton.rs:96-104). Writes the equal range [lo, hi) in the SA for each (unfiltered). */
ASGART_B200_API int32_t asgart_b200_ctx_probe_ranges(asgart_b200_ctx *ctx, const asgart_b200_chunk *chunk,
                                                     const asgart_b200_settings *settings, int64_t *lo, int64_t *hi,
                                                     int64_t n_probes);

/* ---- exact-match queries against the resident index ------------------------------------------------------------
 * sa_search64 (libdivsufsort/lib/utils.c:282-349; bound by the reference at src/divsufsort.rs) for a batch of patterns
 * against the context's index; pattern i = patterns[offsets[i] .. offsets[i+1]) (offsets: n_patterns + 1 entries,
 * non-decreasing). Patterns are any bytes, compared as bytes (_compare, utils.c:244-255; a suffix that ends inside the
 * pattern is smaller). Per pattern: count = number of suffixes that start with it, SA[first .. first + count) = those
 * suffixes; count == 0: first = the reference's insertion point; the empty pattern: first 0, count = entries of the index.
 * On an index built with --trim the answer is the one the reference's own bisection lands on (that array is not sorted
 * for the whole strand it is compared with, SURVEY Q9).
 * max_hits: positions reported per pattern (< 0 all, 0 counts only): SA[first .. first + min(count, max_hits)), in SA
 * order; count itself is never capped. After build_index / build_index_trim / upload_sa. Device memory beyond the index
 * stays bounded (patterns are taken in slices); ASGART_B200_ENOMEM when the positions do not fit in host memory. */
typedef struct asgart_b200_hits asgart_b200_hits;
ASGART_B200_API int32_t asgart_b200_ctx_locate(asgart_b200_ctx *ctx, const uint8_t *patterns, const uint64_t *offsets,
                                               int64_t n_patterns, int64_t max_hits, asgart_b200_hits **out);
ASGART_B200_API int64_t asgart_b200_hits_n_patterns(const asgart_b200_hits *h);
ASGART_B200_API const int64_t *asgart_b200_hits_first(const asgart_b200_hits *h);      /* n_patterns */
ASGART_B200_API const int64_t *asgart_b200_hits_count(const asgart_b200_hits *h);      /* n_patterns, uncapped */
ASGART_B200_API const uint64_t *asgart_b200_hits_offsets(const asgart_b200_hits *h);   /* n_patterns + 1 */
ASGART_B200_API const int64_t *asgart_b200_hits_positions(const asgart_b200_hits *h);  /* offsets[n_patterns] */
ASGART_B200_API void asgart_b200_hits_free(asgart_b200_hits *h);

/* Multi-GPU (one process per GPU; strand + index replicated; probes partitioned by position):
 *   every rank: ctx_search_shard(rank, world) -> partial; exchange the serialised partials (NCCL all-gather);
 *   any rank:   ctx_finish(partials[world]) -> families (identical on every rank and for every world size). */
ASGART_B200_API int32_t asgart_b200_ctx_search_shard(asgart_b200_ctx *ctx, const asgart_b200_chunk *chunks,
                                                     int64_t n_chunks, const asgart_b200_settings *settings,
                                                     int32_t shard, int32_t n_shards, asgart_b200_partial **out);
ASGART_B200_API int64_t asgart_b200_partial_size(const asgart_b200_partial *p);           /* bytes when serialised */
ASGART_B200_API int32_t asgart_b200_partial_serialize(const asgart_b200_partial *p, uint8_t *buf, int64_t cap);
ASGART_B200_API void asgart_b200_partial_free(asgart_b200_partial *p);
ASGART_B200_API int32_t asgart_b200_ctx_finish(asgart_b200_ctx *ctx, const asgart_b200_chunk *chunks, int64_t n_chunks,
                                               const asgart_b200_settings *settings, const uint8_t *const *partials,
                                               const int64_t *partial_sizes, int32_t n_shards, uint32_t post_mask,
                                               asgart_b200_result **out);
/* Device-resident form of the same exchange (what asgart_b200/dist.py uses under NCCL): the partial stays in HBM as one
 * blob owned by the context (valid until its next search_shard_dev call), meta[4] = {p_begin, p_end, events, matches}.
 * finish_dev takes, per shard, a device pointer to that shard's blob (any device memory of this GPU, e.g. the output of
 * an NCCL all-gather) and its 4 meta words. */
ASGART_B200_API int32_t asgart_b200_ctx_search_shard_dev(asgart_b200_ctx *ctx, const asgart_b200_chunk *chunks,
                                                         int64_t n_chunks, const asgart_b200_settings *settings,
                                                         int32_t shard, int32_t n_shards, void **d_blob,
                                                         int64_t *blob_bytes, uint64_t *meta);
ASGART_B200_API int32_t asgart_b200_ctx_finish_dev(asgart_b200_ctx *ctx, const asgart_b200_chunk *chunks, int64_t n_chunks,
                                                   const asgart_b200_settings *settings, const void *const *d_blobs,
                                                   const uint64_t *metas, int32_t n_shards, uint32_t post_mask,
                                                   asgart_b200_result **out);

/* results */
ASGART_B200_API int64_t asgart_b200_result_n_families(const asgart_b200_result *r);
ASGART_B200_API int64_t asgart_b200_result_n_sds(const asgart_b200_result *r);
ASGART_B200_API const uint64_t *asgart_b200_result_family_offsets(const asgart_b200_result *r); /* n_families+1 */
ASGART_B200_API const asgart_b200_protosd *asgart_b200_result_sds(const asgart_b200_result *r);
ASGART_B200_API void asgart_b200_result_free(asgart_b200_result *r);

/* post-steps on caller-provided families (host arrays in, library-owned result out) — FilterNs needs the strand
 * loaded in ctx */
ASGART_B200_API int32_t asgart_b200_ctx_post_steps(asgart_b200_ctx *ctx, const uint64_t *family_offsets,
                                                   int64_t n_families, const asgart_b200_protosd *sds,
                                                   uint32_t post_mask, asgart_b200_result **out);

/* ---- instrumentation (device time from CUDA events on the library's stream) ------------------------------ */
typedef struct asgart_b200_stats {
    /* phases of the last load/build/search, milliseconds */
    double ms_h2d, ms_pack, ms_sa_build, ms_lut, ms_search, ms_automaton, ms_post, ms_d2h;
    /* kernel families inside them: accumulated device ms, launches and algorithmic bytes (DESIGN.md) */
    double ms_sa_sort, ms_sa_gather, ms_sa_rank, ms_probe, ms_emit;
    double ms_sa_scatter;          /* rs_scatter_kernel alone (the dominant kernel), inside ms_sa_sort */
    uint64_t launches_total;
    uint64_t launches_sa_sort, launches_sa_gather, launches_probe, launches_sa_scatter;
    uint64_t bytes_sa_sort, bytes_sa_gather, bytes_probe, bytes_sa_scatter;
    /* counters of the last search */
    uint64_t n_probes, n_searched, n_skipped_n, n_skipped_card, n_matches, n_events, n_segments;
    uint64_t sa_rounds, sa_index_bits;
    uint64_t h2d_bytes, d2h_bytes;
    /* rs_scatter_kernel launches of the initial sort only (every launch moves all n+1 suffixes: the roofline kernel) */
    double ms_sa_scatter_main;
    uint64_t launches_sa_scatter_main, bytes_sa_scatter_main;
    /* ComputeScore: device ms, DP cells (sum of arm-length products) and duplicons scored */
    double ms_score;
    uint64_t score_cells, score_pairs;
    /* FASTA ingest: device ms of the scan passes (the file's H2D copy is in ms_h2d / h2d_bytes), file bytes, records */
    double ms_ingest;
    uint64_t ingest_bytes, ingest_records;
    /* initial sort of the suffix-array build in its MSD form (msd_sort.cuh): partition passes over (key, index) pairs
     * (ms_sa_scatter_main / launches / bytes above then describe msd_scatter_kernel, levels >= 1), the first pass that
     * builds the keys from the text, the per-level histograms, the in-shared-memory finishing sort, levels used */
    double ms_msd_scatter0, ms_msd_hist, ms_msd_local;
    uint64_t bytes_msd_scatter0, bytes_msd_hist, bytes_msd_local, launches_msd_local, msd_levels;
    /* asgart_b200_ctx_locate: accumulated device ms of its search and copy kernels, patterns, reported positions and
     * algorithmic bytes (24 B per bisection step, 16 B per further 32 symbols compared, 8 B per reported position) */
    double ms_locate;
    uint64_t locate_patterns, locate_hits, bytes_locate;
} asgart_b200_stats;
ASGART_B200_API int32_t asgart_b200_ctx_stats(const asgart_b200_ctx *ctx, asgart_b200_stats *out);
ASGART_B200_API void asgart_b200_ctx_reset_stats(asgart_b200_ctx *ctx);
/* probes of search and probe_ranges calls since the last reset_stats whose equal range came from the sorted initial keys
 * that a single-device build_index keeps with the index, instead of from suffix-array entries and text windows
 * (0 for a null context) */
ASGART_B200_API uint64_t asgart_b200_ctx_probe_keys(const asgart_b200_ctx *ctx);
/* a CUDA-event stopwatch on the library's stream, for timing a region of calls on the device */
ASGART_B200_API int32_t asgart_b200_ctx_timer_start(asgart_b200_ctx *ctx);
ASGART_B200_API int32_t asgart_b200_ctx_timer_stop(asgart_b200_ctx *ctx, double *elapsed_ms);

/* ---- host side of the path (C++ mirror of prepare_data / SD conversion / JSON export) -------------------- */
typedef struct asgart_b200_prepared asgart_b200_prepared;
/* prepare_data (src/bin/asgart.rs:273-471) for '\n'-separated FASTA paths; NULL + *err (static storage) on error */
ASGART_B200_API asgart_b200_prepared *asgart_b200_prepare_files(const char *files, int32_t skip_masked, const char **err);
/* the same from an in-memory, already normalised strand WITHOUT '$' and its fragment map */
ASGART_B200_API asgart_b200_prepared *asgart_b200_prepare_memory(const char *file_names, const uint8_t *strand, int64_t n,
                                                                 const char *fragment_names, const uint64_t *frag_pos,
                                                                 const uint64_t *frag_len, int64_t n_fragments);
ASGART_B200_API const uint8_t *asgart_b200_prepared_strand(const asgart_b200_prepared *p, int64_t *n_plus_1);
ASGART_B200_API const asgart_b200_chunk *asgart_b200_prepared_chunks(const asgart_b200_prepared *p, int64_t *n_chunks);
ASGART_B200_API int64_t asgart_b200_prepared_n_fragments(const asgart_b200_prepared *p);
ASGART_B200_API const char *asgart_b200_prepared_fragment(const asgart_b200_prepared *p, int64_t i, uint64_t *position,
                                                          uint64_t *length);
ASGART_B200_API void asgart_b200_prepared_free(asgart_b200_prepared *p);
/* RunResult -> JSON exactly as JSONExporter::save writes it (src/exporters.rs:12-25; ProtoSD->SD src/bin/asgart.rs:776-821).
 * Returns a malloc'd NUL-terminated string; free with asgart_b200_free_string. */
ASGART_B200_API char *asgart_b200_to_json(const asgart_b200_prepared *p, const asgart_b200_settings *settings,
                                          const uint64_t *family_offsets, int64_t n_families,
                                          const asgart_b200_protosd *sds);
ASGART_B200_API void asgart_b200_free_string(char *s);
/* default output file name (src/bin/asgart.rs:642-654, :695-719; src/utils.rs:30-49). malloc'd. */
ASGART_B200_API char *asgart_b200_out_filename(const char *files, const char *prefix, const char *out,
                                               const asgart_b200_settings *settings);
/* whole `asgart FILES...` run on one device: prepare_data -> index -> search -> post-steps -> JSON text (malloc'd) */
ASGART_B200_API char *asgart_b200_run_files(const char *files, const asgart_b200_settings *settings, int32_t device,
                                            const char **err);
/* Several passes over ONE index. The reference needs one `asgart` invocation per orientation (-R / -C / -RC runs never
 * report direct duplications, src/bin/asgart.rs:207-218) — each rebuilding the suffix array — and `asgart-slice a.json
 * b.json` to combine them. Here prepare_data and the index are built once, every settings entry is one pass (they must
 * agree on skip_masked, which changes the strand), and the JSON is what RunResult::from_files (src/structs.rs:114-141)
 * gives for the passes' files in this order: strand and settings of the first pass, families of all passes concatenated
 * (SURVEY §8f row N3: the merge itself; asgart-slice's filters are not part of this). */
ASGART_B200_API char *asgart_b200_run_files_passes(const char *files, const asgart_b200_settings *passes, int32_t n_passes,
                                                   int32_t device, const char **err);
/* the same followed by asgart-slice's duplicon filters (asgart_b200_slice_families below) before the JSON is written */
ASGART_B200_API char *asgart_b200_run_files_sliced(const char *files, const asgart_b200_settings *passes, int32_t n_passes,
                                                   int32_t device, uint32_t slice_flags, uint64_t min_length,
                                                   int64_t max_family_members, const char **err);

/* ---- asgart-slice's duplicon filters on families in memory (SURVEY §8f row N3; host code, no device needed) -------
 * What `asgart-slice` applies to a RunResult before it writes it (src/bin/asgart-slice.rs:126-160), in its order:
 * --no-direct / --no-reversed / --no-uncomplemented / --no-complemented (RunResult::remove_*, src/structs.rs:143-169),
 * --no-inter / --no-intra (:171-194; fragment names as the SD conversion assigns them, src/bin/asgart.rs:776-821, so
 * "unknown" for a position outside every fragment), --min-length (min(left_length, right_length) >= it), every one followed
 * by dropping the empty families (so families that were already empty stay when no such filter is given, as in the
 * reference), then --max-family-members (families with more duplicons are dropped, :196-198). min_length counts only with
 * ASGART_B200_SLICE_MIN_LENGTH (`--min-length 0` still drops empty families); max_family_members < 0 = not given. --collapse, --no-inter-relaxed and the
 * fragment selection (--keep/--restrict/--exclude-fragments) rewrite the fragment map: asgart_b200_run_result_slice below. */
#define ASGART_B200_SLICE_NO_DIRECT          1u
#define ASGART_B200_SLICE_NO_REVERSED        2u
#define ASGART_B200_SLICE_NO_UNCOMPLEMENTED  4u
#define ASGART_B200_SLICE_NO_COMPLEMENTED    8u
#define ASGART_B200_SLICE_NO_INTER          16u
#define ASGART_B200_SLICE_NO_INTRA          32u
#define ASGART_B200_SLICE_MIN_LENGTH        64u
#define ASGART_B200_SLICE_COLLAPSE         128u   /* asgart_b200_run_result_slice only */
#define ASGART_B200_SLICE_NO_INTER_RELAXED 256u   /* asgart_b200_run_result_slice only */
#define ASGART_B200_SLICE_REGEXP           512u   /* asgart_b200_run_result_slice only: fragment lists are patterns */
ASGART_B200_API int32_t asgart_b200_slice_families(const asgart_b200_prepared *p, const uint64_t *family_offsets,
                                                   int64_t n_families, const asgart_b200_protosd *sds, uint32_t flags,
                                                   uint64_t min_length, int64_t max_family_members,
                                                   asgart_b200_result **out);

/* ---- the whole of asgart-slice on the SD-level result (rest of row N3; host code, no device needed) ----------------
 * RunResult as asgart writes it and asgart-slice reads it (src/structs.rs:92-97): strand name / length / fragment map,
 * settings, families of SD records (fragment names and in-fragment positions, src/bin/asgart.rs:776-821).
 * asgart_b200_run_result_slice applies asgart-slice's options in ITS order (src/bin/asgart-slice.rs:126-191):
 *   --collapse            RunResult::flatten (src/structs.rs:350-416): fragments no longer than mean + 1 sd of the fragment
 *                         lengths (f64, n-1 in the variance) whose name is longer than 2 bytes merge into ASGART_COLLAPSED;
 *                         like the reference, its map entry sits at kept_length + 1 and strand.length / global positions
 *                         are left as they were
 *   --no-direct ... --no-inter, --no-inter-relaxed (:178-187: inter-fragment duplicons survive when a leg is collapsed),
 *   --no-intra, --min-length, --max-family-members                          as asgart_b200_slice_families above
 *   --keep-fragments / --restrict-fragments / --exclude-fragments (:232-348): a duplicon stays when a leg / both legs /
 *                         no leg stands on a listed fragment; then empty families go, the map keeps (drops) the listed
 *                         fragments, positions are re-laid end to end and every duplicon's global positions recomputed
 *                         (0 for a fragment no longer in the map; --exclude unwraps instead: ASGART_B200_EPANIC).
 *                         Lists are '\n'-separated names, NULL = option absent. With ASGART_B200_SLICE_REGEXP every entry
 *                         is a pattern, applied one after the other like the reference's loop (unanchored search; the
 *                         reference uses the Rust `regex` crate, this library std::regex ECMAScript — character classes,
 *                         alternation, anchors and quantifiers agree, Rust-only syntax such as (?i) does not exist here).
 * Errors: ASGART_B200_EINVAL (bad pattern) / ASGART_B200_EPANIC with asgart_b200_run_result_error() saying why. */
typedef struct asgart_b200_run_result asgart_b200_run_result;
typedef struct asgart_b200_slice_options {
    uint32_t flags;               /* ASGART_B200_SLICE_* */
    uint32_t reserved;
    uint64_t min_length;          /* with ASGART_B200_SLICE_MIN_LENGTH */
    int64_t max_family_members;   /* < 0: not given */
    const char *keep_fragments, *restrict_fragments, *exclude_fragments;
} asgart_b200_slice_options;
ASGART_B200_API asgart_b200_run_result *asgart_b200_run_result_new(const asgart_b200_prepared *p, const asgart_b200_settings *settings,
                                                                   const uint64_t *family_offsets, int64_t n_families,
                                                                   const asgart_b200_protosd *sds);
ASGART_B200_API int32_t asgart_b200_run_result_slice(asgart_b200_run_result *rr, const asgart_b200_slice_options *options);
ASGART_B200_API char *asgart_b200_run_result_to_json(const asgart_b200_run_result *rr);   /* asgart_b200_free_string */
ASGART_B200_API const char *asgart_b200_run_result_error(const asgart_b200_run_result *rr);
ASGART_B200_API void asgart_b200_run_result_free(asgart_b200_run_result *rr);
/* asgart_b200_run_files_passes followed by asgart_b200_run_result_slice before the JSON is written */
ASGART_B200_API char *asgart_b200_run_files_sliced_ex(const char *files, const asgart_b200_settings *passes, int32_t n_passes,
                                                      int32_t device, const asgart_b200_slice_options *options, const char **err);

/* ---- GPU-side FASTA ingest (SURVEY §8f row N1) ----------------------------------------------------------------
 * read_fasta + find_chunks_to_process of prepare_data (src/bin/asgart.rs:278-366) on the device, for the raw bytes of
 * FASTA / multiFASTA files: record splitting with the semantics of the bio reader the reference calls (:282-290; id =
 * header up to the first white space, sequence lines joined after `trim_end`), per-base normalisation (:291-301),
 * fragment map (:303-308), chunks split at N-runs > 5000 per fragment (:317-366, :381-387), files concatenated with a
 * running offset (:375-395), '$' appended (:430). The strand never exists on the host: ingest_finish leaves the context
 * exactly as ctx_load_strand would (packed, ready for ctx_build_index) and returns the prepare_data result without the
 * strand bytes (asgart_b200_prepared_strand gives NULL and the length; ctx_download_strand reads it back for tests).
 *   ingest_begin -> ingest_fasta (bytes in host memory) | ingest_file (path; read through two pinned staging buffers so
 *   disk reads overlap the copies) once per file, in the order of the command line -> ingest_finish.
 * A file whose first non-empty line is not a header is refused with ASGART_B200_EINVAL ("Unable to parse", as the
 * reference's reader does); an unreadable path with ASGART_B200_EINVAL ("Unable to read FASTA file"). */
ASGART_B200_API int32_t asgart_b200_ctx_ingest_begin(asgart_b200_ctx *ctx);
ASGART_B200_API int32_t asgart_b200_ctx_ingest_fasta(asgart_b200_ctx *ctx, const uint8_t *bytes, int64_t n_bytes,
                                                     int32_t skip_masked);
ASGART_B200_API int32_t asgart_b200_ctx_ingest_file(asgart_b200_ctx *ctx, const char *path, int32_t skip_masked);
/* file_names: '\n'-separated paths as given on the command line (for strand.name of the JSON, src/bin/asgart.rs:466) */
ASGART_B200_API int32_t asgart_b200_ctx_ingest_finish(asgart_b200_ctx *ctx, const char *file_names,
                                                      asgart_b200_prepared **out);
/* the strand held by the context (n+1 bytes incl. '$') back to host memory; cap >= n+1 */
ASGART_B200_API int32_t asgart_b200_ctx_download_strand(asgart_b200_ctx *ctx, uint8_t *out, int64_t cap);

/* ---- deterministic synthetic genomes (bench/test input; DESIGN.md "Synthetic inputs") ---------------------- */
/* Fills out[0..n) (no '$') with the config's sequence (upper/lower case ACGT and N). config: 1..5 = BASELINE.json
 * configs C1..C5 (C5: part 0/1 via `part`), 0 = custom (seed, n_pairs, rc_fraction_percent, no N, no mask).
 * `scale_n` > 0 overrides the config's length (planted-pair count scales with it). Returns the length written. */
ASGART_B200_API int64_t asgart_b200_synth_length(int32_t config, int32_t part, int64_t scale_n);
ASGART_B200_API int64_t asgart_b200_synth_fill(int32_t config, int32_t part, int64_t scale_n, uint64_t seed,
                                               int64_t n_pairs, int32_t rc_percent, uint8_t *out, int64_t cap,
                                               int32_t threads);
/* fragment table of the config (names '\n'-separated into names_buf); returns the fragment count */
ASGART_B200_API int64_t asgart_b200_synth_fragments(int32_t config, int32_t part, int64_t scale_n, char *names_buf,
                                                    int64_t names_cap, uint64_t *pos, uint64_t *len, int64_t cap);

#ifdef __cplusplus
}
#endif
#endif /* ASGART_B200_H */
