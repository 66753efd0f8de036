"""asgart_b200 — B200-native duplication-search hot path of ASGART (SA build, probe search, arm automaton, post-steps)
behind a C ABI (include/asgart_b200.h). Compute runs only in libasgart_b200.so on a CUDA device."""
from .api import (AsgartB200Error, Context, build_index_group, search_group, dist_unique_id, Families, Hits, Prepared, RunSettings, device_count, families_from_lists, normalise,  # noqa: F401
                  out_filename, prepare_data, r_divsufsort, search_duplications, search_duplications_passes, synth_genome, POST_ALL, POST_COMPUTE_SCORE, POST_FILTER_NS,
                  POST_REDUCE_OVERLAP, POST_REORDER, POST_SORT)
