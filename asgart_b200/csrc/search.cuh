// search.cuh — text packing, 8-mer LUT, probe search (stage A) kernels.
//   pack_text_kernel      ASCII strand -> 4-bit packed text, or its complemented / reversed / reverse-complemented
//                         image (the needle of src/bin/asgart.rs:206-218 for every chunk at once)      HBM stream
//   lut_from_keys_kernel  SA interval of every 8-mer (Searcher::new, src/searcher.rs:99-143) and the first suffix of every ACGT
//                         15-mer ("deep table") from the initial sort's sorted keys; deep_fill_kernel closes empty buckets   HBM stream
//   lut_build_kernel      the 8-mer intervals from a finished suffix array (uploaded index, short keys)   HBM gather
//   lut_literal_kernel    the same by the reference's own bisection, for --trim (sorted only where the reference looks)
//   probe_search_kernel   one lane per probe position: LUT narrow -> literal lock-step equal range -> filtered count
//                         (Searcher::search src/searcher.rs:145-180 + src/automaton.rs:100-117)            HBM gather
//   emit (inside the scan's output pass): surviving matches in SA order + event list
#pragma once
#include "common.cuh"
#include "kmer_core.h"
#include "scan.cuh"

namespace ab200 {

enum PackMode : int { PACK_DIRECT = 0, PACK_COMPLEMENT = 1, PACK_REVERSE = 2, PACK_REVCOMP = 3 };

// One u64 word (16 symbols) per thread, 256 words per block. Direct mode packs all n1 bytes (including '$'); the needle
// modes pack the n = n1-1 bases only: needle_image[j] = f(text[j]) (complement) or f(text[n-1-j]) (reversed modes).
// The block's 4096 source bytes are one contiguous stretch of the text in every mode: it is staged in shared memory with
// 16-byte loads (the reversed modes would otherwise read byte by byte, backwards: 8 ms per 3.1 Gbp image).
// err[0] |= 1 if a byte is outside {A,C,G,N,T} or '$' is misplaced.
__global__ void __launch_bounds__(256) pack_text_kernel(const u8* __restrict__ text, u64 n1, int mode, u64* __restrict__ packed, u64 n_words,
                                                        u32* __restrict__ err) {
    __shared__ __align__(16) u8 stage[4096 + 32];
    const u64 w0 = u64(blockIdx.x) * 256;
    const u64 n = n1 - 1;
    const u64 limit = mode == PACK_DIRECT ? n1 : n;
    const u64 p0 = w0 * 16;                                  // first position of the image this block writes
    const u64 p1 = p0 + 4096 < limit ? p0 + 4096 : limit;    // (exclusive); p0 >= limit: padding words only
    u64 lo = 0, hi = 0;                                      // source bytes [lo, hi)
    if (p0 < limit) {
        if (mode & 2) { lo = n - p1; hi = n - p0; } else { lo = p0; hi = p1; }
    }
    const u64 a0 = lo & ~u64(15);                            // stage[i] = text[a0 + i]
    const bool aligned = (reinterpret_cast<uintptr_t>(text) & 15) == 0;
    for (u64 c = a0 + u64(threadIdx.x) * 16; c < hi; c += 256 * 16) {
        if (aligned && c + 16 <= n1) *reinterpret_cast<uint4*>(stage + (c - a0)) = *reinterpret_cast<const uint4*>(text + c);
        else for (u64 q = c; q < c + 16 && q < n1; ++q) stage[q - a0] = text[q];
    }
    __syncthreads();
    const u64 w = w0 + threadIdx.x;
    if (w >= n_words) return;
    const u64 pw = w * 16;
    const u32 valid = pw >= limit ? 0u : (limit - pw >= 16 ? 16u : u32(limit - pw));
    // stage offset of image position pw + j: forwards s0 + j, reversed s0 - j
    const int s0 = (mode & 2) ? int(n - 1 - pw - a0) : int(pw - a0);
    u64 word = 0;
    if (valid == 16) {   // four bytes per instruction when all 16 are bases (kmer_core.h); '$', bytes to reject, ragged ends: below
        const int low = (mode & 2) ? s0 - 15 : s0;
        const u32* sw = reinterpret_cast<const u32*>(stage) + (low >> 2);
        const u32 W[5] = {sw[0], sw[1], sw[2], sw[3], sw[4]};
        if (pack16_fast(W, u32(low) & 3u, (mode & 2) != 0, (mode & 1) != 0, word)) {
            packed[w] = word;
            return;
        }
        word = 0;
    }
    u32 bad = 0;
    const u64 tab = (mode & 1) ? kCodeTabComp : kCodeTab;
    const int step = (mode & 2) ? -1 : 1;
    const i64 s_end = i64(n) - i64(a0);                      // stage offset of the '$' (only the direct mode reaches it)
#pragma unroll 1
    for (u32 j = 0; j < valid; ++j) {
        const int so = s0 + step * int(j);
        const u32 byte = stage[so];
        const u32 c = code_of_byte_tab(byte, tab);
        bad |= u32(c == CODE_BAD) | u32((byte == u32('$')) != (i64(so) == s_end));
        word |= u64(c) << (60 - 4 * int(j));
    }
    packed[w] = word;
    if (bad) atomicOr(err, 1u);
}

// lo/hi of every 8-mer bucket from the suffix array: boundaries where the first 8 symbols change.
template <typename IdxT>
__global__ void lut_build_kernel(const u64* __restrict__ PT, const IdxT* __restrict__ SA, u64 n1, IdxT* __restrict__ lut_lo,
                                 IdxT* __restrict__ lut_hi) {
    const u64 i = u64(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n1) return;
    u32 cur_slot, prev_slot = 0;
    const bool cur_ok = lut_slot(load_window(PT, u64(SA[i])).hi, cur_slot);
    bool prev_ok = false;
    if (i > 0) prev_ok = lut_slot(load_window(PT, u64(SA[i - 1])).hi, prev_slot);
    if (cur_ok && (!prev_ok || prev_slot != cur_slot)) lut_lo[cur_slot] = IdxT(i);
    if (prev_ok && (!cur_ok || prev_slot != cur_slot)) lut_hi[prev_slot] = IdxT(i);
    if (i + 1 == n1 && cur_ok) lut_hi[cur_slot] = IdxT(n1);
}

// Searcher::new with --trim (src/searcher.rs:99-143 over the array of src/bin/asgart.rs:142-147): SA holds the suffixes of
// strand[a..b]+'$' (shifted by a) but sa_searchb64 compares them inside the WHOLE strand, so near b the array is not sorted
// for what it is compared with and the bucket borders are whatever the reference's bisection lands on. One thread per
// 8-mer replays that probe sequence (literal_bucket, kmer_core.h). Slot = 8-mer as base-5 number with digits A,C,G,N,T;
// empty buckets get lo = hi = the reference's insertion point.
template <typename IdxT>
__global__ void lut_literal_kernel(const u8* __restrict__ T, u64 Tsize, const IdxT* __restrict__ SA, u64 SAsize,
                                   IdxT* __restrict__ lut_lo, IdxT* __restrict__ lut_hi) {
    const u32 slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= 390625u) return;
    u8 P[8];
    u32 v = slot;
#pragma unroll
    for (int j = 7; j >= 0; --j) { P[j] = u8("ACGNT"[v % 5u]); v /= 5u; }
    int64_t first = 0, count = 0;
    literal_bucket<IdxT>(T, int64_t(Tsize), P, SA, int64_t(SAsize), first, count);
    lut_lo[slot] = IdxT(first);
    lut_hi[slot] = IdxT(first + count);
}

template <typename IdxT>
__global__ void add_offset_kernel(IdxT* __restrict__ v, u64 n, IdxT off) {
    const u64 stride = u64(gridDim.x) * blockDim.x;
    for (u64 i = u64(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) v[i] += off;
}

struct ChunkDev {
    u64 c0, len;        // global start, length (src/bin/asgart.rs:115)
    u64 n_probes;       // loop iterations (src/automaton.rs:96-98)
    u64 probe_base;     // global index of its first probe
    u64 needle_start;   // position of needle[0] in the packed needle image
};

// chunk of global probe g: last c with probe_base[c] <= g  (n_chunks >= 1, chunks with 0 probes are skipped naturally)
__device__ __forceinline__ u32 chunk_of_probe(const ChunkDev* __restrict__ ch, u32 n_chunks, u64 g) {
    u32 lo = 0, hi = n_chunks;
    while (hi - lo > 1) {
        const u32 mid = (lo + hi) >> 1;
        if (ch[mid].probe_base <= g) lo = mid; else hi = mid;
    }
    return lo;
}

// ---------------------------------------------------------------------------------------------------------------
// Lookup tables as by-products of the suffix-array build's initial sort (sa_build.cuh, SaKeyHook): the sorted keys hold
// the first p0 symbols of every suffix in suffix order, so bucket boundaries need no gather through SA and text.
struct LutCodeMap {
    u8 d5[16];  // dense symbol code -> base-5 digit A,C,G,N,T = 0..4 (255: '$' or padding)
    u8 d4[16];  // dense symbol code -> base-4 digit A,C,G,T = 0..3 (255 otherwise)
    u64 nibbles(const u8* d) const { u64 m = 0; for (int c = 0; c < 16; ++c) m |= u64(d[c] == 255 ? 15u : d[c]) << (4 * c); return m; }
};

// the code maps as 16 nibbles each (0xF = no digit): register-resident, so decoding a key is pure ALU work
__device__ __forceinline__ bool key_slot5(u64 key, int b, int p0, u64 m5, u32& slot) {
    u32 s = 0, bad = 0;
    const u32 mask = (1u << b) - 1u;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const u32 d = u32(m5 >> (4u * (u32(key >> (b * (p0 - 1 - j))) & mask))) & 15u;
        bad |= d;
        s = s * 5u + d;
    }
    slot = s;
    return (bad & 8u) == 0;   // digits are 0..4, 15 = invalid symbol
}
__device__ __forceinline__ bool key_slot4(u64 key, int b, int p0, int depth, u64 m4, u32& slot) {
    u32 s = 0, bad = 0;
    const u32 mask = (1u << b) - 1u;
    int sh = b * (p0 - 1);
    for (int j = 0; j < depth; ++j, sh -= b) {
        const u32 d = u32(m4 >> (4u * (u32(key >> sh) & mask))) & 15u;
        bad |= d;
        s = s * 4u + (d & 3u);
    }
    slot = s;
    return (bad & 12u) == 0;   // digits are 0..3
}

// Base-4 slot of the first `depth` symbols of a key made of 3-bit symbol codes, four symbols per table lookup:
// tab4[12 bits] = the four 2-bit digits (first symbol in the top pair) | 0x8000 when one of the four codes is not A/C/G/T.
// `pad` = 9 bits of a valid code repeated: fills a last group of fewer than four symbols (its digits are dropped again).
// The digit-by-digit decode (key_slot4) made the table kernel ALU-bound: ~90 instructions per bucket border, a third of
// all keys at 3.1 Gbp with 15-symbol buckets.
__device__ __forceinline__ bool key_slot4_tab(u64 key, int p0, int depth, const uint16_t* __restrict__ tab4, u32 pad, u32& slot) {
    u32 s = 0, bad = 0;
    int sh = 3 * p0, rem = depth;
    while (rem >= 4) {
        sh -= 12;
        const u32 e = __ldg(&tab4[u32(key >> sh) & 4095u]);
        s = (s << 8) | (e & 255u);
        bad |= e;
        rem -= 4;
    }
    if (rem) {
        sh -= 3 * rem;
        const int fill = 3 * (4 - rem);
        const u32 grp = ((u32(key >> sh) & ((1u << (3 * rem)) - 1u)) << fill) | (pad & ((1u << fill) - 1u));
        const u32 e = __ldg(&tab4[grp]);
        s = (s << (2 * rem)) | ((e & 255u) >> (2 * (4 - rem)));
        bad |= e;
    }
    slot = s;
    return (bad & 0x8000u) == 0;
}

// 8-mer LUT (Searcher::new, src/searcher.rs:99-143) and, when depth > 0, the first suffix of every ACGT-only
// `depth`-mer (0 = not seen; position 0 is always the '$' suffix) from the sorted initial keys. Needs p0 >= 8, depth.
// Four keys per thread (two 16-byte loads + the predecessor); keys must be 16-byte aligned.
template <typename IdxT>
__global__ void __launch_bounds__(256) lut_from_keys_kernel(const u64* __restrict__ keys, u64 n_local, u64 base, int b, int p0,
                                                            u64 m5, u64 m4, int depth, const uint16_t* __restrict__ tab4, u32 pad4,
                                                            IdxT* __restrict__ lut_lo, IdxT* __restrict__ lut_hi, IdxT* __restrict__ deep) {
    // keys[0 .. n_local) are positions [base, base + n_local) of the sorted keys (sharded build: one member's key range,
    // cut where the first four symbols change, so the first and the last key of the piece are bucket boundaries)
    const u64 i0 = (u64(blockIdx.x) * blockDim.x + threadIdx.x) * 4;
    if (i0 >= n_local) return;
    u64 kk[5];
    kk[0] = i0 > 0 ? keys[i0 - 1] : 0;
    if (i0 + 4 <= n_local) {
        const ulonglong2 v0 = *reinterpret_cast<const ulonglong2*>(keys + i0), v1 = *reinterpret_cast<const ulonglong2*>(keys + i0 + 2);
        kk[1] = v0.x; kk[2] = v0.y; kk[3] = v1.x; kk[4] = v1.y;
    } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) kk[j + 1] = i0 + j < n_local ? keys[i0 + j] : 0;
    }
    if (i0 == 0) kk[0] = ~kk[1];
    const int s8 = b * (p0 - 8);
    const int sd = b * (p0 - depth);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const u64 i = i0 + j;
        if (i >= n_local) break;
        const u64 cur = kk[j + 1], prev = kk[j];
        // slots only change where the leading symbols do: decode the boundaries only
        if ((cur >> s8) != (prev >> s8) || i + 1 == n_local) {
            u32 cs = 0, ps = 0;
            const bool cur_ok = key_slot5(cur, b, p0, m5, cs);
            const bool prev_ok = i > 0 && key_slot5(prev, b, p0, m5, ps);
            if (cur_ok && (!prev_ok || ps != cs)) lut_lo[cs] = IdxT(base + i);
            if (prev_ok && (!cur_ok || ps != cs)) lut_hi[ps] = IdxT(base + i);
            if (i + 1 == n_local && cur_ok) lut_hi[cs] = IdxT(base + n_local);
        }
        if (depth > 0 && (cur >> sd) != (prev >> sd)) {
            u32 cs = 0;
            const bool ok4 = tab4 ? key_slot4_tab(cur, p0, depth, tab4, pad4, cs) : key_slot4(cur, b, p0, depth, m4, cs);
            if (ok4) deep[cs] = IdxT(base + i);
        }
    }
}

// Deep table, empty buckets: a slot no key hit (0) takes the start of the next slot that was hit; deep[M - 1] = n1 closes the
// table. In a genome-sized table few slots are empty and the runs are short (3.1 Gbp in 4^15 slots: 5 %, mostly single), so
// one pass does it: four slots per thread, a thread whose group ends on an empty slot looks ahead, at most kDeepLook slots.
// It may read a slot its owner is filling at that moment — either 0 or the final value, and a filled value is exactly what
// the look-ahead is after. A longer empty run sets *overflow and the caller runs the general scan over what is left (filled
// slots then count as hit ones: same answer). deep must be 16-byte aligned.
constexpr u32 kDeepLook = 256;
template <typename IdxT>
__global__ void __launch_bounds__(256) deep_fill_kernel(IdxT* __restrict__ deep_, u64 M, u32* __restrict__ overflow) {
    volatile IdxT* deep = deep_;                    // the look-ahead reads slots other threads write
    const u64 groups = (M + 3) / 4;
    const u64 stride = u64(gridDim.x) * blockDim.x;
    for (u64 g = u64(blockIdx.x) * blockDim.x + threadIdx.x; g < groups; g += stride) {
        const u64 s0 = g * 4;
        IdxT v[4];
        if (s0 + 4 <= M) {                          // its own four slots (nobody else writes them): vector loads
            if constexpr (sizeof(IdxT) == 4) {
                const uint4 x = *reinterpret_cast<const uint4*>(deep_ + s0);
                v[0] = IdxT(x.x); v[1] = IdxT(x.y); v[2] = IdxT(x.z); v[3] = IdxT(x.w);
            } else {
                const ulonglong2 x = *reinterpret_cast<const ulonglong2*>(deep_ + s0), y = *reinterpret_cast<const ulonglong2*>(deep_ + s0 + 2);
                v[0] = IdxT(x.x); v[1] = IdxT(x.y); v[2] = IdxT(y.x); v[3] = IdxT(y.y);
            }
        } else {
#pragma unroll
            for (int q = 0; q < 4; ++q) v[q] = s0 + q < M ? deep[s0 + q] : IdxT(1);
        }
        if (v[0] != 0 && v[1] != 0 && v[2] != 0 && v[3] != 0) continue;
        IdxT nxt = v[3];
        if (nxt == 0) {
            u64 t = s0 + 4;
            for (u32 look = 0; look < kDeepLook && t < M; ++look, ++t) {
                nxt = deep[t];
                if (nxt != 0) break;
            }
            if (nxt == 0) { atomicOr(overflow, 1u); continue; }
        }
#pragma unroll
        for (int q = 3; q >= 0; --q) {
            if (v[q] == 0) { if (s0 + q < M) deep[s0 + q] = nxt; }
            else nxt = v[q];
        }
    }
}

// slots of the 8-mer LUT whose bucket holds one of the last k-1 suffixes: there the reference's comparator is forced
// to Less (src/searcher.rs:165-166, quirk Q6) and only its literal bisection reproduces its answer
__global__ void q6_mark_kernel(const u64* __restrict__ PT, u64 n1, u32 k, u32* __restrict__ q6_bits) {
    const u64 t = u64(blockIdx.x) * blockDim.x + threadIdx.x;
    const u64 first = n1 >= k ? n1 - k + 1 : 0;
    const u64 x = first + t;
    if (x >= n1) return;
    u32 slot;
    if (lut_slot(load_window(PT, x).hi, slot)) atomicOr(&q6_bits[slot >> 5], 1u << (slot & 31u));
}

template <typename IdxT>
struct ProbeParams {
    const u64* PT;  // packed strand
    const u64* PN;  // packed needle image (== PT when no flag is set)
    const IdxT* SA;
    const IdxT* lut_lo;
    const IdxT* lut_hi;
    const IdxT* deep;     // deep table: 4^deep_depth + 1 non-decreasing bucket starts, or null
    int deep_depth;
    // the build's sorted initial keys (keys[i] = first key_p0 symbols of suffix SA[i], key_b bits each, first symbol on
    // top) and the map strand code -> key code (one nibble per CODE_*); null: deep buckets are compared on the text
    const u64* keys;
    int key_b, key_p0;
    u64 key_map;
    const u32* q6_bits;   // 5^8 bits
    const ChunkDev* chunks;
    u32 n_chunks;
    u64 n1;
    u32 k, s;
    u32 reverse;
    u64 max_card;
    u64 p_begin, p_end;  // probe shard [p_begin, p_end), p_begin % 32 == 0
    // per-probe outputs, indexed g - p_begin
    IdxT* out_lo;
    IdxT* out_raw;
    u32* out_surv;
    u32* proc_bits;   // bit (g - p_begin): iteration processed (neither N-skipped nor over the cardinality cap)
    unsigned long long* counters;  // [0] searched [1] skipped_n [2] skipped_card [3] matches [4] algorithmic bytes [5] deferred
    u64* deferred;    // probes left to the literal kernel (capacity p_end - p_begin)
    // test hook (asgart_b200_ctx_probe_ranges): equal ranges only, no N test, no filters
    i64* rng_lo;
    i64* rng_hi;
};

enum { CTR_SEARCHED = 0, CTR_SKIP_N = 1, CTR_SKIP_CARD = 2, CTR_MATCHES = 3, CTR_ALG_BYTES = 4, CTR_DEFERRED = 5, CTR_COUNT = 8 };

__device__ __forceinline__ u64 warp_sum_u64(u64 v) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    return v;
}

struct ProbeState {
    bool processed = false, searched = false, skip_n = false, skip_card = false;
    u64 lo = 0, hi = 0, surv = 0, alg = 0;
};

constexpr u64 kDeferRange = u64(1) << 63;  // deferred entry: the equal range is known (out_lo / out_raw), only the filters are left
constexpr u64 kInlineMatches = 32;         // longer match intervals are filtered by a whole warp (probe_deferred_kernel)

// per-probe outputs once the equal range [S.lo, S.hi) is known; returns false when the filters are left to a warp
// filters + cardinality: src/automaton.rs:105-117
template <typename IdxT>
__device__ __forceinline__ bool probe_finish(const ProbeParams<IdxT>& P, const ChunkDev& ch, u64 g, u64 i, u64 bucket8, bool may_defer,
                                             ProbeState& S) {
    S.searched = true;
    S.alg = 24ull * (ceil_log2_u64(bucket8 + 1) + 1) + 8ull * (S.hi - S.lo);  // SURVEY §8d
    const u64 o = g - P.p_begin;
    if (P.rng_lo) { P.rng_lo[o] = i64(S.lo); P.rng_hi[o] = i64(S.hi); return true; }
    P.out_lo[o] = IdxT(S.lo);
    P.out_raw[o] = IdxT(S.hi - S.lo);
    if (may_defer && S.hi - S.lo > kInlineMatches) return false;
    const bool rev = P.reverse != 0;
    for (u64 j = S.lo; j < S.hi; ++j) {
        if (match_survives(u64(P.SA[j]), i, ch.c0, ch.len, rev)) {
            if (++S.surv > P.max_card) break;
        }
    }
    if (S.surv > P.max_card) { S.skip_card = true; S.surv = 0; } else S.processed = true;
    P.out_surv[o] = u32(S.surv);
    return true;
}

// the reference's own search: 8-mer bucket, then the literal lock-step bisection with the forced-Less comparator
template <typename IdxT>
__device__ __forceinline__ u64 probe_literal(const ProbeParams<IdxT>& P, u64 q, const Win& pw_raw, ProbeState& S) {
    const int k = int(P.k);
    const Win pw0 = mask_window(pw_raw, k < 32 ? k : 32);
    u32 slot = 0;
    u64 lstart = 0, rstart = 0;
    if (lut_slot(pw_raw.hi, slot)) { lstart = u64(P.lut_lo[slot]); rstart = u64(P.lut_hi[slot]); }
    const IdxT* __restrict__ sub = P.SA + lstart;
    const u64 n1 = P.n1;
    const u64* __restrict__ PT = P.PT;
    const u64* __restrict__ PN = P.PN;
    u64 r0, r1;
    equal_range_lockstep(rstart - lstart, [&](u64 ix) -> int {
        const u64 x = u64(sub[ix]);
        if (x + u64(k) > n1) return -1;  // src/searcher.rs:165-166 (Q6)
        return cmp_kmer(PT, x, PN, q, k, pw0);
    }, r0, r1);
    if (r1 < r0) r1 = r0;  // only reachable through Q6; the reference would panic on the slice
    S.lo = lstart + r0;
    S.hi = lstart + r1;
    return rstart - lstart;
}

// The block's counts go to the counters with one atomic per counter: same-address atomics serialise in one L2 slice, and
// with one per warp and counter they bounded this kernel once the keys had shortened the search (on B200 at C4 size, one
// more per-warp counter took the keys comparison from 44 to 59 ms). Every thread of the block calls this (it synchronises
// the block); blockDim.x == 256.
template <typename IdxT>
__device__ __forceinline__ void probe_account(const ProbeParams<IdxT>& P, const ProbeState& S) {
    __shared__ u64 part[8][5];
    const u64 v[5] = {__popc(__ballot_sync(0xffffffffu, S.searched)), __popc(__ballot_sync(0xffffffffu, S.skip_n)),
                      __popc(__ballot_sync(0xffffffffu, S.skip_card)), warp_sum_u64(S.surv), warp_sum_u64(S.alg)};
    if (lane_id() == 0) {
#pragma unroll
        for (int c = 0; c < 5; ++c) part[threadIdx.x >> 5][c] = v[c];
    }
    __syncthreads();
    if (threadIdx.x < 5) {
        u64 sum = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) sum += part[w][threadIdx.x];
        const int ctr[5] = {CTR_SEARCHED, CTR_SKIP_N, CTR_SKIP_CARD, CTR_MATCHES, CTR_ALG_BYTES};
        if (sum) atomicAdd(&P.counters[ctr[threadIdx.x]], (unsigned long long)sum);
    }
}

// equal range of a deep bucket [lo0, lo0 + B) from the sorted keys: keys[lo0 ..] are compared with the probe's first
// m = min(k, p0) symbols, and only suffixes whose key equals them, when k > p0, are compared on the text (cmp_kmer).
// The bucket holds none of the last k-1 suffixes, so the m compared symbols of every key are text symbols (a '$' among
// them already differs from the probe, which has none): the key comparison is the text comparison of those m symbols.
template <typename IdxT, int kProbeLinear>
__device__ __forceinline__ void probe_keys(const ProbeParams<IdxT>& P, u64 lo0, u64 B, u64 q, const Win& pw_raw, const Win& pw0,
                                           ProbeState& S) {
    const int k = int(P.k), b = P.key_b, p0 = P.key_p0;
    const int m = k < p0 ? k : p0;
    u64 pk = 0;   // the probe's first m symbols as a key (every needle symbol has a key code: run_probe_kernels)
    for (int j = 0; j < m; ++j) {
        const u32 sym = u32((j < 16 ? pw_raw.hi : pw_raw.lo) >> (60 - 4 * (j & 15))) & 15u;
        pk = (pk << b) | ((P.key_map >> (4 * sym)) & 15u);
    }
    const int sh = b * (p0 - m);
    const u64* __restrict__ K = P.keys + lo0;
    u64 r0, r1;
    if (B <= kProbeLinear) {
        u64 kv[kProbeLinear];
#pragma unroll
        for (int j = 0; j < kProbeLinear; ++j) kv[j] = u64(j) < B ? K[j] : 0;
        u32 lt = 0, le = 0;
#pragma unroll
        for (int j = 0; j < kProbeLinear; ++j) {
            const u64 v = kv[j] >> sh;
            if (u64(j) < B) { lt += v < pk; le += v <= pk; }
        }
        r0 = lt; r1 = le;
        if (k > p0 && r1 > r0) {   // keys equal to the probe's on [r0, r1): the k-mers there run smaller, equal, greater
            u64 lo = r0, hi = r1;
#pragma unroll 1
            for (u64 j = r0; j < r1; ++j) {
                const int c = cmp_kmer(P.PT, u64(P.SA[lo0 + j]), P.PN, q, k, pw0);
                if (c > 0) { hi = j; break; }
                lo += c < 0;
            }
            r0 = lo; r1 = hi;
        }
    } else {
        equal_range_lockstep(B, [&](u64 ix) -> int {
            const u64 v = K[ix] >> sh;
            if (v != pk) return v < pk ? -1 : 1;
            return k > p0 ? cmp_kmer(P.PT, u64(P.SA[lo0 + ix]), P.PN, q, k, pw0) : 0;
        }, r0, r1);
    }
    S.lo = lo0 + r0; S.hi = lo0 + r1;
}

// deep buckets up to LINEAR suffixes are compared in one go instead of bisected (template parameter of the kernel)

// One lane per probe position. Probes whose first deep_depth bases are all ACGT start from the deep table's bucket
// (a few suffixes) and compare them all at once; the equal range of a monotone comparator does not depend on how it is
// searched, so this is the reference's answer whenever its own 8-mer bucket holds none of the last k-1 suffixes. KEYS:
// the bucket is compared in the sorted initial keys (probe_keys), else on the text through SA. Every other probe (N among
// the first bases, flagged bucket, no deep table) takes probe_literal, in this kernel when P.deferred is null and in
// probe_deferred_kernel otherwise (keeps the long bisections out of the short warps); probes with long match intervals
// leave the filter pass to that kernel as well. The keys only come with a deep table, so KEYS always defers.
template <typename IdxT, int kProbeLinear, int MINB, bool KEYS>
__global__ void __launch_bounds__(256, MINB) probe_search_kernel(const ProbeParams<IdxT> P) {
    const u64 g = P.p_begin + u64(blockIdx.x) * blockDim.x + threadIdx.x;
    const bool in_range = g < P.p_end;
    ProbeState S;
    u64 defer = 0;
    if (in_range) {
        const ChunkDev ch = P.chunks[chunk_of_probe(P.chunks, P.n_chunks, g)];
        const u64 i = (g - ch.probe_base + 1) * P.s;
        const u64 q = ch.needle_start + i;
        const int k = int(P.k);
        const Win pw_raw = load_window(P.PN, q);
        u32 slot4 = 0, slot8 = 0;
        if (!P.rng_lo && (pw_raw.hi >> 60) == CODE_N) {
            S.skip_n = true;  // src/automaton.rs:100-102
            const u64 o = g - P.p_begin;
            P.out_lo[o] = 0; P.out_raw[o] = 0; P.out_surv[o] = 0;
        } else if (P.deep && deep_slot(pw_raw.hi, P.deep_depth, slot4) && lut_slot(pw_raw.hi, slot8) &&
                   !((P.q6_bits[slot8 >> 5] >> (slot8 & 31u)) & 1u)) {
            const u64 lo0 = u64(P.deep[slot4]), hi0 = u64(P.deep[slot4 + 1]);
            const u64 bucket8 = u64(P.lut_hi[slot8]) - u64(P.lut_lo[slot8]);
            const Win pw0 = mask_window(pw_raw, k < 32 ? k : 32);
            const IdxT* __restrict__ sub = P.SA + lo0;
            const u64* __restrict__ PT = P.PT;
            const u64* __restrict__ PN = P.PN;
            const u64 B = hi0 - lo0;
            if constexpr (KEYS) {
                probe_keys<IdxT, kProbeLinear>(P, lo0, B, q, pw_raw, pw0, S);
            } else if (B <= kProbeLinear) {
                u64 xs[kProbeLinear];
#pragma unroll
                for (int j = 0; j < kProbeLinear; ++j) xs[j] = u64(j) < B ? u64(sub[j]) : 0;
                Win ws[kProbeLinear];
#pragma unroll
                for (int j = 0; j < kProbeLinear; ++j) ws[j] = load_window(PT, xs[j]);
                u32 lt = 0, le = 0;
#pragma unroll
                for (int j = 0; j < kProbeLinear; ++j) {
                    if (u64(j) < B) {
                        int c = cmp_window(mask_window(ws[j], k < 32 ? k : 32), pw0);
                        if (c == 0 && k > 32) c = cmp_kmer(PT, xs[j], PN, q, k, pw0);
                        lt += c < 0; le += c <= 0;
                    }
                }
                S.lo = lo0 + lt; S.hi = lo0 + le;
            } else {
                u64 r0, r1;
                equal_range_lockstep(B, [&](u64 ix) -> int { return cmp_kmer(PT, u64(sub[ix]), PN, q, k, pw0); }, r0, r1);
                S.lo = lo0 + r0; S.hi = lo0 + r1;
            }
            if (!probe_finish(P, ch, g, i, bucket8, P.deferred != nullptr, S)) defer = g | kDeferRange;
        } else if (KEYS || P.deferred) {
            defer = g | (u64(1) << 62);  // bit 62 only marks the entry as present (g may be 0)
        } else {
            const u64 bucket8 = probe_literal(P, q, pw_raw, S);
            probe_finish(P, ch, g, i, bucket8, false, S);
        }
    }
    const unsigned dm = __ballot_sync(0xffffffffu, defer != 0);
    if (dm) {
        unsigned long long base = 0;
        if (lane_id() == 0) base = atomicAdd(&P.counters[CTR_DEFERRED], (unsigned long long)__popc(dm));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (defer) P.deferred[base + __popc(dm & lanemask_lt())] = defer;
    }
    const unsigned bits = __ballot_sync(0xffffffffu, S.processed);
    if (lane_id() == 0 && !P.rng_lo) {
        const u64 word = (u64(blockIdx.x) * blockDim.x + (threadIdx.x & ~31u)) >> 5;
        if (P.p_begin + word * 32 < P.p_end) P.proc_bits[word] = bits;
    }
    probe_account(P, S);
}

// The probes probe_search_kernel left over, one warp each: the lanes run the literal search in lock step (same
// addresses: one transaction per load) and share the filter pass over the match interval.
template <typename IdxT>
__global__ void __launch_bounds__(256) probe_deferred_kernel(const ProbeParams<IdxT> P, u64 n_deferred) {
    const u64 j = (u64(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    if (j >= n_deferred) return;
    const u64 e = P.deferred[j];
    const u64 g = e & ~(kDeferRange | (u64(1) << 62));
    const u64 o = g - P.p_begin;
    const ChunkDev ch = P.chunks[chunk_of_probe(P.chunks, P.n_chunks, g)];
    const u64 i = (g - ch.probe_base + 1) * P.s;
    const u64 q = ch.needle_start + i;
    ProbeState S;
    u64 alg = 0;
    if (e & kDeferRange) {
        S.lo = u64(P.out_lo[o]); S.hi = S.lo + u64(P.out_raw[o]);   // searched and accounted by probe_search_kernel
    } else {
        const u64 bucket8 = probe_literal(P, q, load_window(P.PN, q), S);
        alg = 24ull * (ceil_log2_u64(bucket8 + 1) + 1) + 8ull * (S.hi - S.lo);
        if (P.rng_lo) {
            if (lane_id() == 0) { P.rng_lo[o] = i64(S.lo); P.rng_hi[o] = i64(S.hi); }
            return;
        }
    }
    const bool rev = P.reverse != 0;
    u64 surv = 0;
    for (u64 j0 = S.lo; j0 < S.hi && surv <= P.max_card; j0 += 32) {
        const u64 jj = j0 + lane_id();
        const bool keep = jj < S.hi && match_survives(u64(P.SA[jj]), i, ch.c0, ch.len, rev);
        surv += __popc(__ballot_sync(0xffffffffu, keep));
    }
    if (lane_id() == 0) {
        const bool skip_card = surv > P.max_card;
        if (skip_card) surv = 0;
        P.out_lo[o] = IdxT(S.lo); P.out_raw[o] = IdxT(S.hi - S.lo); P.out_surv[o] = u32(surv);
        if (!skip_card) atomicOr(&P.proc_bits[o >> 5], 1u << (o & 31u));
        if (!(e & kDeferRange)) atomicAdd(&P.counters[CTR_SEARCHED], 1ull);
        if (skip_card) atomicAdd(&P.counters[CTR_SKIP_CARD], 1ull);
        if (surv) atomicAdd(&P.counters[CTR_MATCHES], (unsigned long long)surv);
        if (alg) atomicAdd(&P.counters[CTR_ALG_BYTES], (unsigned long long)alg);
    }
}

// pair of running sums: match offset and event index
struct Sum2 {
    u64 a, b;
    Sum2() = default;
    __host__ __device__ explicit Sum2(int) : a(0), b(0) {}
    __host__ __device__ Sum2(u64 x, u64 y) : a(x), b(y) {}
};
struct Sum2Op {
    __device__ __forceinline__ Sum2 operator()(const Sum2& x, const Sum2& y) const { return Sum2(x.a + y.a, x.b + y.b); }
};

// one warp per event: stream SA[lo, lo+raw), keep the survivors of the two filters in SA order
template <typename IdxT>
__global__ void __launch_bounds__(256) emit_matches_kernel(const IdxT* __restrict__ SA, const u64* __restrict__ ev_probe,
                                                           const u64* __restrict__ ev_moff, const IdxT* __restrict__ ev_lo,
                                                           const IdxT* __restrict__ ev_raw, u64 n_events,
                                                           const ChunkDev* __restrict__ chunks, u32 n_chunks, u32 s, u32 reverse,
                                                           u64* __restrict__ matches) {
    const u64 e = (u64(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    if (e >= n_events) return;
    const unsigned lane = lane_id(), lt = lanemask_lt();
    const u64 g = ev_probe[e];
    const ChunkDev ch = chunks[chunk_of_probe(chunks, n_chunks, g)];
    const u64 i = (g - ch.probe_base + 1) * s;
    const u64 b = u64(ev_lo[e]), end = b + u64(ev_raw[e]);
    u64 w = ev_moff[e];
    for (u64 j0 = b; j0 < end; j0 += 32) {
        const u64 j = j0 + lane;
        u64 x = 0;
        bool keep = false;
        if (j < end) { x = u64(SA[j]); keep = match_survives(x, i, ch.c0, ch.len, reverse != 0); }
        const unsigned m = __ballot_sync(0xffffffffu, keep);
        if (keep) matches[w + __popc(m & lt)] = x;
        w += __popc(m);
    }
}

}  // namespace ab200
