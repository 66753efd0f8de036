// locate.cuh — batched exact-match queries against the resident index: sa_search64 (libdivsufsort/lib/utils.c:244-255
// _compare, :282-349 sa_search; bound by the reference at src/divsufsort.rs) for many patterns at once, and the positions
// of their matches.
//   locate_pack_kernel      pattern bytes -> 4-bit codes (kCodeTab order) + per pattern the "cut": the first byte
//                           that has no code                                                          HBM stream
//   locate_short_kernel     full index, patterns of <= 32 symbols: one lane per pattern, deep table / 8-mer LUT narrow,
//                           then lower and upper bound, one 128-bit window per step                    HBM gather
//   locate_long_kernel      full index, longer patterns: one warp per pattern, the lanes compare 16-symbol words from
//                           the prefix already known to match (min(lmatch, rmatch), as sa_search does)  HBM gather
//   locate_literal_kernel   index built with --trim: sa_search step for step, one thread per pattern   latency
//   locate_copy_kernel      one warp per pattern: SA[first .. first + min(count, max_hits)) -> int64     HBM stream
//
// Comparison (what _compare does): bytes compared as bytes, a suffix that ends inside P is smaller. Up to the cut both
// sides are packed codes, whose order is the byte order of {$,A,C,G,N,T}; the strand holds nothing else, so at the cut
// the text byte always differs from the pattern byte (or the text has ended: smaller).
#pragma once
#include "common.cuh"
#include "kmer_core.h"
#include "scan.cuh"
#include "search.cuh"

namespace ab200 {

template <typename IdxT>
struct LocateParams {
    const u64* PT;        // packed strand
    u64 n1;               // strand length including '$'
    const IdxT* SA;
    u64 sa_len;
    const IdxT* lut_lo;   // 8-mer LUT (full index only)
    const IdxT* lut_hi;
    const IdxT* deep;     // deep table or null
    int deep_depth;
    const u8* pat;        // pattern bytes of the slice
    const u64* PP;        // packed pattern bytes (same positions)
    const u64* off;       // slice-local offsets, n_patterns + 1
    const u64* cut;       // first byte without a code, relative to the pattern (>= its length: none)
    const u32* list;      // patterns this launch takes (null: all)
    u64 n_list;
    i64* first;
    i64* count;
    unsigned long long* alg_bytes;
};

// symbol -> byte of the strand alphabet (codes 1..6)
__device__ __forceinline__ u32 byte_of_code(u32 c) { return u32(u64(0x54'4E'47'43'41'24'00ull) >> (8 * c)) & 0xFFu; }

// 16 symbols of a packed array from symbol `pos` on
__device__ __forceinline__ u64 load16(const u64* __restrict__ P, u64 pos) {
    const u64 w = pos >> 4;
    const unsigned o = unsigned(pos & 15u) * 4u;
    const u64 a = P[w];
    return o == 0 ? a : (a << o) | (P[w + 1] >> (64u - o));
}
__device__ __forceinline__ u64 mask16(u64 v, u64 k) { return k >= 16 ? v : (k == 0 ? 0 : v & ~(~u64(0) >> (4 * k))); }

// what _compare decides once `m` (== eff) symbols are known equal
__device__ __forceinline__ int cmp_at_cut(const u64* __restrict__ PT, u64 n1, u64 x, const u8* __restrict__ pb, u64 len, u64 m) {
    if (m >= len) return 0;
    if (x + m >= n1) return -1;                                   // the suffix ends inside P
    const u32 tc = u32(PT[(x + m) >> 4] >> (60 - 4 * ((x + m) & 15u))) & 15u;
    return int(byte_of_code(tc)) - int(pb[m]);
}

// algorithmic bytes of one bisection step that compared `symbols` symbols (SURVEY §8d, extended): 24 B for the SA entry
// and the first 32-symbol window, 16 B per further 32 symbols
__device__ __forceinline__ u64 alg_of_compare(u64 symbols) { return 24 + (symbols > 32 ? 16 * ((symbols - 1) / 32) : 0); }

// sign of (suffix x) - P over P's len bytes, one thread, from symbol m on (m symbols already known equal); m becomes the
// number of leading symbols found equal (compare_skip of the oracle, one 32-symbol window per step)
__device__ __forceinline__ int cmp_pattern(const u64* __restrict__ PT, u64 n1, u64 x, const u64* __restrict__ PP, u64 po,
                                           const u8* __restrict__ pb, u64 len, u64 eff, u64& m, u64& alg) {
    const u64 m0 = m;
    u64 k = m;
    while (k < eff && x + k < n1) {   // a suffix shorter than the known prefix (trimmed index only) has ended: smaller
        const int w = eff - k < 32 ? int(eff - k) : 32;
        const Win t = mask_window(load_window(PT, x + k), w), p = mask_window(load_window(PP, po + k), w);
        if (t.hi != p.hi || t.lo != p.lo) {
            k += t.hi != p.hi ? u64(__clzll(t.hi ^ p.hi) >> 2) : 16 + u64(__clzll(t.lo ^ p.lo) >> 2);
            m = k;
            alg += alg_of_compare(k + 1 - m0);
            return cmp_window(t, p);
        }
        k += u64(w);
    }
    m = k;
    alg += alg_of_compare(k + 1 - m0);
    return cmp_at_cut(PT, n1, x, pb, len, k);
}

// The same with a whole warp (every lane passes the same arguments and gets the same answer): lane l compares the 16
// symbols at m + 16 l, 512 symbols per round
__device__ __forceinline__ int cmp_pattern_warp(const u64* __restrict__ PT, u64 n1, u64 x, const u64* __restrict__ PP, u64 po,
                                                const u8* __restrict__ pb, u64 len, u64 eff, u64& m, u64& alg) {
    const unsigned lane = lane_id();
    const u64 m0 = m;
    u64 k = m;
    while (k < eff) {
        const u64 q = k + 16 * u64(lane);
        u64 tw = 0, pw = 0;
        if (q < eff) {
            const u64 w = eff - q;
            tw = x + q < n1 ? mask16(load16(PT, x + q), w) : 0;     // past the end of the strand: padding (code 0)
            pw = mask16(load16(PP, po + q), w);
        }
        const unsigned diff = __ballot_sync(0xffffffffu, tw != pw);
        if (diff) {
            const int l = __ffs(diff) - 1;
            const u64 t = __shfl_sync(0xffffffffu, tw, l), p = __shfl_sync(0xffffffffu, pw, l);
            m = k + 16 * u64(l) + u64(__clzll(t ^ p) >> 2);
            alg += alg_of_compare(m + 1 - m0);
            return t < p ? -1 : 1;
        }
        k += eff - k < 512 ? eff - k : 512;
    }
    m = k;
    alg += alg_of_compare(k + 1 - m0);
    return cmp_at_cut(PT, n1, x, pb, len, k);
}

// The part of a sorted index that can hold P: the deep bucket of its first deep_depth symbols when they are ACGT, else
// the 8-mer bucket when its first 8 are in ACGNT; only buckets that are not empty (an empty 8-mer bucket's values are
// unspecified, and between two deep buckets lie suffixes with N or '$' early on, which P may sort before). A deep range
// [deep[s], deep[s+1]) starts with every suffix that begins with s; what follows it sorts after every such suffix.
template <typename IdxT>
__device__ __forceinline__ void locate_narrow(const LocateParams<IdxT>& P, const Win& pw0, u64 eff, u64& L, u64& R) {
    L = 0; R = P.sa_len;
    u32 slot = 0;
    if (P.deep && eff >= u64(P.deep_depth) && deep_slot(pw0.hi, P.deep_depth, slot)) {
        const u64 lo = u64(P.deep[slot]), hi = u64(P.deep[slot + 1]);
        if (lo < hi) { L = lo; R = hi; return; }
    }
    if (eff >= 8 && lut_slot(pw0.hi, slot)) {
        const u64 lo = u64(P.lut_lo[slot]), hi = u64(P.lut_hi[slot]);
        if (lo < hi) { L = lo; R = hi; }
    }
}

__device__ __forceinline__ void locate_account(unsigned long long* ctr, u64 alg) {
    const u64 w = warp_sum_u64(alg);
    if (lane_id() == 0 && w) atomicAdd(ctr, (unsigned long long)w);
}

// Full index, patterns of <= 32 bytes: one lane each. Lower bound (first suffix >= P), then upper bound from there.
template <typename IdxT>
__global__ void __launch_bounds__(256) locate_short_kernel(const LocateParams<IdxT> P) {
    const u64 t = u64(blockIdx.x) * blockDim.x + threadIdx.x;
    u64 alg = 0;
    if (t < P.n_list) {
        const u64 p = P.list ? u64(P.list[t]) : t;
        const u64 po = P.off[p], len = P.off[p + 1] - po;
        const u64 eff = P.cut[p] < len ? P.cut[p] : len;
        const u8* pb = P.pat + po;
        const Win pw0 = mask_window(load_window(P.PP, po), eff == 0 ? 1 : int(eff));   // eff 0: unused
        u64 L, R;
        if (eff == 0) { L = 0; R = P.sa_len; } else locate_narrow(P, pw0, eff, L, R);
        const IdxT* __restrict__ SA = P.SA;
        u64 lo = L, hi = R;
        while (lo < hi) {
            const u64 mid = lo + ((hi - lo) >> 1);
            u64 m = 0;
            if (cmp_pattern(P.PT, P.n1, u64(SA[mid]), P.PP, po, pb, len, eff, m, alg) < 0) lo = mid + 1; else hi = mid;
        }
        const u64 first = lo;
        hi = R;
        while (lo < hi) {
            const u64 mid = lo + ((hi - lo) >> 1);
            u64 m = 0;
            if (cmp_pattern(P.PT, P.n1, u64(SA[mid]), P.PP, po, pb, len, eff, m, alg) <= 0) lo = mid + 1; else hi = mid;
        }
        P.first[p] = i64(first);
        P.count[p] = i64(lo - first);
    }
    locate_account(P.alg_bytes, alg);
}

// Full index, patterns longer than 32 bytes: one warp each, the bisection skips the prefix both bounds already share
// with P (sorted array: every suffix between them shares it too), so a long pattern is not read again from its start at
// every step.
template <typename IdxT>
__global__ void __launch_bounds__(256) locate_long_kernel(const LocateParams<IdxT> P) {
    const u64 t = (u64(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    if (t >= P.n_list) return;
    const u64 p = P.list ? u64(P.list[t]) : t;
    const u64 po = P.off[p], len = P.off[p + 1] - po;
    const u64 eff = P.cut[p] < len ? P.cut[p] : len;
    const u8* pb = P.pat + po;
    u64 alg = 0, L, R;
    if (eff == 0) { L = 0; R = P.sa_len; }
    else locate_narrow(P, mask_window(load_window(P.PP, po), eff < 32 ? int(eff) : 32), eff, L, R);
    const IdxT* __restrict__ SA = P.SA;
    u64 lo = L, hi = R, lm = 0, rm = 0;
    while (lo < hi) {
        const u64 mid = lo + ((hi - lo) >> 1);
        u64 m = lm < rm ? lm : rm;
        if (cmp_pattern_warp(P.PT, P.n1, u64(SA[mid]), P.PP, po, pb, len, eff, m, alg) < 0) { lo = mid + 1; lm = m; }
        else { hi = mid; rm = m; }
    }
    const u64 first = lo;
    hi = R; lm = 0; rm = 0;
    while (lo < hi) {
        const u64 mid = lo + ((hi - lo) >> 1);
        u64 m = lm < rm ? lm : rm;
        if (cmp_pattern_warp(P.PT, P.n1, u64(SA[mid]), P.PP, po, pb, len, eff, m, alg) <= 0) { lo = mid + 1; lm = m; }
        else { hi = mid; rm = m; }
    }
    if (lane_id() == 0) {
        P.first[p] = i64(first);
        P.count[p] = i64(lo - first);
        if (alg) atomicAdd(P.alg_bytes, (unsigned long long)alg);
    }
}

// Index built with --trim: not sorted for the strand it is compared with (SURVEY Q9), so the answer is whatever the
// reference's own bisection lands on. literal_bucket / literal_descent (kmer_core.h) for any pattern length: the same
// middles and the same `match` skipping as sa_search (oracle: sa_search_literal).
template <typename IdxT>
__global__ void __launch_bounds__(256) locate_literal_kernel(const LocateParams<IdxT> P) {
    const u64 t = u64(blockIdx.x) * blockDim.x + threadIdx.x;
    u64 alg = 0;
    if (t < P.n_list) {
        const u64 p = P.list ? u64(P.list[t]) : t;
        const u64 po = P.off[p], len = P.off[p + 1] - po;
        const u64 eff = P.cut[p] < len ? P.cut[p] : len;
        const u8* pb = P.pat + po;
        const IdxT* __restrict__ SA = P.SA;
        i64 first = 0, count = i64(P.sa_len);
        if (len > 0) {
            auto cmp = [&](u64 ix, u64& m) { return cmp_pattern(P.PT, P.n1, u64(SA[ix]), P.PP, po, pb, len, eff, m, alg); };
            i64 i = 0, j = 0, k = 0;
            u64 lmatch = 0, rmatch = 0;
            i64 size = i64(P.sa_len), half = size >> 1;
            while (size > 0) {
                u64 match = lmatch < rmatch ? lmatch : rmatch;
                const int r = cmp(u64(i + half), match);
                if (r < 0) {
                    i += half + 1;
                    half -= (size & 1) ^ 1;
                    lmatch = match;
                } else if (r > 0) {
                    rmatch = match;
                } else {
                    i64 lsize = half, rsize = size - half - 1;
                    j = i; k = i + half + 1;
                    u64 llmatch = lmatch, lrmatch = match;
                    for (i64 h = lsize >> 1; lsize > 0; lsize = h, h >>= 1) {      // first suffix >= P in the left part
                        u64 mm = llmatch < lrmatch ? llmatch : lrmatch;
                        if (cmp(u64(j + h), mm) < 0) { j += h + 1; h -= (lsize & 1) ^ 1; llmatch = mm; }
                        else lrmatch = mm;
                    }
                    u64 rlmatch = match, rrmatch = rmatch;
                    for (i64 h = rsize >> 1; rsize > 0; rsize = h, h >>= 1) {      // first suffix > P in the right part
                        u64 mm = rlmatch < rrmatch ? rlmatch : rrmatch;
                        if (cmp(u64(k + h), mm) <= 0) { k += h + 1; h -= (rsize & 1) ^ 1; rlmatch = mm; }
                        else rrmatch = mm;
                    }
                    break;
                }
                size = half; half >>= 1;
            }
            first = (k - j) > 0 ? j : i;
            count = k - j;
        }
        P.first[p] = first;
        P.count[p] = count;
    }
    locate_account(P.alg_bytes, alg);
}

// pattern bytes -> packed codes, 16 per thread; a byte without a code packs as 0 and lowers its pattern's cut
__global__ void __launch_bounds__(256) locate_pack_kernel(const u8* __restrict__ pat, u64 n_bytes, const u64* __restrict__ off,
                                                          u64 n_patterns, u64* __restrict__ packed, u64 n_words,
                                                          unsigned long long* __restrict__ cut) {   // cut: u64 viewed for atomicMin
    const u64 w = u64(blockIdx.x) * blockDim.x + threadIdx.x;
    if (w >= n_words) return;
    u64 word = 0, seen_end = 0;   // bytes before seen_end belong to a pattern whose cut this thread has lowered already
#pragma unroll 4
    for (u32 j = 0; j < 16; ++j) {
        const u64 pos = w * 16 + j;
        if (pos >= n_bytes) break;
        const u32 c = code_of_byte_tab(pat[pos], kCodeTab);
        if (c != CODE_BAD) { word |= u64(c) << (60 - 4 * j); continue; }
        if (pos < seen_end) continue;
        u64 lo = 0, hi = n_patterns;   // last pattern p with off[p] <= pos (the one that holds the byte)
        while (hi - lo > 1) {
            const u64 mid = (lo + hi) >> 1;
            if (off[mid] <= pos) lo = mid; else hi = mid;
        }
        seen_end = off[lo + 1];
        atomicMin(&cut[lo], (unsigned long long)(pos - off[lo]));
    }
    packed[w] = word;
}

// positions: pattern p's hits are out-slots [moff[p], moff[p] + min(count[p], cap)) of the slice; this launch writes the
// window [w0, w1) of them, to out[0 .. w1 - w0)
template <typename IdxT>
__global__ void __launch_bounds__(256) locate_copy_kernel(const IdxT* __restrict__ SA, const i64* __restrict__ first,
                                                          const i64* __restrict__ count, const u64* __restrict__ moff, u64 n_patterns,
                                                          u64 cap, u64 w0, u64 w1, i64* __restrict__ out) {
    const u64 p = (u64(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    if (p >= n_patterns) return;
    const u64 c = u64(count[p]) < cap ? u64(count[p]) : cap;
    const u64 o = moff[p];
    const u64 s = o > w0 ? o : w0, e = o + c < w1 ? o + c : w1;
    if (s >= e) return;
    const IdxT* __restrict__ src = SA + (u64(first[p]) + (s - o));
    i64* __restrict__ dst = out + (s - w0);
    for (u64 j = lane_id(); j < e - s; j += 32) dst[j] = i64(src[j]);
}

}  // namespace ab200
