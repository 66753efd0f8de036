// sa_build.cuh — on-GPU suffix-array construction by prefix doubling (replaces libdivsufsort behind
// src/divsufsort.rs:10 / r_divsufsort, src/bin/asgart.rs:473-479, of the reference).
//
// The suffix array of a text is unique, so any correct construction reproduces divsufsort64's output bit for bit
// (checked against the reference's own library in tests/). Algorithm (Larsson–Sadakane doubling with discarding,
// laid out for a GPU):
//   0. byte histogram -> dense symbol codes 1..sigma (0 = "past the end", which orders a suffix that is a prefix of
//      another one first, as divsufsort does); b bits per symbol.
//   1. initial sort of (key, i), key[i] = first p0 symbols of suffix i. Genome-sized texts over small alphabets: the MSD
//      sort of msd_sort.cuh (12-bit partition levels while a bucket is large, then one sort in shared memory) with as many
//      symbols as 63 bits hold (DNA + '$': sigma = 6, b = 3, p0 = 21). Short texts, wide alphabets, or when the MSD sort
//      declines: key generation + stable LSD radix passes over b*p0 bits, p0 sized so that random text is almost resolved.
//   2. group heads by key change (hp_reduce / hp_emit) -> SA[] for all; suffixes in groups of size > 1 are compacted into
//      the work list (G = group head index, I = suffix), those whose p0 symbols are all equal into the run round's list.
//      rank[] (= SA index of the group head) is NOT materialised after the MSD sort: it starts as a sentinel and a gather
//      that meets the sentinel looks the initial rank up in the sorted keys (initial_rank below: "lazy ranks"); builds
//      without lookup tables write rank[SA[i]] = head(i) for every i (scatter.cuh).
//   3. run round: runs of >= p0 equal symbols (N-runs) ordered by (symbol after the run, run length) in one sort.
//   4. doubling rounds h = p0, 2p0, ...: key2 = rank[I + h] + 1 (0 past the end)  [random gather],
//      segmented sort of the work list by (G, key2), re-rank, write SA for suffixes that became unique, drop them,
//      until the work list is empty.
// Sharded form (SaGroup, sa_group.h; world > 1): member r owns the suffixes whose first four symbols fall into its range of
// level-0 bins (ranges cut from the histogram the members count together, ~n/world suffixes each) and runs steps 1-4 on
// them; group heads and SA slots are global indices (range base + local position). The rank array is cut into contiguous
// slices by position (RankView): every re-ranking is stored straight into the owner's memory and the gather of step 4
// reads from it (NVLink peer access); a lazy initial rank is looked up in the sorted keys of the member that owns the
// key's bin (RankLookup: peer pointers to every member's keys). Two collectives per doubling round keep reads and writes
// of rank[] apart; the SA pieces are exchanged once at the end.
// Index width is a template parameter: u32 when n < 2^32 - 1 (all BASELINE configs), u64 beyond (composite keys then
// need 128 bits: U128). Both paths are exercised by the tests on small inputs.
#pragma once
#include <cmath>
#include <cstdlib>
#include <vector>

#include "common.cuh"
#include "msd_sort.cuh"
#include "radix_sort.cuh"
#include "sa_group.h"
#include "scan.cuh"
#include "scatter.cuh"
#include "search.cuh"

namespace ab200 {

struct SaStats {
    FamilyTimer* sort = nullptr;    // radix passes
    FamilyTimer* scatter = nullptr; // rs_scatter_kernel alone (sorts of the run round and the doubling rounds)
    FamilyTimer* scatter_main = nullptr; // rs_scatter_kernel of the initial sort: every launch moves all n suffixes
    FamilyTimer* gather = nullptr;  // rank[I + h] gathers
    FamilyTimer* rank = nullptr;    // re-rank / compaction scans
    MsdStats msd;                   // initial sort, MSD form (msd_sort.cuh)
    bool used_msd = false;
    u64 rounds = 0;
};

// ---------------------------------------------------------------------------------------------------------------
__global__ void byte_hist_kernel(const u8* __restrict__ t, u64 n, unsigned long long* __restrict__ hist) {
    __shared__ u32 h[256];
    h[threadIdx.x] = 0;  // 256 threads
    __syncthreads();
    const u64 stride = u64(gridDim.x) * blockDim.x * 16;
    for (u64 i = (u64(blockIdx.x) * blockDim.x + threadIdx.x) * 16; i < n; i += stride) {
        if (i + 16 <= n && (reinterpret_cast<uintptr_t>(t + i) & 15) == 0) {
            uint4 v = *reinterpret_cast<const uint4*>(t + i);
            u32 w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                atomicAdd(&h[w[k] & 255], 1u); atomicAdd(&h[(w[k] >> 8) & 255], 1u);
                atomicAdd(&h[(w[k] >> 16) & 255], 1u); atomicAdd(&h[w[k] >> 24], 1u);
            }
        } else {
            for (u64 j = i; j < n && j < i + 16; ++j) atomicAdd(&h[t[j]], 1u);
        }
    }
    __syncthreads();
    if (h[threadIdx.x]) atomicAdd(&hist[threadIdx.x], (unsigned long long)h[threadIdx.x]);
}

constexpr int kInitThreads = 256;
constexpr int kInitItems = 16;
constexpr int kInitTile = kInitThreads * kInitItems;

// key[i] = codes of T[i .. i+p0) packed most-significant-first, b bits each; vals[i] = i.
// Each thread rolls the key over 16 consecutive positions; the tile's keys go through shared memory (padded against
// bank conflicts) so that they leave the SM as coalesced stores.
template <typename IdxT>
__global__ void __launch_bounds__(kInitThreads) init_keys_kernel(const u8* __restrict__ text, u64 n, const uint16_t* __restrict__ code,
                                                                  int b, int p0, u64* __restrict__ keys, IdxT* __restrict__ vals) {
    __shared__ uint16_t sc[kInitTile + 64];   // codes reach 256 when every byte value occurs
    __shared__ uint16_t scode[256];
    __shared__ u64 skey[kInitTile + kInitThreads];
    scode[threadIdx.x] = code[threadIdx.x];
    __syncthreads();
    const u64 base = u64(blockIdx.x) * kInitTile;
    for (u32 i = threadIdx.x; i < kInitTile + 64; i += kInitThreads) {
        u64 p = base + i;
        sc[i] = p < n ? scode[text[p]] : uint16_t(0);
    }
    __syncthreads();
    const u32 t0 = threadIdx.x * kInitItems;
    const u64 mask = (b * p0 >= 64) ? ~u64(0) : ((u64(1) << (b * p0)) - 1);
    u64 key = 0;
    for (int j = 0; j < p0; ++j) key = (key << b) | sc[t0 + j];
#pragma unroll
    for (int j = 0; j < kInitItems; ++j) {
        skey[t0 + j + threadIdx.x] = key;   // element e lives at e + e / kInitItems
        key = ((key << b) & mask) | sc[t0 + j + p0];
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < kInitItems; ++j) {
        const u32 e = j * kInitThreads + threadIdx.x;
        const u64 p = base + e;
        if (p < n) { keys[p] = skey[e + e / kInitItems]; vals[p] = IdxT(p); }
    }
}


// ---- first re-ranking (step 2): group heads, rank by sorted position and the two work lists, from the sorted initial keys ----
// The generic flag scan (scan.cuh) spends ~80 (reduce) + ~160 (output) instructions per element on this pass — at 3.1 G
// suffixes it is bound by issue slots, not by HBM. Here one thread owns 8 consecutive keys (four 128-bit loads), the
// flags of its keys need two neighbour keys only, and the scan state is three words per thread:
//   latest head inside the tile (1-based, 0 = none)   -> running maximum
//   #unsorted ordinary | #unsorted pure << 16          -> running sums   (pure: all p0 symbols equal, the run round's share)
//   #unsorted ordinary heads                           -> running sum
constexpr int kHpThreads = 256;
constexpr int kHpItems = 8;
constexpr int kHpTile = kHpThreads * kHpItems;

struct HpThreadAcc {
    u32 head1, cd, e;
    HpThreadAcc() = default;
    __host__ __device__ explicit HpThreadAcc(int) : head1(0), cd(0), e(0) {}
};
struct HpThreadOp {
    __device__ __forceinline__ HpThreadAcc operator()(const HpThreadAcc& x, const HpThreadAcc& y) const {
        HpThreadAcc r(0);
        r.head1 = x.head1 > y.head1 ? x.head1 : y.head1;
        r.cd = x.cd + y.cd;
        r.e = x.e + y.e;
        return r;
    }
};
struct HpTileAcc {   // per tile / grand total: head1 = 1-based index (inside the member's piece) of the latest head
    u64 head1, c, d, e;
    HpTileAcc() = default;
    __host__ __device__ explicit HpTileAcc(int) : head1(0), c(0), d(0), e(0) {}
};
struct HpTileOp {
    __device__ __forceinline__ HpTileAcc operator()(const HpTileAcc& x, const HpTileAcc& y) const {
        HpTileAcc r(0);
        r.head1 = x.head1 > y.head1 ? x.head1 : y.head1;
        r.c = x.c + y.c; r.d = x.d + y.d; r.e = x.e + y.e;
        return r;
    }
};

// this thread's 8 keys, its flag masks (bit j = key j) and its summary
struct HpThread {
    u64 k[kHpItems];
    u64 i0;
    u32 valid, head, unsorted, pure;
};

__device__ __forceinline__ void hp_load(const u64* __restrict__ kk, u64 n, u64 rep_unit, u64 sym_mask, HpThread& t) {
    t.i0 = u64(blockIdx.x) * kHpTile + u64(threadIdx.x) * kHpItems;
    const u32 cnt = t.i0 >= n ? 0u : u32(n - t.i0 < u64(kHpItems) ? n - t.i0 : u64(kHpItems));
    t.valid = (1u << cnt) - 1u;
    t.head = t.unsorted = t.pure = 0;
    if (cnt == 0) return;
    if (cnt == kHpItems) {
        const ulonglong2* p = reinterpret_cast<const ulonglong2*>(kk + t.i0);
#pragma unroll
        for (int q = 0; q < kHpItems / 2; ++q) { const ulonglong2 v = p[q]; t.k[2 * q] = v.x; t.k[2 * q + 1] = v.y; }
    } else {
#pragma unroll
        for (int j = 0; j < kHpItems; ++j) t.k[j] = u32(j) < cnt ? kk[t.i0 + j] : 0;
    }
    const bool has_prev = t.i0 > 0, has_next = t.i0 + cnt < n;
    const u64 prev = has_prev ? kk[t.i0 - 1] : 0, next = has_next ? kk[t.i0 + cnt] : 0;
    u32 tail = 0;
#pragma unroll
    for (int j = 0; j < kHpItems; ++j) {
        if (u32(j) < cnt) {
            const u64 cur = t.k[j];
            const bool hd = j == 0 ? (!has_prev || prev != cur) : (t.k[j - 1] != cur);
            const bool tl = u32(j) + 1 == cnt ? (!has_next || next != cur) : (t.k[j + 1] != cur);
            t.head |= u32(hd) << j;
            tail |= u32(tl) << j;
            t.pure |= u32(cur == (cur & sym_mask) * rep_unit) << j;
        }
    }
    t.unsorted = ~(t.head & tail) & t.valid;
}

__device__ __forceinline__ HpThreadAcc hp_thread_acc(const HpThread& t) {
    HpThreadAcc a(0);
    a.head1 = t.head ? u32(threadIdx.x) * kHpItems + (31 - __clz(t.head)) + 1 : 0u;
    const u32 ord = t.unsorted & ~t.pure;
    a.cd = u32(__popc(ord)) | (u32(__popc(t.unsorted & t.pure)) << 16);
    a.e = u32(__popc(ord & t.head));
    return a;
}

__global__ void __launch_bounds__(kHpThreads) hp_reduce_kernel(const u64* __restrict__ kk, u64 n, u64 rep_unit, u64 sym_mask,
                                                               HpTileAcc* __restrict__ tile_acc) {
    __shared__ HpThreadAcc sm[32];
    HpThread t;
    hp_load(kk, n, rep_unit, sym_mask, t);
    HpThreadAcc total;
    block_exclusive_scan(hp_thread_acc(t), HpThreadOp(), total, sm);
    if (threadIdx.x == 0) {
        HpTileAcc r(0);
        r.head1 = total.head1 ? u64(blockIdx.x) * kHpTile + total.head1 : 0;
        r.c = total.cd & 0xffffu; r.d = total.cd >> 16; r.e = total.e;
        tile_acc[blockIdx.x] = r;
    }
}

// rpos[i] = b0 + index of the head of i's group; unsorted suffixes go to the ordinary list (ga, ia; hsa = list index of every
// group's first entry) or, when their p0 symbols are all equal, to the run round's list (gs, is)
template <typename IdxT>
__global__ void __launch_bounds__(kHpThreads) hp_emit_kernel(const u64* __restrict__ kk, const IdxT* __restrict__ vv, u64 n, u64 rep_unit,
                                                             u64 sym_mask, const HpTileAcc* __restrict__ tile_pre, IdxT b0,
                                                             IdxT* __restrict__ rpos, IdxT* __restrict__ ga, IdxT* __restrict__ ia,
                                                             IdxT* __restrict__ hsa, IdxT* __restrict__ gs, IdxT* __restrict__ is) {
    __shared__ HpThreadAcc sm[32];
    HpThread t;
    hp_load(kk, n, rep_unit, sym_mask, t);
    HpThreadAcc total;
    const HpThreadAcc exc = block_exclusive_scan(hp_thread_acc(t), HpThreadOp(), total, sm);
    if (t.valid == 0) return;
    const HpTileAcc pre = tile_pre[blockIdx.x];
    const u64 tile0 = u64(blockIdx.x) * kHpTile;
    u64 head1 = exc.head1 ? tile0 + exc.head1 : pre.head1;     // 1-based index of the latest head before this thread
    u64 c = pre.c + (exc.cd & 0xffffu), d = pre.d + (exc.cd >> 16), e = pre.e + exc.e;
    IdxT hd[kHpItems];
#pragma unroll
    for (int j = 0; j < kHpItems; ++j) {
        if ((t.head >> j) & 1u) head1 = t.i0 + j + 1;
        hd[j] = b0 + IdxT(head1 - 1);
    }
    if (rpos == nullptr) {
        // lazy ranks: no rank-by-sorted-position array is written
    } else if (t.valid == (1u << kHpItems) - 1u) {
        if constexpr (sizeof(IdxT) == 4) {
            uint4* o = reinterpret_cast<uint4*>(rpos + t.i0);
            o[0] = make_uint4(u32(hd[0]), u32(hd[1]), u32(hd[2]), u32(hd[3]));
            o[1] = make_uint4(u32(hd[4]), u32(hd[5]), u32(hd[6]), u32(hd[7]));
        } else {
            ulonglong2* o = reinterpret_cast<ulonglong2*>(rpos + t.i0);
#pragma unroll
            for (int q = 0; q < kHpItems / 2; ++q) o[q] = make_ulonglong2(u64(hd[2 * q]), u64(hd[2 * q + 1]));
        }
    } else {
#pragma unroll
        for (int j = 0; j < kHpItems; ++j) if ((t.valid >> j) & 1u) rpos[t.i0 + j] = hd[j];
    }
    if (t.unsorted == 0) return;
#pragma unroll
    for (int j = 0; j < kHpItems; ++j) {
        if ((t.unsorted >> j) & 1u) {
            const IdxT idx = vv[t.i0 + j];
            if ((t.pure >> j) & 1u) { gs[d] = hd[j]; is[d] = idx; ++d; }
            else {
                ga[c] = hd[j]; ia[c] = idx;
                if ((t.head >> j) & 1u) hsa[e++] = IdxT(c);
                ++c;
            }
        }
    }
}

// ---- sharded build: key-range selection -----------------------------------------------------------------------
// histogram of the first `psym` symbols (b bits each) of every suffix: the members cut their key ranges from it
__global__ void __launch_bounds__(256) key_prefix_hist_kernel(const u8* __restrict__ text, u64 n, const uint16_t* __restrict__ code, int b,
                                                              int psym, unsigned long long* __restrict__ hist) {
    extern __shared__ u32 kp_hist[];
    __shared__ uint16_t scode[256];
    const u32 nb = 1u << (b * psym);
    for (u32 i = threadIdx.x; i < nb; i += blockDim.x) kp_hist[i] = 0;
    scode[threadIdx.x] = code[threadIdx.x];
    __syncthreads();
    const u64 stride = u64(gridDim.x) * blockDim.x;
    const u64 n_up = (n + 31) / 32 * 32;   // whole warps stay in the loop: the vote below needs all lanes
    for (u64 p = u64(blockIdx.x) * blockDim.x + threadIdx.x; p < n_up; p += stride) {
        u32 pre = 0;
        for (int j = 0; j < psym; ++j) pre = (pre << b) | ((p + j < n) ? u32(scode[text[p + j]]) : 0u);
        const bool valid = p < n;
        // runs of one symbol put the whole warp on one counter: one add for all of them
        const u32 first = __shfl_sync(0xffffffffu, pre, 0);
        if (__all_sync(0xffffffffu, valid && pre == first)) { if (lane_id() == 0) atomicAdd(&kp_hist[pre], 32u); }
        else if (valid) atomicAdd(&kp_hist[pre], 1u);
    }
    __syncthreads();
    for (u32 i = threadIdx.x; i < nb; i += blockDim.x)
        if (kp_hist[i]) atomicAdd(&hist[i], (unsigned long long)kp_hist[i]);
}

// init_keys_kernel restricted to the keys whose prefix (key >> pshift) lies in [pre_lo, pre_hi): WRITE = false counts them
// per tile, WRITE = true writes them, in text order, behind the tile's offset.
template <typename IdxT, bool WRITE>
__global__ void __launch_bounds__(kInitThreads) init_keys_range_kernel(const u8* __restrict__ text, u64 n, const uint16_t* __restrict__ code, int b,
                                                                        int p0, int pshift, u32 pre_lo, u32 pre_hi, u64* __restrict__ tile_cnt,
                                                                        const u64* __restrict__ tile_off, u64* __restrict__ keys,
                                                                        IdxT* __restrict__ vals) {
    __shared__ uint16_t sc[kInitTile + 64];
    __shared__ uint16_t scode[256];
    __shared__ u32 wsm[32];
    scode[threadIdx.x] = code[threadIdx.x];
    __syncthreads();
    const u64 base = u64(blockIdx.x) * kInitTile;
    for (u32 i = threadIdx.x; i < kInitTile + 64; i += kInitThreads) {
        const u64 p = base + i;
        sc[i] = p < n ? scode[text[p]] : uint16_t(0);
    }
    __syncthreads();
    const u32 t0 = threadIdx.x * kInitItems;
    const u64 mask = (b * p0 >= 64) ? ~u64(0) : ((u64(1) << (b * p0)) - 1);
    u64 key = 0;
    for (int j = 0; j < p0; ++j) key = (key << b) | sc[t0 + j];
    u64 kk[kInitItems];
    u32 sel = 0, cnt = 0;
#pragma unroll
    for (int j = 0; j < kInitItems; ++j) {
        kk[j] = key;
        const u32 pre = u32(key >> pshift);
        if (base + t0 + j < n && pre >= pre_lo && pre < pre_hi) { sel |= 1u << j; ++cnt; }
        key = ((key << b) & mask) | sc[t0 + j + p0];
    }
    u32 total;
    const u32 exc = block_exclusive_scan(cnt, SumOp(), total, wsm);
    if (!WRITE) {
        if (threadIdx.x == 0) tile_cnt[blockIdx.x] = total;
    } else {
        u64 w = tile_off[blockIdx.x] + exc;
#pragma unroll
        for (int j = 0; j < kInitItems; ++j)
            if ((sel >> j) & 1u) { keys[w] = kk[j]; vals[w] = IdxT(base + t0 + j); ++w; }
    }
}

// rank[suffix] = value, through the view (sharded build: most targets live in a peer's memory)
template <typename IdxT>
__global__ void __launch_bounds__(256) scatter_view_kernel(const IdxT* __restrict__ idx, const IdxT* __restrict__ val, u64 n, RankView<IdxT> rv) {
    const u64 stride = u64(gridDim.x) * blockDim.x;
    for (u64 i = u64(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) *rv.ptr(u64(idx[i])) = val[i];
}

// ---------------------------------------------------------------------------------------------------------------
// composite (group, key2) keys of the large-group radix path
template <typename IdxT> struct CompKey;
template <> struct CompKey<u32> {
    using type = u64;
    __device__ static __forceinline__ u64 make(u32 g, u32 k2, int kb) { return (u64(g) << kb) | u64(k2); }
    __device__ static __forceinline__ u32 key2(u64 k, int kb) { return u32(k & ((u64(1) << kb) - 1)); }
};
template <> struct CompKey<u64> {
    using type = U128;
    __device__ static __forceinline__ U128 make(u64 g, u64 k2, int) { return U128{g, k2}; }
    __device__ static __forceinline__ u64 key2(const U128& k, int) { return k.lo; }
};

constexpr int kSmallGroup = 32;  // groups up to this size are sorted in place by one thread; larger ones go through radix passes

// key2 = rank of the suffix D symbols further on (+1; 0 = past the end): the random gather of prefix doubling
// ---- lazy ranks (single-device build) ---------------------------------------------------------------------------
// rank[j] = sorted position of the head of j's group. Right after the initial sort that is lower_bound(sorted keys,
// key(j)) for EVERY position j, and only 9 % of the suffixes (the unsorted ones) ever ask for a rank — of positions further
// on in the text. So the inverse permutation rank[SA[i]] = head(i) is never materialised (3.09 G pairs through two
// partition passes and a bucket scatter: 55 ms at 3.1 Gbp): rank[] starts as all-ones = "still the initial head", the
// re-ranking stores explicit values for suffixes that leave the first sub-group of their group (a first sub-group keeps its
// head, so the sentinel stays true), and a gather that meets the sentinel computes the initial head from the text: key of
// the suffix -> bucket of its first `depth` symbols in the deep table (~3 sorted keys) -> position of its key among them.
template <typename IdxT>
struct RankLookup {
    const u64* keys[kMaxWorld] = {};   // sorted initial keys: member r holds sorted positions [piece[r], piece[r + 1])
    u64 piece[kMaxWorld + 1] = {};
    u32 world = 1;
    const u8* text = nullptr;
    const uint16_t* code = nullptr;
    u64 n = 0;
    int b = 0, p0 = 0, depth = 0;
    const IdxT* deep = nullptr;
    const IdxT* lut_lo = nullptr;
    const IdxT* lut_hi = nullptr;
    u64 m4 = 0, m5 = 0;
    __device__ __forceinline__ u32 owner(u64 p) const {
        u32 r = 0;
        while (r + 1 < world && p >= piece[r + 1]) ++r;
        return r;
    }
};

template <typename IdxT>
__device__ __forceinline__ IdxT initial_rank(const RankLookup<IdxT>& L, u64 j) {
    u64 key = 0;
    for (int t = 0; t < L.p0; ++t) {
        const u64 p = j + u64(t);
        key = (key << L.b) | (p < L.n ? u64(__ldg(&L.code[L.text[p]])) : 0);
    }
    u64 lo = 0, hi = L.n;
    u32 slot = 0;
    bool one_owner = L.world == 1;
    if (L.depth > 0 && key_slot4(key, L.b, L.p0, L.depth, L.m4, slot)) { lo = u64(L.deep[slot]); hi = u64(L.deep[slot + 1]); one_owner = true; }
    else if (L.p0 >= 8 && key_slot5(key, L.b, L.p0, L.m5, slot)) { lo = u64(L.lut_lo[slot]); hi = u64(L.lut_hi[slot]); one_owner = true; }
    if (one_owner) {
        // a bucket of >= 4 leading symbols lies inside one member's piece (the pieces are cut where the first four symbols change)
        const u32 r = L.owner(lo);
        const u64* __restrict__ kk = L.keys[r] - L.piece[r];
        while (hi - lo > 4) {   // first entry >= key (the suffix's own key is in there)
            const u64 mid = (lo + hi) >> 1;
            if (kk[mid] < key) lo = mid + 1; else hi = mid;
        }
        while (lo < hi && kk[lo] < key) ++lo;
    } else {
        while (lo < hi) {       // the few suffixes that reach past the end of the text: the whole array, whoever holds it
            const u64 mid = (lo + hi) >> 1;
            const u32 r = L.owner(mid);
            if (L.keys[r][mid - L.piece[r]] < key) lo = mid + 1; else hi = mid;
        }
    }
    return IdxT(lo);
}

template <typename IdxT, bool LAZY>
__global__ void gather_rank_kernel(const IdxT* __restrict__ I, const IdxT* __restrict__ D, const RankView<IdxT> rank, u64 U, u64 n,
                                   IdxT* __restrict__ K2, const RankLookup<IdxT> L) {
    const u64 stride = u64(gridDim.x) * blockDim.x;
    for (u64 c = u64(blockIdx.x) * blockDim.x + threadIdx.x; c < U; c += stride) {
        const u64 p = u64(I[c]) + u64(D[c]);
        IdxT v = IdxT(0);
        if (p < n) {
            IdxT* rp = rank.ptr(p);
            v = *rp;
            // never re-ranked: still the head its initial key gives. Written back: positions inside long repeats are asked for
            // again in later rounds (i + D for several (i, D)); measured at 3.1 Gbp: 45 ms of gathers with the store, 55 without
            if (LAZY && v == ~IdxT(0)) {
                v = initial_rank<IdxT>(L, p);
                *rp = v;
            }
            v = IdxT(v + 1);
        }
        K2[c] = v;
    }
}

// one thread per group: groups of <= kSmallGroup suffixes are insertion-sorted by key2 in place, larger ones report
// their size for the radix path
template <typename IdxT>
__global__ void small_group_sort_kernel(const IdxT* __restrict__ hs, u64 n_groups, u64 U, IdxT* __restrict__ K2, IdxT* __restrict__ I,
                                        IdxT* __restrict__ large_sz) {
    const u64 j = u64(blockIdx.x) * blockDim.x + threadIdx.x;
    if (j >= n_groups) return;
    const u64 s = hs[j], m = (j + 1 < n_groups ? u64(hs[j + 1]) : U) - s;
    if (m > kSmallGroup) { large_sz[j] = IdxT(m); return; }
    large_sz[j] = 0;
    for (u64 r = 1; r < m; ++r) {
        const IdxT k = K2[s + r], v = I[s + r];
        u64 w = r;
        while (w > 0 && K2[s + w - 1] > k) { K2[s + w] = K2[s + w - 1]; I[s + w] = I[s + w - 1]; --w; }
        if (w != r) { K2[s + w] = k; I[s + w] = v; }
    }
}

// last j with arr[j] <= v   (arr non-decreasing, arr[0] <= v)
template <typename IdxT>
__device__ __forceinline__ u64 last_le(const IdxT* __restrict__ arr, u64 len, u64 v) {
    u64 lo = 0, hi = len;
    while (hi - lo > 1) {
        const u64 mid = (lo + hi) >> 1;
        if (u64(arr[mid]) <= v) lo = mid; else hi = mid;
    }
    return lo;
}

// one thread per slot of the large-group buffer (not per list entry: large groups are rare, the list is not — a pass
// over all 281 M entries of round 1 at 3.1 Gbp cost 6.3 ms to move a handful of groups)
template <typename IdxT>
__global__ void large_copy_out_kernel(const IdxT* __restrict__ hs, const IdxT* __restrict__ loff, u64 n_groups, u64 UL,
                                      const IdxT* __restrict__ K2, const IdxT* __restrict__ I, int kb,
                                      typename CompKey<IdxT>::type* __restrict__ Lk, IdxT* __restrict__ Li) {
    const u64 q = u64(blockIdx.x) * blockDim.x + threadIdx.x;
    if (q >= UL) return;
    const u64 j = last_le(loff, n_groups, q);  // the large group that owns slot q (last index of the plateau)
    const u64 c = u64(hs[j]) + (q - u64(loff[j]));
    // keyed on the group's ordinal in the list, not its head index: the list is grouped but not globally ordered by head
    // (ordinary groups first, then the run groups), and the sorted elements are copied back in list order
    Lk[q] = CompKey<IdxT>::make(IdxT(j), K2[c], kb);
    Li[q] = I[c];
}

template <typename IdxT>
__global__ void large_copy_back_kernel(const IdxT* __restrict__ hs, const IdxT* __restrict__ loff, u64 n_groups, u64 UL,
                                       const typename CompKey<IdxT>::type* __restrict__ Lk, const IdxT* __restrict__ Li, int kb,
                                       IdxT* __restrict__ K2, IdxT* __restrict__ I) {
    const u64 q = u64(blockIdx.x) * blockDim.x + threadIdx.x;
    if (q >= UL) return;
    const u64 j = last_le(loff, n_groups, q);  // the large group that owns slot q (last index of the plateau)
    const u64 c = u64(hs[j]) + (q - u64(loff[j]));
    K2[c] = CompKey<IdxT>::key2(Lk[q], kb);
    I[c] = Li[q];
}

// secondary key of a suffix that starts a run of >= p0 equal symbols x: with r = run length left and c = the symbol after
// the run, suffixes order by ascending r when c < x and by descending r, after all of those, when c > x.
template <typename IdxT>
__global__ void run_key_kernel(const u8* __restrict__ text, const uint16_t* __restrict__ code, const IdxT* __restrict__ RC,
                               const IdxT* __restrict__ RE, u64 NR, const IdxT* __restrict__ GS, const IdxT* __restrict__ IS, u64 US, u64 n, int kb0, u64* __restrict__ K,
                               IdxT* __restrict__ Gx) {
    const u64 c = u64(blockIdx.x) * blockDim.x + threadIdx.x;
    if (c >= US) return;
    const u64 i = IS[c], e = RE[last_le(RC, NR, c)], r = e - i;   // the long run that holds i: RC = first list index of every run
    const u32 x = code[text[i]];
    const u32 cs = e < n ? code[text[e]] : 0u;
    const u64 flag = cs > x ? 1 : 0;
    const u64 val = flag ? (n - r) : r;
    K[c] = (u64(x) << (kb0 + 1)) | (flag << kb0) | val;
    Gx[x] = GS[c];  // every member of the pure-x group carries the same head index
}

// Optional observer of the initial sort: the keys of all suffixes (first p0 symbols, b bits each, codes by h_code[byte])
// in sorted order — every table that depends only on a bounded prefix of the suffixes (the k-mer lookup tables of the
// probe search) is a by-product of this array and needs no gather through the finished suffix array.
// Sharded build: d_keys holds this member's n_local keys, which are positions [base, base + n_local) of the n_total sorted
// keys; ranges are cut where the first >= 4 symbols change (or the first symbol, for alphabets over 16 symbols), so a
// bucket of 4 or more symbols never spans two members. Every member calls the hook at the same point (collectives allowed).
// Tables the hook may have built from the sorted keys (device pointers of the build's index type): the deep table (start
// of every ACGT `depth`-mer's bucket, closed by one more entry) and the 8-mer LUT, plus the nibble maps dense code -> digit.
struct SaLookupTables {
    const void* deep = nullptr;
    int depth = 0;
    const void* lut_lo = nullptr;
    const void* lut_hi = nullptr;
    u64 m4 = 0, m5 = 0;
};
struct SaKeyHook {
    virtual void on_sorted_keys(const u64* d_keys, u64 n_local, u64 base, u64 n_total, int b, int p0, const uint16_t* h_code,
                                cudaStream_t stream, SaGroup* grp) = 0;
    virtual bool lookup_tables(SaLookupTables&) { return false; }
    // Single-device build that looked ranks up in the sorted keys: the buffer still holds all n keys in suffix-array
    // order when the build ends. The hook may take it (move from `keys`); what it leaves is released.
    virtual void adopt_sorted_keys(DevBuf<u64>& keys) { (void)keys; }
    virtual ~SaKeyHook() = default;
};

template <typename IdxT>
void build_suffix_array(const u8* d_text, u64 n, IdxT* d_sa, const RankView<IdxT> d_rank, cudaStream_t stream, SaStats* st,
                        SaKeyHook* hook = nullptr, SaGroup* grp = nullptr) {
    using KeyT = typename CompKey<IdxT>::type;
    using Acc = FlagAcc<IdxT>;
    if (n == 0) return;
    const int world = grp ? grp->world : 1;
    if (world == 1) grp = nullptr;
    auto sync_read = [&](void* dst, const void* src, size_t bytes) {
        const double t0 = host_now_ms();
        CUDA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, stream));
        CUDA_CHECK(cudaStreamSynchronize(stream));
        g_host_stalls.sync_ms += host_now_ms() - t0;
        g_host_stalls.syncs++;
    };

    // developer aid: ASGART_B200_DEBUG_PHASES=1 prints the wall time of every phase (synchronises the stream at each mark)
    static const bool dbg_phases = getenv("ASGART_B200_DEBUG_PHASES") != nullptr;
    double dbg_t = host_now_ms();
    auto phase = [&](const char* name, u64 count = 0) {
        if (!dbg_phases) return;
        cudaStreamSynchronize(stream);
        const double t = host_now_ms();
        fprintf(stderr, "[sa_build r%d/%d] %-22s %9.3f ms  (%llu)\n", grp ? grp->rank : 0, world, name, t - dbg_t, (unsigned long long)count);
        dbg_t = t;
    };

    NvtxRange nv_all("sa_build");
    NvtxPhases nv;
    // ---- 0. alphabet
    nv.next("sa_build/alphabet+ranges");
    DevBuf<unsigned long long> d_hist(256, stream);
    d_hist.zero();
    {
        int blocks = int(std::min<u64>(ceil_div(n, 256 * 16), u64(kNumSMs) * 8));
        byte_hist_kernel<<<blocks, 256, 0, stream>>>(d_text, n, d_hist.p);
        KERNEL_CHECK();
        count_launch();
    }
    unsigned long long h_hist[256];
    sync_read(h_hist, d_hist.p, sizeof h_hist);
    uint16_t h_code[256];
    int sigma = 0;
    for (int c = 0; c < 256; ++c) h_code[c] = h_hist[c] ? uint16_t(++sigma) : uint16_t(0);
    const int b = std::max(1, bit_width_u64(u64(sigma)));  // codes 0..sigma
    // symbols per initial key: enough that random texts are almost fully resolved by the first sort (p0 * entropy >=
    // log2(n) + 6 bits, i.e. ~n/64 chance collisions), rounded up to whole radix passes, at most what 64 bits hold.
    // 57 Mbp of DNA: 16 symbols = 6 passes instead of 21 symbols = 8 passes; 3.1 Gbp: 18 symbols = 7 passes.
    double entropy = 0;
    for (int c = 0; c < 256; ++c)
        if (h_hist[c]) { const double pr = double(h_hist[c]) / double(n); entropy -= pr * std::log2(pr); }
    const int p0_cap = 64 / b;
    int p0 = int(std::ceil((std::log2(double(n)) + 6.0) / std::max(entropy, 0.25)));
    p0 = std::min(p0_cap, std::max(p0, 1));
    p0 = std::min(p0_cap, (ceil_div_i(i64(b) * p0, 8) * 8) / b);
    // That rule prices an LSD sort, where every 8 key bits are a pass over all pairs. The MSD sort moves a pair once per level
    // only while its bucket is still large, so longer keys cost it next to nothing — and every chance collision they remove is
    // a suffix the doubling rounds never see (3.1 Gbp of DNA: 18 symbols leave 4.4 % of the suffixes with a random twin, 21
    // leave 0.07 %). So: as many symbols as 63 bits hold (all-ones stays free for padding keys).
    if (msd_sort_applicable(b, p0, n)) p0 = std::max(p0, std::min(63 / b, 32));
    DevBuf<uint16_t> d_code(256, stream);
    CUDA_CHECK(cudaMemcpyAsync(d_code.p, h_code, sizeof h_code, cudaMemcpyHostToDevice, stream));
    u64 rep_unit = 0;  // sum of 2^(b*j): a key whose p0 symbols are all equal to c is c * rep_unit
    for (int j = 0; j < p0; ++j) rep_unit |= u64(1) << (b * j);
    const u64 sym_mask = (u64(1) << b) - 1;

    // work list of the suffixes that are not yet unique: group head index, suffix, depth already compared, and the
    // start of every group inside the list (groups are contiguous)
    DevBuf<IdxT> Gw, Iw, Dw, HSw;
    u64 U = 0, NG = 0;

    // ---- 1. initial keys + sort, 2. heads -> rank, SA, work lists (ordinary groups A / single-symbol-run groups S)
    DevBuf<IdxT> GS, IS;
    u64 UA = 0, US = 0, NGA = 0;
    DevBuf<IdxT> GA, IA, HSA;
    // sharded build: this member's key range (prefixes [pre_lo, pre_hi) of `psym` symbols), the global index `base` of its
    // first suffix in the suffix array and the number n_loc of its suffixes; off[] = the pieces of all members
    u64 base = 0, n_loc = n;
    std::vector<u64> piece_off(world + 1, 0);
    piece_off[world] = n;
    int pshift = 0;
    u32 pre_lo = 0, pre_hi = 0;
    // the initial sort runs MSD-first (msd_sort.cuh) for small alphabets and large texts, else as the stable LSD sort
    bool use_msd = msd_sort_applicable(b, p0, n);
    DevBuf<IdxT> msd_table0;   // sharded build: histogram of the level-0 digit of the WHOLE text (the range cuts come from it)
    if (grp) {
        const int psym = std::max(1, std::min(p0, std::min(4, 12 / b)));
        const u32 nb = 1u << (b * psym);
        pshift = b * p0 - b * psym;
        if (b * psym != kMsdDigitBits) use_msd = false;   // the members' ranges must be ranges of level-0 bins
        std::vector<unsigned long long> h_ph(nb);
        if (use_msd) {
            // every member counts the level-0 bins of 1/world of the text; the sums go round as host values
            msd_table0.alloc(kMsdBins, stream);
            msd_table0.zero();
            const u64 tiles = ceil_div(n, u64(kH0Tile));
            const u64 t0 = tiles * u64(grp->rank) / u64(world), t1 = tiles * u64(grp->rank + 1) / u64(world);
            if (t1 > t0) {
                const int blocks = int(std::min<u64>(t1 - t0, u64(kNumSMs) * 2));
                msd_hist_text_kernel<IdxT><<<blocks, kMsdThreads, 0, stream>>>(d_text, n, d_code.p, b, psym, msd_table0.p, t0, t1);
                KERNEL_CHECK();
                count_launch();
            }
            std::vector<IdxT> h_t(nb);
            sync_read(h_t.data(), msd_table0.p, nb * sizeof(IdxT));
            std::vector<u64> sums(nb);
            for (u32 i = 0; i < nb; ++i) sums[i] = u64(h_t[i]);
            grp->allreduce_sum_host(sums.data(), int(nb));
            for (u32 i = 0; i < nb; ++i) { h_ph[i] = (unsigned long long)sums[i]; h_t[i] = IdxT(sums[i]); }
            CUDA_CHECK(cudaMemcpyAsync(msd_table0.p, h_t.data(), nb * sizeof(IdxT), cudaMemcpyHostToDevice, stream));
            CUDA_CHECK(cudaStreamSynchronize(stream));   // h_t leaves scope
        } else {
            DevBuf<unsigned long long> d_ph(nb, stream);
            d_ph.zero();
            const int blocks = int(std::min<u64>(ceil_div(n, 256), u64(kNumSMs) * 8));
            key_prefix_hist_kernel<<<blocks, 256, nb * sizeof(u32), stream>>>(d_text, n, d_code.p, b, psym, d_ph.p);
            KERNEL_CHECK();
            count_launch();
            sync_read(h_ph.data(), d_ph.p, nb * sizeof(unsigned long long));
        }
        // member r starts at the first bin whose preceding bins hold >= r * n / world suffixes (same cut on every member)
        std::vector<u32> cut(world + 1, nb);
        cut[0] = 0;
        u64 cum = 0;
        int r = 1;
        for (u32 bin = 0; bin < nb && r < world; ++bin) {
            while (r < world && cum >= (n / u64(world)) * u64(r) && cum > piece_off[r - 1]) { cut[r] = bin; piece_off[r] = cum; ++r; }
            cum += h_ph[bin];
        }
        for (; r < world; ++r) { cut[r] = nb; piece_off[r] = n; }
        pre_lo = cut[grp->rank]; pre_hi = cut[grp->rank + 1];
        base = piece_off[grp->rank];
        n_loc = piece_off[grp->rank + 1] - base;
    }
    IdxT* const sa_loc = d_sa + base;
    phase("alphabet+ranges", n_loc);
    nv.next("sa_build/init keys");

    // the sorted initial keys outlive the first phase when ranks are looked up lazily (single-device build with lookup tables)
    DevBuf<u64> keysA, keysB;
    RankLookup<IdxT> rl;
    bool lazy = false;
    {
        std::vector<int> shifts;
        for (int s = 0; s < b * p0; s += 8) shifts.push_back(s);
        // the sorted suffix indices must end up in d_sa itself: with an even number of passes they start there
        // (sharded: the piece d_sa + base is not 16-byte aligned, the sort runs in its own buffers and is copied over)
        keysA.alloc(n_loc + 4, stream); keysB.alloc(n_loc + 4, stream);   // + 4: reused as pair buffers by the inverse scatter
        DevBuf<IdxT> valsT(n_loc, stream), valsU(grp ? n_loc : 0, stream);
        u64 *k = keysA.p, *ka = keysB.p;
        IdxT *v, *va;
        bool sorted = false;
        if (use_msd) {
            // MSD-first: keys are built inside the first partition pass; the result lands in (keysA, d_sa / valsT)
            v = grp ? valsT.p : d_sa; va = grp ? valsU.p : valsT.p;
            if (st && st->sort) st->sort->begin();
            sorted = msd_sort_suffixes<IdxT>(d_text, n, d_code.p, b, p0, grp ? pre_lo : 0u, grp ? pre_hi : u32(kMsdBins), n_loc, k, v, ka, va,
                                             grp ? msd_table0.p : nullptr, stream, st ? &st->msd : nullptr);
            if (st && st->sort) st->sort->end(0, 0);
            if (st) st->used_msd = sorted;
            phase(sorted ? "initial sort (msd)" : "initial sort (msd declined)", n_loc);
        }
        if (!sorted) {
        if (!grp) {
            v = (shifts.size() % 2 == 0) ? d_sa : valsT.p; va = (shifts.size() % 2 == 0) ? valsT.p : d_sa;
            init_keys_kernel<IdxT><<<unsigned(ceil_div(n, u64(kInitTile))), kInitThreads, 0, stream>>>(d_text, n, d_code.p, b, p0, k, v);
            KERNEL_CHECK();
            count_launch();
        } else {
            v = valsT.p; va = valsU.p;
            const u64 tiles = ceil_div(n, u64(kInitTile));
            DevBuf<u64> tcnt(tiles, stream), toff(tiles, stream);
            init_keys_range_kernel<IdxT, false><<<unsigned(tiles), kInitThreads, 0, stream>>>(d_text, n, d_code.p, b, p0, pshift, pre_lo, pre_hi,
                                                                                             tcnt.p, nullptr, nullptr, nullptr);
            KERNEL_CHECK();
            const u64* tc = tcnt.p;
            u64* to = toff.p;
            device_scan<u64, SumOp>([tc] __device__(u64 i) { return tc[i]; }, [to] __device__(u64 i, u64 exc, u64) { to[i] = exc; }, tiles,
                                    (u64*)nullptr, stream);
            init_keys_range_kernel<IdxT, true><<<unsigned(tiles), kInitThreads, 0, stream>>>(d_text, n, d_code.p, b, p0, pshift, pre_lo, pre_hi,
                                                                                            nullptr, toff.p, k, v);
            KERNEL_CHECK();
            count_launch(2);
        }
        phase("init keys", n_loc);
        nv.next("sa_build/initial sort");
        radix_sort_pairs<u64, IdxT>(k, ka, v, va, n_loc, shifts.data(), int(shifts.size()), stream, st ? st->sort : nullptr,
                                    st ? st->scatter_main : nullptr);
        phase("initial sort", shifts.size());
        }
        nv.next("sa_build/lookup tables");
        if (grp && n_loc) CUDA_CHECK(cudaMemcpyAsync(sa_loc, v, n_loc * sizeof(IdxT), cudaMemcpyDeviceToDevice, stream));

        if (hook) hook->on_sorted_keys(k, n_loc, base, n, b, p0, h_code, stream, grp);
        phase("lookup tables");
        {
            SaLookupTables lt;
            // (every member of a group takes the same decision: it depends on n, the alphabet and the key length only)
            if (hook && hook->lookup_tables(lt) && lt.depth > 0 && p0 >= 8 && (!grp || b * std::min(p0, 4) >= 8)) {
                lazy = true;
                rl.world = u32(world);
                if (grp) {
                    // the members read each other's sorted keys through peer pointers (k is the start of its block)
                    void* all[kMaxWorld] = {};
                    CUDA_CHECK(cudaStreamSynchronize(stream));
                    grp->exchange_ptr(k, (n_loc + 4) * sizeof(u64), all);
                    for (int r = 0; r < world; ++r) { rl.keys[r] = static_cast<const u64*>(all[r]); rl.piece[r] = piece_off[r]; }
                    rl.piece[world] = piece_off[world];
                } else {
                    rl.keys[0] = k; rl.piece[0] = 0; rl.piece[1] = n;
                }
                rl.text = d_text; rl.code = d_code.p; rl.n = n; rl.b = b; rl.p0 = p0; rl.depth = lt.depth;
                rl.deep = static_cast<const IdxT*>(lt.deep);
                rl.lut_lo = static_cast<const IdxT*>(lt.lut_lo); rl.lut_hi = static_cast<const IdxT*>(lt.lut_hi);
                rl.m4 = lt.m4; rl.m5 = lt.m5;
            }
        }
        nv.next("sa_build/heads+rank scatter");
        const u64* kk = k;
        const IdxT* vv = sa_loc;
        if (st && st->rank) st->rank->begin();
        const u64 hp_tiles = ceil_div(n_loc, u64(kHpTile));
        DevBuf<HpTileAcc> hp_acc(hp_tiles, stream), hp_pre(hp_tiles, stream), hp_total(1, stream);
        HpTileAcc tot(0);
        if (n_loc) {
            hp_reduce_kernel<<<unsigned(hp_tiles), kHpThreads, 0, stream>>>(kk, n_loc, rep_unit, sym_mask, hp_acc.p);
            KERNEL_CHECK();
            count_launch();
            const HpTileAcc* acc = hp_acc.p;
            HpTileAcc* pre = hp_pre.p;
            device_scan<HpTileAcc, HpTileOp>([acc] __device__(u64 i) -> HpTileAcc { return acc[i]; },
                                             [pre] __device__(u64 i, const HpTileAcc& exc, const HpTileAcc&) { pre[i] = exc; }, hp_tiles,
                                             hp_total.p, stream);
            sync_read(&tot, hp_total.p, sizeof tot);
        }
        UA = tot.c; US = tot.d; NGA = tot.e;
        GA.alloc(UA, stream); IA.alloc(UA, stream); HSA.alloc(NGA, stream);
        GS.alloc(US, stream); IS.alloc(US, stream);
        // rank by sorted position goes to the dead half of the value ping-pong, then to text order by the sliced scatter
        IdxT* rpos = lazy ? nullptr : va;
        if (n_loc) {
            hp_emit_kernel<IdxT><<<unsigned(hp_tiles), kHpThreads, 0, stream>>>(kk, vv, n_loc, rep_unit, sym_mask, hp_pre.p, IdxT(base), rpos,
                                                                                GA.p, IA.p, HSA.p, GS.p, IS.p);
            KERNEL_CHECK();
            count_launch();
        }
        if (sorted && US > 1) {
            // The MSD sort leaves equal keys in arbitrary order, but the run round reads the suffixes of every pure key in
            // text order (a stretch of consecutive positions = one run): order the short list by (symbol, position).
            DevBuf<u64> PK(US, stream), PK2(US, stream);
            DevBuf<IdxT> GT(US, stream);
            {
                const IdxT* isp = IS.p;
                const uint16_t* cd = d_code.p;
                u64* pk = PK.p;
                for_each_index(US, [=] __device__(u64 c) { const u64 i = u64(isp[c]); pk[c] = (u64(cd[d_text[i]]) << 58) | i; }, stream);
            }
            std::vector<int> sh;
            for (int s = 0; s < bit_width_u64(n); s += 8) sh.push_back(s);
            for (int s = 0; s < b; s += 8) sh.push_back(58 + s);
            u64 *k1 = PK.p, *k2 = PK2.p;
            IdxT *g1 = GS.p, *g2 = GT.p;
            radix_sort_pairs<u64, IdxT>(k1, k2, g1, g2, US, sh.data(), int(sh.size()), stream, st ? st->sort : nullptr, st ? st->scatter : nullptr);
            {
                IdxT *gsp = GS.p, *isp = IS.p;
                const u64* kk1 = k1;
                const IdxT* gg1 = g1;
                for_each_index(US, [=] __device__(u64 c) {
                    const IdxT g = gg1[c];
                    isp[c] = IdxT(kk1[c] & ((u64(1) << 58) - 1));
                    gsp[c] = g;
                }, stream);
            }
        }
        // the sorted keys are dead from here on: both key buffers serve as scratch of the sort-back scatter
        if (lazy) {   // all-ones: "the initial head"
            if (!grp) CUDA_CHECK(cudaMemsetAsync(d_rank.base[0], 0xFF, n * sizeof(IdxT), stream));
            else {
                CUDA_CHECK(cudaMemsetAsync(d_rank.base[grp->rank], 0xFF, d_rank.slice_len() * sizeof(IdxT), stream));
                CUDA_CHECK(cudaStreamSynchronize(stream));
                grp->barrier();   // nobody stores a refined rank into a slice that is still being cleared
            }
        }
        else if (!grp) inverse_scatter<IdxT>(d_sa, rpos, n, d_rank.base[0], n, stream, k, ka);
        else if (n_loc) {   // group build without a deep table (texts under 256 symbols): plain stores through the view
            const unsigned grid = unsigned(std::min<u64>(ceil_div(n_loc, 256), u64(kNumSMs) * 16));
            scatter_view_kernel<IdxT><<<grid, 256, 0, stream>>>(sa_loc, rpos, n_loc, d_rank);
            KERNEL_CHECK();
            count_launch();
        }
        if (st && st->rank) st->rank->end(4, 0);
        phase("heads+rank scatter", UA + US);
        // the unsorted half of the key ping-pong goes now; the sorted keys stay while ranks are looked up in them
        if (k == keysA.p) keysB.release(); else keysA.release();
        if (!lazy) { keysA.release(); keysB.release(); }
    }
    nv.next("sa_build/run round");

    // ---- 3. run round: suffixes starting a run of >= p0 equal symbols are ordered by (symbol after the run, run length)
    // in one sort and then continue at depth = run length, instead of needing log2(run length) doubling rounds
    DevBuf<IdxT> GS2, IS2, DS2, HSS2;
    u64 US2 = 0, NGS2 = 0;
    if (US > 0) {
        if (st) st->rounds++;
        // the runs of >= p0 equal symbols, read off the list itself: the suffixes of one pure key come out of the stable
        // sort in text order, and the positions i with T[i .. i+p0) all equal to x inside one run [a, e) are exactly
        // a .. e - p0, so a stretch of consecutive positions in the list is one run and its last position + p0 is the run's
        // end. One flag scan over the US list entries (a scan of all n text positions for run starts and ends cost 35 ms at
        // 3.1 Gbp). RC[r] = list index where run r starts, RE[r] = end of that run in the text.
        DevBuf<IdxT> RC, RE;
        u64 NR = 0;
        {
            const IdxT *gsp = GS.p, *isp = IS.p;
            const u64 USc = US;
            const IdxT p0i = IdxT(p0);
            auto rin = [gsp, isp, USc] __device__(u64 c) -> u32 {
                const IdxT g = gsp[c], i = isp[c];
                const bool first = c == 0 || gsp[c - 1] != g || isp[c - 1] + IdxT(1) != i;
                const bool last = c + 1 == USc || gsp[c + 1] != g || isp[c + 1] != i + IdxT(1);
                return (first ? FS_CNT_C : 0u) | (last ? FS_CNT_D : 0u);
            };
            DevBuf<Acc> d_rt(1, stream);
            FlagScanPlan<IdxT> rplan;
            rplan.prepare(rin, US, d_rt.p, stream);
            Acc rt;
            sync_read(&rt, d_rt.p, sizeof rt);
            NR = u64(rt.c);
            RC.alloc(NR, stream); RE.alloc(NR, stream);
            IdxT *rc = RC.p, *re = RE.p;
            rplan.finish(rin, [rc, re, isp, p0i] __device__(u64 c, const Acc& exc, const Acc& inc) {
                if (inc.c != exc.c) rc[exc.c] = IdxT(c);
                if (inc.d != exc.d) re[exc.d] = isp[c] + p0i;
            });
        }
        const int kb0 = std::max(1, bit_width_u64(n));
        DevBuf<u64> KA(US, stream), KB(US, stream);
        DevBuf<IdxT> IB(US, stream), Gx(sigma + 2, stream);
        run_key_kernel<IdxT><<<unsigned(ceil_div(US, 256)), 256, 0, stream>>>(d_text, d_code.p, RC.p, RE.p, NR, GS.p, IS.p, US, n, kb0, KA.p, Gx.p);
        KERNEL_CHECK();
        count_launch();
        std::vector<int> shifts;
        for (int s = 0; s < kb0 + 1 + bit_width_u64(u64(sigma)); s += 8) shifts.push_back(s);
        u64 *k = KA.p, *ka = KB.p;
        IdxT *v = IS.p, *va = IB.p;
        radix_sort_pairs<u64, IdxT>(k, ka, v, va, US, shifts.data(), int(shifts.size()), stream, st ? st->sort : nullptr,
                                    st ? st->scatter : nullptr);
        DevBuf<Acc> d_total(1, stream);
        const u64* kk = k;
        const IdxT* vv = v;
        const u64 USc = US;
        auto in = [kk, USc, kb0] __device__(u64 c) {
            const u64 cur = kk[c];
            bool head_old = true, head_new = true, tail_new = true;
            if (c > 0) { const u64 prev = kk[c - 1]; head_new = prev != cur; head_old = (prev >> (kb0 + 1)) != (cur >> (kb0 + 1)); }
            if (c + 1 < USc) tail_new = kk[c + 1] != cur;
            const bool surv = !(head_new && tail_new);
            return (head_old ? FS_MARK_A : 0u) | (head_new ? FS_MARK_B : 0u) | (surv ? FS_CNT_C : 0u) | ((surv && head_new) ? FS_CNT_D : 0u);
        };
        if (st && st->rank) st->rank->begin();
        FlagScanPlan<IdxT> plan;
        plan.prepare(in, US, d_total.p, stream);
        Acc tot;
        sync_read(&tot, d_total.p, sizeof tot);
        US2 = u64(tot.c); NGS2 = u64(tot.d);
        GS2.alloc(US2, stream); IS2.alloc(US2, stream); DS2.alloc(US2, stream); HSS2.alloc(NGS2, stream);
        IdxT *g2 = GS2.p, *i2 = IS2.p, *d2 = DS2.p, *hs2 = HSS2.p;
        const IdxT* gx = Gx.p;
        plan.finish(in, [=] __device__(u64 c, const Acc& exc, const Acc& inc) {
            const u64 cur = kk[c];
            const bool head_new = c == 0 || kk[c - 1] != cur;
            const bool tail_new = c + 1 == USc || kk[c + 1] != cur;
            const IdxT g = gx[cur >> (kb0 + 1)];
            const IdxT idx = vv[c];
            const IdxT ng = g + (inc.b - inc.a);
            *d_rank.ptr(u64(idx)) = ng;
            if (head_new && tail_new) { d_sa[u64(g) + (c - u64(inc.a))] = idx; return; }
            const u64 val = cur & ((u64(1) << kb0) - 1);
            const u64 r = ((cur >> kb0) & 1) ? (n - val) : val;
            g2[exc.c] = ng; i2[exc.c] = idx; d2[exc.c] = IdxT(r);
            if (head_new) hs2[exc.d] = exc.c;
        });
        if (st && st->rank) st->rank->end(3, 0);
    }
    GS.release(); IS.release();
    phase("run round", US);
    nv.next("sa_build/doubling rounds");

    // ---- 4. merged work list: ordinary groups at depth p0, then the run groups at depth = run length
    U = UA + US2; NG = NGA + NGS2;
    if (U > 0) {
        Gw.alloc(U, stream); Iw.alloc(U, stream); Dw.alloc(U, stream); HSw.alloc(NG, stream);
        IdxT *gw = Gw.p, *iw = Iw.p, *dw = Dw.p, *hw = HSw.p;
        const IdxT *ga = GA.p, *ia = IA.p, *hsa = HSA.p, *g2 = GS2.p, *i2 = IS2.p, *d2 = DS2.p, *hs2 = HSS2.p;
        const u64 UAc = UA, NGAc = NGA, NGc = NG;
        const IdxT p0i = IdxT(p0);
        for_each_index(U, [=] __device__(u64 c) {
            if (c < UAc) { gw[c] = ga[c]; iw[c] = ia[c]; dw[c] = p0i; }
            else { gw[c] = g2[c - UAc]; iw[c] = i2[c - UAc]; dw[c] = d2[c - UAc]; }
            if (c < NGc) hw[c] = c < NGAc ? hsa[c] : IdxT(u64(hs2[c - NGAc]) + UAc);
        }, stream);
    }
    GA.release(); IA.release(); HSA.release(); GS2.release(); IS2.release(); DS2.release(); HSS2.release();

    // ---- 5. doubling rounds: every suffix of the list looks D symbols ahead, where D >= H symbols are already known
    // to be equal inside its group and rank[] orders all suffixes by at least their first H symbols
    const int kb = std::max(1, bit_width_u64(n));  // key2 in [0, n]
    u64 H = u64(p0);
    // Sharded build: a collective at the top of every round (all re-rankings of the previous round have landed in the
    // owners' memory before anyone gathers; its sum also tells when every member's list is empty) and one before the
    // re-ranking (everyone has finished gathering before any rank changes). Members with an empty list only take part in these.
    auto group_sync = [&](u64 v) -> u64 {
        CUDA_CHECK(cudaStreamSynchronize(stream));
        grp->allreduce_sum_host(&v, 1);
        return v;
    };
    while (true) {
        if (grp ? group_sync(U) == 0 : U == 0) break;
        if (st) st->rounds++;
        if (U == 0) { group_sync(0); H <<= 1; continue; }
        DevBuf<IdxT> K2(U, stream), large_sz(NG, stream), loff(NG + 1, stream);
        {
            if (st && st->gather) st->gather->begin();
            int blocks = int(std::min<u64>(ceil_div(U, 256), u64(kNumSMs) * 16));
            if (lazy) gather_rank_kernel<IdxT, true><<<blocks, 256, 0, stream>>>(Iw.p, Dw.p, d_rank, U, n, K2.p, rl);
            else gather_rank_kernel<IdxT, false><<<blocks, 256, 0, stream>>>(Iw.p, Dw.p, d_rank, U, n, K2.p, rl);
            KERNEL_CHECK();
            count_launch();
            if (st && st->gather) st->gather->end(1, U * 3 * sizeof(IdxT));
        }
        if (st && st->rank) st->rank->begin();
        small_group_sort_kernel<IdxT><<<unsigned(ceil_div(NG, 128)), 128, 0, stream>>>(HSw.p, NG, U, K2.p, Iw.p, large_sz.p);
        KERNEL_CHECK();
        count_launch();
        u64 UL = 0;
        {
            const IdxT* lz = large_sz.p;
            IdxT* lo = loff.p;
            device_scan<IdxT, SumOp>([lz] __device__(u64 j) { return lz[j]; }, [lo] __device__(u64 j, IdxT exc, IdxT) { lo[j] = exc; }, NG,
                                     loff.p + NG, stream);
            IdxT h_ul = 0;
            sync_read(&h_ul, loff.p + NG, sizeof h_ul);
            UL = u64(h_ul);
        }
        if (st && st->rank) st->rank->end(4, 0);
        if (UL > 0) {
            DevBuf<KeyT> LA(UL, stream), LB(UL, stream);
            DevBuf<IdxT> LIA(UL, stream), LIB(UL, stream);
            large_copy_out_kernel<IdxT><<<unsigned(ceil_div(UL, 256)), 256, 0, stream>>>(HSw.p, loff.p, NG, UL, K2.p, Iw.p, kb, LA.p, LIA.p);
            KERNEL_CHECK();
            const int jb = std::max(1, bit_width_u64(NG - 1));  // group ordinal in [0, NG)
            std::vector<int> shifts;
            if (sizeof(IdxT) == 4) {
                for (int s = 0; s < kb + jb; s += 8) shifts.push_back(s);
            } else {
                for (int s = 0; s < kb; s += 8) shifts.push_back(s);
                for (int s = 0; s < jb; s += 8) shifts.push_back(64 + s);
            }
            KeyT *k = LA.p, *ka = LB.p;
            IdxT *v = LIA.p, *va = LIB.p;
            radix_sort_pairs<KeyT, IdxT>(k, ka, v, va, UL, shifts.data(), int(shifts.size()), stream, st ? st->sort : nullptr,
                                         st ? st->scatter : nullptr);
            large_copy_back_kernel<IdxT><<<unsigned(ceil_div(UL, 256)), 256, 0, stream>>>(HSw.p, loff.p, NG, UL, k, v, kb, K2.p, Iw.p);
            KERNEL_CHECK();
            count_launch(2);
        }

        DevBuf<Acc> d_total(1, stream);
        const IdxT *gg = Gw.p, *k2 = K2.p, *ii = Iw.p, *dd = Dw.p;
        const u64 Uc = U;
        auto in = [gg, k2, Uc] __device__(u64 c) {
            const IdxT g = gg[c], kv = k2[c];
            bool head_old = true, head_new = true, tail_new = true;
            if (c > 0) { head_old = gg[c - 1] != g; head_new = head_old || k2[c - 1] != kv; }
            if (c + 1 < Uc) tail_new = gg[c + 1] != g || k2[c + 1] != kv;
            const bool surv = !(head_new && tail_new);
            return (head_old ? FS_MARK_A : 0u) | (head_new ? FS_MARK_B : 0u) | (surv ? FS_CNT_C : 0u) | ((surv && head_new) ? FS_CNT_D : 0u);
        };
        if (st && st->rank) st->rank->begin();
        FlagScanPlan<IdxT> plan;
        plan.prepare(in, U, d_total.p, stream);
        Acc tot;
        sync_read(&tot, d_total.p, sizeof tot);
        const u64 U2 = u64(tot.c), NG2 = u64(tot.d);
        if (grp) group_sync(0);
        DevBuf<IdxT> G2(U2, stream), I2(U2, stream), D2(U2, stream), HS2(NG2, stream);
        IdxT *g2 = G2.p, *i2 = I2.p, *d2 = D2.p, *hs2 = HS2.p;
        const IdxT Hi = IdxT(H);
        plan.finish(in, [=] __device__(u64 c, const Acc& exc, const Acc& inc) {
            const IdxT g = gg[c], kv = k2[c];
            const bool head_new = c == 0 || gg[c - 1] != g || k2[c - 1] != kv;
            const bool tail_new = c + 1 == Uc || gg[c + 1] != g || k2[c + 1] != kv;
            const IdxT idx = ii[c];
            const IdxT ng = g + (inc.b - inc.a);
            // rank[] already holds g for every member of the old group: only suffixes that leave its first subgroup need the
            // (random, 4-byte, possibly remote) store
            if (ng != g) *d_rank.ptr(u64(idx)) = ng;
            if (head_new && tail_new) { d_sa[u64(g) + (c - u64(inc.a))] = idx; return; }
            g2[exc.c] = ng; i2[exc.c] = idx; d2[exc.c] = dd[c] + Hi;
            if (head_new) hs2[exc.d] = exc.c;
        });
        if (st && st->rank) st->rank->end(3, 0);
        Gw = std::move(G2); Iw = std::move(I2); Dw = std::move(D2); HSw = std::move(HS2);
        U = U2; NG = NG2;
        H <<= 1;
    }
    if (grp && lazy) { CUDA_CHECK(cudaStreamSynchronize(stream)); grp->barrier(); }   // the peers are done reading these keys
    // The lazy path never writes the sorted keys after the initial sort, and only one of the two buffers is left (the
    // other went after the rank scatter). The doubling rounds only reorder suffixes inside a group of equal keys, and such a
    // group is one contiguous range of the final suffix array, so keys[i] is still the key of SA[i].
    if (lazy && !grp && hook) hook->adopt_sorted_keys(keysA.p ? keysA : keysB);
    keysA.release(); keysB.release();
    phase("doubling rounds", st ? st->rounds : 0);
    nv.next("sa_build/share SA pieces");
    if (grp) grp->share_pieces(d_sa, piece_off.data(), int(sizeof(IdxT)), stream);
    phase("share SA pieces");
}

template <typename IdxT>
void build_suffix_array(const u8* d_text, u64 n, IdxT* d_sa, IdxT* d_rank, cudaStream_t stream, SaStats* st, SaKeyHook* hook = nullptr) {
    build_suffix_array<IdxT>(d_text, n, d_sa, RankView<IdxT>::single(d_rank), stream, st, hook, nullptr);
}

}  // namespace ab200
