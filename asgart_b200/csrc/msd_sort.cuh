// msd_sort.cuh — the initial sort of the suffix-array build as a most-significant-digit-first radix sort (sm_100a).
//
// Job: order the n suffixes of the text by their first p0 symbols (keys of KB = b * p0 <= 64 bits, b bits per symbol,
// most significant symbol first), producing the sorted keys and the suffix indices. Ties may come out in any order
// (the doubling rounds break them); the caller restores text order where it needs it (the run round's list).
//
// Why not the stable LSD sort of radix_sort.cuh: that one moves every (key, index) pair ceil(KB / 8) times (7 passes at
// 3.1 Gbp, 24 B per pair and pass plus a histogram re-read) and pays a stable in-warp ranking (8 ballots per key) in each.
// Here a pair is moved once per 12-bit level while its bucket is still large, with a one-atomic-per-element, non-stable
// ranking, and finished inside shared memory as soon as its bucket is small:
//
//   level l = 0, 1, ...   digit = bits [KB - 12 (l + 1), KB - 12 l) of the key (4 DNA symbols per level), 4096 bins
//     msd_hist          per-row bin counts                       level 0 reads the text (1 B per suffix), others the keys
//     msd_rowscan       bin counts -> child offsets (the row's cursor table); children larger than kLocSmall become the
//                       rows of level l + 1
//     msd_scatter       tile of 4096 pairs -> shared-memory partition by digit -> each digit run appended at its child's
//                       cursor (one global atomicAdd per non-empty bin and tile); level 0 builds the keys from the text
//     msd_local         children of at most kLocSmall pairs: a block loads a window of consecutive children (<= 6400
//                       pairs), sorts it by the remaining low bits with a stable LSD counting sort in shared memory
//                       (6-bit digits, private per-thread counters, no atomics) and writes the final order
//   A row = one bucket that is partitioned at this level. Rows are independent, so levels beyond the first few only
//   see what is still large there: repeats, low-complexity sequence, N-runs. After the last level a bucket holds equal
//   keys only and needs no further work.
//   Buffers: two (key, index) arrays A and B; level l reads one and writes the other, starting with text -> A; the
//   local sort always leaves its result in A (in place after even levels, B -> A after odd ones: that range of A was
//   consumed by the level's own scatter), so A holds the sorted arrays at the end.
//
// HBM traffic per suffix at 3.1 Gbp (levels 0-2 see everything, then buckets are ~184 pairs): 1 + (1 + 12) + 2 * (8 + 24)
// + 24 = 102 B, against 7 * 32 + 13 = 237 B for key generation + the LSD sort.
#pragma once
#include <algorithm>
#include <vector>

#include "common.cuh"
#include "scan.cuh"

namespace ab200 {

constexpr int kMsdDigitBits = 12;
constexpr int kMsdBins = 1 << kMsdDigitBits;
constexpr int kMsdThreads = 512;
constexpr int kMsdItems = 8;
constexpr int kMsdTile = kMsdThreads * kMsdItems;    // 4096 pairs per partition tile
constexpr int kMsdHalo = 64;                         // codes past a tile that its last keys reach into (p0 <= 32, + alignment)
constexpr int kLocThreads = 512;
constexpr int kLocItems = 13;                        // LSD passes: blocked items per thread; odd: their reads are bank-conflict free
constexpr int kLocCap = 6144;                        // pairs per local sort (12 per thread in the striped fast path)
constexpr int kLocSmall = 1536;                      // children up to this size are finished by the local sort
constexpr int kLocWindow = kLocCap - kLocSmall;      // children STARTING inside one window of this many positions form a batch
constexpr int kLocDigitBits = 5;
constexpr int kLocDigits = 1 << kLocDigitBits;
constexpr int kMsdMaxLevels = 6;

struct MsdLevels {
    int key_bits = 0, n = 0;
    int shift[kMsdMaxLevels] = {}, width[kMsdMaxLevels] = {};
    explicit MsdLevels(int kb) : key_bits(kb) {
        for (int top = kb; top > 0 && n < kMsdMaxLevels; top -= kMsdDigitBits) {
            width[n] = std::min(kMsdDigitBits, top);
            shift[n] = top - width[n];
            ++n;
        }
    }
};

__device__ __forceinline__ u32 msd_atomic_add(u32* p, u32 v) { return atomicAdd(p, v); }
__device__ __forceinline__ u64 msd_atomic_add(u64* p, u64 v) { return u64(atomicAdd(reinterpret_cast<unsigned long long*>(p), (unsigned long long)v)); }

// shared-memory histogram bump that returns the element's slot inside its bin; a warp whose lanes all hit one bin (runs of
// one symbol, giant buckets) takes one atomic instead of 32 serialised ones
__device__ __forceinline__ u32 msd_bin_slot(u32* cnt, u32 d, bool valid) {
    const u32 d0 = __shfl_sync(0xffffffffu, d, 0);
    if (__all_sync(0xffffffffu, valid && d == d0)) {
        u32 base = 0;
        if (lane_id() == 0) base = atomicAdd(&cnt[d0], 32u);
        return __shfl_sync(0xffffffffu, base, 0) + lane_id();
    }
    return valid ? atomicAdd(&cnt[d], 1u) : 0u;
}

// One descriptor per partition tile / local window, written by msd_expand_kernel from the rows' (start, size): a block
// finds its work with one load instead of a bisection over the row list (a dependent-load chain longer than the tile's
// own work). Tiles: (base, count) = the tile's pairs. Windows: base = first position, count = ordinal of the window in its row.
struct __align__(16) MsdDesc {
    u64 base;
    u32 count, row;
};

template <bool WINDOWS>
__global__ void __launch_bounds__(128) msd_expand_kernel(const u64* __restrict__ seg_start, const u64* __restrict__ seg_size,
                                                         const u32* __restrict__ first, MsdDesc* __restrict__ out) {
    constexpr u32 unit = WINDOWS ? kLocWindow : kMsdTile;
    const u32 r = blockIdx.x;
    const u64 s = seg_start[r], sz = seg_size[r];
    const u32 t0 = first[r], t1 = first[r + 1];
    for (u32 t = t0 + threadIdx.x; t < t1; t += 128) {
        const u64 off = u64(t - t0) * unit;
        MsdDesc d;
        d.base = s + off;
        d.count = WINDOWS ? (t - t0) : u32(min(u64(unit), sz - off));   // windows: the ordinal inside the row
        d.row = r;
        out[t] = d;
    }
}

// symbol codes of text[base, base + count) -> sc[0, count) (0 past the end of the text); 16 bytes per load where possible
__device__ __forceinline__ void msd_load_codes(const u8* __restrict__ text, u64 n, u64 base, u32 count, const u8* scode, u8* sc) {
    for (u32 c = threadIdx.x * 16; c < count; c += blockDim.x * 16) {
        const u64 p = base + c;
        if (p + 16 <= n && c + 16 <= count && ((reinterpret_cast<uintptr_t>(text) + p) & 15) == 0) {
            const uint4 v = *reinterpret_cast<const uint4*>(text + p);
            const u32 w[4] = {v.x, v.y, v.z, v.w};
            u32 o[4];
#pragma unroll
            for (int q = 0; q < 4; ++q)
                o[q] = u32(scode[w[q] & 255u]) | (u32(scode[(w[q] >> 8) & 255u]) << 8) | (u32(scode[(w[q] >> 16) & 255u]) << 16) |
                       (u32(scode[w[q] >> 24]) << 24);
            *reinterpret_cast<uint4*>(sc + c) = make_uint4(o[0], o[1], o[2], o[3]);
        } else {
            for (u32 j = c; j < c + 16 && j < count; ++j) sc[j] = (base + j < n) ? scode[text[base + j]] : u8(0);
        }
    }
}

// ---- level 0 histogram: bins of the first `msym` symbols (msym * b = width of level 0) of every suffix, from the text ----
constexpr int kH0Items = 16;
constexpr int kH0Tile = kMsdThreads * kH0Items;

// TMA (1-D bulk copy) + mbarrier helpers: one thread arms the barrier with the byte count and starts the copy; the bytes
// land in shared memory without passing through registers and every waiting thread is released when they are all there.
__device__ __forceinline__ void msd_mbar_init(u64* bar, u32 count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(u32(__cvta_generic_to_shared(bar))), "r"(count));
}
__device__ __forceinline__ void msd_bulk_load(void* smem_dst, const void* gmem_src, u32 bytes, u64* bar) {
    const u32 b = u32(__cvta_generic_to_shared(bar));
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(b), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     u32(__cvta_generic_to_shared(smem_dst))),
                 "l"(gmem_src), "r"(bytes), "r"(b)
                 : "memory");
}
__device__ __forceinline__ void msd_mbar_wait(u64* bar, u32 parity) {
    const u32 b = u32(__cvta_generic_to_shared(bar));
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "MSD_WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra MSD_DONE_%=;\n"
        "bra MSD_WAIT_%=;\n"
        "MSD_DONE_%=:\n"
        "}\n" ::"r"(b),
        "r"(parity)
        : "memory");
}

// Persistent blocks; the text tile of the NEXT iteration is fetched by a bulk copy (TMA) into the other half of a
// two-stage buffer while the current one is histogrammed, so the tile's DRAM latency is off the block's critical path.
template <typename OffT>
__global__ void __launch_bounds__(kMsdThreads) msd_hist_text_kernel(const u8* __restrict__ text, u64 n, const uint16_t* __restrict__ code, int b,
                                                                    int msym, OffT* __restrict__ table, u64 tile_begin, u64 tile_end) {
    // positions of the tiles [tile_begin, tile_end) are counted (a sharded build splits the text between the members);
    // the symbols a position looks ahead to are read wherever they lie
    constexpr u32 kNeed = kH0Tile + kMsdHalo;
    __shared__ u32 h[kMsdBins];
    __shared__ __align__(128) u8 raw[2][kNeed];
    __shared__ __align__(8) u64 bar[2];
    __shared__ u8 scode[256];
    for (u32 i = threadIdx.x; i < kMsdBins; i += kMsdThreads) h[i] = 0;
    if (threadIdx.x < 256) scode[threadIdx.x] = u8(code[threadIdx.x]);
    const bool aligned = (reinterpret_cast<uintptr_t>(text) & 15) == 0;
    if (threadIdx.x == 0) {
        msd_mbar_init(&bar[0], 1);
        msd_mbar_init(&bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const u32 wmask = (1u << (b * msym)) - 1u;
    const u64 tiles = min((n + kH0Tile - 1) / kH0Tile, tile_end);
    // bytes of tile t that the bulk copy brings (a multiple of 16 inside the text); the rest is filled by plain loads
    auto bulk_bytes = [&](u64 t) -> u32 {
        const u64 base = t * kH0Tile;
        const u64 avail = n - base;
        return aligned ? u32((avail < u64(kNeed) ? avail : u64(kNeed)) & ~u64(15)) : 0u;
    };
    if (threadIdx.x == 0 && tile_begin + blockIdx.x < tiles) {
        const u32 nb = bulk_bytes(tile_begin + blockIdx.x);
        if (nb) msd_bulk_load(raw[0], text + (tile_begin + blockIdx.x) * kH0Tile, nb, &bar[0]);
    }
    u32 it = 0;
    for (u64 tile = tile_begin + blockIdx.x; tile < tiles; tile += gridDim.x, ++it) {
        const u32 buf = it & 1u;
        const u64 base = tile * kH0Tile;
        const u64 next = tile + gridDim.x;
        if (threadIdx.x == 0 && next < tiles) {   // the other stage was released by the barrier that ended the last iteration
            const u32 nb = bulk_bytes(next);
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            if (nb) msd_bulk_load(raw[buf ^ 1u], text + next * kH0Tile, nb, &bar[buf ^ 1u]);
        }
        const u32 got = bulk_bytes(tile);
        for (u32 i = got + threadIdx.x; i < kNeed; i += kMsdThreads) raw[buf][i] = (base + i < n) ? text[base + i] : u8(0);
        if (got) msd_mbar_wait(&bar[buf], (it >> 1) & 1u);
        __syncthreads();
        const u8* rb = raw[buf];
        const u32 q0 = threadIdx.x * kH0Items;
        u32 w = 0;
        for (int j = 0; j < msym - 1; ++j) w = (w << b) | (base + q0 + j < n ? u32(scode[rb[q0 + j]]) : 0u);
#pragma unroll
        for (int j = 0; j < kH0Items; ++j) {
            const u32 pos = q0 + j + msym - 1;
            w = ((w << b) | (base + pos < n ? u32(scode[rb[pos]]) : 0u)) & wmask;
            msd_bin_slot(h, w, base + q0 + j < n);
        }
        __syncthreads();   // everyone is done with this stage (and, in the first iteration, h / scode were ready before use)
    }
    for (u32 i = threadIdx.x; i < kMsdBins; i += kMsdThreads)
        if (h[i]) msd_atomic_add(&table[i], OffT(h[i]));
}

// ---- levels >= 1: histogram of the digit at `shift` over the tiles of every row ----
template <typename OffT>
__global__ void __launch_bounds__(kMsdThreads) msd_hist_kernel(const u64* __restrict__ keys, const MsdDesc* __restrict__ tiles,
                                                               const u32* __restrict__ n_tiles, int shift, u32 dmask, OffT* __restrict__ table) {
    __shared__ u32 h[kMsdBins];
    if (blockIdx.x >= *n_tiles) return;
    const MsdDesc td = tiles[blockIdx.x];
    const u32 row = td.row, cnt = td.count;
    const u64 base = td.base;
    for (u32 i = threadIdx.x; i < kMsdBins; i += kMsdThreads) h[i] = 0;
    __syncthreads();
    u64 k[kMsdItems];
#pragma unroll
    for (int j = 0; j < kMsdItems; ++j) {
        const u32 li = j * kMsdThreads + threadIdx.x;
        k[j] = li < cnt ? keys[base + li] : 0;
    }
#pragma unroll
    for (int j = 0; j < kMsdItems; ++j) {
        const u32 li = j * kMsdThreads + threadIdx.x;
        msd_bin_slot(h, u32(k[j] >> shift) & dmask, li < cnt);
    }
    __syncthreads();
    OffT* trow = table + u64(row) * kMsdBins;
    for (u32 i = threadIdx.x; i < kMsdBins; i += kMsdThreads)
        if (h[i]) msd_atomic_add(&trow[i], OffT(h[i]));
}

// ---- bin counts -> child starts (the cursors of the scatter); children that stay large become rows of the next level ----
// ctr[0] = number of next rows, ctr[1] = their elements in total. Level 0 of a sharded build keeps bins [bin_lo, bin_hi) only.
template <typename OffT>
__global__ void __launch_bounds__(kMsdThreads) msd_rowscan_kernel(OffT* __restrict__ table, const u64* __restrict__ seg_start, u32 bin_lo,
                                                                  u32 bin_hi, int has_next, u64* __restrict__ next_start,
                                                                  u64* __restrict__ next_size, u64 next_cap, unsigned long long* __restrict__ ctr) {
    __shared__ u64 wsm[32];
    OffT* trow = table + u64(blockIdx.x) * kMsdBins;
    u64 c[kMsdItems], sum = 0;
#pragma unroll
    for (int j = 0; j < kMsdItems; ++j) {
        const u32 bin = threadIdx.x * kMsdItems + j;
        c[j] = (bin >= bin_lo && bin < bin_hi) ? u64(trow[bin]) : 0;
        sum += c[j];
    }
    u64 total;
    u64 start = seg_start[blockIdx.x] + block_exclusive_scan(sum, SumOp(), total, wsm);
#pragma unroll
    for (int j = 0; j < kMsdItems; ++j) {
        trow[threadIdx.x * kMsdItems + j] = OffT(start);
        if (has_next && c[j] > u64(kLocSmall)) {
            const u64 r = atomicAdd(&ctr[0], 1ull);
            if (r < next_cap) { next_start[r] = start; next_size[r] = c[j]; }
            atomicAdd(&ctr[1], (unsigned long long)c[j]);
        }
        start += c[j];
    }
}

// ---- partition of one tile by the level's digit ----
template <typename IdxT, typename OffT>
struct MsdScatterSmem {
    static constexpr size_t bytes = size_t(kMsdBins) * (sizeof(u32) + sizeof(OffT)) + size_t(kMsdTile) * (sizeof(u64) + sizeof(IdxT)) +
                                    (kMsdTile + kMsdHalo) + 256 + 32 * sizeof(u32);
};

// FROM_TEXT (level 0): the tile is kMsdTile text positions, keys are built here (key = first p0 symbols of the suffix, b bits
// each, first symbol most significant; value = position); pairs whose bin lies outside [bin_lo, bin_hi) are dropped (sharded
// build: another member owns them). Otherwise the tile is kMsdTile pairs of one row of (kin, vin).
template <typename IdxT, typename OffT, bool FROM_TEXT>
__global__ void __launch_bounds__(kMsdThreads, 2)
msd_scatter_kernel(const u8* __restrict__ text, u64 n, const uint16_t* __restrict__ code, int b, int p0, u32 bin_lo, u32 bin_hi,
                   const u64* __restrict__ kin, const IdxT* __restrict__ vin, const MsdDesc* __restrict__ tiles, const u32* __restrict__ n_tiles,
                   int shift, u32 dmask, OffT* __restrict__ table, u64* __restrict__ kout, IdxT* __restrict__ vout) {
    extern __shared__ __align__(16) unsigned char msd_smem[];
    u64* skey = reinterpret_cast<u64*>(msd_smem);
    OffT* delta = reinterpret_cast<OffT*>(skey + kMsdTile);
    IdxT* sval = reinterpret_cast<IdxT*>(delta + kMsdBins);
    u32* cnt = reinterpret_cast<u32*>(sval + kMsdTile);
    u32* wsm = cnt + kMsdBins;
    u8* sc = reinterpret_cast<u8*>(wsm + 32);
    u8* scode = sc + kMsdTile + kMsdHalo;

    const u32 tid = threadIdx.x;
    u32 row = 0, count;
    u64 base;
    if (FROM_TEXT) {
        base = u64(blockIdx.x) * kMsdTile;
        count = u32(min(u64(kMsdTile), n - base));
    } else {
        if (blockIdx.x >= *n_tiles) return;
        const MsdDesc td = tiles[blockIdx.x];
        row = td.row; base = td.base; count = td.count;
    }
    u64 keys[kMsdItems];
    IdxT vals[kMsdItems];
    u32 slot[kMsdItems];
    bool ok[kMsdItems];
    if (!FROM_TEXT) {   // the tile's loads are in flight while the counters are cleared
#pragma unroll
        for (int j = 0; j < kMsdItems; ++j) {
            const u32 li = j * kMsdThreads + tid;
            ok[j] = li < count;
            keys[j] = ok[j] ? kin[base + li] : 0;
            vals[j] = ok[j] ? vin[base + li] : IdxT(0);
        }
    }
    for (u32 i = tid; i < kMsdBins; i += kMsdThreads) cnt[i] = 0;
    if (FROM_TEXT) {
        if (tid < 256) scode[tid] = u8(code[tid]);
        __syncthreads();
        msd_load_codes(text, n, base, kMsdTile + kMsdHalo, scode, sc);
        __syncthreads();
        const u32 q0 = tid * kMsdItems;   // blocked: this thread rolls the key over 8 consecutive positions
        const u64 kmask = (b * p0 >= 64) ? ~u64(0) : ((u64(1) << (b * p0)) - 1);
        u64 key = 0;
        for (int j = 0; j < p0; ++j) key = (key << b) | sc[q0 + j];
#pragma unroll
        for (int j = 0; j < kMsdItems; ++j) {
            keys[j] = key;
            vals[j] = IdxT(base + q0 + j);
            const u32 d = u32(key >> shift) & dmask;
            ok[j] = q0 + j < count && d >= bin_lo && d < bin_hi;
            key = ((key << b) & kmask) | sc[q0 + j + p0];
        }
    } else {
        __syncthreads();
    }
#pragma unroll
    for (int j = 0; j < kMsdItems; ++j) slot[j] = msd_bin_slot(cnt, u32(keys[j] >> shift) & dmask, ok[j]);
    __syncthreads();

    // this thread's 8 bins: exclusive offsets inside the tile, and the place their runs go to (one global atomic per non-empty
    // bin, issued before the block scan so that its round trip hides behind the scan's barriers)
    u32 placed;
    {
        u32 c[kMsdItems], sum = 0;
        OffT gbase[kMsdItems];
        OffT* trow = table + u64(row) * kMsdBins;
#pragma unroll
        for (int j = 0; j < kMsdItems; ++j) {
            c[j] = cnt[tid * kMsdItems + j];
            sum += c[j];
            gbase[j] = c[j] ? msd_atomic_add(&trow[tid * kMsdItems + j], OffT(c[j])) : OffT(0);
        }
        u32 run = block_exclusive_scan(sum, SumOp(), placed, wsm);
#pragma unroll
        for (int j = 0; j < kMsdItems; ++j) {
            const u32 bin = tid * kMsdItems + j;
            cnt[bin] = run;
            if (c[j]) delta[bin] = gbase[j] - OffT(run);
            run += c[j];
        }
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < kMsdItems; ++j) {
        if (ok[j]) {
            const u32 lp = cnt[u32(keys[j] >> shift) & dmask] + slot[j];
            skey[lp] = keys[j];
            sval[lp] = vals[j];
        }
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < kMsdItems; ++j) {
        const u32 lp = j * kMsdThreads + tid;
        if (lp < placed) {
            const u64 k = skey[lp];
            const OffT gp = delta[u32(k >> shift) & dmask] + OffT(lp);
            kout[gp] = k;
            vout[gp] = sval[lp];
        }
    }
}

// last level with its result in B: plain copy of the rows' tiles to A
template <typename IdxT>
__global__ void __launch_bounds__(kMsdThreads) msd_copy_tiles_kernel(const u64* __restrict__ kin, const IdxT* __restrict__ vin,
                                                                     const MsdDesc* __restrict__ tiles, const u32* __restrict__ n_tiles,
                                                                     u64* __restrict__ kout, IdxT* __restrict__ vout) {
    if (blockIdx.x >= *n_tiles) return;
    const u64 base = tiles[blockIdx.x].base;
    const u32 count = tiles[blockIdx.x].count;
    for (u32 i = threadIdx.x; i < count; i += kMsdThreads) { kout[base + i] = kin[base + i]; vout[base + i] = vin[base + i]; }
}

// ---- local sort ----
// A batch = the pairs of consecutive small children of one row (at most kLocCap). The children are already in digit order;
// what is left is the order inside each child, by the key bits below the level's digit.
//   fast path   one more partition step inside shared memory: sub-bucket = (child, next w key bits), w as large as the
//               counter budget allows for the number of children in the batch (26 children of ~184 pairs at 3.1 Gbp:
//               w = 7 -> sub-buckets of ~6 pairs), one shared atomic per pair; then every pair finds its rank inside its
//               sub-bucket by comparing its key with the sub-bucket's other keys (one pair per thread and step: O(m) per
//               pair, no divergence beyond the sub-bucket sizes). ~120 instructions per pair.
//   slow path   when some sub-bucket is still long (high-copy repeats, low complexity): stable LSD counting sort of the
//               batch over all bits that can differ (5-bit digits, private per-thread counters) — ~90 instructions per pair
//               and pass, independent of the key distribution (measured: 94 ms for 3 G pairs over 30 bits, the fast path
//               with one thread insertion-sorting each sub-bucket: 166 ms, 41 G warp instructions at half-empty warps).
constexpr int kLocCounters = 2 * kLocCap;  // sub-bucket counters of the fast path: 16 bits each, two per u32 word
constexpr int kLocRankMax = 64;            // longest sub-bucket the fast path finishes by ranking
constexpr int kLocFastItems = kLocCap / kLocThreads;

template <typename IdxT>
struct MsdLocalSmem {
    // fast path: counters + child ordinals; slow path: cnt16[32][512] + row totals — the same 32 KB + 1 KB
    static constexpr size_t aux = size_t(kLocDigits) * kLocThreads * sizeof(uint16_t) + 2 * kLocDigits * sizeof(u32) + 768;
    static constexpr size_t bytes = size_t(kLocCap) * (sizeof(u64) + sizeof(IdxT)) + aux;
};
static_assert(size_t(kLocCounters / 2 + 1) * sizeof(u32) + size_t(kMsdBins) * sizeof(uint16_t) <= MsdLocalSmem<u32>::aux, "fast-path tables must fit");
static_assert(kLocItems * kLocThreads >= kLocCap && kLocFastItems * kLocThreads == kLocCap, "local sort shapes");

// first index i in [0, 4096) with arr[i] >= v (4096 when there is none); arr non-decreasing. Every warp runs the same
// 32-way search (three dependent loads instead of twelve); all lanes return the same value.
template <typename OffT>
__device__ __forceinline__ u32 msd_lower_bound_4096(const OffT* __restrict__ arr, u64 v) {
    const u32 lane = lane_id();
    unsigned m = __ballot_sync(0xffffffffu, u64(arr[lane * 128 + 127]) >= v);
    if (m == 0) return u32(kMsdBins);
    u32 base = (__ffs(m) - 1) * 128;
    m = __ballot_sync(0xffffffffu, u64(arr[base + lane * 4 + 3]) >= v);
    base += (__ffs(m) - 1) * 4;
    m = __ballot_sync(0xffffffffu, lane < 4 && u64(arr[base + (lane & 3u)]) >= v);
    return base + (__ffs(m) - 1);
}

// Stable LSD counting sort of sk/sv[0, count) (in shared memory) by key bits [0, hb): thread t owns pairs [13 t, 13 t + 13)
// of the current order (blocked), counts its digits into its own column of cnt16[digit][thread], the columns are scanned
// digit-major (2 digits per warp, 16 counters per lane), and every pair then knows its place without atomics.
template <typename IdxT>
__device__ __noinline__ void msd_local_lsd(u64* sk, IdxT* sv, u32 count, int hb, uint16_t* cnt16, u32* rowtot, u32* rowbase) {
    const u32 tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const int passes = (hb + kLocDigitBits - 1) / kLocDigitBits;
    u64 key[kLocItems];
    IdxT val[kLocItems];
    const u32 e0 = tid * kLocItems;
    for (int p = 0; p < passes; ++p) {
        const int shift = p * kLocDigitBits;
#pragma unroll
        for (int j = 0; j < kLocItems; ++j)
            if (e0 + j < count) { key[j] = sk[e0 + j]; val[j] = sv[e0 + j]; }
        {   // zero the counters (32 KB)
            uint4* z = reinterpret_cast<uint4*>(cnt16);
            for (u32 i = tid; i < kLocDigits * kLocThreads * sizeof(uint16_t) / 16; i += kLocThreads) z[i] = make_uint4(0, 0, 0, 0);
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < kLocItems; ++j)
            if (e0 + j < count) cnt16[(u32(key[j] >> shift) & (kLocDigits - 1)) * kLocThreads + tid] += 1;
        __syncthreads();
        // exclusive scan inside every digit's row of kLocThreads counters (16 per lane); row totals to rowtot[]
#pragma unroll
        for (int q = 0; q < kLocDigits / (kLocThreads / 32); ++q) {
            const u32 d = warp * (kLocDigits / (kLocThreads / 32)) + q;
            uint4* rowp = reinterpret_cast<uint4*>(cnt16 + d * kLocThreads) + lane * 2;   // 16 counters of 16 bits
            const uint4 v0 = rowp[0], v1 = rowp[1];
            u32 c[16] = {v0.x & 0xffffu, v0.x >> 16, v0.y & 0xffffu, v0.y >> 16, v0.z & 0xffffu, v0.z >> 16, v0.w & 0xffffu, v0.w >> 16,
                         v1.x & 0xffffu, v1.x >> 16, v1.y & 0xffffu, v1.y >> 16, v1.z & 0xffffu, v1.z >> 16, v1.w & 0xffffu, v1.w >> 16};
            u32 s = 0;
#pragma unroll
            for (int i = 0; i < 16; ++i) { const u32 t = c[i]; c[i] = s; s += t; }
            u32 inc = s;
#pragma unroll
            for (int dd = 1; dd < 32; dd <<= 1) { const u32 o = __shfl_up_sync(0xffffffffu, inc, dd); if (lane >= u32(dd)) inc += o; }
            const u32 exc = inc - s;
#pragma unroll
            for (int i = 0; i < 16; ++i) c[i] += exc;
            rowp[0] = make_uint4(c[0] | (c[1] << 16), c[2] | (c[3] << 16), c[4] | (c[5] << 16), c[6] | (c[7] << 16));
            rowp[1] = make_uint4(c[8] | (c[9] << 16), c[10] | (c[11] << 16), c[12] | (c[13] << 16), c[14] | (c[15] << 16));
            if (lane == 31) rowtot[d] = inc;
        }
        __syncthreads();
        if (warp == 0) {   // exclusive scan of the 32 row totals
            const u32 a = rowtot[lane];
            u32 inc = a;
#pragma unroll
            for (int dd = 1; dd < 32; dd <<= 1) { const u32 o = __shfl_up_sync(0xffffffffu, inc, dd); if (lane >= u32(dd)) inc += o; }
            rowbase[lane] = inc - a;
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < kLocItems; ++j) {
            if (e0 + j < count) {
                const u32 d = u32(key[j] >> shift) & (kLocDigits - 1);
                const u32 ci = d * kLocThreads + tid;
                const u32 r = rowbase[d] + cnt16[ci];
                cnt16[ci] += 1;
                sk[r] = key[j];
                sv[r] = val[j];
            }
        }
        __syncthreads();
    }
}

// 16-bit counters packed two per word: bump counter `sub`, return its previous value (the pair's slot in its sub-bucket).
// A warp whose lanes all hit one counter takes one atomic.
__device__ __forceinline__ u32 msd_sub_slot(u32* cnt, u32 sub, bool valid) {
    const u32 sh = (sub & 1u) * 16u;
    const u32 s0 = __shfl_sync(0xffffffffu, sub, 0);
    if (__all_sync(0xffffffffu, valid && sub == s0)) {
        u32 old = 0;
        if (lane_id() == 0) old = atomicAdd(&cnt[s0 >> 1], 32u << sh);
        return ((__shfl_sync(0xffffffffu, old, 0) >> sh) & 0xffffu) + lane_id();
    }
    return valid ? ((atomicAdd(&cnt[sub >> 1], 1u << sh) >> sh) & 0xffffu) : 0u;
}
__device__ __forceinline__ u32 msd_sub_off(const u32* cnt, u32 sub) { return (cnt[sub >> 1] >> ((sub & 1u) * 16u)) & 0xffffu; }

// Sorts pairs [lo, hi) (hi - lo <= kLocCap; whole children of the row, bins [ba, bb) of its table E) of (src_k, src_v) by
// the key bits below `shift` inside every child, into (dst_k, dst_v) at the same positions. The batch is fetched with
// cp.async while the child ordinals are worked out from the row's table.
template <typename IdxT, typename OffT>
__device__ void msd_local_sort_range(const u64* __restrict__ src_k, const IdxT* __restrict__ src_v, u64* __restrict__ dst_k,
                                     IdxT* __restrict__ dst_v, u64 lo, u32 count, const OffT* __restrict__ E, u32 ba, u32 bb,
                                     int shift, u32 dmask, u64* sk, IdxT* sv, unsigned char* aux) {
    __shared__ u32 wsm[32];
    __shared__ u32 s_max;
    const u32 tid = threadIdx.x;
    u32* cnt = reinterpret_cast<u32*>(aux);                                       // [kLocCounters / 2 + 1] packed 16-bit counters
    uint16_t* ord = reinterpret_cast<uint16_t*>(cnt + kLocCounters / 2 + 1);       // [bb - ba] dense ordinal of every non-empty child
    // ---- the batch starts to travel: 8 bytes per key, 4 or 8 per value, striped over the threads
    for (u32 i = tid; i < count; i += kLocThreads) {
        const u32 dk = u32(__cvta_generic_to_shared(sk + i));
        asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dk), "l"(src_k + lo + i));
        const u32 dv = u32(__cvta_generic_to_shared(sv + i));
        if constexpr (sizeof(IdxT) == 4) asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dv), "l"(src_v + lo + i));
        else asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dv), "l"(src_v + lo + i));
    }
    asm volatile("cp.async.commit_group;");
    // ---- dense child ordinals over the bins of the range
    const u32 span = bb - ba;
    u32 nchild;
    {
        constexpr int PER = kMsdBins / kLocThreads;   // 8
        u32 flags = 0, c = 0;
#pragma unroll
        for (int q = 0; q < PER; ++q) {
            const u32 r = tid * PER + q;
            if (r < span) {
                const u32 bin = ba + r;
                const u64 s = r == 0 ? lo : u64(E[bin - 1]);
                if (u64(E[bin]) > s) { flags |= 1u << q; ++c; }
            }
        }
        u32 run = block_exclusive_scan(c, SumOp(), nchild, wsm);
#pragma unroll
        for (int q = 0; q < PER; ++q) {
            const u32 r = tid * PER + q;
            if (r < span) { ord[r] = uint16_t(run); run += (flags >> q) & 1u; }
        }
    }
    // w = key bits of the in-smem partition step: as many as the counters allow for this many children
    int w = 0;
    while (w < 12 && w < shift && (u64(nchild) << (w + 1)) <= u64(kLocCounters)) ++w;
    const bool fast = nchild >= 1 && nchild <= u32(kLocCounters) && shift > 0;
    const u32 nsub = fast ? (nchild << w) : 0;
    for (u32 i = tid; i <= nsub / 2; i += kLocThreads) cnt[i] = 0;
    if (tid == 0) s_max = 0;
    asm volatile("cp.async.wait_group 0;");
    __syncthreads();
    bool ranked = false;
    if (fast) {
        // Register budget: 64 per thread (two blocks of 512 per SM): slots / ranks are kept as 16-bit halves
        u32 slot2[kLocFastItems / 2];
        const int wshift = shift - w;
        const u32 wmask = (1u << w) - 1u;
#pragma unroll
        for (int j = 0; j < kLocFastItems; ++j) {
            const u32 li = j * kLocThreads + tid;
            const bool ok = li < count;
            const u64 k = ok ? sk[li] : 0;
            const u32 d = (u32(k >> shift) & dmask) - ba;
            const u32 sub = ok ? ((u32(ord[d]) << w) | (u32(k >> wshift) & wmask)) : 0u;
            const u32 sl = msd_sub_slot(cnt, sub, ok);
            if (j & 1) slot2[j >> 1] |= sl << 16; else slot2[j >> 1] = sl;
        }
        __syncthreads();
        {   // exclusive scan of the sub-bucket counts in place (packed; cnt word nsub / 2 also closes the table); longest sub-bucket
            constexpr int PER = kLocCounters / 2 / kLocThreads;   // 12 words = 24 counters per thread, read twice rather than kept
            const u32 nw = nsub / 2 + 1;
            u32 sum = 0, mx = 0;
#pragma unroll
            for (int q = 0; q < PER + 1; ++q) {
                const u32 i = tid * PER + q;
                if (q < PER || tid == kLocThreads - 1) {
                    const u32 v = i < nw ? cnt[i] : 0;
                    sum += (v & 0xffffu) + (v >> 16);
                    mx = max(mx, max(v & 0xffffu, v >> 16));
                }
            }
            u32 total;
            u32 run = block_exclusive_scan(sum, SumOp(), total, wsm);
#pragma unroll
            for (int q = 0; q < PER + 1; ++q) {
                const u32 i = tid * PER + q;
                if ((q < PER || tid == kLocThreads - 1) && i < nw) {
                    const u32 v = cnt[i];
                    const u32 a0 = run, a1 = run + (v & 0xffffu);
                    cnt[i] = a0 | (a1 << 16);
                    run = a1 + (v >> 16);
                }
            }
#pragma unroll
            for (int dd = 16; dd; dd >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, dd));
            if ((tid & 31u) == 0) atomicMax(&s_max, mx);
        }
        __syncthreads();
        ranked = s_max <= u32(kLocRankMax);
        {   // place: the pairs move from their striped places to their sub-buckets (through registers: in place)
            u64 key[kLocFastItems];
            IdxT val[kLocFastItems];
#pragma unroll
            for (int j = 0; j < kLocFastItems; ++j) {
                const u32 li = j * kLocThreads + tid;
                if (li < count) { key[j] = sk[li]; val[j] = sv[li]; }
            }
            __syncthreads();
#pragma unroll
            for (int j = 0; j < kLocFastItems; ++j) {
                const u32 li = j * kLocThreads + tid;
                if (li < count) {
                    const u64 k = key[j];
                    const u32 d = (u32(k >> shift) & dmask) - ba;
                    const u32 sub = (u32(ord[d]) << w) | (u32(k >> wshift) & wmask);
                    const u32 pos = msd_sub_off(cnt, sub) + ((slot2[j >> 1] >> ((j & 1) * 16)) & 0xffffu);
                    sk[pos] = k;
                    sv[pos] = val[j];
                }
            }
        }
        __syncthreads();
        if (ranked) {
            // every pair: its rank among the keys of its sub-bucket (ties by position) -> final place. Inside a sub-bucket only
            // the bits below wshift differ: when those fit a word the comparisons run on the low words.
            const bool low32 = wshift <= 32;
#pragma unroll
            for (int j = 0; j < kLocFastItems; ++j) {
                const u32 p = j * kLocThreads + tid;
                u32 r = 0xffffu;
                if (p < count) {
                    const u64 k = sk[p];
                    const u32 d = (u32(k >> shift) & dmask) - ba;
                    const u32 sub = (u32(ord[d]) << w) | (u32(k >> wshift) & wmask);
                    const u32 s0 = msd_sub_off(cnt, sub), s1 = msd_sub_off(cnt, sub + 1);
                    r = s0;
                    if (low32) {
                        const u32 kl = u32(k);
                        const u32* skl = reinterpret_cast<const u32*>(sk);
                        for (u32 q = s0; q < s1; ++q) {
                            const u32 o = skl[2 * q];
                            r += (o < kl || (o == kl && q < p)) ? 1u : 0u;
                        }
                    } else {
                        for (u32 q = s0; q < s1; ++q) {
                            const u64 o = sk[q];
                            r += (o < k || (o == k && q < p)) ? 1u : 0u;
                        }
                    }
                }
                if (j & 1) slot2[j >> 1] |= r << 16; else slot2[j >> 1] = r;
            }
            {   // permute the keys, then the values (one array at a time: half the registers)
                u64 key[kLocFastItems];
#pragma unroll
                for (int j = 0; j < kLocFastItems; ++j) { const u32 p = j * kLocThreads + tid; if (p < count) key[j] = sk[p]; }
                __syncthreads();
#pragma unroll
                for (int j = 0; j < kLocFastItems; ++j) { const u32 p = j * kLocThreads + tid; if (p < count) sk[(slot2[j >> 1] >> ((j & 1) * 16)) & 0xffffu] = key[j]; }
            }
            {
                IdxT val[kLocFastItems];
#pragma unroll
                for (int j = 0; j < kLocFastItems; ++j) { const u32 p = j * kLocThreads + tid; if (p < count) val[j] = sv[p]; }
                __syncthreads();
#pragma unroll
                for (int j = 0; j < kLocFastItems; ++j) { const u32 p = j * kLocThreads + tid; if (p < count) sv[(slot2[j >> 1] >> ((j & 1) * 16)) & 0xffffu] = val[j]; }
            }
            __syncthreads();
        }
    }
    if (!ranked) {
        // the batch sits in shared memory (in child order, grouped by sub-bucket when the fast path ran): sort it over every
        // bit that can differ — the children are in digit order, so the first and the last key bound the digit bits
        uint16_t* cnt16 = reinterpret_cast<uint16_t*>(aux);
        u32* rowtot = reinterpret_cast<u32*>(cnt16 + kLocDigits * kLocThreads);
        const u64 x = (sk[0] ^ sk[count - 1]) >> shift;
        const int hb = shift + (x ? 64 - __clzll((long long)x) : 0);
        __syncthreads();
        msd_local_lsd<IdxT>(sk, sv, count, hb, cnt16, rowtot, rowtot + kLocDigits);
    }
    for (u32 i = tid; i < count; i += kLocThreads) { dst_k[lo + i] = sk[i]; dst_v[lo + i] = sv[i]; }
    __syncthreads();
}

// A batch of the local sort: consecutive small children of one row, at most kLocCap pairs.
struct MsdBatch {
    u64 lo;
    u32 count, row, ba, bb;
};

// One warp per window of kLocWindow positions of a row: the children that START inside the window, except those that went
// on to the next level (larger than kLocSmall), become one batch — or several, when large children lie in between.
// `table` holds the children's END offsets (the scatter advanced every cursor from the child's start to its end).
// Doing this ahead of the sort takes a chain of eight dependent table reads out of every sorting block, and windows
// without small children (levels whose children all went on) cost one warp here instead of one block there.
template <typename OffT>
__global__ void __launch_bounds__(256) msd_batches_kernel(const OffT* __restrict__ table, const MsdDesc* __restrict__ wins,
                                                          const u32* __restrict__ n_wins, MsdBatch* __restrict__ batches,
                                                          u32* __restrict__ n_batches, u32 cap, u32* __restrict__ err) {
    const u32 win = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31u;
    if (win >= *n_wins) return;
    const MsdDesc wd = wins[win];     // base = first position of the window, count = index of the window inside its row
    const OffT* E = table + u64(wd.row) * kMsdBins;
    const u64 seg_hi = u64(E[kMsdBins - 1]);  // the last child ends where the row ends
    const u64 wlo = wd.base, whi = min(wlo + u64(kLocWindow), seg_hi);
    // child b starts at E[b - 1] (child 0 at the row's start = the first window's wlo): the children starting in [wlo, whi)
    const u32 b0 = wd.count == 0 ? 0u : 1u + msd_lower_bound_4096(E, wlo);
    const u32 b1 = whi == seg_hi ? u32(kMsdBins) : 1u + msd_lower_bound_4096(E, whi);
    if (b0 >= b1) return;
    const u64 lo = b0 == 0 ? wlo : u64(E[b0 - 1]);
    const u64 hi = u64(E[b1 - 1]);
    if (lo >= hi) return;
    auto emit = [&](u64 from, u64 to, u32 ba, u32 bb) {
        if (lane != 0) return;
        if (to - from > u64(kLocCap)) { atomicOr(err, 2u); return; }
        const u32 i = atomicAdd(n_batches, 1u);
        if (i >= cap) { atomicOr(err, 4u); return; }
        MsdBatch bt;
        bt.lo = from; bt.count = u32(to - from); bt.row = wd.row; bt.ba = ba; bt.bb = bb;
        batches[i] = bt;
    };
    u64 cur = lo;
    u32 cur_b = b0;
    for (u32 base = b0; base < b1; base += 32) {
        const u32 bq = base + lane;
        u64 s = 0, e = 0;
        if (bq < b1) { s = bq == b0 ? lo : u64(E[bq - 1]); e = u64(E[bq]); }
        unsigned big = __ballot_sync(0xffffffffu, bq < b1 && e - s > u64(kLocSmall));
        while (big) {
            const int l = __ffs(big) - 1;
            const u64 bs = __shfl_sync(0xffffffffu, s, l), be = __shfl_sync(0xffffffffu, e, l);
            if (bs > cur) emit(cur, bs, cur_b, base + l);
            cur = be;
            cur_b = base + l + 1;
            big &= big - 1;
        }
    }
    if (hi > cur) emit(cur, hi, cur_b, b1);
}

template <typename IdxT, typename OffT>
__global__ void __launch_bounds__(kLocThreads, 2)
msd_local_kernel(const u64* __restrict__ src_k, const IdxT* __restrict__ src_v, u64* __restrict__ dst_k, IdxT* __restrict__ dst_v,
                 const OffT* __restrict__ table, const MsdBatch* __restrict__ batches, const u32* __restrict__ n_batches, int shift,
                 u32 dmask) {
    extern __shared__ __align__(16) unsigned char msd_smem[];
    u64* sk = reinterpret_cast<u64*>(msd_smem);
    IdxT* sv = reinterpret_cast<IdxT*>(sk + kLocCap);
    unsigned char* aux = reinterpret_cast<unsigned char*>(sv + kLocCap);
    if (blockIdx.x >= *n_batches) return;
    const MsdBatch bt = batches[blockIdx.x];
    msd_local_sort_range<IdxT, OffT>(src_k, src_v, dst_k, dst_v, bt.lo, bt.count, table + u64(bt.row) * kMsdBins, bt.ba, bt.bb, shift, dmask,
                                     sk, sv, aux);
}

// ---------------------------------------------------------------------------------------------------------------
struct MsdStats {
    FamilyTimer* scatter = nullptr;    // msd_scatter_kernel, levels >= 1 (24 B per pair)
    FamilyTimer* scatter0 = nullptr;   // level 0 (text -> pairs: 1 + 12 B per suffix)
    FamilyTimer* hist = nullptr;
    FamilyTimer* local = nullptr;
    int levels = 0;
};

inline bool msd_sort_applicable(int b, int p0, u64 n) {
    static const char* knob = getenv("ASGART_B200_MSD_MIN");   // developer/test knob: smallest n that takes the MSD path
    const u64 min_n = knob ? u64(strtoull(knob, nullptr, 10)) : (u64(1) << 21);
    return (b == 2 || b == 3 || b == 4) && b * p0 >= 2 * kMsdDigitBits && p0 <= 32 && n >= min_n && n >= 1;
}

// Sorts the suffixes of text[0, n) whose level-0 bin lies in [bin_lo, bin_hi) (all of them: 0, 4096) by their first p0
// symbols. On return (keys_a, vals_a) hold the n_out sorted pairs. keys_b / vals_b: scratch of the same size.
// `table0` (optional, 4096 entries, already holding the level-0 histogram of the WHOLE text) lets a sharded build reuse the
// histogram it cut the members' ranges from. Returns false when a level's tables would not fit `table_budget` bytes
// (pathological bucket structure): the caller then falls back to the LSD sort.
template <typename IdxT>
bool msd_sort_suffixes(const u8* d_text, u64 n, const uint16_t* d_code, int b, int p0, u32 bin_lo, u32 bin_hi, u64 n_out, u64* keys_a,
                       IdxT* vals_a, u64* keys_b, IdxT* vals_b, IdxT* d_table0, cudaStream_t stream, MsdStats* st = nullptr,
                       size_t table_budget = size_t(12) << 30) {
    using OffT = IdxT;
    const MsdLevels L(b * p0);
    if (n == 0 || n_out == 0) return true;
    static std::atomic<unsigned long long> prepared{0};   // per IdxT instantiation, one bit per device
    unsigned long long dev_bit = 0;
    constexpr size_t smem_sc = MsdScatterSmem<IdxT, OffT>::bytes, smem_loc = MsdLocalSmem<IdxT>::bytes;
    if (device_needs_prepare(prepared, dev_bit)) {
        CUDA_CHECK(cudaFuncSetAttribute(msd_scatter_kernel<IdxT, OffT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem_sc)));
        CUDA_CHECK(cudaFuncSetAttribute(msd_scatter_kernel<IdxT, OffT, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem_sc)));
        CUDA_CHECK(cudaFuncSetAttribute(msd_local_kernel<IdxT, OffT>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem_loc)));
        device_prepared(prepared, dev_bit);
    }
    DevBuf<unsigned long long> d_ctr(2, stream);
    DevBuf<u32> d_err(1, stream);
    d_err.zero();
    auto read_ctr = [&](unsigned long long* h) {
        CUDA_CHECK(cudaMemcpyAsync(h, d_ctr.p, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, stream));
        CUDA_CHECK(cudaStreamSynchronize(stream));
    };

    // rows of the current level
    u64 rows = 1, elems = n_out;
    DevBuf<u64> seg_start(1, stream), seg_size(1, stream);
    {
        const u64 h_seg[2] = {0, n_out};
        CUDA_CHECK(cudaMemcpyAsync(seg_start.p, &h_seg[0], sizeof(u64), cudaMemcpyHostToDevice, stream));
        CUDA_CHECK(cudaMemcpyAsync(seg_size.p, &h_seg[1], sizeof(u64), cudaMemcpyHostToDevice, stream));
    }
    DevBuf<u32> tile_first, win_first;
    u64 *src_k = nullptr, *dst_k = keys_a;   // level 0 writes A
    IdxT *src_v = nullptr, *dst_v = vals_a;

    for (int lv = 0; lv < L.n; ++lv) {
        const int shift = L.shift[lv];
        const u32 dmask = (1u << L.width[lv]) - 1u;
        const bool has_next = lv + 1 < L.n;
        const bool to_a = dst_k == keys_a;
        if (st) st->levels = lv + 1;
        // ---- tiles / windows of the rows: one descriptor each (upper bounds size the grids; the true counts sit at first[rows])
        u64 tiles_ub, wins_ub;
        if (lv == 0) {
            tiles_ub = ceil_div(n, u64(kMsdTile));
            wins_ub = ceil_div(n_out, u64(kLocWindow));
            tile_first.alloc(2, stream);
            win_first.alloc(2, stream);
            const u32 h_t[2] = {0, u32(tiles_ub)}, h_w[2] = {0, u32(wins_ub)};
            CUDA_CHECK(cudaMemcpyAsync(tile_first.p, h_t, sizeof h_t, cudaMemcpyHostToDevice, stream));
            CUDA_CHECK(cudaMemcpyAsync(win_first.p, h_w, sizeof h_w, cudaMemcpyHostToDevice, stream));
        } else {
            tiles_ub = elems / kMsdTile + rows;
            wins_ub = elems / kLocWindow + rows;
            tile_first.alloc(rows + 1, stream);
            win_first.alloc(rows + 1, stream);
            const u64* sz = seg_size.p;
            u32 *tf = tile_first.p, *wf = win_first.p;
            device_scan<u32, SumOp>([sz] __device__(u64 r) { return u32((sz[r] + kMsdTile - 1) / kMsdTile); },
                                    [tf] __device__(u64 r, u32 exc, u32) { tf[r] = exc; }, rows, tile_first.p + rows, stream);
            device_scan<u32, SumOp>([sz] __device__(u64 r) { return u32((sz[r] + kLocWindow - 1) / kLocWindow); },
                                    [wf] __device__(u64 r, u32 exc, u32) { wf[r] = exc; }, rows, win_first.p + rows, stream);
        }
        DevBuf<MsdDesc> tile_desc(lv == 0 ? 0 : tiles_ub, stream), win_desc(has_next ? wins_ub : 0, stream);
        if (lv > 0) {
            msd_expand_kernel<false><<<unsigned(rows), 128, 0, stream>>>(seg_start.p, seg_size.p, tile_first.p, tile_desc.p);
            KERNEL_CHECK();
            count_launch();
        }
        if (has_next) {
            msd_expand_kernel<true><<<unsigned(rows), 128, 0, stream>>>(seg_start.p, seg_size.p, win_first.p, win_desc.p);
            KERNEL_CHECK();
            count_launch();
        }
        const u32* n_tiles = tile_first.p + rows;
        const u32* n_wins = win_first.p + rows;
        // ---- histogram
        if (rows * kMsdBins * sizeof(OffT) > table_budget) return false;
        DevBuf<OffT> table;
        OffT* tp;
        if (lv == 0 && d_table0) tp = d_table0;
        else {
            table.alloc(rows * kMsdBins, stream);
            table.zero();
            tp = table.p;
            if (st && st->hist) st->hist->begin();
            if (lv == 0) {
                const int blocks = int(std::min<u64>(ceil_div(n, u64(kH0Tile)), u64(kNumSMs) * 2));
                msd_hist_text_kernel<OffT><<<blocks, kMsdThreads, 0, stream>>>(d_text, n, d_code, b, L.width[0] / b, tp, 0, ~u64(0));
            } else {
                msd_hist_kernel<OffT><<<unsigned(tiles_ub), kMsdThreads, 0, stream>>>(src_k, tile_desc.p, n_tiles, shift, dmask, tp);
            }
            KERNEL_CHECK();
            count_launch();
            if (st && st->hist) st->hist->end(1, lv == 0 ? n : elems * sizeof(u64));
        }
        // ---- child offsets; the next level's rows
        const u64 next_cap = has_next ? std::min<u64>(elems / kLocSmall + 1, rows * kMsdBins) : 1;
        DevBuf<u64> next_start(next_cap, stream), next_size(next_cap, stream);
        d_ctr.zero();
        msd_rowscan_kernel<OffT><<<unsigned(rows), kMsdThreads, 0, stream>>>(tp, seg_start.p, lv == 0 ? bin_lo : 0u, lv == 0 ? bin_hi : u32(kMsdBins),
                                                                            has_next ? 1 : 0, next_start.p, next_size.p, next_cap, d_ctr.p);
        KERNEL_CHECK();
        count_launch();
        // ---- scatter
        if (lv == 0) {
            if (st && st->scatter0) st->scatter0->begin();
            msd_scatter_kernel<IdxT, OffT, true><<<unsigned(tiles_ub), kMsdThreads, smem_sc, stream>>>(
                d_text, n, d_code, b, p0, bin_lo, bin_hi, nullptr, nullptr, nullptr, nullptr, shift, dmask, tp, dst_k, dst_v);
            KERNEL_CHECK();
            if (st && st->scatter0) st->scatter0->end(1, n + n_out * (sizeof(u64) + sizeof(IdxT)));
        } else {
            if (st && st->scatter) st->scatter->begin();
            msd_scatter_kernel<IdxT, OffT, false><<<unsigned(tiles_ub), kMsdThreads, smem_sc, stream>>>(
                nullptr, 0, nullptr, b, p0, 0, kMsdBins, src_k, src_v, tile_desc.p, n_tiles, shift, dmask, tp, dst_k, dst_v);
            KERNEL_CHECK();
            if (st && st->scatter) st->scatter->end(1, elems * 2 * (sizeof(u64) + sizeof(IdxT)));
        }
        count_launch();
        // ---- finish the small children (or, after the last level, bring the rows home to A)
        unsigned long long h_ctr[2] = {0, 0};
        if (has_next) {
            read_ctr(h_ctr);    // rows of the next level, pairs in them: everything else of this level is a small child
            if (h_ctr[0] > next_cap) throw CudaError(ASGART_B200_ECUDA, "msd sort: more large children than fit the row list");
            if (elems > h_ctr[1]) {
                if (st && st->local) st->local->begin();
                // windows -> batches (a window yields one batch, plus one per large child inside it), then one block per batch
                const u64 cap = wins_ub + h_ctr[0] + 1;
                DevBuf<MsdBatch> batches(cap, stream);
                DevBuf<u32> n_batches(1, stream);
                n_batches.zero();
                msd_batches_kernel<OffT><<<unsigned(ceil_div(wins_ub, 8)), 256, 0, stream>>>(tp, win_desc.p, n_wins, batches.p, n_batches.p, u32(cap), d_err.p);
                KERNEL_CHECK();
                msd_local_kernel<IdxT, OffT><<<unsigned(cap), kLocThreads, smem_loc, stream>>>(dst_k, dst_v, keys_a, vals_a, tp, batches.p, n_batches.p,
                                                                                              shift, dmask);
                KERNEL_CHECK();
                count_launch(2);
                if (st && st->local) st->local->end(1, (elems - h_ctr[1]) * 2 * (sizeof(u64) + sizeof(IdxT)));
            }
        } else if (!to_a) {
            msd_copy_tiles_kernel<IdxT><<<unsigned(tiles_ub), kMsdThreads, 0, stream>>>(dst_k, dst_v, tile_desc.p, n_tiles, keys_a, vals_a);
            KERNEL_CHECK();
            count_launch();
        }
        if (!has_next || h_ctr[0] == 0) break;
        rows = h_ctr[0];
        elems = h_ctr[1];
        seg_start = std::move(next_start);
        seg_size = std::move(next_size);
        // the next level reads what this one wrote
        src_k = dst_k; src_v = dst_v;
        dst_k = to_a ? keys_b : keys_a;
        dst_v = to_a ? vals_b : vals_a;
    }
    u32 h_err = 0;
    CUDA_CHECK(cudaMemcpyAsync(&h_err, d_err.p, sizeof h_err, cudaMemcpyDeviceToHost, stream));
    CUDA_CHECK(cudaStreamSynchronize(stream));
    if (h_err) throw CudaError(ASGART_B200_ECUDA, "msd sort: local-sort window overflow (internal error)");
    return true;
}

}  // namespace ab200
