// scatter.cuh — out[idx[i]] = val[i] for an injective idx: the inverse-permutation scatter that turns "rank by sorted
// position" into "rank by text position" in the suffix-array build. The build only comes here when it has no lookup tables
// for the lazy ranks of sa_build.cuh: the divsufsort64 drop-in, --trim, and texts under 256 symbols.
//
// A plain scatter of 4-byte values to random addresses costs a DRAM read-modify-write per element (B200, measured with
// tools/scatter_bench.cu: 30.8 G elem/s for 57 M targets, 22.7 G elem/s for 1 G). When all targets of a launch fall
// inside a slice of `out` that the L2 holds (<= 48 MB), the writes combine in L2 and leave as whole lines: 98 G elem/s
// with four sweeps over 57 M elements. So:
//   out fits one slice          -> plain scatter
//   a few slices (<= kSweepMax) -> one sweep over (idx, val) per slice, each writing only its slice's targets
//   more, idx a permutation     -> sort the pairs back by target: two partition passes by bits [16, 32) of idx leave
//                                  the pairs of every 65 536-target bucket contiguous (bucket b = pairs [b << 16, (b+1) << 16),
//                                  because idx is a permutation); one block per bucket then scatters inside shared memory
//                                  and writes its slice of `out` as whole lines. The order inside a bucket is irrelevant, so
//                                  the passes need not be stable: most significant digit first (regions of 2^24 targets,
//                                  which a permutation fills exactly), then the next digit inside every region, each element
//                                  ranked by one shared-memory atomic instead of the stable sort's ballot matching. No random access reaches L2 or DRAM:
//                                  52 B of streamed traffic per element instead of a 64 B DRAM read-modify-write at
//                                  random-access efficiency (C4, 3.1 G targets: 132 ms for the plain scatter).
//   more, otherwise             -> plain scatter. Tried and dropped: one radix partition pass of the pairs by slice number
//                                  followed by an in-order scatter into L2-sized slices (profiles/r1_scatter_bench.log):
//                                  the L2 takes 26-51 G scattered elem/s only.
#pragma once
#include "common.cuh"
#include "radix_sort.cuh"

namespace ab200 {

constexpr u64 kScatterSliceBytes = u64(48) << 20;
constexpr int kSweepMax = 6;

template <typename IdxT>
__global__ void __launch_bounds__(256) scatter_slice_kernel(const IdxT* __restrict__ idx, const IdxT* __restrict__ val, u64 n,
                                                            IdxT* __restrict__ out, u64 lo, u64 hi) {
    constexpr int V = 16 / sizeof(IdxT);
    const u64 stride = u64(gridDim.x) * blockDim.x * V;
    for (u64 i = (u64(blockIdx.x) * blockDim.x + threadIdx.x) * V; i < n; i += stride) {
        if (i + V <= n) {
            IdxT p[V], v[V];
            *reinterpret_cast<uint4*>(p) = __ldcs(reinterpret_cast<const uint4*>(idx + i));   // streaming: the L2 is for the written lines
            *reinterpret_cast<uint4*>(v) = __ldcs(reinterpret_cast<const uint4*>(val + i));
#pragma unroll
            for (int j = 0; j < V; ++j)
                if (u64(p[j]) >= lo && u64(p[j]) < hi) out[p[j]] = v[j];
        } else {
            for (u64 j = i; j < n; ++j) { const u64 p = u64(idx[j]); if (p >= lo && p < hi) out[p] = val[j]; }
        }
    }
}

// One block per bucket of 2^kBucketBits targets whose pairs are contiguous: the values are placed in shared memory, half a
// bucket (128 KB) at a time, and leave as coalesced 16-byte stores. The second half re-reads the pairs (L2 hits).
constexpr int kBucketBits = 16;
constexpr int kBucketHalfBits = kBucketBits - 1;
constexpr int kBucketThreads = 1024;

__global__ void __launch_bounds__(kBucketThreads, 1) bucket_scatter_kernel(const u32* __restrict__ idx, const u32* __restrict__ val, u64 n,
                                                                          u32* __restrict__ out) {
    extern __shared__ __align__(16) u32 bs_slot[];   // 2^kBucketHalfBits values
    const u64 b0 = u64(blockIdx.x) << kBucketBits;
    const u32 cnt = u32(min(u64(1) << kBucketBits, n - b0));
    const u32* __restrict__ pi = idx + b0;
    const u32* __restrict__ pv = val + b0;
    const u32 tid = threadIdx.x;
    for (u32 half = 0; half < 2; ++half) {
        const u32 lo = half << kBucketHalfBits;
        if (lo >= cnt) break;
#pragma unroll 4
        for (u32 i = tid * 4; i < cnt; i += kBucketThreads * 4) {
            if (i + 4 <= cnt) {
                const uint4 p = *reinterpret_cast<const uint4*>(pi + i);
                const uint4 v = *reinterpret_cast<const uint4*>(pv + i);
                const u32 m = (1u << kBucketHalfBits) - 1u;
                if (((p.x >> kBucketHalfBits) & 1u) == half) bs_slot[p.x & m] = v.x;
                if (((p.y >> kBucketHalfBits) & 1u) == half) bs_slot[p.y & m] = v.y;
                if (((p.z >> kBucketHalfBits) & 1u) == half) bs_slot[p.z & m] = v.z;
                if (((p.w >> kBucketHalfBits) & 1u) == half) bs_slot[p.w & m] = v.w;
            } else {
                for (u32 j = i; j < cnt; ++j) {
                    const u32 p = pi[j];
                    if (((p >> kBucketHalfBits) & 1u) == half) bs_slot[p & ((1u << kBucketHalfBits) - 1u)] = pv[j];
                }
            }
        }
        __syncthreads();
        const u32 m = min(1u << kBucketHalfBits, cnt - lo);
        u32* __restrict__ po = out + b0 + lo;
        for (u32 i = tid * 4; i < m; i += kBucketThreads * 4) {
            if (i + 4 <= m) *reinterpret_cast<uint4*>(po + i) = *reinterpret_cast<const uint4*>(bs_slot + i);
            else for (u32 j = i; j < m; ++j) po[j] = bs_slot[j];
        }
        __syncthreads();
    }
}

// ---- non-stable partition of (idx, val) pairs by an 8-bit digit of idx, optionally inside regions of `rt` tiles ----
// Table row of (tile, digit): regions are laid out one after the other, digit-major inside a region, so one exclusive scan
// of the whole table yields global offsets in (region, digit, tile) order. rt = number of tiles: one region, plain digit-major.
constexpr int kPtThreads = 512;
constexpr int kPtItems = 8;
constexpr int kPtTile = kPtThreads * kPtItems;

__device__ __forceinline__ u64 pt_row(u64 tile, u32 d, u64 rt) { return ((tile / rt) * 256 + d) * rt + tile % rt; }

__global__ void __launch_bounds__(kPtThreads) pt_hist_kernel(const u32* __restrict__ idx, u64 n, int shift, u32* __restrict__ hist, u64 rt) {
    __shared__ u32 h[256];
    if (threadIdx.x < 256) h[threadIdx.x] = 0;
    __syncthreads();
    const u64 base = u64(blockIdx.x) * kPtTile;
    const u32 cnt = u32(min(u64(kPtTile), n - base));
    u32 k[kPtItems];
#pragma unroll
    for (int j = 0; j < kPtItems; ++j) { const u32 li = j * kPtThreads + threadIdx.x; if (li < cnt) k[j] = idx[base + li]; }
#pragma unroll
    for (int j = 0; j < kPtItems; ++j) { const u32 li = j * kPtThreads + threadIdx.x; if (li < cnt) atomicAdd(&h[(k[j] >> shift) & 255u], 1u); }
    __syncthreads();
    if (threadIdx.x < 256) hist[pt_row(blockIdx.x, threadIdx.x, rt)] = h[threadIdx.x];
}

// Three blocks per SM (42 registers): the kernel is a chain of short phases between barriers and runs at the speed at
// which other blocks fill the waits (profiles/r2_launches_c4_v1.summary.txt: 18 ms per pass over 3.09 G pairs at two).
__global__ void __launch_bounds__(kPtThreads, 3) pt_scatter_kernel(const u32* __restrict__ idx, const u32* __restrict__ val, u64 n, int shift,
                                                                  const u32* __restrict__ offs, u64 rt, u32* __restrict__ oidx,
                                                                  u32* __restrict__ oval) {
    __shared__ u32 cnt_d[256], tile_off[256], delta[256];
    __shared__ __align__(16) u32 si[kPtTile], sv[kPtTile];
    const u32 tid = threadIdx.x, lane = tid & 31u;
    const u64 base = u64(blockIdx.x) * kPtTile;
    const u32 cnt = u32(min(u64(kPtTile), n - base));
    u32 k[kPtItems], slot[kPtItems];
#pragma unroll
    for (int j = 0; j < kPtItems; ++j) {   // the tile's loads are in flight while the counters are cleared
        const u32 li = j * kPtThreads + tid;
        k[j] = li < cnt ? idx[base + li] : 0u;
    }
    if (tid < 256) cnt_d[tid] = 0;
    __syncthreads();
#pragma unroll
    for (int j = 0; j < kPtItems; ++j) {
        const u32 li = j * kPtThreads + tid;
        if (li < cnt) slot[j] = atomicAdd(&cnt_d[(k[j] >> shift) & 255u], 1u);
    }
    __syncthreads();
    if (tid < 32) {   // exclusive scan of the 256 digit counts: 8 per lane + warp scan
        u32 c[8], ssum = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) { c[j] = cnt_d[lane * 8 + j]; ssum += c[j]; }
        u32 inc = ssum;
#pragma unroll
        for (int dd = 1; dd < 32; dd <<= 1) { const u32 o = __shfl_up_sync(0xffffffffu, inc, dd); if (lane >= u32(dd)) inc += o; }
        u32 run = inc - ssum;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const u32 d = lane * 8 + j;
            tile_off[d] = run;
            delta[d] = offs[pt_row(blockIdx.x, d, rt)] - run;
            run += c[j];
        }
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < kPtItems; ++j) {
        const u32 li = j * kPtThreads + tid;
        if (li < cnt) {
            const u32 lp = tile_off[(k[j] >> shift) & 255u] + slot[j];
            si[lp] = k[j];
            sv[lp] = val[base + li];   // read here, not kept through the ranking: registers for a third block
        }
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < kPtItems; ++j) {
        const u32 lp = j * kPtThreads + tid;
        if (lp < cnt) {
            const u32 kk = si[lp];
            const u32 gp = delta[(kk >> shift) & 255u] + lp;
            oidx[gp] = kk;
            oval[gp] = sv[lp];
        }
    }
}

// one partition pass; `region_elems` = 0: the whole array is one region, else regions of that many elements (a multiple
// of the tile) that the previous pass has made contiguous
inline void partition_pass(const u32* idx, const u32* val, u64 n, int shift, u64 region_elems, u32* oidx, u32* oval, DevBuf<u32>& hist,
                           DevBuf<u32>& offs, cudaStream_t stream) {
    const u64 tiles = ceil_div(n, u64(kPtTile));
    const u64 rt = region_elems ? region_elems / kPtTile : tiles;
    const u64 table = ceil_div(tiles, rt) * 256 * rt;
    hist.alloc(table, stream);
    offs.alloc(table, stream);
    if (region_elems) hist.zero();    // rows of tiles the last region does not have
    pt_hist_kernel<<<unsigned(tiles), kPtThreads, 0, stream>>>(idx, n, shift, hist.p, rt);
    KERNEL_CHECK();
    const u32* hp = hist.p;
    u32* op = offs.p;
    device_scan<u32, SumOp>([hp] __device__(u64 i) { return hp[i]; }, [op] __device__(u64 i, u32 exc, u32) { op[i] = exc; }, table,
                            (u32*)nullptr, stream);
    pt_scatter_kernel<<<unsigned(tiles), kPtThreads, 0, stream>>>(idx, val, n, shift, offs.p, rt, oidx, oval);
    KERNEL_CHECK();
    count_launch(2);
}

// out[idx[i]] = val[i] for idx a permutation of [0, n), n < 2^32. ws_a and ws_b hold 2 * (n + 4) u32 each; `val` may be
// overwritten (nothing here does), idx and val are left intact. All of idx/val/out/ws_* 16-byte aligned.
inline void inverse_permutation_scatter(const u32* idx, const u32* val, u64 n, u32* out, u32* ws_a, u32* ws_b, cudaStream_t stream,
                                        FamilyTimer* timer = nullptr) {
    if (n == 0) return;
    const u64 half = (n + 3) / 4 * 4;   // the value halves stay 16-byte aligned
    const int bits = bit_width_u64(n - 1);
    const u32 *ki = idx, *vi = val;
    u32* bufs[2] = {ws_a, ws_b};
    int w = 0;
    DevBuf<u32> hist, offs;
    // most significant digit first; a digit at [24, 32) splits the pairs into regions of 2^24 targets = 2^24 pairs each
    for (int shift = bits > kBucketBits ? kBucketBits + 8 * ((bits - kBucketBits - 1) / 8) : -1; shift >= kBucketBits; shift -= 8) {
        const u64 region = (shift + 8 < bits) ? (u64(1) << (shift + 8)) : 0;
        if (timer) timer->begin();
        partition_pass(ki, vi, n, shift, region, bufs[w], bufs[w] + half, hist, offs, stream);
        if (timer) timer->end(5, n * 4 * sizeof(u32));
        ki = bufs[w]; vi = bufs[w] + half;
        w ^= 1;
    }
    static std::atomic<unsigned long long> prepared{0};   // one bit per device
    constexpr int smem = int(sizeof(u32)) << kBucketHalfBits;
    unsigned long long dev_bit = 0;
    if (device_needs_prepare(prepared, dev_bit)) {
        CUDA_CHECK(cudaFuncSetAttribute(bucket_scatter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        device_prepared(prepared, dev_bit);
    }
    if (timer) timer->begin();
    bucket_scatter_kernel<<<unsigned(ceil_div(n, u64(1) << kBucketBits)), kBucketThreads, smem, stream>>>(ki, vi, n, out);
    KERNEL_CHECK();
    count_launch();
    if (timer) timer->end(1, n * 3 * sizeof(u32));
}

// out[idx[i]] = val[i]. perm_ws_a/b (optional, see inverse_permutation_scatter) enable the sort-back path when idx is
// a permutation of [0, n) = [0, out_len).
template <typename IdxT>
void inverse_scatter(const IdxT* idx, const IdxT* val, u64 n, IdxT* out, u64 out_len, cudaStream_t stream, void* perm_ws_a = nullptr,
                     void* perm_ws_b = nullptr, FamilyTimer* timer = nullptr) {
    if (n == 0) return;
    const u64 slice = kScatterSliceBytes / sizeof(IdxT);
    u64 sweeps = ceil_div(out_len, slice);
    if constexpr (sizeof(IdxT) == 4) {
        // developer/test knob: ASGART_B200_PERM_SCATTER_MIN=<elements> moves the threshold of the sort-back path
        static const char* knob = getenv("ASGART_B200_PERM_SCATTER_MIN");
        const bool big = knob ? n >= u64(strtoull(knob, nullptr, 10)) : sweeps > u64(kSweepMax);
        if (big && perm_ws_a && perm_ws_b && n == out_len) {
            inverse_permutation_scatter(reinterpret_cast<const u32*>(idx), reinterpret_cast<const u32*>(val), n, reinterpret_cast<u32*>(out),
                                        static_cast<u32*>(perm_ws_a), static_cast<u32*>(perm_ws_b), stream, timer);
            return;
        }
    }
    if (sweeps > u64(kSweepMax)) sweeps = 1;
    const unsigned grid = unsigned(std::min<u64>(ceil_div(n, 256 * (16 / sizeof(IdxT))), u64(kNumSMs) * 16));
    for (u64 k = 0; k < sweeps; ++k) {
        const u64 lo = out_len * k / sweeps, hi = out_len * (k + 1) / sweeps;
        scatter_slice_kernel<IdxT><<<grid, 256, 0, stream>>>(idx, val, n, out, lo, hi);
        KERNEL_CHECK();
    }
    count_launch(sweeps);
}

}  // namespace ab200
