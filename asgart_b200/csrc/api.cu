// api.cu — context, orchestration of the device pipeline and the C ABI of include/asgart_b200.h.
#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include "automaton.cuh"
#include "common.cuh"
#include "dist_group.cuh"
#include "fasta_ingest.cuh"
#include "host_internal.h"
#include "sa_build.cuh"
#include "levenshtein.cuh"
#include "locate.cuh"
#include "search.cuh"

namespace ab200 {
thread_local LaunchCounter* g_launch_counter = nullptr;
thread_local HostStalls g_host_stalls;   // per thread: the members of build_index_group count their own stalls
thread_local DevicePool* g_device_pool = nullptr;

// keys: the build's sorted initial keys (keys[i] = first key_p0 symbols of suffix SA[i], key_b bits each, first symbol on
// top), kept for the probe search when build_index ran on one device with lazy ranks; key_map = strand code (CODE_*) ->
// key code, one nibble each (0xF: the symbol does not occur in the strand)
struct Index32 { DevBuf<u32> sa, lut_lo, lut_hi, deep; int deep_depth = 0; DevBuf<u64> keys; int key_b = 0, key_p0 = 0; u64 key_map = 0; };
struct Index64 { DevBuf<u64> sa, lut_lo, lut_hi, deep; int deep_depth = 0; DevBuf<u64> keys; int key_b = 0, key_p0 = 0; u64 key_map = 0; };

struct ChunkPlan {
    std::vector<ChunkDev> host;
    DevBuf<ChunkDev> dev;
    u64 total_probes = 0;
    u32 k = 0, s = 0;
    int mode = PACK_DIRECT;
    AutoParams ap{};
};

struct StageA {
    u64 p_begin = 0, p_end = 0, n_events = 0, n_matches = 0;
    DevBuf<u32> bits;
    DevBuf<u64> ev_probe, ev_moff, matches;
    DevBuf<u32> ev_cnt;
};
}  // namespace ab200

using namespace ab200;

struct asgart_b200_partial {
    u64 p_begin = 0, p_end = 0;
    std::vector<u32> bits;
    std::vector<u64> ev_probe;
    std::vector<u32> ev_cnt;
    std::vector<u64> matches;
};

struct asgart_b200_ctx {
    DevicePool pool;   // first member: destroyed last, after every buffer that came from it
    int device = 0;
    cudaStream_t stream = nullptr;
    std::string err;
    u64 n1 = 0;
    u64 sa_len = 0;    // entries of the suffix array: n1, or b - a + 1 for an index built with --trim (a, b)
    bool have_strand = false, have_index = false;
    int want_bits = 0, idx_bits = 0;
    DevBuf<u8> d_text;
    DevBuf<u64> d_pt, d_pn;
    DevBuf<u8> shard_blob;   // device-resident partial of the last search_shard_dev call
    int pn_mode = -1;
    Index32 ix32;
    Index64 ix64;
    asgart_b200_stats st{};
    FamilyTimer t_sort, t_gather, t_rank, t_probe, t_emit, t_scatter, t_scatter_main, t_msd0, t_msd_hist, t_msd_local;
    cudaEvent_t ev_a = nullptr, ev_b = nullptr;
    LaunchCounter launches;
    // sharded index build: the group this context is a member of (null: builds alone) and this member's slice of the
    // block-cyclic rank array, kept between builds so that the peers' mappings of it stay valid
    SaGroup* group = nullptr;
    bool group_owned = false;
    void* rank_slice = nullptr;
    size_t rank_slice_bytes = 0;
    std::vector<void*> retired_slices;
    // GPU-side FASTA ingest: one piece per file between ingest_begin and ingest_finish; pinned staging for ingest_file
    bool ingesting = false;
    std::vector<IngestPiece> pieces;
    u8* stage[2] = {nullptr, nullptr};
    cudaEvent_t stage_ev[2] = {nullptr, nullptr};
    // ctx_locate: its kernels' device time, pinned staging of its copies
    FamilyTimer t_locate;
    u64 n_probe_keys = 0;   // asgart_b200_ctx_probe_keys
    u8* loc_stage = nullptr;
};

struct asgart_b200_hits {
    std::vector<int64_t> first, count;
    std::vector<uint64_t> offsets;
    std::vector<int64_t> positions;
};

namespace ab200 { namespace detail {

const u64 kPartialMagic = 0x4132303050415254ull;  // "A200PART"

struct ApiGuard {
    asgart_b200_ctx* c;
    explicit ApiGuard(asgart_b200_ctx* ctx) : c(ctx) {
        CUDA_CHECK(cudaSetDevice(ctx->device));   // may throw: the thread-locals are only set once nothing can fail any more
        g_launch_counter = &ctx->launches;
        g_device_pool = &ctx->pool;
    }
    ~ApiGuard() { g_launch_counter = nullptr; g_device_pool = nullptr; }
};

template <typename F>
int32_t guarded(asgart_b200_ctx* ctx, F f) {
    if (!ctx) return ASGART_B200_EINVAL;
    try {
        ApiGuard g(ctx);
        return f();
    } catch (const CudaError& e) {
        ctx->err = e.what();
        cudaGetLastError();
        return e.code;
    } catch (const std::bad_alloc&) {
        ctx->err = "host allocation failed";
        return ASGART_B200_ENOMEM;
    } catch (const std::exception& e) {
        ctx->err = e.what();
        return ASGART_B200_ECUDA;
    }
}

int fail(asgart_b200_ctx* ctx, int code, const char* msg) {
    ctx->err = msg;
    return code;
}

u64 packed_words(u64 n1) { return ceil_div(n1, 16) + 4; }

void pack_image(asgart_b200_ctx* ctx, int mode, DevBuf<u64>& out, u32* d_err) {
    const u64 words = packed_words(ctx->n1);
    out.alloc(words, ctx->stream);
    pack_text_kernel<<<unsigned(ceil_div(words, 256)), 256, 0, ctx->stream>>>(ctx->d_text.p, ctx->n1, mode, out.p, words, d_err);
    KERNEL_CHECK();
    count_launch();
}

// validation + 4-bit packing of the strand in ctx->d_text (n1 bytes): the tail of load_strand and of ingest_finish
int32_t pack_loaded_strand(asgart_b200_ctx* ctx) {
    EventTimer tp(ctx->stream);
    tp.start();
    DevBuf<u32> d_err(1, ctx->stream);
    d_err.zero();
    pack_image(ctx, PACK_DIRECT, ctx->d_pt, d_err.p);
    tp.stop();
    u32 h_err = 0;
    CUDA_CHECK(cudaMemcpyAsync(&h_err, d_err.p, sizeof h_err, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    ctx->st.ms_pack += tp.ms();
    if (h_err) return fail(ctx, ASGART_B200_EINVAL, "strand is not normalised: expected bytes in {A,C,G,N,T} followed by one '$'");
    ctx->have_strand = true;
    return ASGART_B200_OK;
}

void ingest_piece(asgart_b200_ctx* ctx, const u8* d_file, u64 n, bool skip_masked, IngestPiece& piece) {
    EventTimer t(ctx->stream);
    t.start();
    ingest_fasta_device(d_file, n, skip_masked, piece, ctx->stream);
    t.stop();
    ctx->st.ms_ingest += t.ms();
    ctx->st.ingest_bytes += n;
    ctx->st.ingest_records += piece.rec_off.size();
}

// Record ids (header up to the first white space) straight from the file bytes, after the bio reader's end-of-records rule
// (fasta_core.h). fetch(at, buf, cap) -> number of bytes copied from file offset `at` (0 at the end of the file).
template <class Fetch>
void ingest_record_ids(IngestPiece& piece, u64 n, Fetch fetch) {
    auto header = [&](u64 off, bool whole_line, std::string* id) {   // whole_line: is the header blank; else: collect the id
        char buf[256];
        for (u64 at = off + 1; at < n;) {
            const size_t r = fetch(at, buf, sizeof buf);
            if (!r) break;
            for (size_t i = 0; i < r; ++i) {
                const u8 c = u8(buf[i]);
                if (c == '\n') return true;
                if (!fa_space(c)) { if (whole_line) return false; id->push_back(char(c)); }
                else if (!whole_line) return true;
            }
            at += r;
        }
        return true;
    };
    stop_at_empty_record(piece.rec_off, piece.rec_pos, piece.kept, [&](size_t r) { return header(piece.rec_off[r], true, nullptr); });
    for (u64 off : piece.rec_off) {
        std::string id;
        header(off, false, &id);
        piece.names.push_back(std::move(id));
    }
}

template <typename IdxT> struct IxOf;
template <> struct IxOf<u32> { static Index32& get(asgart_b200_ctx* c) { return c->ix32; } };
template <> struct IxOf<u64> { static Index64& get(asgart_b200_ctx* c) { return c->ix64; } };

// the sorted keys describe the strand and the index they were built with: a new strand, a new index or another index
// width makes them stale
void drop_sorted_keys(asgart_b200_ctx* ctx) { ctx->ix32.keys.release(); ctx->ix64.keys.release(); }

int pick_bits(const asgart_b200_ctx* ctx) {
    if (ctx->want_bits == 32 || ctx->want_bits == 64) return ctx->want_bits;
    return (ctx->n1 < 0xFFFFFFFEull) ? 32 : 64;
}

// LUT from the finished suffix array (used when the index is uploaded, or the initial keys were shorter than 8 symbols)
template <typename IdxT>
void build_lut(asgart_b200_ctx* ctx) {
    auto& ix = IxOf<IdxT>::get(ctx);
    ix.lut_lo.alloc(kLutSize, ctx->stream);
    ix.lut_hi.alloc(kLutSize, ctx->stream);
    ix.lut_lo.zero();
    ix.lut_hi.zero();
    ix.deep.release();
    ix.deep_depth = 0;
    ix.keys.release();
    lut_build_kernel<IdxT><<<unsigned(ceil_div(ctx->n1, 256)), 256, 0, ctx->stream>>>(ctx->d_pt.p, ix.sa.p, ctx->n1, ix.lut_lo.p,
                                                                                      ix.lut_hi.p);
    KERNEL_CHECK();
    count_launch();
}

// 8-mer LUT and deep table as by-products of the suffix-array build's sorted initial keys
template <typename IdxT>
struct LutHook : SaKeyHook {
    asgart_b200_ctx* ctx;
    bool done = false;
    double ms = 0;
    u64 m4 = 0, m5 = 0;
    explicit LutHook(asgart_b200_ctx* c) : ctx(c) {}
    bool lookup_tables(SaLookupTables& t) override {
        if (!done) return false;
        auto& ix = IxOf<IdxT>::get(ctx);
        t.deep = ix.deep.p; t.depth = ix.deep_depth; t.lut_lo = ix.lut_lo.p; t.lut_hi = ix.lut_hi.p; t.m4 = m4; t.m5 = m5;
        return ix.deep.p != nullptr;
    }
    void adopt_sorted_keys(DevBuf<u64>& keys) override {
        if (done) IxOf<IdxT>::get(ctx).keys = std::move(keys);
    }
    void on_sorted_keys(const u64* d_keys, u64 n_local, u64 base, u64 n, int b, int p0, const uint16_t* h_code, cudaStream_t stream,
                        SaGroup* grp) override {
        if (p0 < 8 || n != ctx->n1) return;
        auto& ix = IxOf<IdxT>::get(ctx);
        EventTimer t(stream);
        t.start();
        LutCodeMap map;
        memset(&map, 255, sizeof map);
        const char* s5 = "ACGNT";
        const char* s4 = "ACGT";
        for (int d = 0; d < 5; ++d) if (h_code[u8(s5[d])] && h_code[u8(s5[d])] < 16) map.d5[h_code[u8(s5[d])]] = u8(d);
        for (int d = 0; d < 4; ++d) if (h_code[u8(s4[d])] && h_code[u8(s4[d])] < 16) map.d4[h_code[u8(s4[d])]] = u8(d);
        m4 = map.nibbles(map.d4); m5 = map.nibbles(map.d5);
        ix.key_b = b; ix.key_p0 = p0; ix.key_map = ~u64(0);
        for (const char* c = "$ACGNT"; *c; ++c) {
            const u32 code = code_of_byte(u8(*c)), dense = h_code[u8(*c)];
            if (dense && dense < 16) ix.key_map = (ix.key_map & ~(u64(15) << (4 * code))) | (u64(dense) << (4 * code));
        }
        // depth: buckets of a few suffixes (4^depth <= n), inside the initial key, at most kMaxDepth symbols: 4^15 + 1 slots
        // still fit u32 slot arithmetic (4 GiB of u32 starts), and a 3.1 Gbp strand leaves ~3 suffixes per bucket, which one
        // round of parallel loads compares instead of a bisection
        constexpr int kMaxDepth = 15;
        int depth = 0;
        while (depth < kMaxDepth && depth < p0 && (u64(1) << (2 * (depth + 1))) <= n) ++depth;
        if (depth < 4) depth = 0;
        ix.lut_lo.alloc(kLutSize, stream);
        ix.lut_hi.alloc(kLutSize, stream);
        ix.lut_lo.zero();
        ix.lut_hi.zero();
        const u64 M = depth ? (u64(1) << (2 * depth)) + 1 : 0;
        ix.deep.alloc(M, stream);
        ix.deep.zero();
        ix.deep_depth = depth;
        // 3-bit codes (DNA): the deep slot is decoded four symbols per lookup through a 4096-entry table
        DevBuf<uint16_t> tab4;
        u32 pad4 = 0;
        if (b == 3 && depth > 0) {
            std::vector<uint16_t> h_tab(4096);
            for (u32 g = 0; g < 4096; ++g) {
                u32 e = 0;
                for (int q = 0; q < 4; ++q) {
                    const u8 d = map.d4[(g >> (3 * (3 - q))) & 7u];
                    if (d == 255) e |= 0x8000u; else e |= u32(d) << (2 * (3 - q));
                }
                h_tab[g] = uint16_t(e);
            }
            u32 ok_code = 8;
            for (u32 c = 0; c < 8; ++c) if (map.d4[c] != 255) { ok_code = c; break; }
            if (ok_code < 8) {
                pad4 = ok_code | (ok_code << 3) | (ok_code << 6);
                tab4.alloc(4096, stream);
                CUDA_CHECK(cudaMemcpyAsync(tab4.p, h_tab.data(), 4096 * sizeof(uint16_t), cudaMemcpyHostToDevice, stream));
                CUDA_CHECK(cudaStreamSynchronize(stream));   // h_tab goes out of scope
            }
        }
        if (n_local) {
            lut_from_keys_kernel<IdxT><<<unsigned(ceil_div(n_local, 256 * 4)), 256, 0, stream>>>(d_keys, n_local, base, b, p0, map.nibbles(map.d5),
                                                                                                map.nibbles(map.d4), depth, tab4.p, pad4,
                                                                                                ix.lut_lo.p, ix.lut_hi.p, ix.deep.p);
            KERNEL_CHECK();
            count_launch();
        }
        if (grp) {
            // every slot was seen by exactly one member (zero elsewhere; slot values are >= 1): the maximum merges the tables
            grp->allreduce_max_dev(ix.lut_lo.p, kLutSize, int(sizeof(IdxT)), stream);
            grp->allreduce_max_dev(ix.lut_hi.p, kLutSize, int(sizeof(IdxT)), stream);
            if (depth && b == 3 && p0 >= 4) {
                // The members' key ranges are cut where the first four symbols change, so each member's keys fill one
                // contiguous range of deep slots: exchange those pieces (4 GiB / world each at 3.1 Gbp) instead of
                // all-reducing the whole table. Member r's piece starts at the slot of its first key's 4-symbol prefix
                // (slots before it that no key hits belong to nobody and stay 0 everywhere).
                u64 first_key = 0;
                if (n_local) {
                    CUDA_CHECK(cudaMemcpyAsync(&first_key, d_keys, sizeof(u64), cudaMemcpyDeviceToHost, stream));
                    CUDA_CHECK(cudaStreamSynchronize(stream));
                }
                std::vector<u64> lo(size_t(grp->world), 0);
                if (n_local) {
                    const u32 bin = u32(first_key >> (3 * (p0 - 4))) & 4095u;
                    u64 f = 0;   // base-4 value of the smallest all-ACGT 4-mer >= bin's 4 symbols = number of all-ACGT bins below `bin`
                    for (u32 g2 = 0; g2 < bin; ++g2) {
                        bool ok = true;
                        for (int q = 0; q < 4; ++q) ok = ok && map.d4[(g2 >> (3 * q)) & 7u] != 255;
                        f += ok ? 1 : 0;
                    }
                    lo[size_t(grp->rank)] = (f << (2 * (depth - 4))) + 1;   // + 1: 0 = this member has no keys
                }
                CUDA_CHECK(cudaStreamSynchronize(stream));
                grp->allreduce_sum_host(lo.data(), grp->world);
                std::vector<u64> offs(size_t(grp->world) + 1, 0);
                offs[size_t(grp->world)] = M - 1;
                for (int r = grp->world - 1; r >= 0; --r) offs[size_t(r)] = lo[size_t(r)] ? std::min<u64>(lo[size_t(r)] - 1, offs[size_t(r) + 1]) : offs[size_t(r) + 1];
                offs[0] = 0;
                grp->share_pieces(ix.deep.p, offs.data(), int(sizeof(IdxT)), stream);
            } else if (depth) {
                grp->allreduce_max_dev(ix.deep.p, M, int(sizeof(IdxT)), stream);
            }
        }
        if (depth) {
            // unseen slots take the start of the next seen one (empty bucket); the last entry closes the table at n1
            IdxT* dp = ix.deep.p;
            const IdxT n1v = IdxT(n);
            CUDA_CHECK(cudaMemcpyAsync(dp + (M - 1), &n1v, sizeof(IdxT), cudaMemcpyHostToDevice, stream));
            // short empty runs (the rule in a genome-sized table) in one pass; a run past the look-ahead leaves the rest to the scan
            u32 h_over = 0;
            {
                DevBuf<u32> d_over(1, stream);
                d_over.zero();
                deep_fill_kernel<IdxT><<<kNumSMs * 16, 256, 0, stream>>>(dp, M, d_over.p);
                KERNEL_CHECK();
                count_launch();
                CUDA_CHECK(cudaMemcpyAsync(&h_over, d_over.p, sizeof h_over, cudaMemcpyDeviceToHost, stream));
                CUDA_CHECK(cudaStreamSynchronize(stream));
            }
            if (h_over)
            device_scan<IdxT, MaxOp>([dp, M, n1v] __device__(u64 kx) { const IdxT v = dp[M - 1 - kx]; return v ? IdxT(n1v + 1 - v) : IdxT(0); },
                                     [dp, M, n1v] __device__(u64 kx, IdxT, IdxT inc) { dp[M - 1 - kx] = inc ? IdxT(n1v + 1 - inc) : n1v; }, M,
                                     (IdxT*)nullptr, stream);
        }
        t.stop();
        ms = t.ms();
        done = true;
    }
};

template <typename IdxT>
void build_index_t(asgart_b200_ctx* ctx) {
    NvtxRange nv("build_index");
    auto& ix = IxOf<IdxT>::get(ctx);
    ix.keys.release();   // before the sort allocates its key buffers: they take this block again
    EventTimer tsa(ctx->stream), tlut(ctx->stream);
    tsa.start();
    ix.sa.alloc(ctx->n1, ctx->stream);
    LutHook<IdxT> hook(ctx);
    SaStats ss;
    ss.sort = &ctx->t_sort; ss.gather = &ctx->t_gather; ss.rank = &ctx->t_rank; ss.scatter = &ctx->t_scatter; ss.scatter_main = &ctx->t_scatter_main;
    ss.msd.scatter = &ctx->t_scatter_main; ss.msd.scatter0 = &ctx->t_msd0; ss.msd.hist = &ctx->t_msd_hist; ss.msd.local = &ctx->t_msd_local;
    SaGroup* grp = (ctx->group && ctx->group->world > 1) ? ctx->group : nullptr;
    if (!grp) {
        DevBuf<IdxT> rank(ctx->n1, ctx->stream);
        build_suffix_array<IdxT>(ctx->d_text.p, ctx->n1, ix.sa.p, rank.p, ctx->stream, &ss, &hook);
    } else {
        // this member's slice of the rank array: a cudaMalloc block of its own (its address is what the peers map)
        RankView<IdxT> rv;
        rv.world = u32(grp->world);
        rv.g = RankView<IdxT>::pick_g(ctx->n1);
        rv.k = RankView<IdxT>::pick_k(ctx->n1, rv.world, rv.g);
        const size_t need = rv.slice_len() * sizeof(IdxT);
        if (need > ctx->rank_slice_bytes) {   // same decision on every member: n1 and world are the same everywhere
            // the previous build ended with a collective, so nobody still works on the old slice; peers may still have it
            // mapped (CUDA IPC), so it is only freed with the context
            if (ctx->rank_slice) ctx->retired_slices.push_back(ctx->rank_slice);
            ctx->rank_slice = nullptr; ctx->rank_slice_bytes = 0;
            CUDA_CHECK(cudaMalloc(&ctx->rank_slice, need));
            ctx->rank_slice_bytes = need;
        }
        void* all[kMaxWorld] = {};
        grp->exchange_ptr(ctx->rank_slice, ctx->rank_slice_bytes, all);
        for (int r = 0; r < kMaxWorld; ++r) rv.base[r] = static_cast<IdxT*>(all[r < grp->world ? r : 0]);
        build_suffix_array<IdxT>(ctx->d_text.p, ctx->n1, ix.sa.p, rv, ctx->stream, &ss, &hook, grp);
    }
    ctx->st.sa_rounds = ss.rounds;
    ctx->st.msd_levels = ss.used_msd ? u64(ss.msd.levels) : 0;
    tsa.stop();
    tlut.start();
    if (!hook.done) build_lut<IdxT>(ctx);
    tlut.stop();
    ctx->st.ms_sa_build += tsa.ms() - hook.ms;
    ctx->st.ms_lut += tlut.ms() + hook.ms;
}

template <typename IdxT>
void build_index_trim_t(asgart_b200_ctx* ctx, u64 a, u64 b) {
    auto& ix = IxOf<IdxT>::get(ctx);
    ix.keys.release();
    cudaStream_t s = ctx->stream;
    EventTimer tsa(s), tlut(s);
    tsa.start();
    const u64 m1 = b - a + 1;
    DevBuf<u8> sub(m1, s);
    CUDA_CHECK(cudaMemcpyAsync(sub.p, ctx->d_text.p + a, b - a, cudaMemcpyDeviceToDevice, s));
    CUDA_CHECK(cudaMemsetAsync(sub.p + (b - a), '$', 1, s));
    ix.sa.alloc(m1, s);
    SaStats ss;
    ss.sort = &ctx->t_sort; ss.gather = &ctx->t_gather; ss.rank = &ctx->t_rank; ss.scatter = &ctx->t_scatter; ss.scatter_main = &ctx->t_scatter_main;
    ss.msd.scatter = &ctx->t_scatter_main; ss.msd.scatter0 = &ctx->t_msd0; ss.msd.hist = &ctx->t_msd_hist; ss.msd.local = &ctx->t_msd_local;
    {
        DevBuf<IdxT> rank(m1, s);
        build_suffix_array<IdxT>(sub.p, m1, ix.sa.p, rank.p, s, &ss, nullptr);
    }
    if (a) {
        add_offset_kernel<IdxT><<<unsigned(std::min<u64>(ceil_div(m1, 256), u64(kNumSMs) * 16)), 256, 0, s>>>(ix.sa.p, m1, IdxT(a));
        KERNEL_CHECK();
        count_launch();
    }
    ctx->st.sa_rounds = ss.rounds;
    tsa.stop();
    tlut.start();
    ix.lut_lo.alloc(kLutSize, s);
    ix.lut_hi.alloc(kLutSize, s);
    ix.deep.release();
    ix.deep_depth = 0;
    lut_literal_kernel<IdxT><<<unsigned(ceil_div(kLutSize, 128)), 128, 0, s>>>(ctx->d_text.p, ctx->n1, ix.sa.p, m1, ix.lut_lo.p, ix.lut_hi.p);
    KERNEL_CHECK();
    count_launch();
    tlut.stop();
    ctx->st.ms_sa_build += tsa.ms();
    ctx->st.ms_lut += tlut.ms();
}

template <typename T>
__global__ void widen_to_i64_kernel(const T* __restrict__ in, i64* __restrict__ out, u64 n) {
    const u64 i = u64(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) out[i] = i64(in[i]);
}
template <typename T>
__global__ void narrow_from_i64_kernel(const i64* __restrict__ in, T* __restrict__ out, u64 n) {
    const u64 i = u64(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i < n) out[i] = T(in[i]);
}

template <typename T>
void download_as_i64(const T* d, i64* h, u64 n, cudaStream_t s) {
    const u64 chunk = u64(1) << 26;
    DevBuf<i64> stage(std::min(n, chunk), s);
    for (u64 o = 0; o < n; o += chunk) {
        const u64 m = std::min(chunk, n - o);
        widen_to_i64_kernel<T><<<unsigned(ceil_div(m, 256)), 256, 0, s>>>(d + o, stage.p, m);
        KERNEL_CHECK();
        count_launch();
        CUDA_CHECK(cudaMemcpyAsync(h + o, stage.p, m * sizeof(i64), cudaMemcpyDeviceToHost, s));
        CUDA_CHECK(cudaStreamSynchronize(s));
    }
}
template <typename T>
void upload_from_i64(const i64* h, T* d, u64 n, cudaStream_t s) {
    const u64 chunk = u64(1) << 26;
    DevBuf<i64> stage(std::min(n, chunk), s);
    for (u64 o = 0; o < n; o += chunk) {
        const u64 m = std::min(chunk, n - o);
        CUDA_CHECK(cudaMemcpyAsync(stage.p, h + o, m * sizeof(i64), cudaMemcpyHostToDevice, s));
        narrow_from_i64_kernel<T><<<unsigned(ceil_div(m, 256)), 256, 0, s>>>(stage.p, d + o, m);
        KERNEL_CHECK();
        count_launch();
        CUDA_CHECK(cudaStreamSynchronize(s));
    }
}

template <typename IdxT>
i64 check_sa_t(asgart_b200_ctx* ctx) {
    auto& ix = IxOf<IdxT>::get(ctx);
    const u64 n1 = ctx->n1;
    cudaStream_t s = ctx->stream;
    DevBuf<IdxT> isa(n1, s);
    DevBuf<unsigned long long> bad(1, s);
    bad.zero();
    CUDA_CHECK(cudaMemsetAsync(isa.p, 0xFF, n1 * sizeof(IdxT), s));
    const IdxT* sa = ix.sa.p;
    IdxT* ip = isa.p;
    unsigned long long* bp = bad.p;
    const u8* text = ctx->d_text.p;
    for_each_index(n1, [=] __device__(u64 i) { const u64 x = u64(sa[i]); if (x < n1) ip[x] = IdxT(i); else atomicAdd(bp, 1ull); }, s);
    for_each_index(n1, [=] __device__(u64 p) { const u64 r = u64(ip[p]); if (r >= n1 || u64(sa[r]) != p) atomicAdd(bp, 1ull); }, s);
    for_each_index(n1, [=] __device__(u64 i) {
        if (i == 0) return;
        const u64 a = u64(sa[i - 1]), b = u64(sa[i]);
        if (a >= n1 || b >= n1) return;  // counted above
        const u8 ca = text[a], cb = text[b];
        bool ok;
        if (ca != cb) ok = ca < cb;
        else if (a + 1 == n1) ok = true;    // the shorter suffix is a proper prefix of the other
        else if (b + 1 == n1) ok = false;
        else ok = u64(ip[a + 1]) < u64(ip[b + 1]);
        if (!ok) atomicAdd(bp, 1ull);
    }, s);
    unsigned long long h = 0;
    CUDA_CHECK(cudaMemcpyAsync(&h, bad.p, sizeof h, cudaMemcpyDeviceToHost, s));
    CUDA_CHECK(cudaStreamSynchronize(s));
    return i64(h);
}

// order-sensitive 64-bit fingerprint of the index: sum over i of splitmix64(SA[i] + i * 0x9E3779B97F4A7C15) mod 2^64
__device__ __forceinline__ u64 fp_mix(u64 z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
template <typename IdxT>
__global__ void __launch_bounds__(256) sa_fingerprint_kernel(const IdxT* __restrict__ sa, u64 n, unsigned long long* __restrict__ out) {
    u64 acc = 0;
    const u64 stride = u64(gridDim.x) * blockDim.x;
    for (u64 i = u64(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += stride) acc += fp_mix(u64(sa[i]) + i * 0x9E3779B97F4A7C15ull);
#pragma unroll
    for (int d = 16; d; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
    if ((threadIdx.x & 31u) == 0) atomicAdd(out, (unsigned long long)acc);
}
template <typename IdxT>
u64 sa_fingerprint_t(asgart_b200_ctx* ctx) {
    auto& ix = IxOf<IdxT>::get(ctx);
    cudaStream_t s = ctx->stream;
    DevBuf<unsigned long long> acc(1, s);
    acc.zero();
    const unsigned grid = unsigned(std::min<u64>(ceil_div(ctx->sa_len, 256), u64(kNumSMs) * 16));
    sa_fingerprint_kernel<IdxT><<<grid, 256, 0, s>>>(ix.sa.p, ctx->sa_len, acc.p);
    KERNEL_CHECK();
    count_launch();
    unsigned long long h = 0;
    CUDA_CHECK(cudaMemcpyAsync(&h, acc.p, sizeof h, cudaMemcpyDeviceToHost, s));
    CUDA_CHECK(cudaStreamSynchronize(s));
    return u64(h);
}

// ---------------------------------------------------------------------------------------------- chunk plan
int make_plan(asgart_b200_ctx* ctx, const asgart_b200_chunk* chunks, i64 n_chunks, const asgart_b200_settings* st, ChunkPlan& plan) {
    if (!chunks || n_chunks < 0 || !st) return fail(ctx, ASGART_B200_EINVAL, "null chunks/settings");
    if (st->probe_size < 8) return fail(ctx, ASGART_B200_EINVAL, "probe_size must be >= 8 (the reference indexes the first 8 bases, src/searcher.rs:95-97)");
    if (st->probe_size > 4096) return fail(ctx, ASGART_B200_EINVAL, "probe_size > 4096 not supported");
    const u64 n = ctx->n1 - 1;
    plan.k = u32(st->probe_size);
    plan.s = u32(st->probe_size / 2);
    plan.mode = (st->reverse ? 2 : 0) | (st->complement ? 1 : 0);
    plan.host.clear();
    u64 base = 0;
    for (i64 c = 0; c < n_chunks; ++c) {
        ChunkDev d{};
        d.c0 = chunks[c].start; d.len = chunks[c].length;
        if (d.c0 > n || d.len > n - d.c0) return fail(ctx, ASGART_B200_EINVAL, "chunk outside the strand");
        d.n_probes = probes_in_chunk(d.len, plan.k, plan.s, st->min_duplication_length);
        d.probe_base = base;
        d.needle_start = st->reverse ? (n - d.c0 - d.len) : d.c0;
        base += d.n_probes;
        plan.host.push_back(d);
    }
    plan.total_probes = base;
    if (plan.host.empty()) plan.host.push_back(ChunkDev{});
    plan.dev.alloc(plan.host.size(), ctx->stream);
    CUDA_CHECK(cudaMemcpyAsync(plan.dev.p, plan.host.data(), plan.host.size() * sizeof(ChunkDev), cudaMemcpyHostToDevice, ctx->stream));
    CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
    AutoParams& ap = plan.ap;
    ap.k = plan.k; ap.s = plan.s; ap.G = st->max_gap_size; ap.min_len = st->min_duplication_length;
    const u64 q = (ap.G + ap.s - 1) / ap.s;
    ap.q_ext = std::max<u64>(1, q);
    ap.q_new = q > 0 ? q - 1 : 0;
    ap.reverse = st->reverse ? 1 : 0;
    return ASGART_B200_OK;
}

void ensure_needle(asgart_b200_ctx* ctx, int mode) {
    if (mode == PACK_DIRECT) return;
    if (ctx->pn_mode == mode && ctx->d_pn.p) return;
    DevBuf<u32> d_err(1, ctx->stream);
    d_err.zero();
    pack_image(ctx, mode, ctx->d_pn, d_err.p);
    ctx->pn_mode = mode;
}

// ---------------------------------------------------------------------------------------------- stage A
// probe_search_kernel over [p_begin, p_end) and, when the deep table is usable (k >= its depth), probe_deferred_kernel over
// the probes it left to the literal search. Reads the counters back (one sync). mode: the needle image (PackMode).
// Returns the number of probes answered from the sorted keys.
template <typename IdxT>
u64 run_probe_kernels(asgart_b200_ctx* ctx, ProbeParams<IdxT>& P, int mode, unsigned long long* h_ctr) {
    auto& ix = IxOf<IdxT>::get(ctx);
    cudaStream_t s = ctx->stream;
    const u64 np = P.p_end - P.p_begin;
    DevBuf<u32> q6(ceil_div(kLutSize, 32), s);
    DevBuf<u64> deferred;
    const bool deep = ix.deep.p && ix.deep_depth > 0 && int(P.k) >= ix.deep_depth;
    if (deep) {
        q6.zero();
        q6_mark_kernel<<<unsigned(ceil_div(P.k, 128)), 128, 0, s>>>(P.PT, P.n1, P.k, q6.p);
        KERNEL_CHECK();
        count_launch();
        deferred.alloc(np, s);
        P.deep = ix.deep.p; P.deep_depth = ix.deep_depth; P.q6_bits = q6.p; P.deferred = deferred.p;
    }
    // The deep buckets are compared in the sorted keys when the build left them, and when every symbol of the needle
    // image has a key code: the codes are those of the bytes that occur in the strand, so a strand with A but no T,
    // searched with its complement, compares on the text.
    bool keys = deep && ix.keys.p;
    const auto has_code = [&](u32 c) { return ((ix.key_map >> (4 * c)) & 15u) != 15u; };
    for (u32 c : {CODE_A, CODE_C, CODE_G, CODE_N, CODE_T})
        if (has_code(c) && !has_code((mode & PACK_COMPLEMENT) ? complement_code(c) : c)) keys = false;
    if (keys) { P.keys = ix.keys.p; P.key_b = ix.key_b; P.key_p0 = ix.key_p0; P.key_map = ix.key_map; }
    // shape of the text comparison (LINEAR = 8 suffixes compared at once, 2 blocks per SM = 128 registers) picked on B200
    // at C4 size: more blocks per SM or a shorter LINEAR are slower, the kernel is bound by random DRAM sectors
    // (profiles/r1_experiments.log). The keys comparison needs 71 (u32) / 75 (u64) registers at that shape, no spills;
    // tried on one B200 (1000 W) at C4 size, while the counters still took one atomic per warp: LINEAR 4, 8, 16 with 2, 3,
    // 4 blocks per SM all within 1 ms of each other (LINEAR 4 with 4 blocks: 44.0 ms, this shape: 44.2 ms), so it keeps
    // the text comparison's shape (22.2 ms with the per-block counters; the other shapes were not timed again).
    if (keys) probe_search_kernel<IdxT, 8, 2, true><<<unsigned(ceil_div(np, 256)), 256, 0, s>>>(P);
    else probe_search_kernel<IdxT, 8, 2, false><<<unsigned(ceil_div(np, 256)), 256, 0, s>>>(P);
    KERNEL_CHECK();
    count_launch();
    u64 n_keys = 0;
    if (deep) {
        // with the keys, every probe probe_search_kernel searched itself was answered from them (it defers all others)
        unsigned long long first[CTR_DEFERRED + 1];
        CUDA_CHECK(cudaMemcpyAsync(first, P.counters, sizeof first, cudaMemcpyDeviceToHost, s));
        CUDA_CHECK(cudaStreamSynchronize(s));
        const u64 n_def = first[CTR_DEFERRED];
        if (keys) n_keys = first[CTR_SEARCHED];
        if (n_def) {
            probe_deferred_kernel<IdxT><<<unsigned(ceil_div(n_def * 32, 256)), 256, 0, s>>>(P, n_def);
            KERNEL_CHECK();
            count_launch();
        }
    }
    CUDA_CHECK(cudaMemcpyAsync(h_ctr, P.counters, sizeof(unsigned long long) * CTR_COUNT, cudaMemcpyDeviceToHost, s));
    CUDA_CHECK(cudaStreamSynchronize(s));
    return n_keys;
}

template <typename IdxT>
void run_stage_a(asgart_b200_ctx* ctx, const ChunkPlan& plan, const asgart_b200_settings* st, u64 p_begin, u64 p_end, StageA& A) {
    NvtxRange nv("search/stage A: probe search + emit");
    auto& ix = IxOf<IdxT>::get(ctx);
    cudaStream_t s = ctx->stream;
    A.p_begin = p_begin; A.p_end = p_end;
    const u64 np = p_end - p_begin;
    const u64 words = ceil_div(np, 32);
    A.bits.alloc(words, s);
    if (np == 0) return;
    DevBuf<IdxT> out_lo(np, s), out_raw(np, s);
    DevBuf<u32> out_surv(np, s);
    DevBuf<unsigned long long> counters(CTR_COUNT, s);
    counters.zero();
    ProbeParams<IdxT> P{};
    P.PT = ctx->d_pt.p;
    P.PN = plan.mode == PACK_DIRECT ? ctx->d_pt.p : ctx->d_pn.p;
    P.SA = ix.sa.p; P.lut_lo = ix.lut_lo.p; P.lut_hi = ix.lut_hi.p;
    P.chunks = plan.dev.p; P.n_chunks = u32(plan.host.size());
    P.n1 = ctx->n1; P.k = plan.k; P.s = plan.s; P.reverse = st->reverse ? 1 : 0; P.max_card = st->max_cardinality;
    P.p_begin = p_begin; P.p_end = p_end;
    P.out_lo = out_lo.p; P.out_raw = out_raw.p; P.out_surv = out_surv.p; P.proc_bits = A.bits.p; P.counters = counters.p;
    unsigned long long h_ctr[CTR_COUNT];
    ctx->t_probe.begin();
    const u64 n_keys = run_probe_kernels<IdxT>(ctx, P, plan.mode, h_ctr);
    ctx->t_probe.end(1, h_ctr[CTR_ALG_BYTES]);
    ctx->st.n_probes += np;
    ctx->st.n_searched += h_ctr[CTR_SEARCHED];
    ctx->st.n_skipped_n += h_ctr[CTR_SKIP_N];
    ctx->st.n_skipped_card += h_ctr[CTR_SKIP_CARD];
    ctx->st.n_matches += h_ctr[CTR_MATCHES];
    ctx->n_probe_keys += n_keys;

    // match offsets + event list + emission, fused into one scan
    ctx->t_emit.begin();
    const u32* surv = out_surv.p;
    auto in = [surv] __device__(u64 o) { const u32 v = surv[o]; return Sum2(u64(v), v ? 1ull : 0ull); };
    DevBuf<Sum2> d_total(1, s);
    ScanPlan<Sum2, Sum2Op> scan;
    scan.prepare(in, np, d_total.p, s);
    Sum2 tot;
    CUDA_CHECK(cudaMemcpyAsync(&tot, d_total.p, sizeof tot, cudaMemcpyDeviceToHost, s));
    CUDA_CHECK(cudaStreamSynchronize(s));
    A.n_matches = tot.a; A.n_events = tot.b;
    A.ev_probe.alloc(A.n_events, s); A.ev_cnt.alloc(A.n_events, s); A.ev_moff.alloc(A.n_events, s);
    A.matches.alloc(A.n_matches, s);
    {
        DevBuf<IdxT> ev_lo(A.n_events, s), ev_raw(A.n_events, s);
        u64* ev_probe = A.ev_probe.p; u32* ev_cnt = A.ev_cnt.p; u64* ev_moff = A.ev_moff.p;
        IdxT* elo = ev_lo.p; IdxT* eraw = ev_raw.p;
        const IdxT* lo = out_lo.p; const IdxT* raw = out_raw.p;
        scan.finish(in, [=] __device__(u64 o, const Sum2& exc, const Sum2&) {
            const u32 v = surv[o];
            if (!v) return;
            ev_probe[exc.b] = p_begin + o; ev_cnt[exc.b] = v; ev_moff[exc.b] = exc.a;
            elo[exc.b] = lo[o]; eraw[exc.b] = raw[o];
        });
        if (A.n_events) {
            emit_matches_kernel<IdxT><<<unsigned(ceil_div(A.n_events * 32, 256)), 256, 0, s>>>(
                ix.sa.p, A.ev_probe.p, A.ev_moff.p, ev_lo.p, ev_raw.p, A.n_events, plan.dev.p, u32(plan.host.size()), plan.s,
                st->reverse ? 1 : 0, A.matches.p);
            KERNEL_CHECK();
            count_launch();
        }
    }
    ctx->t_emit.end(3, 0);
}

// ---------------------------------------------------------------------------------------------- post-steps
// d_sds / d_off are replaced by the post-processed families
void run_post(asgart_b200_ctx* ctx, DevBuf<asgart_b200_protosd>& d_sds, DevBuf<u64>& d_off, u64& n_fam, u64& n_sds, u32 post_mask) {
    NvtxRange nv("post-steps: FilterNs/ReOrder/ReduceOverlap/Sort");
    cudaStream_t s = ctx->stream;
    if (n_fam == 0 || post_mask == 0) return;
    DevBuf<u8> keep(n_sds, s);
    if (post_mask & ASGART_B200_POST_FILTER_NS) {
        DevBuf<u32> oob(1, s);
        oob.zero();
        n_content_kernel<<<unsigned(n_sds), 256, 0, s>>>(ctx->d_text.p, ctx->n1, d_sds.p, n_sds, keep.p, oob.p);
        KERNEL_CHECK();
        count_launch();
        u32 h_oob = 0;
        CUDA_CHECK(cudaMemcpyAsync(&h_oob, oob.p, sizeof h_oob, cudaMemcpyDeviceToHost, s));
        CUDA_CHECK(cudaStreamSynchronize(s));
        if (h_oob)
            throw CudaError(ASGART_B200_EPANIC, "FilterNs: an arm's inclusive range reaches past the strand; the reference panics here "
                                                "(slice index out of range, src/structs.rs:455-466)");
    }
    DevBuf<u64> new_count(n_fam, s);
    post_family_kernel<<<unsigned(ceil_div(n_fam, 64)), 64, 0, s>>>(d_sds.p, d_off.p, n_fam, keep.p, post_mask, new_count.p);
    KERNEL_CHECK();
    count_launch();
    const u64* nc = new_count.p;
    auto in = [nc] __device__(u64 f) { const u64 v = nc[f]; return Sum2(v, v ? 1ull : 0ull); };
    DevBuf<Sum2> d_total(1, s);
    ScanPlan<Sum2, Sum2Op> scan;
    scan.prepare(in, n_fam, d_total.p, s);
    Sum2 tot;
    CUDA_CHECK(cudaMemcpyAsync(&tot, d_total.p, sizeof tot, cudaMemcpyDeviceToHost, s));
    CUDA_CHECK(cudaStreamSynchronize(s));
    DevBuf<asgart_b200_protosd> out_sds(tot.a, s);
    DevBuf<u64> out_off(tot.b + 1, s);
    {
        const asgart_b200_protosd* src = d_sds.p; const u64* off = d_off.p;
        asgart_b200_protosd* dst = out_sds.p; u64* ooff = out_off.p;
        scan.finish(in, [=] __device__(u64 f, const Sum2& exc, const Sum2&) {
            const u64 v = nc[f];
            if (!v) return;
            ooff[exc.b] = exc.a;
            const u64 b = off[f];
            for (u64 r = 0; r < v; ++r) dst[exc.a + r] = src[b + r];
        });
    }
    CUDA_CHECK(cudaMemcpyAsync(out_off.p + tot.b, &tot.a, sizeof(u64), cudaMemcpyHostToDevice, s));
    CUDA_CHECK(cudaStreamSynchronize(s));
    d_sds = std::move(out_sds);
    d_off = std::move(out_off);
    n_sds = tot.a;
    n_fam = tot.b;
}

// ComputeScore (src/bin/asgart.rs:98-111): the reference runs it between ReduceOverlap and Sort; the identity of a duplicon
// depends on its own fields only and Sort only permutes, so it is computed on the final list.
void run_score(asgart_b200_ctx* ctx, DevBuf<asgart_b200_protosd>& d_sds, u64 n_sds) {
    NvtxRange nv("post-steps: ComputeScore");
    if (n_sds == 0) return;
    if (!ctx->have_strand) throw CudaError(ASGART_B200_ESTATE, "ComputeScore needs a loaded strand");
    LevStats ls;
    const int rc = compute_score(ctx->d_text.p, ctx->n1, d_sds.p, n_sds, ctx->stream, &ls);
    ctx->st.ms_score += ls.ms;
    ctx->st.score_cells += ls.cells;
    ctx->st.score_pairs += ls.pairs;
    if (rc == 1)
        throw CudaError(ASGART_B200_EPANIC, "ComputeScore: a complemented right arm ends on the '$' terminator; the reference panics here "
                                            "(\"Unknown nucleotide\", src/structs.rs:28-34)");
    if (rc == 2)
        throw CudaError(ASGART_B200_EPANIC, "ComputeScore: an arm's inclusive range reaches past the strand; the reference panics here "
                                            "(slice index out of range, src/structs.rs:441-442)");
}

void download_result(asgart_b200_ctx* ctx, const DevBuf<asgart_b200_protosd>& d_sds, const DevBuf<u64>& d_off, u64 n_fam, u64 n_sds,
                     asgart_b200_result* r) {
    r->fam_off.assign(n_fam + 1, 0);
    r->sds.resize(n_sds);
    EventTimer t(ctx->stream);
    t.start();
    if (n_fam) CUDA_CHECK(cudaMemcpyAsync(r->fam_off.data(), d_off.p, (n_fam + 1) * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    if (n_sds) CUDA_CHECK(cudaMemcpyAsync(r->sds.data(), d_sds.p, n_sds * sizeof(asgart_b200_protosd), cudaMemcpyDeviceToHost, ctx->stream));
    t.stop();
    ctx->st.ms_d2h += t.ms();
    ctx->st.d2h_bytes += (n_fam + 1) * sizeof(u64) + n_sds * sizeof(asgart_b200_protosd);
}

// ---------------------------------------------------------------------------------------------- stage B
__global__ void chunk_tc_kernel(const ChunkDev* __restrict__ chunks, u32 n_chunks, const u32* __restrict__ bits,
                                const u64* __restrict__ wpre, u64* __restrict__ tc) {
    const u32 c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_chunks) return;
    const u64 b = chunks[c].probe_base;
    tc[c] = processed_before(bits, wpre, b + chunks[c].n_probes) - processed_before(bits, wpre, b);
}

// bits: processed bitmask over all probes; events sorted by probe; ev_moff = exclusive scan of ev_cnt
void run_stage_b(asgart_b200_ctx* ctx, const ChunkPlan& plan, const asgart_b200_settings* st, const u32* d_bits, u64 n_events,
                 const u64* ev_probe, const u32* ev_cnt, const u64* ev_moff, const u64* matches, u64 n_matches, u32 post_mask,
                 asgart_b200_result* result) {
    NvtxRange nv("search/stage B: automaton + families");
    cudaStream_t s = ctx->stream;
    EventTimer tauto(s), tpost(s);
    tauto.start();
    ctx->st.n_events = n_events;
    u64 n_fam = 0, n_sds = 0;
    DevBuf<asgart_b200_protosd> d_sds;
    DevBuf<u64> d_off;
    if (n_events > 0) {
        const u64 words = ceil_div(plan.total_probes, 32);
        DevBuf<u64> wpre(words + 1, s);
        {
            u64* wp = wpre.p;
            device_scan<u64, SumOp>([d_bits] __device__(u64 w) { return u64(__popc(d_bits[w])); },
                                    [wp] __device__(u64 w, u64 exc, u64) { wp[w] = exc; }, words, wpre.p + words, s);
        }
        const u32 n_chunks = u32(plan.host.size());
        DevBuf<u64> tc(n_chunks, s);
        chunk_tc_kernel<<<ceil_div_i(n_chunks, 128), 128, 0, s>>>(plan.dev.p, n_chunks, d_bits, wpre.p, tc.p);
        KERNEL_CHECK();
        DevBuf<u64> ev_i(n_events, s), ev_t(n_events, s);
        DevBuf<u32> ev_chunk(n_events, s);
        DevBuf<u8> ev_head(n_events, s);
        event_info_kernel<<<unsigned(ceil_div(n_events, 256)), 256, 0, s>>>(ev_probe, n_events, plan.dev.p, n_chunks, d_bits, wpre.p,
                                                                          plan.s, plan.ap.q_ext, ev_i.p, ev_t.p, ev_chunk.p, ev_head.p);
        KERNEL_CHECK();
        count_launch(2);
        // segments
        const u8* hd = ev_head.p;
        auto in_seg = [hd] __device__(u64 e) { return u64(hd[e]); };
        DevBuf<u64> d_nseg(1, s);
        ScanPlan<u64, SumOp> seg_scan;
        seg_scan.prepare(in_seg, n_events, d_nseg.p, s);
        u64 n_seg = 0;
        CUDA_CHECK(cudaMemcpyAsync(&n_seg, d_nseg.p, sizeof n_seg, cudaMemcpyDeviceToHost, s));
        CUDA_CHECK(cudaStreamSynchronize(s));
        ctx->st.n_segments = n_seg;
        DevBuf<u64> seg_first(n_seg + 1, s);
        {
            u64* sf = seg_first.p;
            seg_scan.finish(in_seg, [hd, sf] __device__(u64 e, u64 exc, u64) { if (hd[e]) sf[exc] = e; });
            CUDA_CHECK(cudaMemcpyAsync(seg_first.p + n_seg, &n_events, sizeof(u64), cudaMemcpyHostToDevice, s));
        }
        // automaton
        DevBuf<i64> op_target(n_matches, s);
        DevBuf<u64> a_ls(n_matches, s), a_le(n_matches, s), a_rs(n_matches, s), a_re(n_matches, s);
        DevBuf<u32> act_arm(n_matches, s);
        DevBuf<u64> act_wlo(n_matches, s), act_whi(n_matches, s), act_death(n_matches, s), act_ls(n_matches, s);
        DevBuf<asgart_b200_protosd> out_sd(n_matches, s);
        DevBuf<u8> out_flag(n_matches, s);
        out_flag.zero();
        AutoBuffers B{};
        B.ev_i = ev_i.p; B.ev_t = ev_t.p; B.ev_moff = ev_moff; B.ev_cnt = ev_cnt; B.ev_chunk = ev_chunk.p;
        B.seg_first = seg_first.p; B.matches = matches; B.op_target = op_target.p;
        B.a_ls = a_ls.p; B.a_le = a_le.p; B.a_rs = a_rs.p; B.a_re = a_re.p;
        B.act_arm = act_arm.p; B.act_ls = act_ls.p; B.act_wlo = act_wlo.p; B.act_whi = act_whi.p; B.act_death = act_death.p;
        B.out_sd = out_sd.p; B.out_flag = out_flag.p; B.chunk_tc = tc.p; B.chunks = plan.dev.p;
        // light segments: one warp each; heavy segments: one 8-warp block each (every block checks which launch owns it)
        automaton_segment_kernel<1, kActCapLight><<<unsigned(n_seg), 32, 0, s>>>(B, plan.ap, n_seg, n_matches, n_events,
                                                                                 st->reverse ? 1 : 0, st->complement ? 1 : 0);
        KERNEL_CHECK();
        automaton_segment_kernel<kHeavyWarps, kActCapHeavy><<<unsigned(n_seg), kHeavyWarps * 32, 0, s>>>(
            B, plan.ap, n_seg, n_matches, n_events, st->reverse ? 1 : 0, st->complement ? 1 : 0);
        count_launch();
        KERNEL_CHECK();
        count_launch();
        // compaction into CSR families
        const u8* fl = out_flag.p;
        auto in_c = [fl] __device__(u64 j) { const u8 f = fl[j]; return Sum2(f ? 1ull : 0ull, f == 3 ? 1ull : 0ull); };
        DevBuf<Sum2> d_tot(1, s);
        ScanPlan<Sum2, Sum2Op> cscan;
        cscan.prepare(in_c, n_matches, d_tot.p, s);
        Sum2 tot;
        CUDA_CHECK(cudaMemcpyAsync(&tot, d_tot.p, sizeof tot, cudaMemcpyDeviceToHost, s));
        CUDA_CHECK(cudaStreamSynchronize(s));
        n_sds = tot.a; n_fam = tot.b;
        d_sds.alloc(n_sds, s);
        d_off.alloc(n_fam + 1, s);
        {
            const asgart_b200_protosd* src = out_sd.p; asgart_b200_protosd* dst = d_sds.p; u64* off = d_off.p;
            cscan.finish(in_c, [=] __device__(u64 j, const Sum2& exc, const Sum2&) {
                const u8 f = fl[j];
                if (!f) return;
                dst[exc.a] = src[j];
                if (f == 3) off[exc.b] = exc.a;
            });
            CUDA_CHECK(cudaMemcpyAsync(d_off.p + n_fam, &n_sds, sizeof(u64), cudaMemcpyHostToDevice, s));
            CUDA_CHECK(cudaStreamSynchronize(s));
        }
    }
    tauto.stop();
    tpost.start();
    run_post(ctx, d_sds, d_off, n_fam, n_sds, post_mask);
    tpost.stop();
    ctx->st.ms_automaton += tauto.ms();
    ctx->st.ms_post += tpost.ms();
    if (post_mask & ASGART_B200_POST_COMPUTE_SCORE) run_score(ctx, d_sds, n_sds);
    download_result(ctx, d_sds, d_off, n_fam, n_sds, result);
}

void shard_range(u64 total, int shard, int n_shards, u64& b, u64& e) {
    u64 per = ceil_div(ceil_div(total, u64(n_shards)), 32) * 32;
    if (per == 0) per = 32;
    b = std::min(total, u64(shard) * per);
    e = std::min(total, u64(shard + 1) * per);
}

void fold_family_timers(asgart_b200_ctx* ctx) {
    ctx->t_sort.drain(); ctx->t_gather.drain(); ctx->t_rank.drain(); ctx->t_probe.drain(); ctx->t_emit.drain(); ctx->t_scatter.drain(); ctx->t_scatter_main.drain();
    ctx->t_msd0.drain(); ctx->t_msd_hist.drain(); ctx->t_msd_local.drain();
    asgart_b200_stats& S = ctx->st;
    S.ms_msd_scatter0 = ctx->t_msd0.total_ms; S.bytes_msd_scatter0 = ctx->t_msd0.bytes;
    S.ms_msd_hist = ctx->t_msd_hist.total_ms; S.bytes_msd_hist = ctx->t_msd_hist.bytes;
    S.ms_msd_local = ctx->t_msd_local.total_ms; S.bytes_msd_local = ctx->t_msd_local.bytes; S.launches_msd_local = ctx->t_msd_local.launches;
    S.ms_sa_sort = ctx->t_sort.total_ms; S.launches_sa_sort = ctx->t_sort.launches; S.bytes_sa_sort = ctx->t_sort.bytes;
    S.ms_sa_gather = ctx->t_gather.total_ms; S.launches_sa_gather = ctx->t_gather.launches; S.bytes_sa_gather = ctx->t_gather.bytes;
    S.ms_sa_rank = ctx->t_rank.total_ms;
    S.ms_probe = ctx->t_probe.total_ms; S.launches_probe = ctx->t_probe.launches; S.bytes_probe = ctx->t_probe.bytes;
    S.ms_emit = ctx->t_emit.total_ms;
    S.ms_sa_scatter_main = ctx->t_scatter_main.total_ms; S.launches_sa_scatter_main = ctx->t_scatter_main.launches;
    S.bytes_sa_scatter_main = ctx->t_scatter_main.bytes;
    S.ms_sa_scatter = ctx->t_scatter.total_ms + S.ms_sa_scatter_main; S.launches_sa_scatter = ctx->t_scatter.launches + S.launches_sa_scatter_main;
    S.bytes_sa_scatter = ctx->t_scatter.bytes + S.bytes_sa_scatter_main;
    ctx->t_locate.drain();
    S.ms_locate = ctx->t_locate.total_ms;
    S.launches_total = ctx->launches.total;
    S.sa_index_bits = u64(ctx->idx_bits);
}


// ---- ctx_locate (locate.cuh) -----------------------------------------------------------------------------------
constexpr u64 kLocSliceBytes = u64(1) << 28;      // pattern bytes on the device at a time
constexpr u64 kLocSlicePatterns = u64(1) << 24;   // patterns on the device at a time (list entries are u32)
constexpr u64 kLocWindow = u64(1) << 26;          // positions per copy launch (512 MB of int64)
constexpr size_t kLocStage = size_t(1) << 25;     // pinned staging buffer of the host copies

// host <-> device through the context's pinned staging buffer, on its stream
void loc_copy(asgart_b200_ctx* ctx, void* dst, const void* src, size_t bytes, bool to_device) {
    if (!bytes) return;
    if (!ctx->loc_stage) CUDA_CHECK(cudaHostAlloc(reinterpret_cast<void**>(&ctx->loc_stage), kLocStage, cudaHostAllocDefault));
    for (size_t o = 0; o < bytes; o += kLocStage) {
        const size_t m = std::min(kLocStage, bytes - o);
        if (to_device) {
            memcpy(ctx->loc_stage, static_cast<const u8*>(src) + o, m);
            CUDA_CHECK(cudaMemcpyAsync(static_cast<u8*>(dst) + o, ctx->loc_stage, m, cudaMemcpyHostToDevice, ctx->stream));
            CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
        } else {
            CUDA_CHECK(cudaMemcpyAsync(ctx->loc_stage, static_cast<const u8*>(src) + o, m, cudaMemcpyDeviceToHost, ctx->stream));
            CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
            memcpy(static_cast<u8*>(dst) + o, ctx->loc_stage, m);
        }
    }
    (to_device ? ctx->st.h2d_bytes : ctx->st.d2h_bytes) += bytes;
}

// returns false when the positions do not fit in host memory
template <typename IdxT>
bool locate_t(asgart_b200_ctx* ctx, const u8* patterns, const u64* offsets, u64 n, i64 max_hits, asgart_b200_hits& H) {
    auto& ix = IxOf<IdxT>::get(ctx);
    cudaStream_t s = ctx->stream;
    const bool literal = ctx->sa_len != ctx->n1;   // --trim: the literal search (SURVEY Q9)
    const u64 cap = max_hits < 0 ? ~u64(0) : u64(max_hits);
    H.first.assign(n, 0);
    H.count.assign(n, 0);
    H.offsets.assign(n + 1, 0);
    DevBuf<unsigned long long> d_alg(1, s);
    d_alg.zero();
    u64 hits = 0;
    for (u64 p0 = 0; p0 < n;) {
        u64 p1 = p0 + 1;   // a slice: bounded bytes and patterns (a single longer pattern makes a slice of its own)
        while (p1 < n && p1 - p0 < kLocSlicePatterns && offsets[p1 + 1] - offsets[p0] <= kLocSliceBytes) ++p1;
        const u64 np = p1 - p0, base = offsets[p0], nb = offsets[p1] - base, nw = ceil_div(nb, 16) + 4;
        std::vector<u64> off(np + 1);
        for (u64 i = 0; i <= np; ++i) off[i] = offsets[p0 + i] - base;
        std::vector<u32> list_short, list_long;   // keeps the long patterns out of the warps of the short ones
        if (!literal)
            for (u64 i = 0; i < np; ++i) (off[i + 1] - off[i] <= 32 ? list_short : list_long).push_back(u32(i));
        DevBuf<u8> d_pat(nb, s);
        DevBuf<u64> d_off(np + 1, s), d_pp(nw, s), d_cut(np, s);
        DevBuf<i64> d_first(np, s), d_count(np, s);
        DevBuf<u32> d_short(list_short.size(), s), d_long(list_long.size(), s);
        loc_copy(ctx, d_pat.p, patterns + base, nb, true);
        loc_copy(ctx, d_off.p, off.data(), (np + 1) * 8, true);
        loc_copy(ctx, d_short.p, list_short.data(), list_short.size() * 4, true);
        loc_copy(ctx, d_long.p, list_long.data(), list_long.size() * 4, true);
        CUDA_CHECK(cudaMemsetAsync(d_cut.p, 0xFF, np * 8, s));
        locate_pack_kernel<<<unsigned(ceil_div(nw, 256)), 256, 0, s>>>(d_pat.p, nb, d_off.p, np, d_pp.p, nw,
                                                                      reinterpret_cast<unsigned long long*>(d_cut.p));
        KERNEL_CHECK();
        count_launch();
        LocateParams<IdxT> P{};
        P.PT = ctx->d_pt.p; P.n1 = ctx->n1; P.SA = ix.sa.p; P.sa_len = ctx->sa_len;
        P.lut_lo = ix.lut_lo.p; P.lut_hi = ix.lut_hi.p; P.deep = ix.deep.p; P.deep_depth = ix.deep.p ? ix.deep_depth : 0;
        P.pat = d_pat.p; P.PP = d_pp.p; P.off = d_off.p; P.cut = d_cut.p;
        P.first = d_first.p; P.count = d_count.p; P.alg_bytes = d_alg.p;
        ctx->t_locate.begin();
        u64 launches = 0;
        if (literal) {
            P.list = nullptr; P.n_list = np;
            locate_literal_kernel<IdxT><<<unsigned(ceil_div(np, 256)), 256, 0, s>>>(P);
            KERNEL_CHECK();
            ++launches;
        } else {
            if (!list_short.empty()) {
                P.list = d_short.p; P.n_list = list_short.size();
                locate_short_kernel<IdxT><<<unsigned(ceil_div(P.n_list, 256)), 256, 0, s>>>(P);
                KERNEL_CHECK();
                ++launches;
            }
            if (!list_long.empty()) {
                P.list = d_long.p; P.n_list = list_long.size();
                locate_long_kernel<IdxT><<<unsigned(ceil_div(P.n_list * 32, 256)), 256, 0, s>>>(P);
                KERNEL_CHECK();
                ++launches;
            }
        }
        ctx->t_locate.end(launches, 0);
        count_launch(launches);
        loc_copy(ctx, H.first.data() + p0, d_first.p, np * 8, false);
        loc_copy(ctx, H.count.data() + p0, d_count.p, np * 8, false);
        u64 hs = 0;
        for (u64 i = 0; i < np; ++i) {
            hs += std::min(u64(H.count[p0 + i]), cap);
            H.offsets[p0 + i + 1] = hits + hs;
        }
        if (hs) {
            try {
                H.positions.resize(hits + hs);
            } catch (const std::exception&) {
                return false;
            }
            DevBuf<u64> d_moff(np, s);
            const i64* cp = d_count.p;
            u64* mp = d_moff.p;
            device_scan<u64, SumOp>([cp, cap] __device__(u64 i) { const u64 c = u64(cp[i]); return c < cap ? c : cap; },
                                    [mp] __device__(u64 i, u64 exc, u64) { mp[i] = exc; }, np, (u64*)nullptr, s);
            DevBuf<i64> d_out(std::min(hs, kLocWindow), s);
            for (u64 w0 = 0; w0 < hs; w0 += kLocWindow) {
                const u64 w1 = std::min(hs, w0 + kLocWindow);
                ctx->t_locate.begin();
                locate_copy_kernel<IdxT><<<unsigned(ceil_div(np * 32, 256)), 256, 0, s>>>(ix.sa.p, d_first.p, d_count.p, d_moff.p, np,
                                                                                         cap, w0, w1, d_out.p);
                KERNEL_CHECK();
                ctx->t_locate.end(1, 0);
                count_launch();
                loc_copy(ctx, H.positions.data() + hits + w0, d_out.p, (w1 - w0) * 8, false);
            }
        }
        hits += hs;
        p0 = p1;
    }
    unsigned long long alg = 0;
    CUDA_CHECK(cudaMemcpyAsync(&alg, d_alg.p, sizeof alg, cudaMemcpyDeviceToHost, s));
    CUDA_CHECK(cudaStreamSynchronize(s));
    ctx->st.locate_patterns += n;
    ctx->st.locate_hits += hits;
    ctx->st.bytes_locate += u64(alg) + 8 * hits;
    return true;
}

} }  // namespace ab200::detail
using namespace ab200::detail;

// ================================================================================================ C ABI
extern "C" {

const char* asgart_b200_version(void) { return "asgart_b200 0.1.0 (sm_100a; prefix-doubling SA, lock-step probe search)"; }

int32_t asgart_b200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int32_t asgart_b200_ctx_create(int32_t device, asgart_b200_ctx** out) {
    if (!out) return ASGART_B200_EINVAL;
    *out = nullptr;
    int n = asgart_b200_device_count();
    if (n <= 0) return ASGART_B200_ENODEVICE;
    if (device < 0 || device >= n) return ASGART_B200_EINVAL;
    asgart_b200_ctx* ctx = new (std::nothrow) asgart_b200_ctx();
    if (!ctx) return ASGART_B200_ENOMEM;
    ctx->device = device;
    try {
        CUDA_CHECK(cudaSetDevice(device));
        CUDA_CHECK(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        cudaMemPool_t pool;
        CUDA_CHECK(cudaDeviceGetDefaultMemPool(&pool, device));
        u64 thr = ~u64(0);
        CUDA_CHECK(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr));
        ctx->t_sort.init(ctx->stream); ctx->t_gather.init(ctx->stream); ctx->t_rank.init(ctx->stream);
        ctx->t_probe.init(ctx->stream); ctx->t_emit.init(ctx->stream); ctx->t_scatter.init(ctx->stream); ctx->t_scatter_main.init(ctx->stream);
        ctx->t_msd0.init(ctx->stream); ctx->t_msd_hist.init(ctx->stream); ctx->t_msd_local.init(ctx->stream);
        ctx->t_locate.init(ctx->stream);
        CUDA_CHECK(cudaEventCreate(&ctx->ev_a)); CUDA_CHECK(cudaEventCreate(&ctx->ev_b));
    } catch (const CudaError& e) {
        int code = e.code;
        delete ctx;
        cudaGetLastError();
        return code;
    }
    *out = ctx;
    return ASGART_B200_OK;
}

void asgart_b200_ctx_destroy(asgart_b200_ctx* ctx) {
    if (!ctx) return;
    if (getenv("ASGART_B200_DEBUG_TIMING"))
        fprintf(stderr, "[asgart_b200] host stalls: %llu cudaMallocAsync %.2f ms, %llu SA-build read-backs %.2f ms (includes the kernels they wait for)\n",
                (unsigned long long)g_host_stalls.allocs, g_host_stalls.alloc_ms, (unsigned long long)g_host_stalls.syncs, g_host_stalls.sync_ms);
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    ctx->t_sort.destroy(); ctx->t_gather.destroy(); ctx->t_rank.destroy(); ctx->t_probe.destroy(); ctx->t_emit.destroy(); ctx->t_scatter.destroy(); ctx->t_scatter_main.destroy();
    ctx->t_msd0.destroy(); ctx->t_msd_hist.destroy(); ctx->t_msd_local.destroy(); ctx->t_locate.destroy();
    if (ctx->loc_stage) cudaFreeHost(ctx->loc_stage);
    if (ctx->ev_a) cudaEventDestroy(ctx->ev_a);
    if (ctx->ev_b) cudaEventDestroy(ctx->ev_b);
    if (ctx->group_owned && ctx->group) { delete ctx->group; }
    ctx->group = nullptr;
    if (ctx->rank_slice) cudaFree(ctx->rank_slice);
    for (void* p : ctx->retired_slices) cudaFree(p);
    ctx->pieces.clear();
    for (int i = 0; i < 2; ++i) {
        if (ctx->stage[i]) cudaFreeHost(ctx->stage[i]);
        if (ctx->stage_ev[i]) cudaEventDestroy(ctx->stage_ev[i]);
    }
    ctx->d_text.release(); ctx->d_pt.release(); ctx->d_pn.release(); ctx->shard_blob.release();
    ctx->ix32 = Index32();
    ctx->ix64 = Index64();
    cudaStreamSynchronize(ctx->stream);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
}

const char* asgart_b200_ctx_last_error(const asgart_b200_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int32_t asgart_b200_ctx_set_index_bits(asgart_b200_ctx* ctx, int32_t bits) {
    if (!ctx || (bits != 0 && bits != 32 && bits != 64)) return ASGART_B200_EINVAL;
    ctx->want_bits = bits;
    drop_sorted_keys(ctx);
    return ASGART_B200_OK;
}

int32_t asgart_b200_ctx_load_strand(asgart_b200_ctx* ctx, const uint8_t* T, int64_t n_plus_1) {
    return guarded(ctx, [&]() -> int32_t {
        if (!T || n_plus_1 < 1) return fail(ctx, ASGART_B200_EINVAL, "null strand or n_plus_1 < 1");
        ctx->have_strand = ctx->have_index = false;
        drop_sorted_keys(ctx);
        ctx->pn_mode = -1;
        ctx->n1 = u64(n_plus_1);
        EventTimer th(ctx->stream);
        th.start();
        ctx->d_text.alloc(ctx->n1, ctx->stream);
        u64 copied = ctx->n1;
        if (ctx->group && ctx->group_owned && ctx->group->world > 1) {
            // one process per GPU, every rank was handed the same strand: each rank moves 1/world of it over PCIe and the
            // ranks exchange the pieces over NVLink (N full host copies made the N-GPU end-to-end time worse than N = 1)
            const int world = ctx->group->world, rank = ctx->group->rank;
            std::vector<u64> offs(size_t(world) + 1);
            for (int r = 0; r <= world; ++r) offs[size_t(r)] = (ctx->n1 * u64(r) / u64(world)) & ~u64(15);
            offs[size_t(world)] = ctx->n1;
            const u64 o = offs[size_t(rank)];
            copied = offs[size_t(rank) + 1] - o;
            if (copied) CUDA_CHECK(cudaMemcpyAsync(ctx->d_text.p + o, T + o, copied, cudaMemcpyHostToDevice, ctx->stream));
            ctx->group->share_pieces(ctx->d_text.p, offs.data(), 1, ctx->stream);
        } else {
            CUDA_CHECK(cudaMemcpyAsync(ctx->d_text.p, T, ctx->n1, cudaMemcpyHostToDevice, ctx->stream));
        }
        th.stop();
        const int32_t rc = pack_loaded_strand(ctx);
        ctx->st.ms_h2d += th.ms();
        ctx->st.h2d_bytes += copied;
        return rc;
    });
}

// ---- GPU-side FASTA ingest (fasta_ingest.cuh) -----------------------------------------------------------------
int32_t asgart_b200_ctx_ingest_begin(asgart_b200_ctx* ctx) {
    return guarded(ctx, [&]() -> int32_t {
        ctx->have_strand = ctx->have_index = false;
        drop_sorted_keys(ctx);
        ctx->pn_mode = -1;
        ctx->pieces.clear();
        ctx->ingesting = true;
        return ASGART_B200_OK;
    });
}

int32_t asgart_b200_ctx_ingest_fasta(asgart_b200_ctx* ctx, const uint8_t* bytes, int64_t n_bytes, int32_t skip_masked) {
    return guarded(ctx, [&]() -> int32_t {
        if (!ctx->ingesting) return fail(ctx, ASGART_B200_ESTATE, "ingest_fasta before ingest_begin");
        if ((!bytes && n_bytes > 0) || n_bytes < 0) return fail(ctx, ASGART_B200_EINVAL, "null bytes or negative size");
        const u64 n = u64(n_bytes);
        if (!first_byte_ok(n, n ? bytes[0] : 0)) return fail(ctx, ASGART_B200_EINVAL, "Unable to parse FASTA: expected > at record start");
        DevBuf<u8> d_file(n, ctx->stream);
        EventTimer th(ctx->stream);
        th.start();
        if (n) CUDA_CHECK(cudaMemcpyAsync(d_file.p, bytes, n, cudaMemcpyHostToDevice, ctx->stream));
        th.stop();
        ctx->pieces.emplace_back();
        IngestPiece& piece = ctx->pieces.back();
        ingest_piece(ctx, d_file.p, n, skip_masked != 0, piece);
        ingest_record_ids(piece, n, [&](u64 at, char* buf, size_t cap) {
            const size_t r = size_t(std::min<u64>(cap, n - at));
            memcpy(buf, bytes + at, r);
            return r;
        });
        ctx->st.ms_h2d += th.ms();
        ctx->st.h2d_bytes += n;
        return ASGART_B200_OK;
    });
}

int32_t asgart_b200_ctx_ingest_file(asgart_b200_ctx* ctx, const char* path, int32_t skip_masked) {
    return guarded(ctx, [&]() -> int32_t {
        if (!ctx->ingesting) return fail(ctx, ASGART_B200_ESTATE, "ingest_file before ingest_begin");
        if (!path) return fail(ctx, ASGART_B200_EINVAL, "null path");
        struct FdGuard { int fd; ~FdGuard() { if (fd >= 0) close(fd); } } f{open(path, O_RDONLY)};
        struct stat sb;
        if (f.fd < 0 || fstat(f.fd, &sb) != 0 || !S_ISREG(sb.st_mode)) {
            ctx->err = std::string("Unable to read FASTA file `") + path + "`";
            return ASGART_B200_EINVAL;
        }
        const u64 n = u64(sb.st_size);
        constexpr size_t kStage = size_t(32) << 20;
        for (int i = 0; i < 2; ++i) {
            if (!ctx->stage[i]) CUDA_CHECK(cudaHostAlloc(reinterpret_cast<void**>(&ctx->stage[i]), kStage, cudaHostAllocDefault));
            if (!ctx->stage_ev[i]) CUDA_CHECK(cudaEventCreateWithFlags(&ctx->stage_ev[i], cudaEventDisableTiming));
        }
        DevBuf<u8> d_file(n, ctx->stream);
        EventTimer th(ctx->stream);
        th.start();
        bool bad_first = false;
        u64 done = 0;
        for (int slot = 0; done < n; slot ^= 1) {
            CUDA_CHECK(cudaEventSynchronize(ctx->stage_ev[slot]));   // the copy that last used this buffer has finished
            const size_t want = size_t(std::min<u64>(kStage, n - done));
            // the page cache hands out ~6 GB/s per reading thread: four readers per staging buffer keep the link busier
            constexpr int kReaders = 4;
            bool ok[kReaders];
            std::thread readers[kReaders];
            const size_t part = (want + kReaders - 1) / kReaders;
            for (int r = 0; r < kReaders; ++r) {
                const size_t b = std::min(want, part * size_t(r)), e = std::min(want, b + part);
                u8* dst = ctx->stage[slot];
                const int fd = f.fd;
                bool* flag = &ok[r];
                readers[r] = std::thread([=]() {
                    size_t at = b;
                    while (at < e) {
                        const ssize_t k = pread(fd, dst + at, e - at, off_t(done + at));
                        if (k <= 0) break;
                        at += size_t(k);
                    }
                    *flag = at == e;
                });
            }
            bool all = true;
            for (int r = 0; r < kReaders; ++r) { readers[r].join(); all = all && ok[r]; }
            if (!all) { ctx->err = std::string("Unable to read FASTA file `") + path + "`"; return ASGART_B200_EINVAL; }
            const size_t got = want;
            if (done == 0 && !first_byte_ok(n, ctx->stage[slot][0])) { bad_first = true; break; }
            CUDA_CHECK(cudaMemcpyAsync(d_file.p + done, ctx->stage[slot], got, cudaMemcpyHostToDevice, ctx->stream));
            CUDA_CHECK(cudaEventRecord(ctx->stage_ev[slot], ctx->stream));
            done += got;
        }
        th.stop();
        if (bad_first) {
            CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
            ctx->err = std::string("Unable to parse `") + path + "`";
            return ASGART_B200_EINVAL;
        }
        ctx->pieces.emplace_back();
        IngestPiece& piece = ctx->pieces.back();
        ingest_piece(ctx, d_file.p, n, skip_masked != 0, piece);
        ingest_record_ids(piece, n, [&](u64 at, char* buf, size_t cap) {   // the few bytes after each '>' straight from the file
            const ssize_t r = pread(f.fd, buf, cap, off_t(at));
            return r > 0 ? size_t(r) : size_t(0);
        });
        ctx->st.ms_h2d += th.ms();
        ctx->st.h2d_bytes += n;
        return ASGART_B200_OK;
    });
}

int32_t asgart_b200_ctx_ingest_finish(asgart_b200_ctx* ctx, const char* file_names, asgart_b200_prepared** out) {
    return guarded(ctx, [&]() -> int32_t {
        if (!ctx->ingesting) return fail(ctx, ASGART_B200_ESTATE, "ingest_finish before ingest_begin");
        if (!out) return fail(ctx, ASGART_B200_EINVAL, "null out");
        *out = nullptr;
        u64 total = 0;
        for (const IngestPiece& p : ctx->pieces) total += p.kept;
        ctx->n1 = total + 1;
        ctx->d_text.alloc(ctx->n1, ctx->stream);
        std::vector<std::string> names;
        std::vector<u64> pos, len;
        std::vector<asgart_b200_chunk> chunks;
        u64 off = 0;
        for (IngestPiece& p : ctx->pieces) {    // src/bin/asgart.rs:375-395: files concatenated with a running offset
            if (p.kept) CUDA_CHECK(cudaMemcpyAsync(ctx->d_text.p + off, p.strand.p, p.kept, cudaMemcpyDeviceToDevice, ctx->stream));
            ingest_chunks(p, off, chunks, pos, len);
            for (std::string& s : p.names) names.push_back(std::move(s));
            off += p.kept;
        }
        CUDA_CHECK(cudaMemsetAsync(ctx->d_text.p + total, '$', 1, ctx->stream));   // src/bin/asgart.rs:430
        const int32_t rc = pack_loaded_strand(ctx);
        ctx->pieces.clear();
        ctx->ingesting = false;
        if (rc) return rc;
        std::string joined;                     // src/bin/asgart.rs:466
        for (const char* c = file_names ? file_names : ""; *c;) {
            const char* e = strchr(c, '\n');
            const size_t l = e ? size_t(e - c) : strlen(c);
            if (l) { if (!joined.empty()) joined += ", "; joined.append(c, l); }
            c += l + (e ? 1 : 0);
        }
        *out = ab200_prepared_device_only(joined, total, names, pos, len, chunks);
        return ASGART_B200_OK;
    });
}

int32_t asgart_b200_ctx_download_strand(asgart_b200_ctx* ctx, uint8_t* out, int64_t cap) {
    return guarded(ctx, [&]() -> int32_t {
        if (!ctx->have_strand) return fail(ctx, ASGART_B200_ESTATE, "download_strand without a strand");
        if (!out || cap < int64_t(ctx->n1)) return fail(ctx, ASGART_B200_EINVAL, "null out or cap < n + 1");
        CUDA_CHECK(cudaMemcpyAsync(out, ctx->d_text.p, ctx->n1, cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
        ctx->st.d2h_bytes += ctx->n1;
        return ASGART_B200_OK;
    });
}

int32_t asgart_b200_ctx_build_index(asgart_b200_ctx* ctx) {
    return guarded(ctx, [&]() -> int32_t {
        if (!ctx->have_strand) return fail(ctx, ASGART_B200_ESTATE, "build_index before load_strand");
        ctx->have_index = false;
        ctx->idx_bits = pick_bits(ctx);
        if (ctx->idx_bits == 32 && ctx->n1 >= 0xFFFFFFFEull) return fail(ctx, ASGART_B200_EINVAL, "32-bit indices need n+1 < 2^32-2");
        if (ctx->idx_bits == 32) { ctx->ix64 = Index64(); build_index_t<u32>(ctx); }
        else { ctx->ix32 = Index32(); build_index_t<u64>(ctx); }
        CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
        ctx->sa_len = ctx->n1;
        ctx->have_index = true;
        return ASGART_B200_OK;
    });
}

// --trim (src/bin/asgart.rs:142-147): suffix array of strand[a..b]+'$' shifted by a; LUT by the reference's own bisection
// over the whole strand (lut_literal_kernel); no deep table, so every probe takes the literal search (Q9).
int32_t asgart_b200_ctx_build_index_trim(asgart_b200_ctx* ctx, uint64_t a, uint64_t b) {
    return guarded(ctx, [&]() -> int32_t {
        if (!ctx->have_strand) return fail(ctx, ASGART_B200_ESTATE, "build_index_trim before load_strand");
        if (ctx->group && ctx->group->world > 1) return fail(ctx, ASGART_B200_ESTATE, "--trim builds on one device");
        if (!(a < b) || b > ctx->n1 - 1) return fail(ctx, ASGART_B200_EINVAL, "trim needs start < stop <= strand length (see asgart_b200_effective_trim)");
        ctx->have_index = false;
        ctx->idx_bits = pick_bits(ctx);
        if (ctx->idx_bits == 32 && ctx->n1 >= 0xFFFFFFFEull) return fail(ctx, ASGART_B200_EINVAL, "32-bit indices need n+1 < 2^32-2");
        if (ctx->idx_bits == 32) { ctx->ix64 = Index64(); build_index_trim_t<u32>(ctx, a, b); }
        else { ctx->ix32 = Index32(); build_index_trim_t<u64>(ctx, a, b); }
        CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
        ctx->sa_len = b - a + 1;
        ctx->have_index = true;
        return ASGART_B200_OK;
    });
}

// prepare_data's validation of --trim (src/bin/asgart.rs:432-463; n_plus_1 = strand length with '$'): stop is clamped to
// the last base; returns 1 and the effective values, or 0 when the reference skips trimming.
int32_t asgart_b200_effective_trim(uint64_t start, uint64_t stop, int64_t n_plus_1, uint64_t* eff_start, uint64_t* eff_stop) {
    if (n_plus_1 < 1) return 0;
    const uint64_t len = uint64_t(n_plus_1);
    if (stop >= len) stop = len - 1;
    if (stop <= start || start >= len) return 0;
    if (eff_start) *eff_start = start;
    if (eff_stop) *eff_stop = stop;
    return 1;
}

// ---- sharded index build ------------------------------------------------------------------------------------
int32_t asgart_b200_build_index_group(asgart_b200_ctx* const* ctxs, int32_t world) {
    if (!ctxs || world < 1 || world > kMaxWorld) return ASGART_B200_EINVAL;
    for (int r = 0; r < world; ++r) {
        if (!ctxs[r] || ctxs[r]->group) return ASGART_B200_EINVAL;
        if (!ctxs[r]->have_strand || ctxs[r]->n1 != ctxs[0]->n1) return fail(ctxs[r], ASGART_B200_ESTATE, "every member needs the same strand loaded");
    }
    // members on different devices reach each other's rank slices through peer access
    for (int a = 0; a < world; ++a)
        for (int b2 = 0; b2 < world; ++b2) {
            if (ctxs[a]->device == ctxs[b2]->device) continue;
            int can = 0;
            if (cudaDeviceCanAccessPeer(&can, ctxs[a]->device, ctxs[b2]->device) != cudaSuccess || !can)
                return fail(ctxs[a], ASGART_B200_EINVAL, "no peer access between the devices of the group");
            cudaSetDevice(ctxs[a]->device);
            cudaError_t e = cudaDeviceEnablePeerAccess(ctxs[b2]->device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return fail(ctxs[a], ASGART_B200_ECUDA, cudaGetErrorString(e));
            cudaGetLastError();
        }
    ThreadGroupShared shared(world);
    std::vector<int32_t> rc(world, ASGART_B200_OK);
    std::vector<std::thread> threads;
    for (int r = 0; r < world; ++r)
        threads.emplace_back([&, r] {
            asgart_b200_ctx* ctx = ctxs[r];
            ThreadGroup member(&shared, r, ctx->stream);
            ctx->group = &member;
            rc[r] = asgart_b200_ctx_build_index(ctx);
            if (rc[r] != ASGART_B200_OK) shared.fail();
            ctx->group = nullptr;
        });
    for (auto& t : threads) t.join();
    for (int r = 0; r < world; ++r)
        if (rc[r] != ASGART_B200_OK) return rc[r];
    return ASGART_B200_OK;
}

int32_t asgart_b200_dist_unique_id(uint8_t* out, int64_t cap) {
    if (!out || cap < int64_t(sizeof(ncclUniqueId))) return ASGART_B200_EINVAL;
    if (!nccl_api().load()) return ASGART_B200_ECUDA;
    ncclUniqueId id;
    if (nccl_api().GetUniqueId(&id) != ncclSuccess) return ASGART_B200_ECUDA;
    memcpy(out, &id, sizeof id);
    return int32_t(sizeof id);
}

int32_t asgart_b200_ctx_dist_init(asgart_b200_ctx* ctx, int32_t rank, int32_t world, const uint8_t* unique_id, int64_t id_bytes) {
    return guarded(ctx, [&]() -> int32_t {
        if (world < 1 || world > kMaxWorld || rank < 0 || rank >= world || !unique_id || id_bytes != int64_t(sizeof(ncclUniqueId)))
            return fail(ctx, ASGART_B200_EINVAL, "bad rank/world/unique id");
        if (ctx->group) return fail(ctx, ASGART_B200_ESTATE, "context already belongs to a group");
        if (!nccl_api().load()) return fail(ctx, ASGART_B200_ECUDA, nccl_api().error.c_str());
        ncclUniqueId id;
        memcpy(&id, unique_id, sizeof id);
        ctx->group = new NcclGroup(rank, world, id, ctx->stream);
        ctx->group_owned = true;
        return ASGART_B200_OK;
    });
}

int32_t asgart_b200_ctx_dist_shutdown(asgart_b200_ctx* ctx) {
    return guarded(ctx, [&]() -> int32_t {
        CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
        if (ctx->group_owned && ctx->group) delete ctx->group;
        ctx->group = nullptr;
        ctx->group_owned = false;
        return ASGART_B200_OK;
    });
}

int32_t asgart_b200_ctx_upload_sa(asgart_b200_ctx* ctx, const int64_t* SA) {
    return guarded(ctx, [&]() -> int32_t {
        if (!ctx->have_strand) return fail(ctx, ASGART_B200_ESTATE, "upload_sa before load_strand");
        if (!SA) return fail(ctx, ASGART_B200_EINVAL, "null SA");
        ctx->have_index = false;
        ctx->idx_bits = pick_bits(ctx);
        if (ctx->idx_bits == 32) {
            ctx->ix64 = Index64();
            ctx->ix32.sa.alloc(ctx->n1, ctx->stream);
            upload_from_i64<u32>(SA, ctx->ix32.sa.p, ctx->n1, ctx->stream);
            build_lut<u32>(ctx);
        } else {
            ctx->ix32 = Index32();
            ctx->ix64.sa.alloc(ctx->n1, ctx->stream);
            upload_from_i64<u64>(SA, ctx->ix64.sa.p, ctx->n1, ctx->stream);
            build_lut<u64>(ctx);
        }
        CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
        ctx->sa_len = ctx->n1;
        ctx->have_index = true;
        return ASGART_B200_OK;
    });
}

int32_t asgart_b200_ctx_download_sa(asgart_b200_ctx* ctx, int64_t* SA) {
    return guarded(ctx, [&]() -> int32_t {
        if (!ctx->have_index) return fail(ctx, ASGART_B200_ESTATE, "download_sa before build_index");
        if (!SA) return fail(ctx, ASGART_B200_EINVAL, "null SA");
        if (ctx->idx_bits == 32) download_as_i64<u32>(ctx->ix32.sa.p, SA, ctx->sa_len, ctx->stream);
        else download_as_i64<u64>(ctx->ix64.sa.p, SA, ctx->sa_len, ctx->stream);
        return ASGART_B200_OK;
    });
}

int32_t asgart_b200_ctx_check_sa(asgart_b200_ctx* ctx, int64_t* n_bad) {
    return guarded(ctx, [&]() -> int32_t {
        if (!ctx->have_index) return fail(ctx, ASGART_B200_ESTATE, "check_sa before build_index");
        if (!n_bad) return fail(ctx, ASGART_B200_EINVAL, "null output");
        if (ctx->sa_len != ctx->n1) return fail(ctx, ASGART_B200_ESTATE, "check_sa: the index was built with --trim (it is not a suffix array of the strand)");
        if (ctx->idx_bits == 32) *n_bad = check_sa_t<u32>(ctx); else *n_bad = check_sa_t<u64>(ctx);
        return ASGART_B200_OK;
    });
}

int32_t asgart_b200_ctx_sa_fingerprint(asgart_b200_ctx* ctx, uint64_t* fingerprint) {
    return guarded(ctx, [&]() -> int32_t {
        if (!ctx->have_index) return fail(ctx, ASGART_B200_ESTATE, "sa_fingerprint before build_index");
        if (!fingerprint) return fail(ctx, ASGART_B200_EINVAL, "null output");
        *fingerprint = ctx->idx_bits == 32 ? sa_fingerprint_t<u32>(ctx) : sa_fingerprint_t<u64>(ctx);
        return ASGART_B200_OK;
    });
}

int32_t asgart_b200_ctx_download_lut(asgart_b200_ctx* ctx, int64_t* lo, int64_t* hi) {
    return guarded(ctx, [&]() -> int32_t {
        if (!ctx->have_index) return fail(ctx, ASGART_B200_ESTATE, "download_lut before build_index");
        if (!lo || !hi) return fail(ctx, ASGART_B200_EINVAL, "null output");
        if (ctx->idx_bits == 32) {
            download_as_i64<u32>(ctx->ix32.lut_lo.p, lo, kLutSize, ctx->stream);
            download_as_i64<u32>(ctx->ix32.lut_hi.p, hi, kLutSize, ctx->stream);
        } else {
            download_as_i64<u64>(ctx->ix64.lut_lo.p, lo, kLutSize, ctx->stream);
            download_as_i64<u64>(ctx->ix64.lut_hi.p, hi, kLutSize, ctx->stream);
        }
        return ASGART_B200_OK;
    });
}

int32_t asgart_b200_ctx_probe_ranges(asgart_b200_ctx* ctx, const asgart_b200_chunk* chunk, const asgart_b200_settings* st,
                                     int64_t* lo, int64_t* hi, int64_t n_probes) {
    return guarded(ctx, [&]() -> int32_t {
        if (!ctx->have_index) return fail(ctx, ASGART_B200_ESTATE, "probe_ranges before build_index");
        if (!lo || !hi || n_probes < 0) return fail(ctx, ASGART_B200_EINVAL, "bad output arrays");
        ChunkPlan plan;
        asgart_b200_settings s2 = *st;
        s2.min_duplication_length = 0;
        int rc = make_plan(ctx, chunk, 1, &s2, plan);
        if (rc) return rc;
        if (u64(n_probes) > plan.host[0].n_probes) return fail(ctx, ASGART_B200_EINVAL, "n_probes exceeds the chunk's probe count");
        if (n_probes == 0) return ASGART_B200_OK;
        ensure_needle(ctx, plan.mode);
        DevBuf<i64> d_lo(n_probes, ctx->stream), d_hi(n_probes, ctx->stream);
        auto launch = [&](auto tag) {
            using IdxT = decltype(tag);
            auto& ix = IxOf<IdxT>::get(ctx);
            ProbeParams<IdxT> P{};
            P.PT = ctx->d_pt.p; P.PN = plan.mode == PACK_DIRECT ? ctx->d_pt.p : ctx->d_pn.p;
            P.SA = ix.sa.p; P.lut_lo = ix.lut_lo.p; P.lut_hi = ix.lut_hi.p;
            P.chunks = plan.dev.p; P.n_chunks = 1; P.n1 = ctx->n1; P.k = plan.k; P.s = plan.s;
            P.p_begin = 0; P.p_end = u64(n_probes);
            P.rng_lo = d_lo.p; P.rng_hi = d_hi.p;
            DevBuf<unsigned long long> counters(CTR_COUNT, ctx->stream);
            counters.zero();
            P.counters = counters.p;
            unsigned long long h_ctr[CTR_COUNT];
            ctx->n_probe_keys += run_probe_kernels<IdxT>(ctx, P, plan.mode, h_ctr);
        };
        if (ctx->idx_bits == 32) launch(u32(0)); else launch(u64(0));
        CUDA_CHECK(cudaMemcpyAsync(lo, d_lo.p, n_probes * sizeof(i64), cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_CHECK(cudaMemcpyAsync(hi, d_hi.p, n_probes * sizeof(i64), cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_CHECK(cudaStreamSynchronize(ctx->stream));
        return ASGART_B200_OK;
    });
}

int32_t asgart_b200_ctx_search(asgart_b200_ctx* ctx, const asgart_b200_chunk* chunks, int64_t n_chunks,
                               const asgart_b200_settings* st, uint32_t post_mask, asgart_b200_result** out) {
    return guarded(ctx, [&]() -> int32_t {
        if (!out) return fail(ctx, ASGART_B200_EINVAL, "null out");
        *out = nullptr;
        if (!ctx->have_index) return fail(ctx, ASGART_B200_ESTATE, "search before build_index");
        ChunkPlan plan;
        int rc = make_plan(ctx, chunks, n_chunks, st, plan);
        if (rc) return rc;
        ensure_needle(ctx, plan.mode);
        EventTimer ts(ctx->stream);
        ts.start();
        StageA A;
        if (ctx->idx_bits == 32) run_stage_a<u32>(ctx, plan, st, 0, plan.total_probes, A);
        else run_stage_a<u64>(ctx, plan, st, 0, plan.total_probes, A);
        ts.stop();
        ctx->st.ms_search += ts.ms();
        asgart_b200_result* r = new asgart_b200_result();
        try {
            run_stage_b(ctx, plan, st, A.bits.p, A.n_events, A.ev_probe.p, A.ev_cnt.p, A.ev_moff.p, A.matches.p, A.n_matches, post_mask, r);
        } catch (...) { delete r; throw; }
        *out = r;
        return ASGART_B200_OK;
    });
}

int32_t asgart_b200_ctx_search_shard(asgart_b200_ctx* ctx, const asgart_b200_chunk* chunks, int64_t n_chunks,
                                     const asgart_b200_settings* st, int32_t shard, int32_t n_shards, asgart_b200_partial** out) {
    return guarded(ctx, [&]() -> int32_t {
        if (!out || n_shards < 1 || shard < 0 || shard >= n_shards) return fail(ctx, ASGART_B200_EINVAL, "bad shard arguments");
        *out = nullptr;
        if (!ctx->have_index) return fail(ctx, ASGART_B200_ESTATE, "search before build_index");
        ChunkPlan plan;
        int rc = make_plan(ctx, chunks, n_chunks, st, plan);
        if (rc) return rc;
        ensure_needle(ctx, plan.mode);
        u64 b, e;
        shard_range(plan.total_probes, shard, n_shards, b, e);
        EventTimer ts(ctx->stream);
        ts.start();
        StageA A;
        if (ctx->idx_bits == 32) run_stage_a<u32>(ctx, plan, st, b, e, A);
        else run_stage_a<u64>(ctx, plan, st, b, e, A);
        ts.stop();
        ctx->st.ms_search += ts.ms();
        asgart_b200_partial* p = new asgart_b200_partial();
        p->p_begin = b; p->p_end = e;
        p->bits.resize(ceil_div(e - b, 32));
        p->ev_probe.resize(A.n_events); p->ev_cnt.resize(A.n_events); p->matches.resize(A.n_matches);
        cudaStream_t s = ctx->stream;
        if (!p->bits.empty()) CUDA_CHECK(cudaMemcpyAsync(p->bits.data(), A.bits.p, p->bits.size() * 4, cudaMemcpyDeviceToHost, s));
        if (A.n_events) {
            CUDA_CHECK(cudaMemcpyAsync(p->ev_probe.data(), A.ev_probe.p, A.n_events * 8, cudaMemcpyDeviceToHost, s));
            CUDA_CHECK(cudaMemcpyAsync(p->ev_cnt.data(), A.ev_cnt.p, A.n_events * 4, cudaMemcpyDeviceToHost, s));
        }
        if (A.n_matches) CUDA_CHECK(cudaMemcpyAsync(p->matches.data(), A.matches.p, A.n_matches * 8, cudaMemcpyDeviceToHost, s));
        CUDA_CHECK(cudaStreamSynchronize(s));
        ctx->st.d2h_bytes += p->bits.size() * 4 + A.n_events * 12 + A.n_matches * 8;
        *out = p;
        return ASGART_B200_OK;
    });
}

int64_t asgart_b200_partial_size(const asgart_b200_partial* p) {
    if (!p) return 0;
    return int64_t(6 * 8 + p->bits.size() * 4 + p->ev_probe.size() * 8 + p->ev_cnt.size() * 4 + p->matches.size() * 8);
}

int32_t asgart_b200_partial_serialize(const asgart_b200_partial* p, uint8_t* buf, int64_t cap) {
    if (!p || !buf || cap < asgart_b200_partial_size(p)) return ASGART_B200_EINVAL;
    u64 hdr[6] = {kPartialMagic, p->p_begin, p->p_end, u64(p->bits.size()), u64(p->ev_probe.size()), u64(p->matches.size())};
    uint8_t* w = buf;
    memcpy(w, hdr, sizeof hdr); w += sizeof hdr;
    memcpy(w, p->bits.data(), p->bits.size() * 4); w += p->bits.size() * 4;
    memcpy(w, p->ev_probe.data(), p->ev_probe.size() * 8); w += p->ev_probe.size() * 8;
    memcpy(w, p->ev_cnt.data(), p->ev_cnt.size() * 4); w += p->ev_cnt.size() * 4;
    memcpy(w, p->matches.data(), p->matches.size() * 8);
    return ASGART_B200_OK;
}

void asgart_b200_partial_free(asgart_b200_partial* p) { delete p; }

int32_t asgart_b200_ctx_finish(asgart_b200_ctx* ctx, const asgart_b200_chunk* chunks, int64_t n_chunks, const asgart_b200_settings* st,
                               const uint8_t* const* partials, const int64_t* sizes, int32_t n_shards, uint32_t post_mask,
                               asgart_b200_result** out) {
    return guarded(ctx, [&]() -> int32_t {
        if (!out || !partials || !sizes || n_shards < 1) return fail(ctx, ASGART_B200_EINVAL, "bad finish arguments");
        *out = nullptr;
        if (!ctx->have_strand) return fail(ctx, ASGART_B200_ESTATE, "finish before load_strand");
        ChunkPlan plan;
        int rc = make_plan(ctx, chunks, n_chunks, st, plan);
        if (rc) return rc;
        const u64 words = ceil_div(plan.total_probes, 32);
        std::vector<u32> bits(words, 0);
        std::vector<u64> ev_probe, matches;
        std::vector<u32> ev_cnt;
        u64 expect = 0;
        for (int r = 0; r < n_shards; ++r) {
            const uint8_t* b = partials[r];
            if (!b || sizes[r] < 48) return fail(ctx, ASGART_B200_EINVAL, "partial too small");
            u64 hdr[6];
            memcpy(hdr, b, sizeof hdr);
            if (hdr[0] != kPartialMagic) return fail(ctx, ASGART_B200_EINVAL, "bad partial magic");
            const u64 pb = hdr[1], pe = hdr[2], nb = hdr[3], ne = hdr[4], nm = hdr[5];
            if (pb != expect || pe < pb || pe > plan.total_probes || ((pb & 31) && pb != plan.total_probes) || nb != ceil_div(pe - pb, 32) ||
                u64(sizes[r]) != 48 + nb * 4 + ne * 12 + nm * 8)
                return fail(ctx, ASGART_B200_EINVAL, "partials are not the consecutive shards of this plan");
            expect = pe;
            const uint8_t* p = b + 48;
            memcpy(bits.data() + (pb >> 5), p, nb * 4); p += nb * 4;
            size_t e0 = ev_probe.size(), m0 = matches.size();
            ev_probe.resize(e0 + ne); ev_cnt.resize(e0 + ne); matches.resize(m0 + nm);
            memcpy(ev_probe.data() + e0, p, ne * 8); p += ne * 8;
            memcpy(ev_cnt.data() + e0, p, ne * 4); p += ne * 4;
            memcpy(matches.data() + m0, p, nm * 8);
        }
        if (expect != plan.total_probes) return fail(ctx, ASGART_B200_EINVAL, "partials do not cover all probes");
        cudaStream_t s = ctx->stream;
        const u64 ne = ev_probe.size(), nm = matches.size();
        DevBuf<u32> d_bits(words, s), d_cnt(ne, s);
        DevBuf<u64> d_probe(ne, s), d_moff(ne, s), d_matches(nm, s);
        if (words) CUDA_CHECK(cudaMemcpyAsync(d_bits.p, bits.data(), words * 4, cudaMemcpyHostToDevice, s));
        if (ne) {
            CUDA_CHECK(cudaMemcpyAsync(d_probe.p, ev_probe.data(), ne * 8, cudaMemcpyHostToDevice, s));
            CUDA_CHECK(cudaMemcpyAsync(d_cnt.p, ev_cnt.data(), ne * 4, cudaMemcpyHostToDevice, s));
            const u32* cp = d_cnt.p; u64* mp = d_moff.p;
            device_scan<u64, SumOp>([cp] __device__(u64 e) { return u64(cp[e]); }, [mp] __device__(u64 e, u64 exc, u64) { mp[e] = exc; },
                                    ne, (u64*)nullptr, s);
        }
        if (nm) CUDA_CHECK(cudaMemcpyAsync(d_matches.p, matches.data(), nm * 8, cudaMemcpyHostToDevice, s));
        ctx->st.h2d_bytes += words * 4 + ne * 12 + nm * 8;
        asgart_b200_result* r = new asgart_b200_result();
        try {
            run_stage_b(ctx, plan, st, d_bits.p, ne, d_probe.p, d_cnt.p, d_moff.p, d_matches.p, nm, post_mask, r);
        } catch (...) { delete r; throw; }
        *out = r;
        return ASGART_B200_OK;
    });
}

// Device-resident form of search_shard / finish: the partial stays in HBM as one blob
//   [ processed bits (4 B x words, padded to 8) | ev_probe (8 B x events) | matches (8 B x matches) | ev_cnt (4 B x events) ]
// so that the exchange is a plain NCCL all-gather of device memory (meta = {p_begin, p_end, events, matches} travels apart).
static u64 blob_bytes_of(u64 pb, u64 pe, u64 ne, u64 nm) { return ceil_div(ceil_div(pe - pb, 32) * 4, 8) * 8 + ne * 8 + nm * 8 + ne * 4; }

int32_t asgart_b200_ctx_search_shard_dev(asgart_b200_ctx* ctx, const asgart_b200_chunk* chunks, int64_t n_chunks,
                                         const asgart_b200_settings* st, int32_t shard, int32_t n_shards, void** d_blob,
                                         int64_t* blob_bytes, uint64_t* meta) {
    return guarded(ctx, [&]() -> int32_t {
        if (!d_blob || !blob_bytes || !meta || n_shards < 1 || shard < 0 || shard >= n_shards) return fail(ctx, ASGART_B200_EINVAL, "bad shard arguments");
        if (!ctx->have_index) return fail(ctx, ASGART_B200_ESTATE, "search before build_index");
        ChunkPlan plan;
        int rc = make_plan(ctx, chunks, n_chunks, st, plan);
        if (rc) return rc;
        ensure_needle(ctx, plan.mode);
        u64 b, e;
        shard_range(plan.total_probes, shard, n_shards, b, e);
        EventTimer ts(ctx->stream);
        ts.start();
        StageA A;
        if (ctx->idx_bits == 32) run_stage_a<u32>(ctx, plan, st, b, e, A);
        else run_stage_a<u64>(ctx, plan, st, b, e, A);
        cudaStream_t s = ctx->stream;
        const u64 words = ceil_div(e - b, 32), wbytes = ceil_div(words * 4, 8) * 8;
        const u64 total = blob_bytes_of(b, e, A.n_events, A.n_matches);
        ctx->shard_blob.alloc(std::max<u64>(total, 8), s);
        u8* p = ctx->shard_blob.p;
        if (words) CUDA_CHECK(cudaMemcpyAsync(p, A.bits.p, words * 4, cudaMemcpyDeviceToDevice, s));
        p += wbytes;
        if (A.n_events) CUDA_CHECK(cudaMemcpyAsync(p, A.ev_probe.p, A.n_events * 8, cudaMemcpyDeviceToDevice, s));
        p += A.n_events * 8;
        if (A.n_matches) CUDA_CHECK(cudaMemcpyAsync(p, A.matches.p, A.n_matches * 8, cudaMemcpyDeviceToDevice, s));
        p += A.n_matches * 8;
        if (A.n_events) CUDA_CHECK(cudaMemcpyAsync(p, A.ev_cnt.p, A.n_events * 4, cudaMemcpyDeviceToDevice, s));
        ts.stop();
        ctx->st.ms_search += ts.ms();   // synchronises: the blob is complete when this call returns
        meta[0] = b; meta[1] = e; meta[2] = A.n_events; meta[3] = A.n_matches;
        *d_blob = ctx->shard_blob.p;
        *blob_bytes = int64_t(total);
        return ASGART_B200_OK;
    });
}

int32_t asgart_b200_ctx_finish_dev(asgart_b200_ctx* ctx, const asgart_b200_chunk* chunks, int64_t n_chunks, const asgart_b200_settings* st,
                                   const void* const* d_blobs, const uint64_t* metas, int32_t n_shards, uint32_t post_mask,
                                   asgart_b200_result** out) {
    return guarded(ctx, [&]() -> int32_t {
        if (!out || !d_blobs || !metas || n_shards < 1) return fail(ctx, ASGART_B200_EINVAL, "bad finish arguments");
        *out = nullptr;
        if (!ctx->have_strand) return fail(ctx, ASGART_B200_ESTATE, "finish before load_strand");
        ChunkPlan plan;
        int rc = make_plan(ctx, chunks, n_chunks, st, plan);
        if (rc) return rc;
        u64 expect = 0, ne = 0, nm = 0;
        for (int r = 0; r < n_shards; ++r) {
            const u64 pb = metas[4 * r], pe = metas[4 * r + 1];
            if (pb != expect || pe < pb || pe > plan.total_probes || ((pb & 31) && pb != plan.total_probes) || (!d_blobs[r] && pe > pb))
                return fail(ctx, ASGART_B200_EINVAL, "partials are not the consecutive shards of this plan");
            expect = pe;
            ne += metas[4 * r + 2]; nm += metas[4 * r + 3];
        }
        if (expect != plan.total_probes) return fail(ctx, ASGART_B200_EINVAL, "partials do not cover all probes");
        cudaStream_t s = ctx->stream;
        const u64 words = ceil_div(plan.total_probes, 32);
        DevBuf<u32> d_bits(words, s), d_cnt(ne, s);
        DevBuf<u64> d_probe(ne, s), d_moff(ne, s), d_matches(nm, s);
        u64 e0 = 0, m0 = 0;
        for (int r = 0; r < n_shards; ++r) {
            const u64 pb = metas[4 * r], pe = metas[4 * r + 1], re = metas[4 * r + 2], rm = metas[4 * r + 3];
            const u64 w = ceil_div(pe - pb, 32), wbytes = ceil_div(w * 4, 8) * 8;
            const u8* p = static_cast<const u8*>(d_blobs[r]);
            if (w) CUDA_CHECK(cudaMemcpyAsync(d_bits.p + (pb >> 5), p, w * 4, cudaMemcpyDeviceToDevice, s));
            p += wbytes;
            if (re) CUDA_CHECK(cudaMemcpyAsync(d_probe.p + e0, p, re * 8, cudaMemcpyDeviceToDevice, s));
            p += re * 8;
            if (rm) CUDA_CHECK(cudaMemcpyAsync(d_matches.p + m0, p, rm * 8, cudaMemcpyDeviceToDevice, s));
            p += rm * 8;
            if (re) CUDA_CHECK(cudaMemcpyAsync(d_cnt.p + e0, p, re * 4, cudaMemcpyDeviceToDevice, s));
            e0 += re; m0 += rm;
        }
        if (ne) {
            const u32* cp = d_cnt.p; u64* mp = d_moff.p;
            device_scan<u64, SumOp>([cp] __device__(u64 e) { return u64(cp[e]); }, [mp] __device__(u64 e, u64 exc, u64) { mp[e] = exc; },
                                    ne, (u64*)nullptr, s);
        }
        asgart_b200_result* r = new asgart_b200_result();
        try {
            run_stage_b(ctx, plan, st, d_bits.p, ne, d_probe.p, d_cnt.p, d_moff.p, d_matches.p, nm, post_mask, r);
        } catch (...) { delete r; throw; }
        *out = r;
        return ASGART_B200_OK;
    });
}

int32_t asgart_b200_ctx_post_steps(asgart_b200_ctx* ctx, const uint64_t* family_offsets, int64_t n_families,
                                   const asgart_b200_protosd* sds, uint32_t post_mask, asgart_b200_result** out) {
    return guarded(ctx, [&]() -> int32_t {
        if (!out || !family_offsets || n_families < 0) return fail(ctx, ASGART_B200_EINVAL, "bad post_steps arguments");
        *out = nullptr;
        if ((post_mask & (ASGART_B200_POST_FILTER_NS | ASGART_B200_POST_COMPUTE_SCORE)) && !ctx->have_strand)
            return fail(ctx, ASGART_B200_ESTATE, "FilterNs / ComputeScore need a loaded strand");
        u64 n_fam = u64(n_families), n_sds = family_offsets[n_families];
        if (n_sds && !sds) return fail(ctx, ASGART_B200_EINVAL, "null sds");
        cudaStream_t s = ctx->stream;
        DevBuf<asgart_b200_protosd> d_sds(n_sds, s);
        DevBuf<u64> d_off(n_fam + 1, s);
        CUDA_CHECK(cudaMemcpyAsync(d_off.p, family_offsets, (n_fam + 1) * 8, cudaMemcpyHostToDevice, s));
        if (n_sds) CUDA_CHECK(cudaMemcpyAsync(d_sds.p, sds, n_sds * sizeof(asgart_b200_protosd), cudaMemcpyHostToDevice, s));
        CUDA_CHECK(cudaStreamSynchronize(s));
        run_post(ctx, d_sds, d_off, n_fam, n_sds, post_mask);
        if (post_mask & ASGART_B200_POST_COMPUTE_SCORE) run_score(ctx, d_sds, n_sds);
        asgart_b200_result* r = new asgart_b200_result();
        try { download_result(ctx, d_sds, d_off, n_fam, n_sds, r); } catch (...) { delete r; throw; }
        CUDA_CHECK(cudaStreamSynchronize(s));
        *out = r;
        return ASGART_B200_OK;
    });
}

int64_t asgart_b200_result_n_families(const asgart_b200_result* r) { return r ? int64_t(r->fam_off.size()) - 1 : 0; }
int64_t asgart_b200_result_n_sds(const asgart_b200_result* r) { return r ? int64_t(r->sds.size()) : 0; }
const uint64_t* asgart_b200_result_family_offsets(const asgart_b200_result* r) { return r ? r->fam_off.data() : nullptr; }
const asgart_b200_protosd* asgart_b200_result_sds(const asgart_b200_result* r) { return r ? r->sds.data() : nullptr; }
void asgart_b200_result_free(asgart_b200_result* r) { delete r; }

// ---- exact-match queries (locate.cuh) --------------------------------------------------------------------------
int32_t asgart_b200_ctx_locate(asgart_b200_ctx* ctx, const uint8_t* patterns, const uint64_t* offsets, int64_t n_patterns,
                               int64_t max_hits, asgart_b200_hits** out) {
    if (asgart_b200_device_count() <= 0) return ASGART_B200_ENODEVICE;
    return guarded(ctx, [&]() -> int32_t {
        if (!out) return fail(ctx, ASGART_B200_EINVAL, "null out");
        *out = nullptr;
        if (!ctx->have_index) return fail(ctx, ASGART_B200_ESTATE, "locate before build_index");
        if (n_patterns < 0 || (n_patterns > 0 && !offsets)) return fail(ctx, ASGART_B200_EINVAL, "locate: bad pattern count or null offsets");
        const u64 n = u64(n_patterns);
        for (u64 i = 0; i < n; ++i)
            if (offsets[i + 1] < offsets[i]) return fail(ctx, ASGART_B200_EINVAL, "locate: offsets are not non-decreasing");
        if (n > 0 && offsets[n] > offsets[0] && !patterns) return fail(ctx, ASGART_B200_EINVAL, "locate: null patterns");
        std::unique_ptr<asgart_b200_hits> H(new asgart_b200_hits());
        const bool ok = ctx->idx_bits == 32 ? locate_t<u32>(ctx, patterns, offsets, n, max_hits, *H)
                                            : locate_t<u64>(ctx, patterns, offsets, n, max_hits, *H);
        if (!ok) return fail(ctx, ASGART_B200_ENOMEM, "locate: the reported positions do not fit in host memory (lower max_hits)");
        *out = H.release();
        return ASGART_B200_OK;
    });
}
int64_t asgart_b200_hits_n_patterns(const asgart_b200_hits* h) { return h ? int64_t(h->first.size()) : 0; }
const int64_t* asgart_b200_hits_first(const asgart_b200_hits* h) { return h ? h->first.data() : nullptr; }
const int64_t* asgart_b200_hits_count(const asgart_b200_hits* h) { return h ? h->count.data() : nullptr; }
const uint64_t* asgart_b200_hits_offsets(const asgart_b200_hits* h) { return h ? h->offsets.data() : nullptr; }
const int64_t* asgart_b200_hits_positions(const asgart_b200_hits* h) { return h ? h->positions.data() : nullptr; }
void asgart_b200_hits_free(asgart_b200_hits* h) { delete h; }

int32_t asgart_b200_ctx_stats(const asgart_b200_ctx* ctx, asgart_b200_stats* out) {
    if (!ctx || !out) return ASGART_B200_EINVAL;
    asgart_b200_ctx* c = const_cast<asgart_b200_ctx*>(ctx);
    try {
        CUDA_CHECK(cudaSetDevice(c->device));
        fold_family_timers(c);
    } catch (const CudaError& e) {
        c->err = e.what();
        return e.code;
    }
    *out = c->st;
    return ASGART_B200_OK;
}

void asgart_b200_ctx_reset_stats(asgart_b200_ctx* ctx) {
    if (!ctx) return;
    try {
        cudaSetDevice(ctx->device);
        ctx->t_sort.reset(); ctx->t_gather.reset(); ctx->t_rank.reset(); ctx->t_probe.reset(); ctx->t_emit.reset(); ctx->t_scatter.reset(); ctx->t_scatter_main.reset();
        ctx->t_msd0.reset(); ctx->t_msd_hist.reset(); ctx->t_msd_local.reset(); ctx->t_locate.reset();
    } catch (...) {}
    ctx->launches.total = 0;
    ctx->st = asgart_b200_stats{};
    ctx->n_probe_keys = 0;
}

uint64_t asgart_b200_ctx_probe_keys(const asgart_b200_ctx* ctx) { return ctx ? ctx->n_probe_keys : 0; }

int32_t asgart_b200_ctx_timer_start(asgart_b200_ctx* ctx) {
    return guarded(ctx, [&]() -> int32_t { CUDA_CHECK(cudaEventRecord(ctx->ev_a, ctx->stream)); return ASGART_B200_OK; });
}
int32_t asgart_b200_ctx_timer_stop(asgart_b200_ctx* ctx, double* elapsed_ms) {
    return guarded(ctx, [&]() -> int32_t {
        if (!elapsed_ms) return fail(ctx, ASGART_B200_EINVAL, "null elapsed_ms");
        CUDA_CHECK(cudaEventRecord(ctx->ev_b, ctx->stream));
        CUDA_CHECK(cudaEventSynchronize(ctx->ev_b));
        float t = 0;
        CUDA_CHECK(cudaEventElapsedTime(&t, ctx->ev_a, ctx->ev_b));
        *elapsed_ms = double(t);
        return ASGART_B200_OK;
    });
}

// ---- divsufsort64 drop-in -----------------------------------------------------------------------------
int32_t asgart_b200_divsufsort64_ex(const uint8_t* T, int64_t* SA, int64_t n, int32_t device, int32_t index_bits) {
    if (!T || !SA || n < 0) return ASGART_B200_EINVAL;  // divsufsort.c:337
    if (n == 0) return ASGART_B200_OK;
    if (n == 1) { SA[0] = 0; return ASGART_B200_OK; }
    if (asgart_b200_device_count() <= 0) return ASGART_B200_ENODEVICE;
    cudaStream_t s = nullptr;
    try {
        CUDA_CHECK(cudaSetDevice(device));
        CUDA_CHECK(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
        int bits = index_bits ? index_bits : (u64(n) < 0xFFFFFFFEull ? 32 : 64);
        {
            DevBuf<u8> d_text(u64(n), s);
            CUDA_CHECK(cudaMemcpyAsync(d_text.p, T, size_t(n), cudaMemcpyHostToDevice, s));
            if (bits == 32) {
                if (u64(n) >= 0xFFFFFFFEull) { cudaStreamDestroy(s); return ASGART_B200_EINVAL; }
                DevBuf<u32> sa(u64(n), s), rank(u64(n), s);
                build_suffix_array<u32>(d_text.p, u64(n), sa.p, rank.p, s, nullptr);
                rank.release();
                download_as_i64<u32>(sa.p, SA, u64(n), s);
            } else {
                DevBuf<u64> sa(u64(n), s), rank(u64(n), s);
                build_suffix_array<u64>(d_text.p, u64(n), sa.p, rank.p, s, nullptr);
                rank.release();
                download_as_i64<u64>(sa.p, SA, u64(n), s);
            }
        }
        CUDA_CHECK(cudaStreamSynchronize(s));
        cudaStreamDestroy(s);
        return ASGART_B200_OK;
    } catch (const CudaError& e) {
        fprintf(stderr, "asgart_b200_divsufsort64: %s\n", e.what());
        cudaGetLastError();
        if (s) cudaStreamDestroy(s);
        return e.code;
    } catch (const std::bad_alloc&) {
        if (s) cudaStreamDestroy(s);
        return ASGART_B200_ENOMEM;
    }
}

int32_t asgart_b200_divsufsort64(const uint8_t* T, int64_t* SA, int64_t n) {
    int dev = 0;
    if (asgart_b200_device_count() > 0 && cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); dev = 0; }
    return asgart_b200_divsufsort64_ex(T, SA, n, dev, 0);
}

}  // extern "C"
