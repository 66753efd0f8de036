// sa_group.h — the group of devices that build one suffix array together (sharded SA build, sa_build.cuh).
//
// The reference builds its suffix array on one CPU thread (r_divsufsort, src/bin/asgart.rs:473-479) and has no
// distributed mode; this is the multi-GPU side of the replacement. Member r of a group of `world` devices owns
//   * the suffixes whose initial key falls into its key range = one contiguous range of the final suffix array, and
//   * every world-th block of the rank array (RankView): ranks are written to and gathered from the owners'
//     memory directly (peer stores / loads over NVLink), there is no staging copy.
// Collectives are only needed at phase boundaries (a few per doubling round) and for the final exchange of SA pieces.
// Two back ends: ThreadGroup (members = host threads of one process, any devices with peer access; also how the sharded
// build is tested on a single GPU) and NcclGroup (one process per GPU: NCCL for the collectives, CUDA IPC for the peer
// pointers) — both in dist_group.cuh.
#pragma once
#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>

namespace ab200 {

constexpr int kMaxWorld = 16;

struct SaGroup {
    int rank = 0, world = 1;
    // Sum of host values over the members. Every member calls it after synchronising its stream, so when it returns all
    // device work issued before it — on every member, including stores into peer memory — is complete and visible.
    virtual void allreduce_sum_host(uint64_t* vals, int n) = 0;
    void barrier() { uint64_t z = 0; allreduce_sum_host(&z, 1); }
    // element-wise maximum of a device array over the members (elem_bytes 4 or 8, unsigned); stream-ordered on return
    virtual void allreduce_max_dev(void* buf, size_t count, int elem_bytes, cudaStream_t stream) = 0;
    // member s holds elements [offs[s], offs[s+1]) of the array at `base`; afterwards every member holds all of it
    virtual void share_pieces(void* base, const uint64_t* offs, int elem_bytes, cudaStream_t stream) = 0;
    // pointers through which this member's kernels can reach every member's buffer (`mine` = start of a cudaMalloc block)
    virtual void exchange_ptr(void* mine, size_t bytes, void** all) = 0;
    virtual ~SaGroup() = default;
};

// Rank array of the suffix-array build, one contiguous slice per member. Positions come in regions of 2^g (at most 256
// regions; g >= 16), member r owns regions [r k, (r + 1) k), k = ceil(regions / world): slices are balanced to one region,
// and ptr() finds a position's owner with a shift and a 32-bit divide (every rank store and gather of the build goes
// through it). world == 1 is the plain array.
template <typename IdxT>
struct RankView {
    IdxT* base[kMaxWorld];
    uint32_t world;
    uint32_t g;   // region shift
    uint32_t k;   // regions per member
    __host__ __device__ __forceinline__ IdxT* ptr(uint64_t p) const {
        if (world == 1) return base[0] + p;
        const uint32_t o = uint32_t(p >> g) / k;
        return base[o] + (p - ((uint64_t(o) * k) << g));
    }
    static RankView single(IdxT* p) {
        RankView v;
        for (int i = 0; i < kMaxWorld; ++i) v.base[i] = p;
        v.world = 1;
        v.g = 16;
        v.k = 1;
        return v;
    }
    // region shift: at most 256 regions of at least 2^16 positions
    static uint32_t pick_g(uint64_t n) {
        int bits = 0;
        for (uint64_t v = n ? n - 1 : 0; v; v >>= 1) ++bits;
        return bits <= 16 ? 16u : uint32_t(16 + 8 * ((bits - 17) / 8));
    }
    static uint32_t pick_k(uint64_t n, uint32_t world, uint32_t g) {
        const uint64_t regions = (n + (uint64_t(1) << g) - 1) >> g;
        const uint64_t k = (regions + world - 1) / world;
        return uint32_t(k ? k : 1);
    }
    // positions a member must hold
    uint64_t slice_len() const { return uint64_t(k) << g; }
};

}  // namespace ab200
