// automaton.cuh — stage B kernels: processed-index bookkeeping, segment detection, the arm automaton, family
// compaction, and the post-steps FilterNs / ReOrder / ReduceOverlap / Sort (src/bin/asgart.rs:33-96, :481-562).
#pragma once
#include "automaton_core.h"
#include "common.cuh"
#include "scan.cuh"
#include "search.cuh"

namespace ab200 {

// processed index of global probe g = number of processed iterations before it (over all chunks)
__device__ __forceinline__ u64 processed_before(const u32* __restrict__ bits, const u64* __restrict__ wpre, u64 g) {
    const u64 w = g >> 5;
    const u32 r = u32(g & 31u);
    u64 t = wpre[w];
    if (r) t += __popc(bits[w] & ((1u << r) - 1u));
    return t;
}

// per event: chunk, needle-local i, chunk-relative processed index t, segment-head flag
__global__ void event_info_kernel(const u64* __restrict__ ev_probe, u64 n_events, const ChunkDev* __restrict__ chunks,
                                  u32 n_chunks, const u32* __restrict__ bits, const u64* __restrict__ wpre, u32 s, u64 q_ext,
                                  u64* __restrict__ ev_i, u64* __restrict__ ev_t, u32* __restrict__ ev_chunk,
                                  u8* __restrict__ ev_head) {
    const u64 e = u64(blockIdx.x) * blockDim.x + threadIdx.x;
    if (e >= n_events) return;
    const u64 g = ev_probe[e];
    const u32 c = chunk_of_probe(chunks, n_chunks, g);
    const u64 base_t = processed_before(bits, wpre, chunks[c].probe_base);
    const u64 t = processed_before(bits, wpre, g) - base_t;
    bool head = true;
    if (e > 0) {
        const u64 gp = ev_probe[e - 1];
        const u32 cp = chunk_of_probe(chunks, n_chunks, gp);
        if (cp == c) {
            const u64 tp = processed_before(bits, wpre, gp) - base_t;
            head = (t - tp) > q_ext;  // every arm is inactive and flushed before t: hard reset
        }
    }
    ev_i[e] = (g - chunks[c].probe_base + 1) * u64(s);
    ev_t[e] = t;
    ev_chunk[e] = c;
    ev_head[e] = head ? 1 : 0;
}

struct AutoBuffers {
    const u64* ev_i;
    const u64* ev_t;
    const u64* ev_moff;
    const u32* ev_cnt;
    const u32* ev_chunk;
    const u64* seg_first;  // n_segments + 1 entries (last = n_events)
    const u64* matches;
    i64* op_target;
    u64 *a_ls, *a_le, *a_rs, *a_re;  // arm store, indexed like matches
    // active list of the warp kernel (arms that can still be extended), same capacity, creation order preserved
    u32* act_arm;   // index into the segment's arm store
    u64* act_ls;
    u64* act_wlo;   // a match at ms extends the arm iff wlo <= ms < whi (and the arm is active):
    u64* act_whi;   //   wlo = right.end - k + 1, whi = right.end + max(G, trunc(0.1 * left length))   (see arm_window)
    u64* act_death;
    asgart_b200_protosd* out_sd;               // slot array, indexed like matches
    u8* out_flag;                              // 0 empty, 1 duplicon, 3 duplicon that opens a family
    const u64* chunk_tc;                       // processed iterations per chunk
    const ChunkDev* chunks;
};

// One warp per segment. Same event-driven semantics as simulate_segment (automaton_core.h), with the work of one
// event spread over the lanes:
//   phase 1  lane = match: scan the active arms in creation order for the first one the match extends (snapshot
//            semantics: nothing is modified until every match has been classified)          src/automaton.rs:122-134
//   phase 2  ExtendArm ops: per arm the last match in SA order wins (__match_any_sync picks it)              :136-143
//   phase 3  NewArm ops appended in match order (ballot + prefix popcount)                                   :145-163
// Arms that can no longer be extended (death < t) are dropped from the active list by an order-preserving warp
// compaction; the arm store keeps every arm of the open family for the flush (:182-200).
// The critical path is the longest segment (a 50 kbp duplication = 5000 events in sequence), so per-event latency is
// what matters: the active list lives in shared memory (it moves to its global slice only beyond kActCap arms, until
// the next flush), and the first match of every event is prefetched together with the batch of 32 event records.
// Segments whose matches add up to kHeavySegment or more get a whole block of kHeavyWarps warps: warp 0 runs the event loop
// exactly as in the one-warp case and wakes the helper warps (named barriers 1/2) only for events whose
// matches x active-arms product is large; phase 1 of such an event is then spread over all warps. The named barriers are
// the non-aligned form (barrier.sync, not bar.sync): warp 0 reaches them from inside its data-dependent event loop, where
// the compiler need not have reconverged the lanes (compute-sanitizer synccheck flags the aligned form there).
constexpr int kActCapLight = 128;
constexpr int kActCapHeavy = 768;
constexpr int kHeavyWarps = 8;
constexpr u64 kHeavySegment = 512;
constexpr u64 kHeavyEvent = 4096;  // cnt * active arms

struct AutoCmd {
    u64 t, m0, snap;
    u32 cnt, op;  // op: 1 = classify matches, 0 = exit
    u32 in_smem;
};

// try_extend_arms (src/automaton.rs:66-85) as a window test. With m.end > a.right.end, d_ss (:207-216) is 0 when
// m.start <= a.right.end and m.start - a.right.end otherwise (arms are at least k long), so
//   d_ss(a.right, m) < thr  and  m.end > a.right.end    <=>    a.right.end - k < m.start < a.right.end + thr,
// thr = max(G, trunc(0.1 * left length)) > 0 (:69, the f64 product truncated like `as i64`).
__device__ __forceinline__ void arm_window(u64 re, u64 left_len, u64 k, i64 G, u64& wlo, u64& whi) {
    const i64 tenth = i64(0.1 * double(left_len));
    wlo = re - k + 1;
    whi = re + u64(G > tenth ? G : tenth);
}

template <int W, int CAP>
__global__ void __launch_bounds__(W * 32) automaton_segment_kernel(AutoBuffers B, AutoParams P, u64 n_segments, u64 n_matches, u64 n_events,
                                                                   u32 reversed_flag, u32 complemented_flag) {
    __shared__ u64 s_wlo[CAP], s_whi[CAP], s_ls[CAP], s_death[CAP];
    __shared__ u32 s_arm[CAP];
    __shared__ AutoCmd s_cmd;
    const u64 sidx = blockIdx.x;
    if (sidx >= n_segments) return;
    const u64 e0 = B.seg_first[sidx], e1 = B.seg_first[sidx + 1];
    const u64 slot0 = B.ev_moff[e0];
    const u64 seg_matches = (e1 < n_events ? B.ev_moff[e1] : n_matches) - slot0;
    if ((W > 1) != (seg_matches >= kHeavySegment)) return;  // the other launch owns this segment (whole block leaves)
    const unsigned lane = lane_id();
    const unsigned warp = threadIdx.x >> 5;
    const unsigned lt = lanemask_lt();
    const unsigned FULL = 0xffffffffu;
    const u64* matches = B.matches;
    i64* op_target = B.op_target;
    u32* g_arm = B.act_arm + slot0; u64* g_wlo = B.act_wlo + slot0; u64* g_whi = B.act_whi + slot0; u64* g_ls = B.act_ls + slot0;
    u64* g_death = B.act_death + slot0;

    // classify matches [r_begin, cnt) step r_step*32 of one event against the snapshot of the active list
    auto classify = [&](u64 t, u64 m0, u32 cnt, u64 snap, bool smem, u32 w_first, u32 w_step) {
        const u64* c_wlo = smem ? s_wlo : g_wlo; const u64* c_whi = smem ? s_whi : g_whi;
        const u64* c_death = smem ? s_death : g_death;
        for (u32 r0 = w_first * 32; r0 < cnt; r0 += w_step * 32) {
            const u32 r = r0 + lane;
            const bool valid = r < cnt;
            const u64 ms = valid ? matches[m0 + r] : 0;
            i64 target = -1;
            bool searching = valid;
            for (u64 a = 0; a < snap; ++a) {
                if (__ballot_sync(FULL, searching) == 0) break;
                if (searching && ms >= c_wlo[a] && ms < c_whi[a] && c_death[a] >= t) { target = i64(a); searching = false; }
            }
            if (valid) op_target[m0 + r] = target;
        }
    };

    if (W > 1 && warp > 0) {  // helper warps
        for (;;) {
            asm volatile("barrier.sync 1, %0;" ::"r"(W * 32) : "memory");
            const AutoCmd cmd = s_cmd;
            if (cmd.op == 0) return;
            classify(cmd.t, cmd.m0, cmd.cnt, cmd.snap, cmd.in_smem != 0, warp, W);
            asm volatile("barrier.sync 2, %0;" ::"r"(W * 32) : "memory");
        }
    }

    // ---- warp 0: the event loop
    const u32 c = B.ev_chunk[e0];
    const ChunkDev ch = B.chunks[c];
    const u64 Tc = B.chunk_tc[c];
    u64* a_ls = B.a_ls + slot0; u64* a_le = B.a_le + slot0; u64* a_rs = B.a_rs + slot0; u64* a_re = B.a_re + slot0;
    u32* act_arm = s_arm; u64* act_wlo = s_wlo; u64* act_whi = s_whi; u64* act_ls = s_ls; u64* act_death = s_death;
    bool in_smem = true;
    u64 n_arms = 0, fam_start = 0, n_act = 0, max_death = 0, act_min_death = ~u64(0), cursor = slot0;
    const i64 Gi = i64(P.G);
    bool chain_live = false;                        // the previous event had one match and it went to the first active arm
    u64 last_t = 0, last_ms = 0; u32 last_cnt = 0;   // last event of the previous batch of 32
    u64 new_wlo_off, new_whi_off;   // window of a fresh arm relative to its match start: [ms + 1, ms + k + thr(k))
    {
        u64 wl, wh;
        arm_window(P.k, P.k, P.k, Gi, wl, wh);
        new_wlo_off = wl; new_whi_off = wh;   // computed for ms = 0: re = k
    }

    auto to_smem = [&]() {
        act_arm = s_arm; act_wlo = s_wlo; act_whi = s_whi; act_ls = s_ls; act_death = s_death;
        in_smem = true;
    };
    auto to_global = [&]() {  // copy the live entries to the segment's global slice and continue there
        for (u64 a = lane; a < n_act; a += 32) {
            g_arm[a] = act_arm[a]; g_wlo[a] = act_wlo[a]; g_whi[a] = act_whi[a]; g_ls[a] = act_ls[a]; g_death[a] = act_death[a];
        }
        act_arm = g_arm; act_wlo = g_wlo; act_whi = g_whi; act_ls = g_ls; act_death = g_death;
        in_smem = false;
        __syncwarp();
    };

    auto flush = [&]() {
        bool first = true;
        for (u64 base = fam_start; base < n_arms; base += 32) {
            const u64 a = base + lane;
            bool ok = false;
            u64 rl = 0, ll = 0;
            if (a < n_arms) { rl = a_re[a] - a_rs[a]; ll = a_le[a] - a_ls[a]; ok = rl >= P.min_len; }
            const unsigned m = __ballot_sync(FULL, ok);
            if (ok) {
                const u64 slot = cursor + __popc(m & lt);
                asgart_b200_protosd o;
                o.left = P.reverse ? (ch.c0 + ch.len - a_ls[a] - ll) : (a_ls[a] + ch.c0);
                o.right = a_rs[a];
                o.left_length = ll; o.right_length = rl;
                o.identity = 0.f;
                o.reversed = u8(reversed_flag); o.complemented = u8(complemented_flag);
                o._pad[0] = o._pad[1] = 0;
                B.out_sd[slot] = o;
                B.out_flag[slot] = (first && (m & lt) == 0) ? 3 : 1;
            }
            if (m) { first = false; cursor += __popc(m); }
        }
        fam_start = n_arms;
        n_act = 0;
        max_death = 0;
        act_min_death = ~u64(0);
        to_smem();
        __syncwarp();
    };

    auto compact = [&](u64 t) {  // drop arms with death < t, keep order; recompute the exact minimum death
        u64 w = 0, mn = ~u64(0);
        for (u64 base = 0; base < n_act; base += 32) {
            const u64 a = base + lane;
            u32 arm = 0; u64 wlo = 0, whi = 0, ls = 0, death = 0;
            bool keep = false;
            if (a < n_act) {
                arm = act_arm[a]; wlo = act_wlo[a]; whi = act_whi[a]; ls = act_ls[a]; death = act_death[a];
                keep = death >= t;
            }
            const unsigned m = __ballot_sync(FULL, keep);
            __syncwarp();  // all reads of this block of 32 done before anyone overwrites (w <= base)
            if (keep) {
                const u64 d = w + __popc(m & lt);
                act_arm[d] = arm; act_wlo[d] = wlo; act_whi[d] = whi; act_ls[d] = ls; act_death[d] = death;
                mn = death < mn ? death : mn;
            }
            w += __popc(m);
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) { const u64 o = __shfl_xor_sync(FULL, mn, d); mn = o < mn ? o : mn; }
        n_act = w;
        act_min_death = mn;
        __syncwarp();
    };

    // ExtendArm applied to active entry a (:136-143)
    auto extend = [&](u64 a, u64 i, u64 ms, u64 t) {
        const u32 arm = act_arm[a];
        const u64 le = i + P.k, re = ms + P.k;
        a_le[arm] = le; a_re[arm] = re;
        u64 wl, wh;
        arm_window(re, le - act_ls[a], P.k, Gi, wl, wh);
        act_wlo[a] = wl; act_whi[a] = wh;
        act_death[a] = t + P.q_ext;
    };

    for (u64 eb = e0; eb < e1; eb += 32) {
        u64 my_t = 0, my_i = 0, my_moff = 0, my_m0 = 0; u32 my_cnt = 0;
        if (eb + lane < e1) {
            my_t = B.ev_t[eb + lane]; my_i = B.ev_i[eb + lane]; my_moff = B.ev_moff[eb + lane]; my_cnt = B.ev_cnt[eb + lane];
            my_m0 = matches[my_moff];
        }
        const int nev = int(min(u64(32), e1 - eb));
        // Chain test, independent of the automaton's state: event e "chains" when it and its predecessor carry one match
        // each and, provided the predecessor extended (or created) some arm, that arm is still active at e and e's match
        // falls into its window: t_e <= t_(e-1) + q_new and ms_(e-1) < ms_e < ms_(e-1) + k + G (the arm's true window is
        // at least this wide). If that arm is the first of the active list it wins the match whatever else is active, the
        // event changes nothing else, and a run of chained events collapses into its last one.
        unsigned chain_mask;
        {
            u64 p_t = __shfl_up_sync(FULL, my_t, 1), p_ms = __shfl_up_sync(FULL, my_m0, 1);
            u32 p_cnt = __shfl_up_sync(FULL, my_cnt, 1);
            if (lane == 0) { p_t = last_t; p_ms = last_ms; p_cnt = last_cnt; }
            const bool ch_ok = eb + lane < e1 && my_cnt == 1 && p_cnt == 1 && my_t <= p_t + P.q_new && my_m0 > p_ms &&
                               my_m0 < p_ms + P.k + P.G;
            chain_mask = __ballot_sync(FULL, ch_ok);
            last_t = __shfl_sync(FULL, my_t, 31); last_ms = __shfl_sync(FULL, my_m0, 31); last_cnt = __shfl_sync(FULL, my_cnt, 31);
        }
        for (int j = 0; j < nev; ++j) {
            if (chain_live && ((chain_mask >> j) & 1u)) {
                // run of chained events starting at j: only the last one leaves a trace (on the first active arm)
                const unsigned rest = ~(chain_mask >> j);
                const int run = rest ? (__ffs(rest) - 1) : (32 - j);
                const int last = j + run - 1;
                const u64 t = __shfl_sync(FULL, my_t, last), i = __shfl_sync(FULL, my_i, last), ms = __shfl_sync(FULL, my_m0, last);
                if (lane == 0) extend(0, i, ms, t);
                if (t + P.q_ext > max_death) max_death = t + P.q_ext;
                __syncwarp();
                j = last;
                continue;
            }
            const u64 t = __shfl_sync(FULL, my_t, j), i = __shfl_sync(FULL, my_i, j), m0 = __shfl_sync(FULL, my_moff, j);
            const u64 first_ms = __shfl_sync(FULL, my_m0, j);
            const u32 cnt = __shfl_sync(FULL, my_cnt, j);
            if (n_arms > fam_start && max_death < t) flush();
            if (n_act > 0 && act_min_death < t) compact(t);
            if (in_smem && n_act + cnt > CAP) to_global();
            if (cnt == 1) {
                // fast path (9 events in 10): one match, lanes = active arms, first hit in creation order by ballot
                const u64 ms = first_ms;
                i64 target = -1;
                for (u64 base = 0; base < n_act; base += 32) {
                    const u64 a = base + lane;
                    bool hit = false;
                    if (a < n_act) hit = ms >= act_wlo[a] && ms < act_whi[a] && act_death[a] >= t;
                    const unsigned m = __ballot_sync(FULL, hit);
                    if (m) { target = i64(base) + (__ffs(m) - 1); break; }
                }
                __syncwarp();   // every lane has read its entries before lane 0 rewrites the winner (racecheck: WAR)
                if (target >= 0) {
                    if (lane == 0) extend(u64(target), i, ms, t);
                    if (t + P.q_ext > max_death) max_death = t + P.q_ext;
                } else {
                    if (lane == 0) {
                        a_ls[n_arms] = i; a_le[n_arms] = i + P.k; a_rs[n_arms] = ms; a_re[n_arms] = ms + P.k;
                        act_arm[n_act] = u32(n_arms); act_wlo[n_act] = ms + new_wlo_off; act_whi[n_act] = ms + new_whi_off; act_ls[n_act] = i;
                        act_death[n_act] = t + P.q_new;
                    }
                    target = i64(n_act);
                    ++n_arms; ++n_act;
                    if (t + P.q_new > max_death) max_death = t + P.q_new;
                    if (t + P.q_new < act_min_death) act_min_death = t + P.q_new;
                }
                chain_live = target == 0;
                __syncwarp();
                continue;
            }
            chain_live = false;
            const u64 snap = n_act;
            const bool single = cnt <= 32;
            i64 my_target = -1;
            u64 my_ms = 0;
            // phase 1
            if (single) {
                const bool valid = lane < cnt;
                const u64 ms = valid ? matches[m0 + lane] : 0;
                bool searching = valid;
                for (u64 a = 0; a < snap; ++a) {
                    if (__ballot_sync(FULL, searching) == 0) break;
                    if (searching && ms >= act_wlo[a] && ms < act_whi[a] && act_death[a] >= t) { my_target = i64(a); searching = false; }
                }
                my_ms = ms;
            } else if (W > 1 && u64(cnt) * snap >= kHeavyEvent) {
                if (lane == 0) { s_cmd.t = t; s_cmd.m0 = m0; s_cmd.snap = snap; s_cmd.cnt = cnt; s_cmd.op = 1; s_cmd.in_smem = in_smem ? 1 : 0; }
                __syncwarp();
                asm volatile("barrier.sync 1, %0;" ::"r"(W * 32) : "memory");
                classify(t, m0, cnt, snap, in_smem, 0, W);
                asm volatile("barrier.sync 2, %0;" ::"r"(W * 32) : "memory");
            } else {
                classify(t, m0, cnt, snap, in_smem, 0, 1);
            }
            __syncwarp();
            // phase 2: extends, last match per arm wins
            bool any_ext = false, any_new = false;
            for (u32 r0 = 0; r0 < cnt; r0 += 32) {
                const u32 r = r0 + lane;
                const bool valid = r < cnt;
                i64 target = -1; u64 ms = 0;
                if (single) { target = my_target; ms = my_ms; }
                else if (valid) { target = op_target[m0 + r]; ms = matches[m0 + r]; }
                const bool ext = valid && target >= 0;
                const unsigned any = __ballot_sync(FULL, ext);
                if (any) {
                    const unsigned peers = __match_any_sync(FULL, ext ? target : i64(-1) - i64(lane));
                    if (ext && (31 - __clz(peers)) == int(lane)) extend(u64(target), i, ms, t);
                    any_ext = true;
                    __syncwarp();  // a later round may extend the same arm again: keep rounds ordered
                }
            }
            // phase 3: new arms in match order
            for (u32 r0 = 0; r0 < cnt; r0 += 32) {
                const u32 r = r0 + lane;
                const bool valid = r < cnt;
                i64 target = 0; u64 ms = 0;
                if (single) { target = my_target; ms = my_ms; }
                else if (valid) { target = op_target[m0 + r]; ms = matches[m0 + r]; }
                const bool isnew = valid && target < 0;
                const unsigned m = __ballot_sync(FULL, isnew);
                if (isnew) {
                    const u64 off = __popc(m & lt);
                    const u64 arm = n_arms + off, a = n_act + off;
                    a_ls[arm] = i; a_le[arm] = i + P.k; a_rs[arm] = ms; a_re[arm] = ms + P.k;
                    act_arm[a] = u32(arm); act_wlo[a] = ms + new_wlo_off; act_whi[a] = ms + new_whi_off; act_ls[a] = i;
                    act_death[a] = t + P.q_new;
                }
                if (m) { any_new = true; n_arms += __popc(m); n_act += __popc(m); }
            }
            if (any_ext && t + P.q_ext > max_death) max_death = t + P.q_ext;
            if (any_new) {
                if (t + P.q_new > max_death) max_death = t + P.q_new;
                if (t + P.q_new < act_min_death) act_min_death = t + P.q_new;
            }
            __syncwarp();
        }
    }
    if (n_arms > fam_start && max_death + 1 <= Tc) flush();
    if (W > 1) {  // release the helpers
        if (lane == 0) s_cmd.op = 0;
        __syncwarp();
        asm volatile("barrier.sync 1, %0;" ::"r"(W * 32) : "memory");
    }
}

// ------------------------------------------------------------------------------------------------ post-steps
// FilterNs: count of N over strand[p ..= p+len] for both arms (src/structs.rs:454-467), one block per duplicon
// An arm whose inclusive range passes the end of the strand (n1 bytes, '$' included) makes the reference panic on the slice
// (src/structs.rs:455-466); here it raises *oob and the duplicon is left alone — nothing is read out of bounds.
__global__ void __launch_bounds__(256) n_content_kernel(const u8* __restrict__ text, u64 n1, const asgart_b200_protosd* __restrict__ sds,
                                                        u64 n_sds, u8* __restrict__ keep, u32* __restrict__ oob) {
    __shared__ u64 s_l[8], s_r[8];
    const u64 j = blockIdx.x;
    if (j >= n_sds) return;
    const asgart_b200_protosd sd = sds[j];
    if (sd.left >= n1 || sd.left_length >= n1 - sd.left || sd.right >= n1 || sd.right_length >= n1 - sd.right) {
        if (threadIdx.x == 0) { keep[j] = 0; atomicOr(oob, 1u); }
        return;
    }
    u64 cl = 0, cr = 0;
    for (u64 p = sd.left + threadIdx.x; p <= sd.left + sd.left_length; p += 256) { u8 c = text[p]; cl += (c == 'N' || c == 'n'); }
    for (u64 p = sd.right + threadIdx.x; p <= sd.right + sd.right_length; p += 256) { u8 c = text[p]; cr += (c == 'N' || c == 'n'); }
    cl = warp_sum_u64(cl);
    cr = warp_sum_u64(cr);
    if (lane_id() == 0) { s_l[threadIdx.x >> 5] = cl; s_r[threadIdx.x >> 5] = cr; }
    __syncthreads();
    if (threadIdx.x == 0) {
        cl = cr = 0;
        for (int w = 0; w < 8; ++w) { cl += s_l[w]; cr += s_r[w]; }
        const float l = float(cl) / float(sd.left_length);   // f32 arithmetic like the reference
        const float r = float(cr) / float(sd.right_length);
        keep[j] = fmaxf(l, r) <= 0.2f ? 1 : 0;
    }
}

__device__ __forceinline__ bool subsegment_d(u64 xs, u64 xl, u64 ys, u64 yl) { return xs >= ys && xs + xl <= ys + yl; }
__device__ __forceinline__ bool overlap_d(u64 xs, u64 xl, u64 ys, u64 yl) {
    const u64 xe = xs + xl, ye = ys + yl;
    return (xs >= ys && xs <= ye && xe >= ye) || (ys >= xs && ys <= xe && ye >= xe);
}

// one pass of _reduce (src/bin/asgart.rs:516-551) in place over f[0..n): returns the new length
__device__ u64 reduce_once_d(asgart_b200_protosd* f, u64 n) {
    u64 m = 0;  // `news` = f[0..m); m <= index of the element being inserted, so in-place is safe
    for (u64 r = 0; r < n; ++r) {
        const asgart_b200_protosd x = f[r];
        bool absorbed = false;
        for (u64 w = 0; w < m; ++w) {
            asgart_b200_protosd& y = f[w];
            if (subsegment_d(x.left, x.left_length, y.left, y.left_length) &&
                subsegment_d(x.right, x.right_length, y.right, y.right_length)) { absorbed = true; break; }
            if (subsegment_d(y.left, y.left_length, x.left, x.left_length) &&
                subsegment_d(y.right, y.right_length, x.right, x.right_length)) {
                y.left = x.left; y.right = x.right; y.left_length = x.left_length; y.right_length = x.right_length;
                absorbed = true; break;
            }
            if (overlap_d(x.left, x.left_length, y.left, y.left_length) &&
                overlap_d(x.right, x.right_length, y.right, y.right_length)) {
                // merge (src/bin/asgart.rs:497-513) with its mixed-up lengths (quirk Q5)
                const u64 nl = min(x.left, y.left);
                const u64 ls = max(x.left + x.left_length, y.left + y.right_length) - nl;
                const u64 nr = min(x.right, y.right);
                const u64 rs = max(x.right + x.left_length, y.right + y.right_length) - nr;
                y.left = nl; y.right = nr; y.left_length = ls; y.right_length = rs;
                absorbed = true; break;
            }
        }
        if (!absorbed) { f[m] = x; ++m; }
    }
    return m;
}

// per family (v1: one thread each): drop filtered duplicons, ReOrder, ReduceOverlap to fixpoint, stable Sort by left
__global__ void post_family_kernel(asgart_b200_protosd* __restrict__ sds, const u64* __restrict__ fam_off, u64 n_fam,
                                   const u8* __restrict__ keep, u32 post_mask, u64* __restrict__ new_count) {
    const u64 fidx = u64(blockIdx.x) * blockDim.x + threadIdx.x;
    if (fidx >= n_fam) return;
    const u64 b = fam_off[fidx], e = fam_off[fidx + 1];
    asgart_b200_protosd* f = sds + b;
    u64 n = e - b;
    if (post_mask & ASGART_B200_POST_FILTER_NS) {
        u64 m = 0;
        for (u64 r = 0; r < n; ++r)
            if (keep[b + r]) { if (m != r) f[m] = f[r]; ++m; }
        n = m;
    }
    if (post_mask & ASGART_B200_POST_REORDER)
        for (u64 r = 0; r < n; ++r)
            if (f[r].left > f[r].right) { const u64 t = f[r].left; f[r].left = f[r].right; f[r].right = t; }  // positions only (Q4)
    if (post_mask & ASGART_B200_POST_REDUCE_OVERLAP) {
        u64 old_size = n;
        u64 cur = reduce_once_d(f, n);
        while (cur < old_size) { old_size = cur; cur = reduce_once_d(f, cur); }
        n = cur;
    }
    if (post_mask & ASGART_B200_POST_SORT) {  // insertion sort is stable, like sort_by
        for (u64 r = 1; r < n; ++r) {
            const asgart_b200_protosd x = f[r];
            u64 w = r;
            while (w > 0 && f[w - 1].left > x.left) { f[w] = f[w - 1]; --w; }
            f[w] = x;
        }
    }
    new_count[fidx] = n;
}

}  // namespace ab200
