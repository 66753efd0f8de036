// tests/emul/emul.cpp — TEST-ONLY host build of the device logic headers (kmer_core.h, automaton_core.h).
// There is no GPU in the development container, so the arithmetic the kernels share with these headers (packed
// windows, the comparator, the literal lock-step equal range, the LUT slot, the match filters, the event/segment/death
// reformulation of the automaton) is exercised here on the CPU against the oracle. The glue below restates what the
// kernels in search.cuh / automaton.cuh do around those functions, one "thread" at a time. It is never shipped and the
// product never calls it.
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../asgart_b200/csrc/automaton_core.h"
#include "../../asgart_b200/csrc/fasta_core.h"
#include "../../asgart_b200/csrc/kmer_core.h"
#include "../../include/asgart_b200.h"

using namespace ab200;
using u64 = uint64_t;
using u32 = uint32_t;
using i64 = int64_t;

namespace {
struct Chunk { u64 c0, len, n_probes, probe_base, needle_start; };

u64 g_pack_fast_words = 0, g_pack_fast_mismatches = 0, g_pack_tab_mismatches = 0;

std::vector<u64> pack(const uint8_t* text, u64 n1, int mode) {  // pack_text_kernel, one word ("thread") per iteration
    const u64 n = n1 - 1, words = (n1 + 15) / 16 + 4, limit = mode == 0 ? n1 : n;
    std::vector<u64> P(words, 0);
    for (u64 w = 0; w < words; ++w) {
        u64 word = 0;
        for (int j = 0; j < 16; ++j) {            // the definition: byte by byte, plain switches
            const u64 p = w * 16 + j;
            u32 c = CODE_PAD;
            if (p < limit) {
                const u64 src = (mode & 2) ? (n - 1 - p) : p;
                c = code_of_byte(text[src]);
                if (mode & 1) c = complement_code(c);
                if (code_of_byte_tab(text[src], (mode & 1) ? kCodeTabComp : kCodeTab) != c) ++g_pack_tab_mismatches;   // the kernel's slow path
            }
            word |= u64(c & 15u) << (60 - 4 * j);
        }
        P[w] = word;
        // the kernel's fast path on the same 16 bytes: the five aligned words around them as the kernel loads them from its stage
        const u64 pw = w * 16;
        if (pw < limit && limit - pw >= 16) {
            const u64 low = (mode & 2) ? n - 1 - pw - 15 : pw;
            u32 W[5];
            for (int k = 0; k < 5; ++k) {
                u32 x = 0;
                for (int r = 0; r < 4; ++r) {
                    const u64 at = (low & ~u64(3)) + 4 * k + r;
                    x |= u32(at < n1 ? text[at] : uint8_t(0xAA)) << (8 * r);   // past the text: whatever the stage held
                }
                W[k] = x;
            }
            u64 fast = 0;
            if (pack16_fast(W, u32(low & 3), (mode & 2) != 0, (mode & 1) != 0, fast)) {
                ++g_pack_fast_words;
                if (fast != word) ++g_pack_fast_mismatches;
            } else {
                bool all_bases = true;                                         // the fast path may only decline what is not 16 bases
                for (int j = 0; j < 16; ++j) {
                    const uint8_t c = text[(mode & 2) ? (n - 1 - pw - j) : pw + j];
                    all_bases = all_bases && (c == 'A' || c == 'C' || c == 'G' || c == 'N' || c == 'T');
                }
                if (all_bases) ++g_pack_fast_mismatches;
            }
        }
    }
    return P;
}

struct Result { std::vector<int64_t> fam_off{0}; std::vector<u64> fields; };
}  // namespace

extern "C" {

// pack_text_kernel's two paths on an arbitrary byte string (any bytes: the error flag is not modelled, the codes are), all four
// modes: out[0] = words the fast path produced, out[1] = fast-path words differing from the byte-by-byte definition or
// declined although all 16 bytes were bases, out[2] = table-path codes differing from the switches
void emul_pack_check(const uint8_t* text, int64_t n1, uint64_t* out) {
    g_pack_fast_words = g_pack_fast_mismatches = g_pack_tab_mismatches = 0;
    for (int mode = 0; mode < 4; ++mode) pack(text, u64(n1), mode);
    out[0] = g_pack_fast_words; out[1] = g_pack_fast_mismatches; out[2] = g_pack_tab_mismatches;
}

// the branch-free byte -> code maps of the packing kernel against the plain switches, all 256 bytes: number of mismatches
int emul_code_tab_mismatches() {
    int bad = 0;
    for (u32 c = 0; c < 256; ++c) {
        bad += code_of_byte_tab(c, kCodeTab) != code_of_byte(uint8_t(c));
        bad += code_of_byte_tab(c, kCodeTabComp) != complement_code(code_of_byte(uint8_t(c)));
    }
    return bad;
}

// windows / comparator unit hooks
void emul_window(const uint8_t* text, int64_t n1, int mode, uint64_t pos, int k, uint64_t* hi, uint64_t* lo) {
    auto P = pack(text, u64(n1), mode);
    Win w = mask_window(load_window(P.data(), pos), k);
    *hi = w.hi; *lo = w.lo;
}

// lut_literal_kernel (search.cuh), one "thread" per requested pattern: (first, count) of the reference's sa_search
void emul_literal_bucket(const uint8_t* text, int64_t tsize, const uint8_t* P8, const int64_t* SA, int64_t sa_size, int64_t* first,
                         int64_t* count) {
    literal_bucket<int64_t>(text, tsize, P8, SA, sa_size, *first, *count);
}

int emul_lut(const uint8_t* text, int64_t n1, const int64_t* SA, int64_t* lo, int64_t* hi) {  // lut_build_kernel
    auto P = pack(text, u64(n1), 0);
    for (u32 s = 0; s < kLutSize; ++s) lo[s] = hi[s] = 0;
    for (u64 i = 0; i < u64(n1); ++i) {
        u32 cur = 0, prev = 0;
        const bool cur_ok = lut_slot(load_window(P.data(), u64(SA[i])).hi, cur);
        bool prev_ok = false;
        if (i > 0) prev_ok = lut_slot(load_window(P.data(), u64(SA[i - 1])).hi, prev);
        if (cur_ok && (!prev_ok || prev != cur)) lo[cur] = int64_t(i);
        if (prev_ok && (!cur_ok || prev != cur)) hi[prev] = int64_t(i);
        if (i + 1 == u64(n1) && cur_ok) hi[cur] = n1;
    }
    return 0;
}

void* emul_search(const uint8_t* text, int64_t n1_, const int64_t* SA, const asgart_b200_chunk* chunks, int64_t n_chunks,
                  const asgart_b200_settings* st, uint64_t* counters /* probes, searched, skip_n, skip_card, matches, alg */) {
    const u64 n1 = u64(n1_), n = n1 - 1, k = st->probe_size, s = k / 2;
    const int mode = (st->reverse ? 2 : 0) | (st->complement ? 1 : 0);
    auto PT = pack(text, n1, 0);
    auto PN = mode ? pack(text, n1, mode) : PT;
    std::vector<int64_t> lut_lo(kLutSize), lut_hi(kLutSize);
    emul_lut(text, n1_, SA, lut_lo.data(), lut_hi.data());
    std::vector<Chunk> ch;
    u64 base = 0;
    for (int64_t c = 0; c < n_chunks; ++c) {
        Chunk d{chunks[c].start, chunks[c].length, probes_in_chunk(chunks[c].length, k, s, st->min_duplication_length), base,
                st->reverse ? (n - chunks[c].start - chunks[c].length) : chunks[c].start};
        base += d.n_probes;
        ch.push_back(d);
    }
    const u64 total = base;
    // stage A
    std::vector<uint8_t> processed(total, 0);
    std::vector<u64> ev_probe, ev_moff, matches;
    std::vector<u32> ev_cnt;
    u64 ctr[6] = {total, 0, 0, 0, 0, 0};
    for (u64 g = 0; g < total; ++g) {
        size_t c = 0;
        while (c + 1 < ch.size() && ch[c + 1].probe_base <= g) ++c;
        const Chunk& cd = ch[c];
        const u64 i = (g - cd.probe_base + 1) * s, q = cd.needle_start + i;
        const Win pw_raw = load_window(PN.data(), q);
        if ((pw_raw.hi >> 60) == CODE_N) { ++ctr[2]; continue; }
        ++ctr[1];
        const Win pw0 = mask_window(pw_raw, k < 32 ? int(k) : 32);
        u32 slot = 0;
        u64 lstart = 0, rstart = 0;
        if (lut_slot(pw_raw.hi, slot)) { lstart = u64(lut_lo[slot]); rstart = u64(lut_hi[slot]); }
        u64 r0, r1;
        equal_range_lockstep(rstart - lstart, [&](u64 ix) -> int {
            const u64 x = u64(SA[lstart + ix]);
            if (x + k > n1) return -1;
            return cmp_kmer(PT.data(), x, PN.data(), q, int(k), pw0);
        }, r0, r1);
        if (r1 < r0) r1 = r0;
        ctr[5] += 24ull * (ceil_log2_u64(rstart - lstart + 1) + 1) + 8ull * (r1 - r0);
        std::vector<u64> surv;
        for (u64 j = lstart + r0; j < lstart + r1; ++j)
            if (match_survives(u64(SA[j]), i, cd.c0, cd.len, st->reverse != 0)) surv.push_back(u64(SA[j]));
        if (surv.size() > st->max_cardinality) { ++ctr[3]; continue; }
        processed[g] = 1;
        if (!surv.empty()) {
            ev_probe.push_back(g); ev_cnt.push_back(u32(surv.size())); ev_moff.push_back(matches.size());
            matches.insert(matches.end(), surv.begin(), surv.end());
            ctr[4] += surv.size();
        }
    }
    if (counters) memcpy(counters, ctr, sizeof ctr);
    // stage B bookkeeping (event_info_kernel / chunk_tc_kernel)
    std::vector<u64> pre(total + 1, 0);
    for (u64 g = 0; g < total; ++g) pre[g + 1] = pre[g] + processed[g];
    AutoParams P{};
    P.k = k; P.s = s; P.G = st->max_gap_size; P.min_len = st->min_duplication_length;
    const u64 qq = (P.G + P.s - 1) / P.s;
    P.q_ext = qq > 1 ? qq : 1; P.q_new = qq > 0 ? qq - 1 : 0; P.reverse = st->reverse ? 1 : 0;
    const u64 ne = ev_probe.size();
    std::vector<u64> ev_i(ne), ev_t(ne);
    std::vector<u32> ev_chunk(ne);
    std::vector<u64> seg_first;
    for (u64 e = 0; e < ne; ++e) {
        const u64 g = ev_probe[e];
        size_t c = 0;
        while (c + 1 < ch.size() && ch[c + 1].probe_base <= g) ++c;
        ev_chunk[e] = u32(c);
        ev_i[e] = (g - ch[c].probe_base + 1) * s;
        ev_t[e] = pre[g] - pre[ch[c].probe_base];
        bool head = true;
        if (e > 0 && ev_chunk[e - 1] == c) head = (ev_t[e] - ev_t[e - 1]) > P.q_ext;
        if (head) seg_first.push_back(e);
    }
    seg_first.push_back(ne);
    // automaton, one segment at a time (simulate_segment)
    Result* R = new Result();
    const u64 nm = matches.size();
    std::vector<int64_t> op(nm);
    std::vector<u64> a_ls(nm), a_le(nm), a_rs(nm), a_re(nm), a_death(nm);
    for (size_t sidx = 0; sidx + 1 < seg_first.size(); ++sidx) {
        const u64 e0 = seg_first[sidx], e1 = seg_first[sidx + 1];
        const Chunk& cd = ch[ev_chunk[e0]];
        const u64 slot0 = ev_moff[e0];
        ArmStore arms{a_ls.data() + slot0, a_le.data() + slot0, a_rs.data() + slot0, a_re.data() + slot0, a_death.data() + slot0};
        const u64 Tc = pre[cd.probe_base + cd.n_probes] - pre[cd.probe_base];
        simulate_segment(e0, e1, ev_i.data(), ev_t.data(), ev_moff.data(), ev_cnt.data(), matches.data(), op.data(), arms, P, cd.c0,
                         cd.len, Tc, [&](const SdOut& sd, bool head) {
                             if (head && !R->fields.empty()) R->fam_off.push_back(int64_t(R->fields.size() / 4));
                             R->fields.push_back(sd.left); R->fields.push_back(sd.right);
                             R->fields.push_back(sd.left_length); R->fields.push_back(sd.right_length);
                         });
    }
    if (!R->fields.empty()) R->fam_off.push_back(int64_t(R->fields.size() / 4));
    return R;
}
int64_t emul_result_n_families(void* h) { return int64_t(static_cast<Result*>(h)->fam_off.size()) - 1; }
int64_t emul_result_n_sds(void* h) { return int64_t(static_cast<Result*>(h)->fields.size() / 4); }
void emul_result_copy(void* h, int64_t* fam_off, uint64_t* fields) {
    Result* R = static_cast<Result*>(h);
    memcpy(fam_off, R->fam_off.data(), R->fam_off.size() * 8);
    if (!R->fields.empty()) memcpy(fields, R->fields.data(), R->fields.size() * 8);
}
void emul_result_free(void* h) { delete static_cast<Result*>(h); }
}


// ---------------------------------------------------------------------------------------------------------------
// GPU-side FASTA ingest (fasta_ingest.cuh), one "thread" (32 file bytes) at a time with the functions of fasta_core.h:
// classification, keep / base masks, per-thread counts exactly as the kernels use them. What the kernels do with warp
// ballots and tile-level scans — carrying the two one-bit states and the running counts from thread to thread — is a
// plain sequential carry here; the emit step restates fi_emit_kernel (records, compaction + normalisation, long N-runs
// reported by the first base after them) and the host side of ingest_fasta_device / ingest_chunks.
// Returns the number of kept bytes, or -1 when a buffer is too small.
extern "C" int64_t emul_ingest(const uint8_t* file, int64_t n_, int skip_masked, uint8_t* strand, int64_t strand_cap, uint64_t* rec_off,
                               uint64_t* rec_pos, int64_t rec_cap, int64_t* n_rec, uint64_t* chunks, int64_t chunk_cap, int64_t* n_chunks,
                               uint64_t* frag, int64_t frag_cap, int64_t* n_frag) {
    const u64 n = u64(n_);
    const u64 nthreads = (n + kFiBytes - 1) / kFiBytes;
    std::vector<FiThread> th(nthreads);
    for (u64 g = 0; g < nthreads; ++g) {   // fi_load
        FiThread& t = th[g];
        t.base = g * kFiBytes;
        t.valid = int(n - t.base < u64(kFiBytes) ? n - t.base : u64(kFiBytes));
        t.vmask = t.valid == kFiBytes ? 0xffffffffu : ((1u << t.valid) - 1u);
        for (int q = 0; q < kFiBytes / 4; ++q) {
            u32 x = 0;
            for (int r = 0; r < 4; ++r) { const int j = 4 * q + r; x |= u32(j < t.valid ? file[t.base + j] : uint8_t('\n')) << (8 * r); }
            t.w[q] = x;
        }
        fi_classify(t, (t.base == 0 || t.valid == 0) ? 1u : u32(file[t.base - 1] == '\n'));
    }
    std::vector<u32> h_in(nthreads), r_in(nthreads);
    u32 st = 0;
    for (u64 g = 0; g < nthreads; ++g) { h_in[g] = st; if (th[g].h_last != FI_NONE) st = th[g].h_last == FI_SET; }
    st = 1;
    for (u64 g = nthreads; g-- > 0;) { r_in[g] = st; if (th[g].r_first != FI_NONE) st = th[g].r_first == FI_SET; }
    std::vector<u64> roff, rpos, run_start, run_len;
    u64 outpos = 0, after_last = 0;
    for (u64 g = 0; g < nthreads; ++g) {
        const FiThread& t = th[g];
        const u32 keep = fi_keep_mask(t, h_in[g], r_in[g]);
        u32 norm[kFiBytes / 4];
        const u32 base = fi_base_mask(t, skip_masked != 0, norm);
        u64 packed;
        u32 upto;
        fi_thread_counts(t, keep, base, packed, upto);
        for (u32 m = t.heads; m; m &= m - 1) {
            const int j = fc_ffs(m) - 1;
            roff.push_back(t.base + j);
            rpos.push_back(outpos + fc_popc(keep & ((1u << j) - 1u)));
        }
        const u32 kb = keep & base;
        if (kb) {
            const u64 first_base = outpos + fc_popc(keep & ((1u << (fc_ffs(kb) - 1)) - 1u));
            const u64 len = first_base - after_last;
            if (len > kLongNRun) { run_start.push_back(after_last); run_len.push_back(len); }
        }
        u64 at = outpos;
        for (int j = 0; j < kFiBytes; ++j)
            if ((keep >> j) & 1u) {
                if (i64(at) >= strand_cap) return -1;
                strand[at++] = uint8_t(norm[j >> 2] >> ((j & 3) * 8));
            }
        if (at - outpos != (packed & 0xffffffffull) || (packed >> 32) != u64(fc_popc(t.heads))) return -2;
        if (upto) after_last = outpos + upto;
        outpos = at;
    }
    u64 kept = outpos;
    if (kept - after_last > kLongNRun) { run_start.push_back(after_last); run_len.push_back(kept - after_last); }
    if (!first_byte_ok(n, n ? file[0] : 0)) return -3;
    stop_at_empty_record(roff, rpos, kept, [&](size_t r) {
        for (u64 at = roff[r] + 1; at < n && file[at] != '\n'; ++at)
            if (!fa_space(file[at])) return false;
        return true;
    });
    if (i64(roff.size()) > rec_cap) return -1;
    for (size_t r = 0; r < roff.size(); ++r) { rec_off[r] = roff[r]; rec_pos[r] = rpos[r]; }
    *n_rec = i64(roff.size());
    std::vector<asgart_b200_chunk> ch;
    std::vector<u64> fpos, flen;
    chunks_from_runs(rpos, kept, run_start, run_len, 0, ch, fpos, flen);
    if (i64(ch.size()) > chunk_cap || i64(fpos.size()) > frag_cap) return -1;
    for (size_t c = 0; c < ch.size(); ++c) { chunks[2 * c] = ch[c].start; chunks[2 * c + 1] = ch[c].length; }
    for (size_t f = 0; f < fpos.size(); ++f) { frag[2 * f] = fpos[f]; frag[2 * f + 1] = flen[f]; }
    *n_chunks = i64(ch.size());
    *n_frag = i64(fpos.size());
    return i64(kept);
}
