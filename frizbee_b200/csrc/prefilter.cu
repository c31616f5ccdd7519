// prefilter.cu — stage 1 of match_list: length gate → ordered char-mask prefilter → window trim
// → survivor records.
//
// Reference path replaced (per haystack, src/matcher/algo.rs:85-100):
//     if len >= min_haystack_len { (matched,start,end) = prefilter_haystack(..); trim_haystack(..) }
// with Prefilter::match_haystack (src/prefilter/algo/ascii.rs:6-54), match_haystack_1_typo /
// _2_typos / _many_typos (src/prefilter/algo/ascii_typos.rs:15-360) and trim_haystack
// (src/matcher/algo.rs:331-338).  Literal modes (src/literal/algo.rs:234-255) are decided here too.
//
// Structure (persistent, warp-autonomous, no block barriers — the first version synchronised a
// block per tile and spent 65% of its issue slots waiting at barriers, profiles/r01a_*):
//   phase A  warp per group, lane per haystack: length gate + the byte-class SIGNATURE test (8 bytes per
//            haystack, written at pack time — pack.cu: k_pack_sig): "at most k needle bytes lack a partner
//            in this haystack", a necessary condition of every prefilter of the reference.  The haystack bytes
//            are not read for rejected haystacks.  Passing lanes queue in the warp's shared-memory ring.
//            (Rounds 1's phase A streamed every haystack byte through word-parallel probes: 0.35 of the HBM
//            roofline, ALU-issue-bound; the signature test reads 12 bytes per haystack instead of len + 8.)
//   phase B  whenever 32 candidates are queued: lane per candidate, the exact reference window
//            (chunk-emulating for k >= 1) from occurrence masks of the candidate's bytes, all lanes busy.
//   emit     survivors go to per-SW-class lists (warp-aggregated atomics) and set their bit in a
//            per-tile bitmap; k_tile_rank turns the bitmap into index-order ranks so that the
//            scoring stage can write each match straight to its index-ordered position.
#include "frz_device.cuh"
#include <cuda_pipeline.h>
#include <algorithm>

#include "frz_host.h"
#include "indices_path.cuh"
#include "prefilter_masks.cuh"

namespace {

using namespace frzpf;

constexpr int kThreads = 128;
constexpr int kWarps = kThreads / 32;

struct GlobalAcc {
    const uint4* base;  // unit 0 of this slot; its units (and so its bytes) are contiguous
    __device__ __forceinline__ uint32_t word(uint32_t w) const { return reinterpret_cast<const uint32_t*>(base)[w]; }
};


// first position in [from, to) whose byte b satisfies (b | om) == tg, else -1
template <class A>
__device__ __forceinline__ int find_first(const A& a, uint32_t om4, uint32_t tg4, int from, int to) {
    if (from >= to) return -1;
    int w = from >> 2;
    const int wend = (to + 3) >> 2;
    uint32_t x = (a.word(w) | om4) ^ tg4;
    x |= (1u << ((from & 3) * 8)) - 1;  // bytes below `from` can never look like a hit
    for (;;) {
        // lowest flagged byte is always a true zero byte (borrows only travel upwards)
        uint32_t z = (x - 0x01010101u) & ~x & 0x80808080u;
        if (z) {
            int p = w * 4 + ((__ffs(z) - 1) >> 3);
            return p < to ? p : -1;
        }
        if (++w >= wend) return -1;
        x = (a.word(w) | om4) ^ tg4;
    }
}

__device__ __forceinline__ uint32_t zero_bytes_exact(uint32_t x) {
    return ~(((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x | 0x7f7f7f7fu);  // 0x80 in every zero byte
}

// last position in [from, to) matching either probe (om1,tg1) or (om2,tg2), else -1
template <class A>
__device__ __forceinline__ int find_last2(const A& a, uint32_t om1, uint32_t tg1, uint32_t om2, uint32_t tg2, int from, int to) {
    if (from >= to) return -1;
    int w = (to - 1) >> 2;
    const int w0 = from >> 2;
    for (;;) {
        uint32_t v = a.word(w);
        uint32_t z = zero_bytes_exact((v | om1) ^ tg1) | zero_bytes_exact((v | om2) ^ tg2);
        int lo = w * 4;
        if (to - lo < 4) z &= (1u << ((to - lo) * 8)) - 1;          // drop bytes >= to
        if (from > lo) z &= ~((1u << ((from - lo) * 8)) - 1);       // drop bytes < from
        if (z) return lo + ((31 - __clz(z)) >> 3);
        if (--w < w0) return -1;
    }
}

struct Probe {
    uint32_t om, tg;
};
__device__ __forceinline__ Probe probe_of(const FrzPatternDev& p, int i) { return Probe{splat4(p.om[i]), splat4(p.tg[i])}; }

// ---- Prefilter::match_haystack (0 typos): closed form of src/prefilter/algo/ascii.rs:6-54 ----
// start = first occurrence of needle[0]; greedy in-order scan; end = 1 + last occurrence of needle[n-1]
template <class A>
__device__ bool window_k0(const A& a, const FrzPatternDev& p, int len, int* ostart, int* oend) {
    if (len == 0) return false;
    int pos = 0, start = 0, q = 0;
    for (int i = 0; i < p.n; i++) {
        Probe pr = probe_of(p, i);
        q = find_first(a, pr.om, pr.tg, pos, len);
        if (q < 0) return false;
        if (i == 0) start = q;
        pos = q + 1;
    }
    Probe last = probe_of(p, p.n - 1);
    *ostart = start;
    *oend = 1 + find_last2(a, last.om, last.tg, last.om, last.tg, q, len);
    return true;
}

// find_end_pos_with_typos (src/prefilter/algo/ascii_typos.rs:375-397): 1 + last occurrence of any of
// the last (k+1) needle bytes, else len.  Chunk-independent.
template <class A>
__device__ int end_pos_with_typos(const A& a, const FrzPatternDev& p, int len, int k) {
    int best = -1;
    int first = p.n - 1 - k;
    for (int i = first; i < p.n; i += 2) {
        Probe p1 = probe_of(p, i);
        Probe p2 = probe_of(p, i + 1 < p.n ? i + 1 : i);
        int q = find_last2(a, p1.om, p1.tg, p2.om, p2.tg, best < 0 ? 0 : best, len);
        if (q > best) best = q;
    }
    return best < 0 ? len : best + 1;
}

// ---- match_haystack_1_typo (src/prefilter/algo/ascii_typos.rs:15-110), chunk-emulating ----
// Both paths' chunk masks are always suffixes [pos, chunk_end) of the chunk, so a path is the pair
// (needle index, position) and `first_path_chunk_mask > second_path_chunk_mask` ⇔ pf < ps.
template <class A>
__device__ bool window_k1(const A& a, const FrzPatternDev& p, int len, int* ostart, int* oend) {
    const int n = p.n;
    if (n <= 1) { *ostart = 0; *oend = len; return true; }
    if (len == 0) return false;
    int f = 0, s = 1;
    int ms = 0x7fffffff;
    const int L = p.pf_lanes;
    for (int cs = 0; cs < len; cs += L) {
        const int ce = min(cs + L, len);
        int pf = cs, ps = cs;
        bool f_dead = false, s_dead = false;  // path already failed to find its byte in [pos, ce)
        for (;;) {
            bool adv = false;
            int cand = f + 1;
            if (cand > s) {
                if (cand == n) goto found;
                s = cand; ps = pf; s_dead = false;
            } else if (cand == s && pf < ps) {
                ps = pf; s_dead = false;
            }
            if (!f_dead) {
                Probe pr = probe_of(p, f);
                int q = find_first(a, pr.om, pr.tg, pf, ce);
                if (q >= 0) { ms = min(ms, q); f++; pf = q + 1; adv = true; }
                else f_dead = true;
            }
            if (!s_dead) {
                Probe pr = probe_of(p, s);
                int q = find_first(a, pr.om, pr.tg, ps, ce);
                if (q >= 0) {
                    ms = min(ms, q); s++;
                    if (s >= n) goto found;
                    ps = q + 1; adv = true;
                } else s_dead = true;
            }
            if (!adv) break;
        }
    }
    return false;
found:
    *ostart = ms;
    *oend = end_pos_with_typos(a, p, len, 1);
    return true;
}

// ---- match_haystack_many_typos_impl (ascii_typos.rs:254-360); also used for k == 2 ----
// NOTE the 2-typo specialisation (ascii_typos.rs:113-251) advances each path on its OWN first hit,
// the N-typo version advances all paths on the single lowest hit; they are distinct algorithms.
template <class A>
__device__ bool window_k2(const A& a, const FrzPatternDev& p, int len, int* ostart, int* oend) {
    const int n = p.n;
    if (n <= 2) { *ostart = 0; *oend = len; return true; }
    if (len == 0) return false;
    int idx[3] = {0, 1, 2};
    int ms = 0x7fffffff;
    const int L = p.pf_lanes;
    for (int cs = 0; cs < len; cs += L) {
        const int ce = min(cs + L, len);
        int pos[3] = {cs, cs, cs};
        for (;;) {
            bool adv = false;
#pragma unroll
            for (int k = 1; k < 3; k++) {
                int cand = idx[k - 1] + 1;
                if (cand > idx[k]) {
                    if (cand == n) goto found;
                    idx[k] = cand; pos[k] = pos[k - 1];
                } else if (cand == idx[k] && pos[k - 1] < pos[k]) {
                    pos[k] = pos[k - 1];
                }
            }
#pragma unroll
            for (int k = 0; k < 3; k++) {
                Probe pr = probe_of(p, idx[k]);
                int q = find_first(a, pr.om, pr.tg, pos[k], ce);
                if (q >= 0) {
                    ms = min(ms, q); idx[k]++;
                    if (k > 0 && idx[k] >= n) goto found;
                    pos[k] = q + 1; adv = true;
                }
            }
            if (!adv) break;
        }
    }
    return false;
found:
    *ostart = ms;
    *oend = end_pos_with_typos(a, p, len, 2);
    return true;
}

constexpr int kMaxPaths = 16;  // FRZ_T_MANY supports max_typos <= 15 on the GPU path

template <class A>
__device__ bool window_many(const A& a, const FrzPatternDev& p, int len, int* ostart, int* oend) {
    const int n = p.n, k = p.max_typos;
    if (n <= k) { *ostart = 0; *oend = len; return true; }
    if (len == 0) return false;
    const int paths = k + 1;
    int idx[kMaxPaths];
    for (int i = 0; i < paths; i++) idx[i] = 0;
    int ms = 0x7fffffff;
    const int L = p.pf_lanes;
    for (int cs = 0; cs < len; cs += L) {
        const int ce = min(cs + L, len);
        int pos = cs;  // one shared chunk mask (ascii_typos.rs:286,350)
        for (;;) {
            for (int j = 1; j < paths; j++) {
                int cand = idx[j - 1] + 1;
                if (cand > idx[j]) {
                    if (cand == n) goto found;
                    idx[j] = cand;
                }
            }
            // lowest hit over all paths
            int hit = 0x7fffffff;
            for (int j = 0; j < paths; j++) {
                Probe pr = probe_of(p, idx[j]);
                int q = find_first(a, pr.om, pr.tg, pos, min(ce, hit == 0x7fffffff ? ce : hit + 1));
                if (q >= 0 && q < hit) hit = q;
            }
            if (hit == 0x7fffffff) break;
            ms = min(ms, hit);
            uint32_t hb = a.word(hit >> 2) >> ((hit & 3) * 8) & 0xff;
            for (int j = 0; j < paths; j++) {
                int i = idx[j];
                if (((hb | p.om[i]) & 0xff) != p.tg[i]) continue;
                idx[j] = i + 1;
                if (idx[j] == n) goto found;
            }
            pos = hit + 1;
        }
    }
    return false;
found:
    *ostart = ms;
    *oend = end_pos_with_typos(a, p, len, k);
    return true;
}

// ---- literal matcher, ASCII path (src/literal/algo.rs:159-255) ----
__device__ __forceinline__ bool lit_is_delim(uint32_t b) {
    bool alnum = (b - '0' <= 9u) || (b - 'a' <= 25u) || (b - 'A' <= 25u);
    return b <= 127 && !alnum;
}
template <class A>
__device__ __forceinline__ uint32_t byte_at(const A& a, int i) { return (a.word(i >> 2) >> ((i & 3) * 8)) & 0xff; }

template <class A>
__device__ bool lit_matches_at(const A& a, const FrzPatternDev& p, int pos) {
    for (int k = 0; k < p.n; k++) {
        uint32_t b = byte_at(a, pos + k);
        if (b != p.c[k] && b != p.flip[k]) return false;
    }
    return true;
}
template <class A>
__device__ uint32_t lit_score_at(const A& a, const FrzPatternDev& p, int len, int pos) {
    uint32_t score = 0;
    uint32_t prev = pos > 0 ? byte_at(a, pos - 1) : 0;
    for (int k = 0; k < p.n; k++) {
        int st = pos + k;
        uint32_t b = byte_at(a, st);
        uint32_t sc = p.raw_match;
        if (b == p.c[k]) sc += p.raw_case;
        if (st == 0) sc += p.raw_prefix;
        else {
            if (b - 'A' <= 25u && prev - 'a' <= 25u) sc += p.raw_cap;
            if (lit_is_delim(prev) && !lit_is_delim(b)) sc += p.raw_delim;
        }
        score += sc;
        prev = b;
    }
    if (pos == 0 && p.n == len) score += p.exact_bonus;
    return score & 0xffff;
}
// returns true on match; *opos, *oscore
template <class A>
__device__ bool lit_find(const A& a, const FrzPatternDev& p, int len, int* opos, uint32_t* oscore) {
    const int n = p.n;
    if (len < n) return false;
    switch (p.matching) {
        case FRZ_MATCHING_EXACT:
            if (len != n || !lit_matches_at(a, p, 0)) return false;
            *opos = 0; *oscore = lit_score_at(a, p, len, 0); return true;
        case FRZ_MATCHING_PREFIX:
            if (!lit_matches_at(a, p, 0)) return false;
            *opos = 0; *oscore = lit_score_at(a, p, len, 0); return true;
        case FRZ_MATCHING_SUFFIX:
            if (!lit_matches_at(a, p, len - n)) return false;
            *opos = len - n; *oscore = lit_score_at(a, p, len, len - n); return true;
        default: {  // SUBSTRING: best score, earliest on ties (find_substring :262-313)
            bool have = false;
            Probe p0 = probe_of(p, 0);
            int from = 0;
            const int last_start = len - n + 1;
            for (;;) {
                int q = find_first(a, p0.om, p0.tg, from, last_start);
                if (q < 0) break;
                if (lit_matches_at(a, p, q)) {
                    uint32_t sc = lit_score_at(a, p, len, q);
                    if (!have || sc > *oscore) { have = true; *opos = q; *oscore = sc; }
                }
                from = q + 1;
            }
            return have;
        }
    }
}


struct OccTable {
    uint2 occ[kMaxDistinct][32];             // per-lane occurrence masks of the distinct needle byte classes
};

__device__ __forceinline__ int sw_class_of(int window, const FrzPatternDev& pat) {
    if (window > 128) return FRZ_C_GENERIC;
    if (window > 64) return FRZ_C_COLS128;
    if (!pat.col_classes) return FRZ_C_COLS64;
    // columns whose cells can reach the score: the window, needle_len diagonal steps past its end, and never
    // more than the chunks the reference evaluates
    const int chunk_cols = (window + pat.sw_lanes - 1) / pat.sw_lanes * pat.sw_lanes;
    const int need = min(window + pat.n, chunk_cols);
    // four classes: two (48 / 64) were measured 3% SLOWER on B200 (the extra columns cost more than the smaller kernel saves)
    return need <= 40 ? FRZ_C_CC40 : need <= 48 ? FRZ_C_CC48 : need <= 56 ? FRZ_C_CC56 : FRZ_C_COLS64;
}

// Exact window of one queued candidate (phase B) + survivor emission.  All 32 lanes of the warp call
// this together (`active` lanes have an entry); emission uses warp-aggregated atomics.
// One candidate as phase B sees it.  `units` is where the mask builders read the haystack's 16-byte units from (unit k at
// units + k): the packed corpus itself, or this lane's row of a shared-memory stage filled by cp.async.
struct Cand {
    uint32_t tile, slot, li;   // li = index of the haystack inside its tile
    int len;
    const uint4* base;         // unit 0 of the slot in the packed corpus
    const uint4* units;
};
// resolves (tile, slot) through the group descriptor and the slot metadata (candidate lists of the multi-pattern path)
__device__ __forceinline__ Cand resolve_cand(const FrzCorpusView& cv, uint32_t tile, uint32_t slot, int len) {
    Cand c;
    c.tile = tile; c.slot = slot; c.len = len;
    const FrzGroupDesc gd = cv.groups[tile * FRZ_GROUPS_PER_TILE + (slot >> 5)];
    c.base = cv.data + frz_slot_unit0(gd, slot & 31);
    c.units = c.base;
    c.li = cv.slot_meta[(uint64_t)tile * FRZ_TILE + slot] & (FRZ_TILE - 1);
    return c;
}

// what process_candidate found for one lane's candidate, on its way to the per-class survivor lists
struct Emit {
    FrzSurvivor rec;
    unsigned long long base_raw;   // leader lanes: the reserved list position (result of the atomic, may still be in flight)
    uint32_t peers;                // lanes of the warp with the same SW class
    int cls;
    bool ok;
};

template <int MODE>
__device__ __forceinline__ void process_candidate(const FrzCorpusView& cv, const FrzPatternDev& pat, const uint8_t* __restrict__ cid_s,
                                                  uint2 (*occ)[32], const Cand& cd, bool active,
                                                  uint32_t* __restrict__ surv_bitmap, Emit* out, bool single_chunk = false) {
    bool ok = false;
    int cls = 0;
    FrzSurvivor rec;
    rec.tile = 0; rec.slot_rank = 0; rec.start = 0; rec.end = 0;
    const uint32_t tile = cd.tile, slot = cd.slot;
    const int len = active ? cd.len : 0;
    GlobalAcc ga{active ? cd.base : nullptr};
    const uint4* units = active ? cd.units : nullptr;
    // warp-wide occurrence-mask windows (uniform code) for the 0- and 1-typo modes
    bool flat_done = false, flat_ok = false;
    int flat_start = 0, flat_end = 0;
    if ((MODE == FRZ_T_0 || MODE == FRZ_T_1) && pat.n_distinct > 0) {
        if (single_chunk) {   // warp-uniform: corpus of <= 64-byte haystacks at the 64-lane width (prefilter_masks.cuh)
            if (MODE == FRZ_T_0) flat_ok = masks_k0_single(units, pat, occ, len, active, &flat_start, &flat_end);
            else flat_ok = masks_k1_single(units, pat, occ, len, active, &flat_start, &flat_end);
        } else {
            if (MODE == FRZ_T_0) flat_ok = masks_k0(units, pat, cid_s, occ, len, active, &flat_start, &flat_end);
            else flat_ok = masks_k1(units, pat, cid_s, occ, len, active, &flat_start, &flat_end);
        }
        flat_done = true;
    }
    // 2-typo / N-typo trackers on the same occurrence masks (prefilter_masks.cuh: masks_paths<3>, masks_many).  Measured on
    // B200 against the scanning forms window_k2 / window_many (profiles/r02b_sw_variants.txt, 10 M haystacks): k = 2
    // 2.79 -> 0.21 ms, k = 3 2.25 -> 0.42 ms.  The scanning forms remain for needles with > 16 distinct byte classes.
    if ((MODE == FRZ_T_2 || MODE == FRZ_T_MANY) && pat.n_distinct > 0) {
        if (MODE == FRZ_T_2) flat_ok = masks_paths<3>(units, pat, cid_s, occ, len, active, &flat_start, &flat_end);
        else flat_ok = masks_many(units, pat, cid_s, occ, len, active, &flat_start, &flat_end);
        flat_done = true;
    }
    if (active) {
        const uint32_t li = cd.li;
        int start = 0, end = len;
        uint32_t lit_score = 0;
        if (flat_done) { ok = flat_ok; start = flat_start; end = flat_end; }
        else if (MODE == FRZ_T_0) ok = window_k0(ga, pat, len, &start, &end);
        else if (MODE == FRZ_T_1) ok = window_k1(ga, pat, len, &start, &end);
        else if (MODE == FRZ_T_2) ok = window_k2(ga, pat, len, &start, &end);
        else if (MODE == FRZ_T_MANY) ok = window_many(ga, pat, len, &start, &end);
        else if (MODE == FRZ_T_LITERAL) {
            int pos = 0;
            ok = lit_find(ga, pat, len, &pos, &lit_score);
            start = pos; end = pos + pat.n;
        } else ok = true;  // FRZ_T_NONE: NO_PREFILTER (src/matcher/algo.rs:178)
        if (ok) {
            rec.tile = tile;
            rec.slot_rank = slot | (li << 10);
            if (MODE == FRZ_T_LITERAL) {
                // literal matches are final: carry (score, exact) through start/end
                cls = FRZ_C_COLS64;
                rec.start = lit_score;
                rec.end = (start == 0 && pat.n == len) ? 1u : 0u;
            } else {
                start = start > 0 ? start - 1 : 0;  // trim_haystack (src/matcher/algo.rs:331-338)
                cls = sw_class_of(end - start, pat);
                if (cls < FRZ_C_GENERIC) {
                    // window record (frz_device.cuh): everything the SW kernel needs, including the address of the
                    // window's first 16-byte unit, so that it never touches the group descriptors
                    const uint64_t addr = (uint64_t)(ga.base - cv.data) + (uint64_t)(start >> 4);
                    rec.slot_rank |= (uint32_t)(end - start) << 20 | (uint32_t)(end == len) << 28 | (uint32_t)(start == 0) << 29;
                    rec.start = (uint32_t)addr;
                    rec.end = (uint32_t)(addr >> 32) | ((uint32_t)start & 15u) << 8;
                } else {
                    rec.start = (uint32_t)start;
                    rec.end = (uint32_t)end | ((uint32_t)(end == len) << 31);
                }
            }
            atomicOr(&surv_bitmap[(uint64_t)tile * 32 + (li >> 5)], 1u << (li & 31));
        }
    }
    out->rec = rec;
    out->ok = ok;
    out->cls = cls;
}

// Survivor emission, split in two so that the round trip of the list-space atomic overlaps the NEXT item's work:
//   emit_request  the lowest lane of every SW class present reserves list slots for its peers (one atomic per class);
//                 the result stays in flight
//   emit_commit   (one item later) broadcast of the reserved base, then the 16-byte record stores
__device__ __forceinline__ void emit_request(Emit& e, FrzCounters* __restrict__ ctr) {
    const uint32_t lane = frz_lane();
    e.peers = __match_any_sync(0xffffffffu, e.ok ? e.cls : -1);
    e.base_raw = 0;
    if (e.ok && (int)lane == __ffs(e.peers) - 1)
        e.base_raw = atomicAdd(&ctr->class_count[e.cls], (unsigned long long)__popc(e.peers));
}
__device__ __forceinline__ void emit_commit(const Emit& e, const FrzSurvLists& lists, unsigned long long surv_cap,
                                            FrzCounters* __restrict__ ctr) {
    if (!__any_sync(0xffffffffu, e.ok)) return;
    const uint32_t lane = frz_lane();
    const unsigned long long base = __shfl_sync(0xffffffffu, e.base_raw, __ffs(e.peers) - 1);
    if (e.ok) {
        const unsigned long long pos = base + __popc(e.peers & ((1u << lane) - 1));
        if (pos < surv_cap) lists.p[e.cls][pos] = e.rec;
        else atomicOr(&ctr->error, FRZ_DEVERR_SURVIVOR_OVERFLOW);
    }
}

// ================================================================================================================
// Stage 1a  k_sig_scan — the streaming half.  Lane per FOUR consecutive haystacks: one 16-byte load of their lengths and
// two 16-byte loads of their byte-class signatures (written at pack time, pack.cu: k_pack_sig) decide "can this
// haystack hold the needle up to the typo budget?" (two POPCs each).  The haystack bytes themselves are never touched
// here: a rejected haystack costs 12 bytes of HBM traffic instead of len + 8.  Survivors of the test become 16-byte
// candidate records {tile << 10 | slot, len << 10 | index-in-tile, address of unit 0}: the group descriptor is resolved
// here (four contiguous 16-byte descriptors per trip, L2-resident), so stage 1b starts its unit loads straight from the
// record.  Warp-autonomous: a per-warp ring in shared memory collects candidates, every 32 are flushed with ONE atomic
// and one coalesced 512-byte store.  Small (about 40 registers): 12 blocks per SM keep enough bytes in flight to stream
// at HBM speed — in the fused kernel the same loop sat at 47% of the stall samples waiting on its own loads behind
// the 76-register window code (profiles/r02b_*).
constexpr int kScanThreads = 128;
constexpr int kScanWarps = kScanThreads / 32;
constexpr int kScanRing = 256;   // entries per warp: up to 31 left over + up to 128 new per trip

struct __align__(16) CandRec {
    uint32_t tile_slot;   // tile << 10 | slot
    uint32_t meta;        // len << 10 | index inside the tile
    uint64_t unit0;       // unit index (16-byte units from the start of the packed data) of the slot's unit 0
};

// ---- TMA staging (cp.async.bulk, 1-D) of the phase-A arrays ---------------------------------------------------------
// The metadata, signature and group-descriptor arrays are contiguous, so a warp's next 128-slot chunk is three bulk
// copies (512 + 1024 + 64 bytes) that complete on the warp's OWN mbarrier: warp-autonomous, no block barrier, and the
// bytes in flight hold no registers (a register-prefetch form pays 14 registers per chunk in flight and ptxas sinks such
// loads towards their use: it measured 0.1596 against 0.1568 ms for the stage, profiles/r02_experiments.md).  Three stages
// per warp.
constexpr int kScanStages = 3;
struct __align__(16) ScanStage {
    uint32_t meta[128];
    uint2 sig[128];
    FrzGroupDesc desc[4];
};
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src),
                 "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

__global__ void __launch_bounds__(kScanThreads, 6) k_sig_scan(const FrzCorpusView cv, int use_sig, uint32_t need1, uint32_t need2,
                                                               int sig_k, int min_len, CandRec* __restrict__ cand,
                                                               unsigned long long cand_cap, FrzCounters* __restrict__ ctr) {
    extern __shared__ __align__(16) unsigned char scan_smem[];
    const uint32_t lane = frz_lane(), warp = threadIdx.x >> 5;
    CandRec* ring = reinterpret_cast<CandRec*>(scan_smem) + (size_t)warp * kScanRing;
    const uint32_t n_warps = gridDim.x * kScanWarps;
    const uint32_t total_chunks = cv.n_tiles * (FRZ_TILE / 128);   // 128 slots (4 groups) per chunk
    uint32_t head = 0, count = 0;
    // ---- candidate ring → global list, in two steps so that the atomic's round trip overlaps the next chunk:
    //      flush_request reserves list space for the 32 oldest entries (they stay in the ring), flush_commit stores them
    unsigned long long pend_base = 0;
    uint32_t pend_head = 0, pend_n = 0;
    auto flush_commit = [&]() {
        if (pend_n == 0) return;
        const unsigned long long base = __shfl_sync(0xffffffffu, pend_base, 0);
        if (lane < pend_n) {
            const unsigned long long pos = base + lane;
            if (pos < cand_cap) reinterpret_cast<uint4*>(cand)[pos] = reinterpret_cast<const uint4*>(ring)[(pend_head + lane) & (kScanRing - 1)];
            else atomicOr(&ctr->error, FRZ_DEVERR_SURVIVOR_OVERFLOW);
        }
        pend_n = 0;
    };
    auto flush_request = [&](uint32_t n_out) {
        flush_commit();   // at most one reservation in flight
        if (lane == 0) pend_base = atomicAdd(&ctr->cand_count, (unsigned long long)n_out);
        pend_head = head;
        pend_n = n_out;
        head = (head + n_out) & (kScanRing - 1);
        count -= n_out;
    };
    // length gate + signature test of one slot; passing lanes append their record to the ring
    auto test_slot = [&](uint32_t m, uint32_t p1, uint32_t p2, uint32_t slot_global, unsigned long long unit0) {
        bool pass = m != FRZ_INVALID_SLOT && (int)(m >> FRZ_TILE_SHIFT) >= min_len;
        if (use_sig) pass = pass && frz_sig_pass(need1, need2, sig_k, p1, p2);
        const uint32_t ballot = __ballot_sync(0xffffffffu, pass);
        if (pass)   // one 16-byte shared-memory store (a CandRec, field by field)
            reinterpret_cast<uint4*>(ring)[(head + count + __popc(ballot & ((1u << lane) - 1))) & (kScanRing - 1)] =
                make_uint4(slot_global, m, (uint32_t)unit0, (uint32_t)(unit0 >> 32));
        count += __popc(ballot);
    };
    // one chunk = 128 consecutive slots (4 groups): lane L owns slots 4L .. 4L+3, all in group L / 8 of the chunk
    auto process = [&](uint32_t idx, const uint4& meta, const uint4& sig0, const uint4& sig1, unsigned long long grp_off, uint32_t gunits) {
        const uint32_t slot_g = idx * 128 + lane * 4;                   // == tile << 10 | slot of this lane's first slot
        const unsigned long long unit0 = grp_off + (unsigned long long)((lane * 4) & 31) * gunits;   // unit 0 of that slot (slot-major group)
        test_slot(meta.x, sig0.x, sig0.y, slot_g, unit0);
        test_slot(meta.y, sig0.z, sig0.w, slot_g + 1, unit0 + gunits);
        test_slot(meta.z, sig1.x, sig1.y, slot_g + 2, unit0 + 2 * gunits);
        test_slot(meta.w, sig1.z, sig1.w, slot_g + 3, unit0 + 3 * gunits);
        __syncwarp();
        flush_commit();                       // the reservation made one chunk ago has arrived
        while (count >= 32) flush_request(32);
        __syncwarp();
    };
    {   // the chunk pipeline: three TMA stages per warp, each completing on its own mbarrier
        ScanStage* stages = reinterpret_cast<ScanStage*>(scan_smem + sizeof(CandRec) * kScanRing * kScanWarps) + warp * kScanStages;
        uint64_t* bars = reinterpret_cast<uint64_t*>(scan_smem + (sizeof(CandRec) * kScanRing + sizeof(ScanStage) * kScanStages) * kScanWarps) +
                         warp * kScanStages;
        if (lane == 0)
            for (int i = 0; i < kScanStages; i++) mbar_init(&bars[i], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        __syncwarp();
        const uint32_t tx_bytes = (uint32_t)(sizeof(uint32_t) * 128 + sizeof(FrzGroupDesc) * 4) + (use_sig ? (uint32_t)sizeof(uint2) * 128 : 0u);
        uint32_t req = blockIdx.x * kScanWarps + warp;   // next chunk to REQUEST
        auto issue = [&](int st) {
            if (req < total_chunks && lane == 0) {
                const uint64_t slot0 = (uint64_t)req * 128;
                mbar_expect_tx(&bars[st], tx_bytes);
                bulk_g2s(stages[st].meta, cv.slot_meta + slot0, (uint32_t)sizeof(uint32_t) * 128, &bars[st]);
                if (use_sig) bulk_g2s(stages[st].sig, cv.slot_sig + slot0, (uint32_t)sizeof(uint2) * 128, &bars[st]);
                bulk_g2s(stages[st].desc, cv.groups + (size_t)req * 4, (uint32_t)sizeof(FrzGroupDesc) * 4, &bars[st]);
            }
            req += n_warps;
        };
        uint32_t cur = req;
#pragma unroll
        for (int i = 0; i < kScanStages; i++) issue(i);
        int st = 0;
        uint32_t parity = 0;
        while (cur < total_chunks) {
            mbar_wait(&bars[st], parity);
            const uint4 meta = reinterpret_cast<const uint4*>(stages[st].meta)[lane];
            uint4 sig0 = make_uint4(0u, 0u, 0u, 0u), sig1 = sig0;
            if (use_sig) {
                sig0 = reinterpret_cast<const uint4*>(stages[st].sig)[2 * lane];
                sig1 = reinterpret_cast<const uint4*>(stages[st].sig)[2 * lane + 1];
            }
            const unsigned long long grp_off = stages[st].desc[lane >> 3].abs_off;
            const uint32_t grp_units = stages[st].desc[lane >> 3].gunits;
            __syncwarp();
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic reads of the stage before its async refill
            issue(st);
            process(cur, meta, sig0, sig1, grp_off, grp_units);
            cur += n_warps;
            if (++st == kScanStages) { st = 0; parity ^= 1; }
        }
    }
    flush_commit();
    if (count) { flush_request(count); flush_commit(); }
}

// ================================================================================================================
// Stage 1b  k_window — the exact reference window (process_candidate) on the candidates, lane per candidate.
// Work items are 32 consecutive candidate records, claimed from a device counter.  The loop is software-pipelined two
// items deep: while item i is in the mask builders / state machine, item i+1's haystack units travel global → shared
// with cp.async (the record carries the unit address: no dependent descriptor load) and item i+2's records are in
// flight — the scattered unit loads are what phase B of the fused kernel stalled on.
constexpr int kWinThreads = 128;
constexpr int kWinWarps = kWinThreads / 32;
struct WinStage {
    uint4 units[32][5];   // [lane][unit]: the lane's four units contiguous like in the packed corpus; the fifth pads the row
                          // to 80 bytes, which makes the warp's 16-byte accesses bank-conflict-free (rows of 64 would be 4-way)
};
struct WinSmem {
    uint2 occ[kMaxDistinct][32];
    WinStage stage[2];
    uint4 rec[3][32];     // candidate records of items k, k+1, k+2 (ring), also filled by cp.async
};

template <int MODE>
__global__ void __launch_bounds__(kWinThreads, 4) k_window(const FrzCorpusView cv, const __grid_constant__ FrzPatternDev pat,
                                                           const CandRec* __restrict__ cand, unsigned long long cand_cap,
                                                           const FrzSurvLists lists, unsigned long long surv_cap,
                                                           uint32_t* __restrict__ surv_bitmap, FrzCounters* __restrict__ ctr) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const uint32_t lane = frz_lane(), warp = threadIdx.x >> 5;
    WinSmem& sm = reinterpret_cast<WinSmem*>(smem_raw)[warp];
    __shared__ uint8_t cid_s[FRZ_MAX_NEEDLE];
    if (threadIdx.x < FRZ_MAX_NEEDLE) cid_s[threadIdx.x] = pat.cid[threadIdx.x];
    __syncthreads();
    const unsigned long long n_cand = min(ctr->cand_count, cand_cap);
    const uint32_t n_items = (uint32_t)((n_cand + 31) >> 5);
    const bool staged = cv.max_gunits <= 4;   // every haystack fits the four staged units
    const bool single = (MODE == FRZ_T_0 || MODE == FRZ_T_1) && single_chunk_ok(pat, cv.max_gunits);

    // Work items are strided statically over the warps of the grid (their cost is uniform), so the item sequence of a warp
    // is known ahead: item k's units AND item k+1's records were requested with cp.async one iteration earlier (records
    // fetched into registers were sunk by ptxas to their first use: 27% of the stall samples, profiles/r02e).
    //   group G_k (committed in iteration k) = { units of item k+1 , records of item k+2 }
    const uint32_t n_warps = gridDim.x * kWinWarps;
    const uint32_t item0 = blockIdx.x * kWinWarps + warp;
    auto fetch_rec = [&](uint32_t k) {   // records of this warp's k-th item → ring slot k % 3
        const uint32_t item = item0 + k * n_warps;
        const unsigned long long j = (unsigned long long)item * 32 + lane;
        uint4* dst = &sm.rec[k % 3][lane];
        if (item < n_items && j < n_cand) __pipeline_memcpy_async(dst, reinterpret_cast<const uint4*>(cand) + j, 16);
        else *dst = make_uint4(0xFFFFFFFFu, 0u, 0u, 0u);
    };
    auto unit0_of = [](const uint4& r) { return ((unsigned long long)r.w << 32) | r.z; };
    auto fetch_units = [&](const uint4& r, int st) {
        if (staged && r.x != 0xFFFFFFFFu) {
            const int units = ((int)(r.y >> FRZ_TILE_SHIFT) + 15) >> 4;
            const uint4* base = cv.data + unit0_of(r);
#pragma unroll
            for (int k = 0; k < 4; k++)
                if (k < units) __pipeline_memcpy_async(&sm.stage[st].units[lane][k], base + k, 16);
        }
    };
    fetch_rec(0);
    fetch_rec(1);
    __pipeline_commit();
    __pipeline_wait_prior(0);
    __syncwarp();
    fetch_units(sm.rec[0][lane], 0);
    __pipeline_commit();
    Emit pending;
    pending.ok = false; pending.cls = 0; pending.peers = 0; pending.base_raw = 0;
    pending.rec.tile = 0; pending.rec.slot_rank = 0; pending.rec.start = 0; pending.rec.end = 0;
    for (uint32_t k = 0; item0 + k * n_warps < n_items; k++) {
        __pipeline_wait_prior(0);                        // G_{k-1}: this item's units and the next item's records
        __syncwarp();
        const uint4 rec0 = sm.rec[k % 3][lane];
        fetch_units(sm.rec[(k + 1) % 3][lane], (k + 1) & 1);
        fetch_rec(k + 2);
        __pipeline_commit();                             // G_k flies while item k is processed
        const int st = k & 1;
        const bool active = rec0.x != 0xFFFFFFFFu;
        Cand cd;
        cd.tile = rec0.x >> FRZ_TILE_SHIFT;
        cd.slot = rec0.x & (FRZ_TILE - 1);
        cd.li = rec0.y & (FRZ_TILE - 1);
        cd.len = (int)(rec0.y >> FRZ_TILE_SHIFT);
        cd.base = cv.data + unit0_of(rec0);
        cd.units = staged ? &sm.stage[st].units[lane][0] : cd.base;
        Emit cur;
        process_candidate<MODE>(cv, pat, cid_s, sm.occ, cd, active, surv_bitmap, &cur, single);
        emit_commit(pending, lists, surv_cap, ctr);      // the previous item's list space has arrived by now
        emit_request(cur, ctr);
        pending = cur;
        __syncwarp();
    }
    emit_commit(pending, lists, surv_cap, ctr);
    __pipeline_wait_prior(0);
}

// Candidate-list mode (multi-pattern, src/matcher/multi.rs:108-120): the extra patterns are evaluated only
// on the haystacks that survived the previous patterns.  The list is already compact, so each warp takes 32
// candidates at a time straight to phase B.
template <int MODE>
__global__ void __launch_bounds__(kThreads) k_prefilter_list(const FrzCorpusView cv, const __grid_constant__ FrzPatternDev pat,
                                                             const FrzMatchDev* __restrict__ cand, unsigned long long n_cand,
                                                             uint32_t index_offset,
                                                             const FrzSurvLists lists, unsigned long long surv_cap,
                                                             uint32_t* __restrict__ surv_bitmap, FrzCounters* __restrict__ ctr) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const uint32_t lane = frz_lane(), warp = threadIdx.x >> 5;
    uint2 (*occ)[32] = reinterpret_cast<OccTable*>(smem_raw)[warp].occ;
    __shared__ uint8_t cid_s[FRZ_MAX_NEEDLE];
    if (threadIdx.x < FRZ_MAX_NEEDLE) cid_s[threadIdx.x] = pat.cid[threadIdx.x];
    __syncthreads();
    const unsigned long long n_warps = (unsigned long long)gridDim.x * kWarps;
    for (unsigned long long base = ((unsigned long long)blockIdx.x * kWarps + warp) * 32; base < n_cand; base += n_warps * 32) {
        const unsigned long long i = base + lane;
        bool active = i < n_cand;
        Cand cd;
        cd.tile = 0; cd.slot = 0; cd.li = 0; cd.len = 0; cd.base = nullptr; cd.units = nullptr;
        if (active) {
            const uint32_t idx = cand[i].index - index_offset;
            const uint32_t tile = idx >> FRZ_TILE_SHIFT, li = idx & (FRZ_TILE - 1);
            const uint32_t slot = cv.slot_of[(uint64_t)tile * FRZ_TILE + li];
            const uint32_t len = cv.slot_meta[(uint64_t)tile * FRZ_TILE + slot] >> FRZ_TILE_SHIFT;
            active = (int)len >= pat.min_hay_len;   // length gate (src/matcher/algo.rs:88)
            cd = resolve_cand(cv, tile, slot, (int)len);
        }
        __syncwarp();
        Emit e;
        process_candidate<MODE>(cv, pat, cid_s, occ, cd, active, surv_bitmap, &e);
        emit_request(e, ctr);
        emit_commit(e, lists, surv_cap, ctr);
        __syncwarp();
    }
}

// Per tile: exclusive prefix popcount of the 32 survivor-bitmap words (→ rank of a survivor among
// its tile's survivors in index order) and the tile's survivor count.  One warp per tile.
__global__ void __launch_bounds__(256) k_tile_rank(const uint32_t* __restrict__ surv_bitmap, uint16_t* __restrict__ word_prefix,
                                                   uint32_t* __restrict__ tile_count, uint32_t n_tiles) {
    const uint32_t tile = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = frz_lane();
    if (tile >= n_tiles) return;
    const uint32_t c = __popc(surv_bitmap[(uint64_t)tile * 32 + lane]);
    uint32_t x = c;
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t y = __shfl_up_sync(0xffffffffu, x, d);
        if (lane >= (uint32_t)d) x += y;
    }
    word_prefix[(uint64_t)tile * 32 + lane] = (uint16_t)(x - c);
    if (lane == 31) tile_count[tile] = x;
}

// exclusive scan of tile_count → tile_out_base; total → counters.total.  One block; every thread owns a CONTIGUOUS run
// of ceil(n / 1024) tiles, so the block makes one pass (two for > 1 M tiles) instead of n / 1024 barrier rounds
// (12 us → 3 us at 9766 tiles, profiles/r02b_launches.csv vs r02d).
// `carry` (optional): the scan starts at *carry and leaves the new total there too — streamed calls (host.cu:
// frz_match_shard_streamed) run the pipeline over consecutive tile ranges and append each range's matches to the same list.
__global__ void __launch_bounds__(1024) k_tile_scan(const uint32_t* __restrict__ tile_count, uint64_t* __restrict__ out,
                                                    uint32_t n, FrzCounters* __restrict__ ctr, unsigned long long* carry) {
    __shared__ uint64_t warp_sum[32];
    const uint32_t per = (n + blockDim.x - 1) / blockDim.x;
    const uint32_t lo = min(threadIdx.x * per, n), hi = min(lo + per, n);
    uint64_t sum = 0;
    for (uint32_t i = lo; i < hi; i++) sum += tile_count[i];
    uint64_t x = sum;
    for (int d = 1; d < 32; d <<= 1) {
        uint64_t y = __shfl_up_sync(0xffffffffu, x, d);
        if (frz_lane() >= (uint32_t)d) x += y;
    }
    if (frz_lane() == 31) warp_sum[threadIdx.x >> 5] = x;
    __syncthreads();
    if (threadIdx.x < 32) {
        uint64_t w = warp_sum[threadIdx.x], xs = w;
        for (int d = 1; d < 32; d <<= 1) {
            uint64_t y = __shfl_up_sync(0xffffffffu, xs, d);
            if (frz_lane() >= (uint32_t)d) xs += y;
        }
        warp_sum[threadIdx.x] = xs - w;
    }
    __syncthreads();
    const uint64_t start = carry ? *carry : 0ull;
    __syncthreads();                                        // everybody has read the carry before the last thread replaces it
    uint64_t run = start + warp_sum[threadIdx.x >> 5] + x - sum;   // exclusive prefix of this thread's run
    for (uint32_t i = lo; i < hi; i++) {
        out[i] = run;
        run += tile_count[i];
    }
    if (threadIdx.x == blockDim.x - 1) {   // the last thread's run ends at n (empty runs carry the total)
        ctr->total = run;
        if (carry) *carry = run;
    }
}

// Matcher::match_list_indices for chosen haystacks (src/matcher/mod.rs:234-262 → match_one_indices_impl,
// src/matcher/algo.rs:138-169, src/literal/algo.rs:134-155).  One thread per requested haystack; the scoring with
// full matrices and the traceback are in indices_path.cuh (shared with the CPU test build), the ASCII windows come
// from the scanning prefilters above.  Not a hot path: the reference documents it as unoptimised too.
__global__ void __launch_bounds__(128) k_match_indices(const FrzCorpusView cv, const __grid_constant__ FrzPatternDev pat,
                                                       const __grid_constant__ FrzUNeedle un, const FrzUScoring usc, int unicode,
                                                       const uint32_t* __restrict__ which, unsigned long long n,
                                                       FrzMatchDev* __restrict__ out_matches, uint32_t* __restrict__ out_idx,
                                                       uint32_t stride, uint32_t* __restrict__ out_cnt,
                                                       uint16_t* __restrict__ scratch, unsigned long long scratch_stride) {
    const unsigned long long tid = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned long long nthreads = (unsigned long long)gridDim.x * blockDim.x;
    uint16_t* my_scratch = scratch + tid * scratch_stride;
    const int max_typos = pat.typo_mode == FRZ_T_NONE ? -1 : pat.typo_mode == FRZ_T_0 ? 0 : pat.typo_mode == FRZ_T_1 ? 1
                        : pat.typo_mode == FRZ_T_2 ? 2 : pat.max_typos;
    for (unsigned long long j = tid; j < n; j += nthreads) {
        const uint32_t idx = which[j];
        out_cnt[j] = 0xFFFFFFFFu;
        if (idx >= cv.n) continue;
        const uint32_t tile = idx >> FRZ_TILE_SHIFT;
        const uint32_t slot = cv.slot_of[idx];
        const uint32_t meta = cv.slot_meta[(uint64_t)tile * FRZ_TILE + slot];
        const int len = (int)(meta >> FRZ_TILE_SHIFT);
        const FrzGroupDesc gd = cv.groups[tile * FRZ_GROUPS_PER_TILE + (slot >> 5)];
        const GlobalAcc ga{cv.data + frz_slot_unit0(gd, slot & 31)};
        const FrzPackedHay hay{ga.base, 0};
        uint32_t* my_out = out_idx + j * (unsigned long long)stride;
        uint32_t score = 0;
        bool exact = false;
        int cnt = 0;
        if (pat.matching != FRZ_MATCHING_FUZZY) {
            int pos = 0;
            const bool ok = unicode ? frzu::lit_find(un, usc, hay, len, pat.matching, &pos, &score) : lit_find(ga, pat, len, &pos, &score);
            if (!ok) continue;
            exact = pos == 0 && pat.n == len;
            for (int i = pos + pat.n - 1; i >= pos; i--) { if (cnt < (int)stride) my_out[cnt] = (uint32_t)i; cnt++; }
        } else {
            if (len < pat.min_hay_len) continue;
            int start = 0, end = len;
            bool ok;
            if (unicode) ok = frzu::prefilter(un, hay, len, pat.pf_lanes, max_typos, &start, &end);
            else if (pat.typo_mode == FRZ_T_0) ok = window_k0(ga, pat, len, &start, &end);
            else if (pat.typo_mode == FRZ_T_1) ok = window_k1(ga, pat, len, &start, &end);
            else if (pat.typo_mode == FRZ_T_2) ok = window_k2(ga, pat, len, &start, &end);
            else if (pat.typo_mode == FRZ_T_MANY) ok = window_many(ga, pat, len, &start, &end);
            else ok = true;
            if (!ok) continue;
            start = start > 0 ? start - 1 : 0;   // trim_haystack
            const int W = end - start;
            const FrzPackedHay win{ga.base, start};
            score = frzi::sw_indices(un, unicode != 0, usc, win, W, start, max_typos, pat.sw_lanes, pat.score_bits == 8, my_scratch,
                                     my_out, (int)stride, &cnt);
            exact = start == 0 && end == len && W == pat.n;
            for (int k = 0; exact && k < W; k++) exact = win(k) == pat.c[k];
            if (exact) score = (score + (uint32_t)pat.exact_bonus) & 0xffffu;
        }
        FrzMatchDev m;
        m.index = idx; m.score = (uint16_t)score; m.exact = exact ? 1 : 0; m.pad = 0;
        out_matches[j] = m;
        out_cnt[j] = (uint32_t)cnt;   // untruncated (only the first `stride` offsets were stored)
    }
}

}  // namespace

frz_status frz_launch_prefilter_list(const FrzCorpusView& cv, const FrzPatternDev& pat, const FrzMatchDev* cand,
                                     uint64_t n_cand, uint32_t index_offset, FrzWorkspace& ws, cudaStream_t stream,
                                     FrzLaunchStats* st) {
    if (cv.n_tiles == 0) return FRZ_OK;
    const size_t smem = sizeof(OccTable) * kWarps;
    FRZ_CUDA_TRY(cudaMemsetAsync(ws.surv_bitmap, 0, (size_t)cv.n_tiles * 32 * sizeof(uint32_t), stream));
    if (n_cand == 0) return FRZ_OK;
    const uint32_t grid = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(148 * 4, (n_cand + kThreads - 1) / kThreads));
#define FRZ_PFL_LAUNCH(MODE)                                                                                     \
    k_prefilter_list<MODE><<<grid, kThreads, smem, stream>>>(cv, pat, cand, n_cand, index_offset, ws.lists(),    \
                                                             ws.survivor_cap, ws.surv_bitmap, ws.counters)
    switch (pat.typo_mode) {
        case FRZ_T_0: FRZ_PFL_LAUNCH(FRZ_T_0); break;
        case FRZ_T_1: FRZ_PFL_LAUNCH(FRZ_T_1); break;
        case FRZ_T_2: FRZ_PFL_LAUNCH(FRZ_T_2); break;
        case FRZ_T_MANY: FRZ_PFL_LAUNCH(FRZ_T_MANY); break;
        case FRZ_T_NONE: FRZ_PFL_LAUNCH(FRZ_T_NONE); break;
        case FRZ_T_LITERAL: FRZ_PFL_LAUNCH(FRZ_T_LITERAL); break;
        default: return frz_fail(FRZ_ERR_INVALID_ARG, "bad typo mode %d", pat.typo_mode);
    }
#undef FRZ_PFL_LAUNCH
    FRZ_CUDA_TRY(cudaGetLastError());
    if (st) st->launches++;
    return FRZ_OK;
}

// Stage 1a alone: the streaming signature scan over the whole corpus → candidate records in ws.cand_list, their number in
// ws.counters->cand_count.  Shared by the byte path (k_window consumes the records) and the unicode path (k_unicode does).
frz_status frz_launch_sig_scan(const FrzCorpusView& cv, const FrzPatternDev& pat, FrzWorkspace& ws, cudaStream_t stream, FrzLaunchStats* st) {
    if (cv.n_tiles == 0) return FRZ_OK;
    int sms = 0, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (sms <= 0) sms = 148;
    CandRec* cand = reinterpret_cast<CandRec*>(ws.cand_list);
    {   // persistent warps, as many blocks as fit
        const uint32_t total_chunks = cv.n_tiles * (FRZ_TILE / 128);
        const int use_sig = pat.typo_mode != FRZ_T_NONE && pat.sig_on;
        const size_t smem = (sizeof(CandRec) * kScanRing + sizeof(ScanStage) * kScanStages + sizeof(uint64_t) * kScanStages) * kScanWarps;
        static int bps_dev[64] = {};
        int& bps = bps_dev[frz_current_device() & 63];
        if (!bps) {
            FRZ_CUDA_TRY(cudaFuncSetAttribute(k_sig_scan, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            FRZ_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, k_sig_scan, kScanThreads, smem));
            if (bps < 1) bps = 1;
        }
        const uint32_t grid = std::max<uint32_t>(1, std::min<uint32_t>((uint32_t)(sms * bps), (total_chunks + kScanWarps - 1) / kScanWarps));
        k_sig_scan<<<grid, kScanThreads, smem, stream>>>(cv, use_sig, pat.sig_need1, pat.sig_need2, pat.sig_k, pat.min_hay_len, cand,
                                                         ws.cand_cap, ws.counters);
    }
    FRZ_CUDA_TRY(cudaGetLastError());
    if (st) st->launches++;
    return FRZ_OK;
}

// Stage 1 of match_list over the whole corpus: k_sig_scan (streaming signature test → candidate records) and
// k_window (exact windows of the candidates → survivor records + per-tile survivor bitmap).
frz_status frz_launch_prefilter(const FrzCorpusView& cv, const FrzPatternDev& pat, FrzWorkspace& ws, cudaStream_t stream,
                                FrzLaunchStats* st) {
    if (cv.n_tiles == 0) return FRZ_OK;
    int sms = 0, dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (sms <= 0) sms = 148;
    FRZ_CUDA_TRY(cudaMemsetAsync(ws.surv_bitmap, 0, (size_t)cv.n_tiles * 32 * sizeof(uint32_t), stream));
    CandRec* cand = reinterpret_cast<CandRec*>(ws.cand_list);
    FRZ_TRY(frz_launch_sig_scan(cv, pat, ws, stream, st));   // 1a
    const size_t smem = sizeof(WinSmem) * kWinWarps;
#define FRZ_PF_LAUNCH(MODE)                                                                                              \
    do {                                                                                                                 \
        static int bps_dev[64] = {};                                                                                     \
        int& bps = bps_dev[frz_current_device() & 63];                                                                   \
        if (!bps) {                                                                                                      \
            FRZ_CUDA_TRY(cudaFuncSetAttribute(k_window<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));  \
            FRZ_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, k_window<MODE>, kWinThreads, smem));        \
            /* measured on B200, slot-major layout (profiles/r02j_variants.txt): 5 / 4 / 3 resident blocks per SM give */ \
            /* 0.1302 / 0.1328 / 0.1429 ms for the stage (with the interleaved layout 4 beat 5: each candidate touched */  \
            /* four lines and more warps thrashed L1, profiles/r02f_variants.txt) */                                      \
            if (bps > 5) bps = 5;                                                                                        \
            if (bps < 1) bps = 1;                                                                                        \
        }                                                                                                                \
        k_window<MODE><<<sms * bps, kWinThreads, smem, stream>>>(cv, pat, cand, ws.cand_cap, ws.lists(), ws.survivor_cap, \
                                                                 ws.surv_bitmap, ws.counters);                           \
    } while (0)
    switch (pat.typo_mode) {
        case FRZ_T_0: FRZ_PF_LAUNCH(FRZ_T_0); break;
        case FRZ_T_1: FRZ_PF_LAUNCH(FRZ_T_1); break;
        case FRZ_T_2: FRZ_PF_LAUNCH(FRZ_T_2); break;
        case FRZ_T_MANY: FRZ_PF_LAUNCH(FRZ_T_MANY); break;
        case FRZ_T_NONE: FRZ_PF_LAUNCH(FRZ_T_NONE); break;
        case FRZ_T_LITERAL: FRZ_PF_LAUNCH(FRZ_T_LITERAL); break;
        default: return frz_fail(FRZ_ERR_INVALID_ARG, "bad typo mode %d", pat.typo_mode);
    }
#undef FRZ_PF_LAUNCH
    FRZ_CUDA_TRY(cudaGetLastError());
    if (st) st->launches++;
    return FRZ_OK;
}

frz_status frz_launch_tile_scan(const FrzCorpusView& cv, FrzWorkspace& ws, cudaStream_t stream, FrzLaunchStats* st,
                                unsigned long long* carry) {
    if (cv.n_tiles) {
        k_tile_rank<<<(cv.n_tiles * 32 + 255) / 256, 256, 0, stream>>>(ws.surv_bitmap, ws.word_prefix, ws.tile_count, cv.n_tiles);
        if (st) st->launches++;
    }
    k_tile_scan<<<1, 1024, 0, stream>>>(ws.tile_count, ws.tile_out_base, cv.n_tiles, ws.counters, carry);
    FRZ_CUDA_TRY(cudaGetLastError());
    if (st) st->launches++;
    return FRZ_OK;
}

frz_status frz_launch_match_indices(const FrzCorpusView& cv, const FrzPatternDev& pat, const FrzUNeedle& un, const FrzUScoring& usc,
                                    bool unicode, const uint32_t* d_which, uint64_t n, FrzMatchDev* d_matches, uint32_t* d_idx,
                                    uint32_t stride, uint32_t* d_cnt, uint16_t* d_scratch, uint64_t scratch_stride, uint32_t threads,
                                    cudaStream_t stream) {
    if (n == 0) return FRZ_OK;
    const uint32_t grid = (threads + 127) / 128;
    k_match_indices<<<grid, 128, 0, stream>>>(cv, pat, un, usc, unicode ? 1 : 0, d_which, n, d_matches, d_idx, stride, d_cnt,
                                              d_scratch, scratch_stride);
    FRZ_CUDA_TRY(cudaGetLastError());
    return FRZ_OK;
}
