// kc_jsongpu.cuh — H1g: the JSON-in / JSON-out path of the consolidator ON THE DEVICE.
//
// The reference's unit of work is n candidate JSON texts -> consensus JSON (+ likelihoods): json.loads per candidate
// (consolidation.py:25-38), the dict part of recursive_list_alignments (consensus_utils.py:516-548: every candidate gets
// every key, keys SORTED), the dispatcher (:1376-1454), sanitize_value (:925-933), the vote / numeric consensus (K1 / K2),
// and json.dumps of the result (consolidation.py:41-60).  Round 1 did everything around K1/K2 on host threads (H1,
// kc_json.cpp): 211 k records/s against 2 G records/s for the kernels.  Here the candidate texts are copied to the GPU as
// they are and the GPU does the whole chain; the host only moves bytes:
//
//   A0  count_kernel    one thread per record scans candidate 0 -> number of fields F_r        (then an exclusive scan: slots)
//   A1  plan_kernel     a TEAM of lanes per record (team size = n rounded up to a power of two, <= 32):
//         parse   lane c scans candidate c, one 16-byte token (key span, value span, kind) per field
//         type    lane j (one per token): same shape in every candidate (same keys, nested objects open / close at the same
//                 positions), duplicate / special keys, rank of the key among its siblings in sorted order, which kernel
//                 decides the field (plan_leaf of kc_json.cpp)
//         order   nested records: the token's position in output order (depth-first, keys sorted at every level)
//         slots   the team leader numbers the record's vote / numeric groups and reserves rows in the batch's cell matrices
//         encode  lane j: sanitised-equality classes -> int8 local codes (K1 cells), exact decimal -> float64 (K2 cells)
//   A2  medoid_kernel   only when the chunk has multi-word string fields (three exclusive scans of the per-record counts first):
//                       lane j writes its field's normalised strings and their offsets in K4's CSR form
//   K1  kc_vote_i8, K2  kc_numeric_f64, K4  kc_medoid_str on the cell matrices / string groups — the kernels of the columnar path
//   C0  len_kernel      lane j formats its field's value and confidence (float.__repr__ by Ryu) to learn the lengths; the
//                       leader turns them into piece offsets and record lengths          (then two exclusive scans: offsets)
//   C1  write_kernel    lane j writes `"key": value` / `"key": confidence` at its offset of the two output blobs
//
// A record the device path does not model exactly (\u escapes, escapes in keys, non-ASCII, nested values or lists, candidates with different
// keys, multi-word strings outside K4's contract, numbers outside the exact-conversion range, ...) gets a non-zero status and is
// consolidated by the host path (kc_consolidate_json) instead: the device path never guesses.
//
// The phases are plain __host__ __device__ functions of (chunk, record, lane, team size) that communicate through global
// arrays only — no warp intrinsics — so the CPU tests run the SAME code on the host, lane by lane (kc_debug_jsongpu_*).
#pragma once

#include "kc_jsoncore.cuh"

namespace kc {
namespace js {

constexpr int32_t kMaxFields = 1024;  // per record; the key ranking is quadratic in it

// field descriptor word: kind:3 | last of its siblings in key order:1 | rank among its siblings:12 | group index within the record:16
KC_HD inline uint32_t fdesc_pack(uint32_t kind, uint32_t last, uint32_t rank, uint32_t gidx) { return kind | (last << 3) | (rank << 4) | (gidx << 16); }
KC_HD inline uint32_t fdesc_kind(uint32_t d) { return d & 7u; }
KC_HD inline uint32_t fdesc_last(uint32_t d) { return (d >> 3) & 1u; }
KC_HD inline uint32_t fdesc_rank(uint32_t d) { return (d >> 4) & 0xFFFu; }
KC_HD inline uint32_t fdesc_gidx(uint32_t d) { return d >> 16; }

struct Chunk {
    const uint8_t *text;  // the chunk's candidate texts (device copy), text[0] is byte off[0] of the caller's blob
    const int64_t *off;   // [R*n + 1] byte offsets of the candidate texts in the caller's blob (record-major)
    int32_t R, n;
    uint32_t *fcount;   // [R]   A0: tokens of candidate 0 (0 when it does not scan)
    uint8_t *nest;      // [R]   A0: 1 when candidate 0 holds a nested object
    uint32_t *gpos;     // [slots] nested records only: the token's position in OUTPUT order (sorted keys at every level)
    uint32_t *slot;     // [R+1] exclusive scan of fcount: the record's first field slot
    uint8_t *status;    // [R]   0 = on the device path, else D_*
    Tok *toks;          // [slots * n] token of (field slot, candidate)
    uint32_t *fdesc;    // [slots]
    uint32_t *vbase, *xbase;        // [R] first vote / numeric group of the record
    unsigned long long *counters;   // [0] vote groups, [1] numeric groups, [2] medoid groups of the chunk
    int8_t *vcells;     // [vote groups][n]   K1 cells
    double *xcells;     // [numeric groups][n] K2 cells
    // medoid fields (multi-word strings): per record the groups of >= 2 strings, their strings and normalised characters;
    // after the exclusive scans (in place, entry R = the totals) the record's first group / string / character
    uint32_t *mcount, *scount, *ccount;  // [R+1]
    uint8_t *mchars;                     // K4 input: normalised strings back to back
    int32_t *mstr_off, *mgrp_off;        //           [strings + 1], [groups + 1]
    const int32_t *midx;                 // K4 results: medoid's index within its group,
    const double *mavg;                  //             its mean similarity
    const uint32_t *vmeta;   // K1 result words
    int32_t *vrec;           // likelihood-weighted entry only (else NULL): [vote groups] the record of each vote group (slots)
    const float *vsums;      // likelihood-weighted entry only (else NULL): [vote groups][2] (W_win, W_present) of the weighted vote
    const double *xvalue;    // K2 values
    const uint32_t *xmeta;   // K2 result words
    uint32_t *piece_c, *piece_l;  // [slots] by (slot + rank): piece length, then (after the leader's pass) piece offset
    int64_t *len_c, *len_l;       // [R+1] record lengths -> (exclusive scan, in place) record offsets in the output blobs
    uint8_t *out_c, *out_l;       // output blobs: consensus texts, likelihoods texts
};

KC_HD inline uint8_t load_status(const Chunk &ch, int32_t r) { return *(volatile const uint8_t *)(ch.status + r); }
KC_HD inline void decline(const Chunk &ch, int32_t r, int32_t why) { *(volatile uint8_t *)(ch.status + r) = (uint8_t)why; }

// ---------------------------------------------------------------- A0

KC_HD inline void count_record(const Chunk &ch, int32_t r) {
    const int64_t b = ch.off[(int64_t)r * ch.n], e = ch.off[(int64_t)r * ch.n + 1];
    int32_t f = -D_TOO_LONG;
    bool nested = false;
    if (e - b < ((int64_t)1 << 31)) f = scan_object(ch.text + (b - ch.off[0]), (uint32_t)(e - b), 0, nullptr, 0, kMaxFields, &nested);
    ch.fcount[r] = f > 0 ? (uint32_t)f : 0u;
    ch.nest[r] = nested ? 1 : 0;
    ch.status[r] = f > 0 ? (uint8_t)D_OK : (uint8_t)(-f);
}

// ---------------------------------------------------------------- A1

KC_HD inline void parse_phase(const Chunk &ch, int32_t r, int32_t lane, int32_t team) {
    if (load_status(ch, r)) return;
    const int32_t F = (int32_t)ch.fcount[r];
    const int64_t base0 = ch.off[0];
    for (int32_t c = lane; c < ch.n; c += team) {
        const int64_t b = ch.off[(int64_t)r * ch.n + c], e = ch.off[(int64_t)r * ch.n + c + 1];
        int32_t f = -D_TOO_LONG;
        if (e - b < ((int64_t)1 << 31) && (b - base0) + (e - b) < ((int64_t)1 << 32))
            f = scan_object(ch.text + (b - base0), (uint32_t)(e - b), (uint32_t)(b - base0), ch.toks + (int64_t)ch.slot[r] * ch.n + c, ch.n, F);
        if (f < 0) decline(ch, r, f == -D_TOO_MANY_FIELDS ? D_KEYS_DIFFER : -f);
        else if (f != F) decline(ch, r, D_KEYS_DIFFER);
    }
}

// The siblings of a token at depth d: the tokens of depth d (other than K_CLOSE) in [lo, hi), the widest range around it in which
// no token is shallower.  A flat record: every token.
KC_HD inline void sibling_range(const Tok *rt, int32_t n, int32_t F, int32_t j, uint32_t d, bool flat, int32_t &lo, int32_t &hi) {
    lo = 0;
    hi = F;
    if (flat) return;
    lo = j;
    while (lo > 0 && tok_depth(rt[(int64_t)(lo - 1) * n]) >= d) --lo;
    hi = j + 1;
    while (hi < F && tok_depth(rt[(int64_t)hi * n]) >= d) ++hi;
}

KC_HD inline void type_phase(const Chunk &ch, int32_t r, int32_t lane, int32_t team) {
    if (load_status(ch, r)) return;
    const int32_t F = (int32_t)ch.fcount[r], n = ch.n;
    const bool flat = ch.nest[r] == 0;
    const Tok *rt = ch.toks + (int64_t)ch.slot[r] * n;
    for (int32_t j = lane; j < F; j += team) {
        const Tok *row = rt + (int64_t)j * n;
        const uint32_t k0 = row[0].kind, d = tok_depth(row[0]);
        // the same SHAPE in every candidate: the same key at position j, nested objects open and close at the same positions
        // (else the key union / missing -> None / None -> dict of Nones logic of the pre-pass is the host path's, cu:516-548)
        int32_t ref = j;  // the token whose key orders this one among its siblings: itself, or a K_CLOSE's K_OPEN
        if (k0 == K_CLOSE) {
            for (int32_t c = 1; c < n; ++c)
                if (row[c].kind != K_CLOSE || tok_depth(row[c]) != d) {
                    decline(ch, r, D_KEYS_DIFFER);
                    return;
                }
            ref = j - 1;  // its K_OPEN: the nearest token to the left at the same depth (everything between them is deeper)
            while (ref > 0 && tok_depth(rt[(int64_t)ref * n]) != d) --ref;
        }
        const uint8_t *key = ch.text + rt[(int64_t)ref * n].kstart;
        const uint32_t klen = rt[(int64_t)ref * n].klen;
        if (k0 != K_CLOSE) {
            for (int32_t c = 1; c < n; ++c) {
                if ((row[c].kind == K_OPEN) != (k0 == K_OPEN) || row[c].kind == K_CLOSE) {  // an object here, a scalar / None there
                    decline(ch, r, D_NESTED);
                    return;
                }
                if (tok_depth(row[c]) != d || row[c].klen != klen || key_compare(ch.text + row[c].kstart, klen, key, klen) != 0) {
                    decline(ch, r, D_KEYS_DIFFER);
                    return;
                }
            }
            if (contains(key, klen, "reasoning___", 12) || contains(key, klen, "source___", 9) ||  // skipped by consensus_dict (cu:1287-1294)
                (F == 1 && klen == 4 && key_compare(key, 4, (const uint8_t *)"text", 4) == 0)) {   // {"text": s} -> s (cons:55-57)
                decline(ch, r, D_SPECIAL_KEY);
                return;
            }
        }
        // position of the key among its siblings in sorted order (cu:521-522, at every level); duplicates: dict semantics, host path
        int32_t lo, hi;
        sibling_range(rt, n, F, ref, d, flat, lo, hi);
        uint32_t rank = 0, after = 0;
        for (int32_t i = lo; i < hi; ++i) {
            const Tok &o = rt[(int64_t)i * n];
            if (i == ref || (!flat && (tok_depth(o) != d || o.kind == K_CLOSE))) continue;
            const int cmp = key_compare(ch.text + o.kstart, o.klen, key, klen);
            if (cmp == 0) {
                decline(ch, r, D_DUP_KEY);
                return;
            }
            rank += cmp < 0 ? 1u : 0u;
            after += cmp > 0 ? 1u : 0u;
        }
        const uint32_t last = after == 0 ? 1u : 0u;
        if (k0 == K_OPEN || k0 == K_CLOSE) {
            ch.fdesc[ch.slot[r] + j] = fdesc_pack(k0 == K_OPEN ? F_OPEN : F_CLOSE, last, rank, 0);
            continue;
        }
        // which kernel decides the field (plan_leaf, kc_json.cpp; cu:1405-1411, :1443-1453)
        int32_t first = -1;
        for (int32_t c = 0; c < n && first < 0; ++c)
            if (row[c].kind != K_NULL) first = c;
        uint32_t kind;
        if (first < 0) {
            kind = F_ALLNULL;
        } else if (row[first].kind == K_STR) {
            kind = F_VOTE_STR;
            for (int32_t c = 0; c < n; ++c) {
                if (row[c].kind == K_NULL) continue;
                if (row[c].kind != K_STR) {  // str(v) of numbers / bools inside a string field: host path
                    decline(ch, r, D_MIXED_TYPES);
                    return;
                }
                if (row[c].flags & TOK_MULTIWORD) kind = F_MEDOID;  // not enum-like (cu:1405): the similarity medoid (cu:1221-1237)
            }
            if (kind == F_MEDOID) {
                // K4 takes the group when every pair is a Levenshtein pair inside its contract (plan_leaf of kc_json.cpp, the
                // rule of columnar.Plan._medoid_on_device under the default similarity method): at most one string longer than
                // 50 characters (two would go to the embeddings service, cu:813), at most one normalised string longer than 64
                uint32_t live = 0, chars = 0, long_raw = 0, long_norm = 0;
                bool fits = true;
                for (int32_t c = 0; c < n; ++c) {
                    if (row[c].kind == K_NULL) continue;
                    const uint32_t nl = sanitized_copy(ch.text + row[c].vstart, row[c].vlen, nullptr);
                    ++live;
                    chars += nl;
                    const uint32_t raw = (row[c].flags & TOK_ESCAPED) ? unescaped_length(ch.text + row[c].vstart, row[c].vlen) : row[c].vlen;
                    long_raw += raw > 50u ? 1u : 0u;
                    long_norm += nl > 64u ? 1u : 0u;
                    fits &= nl <= 2000u;
                }
                if (live >= 2 && (!fits || long_raw > 1 || long_norm > 1)) {
                    decline(ch, r, D_MULTIWORD);
                    return;
                }
                ch.piece_c[ch.slot[r] + j] = live;   // scratch until C0: read by the leader in slots_phase
                ch.piece_l[ch.slot[r] + j] = chars;
            }
        } else if (row[first].kind == K_TRUE || row[first].kind == K_FALSE) {
            kind = F_VOTE_BOOL;
            for (int32_t c = 0; c < n; ++c)
                if (row[c].kind > K_FALSE) {  // a string may be multi-word, `v or False` of other objects: host path
                    decline(ch, r, D_MIXED_TYPES);
                    return;
                }
        } else {
            kind = F_NUMERIC;  // strings / bools among the cells are "present, not a number" (cu:1105-1114)
        }
        ch.fdesc[ch.slot[r] + j] = fdesc_pack(kind, last, rank, 0);
    }
}

// Nested records only, after type_phase: the token's position in output order.  Output is a depth-first walk with the members
// of every object in key order, so a token comes after its parent's K_OPEN and after the whole subtrees of the siblings that
// sort before it; a K_CLOSE comes last in its object's subtree.
KC_HD inline void order_phase(const Chunk &ch, int32_t r, int32_t lane, int32_t team) {
    if (load_status(ch, r) || ch.nest[r] == 0) return;
    const int32_t F = (int32_t)ch.fcount[r], n = ch.n;
    const Tok *rt = ch.toks + (int64_t)ch.slot[r] * n;
    const uint32_t *fd = ch.fdesc + ch.slot[r];
    auto subtree = [&](int32_t i) -> uint32_t {  // tokens in the subtree of token i (itself included)
        if (rt[(int64_t)i * n].kind != K_OPEN) return 1u;
        const uint32_t d = tok_depth(rt[(int64_t)i * n]);
        int32_t e = i + 1;
        while (tok_depth(rt[(int64_t)e * n]) != d) ++e;  // its K_CLOSE
        return (uint32_t)(e - i + 1);
    };
    for (int32_t j = lane; j < F; j += team) {
        const bool closing = rt[(int64_t)j * n].kind == K_CLOSE;
        uint32_t d = tok_depth(rt[(int64_t)j * n]);
        int32_t cur = j;
        if (closing) {
            cur = j - 1;
            while (cur > 0 && tok_depth(rt[(int64_t)cur * n]) != d) --cur;
        }
        uint32_t pos = closing ? subtree(cur) - 1u : 0u;
        for (;;) {
            int32_t lo, hi;
            sibling_range(rt, n, F, cur, d, false, lo, hi);
            const uint32_t rank = fdesc_rank(fd[cur]);
            for (int32_t i = lo; i < hi; ++i) {
                const Tok &o = rt[(int64_t)i * n];
                if (i == cur || tok_depth(o) != d || o.kind == K_CLOSE) continue;
                if (fdesc_rank(fd[i]) < rank) pos += subtree(i);
            }
            if (d == 0) break;
            pos += 1u;     // the parent's K_OPEN, the token just before the first sibling
            cur = lo - 1;
            --d;
        }
        ch.gpos[ch.slot[r] + j] = pos;
    }
}

KC_HD inline uint32_t out_pos(const Chunk &ch, int32_t r, int32_t j) {
    return ch.nest[r] ? ch.gpos[ch.slot[r] + j] : fdesc_rank(ch.fdesc[ch.slot[r] + j]);
}

// team leader only: number the groups, reserve rows of the cell matrices (chunk-wide counters)
KC_HD inline void slots_phase(const Chunk &ch, int32_t r) {
    if (load_status(ch, r)) return;
    const int32_t F = (int32_t)ch.fcount[r];
    uint32_t *fd = ch.fdesc + ch.slot[r];
    uint32_t nv = 0, nx = 0, nm = 0, ns = 0, nc = 0;
    for (int32_t j = 0; j < F; ++j) {
        const uint32_t d = fd[j], kind = fdesc_kind(d);
        uint32_t g = 0;
        if (kind == F_VOTE_STR || kind == F_VOTE_BOOL) {
            g = nv++;
        } else if (kind == F_NUMERIC) {
            g = nx++;
        } else if (kind == F_MEDOID) {
            uint32_t *pc = ch.piece_c + ch.slot[r] + j, *pl = ch.piece_l + ch.slot[r] + j;
            const uint32_t live = *pc, chars = *pl;
            if (live >= 2) {  // one string alone is its own consensus (cu:1085-1086): no group
                g = nm++;
                *pc = ns;     // the group's first string / character within the record, for medoid_phase
                *pl = nc;
                ns += live;
                nc += chars;
            }
        }
        fd[j] = d | (g << 16);
    }
    ch.mcount[r] = nm;
    ch.scount[r] = ns;
    ch.ccount[r] = nc;
#ifdef __CUDA_ARCH__
    ch.vbase[r] = (uint32_t)atomicAdd(ch.counters + 0, (unsigned long long)nv);
    ch.xbase[r] = (uint32_t)atomicAdd(ch.counters + 1, (unsigned long long)nx);
    if (nm) atomicAdd(ch.counters + 2, (unsigned long long)nm);
#else
    ch.vbase[r] = (uint32_t)ch.counters[0];
    ch.counters[0] += nv;
    ch.xbase[r] = (uint32_t)ch.counters[1];
    ch.counters[1] += nx;
    ch.counters[2] += nm;
#endif
    if (ch.vrec)  // the weighted vote finds the record's weight row through it; a record's groups are contiguous
        for (uint32_t k = 0; k < nv; ++k) ch.vrec[ch.vbase[r] + k] = r;
}

// A2, after the exclusive scans of mcount / scount / ccount: lane j writes its medoid group in K4's CSR form.  Group, string
// and character ranges follow RECORD order (scans, not atomics), so the three offset arrays are monotonic as CSR needs.  A
// record that was declined after slots_phase (a number out of range) still owns its ranges and fills them: K4 reads every group.
KC_HD inline void medoid_phase(const Chunk &ch, int32_t r, int32_t lane, int32_t team) {
    const uint32_t g0 = ch.mcount[r], g1 = ch.mcount[r + 1];
    if (g0 == g1) return;
    const int32_t F = (int32_t)ch.fcount[r], n = ch.n;
    const Tok *rt = ch.toks + (int64_t)ch.slot[r] * n;
    const uint32_t n_groups = ch.mcount[ch.R], n_strings = ch.scount[ch.R];
    for (int32_t j = lane; j < F; j += team) {
        const uint32_t d = ch.fdesc[ch.slot[r] + j];
        if (fdesc_kind(d) != F_MEDOID) continue;
        const Tok *row = rt + (int64_t)j * n;
        uint32_t live = 0;
        for (int32_t c = 0; c < n; ++c) live += row[c].kind != K_NULL ? 1u : 0u;
        if (live < 2) continue;
        const uint32_t g = g0 + fdesc_gidx(d);
        uint32_t s = ch.scount[r] + ch.piece_c[ch.slot[r] + j], at = ch.ccount[r] + ch.piece_l[ch.slot[r] + j];
        ch.mgrp_off[g] = (int32_t)s;
        for (int32_t c = 0; c < n; ++c) {
            if (row[c].kind == K_NULL) continue;
            ch.mstr_off[s++] = (int32_t)at;
            at += sanitized_copy(ch.text + row[c].vstart, row[c].vlen, ch.mchars + at);
        }
        if (g + 1 == n_groups) {  // the chunk's last group closes both offset arrays
            ch.mgrp_off[n_groups] = (int32_t)n_strings;
            ch.mstr_off[n_strings] = (int32_t)at;
        }
    }
}

KC_HD inline void encode_phase(const Chunk &ch, int32_t r, int32_t lane, int32_t team) {
    if (load_status(ch, r)) return;
    const int32_t F = (int32_t)ch.fcount[r], n = ch.n;
    const Tok *rt = ch.toks + (int64_t)ch.slot[r] * n;
    for (int32_t j = lane; j < F; j += team) {
        const Tok *row = rt + (int64_t)j * n;
        const uint32_t d = ch.fdesc[ch.slot[r] + j], kind = fdesc_kind(d), g = fdesc_gidx(d);
        if (kind == F_VOTE_STR) {
            // local dictionary codes: the class of a cell is the first earlier cell with the same sanitised text
            int8_t *cells = ch.vcells + ((int64_t)ch.vbase[r] + g) * n;
            int32_t n_classes = 0;
            for (int32_t c = 0; c < n; ++c) {
                if (row[c].kind == K_NULL) {
                    cells[c] = (int8_t)KC_CODE_NONE;
                    continue;
                }
                int32_t code = -1;
                for (int32_t p = 0; p < c && code < 0; ++p)
                    if (row[p].kind != K_NULL && cells[p] >= 0 &&
                        sanitized_equal(ch.text + row[p].vstart, row[p].vlen, ch.text + row[c].vstart, row[c].vlen))
                        code = cells[p];
                cells[c] = (int8_t)(code >= 0 ? code : n_classes++);
            }
        } else if (kind == F_VOTE_BOOL) {
            int8_t *cells = ch.vcells + ((int64_t)ch.vbase[r] + g) * n;
            for (int32_t c = 0; c < n; ++c) cells[c] = row[c].kind == K_TRUE ? 1 : 0;  // None and False -> False (cu:956)
        } else if (kind == F_NUMERIC) {
            double *cells = ch.xcells + ((int64_t)ch.xbase[r] + g) * n;
            for (int32_t c = 0; c < n; ++c) {
                const Tok &t = row[c];
                double v;
                if (t.kind == K_NULL) {
                    v = bits_f64(KC_F64_NONE_BITS);
                } else if (t.kind == K_INT || t.kind == K_FLOAT) {
                    if (!to_double(ch.text + t.vstart, t.vlen, v)) {
                        decline(ch, r, D_NUMBER_RANGE);  // rows stay reserved; the emit phases skip the record
                        return;
                    }
                    if (t.kind == K_INT && v == 0.0) v = 0.0;  // int("-0") is 0: no negative zero from integers
                } else {
                    v = bits_f64(0x7FF8000000000000ull);  // bool / str: counted, never clustered
                }
                cells[c] = v;
            }
        }
    }
}

// ---------------------------------------------------------------- C0 / C1

// value and confidence of one field, formatted into the two sinks (the epilogue emit_leaf of kc_json.cpp:
// cu:971-982, cu:1085-1086, cu:1116, cu:1177-1219)
KC_HD inline void format_field(const Chunk &ch, int32_t r, int32_t j, Sink &content, Sink &lik) {
    const int32_t n = ch.n;
    const Tok *row = ch.toks + ((int64_t)ch.slot[r] + j) * n;
    const uint32_t d = ch.fdesc[ch.slot[r] + j], kind = fdesc_kind(d), g = fdesc_gidx(d);
    double conf = 0.0;
    if (kind == F_VOTE_STR || kind == F_VOTE_BOOL) {
        const uint32_t m = ch.vmeta[(int64_t)ch.vbase[r] + g];
        const uint32_t idx = KC_META_IDX(m), support = KC_META_SUPPORT(m), present = KC_META_PRESENT(m);
        if (kind == F_VOTE_BOOL) {
            content.lit(row[idx].kind == K_TRUE ? "true" : "false");  // the processed key (cu:958)
        } else {
            content.json_string(ch.text + row[idx].vstart, row[idx].vlen, row[idx].flags & TOK_ESCAPED);  // first original whose sanitised form wins (cu:971)
        }
        if (ch.vsums) {  // likelihood-weighted: the weighted form of support / present (DESIGN.md §5)
            const float *ws = ch.vsums + 2 * ((int64_t)ch.vbase[r] + g);
            conf = py_round5(1.0 * ((double)ws[0] / (double)ws[1]));
        } else {
            conf = py_round5(1.0 * ((double)support / (double)present));
        }
    } else if (kind == F_NUMERIC) {
        const uint32_t m = ch.xmeta[(int64_t)ch.xbase[r] + g];
        const uint32_t idx = KC_META_IDX(m), support = KC_META_SUPPORT(m), nn = KC_META_NN(m), present = KC_META_PRESENT(m);
        const uint32_t flags = KC_META_FLAGS(m);
        if (flags & KC_FLAG_HAS_VALUE) {
            if (flags & KC_FLAG_SINGLE) {  // the original object, confidence unrounded (cu:1085-1086)
                const Tok &t = row[idx];
                if (t.kind == K_INT) {
                    if (t.vlen == 2 && ch.text[t.vstart] == '-' && ch.text[t.vstart + 1] == '0') content.put('0');
                    else content.put(ch.text + t.vstart, t.vlen);
                } else if (t.kind == K_FLOAT) {
                    double v = 0.0;
                    to_double(ch.text + t.vstart, t.vlen, v);
                    float_repr(v, content);
                } else if (t.kind == K_STR) {
                    content.json_string(ch.text + t.vstart, t.vlen, t.flags & TOK_ESCAPED);
                } else {
                    content.lit(t.kind == K_TRUE ? "true" : (t.kind == K_FALSE ? "false" : "null"));
                }
                conf = 1.0 * (1.0 / (double)present) * (1.0 / 1.0);
            } else {
                float_repr(ch.xvalue[(int64_t)ch.xbase[r] + g], content);
                conf = py_round5((double)support / (double)nn);
            }
        } else {
            content.lit("null");
            if (flags & KC_FLAG_NO_FINITE) conf = 1.0 * ((double)nn / (double)present);
            else conf = present == 0 ? 1.0 : 0.0;
        }
    } else if (kind == F_MEDOID) {
        // cu:1444 then cu:1085-1086 (one non-None string: itself, unrounded) or cu:1233-1237 (the medoid, rounded)
        uint32_t live = 0;
        for (int32_t c = 0; c < n; ++c) live += row[c].kind != K_NULL ? 1u : 0u;
        const double sub = 1.0 * ((double)live / (double)n);
        int32_t want = 0;
        if (live >= 2) {
            const uint32_t gi = ch.mcount[r] + g;
            want = ch.midx[gi];
            conf = py_round5(sub * ch.mavg[gi]);
        } else {
            conf = sub * (1.0 / 1.0);
        }
        for (int32_t c = 0; c < n; ++c) {
            if (row[c].kind == K_NULL) continue;
            if (want-- == 0) {
                content.json_string(ch.text + row[c].vstart, row[c].vlen, row[c].flags & TOK_ESCAPED);
                break;
            }
        }
    } else {
        content.lit("null");  // all None: (None, 0.0) (cu:1401-1402)
    }
    float_repr(conf, lik);
}

KC_HD inline void len_phase(const Chunk &ch, int32_t r, int32_t lane, int32_t team) {
    if (load_status(ch, r)) return;
    const int32_t F = (int32_t)ch.fcount[r], n = ch.n;
    for (int32_t j = lane; j < F; j += team) {
        const uint32_t d = ch.fdesc[ch.slot[r] + j], kind = fdesc_kind(d), sep = fdesc_last(d) ? 0u : 2u;  // ", " unless last of its siblings
        const uint32_t klen = ch.toks[((int64_t)ch.slot[r] + j) * n].klen;
        const uint32_t pos = out_pos(ch, r, j);
        uint32_t lc, ll;
        if (kind == F_OPEN) {
            lc = ll = klen + 5u;  // "key": {
        } else if (kind == F_CLOSE) {
            lc = ll = 1u + sep;   // }
        } else {
            Sink c{nullptr, 0}, l{nullptr, 0};
            format_field(ch, r, j, c, l);
            lc = klen + 4u + (uint32_t)c.n + sep;  // "key": value
            ll = klen + 4u + (uint32_t)l.n + sep;
        }
        ch.piece_c[ch.slot[r] + pos] = lc;
        ch.piece_l[ch.slot[r] + pos] = ll;
    }
}

// team leader only: piece lengths (in key order) -> piece offsets; record lengths
KC_HD inline void offsets_phase(const Chunk &ch, int32_t r) {
    if (load_status(ch, r)) {
        ch.len_c[r] = 0;
        ch.len_l[r] = 0;
        return;
    }
    const int32_t F = (int32_t)ch.fcount[r];
    uint32_t *pc = ch.piece_c + ch.slot[r], *pl = ch.piece_l + ch.slot[r];
    uint32_t oc = 1, ol = 1;  // after '{'
    for (int32_t k = 0; k < F; ++k) {  // pieces in output order, separators included
        const uint32_t lc = pc[k], ll = pl[k];
        pc[k] = oc;
        pl[k] = ol;
        oc += lc;
        ol += ll;
    }
    ch.len_c[r] = (int64_t)oc + 1;  // '}'
    ch.len_l[r] = (int64_t)ol + 1;
}

KC_HD inline void write_phase(const Chunk &ch, int32_t r, int32_t lane, int32_t team) {
    if (load_status(ch, r)) return;
    const int32_t F = (int32_t)ch.fcount[r], n = ch.n;
    uint8_t *oc = ch.out_c + ch.len_c[r], *ol = ch.out_l + ch.len_l[r];  // len_* hold the scanned offsets now
    for (int32_t j = lane; j < F; j += team) {
        const Tok &t0 = ch.toks[((int64_t)ch.slot[r] + j) * n];
        const uint32_t d = ch.fdesc[ch.slot[r] + j], kind = fdesc_kind(d);
        const uint32_t pos = out_pos(ch, r, j);
        Sink c{oc + ch.piece_c[ch.slot[r] + pos], 0}, l{ol + ch.piece_l[ch.slot[r] + pos], 0};
        if (pos == 0) {
            oc[0] = '{';
            ol[0] = '{';
        }
        if (kind == F_CLOSE) {
            c.put('}');
            l.put('}');
        } else {
            c.put('"');
            c.put(ch.text + t0.kstart, t0.klen);
            c.lit("\": ");
            l.put('"');
            l.put(ch.text + t0.kstart, t0.klen);
            l.lit("\": ");
            if (kind == F_OPEN) {
                c.put('{');
                l.put('{');
                continue;
            }
            format_field(ch, r, j, c, l);
        }
        if (!fdesc_last(d)) {
            c.lit(", ");
            l.lit(", ");
        } else if (tok_depth(t0) == 0) {  // the last piece of the record closes the top-level object
            c.put('}');
            l.put('}');
        }
    }
}

// ---------------------------------------------------------------- kernels

#ifdef __CUDACC__

__global__ void __launch_bounds__(128) count_kernel(const Chunk ch) {
    for (int32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < ch.R; r += gridDim.x * blockDim.x) count_record(ch, r);
}

// Team t of a warp owns record (warp_index * teams_per_warp + t) of every grid-stride round; all lanes of the warp walk the
// same phases and meet at __syncwarp() (which also orders the team's global-memory traffic between phases).
__global__ void __launch_bounds__(128) plan_kernel(const Chunk ch, int32_t team) {
    const int32_t lane_w = threadIdx.x & 31, tpw = 32 / team;
    const int32_t lane = lane_w % team, t = lane_w / team;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t rounds = ((int64_t)ch.R + tpw - 1) / tpw;
    for (int64_t w = warp; w < rounds; w += n_warps) {
        const int64_t r64 = w * tpw + t;
        const bool live = r64 < ch.R;
        const int32_t r = (int32_t)r64;
        if (live) parse_phase(ch, r, lane, team);
        __syncwarp();
        if (live) type_phase(ch, r, lane, team);
        __syncwarp();
        if (live) order_phase(ch, r, lane, team);  // nested records only; reads the ranks its team wrote
        __syncwarp();
        if (live && lane == 0) slots_phase(ch, r);
        __syncwarp();
        if (live) encode_phase(ch, r, lane, team);
        __syncwarp();
    }
}

__global__ void __launch_bounds__(128) medoid_kernel(const Chunk ch, int32_t team) {
    const int32_t lane_w = threadIdx.x & 31, tpw = 32 / team;
    const int32_t lane = lane_w % team, t = lane_w / team;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t rounds = ((int64_t)ch.R + tpw - 1) / tpw;
    for (int64_t w = warp; w < rounds; w += n_warps) {
        const int64_t r64 = w * tpw + t;
        if (r64 < ch.R) medoid_phase(ch, (int32_t)r64, lane, team);
    }
}

__global__ void __launch_bounds__(128) len_kernel(const Chunk ch, int32_t team) {
    const int32_t lane_w = threadIdx.x & 31, tpw = 32 / team;
    const int32_t lane = lane_w % team, t = lane_w / team;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t rounds = ((int64_t)ch.R + tpw - 1) / tpw;
    for (int64_t w = warp; w < rounds; w += n_warps) {
        const int64_t r64 = w * tpw + t;
        const bool live = r64 < ch.R;
        const int32_t r = (int32_t)r64;
        if (live) len_phase(ch, r, lane, team);
        __syncwarp();
        if (live && lane == 0) offsets_phase(ch, r);
        __syncwarp();
    }
}

__global__ void __launch_bounds__(128) write_kernel(const Chunk ch, int32_t team) {
    const int32_t lane_w = threadIdx.x & 31, tpw = 32 / team;
    const int32_t lane = lane_w % team, t = lane_w / team;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int64_t rounds = ((int64_t)ch.R + tpw - 1) / tpw;
    for (int64_t w = warp; w < rounds; w += n_warps) {
        const int64_t r64 = w * tpw + t;
        if (r64 < ch.R) write_phase(ch, (int32_t)r64, lane, team);
    }
}

#endif  // __CUDACC__

}  // namespace js
}  // namespace kc
