// kc_extra.cuh — confidences (exact Python round(x, 5)) and K3, the per-candidate logprob sum.
#pragma once

#include "kc_common.cuh"
#include "kc_vote.cuh"

namespace kc {

// CPython float.__round__(x, 5) for finite x >= 0 (Objects/floatobject.c double_round: dtoa mode 3, i.e. the
// EXACT binary value rounded half-even to 5 decimals, then strtod).  x = M * 2^-sh exactly; q = x*1e5 rounded
// half-even in 128-bit integer arithmetic; q / 1e5 in IEEE double is the double nearest to the decimal
// q*10^-5, which is what strtod returns.  Used by cu:982,1178,1187,1219.
__device__ __forceinline__ double py_round5(double x) {
    const uint64_t bits = (uint64_t)__double_as_longlong(x);
    const int biased = (int)((bits >> 52) & 0x7FF);
    uint64_t mant = bits & 0xFFFFFFFFFFFFFull;
    int exp2;  // x = mant * 2^exp2
    if (biased == 0) {
        exp2 = -1074;
    } else {
        mant |= 1ull << 52;
        exp2 = biased - 1075;
    }
    if (mant == 0) return x;
    if (exp2 >= 0) return x;  // integer-valued: nothing to round
    const int sh = -exp2;     // >= 1
    if (sh >= 128) return 0.0;
    const uint64_t lo = mant * 100000ull;  // low 64 bits of the 70-bit product
    const uint64_t hi = __umul64hi(mant, 100000ull);
    uint64_t q, rem_hi, rem_lo, half_hi, half_lo;
    if (sh >= 64) {
        const int s = sh - 64;  // 0..63
        q = s == 0 ? hi : (hi >> s);
        rem_hi = s == 0 ? 0 : (hi & ((1ull << s) - 1));
        rem_lo = lo;
        half_hi = s == 0 ? 0 : (1ull << (s - 1));
        half_lo = s == 0 ? (1ull << 63) : 0;
    } else {
        q = (hi << (64 - sh)) | (lo >> sh);  // sh in 1..63; hi < 2^6 so no bits are lost for sh >= 6,
                                             // and for sh < 6 the product fits 64 bits only if hi == 0 (x >= 2^46: not a confidence)
        rem_hi = 0;
        rem_lo = lo & ((1ull << sh) - 1);
        half_hi = 0;
        half_lo = 1ull << (sh - 1);
    }
    const bool gt = rem_hi > half_hi || (rem_hi == half_hi && rem_lo > half_lo);
    const bool eq = rem_hi == half_hi && rem_lo == half_lo;
    if (gt || (eq && (q & 1))) ++q;
    return __ddiv_rn((double)q, 100000.0);
}

// One thread per group: the confidence the reference attaches to the group's consensus value.
__global__ void __launch_bounds__(256) confidence_kernel(const uint32_t *__restrict__ meta, int64_t n_groups, bool numeric,
                                                         const double *__restrict__ pvf_in, double *__restrict__ conf) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < n_groups; g += stride) {
        const uint32_t m = __ldg(meta + g);
        const double pvf = pvf_in ? __ldg(pvf_in + g) : 1.0;
        const double support = (double)KC_META_SUPPORT(m), nn = (double)KC_META_NN(m), present = (double)KC_META_PRESENT(m);
        const uint32_t flags = KC_META_FLAGS(m);
        double c;
        if (flags & KC_FLAG_HAS_VALUE) {
            if (!numeric)
                c = py_round5(__dmul_rn(pvf, __ddiv_rn(support, present)));  // cu:973,982
            else if (flags & KC_FLAG_SINGLE)
                c = __dmul_rn(__dmul_rn(pvf, __ddiv_rn(1.0, present)), 1.0);  // cu:1444,1086 (unrounded)
            else
                c = py_round5(__ddiv_rn(support, nn));  // cu:1177-1178,1186-1187,1218-1219
        } else if (flags & KC_FLAG_NO_FINITE) {
            c = __dmul_rn(pvf, __ddiv_rn(nn, present));  // cu:1444,1116
        } else {
            c = present == 0.0 ? pvf : 0.0;  // cu:1396 / cu:1402
        }
        conf[g] = c;
    }
}

// K3: one warp per sequence.  Lane l adds elements l, l+32, ... (coalesced 128-byte warp loads), then a
// xor butterfly 16,8,4,2,1 — the fixed order include/kllms_b200.h documents and oracle/consensus_oracle.c restates.
__global__ void __launch_bounds__(256) logprob_sum_kernel(const float *__restrict__ lp, const int64_t *__restrict__ offsets,
                                                          int64_t n_seq, float *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t s = warp; s < n_seq; s += n_warps) {
        const int64_t b = __ldg(offsets + s), e = __ldg(offsets + s + 1);
        float acc = 0.0f;
        for (int64_t i = b + lane; i < e; i += 32) acc = __fadd_rn(acc, __ldg(lp + i));
#pragma unroll
        for (int st = 16; st >= 1; st >>= 1) acc = __fadd_rn(acc, __shfl_xor_sync(0xFFFFFFFFu, acc, st));
        if (lane == 0) out[s] = acc;
    }
}

// K3, staged: sequences of a few dozen tokens leave a warp-per-sequence kernel with one or two elements per lane and
// ~25 instructions of bookkeeping per sequence (measured 0.36 of HBM peak on config 4).  Here a CTA copies the CONTIGUOUS
// token range of its T sequences into shared memory with 16-byte cp.async (coalesced, no register staging), then every
// thread sums ONE sequence in exactly the documented order: partial l = elements l, l+32, ... added left to right from
// +0.0f, then the tree the xor butterfly 16,8,4,2,1 forms (lane 0's view of it).  A tile whose tokens do not fit CAP
// floats (long sequences) falls back to the warp-per-sequence loop.
template <int T, int CAP>
__global__ void __launch_bounds__(T) logprob_sum_tile_kernel(const float *__restrict__ lp, const int64_t *__restrict__ offsets,
                                                             int64_t n_seq, float *__restrict__ out) {
    extern __shared__ __align__(16) float tok[];  // CAP + 4 floats
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t n_tiles = (n_seq + T - 1) / T;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t s0 = tile * T;
        const int cnt = (int)min((int64_t)T, n_seq - s0);
        // all four offset loads in flight together: the tile's range and this thread's sequence
        const int64_t t0 = __ldg(offsets + s0), t1 = __ldg(offsets + s0 + cnt);
        const int64_t my_b = __ldg(offsets + s0 + (tid < cnt ? tid : 0)), my_e = __ldg(offsets + s0 + (tid < cnt ? tid + 1 : 0));
        const int64_t t0a = t0 & ~int64_t(3);  // the copy starts at the 16-byte boundary at or below t0
        const int64_t span = t1 - t0a;
        if (span <= CAP) {
            const int n_vec = (int)(span >> 2);  // whole 16-byte pieces inside [t0a, t1)
            const uint32_t dst = smem_u32(tok);
            for (int v = tid; v < n_vec; v += T)
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + (uint32_t)v * 16u), "l"(lp + t0a + (int64_t)v * 4) : "memory");
            for (int i = (n_vec << 2) + tid; i < (int)span; i += T) tok[i] = __ldg(lp + t0a + i);  // < 4 stragglers
            asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
            __syncthreads();
            if (tid < cnt) {
                const int64_t b = my_b, e = my_e;
                const float *x = tok + (b - t0a);
                const int len = (int)(e - b);
                float p[32];
#pragma unroll
                for (int l = 0; l < 32; ++l) p[l] = 0.0f;
                for (int k = 0; k < len; k += 32) {
#pragma unroll
                    for (int l = 0; l < 32; ++l)
                        if (k + l < len) p[l] = __fadd_rn(p[l], x[k + l]);
                }
#pragma unroll
                for (int st = 16; st >= 1; st >>= 1) {
#pragma unroll
                    for (int l = 0; l < st; ++l) p[l] = __fadd_rn(p[l], p[l + st]);
                }
                out[s0 + tid] = p[0];
            }
            __syncthreads();  // the tile buffer is reused
        } else {
            for (int q = warp; q < cnt; q += T / 32) {
                const int64_t b = __ldg(offsets + s0 + q), e = __ldg(offsets + s0 + q + 1);
                float acc = 0.0f;
                for (int64_t i = b + lane; i < e; i += 32) acc = __fadd_rn(acc, __ldg(lp + i));
#pragma unroll
                for (int st = 16; st >= 1; st >>= 1) acc = __fadd_rn(acc, __shfl_xor_sync(0xFFFFFFFFu, acc, st));
                if (lane == 0) out[s0 + q] = acc;
            }
        }
    }
}

// ---------------------------------------------------------------- K3b: likelihood-weighted vote (self-defined spec)

// exp(x) for x <= 0, built only from single IEEE fp32 operations in a fixed order so that the C oracle
// (oracle/consensus_oracle.c: ko_exp_f32) reproduces it bit for bit: t = x*log2(e); k = floor(t + 0.5); f = t - k;
// 2^f by a degree-5 polynomial (Horner, separate multiply and add); scale by 2^k through the exponent field.
__device__ __forceinline__ float kexp(float x) {
    x = x < -87.0f ? -87.0f : x;
    const float t = __fmul_rn(x, 1.44269504f);
    const float k = floorf(__fadd_rn(t, 0.5f));
    const float f = __fadd_rn(t, -k);
    float p = 0.00133336f;
    p = __fadd_rn(__fmul_rn(p, f), 0.00961813f);
    p = __fadd_rn(__fmul_rn(p, f), 0.05550411f);
    p = __fadd_rn(__fmul_rn(p, f), 0.24022651f);
    p = __fadd_rn(__fmul_rn(p, f), 0.69314718f);
    p = __fadd_rn(__fmul_rn(p, f), 1.0f);
    return __fmul_rn(p, __int_as_float(((int)k + 127) << 23));
}

// One thread per group.  Candidate weight w_c = kexp(s_c - max_k s_k) with s = seq_logprob[record]; class weight =
// sum of its cells' weights in ascending candidate order (fp32); the heaviest class wins, ties -> first seen.
template <int NP>
__global__ void __launch_bounds__(128) weighted_vote_kernel(const int32_t *__restrict__ codes, const float *__restrict__ seq_lp,
                                                            int64_t n_groups, int n, FieldMap fm, bool has_nc,
                                                            int32_t *__restrict__ win, uint32_t *__restrict__ meta,
                                                            float *__restrict__ weight) {
    using M = typename MaskOf<NP>::type;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < n_groups; g += stride) {
        const int64_t rec = g / fm.n_fields;
        const uint32_t field = (uint32_t)(g - rec * fm.n_fields);
        const int32_t nc = has_nc ? __ldg(fm.none_code + field) : KC_CODE_NONE;
        int32_t x[NP];
        float w[NP];
        float smax = -3.0e38f;
#pragma unroll
        for (int i = 0; i < NP; ++i) {
            int32_t c = (i < n) ? __ldg(codes + g * n + i) : KC_CODE_ABSENT;
            const float s = (i < n) ? __ldg(seq_lp + rec * n + i) : -3.0e38f;
            w[i] = s;
            smax = (i < n && s > smax) ? s : smax;
            c = (c == KC_CODE_NONE) ? nc : c;           // None votes as none_code where it is >= 0
            x[i] = c < KC_CODE_NONE ? KC_CODE_NONE : c;  // absent cells never vote
        }
        M live = 0;
        int present = 0;
        float total = 0.0f;
#pragma unroll
        for (int i = 0; i < NP; ++i) {
            w[i] = kexp(__fadd_rn(w[i], -smax));
            const bool absent = (i >= n) || __ldg(codes + g * n + (i < n ? i : 0)) < KC_CODE_NONE;
            present += absent ? 0 : 1;
            if (x[i] >= 0) {
                live |= M(1) << i;
                total = __fadd_rn(total, w[i]);
            }
        }
        const int voters = popc_m(live);
        float best_w = -1.0f;
        int best_idx = 0, best_cnt = 0;
        int32_t best_code = KC_CODE_NONE;
        bool tie = false;
#pragma unroll
        for (int i = 0; i < NP; ++i) {
            if ((live >> i) & 1) {
                const int32_t c = x[i];
                M eq = 0;
                float cw = 0.0f;
#pragma unroll
                for (int j = i; j < NP; ++j) {
                    const bool e = x[j] == c;
                    eq |= e ? (M(1) << j) : M(0);
                    cw = e ? __fadd_rn(cw, w[j]) : cw;
                }
                if (cw > best_w) {
                    best_w = cw;
                    best_idx = i;
                    best_cnt = popc_m(eq);
                    best_code = c;
                    tie = false;
                } else if (cw == best_w) {
                    tie = true;
                }
                live &= ~eq;
            }
        }
        win[g] = best_code;
        meta[g] = pack_meta(best_idx, best_cnt, voters, present,
                            voters > 0 ? (KC_FLAG_HAS_VALUE | (tie ? KC_FLAG_TIE : 0u)) : 0u);
        weight[g] = voters > 0 ? __fdiv_rn(best_w, total) : 0.0f;
    }
}

// The weighted vote of ONE group by one thread: rawrow = the group's cells (code >= 0, KC_CODE_NONE, absent < KC_CODE_NONE), nc = the
// code None votes as (KC_CODE_NONE: it does not), w = the weights of the group's cells (shared memory).  best_w = the winning class's
// weight, total = the weight of the voting cells (both fp32 sums in cell order).
template <int NP>
__device__ __forceinline__ void weighted_walk(const int32_t (&rawrow)[NP], int32_t nc, const float *w, int32_t &out_code,
                                              uint32_t &out_meta, float &out_best_w, float &out_total) {
    using M = typename MaskOf<NP>::type;
    int32_t x[NP];
    M live = 0;
    int present = 0;
    float total = 0.0f, wmax = -1.0f;
    int32_t cmax = KC_CODE_NONE;  // the code of this group's heaviest VOTING cell (first of equals)
#pragma unroll
    for (int i = 0; i < NP; ++i) {
        const int32_t raw = rawrow[i];
        int32_t c = (raw == KC_CODE_NONE) ? nc : raw;  // None votes as none_code where it is >= 0
        c = c < KC_CODE_NONE ? KC_CODE_NONE : c;        // absent cells never vote
        x[i] = c;
        present += raw < KC_CODE_NONE ? 0 : 1;
        if (c >= 0) {
            live |= M(1) << i;
            const float wi = w[i];
            total = __fadd_rn(total, wi);
            if (wi > wmax) {
                wmax = wi;
                cmax = c;
            }
        }
    }
    const int voters = popc_m(live);
    float best_w = -1.0f;
    int best_idx = 0, best_cnt = 0;
    int32_t best_code = KC_CODE_NONE;
    bool tie = false;
    float consumed = 0.0f;
    // Order of the walk: always the class of the heaviest cell still waiting (the first one: this group's heaviest
    // voting cell).  The outcome does not depend on the order (the heaviest class wins, equal weights go to the class
    // seen first = smaller first index, `tie` says whether another class equals the winner), but the COST does: a warp
    // loops until its slowest lane is done.  The heaviest voter's class usually holds more than half of the weight and
    // ends the walk at once; where it does not, going by weight makes the remainder shrink fastest.  (Round 1 walked
    // in first-seen order after the record's heaviest candidate: 4.3 class passes per warp, and it parked every
    // group's codes in a shared-memory plane to fetch the next class's code by a data-dependent index; here the pass
    // over the cells finds the next class itself — no shared memory for the codes at all.)
    int32_t c = cmax;
    while (live) {
        // Every class still waiting sums a subset of the unconsumed weights, so its fp32 sum is at most
        // (total - consumed) up to rounding (< 32 * 2^-23 relative on each side); 5e-5 * total is a safe slack.
        // Below best_w it can neither win nor tie: stop.
        if (__fadd_rn(__fadd_rn(total, -consumed), __fmul_rn(total, 5e-5f)) < best_w) break;
        M eq = 0;
        float cw = 0.0f, nw = -1.0f;
        int32_t nc2 = KC_CODE_NONE;
#pragma unroll
        for (int j = 0; j < NP; ++j) {
            const bool e = x[j] == c;  // cells with this code that came earlier were consumed with their class
            const float wj = w[j];
            eq |= e ? (M(1) << j) : M(0);
            cw = e ? __fadd_rn(cw, wj) : cw;
            const bool waiting = !e && ((live >> j) & 1);
            if (waiting && wj > nw) {  // heaviest cell of the classes still waiting (first of equals)
                nw = wj;
                nc2 = x[j];
            }
        }
        const int i = ffs_mask(eq) - 1;  // the class's first cell
        if (cw > best_w) {
            best_w = cw;
            best_idx = i;
            best_cnt = popc_m(eq);
            best_code = c;
            tie = false;
        } else if (cw == best_w) {
            tie = true;
            if (i < best_idx) {  // an equally heavy class that was seen earlier
                best_idx = i;
                best_cnt = popc_m(eq);
                best_code = c;
            }
        }
        consumed = __fadd_rn(consumed, cw);
        live &= ~eq;
        c = nc2;
        if (c < 0) break;  // no waiting cell had a comparable weight (NaN logprobs: outside the spec); never spin
    }
    out_code = best_code;
    out_meta = pack_meta(best_idx, best_cnt, voters, present, voters > 0 ? (KC_FLAG_HAS_VALUE | (tie ? KC_FLAG_TIE : 0u)) : 0u);
    out_best_w = best_w;
    out_total = total;
}

template <int NP>
__device__ __forceinline__ void weighted_core(const int32_t (&rawrow)[NP], int32_t nc, const float *w, int32_t &out_code,
                                              uint32_t &out_meta, float &out_weight) {
    float best_w, total;
    weighted_walk<NP>(rawrow, nc, w, out_code, out_meta, best_w, total);
    out_weight = (KC_META_FLAGS(out_meta) & KC_FLAG_HAS_VALUE) ? __fdiv_rn(best_w, total) : 0.0f;
}

// K3b, weights once per record: the candidate weights depend on the record only, not on the field.  A CTA of T threads
// covers T consecutive groups (fields of a handful of records); its warps first compute w_c = kexp(s_c - max s) for
// those records into shared memory (lane = candidate, warp max by shuffles), then every thread votes its group with the
// weights read from there (same class sums, same order as weighted_vote_kernel).
template <int NP, int T>
__global__ void __launch_bounds__(T) weighted_vote_rec_kernel(const int32_t *__restrict__ codes, const float *__restrict__ seq_lp,
                                                              int64_t n_groups, int n, FieldMap fm, bool has_nc,
                                                              int32_t *__restrict__ win, uint32_t *__restrict__ meta,
                                                              float *__restrict__ weight) {
    using M = typename MaskOf<NP>::type;
    extern __shared__ float wts[];  // [records of the tile][NP]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t n_tiles = (n_groups + T - 1) / T;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t g0 = tile * T, g1 = min(g0 + T, n_groups);
        const int64_t r0 = g0 / fm.n_fields, r1 = (g1 - 1) / fm.n_fields;
        for (int64_t r = r0 + warp; r <= r1; r += T / 32) {
            float s_lo = (lane < n) ? __ldg(seq_lp + r * n + lane) : -3.0e38f;
            float s_hi = (NP > 32 && lane + 32 < n) ? __ldg(seq_lp + r * n + lane + 32) : -3.0e38f;
            float smax = fmaxf(s_lo, s_hi);
#pragma unroll
            for (int st = 16; st >= 1; st >>= 1) smax = fmaxf(smax, __shfl_xor_sync(0xFFFFFFFFu, smax, st));
            float *w = wts + (r - r0) * NP;
            if (lane < NP) w[lane] = kexp(__fadd_rn(s_lo, -smax));
            if (NP > 32) w[lane + 32] = kexp(__fadd_rn(s_hi, -smax));
        }
        __syncthreads();
        const int64_t g = g0 + tid;
        if (g < g1) {
            // record and field of this thread without a 64-bit division: offset inside the tile's first record
            const uint32_t fpos = (uint32_t)(g0 - r0 * fm.n_fields) + (uint32_t)tid;
            const uint32_t rec_local = fm.div_small(fpos);
            const uint32_t field = fpos - rec_local * fm.n_fields;
            const int32_t nc = has_nc ? __ldg(fm.none_code + field) : KC_CODE_NONE;
            const float *w = wts + rec_local * NP;
            // (requesting the row BEFORE the weights phase was tried: it keeps 32 more registers live across the barrier,
            // 67 -> 94, and the lost occupancy cost more than the overlap gained: 0.357 -> 0.379 ms)
            int32_t rawrow[NP];
            if (n == NP) load_row<NP, true>(codes, g, n, rawrow);
            else load_row<NP, false>(codes, g, n, rawrow);
            weighted_core<NP>(rawrow, nc, w, win[g], meta[g], weight[g]);
        }
        __syncthreads();
    }
}

// ---- K3b, TMA front-end: first pass per lane, undecided groups by the whole warp

// What a lane knows about its group after ONE pass over the cells: the mapped codes, the total weight of the voting cells and the
// class of the record's heaviest candidate (the guess), summed in index order exactly as a walk pass would.
template <int N>
struct WvFirst {
    using M = typename MaskOf<N>::type;
    int32_t x[N];
    M eq_g;
    float total, cw_g;
    int32_t guess;
    int voters, present;
    bool decided;  // the guess's class holds a strict majority of the weight: it is the unique winner
};

template <int N>
__device__ __forceinline__ void wv_first_pass(const int32_t (&raw)[N], int32_t lo, int32_t nc, const float *w, int32_t graw, WvFirst<N> &f) {
    using M = typename MaskOf<N>::type;
    f.eq_g = 0;
    f.total = 0.0f;
    f.cw_g = 0.0f;
    if (lo >= 0) {
        // every cell votes with its own code (no None, no absent cell — the common row): 2-3 ALU instructions per cell
        f.guess = graw < 0 ? KC_CODE_NONE : graw;
        f.voters = f.present = N;
#pragma unroll
        for (int i = 0; i < N; ++i) {
            const float wi = w[i];
            const bool e = raw[i] == f.guess;
            f.x[i] = raw[i];
            f.total = __fadd_rn(f.total, wi);
            if (e) {
                f.eq_g |= M(1) << i;
                f.cw_g = __fadd_rn(f.cw_g, wi);
            }
        }
    } else {
        int32_t guess = (graw == KC_CODE_NONE) ? nc : graw;
        f.guess = guess < KC_CODE_NONE ? KC_CODE_NONE : guess;  // the heaviest candidate does not vote here: no guess
        M live = 0;
        int present = 0;
#pragma unroll
        for (int i = 0; i < N; ++i) {
            const int32_t r = raw[i];
            int32_t c = (r == KC_CODE_NONE) ? nc : r;  // None votes as none_code where it is >= 0
            c = c < KC_CODE_NONE ? KC_CODE_NONE : c;    // absent cells never vote
            f.x[i] = c;
            present += r < KC_CODE_NONE ? 0 : 1;
            if (c >= 0) {
                live |= M(1) << i;
                const float wi = w[i];
                f.total = __fadd_rn(f.total, wi);
                if (c == f.guess) {
                    f.eq_g |= M(1) << i;
                    f.cw_g = __fadd_rn(f.cw_g, wi);
                }
            }
        }
        f.voters = popc_m(live);
        f.present = present;
    }
    // every other class sums a subset of the remaining weights: at most (total - cw_g) up to rounding (< 64 * 2^-23 relative on
    // each side; 5e-5 * total is a safe slack).  Strictly below cw_g it can neither win nor tie.
    f.decided = f.guess >= 0 && f.cw_g > __fadd_rn(__fadd_rn(f.total, -f.cw_g), __fmul_rn(f.total, 5e-5f));
}

// The general walk (see weighted_core) for ONE group by the WHOLE warp: lane j holds cells j and j + 32 of the owner's group.  A
// thread-per-group walk makes the warp wait for its slowest lane — a few percent of the groups are undecided after the first
// pass, but most warps hold one — and spends 32 lanes on one lane's work; here an undecided group costs ~150 warp instructions.
// Same visiting order (the class of the heaviest cell still waiting, first of equals), same class sums (index order, one
// rounding per addition), same tie rules: the result is bit-identical.  All arguments except `owner` are the OWNER's values.
template <int N>
__device__ __forceinline__ void wv_warp_walk(uint32_t lane, uint32_t owner, const WvFirst<N> &f, const float *wts, uint32_t rec_local, int WROW,
                                             int32_t &out_code, uint32_t &out_meta, float &out_weight) {
    constexpr uint32_t FULL = 0xFFFFFFFFu;
    // the owner's cells, one (two) per lane
    int32_t c_lo = KC_CODE_NONE, c_hi = KC_CODE_NONE;
#pragma unroll
    for (int j = 0; j < N; ++j) {
        const int32_t v = __shfl_sync(FULL, f.x[j], owner);
        if (lane == (uint32_t)(j & 31)) {
            if (j < 32) c_lo = v;
            else c_hi = v;
        }
    }
    const float *w = wts + __shfl_sync(FULL, rec_local, owner) * WROW;
    const float w_lo = w[lane], w_hi = N > 32 ? w[lane + 32] : 0.0f;
    const float total = __shfl_sync(FULL, f.total, owner);
    const int32_t guess = __shfl_sync(FULL, f.guess, owner);
    const float cw_g = __shfl_sync(FULL, f.cw_g, owner);
    uint32_t live_lo = __ballot_sync(FULL, c_lo >= 0), live_hi = N > 32 ? __ballot_sync(FULL, c_hi >= 0) : 0u;
    float best_w = -1.0f, consumed = 0.0f;
    int best_idx = 0, best_cnt = 0;
    int32_t best_code = KC_CODE_NONE;
    bool tie = false;
    if (guess >= 0) {  // the first pass summed the guess's class: it is the best so far
        const uint32_t g_lo = __ballot_sync(FULL, c_lo == guess), g_hi = N > 32 ? __ballot_sync(FULL, c_hi == guess) : 0u;
        best_w = cw_g;
        best_idx = g_lo ? __ffs((int)g_lo) - 1 : 31 + __ffs((int)g_hi);
        best_cnt = __popc(g_lo) + __popc(g_hi);
        best_code = guess;
        consumed = cw_g;
        live_lo &= ~g_lo;
        live_hi &= ~g_hi;
    }
    while (live_lo | live_hi) {
        if (__fadd_rn(__fadd_rn(total, -consumed), __fmul_rn(total, 5e-5f)) < best_w) break;  // the rest can neither win nor tie
        // the heaviest cell still waiting, first of equals
        float mx = fmaxf(((live_lo >> lane) & 1u) ? w_lo : -1.0f, (N > 32 && ((live_hi >> lane) & 1u)) ? w_hi : -1.0f);
#pragma unroll
        for (int st = 16; st >= 1; st >>= 1) mx = fmaxf(mx, __shfl_xor_sync(FULL, mx, st));
        const uint32_t a_lo = __ballot_sync(FULL, ((live_lo >> lane) & 1u) && w_lo == mx);
        const uint32_t a_hi = N > 32 ? __ballot_sync(FULL, ((live_hi >> lane) & 1u) && w_hi == mx) : 0u;
        if (!(a_lo | a_hi)) break;  // only NaN weights are left (NaN logprobs: outside the spec); never spin
        const int32_t c = a_lo ? __shfl_sync(FULL, c_lo, __ffs((int)a_lo) - 1) : __shfl_sync(FULL, c_hi, __ffs((int)a_hi) - 1);
        const uint32_t e_lo = __ballot_sync(FULL, c_lo == c), e_hi = N > 32 ? __ballot_sync(FULL, c_hi == c) : 0u;
        float cw = 0.0f;  // the class's weights in index order
        for (uint32_t m = e_lo; m; m &= m - 1) cw = __fadd_rn(cw, __shfl_sync(FULL, w_lo, __ffs((int)m) - 1));
        if (N > 32)
            for (uint32_t m = e_hi; m; m &= m - 1) cw = __fadd_rn(cw, __shfl_sync(FULL, w_hi, __ffs((int)m) - 1));
        const int i = e_lo ? __ffs((int)e_lo) - 1 : 31 + __ffs((int)e_hi);
        const int cnt = __popc(e_lo) + __popc(e_hi);
        if (cw > best_w) {
            best_w = cw;
            best_idx = i;
            best_cnt = cnt;
            best_code = c;
            tie = false;
        } else if (cw == best_w) {
            tie = true;
            if (i < best_idx) {  // an equally heavy class that was seen earlier
                best_idx = i;
                best_cnt = cnt;
                best_code = c;
            }
        }
        consumed = __fadd_rn(consumed, cw);
        live_lo &= ~e_lo;
        live_hi &= ~e_hi;
    }
    if (lane == owner) {
        out_code = best_code;
        out_meta = pack_meta(best_idx, best_cnt, f.voters, f.present, f.voters > 0 ? (KC_FLAG_HAS_VALUE | (tie ? KC_FLAG_TIE : 0u)) : 0u);
        out_weight = f.voters > 0 ? __fdiv_rn(best_w, total) : 0.0f;
    }
}

// K3b with K1's TMA front-end (n in {32, 64} cells per group = 128 / 256 byte rows): every WARP runs its own pipeline of STAGES
// tiles of 32 consecutive groups (one cp.async.bulk.tensor.2d per tile, hardware swizzle, the warp's own mbarrier, conflict-free
// LDS.128; see vote_tma_kernel) instead of one 128-byte row per thread straight from global memory (latency-bound at 0.39 of the
// HBM peak: a warp's 32 rows are 32 separate lines per load instruction).  The weights of the tile's records (32 groups span
// 32 / n_fields + 2 records at most) are computed by the warp itself into its own shared-memory rows (lane = candidate, warp
// max by shuffles), padded by one float so that lanes of different records read different banks; the pad slot carries the index of
// the record's heaviest candidate, whose class weighted_core sums in its first pass (one pass decides most groups).  No block-wide
// barrier.
template <int N, int WARPS, int STAGES, int MIN_CTAS, bool PREFETCH>
__global__ void __launch_bounds__(WARPS * 32, MIN_CTAS) weighted_vote_tma_kernel(const __grid_constant__ CUtensorMap tmap, const float *__restrict__ seq_lp,
                                                                       uint32_t n_groups, FieldMap fm, bool has_nc, int rec_cap, uint64_t inv_fields,
                                                                       int32_t *__restrict__ win, uint32_t *__restrict__ meta,
                                                                       float *__restrict__ weight) {
    constexpr int ROW_BYTES = N * 4;
    constexpr int BOX_ROWS_PER_GROUP = ROW_BYTES > 128 ? ROW_BYTES / 128 : 1;
    constexpr uint32_t TILE_BYTES = 32 * ROW_BYTES;
    constexpr int WROW = N + 1;
    // x / n_fields for any 32-bit x without a division: inv_fields = floor(2^64 / n_fields) + 1 (exact for n_fields >= 2)
    auto record_of = [&](uint32_t x) -> uint32_t { return fm.n_fields == 1u ? x : (uint32_t)__umul64hi((uint64_t)x, inv_fields); };
    static_assert(TILE_BYTES % 1024 == 0, "warp tile must keep the swizzle atom alignment");
    static_assert((STAGES & (STAGES - 1)) == 0, "STAGES must be a power of two");
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t full_bar[WARPS * STAGES];

    const uint32_t lane = threadIdx.x & 31;
    const uint32_t warp = __shfl_sync(0xFFFFFFFFu, threadIdx.x >> 5, 0);
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t my_smem = smem_base + warp * (STAGES * TILE_BYTES);
    const uint32_t my_bar = smem_u32(full_bar) + warp * (STAGES * 8);
    // the weight rows live behind the tiles of all warps
    float *wts = reinterpret_cast<float *>(smem_raw + (smem_base - smem_u32(smem_raw)) + (size_t)WARPS * STAGES * TILE_BYTES) +
                 (size_t)warp * rec_cap * WROW;

    const uint32_t n_tiles = (n_groups + 31u) >> 5;
    const uint32_t first = blockIdx.x * WARPS + warp;
    const uint32_t step = gridDim.x * WARPS;
    uint64_t policy = 0;
    if (lane == 0) {
        tma_prefetch_desc(&tmap);
#pragma unroll
        for (int s = 0; s < STAGES; ++s) mbar_init_a(my_bar + s * 8, 1);
        fence_barrier_init();
        policy = policy_evict_first();
#pragma unroll
        for (int s = 0; s < STAGES; ++s) {
            const uint32_t t = first + (uint32_t)s * step;
            if (t < n_tiles) {
                mbar_arrive_expect_tx_a(my_bar + s * 8, TILE_BYTES);
                tma_load_2d_a(my_smem + s * TILE_BYTES, &tmap, 0, (int32_t)(t * 32 * BOX_ROWS_PER_GROUP), my_bar + s * 8, policy, 0);
            }
        }
    }
    __syncwarp();
    uint32_t piece[N / 4];
#pragma unroll
    for (int q = 0; q < N / 4; ++q) piece[q] = Swizzle<ROW_BYTES>::apply(lane * ROW_BYTES + q * 16);

    // The sequence logprobs of a tile's records are requested one tile AHEAD (a warp works through its tiles one after the other:
    // a global-memory round trip per tile in front of the weights would be exposed every time).  Up to PF records per tile are
    // prefetched (32 groups span 31 / n_fields + 2 records); wider tiles load them on the spot.
    constexpr int PF = 4;
    const bool prefetch = PREFETCH && rec_cap <= PF;
    float cur_lo[PF], cur_hi[PF], nxt_lo[PF], nxt_hi[PF];
    auto fetch = [&](uint32_t tt, float (&lo)[PF], float (&hi)[PF]) {
        const uint32_t a = tt * 32, b = min(a + 31u, n_groups - 1u);
        const uint32_t ra = record_of(a), rb = record_of(b);
#pragma unroll
        for (int k = 0; k < PF; ++k) {
            lo[k] = hi[k] = -3.0e38f;
            if (ra + k <= rb) {
                const float *s = seq_lp + (size_t)(ra + k) * N;
                lo[k] = __ldg(s + lane);
                if (N > 32) hi[k] = __ldg(s + lane + 32);
            }
        }
    };
    if (prefetch && first < n_tiles) fetch(first, cur_lo, cur_hi);

    uint32_t it = 0;
    for (uint32_t t = first; t < n_tiles; t += step, ++it) {
        const uint32_t stage = it & (STAGES - 1);
        const uint32_t parity = (it / STAGES) & 1;
        const uint32_t bar = my_bar + stage * 8;
        const uint32_t tile = my_smem + stage * TILE_BYTES;
        if (prefetch && t + step < n_tiles) fetch(t + step, nxt_lo, nxt_hi);
        // the weights of this tile's records, while the tile is still on its way
        const uint32_t g0 = t * 32, g_last = min(g0 + 31u, n_groups - 1u);
        const uint32_t r0 = record_of(g0), r_last = record_of(g_last);
        for (uint32_t r = r0; r <= r_last; ++r) {
            const float *s = seq_lp + (size_t)r * N;
            float s_lo, s_hi = -3.0e38f;
            if (prefetch) {
                const uint32_t k = r - r0;  // < PF
                s_lo = k == 0 ? cur_lo[0] : k == 1 ? cur_lo[1] : k == 2 ? cur_lo[2] : cur_lo[3];
                if (N > 32) s_hi = k == 0 ? cur_hi[0] : k == 1 ? cur_hi[1] : k == 2 ? cur_hi[2] : cur_hi[3];
            } else {
                s_lo = __ldg(s + lane);
                if (N > 32) s_hi = __ldg(s + lane + 32);
            }
            float smax = fmaxf(s_lo, s_hi);
#pragma unroll
            for (int st = 16; st >= 1; st >>= 1) smax = fmaxf(smax, __shfl_xor_sync(0xFFFFFFFFu, smax, st));
            float *w = wts + (r - r0) * WROW;
            w[lane] = kexp(__fadd_rn(s_lo, -smax));
            if (N > 32) w[lane + 32] = kexp(__fadd_rn(s_hi, -smax));
            // the record's heaviest candidate (first of the largest sums; N = none, e.g. all NaN) rides in the row's pad slot
            const uint32_t b_lo = __ballot_sync(0xFFFFFFFFu, s_lo == smax), b_hi = __ballot_sync(0xFFFFFFFFu, N > 32 && s_hi == smax);
            const int imax = b_lo ? __ffs((int)b_lo) - 1 : (b_hi ? 31 + __ffs((int)b_hi) : N);
            if (lane == 0) w[N] = __int_as_float(imax);
        }
        __syncwarp();
        mbar_wait_a(bar, parity);
        int32_t raw[N];
#pragma unroll
        for (int q = 0; q < N / 4; ++q) {
            const int4 v4 = lds_v4(tile + piece[q]);
            raw[4 * q + 0] = v4.x;
            raw[4 * q + 1] = v4.y;
            raw[4 * q + 2] = v4.z;
            raw[4 * q + 3] = v4.w;
        }
        const uint32_t g = g0 + lane;
        const uint32_t fpos = (g0 - r0 * fm.n_fields) + lane;  // offset inside the tile's first record: < n_fields + 32
        const uint32_t rec_local = g < n_groups ? fm.div_small(fpos) : 0u;
        const float *wrow = wts + rec_local * WROW;
        // this group's cell of its record's heaviest candidate: read from the tile while the stage is still ours
        const int imax = __float_as_int(wrow[N]);
        int32_t graw = KC_CODE_NONE - 1;
        if (imax < N) {
            asm volatile("ld.shared.s32 %0, [%1];" : "=r"(graw) : "r"(tile + Swizzle<ROW_BYTES>::apply(lane * ROW_BYTES + (uint32_t)imax * 4u)));
        }
        // hand the stage back to the TMA unit only after every lane's row is in registers (see vote_tma_kernel)
        const int32_t lo = min(row_min<N>(raw), graw);
        const uint32_t order = __shfl_sync(0xFFFFFFFFu, (uint32_t)lo, 0) ^ (uint32_t)lo;
        const uint32_t tn = t + STAGES * step;
        if (lane == 0 && tn < n_tiles) {
            mbar_arrive_expect_tx_a(bar, TILE_BYTES);
            tma_load_2d_a(tile, &tmap, 0, (int32_t)(tn * 32 * BOX_ROWS_PER_GROUP + order), bar, policy, 0);
        }
        WvFirst<N> f;
        bool undecided = false;
        int32_t o_code = KC_CODE_NONE;
        uint32_t o_meta = 0;
        float o_weight = 0.0f;
        if (g < n_groups) {
            const uint32_t field = fpos - rec_local * fm.n_fields;
            const int32_t nc = has_nc ? __ldg(fm.none_code + field) : KC_CODE_NONE;
            wv_first_pass<N>(raw, lo, nc, wrow, graw, f);
            undecided = !f.decided;
            if (f.decided) {
                o_code = f.guess;
                o_meta = pack_meta(ffs_mask(f.eq_g) - 1, popc_m(f.eq_g), f.voters, f.present, KC_FLAG_HAS_VALUE);
                o_weight = __fdiv_rn(f.cw_g, f.total);
            }
        }
        for (uint32_t todo = __ballot_sync(0xFFFFFFFFu, undecided); todo; todo &= todo - 1)
            wv_warp_walk<N>(lane, (uint32_t)__ffs((int)todo) - 1u, f, wts, rec_local, WROW, o_code, o_meta, o_weight);
        if (g < n_groups) {
            win[g] = o_code;
            meta[g] = o_meta;
            weight[g] = o_weight;
        }
        __syncwarp();  // the next tile's weights overwrite these rows
        if (prefetch) {
#pragma unroll
            for (int k = 0; k < PF; ++k) {
                cur_lo[k] = nxt_lo[k];
                cur_hi[k] = nxt_hi[k];
            }
        }
    }
}

// ---- K3b with the weights OUT of the tile loop.  A pre-pass writes, once per record, the row [w_0 .. w_{N-1}, index of the heaviest
// candidate, 3 pad words] (N + 4 floats: rows stay 16-byte multiples and consecutive rows start 4 banks apart); the vote kernel
// fetches the rows of a tile's records with ONE cp.async.bulk next to the tile's tensor copy, completing on the same mbarrier.
//
// The same pre-pass gives the plain weight rows of kc_candidate_weights_f32: any n <= 64, row stride wrow = n (no pad words; with
// wrow >= n + 4 the four pad words above follow the weights).  One warp per record, lane = candidate (and candidate + 32).

__global__ void __launch_bounds__(256) weight_rows_kernel(const float *__restrict__ seq_lp, int64_t n_records, int n, int wrow,
                                                          float *__restrict__ rows) {
    const uint32_t lane = threadIdx.x & 31;
    const bool lo_in = (int)lane < n, hi_in = (int)lane + 32 < n;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = warp; r < n_records; r += n_warps) {
        const float *s = seq_lp + r * n;
        const float s_lo = lo_in ? __ldg(s + lane) : -3.0e38f, s_hi = hi_in ? __ldg(s + lane + 32) : -3.0e38f;
        float smax = fmaxf(s_lo, s_hi);
#pragma unroll
        for (int st = 16; st >= 1; st >>= 1) smax = fmaxf(smax, __shfl_xor_sync(0xFFFFFFFFu, smax, st));
        float *w = rows + r * wrow;
        if (lo_in) w[lane] = kexp(__fadd_rn(s_lo, -smax));
        if (hi_in) w[lane + 32] = kexp(__fadd_rn(s_hi, -smax));
        if (wrow >= n + 4) {
            const uint32_t b_lo = __ballot_sync(0xFFFFFFFFu, lo_in && s_lo == smax), b_hi = __ballot_sync(0xFFFFFFFFu, hi_in && s_hi == smax);
            const int imax = b_lo ? __ffs((int)b_lo) - 1 : (b_hi ? 31 + __ffs((int)b_hi) : n);
            if (lane < 4) w[n + lane] = lane == 0 ? __int_as_float(imax) : 0.0f;
        }
    }
}

// Likelihood-weighted vote over IRREGULAR groups (self-defined, DESIGN.md §5): group g belongs to record rec[g] and holds n cells
// (K1's coding; CellT = int8 for the device JSON path's cell matrix, int32 for the planner's); cell i carries the weight of
// candidate cand[g][i] (cand == NULL: candidate i) of its record.  The vote itself is K3b's (weighted_walk: class sums in cell
// order, heaviest class, ties to the class seen first).  Out: K1's result word and (W_win, W_present), W_present = the fp32 sum of
// the weights of the present cells (None cells included) in cell order.  One thread per group; its cells' weights sit in a
// private shared-memory row (stride NP + 1: the rows of a warp's lanes start in different banks) for the walk to read.
template <int NP, typename CellT>
__global__ void __launch_bounds__(128) weighted_vote_groups_kernel(const CellT *__restrict__ cells, int64_t n_groups, int n,
                                                                   const int32_t *__restrict__ rec, const int8_t *__restrict__ cand,
                                                                   const float *__restrict__ weight, uint32_t *__restrict__ meta,
                                                                   float2 *__restrict__ sums) {
    __shared__ float wsh[128 * (NP + 1)];
    float *w = wsh + threadIdx.x * (NP + 1);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < n_groups; g += stride) {
        const float *wr = weight + (int64_t)__ldg(rec + g) * n;
        int32_t raw[NP];
        float w_present = 0.0f;
#pragma unroll
        for (int i = 0; i < NP; ++i) {
            const int32_t c = i < n ? (int32_t)__ldg(cells + g * n + i) : KC_CODE_ABSENT;
            raw[i] = c;
            float wi = 0.0f;
            if (c >= KC_CODE_NONE) {
                const int k = cand ? (int)__ldg(cand + g * n + i) : i;
                wi = __ldg(wr + k);
                w_present = __fadd_rn(w_present, wi);
            }
            w[i] = wi;
        }
        int32_t code;
        uint32_t m;
        float best_w, total;
        weighted_walk<NP>(raw, KC_CODE_NONE, w, code, m, best_w, total);
        meta[g] = m;
        sums[g] = make_float2((KC_META_FLAGS(m) & KC_FLAG_HAS_VALUE) ? best_w : 0.0f, w_present);
    }
}

__device__ __forceinline__ void bulk_load_1d_a(uint32_t smem_dst, const void *src, uint32_t bytes, uint32_t bar, uint32_t dep) {
    asm volatile(
        "{\n\t"
        ".reg .b32 kc_dep1;\n\t"
        "mov.b32 kc_dep1, %4;\n\t"
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n\t"
        "}\n" ::"r"(smem_dst),
        "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(bar), "r"(dep)
        : "memory");
}

template <int N, int WARPS, int STAGES, int MIN_CTAS>
__global__ void __launch_bounds__(WARPS * 32, MIN_CTAS) weighted_vote_rows_kernel(const __grid_constant__ CUtensorMap tmap, const float *__restrict__ wrows,
                                                                        uint32_t n_groups, FieldMap fm, bool has_nc, int rec_cap, uint64_t inv_fields,
                                                                        int32_t *__restrict__ win, uint32_t *__restrict__ meta,
                                                                        float *__restrict__ weight) {
    constexpr int ROW_BYTES = N * 4;
    constexpr int BOX_ROWS_PER_GROUP = ROW_BYTES > 128 ? ROW_BYTES / 128 : 1;
    constexpr uint32_t TILE_BYTES = 32 * ROW_BYTES;
    constexpr int WROW = N + 4;
    constexpr int WSLOTS = STAGES + 1;  // the slot of the tile being voted is not the one the re-arm refills
    auto record_of = [&](uint32_t x) -> uint32_t { return fm.n_fields == 1u ? x : (uint32_t)__umul64hi((uint64_t)x, inv_fields); };
    static_assert(TILE_BYTES % 1024 == 0, "warp tile must keep the swizzle atom alignment");
    static_assert((STAGES & (STAGES - 1)) == 0, "STAGES must be a power of two");
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t full_bar[WARPS * STAGES];

    const uint32_t lane = threadIdx.x & 31;
    const uint32_t warp = __shfl_sync(0xFFFFFFFFu, threadIdx.x >> 5, 0);
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t my_smem = smem_base + warp * (STAGES * TILE_BYTES);
    const uint32_t my_bar = smem_u32(full_bar) + warp * (STAGES * 8);
    const uint32_t slot_bytes = (uint32_t)rec_cap * WROW * 4;
    const uint32_t my_rows = smem_base + WARPS * STAGES * TILE_BYTES + warp * (WSLOTS * slot_bytes);     // shared-space address
    const float *my_rows_p = reinterpret_cast<const float *>(smem_raw + (my_rows - smem_u32(smem_raw)));  // the same, generic

    const uint32_t n_tiles = (n_groups + 31u) >> 5;
    const uint32_t first = blockIdx.x * WARPS + warp;
    const uint32_t step = gridDim.x * WARPS;
    uint64_t policy = 0;
    // one tile's copies: the 32 rows of cells and the weight rows of the records they belong to, on one barrier
    auto request = [&](uint32_t t, uint32_t stage, uint32_t slot, uint32_t dep) {
        const uint32_t a = t * 32, b = min(a + 31u, n_groups - 1u);
        const uint32_t ra = record_of(a), rb = record_of(b);
        const uint32_t wbytes = (rb - ra + 1u) * WROW * 4;
        const uint32_t bar = my_bar + stage * 8;
        mbar_arrive_expect_tx_a(bar, TILE_BYTES + wbytes);
        tma_load_2d_a(my_smem + stage * TILE_BYTES, &tmap, 0, (int32_t)(t * 32 * BOX_ROWS_PER_GROUP + dep), bar, policy, 0);
        bulk_load_1d_a(my_rows + slot * slot_bytes, wrows + (size_t)ra * WROW, wbytes, bar, dep);
    };
    if (lane == 0) {
        tma_prefetch_desc(&tmap);
#pragma unroll
        for (int s = 0; s < STAGES; ++s) mbar_init_a(my_bar + s * 8, 1);
        fence_barrier_init();
        policy = policy_evict_first();
#pragma unroll
        for (int s = 0; s < STAGES; ++s) {
            const uint32_t t = first + (uint32_t)s * step;
            if (t < n_tiles) request(t, (uint32_t)s, (uint32_t)s, 0u);
        }
    }
    __syncwarp();
    uint32_t piece[N / 4];
#pragma unroll
    for (int q = 0; q < N / 4; ++q) piece[q] = Swizzle<ROW_BYTES>::apply(lane * ROW_BYTES + q * 16);

    uint32_t it = 0, slot = 0;  // slot = it % WSLOTS
    for (uint32_t t = first; t < n_tiles; t += step, ++it) {
        const uint32_t stage = it & (STAGES - 1);
        const uint32_t parity = (it / STAGES) & 1;
        const uint32_t bar = my_bar + stage * 8;
        const uint32_t tile = my_smem + stage * TILE_BYTES;
        const uint32_t g0 = t * 32, g = g0 + lane;
        const uint32_t r0 = record_of(g0);
        const uint32_t fpos = (g0 - r0 * fm.n_fields) + lane;  // offset inside the tile's first record: < n_fields + 32
        const uint32_t rec_local = g < n_groups ? fm.div_small(fpos) : 0u;
        const float *wts = my_rows_p + slot * (slot_bytes / 4);
        const float *wrow = wts + rec_local * WROW;
        mbar_wait_a(bar, parity);
        int32_t raw[N];
#pragma unroll
        for (int q = 0; q < N / 4; ++q) {
            const int4 v4 = lds_v4(tile + piece[q]);
            raw[4 * q + 0] = v4.x;
            raw[4 * q + 1] = v4.y;
            raw[4 * q + 2] = v4.z;
            raw[4 * q + 3] = v4.w;
        }
        // this group's cell of its record's heaviest candidate: read from the tile while the stage is still ours
        const int imax = __float_as_int(wrow[N]);
        int32_t graw = KC_CODE_NONE - 1;
        if (imax < N) {
            asm volatile("ld.shared.s32 %0, [%1];" : "=r"(graw) : "r"(tile + Swizzle<ROW_BYTES>::apply(lane * ROW_BYTES + (uint32_t)imax * 4u)));
        }
        // hand the stage back only after every lane's row is in registers (see vote_tma_kernel); the shuffle also means that
        // every lane has left the previous tile, whose weight slot the request below refills
        const int32_t lo = min(row_min<N>(raw), graw);
        const uint32_t order = __shfl_sync(0xFFFFFFFFu, (uint32_t)lo, 0) ^ (uint32_t)lo;
        const uint32_t tn = t + STAGES * step;
        if (lane == 0 && tn < n_tiles) request(tn, stage, (slot + STAGES) % WSLOTS, order);
        WvFirst<N> f;
        bool undecided = false;
        int32_t o_code = KC_CODE_NONE;
        uint32_t o_meta = 0;
        float o_weight = 0.0f;
        if (g < n_groups) {
            const uint32_t field = fpos - rec_local * fm.n_fields;
            const int32_t nc = has_nc ? __ldg(fm.none_code + field) : KC_CODE_NONE;
            wv_first_pass<N>(raw, lo, nc, wrow, graw, f);
            undecided = !f.decided;
            if (f.decided) {
                o_code = f.guess;
                o_meta = pack_meta(ffs_mask(f.eq_g) - 1, popc_m(f.eq_g), f.voters, f.present, KC_FLAG_HAS_VALUE);
                o_weight = __fdiv_rn(f.cw_g, f.total);
            }
        }
        for (uint32_t todo = __ballot_sync(0xFFFFFFFFu, undecided); todo; todo &= todo - 1)
            wv_warp_walk<N>(lane, (uint32_t)__ffs((int)todo) - 1u, f, wts, rec_local, WROW, o_code, o_meta, o_weight);
        if (g < n_groups) {
            win[g] = o_code;
            meta[g] = o_meta;
            weight[g] = o_weight;
        }
        slot = slot + 1 == WSLOTS ? 0u : slot + 1;
    }
}

}  // namespace kc
