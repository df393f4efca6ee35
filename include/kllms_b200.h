/*
 * kllms_b200.h — C ABI of the B200-native n-way consensus consolidator.
 *
 * The reference (retab-dev/k-LLMs) is pure Python and has NO plugin / FFI boundary; its seam is
 * the import at k_llms/utils/consolidation.py:11-19 (`consensus_values`, `ConsensusSettings`, ...).
 * This header therefore declares the columnar entry points a binding for that seam calls
 * (SURVEY.md §8b "what a C-ABI replacement must export"); each cites the reference code it replaces.
 * INTEGRATION.md shows the ctypes stub a k_llms maintainer would add.
 *
 * Conventions: plain pointers and sizes, no torch types; 0 on success, negative KC_E* on failure,
 * never an exception; caller owns every buffer; `d_` pointers are device memory on the CURRENT
 * CUDA device, `h_` pointers host memory; calls are stream-ordered on `stream` (a cudaStream_t
 * passed as void*, NULL = legacy default stream) and re-entrant.
 *
 * DATA MODEL — a "group" is the n candidate values of ONE field of ONE record (what one call of
 * the reference's consensus_values() sees for a scalar field).  Groups are stored row-major,
 * candidate index innermost: cells[g*n + c], g = record*n_fields + field.
 */
#ifndef KLLMS_B200_H
#define KLLMS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KC_VERSION 200 /* 0.2.0 */
#define KC_MAX_CANDIDATES 64

/* ---- error codes ---- */
#define KC_OK 0
#define KC_EINVAL (-1)  /* bad argument (n out of [1,64], NULL pointer, misaligned buffer, negative eps) */
#define KC_ECUDA (-2)   /* CUDA runtime error; text via kc_last_error() */
#define KC_ENODEV (-3)  /* no sm_100 device */
#define KC_ENOMEM (-4)

/* ---- vote cells (int32) ---- */
#define KC_CODE_NONE (-1)   /* candidate present, value is None (cu:947,964) */
#define KC_CODE_ABSENT (-2) /* candidate is not part of `values` at this node (parent was not a dict/list, cu:1416,1431) */
/* codes >= 0: dictionary code of the processed value (sanitize_value(v) for strings, cu:925-933;
 * `v or False` for bool groups, cu:956); equal code <=> equal processed value. */

/* ---- numeric cells (float64) ---- */
#define KC_F64_NONE_BITS 0x7FF8C0DE00000000ULL   /* quiet NaN whose HIGH 32 bits are 0x7FF8C0DE: None */
#define KC_F64_ABSENT_BITS 0x7FF8C0DF00000000ULL /* quiet NaN whose HIGH 32 bits are 0x7FF8C0DF: absent (see KC_CODE_ABSENT) */
/* Only the high word is examined (the low word is ignored), so a cell is tagged by one 32-bit compare.
 * any OTHER non-finite value means "present, non-None, but not a finite number" (bool, str, nan,
 * inf inside a numeric group): counted in the total, excluded from clustering (cu:1105-1114). */

/* ---- packed per-group result word ("meta") ----
 * bits  0..5  idx      vote: candidate index of the FIRST cell of the winning class (cu:971)
 *                      numeric: index of the single non-None cell when KC_FLAG_SINGLE
 * bits  6..12 support  vote: best_count (cu:958,969); numeric: support of the chosen cluster (cu:1177,1186,1218)
 * bits 13..19 nn       vote: number of voting cells; numeric: number of non-None cells == `total` (cu:1100)
 * bits 20..26 present  len(values) at this node == n - #absent (vote confidence denominator, cu:944,973)
 * bits 27..31 flags    KC_FLAG_*
 */
#define KC_META_IDX(m) ((uint32_t)(m) & 0x3Fu)
#define KC_META_SUPPORT(m) (((uint32_t)(m) >> 6) & 0x7Fu)
#define KC_META_NN(m) (((uint32_t)(m) >> 13) & 0x7Fu)
#define KC_META_PRESENT(m) (((uint32_t)(m) >> 20) & 0x7Fu)
#define KC_META_FLAGS(m) (((uint32_t)(m) >> 27) & 0x1Fu)
#define KC_META_PACK(idx, support, nn, present, flags) \
    (((uint32_t)(idx) & 0x3Fu) | (((uint32_t)(support) & 0x7Fu) << 6) | (((uint32_t)(nn) & 0x7Fu) << 13) | \
     (((uint32_t)(present) & 0x7Fu) << 20) | (((uint32_t)(flags) & 0x1Fu) << 27))

#define KC_FLAG_HAS_VALUE 1u  /* a consensus value exists (else the reference returns None) */
#define KC_FLAG_SINGLE 2u     /* numeric: exactly one non-None cell; value is the ORIGINAL object, confidence unrounded (cu:1085-1086) */
#define KC_FLAG_TIE 4u        /* vote: the maximum count was shared; numeric: tie resolution cu:1189-1219 ran */
#define KC_FLAG_NO_FINITE 8u  /* numeric: >=2 non-None cells, none finite (cu:1115-1116) */

/* ---- library ---- */
int kc_version(void);
const char *kc_last_error(void); /* thread-local text of the last KC_ECUDA / KC_EINVAL */
int kc_device_count(void);       /* number of visible CUDA devices with compute capability 10.x */
int kc_sm_count(int device);     /* multiprocessor count (148 on B200) or KC_E* */
int kc_set_device(int device);   /* make `device` current for this thread's subsequent d_* calls (this library links its own
                                    CUDA runtime instance; a torch caller passes torch.cuda.current_device()) */

/*
 * K1 — vote consensus over dictionary-coded str/bool groups.
 * Replaces voting_consensus (consensus_utils.py:936-982) on pre-sanitised input.
 *   d_codes     int32[n_groups][n]   KC_CODE_* or code >= 0; 16-byte aligned
 *   d_none_code int32[n_fields] or NULL.  Per field (field = g % n_fields): -1 => None cells do not
 *               vote (string fields, cu:964); c >= 0 => None cells vote as code c (bool fields map
 *               None to False, cu:956; allow_none_as_candidate maps None to its own code, cu:961-962).
 *   d_win_code  int32[n_groups]      code of the winning class, KC_CODE_NONE if no cell voted
 *   d_meta      uint32[n_groups]     packed result word
 * Ties go to the class seen first (cu:958,969: Counter insertion order).  1 <= n <= 64.
 */
int kc_vote_i32(const int32_t *d_codes, int64_t n_groups, int32_t n, const int32_t *d_none_code, int32_t n_fields,
                int32_t *d_win_code, uint32_t *d_meta, void *stream);

/*
 * K1 on COMPACT cells: votes only need equality inside a group, so a group can always be re-coded with local codes
 * 0..n-1; int8 cells (-1 None, -2 absent, 0..127 codes) are a lossless format at a quarter of the bytes.  Same outputs.
 */
int kc_vote_i8(const int8_t *d_codes, int64_t n_groups, int32_t n, const int32_t *d_none_code, int32_t n_fields,
               int32_t *d_win_code, uint32_t *d_meta, void *stream);

/*
 * K2 — numeric consensus: sort, 1-D tolerance clustering, largest cluster, numpy-order mean.
 * Replaces the numeric branch of consensus_as_primitive (consensus_utils.py:1098-1219).
 *   d_vals   float64[n_groups][n]  finite value, KC_F64_NONE_BITS, KC_F64_ABSENT_BITS, or any other
 *            non-finite ("present but not a number"); 16-byte aligned
 *   d_value  float64[n_groups]     float(np.mean(cluster)) bit-exact (numpy pairwise order); for
 *            KC_FLAG_SINGLE the cell itself; NaN when no value
 *   rel_eps, abs_eps >= 0          ConsensusSettings.rel_eps / abs_eps (cu:63-64)
 */
int kc_numeric_f64(const double *d_vals, int64_t n_groups, int32_t n, double rel_eps, double abs_eps, double *d_value,
                   uint32_t *d_meta, void *stream);

/*
 * Fused compute + reassembly for multi-GPU batches.  With out_mode == KC_OUT_MULTIMEM the output pointers are
 * NVSwitch MULTICAST addresses (a CUDA multicast object bound on every GPU of the group, e.g. torch symmetric
 * memory's multicast_ptr + this rank's slot offset): results are written with `multimem.st`, so the switch replicates
 * every store into all GPUs' copies of the buffer — the all-gather of the output columns happens inside the
 * producing kernel instead of a separate NCCL collective.  The caller runs a cross-GPU barrier before reading.
 */
#define KC_OUT_LOCAL 0u
#define KC_OUT_MULTIMEM 1u
int kc_vote_i32_ex(const int32_t *d_codes, int64_t n_groups, int32_t n, const int32_t *d_none_code, int32_t n_fields,
                   int32_t *d_win_code, uint32_t *d_meta, uint32_t out_mode, void *stream);
int kc_numeric_f64_ex(const double *d_vals, int64_t n_groups, int32_t n, double rel_eps, double abs_eps, double *d_value,
                      uint32_t *d_meta, uint32_t out_mode, void *stream);

/*
 * The same fusion over peer-to-peer stores (KC_OUT_PEERS): the output pointers are LOCAL addresses inside a buffer that
 * n_peers (<= 7) other GPUs map as well (e.g. torch symmetric memory's buffer_ptrs); every result is stored locally and
 * at address + peer_delta_bytes[k] for each peer k (the distance from this GPU's mapping of the buffer to peer k's, a
 * multiple of 8).  A multicast store also comes back to its sender, so every GPU receives world x its share; with P2P
 * stores it receives (world - 1) shares and sends as many — the better trade on full-duplex NVLink (measured: DESIGN §7).
 */
#define KC_OUT_PEERS 2u
int kc_vote_i32_peers(const int32_t *d_codes, int64_t n_groups, int32_t n, const int32_t *d_none_code, int32_t n_fields,
                      int32_t *d_win_code, uint32_t *d_meta, int32_t n_peers, const int64_t *peer_delta_bytes, void *stream);
int kc_numeric_f64_peers(const double *d_vals, int64_t n_groups, int32_t n, double rel_eps, double abs_eps, double *d_value,
                         uint32_t *d_meta, int32_t n_peers, const int64_t *peer_delta_bytes, void *stream);

/*
 * K1 with a PACKED gathered result.  The full result (d_win_code, d_meta: plain local arrays, not shared) stays on the
 * owning GPU — its decoder needs the first-seen index in the result word — and one word per group,
 *     KC_PACKED_VOTE: code:18 | support:7 | present:7      (support == 0: no value; confidence = support / present)
 * goes to d_packed (a LOCAL address inside the shared buffer) and to d_packed + peer_delta_bytes[k] on every peer: 4 instead
 * of 8 bytes per vote field cross NVLink, and the fused reassembly is NVLink-ingress-bound.  A winning code >= 2^18 cannot
 * be packed: the kernel sets *d_overflow (device uint32, zeroed by the caller) and the caller repeats with kc_vote_i32_peers.
 */
#define KC_PACKED_CODE(w) ((uint32_t)(w) & 0x3FFFFu)
#define KC_PACKED_SUPPORT(w) (((uint32_t)(w) >> 18) & 0x7Fu)
#define KC_PACKED_PRESENT(w) (((uint32_t)(w) >> 25) & 0x7Fu)
int kc_vote_i32_peers_packed(const int32_t *d_codes, int64_t n_groups, int32_t n, const int32_t *d_none_code, int32_t n_fields,
                             int32_t *d_win_code, uint32_t *d_meta, uint32_t *d_packed, int32_t n_peers,
                             const int64_t *peer_delta_bytes, uint32_t *d_overflow, void *stream);

/*
 * Reassembly of a sharded batch in the WIRE format (k_llms_b200/csrc/kc_push.cuh).  K1 / K2 keep their full results in plain
 * local arrays (fast local-store kernels); this call packs the results of one chunk of the shard and writes them — as whole
 * 16-byte vectors — into this rank's slot of a gathered buffer that n_peers other GPUs map as well (symmetric memory), i.e. to
 * d_wire_* and to d_wire_* + peer_delta_bytes[k] for every peer.  Launched on a second stream for chunk c while chunk c + 1 is
 * computed, it overlaps the NVLink transfer with the kernels without slowing them down.
 *   wide == 0 (n <= 31):  vote word u16 code:6 | support:5 | present:5;  numeric: f64 value + u16 kind:2 | payload:10
 *                         (kind 0 value, payload support | nn<<5;  1 single cell, payload present;  2 no finite value, payload
 *                         nn | present<<5;  3 no value, payload present) — 128 B per S32 record
 *   wide == 1:            vote word u32 KC_PACKED_*;  numeric: f64 value + the u32 result word — 192 B per S32 record
 * A result that does not fit the narrow words (winning code >= 64, a count > 31) sets *d_overflow (device uint32, zeroed by
 * the caller); the caller repeats the step with wide = 1.  n_vote_groups and n_num_groups must be multiples of 8; every buffer
 * and every peer_delta_bytes[k] 16-byte aligned.  max_ctas <= 0: twice the SM count.
 */
#define KC_WIRE_VOTE16_CODE(w) ((uint32_t)(w) & 63u)
#define KC_WIRE_VOTE16_SUPPORT(w) (((uint32_t)(w) >> 6) & 31u)
#define KC_WIRE_VOTE16_PRESENT(w) (((uint32_t)(w) >> 11) & 31u)
#define KC_WIRE_NUM16_KIND(w) (((uint32_t)(w) >> 10) & 3u)
/* K1 that also writes the wire word of every group (u16, or u32 when wide) to d_wire_words — this rank's slot of the gathered
 * buffer — next to the full local result, and (n_peers > 0: fused reassembly) to d_wire_words + peer_delta_bytes[k] in every
 * peer's copy; with n_peers == 0, kc_push_results(d_win_code = NULL, ...) replicates the words afterwards.  K2 needs no twin:
 * point its d_value into the slot and pass the same pointer as d_value and d_wire_value to kc_push_results. */
int kc_vote_i32_wire(const int32_t *d_codes, int64_t n_groups, int32_t n, const int32_t *d_none_code, int32_t n_fields,
                     int32_t *d_win_code, uint32_t *d_meta, void *d_wire_words, int32_t wide, int32_t n_peers,
                     const int64_t *peer_delta_bytes, uint32_t *d_overflow, void *stream);
int kc_push_results(const int32_t *d_win_code, const uint32_t *d_vote_meta, int64_t n_vote_groups, const double *d_value,
                    const uint32_t *d_num_meta, int64_t n_num_groups, void *d_wire_votes, void *d_wire_value, void *d_wire_num_meta,
                    int32_t wide, int32_t n_peers, const int64_t *peer_delta_bytes, uint32_t *d_overflow, int32_t max_ctas, void *stream);

/*
 * Confidences from result words, bit-exact with Python's round(x, 5) (cu:982,1178,1187,1219):
 *   vote    (numeric == 0): round(pvf * (support / present), 5)          cu:973,982
 *   numeric (numeric == 1): round(support / nn, 5); SINGLE: pvf * (1/present) unrounded (cu:1086,1444)
 *   no value: all-None -> 0.0 (cu:1402); empty -> pvf (cu:1396); NO_FINITE -> pvf * nn/present (cu:1116)
 * d_pvf float64[n_groups] or NULL (=1.0): parent_valid_frac of each group.
 */
int kc_confidence_f64(const uint32_t *d_meta, int64_t n_groups, int32_t numeric, const double *d_pvf, double *d_conf,
                      void *stream);

/*
 * K3 — per-candidate sequence log-likelihood: fp32 sum of per-token logprobs (NEW feature: the
 * reference only passes `logprobs` through, consolidation.py:129,135; SURVEY.md §0.3 — spec in DESIGN.md).
 *   d_logprobs float32[offsets[n_seq]]   d_offsets int64[n_seq+1] (ascending)   d_sum float32[n_seq]
 * Summation order is fixed (32 strided partial sums, then a xor-butterfly 16,8,4,2,1) so results are
 * bit-reproducible; the oracle restates the same order.
 */
int kc_logprob_sum_f32(const float *d_logprobs, const int64_t *d_offsets, int64_t n_seq, float *d_sum, void *stream);

/*
 * K3b — likelihood-weighted vote (NEW feature, self-defined: DESIGN.md §5).  Candidate weight
 * w_c = kexp(seq_logprob[record][c] - max_k seq_logprob[record][k]); class weight = sum of its cells' weights
 * (fp32, ascending candidate order); the heaviest class wins, ties -> first seen.
 *   d_codes int32[n_records*n_fields][n] as kc_vote_i32; d_seq_logprob float32[n_records][n] (e.g. kc_logprob_sum_f32)
 *   d_weight float32[n_groups]: winning class weight / total voting weight (0 if nothing voted)
 */
int kc_weighted_vote_i32(const int32_t *d_codes, const float *d_seq_logprob, int64_t n_records, int32_t n_fields,
                         int32_t n, const int32_t *d_none_code, int32_t *d_win_code, uint32_t *d_meta, float *d_weight,
                         void *stream);

/*
 * Candidate weights of likelihood-weighted consolidation (NEW feature, self-defined: DESIGN.md §5) — K3b's weight pre-pass:
 *   d_seq_logprob float32[n_records][n]  ->  d_weight float32[n_records][n],  w_c = kexp(s_c - max_k s_k) per record
 * (kexp: the fixed-order fp32 exp of K3b).  1 <= n <= 64.  A slot that is not a candidate of its record can be filled with
 * -3.0e38f: it never raises the record's maximum.
 */
int kc_candidate_weights_f32(const float *d_seq_logprob, int64_t n_records, int32_t n, float *d_weight, void *stream);

/*
 * Likelihood-weighted vote over IRREGULAR groups (NEW feature, self-defined: DESIGN.md §5): K3b's vote (class weight = fp32 sum of
 * its cells' weights in cell order; the heaviest class wins; among equal weights the class whose first cell comes first) for
 * groups that need not be fields of one fixed record layout.
 *   d_cells        [n_groups][n]  K1's coding (code >= 0 class, KC_CODE_NONE, < KC_CODE_NONE absent); None cells do not vote
 *                  (int8: the device JSON path's cell matrix, int32: the planner's)
 *   d_group_record int32[n_groups]  the record of each group (index into d_weight's rows)
 *   d_cand         int8[n_groups][n] or NULL: the candidate of each present cell (NULL: cell c is candidate c)
 *   d_weight       float32[n_records][n] (kc_candidate_weights_f32)
 *   d_meta         uint32[n_groups]  K1's result word: idx | support | nn | present | flags; KC_FLAG_TIE when another class
 *                  weighs exactly as much as the winner
 *   d_sums         float32[n_groups][2] (8-byte aligned): W_win (0 if no cell voted), W_present = fp32 sum of the weights of the
 *                  present cells, None cells included, in cell order.  Confidence: round(pvf * (W_win / W_present), 5) in double.
 * 1 <= n <= 64.
 */
int kc_weighted_vote_groups_i8(const int8_t *d_cells, int64_t n_groups, int32_t n, const int32_t *d_group_record, const int8_t *d_cand,
                               const float *d_weight, uint32_t *d_meta, float *d_sums, void *stream);
int kc_weighted_vote_groups_i32(const int32_t *d_cells, int64_t n_groups, int32_t n, const int32_t *d_group_record, const int8_t *d_cand,
                                const float *d_weight, uint32_t *d_meta, float *d_sums, void *stream);

/*
 * K4 — similarity medoid of string groups (consensus_as_primitive fallback, consensus_utils.py:1221-1237, with
 * levenshtein_similarity :745-761): pairwise 1 - dist/max_len (floored at 1e-8) on NORMALISED strings (lower-case [a-z0-9],
 * normalize_string :660-673, done by the caller), np.nanmean of each row in numpy's summation order, first argmax.
 *   d_chars uint8[...]   all strings back to back       d_str_off int32[S+1]  string s = chars[str_off[s] .. str_off[s+1])
 *   d_grp_off int32[G+1] group g = strings grp_off[g] .. grp_off[g+1]  (2..max_group strings per group, max_group <= 64:
 *                        it sizes the per-warp shared memory, so pass the real maximum, not 64)
 *   contract: for every pair of one group, the shorter string has at most 64 characters (Myers' bit-parallel distance),
 *             and no string is longer than 65535 characters
 *   d_best_idx int32[G] index (within the group) of the medoid; d_best_avg float64[G] its mean similarity (unrounded)
 */
int kc_medoid_str(const uint8_t *d_chars, const int32_t *d_str_off, const int32_t *d_grp_off, int64_t n_groups,
                  int32_t max_group, int32_t *d_best_idx, double *d_best_avg, void *stream);

/* K4 with the other string similarities of the reference (ConsensusSettings.string_similarity_method, cu:56): KC_SIM_LEVENSHTEIN
 * as above; KC_SIM_JACCARD = |A & B| / |A | B| on the character SETS (jaccard_similarity, cu:720-742); KC_SIM_HAMMING = 1 -
 * mismatches / max_len position by position, the shorter string padded (hamming_similarity, cu:676-717); both floored at 1e-8.
 * The 64-character contract applies to KC_SIM_LEVENSHTEIN only. */
#define KC_SIM_LEVENSHTEIN 0
#define KC_SIM_JACCARD 1
#define KC_SIM_HAMMING 2
int kc_medoid_str_method(const uint8_t *d_chars, const int32_t *d_str_off, const int32_t *d_grp_off, int64_t n_groups,
                         int32_t max_group, int32_t method, int32_t *d_best_idx, double *d_best_avg, void *stream);

/* K4 with HOST buffers (H2D, one launch, D2H; synchronous): what the host planners call for a batch of string groups. */
int kc_medoid_str_host(const uint8_t *h_chars, int64_t n_chars, const int32_t *h_str_off, const int32_t *h_grp_off, int64_t n_groups,
                       int32_t max_group, int32_t *h_best_idx, double *h_best_avg, int device);

/*
 * End-to-end entry with HOST buffers (the call a k_llms binding makes for a batch of records of one
 * flat schema): chunked, double-buffered H2D -> K1/K2 -> D2H on internal streams of `device`.
 * Either half may be absent (n_vote_fields == 0 or n_num_fields == 0).  Blocks until results are in
 * host memory.  Host buffers should be page-locked (kc_host_alloc) for full PCIe bandwidth.
 */
int kc_consensus_host(const int32_t *h_codes, int32_t n_vote_fields, const int32_t *h_none_code, const double *h_vals,
                      int32_t n_num_fields, int64_t n_records, int32_t n, double rel_eps, double abs_eps,
                      int32_t *h_win_code, uint32_t *h_vote_meta, double *h_value, uint32_t *h_num_meta, int device,
                      float *device_ms /* optional: CUDA-event time of the whole call (copies + kernels), NULL to skip */);

/* Same with int8 vote cells (see kc_vote_i8): 2.56 GB -> 1.41 GB over PCIe for 1M x 32 fields at n = 16. */
int kc_consensus_host_i8(const int8_t *h_codes, int32_t n_vote_fields, const int32_t *h_none_code, const double *h_vals,
                         int32_t n_num_fields, int64_t n_records, int32_t n, double rel_eps, double abs_eps,
                         int32_t *h_win_code, uint32_t *h_vote_meta, double *h_value, uint32_t *h_num_meta, int device,
                         float *device_ms);

/*
 * H1 in two phases, for callers that run K1 / K2 / K4 themselves (own streams, another device; the CPU tests put the oracle
 * in their place to check the host logic without a GPU).  kc_json_plan parses, plans and encodes a batch into host arrays owned
 * by the handle; kc_json_inputs exposes them (vote cells int8[n_vote_groups][n] as kc_vote_i8 takes them with n_fields = 1 and
 * no none_code; numeric cells float64[n_num_groups][n]; medoid groups in kc_medoid_str's CSR form); the caller computes
 * vote_meta uint32[n_vote_groups], num_value float64 / num_meta uint32 [n_num_groups], medoid_idx int32 / medoid_avg float64
 * [n_medoid_groups]; kc_json_emit turns them into the texts kc_consolidate_json returns.  The candidate texts must stay alive
 * until kc_json_emit has returned (cells are views into them).
 */
typedef struct kc_json_batch kc_json_batch;
int kc_json_plan(const char *const *texts, const int64_t *lens, int64_t n_records, int32_t n, int32_t threads, kc_json_batch **out);
int kc_json_inputs(const kc_json_batch *h, const int8_t **vote_cells, int64_t *n_vote_groups, const double **num_cells,
                   int64_t *n_num_groups, const uint8_t **medoid_chars, const int32_t **medoid_str_off, const int32_t **medoid_grp_off,
                   int64_t *n_medoid_groups, int32_t *max_medoid_group);
int kc_json_emit(kc_json_batch *h, const uint32_t *vote_meta, const double *num_value, const uint32_t *num_meta, const int32_t *medoid_idx,
                 const double *medoid_avg, char **out_content, char **out_likelihoods, uint8_t *out_status);
void kc_json_free(kc_json_batch *h);

/*
 * H2 — the alignment pre-pass of the client path, natively (SURVEY.md §8f-3): recursive_list_alignments
 * (consensus_utils.py:458-613; lists_alignment :383-430 with the dynamic threshold :185-252, the reference list :255-333, the
 * min-cost assignment :336-380 = scipy's linear_sum_assignment restated, pruning :109-149; majority ordering
 * majority_sorting.py:8-112) for ONE record: n candidate values as JSON texts ("null" = None) in, out_texts[c] = json.dumps of
 * candidate c's aligned value (free with kc_free_strings).  Host code, no GPU.  The default string similarity method
 * ("embeddings") is assumed.  Returns 0; 1 = the record needs the Python path (two strings both longer than 50 characters
 * would be compared through the embeddings service, consensus_utils.py:813; non-ASCII text); KC_EINVAL for invalid JSON.
 * Dict-field similarities are summed in sorted key order (the reference's order depends on PYTHONHASHSEED): similarities agree
 * to an ulp, alignments are pinned on the reference's goldens (tests/test_align_native.py).
 */
int kc_align_json(const char *const *texts, const int64_t *lens, int32_t n, double min_support_ratio, char **out_texts);
/* test hooks of H2: generic_similarity (consensus_utils.py:892-917) of two JSON values; scipy.optimize.linear_sum_assignment */
int kc_debug_similarity_json(const char *a, const char *b, double *out);
int kc_debug_lsap(int32_t nr, int32_t nc, const double *cost, int32_t *row_ind, int32_t *col_ind);

/*
 * H1 — native columnariser / decoder for records of scalars, nested objects and lists (SURVEY.md §8f-1, §8f-3): for each record, n candidate JSON texts in ->
 * consensus JSON text + likelihoods JSON text out, multi-threaded on the host with K1/K2 in between.  Replaces, for such
 * records, the Python around the hot path: _safe_parse_content (consolidation.py:25-38), the dict part of
 * recursive_list_alignments (consensus_utils.py:516-548: keys sorted, missing -> None), the dispatcher
 * (consensus_utils.py:1376-1454), sanitize_value (:925-933) and _format_consensus_content (consolidation.py:41-60).
 *   texts   [n_records * n] candidate contents (record-major); lens [n_records * n] byte lengths or NULL (NUL-terminated)
 *   out_content / out_likelihoods [n_records] malloc'ed NUL-terminated strings (free with kc_free_strings), byte-identical
 *           to the reference's json.dumps output; out_status [n_records]: 0 = consolidated here, 1 = not expressible as
 *           groups for K1/K2/K4 (a key mixing objects with other types, string pairs that need the embeddings service, non-ASCII,
 *           empty content, ...) -> caller uses the Python path.  Implements the reference's DEFAULT settings (similarity method
 *           "embeddings", min_support_ratio 0.51, Nones do not vote); other settings: Python path
 *   threads <= 0: min(32, hardware threads).  Blocks until done; callers are serialised (one staging pool per process).
 */
int kc_consolidate_json(const char *const *texts, const int64_t *lens, int64_t n_records, int32_t n, double rel_eps,
                        double abs_eps, int device, int32_t threads, char **out_content, char **out_likelihoods,
                        uint8_t *out_status);
void kc_free_strings(char **arr, int64_t count);

/*
 * H1g — the same consolidation with the JSON work ON THE DEVICE (k_llms_b200/csrc/kc_jsongpu.cuh): the candidate texts are
 * copied to the GPU as they are; kernels scan them (json.loads, consolidation.py:25-38), sort and check the keys (the dict part
 * of recursive_list_alignments, consensus_utils.py:516-548), type the fields (dispatcher :1376-1454), build K1 cells by
 * sanitised equality (sanitize_value :925-933) and K2 cells by exact decimal -> float64 conversion, run K1 / K2, and write the
 * consensus and likelihoods texts (json.dumps, consolidation.py:41-60; float.__repr__ by shortest-digits conversion).  The host
 * only moves bytes.  Records the device path does not model exactly (escapes, non-ASCII, nested values / lists, candidates with
 * different key sequences, multi-word strings, NaN / Infinity, > 19 significant digits, ...) are consolidated by the host path
 * (kc_consolidate_json) inside the same call; what that declines too is left to the caller's Python path.
 *   h_text   all candidate texts back to back (ideally page-locked: kc_host_alloc)
 *   h_off    int64[n_records * n + 1]  candidate c of record r is h_text[h_off[r*n+c] .. h_off[r*n+c+1])  (record-major)
 *   flags    KC_JSON_DEVICE_ONLY: skip the host path (declined records keep status 1)
 *   *out     result handle: one text blob + per-record spans (kc_json_result_view), released with kc_json_result_free
 * status per record: 0 = consolidated on the device, 2 = consolidated by the host path, 1 = needs the Python path.
 * Texts are byte-identical to the reference's json.dumps output.  Re-entrant (pooled per-call streams and buffers).
 */
#define KC_JSON_DEVICE_ONLY 1u
typedef struct kc_json_result kc_json_result;
typedef struct {
    int64_t n_records, n_device, n_host, n_python; /* where the records were consolidated */
    int64_t input_bytes, output_bytes;
    int32_t chunks, streams;
    /* device time by stage, summed over the chunks (CUDA events on each chunk's stream; chunks overlap, so the sum of the
     * stages can exceed the wall time) */
    double h2d_ms, plan_ms /* A0 + A1 (+ A2): scan, type, encode */, kernel_ms /* K1 + K2 (+ K4) */, emit_ms /* C0 + C1 */, d2h_ms;
    double device_path_wall_ms, host_path_wall_ms, wall_ms;
} kc_json_stats;
int kc_consolidate_json_packed(const char *h_text, const int64_t *h_off, int64_t n_records, int32_t n, double rel_eps, double abs_eps,
                               int device, int32_t threads, uint32_t flags, kc_json_result **out);
/*
 * H1g with the likelihood-weighted vote (NEW feature, self-defined: DESIGN.md §5).  The arguments of kc_consolidate_json_packed plus
 *   h_lp      float32 token logprobs of every candidate, back to back
 *   h_lp_off  int64[n_records * n + 1]  candidate c of record r has the tokens h_lp[h_lp_off[r*n+c] .. h_lp_off[r*n+c+1]) (ascending)
 * Per chunk the logprobs go to the device next to the texts; K3 sums them per candidate, kc_candidate_weights_f32 turns the sums
 * into weights, and the vote fields are decided by kc_weighted_vote_groups_i8 (confidence round(W_win / W_present, 5)).  Numeric
 * and multi-word fields are not weighted.  The host path H1 does not weight: records the device path declines keep status 1 (as
 * with KC_JSON_DEVICE_ONLY).  stats.input_bytes counts the logprob bytes.
 */
int kc_consolidate_json_packed_weighted(const char *h_text, const int64_t *h_off, const float *h_lp, const int64_t *h_lp_off,
                                        int64_t n_records, int32_t n, double rel_eps, double abs_eps, int device, int32_t threads,
                                        uint32_t flags, kc_json_result **out);
/* record r: content = text[content_off[r] .. +content_len[r]), likelihoods likewise; `why` = the device path's reason code for
 * declining (0 = not declined; kc_jsoncore.cuh D_*).  Pointers stay valid until kc_json_result_free.  Any output may be NULL. */
int kc_json_result_view(kc_json_result *res, const char **text, const int64_t **content_off, const int64_t **content_len,
                        const int64_t **likelihoods_off, const int64_t **likelihoods_len, const uint8_t **status, const uint8_t **why,
                        kc_json_stats *stats);
void kc_json_result_free(kc_json_result *res);

/* Test hooks of H1g: the device phases instantiated on the host (same source), in the two-phase shape of kc_json_plan /
 * kc_json_emit, so the CPU tests can put the oracle in K1 / K2's place.  Not a product path. */
typedef struct kc_debug_jsongpu kc_debug_jsongpu;
int kc_debug_jsongpu_plan(const char *h_text, const int64_t *h_off, int64_t n_records, int32_t n, kc_debug_jsongpu **out);
int kc_debug_jsongpu_inputs(const kc_debug_jsongpu *h, const int8_t **vote_cells, int64_t *n_vote_groups, const double **num_cells,
                            int64_t *n_num_groups, const uint8_t **status);
int kc_debug_jsongpu_emit(kc_debug_jsongpu *h, const uint32_t *vote_meta, const double *num_value, const uint32_t *num_meta,
                          const char **content, const int64_t **content_off, const char **likelihoods, const int64_t **likelihoods_off);
/* the batch's medoid groups (multi-word string fields) in kc_medoid_str's CSR form; K4's results go in through _set_medoid
 * (before _emit; the arrays must stay alive until _emit has returned) */
int kc_debug_jsongpu_medoid_inputs(const kc_debug_jsongpu *h, const uint8_t **chars, const int32_t **str_off, const int32_t **grp_off,
                                   int64_t *n_groups);
int kc_debug_jsongpu_set_medoid(kc_debug_jsongpu *h, const int32_t *medoid_idx, const double *medoid_avg);
/* the weighted entry's phases (self-defined, DESIGN.md §5): the record of every vote group (kc_weighted_vote_groups_i8's
 * d_group_record), and the emit with the weighted vote's float32[n_vote_groups][2] (W_win, W_present) */
int kc_debug_jsongpu_vote_records(const kc_debug_jsongpu *h, const int32_t **vote_records);
int kc_debug_jsongpu_emit_weighted(kc_debug_jsongpu *h, const uint32_t *vote_meta, const float *vote_sums, const double *num_value,
                                   const uint32_t *num_meta, const char **content, const int64_t **content_off, const char **likelihoods,
                                   const int64_t **likelihoods_off);
void kc_debug_jsongpu_free(kc_debug_jsongpu *h);
int kc_debug_parse_doubles(const char *text, const int64_t *off, int64_t count, double *out, uint8_t *ok);
int kc_debug_float_reprs(const double *xs, int64_t count, char *out /* [count][32] */, int32_t *lens);
int kc_debug_round5(const double *xs, int64_t count, double *out);
/* Bench / test input: n_records records of schema S32 (SURVEY.md §8d) as candidate texts, exactly as json.dumps prints them.
 * Call with out == NULL to get the offsets (off[n_records*n] = bytes needed), then with a buffer of that size. */
int kc_debug_s32_texts(uint64_t seed, int64_t n_records, int32_t n, int32_t threads, char *out, int64_t cap, int64_t *off);

/* Host helper: unit-cost edit distance of two byte strings (python-Levenshtein `distance`, consensus_utils.py:759),
 * used by the host similarity medoid / list alignment.  -1 on bad arguments. */
int32_t kc_levenshtein(const char *a, int32_t alen, const char *b, int32_t blen);

void *kc_host_alloc(uint64_t bytes); /* page-locked host memory, NULL on failure */
void kc_host_free(void *p);

#ifdef __cplusplus
}
#endif
#endif /* KLLMS_B200_H */
