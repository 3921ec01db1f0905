/*
 * xmve.h -- C ABI of the B200-native retrieval scoring library (libxmve.so, sm_100a only).
 *
 * The reference (WWWindrunner/Cross-Modal-Video-Engine) is 100 % Python and has no FFI: its
 * boundary for this path is a set of Python call signatures (SURVEY.md section 8b).  Each entry
 * point below names the reference lines whose arithmetic it replaces; the Python mirror of the
 * reference modules (cross-modal-video-engine_b200/{evaluation,validate,metrics,...}.py) binds
 * them through ctypes.  INTEGRATION.md shows the binding a reference maintainer would add.
 *
 * Conventions
 *   - every function returns 0 on success or a negative xmve_status; xmve_last_error() gives a
 *     thread-local message for the last failure.
 *   - all data pointers are DEVICE pointers borrowed from the caller (e.g. torch data_ptr());
 *     nothing is allocated, owned or freed by the library.  `stream` is a cudaStream_t passed as
 *     void*; work is enqueued on it and the call returns without synchronising.
 *   - matrices are row-major; `ld` arguments are row strides in ELEMENTS.
 *   - there is no CPU path: on a device that is not compute capability 10.x every call fails
 *     with XMVE_ERR_DEVICE.
 */
#ifndef XMVE_H_
#define XMVE_H_

#include <stdint.h>

#if defined(__GNUC__)
#define XMVE_API __attribute__((visibility("default")))
#else
#define XMVE_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef enum xmve_status {
  XMVE_OK = 0,
  XMVE_ERR_ARG = -1,     /* bad argument (null pointer, misaligned, out of range) */
  XMVE_ERR_DEVICE = -2,  /* no CUDA device / not sm_100 */
  XMVE_ERR_CUDA = -3,    /* a CUDA runtime / driver call failed */
  XMVE_ERR_LIMIT = -4    /* a size exceeds what the kernel supports (see each function) */
} xmve_status;

enum { XMVE_F32 = 0, XMVE_F64 = 1 };

/* operand layouts written by xmve_prepare_rows (how one embedding space is laid out along K) */
enum {
  XMVE_OP_X1 = 0,        /* [hi]            K = dpad      bf16(w * x_hat)                        */
  XMVE_OP_X3_QUERY = 1,  /* [hi | hi | lo]  K = 3 * dpad  split-bf16, query side                  */
  XMVE_OP_X3_CORPUS = 2  /* [hi | lo | hi]  K = 3 * dpad  split-bf16, corpus side                 */
};

enum { XMVE_NORM_PLAIN = 0,   /* x / ||x||            (evaluation.py:10-14, no epsilon)          */
       XMVE_NORM_EPS = 1 };   /* x / max(||x||,1e-12) (torch F.normalize, MultiFusion validate.py:55) */

XMVE_API int xmve_version(void);
XMVE_API const char* xmve_last_error(void);
/* Fails unless `device` (or the current device if < 0) is compute capability 10.x. */
XMVE_API int xmve_device_check(int device);
/* Number of SMs of the current device (grid sizing); < 0 on error. */
XMVE_API int xmve_sm_count(void);

/* ---- K1: row normalise + cast (corpus-resident store, query prep) -----------------------------
 * Replaces evaluation.l2norm (LINAS-engine/evaluation.py:10-14), the re-normalisation inside
 * cal_error (:19-20), F.normalize(index).float() (MultiFusion/src/validate.py:55) and, with
 * frames > 1, Combiner.time_process = mean over frames (MultiFusion/src/combiner.py:140-143).
 *
 * src       [n, frames, d] fp32/fp64 (src_dtype), row stride src_ld elements (>= frames*d)
 * raw_out   optional fp32 [n, raw_ld]: the (frame-pooled) raw row is written at column raw_off
 * norm_out  optional fp64 [n]: ||x||_2 accumulated in double
 * resid_out optional fp32 [n]: ||w*x_hat - bf16(w*x_hat)||^2 of the row's hi plane, rounded up (the measured
 *           bf16 quantisation residual; engine.py turns the maxima of both sides into the rigorous bound
 *           eps on |tensor-core score - exact score| that certifies the top-k)
 * op_out    optional bf16 [n, op_ld]: operand planes per op_layout written at column op_off,
 *           plane stride dpad = round_up(d, 64); columns d..dpad of each plane are zero-filled
 * weight    folded into the operand (per-space fusion weight; 1.0 on the corpus side)
 */
XMVE_API int xmve_prepare_rows(const void* src, int src_dtype, int64_t n, int d, int frames, int64_t src_ld,
                      float* raw_out, int64_t raw_ld, int64_t raw_off,
                      double* norm_out, float* resid_out,
                      void* op_out, int64_t op_ld, int64_t op_off, int op_layout,
                      float weight, int norm_mode, void* stream);

/* ---- K2: query x corpus score kernel (tcgen05 / TMEM / TMA, bf16 operands, fp32 accumulate) ----
 * Replaces np.dot(l2norm(captions), l2norm(videos).T) (LINAS-engine/evaluation.py:21,45,79) and
 * P @ index.T (MultiFusion/src/validate.py:73,90; inference.py:63).  a_op [nq, a_ld] and
 * b_op [nv, b_ld] are bf16 operands from xmve_prepare_rows (16-byte aligned, ld % 8 == 0), k is the
 * contraction length in elements (multiple of 64).  b_row_step > 1 scores every b_row_step-th
 * corpus row only (a strided TMA view; nv is then the number of sampled rows).
 *
 * store : out[q, v] = alpha * <a_q, b_v>   fp32 [nq, out_ld]     (cal_error: alpha = -1)
 */
XMVE_API int xmve_score_store(const void* a_op, int64_t nq, int64_t a_ld,
                     const void* b_op, int64_t nv, int64_t b_ld, int64_t b_row_step, int k,
                     float alpha, float* out, int64_t out_ld, void* stream);

/* filter: the score matrix never reaches HBM.  Per query row q with window (lo[q], hi[q]]:
 *   s >  hi[q]            -> count_above[q] += 1                    (hi may be NULL = +inf)
 *   lo[q] < s <= hi[q]    -> slot = cand_count[q]++ ; if slot < cap:
 *                            cand_score[q*cap+slot] = s, cand_idx[q*cap+slot] = v
 * cand_count keeps counting past cap so the caller can detect overflow.  b_row_step as in xmve_score_store (v is
 * then the index of the sampled row).  Replaces the full
 * argsort of every row (LINAS-engine/inference.py:79; MultiFusion/src/validate.py:74,92) as a
 * streaming threshold top-k, and the rank-of-ground-truth search (util/metrics.py:139-145) as
 * count_above with a guard band.
 */
XMVE_API int xmve_score_filter(const void* a_op, int64_t nq, int64_t a_ld,
                      const void* b_op, int64_t nv, int64_t b_ld, int64_t b_row_step, int k,
                      const float* lo, const float* hi,
                      int32_t* count_above, int32_t* cand_count,
                      float* cand_score, int32_t* cand_idx, int32_t cap, void* stream);

/* filter_labeled: xmve_score_filter restricted per query row to the corpus rows whose label it allows.  Column v
 * (a sampled row when b_row_step > 1) has the label labels[v * b_row_step], 0 <= label < 64 (DEVICE uint8); row q
 * may list -- and count above hi -- only columns whose label bit is set in allow[q] (DEVICE uint64 [nq]).  Every
 * other score is skipped, so cand_count[q] and count_above[q] count eligible columns only.  The labels are read
 * only for scores that enter the window (lo[q], ...), from a shared-memory copy of the tile's labels: the extra cost
 * grows with the candidates, not with nv.  The wide tile (XMVE_TILE=2 / 6) has no shared memory left for the
 * labels and returns XMVE_ERR_ARG.
 */
XMVE_API int xmve_score_filter_labeled(const void* a_op, int64_t nq, int64_t a_ld,
                      const void* b_op, int64_t nv, int64_t b_ld, int64_t b_row_step, int k,
                      const float* lo, const float* hi,
                      int32_t* count_above, int32_t* cand_count,
                      float* cand_score, int32_t* cand_idx, int32_t cap,
                      const uint8_t* labels, const uint64_t* allow, void* stream);

/* mask_scores: in place, scores[r * ld + c] = -inf for every column c whose label labels[c * label_step] is not set
 * in allow[r] (DEVICE uint64 [rows]).  dtype XMVE_F32 or XMVE_F64.  Restricts a sampled STORE matrix
 * or an fp64 score matrix to the eligible corpus rows; the selection kernels skip -inf entries.
 */
XMVE_API int xmve_mask_scores(void* scores, int dtype, int64_t rows, int64_t cols, int64_t ld,
                              const uint8_t* labels, int64_t label_step, const uint64_t* allow, void* stream);

/* ---- order statistics of score rows ------------------------------------------------------------
 * out[r] = max( kth_largest(row r, j1) - sub , kth_largest(row r, j2) )   (j2 <= 0: first term only)
 * Row r holds min(counts[r], cols) valid floats (counts == NULL: cols).  Fewer than j valid values
 * give -inf for that term.  Used for the sampled filter threshold and the candidate pre-filter.
 * sub_dev (DEVICE scalar, may be NULL) multiplies sub: with the error bound eps living on the device (xmve_eps_bound)
 * "kth - 2 eps" is sub = 2, sub_dev = eps -- no host round trip, the step stays capturable in a CUDA graph.
 */
XMVE_API int xmve_row_kth(const float* vals, int64_t rows, int64_t cols, int64_t ld, const int32_t* counts,
                 int32_t j1, float sub, const float* sub_dev, int32_t j2, float* out, void* stream);

/* ---- exact rescoring of candidates in double precision -----------------------------------------
 * exact[q, c] = sum_s w[s] * <q_s, v_s> / (||q_s|| * ||v_s||)  for candidate c of row q whose
 * approximate score is >= bound[q] (bound == NULL: all), else -inf.  With bound_hi != NULL (the second round of the
 * two-round rescore) only candidates with bound[q] <= approx < bound_hi[q] are computed and the entries at or above
 * bound_hi[q] -- written by the first round -- are left untouched.  Raw rows are fp32 (values the
 * reference keeps in float64 arrays, evaluation.py:102-105); products and sums are in fp64, i.e.
 * the arithmetic of cal_error on float64 inputs (evaluation.py:19-21) up to rounding order.
 * space_off[n_space+1] (HOST array) are column offsets into the raw rows, weights[n_space] is a HOST
 * array, q_norm is DEVICE [n_space, nq] fp64 and v_norm DEVICE [n_space, nv] fp64: nv is the row stride of v_norm
 * (a corpus store's capacity, which may exceed the number of rows filled), the norm of corpus row v in space s is
 * v_norm[s * nv + v].  exact[q, c] is written for c < cand_count[q] only.
 * norm_mode as in xmve_prepare_rows.  Limit: total raw dim <= 6000.
 */
XMVE_API int xmve_rescore(const float* q_raw, int64_t nq, int64_t q_ld, const double* q_norm,
                 const float* v_raw, int64_t nv, int64_t v_ld, const double* v_norm,
                 int n_space, const int32_t* space_off, const double* weights, int norm_mode,
                 const float* cand_score, const int32_t* cand_idx, const int32_t* cand_count,
                 int32_t cap, const float* bound, const float* bound_hi, double* exact, void* stream);

/* ---- two-round rescore: the pilot -----------------------------------------------------------------------
 * Round one rescores the m best approximate candidates of every shard exactly.  xmve_pilot_top writes the (up to) m
 * largest finite entries of exact[r, :min(counts[r], cap)] in descending order, -inf padded, skipping the entry whose
 * global index idx + idx_offset equals exclude[r]: out fp64 [rows, m] (m <= 1024).  After the lists of all shards are
 * gathered ([n_seg, rows, m]), xmve_pilot_bound gives bound[r] = round_down(kth largest of the union - eps) (-inf if
 * the union has fewer than k finite scores): a candidate whose approximate score is below it cannot belong to the
 * top-k, because the k-th largest of ANY set of exact scores is a lower bound on the true k-th best and
 * |approx - exact| <= eps.  eps_dev as sub_dev above.  (Halves the rows gathered by the rescore against the one-round
 * window "approximate k-th - 2 eps".)
 */
XMVE_API int xmve_pilot_top(const double* exact, const int32_t* idx, const int32_t* counts, int64_t rows, int32_t cap,
                   int64_t idx_offset, const int64_t* exclude, int32_t m, double* out, void* stream);
XMVE_API int xmve_pilot_bound(const double* lists, int32_t n_seg, int64_t rows, int32_t m, int32_t k, float eps,
                     const float* eps_dev, float* bound, void* stream);

/* The rigorous bound eps on |tensor-core score - exact score| from the MEASURED bf16 residuals, on the device:
 * dq^2 = max_q sum_s q_resid[s, q], dv^2 = dv2[0] (max over corpus rows, all shards),
 * eps = dq*vn + qn*dv + k_len * 2^-22 * qn * vn + 1e-6, qn = w_norm + dq, vn = sqrt(n_space) * (1 + 2^-8), rounded up;
 * `fallback` when a residual is NaN (zero rows under XMVE_NORM_PLAIN).  eps_out: DEVICE float[1].
 */
XMVE_API int xmve_eps_bound(const float* q_resid, int32_t n_space, int64_t nq, const float* dv2, double w_norm,
                   int32_t k_len, float fallback, float* eps_out, void* stream);

/* ---- final top-k of each row from (score, index) pairs -----------------------------------------
 * Sorts the valid entries (score > -inf, index != exclude[r]) of row r by (score desc, index asc)
 * and writes the first k: out_score fp64 [rows, k] (-inf padded), out_idx int64 [rows, k]
 * (-1 padded; idx + idx_offset otherwise; idx == NULL means idx[r, c] = c), out_valid[r] = number
 * of valid entries.
 * Certification (thr != NULL): cert[r] = 1 iff counts[r] <= cols, at least k entries are valid and
 * kth_score - eps >= thr[r] -- then no corpus item outside the candidate set can belong to the
 * top-k given |approx - exact| <= eps.  thr_next[r] is the threshold to re-run an uncertified row
 * with (kth - eps when k entries were found; bound[r] = approximate kth of the retained candidates
 * - 2 eps after a candidate-list overflow).  The sort holds 16384 entries per row; rows with more valid entries
 * are first cut at the k-th largest score rounded to float (a superset of the exact top-k), so only > 16384
 * scores that agree with the k-th to float precision defeat it (reported as not certified).  (With 512 rows or more
 * the sort holds max(2048, 4k) entries so that several rows are resident per SM; a row that does not fit comes
 * back uncertified and must be re-run in a batch of fewer than 512 rows to get the full capacity.)
 * Without thr (a shard's local list that a later merge certifies), cert may still be given: cert[r] = 1 iff the
 * list is exact -- counts[r] <= cols and every entry that can belong to the top-k fit the sort -- and 0 when the
 * sort held only an arbitrary subset of tied entries; thr_next must then be NULL.
 * eps_dev (DEVICE scalar, may be NULL) multiplies eps.  n_uncertified (DEVICE int32, may be NULL) is incremented once
 * per uncertified row: the caller reads ONE scalar, asynchronously, instead of scanning cert on the host.
 */
XMVE_API int xmve_select_topk_i32(const double* score, const int32_t* idx, int64_t rows, int64_t cols,
                         const int32_t* counts, int64_t idx_offset, const int64_t* exclude, int32_t k,
                         const float* thr, float eps, const float* eps_dev, const float* bound,
                         double* out_score, int64_t* out_idx, int32_t* out_valid,
                         int32_t* cert, float* thr_next, int32_t* n_uncertified, void* stream);
/* K3: G-way merge of per-shard top-k lists after the all-gather: rows x (G*k) pairs with global
 * int64 indices -> top-k.  Same ordering rule.  With thr != NULL the merged list is certified like above
 * (cert, thr_next); overflow[r] != 0 says that some shard's candidate list of row r overflowed. */
XMVE_API int xmve_select_topk_i64(const double* score, const int64_t* idx, int64_t rows, int64_t cols,
                         const int64_t* exclude, int32_t k,
                         const float* thr, float eps, const float* eps_dev, const int32_t* overflow,
                         double* out_score, int64_t* out_idx, int32_t* out_valid,
                         int32_t* cert, float* thr_next, int32_t* n_uncertified, void* stream);
/* K3 on the result of ONE all-gather: every rank contributes one packed block of seg_bytes bytes
 *   [ score fp64 rows x len | global index int64 rows x len | overflow flag int32 rows | pad to 16 ]
 * (xmve_packed_topk_bytes(rows, len) bytes), `packed` holds the n_seg blocks back to back.  Same ordering rule,
 * certificate and outputs as xmve_select_topk_i64; a row is treated as overflowed if any block flags it.
 */
XMVE_API int64_t xmve_packed_topk_bytes(int64_t rows, int32_t len);
XMVE_API int xmve_merge_topk_packed(const void* packed, int32_t n_seg, int64_t seg_bytes, int64_t rows, int32_t len,
                           const int64_t* exclude, int32_t k, const float* thr, float eps, const float* eps_dev,
                           double* out_score, int64_t* out_idx, int32_t* cert, float* thr_next,
                           int32_t* n_uncertified, void* stream);
/* ---- range search: every corpus row whose exact score reaches a per-row minimum -------------------------------
 * A new capability with no counterpart in the reference, which only ranks whole score rows.  The caller has listed,
 * with xmve_score_filter at lo[r] <= min_score[r] - eps, every row that can reach min_score[r] and rescored the list
 * (xmve_rescore, bound = NULL).  Entry c < min(cand_count[r], cap) of row r matches iff exact[r, c] > -inf,
 * exact[r, c] >= min_score[r] (NaN never matches) and its global row cand_idx + idx_offset differs from exclude[r]
 * (exclude may be NULL).  min_score fp64 [rows], exact fp64 [rows, cap], cand_idx int32 [rows, cap].
 *   count (off == NULL): counts[r] = the number of matches of row r (int64 [rows], written).
 *   fill  (off != NULL): counts is the count mode's result (read); the matches of row r are written, sorted by
 *         (score desc, global row asc), to out_score / out_idx [off[r], off[r] + counts[r]).  off int64 [rows] holds
 *         the start positions, normally the exclusive cumsum of counts (the first rows of a CSR's offsets); any starts
 *         whose ranges do not overlap will do, so a subset of rows can be filled into a larger CSR.  max_len >=
 *         max_r counts[r] sizes the sort.  Rows of up to 16384 matches are sorted in shared memory; longer rows need
 *         scratch (DEVICE, 24 bytes per output entry: row r uses bytes [24 off[r], 24 (off[r] + counts[r]))) and
 *         return XMVE_ERR_LIMIT without it.
 * xmve_range_merge joins the per-shard results: run (s, r) of segment s < n_seg is the sorted entries
 * score / idx [seg_off[s, r], seg_off[s, r + 1]) (seg_off int64 [n_seg, rows + 1], positions into score and idx,
 * which are DEVICE fp64 / int64 with global rows).  Row r's runs are merged, in the same order, into
 * out_score / out_idx [off[r], off[r + 1]) (off int64 [rows + 1]); the runs of a row must hold off[r + 1] - off[r]
 * entries in all and no (score, row) pair twice (shards own disjoint rows).  max_len >= max_r off[r + 1] - off[r]
 * sizes the grid.  Runs are merged by binary search, so runs of any length need no scratch.
 */
XMVE_API int xmve_range_select(const double* exact, const int32_t* cand_idx, const int32_t* cand_count, int64_t rows,
                      int32_t cap, int64_t idx_offset, const int64_t* exclude, const double* min_score,
                      int64_t* counts, const int64_t* off, int64_t max_len, void* scratch,
                      double* out_score, int64_t* out_idx, void* stream);
/* xmve_pair_select is xmve_range_select with one more condition, for the similar-pairs join of a corpus with itself
 * (row r of the lists is the stored row after[r] used as a query): an entry matches only if, in addition, its global
 * row cand_idx + idx_offset is greater than after[r] (after int64 [rows], DEVICE, never NULL).  This drops the row
 * itself and every pair the join lists from the other side.  Count and fill apply the same test; arguments, modes and
 * limits are those of xmve_range_select.  after[r] = -1 gives xmve_range_select's result. */
XMVE_API int xmve_pair_select(const double* exact, const int32_t* cand_idx, const int32_t* cand_count, int64_t rows,
                     int32_t cap, int64_t idx_offset, const int64_t* exclude, const double* min_score,
                     int64_t* counts, const int64_t* off, int64_t max_len, void* scratch,
                     double* out_score, int64_t* out_idx, const int64_t* after, void* stream);
XMVE_API int xmve_range_merge(const double* score, const int64_t* idx, int32_t n_seg, const int64_t* seg_off,
                     int64_t rows, const int64_t* off, int64_t max_len, double* out_score, int64_t* out_idx,
                     void* stream);
/* The j largest values of each row in descending order, -inf padded: out fp32 [rows, j] (j <= 4096).
 * Row r holds min(counts[r], cols) valid values (counts == NULL: cols).  The j-th largest value of a corpus
 * that is sharded over GPUs is the j-th largest of the union of the shards' top-j lists. */
XMVE_API int xmve_row_topj(const float* vals, int64_t rows, int64_t cols, int64_t ld, const int32_t* counts,
                  int32_t j, float* out, void* stream);

/* ---- exact fp64 score matrix (small problems; the cal_error drop-in on float64 inputs) ----------
 * out[q, v] = alpha * <a_q, b_v>, a [nq, a_ld], b [nv, b_ld], out [nq, out_ld], all fp64, k columns.
 * a and b are already normalised (xmve_normalize_f64).  LINAS-engine/evaluation.py:21.
 */
XMVE_API int xmve_normalize_f64(const void* src, int src_dtype, int64_t n, int d, int64_t src_ld,
                       double* dst, int64_t dst_ld, int norm_mode, void* stream);
XMVE_API int xmve_score_f64(const double* a, int64_t nq, int64_t a_ld, const double* b, int64_t nv, int64_t b_ld,
                   int k, double alpha, double* out, int64_t out_ld, void* stream);
/* The same with the multi-space fusion (SURVEY.md section 8a row F) in the epilogue:
 *   first != 0: out = w * (alpha * <a_q, b_v>);   first == 0: out = out + w * (alpha * <a_q, b_v>)
 * every product and sum rounded on its own, i.e. exactly `acc = w * e` / `acc = acc + w * e` of NumPy on the matrix
 * xmve_score_f64 would have written -- without writing and re-reading that matrix.  Needs even row strides and
 * 16-byte aligned operands (the DMMA kernel); XMVE_ERR_ARG otherwise.
 */
XMVE_API int xmve_score_f64_fused(const double* a, int64_t nq, int64_t a_ld, const double* b, int64_t nv, int64_t b_ld,
                         int k, double alpha, double w, int first, double* out, int64_t out_ld, void* stream);

/* ---- non-cosine measures of cal_error (LINAS-engine/evaluation.py:22-35; scipy cdist / loss.jaccard_sim) -------
 * out[q, v] = alpha * f(a_q, b_v) + beta,  f = sum_i |a_i - b_i| (L1), sqrt(sum_i (a_i - b_i)^2) (L2) or
 * sum_i min(a_i, b_i) / sum_i max(a_i, b_i) (JACCARD); a [nq, a_ld], b [nv, b_ld], out [nq, out_ld] fp64, k columns.
 * 'l1' / 'l2' / 'euclidean': alpha = 1, beta = 0; 'l1_norm' / 'l2_norm': alpha = -1/k, beta = -1; 'jaccard': alpha = -1.
 * CUDA-core kernel (ALU-bound); at most 65535 * 64 query rows per call.
 */
enum { XMVE_MEASURE_L1 = 0, XMVE_MEASURE_L2 = 1, XMVE_MEASURE_JACCARD = 2,
       /* the similarity functions of the training loss (LINAS-engine/loss.py:7-73) */
       XMVE_MEASURE_SQL2 = 3,   /* sum_i (a_i - b_i)^2           (euclidean_sim / L2_sim / L2_sim_norm: no root) */
       XMVE_MEASURE_DOT = 4,    /* sum_i a_i * b_i                (cosine_sim on already normalised rows)        */
       XMVE_MEASURE_ORDER = 5   /* sqrt(sum_i max(b_i - a_i, 0)^2) (order_sim)                                  */ };
XMVE_API int xmve_pairwise_f64(const double* a, int64_t nq, int64_t a_ld, const double* b, int64_t nv, int64_t b_ld,
                      int k, int measure, double alpha, double beta, double* out, int64_t out_ld, void* stream);

/* ---- triplet ranking cost of a batch score matrix (LINAS-engine/loss.py:112-153, forward value only) ------------
 * scores fp64 [n, n] = sim(im, s) (xmve_pairwise_f64).  With the diagonal cleared,
 *   out[0] = sum of cost_s  = max(0, margin + scores[i, j] - scores[i, i])  (max_violation: of each ROW's maximum)
 *   out[1] = sum of cost_im = max(0, margin + scores[i, j] - scores[j, j])  (max_violation: of each COLUMN's maximum)
 * out: DEVICE double[2] (zeroed by the call).  loss.py:147-150: 'sum' adds them, 'mean' divides by n*n (or n).
 */
XMVE_API int xmve_triplet_cost(const double* scores, int64_t n, int64_t ld, double margin, int max_violation,
                      double* out, void* stream);

/* ---- K4: bit-exact rank / metric kernels --------------------------------------------------------
 * errors is the caller's [n_row, n_col] matrix (fp32/fp64, smaller = better, as cal_error returns).
 * gt_off[n_query+1], gt_ids[] is a CSR of ground-truth positions per query.
 * axis = 0: query i is ROW i, memories are columns   (eval_q2m(errors, t2v_gt), util/metrics.py:124-157)
 * axis = 1: query i is COLUMN i, memories are rows   (eval_q2m(errors.T, v2t_gt), validate.py:22)
 * ranks[e] (1-based, one per CSR entry) = 1 + #{m : x[m] < x[g]} + #{m < g : x[m] == x[g]}, the
 * position of g in a stable ascending argsort (np.argsort(line, kind="stable")).  As there, NaN sorts after every
 * number, NaNs in index order: a NaN x[g] has rank 1 + #{m : x[m] is not NaN} + #{m < g : x[m] is NaN}, and a NaN
 * element never precedes a number.  -0.0 and +0.0 are equal.  n_entries = gt_off[n_query] and max_gt = the largest
 * number of entries of any query are passed by the caller (it built the CSR) to avoid a device sync.
 */
XMVE_API int xmve_gt_ranks(const void* errors, int dtype, int64_t n_row, int64_t n_col, int64_t ld, int axis,
                  const int64_t* gt_off, const int32_t* gt_ids, int64_t n_query,
                  int64_t n_entries, int32_t max_gt, int32_t* ranks, void* stream);
/* Per-query reduction of the CSR ranks (n_mem = number of memories):
 *   best[i]   = min rank over the query's GT entries, n_mem + 1 if none   (util/metrics.py:140-147)
 *   ap[i]     = APScorer(ap_k).score of the label list with the GT entries relevant: ranks sorted
 *               ascending, ap += j / rank_j in that order, / nr_relevant (basic/metric.py:31-46);
 *               first_only != 0 marks only the FIRST GT entry (t2v_map, util/metrics.py:72-73)
 *   recall_counts[0..2] += #{best <= 1, 5, 10}; rank_sum += best; hist[best] += 1 (hist[n_mem+2])
 * max_gt = the largest number of entries of any query (the caller built the CSR).  Lists of up to 16384 entries are
 * sorted in shared memory; beyond that sort_scratch (int32 [n_entries], DEVICE) is required (XMVE_ERR_LIMIT without it)
 * and the longer lists are sorted there.
 */
XMVE_API int xmve_rank_metrics(const int32_t* ranks, const int64_t* gt_off, int64_t n_query, int64_t n_mem,
                      int first_only, int ap_k, int32_t max_gt, int32_t* sort_scratch,
                      int32_t* best, double* ap, int64_t* recall_counts, int64_t* rank_sum,
                      int32_t* hist, void* stream);

/* Ranks from top-k LISTS instead of a score matrix (corpora whose matrix cannot exist): lists int64 [n_query, len]
 * (row stride ld) are ranked memory ids (np.argsort(errors)[:topK], LINAS-engine/inference.py:79-80); for CSR entry e
 * of query q (off[n_query+1], wanted[n_entries]) rank[e] = 1 + the position of wanted[e] in row q, or `absent` when
 * the list does not hold it.  Feeds xmve_rank_metrics (AP@k of basic/metric.py:31-46, R@K of util/metrics.py:149-151).
 */
XMVE_API int xmve_list_ranks(const int64_t* lists, int64_t n_query, int64_t len, int64_t ld, const int64_t* off,
                    const int64_t* wanted, int64_t n_entries, int32_t absent, int32_t* rank, void* stream);

/* ---- rank of the ground truth when the score matrix cannot exist (util/metrics.py:139-145 at C3-C5 scale) ---------
 * Entry e = (query, ground-truth item g[e]) with the item's exact score s_gt[e].  The tensor-core pass
 * (xmve_score_filter with lo = s_gt - eps, hi = s_gt + eps) counts the rows certainly above and lists the rows inside
 * the guard band; after xmve_rescore of those, xmve_count_before adds
 *   before[e] += #{c < min(counts[e], cap) : exact[e, c] > s_gt[e]  or  (exact[e, c] == s_gt[e] and idx + idx_offset < g[e])}
 * so that rank = 1 + count_above + before is the position of g in a stable ascending argsort of the errors.
 * Shards add their counts (one all-reduce).  xmve_count_band_f64 is the fallback for entries whose band overflowed
 * (very deep ground truths): against a chunk of an exact fp64 score matrix [n_entries, cols] it adds the columns above
 * s_gt + delta to above[e] and lists the columns with |x - s_gt| <= delta (chunk-local numbers) for the same settle step.
 */
XMVE_API int xmve_count_before(const double* exact, const int32_t* idx, const int32_t* counts, int64_t n_entries,
                      int32_t cap, int64_t idx_offset, const double* s_gt, const int64_t* g, int64_t* before,
                      void* stream);
XMVE_API int xmve_count_band_f64(const double* scores, int64_t n_entries, int64_t cols, int64_t ld, int64_t col0,
                        const double* s_gt, double delta, int64_t* above, int32_t* band_count, int32_t* band_idx,
                        int32_t band_cap, void* stream);

/* ---- norm_score (LINAS-engine/validate.py:7-11) -------------------------------------------------
 * minmax[0] = min(-E), minmax[1] = max(-E - min) over the whole matrix (two launches inside);
 * then out = -((-E - min) / max) with the reference's operation order, in the input's precision.  NumPy semantics on
 * non-finite input: a NaN anywhere makes min, max and every output NaN; an infinite min (an error of +inf, or all
 * errors -inf) makes every output NaN; an error of -inf alone makes max = inf, so that element's output is NaN and
 * every other one -0.0; a constant matrix gives 0 / 0 = NaN.  minmax_scratch: DEVICE, 2 doubles.
 */
XMVE_API int xmve_norm_score(const void* errors, int dtype, int64_t n_row, int64_t n_col, int64_t ld,
                    void* out, int64_t out_ld, double* minmax_scratch, void* stream);

/* ---- multi-space fusion of score matrices (SURVEY.md section 8a row F) ---------------------------------
 * acc = w * e (first != 0) or acc = acc + w * e, element-wise on [n_row, n_col] matrices of `dtype`, every
 * multiplication and addition rounded on its own (what NumPy's `acc + w * e` does; no fused multiply-add), w
 * rounded to `dtype` first.  Composes `errors = sum_s w_s * cal_error_s` and `sum_s w_s * norm_score(cal_error_s)`.
 */
XMVE_API int xmve_fuse_accumulate(void* acc, int64_t acc_ld, const void* e, int64_t e_ld, int dtype,
                         int64_t n_row, int64_t n_col, double w, int first, void* stream);

#ifdef __cplusplus
}
#endif
#endif  /* XMVE_H_ */
