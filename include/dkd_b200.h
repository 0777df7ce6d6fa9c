/*
 * dkd_b200.h — C ABI of the B200-native DL-DKD++ corpus retrieval scoring path.
 *
 * The reference (HuiGuanLab/DL-DKD) has no FFI: its seam for this path is plain Python
 * (bound methods of DLDKD(nn.Module), method/model.py, and module functions of
 * method/eval.py).  Each entry point below names the reference interface (file:line under
 * /root/reference) whose arithmetic it replaces; INTEGRATION.md shows the ctypes stub a
 * maintainer adds on the reference side.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in `_host`;
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream);
 *   - no allocation, no host synchronisation, no global state inside any call;
 *   - return value: 0 = ok, <0 = DKD_ERR_* (bad argument), >0 = cudaError_t;
 *   - dense score matrices are query-major: element (m, n) at out[m * ld + n];
 *   - "rows per video" R: the scoring kernels see the corpus as Nv * R rows of D
 *     features; R = L (frames, reference path) or R = P = T(T+1)/2 (clip proposals).
 *
 * All arithmetic types: fp32 scores, int32 indices, bf16 (uint16_t storage) GEMM operands, fp16 (uint16_t
 * storage) operands of the approximate frame-scale gather.
 */
#ifndef DKD_B200_H_
#define DKD_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DKD_OK 0
#define DKD_ERR_ARG (-1)       /* null pointer / non-positive size */
#define DKD_ERR_SHAPE (-2)     /* unsupported shape (D % 64, T > 32, K > 256, ...) */
#define DKD_ERR_ALIGN (-3)     /* pointer or leading dimension not aligned as required */
#define DKD_ERR_DRIVER (-4)    /* cuTensorMapEncodeTiled unavailable */
#define DKD_ERR_WORKSPACE (-5) /* workspace too small */

#define DKD_MASKED_SCORE (-1e10f) /* method/model.py:444-445 mask_logits fill value */

int dkd_version(void);
const char* dkd_error_string(int code);

/* ---------------------------------------------------------------------------------------
 * Row preparation: L2-normalise every D-vector (x / max(||x||, eps)), write fp32 and/or bf16 and/or fp16.
 * Replaces F.normalize(modularied_query) / F.normalize(context_feat), method/model.py:318-319
 * (hoisted out of the per-query-batch loop of method/eval.py:188-208).
 * rows_out_pad >= rows: extra output rows are zero-filled (GEMM M padding). Any output may be NULL
 * (bf16: GEMM operands; fp16: operands of the frame-scale gather).
 */
int dkd_normalize_rows(const float* x, int64_t rows, int32_t D, float eps, float* out_f32,
                       uint16_t* out_bf16, uint16_t* out_f16, int64_t rows_out_pad, void* stream);

/* ---------------------------------------------------------------------------------------
 * Clip downsample: encoded frames (Nv, L, D) + valid lengths -> (Nv, T, D) clip features with
 * the arithmetic of average_to_fixed_length, method/data_provider.py:30-50.
 */
int dkd_downsample_clips(const float* frames, const int32_t* lengths, int32_t Nv, int32_t L,
                         int32_t D, int32_t T, float* clips, void* stream);

/* ---------------------------------------------------------------------------------------
 * Clip-proposal builder (north_star "prefix-sum kernel"; SURVEY §8 N2): for every video the
 * P = T(T+1)/2 sliding-window means, ordered by window length w = 1..T then start s,
 *   p(w, s) = (w-1)*T - (w-1)(w-2)/2 + s,   prop[p] = mean(clips[s : s+w]).
 * Outputs (any may be NULL):
 *   prop_bf16   (Nv, P, D)  L2-normalised proposals, bf16 — B operand of the clip-scale GEMM;
 *   prop_scale  (Nv, P)     1 / (w * max(||mean||, 1e-12)) — turns a window SUM of per-clip dot
 *                           products into the cosine (exact fp32 path);
 *   prop_f32    (Nv, P, D)  un-normalised fp32 means (tests / small shapes only).
 * Requires T <= 32, D % 64 == 0, D <= 512.
 */
int dkd_build_proposals(const float* clips, int32_t Nv, int32_t T, int32_t D,
                        uint16_t* prop_bf16, float* prop_scale, float* prop_f32, void* stream);

/* ---------------------------------------------------------------------------------------
 * Exact fp32 scoring (SIMT).  Replaces DLDKD.get_sim_scores, method/model.py:307-329, with the
 * corpus normalisation hoisted:
 *   out_max[m, n] = max_r  qn[m] . xn[n, r]   (masked rows score exactly -1e10, mask_logits :444)
 *   out_arg[m, n] = first r attaining the max (torch.max tie rule)
 * qn (M, D) and xn (Nv, R, D) are L2-normalised fp32; mask (Nv, R) uint8 or NULL; R <= 128.
 * out_rows (optional) is the reference's second return value laid out (M, R, Nv).
 * q_list / vid_ptr (optional, both or neither): CSR restriction — for video n only queries
 * q_list[vid_ptr[n] .. vid_ptr[n+1]) are scored and results go to out_max[e] / out_arg[e]
 * (entry order) instead of the dense matrix.
 */
int dkd_score_max_f32(const float* qn, int32_t M, const float* xn, int32_t Nv, int32_t R,
                      int32_t D, const uint8_t* mask, float* out_max, int32_t* out_arg,
                      int64_t ld_out, float* out_rows, const int32_t* vid_ptr,
                      const int32_t* q_list, void* stream);

/* ---------------------------------------------------------------------------------------
 * Exact (fp32-grade) scoring on the tcgen05 tensor cores: kind::tf32 with operands split on the fly
 * (x = hi + lo; lo.hi + hi.lo + hi.hi, fp32 accumulate in TMEM — error inside the summation-order noise of an
 * fp32 einsum).  The corpus-side operand is pre-packed once per corpus into the shared-memory image of the
 * MMA's B operand (tf32 hi / lo planes, K-major 128-byte swizzle):
 *   dkd_pack_rows_tf32  xn (Nv, R, D) normalised rows, R <= 128   -> dkd_row_planes_bytes(Nv, R, D) bytes
 *   dkd_pack_clips_tf32 clips (Nv, T, D), T <= 32                  -> dkd_clip_planes_bytes(Nv, D) bytes
 *
 * dkd_score_max_exact: same results and options as dkd_score_max_f32 (max / first argmax over the R rows of a
 * video, masked rows exactly -1e10, dense or CSR) without the per-row output; replaces DLDKD.get_sim_scores,
 * method/model.py:307-329.  D % 32 == 0, D <= 512.
 *
 * dkd_clip_score_f32: clip-scale scores through per-clip dot products (SURVEY §7 "linearity"):
 *   d[m, n, i] = qn[m] . clips[n, i];  S[m, n, p(w,s)] = (sum_{i=s}^{s+w-1} d[m,n,i]) * prop_scale[n, p]
 *   out_max = max_p S, out_arg = first argmax_p.  T <= 32, D % 32 == 0, D <= 512, 16-byte aligned rows.
 * Same CSR option (vid_cnt, optional: video n owns vid_cnt[n] entries from vid_ptr[n] instead of the CSR run
 * vid_ptr[n] .. vid_ptr[n+1]); with out_slot (list form only) entry e is written to out_max[out_slot[e]] /
 * out_arg[out_slot[e]] (scatter into a dense matrix) instead of out_max[e].
 * known_key (list form, T = 32, optional): dense (M, known_ld) key clips already fixed by the approximate pass (entry
 * (q, n) reads known_key[q * known_ld + n]); the kernel confirms the key against the exact maximum at a third of the
 * full scan's cost and falls back to the full first-argmax search for any entry whose key is not the maximum — the
 * results are those of the call without known_key.
 * Replaces get_clip_scale_scores of the two-scale head (SURVEY §8 N3), fp32 reference flavour.
 */
int64_t dkd_row_planes_bytes(int32_t Nv, int32_t R, int32_t D);
int dkd_pack_rows_tf32(const float* xn, int32_t Nv, int32_t R, int32_t D, float* planes, void* stream);
int dkd_score_max_exact(const float* qn, int32_t M, const float* row_planes, int32_t Nv, int32_t R,
                        int32_t D, const uint8_t* mask, float* out_max, int32_t* out_arg, int64_t ld_out,
                        const int32_t* vid_ptr, const int32_t* q_list, void* stream);
int64_t dkd_clip_planes_bytes(int32_t Nv, int32_t D);
int dkd_pack_clips_tf32(const float* clips, int32_t Nv, int32_t T, int32_t D, float* planes, void* stream);
int dkd_clip_score_f32(const float* qn, int32_t M, const float* clip_planes, const float* prop_scale,
                       int32_t Nv, int32_t T, int32_t D, float* out_max, int32_t* out_arg,
                       int64_t ld_out, const int32_t* vid_ptr, const int32_t* vid_cnt,
                       const int32_t* q_list, const int32_t* out_slot, const int32_t* known_key,
                       int64_t known_ld, void* stream);

/* ---------------------------------------------------------------------------------------
 * bf16 tcgen05/TMEM scoring GEMM with fused max/argmax epilogue (the hot kernel).
 *   q_bf16 (Mpad, D) normalised queries, Mpad % 128 == 0, rows >= M zero;
 *   x_bf16 (Nv * R, D) normalised corpus rows; R % 16 == 0, D % 64 == 0, D <= 512;
 *   mask   (Nv, R) uint8 (non-zero = valid, method/model.py:444-445) or NULL; 16-byte aligned (DKD_ERR_ALIGN
 *          otherwise): the kernel reads it 16 columns at a time.  A video with no valid row scores exactly
 *          DKD_MASKED_SCORE with argmax 0 (torch.max: first index).
 * Outputs as dkd_score_max_f32 (dense only), except for the tie rule below.  Replaces method/model.py:318-327 (R = L) and the
 * clip-scale contraction of SURVEY §8 N3 (R = P = 528).  Videos of R <= 128 rows (the reference's frame head) are
 * scored two per N = 2 R MMA tile on CTA pairs.
 * TMA descriptors are encoded on the host per call (cuTensorMapEncodeTiled fetched through
 * cudaGetDriverEntryPoint) and passed as kernel parameters: no workspace.
 * out_gap (optional): best score minus the runner-up score of the same (query, video) — pairs whose
 * gap is below the bf16 noise floor have an ambiguous argmax and are re-resolved in fp32
 * (dkd_select_pairs_csr -> dkd_clip_score_f32 (CSR, out_slot)).  Scores carry the column
 * position in their 4 low mantissa bits inside the kernel: returned values are exact to 8 ulp.
 * Tie rule (narrower than torch.max): rows whose scores are equal above those 4 bits are tied, and out_arg is one of
 * them, which one is unspecified (for a negative score or across 16-row chunks it need not be the first).  Such a pair
 * always has gap 0 (a fully masked video: gap <= 0), so any tau > 0 flags it for the exact kernels, which return
 * the first argmax.
 * out_flags (optional, caller-zeroed, (M, ceil(Nv/32)) uint32): bit (n & 31) of word [m][n >> 5] is set when
 * that gap is below tau — the compact form consumed by dkd_select_flagged (no dense gap round trip).
 */
int dkd_score_max_bf16(const uint16_t* q_bf16, int32_t M, int32_t Mpad, const uint16_t* x_bf16,
                       int32_t Nv, int32_t R, int32_t D, const uint8_t* mask, float* out_max,
                       int32_t* out_arg, float* out_gap, int64_t ld_out, uint32_t* out_flags, float tau,
                       void* stream);

/* The same kernel on IEEE-half operands (kind::f16 with the f16 formats: same tensor rate and bytes as bf16, 11
 * instead of 8 significant bits — operand rounding error 8 x smaller; values are L2-normalised, so the narrower
 * exponent range costs nothing).  A reported variant (DESIGN.md): north_star specifies bf16, which stays the default. */
int dkd_score_max_f16(const uint16_t* q_f16, int32_t M, int32_t Mpad, const uint16_t* x_f16,
                      int32_t Nv, int32_t R, int32_t D, const uint8_t* mask, float* out_max,
                      int32_t* out_arg, float* out_gap, int64_t ld_out, uint32_t* out_flags, float tau,
                      void* stream);
/* dkd_build_proposals with IEEE-half rows (B operand of dkd_score_max_f16). */
int dkd_build_proposals_f16(const float* clips, int32_t Nv, int32_t T, int32_t D, uint16_t* prop_f16,
                            float* prop_scale, void* stream);

/* The same GEMM with the ambiguous-pair lists written straight from its epilogue (one atomic per flagged pair; no bit
 * matrix and no selection pass): flag_cnt (Nv, caller-zeroed) = number of pairs of each video whose gap is below tau,
 * flag_list = their query indices, video n at [n * flag_cap, n * flag_cap + flag_cnt[n]) in any order (flag_cap >= M
 * rules out overflow; entries beyond flag_cap are dropped).  f16_operands: IEEE-half instead of bf16 operands.
 * dkd_clip_score_list consumes the lists: exact clip score / key clip of every listed pair (arithmetic of
 * dkd_clip_score_f32) scattered into the dense matrices at (query, video). */
int dkd_score_max_bf16_lists(const uint16_t* q, int32_t M, int32_t Mpad, const uint16_t* x, int32_t Nv, int32_t R,
                             int32_t D, const uint8_t* mask, float* out_max, int32_t* out_arg, int64_t ld_out,
                             float tau, int32_t* flag_cnt, int32_t* flag_list, int64_t flag_cap,
                             int32_t f16_operands, void* stream);
int dkd_clip_score_list(const float* qn, int32_t M, const float* clip_planes, const float* prop_scale, int32_t Nv,
                        int32_t T, int32_t D, float* out_max, int32_t* out_arg, int64_t ld_out,
                        const int32_t* vid_cnt, const int32_t* q_list, int64_t list_stride, void* stream);

/* Per-video lists of the flagged pairs of a dkd_score_max_bf16 bit matrix: video n owns entries
 * [vid_begin[n], vid_begin[n] + vid_cnt[n]) of q_list (query index) / slot (m * ld + n), in any order; runs
 * are placed by a global cursor (1 int scratch).  One pass over the bit matrix, one block per 32 videos. */
int dkd_select_flagged(const uint32_t* flags, int32_t M, int32_t Nv, int64_t ld, int64_t cap, int32_t* cursor,
                       int32_t* vid_begin, int32_t* vid_cnt, int32_t* q_list, int32_t* slot, void* stream);

/* Ambiguous-pair bookkeeping: CSR (by video) of all pairs (m, n) with gap[m, n] < tau.
 * counts (Nv) scratch; vid_ptr (Nv+1); q_list / slot (cap entries; slot = m * ld + n).  Entries beyond
 * `cap` are dropped (size cap = M * Nv to make that impossible). */
int dkd_select_pairs_csr(const float* gap, int32_t M, int32_t Nv, int64_t ld, float tau, int64_t cap,
                         int32_t* counts, int32_t* vid_ptr, int32_t* q_list, int32_t* slot, void* stream);

/* ---------------------------------------------------------------------------------------
 * Key-clip-guided frame attention, query-independent table form (SURVEY §8 N4, §7):
 *   E[n, l, i]      = key[n, l] . clips[n, i]                       (dkd_key_clip_dots)
 *   logit[n, p, l]  = (sum_{i in window p} E[n, l, i]) / w
 *   a               = softmax over valid frames l < lengths[n]
 *   g[n, p]         = sum_l a_l * val[n, l];   table = g / max(||g||, 1e-12)
 * key/val (Nv, L, D) fp32 are the W_k / W_v projections of the encoded frames.
 * Outputs (either may be NULL): table_f32, table_f16 (Nv, P, D; IEEE half). L <= 128, T <= 32, D % 64 == 0,
 * D <= 512.  E is a caller-provided scratch of Nv*L*T floats.
 */
int dkd_key_clip_dots(const float* key, const float* clips, int32_t Nv, int32_t L, int32_t T,
                      int32_t D, float* E, void* stream);
int dkd_frame_attn_table(const float* E, const float* val, const int32_t* lengths, int32_t Nv,
                         int32_t L, int32_t T, int32_t D, float* table_f32, uint16_t* table_f16,
                         void* stream);

/* Frame-scale score + branch fusion (SURVEY §8 N5; cross-branch weights method/eval.py:254):
 *   frame[m, n]  = q[m] . table[n, key_clip[m, n]]
 *   branch[m, n] = fl(w_clip * clip[m, n]) + fl(w_frame * frame[m, n])
 *   fused[m, n]  = accumulate ? fused[m, n] + fl(w_branch * branch) : fl(w_branch * branch)
 * q/table both fp32 (is_f16 = 0: exact path) or both fp16 (is_f16 = 1: half2 FMA in chunks of 4 products,
 * fp32 accumulation across chunks; D % 64 == 0).  out_frame / fused may be NULL.
 */
int dkd_frame_fuse(const void* q, const void* table, int32_t is_f16, const float* clip_scores,
                   const int32_t* key_clip, int32_t M, int32_t Nv, int32_t P, int32_t D,
                   int64_t ld, float w_clip, float w_frame, float w_branch, int32_t accumulate,
                   float* out_frame, float* fused, void* stream);

/* fused = fl(wa * a) + fl(wb * b), elementwise, numpy rounding order of method/eval.py:254. */
int dkd_fuse_scores(const float* a, const float* b, float wa, float wb, float* out, int64_t n,
                    void* stream);

/* ---------------------------------------------------------------------------------------
 * Ranking.  dkd_topk: per query the K best (score desc, video id asc on equal scores) of a
 * dense (M, Nv) matrix; ids are offset by id_base (global ids of a corpus shard). K <= 256.
 * Replaces the np.argsort of eval_q2m, method/eval.py:75 (only the top-100 matter for R@K).
 */
int dkd_topk(const float* scores, int32_t M, int32_t Nv, int64_t ld, int32_t K, int32_t id_base,
             float* out_scores, int32_t* out_ids, void* stream);

/* Top-K SELECTION without ordering (radix select on the score key, one warp per row): out_ids (M, K) = the ids of the K
 * best entries of every row in column order (same order rule: ties at the K-th score go to the lower ids), padded with
 * -1 when Nv < K; out_kth (M) = the K-th best score (-inf when Nv <= K).  For the candidate pass of the ranking, which
 * rescored and sorts its candidates afterwards and needs only their set and the K-th approximate score. */
int dkd_select_topk(const float* scores, int32_t M, int32_t Nv, int64_t ld, int32_t K, int32_t id_base,
                    int32_t* out_ids, float* out_kth, void* stream);

/* Merge G per-shard top-K lists (G, M, K) (e.g. after an NCCL all-gather) into one (M, K). */
int dkd_merge_topk(const float* scores, const int32_t* ids, int32_t G, int32_t M, int32_t K,
                   float* out_scores, int32_t* out_ids, void* stream);
/* dkd_merge_topk with a payload: every entry carries C <= 8 opaque 32-bit words, payload (G, M, K, C); out_scores /
 * out_ids are bit-identical to dkd_merge_topk's, and out_payload (M, K, C) row j holds the words of the entry ranked j.
 * Output ranks without an entry (id -1) are not written: the caller pre-fills them.  Precondition: within one query
 * the ids of the G lists are distinct (disjoint shards, or the running list and a chunk of new videos), so every
 * (score, id) key is unique.  Carries the per-hit detail of a ranking (key clip, branch scores) through the shard and
 * chunk merges that replace the np.argsort of eval_q2m, method/eval.py:75. */
int dkd_merge_topk_payload(const float* scores, const int32_t* ids, const uint32_t* payload, int32_t G, int32_t M,
                           int32_t K, int32_t C, float* out_scores, int32_t* out_ids, uint32_t* out_payload,
                           void* stream);

/* Rank of the best ground-truth video per query (1-based), eval_q2m method/eval.py:73-82:
 * rank = 1 + #{n : s[n] > s[gt]} + #{n < gt : s[n] == s[gt]}, min over the query's GT list
 * (CSR gt_ptr / gt_ids).  Dense scores. */
int dkd_rank_of_gt(const float* scores, int32_t M, int32_t Nv, int64_t ld, const int32_t* gt_ptr,
                   const int32_t* gt_ids, int32_t* out_rank, void* stream);

/* Candidate bookkeeping for exact rescoring: invert (M, K) candidate ids into a per-video CSR.
 * Candidate ids are global (id_base + local video index); ids outside the shard are skipped.
 * counts (Nv) scratch; vid_ptr (Nv+1), q_list (M*K), slot (M*K) outputs. */
int dkd_candidates_to_csr(const int32_t* cand_ids, int32_t M, int32_t K, int32_t Nv,
                          int32_t id_base, int32_t* counts, int32_t* vid_ptr, int32_t* q_list,
                          int32_t* slot, void* stream);
/* Per-CSR-entry frame score + fusion (exact rescoring of candidates), then scatter to (M, K).
 * clip_scores / key_clip: per-entry arrays (dense_ld = 0), or dense (M, ld) matrices read at (q_list[e], video)
 * (dense_ld = ld >= Nv) when the exact clip scores of every pair already exist. */
int dkd_frame_fuse_csr(const float* q, const float* table, const float* clip_scores,
                       const int32_t* key_clip, const int32_t* vid_ptr, const int32_t* q_list,
                       const int32_t* slot, int32_t Nv, int32_t P, int32_t D, float w_clip,
                       float w_frame, float w_branch, int32_t accumulate, float* cand_scores,
                       int64_t dense_ld, void* stream);
/* dkd_frame_fuse_csr plus the per-hit detail of this branch: the same kernel writes cand_scores exactly as
 * dkd_frame_fuse_csr does and, at payload[slot[e] * C + c0 ..], three words: the key clip used (int32, clamped to
 * [0, P)), the clip-scale score and the frame-scale score (fp32 bits) that the fused score was computed from
 * (fuse_branch order: branch = fl(w_clip * clip) + fl(w_frame * frame), times w_branch).  c0 + 3 <= C.
 * Serves the moment behind each hit of the two-scale ranking (key clip of SURVEY §8 N3, frame score of N5). */
int dkd_frame_fuse_csr_detail(const float* q, const float* table, const float* clip_scores,
                              const int32_t* key_clip, const int32_t* vid_ptr, const int32_t* q_list,
                              const int32_t* slot, int32_t Nv, int32_t P, int32_t D, float w_clip,
                              float w_frame, float w_branch, int32_t accumulate, float* cand_scores,
                              int64_t dense_ld, uint32_t* payload, int32_t C, int32_t c0, void* stream);
/* Per-CSR-entry fusion + scatter (reference frame path rescoring): out[slot[e]] =
 * fl(wa*a[e]) + fl(wb*b[e]) for e < vid_ptr[Nv] (b == NULL: plain scatter of a). */
int dkd_scatter_fuse(const float* a, const float* b, float wa, float wb, const int32_t* slot,
                     const int32_t* vid_ptr, int32_t Nv, int64_t max_entries, float* out, void* stream);
/* dkd_scatter_fuse plus the per-hit detail of the frame head: out as dkd_scatter_fuse, and payload[slot[e] * C ..] =
 * (arg_a[e], bits of a[e]) and, when b is given, (arg_b[e], bits of b[e]): each branch's best frame (the first argmax of
 * dkd_score_max_exact / dkd_score_max_f32 in CSR form) and its max-over-frames cosine, get_sim_scores of
 * method/model.py:307-329.  arg_b and b both given or both NULL; C >= 4 with b, C >= 2 without. */
int dkd_scatter_fuse_detail(const float* a, const float* b, float wa, float wb, const int32_t* arg_a,
                            const int32_t* arg_b, const int32_t* slot, const int32_t* vid_ptr, int32_t Nv,
                            int64_t max_entries, float* out, uint32_t* payload, int32_t C, void* stream);
/* Sort each query's K candidates (score desc, id asc) and keep the first K_out. */
int dkd_sort_candidates(const float* cand_scores, const int32_t* cand_ids, int32_t M, int32_t K,
                        int32_t K_out, float* out_scores, int32_t* out_ids, void* stream);
/* dkd_sort_candidates with a payload of C <= 8 opaque 32-bit words per candidate, payload (M, K, C): out_scores /
 * out_ids are bit-identical to dkd_sort_candidates's, out_payload (M, K_out, C) row j holds the words of the candidate
 * ranked j.  Output ranks without a candidate are not written (the caller pre-fills them).  Precondition: the valid
 * ids of one query's candidates are distinct (dkd_select_topk gives distinct ids), so every key is unique. */
int dkd_sort_candidates_payload(const float* cand_scores, const int32_t* cand_ids, const uint32_t* payload,
                                int32_t M, int32_t K, int32_t K_out, int32_t C, float* out_scores, int32_t* out_ids,
                                uint32_t* out_payload, void* stream);

/* ---------------------------------------------------------------------------------------
 * Training-step similarity (BASELINE.json configs[4]; SURVEY §8f #2).  Replaces, inside DLDKD.forward
 * (method/model.py:109-157), the back-to-back get_sim_scores (:307-329) / get_unnormalized_sim_scores (:331-350)
 * calls on the same operands and the column gather of compute_kl_loss (:184-188), forward and backward.
 *
 * dkd_row_inv_norms: out[r] = 1 / max(||x_r||, eps) — the denominator of F.normalize (:318-319).
 *
 * dkd_train_sim_fwd: q (M, D) raw queries, x (N, L, D) raw frames, rq (M) / rx (N*L) their inverse norms,
 *   mask (N, L) uint8 or NULL, labels (M) positive video of each query (needed for curve).  One pass of fp32 dots:
 *     max_n[m, n] = max_l cos(q_m, x_nl), arg_n = first argmax      (masked frames score exactly -1e10)
 *     max_u[m, n] = max_l q_m . x_nl,     arg_u = first argmax
 *     curve[m, l] = cos(q_m, x_{labels[m], l})  (masked: -1e10) — rows[m, :, labels[m]] of the reference
 *   Any output may be NULL.  L <= 128, D % 32 == 0, 16-byte aligned q / x.
 *
 * dkd_train_sim_bwd: gradients of a scalar loss with respect to q and x given the upstream gradients of max_n,
 *   max_u (M, N) and curve (M, L) (any may be NULL): the max routes to its argmax frame, masked frames get none,
 *   cos differentiates through both norms.  grad_q (M, D) / grad_x (N, L, D) are overwritten (either may be
 *   NULL).  Deterministic (no atomics).  D <= 512.
 *
 * dkd_kl_curve_loss: loss[m] = KL(softmax(target[m, :len] / temp) || softmax(pred[m, :len] / temp)), len = lens[m]
 *   (F.kl_div(..., reduction='sum') per query, method/model.py:190-195), dpred = d loss[m] / d pred[m, l]
 *   (zero beyond len).  L <= 128.
 */
int dkd_row_inv_norms(const float* x, int64_t rows, int32_t D, float eps, float* out, void* stream);
/* The positive video's frame curve alone, from L2-normalised operands (the tensor-core forward: the two maxima come
 * from dkd_score_max_exact on the normalised / the raw operands, tcgen05 kind::tf32 x 3, and only this gather of
 * M * L dot products — rows[m, :, labels[m]] of method/model.py:184-188 — stays a SIMT kernel). */
int dkd_train_curve(const float* qn, const float* xn, const uint8_t* mask, const int32_t* labels, int32_t M, int32_t L,
                    int32_t D, float* curve, void* stream);
int dkd_train_sim_fwd(const float* q, const float* x, const float* rq, const float* rx, const uint8_t* mask,
                      const int32_t* labels, int32_t M, int32_t N, int32_t L, int32_t D, float* max_n,
                      int32_t* arg_n, float* max_u, int32_t* arg_u, float* curve, void* stream);
int dkd_train_sim_bwd(const float* q, const float* x, const float* rq, const float* rx, const uint8_t* mask,
                      const int32_t* labels, int32_t M, int32_t N, int32_t L, int32_t D, const float* max_n,
                      const int32_t* arg_n, const int32_t* arg_u, const float* curve, const float* g_max_n,
                      const float* g_max_u, const float* g_curve, float* grad_q, float* grad_x, void* stream);
int dkd_kl_curve_loss(const float* pred, const float* target, const int32_t* lens, int32_t M, int32_t L,
                      float temp, float* loss, float* dpred, void* stream);

/* Fused triplet + NCE losses of one branch on the (M, N) in-batch score matrices, value and gradient together.
 * Replaces get_clip_triplet_loss (method/model.py:352-388) on s_n (cosine maxima) and clip_nce / clip_nce_soft
 * (method/model_components.py:106-233, reduction 'mean') on s_u (raw maxima):
 *   labels (M)      positive video of each query;
 *   t2v_draw (M)    position (>= 1) in the descending order of the query's row with the positive first — the
 *                   torch.randint(1, max_idx) draw of :376-380 (1 = hardest negative);
 *   v2t_pick (N)    rank (>= 0) among the video's negative queries, descending — 0 = hardest (:363-364), or the
 *                   torch.randint(0, n_neg) draw of :366-368;
 *   soft = 1        clip_nce_soft with soft targets from `sims` (teacher maxima, or s_u itself for the
 *                   self-distilled exploration branch: the gradient through the targets is then included);
 *   soft = 0        clip_nce (sims ignored).
 * out_terms[0] = triplet loss, out_terms[1] = NCE loss (unweighted); g_n / g_u (M, N) = d out_terms[0] / d s_n and
 * d out_terms[1] / d s_u.  workspace: dkd_train_losses_workspace_floats(M, N) floats.  Deterministic.
 * N <= 2048, M <= 8192.
 */
int64_t dkd_train_losses_workspace_floats(int32_t M, int32_t N);
int dkd_train_losses(const float* s_n, const float* s_u, const float* sims, const int32_t* labels,
                     const int32_t* t2v_draw, const int32_t* v2t_pick, int32_t M, int32_t N, float margin,
                     int32_t soft, float alpha, float belta, float* out_terms, float* g_n, float* g_u,
                     float* workspace, void* stream);

/* ---------------------------------------------------------------------------------------
 * Corpus-side encoder (SURVEY section 8 f1).  Replaces, inside DLDKD.encode_context -> encode_input
 * (method/model.py:215-243), the arithmetic of LinearLayer (LayerNorm -> Linear -> ReLU, method/model_components.py:294-312),
 * TrainablePositionalEncoding (:269-291), BertAttention (:339-436: query / key / value / dense linears, 4-head attention
 * with the additive -10000 key mask of :420-422, post-LayerNorm residual) and out_mapping_linear; also the W_k / W_v
 * projections of the key-clip attention.  fp32-grade throughout: the linears run on tcgen05 kind::tf32 with both
 * operands split hi + lo (3 products, fp32 TMEM accumulation — the pipeline of dkd_score_max_exact).
 *
 * dkd_pack_weight_tf32: w (N, K) row-major (nn.Linear.weight) -> the shared-memory image of the MMA's B operand,
 *   128-row tiles, tf32 hi / lo planes (dkd_weight_planes_bytes(N, K) bytes; once per model).  K % 32 == 0.
 * dkd_linear_exact: out[m, n] = act(sum_k xh[m, k] * w[n, k] + bias[n]),  xh = x * scale_m + shift_m when
 *   row_scale_shift ((M, 2): dkd_row_stats) is given — the LayerNorm in front of the projection applied on the fly
 *   (its gamma / beta are folded into w / bias by the caller) — else xh = x.  relu: act = max(., 0).
 *   x (M, K) fp32, out (M, ld_out) fp32, N % 4 == 0, ld_out % 4 == 0, 16-byte aligned pointers.
 * dkd_row_stats: (scale, shift) = (rstd, -mean * rstd) of every row, rstd = 1 / sqrt(var + eps) (biased variance).
 * dkd_layernorm_rows: out = LayerNorm(x [+ pos[row % L]] [+ residual]) * gamma + beta over D <= 512; x / residual are
 *   column blocks of wider matrices (row strides x_ld / res_ld), out is dense (rows, D).
 * dkd_mha_small: per (video, head) softmax(q k^T * scale + (1 - mask) * -10000) v for L <= 128 frames; q / k / v are
 *   column blocks of one (Nv * L, ld) matrix (a fused QKV projection) at q_off / k_off / v_off + head * dh,
 *   dh in {16, 32, 64, 96, 128}; mask (Nv, L) uint8 or NULL; out (Nv * L, out_ld) at column head * dh.
 */
int64_t dkd_weight_planes_bytes(int32_t N, int32_t K);
int dkd_pack_weight_tf32(const float* w, int32_t N, int32_t K, float* planes, void* stream);
int dkd_linear_exact(const float* x, int64_t M, int32_t K, const float* w_planes, int32_t N, const float* bias,
                     int32_t relu, const float* row_scale_shift, float* out, int64_t ld_out, void* stream);
int dkd_row_stats(const float* x, int64_t rows, int32_t D, float eps, float* scale_shift, void* stream);
int dkd_layernorm_rows(const float* x, int64_t x_ld, int64_t rows, int32_t D, const float* gamma, const float* beta,
                       float eps, const float* residual, int64_t res_ld, const float* pos, int32_t L, float* out,
                       void* stream);
int dkd_mha_small(const float* qkv, int64_t ld, int32_t q_off, int32_t k_off, int32_t v_off, const uint8_t* mask,
                  int32_t Nv, int32_t L, int32_t heads, int32_t dh, float scale, float* out, int64_t out_ld,
                  void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DKD_B200_H_ */
