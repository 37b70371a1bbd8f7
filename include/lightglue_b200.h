/*
 * lightglue_b200.h -- C ABI of the B200-native LightGlue matcher hot path.
 *
 * The reference (ipastore/glue-factory-colon) has NO native boundary: every op
 * of gluefactory/models/matchers/lightglue.py is a PyTorch library call.  Each
 * entry point below replaces the library call sites of one kernel family; the
 * reference file:line it replaces is cited per function (paths relative to the
 * reference checkout).  The Python host mirror glue_factory_colon_b200/lightglue.py
 * calls the kernel entry points (ctypes; see INTEGRATION.md); a native caller can
 * run the whole matcher with lgb200_pack_weights + lgb200_match ("whole matcher",
 * at the end; tools/native_match_demo.cpp uses nothing but this header).
 *
 * Conventions
 *   - All pointers are DEVICE pointers unless stated otherwise.  No entry point
 *     allocates, synchronises or keeps mutable global state; every launch goes
 *     to the `stream` argument (a cudaStream_t passed as void*).
 *   - Return value: 0 on success; LGB200_ERR_* (negative) for bad arguments;
 *     a positive value is a cudaError_t from the launch.
 *   - Token storage ("sequence-major"): S = 2*B sequences, sequence s = 2*b+i
 *     is image i of pair b; every sequence owns Lp rows (Lp % 128 == 0) of
 *     which the first lens[s] are valid.  `lens` is a DEVICE int32[S] so that
 *     point pruning can shrink it without a host round trip; a sequence with
 *     lens[s] == 0 is skipped by every kernel (used for early-exited pairs).
 *   - precision: LGB200_F32 runs hand-written CUDA-core fp32 kernels (the
 *     parity mode, 1e-3 on log_assignment); LGB200_BF16 runs tcgen05/TMEM/TMA
 *     kernels with bf16 operands and fp32 accumulation (the throughput mode);
 *     LGB200_F32X3 is the fp32-accurate mode ON the tensor cores: every MMA
 *     operand is a pair of fp16 planes [2][rows][K] (x = hi + lo, 22 mantissa
 *     bits), every product is three tcgen05 MMAs with fp32 accumulation,
 *     softmax / LayerNorm / GELU(erf) / residuals stay in fp32 (lg_x3*.cu).
 *     In that mode the operand pointers of lgb200_linear (A0, A1, W, out16,
 *     outp0..2) and of lgb200_attention (Q, K, V, ctx) are split planes.
 */
#ifndef LIGHTGLUE_B200_H_
#define LIGHTGLUE_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LGB200_ABI_VERSION 8

enum { LGB200_F32 = 0, LGB200_BF16 = 1, LGB200_F32X3 = 2 };

enum {
  LGB200_OK = 0,
  LGB200_ERR_SHAPE = -1,     /* unsupported extent / alignment            */
  LGB200_ERR_NULL = -2,      /* required pointer missing                  */
  LGB200_ERR_PRECISION = -3, /* unknown precision / epilogue enum         */
  LGB200_ERR_DRIVER = -4,    /* cuTensorMapEncodeTiled unavailable/failed */
  LGB200_ERR_ARCH = -5,      /* device is not sm_100                      */
  LGB200_ERR_WEIGHTS = -6    /* required weight missing (lgb200_pack_weights) */
};

/* epilogues of lgb200_linear */
enum {
  LGB200_EPI_ROWMAJOR = 0, /* out[r,c] = (acc + bias[c]) * scale0 (+ resid[r,c])            */
  LGB200_EPI_HEADS = 1,    /* split into parts of 256 cols, optional rotary, head-major out */
  LGB200_EPI_LN_GELU = 2   /* N == 512: gelu(layernorm(acc + bias) * gamma + beta)          */
};

int lgb200_abi_version(void);
/* 0 if the current device can run the kernels (compute capability 10.x). */
int lgb200_device_ok(void);
const char* lgb200_error_string(int code);
/* Number of kernels this library has launched in the process so far (statistics for bench.py). */
unsigned long long lgb200_launch_count(void);

/* ---- input staging ------------------------------------------------------
 * Replaces descriptors.contiguous() + the implicit [B,N,d] layout,
 * lightglue.py:456-465 (input_proj itself goes through lgb200_linear).
 * src [B, n, dim] fp32 -> rows of sequences (2*b + img): x32 [S,Lp,dim] fp32 and/or
 * x16 (bf16); either may be NULL, not both.  Rows >= n are zero-filled. */
int lgb200_pack_rows(const float* src, int B, int n, int dim, int img, int Lp,
                     float* x32, void* x16, void* stream);

/* ---- positional encoding --------------------------------------------------
 * Replaces normalize_keypoints (lightglue.py:28-40) and
 * LearnableFourierPositionalEncoding.forward (lightglue.py:61-66).
 * kpts [B,n,kdim] fp32 (kdim 2, or 4 with scale/orientation appended),
 * size [B,2] (W,H) or NULL (extent of the valid points), Wr [32,kdim].
 * rot [S,Lp,64] fp32 receives (cos_f, sin_f) pairs, f = 0..31, for sequence
 * 2*b+img; one table serves the 4 heads and all layers (the reference's
 * repeat_interleave(2) is implicit: rotary pair f uses entry f).
 * rot16 [S,Lp,32] (nullable) receives the same pairs as packed fp16 (cos, sin):
 * the 128-byte-per-token table the bf16 QKV epilogue fetches by TMA.
 * At least one of rot / rot16 must be given. */
int lgb200_posenc(const float* kpts, int B, int n, int kdim, const float* size,
                  const float* Wr, const int32_t* lens, int img, int Lp,
                  float* rot, void* rot16, void* stream);

/* ---- linear layers with fused epilogues -------------------------------------
 * Replaces nn.Linear + the elementwise ops around it:
 *   Wqkv + unflatten + rotary   lightglue.py:157-161, 43-50
 *   to_qk / to_v                lightglue.py:196-201, 208
 *   out_proj / to_out           lightglue.py:163, 219
 *   ffn (cat, Linear, LayerNorm, GELU, Linear, residual)  lightglue.py:144-149,164,220-221
 *   final_proj / d**.25         lightglue.py:281-283
 *   input_proj                  lightglue.py:464-465
 * Y[T,N] = A[T,K] . W[N,K]^T, T = S*Lp.  A is A0[T,K0] followed column-wise by
 * A1[T,K-K0] (A1 NULL when K0 == K) -- this is the ffn's torch.cat([x,msg],-1).
 * A and W are fp32 (LGB200_F32) or bf16 (LGB200_BF16); bias/gamma/beta fp32.
 *   ROWMAJOR: out32 (fp32, nullable) / out16 (bf16, nullable), leading dim N;
 *             residual: resid32 [T,N] fp32 or resid16 [T,N] bf16 (at most one).
 *             The bf16 throughput path keeps the residual stream in bf16 only
 *             (resid16 == out16 updates it in place).
 *   HEADS:    N = parts*256, column c = part*256 + head*64 + d (the caller
 *             permutes Wqkv rows from the reference's head*192 + d*3 + part).
 *             Parts < n_rot get the rotary embedding from rot [T,64] fp32 or
 *             rot16 [T,32] packed fp16 (cos,sin) (LGB200_BF16 prefers rot16);
 *             part p is scaled by scale[p] and written to outp[p] laid out
 *             [S,4,Lp,64] in the precision's element type.
 *   LN_GELU:  N = 512; out as ROWMAJOR. */
int lgb200_linear(int precision, int epilogue, const void* A0, const void* A1, int K0,
                  const void* W, const float* bias, int T, int N, int K,
                  const int32_t* lens, int Lp,
                  float scale0, float scale1, float scale2,
                  const float* resid32, const void* resid16, float* out32, void* out16,
                  const float* rot, const void* rot16, int n_rot,
                  void* outp0, void* outp1, void* outp2,
                  const float* gamma, const float* beta, void* stream);

/* ---- attention ---------------------------------------------------------------
 * Replaces Attention.forward / F.scaled_dot_product_attention and the einsum
 * cross attention, lightglue.py:112-129, 203-217.  Q,K,V [S,4,Lp,64]; Q is
 * expected pre-scaled so that softmax uses exp2 (log2(e)/sqrt(64) folded in by
 * the producing lgb200_linear).  Sequence s attends to sequence s ^ kv_xor
 * (0 = self attention, 1 = the other image of the pair = cross attention);
 * keys >= lens[s ^ kv_xor] are masked, a sequence with no keys yields zeros
 * (nan_to_num, lightglue.py:118,217).  ctx [S,Lp,256] token-major, column
 * head*64+d (= transpose(1,2).flatten(-2), lightglue.py:163,218). */
int lgb200_attention(int precision, const void* Q, const void* K, const void* V,
                     int S, int Lp, const int32_t* lens, int kv_xor,
                     void* ctx, void* stream);
/* Same, with a launch order for ragged batches: order[S] (DEVICE int32, a permutation of 0..S-1, or NULL) lists the
 * sequences in the order their query tiles are handed to the SMs.  Sorted by key count, longest first, the kernel's
 * tail consists of the shortest work items (a CTA's duration is proportional to lens[s ^ kv_xor]).  The result does
 * not depend on it; the fp32 kernels ignore it. */
int lgb200_attention_ordered(int precision, const void* Q, const void* K, const void* V,
                             int S, int Lp, const int32_t* lens, const int32_t* order, int kv_xor,
                             void* ctx, void* stream);

/* ---- per-token heads -----------------------------------------------------------
 * Replaces matchability / token-confidence Linear(256,1) (+ sigmoid),
 * lightglue.py:72,75-80,285-286,290-291.  out[r] = dot(x[r,:], w) + b with x
 * [S*Lp,256] fp32 (LGB200_F32) or bf16 (LGB200_BF16), w/b fp32; sigmoid applied
 * when apply_sigmoid != 0; rows >= lens[s] are left untouched. */
int lgb200_rowdot(int precision, const void* x, const float* w, const float* b, int S, int Lp,
                  const int32_t* lens, int apply_sigmoid, float* out, void* stream);

/* ---- log assignment ---------------------------------------------------------------
 * Replaces the similarity einsum + sigmoid_log_double_softmax,
 * lightglue.py:257-269, 284-288.  md [S,Lp,256] = final_proj(desc)/4 (from
 * lgb200_linear), z [S,Lp] = matchability logits.
 *   pass 1 (lgb200_assign_lse): lse[s,l] = logsumexp_j <md[s,l], md[s^1,j]>,
 *          j < lens[s^1]  (row normaliser of image 0, column normaliser of image 1);
 *   pass 2 (lgb200_assign_scores): recomputes the similarity tile and writes
 *          scores [B,R,C] fp32 (R = n0max+1, C = n1max+1) exactly once:
 *          valid block 2*sim - lse0[i] - lse1[j] + logsigmoid(z0[i]) + logsigmoid(z1[j]),
 *          dustbin column C-1 = logsigmoid(-z0), dustbin row R-1 = logsigmoid(-z1),
 *          everything else (padding, corner) 0.
 *          best_ws (nullable, 8*B*(R+C) bytes, LGB200_BF16 only): the kernel also leaves the packed
 *          row / column maxima of the valid block there (computed on exactly the values it writes),
 *          which lgb200_filter_matches accepts with workspace_has_best = 1 and then does not
 *          re-read the score matrix at all. */
int lgb200_assign_lse(int precision, const void* md, int S, int Lp, const int32_t* lens,
                      float* lse, void* stream);
int lgb200_assign_scores(int precision, const void* md, const float* z, const float* lse,
                         int B, int Lp, const int32_t* lens, int R, int C,
                         float* scores, void* best_ws, void* stream);

/* ---- filter_matches -------------------------------------------------------------------
 * Replaces filter_matches, lightglue.py:294-319 (and the scatter back to
 * un-pruned indices, lightglue.py:527-536).  scores [B,R,C] fp32; pair b uses
 * rows < n0 = lens[2b], cols < n1 = lens[2b+1] (lens NULL: n0 = R-1, n1 = C-1).
 * Ties resolve to the lowest index, NaN counts as the maximum (torch.max).
 * ind0/ind1 (int32 [B,ind_ld], nullable) map current rows to original indices;
 * outputs are indexed by ORIGINAL index: m0 [B,N0] int64, m1 [B,N1] int64,
 * ms0 [B,N0], ms1 [B,N1] fp32; untouched entries are -1 / 0.
 * workspace: 8 * B * (R + C) bytes; workspace_has_best != 0 means it already holds the packed maxima
 * written by lgb200_assign_scores (scores may then be NULL). */
int lgb200_filter_matches(const float* scores, int B, int R, int C, const int32_t* lens,
                          float threshold, const int32_t* ind0, const int32_t* ind1, int ind_ld,
                          int N0, int N1, int64_t* m0, int64_t* m1, float* ms0, float* ms1,
                          void* workspace, int workspace_has_best, void* stream);

/* ---- nearest-neighbour matcher ----------------------------------------------------------
 * Replaces NearestNeighborMatcher._forward, gluefactory/models/matchers/nearest_neighbor_matcher.py:63-83
 * (fp32).  d [S,Lp,256] = descriptors packed like the LightGlue activations (rows >= count and columns
 * >= the descriptor dimension zero), lse from lgb200_assign_lse(LGB200_F32, d, ...).
 *   lgb200_nn_scores: similarity [B,R-1,C-1] (nullable) = <d0[i], d1[j]> (:64) and log_assignment [B,R,C] =
 *          log_softmax(sim, rows) + log_softmax(sim, columns) on the valid block, zeros elsewhere incl. the
 *          dustbin row / column (:72-74).
 *   lgb200_nn_match: find_nn (:15-31) for both images -- nearest neighbour by similarity, rejected if
 *          2(1-s1) > ratio^2 * 2(1-s2) (ratio_thresh > 0, more than one candidate) or 2(1-s1) > distance_thresh^2
 *          (distance_thresh > 0); lowest index among equal similarities -- then mutual_check (:34-43) if
 *          `mutual`; scores = (match > -1).  similarity [B,N,M]; workspace: 8 * B * (N + M) bytes. */
int lgb200_nn_scores(const float* d, const float* lse, int B, int Lp, const int32_t* lens, int R, int C,
                     float* similarity, float* log_assignment, void* stream);
int lgb200_nn_match(const float* similarity, int B, int N, int M, const int32_t* lens, float ratio_thresh,
                    float distance_thresh, int mutual, int64_t* workspace, int64_t* m0, int64_t* m1,
                    float* ms0, float* ms1, void* stream);

/* N_pair loss of the nearest-neighbour matcher, forward values.  Replaces
 * NearestNeighborMatcher.loss, nearest_neighbor_matcher.py:85-109:
 * scores = T (2 - sqrt(clamp(2 (1 - sim), 1e-6))), prob0 / prob1 = row / column
 * log-softmax of scores.  similarity [B,N,M] fp32, gt_assignment [B,N,M] bytes
 * (non-zero = match).  Outputs per row: row_sum[b,i] = sum_j a (prob0 + prob1),
 * row_cnt[b,i] = sum_j a; the caller forms nll = -sum_i row_sum / (2 max(sum_i row_cnt, 1)).
 * workspace: B * (N + M) floats. */
int lgb200_npair_loss(const float* similarity, const uint8_t* gt_assignment, int B, int N, int M,
                      float temperature, float* workspace, float* row_sum, float* row_cnt, void* stream);
/* Backward of lgb200_npair_loss (what autograd derives for nearest_neighbor_matcher.py:85-109), on the same
 * similarity, gt_assignment and temperature, after that call: workspace = its row / column log-sum-exps LR | LC,
 * row_cnt = its r.  coef [B] = -g_b / (2 num_b) with g_b the gradient of nll_b.  With s = T (2 - q),
 * q = sqrt(clamp(2 (1 - sim), 1e-6)) and c_j = sum_i a_ij:
 *   d nll / d s_ij = coef_b (2 a_ij - r_i exp(s_ij - LR_i) - c_j exp(s_ij - LC_j));
 *   dsim [B,N,M] (nullable: then nothing is written) = d nll / d s_ij * T / q_ij where 2 (1 - sim) >= 1e-6,
 *          0 where the clamp holds (torch's rule);
 *   dtemp_rows [B,N] = sum_j d nll / d s_ij (2 - q_ij), per-row partials of d nll / d T (no atomics: bit-reproducible;
 *          the caller adds them).
 * col_cnt [B,M]: scratch, receives c. */
int lgb200_npair_loss_bwd(const float* similarity, const uint8_t* gt_assignment, int B, int N, int M,
                          float temperature, const float* workspace, const float* row_cnt, const float* coef,
                          float* col_cnt, float* dsim, float* dtemp_rows, void* stream);

/* ---- loss-side reductions (SURVEY.md 8(f) rank 2; forward values only) -------------------
 * Replaces the dense [B,R,C] reductions behind LightGlue.loss, lightglue.py:588-637:
 *   NLLLoss / weight_loss, gluefactory/models/utils/losses.py:6-26 -- row_pos[b,i] = sum_j la[b,i,j] *
 *          gt[b,i,j] and row_cnt[b,i] = sum_j gt[b,i,j] over the inner block (i < R-1, j < C-1);
 *   losses["row_norm"], lightglue.py:606 -- row_exp[b,i] = sum_{j<C} exp(la[b,i,j]);
 *   TokenConfidence.loss, lightglue.py:86-91 -- row_arg[b,i] = argmax_{j<C} la[b,i,j] for i < R-1 and
 *          col_arg[b,j] = argmax_{i<R} la[b,i,j] for j < C-1 (torch.max: lowest index among equal values).
 * gt_assignment is the reference's bool tensor data["gt_assignment"] [B,R-1,C-1] (one byte per entry).
 * Any output pointer may be NULL; per-row results are written without atomics (bit-reproducible). */
int lgb200_loss_reduce(const float* log_assignment, int B, int R, int C, const uint8_t* gt_assignment,
                       float* row_pos, float* row_cnt, float* row_exp, int32_t* row_arg, int32_t* col_arg,
                       void* stream);
/* lgb200_loss_reduce_ragged: the same for a padded batch with per-pair counts lens [2B] (device; lens[2b] rows of
 * image 0, lens[2b+1] of image 1, each at most R-1 / C-1) in the inference layout of such a batch -- dustbin column
 * C-1 and dustbin row R-1 whatever the counts.  Pair b is reduced over rows i < lens[2b] and columns j < lens[2b+1]
 * of the inner block plus the dustbins: row_pos / row_cnt / row_exp sum over that region only (gt_assignment is read
 * only inside it), row_arg covers the valid columns plus the dustbin C-1, col_arg the valid rows plus the dustbin
 * R-1.  Rows i >= lens[2b] get row_pos = row_cnt = row_exp = 0 and row_arg = -1; columns j >= lens[2b+1] get
 * col_arg = -1.  lens must not be NULL (full counts: lgb200_loss_reduce). */
int lgb200_loss_reduce_ragged(const float* log_assignment, int B, int R, int C, const int32_t* lens,
                              const uint8_t* gt_assignment, float* row_pos, float* row_cnt, float* row_exp,
                              int32_t* row_arg, int32_t* col_arg, void* stream);

/* Fused form for LGB200_BF16 (tcgen05): MatchAssignment pass 2 of lgb200_assign_scores with the reductions above in
 * its epilogue instead of the store -- the [B,R,C] matrix of a layer that only the loss looks at (every layer but
 * the last in training mode, lightglue.py:607-608) is never written.  Same outputs as lgb200_loss_reduce on the
 * matrix lgb200_assign_scores would have produced; md / z / lse as for lgb200_assign_scores.  lens (nullable when
 * R-1 == C-1 == Lp) holds per-pair counts of at most R-1 / C-1: with counts below R-1 / C-1 the outputs are those of
 * lgb200_loss_reduce_ragged with the same lens (rows and columns past the counts: sums 0, arg-maximum -1; the
 * dustbin folded in only inside the counts).  workspace: 8 * B * (R + C) bytes.  LGB200_F32 is refused
 * (LGB200_ERR_PRECISION): the fp32 parity mode materialises and calls lgb200_loss_reduce(_ragged). */
int lgb200_assign_loss(int precision, const void* md, const float* z, const float* lse, int B, int Lp,
                       const int32_t* lens, int R, int C, const uint8_t* gt_assignment, float* row_pos,
                       float* row_cnt, float* row_exp, int32_t* row_arg, int32_t* col_arg, void* workspace,
                       void* stream);

/* ---- adaptive depth (early exit) ---------------------------------------------------------
 * Replaces check_if_stop, lightglue.py:569-580.  conf [S,Lp] = sigmoid token
 * confidences; pair b stops iff 1 - count(conf < thr)/total[b] > depth_conf
 * (fp32 arithmetic as in the reference).  done[b] is set to layer+1 for pairs
 * that stop now (pairs with done[b] != 0 are left alone) and their entries of
 * `lens_active` are zeroed so later kernels skip them. */
int lgb200_exit_check(const float* conf, int B, int Lp, const int32_t* lens,
                      const int32_t* total, float thr, float depth_conf, int layer,
                      int32_t* done, int32_t* lens_active, void* stream);

/* ---- adaptive width (point pruning) --------------------------------------------------------
 * Replaces get_pruning_mask + torch.where + index_select + prune += 1,
 * lightglue.py:506-521, 560-567.  keep[l] = match[s,l] > 1 - width_conf ||
 * (conf != NULL && conf[s,l] <= thr).  Rows are compacted from the *_src
 * buffers into the *_dst buffers (stable order), lens[s] is updated on the
 * device, prune_cnt[s, ind] += 1 for kept rows.  Sequences with
 * lens_active[s] == 0 are copied through unchanged in count (not pruned).
 * Each of the x32 / x16 / rot / rot16 buffer pairs may be NULL (not in use). */
int lgb200_prune_compact(const float* match, const float* conf, float thr, float width_conf,
                         int S, int Lp, int32_t* lens, int32_t* lens_active,
                         const float* x32_src, float* x32_dst,
                         const void* x16_src, void* x16_dst,
                         const float* rot_src, float* rot_dst,
                         const void* rot16_src, void* rot16_dst,
                         const int32_t* ind_src, int32_t* ind_dst,
                         int32_t* prune_cnt, void* stream);

/* ---- fp32-accurate tensor-core mode (LGB200_F32X3): helpers -------------------------------------
 * lgb200_split_rows: x [n] fp32 -> xs [2][n] fp16 planes (hi = fp16(x), lo = fp16(x - hi)); n % 4 == 0.
 * Used for the staged descriptors (lightglue.py:456-465) and after point pruning (:506-521). */
int lgb200_split_rows(const float* x, long long n, void* xs, void* stream);
/* lgb200_split_dynamic: the same for tensors without a fixed range (gradients): xs [2][n] = planes of g x with g the
 * power of two that brings max |x| into [256, 512) (1 for an all-zero tensor); inv_scale[0] = 1 / g on the device,
 * inv_scale[1] is scratch (two floats).  Feeds the three-product tensor-core GEMMs of the backward pass (train.py).
 * colsum_partials (nullable): x is read as [n / cols][cols] and colsum_partials [n_partials][cols] receives per-CTA
 * column sums from the same pass (the caller adds the n_partials rows: the bias gradient dY^T 1); cols % 4 == 0.
 * lgb200_merge_rows: planes [2][n] -> x [n] = (hi + lo) * inv_scale. */
int lgb200_split_dynamic(const float* x, long long n, void* xs, float* inv_scale, int cols, float* colsum_partials,
                         int n_partials, void* stream);
int lgb200_merge_rows(const void* xs, long long n, float inv_scale, float* x, void* stream);
/* Similarity of MatchAssignment (the einsum of lightglue.py:284) for all pairs: mds = split planes of
 * final_proj(desc)/4 [2][S*Lp][256]; sim [B][Lp][Lp] fp32 receives <md[2b,i], md[2b+1,j]> for i < lens[2b],
 * j < lens[2b+1] (tiles past the valid counts are not touched). Lp % 256 == 0. */
int lgb200_x3_similarity(const void* mds, int B, int Lp, const int32_t* lens, float* sim, void* stream);
/* lse [S*Lp]: row normaliser log_softmax(sim, 2) for image 0, column normaliser log_softmax(sim, 1) for image 1
 * (lightglue.py:262-263), natural log; n0 / n1 = counts when lens is NULL. */
int lgb200_x3_assign_lse(const float* sim, int B, int Lp, const int32_t* lens, int n0, int n1, float* lse,
                         void* stream);
/* scores [B][R][C] (lightglue.py:257-269) from sim, z (matchability logits [S*Lp]) and lse. */
int lgb200_x3_assign_scores(const float* sim, const float* z, const float* lse, int B, int Lp,
                            const int32_t* lens, int R, int C, float* scores, void* stream);

/* ---- training path: backward kernels (SURVEY.md 8(f) rank 2) -------------------------------------
 * The reference trains through this path with autograd (train.py -> LightGlue.forward, lightglue.py:484-498, and
 * LightGlue.loss, :588-637).  fp32 (the layouts of LGB200_F32).  Plain GEMMs of the backward pass (dX = dY.W,
 * dW = dY^T.X) are cuBLAS calls on the host side (glue_factory_colon_b200/train.py); the fused forward ops have
 * these fused backward ops:
 *
 * lgb200_attention_bwd: backward of lgb200_attention (flash-style: the score matrix is recomputed tile by tile,
 *   nothing N x M is stored).  Q, K, V [S,4,Lp,64] as given to the forward (Q pre-scaled, log2 domain), ctx / dctx
 *   [S,Lp,256] = forward output and its gradient.  dQ, dK, dV [S,4,Lp,64]: gradients w.r.t. the given (scaled) Q,
 *   K and V; with kv_xor = 1, dK / dV of sequence s collect the queries of sequence s ^ 1.  Rows >= lens are zero.
 *   Runs on tcgen05 in the fp32-accurate split-fp16 mode (csrc/lg_x3_attn_bwd.cu).  workspace:
 *   lgb200_attention_bwd_workspace(S, Lp) floats (row log-sum-exp, <dO, O>, and the fp16 plane pairs of Q, K, V, dO).
 * lgb200_attention_bwd_workspace: *n_floats = the workspace size of lgb200_attention_bwd for (S, Lp).
 * lgb200_heads_bwd: backward of the HEADS epilogue of lgb200_linear (unflatten + rotary + scale, lightglue.py:43-50,
 *   157-161, 196-201).  n_parts = 3: out [T,768] = [scale0 R^T dQ | scale1 R^T dK | scale2 dV] in the packed column
 *   order part*256 + head*64 + d, R^T = inverse rotation by the angles in rot [T,64]; dtheta [T,32] (nullable) +=
 *   the gradient of the rotary angles summed over heads and q / k (accumulates over layers; feeds posenc.Wr).
 *   n_parts = 2 (cross block): out [T,512] = [scale0 (dQ + dK) | scale1 dV]; Q, K, rot, dtheta unused.
 * lgb200_ln_gelu_bwd: backward of GELU(LayerNorm(h) gamma + beta) on rows of 512 (lightglue.py:144-149): h = the
 *   pre-LayerNorm activations, da = gradient of the GELU output; dh = gradient of h, act (nullable) = the GELU
 *   output recomputed (the A operand of d W2); partials [n_partials][1024] receives per-CTA column sums of
 *   (d gamma | d beta) -- the caller adds the n_partials rows.  Rows >= lens get zeros.
 * lgb200_assign_dsim: backward of sigmoid_log_double_softmax (lightglue.py:257-269) w.r.t. the similarity, for a
 *   loss that is linear in log_assignment (NLLLoss, losses.py:6-26): sim [B,m,n] is replaced in place by
 *   2 g_pos[b] gt - r[b,i] exp(sim - lse0[i]) - c[b,j] exp(sim - lse1[j]); lse as written by lgb200_assign_lse
 *   ([S,Lp]: rows of image 0, columns of image 1), r / c = g_pos times the row / column sums of gt.
 * lgb200_assign_dsim_ragged: the same for a padded batch (m, n = padded sizes) with per-pair counts lens [2B]
 *   (device, not NULL): entries of pair b with i >= lens[2b] or j >= lens[2b+1] become exactly 0, and gt, r, c and
 *   lse are read only inside the valid block. */
int lgb200_attention_bwd(const float* Q, const float* K, const float* V, const float* ctx, const float* dctx,
                         int S, int Lp, const int32_t* lens, int kv_xor, float* dQ, float* dK, float* dV,
                         float* workspace, void* stream);
int lgb200_attention_bwd_workspace(int S, int Lp, long long* n_floats);
/* lgb200_attention_bwd_bf16: backward of lgb200_attention(LGB200_BF16, ...) on what that forward read and wrote --
 *   Q, K, V bf16 [S,4,Lp,64] (Q pre-scaled into the log2 domain; rows >= lens must be finite, as for the forward),
 *   ctx bf16 [S,Lp,256] = the forward's output, dctx fp32 [S,Lp,256] = its gradient.  dQ, dK, dV fp32 [S,4,Lp,64] as
 *   for lgb200_attention_bwd (the layout lgb200_heads_bwd reads); rows >= lens are zero.  tcgen05, one bf16 MMA per
 *   product with fp32 accumulation; <dO, O> is formed in fp32.  workspace: lgb200_attention_bwd_bf16_workspace(S, Lp)
 *   floats (row log-sum-exp, <dO, O>, and dO as head-major bf16).
 * lgb200_attention_bwd_bf16_workspace: *n_floats = the workspace size of lgb200_attention_bwd_bf16 for (S, Lp). */
int lgb200_attention_bwd_bf16(const void* Q, const void* K, const void* V, const void* ctx, const float* dctx,
                              int S, int Lp, const int32_t* lens, int kv_xor, float* dQ, float* dK, float* dV,
                              float* workspace, void* stream);
int lgb200_attention_bwd_bf16_workspace(int S, int Lp, long long* n_floats);
int lgb200_heads_bwd(const float* dQ, const float* dK, const float* dV, const float* Q, const float* K,
                     const float* rot, int S, int Lp, const int32_t* lens, int n_parts, float scale0,
                     float scale1, float scale2, float* out, float* dtheta, void* stream);
int lgb200_ln_gelu_bwd(const float* h, const float* gamma, const float* beta, const float* da, int T, int Lp,
                       const int32_t* lens, float* dh, float* act, float* partials, int n_partials,
                       void* stream);
int lgb200_assign_dsim(float* sim, int B, int m, int n, const float* lse, int Lp,
                       const uint8_t* gt_assignment, const float* g_pos, const float* r, const float* c,
                       void* stream);
int lgb200_assign_dsim_ragged(float* sim, int B, int m, int n, const float* lse, int Lp, const int32_t* lens,
                              const uint8_t* gt_assignment, const float* g_pos, const float* r, const float* c,
                              void* stream);
/* lgb200_assign_bwd: backward of sigmoid_log_double_softmax (lightglue.py:257-269) for ANY upstream gradient
 *   G [B,m+1,n+1] fp32 = d loss / d log_assignment in the forward's layout (dustbin column n, dustbin row m).  Pair b
 *   uses rows i < n0 = lens[2b] and columns j < n1 = lens[2b+1] (lens NULL: n0 = m, n1 = n; an empty side is allowed);
 *   R_i / C_j are the row / column sums of G over that block.  sim [B,m,n] (the recomputed similarity) is replaced in
 *   place by d sim = 2 G_ij - R_i exp(sim_ij - lse0_i) - C_j exp(sim_ij - lse1_j) inside the block and exactly 0
 *   outside it; lse as written by lgb200_assign_lse ([S,Lp]: rows of image 0, columns of image 1).  z [S,Lp]
 *   (matchability logits, nullable): then dz0 [B,m] = R_i sigmoid(-z0_i) - G_{i,n} sigmoid(z0_i) and dz1 [B,n] =
 *   C_j sigmoid(-z1_j) - G_{m,j} sigmoid(z1_j), 0 past the counts.  Nothing outside the valid block (and its
 *   dustbin entries) is read.  No atomics: bit-reproducible.  workspace: lgb200_assign_bwd_workspace(B, m, n) floats.
 * lgb200_assign_bwd_workspace: *n_floats = B m + B n + B ceil(m / 32) n (row sums, column sums, per-warp column
 *   partials). */
int lgb200_assign_bwd(const float* G, float* sim, int B, int m, int n, const float* lse, int Lp, const int32_t* lens,
                      const float* z, float* dz0, float* dz1, float* workspace, void* stream);
int lgb200_assign_bwd_workspace(int B, int m, int n, long long* n_floats);
/* lgb200_posenc_bwd: gradient w.r.t. the keypoints of lgb200_posenc with the same kpts / B / n / kdim / size / Wr /
 *   lens / img / Lp.  dtheta [S,Lp,32] = gradient of the rotary angles (what lgb200_heads_bwd accumulates);
 *   dkpts [B,n,kdim] receives d kpts: through normalize_keypoints (lightglue.py:28-40) on the two coordinates -- with
 *   size NULL also through the extent 1 + max - min of the valid points, to the first arg-maximum / arg-minimum (torch's
 *   tie rule; the x extent wins a tie between W and H) -- and unchanged on scale / orientation.  Rows >= lens[2b+img]
 *   are 0.  Gradients w.r.t. size are not formed. */
int lgb200_posenc_bwd(const float* kpts, int B, int n, int kdim, const float* size, const float* Wr,
                      const int32_t* lens, int img, int Lp, const float* dtheta, float* dkpts, void* stream);

/* ---- whole matcher ------------------------------------------------------------------------------------------------
 * The no-grad forward of LightGlue in eval mode with depth_confidence <= 0 and width_confidence <= 0 (lightglue.py:
 * 422-553) behind two calls, for callers without the Python package (a C++ / LibTorch consumer of the plain-dict
 * state dict, weights.py).  lgb200_match makes exactly the calls of LightGlue._forward_impl in the same order, with the
 * same arguments, so its outputs are bit-equal to LightGlue.forward with the same weights, precision and counts. */
typedef struct {
  int precision;          /* LGB200_BF16 or LGB200_F32X3 (LightGlue precision "bf16" / "fp32"); else LGB200_ERR_PRECISION */
  int n_layers;           /* >= 1 */
  int input_dim;          /* 256, or the input_proj width: a positive multiple of 64 */
  int kdim;               /* 2, or 4 with add_scale_ori (scale, orientation appended to the keypoints) */
  float filter_threshold;
} lgb200_match_config;

/* Packed-weight table for `cfg`: *entries = 16 n_layers + 5 (+ 2 when input_dim != 256) and *pack_bytes = the device
 * bytes lgb200_pack_weights fills (every entry starts on a 256-byte boundary).
 *
 * Entry order -- per layer l = 0 .. n_layers-1, at 16 l + j (the names of LightGlue._pack):
 *    j  0 qkv_w  W [768][256]  Wqkv.weight, rows permuted head*192 + d*3 + part -> part*256 + head*64 + d
 *       1 qkv_b  F [768]       Wqkv.bias, same permutation
 *       2 sf0_w  W [512][512]  [W1x | W1m Wo]: self ffn.0 with out_proj folded in (float64, rounded to fp32 once)
 *       3 sf0_b  F [512]       b1 + W1m bo
 *       4 sln_g  F [512]       self ffn.1.weight       5 sln_b  F [512]  ffn.1.bias
 *       6 sf3_w  W [256][512]  self ffn.3.weight       7 sf3_b  F [256]  ffn.3.bias
 *       8 cqv_w  W [512][256]  to_qk.weight | to_v.weight (rows concatenated)
 *       9 cqv_b  F [512]       to_qk.bias | to_v.bias
 *      10 cf0_w  W [512][512]  cross ffn.0 with to_out folded in      11 cf0_b  F [512]
 *      12 cln_g  F [512]       13 cln_b  F [512]       14 cf3_w  W [256][512]       15 cf3_b  F [256]
 * then the tail, at t = 16 n_layers + j:
 *    j  0 wr     F [32][kdim]  posenc.Wr.weight
 *       1 fp_w   W [256][256]  log_assignment.{n_layers-1}.final_proj.weight     2 fp_b  F [256]
 *       3 m_w    F [256]       log_assignment.{n_layers-1}.matchability.weight   4 m_b   F [1]
 *       5 in_w   W [256][input_dim]  input_proj.weight (input_dim != 256 only)   6 in_b  F [256]
 * W = weight matrix in the operand format of the precision: LGB200_BF16 bf16 [N][K]; LGB200_F32X3 fp16 planes
 * [2][N][K] with 256 w = hi + lo (hi = fp16(256 w), lo = fp16(256 w - hi)).  F = fp32, copied as it is. */
int lgb200_weight_table_size(const lgb200_match_config* cfg, int* entries, long long* pack_bytes);

/* Packs the weights: tensors[i] (fp32, contiguous, DEVICE, the reference's shapes, which are not checked) is the
 * state-dict tensor called names[i] (host strings, the keys of LightGlue.state_dict() with prefixes stripped as
 * weights.strip_prefixes does).  Names not listed below are ignored; a missing one returns LGB200_ERR_WEIGHTS and a
 * NULL tensor of a required name LGB200_ERR_NULL, before anything is launched.  Required names:
 * BEGIN REQUIRED WEIGHTS
 *   transformers.{l}.self_attn.Wqkv.weight          transformers.{l}.self_attn.Wqkv.bias
 *   transformers.{l}.self_attn.out_proj.weight      transformers.{l}.self_attn.out_proj.bias
 *   transformers.{l}.self_attn.ffn.0.weight         transformers.{l}.self_attn.ffn.0.bias
 *   transformers.{l}.self_attn.ffn.1.weight         transformers.{l}.self_attn.ffn.1.bias
 *   transformers.{l}.self_attn.ffn.3.weight         transformers.{l}.self_attn.ffn.3.bias
 *   transformers.{l}.cross_attn.to_qk.weight        transformers.{l}.cross_attn.to_qk.bias
 *   transformers.{l}.cross_attn.to_v.weight         transformers.{l}.cross_attn.to_v.bias
 *   transformers.{l}.cross_attn.to_out.weight       transformers.{l}.cross_attn.to_out.bias
 *   transformers.{l}.cross_attn.ffn.0.weight        transformers.{l}.cross_attn.ffn.0.bias
 *   transformers.{l}.cross_attn.ffn.1.weight        transformers.{l}.cross_attn.ffn.1.bias
 *   transformers.{l}.cross_attn.ffn.3.weight        transformers.{l}.cross_attn.ffn.3.bias
 *   posenc.Wr.weight
 *   log_assignment.{L-1}.final_proj.weight          log_assignment.{L-1}.final_proj.bias
 *   log_assignment.{L-1}.matchability.weight        log_assignment.{L-1}.matchability.bias
 *   input_proj.weight                               input_proj.bias              (input_dim != 256 only)
 * END REQUIRED WEIGHTS
 * for every layer l < L = n_layers.  (token_confidence and the other layers' log_assignment serve adaptive depth /
 * width and the loss only.)  Writes the table's entries into pack_buf (pack_bytes from lgb200_weight_table_size) and
 * the HOST array table[entries] with device pointers into pack_buf (256-byte aligned).  Runs on `stream`; no allocation, no
 * synchronisation: the source tensors must stay valid until the stream has run the packing. */
int lgb200_pack_weights(const lgb200_match_config* cfg, int n, const char* const* names,
                        const float* const* tensors, void* pack_buf, long long pack_bytes,
                        const void** table, void* stream);

/* *bytes = the workspace of lgb200_match for B pairs of capacity m x n (it does not depend on the counts). */
int lgb200_match_workspace(const lgb200_match_config* cfg, int B, int m, int n, long long* bytes);

/* The forward.  table = the table filled by lgb200_pack_weights (or the same layouts built elsewhere).  Inputs fp32
 * contiguous: kpts0/1 [B,m|n,kdim], desc0/1 [B,m|n,input_dim], size0/1 [B,2] (W,H) or NULL (extent of the valid
 * points), counts0/1 DEVICE int32 [B] or NULL: per-pair valid counts of a padded batch (num_keypoints0/1), clamped to
 * [0, m] / [0, n] on the device.  Outputs (every pointer non-NULL, also when m or n is 0, except desc_out0/1):
 * matches0/1 int64 [B,m|n], scores0/1 fp32 [B,m|n] (matching_scores), log_assignment fp32 [B,m+1,n+1] (dustbin column
 * n, dustbin row m: the padded layout of LightGlue.forward), desc_out0/1 (nullable) [B,m|n,256] in the activation dtype
 * (bf16 / fp32) = the last layer's ref_descriptors.  workspace: lgb200_match_workspace bytes, 256-byte aligned.
 * Kernel launches: those of LightGlue.forward with the same inputs, plus one (device-side lens and attention launch
 * order) unless counts are NULL and m == n == Lp (Lp = max(m, n) rounded up to 128 in bf16, 256 in fp32, at least
 * that granule: lens is then NULL, as in the Python forward); besides, cudaMemsetAsync where
 * the Python forward allocates zeros and cudaMemcpy2DAsync for desc_out0/1.  No allocation, no synchronisation, no
 * host read of device data, every operation on `stream`: a call can be captured into a CUDA graph at a capacity m x n
 * and replayed with other inputs and counts written into the same buffers. */
int lgb200_match(const lgb200_match_config* cfg, const void* const* table, int B, int m, int n,
                 const float* kpts0, const float* kpts1, const float* desc0, const float* desc1,
                 const float* size0, const float* size1, const int32_t* counts0, const int32_t* counts1,
                 int64_t* matches0, int64_t* matches1, float* scores0, float* scores1,
                 float* log_assignment, void* desc_out0, void* desc_out1,
                 void* workspace, long long workspace_bytes, void* stream);

/* ---- adaptive matcher ---------------------------------------------------------------------------------------------
 * The same forward with LightGlue's adaptive depth (early exit, lightglue.py:501-505, 569-580) and adaptive width
 * (point pruning, :506-521, 560-567).  lgb200_match_adaptive makes the calls of LightGlue._forward_impl with every
 * layer launched (pairs that stopped cost empty kernels) and its tail -- MatchAssignment of each pair's exit layer,
 * filter_matches at the pruned counts -- on the device: no allocation, no synchronisation, no host read.  One capture
 * at B x K x K serves every input and every count, as for lgb200_match; the outputs are bit-equal to LightGlue.forward
 * with the same conf, in the layouts below. */
typedef struct {
  float depth_confidence; /* > 0: early exit after layers 0 .. n_layers-2; else off */
  float width_confidence; /* > 0: point pruning; else off */
} lgb200_adaptive_config;

/* Adaptive table: *entries = the lgb200_weight_table_size entries + 6 (n_layers - 1), *pack_bytes likewise (every
 * entry 256-byte aligned).  The first entries are exactly lgb200_pack_weights' table (an adaptive table also serves
 * lgb200_match); then, per layer l < n_layers-1, at base + 6 l + j (base = 16 n_layers + 5 (+ 2)):
 *    j  0 fp_w  W [256][256]  log_assignment.{l}.final_proj.weight     1 fp_b  F [256]  final_proj.bias
 *       2 m_w   F [256]       log_assignment.{l}.matchability.weight   3 m_b   F [1]    matchability.bias
 *       4 tk_w  F [256]       token_confidence.{l}.token.0.weight      5 tk_b  F [1]    token.0.bias
 * (layer n_layers-1's MatchAssignment is the tail of the first part).  W and F as for lgb200_weight_table_size. */
int lgb200_adaptive_table_size(const lgb200_match_config* cfg, int* entries, long long* pack_bytes);

/* lgb200_pack_weights for the adaptive table: same arguments and rules, with these names required besides the
 * REQUIRED WEIGHTS above (a missing one returns LGB200_ERR_WEIGHTS before anything is launched):
 * BEGIN ADAPTIVE WEIGHTS
 *   log_assignment.{l}.final_proj.weight            log_assignment.{l}.final_proj.bias
 *   log_assignment.{l}.matchability.weight          log_assignment.{l}.matchability.bias
 *   token_confidence.{l}.token.0.weight             token_confidence.{l}.token.0.bias
 * END ADAPTIVE WEIGHTS
 * for every layer l < L-1.  The confidence thresholds are not read: lgb200_match_adaptive computes
 * LightGlue.confidence_threshold, clip(0.8 + 0.1 exp(-4 l / L), 0, 1) in double rounded to float, on the host. */
int lgb200_pack_weights_adaptive(const lgb200_match_config* cfg, int n, const char* const* names,
                                 const float* const* tensors, void* pack_buf, long long pack_bytes,
                                 const void** table, void* stream);

/* *bytes = the workspace of lgb200_match_adaptive for B pairs of capacity m x n.  It depends on neither the counts nor
 * the confidences: lgb200_match_workspace's layout followed by, each 256-byte aligned, with T = 2 B Lp,
 * act = 2 (bf16) / 4 (fp32) bytes and rot = 128 (bf16) / 256 (fp32) bytes per token:
 *   ind, prune_cnt, conf, msig, ind_b   5 x T x 4      x_b  T x 256 x act      rot_b  T x rot
 *   done | lens_active | total  (2 B + 2 B) x 4        per-exit-layer counts  n_layers x 2 B x 4 */
int lgb200_match_adaptive_workspace(const lgb200_match_config* cfg, int B, int m, int n, long long* bytes);

/* The adaptive forward.  cfg, table (from lgb200_pack_weights_adaptive), B, m, n and the inputs and outputs up to
 * desc_out0/1 as for lgb200_match, with:
 *   log_assignment  fp32 [B, m+1, n+1], dustbin row m, dustbin column n; pair b's valid block is [:k0_b, :k1_b] at its
 *                   pruned counts (LightGlue.forward returns [B, max k0 + 1, max k1 + 1]: crop_log_assignment).
 *   matches0/1, scores0/1  indexed by the un-pruned keypoint, as LightGlue.forward returns them.
 *   desc_out0/1     the exit layer's descriptors, compacted by the pruning: rows < k_b, zeros past them.
 * and, each nullable:
 *   prune0/1        int32 [B, m|n]: the layer count of each keypoint (LightGlue.forward's prune0/1; n_layers for
 *                   every keypoint without width pruning);
 *   exit_layer      int32 [B]: the layer whose MatchAssignment gave the pair's outputs (n_layers-1 if it never exited);
 *   final_counts    int32 [B][2]: the pruned counts (k0_b, k1_b).
 * acfg NULL: LGB200_ERR_NULL.  Width pruning with Lp > 8192 (lgb200_prune_compact's limit): LGB200_ERR_SHAPE.  Both
 * argument checks come before any launch; with either mode on, every table entry must be non-NULL.
 * workspace: lgb200_match_adaptive_workspace bytes, 256-byte aligned.
 * Both confidences <= 0: exactly the calls of lgb200_match (same outputs), then one kernel that fills prune0/1,
 * exit_layer and final_counts if any of them is non-NULL.
 * Otherwise, with d = 1 under depth and 0 else, w likewise for width, x = 1 in LGB200_F32X3 and 0 in LGB200_BF16, the
 * kernel launches are those of lgb200_match with non-NULL counts on the same cfg and shapes, plus
 *     1                                 the adaptive state (lens_active, total, done, ind, prune_cnt)
 *   + (n_layers - 1) (2 d + (2 + x) w)  per layer but the last: token head + exit check, matchability + compaction
 *                                       (+ the plane split in LGB200_F32X3)
 *   + d (1 + (n_layers - 1) g)          the per-exit-layer counts and n_layers MatchAssignment groups instead of
 *                                       one, g = the group's launches: final_proj, matchability and lgb200_assign_lse
 *                                       (3) in LGB200_BF16; final_proj, matchability, lgb200_x3_similarity and
 *                                       lgb200_x3_assign_lse (3 + [m > 0] + [n > 0]) in LGB200_F32X3
 *   + 1                                 the descriptors, prune0/1, exit_layer and final_counts (when any is non-NULL)
 * besides cudaMemsetAsync where the Python forward allocates zeros.  No cudaMemcpy: desc_out0/1 follow device counts. */
int lgb200_match_adaptive(const lgb200_match_config* cfg, const lgb200_adaptive_config* acfg,
                          const void* const* table, int B, int m, int n,
                          const float* kpts0, const float* kpts1, const float* desc0, const float* desc1,
                          const float* size0, const float* size1, const int32_t* counts0, const int32_t* counts1,
                          int64_t* matches0, int64_t* matches1, float* scores0, float* scores1,
                          float* log_assignment, void* desc_out0, void* desc_out1,
                          int32_t* prune0, int32_t* prune1, int32_t* exit_layer, int32_t* final_counts,
                          void* workspace, long long workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LIGHTGLUE_B200_H_ */
