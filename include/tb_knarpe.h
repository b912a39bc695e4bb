/*
 * tb_knarpe.h — C ABI of libtbknarpe.so: hand-written sm_100a kernels for the TrafficBots-V1.5 hot path
 * (HPTR KNARPE attention + per-step closed-loop rollout).
 *
 * The reference (zhejz/TrafficBotsV1.5) is pure PyTorch and has no FFI; each entry point below replaces the
 * chain of eager ATen ops behind the cited reference function (paths relative to the reference's src/).
 *
 * Conventions (all entry points):
 *   - plain device pointers + sizes, no torch types; all buffers are caller-owned, on the current device;
 *   - float = fp32 row-major; masks are uint8 (torch.bool storage), nonzero = INVALID unless stated;
 *     indices are int32;
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*); nothing allocates, nothing
 *     synchronises, no global mutable state => CUDA-graph capturable and thread-safe per stream;
 *   - return value: 0 (TB_OK) or a negative TB_ERR_* code; never throws.
 */
#ifndef TB_KNARPE_H_
#define TB_KNARPE_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TB_OK 0
#define TB_ERR_BAD_SHAPE (-1)    /* non-positive / inconsistent dims                                  */
#define TB_ERR_KNN_RANGE (-2)    /* needs 0 < K < T            (reference assert: utils/rpe.py:79)     */
#define TB_ERR_UNSUPPORTED (-3)  /* size outside the compiled variants (e.g. T > 2048, D not 128/256) */
#define TB_ERR_MISALIGNED (-4)   /* pointer / leading dimension not 16-byte aligned where required    */
#define TB_ERR_NULL (-5)         /* required pointer is NULL                                          */
#define TB_ERR_CUDA (-6)         /* kernel launch failed (cudaGetLastError)                           */

const char* tb_strerror(int code);
int tb_version(void);

/* fp16 range guard of the tensor-core mode. The reference computes in fp32 (or AMP fp16 with a GradScaler,
 * configs/trainer/default.yaml:16); this library's 16-bit intermediates ([q|u], [k|v] tables, ReLU hidden rows, the
 * fused history encoder's MLP rows) are converted with saturation (never inf) and, when `d_flag` (one device word,
 * caller-owned, zeroed by the caller) is registered, every producing kernel ORs bit 0 into it if a converted value
 * reached +-65504. NULL unregisters. Host-side setting, not stream ordered: register before launching. */
int tb_set_fp16_flag(unsigned int* d_flag);

/* ---------------------------------------------------------------------------------------------------
 * Fused pairwise relative pose + K-nearest-target selection.
 * Replaces utils/rpe.py:9-37 (get_rel_pose) + :62-90 (get_tgt_knn_idx) + the row gathers of the winners.
 * For every source token (b,s): rel pose of every target in the source frame
 *   x' = dx cos(yaw_s) + dy sin(yaw_s), y' = -dx sin(yaw_s) + dy cos(yaw_s), dyaw = yaw_t - yaw_s (unwrapped),
 * dist = |(x',y')|, +inf if source or target invalid; the K smallest (ties: lower target index) are emitted
 * in ascending target-index order with  invalid = tgt_invalid | dist > dist_limit.
 * Targets of batch row b are taken from tgt batch (b / tgt_batch_div): the 32 WOSAC rollouts of one scene
 * share the scene's map / traffic-light table instead of a repeat_interleave copy
 * (pl_modules/waymo_motion.py:458-462).
 * Outputs are written at column offset `out_koff` of rows with `out_ldk` columns, so several selections
 * can be concatenated in place (agent_encoder.py:165-167).
 *   src_pose [B,S,3] src_invalid [B,S]  tgt_pose [B/div,T,3] tgt_invalid [B/div,T]
 *   out_idx [B,S,ldk] int32   out_invalid [B,S,ldk] u8   out_rel [B,S,ldk,3] f32
 * Optional (all may be NULL / 0) — repeated selections against STATIC targets (agent -> map, every rollout step):
 *   tgt_index_map [B/div,T] int32: the targets are passed in a caller-chosen order and out_idx reports
 *     tgt_index_map[position] (ties and output order then follow the passed order);
 *   flags & TB_KNN_SORTED_BY_X: the caller promises tgt_pose[..,0] ascending within each target batch;
 *   row_state [B,S,3] f32 (in/out): (x, y, K-th smallest squared distance) of the previous call for the same row,
 *     K-th = +inf to start. With sorted targets only the slab |x_t - x_s| <= sqrt(K-th) + |displacement| is scanned
 *     (the K nearest of the previous call still lie within that radius: same result as a full scan). Without
 *     sorted targets the state still brackets the bisection for the K-th distance. A row state REQUIRES static targets.
 * `flags` (the former sorted_by_x argument; 1 keeps its meaning):
 *   TB_KNN_SORTED_BY_X  the caller promises tgt_pose[..,0] ascending within each target batch (above);
 *   TB_KNN_REFERENCE    run the previous kernels (full-length bisections, one kernel for every path) instead of the
 *                       current ones. Both emit the same lists and row states bit for bit; kept for A/B and tests.
 * Limits: 0 < K < T <= 2048.
 * ------------------------------------------------------------------------------------------------- */
#define TB_KNN_SORTED_BY_X 1
#define TB_KNN_REFERENCE 2
int tb_knn_select(const float* src_pose, const uint8_t* src_invalid, const float* tgt_pose,
                  const uint8_t* tgt_invalid, int B, int S, int T, int tgt_batch_div, int K, float dist_limit,
                  int32_t* out_idx, uint8_t* out_invalid, float* out_rel, int out_ldk, int out_koff,
                  const int32_t* tgt_index_map, float* row_state, int flags, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * KNARPE attention core (gather + relative-pose bias + masked softmax + weighted sum).
 * Replaces modules/attention_rpe.py:137-190 between the input projections and the output projection, in the
 * re-associated form (DESIGN.md §3):
 *   logit_hj = q_h . k_hj + u_h . e_j           (u_h = W_rk,h^T q_h, computed by the caller's projection)
 *   a_h = softmax_j(logit_hj)  over the non-masked neighbours   (q, u already carry 1/sqrt(d_head)*log2 e)
 *   ov_h = sum_j a_hj v_hj ,  z_h = sum_j a_hj e_j
 * e_j = PoseEmb("pe_xy_yaw") of the neighbour's relative pose (utils/pose_emb.py:50-55) evaluated in
 * registers from `rel` [B,S,K,3], or read from `emb` [B,S,K,D] when the caller has it materialised
 * (exactly one of rel/emb non-NULL). Neighbour j < K0 is row idx of table kv0, j >= K0 of table kv1
 * (K1 may be 0); a table row is [k(D) | v(D)] at `kvX + (b/divX * TX + row) * ldkvX`.
 * Rows whose neighbours are all masked produce zeros and none_valid = 1 (attention_rpe.py:112-118,188-190).
 *   q [B*S] rows, leading dim ldq (D floats used);  u [B*S] rows, leading dim ldu (H*D floats, head-major)
 *   out_ov / out_z: rows with leading dim ldo (D and H*D floats)
 *   pe_freq_xy: D/8 floats = PositionalEmbedding(dim=D/4, theta).freqs[::2] (utils/positional_emb.py:11)
 * flags bit 0: evaluate the embedding angles with the SFU's own range reduction (no 2-term Cody-Waite step): abs error
 *   grows with |angle| (<= ~2e-5 at 150 rad, the fp32 rounding of a 150 m coordinate); used with the tf32 projections.
 * flags bit 1: 16-bit mode. kv0 / kv1 are IEEE fp16 tables (leading dims in halves, multiples of 8) as written
 *   by tb_linear's Yh output. For D == 128 and K0 + K1 <= 128 all four contractions (q.k, u.e, sum a e, sum a v) run
 *   on mma.sync (f16 operands, f32 accumulate; q, u and a are split into fp16 head + residual, k, v and e are rounded
 *   to fp16: 2^-11 relative per component, the rounding a tf32 projection applies to its inputs anyway; implies the
 *   bit-0 trig). Other shapes (D == 256: BASELINE config 2; longer lists) gather the fp16 rows with the fp32-arithmetic
 *   kernel: they need bit 0 and bits 2 and 3 both set or both clear. Needs rel != NULL.
 * flags bit 2: out_ov / out_z are IEEE fp16 rows (ldo in halves, multiple of 8) — what tb_linear precision 2 consumes.
 *   Needs D == 128, rel != NULL and bit 0 (or bit 1).
 * flags bit 3: q / u are IEEE fp16 rows (ldq, ldu in halves, multiples of 8) as written by tb_linear's Yh output;
 *   with bit 1 they are MMA operands as they are (no residual). Needs bit 2 when bit 1 is not set.
 * flags bit 4: head-interleaved channels. The q rows and the K and V halves of the table rows store channel c
 *   (0..31) of head h at position 64*(h>>1) + 16*(c>>3) + 8*(h&1) + (c&7), so that a lane reads 32 contiguous bytes
 *   (one 256-bit load) holding its MMA fragments of two heads - half the L1 wavefronts per gathered row. The caller
 *   gets the layout for free by permuting the output features of the q / k / v projection weights; u, out_ov and
 *   out_z keep the natural order. Needs bits 1 and 3, K0 + K1 <= 128, table pointers 32-byte aligned and table leading
 *   dims multiples of 16 halves.
 * Limits: D in {128,256} (d_rpe == D), H == 4, all leading dims and pointers 16-byte aligned.
 * ------------------------------------------------------------------------------------------------- */
int tb_knarpe_attn(const void* q, int ldq, const void* u, int ldu,
                   const void* kv0, int ldkv0, int T0, int div0, int K0,
                   const void* kv1, int ldkv1, int T1, int div1, int K1,
                   const int32_t* idx, const uint8_t* invalid, const float* rel, const float* emb,
                   const float* pe_freq_xy, int B, int S, int D, int H,
                   void* out_ov, void* out_z, int ldo, uint8_t* out_none_valid, int flags, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Backward of the KNARPE attention core (SURVEY.md 8(f) rank 2, first piece; autograd through
 * modules/attention_rpe.py:137-190 in the re-associated form above). Inputs as tb_knarpe_attn (fp32 tables, rel pose
 * form, D == 128, H == 4, K0 + K1 <= 128) plus the upstream gradients d_ov [B*S, D] / d_z [B*S, H*D] (ld ldo).
 * Outputs: d_qu rows [d_q (D) | d_u (H*D)] (ld ldg); d_kv0 / d_kv1: gradient tables with the layout and leading
 * dimension of kv0 / kv1, ACCUMULATED with vector atomics (the caller zero-fills them). No gradient flows into the
 * relative pose. All-masked rows contribute zeros.
 * ------------------------------------------------------------------------------------------------- */
int tb_knarpe_attn_bwd(const float* q, int ldq, const float* u, int ldu, const float* kv0, int ldkv0, int T0, int div0,
                       int K0, const float* kv1, int ldkv1, int T1, int div1, int K1, const int32_t* idx,
                       const uint8_t* invalid, const float* rel, const float* pe_freq_xy, int B, int S, int D, int H,
                       const float* d_ov, const float* d_z, int ldo, float* d_qu, int ldg, float* d_kv0, float* d_kv1,
                       void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Dense projection  Y = epilogue(X W^T + bias)  — replaces F.linear / nn.Linear call sites
 * (attention_rpe.py:96-97,147,186; transformer_rpe.py:237-238; modules/mlp.py:69).
 *   X [M,K] ld ldx;  W [N,K] (nn.Linear layout) ld K;  Y [M,N] ld ldy
 *   v = acc + bias[n]  (bias_group == 0)  or  acc + bias[(m / bias_group) * N + n]  (one bias row per group of
 *   bias_group consecutive rows: the PointNet "concat the group max" term W_right max_g + b, polyline_encoder.py:52);
 *   if relu: v = max(v,0); if mask_pre[m]: v = 0; if res: v += res[m*ldr+n]; if mask_post[m]: v = 0.
 * precision: 0 = fp32 FFMA (parity path), 1 = tf32 tcgen05 tensor cores (fp32 operands read as tf32, fp32 accumulate),
 *   2 = X and W are IEEE fp16 arrays (ldx in halves; tcgen05 kind::f16, fp32 accumulate) — the consumer side of the
 *   fp16 intermediates of the tensor-core mode (attention output [ov|z], FFN hidden); bias / residual / Y stay fp32.
 * Yh (optional, precision 1 or 2): columns [col_h, N) of the result are written as IEEE fp16 to
 *   Yh[row*ldyh + col - col_h] instead of Y (col_h a multiple of 32; col_h == 0 => Y may be NULL). This is how the
 *   K|V tables consumed by tb_knarpe_attn flags bit 1 are produced without a conversion pass.
 * ------------------------------------------------------------------------------------------------- */
int tb_linear(const void* X, int ldx, const void* W, const float* bias, int bias_group, float* Y, int ldy, int M,
              int N, int K, int relu, const uint8_t* mask_pre, const float* res, int ldr, const uint8_t* mask_post,
              int precision, void* Yh, int ldyh, int col_h, void* stream);

/* 3xTF32 operand split for fp32-accurate projections on the tf32 tensor cores (the strict-parity mode of the engine):
 *   out[m, :] = [ X[m, :] | X[m, :] - trunc_tf32(X[m, :]) | X[m, :] ]   (3K columns, ld ldo)
 * With W3 = [W | W | W - trunc_tf32(W)] (built once per weight by the host), tb_linear(precision 1) over K' = 3K computes
 * x_hi W_hi + x_lo W_hi + x_hi W_lo: fp32-class accuracy (2^-20 relative) at tensor-core speed, same epilogue.
 * K and the leading dims multiples of 4, pointers 16-byte aligned. */
int tb_tf32_split3(const float* X, int ldx, int M, int K, float* out, int ldo, void* stream);

/* tb_linear with the LayerNorm of its result fused into the epilogue (tensor-core mode, N == 128):
 *   Y = X W^T + bias, masks / residual as tb_linear (no ReLU); ln_out[row] = fp16(LayerNorm(Y[row]) * gamma + beta),
 *   eps 1e-5 (transformer_rpe.py:156-171 applied to the residual stream right after attention / FFN, :233-245) —
 *   the rows the next kind::f16 projection reads, so the residual stream is not re-read by a LayerNorm launch.
 *   precision 1 (fp32 X, W) or 2 (fp16 X, W). Y, res, bias, gamma, beta 16-byte aligned, ln_out 8-byte aligned,
 *   leading dims multiples of 4; anything else: TB_ERR_UNSUPPORTED / TB_ERR_MISALIGNED (call tb_linear + tb_layernorm).
 *   Statistics in fp32 without cancellation: per 32 columns the sum and M2 of the values shifted by the first of them,
 *   merged over the row with Chan's formula M2 = sum M2_h + 32 sum (mean_h - mean)^2, variance M2 / 128. */
int tb_linear_ln(const void* X, int ldx, const void* W, const float* bias, float* Y, int ldy, int M, int N, int K,
                 const uint8_t* mask_pre, const float* res, int ldr, const uint8_t* mask_post, int precision,
                 const float* ln_gamma, const float* ln_beta, void* ln_out, int ld_ln, void* stream);

/* LayerNorm over the last dim (eps 1e-5, affine) — transformer_rpe.py:156-171. flags bit 0: ReLU on the result (the
 * Linear -> LayerNorm -> ReLU layers of modules/mlp.py:47-51 with use_layernorm); bit 1: Y rows are IEEE fp16 (ldy in
 * halves, multiple of 8) — the operand a tb_linear precision-2 projection reads. D in {128,256}. */
int tb_layernorm(const float* X, int ldx, const float* gamma, const float* beta, void* Y, int ldy, int M, int D,
                 int flags, void* stream);

/* LayerNorm backward (training path, SURVEY 8(f) rank 2; nn.LayerNorm of transformer_rpe.py:156-171):
 *   dX[row] = rstd (g - mean(g) - xhat mean(g xhat)), g = dY gamma, xhat = (X - mean) rstd (statistics recomputed);
 *   dgamma[c] += sum_rows dY xhat, dbeta[c] += sum_rows dY  (the caller zeroes dgamma / dbeta; atomics).
 *   D in {128, 256}; pointers 16-byte aligned, leading dims multiples of 4. */
int tb_layernorm_bwd(const float* X, int ldx, const float* gamma, const float* dY, int lddy, float* dX, int lddx,
                     float* dgamma, float* dbeta, int M, int D, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Training path (SURVEY.md 8(f) rank 2, BASELINE config 4): gradients of the layers above and the differentiable
 * part of the closed loop. Reference: pl_modules/waymo_motion.py:313-385 (training_step body), autograd through
 * modules/mlp.py:69, transformer_rpe.py:175-245, polyline_encoder.py:50-53, utils/dynamics.py:66-141,237-274,
 * utils/rewards.py:35-85, models/metrics/loss.py:9-37, models/metrics/training.py:76-160.
 * ------------------------------------------------------------------------------------------------- */

/* Weight gradient of Y = X W^T + b:  dW[n,k] += sum_m dY[m,n] X[m,k],  db[n] += sum_m dY[m,n]  (db may be NULL).
 * Split over M with fp32 atomics: dW (ld lddw) / db are ACCUMULATED (the caller zero-fills them once and may collect
 * every use of a shared weight in the same buffer). precision 0: fp32 FFMA; 1: tcgen05 kind::tf32 with both operands
 * MN-major straight from the row-major activations via TMA (csrc/wgrad_tc.cu; leading dims multiples of 4 floats and
 * 16-byte aligned pointers, else the FFMA kernel runs). The data gradient dX = dY W is tb_linear with W^T. */
int tb_linear_wgrad(const float* dY, int lddy, const float* X, int ldx, int M, int N, int K, float* dW, int lddw,
                    float* db, int precision, void* stream);

/* out[n] += sum over the M rows of X[m, n] (bias gradient; out is accumulated with atomics). */
int tb_colsum(const float* X, int ldx, int M, int N, float* out, void* stream);

/* Backward of a tb_linear epilogue: out[m,n] = dY[m,n] where the row is in neither mask and (Y == NULL or Y[m,n] > 0),
 * else 0. Y is the epilogue's own output (ReLU and pre/post row masks all leave zeros there). */
int tb_grad_mask(const float* dY, int lddy, const float* Y, int ldy, const uint8_t* mask_a, const uint8_t* mask_b, int M,
                 int N, float* out, int ldo, void* stream);

/* out[g, :] = sum of the L consecutive rows of group g of X: gradient of a grouped bias (tb_linear bias_group). */
int tb_group_sum(const float* X, int ldx, int G, int L, int N, float* out, int ldo, void* stream);

/* Backward of tb_pointnet_pool modes 1 / 2 (x.amax over the valid rows of a group, polyline_encoder.py:52,
 * utils/pooling.py:38): dX[row, c] = dOut[g, c] (+ dOut[g, C + c] in mode 2) on the first valid row attaining the
 * maximum, 0 elsewhere (ties only occur at ReLU zeros, where the ReLU backward drops the gradient). */
int tb_pointnet_pool_bwd(const float* X, int ldx, const uint8_t* invalid, int G, int L, int C, int mode,
                         const float* dOut, int ldo, float* dX, int lddx, void* stream);

/* Imitation loss of a recorded closed-loop rollout and its gradient w.r.t. the action-head outputs of every step.
 * The policy inputs are detached in training (waymo_motion.py:158-161), so the chain through time is the state
 * recurrence only (dynamics.py:84-141, MultiPathPP :237-274; teacher-forced / spawned rows are replaced by the ground
 * truth, which cuts the chain). One thread per (rollout-scene, agent).
 *   act [T, B*A, 6] action-head outputs (pre-tanh; (veh, ped, cyc) x (acc, yaw rate)); pred_valid [B*A, T] u8 as
 *   recorded by tb_dyn_step; pose0 / motion0 [B*A, 3] state at time 0; gt_* [B/sc_div, A, n_gt(, 3)]; tf_mask as
 *   tb_dyn_step; loss_mask [B*A] u8 or NULL (relevant-agent mask, training.py:93-98); step_start: first counted
 *   buffer index (training.py:99-101); weights of rewards.py:62-70 (SmoothL1 position / speed, 0.5 (1 - cos) heading).
 * fwd: state_in [T, B*A, 4] (16-byte aligned) <- (x, y, yaw, speed) before every step; out[0] += sum of the weighted
 *   errors, out[1] += number of counted entries (caller zero-fills; loss = -w_diffbar_reward * (-out[0]) / out[1]).
 * bwd: d_act [T, B*A, 6] <- g_out[0] * d out[0] / d act (every element written). */
int tb_il_loss_fwd(const float* act, const uint8_t* ag_type, const float* max_acc, const float* max_yaw_rate, float dt,
                   const uint8_t* pred_valid, const float* pose0, const float* motion0, const uint8_t* gt_valid,
                   const float* gt_pose, const float* gt_motion, const uint8_t* tf_mask, const uint8_t* loss_mask,
                   int n_gt, int sc_div, int B, int A, int T, int step_start, float w_pos, float w_rot, float w_spd,
                   float* state_in, float* out, void* stream);
int tb_il_loss_bwd(const float* act, const uint8_t* ag_type, const float* max_acc, const float* max_yaw_rate, float dt,
                   const uint8_t* pred_valid, const uint8_t* gt_valid, const float* gt_pose, const float* gt_motion,
                   const uint8_t* tf_mask, const uint8_t* loss_mask, int n_gt, int sc_div, int B, int A, int T,
                   int step_start, float w_pos, float w_rot, float w_spd, const float* state_in, const float* g_out,
                   float* d_act, void* stream);

/* Traffic-light state NLL of all steps (waymo_motion.py:270-277, traffic_light.py:284-286, training.py:155-160):
 * -log_softmax(clamp(logits, -3, 3))[argmax gt] over valid lights and steps s < n_gt.
 *   logits [T, n, 5] (step s at index s - 1), tl_invalid [n] u8, gt_tl [n, n_gt, 5] u8.
 * out != NULL: out[0] += sum, out[1] += count. d_logits != NULL: d_logits <- g_out[0] * d out[0] / d logits. */
int tb_tl_nll(const float* logits, const uint8_t* tl_invalid, const uint8_t* gt_tl, int n_gt, int n, int T, float* out,
              const float* g_out, float* d_logits, void* stream);

/* Categorical NLL of the destination classifier (navigation.py:265-278 logits with -inf on excluded polylines,
 * training.py:146-153): nll[r] = logsumexp(logits[r, :]) - logits[r, target[r]] on rows with row_valid != 0.
 *   logits [R, C] ld ld, target int64 [R], row_valid u8 [R]. out != NULL: out[0] += sum, out[1] += count.
 *   d_logits != NULL (ld ldd): g_out[0] * (softmax - onehot) on valid rows, 0 elsewhere (every element written). */
int tb_softmax_nll(const float* logits, int ld, const int64_t* target, const uint8_t* row_valid, int R, int C, float* out,
                   const float* g_out, float* d_logits, int ldd, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * PointNet pooling step over groups of L consecutive rows — modules/polyline_encoder.py:50-53 and
 * utils/pooling.py:18-19,38. X rows have 2*C columns; the left C columns hold relu(Linear(x)).
 * mode 0 (layer): right half <- max over the group's valid rows of the left half; invalid rows <- 0 (both halves)
 * mode 1 (final): out[g, 0:C2] = max over valid rows of X (0 if the group has no valid row)
 * mode 2: as mode 1 but written twice, out[g] = [max | max] (C2 columns each)
 *   X [G*L, 2C] ld ldx, invalid [G*L] u8, out [G, 2C] (mode 1 only). 2C in {128,256}.
 * ------------------------------------------------------------------------------------------------- */
int tb_pointnet_pool(float* X, int ldx, const uint8_t* invalid, int G, int L, int C2, int mode, float* out, int ldo,
                     void* stream);

/* ---------------------------------------------------------------------------------------------------
 * PoseEmb("pe_xy_yaw") of poses expressed in a reference frame — utils/pose_emb.py:50-55 with
 * transform_utils.py:146-157,200-213 (cast=False). For row m: (x,y,yaw) = pose[m] seen from frame[m / frame_div]
 * (frame NULL => identity). Writes pe_dim floats at out[m*ldo .. ]. pe_dim in {64,128,256}.
 * freq_xy: pe_dim/8 floats.
 * ------------------------------------------------------------------------------------------------- */
int tb_pose_emb(const float* pose, const float* frame, int frame_div, const float* freq_xy, int M, int pe_dim,
                float* out, int ldo, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Rollout state (DESIGN.md §4): ring buffers of the last W=11 steps, slot = time % W.
 * `d_step` points to the device-resident loop counter s (1-based policy step, waymo_motion.py:233);
 * the state in the ring covers times max(0,s-W) .. s-1.
 * ------------------------------------------------------------------------------------------------- */

/* Agent history tokens — agent_encoder.py:130-157 and pooling.py:24-29 (last_valid).
 *   hist_valid [B,A,W] u8 (1 = valid), hist_pose/hist_motion [B,A,W,3], ag_attr [B,A,6]
 * out: tok_pose [B,A,3], tok_invalid [B,A], row_invalid [B,A,W] (window order, oldest first; absent = 1),
 *      attr rows [B*A*W, 20] = [attr6 | motion3 | one-hot11 (agent_encoder.py:154)] (ld lda),
 *      pe rows: PoseEmb pe_dim=64 of the history pose in the token frame, written at pe_out (ld ldpe).
 * row_invalid, attr_out and pe_out may all be NULL: only tok_pose / tok_invalid are produced (used to start the KNN
 * selects while tb_ag_frontend encodes the history). */
int tb_ag_featurize(const uint8_t* hist_valid, const float* hist_pose, const float* hist_motion,
                    const float* ag_attr, const int* d_step, const float* freq_xy, int B, int A, int W,
                    float* tok_pose, uint8_t* tok_invalid, uint8_t* row_invalid, float* attr_out, int lda,
                    float* pe_out, int ldpe, void* stream);
/* Same with one loop counter per batch row: s(b) = d_step[b * step_stride] (step_stride 0 = the shared scalar above).
 * The training path evaluates the policy of ALL steps of a recorded rollout as one batch of scenes x steps rows
 * (waymo_motion.py:158-161: the policy inputs are detached, so every step's forward / backward is independent). */
int tb_ag_featurize_ex(const uint8_t* hist_valid, const float* hist_pose, const float* hist_motion,
                       const float* ag_attr, const int* d_step, int step_stride, const float* freq_xy, int B, int A,
                       int W, float* tok_pose, uint8_t* tok_invalid, uint8_t* row_invalid, float* attr_out, int lda,
                       float* pe_out, int ldpe, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Fused agent history encoder of the tensor-core mode — agent_encoder.py:130-162 in one kernel (one warp per agent):
 * tb_ag_featurize's rows -> input MLP [9+W -> 64 -> 64 -> 64] ++ PoseEmb64 -> PointNet 3 x (128 -> 64, max over the
 * valid steps) -> token [max h | max h]; mma.sync f16 operands / f32 accumulate, activations never leave registers.
 *   wblob: tb_ag_frontend_blob_halves() fp16 values = the six weight matrices, row-major [64 outputs][inputs] with
 *   row strides 40 (W1, inputs zero-padded to 32), 72 (W2, W3), 136 (P0, P1, P2), in that order; bias: fp32 [6][64].
 *   tok_out [B*A, 128] fp32 (ld ldo): zeros for agents without a valid step; tok_pose [B,A,3], tok_invalid [B,A].
 *   ln_out (may be NULL): fp16 rows [B*A, 128] (ld ld_ln, multiple of 2) = LayerNorm(token) * ln_gamma + ln_beta, eps
 *   1e-5 — the first LayerNorm of the agent transformer (transformer_rpe.py:156-171) from the same warp.
 * W <= 16 (one MMA tile of history rows). */
int tb_ag_frontend_blob_halves(void);
int tb_ag_frontend(const uint8_t* hist_valid, const float* hist_pose, const float* hist_motion, const float* ag_attr,
                   const int* d_step, const float* freq_xy, int B, int A, int W, const void* wblob, const float* bias,
                   float* tok_out, int ldo, float* tok_pose, uint8_t* tok_invalid, const float* ln_gamma,
                   const float* ln_beta, void* ln_out, int ld_ln, void* stream);
/* Same with one loop counter per batch row, s(b) = d_step[b * step_stride] (see tb_ag_featurize_ex): the engine encodes
 * the rollout-invariant warm-start steps of all scenes as one batch of (scene, step) rows. */
int tb_ag_frontend_ex(const uint8_t* hist_valid, const float* hist_pose, const float* hist_motion, const float* ag_attr,
                      const int* d_step, int step_stride, const float* freq_xy, int B, int A, int W, const void* wblob,
                      const float* bias, float* tok_out, int ldo, float* tok_pose, uint8_t* tok_invalid,
                      const float* ln_gamma, const float* ln_beta, void* ln_out, int ld_ln, void* stream);

/* Traffic-light history rows — traffic_light.py:223-225: [state5 | one-hot11] per (b,tl,window slot).
 *   hist_tl [B,TL,W,5] u8 one-hot, tl_invalid [B,TL]; out rows [B*TL*W,16] (ld lda), row_invalid [B,TL,W]. */
int tb_tl_featurize(const uint8_t* hist_tl, const uint8_t* tl_invalid, const int* d_step, int B, int TL, int W,
                    float* attr_out, int lda, uint8_t* row_invalid, void* stream);
/* Same with one loop counter per batch row, s(b) = d_step[b * step_stride] (see tb_ag_featurize_ex). */
int tb_tl_featurize_ex(const uint8_t* hist_tl, const uint8_t* tl_invalid, const int* d_step, int step_stride, int B,
                       int TL, int W, float* attr_out, int lda, uint8_t* row_invalid, void* stream);

/* Agent dynamics + closed-loop bookkeeping for one step — utils/dynamics.py:66-141,166-204 (update_ag,
 * override_ag, disable_ag, disable_navi), MultiPathPP :237-274, teacher_forcing.py:126-147,
 * traffic_rule_checker.py:107-116 (outside map) and :291-319 (dest reached), waymo_motion.py:179-190,250,289-290.
 *   act_branch [B*A, 3*2]: per-type action-head outputs (veh,ped,cyc) (action_head.py:78-82)
 *   ag_type [B,A,3] u8 one-hot, max_acc[3], max_yaw_rate[3] (HOST arrays; veh,ped,cyc), dt
 *   state (in/out): valid/disabled/navi_invalid/dest_reached [B,A] u8 (1 = true), pose/motion [B,A,3]
 *   gt_* [B/sc_div, A, n_gt(,3)], tf_mask [B/sc_div, A, n_gt] (teacher_forcing.py:51-82); sc_div = rollouts per scene
 *   boundary [B/sc_div,4] (xmin,xmax,ymin,ymax); dest_idx [B,A] int32 polyline index of each agent's destination;
 *   per-scene destination tables (traffic_rule_checker.py:86-105): mp_pos [B/sc_div,n_mp,n_node,2],
 *   mp_dirn (unit direction) same shape, mp_node_invalid [B/sc_div,n_mp,n_node] u8,
 *   mp_kind [B/sc_div,n_mp] u8 (1 = lane types 0..3, 2 = road edge type 4, 0 = never reached);
 *   thresh_lane / thresh_edge (50 m / 50*(1-0.8) m) and cos_rot = cos(30 deg) as the reference rounds them
 *   out: pred_valid [B,A,T] u8, pred_pose/pred_motion [B,A,T,3] at index s-1; ring slot s%W of hist_*. */
int tb_dyn_step(const float* act_branch, const uint8_t* ag_type, const float* max_acc, const float* max_yaw_rate,
                float dt, uint8_t* valid, uint8_t* disabled, uint8_t* navi_invalid, uint8_t* dest_reached,
                float* pose, float* motion, const uint8_t* gt_valid, const float* gt_pose, const float* gt_motion,
                const uint8_t* tf_mask, int n_gt, int sc_div, const float* boundary, const int32_t* dest_idx,
                const float* mp_pos, const float* mp_dirn, const uint8_t* mp_node_invalid, const uint8_t* mp_kind,
                int n_mp, int n_node, float thresh_lane, float thresh_edge, float cos_rot, const int* d_step, int B,
                int A, int W, int T, uint8_t* hist_valid, float* hist_pose, float* hist_motion, uint8_t* pred_valid,
                float* pred_pose, float* pred_motion, void* stream);
/* tb_dyn_step + the two per-step feedback flags RolloutBuffer.violation keeps (buffer.py:57-60):
 *   o_outside / o_reached [B,A,T] u8 (optional, NULL = not recorded): outside_map_this_step / dest_reached_this_step
 *   of step s at index s-1 (traffic_rule_checker.py:107-116, 291-319). */
int tb_dyn_step_ex(const float* act_branch, const uint8_t* ag_type, const float* max_acc, const float* max_yaw_rate,
                   float dt, uint8_t* valid, uint8_t* disabled, uint8_t* navi_invalid, uint8_t* dest_reached,
                   float* pose, float* motion, const uint8_t* gt_valid, const float* gt_pose, const float* gt_motion,
                   const uint8_t* tf_mask, int n_gt, int sc_div, const float* boundary, const int32_t* dest_idx,
                   const float* mp_pos, const float* mp_dirn, const uint8_t* mp_node_invalid, const uint8_t* mp_kind,
                   int n_mp, int n_node, float thresh_lane, float thresh_edge, float cos_rot, const int* d_step, int B,
                   int A, int W, int T, uint8_t* hist_valid, float* hist_pose, float* hist_motion, uint8_t* pred_valid,
                   float* pred_pose, float* pred_motion, uint8_t* o_outside, uint8_t* o_reached, void* stream);
/* tb_dyn_step_ex + the player override of Dynamics.update_ag (utils/dynamics.py:96-99, waymo_motion.py:206-217):
 *   player_valid [B*A] u8 (optional, NULL = no player; then the bits of tb_dyn_step_ex), player_action [B*A, T, 2]
 *   physical (acc m/s^2, yaw rate rad/s), required with player_valid. Step s of a valid, typed agent with
 *   player_valid set uses player_action[.., s-1, :] instead of the tanh-scaled action head; pred_* record that
 *   prediction, then teacher forcing and the outside-map / destination checks run unchanged. */
int tb_dyn_step_player(const float* act_branch, const uint8_t* ag_type, const float* max_acc,
                       const float* max_yaw_rate, float dt, uint8_t* valid, uint8_t* disabled, uint8_t* navi_invalid,
                       uint8_t* dest_reached, float* pose, float* motion, const uint8_t* gt_valid, const float* gt_pose,
                       const float* gt_motion, const uint8_t* tf_mask, int n_gt, int sc_div, const float* boundary,
                       const int32_t* dest_idx, const float* mp_pos, const float* mp_dirn,
                       const uint8_t* mp_node_invalid, const uint8_t* mp_kind, int n_mp, int n_node, float thresh_lane,
                       float thresh_edge, float cos_rot, const int* d_step, int B, int A, int W, int T,
                       uint8_t* hist_valid, float* hist_pose, float* hist_motion, uint8_t* pred_valid, float* pred_pose,
                       float* pred_motion, uint8_t* o_outside, uint8_t* o_reached, const uint8_t* player_valid,
                       const float* player_action, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Fused MLP chain (csrc/mlp_chain.cu): a sequence of dense layers over 128-row tiles with every intermediate kept on
 * the SM (tcgen05 MMAs, fp16 activation tiles in shared memory, fp32 accumulators in TMEM). One launch replaces the
 * head chain of a policy step — NaviEncoder.mlp_pe, AddNaviLatent x 2, ActionHead (models/traffic_bots.py:191-217,
 * modules/add_navi_latent.py:46-64, modules/action_head.py:78-82) — or the FFN of a transformer layer with its residual
 * and LayerNorm (modules/transformer_rpe.py:236-245).
 * A program is a list of units executed in order for every tile; `buffers` are on-chip fp16 tiles [128 rows x 128 cols]:
 *   kind 1 LOAD: rows of an external tensor (binding `src`, leading dim lds, first column src_col; fp32 or, with src_f16,
 *     IEEE fp16) -> buffer out_buf.
 *   kind 0 GEMM: acc[128 x 128] = A W[n0 : n0+128, :]^T with A = the 128-column buffers a_buf[0 .. K/128) side by side
 *     (K a multiple of 64, <= 512) and W [N, K] fp16 row-major (rows past N read as zero);
 *     v = acc + bias[n0 + c]; relu; if mask_pre[row]: 0; += res[row, res_col + c]; if mask_post[row]: 0 — the epilogue of
 *     tb_linear. v goes to buffer out_buf as fp16 (all 128 columns) and/or to fp32 rows out_g[row, g_col + c] and/or
 *     fp16 rows out_h[row, h_col + c], both for c < n_valid only (0 = 128); with ln_out, fp16(LayerNorm(v) * ln_gamma +
 *     ln_beta) of all 128 columns (eps 1e-5) goes to ln_out[row, c]. The residual rows are read for all 128 columns.
 *     fp16 conversions (LOAD of fp32, out_buf, out_h, ln_out) round to nearest and saturate at +-65504; a buffer or out_h
 *     value that reaches the bound sets the tb_set_fp16_flag word.
 * bias / ln_gamma / ln_beta / W are device pointers baked into the program (model constants; bias must hold n0 + 128
 * floats, ln_gamma / ln_beta 128, W / ln_gamma / ln_beta 16-byte aligned); mask_pre, mask_post, res, out_g, out_h,
 * ln_out, src are indices into the `bindings` array passed at run time.
 * Aliasing within one launch:
 *   - a LOAD source is read through the non-coherent cache (ld.global.nc): no unit of the launch may write what a LOAD
 *     reads. tb_chain_run refuses (TB_ERR_UNSUPPORTED) a LOAD whose binding pointer is also an out_g / out_h / ln_out
 *     binding unless both have the same row pitch and disjoint column ranges inside one row.
 *   - residual rows are read with plain loads, by the thread that owns the row slice [32 q, 32 q + 32) of the unit, so a
 *     residual may read what an EARLIER unit of the launch wrote through out_g at the same binding, leading dimension and
 *     column offset (the head chain: add_latent reads add_navi's output this way). Two units that touch the same global
 *     element must use the same binding, leading dimension and column offset; other overlaps race.
 * ------------------------------------------------------------------------------------------------- */
#define TB_CHAIN_MAX_UNITS 32
#define TB_CHAIN_MAX_KB 8
#define TB_CHAIN_MAX_BIND 16
typedef struct tb_chain_unit {
  int kind;
  const void* W; int K, N, n0;
  int a_buf[4];
  const float* bias; int relu, n_valid;
  int mask_pre, mask_post, res, ldr, res_col;
  int out_buf;
  int out_g, ldg, g_col;
  int out_h, ldh, h_col;
  int ln_out, ld_ln; const float* ln_gamma; const float* ln_beta;
  int src, lds, src_col, src_f16;
} tb_chain_unit;
int tb_chain_program_bytes(void);
/* host_blob: tb_chain_program_bytes() bytes of host memory; copy it to 128-byte aligned device memory afterwards.
 * n_buf: on-chip activation buffers, 2..5 (else TB_ERR_BAD_SHAPE). The rest of the 227 KB of shared memory is the weight
 * ring: (227 KB - 1 KB - 32 KB n_buf - 704 n_units - 4928) / 16 KB stages, at most 8, i.e.
 *   n_buf 2: 8 | 3: 7 (1-19 units), 6 (20-32) | 4: 5, 4 | 5: 3, 2 — n_stage, the 4th int of the host blob.
 * A GEMM unit waits for the last writer of each of its (at most 4) input buffers and, from the 5th GEMM on, for the
 * epilogue of the GEMM 4 earlier (the 4 TMEM accumulator regions are used in turn): at most 5 waits.
 * Errors: n_units outside 1..32, n_buf outside 2..5, out_buf >= n_buf, a binding index outside -1..14, a misshapen LOAD
 * (lds / src_col not multiples of 4 (fp32) or 8 (fp16)) or GEMM (K not a multiple of 64 or > 512, n0 >= N, n_valid
 * > 128), reading a buffer nobody wrote -> TB_ERR_BAD_SHAPE; misaligned W / bias / ln_gamma / ln_beta, ldr / res_col
 * not multiples of 4, ldh / h_col / ld_ln not multiples of 8, ln_out without gamma / beta -> TB_ERR_MISALIGNED; more than
 * 24 distinct (W, K, N) weights -> TB_ERR_UNSUPPORTED. All of these are returned before any device work. */
int tb_chain_encode(const tb_chain_unit* units, int n_units, int n_buf, void* host_blob);
/* bindings: HOST array of n_bind (<= 15) device pointers. Rows >= M of the last tile are neither read nor written.
 * Before the launch every binding the program uses is checked: index >= n_bind -> TB_ERR_BAD_SHAPE, NULL -> TB_ERR_NULL,
 * base not 16-byte aligned (LOAD sources, residual, out_h, ln_out, out_g with (ldg | g_col) % 4 == 0) or 4-byte aligned
 * (other out_g) -> TB_ERR_MISALIGNED, a LOAD source written by the launch (see Aliasing) -> TB_ERR_UNSUPPORTED. */
int tb_chain_run(const void* d_program, const void* host_blob, void* const* bindings, int n_bind, int M, void* stream);

/* Traffic-light feedback — utils/dynamics.py:144-163 (override_tl), traffic_light.py:286 (clamp +-3).
 *   logits [B*TL,5] (pre-clamp, invalid rows are zeroed here), tl_invalid [B,TL], gt_tl [B,TL,n_gt,5] u8.
 *   writes the new one-hot state into ring slot s%W of hist_tl [B,TL,W,5] and tl_out [B,TL,T,5] at s-1. */
int tb_tl_step(const float* logits, const uint8_t* tl_invalid, const uint8_t* gt_tl, int n_gt, const int* d_step,
               int B, int TL, int W, int T, uint8_t* hist_tl, uint8_t* tl_out, void* stream);
/* tb_tl_step + RolloutBuffer.tl_state_nll (waymo_motion.py:270-277): o_nll [B,TL,T] (optional) receives, at s-1,
 * -log_softmax(clamp(logits))[argmax gt state] while s < n_gt and 0 afterwards. */
int tb_tl_step_ex(const float* logits, const uint8_t* tl_invalid, const uint8_t* gt_tl, int n_gt, const int* d_step,
                  int B, int TL, int W, int T, uint8_t* hist_tl, uint8_t* tl_out, float* o_nll, void* stream);

/* Dynamics.update_ag of a stand-alone Dynamics object (utils/dynamics.py:66-120, MultiPathPP :237-274):
 *   action_unbounded [n,2] (mean or sample of the action distribution), ag_type [n,3] u8, valid [n] u8,
 *   player_valid [n] u8 / player_action [n,2] (optional override of the physical action, :96-99),
 *   max_acc[3], max_yaw_rate[3] (HOST arrays: veh, ped, cyc), dt; pose / motion [n,3] in;
 *   out_pose / out_motion [n,3], out_action [n,2] (physical action: m/s^2, rad/s). Invalid agents -> zeros. */
int tb_dyn_update(const float* action_unbounded, const uint8_t* ag_type, const uint8_t* valid,
                  const uint8_t* player_valid, const float* player_action, const float* max_acc,
                  const float* max_yaw_rate, float dt, int n, const float* pose, const float* motion, float* out_pose,
                  float* out_motion, float* out_action, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Logging-only traffic-rule checks of one step (SURVEY.md 8(f) rank 1) — TrafficRuleChecker.check
 * (utils/traffic_rule_checker.py:343-451): _check_collided (:119-149), check_collided_wosac
 * (utils/wosac_collision.py:196-239), _check_run_road_edge (:152-173), _check_run_red_light (:176-218),
 * _check_passive (:221-274). Evaluated on the step's prediction (pred_* at index s-1) and the traffic-light state
 * after override_tl (ring slot s%W). One CTA per rollout-scene.
 *   ag_size [B/sc_div,A,3] (length,width,height; collision boxes use size_scale = 1.1, :27), ag_type [B,A,3] u8
 *   per-scene map tables (:452-497): seg [B/sc_div,n_mp,n_node,4] = (pos, pos+dir), node_invalid [.,n_mp,n_node] u8,
 *   poly_circle [.,n_mp,3] = bounding circle (cx,cy,r) of each polyline's segments, poly_kind [.,n_mp] u8
 *   (bit0: road-edge types 4,5,7; bit1: lane-centre types 0..2)
 *   passive_counter [B,A] f32 (in/out); outputs "*_this_step" flags [B,A,T] u8 at index s-1.
 * Limit: A <= 256.
 * ------------------------------------------------------------------------------------------------- */
int tb_rule_check(const uint8_t* pred_valid, const float* pred_pose, const float* pred_motion, const uint8_t* ag_type,
                  const float* ag_size, const uint8_t* hist_tl, const uint8_t* tl_invalid, const float* tl_pose,
                  const float* seg, const uint8_t* node_invalid, const float* poly_circle, const uint8_t* poly_kind,
                  int n_mp, int n_node, float* passive_counter, uint8_t* o_collided, uint8_t* o_collided_wosac,
                  uint8_t* o_run_road_edge, uint8_t* o_run_red_light, uint8_t* o_passive, const int* d_step, int B, int A,
                  int T, int W, int n_tl, int sc_div, int tl_div, float size_scale, void* stream);

/* s <- s + 1 on the device (single thread); keeps the step graph replayable. */
int tb_step_advance(int* d_step, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Batched row copy (csrc/state_copy.cu): the rollout engine's snapshot / restore / fork of its device state in one
 * launch. Item i copies n_rows rows of row_bytes bytes from src to dst (both dense). With `src_rollout` (int32, one
 * entry per row of the longest per-rollout item) every item with per_rollout != 0 is a row gather over the R rollouts
 * of a scene: row b = sc * R + r of dst receives row sc * R + src_rollout[b] of src; an entry outside [0, R) copies
 * row b itself (defined, never an out-of-range read). Other items, and all items when src_rollout is NULL, are plain
 * copies. Accesses are 16 bytes wide where src, dst and row_bytes allow it, narrower otherwise. Items must not
 * overlap each other. The item table travels in the kernel parameters: no allocation, no synchronisation.
 * Errors: items / src / dst NULL -> TB_ERR_NULL; n_items outside 1..TB_COPY_ROWS_MAX, row_bytes or n_rows <= 0, a
 * per-rollout item with R <= 0 or n_rows not a multiple of R -> TB_ERR_BAD_SHAPE; a gathered item with src == dst
 * (rows would be overwritten before they are read) or of 2^32 access units or more -> TB_ERR_UNSUPPORTED.
 * ------------------------------------------------------------------------------------------------- */
#define TB_COPY_ROWS_MAX 64
typedef struct tb_row_copy_t {
  const void* src;
  void* dst;
  long long row_bytes;
  int n_rows;
  int per_rollout;
} tb_row_copy_t;
int tb_copy_rows(const tb_row_copy_t* items, int n_items, const int32_t* src_rollout, int R, void* stream);

/* Gather rows: out[m, 0:C] = table[(m / rows_per_batch / div) * T + idx[m], 0:C] — navigation.py:69,
 * traffic_light.py:115. */
int tb_gather_rows(const float* table, int ldt, int T, const int32_t* idx, int M, int rows_per_batch, int div, int C,
                   float* out, int ldo, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * WOSAC post-processing on the device (the step right after the loop; SURVEY.md 8(f) rank 4).
 * tb_future_filter — data_modules/wosac_post_processing.py:31-64 (`_filter_futures`): per joint future k of scene sc
 *   score[sc,k] = sum_a role_any[sc,a] * any_{t>=t0} collided[(sc K + k), a, t]
 *               + w_road_edge * sum_a role_any[sc,a] * any_{t>=t0} run_road_edge[...]
 *   and sel[sc, 0:n_keep] = the n_keep futures with the smallest score, ascending by (score, index) (the reference's
 *   torch.topk(sorted=False) leaves order and tie-break unspecified). Flags [n_sc*K, A, T] u8 as written by
 *   tb_rule_check; role_any [n_sc, A] u8; score [n_sc, K] f32, sel [n_sc, n_keep] i32. K <= 1024.
 * tb_traj_global — wosac_post_processing.py:66-75 with transform_utils.py:160-171,215-225: gathers the selected
 *   futures (sel NULL: all K in order) and maps them to the global frame:
 *   out_pos[sc,i,a,t,:] = R(yaw[sc]) pose_xy[(sc K + sel[sc,i]), a, t0+t] + center[sc];
 *   out_yaw[sc,i,a,t] = wrap_[-pi,pi)(pose_yaw + yaw[sc]). pose [n_sc*K, A, T, 3]; out_pos [n_sc,n_keep,A,T-t0,2].
 * ------------------------------------------------------------------------------------------------- */
int tb_future_filter(const uint8_t* collided, const uint8_t* run_road_edge, const uint8_t* role_any, int n_sc, int K,
                     int A, int T, int t0, float w_road_edge, int n_keep, float* score, int32_t* sel, void* stream);
int tb_traj_global(const float* pose, const int32_t* sel, const float* center, const float* yaw, int n_sc, int K,
                   int n_keep, int A, int T, int t0, float* out_pos, float* out_yaw, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * WOMD post-processing on the device (SURVEY.md 8(f) rank 4) — data_modules/womd_post_processing.py:36-106 with the
 * configured parameters of configs/model/sim_agent.yaml:170-177 (top-k + `mpa_nms`; `mtr_nms` / `traj_aggr` are not
 * configured and not built). Per (scene, agent):
 *   p = softmax_k(scores[sc, k, a])                (scores NULL: uniform)                               :48-53
 *   K > k_pred: keep the k_pred most probable futures (descending p, ties by lower index; the reference's
 *     topk(sorted=False) leaves the order unspecified) and renormalise                                   :170-190
 *   nms_on: d(m,n) = mean_t |xy_m(t) - xy_n(t)| (use_ade) or the distance at the last step; visiting the modes in
 *     descending score order, a mode with d < thresh(type) to a currently higher-scored mode drops to 1e-3; then
 *     renormalise. thresh = sum_i ag_type[sc,a,i] * thr_i                                                :75-106
 *   score_temperature > 0: p = softmax(log p / temperature)                                              :66-67
 *   out_trajs[sc, a, m, j, :] = trajs[sc, mode m, a, t_first + j * t_stride, :], t < min(t_end, T)      :69
 * trajs [n_sc, K, A, T, 3] f32 (the rollout's layout), scores [n_sc, K, A] f32 log-probs, ag_type [n_sc, A, 3] u8;
 * out_trajs [n_sc, A, k, n_out, 3], out_scores / out_mode (may be NULL) [n_sc, A, k] with k = min(K, k_pred).
 * Limits: K <= 128, k_pred <= 8 (TB_ERR_UNSUPPORTED).
 * ------------------------------------------------------------------------------------------------- */
int tb_womd_post(const float* trajs, const float* scores, const uint8_t* ag_type, int n_sc, int K, int A, int T,
                 int k_pred, int use_ade, int nms_on, float thr_veh, float thr_ped, float thr_cyc,
                 float score_temperature, int t_first, int t_stride, int t_end, float* out_trajs, float* out_scores,
                 int32_t* out_mode, void* stream);

/* Sum of the three type-masked branches is done inside tb_dyn_step; this helper exposes the masked action
 * mean [B,A,2] for the module-level API (action_head.py:78-82). */
int tb_action_mean(const float* act_branch, const uint8_t* ag_type, const uint8_t* valid, int M, float* mean,
                   void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TB_KNARPE_H_ */
