// Per-step closed-loop kernels: history featurisation, dynamics + teacher forcing + feedback checks, TL feedback.
// Rollout state lives in HBM ring buffers for the whole rollout (slot = time % W); the loop counter is a device
// scalar so one captured CUDA graph replays for all 90 steps (no host sync, cf. the .any() syncs of the reference:
// attention_rpe.py:115, dynamics.py:136,161,179).
#include "common.cuh"

namespace {

__device__ __forceinline__ float pe_component64(int c, float x, float y, float w, const float* __restrict__ freq_xy) {
  // PoseEmb pe_dim = 64 (agent_encoder.py:50): [cos(x f0..7)|sin(x f)|cos(y f)|sin(y f)|cos(w 1..16)|sin(w 1..16)]
  float a;
  bool is_sin;
  if (c < 16) { a = x * __ldg(freq_xy + (c & 7)); is_sin = c >= 8; }
  else if (c < 32) { a = y * __ldg(freq_xy + (c & 7)); is_sin = c >= 24; }
  else { a = w * (float)(((c - 32) & 15) + 1); is_sin = c >= 48; }
  const float r = tb_reduce_2pi(a);
  return is_sin ? __sinf(r) : __cosf(r);
}

// one warp per (b, agent)
__global__ void __launch_bounds__(256)
ag_featurize_kernel(const uint8_t* __restrict__ hist_valid, const float* __restrict__ hist_pose,
                    const float* __restrict__ hist_motion, const float* __restrict__ ag_attr,
                    const int* __restrict__ d_step, int step_stride, int A, const float* __restrict__ freq_xy,
                    int n_ag_tot, int W, float* __restrict__ tok_pose, uint8_t* __restrict__ tok_invalid,
                    uint8_t* __restrict__ row_invalid, float* __restrict__ attr_out, int lda,
                    float* __restrict__ pe_out, int ldpe) {
  const int ba = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (ba >= n_ag_tot) return;
  const int s = d_step[step_stride ? (size_t)(ba / A) * step_stride : 0];  // one step for all, or one per batch row
  const int n_step = min(s, W);
  const size_t hb = (size_t)ba * W;
  // window position wp in [W-n_step, W) <-> time t = s - W + wp, slot t % W ; wp < W-n_step: absent
  int last_wp = -1;
  for (int wp = W - n_step; wp < W; ++wp) {
    const int t = s - W + wp;
    if (hist_valid[hb + (t % W)]) last_wp = wp;
  }
  float px = 0.f, py = 0.f, pw = 0.f;
  if (last_wp >= 0) {
    const int slot = (s - W + last_wp) % W;
    px = hist_pose[(hb + slot) * 3];
    py = hist_pose[(hb + slot) * 3 + 1];
    pw = hist_pose[(hb + slot) * 3 + 2];
  }
  if (lane == 0) {
    tok_pose[(size_t)ba * 3] = px; tok_pose[(size_t)ba * 3 + 1] = py; tok_pose[(size_t)ba * 3 + 2] = pw;
    tok_invalid[ba] = last_wp < 0;
  }
  if (!attr_out) return;  // token-only mode (the fused front-end builds the rows itself)
  float sn, cs;
  sincosf(pw, &sn, &cs);
  for (int wp = 0; wp < W; ++wp) {
    const size_t orow = hb + wp;
    const bool present = wp >= W - n_step;
    const int slot = present ? (s - W + wp) % W : 0;
    const bool valid = present && hist_valid[hb + slot];
    if (lane == 0) row_invalid[orow] = !valid;
    // attr row: [attr6 | motion3 | one-hot W]
    float* ar = attr_out + orow * lda;
    if (lane < 6) ar[lane] = present ? ag_attr[(size_t)ba * 6 + lane] : 0.f;
    else if (lane < 9) ar[lane] = present ? hist_motion[(hb + slot) * 3 + (lane - 6)] : 0.f;
    else if (lane < 9 + W) ar[lane] = (present && (lane - 9) == wp) ? 1.f : 0.f;
    // pose embedding of the history pose in the token frame (agent_encoder.py:147-148,159)
    float x = 0.f, y = 0.f, w = 0.f;
    if (present) {
      const float dx = hist_pose[(hb + slot) * 3] - px, dy = hist_pose[(hb + slot) * 3 + 1] - py;
      x = fmaf(dx, cs, dy * sn);
      y = fmaf(dy, cs, -dx * sn);
      w = hist_pose[(hb + slot) * 3 + 2] - pw;
    }
    float* pr = pe_out + orow * ldpe;
    pr[lane] = pe_component64(lane, x, y, w, freq_xy);
    pr[lane + 32] = pe_component64(lane + 32, x, y, w, freq_xy);
  }
}

__global__ void tl_featurize_kernel(const uint8_t* __restrict__ hist_tl, const uint8_t* __restrict__ tl_invalid,
                                    const int* __restrict__ d_step, int step_stride, int TL, int n_rows, int W,
                                    float* __restrict__ attr_out, int lda, uint8_t* __restrict__ row_invalid) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;  // (b*TL + tl)*W + wp
  if (i >= n_rows) return;
  const int wp = i % W, bt = i / W;
  const int s = d_step[step_stride ? (size_t)(bt / TL) * step_stride : 0];
  const int n_step = min(s, W);
  const bool present = wp >= W - n_step;
  const int slot = present ? (s - W + wp) % W : 0;
  float* ar = attr_out + (size_t)i * lda;
#pragma unroll
  for (int c = 0; c < 5; ++c) ar[c] = present ? (float)hist_tl[((size_t)bt * W + slot) * 5 + c] : 0.f;
  for (int c = 0; c < W; ++c) ar[5 + c] = (present && c == wp) ? 1.f : 0.f;
  row_invalid[i] = !present || tl_invalid[bt];
}

struct DynArgs {
  const float* act_branch; const uint8_t* ag_type; float max_acc[3]; float max_yaw[3]; float dt;
  uint8_t* valid; uint8_t* disabled; uint8_t* navi_invalid; uint8_t* dest_reached; float* pose; float* motion;
  const uint8_t* gt_valid; const float* gt_pose; const float* gt_motion; const uint8_t* tf_mask; int n_gt; int sc_div;
  const float* boundary; const int32_t* dest_idx; const float* mp_pos; const float* mp_dirn;
  const uint8_t* mp_node_invalid; const uint8_t* mp_kind; int n_mp; int n_node; float thresh_lane; float thresh_edge;
  float cos_rot; const int* d_step; int n_tot; int A; int W; int T;
  uint8_t* hist_valid; float* hist_pose; float* hist_motion; uint8_t* pred_valid; float* pred_pose; float* pred_motion;
  uint8_t* o_outside; uint8_t* o_reached;  // optional [B,A,T]: outside_map_this_step / dest_reached_this_step (buffer.py:57-60)
  const uint8_t* player_valid; const float* player_action;  // optional [B*A] / [B*A,T,2]: player override (dynamics.py:96-99)
};

__global__ void __launch_bounds__(128) dyn_step_kernel(DynArgs p) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;  // b*A + a
  if (i >= p.n_tot) return;
  const int s = *p.d_step;
  if (s < 1 || s > p.T) return;  // pred_*[.., s - 1] would be out of bounds: the step counter ran past step_end
  const int b = i / p.A, a = i - b * p.A, sc = b / p.sc_div;
  const bool v_old = p.valid[i] != 0;
  // ---- action head branches -> physical action (action_head.py:78-82, dynamics.py:84-101, :237-246)
  int type = -1;
#pragma unroll
  for (int t = 0; t < 3; ++t) if (p.ag_type[(size_t)i * 3 + t]) type = t;  // one-hot
  float acc = 0.f, yr = 0.f;
  if (v_old && type >= 0) {
    acc = tanhf(p.act_branch[(size_t)i * 6 + type * 2 + 0]) * p.max_acc[type];
    yr = tanhf(p.act_branch[(size_t)i * 6 + type * 2 + 1]) * p.max_yaw[type];
    if (p.player_valid && p.player_valid[i]) {  // the player's physical action replaces the policy's (dynamics.py:96-99)
      const size_t o = ((size_t)i * p.T + (s - 1)) * 2;
      acc = p.player_action[o];
      yr = p.player_action[o + 1];
    }
  }
  // ---- MultiPathPP.update (dynamics.py:248-274), same operation order as the reference (no FMA contraction)
  float x = p.pose[(size_t)i * 3], y = p.pose[(size_t)i * 3 + 1], w = p.pose[(size_t)i * 3 + 2];
  float spd = p.motion[(size_t)i * 3];
  const float hdt = 0.5f * p.dt;
  const float v_t = __fadd_rn(spd, __fmul_rn(hdt, acc));
  const float th_t = __fadd_rn(w, __fmul_rn(hdt, yr));
  float sn, cs;
  sincosf(th_t, &sn, &cs);
  float nx = __fadd_rn(x, __fmul_rn(p.dt, __fmul_rn(v_t, cs)));
  float ny = __fadd_rn(y, __fmul_rn(p.dt, __fmul_rn(v_t, sn)));
  float nw = __fadd_rn(w, __fmul_rn(p.dt, yr));
  float nspd = __fadd_rn(spd, __fmul_rn(p.dt, acc));
  float nacc = acc, nyr = yr;
  if (!(v_old && type >= 0)) { nx = ny = nw = nspd = nacc = nyr = 0.f; }  // dynamics.py:108-119
  // ---- record prediction (buffer.py:54-56): index s-1
  {
    const size_t o = (size_t)i * p.T + (s - 1);
    p.pred_valid[o] = v_old;
    p.pred_pose[o * 3] = nx; p.pred_pose[o * 3 + 1] = ny; p.pred_pose[o * 3 + 2] = nw;
    p.pred_motion[o * 3] = nspd; p.pred_motion[o * 3 + 1] = nacc; p.pred_motion[o * 3 + 2] = nyr;
  }
  // ---- feedback checks on the prediction (traffic_rule_checker.py:107-116, 291-319)
  const float* bd = p.boundary + (size_t)sc * 4;
  const bool outside = v_old && ((nx > bd[1]) || (nx < bd[0]) || (ny > bd[3]) || (ny < bd[2]));
  bool reached = false;
  if (v_old && !p.dest_reached[i]) {
    const int di = p.dest_idx[i];
    const size_t mrow = (size_t)sc * p.n_mp + di;
    const int kind = p.mp_kind[mrow];
    if (kind) {
      const float thr = kind == 2 ? p.thresh_edge : p.thresh_lane;
      float hs, hc;
      sincosf(nw, &hs, &hc);
      bool pos_ok = false, rot_ok = false;
      for (int n = 0; n < p.n_node; ++n) {
        const size_t q = mrow * p.n_node + n;
        if (p.mp_node_invalid[q]) continue;
        const float dx = nx - p.mp_pos[q * 2], dy = ny - p.mp_pos[q * 2 + 1];
        pos_ok |= sqrtf(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy))) < thr;
        rot_ok |= __fadd_rn(__fmul_rn(hc, p.mp_dirn[q * 2]), __fmul_rn(hs, p.mp_dirn[q * 2 + 1])) > p.cos_rot;
      }
      reached = kind == 2 ? pos_ok : (pos_ok && rot_ok);
    }
  }
  if (p.o_outside) p.o_outside[(size_t)i * p.T + (s - 1)] = outside;
  if (p.o_reached) p.o_reached[(size_t)i * p.T + (s - 1)] = reached;
  // ---- teacher forcing / spawn override (teacher_forcing.py:126-147, dynamics.py:122-141)
  bool v_new = v_old;
  const bool dis_old = p.disabled[i] != 0;
  bool gtv = false;
  if (s < p.n_gt) {
    const size_t g = ((size_t)sc * p.A + a) * p.n_gt + s;
    gtv = p.gt_valid[g] != 0;
    if (p.tf_mask[g] && !dis_old) {
      v_new = true;
      nx = p.gt_pose[g * 3]; ny = p.gt_pose[g * 3 + 1]; nw = p.gt_pose[g * 3 + 2];
      nspd = p.gt_motion[g * 3]; nacc = p.gt_motion[g * 3 + 1]; nyr = p.gt_motion[g * 3 + 2];
    }
  }
  // ---- disable agents outside the map / navigation reached (dynamics.py:166-204)
  const bool dis = outside && !(s < p.n_gt && gtv);
  if (dis) { p.disabled[i] = 1; v_new = false; }
  if (reached) { p.dest_reached[i] = 1; p.navi_invalid[i] = 1; }
  p.valid[i] = v_new;
  p.pose[(size_t)i * 3] = nx; p.pose[(size_t)i * 3 + 1] = ny; p.pose[(size_t)i * 3 + 2] = nw;
  p.motion[(size_t)i * 3] = nspd; p.motion[(size_t)i * 3 + 1] = nacc; p.motion[(size_t)i * 3 + 2] = nyr;
  // ---- history ring (traffic_bots.py:123-143): state at time s
  const size_t h = (size_t)i * p.W + (s % p.W);
  p.hist_valid[h] = v_new;
  p.hist_pose[h * 3] = nx; p.hist_pose[h * 3 + 1] = ny; p.hist_pose[h * 3 + 2] = nw;
  p.hist_motion[h * 3] = nspd; p.hist_motion[h * 3 + 1] = nacc; p.hist_motion[h * 3 + 2] = nyr;
}

__global__ void tl_step_kernel(const float* __restrict__ logits, const uint8_t* __restrict__ tl_invalid,
                               const uint8_t* __restrict__ gt_tl, int n_gt, const int* __restrict__ d_step, int n_tot,
                               int W, int T, uint8_t* __restrict__ hist_tl, uint8_t* __restrict__ tl_out,
                               float* __restrict__ o_nll) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;  // b*TL + tl
  if (i >= n_tot) return;
  const int s = *d_step;
  if (s < 1 || s > T) return;  // tl_out[.., s - 1] would be out of bounds
  uint8_t st[5];
  if (o_nll) {  // tl_state_nll of the step (waymo_motion.py:270-277): -log_softmax(clamped logits)[gt state], 0 past the gt
    float nll = 0.f;
    if (s < n_gt) {
      const bool inv = tl_invalid[i] != 0;
      float v[5], mx = -INFINITY;
      int gt = 0;
#pragma unroll
      for (int c = 0; c < 5; ++c) {
        v[c] = inv ? 0.f : fminf(fmaxf(logits[(size_t)i * 5 + c], -3.f), 3.f);
        mx = fmaxf(mx, v[c]);
      }
      uint8_t best = 0;
#pragma unroll
      for (int c = 0; c < 5; ++c) {  // max(-1)[1] of a bool one-hot: first maximal entry
        const uint8_t g = gt_tl[((size_t)i * n_gt + s) * 5 + c];
        if (g > best) { best = g; gt = c; }
      }
      float se = 0.f;
#pragma unroll
      for (int c = 0; c < 5; ++c) se += expf(v[c] - mx);
      nll = -(v[gt] - mx - logf(se));
    }
    o_nll[(size_t)i * T + (s - 1)] = nll;
  }
  if (s < n_gt) {  // ground-truth traffic lights while available (teacher_forcing.py:65,159-160)
#pragma unroll
    for (int c = 0; c < 5; ++c) st[c] = gt_tl[((size_t)i * n_gt + s) * 5 + c];
  } else {  // one-hot(argmax softmax(clamp(logits, +-3))) (traffic_light.py:285-286, dynamics.py:154-159)
    int best = 0;
    float bv = -INFINITY;
    const bool inv = tl_invalid[i] != 0;
#pragma unroll
    for (int c = 0; c < 5; ++c) {
      float v = inv ? 0.f : fminf(fmaxf(logits[(size_t)i * 5 + c], -3.f), 3.f);
      if (v > bv) { bv = v; best = c; }
    }
#pragma unroll
    for (int c = 0; c < 5; ++c) st[c] = c == best;
  }
#pragma unroll
  for (int c = 0; c < 5; ++c) {
    hist_tl[((size_t)i * W + (s % W)) * 5 + c] = st[c];
    tl_out[((size_t)i * T + (s - 1)) * 5 + c] = st[c];
  }
}

__global__ void step_advance_kernel(int* d_step) { *d_step += 1; }

__global__ void action_mean_kernel(const float* __restrict__ act_branch, const uint8_t* __restrict__ ag_type,
                                   const uint8_t* __restrict__ valid, int M, float* __restrict__ mean) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M) return;
  float m0 = 0.f, m1 = 0.f;
  if (valid[i]) {
#pragma unroll
    for (int t = 0; t < 3; ++t)
      if (ag_type[(size_t)i * 3 + t]) { m0 += act_branch[(size_t)i * 6 + t * 2]; m1 += act_branch[(size_t)i * 6 + t * 2 + 1]; }
  }
  mean[(size_t)i * 2] = m0;
  mean[(size_t)i * 2 + 1] = m1;
}

}  // namespace

extern "C" int tb_ag_featurize_ex(const uint8_t* hist_valid, const float* hist_pose, const float* hist_motion,
                                  const float* ag_attr, const int* d_step, int step_stride, const float* freq_xy, int B,
                                  int A, int W, float* tok_pose, uint8_t* tok_invalid, uint8_t* row_invalid,
                                  float* attr_out, int lda, float* pe_out, int ldpe, void* stream) {
  if (!hist_valid || !hist_pose || !hist_motion || !ag_attr || !d_step || !freq_xy || !tok_pose || !tok_invalid)
    return TB_ERR_NULL;
  const bool rows = attr_out || pe_out || row_invalid;  // all three or none (none: token pose / validity only)
  if (rows && (!row_invalid || !attr_out || !pe_out)) return TB_ERR_NULL;
  if (B <= 0 || A <= 0 || W <= 0 || W > 23 || step_stride < 0 || (rows && (lda < 9 + W || ldpe < 64)))
    return TB_ERR_BAD_SHAPE;
  const int n = B * A;
  ag_featurize_kernel<<<(n + 7) / 8, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      hist_valid, hist_pose, hist_motion, ag_attr, d_step, step_stride, A, freq_xy, n, W, tok_pose, tok_invalid,
      row_invalid, attr_out, lda, pe_out, ldpe);
  TB_CHECK_LAUNCH();
  return TB_OK;
}

extern "C" int tb_ag_featurize(const uint8_t* hist_valid, const float* hist_pose, const float* hist_motion,
                               const float* ag_attr, const int* d_step, const float* freq_xy, int B, int A, int W,
                               float* tok_pose, uint8_t* tok_invalid, uint8_t* row_invalid, float* attr_out, int lda,
                               float* pe_out, int ldpe, void* stream) {
  return tb_ag_featurize_ex(hist_valid, hist_pose, hist_motion, ag_attr, d_step, 0, freq_xy, B, A, W, tok_pose,
                            tok_invalid, row_invalid, attr_out, lda, pe_out, ldpe, stream);
}

extern "C" int tb_tl_featurize_ex(const uint8_t* hist_tl, const uint8_t* tl_invalid, const int* d_step, int step_stride,
                                  int B, int TL, int W, float* attr_out, int lda, uint8_t* row_invalid, void* stream) {
  if (!hist_tl || !tl_invalid || !d_step || !attr_out || !row_invalid) return TB_ERR_NULL;
  if (B <= 0 || TL <= 0 || W <= 0 || lda < 5 + W || step_stride < 0) return TB_ERR_BAD_SHAPE;
  const int n = B * TL * W;
  tl_featurize_kernel<<<(n + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      hist_tl, tl_invalid, d_step, step_stride, TL, n, W, attr_out, lda, row_invalid);
  TB_CHECK_LAUNCH();
  return TB_OK;
}

extern "C" int tb_tl_featurize(const uint8_t* hist_tl, const uint8_t* tl_invalid, const int* d_step, int B, int TL,
                               int W, float* attr_out, int lda, uint8_t* row_invalid, void* stream) {
  return tb_tl_featurize_ex(hist_tl, tl_invalid, d_step, 0, B, TL, W, attr_out, lda, row_invalid, stream);
}

extern "C" int tb_dyn_step_player(const float* act_branch, const uint8_t* ag_type, const float* max_acc,
                                  const float* max_yaw_rate, float dt, uint8_t* valid, uint8_t* disabled,
                                  uint8_t* navi_invalid, uint8_t* dest_reached, float* pose, float* motion,
                                  const uint8_t* gt_valid, const float* gt_pose, const float* gt_motion,
                                  const uint8_t* tf_mask, int n_gt, int sc_div, const float* boundary,
                                  const int32_t* dest_idx, const float* mp_pos, const float* mp_dirn,
                                  const uint8_t* mp_node_invalid, const uint8_t* mp_kind, int n_mp, int n_node,
                                  float thresh_lane, float thresh_edge, float cos_rot, const int* d_step, int B, int A,
                                  int W, int T, uint8_t* hist_valid, float* hist_pose, float* hist_motion,
                                  uint8_t* pred_valid, float* pred_pose, float* pred_motion, uint8_t* o_outside,
                                  uint8_t* o_reached, const uint8_t* player_valid, const float* player_action,
                                  void* stream) {
  if (!act_branch || !ag_type || !max_acc || !max_yaw_rate || !valid || !disabled || !navi_invalid || !dest_reached ||
      !pose || !motion || !gt_valid || !gt_pose || !gt_motion || !tf_mask || !boundary || !dest_idx || !mp_pos ||
      !mp_dirn || !mp_node_invalid || !mp_kind || !d_step || !hist_valid || !hist_pose || !hist_motion || !pred_valid ||
      !pred_pose || !pred_motion || (player_valid && !player_action))
    return TB_ERR_NULL;
  if (B <= 0 || A <= 0 || W <= 0 || T <= 0 || n_gt <= 0 || sc_div <= 0 || n_mp <= 0 || n_node <= 0)
    return TB_ERR_BAD_SHAPE;
  DynArgs p;
  p.act_branch = act_branch; p.ag_type = ag_type;
  for (int t = 0; t < 3; ++t) { p.max_acc[t] = max_acc[t]; p.max_yaw[t] = max_yaw_rate[t]; }  // host arrays
  p.dt = dt; p.valid = valid; p.disabled = disabled; p.navi_invalid = navi_invalid; p.dest_reached = dest_reached;
  p.pose = pose; p.motion = motion; p.gt_valid = gt_valid; p.gt_pose = gt_pose; p.gt_motion = gt_motion;
  p.tf_mask = tf_mask; p.n_gt = n_gt; p.sc_div = sc_div; p.boundary = boundary; p.dest_idx = dest_idx;
  p.mp_pos = mp_pos; p.mp_dirn = mp_dirn; p.mp_node_invalid = mp_node_invalid; p.mp_kind = mp_kind; p.n_mp = n_mp;
  p.n_node = n_node; p.thresh_lane = thresh_lane; p.thresh_edge = thresh_edge; p.cos_rot = cos_rot; p.d_step = d_step;
  p.n_tot = B * A; p.A = A; p.W = W; p.T = T; p.hist_valid = hist_valid; p.hist_pose = hist_pose;
  p.hist_motion = hist_motion; p.pred_valid = pred_valid; p.pred_pose = pred_pose; p.pred_motion = pred_motion;
  p.o_outside = o_outside; p.o_reached = o_reached; p.player_valid = player_valid; p.player_action = player_action;
  dyn_step_kernel<<<(p.n_tot + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(p);
  TB_CHECK_LAUNCH();
  return TB_OK;
}

extern "C" int tb_dyn_step_ex(const float* act_branch, const uint8_t* ag_type, const float* max_acc,
                              const float* max_yaw_rate, float dt, uint8_t* valid, uint8_t* disabled, uint8_t* navi_invalid,
                              uint8_t* dest_reached, float* pose, float* motion, const uint8_t* gt_valid,
                              const float* gt_pose, const float* gt_motion, const uint8_t* tf_mask, int n_gt, int sc_div,
                              const float* boundary, const int32_t* dest_idx, const float* mp_pos, const float* mp_dirn,
                              const uint8_t* mp_node_invalid, const uint8_t* mp_kind, int n_mp, int n_node,
                              float thresh_lane, float thresh_edge, float cos_rot, const int* d_step, int B, int A, int W,
                              int T, uint8_t* hist_valid, float* hist_pose, float* hist_motion, uint8_t* pred_valid,
                              float* pred_pose, float* pred_motion, uint8_t* o_outside, uint8_t* o_reached, void* stream) {
  return tb_dyn_step_player(act_branch, ag_type, max_acc, max_yaw_rate, dt, valid, disabled, navi_invalid, dest_reached,
                            pose, motion, gt_valid, gt_pose, gt_motion, tf_mask, n_gt, sc_div, boundary, dest_idx, mp_pos,
                            mp_dirn, mp_node_invalid, mp_kind, n_mp, n_node, thresh_lane, thresh_edge, cos_rot, d_step, B,
                            A, W, T, hist_valid, hist_pose, hist_motion, pred_valid, pred_pose, pred_motion, o_outside,
                            o_reached, nullptr, nullptr, stream);
}

extern "C" int tb_dyn_step(const float* act_branch, const uint8_t* ag_type, const float* max_acc,
                           const float* max_yaw_rate, float dt, uint8_t* valid, uint8_t* disabled, uint8_t* navi_invalid,
                           uint8_t* dest_reached, float* pose, float* motion, const uint8_t* gt_valid,
                           const float* gt_pose, const float* gt_motion, const uint8_t* tf_mask, int n_gt, int sc_div,
                           const float* boundary, const int32_t* dest_idx, const float* mp_pos, const float* mp_dirn,
                           const uint8_t* mp_node_invalid, const uint8_t* mp_kind, int n_mp, int n_node,
                           float thresh_lane, float thresh_edge, float cos_rot, const int* d_step, int B, int A, int W,
                           int T, uint8_t* hist_valid, float* hist_pose, float* hist_motion, uint8_t* pred_valid,
                           float* pred_pose, float* pred_motion, void* stream) {
  return tb_dyn_step_ex(act_branch, ag_type, max_acc, max_yaw_rate, dt, valid, disabled, navi_invalid, dest_reached, pose,
                        motion, gt_valid, gt_pose, gt_motion, tf_mask, n_gt, sc_div, boundary, dest_idx, mp_pos, mp_dirn,
                        mp_node_invalid, mp_kind, n_mp, n_node, thresh_lane, thresh_edge, cos_rot, d_step, B, A, W, T,
                        hist_valid, hist_pose, hist_motion, pred_valid, pred_pose, pred_motion, nullptr, nullptr, stream);
}

extern "C" int tb_tl_step_ex(const float* logits, const uint8_t* tl_invalid, const uint8_t* gt_tl, int n_gt,
                             const int* d_step, int B, int TL, int W, int T, uint8_t* hist_tl, uint8_t* tl_out,
                             float* o_nll, void* stream) {
  if (!logits || !tl_invalid || !gt_tl || !d_step || !hist_tl || !tl_out) return TB_ERR_NULL;
  if (B <= 0 || TL <= 0 || W <= 0 || T <= 0 || n_gt <= 0) return TB_ERR_BAD_SHAPE;
  const int n = B * TL;
  tl_step_kernel<<<(n + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(logits, tl_invalid, gt_tl, n_gt, d_step,
                                                                               n, W, T, hist_tl, tl_out, o_nll);
  TB_CHECK_LAUNCH();
  return TB_OK;
}

extern "C" int tb_tl_step(const float* logits, const uint8_t* tl_invalid, const uint8_t* gt_tl, int n_gt,
                          const int* d_step, int B, int TL, int W, int T, uint8_t* hist_tl, uint8_t* tl_out,
                          void* stream) {
  return tb_tl_step_ex(logits, tl_invalid, gt_tl, n_gt, d_step, B, TL, W, T, hist_tl, tl_out, nullptr, stream);
}

// Dynamics.update_ag for a stand-alone Dynamics object (utils/dynamics.py:66-120 + MultiPathPP :237-274): unbounded
// action (the distribution's mean or sample) -> physical action per agent type -> optional player override ->
// unicycle update; invalid agents and agents without a type come out as zeros (:108-119).
__global__ void dyn_update_kernel(const float* __restrict__ act, const uint8_t* __restrict__ ag_type,
                                  const uint8_t* __restrict__ valid, const uint8_t* __restrict__ player_valid,
                                  const float* __restrict__ player_action, float3 max_acc, float3 max_yaw, float dt, int n,
                                  const float* __restrict__ pose, const float* __restrict__ motion,
                                  float* __restrict__ o_pose, float* __restrict__ o_motion, float* __restrict__ o_action) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const bool v = valid[i] != 0;
  const float ma[3] = {max_acc.x, max_acc.y, max_acc.z}, my[3] = {max_yaw.x, max_yaw.y, max_yaw.z};
  float acc = 0.f, yr = 0.f, n_type = 0.f;
  const float t0 = tanhf(act[(size_t)i * 2]), t1 = tanhf(act[(size_t)i * 2 + 1]);
#pragma unroll
  for (int t = 0; t < 3; ++t)
    if (ag_type[(size_t)i * 3 + t]) { acc += t0 * ma[t]; yr += t1 * my[t]; n_type += 1.f; }  // masked sum over the types
  if (!v) { acc = 0.f; yr = 0.f; }
  if (player_valid && player_valid[i] && v) { acc = player_action[(size_t)i * 2]; yr = player_action[(size_t)i * 2 + 1]; }
  const float x = pose[(size_t)i * 3], y = pose[(size_t)i * 3 + 1], w = pose[(size_t)i * 3 + 2], spd = motion[(size_t)i * 3];
  const float hdt = 0.5f * dt;
  const float v_t = __fadd_rn(spd, __fmul_rn(hdt, acc)), th_t = __fadd_rn(w, __fmul_rn(hdt, yr));
  float sn, cs;
  sincosf(th_t, &sn, &cs);
  // every type's MultiPathPP.update gives the same state; the masked sum over types multiplies it by the type count
  float nx = __fadd_rn(x, __fmul_rn(dt, __fmul_rn(v_t, cs))) * n_type, ny = __fadd_rn(y, __fmul_rn(dt, __fmul_rn(v_t, sn))) * n_type;
  float nw = __fadd_rn(w, __fmul_rn(dt, yr)) * n_type, nspd = __fadd_rn(spd, __fmul_rn(dt, acc)) * n_type;
  float nacc = acc * n_type, nyr = yr * n_type;
  if (!v) { nx = ny = nw = nspd = nacc = nyr = 0.f; }
  o_pose[(size_t)i * 3] = nx; o_pose[(size_t)i * 3 + 1] = ny; o_pose[(size_t)i * 3 + 2] = nw;
  o_motion[(size_t)i * 3] = nspd; o_motion[(size_t)i * 3 + 1] = nacc; o_motion[(size_t)i * 3 + 2] = nyr;
  o_action[(size_t)i * 2] = acc; o_action[(size_t)i * 2 + 1] = yr;
}

extern "C" int tb_dyn_update(const float* action_unbounded, const uint8_t* ag_type, const uint8_t* valid,
                             const uint8_t* player_valid, const float* player_action, const float* max_acc,
                             const float* max_yaw_rate, float dt, int n, const float* pose, const float* motion,
                             float* out_pose, float* out_motion, float* out_action, void* stream) {
  if (!action_unbounded || !ag_type || !valid || !max_acc || !max_yaw_rate || !pose || !motion || !out_pose || !out_motion ||
      !out_action || (player_valid && !player_action))
    return TB_ERR_NULL;
  if (n <= 0) return TB_ERR_BAD_SHAPE;
  dyn_update_kernel<<<(n + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      action_unbounded, ag_type, valid, player_valid, player_action, make_float3(max_acc[0], max_acc[1], max_acc[2]),
      make_float3(max_yaw_rate[0], max_yaw_rate[1], max_yaw_rate[2]), dt, n, pose, motion, out_pose, out_motion, out_action);
  TB_CHECK_LAUNCH();
  return TB_OK;
}

extern "C" int tb_step_advance(int* d_step, void* stream) {
  if (!d_step) return TB_ERR_NULL;
  step_advance_kernel<<<1, 1, 0, static_cast<cudaStream_t>(stream)>>>(d_step);
  TB_CHECK_LAUNCH();
  return TB_OK;
}

extern "C" int tb_action_mean(const float* act_branch, const uint8_t* ag_type, const uint8_t* valid, int M,
                              float* mean, void* stream) {
  if (!act_branch || !ag_type || !valid || !mean) return TB_ERR_NULL;
  if (M <= 0) return TB_ERR_BAD_SHAPE;
  action_mean_kernel<<<(M + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(act_branch, ag_type, valid, M, mean);
  TB_CHECK_LAUNCH();
  return TB_OK;
}
