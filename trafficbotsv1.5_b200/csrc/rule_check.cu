// Logging-only traffic-rule checks of one rollout step (tb_rule_check) — SURVEY.md 8(f) rank 1.
// Reference behaviour: TrafficRuleChecker.check (utils/traffic_rule_checker.py:343-451) with _check_collided (:119-149),
// check_collided_wosac (utils/wosac_collision.py:196-239), _check_run_road_edge (:152-173), _check_run_red_light
// (:176-218) and _check_passive (:221-274). The reference materialises [n_sc,n_ag,n_ag,4,4,3], [n_sc,n_ag,n_mp*20,4,2]
// ... tensors every step (3x the model's CPU time, BASELINE.md); here one CTA owns one rollout-scene, agents live in
// shared memory, agent pairs are pre-filtered by an exact conservative distance bound, and map segments / lane points
// are reached through per-polyline bounding circles (computed once per scene), so an agent only visits the nodes of
// the few polylines it can touch.
// Comparisons replicate the reference's fp32 operation order without FMA contraction (__fmul_rn / __fadd_rn), so flags
// can differ from the CPU reference only on knife-edge inputs (cos/sin of the heading may differ by 1 ulp).
#include "common.cuh"

namespace {

// tests/_rule_scenes.py mirrors MAX_A and QCAP: its crowd and dense-map scenes overflow both queues (more than QCAP
// agent pairs / (polyline, vehicle) pairs), so the inline fallbacks run under test.
constexpr int MAX_A = 256;
constexpr int QCAP = 4096;  // candidate queue per rollout-scene: agent pairs, then (polyline, vehicle) pairs
enum : unsigned { F_COL = 1, F_WOSAC = 2, F_EDGE = 4, F_RED = 8, F_LANE = 16, F_TLAHEAD = 32, F_AGAHEAD = 64 };

struct Args {
  const uint8_t* pred_valid; const float* pred_pose; const float* pred_motion;  // [B,A,T(,3)], step index s-1
  const uint8_t* ag_type;  // [B,A,3]
  const float* ag_size;    // [B/div,A,3]
  const uint8_t* hist_tl;  // [B/tl_div, n_tl, W, 5], slot s%W = state after override_tl
  const uint8_t* tl_invalid; const float* tl_pose;  // [B/div, n_tl(,3)]
  const float* seg;             // [B/div, n_mp, n_node, 4] (x0,y0,x1,y1) = (pos, pos + dir)
  const uint8_t* node_invalid;  // [B/div, n_mp, n_node]
  const float* poly_circle;     // [B/div, n_mp, 3] bounding circle (cx, cy, r) of each polyline
  const uint8_t* poly_kind;     // [B/div, n_mp]: bit0 road-edge types (4,5,7), bit1 lane-centre types (0..2)
  int n_mp, n_node;
  float* passive_counter;  // [B,A]
  uint8_t *o_col, *o_wosac, *o_edge, *o_red, *o_passive;  // [B,A,T]
  const int* d_step; int A, T, W, n_tl, div, tl_div; float size_scale;
};

__device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }

// get_ag_bbox (wosac_collision.py:22-48): corners [of-or, -of-or, -of+or, of+or] + position
__device__ __forceinline__ void make_box(float x, float y, float c, float s, float len, float wid, float* bx, float* by) {
  const float ofx = mul(mul(0.5f, len), c), ofy = mul(mul(0.5f, len), s);
  const float orx = mul(mul(0.5f, wid), s), ory = mul(mul(0.5f, wid), -c);
  bx[0] = add(x, sub(ofx, orx));        by[0] = add(y, sub(ofy, ory));
  bx[1] = add(x, sub(-ofx, orx));       by[1] = add(y, sub(-ofy, ory));
  bx[2] = add(x, add(-ofx, orx));       by[2] = add(y, add(-ofy, ory));
  bx[3] = add(x, add(ofx, orx));        by[3] = add(y, add(ofy, ory));
}

// all 4 corners of box q on the outer side of one edge line of box p (traffic_rule_checker.py:126-143)
__device__ __forceinline__ bool separated_by_edges(const float* px, const float* py, const float* qx, const float* qy) {
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const int n = (e + 1) & 3;
    const float a = sub(py[n], py[e]), b = sub(px[e], px[n]);
    const float c = sub(mul(px[n], py[e]), mul(py[n], px[e]));
    bool all_out = true;
#pragma unroll
    for (int k = 0; k < 4; ++k) all_out &= add(add(mul(a, qx[k]), mul(b, qy[k])), c) > 0.f;  // sum over (a,b,c)*(x,y,1)
    if (all_out) return true;
  }
  return false;
}

__device__ __forceinline__ bool ccw(float ax, float ay, float bx, float by, float cx, float cy) {
  return mul(sub(cy, ay), sub(bx, ax)) > mul(sub(by, ay), sub(cx, ax));
}

// signed distance from the origin to the Minkowski difference of two boxes (wosac_collision.py:51-192)
__device__ float wosac_signed_distance(const float* ax, const float* ay, const float* bx0, const float* by0) {
  float bx[4], by[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) { bx[k] = mul(-1.0f, bx0[k]); by[k] = mul(-1.0f, by0[k]); }
  int s1 = 0, s2 = 0;  // downmost vertex = first arg-min of y
#pragma unroll
  for (int k = 1; k < 4; ++k) { if (ay[k] < ay[s1]) s1 = k; if (by[k] < by[s2]) s2 = k; }
  auto edge_dir = [](const float* x, const float* y, int s, float* dx, float* dy) {
    const int n = (s + 1) & 3;
    const float ex = sub(x[n], x[s]), ey = sub(y[n], y[s]);
    const float l = sqrtf(add(mul(ex, ex), mul(ey, ey)));
    *dx = ex / l; *dy = ey / l;
  };
  float d1x, d1y, d2x, d2y;
  edge_dir(ax, ay, s1, &d1x, &d1y);
  edge_dir(bx, by, s2, &d2x, &d2y);
  const bool cond = sub(mul(d1x, d2y), mul(d1y, d2x)) >= 0.0f;
  float px[8], py[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int o1 = k >> 1, o2 = ((k + 1) >> 1) & 3;  // point_order_1 = 0,0,1,1,.. ; point_order_2 = 0,1,1,2,2,3,3,0
    const int i1 = ((cond ? o2 : o1) + s1) & 3, i2 = ((cond ? o1 : o2) + s2) & 3;
    px[k] = add(ax[i1], bx[i2]);
    py[k] = add(ay[i1], by[i2]);
  }
  bool inside = true;
  float md = 1e10f;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int n = (k + 1) & 7;
    const float ex = sub(px[n], px[k]), ey = sub(py[n], py[k]);
    const float el = sqrtf(add(mul(ex, ex), mul(ey, ey)));
    const float tx = ex / el, ty = ey / el;
    const float vx = -px[k], vy = -py[k];                 // vertex -> query (origin)
    const float vd = sqrtf(add(mul(vx, vx), mul(vy, vy)));
    const float sperp = add(mul(ty, vx), mul(-tx, vy));   // sum(-normal * v), normal = (-ty, tx)
    inside &= sperp <= 0.f;
    const float prop = add(mul(tx, vx), mul(ty, vy)) / el;
    const float ed = (prop >= 0.0f && prop <= 1.0f) ? fabsf(sperp) : 1e10f;
    md = fminf(md, fminf(ed, vd));
  }
  return inside ? -md : md;
}

__global__ void __launch_bounds__(256) rule_check_kernel(Args p) {
  __shared__ float s_x[MAX_A], s_y[MAX_A], s_c[MAX_A], s_s[MAX_A], s_spd[MAX_A], s_rad[MAX_A], s_shrink[MAX_A];
  __shared__ float s_len[MAX_A], s_wid[MAX_A];
  __shared__ float s_bx[MAX_A][4], s_by[MAX_A][4], s_wx[MAX_A][4], s_wy[MAX_A][4];
  __shared__ uint8_t s_valid[MAX_A], s_veh[MAX_A], s_ped[MAX_A];
  __shared__ unsigned s_flag[MAX_A];
  __shared__ unsigned s_q[QCAP];
  __shared__ int s_qn;
  __shared__ float4 s_veh4[MAX_A];  // valid vehicles, compacted: (x, y, map reach, agent id bits)
  __shared__ int s_nveh;
  __shared__ float s_bb[4];         // their bounding box grown by the reach: x0, y0, x1, y1

  const int b = blockIdx.x, sc = b / p.div, A = p.A;
  const int s = *p.d_step;
  if (s < 1 || s > p.T) return;  // block-uniform: the flags of step s live at [.., s - 1] < T
  for (int a = threadIdx.x; a < A; a += blockDim.x) {
    const size_t i = (size_t)b * A + a, o = i * p.T + (s - 1);
    const float x = p.pred_pose[o * 3], y = p.pred_pose[o * 3 + 1], w = p.pred_pose[o * 3 + 2];
    const float c = cosf(w), sn = sinf(w);
    const float* sz = p.ag_size + ((size_t)sc * A + a) * 3;
    const float len = mul(sz[0], p.size_scale), wid = mul(sz[1], p.size_scale);  // self.ag_size (:27)
    s_x[a] = x; s_y[a] = y; s_c[a] = c; s_s[a] = sn; s_spd[a] = p.pred_motion[o * 3];
    s_len[a] = sz[0]; s_wid[a] = sz[1];
    s_valid[a] = p.pred_valid[o]; s_veh[a] = p.ag_type[i * 3]; s_ped[a] = p.ag_type[i * 3 + 1];
    make_box(x, y, c, sn, len, wid, s_bx[a], s_by[a]);
    const float shrink = mul(fminf(len, wid), 0.7f) / 2.0f;                       // wosac_collision.py:216
    s_shrink[a] = shrink;
    make_box(x, y, c, sn, sub(len, mul(2.0f, shrink)), sub(wid, mul(2.0f, shrink)), s_wx[a], s_wy[a]);
    s_rad[a] = 0.5f * sqrtf(len * len + wid * wid) + 1e-3f;                       // conservative circumradius
    s_flag[a] = 0u;
  }
  if (threadIdx.x == 0) { s_qn = 0; s_nveh = 0; }
  __syncthreads();
  // valid vehicles for the map phase (ncu: 60 % of the kernel's instructions were the polyline x agent circle tests
  // re-reading validity / type bytes and three floats per pair)
  for (int a = threadIdx.x; a < A; a += blockDim.x)
    if (s_valid[a] && s_veh[a])
      s_veh4[atomicAdd(&s_nveh, 1)] = make_float4(s_x[a], s_y[a], fmaxf(s_rad[a], 2.001f), __int_as_float(a));
  __syncthreads();
  if (threadIdx.x < 32) {
    float x0 = 3.0e38f, y0 = 3.0e38f, x1 = -3.0e38f, y1 = -3.0e38f;
    for (int i = threadIdx.x; i < s_nveh; i += 32) {
      const float4 g = s_veh4[i];
      x0 = fminf(x0, g.x - g.z); y0 = fminf(y0, g.y - g.z); x1 = fmaxf(x1, g.x + g.z); y1 = fmaxf(y1, g.y + g.z);
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      x0 = fminf(x0, __shfl_xor_sync(TB_FULL_MASK, x0, o)); y0 = fminf(y0, __shfl_xor_sync(TB_FULL_MASK, y0, o));
      x1 = fmaxf(x1, __shfl_xor_sync(TB_FULL_MASK, x1, o)); y1 = fmaxf(y1, __shfl_xor_sync(TB_FULL_MASK, y1, o));
    }
    if (threadIdx.x == 0) { s_bb[0] = x0; s_bb[1] = y0; s_bb[2] = x1; s_bb[3] = y1; }
  }
  // (s_bb is first read after the __syncthreads() calls of the agent x agent phase)

  // ---- agent x agent: collision (SAT), WOSAC collision, "agent ahead" of the passive check.
  // Pass 1 runs the cheap distance tests over all A^2 ordered pairs and queues the few whose circumcircles touch;
  // pass 2 runs SAT + the Minkowski signed distance densely over the queue (inline in pass 1 the ~550-instruction
  // branch was taken by one or two lanes of half the warps' iterations).
  auto near_pair = [&](int a, int j) {
    unsigned f = 0u;
    if (!(s_ped[a] && s_ped[j])) {  // collision_invalid_mask (:48-51)
      const bool no_col = separated_by_edges(s_bx[a], s_by[a], s_bx[j], s_by[j]) ||
                          separated_by_edges(s_bx[j], s_by[j], s_bx[a], s_by[a]);
      if (!no_col) f |= F_COL;
    }
    float sd = wosac_signed_distance(s_wx[a], s_wy[a], s_wx[j], s_wy[j]);
    sd = sub(sub(sd, s_shrink[j]), s_shrink[a]);                                 // :231-232
    if (sd < 0.0f) f |= F_WOSAC;
    if (f) atomicOr(&s_flag[a], f);
  };
  for (int q = threadIdx.x; q < A * A; q += blockDim.x) {
    const int a = q / A, j = q - a * A;
    if (a == j || !s_valid[a] || !s_valid[j]) continue;
    const float dx = sub(s_x[j], s_x[a]), dy = sub(s_y[j], s_y[a]);
    const float d2 = dx * dx + dy * dy;
    const float reach = s_rad[a] + s_rad[j];
    if (d2 <= reach * reach) {
      const int k = atomicAdd(&s_qn, 1);
      if (k < QCAP) s_q[k] = ((unsigned)a << 8) | (unsigned)j;
      else near_pair(a, j);  // queue full (a crowd): inline
    }
    if (d2 < 101.f) {  // _check_passive (:262-268): norm < 10 m and cos(angle to heading) > 0.95
      const float n = sqrtf(add(mul(dx, dx), mul(dy, dy)));
      if (n < 10.f && (add(mul(s_c[a], dx), mul(s_s[a], dy)) / n) > 0.95f) atomicOr(&s_flag[a], F_AGAHEAD);
    }
  }
  __syncthreads();
  {
    const int npair = min(s_qn, QCAP);
    for (int it = threadIdx.x; it < npair; it += blockDim.x) near_pair((int)(s_q[it] >> 8), (int)(s_q[it] & 255u));
  }
  __syncthreads();
  if (threadIdx.x == 0) s_qn = 0;  // the queue is reused by the map phase
  __syncthreads();

  // ---- agent x traffic light: red-light running (:176-218) and "red light ahead" of the passive check (:250-256)
  const int slot = s % p.W;
  for (int q = threadIdx.x; q < A * p.n_tl; q += blockDim.x) {
    const int a = q / p.n_tl, t = q - a * p.n_tl;
    if (!s_valid[a] || !s_veh[a]) continue;
    const size_t ti = (size_t)sc * p.n_tl + t;
    if (p.tl_invalid[ti]) continue;
    const uint8_t* st = p.hist_tl + (((size_t)(b / p.tl_div) * p.n_tl + t) * p.W + slot) * 5;
    const float tx = p.tl_pose[ti * 3], ty = p.tl_pose[ti * 3 + 1];
    unsigned f = 0u;
    if (st[1]) {
      const float c = s_c[a], sn = s_s[a];
      const float ln = mul(mul(s_len[a], 0.5f), 0.6f), wd = mul(mul(s_wid[a], 0.5f), 1.8f);  // :61-62 (unscaled size)
      const float x0 = s_x[a], y0 = s_y[a];
      const float step = mul(0.1f, s_spd[a]);
      const float x1 = add(x0, mul(step, c)), y1 = add(y0, mul(step, sn));
      auto inside = [&](float px, float py) {
        const float ex = sub(tx, px), ey = sub(ty, py);
        return fabsf(add(mul(ex, c), mul(ey, sn))) < ln && fabsf(add(mul(ex, sn), mul(ey, -c))) < wd;
      };
      if (inside(x0, y0) && !inside(x1, y1)) f |= F_RED;
    }
    if (st[0] || st[1] || st[2] || st[4]) {
      const float vx = sub(tx, s_x[a]), vy = sub(ty, s_y[a]);
      const float n = sqrtf(add(mul(vx, vx), mul(vy, vy)));
      if (n < 10.f && (add(mul(s_c[a], vx), mul(s_s[a], vy)) / n) > 0.95f) f |= F_TLAHEAD;
    }
    if (f) atomicOr(&s_flag[a], f);
  }

  // ---- agent x map: road-edge crossing (:152-173) and "close to lane" of the passive check (:243-247).
  // Phase 1: polylines strided over threads, every (polyline, agent) whose bounding circles touch is queued.
  // Phase 2: the queue is expanded to (pair, node) items over all threads — no divergent per-lane node loops.
  auto test_node = [&](int a, size_t ni, unsigned kind) {
    if (p.node_invalid[ni]) return;
    const float cx = p.seg[ni * 4], cy = p.seg[ni * 4 + 1];
    if ((kind & 1u) && !(s_flag[a] & F_EDGE)) {
      const float dx = p.seg[ni * 4 + 2], dy = p.seg[ni * 4 + 3];
      bool hit = false;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int m = (k + 1) & 3;
        const float ax = s_bx[a][k], ay = s_by[a][k], bx = s_bx[a][m], by = s_by[a][m];
        hit |= (ccw(ax, ay, cx, cy, dx, dy) != ccw(bx, by, cx, cy, dx, dy)) &&
               (ccw(ax, ay, bx, by, cx, cy) != ccw(ax, ay, bx, by, dx, dy));
      }
      if (hit) atomicOr(&s_flag[a], F_EDGE);
    }
    if ((kind & 2u) && !(s_flag[a] & F_LANE)) {
      const float ex = sub(s_x[a], cx), ey = sub(s_y[a], cy);
      if (sqrtf(add(mul(ex, ex), mul(ey, ey))) < 2.f) atomicOr(&s_flag[a], F_LANE);
    }
  };
  for (int pl = threadIdx.x; pl < p.n_mp; pl += blockDim.x) {
    const size_t pi = (size_t)sc * p.n_mp + pl;
    const unsigned kind = p.poly_kind[pi];
    if (!kind) continue;
    const float pcx = p.poly_circle[pi * 3], pcy = p.poly_circle[pi * 3 + 1], pr = p.poly_circle[pi * 3 + 2];
    if (pcx + pr < s_bb[0] || pcy + pr < s_bb[1] || pcx - pr > s_bb[2] || pcy - pr > s_bb[3]) continue;
    const int n_veh = s_nveh;
    for (int i = 0; i < n_veh; ++i) {
      const float4 g = s_veh4[i];
      const float rx = pcx - g.x, ry = pcy - g.y, reach = pr + g.z;
      if (rx * rx + ry * ry > reach * reach) continue;
      const int a = __float_as_int(g.w);
      const int k = atomicAdd(&s_qn, 1);
      if (k < QCAP) s_q[k] = ((unsigned)pl << 8) | (unsigned)a;
      else for (int n = 0; n < p.n_node; ++n) test_node(a, pi * p.n_node + n, kind);  // queue full: inline (rare)
    }
  }
  __syncthreads();
  const int nq = min(s_qn, QCAP);
  for (int it = threadIdx.x; it < nq * p.n_node; it += blockDim.x) {
    const int h = it / p.n_node, n = it - h * p.n_node;
    const unsigned e = s_q[h];
    const int pl = (int)(e >> 8), a = (int)(e & 255u);
    const size_t pi = (size_t)sc * p.n_mp + pl;
    test_node(a, pi * p.n_node + n, p.poly_kind[pi]);
  }
  __syncthreads();

  for (int a = threadIdx.x; a < A; a += blockDim.x) {
    const size_t i = (size_t)b * A + a, o = i * p.T + (s - 1);
    const unsigned f = s_flag[a];
    const bool valid = s_valid[a] != 0, veh = s_veh[a] != 0;
    p.o_col[o] = (f & F_COL) != 0;
    p.o_wosac[o] = (f & F_WOSAC) != 0;
    p.o_edge[o] = (f & F_EDGE) != 0;
    p.o_red[o] = (f & F_RED) != 0;
    const bool passive = valid && veh && (f & F_LANE) && (s_spd[a] < 5.f) && !(f & F_TLAHEAD) && !(f & F_AGAHEAD);
    const float cnt = passive ? p.passive_counter[i] + 1.f : 0.f;  // (counter + p) * p   (:271)
    p.passive_counter[i] = cnt;
    p.o_passive[o] = cnt > 20.f;
  }
}

}  // namespace

extern "C" int tb_rule_check(const uint8_t* pred_valid, const float* pred_pose, const float* pred_motion,
                             const uint8_t* ag_type, const float* ag_size, const uint8_t* hist_tl,
                             const uint8_t* tl_invalid, const float* tl_pose, const float* seg,
                             const uint8_t* node_invalid, const float* poly_circle, const uint8_t* poly_kind, int n_mp,
                             int n_node, float* passive_counter,
                             uint8_t* o_collided, uint8_t* o_collided_wosac, uint8_t* o_run_road_edge,
                             uint8_t* o_run_red_light, uint8_t* o_passive, const int* d_step, int B, int A, int T, int W,
                             int n_tl, int sc_div, int tl_div, float size_scale, void* stream) {
  if (!pred_valid || !pred_pose || !pred_motion || !ag_type || !ag_size || !hist_tl || !tl_invalid || !tl_pose ||
      !seg || !node_invalid || !poly_circle || !poly_kind || !passive_counter || !o_collided || !o_collided_wosac ||
      !o_run_road_edge || !o_run_red_light || !o_passive || !d_step)
    return TB_ERR_NULL;
  if (B <= 0 || A <= 0 || T <= 0 || W <= 0 || n_tl <= 0 || sc_div <= 0 || tl_div <= 0 || n_mp <= 0 || n_node <= 0)
    return TB_ERR_BAD_SHAPE;
  if (A > MAX_A) return TB_ERR_UNSUPPORTED;
  Args p{pred_valid, pred_pose, pred_motion, ag_type, ag_size, hist_tl, tl_invalid, tl_pose, seg, node_invalid, poly_circle,
         poly_kind, n_mp, n_node, passive_counter, o_collided, o_collided_wosac, o_run_road_edge, o_run_red_light,
         o_passive, d_step, A, T, W, n_tl, sc_div, tl_div, size_scale};
  rule_check_kernel<<<B, 256, 0, static_cast<cudaStream_t>(stream)>>>(p);
  TB_CHECK_LAUNCH();
  return TB_OK;
}
