// Fused pairwise relative pose + top-K nearest-target selection (tb_knn_select).
// Reference behaviour: utils/rpe.py:9-37 (get_rel_pose) + :62-90 (get_tgt_knn_idx).
//
// One warp per source token. The scene's targets (x, y, yaw, invalid) are staged once per CTA in shared
// memory and shared by all of the CTA's source rows; each lane keeps T/32 candidate keys (squared distances) in
// registers (never materialising the [S,T,3] rel-pose / [S,T] distance tensors of the reference).
// Selection: (1) prune — the per-lane two smallest keys give 64 candidates whose maximum U bounds the K-th smallest
// from above, so only keys <= U (typically ~15 % of T) survive and are ballot-compacted into a per-warp list;
// (2) the K-th smallest of the survivors is found by bisection on the fp32 bit pattern (non-negative floats order
// like unsigned ints) with one REDUX per probe; (3) winners are compacted in ascending target-index order (ties: lower
// index) and their rotated relative pose / exact distance are evaluated from shared memory. Rows whose survivor list
// would overflow (many invalid targets, K > 64, T <= 128) take the general path: bisection over all T keys.
// Repeated selections against static x-sorted targets with a row state (agent -> map, every rollout step) run in
// knn_slab_kernel instead: it scans only an x-slab around the source and holds no per-lane key array, so it keeps
// 4 CTAs per SM where knn_select_kernel<32> keeps 2.
#include "common.cuh"

namespace {

constexpr int kWarps = 8;
constexpr int kRowsPerWarp = 8;  // source rows per warp => 64 rows per CTA amortise the target staging
constexpr int kCap = 12;         // pruned candidate list: up to kCap*32 survivors per row

// K-th smallest of the warp's keys (N per lane) by bisection on the bit pattern; returns tau and #keys < tau.
// Returns the smallest v in [lo, hi] with #keys <= v >= K (hi if none). kFast stops early with that same value: when
// fewer than K keys lie below hi (e.g. a K-th key of +inf), and at the first probe with exactly K keys <= mid (the
// largest of them is the K-th smallest) - usually a handful of probes instead of ~log2(hi - lo). Exact ties at the
// K-th key never give a count of exactly K and take the full bisection.
template <int N, bool kFast>
__device__ __forceinline__ uint32_t kth_smallest(const uint32_t (&key)[N], int K, uint32_t hi, int* c_lt_out,
                                                 uint32_t lo = 0u) {
  if (kFast && lo < hi) {
    int c = 0;
#pragma unroll
    for (int i = 0; i < N; ++i) c += (key[i] < hi);
    if (__reduce_add_sync(TB_FULL_MASK, c) < K) lo = hi;
  }
  while (lo < hi) {
    const uint32_t mid = lo + ((hi - lo) >> 1);
    int c = 0;
#pragma unroll
    for (int i = 0; i < N; ++i) c += (key[i] <= mid);
    c = __reduce_add_sync(TB_FULL_MASK, c);
    if (kFast && c == K) {
      uint32_t m = 0u;
#pragma unroll
      for (int i = 0; i < N; ++i) m = key[i] <= mid ? max(m, key[i]) : m;
      lo = max(lo, __reduce_max_sync(TB_FULL_MASK, m));  // lo > lo_in only after a probe below the K-th key
      break;
    }
    if (c >= K) hi = mid; else lo = mid + 1u;
  }
  int c_lt = 0;
#pragma unroll
  for (int i = 0; i < N; ++i) c_lt += (key[i] < lo);
  *c_lt_out = __reduce_add_sync(TB_FULL_MASK, c_lt);
  return lo;
}

struct RowCtx {
  float sx, sy, syaw, sn, cs, dist_limit;
  const float *tx, *ty, *tyaw;
  const uint8_t* tinv;
  bool sinv;
  const int32_t* tmap;  // staged target position -> caller's target index (NULL: identity)
  int32_t* out_idx; uint8_t* out_invalid; float* out_rel;
  size_t obase;
};

// winner t -> outputs (relative pose in the source frame, utils/rpe.py:26-36; invalid flag :85-86)
__device__ __forceinline__ void emit(const RowCtx& c, int pos, int t) {
  const float dx = c.tx[t] - c.sx, dy = c.ty[t] - c.sy;
  const float lx = fmaf(dx, c.cs, dy * c.sn), ly = fmaf(dy, c.cs, -dx * c.sn);
  const bool dead = c.sinv || c.tinv[t];
  const float d = dead ? __int_as_float(0x7f800000) : sqrtf(fmaf(lx, lx, ly * ly));
  c.out_idx[c.obase + pos] = c.tmap ? c.tmap[t] : t;
  c.out_invalid[c.obase + pos] = (uint8_t)((c.tinv[t] != 0) | (d > c.dist_limit));
  float* r = c.out_rel + (c.obase + pos) * 3;
  r[0] = lx; r[1] = ly; r[2] = c.tyaw[t] - c.syaw;
}

// selection key of staged target t: squared distance (the rotation into the source frame preserves it; the winners'
// rotated pose and exact distance are evaluated in emit()), +inf if either end is invalid, beyond T never selected
__device__ __forceinline__ uint32_t target_key(const RowCtx& c, int t, int T) {
  if (t >= T) return 0xffffffffu;
  const float dx = c.tx[t] - c.sx, dy = c.ty[t] - c.sy;
  return (c.sinv || c.tinv[t]) ? 0x7f800000u : __float_as_uint(fmaf(dx, dx, dy * dy));
}

// K smallest of a compacted candidate list (keys + staged target positions, ascending position order): bisection on
// [lo, hi], winners emitted in list order (ties: earlier entries). Returns the K-th smallest key.
template <int NC, bool kFast>
__device__ __forceinline__ uint32_t select_from_list(const RowCtx& c, const uint32_t* ckey, const uint16_t* cidx, int cnt,
                                                     int K, uint32_t lo, uint32_t hi, int lane, unsigned lt_mask) {
  uint32_t ck[NC];
#pragma unroll
  for (int j = 0; j < NC; ++j) ck[j] = (j * 32 + lane < cnt) ? ckey[j * 32 + lane] : 0xffffffffu;
  int c_lt;
  const uint32_t tau = kth_smallest<NC, kFast>(ck, K, hi, &c_lt, lo);
  const int need_ties = K - c_lt;
  int n_out = 0, n_tie = 0;
#pragma unroll
  for (int j = 0; j < NC; ++j) {
    if (j * 32 >= cnt) break;  // warp-uniform
    const bool is_tie = ck[j] == tau;
    const unsigned tie_b = __ballot_sync(TB_FULL_MASK, is_tie);
    const bool sel = (ck[j] < tau) || (is_tie && n_tie + __popc(tie_b & lt_mask) < need_ties);
    const unsigned sel_b = __ballot_sync(TB_FULL_MASK, sel);
    if (sel) emit(c, n_out + __popc(sel_b & lt_mask), cidx[j * 32 + lane]);
    n_out += __popc(sel_b);
    n_tie += __popc(tie_b);
  }
  return tau;
}

// The scene's targets -> shared memory (x, y, yaw planes, then the invalid bytes); returns the staged planes and the
// per-warp candidate lists behind them.
struct Staged {
  float *tx, *ty, *tyaw;
  uint8_t* tinv;
  uint32_t* ckey;
  uint16_t* cidx;
  const int32_t* tmap;
};

__device__ __forceinline__ Staged stage_targets(float* smem, const float* tgt_pose, const uint8_t* tgt_invalid,
                                                const int32_t* tgt_index_map, int T, int bt) {
  Staged g;
  g.tx = smem;
  g.ty = g.tx + T;
  g.tyaw = g.ty + T;
  g.tinv = reinterpret_cast<uint8_t*>(g.tyaw + T);
  uint32_t* ckey_all = reinterpret_cast<uint32_t*>(smem + 3 * T + ((T + 15) / 16) * 4);
  uint16_t* cidx_all = reinterpret_cast<uint16_t*>(ckey_all + kWarps * kCap * 32);
  const int warp = threadIdx.x >> 5;
  g.ckey = ckey_all + warp * kCap * 32;
  g.cidx = cidx_all + warp * kCap * 32;
  g.tmap = tgt_index_map ? tgt_index_map + (size_t)bt * T : nullptr;
  const float* tp = tgt_pose + (size_t)bt * T * 3;
  const uint8_t* ti = tgt_invalid + (size_t)bt * T;
  for (int i = threadIdx.x; i < T; i += blockDim.x) {
    g.tx[i] = tp[i * 3 + 0];
    g.ty[i] = tp[i * 3 + 1];
    g.tyaw[i] = tp[i * 3 + 2];
    g.tinv[i] = ti[i];
  }
  __syncthreads();
  return g;
}

__device__ __forceinline__ RowCtx row_ctx(const Staged& g, const float* src_pose, const uint8_t* src_invalid,
                                          size_t row, float dist_limit, int32_t* out_idx, uint8_t* out_invalid,
                                          float* out_rel, int ldk, int koff) {
  RowCtx c;
  c.sx = src_pose[row * 3 + 0]; c.sy = src_pose[row * 3 + 1]; c.syaw = src_pose[row * 3 + 2];
  c.sinv = src_invalid[row] != 0;
  sincosf(c.syaw, &c.sn, &c.cs);
  c.dist_limit = dist_limit; c.tx = g.tx; c.ty = g.ty; c.tyaw = g.tyaw; c.tinv = g.tinv;
  c.out_idx = out_idx; c.out_invalid = out_invalid; c.out_rel = out_rel; c.tmap = g.tmap;
  c.obase = row * (size_t)ldk + koff;
  return c;
}

// invalid source: every distance is +inf, the (always masked) fillers are targets 0..K-1
__device__ __forceinline__ void emit_invalid_row(const RowCtx& c, float* rs, int K, int lane) {
  for (int pos = lane; pos < K; pos += 32) emit(c, pos, pos);
  if (rs && lane == 0) rs[2] = __int_as_float(0x7f800000);
}

// ---- temporal-coherence fast path (static targets sorted by x, e.g. agent -> map): at least K valid targets lay
// within sqrt(kth_prev) of the previous source position, so they lie within r = sqrt(kth_prev) + |displacement|
// of the current one (triangle inequality): the K nearest are among the targets with |x - sx| <= r and d <= r.
// Only that x-slab is scanned (binary search in the staged, x-sorted coordinates); everything else is unchanged.
// Returns false (nothing written) for a first call (state +inf), a survivor list overflow or fewer than K survivors.
template <bool kFast>
__device__ __forceinline__ bool slab_select(const RowCtx& c, float* rs, uint32_t* ckey, uint16_t* cidx, int T, int K,
                                            int lane, unsigned lt_mask) {
  const float kprev = rs[2];
  if (!(kprev < 3.0e38f)) return false;
  const float ddx = c.sx - rs[0], ddy = c.sy - rs[1];
  const float r = (sqrtf(kprev) + sqrtf(fmaf(ddx, ddx, ddy * ddy))) * 1.00001f + 1e-3f;
  const float r2 = r * r;
  int lo = 0, hi = T;  // lo = first t with tx[t] >= sx - r, hi = first t with tx[t] > sx + r
  {
    int a = 0, b2 = T;
    const float xl = c.sx - r, xh = c.sx + r;
    while (a < b2) { const int m = (a + b2) >> 1; if (c.tx[m] < xl) a = m + 1; else b2 = m; }
    lo = a;
    b2 = T;
    while (a < b2) { const int m = (a + b2) >> 1; if (c.tx[m] <= xh) a = m + 1; else b2 = m; }
    hi = a;
  }
  __syncwarp();
  int cnt = 0;
  bool overflow = false;
  for (int base = lo; base < hi; base += 32) {  // warp-uniform bounds
    const int t = base + lane;
    uint32_t k = 0xffffffffu;
    if (t < hi) {
      const float dx = c.tx[t] - c.sx, dy = c.ty[t] - c.sy;
      k = c.tinv[t] ? 0x7f800000u : __float_as_uint(fmaf(dx, dx, dy * dy));
    }
    const bool sel = k <= __float_as_uint(r2);
    const unsigned sb = __ballot_sync(TB_FULL_MASK, sel);
    if (cnt + __popc(sb) > kCap * 32) { overflow = true; break; }
    if (sel) {
      const int p = cnt + __popc(sb & lt_mask);
      ckey[p] = k;
      cidx[p] = (uint16_t)t;
    }
    cnt += __popc(sb);
  }
  __syncwarp();
  if (overflow || cnt < K) return false;
  // the K-th distance cannot have shrunk by more than the displacement either: bracket for the bisection
  const float dl = (sqrtf(kprev) - sqrtf(fmaf(ddx, ddx, ddy * ddy))) * 0.9999f - 1e-3f;
  const uint32_t lo_bits = dl > 0.f ? __float_as_uint(dl * dl) : 0u;
  uint32_t tau;
  if (cnt <= 4 * 32) {  // the usual case: K + a few survivors
    tau = select_from_list<4, kFast>(c, ckey, cidx, cnt, K, lo_bits, __float_as_uint(r2), lane, lt_mask);
  } else {
    tau = select_from_list<kCap, kFast>(c, ckey, cidx, cnt, K, lo_bits, __float_as_uint(r2), lane, lt_mask);
  }
  if (lane == 0) { rs[0] = c.sx; rs[1] = c.sy; rs[2] = __uint_as_float(tau); }
  return true;
}

// Bisection bracket of the general path: with a row state (static targets) |sqrt(kth) - sqrt(kth_prev)| <=
// |displacement|.
__device__ __forceinline__ void state_bracket(const RowCtx& c, const float* rs, uint32_t* b_lo, uint32_t* b_hi) {
  *b_lo = 0u;
  *b_hi = 0x7f800000u;
  if (rs && rs[2] < 3.0e38f) {
    const float ddx = c.sx - rs[0], ddy = c.sy - rs[1];
    const float disp = sqrtf(fmaf(ddx, ddx, ddy * ddy)), dk = sqrtf(rs[2]);
    const float dh = (dk + disp) * 1.00001f + 1e-3f, dl = (dk - disp) * 0.9999f - 1e-3f;
    *b_hi = __float_as_uint(dh * dh);
    *b_lo = dl > 0.f ? __float_as_uint(dl * dl) : 0u;
  }
}

// General kernel: every path, keys in registers. kFast = false is the previous selection (full-length bisections, the
// slab path in this kernel), kept as the reference of the fast one; both give the same lists bit for bit.
template <int TPL, bool kFast>
__global__ void __launch_bounds__(kWarps * 32)
knn_select_kernel(const float* __restrict__ src_pose, const uint8_t* __restrict__ src_invalid,
                  const float* __restrict__ tgt_pose, const uint8_t* __restrict__ tgt_invalid, int S, int T, int div,
                  int K, float dist_limit, int32_t* __restrict__ out_idx, uint8_t* __restrict__ out_invalid,
                  float* __restrict__ out_rel, int ldk, int koff, const int32_t* __restrict__ tgt_index_map,
                  float* __restrict__ row_state, int sorted_by_x) {
  extern __shared__ float smem[];
  const int b = blockIdx.y;
  const Staged g = stage_targets(smem, tgt_pose, tgt_invalid, tgt_index_map, T, b / div);
  uint32_t* ckey = g.ckey;
  uint16_t* cidx = g.cidx;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const unsigned lt_mask = (1u << lane) - 1u;
  const int row0 = (blockIdx.x * kWarps + warp) * kRowsPerWarp;

  for (int rr = 0; rr < kRowsPerWarp; ++rr) {
    const int s = row0 + rr;
    if (s >= S) break;  // warp-uniform
    const size_t row = (size_t)b * S + s;
    const RowCtx c = row_ctx(g, src_pose, src_invalid, row, dist_limit, out_idx, out_invalid, out_rel, ldk, koff);
    float* rs = row_state ? row_state + row * 3 : nullptr;  // (x, y, K-th smallest squared distance) of the last call

    if (c.sinv) {
      emit_invalid_row(c, rs, K, lane);
      continue;
    }
    if (!kFast && rs && sorted_by_x && TPL >= 8 && slab_select<false>(c, rs, ckey, cidx, T, K, lane, lt_mask)) continue;

    uint32_t key[TPL];  // this lane's candidates t = i*32 + lane
#pragma unroll
    for (int i = 0; i < TPL; ++i) key[i] = target_key(c, i * 32 + lane, T);

    bool done = false;
    if (TPL >= 8 && K <= 64) {
      // ---- prune: the 64 (32) per-lane two-smallest (smallest) keys bound the K-th smallest from above
      uint32_t m1 = 0xffffffffu, m2 = 0xffffffffu;
#pragma unroll
      for (int i = 0; i < TPL; ++i) {
        m2 = min(m2, max(m1, key[i]));
        m1 = min(m1, key[i]);
      }
      const uint32_t U = __reduce_max_sync(TB_FULL_MASK, K <= 32 ? m1 : m2);
      int cnt = 0;
#pragma unroll
      for (int i = 0; i < TPL; ++i) cnt += (key[i] <= U);
      cnt = __reduce_add_sync(TB_FULL_MASK, cnt);
      if (cnt <= kCap * 32) {  // warp-uniform
        __syncwarp();
        int base = 0;
#pragma unroll
        for (int i = 0; i < TPL; ++i) {  // compaction keeps ascending target-index order
          const bool sel = key[i] <= U;
          const unsigned sb = __ballot_sync(TB_FULL_MASK, sel);
          if (sel) {
            const int p = base + __popc(sb & lt_mask);
            ckey[p] = key[i];
            cidx[p] = (uint16_t)(i * 32 + lane);
          }
          base += __popc(sb);
        }
        __syncwarp();
        const uint32_t tau = select_from_list<kCap, kFast>(c, ckey, cidx, cnt, K, 0u, U, lane, lt_mask);
        if (rs && lane == 0) { rs[0] = c.sx; rs[1] = c.sy; rs[2] = __uint_as_float(tau); }
        done = true;
      }
    }
    if (done) continue;

    // ---- general path: bisection over all T keys
    uint32_t b_lo, b_hi;
    state_bracket(c, rs, &b_lo, &b_hi);
    int c_lt;
    const uint32_t tau = kth_smallest<TPL, kFast>(key, K, b_hi, &c_lt, b_lo);
    const int need_ties = K - c_lt;  // >= 1
    int n_out = 0, n_tie = 0;
#pragma unroll
    for (int i = 0; i < TPL; ++i) {  // compaction in ascending target index (i-major, then lane)
      const bool is_tie = key[i] == tau;
      const unsigned tie_b = __ballot_sync(TB_FULL_MASK, is_tie);
      const bool sel = (key[i] < tau) || (is_tie && n_tie + __popc(tie_b & lt_mask) < need_ties);
      const unsigned sel_b = __ballot_sync(TB_FULL_MASK, sel);
      if (sel) emit(c, n_out + __popc(sel_b & lt_mask), i * 32 + lane);
      n_out += __popc(sel_b);
      n_tie += __popc(tie_b);
    }
    if (rs && lane == 0) { rs[0] = c.sx; rs[1] = c.sy; rs[2] = __uint_as_float(tau); }
  }
}

// Static x-sorted targets with a row state, T > 128 (agent -> map, every rollout step). Nearly every row takes the slab
// path; the others (first call, slab overflow, fewer than K survivors) take the same decisions as
// knn_select_kernel<TPL> - prune when K <= 64 and the survivors fit the list, else bisection over all keys - with the
// keys recomputed from shared memory at each pass instead of held in a TPL-key register array.
__global__ void __launch_bounds__(kWarps * 32, 4)
knn_slab_kernel(const float* __restrict__ src_pose, const uint8_t* __restrict__ src_invalid,
                const float* __restrict__ tgt_pose, const uint8_t* __restrict__ tgt_invalid, int S, int T, int div,
                int K, float dist_limit, int32_t* __restrict__ out_idx, uint8_t* __restrict__ out_invalid,
                float* __restrict__ out_rel, int ldk, int koff, const int32_t* __restrict__ tgt_index_map,
                float* __restrict__ row_state) {
  extern __shared__ float smem[];
  const int b = blockIdx.y;
  const Staged g = stage_targets(smem, tgt_pose, tgt_invalid, tgt_index_map, T, b / div);
  uint32_t* ckey = g.ckey;
  uint16_t* cidx = g.cidx;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const unsigned lt_mask = (1u << lane) - 1u;
  const int row0 = (blockIdx.x * kWarps + warp) * kRowsPerWarp;
  const int n_i = (T + 31) >> 5;  // lane rows of keys; beyond n_i every key is padding (never selected, never <= U)

  for (int rr = 0; rr < kRowsPerWarp; ++rr) {
    const int s = row0 + rr;
    if (s >= S) break;  // warp-uniform
    const size_t row = (size_t)b * S + s;
    const RowCtx c = row_ctx(g, src_pose, src_invalid, row, dist_limit, out_idx, out_invalid, out_rel, ldk, koff);
    float* rs = row_state + row * 3;

    if (c.sinv) {
      emit_invalid_row(c, rs, K, lane);
      continue;
    }
    if (slab_select<true>(c, rs, ckey, cidx, T, K, lane, lt_mask)) continue;

    if (K <= 64) {  // prune
      uint32_t m1 = 0xffffffffu, m2 = 0xffffffffu;
      for (int i = 0; i < n_i; ++i) {
        const uint32_t k = target_key(c, i * 32 + lane, T);
        m2 = min(m2, max(m1, k));
        m1 = min(m1, k);
      }
      const uint32_t U = __reduce_max_sync(TB_FULL_MASK, K <= 32 ? m1 : m2);
      int cnt = 0;
      for (int i = 0; i < n_i; ++i) cnt += (target_key(c, i * 32 + lane, T) <= U);
      cnt = __reduce_add_sync(TB_FULL_MASK, cnt);
      if (cnt <= kCap * 32) {  // warp-uniform
        __syncwarp();
        int base = 0;
        for (int i = 0; i < n_i; ++i) {
          const uint32_t k = target_key(c, i * 32 + lane, T);
          const bool sel = k <= U;
          const unsigned sb = __ballot_sync(TB_FULL_MASK, sel);
          if (sel) {
            const int p = base + __popc(sb & lt_mask);
            ckey[p] = k;
            cidx[p] = (uint16_t)(i * 32 + lane);
          }
          base += __popc(sb);
        }
        __syncwarp();
        const uint32_t tau = select_from_list<kCap, true>(c, ckey, cidx, cnt, K, 0u, U, lane, lt_mask);
        if (lane == 0) { rs[0] = c.sx; rs[1] = c.sy; rs[2] = __uint_as_float(tau); }
        continue;
      }
    }

    // general path: the bisection of kth_smallest<TPL, false> over all keys, one pass over shared memory per probe
    uint32_t lo, hi;
    state_bracket(c, rs, &lo, &hi);
    while (lo < hi) {
      const uint32_t mid = lo + ((hi - lo) >> 1);
      int cn = 0;
      for (int i = 0; i < n_i; ++i) cn += (target_key(c, i * 32 + lane, T) <= mid);
      cn = __reduce_add_sync(TB_FULL_MASK, cn);
      if (cn >= K) hi = mid; else lo = mid + 1u;
    }
    const uint32_t tau = lo;
    int c_lt = 0;
    for (int i = 0; i < n_i; ++i) c_lt += (target_key(c, i * 32 + lane, T) < tau);
    const int need_ties = K - __reduce_add_sync(TB_FULL_MASK, c_lt);
    int n_out = 0, n_tie = 0;
    for (int i = 0; i < n_i; ++i) {
      const uint32_t k = target_key(c, i * 32 + lane, T);
      const bool is_tie = k == tau;
      const unsigned tie_b = __ballot_sync(TB_FULL_MASK, is_tie);
      const bool sel = (k < tau) || (is_tie && n_tie + __popc(tie_b & lt_mask) < need_ties);
      const unsigned sel_b = __ballot_sync(TB_FULL_MASK, sel);
      if (sel) emit(c, n_out + __popc(sel_b & lt_mask), i * 32 + lane);
      n_out += __popc(sel_b);
      n_tie += __popc(tie_b);
    }
    if (lane == 0) { rs[0] = c.sx; rs[1] = c.sy; rs[2] = __uint_as_float(tau); }
  }
}

size_t smem_bytes(int T) { return (size_t)T * 12 + ((T + 15) / 16) * 16 + (size_t)kWarps * kCap * 32 * 6; }

template <int TPL, bool kFast>
int launch(const float* src_pose, const uint8_t* src_invalid, const float* tgt_pose, const uint8_t* tgt_invalid,
           int B, int S, int T, int div, int K, float dist_limit, int32_t* out_idx, uint8_t* out_invalid,
           float* out_rel, int ldk, int koff, const int32_t* tgt_index_map, float* row_state, int sorted_by_x,
           cudaStream_t st) {
  dim3 grid((S + kWarps * kRowsPerWarp - 1) / (kWarps * kRowsPerWarp), B);
  if (kFast && row_state && sorted_by_x && TPL >= 8) {
    knn_slab_kernel<<<grid, kWarps * 32, smem_bytes(T), st>>>(src_pose, src_invalid, tgt_pose, tgt_invalid, S, T, div,
                                                              K, dist_limit, out_idx, out_invalid, out_rel, ldk, koff,
                                                              tgt_index_map, row_state);
  } else {
    knn_select_kernel<TPL, kFast><<<grid, kWarps * 32, smem_bytes(T), st>>>(
        src_pose, src_invalid, tgt_pose, tgt_invalid, S, T, div, K, dist_limit, out_idx, out_invalid, out_rel, ldk,
        koff, tgt_index_map, row_state, sorted_by_x);
  }
  TB_CHECK_LAUNCH();
  return TB_OK;
}

template <bool kFast>
int dispatch(const float* src_pose, const uint8_t* src_invalid, const float* tgt_pose, const uint8_t* tgt_invalid,
             int B, int S, int T, int div, int K, float dist_limit, int32_t* out_idx, uint8_t* out_invalid,
             float* out_rel, int ldk, int koff, const int32_t* tgt_index_map, float* row_state, int sorted_by_x,
             cudaStream_t st) {
#define TB_KNN_ARGS src_pose, src_invalid, tgt_pose, tgt_invalid, B, S, T, div, K, dist_limit, out_idx, out_invalid, \
                    out_rel, ldk, koff, tgt_index_map, row_state, sorted_by_x, st
  if (T <= 64) return launch<2, kFast>(TB_KNN_ARGS);
  if (T <= 128) return launch<4, kFast>(TB_KNN_ARGS);
  if (T <= 256) return launch<8, kFast>(TB_KNN_ARGS);
  if (T <= 512) return launch<16, kFast>(TB_KNN_ARGS);
  if (T <= 1024) return launch<32, kFast>(TB_KNN_ARGS);
  if (T <= 2048) return launch<64, kFast>(TB_KNN_ARGS);
#undef TB_KNN_ARGS
  return TB_ERR_UNSUPPORTED;
}

}  // namespace

extern "C" int tb_knn_select(const float* src_pose, const uint8_t* src_invalid, const float* tgt_pose,
                             const uint8_t* tgt_invalid, int B, int S, int T, int tgt_batch_div, int K,
                             float dist_limit, int32_t* out_idx, uint8_t* out_invalid, float* out_rel, int out_ldk,
                             int out_koff, const int32_t* tgt_index_map, float* row_state, int flags,
                             void* stream) {
  if (!src_pose || !src_invalid || !tgt_pose || !tgt_invalid || !out_idx || !out_invalid || !out_rel)
    return TB_ERR_NULL;
  if (B <= 0 || S <= 0 || T <= 0 || tgt_batch_div <= 0 || out_koff < 0 || out_ldk < out_koff + K)
    return TB_ERR_BAD_SHAPE;
  if (!(0 < K && K < T)) return TB_ERR_KNN_RANGE;
  if (B > 65535) return TB_ERR_UNSUPPORTED;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int sorted_by_x = flags & TB_KNN_SORTED_BY_X;
  if (flags & TB_KNN_REFERENCE)
    return dispatch<false>(src_pose, src_invalid, tgt_pose, tgt_invalid, B, S, T, tgt_batch_div, K, dist_limit,
                           out_idx, out_invalid, out_rel, out_ldk, out_koff, tgt_index_map, row_state, sorted_by_x, st);
  return dispatch<true>(src_pose, src_invalid, tgt_pose, tgt_invalid, B, S, T, tgt_batch_div, K, dist_limit, out_idx,
                        out_invalid, out_rel, out_ldk, out_koff, tgt_index_map, row_state, sorted_by_x, st);
}
