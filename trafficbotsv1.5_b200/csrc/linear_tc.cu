// Tensor-core projection path (tb_linear precision 1): Y = epilogue(X W^T + bias) on the 5th-gen tensor cores.
//   tcgen05.mma kind::tf32 (fp32 operands straight from HBM, no conversion pass), fp32 accumulators in TMEM,
//   operands staged by TMA (cp.async.bulk.tensor.2d, 128-byte swizzle) through a 4-stage mbarrier pipeline,
//   warp-specialised: warps 0-7 epilogue (tcgen05.ld -> bias/ReLU/mask/residual -> global), warp 8 TMA producer,
//   warp 9 MMA issuer + TMEM allocator. Two TMEM accumulator buffers overlap the epilogue of tile n with the MMAs of
//   tile n+1. Persistent CTAs (one per SM) walk the (m, n) tiles n-fastest, so an A tile is fetched from HBM once and
//   re-read from L2 by the neighbouring SMs; the epilogue transposes each 32x32 accumulator block through swizzled
//   shared memory so that global stores / residual loads are full 128-byte lines.
// Shapes the TMA constraints do not cover (K or ldx not a multiple of 4 floats, misaligned pointers) are executed by
// the fp32 FFMA kernel instead (higher precision, same semantics). Narrow outputs (N = 2, 5, 6) run as one 128-wide
// tile whose missing weight rows are TMA zero fill.
#include <cuda.h>
#include <cuda_fp16.h>
#include "common.cuh"

int tb_linear_f32(const float* X, int ldx, const float* W, const float* bias, int bias_group, float* Y, int ldy, int M,
                  int N, int K,
                  int relu, const uint8_t* mask_pre, const float* res, int ldr, const uint8_t* mask_post,
                  cudaStream_t st);

namespace {

constexpr int BM = 128, BN = 128;
constexpr int BK_BYTES = 128;  // one k-block = one swizzle-128B row per operand row: 32 tf32/fp32 or 64 fp16 elements
constexpr int STAGES = 4;
constexpr int A_BYTES = BM * BK_BYTES, B_BYTES = BN * BK_BYTES;
constexpr int EPI_WARPS = 16;                 // 4 warps per TMEM lane quarter, each owning BN/4 of the tile's columns
constexpr int COLS_PER_WARP = BN / (EPI_WARPS / 4);
constexpr int NUM_THREADS = (EPI_WARPS + 2) * 32;
constexpr int TMEM_COLS = 2 * BN;
constexpr int EPI_BYTES = EPI_WARPS * 32 * 32 * 4;  // one 32x32 fp32 staging block per epilogue warp
constexpr int LN_BYTES = 2 * 4 * 4 * 32 * 8;          // fused LayerNorm: (sum, M2) partials [parity][quarter][col block][row]
constexpr size_t SMEM_BYTES = 1024 /*align slack*/ + (size_t)STAGES * (A_BYTES + B_BYTES) + EPI_BYTES + LN_BYTES + 256;

struct Epi {
  const float* bias; int bgroup; int relu; const uint8_t* mask_pre; const float* res; int ldr; const uint8_t* mask_post;
  __half* yh; int ldyh; int colh;  // columns >= colh (multiple of 32) are written as fp16 to yh[row*ldyh + col - colh]
  // fused LayerNorm of the output rows (N == 128, one n tile): ln_out[row] = fp16(LN(Y[row]) * gamma + beta)
  const float* ln_g; const float* ln_b; __half* ln_out; int ld_ln;
  unsigned int* sat_flag;  // fp16 range guard (common.cuh): ORed with 1 when an fp16 output value saturated
};
struct LnCtx { float2* part; uint32_t st_s; int quarter, half, parity; };

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "DONE:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
template <bool F16>
__device__ __forceinline__ void umma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                     uint32_t accumulate) {
  if (F16)
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
  else
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// K-major operand tile, 128-byte swizzle: rows of 128 B, 8-row atoms of 1024 B (SBO), LBO unused (canonical 1),
// descriptor version 1 (Blackwell), layout type 2 = SWIZZLE_128B (cute/arch/mma_sm100_desc.hpp bit layout).
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr) {
  return (uint64_t)((saddr & 0x3FFFF) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
// Instruction descriptor: D fp32 (bit 4), A/B format at bits 7 / 10 (kind::tf32: 2 = tf32; kind::f16: 0 = fp16),
// K-major A and B, N>>3 at bit 17, M>>4 at bit 24.
__host__ __device__ constexpr uint32_t make_idesc(int m, int n, bool f16) {
  return (1u << 4) | ((f16 ? 0u : 2u) << 7) | ((f16 ? 0u : 2u) << 10) | ((uint32_t)(n >> 3) << 17) |
         ((uint32_t)(m >> 4) << 24);
}

// Store phase of the epilogue for one 32x32 block: lane -> (row 4i + rsub, 16-byte chunk cc), 8 rows per lane.
// Everything that does not change inside the loop is a template parameter or hoisted (ncu source page of the first
// version: 339 warp instructions per block, ~20 per stored row of which 10 were 64-bit address arithmetic and row
// bound checks; the projections with K = 128 are bound by the epilogue's instruction issue). ALL: the block has all
// 32 rows (every block but the last M tile's). Residual rows and row masks (EXTRA) are fetched by `Prefetch` before the
// accumulator is waited for, so their latency overlaps the MMAs of the tile.
struct Prefetch {
  float4 rv[8];
  uint32_t zero_pre, zero_post;  // bit i: row 4i + rsub is masked
};
template <bool ALL>
__device__ __forceinline__ void prefetch_rows(Prefetch& pf, int rsub, int rbase, int col, int M, const Epi& ep) {
  pf.zero_pre = pf.zero_post = 0u;
  const int row0 = rbase + rsub;
  const float* rp = ep.res ? ep.res + (size_t)row0 * ep.ldr + col : nullptr;
  const size_t rstep = (size_t)4 * ep.ldr;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    pf.rv[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (ALL || row0 + 4 * i < M) {
      if (rp) pf.rv[i] = *reinterpret_cast<const float4*>(rp);
      if (ep.mask_pre && ep.mask_pre[row0 + 4 * i]) pf.zero_pre |= 1u << i;
      if (ep.mask_post && ep.mask_post[row0 + 4 * i]) pf.zero_post |= 1u << i;
    }
    if (rp) rp += rstep;
  }
}
// Store-phase row sums: q[i] is this lane's partial of row 4 i + rsub; a butterfly over the 8 lanes of the row group
// (7 shuffles) leaves lane (rsub, cc) with the full 32-column sum of row 4 cc + rsub.
__device__ __forceinline__ float rowgroup_sum(const float (&q)[8], int cc) {
  const bool b2 = cc & 4, b1 = cc & 2, b0 = cc & 1;
  float t[4], u[2];
#pragma unroll
  for (int j = 0; j < 4; ++j) t[j] = (b2 ? q[j + 4] : q[j]) + __shfl_xor_sync(TB_FULL_MASK, b2 ? q[j] : q[j + 4], 4);
#pragma unroll
  for (int j = 0; j < 2; ++j) u[j] = (b1 ? t[j + 2] : t[j]) + __shfl_xor_sync(TB_FULL_MASK, b1 ? t[j] : t[j + 2], 2);
  return (b0 ? u[1] : u[0]) + __shfl_xor_sync(TB_FULL_MASK, b0 ? u[0] : u[1], 1);
}
template <bool RELU, bool TO_H, bool EXTRA, bool ALL, bool LN = false>
__device__ __forceinline__ void store_block(uint32_t st_s, int rsub, int cc, int rbase, int col, int M, float4 bv,
                                            float* __restrict__ Y, int ldy, const Epi& ep, const Prefetch& pf,
                                            const LnCtx* ln = nullptr) {
  const int row0 = rbase + rsub;
  float* yp = Y + (size_t)row0 * ldy + col;
  const size_t ystep = (size_t)4 * ldy;
  __half* hp = TO_H ? ep.yh + (size_t)row0 * ep.ldyh + (col - ep.colh) : nullptr;
  const size_t hstep = (size_t)4 * ep.ldyh;
  // row rr = 4 i + rsub sits at rr * 128 bytes, chunk cc ^ (rr & 7): (rr & 7) alternates between rsub and rsub + 4
  const uint32_t sa0 = st_s + (uint32_t)rsub * 128u + ((uint32_t)(cc ^ rsub) << 4);
  const uint32_t sa1 = st_s + (uint32_t)rsub * 128u + ((uint32_t)(cc ^ (rsub + 4)) << 4);
  uint32_t hmax = 0u;  // TO_H: running |max| of the converted halves (fp16 range guard)
  float4 vv[8];  // all eight rows in flight before the first store (measured: 43 -> 38 us on the N = 896 projection)
#pragma unroll
  for (int i = 0; i < 8; ++i)
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(vv[i].x), "=f"(vv[i].y), "=f"(vv[i].z), "=f"(vv[i].w)
                 : "r"(((i & 1) ? sa1 : sa0) + (uint32_t)i * 512u));
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    if (ALL || row0 + 4 * i < M) {
      float4 v = vv[i];
      v.x += bv.x; v.y += bv.y; v.z += bv.z; v.w += bv.w;
      if (RELU) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
      if (EXTRA) {
        if (pf.zero_pre & (1u << i)) v = make_float4(0.f, 0.f, 0.f, 0.f);
        v.x += pf.rv[i].x; v.y += pf.rv[i].y; v.z += pf.rv[i].z; v.w += pf.rv[i].w;
        if (pf.zero_post & (1u << i)) v = make_float4(0.f, 0.f, 0.f, 0.f);
      }
      if (TO_H) {
        const uint32_t h0 = tb_pack_h2_sat(v.x, v.y), h1 = tb_pack_h2_sat(v.z, v.w);
        tb_track_h2(hmax, h0);
        tb_track_h2(hmax, h1);
        *reinterpret_cast<uint2*>(hp) = make_uint2(h0, h1);
      } else {
        *reinterpret_cast<float4*>(yp) = v;
      }
      if (LN) vv[i] = v;
    }
    if (TO_H) hp += hstep; else yp += ystep;
  }
  if (TO_H) tb_flag_if_sat(hmax, ep.sat_flag);
  if (LN) {
    // ---- LayerNorm of the finished rows (transformer_rpe.py:156-171, eps 1e-5): a row's 128 columns sit in the four
    // warps of this TMEM lane quarter. Each warp sums its 32 columns of a row shifted by c, the row's value in the
    // warp's first column (one broadcast from lane (rsub, 0)), and the squares of the shifted values, by a butterfly
    // over the 8 lanes of a row group (lane (rsub, cc) ends up owning row 4 cc + rsub). c is one of the 32 values, so
    // (mean_h - c)^2 <= M2_h and M2_h = sum (y - c)^2 - (sum (y - c))^2 / 32 loses at most a factor 33 to cancellation,
    // whatever the row's offset. The four warps' (sum, M2) partials go through shared memory + a 128-thread named
    // barrier and merge with Chan's formula M2 = sum M2_h + 32 sum (mean_h - mean)^2. Statistics back to the lanes
    // through the warp's staging block.
    float c[8], q1[8], q2[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      c[i] = __shfl_sync(TB_FULL_MASK, vv[i].x, rsub << 3);
      const float dx = vv[i].x - c[i], dy = vv[i].y - c[i], dz = vv[i].z - c[i], dw = vv[i].w - c[i];
      q1[i] = (dx + dy) + (dz + dw);
      q2[i] = fmaf(dx, dx, fmaf(dy, dy, fmaf(dz, dz, dw * dw)));
    }
    const float w1 = rowgroup_sum(q1, cc), w2 = rowgroup_sum(q2, cc);
    float c_own = c[0];  // the shift of the row this lane owns (row 4 cc + rsub: i = cc)
#pragma unroll
    for (int i = 1; i < 8; ++i) c_own = cc == i ? c[i] : c_own;
    const int own = 4 * cc + rsub;  // the block row this lane now holds the 32-column (sum, M2) of
    float2* part = ln->part + (ln->parity * 4 + ln->quarter) * 4 * 32;
    part[ln->half * 32 + own] = make_float2(fmaf(32.f, c_own, w1), fmaf(-w1, w1 * (1.f / 32.f), w2));
    asm volatile("bar.sync %0, 128;" ::"r"(1 + ln->quarter) : "memory");
    float S1 = 0.f;
#pragma unroll
    for (int h = 0; h < 4; ++h) S1 += part[h * 32 + own].x;
    const float mean = S1 * (1.f / BN);
    float M2 = 0.f;
#pragma unroll
    for (int h = 0; h < 4; ++h) {
      const float2 pp = part[h * 32 + own];
      const float d = fmaf(pp.x, 1.f / 32.f, -mean);
      M2 = fmaf(32.f * d, d, M2 + pp.y);
    }
    const float rstd = 1.f / sqrtf(M2 * (1.f / BN) + 1e-5f);
    __syncwarp();  // every lane has read its rows from the staging block
    asm volatile("st.shared.v2.f32 [%0], {%1,%2};" ::"r"(st_s + (uint32_t)own * 8u), "f"(mean), "f"(rstd) : "memory");
    __syncwarp();
    const float4 gg = __ldg(reinterpret_cast<const float4*>(ep.ln_g + col));
    const float4 be = __ldg(reinterpret_cast<const float4*>(ep.ln_b + col));
    __half* lp = ep.ln_out + (size_t)row0 * ep.ld_ln + col;
    const size_t lstep = (size_t)4 * ep.ld_ln;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      if (ALL || row0 + 4 * i < M) {
        float mu, rs;
        asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(mu), "=f"(rs) : "r"(st_s + (uint32_t)(4 * i + rsub) * 8u));
        const __half2 h0 = __floats2half2_rn((vv[i].x - mu) * rs * gg.x + be.x, (vv[i].y - mu) * rs * gg.y + be.y);
        const __half2 h1 = __floats2half2_rn((vv[i].z - mu) * rs * gg.z + be.z, (vv[i].w - mu) * rs * gg.w + be.w);
        *reinterpret_cast<uint2*>(lp) =
            make_uint2(*reinterpret_cast<const uint32_t*>(&h0), *reinterpret_cast<const uint32_t*>(&h1));
      }
      lp += lstep;
    }
  }
}

// F16: operands are fp16 in memory (kind::f16, 64 elements per k-block) instead of fp32 read as tf32 (32 per k-block)
// LN: the fused-LayerNorm epilogue (its own instantiation: its register pressure must not leak into the others)
template <bool F16, bool LN>
__global__ void __launch_bounds__(NUM_THREADS, 1)
linear_tc_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                 float* __restrict__ Y, int ldy, int M, int N, int K, Epi ep) {
  constexpr int BK = F16 ? 64 : 32;  // elements per k-block
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sA = smem;
  uint8_t* sB = smem + STAGES * A_BYTES;
  float* sE = reinterpret_cast<float*>(smem + STAGES * (A_BYTES + B_BYTES));
  float2* sLN = reinterpret_cast<float2*>(smem + STAGES * (A_BYTES + B_BYTES) + EPI_BYTES);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + STAGES * (A_BYTES + B_BYTES) + EPI_BYTES + LN_BYTES);
  uint64_t* empty = full + STAGES;
  uint64_t* tfull = empty + STAGES;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = (N + BN - 1) / BN;
  const int total_tiles = ((M + BM - 1) / BM) * n_tiles;
  const int num_k = (K + BK - 1) / BK;

  if (warp == EPI_WARPS && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapA)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapB)) : "memory");
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], EPI_WARPS * 32); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == EPI_WARPS + 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;

  if (warp == EPI_WARPS) {
    // ===== TMA producer =====
    if (lane == 0) {
      int it = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const int m0 = (tile / n_tiles) * BM, n0 = (tile % n_tiles) * BN;
        for (int k = 0; k < num_k; ++k, ++it) {
          const int s = it % STAGES;
          mbar_wait(&empty[s], ((it / STAGES) & 1) ^ 1);
          mbar_expect_tx(&full[s], A_BYTES + B_BYTES);
          tma_load_2d(&mapA, &full[s], sA + s * A_BYTES, k * BK, m0);
          tma_load_2d(&mapB, &full[s], sB + s * B_BYTES, k * BK, n0);
        }
      }
    }
  } else if (warp == EPI_WARPS + 1) {
    // ===== MMA issuer (one elected lane) =====
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc(BM, BN, F16);
      int it = 0, lt = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++lt) {
        const int buf = lt & 1;
        mbar_wait(&tempty[buf], ((lt >> 1) & 1) ^ 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        for (int k = 0; k < num_k; ++k, ++it) {
          const int s = it % STAGES;
          mbar_wait(&full[s], (it / STAGES) & 1);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint64_t adesc = make_desc(smem_u32(sA + s * A_BYTES));
          const uint64_t bdesc = make_desc(smem_u32(sB + s * B_BYTES));
#pragma unroll
          for (int kk = 0; kk < BK_BYTES / 32; ++kk)  // UMMA_K = 8 tf32 / 16 fp16 = 32 bytes -> +2 in 16-byte units
            umma<F16>(tmem_base + buf * BN, adesc + 2 * kk, bdesc + 2 * kk, idesc, (k | kk) != 0);
          umma_commit(&empty[s]);  // frees the smem stage when these MMAs have read it
        }
        umma_commit(&tfull[buf]);  // accumulator of this tile complete
      }
    }
  } else {
    // ===== epilogue warps 0..7: warp w reads TMEM lanes [32*(w&3), +32) (rows m0 + 32*(w&3) + lane) and owns the
    // column slice (w>>2) of the tile =====
    const int quarter = warp & 3, half = warp >> 2;
    float* st = sE + warp * (32 * 32);  // this warp's 32x32 staging block, 16-byte chunks XOR-swizzled by row
    const uint32_t st_s = smem_u32(st);
    const bool extra = ep.mask_pre || ep.res || ep.mask_post;  // row masks / residual: the slower store variant
    const bool vec_ok = ((ldy & 3) == 0) && ((reinterpret_cast<uintptr_t>(Y) & 15) == 0) &&
                        (!ep.yh || (((ep.ldyh & 3) == 0) && ((reinterpret_cast<uintptr_t>(ep.yh) & 7) == 0))) &&
                        (!ep.res || (((ep.ldr & 3) == 0) && ((reinterpret_cast<uintptr_t>(ep.res) & 15) == 0))) &&
                        (!ep.bias || (((reinterpret_cast<uintptr_t>(ep.bias) & 15) == 0) && (!ep.bgroup || (N & 3) == 0)));
    const int rsub = lane >> 3, cc = lane & 7;  // store phase: lane -> (row i*4 + rsub, 16-byte chunk cc)
    int lt = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++lt) {
      const unsigned tmi = (unsigned)tile / (unsigned)n_tiles;
      const int m0 = (int)tmi * BM, n0 = (tile - (int)tmi * n_tiles) * BN;
      const int buf = lt & 1;
      const int rbase = m0 + quarter * 32;
      const bool all_rows = rbase + 32 <= M;
      bool waited = false;
      // grouped bias: this thread's accumulator row (TMEM lane) is fixed for the tile -> one division per tile
      const float* gb_row = (ep.bgroup && rbase + lane < M)
                                ? ep.bias + (size_t)((rbase + lane) / ep.bgroup) * N : nullptr;
#pragma unroll 1
      for (int c0 = half * COLS_PER_WARP; c0 < (half + 1) * COLS_PER_WARP; c0 += 32) {
        const int cbase = n0 + c0;
        if (cbase >= N) break;  // warp-uniform
        const bool fast = vec_ok && cbase + 32 <= N;
        Prefetch pf;
        if ((extra || LN) && fast) {  // residual rows / row masks of this block: in flight while the accumulator completes
          if (all_rows) prefetch_rows<true>(pf, rsub, rbase, cbase + cc * 4, M, ep);
          else prefetch_rows<false>(pf, rsub, rbase, cbase + cc * 4, M, ep);
        }
        if (!waited) {
          mbar_wait(&tfull[buf], (lt >> 1) & 1);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          waited = true;
        }
        uint32_t r[32];
        const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(buf * BN + c0);
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
            "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
            "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
            : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
              "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
              "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
              "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
            : "r"(taddr));
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        if (gb_row) {  // add the group's bias row while the accumulators are still row-per-thread
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            if (vec_ok && cbase + 32 <= N) {
              const float4 b4 = __ldg(reinterpret_cast<const float4*>(gb_row + cbase + j));
              r[j] = __float_as_uint(__uint_as_float(r[j]) + b4.x);
              r[j + 1] = __float_as_uint(__uint_as_float(r[j + 1]) + b4.y);
              r[j + 2] = __float_as_uint(__uint_as_float(r[j + 2]) + b4.z);
              r[j + 3] = __float_as_uint(__uint_as_float(r[j + 3]) + b4.w);
            } else {
#pragma unroll
              for (int q = 0; q < 4; ++q)
                if (cbase + j + q < N) r[j + q] = __float_as_uint(__uint_as_float(r[j + q]) + __ldg(gb_row + cbase + j + q));
            }
          }
        }
        // registers (row = lane) -> swizzled staging block
#pragma unroll
        for (int c = 0; c < 8; ++c)
          asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(st_s + (uint32_t)(lane * 32 + ((c ^ (lane & 7)) << 2)) * 4),
                       "r"(r[4 * c]), "r"(r[4 * c + 1]), "r"(r[4 * c + 2]), "r"(r[4 * c + 3]) : "memory");
        __syncwarp();
        const bool to_h = ep.yh != nullptr && cbase >= ep.colh;  // warp-uniform: colh is a multiple of 32
        if (fast) {
          const int col = cbase + cc * 4;
          float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
          if (ep.bias && !ep.bgroup) bv = __ldg(reinterpret_cast<const float4*>(ep.bias + col));
#define TB_STORE(R, H, X)                                                                          \
  do {                                                                                             \
    if (all_rows) store_block<R, H, X, true>(st_s, rsub, cc, rbase, col, M, bv, Y, ldy, ep, pf);   \
    else store_block<R, H, X, false>(st_s, rsub, cc, rbase, col, M, bv, Y, ldy, ep, pf);           \
  } while (0)
          if (LN) {  // host guarantees: N == BN, fp32 output, this (vectorised) path
            const LnCtx ln{sLN, st_s, quarter, half, lt & 1};
            if (all_rows) store_block<false, false, true, true, LN>(st_s, rsub, cc, rbase, col, M, bv, Y, ldy, ep, pf, &ln);
            else store_block<false, false, true, false, LN>(st_s, rsub, cc, rbase, col, M, bv, Y, ldy, ep, pf, &ln);
          } else if (extra) {
            if (ep.relu) { if (to_h) TB_STORE(true, true, true); else TB_STORE(true, false, true); }
            else { if (to_h) TB_STORE(false, true, true); else TB_STORE(false, false, true); }
          } else {
            if (ep.relu) { if (to_h) TB_STORE(true, true, false); else TB_STORE(true, false, false); }
            else { if (to_h) TB_STORE(false, true, false); else TB_STORE(false, false, false); }
          }
#undef TB_STORE
        } else {  // N tail / unaligned views: scalar, bounds-checked
#pragma unroll 1
          for (int i = 0; i < 32; ++i) {
            const int row = rbase + i, col = cbase + lane;
            if (row < M && col < N) {
              float t = st[i * 32 + ((((lane >> 2) ^ (i & 7)) << 2) | (lane & 3))];
              if (ep.bias && !ep.bgroup) t += __ldg(ep.bias + col);
              if (ep.relu) t = fmaxf(t, 0.f);
              if (ep.mask_pre && ep.mask_pre[row]) t = 0.f;
              if (ep.res) t += ep.res[(size_t)row * ep.ldr + col];
              if (ep.mask_post && ep.mask_post[row]) t = 0.f;
              if (to_h) {
                const uint32_t hv = tb_pack_h2_sat(t, 0.f);
                tb_flag_if_sat(hv & 0x7FFFu, ep.sat_flag);
                ep.yh[(size_t)row * ep.ldyh + (col - ep.colh)] = __ushort_as_half((unsigned short)(hv & 0xFFFFu));
              }
              else Y[(size_t)row * ldy + col] = t;
            }
          }
        }
        __syncwarp();
      }
      if (!waited) mbar_wait(&tfull[buf], (lt >> 1) & 1);  // column slice entirely past N: keep the phases in step
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      mbar_arrive(&tempty[buf]);
    }
  }

  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == EPI_WARPS + 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = []() -> EncodeTiledFn {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      return nullptr;
    return reinterpret_cast<EncodeTiledFn>(p);
  }();
  return fn;
}

// 2-D fp32 / fp16 tensor [rows, cols] with row stride ld (elements); box = 128 B of columns x box_rows, 128-byte
// swizzle, out-of-bounds elements read as zero (handles the M / N / K tails).
bool make_map(CUtensorMap* map, const void* ptr, int rows, int cols, int ld, int box_rows, bool f16) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return false;
  const int esz = f16 ? 2 : 4;
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstr[1] = {(cuuint64_t)ld * esz};
  cuuint32_t box[2] = {(cuuint32_t)(BK_BYTES / esz), (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  return enc(map, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(ptr), gdim,
             gstr, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace

int tb_linear_tc(const void* X, int ldx, const void* W, int in_f16, const float* bias, int bias_group, float* Y,
                 int ldy, int M, int N, int K,
                 int relu, const uint8_t* mask_pre, const float* res, int ldr, const uint8_t* mask_post,
                 void* Yh, int ldyh, int colh, cudaStream_t st, const float* ln_g, const float* ln_b, void* ln_out,
                 int ld_ln) {
  const int ea = in_f16 ? 8 : 4;  // elements per 16 bytes: TMA needs 16-byte aligned rows
  const bool ok = (K % ea == 0) && (ldx % ea == 0) && tb_aligned16(X) && tb_aligned16(W);
  if (ln_out) {  // fused LayerNorm: one n tile, the vectorised epilogue path, no ReLU / fp16 split / grouped bias
    if (!ok || N != BN || relu || Yh || bias_group) return TB_ERR_UNSUPPORTED;
    if ((ldy & 3) || !tb_aligned16(Y) || (res && ((ldr & 3) || !tb_aligned16(res))) || (bias && !tb_aligned16(bias)) ||
        !tb_aligned16(ln_g) || !tb_aligned16(ln_b) || (ld_ln & 3) || (reinterpret_cast<uintptr_t>(ln_out) & 7))
      return TB_ERR_MISALIGNED;
  }
  if (!ok) {
    if (Yh || in_f16) return TB_ERR_UNSUPPORTED;  // the fp32 kernel has no fp16 input / output path
    return tb_linear_f32(static_cast<const float*>(X), ldx, static_cast<const float*>(W), bias, bias_group, Y, ldy, M, N, K,
                         relu, mask_pre, res, ldr, mask_post, st);
  }
  CUtensorMap mapA, mapB;
  if (!make_map(&mapA, X, M, K, ldx, BM, in_f16) || !make_map(&mapB, W, N, K, K, BN, in_f16)) return TB_ERR_CUDA;
  static bool attr_set = false;
  if (!attr_set) {
    if (cudaFuncSetAttribute(linear_tc_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)SMEM_BYTES) != cudaSuccess ||
        cudaFuncSetAttribute(linear_tc_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)SMEM_BYTES) != cudaSuccess ||
        cudaFuncSetAttribute(linear_tc_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)SMEM_BYTES) != cudaSuccess ||
        cudaFuncSetAttribute(linear_tc_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)SMEM_BYTES) != cudaSuccess)
      return TB_ERR_CUDA;
    attr_set = true;
  }
  const int m_tiles = (M + BM - 1) / BM, n_tiles = (N + BN - 1) / BN;
  static int num_sms = 0;
  if (num_sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || num_sms <= 0)
      num_sms = 148;
  }
  const int total = m_tiles * n_tiles;
  const int grid = total < num_sms ? total : num_sms;  // persistent: one CTA per SM
  Epi ep{bias, bias_group, relu, mask_pre, res, ldr, mask_post, static_cast<__half*>(Yh), ldyh, colh,
         ln_g, ln_b, static_cast<__half*>(ln_out), ld_ln, tb_fp16_flag_ptr};
  if (ln_out) {
    if (in_f16) linear_tc_kernel<true, true><<<grid, NUM_THREADS, SMEM_BYTES, st>>>(mapA, mapB, Y, ldy, M, N, K, ep);
    else linear_tc_kernel<false, true><<<grid, NUM_THREADS, SMEM_BYTES, st>>>(mapA, mapB, Y, ldy, M, N, K, ep);
  } else {
    if (in_f16) linear_tc_kernel<true, false><<<grid, NUM_THREADS, SMEM_BYTES, st>>>(mapA, mapB, Y, ldy, M, N, K, ep);
    else linear_tc_kernel<false, false><<<grid, NUM_THREADS, SMEM_BYTES, st>>>(mapA, mapB, Y, ldy, M, N, K, ep);
  }
  TB_CHECK_LAUNCH();
  return TB_OK;
}
