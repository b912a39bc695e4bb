// Fused MLP chain on the 5th-gen tensor cores (tb_chain_*): a whole sequence of small dense layers
// (Linear + bias + ReLU + row masks + residual [+ LayerNorm]) over one 128-row tile per CTA, with every intermediate
// activation kept on the SM. Replaces, per policy iteration of the rollout,
//   * the 20-launch head chain navi_encoder.mlp_pe -> add_navi (mlp_in, mlp) -> add_latent (mlp) -> action head
//     (models/traffic_bots.py:191-217, modules/add_navi_latent.py:46-64, modules/action_head.py:78-82) by ONE launch,
//   * FFN-1 -> ReLU -> FFN-2 -> +residual -> LayerNorm of every transformer layer (transformer_rpe.py:236-245) by
//     one launch: the [rows, 512] hidden tensor never reaches HBM.
// The separate launches are bound by their epilogues and by HBM round trips of 32-100 MB each, not by the MMAs
// (profiles/r1/ncu_final_linear_tc.summary.txt); here a tile's chain is
//   tcgen05.mma (A: fp16 activation tile in shared memory, 128-byte-swizzled K-major; B: fp16 weight k-blocks streamed
//   by TMA through an mbarrier ring; D: fp32 in TMEM)  ->  tcgen05.ld  ->  bias / ReLU / mask / residual in registers
//   ->  fp16 rows written straight into the NEXT layer's A-operand layout (no transpose: a thread owns an accumulator
//   row, and a K-major operand row is contiguous)  ->  fence.proxy.async  ->  mbarrier  ->  next tcgen05.mma.
// A chain is a "program": up to 32 units (GEMM units of <= 128 output features and LOAD units that bring a tile of an
// external fp32 / fp16 row-major tensor into an activation buffer), encoded once by the host together with the TMA
// descriptors of its weight matrices. Warp roles: 16 epilogue warps (4 per TMEM lane quarter, 32 columns each),
// 1 TMA producer, 1 MMA issuer. Persistent CTAs, one per SM.
#include <cuda.h>
#include <cuda_fp16.h>

#include <cstring>

#include "common.cuh"

namespace {

constexpr int TM = 128;                       // rows per tile
constexpr int KB_BYTES = TM * 128;            // one k-block of an activation buffer: [128 rows x 64 halves]
constexpr int BUF_BYTES = 2 * KB_BYTES;       // activation buffer: 128 columns = two k-blocks
constexpr int WSTAGE_BYTES = 128 * 128;       // weight stage: [128 output features x 64 halves]
constexpr int EPI_WARPS = 16;
constexpr int NUM_THREADS = (EPI_WARPS + 2) * 32;
constexpr int MAX_UNITS = TB_CHAIN_MAX_UNITS;
constexpr int MAX_MAPS = 24;
constexpr int MAX_BUF = 5;
constexpr int SMEM_MAX = 227 * 1024;

// Device-side unit record (192 bytes, staged in shared memory). The fields a warp needs on its critical path sit in
// 16-byte groups that are fetched with ONE ld.shared.v4 (ncu: a chain of load -> compare -> branch on individual
// fields cost more than the arithmetic of the epilogue).
enum : int { F_LOAD = 1, F_RELU = 2, F_MPRE = 4, F_MPOST = 8, F_RES = 16, F_OBUF = 32, F_OG = 64, F_OH = 128, F_LN = 256,
             F_SRC16 = 512 };
struct UnitDev {
  int flags, tmem_col, out_off, n_valid;   // epilogue group
  int map, n0, nk, n_wait;                 // producer / MMA group
  int wait[8];                             // units whose epilogue must have arrived before this unit's MMAs (n_wait used)
  int a_off[TB_CHAIN_MAX_KB];              // byte offset of every k-block's A tile in the activation area
  const float* bias;                       // [>= n0 + 128] or NULL (model constants, baked device pointers)
  const float* ln_g;
  const float* ln_b;
  int mask_pre, mask_post;                 // binding indices
  int res, ldr, res_col;                   // fp32 residual rows
  int out_g, ldg, g_col;                   // fp32 global output
  int out_h, ldh, h_col;                   // fp16 global output
  int ln_out, ld_ln;                       // fp16 LayerNorm(output row) -> global
  int src, lds, src_col;                   // LOAD source
  int pad_[2];
};
static_assert(sizeof(UnitDev) == 192, "unit record layout");

struct Header {
  int n_units, n_maps, n_buf, n_stage, total_boxes, pad[3];
};

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
      "CH_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra CH_DONE;\n\t"
      "bra CH_WAIT;\n\t"
      "CH_DONE:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_2d(const void* map, uint64_t* bar, void* dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// K-major tile, 128-byte swizzle, 8-row atoms of 1024 B (same encoding as linear_tc.cu)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr) {
  return (uint64_t)((saddr & 0x3FFFF) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)2 << 61);
}
constexpr uint32_t kIdesc = (1u << 4) | ((uint32_t)(128 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);  // f16 x f16 -> f32, M = N = 128

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}

struct Bind { void* p[TB_CHAIN_MAX_BIND]; };

// byte address of the 16-byte chunk `chunk` (0..7) of row `row` in a k-block tile (SWIZZLE_128B K-major layout)
__device__ __forceinline__ uint32_t kb_chunk_addr(uint32_t kb_base, int row, int chunk) {
  return kb_base + (uint32_t)(row >> 3) * 1024u + (uint32_t)(row & 7) * 128u + (uint32_t)((chunk ^ (row & 7)) << 4);
}

__device__ __forceinline__ int4 lds128(uint32_t a) {
  int4 v;
  asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ int lds32(uint32_t a) {
  int v;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ uint64_t lds64(uint32_t a) {
  uint64_t v;
  asm volatile("ld.shared.b64 %0, [%1];" : "=l"(v) : "r"(a));
  return v;
}
#define UOFF(f) ((uint32_t)offsetof(UnitDev, f))

__global__ void __launch_bounds__(NUM_THREADS, 1)
mlp_chain_kernel(const uint8_t* __restrict__ prog, const Bind bind, int M) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const Header* hd = reinterpret_cast<const Header*>(prog);
  const UnitDev* g_units = reinterpret_cast<const UnitDev*>(prog + 64);
  const uint8_t* maps = prog + 64 + ((sizeof(UnitDev) * MAX_UNITS + 63) & ~(size_t)63);
  const int n_units = hd->n_units, n_buf = hd->n_buf, n_stage = hd->n_stage;

  uint8_t* sAct = smem;                                   // n_buf activation buffers
  uint8_t* sW = smem + (size_t)n_buf * BUF_BYTES;         // weight ring
  uint8_t* tail = sW + (size_t)n_stage * WSTAGE_BYTES;
  UnitDev* units = reinterpret_cast<UnitDev*>(tail);      // the program's unit table
  tail += (size_t)n_units * sizeof(UnitDev);
  float* sBias = reinterpret_cast<float*>(tail);          // [n_units][128] bias of every unit (zeros when absent)
  tail += (size_t)n_units * 128 * 4;
  float2* sLN = reinterpret_cast<float2*>(tail);          // [4 column quarters][128 rows] partial (sum, sum of squares)
  tail += 4 * TM * 8;
  uint64_t* sBind = reinterpret_cast<uint64_t*>(tail);    // the binding pointers (indexed dynamically: not from param space)
  tail += TB_CHAIN_MAX_BIND * 8;
  uint64_t* full = reinterpret_cast<uint64_t*>(tail);
  uint64_t* empty = full + 8;
  uint64_t* acc_bar = empty + 8;                          // [MAX_UNITS] accumulator of unit u complete (MMA commit)
  uint64_t* act_bar = acc_bar + MAX_UNITS;                // [MAX_UNITS] epilogue / load of unit u done (one arrival per warp)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(act_bar + MAX_UNITS);
  const uint32_t units_s = smem_u32(units), bind_s = smem_u32(sBind), act_s = smem_u32(sAct);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = (M + TM - 1) / TM;

  for (int i = threadIdx.x; i < n_units * (int)(sizeof(UnitDev) / 4); i += NUM_THREADS)
    reinterpret_cast<uint32_t*>(units)[i] = reinterpret_cast<const uint32_t*>(g_units)[i];
  for (int i = threadIdx.x; i < n_units * 128; i += NUM_THREADS) {
    const UnitDev& gu = g_units[i >> 7];
    sBias[i] = (!(gu.flags & F_LOAD) && gu.bias) ? __ldg(gu.bias + gu.n0 + (i & 127)) : 0.f;
  }
  if (threadIdx.x < TB_CHAIN_MAX_BIND) sBind[threadIdx.x] = reinterpret_cast<uint64_t>(bind.p[threadIdx.x]);
  if (warp == EPI_WARPS && lane == 0) {
    for (int i = 0; i < hd->n_maps; ++i)
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(maps + (size_t)i * 128)) : "memory");
    for (int i = 0; i < n_stage; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    for (int i = 0; i < MAX_UNITS; ++i) { mbar_init(&acc_bar[i], 1); mbar_init(&act_bar[i], EPI_WARPS); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == EPI_WARPS + 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;

  if (warp == EPI_WARPS) {
    // ===== TMA producer: the weight k-blocks of every GEMM unit, in program order, once per tile =====
    if (lane == 0) {
      int it = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        for (int u = 0; u < n_units; ++u) {
          const int4 gq = lds128(units_s + u * (uint32_t)sizeof(UnitDev) + UOFF(map));  // map, n0, nk, n_wait
          for (int kb = 0; kb < gq.z; ++kb, ++it) {                                      // nk == 0 for LOAD units
            const int s = it % n_stage;
            mbar_wait(&empty[s], ((it / n_stage) & 1) ^ 1);
            mbar_expect_tx(&full[s], WSTAGE_BYTES);
            tma_load_2d(maps + (size_t)gq.x * 128, &full[s], sW + (size_t)s * WSTAGE_BYTES, kb * 64, gq.y);
          }
        }
      }
    }
  } else if (warp == EPI_WARPS + 1) {
    // ===== MMA issuer =====
    if (lane == 0) {
      int it = 0, lt = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++lt) {
        const uint32_t par = lt & 1;
        for (int u = 0; u < n_units; ++u) {
          const uint32_t ua = units_s + u * (uint32_t)sizeof(UnitDev);
          const int4 gq = lds128(ua + UOFF(map));  // map, n0, nk, n_wait
          if (gq.z == 0) continue;
          const int4 w0 = lds128(ua + UOFF(wait)), w1 = lds128(ua + UOFF(wait) + 16);
          const int4 a0 = lds128(ua + UOFF(a_off)), a1 = lds128(ua + UOFF(a_off) + 16);
          const int tcol = lds32(ua + UOFF(tmem_col));
          const int wl[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
          const int al[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
          for (int w = 0; w < 6; ++w)
            if (w < gq.w) mbar_wait(&act_bar[wl[w]], par);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
          for (int kb = 0; kb < TB_CHAIN_MAX_KB; ++kb) {
            if (kb < gq.z) {
              const int s = it % n_stage;
              mbar_wait(&full[s], (it / n_stage) & 1);
              asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
              const uint64_t adesc = make_desc(act_s + (uint32_t)al[kb]);
              const uint64_t bdesc = make_desc(smem_u32(sW + (size_t)s * WSTAGE_BYTES));
#pragma unroll
              for (int kk = 0; kk < 4; ++kk)  // UMMA_K = 16 halves = 32 bytes
                umma_f16(tmem_base + tcol, adesc + 2 * kk, bdesc + 2 * kk, kIdesc, (kb | kk) != 0);
              umma_commit(&empty[s]);
              ++it;
            }
          }
          umma_commit(&acc_bar[u]);
        }
      }
    }
  } else {
    // ===== epilogue / load warps: thread <-> tile row (TMEM lane); the four warps of a lane quarter (w & 3) split
    // the 128 columns of a unit into 32-column slices (w >> 2) =====
    const int quarter = warp & 3, cq = warp >> 2;
    const int row = quarter * 32 + lane;
    const int kblk = cq >> 1, chunk0 = (cq & 1) * 4;   // this slice inside a buffer: k-block, first 16-byte chunk
    auto bptr = [&](int i) { return reinterpret_cast<void*>(lds64(bind_s + 8u * (uint32_t)i)); };
    int lt = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++lt) {
      const uint32_t par = lt & 1;
      const int grow = tile * TM + row;
      const bool rok = grow < M;
      // the NEXT tile's external rows (LOAD sources, residuals) on their way to L2 while this tile computes: with one
      // tile in flight per SM every DRAM round trip is exposed otherwise (first tile: also its own rows, just in time)
      for (int pass = (lt == 0 ? 0 : 1); pass < 2; ++pass) {
        const int pr = pass == 0 ? grow : grow + (int)gridDim.x * TM;
        if (pr < M) {
          for (int u = 0; u < n_units; ++u) {
            const uint32_t ua = units_s + u * (uint32_t)sizeof(UnitDev);
            const int flags = lds32(ua);
            if (flags & F_LOAD) {
              const char* pp = static_cast<const char*>(bptr(lds32(ua + UOFF(src)))) +
                               ((size_t)pr * lds32(ua + UOFF(lds)) + lds32(ua + UOFF(src_col)) + cq * 32) * ((flags & F_SRC16) ? 2 : 4);
              asm volatile("prefetch.global.L2 [%0];" ::"l"(pp));
            } else if (flags & F_RES) {
              const float* pp = static_cast<const float*>(bptr(lds32(ua + UOFF(res)))) + (size_t)pr * lds32(ua + UOFF(ldr)) +
                                lds32(ua + UOFF(res_col)) + cq * 32;
              asm volatile("prefetch.global.L2 [%0];" ::"l"(pp));
            }
          }
        }
      }
      for (int u = 0; u < n_units; ++u) {
        const uint32_t ua = units_s + u * (uint32_t)sizeof(UnitDev);
        const int4 hq = lds128(ua);  // flags, tmem_col, out_off, n_valid
        const int flags = hq.x;
        if (flags & F_LOAD) {
          // ---- LOAD: 32 columns of this thread's row of an external tensor -> its slice of a buffer
          const uint32_t kb_base = act_s + (uint32_t)hq.z + (uint32_t)kblk * KB_BYTES;
          const int src = lds32(ua + UOFF(src)), lds_ = lds32(ua + UOFF(lds)), scol = lds32(ua + UOFF(src_col));
          if (flags & F_SRC16) {
            const __half* sp = static_cast<const __half*>(bptr(src)) + (size_t)grow * lds_ + scol + cq * 32;
            uint4 v[4];
#pragma unroll
            for (int c = 0; c < 4; ++c) v[c] = rok ? __ldg(reinterpret_cast<const uint4*>(sp + c * 8)) : make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
            for (int c = 0; c < 4; ++c)
              asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(kb_chunk_addr(kb_base, row, chunk0 + c)), "r"(v[c].x),
                           "r"(v[c].y), "r"(v[c].z), "r"(v[c].w) : "memory");
          } else {
            const float* sp = static_cast<const float*>(bptr(src)) + (size_t)grow * lds_ + scol + cq * 32;
            float4 a[8];
#pragma unroll
            for (int c = 0; c < 8; ++c) a[c] = rok ? ldg4(sp + c * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int c = 0; c < 4; ++c)
              asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(kb_chunk_addr(kb_base, row, chunk0 + c)),
                           "r"(tb_pack_h2_sat(a[2 * c].x, a[2 * c].y)), "r"(tb_pack_h2_sat(a[2 * c].z, a[2 * c].w)),
                           "r"(tb_pack_h2_sat(a[2 * c + 1].x, a[2 * c + 1].y)),
                           "r"(tb_pack_h2_sat(a[2 * c + 1].z, a[2 * c + 1].w)) : "memory");
          }
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          __syncwarp();
          if (lane == 0) mbar_arrive(&act_bar[u]);  // one arrival per warp
          continue;
        }
        // ---- GEMM epilogue: everything that does not depend on the accumulator is in flight before the wait
        bool z_pre = false, z_post = false;
        float4 rv[8];
        if (flags & (F_MPRE | F_MPOST | F_RES)) {  // rare units: masks / residual rows
          if (rok && (flags & F_MPRE)) z_pre = static_cast<const uint8_t*>(bptr(lds32(ua + UOFF(mask_pre))))[grow] != 0;
          if (rok && (flags & F_MPOST)) z_post = static_cast<const uint8_t*>(bptr(lds32(ua + UOFF(mask_post))))[grow] != 0;
          if (flags & F_RES) {
            const float* resp = static_cast<const float*>(bptr(lds32(ua + UOFF(res)))) +
                                (size_t)(rok ? grow : 0) * lds32(ua + UOFF(ldr)) + lds32(ua + UOFF(res_col)) + cq * 32;
#pragma unroll
            for (int j = 0; j < 8; ++j) rv[j] = *reinterpret_cast<const float4*>(resp + 4 * j);
          }
        }
        mbar_wait(&acc_bar[u], par);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (cq * 32 >= hq.w && !(flags & (F_OBUF | F_LN))) {  // narrow output (e.g. the 6-wide action head): nothing to read here
          asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
          __syncwarp();
          if (lane == 0) mbar_arrive(&act_bar[u]);
          continue;
        }
        float v[32];
        {
          uint32_t r[32];
          tmem_ld32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(hq.y + cq * 32), r);
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
        }
        {
          const uint32_t ba = smem_u32(sBias) + (uint32_t)(u * 128 + cq * 32) * 4u;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int4 b4 = lds128(ba + 16u * j);
            v[4 * j] += __int_as_float(b4.x); v[4 * j + 1] += __int_as_float(b4.y);
            v[4 * j + 2] += __int_as_float(b4.z); v[4 * j + 3] += __int_as_float(b4.w);
          }
        }
        if (flags & F_RELU) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
        }
        if (flags & (F_MPRE | F_MPOST | F_RES)) {
          if (z_pre) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = 0.f;
          }
          if (flags & F_RES) {
#pragma unroll
            for (int j = 0; j < 8; ++j) { v[4 * j] += rv[j].x; v[4 * j + 1] += rv[j].y; v[4 * j + 2] += rv[j].z; v[4 * j + 3] += rv[j].w; }
          }
          if (z_post) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = 0.f;
          }
        }
        const int nv = hq.w - cq * 32;  // columns of this slice that exist for out_g / out_h (< 32: narrow output)
        if (flags & (F_OBUF | F_OH)) {
          uint32_t h[16], hm = 0u;
#pragma unroll
          for (int j = 0; j < 16; ++j) { h[j] = tb_pack_h2_sat(v[2 * j], v[2 * j + 1]); tb_track_h2(hm, h[j]); }
          if (!(flags & F_OBUF) && nv < 32) {  // only out_h's c < n_valid are stored: only they can raise the flag
            hm = 0u;
#pragma unroll
            for (int j = 0; j < 16; ++j) tb_track_h2(hm, 2 * j + 1 < nv ? h[j] : 2 * j < nv ? (h[j] & 0xFFFFu) : 0u);
          }
          if (flags & F_OBUF) {  // fp16 row slice -> the next A operand (K-major, 128-byte swizzle)
            const uint32_t kb_base = act_s + (uint32_t)hq.z + (uint32_t)kblk * KB_BYTES;
#pragma unroll
            for (int c = 0; c < 4; ++c)
              asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(kb_chunk_addr(kb_base, row, chunk0 + c)), "r"(h[4 * c]),
                           "r"(h[4 * c + 1]), "r"(h[4 * c + 2]), "r"(h[4 * c + 3]) : "memory");
          }
          if ((flags & F_OH) && rok) {
            __half* hp = static_cast<__half*>(bptr(lds32(ua + UOFF(out_h)))) + (size_t)grow * lds32(ua + UOFF(ldh)) +
                         lds32(ua + UOFF(h_col)) + cq * 32;
            if (nv >= 32) {
#pragma unroll
              for (int c = 0; c < 4; ++c)
                *reinterpret_cast<uint4*>(hp + 8 * c) = make_uint4(h[4 * c], h[4 * c + 1], h[4 * c + 2], h[4 * c + 3]);
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (j < nv) hp[j] = __ushort_as_half((unsigned short)(h[j >> 1] >> (16 * (j & 1))));
            }
          }
          if (rok) tb_flag_if_sat(hm, static_cast<unsigned int*>(bptr(TB_CHAIN_MAX_BIND - 1)));
        }
        if ((flags & F_OG) && rok) {
          const int ldg = lds32(ua + UOFF(ldg)), gcol = lds32(ua + UOFF(g_col));
          float* gp = static_cast<float*>(bptr(lds32(ua + UOFF(out_g)))) + (size_t)grow * ldg + gcol + cq * 32;
          if (nv >= 32 && ((ldg | gcol) & 3) == 0) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) *reinterpret_cast<float4*>(gp + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (j < nv) gp[j] = v[j];
          }
        }
        if (flags & F_LN) {
          // LayerNorm of the 128-wide output row (transformer_rpe.py:156-171, eps 1e-5): this thread holds 32 of its
          // columns, the other three warps of the lane quarter the rest -> exchange (sum, M2) of the 32 columns through smem
          // and merge them with Chan's formula M2 = sum M2_q + 32 sum (mean_q - mean)^2. The 32 columns are summed
          // shifted by their first value c: (mean_q - c)^2 <= M2_q, so sum (v - c)^2 - (sum (v - c))^2 / 32 loses at
          // most a factor 33 to cancellation, whatever the row's offset (no E[v^2] - E[v]^2)
          const float c = v[0];
          float s1 = 0.f, m2 = 0.f;
#pragma unroll
          for (int j = 0; j < 32; ++j) { const float d = v[j] - c; s1 += d; m2 = fmaf(d, d, m2); }
          m2 = fmaf(-s1, s1 * (1.f / 32.f), m2);
          s1 = fmaf(32.f, c, s1);
          sLN[cq * TM + row] = make_float2(s1, m2);
          asm volatile("bar.sync %0, 128;" ::"r"(1 + quarter) : "memory");
          float2 o[4];
          s1 = 0.f;
#pragma unroll
          for (int q = 0; q < 4; ++q) { o[q] = sLN[q * TM + row]; s1 += o[q].x; }
          asm volatile("bar.sync %0, 128;" ::"r"(1 + quarter) : "memory");  // partials consumed: the slots may be rewritten
          const float mean = s1 * (1.f / 128.f);
          m2 = 0.f;
#pragma unroll
          for (int q = 0; q < 4; ++q) { const float d = fmaf(o[q].x, 1.f / 32.f, -mean); m2 = fmaf(32.f * d, d, m2 + o[q].y); }
          const float rstd = 1.f / sqrtf(m2 * (1.f / 128.f) + 1e-5f);
          if (rok) {
            const float* ln_g = reinterpret_cast<const float*>(lds64(ua + UOFF(ln_g)));
            const float* ln_b = reinterpret_cast<const float*>(lds64(ua + UOFF(ln_b)));
            __half* lp = static_cast<__half*>(bptr(lds32(ua + UOFF(ln_out)))) + (size_t)grow * lds32(ua + UOFF(ld_ln)) + cq * 32;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const float4 g0 = ldg4(ln_g + cq * 32 + 8 * c), g1 = ldg4(ln_g + cq * 32 + 8 * c + 4);
              const float4 b0 = ldg4(ln_b + cq * 32 + 8 * c), b1 = ldg4(ln_b + cq * 32 + 8 * c + 4);
              const float* x = v + 8 * c;
              *reinterpret_cast<uint4*>(lp + 8 * c) = make_uint4(
                  tb_pack_h2_sat((x[0] - mean) * rstd * g0.x + b0.x, (x[1] - mean) * rstd * g0.y + b0.y),
                  tb_pack_h2_sat((x[2] - mean) * rstd * g0.z + b0.z, (x[3] - mean) * rstd * g0.w + b0.w),
                  tb_pack_h2_sat((x[4] - mean) * rstd * g1.x + b1.x, (x[5] - mean) * rstd * g1.y + b1.y),
                  tb_pack_h2_sat((x[6] - mean) * rstd * g1.z + b1.z, (x[7] - mean) * rstd * g1.w + b1.w));
            }
          }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(&act_bar[u]);
      }
    }
  }

  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == EPI_WARPS + 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
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

// unit table + biases + LayerNorm partials + mbarriers + TMEM slot
int tail_bytes(int n_units) {
  return n_units * (int)sizeof(UnitDev) + n_units * 512 + 4 * TM * 8 + TB_CHAIN_MAX_BIND * 8 + (16 + 2 * MAX_UNITS) * 8 + 64;
}

size_t blob_bytes() { return 64 + ((sizeof(UnitDev) * MAX_UNITS + 63) & ~(size_t)63) + (size_t)MAX_MAPS * 128; }

// The bindings a program uses, checked from the host copy of the program before any launch: every index is below
// n_bind (else TB_ERR_BAD_SHAPE), not NULL (TB_ERR_NULL) and aligned for the widest access the kernel makes through it
// (TB_ERR_MISALIGNED): 16 bytes for LOAD sources (ldg4 / uint4), residual rows (float4), out_h and ln_out rows (uint4)
// and out_g rows with (ldg | g_col) % 4 == 0 (float4), 4 bytes for other out_g rows. LOAD sources are read through the
// non-coherent path (ld.global.nc), so a LOAD whose binding (same pointer) is also written by the launch through out_g /
// out_h / ln_out is refused (TB_ERR_UNSUPPORTED) unless both rows have the same pitch in bytes and their column byte
// ranges lie inside one row and do not overlap (the head chain reads the right half of the buffer it writes the left
// half of).
int check_bindings(const UnitDev* units, int n_units, void* const* bindings, int n_bind) {
  auto need = [&](int i, uintptr_t align) {
    if (i < 0 || i >= n_bind) return TB_ERR_BAD_SHAPE;
    if (!bindings[i]) return TB_ERR_NULL;
    return (reinterpret_cast<uintptr_t>(bindings[i]) & (align - 1)) ? TB_ERR_MISALIGNED : TB_OK;
  };
  for (int u = 0; u < n_units; ++u) {
    const UnitDev& d = units[u];
    int e = TB_OK;
    if (d.flags & F_LOAD) {
      if ((e = need(d.src, 16))) return e;
      continue;
    }
    if ((d.flags & F_MPRE) && (e = need(d.mask_pre, 1))) return e;
    if ((d.flags & F_MPOST) && (e = need(d.mask_post, 1))) return e;
    if ((d.flags & F_RES) && (e = need(d.res, 16))) return e;
    if ((d.flags & F_OG) && (e = need(d.out_g, ((d.ldg | d.g_col) & 3) ? 4 : 16))) return e;
    if ((d.flags & F_OH) && (e = need(d.out_h, 16))) return e;
    if ((d.flags & F_LN) && (e = need(d.ln_out, 16))) return e;
  }
  for (int u = 0; u < n_units; ++u) {
    const UnitDev& l = units[u];
    if (!(l.flags & F_LOAD)) continue;
    const long es = (l.flags & F_SRC16) ? 2 : 4, pitch = l.lds * es, lo = l.src_col * es, hi = lo + 128 * es;
    for (int v = 0; v < n_units; ++v) {
      const UnitDev& g = units[v];
      if (g.flags & F_LOAD) continue;
      const struct { int flag, idx; long pitch, lo, hi; } outs[3] = {
          {F_OG, g.out_g, g.ldg * 4L, g.g_col * 4L, (g.g_col + (long)g.n_valid) * 4L},
          {F_OH, g.out_h, g.ldh * 2L, g.h_col * 2L, (g.h_col + (long)g.n_valid) * 2L},
          {F_LN, g.ln_out, g.ld_ln * 2L, 0L, 256L}};
      for (const auto& o : outs)
        if ((g.flags & o.flag) && bindings[o.idx] == bindings[l.src] &&
            !(o.pitch == pitch && hi <= pitch && o.hi <= pitch && (hi <= o.lo || o.hi <= lo)))
          return TB_ERR_UNSUPPORTED;
    }
  }
  return TB_OK;
}

}  // namespace

extern "C" int tb_chain_program_bytes(void) { return (int)blob_bytes(); }

// Encode a chain program into `host_blob` (tb_chain_program_bytes() bytes); the caller copies it to 128-byte aligned
// device memory and passes that to tb_chain_run. Validates buffer hazards it can see statically.
extern "C" int tb_chain_encode(const tb_chain_unit* units, int n_units, int n_buf, void* host_blob) {
  if (!units || !host_blob) return TB_ERR_NULL;
  // 6 buffers would leave (227 KB - 1 KB - 192 KB - tail) / 16 KB = 1 weight stage even for one unit: 2..5 only
  if (n_units <= 0 || n_units > MAX_UNITS || n_buf < 2 || n_buf > MAX_BUF) return TB_ERR_BAD_SHAPE;
  EncodeTiledFn enc = get_encode();
  if (!enc) return TB_ERR_CUDA;
  uint8_t* blob = static_cast<uint8_t*>(host_blob);
  memset(blob, 0, blob_bytes());
  Header* hd = reinterpret_cast<Header*>(blob);
  UnitDev* out = reinterpret_cast<UnitDev*>(blob + 64);
  CUtensorMap* maps = reinterpret_cast<CUtensorMap*>(blob + 64 + ((sizeof(UnitDev) * MAX_UNITS + 63) & ~(size_t)63));
  static_assert(sizeof(CUtensorMap) == 128, "tensor map size");
  const int tail = tail_bytes(n_units);
  const int n_stage = (SMEM_MAX - 1024 - n_buf * BUF_BYTES - tail) / WSTAGE_BYTES;
  if (n_stage < 2) return TB_ERR_UNSUPPORTED;
  hd->n_units = n_units; hd->n_buf = n_buf; hd->n_stage = n_stage > 8 ? 8 : n_stage;
  int n_maps = 0, n_gemm = 0, total_boxes = 0;
  const void* map_w[MAX_MAPS];
  int map_k[MAX_MAPS], map_n[MAX_MAPS];
  int writer[8];      // unit that last wrote every activation buffer (-1: nobody yet)
  int gemm_unit[MAX_UNITS];
  for (int b = 0; b < 8; ++b) writer[b] = -1;
  for (int u = 0; u < n_units; ++u) {
    const tb_chain_unit& s = units[u];
    UnitDev& d = out[u];
    d.mask_pre = s.mask_pre; d.mask_post = s.mask_post; d.res = s.res; d.ldr = s.ldr; d.res_col = s.res_col;
    d.out_off = s.out_buf >= 0 ? s.out_buf * BUF_BYTES : 0;
    d.out_g = s.out_g; d.ldg = s.ldg; d.g_col = s.g_col; d.out_h = s.out_h; d.ldh = s.ldh; d.h_col = s.h_col;
    d.ln_out = s.ln_out; d.ld_ln = s.ld_ln; d.ln_g = s.ln_gamma; d.ln_b = s.ln_beta;
    d.src = s.src; d.lds = s.lds; d.src_col = s.src_col;
    d.bias = s.bias; d.n0 = s.n0; d.nk = 0; d.n_wait = 0;
    d.n_valid = s.n_valid > 0 ? s.n_valid : 128;
    d.flags = (s.kind == 1 ? F_LOAD : 0) | (s.relu ? F_RELU : 0) | (s.mask_pre >= 0 ? F_MPRE : 0) |
              (s.mask_post >= 0 ? F_MPOST : 0) | (s.res >= 0 ? F_RES : 0) | (s.out_buf >= 0 ? F_OBUF : 0) |
              (s.out_g >= 0 ? F_OG : 0) | (s.out_h >= 0 ? F_OH : 0) | (s.ln_out >= 0 ? F_LN : 0) | (s.src_f16 ? F_SRC16 : 0);
    if (s.out_buf >= n_buf) return TB_ERR_BAD_SHAPE;
    auto bad_bind = [](int b) { return b < -1 || b >= TB_CHAIN_MAX_BIND - 1; };
    if (bad_bind(s.mask_pre) || bad_bind(s.mask_post) || bad_bind(s.res) || bad_bind(s.out_g) || bad_bind(s.out_h) ||
        bad_bind(s.ln_out) || bad_bind(s.src))
      return TB_ERR_BAD_SHAPE;
    if (s.kind == 1) {  // LOAD
      if (s.src < 0 || s.out_buf < 0 || (s.src_f16 ? (s.lds | s.src_col) & 7 : (s.lds | s.src_col) & 3)) return TB_ERR_BAD_SHAPE;
    } else if (s.kind == 0) {
      if (!s.W || s.K <= 0 || (s.K & 63) || s.K / 64 > TB_CHAIN_MAX_KB || s.N <= 0 || s.n0 < 0 || s.n0 >= s.N ||
          s.n_valid > 128)
        return TB_ERR_BAD_SHAPE;
      if (!tb_aligned16(s.W) || (s.bias && !tb_aligned16(s.bias)) || (s.res >= 0 && ((s.ldr | s.res_col) & 3)) ||
          (s.out_h >= 0 && ((s.ldh | s.h_col) & 7)) ||
          (s.ln_out >= 0 && ((s.ld_ln & 7) || !s.ln_gamma || !s.ln_beta || !tb_aligned16(s.ln_gamma) ||
                             !tb_aligned16(s.ln_beta))))
        return TB_ERR_MISALIGNED;
      d.nk = s.K / 64;
      int m = -1;  // one tensor map per distinct (W, K, N): the same pointer read with another shape needs its own
      for (int i = 0; i < n_maps; ++i)
        if (map_w[i] == s.W && map_k[i] == s.K && map_n[i] == s.N) m = i;
      if (m < 0) {
        if (n_maps == MAX_MAPS) return TB_ERR_UNSUPPORTED;
        cuuint64_t gdim[2] = {(cuuint64_t)s.K, (cuuint64_t)s.N};
        cuuint64_t gstr[1] = {(cuuint64_t)s.K * 2};
        cuuint32_t box[2] = {64, 128};
        cuuint32_t estr[2] = {1, 1};
        if (enc(&maps[n_maps], CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(s.W), gdim, gstr, box, estr,
                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
          return TB_ERR_CUDA;
        map_w[n_maps] = s.W; map_k[n_maps] = s.K; map_n[n_maps] = s.N;
        m = n_maps++;
      }
      d.map = m;
      auto add_wait = [&](int unit) {
        if (unit < 0) return true;
        for (int i = 0; i < d.n_wait; ++i)
          if (d.wait[i] == unit) return true;
        if (d.n_wait == 6) return false;  // defensive: 4 input buffers + the TMEM region make at most 5 waits
        d.wait[d.n_wait++] = unit;
        return true;
      };
      for (int kb = 0; kb < d.nk; ++kb) {
        const int b = s.a_buf[kb / 2 < 4 ? kb / 2 : 3];  // k-blocks 2i, 2i+1 <- buffer a_buf[i]
        if (b < 0 || b >= n_buf || writer[b] < 0) return TB_ERR_BAD_SHAPE;  // reads a buffer nobody wrote
        d.a_off[kb] = b * BUF_BYTES + (kb & 1) * KB_BYTES;
        if (!add_wait(writer[b])) return TB_ERR_UNSUPPORTED;
      }
      d.tmem_col = (n_gemm % 4) * 128;
      if (n_gemm >= 4 && !add_wait(gemm_unit[n_gemm - 4])) return TB_ERR_UNSUPPORTED;  // accumulator region drained
      gemm_unit[n_gemm++] = u;
      total_boxes += d.nk;
    } else {
      return TB_ERR_BAD_SHAPE;
    }
    if (s.out_buf >= 0) writer[s.out_buf] = u;
  }
  hd->n_maps = n_maps; hd->total_boxes = total_boxes;
  return TB_OK;
}

extern "C" int tb_chain_run(const void* d_program, const void* host_blob, void* const* bindings, int n_bind, int M,
                            void* stream) {
  if (!d_program || !host_blob || !bindings) return TB_ERR_NULL;
  if (M <= 0 || n_bind < 0 || n_bind > TB_CHAIN_MAX_BIND - 1) return TB_ERR_BAD_SHAPE;
  if (reinterpret_cast<uintptr_t>(d_program) & 127) return TB_ERR_MISALIGNED;
  const Header* hd = static_cast<const Header*>(host_blob);
  if (hd->n_units <= 0 || hd->n_units > MAX_UNITS) return TB_ERR_BAD_SHAPE;
  const int err = check_bindings(reinterpret_cast<const UnitDev*>(static_cast<const uint8_t*>(host_blob) + 64),
                                 hd->n_units, bindings, n_bind);
  if (err != TB_OK) return err;
  Bind b;
  for (int i = 0; i < TB_CHAIN_MAX_BIND; ++i) b.p[i] = i < n_bind ? bindings[i] : nullptr;
  b.p[TB_CHAIN_MAX_BIND - 1] = tb_fp16_flag_ptr;  // fp16 range guard word (common.cuh)
  const size_t smem = 1024 + (size_t)hd->n_buf * BUF_BYTES + (size_t)hd->n_stage * WSTAGE_BYTES + tail_bytes(hd->n_units);
  static size_t attr_smem = 0;
  if (smem > attr_smem) {
    if (cudaFuncSetAttribute(mlp_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
      return TB_ERR_CUDA;
    attr_smem = smem;
  }
  static int num_sms = 0;
  if (num_sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || num_sms <= 0) num_sms = 148;
  }
  const int n_tiles = (M + TM - 1) / TM;
  const int grid = n_tiles < num_sms ? n_tiles : num_sms;
  mlp_chain_kernel<<<grid, NUM_THREADS, smem, static_cast<cudaStream_t>(stream)>>>(static_cast<const uint8_t*>(d_program), b, M);
  TB_CHECK_LAUNCH();
  return TB_OK;
}
