// Batched row copy of the rollout state (engine snapshot / restore / fork): many buffers in one launch, with an
// optional per-rollout row gather. Pure data movement; the item table travels in the kernel parameters.
#include "common.cuh"

namespace {

struct CopyItem {
  const unsigned char* src;
  unsigned char* dst;
  unsigned int upr;      // units per row
  int shift;             // log2 of the access width in bytes (0..4)
  int gather;            // route the rows through the rollout map
};

struct CopyTable {
  CopyItem item[TB_COPY_ROWS_MAX];
  long long end[TB_COPY_ROWS_MAX];  // exclusive prefix end of every item's units in the flattened index space
  int n_items;
};

constexpr int kThreads = 256;
constexpr int kUnroll = 4;

__device__ __forceinline__ uint4 load_unit(const unsigned char* p, int shift) {
  uint4 v = make_uint4(0u, 0u, 0u, 0u);
  switch (shift) {
    case 4: v = __ldg(reinterpret_cast<const uint4*>(p)); break;
    case 3: { uint2 t = __ldg(reinterpret_cast<const uint2*>(p)); v.x = t.x; v.y = t.y; } break;
    case 2: v.x = __ldg(reinterpret_cast<const unsigned int*>(p)); break;
    case 1: v.x = __ldg(reinterpret_cast<const unsigned short*>(p)); break;
    default: v.x = __ldg(p); break;
  }
  return v;
}

__device__ __forceinline__ void store_unit(unsigned char* p, int shift, uint4 v) {
  switch (shift) {
    case 4: *reinterpret_cast<uint4*>(p) = v; break;
    case 3: *reinterpret_cast<uint2*>(p) = make_uint2(v.x, v.y); break;
    case 2: *reinterpret_cast<unsigned int*>(p) = v.x; break;
    case 1: *reinterpret_cast<unsigned short*>(p) = static_cast<unsigned short>(v.x); break;
    default: *p = static_cast<unsigned char>(v.x); break;
  }
}

// Byte offset in src of unit u of item it. Gathered rows: row b = sc * R + r reads row sc * R + map[b]; an entry
// outside [0, R) reads the row itself.
__device__ __forceinline__ long long src_offset(const CopyItem& c, long long u, const int32_t* __restrict__ map, int R) {
  if (!c.gather) return u << c.shift;
  const unsigned int uu = static_cast<unsigned int>(u);  // gathered items hold < 2^32 units (host check)
  const unsigned int row = uu / c.upr, col = uu - row * c.upr;
  const int r = __ldg(map + row);
  const unsigned int srow = static_cast<unsigned int>(r) < static_cast<unsigned int>(R) ? row - row % R + r : row;
  return (static_cast<long long>(srow) * c.upr + col) << c.shift;
}

// Grid-stride loop over the units of all items, kUnroll units in flight per thread. A thread's indices only grow,
// so its item cursor only moves forward.
__global__ void __launch_bounds__(kThreads) copy_rows_kernel(const __grid_constant__ CopyTable tab,
                                                             const int32_t* __restrict__ map, int R) {
  const long long total = tab.end[tab.n_items - 1];
  const long long stride = static_cast<long long>(gridDim.x) * kThreads;
  int it = 0;
  for (long long base = static_cast<long long>(blockIdx.x) * kThreads + threadIdx.x; base < total;
       base += stride * kUnroll) {
    uint4 v[kUnroll];
    unsigned char* dst[kUnroll];
    int sh[kUnroll];
#pragma unroll
    for (int k = 0; k < kUnroll; ++k) {
      const long long i = base + k * stride;
      dst[k] = nullptr;
      if (i < total) {
        while (i >= tab.end[it]) ++it;
        const CopyItem& c = tab.item[it];
        const long long u = i - (it ? tab.end[it - 1] : 0);
        sh[k] = c.shift;
        v[k] = load_unit(c.src + src_offset(c, u, map, R), c.shift);
        dst[k] = c.dst + (u << c.shift);
      }
    }
#pragma unroll
    for (int k = 0; k < kUnroll; ++k)
      if (dst[k]) store_unit(dst[k], sh[k], v[k]);
  }
}

int num_sms() {
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
    return 148;
  return n;
}

}  // namespace

extern "C" int tb_copy_rows(const tb_row_copy_t* items, int n_items, const int32_t* src_rollout, int R, void* stream) {
  if (!items) return TB_ERR_NULL;
  if (n_items <= 0 || n_items > TB_COPY_ROWS_MAX) return TB_ERR_BAD_SHAPE;
  CopyTable tab;
  long long total = 0;
  for (int i = 0; i < n_items; ++i) {
    const tb_row_copy_t& x = items[i];
    if (!x.src || !x.dst) return TB_ERR_NULL;
    if (x.row_bytes <= 0 || x.n_rows <= 0) return TB_ERR_BAD_SHAPE;
    const bool gather = src_rollout && x.per_rollout;
    if (x.per_rollout && (R <= 0 || x.n_rows % R != 0)) return TB_ERR_BAD_SHAPE;
    if (gather && x.src == x.dst) return TB_ERR_UNSUPPORTED;  // rows would be read after being overwritten
    const uintptr_t a = reinterpret_cast<uintptr_t>(x.src) | reinterpret_cast<uintptr_t>(x.dst) |
                        static_cast<uintptr_t>(x.row_bytes);
    int shift = 4;
    while (shift > 0 && (a & ((uintptr_t(1) << shift) - 1))) --shift;
    const long long upr = x.row_bytes >> shift;
    if (upr > 0xFFFFFFFFll || (gather && upr * x.n_rows > 0xFFFFFFFFll)) return TB_ERR_UNSUPPORTED;
    CopyItem& c = tab.item[i];
    c.src = static_cast<const unsigned char*>(x.src);
    c.dst = static_cast<unsigned char*>(x.dst);
    c.upr = static_cast<unsigned int>(upr);
    c.shift = shift;
    c.gather = gather;
    total += upr * x.n_rows;
    tab.end[i] = total;
  }
  tab.n_items = n_items;
  const long long want = (total + kThreads * kUnroll - 1) / (kThreads * kUnroll);
  const int grid = static_cast<int>(want < 8ll * num_sms() ? want : 8ll * num_sms());
  copy_rows_kernel<<<grid, kThreads, 0, static_cast<cudaStream_t>(stream)>>>(tab, src_rollout, R);
  TB_CHECK_LAUNCH();
  return TB_OK;
}
