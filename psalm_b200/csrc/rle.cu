// COCO run-length encoding of binary masks on the device (pycocotools maskApi.c rleEncode + rleToString).
//
// Replaces `pycocotools.mask.encode` on the instance / region results: detectron2's instances_to_coco_json (behind
// COCOEvaluator.process, psalm/eval/instance_segmentation.py:128,150) and psalm/eval/region_segmentation.py:282-283
// both copy the dense fp32 [K, H, W] masks to the host first.  Here only the RLE strings leave the device.
//
// Three phases, each a few launches; the caller sizes the exact output buffers between them (two small reads):
//   sizes  pack:     row-major [K, H, W] -> column-major bit words bits[k][w][x] (bit j = pixel (32w + j, x)): one warp per
//                    32 x 32 tile, coalesced row loads, one ballot per row, then a 32 x 32 bit transpose by 32 ballots
//          count:    per column, the transitions (pixel != its column-major predecessor; the predecessor of (0, x) is
//                    (H-1, x-1), that of (0, 0) an implicit 0) and the last transition's linear position
//          colscan:  per mask, exclusive scans over the columns: first run index and previous transition position of
//                    every column; runs of mask k = transitions + 1
//          offsets:  scan over the masks -> run_offsets [K + 1]
//   runs   runs:     per column, run lengths = distance between consecutive transitions (written in place, in order)
//          chars:    per mask, the length of its counts string -> offsets -> str_offsets [K + 1]
//   write  write:    per mask, block scan of the per-run character counts and the 5-bit groups of rleToString
#include <cub/block/block_reduce.cuh>
#include <cub/block/block_scan.cuh>

#include "common.cuh"

namespace psalm {
namespace {

constexpr int kBlock = 256;

struct MaxOp {
  __device__ __forceinline__ uint32_t operator()(uint32_t a, uint32_t b) const { return a > b ? a : b; }
};

// foreground = value != 0 on the raw bits (+0 and -0 are background); U is the unsigned type of the element's width
template <typename U, uint32_t kMag>
// (2 blocks per SM: <= 128 registers with the 32 loads of a lane in flight, no spills)
__global__ void __launch_bounds__(kBlock, 2) rle_pack_kernel(const U* __restrict__ masks, uint32_t* __restrict__ bits,
                                                             int K, int H, int W, int NW) {
  const int lane = threadIdx.x & 31;
  const int w = blockIdx.y * (kBlock / 32) + (threadIdx.x >> 5);   // word row: pixel rows 32w .. 32w + 31
  if (w >= NW) return;                                              // uniform per warp
  const int x = blockIdx.x * 32 + lane;
  const int y0 = w * 32;
  const bool interior = (int)(blockIdx.x + 1) * 32 <= W && y0 + 32 <= H;   // no bounds tests: 32 loads in flight
  for (int k = blockIdx.z; k < K; k += gridDim.z) {
    const U* m = masks + (size_t)k * H * W + (size_t)y0 * W + x;
    bool v[32];
    if (interior) {
#pragma unroll
      for (int r = 0; r < 32; ++r) v[r] = (((uint32_t)__ldg(m + (size_t)r * W)) & kMag) != 0;
    } else {
#pragma unroll
      for (int r = 0; r < 32; ++r) v[r] = x < W && y0 + r < H && (((uint32_t)__ldg(m + (size_t)r * W)) & kMag) != 0;
    }
    uint32_t row = 0;   // lane r: pixel row y0 + r over the tile's 32 columns (bit c = column x0 + c)
#pragma unroll
    for (int r = 0; r < 32; ++r) {
      const uint32_t b = __ballot_sync(0xffffffffu, v[r]);
      if (lane == r) row = b;
    }
    uint32_t col = 0;   // lane c: column x0 + c over the tile's 32 rows (bit r = row y0 + r)
#pragma unroll
    for (int c = 0; c < 32; ++c) {
      const uint32_t b = __ballot_sync(0xffffffffu, (row >> c) & 1u);
      if (lane == c) col = b;
    }
    if (x < W) bits[((size_t)k * NW + w) * W + x] = col;
  }
}

// transitions of word w of a column: bit j set when pixel 32w + j differs from its predecessor
__device__ __forceinline__ uint32_t transitions(uint32_t word, uint32_t& carry, int w, int NW, uint32_t tail) {
  uint32_t t = word ^ ((word << 1) | carry);
  carry = word >> 31;
  return w == NW - 1 ? t & tail : t;
}

__device__ __forceinline__ uint32_t carry_into_column(const uint32_t* col_bits, int x, int H, int W, int NW) {
  return x > 0 ? (col_bits[(size_t)(NW - 1) * W - 1] >> ((H - 1) & 31)) & 1u : 0u;   // pixel (H-1, x-1)
}

__global__ void __launch_bounds__(kBlock) rle_count_kernel(const uint32_t* __restrict__ bits, uint32_t* __restrict__ ncol,
                                                           uint32_t* __restrict__ lastp, int K, int H, int W, int NW) {
  const long long i = (long long)blockIdx.x * kBlock + threadIdx.x;
  if (i >= (long long)K * W) return;
  const int k = (int)(i / W), x = (int)(i % W);
  const uint32_t* b = bits + (size_t)k * NW * W + x;
  const uint32_t tail = (H & 31) ? (1u << (H & 31)) - 1u : 0xffffffffu;
  uint32_t carry = carry_into_column(b, x, H, W, NW);
  uint32_t n = 0, last = 0;
  for (int w = 0; w < NW; ++w) {
    const uint32_t t = transitions(b[(size_t)w * W], carry, w, NW, tail);
    if (t) {
      n += __popc(t);
      last = (uint32_t)x * H + 32u * w + 31u - __clz(t);
    }
  }
  ncol[i] = n;
  lastp[i] = last;
}

// one block per mask: ncol -> index of the column's first transition in the mask, lastp -> position of the last transition
// before the column (0 when none: the first run then starts at 0, as it does after a transition at pixel 0)
__global__ void __launch_bounds__(kBlock) rle_colscan_kernel(uint32_t* __restrict__ ncol, uint32_t* __restrict__ lastp,
                                                             long long* __restrict__ run_offsets, int K, int W) {
  using Scan = cub::BlockScan<uint32_t, kBlock>;
  __shared__ typename Scan::TempStorage tmp;
  for (int k = blockIdx.x; k < K; k += gridDim.x) {
    uint32_t carry_n = 0, carry_p = 0;
    for (int x0 = 0; x0 < W; x0 += kBlock) {
      const int x = x0 + threadIdx.x;
      const size_t i = (size_t)k * W + x;
      const uint32_t n = x < W ? ncol[i] : 0u, p = x < W ? lastp[i] : 0u;
      uint32_t on, op, tn, tp;
      Scan(tmp).ExclusiveSum(n, on, tn);
      __syncthreads();
      Scan(tmp).ExclusiveScan(p, op, 0u, MaxOp(), tp);
      __syncthreads();
      if (x < W) {
        ncol[i] = carry_n + on;
        lastp[i] = max(carry_p, op);
      }
      carry_n += tn;
      carry_p = max(carry_p, tp);
    }
    if (threadIdx.x == 0) run_offsets[k + 1] = (long long)carry_n + 1;
  }
}

// off[1..K] per-mask sizes -> inclusive prefix sums; off[0] = 0 (one block)
__global__ void __launch_bounds__(kBlock) rle_offsets_kernel(long long* __restrict__ off, int K) {
  using Scan = cub::BlockScan<long long, kBlock>;
  __shared__ typename Scan::TempStorage tmp;
  long long carry = 0;
  for (int i0 = 0; i0 < K; i0 += kBlock) {
    const int i = i0 + threadIdx.x;
    long long v = i < K ? off[i + 1] : 0, o, agg;
    Scan(tmp).InclusiveSum(v, o, agg);
    __syncthreads();
    if (i < K) off[i + 1] = carry + o;
    carry += agg;
  }
  if (threadIdx.x == 0) off[0] = 0;
}

__global__ void __launch_bounds__(kBlock) rle_runs_kernel(const uint32_t* __restrict__ bits, const uint32_t* __restrict__ first,
                                                          const uint32_t* __restrict__ prevp,
                                                          const long long* __restrict__ run_offsets,
                                                          uint32_t* __restrict__ counts, int K, int H, int W, int NW) {
  const long long i = (long long)blockIdx.x * kBlock + threadIdx.x;
  if (i >= (long long)K * W) return;
  const int k = (int)(i / W), x = (int)(i % W);
  const uint32_t* b = bits + (size_t)k * NW * W + x;
  const uint32_t tail = (H & 31) ? (1u << (H & 31)) - 1u : 0xffffffffu;
  uint32_t carry = carry_into_column(b, x, H, W, NW);
  uint32_t* out = counts + run_offsets[k] + first[i];
  uint32_t prev = prevp[i];
  for (int w = 0; w < NW; ++w) {
    uint32_t t = transitions(b[(size_t)w * W], carry, w, NW, tail);
    while (t) {
      const uint32_t p = (uint32_t)x * H + 32u * w + (uint32_t)(__ffs(t) - 1);
      t &= t - 1;
      *out++ = p - prev;
      prev = p;
    }
  }
  if (x == W - 1) *out = (uint32_t)H * W - prev;   // the last run ends at the last pixel
}

// rleToString: x = cnts[i] (- cnts[i-2] for i > 2), 5-bit groups least significant first, 0x20 = more groups follow
__device__ __forceinline__ long long rle_delta(const uint32_t* c, long long i) {
  return i > 2 ? (long long)c[i] - (long long)c[i - 2] : (long long)c[i];
}

__device__ __forceinline__ int rle_chars(long long x) {
  int n = 1;
  for (;;) {
    const int c = (int)(x & 0x1f);
    x >>= 5;   // arithmetic
    if (!((c & 0x10) ? x != -1 : x != 0)) return n;
    ++n;
  }
}

__global__ void __launch_bounds__(kBlock) rle_chars_kernel(const uint32_t* __restrict__ counts,
                                                           const long long* __restrict__ run_offsets,
                                                           long long* __restrict__ str_offsets, int K) {
  using Reduce = cub::BlockReduce<long long, kBlock>;
  __shared__ typename Reduce::TempStorage tmp;
  for (int k = blockIdx.x; k < K; k += gridDim.x) {
    const uint32_t* c = counts + run_offsets[k];
    const long long m = run_offsets[k + 1] - run_offsets[k];
    long long n = 0;
    for (long long i = threadIdx.x; i < m; i += kBlock) n += rle_chars(rle_delta(c, i));
    const long long total = Reduce(tmp).Sum(n);
    if (threadIdx.x == 0) str_offsets[k + 1] = total;
    __syncthreads();
  }
}

__global__ void __launch_bounds__(kBlock) rle_write_kernel(const uint32_t* __restrict__ counts,
                                                           const long long* __restrict__ run_offsets,
                                                           const long long* __restrict__ str_offsets,
                                                           char* __restrict__ strings, int K) {
  using Scan = cub::BlockScan<long long, kBlock>;
  __shared__ typename Scan::TempStorage tmp;
  for (int k = blockIdx.x; k < K; k += gridDim.x) {
    const uint32_t* c = counts + run_offsets[k];
    const long long m = run_offsets[k + 1] - run_offsets[k];
    char* s = strings + str_offsets[k];
    for (long long i0 = 0; i0 < m; i0 += kBlock) {
      const long long i = i0 + threadIdx.x;
      long long x = i < m ? rle_delta(c, i) : 0;
      long long n = i < m ? rle_chars(x) : 0, o, agg;
      Scan(tmp).ExclusiveSum(n, o, agg);
      __syncthreads();
      for (long long j = 0; j < n; ++j) {
        int ch = (int)(x & 0x1f);
        x >>= 5;
        if (j + 1 < n) ch |= 0x20;
        s[o + j] = (char)(ch + 48);
      }
      s += agg;
    }
  }
}

int grid_of(long long threads) { return (int)((threads + kBlock - 1) / kBlock); }

struct Workspace {
  uint32_t *bits, *ncol, *lastp;
  static size_t align(size_t b) { return (b + 255) & ~(size_t)255; }
  static size_t bytes(int K, int H, int W) {
    const size_t NW = (size_t)(H + 31) / 32;
    return align((size_t)K * NW * W * 4) + 2 * align((size_t)K * W * 4);
  }
  Workspace(void* ws, int K, int H, int W) {
    const size_t NW = (size_t)(H + 31) / 32;
    char* p = (char*)ws;
    bits = (uint32_t*)p;
    p += align((size_t)K * NW * W * 4);
    ncol = (uint32_t*)p;
    p += align((size_t)K * W * 4);
    lastp = (uint32_t*)p;
  }
};

int check_shape(int K, int H, int W) {
  PSALM_REQUIRE(K > 0 && H > 0 && W > 0, "mask_rle: bad shape K=%d H=%d W=%d", K, H, W);
  PSALM_REQUIRE((long long)H * W < (1ll << 31), "mask_rle: H*W=%lld pixels per mask exceeds 2^31 - 1",
                (long long)H * W);
  return PSALM_OK;
}

}  // namespace
}  // namespace psalm

extern "C" size_t psalm_mask_rle_workspace_bytes(int K, int H, int W) {
  if (K <= 0 || H <= 0 || W <= 0) return 0;
  return psalm::Workspace::bytes(K, H, W);
}

extern "C" int psalm_mask_rle_sizes(const void* masks, void* workspace, size_t workspace_bytes, int64_t* run_offsets, int K,
                                    int H, int W, int dtype, void* stream) {
  using namespace psalm;
  PSALM_REQUIRE(masks && workspace && run_offsets, "mask_rle_sizes: null pointer");
  if (int rc = check_shape(K, H, W)) return rc;
  PSALM_REQUIRE(workspace_bytes >= Workspace::bytes(K, H, W), "mask_rle_sizes: workspace of %zu bytes, %zu needed",
                workspace_bytes, Workspace::bytes(K, H, W));
  cudaStream_t st = (cudaStream_t)stream;
  Workspace ws(workspace, K, H, W);
  const int NW = (H + 31) / 32;
  const dim3 grid((W + 31) / 32, (NW + kBlock / 32 - 1) / (kBlock / 32), K < 65535 ? K : 65535);
  switch (dtype) {
    case PSALM_F32:
      rle_pack_kernel<uint32_t, 0x7fffffffu><<<grid, kBlock, 0, st>>>((const uint32_t*)masks, ws.bits, K, H, W, NW);
      break;
    case PSALM_F16:
    case PSALM_BF16:
      rle_pack_kernel<unsigned short, 0x7fffu><<<grid, kBlock, 0, st>>>((const unsigned short*)masks, ws.bits, K, H, W, NW);
      break;
    case PSALM_U8:
      rle_pack_kernel<unsigned char, 0xffu><<<grid, kBlock, 0, st>>>((const unsigned char*)masks, ws.bits, K, H, W, NW);
      break;
    default:
      set_error("mask_rle_sizes: unknown dtype %d", dtype);
      return PSALM_E_ARG;
  }
  if (int rc = check_launch("rle_pack_kernel")) return rc;
  rle_count_kernel<<<grid_of((long long)K * W), kBlock, 0, st>>>(ws.bits, ws.ncol, ws.lastp, K, H, W, NW);
  if (int rc = check_launch("rle_count_kernel")) return rc;
  rle_colscan_kernel<<<K, kBlock, 0, st>>>(ws.ncol, ws.lastp, (long long*)run_offsets, K, W);
  if (int rc = check_launch("rle_colscan_kernel")) return rc;
  rle_offsets_kernel<<<1, kBlock, 0, st>>>((long long*)run_offsets, K);
  return check_launch("rle_offsets_kernel");
}

extern "C" int psalm_mask_rle_runs(const void* workspace, size_t workspace_bytes, const int64_t* run_offsets, uint32_t* counts,
                                   int64_t* str_offsets, int K, int H, int W, void* stream) {
  using namespace psalm;
  PSALM_REQUIRE(workspace && run_offsets && counts && str_offsets, "mask_rle_runs: null pointer");
  if (int rc = check_shape(K, H, W)) return rc;
  PSALM_REQUIRE(workspace_bytes >= Workspace::bytes(K, H, W), "mask_rle_runs: workspace of %zu bytes, %zu needed",
                workspace_bytes, Workspace::bytes(K, H, W));
  cudaStream_t st = (cudaStream_t)stream;
  Workspace ws(const_cast<void*>(workspace), K, H, W);
  const int NW = (H + 31) / 32;
  rle_runs_kernel<<<grid_of((long long)K * W), kBlock, 0, st>>>(ws.bits, ws.ncol, ws.lastp, (const long long*)run_offsets,
                                                                 counts, K, H, W, NW);
  if (int rc = check_launch("rle_runs_kernel")) return rc;
  rle_chars_kernel<<<K, kBlock, 0, st>>>(counts, (const long long*)run_offsets, (long long*)str_offsets, K);
  if (int rc = check_launch("rle_chars_kernel")) return rc;
  rle_offsets_kernel<<<1, kBlock, 0, st>>>((long long*)str_offsets, K);
  return check_launch("rle_offsets_kernel");
}

extern "C" int psalm_mask_rle_write(const uint32_t* counts, const int64_t* run_offsets, const int64_t* str_offsets,
                                    char* strings, int K, void* stream) {
  using namespace psalm;
  PSALM_REQUIRE(counts && run_offsets && str_offsets && strings, "mask_rle_write: null pointer");
  PSALM_REQUIRE(K > 0, "mask_rle_write: bad K=%d", K);
  rle_write_kernel<<<K, kBlock, 0, (cudaStream_t)stream>>>(counts, (const long long*)run_offsets,
                                                           (const long long*)str_offsets, strings, K);
  return check_launch("rle_write_kernel");
}
