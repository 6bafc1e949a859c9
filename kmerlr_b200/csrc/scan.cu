// scan.cu -- exclusive prefix sums used for row pointers, column pointers and bitmap ranks.
// Three launches: per-tile sums, one block scanning the tile sums, per-tile scan + offset.
#include "common.cuh"

namespace kl {

namespace {

constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 8;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

template <typename TIn>
__global__ void scan_tile_sums(const TIn *__restrict__ in, int64_t n, int64_t *__restrict__ tile_sum) {
  __shared__ int64_t warp_part[SCAN_THREADS / 32];
  int64_t base = (int64_t)blockIdx.x * SCAN_TILE;
  int64_t s = 0;
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; i++) {
    int64_t j = base + (int64_t)i * SCAN_THREADS + threadIdx.x;
    if (j < n) s += (int64_t)in[j];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) warp_part[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    int64_t t = 0;
    for (int w = 0; w < SCAN_THREADS / 32; w++) t += warp_part[w];
    tile_sum[blockIdx.x] = t;
  }
}

// one block: exclusive scan of the tile sums in place; total written to tile_sum[nt]
__global__ void scan_tile_offsets(int64_t *tile_sum, int64_t nt) {
  __shared__ int64_t warp_part[32];
  __shared__ int64_t carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  for (int64_t base = 0; base < nt; base += blockDim.x) {
    int64_t j = base + threadIdx.x;
    int64_t v = j < nt ? tile_sum[j] : 0, x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int64_t y = __shfl_up_sync(0xffffffffu, x, o);
      if ((threadIdx.x & 31) >= o) x += y;
    }
    if ((threadIdx.x & 31) == 31) warp_part[threadIdx.x >> 5] = x;
    __syncthreads();
    if (threadIdx.x < 32) {
      int64_t w = threadIdx.x < (blockDim.x >> 5) ? warp_part[threadIdx.x] : 0, z = w;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        int64_t y = __shfl_up_sync(0xffffffffu, z, o);
        if (threadIdx.x >= o) z += y;
      }
      warp_part[threadIdx.x] = z - w;  // exclusive over warps
    }
    __syncthreads();
    int64_t excl = carry + warp_part[threadIdx.x >> 5] + x - v;
    if (j < nt) tile_sum[j] = excl;
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) carry = excl + v;
    __syncthreads();
  }
  if (threadIdx.x == 0) tile_sum[nt] = carry;
}

template <typename TIn, typename TOut>
__global__ void scan_tiles(const TIn *__restrict__ in, int64_t n, const int64_t *__restrict__ tile_off,
                           TOut *__restrict__ out, int64_t nt) {
  __shared__ int64_t warp_part[SCAN_THREADS / 32];
  // blocked arrangement: thread t owns items [t*ITEMS, (t+1)*ITEMS)
  int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
  int64_t v[SCAN_ITEMS], s = 0;
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; i++) {
    int64_t j = base + i;
    v[i] = j < n ? (int64_t)in[j] : 0;
    s += v[i];
  }
  int64_t x = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int64_t y = __shfl_up_sync(0xffffffffu, x, o);
    if ((threadIdx.x & 31) >= o) x += y;
  }
  if ((threadIdx.x & 31) == 31) warp_part[threadIdx.x >> 5] = x;
  __syncthreads();
  int64_t woff = 0;
  for (int w = 0; w < (int)(threadIdx.x >> 5); w++) woff += warp_part[w];
  int64_t run = tile_off[blockIdx.x] + woff + x - s;
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; i++) {
    int64_t j = base + i;
    if (j < n) out[j] = (TOut)run;
    run += v[i];
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) out[n] = (TOut)tile_off[nt];
}

int64_t tile_count(int64_t n) {
  const int64_t nt = (n + SCAN_TILE - 1) / SCAN_TILE;
  return nt == 0 ? 1 : nt;
}

template <typename TIn, typename TOut>
void scan_launch(const TIn *in, TOut *out, int64_t n, int64_t *tiles) {
  const int64_t nt = tile_count(n);
  KL_LAUNCH((scan_tile_sums<TIn>), (unsigned)nt, SCAN_THREADS, 0, in, n, tiles);
  KL_LAUNCH(scan_tile_offsets, 1, 1024, 0, tiles, nt);
  KL_LAUNCH((scan_tiles<TIn, TOut>), (unsigned)nt, SCAN_THREADS, 0, in, n, tiles, out, nt);
}

template <typename TIn, typename TOut>
void scan_impl(const TIn *in, TOut *out, int64_t n) {
  DevBuf<int64_t> tiles((size_t)tile_count(n) + 1);
  scan_launch(in, out, n, tiles.p);
  sync_stream();  // tiles is freed on return
}

}  // namespace

int64_t exclusive_scan_workspace(int64_t n) { return tile_count(n) + 1; }
void exclusive_scan_u32_async(const uint32_t *in, uint32_t *out, int64_t n, int64_t *workspace) {
  scan_launch<uint32_t, uint32_t>(in, out, n, workspace);
}

void exclusive_scan_i64(const int64_t *in, int64_t *out, int64_t n) { scan_impl<int64_t, int64_t>(in, out, n); }
void exclusive_scan_u32_to_i64(const uint32_t *in, int64_t *out, int64_t n) { scan_impl<uint32_t, int64_t>(in, out, n); }
void exclusive_scan_u32(const uint32_t *in, uint32_t *out, int64_t n) { scan_impl<uint32_t, uint32_t>(in, out, n); }

}  // namespace kl
