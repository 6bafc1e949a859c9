// matrix.cu -- KmerDataSet in HBM: CSR import/export, labels, the stable CSR -> CSC transpose that
// makes X^T w deterministic, featureSelection.Data (reduced matrix) and the step-size row norm.
#include "common.cuh"

#include <cmath>

namespace kl {

namespace {

// ---- stable transpose: LSD radix sort of the entries by column ---------------------------------------
// The CSC view must list the entries of a column in ascending row order (the order the reference
// accumulates a gradient entry in, kmerLr_logistic_regression.go:166-181) and must not depend on
// scheduling.  Entries start in row order (CSR), so a STABLE sort by column gives exactly that:
// 8-bit digits, least significant first; every pass = per-tile digit histogram, one scan, and a
// scatter whose local ranks come from warp match (no atomics in the ranking, fully deterministic).
constexpr int RS_THREADS = 256;
constexpr int RS_GROUPS = 32;                       // 32 consecutive entries per lane-group
constexpr int RS_WARP_ITEMS = 32 * RS_GROUPS;       // 1024 consecutive entries per warp
constexpr int RS_TILE = (RS_THREADS / 32) * RS_WARP_ITEMS;   // 8192 entries per CTA

__global__ void __launch_bounds__(RS_THREADS) radix_hist(const uint32_t *__restrict__ keys, int64_t nnz, int shift,
                                                         uint32_t *__restrict__ hist, int64_t ntiles) {
  __shared__ uint32_t h[256];
  h[threadIdx.x] = 0;
  __syncthreads();
  int64_t base = (int64_t)blockIdx.x * RS_TILE;
#pragma unroll 8
  for (int i = 0; i < RS_TILE / RS_THREADS; i++) {
    int64_t p = base + (int64_t)i * RS_THREADS + threadIdx.x;
    if (p < nnz) atomicAdd(&h[(keys[p] >> shift) & 255u], 1u);
  }
  __syncthreads();
  hist[(int64_t)threadIdx.x * ntiles + blockIdx.x] = h[threadIdx.x];   // digit-major: one flat scan gives offsets
}

template <typename VT, bool FIRST>
__global__ void __launch_bounds__(RS_THREADS) radix_scatter(const uint32_t *__restrict__ keys,
                                                            const uint32_t *__restrict__ rows_in,
                                                            const int64_t *__restrict__ rowptr, int64_t nrows,
                                                            const VT *__restrict__ vals, int64_t nnz, int shift,
                                                            const int64_t *__restrict__ offs, int64_t ntiles,
                                                            uint32_t *__restrict__ keys_out,
                                                            uint32_t *__restrict__ rows_out,
                                                            VT *__restrict__ vals_out) {
  // dynamic smem: the tile in sorted order (keys, rows, values), written out as coalesced runs
  extern __shared__ __align__(16) unsigned char rs_smem[];
  uint32_t *skey = (uint32_t *)rs_smem;
  uint32_t *srow = skey + RS_TILE;
  VT *sval = (VT *)(srow + RS_TILE);
  __shared__ uint32_t wcnt[RS_THREADS / 32][256];
  __shared__ uint32_t tdig[257];
  __shared__ int64_t goff[256];
  const unsigned lane = lane_id(), w = threadIdx.x >> 5;
  const int64_t tbase = (int64_t)blockIdx.x * RS_TILE;
  const int64_t wbase = tbase + (int64_t)w * RS_WARP_ITEMS;
  for (int i = lane; i < 256; i += 32) wcnt[w][i] = 0;
  __syncwarp();
  // sub-pass 1: rank of every entry among the earlier entries of its warp with the same digit
  uint32_t lr[RS_GROUPS];
#pragma unroll
  for (int g = 0; g < RS_GROUPS; g++) {
    int64_t p = wbase + g * 32 + lane;
    bool valid = p < nnz;
    uint32_t d = valid ? ((keys[p] >> shift) & 255u) : 0u;
    // lanes holding the same digit: 8 ballots (match.any serialises over the distinct values)
    unsigned mask = __ballot_sync(0xffffffffu, valid);
#pragma unroll
    for (int b = 0; b < 8; b++) {
      unsigned bal = __ballot_sync(0xffffffffu, (d >> b) & 1u);
      mask &= ((d >> b) & 1u) ? bal : ~bal;
    }
    uint32_t old = valid ? wcnt[w][d] : 0u;
    __syncwarp();
    if (valid && (unsigned)(__ffs(mask) - 1) == lane) wcnt[w][d] = old + __popc(mask);
    __syncwarp();
    lr[g] = old + __popc(mask & lanemask_lt());
  }
  __syncthreads();
  // bases: digit = threadIdx.x; earlier warps of the tile come first
  {
    uint32_t run = 0;
#pragma unroll
    for (int ww = 0; ww < RS_THREADS / 32; ww++) {
      uint32_t c = wcnt[ww][threadIdx.x];
      wcnt[ww][threadIdx.x] = run;
      run += c;
    }
    // exclusive scan of the tile's digit counts (256 threads = 256 digits)
    uint32_t x = run;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= (unsigned)o) x += y;
    }
    __shared__ uint32_t wtot[RS_THREADS / 32];
    if (lane == 31) wtot[w] = x;
    __syncthreads();
    uint32_t before = 0;
    for (unsigned ww = 0; ww < w; ww++) before += wtot[ww];
    tdig[threadIdx.x] = before + x - run;
    if (threadIdx.x == 255) tdig[256] = before + x;
    goff[threadIdx.x] = offs[(int64_t)threadIdx.x * ntiles + blockIdx.x];
  }
  __syncthreads();
  // row of the warp's first entry (first pass: rows are implicit in the CSR row pointers)
  int64_t rcur = 0;
  if (FIRST) {
    if (wbase < nnz) {
      int64_t lo = 0, hi = nrows;   // last row with rowptr[row] <= wbase
      while (hi - lo > 1) { int64_t mid = (lo + hi) >> 1; if (rowptr[mid] <= wbase) lo = mid; else hi = mid; }
      rcur = lo;
    }
  }
  // sub-pass 2: place every entry at its sorted position inside the tile
#pragma unroll
  for (int g = 0; g < RS_GROUPS; g++) {
    int64_t p = wbase + g * 32 + lane;
    bool valid = p < nnz;
    uint32_t row = 0;
    if (FIRST) {
      int64_t r = rcur;
      if (valid) while (rowptr[r + 1] <= p) r++;
      row = (uint32_t)r;
      rcur = __shfl_sync(0xffffffffu, r, 0);
    }
    if (valid) {
      uint32_t key = keys[p], d = (key >> shift) & 255u;
      uint32_t slot = tdig[d] + wcnt[w][d] + lr[g];
      skey[slot] = key;
      srow[slot] = FIRST ? row : rows_in[p];
      if (vals) sval[slot] = vals[p];
    }
  }
  __syncthreads();
  // write out: consecutive threads -> consecutive slots -> consecutive addresses inside a digit run
  const uint32_t tile_n = tdig[256];
  for (uint32_t i = threadIdx.x; i < tile_n; i += RS_THREADS) {
    uint32_t key = skey[i], d = (key >> shift) & 255u;
    int64_t dst = goff[d] + (i - tdig[d]);
    keys_out[dst] = key;
    rows_out[dst] = srow[i];
    if (vals) vals_out[dst] = sval[i];
  }
}

// colptr[c] = first position of a key >= c in the sorted key array
__global__ void lower_bounds(const uint32_t *__restrict__ sorted, int64_t nnz, int64_t m, int64_t *__restrict__ colptr) {
  int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c > m) return;
  int64_t lo = 0, hi = nnz;
  while (lo < hi) { int64_t mid = (lo + hi) >> 1; if ((int64_t)sorted[mid] < c) lo = mid + 1; else hi = mid; }
  colptr[c] = lo;
}

// ---- featureSelection.Data (kmerLr_feature_selection.go:309-343) ----------------------------------
template <typename VT>
__device__ __forceinline__ double row_value(const uint32_t *col, const VT *val, int64_t a, int64_t b, uint32_t c) {
  int64_t lo = a, hi = b;
  while (lo < hi) {
    int64_t mid = (lo + hi) >> 1;
    if (col[mid] < c) lo = mid + 1; else hi = mid;
  }
  if (lo < b && col[lo] == c) return val ? (double)val[lo] : 1.0;
  return 0.0;
}

template <typename VT, bool WRITE>
__global__ void reduce_rows(const Rows R, const uint32_t *__restrict__ col,
                            const VT *__restrict__ val, int64_t n, const int64_t *__restrict__ selA,
                            const int64_t *__restrict__ selB, int64_t nsel, uint32_t *__restrict__ cnt_out,
                            const int64_t *__restrict__ orowptr, uint32_t *__restrict__ ocol,
                            double *__restrict__ oval) {
  int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= n) return;
  unsigned lane = lane_id();
  int64_t a, b;
  R.range(row, a, b);
  int64_t outp = WRITE ? orowptr[row] : 0;
  uint32_t tot = 0;
  for (int64_t j0 = 0; j0 < nsel; j0 += 32) {
    int64_t j = j0 + lane;
    double v = 0.0;
    if (j < nsel) {
      v = row_value(col, val, a, b, (uint32_t)selA[j]);
      if (selB[j] >= 0 && v != 0.0) v = v * row_value(col, val, a, b, (uint32_t)selB[j]);
    }
    unsigned km = __ballot_sync(0xffffffffu, v != 0.0);
    if (WRITE && v != 0.0) {
      int64_t pos = outp + __popc(km & lanemask_lt());
      ocol[pos] = (uint32_t)j;
      oval[pos] = v;
    }
    outp += __popc(km);
    tot += __popc(km);
  }
  if (!WRITE && lane == 0) cnt_out[row] = tot;
}

template <typename VT>
__global__ void row_sqnorm_max(const Rows R, const VT *__restrict__ val, int64_t n,
                               unsigned long long *__restrict__ out) {
  int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= n) return;
  unsigned lane = lane_id();
  double s = 0.0;
  int64_t a, b;
  R.range(row, a, b);
  if (val) {
    for (int64_t p = a + lane; p < b; p += 32) { double v = (double)val[p]; s += v * v; }
    s = warp_sum(s);
  } else {
    s = (double)(b - a);
  }
  // non-negative doubles compare like their bit patterns
  if (lane == 0) atomicMax(out, (unsigned long long)__double_as_longlong(s));
}

// max_i ||x~_i||^2 of the pair-expanded rows x~ = (v_j)_j u (v_a v_b)_{a<b}: ||x~||^2 = S2 + (S2^2 - S4) / 2 with
// S2 = sum v^2 and S4 = sum v^4 over the row, one warp per row.  Integer values (u32 counts, binarized rows) whose S2 is
// below 2^32 take exact 64-bit integer sums (then S2^2 < 2^64), rounded to a double once: the bits of the explicit
// expansion's row_sqnorm_max whenever its sums are exact (below 2^53).  Real values, and larger integer rows, in fp64
// (S2^2 is rounded before the subtraction, so that a row of one entry gives S2 exactly).
template <typename VT>
__global__ void row_sqnorm_pairs_max(const Rows R, const VT *__restrict__ val, int64_t n, unsigned long long *__restrict__ out) {
  int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= n) return;
  unsigned lane = lane_id();
  int64_t a, b;
  R.range(row, a, b);
  constexpr bool INT = std::is_same<VT, uint32_t>::value;
  double d2 = 0.0, d4 = 0.0;
  unsigned long long i2 = 0ull, i4 = 0ull;
  for (int64_t p = a + lane; p < b; p += 32) {
    const double v = val ? (double)val[p] : 1.0, v2 = v * v;
    d2 += v2; d4 += v2 * v2;
    if (INT) { const unsigned long long u = val ? (unsigned long long)val[p] : 1ull, u2 = u * u; i2 += u2; i4 += u2 * u2; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    d2 += __shfl_xor_sync(0xffffffffu, d2, o); d4 += __shfl_xor_sync(0xffffffffu, d4, o);
    i2 += __shfl_xor_sync(0xffffffffu, i2, o); i4 += __shfl_xor_sync(0xffffffffu, i4, o);
  }
  if (lane != 0) return;
  double s;
  if (INT && d2 < 4294967296.0) s = (double)(i2 + (i2 * i2 - i4) / 2ull);   // (v < 2^16 everywhere: no product wraps)
  else s = d2 + 0.5 * (__dmul_rn(d2, d2) - d4);
  atomicMax(out, (unsigned long long)__double_as_longlong(s));
}

template <typename VT>
__global__ void abs_max(const VT *__restrict__ val, int64_t nnz, unsigned long long *__restrict__ out) {
  double mx = 0.0;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < nnz; p += (int64_t)gridDim.x * blockDim.x)
    mx = fmax(mx, fabs((double)val[p]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if (lane_id() == 0 && mx > 0.0) atomicMax(out, (unsigned long long)__double_as_longlong(mx));
}

// per column: sum of the values, sum of their squares, largest |value|, number of stored entries
// (TransformFull.Fit, kmerLr_transform.go:59-252).  Counts are integers: exact 64-bit sums in any order.
template <typename VT>
__global__ void column_moments(const Rows R, const uint32_t *__restrict__ col, const VT *__restrict__ val, int64_t n,
                               unsigned long long *__restrict__ s1, unsigned long long *__restrict__ s2,
                               unsigned long long *__restrict__ mx, unsigned long long *__restrict__ cnt) {
  int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= n) return;
  int64_t a, b;
  R.range(row, a, b);
  for (int64_t p = a + lane_id(); p < b; p += 32) {
    const unsigned long long v = val ? (unsigned long long)val[p] : 1ull;
    const uint32_t c = col[p];
    atomicAdd(s1 + c, v);
    atomicAdd(s2 + c, v * v);
    atomicMax(mx + c, v);
    atomicAdd(cnt + c, 1ull);
  }
}

// the same four moments for the pair features v_a v_b, a < b (TransformFull.Fit with cooccurrence,
// kmerLr_transform.go:90-99,118-127): one warp per pair intersects the two CSC columns; integer values, exact
// sums.  Output position = CoeffIndex(m).Ind2Sub(a, b) - (m + 1).
template <typename VT>
__global__ void pair_moments(const int64_t *__restrict__ colptr, const uint32_t *__restrict__ crow,
                             const VT *__restrict__ cval, int64_t m, unsigned long long *__restrict__ s1,
                             unsigned long long *__restrict__ s2, unsigned long long *__restrict__ mx,
                             unsigned long long *__restrict__ cnt) {
  const int64_t npairs = m * (m - 1) / 2, warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const unsigned lane = lane_id();
  for (int64_t pi = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; pi < npairs; pi += warps) {
    // pair index -> (a, b), a < b, row-major over the strict upper triangle (= CoeffIndex order)
    int64_t a = (int64_t)floor(((double)(2 * m - 1) - sqrt((double)(2 * m - 1) * (double)(2 * m - 1) - 8.0 * (double)pi)) / 2.0);
    while (a > 0 && a * (2 * m - a - 1) / 2 > pi) a--;
    while ((a + 1) * (2 * m - a - 2) / 2 <= pi) a++;
    const int64_t b = pi - a * (2 * m - a - 1) / 2 + a + 1;
    const int64_t a0 = colptr[a], a1 = colptr[a + 1], b0 = colptr[b], b1 = colptr[b + 1];
    const bool swap = (a1 - a0) > (b1 - b0);
    const int64_t q0 = swap ? b0 : a0, q1 = swap ? b1 : a1, l0 = swap ? a0 : b0, l1 = swap ? a1 : b1;
    unsigned long long t1 = 0, t2 = 0, tm = 0, tc = 0;
    for (int64_t p = q0 + lane; p < q1; p += 32) {
      const uint32_t r = crow[p];
      int64_t lo = l0, hi = l1;
      while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (crow[mid] < r) lo = mid + 1; else hi = mid; }
      if (lo < l1 && crow[lo] == r) {
        const unsigned long long v = (cval ? (unsigned long long)cval[p] : 1ull) * (cval ? (unsigned long long)cval[lo] : 1ull);
        t1 += v; t2 += v * v; tm = v > tm ? v : tm; tc += 1;
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      t1 += __shfl_xor_sync(0xffffffffu, t1, o); t2 += __shfl_xor_sync(0xffffffffu, t2, o);
      tc += __shfl_xor_sync(0xffffffffu, tc, o);
      const unsigned long long y = __shfl_xor_sync(0xffffffffu, tm, o);
      tm = y > tm ? y : tm;
    }
    if (lane == 0) { s1[pi] = t1; s2[pi] = t2; mx[pi] = tm; cnt[pi] = tc; }
  }
}

// Transform.Apply (kmerLr_transform.go:584-629) on the rows of a (reduced) matrix.  With an offset every entry of
// every row, zeros included, becomes (v - offset_j) scale_j: the rows turn dense.  Scale only: v scale_j, the
// sparsity stays.  offset / scale are indexed by coefficient (index 0 = bias, untouched).
template <typename VT>
__global__ void transform_dense(const Rows R, const uint32_t *__restrict__ col, const VT *__restrict__ val, int64_t n,
                                int64_t m, const double *__restrict__ offset, const double *__restrict__ scale,
                                uint32_t *__restrict__ ocol, double *__restrict__ oval) {
  const int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= n) return;
  int64_t a, b;
  R.range(row, a, b);
  for (int64_t j = lane_id(); j < m; j += 32) {
    int64_t lo = a, hi = b;
    while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (col[mid] < (uint32_t)j) lo = mid + 1; else hi = mid; }
    const double v = (lo < b && col[lo] == (uint32_t)j) ? (val ? (double)val[lo] : 1.0) : 0.0;
    double t = v - offset[j + 1];
    if (scale) t *= scale[j + 1];
    ocol[row * m + j] = (uint32_t)j;
    oval[row * m + j] = t;
  }
}
template <typename VT>
__global__ void transform_scale(const uint32_t *__restrict__ col, const VT *__restrict__ val, int64_t nnz,
                                const double *__restrict__ scale, double *__restrict__ oval) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p < nnz) oval[p] = (val ? (double)val[p] : 1.0) * scale[col[p] + 1];
}

}  // namespace

std::shared_ptr<Matrix> matrix_transform(Matrix &M, const double *offset, const double *scale, int64_t len) {
  require_ready();
  KL_REQUIRE(len == M.m + 1, "transform: offset / scale must have one entry per coefficient (m + 1)");
  KL_REQUIRE(offset || scale, "transform: neither offset nor scale given");
  auto R = std::make_shared<Matrix>();
  R->n = M.n; R->m = M.m; R->vt = VAL_F64;
  R->sharded = M.sharded; R->n_global = M.n_global;
  R->n_classes = M.n_classes; R->class_k = M.class_k; R->class_code = M.class_code;
  DevBuf<double> doff, dsc;
  if (offset) { doff.alloc((size_t)len); doff.upload(offset, (size_t)len); }
  if (scale) { dsc.alloc((size_t)len); dsc.upload(scale, (size_t)len); }
  R->rowptr.alloc((size_t)M.n + 1);
  if (offset) {
    KL_REQUIRE(M.n * M.m < ((int64_t)1 << 31), "transform: a data transform with an offset makes the rows dense; "
               "this matrix would not fit (apply it to the reduced matrix of the selected features)");
    R->nnz = M.n * M.m;
    R->col.alloc((size_t)(R->nnz ? R->nnz : 1));
    R->val_f64.alloc((size_t)(R->nnz ? R->nnz : 1));
    std::vector<int64_t> rp((size_t)M.n + 1);
    for (int64_t i = 0; i <= M.n; i++) rp[(size_t)i] = i * M.m;
    R->rowptr.upload(rp.data(), (size_t)M.n + 1);
    if (M.n > 0 && M.m > 0) {
      const unsigned grid = (unsigned)((M.n * 32 + 127) / 128);
      if (M.vt == VAL_U32)
        KL_LAUNCH((transform_dense<uint32_t>), grid, 128, 0, M.rows(), M.col.p, M.val_u32.p, M.n, M.m, doff.p, dsc.p, R->col.p, R->val_f64.p);
      else if (M.vt == VAL_F64)
        KL_LAUNCH((transform_dense<double>), grid, 128, 0, M.rows(), M.col.p, M.val_f64.p, M.n, M.m, doff.p, dsc.p, R->col.p, R->val_f64.p);
      else
        KL_LAUNCH((transform_dense<uint32_t>), grid, 128, 0, M.rows(), M.col.p, (const uint32_t *)nullptr, M.n, M.m, doff.p, dsc.p, R->col.p, R->val_f64.p);
    }
    sync_stream();
  } else {
    matrix_compact(M);
    R->nnz = M.nnz;
    R->col.alloc((size_t)(R->nnz ? R->nnz : 1));
    R->val_f64.alloc((size_t)(R->nnz ? R->nnz : 1));
    KL_CUDA(cudaMemcpyAsync(R->rowptr.p, M.rowptr.p, (size_t)(M.n + 1) * sizeof(int64_t), cudaMemcpyDeviceToDevice, ctx().stream));
    if (M.nnz > 0) {
      KL_CUDA(cudaMemcpyAsync(R->col.p, M.col.p, (size_t)M.nnz * sizeof(uint32_t), cudaMemcpyDeviceToDevice, ctx().stream));
      const unsigned grid = (unsigned)((M.nnz + 255) / 256);
      if (M.vt == VAL_U32) KL_LAUNCH((transform_scale<uint32_t>), grid, 256, 0, M.col.p, M.val_u32.p, M.nnz, dsc.p, R->val_f64.p);
      else if (M.vt == VAL_F64) KL_LAUNCH((transform_scale<double>), grid, 256, 0, M.col.p, M.val_f64.p, M.nnz, dsc.p, R->val_f64.p);
      else KL_LAUNCH((transform_scale<uint32_t>), grid, 256, 0, M.col.p, (const uint32_t *)nullptr, M.nnz, dsc.p, R->val_f64.p);
    }
    sync_stream();
  }
  if (M.has_labels) {
    R->labels.alloc((size_t)(M.n ? M.n : 1));
    KL_CUDA(cudaMemcpyAsync(R->labels.p, M.labels.p, (size_t)M.n, cudaMemcpyDeviceToDevice, ctx().stream));
    matrix_label_counts_local(M);
    R->n_pos = M.n_pos; R->n_neg = M.n_neg; R->counts_global = M.counts_global; R->has_labels = true;
    sync_stream();
  }
  return R;
}

void matrix_pair_moments(Matrix &M, double *sum, double *sumsq, double *absmax, int64_t *count) {
  require_ready();
  KL_REQUIRE(M.vt != VAL_F64, "pair_moments: only count / binarized matrices (integer values) are supported");
  KL_REQUIRE(!M.sharded, "pair_moments: not available on a sharded matrix");
  const int64_t np = M.m * (M.m - 1) / 2;
  if (np <= 0) return;
  ensure_csc(M);
  DevBuf<unsigned long long> d((size_t)(4 * np));
  if (M.vt == VAL_U32)
    KL_LAUNCH((pair_moments<uint32_t>), (unsigned)(ctx().sm_count * 8), 256, 0, M.colptr.p, M.crow.p, M.cval_u32.p, M.m, d.p,
              d.p + np, d.p + 2 * np, d.p + 3 * np);
  else
    KL_LAUNCH((pair_moments<uint32_t>), (unsigned)(ctx().sm_count * 8), 256, 0, M.colptr.p, M.crow.p, (const uint32_t *)nullptr,
              M.m, d.p, d.p + np, d.p + 2 * np, d.p + 3 * np);
  std::vector<unsigned long long> h((size_t)(4 * np));
  d.download(h.data(), (size_t)(4 * np));
  sync_stream();
  for (int64_t j = 0; j < np; j++) {
    sum[j] = (double)h[(size_t)j]; sumsq[j] = (double)h[(size_t)(np + j)];
    absmax[j] = (double)h[(size_t)(2 * np + j)]; count[j] = (int64_t)h[(size_t)(3 * np + j)];
  }
}

void matrix_column_moments(Matrix &M, double *sum, double *sumsq, double *absmax, int64_t *count) {
  require_ready();
  KL_REQUIRE(M.vt != VAL_F64, "column_moments: only count / binarized matrices (integer values) are supported");
  DevBuf<unsigned long long> d((size_t)(4 * (M.m ? M.m : 1)));
  d.zero();
  if (M.n > 0 && M.m > 0)
    KL_LAUNCH((column_moments<uint32_t>), (unsigned)((M.n * 32 + 255) / 256), 256, 0, M.rows(), M.col.p,
              M.vt == VAL_U32 ? M.val_u32.p : (const uint32_t *)nullptr, M.n, d.p, d.p + M.m, d.p + 2 * M.m, d.p + 3 * M.m);
  if (M.sharded) {
    // sums and counts add up over the ranks, the maximum is taken separately
    DevBuf<double> mxd((size_t)(M.m ? M.m : 1));
    std::vector<unsigned long long> tmp((size_t)M.m);
    KL_CUDA(cudaMemcpyAsync(tmp.data(), d.p + 2 * M.m, (size_t)M.m * 8, cudaMemcpyDeviceToHost, ctx().stream));
    sync_stream();
    std::vector<double> hm((size_t)M.m);
    for (int64_t j = 0; j < M.m; j++) hm[(size_t)j] = (double)tmp[(size_t)j];
    mxd.upload(hm.data(), (size_t)M.m);
    comm_allreduce_max_f64(mxd.p, M.m);
    mxd.download(hm.data(), (size_t)M.m);
    KL_CUDA(cudaMemsetAsync(d.p + 2 * M.m, 0, (size_t)M.m * 8, ctx().stream));
    comm_allreduce_sum_i64((int64_t *)d.p, 4 * M.m);
    sync_stream();
    for (int64_t j = 0; j < M.m; j++) absmax[j] = hm[(size_t)j];
  }
  std::vector<unsigned long long> h((size_t)(4 * M.m));
  d.download(h.data(), (size_t)(4 * M.m));
  sync_stream();
  for (int64_t j = 0; j < M.m; j++) {
    sum[j] = (double)h[(size_t)j];
    sumsq[j] = (double)h[(size_t)(M.m + j)];
    if (!M.sharded) absmax[j] = (double)h[(size_t)(2 * M.m + j)];
    count[j] = (int64_t)h[(size_t)(3 * M.m + j)];
  }
}

// ---------------------------------------------------------------------------------------------------
std::shared_ptr<Matrix> matrix_from_csr(int64_t n, int64_t m, const int64_t *rowptr, const int32_t *col,
                                        const double *val, int flags) {
  require_ready();
  KL_REQUIRE(n >= 0 && m >= 0 && rowptr && rowptr[0] == 0, "from_csr: bad arguments");
  int64_t nnz = rowptr[n];
  for (int64_t i = 0; i < n; i++) {
    KL_REQUIRE(rowptr[i + 1] >= rowptr[i], "from_csr: rowptr must be non-decreasing");
    for (int64_t p = rowptr[i]; p < rowptr[i + 1]; p++) {
      KL_REQUIRE(col[p] >= 0 && col[p] < m, "from_csr: column out of range");
      KL_REQUIRE(p == rowptr[i] || col[p] > col[p - 1], "from_csr: columns must be strictly increasing in a row");
    }
  }
  auto M = std::make_shared<Matrix>();
  M->n = n; M->m = m; M->nnz = nnz; M->vt = VAL_F64;
  M->sharded = (flags & KMERLR_FLAG_SHARDED) != 0 && ctx().world > 1;
  M->n_global = n;
  M->rowptr.alloc((size_t)n + 1);
  M->col.alloc((size_t)(nnz ? nnz : 1));
  M->val_f64.alloc((size_t)(nnz ? nnz : 1));
  M->rowptr.upload(rowptr, (size_t)n + 1);
  std::vector<uint32_t> c32((size_t)nnz);
  for (int64_t p = 0; p < nnz; p++) c32[p] = (uint32_t)col[p];
  M->col.upload(c32.data(), (size_t)nnz);
  M->val_f64.upload(val, (size_t)nnz);
  if (M->sharded) {
    DevBuf<int64_t> tmp(1);
    int64_t nn = n;
    tmp.upload(&nn, 1);
    comm_allreduce_sum_i64(tmp.p, 1);
    tmp.download(&nn, 1);
    sync_stream();
    M->n_global = nn;
  }
  sync_stream();
  return M;
}

// padded rows (extraction layout) -> compact CSR: one gather, the padded arrays are released
template <typename VT>
__global__ void gather_rows(const uint32_t *__restrict__ rowcnt, int64_t stride, int64_t n,
                            const int64_t *__restrict__ rowptr, const uint32_t *__restrict__ col,
                            const VT *__restrict__ val, uint32_t *__restrict__ ocol, VT *__restrict__ oval) {
  int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= n) return;
  const unsigned lane = lane_id();
  const int64_t a = row * stride, o = rowptr[row];
  const uint32_t c = rowcnt[row];
  for (uint32_t j = lane; j < c; j += 32) {
    ocol[o + j] = col[a + j];
    if (val) oval[o + j] = val[a + j];
  }
}

void matrix_compact(Matrix &M) {
  if (M.row_stride == 0) return;
  require_ready();
  M.rowptr.alloc((size_t)M.n + 1);
  if (M.n > 0) exclusive_scan_u32_to_i64(M.rowcnt.p, M.rowptr.p, M.n); else M.rowptr.zero();
  DevBuf<uint32_t> ncol((size_t)(M.nnz ? M.nnz : 1)), nval;
  if (M.vt == VAL_U32) nval.alloc((size_t)(M.nnz ? M.nnz : 1));
  if (M.n > 0)
    KL_LAUNCH((gather_rows<uint32_t>), (unsigned)((M.n * 32 + 127) / 128), 128, 0, M.rowcnt.p, M.row_stride, M.n,
              M.rowptr.p, M.col.p, M.vt == VAL_U32 ? M.val_u32.p : (const uint32_t *)nullptr, ncol.p,
              M.vt == VAL_U32 ? nval.p : (uint32_t *)nullptr);
  sync_stream();
  M.col = std::move(ncol);
  if (M.vt == VAL_U32) M.val_u32 = std::move(nval);
  M.rowcnt.release();
  M.row_stride = 0;
}

void matrix_rows(Matrix &M, int64_t *rowptr, int32_t *col, double *val) {
  require_ready();
  matrix_compact(M);
  M.rowptr.download(rowptr, (size_t)M.n + 1);
  std::vector<uint32_t> c32((size_t)M.nnz);
  M.col.download(c32.data(), (size_t)M.nnz);
  std::vector<uint32_t> v32;
  if (M.vt == VAL_U32) { v32.resize((size_t)M.nnz); M.val_u32.download(v32.data(), (size_t)M.nnz); }
  else if (M.vt == VAL_F64) M.val_f64.download(val, (size_t)M.nnz);
  sync_stream();
  for (int64_t p = 0; p < M.nnz; p++) {
    col[p] = (int32_t)c32[p];
    if (M.vt == VAL_U32) val[p] = (double)v32[p];
    else if (M.vt == VAL_ONE) val[p] = 1.0;
  }
}

// labels[i] = raw[i] != 0 in place, *ones += the number of ones
__global__ void normalize_labels(uint8_t *__restrict__ labels, int64_t n, unsigned long long *__restrict__ ones) {
  __shared__ unsigned int sh;
  if (threadIdx.x == 0) sh = 0u;
  __syncthreads();
  unsigned int c = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const uint8_t v = labels[i] != 0;
    labels[i] = v;
    c += v;
  }
  if (c) atomicAdd(&sh, c);
  __syncthreads();
  if (threadIdx.x == 0 && sh) atomicAdd(ones, (unsigned long long)sh);
}

// the labels go up through the pinned staging buffer and are normalised and counted on the device: no host pass
// over them and no wait for the device (the count is read when somebody asks for it)
void matrix_set_labels(Matrix &M, const uint8_t *labels, int64_t n) {
  require_ready();
  KL_REQUIRE(n == M.n, "labels: length does not match the number of rows");
  M.labels.alloc((size_t)(n ? n : 1));
  M.label_ones.alloc(1);
  M.label_ones.zero();
  if (n > 0) {
    uint8_t *h = (uint8_t *)host_staging((size_t)n);
    memcpy(h, labels, (size_t)n);
    M.labels.upload(h, (size_t)n);
    host_staging_done();
    int64_t blocks = (n + 255) / 256;
    if (blocks > 4 * ctx().sm_count) blocks = 4 * ctx().sm_count;
    KL_LAUNCH(normalize_labels, (unsigned)blocks, 256, 0, M.labels.p, n, M.label_ones.p);
  }
  // the global counts (class weights) are summed over the ranks when somebody asks: no collective here
  M.counts_pending = true;
  M.counts_global = !M.sharded;
  M.has_labels = true;
}

void matrix_label_counts_local(Matrix &M) {
  if (!M.counts_pending) return;
  unsigned long long ones = 0;
  M.label_ones.download(&ones, 1);
  sync_stream();
  M.n_pos = (int64_t)ones; M.n_neg = M.n - (int64_t)ones;
  M.counts_pending = false;
}

void matrix_label_counts(Matrix &M) {
  matrix_label_counts_local(M);
  if (M.counts_global) return;
  int64_t cnt[2] = {M.n_neg, M.n_pos};
  DevBuf<int64_t> tmp(2);
  tmp.upload(cnt, 2);
  comm_allreduce_sum_i64(tmp.p, 2);
  tmp.download(cnt, 2);
  sync_stream();
  M.n_neg = cnt[0]; M.n_pos = cnt[1];
  M.counts_global = true;
}

template <typename VT>
static void build_csc(Matrix &M, const VT *val, VT *cval) {
  const int64_t nnz = M.nnz, ntiles = (nnz + RS_TILE - 1) / RS_TILE;
  int bits = 1;
  while (((int64_t)1 << bits) < M.m) bits++;
  const int passes = (bits + 7) / 8;
  Trace tr("csc");
  DevBuf<uint32_t> hist((size_t)(256 * ntiles));
  DevBuf<int64_t> offs((size_t)(256 * ntiles) + 1);
  // ping-pong buffers; the last pass writes straight into the CSC arrays
  DevBuf<uint32_t> kA((size_t)nnz), kB(passes > 1 ? (size_t)nnz : 1), rA(passes > 1 ? (size_t)nnz : 1),
      rB(passes > 2 ? (size_t)nnz : 1);
  DevBuf<VT> vA(val && passes > 1 ? (size_t)nnz : 1), vB(val && passes > 2 ? (size_t)nnz : 1);
  const uint32_t *kin = M.col.p, *rin = nullptr;
  const VT *vin = val;
  tr.mark("alloc");
  for (int ps = 0; ps < passes; ps++) {
    const bool last = ps == passes - 1;
    uint32_t *kout = (ps & 1) ? kB.p : kA.p;
    if (passes == 1) kout = kA.p;
    uint32_t *rout = last ? M.crow.p : ((ps & 1) ? rB.p : rA.p);
    VT *vout = val ? (last ? cval : ((ps & 1) ? vB.p : vA.p)) : nullptr;
    KL_LAUNCH(radix_hist, (unsigned)ntiles, RS_THREADS, 0, kin, nnz, 8 * ps, hist.p, ntiles);
    exclusive_scan_u32_to_i64(hist.p, offs.p, 256 * ntiles);
    const size_t smem = (size_t)RS_TILE * (8 + (val ? sizeof(VT) : 0));
    if (ps == 0) {
      KL_CUDA(cudaFuncSetAttribute(radix_scatter<VT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      KL_LAUNCH((radix_scatter<VT, true>), (unsigned)ntiles, RS_THREADS, smem, kin, rin, M.rowptr.p, M.n, vin, nnz, 8 * ps,
                offs.p, ntiles, kout, rout, vout);
    } else {
      KL_CUDA(cudaFuncSetAttribute(radix_scatter<VT, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      KL_LAUNCH((radix_scatter<VT, false>), (unsigned)ntiles, RS_THREADS, smem, kin, rin, M.rowptr.p, M.n, vin, nnz, 8 * ps,
                offs.p, ntiles, kout, rout, vout);
    }
    kin = kout; rin = rout; vin = vout;
    tr.mark("pass");
  }
  KL_LAUNCH(lower_bounds, (unsigned)((M.m + 1 + 255) / 256), 256, 0, kin, nnz, M.m, M.colptr.p);
  sync_stream();
}

void ensure_csc(Matrix &M) {
  if (M.has_csc) return;
  matrix_compact(M);          // the transpose walks the stored entries as one contiguous array
  M.colptr.alloc((size_t)M.m + 1);
  M.crow.alloc((size_t)(M.nnz ? M.nnz : 1));
  if (M.m == 0 || M.n == 0 || M.nnz == 0) {
    M.colptr.zero();
  } else if (M.vt == VAL_U32) {
    M.cval_u32.alloc((size_t)(M.nnz ? M.nnz : 1));
    build_csc<uint32_t>(M, M.val_u32.p, M.cval_u32.p);
  } else if (M.vt == VAL_F64) {
    M.cval_f64.alloc((size_t)(M.nnz ? M.nnz : 1));
    build_csc<double>(M, M.val_f64.p, M.cval_f64.p);
  } else {
    build_csc<uint32_t>(M, nullptr, nullptr);
  }
  sync_stream();
  M.has_csc = true;
}

// ---- sliced view: slices of 32 rows, column-major inside a slice -----------------------------------------------
__global__ void slice_widths(const int64_t *__restrict__ rowptr, int64_t n, int64_t nslices, uint32_t *__restrict__ width32) {
  const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= nslices) return;
  int64_t w = 0;
  for (int64_t r = 32 * s; r < 32 * s + 32 && r < n; r++) w = max(w, rowptr[r + 1] - rowptr[r]);
  width32[s] = (uint32_t)w;                  // slots of the slice = 32 w
}

template <typename VT>
__global__ void slice_fill(const int64_t *__restrict__ rowptr, const uint32_t *__restrict__ col, const VT *__restrict__ val,
                           int64_t n, const int64_t *__restrict__ slice_off, uint32_t *__restrict__ scol, VT *__restrict__ sval) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n) return;
  const int64_t a = rowptr[row], b = rowptr[row + 1], base = 32 * slice_off[row >> 5] + (row & 31);
  for (int64_t p = a; p < b; p++) {
    scol[base + 32 * (p - a)] = col[p];
    if (val) sval[base + 32 * (p - a)] = val[p];
  }
}

void ensure_sliced(Matrix &M) {
  if (M.has_sliced) return;
  matrix_compact(M);
  const int64_t ns = (M.n + 31) / 32;
  M.slice_off.alloc((size_t)ns + 1);
  if (ns == 0) { M.slice_off.zero(); M.has_sliced = true; return; }
  DevBuf<uint32_t> w((size_t)ns);
  KL_LAUNCH(slice_widths, (unsigned)((ns + 255) / 256), 256, 0, M.rowptr.p, M.n, ns, w.p);
  exclusive_scan_u32_to_i64(w.p, M.slice_off.p, ns);            // in units of 32 slots
  int64_t total = 0;
  KL_CUDA(cudaMemcpyAsync(&total, M.slice_off.p + ns, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx().stream));
  sync_stream();
  const size_t slots = (size_t)(32 * total > 0 ? 32 * total : 1);
  M.scol.alloc(slots);
  const unsigned blocks = (unsigned)((M.n + 255) / 256);
  if (M.vt == VAL_U32) {
    M.sval_u32.alloc(slots);
    KL_LAUNCH((slice_fill<uint32_t>), blocks, 256, 0, M.rowptr.p, M.col.p, M.val_u32.p, M.n, M.slice_off.p, M.scol.p, M.sval_u32.p);
  } else if (M.vt == VAL_F64) {
    M.sval_f64.alloc(slots);
    KL_LAUNCH((slice_fill<double>), blocks, 256, 0, M.rowptr.p, M.col.p, M.val_f64.p, M.n, M.slice_off.p, M.scol.p, M.sval_f64.p);
  } else {
    KL_LAUNCH((slice_fill<uint32_t>), blocks, 256, 0, M.rowptr.p, M.col.p, (const uint32_t *)nullptr, M.n, M.slice_off.p, M.scol.p,
              (uint32_t *)nullptr);
  }
  M.has_sliced = true;
}

template <typename VT>
__global__ void pack_entries(const uint32_t *__restrict__ idx, const VT *__restrict__ val, int64_t count, int shift,
                             uint32_t *__restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) out[i] = idx[i] | ((val ? (uint32_t)val[i] : 1u) << shift);
}

// real values that are all small counts (what a reduced count matrix holds)?
__global__ void count_non_counts(const double *__restrict__ val, int64_t count, double limit, unsigned int *__restrict__ bad) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const double v = val[i];
  if (!(v >= 0.0 && v < limit && v == floor(v))) atomicAdd(bad, 1u);
}

bool ensure_packed(Matrix &M) {
  if (M.has_packed) return M.packable;
  M.has_packed = true;
  M.packable = false;
  if (M.m > 1024 || M.n < 1 || M.nnz < 1) return false;
  int rb = 1;
  while (((int64_t)1 << rb) < M.n) rb++;
  if (rb > 24) return false;
  const double limit = (double)(1u << (32 - rb < 22 ? 32 - rb : 22));
  matrix_compact(M);
  if (M.vt == VAL_U32) {
    if (matrix_vmax(M) >= limit) return false;                       // (cached by the callers: no collective here)
  } else if (M.vt == VAL_F64) {
    DevBuf<unsigned int> bad(1);
    bad.zero();
    KL_LAUNCH(count_non_counts, (unsigned)((M.nnz + 255) / 256), 256, 0, M.val_f64.p, M.nnz, limit, bad.p);
    unsigned int nbad = 0;
    bad.download(&nbad, 1);
    sync_stream();
    if (nbad) return false;
  }
  ensure_sliced(M);
  ensure_csc(M);
  M.pack_row_bits = rb;
  const int64_t slots = (int64_t)M.scol.n;
  M.spack.alloc((size_t)slots);
  M.cpack.alloc((size_t)M.nnz);
  // (padding slots of the sliced view hold whatever the allocation held; nobody reads them)
  const unsigned sb = (unsigned)((slots + 255) / 256), cb = (unsigned)((M.nnz + 255) / 256);
  if (M.vt == VAL_F64) {
    KL_LAUNCH((pack_entries<double>), sb, 256, 0, M.scol.p, M.sval_f64.p, slots, 10, M.spack.p);
    KL_LAUNCH((pack_entries<double>), cb, 256, 0, M.crow.p, M.cval_f64.p, M.nnz, rb, M.cpack.p);
  } else {
    const uint32_t *sval = M.vt == VAL_U32 ? M.sval_u32.p : nullptr, *cval = M.vt == VAL_U32 ? M.cval_u32.p : nullptr;
    KL_LAUNCH((pack_entries<uint32_t>), sb, 256, 0, M.scol.p, sval, slots, 10, M.spack.p);
    KL_LAUNCH((pack_entries<uint32_t>), cb, 256, 0, M.crow.p, cval, M.nnz, rb, M.cpack.p);
  }
  M.packable = true;
  return true;
}

// ---- block-local column-major view (see Matrix::bv_*) ---------------------------------------------------------------
// first entry of column c with row >= n b / grid, for b = 0 .. grid (b = grid: the end of the column)
__global__ void bv_bounds(const int64_t *__restrict__ colptr, const uint32_t *__restrict__ cpack, uint32_t rmask, int64_t n,
                          int64_t m, int grid, int64_t *__restrict__ lb) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)(grid + 1) * m) return;
  const int64_t b = idx / m, c = idx % m;
  const int64_t row_lo = n * b / grid;
  int64_t lo = colptr[c], hi = colptr[c + 1];
  while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if ((int64_t)(cpack[mid] & rmask) < row_lo) lo = mid + 1; else hi = mid; }
  lb[idx] = lo;
}
// per block: position of its first entry of every column in the block's list, number of entries, share width
__global__ void bv_starts(const int64_t *__restrict__ lb, int64_t m, int grid, int64_t *__restrict__ start,
                          uint32_t *__restrict__ width) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= grid) return;
  int64_t run = 0;
  for (int64_t c = 0; c < m; c++) { start[b * m + c] = run; run += lb[(b + 1) * m + c] - lb[b * m + c]; }
  width[b] = (uint32_t)((run + 255) / 256);
}
__global__ void bv_fill(const int64_t *__restrict__ lb, const int64_t *__restrict__ start, const uint32_t *__restrict__ width,
                        const int64_t *__restrict__ off, const uint32_t *__restrict__ cpack, int crow_bits, int64_t n, int64_t m,
                        int grid, int row_bits, uint32_t *__restrict__ out, unsigned int *__restrict__ bad) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)grid * m) return;
  const int64_t b = idx / m, c = idx % m;
  const int64_t p0 = lb[b * m + c], p1 = lb[(b + 1) * m + c], row_lo = n * b / grid;
  const int64_t w = width[b];
  const uint32_t rmask = (1u << crow_bits) - 1u;
  for (int64_t p = p0; p < p1; p++) {
    const uint32_t e = cpack[p], cnt = e >> crow_bits;
    const int64_t lr = (int64_t)(e & rmask) - row_lo;
    if (lr < 0 || lr >= ((int64_t)1 << row_bits) || (row_bits + 10 < 32 && (cnt >> (32 - row_bits - 10)) != 0u)) { atomicAdd(bad, 1u); continue; }
    const int64_t q = start[b * m + c] + (p - p0), t = q / w, j = q % w;
    out[256 * (off[b] + j) + t] = (uint32_t)lr | ((uint32_t)c << row_bits) | (cnt << (row_bits + 10));
  }
}

bool ensure_blockview(Matrix &M, int grid) {
  if (M.bv_grid == grid) return M.bv_ok;
  M.bv_grid = grid; M.bv_ok = false;
  if (!ensure_packed(M) || grid < 1 || M.m < 1 || M.m > 1024) return false;
  const int64_t rows = (M.n + grid - 1) / grid + 1;             // upper bound of the rows of one block
  int rb = 1;
  while (((int64_t)1 << rb) < rows) rb++;
  if (rb + 10 > 28 || rows * 8 > 32 * 1024) return false;       // (at least 4 bits of count; the block's weights live in 32 KB)
  DevBuf<int64_t> lb((size_t)(grid + 1) * M.m), start((size_t)grid * M.m);
  DevBuf<uint32_t> width((size_t)grid);
  const uint32_t rmask = (1u << M.pack_row_bits) - 1u;
  KL_LAUNCH(bv_bounds, (unsigned)(((int64_t)(grid + 1) * M.m + 255) / 256), 256, 0, M.colptr.p, M.cpack.p, rmask, M.n, M.m, grid, lb.p);
  KL_LAUNCH(bv_starts, (unsigned)((grid + 127) / 128), 128, 0, lb.p, M.m, grid, start.p, width.p);
  M.bv_off.alloc((size_t)grid + 1);
  exclusive_scan_u32_to_i64(width.p, M.bv_off.p, grid);
  int64_t total = 0;
  KL_CUDA(cudaMemcpyAsync(&total, M.bv_off.p + grid, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx().stream));
  sync_stream();
  M.bv_pack.alloc((size_t)(total > 0 ? 256 * total : 1));
  KL_CUDA(cudaMemsetAsync(M.bv_pack.p, 0xFF, (size_t)(total > 0 ? 256 * total : 1) * sizeof(uint32_t), ctx().stream));
  DevBuf<unsigned int> bad(1);
  bad.zero();
  KL_LAUNCH(bv_fill, (unsigned)(((int64_t)grid * M.m + 255) / 256), 256, 0, lb.p, start.p, width.p, M.bv_off.p, M.cpack.p,
            M.pack_row_bits, M.n, M.m, grid, rb, M.bv_pack.p, bad.p);
  unsigned int nbad = 0;
  bad.download(&nbad, 1);
  sync_stream();
  if (nbad) return false;                                       // a count does not fit beside the row and the column
  M.bv_row_bits = rb; M.bv_rows = (int)rows;
  M.bv_ok = true;
  return true;
}

std::shared_ptr<Matrix> matrix_reduce(Matrix &M, const int64_t *sel, int64_t nsel) {
  require_ready();
  KL_REQUIRE(nsel >= 1 && sel[0] == 0, "reduce: sel[0] must be the bias (0)");
  const int64_t dim = kmerlr_coeff_dim(M.m);
  std::vector<int64_t> A((size_t)(nsel - 1)), B((size_t)(nsel - 1));
  for (int64_t j = 1; j < nsel; j++) {
    KL_REQUIRE(sel[j] > sel[j - 1] && sel[j] < dim, "reduce: coefficient indices must be ascending and in range");
    if (sel[j] >= M.m + 1) {
      int64_t i1, i2;
      kmerlr_coeff_sub2ind(M.m, sel[j] - 1, &i1, &i2);
      A[j - 1] = i1; B[j - 1] = i2;
    } else {
      A[j - 1] = sel[j] - 1; B[j - 1] = -1;
    }
  }
  auto R = std::make_shared<Matrix>();
  R->n = M.n; R->m = nsel - 1; R->vt = VAL_F64;
  R->sharded = M.sharded; R->n_global = M.n_global;
  const int64_t ns = nsel - 1;
  DevBuf<int64_t> dA((size_t)(ns ? ns : 1)), dB((size_t)(ns ? ns : 1));
  dA.upload(A.data(), (size_t)ns); dB.upload(B.data(), (size_t)ns);
  DevBuf<uint32_t> cnt((size_t)(M.n ? M.n : 1));
  R->rowptr.alloc((size_t)M.n + 1);
  unsigned wgrid = (unsigned)((M.n * 32 + 127) / 128);
  auto run = [&](auto *valp) {
    using VT = typename std::remove_const<typename std::remove_pointer<decltype(valp)>::type>::type;
    if (M.n > 0) {
      KL_LAUNCH((reduce_rows<VT, false>), wgrid, 128, 0, M.rows(), M.col.p, valp, M.n, dA.p, dB.p, ns, cnt.p,
                nullptr, nullptr, nullptr);
      exclusive_scan_u32_to_i64(cnt.p, R->rowptr.p, M.n);
      KL_CUDA(cudaMemcpyAsync(&R->nnz, R->rowptr.p + M.n, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx().stream));
      sync_stream();
    } else {
      R->rowptr.zero(); R->nnz = 0;
    }
    R->col.alloc((size_t)(R->nnz ? R->nnz : 1));
    R->val_f64.alloc((size_t)(R->nnz ? R->nnz : 1));
    if (M.n > 0)
      KL_LAUNCH((reduce_rows<VT, true>), wgrid, 128, 0, M.rows(), M.col.p, valp, M.n, dA.p, dB.p, ns, nullptr,
                R->rowptr.p, R->col.p, R->val_f64.p);
    sync_stream();
  };
  if (M.vt == VAL_U32) run((const uint32_t *)M.val_u32.p);
  else if (M.vt == VAL_F64) run((const double *)M.val_f64.p);
  else run((const uint32_t *)nullptr);
  if (M.has_labels) {
    R->labels.alloc((size_t)(M.n ? M.n : 1));
    KL_CUDA(cudaMemcpyAsync(R->labels.p, M.labels.p, (size_t)M.n, cudaMemcpyDeviceToDevice, ctx().stream));
    matrix_label_counts_local(M);
    R->n_pos = M.n_pos; R->n_neg = M.n_neg; R->counts_global = M.counts_global; R->has_labels = true;
    sync_stream();
  }
  return R;
}

// max_i ||x_i||^2 without the bias (estimate_step_size, kmerLr_estimator_proximal.go:54-69) and
// max |x_ij| over the stored entries (fixed-point scale of the gradient accumulation): computed together,
// one MAX all-reduce over the ranks
static void ensure_stats(Matrix &M) {
  if (M.has_maxsq && M.has_vmax) return;
  double v[2] = {0.0, 0.0};
  if (M.has_local_stats) {
    v[0] = M.local_maxsq; v[1] = M.local_vmax;
  } else {
    matrix_compact(M);
    DevBuf<unsigned long long> d(2);
    d.zero();
    if (M.n > 0) {
      unsigned wgrid = (unsigned)((M.n * 32 + 127) / 128);
      if (M.vt == VAL_U32) KL_LAUNCH((row_sqnorm_max<uint32_t>), wgrid, 128, 0, M.rows(), M.val_u32.p, M.n, d.p);
      else if (M.vt == VAL_F64) KL_LAUNCH((row_sqnorm_max<double>), wgrid, 128, 0, M.rows(), M.val_f64.p, M.n, d.p);
      else KL_LAUNCH((row_sqnorm_max<uint32_t>), wgrid, 128, 0, M.rows(), (const uint32_t *)nullptr, M.n, d.p);
    }
    if (M.nnz > 0) {
      if (M.vt == VAL_U32) KL_LAUNCH((abs_max<uint32_t>), 1024, 256, 0, M.val_u32.p, M.nnz, d.p + 1);
      else if (M.vt == VAL_F64) KL_LAUNCH((abs_max<double>), 1024, 256, 0, M.val_f64.p, M.nnz, d.p + 1);
    }
    unsigned long long bits[2] = {0, 0};
    d.download(bits, 2);
    sync_stream();
    memcpy(v, bits, sizeof(v));
    if (M.vt == VAL_ONE) v[1] = M.nnz > 0 ? 1.0 : 0.0;
  }
  if (M.sharded) {
    DevBuf<double> t(2);
    t.upload(v, 2);
    comm_allreduce_max_f64(t.p, 2);
    t.download(v, 2);
    sync_stream();
  }
  M.maxsq = v[0]; M.has_maxsq = true;
  M.vmax = v[1]; M.has_vmax = true;
}

double matrix_maxsq(Matrix &M) {
  ensure_stats(M);
  return M.maxsq;
}

double matrix_maxsq_pairs(Matrix &M) {
  KL_INVARIANT(!M.sharded);
  if (M.has_maxsq_pairs) return M.maxsq_pairs;
  matrix_compact(M);
  DevBuf<unsigned long long> d(1);
  d.zero();
  if (M.n > 0) {
    unsigned wgrid = (unsigned)((M.n * 32 + 127) / 128);
    if (M.vt == VAL_F64) KL_LAUNCH((row_sqnorm_pairs_max<double>), wgrid, 128, 0, M.rows(), M.val_f64.p, M.n, d.p);
    else KL_LAUNCH((row_sqnorm_pairs_max<uint32_t>), wgrid, 128, 0, M.rows(), M.vt == VAL_U32 ? M.val_u32.p : nullptr, M.n, d.p);
  }
  unsigned long long bits = 0;
  d.download(&bits, 1);
  sync_stream();
  memcpy(&M.maxsq_pairs, &bits, sizeof(double));
  M.has_maxsq_pairs = true;
  return M.maxsq_pairs;
}

double matrix_vmax(Matrix &M) {
  ensure_stats(M);
  return M.vmax;
}

}  // namespace kl
