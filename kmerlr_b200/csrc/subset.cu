// subset.cu -- a row subset of a resident matrix (filterCvGroup, kmerLr_crossvalidation.go:95): the folds of a
// cross-validation and the subsamples of an ensemble are row subsets of ONE compiled data set, so they keep its
// columns, its class numbering and every view it has.  Stored rows and labels are gathered; the matrix-free view
// gathers only per-row metadata and points into the parent's packed sequences.
#include "common.cuh"

namespace kl {

namespace {

// totals the host reads back in one round trip
enum : int { ST_NNZ = 0, ST_ONES, ST_MAXLEN, ST_BASES, ST_MAXSQ, ST_VMAX, ST_COUNT };

// thread per subset row: row lengths (the layout's count, or the scan input of a compact subset), labels, and the
// per-row arrays of the matrix-free view; the entries, ones and bases are summed and the longest sequence taken per
// block, one atomic each per block
__global__ void __launch_bounds__(256) subset_rows(const int64_t *__restrict__ rows, int64_t nrows, const Rows R,
                                                   uint32_t *__restrict__ cnt, const uint8_t *__restrict__ labels,
                                                   uint8_t *__restrict__ olabels, const int64_t *__restrict__ len,
                                                   const int64_t *__restrict__ blk, int64_t *__restrict__ olen,
                                                   int64_t *__restrict__ oblk, const int64_t *__restrict__ evptr,
                                                   uint32_t *__restrict__ evcnt, unsigned long long *__restrict__ st) {
  __shared__ unsigned long long part[4][8];
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long v[4] = {0, 0, 0, 0};       // entries, ones, bases, longest sequence
  if (i < nrows) {
    const int64_t r = rows[i];
    int64_t a, b;
    R.range(r, a, b);
    cnt[i] = (uint32_t)(b - a);
    v[0] = (unsigned long long)(b - a);
    if (labels) { const uint8_t l = labels[r]; olabels[i] = l; v[1] = l; }
    if (len) {
      const int64_t L = len[r];
      olen[i] = L; oblk[i] = blk[r];
      v[2] = v[3] = (unsigned long long)L;
    }
    if (evptr) evcnt[i] = (uint32_t)(evptr[r + 1] - evptr[r]);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
    for (int q = 0; q < 3; q++) v[q] += __shfl_xor_sync(0xffffffffu, v[q], o);
    const unsigned long long y = __shfl_xor_sync(0xffffffffu, v[3], o);
    v[3] = y > v[3] ? y : v[3];
  }
  const int w = threadIdx.x >> 5;
  if (lane_id() == 0)
    for (int q = 0; q < 4; q++) part[q][w] = v[q];
  __syncthreads();
  if (threadIdx.x < 4) {
    unsigned long long s = 0;
    for (int u = 0; u < (int)(blockDim.x >> 5); u++)
      s = threadIdx.x == 3 ? (part[3][u] > s ? part[3][u] : s) : s + part[threadIdx.x][u];
    const int slot = threadIdx.x == 0 ? ST_NNZ : (threadIdx.x == 1 ? ST_ONES : (threadIdx.x == 2 ? ST_BASES : ST_MAXLEN));
    if (s) {
      if (threadIdx.x == 3) atomicMax(st + slot, s);
      else atomicAdd(st + slot, s);
    }
  }
}

template <int V> struct Vec;
template <> struct Vec<1> { using T = uint32_t; };
template <> struct Vec<2> { using T = uint2; };
template <> struct Vec<4> { using T = uint4; };

__device__ __forceinline__ uint32_t vget(uint32_t x, int) { return x; }
__device__ __forceinline__ uint32_t vget(uint2 x, int q) { return q ? x.y : x.x; }
__device__ __forceinline__ uint32_t vget(uint4 x, int q) { return q == 0 ? x.x : (q == 1 ? x.y : (q == 2 ? x.z : x.w)); }

// padded rows (straight from the extraction): warp per subset row, V slots per lane and load (V divides the stride,
// so rounding a row up to V slots stays inside its own slots); the row's sum of squares and largest value go to the
// statistics the step size and the fixed-point scale need (the extraction computes them the same way)
template <int V>
__global__ void __launch_bounds__(128) subset_padded(const int64_t *__restrict__ rows, int64_t nrows, int64_t stride,
                                                     const uint32_t *__restrict__ cnt, const uint32_t *__restrict__ col,
                                                     const uint32_t *__restrict__ val, uint32_t *__restrict__ ocol,
                                                     uint32_t *__restrict__ oval, unsigned long long *__restrict__ st) {
  using T = typename Vec<V>::T;
  const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (i >= nrows) return;
  const unsigned lane = lane_id();
  const uint32_t c = cnt[i];
  const int64_t nv = (c + V - 1) / V;
  const T *sc = (const T *)(col + rows[i] * stride), *sv = val ? (const T *)(val + rows[i] * stride) : nullptr;
  T *dc = (T *)(ocol + i * stride), *dv = val ? (T *)(oval + i * stride) : nullptr;
  double sq = 0.0;
  uint32_t mx = 0;
  for (int64_t j = lane; j < nv; j += 32) {
    dc[j] = __ldcs(sc + j);
    if (val) {
      const T x = __ldcs(sv + j);
      dv[j] = x;
#pragma unroll
      for (int q = 0; q < V; q++)
        if (j * V + q < c) { const uint32_t v = vget(x, q); sq += (double)v * (double)v; mx = v > mx ? v : mx; }
    }
  }
  if (!val) { sq = (double)c; mx = c ? 1u : 0u; }
  else {
    sq = warp_sum(sq);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { const uint32_t y = __shfl_xor_sync(0xffffffffu, mx, o); mx = y > mx ? y : mx; }
  }
  // non-negative doubles compare like their bit patterns
  if (lane == 0) {
    atomicMax(st + ST_MAXSQ, (unsigned long long)__double_as_longlong(sq));
    if (mx) atomicMax(st + ST_VMAX, (unsigned long long)__double_as_longlong((double)mx));
  }
}

// compact rows, and the repeat events of the matrix-free view: warp per subset row copies the range sptr[rows[i]] ..
// of the parent to dptr[i] .. (b: values beside a, or nullptr)
template <typename VT>
__global__ void __launch_bounds__(128) subset_ranges(const int64_t *__restrict__ rows, int64_t nrows,
                                                     const int64_t *__restrict__ sptr, const int64_t *__restrict__ dptr,
                                                     const uint32_t *__restrict__ a, const VT *__restrict__ b,
                                                     uint32_t *__restrict__ oa, VT *__restrict__ ob) {
  const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (i >= nrows) return;
  const int64_t r = rows[i], s = sptr[r], c = sptr[r + 1] - s, d = dptr[i];
  for (int64_t j = lane_id(); j < c; j += 32) {
    oa[d + j] = __ldcs(a + s + j);
    if (b) ob[d + j] = __ldcs(b + s + j);
  }
}

// fixed-width per-row words (the class bitmaps of binarized rows): thread per word
__global__ void subset_words(const int64_t *__restrict__ rows, int64_t nrows, int width, const uint32_t *__restrict__ src,
                             uint32_t *__restrict__ dst) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nrows * width) return;
  const int64_t i = t / width, j = t % width;
  dst[t] = src[rows[i] * width + j];
}

template <typename VT>
void gather_compact(const Matrix &P, Matrix &R, const int64_t *drows, const VT *val, VT *oval) {
  KL_LAUNCH((subset_ranges<VT>), (unsigned)((R.n * 32 + 127) / 128), 128, 0, drows, R.n, P.rowptr.p, R.rowptr.p, P.col.p,
            val, R.col.p, oval);
}

}  // namespace

std::shared_ptr<Matrix> matrix_subset(Matrix &P, const int64_t *rows, int64_t nrows) {
  require_ready();
  KL_REQUIRE(!P.sharded, "matrix_subset: a sharded matrix is refused (the row indices of a shard cannot be checked against "
             "the rows of the other ranks); take the subset before sharding");
  KL_REQUIRE(nrows > 0, "matrix_subset: nrows must be at least 1");
  KL_REQUIRE(rows, "matrix_subset: null argument");
  for (int64_t i = 0; i < nrows; i++)
    KL_REQUIRE(rows[i] >= 0 && rows[i] < P.n, "matrix_subset: row index " + std::to_string(rows[i]) + " at position " +
               std::to_string(i) + " is outside [0, " + std::to_string(P.n) + ")");
  const bool padded = P.row_stride > 0;
  KL_INVARIANT(!padded || P.vt != VAL_F64);
  auto R = std::make_shared<Matrix>();
  R->n = nrows; R->m = P.m; R->vt = P.vt; R->n_global = nrows;
  // the class list of the parent, as it is (on the device or decoded)
  R->n_classes = P.n_classes;
  R->class_M = P.class_M; R->class_N = P.class_N; R->classes_on_host = P.classes_on_host;
  for (int k = 0; k < 16; k++) R->class_level_off[k] = P.class_level_off[k];
  R->class_k = P.class_k; R->class_code = P.class_code;
  if (P.class_ids.n) {
    R->class_ids.alloc(P.class_ids.n);
    KL_CUDA(cudaMemcpyAsync(R->class_ids.p, P.class_ids.p, P.class_ids.bytes(), cudaMemcpyDeviceToDevice, ctx().stream));
  }
  DevBuf<int64_t> drows((size_t)nrows);
  drows.upload(rows, (size_t)nrows);
  DevBuf<unsigned long long> st(ST_COUNT);
  st.zero();

  // ---- per-row pass: lengths, labels, the matrix-free view's row metadata -------------------------------------------
  const Implicit *I = P.imp.get();
  std::shared_ptr<Implicit> imp;
  std::shared_ptr<SeqSet> seqs;
  DevBuf<uint32_t> cnt(padded ? 0 : (size_t)nrows), evcnt;
  if (padded) R->rowcnt.alloc((size_t)nrows);
  if (P.has_labels) {
    R->labels.alloc((size_t)nrows);
    R->label_ones.alloc(1);
  }
  if (I) {
    imp = std::make_shared<Implicit>();
    seqs = std::make_shared<SeqSet>();
    seqs->n = nrows;
    seqs->len.alloc((size_t)nrows);
    seqs->blk.alloc((size_t)nrows);
    if (I->binarized) evcnt.alloc((size_t)nrows);
  }
  KL_LAUNCH(subset_rows, (unsigned)((nrows + 255) / 256), 256, 0, drows.p, nrows, P.rows(), padded ? R->rowcnt.p : cnt.p,
            P.has_labels ? P.labels.p : (const uint8_t *)nullptr, R->labels.p, I ? I->seqs->len.p : (const int64_t *)nullptr,
            I ? I->seqs->blk.p : (const int64_t *)nullptr, I ? seqs->len.p : (int64_t *)nullptr,
            I ? seqs->blk.p : (int64_t *)nullptr, I && I->binarized ? I->evptr.p : (const int64_t *)nullptr, evcnt.p, st.p);
  if (!padded) {
    R->rowptr.alloc((size_t)nrows + 1);
    exclusive_scan_u32_to_i64(cnt.p, R->rowptr.p, nrows);
  }
  DevBuf<int64_t> evptr;
  if (I && I->binarized) {
    evptr.alloc((size_t)nrows + 1);
    exclusive_scan_u32_to_i64(evcnt.p, evptr.p, nrows);
  }
  unsigned long long hst[ST_COUNT];
  int64_t n_events = 0;
  st.download(hst, ST_COUNT);
  if (I && I->binarized)
    KL_CUDA(cudaMemcpyAsync(&n_events, evptr.p + nrows, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx().stream));
  sync_stream();
  R->nnz = (int64_t)hst[ST_NNZ];

  // ---- stored rows ------------------------------------------------------------------------------------------------
  if (padded) {
    const int64_t stride = P.row_stride;
    R->row_stride = stride;
    R->col.alloc((size_t)(nrows * stride));
    if (P.vt == VAL_U32) R->val_u32.alloc((size_t)(nrows * stride));
    const uint32_t *val = P.vt == VAL_U32 ? P.val_u32.p : nullptr;
    uint32_t *oval = P.vt == VAL_U32 ? R->val_u32.p : nullptr;
    const unsigned grid = (unsigned)((nrows * 32 + 127) / 128);
    if (stride % 4 == 0)
      KL_LAUNCH(subset_padded<4>, grid, 128, 0, drows.p, nrows, stride, R->rowcnt.p, P.col.p, val, R->col.p, oval, st.p);
    else if (stride % 2 == 0)
      KL_LAUNCH(subset_padded<2>, grid, 128, 0, drows.p, nrows, stride, R->rowcnt.p, P.col.p, val, R->col.p, oval, st.p);
    else
      KL_LAUNCH(subset_padded<1>, grid, 128, 0, drows.p, nrows, stride, R->rowcnt.p, P.col.p, val, R->col.p, oval, st.p);
    KL_CUDA(cudaMemcpyAsync(hst + ST_MAXSQ, st.p + ST_MAXSQ, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost,
                            ctx().stream));
  } else {
    R->col.alloc((size_t)(R->nnz ? R->nnz : 1));
    if (P.vt == VAL_U32) {
      R->val_u32.alloc((size_t)(R->nnz ? R->nnz : 1));
      gather_compact<uint32_t>(P, *R, drows.p, P.val_u32.p, R->val_u32.p);
    } else if (P.vt == VAL_F64) {
      R->val_f64.alloc((size_t)(R->nnz ? R->nnz : 1));
      gather_compact<double>(P, *R, drows.p, P.val_f64.p, R->val_f64.p);
    } else {
      gather_compact<uint32_t>(P, *R, drows.p, (const uint32_t *)nullptr, (uint32_t *)nullptr);
    }
  }

  // ---- labels: the counts stay on the device until somebody asks (matrix_label_counts) ------------------------------
  if (P.has_labels) {
    KL_CUDA(cudaMemcpyAsync(R->label_ones.p, st.p + ST_ONES, sizeof(unsigned long long), cudaMemcpyDeviceToDevice,
                            ctx().stream));
    R->has_labels = true; R->counts_pending = true; R->counts_global = true;
  }

  // ---- matrix-free view: the parent's packed words, gathered row metadata -------------------------------------------
  if (I) {
    seqs->words = I->seqs->words ? I->seqs->words : I->seqs;
    seqs->max_len = (int64_t)hst[ST_MAXLEN];
    seqs->total_bases = (int64_t)hst[ST_BASES];
    seqs->total_blocks = seqs->words->total_blocks;
    imp->seqs = seqs;
    imp->M = I->M; imp->N = I->N; imp->op = I->op; imp->Mlo = I->Mlo;
    for (int k = 0; k < 16; k++) { imp->level_off[k] = I->level_off[k]; imp->fo[k] = I->fo[k]; }
    imp->num = I->num;
    if (I->binarized) {
      imp->binarized = true;
      imp->low_words = I->low_words;
      imp->lowcol.alloc(I->lowcol.n);
      KL_CUDA(cudaMemcpyAsync(imp->lowcol.p, I->lowcol.p, I->lowcol.bytes(), cudaMemcpyDeviceToDevice, ctx().stream));
      if (I->low_words) {
        imp->lowbits.alloc((size_t)(nrows * I->low_words));
        KL_LAUNCH(subset_words, (unsigned)((nrows * I->low_words + 255) / 256), 256, 0, drows.p, nrows, I->low_words,
                  I->lowbits.p, imp->lowbits.p);
      }
      imp->events.alloc((size_t)(n_events ? n_events : 1));
      KL_LAUNCH((subset_ranges<uint32_t>), (unsigned)((nrows * 32 + 127) / 128), 128, 0, drows.p, nrows, I->evptr.p,
                evptr.p, I->events.p, (const uint32_t *)nullptr, imp->events.p, (uint32_t *)nullptr);
      imp->evptr = std::move(evptr);
    }
    R->imp = imp;
  }
  sync_stream();
  if (padded) {
    double v[2];
    memcpy(v, hst + ST_MAXSQ, sizeof(v));
    R->has_local_stats = true;
    R->local_maxsq = v[0]; R->local_vmax = v[1];
  }
  return R;
}

}  // namespace kl
