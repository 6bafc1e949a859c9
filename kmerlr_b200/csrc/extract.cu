// extract.cu -- stage 1 of the hot path: sequences -> sparse k-mer count rows.
//
// Replaces scan_sequences + NewKmerCountsList/SetKmers + convert_counts_list
// (kmerLr_data.go:197-284,306-357; k-mer semantics of gonetics restated in SURVEY.md 8c).
//
// Design (one warp per sequence, no hash tables, no float atomics).  Sequences are 2-bit packed in
// HBM (+1 invalid bit per base, see SeqSet); every lane rolls the forward code and the image under
// the strand operation (revcomp / complement / reverse) over its stretch of positions, so the
// canonical code min(u, op(u)) of the k-mer starting at a position costs a shift and a min.  Levels:
//   * k <= 5   "table levels": forward counts of the deepest table level in a per-warp shared
//              memory table (one atomic per position), shallower levels are sums of 4 children; the
//              classes are walked through a precomputed list (code, image, id);
//   * k = 6, 7 "bitmap levels": one bit per canonical code in a per-warp shared memory bitmap
//              (4^k bits), set with atomicOr; the rare repeats go to a small list and are added to
//              the counts afterwards.  Walking the bitmap emits the row in code order.  Level 8 is a
//              bitmap level too when the rows are too long for the register sort;
//   * k >= 8   "sorted levels": per level ONE bitonic sort of the canonical codes in registers --
//              in-register compare-exchanges below distance E, warp shuffles above; a run of equal
//              keys is a class, its length the count.  Under revcomp with N <= 8 the keys are 16-bit,
//              two to a register (warp_sort16).
// Rows leave the kernel sorted by (k, code) = by final column index; columns are ranks in the
// bitmap of observed (or frozen) classes; observed classes are gathered per block in shared memory.
// Host sequences (kmerlr_extract) arrive in chunks on a copy stream while earlier chunks are
// packed and extracted.
#include <cmath>

#include "extract_kernel.cuh"

namespace kl {

namespace {

using namespace xk;

// ---- pack: ASCII -> 2 bit codes + invalid mask --------------------------------------------------
__global__ void pack_kernel(const uint8_t *__restrict__ seq, const int64_t *__restrict__ off,
                            const int64_t *__restrict__ blk, int64_t n, int64_t total_blocks, int64_t w0, int64_t w1,
                            uint32_t *__restrict__ bits2, uint16_t *__restrict__ inv16) {
  int64_t w = w0 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= w1) return;
  // sequence owning word w: the last i with blk[i] <= b, b = the 64-base block of w.  Start from the row a
  // set of equal-length sequences would give, gallop to a bracket, bisect inside it: a few probes (all in
  // L1) instead of log2(n) for every word.
  const int64_t b = w >> 2;
  int64_t g = (int64_t)((double)b * (double)n / (double)total_blocks);
  g = g < 0 ? 0 : (g > n - 1 ? n - 1 : g);
  int64_t lo, hi, stepw = 1;
  if (blk[g] <= b) {
    lo = g; hi = g + 1;
    while (hi < n && blk[hi] <= b) { lo = hi; stepw <<= 1; hi = hi + stepw < n ? hi + stepw : n; }
  } else {
    hi = g; lo = g - 1;
    while (lo > 0 && blk[lo] > b) { hi = lo; stepw <<= 1; lo = lo - stepw > 0 ? lo - stepw : 0; }
  }
  while (hi - lo > 1) {
    int64_t mid = (lo + hi) >> 1;
    if (blk[mid] <= b) lo = mid; else hi = mid;
  }
  int64_t i = lo, j0 = (w - blk[i] * 4) * 16, L = off[i + 1] - off[i];
  const uint8_t *s = seq + off[i];
  uint32_t bits = 0, inv = 0;
#pragma unroll
  for (int j = 0; j < 16; j++) {
    if (j0 + j < L) {
      uint32_t ch = s[j0 + j] | 0x20u, c;   // fold case
      if (ch == 'a') c = 0; else if (ch == 'c') c = 1; else if (ch == 'g') c = 2; else if (ch == 't') c = 3;
      else { c = 0; inv |= 1u << j; }
      bits |= c << (2 * j);
    }
  }
  bits2[w] = bits;
  inv16[w] = (uint16_t)inv;
}

// ---- bitmap helpers -------------------------------------------------------------------------------
__global__ void popc_words(const uint32_t *__restrict__ bm, int64_t nw, uint32_t *__restrict__ out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nw) out[i] = __popc(bm[i]);
}
// sharded extraction: ONE exchange.  Every rank contributes [bitmap words | rows | max row norm | max value];
// the merge ORs the bitmaps, adds the row counts and takes the maxima of the statistics.
__global__ void pack_exchange(const uint32_t *__restrict__ bm, int64_t nw, unsigned long long n_local,
                              const unsigned long long *__restrict__ stats, uint32_t *__restrict__ out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nw) out[i] = bm[i];
  if (i == 0) {
    unsigned long long v[3] = {n_local, stats[0], stats[1]};
    for (int k = 0; k < 3; k++) { out[nw + 2 * k] = (uint32_t)v[k]; out[nw + 2 * k + 1] = (uint32_t)(v[k] >> 32); }
  }
}
__global__ void merge_exchange(const uint32_t *__restrict__ all, int world, int64_t nw, uint32_t *__restrict__ bm,
                               unsigned long long *__restrict__ res) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t per = nw + 6;
  if (i < nw) {
    uint32_t v = 0;
    for (int r = 0; r < world; r++) v |= all[(int64_t)r * per + i];
    bm[i] = v;
  }
  if (i == 0) {
    unsigned long long n = 0, a = 0, b = 0;
    for (int r = 0; r < world; r++) {
      const uint32_t *t = all + (int64_t)r * per + nw;
      n += (unsigned long long)t[0] | ((unsigned long long)t[1] << 32);
      const unsigned long long x = (unsigned long long)t[2] | ((unsigned long long)t[3] << 32);
      const unsigned long long y = (unsigned long long)t[4] | ((unsigned long long)t[5] << 32);
      a = x > a ? x : a; b = y > b ? y : b;
    }
    res[0] = n; res[1] = a; res[2] = b;
  }
}
// ids of the set bits at their rank positions
__global__ void enumerate_bits(const uint32_t *__restrict__ bm, const uint32_t *__restrict__ rank, int64_t nw,
                               uint32_t *__restrict__ ids) {
  int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= nw) return;
  uint32_t v = bm[w], r = rank[w];
  while (v) {
    int b = __ffs(v) - 1;
    ids[r++] = (uint32_t)(w * 32 + b);
    v &= v - 1;
  }
}

// ---- numbering set helpers --------------------------------------------------------------------------
struct LevelInfo {
  int M, N, op;
  uint32_t level_off[16];
};
// every class the configuration can produce: the codes u <= image(u) of every level
__global__ void all_classes_bits(const LevelInfo I, uint32_t *__restrict__ bm, int64_t nw) {
  int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= nw) return;
  const uint32_t id0 = (uint32_t)(w * 32);
  int k = I.M;
  while (k < I.N && id0 >= I.level_off[k + 1]) k++;
  const uint32_t u0 = id0 - I.level_off[k], nk = 1u << (2 * k);   // levels start on multiples of 32
  uint32_t v = 0;
  for (int b = 0; b < 32; b++) {
    const uint32_t u = u0 + b;
    if (u < nk && (I.op == 0 || u <= kmer_op(u, k, I.op))) v |= 1u << b;
  }
  bm[w] = v;
}
__global__ void interleave_numbering(const uint32_t *__restrict__ bits, const uint32_t *__restrict__ rank, int64_t nw,
                                     uint2 *__restrict__ out) {
  int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w < nw) out[w] = make_uint2(bits[w], rank[w]);
}
// after the extraction kernel: tot[0] += the stored entries (sum of the row counts), tot[3] = 1 if the observed
// classes a differ from the numbering set b (b == nullptr: no check)
__global__ void extract_totals(const uint32_t *__restrict__ rowcnt, int64_t n, const uint32_t *__restrict__ a,
                               const uint32_t *__restrict__ b, int64_t nw, unsigned long long *__restrict__ tot) {
  __shared__ unsigned long long sh;
  if (threadIdx.x == 0) sh = 0ull;
  __syncthreads();
  const int64_t stride = (int64_t)gridDim.x * blockDim.x, i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long s = 0ull;
  for (int64_t i = i0; i < n; i += stride) s += rowcnt[i];
  if (b)
    for (int64_t w = i0; w < nw; w += stride)
      if (a[w] != b[w]) tot[3] = 1ull;
  if (s) atomicAdd(&sh, s);
  __syncthreads();
  if (threadIdx.x == 0 && sh) atomicAdd(tot, sh);
}
// columns numbered in the numbering set -> ranks among the observed classes, in place (warp per row)
__global__ void renumber_rows(uint32_t *__restrict__ col, const uint32_t *__restrict__ rowcnt, int64_t stride, int64_t n,
                              const uint32_t *__restrict__ ids, const uint32_t *__restrict__ bm,
                              const uint32_t *__restrict__ rank, const uint32_t *__restrict__ rowdup) {
  int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= n) return;
  const unsigned lane = lane_id();
  uint32_t *c = col + row * stride;
  const uint32_t cnt = rowcnt[row];
  for (uint32_t j = lane; j < cnt; j += 32) {
    const uint32_t id = __ldg(ids + c[j]), w = __ldg(bm + (id >> 5));
    c[j] = __ldg(rank + (id >> 5)) + __popc(w & ((1u << (id & 31)) - 1u));
  }
  // repeat events of binarized rows (columns too), stored downwards from the row's last slot
  const uint32_t nd = rowdup ? rowdup[row] : 0u;
  uint32_t *t = c + stride - 1;
  for (uint32_t j = lane; j < nd; j += 32) {
    const uint32_t id = __ldg(ids + t[-(int64_t)j]), w = __ldg(bm + (id >> 5));
    t[-(int64_t)j] = __ldg(rank + (id >> 5)) + __popc(w & ((1u << (id & 31)) - 1u));
  }
}
// repeat events of binarized rows: from the tail of each row's slots into one compact array (the row layout
// may be compacted away later, the matrix-free logistic pass keeps its own copy)
__global__ void gather_events(const uint32_t *__restrict__ col, int64_t stride, int64_t n,
                              const int64_t *__restrict__ evptr, uint32_t *__restrict__ events) {
  int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= n) return;
  const unsigned lane = lane_id();
  const int64_t a = evptr[row], cnt = evptr[row + 1] - a;
  const uint32_t *t = col + (row + 1) * stride - 1;
  for (int64_t j = lane; j < cnt; j += 32) events[a + j] = t[-j];
}
// column of every class of the table levels (flat list tl), NOCOL when the class is not numbered
__global__ void low_columns(const uint2 *__restrict__ tl, uint32_t tl_cnt, int slots, const uint32_t *__restrict__ bm,
                            const uint32_t *__restrict__ rank, uint32_t *__restrict__ lowcol) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= slots) return;
  uint32_t col = NOCOL;
  if ((uint32_t)j < tl_cnt) {
    const uint32_t id = tl[j].y, w = bm[id >> 5], bit = 1u << (id & 31);
    if (w & bit) col = rank[id >> 5] + __popc(w & (bit - 1u));
  }
  lowcol[j] = col;
}

// ---- explicit feature lists: singles and pair products (convert_counts, kmerLr_data.go:210-229) ----
__device__ __forceinline__ uint32_t row_lookup(const uint32_t *col, const uint32_t *val, int64_t a, int64_t b, uint32_t c) {
  int64_t lo = a, hi = b;
  while (lo < hi) {
    int64_t mid = (lo + hi) >> 1;
    if (col[mid] < c) lo = mid + 1; else hi = mid;
  }
  if (lo < b && col[lo] == c) return val ? val[lo] : 1u;
  return 0u;
}
template <bool WRITE>
__global__ void features_rows(const Rows R, const uint32_t *__restrict__ col,
                              const uint32_t *__restrict__ val, int64_t n, const int32_t *__restrict__ feat,
                              int64_t nf, uint32_t *__restrict__ cnt_out, const int64_t *__restrict__ orowptr,
                              uint32_t *__restrict__ ocol, uint32_t *__restrict__ oval) {
  int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= n) return;
  unsigned lane = lane_id();
  int64_t a, b;
  R.range(row, a, b);
  int64_t outp = WRITE ? orowptr[row] : 0;
  uint32_t tot = 0;
  for (int64_t j0 = 0; j0 < nf; j0 += 32) {
    int64_t j = j0 + lane;
    uint32_t v = 0;
    if (j < nf) {
      int32_t i1 = feat[2 * j], i2 = feat[2 * j + 1];
      uint32_t c1 = row_lookup(col, val, a, b, (uint32_t)i1);
      if (i1 == i2) v = c1;
      else if (c1) v = c1 * row_lookup(col, val, a, b, (uint32_t)i2);
    }
    unsigned km = __ballot_sync(0xffffffffu, v != 0);
    if (WRITE && v != 0) {
      int64_t pos = outp + __popc(km & lanemask_lt());
      ocol[pos] = (uint32_t)j;
      if (oval) oval[pos] = v;
    }
    outp += __popc(km);
    tot += __popc(km);
  }
  if (!WRITE && lane == 0) cnt_out[row] = tot;
}

// the classes of the table levels [t_lo, t_hi] in (k, code) order: table index of the code, table
// index of its image under the strand operation (the same index when the code is its own image), id
const uint2 *table_classes(int op, int t_lo, int t_hi, const uint32_t *level_off, uint32_t *count) {
  struct Entry { int op, lo, hi; uint32_t off0; DevBuf<uint2> dev; uint32_t cnt; };
  static std::vector<std::unique_ptr<Entry>> cache;
  for (auto &e : cache)
    if (e->op == op && e->lo == t_lo && e->hi == t_hi && e->off0 == level_off[t_lo]) { *count = e->cnt; return e->dev.p; }
  std::vector<uint2> list;
  for (int k = t_lo; k <= t_hi; k++) {
    const uint32_t toff = ((1u << (2 * k)) - 4u) / 3u;
    for (uint32_t u = 0; u < (1u << (2 * k)); u++) {
      uint32_t r = u;
      if (op) {
        r = 0;
        for (int i = 0; i < k; i++) {
          uint32_t d = (u >> (2 * i)) & 3u;               // digit i from the right
          if (op == 1) r |= (3u - d) << (2 * (k - 1 - i));
          else if (op == 2) r |= (3u - d) << (2 * i);
          else r |= d << (2 * (k - 1 - i));
        }
      }
      // BYTE offsets of the two 16-bit counters inside the warp's table (word index swizzled as the kernel does,
      // xk::sw); a code that is its own image gets a counter of the padding (always 0) as its second one
      auto pos = [](uint32_t i) { return (sw(i >> 1) << 2) | ((i & 1u) << 1); };
      const uint32_t zero_slot = 2u * TAB_WORDS - 2u;
      if (u <= r) list.push_back(make_uint2(pos(toff + u) | (pos(u == r ? zero_slot : toff + r) << 16), level_off[k] + u));
    }
  }
  auto e = std::make_unique<Entry>();
  e->op = op; e->lo = t_lo; e->hi = t_hi; e->off0 = level_off[t_lo]; e->cnt = (uint32_t)list.size();
  e->dev.alloc(list.size());
  e->dev.upload(list.data(), list.size());
  sync_stream();
  *count = e->cnt;
  cache.push_back(std::move(e));
  return cache.back()->dev.p;
}

}  // namespace

// Per-sequence metadata on the device from ONE upload of the caller's offsets: len[i], and blk = the
// exclusive scan of ceil(len / 64).
static __global__ void seq_meta_kernel(const int64_t *__restrict__ off, int64_t n, int64_t *__restrict__ len,
                                uint32_t *__restrict__ nblk) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int64_t l = off[i + 1] - off[i];
  len[i] = l;
  nblk[i] = (uint32_t)((l + 63) >> 6);
}

// Host sequences feeding an extraction: the ASCII bytes go to the device in chunks on the copy stream
// while the previous chunk is packed and extracted on the main stream.  The host keeps only the chunk
// boundaries (rows, 64-base blocks, bytes); the per-sequence arrays are derived on the device.
struct HostFeed {
  const uint8_t *seq = nullptr;   // base 0 of the caller's buffer (offsets are absolute)
  int nchunks = 1;
  int64_t row[CTX_COPY_EVENTS] = {0}, blk[CTX_COPY_EVENTS] = {0}, byte[CTX_COPY_EVENTS] = {0};
  // Chunk sizes grow geometrically: the first kernel starts after a short copy, and the copy of chunk c+1
  // must end before the extraction of chunk c does, or the GPU idles.  At C2 the extraction (+ pack) of a
  // chunk takes 1.45 x its copy time (2.8 ms vs 1.9 ms for the whole set), so the growth factor has to
  // stay below that: 1.35 (doubling sizes left the GPU waiting at every chunk: 3.9 ms vs 3.4 ms).
  static int64_t cut(int64_t n, int c, int nchunks) {
    if (c <= 0) return 0;
    if (c >= nchunks) return n;
    const double g = 0.01 * (double)ctx().feed_growth;      // kmerlr_option("feed_growth"), per cent
    if (g <= 1.0001) return n * c / nchunks;
    return (int64_t)((double)n * (pow(g, c) - 1.0) / (pow(g, nchunks) - 1.0));
  }
  DevBuf<uint8_t> raw;            // bytes [byte[0], byte[nchunks])
  DevBuf<int64_t> doff;           // the caller's offsets
  // copy the bases of chunk c (every chunk for c < 0) and pack them (main stream waits for the copy)
  void feed(SeqSet &s, int c) {
    const int c0 = c < 0 ? 0 : c, c1 = c < 0 ? nchunks : c + 1;
    const int64_t b0 = byte[c0], b1 = byte[c1];
    if (b1 > b0) {
      KL_CUDA(cudaMemcpyAsync(raw.p + (b0 - byte[0]), seq + b0, (size_t)(b1 - b0), cudaMemcpyHostToDevice,
                              ctx().copy_stream));
      KL_CUDA(cudaEventRecord(ctx().copy_ev[c0], ctx().copy_stream));
      KL_CUDA(cudaStreamWaitEvent(ctx().stream, ctx().copy_ev[c0], 0));
    }
    const int64_t w0 = blk[c0] * 4, w1 = blk[c1] * 4;
    if (w1 > w0)
      KL_LAUNCH(pack_kernel, (unsigned)((w1 - w0 + 255) / 256), 256, 0, raw.p - byte[0], doff.p, s.blk.p, s.n,
                s.total_blocks, w0, w1,
                s.bits2.p, s.inv16.p);
  }
};

// by_bytes: few long sequences (the contigs of a genome on their way to the window scoring) -- chunks of whole
// rows of about equal size in bytes instead of the growing row counts of a training set
static std::shared_ptr<SeqSet> sequences_begin(const uint8_t *seq, const int64_t *off, int64_t n, HostFeed &hf,
                                               bool by_bytes = false) {
  require_ready();
  KL_REQUIRE(n >= 0 && off != nullptr, "sequences: bad arguments");
  auto s = std::make_shared<SeqSet>();
  s->n = n;
  hf.seq = seq;
  int64_t cutrow[CTX_COPY_EVENTS + 1];
  if (by_bytes) {
    const int64_t total = off[n] - off[0], per = (int64_t)8 << 20;
    hf.nchunks = (int)(total / per < 1 ? 1 : (total / per > CTX_COPY_EVENTS - 1 ? CTX_COPY_EVENTS - 1 : total / per));
    if (hf.nchunks > n) hf.nchunks = n > 0 ? (int)n : 1;
    int64_t i = 0;
    for (int c = 0; c <= hf.nchunks; c++) {
      const int64_t want = c == hf.nchunks ? total : total / hf.nchunks * c;
      while (i < n && off[i] - off[0] < want) i++;
      cutrow[c] = c == hf.nchunks ? n : i;
    }
  } else {
    hf.nchunks = (int)(n / 8192 < 1 ? 1 : (n / 8192 > CTX_COPY_EVENTS - 1 ? CTX_COPY_EVENTS - 1 : n / 8192));
    for (int c = 0; c <= hf.nchunks; c++) cutrow[c] = HostFeed::cut(n, c, hf.nchunks);
  }
  Trace tr("feed");
  // one pass over the offsets: validation, longest sequence, block counts at the chunk boundaries
  int64_t blocks = 0, max_len = 0, min_len = 0;
  for (int c = 0; c < hf.nchunks; c++) {
    const int64_t r0 = cutrow[c], r1 = cutrow[c + 1];
    hf.row[c] = r0; hf.blk[c] = blocks; hf.byte[c] = off[r0];
    for (int64_t i = r0; i < r1; i++) {
      const int64_t l = off[i + 1] - off[i];
      max_len = l > max_len ? l : max_len;
      min_len = l < min_len ? l : min_len;
      blocks += (l + 63) >> 6;
    }
  }
  KL_REQUIRE(min_len >= 0, "sequences: offsets must be non-decreasing");
  hf.row[hf.nchunks] = n; hf.blk[hf.nchunks] = blocks; hf.byte[hf.nchunks] = off[n];
  s->max_len = max_len;
  s->total_bases = off[n] - off[0];
  s->total_blocks = blocks;
  tr.mark("host pass", false);
  hf.doff.alloc((size_t)n + 1);
  hf.doff.upload(off, (size_t)n + 1);
  s->len.alloc((size_t)(n ? n : 1));
  s->blk.alloc((size_t)n + 1);
  if (n > 0) {
    DevBuf<uint32_t> nblk((size_t)n);
    KL_LAUNCH(seq_meta_kernel, (unsigned)((n + 255) / 256), 256, 0, hf.doff.p, n, s->len.p, nblk.p);
    exclusive_scan_u32_to_i64(nblk.p, s->blk.p, n);
  } else {
    s->blk.zero();
  }
  const int64_t words = blocks * 4;
  s->bits2.alloc((size_t)words + 4);     // + 4: the kernels read up to two words past the last base
  s->inv16.alloc((size_t)words + 4);
  KL_CUDA(cudaMemsetAsync(s->bits2.p + words, 0, 4 * sizeof(uint32_t), ctx().stream));
  KL_CUDA(cudaMemsetAsync(s->inv16.p + words, 0, 4 * sizeof(uint16_t), ctx().stream));
  hf.raw.alloc((size_t)(s->total_bases ? s->total_bases : 1));
  // the copy stream must not run ahead of the allocation / earlier work on the main stream
  KL_CUDA(cudaEventRecord(ctx().copy_ev[CTX_COPY_EVENTS - 1], ctx().stream));
  KL_CUDA(cudaStreamWaitEvent(ctx().copy_stream, ctx().copy_ev[CTX_COPY_EVENTS - 1], 0));
  tr.mark("offsets, metadata");
  return s;
}

// host sequences arriving in chunks of whole rows, for a consumer that works chunk by chunk (score.cu)
namespace {
struct FeedImpl : SeqFeed {
  HostFeed hf;
  std::shared_ptr<SeqSet> s;
  int chunks() const override { return hf.nchunks; }
  int64_t first_row(int c) const override { return hf.row[c]; }
  void feed(int c) override { if (s->n > 0) hf.feed(*s, c); }
};
}  // namespace

std::shared_ptr<SeqSet> sequences_begin_chunked(const uint8_t *seq, const int64_t *off, int64_t n, std::unique_ptr<SeqFeed> &feed) {
  auto f = std::make_unique<FeedImpl>();
  f->s = sequences_begin(seq, off, n, f->hf, true);
  auto s = f->s;
  feed = std::move(f);
  return s;
}

std::shared_ptr<SeqSet> sequences_create(const uint8_t *seq, const int64_t *off, int64_t n) {
  HostFeed hf;
  auto s = sequences_begin(seq, off, n, hf);
  if (n > 0) hf.feed(*s, -1);
  sync_stream();
  return s;
}

static std::shared_ptr<Matrix> apply_features(Matrix &cls, const int32_t *features, int64_t nf) {
  for (int64_t j = 0; j < nf; j++) {
    KL_REQUIRE(features[2 * j] >= 0 && features[2 * j] < cls.m && features[2 * j + 1] >= 0 && features[2 * j + 1] < cls.m,
               "features: class index out of range");
  }
  auto out = std::make_shared<Matrix>();
  out->n = cls.n; out->m = nf; out->vt = cls.vt;
  matrix_class_list(cls);
  out->class_k = cls.class_k; out->class_code = cls.class_code; out->n_classes = cls.n_classes;
  out->sharded = cls.sharded; out->n_global = cls.n_global;
  DevBuf<int32_t> dfeat((size_t)(2 * nf));
  dfeat.upload(features, (size_t)(2 * nf));
  DevBuf<uint32_t> cnt((size_t)(cls.n ? cls.n : 1));
  const uint32_t *val = cls.vt == VAL_U32 ? cls.val_u32.p : nullptr;
  unsigned grid = (unsigned)((cls.n * 32 + 127) / 128);
  out->rowptr.alloc((size_t)cls.n + 1);
  if (cls.n > 0) {
    KL_LAUNCH((features_rows<false>), grid, 128, 0, cls.rows(), cls.col.p, val, cls.n, dfeat.p, nf, cnt.p, nullptr,
              nullptr, nullptr);
    exclusive_scan_u32_to_i64(cnt.p, out->rowptr.p, cls.n);
    KL_CUDA(cudaMemcpyAsync(&out->nnz, out->rowptr.p + cls.n, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx().stream));
    sync_stream();
  } else {
    out->rowptr.zero(); out->nnz = 0;
  }
  out->col.alloc((size_t)(out->nnz ? out->nnz : 1));
  if (out->vt == VAL_U32) out->val_u32.alloc((size_t)(out->nnz ? out->nnz : 1));
  if (cls.n > 0)
    KL_LAUNCH((features_rows<true>), grid, 128, 0, cls.rows(), cls.col.p, val, cls.n, dfeat.p, nf, nullptr,
              out->rowptr.p, out->col.p, out->vt == VAL_U32 ? out->val_u32.p : nullptr);
  sync_stream();
  return out;
}

// rank, count and interleaved words of a numbering set whose bits are in place
static void number_set(Numbering &S) {
  const int64_t nw = S.nw;
  DevBuf<uint32_t> pc((size_t)nw);
  KL_LAUNCH(popc_words, (unsigned)((nw + 255) / 256), 256, 0, S.bits.p, nw, pc.p);
  exclusive_scan_u32(pc.p, S.rank.p, nw);
  S.nbx.alloc((size_t)nw);
  KL_LAUNCH(interleave_numbering, (unsigned)((nw + 255) / 256), 256, 0, S.bits.p, S.rank.p, nw, S.nbx.p);
}

// every class the configuration can produce, built once per (M, N, strand op) and kept by the context
static std::shared_ptr<const Numbering> numbering_all(const LevelInfo &LI, int64_t nw) {
  for (auto &s : ctx().numbering)
    if (s->M == LI.M && s->N == LI.N && s->op == LI.op) return s;
  auto S = std::make_shared<Numbering>();
  S->M = LI.M; S->N = LI.N; S->op = LI.op; S->nw = nw;
  S->bits.alloc((size_t)nw); S->rank.alloc((size_t)nw + 1);
  KL_LAUNCH(all_classes_bits, (unsigned)((nw + 255) / 256), 256, 0, LI, S->bits.p, nw);
  number_set(*S);
  KL_CUDA(cudaMemcpyAsync(&S->count, S->rank.p + nw, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx().stream));
  sync_stream();
  ctx().numbering.push_back(S);
  return S;
}

static std::shared_ptr<Matrix> extract_impl(const kmerlr_config &cfg, std::shared_ptr<SeqSet> seqs,
                                            const int32_t *frozen_k, const uint64_t *frozen_code, int64_t n_frozen,
                                            const int32_t *features, int64_t n_features, int flags, HostFeed *feed) {
  require_ready();
  const SeqSet &s = *seqs;
  KL_REQUIRE(cfg.alphabet == 0 || cfg.alphabet == 1, "alphabet: 0 = nucleotide, 1 = gapped nucleotide (IUPAC is not implemented)");
  if (cfg.alphabet == 1) {
    // gapped alphabet: the sort-based path of gapped.cu (needs the whole set packed)
    KL_REQUIRE(n_features == 0 || n_frozen > 0, "an explicit feature list needs a frozen class list");
    if (feed && s.n > 0) feed->feed(*seqs, -1);
    auto g = extract_gapped(cfg, seqs, frozen_k, frozen_code, n_frozen, flags);
    if (n_features > 0) return apply_features(*g, features, n_features);
    return g;
  }
  KL_REQUIRE(cfg.M >= 1 && cfg.M <= cfg.N, "need 1 <= M <= N");
  KL_REQUIRE(n_features == 0 || n_frozen > 0, "an explicit feature list needs a frozen class list");
  {
    // What the warp-per-row kernel does not take goes through the sort-based path of gapped.cu (not tuned):
    // several strand flags at once, k-mers of 14 bases, k > 8 on rows too long for the register sort.
    const int nops = (cfg.complement != 0) + (cfg.reverse != 0) + (cfg.revcomp != 0);
    const bool long_sorted = cfg.N > KB_MAX && (s.max_len + 31) / 32 > 64;
    const bool long_tables = s.max_len >= 65536 && cfg.M <= KT_MAX;      // (16-bit count tables)
    if (nops > 1 || cfg.N > MAX_N || long_sorted || long_tables) {
      if (feed && s.n > 0) feed->feed(*seqs, -1);
      auto g = extract_gapped(cfg, seqs, frozen_k, frozen_code, n_frozen, flags);
      if (n_features > 0) return apply_features(*g, features, n_features);
      return g;
    }
  }
  const bool sharded = (flags & KMERLR_FLAG_SHARDED) != 0 && ctx().world > 1;

  XParams P{};
  P.M = cfg.M; P.N = cfg.N; P.binarize = cfg.binarize != 0;
  P.op = cfg.revcomp ? 1 : (cfg.complement ? 2 : (cfg.reverse ? 3 : 0));
  P.t_lo = cfg.M; P.t_hi = cfg.N < KT_MAX ? cfg.N : KT_MAX;
  // levels above the tables: per-row bitmaps up to level 7, a register sort per level above that;
  // rows too long for the register sort (more than 64 positions per lane) keep level 8 on a bitmap
  const int64_t steps = (s.max_len + 31) / 32;           // start positions per lane
  const int kb = steps > 64 ? KB_MAX : KB_DEFAULT;
  P.b_lo = cfg.M > KT_MAX + 1 ? cfg.M : KT_MAX + 1; P.b_hi = cfg.N < kb ? cfg.N : kb;
  P.s_lo = cfg.M > kb + 1 ? cfg.M : kb + 1;
  P.n = s.n;
  P.len = s.len.p; P.blk = s.blk.p; P.bits2 = s.bits2.p; P.inv16 = s.inv16.p;
  // dense class ids: every level starts on a multiple of 32 so that bitmap words never straddle levels
  uint64_t dense = 0;
  for (int k = cfg.M; k <= cfg.N; k++) {
    P.level_off[k] = (uint32_t)dense;
    dense += ((1ull << (2 * k)) + 31) / 32 * 32;
  }
  P.level_off[cfg.N + 1] = (uint32_t)dense;
  const int64_t nbits = (int64_t)dense, nw = (nbits + 31) / 32;
  // row stride of the matrix: upper bound on the distinct classes of one sequence
  int64_t stride = 0;
  for (int k = cfg.M; k <= cfg.N; k++) {
    int64_t inst = s.max_len - k + 1; if (inst < 0) inst = 0;
    int64_t cls = (int64_t)1 << (2 * k);
    stride += inst < cls ? inst : cls;
  }
  if (stride < 1) stride = 1;
  P.stride = stride;
  // Binarized rows keep what the matrix-free logistic pass needs (Implicit): the class bitmap of the table
  // levels and one event per repeat of a class of the levels above them.  The events sit in the unused tail
  // of the row's slots: for a level whose stride term is its number of instances, entries + events = instances.
  bool hybrid = P.binarize && cfg.N <= IMP_MAX_N && n_features == 0 && s.n > 0;
  for (int k = cfg.M > KT_MAX + 1 ? cfg.M : KT_MAX + 1; k <= cfg.N && hybrid; k++)
    if (s.max_len - k + 1 > ((int64_t)1 << (2 * k))) hybrid = false;
  KL_INVARIANT(s.max_len < 65536 || P.t_lo > P.t_hi);
  KL_REQUIRE(s.max_len < ((int64_t)1 << 30), "sequence too long");
  // keys per lane of the register sort
  int E = 0;
  if (P.s_lo <= cfg.N) {
    E = 2; while (E < steps && E < 128) E <<= 1;
    KL_INVARIANT(E <= 64);        // (longer rows went to the sort-based path above)
  }
  // per-warp shared memory
  P.bm_words = 0; P.pf_words = 0;
  int nbl = 0;
  for (int k = P.b_lo; k <= P.b_hi; k++) {
    P.bm_off[k] = (uint32_t)P.bm_words; P.pf_off[k] = (uint32_t)P.pf_words;
    P.bm_words += 1 << (2 * k - 5); P.pf_words += 1 << (2 * k - 7);
    nbl++;
  }
  P.pf_words = (P.pf_words + 3) / 4 * 4;
  P.ts_words = 32 * E > TAB_WORDS ? 32 * E : TAB_WORDS;
  P.warp_words = P.bm_words + P.pf_words + P.ts_words + 8;     // + repeat count, ticket, row slots of the bitmap levels
  P.warp_words = (P.warp_words + 3) / 4 * 4;
  // the block's bitmap of observed classes covers the levels up to OBS_MAX_LEVEL
  {
    int top = cfg.N < OBS_MAX_LEVEL ? cfg.N : OBS_MAX_LEVEL;
    P.obs_id_words = top >= cfg.M ? (int)(P.level_off[top + 1] / 32) : 0;
    P.obs_id_words = (P.obs_id_words + 3) / 4 * 4;
  }
  // classes of the table levels (their marks sit behind the marks by class id, one bit per list entry)
  if (P.t_lo <= P.t_hi) P.tl = table_classes(P.op, P.t_lo, P.t_hi, P.level_off, &P.tl_cnt);
  P.obs_words = P.obs_id_words + (P.t_lo <= P.t_hi ? (int)((P.tl_cnt + 127) / 128 * 4) : 0);
  Trace tr("extract");
  auto out = std::make_shared<Matrix>();
  out->n = s.n; out->vt = P.binarize ? VAL_ONE : VAL_U32;
  out->sharded = sharded; out->n_global = s.n;
  // the kernel writes the rows of the matrix itself: fixed stride, final column numbers
  out->row_stride = stride;
  out->col.alloc((size_t)(s.n ? s.n * stride : 1));
  if (!P.binarize) out->val_u32.alloc((size_t)(s.n ? s.n * stride : 1));
  out->rowcnt.alloc((size_t)(s.n ? s.n : 1));
  DevBuf<uint32_t> dummy_cnt(1);
  // numbering set: the frozen list, or every class the configuration can produce (then the columns
  // are final unless some class never shows up, see below)
  DevBuf<uint32_t> bitmap((size_t)nw);
  std::vector<uint32_t> frozen_bits;       // host image of the frozen class set (alive until the next sync)
  LevelInfo LI{};
  LI.M = cfg.M; LI.N = cfg.N; LI.op = P.op;
  for (int k = cfg.M; k <= cfg.N + 1; k++) LI.level_off[k] = P.level_off[k];
  std::shared_ptr<const Numbering> num;
  if (n_frozen > 0) {
    frozen_bits.assign((size_t)nw, 0u);
    uint64_t prev = 0;
    for (int64_t j = 0; j < n_frozen; j++) {
      int k = frozen_k[j];
      KL_REQUIRE(k >= cfg.M && k <= cfg.N && frozen_code[j] < (1ull << (2 * k)), "frozen class outside [M,N]");
      uint64_t id = (uint64_t)P.level_off[k] + frozen_code[j];
      KL_REQUIRE(j == 0 || id > prev, "frozen class list must be sorted by (k, code) without duplicates");
      prev = id;
      frozen_bits[id >> 5] |= 1u << (id & 31);
    }
    auto F = std::make_shared<Numbering>();
    F->M = cfg.M; F->N = cfg.N; F->op = P.op; F->nw = nw; F->count = (uint32_t)n_frozen;
    F->bits.alloc((size_t)nw); F->rank.alloc((size_t)nw + 1);
    F->bits.upload(frozen_bits.data(), (size_t)nw);
    number_set(*F);
    num = F;
  } else {
    num = numbering_all(LI, nw);
  }
  // one zeroed block for everything the host reads after the kernel: [0] stored entries, [1, 2] row statistics,
  // [3] "observed classes differ from the numbering set", [4] repeat events, [6, 9) the sharded exchange's totals
  DevBuf<unsigned long long> tot(9);
  tot.zero();
  bitmap.zero();
  DevBuf<uint32_t> full(1);                 // "every class has been observed" (set by the kernel, ends the marks)
  full.zero();
  P.full = full.p; P.nb_words = nw;
  P.st_id = out->col.p; P.st_cnt = P.binarize ? dummy_cnt.p : out->val_u32.p; P.rowcnt = out->rowcnt.p;
  P.bitmap = bitmap.p; P.nbx = num->nbx.p; P.filter = n_frozen > 0; P.stats = tot.p + 1;
  P.mark = n_frozen == 0;
  DevBuf<uint32_t> lowbits, rowdup;
  if (hybrid) {
    P.events = 1;
    P.low_words = P.t_lo <= P.t_hi ? (int)((P.tl_cnt + 31) / 32) : 0;
    if (P.low_words) { lowbits.alloc((size_t)s.n * P.low_words); P.lowbits = lowbits.p; }
    rowdup.alloc((size_t)s.n);
    P.rowdup = rowdup.p;
  }
  // repeats of the bitmap levels: one list per warp in global memory (L2 resident)
  DevBuf<uint32_t> ovf;
  P.ovf_stride = nbl * (s.max_len > 0 ? s.max_len : 1);
  if (nbl && (!P.binarize || hybrid) && s.n > 0) {
    ovf.alloc((size_t)ctx().sm_count * 64 * (size_t)P.ovf_stride);
    P.ovf = ovf.p;
  }
  tr.mark("alloc");

  if (s.n > 0) {
    // host sequences arrive in chunks: copy of chunk c+1 overlaps pack + extraction of chunk c
    const int nchunks = feed ? feed->nchunks : 1;
    DevBuf<uint32_t> ticket((size_t)nchunks);     // next group of rows of each launch
    ticket.zero();
    // A chunk's kernel ends with a tail of about one row time (64 us at C2) in which the SMs run dry.  Odd
    // chunks therefore run on a second stream: their blocks move in as the blocks of the chunk before
    // them leave.  Two kernels can then be in flight, each with its own lists of repeats.
    const bool two_streams = feed && nchunks > 1;
    DevBuf<uint32_t> ovf2;
    if (two_streams && P.ovf) ovf2.alloc((size_t)ctx().sm_count * 64 * (size_t)P.ovf_stride);
    struct StreamSwap {            // launches go to ctx().stream: point it at the chunk's stream for a while
      cudaStream_t saved;
      explicit StreamSwap(cudaStream_t run) : saved(ctx().stream) { ctx().stream = run; }
      ~StreamSwap() { ctx().stream = saved; }
    };
    if (two_streams) {
      KL_CUDA(cudaEventRecord(ctx().join_ev[0], ctx().stream));
      KL_CUDA(cudaStreamWaitEvent(ctx().alt_stream, ctx().join_ev[0], 0));
    }
    uint32_t *const ovf_even = P.ovf;
    for (int c = 0; c < nchunks; c++) {
      StreamSwap on((two_streams && (c & 1)) ? ctx().alt_stream : ctx().stream);
      P.ovf = (two_streams && (c & 1) && ovf_even) ? ovf2.p : ovf_even;
      P.ticket = ticket.p + c;
      const int64_t r0 = feed ? feed->row[c] : 0, r1 = feed ? feed->row[c + 1] : s.n;
      if (feed) feed->feed(*seqs, c);
      P.row0 = r0; P.n = r1;
      switch (E) {
        case 0: launch_extract<0>(P); break;
        case 2: launch_extract<2>(P); break;
        case 4: launch_extract<4>(P); break;
        case 8: launch_extract<8>(P); break;
        case 16: launch_extract<16>(P); break;
        case 32: launch_extract<32>(P); break;
        default: launch_extract<64>(P); break;
      }
    }
    P.ovf = ovf_even;
    if (two_streams) {
      KL_CUDA(cudaEventRecord(ctx().join_ev[1], ctx().alt_stream));
      KL_CUDA(cudaStreamWaitEvent(ctx().stream, ctx().join_ev[1], 0));
    }
    P.row0 = 0; P.n = s.n;
  }
  tr.mark("extract_kernel");
  // observed classes, row count and row statistics of all ranks in ONE exchange; do the classes cover the
  // numbering set?
  unsigned long long *const gres = tot.p + 6;
  if (sharded) {
    const int64_t xw = n_frozen == 0 ? nw : 0, per = xw + 6;
    DevBuf<uint32_t> mine((size_t)per), all((size_t)(per * ctx().world));
    KL_LAUNCH(pack_exchange, (unsigned)((xw + 256) / 256), 256, 0, bitmap.p, xw, (unsigned long long)s.n, tot.p + 1, mine.p);
    comm_allgather_bytes(mine.p, all.p, per * 4);
    KL_LAUNCH(merge_exchange, (unsigned)((xw + 256) / 256), 256, 0, all.p, ctx().world, xw, bitmap.p, gres);
  }
  {
    int64_t blocks = ((s.n > nw ? s.n : nw) + 255) / 256;
    if (blocks > 4 * ctx().sm_count) blocks = 4 * ctx().sm_count;
    KL_LAUNCH(extract_totals, (unsigned)(blocks ? blocks : 1), 256, 0, out->rowcnt.p, s.n, bitmap.p,
              n_frozen == 0 ? num->bits.p : (const uint32_t *)nullptr, nw, tot.p);
  }
  DevBuf<int64_t> evptr;
  if (hybrid) {
    evptr.alloc((size_t)s.n + 1);
    exclusive_scan_u32_to_i64(rowdup.p, evptr.p, s.n);
    KL_CUDA(cudaMemcpyAsync(tot.p + 4, evptr.p + s.n, sizeof(int64_t), cudaMemcpyDeviceToDevice, ctx().stream));
  }
  // the class list of the numbering set goes out before the one round trip (a renumbering below redoes it)
  uint32_t m32 = num->count;
  out->class_ids.alloc((size_t)(m32 ? m32 : 1));
  KL_LAUNCH(enumerate_bits, (unsigned)((nw + 255) / 256), 256, 0, num->bits.p, num->rank.p, nw, out->class_ids.p);
  // one round trip: stored entries, "columns are final", row statistics, repeat events, global number of rows
  unsigned long long *htot = (unsigned long long *)host_staging(9 * sizeof(unsigned long long));
  tot.download(htot, 9);
  host_staging_done();
  sync_stream();
  out->nnz = (int64_t)htot[0];
  const unsigned long long hstats[2] = {htot[1], htot[2]}, hres[3] = {htot[6], htot[7], htot[8]};
  const bool hdiffer = htot[3] != 0;
  const int64_t n_events = (int64_t)htot[4];
  int64_t nn = s.n;
  if (sharded) {
    // the statistics are global already: no collective later (step size, fixed-point scale)
    nn = (int64_t)hres[0];
    out->maxsq = (double)hres[1]; out->vmax = (double)hres[2];
    out->has_maxsq = out->has_vmax = true;
  }
  out->n_global = nn;
  out->has_local_stats = true;
  out->local_maxsq = (double)hstats[0]; out->local_vmax = (double)hstats[1];
  tr.mark("sizes");
  if (hdiffer) {
    // some class of the configuration never occurs: the columns are the ranks among the OBSERVED
    // classes (kmerLr_data.go:316-324), renumber the stored columns in place
    auto obs = std::make_shared<Numbering>();
    obs->M = cfg.M; obs->N = cfg.N; obs->op = P.op; obs->nw = nw;
    obs->rank.alloc((size_t)nw + 1);
    {
      DevBuf<uint32_t> pc((size_t)nw);
      KL_LAUNCH(popc_words, (unsigned)((nw + 255) / 256), 256, 0, bitmap.p, nw, pc.p);
      exclusive_scan_u32(pc.p, obs->rank.p, nw);
    }
    if (s.n > 0)
      KL_LAUNCH(renumber_rows, (unsigned)((s.n * 32 + 127) / 128), 128, 0, out->col.p, out->rowcnt.p, stride, s.n,
                out->class_ids.p, bitmap.p, obs->rank.p, hybrid ? rowdup.p : (const uint32_t *)nullptr);
    KL_CUDA(cudaMemcpyAsync(&obs->count, obs->rank.p + nw, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx().stream));
    sync_stream();
    obs->bits = std::move(bitmap);
    m32 = obs->count;
    num = obs;
    out->class_ids.alloc((size_t)(m32 ? m32 : 1));
    KL_LAUNCH(enumerate_bits, (unsigned)((nw + 255) / 256), 256, 0, num->bits.p, num->rank.p, nw, out->class_ids.p);
    tr.mark("renumber");
  }
  out->m = (int64_t)m32;
  // class list: dense ids stay on the device, (k, code) pairs are decoded on demand
  out->n_classes = (int64_t)m32;
  out->class_M = cfg.M; out->class_N = cfg.N; out->classes_on_host = false;
  for (int k = cfg.M; k <= cfg.N + 1; k++) out->class_level_off[k] = P.level_off[k];
  if (n_features > 0) { sync_stream(); return apply_features(*out, features, n_features); }
  // matrices with one column per class keep what the matrix-free logistic pass needs
  if ((!P.binarize || hybrid) && cfg.N <= IMP_MAX_N && s.n > 0 && m32 > 0) {
    auto imp = std::make_shared<Implicit>();
    imp->seqs = seqs; imp->M = cfg.M; imp->N = cfg.N; imp->op = P.op;
    imp->Mlo = P.binarize ? (cfg.M > KT_MAX + 1 ? cfg.M : KT_MAX + 1) : cfg.M;
    uint32_t fo = 0;
    for (int k = cfg.M; k <= cfg.N + 1; k++) {
      imp->level_off[k] = P.level_off[k];
      imp->fo[k] = fo;
      if (k <= cfg.N && k >= imp->Mlo) fo += 1u << (2 * k);
    }
    if (P.binarize) {
      imp->binarized = true;
      imp->low_words = P.low_words;
      imp->lowcol.alloc((size_t)(P.low_words ? P.low_words * 32 : 1));
      if (P.low_words)
        KL_LAUNCH(low_columns, (unsigned)((P.low_words * 32 + 127) / 128), 128, 0, P.tl, P.tl_cnt, P.low_words * 32,
                  num->bits.p, num->rank.p, imp->lowcol.p);
      imp->lowbits = std::move(lowbits);
      imp->events.alloc((size_t)(n_events ? n_events : 1));
      KL_LAUNCH(gather_events, (unsigned)((s.n * 32 + 127) / 128), 128, 0, out->col.p, stride, s.n, evptr.p, imp->events.p);
      imp->evptr = std::move(evptr);
    }
    imp->num = num;
    out->imp = imp;
  }
  sync_stream();
  return out;
}

void matrix_class_list(Matrix &M) {
  if (M.classes_on_host) return;
  std::vector<uint32_t> hid((size_t)M.n_classes);
  M.class_ids.download(hid.data(), (size_t)M.n_classes);
  sync_stream();
  M.class_k.resize((size_t)M.n_classes); M.class_code.resize((size_t)M.n_classes);
  int k = M.class_M;
  for (size_t j = 0; j < hid.size(); j++) {
    while (k < M.class_N && hid[j] >= M.class_level_off[k + 1]) k++;
    M.class_k[j] = k; M.class_code[j] = hid[j] - M.class_level_off[k];
  }
  M.classes_on_host = true;
}

std::shared_ptr<Matrix> extract(const kmerlr_config &cfg, std::shared_ptr<SeqSet> seqs, const int32_t *frozen_k,
                                const uint64_t *frozen_code, int64_t n_frozen, const int32_t *features,
                                int64_t n_features, int flags) {
  return extract_impl(cfg, seqs, frozen_k, frozen_code, n_frozen, features, n_features, flags, nullptr);
}

// kmerlr_extract: sequences in host memory; upload, packing and extraction are pipelined
std::shared_ptr<Matrix> extract_host(const kmerlr_config &cfg, const uint8_t *seq, const int64_t *off, int64_t n,
                                     const int32_t *frozen_k, const uint64_t *frozen_code, int64_t n_frozen,
                                     const int32_t *features, int64_t n_features, int flags) {
  HostFeed hf;
  auto s = sequences_begin(seq, off, n, hf);
  auto out = extract_impl(cfg, s, frozen_k, frozen_code, n_frozen, features, n_features, flags, &hf);
  sync_stream();
  return out;
}

}  // namespace kl
