// score.cu -- stage 3 of the hot path: sliding-window genomic scoring.
//
// Replaces genomicKmerLr.Predict + predict_window_genomic (kmerLr_predict_genomic.go:134-171):
// for every window start j = 0, step, 2 step, ... < len - W of every region, count the model's
// k-mer classes in the window, build the feature vector (singles, pair products, binarize),
// evaluate log sigma(x . theta) per ensemble member, summarize, and sum over models.
// Quirks kept (SURVEY 8a row 11): slot count n/step+1 with a strict loop bound (the last slot may
// stay 0.0), regions with len <= W give no output, the model Transform is not applied.
//
// A model class (k, code) is looked up by its dense id level_off[k] + code, the column numbering of the
// extraction (gapped.cu).  Every model the extraction accepts is scored: the nucleotide alphabet with k <= 14
// and any subset of the strand flags, and the gapped alphabet with k <= 11.
//
// Three kernels:
//   score_linear   models whose score is linear in the counts (no binarize, no pair features):
//                  per tile of the region, per-level prefix sums of the per-position coefficient
//                  (in shared memory, or in a per-block scratch buffer when W + step does not fit);
//                  a window is 2 reads per level.  The nucleotide alphabet with at most one strand flag
//                  and k <= 13 takes a specialised instantiation; every other class rule enumerates the
//                  instance's variants with kmer_class.cuh
//   score_generic  everything else with at most 8192 classes, nucleotide, one strand flag, k <= 13:
//                  one warp per window, counts in shared memory
//   score_hits     the remaining generic models: one warp per window, the window's model-class hits in a
//                  per-warp ordered hash table in global memory; the cost follows the hits
#include "common.cuh"
#include "kmer_class.cuh"

#include <cmath>

namespace kl {

namespace {

constexpr uint32_t HEMPTY = 0xFFFFFFFFu;

struct DevModel {
  int M, N, op, binarize, summary;
  int n_classes, n_features, n_members;
  uint32_t hmask;          // hash table size - 1
  uint32_t levels;         // bit k set: the model has a class of length k
  ClassRule rule;          // class rule of the extraction (kmer_class.cuh)
  uint32_t level_off[16];  // dense id of (k, code 0), as in gapped.cu: key of class (k, code) = level_off[k] + code
  uint32_t hit_cap;        // score_hits: hash range of the window table (power of 2)
  uint32_t hit_size;       // score_hits: window table slots (hit_cap + most distinct hits + 1)
  const uint32_t *hkeys;   // dense class id, HEMPTY = free
  const int32_t *hvals;    // class index
  const int32_t *feat;     // n_features x 2
  const double *theta;     // n_members x (n_features + 1)
  const double *cweight;   // n_members x n_classes: sum of theta over single features of the class
  const double *wtab;      // nucleotide: class weight (member 0) of every code of the levels k <= SCORE_KD
  const int32_t *adj_off;  // score_hits: features whose first class is c are adj_feat[adj_off[c] .. adj_off[c + 1])
  const int32_t *adj_feat;
};

__device__ __forceinline__ uint32_t hash_u32(uint32_t x) {
  x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
  return x;
}
__device__ __forceinline__ int model_lookup(const DevModel &md, uint32_t key) {
  uint32_t h = hash_u32(key) & md.hmask;
  while (true) {
    uint32_t kk = __ldg(md.hkeys + h);
    if (kk == key) return __ldg(md.hvals + h);
    if (kk == HEMPTY) return -1;
    h = (h + 1) & md.hmask;
  }
}
// the same probe sequence over a copy of the table (shared memory)
__device__ __forceinline__ int table_lookup(const uint32_t *keys, const int32_t *vals, uint32_t hmask, uint32_t key) {
  uint32_t h = hash_u32(key) & hmask;
  while (true) {
    uint32_t kk = keys[h];
    if (kk == key) return vals[h];
    if (kk == HEMPTY) return -1;
    h = (h + 1) & hmask;
  }
}

__device__ __forceinline__ double summarize(int summary, const double *x, int n) {
  double r;
  switch (summary) {
    case KMERLR_SUMMARY_MEAN: r = 0.0; for (int j = 0; j < n; j++) r += x[j]; return r / (double)n;
    case KMERLR_SUMMARY_PRODUCT: r = 1.0; for (int j = 0; j < n; j++) r *= x[j]; return r;
    case KMERLR_SUMMARY_MIN: r = x[0]; for (int j = 1; j < n; j++) if (r > x[j]) r = x[j]; return r;
    case KMERLR_SUMMARY_MAX: r = x[0]; for (int j = 1; j < n; j++) if (r < x[j]) r = x[j]; return r;
    default: return x[0];
  }
}

constexpr int MAX_MEMBERS = 16;

// one warp per window
__global__ void score_generic(const DevModel *__restrict__ models, int n_models, const int64_t *__restrict__ len,
                              const int64_t *__restrict__ blk, const uint32_t *__restrict__ bits2,
                              const uint16_t *__restrict__ inv16, int64_t n_regions,
                              const int64_t *__restrict__ win_off, const int64_t *__restrict__ slot_off,
                              int64_t total_windows, int64_t W, int64_t step, int max_classes,
                              int64_t slot_stride, double *__restrict__ out) {
  extern __shared__ uint32_t smem[];
  const unsigned lane = lane_id();
  uint32_t *cnt = smem + (size_t)(threadIdx.x >> 5) * max_classes;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t wi = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; wi < total_windows; wi += nwarps) {
    // region of window wi
    int64_t lo = 0, hi = n_regions;
    while (hi - lo > 1) { int64_t mid = (lo + hi) >> 1; if (win_off[mid] <= wi) lo = mid; else hi = mid; }
    const int64_t r = lo, w = wi - win_off[r], a = w * step;
    const uint32_t *b2 = bits2 + blk[r] * 4;
    const uint16_t *iv = inv16 + blk[r] * 4;
    double total = 0.0;
    for (int mi = 0; mi < n_models; mi++) {
      const DevModel md = models[mi];
      const uint32_t *level_off = models[mi].level_off;
      for (int i = lane; i < md.n_classes; i += 32) cnt[i] = 0;
      __syncwarp();
      // CountKmers / IdentifyKmers restricted to the model classes
      for (int64_t i = lane; i < W; i += 32) {
        uint32_t fw = 0, im = 0;
        for (int k = 1; k <= md.N && i + k <= W; k++) {
          int64_t idx = a + i + k - 1;
          uint32_t word = __ldg(b2 + (idx >> 4)), inv = (__ldg(iv + (idx >> 4)) >> (idx & 15)) & 1u;
          if (inv) break;
          uint32_t x = (word >> (2 * (idx & 15))) & 3u;
          fw = (fw << 2) | x;
          if (md.op == 1) im |= (3u - x) << (2 * (k - 1));
          else if (md.op == 2) im = (im << 2) | (3u - x);
          else if (md.op == 3) im |= x << (2 * (k - 1));
          if (k >= md.M && ((md.levels >> k) & 1u)) {
            uint32_t code = md.op ? min(fw, im) : fw;
            int ci = model_lookup(md, level_off[k] + code);
            if (ci >= 0) atomicAdd(cnt + ci, 1u);
          }
        }
      }
      __syncwarp();
      // convert_counts(counts, features, false) (kmerLr_data.go:210-229) and x . theta per member
      double z[MAX_MEMBERS];
      for (int e = 0; e < md.n_members; e++) z[e] = 0.0;
      for (int j = lane; j < md.n_features; j += 32) {
        int i1 = md.feat[2 * j], i2 = md.feat[2 * j + 1];
        uint32_t c1 = cnt[i1], c2 = cnt[i2];
        if (md.binarize) { c1 = c1 ? 1 : 0; c2 = c2 ? 1 : 0; }
        double v = i1 == i2 ? (double)c1 : ((c1 && c2) ? (double)(c1 * c2) : 0.0);
        if (v != 0.0)
          for (int e = 0; e < md.n_members; e++) z[e] += v * md.theta[(int64_t)e * (md.n_features + 1) + j + 1];
      }
      double lp[MAX_MEMBERS];
      for (int e = 0; e < md.n_members; e++) {
        double zz = md.theta[(int64_t)e * (md.n_features + 1)] + warp_sum(z[e]);
        lp[e] = -log_add0(-zz);
      }
      total += summarize(md.summary, lp, md.n_members);
      __syncwarp();
    }
    if (lane == 0) out[slot_off[r] + w * slot_stride] = total;
  }
}

// ---- linear fast path -----------------------------------------------------------------------------
// One block per tile of TP window-start positions of one region.  For every level k of the model, the
// block holds the inclusive prefix sum Q_k over tile positions of
//   t_k(p) = sum over the variants of the k-mer starting at p of the class weight (0 if not a model class /
//            invalid; one variant unless the alphabet is gapped),
// so that  z(window at a) = theta_0 + sum_k Q_k[a + W - k] - Q_k[a - 1].  The prefix spans one tile (about
// W + step positions or more), never a whole region, so its rounding stays that of a sum of tile length.
// GEN: the class rule of kmer_class.cuh (gapped alphabet, several strand flags, k = 14); otherwise the
// nucleotide alphabet with at most one strand flag and k <= 13, with the class computed from the packed bits.
// SCRATCH: the prefix rows live in a per-block buffer in global memory (W + step larger than shared memory
// allows); the grid is then bounded and each block walks its tiles.
struct LinearTile { int64_t region, p0; };

constexpr int SCORE_THREADS = 1024;
// levels k <= SCORE_KD of a small nucleotide model: the class weight of every code in a direct table in shared
// memory (one LDS per position and level instead of a hash probe sequence + a gather of the weight)
constexpr int SCORE_KD = 5;
constexpr int SCORE_WT = (4 + 16 + 64 + 256 + 1024);     // sum_{k=1..5} 4^k entries
__host__ __device__ __forceinline__ uint32_t score_doff(int k) { return ((1u << (2 * k)) - 4u) / 3u; }   // sum_{j<k} 4^j
__device__ __forceinline__ int level_slot(uint32_t levels, int k) {   // index of level k among the model's levels
  return ((levels >> k) & 1u) ? __popc(levels & ((1u << k) - 1u)) : -1;
}

template <bool GEN, bool SCRATCH>
__global__ void __launch_bounds__(SCORE_THREADS) score_linear(const DevModel *__restrict__ models, int member,
                                                    int accumulate, const int64_t *__restrict__ len,
                                                    const int64_t *__restrict__ blk,
                                                    const uint32_t *__restrict__ bits2,
                                                    const uint16_t *__restrict__ inv16,
                                                    const LinearTile *__restrict__ tiles, int64_t n_tiles,
                                                    const int64_t *__restrict__ slot_off, int64_t W, int64_t step,
                                                    int TP, int model_index, int hs_smem, int64_t slot_stride,
                                                    double *__restrict__ scratch, double *__restrict__ out) {
  // shared: nlev x (TP + 1) prefix rows, q[.][0] = 0 (unless SCRATCH); then a copy of the class table and the
  // direct weight table
  extern __shared__ double smem_d[];
  __shared__ double warp_tot[SCORE_THREADS / 32];
  __shared__ uint32_t slo[16];
  const DevModel md = models[model_index];
  const int N = md.N;
  const uint32_t maskN = (1u << (2 * N)) - 1u;
  const int nlev = __popc(md.levels);
  const int stride = TP + 1;
  double *q = SCRATCH ? scratch + (size_t)blockIdx.x * nlev * stride : smem_d;
  // small class tables are probed in shared memory (most probes miss: one LDS instead of one LDG each)
  uint32_t *skeys = reinterpret_cast<uint32_t *>(SCRATCH ? smem_d : smem_d + (size_t)nlev * stride);
  int32_t *svals = reinterpret_cast<int32_t *>(skeys + hs_smem);
  double *wtab = reinterpret_cast<double *>(svals + hs_smem);
  const bool direct = hs_smem && md.wtab;
  for (int i = threadIdx.x; i < hs_smem; i += blockDim.x) { skeys[i] = md.hkeys[i]; svals[i] = md.hvals[i]; }
  if (direct)
    for (int i = threadIdx.x; i < SCORE_WT; i += blockDim.x) wtab[i] = __ldg(md.wtab + i);
  if (threadIdx.x < 16) slo[threadIdx.x] = models[model_index].level_off[threadIdx.x];
  __syncthreads();
  auto weight = [&](int k, uint32_t code) -> double {
    if (direct && k <= SCORE_KD) return wtab[score_doff(k) + code];
    const uint32_t key = slo[k] + code;
    int ci = hs_smem ? table_lookup(skeys, svals, md.hmask, key) : model_lookup(md, key);
    return ci >= 0 ? __ldg(md.cweight + (int64_t)member * md.n_classes + ci) : 0.0;
  };
  const int per = (TP + blockDim.x - 1) / blockDim.x;
  for (int64_t ti = blockIdx.x; ti < n_tiles; ti += gridDim.x) {
    const LinearTile tl = tiles[ti];
    const int64_t L = len[tl.region];
    const uint32_t *b2 = bits2 + blk[tl.region] * 4;
    const uint16_t *iv = inv16 + blk[tl.region] * 4;
    // phase 1: t_k(p) for p in [p0, p0 + TP).  The N bases starting at p are 2N consecutive bits of the
    // packed words (one funnel shift, first base in the low bits): no rolling state, so the positions
    // are simply dealt to the threads
    for (int i = threadIdx.x; i < TP; i += blockDim.x) {
      const int64_t p = tl.p0 + i;
      int len_f = 0;
      uint32_t e = 0, FW = 0, IM = 0;
      if (p < L) {
        const int64_t wi = p >> 4;
        const int sh = (int)(p & 15);
        e = __funnelshift_r(__ldg(b2 + wi), __ldg(b2 + wi + 1), 2 * sh) & maskN;
        const int64_t rest = L - p;
        const uint32_t ivb = (((uint32_t)__ldg(iv + wi) | ((uint32_t)__ldg(iv + wi + 1) << 16)) >> sh) |
                             (1u << (rest < N ? (int)rest : N));
        len_f = __ffs(ivb) - 1;
        if (!GEN) {
          FW = swap_pairs(__brev(e)) >> (32 - 2 * N);
          IM = md.op == 1 ? (~e) & maskN : e;       // image of the window under revcomp / reverse
        }
      }
      for (int k = md.M; k <= N; k++) {
        const int sl = level_slot(md.levels, k);
        if (sl < 0) continue;
        double t = 0.0;
        if (len_f >= k) {
          if (GEN) {
            const uint32_t nm = kmer_masks(md.rule, k);
            for (uint32_t mask = 0; mask < nm; mask++) {
              const uint32_t code = kmer_variant_class(md.rule, e, k, mask);
              if (code != KMER_NONE) t += weight(k, code);
            }
          } else {
            uint32_t fw = FW >> (2 * (N - k)), code = fw;
            if (md.op == 1 || md.op == 3) code = min(fw, IM & ((1u << (2 * k)) - 1u));
            else if (md.op == 2) code = min(fw, (~fw) & ((1u << (2 * k)) - 1u));
            t = weight(k, code);
          }
        }
        q[sl * stride + 1 + i] = t;
      }
    }
    if ((int)threadIdx.x < nlev) q[threadIdx.x * stride] = 0.0;
    __syncthreads();
    // phase 2: inclusive scan per level (blocked: thread-local runs, warp scan, block carry)
    for (int sl = 0; sl < nlev; sl++) {
      double *row = q + sl * stride + 1;
      int i0 = threadIdx.x * per, i1 = min(TP, i0 + per);
      double s = 0.0;
      for (int i = i0; i < i1; i++) { s += row[i]; row[i] = s; }
      double x = s;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        double y = __shfl_up_sync(0xffffffffu, x, o);
        if ((int)lane_id() >= o) x += y;
      }
      if (lane_id() == 31) warp_tot[threadIdx.x >> 5] = x;
      __syncthreads();
      double carry = x - s;
      for (int wv = 0; wv < (int)(threadIdx.x >> 5); wv++) carry += warp_tot[wv];
      for (int i = i0; i < i1; i++) row[i] += carry;
      __syncthreads();
    }
    // phase 3: windows starting inside this tile whose k-mers all lie inside the tile
    const int64_t nwin_region = (L - W > 0) ? (L - W + step - 1) / step : 0;
    const int64_t w_first = (tl.p0 + step - 1) / step;
    for (int64_t w = w_first + threadIdx.x; w < nwin_region; w += blockDim.x) {
      int64_t a = w * step - tl.p0;           // tile-relative start
      if (a + W > TP) break;
      double z = md.theta[(int64_t)member * (md.n_features + 1)];
      for (int k = md.M; k <= N; k++) {
        const int sl = level_slot(md.levels, k);
        if (sl < 0 || W < k) continue;
        const double *row = q + sl * stride;  // row[i+1] = inclusive prefix through position i
        z += row[a + W - k + 1] - row[a];
      }
      double lp = -log_add0(-z);
      int64_t o = slot_off[tl.region] + w * slot_stride;
      if (accumulate) out[o] += lp; else out[o] = lp;
    }
    if (ti + gridDim.x < n_tiles) __syncthreads();   // phase 3 reads the rows the next tile overwrites
  }
}

// ---- generic models without the limits of score_generic ------------------------------------------------
// One warp per window.  The window's hits (model class indices, one per counted variant) go into an ordered
// linear-probing hash table (Amble & Knuth): inserted with atomicMin, smaller keys stay, displaced keys move on.
// Its layout depends on the key set only, not on the order of the atomics, so the walk over its slots -- and the
// floating-point sums -- are the same in every run.  Pass 1 inserts, pass 2 counts (the table no longer moves),
// pass 3 walks the slots: every present class adds its features (class -> feature adjacency built on the host;
// a pair partner is looked up in the same table), pass 4 clears what it used.  The table of a warp has
// hit_size slots; nothing scales with n_features or n_classes x warps.
__device__ __forceinline__ void hit_insert(uint32_t *tab, uint32_t cap, uint32_t x) {
  uint32_t h = hash_u32(x) & (cap - 1);
  while (true) {
    const uint32_t old = atomicMin(tab + h, x);
    if (old == HEMPTY || old == x) return;
    if (old > x) x = old;                     // x took the slot: carry on with the key it displaced
    h++;
  }
}
// slot of x, or of the first larger key / the empty slot where x would be: keys along a probe run increase
__device__ __forceinline__ uint32_t hit_find(const uint32_t *tab, uint32_t cap, uint32_t x) {
  uint32_t h = hash_u32(x) & (cap - 1);
  while (__ldcg(tab + h) < x) h++;
  return h;
}

// every counted variant of every k-mer inside the window [a, a + W) that is a model class: f(class index)
template <class F>
__device__ __forceinline__ void window_hits(const DevModel &md, const uint32_t *level_off, const uint32_t *b2,
                                            const uint16_t *iv, int64_t a, int64_t W, F f) {
  const int N = md.N;
  const uint32_t maskN = (1u << (2 * N)) - 1u;
  for (int64_t i = lane_id(); i < W; i += 32) {
    const int64_t p = a + i, wi = p >> 4, rest = W - i;
    const int sh = (int)(p & 15);
    const uint32_t e = __funnelshift_r(__ldg(b2 + wi), __ldg(b2 + wi + 1), 2 * sh) & maskN;
    const uint32_t ivb = (((uint32_t)__ldg(iv + wi) | ((uint32_t)__ldg(iv + wi + 1) << 16)) >> sh) |
                         (1u << (rest < N ? (int)rest : N));
    const int len_f = __ffs(ivb) - 1;
    for (int k = md.M; k <= N && k <= len_f; k++) {
      if (!((md.levels >> k) & 1u)) continue;
      const uint32_t nm = kmer_masks(md.rule, k), lo = level_off[k];
      for (uint32_t mask = 0; mask < nm; mask++) {
        const uint32_t code = kmer_variant_class(md.rule, e, k, mask);
        if (code == KMER_NONE) continue;
        const int ci = model_lookup(md, lo + code);
        if (ci >= 0) f((uint32_t)ci);
      }
    }
  }
}

__global__ void score_hits(const DevModel *__restrict__ models, int n_models, const int64_t *__restrict__ blk,
                           const uint32_t *__restrict__ bits2, const uint16_t *__restrict__ inv16, int64_t n_regions,
                           const int64_t *__restrict__ win_off, const int64_t *__restrict__ slot_off,
                           int64_t total_windows, int64_t W, int64_t step, int64_t slot_stride,
                           uint32_t *__restrict__ scratch, int64_t tab_stride, double *__restrict__ out) {
  const unsigned lane = lane_id();
  const int64_t gw = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  uint32_t *tab = scratch + gw * tab_stride;                // keys, HEMPTY = free
  uint32_t *cnt = scratch + (nwarps + gw) * tab_stride;     // counts, 0 = free
  for (int64_t wi = gw; wi < total_windows; wi += nwarps) {
    int64_t lo = 0, hi = n_regions;
    while (hi - lo > 1) { int64_t mid = (lo + hi) >> 1; if (win_off[mid] <= wi) lo = mid; else hi = mid; }
    const int64_t r = lo, w = wi - win_off[r], a = w * step;
    const uint32_t *b2 = bits2 + blk[r] * 4;
    const uint16_t *iv = inv16 + blk[r] * 4;
    double total = 0.0;
    for (int mi = 0; mi < n_models; mi++) {
      const DevModel &md = models[mi];
      const uint32_t *level_off = md.level_off;
      const uint32_t cap = md.hit_cap, size = md.hit_size;
      window_hits(md, level_off, b2, iv, a, W, [&](uint32_t ci) { hit_insert(tab, cap, ci); });
      __syncwarp();
      window_hits(md, level_off, b2, iv, a, W, [&](uint32_t ci) { atomicAdd(cnt + hit_find(tab, cap, ci), 1u); });
      __syncwarp();
      // convert_counts(counts, features, false) (kmerLr_data.go:210-229) and x . theta per member
      const int nf = md.n_features, nm = md.n_members, bin = md.binarize;
      double z[MAX_MEMBERS];
      for (int e = 0; e < nm; e++) z[e] = 0.0;
      for (uint32_t sl = lane; sl < size; sl += 32) {
        const uint32_t c = __ldcg(tab + sl);
        if (c == HEMPTY) continue;
        const uint32_t c1 = bin ? 1u : __ldcg(cnt + sl);
        for (int j0 = __ldg(md.adj_off + c), j1 = __ldg(md.adj_off + c + 1); j0 < j1; j0++) {
          const int j = __ldg(md.adj_feat + j0);
          const uint32_t c2i = (uint32_t)__ldg(md.feat + 2 * j + 1);
          double v;
          if (c2i == c) {
            v = (double)c1;
          } else {
            const uint32_t h = hit_find(tab, cap, c2i);
            const uint32_t c2 = __ldcg(tab + h) == c2i ? (bin ? 1u : __ldcg(cnt + h)) : 0u;
            v = c2 ? (double)(c1 * c2) : 0.0;
          }
          if (v != 0.0)
            for (int e = 0; e < nm; e++) z[e] += v * __ldg(md.theta + (int64_t)e * (nf + 1) + j + 1);
        }
      }
      __syncwarp();
      for (uint32_t sl = lane; sl < size; sl += 32)
        if (__ldcg(tab + sl) != HEMPTY) { __stcg(tab + sl, HEMPTY); __stcg(cnt + sl, 0u); }
      double lp[MAX_MEMBERS];
      for (int e = 0; e < nm; e++) {
        double zz = __ldg(md.theta + (int64_t)e * (nf + 1)) + warp_sum(z[e]);
        lp[e] = -log_add0(-zz);
      }
      total += summarize(md.summary, lp, nm);
      __syncwarp();
    }
    if (lane == 0) out[slot_off[r] + w * slot_stride] = total;
  }
}

struct HostModel {
  DevModel d;
  DevBuf<uint32_t> hkeys;
  DevBuf<int32_t> hvals, feat, adj_off, adj_feat;
  DevBuf<double> theta, cweight, wtab;
  bool linear;
  bool gen;                // class rule beyond the nucleotide alphabet with one strand flag and k <= 13
  uint64_t max_hits;       // most counted variants of model classes in one window
};

}  // namespace

// layout 0: predict_window_genomic -- n/step + 1 slots per region, window j*step in slot j
// layout 1: predict_window (kmerLr_predict.go:89-124) -- n = len - W slots, window starting at j in slot j
// feed: the sequences are still on the host and arrive in chunks of whole rows (kmerlr_score_windows with host
// buffers).  Count models without pair features then work chunk by chunk: the copy of chunk c + 1 (copy stream)
// and the copy of the scores of chunk c - 1 back to the host (third stream) overlap the scoring of chunk c.
void score_windows(const kmerlr_model *models, int n_models, const SeqSet &s, int64_t W, int64_t step,
                   double *out_host, std::shared_ptr<Object> *out_dev, int layout, SeqFeed *feed) {
  require_ready();
  KL_REQUIRE(n_models >= 1 && W >= 1 && step >= 1, "score_windows: bad arguments");
  std::vector<std::unique_ptr<HostModel>> hm;
  int max_classes = 1;
  bool all_linear = true, any_hits = false;
  for (int mi = 0; mi < n_models; mi++) {
    const kmerlr_model &m = models[mi];
    KL_REQUIRE(m.cfg.alphabet == 0 || m.cfg.alphabet == 1,
               "score_windows: alphabet: 0 = nucleotide, 1 = gapped nucleotide (IUPAC is not implemented)");
    const bool gapped = m.cfg.alphabet == 1;
    KL_REQUIRE(m.cfg.M >= 1 && m.cfg.M <= m.cfg.N && m.cfg.N <= (gapped ? 11 : 14),
               "score_windows: need 1 <= M <= N <= 14 (nucleotide) or <= 11 (gapped nucleotide)");
    int nops = (m.cfg.complement != 0) + (m.cfg.reverse != 0) + (m.cfg.revcomp != 0);
    KL_REQUIRE(m.n_members >= 1 && m.n_members <= MAX_MEMBERS, "score_windows: 1..16 ensemble members");
    KL_REQUIRE(m.n_members == 1 || m.summary != KMERLR_SUMMARY_NONE, "no summary given for ensemble classifier");
    KL_REQUIRE(m.n_classes >= 0 && m.n_classes < ((int64_t)1 << 31), "score_windows: too many model classes");
    auto h = std::make_unique<HostModel>();
    DevModel &d = h->d;
    d.M = m.cfg.M; d.N = m.cfg.N; d.binarize = m.cfg.binarize != 0; d.summary = m.summary;
    d.op = m.cfg.revcomp ? 1 : (m.cfg.complement ? 2 : (m.cfg.reverse ? 3 : 0));
    d.rule = ClassRule{gapped ? 5 : 4, gapped ? m.cfg.max_ambiguous : -1, m.cfg.complement != 0, m.cfg.reverse != 0,
                       m.cfg.revcomp != 0};
    h->gen = gapped || nops > 1 || m.cfg.N > 13;
    d.n_classes = (int)m.n_classes; d.n_features = (int)m.n_features; d.n_members = (int)m.n_members;
    // dense class ids, as the extraction numbers its columns (gapped.cu)
    uint64_t dense = 0, pk = 1, ncodes[16] = {0};
    for (int k = 1; k <= d.N; k++) {
      pk *= (uint64_t)d.rule.A;
      ncodes[k] = pk;
      if (k < d.M) continue;
      d.level_off[k] = (uint32_t)dense;
      dense += (pk + 31) / 32 * 32;
    }
    uint32_t hs = 16; while (hs < 2 * (uint32_t)m.n_classes + 2) hs <<= 1;
    std::vector<uint32_t> keys(hs, HEMPTY); std::vector<int32_t> vals(hs, -1);
    d.levels = 0;
    auto mix = [](uint32_t x) { x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16; return x; };
    for (int64_t c = 0; c < m.n_classes; c++) {
      int k = m.class_k[c];
      KL_REQUIRE(k >= d.M && k <= d.N && m.class_code[c] < ncodes[k], "score_windows: class outside [M,N]");
      uint32_t key = d.level_off[k] + (uint32_t)m.class_code[c], hh = mix(key) & (hs - 1);
      while (keys[hh] != HEMPTY) { KL_REQUIRE(keys[hh] != key, "score_windows: duplicate model class"); hh = (hh + 1) & (hs - 1); }
      keys[hh] = key; vals[hh] = (int32_t)c;
      d.levels |= 1u << k;
    }
    d.hmask = hs - 1;
    h->linear = !d.binarize;
    std::vector<double> cwt((size_t)(m.n_members * (m.n_classes ? m.n_classes : 1)), 0.0);
    std::vector<int32_t> adj_off((size_t)m.n_classes + 1, 0), adj_feat((size_t)(m.n_features ? m.n_features : 1));
    for (int64_t j = 0; j < m.n_features; j++) {
      int32_t i1 = m.features[2 * j], i2 = m.features[2 * j + 1];
      KL_REQUIRE(i1 >= 0 && i1 < m.n_classes && i2 >= 0 && i2 < m.n_classes, "score_windows: feature index out of range");
      adj_off[(size_t)i1 + 1]++;
      if (i1 != i2) h->linear = false;
      else for (int64_t e = 0; e < m.n_members; e++) cwt[(size_t)(e * m.n_classes + i1)] += m.theta[e * (m.n_features + 1) + j + 1];
    }
    for (int64_t c = 0; c < m.n_classes; c++) adj_off[(size_t)c + 1] += adj_off[(size_t)c];
    {
      std::vector<int32_t> fill(adj_off.begin(), adj_off.end() - 1);
      for (int64_t j = 0; j < m.n_features; j++) adj_feat[(size_t)fill[(size_t)m.features[2 * j]]++] = (int32_t)j;
    }
    // most counted variants of the model's levels in one window, and the window table of score_hits
    h->max_hits = 0;
    for (int k = d.M; k <= d.N; k++) {
      if (!((d.levels >> k) & 1u) || W < k) continue;
      const int nin = gapped && k >= 2 ? k - 2 : 0;
      uint64_t nv = 0, binom = 1;                        // variants with at most max_ambiguous wildcards
      for (int j = 0; j <= nin; j++) {
        if (d.rule.max_amb < 0 || j <= d.rule.max_amb) nv += binom;
        binom = binom * (uint64_t)(nin - j) / (uint64_t)(j + 1);
      }
      h->max_hits += (uint64_t)(W - k + 1) * nv;
    }
    const uint64_t distinct = std::min<uint64_t>(h->max_hits, (uint64_t)m.n_classes);
    uint64_t cap = 32; while (cap < 2 * distinct) cap <<= 1;
    KL_REQUIRE(cap + distinct + 1 < ((uint64_t)1 << 32), "score_windows: window too large for the hit table");
    d.hit_cap = (uint32_t)cap; d.hit_size = (uint32_t)(cap + distinct + 1);
    if (!h->linear) all_linear = false;
    h->hkeys.alloc(hs); h->hvals.alloc(hs);
    h->hkeys.upload(keys.data(), hs); h->hvals.upload(vals.data(), hs);
    h->feat.alloc((size_t)(m.n_features ? 2 * m.n_features : 1));
    h->feat.upload(m.features, (size_t)(2 * m.n_features));
    h->theta.alloc((size_t)(m.n_members * (m.n_features + 1)));
    h->theta.upload(m.theta, (size_t)(m.n_members * (m.n_features + 1)));
    h->cweight.alloc(cwt.size());
    h->cweight.upload(cwt.data(), cwt.size());
    h->adj_off.alloc(adj_off.size()); h->adj_feat.alloc(adj_feat.size());
    h->adj_off.upload(adj_off.data(), adj_off.size()); h->adj_feat.upload(adj_feat.data(), adj_feat.size());
    d.wtab = nullptr;
    if (!gapped) {
      std::vector<double> wt(SCORE_WT, 0.0);
      for (int64_t c = 0; c < m.n_classes; c++)
        if (m.class_k[c] <= SCORE_KD) wt[score_doff(m.class_k[c]) + m.class_code[c]] = cwt[(size_t)c];
      h->wtab.alloc(SCORE_WT);
      h->wtab.upload(wt.data(), SCORE_WT);
      d.wtab = h->wtab.p;
    }
    d.hkeys = h->hkeys.p; d.hvals = h->hvals.p; d.feat = h->feat.p; d.theta = h->theta.p; d.cweight = h->cweight.p;
    d.adj_off = h->adj_off.p; d.adj_feat = h->adj_feat.p;
    if (d.n_classes > max_classes) max_classes = d.n_classes;
    if (h->gen || d.n_classes > 8192) any_hits = true;
    hm.push_back(std::move(h));
  }
  sync_stream();
  // a summary of several members is not linear in the per-member scores unless it is the mean
  for (auto &h : hm)
    if (h->d.n_members > 1) all_linear = false;
  std::vector<DevModel> dm;
  for (auto &h : hm) dm.push_back(h->d);
  DevBuf<DevModel> dmodels((size_t)n_models);
  dmodels.upload(dm.data(), (size_t)n_models);
  // slots and windows per region
  std::vector<int64_t> len((size_t)s.n);
  s.len.download(len.data(), (size_t)s.n);
  sync_stream();
  std::vector<int64_t> slot_off((size_t)s.n + 1, 0), win_off((size_t)s.n + 1, 0);
  for (int64_t r = 0; r < s.n; r++) {
    slot_off[r + 1] = slot_off[r] + (layout == 1 ? (len[r] - W > 0 ? len[r] - W : 0) : kmerlr_window_slots(len[r], W, step));
    win_off[r + 1] = win_off[r] + (len[r] - W > 0 ? (len[r] - W + step - 1) / step : 0);
  }
  const int64_t total_slots = slot_off[s.n], total_windows = win_off[s.n];
  auto outbuf = std::make_shared<Matrix>();   // reuse Matrix.val_f64 as a plain device vector
  outbuf->val_f64.alloc((size_t)(total_slots ? total_slots : 1));
  outbuf->val_f64.zero();
  outbuf->n = total_slots;
  DevBuf<int64_t> dslot((size_t)s.n + 1), dwin((size_t)s.n + 1);
  dslot.upload(slot_off.data(), (size_t)s.n + 1);
  dwin.upload(win_off.data(), (size_t)s.n + 1);
  bool copied_home = false;       // the scores went to out_host chunk by chunk
  if (total_windows > 0) {
    if (all_linear) {
      for (int mi = 0; mi < n_models; mi++) {
        const DevModel &d = dm[mi];
        const bool gen = hm[mi]->gen;
        int nlev = __builtin_popcount(d.levels);
        if (nlev == 0) nlev = 1;
        // tile: as many positions as 200 KB of prefix sums allow, at least W + step
        const int64_t hs = (int64_t)d.hmask + 1;
        const int hs_smem = hs * 8 <= 16 * 1024 ? (int)hs : 0;
        const int wt_bytes = hs_smem && d.wtab ? SCORE_WT * 8 : 0;   // direct weight tables of the levels <= SCORE_KD
        int64_t TP = (200 * 1024 - hs_smem * 8 - wt_bytes) / (8 * nlev) - 1;
        if (TP > 16384) TP = 16384;
        // W + step does not fit: the prefix rows go to a per-block scratch buffer, a tile spans W plus at most
        // 16 384 positions of further window starts, and the grid is bounded by the SM count
        const bool scratch = TP < W + step;
        if (scratch) {
          const int64_t more = std::max<int64_t>(0, std::min<int64_t>(W, 16384) / step - 1);
          TP = W + more * step;
          KL_REQUIRE(TP < ((int64_t)1 << 30), "score_windows: window too large");
        }
        // windows per tile: starts a with a + W <= TP (a tile advances by that many steps)
        int64_t starts = (TP - W) / step + 1;
        std::vector<LinearTile> tiles;
        for (int64_t r = 0; r < s.n; r++) {
          int64_t nw = win_off[r + 1] - win_off[r];
          for (int64_t w0 = 0; w0 < nw; w0 += starts) tiles.push_back(LinearTile{r, w0 * step});
        }
        DevBuf<LinearTile> dt(tiles.size() ? tiles.size() : 1);
        dt.upload(tiles.data(), tiles.size());
        const int64_t grid_cap = scratch ? (int64_t)ctx().sm_count : INT64_MAX;
        DevBuf<double> qbuf;
        if (scratch) qbuf.alloc((size_t)std::min<int64_t>(grid_cap, (int64_t)tiles.size()) * nlev * (size_t)(TP + 1));
        size_t smem = (scratch ? 0 : (size_t)nlev * (size_t)(TP + 1) * sizeof(double)) + (size_t)hs_smem * 8 + (size_t)wt_bytes;
        auto kern = gen ? (scratch ? score_linear<true, true> : score_linear<true, false>)
                        : (scratch ? score_linear<false, true> : score_linear<false, false>);
        KL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        // chunk by chunk (one chunk when the sequences are resident): the tiles are sorted by region
        const int nch = feed ? feed->chunks() : 1;
        size_t t0 = 0;
        for (int c = 0; c < nch; c++) {
          const int64_t r0 = feed ? feed->first_row(c) : 0, r1 = feed ? feed->first_row(c + 1) : s.n;
          if (feed && mi == 0) feed->feed(c);
          size_t t1 = t0;
          while (t1 < tiles.size() && tiles[t1].region < r1) t1++;
          if (t1 > t0) {
            const int64_t nt = (int64_t)(t1 - t0);
            const unsigned grid = (unsigned)std::min<int64_t>(nt, grid_cap);
            const int64_t stride = layout == 1 ? step : (int64_t)1;
            if (!gen && !scratch)
              KL_LAUNCH((score_linear<false, false>), grid, SCORE_THREADS, smem, dmodels.p, 0, mi > 0 ? 1 : 0, s.len.p,
                        s.blk.p, s.bits2.p, s.inv16.p, dt.p + t0, nt, dslot.p, W, step, (int)TP, mi, hs_smem, stride,
                        qbuf.p, outbuf->val_f64.p);
            else if (!gen)
              KL_LAUNCH((score_linear<false, true>), grid, SCORE_THREADS, smem, dmodels.p, 0, mi > 0 ? 1 : 0, s.len.p,
                        s.blk.p, s.bits2.p, s.inv16.p, dt.p + t0, nt, dslot.p, W, step, (int)TP, mi, hs_smem, stride,
                        qbuf.p, outbuf->val_f64.p);
            else if (!scratch)
              KL_LAUNCH((score_linear<true, false>), grid, SCORE_THREADS, smem, dmodels.p, 0, mi > 0 ? 1 : 0, s.len.p,
                        s.blk.p, s.bits2.p, s.inv16.p, dt.p + t0, nt, dslot.p, W, step, (int)TP, mi, hs_smem, stride,
                        qbuf.p, outbuf->val_f64.p);
            else
              KL_LAUNCH((score_linear<true, true>), grid, SCORE_THREADS, smem, dmodels.p, 0, mi > 0 ? 1 : 0, s.len.p,
                        s.blk.p, s.bits2.p, s.inv16.p, dt.p + t0, nt, dslot.p, W, step, (int)TP, mi, hs_smem, stride,
                        qbuf.p, outbuf->val_f64.p);
          }
          t0 = t1;
          // the scores of the chunk go home while the next chunk is scored (last model only: the models add up)
          if (feed && out_host && mi == n_models - 1 && slot_off[r1] > slot_off[r0]) {
            cudaEvent_t ev;
            KL_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
            KL_CUDA(cudaEventRecord(ev, ctx().stream));
            KL_CUDA(cudaStreamWaitEvent(ctx().alt_stream, ev, 0));
            KL_CUDA(cudaMemcpyAsync(out_host + slot_off[r0], outbuf->val_f64.p + slot_off[r0],
                                    (size_t)(slot_off[r1] - slot_off[r0]) * sizeof(double), cudaMemcpyDeviceToHost, ctx().alt_stream));
            KL_CUDA(cudaEventDestroy(ev));            // (released once the event has completed)
            copied_home = true;
          }
        }
        sync_stream();
      }
      if (copied_home) KL_CUDA(cudaStreamSynchronize(ctx().alt_stream));
    } else if (any_hits) {
      // a warp's window table: keys and counts of the largest model; as many warps as 512 MB of tables allow
      if (feed) feed->feed(-1);
      int64_t tab = 32;
      for (auto &h : hm) tab = std::max<int64_t>(tab, (int64_t)h->d.hit_size);
      tab = (tab + 31) / 32 * 32;
      const int64_t per_warp = 2 * tab * (int64_t)sizeof(uint32_t);
      int64_t warps = std::min<int64_t>((int64_t)ctx().sm_count * 64, std::max<int64_t>(32, ((int64_t)512 << 20) / per_warp));
      warps = std::min<int64_t>(warps, (total_windows + 3) / 4 * 4);
      const int64_t blocks = (warps + 3) / 4;
      DevBuf<uint32_t> tabs((size_t)(blocks * 4 * 2 * tab));       // the keys of every warp, then the counts
      KL_CUDA(cudaMemsetAsync(tabs.p, 0xFF, (size_t)(blocks * 4 * tab) * sizeof(uint32_t), ctx().stream));
      KL_CUDA(cudaMemsetAsync(tabs.p + blocks * 4 * tab, 0, (size_t)(blocks * 4 * tab) * sizeof(uint32_t), ctx().stream));
      KL_LAUNCH(score_hits, (unsigned)blocks, 128, 0, dmodels.p, n_models, s.blk.p, s.bits2.p, s.inv16.p, s.n, dwin.p,
                dslot.p, total_windows, W, step, layout == 1 ? step : (int64_t)1, tabs.p, tab, outbuf->val_f64.p);
    } else {
      if (feed) feed->feed(-1);
      size_t smem = (size_t)4 * (size_t)max_classes * sizeof(uint32_t);
      KL_CUDA(cudaFuncSetAttribute(score_generic, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      int64_t blocks = (total_windows + 3) / 4, cap = (int64_t)ctx().sm_count * 16;
      if (blocks > cap) blocks = cap;
      KL_LAUNCH(score_generic, (unsigned)blocks, 128, smem, dmodels.p, n_models, s.len.p, s.blk.p, s.bits2.p,
                s.inv16.p, s.n, dwin.p, dslot.p, total_windows, W, step, max_classes, layout == 1 ? step : (int64_t)1,
                outbuf->val_f64.p);
    }
  }
  else if (feed) feed->feed(-1);
  if (out_host && !copied_home) outbuf->val_f64.download(out_host, (size_t)total_slots);
  sync_stream();
  if (out_dev) *out_dev = outbuf;
}

}  // namespace kl
