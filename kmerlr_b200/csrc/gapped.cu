// gapped.cu -- the sort-based extraction path: every (row, class) instance becomes a 64-bit key, the keys are
// sorted (CUB radix sort) and run-length encoded; the runs are the stored entries in CSR order.  A correctness
// path, not a tuned one, for everything the warp-per-row kernel of extract.cu does not take:
//   * the gapped nucleotide alphabet {a, c, g, t, n} (SURVEY 8c items 3-6, 8f-3): every k-mer instance
//     contributes all its variants in which a subset of the INTERIOR positions is replaced by the wildcard n
//     (2^(k-2) variants, or those with at most max_ambiguous wildcards); codes are base-5 numbers.  This is the
//     configuration the reference's own exact pins use (kmerLr_test.go:30-68);
//   * the nucleotide alphabet with SEVERAL strand flags at once (kmerLr_learn.go:94 passes complement, reverse and
//     revcomp independently: class = min over the k-mer and every enabled image), with k-mers of 14 bases, or
//     with k > 8 on rows too long for the register sort of the main kernel.
// Codes are base-|alphabet| numbers (first letter most significant), class = min over the k-mer and its images.
#include "common.cuh"
#include "kmer_class.cuh"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_run_length_encode.cuh>

namespace kl {

namespace {

constexpr int GAP_MAX_N = 11;                       // gapped alphabet: 5^1 + ... + 5^11 < 2^26 dense ids
constexpr int SORT_MAX_N = 14;                      // nucleotide alphabet: 4^1 + ... + 4^14 < 2^29 dense ids
constexpr unsigned long long GAP_NONE = ~0ull;

struct GapParams {
  int M, N;
  ClassRule R;                  // alphabet, max_ambiguous, strand flags (kmer_class.cuh)
  uint32_t level_off[16];       // dense id of (k, code 0), multiples of 32
  uint32_t slots_per_pos;       // sum over k of 2^max(k-2, 0)
  uint32_t slot_off[16];        // offset of level k inside the slots of one position
};

// one thread per base position of the whole set: writes slots_per_pos keys
__global__ void gapped_fill(const GapParams P, int64_t n, const int64_t *__restrict__ len,
                            const int64_t *__restrict__ blk, const int64_t *__restrict__ posoff,
                            const uint32_t *__restrict__ bits2, const uint16_t *__restrict__ inv16,
                            int64_t total_pos, unsigned long long *__restrict__ keys) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total_pos) return;
  // row of this position: last row with posoff[row] <= t
  int64_t lo = 0, hi = n;
  while (hi - lo > 1) { int64_t mid = (lo + hi) >> 1; if (posoff[mid] <= t) lo = mid; else hi = mid; }
  const int64_t row = lo, p = t - posoff[row], L = len[row];
  const uint32_t *b2 = bits2 + blk[row] * 4;
  const uint16_t *iv = inv16 + blk[row] * 4;
  unsigned long long *out = keys + t * P.slots_per_pos;
  uint32_t e = 0;                                   // letter j in bits 2j, 2j+1
  int valid = 0;                                    // valid bases from p on
  for (int j = 0; j < P.N && p + j < L; j++) {
    const int64_t idx = p + j;
    if ((iv[idx >> 4] >> (idx & 15)) & 1u) break;
    e |= ((b2[idx >> 4] >> (2 * (idx & 15))) & 3u) << (2 * j);
    valid = j + 1;
  }
  for (int k = P.M; k <= P.N; k++) {
    unsigned long long *o = out + P.slot_off[k];
    const uint32_t nm = kmer_masks(P.R, k);
    for (uint32_t mask = 0; mask < nm; mask++) {
      unsigned long long key = GAP_NONE;
      if (valid >= k) {
        const uint32_t c = kmer_variant_class(P.R, e, k, mask);
        if (c != KMER_NONE) key = ((unsigned long long)row << 40) | (unsigned long long)(P.level_off[k] + c);
      }
      o[mask] = key;
    }
  }
}

__global__ void gapped_mark(const unsigned long long *__restrict__ ukeys, int64_t nu, uint32_t *__restrict__ bitmap) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nu || ukeys[i] == GAP_NONE) return;
  const uint32_t id = (uint32_t)(ukeys[i] & 0xFFFFFFFFFFull);
  atomicOr(bitmap + (id >> 5), 1u << (id & 31));
}

// keep flag per run (class in the set, not the sentinel) and the number of kept runs per row
__global__ void gapped_keep(const unsigned long long *__restrict__ ukeys, int64_t nu, const uint32_t *__restrict__ bitmap,
                            uint32_t *__restrict__ keep, uint32_t *__restrict__ rowcnt) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nu) return;
  uint32_t k = 0;
  if (ukeys[i] != GAP_NONE) {
    const uint32_t id = (uint32_t)(ukeys[i] & 0xFFFFFFFFFFull);
    k = (bitmap[id >> 5] >> (id & 31)) & 1u;
    if (k) atomicAdd(rowcnt + (ukeys[i] >> 40), 1u);
  }
  keep[i] = k;
}

__global__ void gapped_write(const unsigned long long *__restrict__ ukeys, const int *__restrict__ runlen, int64_t nu,
                             const uint32_t *__restrict__ keep, const uint32_t *__restrict__ pos,
                             const uint32_t *__restrict__ bitmap, const uint32_t *__restrict__ rank,
                             uint32_t *__restrict__ col, uint32_t *__restrict__ val) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nu || !keep[i]) return;
  const uint32_t id = (uint32_t)(ukeys[i] & 0xFFFFFFFFFFull), w = bitmap[id >> 5];
  col[pos[i]] = rank[id >> 5] + __popc(w & ((1u << (id & 31)) - 1u));
  if (val) val[pos[i]] = (uint32_t)runlen[i];
}

__global__ void gap_popc_words(const uint32_t *__restrict__ bm, int64_t nw, uint32_t *__restrict__ out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nw) out[i] = __popc(bm[i]);
}
__global__ void gap_enumerate_bits(const uint32_t *__restrict__ bm, const uint32_t *__restrict__ rank, int64_t nw,
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
__global__ void gap_or_ranks(const uint32_t *__restrict__ all, int world, int64_t nw, uint32_t *__restrict__ bm) {
  const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= nw) return;
  uint32_t v = 0;
  for (int r = 0; r < world; r++) v |= all[(int64_t)r * nw + w];
  bm[w] = v;
}

}  // namespace

std::shared_ptr<Matrix> extract_gapped(const kmerlr_config &cfg, std::shared_ptr<SeqSet> seqs, const int32_t *frozen_k,
                                       const uint64_t *frozen_code, int64_t n_frozen, int flags) {
  require_ready();
  const SeqSet &s = *seqs;
  const bool gapped = cfg.alphabet == 1;
  KL_REQUIRE(cfg.M >= 1 && cfg.M <= cfg.N, "need 1 <= M <= N");
  if (gapped) KL_REQUIRE(cfg.N <= GAP_MAX_N, "gapped alphabet: k-mer length above 11 is not supported on the GPU path");
  else KL_REQUIRE(cfg.N <= SORT_MAX_N, "k-mer length above 14 is not supported on the GPU path");
  KL_REQUIRE(s.n < ((int64_t)1 << 24), "sort-based extraction path: at most 2^24 sequences per call");
  const bool sharded = (flags & KMERLR_FLAG_SHARDED) != 0 && ctx().world > 1;
  GapParams P{};
  P.M = cfg.M; P.N = cfg.N;
  P.R = ClassRule{gapped ? 5 : 4, gapped ? cfg.max_ambiguous : -1, cfg.complement != 0, cfg.reverse != 0, cfg.revcomp != 0};
  uint64_t dense = 0, p5 = 1;
  for (int k = 1; k <= cfg.N; k++) {
    p5 *= (uint64_t)P.R.A;
    if (k < cfg.M) continue;
    P.level_off[k] = (uint32_t)dense;
    dense += (p5 + 31) / 32 * 32;
  }
  P.level_off[cfg.N + 1] = (uint32_t)dense;
  const int64_t nbits = (int64_t)dense, nw = nbits / 32;
  P.slots_per_pos = 0;
  for (int k = cfg.M; k <= cfg.N; k++) { P.slot_off[k] = P.slots_per_pos; P.slots_per_pos += gapped ? 1u << (k >= 2 ? k - 2 : 0) : 1u; }
  // positions of every row (host: the lengths are needed for the offsets)
  std::vector<int64_t> len((size_t)s.n), posoff((size_t)s.n + 1, 0);
  s.len.download(len.data(), (size_t)s.n);
  sync_stream();
  for (int64_t i = 0; i < s.n; i++) posoff[i + 1] = posoff[i] + len[i];
  const int64_t total_pos = posoff[s.n], total_slots = total_pos * (int64_t)P.slots_per_pos;
  KL_REQUIRE(total_slots <= ((int64_t)1 << 30), "input too large for the sort-based extraction path (2^30 k-mer instances per call)");

  auto out = std::make_shared<Matrix>();
  out->n = s.n; out->vt = cfg.binarize ? VAL_ONE : VAL_U32;
  out->sharded = sharded; out->n_global = s.n;
  DevBuf<uint32_t> bitmap((size_t)(nw ? nw : 1));
  bitmap.zero();
  int64_t nu = 0;
  DevBuf<unsigned long long> ukeys((size_t)(total_slots ? total_slots : 1));
  DevBuf<int> runlen((size_t)(total_slots ? total_slots : 1));
  if (total_slots > 0) {
    DevBuf<int64_t> dposoff((size_t)s.n + 1);
    dposoff.upload(posoff.data(), (size_t)s.n + 1);
    DevBuf<unsigned long long> keys((size_t)total_slots), sorted((size_t)total_slots);
    KL_LAUNCH(gapped_fill, (unsigned)((total_pos + 127) / 128), 128, 0, P, s.n, s.len.p, s.blk.p, dposoff.p, s.bits2.p,
              s.inv16.p, total_pos, keys.p);
    size_t tb1 = 0, tb2 = 0;
    DevBuf<int> nruns(1);
    KL_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, tb1, keys.p, sorted.p, (int)total_slots, 0, 64, ctx().stream));
    KL_CUDA(cub::DeviceRunLengthEncode::Encode(nullptr, tb2, sorted.p, ukeys.p, runlen.p, nruns.p, (int)total_slots, ctx().stream));
    DevBuf<uint8_t> tmp(tb1 > tb2 ? tb1 : tb2);
    KL_CUDA(cub::DeviceRadixSort::SortKeys(tmp.p, tb1, keys.p, sorted.p, (int)total_slots, 0, 64, ctx().stream));
    ctx().launches += 4;
    KL_CUDA(cub::DeviceRunLengthEncode::Encode(tmp.p, tb2, sorted.p, ukeys.p, runlen.p, nruns.p, (int)total_slots, ctx().stream));
    ctx().launches += 2;
    int hn = 0;
    nruns.download(&hn, 1);
    sync_stream();
    nu = hn;
  }
  // class set: the frozen list or the observed classes (of all ranks)
  if (n_frozen > 0) {
    std::vector<uint32_t> hb((size_t)nw, 0u);
    uint64_t prev = 0;
    for (int64_t j = 0; j < n_frozen; j++) {
      int k = frozen_k[j];
      KL_REQUIRE(k >= cfg.M && k <= cfg.N, "frozen class outside [M,N]");
      uint64_t id = (uint64_t)P.level_off[k] + frozen_code[j];
      KL_REQUIRE(id < (uint64_t)P.level_off[k + 1], "frozen class code out of range");
      KL_REQUIRE(j == 0 || id > prev, "frozen class list must be sorted by (k, code) without duplicates");
      prev = id;
      hb[id >> 5] |= 1u << (id & 31);
    }
    bitmap.upload(hb.data(), (size_t)nw);
    sync_stream();
  } else {
    if (nu > 0) KL_LAUNCH(gapped_mark, (unsigned)((nu + 255) / 256), 256, 0, ukeys.p, nu, bitmap.p);
    if (sharded && nw > 0) {
      DevBuf<uint32_t> all((size_t)(nw * ctx().world));
      comm_allgather_bytes(bitmap.p, all.p, nw * 4);
      KL_LAUNCH(gap_or_ranks, (unsigned)((nw + 255) / 256), 256, 0, all.p, ctx().world, nw, bitmap.p);
    }
  }
  DevBuf<uint32_t> pc((size_t)(nw ? nw : 1)), rank((size_t)nw + 1);
  KL_LAUNCH(gap_popc_words, (unsigned)((nw + 255) / 256), 256, 0, bitmap.p, nw, pc.p);
  exclusive_scan_u32(pc.p, rank.p, nw);
  // kept runs -> CSR
  DevBuf<uint32_t> keep((size_t)(nu ? nu : 1)), pos((size_t)nu + 1), rowcnt((size_t)(s.n ? s.n : 1));
  rowcnt.zero();
  out->rowptr.alloc((size_t)s.n + 1);
  if (nu > 0) {
    KL_LAUNCH(gapped_keep, (unsigned)((nu + 255) / 256), 256, 0, ukeys.p, nu, bitmap.p, keep.p, rowcnt.p);
    exclusive_scan_u32(keep.p, pos.p, nu);
  }
  if (s.n > 0) exclusive_scan_u32_to_i64(rowcnt.p, out->rowptr.p, s.n); else out->rowptr.zero();
  uint32_t m32 = 0;
  KL_CUDA(cudaMemcpyAsync(&m32, rank.p + nw, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx().stream));
  KL_CUDA(cudaMemcpyAsync(&out->nnz, out->rowptr.p + s.n, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx().stream));
  DevBuf<int64_t> nglob(1);
  int64_t nn = s.n;
  if (sharded) {
    nglob.upload(&nn, 1);
    comm_allreduce_sum_i64(nglob.p, 1);
    nglob.download(&nn, 1);
  }
  sync_stream();
  out->m = (int64_t)m32; out->n_global = nn;
  out->col.alloc((size_t)(out->nnz ? out->nnz : 1));
  if (out->vt == VAL_U32) out->val_u32.alloc((size_t)(out->nnz ? out->nnz : 1));
  if (nu > 0)
    KL_LAUNCH(gapped_write, (unsigned)((nu + 255) / 256), 256, 0, ukeys.p, runlen.p, nu, keep.p, pos.p, bitmap.p, rank.p,
              out->col.p, out->vt == VAL_U32 ? out->val_u32.p : (uint32_t *)nullptr);
  // class list
  out->n_classes = (int64_t)m32;
  out->class_ids.alloc((size_t)(m32 ? m32 : 1));
  KL_LAUNCH(gap_enumerate_bits, (unsigned)((nw + 255) / 256), 256, 0, bitmap.p, rank.p, nw, out->class_ids.p);
  out->class_M = cfg.M; out->class_N = cfg.N; out->classes_on_host = false;
  for (int k = cfg.M; k <= cfg.N + 1; k++) out->class_level_off[k] = P.level_off[k];
  sync_stream();
  return out;
}

}  // namespace kl
