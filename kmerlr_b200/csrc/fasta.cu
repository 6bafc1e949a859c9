// fasta.cu -- FASTA text -> resident sequence set on the device, regions cut out of a resident set, and the
// read-back of a set as letters.
//
// Replaces import_fasta (kmerLr_data.go:101-121, gonetics' reader) and the slicing of extractFasta
// (kmerLr_predict_genomic.go:93-112).  The rule (DESIGN §4.7), on bytes:
//   * lines end at '\n' (the last line of a text needs none); a lone '\r' inside a line is a byte of the line;
//   * every line is stripped of leading and trailing ' ', '\t', '\r', '\v', '\f'; empty lines are skipped;
//   * a stripped line starting with '>' begins a record, its name = the rest of the line, stripped;
//   * every other line is appended to the current record as it is (bytes other than a/c/g/t in either case
//     are invalid positions, as pack_kernel treats them); sequence data before the first header of a text is
//     an error, and so is a text that starts with the gzip magic 1f 8b.
// Pipeline (all indices 64-bit): the texts are copied into one buffer with a '\n' after each, so that no line
// crosses a text; the line pass counts '\n' per 4 KiB tile and writes every line end; one thread per line finds
// its stripped bounds and kind; scans give each line's record and its offset in the record's bases; the packing
// locates the line of every 16-base output word by a galloping search over those offsets and reads the bytes
// straight from the text.
#include "common.cuh"

namespace kl {

namespace {

constexpr int TILE_THREADS = 256;
constexpr int64_t TILE_BYTES = TILE_THREADS * 16;

__device__ __forceinline__ bool fasta_space(uint32_t c) {
  return c == ' ' || c == '\t' || c == '\r' || c == '\v' || c == '\f';
}

// last i in [0, n) with a[i] <= key, for non-decreasing a with a[0] <= key: gallop from the guess g to a
// bracket, bisect inside it (a few probes when the guess is close, as for a genome of equal lines)
__device__ __forceinline__ int64_t last_le(const int64_t *__restrict__ a, int64_t n, int64_t key, int64_t g) {
  g = g < 0 ? 0 : (g > n - 1 ? n - 1 : g);
  int64_t lo, hi, step = 1;
  if (a[g] <= key) {
    lo = g; hi = g + 1;
    while (hi < n && a[hi] <= key) { lo = hi; step <<= 1; hi = hi + step < n ? hi + step : n; }
  } else {
    hi = g; lo = g - 1;
    while (lo > 0 && a[lo] > key) { hi = lo; step <<= 1; lo = lo - step > 0 ? lo - step : 0; }
  }
  while (hi - lo > 1) {
    const int64_t mid = (lo + hi) >> 1;
    if (a[mid] <= key) lo = mid; else hi = mid;
  }
  return lo;
}

// sequence of a 64-base block of a set (blk = n + 1 block offsets)
__device__ __forceinline__ int64_t seq_of_block(const int64_t *__restrict__ blk, int64_t n, int64_t total_blocks,
                                                int64_t b) {
  return last_le(blk, n, b, (int64_t)((double)b * (double)n / (double)total_blocks));
}

__device__ __forceinline__ uint32_t newline_mask16(uint4 v, int64_t base, int64_t nbytes) {
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
  uint32_t m = 0;
#pragma unroll
  for (int q = 0; q < 4; q++)
#pragma unroll
    for (int b = 0; b < 4; b++)
      if (((w[q] >> (8 * b)) & 0xFFu) == '\n') m |= 1u << (4 * q + b);
  const int64_t left = nbytes - base;
  if (left < 16) m &= left <= 0 ? 0u : (1u << left) - 1u;
  return m;
}

// ---- line pass: '\n' per tile, then the position of every '\n' -------------------------------------------
__global__ void fasta_count_lines(const uint4 *__restrict__ text, int64_t nbytes, uint32_t *__restrict__ tile_cnt) {
  __shared__ uint32_t part[TILE_THREADS / 32];
  const int64_t base = (int64_t)blockIdx.x * TILE_BYTES + (int64_t)threadIdx.x * 16;
  uint32_t c = 0;
  if (base < nbytes) c = __popc(newline_mask16(text[base >> 4], base, nbytes));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t t = 0;
    for (int w = 0; w < TILE_THREADS / 32; w++) t += part[w];
    tile_cnt[blockIdx.x] = t;
  }
}

__global__ void fasta_line_ends(const uint4 *__restrict__ text, int64_t nbytes, const int64_t *__restrict__ tile_off,
                                int64_t *__restrict__ lend) {
  __shared__ uint32_t part[TILE_THREADS / 32];
  const int64_t base = (int64_t)blockIdx.x * TILE_BYTES + (int64_t)threadIdx.x * 16;
  uint32_t m = 0;
  if (base < nbytes) m = newline_mask16(text[base >> 4], base, nbytes);
  const uint32_t c = __popc(m);
  uint32_t x = c;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
    if ((threadIdx.x & 31) >= (unsigned)o) x += y;
  }
  if ((threadIdx.x & 31) == 31) part[threadIdx.x >> 5] = x;
  __syncthreads();
  uint32_t woff = 0;
  for (int w = 0; w < (int)(threadIdx.x >> 5); w++) woff += part[w];
  int64_t k = tile_off[blockIdx.x] + woff + x - c;
  while (m) {
    const int b = __ffs(m) - 1;
    lend[k++] = base + b;
    m &= m - 1;
  }
}

// ---- per line: stripped bounds, header or sequence, bases kept ------------------------------------------
__global__ void fasta_classify(const uint8_t *__restrict__ text, const int64_t *__restrict__ lend, int64_t L,
                               int64_t *__restrict__ lstart, int64_t *__restrict__ kept, int64_t *__restrict__ hdr) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= L) return;
  int64_t s = i ? lend[i - 1] + 1 : 0, e = lend[i];
  while (s < e && fasta_space(text[s])) s++;
  while (e > s && fasta_space(text[e - 1])) e--;
  const bool h = s < e && text[s] == '>';
  lstart[i] = s;
  kept[i] = h ? 0 : e - s;
  hdr[i] = h ? 1 : 0;
}

// first line of every text (tline[t] = the number of '\n' before the text starts; tline[n_texts] = L) and the
// records of every text from the header ranks
__global__ void fasta_texts(const int64_t *__restrict__ lend, int64_t L, const int64_t *__restrict__ tbase,
                            int64_t n_texts, const int64_t *__restrict__ hrank, int64_t *__restrict__ tline,
                            int64_t *__restrict__ trec) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t > n_texts) return;
  int64_t lo = 0, hi = L;   // lower bound of tbase[t] in lend
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (lend[mid] < tbase[t]) lo = mid + 1; else hi = mid;
  }
  tline[t] = lo;
  trec[t] = hrank[lo];
}

// header line of every record; err = 1 + the first text with sequence data before its first header
__global__ void fasta_records(const int64_t *__restrict__ kept, const int64_t *__restrict__ hdr,
                              const int64_t *__restrict__ hrank, int64_t L, const int64_t *__restrict__ tline,
                              int64_t n_texts, int64_t *__restrict__ hline, unsigned long long *__restrict__ err) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= L) return;
  if (hdr[i]) { hline[hrank[i]] = i; return; }
  if (kept[i] == 0) return;
  int64_t lo = 0, hi = n_texts;   // text of line i: last t with tline[t] <= i
  while (hi - lo > 1) {
    const int64_t mid = (lo + hi) >> 1;
    if (tline[mid] <= i) lo = mid; else hi = mid;
  }
  if (hrank[i] == hrank[tline[lo]]) atomicMin(err, (unsigned long long)lo + 1);
}

// per record: offset of its first base among the kept bytes, length, 64-base blocks, name bounds
__global__ void fasta_record_meta(const uint8_t *__restrict__ text, const int64_t *__restrict__ lend,
                                  const int64_t *__restrict__ lstart, const int64_t *__restrict__ koff,
                                  const int64_t *__restrict__ hline, int64_t nrec, int64_t L,
                                  int64_t *__restrict__ kst, int64_t *__restrict__ len, int64_t *__restrict__ nblk,
                                  int64_t *__restrict__ nst, int64_t *__restrict__ nlen,
                                  unsigned long long *__restrict__ max_len) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= nrec) return;
  const int64_t i0 = hline[r], i1 = r + 1 < nrec ? hline[r + 1] : L;
  const int64_t l = koff[i1] - koff[i0];
  kst[r] = koff[i0];
  len[r] = l;
  nblk[r] = (l + 63) >> 6;
  atomicMax(max_len, (unsigned long long)l);
  int64_t s = lstart[i0] + 1, e = lend[i0];
  while (e > s && fasta_space(text[e - 1])) e--;
  while (s < e && fasta_space(text[s])) s++;
  nst[r] = s;
  nlen[r] = e - s;
}

__global__ void fasta_names(const uint8_t *__restrict__ text, const int64_t *__restrict__ nst,
                            const int64_t *__restrict__ noff, int64_t nrec, uint8_t *__restrict__ out) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= nrec) return;
  const uint8_t *s = text + nst[r];
  uint8_t *d = out + noff[r];
  for (int64_t j = 0, n = noff[r + 1] - noff[r]; j < n; j++) d[j] = s[j];
}

// ---- pack: every 16-base output word from the text ---------------------------------------------------------
__device__ __forceinline__ uint32_t base_code(uint32_t ch, int j, uint32_t &inv) {
  ch |= 0x20u;   // fold case
  if (ch == 'a') return 0;
  if (ch == 'c') return 1;
  if (ch == 'g') return 2;
  if (ch == 't') return 3;
  inv |= 1u << j;
  return 0;
}

__global__ void fasta_pack(const uint8_t *__restrict__ text, const int64_t *__restrict__ lstart,
                           const int64_t *__restrict__ kept, const int64_t *__restrict__ koff, int64_t L,
                           const int64_t *__restrict__ kst, const int64_t *__restrict__ len,
                           const int64_t *__restrict__ blk, int64_t n, int64_t total_blocks,
                           uint32_t *__restrict__ bits2, uint16_t *__restrict__ inv16) {
  const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= total_blocks * 4) return;
  const int64_t r = seq_of_block(blk, n, total_blocks, w >> 2);
  const int64_t j0 = (w - blk[r] * 4) * 16, lr = len[r];
  uint32_t bits = 0, inv = 0;
  if (j0 < lr) {
    const int cnt = lr - j0 < 16 ? (int)(lr - j0) : 16;
    const int64_t k = kst[r] + j0;   // offset among the kept bytes of all records
    int64_t i = last_le(koff, L, k, (int64_t)((double)k * (double)L / (double)koff[L]));
    int64_t pos = lstart[i] + (k - koff[i]), rem = koff[i] + kept[i] - k;
    for (int j = 0; j < cnt; j++) {
      while (rem == 0) { i++; pos = lstart[i]; rem = kept[i]; }
      bits |= base_code(text[pos], j, inv) << (2 * j);
      pos++; rem--;
    }
  }
  bits2[w] = bits;
  inv16[w] = (uint16_t)inv;
}

// ---- regions: row i = bases [from_i, from_i + len_i) of sequence src_i, funnel-shifted out of the packed words
__global__ void regions_pack(const uint32_t *__restrict__ sbits, const uint16_t *__restrict__ sinv,
                             const int64_t *__restrict__ sblk, const int64_t *__restrict__ src,
                             const int64_t *__restrict__ from, const int64_t *__restrict__ len,
                             const int64_t *__restrict__ blk, int64_t n, int64_t total_blocks,
                             uint32_t *__restrict__ bits2, uint16_t *__restrict__ inv16) {
  const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= total_blocks * 4) return;
  const int64_t i = seq_of_block(blk, n, total_blocks, w >> 2);
  const int64_t j0 = (w - blk[i] * 4) * 16;
  uint32_t bits = 0, inv = 0;
  if (j0 < len[i]) {
    const int64_t p = from[i] + j0, q = sblk[src[i]] * 4 + (p >> 4);
    const int sh = (int)(p & 15);
    bits = (uint32_t)((((uint64_t)sbits[q + 1] << 32) | sbits[q]) >> (2 * sh));
    inv = ((((uint32_t)sinv[q + 1] << 16) | sinv[q]) >> sh) & 0xFFFFu;
    const int64_t cnt = len[i] - j0;
    if (cnt < 16) {
      bits &= (1u << (2 * cnt)) - 1u;
      inv &= (1u << cnt) - 1u;
    }
  }
  bits2[w] = bits;
  inv16[w] = (uint16_t)inv;
}

// ---- read-back: the bases of every sequence as a/c/g/t, 'n' at invalid positions ---------------------------
__global__ void letters_kernel(const uint32_t *__restrict__ bits2, const uint16_t *__restrict__ inv16,
                                  const int64_t *__restrict__ blk, const int64_t *__restrict__ len,
                                  const int64_t *__restrict__ soff, int64_t n, int64_t total_blocks,
                                  uint8_t *__restrict__ out) {
  const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= total_blocks * 4) return;
  const int64_t r = seq_of_block(blk, n, total_blocks, w >> 2);
  const int64_t j0 = (w - blk[r] * 4) * 16;
  const uint32_t bits = bits2[w], inv = inv16[w];
  for (int j = 0; j < 16 && j0 + j < len[r]; j++)
    out[soff[r] + j0 + j] = (inv >> j) & 1u ? 'n' : "acgt"[(bits >> (2 * j)) & 3u];
}

unsigned grid_of(int64_t n, int threads) { return (unsigned)((n + threads - 1) / threads); }

template <typename T>
T fetch(const T *dev) {
  T v;
  KL_CUDA(cudaMemcpyAsync(&v, dev, sizeof(T), cudaMemcpyDeviceToHost, ctx().stream));
  sync_stream();
  return v;
}

// bits2 / inv16 of a set whose blk is known: total_blocks words of each + the zero words the kernels read past
// the last base
void alloc_packed(SeqSet &s) {
  const int64_t words = s.total_blocks * 4;
  s.bits2.alloc((size_t)words + 4);
  s.inv16.alloc((size_t)words + 4);
  KL_CUDA(cudaMemsetAsync(s.bits2.p + words, 0, 4 * sizeof(uint32_t), ctx().stream));
  KL_CUDA(cudaMemsetAsync(s.inv16.p + words, 0, 4 * sizeof(uint16_t), ctx().stream));
}

}  // namespace

std::shared_ptr<SeqSet> sequences_from_fasta(const uint8_t *const *texts, const int64_t *nbytes, int64_t n_texts,
                                             int64_t *records_out) {
  require_ready();
  KL_REQUIRE(n_texts >= 0 && (n_texts == 0 || (texts && nbytes && records_out)), "sequences_from_fasta: null argument");
  // text t occupies [tbase[t], tbase[t] + nbytes[t]) of one buffer and is followed by a '\n'
  std::vector<int64_t> tbase((size_t)n_texts + 1, 0);
  for (int64_t t = 0; t < n_texts; t++) {
    KL_REQUIRE(nbytes[t] >= 0 && (nbytes[t] == 0 || texts[t]), "sequences_from_fasta: bad text");
    KL_REQUIRE(!(nbytes[t] >= 2 && texts[t][0] == 0x1f && texts[t][1] == 0x8b),
               "sequences_from_fasta: text " + std::to_string(t) +
                   " is gzip-compressed (starts with 1f 8b); decompress it before the call");
    tbase[t + 1] = tbase[t] + nbytes[t] + 1;
  }
  Trace tr("fasta");
  const int64_t T = tbase[n_texts];
  auto s = std::make_shared<SeqSet>();
  DevBuf<uint8_t> raw((size_t)(T ? T : 1));
  DevBuf<int64_t> dtbase((size_t)n_texts + 1);
  dtbase.upload(tbase.data(), (size_t)n_texts + 1);
  for (int64_t t = 0; t < n_texts; t++) {
    if (nbytes[t])
      KL_CUDA(cudaMemcpyAsync(raw.p + tbase[t], texts[t], (size_t)nbytes[t], cudaMemcpyHostToDevice, ctx().stream));
    KL_CUDA(cudaMemsetAsync(raw.p + tbase[t + 1] - 1, '\n', 1, ctx().stream));
  }
  tr.mark("copy in");
  // lines
  const int64_t ntiles = T ? (T + TILE_BYTES - 1) / TILE_BYTES : 1;
  DevBuf<uint32_t> tile_cnt((size_t)ntiles);
  DevBuf<int64_t> tile_off((size_t)ntiles + 1);
  KL_LAUNCH(fasta_count_lines, (unsigned)ntiles, TILE_THREADS, 0, (const uint4 *)raw.p, T, tile_cnt.p);
  exclusive_scan_u32_to_i64(tile_cnt.p, tile_off.p, ntiles);
  const int64_t L = fetch(tile_off.p + ntiles);   // one line per '\n': every text ends with one
  DevBuf<int64_t> lend((size_t)(L ? L : 1));
  if (L) KL_LAUNCH(fasta_line_ends, (unsigned)ntiles, TILE_THREADS, 0, (const uint4 *)raw.p, T, tile_off.p, lend.p);
  tile_cnt.release(); tile_off.release();
  tr.mark("line pass");
  DevBuf<int64_t> lstart((size_t)L + 1), kept((size_t)L + 1), hdr((size_t)L + 1), koff((size_t)L + 1),
      hrank((size_t)L + 1);
  if (L) {
    KL_LAUNCH(fasta_classify, grid_of(L, 256), 256, 0, raw.p, lend.p, L, lstart.p, kept.p, hdr.p);
    exclusive_scan_i64(hdr.p, hrank.p, L);
    exclusive_scan_i64(kept.p, koff.p, L);
  } else {
    hrank.zero(); koff.zero();
  }
  DevBuf<int64_t> tline((size_t)n_texts + 1), trec((size_t)n_texts + 1);
  DevBuf<unsigned long long> stat(2);   // [0] = 1 + first text with data before a header (0: none), [1] = max length
  KL_CUDA(cudaMemsetAsync(stat.p, 0xFF, sizeof(unsigned long long), ctx().stream));
  KL_CUDA(cudaMemsetAsync(stat.p + 1, 0, sizeof(unsigned long long), ctx().stream));
  KL_LAUNCH(fasta_texts, grid_of(n_texts + 1, 128), 128, 0, lend.p, L, dtbase.p, n_texts, hrank.p, tline.p, trec.p);
  std::vector<int64_t> h2(2);
  KL_CUDA(cudaMemcpyAsync(h2.data(), hrank.p + L, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx().stream));
  KL_CUDA(cudaMemcpyAsync(h2.data() + 1, koff.p + L, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx().stream));
  sync_stream();
  const int64_t nrec = h2[0];
  DevBuf<int64_t> hline((size_t)(nrec ? nrec : 1));
  if (L)
    KL_LAUNCH(fasta_records, grid_of(L, 256), 256, 0, kept.p, hdr.p, hrank.p, L, tline.p, n_texts, hline.p, stat.p);
  const unsigned long long bad = fetch(stat.p);
  if (bad != ~0ull)
    fail(KMERLR_ERR_ARG, "sequences_from_fasta: text " + std::to_string(bad - 1) +
                             " has sequence data before its first header ('>' line)");
  {
    std::vector<int64_t> tr_h((size_t)n_texts + 1);
    trec.download(tr_h.data(), (size_t)n_texts + 1);
    sync_stream();
    for (int64_t t = 0; t < n_texts; t++) records_out[t] = tr_h[t + 1] - tr_h[t];
  }
  tr.mark("lines, records");
  // records
  s->n = nrec;
  s->total_bases = h2[1];
  s->len.alloc((size_t)(nrec ? nrec : 1));
  s->blk.alloc((size_t)nrec + 1);
  DevBuf<int64_t> kst((size_t)(nrec ? nrec : 1)), nblk((size_t)(nrec ? nrec : 1)), nst((size_t)(nrec ? nrec : 1)),
      nlen((size_t)(nrec ? nrec : 1)), noff((size_t)nrec + 1);
  if (nrec) {
    KL_LAUNCH(fasta_record_meta, grid_of(nrec, 256), 256, 0, raw.p, lend.p, lstart.p, koff.p, hline.p, nrec, L, kst.p,
              s->len.p, nblk.p, nst.p, nlen.p, stat.p + 1);
    exclusive_scan_i64(nblk.p, s->blk.p, nrec);
    exclusive_scan_i64(nlen.p, noff.p, nrec);
  } else {
    s->blk.zero(); noff.zero();
  }
  int64_t h3[3];
  KL_CUDA(cudaMemcpyAsync(h3, s->blk.p + nrec, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx().stream));
  KL_CUDA(cudaMemcpyAsync(h3 + 1, stat.p + 1, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx().stream));
  KL_CUDA(cudaMemcpyAsync(h3 + 2, noff.p + nrec, sizeof(int64_t), cudaMemcpyDeviceToHost, ctx().stream));
  sync_stream();
  s->total_blocks = h3[0];
  s->max_len = h3[1];
  tr.mark("record metadata");
  // bases
  alloc_packed(*s);
  if (s->total_blocks)
    KL_LAUNCH(fasta_pack, grid_of(s->total_blocks * 4, 256), 256, 0, raw.p, lstart.p, kept.p, koff.p, L, kst.p,
              s->len.p, s->blk.p, nrec, s->total_blocks, s->bits2.p, s->inv16.p);
  // names: only the header bytes come back
  s->name_off.assign((size_t)nrec + 1, 0);
  s->names.assign((size_t)h3[2], '\0');
  if (h3[2]) {
    DevBuf<uint8_t> names((size_t)h3[2]);
    KL_LAUNCH(fasta_names, grid_of(nrec, 256), 256, 0, raw.p, nst.p, noff.p, nrec, names.p);
    names.download((uint8_t *)&s->names[0], (size_t)h3[2]);
  }
  noff.download(s->name_off.data(), (size_t)nrec + 1);
  sync_stream();
  tr.mark("pack, names");
  return s;
}

std::shared_ptr<SeqSet> sequences_regions(const SeqSet &src, const int64_t *seq_index, const int64_t *from,
                                          const int64_t *to, int64_t n) {
  require_ready();
  KL_REQUIRE(n >= 0 && (n == 0 || (seq_index && from && to)), "sequences_regions: null argument");
  std::vector<int64_t> slen((size_t)src.n);
  src.len.download(slen.data(), (size_t)src.n);
  sync_stream();
  auto s = std::make_shared<SeqSet>();
  s->n = n;
  std::vector<int64_t> len((size_t)(n ? n : 1), 0), blk((size_t)n + 1, 0);
  for (int64_t i = 0; i < n; i++) {
    KL_REQUIRE(seq_index[i] >= 0 && seq_index[i] < src.n,
               "sequences_regions: region " + std::to_string(i) + ": sequence index " + std::to_string(seq_index[i]) +
                   " out of range [0, " + std::to_string(src.n) + ")");
    const int64_t l = slen[(size_t)seq_index[i]];
    KL_REQUIRE(from[i] >= 0 && from[i] <= to[i] && to[i] <= l,
               "sequences_regions: region " + std::to_string(i) + ": [" + std::to_string(from[i]) + ", " +
                   std::to_string(to[i]) + ") is not a slice of sequence " + std::to_string(seq_index[i]) +
                   " (length " + std::to_string(l) + ")");
    len[(size_t)i] = to[i] - from[i];
    blk[(size_t)i + 1] = blk[(size_t)i] + ((len[(size_t)i] + 63) >> 6);
    s->total_bases += len[(size_t)i];
    s->max_len = len[(size_t)i] > s->max_len ? len[(size_t)i] : s->max_len;
  }
  s->total_blocks = blk[(size_t)n];
  s->len.alloc(len.size());
  s->len.upload(len.data(), len.size());
  s->blk.alloc((size_t)n + 1);
  s->blk.upload(blk.data(), (size_t)n + 1);
  alloc_packed(*s);
  if (s->total_blocks) {
    DevBuf<int64_t> dsrc((size_t)n), dfrom((size_t)n);
    dsrc.upload(seq_index, (size_t)n);
    dfrom.upload(from, (size_t)n);
    KL_LAUNCH(regions_pack, grid_of(s->total_blocks * 4, 256), 256, 0, src.bits2.p, src.inv16.p, src.blk.p, dsrc.p,
              dfrom.p, s->len.p, s->blk.p, n, s->total_blocks, s->bits2.p, s->inv16.p);
    sync_stream();   // dsrc / dfrom and the host arrays are freed on return
  } else {
    sync_stream();
  }
  return s;
}

void sequences_letters(const SeqSet &s, char *out) {
  require_ready();
  if (s.total_bases == 0) return;
  DevBuf<int64_t> soff((size_t)s.n + 1);
  exclusive_scan_i64(s.len.p, soff.p, s.n);
  DevBuf<uint8_t> dout((size_t)s.total_bases);
  KL_LAUNCH(letters_kernel, grid_of(s.total_blocks * 4, 256), 256, 0, s.bits2.p, s.inv16.p, s.blk.p, s.len.p,
            soff.p, s.n, s.total_blocks, dout.p);
  dout.download((uint8_t *)out, (size_t)s.total_bases);
  sync_stream();
}

}  // namespace kl
