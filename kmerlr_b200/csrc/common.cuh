// common.cuh -- shared infrastructure of libkmerlr_b200.so (context, errors, device buffers,
// matrix / sequence objects, small device helpers).  sm_100a only.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "../../include/kmerlr_b200.h"

namespace kl {

// ---------------------------------------------------------------------------------------------
// errors: C++ exceptions inside, status codes at the C ABI (reference style: log.Fatal for
// argument / IO errors, panic("internal error") for invariants -- SURVEY 8b)
// ---------------------------------------------------------------------------------------------
struct Error {
  int code;
  std::string msg;
};

[[noreturn]] inline void fail(int code, const std::string &msg) { throw Error{code, msg}; }

#define KL_CUDA(expr)                                                                              \
  do {                                                                                             \
    cudaError_t _e = (expr);                                                                       \
    if (_e != cudaSuccess)                                                                         \
      ::kl::fail(KMERLR_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e) + " (" +      \
                                      __FILE__ + ":" + std::to_string(__LINE__) + ")");            \
  } while (0)

#define KL_REQUIRE(cond, msg)                                                                      \
  do {                                                                                             \
    if (!(cond)) ::kl::fail(KMERLR_ERR_ARG, std::string(msg));                                     \
  } while (0)

#define KL_INVARIANT(cond)                                                                         \
  do {                                                                                             \
    if (!(cond)) ::kl::fail(KMERLR_ERR_INTERNAL, std::string("internal error: ") + #cond + " (" +  \
                                                     __FILE__ + ":" + std::to_string(__LINE__) + ")"); \
  } while (0)

// ---------------------------------------------------------------------------------------------
// context: one process drives one GPU
// ---------------------------------------------------------------------------------------------
// Mailboxes of the peer-memory exchange: rank r's mailbox holds, for both parities of the sequence
// number, one payload slot per sender and one flag per sender (the sender's sequence number).
constexpr int PEER_MAX_WORLD = 8;
constexpr int PEER_PAYLOAD = 1024 + 8;          // 64-bit words per slot
struct PeerMail {
  unsigned long long slot[2][PEER_MAX_WORLD][PEER_PAYLOAD];
  unsigned long long flag[2][PEER_MAX_WORLD];
  unsigned long long seq;                        // local: sequence number of the last exchange
  unsigned int senders_done;                     // local: sender blocks of the running exchange that are through
  // all-reduce over peer memory (comm.cu: p2p_allreduce_kernel): two barriers per exchange
  unsigned long long ar_flag[2][PEER_MAX_WORLD]; // ar_flag[b][s] = sequence number of sender s at barrier b
  unsigned long long ar_seq;                     // local: sequence number of the last all-reduce
  unsigned int ar_error;                         // local: a peer did not show up at a barrier
};
constexpr int64_t PEER_AR_CAP = (int64_t)4 << 20;   // 64-bit words per all-reduce over peer memory (32 MB in, 32 MB out)
struct PeerBox {
  PeerMail *box[PEER_MAX_WORLD];                 // box[r] = rank r's mailbox as mapped into this process
  unsigned long long *sym[PEER_MAX_WORLD];       // sym[r] = rank r's all-reduce buffer: IN[PEER_AR_CAP] then OUT[PEER_AR_CAP]
  int rank, world;
};

constexpr int CTX_COPY_EVENTS = 11;   // chunks of a pipelined host feed + 1
struct Numbering;
struct Ctx {
  bool ready = false;
  int device = 0;
  int sm_count = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr;            // host -> device feeds overlapping the kernels
  cudaStream_t alt_stream = nullptr;             // odd chunks of a pipelined feed: their kernels overlap the tails of the even ones
  cudaEvent_t join_ev[2] = {nullptr, nullptr};
  cudaEvent_t copy_ev[CTX_COPY_EVENTS] = {nullptr};
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  // pinned host staging of the small per-call transfers (labels, theta, iteration state): see host_staging()
  void *staging = nullptr;
  size_t staging_bytes = 0;
  cudaEvent_t staging_ev = nullptr;              // recorded after the last transfer that used the staging buffer
  // numbering sets of every class a configuration can produce, one per (M, N, strand op) seen (extract.cu)
  std::vector<std::shared_ptr<const Numbering>> numbering;
  int64_t launches = 0;
  double last_ms = 0.0;
  bool profiling = false;
  bool implicit_ok = true;   // kmerlr_option("implicit")
  int super_len = -1;        // kmerlr_option("super_len"): length of the super k-mer tables (-1 = automatic, 0 = off)
  int hot_cols = 6144;       // kmerlr_option("hot_cols"): columns of the CSR pass that accumulate in shared memory
  int fused_ticket = 8;      // kmerlr_option("fused_ticket"): rows per ticket of the CSR pass (0 = static grid); measured
                             // at C3 / C2 per iteration: 8: 16.2 / 3.07 ms, 32: 16.7, 128: 19.8, static: 16.7 / 3.49 ms
  // communicator (NCCL via dlopen, see comm.cu)
  void *comm = nullptr;
  int rank = 0, world = 1;
  // peer-memory exchange over NVLink (comm.cu): every rank owns one mailbox, mapped into all ranks
  PeerBox *peer = nullptr;   // device copy of the mailbox table, nullptr = not available (NCCL is used)
  bool p2p_ok = true;        // kmerlr_option("p2p")
  bool p2p_allreduce = false; // kmerlr_option("p2p_allreduce"): full-space gradient all-reduce over peer memory instead of NCCL
  int feed_growth = 135;     // kmerlr_option("feed_growth"): growth of the chunk sizes of a host feed, per cent
  int small_long = -1;       // kmerlr_option("small_long"): reduced-matrix solver on the sliced + column-major layouts (1), on the rows (0), by row length (-1)
  int persist_bps = 0;       // kmerlr_option("persist_bps"): blocks per SM of the persistent reduced-matrix solver (0 = all that fit)
  bool coop_supported = true;
  bool coop_ok = true;       // kmerlr_option("persistent"); false when the device cannot launch cooperatively
};
Ctx &ctx();
void require_ready();

// per-kernel device timing (bench.py: roofline of the dominant kernel, measured with CUDA events on
// the launching stream); off by default
void profile_begin(const char *name);
void profile_end();

// launch helper: counts launches (bench.py reports gpu_launches) and checks the launch
#define KL_LAUNCH(kernel, grid, block, smem, ...)                                                  \
  do {                                                                                             \
    if (::kl::ctx().profiling) ::kl::profile_begin(#kernel);                                       \
    kernel<<<(grid), (block), (smem), ::kl::ctx().stream>>>(__VA_ARGS__);                          \
    if (::kl::ctx().profiling) ::kl::profile_end();                                                \
    ::kl::ctx().launches++;                                                                        \
    KL_CUDA(cudaGetLastError());                                                                   \
  } while (0)

inline void sync_stream() { KL_CUDA(cudaStreamSynchronize(ctx().stream)); }

// Pinned host buffer of at least `bytes` (grown on demand, owned by the context) for copies on ctx().stream:
// copies from and to pageable memory stage through a driver buffer and block the host.  The caller records
// the end of its copies with host_staging_done(); the next host_staging() waits for them before it hands the
// buffer out again.
void *host_staging(size_t bytes);
inline void host_staging_done() { KL_CUDA(cudaEventRecord(ctx().staging_ev, ctx().stream)); }

// KMERLR_TRACE=1: host-side phase timestamps on stderr (where does a call spend its wall time)
struct Trace {
  bool on;
  std::chrono::steady_clock::time_point t0, last;
  const char *what;
  explicit Trace(const char *w) : what(w) {
    static int env = -1;
    if (env < 0) { const char *e = getenv("KMERLR_TRACE"); env = (e && *e == '1') ? 1 : 0; }
    on = env == 1;
    if (on) t0 = last = std::chrono::steady_clock::now();
  }
  void mark(const char *phase, bool sync = true) {
    if (!on) return;
    if (sync) cudaStreamSynchronize(ctx().stream);
    auto t = std::chrono::steady_clock::now();
    fprintf(stderr, "[trace %s] %-28s %8.3f ms (total %8.3f)\n", what, phase,
            std::chrono::duration<double, std::milli>(t - last).count(),
            std::chrono::duration<double, std::milli>(t - t0).count());
    last = t;
  }
};

// ---------------------------------------------------------------------------------------------
// device buffer (RAII)
// ---------------------------------------------------------------------------------------------
void *arena_alloc(size_t bytes);
void arena_free(void *p);
void arena_release_all();

template <typename T>
struct DevBuf {
  T *p = nullptr;
  size_t n = 0;
  DevBuf() = default;
  explicit DevBuf(size_t count) { alloc(count); }
  DevBuf(const DevBuf &) = delete;
  DevBuf &operator=(const DevBuf &) = delete;
  DevBuf(DevBuf &&o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
  DevBuf &operator=(DevBuf &&o) noexcept {
    if (this != &o) { release(); p = o.p; n = o.n; o.p = nullptr; o.n = 0; }
    return *this;
  }
  ~DevBuf() { release(); }
  // device memory comes from a caching arena (abi.cu): freed blocks are kept and handed out again,
  // so that after the first step no call reaches the driver's allocator.  Everything runs on one
  // stream, which makes reuse safe without events.
  void alloc(size_t count) {
    release();
    n = count;
    if (count) p = (T *)arena_alloc(count * sizeof(T) + 32);   // + 32: kernels read whole aligned 16-byte groups
  }
  void release() {
    if (p) arena_free(p);
    p = nullptr; n = 0;
  }
  void zero() { if (n) KL_CUDA(cudaMemsetAsync(p, 0, n * sizeof(T), ctx().stream)); }
  void upload(const T *h, size_t count) {
    if (count) KL_CUDA(cudaMemcpyAsync(p, h, count * sizeof(T), cudaMemcpyHostToDevice, ctx().stream));
  }
  void download(T *h, size_t count) const {
    if (count) KL_CUDA(cudaMemcpyAsync(h, p, count * sizeof(T), cudaMemcpyDeviceToHost, ctx().stream));
  }
  size_t bytes() const { return n * sizeof(T); }
};

// ---------------------------------------------------------------------------------------------
// objects behind handles
// ---------------------------------------------------------------------------------------------
struct Object {
  virtual ~Object() {}
};

// 2-bit packed sequences resident in HBM.  Every sequence starts on a 64-base block
// (16 B of codes + 8 B of invalid mask); base j of sequence i is bits [2(j&15), 2(j&15)+1] of
// bits2[blk[i]*4 + (j>>4)], its "not ACGT" flag is bit (j&15) of inv16[blk[i]*4 + (j>>4)].
struct SeqSet : Object {
  int64_t n = 0;
  int64_t total_bases = 0;
  int64_t total_blocks = 0;
  int64_t max_len = 0;
  DevBuf<int64_t> len;      // n
  DevBuf<int64_t> blk;      // n+1, in 64-base blocks
  DevBuf<uint32_t> bits2;   // total_blocks*4
  DevBuf<uint16_t> inv16;   // total_blocks*4
  // record names of a set parsed from FASTA text (fasta.cu): name i = names[name_off[i], name_off[i+1]); empty
  // for every other set
  std::string names;
  std::vector<int64_t> name_off;
  // a row subset's set (subset.cu): len / blk are gathered from the set `words`, whose packed words they point into
  // (bits2 / inv16 stay empty here).  Its rows need not tile the words, so only the matrix-free logistic pass reads
  // it; it is never handed out as a handle.  nullptr: the set owns its words.
  std::shared_ptr<const SeqSet> words;
  const SeqSet &word_owner() const { return words ? *words : *this; }
};

enum ValType : int { VAL_ONE = 0, VAL_U32 = 1, VAL_F64 = 2 };

// What the matrix-free logistic pass needs (logistic.cu).  A matrix that came straight out of the
// extraction (one column per observed / frozen class) is a function of the k-mer occurrences, so X theta
// and X^T w can be evaluated from the packed sequences instead of the stored rows:
//   * count matrices: linear in the occurrences, every level M..N is matrix-free (Mlo = M);
//   * binarized matrices: the table levels (k <= 5, where nearly every class repeats) are a per-row bitmap
//     over the classes of those levels (lowbits), the levels k >= 6 are matrix-free with one correction per
//     REPEAT of a class inside a row (the events the extraction leaves at the tail of the row's slots).
// The numbering set of an extraction: the classes that get a column (column = rank of the class among them) as a
// bitmap over the dense class ids, the rank of every word's first bit (rank[nw] = count), and both interleaved for
// the extraction kernel.  Never changed once built: the set of every class of an unfrozen configuration depends
// on (M, N, strand op) only, so the context keeps one per configuration and the matrices share it.
struct Numbering {
  int M = 0, N = 0, op = 0;
  int64_t nw = 0;
  uint32_t count = 0;
  DevBuf<uint32_t> bits, rank;     // nw, nw + 1
  DevBuf<uint2> nbx;               // nw (empty for the observed-class sets of a renumbered matrix)
};

constexpr int IMP_MAX_N = 10;      // forward-code tables of 4^1 + ... + 4^N entries
constexpr int IMP_SUPER_MAX = 11;  // longest "super k-mer" table (4^11 entries of 8 bytes = 32 MB)
constexpr uint32_t NOCOL = 0xFFFFFFFFu;
struct Implicit {
  std::shared_ptr<SeqSet> seqs;
  int M = 0, N = 0, op = 0;
  int Mlo = 0;                     // first matrix-free level (>= M)
  uint32_t level_off[16] = {0};    // dense class id of (k, code 0)
  uint32_t fo[16] = {0};           // offset of level j (Mlo..N) in the forward-code tables, fo[N+1] = total
  std::shared_ptr<const Numbering> num;   // class set over dense ids: column = rank[id>>5] + popc(bits below)
  // binarized matrices only
  bool binarized = false;
  int low_words = 0;               // 32-bit words of a row's bitmap over the table-level classes
  DevBuf<uint32_t> lowbits;        // n * low_words
  DevBuf<uint32_t> lowcol;         // low_words * 32: column of the j-th table-level class (NOCOL: not a column)
  DevBuf<int64_t> evptr;           // n + 1: the repeat events of row i are events[evptr[i] .. evptr[i+1])
  DevBuf<uint32_t> events;         // the column of the repeated class, once per repeat
};                                 // (the dense class id of every column is Matrix::class_ids)

// where row i of a matrix lives: compact CSR (rowptr) or fixed-stride rows straight from the extraction
struct Rows {
  const int64_t *rowptr;     // compact: row i = [rowptr[i], rowptr[i+1])
  const uint32_t *rowcnt;    // padded:  row i = [i*stride, i*stride + rowcnt[i])
  int64_t stride;            // 0 = compact
#ifdef __CUDACC__
  __device__ __forceinline__ void range(int64_t row, int64_t &a, int64_t &b) const {
    if (stride) { a = row * stride; b = a + rowcnt[row]; }
    else { a = rowptr[row]; b = rowptr[row + 1]; }
  }
#endif
};

// KmerDataSet in HBM: sparse rows (without the bias column) + labels + classes; a CSC view is built
// lazily for the pair-feature (co-occurrence) gradient only.  Matrices that come out of the extraction
// keep the fixed-stride row layout the kernel wrote (no second copy); matrix_compact() turns them into
// compact CSR for the few consumers that need contiguous entries (export, CSC transpose).
struct Matrix : Object {
  int64_t n = 0, m = 0, nnz = 0;
  ValType vt = VAL_U32;
  int64_t row_stride = 0;    // > 0: padded rows, rowcnt valid, rowptr unused
  DevBuf<uint32_t> rowcnt;   // n (padded layout)
  DevBuf<int64_t> rowptr;    // n+1 (compact layout)
  DevBuf<uint32_t> col;      // nnz, or n*row_stride
  DevBuf<uint32_t> val_u32;  // (VAL_U32)
  DevBuf<double> val_f64;    // (VAL_F64)
  Rows rows() const { return Rows{rowptr.p, rowcnt.p, row_stride}; }
  // CSC view (built on first use by ensure_csc): entries of column c in ascending row order
  bool has_csc = false;
  DevBuf<int64_t> colptr;    // m+1
  DevBuf<uint32_t> crow;     // nnz
  DevBuf<uint32_t> cval_u32;
  DevBuf<double> cval_f64;
  // sliced view (built on first use by ensure_sliced): slices of 32 rows, entry k of the 32 rows side by side
  // (entry k of row r at slice_off[r / 32] + 32 k + r % 32), so that one thread per row reads coalesced
  bool has_sliced = false;
  DevBuf<int64_t> slice_off;   // n/32 + 1
  DevBuf<uint32_t> scol;
  DevBuf<uint32_t> sval_u32;
  DevBuf<double> sval_f64;
  // both views with the count packed beside the index, one 32-bit word per entry (ensure_packed; counts and at
  // most 1 024 columns only): sliced = column | count << 10, column-major = row | count << pack_row_bits
  bool has_packed = false, packable = false;
  int pack_row_bits = 0;
  DevBuf<uint32_t> spack, cpack;
  // block-local column-major view for the persistent reduced-matrix solver (ensure_blockview): block b of a grid of
  // bv_grid blocks owns the rows [n b / bv_grid, n (b+1) / bv_grid); its entries, sorted by (column, row), are dealt
  // to the 256 threads of the block in contiguous shares of width_b entries and stored share-interleaved (entry j of
  // thread t at 256 (bv_off[b] + j) + t), one word each: local row | column << bv_row_bits | count << (bv_row_bits
  // + 10); 0xFFFFFFFF pads the last shares
  int bv_grid = 0, bv_row_bits = 0, bv_rows = 0;
  bool bv_ok = false;
  DevBuf<int64_t> bv_off;
  DevBuf<uint32_t> bv_pack;
  // labels
  bool has_labels = false;
  DevBuf<uint8_t> labels;    // n
  int64_t n_pos = 0, n_neg = 0;   // label counts: this rank's until matrix_label_counts() has summed them over the ranks
  bool counts_global = true;
  bool counts_pending = false;    // n_pos is still on the device (label_ones), read when somebody needs the counts
  DevBuf<unsigned long long> label_ones;
  // class list: dense class ids on the device (extraction), decoded to (k, code) on the host the first
  // time somebody asks (matrix_class_list)
  int64_t n_classes = 0;
  DevBuf<uint32_t> class_ids;
  int class_M = 0, class_N = 0;
  uint32_t class_level_off[16] = {0};
  bool classes_on_host = true;
  std::vector<int32_t> class_k;
  std::vector<uint64_t> class_code;
  // sample sharding
  bool sharded = false;
  int64_t n_global = 0;
  // cached max_i ||x_i||^2 (without bias) and max |x_ij|, global
  bool has_maxsq = false;
  double maxsq = 0.0;
  bool has_vmax = false;
  double vmax = 0.0;
  // cached max_i ||x~_i||^2 of the pair-expanded rows x~ = (v_j)_j u (v_a v_b)_{a<b} (pair mode's step size)
  bool has_maxsq_pairs = false;
  double maxsq_pairs = 0.0;
  // matrix-free view (count matrices produced by extract() without an explicit feature list)
  std::shared_ptr<Implicit> imp;
  // the same two numbers over this rank's rows, when the kernel that wrote the rows computed them
  bool has_local_stats = false;
  double local_maxsq = 0.0, local_vmax = 0.0;
};

// handle registry (abi.cu)
uint64_t register_object(std::shared_ptr<Object> o);
std::shared_ptr<Object> lookup_object(uint64_t h);
template <typename T>
std::shared_ptr<T> lookup(uint64_t h, const char *what) {
  auto o = std::dynamic_pointer_cast<T>(lookup_object(h));
  if (!o) fail(KMERLR_ERR_ARG, std::string("invalid ") + what + " handle");
  return o;
}

// ---------------------------------------------------------------------------------------------
// module entry points (one .cu file each)
// ---------------------------------------------------------------------------------------------
// scan.cu
void exclusive_scan_i64(const int64_t *in, int64_t *out, int64_t n);            // out[n] = total
void exclusive_scan_u32_to_i64(const uint32_t *in, int64_t *out, int64_t n);    // out[n] = total
void exclusive_scan_u32(const uint32_t *in, uint32_t *out, int64_t n);          // out[n] = total
// the same scan queued on the stream with a caller-owned workspace of exclusive_scan_workspace(n) words: no
// allocation and no synchronisation (a solver's iteration scans without a host round trip)
int64_t exclusive_scan_workspace(int64_t n);
void exclusive_scan_u32_async(const uint32_t *in, uint32_t *out, int64_t n, int64_t *workspace);
// extract.cu
std::shared_ptr<SeqSet> sequences_create(const uint8_t *seq, const int64_t *off, int64_t n);
// host sequences that arrive in chunks of whole rows: feed(c) copies chunk c on the copy stream and packs it on the
// main stream (asynchronously; c < 0: everything); rows [first_row(c), first_row(c + 1))
struct SeqFeed {
  virtual ~SeqFeed() {}
  virtual int chunks() const = 0;
  virtual int64_t first_row(int c) const = 0;
  virtual void feed(int c) = 0;
};
std::shared_ptr<SeqSet> sequences_begin_chunked(const uint8_t *seq, const int64_t *off, int64_t n, std::unique_ptr<SeqFeed> &feed);
std::shared_ptr<Matrix> extract(const kmerlr_config &cfg, std::shared_ptr<SeqSet> seqs, const int32_t *frozen_k,
                                const uint64_t *frozen_code, int64_t n_frozen, const int32_t *features,
                                int64_t n_features, int flags);
std::shared_ptr<Matrix> extract_host(const kmerlr_config &cfg, const uint8_t *seq, const int64_t *off, int64_t n,
                                     const int32_t *frozen_k, const uint64_t *frozen_code, int64_t n_frozen,
                                     const int32_t *features, int64_t n_features, int flags);
// fasta.cu
std::shared_ptr<SeqSet> sequences_from_fasta(const uint8_t *const *texts, const int64_t *nbytes, int64_t n_texts,
                                             int64_t *records_out);
std::shared_ptr<SeqSet> sequences_regions(const SeqSet &src, const int64_t *seq_index, const int64_t *from,
                                          const int64_t *to, int64_t n);
void sequences_letters(const SeqSet &s, char *out);   // total_bases bytes: a/c/g/t, 'n' at invalid positions
// gapped.cu
std::shared_ptr<Matrix> extract_gapped(const kmerlr_config &cfg, std::shared_ptr<SeqSet> seqs, const int32_t *frozen_k,
                                       const uint64_t *frozen_code, int64_t n_frozen, int flags);
void matrix_class_list(Matrix &M);   // fills class_k / class_code if they are still on the device
// matrix.cu
std::shared_ptr<Matrix> matrix_from_csr(int64_t n, int64_t m, const int64_t *rowptr, const int32_t *col,
                                        const double *val, int flags);
void matrix_rows(Matrix &M, int64_t *rowptr, int32_t *col, double *val);
void matrix_set_labels(Matrix &M, const uint8_t *labels, int64_t n);
void matrix_label_counts_local(Matrix &M);   // n_pos / n_neg of this rank's rows on the host
void matrix_label_counts(Matrix &M);   // n_pos / n_neg over all ranks (collective on a sharded matrix, first call only)
void matrix_column_moments(Matrix &M, double *sum, double *sumsq, double *absmax, int64_t *count);
void matrix_pair_moments(Matrix &M, double *sum, double *sumsq, double *absmax, int64_t *count);   // m (m - 1) / 2 pairs
std::shared_ptr<Matrix> matrix_transform(Matrix &M, const double *offset, const double *scale, int64_t len);
void matrix_compact(Matrix &M);      // padded rows -> compact CSR (no-op for compact matrices)
void ensure_csc(Matrix &M);
void ensure_sliced(Matrix &M);
bool ensure_packed(Matrix &M);      // false: the entries do not fit (real values, large counts, > 1 024 columns)
bool ensure_blockview(Matrix &M, int grid);   // false: rows per block / counts do not fit the packed word
std::shared_ptr<Matrix> matrix_reduce(Matrix &M, const int64_t *sel, int64_t nsel);
// subset.cu
std::shared_ptr<Matrix> matrix_subset(Matrix &M, const int64_t *rows, int64_t nrows);
double matrix_maxsq(Matrix &M);
double matrix_maxsq_pairs(Matrix &M);   // max_i ||x~_i||^2 of the pair-expanded rows (one GPU)
double matrix_vmax(Matrix &M);
// logistic.cu
void linear_pdf(Matrix &M, const double *theta, int64_t ntheta, int cooc, double *out_host, bool logpdf);
void gradient(Matrix &M, const double *theta, int64_t ntheta, const double cw[2], double lambda, int cooc,
              double *g_host, DevBuf<double> *g_dev = nullptr);   // g_dev: the gradient stays on the device
double loss(Matrix &M, const double *theta, int64_t ntheta, const double cw[2], double lambda, int cooc);
void coordinate(Matrix &M, double *theta, int64_t ntheta, const double cw_hook[2], double l1reg, double l2reg,
                double epsilon, double epsilon_loss, int64_t max_iter, double hook[2], int64_t *sweeps_out,
                double *delta_out);
void proxgrad(Matrix &M, double *theta, int64_t ntheta, const double cw[2], double lambda, double l2,
              double step_factor, double epsilon, double epsilon_loss, int64_t max_iter, double hook[2],
              int64_t *iters, double *delta);
void proxgrad_accel(Matrix &M, double *theta, double *y, double *t, int64_t ntheta, const double cw[2], double lambda,
                    double l2, double step_factor, double epsilon, double epsilon_loss, int64_t max_iter, double hook[2],
                    int64_t *iters, double *delta, int64_t *restarts);
void proxgrad_accel_full(Matrix &M, double *theta, double *y, double *t, int64_t ntheta, const double cw[2],
                         double lambda, double l2, double step_factor, double epsilon, double epsilon_loss,
                         int64_t max_iter, double hook[2], int64_t *iters, double *delta, int64_t *restarts);
void proxgrad_pairs(Matrix &M, double *theta, int64_t ntheta, const double cw[2], double lambda, double l2,
                    double step_factor, double epsilon, double epsilon_loss, int64_t max_iter, double hook[2],
                    int64_t *iters, double *delta);
void proxgrad_pairs_accel(Matrix &M, double *theta, double *y, double *t, int64_t ntheta, const double cw[2],
                          double lambda, double l2, double step_factor, double epsilon, double epsilon_loss,
                          int64_t max_iter, double hook[2], int64_t *iters, double *delta, int64_t *restarts);
// select.cu
void select(Matrix &M, const double cw[2], int cooc, int64_t N, double theta0, const int64_t *active_idx,
            const double *active_theta, int64_t n_active, int tie, double eps_lambda, double prev_lambda,
            uint8_t *mask, int64_t ntheta, double *lambda_out, int64_t *c_out, int *ok_out, double *g_out);
void select_from_gradient(const double *g, int64_t ntheta, int64_t N, const int64_t *active_idx, const double *active_theta,
                          int64_t n_active, int tie, double eps_lambda, double prev_lambda, uint8_t *mask,
                          double *lambda_out, int64_t *c_out, int *ok_out);
// score.cu
void score_windows(const kmerlr_model *models, int n_models, const SeqSet &s, int64_t W, int64_t step,
                   double *out_host, std::shared_ptr<Object> *out_dev, int layout = 0, SeqFeed *feed = nullptr);
// formats.cu: the on-disk formats either side of the path
int64_t wiggle_records(const double *pred, bool pred_on_device, int64_t n, char *out);
void save_wiggle(const char *filename, const char *track_name, int64_t n_regions, const char *const *seqnames,
                 const int64_t *from, const int64_t *slot_off, const double *pred, bool pred_on_device, int64_t window_size,
                 int64_t window_step);
std::string class_name(const kmerlr_config &cfg, int k, uint64_t code);
void export_kmers(Matrix &M, const kmerlr_config &cfg, const char *filename, bool as_float);
void export_path(const char *filename, int64_t n, const int64_t *estimator, const double *lambda, const double *norm,
                 const int64_t *theta_off, const double *theta);
void export_trace(const char *filename, int64_t n, const int64_t *duration_ns, const int64_t *iteration, const double *change,
                  const int64_t *nonzero, const double *lambda, const double *loss);

// comm.cu
void comm_unique_id(void *id128);
void comm_init(int rank, int world, const void *id128);
void comm_destroy();
void comm_allreduce_sum_f64(double *dev, int64_t count);
void comm_allreduce_sum_i64(int64_t *dev, int64_t count);
void comm_allreduce_sum_i64_fast(int64_t *dev, int64_t count);   // over NVLink peer memory when available, else NCCL
void comm_check_peer_errors();                                   // throws when a peer-memory all-reduce timed out
void comm_allreduce_max_f64(double *dev, int64_t count);
void comm_allreduce_max_u8(uint8_t *dev, int64_t count);
void comm_allgather_f64(const double *dev_in, double *dev_out, int64_t count_per_rank);
void comm_allgather_bytes(const void *dev_in, void *dev_out, int64_t bytes_per_rank);

// exponent e of the fixed-point sums (scale 2^e): 60 - ceil(log2(bound)), so a sum bounded by `bound` stays below
// 2^60.  Clamped so that 2^e and 2^-e stay finite; a bound of 0 (an empty matrix) takes the exponent of 1
inline int fixed_point_exponent(double bound) {
  if (!(bound > 0.0) || !std::isfinite(bound)) bound = 1.0;
  const int e = 60 - (int)std::ceil(std::log2(bound));
  return e > 1000 ? 1000 : e;
}

// ---------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ unsigned lane_id() { return threadIdx.x & 31u; }
__device__ __forceinline__ unsigned lanemask_lt() {
  unsigned m;
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
  return m;
}
__device__ __forceinline__ uint32_t swap_pairs(uint32_t y) {
  return ((y >> 1) & 0x55555555u) | ((y & 0x55555555u) << 1);
}
// image of the k-mer code u under the strand operation (1 revcomp, 2 complement, 3 reverse)
__device__ __forceinline__ uint32_t kmer_op(uint32_t u, int k, int op) {
  if (op == 1) return swap_pairs(__brev(~u)) >> (32 - 2 * k);
  if (op == 2) return (~u) & ((1u << (2 * k)) - 1u);
  return swap_pairs(__brev(u)) >> (32 - 2 * k);
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
// reduction in a fixed order that depends only on the lane layout (deterministic)
__device__ __forceinline__ double warp_sum_down(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}
// ---- TMA bulk copy (cp.async.bulk, 1-D: no tensor map) global -> shared, completion on an mbarrier -------------
// dst, src 16-byte aligned, bytes a multiple of 16.  One thread arms the barrier with the byte count and issues the
// copy; every consumer waits on the barrier's phase.
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, uint32_t arrivals) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(arrivals) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void bulk_copy_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, unsigned long long *bar) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "KL_MBAR_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra KL_MBAR_DONE;\n"
      "bra KL_MBAR_WAIT;\n"
      "KL_MBAR_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}

// log(1+exp(x)) with a = 0: LogAdd(0, x) of autodiff's logarithmetic package, restated as
// max(0,x) + log1p(exp(-|x|))  (kmerLr_logistic_regression.go:138-145)
__device__ __forceinline__ double log_add0(double x) {
  return x > 0.0 ? x + log1p(exp(-x)) : log1p(exp(x));
}

// value of CSR entry p; val == nullptr: a binarized matrix, every stored entry is 1
template <typename VT>
__device__ __forceinline__ double valf(const VT *val, int64_t p) { return val ? (double)val[p] : 1.0; }

// proximal step of the L1 penalty on one coefficient: sign(x) max(|x| - t, 0) (kmerLr_estimator_proximal.go:88-98)
__device__ __forceinline__ double soft_threshold(double x, double t) {
  return x >= 0.0 ? fmax(fabs(x) - t, 0.0) : -fmax(fabs(x) - t, 0.0);
}

// eval_stopping (kmerLr_estimator_proximal.go:30-52) from max |x1|, max |x1 - x0| and whether x1 holds a NaN:
// delta = max|dx| / max|x| (max|dx| when x = 0, NaN on a NaN); stop when delta <= eps, on x = dx = 0 or on a NaN
__host__ __device__ __forceinline__ bool eval_stopping(double mx, double md, bool nan_seen, double eps, double *delta) {
  if (nan_seen) { *delta = nan(""); return true; }
  *delta = mx != 0.0 ? md / mx : md;
  return (mx != 0.0 && md / mx <= eps) || (mx == 0.0 && md == 0.0);
}
#endif

}  // namespace kl
