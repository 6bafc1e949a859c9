// abi.cu -- the C ABI of libkmerlr_b200.so (include/kmerlr_b200.h): handle registry, error
// conversion, per-call device timing.  No CPU fallback: without an sm_100 device every entry point
// that computes returns KMERLR_ERR_NOGPU.
#include <cmath>
#include <map>
#include <mutex>
#include <unordered_map>
#include <vector>

#include "common.cuh"

namespace kl {

namespace {
Ctx g_ctx;
std::mutex g_mutex;   // the library is re-entrant: one call at a time per process / device
std::unordered_map<uint64_t, std::shared_ptr<Object>> g_objects;
uint64_t g_next = 1;
thread_local std::string g_error;
}  // namespace

Ctx &ctx() { return g_ctx; }

// ---- caching arena ------------------------------------------------------------------------------------
namespace {
std::multimap<size_t, void *> g_free_blocks;            // size -> block
std::unordered_map<void *, size_t> g_block_size;        // every block we own
constexpr size_t ARENA_GRAIN = (size_t)2 << 20;         // 2 MiB
}  // namespace
void *arena_alloc(size_t bytes) {
  size_t want = (bytes + ARENA_GRAIN - 1) / ARENA_GRAIN * ARENA_GRAIN;
  auto it = g_free_blocks.lower_bound(want);
  // reuse a cached block unless it would waste more than half of itself
  if (it != g_free_blocks.end() && it->first <= 2 * want + 8 * ARENA_GRAIN) {
    void *p = it->second;
    g_free_blocks.erase(it);
    return p;
  }
  void *p = nullptr;
  cudaError_t e = cudaMalloc(&p, want);
  if (e != cudaSuccess) {
    // out of memory: give the cache back to the driver and retry once
    cudaGetLastError();
    cudaStreamSynchronize(g_ctx.stream);
    for (auto &kv : g_free_blocks) { cudaFree(kv.second); g_block_size.erase(kv.second); }
    g_free_blocks.clear();
    KL_CUDA(cudaMalloc(&p, want));
  }
  g_block_size[p] = want;
  return p;
}
void arena_free(void *p) {
  auto it = g_block_size.find(p);
  if (it == g_block_size.end()) return;
  g_free_blocks.emplace(it->second, p);
}
void arena_release_all() {
  for (auto &kv : g_block_size) cudaFree(kv.first);
  g_block_size.clear();
  g_free_blocks.clear();
}

void *host_staging(size_t bytes) {
  KL_CUDA(cudaEventSynchronize(g_ctx.staging_ev));
  if (bytes > g_ctx.staging_bytes) {
    if (g_ctx.staging) KL_CUDA(cudaFreeHost(g_ctx.staging));
    g_ctx.staging = nullptr; g_ctx.staging_bytes = 0;
    const size_t want = (bytes + ARENA_GRAIN - 1) / ARENA_GRAIN * ARENA_GRAIN;
    KL_CUDA(cudaMallocHost(&g_ctx.staging, want));
    g_ctx.staging_bytes = want;
  }
  return g_ctx.staging;
}

// ---- per-kernel profiling ---------------------------------------------------------------------------
namespace {
struct ProfRec { std::string name; cudaEvent_t e0, e1; };
std::vector<ProfRec> g_prof_pending;
std::vector<cudaEvent_t> g_prof_pool;
std::unordered_map<std::string, std::pair<double, int64_t>> g_prof_totals;
cudaEvent_t prof_event() {
  if (!g_prof_pool.empty()) { cudaEvent_t e = g_prof_pool.back(); g_prof_pool.pop_back(); return e; }
  cudaEvent_t e;
  KL_CUDA(cudaEventCreate(&e));
  return e;
}
void prof_resolve() {
  if (g_prof_pending.empty()) return;
  KL_CUDA(cudaStreamSynchronize(g_ctx.stream));
  for (auto &r : g_prof_pending) {
    float ms = 0.f;
    KL_CUDA(cudaEventElapsedTime(&ms, r.e0, r.e1));
    auto &t = g_prof_totals[r.name];
    t.first += ms; t.second += 1;
    g_prof_pool.push_back(r.e0); g_prof_pool.push_back(r.e1);
  }
  g_prof_pending.clear();
}
}  // namespace
void profile_begin(const char *name) {
  if (g_prof_pending.size() > 8192) prof_resolve();
  ProfRec r{name, prof_event(), prof_event()};
  KL_CUDA(cudaEventRecord(r.e0, g_ctx.stream));
  g_prof_pending.push_back(r);
}
void profile_end() { KL_CUDA(cudaEventRecord(g_prof_pending.back().e1, g_ctx.stream)); }

void require_ready() {
  if (!g_ctx.ready) fail(KMERLR_ERR_NOGPU, "kmerlr_init() has not succeeded: no usable sm_100 GPU (there is no CPU fallback)");
}

uint64_t register_object(std::shared_ptr<Object> o) {
  uint64_t h = g_next++;
  g_objects[h] = std::move(o);
  return h;
}
std::shared_ptr<Object> lookup_object(uint64_t h) {
  auto it = g_objects.find(h);
  return it == g_objects.end() ? nullptr : it->second;
}

template <typename F>
int guarded(F &&f, bool timed = true) {
  std::lock_guard<std::mutex> lock(g_mutex);
  try {
    // the current device is per host THREAD: cgo moves goroutines between OS threads, and kmerlr_init
    // bound only the thread that ran it
    if (g_ctx.ready) KL_CUDA(cudaSetDevice(g_ctx.device));
    if (timed && g_ctx.ready) KL_CUDA(cudaEventRecord(g_ctx.ev0, g_ctx.stream));
    f();
    if (timed && g_ctx.ready) {
      KL_CUDA(cudaEventRecord(g_ctx.ev1, g_ctx.stream));
      KL_CUDA(cudaEventSynchronize(g_ctx.ev1));
      float ms = 0.f;
      KL_CUDA(cudaEventElapsedTime(&ms, g_ctx.ev0, g_ctx.ev1));
      g_ctx.last_ms = ms;
    }
    return KMERLR_OK;
  } catch (const Error &e) {
    g_error = e.msg;
    if (g_ctx.ready) cudaGetLastError();
    return e.code;
  } catch (const std::exception &e) {
    g_error = e.what();
    return KMERLR_ERR_INTERNAL;
  }
}

}  // namespace kl

using namespace kl;

extern "C" {

int kmerlr_version(void) { return 100; }

const char *kmerlr_last_error(void) { return g_error.c_str(); }

double kmerlr_last_device_ms(void) { return g_ctx.last_ms; }

int64_t kmerlr_launch_count(void) { return g_ctx.launches; }

int kmerlr_profile(int enable) {
  return guarded([&] {
    prof_resolve();
    if (enable) g_prof_totals.clear();
    g_ctx.profiling = enable != 0;
  }, false);
}

int kmerlr_profile_read(const char *kernel_substr, double *ms_total, int64_t *launches) {
  return guarded([&] {
    prof_resolve();
    double ms = 0.0; int64_t n = 0;
    for (auto &kv : g_prof_totals)
      if (kv.first.find(kernel_substr) != std::string::npos) { ms += kv.second.first; n += kv.second.second; }
    *ms_total = ms; *launches = n;
  }, false);
}

int kmerlr_profile_dump(char *buf, int64_t buflen) {
  return guarded([&] {
    prof_resolve();
    std::string out;
    for (auto &kv : g_prof_totals)
      out += kv.first + "\t" + std::to_string(kv.second.first) + "\t" + std::to_string(kv.second.second) + "\n";
    KL_REQUIRE((int64_t)out.size() + 1 <= buflen, "profile_dump: buffer too small");
    memcpy(buf, out.c_str(), out.size() + 1);
  }, false);
}

int kmerlr_option(const char *name, int64_t value) {
  return guarded([&] {
    KL_REQUIRE(name != nullptr, "option: null name");
    if (!strcmp(name, "implicit")) g_ctx.implicit_ok = value != 0;
    else if (!strcmp(name, "super_len")) g_ctx.super_len = (int)(value < 0 ? -1 : (value > IMP_SUPER_MAX ? IMP_SUPER_MAX : value));
    else if (!strcmp(name, "p2p")) g_ctx.p2p_ok = value != 0;
    else if (!strcmp(name, "feed_growth")) g_ctx.feed_growth = (int)(value < 100 ? 100 : (value > 400 ? 400 : value));
    else if (!strcmp(name, "small_long")) g_ctx.small_long = (int)(value < 0 ? -1 : (value > 2 ? 2 : value));
    else if (!strcmp(name, "persist_bps")) g_ctx.persist_bps = (int)(value < 0 ? 0 : value);
    else if (!strcmp(name, "p2p_allreduce")) g_ctx.p2p_allreduce = value != 0;
    else if (!strcmp(name, "persistent")) g_ctx.coop_ok = value != 0 && g_ctx.coop_supported;
    else if (!strcmp(name, "fused_ticket")) g_ctx.fused_ticket = (int)(value < 0 ? 0 : (value > 4096 ? 4096 : value));
    else if (!strcmp(name, "hot_cols")) g_ctx.hot_cols = (int)(value < 0 ? 0 : (value > 16384 ? 16384 : value));
    else fail(KMERLR_ERR_ARG, std::string("unknown option ") + name);
  }, false);
}

int kmerlr_init(int device) {
  return guarded([&] {
    if (g_ctx.ready) {
      KL_REQUIRE(device == g_ctx.device, "kmerlr_init: already initialised on another device");
      return;
    }
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
      cudaGetLastError();
      fail(KMERLR_ERR_NOGPU, "no CUDA device visible (there is no CPU fallback)");
    }
    KL_REQUIRE(device >= 0 && device < count, "kmerlr_init: device index out of range");
    cudaDeviceProp prop;
    KL_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) fail(KMERLR_ERR_NOGPU, std::string("device is ") + prop.name + " (sm_" + std::to_string(prop.major) + std::to_string(prop.minor) + "); this library is built for sm_100a only");
    KL_CUDA(cudaSetDevice(device));
    g_ctx.device = device;
    g_ctx.sm_count = prop.multiProcessorCount;
    g_ctx.coop_supported = prop.cooperativeLaunch != 0;
    g_ctx.coop_ok = g_ctx.coop_supported;
    KL_CUDA(cudaStreamCreateWithFlags(&g_ctx.stream, cudaStreamNonBlocking));
    KL_CUDA(cudaStreamCreateWithFlags(&g_ctx.copy_stream, cudaStreamNonBlocking));
    KL_CUDA(cudaStreamCreateWithFlags(&g_ctx.alt_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; i++) KL_CUDA(cudaEventCreateWithFlags(&g_ctx.join_ev[i], cudaEventDisableTiming));
    for (int i = 0; i < CTX_COPY_EVENTS; i++) KL_CUDA(cudaEventCreateWithFlags(&g_ctx.copy_ev[i], cudaEventDisableTiming));

    KL_CUDA(cudaEventCreate(&g_ctx.ev0));
    KL_CUDA(cudaEventCreate(&g_ctx.ev1));
    KL_CUDA(cudaEventCreateWithFlags(&g_ctx.staging_ev, cudaEventDisableTiming));
    g_ctx.ready = true;
  }, false);
}

int kmerlr_shutdown(void) {
  return guarded([&] {
    g_objects.clear();
    if (g_ctx.ready) {
      cudaStreamSynchronize(g_ctx.stream);
      arena_release_all();
      comm_destroy();
      cudaEventDestroy(g_ctx.ev0); cudaEventDestroy(g_ctx.ev1);
      cudaEventDestroy(g_ctx.staging_ev);
      if (g_ctx.staging) cudaFreeHost(g_ctx.staging);
      cudaStreamSynchronize(g_ctx.copy_stream);
      for (int i = 0; i < CTX_COPY_EVENTS; i++) cudaEventDestroy(g_ctx.copy_ev[i]);
      cudaStreamDestroy(g_ctx.copy_stream);
      cudaStreamSynchronize(g_ctx.alt_stream);
      cudaStreamDestroy(g_ctx.alt_stream);
      for (int i = 0; i < 2; i++) cudaEventDestroy(g_ctx.join_ev[i]);
      cudaStreamDestroy(g_ctx.stream);
      g_ctx = Ctx();
    }
  }, false);
}

int kmerlr_comm_unique_id(void *id128) { return guarded([&] { comm_unique_id(id128); }, false); }
int kmerlr_comm_init(int rank, int world, const void *id128) { return guarded([&] { comm_init(rank, world, id128); }, false); }
int kmerlr_comm_destroy(void) { return guarded([&] { comm_destroy(); }, false); }

int kmerlr_sequences_create(const uint8_t *seq, const int64_t *off, int64_t n, kmerlr_handle *out) {
  return guarded([&] {
    KL_REQUIRE(out, "null output handle");
    *out = register_object(sequences_create(seq, off, n));
  });
}

// import_fasta (kmerLr_data.go:101-121)
int kmerlr_sequences_from_fasta(const uint8_t *const *texts, const int64_t *nbytes, int64_t n_texts,
                                int64_t *records_out, kmerlr_handle *out) {
  return guarded([&] {
    KL_REQUIRE(out, "null output handle");
    *out = register_object(sequences_from_fasta(texts, nbytes, n_texts, records_out));
  });
}

int kmerlr_sequences_info(kmerlr_handle sequences, int64_t *n, int64_t *total_bases, int64_t *len_out_or_null) {
  return guarded([&] {
    auto s = lookup<SeqSet>(sequences, "sequences");
    if (n) *n = s->n;
    if (total_bases) *total_bases = s->total_bases;
    if (len_out_or_null && s->n) {
      s->len.download(len_out_or_null, (size_t)s->n);
      sync_stream();
    }
  }, false);
}

int kmerlr_sequences_names(kmerlr_handle sequences, char *buf_or_null, int64_t buflen, int64_t *name_off) {
  return guarded([&] {
    KL_REQUIRE(name_off, "null argument");
    auto s = lookup<SeqSet>(sequences, "sequences");
    const bool named = (int64_t)s->name_off.size() == s->n + 1;
    for (int64_t i = 0; i <= s->n; i++) name_off[i] = named ? s->name_off[(size_t)i] : 0;
    if (!buf_or_null) return;
    KL_REQUIRE(buflen >= name_off[s->n], "sequences_names: buffer too small");
    if (name_off[s->n]) memcpy(buf_or_null, s->names.data(), (size_t)name_off[s->n]);
  }, false);
}

// the slicing of extractFasta (kmerLr_predict_genomic.go:93-112)
int kmerlr_sequences_regions(kmerlr_handle sequences, const int64_t *seq_index, const int64_t *from,
                             const int64_t *to, int64_t n, kmerlr_handle *out) {
  return guarded([&] {
    KL_REQUIRE(out, "null output handle");
    *out = register_object(sequences_regions(*lookup<SeqSet>(sequences, "sequences"), seq_index, from, to, n));
  });
}

int kmerlr_sequences_bases(kmerlr_handle sequences, char *out) {
  return guarded([&] {
    auto s = lookup<SeqSet>(sequences, "sequences");
    KL_REQUIRE(out || s->total_bases == 0, "null argument");
    sequences_letters(*s, out);
  });
}

int kmerlr_extract_resident(const kmerlr_config *cfg, kmerlr_handle sequences, const int32_t *frozen_k,
                            const uint64_t *frozen_code, int64_t n_frozen, const int32_t *features,
                            int64_t n_features, int flags, kmerlr_handle *out) {
  return guarded([&] {
    KL_REQUIRE(cfg && out, "null argument");
    auto s = lookup<SeqSet>(sequences, "sequences");
    *out = register_object(extract(*cfg, s, frozen_k, frozen_code, n_frozen, features, n_features, flags));
  });
}

int kmerlr_extract(const kmerlr_config *cfg, const uint8_t *seq, const int64_t *off, int64_t n,
                   const int32_t *frozen_k, const uint64_t *frozen_code, int64_t n_frozen,
                   const int32_t *features, int64_t n_features, int flags, kmerlr_handle *out) {
  return guarded([&] {
    KL_REQUIRE(cfg && out, "null argument");
    *out = register_object(extract_host(*cfg, seq, off, n, frozen_k, frozen_code, n_frozen, features, n_features, flags));
  });
}

int kmerlr_matrix_info(kmerlr_handle h, int64_t *n, int64_t *m, int64_t *nnz, int64_t *n_classes) {
  return guarded([&] {
    auto M = lookup<Matrix>(h, "matrix");
    if (n) *n = M->n;
    if (m) *m = M->m;
    if (nnz) *nnz = M->nnz;
    if (n_classes) *n_classes = M->n_classes;
  }, false);
}

int kmerlr_matrix_rows_global(kmerlr_handle h, int64_t *n_global) {
  return guarded([&] {
    KL_REQUIRE(n_global, "null argument");
    *n_global = lookup<Matrix>(h, "matrix")->n_global;
  }, false);
}

int kmerlr_matrix_classes(kmerlr_handle h, int32_t *k_out, uint64_t *code_out) {
  return guarded([&] {
    auto M = lookup<Matrix>(h, "matrix");
    matrix_class_list(*M);
    for (size_t j = 0; j < M->class_k.size(); j++) { k_out[j] = M->class_k[j]; code_out[j] = M->class_code[j]; }
  }, false);
}

int kmerlr_matrix_rows(kmerlr_handle h, int64_t *rowptr, int32_t *col, double *val) {
  return guarded([&] { matrix_rows(*lookup<Matrix>(h, "matrix"), rowptr, col, val); });
}

int kmerlr_matrix_set_labels(kmerlr_handle h, const uint8_t *labels, int64_t n) {
  return guarded([&] { matrix_set_labels(*lookup<Matrix>(h, "matrix"), labels, n); });
}

int kmerlr_matrix_from_csr(int64_t n, int64_t m, const int64_t *rowptr, const int32_t *col, const double *val,
                           int flags, kmerlr_handle *out) {
  return guarded([&] {
    KL_REQUIRE(out, "null output handle");
    *out = register_object(matrix_from_csr(n, m, rowptr, col, val, flags));
  });
}

int kmerlr_column_moments(kmerlr_handle h, double *sum, double *sumsq, double *absmax, int64_t *count) {
  return guarded([&] {
    KL_REQUIRE(sum && sumsq && absmax && count, "null argument");
    matrix_column_moments(*lookup<Matrix>(h, "matrix"), sum, sumsq, absmax, count);
  });
}

int kmerlr_pair_moments(kmerlr_handle h, double *sum, double *sumsq, double *absmax, int64_t *count) {
  return guarded([&] {
    KL_REQUIRE(sum && sumsq && absmax && count, "null argument");
    matrix_pair_moments(*lookup<Matrix>(h, "matrix"), sum, sumsq, absmax, count);
  });
}

int kmerlr_matrix_transform(kmerlr_handle h, const double *offset_or_null, const double *scale_or_null, int64_t len,
                            kmerlr_handle *out) {
  return guarded([&] {
    KL_REQUIRE(out, "null output handle");
    *out = register_object(matrix_transform(*lookup<Matrix>(h, "matrix"), offset_or_null, scale_or_null, len));
  });
}

int kmerlr_free(kmerlr_handle h) {
  return guarded([&] {
    KL_REQUIRE(g_objects.erase(h) == 1, "kmerlr_free: invalid handle");
  }, false);
}

int64_t kmerlr_coeff_dim(int64_t n) { return (n + 1) * n / 2 + 1; }
int64_t kmerlr_coeff_ind2sub(int64_t n, int64_t k1, int64_t k2) {
  if (k1 == k2) return k1 + 1;
  return n + (n * (n - 1) / 2) - (n - k1) * ((n - k1) - 1) / 2 + k2 - k1;
}
void kmerlr_coeff_sub2ind(int64_t n, int64_t i, int64_t *k1, int64_t *k2) {
  if (i < n) { *k1 = i; *k2 = i; return; }
  i = i - n;
  int64_t a = n - 2 - (int64_t)std::floor(std::sqrt((double)(-8 * i + 4 * n * (n - 1) - 7)) / 2.0 - 0.5);
  *k1 = a;
  *k2 = i + a + 1 - n * (n - 1) / 2 + (n - a) * ((n - a) - 1) / 2;
}

int kmerlr_linear_pdf(kmerlr_handle h, const double *theta, int64_t ntheta, int cooccurrence, double *out_n) {
  return guarded([&] { linear_pdf(*lookup<Matrix>(h, "matrix"), theta, ntheta, cooccurrence, out_n, false); });
}
int kmerlr_logpdf(kmerlr_handle h, const double *theta, int64_t ntheta, int cooccurrence, double *out_n) {
  return guarded([&] { linear_pdf(*lookup<Matrix>(h, "matrix"), theta, ntheta, cooccurrence, out_n, true); });
}
int kmerlr_gradient(kmerlr_handle h, const double *theta, int64_t ntheta, const double class_w[2], double lambda,
                    int cooccurrence, double *g_out) {
  return guarded([&] { gradient(*lookup<Matrix>(h, "matrix"), theta, ntheta, class_w, lambda, cooccurrence, g_out); });
}
int kmerlr_loss(kmerlr_handle h, const double *theta, int64_t ntheta, const double class_w[2], double lambda,
                int cooccurrence, double *loss_out) {
  return guarded([&] { *loss_out = loss(*lookup<Matrix>(h, "matrix"), theta, ntheta, class_w, lambda, cooccurrence); });
}
int kmerlr_class_weights(kmerlr_handle h, double class_w_out[2]) {
  return guarded([&] {
    auto M = lookup<Matrix>(h, "matrix");
    KL_REQUIRE(M->has_labels, "class_weights: the matrix has no labels");
    matrix_label_counts(*M);
    double n0 = (double)M->n_neg, n1 = (double)M->n_pos;
    class_w_out[0] = (n0 + n1) / (2.0 * n0);
    class_w_out[1] = (n0 + n1) / (2.0 * n1);
  }, false);
}

int kmerlr_select(kmerlr_handle h, const double class_w[2], int cooccurrence, int64_t N, double theta0,
                  const int64_t *active_idx, const double *active_theta, int64_t n_active, int tie,
                  double epsilon_lambda, double prev_lambda, uint8_t *mask_out, int64_t ntheta, double *lambda_out,
                  int64_t *c_out, int *ok_out, double *g_out_or_null) {
  return guarded([&] {
    KL_REQUIRE(mask_out && lambda_out && c_out && ok_out, "null argument");
    select(*lookup<Matrix>(h, "matrix"), class_w, cooccurrence, N, theta0, active_idx, active_theta, n_active, tie,
           epsilon_lambda, prev_lambda, mask_out, ntheta, lambda_out, c_out, ok_out, g_out_or_null);
  });
}

int kmerlr_select_from_gradient(const double *g, int64_t ntheta, int64_t N, const int64_t *active_idx,
                                const double *active_theta, int64_t n_active, int tie, double epsilon_lambda,
                                double prev_lambda, uint8_t *mask_out, double *lambda_out, int64_t *c_out, int *ok_out) {
  return guarded([&] {
    KL_REQUIRE(g && mask_out && lambda_out && c_out && ok_out && ntheta >= 1, "null argument");
    select_from_gradient(g, ntheta, N, active_idx, active_theta, n_active, tie, epsilon_lambda, prev_lambda, mask_out,
                         lambda_out, c_out, ok_out);
  }, false);
}

int kmerlr_reduce(kmerlr_handle h, const int64_t *sel, int64_t nsel, kmerlr_handle *out) {
  return guarded([&] {
    KL_REQUIRE(out, "null output handle");
    *out = register_object(matrix_reduce(*lookup<Matrix>(h, "matrix"), sel, nsel));
  });
}

int kmerlr_step_size(kmerlr_handle h, double l2, double step_factor, double *step_out) {
  return guarded([&] {
    auto M = lookup<Matrix>(h, "matrix");
    KL_REQUIRE(M->n_global > 0, "step_size: empty data set");
    double L = 0.25 * (matrix_maxsq(*M) + 1.0) + l2 / (double)M->n_global;
    *step_out = 1.0 / (2.0 * L + std::fmin(2.0 * l2, L)) * step_factor;
  });
}

int kmerlr_proxgrad(kmerlr_handle h, double *theta_inout, int64_t ntheta, const double class_w[2], double lambda,
                    double l2, double step_factor, double epsilon, double epsilon_loss, int64_t max_iter,
                    double hook_state[2], int64_t *iters_out, double *delta_out) {
  return guarded([&] {
    proxgrad(*lookup<Matrix>(h, "matrix"), theta_inout, ntheta, class_w, lambda, l2, step_factor, epsilon,
             epsilon_loss, max_iter, hook_state, iters_out, delta_out);
  });
}

int kmerlr_coordinate(kmerlr_handle h, double *theta_inout, int64_t ntheta, const double class_w_hook[2], double l1reg,
                      double l2reg, double epsilon, double epsilon_loss, int64_t max_iter, double hook_state[2],
                      int64_t *sweeps_out, double *delta_out) {
  return guarded([&] {
    KL_REQUIRE(theta_inout && class_w_hook, "coordinate: null argument");
    coordinate(*lookup<Matrix>(h, "matrix"), theta_inout, ntheta, class_w_hook, l1reg, l2reg, epsilon, epsilon_loss,
               max_iter, hook_state, sweeps_out, delta_out);
  });
}

int64_t kmerlr_window_slots(int64_t len, int64_t W, int64_t step) {
  int64_t n = len - W;
  return n > 0 ? n / step + 1 : 0;
}

int kmerlr_score_windows(const kmerlr_model *models, int n_models, const uint8_t *seq, const int64_t *region_off,
                         int64_t n_regions, int64_t W, int64_t step, double *out) {
  return guarded([&] {
    // the contigs arrive in chunks: copies in both directions overlap the scoring (score.cu)
    std::unique_ptr<SeqFeed> feed;
    auto s = sequences_begin_chunked(seq, region_off, n_regions, feed);
    score_windows(models, n_models, *s, W, step, out, nullptr, 0, feed.get());
  });
}

// predict_window (kmerLr_predict.go:89-124): one classifier, len - W slots per sequence, slot j = window at j
int kmerlr_predict_windows(const kmerlr_model *model, const uint8_t *seq, const int64_t *seq_off, int64_t n_seq,
                           int64_t W, int64_t step, double *out) {
  return guarded([&] {
    KL_REQUIRE(model && out, "null argument");
    auto s = sequences_create(seq, seq_off, n_seq);
    score_windows(model, 1, *s, W, step, out, nullptr, 1);
  });
}

int kmerlr_score_windows_resident(const kmerlr_model *models, int n_models, kmerlr_handle sequences, int64_t W,
                                  int64_t step, double *out_host_or_null, kmerlr_handle *out_dev_or_null) {
  return guarded([&] {
    auto s = lookup<SeqSet>(sequences, "sequences");
    std::shared_ptr<Object> dev;
    score_windows(models, n_models, *s, W, step, out_host_or_null, out_dev_or_null ? &dev : nullptr);
    if (out_dev_or_null) *out_dev_or_null = register_object(dev);
  });
}

// ---- on-disk formats (formats.cu) -----------------------------------------------------------------------------
int kmerlr_wiggle_records(const double *pred, int64_t n, char *out, int64_t *n_irregular_out) {
  return guarded([&] {
    const int64_t irr = wiggle_records(pred, false, n, out);
    if (n_irregular_out) *n_irregular_out = irr;
  });
}

int kmerlr_save_wiggle(const char *filename, const char *track_name, int64_t n_regions, const char *const *seqnames,
                       const int64_t *from, const int64_t *slot_off, const double *pred_or_null, kmerlr_handle scores,
                       int64_t window_size, int64_t window_step) {
  return guarded([&] {
    require_ready();
    if (n_regions == 0) { save_wiggle(filename, track_name, 0, nullptr, nullptr, nullptr, nullptr, false, window_size, window_step); return; }
    if (pred_or_null) { save_wiggle(filename, track_name, n_regions, seqnames, from, slot_off, pred_or_null, false, window_size, window_step); return; }
    auto S = lookup<Matrix>(scores, "scores");
    KL_REQUIRE(n_regions == 0 || (slot_off && (size_t)slot_off[n_regions] <= S->val_f64.n), "save_wiggle: more slots than scores");
    save_wiggle(filename, track_name, n_regions, seqnames, from, slot_off, S->val_f64.p, true, window_size, window_step);
  });
}

int kmerlr_export_kmers(kmerlr_handle data, const kmerlr_config *cfg, const char *filename, int as_float) {
  return guarded([&] {
    KL_REQUIRE(cfg, "null configuration");
    export_kmers(*lookup<Matrix>(data, "matrix"), *cfg, filename, as_float != 0);
  });
}

int kmerlr_class_name(const kmerlr_config *cfg, int32_t k, uint64_t code, char *buf, int64_t buflen) {
  return guarded([&] {
    KL_REQUIRE(cfg && buf && buflen > 0, "null argument");
    const std::string s = class_name(*cfg, k, code);
    KL_REQUIRE((int64_t)s.size() < buflen, "class_name: buffer too small");
    memcpy(buf, s.c_str(), s.size() + 1);
  }, false);
}

int kmerlr_export_path(const char *filename, int64_t n, const int64_t *estimator_or_null, const double *lambda,
                       const double *norm, const int64_t *theta_off, const double *theta) {
  return guarded([&] { export_path(filename, n, estimator_or_null, lambda, norm, theta_off, theta); }, false);
}

int kmerlr_export_trace(const char *filename, int64_t n, const int64_t *duration_ns, const int64_t *iteration,
                        const double *change, const int64_t *nonzero, const double *lambda_or_null,
                        const double *loss_or_null) {
  return guarded([&] { export_trace(filename, n, duration_ns, iteration, change, nonzero, lambda_or_null, loss_or_null); }, false);
}

}  // extern "C"
