// logistic.cu -- stage 2 of the hot path: sparse logistic loss / gradient and the proximal-gradient
// estimator.
//
// Replaces logisticRegression.LinearPdf / LogPdf / Gradient / Loss
// (kmerLr_logistic_regression.go:47-272) and estimate_proximal + eval_stopping + estimate_step_size
// (kmerLr_estimator_proximal.go:30-120, hook kmerLr_estimator_hook.go:46-99).
//
// ONE pass over the matrix per gradient (CSR, warp per row): z_i = theta_0 + sum_j v_ij theta_j, the
// loss term and the weight w_i, then the row's contributions w_i v_ij are added to the gradient in
// 64-bit FIXED POINT (scale 2^e, e chosen so that the worst case sum fits): integer addition is
// associative, so the result does not depend on the order of the atomics -- it is deterministic,
// two features with identical columns get bit-identical gradients (what leapfrog tie handling
// needs, SURVEY 7.2), and an int64 all-reduce over the ranks gives the same bits as one GPU.
// The first columns (the dense low-k classes) accumulate in shared memory, the rest in L2.
#include <cooperative_groups.h>

#include "common.cuh"

#include <cmath>

namespace kl {

namespace {

constexpr int RED_BLOCKS = 256;

struct PgState {
  long long iter;
  int done;          // 0 running, 1 stopped, 2 final loss evaluation pending
  int first;
  double delta, loss_old, loss_new, lossval;
  int error;         // 1: a peer never answered the gradient exchange
};

// the hook's state transition (kmerLr_estimator_hook.go:46-99) for the loss l at the current theta
__device__ __forceinline__ void hook_update(PgState *st, double l, double eps_loss) {
  st->lossval = l;
  if (st->first) { st->first = 0; return; }   // loss at the start point: no hook call yet
  const double t = st->loss_old; st->loss_old = st->loss_new; st->loss_new = t;
  if (eps_loss != 0.0) {
    st->loss_new = l;
    if (st->done == 0 && fabs(st->loss_old - st->loss_new) < eps_loss) st->done = 1;
  }
  if (st->done == 2) st->done = 1;
}

// end of a prox step: eval_stopping on max |theta|, max |delta| and the NaN flag of the new theta; after max_iter
// steps one more pass evaluates the hook's loss (done = 2)
__device__ __forceinline__ void pg_stop(PgState *st, double mx, double md, double nn, double eps, long long max_iter) {
  st->iter += 1;
  if (eval_stopping(mx, md, nn != 0.0, eps, &st->delta)) st->done = 1;
  else if (st->iter >= max_iter) st->done = 2;
}

__device__ __forceinline__ int64_t ind2sub(int64_t n, int64_t k1, int64_t k2) {
  return n + (n * (n - 1) / 2) - (n - k1) * ((n - k1) - 1) / 2 + k2 - k1;
}

// a non-zero pair coefficient theta[Ind2Sub(a, b)], a < b (pair mode with a sparse theta)
struct PairTerm {
  uint32_t a, b;
  double theta;
};
// value of column c in the row [a, b) (columns ascending), 0 when absent
template <typename VT>
__device__ __forceinline__ double row_value(const uint32_t *__restrict__ col, const VT *__restrict__ val, int64_t a, int64_t b,
                                            uint32_t c) {
  int64_t lo = a, hi = b;
  while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (col[mid] < c) lo = mid + 1; else hi = mid; }
  return (lo < b && col[lo] == c) ? valf(val, lo) : 0.0;
}

// Gradient weight (kmerLr_logistic_regression.go:166-178) and Loss term (:257-263) of a row with label y and
// z = x theta: returns w, the loss term goes to `lossterm`.  The label and the weights are references so that they
// are read where the formula uses them: read ahead of the logarithm, they stay live across it and ptxas spills in
// imp_pass<8, true>.
__device__ __forceinline__ double row_weight(double z, const uint8_t &y, const double &cw0, const double &cw1, const double &inv_n,
                                             double &lossterm) {
  const double r = -log_add0(-z);
  double w;
  if (y) { w = inv_n * cw1 * (exp(r) - 1.0); lossterm = -cw1 * r; }
  else   { w = inv_n * cw0 * exp(r);         lossterm = cw0 * log_add0(z); }
  return w;
}

// rows pass: MODE 0 = z only, 1 = log sigma(z), 2 = w_i and loss term.
// cooc = 1: pair terms over all pairs of entries of the row (O(q^2) gathers of theta); cooc = 2: over the list of
// non-zero pair coefficients (`terms`, sorted by coefficient index): two lookups per term and row -- an L1-regularised
// theta has a handful of them, and 3.84 M coefficients at C4
template <typename VT, int MODE>
__global__ void rows_kernel(const Rows R, const uint32_t *__restrict__ col,
                            const VT *__restrict__ val, int64_t n, int64_t m, const double *__restrict__ theta,
                            int cooc, const uint8_t *__restrict__ labels, double cw0, double cw1, double inv_n,
                            double *__restrict__ out, double *__restrict__ lossterm, const PgState *st,
                            const PairTerm *__restrict__ terms, int nterms) {
  if (st && st->done == 1) return;
  int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= n) return;
  unsigned lane = lane_id();
  int64_t a, b;
  R.range(row, a, b);
  double s = 0.0;
  for (int64_t p = a + lane; p < b; p += 32) s += valf(val, p) * __ldg(theta + col[p] + 1);
  if (cooc == 2) {
    for (int t = (int)lane; t < nterms; t += 32) {
      const PairTerm pt = terms[t];
      const double v1 = row_value(col, val, a, b, pt.a);
      if (v1 != 0.0) s += v1 * row_value(col, val, a, b, pt.b) * pt.theta;
    }
  } else if (cooc) {
    // pair terms (kmerLr_logistic_regression.go:69-84)
    for (int64_t p1 = a; p1 < b; p1++) {
      double v1 = valf(val, p1);
      int64_t c1 = col[p1];
      for (int64_t p2 = p1 + 1 + lane; p2 < b; p2 += 32)
        s += v1 * valf(val, p2) * __ldg(theta + ind2sub(m, c1, (int64_t)col[p2]));
    }
  }
  s = warp_sum_down(s);
  if (lane == 0) {
    double z = theta[0] + s;
    if (MODE == 0) out[row] = z;
    else if (MODE == 1) out[row] = -log_add0(-z);
    else out[row] = row_weight(z, labels[row], cw0, cw1, inv_n, lossterm[row]);
  }
}

// 64-bit accumulators as two 32-bit words (acc_lo[c], acc_hi[c]): shared memory has native 32-bit atomic adds only (a
// 64-bit add would be a compare-and-swap loop); the carry out of the low word is added to the high word by the thread
// whose add wrapped, so the pair is an exact 64-bit sum
__device__ __forceinline__ void acc64_add(uint32_t *acc_lo, uint32_t *acc_hi, uint32_t c, unsigned long long q) {
  const uint32_t lo = (uint32_t)q, hi = (uint32_t)(q >> 32);
  const uint32_t old = atomicAdd(&acc_lo[c], lo);
  const uint32_t add_hi = hi + ((old + lo) < old ? 1u : 0u);
  if (add_hi) atomicAdd(&acc_hi[c], add_hi);
}
// G[i] += the pair i for i < count, by the threads of the block once its adds are done (after a barrier).  `count` is
// an int: a 64-bit bound widens the loop index and ptxas spills in fused_kernel<uint32_t>.
__device__ __forceinline__ void acc64_flush(const uint32_t *acc_lo, const uint32_t *acc_hi, int count, unsigned long long *G) {
  for (int i = threadIdx.x; i < count; i += blockDim.x) {
    const unsigned long long v = ((unsigned long long)acc_hi[i] << 32) | acc_lo[i];
    if (v) atomicAdd(&G[i], v);
  }
}

// the fused pass over the stored rows: one warp per row
//   G[0]    += round(w_i * S)                 (bias, Go index 0)
//   G[c+1]  += round(w_i * v_ic * S)          for every entry of the row
// Lane l reads the entries l, l + 32, ... of the row: one warp-level gather of theta then covers 32 CONSECUTIVE
// entries of the sorted row, i.e. neighbouring columns that share cache lines.  (128-bit loads of four entries
// per lane were measured slower, 15.3 vs 14.1 ms at C3: the gathers of one instruction then span 128 entries
// and touch four times as many lines, and the gathers, not the streams, bound this kernel -- ncu: 44 % of the
// stall samples on the theta gather, LSU wavefronts at 59 % of peak.)
// Rows: ticket == nullptr: block b owns the rows [b rpb, (b+1) rpb) (fine static grid); else the warps take
// `rpb` rows per atomic ticket.
constexpr int FUSED_RPB = 256;         // rows per block (static grid)
constexpr int HOT_COLS_MAX = 16384;    // at most this many columns accumulate in shared memory (8 B each)

template <typename VT>
__global__ void __launch_bounds__(256) fused_kernel(const Rows R, const uint32_t *__restrict__ col,
                                                    const VT *__restrict__ val, int64_t n, int64_t m,
                                                    const double *__restrict__ theta,
                                                    const uint8_t *__restrict__ labels, double cw0, double cw1,
                                                    double inv_n, double scale, double scale0,
                                                    unsigned long long *__restrict__ G,
                                                    double *__restrict__ lossterm, const PgState *st, int scatter,
                                                    int hot_limit, int rpb, unsigned long long *__restrict__ ticket) {
  if (st && st->done == 1) return;
  extern __shared__ uint32_t hot_smem[];
  uint32_t *hot_lo = hot_smem, *hot_hi = hot_smem + hot_limit;
  const int64_t hot_cols = m < hot_limit ? m : hot_limit;
  for (int i = threadIdx.x; i < hot_cols; i += blockDim.x) { hot_lo[i] = 0u; hot_hi[i] = 0u; }
  __syncthreads();
  const unsigned lane = lane_id();
  long long bias_acc = 0;
  auto do_row = [&](int64_t row) {
    int64_t a, b;
    R.range(row, a, b);
    double s = 0.0;
    for (int64_t p = a + lane; p < b; p += 32) s += valf(val, p) * __ldg(theta + col[p] + 1);
    s = warp_sum_down(s);
    double w = 0.0;
    if (lane == 0) {
      w = row_weight(theta[0] + s, labels[row], cw0, cw1, inv_n, lossterm[row]);
      bias_acc += __double2ll_rn(w * scale0);
    }
    if (!scatter) return;                 // loss-only pass (the hook after the last iteration)
    w = __shfl_sync(0xffffffffu, w, 0);
    const double ws = w * scale;          // scale is a power of two: exact
    for (int64_t p = a + lane; p < b; p += 32) {
      const uint32_t c = col[p];
      const unsigned long long q = (unsigned long long)__double2ll_rn(ws * valf(val, p));
      if (c < (uint32_t)hot_cols) acc64_add(hot_lo, hot_hi, c, q);
      else atomicAdd(&G[c + 1], q);
    }
  };
  if (ticket) {
    for (;;) {
      unsigned long long t0 = 0;
      if (lane == 0) t0 = atomicAdd(ticket, (unsigned long long)rpb);
      const int64_t first = (int64_t)__shfl_sync(0xffffffffu, t0, 0);
      if (first >= n) break;
      const int64_t last = first + rpb < n ? first + rpb : n;
      for (int64_t row = first; row < last; row++) do_row(row);
    }
  } else {
    const int64_t first = (int64_t)blockIdx.x * rpb, last = first + rpb < n ? first + rpb : n;
    for (int64_t row = first + (threadIdx.x >> 5); row < last; row += (blockDim.x >> 5)) do_row(row);
  }
  if (lane == 0 && bias_acc != 0) atomicAdd(&G[0], (unsigned long long)bias_acc);
  __syncthreads();
  acc64_flush(hot_lo, hot_hi, hot_cols, G + 1);
}

// ---- matrix-free pass (matrices straight from the extraction, Matrix::imp) ----------------------------
// The count of class c in row i is the number of positions p of sequence i whose k-mer belongs to c, so
//   z_i = theta_0 + sum_p T[len_p][code_p],   T[j][u] = sum_{k=Mlo..j} theta[class of the k-prefix of u]
//   g_c = sum over the codes u of c and the levels j >= k of F_k, F_k[u] = H_k[u] + sum_x F_{k+1}[4u+x]
// where (len_p, code_p) = the longest valid k-mer (<= N bases) starting at p and H[len_p][code_p]
// collects round(w_i S) of every position.  No CSR traffic at all; the integer sums are exact, so the
// result equals sum_i round(w_i S) count_ic bit for bit in any order.
//
// SUPER K-MERS: c = S - N + 1 consecutive positions whose S bases are all valid share ONE table entry,
//   TS[U] = sum_{t<c} T[N][N-mer at offset t of U],   HS[U] += round(w_i S)
// (U = the S-mer starting at the first of them; HS is scattered back into H[N] before the level fold), so a
// row costs one gather and one RED.64 per GROUP of c positions instead of one per position; the positions of
// a group that reaches past the end of the row or over an invalid base fall back to their own entries.
//
// BINARIZED rows (x_ic = [count_ic > 0]): the levels k >= Mlo = 6 are the count formulation minus one
// correction per REPEAT of a class inside a row (the extraction leaves the columns of those repeats in
// Implicit::events: theta is subtracted once per event, round(w_i S) likewise); the table levels
// (k <= 5, where nearly every class of a row repeats) are a per-row bitmap over their classes: X theta through
// sums precomputed per 4-bit group of the bitmap (lowtab), X^T w by low_accumulate from the stored q_i.
struct ImpParams {
  int M, N, op;
  int Mlo;                 // first matrix-free level
  int S, c;                // super k-mer length, positions per group (c = S - N + 1; c = 1: S = N)
  uint32_t sup0;           // table offset of the super level (c = 1: the offset of level N itself)
  uint32_t level_off[16], fo[16];
};

__global__ void imp_build_T(const ImpParams P, const uint32_t *__restrict__ bitmap, const uint32_t *__restrict__ rank,
                            const double *__restrict__ theta, double *__restrict__ T, int64_t total,
                            const PgState *st) {
  if (st && st->done == 1) return;
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  int j = P.Mlo;
  while (j < P.N && t >= (int64_t)P.fo[j + 1]) j++;
  const uint32_t u = (uint32_t)(t - P.fo[j]);
  double s = 0.0;
  for (int k = P.Mlo; k <= j; k++) {
    uint32_t c = u >> (2 * (j - k));
    if (P.op) c = min(c, kmer_op(c, k, P.op));
    const uint32_t id = P.level_off[k] + c, w = bitmap[id >> 5], bit = 1u << (id & 31);
    if (w & bit) s += theta[rank[id >> 5] + __popc(w & (bit - 1u)) + 1];
  }
  T[t] = s;
}

// TS[U] = sum of the level-N entries of the c N-mers inside the S-mer U
__global__ void imp_build_TS(const ImpParams P, double *__restrict__ T, const PgState *st) {
  if (st && st->done == 1) return;
  const uint32_t U = blockIdx.x * blockDim.x + threadIdx.x;
  if (U >= (1u << (2 * P.S))) return;
  const uint32_t maskN = (1u << (2 * P.N)) - 1u;
  const double *TN = T + P.fo[P.N];
  double s = 0.0;
  for (int t = 0; t < P.c; t++) s += TN[(U >> (2 * (P.S - P.N - t))) & maskN];
  T[P.sup0 + U] = s;
}

// true in every thread of the block that arrives last at `ticket` (one arrival per block of the grid): its reads
// then see what the other blocks wrote before they arrived.  The caller resets the ticket.
__device__ __forceinline__ bool last_block(unsigned int *ticket) {
  __shared__ int s_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(ticket, 1u) == gridDim.x - 1 ? 1 : 0;
  __syncthreads();
  if (!s_last) return false;
  __threadfence();
  return true;
}

// The fold of the forward-code tables after the pass, F_j[u] = H_j[u] + F_{j+1}[4u .. 4u+3] from level N-1 down to
// Mlo, preceded by H[N][N-mer at offset t of U] += HS[U] when there is a super level.  The grid of one launch folds
// `level` (P.N: the super level into level N) -- the large steps, one launch each; the block that finishes last then
// folds the levels tail_top .. Mlo (at most 4^IMP_FOLD_TAIL entries each) in place of one launch per level.  The
// integer sums are exact, so the order does not matter.  `ticket` is zero on entry and left zero.
constexpr int IMP_FOLD_TAIL = 7;
constexpr int IMP_FOLD_THREADS = 1024;
__global__ void __launch_bounds__(IMP_FOLD_THREADS) imp_fold(const ImpParams P, int level, int tail_top,
                                                             unsigned long long *__restrict__ H, unsigned int *ticket,
                                                             const PgState *st) {
  if (st && st->done == 1) return;
  const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
  if (level == P.N) {
    if (u < (1u << (2 * P.S))) {
      const unsigned long long h = H[P.sup0 + u];
      const uint32_t maskN = (1u << (2 * P.N)) - 1u;
      if (h)
        for (int t = 0; t < P.c; t++) atomicAdd(H + P.fo[P.N] + ((u >> (2 * (P.S - P.N - t))) & maskN), h);
    }
  } else if (level >= P.Mlo && u < (1u << (2 * level))) {
    const unsigned long long *c = H + P.fo[level + 1] + 4ull * u;
    H[P.fo[level] + u] += c[0] + c[1] + c[2] + c[3];
  }
  if (tail_top < P.Mlo || !last_block(ticket)) return;
  for (int j = tail_top; j >= P.Mlo; j--) {
    for (uint32_t v = threadIdx.x; v < (1u << (2 * j)); v += blockDim.x) {   // (L2 reads: other blocks wrote there)
      const unsigned long long *c = H + P.fo[j + 1] + 4ull * v;
      H[P.fo[j] + v] = __ldcg(H + P.fo[j] + v) + __ldcg(c) + __ldcg(c + 1) + __ldcg(c + 2) + __ldcg(c + 3);
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) *ticket = 0u;
}

// binarized rows: lowtab[(i * 16 + v) * lwp + l] = sum of theta over the classes (l * 32 + 4 i + b) with bit b
// of v set -- X theta of the table levels is 8 shared-memory reads per bitmap word
__global__ void imp_build_low(const uint32_t *__restrict__ lowcol, int low_words, int lwp,
                              const double *__restrict__ theta, double *__restrict__ lowtab, const PgState *st) {
  if (st && st->done == 1) return;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= 128 * lwp) return;
  const int l = e % lwp, v = (e / lwp) & 15, i = e / (16 * lwp);
  double s = 0.0;
  if (l < low_words)
    for (int b = 0; b < 4; b++)
      if ((v >> b) & 1) {
        const uint32_t col = lowcol[l * 32 + 4 * i + b];
        if (col != NOCOL) s += theta[col + 1];
      }
  lowtab[e] = s;
}

constexpr uint32_t IMP_NOIDX = 0xFFFFFFFFu, IMP_SINGLES = 0xFFFFFFFEu;

// A lane's view of a row: up to 32 consecutive bases starting at p0, digit-reversed so that the first base
// sits in the two top bits (a k-mer starting at base x of the window is a shift and a mask: code order,
// first base most significant), and one "not usable" bit per base (invalid letter, or past the end of the row).
struct ImpWindow {
  unsigned long long rev;
  uint32_t inv;
  int left;                                     // bases of the row from the window's first base on (<= 0: none)
  __device__ __forceinline__ void load(const uint32_t *__restrict__ b2, const uint16_t *__restrict__ iv, int L, int p0) {
    left = L - p0;
    if (p0 >= L) { rev = 0ull; inv = 0xFFFFFFFFu; return; }     // (and no load past the row)
    const int wi = p0 >> 4, sh = p0 & 15;
    const uint32_t w0 = __ldg(b2 + wi), w1 = __ldg(b2 + wi + 1), w2 = __ldg(b2 + wi + 2);
    const uint32_t lo = __funnelshift_r(w0, w1, 2 * sh), hi = __funnelshift_r(w1, w2, 2 * sh);
    rev = ((unsigned long long)swap_pairs(__brev(lo)) << 32) | swap_pairs(__brev(hi));
    const unsigned long long iw = (unsigned long long)__ldg(iv + wi) | ((unsigned long long)__ldg(iv + wi + 1) << 16) |
                                  ((unsigned long long)__ldg(iv + wi + 2) << 32);
    inv = (uint32_t)(iw >> sh);
    if (left < 32) inv |= 0xFFFFFFFFu << left;
  }
  // the k bases starting at base x of the window (x + k <= 32)
  __device__ __forceinline__ uint32_t code(int x, int k) const {
    return (uint32_t)(rev >> (64 - 2 * (x + k))) & ((1u << (2 * k)) - 1u);
  }
};

// group at base x of the window = c positions.  Table index of its super k-mer, IMP_SINGLES when the S bases
// are not all usable, IMP_NOIDX when the group starts past the end of the row
__device__ __forceinline__ uint32_t imp_group(const ImpParams &P, const ImpWindow &W, int x) {
  if (x >= W.left) return IMP_NOIDX;            // the group starts past the end of the row: nothing to look at
  const uint32_t bits = (W.inv >> x) & ((1u << P.S) - 1u);
  return bits == 0u ? P.sup0 + W.code(x, P.S) : IMP_SINGLES;
}
// position at base x of the window: table index of the longest valid k-mer starting there (x + N <= 32)
__device__ __forceinline__ uint32_t imp_single(const ImpParams &P, const ImpWindow &W, int x) {
  const uint32_t bits = W.inv >> x;
  int lf = bits ? __ffs(bits) - 1 : P.N;
  if (lf > P.N) lf = P.N;
  if (lf < P.Mlo) return IMP_NOIDX;
  return P.fo[lf] + W.code(x, lf);
}

struct ImpArgs {
  int64_t n;
  const int64_t *len, *blk;
  const uint32_t *bits2;
  const uint16_t *inv16;
  const double *T, *theta;
  const uint8_t *labels;
  double cw0, cw1, inv_n, scale;
  unsigned long long *H, *G;
  double *lossterm;
  const PgState *st;
  int scatter;
  int rpb;                     // rows per block
  int gw;                      // groups per window: (gw - 1) c + S <= 32
  // binarized rows
  const uint32_t *lowbits;
  int low_words, lwp;
  const double *lowtab;
  const int64_t *evptr;
  const uint32_t *events;
  unsigned long long *q_out;
};

constexpr int IMP_R = 2;           // rows per warp and round

// One warp per sequence, 8 warps per block; block b owns the rows [b rpb, (b+1) rpb) and works through them in
// rounds of 8 IMP_R rows: (A) every warp decodes its rows and gathers, (B) the weights of all rows of the round
// are computed together -- the fp64 exp / log1p of a row are ~300 instructions for ONE lane, a third of the
// whole row when every warp did them for itself -- (C) every warp scatters.  A fine grid of short blocks: the
// hardware block scheduler balances the SMs.  A lane owns CONSECUTIVE groups of its row, so one 64-bit window of
// packed bases (digit-reversed once) serves all of them.
// CACHE > 0: the lane's groups fit one window and their table indices stay in registers between gather and
// scatter (rows of up to 32 CACHE groups); CACHE = 0: window after window, decoded twice (rows of any length).
#ifndef KL_IMP_MINB
#define KL_IMP_MINB 0      // resident blocks per SM the compiler has to make room for (0: its own choice, 62-64 registers,
                           // 4 blocks; measured with 5 blocks / 48 registers: the same at C2, 3 % faster at C3; with 6 / 40: 25 % slower)
#endif
template <int CACHE, bool BIN>
__global__ void
#if KL_IMP_MINB > 0
__launch_bounds__(256, KL_IMP_MINB)
#else
__launch_bounds__(256)
#endif
imp_pass(const ImpParams P, const ImpArgs A) {
  if (A.st && A.st->done == 1) return;
  constexpr int CC = CACHE > 0 ? CACHE : 1;
  constexpr int RR = 8 * IMP_R;
  extern __shared__ __align__(16) double s_low[];
  __shared__ double s_z[RR];
  __shared__ unsigned long long s_q[RR];
  __shared__ unsigned long long s_bias;
  __shared__ __align__(8) unsigned long long s_bar;
  if (threadIdx.x == 0) {
    s_bias = 0ull;
    if (BIN) mbar_init(&s_bar, 1);
  }
  __syncthreads();
  // binarized rows: the block's copy of lowtab (32 / 64 KB) arrives by ONE TMA bulk copy while the first round
  // decodes and gathers; the warps wait on its mbarrier right before they first read the table
  if (BIN && threadIdx.x == 0) bulk_copy_g2s(s_low, A.lowtab, (uint32_t)(128 * A.lwp * sizeof(double)), &s_bar);
  bool low_ready = !BIN;
  const unsigned lane = lane_id();
  const int wib = threadIdx.x >> 5;
  const int c = P.c;
  long long bias_acc = 0;
  const int64_t first = (int64_t)blockIdx.x * A.rpb, last = first + A.rpb < A.n ? first + A.rpb : A.n;
  for (int64_t base = first; base < last; base += RR) {
    ImpWindow W[IMP_R];
    uint32_t IDX[IMP_R][CC];
    int gpl[IMP_R];                         // groups per lane of the row
    // ---- (A) decode + gather ----
#pragma unroll
    for (int r = 0; r < IMP_R; r++) {
      const int64_t row = base + wib * IMP_R + r;
      gpl[r] = 0;
      if (row >= last) continue;
      const int L = (int)A.len[row];
      const uint32_t *b2 = A.bits2 + A.blk[row] * 4;
      const uint16_t *iv = A.inv16 + A.blk[row] * 4;
      const int ngroups = P.Mlo <= P.N ? (L + c - 1) / c : 0;
      const int G = (ngroups + 31) >> 5;
      gpl[r] = G;
      const int p0 = (int)lane * G * c;
      double s = 0.0;
      if (CACHE > 0) {
        W[r].load(b2, iv, L, p0);
#pragma unroll
        for (int i = 0; i < CC; i++) {
          uint32_t ix = IMP_NOIDX;
          if (i < G) {
            ix = imp_group(P, W[r], i * c);
            if (ix == IMP_SINGLES)
              for (int t = 0; t < c; t++) {
                const uint32_t i1 = imp_single(P, W[r], i * c + t);
                if (i1 != IMP_NOIDX) s += __ldg(A.T + i1);
              }
          }
          IDX[r][i] = ix;
        }
#pragma unroll
        for (int i = 0; i < CC; i++)
          if (IDX[r][i] < IMP_SINGLES) s += __ldg(A.T + IDX[r][i]);
      } else {
        for (int g0 = 0; g0 < G; g0 += A.gw) {
          ImpWindow V;
          V.load(b2, iv, L, p0 + g0 * c);
          const int ge = G - g0 < A.gw ? G - g0 : A.gw;
          for (int i = 0; i < ge; i++) {
            const uint32_t ix = imp_group(P, V, i * c);
            if (ix == IMP_SINGLES) {
              for (int t = 0; t < c; t++) {
                const uint32_t i1 = imp_single(P, V, i * c + t);
                if (i1 != IMP_NOIDX) s += __ldg(A.T + i1);
              }
            } else if (ix != IMP_NOIDX) s += __ldg(A.T + ix);
          }
        }
      }
      if (BIN) {
        if (!low_ready) { mbar_wait(&s_bar, 0); low_ready = true; }
        // table levels: 8 precomputed sums per word of the row's class bitmap
        for (int l = (int)lane; l < A.low_words; l += 32) {
          const uint32_t w = __ldcs(A.lowbits + row * A.low_words + l);
#pragma unroll
          for (int i = 0; i < 8; i++) s += s_low[(i * 16 + ((w >> (4 * i)) & 15u)) * A.lwp + l];
        }
        // repeats of a class inside the row: the count formulation counted them, a binarized row does not
        const int64_t e0 = A.evptr[row];
        const uint32_t nd = (uint32_t)(A.evptr[row + 1] - e0);
        for (uint32_t e = lane; e < nd; e += 32) s -= __ldg(A.theta + A.events[e0 + e] + 1);
      }
      s = warp_sum_down(s);
      if (lane == 0) s_z[wib * IMP_R + r] = s;
    }
    __syncthreads();
    // ---- (B) Gradient weight (:166-178) and Loss term (:257-263) of the round's rows, one lane per row ----
    if (threadIdx.x < RR && base + threadIdx.x < last) {
      const int64_t row = base + threadIdx.x;
      const double w = row_weight(A.theta[0] + s_z[threadIdx.x], A.labels[row], A.cw0, A.cw1, A.inv_n, A.lossterm[row]);
      const unsigned long long q = (unsigned long long)__double2ll_rn(w * A.scale);
      s_q[threadIdx.x] = q;
      if (A.scatter) { bias_acc += (long long)q; if (BIN) A.q_out[row] = q; }
    }
    __syncthreads();
    if (!A.scatter) continue;               // loss-only pass (the hook after the last iteration)
    // ---- (C) scatter ----
#pragma unroll
    for (int r = 0; r < IMP_R; r++) {
      const int64_t row = base + wib * IMP_R + r;
      if (row >= last) continue;
      const unsigned long long q = s_q[wib * IMP_R + r];
      const int G = gpl[r];
      if (CACHE > 0) {
#pragma unroll
        for (int i = 0; i < CC; i++) {
          if (IDX[r][i] < IMP_SINGLES) atomicAdd(A.H + IDX[r][i], q);
          else if (IDX[r][i] == IMP_SINGLES)
            for (int t = 0; t < c; t++) {
              const uint32_t i1 = imp_single(P, W[r], i * c + t);
              if (i1 != IMP_NOIDX) atomicAdd(A.H + i1, q);
            }
        }
      } else {
        const int L = (int)A.len[row];
        const uint32_t *b2 = A.bits2 + A.blk[row] * 4;
        const uint16_t *iv = A.inv16 + A.blk[row] * 4;
        const int p0 = (int)lane * G * c;
        for (int g0 = 0; g0 < G; g0 += A.gw) {
          ImpWindow V;
          V.load(b2, iv, L, p0 + g0 * c);
          const int ge = G - g0 < A.gw ? G - g0 : A.gw;
          for (int i = 0; i < ge; i++) {
            const uint32_t ix = imp_group(P, V, i * c);
            if (ix == IMP_SINGLES) {
              for (int t = 0; t < c; t++) {
                const uint32_t i1 = imp_single(P, V, i * c + t);
                if (i1 != IMP_NOIDX) atomicAdd(A.H + i1, q);
              }
            } else if (ix != IMP_NOIDX) atomicAdd(A.H + ix, q);
          }
        }
      }
      if (BIN) {
        const unsigned long long nq = 0ull - q;
        const int64_t e0 = A.evptr[row];
        const uint32_t nd = (uint32_t)(A.evptr[row + 1] - e0);
        for (uint32_t e = lane; e < nd; e += 32) atomicAdd(A.G + A.events[e0 + e] + 1, nq);
      }
    }
  }
  // bias column: one atomic per block
  if (bias_acc != 0) atomicAdd(&s_bias, (unsigned long long)bias_acc);
  __syncthreads();
  if (threadIdx.x == 0 && s_bias != 0ull) atomicAdd(&A.G[0], s_bias);
}

// binarized rows, table levels: G[column of class j] += sum_i q_i [bit j of row i].  A warp walks rows; lane l
// owns word w0 + l of the row's bitmap and keeps one 64-bit accumulator per bit in registers (no atomics in
// the loop); the warps of a block are summed in shared memory, one atomic per class and block at the end.
// (Folding this into imp_pass -- register accumulators per thread, flushed per block -- made the pass slower
// than the two kernels together: 4.86 vs 3.8 + 0.65 ms at C3; imp_pass is bound by its scattered accesses and
// lost a resident block per SM to the extra registers.)
__global__ void __launch_bounds__(256) low_accumulate(const uint32_t *__restrict__ lowbits, int low_words, int w0, int64_t n,
                                                      const unsigned long long *__restrict__ q,
                                                      const uint32_t *__restrict__ lowcol, unsigned long long *__restrict__ G,
                                                      const PgState *st) {
  if (st && st->done == 1) return;
  __shared__ unsigned long long sacc[32 * 32];
  const unsigned lane = lane_id();
  const int word = w0 + (int)lane, wib = threadIdx.x >> 5;
  const bool on = word < low_words;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  unsigned long long acc[32];
#pragma unroll
  for (int b = 0; b < 32; b++) acc[b] = 0ull;
  for (int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < n; row += nwarps) {
    const unsigned long long qq = q[row];
    const uint32_t w = on ? __ldcs(lowbits + row * low_words + word) : 0u;
#pragma unroll
    for (int b = 0; b < 32; b++)
      if ((w >> b) & 1u) acc[b] += qq;
  }
  for (int i = threadIdx.x; i < 1024; i += blockDim.x) sacc[i] = 0ull;
  __syncthreads();
  for (int v = 0; v < (int)(blockDim.x >> 5); v++) {
    if (wib == v) {
#pragma unroll
      for (int b = 0; b < 32; b++) sacc[b * 32 + lane] += acc[b];
    }
    __syncthreads();
  }
  for (int i = threadIdx.x; i < 1024; i += blockDim.x) {
    const int b = i >> 5, l = i & 31;
    const unsigned long long v = sacc[i];
    if (v && w0 + l < low_words) {
      const uint32_t col = lowcol[(w0 + l) * 32 + b];
      if (col != NOCOL) atomicAdd(G + col + 1, v);
    }
  }
}

// G[col + 1] += F_k[code] + F_k[image(code)] for column j if it is one of the matrix-free levels (G holds the repeat
// corrections of binarized rows by now, zero otherwise)
__device__ __forceinline__ void imp_column(const ImpParams &P, const uint32_t *__restrict__ col_id, int64_t j,
                                           const unsigned long long *__restrict__ F, unsigned long long *__restrict__ G) {
  const uint32_t id = col_id[j];
  int k = P.M;
  while (k < P.N && id >= P.level_off[k + 1]) k++;
  if (k < P.Mlo) return;
  const uint32_t c = id - P.level_off[k];
  unsigned long long g = F[P.fo[k] + c];
  if (P.op) { const uint32_t r = kmer_op(c, k, P.op); if (r != c) g += F[P.fo[k] + r]; }
  G[j + 1] += g;
}

// pair mode: the weights come from the pair-aware rows kernel; same fixed-point accumulation
template <typename VT>
__global__ void scatter_w(const Rows R, const uint32_t *__restrict__ col,
                          const VT *__restrict__ val, int64_t n, const double *__restrict__ w, double scale,
                          double scale0, unsigned long long *__restrict__ G) {
  int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (row >= n) return;
  unsigned lane = lane_id();
  const double ws = w[row] * scale;
  if (lane == 0) atomicAdd(&G[0], (unsigned long long)__double2ll_rn(w[row] * scale0));
  int64_t a, b;
  R.range(row, a, b);
  for (int64_t p = a + lane; p < b; p += 32)
    atomicAdd(&G[col[p] + 1], (unsigned long long)__double2ll_rn(ws * valf(val, p)));
}

// g[j] = G[j] / S for the single-feature coefficients (the bias has a scale of its own, see set_scale)
__global__ void finalize_g(const unsigned long long *__restrict__ G, int64_t count, double inv_scale, double inv_scale0,
                           double *__restrict__ g) {
  int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j < count) g[j] = (double)(long long)G[j] * (j == 0 ? inv_scale0 : inv_scale);
}

// pair coefficients (kmerLr_logistic_regression.go:183-195): g[Ind2Sub(a,b)] = sum_i (w_i v_ia) v_ib, a < b.
// One block per pair of column tiles (32 x 32 pair accumulators in registers: warp = 4 columns a, lane = column
// b).  The rows go by in chunks: the block spreads the B tile's entries of the chunk into a dense [row][b] array
// in shared memory, then every warp walks the entries of its a columns IN ROW ORDER and adds (w_r v_ra) x the
// dense row to its 32 accumulators -- a zero of the dense row adds +0.0, which changes nothing.  Every pair is
// therefore summed in increasing sample order with the reference's product (w v1) v2, i.e. bit for bit what the
// serial Go loop computes, without the per-element binary search of one warp per pair (227 ms at C4 before).
constexpr int PAIR_T = 32;         // tile edge, columns
constexpr int PAIR_CH = 256;       // rows per chunk: PAIR_CH x PAIR_T doubles = 64 KB of shared memory
template <typename VT>
__global__ void __launch_bounds__(256) pairs_gradient(const int64_t *__restrict__ colptr, const uint32_t *__restrict__ crow,
                                                      const VT *__restrict__ cval, int64_t m, int64_t n, int ntile,
                                                      const double *__restrict__ w, double *__restrict__ g) {
  extern __shared__ __align__(16) double Bd[];            // [PAIR_CH][PAIR_T], then the warps' staging areas
  __shared__ int64_t pb[PAIR_T];
  double *st_t = Bd + PAIR_CH * PAIR_T + (threadIdx.x >> 5) * PAIR_CH;                                       // w_r v_ra
  unsigned short *st_r = reinterpret_cast<unsigned short *>(Bd + PAIR_CH * PAIR_T + 8 * PAIR_CH) + (threadIdx.x >> 5) * PAIR_CH;   // local row
  // tile pair (ta <= tb) of this block: row-major over the upper triangle, diagonal included
  int64_t rest = blockIdx.x;
  int ta = 0;
  while (rest >= ntile - ta) { rest -= ntile - ta; ta++; }
  const int tb = ta + (int)rest;
  const int64_t a0 = (int64_t)ta * PAIR_T, b0 = (int64_t)tb * PAIR_T;
  const unsigned lane = lane_id();
  const int wib = threadIdx.x >> 5;
  int64_t pa[4], ea[4];
  double acc[4];
#pragma unroll
  for (int i = 0; i < 4; i++) {
    const int64_t a = a0 + wib * 4 + i;
    pa[i] = a < m ? colptr[a] : 0; ea[i] = a < m ? colptr[a + 1] : 0;
    acc[i] = 0.0;
  }
  if (threadIdx.x < PAIR_T) pb[threadIdx.x] = b0 + threadIdx.x < m ? colptr[b0 + threadIdx.x] : 0;
  for (int64_t lo = 0; lo < n; lo += PAIR_CH) {
    const int64_t hi = lo + PAIR_CH < n ? lo + PAIR_CH : n;
    for (int i = threadIdx.x; i < PAIR_CH * PAIR_T / 2; i += blockDim.x) reinterpret_cast<double2 *>(Bd)[i] = make_double2(0.0, 0.0);
    __syncthreads();
    // the B tile's entries of this chunk -> dense rows (a warp takes 4 columns; the entries of a column are sorted by row)
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const int bc = wib * 4 + i;
      const int64_t b = b0 + bc;
      if (b >= m) continue;
      int64_t p = pb[bc];
      const int64_t end = colptr[b + 1];
      for (;;) {
        const int64_t q = p + lane;
        const uint32_t r = q < end ? crow[q] : 0xFFFFFFFFu;
        const bool in = q < end && (int64_t)r < hi;
        if (in) Bd[(r - lo) * PAIR_T + bc] = valf(cval, q);
        const int cnt = __popc(__ballot_sync(0xffffffffu, in));
        p += cnt;
        if (cnt < 32) break;
      }
      __syncwarp();
      if (lane == 0) pb[bc] = p;
    }
    __syncthreads();
    // the a columns of this warp, entries in row order: acc[a][b] += (w_r v_ra) v_rb.  The lanes stage the
    // column's entries of the chunk (local row, w_r v_ra) in shared memory with coalesced loads; the serial
    // walk then reads broadcasts whose addresses are known ahead, so only the chain of additions is left
#pragma unroll
    for (int i = 0; i < 4; i++) {
      int64_t p = pa[i];
      int cnt_tot = 0;
      for (;;) {
        const int64_t q = p + lane;
        const uint32_t r = q < ea[i] ? crow[q] : 0xFFFFFFFFu;
        const bool in = q < ea[i] && (int64_t)r < hi;
        if (in) { st_r[cnt_tot + lane] = (unsigned short)(r - lo); st_t[cnt_tot + lane] = __ldg(w + r) * valf(cval, q); }
        const int cnt = __popc(__ballot_sync(0xffffffffu, in));
        p += cnt; cnt_tot += cnt;
        if (cnt < 32) break;
      }
      pa[i] = p;
      __syncwarp();
      double a_ = acc[i];
      int e = 0;
      for (; e + 4 <= cnt_tot; e += 4) {
        double d[4], t[4];
#pragma unroll
        for (int q = 0; q < 4; q++) { t[q] = st_t[e + q]; d[q] = Bd[(int)st_r[e + q] * PAIR_T + lane]; }
#pragma unroll
        for (int q = 0; q < 4; q++) a_ += t[q] * d[q];
      }
      for (; e < cnt_tot; e++) a_ += st_t[e] * Bd[(int)st_r[e] * PAIR_T + lane];
      acc[i] = a_;
      __syncwarp();
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; i++) {
    const int64_t a = a0 + wib * 4 + i, b = b0 + lane;
    if (a < m && b < m && a < b) g[ind2sub(m, a, b)] = acc[i];
  }
}

__global__ void add_l1_sign(const double *__restrict__ theta, double *__restrict__ g, int64_t ntheta, double lambda) {
  int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j < 1 || j >= ntheta) return;
  if (theta[j] < 0) g[j] -= lambda; else if (theta[j] > 0) g[j] += lambda;
}

// sum over ranks in rank order (deterministic, identical on every rank)
__global__ void sum_ranks(const double *__restrict__ gathered, int world, int64_t count, double *__restrict__ out) {
  int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= count) return;
  double s = 0.0;
  for (int r = 0; r < world; r++) s += gathered[(int64_t)r * count + j];
  out[j] = s;
}

// Sharded loss: the per-rank loss sums ride in the gradient all-reduce.  Rank r puts the bits of its sum into
// slot r and zeros into the other slots: the int64 sum over the ranks then returns every rank's bits
// unchanged, and every rank adds the sums in rank order (the same bits everywhere).
__global__ void pack_loss_slots(const PgState *st, const double *__restrict__ local, unsigned long long *__restrict__ slots,
                                int rank, int world) {
  if (st && st->done == 1) return;
  const int r = threadIdx.x;
  if (r < world) slots[r] = r == rank ? (unsigned long long)__double_as_longlong(local[0]) : 0ull;
}

// hook (kmerLr_estimator_hook.go:46-99): loss = mean + lambda * sum_{j=1..m} |theta_j|, run by one warp.  losssum:
// the sum of the loss terms (lane 0); l1part[b] = sum over block b's stride of lambda |theta_j|, j >= 1, added up
// in a fixed order (deterministic)
__device__ __forceinline__ void hook_warp(PgState *st, double losssum, const double *l1part, int nparts, double inv_n,
                                          double eps_loss) {
  double l1 = 0.0;
  for (int b = (int)lane_id(); b < nparts; b += 32) l1 += __ldcg(l1part + b);
  l1 = warp_sum_down(l1);
  if (lane_id() == 0) hook_update(st, losssum * inv_n + l1, eps_loss);
}

// the loss sums of the ranks in rank order, then the hook (one warp)
__global__ void unpack_loss_hook(PgState *st, const unsigned long long *__restrict__ slots, int world,
                                 double *__restrict__ out, const double *l1part, int nparts, double inv_n, double eps_loss) {
  if (st->done == 1) return;
  double s = 0.0;
  if (threadIdx.x == 0) {
    for (int r = 0; r < world; r++) s += __longlong_as_double((long long)slots[r]);
    out[0] = s;
  }
  hook_warp(st, s, l1part, nparts, inv_n, eps_loss);
}

// sum of v over the 256 threads of the block in a fixed tree (deterministic), returned to every thread
__device__ __forceinline__ double block_sum_256(double *sh, double v) {
  sh[threadIdx.x] = v;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
    __syncthreads();
  }
  const double r = sh[0];
  __syncthreads();
  return r;
}

// The tail of a pass, one launch of RED_BLOCKS x 256 threads: the columns of the matrix-free levels (F != nullptr:
// a gradient pass over the forward-code tables), the block's partial sum of the loss terms (a fixed grid over
// strided elements) and the block's partial sum of lambda |theta_j|.  The block that finishes last adds the loss
// partials (one warp, lane l the partials l, l + 32, ..., then a fixed shuffle tree) into losssum[0] and, unless
// the loss sums of the ranks have to be exchanged first (hook = 0), runs the hook.  `ticket` is zero on entry and
// left zero.
__global__ void __launch_bounds__(256) pass_tail(PgState *st, const ImpParams P, const uint32_t *__restrict__ col_id,
                                                 int64_t m, const unsigned long long *__restrict__ F,
                                                 unsigned long long *__restrict__ G, const double *__restrict__ lossterm,
                                                 int64_t n, double *__restrict__ part, double *__restrict__ losssum,
                                                 const double *__restrict__ theta, int64_t ntheta, double lambda,
                                                 double *__restrict__ l1part, int hook, double inv_n, double eps_loss,
                                                 unsigned int *ticket) {
  if (st && st->done == 1) return;
  __shared__ double sh[256];
  const int64_t stride = (int64_t)gridDim.x * blockDim.x, i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (F)
    for (int64_t j = i0; j < m; j += stride) imp_column(P, col_id, j, F, G);
  double s = 0.0;
  for (int64_t i = i0; i < n; i += stride) s += lossterm[i];
  s = block_sum_256(sh, s);
  if (threadIdx.x == 0) part[blockIdx.x] = s;
  double l1 = 0.0;
  if (!isnan(lambda) && lambda != 0.0)
    for (int64_t j = 1 + i0; j < ntheta; j += stride) l1 += lambda * fabs(theta[j]);
  l1 = block_sum_256(sh, l1);
  if (threadIdx.x == 0) l1part[blockIdx.x] = l1;
  if (!last_block(ticket)) return;
  if (threadIdx.x < 32) {
    double t = 0.0;
    for (int i = threadIdx.x; i < (int)gridDim.x; i += 32) t += __ldcg(part + i);
    t = warp_sum_down(t);
    if (threadIdx.x == 0) { losssum[0] = t; *ticket = 0u; }
    if (hook) hook_warp(st, t, l1part, (int)gridDim.x, inv_n, eps_loss);
  }
}

// theta <- prox(theta - s g), eval_stopping (kmerLr_estimator_proximal.go:30-52,88-98): a grid-wide update with
// per-block max |theta|, max |delta| and NaN flag; the block that finishes last takes the decision.  `ticket` is
// zero on entry and left zero.
__global__ void prox_update(PgState *st, double *__restrict__ theta, const unsigned long long *__restrict__ G,
                            double inv_scale, double inv_scale0, int64_t ntheta, double step, double lambda,
                            double *__restrict__ blockmax, double eps, long long max_iter, unsigned int *ticket) {
  if (st->done) return;
  __shared__ double shx[256], shd[256], shn[256];
  double mx = 0.0, md = 0.0, nn = 0.0;
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < ntheta; k += (int64_t)gridDim.x * blockDim.x) {
    double g = (double)(long long)G[k] * (k == 0 ? inv_scale0 : inv_scale);
    double t0 = theta[k], t1 = t0 - step * g;
    if (k > 0) t1 = soft_threshold(t1, step * lambda);
    theta[k] = t1;
    if (isnan(t1)) nn = 1.0;
    mx = fmax(mx, fabs(t1));
    md = fmax(md, fabs(t1 - t0));
  }
  shx[threadIdx.x] = mx; shd[threadIdx.x] = md; shn[threadIdx.x] = nn;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) {
      shx[threadIdx.x] = fmax(shx[threadIdx.x], shx[threadIdx.x + o]);
      shd[threadIdx.x] = fmax(shd[threadIdx.x], shd[threadIdx.x + o]);
      shn[threadIdx.x] = fmax(shn[threadIdx.x], shn[threadIdx.x + o]);
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) { blockmax[3 * blockIdx.x] = shx[0]; blockmax[3 * blockIdx.x + 1] = shd[0]; blockmax[3 * blockIdx.x + 2] = shn[0]; }
  if (!last_block(ticket) || threadIdx.x >= 32) return;
  mx = 0.0; md = 0.0; nn = 0.0;
  for (int i = threadIdx.x; i < (int)gridDim.x; i += 32) {
    mx = fmax(mx, __ldcg(blockmax + 3 * i)); md = fmax(md, __ldcg(blockmax + 3 * i + 1)); nn = fmax(nn, __ldcg(blockmax + 3 * i + 2));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    md = fmax(md, __shfl_xor_sync(0xffffffffu, md, o));
    nn = fmax(nn, __shfl_xor_sync(0xffffffffu, nn, o));
  }
  if (threadIdx.x == 0) {
    *ticket = 0u;
    pg_stop(st, mx, md, nn, eps, max_iter);
  }
}

// ---- small problems (reduced matrices of the leapfrog path: <= 1023 columns, short rows) -----------------
// An iteration is latency / launch bound there.  Sharded matrices: ONE launch of fused_small_kernel per
// iteration (one thread per row, theta and the fixed-point gradient accumulators in shared memory, loss
// partial per block; without a communicator the block that finishes last runs small_tail: loss, hook,
// prox update, stopping rule, clears G).  One GPU: fused_small_persistent, thousands of iterations per
// cooperative launch.
constexpr int SMALL_MAX_THETA = 1024;

// hook (kmerLr_estimator_hook.go:46-99) + prox step + eval_stopping (kmerLr_estimator_proximal.go:30-52,88-98),
// run by ONE block of 256 threads once every block's partials are in
template <int BT = 256>
__device__ __forceinline__ void small_tail(PgState *st, const double *blockloss, int nblocks, double *theta,
                                           unsigned long long *G,
                                           double inv_scale, double inv_scale0, int64_t ntheta, double inv_n, double lambda,
                                           double eps_loss, double step, double eps, long long max_iter,
                                           bool clear_g = true, int replicas = 1) {
  constexpr int NW = BT / 32;
  __shared__ double sh[3][NW];
  __shared__ int s_done;
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
  // loss = sum of the block partials (index order inside a thread, fixed tree across threads) + L1 term;
  // the partials were written by other blocks (read in L2), four loads in flight per thread
  double s = 0.0, l1 = 0.0;
  for (int i = t; i < nblocks; i += 4 * BT) {
    const double v0 = __ldcg(blockloss + i);
    const double v1 = i + BT < nblocks ? __ldcg(blockloss + i + BT) : 0.0;
    const double v2 = i + 2 * BT < nblocks ? __ldcg(blockloss + i + 2 * BT) : 0.0;
    const double v3 = i + 3 * BT < nblocks ? __ldcg(blockloss + i + 3 * BT) : 0.0;
    s += v0; s += v1; s += v2; s += v3;
  }
  if (!isnan(lambda) && lambda != 0.0)
    for (int64_t j = 1 + t; j < ntheta; j += BT) l1 += lambda * fabs(theta[j]);
  // block sums: shuffle tree inside the warps, then the 8 warp sums in warp order (fixed: deterministic)
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { s += __shfl_down_sync(0xffffffffu, s, o); l1 += __shfl_down_sync(0xffffffffu, l1, o); }
  if (lane == 0) { sh[0][wid] = s; sh[1][wid] = l1; }
  __syncthreads();
  if (t == 0) {
    double ssum = sh[0][0], lsum = sh[1][0];
    for (int w = 1; w < NW; w++) { ssum += sh[0][w]; lsum += sh[1][w]; }
    hook_update(st, ssum * inv_n + lsum, eps_loss);
    s_done = st->done;
  }
  __syncthreads();
  if (!s_done) {
    double mx = 0.0, md = 0.0, nn = 0.0;
    for (int64_t k = t; k < ntheta; k += BT) {
      unsigned long long gi = __ldcg(G + k);
      for (int r = 1; r < replicas; r++) gi += __ldcg(G + r * ntheta + k);     // exact integer sum: any order
      double g = (double)(long long)gi * (k == 0 ? inv_scale0 : inv_scale);
      double t0 = theta[k], t1 = t0 - step * g;
      if (k > 0) t1 = soft_threshold(t1, step * lambda);
      theta[k] = t1;
      if (isnan(t1)) nn = 1.0;
      mx = fmax(mx, fabs(t1));
      md = fmax(md, fabs(t1 - t0));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      mx = fmax(mx, __shfl_down_sync(0xffffffffu, mx, o));
      md = fmax(md, __shfl_down_sync(0xffffffffu, md, o));
      nn = fmax(nn, __shfl_down_sync(0xffffffffu, nn, o));
    }
    if (lane == 0) { sh[0][wid] = mx; sh[1][wid] = md; sh[2][wid] = nn; }
    __syncthreads();
    if (t == 0) {
      for (int w = 1; w < NW; w++) { mx = fmax(mx, sh[0][w]); md = fmax(md, sh[1][w]); nn = fmax(nn, sh[2][w]); }
      pg_stop(st, mx, md, nn, eps, max_iter);
    }
  }
  if (clear_g)
    for (int64_t k = t; k < ntheta; k += BT) G[k] = 0ull;     // the next pass accumulates from zero
}

#ifndef KL_SMALL_BPS
#define KL_SMALL_BPS 6
#endif
#ifndef KL_SMALL_REPLICAS
#define KL_SMALL_REPLICAS 4
#endif
constexpr int SMALL_REPLICAS = KL_SMALL_REPLICAS;   // copies of the gradient accumulators (persistent kernel)
constexpr int SMALL_BLOCKS_PER_SM = KL_SMALL_BPS;   // resident blocks per SM the register budget is held to
// the row pass of one block: z, loss terms, weights, fixed-point gradient into G; loss partial into blockloss.
// ONE THREAD PER ROW: the rows are a handful of entries long, so a lane walks its row serially (the sum
// runs in entry order, as the reference's does) and nothing is spent on lane hand-offs; the rows of a warp
// are consecutive, their entries sit next to each other in memory.  (8 lanes per row cost 107 warp
// instructions per row at C2 and made the iteration instruction bound.)
template <typename VT, bool LOAD_THETA = true>
__device__ __forceinline__ void small_rows(const Rows &R, const uint32_t *__restrict__ col, const VT *__restrict__ val,
                                           int64_t n, int64_t ntheta, const double *theta,
                                           const uint8_t *__restrict__ labels, double cw0, double cw1, double inv_n,
                                           double scale, double scale0, unsigned long long *G, double *blockloss,
                                           int scatter, uint32_t *acc_lo, uint32_t *acc_hi, double *sth, double *red) {
  for (int i = threadIdx.x; i < ntheta; i += blockDim.x) {
    acc_lo[i] = 0u; acc_hi[i] = 0u;
    if (LOAD_THETA) sth[i] = theta[i];
  }
  __syncthreads();
  double lacc = 0.0;
  // every block takes an equal, contiguous share of the rows
  const int64_t row_lo = n * blockIdx.x / gridDim.x, row_hi = n * (blockIdx.x + 1) / gridDim.x;
  for (int64_t row = row_lo + threadIdx.x; row < row_hi; row += blockDim.x) {
    int64_t a, b;
    R.range(row, a, b);
    double s = 0.0;
    for (int64_t p = a; p < b; p++) s += valf(val, p) * sth[col[p] + 1];
    double lt;
    const double w = row_weight(sth[0] + s, labels[row], cw0, cw1, inv_n, lt);
    lacc += lt;
    if (!scatter) continue;
    const double ws = w * scale;                    // scale is a power of two: exact
    acc64_add(acc_lo, acc_hi, 0u, (unsigned long long)__double2ll_rn(w * scale0));
    for (int64_t p = a; p < b; p++) acc64_add(acc_lo, acc_hi, col[p] + 1u, (unsigned long long)__double2ll_rn(ws * valf(val, p)));
  }
  // loss partial of the block: shuffle tree inside the warps, then the warp sums in warp order (fixed)
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) lacc += __shfl_down_sync(0xffffffffu, lacc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = lacc;
  __syncthreads();                      // (also: every row of the block is in the accumulators)
  if (threadIdx.x == 0) {
    double l = red[0];
    for (int w = 1; w < (int)(blockDim.x >> 5); w++) l += red[w];
    blockloss[blockIdx.x] = l;
  }
  if (scatter) acc64_flush(acc_lo, acc_hi, ntheta, G);
}

#ifndef KL_LONG_U
#define KL_LONG_U 8
#endif
constexpr int LONG_U = KL_LONG_U;     // loads in flight per thread in the long-row passes (8 against 4, block-local view:
                                      // 40.6 vs 41.8 us at 50 entries per row, 62.4 vs 67.7 at 98, 137 vs 148 at 249)
// Reduced matrices with LONG rows (late epochs of a leapfrog path: the classes of the short k-mers are in every
// row -- 47 entries per row at 100 features of C2).  One thread per row over the compact rows then costs one L1
// wavefront PER LANE and load (the rows of a warp are 200 bytes apart), and the rows of a warp add to the same
// shared-memory accumulator at the same time (every row starts with the same columns): 138 us per iteration at
// 9.4 M entries.  Two more views of the same matrix remove both: the forward sum reads the SLICED view (entry k of
// 32 consecutive rows side by side: one wavefront per warp and load; the sum of a row still runs in entry order,
// so z has the same bits as on the compact rows), leaves the scaled weights in wbuf, and after a grid barrier
// the gradient is a segmented sum over the COLUMN-MAJOR view (contiguous entries, weights gathered by row, a
// thread's entries of one column summed in a register): exact integers -- the same G as the row-wise scatter.
template <typename VT>
struct LongView {
  const int64_t *slice_off; const uint32_t *scol; const VT *sval;     // sliced view (Matrix::ensure_sliced)
  const int64_t *colptr; const uint32_t *crow; const VT *cval;        // column-major view (ensure_csc)
  const uint32_t *spack, *cpack;                                      // both with the count packed in (ensure_packed), or null
  int row_bits;
  double *wbuf;                                                       // n scaled row weights
  int64_t nnz;
  // block-local column-major view (Matrix::bv_*, LONG == 2): the weights of the block's rows stay in shared memory and
  // the gradient of the block's rows is summed by the block itself -- one grid barrier per iteration instead of two
  const int64_t *bv_off; const uint32_t *bv_pack; int bv_row_bits;
};

template <typename VT>
__device__ __forceinline__ void long_forward(const Rows &R, const LongView<VT> &V, int64_t n, int64_t ntheta,
                                             const uint8_t *__restrict__ labels, double cw0, double cw1, double inv_n,
                                             double scale, double scale0, double *blockloss, int scatter, uint32_t *acc_lo,
                                             uint32_t *acc_hi, const double *sth, double *red, double *w_local = nullptr) {
  for (int i = threadIdx.x; i < ntheta; i += blockDim.x) { acc_lo[i] = 0u; acc_hi[i] = 0u; }
  __syncthreads();
  double lacc = 0.0;
  long long bias = 0;
  const int64_t row_lo = n * blockIdx.x / gridDim.x, row_hi = n * (blockIdx.x + 1) / gridDim.x;
  for (int64_t row = row_lo + threadIdx.x; row < row_hi; row += blockDim.x) {
    int64_t a, b;
    R.range(row, a, b);
    const int64_t base = 32 * V.slice_off[row >> 5] + (row & 31);
    const int len = (int)(b - a);
    double s = 0.0;
    if (V.spack) {
      // four loads in flight, the sum in entry order
      const uint32_t *sp = V.spack + base;
      int k = 0;
      for (; k + LONG_U <= len; k += LONG_U) {
        uint32_t e[LONG_U];
#pragma unroll
        for (int j = 0; j < LONG_U; j++) e[j] = __ldg(sp + 32 * (k + j));
#pragma unroll
        for (int j = 0; j < LONG_U; j++) s += (double)(e[j] >> 10) * sth[(e[j] & 1023u) + 1];
      }
      for (; k < len; k++) { const uint32_t e = __ldg(sp + 32 * k); s += (double)(e >> 10) * sth[(e & 1023u) + 1]; }
    } else {
      for (int k = 0; k < len; k++) s += valf(V.sval, base + 32 * k) * sth[V.scol[base + 32 * k] + 1];
    }
    double lt;
    const double w = row_weight(sth[0] + s, labels[row], cw0, cw1, inv_n, lt);
    lacc += lt;
    if (!scatter) continue;
    const double ws = w * scale;
    if (w_local) w_local[row - row_lo] = ws; else V.wbuf[row] = ws;
    bias += __double2ll_rn(w * scale0);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { lacc += __shfl_down_sync(0xffffffffu, lacc, o); bias += __shfl_down_sync(0xffffffffu, bias, o); }
  if ((threadIdx.x & 31) == 0) {
    red[threadIdx.x >> 5] = lacc;
    if (bias) acc64_add(acc_lo, acc_hi, 0u, (unsigned long long)bias);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double l = red[0];
    for (int w = 1; w < (int)(blockDim.x >> 5); w++) l += red[w];
    blockloss[blockIdx.x] = l;
  }
}

// gradient of the block's share of the column-major entries into the block's accumulators, then into G
template <typename VT>
__device__ __forceinline__ void long_columns(const LongView<VT> &V, int64_t ntheta, unsigned long long *G, uint32_t *acc_lo,
                                             uint32_t *acc_hi, const long long *scp, int c_first) {
  const int64_t lo = V.nnz * blockIdx.x / gridDim.x, hi = V.nnz * (blockIdx.x + 1) / gridDim.x;
  int64_t p = lo + threadIdx.x;
  long long acc = 0;
  int c = -1;
  if (p < hi) {
    c = c_first;
    long long cend = scp[c + 1];
    auto boundary = [&](int64_t q) {
      if (q >= cend) {
        if (acc) acc64_add(acc_lo, acc_hi, (uint32_t)c + 1u, (unsigned long long)acc);
        acc = 0;
        do { c++; cend = scp[c + 1]; } while (q >= cend);
      }
    };
    if (V.cpack) {
      const uint32_t rmask = (1u << V.row_bits) - 1u;
      const int64_t bd = blockDim.x;
      for (; p < hi; p += LONG_U * bd) {
        uint32_t e[LONG_U];
        double ws[LONG_U];
#pragma unroll
        for (int j = 0; j < LONG_U; j++) e[j] = p + j * bd < hi ? __ldg(V.cpack + p + j * bd) : 0u;
#pragma unroll
        for (int j = 0; j < LONG_U; j++) ws[j] = __ldcg(V.wbuf + (e[j] & rmask));     // (written by other blocks before the barrier)
#pragma unroll
        for (int j = 0; j < LONG_U; j++) {
          if (p + j * bd < hi) {
            boundary(p + j * bd);
            acc += __double2ll_rn(ws[j] * (double)(e[j] >> V.row_bits));
          }
        }
      }
    } else {
      for (; p < hi; p += blockDim.x) {
        boundary(p);
        const double ws = __ldcg(V.wbuf + V.crow[p]);
        acc += __double2ll_rn(ws * valf(V.cval, p));
      }
    }
  }
  // the threads of a warp mostly end in the same column: one add per warp
  const int c0 = __shfl_sync(0xffffffffu, c, 0);
  if (__all_sync(0xffffffffu, c == c0)) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0 && c >= 0 && acc) acc64_add(acc_lo, acc_hi, (uint32_t)c + 1u, (unsigned long long)acc);
  } else if (c >= 0 && acc) {
    acc64_add(acc_lo, acc_hi, (uint32_t)c + 1u, (unsigned long long)acc);
  }
  __syncthreads();
  acc64_flush(acc_lo, acc_hi, ntheta, G);
}

// LONG == 2: gradient of the block's OWN rows from the block-local view (thread t sums its contiguous share of the
// block's entries, which are sorted by column: a register run per column, a shared-memory add when the column
// changes), the weights read from shared memory; then into G.  The same integer terms as long_columns.
template <typename VT>
__device__ __forceinline__ void block_columns(const LongView<VT> &V, int64_t ntheta, unsigned long long *G, uint32_t *acc_lo,
                                              uint32_t *acc_hi, const double *w_s) {
  const int64_t o0 = V.bv_off[blockIdx.x], wdt = V.bv_off[blockIdx.x + 1] - o0;
  const uint32_t *bp = V.bv_pack + 256 * o0 + threadIdx.x;
  const uint32_t rmask = (1u << V.bv_row_bits) - 1u;
  const int cs = V.bv_row_bits, vs = V.bv_row_bits + 10;
  long long acc = 0;
  int cur = -1;
  for (int64_t j = 0; j < wdt; j += LONG_U) {
    uint32_t e[LONG_U];
#pragma unroll
    for (int i = 0; i < LONG_U; i++) e[i] = j + i < wdt ? __ldg(bp + 256 * (j + i)) : 0xFFFFFFFFu;
#pragma unroll
    for (int i = 0; i < LONG_U; i++) {
      if (e[i] == 0xFFFFFFFFu) continue;
      const int c = (int)((e[i] >> cs) & 1023u);
      if (c != cur) {
        if (acc) acc64_add(acc_lo, acc_hi, (uint32_t)cur + 1u, (unsigned long long)acc);
        acc = 0; cur = c;
      }
      acc += __double2ll_rn(w_s[e[i] & rmask] * (double)(e[i] >> vs));
    }
  }
  if (acc) acc64_add(acc_lo, acc_hi, (uint32_t)cur + 1u, (unsigned long long)acc);
  __syncthreads();
  acc64_flush(acc_lo, acc_hi, ntheta, G);
}

template <typename VT>
__global__ void __launch_bounds__(256, SMALL_BLOCKS_PER_SM) fused_small_kernel(const Rows R, const uint32_t *__restrict__ col,
                                                          const VT *__restrict__ val, int64_t n, int64_t ntheta,
                                                          double *theta, const uint8_t *__restrict__ labels,
                                                          double cw0, double cw1, double inv_n, double scale,
                                                          double scale0, unsigned long long *G, double *blockloss,
                                                          PgState *st, int scatter, unsigned int *counter,
                                                          double inv_scale, double inv_scale0, double lambda, double eps_loss, double step, double eps,
                                                          long long max_iter) {
  if (st->done == 1) return;
  __shared__ uint32_t acc_lo[SMALL_MAX_THETA], acc_hi[SMALL_MAX_THETA];
  __shared__ double sth[SMALL_MAX_THETA];
  __shared__ double red[256];
  small_rows<VT>(R, col, val, n, ntheta, theta, labels, cw0, cw1, inv_n, scale, scale0, G, blockloss, scatter, acc_lo, acc_hi,
                 sth, red);
  // the block that finishes last runs the tail of the iteration (its reads see every block's results)
  if (!counter) return;                 // sharded: the collectives come first, the tail is its own launch
  if (!last_block(counter)) return;
  small_tail(st, blockloss, (int)gridDim.x, theta, G, inv_scale, inv_scale0, ntheta, inv_n, lambda, eps_loss, step, eps,
             max_iter);
  if (threadIdx.x == 0) *counter = 0u;
}

// One GPU, reduced matrix: MANY iterations in one cooperative launch, ONE grid barrier per iteration and no
// serial section.  Every block keeps theta and the iteration state in shared memory; a pass is the row
// pass of all blocks (gradient into G[pass % 3], loss partials into blockloss[pass & 1]), the grid
// barrier, and the tail of the iteration (small_tail: loss, hook, prox step, stopping rule) run by EVERY
// block on the same inputs in the same order -- the same result everywhere, bit for bit, so nobody waits
// for a block 0.  G is triple buffered: block 0 clears G[(pass + 1) % 3] during pass `pass`; that buffer
// was last read in the tail of pass - 2, which every block left before it arrived at the barrier of
// pass - 1.  The loss partials of pass + 2 overwrite those of `pass` for the same reason.  The passes of
// one launch are pass0, pass0 + 1, ...; pass number max_iter only evaluates the hook's loss.
// (1024-thread blocks, one per SM -- fewer loss partials, a cheaper barrier -- measured no faster: 23 vs 21 us)
constexpr int PERSIST_THREADS = 256;
// SHARDED: the rows are this rank's shard and the ranks are connected by NVLink peer memory.  After the grid
// barrier block 0 exchanges the rank's payload (fixed-point gradient + loss partial) with all ranks through
// the mailboxes -- stores into every rank's slot, a flag, a wait for the flags of the others, the sum in rank
// order (integers: the same bits on every rank) -- and a second grid barrier releases the tail.  The
// collective lives INSIDE the persistent kernel: no launch and no NCCL call per iteration.
template <typename VT, bool SHARDED, int LONG>
__global__ void __launch_bounds__(PERSIST_THREADS, SMALL_BLOCKS_PER_SM) fused_small_persistent(
    const Rows R, const uint32_t *__restrict__ col, const VT *__restrict__ val, int64_t n, int64_t ntheta, double *theta,
    const uint8_t *__restrict__ labels, double cw0, double cw1, double inv_n, double scale, double scale0,
    unsigned long long *G3, double *blockloss2, PgState *st, long long pass0, int npass, double inv_scale,
    double inv_scale0, double lambda, double eps_loss,
    double step, double eps, long long max_iter, const PeerBox *pb, unsigned long long *Gx, double *scratch,
    unsigned int *abort_flag, const LongView<VT> LV) {
  cooperative_groups::grid_group grid = cooperative_groups::this_grid();
  __shared__ uint32_t acc_lo[SMALL_MAX_THETA], acc_hi[SMALL_MAX_THETA];
  __shared__ double sth[SMALL_MAX_THETA];
  __shared__ double red[256];
  __shared__ PgState ls;
  __shared__ unsigned long long s_seq;
  __shared__ int s_timeout;
  if (threadIdx.x == 0) {
    ls = *st;
    if (SHARDED) s_seq = pb->box[pb->rank]->seq;
  }
  for (int i = threadIdx.x; i < ntheta; i += blockDim.x) sth[i] = theta[i];
  // LONG: the column offsets stay in shared memory; c_first = the column of this thread's first column-major entry
  __shared__ long long scp[LONG == 1 ? SMALL_MAX_THETA + 1 : 1];
  extern __shared__ __align__(16) double w_s[];          // LONG == 2: the scaled weights of the block's rows
  int c_first = 0;
  if constexpr (LONG == 1) {
    for (int i = threadIdx.x; i < ntheta; i += blockDim.x) scp[i] = LV.colptr[i];        // m + 1 = ntheta offsets
    __syncthreads();
    const int64_t p = LV.nnz * blockIdx.x / gridDim.x + threadIdx.x;
    int a = 0, b = (int)ntheta - 1;                 // scp[a] <= p < scp[b] (empty columns skipped)
    while (b - a > 1) { const int mid = (a + b) >> 1; if (scp[mid] <= p) a = mid; else b = mid; }
    c_first = a;
  }
  __syncthreads();
  const int nblocks = (int)gridDim.x;
  for (int it = 0; it < npass; it++) {
    if (ls.done == 1) break;
    const long long pass = pass0 + it;
    const int scatter = pass < max_iter ? 1 : 0;
    // SMALL_REPLICAS copies of the accumulators (block b adds to copy b mod SMALL_REPLICAS): the L2 serialises
    // atomics on one address, and every block adds to the same ntheta addresses at the end of its rows
    unsigned long long *G = G3 + (pass % 3) * SMALL_REPLICAS * ntheta, *Gnext = G3 + ((pass + 1) % 3) * SMALL_REPLICAS * ntheta;
    double *blockloss = blockloss2 + (pass & 1) * nblocks;
    if (blockIdx.x == 0)
      for (int i = threadIdx.x; i < SMALL_REPLICAS * ntheta; i += blockDim.x) Gnext[i] = 0ull;
    if constexpr (LONG == 1) {
      long_forward<VT>(R, LV, n, ntheta, labels, cw0, cw1, inv_n, scale, scale0, blockloss, scatter, acc_lo, acc_hi, sth,
                       red);
      if (scatter) {
        grid.sync();
        long_columns<VT>(LV, ntheta, G + (blockIdx.x % SMALL_REPLICAS) * ntheta, acc_lo, acc_hi, scp, c_first);
      }
    } else if constexpr (LONG == 2) {
      long_forward<VT>(R, LV, n, ntheta, labels, cw0, cw1, inv_n, scale, scale0, blockloss, scatter, acc_lo, acc_hi, sth,
                       red, w_s);
      if (scatter) block_columns<VT>(LV, ntheta, G + (blockIdx.x % SMALL_REPLICAS) * ntheta, acc_lo, acc_hi, w_s);
    } else {
      small_rows<VT, false>(R, col, val, n, ntheta, sth, labels, cw0, cw1, inv_n, scale, scale0,
                            G + (blockIdx.x % SMALL_REPLICAS) * ntheta, blockloss, scatter, acc_lo, acc_hi, sth, red);
    }
    grid.sync();
    if (!SHARDED) {
      small_tail<PERSIST_THREADS>(&ls, blockloss, nblocks, sth, G, inv_scale, inv_scale0, ntheta, inv_n, lambda, eps_loss,
                                  step, eps, max_iter, false, SMALL_REPLICAS);
    } else {
      if (blockIdx.x == 0) {
        const int t = threadIdx.x, me = pb->rank, world = pb->world;
        PeerMail *mine = pb->box[me];
        const unsigned long long seq = s_seq + 1ull;
        const int par = (int)(seq & 1ull);
        if (t == 0) s_timeout = 0;
        // loss partial of this rank: block partials in a fixed order
        double s = 0.0;
        for (int i = t; i < nblocks; i += PERSIST_THREADS) s += __ldcg(blockloss + i);
        s = block_sum_256(red, s);
        // payload into every mailbox (NVLink stores), one system fence, then the flags
        for (int64_t k = t; k < ntheta; k += PERSIST_THREADS) {
          unsigned long long g = 0ull;
          for (int r = 0; r < SMALL_REPLICAS; r++) g += __ldcg(G + r * ntheta + k);
          for (int r = 0; r < world; r++) pb->box[r]->slot[par][me][k] = g;
        }
        if (t < world) pb->box[t]->slot[par][me][ntheta] = (unsigned long long)__double_as_longlong(s);
        __syncthreads();
        if (t == 0) __threadfence_system();
        __syncthreads();
        if (t < world) {
          *(volatile unsigned long long *)&pb->box[t]->flag[par][me] = seq;
          volatile unsigned long long *f = &mine->flag[par][t];
          const long long t0 = clock64();
          while (*f < seq)
            if (clock64() - t0 > 6000000000LL) { s_timeout = 1; break; }      // ~3 s: a peer is gone
          __threadfence_system();
        }
        __syncthreads();
        if (s_timeout) {
          if (t == 0) *abort_flag = 1u;
        } else {
          for (int64_t k = t; k < ntheta; k += PERSIST_THREADS) {
            unsigned long long g = 0ull;
            for (int r = 0; r < world; r++) g += __ldcv(&mine->slot[par][r][k]);
            Gx[k] = g;
          }
          if (t < world) scratch[t] = __longlong_as_double((long long)__ldcv(&mine->slot[par][t][ntheta]));
        }
        __threadfence();
        if (t == 0) s_seq = seq;
        __syncthreads();
      }
      grid.sync();
      if (*(volatile unsigned int *)abort_flag) {
        if (threadIdx.x == 0) { ls.error = 1; ls.done = 1; }
        __syncthreads();
        break;
      }
      small_tail<PERSIST_THREADS>(&ls, scratch, pb->world, sth, Gx, inv_scale, inv_scale0, ntheta, inv_n, lambda, eps_loss,
                                  step, eps, max_iter, false, 1);
    }
    __syncthreads();
  }
  if (blockIdx.x == 0) {
    for (int i = threadIdx.x; i < ntheta; i += blockDim.x) theta[i] = sth[i];
    if (threadIdx.x == 0) {
      *st = ls;
      if (SHARDED) pb->box[pb->rank]->seq = s_seq;
    }
  }
}

// sharded reduced matrices: sum of the block loss partials (fixed order) -> one double per rank ...
__global__ void __launch_bounds__(256) small_presum_kernel(const PgState *st, const double *__restrict__ blockloss,
                                                           int nblocks, double *__restrict__ out) {
  if (st->done == 1) return;
  __shared__ double sh[256];
  double s = 0.0;
  for (int i = threadIdx.x; i < nblocks; i += 256) s += blockloss[i];
  s = block_sum_256(sh, s);
  if (threadIdx.x == 0) out[0] = s;
}
// ... and the tail over the gathered per-rank losses (rank order) and the all-reduced gradient
__global__ void __launch_bounds__(256) small_tail_kernel(PgState *st, const double *partials, int nparts, double *theta,
                                                         unsigned long long *G, double inv_scale, double inv_scale0,
                                                         int64_t ntheta, double inv_n, double lambda, double eps_loss,
                                                         double step, double eps, long long max_iter) {
  if (st->done == 1) return;
  small_tail(st, partials, nparts, theta, G, inv_scale, inv_scale0, ntheta, inv_n, lambda, eps_loss, step, eps, max_iter);
}

// Sharded reduced matrices, ranks connected by NVLink: the gradient all-reduce, the loss all-gather and
// the tail of the iteration in ONE launch of world + 1 blocks.  Block b < world stores this rank's payload
// (fixed-point gradient + loss partial) straight into rank b's mailbox (peer memory, CUDA IPC) and raises
// this rank's flag there -- the world stores travel in parallel; block `world` waits for the flags of all
// senders in its own mailbox, sums the payloads in rank order -- integers, so every rank holds the same
// bits -- and runs hook / prox step / stopping rule.  Two parities of slots: a sender can be at most one
// exchange ahead of a receiver.  (One block doing the world stores one after the other: 36 us per
// iteration at 8 ranks against 20 us on one GPU.)
__global__ void __launch_bounds__(256) small_p2p_tail_kernel(PgState *st, const PeerBox *pb, const double *__restrict__ blockloss,
                                                             int nblocks, double *theta, unsigned long long *G,
                                                             double *scratch, double inv_scale, double inv_scale0,
                                                             int64_t ntheta, double inv_n,
                                                             double lambda, double eps_loss, double step, double eps,
                                                             long long max_iter) {
  if (st->done == 1) return;
  __shared__ double shs[256];
  __shared__ int s_timeout;
  const int t = threadIdx.x, me = pb->rank, world = pb->world;
  PeerMail *mine = pb->box[me];
  // (the sequence number is bumped by the last block only after every sender block of this launch is through)
  const unsigned long long seq = mine->seq + 1ull;
  const int par = (int)(seq & 1ull);
  if ((int)blockIdx.x < world) {
    // ---- sender: payload into mailbox blockIdx.x (NVLink stores), then the flag ----
    const int dst_rank = (int)blockIdx.x;
    double s = 0.0;
    for (int i = t; i < nblocks; i += 256) s += blockloss[i];      // loss partial of this rank, fixed order
    s = block_sum_256(shs, s);
    unsigned long long *dst = pb->box[dst_rank]->slot[par][me];
    for (int64_t k = t; k < ntheta; k += 256) dst[k] = G[k];
    if (t == 0) dst[ntheta] = (unsigned long long)__double_as_longlong(s);
    __threadfence_system();
    __syncthreads();
    if (t == 0) {
      *(volatile unsigned long long *)&pb->box[dst_rank]->flag[par][me] = seq;
      __threadfence();
      atomicAdd(&mine->senders_done, 1u);
    }
    return;
  }
  // ---- receiver: wait for every sender's flag in my own mailbox ----
  if (t == 0) s_timeout = 0;
  __syncthreads();
  if (t < world) {
    volatile unsigned long long *g = &mine->flag[par][t];
    const long long t0 = clock64();
    while (*g < seq)
      if (clock64() - t0 > 6000000000LL) { s_timeout = 1; break; }      // ~3 s: a peer is gone
  }
  // ... and for my own sender blocks: they read G and the sequence number, both change below
  if (t == 32) {
    volatile unsigned int *d = &mine->senders_done;
    const long long t0 = clock64();
    while (*d < (unsigned)world)
      if (clock64() - t0 > 6000000000LL) { s_timeout = 1; break; }
  }
  __syncthreads();
  if (s_timeout) {
    if (t == 0) { st->error = 1; st->done = 1; mine->senders_done = 0u; }
    return;
  }
  __threadfence_system();
  for (int64_t k = t; k < ntheta; k += 256) {
    unsigned long long g = 0ull;
    for (int r = 0; r < world; r++) g += __ldcv(&mine->slot[par][r][k]);
    G[k] = g;
  }
  if (t < world) scratch[t] = __longlong_as_double((long long)__ldcv(&mine->slot[par][t][ntheta]));
  __threadfence();
  __syncthreads();
  if (t == 0) { mine->senders_done = 0u; mine->seq = seq; }
  small_tail(st, scratch, world, theta, G, inv_scale, inv_scale0, ntheta, inv_n, lambda, eps_loss, step, eps, max_iter);
}

constexpr int PROX_BLOCKS = 256;

struct Work {
  DevBuf<double> theta, w, lossterm, g, red, scalars, gathered, blockmax;
  DevBuf<unsigned long long> G, H;     // H: forward-code tables of the matrix-free pass
  DevBuf<double> T, lowtab;
  DevBuf<unsigned long long> q;        // binarized rows: round(w_i S) of every row, for low_accumulate
  DevBuf<unsigned int> tickets;        // last-block counters of imp_fold, pass_tail, prox_update (zero between launches)
  double scale = 1.0, inv_scale = 1.0;      // the columns of the matrix
  double scale0 = 1.0, inv_scale0 = 1.0;    // the bias (its value is 1 in every row)
  // after a matrix-free gradient pass: the folded tables whose columns pass_tail adds to G (nullptr: none pending)
  const unsigned long long *F = nullptr;
  ImpParams P{};
};

template <typename VT>
const VT *csr_val(const Matrix &M);
template <> const uint32_t *csr_val<uint32_t>(const Matrix &M) { return M.vt == VAL_U32 ? M.val_u32.p : nullptr; }
template <> const double *csr_val<double>(const Matrix &M) { return M.val_f64.p; }
template <typename VT>
const VT *sliced_val(const Matrix &M);
template <> const uint32_t *sliced_val<uint32_t>(const Matrix &M) { return M.vt == VAL_U32 ? M.sval_u32.p : nullptr; }
template <> const double *sliced_val<double>(const Matrix &M) { return M.sval_f64.p; }
template <typename VT>
const void *persistent_kernel(bool sharded, int long_mode) {
  if (sharded) return long_mode == 2 ? (const void *)fused_small_persistent<VT, true, 2>
                    : long_mode == 1 ? (const void *)fused_small_persistent<VT, true, 1> : (const void *)fused_small_persistent<VT, true, 0>;
  return long_mode == 2 ? (const void *)fused_small_persistent<VT, false, 2>
       : long_mode == 1 ? (const void *)fused_small_persistent<VT, false, 1> : (const void *)fused_small_persistent<VT, false, 0>;
}
template <typename VT>
const VT *csc_val(const Matrix &M);
template <> const uint32_t *csc_val<uint32_t>(const Matrix &M) { return M.vt == VAL_U32 ? M.cval_u32.p : nullptr; }
template <> const double *csc_val<double>(const Matrix &M) { return M.cval_f64.p; }

inline unsigned warp_grid(int64_t items, int threads) { return (unsigned)((items * 32 + threads - 1) / threads); }

// the non-zero pair coefficients of a host theta, in coefficient order; empty optional = too many (dense theta)
constexpr int64_t PAIR_TERMS_MAX = 8192;
struct PairTerms {
  bool sparse = false;
  DevBuf<PairTerm> dev;
  int n = 0;
};
void collect_pair_terms(const Matrix &M, const double *theta_host, int64_t ntheta, int cooc, PairTerms &T) {
  if (!cooc) return;
  std::vector<PairTerm> h;
  const uint64_t *bits = reinterpret_cast<const uint64_t *>(theta_host);
  for (int64_t j = M.m + 1; j < ntheta; j++) {
    // (blocks of eight zeros -- the normal case -- are skipped with integer ORs; the shift drops the sign of -0.0)
    if (j + 8 <= ntheta && (((bits[j] | bits[j + 1] | bits[j + 2] | bits[j + 3] | bits[j + 4] | bits[j + 5] | bits[j + 6] | bits[j + 7]) << 1) == 0)) { j += 7; continue; }
    if (theta_host[j] == 0.0) continue;
    if ((int64_t)h.size() >= PAIR_TERMS_MAX) return;          // dense theta: the O(q^2) path
    int64_t a, b;
    kmerlr_coeff_sub2ind(M.m, j - 1, &a, &b);
    h.push_back(PairTerm{(uint32_t)a, (uint32_t)b, theta_host[j]});
  }
  T.sparse = true; T.n = (int)h.size();
  T.dev.alloc(h.size() ? h.size() : 1);
  T.dev.upload(h.data(), h.size());
  sync_stream();                                                // (h goes out of scope)
}

template <typename VT, int MODE>
void launch_rows(const Matrix &M, const double *theta, int cooc, const double cw[2], double *out, double *lossterm,
                 const PgState *st, const PairTerms *T = nullptr) {
  if (M.n == 0) return;
  double inv_n = 1.0 / (double)M.n_global;
  const bool sparse = cooc && T && T->sparse;
  KL_LAUNCH((rows_kernel<VT, MODE>), warp_grid(M.n, 256), 256, 0, M.rows(), M.col.p, csr_val<VT>(M), M.n, M.m,
            theta, sparse ? 2 : cooc, M.labels.p, cw ? cw[0] : 1.0, cw ? cw[1] : 1.0, inv_n, out, lossterm, st,
            sparse ? T->dev.p : (const PairTerm *)nullptr, sparse ? T->n : 0);
}

// fixed-point scales: sum_i |w_i v_ic| <= max(cw) * max|v| for a column, <= max(cw) for the bias, each kept below
// 2^60.  The columns of a matrix whose values are all below 1 get the finer scale their bound allows (a matrix of
// frequencies would otherwise lose the bits between max|v| and 1); the bias keeps max(cw) * max(max|v|, 1).  Both
// are the same whenever max|v| >= 1, as in every count and binarized matrix.
void set_scale(Matrix &M, Work &wk, const double cw[2]) {
  const double cmax = std::fmax(std::fabs(cw[0]), std::fabs(cw[1])), vmax = matrix_vmax(M);
  const int e = fixed_point_exponent(cmax * (vmax > 0.0 ? vmax : 1.0)), e0 = fixed_point_exponent(cmax * std::fmax(vmax, 1.0));
  wk.scale = std::ldexp(1.0, e);
  wk.inv_scale = std::ldexp(1.0, -e);
  wk.scale0 = std::ldexp(1.0, e0);
  wk.inv_scale0 = std::ldexp(1.0, -e0);
}

// kmerlr_option("implicit", 0) or KMERLR_IMPLICIT=0 forces the pass over the stored rows (tests compare the two)
bool use_implicit(const Matrix &M) {
  static int env = -1;
  if (env < 0) { const char *e = getenv("KMERLR_IMPLICIT"); env = (e && *e == '0') ? 0 : 1; }
  if (!(env == 1 && ctx().implicit_ok && M.imp)) return false;      // (rank invariant: no look at the local row count)
  return M.imp->binarized ? M.vt == VAL_ONE : M.vt == VAL_U32;
}

// length of the super k-mer tables for k-mers of up to N bases: 4^S entries of 8 bytes for T and for H must
// stay L2 resident (S = 10: 8 MB each, S = 11: 32 MB each)
int super_length(int N) {
  int S = ctx().super_len;
  if (S < 0) S = N <= 8 ? 10 : IMP_SUPER_MAX;
  if (S > IMP_SUPER_MAX) S = IMP_SUPER_MAX;
  return S < N ? N : S;
}

template <int CACHE, bool BIN>
void launch_imp_pass(const ImpParams &P, const ImpArgs &A, size_t smem) {
  if (smem > 48 * 1024)
    KL_CUDA(cudaFuncSetAttribute((imp_pass<CACHE, BIN>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t blocks = (A.n + A.rpb - 1) / A.rpb;
  KL_LAUNCH((imp_pass<CACHE, BIN>), (unsigned)blocks, 256, smem, P, A);
}

void launch_implicit(Matrix &M, Work &wk, const double cw[2], const PgState *st, int scatter) {
  KL_INVARIANT(wk.scale == wk.scale0);       // (one round(w_i S) per row serves the bias and the columns)
  const Implicit &I = *M.imp;
  const SeqSet &S = *I.seqs;
  ImpParams P{};
  P.M = I.M; P.N = I.N; P.op = I.op; P.Mlo = I.Mlo;
  for (int k = 0; k < 16; k++) { P.level_off[k] = I.level_off[k]; P.fo[k] = I.fo[k]; }
  const bool levels = I.Mlo <= I.N;            // (a binarized matrix with N <= 5 has table levels only)
  wk.F = nullptr;
  P.S = levels ? super_length(I.N) : I.N;
  P.c = P.S - I.N + 1;
  const int64_t tlev = levels ? I.fo[I.N + 1] : 0, tsup = P.c > 1 ? (int64_t)1 << (2 * P.S) : 0, total = tlev + tsup;
  P.sup0 = P.c > 1 ? (uint32_t)tlev : I.fo[I.N];
  if (wk.T.n < (size_t)(total ? total : 1)) { wk.T.alloc((size_t)(total ? total : 1)); wk.H.alloc((size_t)(total ? total : 1)); }
  if (scatter && total) KL_CUDA(cudaMemsetAsync(wk.H.p, 0, (size_t)total * sizeof(unsigned long long), ctx().stream));
  if (levels) {
    KL_LAUNCH(imp_build_T, (unsigned)((tlev + 255) / 256), 256, 0, P, I.num->bits.p, I.num->rank.p, wk.theta.p, wk.T.p, tlev, st);
    if (P.c > 1) KL_LAUNCH(imp_build_TS, (unsigned)((tsup + 255) / 256), 256, 0, P, wk.T.p, st);
  }
  ImpArgs A{};
  A.n = M.n; A.len = S.len.p; A.blk = S.blk.p; A.bits2 = S.bits2.p; A.inv16 = S.inv16.p;
  A.T = wk.T.p; A.theta = wk.theta.p; A.labels = M.labels.p;
  A.cw0 = cw[0]; A.cw1 = cw[1]; A.inv_n = 1.0 / (double)M.n_global; A.scale = wk.scale;
  A.H = wk.H.p; A.G = wk.G.p; A.lossterm = wk.lossterm.p; A.st = st; A.scatter = scatter;
  // rows per block: 8 warps x 4 rows; binarized rows amortise the block's copy of lowtab (32 KB) over 16 per warp
  A.rpb = I.binarized ? 128 : 32;
  while ((M.n + A.rpb - 1) / A.rpb > 0x7fffffffLL) A.rpb *= 2;
  size_t smem = 0;
  if (I.binarized) {
    A.lowbits = I.lowbits.p; A.low_words = I.low_words; A.lwp = I.low_words <= 32 ? 32 : 64;
    if (!wk.lowtab.p) { wk.lowtab.alloc((size_t)128 * 64); wk.q.alloc((size_t)M.n); }
    A.lowtab = wk.lowtab.p; A.evptr = I.evptr.p; A.events = I.events.p; A.q_out = wk.q.p;
    smem = (size_t)128 * A.lwp * sizeof(double);
    KL_LAUNCH(imp_build_low, (unsigned)((128 * A.lwp + 255) / 256), 256, 0, I.lowcol.p, I.low_words, A.lwp, wk.theta.p,
              wk.lowtab.p, st);
  }
  // a lane's groups share one 64-bit window of bases when (groups - 1) c + S <= 32
  A.gw = (32 - P.S) / P.c + 1;
  const int64_t groups_per_lane = ((S.max_len + P.c - 1) / P.c + 31) / 32;
  const int64_t cached = groups_per_lane <= A.gw ? groups_per_lane : 1000;
  if (I.binarized) {
    if (cached <= 4) launch_imp_pass<4, true>(P, A, smem);
    else if (cached <= 8) launch_imp_pass<8, true>(P, A, smem);
    else launch_imp_pass<0, true>(P, A, smem);
  } else {
    if (cached <= 4) launch_imp_pass<4, false>(P, A, smem);
    else if (cached <= 8) launch_imp_pass<8, false>(P, A, smem);
    else launch_imp_pass<0, false>(P, A, smem);
  }
  if (!scatter) return;
  if (I.binarized)
    for (int w0 = 0; w0 < I.low_words; w0 += 32)
      KL_LAUNCH(low_accumulate, (unsigned)(ctx().sm_count * 2), 256, 0, I.lowbits.p, I.low_words, w0, M.n, wk.q.p, I.lowcol.p,
                wk.G.p, st);
  if (!scatter) return;
  if (!levels) return;
  // the fold: the super level and the levels above IMP_FOLD_TAIL one launch each, the small levels in the last
  // block of the last of those launches (or of a one-block launch when there is none)
  const int small_top = I.N - 1 < IMP_FOLD_TAIL ? I.N - 1 : IMP_FOLD_TAIL;
  int steps[IMP_MAX_N + 1], nsteps = 0;
  if (P.c > 1) steps[nsteps++] = I.N;
  for (int j = I.N - 1; j > small_top && j >= I.Mlo; j--) steps[nsteps++] = j;
  if (nsteps == 0 && small_top >= I.Mlo) steps[nsteps++] = -1;
  for (int s = 0; s < nsteps; s++) {
    const int j = steps[s];
    const int64_t items = j == I.N ? tsup : (j < 0 ? 1 : (int64_t)1 << (2 * j));
    KL_LAUNCH(imp_fold, (unsigned)((items + IMP_FOLD_THREADS - 1) / IMP_FOLD_THREADS), IMP_FOLD_THREADS, 0, P, j,
              s == nsteps - 1 ? small_top : -1, wk.H.p, wk.tickets.p, st);
  }
  // the columns are read off the folded tables by the pass tail (pass_tail)
  wk.P = P;
  wk.F = wk.H.p;
}

// the fused pass: loss terms + fixed-point gradient of the single-feature coefficients of THIS rank's rows
// (the caller reduces over the ranks); scatter = 0: loss terms only (G is left untouched)
template <typename VT>
void launch_fused(Matrix &M, Work &wk, const double cw[2], const PgState *st, int scatter = 1) {
  // G: [0, m] gradient | [m+1, m+1+world) loss slots of the ranks | [m+1+PEER_MAX_WORLD] row ticket (fused_kernel)
  if (scatter) KL_CUDA(cudaMemsetAsync(wk.G.p, 0, (size_t)(M.m + 2 + PEER_MAX_WORLD) * sizeof(unsigned long long), ctx().stream));
  if (M.n > 0) {
    if (use_implicit(M)) {
      launch_implicit(M, wk, cw, st, scatter);
    } else {
      int hot = ctx().hot_cols;
      if (hot > M.m) hot = (int)M.m;
      const size_t smem = (size_t)hot * 8;
      KL_CUDA(cudaFuncSetAttribute(fused_kernel<VT>, cudaFuncAttributeMaxDynamicSharedMemorySize, HOT_COLS_MAX * 8));
      const int tk = ctx().fused_ticket;
      if (tk > 0) {
        // persistent blocks, `tk` rows per warp and ticket (the counter sits behind the loss slots of G)
        unsigned long long *ticket = wk.G.p + M.m + 1 + PEER_MAX_WORLD;
        KL_CUDA(cudaMemsetAsync(ticket, 0, sizeof(unsigned long long), ctx().stream));
        int per_sm = 0;
        KL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fused_kernel<VT>, 256, smem));
        if (per_sm < 1) per_sm = 1;
        int64_t blocks = (int64_t)ctx().sm_count * per_sm, need = (M.n + 8 * tk - 1) / (8 * tk);
        if (blocks > need) blocks = need;
        KL_LAUNCH((fused_kernel<VT>), (unsigned)blocks, 256, smem, M.rows(), M.col.p, csr_val<VT>(M), M.n, M.m, wk.theta.p,
                  M.labels.p, cw[0], cw[1], 1.0 / (double)M.n_global, wk.scale, wk.scale0, wk.G.p, wk.lossterm.p, st, scatter, hot, tk,
                  ticket);
      } else {
        int rpb = FUSED_RPB;
        while ((M.n + rpb - 1) / rpb > 0x7fffffffLL) rpb *= 2;
        KL_LAUNCH((fused_kernel<VT>), (unsigned)((M.n + rpb - 1) / rpb), 256, smem, M.rows(), M.col.p, csr_val<VT>(M), M.n,
                  M.m, wk.theta.p, M.labels.p, cw[0], cw[1], 1.0 / (double)M.n_global, wk.scale, wk.scale0, wk.G.p, wk.lossterm.p, st,
                  scatter, hot, rpb, (unsigned long long *)nullptr);
      }
    }
  }
}

void alloc_work(const Matrix &M, int64_t ntheta, Work &wk) {
  wk.theta.alloc((size_t)ntheta);
  wk.w.alloc((size_t)(M.n ? M.n : 1));
  wk.lossterm.alloc((size_t)(M.n ? M.n : 1));
  wk.g.alloc((size_t)ntheta);
  wk.G.alloc((size_t)M.m + 2 + PEER_MAX_WORLD);      // + loss slots of the ranks
  wk.red.alloc(RED_BLOCKS);
  wk.scalars.alloc(8);
  wk.blockmax.alloc(4 * PROX_BLOCKS);    // max |theta|, max |delta|, NaN flag per block + the L1 partials of the hook
  wk.gathered.alloc((size_t)(M.sharded ? ntheta * ctx().world : 1));
  wk.tickets.alloc(3);
  wk.tickets.zero();
}

// the tail of a pass (pass_tail): the pending matrix-free columns, the sum of the first n loss terms into
// wk.scalars[0], the L1 partials of theta[1, ntheta) and, with a state and hook = 1, the hook
void launch_pass_tail(const Matrix &M, Work &wk, PgState *st, int64_t n, int64_t ntheta, double lambda, int hook,
                      double eps_loss) {
  static_assert(RED_BLOCKS == PROX_BLOCKS, "the L1 partials of pass_tail are the hook's PROX_BLOCKS partials");
  KL_LAUNCH(pass_tail, RED_BLOCKS, 256, 0, st, wk.P, M.class_ids.p, M.m, wk.F, wk.G.p, wk.lossterm.p, n,
            wk.red.p, wk.scalars.p, wk.theta.p, ntheta, lambda, wk.blockmax.p + 3 * PROX_BLOCKS, hook,
            1.0 / (double)M.n_global, eps_loss, wk.tickets.p + 1);
  wk.F = nullptr;
}

void check_theta(const Matrix &M, int64_t ntheta, int cooc) {
  if (cooc) KL_INVARIANT(ntheta == kmerlr_coeff_dim(M.m));
  else KL_INVARIANT(ntheta == M.m + 1);
}

template <typename F>
void dispatch_vt(const Matrix &M, F &&f) {
  if (M.vt == VAL_F64) f((double *)nullptr);
  else f((uint32_t *)nullptr);
}

}  // namespace

// ---------------------------------------------------------------------------------------------------
void linear_pdf(Matrix &M, const double *theta, int64_t ntheta, int cooc, double *out_host, bool logpdf) {
  require_ready();
  check_theta(M, ntheta, cooc);
  DevBuf<double> dth((size_t)ntheta), out((size_t)(M.n ? M.n : 1));
  dth.upload(theta, (size_t)ntheta);
  PairTerms terms;
  collect_pair_terms(M, theta, ntheta, cooc, terms);
  dispatch_vt(M, [&](auto *tag) {
    using VT = typename std::remove_pointer<decltype(tag)>::type;
    if (logpdf) launch_rows<VT, 1>(M, dth.p, cooc, nullptr, out.p, nullptr, nullptr, &terms);
    else launch_rows<VT, 0>(M, dth.p, cooc, nullptr, out.p, nullptr, nullptr, &terms);
  });
  out.download(out_host, (size_t)M.n);
  sync_stream();
}

void gradient(Matrix &M, const double *theta, int64_t ntheta, const double cw[2], double lambda, int cooc,
              double *g_host, DevBuf<double> *g_dev) {
  require_ready();
  check_theta(M, ntheta, cooc);
  KL_REQUIRE(M.has_labels, "gradient: the matrix has no labels (kmerlr_matrix_set_labels)");
  Work wk; alloc_work(M, ntheta, wk);
  set_scale(M, wk, cw);
  wk.theta.upload(theta, (size_t)ntheta);
  wk.g.zero();
  dispatch_vt(M, [&](auto *tag) {
    using VT = typename std::remove_pointer<decltype(tag)>::type;
    if (!cooc) {
      launch_fused<VT>(M, wk, cw, nullptr);
      if (wk.F) launch_pass_tail(M, wk, nullptr, 0, 0, NAN, 0, 0.0);
      if (M.sharded) comm_allreduce_sum_i64_fast((int64_t *)wk.G.p, M.m + 1);
    } else {
      // pair mode: z needs the pair terms, so the weights come from the general rows kernel; the
      // single-feature part still goes through the fixed-point pass with theta restricted to it
      // being irrelevant: w is what matters.  Reuse the fused kernel's scatter by running the pair
      // aware rows kernel for w and the CSC kernels for the pairs.
      PairTerms terms;
      collect_pair_terms(M, theta, ntheta, cooc, terms);
      launch_rows<VT, 2>(M, wk.theta.p, cooc, cw, wk.w.p, wk.lossterm.p, nullptr, &terms);
      ensure_csc(M);
      KL_CUDA(cudaMemsetAsync(wk.G.p, 0, (size_t)(M.m + 1) * sizeof(unsigned long long), ctx().stream));
      if (M.n > 0)
        KL_LAUNCH((scatter_w<VT>), warp_grid(M.n, 256), 256, 0, M.rows(), M.col.p, csr_val<VT>(M), M.n, wk.w.p,
                  wk.scale, wk.scale0, wk.G.p);
      if (M.sharded) comm_allreduce_sum_i64((int64_t *)wk.G.p, M.m + 1);
      if (M.m > 1) {
        const int ntile = (int)((M.m + PAIR_T - 1) / PAIR_T);
        const size_t smem = (size_t)PAIR_CH * PAIR_T * sizeof(double) + (size_t)8 * PAIR_CH * (sizeof(double) + sizeof(unsigned short));
        KL_CUDA(cudaFuncSetAttribute(pairs_gradient<VT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        KL_LAUNCH((pairs_gradient<VT>), (unsigned)((int64_t)ntile * (ntile + 1) / 2), 256, smem, M.colptr.p, M.crow.p,
                  csc_val<VT>(M), M.m, M.n, ntile, wk.w.p, wk.g.p);
        if (M.sharded) {
          // pair entries: every rank sums the per-rank values in rank order
          comm_allgather_f64(wk.g.p, wk.gathered.p, ntheta);
          KL_LAUNCH(sum_ranks, (unsigned)((ntheta + 255) / 256), 256, 0, wk.gathered.p, ctx().world, ntheta, wk.g.p);
        }
      }
    }
  });
  KL_LAUNCH(finalize_g, (unsigned)((M.m + 1 + 255) / 256), 256, 0, wk.G.p, M.m + 1, wk.inv_scale, wk.inv_scale0, wk.g.p);
  if (!std::isnan(lambda) && lambda != 0.0)
    KL_LAUNCH(add_l1_sign, (unsigned)((ntheta + 255) / 256), 256, 0, wk.theta.p, wk.g.p, ntheta, lambda);
  if (g_host) wk.g.download(g_host, (size_t)ntheta);
  sync_stream();
  if (M.sharded) comm_check_peer_errors();
  if (g_dev) *g_dev = std::move(wk.g);
}

double loss(Matrix &M, const double *theta, int64_t ntheta, const double cw[2], double lambda, int cooc) {
  require_ready();
  check_theta(M, ntheta, cooc);
  KL_REQUIRE(M.has_labels, "loss: the matrix has no labels (kmerlr_matrix_set_labels)");
  if (M.n_global == 0) return 0.0;
  Work wk; alloc_work(M, ntheta, wk);
  wk.theta.upload(theta, (size_t)ntheta);
  PairTerms terms;
  collect_pair_terms(M, theta, ntheta, cooc, terms);
  dispatch_vt(M, [&](auto *tag) {
    using VT = typename std::remove_pointer<decltype(tag)>::type;
    launch_rows<VT, 2>(M, wk.theta.p, cooc, cw, wk.w.p, wk.lossterm.p, nullptr, &terms);
  });
  launch_pass_tail(M, wk, nullptr, M.n, 0, NAN, 0, 0.0);
  if (M.sharded) {
    // the sums of the ranks in rank order (the same bits on every rank)
    comm_allgather_f64(wk.scalars.p, wk.gathered.p, 1);
    KL_LAUNCH(sum_ranks, 1, 32, 0, wk.gathered.p, ctx().world, (int64_t)1, wk.scalars.p);
  }
  double s = 0.0;
  wk.scalars.download(&s, 1);
  sync_stream();
  double r = s / (double)M.n_global;
  // the L1 loop bound of the reference is data[0].Dim() = m+1, also in pair mode (:255,267)
  if (!std::isnan(lambda) && lambda != 0.0)
    for (int64_t j = 1; j < M.m + 1; j++) r += lambda * std::fabs(theta[j]);
  return r;
}

void proxgrad(Matrix &M, double *theta, int64_t ntheta, const double cw[2], double lambda, double l2,
              double step_factor, double epsilon, double epsilon_loss, int64_t max_iter, double hook[2],
              int64_t *iters, double *delta) {
  require_ready();
  check_theta(M, ntheta, 0);
  KL_REQUIRE(M.has_labels, "proxgrad: the matrix has no labels (kmerlr_matrix_set_labels)");
  KL_REQUIRE(M.n_global > 0, "proxgrad: empty data set");
  Trace tr("proxgrad");
  // estimate_step_size (kmerLr_estimator_proximal.go:54-76)
  double L = 0.25 * (matrix_maxsq(M) + 1.0) + l2 / (double)M.n_global;
  double step = 1.0 / (2.0 * L + std::fmin(2.0 * l2, L)) * step_factor;
  Work wk; alloc_work(M, ntheta, wk);
  set_scale(M, wk, cw);
  // theta and the iteration state travel through the pinned staging buffer (theta first, the state behind it)
  double *hth = (double *)host_staging((size_t)ntheta * sizeof(double) + sizeof(PgState));
  PgState *hst = reinterpret_cast<PgState *>(hth + ntheta);
  memcpy(hth, theta, (size_t)ntheta * sizeof(double));
  wk.theta.upload(hth, (size_t)ntheta);
  DevBuf<PgState> st(1);
  PgState h{};
  h.iter = 0; h.done = max_iter > 0 ? 0 : 1; h.first = 1; h.delta = 0.0;
  h.loss_old = hook ? hook[0] : NAN; h.loss_new = hook ? hook[1] : NAN; h.lossval = NAN; h.error = 0;
  *hst = h;
  st.upload(hst, 1);
  const double inv_n = 1.0 / (double)M.n_global;
  // reduced matrices: long batches between host round trips.  The choice of the path uses quantities that are
  // the same on every rank (a rank with an empty shard must issue the same collectives as the others)
  const bool small = ntheta <= SMALL_MAX_THETA && !use_implicit(M);
  // the kernels of reduced matrices accumulate the columns and the bias with their own scales (set_scale), as the
  // full-space pass does: the same integers G as fused_kernel
  // the passes of a batch are ONE cooperative launch (grid barriers instead of launches); sharded matrices
  // exchange the gradient inside that kernel over NVLink peer memory
  const bool p2p = M.sharded && ctx().peer && ctx().p2p_ok;
  bool persistent = small && ctx().coop_ok && (!M.sharded || p2p);
  // long rows: sliced + column-major views (the iterates are the same bits on either path, so a rank may choose by
  // its own shard)
  // (by row length: the block-local view from 4 entries per row, the two global views from 8)
  bool long_rows = persistent && M.nnz > 0 && (ctx().small_long >= 1 || (ctx().small_long < 0 && M.nnz >= 4 * M.n));
  DevBuf<double> wbuf;
  bool packed = false;
  if (long_rows) { ensure_sliced(M); ensure_csc(M); packed = ensure_packed(M); wbuf.alloc((size_t)M.n); }
  // long_mode 2: the block-local view (one grid barrier per iteration); it is built for the grid of this launch
  int long_mode = long_rows ? 1 : 0;
  size_t dyn_smem = 0;
  // (measured at C2 rows, 100 columns, 5 / 14 / 24 / 50 / 98 / 249 entries per row: 19.0 / 23.5 / 28.2 / 40.6 / 62.4 / 137 us
  // against 23.2 / 27.4 / 32.5 / 42.5 / 67.0 / 141 us on the sliced + column-major views: chosen whenever it fits)
  const bool want_block = long_rows && packed && (ctx().small_long == 2 || ctx().small_long < 0);
  const int64_t BATCH = persistent ? 4096 : (small ? 256 : 16);
  int small_blocks = 0;
  DevBuf<double> blockloss;
  DevBuf<unsigned int> counter;
  DevBuf<unsigned long long> G3;      // persistent path: triple-buffered gradient accumulators
  if (small) {
    // one wave: as many blocks as are resident at once (a second, partly filled wave costs a whole round)
    int64_t nb = (int64_t)ctx().sm_count * SMALL_BLOCKS_PER_SM, need = (M.n + 63) / 64;   // >= 64 rows per block
    if (persistent) {
      auto resident = [&](int mode, size_t smem) {
        int per_sm = 0;
        dispatch_vt(M, [&](auto *tag) {
          using VT = typename std::remove_pointer<decltype(tag)>::type;
          if (smem > 16 * 1024)
            KL_CUDA(cudaFuncSetAttribute(persistent_kernel<VT>(M.sharded, mode), cudaFuncAttributeMaxDynamicSharedMemorySize, 32 * 1024));
          KL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, persistent_kernel<VT>(M.sharded, mode), PERSIST_THREADS, smem));
        });
        if (ctx().persist_bps > 0 && ctx().persist_bps < per_sm) per_sm = ctx().persist_bps;
        return per_sm;
      };
      if (want_block) {
        // the grid fixes the rows per block, the rows per block fix the shared memory, the shared memory the grid
        int per_sm = resident(2, 0);
        for (int round = 0; round < 4 && per_sm >= 1; round++) {
          int64_t g = (int64_t)ctx().sm_count * per_sm;
          if (g > need) g = need;
          const size_t smem = (size_t)((M.n + g - 1) / g + 1) * sizeof(double);
          const int p2 = smem <= 32 * 1024 ? resident(2, smem) : 0;
          if (p2 >= per_sm) { dyn_smem = smem; break; }
          per_sm = p2;
        }
        if (per_sm >= 1 && dyn_smem > 0) {
          int64_t g = (int64_t)ctx().sm_count * per_sm;
          if (g > need) g = need;
          if (ensure_blockview(M, (int)g)) { long_mode = 2; nb = (int64_t)ctx().sm_count * per_sm; }
          else dyn_smem = 0;
        } else dyn_smem = 0;
      }
      if (long_mode != 2 && long_rows && ctx().small_long < 0 && M.nnz < 8 * M.n) { long_rows = false; long_mode = 0; }
      if (long_mode != 2) {
        const int per_sm = resident(long_mode, 0);
        KL_INVARIANT(per_sm >= 1);
        nb = (int64_t)ctx().sm_count * per_sm;       // a cooperative grid must be resident as a whole
      }
    }
    small_blocks = (int)(nb < need ? nb : need);
    if (small_blocks < 1) small_blocks = 1;        // (an empty shard still takes part in the exchange)
    blockloss.alloc((size_t)small_blocks * (persistent ? 2 : 1));
    if (persistent) { G3.alloc((size_t)(3 * SMALL_REPLICAS * ntheta)); G3.zero(); }
    counter.alloc(1);
    counter.zero();
    KL_CUDA(cudaMemsetAsync(wk.G.p, 0, (size_t)ntheta * sizeof(unsigned long long), ctx().stream));
  }
  int64_t issued = 0;
  while (true) {
    // max_iter prox steps need max_iter + 1 row passes (the last one only evaluates the hook)
    int64_t nb = max_iter + 1 - issued;
    if (nb > BATCH) nb = BATCH;
    if (nb < 1) nb = 1;
    issued += nb;
    if (persistent) {
      dispatch_vt(M, [&](auto *tag) {
        using VT = typename std::remove_pointer<decltype(tag)>::type;
        Rows rows = M.rows();
        const uint32_t *colp = M.col.p;
        const VT *valp = csr_val<VT>(M);
        int64_t n = M.n, nt = ntheta;
        double *thp = wk.theta.p;
        const uint8_t *lab = M.labels.p;
        double cw0 = cw[0], cw1 = cw[1], invn = inv_n, scale = wk.scale, inv_scale = wk.inv_scale;
        double scale0 = wk.scale0, inv_scale0 = wk.inv_scale0;
        unsigned long long *Gp = G3.p;
        double *bl = blockloss.p;
        PgState *stp = st.p;
        long long pass0 = (long long)(issued - nb), mi = (long long)max_iter;
        int npass = (int)nb;
        double lam = lambda, el = epsilon_loss, stp_size = step, eps = epsilon;
        const PeerBox *pbp = ctx().peer;
        unsigned long long *gx = wk.G.p;
        double *scr = wk.gathered.p;
        unsigned int *abortp = counter.p;
        LongView<VT> lv{};
        if (long_rows) {
          lv.slice_off = M.slice_off.p; lv.scol = M.scol.p; lv.sval = sliced_val<VT>(M);
          lv.colptr = M.colptr.p; lv.crow = M.crow.p; lv.cval = csc_val<VT>(M);
          if (packed) { lv.spack = M.spack.p; lv.cpack = M.cpack.p; lv.row_bits = M.pack_row_bits; }
          lv.wbuf = wbuf.p; lv.nnz = M.nnz;
          if (long_mode == 2) { lv.bv_off = M.bv_off.p; lv.bv_pack = M.bv_pack.p; lv.bv_row_bits = M.bv_row_bits; }
        }
        void *args[] = {&rows, &colp, &valp, &n, &nt, &thp, &lab, &cw0, &cw1, &invn, &scale, &scale0, &Gp, &bl, &stp, &pass0,
                        &npass, &inv_scale, &inv_scale0, &lam, &el, &stp_size, &eps, &mi, &pbp, &gx, &scr, &abortp, &lv};
        if (ctx().profiling) profile_begin("fused_small_persistent");
        const cudaError_t e = cudaLaunchCooperativeKernel(
            persistent_kernel<VT>(M.sharded, long_mode),
            dim3((unsigned)small_blocks), dim3(PERSIST_THREADS), args, dyn_smem, ctx().stream);
        if (ctx().profiling) profile_end();
        if (e == cudaErrorCooperativeLaunchTooLarge && !M.sharded) {
          // the GPU is shared (MPS, another context): the grid cannot be resident as a whole right now.
          // Nothing was launched; this call goes on with one launch per iteration.  (Not on a sharded matrix:
          // the other ranks are inside their exchange by now, a rank that changes path would leave them waiting.)
          (void)cudaGetLastError();
          persistent = false;
        } else {
          KL_CUDA(e);
          ctx().launches++;
        }
      });
    }
    for (int64_t it = 0; it < nb && !persistent; it++) {
      // pass number max_iter (0-based) only evaluates the hook's loss at the final theta: no gradient
      const int scatter = (issued - nb + it) < max_iter ? 1 : 0;
      if (small) {
        dispatch_vt(M, [&](auto *tag) {
          using VT = typename std::remove_pointer<decltype(tag)>::type;
          KL_LAUNCH((fused_small_kernel<VT>), (unsigned)small_blocks, 256, 0, M.rows(), M.col.p, csr_val<VT>(M), M.n, ntheta,
                    wk.theta.p, M.labels.p, cw[0], cw[1], inv_n, wk.scale, wk.scale0, wk.G.p, blockloss.p, st.p, scatter,
                    M.sharded ? (unsigned int *)nullptr : counter.p, wk.inv_scale, wk.inv_scale0, lambda, epsilon_loss, step,
                    epsilon, (long long)max_iter);
        });
        if (M.sharded && ctx().peer && ctx().p2p_ok) {
          // exchange over peer memory fused with the tail of the iteration
          KL_LAUNCH(small_p2p_tail_kernel, (unsigned)(ctx().world + 1), 256, 0, st.p, ctx().peer, blockloss.p, small_blocks, wk.theta.p, wk.G.p,
                    wk.gathered.p, wk.inv_scale, wk.inv_scale0, ntheta, inv_n, lambda, epsilon_loss, step, epsilon,
                    (long long)max_iter);
        } else if (M.sharded) {
          // gradient: exact int64 all-reduce; loss: per-rank sums gathered and added in rank order
          unsigned long long *slots = wk.G.p + ntheta;
          KL_LAUNCH(small_presum_kernel, 1, 256, 0, st.p, blockloss.p, small_blocks, wk.scalars.p);
          KL_LAUNCH(pack_loss_slots, 1, 32, 0, st.p, wk.scalars.p, slots, ctx().rank, ctx().world);
          if (scatter) comm_allreduce_sum_i64((int64_t *)wk.G.p, ntheta + ctx().world);
          else comm_allreduce_sum_i64((int64_t *)slots, ctx().world);
          KL_LAUNCH(small_tail_kernel, 1, 256, 0, st.p, reinterpret_cast<const double *>(slots), ctx().world, wk.theta.p,
                    wk.G.p, wk.inv_scale, wk.inv_scale0, ntheta, inv_n, lambda, epsilon_loss, step, epsilon, (long long)max_iter);
        }
        continue;
      }
      dispatch_vt(M, [&](auto *tag) {
        using VT = typename std::remove_pointer<decltype(tag)>::type;
        launch_fused<VT>(M, wk, cw, st.p, scatter);
        // columns, loss and L1 partials; one GPU: the loss sum and the hook in the same launch
        launch_pass_tail(M, wk, st.p, M.n, M.m + 1, lambda, M.sharded ? 0 : 1, epsilon_loss);
        if (M.sharded) {
          // ONE collective per iteration: gradient words + the loss sums of the ranks
          unsigned long long *slots = wk.G.p + M.m + 1;
          KL_LAUNCH(pack_loss_slots, 1, 32, 0, st.p, wk.scalars.p, slots, ctx().rank, ctx().world);
          if (scatter) comm_allreduce_sum_i64_fast((int64_t *)wk.G.p, M.m + 1 + ctx().world);
          else comm_allreduce_sum_i64_fast((int64_t *)slots, ctx().world);
          KL_LAUNCH(unpack_loss_hook, 1, 32, 0, st.p, slots, ctx().world, wk.scalars.p, wk.blockmax.p + 3 * PROX_BLOCKS,
                    PROX_BLOCKS, inv_n, epsilon_loss);
        }
        // the loss-only pass (number max_iter) follows the last prox step: the state is stopped (done != 0) by then
        if (scatter)
          KL_LAUNCH(prox_update, PROX_BLOCKS, 256, 0, st.p, wk.theta.p, wk.G.p, wk.inv_scale, wk.inv_scale0, ntheta, step, lambda,
                    wk.blockmax.p, epsilon, (long long)max_iter, wk.tickets.p + 2);
      });
    }
    // theta comes down with the state: a batch is usually the last one, and then no second round trip is needed
    st.download(hst, 1);
    wk.theta.download(hth, (size_t)ntheta);
    host_staging_done();
    sync_stream();
    h = *hst;
    if (h.error) fail(KMERLR_ERR_CUDA, "proxgrad: a rank did not answer the gradient exchange over peer memory");
    if (M.sharded) comm_check_peer_errors();
    if (h.done == 1) break;
  }
  memcpy(theta, hth, (size_t)ntheta * sizeof(double));
  tr.mark("iterations");
  if (hook) { hook[0] = h.loss_old; hook[1] = h.loss_new; }
  if (iters) *iters = (int64_t)h.iter;
  if (delta) *delta = h.delta;
}

}  // namespace kl
