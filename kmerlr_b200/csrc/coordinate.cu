// coordinate.cu -- the IRLS + coordinate-descent estimator of the reference
// (kmerLr_estimator_coordinate.go:31-139; SURVEY 8a row 8), for reduced matrices (<= 1023 columns).
// PARITY UNPINNED IN THE REFERENCE ITSELF: the function has no caller, no test and no golden there; the numpy
// restatement the tests compare this kernel with is pinned by optimality properties only.
//
//   outer iteration: r_i = x_i theta, p_i = sigma(r_i), w_i = p_i (1 - p_i), z_i = r_i + (y_i - p_i) / w_i,
//                    w_i *= class weight of y_i                                          (:97-111)
//   inner loop:      xy_j = sum_i w_i z_i x_ij,  xx_jk = sum_i w_i x_ij x_ik  (norm_j = xx_jj)   (:32-52)
//                    cyclic sweeps  t = xy_j + norm_j theta_j - sum_k xx_jk theta_k,
//                    soft threshold by L1Reg (j > 0), t / (norm_j + L2Reg)               (:55-72)
//   eval_stopping after every sweep and after every outer iteration, then the hook (:74-82, :117-125).
//
// The reference never calls this function and, as written, all of its theta slices alias one array
// (:89-91) so that it would stop after the first sweep; like estimate_proximal it is built here with
// the slices de-aliased (theta0 = start of the outer iteration, theta0_ = before the sweep).
//
// Device work: the row pass (one thread per row, the Gram matrix and xy as exact 64-bit fixed-point
// sums: deterministic, any order) and the sweeps (one block: the dot product of a Gram row with theta
// is a fixed tree over 1024 threads).  The host only sequences the launches and reads the stopping state.
#include <cmath>

#include "common.cuh"

namespace kl {

namespace {

constexpr int CD_MAX_THETA = 1024;
constexpr int CD_THREADS = 1024;

// the powers of two of the fixed-point sums, one per class of entry: xy of the bias and of a column; xx of
// (bias, bias), (bias, column) and (column, column).  The bias is 1 in every row, a column at most max|v|: a matrix
// whose values are all below 1 keeps the bits between max|v| and 1 in its column entries.
struct CdScales {
  double xy0, xy, xx00, xx0c, xxcc;
};

// row pass: Gram and xy of the weighted least-squares problem of this outer iteration
template <typename VT>
__global__ void __launch_bounds__(256) cd_rows_kernel(const Rows R, const uint32_t *__restrict__ col,
                                                      const VT *__restrict__ val, int64_t n, int64_t ntheta,
                                                      const double *__restrict__ theta,
                                                      const uint8_t *__restrict__ labels, double cw0, double cw1,
                                                      CdScales S, long long *__restrict__ XY, long long *__restrict__ XX,
                                                      int *__restrict__ bad) {
  __shared__ double sth[CD_MAX_THETA];
  for (int i = threadIdx.x; i < ntheta; i += blockDim.x) sth[i] = theta[i];
  __syncthreads();
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= n) return;
  int64_t a, b;
  R.range(row, a, b);
  double s = 0.0;
  for (int64_t p = a; p < b; p++) s += valf(val, p) * sth[col[p] + 1];
  const double r = sth[0] + s;                                   // LinearPdf (:98)
  const double pr = exp(-log_add0(-r));                          // (:99)
  double w = pr * (1.0 - pr);                                    // (:100)
  const bool y = labels[row] != 0;
  const double z = y ? r + (1.0 - pr) / w : r + (0.0 - pr) / w;  // (:101-105)
  w *= y ? cw1 : cw0;                                            // (:106-110)
  const double wz = w * z;
  if (!isfinite(wz) || !isfinite(w)) { atomicExch(bad, 1); return; }   // the reference's sums turn NaN here
  // entry -1 = the bias column (index 0, value 1)
  for (int64_t p1 = a - 1; p1 < b; p1++) {
    const int64_t j1 = p1 < a ? 0 : (int64_t)col[p1] + 1;
    const double v1 = p1 < a ? 1.0 : valf(val, p1);
    atomicAdd((unsigned long long *)&XY[j1], (unsigned long long)__double2ll_rn(wz * v1 * (j1 == 0 ? S.xy0 : S.xy)));
    const double wv1 = w * v1;
    const double sb = j1 == 0 ? S.xx00 : S.xx0c, sc = j1 == 0 ? S.xx0c : S.xxcc;     // the scales of (j1, bias), (j1, column)
    for (int64_t p2 = a - 1; p2 < b; p2++) {
      const int64_t j2 = p2 < a ? 0 : (int64_t)col[p2] + 1;
      const double v2 = p2 < a ? 1.0 : valf(val, p2);
      atomicAdd((unsigned long long *)&XX[j1 * ntheta + j2],
                (unsigned long long)__double2ll_rn(wv1 * v2 * (j2 == 0 ? sb : sc)));
    }
  }
}

__global__ void cd_convert_kernel(const long long *__restrict__ XY, const long long *__restrict__ XX, int64_t ntheta,
                                  CdScales inv, double *__restrict__ xy, double *__restrict__ xx) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < ntheta) xy[i] = (double)XY[i] * (i == 0 ? inv.xy0 : inv.xy);
  if (i < ntheta * ntheta) {
    const bool b1 = i < ntheta, b2 = i % ntheta == 0;
    xx[i] = (double)XX[i] * (b1 && b2 ? inv.xx00 : (b1 || b2 ? inv.xx0c : inv.xxcc));
  }
}

struct CdState {
  double delta;     // eval_stopping's delta of the last sweep
  int stop;         // eval_stopping said stop
};

// one cyclic sweep over the coordinates (:57-72) + eval_stopping(theta0_, theta1) (:74), one block
__global__ void __launch_bounds__(CD_THREADS) cd_sweep_kernel(const double *__restrict__ xy, const double *__restrict__ xx,
                                                               int64_t ntheta, double l1, double l2, double eps,
                                                               double *theta, CdState *st) {
  __shared__ double sth[CD_MAX_THETA];
  __shared__ double red[CD_THREADS / 32];
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
  for (int i = t; i < ntheta; i += CD_THREADS) sth[i] = theta[i];
  __syncthreads();
  double max_x = 0.0, max_d = 0.0;
  bool isnan_seen = false;
  for (int64_t j = 0; j < ntheta; j++) {
    // sum_k xx[j][k] theta1[k]: one product per thread, fixed tree
    double v = t < ntheta ? xx[j * ntheta + t] * sth[t] : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if (lane == 0) red[wid] = v;
    __syncthreads();
    if (t == 0) {
      double dot = red[0];
      for (int w = 1; w < CD_THREADS / 32; w++) dot += red[w];
      const double norm = xx[j * ntheta + j];
      double tj = xy[j] + norm * sth[j];
      tj -= dot;
      if (j > 0) tj = soft_threshold(tj, l1);
      tj /= (norm + l2);
      const double old = sth[j];
      sth[j] = tj;
      if (isnan(tj)) isnan_seen = true;
      max_x = fmax(max_x, fabs(tj));
      max_d = fmax(max_d, fabs(tj - old));
    }
    __syncthreads();
  }
  for (int i = t; i < ntheta; i += CD_THREADS) theta[i] = sth[i];
  if (t == 0) st->stop = eval_stopping(max_x, max_d, isnan_seen, eps, &st->delta) ? 1 : 0;
}

}  // namespace

void coordinate(Matrix &M, double *theta, int64_t ntheta, const double cw_hook[2], double l1reg, double l2reg,
                double epsilon, double epsilon_loss, int64_t max_iter, double hook[2], int64_t *sweeps_out,
                double *delta_out) {
  require_ready();
  KL_REQUIRE(ntheta == M.m + 1, "coordinate: theta must have one entry per column plus the bias");
  KL_REQUIRE(ntheta <= CD_MAX_THETA, "coordinate: the coordinate-descent estimator keeps a dense Gram matrix; use it on a "
                                     "reduced matrix (at most 1023 columns)");
  KL_REQUIRE(M.has_labels, "coordinate: the matrix has no labels (kmerlr_matrix_set_labels)");
  KL_REQUIRE(!M.sharded, "coordinate: single GPU only");
  KL_REQUIRE(M.n > 0, "coordinate: empty data set");
  // compute_class_weights(data_train.Labels) (:88; kmerLr_data.go:178-193)
  matrix_label_counts(M);
  KL_REQUIRE(M.n_pos > 0 && M.n_neg > 0, "coordinate: both classes must be present");
  const double ntot = (double)(M.n_pos + M.n_neg);
  const double cw[2] = {ntot / (2.0 * (double)M.n_neg), ntot / (2.0 * (double)M.n_pos)};
  const double cwmax = std::fmax(cw[0], cw[1]);
  const double vmax = matrix_vmax(M), v1 = std::fmax(vmax, 1.0), maxsq = matrix_maxsq(M);

  DevBuf<double> dtheta((size_t)ntheta), xy((size_t)ntheta), xx((size_t)(ntheta * ntheta));
  DevBuf<long long> XY((size_t)ntheta), XX((size_t)(ntheta * ntheta));
  DevBuf<int> bad(1);
  DevBuf<CdState> dst(1);
  std::vector<double> th1(theta, theta + ntheta), th0((size_t)ntheta);
  double hk_old = hook ? hook[0] : NAN, hk_new = hook ? hook[1] : NAN;
  // the hook (kmerLr_estimator_hook.go:46-99): loss at theta (the ESTIMATOR's class weights, lambda = L1Reg / n),
  // stop when it moved by less than epsilon_loss
  auto run_hook = [&](const std::vector<double> &th) -> bool {
    double t = hk_old; hk_old = hk_new; hk_new = t;
    if (epsilon_loss != 0.0) {
      hk_new = loss(M, th.data(), ntheta, cw_hook, l1reg / (double)M.n, 0);
      if (std::fabs(hk_old - hk_new) < epsilon_loss) return true;
    }
    return false;
  };
  int64_t sweeps = 0;
  double delta = 0.0;
  const unsigned row_grid = (unsigned)((M.n + 255) / 256);
  const unsigned cv_grid = (unsigned)((ntheta * ntheta + 255) / 256);
  bool nan_abort = false;
  for (int64_t iter = 0; iter < max_iter; iter++) {
    // scales of the fixed-point sums: |w x_j x_k| <= cw |x_j| |x_k| / 4, |w z x_j| <= cw |x_j| (|r| / 4 + 1), with
    // |x_0| = 1 for the bias and |x_j| <= vmax for a column; the bias bounds take max(vmax, 1) (v1), so every
    // exponent is the same whenever vmax >= 1
    double th2 = 0.0;
    for (int64_t k = 1; k < ntheta; k++) th2 += th1[k] * th1[k];
    const double rmax = std::fabs(th1[0]) + std::sqrt(th2 * maxsq);
    const double bxy0 = (double)M.n * cwmax * v1 * (0.25 * rmax + 1.0);
    if (!(bxy0 > 0.0) || !std::isfinite(bxy0)) { nan_abort = true; break; }
    const int exy0 = fixed_point_exponent(bxy0),
              exy = fixed_point_exponent((double)M.n * cwmax * vmax * (0.25 * rmax + 1.0));
    const int exx00 = fixed_point_exponent((double)M.n * 0.25 * cwmax * v1 * v1),
              exx0c = fixed_point_exponent((double)M.n * 0.25 * cwmax * v1 * vmax),
              exxcc = fixed_point_exponent((double)M.n * 0.25 * cwmax * vmax * vmax);
    const CdScales S{std::ldexp(1.0, exy0), std::ldexp(1.0, exy), std::ldexp(1.0, exx00), std::ldexp(1.0, exx0c),
                     std::ldexp(1.0, exxcc)};
    const CdScales inv{std::ldexp(1.0, -exy0), std::ldexp(1.0, -exy), std::ldexp(1.0, -exx00), std::ldexp(1.0, -exx0c),
                       std::ldexp(1.0, -exxcc)};
    dtheta.upload(th1.data(), (size_t)ntheta);
    XY.zero(); XX.zero(); bad.zero();
    if (M.vt == VAL_F64)
      KL_LAUNCH((cd_rows_kernel<double>), row_grid, 256, 0, M.rows(), M.col.p, M.val_f64.p, M.n, ntheta, dtheta.p, M.labels.p,
                cw[0], cw[1], S, XY.p, XX.p, bad.p);
    else
      KL_LAUNCH((cd_rows_kernel<uint32_t>), row_grid, 256, 0, M.rows(), M.col.p,
                M.vt == VAL_U32 ? M.val_u32.p : (const uint32_t *)nullptr, M.n, ntheta, dtheta.p, M.labels.p, cw[0], cw[1],
                S, XY.p, XX.p, bad.p);
    KL_LAUNCH(cd_convert_kernel, cv_grid, 256, 0, XY.p, XX.p, ntheta, inv, xy.p, xx.p);
    int hbad = 0;
    bad.download(&hbad, 1);
    sync_stream();
    if (hbad) { nan_abort = true; break; }
    th0 = th1;                                                   // (:112-115)
    // estimate_coordinate_loop (:55-83): sweeps until eval_stopping or the hook says stop
    for (; iter < max_iter; iter++) {
      KL_LAUNCH(cd_sweep_kernel, 1, CD_THREADS, 0, xy.p, xx.p, ntheta, l1reg, l2reg, epsilon, dtheta.p, dst.p);
      CdState hs{};
      dst.download(&hs, 1);
      dtheta.download(th1.data(), (size_t)ntheta);
      sync_stream();
      sweeps++;
      delta = hs.delta;
      if (hs.stop) break;
      if (run_hook(th1)) break;
    }
    // (:117-125) eval_stopping over the outer iteration
    double max_x = 0.0, max_d = 0.0;
    bool isnan_seen = false;
    for (int64_t k = 0; k < ntheta && !isnan_seen; k++) {
      isnan_seen = std::isnan(th1[k]);
      max_x = std::fmax(max_x, std::fabs(th1[k]));
      max_d = std::fmax(max_d, std::fabs(th1[k] - th0[k]));
    }
    if (eval_stopping(max_x, max_d, isnan_seen, epsilon, &delta)) break;
    if (run_hook(th1)) break;
  }
  if (nan_abort) {
    for (auto &v : th1) v = NAN;
    delta = NAN;
  }
  for (int64_t k = 0; k < ntheta; k++) theta[k] = th1[k];
  if (hook) { hook[0] = hk_old; hook[1] = hk_new; }
  if (sweeps_out) *sweeps_out = sweeps;
  if (delta_out) *delta_out = delta;
}

}  // namespace kl
