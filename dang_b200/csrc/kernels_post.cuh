// kernels_post.cuh -- running posterior mean and variance of the chain state (dang_gpu_posterior_*; not in the
// reference, whose users write every sample with write_maps and average offline).  Accumulators hold one 16-byte
// {mean, M2} pair per element, and with batch means a 16-byte {bmean, bM2} pair and an 8-byte bsum.  Every step is spelled with _rn intrinsics: the build contracts a*b+c to an FMA by
// default, and the update is defined as separately rounded operations so that a numpy restatement equals it bit
// for bit.  Elements are independent, so no result depends on the grid.
#pragma once
#include <math_constants.h>

#include "common.cuh"
#include "kernels_data.cuh"

// One sample x, n = the count after adding it:  d = x - mean;  mean += d / n;  M2 += d * (x - mean)
__device__ __forceinline__ double2 post_update(double2 a, double x, double n) {
  const double d = __dsub_rn(x, a.x);
  a.x = __dadd_rn(a.x, __ddiv_rn(d, n));
  a.y = __dadd_rn(a.y, __dmul_rn(d, __dsub_rn(x, a.x)));
  return a;
}

// ---------------------------------------------------------------- amplitudes, index maps, template amplitudes
// One entry per accumulated array: a (component, plane) map of Ppad elements, or a component's [3][DG_MAX_BANDS]
// template-amplitude table.  Lengths are even and every array is 16-byte aligned, so samples move as double2.
const int DG_POST_ENTRIES = 128;
struct PostEntry {
  const double *src;  // the sample, read where it lives (c.amp / c.idx[l] / c.tamp)
  double2 *acc;       // its accumulators
  int64_t n;          // elements (even)
};
struct PostTable {
  int count;
  PostEntry e[DG_POST_ENTRIES];
};

// grid = (x, count): blockIdx.y picks the array, x strides over its element pairs.  40 bytes per element.
static __global__ void __launch_bounds__(DG_THREADS) post_stream_kernel(const PostTable t, double n) {
  const PostEntry &e = t.e[blockIdx.y];
  const double2 *src = reinterpret_cast<const double2 *>(e.src);
  const int64_t npair = e.n / 2, stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < npair; i += stride) {
    const double2 x = __ldcs(src + i);
    const double2 a0 = __ldcs(e.acc + 2 * i), a1 = __ldcs(e.acc + 2 * i + 1);
    __stcs(e.acc + 2 * i, post_update(a0, x.x, n));
    __stcs(e.acc + 2 * i + 1, post_update(a1, x.y, n));
  }
}

// ---------------------------------------------------------------- batch means (dang_gpu_posterior_begin_batched)
// Next to {mean, M2}, a batched array holds per element the running sum of the open batch, bsum, and Welford
// moments of the completed batch means, {bmean, bM2}.  Sample n sits at position j = ((n-1) mod b) + 1 of its batch;
// the host knows j, so the phase is a launch parameter: OPEN (j == 1) sets bsum = x without reading it, CLOSE
// (j == b, k = n / b) folds y = bsum / b into {bmean, bM2} with post_update and does not store bsum.  b = 1 is both.
struct PostBatch {
  double b, k;  // batch length; completed batches after this sample (read only when closing)
  bool open, close;
};

// One batched element: {mean, M2} as post_update, then the batch sum and, when the batch closes, its mean
__device__ __forceinline__ void post_batch_update(double2 *acc, double *bsum, double2 *bacc, size_t i, double x,
                                                  double n, const PostBatch &p) {
  acc[i] = post_update(acc[i], x, n);
  const double s = p.open ? x : __dadd_rn(bsum[i], x);
  if (p.close) bacc[i] = post_update(bacc[i], __ddiv_rn(s, p.b), p.k);
  else bsum[i] = s;
}

// The table of post_stream_kernel with the two batch arrays of each entry.  128 entries of 40 B exceed the classic
// 4 KB of kernel parameters; sm_70 and later take up to 32 KB since CUDA 12.1, so the table stays a by-value argument.
struct PostBatchEntry {
  const double *src;
  double2 *acc;   // {mean, M2}
  double *bsum;   // the open batch's running sum
  double2 *bacc;  // {bmean, bM2} of the completed batch means
  int64_t n;      // elements (even)
};
struct PostBatchTable {
  int count;
  PostBatchEntry e[DG_POST_ENTRIES];
};

// grid = (x, count), as post_stream_kernel.  Bytes per element: OPEN 48 (bsum not read), middle 56, CLOSE 80 (bsum
// not written), OPEN and CLOSE (b = 1) 72.
template <bool OPEN, bool CLOSE>
static __global__ void __launch_bounds__(DG_THREADS)
post_stream_batch_kernel(const PostBatchTable t, double n, double b, double k) {
  const PostBatchEntry &e = t.e[blockIdx.y];
  const double2 *src = reinterpret_cast<const double2 *>(e.src);
  double2 *bsum = reinterpret_cast<double2 *>(e.bsum);
  const int64_t npair = e.n / 2, stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < npair; i += stride) {
    const double2 x = __ldcs(src + i);
    const double2 a0 = __ldcs(e.acc + 2 * i), a1 = __ldcs(e.acc + 2 * i + 1);
    __stcs(e.acc + 2 * i, post_update(a0, x.x, n));
    __stcs(e.acc + 2 * i + 1, post_update(a1, x.y, n));
    double2 s = x;
    if (!OPEN) {
      const double2 p = __ldcs(bsum + i);
      s = make_double2(__dadd_rn(p.x, x.x), __dadd_rn(p.y, x.y));
    }
    if (CLOSE) {
      const double2 b0 = __ldcs(e.bacc + 2 * i), b1 = __ldcs(e.bacc + 2 * i + 1);
      __stcs(e.bacc + 2 * i, post_update(b0, __ddiv_rn(s.x, b), k));
      __stcs(e.bacc + 2 * i + 1, post_update(b1, __ddiv_rn(s.y, b), k));
    } else {
      __stcs(bsum + i, s);
    }
  }
}

// ---------------------------------------------------------------- residual and chi-square maps
// The K6 sink of dang_gpu_posterior_accumulate (chisq_kernel<NC, ChisqPost>): t and chi(k) / nbands go into
// accumulators instead of res_map and chi_map, so the model arithmetic is the code dang_gpu_get_sky_model runs.
// No chi-square reduction.
struct ChisqPost {
  static constexpr bool kMaps = true, kReduce = false;
  double2 *acc_res;  // [nbands][nmaps][Ppad] or nullptr
  double2 *acc_chi;  // [nmaps][Ppad] or nullptr
  double n;
  __device__ __forceinline__ void sky(const ChisqView &, size_t, double) const {}
  __device__ __forceinline__ void res(const ChisqView &, size_t off, double v) const {
    if (acc_res) acc_res[off] = post_update(acc_res[off], v, n);
  }
  __device__ __forceinline__ void chi(const ChisqView &, size_t off, double v) const {
    if (acc_chi) acc_chi[off] = post_update(acc_chi[off], v, n);
  }
};

// ChisqPost with batch means (chisq_kernel<NC, ChisqPostBatch>).  The phase is uniform over the launch.
struct ChisqPostBatch {
  static constexpr bool kMaps = true, kReduce = false;
  double2 *acc_res, *bacc_res;  // [nbands][nmaps][Ppad] or nullptr
  double *bsum_res;
  double2 *acc_chi, *bacc_chi;  // [nmaps][Ppad] or nullptr
  double *bsum_chi;
  double n;
  PostBatch p;
  __device__ __forceinline__ void sky(const ChisqView &, size_t, double) const {}
  __device__ __forceinline__ void res(const ChisqView &, size_t off, double v) const {
    if (acc_res) post_batch_update(acc_res, bsum_res, bacc_res, off, v, n, p);
  }
  __device__ __forceinline__ void chi(const ChisqView &, size_t off, double v) const {
    if (acc_chi) post_batch_update(acc_chi, bsum_chi, bacc_chi, off, v, n, p);
  }
};

// ---------------------------------------------------------------- read-out
// mean and standard deviation sqrt(M2 / (n - 1)) of `len` elements; NaN for n < 2
static __global__ void post_finalize_kernel(const double2 *acc, int64_t len, int64_t n, double *mean, double *stddev) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const double nm1 = (double)(n - 1);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += stride) {
    const double2 a = acc[i];
    mean[i] = a.x;
    if (stddev) stddev[i] = n < 2 ? CUDART_NAN : __dsqrt_rn(__ddiv_rn(a.y, nm1));
  }
}

// Classic Gelman-Rubin R-hat per element over m chains of n samples each (same element layout), summed over the
// chains in the order given:  W = (sum_c M2_c / (n-1)) / m,  mu = (sum_c mean_c) / m,
// B/n = (sum_c (mean_c - mu)^2) / (m - 1),  R = sqrt((((n-1)/n) W + B/n) / W);  NaN where W = 0.
const int DG_RHAT_MAX = 256;
struct RhatView {
  int m;
  const double2 *acc[DG_RHAT_MAX];
};
static __global__ void post_rhat_kernel(const RhatView v, int64_t len, int64_t n, double *rhat) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const double nd = (double)n, nm1 = (double)(n - 1), md = (double)v.m;
  const double shrink = __ddiv_rn(nm1, nd);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += stride) {
    double W = 0.0, mu = 0.0;
    for (int c = 0; c < v.m; c++) {
      const double2 a = v.acc[c][i];
      W = __dadd_rn(W, __ddiv_rn(a.y, nm1));
      mu = __dadd_rn(mu, a.x);
    }
    W = __ddiv_rn(W, md);
    mu = __ddiv_rn(mu, md);
    double B = 0.0;
    for (int c = 0; c < v.m; c++) {
      const double d = __dsub_rn(v.acc[c][i].x, mu);
      B = __dadd_rn(B, __dmul_rn(d, d));
    }
    B = __ddiv_rn(B, md - 1.0);
    rhat[i] = W == 0.0 ? CUDART_NAN : __dsqrt_rn(__ddiv_rn(__dadd_rn(__dmul_rn(shrink, W), B), W));
  }
}

// Batch-means effective sample size and Monte Carlo standard error per element over m chains (m = 1: one chain) of
// n samples and K = n / b complete batches each; {bmean, bM2} of chain c sits `boff` pairs after its {mean, M2}.
// Sums over the chains in the order given, each operation rounded separately:
//   mu = (sum mean_c) / m,   A = sum M2_c,   D = sum (mean_c - mu)^2,    s2 = (A + n D) / (m n - 1)
//   mub = (sum bmean_c) / m, Ab = sum bM2_c, Db = sum (bmean_c - mub)^2, sig2 = b (Ab + K Db) / (m K - 1)
//   ess = (m n) s2 / sig2,   mcse = sqrt(sig2 / (m n));  both NaN where sig2 = 0.
static __global__ void post_ess_kernel(const RhatView v, int64_t boff, int64_t len, int64_t n, int64_t K, double b,
                                       double *ess, double *mcse) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const double md = (double)v.m, nd = (double)n, kd = (double)K, mn = (double)(v.m * n);
  const double mn1 = (double)(v.m * n - 1), mk1 = (double)(v.m * K - 1);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += stride) {
    double mu = 0.0, A = 0.0, mub = 0.0, Ab = 0.0;
    for (int c = 0; c < v.m; c++) {
      const double2 a = v.acc[c][i], ab = v.acc[c][boff + i];
      mu = __dadd_rn(mu, a.x);
      A = __dadd_rn(A, a.y);
      mub = __dadd_rn(mub, ab.x);
      Ab = __dadd_rn(Ab, ab.y);
    }
    mu = __ddiv_rn(mu, md);
    mub = __ddiv_rn(mub, md);
    double D = 0.0, Db = 0.0;
    for (int c = 0; c < v.m; c++) {
      const double d = __dsub_rn(v.acc[c][i].x, mu), db = __dsub_rn(v.acc[c][boff + i].x, mub);
      D = __dadd_rn(D, __dmul_rn(d, d));
      Db = __dadd_rn(Db, __dmul_rn(db, db));
    }
    const double s2 = __ddiv_rn(__dadd_rn(A, __dmul_rn(nd, D)), mn1);
    const double sig2 = __ddiv_rn(__dmul_rn(b, __dadd_rn(Ab, __dmul_rn(kd, Db))), mk1);
    if (ess) ess[i] = sig2 == 0.0 ? CUDART_NAN : __ddiv_rn(__dmul_rn(mn, s2), sig2);
    if (mcse) mcse[i] = sig2 == 0.0 ? CUDART_NAN : __dsqrt_rn(__ddiv_rn(sig2, mn));
  }
}
