// kernels_post.cuh -- running posterior mean and variance of the chain state (dang_gpu_posterior_*; not in the
// reference, whose users write every sample with write_maps and average offline).  Accumulators hold one 16-byte
// {mean, M2} pair per element.  Every step is spelled with _rn intrinsics: the build contracts a*b+c to an FMA by
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
