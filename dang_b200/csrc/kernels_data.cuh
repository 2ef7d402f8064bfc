// kernels_data.cuh -- K6: update_sky_model + compute_chisq (SURVEY rows a20, a21),
// src/dang_data_mod.f90:339-396, 494-526, fused into one pass over sig/rms.
// sky_model / res_map / chi_map are only materialised when the host asks for them
// (write_maps cadence, src/dang.f90:119-121); the per-iteration call just reduces chi-square.
#pragma once
#include "common.cuh"

struct ChisqView {
  int k_lo, k_hi;     // 0-based plane range of ddata%pol_type
  double *sky, *res;  // [nbands][nmaps][Ppad] or nullptr
  double *chi_map;    // [nmaps][Ppad] or nullptr
};

// Where K6 puts what it computes per pixel: the sky model and residual t of every (band, plane), and chi_map(:,k).
// ChisqStore writes the maps the host asked for and reduces chi-square (dang_gpu_chisq / dang_gpu_get_sky_model);
// the posterior sink of kernels_post.cuh folds them into running moments instead.  kMaps: the sink always takes
// the maps (every plane, every pixel, as dang_gpu_get_sky_model); kReduce: the chi-square sums go to `out`.
struct ChisqStore {
  static constexpr bool kMaps = false, kReduce = true;
  __device__ __forceinline__ void sky(const ChisqView &cv, size_t off, double v) const { if (cv.sky) cv.sky[off] = v; }
  __device__ __forceinline__ void res(const ChisqView &cv, size_t off, double v) const { if (cv.res) cv.res[off] = v; }
  __device__ __forceinline__ void chi(const ChisqView &cv, size_t off, double v) const { if (cv.chi_map) cv.chi_map[off] = v; }
};

// K6.  out[0..2] = sum over unmasked pixels of chi_map(:,k) (already / nbands), out[3] = #unmasked (ChisqStore)
template <int NC, class Sink = ChisqStore>
__global__ void __launch_bounds__(DG_THREADS)
chisq_kernel(const ModelView mv, const ChisqView cv, double *partials, unsigned int *ticket,
             double *out, const Sink sink = Sink()) {
  __shared__ double smem[4 * 32];
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
  const bool maps = Sink::kMaps || cv.sky != nullptr || cv.res != nullptr;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < mv.P; p += stride) {
    const bool use = mv.mask[p] != 0;
    if (use) acc[3] += 1.0;
    if (!use && !maps) {
      if (cv.chi_map)
        for (int k = 0; k < mv.nmaps; k++) cv.chi_map[(size_t)k * mv.Ppad + p] = 0.0;
      continue;
    }
    // update_sky_model covers every plane and every pixel; compute_chisq only pol_type planes
    const int ka = maps ? 0 : cv.k_lo, kb = maps ? mv.nmaps - 1 : cv.k_hi;
    double a[3][NC], th[3][NC][DG_MAXIND];
#pragma unroll
    for (int k = 0; k < 3; k++) {
      if (k < ka || k > kb) continue;
      const size_t kp = (size_t)k * mv.Ppad + p;
#pragma unroll
      for (int c = 0; c < NC; c++) {
        if (c < mv.ncomp) {
          const CompView &cc = mv.comp[c];
          a[k][c] = cc.amp[kp];
          th[k][c][0] = cc.nind > 0 ? cc.idx[0][kp] : 0.0;
          th[k][c][1] = cc.nind > 1 ? cc.idx[1][kp] : 0.0;
        }
      }
    }
    double chi[3] = {0.0, 0.0, 0.0};
    for (int j = 0; j < mv.nbands; j++) {
      double sed[3][NC];
#pragma unroll
      for (int k = 0; k < 3; k++) {
        if (k < ka || k > kb) continue;
#pragma unroll
        for (int c = 0; c < NC; c++) {
          if (c < mv.ncomp) {
            if (k > ka && mv.comp[c].tamp == nullptr && sed_uniform(mv, c, k) == sed_uniform(mv, c, k > 0 ? k - 1 : 0) && th[k][c][0] == th[k > 0 ? k - 1 : 0][c][0] && th[k][c][1] == th[k > 0 ? k - 1 : 0][c][1])
              sed[k][c] = sed[k > 0 ? k - 1 : 0][c];
            else
              sed[k][c] = sed_eval(mv, c, k, j, th[k][c][0], th[k][c][1]);
          }
        }
      }
#pragma unroll
      for (int k = 0; k < 3; k++) {
        if (k < ka || k > kb) continue;
        const size_t off = plane_off(mv, j, k) + p;
        double sky = 0.0;  // :354, :367
#pragma unroll
        for (int c = 0; c < NC; c++)
          if (c < mv.ncomp && mv.comp[c].in_sky) sky = sky + a[k][c] * sed[k][c];  // (monopoles are offsets, :357-361)
        const double sig = ldg_stream(mv.sig + off);
        const double t = (k == 0) ? (sig - mv.offset[j]) / mv.gain[j] - sky : sig - sky;  // :384-387
        sink.sky(cv, off, sky);
        sink.res(cv, off, t);
        if (use && k >= cv.k_lo && k <= cv.k_hi) {
          const double rms = ldg_stream(mv.rms + off);
          chi[k] = chi[k] + (t * t) / (rms * rms);  // :510-516
        }
      }
    }
#pragma unroll
    for (int k = 0; k < 3; k++) {
      if (k >= mv.nmaps) continue;
      const double v = (use && k >= cv.k_lo && k <= cv.k_hi) ? chi[k] / mv.nbands : 0.0;  // :523
      sink.chi(cv, (size_t)k * mv.Ppad + p, v);
      acc[k] += v;
    }
  }
  if constexpr (Sink::kReduce) grid_reduce<4>(acc, smem, partials, ticket, out);
}

// mask_avg, src/dang_util_mod.f90:186-206: out[0] = sum over unmasked of map, out[1] = count
static __global__ void __launch_bounds__(DG_THREADS)
masked_sum_kernel(const double *map, const unsigned char *mask, int64_t P, double *partials,
                  unsigned int *ticket, double *out) {
  __shared__ double smem[4 * 32];
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < P; p += stride)
    if (!mask || mask[p]) {  // (mask == nullptr: the plain sum over every pixel)
      acc[0] += map[p];
      acc[1] += 1.0;
    }
  grid_reduce<4>(acc, smem, partials, ticket, out);
}

static __global__ void fill_kernel(double *dst, int64_t n, double v) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) dst[i] = v;
}

// mask (double, 0 / missval = masked) -> bytes, src/dang_data_mod.f90:153-161
static __global__ void mask_to_bytes_kernel(const double *mask, unsigned char *out, int64_t P, int64_t Ppad) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < Ppad; i += stride)
    out[i] = (i < P && mask[i] != 0.0 && mask[i] != -1.6375e30) ? 1 : 0;
}

// ---------------------------------------------------------------- SED tables
// uniform_check_kernel: does index map (c, l) hold one value on plane k (over ALL local pixels)?
// grid = (blocks, ncomp * 3 * DG_MAXIND); the nonuni flags of the maps selected by check_mask must
// be zero on entry.  Maps written by the samplers are never re-scanned: a full-sky draw leaves a
// constant plane, a per-pixel draw a varying one, and the host sets their flags directly.
static __global__ void __launch_bounds__(DG_THREADS)
uniform_check_kernel(const ModelView mv, SedTable *tab, unsigned long long check_mask) {
  const int m = blockIdx.y;
  const int l = m % DG_MAXIND, k = (m / DG_MAXIND) % 3, c = m / (DG_MAXIND * 3);
  if (c >= mv.ncomp || k >= mv.nmaps || l >= mv.comp[c].nind) return;
  if (!((check_mask >> m) & 1ull)) return;  // this map's flag is already known
  const double *map = mv.comp[c].idx[l] + (size_t)k * mv.Ppad;
  const double first = map[0];
  bool bad = false;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < mv.P; p += stride)
    bad = bad || !(map[p] == first);  // NaN counts as non-uniform
  if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(&tab->nonuni[c * 3 + k][l], 1);
}

// sed_table_kernel<<<ncomp*3, 32>>>: tabulate the per-band SED of every uniform (component, plane)
static __global__ void sed_table_kernel(const ModelView mv, SedTable *tab) {
  const int ck = blockIdx.x, c = ck / 3, k = ck % 3;
  if (c >= mv.ncomp || k >= mv.nmaps) {
    if (threadIdx.x == 0) tab->uni[ck] = 0;
    return;
  }
  const CompView &cv = mv.comp[c];
  bool uni = true;
  for (int l = 0; l < cv.nind; l++) uni = uni && tab->nonuni[ck][l] == 0;
  if (cv.tamp && cv.type != 9) {  // 'template' / 'monopole': eval_signal = template_amplitudes(band, plane) * template(pix, plane)
    for (int j = threadIdx.x; j < mv.nbands; j += blockDim.x) tab->sed[ck][j] = cv.tamp[k * DG_MAX_BANDS + j];
  } else if (uni) {
    const double t0 = cv.nind > 0 ? cv.idx[0][(size_t)k * mv.Ppad] : 0.0;
    const double t1 = cv.nind > 1 ? cv.idx[1][(size_t)k * mv.Ppad] : 0.0;
    for (int j = threadIdx.x; j < mv.nbands; j += blockDim.x) tab->sed[ck][j] = sed_theta(mv, c, j, t0, t1, k);
  }
  if (threadIdx.x == 0) tab->uni[ck] = uni ? 1 : 0;
}

// fit_band_gain, src/dang_sample_mod.f90:570-621: the two masked, noise-weighted dot products of
// one band against the current sky model.  out[0] = sum(map2*N_inv*map1), out[1] = sum(map1*N_inv*map1)
// with map1 = sky_model, map2 = res_map + sky_model (update_sky_model :384-387 fused in).
static __global__ void __launch_bounds__(DG_THREADS)
band_gain_kernel(const ModelView mv, int k, int band, double *partials, unsigned int *ticket, double *out) {
  __shared__ double smem[4 * 32];
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < mv.P; p += stride) {
    if (!mv.mask[p]) continue;
    const size_t kp = (size_t)k * mv.Ppad + p;
    double sky = 0.0;
    for (int c = 0; c < mv.ncomp; c++) {
      const CompView &cc = mv.comp[c];
      if (!cc.in_sky) continue;
      const double t0 = cc.nind > 0 ? cc.idx[0][kp] : 0.0, t1 = cc.nind > 1 ? cc.idx[1][kp] : 0.0;
      sky = sky + cc.amp[kp] * sed_eval(mv, c, k, band, t0, t1);
    }
    const size_t off = plane_off(mv, band, k) + p;
    const double sig = mv.sig[off], noise = mv.rms[off];
    const double res = (k == 0) ? (sig - mv.offset[band]) / mv.gain[band] - sky : sig - sky;
    const double map1 = sky, map2 = res + sky;
    const double N_inv = 1.0 / (noise * noise);
    acc[0] += map2 * N_inv * map1;
    acc[1] += map1 * N_inv * map1;
  }
  grid_reduce<4>(acc, smem, partials, ticket, out);
}
