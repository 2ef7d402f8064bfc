// kernels_mh_fast.cuh -- K5 with certified single-precision screening.
//
// Per-pixel branch of sample_index_mh (src/dang_sample_mod.f90:332-481), chisq likelihood with a
// uniform / Gaussian prior, delta bands, power-law beta / mbb beta / mbb T: the configurations whose
// cost is nsample * nbands fp64 exp() per pixel in mh_perpixel_kernel (FP64-pipe / issue bound:
// 157 ms per index at nside 2048 x 20 bands against 6 ms of compulsory HBM traffic).
//
// A Metropolis step only needs the SIGN of (lnL(theta') - lnL(cur)) - ln u.  With the residuals of the
// chain's CURRENT point held per (band, Stokes),
//     t = (d - a s_cur) / sigma,   g = a s_cur / sigma,
//     s(theta') = s_cur (1 + rho),  rho = exp((theta' - cur) L_j) - 1           (beta)
//                                   rho = P_j(T')/P_j(cur) - 1                  (T, Planck ratio, see below)
//     lnL(theta') - lnL(cur) = 1/2 sum a (2 t - a),   a = g rho,
// the data term has cancelled analytically and what is left is a short sum of well-scaled products
// that fp32 evaluates to ~1e-6 of E = sum |g| b (2 |t| + 2 |g| b), b >= |rho| being the magnitude the
// rounding error of rho scales with (rho comes from expm1f of an fp64-exact difference theta' - cur).
// t and g start from an fp64 evaluation at the chain's first point and follow accepted moves in fp32
// (t -= a, g += a); a running bound dT on the error this leaves in t enters the error budget.
// Every proposal is screened with
//     diff~ = 1/2 sum a (2 t - a) + (prior' - prior_cur),   eps = kappa E + 2 dT sum |a| + eps_u
// and decided from diff~ when |diff~ - ln u| > eps.  Otherwise (~1e-4 of the proposals) the warp
// re-evaluates lnL(theta') and lnL(cur) in fp64 with exactly the arithmetic of mh_perpixel_kernel and
// decides from that.  Either way the decision is the one the fp64 kernel takes; accepted proposals
// are stored verbatim, so the index maps carry the same bits.  Per proposal and band the fp64 exp
// (~50 issue slots, 2 cycles each on the FP64 pipe) becomes ~25 fp32 instructions.
//
// In record mode (DANG_OPT_RECORD_DECISIONS) the kernel also evaluates every proposal in fp64, writes
// that lnL to the trace, and counts (out[2]) the proposals whose screened quantities broke the bound
// or whose certain decision differs from the fp64 one -- the parity tests require zero.
// out[0] = accepted proposals, out[1] = proposals decided by the fp64 fallback, out[2] = violations.
#pragma once
#include "kernels_mh.cuh"

// T mode: with y = h nu / (k T_cur), w = 1/T' - 1/T_cur and em1 = exp() - 1,
//   em1(y T_cur/T') / em1(y) = 1 + K em1(h nu w / k),  K = 1 / (1 - exp(-y)) = 1 + 1/em1(y),
// so rho_j = (K_ref em1(c_ref w) - K_j em1(c_j w)) / (1 + K_j em1(c_j w)): every term is O(w), which keeps
// the RELATIVE accuracy of rho at fp32 level for small steps (a plain ratio of four fp32 expm1 values
// would carry an absolute error of ~1e-6 and force a fallback on every bright pixel).
#define DG_K5_KAPPA_BETA 1.0e-6f
#define DG_K5_KAPPA_T 1.5e-6f

// exp(x) - 1 in single precision: Taylor to x^7 for |x| < 0.35 (relative error ~2 ulp), ex2.approx beyond
// (where exp(x) - 1 is no longer small against the absolute error of exp; relative error < 1e-6 (1 + |x|/3)).
// `w` returns the weight of the result in the error budget: 1 on the Taylor branch, 4 (1 + |x|/3) beyond.
__device__ __forceinline__ float k5_em1f(float x, float &w) {
  w = fabsf(x) < 0.35f ? 1.0f : fmaf(fabsf(x), 4.0f / 3.0f, 4.0f);
  float p = fmaf(x, 1.0f / 5040.0f, 1.0f / 720.0f);
  p = fmaf(p, x, 1.0f / 120.0f);
  p = fmaf(p, x, 1.0f / 24.0f);
  p = fmaf(p, x, 1.0f / 6.0f);
  p = fmaf(p, x, 0.5f);
  p = fmaf(p, x, 1.0f);
  const float e = __expf(x) - 1.0f;
  return fabsf(x) < 0.35f ? p * x : e;
}
__device__ __forceinline__ float k5_em1f(float x) {
  float p = fmaf(x, 1.0f / 5040.0f, 1.0f / 720.0f);
  p = fmaf(p, x, 1.0f / 120.0f);
  p = fmaf(p, x, 1.0f / 24.0f);
  p = fmaf(p, x, 1.0f / 6.0f);
  p = fmaf(p, x, 0.5f);
  p = fmaf(p, x, 1.0f);
  const float e = __expf(x) - 1.0f;
  return fabsf(x) < 0.35f ? p * x : e;
}

// data_raw and 1/sigma of one (band, plane, pixel): out of line, so that the (large) SED dispatch of the
// other components exists once in the kernel instead of once per call site
static __device__ __noinline__ void k5_fetch(const ModelView &mv, int ic, int j, int k, int64_t pp, double &D, double &sig) {
  D = mh_data_value(mv, ic, j, k, pp);
  sig = ldg_stream(mv.rms + plane_off(mv, j, k) + pp);
}

// this lane's share of lnL(xe) in fp64: the arithmetic (and order) of mh_perpixel_kernel, on the data
// residuals D and noise sigma this thread parked in shared memory (dw[(q * BPL + i) * threads + tid],
// q = 0..3: D0, sigma0, D1, sigma1)
template <int BPL, int MODE>
__device__ __noinline__ double k5_exact_part(const ModelView &mv, const MhView &mh, const double *dw, int r, double xe,
                                             double idx0, double idx1, double amp0, double amp1) {
  constexpr int L = DG_MH_LANES;
  const int B = mv.nbands, S = mh.S;
  const CompView &cv = mv.comp[mh.ic];
  const SedTable &tab = *mv.tab;
  const double nu_ref = cv.nu_ref;
  double zT = 0.0, eref = 0.0, zF = 0.0, erefF = 0.0;
  if (MODE == MH_SED_MBB_T) {
    zT = DG_H / (DG_KB * xe);
    eref = exp(zT * nu_ref) - 1.0;
  }
  if (MODE == MH_SED_MBB_BETA) {
    zF = DG_H / (DG_KB * idx1);
    erefF = exp(zF * nu_ref) - 1.0;
  }
  double part = 0.0;
#pragma unroll 1
  for (int i = 0; i < BPL; i++) {
    const int j = r + i * L;
    if (j < B) {
      const double Lh = tab.lnr_hi[mh.ic][j], Ll = tab.lnr_lo[mh.ic][j], nuc = mv.band[j].nu_c;
      const double D0 = dw[(0 * BPL + i) * DG_MH_THREADS];
      const double W0 = 1.0 / dw[(1 * BPL + i) * DG_MH_THREADS];
      double sed;
      if (MODE == MH_SED_POWERLAW) {
        sed = exp_scaled(xe, Lh, Ll);
      } else if (MODE == MH_SED_MBB_BETA) {
        const double F = erefF / (exp(zF * nuc) - 1.0);
        sed = F * exp_scaled(xe + 1.0, Lh, Ll);
      } else {
        const double F = exp_scaled(idx0 + 1.0, Lh, Ll);
        sed = eref * mh_fast_rcp(exp(zT * nuc) - 1.0) * F;
      }
      const double t0 = (D0 - amp0 * sed) * W0;
      part = part - 0.5 * (t0 * t0);
      if (S > 1) {
        const double D1 = dw[(2 * BPL + i) * DG_MH_THREADS];
        const double W1 = 1.0 / dw[(3 * BPL + i) * DG_MH_THREADS];
        const double t1 = (D1 - amp1 * sed) * W1;
        part = part - 0.5 * (t1 * t1);
      }
    }
  }
  return part;
}

template <int BPL, int MODE>
__global__ void __launch_bounds__(DG_MH_THREADS, 4)
mh_perpixel_fast_kernel(const __grid_constant__ ModelView mv, const __grid_constant__ MhView mh, double *partials,
                        unsigned int *ticket, double *out) {
  constexpr int L = DG_MH_LANES;
  constexpr int PB = DG_MH_THREADS / L;  // pixels per block iteration
  constexpr int PW = 32 / L;             // pixels per warp
  extern __shared__ double dyn[];        // zs[PB][nsample], us[PB][nsample], dw[4 * BPL][threads]
  __shared__ double smem[4 * 32];
  const int tid = threadIdx.x, lane = tid & 31, r = tid % L, g = tid / L, B = mv.nbands, S = mh.S;
  const int nsample = mh.nsample;
  const unsigned full = 0xffffffffu;
  double *zs = dyn + (size_t)g * nsample, *us = dyn + (size_t)(PB + g) * nsample;
  double *wzs = dyn + (size_t)(g - lane / L) * nsample;  // first pixel of this warp
  double *wus = wzs + (size_t)PB * nsample;
  double *dw = dyn + (size_t)2 * PB * nsample + tid;  // fp64 data residuals / sigma of this thread's bands
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
  const CompView &cv = mv.comp[mh.ic];
  const SedTable &tab = *mv.tab;
  const double nu_ref = cv.nu_ref;
  const double ln_denom = log(mh.gauss[1] * sqrt(2.0 * DG_PI));
  const double inv2var = 1.0 / (2 * (mh.gauss[1] * mh.gauss[1]));
  const bool record = mh.decisions != nullptr;
  const float kappa = MODE == MH_SED_MBB_T ? DG_K5_KAPPA_T : DG_K5_KAPPA_BETA;

  // band constants in single precision: ln(nu/nu_ref) (beta modes) or h nu / k (T mode); in shared memory
  // (indexed by band) rather than BPL registers per lane: the chain loop is register-bound
  __shared__ float scf[BPL * L];
  if (tid < BPL * L) {
    const int j = tid;
    if (MODE == MH_SED_MBB_T) scf[j] = j < B ? (float)(DG_H / DG_KB * mv.band[j].nu_c) : 0.0f;
    else scf[j] = j < B ? (float)tab.lnr_hi[mh.ic][j] : 0.0f;
  }
  __syncthreads();
  const float *cf = scf + r;  // band r + i L -> cf[i * L]
  const float cref = (float)(DG_H / DG_KB * nu_ref);

  const int64_t ngroups = (int64_t)gridDim.x * PB;
  const int64_t niter = (mv.P + ngroups - 1) / ngroups;
  for (int64_t itp = 0; itp < niter; itp++) {
    const int64_t p = itp * ngroups + (int64_t)blockIdx.x * PB + g;
    const bool valid = p < mv.P;
    const bool use = valid && mv.mask[p] != 0;
    if (!use && valid && r == 0) {  // :362; index_map stays 0 for masked pixels (:223, :465, :483)
      for (int s = 0; s < S; s++) cv.idx[mh.nind][(size_t)mh.plane[s] * mv.Ppad + p] = 0.0;
      if (mh.decisions)
        for (int l = 0; l < nsample; l++) mh.decisions[(size_t)l * mv.P + p] = 3;
    }
    if (!__any_sync(full, use)) continue;
    const int64_t pp = use ? p : 0;
    const size_t kp0 = (size_t)mh.plane[0] * mv.Ppad + pp;
    const double idx0 = cv.nind > 0 ? cv.idx[0][kp0] : 0.0;  // :372-374
    const double idx1 = cv.nind > 1 ? cv.idx[1][kp0] : 0.0;
    const double theta_ref = mh.nind == 0 ? idx0 : idx1;
    double cur = theta_ref;
    const double amp0 = cv.amp[(size_t)mh.plane[0] * mv.Ppad + pp];
    const double amp1 = S > 1 ? cv.amp[(size_t)mh.plane[1] * mv.Ppad + pp] : 0.0;

    // ---- state at the chain's first point, evaluated in fp64, kept in fp32: t, g per (band, Stokes),
    //      gs = |g0| + |g1|; T mode: K_j = 1 + 1/em1(h nu_j / k T) per band and for the reference frequency
    float tr0[BPL], tr1[BPL], g0[BPL], g1[BPL], kj[BPL];
    float kref = 1.0f;
    {
      double zF = 0.0, erefF = 0.0;
      if (MODE != MH_SED_POWERLAW) {
        zF = DG_H / (DG_KB * idx1);             // T of the first point (idx1 == cur in T mode)
        erefF = exp(zF * nu_ref) - 1.0;
        kref = (float)(1.0 + 1.0 / erefF);
      }
#pragma unroll
      for (int i = 0; i < BPL; i++) {
        const int j = r + i * L;
        tr0[i] = tr1[i] = g0[i] = g1[i] = 0.0f;
        kj[i] = 1.0f;
        if (j < B) {
          const double Lh = tab.lnr_hi[mh.ic][j], Ll = tab.lnr_lo[mh.ic][j];
          double sed;
          if (MODE == MH_SED_POWERLAW) {
            sed = exp_scaled(idx0, Lh, Ll);
          } else {
            const double em1 = exp(zF * mv.band[j].nu_c) - 1.0;
            const double iem1 = mh_fast_rcp(em1);
            sed = erefF * iem1 * exp_scaled(idx0 + 1.0, Lh, Ll);
            kj[i] = (float)(1.0 + iem1);
          }
          double D0, s0;
          k5_fetch(mv, mh.ic, j, mh.plane[0], pp, D0, s0);
          dw[(0 * BPL + i) * DG_MH_THREADS] = D0;
          dw[(1 * BPL + i) * DG_MH_THREADS] = s0;
          const double W0 = mh_fast_rcp(s0), m0 = amp0 * sed;
          tr0[i] = (float)((D0 - m0) * W0);
          g0[i] = (float)(m0 * W0);
          if (S > 1) {
            double D1, s1;
            k5_fetch(mv, mh.ic, j, mh.plane[1], pp, D1, s1);
            dw[(2 * BPL + i) * DG_MH_THREADS] = D1;
            dw[(3 * BPL + i) * DG_MH_THREADS] = s1;
            const double W1 = mh_fast_rcp(s1), m1 = amp1 * sed;
            tr1[i] = (float)((D1 - m1) * W1);
            g1[i] = (float)(m1 * W1);
          }
        }
      }
    }
    // deviates of this warp's PW chains, slot-indexed (Q5), generated by all 32 lanes
    __syncwarp();
    {
      const int64_t p_first = itp * ngroups + (int64_t)blockIdx.x * PB + (g - lane / L);
      for (int q = lane; q < PW * nsample; q += 32) {
        const int gq = q / nsample, l = q - gq * nsample;
        int64_t pq = p_first + gq;
        if (pq >= mv.P) pq = 0;
        const size_t slot = (size_t)l * mv.P + pq;
        const uint64_t gslot = (uint64_t)l * (uint64_t)mv.npix + (uint64_t)(mv.pix_lo + pq);
        wzs[(size_t)gq * nsample + l] = mh.z ? mh.z[slot] : philox_normal(mh.seed, DG_STREAM_MH_Z, gslot);
        double uu = 1.0, u2;
        if (mh.ml_mode != 0) {
          if (mh.u) uu = mh.u[slot];
          else philox_uniform2(mh.seed, DG_STREAM_MH_U, gslot, uu, u2);
        }
        wus[(size_t)gq * nsample + l] = uu;
      }
    }
    __syncwarp();

    auto prior_of = [&](double xe) -> double {
      if (mh.prior_type != 1) return 0.0;
      const double a = ((xe - mh.gauss[0]) * (xe - mh.gauss[0])) * inv2var;
      return a < 700.0 ? -a - ln_denom : log_normal_prior(xe, mh.gauss[0], mh.gauss[1]);
    };
    auto exact_lnl = [&](double xe) -> double {  // the fp64 kernel's lnl_new for xe
      double part = k5_exact_part<BPL, MODE>(mv, mh, dw, r, xe, idx0, idx1, amp0, amp1);
      part += __shfl_xor_sync(full, part, 1);
      part += __shfl_xor_sync(full, part, 2);
      return part + prior_of(xe);
    };

    // bound on |t| over this pixel's bands (for the state-error budget)
    float tmax = 0.0f;
#pragma unroll
    for (int i = 0; i < BPL; i++) tmax = fmaxf(tmax, fmaxf(fabsf(tr0[i]), fabsf(tr1[i])));
    tmax = fmaxf(tmax, __shfl_xor_sync(full, tmax, 1));
    tmax = fmaxf(tmax, __shfl_xor_sync(full, tmax, 2));
    float dT = 1.2e-7f * tmax;  // error bound of the fp32 copies of t
    float kap = kappa;          // grows with every accepted move (relative error of g, em1)
    double prior_cur = prior_of(cur), naccept = 0.0;
    double lnl_cur_x = 0.0;   // fp64 lnL(cur) when a fallback has already evaluated it
    bool have_cur_x = false, need_tmax = false;
    for (int l = 0; l < nsample; l++) {
      const double x = cur + (0.0 + mh.step * zs[l]);       // :414
      const bool oob = x < mh.uni[0] || x > mh.uni[1];      // :415, Q5
      const size_t slot = (size_t)l * mv.P + pp;
      // ---- screened evaluation: this lane's share of the difference, of A1 = sum |g| b (b >= |rho| is the
      //      magnitude the rounding error of rho scales with) and of A2 = sum |a|
      float lam = 0.0f, A1 = 0.0f, A2 = 0.0f, n1 = 0.0f, w1 = 1.0f;
      float rho[BPL];
#pragma unroll
      for (int i = 0; i < BPL; i++) rho[i] = 0.0f;
      if (!oob) {
        float d;
        if (MODE == MH_SED_MBB_T) {
          d = (float)((cur - x) * mh_fast_rcp(x * cur));    // w = 1/T' - 1/T_cur
          n1 = kref * k5_em1f(cref * d, w1);
        } else {
          d = (float)(x - cur);
        }
#pragma unroll
        for (int i = 0; i < BPL; i++) {
          float b, w2;
          if (MODE == MH_SED_MBB_T) {
            const float n2 = kj[i] * k5_em1f(cf[i * L] * d, w2);
            const float inv = __frcp_rn(1.0f + n2);
            rho[i] = (n1 - n2) * inv;
            b = fmaf(fabsf(n1), w1, fabsf(n2) * w2) * inv;
          } else {
            const float xx = d * cf[i * L];
            rho[i] = k5_em1f(xx, w2);
            b = fabsf(rho[i]) * w2 * (1.0f + fabsf(xx));
          }
          const float a0 = g0[i] * rho[i], a1 = g1[i] * rho[i];
          lam = fmaf(a0, fmaf(2.0f, tr0[i], -a0), lam);
          lam = fmaf(a1, fmaf(2.0f, tr1[i], -a1), lam);
          A1 = fmaf(fabsf(g0[i]) + fabsf(g1[i]), b, A1);
          A2 += fabsf(a0) + fabsf(a1);
        }
      }
      lam += __shfl_xor_sync(full, lam, 1);
      lam += __shfl_xor_sync(full, lam, 2);
      A1 += __shfl_xor_sync(full, A1, 1);
      A1 += __shfl_xor_sync(full, A1, 2);
      A2 += __shfl_xor_sync(full, A2, 1);
      A2 += __shfl_xor_sync(full, A2, 2);
      const float E = 2.0f * A1 * (tmax + A2);              // >= sum |g| b (2 |t| + 2 |a|)
      const double prior_new = oob ? prior_cur : prior_of(x);
      const double diff_s = 0.5 * (double)lam + (prior_new - prior_cur);
      const double uu = us[l];
      float lu = 0.0f, eps_u = 0.0f;
      if (mh.ml_mode != 0) {
        lu = __logf((float)uu);                             // :450 (Q4), screened
        eps_u = 1.5e-6f * (1.0f + fabsf(lu));
      }
      const float eps = kap * E + 2.0f * dT * A2 + 2.5e-7f * A2 * (tmax + A2) + eps_u + 1.0e-30f;
      const bool certain = fabs(diff_s - (double)lu) > (double)eps;  // false for NaN / inf
      bool accept = diff_s > (double)lu;
      const bool need = use && !oob && !certain;
      const bool fallback = __any_sync(full, need) || record;
      if (fallback) {  // fp64 re-evaluation for the whole warp (shuffles stay convergent)
        const double xe = oob ? cur : x;
        const double lnl_new = exact_lnl(xe);
        if (__any_sync(full, !have_cur_x)) {
          const double v = exact_lnl(cur);
          if (!have_cur_x) lnl_cur_x = v;
          have_cur_x = true;
        }
        const double lnl_old = lnl_cur_x;
        const double diff = lnl_new - lnl_old;
        const bool acc_x = (mh.ml_mode == 0) ? (diff > 0.0) : (diff > log(uu));
        if (record && !oob && use && r == 0) {
          if (mh.lnl_trace) mh.lnl_trace[slot] = lnl_new;
          const double scale = fmax(1.0, fmax(fabs(lnl_new), fabs(lnl_old)));
          const bool bound_ok = fabs(diff_s - diff) <= (double)eps + 1e-13 * scale;
          if (!bound_ok || (certain && acc_x != accept)) acc[2] += 1.0;
        }
        if (need) {
          accept = acc_x;
          if (r == 0) acc[1] += 1.0;
        }
        if (accept && !oob) lnl_cur_x = lnl_new;   // stays valid for the new point
      } else if (accept && !oob) {
        have_cur_x = false;
      }
      // (accept is only meaningful for in-bounds proposals)
      if (oob) accept = false;  // (no divergent `continue`: the warp meets again at the shuffles below)
      if (accept) {  // the state follows the chain: t -= a, g += a (s_new = s_cur (1 + rho))
        cur = x;
        prior_cur = prior_new;
        naccept += 1.0;
        float iT = 0.0f;
        if (MODE == MH_SED_MBB_T) {  // K_j at the new temperature, from scratch (no error accumulation)
          iT = (float)mh_fast_rcp(cur);
          kref = 1.0f + __frcp_rn(k5_em1f(cref * iT));
        }
#pragma unroll
        for (int i = 0; i < BPL; i++) {
          const float a0 = g0[i] * rho[i], a1 = g1[i] * rho[i];
          tr0[i] -= a0;
          tr1[i] -= a1;
          g0[i] += a0;
          g1[i] += a1;
          // (padding bands keep K = 1: with c_j = 0, 1 / em1(0) would make every later proposal NaN)
          if (MODE == MH_SED_MBB_T && r + i * L < B) kj[i] = 1.0f + __frcp_rn(k5_em1f(cf[i * L] * iT));
        }
        dT += kap * A1 + 1.2e-7f * (tmax + A2);       // error of a (b-scaled) + rounding of t - a
        kap += 1.5e-7f;                               // g picks up ~1 ulp per update
        need_tmax = true;
      }
      if (__any_sync(full, need_tmax)) {  // max |t| of the moved state (all lanes take part in the shuffles)
        float m = 0.0f;
#pragma unroll
        for (int i = 0; i < BPL; i++) m = fmaxf(m, fmaxf(fabsf(tr0[i]), fabsf(tr1[i])));
        m = fmaxf(m, __shfl_xor_sync(full, m, 1));
        m = fmaxf(m, __shfl_xor_sync(full, m, 2));
        if (need_tmax) tmax = m;
        need_tmax = false;
      }
      if (use && r == 0 && mh.decisions) mh.decisions[slot] = oob ? 2 : (accept ? 1 : 0);
    }
    if (use && r == 0) {
      for (int s = 0; s < S; s++) cv.idx[mh.nind][(size_t)mh.plane[s] * mv.Ppad + p] = cur;  // :465, :483
      acc[0] += naccept;
    }
  }
  grid_reduce<4>(acc, smem, partials, ticket, out);
}

// ======================================================================================
// Split form (DANG_OPT_PERPIXEL_FAST = 2; a measured experiment, OFF by default):
//   k5_rng_kernel     the chain's deviates z, u for every (proposal, pixel) -> global (fp64 Box-Muller,
//                     fully parallel, off the chains' critical path)
//   k5_state_kernel   the fp64 state at the chain's first point -> fp32 scratch (t, g per band / Stokes)
//   k5_chain_kernel   the screened chains: fp32 hot loop only, register-light; an uncertain proposal
//                     calls the out-of-line fp64 evaluation (maps re-read from HBM, ~5e-4 of the proposals)
// Same arithmetic as the monolithic kernel in every step, so the decisions are the same
// (tests/test_gpu_parity.py::test_perpixel_split_form_matches).  MEASURED (B200, config c4 at nside 512):
// rng 0.84 ms + state + chain 10.1 ms against 7.9 ms for the monolithic kernel: the chain loop alone still
// wants more than 128 registers (5 bands x {t0, t1, g0, g1, |g|, K, c, rho} per lane + the fp64 chain state),
// so occupancy does not improve, and reading z / u from global memory per proposal exposes latency the
// monolithic kernel hides by parking them in shared memory.
// ======================================================================================

// this lane's share of lnL(xe) in fp64 straight from the maps (rare path of the chain kernel)
template <int BPL, int MODE>
__device__ __noinline__ double k5_exact_part_global(const ModelView &mv, const MhView &mh, int r, int64_t pp, double xe,
                                                    double idx0, double idx1, double amp0, double amp1) {
  constexpr int L = DG_MH_LANES;
  const int B = mv.nbands, S = mh.S;
  const CompView &cv = mv.comp[mh.ic];
  const SedTable &tab = *mv.tab;
  const double nu_ref = cv.nu_ref;
  double zT = 0.0, eref = 0.0, zF = 0.0, erefF = 0.0;
  if (MODE == MH_SED_MBB_T) {
    zT = DG_H / (DG_KB * xe);
    eref = exp(zT * nu_ref) - 1.0;
  }
  if (MODE == MH_SED_MBB_BETA) {
    zF = DG_H / (DG_KB * idx1);
    erefF = exp(zF * nu_ref) - 1.0;
  }
  double part = 0.0;
#pragma unroll 1
  for (int i = 0; i < BPL; i++) {
    const int j = r + i * L;
    if (j < B) {
      const double Lh = tab.lnr_hi[mh.ic][j], Ll = tab.lnr_lo[mh.ic][j], nuc = mv.band[j].nu_c;
      double D0, s0;
      k5_fetch(mv, mh.ic, j, mh.plane[0], pp, D0, s0);
      const double W0 = 1.0 / s0;
      double sed;
      if (MODE == MH_SED_POWERLAW) {
        sed = exp_scaled(xe, Lh, Ll);
      } else if (MODE == MH_SED_MBB_BETA) {
        const double F = erefF / (exp(zF * nuc) - 1.0);
        sed = F * exp_scaled(xe + 1.0, Lh, Ll);
      } else {
        const double F = exp_scaled(idx0 + 1.0, Lh, Ll);
        sed = eref * mh_fast_rcp(exp(zT * nuc) - 1.0) * F;
      }
      const double t0 = (D0 - amp0 * sed) * W0;
      part = part - 0.5 * (t0 * t0);
      if (S > 1) {
        double D1, s1;
        k5_fetch(mv, mh.ic, j, mh.plane[1], pp, D1, s1);
        const double W1 = 1.0 / s1;
        const double t1 = (D1 - amp1 * sed) * W1;
        part = part - 0.5 * (t1 * t1);
      }
    }
  }
  return part;
}

// z[l][p], u[l][p] for this handle's pixels (slot-indexed by the GLOBAL pixel number, Q5 / DESIGN.md "RNG")
static __global__ void __launch_bounds__(256)
k5_rng_kernel(const ModelView mv, const MhView mh, double *z, double *u) {
  const int64_t n = (int64_t)mh.nsample * mv.P, stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const int64_t l = i / mv.P, p = i - l * mv.P;
    if (!mv.mask[p]) continue;
    const uint64_t gslot = (uint64_t)l * (uint64_t)mv.npix + (uint64_t)(mv.pix_lo + p);
    z[i] = philox_normal(mh.seed, DG_STREAM_MH_Z, gslot);
    double uu = 1.0, u2;
    if (mh.ml_mode != 0) philox_uniform2(mh.seed, DG_STREAM_MH_U, gslot, uu, u2);
    u[i] = uu;
  }
}

// fp64 state at the chain's first point -> st4[(i * P + p) * L + r] = {t0, t1, g0, g1}, kj[...] (T mode: K_j)
template <int BPL, int MODE>
__global__ void __launch_bounds__(DG_MH_THREADS)
k5_state_kernel(const __grid_constant__ ModelView mv, const __grid_constant__ MhView mh, float4 *st4, float *kjs) {
  constexpr int L = DG_MH_LANES;
  constexpr int PB = DG_MH_THREADS / L;
  const int tid = threadIdx.x, r = tid % L, g = tid / L, B = mv.nbands, S = mh.S;
  const CompView &cv = mv.comp[mh.ic];
  const SedTable &tab = *mv.tab;
  const double nu_ref = cv.nu_ref;
  const int64_t ngroups = (int64_t)gridDim.x * PB;
  for (int64_t p = (int64_t)blockIdx.x * PB + g; p < mv.P; p += ngroups) {
    if (!mv.mask[p]) continue;
    const size_t kp0 = (size_t)mh.plane[0] * mv.Ppad + p;
    const double idx0 = cv.nind > 0 ? cv.idx[0][kp0] : 0.0;
    const double idx1 = cv.nind > 1 ? cv.idx[1][kp0] : 0.0;
    const double amp0 = cv.amp[(size_t)mh.plane[0] * mv.Ppad + p];
    const double amp1 = S > 1 ? cv.amp[(size_t)mh.plane[1] * mv.Ppad + p] : 0.0;
    double zF = 0.0, erefF = 0.0;
    if (MODE != MH_SED_POWERLAW) {
      zF = DG_H / (DG_KB * idx1);
      erefF = exp(zF * nu_ref) - 1.0;
    }
#pragma unroll
    for (int i = 0; i < BPL; i++) {
      const int j = r + i * L;
      float4 o = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      float kj = 1.0f;
      if (j < B) {
        const double Lh = tab.lnr_hi[mh.ic][j], Ll = tab.lnr_lo[mh.ic][j];
        double sed;
        if (MODE == MH_SED_POWERLAW) {
          sed = exp_scaled(idx0, Lh, Ll);
        } else {
          const double em1 = exp(zF * mv.band[j].nu_c) - 1.0;
          const double iem1 = mh_fast_rcp(em1);
          sed = erefF * iem1 * exp_scaled(idx0 + 1.0, Lh, Ll);
          kj = (float)(1.0 + iem1);
        }
        const double D0 = mh_data_value(mv, mh.ic, j, mh.plane[0], p);
        const double W0 = mh_fast_rcp(ldg_stream(mv.rms + plane_off(mv, j, mh.plane[0]) + p)), m0 = amp0 * sed;
        o.x = (float)((D0 - m0) * W0);
        o.z = (float)(m0 * W0);
        if (S > 1) {
          const double D1 = mh_data_value(mv, mh.ic, j, mh.plane[1], p);
          const double W1 = mh_fast_rcp(ldg_stream(mv.rms + plane_off(mv, j, mh.plane[1]) + p)), m1 = amp1 * sed;
          o.y = (float)((D1 - m1) * W1);
          o.w = (float)(m1 * W1);
        }
      }
      const size_t e = ((size_t)i * mv.P + p) * L + r;
      st4[e] = o;
      if (MODE == MH_SED_MBB_T) kjs[e] = kj;
    }
  }
}

// the screened chains.  out[0] = accepted proposals, out[1] = proposals decided by the fp64 fallback
template <int BPL, int MODE>
__global__ void __launch_bounds__(DG_MH_THREADS, 4)
k5_chain_kernel(const __grid_constant__ ModelView mv, const __grid_constant__ MhView mh, const float4 *st4,
                const float *kjs, double *partials, unsigned int *ticket, double *out) {
  constexpr int L = DG_MH_LANES;
  constexpr int PB = DG_MH_THREADS / L;
  __shared__ double smem[4 * 32];
  const int tid = threadIdx.x, r = tid % L, g = tid / L, B = mv.nbands, S = mh.S;
  const int nsample = mh.nsample;
  const unsigned full = 0xffffffffu;
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
  const CompView &cv = mv.comp[mh.ic];
  const double ln_denom = log(mh.gauss[1] * sqrt(2.0 * DG_PI));
  const double inv2var = 1.0 / (2 * (mh.gauss[1] * mh.gauss[1]));
  const float kappa = MODE == MH_SED_MBB_T ? DG_K5_KAPPA_T : DG_K5_KAPPA_BETA;
  float cf[BPL];
#pragma unroll
  for (int i = 0; i < BPL; i++) {
    const int j = r + i * L;
    if (MODE == MH_SED_MBB_T) cf[i] = j < B ? (float)(DG_H / DG_KB * mv.band[j].nu_c) : 0.0f;
    else cf[i] = j < B ? (float)mv.tab->lnr_hi[mh.ic][j] : 0.0f;
  }
  const float cref = (float)(DG_H / DG_KB * cv.nu_ref);

  const int64_t ngroups = (int64_t)gridDim.x * PB;
  const int64_t niter = (mv.P + ngroups - 1) / ngroups;
  for (int64_t itp = 0; itp < niter; itp++) {
    const int64_t p = itp * ngroups + (int64_t)blockIdx.x * PB + g;
    const bool valid = p < mv.P;
    const bool use = valid && mv.mask[p] != 0;
    if (!use && valid && r == 0)  // :362; index_map stays 0 for masked pixels (:223, :465, :483)
      for (int s = 0; s < S; s++) cv.idx[mh.nind][(size_t)mh.plane[s] * mv.Ppad + p] = 0.0;
    if (!__any_sync(full, use)) continue;
    const int64_t pp = use ? p : 0;
    const size_t kp0 = (size_t)mh.plane[0] * mv.Ppad + pp;
    const double idx0 = cv.nind > 0 ? cv.idx[0][kp0] : 0.0;  // :372-374
    const double idx1 = cv.nind > 1 ? cv.idx[1][kp0] : 0.0;
    double cur = mh.nind == 0 ? idx0 : idx1;
    float tr0[BPL], tr1[BPL], g0[BPL], g1[BPL], gs[BPL], kj[BPL];
    float kref = 1.0f;
#pragma unroll
    for (int i = 0; i < BPL; i++) {
      const size_t e = ((size_t)i * mv.P + pp) * L + r;
      const float4 o = use ? __ldg(st4 + e) : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      tr0[i] = o.x;
      tr1[i] = o.y;
      g0[i] = o.z;
      g1[i] = o.w;
      gs[i] = fabsf(o.z) + fabsf(o.w);
      kj[i] = (MODE == MH_SED_MBB_T && use) ? __ldg(kjs + e) : 1.0f;
    }
    if (MODE == MH_SED_MBB_T) kref = 1.0f + __frcp_rn(k5_em1f(cref * (float)mh_fast_rcp(cur)));
    auto prior_of = [&](double xe) -> double {
      if (mh.prior_type != 1) return 0.0;
      const double a = ((xe - mh.gauss[0]) * (xe - mh.gauss[0])) * inv2var;
      return a < 700.0 ? -a - ln_denom : log_normal_prior(xe, mh.gauss[0], mh.gauss[1]);
    };
    float tmax = 0.0f;
#pragma unroll
    for (int i = 0; i < BPL; i++) tmax = fmaxf(tmax, fmaxf(fabsf(tr0[i]), fabsf(tr1[i])));
    tmax = fmaxf(tmax, __shfl_xor_sync(full, tmax, 1));
    tmax = fmaxf(tmax, __shfl_xor_sync(full, tmax, 2));
    float dT = 1.2e-7f * tmax, kap = kappa;
    double prior_cur = prior_of(cur), naccept = 0.0, lnl_cur_x = 0.0;
    bool have_cur_x = false, need_tmax = false;
    for (int l = 0; l < nsample; l++) {
      const size_t slot = (size_t)l * mv.P + pp;
      const double x = cur + (0.0 + mh.step * __ldg(mh.z + slot));  // :414
      const bool oob = x < mh.uni[0] || x > mh.uni[1];               // :415, Q5
      float lam = 0.0f, A1 = 0.0f, A2 = 0.0f, n1 = 0.0f, w1 = 1.0f;
      float rho[BPL];
#pragma unroll
      for (int i = 0; i < BPL; i++) rho[i] = 0.0f;
      if (!oob) {
        float d;
        if (MODE == MH_SED_MBB_T) {
          d = (float)((cur - x) * mh_fast_rcp(x * cur));
          n1 = kref * k5_em1f(cref * d, w1);
        } else {
          d = (float)(x - cur);
        }
#pragma unroll
        for (int i = 0; i < BPL; i++) {
          float b, w2;
          if (MODE == MH_SED_MBB_T) {
            const float n2 = kj[i] * k5_em1f(cf[i] * d, w2);
            const float inv = __frcp_rn(1.0f + n2);
            rho[i] = (n1 - n2) * inv;
            b = fmaf(fabsf(n1), w1, fabsf(n2) * w2) * inv;
          } else {
            const float xx = d * cf[i];
            rho[i] = k5_em1f(xx, w2);
            b = fabsf(rho[i]) * w2 * (1.0f + fabsf(xx));
          }
          const float a0 = g0[i] * rho[i], a1 = g1[i] * rho[i];
          lam = fmaf(a0, fmaf(2.0f, tr0[i], -a0), lam);
          lam = fmaf(a1, fmaf(2.0f, tr1[i], -a1), lam);
          A1 = fmaf(gs[i], b, A1);
          A2 += fabsf(a0) + fabsf(a1);
        }
      }
      lam += __shfl_xor_sync(full, lam, 1);
      lam += __shfl_xor_sync(full, lam, 2);
      A1 += __shfl_xor_sync(full, A1, 1);
      A1 += __shfl_xor_sync(full, A1, 2);
      A2 += __shfl_xor_sync(full, A2, 1);
      A2 += __shfl_xor_sync(full, A2, 2);
      const float E = 2.0f * A1 * (tmax + A2);
      const double prior_new = oob ? prior_cur : prior_of(x);
      const double diff_s = 0.5 * (double)lam + (prior_new - prior_cur);
      const double uu = mh.ml_mode != 0 ? __ldg(mh.u + slot) : 1.0;
      float lu = 0.0f, eps_u = 0.0f;
      if (mh.ml_mode != 0) {
        lu = __logf((float)uu);
        eps_u = 1.5e-6f * (1.0f + fabsf(lu));
      }
      const float eps = kap * E + 2.0f * dT * A2 + 2.5e-7f * A2 * (tmax + A2) + eps_u + 1.0e-30f;
      const bool certain = fabs(diff_s - (double)lu) > (double)eps;
      bool accept = diff_s > (double)lu;
      const bool need = use && !oob && !certain;
      if (__any_sync(full, need)) {  // fp64 re-evaluation for the whole warp (shuffles stay convergent)
        const double amp0 = cv.amp[(size_t)mh.plane[0] * mv.Ppad + pp];
        const double amp1 = S > 1 ? cv.amp[(size_t)mh.plane[1] * mv.Ppad + pp] : 0.0;
        auto exact_lnl = [&](double xe) -> double {
          double part = k5_exact_part_global<BPL, MODE>(mv, mh, r, pp, xe, idx0, idx1, amp0, amp1);
          part += __shfl_xor_sync(full, part, 1);
          part += __shfl_xor_sync(full, part, 2);
          return part + prior_of(xe);
        };
        const double lnl_new = exact_lnl(oob ? cur : x);
        if (__any_sync(full, !have_cur_x)) {
          const double v = exact_lnl(cur);
          if (!have_cur_x) lnl_cur_x = v;
          have_cur_x = true;
        }
        const double diff = lnl_new - lnl_cur_x;
        const bool acc_x = (mh.ml_mode == 0) ? (diff > 0.0) : (diff > log(uu));
        if (need) {
          accept = acc_x;
          if (r == 0) acc[1] += 1.0;
        }
        if (accept && !oob) lnl_cur_x = lnl_new;
      } else if (accept && !oob) {
        have_cur_x = false;
      }
      if (oob) accept = false;
      if (accept) {
        cur = x;
        prior_cur = prior_new;
        naccept += 1.0;
        float iT = 0.0f;
        if (MODE == MH_SED_MBB_T) {
          iT = (float)mh_fast_rcp(cur);
          kref = 1.0f + __frcp_rn(k5_em1f(cref * iT));
        }
#pragma unroll
        for (int i = 0; i < BPL; i++) {
          const float a0 = g0[i] * rho[i], a1 = g1[i] * rho[i];
          tr0[i] -= a0;
          tr1[i] -= a1;
          g0[i] += a0;
          g1[i] += a1;
          gs[i] = fabsf(g0[i]) + fabsf(g1[i]);
          if (MODE == MH_SED_MBB_T && r + i * L < B) kj[i] = 1.0f + __frcp_rn(k5_em1f(cf[i] * iT));  // (padding: K = 1)
        }
        dT += kap * A1 + 1.2e-7f * (tmax + A2);
        kap += 1.5e-7f;
        need_tmax = true;
      }
      if (__any_sync(full, need_tmax)) {
        float m = 0.0f;
#pragma unroll
        for (int i = 0; i < BPL; i++) m = fmaxf(m, fmaxf(fabsf(tr0[i]), fabsf(tr1[i])));
        m = fmaxf(m, __shfl_xor_sync(full, m, 1));
        m = fmaxf(m, __shfl_xor_sync(full, m, 2));
        if (need_tmax) tmax = m;
        need_tmax = false;
      }
    }
    if (use && r == 0) {
      for (int s = 0; s < S; s++) cv.idx[mh.nind][(size_t)mh.plane[s] * mv.Ppad + p] = cur;  // :465, :483
      acc[0] += naccept;
    }
  }
  grid_reduce<4>(acc, smem, partials, ticket, out);
}
