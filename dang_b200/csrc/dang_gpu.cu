// dang_gpu.cu -- C ABI (include/dang_gpu.h) of the B200-native dang Gibbs hot path.
//
// One handle owns one GPU and one contiguous RING pixel range.  All work is enqueued on the
// handle's stream; cross-rank traffic is an NCCL all-gather of a few doubles followed by a
// rank-ordered sum on every rank (deterministic, identical bits everywhere).
// There is deliberately no CPU fallback: every error surfaces as a nonzero return code.
#include <algorithm>

#include "host.cuh"
#include "kernels_data.cuh"

thread_local std::string g_create_error;
NcclApi g_nccl;

void nccl_load() {
  if (g_nccl.lib) return;
  const char *names[] = {"libnccl.so.2", "libnccl.so"};
  for (const char *n : names) {
    g_nccl.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (g_nccl.lib) break;
  }
  if (!g_nccl.lib) fail(DANG_GPU_ENCCL, "cannot dlopen libnccl.so.2: %s", dlerror());
#define SYM(field, name)                                                          \
  *(void **)(&g_nccl.field) = dlsym(g_nccl.lib, name);                            \
  if (!g_nccl.field) fail(DANG_GPU_ENCCL, "libnccl lacks symbol %s", name)
  SYM(GetUniqueId, "ncclGetUniqueId");
  SYM(CommInitRank, "ncclCommInitRank");
  SYM(CommDestroy, "ncclCommDestroy");
  SYM(AllGather, "ncclAllGather");
  SYM(GetErrorString, "ncclGetErrorString");
#undef SYM
}
// static tables: flattened bandpasses, ln(nu/nu_ref) per (component, band [, bandpass sample])
// Gauss quadrature of a tabulated bandpass.  Every bandpass-integrated SED of the reference is a sum
// sum_i tau0_i g(nu0_i) (src/dang_component_mod.f90:909-914, 949-955, 990-996, 1030-1036) with g smooth in
// x = ln(nu / nu_c) over the few per cent a band spans.  The n-point Gauss rule of the discrete measure
// {x_i, tau0_i} -- nodes = eigenvalues of its Jacobi matrix (Lanczos on diag(x) started from sqrt(tau0)),
// weights = total weight x squared first eigenvector components -- integrates every polynomial in x up to
// degree 2n-1 exactly as the full table does, so the two sums differ by the 2n-th order Taylor remainder of g
// across the band.  That remainder is below rounding only while g varies slowly in ln nu: it is for power laws
// and mbb dust at the c3 bands, but not for 'cmb' above ~500 GHz (hnu/kT_CMB up to 15 at 857 GHz: 4e-8 with 8
// nodes over a half-width of 0.25) or for a narrow lognormal near nu_p (2e-6 at w = 0.1).  So upload_bandpasses
// accepts a rule for a band only after verifying it (verify_rule) and otherwise keeps the table.  With a rule
// the device sees n samples per band instead of n_bp (128 at config c3): 16x fewer transcendentals in every
// kernel that evaluates a bandpass-integrated SED.
// Returns false (table kept) if the band is too short, has negative weights, or the rule comes out badly.
static bool gauss_compress(const BandHost &b, int nq, std::vector<double> &nu_q, std::vector<double> &w_q) {
  std::vector<double> x, w;
  double W = 0.0;
  for (int i = 0; i < b.n; i++) {
    if (b.nu0[i] == 0.0) continue;  // skipped by the reference's sums (:911)
    if (b.tau0[i] < 0.0) return false;
    if (b.tau0[i] == 0.0) continue;
    x.push_back((double)logl((long double)b.nu0[i] / (long double)b.nu_c));
    w.push_back(b.tau0[i]);
    W += b.tau0[i];
  }
  const int m = (int)x.size();
  if (m <= 2 * nq || W <= 0.0) return false;
  // the error estimate assumes g varies on scales >~ 0.25 in ln(nu) across a band of half-width <= 0.25
  // (a 16th-order remainder ~ (4 x 0.25)^16 / 16! = 5e-14 for an SED as steep as nu^4); wider bands keep their table
  for (int i = 0; i < m; i++)
    if (fabs(x[i]) > 0.25) return false;
  // Lanczos with full re-orthogonalisation: J = tridiag(beta_k, alpha_k, beta_{k+1})
  std::vector<std::vector<long double>> q(nq, std::vector<long double>(m));
  std::vector<long double> alpha(nq), beta(nq, 0.0L);
  for (int i = 0; i < m; i++) q[0][i] = sqrtl((long double)w[i] / (long double)W);
  for (int k = 0; k < nq; k++) {
    std::vector<long double> v(m);
    long double a = 0.0L;
    for (int i = 0; i < m; i++) {
      v[i] = (long double)x[i] * q[k][i];
      a += q[k][i] * v[i];
    }
    alpha[k] = a;
    if (k + 1 == nq) break;
    for (int i = 0; i < m; i++) v[i] -= a * q[k][i] + (k > 0 ? beta[k] * q[k - 1][i] : 0.0L);
    for (int pass = 0; pass < 2; pass++)
      for (int kk = 0; kk <= k; kk++) {
        long double d = 0.0L;
        for (int i = 0; i < m; i++) d += q[kk][i] * v[i];
        for (int i = 0; i < m; i++) v[i] -= d * q[kk][i];
      }
    long double nrm = 0.0L;
    for (int i = 0; i < m; i++) nrm += v[i] * v[i];
    nrm = sqrtl(nrm);
    if (!(nrm > 1e-14L)) return false;  // the measure has fewer than nq + 1 effective points
    beta[k + 1] = nrm;
    for (int i = 0; i < m; i++) q[k + 1][i] = v[i] / nrm;
  }
  // eigen-decomposition of the nq x nq Jacobi matrix by cyclic Jacobi rotations
  std::vector<std::vector<long double>> A(nq, std::vector<long double>(nq, 0.0L)), V(nq, std::vector<long double>(nq, 0.0L));
  for (int k = 0; k < nq; k++) {
    A[k][k] = alpha[k];
    V[k][k] = 1.0L;
    if (k + 1 < nq) A[k][k + 1] = A[k + 1][k] = beta[k + 1];
  }
  for (int sweep = 0; sweep < 60; sweep++) {
    long double off = 0.0L;
    for (int p = 0; p < nq; p++)
      for (int r = p + 1; r < nq; r++) off += A[p][r] * A[p][r];
    if (off < 1e-40L) break;
    for (int p = 0; p < nq; p++)
      for (int r = p + 1; r < nq; r++) {
        if (fabsl(A[p][r]) < 1e-300L) continue;
        const long double th = (A[r][r] - A[p][p]) / (2.0L * A[p][r]);
        const long double t = (th >= 0 ? 1.0L : -1.0L) / (fabsl(th) + sqrtl(th * th + 1.0L));
        const long double c = 1.0L / sqrtl(t * t + 1.0L), sn = t * c;
        for (int k = 0; k < nq; k++) {
          const long double akp = A[k][p], akr = A[k][r];
          A[k][p] = c * akp - sn * akr;
          A[k][r] = sn * akp + c * akr;
        }
        for (int k = 0; k < nq; k++) {
          const long double apk = A[p][k], ark = A[r][k];
          A[p][k] = c * apk - sn * ark;
          A[r][k] = sn * apk + c * ark;
        }
        for (int k = 0; k < nq; k++) {
          const long double vkp = V[k][p], vkr = V[k][r];
          V[k][p] = c * vkp - sn * vkr;
          V[k][r] = sn * vkp + c * vkr;
        }
      }
  }
  nu_q.assign(nq, 0.0);
  w_q.assign(nq, 0.0);
  long double wsum = 0.0L;
  for (int k = 0; k < nq; k++) {
    const long double wk = V[0][k] * V[0][k] * (long double)W;
    if (!(wk > 0.0L)) return false;
    nu_q[k] = (double)((long double)b.nu_c * expl(A[k][k]));
    w_q[k] = (double)wk;
    wsum += wk;
  }
  return fabsl(wsum - (long double)W) <= 1e-12L * (long double)W;
}

// Verification of a band's rule.  The values of an index a kernel can evaluate an SED at: the range of the maps
// the host uploaded and, when the index is sampled, its uniform-prior box (the samplers never leave it).
static void index_box(const dang_gpu *h, const CompHost &c, int l, double box[2]) {
  box[0] = c.map_range[l][0];
  box[1] = c.map_range[l][1];
  if (c.index[l].sample_index) {
    box[0] = std::min(box[0], c.index[l].uni[0]);
    box[1] = std::max(box[1], c.index[l].uni[1]);
  }
}
// the T_CMB values the 'cmb' SED can see: the current one and every value a 'T_cmb' component can hand over
static void t_cmb_box(const dang_gpu *h, double box[2]) {
  box[0] = box[1] = h->T_cmb;
  for (int c = 0; c < h->ncomp; c++)
    if (h->comp[c].set && h->comp[c].type == DANG_COMP_T_CMB) {
      double b[2];
      index_box(h, h->comp[c], 0, b);
      box[0] = std::min(box[0], b[0]);
      box[1] = std::max(box[1], b[1]);
    }
}
// c%indices(:,:,l) as the host uploads it (full-sky [plane][pix], NULL: the constructor's 1.0): its range here
static void record_map_range(const dang_gpu *h, CompHost &c, int l, const double *indices) {
  double lo = 1.0, hi = 1.0;
  if (indices) {
    lo = INFINITY;
    hi = -INFINITY;
    for (int k = 0; k < h->nmaps; k++)
      for (int64_t p = h->lo; p < h->hi; p++) {
        const double v = indices[(size_t)k * h->npix + p];
        lo = std::min(lo, v);
        hi = std::max(hi, v);
      }
  }
  c.map_range[l][0] = lo;
  c.map_range[l][1] = hi;
}
// true while every index map and T_CMB stays inside the box the current rules were verified on
static bool rules_cover_params(const dang_gpu *h) {
  double box[2];
  for (int c = 0; c < h->ncomp; c++)
    for (int l = 0; h->comp[c].set && l < h->comp[c].nind; l++) {
      index_box(h, h->comp[c], l, box);
      if (!(box[0] >= h->comp[c].verified_box[l][0] && box[1] <= h->comp[c].verified_box[l][1])) return false;
    }
  t_cmb_box(h, box);
  return box[0] >= h->verified_T_cmb[0] && box[1] <= h->verified_T_cmb[1];
}
// A band's SED up to factors constant over the band, in long double: the bodies of sed_powerlaw ... sed_planck_rj
// (common.cuh), which restate evaluate_powerlaw ... evaluate_hi_fit of the reference.  hi_fit's template amplitude
// and T_cmb's / hi_fit's constants cancel in a relative comparison.
static long double sed_ld(int type, long double nu, long double nu_ref, long double t0, long double t1, long double T_cmb) {
  const long double H = (long double)DG_H, KB = (long double)DG_KB;
  switch (type) {
    case DANG_COMP_POWERLAW: return powl(nu / nu_ref, t0);
    case DANG_COMP_MBB: return powl(nu / nu_ref, t0 + 1.0L) / expm1l(H * nu / (KB * t1));
    case DANG_COMP_FREEFREE: {
      const long double g = logl(expl(5.960L - sqrtl(3.0L) / 3.141592653589793238462643383279502884L *
                                                  logl(nu / 1e9L * powl(t0 / 1e4L, -1.5L))) + 2.71828L);
      return g * (nu_ref / nu) * (nu_ref / nu);
    }
    case DANG_COMP_LOGNORMAL: {
      const long double t = logl(nu / (t0 * 1e9L)) / t1;
      return expl(-0.5L * t * t) * (nu_ref / nu) * (nu_ref / nu);
    }
    case DANG_COMP_CMB: {
      const long double y = (nu > 1e7L ? H * nu : H * nu * 1e9L) / (KB * T_cmb);
      return expm1l(y) * expm1l(y) / (y * y * expl(y));
    }
    default: return nu / expm1l(H * nu / (KB * t0));  // T_cmb, hi_fit: B_nu / RJ
  }
}
const int DG_VERIFY_POINTS = 7;  // per index dimension, box edges included
// One point at which a band's rule is verified: an SED type and its parameters, with the full table's sum there.
struct VerifyPoint {
  int type;
  long double nu_ref, t0, t1, full;
};
// The points for band b: for every component on the handle, a DG_VERIFY_POINTS grid over the box each of its indices
// can take (a single point where the box is), each with sum_i tau0_i g(nu0_i) over the whole table.
static std::vector<VerifyPoint> verify_points(const dang_gpu *h, const BandHost &b) {
  std::vector<VerifyPoint> pts;
  const int P = DG_VERIFY_POINTS;
  for (int c = 0; c < h->ncomp; c++) {
    const CompHost &cc = h->comp[c];
    if (!cc.set || cc.type == DANG_COMP_TEMPLATE || cc.type == DANG_COMP_MONOPOLE) continue;
    double box[2][2] = {{0.0, 0.0}, {0.0, 0.0}};  // 'cmb': box[0] is the T_CMB range
    if (cc.type == DANG_COMP_CMB) t_cmb_box(h, box[0]);
    for (int l = 0; l < cc.nind; l++) index_box(h, cc, l, box[l]);
    const int n0 = box[0][1] > box[0][0] ? P : 1, n1 = box[1][1] > box[1][0] ? P : 1;
    for (int a = 0; a < n0; a++)
      for (int e = 0; e < n1; e++) {
        VerifyPoint v;
        v.type = cc.type;
        v.nu_ref = cc.nu_ref;
        v.t0 = box[0][0] + (box[0][1] - box[0][0]) * (long double)a / (P - 1);
        v.t1 = box[1][0] + (box[1][1] - box[1][0]) * (long double)e / (P - 1);
        v.full = 0.0L;
        for (int i = 0; i < b.n; i++)
          if (b.nu0[i] != 0.0) v.full += (long double)b.tau0[i] * sed_ld(v.type, b.nu0[i], v.nu_ref, v.t0, v.t1, v.t0);
        pts.push_back(v);
      }
  }
  return pts;
}
// Does the rule (nu_q, w_q) reproduce the table's sum to 1e-14 relative at every point?
static bool verify_rule(const std::vector<VerifyPoint> &pts, const std::vector<double> &nu_q,
                        const std::vector<double> &w_q) {
  for (const VerifyPoint &v : pts) {
    long double q = 0.0L;
    for (size_t k = 0; k < nu_q.size(); k++) q += (long double)w_q[k] * sed_ld(v.type, nu_q[k], v.nu_ref, v.t0, v.t1, v.t0);
    if (!(fabsl(q - v.full) <= 1e-14L * fabsl(v.full))) return false;
  }
  return true;
}

void upload_bandpasses(dang_gpu *h) {
  if (!h->bp_dirty) return;
  std::vector<double> nu0, tau0;
  for (int j = 0; j < h->nbands; j++) {
    BandHost &b = h->band[j];
    b.n_dev = b.n;
    b.nu0_dev = b.nu0;
    b.tau0_dev = b.tau0;
    // the smallest rule (bp_quad, then 4 nodes more at a time, up to n_bp / 2) that verify_rule accepts
    std::vector<VerifyPoint> pts;
    if (h->bp_quad > 0 && 2 * h->bp_quad <= b.n) pts = verify_points(h, b);
    for (int nq = h->bp_quad; nq > 0 && 2 * nq <= b.n; nq += 4) {
      std::vector<double> nq_nu, nq_w;
      if (!gauss_compress(b, nq, nq_nu, nq_w)) break;
      if (verify_rule(pts, nq_nu, nq_w)) {
        b.n_dev = nq;
        b.nu0_dev = nq_nu;
        b.tau0_dev = nq_w;
        break;
      }
    }
    nu0.insert(nu0.end(), b.nu0_dev.begin(), b.nu0_dev.end());
    tau0.insert(tau0.end(), b.tau0_dev.begin(), b.tau0_dev.end());
  }
  for (int c = 0; c < h->ncomp; c++)
    for (int l = 0; h->comp[c].set && l < h->comp[c].nind; l++) index_box(h, h->comp[c], l, h->comp[c].verified_box[l]);
  t_cmb_box(h, h->verified_T_cmb);
  dfree(h->bp_nu0); dfree(h->bp_tau0); dfree(h->bp_lnr_hi); dfree(h->bp_lnr_lo);
  h->nbp = (int)nu0.size();
  std::vector<double> lhi((size_t)h->ncomp * h->nbp + 1), llo((size_t)h->ncomp * h->nbp + 1);
  std::vector<double> thi(DG_MAX_COMPS * DG_MAX_BANDS, 0.0), tlo(DG_MAX_COMPS * DG_MAX_BANDS, 0.0);
  for (int c = 0; c < h->ncomp; c++) {
    if (!h->comp[c].set) continue;
    for (int j = 0; j < h->nbands; j++)
      if (h->band[j].set) dd_log_ratio(h->band[j].nu_c, h->comp[c].nu_ref, thi[c * DG_MAX_BANDS + j], tlo[c * DG_MAX_BANDS + j]);
    for (int i = 0; i < h->nbp; i++)
      if (nu0[i] != 0.0) dd_log_ratio(nu0[i], h->comp[c].nu_ref, lhi[(size_t)c * h->nbp + i], llo[(size_t)c * h->nbp + i]);
  }
  if (h->nbp) {
    CK(cudaMalloc(&h->bp_nu0, nu0.size() * sizeof(double)));
    CK(cudaMalloc(&h->bp_tau0, tau0.size() * sizeof(double)));
    CK(cudaMalloc(&h->bp_lnr_hi, lhi.size() * sizeof(double)));
    CK(cudaMalloc(&h->bp_lnr_lo, llo.size() * sizeof(double)));
    CK(cudaMemcpyAsync(h->bp_nu0, nu0.data(), nu0.size() * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->bp_tau0, tau0.data(), tau0.size() * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->bp_lnr_hi, lhi.data(), lhi.size() * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->bp_lnr_lo, llo.data(), llo.size() * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  }
  CK(cudaMemcpyAsync((char *)h->tab + offsetof(SedTable, lnr_hi), thi.data(), sizeof(double) * thi.size(),
                     cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync((char *)h->tab + offsetof(SedTable, lnr_lo), tlo.data(), sizeof(double) * tlo.size(),
                     cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));  // the host vectors go out of scope
  h->bp_dirty = false;
  h->tab_dirty = true;
}

ModelView model_view(dang_gpu *h) {
  if (!h->maps_set) fail(DANG_GPU_ESTATE, "dang_gpu_upload_maps has not been called");
  upload_bandpasses(h);
  ModelView mv;
  memset(&mv, 0, sizeof mv);
  mv.nbands = h->nbands;
  mv.ncomp = h->ncomp;
  mv.nmaps = h->nmaps;
  mv.P = h->P;
  mv.Ppad = h->Ppad;
  mv.pix_lo = h->lo;
  mv.npix = h->npix;
  int off = 0;
  for (int j = 0; j < h->nbands; j++) {
    if (!h->band[j].set) fail(DANG_GPU_ESTATE, "band %d has not been set", j);
    mv.band[j].nu_c = h->band[j].nu_c;
    mv.band[j].n = h->band[j].n_dev;
    mv.band[j].off = off;
    off += h->band[j].n_dev;
    mv.gain[j] = h->gain[j];
    mv.offset[j] = h->offset[j];
  }
  mv.T_cmb = h->T_cmb;
  for (int c = 0; c < h->ncomp; c++) {
    if (!h->comp[c].set) fail(DANG_GPU_ESTATE, "component %d has not been set", c);
    mv.comp[c].type = h->comp[c].type;
    mv.comp[c].nind = h->comp[c].nind;
    mv.comp[c].nu_ref = h->comp[c].nu_ref;
    mv.comp[c].amp = h->comp[c].amp;
    for (int l = 0; l < DG_MAXIND; l++) mv.comp[c].idx[l] = h->comp[c].idx[l];
    mv.comp[c].tamp = h->comp[c].is_template ? h->comp[c].tamp : nullptr;  // template / monopole / hi_fit
    mv.comp[c].in_sky = h->comp[c].type == DANG_COMP_MONOPOLE ? 0 : 1;
  }
  mv.bp_nu0 = h->bp_nu0;
  mv.bp_tau0 = h->bp_tau0;
  mv.bp_lnr_hi = h->bp_lnr_hi;
  mv.bp_lnr_lo = h->bp_lnr_lo;
  mv.nbp = h->nbp;
  mv.tab = h->tab;
  mv.sig = h->sig;
  mv.rms = h->rms;
  mv.mask = h->mask;
  if (h->tab_dirty) {  // an index map changed since the SED tables were built
    idx_changed(h);    // (whatever left the device for the next full-sky chain is stale now)
    const bool scanned = h->check_mask != 0;
    if (h->check_mask) {
      // maps uploaded by the host are scanned once; maps written by the samplers are not (their
      // uniformity is known by construction and was recorded by set_nonuni)
      const int nmap = h->ncomp * 3 * DG_MAXIND;
      for (int m = 0; m < nmap; m++)
        if ((h->check_mask >> m) & 1ull)
          CK(cudaMemsetAsync((char *)h->tab + offsetof(SedTable, nonuni) + m * sizeof(int), 0, sizeof(int), h->stream));
      KTimer kt(h, DANG_K_SCALAR, 0);
      dim3 grid(grid_for(h, h->P, DG_THREADS, 1), nmap);
      uniform_check_kernel<<<grid, DG_THREADS, 0, h->stream>>>(mv, h->tab, h->check_mask);
      kt.done();
      h->check_mask = 0;
    }
    KTimer kt(h, DANG_K_SCALAR, 0);
    sed_table_kernel<<<h->ncomp * 3, 32, 0, h->stream>>>(mv, h->tab);
    kt.done();
    // the host picks the streaming (tabulated-SED) kernel variants from these flags; they are read
    // back only after a scan, otherwise the host mirror (kept by set_nonuni) already has them
    if (scanned) {
      int *hu = (int *)((char *)h->pinned + 32 * 1024);
      readback(h, hu, (char *)h->tab + offsetof(SedTable, nonuni), sizeof(h->nonuni_host));
      CK(cudaStreamSynchronize(h->stream));
      memcpy(h->nonuni_host, hu, sizeof(h->nonuni_host));
    }
    for (int c = 0; c < DG_MAX_COMPS; c++)
      for (int k = 0; k < 3; k++) {
        bool uni = c < h->ncomp && k < h->nmaps;
        for (int l = 0; uni && l < h->comp[c].nind; l++) uni = h->nonuni_host[c * 3 + k][l] == 0;
        h->uni_host[c * 3 + k] = uni ? 1 : 0;
      }
    h->tab_dirty = false;
  }
  return mv;
}

// exchange `cnt` doubles of sums_local between ranks; result in h->gathered as [rank][cnt]
void gather(dang_gpu *h, int cnt) {
  if (cnt > GATHER_MAX) fail(DANG_GPU_EINVAL, "gather of %d doubles exceeds %d", cnt, GATHER_MAX);
  if (h->nranks == 1) {
    return;  // h->gathered aliases h->sums_local (set in create / comm_init)
  } else if (h->use_mail) {
    peer_exchange_kernel<<<1, 32, 0, h->stream>>>(h->peer, h->sums_local, cnt, h->gathered);
    CK(cudaGetLastError());
  } else {
    NCK(g_nccl.AllGather(h->sums_local, h->gathered, cnt, NCCL_DOUBLE, h->comm, h->stream));
  }
}
// update_sky_model's side effect for a monopole component (src/dang_data_mod.f90:357-361): ddata%offset takes the
// band monopoles, template_amplitudes(:, 1).  The reference runs update_sky_model after every draw, so the offsets
// always equal the current monopole amplitudes; the library keeps that invariant wherever they change.
void monopole_to_offset(dang_gpu *h, const CompHost &c) {
  if (c.type != DANG_COMP_MONOPOLE) return;
  for (int j = 0; j < h->nbands; j++) h->offset[j] = c.tamp_host[0][j];
}

// template_amplitudes host mirror -> device table; the tabulated "SEDs" must be rebuilt
void upload_tamp(dang_gpu *h, CompHost &c) {
  if (!c.tamp) CK(cudaMalloc(&c.tamp, sizeof c.tamp_host));
  // pageable source: the copy is staged before the call returns, so the mirror may change right after
  CK(cudaMemcpyAsync(c.tamp, c.tamp_host, sizeof c.tamp_host, cudaMemcpyHostToDevice, h->stream));
  h->tab_dirty = true;
}

// unmasked pixels over all ranks (compute_chisq's count, src/dang_data_mod.f90:153-161); counted once per
// upload, the chi-square kernels refresh it as a by-product
int64_t unmasked_count(dang_gpu *h) {
  if (h->n_unmasked >= 0) return h->n_unmasked;
  if (!h->maps_set) fail(DANG_GPU_ESTATE, "dang_gpu_upload_maps has not been called");
  const int grid = grid_for(h, h->P, DG_THREADS, 4);
  KTimer kt(h, DANG_K_SCALAR, 0);
  masked_sum_kernel<<<grid, DG_THREADS, 0, h->stream>>>(h->sig, h->mask, h->P, h->partials, h->tickets, h->sums_local);
  kt.done();
  gather(h, 4);
  double *hp = (double *)h->pinned;
  readback(h, hp, h->gathered, (size_t)h->nranks * 4 * sizeof(double));
  CK(cudaStreamSynchronize(h->stream));
  double n = 0;
  for (int g = 0; g < h->nranks; g++) n += hp[g * 4 + 1];
  h->n_unmasked = (int64_t)(n + 0.5);
  return h->n_unmasked;
}

// ---------------------------------------------------------------- C ABI
#define API_BEGIN                                   \
  if (!h) return DANG_GPU_EINVAL;                   \
  try {                                             \
    set_device(h);
#define API_END_OK                                  \
    if (h->peer_error_host && *h->peer_error_host)  \
      fail(DANG_GPU_ENCCL, "a peer rank did not answer a scalar exchange within the timeout; results of this handle are poisoned"); \
    return DANG_GPU_OK;
#define API_END                                     \
    if (h->peer_error_host && *h->peer_error_host)  \
      fail(DANG_GPU_ENCCL, "a peer rank did not answer a scalar exchange within the timeout; results of this handle are poisoned"); \
    return DANG_GPU_OK;                             \
  } catch (const DgError &e) {                      \
    h->err = e.what();                              \
    return e.code;                                  \
  } catch (const std::exception &e) {               \
    h->err = e.what();                              \
    return DANG_GPU_ECUDA;                          \
  }

extern "C" {

const char *dang_gpu_last_error(const dang_gpu_t *h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int dang_gpu_create(int device, int nside, int64_t npix, int nmaps, int nbands, int ncomp,
                    int64_t pix_lo, int64_t pix_hi, dang_gpu_t **out) {
  if (!out) return DANG_GPU_EINVAL;
  *out = nullptr;
  dang_gpu *h = nullptr;
  try {
    if (npix != 12LL * nside * nside) fail(DANG_GPU_EINVAL, "npix %lld /= 12*nside^2", (long long)npix);
    if (nmaps < 1 || nmaps > 3) fail(DANG_GPU_EINVAL, "nmaps = %d", nmaps);
    if (nbands < 1 || nbands > DG_MAX_BANDS) fail(DANG_GPU_EINVAL, "nbands = %d (max %d)", nbands, DG_MAX_BANDS);
    if (ncomp < 1 || ncomp > DG_MAX_COMPS) fail(DANG_GPU_EINVAL, "ncomp = %d (max %d)", ncomp, DG_MAX_COMPS);
    if (pix_lo < 0 || pix_hi > npix || pix_lo >= pix_hi) fail(DANG_GPU_EINVAL, "bad pixel range [%lld,%lld)", (long long)pix_lo, (long long)pix_hi);
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
      fail(DANG_GPU_ECUDA, "no CUDA device available (%s); this library has no CPU fallback",
           e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (device < 0 || device >= ndev) fail(DANG_GPU_EINVAL, "device %d of %d", device, ndev);
    h = new dang_gpu();
    h->device = device;
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    h->num_sms = prop.multiProcessorCount;
    h->l2_persist_max = (size_t)prop.persistingL2CacheMaxSize;
    h->l2_window_max = (size_t)prop.accessPolicyMaxWindowSize;

    h->nside = nside;
    h->npix = npix;
    h->nmaps = nmaps;
    h->nbands = nbands;
    h->ncomp = ncomp;
    h->lo = pix_lo;
    h->hi = pix_hi;
    h->P = pix_hi - pix_lo;
    h->Ppad = (h->P + 63) / 64 * 64;
    for (int j = 0; j < DG_MAX_BANDS; j++) {
      h->gain[j] = 1.0;  // dang_data_mod.f90:127-128
      h->offset[j] = 0.0;
    }
    CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&h->d2h_stream, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&h->h2d_stream, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&h->ev_compute, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&h->ev_idx_dl, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&h->ev_sync, cudaEventDisableTiming));
    for (int i = 0; i < 2; i++) {
      CK(cudaEventCreateWithFlags(&h->ev_eta[i], cudaEventDisableTiming));
      CK(cudaEventCreateWithFlags(&h->ev_eta_used[i], cudaEventDisableTiming));
    }
    h->grid_cap = h->num_sms * 8;
    CK(cudaMalloc(&h->partials, (size_t)h->grid_cap * GATHER_MAX * sizeof(double)));
    CK(cudaMalloc(&h->tickets, 32 * sizeof(unsigned int)));
    CK(cudaMemset(h->tickets, 0, 32 * sizeof(unsigned int)));
    CK(cudaMalloc(&h->sums_local, GATHER_MAX * sizeof(double)));
    CK(cudaMalloc(&h->gathered_buf, (size_t)GATHER_MAX * 64 * sizeof(double)));
    h->gathered = h->sums_local;  // single rank: no exchange
    CK(cudaMalloc(&h->cg_scalars, sizeof(CgScalars)));
    CK(cudaMalloc(&h->mh_scalars, sizeof(MhScalars)));
    CK(cudaMalloc(&h->tab, sizeof(SedTable)));
    CK(cudaMemset(h->tab, 0, sizeof(SedTable)));
    CK(cudaMallocHost(&h->pinned, 256 * 1024));
    CK(cudaMallocHost(&h->snap, DG_SNAP_SLOTS * DG_SNAP_BYTES));
    for (int i = 0; i < DG_SNAP_SLOTS; i++) CK(cudaEventCreateWithFlags(&h->snap_meta[i].ev, cudaEventDisableTiming));
    {
      const int never = 0x7fffffff;  // no solve has run: x is carried on checkpoint passes only
      CK(cudaMemset(h->cg_scalars, 0, sizeof(CgScalars)));
      CK(cudaMemcpy(&h->cg_scalars->k_pred, &never, sizeof never, cudaMemcpyHostToDevice));
    }
    h->peer.nranks = 1;
    h->peer.rank = 0;
    for (int i = 0; i < 16; i++) CK(cudaEventCreate(&h->ev[i]));
    *out = h;
    return DANG_GPU_OK;
  } catch (const DgError &e) {
    g_create_error = e.what();
    if (h) dang_gpu_destroy(h);  // releases whatever streams, events and buffers were created so far
    return e.code;
  } catch (const std::exception &e) {
    g_create_error = e.what();
    if (h) dang_gpu_destroy(h);
    return DANG_GPU_ECUDA;
  }
}

int dang_gpu_destroy(dang_gpu_t *h) {
  if (!h) return DANG_GPU_EINVAL;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  post_release(h);
  if (h->comm) g_nccl.CommDestroy(h->comm);
  for (int g = 0; g < DG_MAX_RANKS; g++)
    if (h->peer_ptr[g] && g != h->rank) cudaIpcCloseMemHandle(h->peer_ptr[g]);
  if (h->peer.seq) cudaFree(h->peer.seq);
  if (h->peer_error_host) cudaFreeHost((void *)h->peer_error_host);
  if (h->mailbox) cudaFree(h->mailbox);
  if (!h->maps_borrowed) { dfree(h->sig); dfree(h->rms); dfree(h->mask); }
  dfree(h->bp_nu0); dfree(h->bp_tau0);
  for (auto &c : h->comp) {
    dfree(c.amp); dfree(c.amp_alt); dfree(c.idx[0]); dfree(c.idx[1]); dfree(c.tamp);
    if (c.ev_read) cudaEventDestroy(c.ev_read);
    if (c.ev_read_alt) cudaEventDestroy(c.ev_read_alt);
  }
  for (auto &g : h->cg) for (auto &x : g.x) dfree(x);
  dfree(h->M); dfree(h->r); dfree(h->d); dfree(h->eta); dfree(h->D); dfree(h->zbuf); dfree(h->ubuf);
  dfree(h->decisions); dfree(h->lnl_trace); dfree(h->stage); dfree(h->partials); dfree(h->tickets);
  dfree(h->sums_local); dfree(h->gathered_buf); dfree(h->cg_scalars); dfree(h->mh_scalars); dfree(h->tab);
  dfree(h->bp_lnr_hi); dfree(h->bp_lnr_lo); dfree(h->stat_buf); dfree(h->k5_kj); if (h->k5_st4) cudaFree(h->k5_st4); dfree(h->tb); dfree(h->tq); dfree(h->tmpl_scalars);
  if (h->pinned) cudaFreeHost(h->pinned);
  if (h->snap) cudaFreeHost(h->snap);
  for (int i = 0; i < DG_SNAP_SLOTS; i++)
    if (h->snap_meta[i].ev) cudaEventDestroy(h->snap_meta[i].ev);
  for (auto &k : h->kstat) for (auto &p : k.pending) { cudaEventDestroy(p.first); cudaEventDestroy(p.second); }
  for (auto &e : h->ev) if (e) cudaEventDestroy(e);
  if (h->d2h_stream) cudaStreamSynchronize(h->d2h_stream);
  if (h->h2d_stream) cudaStreamSynchronize(h->h2d_stream);
  dfree(h->eta_stage[0]); dfree(h->eta_stage[1]);
  for (cudaEvent_t e : {h->ev_compute, h->ev_idx_dl, h->ev_sync, h->ev_eta[0], h->ev_eta[1], h->ev_eta_used[0], h->ev_eta_used[1]}) if (e) cudaEventDestroy(e);
  for (cudaStream_t st : {h->d2h_stream, h->h2d_stream, h->stream}) if (st) cudaStreamDestroy(st);
  delete h;
  return DANG_GPU_OK;
}

int dang_gpu_set_option(dang_gpu_t *h, int option, double value) {
  API_BEGIN
  switch (option) {
    case DANG_OPT_FIX_SAMPLE_VECTOR: h->fix_q1 = value != 0; break;
    case DANG_OPT_CG_TWO_PASS: h->cg_two_pass = value != 0; break;
    case DANG_OPT_FULLSKY_STREAM: h->fullsky_stream = value != 0; break;
    case DANG_OPT_PROFILE:
      h->profile = value != 0;
      if (h->profile) {  // (re)start the event log here
        resolve_stats(h);
        h->tl.clear();
        if (!h->tl_base) CK(cudaEventCreate(&h->tl_base));
        CK(cudaEventRecord(h->tl_base, h->stream));
      }
      break;
    case DANG_OPT_CG_CHUNK: h->cg_chunk = value < 1 ? 1 : (int)value; break;
    case DANG_OPT_RECORD_DECISIONS: h->record = value != 0; break;
    case DANG_OPT_PERPIXEL_SERIAL: h->perpixel_serial = value != 0; break;
    case DANG_OPT_PERPIXEL_FAST: h->pp_fast = value != 0; h->pp_split = value == 2; h->pp_pix = value == 3; break;
    case DANG_OPT_TMA: h->use_tma = value != 0; break;
    case DANG_OPT_L2_PERSIST_MB: {
      // the set-aside shrinks the L2 every other kernel sees, so it exists only while the option is on
      h->l2_persist_mb = value < 0 ? 0 : (int)value;
      size_t want = (size_t)h->l2_persist_mb << 20;
      if (want > h->l2_persist_max) want = h->l2_persist_max;
      CK(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want));
      if (getenv("DANG_GPU_VERBOSE"))
        fprintf(stderr, "dang_gpu: persisting L2 %zu MB (max %zu MB, window max %zu MB)\n", want >> 20,
                h->l2_persist_max >> 20, h->l2_window_max >> 20);
      break;
    }
    case DANG_OPT_PERPIXEL_BP_SERIES: h->pp_bp_series = value != 0; break;
    case DANG_OPT_CG_PERSISTENT: h->cg_persistent = value != 0; break;
    case DANG_OPT_STREAM_RING: h->stream_ring = value != 0; break;
    case DANG_OPT_DEFER_D2H: h->defer_d2h = value != 0; break;
    case DANG_OPT_DEFER_SCALARS:
      if (h->pend_cg || h->pend_chisq_cg || h->pend_draw)
        fail(DANG_GPU_ESTATE, "results are pending: call dang_gpu_iteration_mark / dang_gpu_iteration_scalars before changing DANG_OPT_DEFER_SCALARS");
      h->defer_scalars = value != 0;
      break;
    case DANG_OPT_BP_QUADRATURE:
      h->bp_quad = value < 0 ? 0 : (value > 32 ? 32 : (int)value);
      h->bp_dirty = true;
      touch(h);
      break;
    case DANG_OPT_STAT_CACHE: h->stat_cache = value != 0; h->stat_valid = false; h->chisq_valid = false; break;
    case DANG_OPT_CG_CHECKPOINT:
      h->cg_ckpt = value < 0 ? 0 : (value > DG_CG_MAXM ? DG_CG_MAXM : (int)value);
      break;
    default: fail(DANG_GPU_EINVAL, "unknown option %d", option);
  }
  API_END
}

int dang_gpu_sync(dang_gpu_t *h) {
  API_BEGIN
  CK(cudaStreamSynchronize(h->stream));
  API_END
}

int dang_gpu_comm_unique_id(char id[128]) {
  try {
    nccl_load();
    nccl_uid_t uid;
    NCK(g_nccl.GetUniqueId(&uid));
    memcpy(id, uid.internal, 128);
    return DANG_GPU_OK;
  } catch (const DgError &e) {
    g_create_error = e.what();
    return e.code;
  }
}

int dang_gpu_comm_init(dang_gpu_t *h, int nranks, int rank, const char id[128]) {
  API_BEGIN
  // every gather buffer (gathered_buf, stat_buf, the pinned read-back area) is sized for DG_MAX_RANKS rows
  if (nranks < 1 || nranks > DG_MAX_RANKS || rank < 0 || rank >= nranks)
    fail(DANG_GPU_EINVAL, "bad rank %d of %d (at most %d ranks)", rank, nranks, DG_MAX_RANKS);
  h->nranks = nranks;
  h->rank = rank;
  h->n_unmasked = -1;
  touch(h);
  h->gathered = nranks > 1 ? h->gathered_buf : h->sums_local;
  if (nranks > 1) {
    nccl_load();
    nccl_uid_t uid;
    memcpy(uid.internal, id, 128);
    NCK(g_nccl.CommInitRank(&h->comm, nranks, uid, rank));
  }
  API_END
}

int dang_gpu_comm_ipc_handle(dang_gpu_t *h, char handle[64]) {
  API_BEGIN
  if (h->nranks < 2) fail(DANG_GPU_ESTATE, "dang_gpu_comm_init with nranks > 1 comes first");
  if (h->nranks > DG_MAX_RANKS) fail(DANG_GPU_EUNSUPPORTED, "mailboxes support up to %d ranks", DG_MAX_RANKS);
  if (!h->mailbox) {
    const size_t n = (size_t)DG_MAIL_SLOTS * h->nranks * sizeof(Mail);
    CK(cudaMalloc(&h->mailbox, n));
    CK(cudaMemset(h->mailbox, 0, n));
    CK(cudaMalloc(&h->peer.seq, sizeof(unsigned long long)));
    CK(cudaMemset(h->peer.seq, 0, sizeof(unsigned long long)));
    // the timeout flag lives in mapped pinned host memory: the kernels set it, every API call checks it
    int *eh = nullptr;
    CK(cudaHostAlloc((void **)&eh, sizeof(int), cudaHostAllocMapped));
    *eh = 0;
    h->peer_error_host = eh;
    CK(cudaHostGetDevicePointer((void **)&h->peer.error, eh, 0));
    {
      int khz = 0;
      CK(cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, h->device));
      const char *ts = getenv("DANG_GPU_PEER_TIMEOUT_S");
      double secs = ts ? atof(ts) : 30.0;
      if (!(secs > 0)) secs = 30.0;
      h->peer.timeout_cycles = (long long)(secs * 1e3 * (double)khz);
    }
    CK(cudaDeviceSynchronize());
  }
  cudaIpcMemHandle_t ih;
  CK(cudaIpcGetMemHandle(&ih, h->mailbox));
  static_assert(sizeof(ih) == 64, "cudaIpcMemHandle_t is 64 bytes");
  memcpy(handle, &ih, 64);
  API_END
}

int dang_gpu_comm_open_peers(dang_gpu_t *h, const char *handles) {
  API_BEGIN
  if (!h->mailbox || !handles) fail(DANG_GPU_ESTATE, "dang_gpu_comm_ipc_handle comes first");
  for (int g = 0; g < h->nranks; g++) {
    if (g == h->rank) {
      h->peer_ptr[g] = h->mailbox;
    } else {
      cudaIpcMemHandle_t ih;
      memcpy(&ih, handles + (size_t)g * 64, 64);
      CK(cudaIpcOpenMemHandle(&h->peer_ptr[g], ih, cudaIpcMemLazyEnablePeerAccess));
    }
    h->peer.box[g] = (Mail *)h->peer_ptr[g];
  }
  h->peer.nranks = h->nranks;
  h->peer.rank = h->rank;
  h->use_mail = true;
  API_END
}

int dang_gpu_comm_check(dang_gpu_t *h) {
  API_BEGIN
  if (h->use_mail) CK(cudaStreamSynchronize(h->stream));  // API_END reads the (host-mapped) timeout flag
  API_END
}

int dang_gpu_comm_probe(dang_gpu_t *h, int reps, int cnt, double *us_per_exchange) {
  API_BEGIN
  if (!h->use_mail) fail(DANG_GPU_ESTATE, "dang_gpu_comm_open_peers comes first");
  if (reps < 1 || cnt < 1 || cnt > 32) fail(DANG_GPU_EINVAL, "comm_probe: reps %d, cnt %d", reps, cnt);
  cudaEvent_t a, b;
  CK(cudaEventCreate(&a));
  CK(cudaEventCreate(&b));
  peer_exchange_probe_kernel<<<1, 32, 0, h->stream>>>(h->peer, h->sums_local, cnt, h->gathered, 8);  // warm-up, aligns the ranks
  CK(cudaEventRecord(a, h->stream));
  peer_exchange_probe_kernel<<<1, 32, 0, h->stream>>>(h->peer, h->sums_local, cnt, h->gathered, reps);
  CK(cudaEventRecord(b, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, a, b));
  cudaEventDestroy(a);
  cudaEventDestroy(b);
  if (us_per_exchange) *us_per_exchange = 1e3 * ms / reps;
  API_END
}

int dang_gpu_set_band(dang_gpu_t *h, int band, double nu_c_hz, int n_bp, const double *nu0_hz,
                      const double *tau0) {
  API_BEGIN
  if (band < 0 || band >= h->nbands) fail(DANG_GPU_EINVAL, "band %d of %d", band, h->nbands);
  if (n_bp < 0 || (n_bp > 0 && (!nu0_hz || !tau0))) fail(DANG_GPU_EINVAL, "bad bandpass table for band %d", band);
  BandHost &b = h->band[band];
  b.set = true;
  b.nu_c = nu_c_hz;
  b.n = n_bp;
  b.nu0.assign(nu0_hz, nu0_hz + n_bp);
  b.tau0.assign(tau0, tau0 + n_bp);
  h->bp_dirty = true;
  touch(h);  // every SED changes: cached statistics / chi-squares are stale
  API_END
}

int dang_gpu_set_gain_offset(dang_gpu_t *h, const double *gain, const double *offset) {
  API_BEGIN
  for (int j = 0; j < h->nbands; j++) {
    if (gain) h->gain[j] = gain[j];
    if (offset) h->offset[j] = offset[j];
  }
  touch(h);
  API_END
}

int dang_gpu_upload_maps(dang_gpu_t *h, const double *sig_map, const double *rms_map,
                         const double *mask, const double *gain, const double *offset) {
  API_BEGIN
  if (!sig_map || !rms_map || !mask) fail(DANG_GPU_EINVAL, "null map pointer");
  if (h->maps_borrowed) fail(DANG_GPU_ESTATE, "this handle borrows its maps (dang_gpu_share_maps): upload through the owner");
  const size_t n3 = (size_t)h->nbands * h->nmaps * h->Ppad;
  if (!h->sig) {
    CK(cudaMalloc(&h->sig, n3 * sizeof(double)));
    CK(cudaMalloc(&h->rms, n3 * sizeof(double)));
    CK(cudaMalloc(&h->mask, h->Ppad));
    CK(cudaMemsetAsync(h->sig, 0, n3 * sizeof(double), h->stream));
    // padding lanes of rms hold 1 so that nothing divides by zero there
    fill_kernel<<<h->num_sms * 4, DG_THREADS, 0, h->stream>>>(h->rms, (int64_t)n3, 1.0);
    CK(cudaGetLastError());
  }
  h2d_planes(h, h->sig, sig_map, h->nbands * h->nmaps);
  h2d_planes(h, h->rms, rms_map, h->nbands * h->nmaps);
  ensure(h->stage, h->stage_len, (size_t)h->Ppad);
  CK(cudaMemcpyAsync(h->stage, mask + h->lo, h->P * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  mask_to_bytes_kernel<<<h->num_sms * 4, DG_THREADS, 0, h->stream>>>(h->stage, h->mask, h->P, h->Ppad);
  CK(cudaGetLastError());
  for (int j = 0; j < h->nbands; j++) {
    if (gain) h->gain[j] = gain[j];
    if (offset) h->offset[j] = offset[j];
  }
  CK(cudaStreamSynchronize(h->stream));
  h->maps_set = true;
  h->n_unmasked = -1;
  touch(h);
  API_END
}

int dang_gpu_share_maps(dang_gpu_t *h, dang_gpu_t *src) {
  API_BEGIN
  if (!src || !src->maps_set) fail(DANG_GPU_ESTATE, "the source handle has no maps");
  if (src->device != h->device || src->npix != h->npix || src->nmaps != h->nmaps || src->nbands != h->nbands ||
      src->lo != h->lo || src->hi != h->hi)
    fail(DANG_GPU_EINVAL, "handles that share maps must have the same device, geometry and pixel range");
  if (h->sig && !h->maps_borrowed) { dfree(h->sig); dfree(h->rms); dfree(h->mask); }
  h->sig = src->sig;
  h->rms = src->rms;
  h->mask = src->mask;
  for (int j = 0; j < h->nbands; j++) {
    h->gain[j] = src->gain[j];
    h->offset[j] = src->offset[j];
  }
  h->maps_borrowed = true;
  h->maps_set = true;
  h->n_unmasked = -1;
  touch(h);
  API_END
}

int dang_gpu_set_component(dang_gpu_t *h, int ic, int type, const char *label, double nu_ref_hz,
                           int cg_group, int sample_amplitude, const double *amplitude,
                           const double *indices) {
  API_BEGIN
  if (ic < 0 || ic >= h->ncomp) fail(DANG_GPU_EINVAL, "component %d of %d", ic, h->ncomp);
  if (type < DANG_COMP_POWERLAW || type > DANG_COMP_HI_FIT) fail(DANG_GPU_EINVAL, "unrecognized component type %d", type);
  CompHost &c = h->comp[ic];
  c.set = true;
  c.type = type;
  c.label = label ? label : "";
  c.nu_ref = nu_ref_hz;
  c.cg_group = cg_group;
  c.sample_amplitude = sample_amplitude != 0;
  c.nind = (type == DANG_COMP_MBB || type == DANG_COMP_LOGNORMAL) ? 2
           : (type == DANG_COMP_CMB || type == DANG_COMP_TEMPLATE || type == DANG_COMP_MONOPOLE) ? 0 : 1;
  // "border" types: amp holds the template map, eval_signal carries template_amplitudes(band, plane)
  c.is_template = type == DANG_COMP_TEMPLATE || type == DANG_COMP_MONOPOLE || type == DANG_COMP_HI_FIT;
  if (c.is_template) {  // until dang_gpu_set_template: empty template, zero amplitudes, no fitted band
    memset(c.tamp_host, 0, sizeof c.tamp_host);
    memset(c.corr, 0, sizeof c.corr);
    c.nfit = 0;
    upload_tamp(h, c);
  }
  const size_t n2 = (size_t)h->nmaps * h->Ppad;
  if (!c.amp) CK(cudaMalloc(&c.amp, n2 * sizeof(double)));
  amp_write_barrier(h, c);
  CK(cudaMemsetAsync(c.amp, 0, n2 * sizeof(double), h->stream));
  if (amplitude && !c.is_template && type != DANG_COMP_T_CMB) h2d_planes(h, c.amp, amplitude, h->nmaps);
  if (type == DANG_COMP_T_CMB) {  // eval_signal = eval_sed (:770-771): an amplitude of exactly 1 everywhere
    fill_kernel<<<h->num_sms * 2, DG_THREADS, 0, h->stream>>>(c.amp, (int64_t)n2, 1.0);
    CK(cudaGetLastError());
  }
  if (type == DANG_COMP_MONOPOLE) {  // :591-594: template = 1 on plane 1, 0 on the polarisation planes
    fill_kernel<<<h->num_sms * 2, DG_THREADS, 0, h->stream>>>(c.amp, (int64_t)h->P, 1.0);
    CK(cudaGetLastError());
  }
  for (int l = 0; l < c.nind; l++) {
    if (!c.idx[l]) CK(cudaMalloc(&c.idx[l], n2 * sizeof(double)));
    // padding lanes get a harmless finite index
    fill_kernel<<<h->num_sms * 2, DG_THREADS, 0, h->stream>>>(c.idx[l], (int64_t)n2, 1.0);
    CK(cudaGetLastError());
    if (indices) h2d_planes(h, c.idx[l], indices + (size_t)l * h->nmaps * h->npix, h->nmaps);
    record_map_range(h, c, l, indices ? indices + (size_t)l * h->nmaps * h->npix : nullptr);
  }
  for (int l = 0; l < DG_MAXIND; l++) {
    c.index[l] = IndexHost();
    c.index[l].sample_nside = h->nside;
  }
  CK(cudaStreamSynchronize(h->stream));
  h->bp_dirty = true;
  h->tab_dirty = true;
  touch(h);
  for (int k = 0; k < 3; k++)
    for (int l = 0; l < DG_MAXIND; l++) h->check_mask |= 1ull << ((ic * 3 + k) * DG_MAXIND + l);
  API_END
}

int dang_gpu_set_template(dang_gpu_t *h, int ic, const double *template_map, const double *template_amplitudes,
                          const int *corr, int nfit) {
  API_BEGIN
  if (ic < 0 || ic >= h->ncomp || !h->comp[ic].set || !h->comp[ic].is_template)
    fail(DANG_GPU_EINVAL, "component %d is not a template component", ic);
  CompHost &c = h->comp[ic];
  if (!corr || (!template_map && c.type != DANG_COMP_MONOPOLE)) fail(DANG_GPU_EINVAL, "null template / corr pointer");
  int count = 0;
  for (int j = 0; j < h->nbands; j++) {
    c.corr[j] = corr[j] != 0;
    count += c.corr[j];
  }
  if (count != nfit) fail(DANG_GPU_EINVAL, "nfit = %d but corr selects %d bands", nfit, count);
  c.nfit = nfit;
  amp_write_barrier(h, c);
  if (c.type != DANG_COMP_MONOPOLE)
    h2d_planes(h, c.amp, template_map, h->nmaps);  // c%template ('template': already divided by temp_norm, :574-577)
  memset(c.tamp_host, 0, sizeof c.tamp_host);
  if (template_amplitudes)  // Fortran template_amplitudes(nbands, nmaps) == C [plane][band]
    for (int k = 0; k < h->nmaps; k++)
      for (int j = 0; j < h->nbands; j++) c.tamp_host[k][j] = template_amplitudes[(size_t)k * h->nbands + j];
  upload_tamp(h, c);
  monopole_to_offset(h, c);
  for (auto &g : h->cg)
    for (int f = 0; f < 3; f++) g.xt_set[f] = false;
  CK(cudaStreamSynchronize(h->stream));
  touch(h);
  API_END
}

int dang_gpu_set_t_cmb(dang_gpu_t *h, double t_cmb) {
  API_BEGIN
  if (!(t_cmb > 0.0)) fail(DANG_GPU_EINVAL, "T_CMB = %g", t_cmb);
  h->T_cmb = t_cmb;
  h->tab_dirty = true;  // the 'cmb' SED (1 / a2t) depends on it
  if (!rules_cover_params(h)) h->bp_dirty = true;
  touch(h);
  API_END
}

int dang_gpu_get_template_amplitudes(dang_gpu_t *h, int ic, double *template_amplitudes) {
  API_BEGIN
  if (ic < 0 || ic >= h->ncomp || !h->comp[ic].set || !h->comp[ic].is_template || !template_amplitudes)
    fail(DANG_GPU_EINVAL, "component %d is not a template component", ic);
  for (int k = 0; k < h->nmaps; k++)
    for (int j = 0; j < h->nbands; j++) template_amplitudes[(size_t)k * h->nbands + j] = h->comp[ic].tamp_host[k][j];
  API_END
}

int dang_gpu_set_index(dang_gpu_t *h, int ic, int nind, int sample_index, int index_mode,
                       int lnl_type, int prior_type, const double gauss_prior[2],
                       const double uni_prior[2], double step_size, int sample_nside,
                       const int *pol_flags, int nflag) {
  API_BEGIN
  if (ic < 0 || ic >= h->ncomp || !h->comp[ic].set) fail(DANG_GPU_EINVAL, "bad component %d", ic);
  CompHost &c = h->comp[ic];
  if (nind < 0 || nind >= c.nind) fail(DANG_GPU_EINVAL, "component %d has no index %d", ic, nind);
  if (nflag < 0 || nflag > 3) fail(DANG_GPU_EINVAL, "nflag = %d", nflag);
  if (index_mode != DANG_INDEX_FULLSKY && index_mode != DANG_INDEX_PERPIXEL) fail(DANG_GPU_EINVAL, "index_mode = %d", index_mode);
  IndexHost &ix = c.index[nind];
  ix.sample_index = sample_index != 0;
  ix.index_mode = index_mode;
  ix.lnl_type = lnl_type;
  ix.prior_type = prior_type;
  if (gauss_prior) { ix.gauss[0] = gauss_prior[0]; ix.gauss[1] = gauss_prior[1]; }
  if (uni_prior) { ix.uni[0] = uni_prior[0]; ix.uni[1] = uni_prior[1]; }
  ix.step = step_size;
  ix.sample_nside = sample_nside;
  ix.nflag = nflag;
  for (int k = 0; k < nflag; k++) ix.pol_flag[k] = pol_flags[k];
  if (!rules_cover_params(h)) h->bp_dirty = true;  // a wider prior box: verify the bandpass rules again
  touch(h);
  API_END
}

int dang_gpu_set_amplitude(dang_gpu_t *h, int ic, const double *amplitude) {
  API_BEGIN
  if (ic < 0 || ic >= h->ncomp || !h->comp[ic].set || !amplitude) fail(DANG_GPU_EINVAL, "bad component %d", ic);
  amp_write_barrier(h, h->comp[ic]);
  h2d_planes(h, h->comp[ic].amp, amplitude, h->nmaps);
  CK(cudaStreamSynchronize(h->stream));
  touch(h);
  API_END
}

int dang_gpu_set_indices(dang_gpu_t *h, int ic, const double *indices) {
  API_BEGIN
  if (ic < 0 || ic >= h->ncomp || !h->comp[ic].set || !indices) fail(DANG_GPU_EINVAL, "bad component %d", ic);
  for (int l = 0; l < h->comp[ic].nind; l++) {
    h2d_planes(h, h->comp[ic].idx[l], indices + (size_t)l * h->nmaps * h->npix, h->nmaps);
    record_map_range(h, h->comp[ic], l, indices + (size_t)l * h->nmaps * h->npix);
  }
  CK(cudaStreamSynchronize(h->stream));
  h->tab_dirty = true;
  if (!rules_cover_params(h)) h->bp_dirty = true;  // values outside the box the bandpass rules were verified on
  touch(h);
  for (int k = 0; k < 3; k++)
    for (int l = 0; l < DG_MAXIND; l++) h->check_mask |= 1ull << ((ic * 3 + k) * DG_MAXIND + l);
  API_END
}

int dang_gpu_get_amplitude(dang_gpu_t *h, int ic, double *amplitude) {
  API_BEGIN
  if (ic < 0 || ic >= h->ncomp || !h->comp[ic].set || !amplitude) fail(DANG_GPU_EINVAL, "bad component %d", ic);
  d2h_planes(h, amplitude, h->comp[ic].amp, h->nmaps);
  CK(cudaStreamSynchronize(h->stream));
  API_END
}

int dang_gpu_get_indices(dang_gpu_t *h, int ic, double *indices) {
  API_BEGIN
  if (ic < 0 || ic >= h->ncomp || !h->comp[ic].set || !indices) fail(DANG_GPU_EINVAL, "bad component %d", ic);
  for (int l = 0; l < h->comp[ic].nind; l++)
    d2h_planes(h, indices + (size_t)l * h->nmaps * h->npix, h->comp[ic].idx[l], h->nmaps);
  CK(cudaStreamSynchronize(h->stream));
  API_END
}

int dang_gpu_get_index_fullsky(dang_gpu_t *h, int ic, int nind, int map_n, double *value) {
  API_BEGIN
  if (ic < 0 || ic >= h->ncomp || !h->comp[ic].set || nind < 0 || nind >= h->comp[ic].nind || map_n < 1 ||
      map_n > h->nmaps || !value)
    fail(DANG_GPU_EINVAL, "bad component/index/map %d/%d/%d", ic, nind, map_n);
  {  // the host already knows the value when the plane's last writer was a full-sky draw
    const IndexHost &ixh = h->comp[ic].index[nind];
    if (!h->tab_dirty && ixh.last_value_epoch == h->idx_epoch && (ixh.last_value_planes >> (map_n - 1)) & 1) {
      *value = ixh.last_value;
      API_END_OK
    }
  }
  model_view(h);  // refreshes the uniformity flags
  if (h->nonuni_host[ic * 3 + (map_n - 1)][nind] != 0)
    fail(DANG_GPU_ESTATE, "plane %d of index %d of component %d is not constant", map_n, nind, ic);
  readback(h, h->pinned, h->comp[ic].idx[nind] + (size_t)(map_n - 1) * h->Ppad, sizeof(double));
  CK(cudaStreamSynchronize(h->stream));
  *value = *(double *)h->pinned;
  API_END
}

int dang_gpu_get_step_size(dang_gpu_t *h, int ic, int nind, double *step_size) {
  API_BEGIN
  if (ic < 0 || ic >= h->ncomp || !h->comp[ic].set || nind < 0 || nind >= h->comp[ic].nind || !step_size)
    fail(DANG_GPU_EINVAL, "bad component/index %d/%d", ic, nind);
  *step_size = h->comp[ic].index[nind].step;
  API_END
}

int dang_gpu_set_cg_group(dang_gpu_t *h, int cg_group, int i_max, double converge,
                          const int *pol_flags, int nflag) {
  API_BEGIN
  if (nflag < 1 || nflag > 3 || !pol_flags) fail(DANG_GPU_EINVAL, "nflag = %d", nflag);
  CgGroupHost *g = nullptr;
  for (auto &gg : h->cg)
    if (gg.cg_group == cg_group) g = &gg;
  if (!g) {
    h->cg.emplace_back();
    g = &h->cg.back();
  }
  g->set = true;
  g->cg_group = cg_group;
  g->i_max = i_max;
  g->converge = converge;
  g->nflag = nflag;
  for (int k = 0; k < nflag; k++) g->pol_flag[k] = pol_flags[k];
  API_END
}

int dang_gpu_cg_solve(dang_gpu_t *h, int cg_group, int flag_n, int ml_mode, const double *eta,
                      uint64_t seed, int *n_iter, double *delta_final) {
  API_BEGIN
  touch(h, 1);  // also when the solve fails half way: the amplitudes may have changed
  cg_solve(h, cg_group, flag_n, ml_mode, eta, seed, n_iter, delta_final);
  API_END
}

int dang_gpu_cg_trace(dang_gpu_t *h, double *delta, int max_len, int *len) {
  API_BEGIN
  int n = (int)h->last_trace.size();
  if (n > max_len) n = max_len;
  for (int i = 0; i < n; i++) delta[i] = h->last_trace[i];
  if (len) *len = n;
  API_END
}

int dang_gpu_get_cg_x(dang_gpu_t *h, int cg_group, int flag_n, double *x) {
  API_BEGIN
  CgGroupHost *g = nullptr;
  for (auto &gg : h->cg)
    if (gg.set && gg.cg_group == cg_group) g = &gg;
  if (!g || flag_n < 0 || flag_n >= g->nflag || !g->x[flag_n] || !x) fail(DANG_GPU_ESTATE, "no saved x for group %d flag %d", cg_group, flag_n);
  const int nplanes = (int)(g->x_len[flag_n] / h->Ppad);
  d2h_planes(h, x, g->x[flag_n], nplanes);
  CK(cudaStreamSynchronize(h->stream));
  API_END
}

// Deferred scalars: the device keeps ONE full-sky draw's outcome (MhScalars) for dang_gpu_iteration_mark.  A second
// full-sky draw -- or the tuner, which runs its chains in the same scalars -- before the mark would overwrite it.
static void deferred_draw_guard(const dang_gpu *h) {
  if (h->defer_scalars && h->pend_draw)
    fail(DANG_GPU_ESTATE, "a deferred full-sky draw is pending: call dang_gpu_iteration_mark before the next full-sky "
                          "draw or step-size tuning (its acceptance, value and chi-square would be lost)");
}

int dang_gpu_sample_index(dang_gpu_t *h, int ic, int nind, int map_n, int nsample, int ml_mode,
                          const double *z, const double *u, uint64_t seed, double *accept) {
  API_BEGIN
  if (nsample < 0) fail(DANG_GPU_EINVAL, "nsample = %d", nsample);
  MhView mh;
  mh_view(h, ic, nind, map_n, nsample, ml_mode, mh);
  const bool perpix = h->comp[ic].index[nind].index_mode == DANG_INDEX_PERPIXEL;
  if (h->idx_dl_pending) {  // the draw overwrites index planes a download may still be reading
    CK(cudaStreamWaitEvent(h->stream, h->ev_idx_dl, 0));
    h->idx_dl_pending = false;
  }
  if (!perpix) deferred_draw_guard(h);
  h->fs_tab_written = false;
  if (perpix) {
    touch(h, 2);
    idx_changed(h);
    sample_perpixel(h, mh, z, u, seed, accept);
  } else {
    sample_fullsky(h, mh, z, u, seed, accept);  // bumps the version itself (after using the cache)
    // planes that were tabulated before the draw stay tabulated, and the chain kernel has already put the new SED
    // into the table: nothing to flag, nothing to rebuild
    IndexHost &ixh = h->comp[ic].index[nind];
    const bool value_known = ixh.last_value_planes != -1;  // (deferred scalars: the draw's outcome is still on the device)
    ixh.last_value_planes = 0;
    for (int s = 0; s < mh.S && value_known; s++) ixh.last_value_planes |= 1 << mh.plane[s];
    if (h->fs_tab_written) {
      ixh.last_value_epoch = h->idx_epoch;
      API_END_OK
    }
    idx_changed(h);
    ixh.last_value_epoch = h->idx_epoch + 1;  // (the table rebuild this draw triggers bumps the epoch once more)
  }
  // the written planes are varying after a per-pixel draw (masked pixels are zeroed, so even a
  // chain that never moved leaves a non-constant plane unless nothing is masked -- treating it as
  // varying is always safe) and constant after a full-sky draw
  for (int s = 0; s < mh.S; s++) set_nonuni(h, ic, mh.plane[s], nind, perpix ? 1 : 0);
  API_END
}

int dang_gpu_get_decisions(dang_gpu_t *h, unsigned char *decisions, double *lnl) {
  API_BEGIN
  if (h->dec_mode == 0) fail(DANG_GPU_ESTATE, "no decisions recorded (per-pixel mode needs option 6)");
  if (h->dec_mode == 1) {
    if (decisions) CK(cudaMemcpyAsync(decisions, h->decisions, h->dec_nsample, cudaMemcpyDeviceToHost, h->stream));
    if (lnl) CK(cudaMemcpyAsync(lnl, h->lnl_trace, h->dec_nsample * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  } else {
    if (decisions)
      CK(cudaMemcpy2DAsync(decisions + h->lo, h->npix, h->decisions, h->P, h->P, h->dec_nsample,
                           cudaMemcpyDeviceToHost, h->stream));
    if (lnl)
      CK(cudaMemcpy2DAsync(lnl + h->lo, h->npix * sizeof(double), h->lnl_trace, h->P * sizeof(double),
                           h->P * sizeof(double), h->dec_nsample, cudaMemcpyDeviceToHost, h->stream));
  }
  CK(cudaStreamSynchronize(h->stream));
  API_END
}

int dang_gpu_perpixel_stats(dang_gpu_t *h, double *fallbacks, double *violations) {
  API_BEGIN
  if (fallbacks) *fallbacks = h->pp_fallbacks;
  if (violations) *violations = h->pp_violations;
  API_END
}

int dang_gpu_tune_index(dang_gpu_t *h, int ic, int nind, int map_n, int nsample, int ml_mode,
                        const double *z, const double *u, uint64_t seed, int max_blocks, int *blocks_run,
                        double *step_size) {
  API_BEGIN
  if (nsample < 0) fail(DANG_GPU_EINVAL, "nsample = %d", nsample);
  MhView mh;
  mh_view(h, ic, nind, map_n, nsample, ml_mode, mh);
  deferred_draw_guard(h);
  double start[DG_MAXIND] = {0.0, 0.0};
  const bool perpix = h->comp[ic].index[nind].index_mode == DANG_INDEX_PERPIXEL;
  if (perpix) {
    // the per-pixel call site (src/dang_sample_mod.f90:341-347) starts the tuner at
    // sample(l) = sum(c%indices(:, map_inds(1), l)) / sum(mask(:,1)) -- the sum runs over EVERY pixel -- and calls it
    // inside the loop over l, i.e. with the later indices still 0: only single-index components survive that
    if (h->comp[ic].nind != 1)
      fail(DANG_GPU_EUNSUPPORTED, "per-pixel step-size tuning of a component with %d indices: the reference calls the tuner "
                                  "with the other index still 0 (src/dang_sample_mod.f90:343-346), which never terminates",
           h->comp[ic].nind);
    model_view(h);
    const int64_t n_unmasked = unmasked_count(h);
    CK(cudaMemsetAsync(h->sums_local, 0, GATHER_MAX * sizeof(double), h->stream));
    const int grid = grid_for(h, h->P, DG_THREADS, 4);
    {
      KTimer kt(h, DANG_K_SCALAR, 0);
      masked_sum_kernel<<<grid, DG_THREADS, 0, h->stream>>>(h->comp[ic].idx[nind] + (size_t)mh.plane[0] * h->Ppad, nullptr, h->P,
                                                            h->partials, h->tickets, h->sums_local);
      kt.done();
    }
    gather(h, 4);
    double *hp = (double *)h->pinned;
    readback(h, hp, h->gathered, (size_t)h->nranks * 4 * sizeof(double));
    CK(cudaStreamSynchronize(h->stream));
    double sum = 0.0;
    for (int g = 0; g < h->nranks; g++) sum += hp[g * 4];
    start[0] = sum / (double)n_unmasked;
  }
  tune_fullsky(h, ic, nind, mh, z, u, seed, max_blocks, blocks_run, step_size, perpix ? start : nullptr);
  API_END
}

int dang_gpu_chisq(dang_gpu_t *h, int pol_lo, int pol_hi, double *chisq_planes, int64_t *n_unmasked) {
  API_BEGIN
  double out4[4];
  run_chisq(h, pol_lo, pol_hi, nullptr, nullptr, nullptr, out4);
  if (chisq_planes)
    for (int k = 0; k < h->nmaps; k++) chisq_planes[k] = out4[k];
  if (n_unmasked) *n_unmasked = (int64_t)(out4[3] + 0.5);
  API_END
}

int dang_gpu_get_sky_model(dang_gpu_t *h, int pol_lo, int pol_hi, double *sky_model, double *res_map,
                           double *chi_map) {
  API_BEGIN
  const size_t n3 = (size_t)h->nbands * h->nmaps * h->Ppad, n2 = (size_t)h->nmaps * h->Ppad;
  double *d_sky = nullptr, *d_res = nullptr, *d_chi = nullptr;
  try {
    CK(cudaMalloc(&d_sky, n3 * sizeof(double)));
    CK(cudaMalloc(&d_res, n3 * sizeof(double)));
    CK(cudaMalloc(&d_chi, n2 * sizeof(double)));
    double out4[4];
    run_chisq(h, pol_lo, pol_hi, d_sky, d_res, d_chi, out4);
    if (sky_model) d2h_planes(h, sky_model, d_sky, h->nbands * h->nmaps);
    if (res_map) d2h_planes(h, res_map, d_res, h->nbands * h->nmaps);
    if (chi_map) d2h_planes(h, chi_map, d_chi, h->nmaps);
    CK(cudaStreamSynchronize(h->stream));
  } catch (...) {
    cudaFree(d_sky); cudaFree(d_res); cudaFree(d_chi);
    throw;
  }
  cudaFree(d_sky); cudaFree(d_res); cudaFree(d_chi);
  API_END
}

int dang_gpu_iteration_mark(dang_gpu_t *h, int64_t *ticket) {
  API_BEGIN
  static_assert(offsetof(CgScalars, ah) <= DG_SNAP_CG && sizeof(MhScalars) <= DG_SNAP_MH, "snapshot sections");
  if (!ticket) fail(DANG_GPU_EINVAL, "ticket is NULL");
  const int64_t t = h->snap_ticket;
  dang_gpu::SnapMeta &m = h->snap_meta[t % DG_SNAP_SLOTS];
  if (m.ticket >= 0 && !m.read)
    fail(DANG_GPU_ESTATE, "ticket %lld has not been read and its slot is needed (at most %d marks may be outstanding)",
         (long long)m.ticket, DG_SNAP_SLOTS);
  unsigned char *slot = h->snap + (size_t)(t % DG_SNAP_SLOTS) * DG_SNAP_BYTES;
  h->snap_ticket++;
  m.ticket = t;
  m.read = false;
  m.cg = h->pend_cg;
  m.chisq_cg = h->pend_chisq_cg;
  m.draw = h->pend_draw;
  m.chisq_draw = h->pend_chisq_draw;
  m.g = h->pend_g;
  m.flag = h->pend_flag;
  m.ic = h->pend_ic;
  m.nind = h->pend_nind;
  m.S = h->pend_S;
  m.plane[0] = h->pend_plane[0];
  m.plane[1] = h->pend_plane[1];
  m.stat_cnt = h->pend_stat_cnt;
  m.cg_T = h->pend_cg_T;
  m.cg_C = h->pend_cg_C;
  m.cg_m = h->pend_cg_m;
  m.cg_vs = h->pend_cg_vs;
  const int n_cg = m.cg ? (int)(offsetof(CgScalars, ah) / 4) : 0;
  const int n_st = m.chisq_cg ? (int)((size_t)h->nranks * m.stat_cnt * 2) : 0;
  const int n_mh = m.draw ? (int)(sizeof(MhScalars) / 4) : 0;
  if (n_cg + n_st + n_mh > 0) {  // one launch, straight into pinned memory (no copy-engine work)
    snapshot_kernel<<<1, 256, 0, h->stream>>>((unsigned int *)slot, (const unsigned int *)h->cg_scalars, n_cg,
                                             (unsigned int *)(slot + DG_SNAP_CG), (const unsigned int *)h->mh_scalars, n_mh,
                                             (unsigned int *)(slot + DG_SNAP_CG + DG_SNAP_MH), (const unsigned int *)h->stat_buf, n_st);
    CK(cudaGetLastError());
    h->launches++;
  }
  CK(cudaEventRecord(m.ev, h->stream));
  h->pend_cg = h->pend_chisq_cg = h->pend_draw = h->pend_chisq_draw = false;
  *ticket = t;
  API_END
}

int dang_gpu_iteration_scalars(dang_gpu_t *h, int64_t ticket, int *n_iter, double *delta_final,
                               double *chisq_after_amplitudes, double *accept, double *index_value,
                               double *chisq_after_index) {
  API_BEGIN
  if (ticket < 0 || ticket >= h->snap_ticket) fail(DANG_GPU_EINVAL, "ticket %lld was never issued", (long long)ticket);
  dang_gpu::SnapMeta &m = h->snap_meta[ticket % DG_SNAP_SLOTS];
  if (m.ticket != ticket) fail(DANG_GPU_ESTATE, "ticket %lld has been overwritten by a later mark", (long long)ticket);
  CK(cudaEventSynchronize(m.ev));
  const unsigned char *slot = h->snap + (size_t)(ticket % DG_SNAP_SLOTS) * DG_SNAP_BYTES;
  const double qnan = nan("");
  if (n_iter) *n_iter = -1;
  if (delta_final) *delta_final = qnan;
  if (accept) *accept = qnan;
  if (index_value) *index_value = qnan;
  for (int k = 0; k < h->nmaps; k++) {
    if (chisq_after_amplitudes) chisq_after_amplitudes[k] = qnan;
    if (chisq_after_index) chisq_after_index[k] = qnan;
  }
  if (m.cg) {
    const CgScalars *hs = (const CgScalars *)slot;
    CgGroupHost &g = h->cg[m.g];
    if (!m.read) {  // book the solve's traffic now that its pass count is known; the prediction it ran with was the
                    // count of the solve before it, which an in-order reader has in last_iter
      const int k_pred = g.last_iter[m.flag] > 1 ? g.last_iter[m.flag] - 1 : 0x7fffffff;
      h->kstat[DANG_K_CG_PASS].bytes += bytes_w(cg_solve_bytes(hs->iter - 1, k_pred, m.cg_m, m.cg_T, m.cg_C, m.cg_vs));
      g.last_iter[m.flag] = hs->iter;
      const int n = hs->iter < 256 ? hs->iter : 256;
      h->last_trace.assign(hs->trace, hs->trace + n);
    }
    if (n_iter) *n_iter = hs->iter;
    if (delta_final) *delta_final = hs->delta_new;
  }
  if (m.chisq_cg && chisq_after_amplitudes) {
    double out4[4];
    chisq_of_statistics(h, (const double *)(slot + DG_SNAP_CG + DG_SNAP_MH), m.stat_cnt, m.S, m.plane, out4);
    for (int k = 0; k < h->nmaps; k++) chisq_after_amplitudes[k] = out4[k];
  }
  if (m.draw) {
    const MhScalars *hs = (const MhScalars *)(slot + DG_SNAP_CG);
    if (accept) *accept = hs->accept;
    if (index_value) *index_value = hs->sample[m.nind];
    if (m.chisq_draw && chisq_after_index) {
      for (int k = 0; k < h->nmaps; k++) chisq_after_index[k] = 0.0;
      for (int s = 0; s < m.S; s++) chisq_after_index[m.plane[s]] = hs->chisq[s];
    }
  }
  m.read = true;
  API_END
}

int dang_gpu_index_mean(dang_gpu_t *h, int ic, int nind, int map_n, double *mean) {
  API_BEGIN
  if (ic < 0 || ic >= h->ncomp || !h->comp[ic].set || nind < 0 || nind >= h->comp[ic].nind || map_n < 1 || map_n > h->nmaps)
    fail(DANG_GPU_EINVAL, "bad component/index/map %d/%d/%d", ic, nind, map_n);
  model_view(h);
  const int grid = grid_for(h, h->P, DG_THREADS, 4);
  KTimer kt(h, DANG_K_SCALAR, 0);
  masked_sum_kernel<<<grid, DG_THREADS, 0, h->stream>>>(h->comp[ic].idx[nind] + (size_t)(map_n - 1) * h->Ppad,
                                                       h->mask, h->P, h->partials, h->tickets, h->sums_local);
  kt.done();
  gather(h, 4);
  double *hp = (double *)h->pinned;
  readback(h, hp, h->gathered, (size_t)h->nranks * 4 * sizeof(double));
  CK(cudaStreamSynchronize(h->stream));
  double s = 0, n = 0;
  for (int g = 0; g < h->nranks; g++) { s += hp[g * 4]; n += hp[g * 4 + 1]; }
  if (mean) *mean = s / n;
  API_END
}

}  // extern "C"

// issue every recorded amplitude download on the d2h stream, ordered after `after` (an event of the compute stream)
void issue_deferred_d2h(dang_gpu *h, cudaEvent_t after) {
  if (h->deferred.empty()) return;
  CK(cudaStreamWaitEvent(h->d2h_stream, after, 0));
  for (const DeferredD2H &r : h->deferred) {
    CompHost &cc = h->comp[r.ic];
    const size_t o = (size_t)(r.k_lo - 1);
    CopyTimer ct(h, DANG_TL_D2H_AMP, h->d2h_stream);
    CK(cudaMemcpy2DAsync(r.dst + o * h->npix + h->lo, h->npix * sizeof(double), r.src + o * h->Ppad,
                         h->Ppad * sizeof(double), h->P * sizeof(double), r.k_hi - r.k_lo + 1, cudaMemcpyDeviceToHost,
                         h->d2h_stream));
    ct.done();
    // the buffer may have changed roles (amp <-> amp_alt) since the request: flag whichever it is now
    if (r.src == cc.amp) {
      CK(cudaEventRecord(cc.ev_read, h->d2h_stream));
      cc.read_pending = true;
    } else {
      CK(cudaEventRecord(cc.ev_read_alt, h->d2h_stream));
      cc.read_pending_alt = true;
    }
  }
  h->deferred.clear();
}

extern "C" {

int dang_gpu_get_amplitude_async(dang_gpu_t *h, int ic, int k_lo, int k_hi, double *amplitude) {
  API_BEGIN
  if (ic < 0 || ic >= h->ncomp || !h->comp[ic].set || !amplitude || k_lo < 1 || k_hi > h->nmaps || k_lo > k_hi)
    fail(DANG_GPU_EINVAL, "bad component / plane range %d %d..%d", ic, k_lo, k_hi);
  CompHost &cc = h->comp[ic];
  if (!cc.ev_read) {
    CK(cudaEventCreateWithFlags(&cc.ev_read, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&cc.ev_read_alt, cudaEventDisableTiming));
  }
  h->deferred.push_back(DeferredD2H{ic, cc.amp, amplitude, k_lo, k_hi});
  cc.read_pending = true;  // (requested: the next draw must not unpack into this buffer)
  if (!h->defer_d2h) {
    CK(cudaEventRecord(h->ev_compute, h->stream));
    issue_deferred_d2h(h, h->ev_compute);
  }
  API_END
}

int dang_gpu_get_indices_async(dang_gpu_t *h, int ic, int nind, int k_lo, int k_hi, double *indices) {
  API_BEGIN
  if (ic < 0 || ic >= h->ncomp || !h->comp[ic].set || nind < 0 || nind >= h->comp[ic].nind || !indices || k_lo < 1 ||
      k_hi > h->nmaps || k_lo > k_hi)
    fail(DANG_GPU_EINVAL, "bad component / index / plane range %d %d %d..%d", ic, nind, k_lo, k_hi);
  CK(cudaEventRecord(h->ev_compute, h->stream));
  CK(cudaStreamWaitEvent(h->d2h_stream, h->ev_compute, 0));
  const size_t o = (size_t)(k_lo - 1);
  CopyTimer ct(h, DANG_TL_D2H_IDX, h->d2h_stream);
  CK(cudaMemcpy2DAsync(indices + ((size_t)nind * h->nmaps + o) * h->npix + h->lo, h->npix * sizeof(double),
                       h->comp[ic].idx[nind] + o * h->Ppad, h->Ppad * sizeof(double), h->P * sizeof(double),
                       k_hi - k_lo + 1, cudaMemcpyDeviceToHost, h->d2h_stream));
  ct.done();
  CK(cudaEventRecord(h->ev_idx_dl, h->d2h_stream));
  h->idx_dl_pending = true;
  API_END
}

int dang_gpu_download_wait(dang_gpu_t *h) {
  API_BEGIN
  if (!h->deferred.empty()) {
    CK(cudaEventRecord(h->ev_compute, h->stream));
    issue_deferred_d2h(h, h->ev_compute);
  }
  CK(cudaStreamSynchronize(h->d2h_stream));
  for (auto &c : h->comp) c.read_pending = c.read_pending_alt = false;
  h->idx_dl_pending = false;
  API_END
}

int dang_gpu_stage_eta(dang_gpu_t *h, const double *eta, int nplanes) {
  API_BEGIN
  if (!eta || nplanes < 1 || nplanes > 2) fail(DANG_GPU_EINVAL, "stage_eta: nplanes = %d", nplanes);
  if (h->eta_count == 2) fail(DANG_GPU_ESTATE, "the deviates of two solves are already staged");
  const int slot = (h->eta_head + h->eta_count) % 2;
  ensure(h->eta_stage[slot], h->eta_stage_len[slot], (size_t)nplanes * h->Ppad);
  // the slot's previous consumer (K1 of an earlier solve) must have read it
  if (h->eta_used_recorded[slot]) CK(cudaStreamWaitEvent(h->h2d_stream, h->ev_eta_used[slot], 0));
  CopyTimer ct(h, DANG_TL_H2D_ETA, h->h2d_stream);
  CK(cudaMemcpy2DAsync(h->eta_stage[slot], h->Ppad * sizeof(double), eta + h->lo, h->npix * sizeof(double),
                       h->P * sizeof(double), nplanes, cudaMemcpyHostToDevice, h->h2d_stream));
  ct.done();
  CK(cudaEventRecord(h->ev_eta[slot], h->h2d_stream));
  h->eta_stage_planes[slot] = nplanes;
  h->eta_count++;
  API_END
}

int dang_gpu_fit_band_gain(dang_gpu_t *h, int map_n, int band, int ml_mode, const double *z, uint64_t seed,
                           double *gain) {
  API_BEGIN
  if (map_n < 1 || map_n > h->nmaps || band < 0 || band >= h->nbands) fail(DANG_GPU_EINVAL, "bad map / band %d / %d", map_n, band);
  ModelView mv = model_view(h);
  const int grid = occ_grid(h, band_gain_kernel, h->P, DG_THREADS);
  {
    KTimer kt(h, DANG_K_SCALAR, 0);
    band_gain_kernel<<<grid, DG_THREADS, 0, h->stream>>>(mv, map_n - 1, band, h->partials, h->tickets, h->sums_local);
    kt.done();
  }
  gather(h, 4);
  double *hp = (double *)h->pinned;
  readback(h, hp, h->gathered, (size_t)h->nranks * 4 * sizeof(double));
  CK(cudaStreamSynchronize(h->stream));
  double mu = 0.0, sigma = 0.0;
  for (int g = 0; g < h->nranks; g++) {
    mu += hp[g * 4 + 0];
    sigma += hp[g * 4 + 1];
  }
  mu = mu / sigma;               // :609-610
  sigma = sqrt(1.0 / sigma);
  double g = mu;
  if (ml_mode != DANG_ML_OPTIMIZE) {
    const double zz = z ? *z : philox_normal(seed, DG_STREAM_GAIN, (uint64_t)band);
    g = mu + sigma * (0.0 + 1.0 * zz);  // rand_normal(0,1), :615
  }
  h->gain[band] = g;             // ddata%gain(band) = gain, :619
  touch(h);
  if (gain) *gain = g;
  API_END
}

int dang_gpu_bandpass_quadrature(double nu_c_hz, int n_bp, const double *nu0_hz, const double *tau0, int nq,
                                 double *nu_q_hz, double *w_q) {
  if (n_bp < 1 || !nu0_hz || !tau0 || nq < 1 || nq > 32 || !nu_q_hz || !w_q) return DANG_GPU_EINVAL;
  BandHost b;
  b.set = true;
  b.nu_c = nu_c_hz;
  b.n = n_bp;
  b.nu0.assign(nu0_hz, nu0_hz + n_bp);
  b.tau0.assign(tau0, tau0 + n_bp);
  std::vector<double> nu, w;
  if (!gauss_compress(b, nq, nu, w)) return DANG_GPU_EUNSUPPORTED;  // the table would be kept
  for (int k = 0; k < nq; k++) {
    nu_q_hz[k] = nu[k];
    w_q[k] = w[k];
  }
  return DANG_GPU_OK;
}

int dang_gpu_band_samples(dang_gpu_t *h, int band, int *n_samples) {
  API_BEGIN
  if (band < 0 || band >= h->nbands || !h->band[band].set || !n_samples) fail(DANG_GPU_EINVAL, "bad band %d", band);
  upload_bandpasses(h);
  *n_samples = h->band[band].n_dev;
  API_END
}

int dang_gpu_host_alloc(void **ptr, uint64_t bytes) {
  return cudaMallocHost(ptr, bytes) == cudaSuccess ? DANG_GPU_OK : DANG_GPU_ECUDA;
}
int dang_gpu_host_free(void *ptr) { return cudaFreeHost(ptr) == cudaSuccess ? DANG_GPU_OK : DANG_GPU_ECUDA; }

int dang_gpu_event_record(dang_gpu_t *h, int slot) {
  API_BEGIN
  if (slot < 0 || slot >= 16) fail(DANG_GPU_EINVAL, "event slot %d", slot);
  CK(cudaEventRecord(h->ev[slot], h->stream));
  API_END
}

int dang_gpu_event_elapsed_ms(dang_gpu_t *h, int a, int b, float *ms) {
  API_BEGIN
  if (a < 0 || a >= 16 || b < 0 || b >= 16 || !ms) fail(DANG_GPU_EINVAL, "event slots %d %d", a, b);
  CK(cudaEventSynchronize(h->ev[b]));
  CK(cudaEventElapsedTime(ms, h->ev[a], h->ev[b]));
  API_END
}

int dang_gpu_launch_count(dang_gpu_t *h, int64_t *launches, int reset) {
  API_BEGIN
  if (launches) *launches = h->launches;
  if (reset) h->launches = 0;
  API_END
}

int dang_gpu_kernel_stats(dang_gpu_t *h, int kernel, int64_t *launches, double *total_ms, double *bytes,
                          int reset) {
  API_BEGIN
  if (kernel < 0 || kernel >= DANG_K_COUNT) fail(DANG_GPU_EINVAL, "kernel id %d", kernel);
  resolve_stats(h);
  KStat &k = h->kstat[kernel];
  if (launches) *launches = k.launches;
  if (total_ms) *total_ms = k.ms;
  if (bytes) *bytes = k.bytes;
  if (reset) { k.launches = 0; k.ms = 0; k.bytes = 0; }
  API_END
}

int dang_gpu_timeline(dang_gpu_t *h, int max_n, int *n, int *kind, double *t0_us, double *t1_us) {
  API_BEGIN
  resolve_stats(h);
  std::sort(h->tl.begin(), h->tl.end(), [](const TlRec &a, const TlRec &b) { return a.t0_us < b.t0_us; });
  int m = (int)h->tl.size();
  if (m > max_n) m = max_n;
  for (int i = 0; i < m; i++) {
    if (kind) kind[i] = h->tl[i].kind;
    if (t0_us) t0_us[i] = h->tl[i].t0_us;
    if (t1_us) t1_us[i] = h->tl[i].t1_us;
  }
  if (n) *n = m;
  API_END
}

const char *dang_gpu_kernel_name(int kernel) {
  static const char *names[DANG_K_COUNT] = {
      "rhs_blocks_kernel", "cg_pass_kernel", "cg_dq_pass_kernel", "cg_update_pass_kernel",
      "chisq_kernel", "chisq_kernel(maps)", "mh_data_kernel", "mh_fullsky_lnl_kernel",
      "mh_suffstat_kernel", "mh_perpixel_kernel", "scalar kernels", "cg_final_pass(x,unpack)"};
  static const char *extra[DANG_TL_EXTRA] = {"h2d:eta (copy stream)", "d2h:amplitude (copy stream)", "d2h:indices (copy stream)"};
  if (kernel >= DANG_K_COUNT && kernel < DANG_K_COUNT + DANG_TL_EXTRA) return extra[kernel - DANG_K_COUNT];
  return (kernel >= 0 && kernel < DANG_K_COUNT) ? names[kernel] : "?";
}

}  // extern "C"
