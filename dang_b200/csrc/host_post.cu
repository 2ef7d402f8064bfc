// host_post.cu -- dang_gpu_posterior_*: posterior mean / standard-deviation maps accumulated on the device, and the
// Gelman-Rubin R-hat across chains.  Not in the reference (its users write every sample and average offline).
#include "host.cuh"
#include "kernels_post.cuh"

namespace {

const int POST_ALL = DANG_POST_AMPLITUDE | DANG_POST_INDICES | DANG_POST_CHI_MAP | DANG_POST_RESIDUAL |
                     DANG_POST_TEMPLATE_AMPLITUDES;

bool has_map_amplitude(const CompHost &c) { return !c.is_template && c.type != DANG_COMP_T_CMB; }

// n elements: {mean, M2}, and with batch means {bmean, bM2} and bsum behind them (PostHost)
double2 *post_alloc(dang_gpu *h, size_t n, bool batched) {
  const size_t bytes = n * (batched ? 2 * sizeof(double2) + sizeof(double) : sizeof(double2));
  double2 *p = nullptr;
  CK(cudaMalloc(&p, bytes));
  CK(cudaMemsetAsync(p, 0, bytes, h->stream));
  return p;
}

const size_t TAMP_LEN = 3 * DG_MAX_BANDS;  // elements of a template-amplitude accumulator allocation

// the batch arrays of element `off` of an allocation of `len` elements
double *post_bsum(double2 *base, size_t len, size_t off) { return reinterpret_cast<double *>(base + 2 * len) + off; }
double2 *post_bacc(double2 *base, size_t len, size_t off) { return base + len + off; }

// the accumulators of one (kind, ic, nind) and their element layout
struct PostSlice {
  const double2 *acc = nullptr;
  int nplanes = 0;     // Ppad-strided planes, or
  bool table = false;  // a [nmaps][DG_MAX_BANDS] template-amplitude table
  int64_t len(const dang_gpu *h) const { return table ? (int64_t)h->nmaps * DG_MAX_BANDS : (int64_t)nplanes * h->Ppad; }
  // elements of the allocation: {bmean, bM2} start this many pairs after acc
  int64_t alloc_len(const dang_gpu *h) const { return table ? (int64_t)TAMP_LEN : len(h); }
};

PostSlice post_slice(const dang_gpu *h, int kind, int ic, int nind, int not_begun_code) {
  const PostHost &ps = h->post;
  if (!ps.what) fail(not_begun_code, "dang_gpu_posterior_begin has not been called");
  if (kind != DANG_POST_AMPLITUDE && kind != DANG_POST_INDICES && kind != DANG_POST_CHI_MAP && kind != DANG_POST_RESIDUAL &&
      kind != DANG_POST_TEMPLATE_AMPLITUDES)
    fail(DANG_GPU_EINVAL, "posterior kind %d is not one DANG_POST_* value", kind);
  if (!(ps.what & kind)) fail(not_begun_code, "posterior kind %d was not begun (what = %d)", kind, ps.what);
  PostSlice s;
  const bool comp_kind = kind == DANG_POST_AMPLITUDE || kind == DANG_POST_INDICES || kind == DANG_POST_TEMPLATE_AMPLITUDES;
  if (comp_kind && (ic < 0 || ic >= h->ncomp)) fail(DANG_GPU_EINVAL, "component %d of %d", ic, h->ncomp);
  switch (kind) {
    case DANG_POST_AMPLITUDE:
      s.acc = ps.amp[ic];
      s.nplanes = h->nmaps;
      if (!s.acc) fail(DANG_GPU_EINVAL, "component %d has no map amplitude (template, monopole, hi_fit or T_cmb)", ic);
      break;
    case DANG_POST_INDICES:
      if (nind < 0 || nind >= h->comp[ic].nind) fail(DANG_GPU_EINVAL, "component %d has no index %d", ic, nind);
      s.acc = ps.idx[ic][nind];
      s.nplanes = h->nmaps;
      break;
    case DANG_POST_TEMPLATE_AMPLITUDES:
      s.acc = ps.tamp[ic];
      s.table = true;
      if (!s.acc) fail(DANG_GPU_EINVAL, "component %d is not a template, monopole or hi_fit component", ic);
      break;
    case DANG_POST_CHI_MAP:
      s.acc = ps.chi;
      s.nplanes = h->nmaps;
      break;
    case DANG_POST_RESIDUAL:
      s.acc = ps.res;
      s.nplanes = h->nbands * h->nmaps;
      break;
  }
  return s;
}

// device planes / table of `s`'s layout -> the caller's array in the layout of the matching getter
void post_d2h(dang_gpu *h, const PostSlice &s, double *dst, const double *src) {
  if (s.table)  // [k][DG_MAX_BANDS] -> Fortran template_amplitudes(nbands, nmaps) == C [k][band]
    CK(cudaMemcpy2DAsync(dst, h->nbands * sizeof(double), src, DG_MAX_BANDS * sizeof(double), h->nbands * sizeof(double),
                         h->nmaps, cudaMemcpyDeviceToHost, h->stream));
  else
    d2h_planes(h, dst, src, s.nplanes);
}

// device scratch of one read-out, freed on every exit
struct DevBuf {
  double *p = nullptr;
  explicit DevBuf(size_t n) { CK(cudaMalloc(&p, n * sizeof(double))); }
  ~DevBuf() { cudaFree(p); }
};

// the accumulators of (kind, ic, nind) on m chains that share the device, geometry, pixel range and n; the slice of
// hs[0] describes them all
PostSlice post_chains(dang_gpu *const *hs, int m, int kind, int ic, int nind, RhatView &v) {
  const dang_gpu *h = hs[0];
  v.m = m;
  PostSlice s0;
  for (int c = 0; c < m; c++) {
    const dang_gpu *g = hs[c];
    if (!g) fail(DANG_GPU_EINVAL, "handle %d is NULL", c);
    if (g->device != h->device || g->npix != h->npix || g->nmaps != h->nmaps || g->nbands != h->nbands ||
        g->lo != h->lo || g->hi != h->hi)
      fail(DANG_GPU_EINVAL, "handle %d: chains must share the device, geometry and pixel range", c);
    const PostSlice s = post_slice(g, kind, ic, nind, DANG_GPU_EINVAL);
    if (g->post.n != h->post.n) fail(DANG_GPU_EINVAL, "handle %d holds %lld samples, handle 0 %lld", c,
                                     (long long)g->post.n, (long long)h->post.n);
    if (c == 0) s0 = s;
    v.acc[c] = s.acc;
  }
  return s0;
}

// the residual / chi-square sink through the component-count ladder of run_chisq's map form (dang_gpu_get_sky_model)
template <class Sink>
void launch_chisq_post(dang_gpu *h, const Sink &sink) {
  const ModelView mv = model_view(h);
  ChisqView cv;
  cv.k_lo = h->post.pol_lo - 1;
  cv.k_hi = h->post.pol_hi - 1;
  cv.sky = cv.res = cv.chi_map = nullptr;
#define LAUNCH_CHISQ_POST(NC)                                                                          \
  chisq_kernel<NC, Sink><<<occ_grid(h, chisq_kernel<NC, Sink>, h->P, DG_THREADS), DG_THREADS, 0, h->stream>>>( \
      mv, cv, nullptr, nullptr, nullptr, sink)
  if (h->ncomp <= 1) LAUNCH_CHISQ_POST(1);
  else if (h->ncomp == 2) LAUNCH_CHISQ_POST(2);
  else if (h->ncomp == 3) LAUNCH_CHISQ_POST(3);
  else if (h->ncomp == 4) LAUNCH_CHISQ_POST(4);
  else LAUNCH_CHISQ_POST(DG_MAX_COMPS);
#undef LAUNCH_CHISQ_POST
  CK(cudaGetLastError());
  h->launches++;
}

template <bool OPEN, bool CLOSE>
void launch_stream_batch(dang_gpu *h, int gx, const PostBatchTable &t, double n, const PostBatch &p) {
  post_stream_batch_kernel<OPEN, CLOSE><<<dim3(gx, t.count), DG_THREADS, 0, h->stream>>>(t, n, p.b, p.k);
}

void post_begin(dang_gpu *h, int what, int pol_lo, int pol_hi, int batch_len) {
  if (what <= 0 || (what & ~POST_ALL)) fail(DANG_GPU_EINVAL, "posterior kinds %d: not a set of DANG_POST_* bits", what);
  if ((what & (DANG_POST_CHI_MAP | DANG_POST_RESIDUAL)) && (pol_lo < 1 || pol_hi > h->nmaps || pol_lo > pol_hi))
    fail(DANG_GPU_EINVAL, "bad pol_type range %d..%d", pol_lo, pol_hi);
  for (int c = 0; c < h->ncomp; c++)
    if (!h->comp[c].set) fail(DANG_GPU_ESTATE, "component %d has not been set", c);
  post_release(h);
  PostHost &ps = h->post;
  const size_t n2 = (size_t)h->nmaps * h->Ppad;
  const bool batched = batch_len > 0;
  try {
    for (int c = 0; c < h->ncomp; c++) {
      const CompHost &cc = h->comp[c];
      if ((what & DANG_POST_AMPLITUDE) && has_map_amplitude(cc)) ps.amp[c] = post_alloc(h, n2, batched);
      if (what & DANG_POST_INDICES)
        for (int l = 0; l < cc.nind; l++) ps.idx[c][l] = post_alloc(h, n2, batched);
      if ((what & DANG_POST_TEMPLATE_AMPLITUDES) && cc.is_template) ps.tamp[c] = post_alloc(h, TAMP_LEN, batched);
    }
    if (what & DANG_POST_RESIDUAL) ps.res = post_alloc(h, (size_t)h->nbands * n2, batched);
    if (what & DANG_POST_CHI_MAP) ps.chi = post_alloc(h, n2, batched);
  } catch (...) {
    ps.what = POST_ALL;  // (release whatever was allocated)
    post_release(h);
    throw;
  }
  ps.what = what;
  ps.pol_lo = pol_lo;
  ps.pol_hi = pol_hi;
  ps.batch_len = batch_len;
  ps.n = 0;
}

}  // namespace

void post_release(dang_gpu *h) {
  PostHost &ps = h->post;
  if (!ps.what) return;
  if (h->stream) cudaStreamSynchronize(h->stream);  // an accumulation may still be writing
  for (int c = 0; c < DG_MAX_COMPS; c++) {
    dfree(ps.amp[c]);
    dfree(ps.tamp[c]);
    for (int l = 0; l < DG_MAXIND; l++) dfree(ps.idx[c][l]);
  }
  dfree(ps.res);
  dfree(ps.chi);
  ps = PostHost();
}

#define API_BEGIN                                   \
  if (!h) return DANG_GPU_EINVAL;                   \
  try {                                             \
    set_device(h);
#define API_END                                     \
    return DANG_GPU_OK;                             \
  } catch (const DgError &e) {                      \
    h->err = e.what();                              \
    return e.code;                                  \
  } catch (const std::exception &e) {               \
    h->err = e.what();                              \
    return DANG_GPU_ECUDA;                          \
  }

extern "C" {

int dang_gpu_posterior_begin(dang_gpu_t *h, int what, int pol_lo, int pol_hi) {
  API_BEGIN
  post_begin(h, what, pol_lo, pol_hi, 0);
  API_END
}

int dang_gpu_posterior_begin_batched(dang_gpu_t *h, int what, int pol_lo, int pol_hi, int batch_len) {
  API_BEGIN
  if (batch_len < 1) fail(DANG_GPU_EINVAL, "batch length %d (>= 1)", batch_len);
  post_begin(h, what, pol_lo, pol_hi, batch_len);
  API_END
}

// Stream ordered, no host wait: the samples are read where the state lives at this point of h->stream.
int dang_gpu_posterior_accumulate(dang_gpu_t *h) {
  API_BEGIN
  PostHost &ps = h->post;
  if (!ps.what) fail(DANG_GPU_ESTATE, "dang_gpu_posterior_begin has not been called");
  const double n = (double)(ps.n + 1);
  const int64_t b = ps.batch_len;
  PostBatch pb{};  // sample n + 1 is at position j of its batch
  if (b) {
    const int64_t j = ps.n % b + 1;
    pb = PostBatch{(double)b, (double)((ps.n + 1) / b), j == 1, j == b};
  }
  PostTable t;
  PostBatchTable tb;
  t.count = tb.count = 0;
  static_assert(DG_MAX_COMPS * (3 * (1 + DG_MAXIND) + 1) <= DG_POST_ENTRIES, "one table entry per accumulated array");
  // element `off` of the allocation `base` of `alen` elements, `len` elements long
  auto add = [&](const double *src, double2 *base, size_t alen, size_t off, int64_t len) {
    t.e[t.count++] = PostEntry{src, base + off, len};
    if (b) tb.e[tb.count++] = PostBatchEntry{src, base + off, post_bsum(base, alen, off), post_bacc(base, alen, off), len};
  };
  const size_t n2 = (size_t)h->nmaps * h->Ppad;
  for (int c = 0; c < h->ncomp; c++) {
    const CompHost &cc = h->comp[c];
    for (int k = 0; k < h->nmaps; k++) {
      const size_t o = (size_t)k * h->Ppad;
      // c.amp now: a solve that ran behind a pending download unpacked into the other buffer and swapped them
      if (ps.amp[c]) add(cc.amp + o, ps.amp[c], n2, o, h->Ppad);
      for (int l = 0; l < cc.nind; l++)
        if (ps.idx[c][l]) add(cc.idx[l] + o, ps.idx[c][l], n2, o, h->Ppad);
    }
    if (ps.tamp[c]) add(cc.tamp, ps.tamp[c], TAMP_LEN, 0, TAMP_LEN);
  }
  if (t.count) {
    const int gx = (grid_for(h, (int64_t)t.count * h->Ppad / 2, DG_THREADS, 4) + t.count - 1) / t.count;
    if (!b) post_stream_kernel<<<dim3(gx, t.count), DG_THREADS, 0, h->stream>>>(t, n);
    else if (pb.open && pb.close) launch_stream_batch<true, true>(h, gx, tb, n, pb);
    else if (pb.open) launch_stream_batch<true, false>(h, gx, tb, n, pb);
    else if (pb.close) launch_stream_batch<false, true>(h, gx, tb, n, pb);
    else launch_stream_batch<false, false>(h, gx, tb, n, pb);
    CK(cudaGetLastError());
    h->launches++;
  }
  if (ps.res || ps.chi) {
    if (!b) {
      launch_chisq_post(h, ChisqPost{ps.res, ps.chi, n});
    } else {
      const size_t rlen = (size_t)h->nbands * n2;
      ChisqPostBatch sink{};
      if (ps.res) {
        sink.acc_res = ps.res;
        sink.bsum_res = post_bsum(ps.res, rlen, 0);
        sink.bacc_res = post_bacc(ps.res, rlen, 0);
      }
      if (ps.chi) {
        sink.acc_chi = ps.chi;
        sink.bsum_chi = post_bsum(ps.chi, n2, 0);
        sink.bacc_chi = post_bacc(ps.chi, n2, 0);
      }
      sink.n = n;
      sink.p = pb;
      launch_chisq_post(h, sink);
    }
  }
  ps.n++;
  API_END
}

int dang_gpu_posterior_get(dang_gpu_t *h, int kind, int ic, int nind, double *mean, double *stddev, int64_t *n) {
  API_BEGIN
  const PostSlice s = post_slice(h, kind, ic, nind, DANG_GPU_ESTATE);
  if (!mean) fail(DANG_GPU_EINVAL, "null mean");
  const int64_t len = s.len(h);
  DevBuf out((size_t)(stddev ? 2 : 1) * len);
  post_finalize_kernel<<<grid_for(h, len, DG_THREADS, 4), DG_THREADS, 0, h->stream>>>(
      s.acc, len, h->post.n, out.p, stddev ? out.p + len : nullptr);
  CK(cudaGetLastError());
  h->launches++;
  post_d2h(h, s, mean, out.p);
  if (stddev) post_d2h(h, s, stddev, out.p + len);
  CK(cudaStreamSynchronize(h->stream));
  if (n) *n = h->post.n;
  API_END
}

int dang_gpu_posterior_end(dang_gpu_t *h) {
  API_BEGIN
  if (!h->post.what) fail(DANG_GPU_ESTATE, "dang_gpu_posterior_begin has not been called");
  post_release(h);
  API_END
}

int dang_gpu_posterior_rhat(dang_gpu_t *const *hs, int m, int kind, int ic, int nind, double *rhat) {
  if (!hs || !hs[0]) return DANG_GPU_EINVAL;
  dang_gpu *h = hs[0];  // errors are reported on the first handle
  API_BEGIN
  if (m < 2 || m > DG_RHAT_MAX) fail(DANG_GPU_EINVAL, "R-hat over %d chains (2..%d)", m, DG_RHAT_MAX);
  if (!rhat) fail(DANG_GPU_EINVAL, "null rhat");
  RhatView v;
  const PostSlice s0 = post_chains(hs, m, kind, ic, nind, v);
  if (h->post.n < 2) fail(DANG_GPU_EINVAL, "R-hat needs n >= 2 samples per chain (n = %lld)", (long long)h->post.n);
  for (int c = 0; c < m; c++) CK(cudaStreamSynchronize(hs[c]->stream));  // every chain's accumulations have landed
  const int64_t len = s0.len(h);
  DevBuf out((size_t)len);
  post_rhat_kernel<<<grid_for(h, len, DG_THREADS, 4), DG_THREADS, 0, h->stream>>>(v, len, h->post.n, out.p);
  CK(cudaGetLastError());
  h->launches++;
  post_d2h(h, s0, rhat, out.p);
  CK(cudaStreamSynchronize(h->stream));
  API_END
}

int dang_gpu_posterior_ess(dang_gpu_t *const *hs, int m, int kind, int ic, int nind, double *ess, double *mcse) {
  if (!hs || !hs[0]) return DANG_GPU_EINVAL;
  dang_gpu *h = hs[0];  // errors are reported on the first handle
  API_BEGIN
  if (m < 1 || m > DG_RHAT_MAX) fail(DANG_GPU_EINVAL, "ESS over %d chains (1..%d)", m, DG_RHAT_MAX);
  if (!ess && !mcse) fail(DANG_GPU_EINVAL, "null ess and mcse");
  for (int c = 0; c < m; c++) {
    const dang_gpu *g = hs[c];
    if (!g) fail(DANG_GPU_EINVAL, "handle %d is NULL", c);
    if (!g->post.what) fail(DANG_GPU_ESTATE, "handle %d: dang_gpu_posterior_begin has not been called", c);
    if (!g->post.batch_len) fail(DANG_GPU_ESTATE, "handle %d was begun without batch means", c);
  }
  RhatView v;
  const PostSlice s0 = post_chains(hs, m, kind, ic, nind, v);
  const int64_t b = h->post.batch_len, n = h->post.n;
  for (int c = 0; c < m; c++)
    if (hs[c]->post.batch_len != b)
      fail(DANG_GPU_EINVAL, "handle %d has batch length %d, handle 0 %lld", c, hs[c]->post.batch_len, (long long)b);
  if (n / b < 2) fail(DANG_GPU_EINVAL, "ESS needs K >= 2 complete batches (n = %lld, b = %lld)", (long long)n, (long long)b);
  for (int c = 0; c < m; c++) CK(cudaStreamSynchronize(hs[c]->stream));  // every chain's accumulations have landed
  const int64_t len = s0.len(h);
  DevBuf out((size_t)(ess && mcse ? 2 : 1) * len);
  double *d_ess = ess ? out.p : nullptr, *d_mcse = mcse ? out.p + (ess ? len : 0) : nullptr;
  post_ess_kernel<<<grid_for(h, len, DG_THREADS, 4), DG_THREADS, 0, h->stream>>>(v, s0.alloc_len(h), len, n, n / b,
                                                                                  (double)b, d_ess, d_mcse);
  CK(cudaGetLastError());
  h->launches++;
  if (ess) post_d2h(h, s0, ess, d_ess);
  if (mcse) post_d2h(h, s0, mcse, d_mcse);
  CK(cudaStreamSynchronize(h->stream));
  API_END
}

}  // extern "C"
