// host.cuh -- host-side state of one handle (struct dang_gpu) and the launch helpers shared by the
// translation units of libdang_gpu.so: dang_gpu.cu (C ABI, tables, maps), host_cg.cu (amplitude
// draw), host_mh_pp.cu / host_mh_fs.cu (spectral-parameter draw), host_data.cu (chi-square).
#pragma once
#include "../../include/dang_gpu.h"

#include <cuda_runtime.h>
#include <dlfcn.h>

#include <cstdarg>
#include <cstddef>
#include <cstdio>
#include <cmath>
#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>

#include "common.cuh"

// ---------------------------------------------------------------- errors

struct DgError : std::runtime_error {
  int code;
  DgError(int c, const std::string &m) : std::runtime_error(m), code(c) {}
};

inline std::string vfmt(const char *f, va_list ap) {
  char buf[1024];
  vsnprintf(buf, sizeof buf, f, ap);
  return buf;
}
[[noreturn]] inline void fail(int code, const char *f, ...) {
  va_list ap;
  va_start(ap, f);
  std::string m = vfmt(f, ap);
  va_end(ap);
  throw DgError(code, m);
}

#define CK(call)                                                                              \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess)                                                                    \
      fail(DANG_GPU_ECUDA, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__,               \
           cudaGetErrorString(e_));                                                           \
  } while (0)

extern thread_local std::string g_create_error;
// ---------------------------------------------------------------- NCCL (loaded lazily)
// Only multi-rank runs touch NCCL; it is dlopen'ed so a single-GPU Fortran host needs no NCCL.
typedef struct { char internal[128]; } nccl_uid_t;
typedef void *nccl_comm_t;
struct NcclApi {
  void *lib = nullptr;
  int (*GetUniqueId)(nccl_uid_t *) = nullptr;
  int (*CommInitRank)(nccl_comm_t *, int, nccl_uid_t, int) = nullptr;
  int (*CommDestroy)(nccl_comm_t) = nullptr;
  int (*AllGather)(const void *, void *, size_t, int, nccl_comm_t, cudaStream_t) = nullptr;
  const char *(*GetErrorString)(int) = nullptr;
};
extern NcclApi g_nccl;
void nccl_load();
#define NCK(call)                                                                       \
  do {                                                                                  \
    int r_ = (call);                                                                    \
    if (r_ != 0) fail(DANG_GPU_ENCCL, "%s failed: %s", #call, g_nccl.GetErrorString(r_)); \
  } while (0)
const int NCCL_DOUBLE = 8;  // ncclFloat64
// ---------------------------------------------------------------- host-side objects
struct BandHost {
  bool set = false;
  double nu_c = 0;
  int n = 0;
  std::vector<double> nu0, tau0;
  // what the device sees: the table itself, or its Gauss-quadrature compression (upload_bandpasses)
  int n_dev = 0;
  std::vector<double> nu0_dev, tau0_dev;
};

struct IndexHost {
  int sample_index = 0, index_mode = DANG_INDEX_PERPIXEL, lnl_type = 0, prior_type = 0;
  double gauss[2] = {0, 1}, uni[2] = {-1e300, 1e300}, step = 0;
  int sample_nside = 0, nflag = 0, pol_flag[3] = {0, 0, 0};
  double last_value = 0;  // value left by the last full-sky draw (the whole plane holds it)
  uint64_t last_value_epoch = 0;  // dang_gpu::idx_epoch right after that draw: the value is current while they agree
  int last_value_planes = 0;      // bit k: plane k holds it
};

struct CompHost {
  bool set = false;
  int type = 0, cg_group = 0, sample_amplitude = 0, nind = 0;
  std::string label;
  double nu_ref = 0;
  double *amp = nullptr;               // [nmaps][Ppad]
  // Second amplitude buffer: while an asynchronous download still reads `amp`, the next solve unpacks
  // into `amp_alt` and the two swap roles, so a download never stalls the solve that follows it.
  double *amp_alt = nullptr;
  // type 'template' (src/dang_component_mod.f90:536-577): amp holds the template map
  bool is_template = false;
  double *tamp = nullptr;                       // device [3][DG_MAX_BANDS] template_amplitudes
  double tamp_host[3][DG_MAX_BANDS] = {};
  int corr[DG_MAX_BANDS] = {};
  int nfit = 0;
  cudaEvent_t ev_read = nullptr, ev_read_alt = nullptr;  // last download that read amp / amp_alt
  bool read_pending = false, read_pending_alt = false;
  double *idx[DG_MAXIND] = {nullptr, nullptr};
  IndexHost index[DG_MAXIND];
  // range of the index maps the host last uploaded (this handle's pixels), and the box of index values the
  // bandpass rules were verified on (upload_bandpasses)
  double map_range[DG_MAXIND][2] = {{1.0, 1.0}, {1.0, 1.0}};
  double verified_box[DG_MAXIND][2] = {{0.0, -1.0}, {0.0, -1.0}};
};

struct CgGroupHost {
  bool set = false;
  int cg_group = 0, i_max = 0, nflag = 0, pol_flag[3] = {0, 0, 0};
  double converge = 0;
  double *x[3] = {nullptr, nullptr, nullptr};  // Q10: persists across Gibbs iterations
  double xt[3][32] = {};                       // ... and so do the template amplitudes in the tail of x
  bool xt_set[3] = {false, false, false};
  size_t x_len[3] = {0, 0, 0};
  int last_iter[3] = {0, 0, 0};  // iterations of the previous solve (sizes the first batch)
};

struct KStat {
  int64_t launches = 0;
  double ms = 0, bytes = 0;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> pending;
};

const int GATHER_MAX = 256;  // doubles per rank in one scalar exchange
const int DG_SNAP_SLOTS = 4;
const size_t DG_SNAP_CG = 4096, DG_SNAP_MH = 1024, DG_SNAP_STAT = (size_t)GATHER_MAX * 32 * 8;  // bytes per slot section
const size_t DG_SNAP_BYTES = DG_SNAP_CG + DG_SNAP_MH + DG_SNAP_STAT;

// event-log kinds beyond the kernel families of dang_gpu.h: staged copies on the side streams
const int DANG_TL_EXTRA = 3;
enum { DANG_TL_H2D_ETA = DANG_K_COUNT, DANG_TL_D2H_AMP = DANG_K_COUNT + 1, DANG_TL_D2H_IDX = DANG_K_COUNT + 2 };
struct TlRec {
  int kind;
  double t0_us, t1_us;
};

struct dang_gpu {
  int device = 0, nside = 0, nmaps = 0, nbands = 0, ncomp = 0, num_sms = 0;
  int64_t npix = 0, lo = 0, hi = 0, P = 0, Ppad = 0;
  cudaStream_t stream = nullptr, d2h_stream = nullptr, h2d_stream = nullptr;
  cudaEvent_t ev_compute = nullptr, ev_idx_dl = nullptr;
  std::vector<struct DeferredD2H> deferred;  // amplitude downloads requested but not issued yet
  int defer_d2h = 1;                         // DANG_OPT_DEFER_D2H
  // deferred scalars (DANG_OPT_DEFER_SCALARS): cg_solve / chisq / full-sky sample_index enqueue their kernels and
  // return without waiting; dang_gpu_iteration_mark snapshots the device-side results into a ring of pinned slots
  // and dang_gpu_iteration_scalars decodes a slot later -- one host wait per Gibbs iteration, one iteration behind
  int defer_scalars = 0;
  bool pend_cg = false, pend_chisq_cg = false, pend_draw = false;  // what the calls since the last mark left behind
  int pend_g = -1, pend_flag = -1, pend_ic = -1, pend_nind = -1, pend_S = 0, pend_plane[2] = {0, 0}, pend_stat_cnt = 0;
  int pend_chisq_lo = 0, pend_chisq_hi = 0;
  int pend_cg_T = 0, pend_cg_C = 0, pend_cg_m = 0;
  double pend_cg_vs = 0.0;
  bool pend_draw_chisq = false;   // the pending draw's MhScalars::chisq is the chi-square of the state it left
  uint64_t pend_draw_version = 0;
  bool pend_chisq_draw = false;   // ... and a dang_gpu_chisq call asked for it
  unsigned char *snap = nullptr;  // pinned: DG_SNAP_SLOTS slots
  int64_t snap_ticket = 0;
  struct SnapMeta {
    int64_t ticket = -1;
    bool read = false;
    bool cg = false, chisq_cg = false, draw = false;
    bool chisq_draw = false;
    int g = -1, flag = -1, ic = -1, nind = -1, S = 0, plane[2] = {0, 0}, stat_cnt = 0, chisq_lo = 0, chisq_hi = 0;
    int cg_T = 0, cg_C = 0, cg_m = 0;
    double cg_vs = 0.0;
    cudaEvent_t ev = nullptr;
  } snap_meta[4];
  cudaEvent_t ev_sync = nullptr;  // host waits for a point of the compute stream (results read back) while later kernels run
  bool idx_dl_pending = false;
  // staged deviates of the next solves: a two-slot FIFO, so the upload for solve k+1 runs while solve k
  // (which consumes the other slot) is still computing
  double *eta_stage[2] = {nullptr, nullptr}; size_t eta_stage_len[2] = {0, 0}; int eta_stage_planes[2] = {0, 0};
  cudaEvent_t ev_eta[2] = {nullptr, nullptr}, ev_eta_used[2] = {nullptr, nullptr};
  bool eta_used_recorded[2] = {false, false};
  int eta_head = 0, eta_count = 0;
  std::string err;

  // options
  int fix_q1 = 0, cg_two_pass = 0, fullsky_stream = 0, profile = 0, cg_chunk = 8, record = 0, perpixel_serial = 0;
  int cg_ckpt = 8;  // checkpoint interval of the recompute CG form (0: streaming form)
  int stream_ring = 1;    // K1 / statistics pass fed by per-thread cp.async rings (DANG_OPT_STREAM_RING)
  int cg_persistent = 1;  // whole solve in one persistent cooperative kernel (DANG_OPT_CG_PERSISTENT)
  int bp_quad = 8;        // nodes of the Gauss-quadrature compression of tabulated bandpasses (0: off)
  int pp_bp_series = 1;   // tabulated bandpasses: moment series in the per-pixel chains (DANG_OPT_PERPIXEL_BP_SERIES)
  int pp_pix = 1;         // 1: one-thread-per-pixel form of the screened kernel (kernels_mh_pix.cuh)
  int pp_split = 0;       // 1: split form of the screened kernel (rng / state / chain kernels), measured slower
  void *k5_st4 = nullptr; float *k5_kj = nullptr; size_t k5_len = 0;  // its fp32 state scratch
  int pp_fast = 1;        // certified fp32 screening in the per-pixel Metropolis kernel (DANG_OPT_PERPIXEL_FAST)
  double pp_fallbacks = 0, pp_violations = 0;  // of the last per-pixel draw (all ranks)
  int l2_persist_mb = 0;  // MB of the CG block matrices kept persisting in L2 during a solve (0: off)
  size_t l2_persist_max = 0, l2_window_max = 0;
  int use_tma = 0;  // TMA-staged K1 (measured slower than the LDG form on B200: kept as an experiment)

  // ddata
  bool maps_set = false, maps_borrowed = false;  // borrowed: sig/rms/mask belong to another handle (ensembles)
  double *sig = nullptr, *rms = nullptr;
  unsigned char *mask = nullptr;
  double gain[DG_MAX_BANDS], offset[DG_MAX_BANDS];
  double T_cmb = 2.7255;  // src/dang_util_mod.f90:15; dang_gpu_set_t_cmb

  BandHost band[DG_MAX_BANDS];
  double *bp_nu0 = nullptr, *bp_tau0 = nullptr, *bp_lnr_hi = nullptr, *bp_lnr_lo = nullptr;
  int nbp = 0;
  bool bp_dirty = true;   // band / component constants changed: rebuild the static tables
  double verified_T_cmb[2] = {0.0, -1.0};  // T_CMB range the 'cmb' SED was verified on
  bool tab_dirty = true;  // an index map changed: re-tabulate SEDs
  unsigned long long check_mask = ~0ull;  // index maps whose uniformity must be re-scanned
  SedTable *tab = nullptr;
  int uni_host[DG_MAX_COMPS * 3] = {};  // host copy of SedTable::uni (refreshed with the tables)
  int nonuni_host[DG_MAX_COMPS * 3][DG_MAXIND] = {};  // host mirror of SedTable::nonuni
  CompHost comp[DG_MAX_COMPS];
  std::vector<CgGroupHost> cg;

  // scratch
  double *tb = nullptr, *tq = nullptr; size_t t_len = 0;  // template CG: b and q planes
  struct TmplScalars *tmpl_scalars = nullptr;
  double *M = nullptr, *r = nullptr, *d = nullptr, *eta = nullptr;
  size_t M_len = 0, v_len = 0, eta_len = 0;
  int cg_layout = -1;
  double *D = nullptr;  size_t D_len = 0;       // streaming full-sky data
  double *zbuf = nullptr, *ubuf = nullptr; size_t zu_len = 0;
  unsigned char *decisions = nullptr; double *lnl_trace = nullptr; size_t dec_len = 0;
  int dec_mode = 0, dec_nsample = 0;            // 1 full-sky, 2 per-pixel
  double *stage = nullptr; size_t stage_len = 0; // device staging for strided host copies
  double *partials = nullptr; unsigned int *tickets = nullptr;
  int grid_cap = 0;
  double *sums_local = nullptr, *gathered = nullptr, *gathered_buf = nullptr;
  CgScalars *cg_scalars = nullptr;
  MhScalars *mh_scalars = nullptr;
  void *pinned = nullptr;  // small pinned buffer for scalar read-back
  std::vector<double> last_trace;

  // statistics cache (DESIGN.md "One statistics pass per Gibbs iteration"): `version` counts changes of
  // the model state (amplitudes, indices, maps, gains).  The per-plane sufficient statistics of the
  // next full-sky draw, gathered when compute_chisq is asked for right after an amplitude draw, serve
  // that chi-square, the draw itself and the chi-square after it.
  int stat_cache = 1;            // DANG_OPT_STAT_CACHE
  uint64_t version = 1;
  int last_mutation = 0;         // 1: amplitude draw, 2: spectral-parameter draw, 0: anything else
  bool stat_valid = false;
  int stat_ic = -1, stat_nind = -1, stat_S = 0, stat_plane[2] = {0, 0}, stat_cnt = 0;
  uint64_t stat_version = 0;
  double *stat_buf = nullptr;    // [nranks][stat_cnt] gathered statistics
  bool chisq_valid = false;
  uint64_t chisq_version = 0;
  int chisq_lo = 0, chisq_hi = 0;
  double chisq_vals[4] = {0, 0, 0, 0};
  int64_t n_unmasked = -1;       // all ranks; -1: not counted yet
  // chain continuity of full-sky draws: after a statistics-form draw of (ic, nind) over planes that were already
  // tabulated, the device holds the next chain's start (MhScalars::sample, s0) and the refreshed SED table, so the
  // next draw of the same index skips the chain-start kernels and the table kernel.  idx_epoch counts every other
  // change to index maps / bands / component constants.
  uint64_t idx_epoch = 1;
  bool fs_cont_valid = false;
  int fs_cont_ic = -1, fs_cont_nind = -1, fs_cont_S = 0, fs_cont_plane0 = -1;
  uint64_t fs_cont_epoch = 0;
  bool fs_tab_written = false;   // set by sample_fullsky for dang_gpu_sample_index: table already refreshed on the device

  // comm
  int nranks = 1, rank = 0;
  nccl_comm_t comm = nullptr;
  // NVLink mailboxes (CUDA IPC); peer.nranks == 1 until dang_gpu_comm_open_peers succeeds
  Mail *mailbox = nullptr;
  void *peer_ptr[DG_MAX_RANKS] = {};
  PeerComm peer{};
  volatile int *peer_error_host = nullptr;  // host view of peer.error (mapped pinned memory)
  bool use_mail = false;

  // instrumentation
  int64_t launches = 0;
  KStat kstat[DANG_K_COUNT + DANG_TL_EXTRA];
  cudaEvent_t tl_base = nullptr;  // origin of the event log
  std::vector<TlRec> tl;
  cudaEvent_t ev[16] = {};
};
// ---------------------------------------------------------------- helpers
inline void set_device(dang_gpu *h) { CK(cudaSetDevice(h->device)); }

template <typename T>
void dfree(T *&p) {
  if (p) cudaFree(p);
  p = nullptr;
}

inline void ensure(double *&buf, size_t &len, size_t need) {
  if (len >= need) return;
  if (buf) CK(cudaFree(buf));
  buf = nullptr;
  CK(cudaMalloc(&buf, need * sizeof(double)));
  len = need;
}

// Persistent-style launch: exactly as many blocks as are resident at once (blocks/SM from the
// occupancy calculator x SM count), or fewer when the work is small; grid-stride loops inside.
template <typename K>
int occ_grid(dang_gpu *h, K kernel, int64_t work, int threads, size_t smem = 0) {
  int per_sm = 0;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem));
  if (per_sm < 1) per_sm = 1;
  int64_t need = (work + threads - 1) / threads;
  int64_t cap = (int64_t)h->num_sms * per_sm;
  if (cap > h->grid_cap) cap = h->grid_cap;
  int64_t g = need < cap ? need : cap;
  return (int)(g < 1 ? 1 : g);
}

inline int grid_for(dang_gpu *h, int64_t work, int threads, int blocks_per_sm) {
  int64_t need = (work + threads - 1) / threads;
  int64_t cap = (int64_t)h->num_sms * blocks_per_sm;
  if (cap > h->grid_cap) cap = h->grid_cap;
  int64_t g = need < cap ? need : cap;
  return (int)(g < 1 ? 1 : g);
}

struct KTimer {
  dang_gpu *h;
  int kid;
  double bytes;
  bool deferred;
  cudaEvent_t a = nullptr, b = nullptr;
  // deferred: the launch is booked later with commit(), once the host knows whether the kernel did any work
  // (a CG pass enqueued after convergence returns at once: it must not be credited with a pass's bytes)
  KTimer(dang_gpu *h_, int kid_, double bytes_, bool deferred_ = false) : h(h_), kid(kid_), bytes(bytes_), deferred(deferred_) {
    h->launches++;
    if (!deferred) {
      h->kstat[kid].launches++;
      h->kstat[kid].bytes += bytes;
    }
    if (h->profile) {
      CK(cudaEventCreate(&a));
      CK(cudaEventCreate(&b));
      CK(cudaEventRecord(a, h->stream));
    }
  }
  void done() {
    CK(cudaGetLastError());
    if (h->profile) {
      CK(cudaEventRecord(b, h->stream));
      if (!deferred) h->kstat[kid].pending.emplace_back(a, b);
    }
  }
  // book a deferred launch: under `kid` with its bytes if it worked, else as a scalar (early-exit) launch
  void commit(bool worked) {
    const int k = worked ? kid : DANG_K_SCALAR;
    h->kstat[k].launches++;
    if (worked) h->kstat[k].bytes += bytes;
    if (a) h->kstat[k].pending.emplace_back(a, b);
  }
};

// Event log (DANG_OPT_PROFILE): while profiling, every timed launch -- and every staged copy on the h2d / d2h
// streams (kinds DANG_K_COUNT + ...) -- also lands in h->tl with its start / end relative to h->tl_base, so a run
// can be laid out as a per-stream timeline (dang_gpu_timeline) without nsys.
inline void resolve_stats(dang_gpu *h) {
  CK(cudaStreamSynchronize(h->stream));
  CK(cudaStreamSynchronize(h->d2h_stream));
  CK(cudaStreamSynchronize(h->h2d_stream));
  for (int k = 0; k < DANG_K_COUNT + DANG_TL_EXTRA; k++) {
    for (auto &pr : h->kstat[k].pending) {
      float ms = 0;
      CK(cudaEventElapsedTime(&ms, pr.first, pr.second));
      h->kstat[k].ms += ms;
      if (h->tl_base && h->tl.size() < 100000) {
        float t0 = 0;
        if (cudaEventElapsedTime(&t0, h->tl_base, pr.first) == cudaSuccess) h->tl.push_back(TlRec{k, 1e3 * t0, 1e3 * (t0 + ms)});
      }
      cudaEventDestroy(pr.first);
      cudaEventDestroy(pr.second);
    }
    h->kstat[k].pending.clear();
  }
}

// a staged copy on one of the side streams, logged like a kernel launch while profiling
struct CopyTimer {
  dang_gpu *h;
  int kind;
  cudaStream_t st;
  cudaEvent_t a = nullptr, b = nullptr;
  CopyTimer(dang_gpu *h_, int kind_, cudaStream_t st_) : h(h_), kind(kind_), st(st_) {
    if (h->profile) {
      CK(cudaEventCreate(&a));
      CK(cudaEventCreate(&b));
      CK(cudaEventRecord(a, st));
    }
  }
  void done() {
    if (h->profile) {
      CK(cudaEventRecord(b, st));
      h->kstat[kind].launches++;
      h->kstat[kind].pending.emplace_back(a, b);
    }
  }
};

// host (npix-strided, full sky) <-> device (Ppad-strided slice) plane copies
inline void h2d_planes(dang_gpu *h, double *dst, const double *src, int nplanes) {
  CK(cudaMemcpy2DAsync(dst, h->Ppad * sizeof(double), src + h->lo, h->npix * sizeof(double),
                       h->P * sizeof(double), nplanes, cudaMemcpyHostToDevice, h->stream));
}
inline void d2h_planes(dang_gpu *h, double *dst, const double *src, int nplanes) {
  CK(cudaMemcpy2DAsync(dst + h->lo, h->npix * sizeof(double), src, h->Ppad * sizeof(double),
                       h->P * sizeof(double), nplanes, cudaMemcpyDeviceToHost, h->stream));
}

// ln(a/b) as a double-double from an extended-precision logarithm
inline void dd_log_ratio(double a, double b, double &hi, double &lo) {
  const long double L = logl((long double)a / (long double)b);
  hi = (double)L;
  lo = (double)(L - (long double)hi);
}
// Compulsory traffic (doubles) of one persistent solve that ran n_pass passes with prediction k_pred: every sweep
// reads M, r (and d after the first checkpoint); checkpoint passes write r, d; sweeps that carry x read it and write
// x + the amplitude planes; a closing sweep follows when x is behind the last pass.
inline double cg_solve_bytes(int n_pass, int k_pred, int ckpt_m, int T, int C, double vs) {
  double per_el = 0.0;
  int x_at = 0;
  for (int pn = 1; pn <= n_pass; pn++) {
    const bool store = pn % ckpt_m == 0, with_x = store || pn >= k_pred;
    per_el += T + C + (pn > ckpt_m ? C : 0) + (store ? 2.0 * C : 0.0) + (with_x ? 3.0 * C : 0.0);
    if (with_x) x_at = pn;
  }
  if (n_pass > x_at) per_el += T + C + (n_pass > ckpt_m ? C : 0) + 3.0 * C;
  return vs * per_el;
}
// device -> pinned host (h->pinned) for small results, stream ordered, bypassing the copy engine
inline void readback(dang_gpu *h, void *dst_pinned, const void *src_dev, size_t bytes) {
  if (bytes % 4 != 0) fail(DANG_GPU_EINVAL, "readback of %zu bytes", bytes);
  readback_kernel<<<1, 128, 0, h->stream>>>((unsigned int *)dst_pinned, (const unsigned int *)src_dev, (int)(bytes / 4));
  CK(cudaGetLastError());
  h->launches++;  // (dang_gpu_launch_count: every kernel of this library counts)
}

// Deferred amplitude downloads (DANG_OPT_DEFER_D2H).  A bulk device->host copy saturates the host link, and while
// it does the GPU's command fetches queue behind it: every small launch of the spectral-parameter block then costs
// 50-70 us instead of 5-10 (profiles/r02_timeline_*.md).  So dang_gpu_get_amplitude_async only RECORDS the request;
// the copy is issued by the next amplitude draw right behind its solve kernel -- one long launch that needs nothing
// from the host for hundreds of microseconds -- reading the buffer the draw just swapped out (CompHost::amp_alt).
// Anything else that needs the data or the buffer (dang_gpu_download_wait, in-place writers) issues them at once.
struct DeferredD2H {
  int ic;
  const double *src;  // device planes (the component's amplitude buffer at request time)
  double *dst;        // host array (full-sky addressing)
  int k_lo, k_hi;
};
void issue_deferred_d2h(dang_gpu *h, cudaEvent_t after);  // dang_gpu.cu
void chisq_of_statistics(const dang_gpu *h, const double *hp, int cnt, int S, const int *plane, double out4[4]);  // host_mh_fs.cu

// anything that overwrites c.amp in place waits for a download that may still be reading it
inline void amp_write_barrier(dang_gpu *h, CompHost &c) {
  if (!h->deferred.empty()) {
    CK(cudaEventRecord(h->ev_compute, h->stream));
    issue_deferred_d2h(h, h->ev_compute);
  }
  if (c.read_pending) {
    CK(cudaStreamWaitEvent(h->stream, c.ev_read, 0));
    c.read_pending = false;
  }
}

// defined in dang_gpu.cu
void upload_bandpasses(dang_gpu *h);
ModelView model_view(dang_gpu *h);
void gather(dang_gpu *h, int cnt);  // exchange `cnt` doubles of sums_local between ranks -> h->gathered [rank][cnt]

inline int flag_planes(int flag, int plane[2]) {  // 0-based planes; returns S
  if (flag & 8) {
    plane[0] = 1;
    plane[1] = 2;
    return 2;
  }
  int k = 0;
  if (flag & 1) k = 0;
  else if (flag & 2) k = 1;
  else if (flag & 4) k = 2;
  else fail(DANG_GPU_EUNSUPPORTED, "pol flag %d (T+Q+U) is dead code in the reference (SURVEY Q2)", flag);
  plane[0] = plane[1] = k;
  return 1;
}

inline double bytes_w(double n) { return n * 8.0; }

// record that index map (c, l) on plane k is known constant (val = 0) or varying (val = 1)
inline void set_nonuni(dang_gpu *h, int c, int k, int l, int val) {
  const int m = (c * 3 + k) * DG_MAXIND + l;
  CK(cudaMemsetAsync((char *)h->tab + offsetof(SedTable, nonuni) + m * sizeof(int), val ? 1 : 0, sizeof(int), h->stream));
  h->nonuni_host[c * 3 + k][l] = val ? 1 : 0;
  h->check_mask &= ~(1ull << m);
  h->tab_dirty = true;
}

inline bool comp_uniform(const dang_gpu *h, int c, int k) { return h->uni_host[c * 3 + k] != 0; }
inline void idx_changed(dang_gpu *h) { h->idx_epoch++; }  // an index map / band / component constant changed outside a full-sky draw

// ---------------------------------------------------------------- entry points of the other translation units
void cg_solve(dang_gpu *h, int cg_group, int flag_n, int ml_mode, const double *eta, uint64_t seed,
              int *n_iter, double *delta_final);                                   // host_cg.cu
int64_t unmasked_count(dang_gpu *h);  // dang_gpu.cu: unmasked pixels over all ranks (cached)
inline void touch(dang_gpu *h, int what = 0) {  // the model state changed
  h->version++;
  h->last_mutation = what;
}
// host_mh_fs.cu: serve compute_chisq from the sufficient statistics of the upcoming full-sky draw
bool chisq_from_statistics(dang_gpu *h, int pol_lo, int pol_hi, double out4[4]);
void prefetch_statistics(dang_gpu *h);  // host_mh_fs.cu: statistics pass of the upcoming full-sky draw, enqueued ahead of time
void cg_solve_template(dang_gpu *h, CgGroupHost &g, int flag_n, int ml_mode, const double *eta, uint64_t seed,
                       const int *comps, int C, const int *borders, int nb, const int *og, int nog, int *n_iter,
                       double *delta_final);                                       // host_tmpl.cu
void monopole_to_offset(dang_gpu *h, const CompHost &c);                          // dang_gpu.cu
void upload_tamp(dang_gpu *h, CompHost &c);                                        // dang_gpu.cu
void run_chisq(dang_gpu *h, int pol_lo, int pol_hi, double *sky, double *res, double *chi_map,
               double out4[4]);                                                    // host_data.cu
void mh_view(dang_gpu *h, int ic, int nind, int map_n, int nsample, int ml_mode, MhView &mh);  // host_mh_fs.cu
void ensure_zu(dang_gpu *h, size_t n);
void ensure_decisions(dang_gpu *h, size_t n);
void sample_perpixel(dang_gpu *h, MhView &mh, const double *z, const double *u, uint64_t seed, double *accept);  // host_mh_pp.cu
void launch_perpixel_pix(dang_gpu *h, const ModelView &mv, const MhView &mh, int mode);  // host_mh_ppx.cu
// fp64 lane-cooperative per-pixel kernel, one translation unit per bands-per-lane value (host_mh_ppd{2,3,5,8}.cu)
void launch_perpixel_fp64_2(dang_gpu *h, const ModelView &mv, const MhView &mh, int mode, int64_t work, size_t smem);
void launch_perpixel_fp64_3(dang_gpu *h, const ModelView &mv, const MhView &mh, int mode, int64_t work, size_t smem);
void launch_perpixel_fp64_5(dang_gpu *h, const ModelView &mv, const MhView &mh, int mode, int64_t work, size_t smem);
void launch_perpixel_fp64_8(dang_gpu *h, const ModelView &mv, const MhView &mh, int mode, int64_t work, size_t smem);
void launch_perpixel_fast(dang_gpu *h, const ModelView &mv, const MhView &mh, int bpl, int mode, int64_t work,
                          size_t smem);                                            // host_mh_ppf.cu
void launch_perpixel_split(dang_gpu *h, const ModelView &mv, MhView &mh, int bpl, int mode, int64_t work);  // host_mh_ppf.cu
void sample_fullsky(dang_gpu *h, MhView &mh, const double *z, const double *u, uint64_t seed, double *accept);   // host_mh_fs.cu
void tune_fullsky(dang_gpu *h, int ic, int nind, MhView &mh, const double *z, const double *u, uint64_t seed,
                  int max_blocks, int *blocks_run, double *step_size, const double *start);  // host_mh_fs.cu
