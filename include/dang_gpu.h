/*
 * dang_gpu.h -- C ABI of the B200-native replacement for hermda02/dang's Gibbs hot path.
 *
 * The reference has no plugin/FFI layer; its "interface" for this path is the set of Fortran
 * call sites in the Gibbs loop (src/dang.f90:87-126) and the three objects they take
 * (dang_params, dang_data, dang_comps).  Each entry point below names the reference routine
 * or call site it replaces; fortran/dang_gpu_mod.f90 is the iso_c_binding shim a maintainer
 * adds (INTEGRATION.md), and dang_b200/engine.py is the same binding through ctypes.
 *
 * Conventions
 *   - real(dp) <-> double, integer(i4b) <-> int32_t (int), logical(lgt) <-> int (0/1).
 *   - Host arrays are the reference's own allocatables, passed by c_loc, in Fortran layout
 *     A(0:npix-1, nmaps [, nbands]) == C [band][stokes][pix]; FULL-SKY size even when the
 *     handle owns only a pixel slice.  Host memory stays owned by the caller; every call copies.
 *   - Plane / map numbers are the reference's 1-based values (1=I, 2=Q, 3=U; map_n -1 = Q+U);
 *     pol flags are the bit flags of return_poltype_flag (src/dang_util_mod.f90:228-292);
 *     component / band / index / cg-group numbers are 0-based except `cg_group`, which is the
 *     value of COMP_CG_GROUPnn (1-based) as stored in c%cg_group.
 *   - One handle == one process == one GPU == one contiguous RING-ordered pixel range
 *     [pix_lo, pix_hi).  Multi-GPU runs use one handle per rank plus dang_gpu_comm_init; the
 *     only cross-rank traffic is the CG / lnL / chi-square scalars (NCCL all-gather).
 *   - Every function returns 0 on success.  On failure it returns a DANG_GPU_E* code and
 *     dang_gpu_last_error() holds the message; the shim prints it and STOPs, mirroring the
 *     reference's `write(*,*) ...; stop` convention (e.g. src/dang_cg_mod.f90:97-101).
 *     There is no CPU fallback anywhere in the library.
 *   - Not thread-safe per handle; call from outside any OpenMP region.
 */
#ifndef DANG_GPU_H
#define DANG_GPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dang_gpu dang_gpu_t;

enum {
  DANG_GPU_OK = 0,
  DANG_GPU_EINVAL = 1,      /* bad argument                                   */
  DANG_GPU_ECUDA = 2,       /* CUDA runtime error (no device, OOM, launch...) */
  DANG_GPU_EUNSUPPORTED = 3,/* valid in the reference, not built yet (DESIGN.md "Out of scope") */
  DANG_GPU_ENCCL = 4,       /* NCCL could not be loaded / failed              */
  DANG_GPU_ESTATE = 5       /* call order violated (e.g. solve before upload) */
};

/* c%type, src/dang_component_mod.f90:791-809 */
enum { DANG_COMP_POWERLAW = 1, DANG_COMP_MBB = 2, DANG_COMP_FREEFREE = 3, DANG_COMP_LOGNORMAL = 4, DANG_COMP_CMB = 5,
       DANG_COMP_TEMPLATE = 6, DANG_COMP_T_CMB = 7, DANG_COMP_MONOPOLE = 8, DANG_COMP_HI_FIT = 9 };
/* c%lnl_type, src/dang_sample_mod.f90:249-258 */
enum { DANG_LNL_CHISQ = 0, DANG_LNL_MARGINAL = 1, DANG_LNL_PRIOR = 2 };
/* c%prior_type, src/dang_sample_mod.f90:260-266 */
enum { DANG_PRIOR_UNIFORM = 0, DANG_PRIOR_GAUSSIAN = 1, DANG_PRIOR_JEFFREYS = 2 };
/* ml_mode, src/dang_cg_mod.f90:254,265 */
enum { DANG_ML_OPTIMIZE = 0, DANG_ML_SAMPLE = 1 };
/* c%index_mode, src/dang_component_mod.f90:166-170 */
enum { DANG_INDEX_FULLSKY = 1, DANG_INDEX_PERPIXEL = 2 };

/* options for dang_gpu_set_option */
enum {
  /* 0 (default): reproduce compute_sample_vector's indexing (SURVEY Q1: every diffuse
   * component writes slot 1, src/dang_cg_mod.f90:1033-1034).  1: offset per component. */
  DANG_OPT_FIX_SAMPLE_VECTOR = 1,
  /* CG iteration form.  0 (default): one fused pass per iteration (d.q from a recurrence);
   * 1: classic two-pass form with d.q summed directly, as cg_search writes it (:296-305). */
  DANG_OPT_CG_TWO_PASS = 2,
  /* Full-sky Metropolis likelihood.  0 (default): per-band sufficient statistics gathered in
   * one pass, proposals evaluated from them; 1: stream the maps once per proposal, the
   * reference's own structure (src/dang_sample_mod.f90:282-324). */
  DANG_OPT_FULLSKY_STREAM = 3,
  /* 1: record CUDA events around every kernel launch (dang_gpu_kernel_stats). */
  DANG_OPT_PROFILE = 4,
  /* CG iterations enqueued between host checks of the convergence flag (default 8). */
  DANG_OPT_CG_CHUNK = 5,
  /* 1: per-pixel chains record every decision / lnL (dang_gpu_get_decisions); parity tests. */
  DANG_OPT_RECORD_DECISIONS = 6,
  /* Per-pixel Metropolis.  0 (default): four lanes share a pixel's bands, lnL summed in a fixed
   * tree order; 1: one thread per pixel, lnL accumulated in exactly the reference's order
   * (Stokes outer, band inner, src/dang_lnl_mod.f90:172-176) -- several times slower. */
  DANG_OPT_PERPIXEL_SERIAL = 7,
  /* CG state checkpoint interval m of the recompute form (default 8): a pass re-runs the
   * block-local recurrences since the last checkpoint in registers instead of reading and
   * writing r, d, x every iteration; 0 selects the streaming form (one r/d/x update per pass). */
  DANG_OPT_CG_CHECKPOINT = 8,
  /* 1: K1 streams sig/rms through a shared-memory ring filled by the TMA bulk-copy engine
   * (cp.async.bulk + mbarrier) when all SEDs are tabulated; 0 (default): 16-byte LDG loads, which
   * measured faster (285 vs 313 us at nside 512: K1 is issue-bound, not load-bound). */
  DANG_OPT_TMA = 9,
  /* 1 (default): dang_gpu_chisq called right after an amplitude draw gathers the per-plane sufficient
   * statistics of the full-sky draw that follows (when the next index in sample_spectral_parameters'
   * order is a full-sky chisq draw over the same planes); that chi-square, the draw, and the chi-square
   * after the draw are then all served by ONE pass over the maps.  0: every call streams the maps. */
  DANG_OPT_STAT_CACHE = 10,
  /* MB of the CG block matrices M marked persisting in L2 (cudaAccessPolicyWindow) for the passes of a
   * solve; the rest of the CG state streams.  0: off. */
  DANG_OPT_L2_PERSIST_MB = 11,
  /* Per-pixel Metropolis, delta bands, power-law / mbb indices.  Screened forms: every proposal is evaluated
   * in single precision from the chi-square DIFFERENCE about the chain's current point (the data term
   * cancels analytically) with a running error bound; a proposal whose |diff - ln u| is inside the bound
   * is re-evaluated in fp64 with the arithmetic of the fp64 kernel, so the decisions are the fp64
   * kernel's (dang_gpu_perpixel_stats counts the fallbacks).
   *   3 (default): one thread per pixel, two numbers of state per band in shared memory (csrc/kernels_mh_pix.cuh;
   *      6.3 ms per index at nside 512 x 20 bands);
   *   1: four lanes per pixel, residuals per band and Stokes parameter in registers (csrc/kernels_mh_fast.cuh; 7.9 ms);
   *   2: form 1 split into deviate / state / chain kernels -- a measured experiment, slower (10.1 ms);
   *   0: every proposal in fp64 (9.4 ms). */
  DANG_OPT_PERPIXEL_FAST = 12,
  /* Per-pixel Metropolis with tabulated bandpasses, power-law beta / mbb beta.  1 (default): the bandpass-
   * integrated SED of a proposal comes from a 9-term moment series about the chain's first point (the n_bp
   * exponentials are evaluated once per pixel and band instead of once per proposal; remainder < 3e-15);
   * 0: every proposal sums the bandpass (evaluate_powerlaw / evaluate_mbb as written). */
  DANG_OPT_PERPIXEL_BP_SERIES = 13,
  /* Tabulated bandpasses are handed to the device as the n-point Gauss quadrature of the discrete measure
   * {ln(nu0_i / nu_c), tau0_i} (default n = 8; 0: the table itself).  The rule reproduces the table's sum for
   * every polynomial in ln nu up to degree 2n-1 while costing n instead of n_bp transcendentals per band
   * (DESIGN.md 4.2).  A band gets a rule only where it reproduces the n_bp-term sums of evaluate_powerlaw /
   * evaluate_mbb / ... of every component on the handle to 1e-14 relative (n, n + 4, ... nodes are tried up to
   * n_bp / 2; dang_gpu_band_samples reports the outcome).  Bands with negative weights or a half-width above 0.25 in
   * ln(nu), and bands no rule passes for, keep their table. */
  DANG_OPT_BP_QUADRATURE = 14,
  /* 1 (default): the whole loop of cg_search (src/dang_cg_mod.f90:293-314) runs as ONE persistent, cooperatively
   * launched kernel -- one sweep of the checkpointed-recompute form per CG iteration, a grid barrier and (on
   * several GPUs) the NVLink mailbox exchange between sweeps, unpack_amplitudes folded into the predicted last
   * sweep -- instead of one launch per iteration.  Same operations in the same order (bit-identical results).
   * Needs the recompute form (DANG_OPT_CG_CHECKPOINT > 0) and one rank or mailboxes; 0: one launch per pass. */
  DANG_OPT_CG_PERSISTENT = 15,
  /* 1 (default): the two passes over sig / rms of a configuration with tabulated SEDs (K1 = rhs + blocks, and the
   * full-sky sufficient statistics) prefetch through per-thread three-stage cp.async rings in shared memory, two band
   * batches ahead of the arithmetic (csrc/kernels_stream.cuh); 0: the 16-byte LDG forms (csrc/kernels_uni.cuh).
   * Same arithmetic; sums agree to rounding (the grid sizes differ). */
  DANG_OPT_STREAM_RING = 16,
  /* 1 (default): dang_gpu_get_amplitude_async records the request and the NEXT amplitude draw issues the copy right
   * behind its solve kernel (from the buffer it swapped out), so the bulk transfer overlaps one long launch instead of
   * the launch-heavy spectral-parameter block: a saturated host link delays the GPU's command fetches, which makes
   * every small kernel behind it cost 50-70 us (profiles/).  dang_gpu_download_wait and in-place writers issue pending
   * requests at once.  0: the copy starts as soon as the compute stream reaches the request. */
  DANG_OPT_DEFER_D2H = 17,
  /* 1: deferred scalars.  The reference's loop prints n_iter / chi-square / accept after each block
   * (write_stats_to_term, src/dang.f90:100-104), and by default every call here waits for the device to hand those
   * numbers back: three host round trips per Gibbs iteration, each leaving the GPU idle for 15-25 us (more on several
   * GPUs).  With this option dang_gpu_cg_solve (persistent form, one solve per iteration), dang_gpu_chisq (when the
   * draw's statistics serve it) and full-sky dang_gpu_sample_index (statistics form) only ENQUEUE their kernels and
   * return n_iter = -1 / NaN; dang_gpu_iteration_mark snapshots the device-side results at that point of the stream
   * and dang_gpu_iteration_scalars returns them later -- typically one iteration behind, so the device never waits
   * for the host.  The kernels, their order and every result are identical to the default mode's; calls that are
   * not covered keep returning their values directly.  0 (default): every call returns its own numbers. */
  DANG_OPT_DEFER_SCALARS = 18
};

/* ---- lifetime: after initialize_cg_groups, src/dang.f90:71-75; mpi_finalize, :127 ---- */
int dang_gpu_create(int device, int nside, int64_t npix, int nmaps, int nbands, int ncomp,
                    int64_t pix_lo, int64_t pix_hi, dang_gpu_t **h);
int dang_gpu_destroy(dang_gpu_t *h);
const char *dang_gpu_last_error(const dang_gpu_t *h); /* h may be NULL: last create() error */
int dang_gpu_set_option(dang_gpu_t *h, int option, double value);
int dang_gpu_sync(dang_gpu_t *h);

/* ---- multi-GPU: replaces the reference's unused MPI (src/dang_util_mod.f90:48-57) ----
 * Rank 0 calls dang_gpu_comm_unique_id and broadcasts the 128 bytes with whatever the host
 * has (MPI_Bcast in Fortran, torch.distributed here); then every rank calls comm_init. */
int dang_gpu_comm_unique_id(char id[128]);
int dang_gpu_comm_init(dang_gpu_t *h, int nranks, int rank, const char id[128]);
/* Optional NVLink fast path for the scalar exchanges (one process per GPU on one node): every
 * rank exports its mailbox (64-byte CUDA IPC handle), the host all-gathers the handles
 * (rank-major, nranks*64 bytes) and every rank opens them.  From then on the exchanges are peer
 * stores + flag waits inside the compute kernels instead of NCCL calls; a CG iteration on N GPUs
 * is a single kernel launch.  dang_gpu_comm_check reports a peer that stopped answering. */
int dang_gpu_comm_ipc_handle(dang_gpu_t *h, char handle[64]);
int dang_gpu_comm_open_peers(dang_gpu_t *h, const char *handles);
int dang_gpu_comm_check(dang_gpu_t *h);
/* instrumentation: latency of one in-kernel scalar exchange of `cnt` doubles (1..32) between all ranks over the NVLink
 * mailboxes, averaged over `reps` back-to-back exchanges by one warp (every rank must call it) */
int dang_gpu_comm_probe(dang_gpu_t *h, int reps, int cnt, double *us_per_exchange);

/* ---- bp(j): type bandinfo, src/dang_bp_mod.f90:7-15 (as left by init_bp_mod :19-60) ----
 * nu_c [Hz]; n_bp == 0 <=> bp%id == 'delta'; nu0 [Hz]; tau0 already normalised (:62-81). */
int dang_gpu_set_band(dang_gpu_t *h, int band, double nu_c_hz, int n_bp, const double *nu0_hz,
                      const double *tau0);

/* ---- ddata: sig_map, rms_map, masks(:,1), gain, offset, src/dang_data_mod.f90:23-34 ----
 * Call after initialize_data_module (:68-86) and again after swap_cg_maps (dang.f90:92-97). */
int dang_gpu_upload_maps(dang_gpu_t *h, const double *sig_map, const double *rms_map,
                         const double *mask, const double *gain, const double *offset);
int dang_gpu_set_gain_offset(dang_gpu_t *h, const double *gain, const double *offset);
/* Ensembles of independent chains on one GPU (BASELINE config c5): `h` uses the device copies of
 * sig_map / rms_map / masks that `src` uploaded instead of holding its own (64 chains at nside 512
 * share 1.2 GB of maps and keep ~0.9 GB of state each).  `src` must outlive `h`. */
int dang_gpu_share_maps(dang_gpu_t *h, dang_gpu_t *src);

/* ---- component_list(ic): type dang_comps, src/dang_component_mod.f90:12-55 ---- */
int dang_gpu_set_component(dang_gpu_t *h, int ic, int type, const char *label,
                           double nu_ref_hz, int cg_group, int sample_amplitude,
                           const double *amplitude /* (npix,nmaps) */,
                           const double *indices /* (npix,nmaps,nindices) */);
/* type 'template' (src/dang_component_mod.f90:536-577), after dang_gpu_set_component(type = DANG_COMP_TEMPLATE,
 * amplitude = indices = NULL): template_map = c%template (npix,nmaps), already divided by temp_norm (:574-577);
 * template_amplitudes = c%template_amplitudes (nbands,nmaps) or NULL for zeros; corr[nbands] = c%corr; nfit = c%nfit.
 * eval_signal of such a component is template_amplitudes(band,plane) * template(pix,plane) everywhere (chi-square,
 * sky model, the data of the Metropolis draws); in a CG group it adds `nfit` scalar unknowns, one per fitted band
 * (compute_rhs :560-587, compute_Ax :745-768,:867-893, compute_sample_vector :1077-1096, unpack :1374-1392).
 * Built for CG_POLTYPE = Q+U with one template per group placed after the group's diffuse components. */
int dang_gpu_set_template(dang_gpu_t *h, int ic, const double *template_map, const double *template_amplitudes,
                          const int *corr, int nfit);
/* The same call completes the two Stokes-I "border" types (after dang_gpu_set_component with that type):
 *   'monopole' (src/dang_component_mod.f90:579-597): template_map = NULL (the constructor's map: 1 on plane 1, 0 on
 *     the polarisation planes); eval_signal = template_amplitudes(band, 1).  update_sky_model leaves it out of the sky
 *     model and copies the amplitudes into ddata%offset instead (src/dang_data_mod.f90:357-361): the library does the
 *     same to its offsets whenever the amplitudes change.
 *   'hi_fit' (:599-700): template_map = the HI template (NOT normalised), indices (npix,nmaps,1) = T_d given to
 *     dang_gpu_set_component; eval_signal = template_amplitudes(band, k) * template(pix, k) * B_nu(T_d) in RJ units
 *     (evaluate_hi_fit :850-884).
 * In a CG group both add one scalar unknown per fitted band like a template, on plane 1 only: CG_POLTYPE = T
 * (compute_rhs :522-559, compute_Ax :717-744 / :833-866, compute_sample_vector :1044-1067).
 * 'T_cmb' (:430 ff., evaluate_T_cmb :815-848) needs no second call: eval_signal = eval_sed = B_nu(T) in RJ units, no
 * amplitude.  After its index has been drawn the host updates the global T_CMB as sample_spectral_parameters does
 * (src/dang_sample_mod.f90:76-78) with dang_gpu_set_t_cmb; the 'cmb' SED (1 / a2t) follows it. */
int dang_gpu_set_t_cmb(dang_gpu_t *h, double t_cmb);
int dang_gpu_get_template_amplitudes(dang_gpu_t *h, int ic, double *template_amplitudes); /* -> (nbands,nmaps) */
int dang_gpu_set_index(dang_gpu_t *h, int ic, int nind, int sample_index, int index_mode,
                       int lnl_type, int prior_type, const double gauss_prior[2],
                       const double uni_prior[2], double step_size, int sample_nside,
                       const int *pol_flags, int nflag);
int dang_gpu_set_amplitude(dang_gpu_t *h, int ic, const double *amplitude);
int dang_gpu_set_indices(dang_gpu_t *h, int ic, const double *indices);
int dang_gpu_get_amplitude(dang_gpu_t *h, int ic, double *amplitude); /* -> c%amplitude */
int dang_gpu_get_indices(dang_gpu_t *h, int ic, double *indices);     /* -> c%indices   */
/* The value every pixel of plane map_n of c%indices(:,:,nind) holds after a full-sky draw (the reference
 * assigns the chain's final sample to the whole plane, src/dang_sample_mod.f90:329,483): 8 bytes instead of
 * a map download; the shim fills c%indices(:,map_n,nind) with it.  DANG_GPU_ESTATE if the plane varies. */
int dang_gpu_get_index_fullsky(dang_gpu_t *h, int ic, int nind, int map_n, double *value);
int dang_gpu_get_step_size(dang_gpu_t *h, int ic, int nind, double *step_size);

/* ---- cg_groups(i): constructor_cg, src/dang_cg_mod.f90:57-120 ---- */
int dang_gpu_set_cg_group(dang_gpu_t *h, int cg_group, int i_max, double converge,
                          const int *pol_flags, int nflag);

/* ---- amplitude draw: compute_rhs + cg_search + unpack_amplitudes for one (group, flag),
 * src/dang_cg_mod.f90:167-169 (bodies :326-596, :179-324, :598-911, :913-1100, :1284-1396).
 * eta: the S*npix standard normals cg_search draws (:256-262), full-sky, [stokes][pix];
 * NULL => generated on the device from `seed` (Philox4x32-10, DESIGN.md "RNG").
 * n_iter: final value of the reference's loop counter i; delta_final: last sum(r*r). */
int dang_gpu_cg_solve(dang_gpu_t *h, int cg_group, int flag_n, int ml_mode, const double *eta,
                      uint64_t seed, int *n_iter, double *delta_final);
/* per-iteration delta trace of the last solve (delta after init, then after each pass) */
int dang_gpu_cg_trace(dang_gpu_t *h, double *delta, int max_len, int *len);
/* the saved solution vector self%x of one (group, flag), full-sky layout [comp][stokes][pix] */
int dang_gpu_get_cg_x(dang_gpu_t *h, int cg_group, int flag_n, double *x);

/* ---- spectral-parameter draw: sample_index_mh(ddata,c,nind,map_n),
 * src/dang_sample_mod.f90:88-485 (+ update_sample_model :520-568, evaluate_lnL etc. in
 * src/dang_lnl_mod.f90, priors src/dang_util_mod.f90:112-121).
 * z, u: injected deviates, slot-indexed (a slot is used only if the reference would draw it):
 *   full-sky: z[l], u[l], l < nsample;  per-pixel: z[l*npix + pix], u[l*npix + pix] (full sky).
 *   NULL => device RNG from `seed`.
 * accept: number of accepted proposals (summed over this handle's pixels in per-pixel mode). */
int dang_gpu_sample_index(dang_gpu_t *h, int ic, int nind, int map_n, int nsample, int ml_mode,
                          const double *z, const double *u, uint64_t seed, double *accept);
/* decisions of the last dang_gpu_sample_index call (parity instrumentation):
 * 0 rejected, 1 accepted, 2 out of prior bounds, 3 masked; full-sky: nsample entries,
 * per-pixel: [l*npix + pix] for this handle's pixels (other entries untouched).
 * lnl: lnl_new of every evaluated proposal, same indexing (may be NULL). */
int dang_gpu_get_decisions(dang_gpu_t *h, unsigned char *decisions, double *lnl);
/* screening statistics of the last per-pixel dang_gpu_sample_index (all ranks): proposals decided by the
 * fp64 fallback; in record mode (option 6) also the proposals whose screened difference broke its error
 * bound or whose certain decision differed from the fp64 one (must be 0). */
int dang_gpu_perpixel_stats(dang_gpu_t *h, double *fallbacks, double *violations);
/* tune_spectral_parameter_length, src/dang_sample_mod.f90:623-717 (full-sky chain).
 * z, u hold max_blocks*nsample slots, [block*nsample + l]. */
int dang_gpu_tune_index(dang_gpu_t *h, int ic, int nind, int map_n, int nsample, int ml_mode,
                        const double *z, const double *u, uint64_t seed, int max_blocks,
                        int *blocks_run, double *step_size);

/* ---- chi-square: update_sky_model + compute_chisq, src/dang_data_mod.f90:339-396,494-526
 * (called from write_stats_to_term :528-570).  pol_lo..pol_hi = ddata%pol_type(1)..(size).
 * chisq_planes[nmaps]: un-normalised sum over this handle's... all ranks' pixels of
 * chi_map(:,k) (already divided by nbands, :523); n_unmasked: unmasked pixel count (all ranks).
 * The host forms chisq = sum(chisq_planes)/nump with its own nump (SURVEY Q9). */
int dang_gpu_chisq(dang_gpu_t *h, int pol_lo, int pol_hi, double *chisq_planes,
                   int64_t *n_unmasked);
/* sky_model, res_map (npix,nmaps,nbands) and chi_map (npix,nmaps): only this handle's pixels
 * are written; any pointer may be NULL.  Needed only when write_maps is due (dang.f90:119). */
int dang_gpu_get_sky_model(dang_gpu_t *h, int pol_lo, int pol_hi, double *sky_model,
                           double *res_map, double *chi_map);
/* ---- band calibration: fit_band_gain(ddata, map_n, band), src/dang_sample_mod.f90:570-621
 * (called for Stokes I by sample_calibrators :487-518).  z: the N(0,1) deviate of :615 or NULL
 * (device stream `seed`).  The fitted gain replaces the handle's gain(band) and is returned. */
int dang_gpu_fit_band_gain(dang_gpu_t *h, int map_n, int band, int ml_mode, const double *z,
                           uint64_t seed, double *gain);

/* ---- resolution changes of the low-resolution sampling branch (src/dang_sample_mod.f90:204-217, 480) as standalone
 * operators on full-sky RING maps in host memory, (npix, nmaps) each:
 *   kind 0  udgrade_ring   HEALPix-F90 udgrade_nr as published: RING -> NESTED, average the (nside_in/nside_out)^2
 *                          children (bad pixels -1.6375e30 skipped, all bad -> bad) or copy the parent, NESTED -> RING
 *   kind 1  udgrade_rms    src/dang_util_mod.f90:341-356: sqrt(udgrade_ring(rms^2)) * nside_out / nside_in
 *   kind 2  udgrade_mask   :358-376: udgrade_ring, then (when degrading) 0 below `threshold`, 1 otherwise
 * dang_gpu_sample_index itself still requires sample_nside == nside (DESIGN.md section 7). */
int dang_gpu_udgrade(dang_gpu_t *h, int kind, const double *in, int nside_in, double *out, int nside_out, int nmaps,
                     double threshold);

/* ---- deferred scalars (DANG_OPT_DEFER_SCALARS): the terminal line of src/dang.f90:100-104 one iteration late ----
 * _mark: snapshot what the deferred calls since the previous mark left on the device (solve count / residual,
 *   statistics rows, chain outcome) into one of four pinned slots, stream ordered, no host wait; returns a ticket.
 *   At most four tickets may be outstanding (unread).  A slot holds ONE full-sky draw: a second full-sky
 *   dang_gpu_sample_index (or a dang_gpu_tune_index) before the next _mark would overwrite the first draw's outcome
 *   and fails with DANG_GPU_ESTATE instead -- mark after each full-sky draw (index poltype 'Q,U', or several
 *   full-sky indices per iteration).
 * _scalars: wait for that snapshot only and decode it.  n_iter / delta_final: the amplitude draw's (as
 *   dang_gpu_cg_solve); chisq_after_amplitudes[nmaps]: the dang_gpu_chisq call that followed it; accept /
 *   index_value: the full-sky draw's acceptance ratio and final value; chisq_after_index[nmaps]: the dang_gpu_chisq
 *   call after the draw.  Entries nothing was deferred for come back as -1 / NaN; any pointer may be NULL.
 *   Tickets should be read in issue order (the traffic accounting of dang_gpu_kernel_stats assumes it). */
int dang_gpu_iteration_mark(dang_gpu_t *h, int64_t *ticket);
int dang_gpu_iteration_scalars(dang_gpu_t *h, int64_t ticket, int *n_iter, double *delta_final,
                               double *chisq_after_amplitudes, double *accept, double *index_value,
                               double *chisq_after_index);

/* mask_avg(c%indices(:,map_n,nind), masks(:,1)), src/dang_util_mod.f90:186-206 */
int dang_gpu_index_mean(dang_gpu_t *h, int ic, int nind, int map_n, double *mean);

/* ---- output / input staging (SURVEY 8f-4): copies on dedicated streams that overlap later calls.
 * dang_gpu_get_*_async start a device->host copy of planes k_lo..k_hi (1-based) of c%amplitude /
 * c%indices(:,:,nind) into the caller's arrays (same addressing as the synchronous getters) and
 * return at once; the library orders them against its own later writes (a solve's unpack waits
 * for a pending amplitude download, a sampler for a pending index download).
 * dang_gpu_download_wait blocks until every pending download has landed.
 * dang_gpu_stage_eta uploads the S*npix normals of a coming dang_gpu_cg_solve while other work runs;
 * that solve is then called with eta == NULL and uses the staged deviates (once).  Up to two solves'
 * deviates can be staged (first in, first out), so the upload for solve k+1 overlaps solve k.
 * Host buffers should be pinned (dang_gpu_host_alloc) or the copies serialise. */
int dang_gpu_get_amplitude_async(dang_gpu_t *h, int ic, int k_lo, int k_hi, double *amplitude);
int dang_gpu_get_indices_async(dang_gpu_t *h, int ic, int nind, int k_lo, int k_hi, double *indices);
int dang_gpu_download_wait(dang_gpu_t *h);
int dang_gpu_stage_eta(dang_gpu_t *h, const double *eta, int nplanes);

/* The n-point Gauss quadrature the library substitutes for a tabulated bandpass (DANG_OPT_BP_QUADRATURE):
 * nodes nu_q [Hz] and weights w_q with sum_q w_q g(nu_q) == sum_i tau0_i g(nu0_i) for every g polynomial in
 * ln(nu) up to degree 2 nq - 1.  Host-only (no device needed); DANG_GPU_EUNSUPPORTED when no rule is built
 * (n_bp <= 2 nq, negative weights, half-width above 0.25 in ln nu).  This is the rule before a handle verifies it
 * against its components' SEDs (dang_gpu_band_samples). */
int dang_gpu_bandpass_quadrature(double nu_c_hz, int n_bp, const double *nu0_hz, const double *tau0, int nq,
                                 double *nu_q_hz, double *w_q);
/* Samples of `band` that the device's bandpass-integrated SEDs sum over: 0 for a delta band, n_bp where the
 * table is kept, otherwise the node count of the Gauss rule that replaced it.  A rule is used only where it
 * reproduces the table's sum of every SED on the handle to 1e-14 relative at 7 points per index spanning the
 * uniform-prior box of each sampled index and the range of the index maps uploaded (and at the T_CMB values 'cmb'
 * can meet) -- a sampled check, not a bound between the points; it has DANG_OPT_BP_QUADRATURE nodes, or 4, 8, ...
 * more (up to n_bp / 2) where that is not enough.  Read-only. */
int dang_gpu_band_samples(dang_gpu_t *h, int band, int *n_samples);

/* ---- posterior summaries on the device.  NOT in the reference: its users set OUTPUT_ITER = 1, let write_maps write
 * every sample and compute mean / std maps offline.  Here the chain stays resident and running moments accumulate
 * next to it; the host downloads only the summaries, when write_maps is due (INTEGRATION.md).
 * _begin: allocate and zero the accumulators of the kinds in `what` (a set of DANG_POST_* bits, fixed until _end or
 *   the next _begin, which starts again from zero), n = 0.  pol_lo..pol_hi: the range dang_gpu_get_sky_model takes,
 *   used by CHI_MAP / RESIDUAL (ignored otherwise).
 *     AMPLITUDE            c%amplitude of every component with a map amplitude (not template / monopole / hi_fit,
 *                          whose map is fixed, nor T_cmb, which has none)
 *     INDICES              every index map of every component, per-pixel or full-sky
 *     CHI_MAP, RESIDUAL    the chi_map / res_map dang_gpu_get_sky_model(h, pol_lo, pol_hi, ...) would return
 *     TEMPLATE_AMPLITUDES  template_amplitudes of template / monopole / hi_fit components
 * _accumulate: add the current state as one sample; stream ordered, no host wait.  Per element, n the count after
 *   adding x, every operation rounded separately (no FMA):  d = x - mean;  mean += d / n;  M2 += d * (x - mean).
 * _get: synchronous; mean and stddev = sqrt(M2 / (n - 1)) (NaN for n < 2; stddev may be NULL) in the layout of the
 *   getter of that quantity: (npix,nmaps) for AMPLITUDE of component ic, INDICES of (ic, nind) and CHI_MAP,
 *   (npix,nmaps,nbands) for RESIDUAL, (nbands,nmaps) for TEMPLATE_AMPLITUDES of ic; only this handle's pixels are
 *   written.  ic / nind are ignored by the kinds that do not use them.
 * _get / _accumulate / _end before _begin, or _get of a kind not begun: DANG_GPU_ESTATE; a bad ic, nind or kind:
 *   DANG_GPU_EINVAL.  Nothing crosses ranks: each rank accumulates its own pixels.
 * _rhat: the classic Gelman-Rubin statistic (not split-chain) per element over the m handles hs[0..m-1] (same device,
 *   same pixel range, the kind begun and the same n >= 2 on each; otherwise DANG_GPU_EINVAL, message on hs[0]),
 *   in _get's layout.  Sums run over the chains in the order given, each operation rounded separately:
 *   W = (sum M2_c / (n-1)) / m,  mu = (sum mean_c) / m,  B/n = (sum (mean_c - mu)^2) / (m - 1),
 *   R = sqrt((((n-1)/n) W + B/n) / W);  NaN where W = 0 (e.g. masked pixels of the chi-square map).
 * _begin_batched: _begin plus batch-means accumulators for every kind in `what` (24 more bytes per element), so
 *   that _ess can estimate how many independent samples the mean rests on.  batch_len = b >= 1, else
 *   DANG_GPU_EINVAL.  _accumulate, _get, _end and _rhat behave as after _begin (_get returns the same mean and
 *   stddev bit for bit).  Sample n at position j = ((n-1) mod b) + 1 of its batch, each operation rounded separately:
 *   {mean, M2} as above;  bsum = (j == 1) ? x : bsum + x;  if j == b:  k = n / b,  y = bsum / b,  d = y - bmean,
 *   bmean += d / k,  bM2 += d * (y - bmean).  A partial batch at the end is left out of {bmean, bM2}.
 * _ess: batch-means effective sample size and Monte Carlo standard error of the posterior mean per element, over
 *   m >= 1 handles hs[0..m-1] (m = 1: one chain; m > 1 pools the chains), in _get's layout; ess or mcse may be
 *   NULL, not both.  Synchronous.  Every handle needs the same device and pixel range, the kind begun batched, the
 *   same n and b, and K = n / b >= 2 complete batches; otherwise DANG_GPU_EINVAL, message on hs[0].  A handle not
 *   begun, or begun without batches: DANG_GPU_ESTATE.  Sums run over the chains in the order given:
 *     mu  = (sum mean_c) / m,   A  = sum M2_c,   D  = sum (mean_c - mu) (mean_c - mu),    s2   = (A + n D) / (m n - 1)
 *     mub = (sum bmean_c) / m,  Ab = sum bM2_c,  Db = sum (bmean_c - mub) (bmean_c - mub), sig2 = b (Ab + K Db) / (m K - 1)
 *     ess = (m n) s2 / sig2,    mcse = sqrt(sig2 / (m n));  both NaN where sig2 = 0.
 *   sig2 estimates the asymptotic variance of the chain mean (Flegal & Jones 2010).  For m > 1, chains that
 *   disagree inflate Db and the ESS collapses.  ESS is not capped at m n.  Choose b near sqrt(planned n), with
 *   K >= 20 for a stable estimate; the library does not choose b. */
enum { DANG_POST_AMPLITUDE = 1, DANG_POST_INDICES = 2, DANG_POST_CHI_MAP = 4,
       DANG_POST_RESIDUAL = 8, DANG_POST_TEMPLATE_AMPLITUDES = 16 };
int dang_gpu_posterior_begin(dang_gpu_t *h, int what, int pol_lo, int pol_hi);
int dang_gpu_posterior_begin_batched(dang_gpu_t *h, int what, int pol_lo, int pol_hi, int batch_len);
int dang_gpu_posterior_accumulate(dang_gpu_t *h);
int dang_gpu_posterior_get(dang_gpu_t *h, int kind, int ic, int nind, double *mean, double *stddev, int64_t *n);
int dang_gpu_posterior_end(dang_gpu_t *h);
int dang_gpu_posterior_rhat(dang_gpu_t *const *hs, int m, int kind, int ic, int nind, double *rhat);
int dang_gpu_posterior_ess(dang_gpu_t *const *hs, int m, int kind, int ic, int nind, double *ess, double *mcse);

/* ---- instrumentation (bench.py) ---- */
int dang_gpu_host_alloc(void **ptr, uint64_t bytes); /* pinned host memory */
int dang_gpu_host_free(void *ptr);
int dang_gpu_event_record(dang_gpu_t *h, int slot);  /* slot 0..15, on the handle's stream */
int dang_gpu_event_elapsed_ms(dang_gpu_t *h, int slot_a, int slot_b, float *ms);
int dang_gpu_launch_count(dang_gpu_t *h, int64_t *launches, int reset);
/* per-kernel totals since the last reset (needs DANG_OPT_PROFILE): kernel ids in dang_gpu.h
 * order below; bytes = algorithmic HBM bytes of those launches (DESIGN.md "Kernels"). */
enum {
  DANG_K_RHS_BLOCKS = 0, DANG_K_CG_PASS = 1, DANG_K_CG_DQ = 2, DANG_K_CG_UPDATE = 3,
  DANG_K_CHISQ = 4, DANG_K_SKYMODEL = 5, DANG_K_MH_DATA = 6, DANG_K_MH_FULLSKY_LNL = 7,
  DANG_K_MH_SUFFSTAT = 8, DANG_K_MH_PERPIXEL = 9, DANG_K_SCALAR = 10, DANG_K_CG_FIXUP = 11,
  DANG_K_COUNT = 12
};
int dang_gpu_kernel_stats(dang_gpu_t *h, int kernel, int64_t *launches, double *total_ms,
                          double *bytes, int reset);
const char *dang_gpu_kernel_name(int kernel);
/* Event log of everything launched since DANG_OPT_PROFILE was switched on: kernel launches on the compute stream
 * (kind = DANG_K_*) and staged copies on the copy streams (kind = DANG_K_COUNT + 0 h2d eta, + 1 d2h amplitude,
 * + 2 d2h indices), start / end in microseconds from that moment, sorted by start.  The per-stream timeline of
 * profiles/ (no nsys in this image). */
int dang_gpu_timeline(dang_gpu_t *h, int max_n, int *n, int *kind, double *t0_us, double *t1_us);

#ifdef __cplusplus
}
#endif
#endif
