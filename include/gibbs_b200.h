/*
 * gibbs_b200.h -- C ABI of libgibbs_b200.so: the B200 (sm_100a) implementation of the
 * constrained-realization + C_l-sampling Gibbs step of Gabriel-Ducrocq/GibbsSampler.
 *
 * The reference has no C ABI at this boundary (SURVEY.md 8b): its samplers call healpy, a
 * forked qcinv, scipy.stats and the Cython module variance_expension.pyx directly from
 * Python.  Each entry point below names the reference call it replaces (file:line in the
 * reference tree).  Conventions:
 *   - every pointer argument is a CALLER-OWNED DEVICE pointer unless the name ends in _host;
 *   - sizes are passed explicitly or fixed by the plan (nside, lmax);
 *   - every call takes the CUDA stream to run on as `void* stream` (a cudaStream_t, NULL =
 *     default stream) and is asynchronous with respect to the host unless stated otherwise;
 *   - the return value is a status (GS_OK = 0, negative = error); no exception crosses the
 *     ABI; gs_last_error_string() describes the last failure on the calling thread;
 *   - a plan is used by one host thread at a time; distinct plans / streams are independent.
 *
 * Layouts (bit-exact integer conventions of the reference, SURVEY.md 8):
 *   GS_ALM_COMPLEX  healpy m-major complex128, idx(l,m) = m(2L+1-m)/2 + l
 *                   (variance_expension.pyx:19, utils.py:123); (L+1)(L+2)/2 complex numbers.
 *   GS_ALM_REAL     the reference's "real convention" (utils.py:49-76,
 *                   variance_expension.pyx:65-100): r[i] = Re a_i for i <= L (m = 0) and
 *                   r[2i-(L+1)] = sqrt2 Re a_i, r[2i-(L+1)+1] = sqrt2 Im a_i for i > L;
 *                   (L+1)^2 doubles.
 *   maps            HEALPix RING order, float64, Npix = 12 nside^2.
 */
#ifndef GIBBS_B200_H
#define GIBBS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GS_OK 0
#define GS_E_BADARG (-1)
#define GS_E_CUDA (-2)
#define GS_E_NOTCONVERGED (-3)
#define GS_E_NCCL (-4)
#define GS_E_NOMEM (-5)

#define GS_ALM_COMPLEX 0
#define GS_ALM_REAL 1

typedef struct gs_plan gs_plan;

/* ---- library / plan ------------------------------------------------------------------ */
const char* gs_last_error_string(void);
int gs_version(void);

/* Builds ring geometry, FP64 recurrence tables and ring-FFT tables for (nside, lmax) on CUDA
 * device `device` (-1 = current).  Replaces the implicit healpy/libsharp geometry + plan that
 * hp.alm2map / hp.map2alm rebuild on every call.  Synchronous. */
int gs_plan_create(gs_plan** plan, int nside, int lmax, int device);
int gs_plan_destroy(gs_plan* plan);
/* Chain batches (SURVEY.md 8b: gs_plan_create(nside, lmax, n_chain, ...); BASELINE config #5 "batched over chains"): sizes the
 * plan's ring-spectra and partial-sum workspaces for n_chain (1 or 2) right-hand sides per launch.  The reference runs one
 * chain per process (SLURM array, job-script.sh:6), every chain repeating the Legendre recurrences of hp.alm2map / hp.map2alm;
 * a batch shares them.  Unsharded plans only; called implicitly by the *_batch entry points. */
int gs_plan_reserve_chains(gs_plan* plan, int n_chain);
int gs_plan_nside(const gs_plan* plan);
int gs_plan_lmax(const gs_plan* plan);
int64_t gs_plan_npix(const gs_plan* plan);
int64_t gs_plan_nalm(const gs_plan* plan);   /* (L+1)(L+2)/2 */
int64_t gs_plan_nreal(const gs_plan* plan);  /* (L+1)^2      */

/* ---- spherical-harmonic transforms ----------------------------------------------------- */
/* hp.alm2map(alm, nside, lmax)  (NonCenteredGibbs.py:179,204; ClsSampler.py:108 via
 * synthesis_hp, variance_expension.pyx:114-123).  `fl` (nullable, L+1 doubles) multiplies a_lm
 * by fl[l] first, i.e. a fused hp.almxfl(alm, fl). */
int gs_alm2map_spin0(gs_plan* plan, const double* alm, int layout, const double* fl, double* map,
                     void* stream);

/* (Q, U) of hp.alm2map([0, almE, almB], pol=True)  (CenteredGibbs.py:505-508, 698-699,
 * 751-753; NonCenteredGibbs.py:350-351; qcinv opfilt_pp.fwd_op).  HEALPix convention
 * Q +- iU = sum -(E +- iB) (+-2)Y_lm. */
int gs_alm2map_spin2(gs_plan* plan, const double* almE, const double* almB, int layout,
                     const double* fl, double* mapQ, double* mapU, void* stream);

/* hp.map2alm(map, lmax, iter=iter, use_weights=False) (utils.py:104; CenteredGibbs.py:209).
 * adjoint != 0 computes the plain transpose A^T f = (Npix/4pi) map2alm_iter0(f) instead
 * (utils.adjoint_synthesis_hp with iter = 0; config.py:72) and ignores `iter`.
 * `pixw` (nullable, Npix doubles) multiplies the map first (fused N^-1); `fl` (nullable)
 * multiplies the result by fl[l].  iter > 0 uses plan-owned scratch. */
int gs_map2alm_spin0(gs_plan* plan, const double* map, const double* pixw, int iter, int adjoint,
                     const double* fl, double* alm, int layout, void* stream);

/* (E, B) of hp.map2alm([0, Q, U], lmax, pol=True, iter=iter)  (CenteredGibbs.py:298-299, 513,
 * 717-719; utils.py:89 with iter=3; NonCenteredGibbs.py:155). */
int gs_map2alm_spin2(gs_plan* plan, const double* mapQ, const double* mapU, const double* pixw,
                     int iter, int adjoint, const double* fl, double* almE, double* almB,
                     int layout, void* stream);

/* n_chain independent right-hand sides per call (hp.alm2map / hp.map2alm of n_chain chains that the reference runs as
 * separate processes): chain c reads / writes alm + c alm_stride and map + c map_stride (strides in doubles; spin 0 ignores
 * almB / mapU).  Chains are transformed two per launch and the two share ONE Legendre recurrence per (ring pair, m)
 * (4 + 8 K DFMA per ring pair and multipole for K = 2 chains instead of 12 K).  Results equal n_chain single calls.
 * gs_map2alm_batch is map2alm(iter = 0) (adjoint != 0: A^T, weight 1); pixw (nullable) multiplies the pixels of every chain. */
int gs_alm2map_batch(gs_plan* plan, int spin, int n_chain, const double* almE, const double* almB,
                     int64_t alm_stride, int layout, const double* fl, double* mapQ, double* mapU,
                     int64_t map_stride, void* stream);
int gs_map2alm_batch(gs_plan* plan, int spin, int n_chain, const double* mapQ, const double* mapU,
                     int64_t map_stride, const double* pixw, int adjoint, const double* fl, double* almE,
                     double* almB, int64_t alm_stride, int layout, void* stream);

/* ---- harmonic-space array utilities (all device pointers) ------------------------------ */
/* utils.real_to_complex (utils.py:49-60) / variance_expension.real_to_complex (.pyx:84-100) */
int gs_real_to_complex(const double* real_alm, double* complex_alm, int lmax, void* stream);
/* utils.complex_to_real (utils.py:63-76) / variance_expension.complex_to_real (.pyx:65-81) */
int gs_complex_to_real(const double* complex_alm, double* real_alm, int lmax, void* stream);
/* Expansion of a per-l array x[0..L] to the real alm layout ((L+1)^2 doubles).
 *   mode 0: x_l                     GibbsSampler.compute_bl_map (GibbsSampler.py:64-74), config.py:75-84
 *   mode 1: C_l = D_l 2pi/(l(l+1))  utils.generate_var_cl (utils.py:114-147), .pyx:8-33 (l = 0 copied)
 *   mode 2: 1/C_l where C_l != 0    CenteredGibbs.py:463-466
 *   mode 3: sqrt(C_l)               ASIS.py:198-203
 *   mode 4: sqrt(1/C_l) where != 0  CenteredGibbs.py:478-479, NonCenteredGibbs.py:192-194 */
int gs_expand_per_l(const double* x, int lmax, int mode, double* out, void* stream);
/* utils.unfold_bins (utils.py:150-162): np.repeat(binned, diff(bins)); bins has nbins + 1
 * ascending int32 edges, out has nout = bins[nbins] - bins[0] entries. */
int gs_unfold_bins(const double* binned, const int* bins, int nbins, double* out, int nout,
                   void* stream);
/* hp.almxfl(alm, fl) (CenteredGibbs.py:304-305, 514-515); out may alias alm. */
int gs_almxfl(const double* alm, int layout, int lmax, const double* fl, double* out, void* stream);
/* hp.alm2cl(alm, lmax) (CenteredGibbs.py:30, 61): (|a_l0|^2 + 2 sum_m |a_lm|^2) / (2l+1). */
int gs_alm2cl(const double* alm, int layout, int lmax, double* cl, void* stream);

/* Same as gs_alm2map_spin2 with separate per-l filters for E and B: the non-centred likelihood
 * synthesises A (b_l sqrt(C^EE_l) s^E, b_l sqrt(C^BB_l) s^B)  (NonCenteredGibbs.py:346-351). */
int gs_alm2map_spin2_fl2(gs_plan* plan, const double* almE, const double* almB, int layout,
                         const double* flE, const double* flB, double* mapQ, double* mapU,
                         void* stream);

/* ---- constrained realization (masked sky: PCG; full sky isotropic: direct) ------------- */
/* Right-hand side of Q x = b for the polarised masked-sky draw (CenteredGibbs.py:469-483):
 *   b = B A^T N^-1 d + B (Npix/4pi) map2alm_{iter=fluct_iter}(N^-1/2 xi_pix) + C^-1/2 xi_alm,
 * RNG order of the reference: xi_Q[Npix], xi_U[Npix], xi_E[(L+1)^2], xi_B[(L+1)^2] (standard
 * normals supplied by the caller: injected numpy draws for parity, gs_randn in production).
 * The data term is what the forked qcinv adds in multigrid_chain.sample (opfilt_pp.calc_prep) and
 * equals second_part_grad (CenteredGibbs.py:298-308); pass it precomputed in bdata_E/B (real
 * layout) or pass d_Q/d_U to have it computed.  dl_* are unbinned D_l (L+1), bl the beam b_l,
 * inv_noise = mask / noise_pol and sqrt_inv_noise its square root (Npix).  fluct_iter = 3
 * reproduces utils.adjoint_synthesis_hp (utils.py:89). */
int gs_cr_rhs_pol(gs_plan* plan, const double* dl_EE, const double* dl_BB, const double* bl,
                  const double* inv_noise, const double* sqrt_inv_noise, const double* bdata_E,
                  const double* bdata_B, const double* d_Q, const double* d_U, const double* xi_Q,
                  const double* xi_U, const double* xi_E, const double* xi_B, int fluct_iter,
                  double* rhs_E, double* rhs_B, void* stream);

/* Preconditioned conjugate gradient for Q x = b, Q = C^-1 + B A^T N^-1 A B, real alm layout:
 * qcinv.multigrid.multigrid_chain(opfilt_pp, [[0, ["diag_cl"], lmax, nside, itermax, eps, tr_cg,
 * cache_mem()]], ...) as configured at ConstrainedRealization.py:40-41 / CenteredGibbs.py:280-282
 * and run at CenteredGibbs.py:486-488.  Preconditioner 1/(1/C_l + b_l^2 sum(N^-1)/(4pi))
 * (ninv_sum_over_4pi = sum(inv_noise)/(4 pi)); stop when <r,r> <= eps^2 <r0,r0> or after itermax
 * iterations.  warm_start = 0 starts from x = 0 (x_E/x_B are overwritten), otherwise from the
 * contents of x_E/x_B (RJPO, CenteredGibbs.py:642-651).  The convergence flag lives on the device;
 * the host polls it every `check_every` iterations (<= 0: 8).  Synchronous on return:
 * *n_iter_out / *resid_out (host, nullable) receive the iteration count and |r|/|r0|.
 * Returns GS_E_NOTCONVERGED if itermax was hit first (x holds the last iterate). */
int gs_cr_pcg_pol(gs_plan* plan, const double* dl_EE, const double* dl_BB, const double* bl,
                  const double* inv_noise, double ninv_sum_over_4pi, const double* rhs_E,
                  const double* rhs_B, double* x_E, double* x_B, int warm_start, double eps,
                  int itermax, int check_every, int* n_iter_out, double* resid_out, void* stream);

/* gs_cr_pcg_pol (cold start) for n_chain = 1 or 2 independent chains on the same data (what n_chain processes of the
 * reference each do at CenteredGibbs.py:486-488): chain c uses dl_* + c (L+1) and rhs / x + c stride (doubles).  While both
 * chains iterate, every mat-vec is one chain-batched launch per stage (shared Legendre recurrence); alpha, beta and the
 * stopping rule stay per chain, so each chain runs the iterations of its own single solve (n_iter_out[c], resid_out[c]). */
int gs_cr_pcg_pol_batch(gs_plan* plan, int n_chain, const double* dl_EE, const double* dl_BB, const double* bl,
                        const double* inv_noise, double ninv_sum_over_4pi, const double* rhs_E,
                        const double* rhs_B, double* x_E, double* x_B, int64_t stride, double eps, int itermax,
                        int check_every, int* n_iter_out, double* resid_out, void* stream);

/* 1 (default): unsharded gs_cr_pcg_* solves capture the `check_every` iterations between two polls of the convergence flag in a
 * CUDA graph (once per solve, on a stream owned by the plan and ordered after `stream`) and replay it; 0: plain launches.
 * Returns the previous setting.  Same arithmetic either way. */
int gs_set_pcg_graph(int on);

/* y = Q x (qcinv opfilt_pp.fwd_op; CenteredGibbs.py:629, 653). */
int gs_cr_apply_q_pol(gs_plan* plan, const double* dl_EE, const double* dl_BB, const double* bl,
                      const double* inv_noise, const double* x_E, const double* x_B, double* y_E,
                      double* y_B, void* stream);

/* Temperature twins of the three entry points above (one spin-0 field; qcinv.opfilt_tt chain of
 * ConstrainedRealization.py:40-41, run at CenteredGibbs.py:141-165 and NonCenteredGibbs.py:57-72).  RNG order
 * of the reference for the right-hand side: xi_alm[(L+1)^2] first, then xi_pix[Npix] (CenteredGibbs.py:145-147).
 * bdata = B A^T N^-1 d is what qcinv adds inside chain.sample; pass it precomputed or pass d. */
int gs_cr_rhs_tt(gs_plan* plan, const double* dl_TT, const double* bl, const double* inv_noise,
                 const double* sqrt_inv_noise, const double* bdata, const double* d, const double* xi_alm,
                 const double* xi_pix, int fluct_iter, double* rhs, void* stream);
int gs_cr_pcg_tt(gs_plan* plan, const double* dl_TT, const double* bl, const double* inv_noise,
                 double ninv_sum_over_4pi, const double* rhs, double* x, int warm_start, double eps, int itermax,
                 int check_every, int* n_iter_out, double* resid_out, void* stream);
int gs_cr_apply_q_tt(gs_plan* plan, const double* dl_TT, const double* bl, const double* inv_noise,
                     const double* x, double* y, void* stream);

/* Joint T/E/B twins: T and E coupled through C^TE on a cut sky (qcinv's joint T+P filter, opfilt_tp upstream, not vendored;
 * the reference only has the full-sky per-coefficient 3x3 solve, utils.compute_inverse_and_cholesky + utils.matrix_product, see
 * gs_inv_chol_3x3).  Real layout, one beam bl for the three fields (the reference applies the temperature beam to E/B):
 *   Q = C^-1 + B A^T N^-1 A B,  C_l = [[TT, TE, 0], [TE, EE, 0], [0, 0, BB]] on (T_j, E_j, B_j) of every coefficient j,
 *   A B x = (alm2map_spin0(b x_T), alm2map_spin2(b x_E, b x_B)),  N^-1 = diag(inv_noise_T, inv_noise_P, inv_noise_P) on (I, Q, U).
 * inv_noise_X = mask_X / noise_X (Npix each; the T and P masks may differ), dl_* unbinned D_l (L+1).
 * Right-hand side  b = B A^T N^-1 d + B (Npix/4pi) map2alm_{iter=fluct_iter}(N^-1/2 xi_pix) + F xi_alm  with F = L^-T on (T, E),
 * C^{TE block}_l = L L^T the lower Cholesky factor, and F = 1/sqrt(C^BB) on B, so F F^T = C^-1: with fluct_iter = 0 the
 * right-hand side has covariance Q and x = Q^-1 b is an exact draw of s | C, d.  RNG order: xi_I, xi_Q, xi_U [Npix each], then
 * xi_T, xi_E, xi_B [(L+1)^2 each] (pixel draws first, as in the polarised reference, CenteredGibbs.py:472-479).  The data terms
 * B A^T N^-1 d are passed precomputed (bdata_T/E/B) or computed from d_I, d_Q, d_U.
 * PCG: preconditioner diag_cl per l, M_l = (C_l^-1 + diag(b_l^2 nT, b_l^2 nP, b_l^2 nP))^-1 with nX = sum(inv_noise_X)/(4 pi)
 * (a 2x2 inverse on (T, E), a scalar on B); stop when <r,r> <= eps^2 <r0,r0> with the sums over all three fields (qcinv
 * monitor_basic).  Singular blocks follow safe_inv: at l < 2 (D_l = 0) C^-1 = 0, a block with C^TE = 0 inverts field by
 * field; where C^TE != 0 the TE block must be positive definite.  warm_start, check_every, the outputs and GS_E_NOTCONVERGED as
 * in gs_cr_pcg_pol.  Unsharded plans only (GS_E_BADARG otherwise). */
int gs_cr_rhs_teb(gs_plan* plan, const double* dl_TT, const double* dl_TE, const double* dl_EE, const double* dl_BB,
                  const double* bl, const double* inv_noise_T, const double* sqrt_inv_noise_T, const double* inv_noise_P,
                  const double* sqrt_inv_noise_P, const double* bdata_T, const double* bdata_E, const double* bdata_B,
                  const double* d_I, const double* d_Q, const double* d_U, const double* xi_I, const double* xi_Q,
                  const double* xi_U, const double* xi_T, const double* xi_E, const double* xi_B, int fluct_iter,
                  double* rhs_T, double* rhs_E, double* rhs_B, void* stream);
int gs_cr_pcg_teb(gs_plan* plan, const double* dl_TT, const double* dl_TE, const double* dl_EE, const double* dl_BB,
                  const double* bl, const double* inv_noise_T, const double* inv_noise_P, double ninvT_sum_over_4pi,
                  double ninvP_sum_over_4pi, const double* rhs_T, const double* rhs_E, const double* rhs_B, double* x_T,
                  double* x_E, double* x_B, int warm_start, double eps, int itermax, int check_every, int* n_iter_out,
                  double* resid_out, void* stream);
int gs_cr_apply_q_teb(gs_plan* plan, const double* dl_TT, const double* dl_TE, const double* dl_EE, const double* dl_BB,
                      const double* bl, const double* inv_noise_T, const double* inv_noise_P, const double* x_T,
                      const double* x_E, const double* x_B, double* y_T, double* y_E, double* y_B, void* stream);

/* Diagonal draw for full sky + isotropic noise, one field, real layout, w = Npix/(noise 4 pi):
 *   mode 0 centred     (CenteredGibbs.py:317-353): sigma = 1/(w b^2 + 1/C), s = sigma b w d + xi sqrt(sigma)
 *   mode 1 non-centred (NonCenteredGibbs.py:138-176, all_sph): sigma = 1/(1 + b^2 C w),
 *                      s = sigma sqrt(C) b w d + xi sqrt(sigma)
 * dl = unbinned D_l, d_alm = data in harmonic space (pix_map["EE"/"BB"]), xi = standard normals. */
int gs_cr_direct(const double* dl, const double* bl, const double* d_alm, const double* xi,
                 double npix_over_noise_4pi, int lmax, int mode, double* out, void* stream);

/* Diagonal TT draw, full sky + isotropic noise, with data and noise fluctuation entering as pixel-space adjoints
 * (utils.adjoint_synthesis_hp, iter = 3): bsum = b_l A^T N^-1 d + b_l A^T N^-1/2 xi_pix in the real layout,
 * w = Npix / (noise 4 pi).  l < l_cut centred (CenteredConstrainedRealization.sample_no_mask, CenteredGibbs.py:100-127),
 * l >= l_cut non-centred (NonCenteredConstrainedRealization.sample_no_mask, NonCenteredGibbs.py:22-41); 0 < l_cut <= L
 * is the recovered TT PNCPConstrainedRealization.sample (PNCP.cpython-38.pyc), which zeroes l < 2 (zero_low). */
int gs_cr_direct_pix(const double* dl, const double* bl, const double* bsum, const double* xi,
                     double npix_over_noise_4pi, int lmax, int l_cut, int zero_low, double* out, void* stream);

/* ---- C_l conditional samplers ------------------------------------------------------------ */
/* PolarizedCenteredClsSampler.sample_one_pol / CenteredClsSampler.sample (CenteredGibbs.py:24-79):
 * cl_hat = alm2cl(s) (L+1); bins = nbins + 1 int32 edges; D_bin = beta / Gamma(alpha, 1) with
 * beta = sum_l (2l+1) l (l+1) cl_hat_l / 4pi, alpha = sum_l (2l+1)/2 - 1, alpha[0] := 1, D[:2] := 0.
 * gamma_inject (nullable, nbins): Gamma(alpha,1) variates from the caller (numpy parity); NULL:
 * Marsaglia-Tsang on a Philox4x32-10 stream keyed by (seed, call, bin).  alpha_out / beta_out
 * (nullable, nbins) return the shape / scale per bin. */
int gs_cls_invgamma(const double* cl_hat, const int* bins, int nbins, const double* gamma_inject,
                    uint64_t seed, uint64_t call, double* dl_binned, double* alpha_out,
                    double* beta_out, void* stream);

/* Truncated-normal proposal on [0, inf) around the current binned D_l (ClsSampler.py:79-92,
 * NonCenteredGibbs.py:292-309): dl_new[b] = ppf(u[b-2]; loc = dl_old[b], scale = sqrt(prop_var[b-2]))
 * for b >= 2, dl_new[0] = dl_new[1] = 0.  u: nbins - 2 uniforms. */
int gs_truncnorm_propose(const double* dl_old, const double* prop_var, int nbins, const double* u,
                         double* dl_new, void* stream);
/* out[b] = truncnorm.logpdf(x[b]; a = -from[b]/scale, b = inf, loc = from[b], scale) for b >= 2,
 * 0 for b < 2 (NonCenteredGibbs.py:313-330). */
int gs_truncnorm_logpdf(const double* x, const double* from, const double* prop_var, int nbins,
                        double* out, void* stream);
/* -1/2 sum_p inv_noise_p [(d_Q - m_Q)^2 + (d_U - m_U)^2] -> out[0] (device); d_U = m_U = NULL
 * for temperature (NonCenteredGibbs.py:353-355; ClsSampler.py:107-108).  scratch: 592 doubles. */
int gs_loglik_pix(const double* d_Q, const double* d_U, const double* m_Q, const double* m_U,
                  const double* inv_noise, int64_t npix, double* scratch, double* out, void* stream);
/* compute_log_likelihood_all_sph (NonCenteredGibbs.py:357-377; full sky, isotropic noise, data given in harmonic space):
 * -1/2 weight sum_i [(d_E_i - fl_E[l(i)] s_E_i)^2 + (d_B_i - fl_B[l(i)] s_B_i)^2] -> out[0] (device), i over the real alm
 * layout ((lmax+1)^2 doubles per array), fl_* = b_l sqrt(C_l) per multipole (gs_mwg_filters), weight = N^-1 Npix / 4 pi
 * (NonCenteredGibbs.py:375-377).  scratch: 592 doubles. */
int gs_loglik_alm(const double* d_E, const double* d_B, const double* s_E, const double* s_B, const double* fl_E,
                  const double* fl_B, int lmax, double weight, double* scratch, double* out, void* stream);

/* ---- Metropolis-within-Gibbs on the binned D_l, device resident ---------------------------- */
/* Per-l synthesis filters fl_X[l] = b_l sqrt(C^X_l) of the candidate state = current binned D_l
 * with bins [b_start, b_end) of spectrum pol (0 EE, 1 BB, -1 none) replaced by the proposal; they feed
 * gs_alm2map_spin2_fl2 for the likelihood of NonCenteredGibbs.py:333-355 (unfold_bins +
 * generate_var_cl + bl_map * sqrt(var_cls) fused per l).  l < l_cut keeps fl = b_l (partially
 * non-centred parametrisation, PNCP); pass l_cut = 0 for the fully non-centred sampler. */
int gs_mwg_filters(const double* cur_E, const double* cur_B, const double* prop_E, const double* prop_B,
                   const int* bins_E, int nbins_E, const int* bins_B, int nbins_B, int pol, int b_start,
                   int b_end, const double* bl, int lmax, int l_cut, double* flE, double* flB,
                   void* stream);
/* Accept/reject of one block (NonCenteredGibbs.py:421-442) without leaving the device:
 * log r = sum_{b in block} logr[b] + new_lik - old_lik; if log(u[0]) < log r the block of `cur` is
 * overwritten with the proposal and old_lik[0] = new_lik[0]; accept_out[0] = 0/1. */
int gs_mwg_accept(double* cur, const double* prop, const double* logr, int b_start, int b_end,
                  const double* new_lik, double* old_lik, const double* u, int* accept_out, void* stream);
/* The whole blocked Metropolis sweep of PolarizationNonCenteredClsSampler.sample (NonCenteredGibbs.py:401-445)
 * in one call, using the linearity of the likelihood's synthesis in the per-l filter (NonCenteredGibbs.py:333-355):
 * r = d - A (b sqrt(C) s_nc) is synthesised once, the map changes dM_k of ALL blocks come from one pass of the
 * Legendre recurrence + one batched ring-FFT launch, and each Metropolis test is a fused chi^2 reduction of
 * r - dM_k followed by a device-side accept (cur <- prop on the block, r <- r - dM_k).  Same accept rule, same
 * order (EE blocks then BB blocks, n_iter tests per block) and same consumption of u as the per-block path
 * (gs_mwg_filters + gs_alm2map_spin2_fl2 + gs_loglik_pix + gs_mwg_accept).
 * snc_*: real-layout alm; cur_* (in/out), prop_*, logr_*: binned arrays; bins_*_host[nbins+1], blocks_*_host[nblk+1]:
 * HOST int arrays (blocks index the binned arrays); u / accept_out: (nblk_E + nblk_B) * n_iter entries;
 * loglik_out (nullable, device): final log-likelihood; workspace_bytes: cap of the plan-owned block workspace
 * (<= 0: 8 GiB).  Needs an unsharded plan with NSIDE <= 1024. */
int gs_mwg_sweep_blocks(gs_plan* plan, const double* snc_E, const double* snc_B, double* cur_E, double* cur_B,
                        const double* prop_E, const double* prop_B, const double* logr_E, const double* logr_B,
                        const int* bins_E_host, int nbins_E, const int* bins_B_host, int nbins_B,
                        const int* blocks_E_host, int nblk_E, const int* blocks_B_host, int nblk_B, int n_iter,
                        const double* bl, int l_cut, const double* d_Q, const double* d_U, const double* inv_noise,
                        const double* u, int* accept_out, double* loglik_out, int64_t workspace_bytes, void* stream);
/* out = a * b elementwise (re-centring s = sqrt(C) s_nc, ASIS.py:181-203; NonCenteredGibbs.py:192-194). */
int gs_mul(const double* a, const double* b, double* out, int64_t n, void* stream);

/* ---- auxiliary-variable constrained realization (CenteredGibbs.py:676-825) --------------- */
/* v | s in pixel space, one component: gamma = mu - N^-1, mean = gamma * map (map = A B s),
 * v = mean + alpha (v_io - mean) + sqrt(1 - alpha^2) sqrt(gamma) xi; v_io <- v; out <- v + N^-1 d
 * (the map whose adjoint transform gives the mean of s | v).  alpha = 0: plain Gibbs draw
 * (CenteredGibbs.py:701-705); alpha = -0.995: over-relaxation (CenteredGibbs.py:796-797). */
int gs_aux_v_update(const double* map, const double* inv_noise, const double* d, const double* xi,
                    double mu, double alpha, double* v_io, double* out, int64_t npix, void* stream);
/* s | v in the real alm layout, one spectrum: var = 1/((mu/w) b_l^2 + 1/C_l), mean = var * badj with
 * badj = b_l A^T (v + N^-1 d); s_io <- mean + alpha (s_io - mean) + sqrt(1 - alpha^2) sqrt(var) xi
 * (CenteredGibbs.py:708-725, 763-781). */
int gs_aux_s_update(const double* badj, const double* dl, const double* bl, const double* xi,
                    double mu_over_w, double alpha, int lmax, double* s_io, void* stream);
/* per-l factor of the partially non-centred parametrisation (PNCP): out[l] = 1 for l < l_cut, else
 * sqrt(1/C_l) (mode 0) or sqrt(C_l) (mode 1). */
int gs_pncp_factor(const double* dl, int lmax, int l_cut, int mode, double* out, void* stream);

/* ---- MALA constrained realization (CenteredGibbs.py:494-603), real alm layout ---------------- */
/* sigma = 1/(w b_l^2 + 1/C_l), w = Npix/(noise 4 pi) (CenteredGibbs.py:569-570). */
int gs_mala_sigma(const double* dl, const double* bl, double npix_over_noise_4pi, int lmax, double* out,
                  void* stream);
/* g = bdata - C^-1 s - y with y = B A^T N^-1 A B s (compute_gradient_mala, CenteredGibbs.py:494-520). */
int gs_mala_grad(const double* bdata, const double* invc, const double* s, const double* y, double* g,
                 int64_t n, void* stream);
/* out = s + tau sigma g + sqrt(2 tau sigma) xi (propose_new_mala, CenteredGibbs.py:523-527). */
int gs_mala_propose(const double* s, const double* g, const double* sigma, const double* xi, double tau,
                    double* out, int64_t n, void* stream);
/* out[0] = -1/2 sum (to - from - tau sigma g_from)^2 / (2 tau sigma) (compute_log_proposal, :530-532). */
int gs_mala_logq(const double* to, const double* from, const double* g_from, const double* sigma,
                 double tau, int64_t n, double* scratch, double* out, void* stream);
/* ULA_no_mask for one spectrum (CenteredGibbs.py:355-446: compute_gradient_no_mask :355-377, compute_log_proposal_no_mask
 * :379-392, compute_log_density_no_mask :394-414, proposal and ratio :417-446), full sky + isotropic noise, diagonal in the
 * real layout: s_new = s_old + tau sigma grad + sqrt(2 tau sigma) xi and log_ratio_out[0] = this spectrum's share of the
 * Metropolis log-ratio; d_alm = harmonic-space data (pix_map["EE"/"BB"]); scratch: 592 doubles. */
int gs_ula_nomask(const double* dl, const double* bl, const double* d_alm, const double* s_old, const double* xi,
                  double npix_over_noise_4pi, double tau, int lmax, double* s_new, double* scratch,
                  double* log_ratio_out, void* stream);
/* remove_monopole_dipole_contributions (variance_expension.pyx:103-111): real-layout entries 0, 1, L+1, L+2 := 0, in place. */
int gs_remove_monopole_dipole(double* alm_real, int lmax, void* stream);
/* out[0] = sum a b c (c nullable), fixed summation order; scratch: 592 doubles. */
int gs_dot3(const double* a, const double* b, const double* c, int64_t n, double* scratch, double* out,
            void* stream);

/* ---- random numbers / reductions --------------------------------------------------------- */
/* n standard normals (Philox4x32-10 keyed by (seed, stream_id), Box-Muller); replaces
 * np.random.normal in production runs. */
int gs_randn(double* out, int64_t n, uint64_t seed, uint64_t stream_id, void* stream);
/* n uniforms on (0,1). */
int gs_randu(double* out, int64_t n, uint64_t seed, uint64_t stream_id, void* stream);
/* out[0] = sum(a[0..n)) in a fixed order; scratch: 592 doubles. */
int gs_sum(const double* a, int64_t n, double* scratch, double* out, void* stream);

/* ---- per-multipole 3x3 TT/TE/EE/BB machinery (one thread per l / per coefficient) -----------------
 * Row-major arrays: per-l matrices (L+1,3,3), per-coefficient matrices ((L+1)^2,3,3), vectors ((L+1)^2,3),
 * component order (T, E, B). */
/* variance_expension.generate_polarization_var_cl_cython (variance_expension.pyx:36-61): D_l (L+1,3,3) ->
 * C_l = D_l 2pi/(l(l+1)) expanded over the real alm layout ((L+1)^2,3,3); l = 0 copied.  The reference
 * indexes cls_[idx] for cls_[l] at :51 (IndexError); the intended per-l lookup is implemented. */
int gs_expand_var_cl_3x3(const double* dls, int lmax, double* out, void* stream);
/* utils.compute_inverse_and_cholesky (recovered from utils.cpython-38.pyc; native twin linear_algebra.pyx
 * compute_inverse_matrices / compute_cholesky, LAPACK dgesv/dpotrf/dpotri): for l >= 2
 * Sigma_l = (blockdiag(inv(C_l[:2,:2]), 1/C_l[2,2]) + diag(pix_part_l))^-1 and its lower Cholesky factor;
 * l < 2 -> zeros.  pix_part is (L+1,3); chol nullable. */
int gs_inv_chol_3x3(const double* all_cls, const double* pix_part, int lmax, double* sigma, double* chol,
                    void* stream);
/* utils.matrix_product (recovered; native twin compute_matrix_product): out[i] = mats[l(i)] v[i] (+ add[i])
 * for every coefficient i of the real layout; add nullable; out may alias add. */
int gs_matvec_3x3(const double* mats, const double* v, const double* add, int lmax, double* out, void* stream);
/* hp.alm2cl(alm1, alm2) in the real layout: cl[l] = sum x y / (2l+1) (TE cross spectrum). */
int gs_alm2cl_cross(const double* alm_x, const double* alm_y, int lmax, double* cl, void* stream);
/* Inverse-Wishart draw of the (TT, TE; TE, EE) block per l >= 2 with df = 2l - 2 and scale (2l+1) Chat_l
 * (.ipynb_checkpoints/main-checkpoint.py:39-44, 333-346) by Bartlett decomposition, one thread per l.
 * cl_* are the empirical spectra (L+1); inject (nullable, (L+1,3)) = (chi2_df, chi2_{df-1}, N(0,1)) from the
 * caller for parity; outputs are C_l (0 for l < 2). */
int gs_cls_invwishart(const double* cl_tt, const double* cl_te, const double* cl_ee, int lmax,
                      const double* inject, uint64_t seed, uint64_t call, double* out_tt, double* out_te,
                      double* out_ee, void* stream);
/* Binned twin of gs_cls_invwishart (.ipynb_checkpoints/main-checkpoint.py:39-44, 333-346 with the binning of
 * CenteredGibbs.py:54-79): D_l = D_b on each bin b, and per bin, one thread each,
 *   D_b | s ~ IW(nu_b, Psi_b),  nu_b = sum_{l in b} (2l+1) - 3,  Psi_b = sum_{l in b} (2l+1) l(l+1)/(2pi) Chat_l,
 * Psi_b summed in ascending l.  With one-l bins this is gs_cls_invwishart times l(l+1)/(2pi) on the same variates.
 * cl_* are the unbinned empirical spectra (L+1); bins = nbins + 1 ascending int32 edges (device) that start 0, 1, 2
 * and end at lmax + 1 (bins 0 and 1 are l = 0 and l = 1 and come out 0); outputs dl_* are nbins binned D each.
 * inject (nullable, (nbins,3)) = (chi2_nu, chi2_{nu-1}, N(0,1)) per bin; NULL: Philox stream of draw b keyed as draw
 * l = b of gs_cls_invwishart.  GS_E_BADARG for null pointers, lmax < 0 or nbins outside [1, lmax + 1].  The edges are
 * checked on the device, bin by bin: a bin whose edges break the conditions above (bin 0 or 1 other than [0,1) / [1,2), an
 * empty bin, a bin below l = 2 or past lmax, a last edge other than lmax + 1) comes out NaN in all three outputs. */
int gs_cls_invwishart_binned(const double* cl_tt, const double* cl_te, const double* cl_ee, int lmax,
                             const int* bins, int nbins, const double* inject, uint64_t seed, uint64_t call,
                             double* dl_tt, double* dl_te, double* dl_ee, void* stream);

/* ---- Blackwell-Rao estimator of the spectrum posterior (Wandelt, Larson & Lakshminarayanan 2004; Chu et al. 2005) ----------
 * The reference has no BR code.  From the empirical spectra sigma^i of the N sky samples of a chain,
 *   log L(theta_k) = log( (1/N) sum_i exp( sum_b log p(D_b^k | sigma^i) ) ),  D in D units, p = the chain's C_l conditional:
 *   GS_BR_IG (one spectrum, edges of gs_cls_invgamma): alpha_b = sum_{l in b} (2l+1)/2 - 1,
 *     beta_b^i = sum_{l in b} (2l+1) l (l+1) sigma_l^i / 4pi (the arithmetic of gs_cls_invgamma's beta_out),
 *     log p = alpha log beta - lgamma(alpha) - (alpha+1) log D_b - beta / D_b;
 *   GS_BR_IW (the (TT, TE; TE, EE) block of gs_cls_invwishart_binned): nu_b = sum (2l+1) - 3,
 *     Psi_b^i = sum (2l+1) l (l+1)/2pi Chat_l^i, log p = (nu/2) log|Psi| - nu log 2 - log Gamma_2(nu/2) - (nu+3)/2 log|D|
 *     - tr(Psi D^-1)/2, log Gamma_2(a) = log(pi)/2 + lgamma(a) + lgamma(a - 1/2).
 * Written x_ik = c_i + sum_j S_ji W_jk + e_k, S is a (K, N) feature-major matrix (IG bin: one row beta_b; IW bin: three rows
 * Psi00, Psi01, Psi11), W a (K, M) one (IG: -1/D_b; IW: -(D^-1)00/2, -(D^-1)01, -(D^-1)11/2); c and e carry the rest.
 * Every bin passed to these calls is evaluated: callers pass the edges of the bins they want (the chains' bins 0 and 1 are
 * fixed at D = 0 and are never evaluated).  bins = nbins + 1 int32 device edges; each thread checks its own bin
 * (0 <= first < last <= ncl) and writes NaN for a broken one instead of reading out of range. */
#define GS_BR_IG 0
#define GS_BR_IW 1
/* Sample features of one spectrum group: sigma (IG) or sigma = TT, sigma_te, sigma_ee (IW), each (nsamp, ncl) row-major
 * (row i = empirical C_l of sample i, ncl = lmax + 1).  Writes rows 0 .. f nbins - 1 of S (f = 1 for IG, 3 for IW; row r at
 * S + r nsamp: pass S offset to the group's first row) and c[i] = (accumulate ? c[i] : 0) + sum_b t_b^i, b ascending, with
 * t_b = alpha_b log beta_b (IG) or (nu_b / 2) log|Psi_b| (IW).  scratch: nbins * nsamp doubles.  GS_E_BADARG for null
 * pointers, a bad kind, nsamp < 1 or nbins outside [1, min(ncl, 65535)]. */
int gs_br_sample_features(int kind, const double* sigma, const double* sigma_te, const double* sigma_ee, int64_t nsamp, int ncl,
                          const int* bins, int nbins, double* S, double* c, int accumulate, double* scratch, void* stream);
/* Model features of one group: dl (IG) or dl = TT, dl_te, dl_ee (IW), each (nmod, nbins) row-major binned D of the group's
 * bins.  Writes rows 0 .. f nbins - 1 of W (row r at W + r nmod) and e[k] = (accumulate ? e[k] : 0) + sum_b u_b^k with
 * u_b = -lgamma(alpha) - (alpha+1) log D_b (IG) or -nu log 2 - log Gamma_2(nu/2) - (nu+3)/2 log|D_b| (IW).  A model with
 * D_b <= 0, or an IW block that is not positive definite, gets W = 0 and e = -inf (its estimate is exactly -inf).
 * scratch: nbins * nmod doubles.  GS_E_BADARG as gs_br_sample_features. */
int gs_br_model_features(int kind, const double* dl, const double* dl_te, const double* dl_ee, int64_t nmod, int ncl,
                         const int* bins, int nbins, double* W, double* e, int accumulate, double* scratch, void* stream);
/* Fused GEMM + log-mean-exp: logl_out[k] = log((1/N) sum_i exp(x_ik)), x = c + S^T W + e (S: (K, nsamp), W: (K, nmod)), and
 * neff_out[k] (nullable) = (sum w_i)^2 / sum w_i^2, w_i = exp(x_ik - max_i x_ik): 0 and -inf for a model with e = -inf, NaN
 * for e = NaN.  Never forms the nsamp x nmod matrix.  The sample axis is split over
 *   P = min(ceil(nsamp / 256), ceil(2368 / ceil(nmod / 64)))
 * CTA columns; scratch: 3 * nmod * P doubles (the per-split partials, merged in a fixed order), as gs_br_logmeanexp_scratch
 * returns.  The split depends on
 * (nsamp, nmod) only, so repeated calls are bit-identical.  GS_E_BADARG for null pointers or nsamp, nmod, K < 1. */
/* Doubles of scratch gs_br_logmeanexp needs for (nsamp, nmod): 3 nmod P (-1 for nsamp or nmod < 1). */
int64_t gs_br_logmeanexp_scratch(int64_t nsamp, int64_t nmod);
int gs_br_logmeanexp(const double* S, const double* c, int64_t nsamp, const double* W, const double* e, int64_t nmod, int K,
                     double* scratch, double* logl_out, double* neff_out, void* stream);
/* Per-bin marginals out[b][g] = log((1/N) sum_i p(grid_b[g] | sigma_b^i)) of one group, p = IG(alpha_b, beta_b^i) for GS_BR_IG
 * (comp = 0; S = the group's nbins rows) and, for GS_BR_IW, the marginal of diagonal entry comp (0 = TT, 2 = EE) of the
 * inverse-Wishart, IG((nu_b - 1)/2, Psi_b,comp / 2) (S = the group's 3 nbins rows).  grid_b = grid + b grid_ld (grid_ld = 0:
 * one grid for all bins), ngrid points; a point <= 0 gives -inf.  out: (nbins, ngrid).  GS_E_BADARG for null pointers, a
 * bad kind / comp, nsamp or ngrid < 1, grid_ld < 0 or nbins outside [1, min(ncl, 65535)]. */
int gs_br_marginal(int kind, const double* S, int64_t nsamp, int ncl, const int* bins, int nbins, int comp, const double* grid,
                   int64_t grid_ld, int ngrid, double* out, void* stream);
/* Gaussianized BR transform (Rudjord et al. 2009) of one group, with the bins, kind, comp and S of gs_br_marginal: for the BR
 * marginal of bin b, the mixture (1/N) sum_i IG(alpha_b, beta_b^i), and dl (nmod, nbins) row-major binned D,
 *   x_out[k][b] = Phi^-1(F_b(D_kb)),  F_b(D) = (1/N) sum_i Q(alpha_b, beta_b^i / D),   logm_out[k][b] = log p_b(D_kb)
 * (Q, P: the regularized upper and lower incomplete gammas; logm is the quantity gs_br_marginal returns).  Sum Q and sum P are
 * kept apart, each sample computing its smaller tail directly (series, continued fraction or Temme's uniform expansion), and
 * x = Phi^-1(F) for F <= 1/2, else -Phi^-1(1 - F).  Broken edges: NaN; D <= 0 (or NaN), or F or 1 - F = 0 in FP64: x = -inf / +inf
 * and logm = -inf.  The sample axis is split over P CTA columns as a function of (nsamp, nmod, nbins) only and the partials merged
 * in a fixed order, so repeated calls are bit-identical; scratch: 4 * nmod * nbins * P doubles, as gs_gbr_transform_scratch
 * returns (-1 for nsamp or nmod < 1 or nbins outside [1, 65535]).  GS_E_BADARG for null pointers, a bad kind / comp, nsamp or
 * nmod < 1 or nbins outside [1, min(ncl, 65535)]. */
int64_t gs_gbr_transform_scratch(int64_t nsamp, int64_t nmod, int nbins);
int gs_gbr_transform(int kind, const double* S, int64_t nsamp, int ncl, const int* bins, int nbins, int comp, const double* dl,
                     int64_t nmod, double* x_out, double* logm_out, double* scratch, void* stream);

/* ---- whole chain in one call (SURVEY.md 8b gs_gibbs_step_centered; BASELINE config #1) -----------------------------------
 * GibbsSampler.run_polarization (GibbsSampler.py:118-180) for the full-sky isotropic-noise centred sampler: every iteration is
 * PolarizedCenteredConstrainedRealization.sample_no_mask (CenteredGibbs.py:317-353) + PolarizedCenteredClsSampler.sample
 * (CenteredGibbs.py:54-93) + utils.unfold_bins, run as three kernels that take the iteration number from device memory; the
 * iteration is captured once in a CUDA graph (use_graph != 0) and replayed n_iter times.  d_E / d_B = pix_map["EE"/"BB"] (real
 * layout), bins_* = nbins_* + 1 int32 edges, init_* = binned D_l of the start.  hist_* receive [n_iter + 1][nbins_*] binned D_l
 * (row 0 = init), last_E / last_B (nullable) the last sky map.  Philox draws (seed); synchronous on return. */
int gs_gibbs_run_centered_fullsky(int lmax, int64_t npix, double noise_pol, const double* bl, const double* d_E,
                                  const double* d_B, const int* bins_EE, int nbins_EE, const int* bins_BB, int nbins_BB,
                                  const double* init_EE, const double* init_BB, int n_iter, uint64_t seed,
                                  double* hist_EE, double* hist_BB, double* last_E, double* last_B, int use_graph,
                                  void* stream);

/* ---- m-sharded transforms over the GPUs of one node (SURVEY.md 8e; BASELINE config #4) --------------
 * The reference has no multi-GPU transform (one chain per SLURM task, job-script.sh:6); this is the
 * single-chain strategy for NSIDE >= 1024.  Rank r of `world` owns the m pairs {j, L-j} with j mod world = r
 * (Legendre stage) and the ring pairs p with p mod world = r (ring-FFT / pixel stage); one NCCL all-to-all
 * per transform moves the ring spectra between the two partitions.  On a sharded plan every plan-based
 * entry point above (gs_alm2map_spin2, gs_map2alm_spin2, gs_cr_rhs_pol, gs_cr_pcg_pol, gs_cr_apply_q_pol, ...)
 * takes LOCAL shards: alm in the local real layout (owned m ascending; m = 0: a_l0, l = 0..L; m > 0:
 * (sqrt2 Re, sqrt2 Im) for l = m..L; layout flag GS_ALM_REAL), maps as the owned rings in ascending RING
 * order; per-l arrays (dl, bl, fl) are replicated.  Scalars that are sums over pixels
 * (ninv_sum_over_4pi) must be global.  All ranks must make the same calls in the same order. */
/* 128-byte NCCL unique id for a new group: call on one rank, broadcast, pass to gs_plan_create_sharded. */
int gs_nccl_unique_id(char* id128_host);
/* Collective over the `world` ranks (each on its own device).  world == 1 is gs_plan_create. */
int gs_plan_create_sharded(gs_plan** plan, int nside, int lmax, int device, int rank, int world,
                           const char* nccl_id128_host);
/* In-process group for verification on ONE GPU: `world` sharded plans on the same device, each driven by
 * its own host thread and stream; the all-to-all / all-reduce are host barriers + device copies. */
int gs_local_group_create(void** group, int world);
int gs_local_group_destroy(void* group);
int gs_plan_create_sharded_local(gs_plan** plan, int nside, int lmax, int device, int rank, int world,
                                 void* local_group);
int gs_plan_world(const gs_plan* plan);
int gs_plan_rank(const gs_plan* plan);
int64_t gs_plan_nreal_local(const gs_plan* plan);  /* doubles in a local alm shard */
int64_t gs_plan_npix_local(const gs_plan* plan);   /* pixels in a local map shard */
/* The partition as pure host functions (no GPU): owned m / owned rings (0-based, ascending) of `rank`;
 * out may be NULL to query the count, which is the return value (negative = error). */
int gs_shard_partition_m(int lmax, int world, int rank, int* out);
int gs_shard_partition_rings(int nside, int world, int rank, int* out);
/* Global index (reference real layout, utils.py:49-76 / RING pixel number) of every entry of the local
 * alm / map shard; out may be NULL to query the length, which is the return value. */
int64_t gs_shard_real_index(int lmax, int world, int rank, int64_t* out);
int64_t gs_shard_pixel_index(int nside, int world, int rank, int64_t* out);
/* gs_expand_per_l over the plan's local real layout. */
int gs_shard_expand_per_l(gs_plan* plan, const double* x, int mode, double* out, void* stream);
/* hp.alm2cl of a sharded real-layout alm: local sums, all-reduce, / (2l+1); cl (L+1) on every rank. */
int gs_shard_alm2cl(gs_plan* plan, const double* alm_local, double* cl, void* stream);
/* In-place sum over the ranks of the plan of n device doubles. */
int gs_shard_allreduce_sum(gs_plan* plan, double* buf, int n, void* stream);

/* Average duration (ms) of one ring <-> m all-to-all of a sharded plan's spectra buffers, timed alone with CUDA events on
 * `stream` (collective: every rank calls it; 0 on unsharded plans).  bench.py reports it for BASELINE config #4. */
int gs_profile_exchange(gs_plan* plan, int nrep, float* ms_out, void* stream);

/* ---- measurement helpers used by bench.py ------------------------------------------------ */
/* Number of kernels this library has launched so far in the SHT stages and PCG vector updates. */
long long gs_launch_count(void);
/* Average duration (ms, CUDA events on `stream`) of the kernels of one PCG mat-vec
 * y = B A^T N^-1 A B x: ms_out[0] Legendre synthesis, [1] ring synthesis, [2] ring analysis,
 * [3] Legendre analysis + finish.  With the fused ring stage (the default, see gs_set_ring_fused)
 * ms_out[1] is the single ring kernel (synthesis -> N^-1 -> analysis per ring) and ms_out[2] = 0.  Synchronous. */
int gs_profile_matvec(gs_plan* plan, const double* x_E, const double* x_B, const double* bl,
                      const double* inv_noise, double* y_E, double* y_B, int nrep, float* ms_out,
                      void* stream);
/* gs_profile_matvec for a chain batch (n_chain = 1 or 2 right-hand sides at x / y + c stride doubles, one launch per stage, fused
 * ring stage): ms_out[0] Legendre synthesis, [1] ring stage, [2] Legendre analysis + finish, each for the whole batch. */
int gs_profile_matvec_batch(gs_plan* plan, int n_chain, const double* x_E, const double* x_B, int64_t stride,
                            const double* bl, const double* inv_noise, double* y_E, double* y_B, int nrep,
                            float* ms_out, void* stream);
/* Average duration (ms, CUDA events on `stream`) of the three vector kernels of one PCG iteration of gs_cr_pcg_pol
 * (spin = 2) / gs_cr_pcg_tt (spin = 0) on the plan's own zero-filled workspace: ms_out[0]  q += C^-1 p with <p, q>
 * (4 arrays of 8 n bytes per field), [1]  x += alpha p, r -= alpha q with <r, r>, <r, M r>  (7 arrays), [2]  p = M r +
 * beta p  (4 arrays); n = (lmax+1)^2, 2 fields for spin 2.  Every launch is timed alone after the plan's analysis workspace
 * (larger than L2 at NSIDE >= 512) has been overwritten.  No solver state is changed.  Synchronous. */
int gs_profile_pcg_vectors(gs_plan* plan, int spin, int nrep, float* ms_out, void* stream);
/* The parts of one gs_cr_pcg_teb iteration, average ms over nrep (CUDA events on `stream`, one warm-up): ms_out[0] the spin-0
 * mat-vec on inv_noise_T, [1] the spin-2 mat-vec on inv_noise_P (each with its own ring flags, as in the solve), [2] <p, Q p>
 * (6 arrays of 8 (L+1)^2 bytes), [3] the x / r update with <r,r>, <r,M r> (18 arrays), [4] p = M r + beta p (9 arrays), the
 * vector kernels on the zero-filled joint workspace after the analysis workspace has been overwritten.  Unsharded plans;
 * no solver state changes.  Synchronous. */
int gs_profile_matvec_teb(gs_plan* plan, const double* bl, const double* inv_noise_T, const double* inv_noise_P, int nrep,
                          float* ms_out, void* stream);
/* Ring stage of the PCG mat-vec (opfilt_pp.fwd_op's alm2map_spin -> N^-1 -> map2alm_spin, CenteredGibbs.py:629,653):
 * fused != 0 (default): one kernel per mat-vec keeps each ring's pixels in shared memory; 0: ring synthesis to the
 * plan's scratch maps, then weighted ring analysis.  Same result to rounding.  Returns the previous setting. */
int gs_set_ring_fused(int fused);
/* Rings whose pixel weights N^-1 vanish identically (inside a mask) contribute exactly nothing to A^T N^-1 A.  on != 0
 * (default): gs_cr_pcg_* / gs_cr_apply_q_* / gs_profile_matvec mark those rings from the weight map they are given (two
 * small kernels per call, no host round trip) and the Legendre and ring kernels of the mat-vec leave them out; 0: every
 * ring is processed.  Same result up to the rounding of a re-associated sum.  On sharded plans the ranks mark their own
 * rings and sum the flags (one small all-reduce per call).  gs_mwg_sweep_blocks skips the ring FFTs of those rings too.
 * Returns the previous setting. */
int gs_set_ring_skip(int on);
/* Rings on which the pixel weights N^-1 are all equal (isotropic noise, noise_covar * ones in the reference's config.py, on
 * every ring that the edge of the mask does not cut): for such a ring the middle of opfilt_pp.fwd_op (alm2map_spin -> N^-1 ->
 * map2alm_spin, CenteredGibbs.py:629,653) is DFT^H diag(w) DFT = n w on the alias-folded ring spectrum.  on != 0 (default,
 * unsharded plans, needs gs_set_ring_skip on): the fused ring stage of the mat-vec takes those rings without any transform,
 * flagged from the weight map of each call, and gs_mwg_sweep_blocks keeps data, model and block maps of those rings as the unitary
 * DFT of Q + iU along the ring (the weighted sums of squares of NonCenteredGibbs.py:380-399 are invariant under it), so their ring
 * FFTs are not run either; 0: every ring is transformed.  Same result to rounding.  Returns the previous setting. */
int gs_set_ring_const(int on);
/* Number of rings (of 4 nside - 1) whose pixel weights were all equal in the weight map of the last gs_cr_pcg_* /
 * gs_cr_apply_q_* / gs_profile_matvec call on this plan (rings inside the mask count: their weight is the constant 0);
 * 0 on sharded plans.  See gs_set_ring_const. */
int gs_constant_rings(gs_plan* plan, int* count_out);
/* Number of ring pairs (north/south) with a non-zero weight found by the last such call on this plan, and the total. */
int gs_active_ring_pairs(gs_plan* plan, int* active_out, int* total_out);
/* FP64 FMA throughput of the current device in TFLOP/s (DFMA microkernel; the roofline
 * denominator of the Legendre kernels).  Synchronous. */
int gs_measure_fp64_peak(double* tflops_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GIBBS_B200_H */
