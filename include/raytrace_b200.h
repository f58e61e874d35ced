/*
 * raytrace_b200.h -- C ABI of libraytrace_b200.so: the B200 (sm_100a) drop-in for the
 * reference's one data-parallel hot path, the 1-D layered-cake forward ray tracer `dff`
 * fused with the Gaussian travel-time likelihood.
 *
 * Reference = AntonBiryukovUofC/RayTracerFortran; citations are file:line in that tree.
 *
 * Conventions shared by every entry point
 *   - plain pointers and sizes only; every scalar of the Fortran-facing entries is passed
 *     BY REFERENCE (what R's .Fortran / .C and Fortran bind(C) callers without VALUE do);
 *   - all reals are IEEE binary64 (c_double), all counts are 32-bit (c_int);
 *   - vels[NLayers+1]  layer P velocities, surface to half-space;
 *     depths[NLayers]  depths of the interfaces below the surface (NOT thicknesses,
 *                      raytracerR-export-data-to-MCMC.Rmd:61);
 *   - the caller owns every buffer; the library keeps no result state between calls
 *     (device buffers and streams are cached internally and reused);
 *   - one context and one GPU per process (device = RTB200_DEVICE, else LOCAL_RANK, else 0,
 *     unless rtb200_init() chose one); every entry takes one process-wide lock, so calls from
 *     several host threads are safe and run one after the other (rtb200_last_error() is the
 *     last error of any thread);
 *   - there is NO CPU fallback: without a usable CUDA device the Fortran-style entries fill
 *     their outputs with NaN, print one line to stderr and record rtb200_last_error();
 *     the int-returning entries return a non-zero status.
 *   - results are bit-identical to the reference algorithm evaluated in IEEE binary64
 *     without FMA contraction (see DESIGN.md, "parity").
 */
#ifndef RAYTRACE_B200_H
#define RAYTRACE_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------
 * Drop-in symbols of the reference
 * ---------------------------------------------------------------------------------------- */

/* Replaces  subroutine dofullforwardproblem(...) bind(C, name="dff_")
 *           subroutineR-quiet.f90:408-463   (the symbol R's .Fortran("dff", ...) resolves,
 *           rayTracerR.R:31-33, raytracerR-export-data-to-MCMC.Rmd:81-83).
 * timeP[k] = direct-ray travel time from source k to the surface receiver; -999 when the
 * reference's `conv` flag stays false (:167-169).  keep_delta > 0 (re)writes ./rays.dat
 * with the per-layer horizontal advances and thicknesses of every ray (:157-164). */
void dff_(const double *vels, const double *depths, const int *NLayers,
          const double *src_offset, const double *src_depth, const int *NSrc,
          double *timeP, const int *keep_delta);

/* The older 7-argument form: subroutineR.f90:405, README.md:16-21, adaptMCMC.Rmd:74-78.
 * A C callee cannot see a missing 8th argument, so the two arities are two symbols; build
 * with -DRTB200_DFF_IS_7ARG to export this one under the name dff_ instead. */
void dff7_(const double *vels, const double *depths, const int *NLayers,
           const double *src_offset, const double *src_depth, const int *NSrc,
           double *timeP);

/* Replaces  subroutine TraceRays(...)  subroutineR-quiet.f90:467-520, the entry the sampler's
 * likelihood calls (ray_tracing_sampling/loglhood.f90:135,144).  Same body as dff_.  The
 * Fortran shim shim/raymod_b200.f90 forwards module raymod's TraceRays to this symbol. */
void tracerays_(const double *vels, const double *depths, const int *NLayers,
                const double *src_offset, const double *src_depth, const int *NSrc,
                double *timeP, const int *keep_delta);

/* The same entry under the names Fortran compilers give  module raymod :: TraceRays  (gfortran,
 * ifort/ifx, nvfortran/PGI), so that objects already compiled against the reference's raymod.mod
 * (ray_tracing_sampling/loglhood.f90 calls TraceRays at :135,144) link against this library as
 * they are; the checked-in raymod.mod is gfortran's.  Explicit-shape dummy arrays are passed as
 * plain pointers and scalars by reference: exactly tracerays_'s ABI. */
void __raymod_MOD_tracerays(const double *vels, const double *depths, const int *NLayers,
                            const double *src_offset, const double *src_depth, const int *NSrc,
                            double *timeP, const int *keep_delta);
void raymod_mp_tracerays_(const double *vels, const double *depths, const int *NLayers,
                          const double *src_offset, const double *src_depth, const int *NSrc,
                          double *timeP, const int *keep_delta);
void raymod_tracerays_(const double *vels, const double *depths, const int *NLayers,
                       const double *src_offset, const double *src_depth, const int *NSrc,
                       double *timeP, const int *keep_delta);

/* ------------------------------------------------------------------------------------------
 * Batched entries (new; the reference evaluates one model per call)
 * ---------------------------------------------------------------------------------------- */

/* B models x NSrc sources in one call; the sources are shared by every model, as in the
 * reference (rjmcmc_com.f90:44-45).  Host pointers.
 *   vels   [B][ldv]  row b holds nlayers[b]+1 velocities   (Fortran: vels(ldv,B))
 *   depths [B][ldz]  row b holds nlayers[b]   interfaces   (Fortran: depths(ldz,B))
 *   timeP  [B][NSrc] or NULL      travel times
 *   p_out  [B][NSrc] or NULL      ray parameter the travel time was summed at
 *   logL   [B]       or NULL      fused LOGLHOOD_RT value (needs tobs[NSrc], sigma[B]):
 *                                 log(1/(2 pi)^(N/2)) - (sum(res^2)/(2 sigma^2) + N log sigma),
 *                                 NaN -> -HUGE            (loglhood.f90:165-166,193-203)
 * Returns 0, or a non-zero status (see rtb200_last_error()). */
int dff_batch(const double *vels, const double *depths, const int *nlayers,
              const int *B, const int *ldv, const int *ldz,
              const double *src_offset, const double *src_depth, const int *NSrc,
              double *timeP, const double *tobs, const double *sigma,
              double *logL, double *p_out);

/* dff_batch for callers that cannot see a C return value: R's .C() and .Fortran() discard it and
 * pass every argument as a pointer.  Same arguments, plus *status = what dff_batch returns
 * (0 = ok; the message is rtb200_last_error()).  Exported as dff_batch_status (R: .C) and
 * dff_batch_status_ (R: .Fortran; Fortran without bind(C)).  R cannot pass NULL for an optional
 * array: pass a length-0 vector and the matching want flag = 0 --
 *   want[0] timeP, want[1] logL (then tobs and sigma are read), want[2] p_out. */
void dff_batch_status(const double *vels, const double *depths, const int *nlayers, const int *B,
                      const int *ldv, const int *ldz, const double *src_offset,
                      const double *src_depth, const int *NSrc, double *timeP, const double *tobs,
                      const double *sigma, double *logL, double *p_out, const int *want,
                      int *status);
void dff_batch_status_(const double *vels, const double *depths, const int *nlayers, const int *B,
                       const int *ldv, const int *ldz, const double *src_offset,
                       const double *src_depth, const int *NSrc, double *timeP, const double *tobs,
                       const double *sigma, double *logL, double *p_out, const int *want,
                       int *status);

/* dff_batch and the gradient of its travel times in one call (host pointers, scalars by
 * reference): the forward, then rtb200_dff_grad_device's vector-Jacobian product with weights
 * w [B][NSrc].  gvels [B][ldv] and gdepths [B][ldz] receive sum_s w dT/dV and sum_s w dT/dz;
 * timeP, p_out, dtdr and dtdd [B][NSrc] may each be NULL.  Returns 0, or a non-zero status
 * (see rtb200_last_error()). */
int dff_batch_grad(const double *vels, const double *depths, const int *nlayers,
                   const int *B, const int *ldv, const int *ldz,
                   const double *src_offset, const double *src_depth, const int *NSrc,
                   const double *w, double *timeP, double *p_out,
                   double *gvels, double *gdepths, double *dtdr, double *dtdd);

/* dff_batch and the Jacobian of its travel times in one call (host pointers, scalars by
 * reference): the forward, then rtb200_dff_jac_device.  jvels [B][NSrc][ldv] and
 * jdepths [B][NSrc][ldz] receive dT/dV and dT/dz per ray; timeP, p_out, dtdr and dtdd
 * [B][NSrc] may each be NULL.  No kmode.  Returns 0, or a non-zero status (see
 * rtb200_last_error()). */
int dff_batch_jac(const double *vels, const double *depths, const int *nlayers, const int *B,
                  const int *ldv, const int *ldz, const double *src_offset,
                  const double *src_depth, const int *NSrc, double *timeP, double *p_out,
                  double *jvels, double *jdepths, double *dtdr, double *dtdd);

/* dff_batch and the Gauss-Newton normal equations of its travel times in one call (host pointers,
 * scalars by reference): the forward, then rtb200_dff_normal_device.  JtJ [B][P][P], P = ldv + ldz;
 * tobs [NSrc] and Jtr [B][P] are both given or both NULL; timeP and p_out [B][NSrc] may each be
 * NULL.  No kmode.  Returns 0, or a non-zero status (see rtb200_last_error()). */
int dff_batch_normal(const double *vels, const double *depths, const int *nlayers, const int *B,
                     const int *ldv, const int *ldz, const double *src_offset,
                     const double *src_depth, const int *NSrc, const double *tobs, double *timeP,
                     double *p_out, double *JtJ, double *Jtr);

/* LOGLHOOD / LOGLHOOD_RT (loglhood.f90:3-32,35-211) over B chain states, with the model
 * mapping of :127-146: state b has k[b] Voronoi nodes, vp[b][0..k-1] = voro(1:k,2),
 * ziface[b][0..k-2] = ziface(1:k-1); k == 1 becomes two equal velocities over one fake
 * interface at 9999.9.  NMODE = 1, ICOV = 1, IAR = 0 (every shipped configuration).
 *   logL [B]; tpred [B][NSrc] or NULL receives DpredRT. */
int loglhood_batch(const int *k, const double *vp, const double *ziface,
                   const int *B, const int *ldv, const int *ldz,
                   const double *src_offset, const double *src_depth, const int *NSrc,
                   const double *tobs, const double *sigma,
                   double *logL, double *tpred);

/* loglhood_batch with the AR(1) residual error model of IAR = 1 (loglhood.f90:171-182;
 * ARPRED_RT :616-653, CHECKBOUNDS_ARMXRT :678-699; off in every shipped parameter file):
 * for states with idxar[b] == 1, DarRT(i) = arpar[b] * DresRT(i-1) for 1 < i < NSrc and 0 at both
 * ends, the residual becomes DresRT - DarRT, and a state whose |DarRT| exceeds *armx (the
 * reference's armxRT = 0.5, rjmcmc_com.f90:93) gets logL = -HUGE.  idxar == NULL is loglhood_batch. */
int loglhood_batch_ar(const int *k, const double *vp, const double *ziface,
                      const int *B, const int *ldv, const int *ldz,
                      const double *src_offset, const double *src_depth, const int *NSrc,
                      const double *tobs, const double *sigma,
                      const int *idxar, const double *arpar, const double *armx,
                      double *logL, double *tpred);

/* INTERPLAYER_novar + LOGLHOOD (loglhood.f90:214-295 then :3-211) over B chain states given as
 * UNSORTED Voronoi nodes: voro[b][0][i] = depth, voro[b][1][i] = vp of node i (Fortran
 * voro(ldk, 2, B)), k[b] <= ldk <= 64 nodes.  The nodes are sorted by depth on the device with
 * the reference's quicksort (quicksort.f90:66-123), ziface(1:k-1) = depth(2:k), and the states
 * are evaluated as by loglhood_batch.  voro_sorted [B][2][ldk] (or NULL) receives the sorted
 * nodes, tpred [B][NSrc] (or NULL) DpredRT. */
int loglhood_batch_voro(const int *k, const double *voro, const int *B, const int *ldk,
                        const double *src_offset, const double *src_depth, const int *NSrc,
                        const double *tobs, const double *sigma, double *logL, double *tpred,
                        double *voro_sorted);

/* ------------------------------------------------------------------------------------------
 * Device-resident entry: every pointer is a CUDA device pointer on the current device and
 * nothing is copied.  Asynchronous on `stream` (a cudaStream_t passed as void*; NULL = the
 * library's own stream, in which case the call synchronises before returning).
 * kmode != 0 : nlayers[] holds node counts k and the LOGLHOOD_RT mapping above is applied.
 * ---------------------------------------------------------------------------------------- */
int rtb200_dff_batch_device(const double *d_vels, const double *d_depths, const int *d_nlayers,
                            int B, int ldv, int ldz,
                            const double *d_src_offset, const double *d_src_depth, int NSrc,
                            double *d_timeP, const double *d_tobs, const double *d_sigma,
                            double *d_logL, double *d_p_out, int kmode, void *stream);

/* Gradient of the travel times with respect to the layered model and the sources, as a
 * vector-Jacobian product over B models x NSrc sources (DESIGN.md section 11).  Device pointers,
 * model and source arrays as for rtb200_dff_batch_device (same kmode mapping), plus what that
 * entry returned for them:
 *   timeP, p   [B][NSrc]   the forward's travel times and ray parameters (d_timeP, d_p_out)
 *   w          [B][NSrc]   weights, e.g. dL/dT of a loss L
 * Out:
 *   gvels      [B][ldv]    gvels[b][i]   = sum_s w[b][s] dT_bs/dV_i
 *   gdepths    [B][ldz]    gdepths[b][j] = sum_s w[b][s] dT_bs/dz_j   (kmode: ziface)
 *   dtdr, dtdd [B][NSrc]   or NULL: dT_bs/d(src_offset[s]), dT_bs/d(src_depth[s])
 * The derivatives are those of the exact travel-time function at the returned p (Fermat:
 * dT/dR = p); rays with timeP = -999 (not converged) contribute 0.  Columns past a model's layers
 * are 0; at k = 1 both layers are vp(1) and the fake interface gets 0.  Each sum runs in source
 * order without atomics, so the result is reproducible bit for bit.  Rows must hold nlayers[b]+1
 * velocities and nlayers[b] interfaces, as for the forward.  Stream semantics of
 * rtb200_dff_batch_device. */
int rtb200_dff_grad_device(const double *d_vels, const double *d_depths, const int *d_nlayers,
                           int B, int ldv, int ldz,
                           const double *d_src_offset, const double *d_src_depth, int NSrc,
                           const double *d_timeP, const double *d_p, const double *d_w,
                           double *d_gvels, double *d_gdepths, double *d_dtdr, double *d_dtdd,
                           int kmode, void *stream);

/* Jacobian of the travel times with respect to the layered model, per ray (DESIGN.md section 12):
 * the terms rtb200_dff_grad_device sums over the sources, written unsummed.  Inputs as for that
 * entry, without w.  Out:
 *   jvels      [B][NSrc][ldv]  dT_bs/dV_i: n >= 2 layers and i < n: -H_i / (V_i^2 cos_i);
 *                              a top-layer ray (n = 1): -T/V_0 at i = 0
 *   jdepths    [B][NSrc][ldz]  dT_bs/dz_j = eta_j - eta_{j+1} for j <= n - 2 (kmode: ziface)
 *   dtdr, dtdd [B][NSrc]       or NULL: as rtb200_dff_grad_device writes them
 * Every other entry is 0, and so is the row of a ray with timeP = -999.  At k = 1 (kmode)
 * jvels[b][s][0] is the sum of both layers' terms and jdepths is 0.  Each term is rounded as in
 * rtb200_dff_grad_device, so that entry with a one-hot w returns the ray's row bit for bit.
 * jdepths may be NULL when ldz = 0.  Stream semantics of rtb200_dff_batch_device. */
int rtb200_dff_jac_device(const double *d_vels, const double *d_depths, const int *d_nlayers,
                          int B, int ldv, int ldz,
                          const double *d_src_offset, const double *d_src_depth, int NSrc,
                          const double *d_timeP, const double *d_p, double *d_jvels,
                          double *d_jdepths, double *d_dtdr, double *d_dtdd, int kmode,
                          void *stream);

/* Gauss-Newton normal equations of the travel times, per model (DESIGN.md section 13), without
 * storing the Jacobian.  Inputs as for rtb200_dff_jac_device, plus the observations d_tobs [NSrc].
 * With J_s = [jvels[b][s][:] | jdepths[b][s][:]] the row rtb200_dff_jac_device writes for ray
 * (b, s), P = ldv + ldz and r_s = tobs_s - timeP[b][s]:
 *   JtJ  [B][P][P]  sum_s J_si J_sj
 *   Jtr  [B][P]     sum_s J_si r_s
 * Each sum runs over s in increasing order from +0.0, one rounded multiply and one rounded add a
 * term (no FMA), and takes only the terms whose columns the ray reaches: velocity column i < n
 * (kmode k = 1: column 0 when n >= 1), depth column j <= n - 2 (none at k = 1), nothing for a ray
 * with timeP = -999.  So the result depends on no launch geometry, JtJ is exactly symmetric, and
 * a column no ray of a model reaches is a zero row and column: JtJ is then singular, and a
 * damped solve (Levenberg-Marquardt) is the caller's remedy.  No weights: with one sigma per
 * model the caller scales the result by 1 / sigma^2.  d_tobs and d_Jtr are NULL together.
 * NSrc = 0 gives zeros; the source arrays, timeP, p and d_tobs may then be NULL.  Stream
 * semantics of rtb200_dff_batch_device. */
int rtb200_dff_normal_device(const double *d_vels, const double *d_depths, const int *d_nlayers,
                             int B, int ldv, int ldz, const double *d_src_offset,
                             const double *d_src_depth, int NSrc, const double *d_timeP,
                             const double *d_p, const double *d_tobs, double *d_JtJ,
                             double *d_Jtr, int kmode, void *stream);

/* One fixed-dimension Metropolis-Hastings move of B independent chains, entirely on the device:
 * PROPOSAL (prjmh_temper_rf.f90:1386-1447, ENOS = 0: Cauchy step on voro(ivo,iwhich), |.| for a
 * depth) -> INTERPLAYER_novar (loglhood.f90:214-295) -> CHECKBOUNDS2 (:1681-1716) -> LOGLHOOD ->
 * the accept test of EXPLORE_MH_NOVARPAR (:739-757: reject iff ran_uni >= EXP(logPr + (logL_new -
 * logL)*beta_mh), logPr = 0; proposals outside the prior bounds are rejected unevaluated).
 * The random numbers are inputs, so the caller owns the generator.  Device pointers:
 *   d_k      [B]          node counts (unchanged: no birth/death)
 *   d_voro   [B][2][ldk]  current states, sorted by depth (row 0 depth, row 1 vp); accepted
 *                         proposals are written back
 *   d_logL   [B]          current logL; updated on accept
 *   d_ivo, d_iwhich [B]   1-based node and parameter (1 = depth, 2 = vp) to perturb; ivo > k,
 *                         or (ivo, iwhich) = (1, 1) (the fixed top node, :730) is a no-op (-1)
 *   d_cauchy [B]          TAN(PI*(ran_uni - 0.5)) deviates;  d_uacc [B] uniforms of the accept test
 *   d_beta   [B]          1/T of each chain;  d_sigma [B] sdparRT
 *   prior    HOST [7]     fact/factor*pertsd(1), fact/factor*pertsd(2), minlim(1), minlim(2),
 *                         maxlim(1), maxlim(2), hmin          (read_input.f90:207-214)
 *   d_accept [B] out      1 accepted, 0 rejected, -1 rejected because outside the bounds
 * Asynchronous on `stream` like rtb200_dff_batch_device; the library's scratch buffers are reused
 * by consecutive calls, so issue them on one stream. */
int rtb200_mh_step_device(const int *d_k, double *d_voro, double *d_logL, int B, int ldk,
                          const int *d_ivo, const int *d_iwhich, const double *d_cauchy,
                          const double *d_uacc, const double *d_beta, const double *d_sigma,
                          const double *prior, const double *d_src_offset,
                          const double *d_src_depth, const double *d_tobs, int NSrc,
                          int *d_accept, void *stream);
/* The same move with the accept test ordered behind a CUDA event (cudaEvent_t, may be NULL): the
 * proposal and likelihood kernels do not read d_beta, so a tempering swap round that is still
 * rewriting the betas on another stream (rtb200_swap_round_device) overlaps with them.
 * enos = 1 selects the even-numbered order statistics prior of the parameter file (ENOS, Green
 * 1995): a depth move draws the node uniformly between its neighbours -- d_cauchy[b] is then the
 * uniform ran_uni itself -- and LOG(zjp1-zp)+LOG(zp-zjm1)-LOG(zjp1-zj)-LOG(zj-zjm1) enters the
 * accept test as logPr (PROPOSAL, prjmh_temper_rf.f90:1418-1431, :743-745). */
int rtb200_mh_step_device_ev(const int *d_k, double *d_voro, double *d_logL, int B, int ldk,
                          const int *d_ivo, const int *d_iwhich, const double *d_cauchy,
                          const double *d_uacc, const double *d_beta, const double *d_sigma,
                          const double *prior, const double *d_src_offset,
                          const double *d_src_depth, const double *d_tobs, int NSrc,
                          int *d_accept, void *stream, void *beta_ready_event, int enos);

/* n_moves consecutive calls of rtb200_mh_step_device in one: move m uses row m of d_ivo, d_iwhich,
 * d_cauchy, d_uacc and writes row m of d_accept (all [n_moves][B]).  The run is captured once into
 * a CUDA graph and replayed for as long as the caller passes the same buffers and sizes (refill
 * them in place) and the options stay as they were, which removes the launch gaps between the
 * three kernels of every move; a changed option or tile geometry takes effect on the next call.
 * n_moves <= 512. */
int rtb200_mh_moves_device(const int *d_k, double *d_voro, double *d_logL, int B, int ldk,
                           int n_moves, const int *d_ivo, const int *d_iwhich,
                           const double *d_cauchy, const double *d_uacc, const double *d_beta,
                           const double *d_sigma, const double *prior, const double *d_src_offset,
                           const double *d_src_depth, const double *d_tobs, int NSrc,
                           int *d_accept, void *stream);
/* The same with the ENOS switch of rtb200_mh_step_device_ev. */
int rtb200_mh_moves_device_ex(const int *d_k, double *d_voro, double *d_logL, int B, int ldk,
                           int n_moves, const int *d_ivo, const int *d_iwhich,
                           const double *d_cauchy, const double *d_uacc, const double *d_beta,
                           const double *d_sigma, const double *prior, const double *d_src_offset,
                           const double *d_src_depth, const double *d_tobs, int NSrc,
                           int *d_accept, void *stream, int enos);

/* The birth/death move at the top of EXPLORE_MH_NOVARPAR (prjmh_temper_rf.f90:658-710) for B
 * independent chains on the device: move choice from ran_unik (:666-680: 1/3 birth, 1/3 death,
 * 1/3 neither; no birth at kmax, no death at kmin), BIRTH_FULL (:997-1103: new node at depth
 * maxpert(1)*u_z with vp minlim(2)+maxpert(2)*u_v) or DEATH_FULL (:917-994: node idel of 2..k
 * removed), INTERPLAYER_novar, CHECKBOUNDS (:1639-1678), LOGLHOOD, accept with
 * logPr = LOG(pk(k'))-LOG(pk(k)) (Poisson prior on k, IPOIPR = 1, ENOS = 0).
 *   d_k [B] in/out; d_voro [B][2][ldk] in/out (slots past k are zero); d_logL [B] in/out
 *   d_uk, d_uz, d_uv, d_uacc [B]  uniforms: move choice, new depth, new vp, accept test
 *   d_idel [B]                    node a death would remove (RANDPERM(k-1)(1)+1, in 2..k)
 *   prior HOST [7] as for rtb200_mh_step_device; pk HOST [kmax] with pk[i-1] = pk(i)
 *                                 (read_input.f90:78-81), or NULL for IPOIPR = 0
 *   d_accept [B] out              1 accepted, 0 rejected, -1 outside the bounds, 2 no move proposed */
int rtb200_bd_step_device(int *d_k, double *d_voro, double *d_logL, int B, int ldk,
                          const double *d_uk, const int *d_idel, const double *d_uz,
                          const double *d_uv, const double *d_uacc, const double *d_beta,
                          const double *d_sigma, const double *prior, const double *pk, int kmin,
                          int kmax, const double *d_src_offset, const double *d_src_depth,
                          const double *d_tobs, int NSrc, int *d_accept, void *stream);
/* The same with enos = 1: the order-statistics terms of DEATH_FULL (prjmh_temper_rf.f90:981-991)
 * and BIRTH_FULL (:1090-1098) are added to logPr (after LOG(pk(k'))-LOG(pk(k)) when pk is given);
 * a birth whose new node cannot be found among the sorted interfaces (the reference would index
 * voro(-1,1)) is rejected as outside. */
int rtb200_bd_step_device_ex(int *d_k, double *d_voro, double *d_logL, int B, int ldk,
                          const double *d_uk, const int *d_idel, const double *d_uz,
                          const double *d_uv, const double *d_uacc, const double *d_beta,
                          const double *d_sigma, const double *prior, const double *pk, int kmin,
                          int kmax, const double *d_src_offset, const double *d_src_depth,
                          const double *d_tobs, int NSrc, int *d_accept, void *stream, int enos);

/* The data-error move of EXPLORE_MH (prjmh_temper_rf.f90:545-575) for B independent chains on the
 * device: chains whose gate uniform is >= 0.10 propose sdparRT + pertsdsdRT*gauss (PROPOSAL_SDRT,
 * :1616-1635; outside unless within [minlimsdRT, maxlimsdRT]), the model is re-evaluated with the
 * proposed sigma, and the move is rejected iff ran_uni >= EXP((logL_new - logL)*beta_mh).
 *   d_voro [B][2][ldk], d_k [B] read only; d_logL [B], d_sigma [B] in/out
 *   d_ugate, d_uacc [B] uniforms; d_gauss [B] standard normal deviates (GASDEVJ)
 *   sd_prior HOST [3] = pertsdsdRT, minlimsdRT, maxlimsdRT          (read_input.f90:237-241)
 *   d_accept [B] out: 1 accepted, 0 rejected, -1 outside the bounds, 2 no move proposed */
int rtb200_sd_step_device(const int *d_k, const double *d_voro, double *d_logL, double *d_sigma,
                          int B, int ldk, const double *d_ugate, const double *d_gauss,
                          const double *d_uacc, const double *d_beta, const double *sd_prior,
                          const double *d_src_offset, const double *d_src_depth,
                          const double *d_tobs, int NSrc, int *d_accept, void *stream);

/* IAR = 1 for the chain move entries: register the chains' AR(1) state (device arrays idxarRT [B],
 * arparRT [B], and armxRT); from then on rtb200_mh_step_device, rtb200_mh_moves_device,
 * rtb200_bd_step_device and rtb200_sd_step_device evaluate LOGLHOOD with the AR residual model
 * (loglhood.f90:171-182) of each chain, as the sampler does when IAR = 1.  NULL, NULL returns to
 * IAR = 0.  rtb200_ar_step_device updates the same arrays when they are the ones passed to it. */
int rtb200_set_chain_ar(const int *d_idxar, const double *d_arpar, double armx);

/* The AR(1) move of EXPLORE_MH (prjmh_temper_rf.f90:583-631, IAR = 1) for B independent chains on
 * the device, with PROPOSAL_ARRT (:1521-1552): a chain without an AR parameter proposes its birth
 * (uniform over [minlimarRT, maxlimarRT], logarp = LOG(0.5)); otherwise death when the choice
 * uniform is >= 0.5 (logarp = LOG(2)) or a perturbation arparRT + pertarsdRT*gauss (logarp = 0).
 * The model is re-evaluated with the proposal (loglhood.f90:171-182) and the move is rejected iff
 * ran_uni >= EXP(logarp + (logL_new - logL)*beta_mh).  d_logL must be the likelihood under the
 * chain's current (idxar, arpar).
 *   d_idxar [B], d_arpar [B] in/out;  d_uchoice, d_uprop, d_uacc [B] uniforms;  d_gauss [B] normal
 *   ar_prior HOST [4] = pertarsdRT, minlimarRT, maxlimarRT, armxRT      (read_input.f90:223-227)
 *   d_accept [B] out: 1 accepted, 0 rejected, -1 outside the bounds */
int rtb200_ar_step_device(const int *d_k, const double *d_voro, double *d_logL,
                          const double *d_sigma, int *d_idxar, double *d_arpar, int B, int ldk,
                          const double *d_uchoice, const double *d_uprop, const double *d_gauss,
                          const double *d_uacc, const double *d_beta, const double *ar_prior,
                          const double *d_src_offset, const double *d_src_depth,
                          const double *d_tobs, int NSrc, int *d_accept, void *stream);

/* One whole iteration of the sampler's worker loop (prjmh_temper_rf.f90:420-458) for B chains,
 * n_iterations times, entirely on the device: the birth/death move (skipped when kmin == kmax),
 * n_moves fixed-dimension moves in which every chain continues its own sweep (ivo, iwhich) =
 * (1,2), (2,1), (2,2), ..., (k,1), (k,2) (:725-731) from d_pos[b], and the data-error move of
 * EXPLORE_MH (:545-575).  Every random deviate is drawn by the library's Philox4x32-10 kernels
 * (key = seed, counter = (chain, *d_counter, purpose)); the iteration is captured once as a CUDA
 * graph and replayed, *d_counter advancing by one per iteration, so there is no host
 * synchronisation and no per-move host work.  With d_idxar / d_arpar / ar_prior (IAR = 1; all
 * three or none) the iteration ends with EXPLORE_MH's AR(1) move (:583-631) and every likelihood
 * of the iteration uses the chains' AR state; without them a state registered through
 * rtb200_set_chain_ar still enters every likelihood.
 *   d_k, d_voro, d_logL, d_sigma in/out; d_beta [B] read at every accept test (a swap round
 *   between calls may rewrite it); d_pos [B] i32 in/out: position of each chain in its sweep
 *   prior HOST [7], sd_prior HOST [3], pk HOST [kmax] or NULL, enos: as for the single moves
 *   d_counter: one device uint64, in/out;  d_workspace: rtb200_mcmc_workspace_bytes(B, n_moves)
 *   bytes holding the iteration's deviates and outcomes (layout: McmcWs in csrc/rt_internal.h,
 *   mirrored by chains.mcmc_workspace_views);  d_tally [5][B] int64 or NULL, accumulated:
 *   fixed-dimension moves accepted, evaluated, births/deaths accepted, sigma moves accepted,
 *   AR moves accepted;  ar_prior HOST [4] as for rtb200_ar_step_device */
size_t rtb200_mcmc_workspace_bytes(int B, int n_moves);
int rtb200_mcmc_iterations_device(int *d_k, double *d_voro, double *d_logL, double *d_sigma,
                                  const double *d_beta, int *d_pos, int B, int ldk, int n_moves,
                                  const double *prior, const double *sd_prior, const double *pk,
                                  int kmin, int kmax, int enos, const double *d_src_offset,
                                  const double *d_src_depth, const double *d_tobs, int NSrc,
                                  unsigned long long seed, unsigned long long *d_counter,
                                  void *d_workspace, long long *d_tally, int n_iterations,
                                  int *d_idxar, double *d_arpar, const double *ar_prior,
                                  void *stream);

/* The parallel-tempering swap round (TEMPSWP_MH, prjmh_temper_rf.f90:1329-1384; master loop
 * :326-349) for n chains spread over the ranks of one job, decisions taken on the device.
 * Every rank calls rtb200_swap_pack_device on its own chains (d_out[i] = (logL[i], beta[i])),
 * all-gathers the packed pairs in rank order (the path's only collective: 16 bytes per chain),
 * and calls rtb200_swap_round_device on the gathered array: the round's pairing (a keyed
 * bijection of [0, n); pair t = (perm(2t), perm(2t+1))) and its uniforms are functions of
 * (seed, round) alone, so all ranks take identical decisions; chain pair (i, j) is accepted iff
 * u <= EXP((beta_j - beta_i)*(logL_i - logL_j)) (:1339-1342) and exchanges betas (the reference
 * exchanges the states and keeps the temperatures in place, :1351-1357: the same Markov kernel).
 *   d_all [n][2] gathered (logL, beta);  this rank owns chains [lo, lo + n_local)
 *   d_beta_local [n_local] out: the betas of this rank's chains after the round
 *   d_accept [n/2] out or NULL: 1/0 per pair;  d_partner [n_local] out or NULL: the partner's
 *   global index when the swap was accepted, -1 - index when rejected, -1 when unpaired (odd n) */
int rtb200_swap_pack_device(const double *d_logL, const double *d_beta, int n, double *d_out,
                            void *stream);
int rtb200_swap_round_device(const double *d_all, int n, int lo, int n_local,
                             unsigned long long seed, unsigned long long round,
                             double *d_beta_local, int *d_accept, int *d_partner, void *stream);

/* ------------------------------------------------------------------------------------------
 * Runtime control and introspection
 * ---------------------------------------------------------------------------------------- */
int         rtb200_init(int device);          /* optional; lazy init picks the device itself   */
void        rtb200_shutdown(void);
const char *rtb200_last_error(void);          /* "" when the last call succeeded               */
int         rtb200_device_count(void);        /* 0 without a driver / device                   */
/* options: "variant" (1 lane state machine, 3 deep-model kernel, 5 variant 1 with one segment of
 *          the sorted ray list per warp; any other value >= 0 means 1;
 *          < 0 default: by shape -- 3 for deep models; for shallow ones 5 when
 *          the batch is at least six tiles per resident CTA or a single wave of full tiles, 1 in
 *          between; rtb200_get_stat("variant") reports 9 for the one-model
 *          latency kernel),
 *          "threads", "tile_models", "tile_sources", "chunk_models", "ctas_per_sm"; <= 0 restores
 *          the default; "comp_streams" (1: host-call chunks run on one compute stream; default 2:
 *          consecutive chunks alternate between two so one chunk's tail overlaps the next);
 *          "static_tiles" (1: CTAs stride over the tiles instead of claiming them from a counter);
 *          "logl_shuffle" (1: reduce the residuals of a model with a warp-shuffle tree instead of
 *          the reference's source order -- same terms, ~N ulp from the ordered sum; default 0);
 *          "stage_pageable" (-1 default: large pageable host inputs are copied by a few host
 *          threads into a pinned ring so that H2D stays asynchronous; 0 never; 1 always);
 *          "latency_path" (1 default: a one-model call without likelihood -- dff_, TraceRays --
 *          runs the one-warp-per-ray kernel on mapped pinned memory; 0: the batch kernel);
 *          "stable_lognorm" (0 default: LOG(1/(2 PI2)**(N/2)) as loglhood.f90:194 writes it, which
 *          is -Inf for N >= 773 sources; 1: the same constant as -(N/2) LOG(2 PI2), finite for any
 *          N -- a deviation from the reference, for likelihoods over more than 771 data);
 *          "ismpprior" (ISMPPRIOR of the parameter file: 1 = the chain move entries sample the
 *          prior -- every proposal's likelihood is LOGLHOOD2's constant 1, loglhood.f90:704-716,
 *          and no ray is traced; default 0) */
int         rtb200_set_option(const char *name, double value);
/* stats of the last batched call: "kernel_ms", "total_ms", "launches" (cumulative),
 *          "tile_models", "tile_sources", "smem_bytes", "grid", "threads", "ctas_per_sm" */
double      rtb200_get_stat(const char *name);
/* sustained FP64 FMA throughput of the current device in TFLOP/s (roofline denominator) */
double      rtb200_fp64_peak_tflops(int repeats);
/* Self-test of the hot loop's rsqrt-seeded square root and divisions: draws `samples` operand
 * triples over the solver's range and compares them bit for bit with CUDA's correctly rounded
 * sqrt and divide.  Returns the number of mismatching results (0 expected), -1 on failure. */
double      rtb200_selftest_fast_division(double samples, unsigned long long seed);
/* contiguous slice [*lo, *hi) of B models owned by `rank` of `world` (model-axis sharding) */
void        rtb200_shard_range(long long B, int rank, int world, long long *lo, long long *hi);

#ifdef __cplusplus
}
#endif
#endif
