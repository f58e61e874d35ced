// rt_internal.h -- shared between the kernels (rt_kernels.cu) and the C ABI (rt_api.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace rtb {

// Solver constants of the reference (subroutineR-quiet.f90).
constexpr double kTol          = 1.0e-1;   // :234, :351   tol = 1.d-1
constexpr int    kNewtonMaxIt  = 15;       // :233
constexpr int    kBisectMaxIt  = 20;       // :346
constexpr double kClampRR      = 1.0e-9;   // :250
constexpr double kSafeEps      = 1.0e-10;  // :142, :388
constexpr double kBisectLo     = 1.0e-10;  // :148
constexpr double kBisectHiEps  = 1.0e-12;  // :148
constexpr int    kHalveCap     = 2200;     // the reference never terminates on a NaN p0 (:125-133)
constexpr double kFakeIface    = 9999.9;   // loglhood.f90:141

// One batched launch.  Every pointer is a device pointer.
struct BatchArgs {
    const double *vels;        // [B][ldv]
    const double *depths;      // [B][ldz]
    const int    *nlayers;     // [B]; kmode: node counts k
    int           B, ldv, ldz;
    int           kmode;       // LOGLHOOD_RT model mapping (loglhood.f90:127-146)
    const double *src_offset;  // [nsrc]
    const double *src_depth;   // [nsrc]
    const double *tobs;        // [nsrc] or null
    int           nsrc;
    const double *sigma;       // [B] or null
    double       *timeP;       // [B][nsrc] or null
    double       *p_out;       // [B][nsrc] or null
    double       *logL;        // [B] or null
    double        logc;        // log(1/(2 pi)^(N/2)), computed once on the host
    int           padded;      // vels/depths are readable up to a whole number of tiles
    // AR(1) residual model (IAR = 1: ARPRED_RT + CHECKBOUNDS_ARMXRT, loglhood.f90:171-182,616-701)
    const int    *idxar;       // [B] or null: obj%idxarRT(1), 1 = apply the AR model to this state
    const double *arpar;       // [B] obj%arparRT(1)
    double        armx;        // armxRT: |DarRT| beyond it rejects the state (logL = -HUGE)
    // dynamic tile scheduling: [0] tiles claimed beyond the first wave, [1] CTAs finished; both
    // zero between launches (the last CTA resets them); null = static stride
    int          *sched;
};

// What every derivative kernel reads: the models and sources of a batch-kernel launch and what it
// returned.  Every pointer is a device pointer; model and source arrays as in BatchArgs.  It is
// the base of GradArgs, JacArgs, NormalArgs and HessArgs, so their fields keep the offsets they would have
// if each declared these itself.
struct DerivArgs {
    const double *vels;        // [B][ldv]
    const double *depths;      // [B][ldz]
    const int    *nlayers;     // [B]; kmode: node counts k
    int           B, ldv, ldz;
    int           kmode;
    const double *src_offset;  // [nsrc]
    const double *src_depth;   // [nsrc]
    int           nsrc;
    const double *timeP;       // [B][nsrc] the batch kernel's travel times
    const double *p;           // [B][nsrc] and ray parameters
};

// One launch of the gradient kernel (the vector-Jacobian product of the travel times, DESIGN.md
// section 11).
struct GradArgs : DerivArgs {
    const double *w;           // [B][nsrc] weights of the product
    double       *gvels;       // [B][ldv]  sum_s w dT/dV_i
    double       *gdepths;     // [B][ldz]  sum_s w dT/dz_j
    double       *dtdr;        // [B][nsrc] or null: dT/d(offset)
    double       *dtdd;        // [B][nsrc] or null: dT/d(depth)
};

// One launch of the Jacobian kernel (the per-ray terms the gradient kernel sums, DESIGN.md
// section 12).
struct JacArgs : DerivArgs {
    double       *jvels;       // [B][nsrc][ldv]  dT_bs/dV_i
    double       *jdepths;     // [B][nsrc][ldz]  dT_bs/dz_j (null when ldz = 0)
    double       *dtdr;        // [B][nsrc] or null: dT/d(offset)
    double       *dtdd;        // [B][nsrc] or null: dT/d(depth)
};

// One launch of the normal-equations kernel (DESIGN.md section 13).  P = ldv + ldz parameter
// columns, [vels | depths].
struct NormalArgs : DerivArgs {
    const double *tobs;        // [nsrc] or null (then Jtr is null)
    double       *JtJ;         // [B][P][P]
    double       *Jtr;         // [B][P] or null
};

// One launch of the second-derivative kernel (DESIGN.md section 14).  P = ldv + ldz parameter
// columns, [vels | depths].
struct HessArgs : DerivArgs {
    const double *w;           // [B][nsrc] weights of the rays
    double       *H;           // [B][P][P]  sum_s w_s d2T_s
};

// Tile geometry chosen by the host for one launch.
struct TileCfg {
    int M;        // models per tile (even unless forced by the tile_models option)
    int SC;       // sources per chunk
    int LP;       // per-model row length of the derived tables (odd, >= max velocities)
    int TS;       // row stride of the travel-time tile (odd)
    int threads;  // CTA size
    int grid;     // persistent CTAs
    int variant;  // 1: lane state machine with refill, 3: the same for deep models,
                  // 5: variant 1 with one list segment per warp
    int use_tma;  // rows are 16-byte aligned: stage with cp.async.bulk
    int logl_shuffle;  // reduce the residuals with warp shuffles (tree order) instead of source order
    size_t smem;  // dynamic shared memory bytes
    // Unused.  It keeps the batch kernel's parameter block at the 1200 bytes its register allocation
    // was tuned with: 104 bytes smaller, ptxas allocates the kernels differently, and on a B200 at
    // 1000 W config 2 took 9.127 ms against 9.044 and config 3 0.1360 ms against 0.1338.
    double reserved[13];
};

// Prior and proposal scales of the fixed-dimension MH move (read_input.f90:207-214).
struct MhPrior {
    double scale[2];    // fact/factor*pertsd(1:2)   Cauchy step widths: depth, vp
    double minlim[2];   // minlim(1:2)
    double maxlim[2];   // maxlim(1:2)
    double hmin;        // minimum layer thickness
    int    enos;        // ENOS: 1 = even-numbered order statistics prior (Green 1995) in the moves
};

// Birth/death move: range of k and the Poisson prior on k (read_input.f90:70-81) as LOG(pk(i)).
struct BdPrior {
    int    kmin, kmax, use_pk;
    double logpk[64];   // logpk[i-1] = LOG(pk(i)), computed on the host
};

// Workspace of one MCMC iteration run as a CUDA graph (rtb200_mcmc_iterations_device): every
// deviate of the iteration, written by the library's Philox kernels and read by the move kernels,
// and every move's outcome.  One caller-owned allocation, laid out as
//   doubles: u_k | u_z | u_v | u_acc_bd | u_gate | gauss | u_acc_sd |
//            u_choice | u_prop_ar | gauss_ar | u_acc_ar                    [B] each
//            dev [M][B] | u_acc [M][B]
//   ints:    idel | acc_bd | acc_sd | acc_ar [B] each,  ivo | iwhich | acc_mh [M][B] each
struct McmcWs {
    double *u_k, *u_z, *u_v, *u_acc_bd, *u_gate, *gauss, *u_acc_sd, *u_choice, *u_prop_ar, *gauss_ar,
           *u_acc_ar, *dev, *u_acc;
    int    *idel, *acc_bd, *acc_sd, *acc_ar, *ivo, *iwhich, *acc_mh;
};
inline size_t mcmc_ws_bytes(size_t B, size_t M) { return (11 + 2 * M) * B * 8 + (4 + 3 * M) * B * 4; }
inline McmcWs mcmc_ws_layout(void *base, size_t B, size_t M) {
    McmcWs w;
    double *d = static_cast<double *>(base);
    w.u_k = d; w.u_z = d + B; w.u_v = d + 2 * B; w.u_acc_bd = d + 3 * B; w.u_gate = d + 4 * B;
    w.gauss = d + 5 * B; w.u_acc_sd = d + 6 * B; w.u_choice = d + 7 * B; w.u_prop_ar = d + 8 * B;
    w.gauss_ar = d + 9 * B; w.u_acc_ar = d + 10 * B; w.dev = d + 11 * B; w.u_acc = d + (11 + M) * B;
    int *i = reinterpret_cast<int *>(d + (11 + 2 * M) * B);
    w.idel = i; w.acc_bd = i + B; w.acc_sd = i + 2 * B; w.acc_ar = i + 3 * B; w.ivo = i + 4 * B;
    w.iwhich = i + (4 + M) * B; w.acc_mh = i + (4 + 2 * M) * B;
    return w;
}
cudaError_t launch_mcmc_draw(const unsigned long long *counter, unsigned long long seed, const int *k,
                             int B, const McmcWs &w, cudaStream_t st);
cudaError_t launch_mcmc_sweep_draw(const unsigned long long *counter, unsigned long long seed,
                                   const int *k, const int *pos, int B, int M, int enos,
                                   const McmcWs &w, cudaStream_t st);
cudaError_t launch_mcmc_finish(unsigned long long *counter, const int *k, int *pos, int B, int M,
                               const McmcWs &w, long long *tally, cudaStream_t st);

size_t      tile_smem_bytes(const TileCfg &c, int ldv, int ldz);
cudaError_t launch_batch(const BatchArgs &a, const TileCfg &c, cudaStream_t st);
cudaError_t launch_grad(const GradArgs &a, cudaStream_t st);
cudaError_t launch_jac(const JacArgs &a, cudaStream_t st);
cudaError_t launch_normal(const NormalArgs &a, cudaStream_t st);
cudaError_t launch_hess(const HessArgs &a, cudaStream_t st);
cudaError_t launch_prep_voro(const int *k, const double *voro, int B, int ldk, double *vels,
                             double *depths, double *sorted, cudaStream_t st);
cudaError_t launch_propose_voro(const int *k, const double *voro, int B, int ldk, const int *ivo,
                                const int *iwhich, const double *cauchy, const MhPrior &pr,
                                double *vels, double *depths, int *keval, double *prop,
                                double *logpr, int *outside, cudaStream_t st);
cudaError_t launch_mh_accept(const int *k, double *voro, const double *prop, double *logL,
                             const double *logL_prop, const double *logpr, const int *outside,
                             const double *u_acc, const double *beta, int B, int ldk, int *accept,
                             cudaStream_t st);
cudaError_t launch_propose_bd(const int *k, const double *voro, int B, int ldk, const double *u_k,
                              const int *idel, const double *u_z, const double *u_v,
                              const MhPrior &pr, const BdPrior &bd, double *vels, double *depths,
                              int *keval, int *kprop, double *prop, double *logpr, int *outside,
                              cudaStream_t st);
cudaError_t launch_bd_accept(int *k, double *voro, const double *prop, const int *kprop,
                             const double *logpr, double *logL, const double *logL_prop,
                             const int *outside, const double *u_acc, const double *beta, int B,
                             int ldk, int *accept, cudaStream_t st);
cudaError_t launch_propose_sd(const int *k, const double *voro, int B, int ldk, const double *sigma,
                              const double *u_gate, const double *gauss, double pert, double smin,
                              double smax, double *vels, double *depths, int *keval,
                              double *sigma_prop, int *outside, cudaStream_t st);
cudaError_t launch_sd_accept(double *sigma, const double *sigma_prop, double *logL,
                             const double *logL_prop, const int *outside, const double *u_acc,
                             const double *beta, int B, int *accept, cudaStream_t st);
cudaError_t launch_propose_ar(const int *k, const double *voro, int B, int ldk, const int *idxar,
                              const double *arpar, const double *u_choice, const double *u_prop,
                              const double *gauss, double pert, double amin, double amax,
                              double log_half, double log_two, double *vels, double *depths,
                              int *keval, int *idx_prop, double *ar_prop, double *logarp,
                              int *outside, cudaStream_t st);
cudaError_t launch_ar_accept(int *idxar, double *arpar, const int *idx_prop, const double *ar_prop,
                             const double *logarp, double *logL, const double *logL_prop,
                             const int *outside, const double *u_acc, const double *beta, int B,
                             int *accept, cudaStream_t st);
cudaError_t launch_dff_latency(const double *in_host, const double *in_dev, int NL, int S, double *out,
                               int want_p, int *done_flag, int *single_cta, cudaStream_t st);
cudaError_t launch_fill_f64(double *p, int n, double value, cudaStream_t st);
cudaError_t launch_swap_pack(const double *logL, const double *beta, int n, double *out,
                             cudaStream_t st);
cudaError_t launch_swap_round(const double *all, int n, int lo, int n_local, unsigned long long seed,
                              unsigned long long round, double *beta_local, int *accept,
                              int *partner, cudaStream_t st);
int         max_ctas_per_sm(const TileCfg &c);   // occupancy of the batch kernel for this geometry
cudaError_t fp64_peak(double *tflops, int repeats, cudaStream_t st);
cudaError_t fastpath_selftest(double samples, unsigned long long seed, double *mismatches,
                              cudaStream_t st);

}  // namespace rtb
