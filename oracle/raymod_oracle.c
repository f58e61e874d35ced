/*
 * raymod_oracle.c -- CPU ORACLE (TEST INFRASTRUCTURE, NOT PRODUCT CODE).  See raymod_oracle.h.
 *
 * Every function cites the reference lines it restates; paths are relative to
 * /root/reference/.  "sq" = subroutineR-quiet.f90, "ll" = ray_tracing_sampling/loglhood.f90.
 *
 * Build: gcc -O2 -ffp-contract=off -fno-fast-math -fopenmp (see oracle/Makefile).
 * No FMA, no reassociation: the bits must equal gfortran -O2 on baseline x86-64.
 */
#include "raymod_oracle.h"

#include <float.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define ORC_TOL            1.0e-1   /* sq:234, sq:351   tol = 1.d-1                     */
#define ORC_NEWTON_MAXIT   15       /* sq:233                                            */
#define ORC_BISECT_MAXIT   20       /* sq:346                                            */
#define ORC_CLAMP_RR       1.0e-9   /* sq:250  rr = 1d-9                                 */
#define ORC_SAFE_EPS       1.0e-10  /* sq:142, sq:388                                    */
#define ORC_BISECT_LO      1.0e-10  /* sq:148  first bracket end                         */
#define ORC_BISECT_HI_EPS  1.0e-12  /* sq:148  1/maxval(vp) - 1d-12                      */
#define ORC_HALVE_CAP      2200     /* the reference loops forever on NaN p0 (sq:125-133);
                                       2200 halvings take any finite double to 0          */
#define ORC_PI             3.141592653589793238462643383279502884197 /* data_type.f90:5 */


/* gfortran list-directed output of a REAL(8) (the format of rays.dat, sq:101-102,160-161):
   17 significant digits, fixed notation for 0.1 <= |x| < 1e17 (right-justified in 21 columns
   followed by 5 blanks), exponent form otherwise. */
static void fprint_ld(FILE *fh, double x)
{
    char buf[64];
    double ax = fabs(x);
    if (x == 0.0) {
        snprintf(buf, sizeof buf, "0.0000000000000000");
    } else if (ax >= 0.1 && ax < 1e17) {
        int e10 = (int)floor(log10(ax));
        int dec = 16 - e10;
        if (e10 < 0) dec = 17;
        if (dec < 0) dec = 0;
        snprintf(buf, sizeof buf, "%.*f", dec, x);
    } else {
        int e10 = (int)floor(log10(ax));
        double m = x / pow(10.0, e10);
        snprintf(buf, sizeof buf, "%.16fE%+04d", m, e10);
        fprintf(fh, "%26s", buf);
        return;
    }
    fprintf(fh, "%21s     ", buf);
}

/* ---- sq:9-32 whichLayer ------------------------------------------------------------ */
int orc_which_layer(const double *depths, int nlayers, double dph)
{
    int    inN  = 0;
    double diff = 0.0;  /* uninitialised in the reference when nlayers == 0 (never called so) */
    for (int i = 1; i <= nlayers; ++i) {
        inN  = i;
        diff = depths[i - 1] - dph;
        if (diff > 0.0) break;
    }
    if (nlayers <= 0) return 1;          /* defined extension: a bare half-space */
    return (diff < 0.0) ? nlayers + 1 : inN;
}

/* ---- sq:184-202 costFunc ----------------------------------------------------------- */
static double cost_f(double x, const double *H, const double *V, int n, double R)
{
    double sum_all = 0.0;
    for (int i = 0; i < n; ++i) {
        double num = (H[i] * V[i]) * x;                       /* H*V*x, left to right */
        double den = sqrt(1.0 - (x * x) * (V[i] * V[i]));     /* sqrt(1-(x**2)*V**2)  */
        sum_all = sum_all + num / den;
    }
    return R - sum_all;
}

/* ---- sq:206-221 costFunc_Prime ----------------------------------------------------- */
static double cost_fp(double x, const double *H, const double *V, int n)
{
    double acc = 0.0;
    for (int i = 0; i < n; ++i) {
        double s     = sqrt(1.0 - (x * x) * (V[i] * V[i]));
        double denom = s * (s * s);                           /* s**3 */
        acc = acc + (H[i] * V[i]) / denom;
    }
    return -acc;
}

static double max_of(const double *V, int n)
{
    double m = V[0];
    for (int i = 1; i < n; ++i) if (V[i] > m) m = V[i];
    return m;
}

/* ---- sq:226-332 solve (Newton) ----------------------------------------------------- */
static double newton_solve(double x0, const double *H, const double *V, int n, double R,
                           int *conv_out, orc_trace *tr, int x0_cached)
{
    int    conv = 0;
    double x = x0, fx = 0.0, fxp = 0.0;
    int    k;
    for (k = 1; k <= ORC_NEWTON_MAXIT; ++k) {
        fx  = cost_f(x, H, V, n, R);                           /* sq:275 */
        fxp = cost_fp(x, H, V, n);                             /* sq:284 */
        if (tr) {
            tr->n_f_ref++; tr->n_fp_ref++;
            int cached = (k == 1) && x0_cached;                /* caller already holds f,f' at x0 */
            if (fabs(fx) < ORC_TOL) { if (!cached) tr->n_f_min++; }
            else if (!cached) tr->n_ffp_min++;
        }
        if (fabs(fx) < ORC_TOL) { conv = 1; break; }           /* sq:287-291 */
        x = x - fx / fxp;                                      /* sq:294-298 */
        if (tr) tr->n_newton++;
        if (x > 1.0 / max_of(V, n)) {                          /* sq:299-304 */
            x = 1.0 / max_of(V, n) - ORC_CLAMP_RR;
            if (tr) tr->n_clamp++;
        }
    }
    if (k > ORC_NEWTON_MAXIT) {                                /* sq:314-317 */
        fx = cost_f(x, H, V, n, R);
        if (tr) { tr->n_f_ref++; tr->n_f_min++; }
    }
    if (fabs(fx) > ORC_TOL) conv = 1;                          /* sq:327-330 (sic) */
    if (tr) tr->f_final = fx;
    *conv_out = conv;
    return x;
}

/* ---- sq:339-405 solvebst (bisection until a Newton jump is safe) ------------------- */
static double bisect_solve(double x1, double x2, const double *H, const double *V, int n,
                           double R, orc_trace *tr, int *x_cached)
{
    double fmid = cost_f(x2, H, V, n, R);                      /* sq:353 */
    double f    = cost_f(x1, H, V, n, R);                      /* sq:354 */
    double x, dx, xmid, fx, fxp, check_x;
    (void)fmid;
    /* f(x2) is dead in the reference: fmid is overwritten at sq:370 before any use */
    if (tr) { tr->n_f_ref += 2; tr->n_f_min += 1; }
    if (f < 0.0) { x = x1; dx = x2 - x1; }                     /* sq:359-365 */
    else         { x = x2; dx = x1 - x2; }
    *x_cached = 0;
    for (int k = 1; k <= ORC_BISECT_MAXIT; ++k) {
        dx   = dx * 0.5;                                       /* sq:368 */
        xmid = x + dx;                                         /* sq:369 */
        fmid = cost_f(xmid, H, V, n, R);                       /* sq:370 */
        if (tr) { tr->n_bisect++; tr->n_f_ref++; }
        *x_cached = 0;
        if (fmid < 0.0) { x = xmid; *x_cached = 1; }           /* sq:371-373 */
        if (fmid == 0.0) { if (tr) tr->n_f_min++; break; }     /* sq:375-377 */
        fx  = cost_f(xmid, H, V, n, R);                        /* sq:378 */
        fxp = cost_fp(xmid, H, V, n);                          /* sq:380 */
        if (tr) { tr->n_f_ref++; tr->n_fp_ref++; tr->n_ffp_min++; }
        check_x = x - fx / fxp;                                /* sq:384-386: x, not xmid */
        if (check_x < 1.0 / max_of(V, n) - ORC_SAFE_EPS) {     /* sq:388-392 */
            x = xmid; *x_cached = 1;
            break;
        }
        if (fabs(fmid) < ORC_TOL) break;                       /* sq:394-396 */
    }
    return x;
}

/* ---- sq:77-178 GetPTime on the truncated column H[0..n-1], V[0..n-1] --------------- */
static double get_ptime(double src_depth, double src_offset, int n,
                        const double *V, const double *H, orc_trace *tr,
                        int keep_delta, const char *rays_path)
{
    double timeP;
    if (n == 1) {                                              /* sq:94-97 */
        timeP = sqrt(src_depth * src_depth + src_offset * src_offset) / V[0];
        if (tr) {
            tr->branch = ORC_BRANCH_TOP; tr->conv = 1;
            /* the reference has no p on this path; report the straight ray's sin(theta)/v */
            tr->p = (src_offset / sqrt(src_depth * src_depth + src_offset * src_offset)) / V[0];
        }
        if (keep_delta > 0 && rays_path) {                     /* sq:98-105 (root copy only) */
            FILE *fh = fopen(rays_path, "a");
            if (fh) {
                fprint_ld(fh, src_offset); fprintf(fh, "\n");
                fprint_ld(fh, src_depth);  fprintf(fh, "\n");
                fclose(fh);
            }
        }
        return timeP;
    }

    int    conv = 0;
    double hv_sum = 0.0;
    for (int i = 0; i < n; ++i) hv_sum = hv_sum + H[i] / V[i];
    double c_harmonic = src_depth / hv_sum;                                            /* sq:112 */
    double cos_t = src_depth / sqrt(src_offset * src_offset + src_depth * src_depth);  /* sq:113 */
    double p0 = cos_t / c_harmonic * 1.0;                                              /* sq:116 */

    for (int guard = 0; guard < ORC_HALVE_CAP; ++guard) {                              /* sq:125-133 */
        double s = 0.0;
        for (int i = 0; i < n; ++i)
            s = s + sqrt(1.0 - (p0 * p0) * ((V[i] + 1.0) * (V[i] + 1.0)));
        if (!isnan(s)) break;
        p0 = p0 / 2.0;
        if (tr) tr->n_halve++;
    }

    double cf  = cost_f(p0, H, V, n, src_offset);                                      /* sq:136 */
    double cfp = cost_fp(p0, H, V, n);                                                 /* sq:137 */
    double check_x = p0 - cf / cfp;                                                    /* sq:138 */
    if (tr) { tr->n_f_ref++; tr->n_fp_ref++; tr->n_ffp_min++; }

    double p_final;
    if (cf < 0.0) {                                                                    /* sq:139-141 */
        if (tr) tr->branch = ORC_BRANCH_NEG;
        p_final = newton_solve(p0, H, V, n, src_offset, &conv, tr, 1);
    } else if (check_x < 1.0 / max_of(V, n) - ORC_SAFE_EPS) {                          /* sq:142-144 */
        if (tr) tr->branch = ORC_BRANCH_SAFE;
        p_final = newton_solve(p0, H, V, n, src_offset, &conv, tr, 1);
    } else {                                                                           /* sq:145-153 */
        int cached = 0;
        if (tr) tr->branch = ORC_BRANCH_BISECT;
        double pb = bisect_solve(ORC_BISECT_LO, 1.0 / max_of(V, n) - ORC_BISECT_HI_EPS,
                                 H, V, n, src_offset, tr, &cached);
        p_final = newton_solve(pb, H, V, n, src_offset, &conv, tr, cached);
    }

    /* sq:156,165-166  cosV = sqrt(1-(p**2)*vp**2); t_int = depths/(vp*cosV); sum */
    timeP = 0.0;
    for (int i = 0; i < n; ++i) {
        double cosV = sqrt(1.0 - (p_final * p_final) * (V[i] * V[i]));
        timeP = timeP + H[i] / (V[i] * cosV);
    }
    if (keep_delta > 0 && rays_path) {                                                 /* sq:157-164 */
        FILE *fh = fopen(rays_path, "a");
        if (fh) {
            for (int i = 0; i < n; ++i) {
                double cosV = sqrt(1.0 - (p_final * p_final) * (V[i] * V[i]));
                double q = H[i] / cosV;
                fprint_ld(fh, sqrt(q * q - H[i] * H[i]));
            }
            fprintf(fh, "\n");
            for (int i = 0; i < n; ++i) fprint_ld(fh, H[i]);
            fprintf(fh, "\n");
            fclose(fh);
        }
    }
    if (!conv) timeP = -999.0;                                                         /* sq:167-169 */
    if (tr) { tr->p = p_final; tr->conv = conv; }
    return timeP;
}

/* ---- sq:436-455 one trip of the source loop: whichLayer, InsertLayer, GetPTime ------ */
static double ray_time_impl(const double *vels, const double *depths, int nlayers,
                            double src_offset, double src_depth, orc_trace *tr,
                            int keep_delta, const char *rays_path)
{
    if (tr) memset(tr, 0, sizeof *tr);
    int nl = orc_which_layer(depths, nlayers, src_depth);
    if (tr) tr->nl = nl;
    if (nl == 1)                                               /* sq:438-441 */
        return get_ptime(src_depth, src_offset, 1, vels, depths, tr, keep_delta, rays_path);

    /* sq:38-69 InsertLayer: the column above the source, interfaces turned into thicknesses.
       Both branches (:51-56 and :57-63) give V(1:nl) = vels(1:nl) and depths_new(1:nl) =
       (z(1:nl-1), dph); :67 differences it in place. */
    double Hs[64], Vs[64];
    double *H = Hs, *V = Vs;
    if (nl > 64) {
        H = (double *)malloc(sizeof(double) * (size_t)nl * 2);
        V = H + nl;
    }
    for (int i = 0; i < nl; ++i) V[i] = vels[i];
    H[0] = depths[0];
    for (int i = 1; i < nl - 1; ++i) H[i] = depths[i] - depths[i - 1];
    H[nl - 1] = src_depth - depths[nl - 2];
    double t = get_ptime(src_depth, src_offset, nl, V, H, tr, keep_delta, rays_path);
    if (H != Hs) free(H);
    return t;
}

double orc_ray_time(const double *vels, const double *depths, int nlayers,
                    double src_offset, double src_depth, orc_trace *tr)
{
    return ray_time_impl(vels, depths, nlayers, src_offset, src_depth, tr, -1, NULL);
}

/* ---- sq:408-463 dofullforwardproblem == sq:467-520 TraceRays ------------------------ */
void orc_trace_rays(const double *vels, const double *depths, int nlayers,
                    const double *src_offset, const double *src_depth, int nsrc,
                    double *timeP, double *p_out, orc_trace *traces,
                    int keep_delta, const char *rays_path)
{
    for (int k = 0; k < nsrc; ++k) timeP[k] = -1.0;            /* sq:430 */
    if (rays_path) {                                           /* sq:432-433: REPLACE, every call */
        FILE *fh = fopen(rays_path, "w");
        if (fh) fclose(fh);
    }
    for (int k = 0; k < nsrc; ++k) {                           /* sq:434-462 */
        orc_trace local;
        orc_trace *tr = traces ? &traces[k] : (p_out ? &local : NULL);
        timeP[k] = ray_time_impl(vels, depths, nlayers, src_offset[k], src_depth[k], tr,
                                 keep_delta, rays_path);
        if (p_out) p_out[k] = tr->p;
    }
}

/* ---- ll:165-166,193-203 ------------------------------------------------------------ */
double orc_loglhood_from_times(const double *tpred, const double *tobs, int ndat, double sigma)
{
    double ss = 0.0;
    for (int k = 0; k < ndat; ++k) {
        double res = tobs[k] - tpred[k];                       /* ll:166 */
        ss = ss + res * res;                                   /* SUM(DresRT**2) */
    }
    double n = (double)ndat;
    double logL = log(1.0 / pow(2.0 * ORC_PI, n / 2.0))        /* ll:194 */
                - (ss / (2.0 * (sigma * sigma)) + n * log(sigma));   /* ll:195-196 */
    if (isnan(logL)) logL = -DBL_MAX;                          /* ll:200-203 */
    return logL;
}

/* ---- ll:127-146 model mapping + ll:165-203 ------------------------------------------ */
double orc_loglhood_rt(int k, const double *vp, const double *ziface,
                       const double *src_offset, const double *src_depth, int nsrc,
                       const double *tobs, double sigma, double *tpred)
{
    double *pred = tpred ? tpred : (double *)malloc(sizeof(double) * (size_t)(nsrc > 0 ? nsrc : 1));
    if (k > 1) {
        orc_trace_rays(vp, ziface, k - 1, src_offset, src_depth, nsrc, pred, NULL, NULL, -1, NULL);
    } else {
        double v2[2] = { vp[0], vp[0] };
        double z1[1] = { 9999.9 };
        orc_trace_rays(v2, z1, 1, src_offset, src_depth, nsrc, pred, NULL, NULL, -1, NULL);
    }
    double logL = orc_loglhood_from_times(pred, tobs, nsrc, sigma);
    if (!tpred) free(pred);
    return logL;
}

/* ---- batched sweeps (workload shape of replica.f90:173-232; new, not in the reference) */
int orc_dff_batch(const double *vels, const double *depths, const int *nlayers,
                  int B, int ldv, int ldz,
                  const double *src_offset, const double *src_depth, int nsrc,
                  double *timeP, const double *tobs, const double *sigma,
                  double *logL, double *p_out, int nthreads)
{
    int used = 1;
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
    used = nthreads;
#else
    (void)nthreads;
#endif
#pragma omp parallel num_threads(used)
    {
        double *tloc = (double *)malloc(sizeof(double) * (size_t)(nsrc > 0 ? nsrc : 1));
        double *ploc = (double *)malloc(sizeof(double) * (size_t)(nsrc > 0 ? nsrc : 1));
#pragma omp for schedule(dynamic, 64)
        for (int b = 0; b < B; ++b) {
            const double *v = vels + (size_t)b * ldv;
            const double *z = depths + (size_t)b * ldz;
            double *t = timeP ? timeP + (size_t)b * nsrc : tloc;
            double *p = p_out ? p_out + (size_t)b * nsrc : NULL;
            orc_trace_rays(v, z, nlayers[b], src_offset, src_depth, nsrc, t, p, NULL, -1, NULL);
            if (logL) logL[b] = orc_loglhood_from_times(t, tobs, nsrc, sigma[b]);
        }
        free(tloc); free(ploc);
    }
    return used;
}

int orc_dff_batch_faithful(const double *vels, const double *depths, const int *nlayers,
                           int B, int ldv, int ldz,
                           const double *src_offset, const double *src_depth, int nsrc,
                           double *timeP, const char *rays_path)
{
    double *tloc = (double *)malloc(sizeof(double) * (size_t)(nsrc > 0 ? nsrc : 1));
    for (int b = 0; b < B; ++b) {
        double *t = timeP ? timeP + (size_t)b * nsrc : tloc;
        orc_trace_rays(vels + (size_t)b * ldv, depths + (size_t)b * ldz, nlayers[b],
                       src_offset, src_depth, nsrc, t, NULL, NULL, -1, rays_path);
    }
    free(tloc);
    return 1;
}

/* ---- work accounting (DESIGN.md "work per evaluation"; sqrt = div = 1 flop) --------- */
void orc_batch_stats(const double *vels, const double *depths, const int *nlayers,
                     int B, int ldv, int ldz,
                     const double *src_offset, const double *src_depth, int nsrc,
                     orc_stats *out)
{
    orc_stats s;
    memset(&s, 0, sizeof s);
    for (int b = 0; b < B; ++b) {
        for (int k = 0; k < nsrc; ++k) {
            orc_trace tr;
            (void)orc_ray_time(vels + (size_t)b * ldv, depths + (size_t)b * ldz, nlayers[b],
                               src_offset[k], src_depth[k], &tr);
            double L = (double)tr.nl;
            s.rays++;
            s.sum_nl += tr.nl;
            if (tr.branch == ORC_BRANCH_TOP) {
                s.top++;
                s.flops_ref += 5.0; s.flops_min += 5.0;
                s.sqrt_ref += 1; s.div_ref += 1; s.sqrt_min += 1; s.div_min += 1;
                continue;
            }
            if (tr.branch == ORC_BRANCH_NEG)    s.neg++;
            if (tr.branch == ORC_BRANCH_SAFE)   s.safe++;
            if (tr.branch == ORC_BRANCH_BISECT) s.bisect++;
            s.n_halve += tr.n_halve; s.n_bisect += tr.n_bisect; s.n_newton += tr.n_newton;
            s.n_clamp += tr.n_clamp; s.not_conv += !tr.conv;
            s.n_f_ref += tr.n_f_ref; s.n_fp_ref += tr.n_fp_ref;
            s.n_ffp_min += tr.n_ffp_min; s.n_f_min += tr.n_f_min;
            int isb = tr.branch == ORC_BRANCH_BISECT;
            /* what the reference executes */
            s.flops_ref += (L - 1.0)                       /* InsertLayer differencing            */
                         + (2.0 * L + 1.0) + 5.0 + 2.0      /* c_harmonic, cos_t, p0               */
                         + (6.0 * L + 1.0) * (1 + tr.n_halve) + tr.n_halve
                         + (8.0 * L + 2.0) * tr.n_f_ref + (9.0 * L + 2.0) * tr.n_fp_ref
                         + 2.0 + 2.0                        /* check_x, 1/vmax - 1e-10             */
                         + (isb ? 2.0 + 6.0 * tr.n_bisect : 0.0)
                         + 3.0 * tr.n_newton + 2.0 * tr.n_clamp
                         + (7.0 * L + 1.0);                 /* travel-time sum                      */
            s.sqrt_ref += (long long)(L * (1 + tr.n_halve) + L * tr.n_f_ref + L * tr.n_fp_ref + L) + 1;
            s.div_ref  += (long long)((L + 1) + 2 + tr.n_halve + L * tr.n_f_ref + L * tr.n_fp_ref
                                      + 2 + (isb ? 1 + 2 * tr.n_bisect : 0) + 2 * tr.n_newton
                                      + tr.n_clamp + L);
            /* de-duplicated count that still yields identical bits */
            s.flops_min += 5.0 + 5.0 + 1.0                  /* last-layer H, hv, c_h; cos_t; p0    */
                         + 5.0 * (1 + tr.n_halve) + tr.n_halve
                         + 1.0 + 1.0                        /* 1/vmax, - 1e-10                      */
                         + (10.0 * L + 3.0) * tr.n_ffp_min + (6.0 * L + 2.0) * tr.n_f_min
                         + 2.0                              /* check_x                              */
                         + (isb ? 1.0 + 4.0 * tr.n_bisect : 0.0)
                         + 2.0 * tr.n_newton + 1.0 * tr.n_clamp
                         + (6.0 * L + 1.0);
            s.sqrt_min += (long long)(1 + L * tr.n_ffp_min + L * tr.n_f_min + L);
            s.div_min  += (long long)(2 + 1 + 1 + tr.n_halve + 1 + 2 * L * tr.n_ffp_min + L * tr.n_f_min
                                      + 1 + (isb ? tr.n_bisect : 0) + tr.n_newton + L);
        }
    }
    *out = s;
}

/* ---- "next" row N1: INTERPLAYER_novar (ll:214-295) ---------------------------------- *
 * Sort the k Voronoi nodes by depth with the reference's own quicksort (Hoare partition,
 * quicksort.f90:66-123: ties keep the order that algorithm gives them), then
 * ziface(1:k-1) = depth(2:k) (ll:258-259) and LOGLHOOD_RT on (vp(1:k), ziface).          */
static void orc_partition2d(double *dep, double *vp, int n, int *marker)
{
    double x = dep[0];                                          /* quicksort.f90:93 */
    int i = 0, j = n + 1;                                       /* 1-based, as in the reference */
    for (;;) {
        j = j - 1;
        while (!(dep[j - 1] <= x)) j = j - 1;                   /* :99-102 */
        i = i + 1;
        while (!(dep[i - 1] >= x)) i = i + 1;                   /* :104-107 */
        if (i < j) {                                            /* :108-115 */
            double t = dep[i - 1]; dep[i - 1] = dep[j - 1]; dep[j - 1] = t;
            t = vp[i - 1]; vp[i - 1] = vp[j - 1]; vp[j - 1] = t;
        } else if (i == j) { *marker = i + 1; return; }         /* :116-118 */
        else { *marker = i; return; }                           /* :119-121 */
    }
}

static void orc_qsortc2d(double *dep, double *vp, int n)
{
    if (n > 1) {                                                /* quicksort.f90:71-75 */
        int iq;
        orc_partition2d(dep, vp, n, &iq);
        orc_qsortc2d(dep, vp, iq - 1);
        orc_qsortc2d(dep + iq - 1, vp + iq - 1, n - iq + 1);
    }
}

void orc_interplayer_novar(int k, double *node_depth, double *node_vp)
{
    orc_qsortc2d(node_depth, node_vp, k);
}

double orc_loglhood_voro(int k, const double *node_depth, const double *node_vp,
                         const double *src_offset, const double *src_depth, int nsrc,
                         const double *tobs, double sigma, double *tpred,
                         double *sorted_depth, double *sorted_vp)
{
    double *d = (double *)malloc(sizeof(double) * (size_t)(2 * k + 2));
    double *v = d + k + 1;
    memcpy(d, node_depth, sizeof(double) * (size_t)k);
    memcpy(v, node_vp, sizeof(double) * (size_t)k);
    orc_interplayer_novar(k, d, v);
    if (sorted_depth) memcpy(sorted_depth, d, sizeof(double) * (size_t)k);
    if (sorted_vp) memcpy(sorted_vp, v, sizeof(double) * (size_t)k);
    double ll = orc_loglhood_rt(k, v, d + 1, src_offset, src_depth, nsrc, tobs, sigma, tpred);
    free(d);
    return ll;
}

/* Chain likelihood used by the MCMC moves below: LOGLHOOD_RT, with the AR(1) residual model when
 * the sampler runs with IAR = 1 (the chain's idxarRT / arparRT, loglhood.f90:171-182).  The chains'
 * AR state is registered with orc_set_chain_ar (NULL: IAR = 0) and indexed by chain.          */
static const int    *g_ar_idx = NULL;
static const double *g_ar_par = NULL;
static double        g_ar_mx  = 0.5;

void orc_set_chain_ar(const int *idxar, const double *arpar, double armx)
{
    g_ar_idx = idxar;
    g_ar_par = arpar;
    g_ar_mx  = armx;
}

/* ISMPPRIOR = 1: the sampler draws from the prior, every likelihood is LOGLHOOD2's constant
 * (loglhood.f90:704-716: obj%logL = 1). */
static int g_ismpprior = 0;
void orc_set_ismpprior(int on) { g_ismpprior = on ? 1 : 0; }

static double chain_loglhood(int chain, int k, const double *vp, const double *ziface,
                             const double *src_offset, const double *src_depth, int nsrc,
                             const double *tobs, double sigma)
{
    if (g_ismpprior) return 1.0;
    if (!g_ar_idx || chain < 0)
        return orc_loglhood_rt(k, vp, ziface, src_offset, src_depth, nsrc, tobs, sigma, NULL);
    double *pred = (double *)malloc(sizeof(double) * (size_t)(nsrc > 0 ? nsrc : 1));
    orc_loglhood_rt(k, vp, ziface, src_offset, src_depth, nsrc, tobs, sigma, pred);
    const double ll = orc_loglhood_from_times_ar(pred, tobs, nsrc, sigma, g_ar_idx[chain],
                                                 g_ar_par[chain], g_ar_mx);
    free(pred);
    return ll;
}

/* ---- "next" rows N1 + N2: one fixed-dimension Metropolis-Hastings move of one chain ---- *
 * The body of EXPLORE_MH_NOVARPAR's sweep for one (ivo, iwhich) (prjmh_temper_rf.f90:725-757):
 * PROPOSAL (:1386-1447, ENOS = 0: Cauchy step on voro(ivo,iwhich), |.| for the depth, then
 * INTERPLAYER_novar), CHECKBOUNDS2 (:1681-1716), LOGLHOOD, and the accept test
 * "reject iff ran_uni >= EXP(logPr + (logL_new - logL)*beta_mh)" (:742-751).
 * The random numbers are inputs: `cauchy` = TAN(PI*(ran_uni-0.5)), `u_acc` = ran_uni of :746.
 * prior = { fact/factor*pertsd(1), fact/factor*pertsd(2), minlim(1), minlim(2), maxlim(1),
 *           maxlim(2), hmin }  (read_input.f90:207-214, rjmcmc_com.f90:80).
 * node_depth/node_vp [k] are the chain's sorted nodes (in/out), *logL its current logL (in/out).
 * prop_depth/prop_vp [k] (may be NULL) receive the proposal after INTERPLAYER_novar, *logL_prop
 * (may be NULL) its logL (untouched when outside).  Returns 1 accepted, 0 rejected, -1 rejected
 * because the proposal left the prior bounds (ioutside).                                     */
/* ENOS (even-numbered order statistics prior, Green 1995; rjmcmc_com.f90) for the move oracles:
 * 0 = Cauchy depth steps and no order-statistics terms, 1 = uniform depth step between the
 * neighbouring nodes (PROPOSAL :1418-1431) and the prior ratios of DEATH_FULL :981-991 /
 * BIRTH_FULL :1090-1098.  With ENOS = 1 the `cauchy` argument of a depth move carries the
 * uniform deviate itself. */
static int g_enos = 0;
void orc_set_enos(int enos) { g_enos = enos ? 1 : 0; }

int orc_mh_step_chain(int chain, int k, double *node_depth, double *node_vp, double *logL,
                int ivo, int iwhich, double cauchy, double u_acc, double beta, double sigma,
                const double *prior,
                const double *src_offset, const double *src_depth, int nsrc, const double *tobs,
                double *prop_depth, double *prop_vp, double *logL_prop)
{
    const double scale[2] = {prior[0], prior[1]}, minlim[2] = {prior[2], prior[3]},
                 maxlim[2] = {prior[4], prior[5]}, hmin = prior[6];
    if (k < 1 || ivo < 1 || ivo > k || iwhich < 1 || iwhich > 2 || (ivo == 1 && iwhich == 1))
        return -1;                                               /* :730 CYCLE: nothing to propose */
    double *d = (double *)malloc(sizeof(double) * (size_t)(2 * k + 2));
    double *v = d + k + 1;
    memcpy(d, node_depth, sizeof(double) * (size_t)k);
    memcpy(v, node_vp, sizeof(double) * (size_t)k);
    double *tgt = (iwhich == 1) ? d : v;
    double logPr = 0.0;
    if (iwhich == 1 && g_enos) {                                 /* :1418-1431 */
        const double zj = d[ivo - 1], zjm1 = d[ivo - 2];
        const double zjp1 = (ivo == k) ? maxlim[0] : d[ivo];     /* hmx = maxlim(1) */
        const double zp = zjm1 + cauchy * (zjp1 - zjm1);
        d[ivo - 1] = zp;
        logPr = log(zjp1 - zp) + log(zp - zjm1) - log(zjp1 - zj) - log(zj - zjm1);
    } else
    tgt[ivo - 1] = tgt[ivo - 1] + scale[iwhich - 1] * cauchy;    /* :1405 / :1416 */
    if (iwhich == 1) d[ivo - 1] = fabs(d[ivo - 1]);              /* :1441-1443 */
    int ordered = 1;
    for (int i = 0; i < k; ++i) ordered = ordered && (d[i] == d[i]);
    if (ordered) orc_interplayer_novar(k, d, v);                 /* :1444 */
    if (prop_depth) memcpy(prop_depth, d, sizeof(double) * (size_t)k);
    if (prop_vp) memcpy(prop_vp, v, sizeof(double) * (size_t)k);
    /* CHECKBOUNDS2: ziface(i) = voro(i+1,1), hiface(1) = ziface(1), hiface(i) = ziface(i)-ziface(i-1) */
    int outside = 0;
    for (int ilay = 1; ilay <= k - 1; ++ilay) {
        const double zi = d[ilay];
        const double hi = (ilay == 1) ? zi : zi - d[ilay - 1];
        if (hmin > hi) outside = 1;                              /* :1693 */
        if (maxlim[0] < zi) outside = 1;                         /* :1694 */
    }
    if (ivo > 1 && (d[ivo - 1] < 0.0 || d[ivo - 1] > maxlim[0])) outside = 1;      /* :1698-1704 */
    {
        const double x = (iwhich == 1) ? d[ivo - 1] : v[ivo - 1];                 /* :1705-1712 */
        if ((x - minlim[iwhich - 1]) < 0.0 || (maxlim[iwhich - 1] - x) < 0.0) outside = 1;
    }
    int ret;
    if (outside) {
        ret = -1;                                                /* :753-757 */
    } else {
        const double ll = chain_loglhood(chain, k, v, d + 1, src_offset, src_depth, nsrc, tobs, sigma);
        if (logL_prop) *logL_prop = ll;
        const double logPLratio = logPr + (ll - *logL) * beta;   /* :743-745 */
        if (u_acc >= exp(logPLratio)) {
            ret = 0;                                             /* :747-749 */
        } else {
            memcpy(node_depth, d, sizeof(double) * (size_t)k);   /* :750 obj = objnew1 */
            memcpy(node_vp, v, sizeof(double) * (size_t)k);
            *logL = ll;
            ret = 1;
        }
    }
    free(d);
    return ret;
}

/* ---- N2: the birth/death move at the top of EXPLORE_MH_NOVARPAR (:658-710) -------------- *
 * Move choice from ran_unik (:666-680): at kmax only death, at kmin only birth, each with
 * probability 0.3333; otherwise birth if <= 0.3333, death if > 0.6666.
 * BIRTH_FULL (:997-1103): new node k+1 with depth maxpert(1)*u_z and vp minlim(2)+maxpert(2)*u_v
 * (maxpert = maxlim - minlim, read_input.f90:213), INTERPLAYER_novar.
 * DEATH_FULL (:917-994): node idel (2..k, the first element of RANDPERM(k-1) plus one) is zeroed,
 * the k nodes are sorted, the first one is dropped (:957-960), INTERPLAYER_novar.
 * logPr = LOG(pk(k_new)) - LOG(pk(k)) with the Poisson prior (IPOIPR = 1, ENOS = 0; :986,:1094),
 * 0 when pk is NULL (IPOIPR = 0).  CHECKBOUNDS (:1639-1678), LOGLHOOD, accept test (:689-699).
 * node_depth/node_vp have ldk slots; slots past k are zero and stay zero.
 * Returns 1 accepted, 0 rejected, -1 outside the bounds, 2 no birth/death proposed.        */
int orc_bd_step_chain(int chain, int *k_io, double *node_depth, double *node_vp, double *logL, int ldk,
                double u_k, int idel, double u_z, double u_v, double u_acc, double beta,
                double sigma, const double *prior, const double *pk, int kmin, int kmax,
                const double *src_offset, const double *src_depth, int nsrc, const double *tobs,
                int *k_prop, double *prop_depth, double *prop_vp, double *logL_prop)
{
    const double minlim[2] = {prior[2], prior[3]}, maxlim[2] = {prior[4], prior[5]}, hmin = prior[6];
    const int k = *k_io;
    int i_bd = 0;
    if (kmin != kmax) {                                          /* :661-680 */
        if (k == kmax)      { if (u_k <= 0.3333) i_bd = 2; }
        else if (k == kmin) { if (u_k <= 0.3333) i_bd = 1; }
        else { if (u_k <= 0.3333) i_bd = 1; if (u_k > 0.6666) i_bd = 2; }
    }
    if (k_prop) *k_prop = k;
    if (i_bd == 0) return 2;
    if (k < 1 || k > ldk || (i_bd == 1 && k + 1 > ldk) || (i_bd == 2 && (k < 2 || idel < 2 || idel > k)))
        return -1;
    double *d = (double *)calloc((size_t)(2 * ldk + 2), sizeof(double));
    double *v = d + ldk + 1;
    memcpy(d, node_depth, sizeof(double) * (size_t)k);
    memcpy(v, node_vp, sizeof(double) * (size_t)k);
    int kn;
    double et[6];                /* the order-statistics terms, added left to right as the Fortran does */
    int net = 0, enos_bad = 0;
    const double hmx = maxlim[0], kk = (double)k;
    if (i_bd == 1) {
        kn = k + 1;
        const double znew = (maxlim[0] - minlim[0]) * u_z;       /* :1035-1040 */
        d[k] = znew;
        v[k] = minlim[1] + (maxlim[1] - minlim[1]) * u_v;        /* :1051 */
        orc_interplayer_novar(kn, d, v);                         /* :1057 */
        if (g_enos) {                                            /* :1061-1073, :1090-1098 */
            int iznew = 0;
            for (int ivo = 1; ivo <= k; ++ivo)
                if (d[ivo] - znew == 0.0) iznew = ivo + 1;       /* ziface(ivo) = voro(ivo+1,1) */
            if (iznew == 0) enos_bad = 1;                        /* the reference would index voro(-1) */
            else {
                const double zj = d[iznew - 2];
                const double zjp1 = (iznew > k) ? hmx : d[iznew];
                et[0] = log(2.0 * kk + 2.0);  et[1] = log(2.0 * kk + 3.0);  et[2] = -(2.0 * log(hmx - hmin));
                et[3] = log(znew - zj);       et[4] = log(zjp1 - znew);     et[5] = -log(zjp1 - zj);
                net = 6;
            }
        }
    } else {
        kn = k - 1;
        if (g_enos) {                                            /* :941-947, :981-991 */
            const double zdel = d[idel - 1], zj = d[idel - 2];
            const double zjp1 = (idel == k) ? hmx : d[idel];
            et[0] = 2.0 * log(hmx - hmin);  et[1] = -log(2.0 * kk * (2.0 * kk + 1.0));
            et[2] = log(zjp1 - zj);         et[3] = -log(zdel - zj);        et[4] = -log(zjp1 - zdel);
            net = 5;
        }
        d[idel - 1] = 0.0;                                       /* :948 */
        v[idel - 1] = 0.0;
        orc_interplayer_novar(k, d, v);                          /* :951-953 QSORTC2D over k nodes */
        for (int i = 0; i < kn; ++i) { d[i] = d[i + 1]; v[i] = v[i + 1]; }   /* :957 */
        d[kn] = 0.0; v[kn] = 0.0;                                /* :959 */
        orc_interplayer_novar(kn, d, v);                         /* :962 */
    }
    double logPr = pk ? log(pk[kn - 1]) - log(pk[k - 1]) : 0.0;             /* :986 / :1094 */
    if (g_enos && net) {                                                    /* :981-991 / :1090-1098 */
        double acc = pk ? logPr + et[0] : et[0];
        for (int i = 1; i < net; ++i) acc = acc + et[i];
        logPr = acc;
    }
    if (k_prop) *k_prop = kn;
    if (prop_depth) memcpy(prop_depth, d, sizeof(double) * (size_t)ldk);
    if (prop_vp) memcpy(prop_vp, v, sizeof(double) * (size_t)ldk);
    int outside = 0;                                             /* CHECKBOUNDS :1650-1674 */
    for (int ilay = 1; ilay <= kn - 1; ++ilay) {
        const double zi = d[ilay];
        const double hi = (ilay == 1) ? zi : zi - d[ilay - 1];
        if (hmin > hi) outside = 1;
        if (maxlim[0] < zi) outside = 1;
    }
    for (int ivo = 1; ivo <= kn; ++ivo) {
        if (ivo > 1 && (d[ivo - 1] < 0.0 || d[ivo - 1] > maxlim[0])) outside = 1;
        if ((v[ivo - 1] - minlim[1]) < 0.0 || (maxlim[1] - v[ivo - 1]) < 0.0) outside = 1;
    }
    if (enos_bad) outside = 1;
    int ret;
    if (outside) {
        ret = -1;                                                /* :700-704 */
    } else {
        const double ll = chain_loglhood(chain, kn, v, d + 1, src_offset, src_depth, nsrc, tobs, sigma);
        if (logL_prop) *logL_prop = ll;
        const double logPLratio = logPr + (ll - *logL) * beta;   /* :689-691 */
        if (u_acc >= exp(logPLratio)) {
            ret = 0;
        } else {
            memcpy(node_depth, d, sizeof(double) * (size_t)ldk);
            memcpy(node_vp, v, sizeof(double) * (size_t)ldk);
            *logL = ll;
            *k_io = kn;
            ret = 1;
        }
    }
    free(d);
    return ret;
}

void orc_bd_step_batch(int *k, double *voro, double *logL, int B, int ldk, const double *u_k,
                       const int *idel, const double *u_z, const double *u_v, const double *u_acc,
                       const double *beta, const double *sigma, const double *prior,
                       const double *pk, int kmin, int kmax,
                       const double *src_offset, const double *src_depth, int nsrc,
                       const double *tobs, int *accept, int *k_prop, double *voro_prop,
                       double *logL_prop)
{
#pragma omp parallel for schedule(dynamic, 16)
    for (int b = 0; b < B; ++b) {
        double *row = voro + (size_t)b * 2 * ldk;
        double *pr = voro_prop ? voro_prop + (size_t)b * 2 * ldk : NULL;
        accept[b] = orc_bd_step_chain(b, &k[b], row, row + ldk, &logL[b], ldk, u_k[b], idel[b], u_z[b], u_v[b],
                                u_acc[b], beta[b], sigma[b], prior, pk, kmin, kmax, src_offset,
                                src_depth, nsrc, tobs, k_prop ? &k_prop[b] : NULL, pr,
                                pr ? pr + ldk : NULL, logL_prop ? &logL_prop[b] : NULL);
    }
}

/* ---- the data-error move of EXPLORE_MH (:545-575): with probability 0.9 (ran_uni_ar >= 0.10)
 * PROPOSAL_SDRT (:1616-1635: sdparRT + pertsdsdRT*gauss, outside unless within [minlimsdRT,
 * maxlimsdRT]), LOGLHOOD (the travel times are recomputed: LOGLHOOD_RT ignores ipred), and
 * "reject iff ran_uni >= EXP((logL_new - logL)*beta_mh)".  sd_prior = { pertsdsdRT, minlimsdRT,
 * maxlimsdRT } (read_input.f90:237-241).  Returns 1 / 0 / -1 outside / 2 no move.            */
int orc_sd_step_chain(int chain, int k, const double *node_depth, const double *node_vp, double *logL, double *sigma,
                double u_gate, double gauss, double u_acc, double beta, const double *sd_prior,
                const double *src_offset, const double *src_depth, int nsrc, const double *tobs,
                double *logL_prop)
{
    if (!(u_gate >= 0.10)) return 2;                             /* :553-554 */
    const double snew = *sigma + sd_prior[0] * gauss;            /* :1630 */
    if ((snew - sd_prior[1]) < 0.0 || (sd_prior[2] - snew) < 0.0) return -1;   /* :1631-1632, :569-573 */
    const double ll = chain_loglhood(chain, k, node_vp, node_depth + 1, src_offset, src_depth, nsrc, tobs,
                                     snew);
    if (logL_prop) *logL_prop = ll;
    const double logPLratio = (ll - *logL) * beta;               /* :560 */
    if (u_acc >= exp(logPLratio)) return 0;                      /* :562-564 */
    *sigma = snew;                                               /* :566 */
    *logL = ll;
    return 1;
}

void orc_sd_step_batch(const int *k, const double *voro, double *logL, double *sigma, int B, int ldk,
                       const double *u_gate, const double *gauss, const double *u_acc,
                       const double *beta, const double *sd_prior,
                       const double *src_offset, const double *src_depth, int nsrc,
                       const double *tobs, int *accept, double *logL_prop)
{
#pragma omp parallel for schedule(dynamic, 16)
    for (int b = 0; b < B; ++b) {
        const double *row = voro + (size_t)b * 2 * ldk;
        accept[b] = orc_sd_step_chain(b, k[b], row, row + ldk, &logL[b], &sigma[b], u_gate[b], gauss[b],
                                u_acc[b], beta[b], sd_prior, src_offset, src_depth, nsrc, tobs,
                                logL_prop ? &logL_prop[b] : NULL);
    }
}

/* ---- the AR(1) move of EXPLORE_MH (:583-631, IAR = 1) with PROPOSAL_ARRT (:1521-1552) --------- *
 * idxarRT == 0: birth (arparRT uniform over [minlimarRT, maxlimarRT], logarp = LOG(0.5));
 * else ran_uni_ar >= 0.5: death (idxarRT = 0, arparRT = minlimarRT - 1, logarp = LOG(2)),
 * otherwise perturb (arparRT + pertarsdRT*gauss, logarp = 0).  LOGLHOOD with the AR model of
 * loglhood.f90:171-182 (LOGLHOOD2's constant 1 under ISMPPRIOR = 1, as for the other moves);
 * reject iff ran_uni >= EXP(logarp + (logL_new - logL)*beta_mh).
 * ar_prior = { pertarsdRT, minlimarRT, maxlimarRT, armxRT }.  Returns 1 / 0 / -1 outside.     */
int orc_ar_step(int k, const double *node_depth, const double *node_vp, double *logL, double sigma,
                int *idxar, double *arpar, double u_choice, double u_prop, double gauss,
                double u_acc, double beta, const double *ar_prior,
                const double *src_offset, const double *src_depth, int nsrc, const double *tobs,
                double *logL_prop)
{
    const double pert = ar_prior[0], amin = ar_prior[1], amax = ar_prior[2], armx = ar_prior[3];
    int idx_new, outside = 0;
    double ar_new, logarp;
    if (*idxar == 0) {                                           /* :588-591, :1531-1537 */
        logarp = log(0.5);
        ar_new = u_prop * (amax - amin) + amin;
        idx_new = 1;
        if ((ar_new - amin) < 0.0 || (amax - ar_new) < 0.0) outside = 1;
    } else if (u_choice >= 0.5) {                                /* :594-597, :1539-1542 */
        logarp = log(2.0);
        ar_new = amin - 1.0;
        idx_new = 0;
    } else {                                                     /* :598-601, :1544-1549 */
        logarp = 0.0;
        ar_new = *arpar + pert * gauss;
        idx_new = *idxar;
        if ((ar_new - amin) < 0.0 || (amax - ar_new) < 0.0) outside = 1;
    }
    if (outside) return -1;                                      /* :621-625 */
    double ll = 1.0;                                             /* ISMPPRIOR = 1: LOGLHOOD2 */
    if (!g_ismpprior) {
        double *pred = (double *)malloc(sizeof(double) * (size_t)(nsrc > 0 ? nsrc : 1));
        orc_loglhood_rt(k, node_vp, node_depth + 1, src_offset, src_depth, nsrc, tobs, sigma, pred);
        ll = orc_loglhood_from_times_ar(pred, tobs, nsrc, sigma, idx_new, ar_new, armx);
        free(pred);
    }
    if (logL_prop) *logL_prop = ll;
    const double logPLratio = logarp + (ll - *logL) * beta;      /* :611 */
    if (u_acc >= exp(logPLratio)) return 0;                      /* :613-615 */
    *idxar = idx_new;                                            /* :617 */
    *arpar = ar_new;
    *logL = ll;
    return 1;
}

void orc_ar_step_batch(const int *k, const double *voro, double *logL, const double *sigma,
                       int *idxar, double *arpar, int B, int ldk, const double *u_choice,
                       const double *u_prop, const double *gauss, const double *u_acc,
                       const double *beta, const double *ar_prior,
                       const double *src_offset, const double *src_depth, int nsrc,
                       const double *tobs, int *accept, double *logL_prop)
{
#pragma omp parallel for schedule(dynamic, 16)
    for (int b = 0; b < B; ++b) {
        const double *row = voro + (size_t)b * 2 * ldk;
        accept[b] = orc_ar_step(k[b], row, row + ldk, &logL[b], sigma[b], &idxar[b], &arpar[b],
                                u_choice[b], u_prop[b], gauss[b], u_acc[b], beta[b], ar_prior,
                                src_offset, src_depth, nsrc, tobs, logL_prop ? &logL_prop[b] : NULL);
    }
}

/* B independent chains, one move each; voro [B][2][ldk] (depth row, vp row), OpenMP over chains. */
void orc_mh_step_batch(const int *k, double *voro, double *logL, int B, int ldk,
                       const int *ivo, const int *iwhich, const double *cauchy, const double *u_acc,
                       const double *beta, const double *sigma, const double *prior,
                       const double *src_offset, const double *src_depth, int nsrc,
                       const double *tobs, int *accept, double *voro_prop, double *logL_prop)
{
#pragma omp parallel for schedule(dynamic, 16)
    for (int b = 0; b < B; ++b) {
        double *row = voro + (size_t)b * 2 * ldk;
        double *pr = voro_prop ? voro_prop + (size_t)b * 2 * ldk : NULL;
        accept[b] = orc_mh_step_chain(b, k[b], row, row + ldk, &logL[b], ivo[b], iwhich[b], cauchy[b],
                                u_acc[b], beta[b], sigma[b], prior, src_offset, src_depth, nsrc,
                                tobs, pr, pr ? pr + ldk : NULL, logL_prop ? &logL_prop[b] : NULL);
    }
}

/* ---- "next" row N4: the AR(1) residual error model of IAR = 1 ------------------------ *
 * ll:171-182: DarRT from ARPRED_RT (ll:616-653, order 1: DarRT(i) = arpar*DresRT(i-1) for
 * 1 < i < N, 0 at both ends), DresRT = DresRT - DarRT, CHECKBOUNDS_ARMXRT (ll:678-699) rejects
 * the state (logL = -HUGE) when MAXVAL(DarRT) > armx or MINVAL(DarRT) < -armx.            */
double orc_loglhood_from_times_ar(const double *tpred, const double *tobs, int ndat, double sigma,
                                  int idxar, double arpar, double armx)
{
    double *res = (double *)malloc(sizeof(double) * (size_t)(ndat > 0 ? ndat : 1));
    double *dar = (double *)calloc((size_t)(ndat > 0 ? ndat : 1), sizeof(double));
    for (int i = 0; i < ndat; ++i) res[i] = tobs[i] - tpred[i];            /* ll:166 */
    if (idxar == 1) {
        for (int i = 1; i < ndat; ++i) dar[i] = 0.0 + arpar * res[i - 1];  /* ll:640-650, k = 1 */
        if (ndat > 0) { dar[0] = 0.0; dar[ndat - 1] = 0.0; }               /* ll:652-653 */
    }
    int bad = 0;
    double mx = -DBL_MAX, mn = DBL_MAX;
    for (int i = 0; i < ndat; ++i) { if (dar[i] > mx) mx = dar[i]; if (dar[i] < mn) mn = dar[i]; }
    if (ndat > 0 && (mx > armx || mn < -armx)) bad = 1;                    /* ll:686-695 */
    double ss = 0.0;
    for (int i = 0; i < ndat; ++i) { double r = res[i] - dar[i]; ss = ss + r * r; }   /* ll:178,195 */
    double n = (double)ndat;
    double logL = log(1.0 / pow(2.0 * ORC_PI, n / 2.0)) - (ss / (2.0 * (sigma * sigma)) + n * log(sigma));
    if (isnan(logL)) logL = -DBL_MAX;
    if (bad) logL = -DBL_MAX;                                              /* ll:204-206 */
    free(res); free(dar);
    return logL;
}
