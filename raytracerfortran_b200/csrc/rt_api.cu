// rt_api.cu -- the C ABI of libraytrace_b200.so (include/raytrace_b200.h) and the host-side
// runtime around the kernels: device selection, cached device buffers, the chunked
// H2D -> kernel -> D2H pipeline for host callers, tile geometry, rays.dat output.
//
// There is deliberately no CPU implementation of the path in this file: if CUDA is not
// usable the entries report the failure (NaN outputs + stderr for the Fortran-style ones,
// non-zero status for the others).
#include "../../include/raytrace_b200.h"
#include "rt_internal.h"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <mutex>
#include <string>
#include <thread>
#include <type_traits>
#include <vector>
#if defined(__x86_64__)
#include <emmintrin.h>
#endif

namespace {

using rtb::BatchArgs;
using rtb::TileCfg;

constexpr double kPi = 3.141592653589793238462643383279502884197;  // data_type.f90:5 (PI2)
constexpr int    kMaxChunks = 64;
constexpr int    kSchedSlots = 256;  // tile-scheduler counter pairs, one per launch in flight
constexpr int    kGraphSlots = 512;  // further pairs owned by the kernel nodes of a captured graph (two graphs)
constexpr int    kDeepLdv = 40;     // models with this many velocities or more use the deep-model kernel

struct DevBuf {
    void  *p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <class T> T *as() const { return static_cast<T *>(p); }
};

// A captured CUDA graph and the key of everything its capture baked in.
struct GraphCache {
    cudaGraphExec_t     exec = nullptr;
    std::vector<size_t> key;
    void reset() {
        if (exec) cudaGraphExecDestroy(exec);
        exec = nullptr;
        key.clear();
    }
};

struct Ctx {
    bool inited = false, ok = false;
    int  device = 0, sms = 0, smem_optin = 0;
    cudaStream_t s_comp = nullptr, s_comp2 = nullptr, s_h2d = nullptr, s_d2h = nullptr;
    cudaEvent_t  ev_h2d[kMaxChunks], ev_d2h[kMaxChunks], ev_k0[kMaxChunks], ev_k1[kMaxChunks];
    cudaEvent_t  ev_t0 = nullptr, ev_t1 = nullptr;
    DevBuf vels, depths, nl, off, dep, tobs, sigma, timeP, pout, logL, arena, voro, vsorted,
        idxar, arparb, sched, mh_ll, mh_out, mh_kp, mh_lpr,
        // the derivative entries': the gradient's weights; the derivatives with respect to the
        // model (the gradient's sums, the Jacobian's rows) and to the sources; the normal equations
        // (JtJ also holds the second derivatives' H)
        w, dvels, ddepths, dtdr, dtdd, JtJ, Jtr;
    // The scratch buffers above (vels ... Jtr) are shared by every entry.  Entries that return
    // without synchronising (a caller stream was given) leave an event behind; any later entry that
    // uses the scratch from another stream first makes that stream wait for it.
    cudaEvent_t  ev_scratch = nullptr;
    cudaStream_t scratch_stream = nullptr;
    bool         scratch_pending = false;
    unsigned sched_seq = 0;        // launches take scheduler slots round robin
    bool     sched_dirty = false;  // a CUDA call failed: a kernel may have left counters behind
    GraphCache   mv;               // a run of MH moves (rtb200_mh_moves_device)
    GraphCache   mc;               // a whole MCMC iteration (rtb200_mcmc_iterations_device)
    cudaStream_t s_cap = nullptr;
    // IAR = 1: the chains' AR(1) state, used by every likelihood evaluation of the move entries
    const int    *chain_idxar = nullptr;
    const double *chain_arpar = nullptr;
    double        chain_armx  = 0.5;
    void  *pin = nullptr;          // pinned staging for small calls
    size_t pin_cap = 0;
    // pinned ring for callers whose arrays are pageable (R vectors, Fortran arrays, numpy)
    void  *stage = nullptr;
    size_t stage_cap = 0;
    void  *stage_out = nullptr;    // pinned bounce buffer for logL
    size_t stage_out_cap = 0;
    cudaEvent_t ev_slot[4] = {nullptr, nullptr, nullptr, nullptr};
    int opt_stage = -1;            // -1 automatic (stage pageable inputs), 0 never, 1 always
    // mapped pinned buffer of the one-model latency path (dff_ / TraceRays)
    void  *lat = nullptr;
    size_t lat_cap = 0;
    int opt_latency = 1;           // 1: one-model calls take the latency kernel; 0: the batch kernel
    int opt_stable_lognorm = 0;    // 1: log-likelihood constant as -(N/2) log(2 pi) (finite for N >= 773)
    int opt_ismpprior = 0;         // 1: the chain moves sample the prior (LOGLHOOD2: logL = 1)
    // options (<= 0: automatic)
    int opt_variant = -1, opt_threads = 0, opt_tile_models = 0, opt_tile_sources = 0,
        opt_chunk_models = 0, opt_ctas = 0, opt_logl_shuffle = 0, opt_comp_streams = 0, opt_static_tiles = 0;
    // stats
    double    kernel_ms = 0.0, total_ms = 0.0;
    long long launches = 0;
    TileCfg   last{};
    int       last_ctas = 0;
    std::string err;
    bool warned = false;
};

Ctx g;

int fail(const std::string &what, cudaError_t e = cudaSuccess) {
    g.err = what;
    if (e != cudaSuccess) {
        g.sched_dirty = true;
        g.err += ": ";
        g.err += cudaGetErrorString(e);
    }
    return e != cudaSuccess ? (int)e : -1;
}

#define CK(call)                                                    \
    do {                                                            \
        cudaError_t e__ = (call);                                   \
        if (e__ != cudaSuccess) return fail(#call, e__);            \
    } while (0)

int pick_device() {
    const char *names[] = {"RTB200_DEVICE", "LOCAL_RANK"};
    for (const char *n : names) {
        const char *v = getenv(n);
        if (v && *v) return atoi(v);
    }
    return 0;
}

int ensure_init(int device = -1) {
    if (g.inited && (device < 0 || device == g.device)) {
        if (!g.ok) return -1;
        cudaSetDevice(g.device);
        return 0;
    }
    if (g.inited && g.ok) rtb200_shutdown();
    g.inited = true;
    g.ok = false;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail("no usable CUDA device (libraytrace_b200 has no CPU fallback)", e);
    g.device = device >= 0 ? device : pick_device();
    if (g.device < 0) return fail("negative CUDA device index (RTB200_DEVICE / LOCAL_RANK)");
    if (g.device >= n) g.device = g.device % n;      // more ranks than GPUs on this node: wrap
    CK(cudaSetDevice(g.device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, g.device));
    if (prop.major < 10)
        return fail(std::string("device '") + prop.name +
                    "' is not sm_100a; this library carries sm_100a code only");
    g.sms = prop.multiProcessorCount;
    CK(cudaDeviceGetAttribute(&g.smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, g.device));
    CK(cudaStreamCreateWithFlags(&g.s_comp, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&g.s_comp2, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&g.s_h2d, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&g.s_d2h, cudaStreamNonBlocking));
    for (int i = 0; i < kMaxChunks; ++i) {
        CK(cudaEventCreateWithFlags(&g.ev_h2d[i], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&g.ev_d2h[i], cudaEventDisableTiming));
        CK(cudaEventCreate(&g.ev_k0[i]));
        CK(cudaEventCreate(&g.ev_k1[i]));
    }
    CK(cudaEventCreate(&g.ev_t0));
    CK(cudaEventCreate(&g.ev_t1));
    CK(cudaEventCreateWithFlags(&g.ev_scratch, cudaEventDisableTiming));
    g.scratch_pending = false;
    CK(g.sched.reserve((kSchedSlots + 2 * kGraphSlots) * 2 * sizeof(int)));
    CK(cudaMemset(g.sched.p, 0, (kSchedSlots + 2 * kGraphSlots) * 2 * sizeof(int)));
    g.ok = true;
    g.err.clear();
    return 0;
}

int even_up(int x) { return (x + 1) & ~1; }

// Order this stream behind the last asynchronous user of the shared scratch (see Ctx).
int scratch_acquire(cudaStream_t st) {
    if (g.scratch_pending && g.scratch_stream != st) CK(cudaStreamWaitEvent(st, g.ev_scratch, 0));
    return 0;
}
// An entry has queued work on the scratch in `st`; `synced`: it has also waited for it.
int scratch_release(cudaStream_t st, bool synced) {
    if (synced) {
        if (g.scratch_stream == st) g.scratch_pending = false;
        return 0;
    }
    CK(cudaEventRecord(g.ev_scratch, st));
    g.scratch_stream = st;
    g.scratch_pending = true;
    return 0;
}

// Counter pair for one launch's dynamic tile scheduling (the kernel leaves it zeroed).
int *next_sched() {
    if (g.opt_static_tiles) return nullptr;
    if (g.sched_dirty) {
        cudaDeviceSynchronize();
        if (cudaMemset(g.sched.p, 0, (kSchedSlots + 2 * kGraphSlots) * 2 * sizeof(int)) != cudaSuccess) return nullptr;
        g.sched_dirty = false;
    }
    return g.sched.as<int>() + 2 * (g.sched_seq++ % kSchedSlots);
}

// Tile geometry for one launch (DESIGN.md "tiling").
int choose_cfg(int B, int ldv, int ldz, int nsrc, bool aligned, TileCfg &c) {
    if (ldv > 255) return fail("more than 254 interfaces per model are not supported");
    // variant: 1 lane state machine; 3 the same with branch-free, unrolled layer loops for deep
    // models (more registers, 2 CTAs/SM); 5 is chosen below.  Default: by depth; the option forces
    // 3 or 5, and any other value means 1
    c.variant = g.opt_variant < 0 ? (ldv >= kDeepLdv ? 3 : 1)
                                  : (g.opt_variant == 3 || g.opt_variant == 5 ? g.opt_variant : 1);
    c.threads = g.opt_threads > 0 ? std::min(256, (g.opt_threads + 31) / 32 * 32) : 256;
    c.LP = std::max(ldv, 2) | 1;
    c.SC = std::min(nsrc, g.opt_tile_sources > 0 ? g.opt_tile_sources : 256);
    c.TS = c.SC | 1;
    c.use_tma = aligned ? 1 : 0;
    c.logl_shuffle = g.opt_logl_shuffle;
    const int rays_target = c.threads * 8;
    int M = g.opt_tile_models > 0 ? g.opt_tile_models : std::max(2, rays_target / c.SC);
    M = g.opt_tile_models > 0 ? std::max(1, std::min(M, B)) : even_up(std::min(M, even_up(B)));
    const int want_ctas = g.opt_ctas > 0 ? g.opt_ctas : (c.variant == 3 ? 2 : 3);
    const size_t budget  = (size_t)g.smem_optin;
    const size_t per_cta = std::min<size_t>(budget, (size_t)(227 * 1024) / want_ctas - 1024);
    for (;;) {
        c.M = M;
        c.smem = rtb::tile_smem_bytes(c, ldv, ldz);
        const bool fits = c.smem <= per_cta && (size_t)M * c.SC <= 65536 && M <= 2048 && c.SC <= 4096 &&
                          (size_t)M * (ldv + ldz) * 8 < (1u << 20);
        if (fits) break;
        if (M > 2) {     // far too large: halve; close: step down
            M = (c.smem > per_cta + per_cta / 3) ? std::max(2, even_up(M / 2)) : M - 2;
            continue;
        }
        if (c.SC > 32) { c.SC = std::max(32, c.SC / 2); c.TS = c.SC | 1; continue; }
        if (c.smem <= budget) break;
        return fail("model rows too large for shared memory");
    }
    int occ = rtb::max_ctas_per_sm(c);
    if (occ < 1) return fail("batch kernel cannot be resident with this tile geometry");
    // few models: shrink the tile so one wave of CTAs covers the batch.  (Measured on 4096 and
    // 8192 trans-dimensional states x 256 sources: tiles of 2..7 or 12 models are no faster than
    // this rule's 8 -- such a batch is one or two waves of latency-bound tiles, not a queue of
    // rounds, so neither finer tiles nor "rounds x tile cost" tuning helps; profiles/r02_*.)
    if (g.opt_tile_models <= 0 && (B + c.M - 1) / c.M < g.sms * occ) {
        const int slots = g.sms * occ;
        const int m2 = std::max(2, even_up((B + slots - 1) / slots));
        if (m2 < c.M) {
            c.M = m2;
            c.smem = rtb::tile_smem_bytes(c, ldv, ldz);
            occ = std::max(occ, rtb::max_ctas_per_sm(c));
        }
    }
    const int ntiles = (B + c.M - 1) / c.M;
    // Shallow models: variant 5 (one segment of the sorted ray list per warp, so a warp's lanes
    // hold rays of one depth: -4.6 % on config 2) where its tiles' longer first-to-last-warp time
    // (nothing rebalances the warps inside a tile) is not exposed at the end of the launch: when
    // every CTA slot works through many tiles (150 000 models x 64 sources, 8 rounds: 5 % faster),
    // and when the launch is a single wave of full tiles anyway (4096 states x 256 sources: 2-3 %
    // faster).  In between it loses: 60 000 models (3 rounds) and the 8192 x 256 shape (2 rounds)
    // are 3-7 % slower with it, so those keep variant 1.
    const int slots = g.sms * occ;
    if (g.opt_variant < 0 && c.variant == 1 &&
        (ntiles >= 6 * slots || (ntiles <= slots && c.M * c.SC >= 1024))) {
        c.variant = 5;
        const int occ5 = rtb::max_ctas_per_sm(c);
        if (occ5 >= occ) occ = occ5; else c.variant = 1;
    }
    c.grid = std::max(1, std::min(ntiles, g.sms * occ));
    g.last_ctas = occ;
    return 0;
}

double log_norm_const(int nsrc) {
    // LOG(1._RP/(2._RP*PI2)**(REAL(NDAT_RT,RP)/2._RP))     loglhood.f90:194
    // For NDAT_RT >= 773 the power overflows, 1/Inf = 0 and the reference's logL is -Inf for every
    // model; that is reproduced by default.  Option "stable_lognorm" (a documented deviation, off
    // by default) evaluates the same constant as -(N/2) LOG(2 PI2), which stays finite.
    const double n = (double)nsrc;
    if (g.opt_stable_lognorm) return -(n / 2.0) * std::log(2.0 * kPi);
    return std::log(1.0 / std::pow(2.0 * kPi, n / 2.0));
}

bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

struct HostCall {
    const double *vels, *depths;
    const int    *nlayers;
    int B, ldv, ldz, kmode;
    const double *off, *dep;
    int nsrc;
    double *timeP;
    const double *tobs, *sigma;
    double *logL, *p_out;
    const int    *idxar = nullptr;     // AR(1) residual model: per-state switch, coefficient, bound
    const double *arpar = nullptr;
    double        armx  = 0.0;
};

// Small calls (the one-model dff_ of R's .Fortran, a handful of proposals): everything goes
// through one pinned staging buffer -- one H2D copy, one launch (cos_t computed in the kernel),
// one D2H copy, one stream -- because here the call is latency, not throughput.
constexpr size_t kSmallBytes = 256 * 1024;

int run_host_small(const HostCall &h, const TileCfg &cfg, int ldz) {
    const size_t B = (size_t)h.B, S = (size_t)h.nsrc, M = (size_t)cfg.M;
    const size_t Bpad = (B + M - 1) / M * M;
    auto up = [](size_t x) { return (x + 15) / 16 * 16; };
    size_t o = 0;
    const size_t o_v = o;   o += up(Bpad * h.ldv * 8);
    const size_t o_z = o;   o += up(Bpad * std::max(ldz, 1) * 8);
    const size_t o_off = o; o += up(S * 8);
    const size_t o_dep = o; o += up(S * 8);
    const size_t o_obs = o; o += up(S * 8);
    const size_t o_sig = o; o += up(B * 8);
    const size_t o_nl = o;  o += up(Bpad * 4);
    const size_t in_bytes = o;
    const size_t o_t = o;   o += h.timeP ? up(B * S * 8) : 0;
    const size_t o_p = o;   o += h.p_out ? up(B * S * 8) : 0;
    const size_t o_l = o;   o += h.logL ? up(B * 8) : 0;
    const size_t total = o;
    if (total > g.pin_cap) {
        if (g.pin) cudaFreeHost(g.pin);
        g.pin = nullptr; g.pin_cap = 0;
        CK(cudaMallocHost(&g.pin, 2 * total + 4096));
        g.pin_cap = 2 * total + 4096;
    }
    CK(g.arena.reserve(total));
    char *hp = static_cast<char *>(g.pin), *dp = g.arena.as<char>();
    memset(hp + o_v, 0, o_off - o_v);
    for (size_t b = 0; b < B; ++b) memcpy(hp + o_v + b * h.ldv * 8, h.vels + b * h.ldv, (size_t)h.ldv * 8);
    if (ldz > 0) memcpy(hp + o_z, h.depths, B * ldz * 8);
    memcpy(hp + o_off, h.off, S * 8);
    memcpy(hp + o_dep, h.dep, S * 8);
    if (h.tobs) memcpy(hp + o_obs, h.tobs, S * 8);
    if (h.sigma) memcpy(hp + o_sig, h.sigma, B * 8);
    memset(hp + o_nl, 0, Bpad * 4);
    memcpy(hp + o_nl, h.nlayers, B * 4);
    cudaStream_t st = g.s_comp;
    CK(cudaMemcpyAsync(dp, hp, in_bytes, cudaMemcpyHostToDevice, st));
    BatchArgs a{};
    a.vels = reinterpret_cast<double *>(dp + o_v);
    a.depths = reinterpret_cast<double *>(dp + o_z);
    a.nlayers = reinterpret_cast<int *>(dp + o_nl);
    a.B = h.B; a.ldv = h.ldv; a.ldz = ldz; a.kmode = h.kmode;
    a.src_offset = reinterpret_cast<double *>(dp + o_off);
    a.src_depth = reinterpret_cast<double *>(dp + o_dep);
    a.tobs = h.tobs ? reinterpret_cast<double *>(dp + o_obs) : nullptr;
    a.nsrc = h.nsrc;
    a.sigma = h.sigma ? reinterpret_cast<double *>(dp + o_sig) : nullptr;
    a.timeP = h.timeP ? reinterpret_cast<double *>(dp + o_t) : nullptr;
    a.p_out = h.p_out ? reinterpret_cast<double *>(dp + o_p) : nullptr;
    a.logL = h.logL ? reinterpret_cast<double *>(dp + o_l) : nullptr;
    a.logc = h.logL ? log_norm_const(h.nsrc) : 0.0;
    a.padded = 1;
    CK(cudaEventRecord(g.ev_k0[0], st));
    a.sched = next_sched();
    CK(rtb::launch_batch(a, cfg, st));
    CK(cudaEventRecord(g.ev_k1[0], st));
    g.launches++;
    g.last = cfg;
    if (total > in_bytes)
        CK(cudaMemcpyAsync(hp + in_bytes, dp + in_bytes, total - in_bytes, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (h.timeP) memcpy(h.timeP, hp + o_t, B * S * 8);
    if (h.p_out) memcpy(h.p_out, hp + o_p, B * S * 8);
    if (h.logL) memcpy(h.logL, hp + o_l, B * 8);
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, g.ev_k0[0], g.ev_k1[0]) == cudaSuccess) g.kernel_ms = g.total_ms = ms;
    return 0;
}

// Is this host pointer ordinary pageable memory (not pinned, not registered, not managed)?
bool is_pageable(const void *p) {
    if (!p) return false;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return true;
    }
    return a.type == cudaMemoryTypeUnregistered;
}

// Copy into the pinned ring with non-temporal stores: the destination is only read by the DMA
// engine, so it need not be fetched into (nor kept in) the caches; on a bandwidth-bound host this
// is a third less memory traffic than memcpy's read-for-ownership.  dst is 16-byte aligned.
void stream_copy(void *dst, const void *src, size_t bytes) {
#if defined(__x86_64__)
    if ((reinterpret_cast<uintptr_t>(dst) & 15u) == 0) {
        char *d = static_cast<char *>(dst);
        const char *s = static_cast<const char *>(src);
        size_t i = 0;
        for (; i + 64 <= bytes; i += 64) {
            const __m128i a = _mm_loadu_si128(reinterpret_cast<const __m128i *>(s + i));
            const __m128i b = _mm_loadu_si128(reinterpret_cast<const __m128i *>(s + i + 16));
            const __m128i c = _mm_loadu_si128(reinterpret_cast<const __m128i *>(s + i + 32));
            const __m128i e = _mm_loadu_si128(reinterpret_cast<const __m128i *>(s + i + 48));
            _mm_stream_si128(reinterpret_cast<__m128i *>(d + i), a);
            _mm_stream_si128(reinterpret_cast<__m128i *>(d + i + 16), b);
            _mm_stream_si128(reinterpret_cast<__m128i *>(d + i + 32), c);
            _mm_stream_si128(reinterpret_cast<__m128i *>(d + i + 48), e);
        }
        _mm_sfence();
        if (i < bytes) memcpy(d + i, s + i, bytes - i);
        return;
    }
#endif
    memcpy(dst, src, bytes);
}

// the copy split over a few host threads: one core moves a few GB/s, the H2D link takes 50+
void parallel_memcpy(void *dst, const void *src, size_t bytes) {
    constexpr size_t kMinPerThread = 1u << 20;
    static const unsigned cap = [] {
        const char *e = getenv("RTB200_COPY_THREADS");
        const unsigned hw = std::thread::hardware_concurrency();
        return e && atoi(e) > 0 ? (unsigned)atoi(e) : std::max(1u, std::min(hw / 2, 8u));
    }();
    size_t nt = std::min<size_t>(cap, std::max<size_t>(1, bytes / kMinPerThread));
    if (nt <= 1) {
        stream_copy(dst, src, bytes);
        return;
    }
    const size_t part = (bytes / nt + 63) & ~(size_t)63;
    std::vector<std::thread> th;
    size_t done_to = std::min(part, bytes);       // [0, done_to) is this thread's; helpers take the rest
    for (size_t t = 1; t < nt; ++t) {
        const size_t o = t * part;
        if (o >= bytes) break;
        try {                                      // a host that cannot start another thread: copy it here
            th.emplace_back([=] { stream_copy((char *)dst + o, (const char *)src + o, std::min(part, bytes - o)); });
        } catch (...) {
            stream_copy((char *)dst + o, (const char *)src + o, bytes - o);
            break;
        }
    }
    stream_copy(dst, src, done_to);
    for (auto &t : th) t.join();
}

// One model, no likelihood (dff_, dff7_, TraceRays): the call is pure latency.  Arguments are
// copied into a mapped pinned buffer the kernel reads and writes directly (zero-copy over PCIe), so
// the call is one memcpy, one launch of the one-warp-per-ray kernel, one stream synchronise.
constexpr int kLatencyMaxSources = 8192;

int run_host_latency(const HostCall &h) {
    const int NL = std::max(h.nlayers[0], 0), S = h.nsrc;
    const size_t n_in = (size_t)(2 * NL + 1) + 2 * (size_t)S, n_out = 2 * (size_t)S;
    const size_t bytes = (n_in + n_out) * 8 + 192;
    if (bytes > g.lat_cap) {
        if (g.lat) cudaFreeHost(g.lat);
        g.lat = nullptr; g.lat_cap = 0;
        CK(cudaHostAlloc(&g.lat, 2 * bytes, cudaHostAllocMapped));
        g.lat_cap = 2 * bytes;
    }
    double *in = static_cast<double *>(g.lat), *out = in + ((n_in + 7) & ~(size_t)7);
    memcpy(in, h.vels, (size_t)(NL + 1) * 8);
    if (NL > 0) memcpy(in + NL + 1, h.depths, (size_t)NL * 8);
    memcpy(in + 2 * NL + 1, h.off, (size_t)S * 8);
    memcpy(in + 2 * NL + 1 + S, h.dep, (size_t)S * 8);
    double *d_in = nullptr;
    CK(cudaHostGetDevicePointer((void **)&d_in, in, 0));
    double *d_out = d_in + (out - in);
    // completion flag after the outputs, on its own cache line
    volatile int *flag = reinterpret_cast<volatile int *>(out + ((n_out + 7) & ~(size_t)7));
    int *d_flag = reinterpret_cast<int *>(d_out + ((n_out + 7) & ~(size_t)7));
    *flag = 0;
    int single = 0;
    CK(rtb::launch_dff_latency(in, d_in, NL, S, d_out, h.p_out ? 1 : 0, d_flag, &single, g.s_comp));
    g.launches++;
    if (single) {
        // a single-CTA launch sets the flag after its last store: spinning on it is ~2 us
        // quicker than the stream synchronise; give up after a while so a faulting kernel
        // still surfaces as an error below
        for (long spin = 0; *flag == 0 && spin < 4000000; ++spin) {}
        if (*flag == 0) CK(cudaStreamSynchronize(g.s_comp));
    } else {
        CK(cudaStreamSynchronize(g.s_comp));
    }
    if (h.timeP) memcpy(h.timeP, out, (size_t)S * 8);
    if (h.p_out) memcpy(h.p_out, out + S, (size_t)S * 8);
    g.last = TileCfg{};
    g.last.variant = 9;            // what rtb200_get_stat("variant") reports for the latency kernel
    g.last.threads = std::min(S, 32) * 32;
    g.last.grid = (S + 31) / 32;
    return 0;
}

// Host buffers in, host buffers out: chunked over the model axis so the copy of chunk j+1
// and the read-back of chunk j-1 overlap the kernel of chunk j.
int run_host(const HostCall &h) {
    if (int rc = ensure_init()) return rc;
    g.err.clear();
    g.kernel_ms = g.total_ms = 0.0;
    if (h.B <= 0 || h.nsrc <= 0) return 0;
    if (h.ldv < 1) return fail("ldv must be >= 1");
    if (h.logL && (!h.tobs || !h.sigma)) return fail("logL needs tobs and sigma");
    const size_t B = (size_t)h.B, S = (size_t)h.nsrc;
    const int ldz = std::max(h.ldz, 0);
    if (g.opt_latency && g.opt_variant < 0 && h.B == 1 && !h.logL && !h.kmode && !h.idxar &&
        h.nsrc <= kLatencyMaxSources) {
        const int nl0 = std::max(h.nlayers[0], 0);
        if (nl0 + 1 <= h.ldv && nl0 <= ldz && nl0 <= 254) return run_host_latency(h);
    }

    TileCfg cfg;
    if (int rc = choose_cfg(h.B, h.ldv, ldz, h.nsrc, true, cfg)) return rc;
    {
        const size_t io = (B * (h.ldv + ldz + 2) + 3 * S) * 8 +
                          ((h.timeP ? B * S : 0) + (h.p_out ? B * S : 0) + (h.logL ? B : 0)) * 8;
        if (io <= kSmallBytes && !h.idxar) return run_host_small(h, cfg, ldz);
    }
    // our own buffers are padded to whole tiles, so TMA is always legal on them
    const size_t Bpad = (B + cfg.M - 1) / cfg.M * cfg.M + cfg.M;
    CK(g.vels.reserve(Bpad * h.ldv * 8));
    CK(g.depths.reserve(Bpad * std::max(ldz, 1) * 8));
    CK(g.nl.reserve(Bpad * 4));
    CK(g.off.reserve(S * 8));
    CK(g.dep.reserve(S * 8));
    if (h.tobs) CK(g.tobs.reserve(S * 8));
    if (h.sigma) CK(g.sigma.reserve(B * 8));
    if (h.timeP) CK(g.timeP.reserve(B * S * 8));
    if (h.p_out) CK(g.pout.reserve(B * S * 8));
    if (h.logL) CK(g.logL.reserve(B * 8));
    if (h.idxar) {
        CK(g.idxar.reserve(B * 4));
        CK(g.arparb.reserve(B * 8));
    }

    if (g.scratch_pending) {       // an asynchronous device-path call may still be reading the scratch
        CK(cudaStreamWaitEvent(g.s_h2d, g.ev_scratch, 0));
        CK(cudaStreamWaitEvent(g.s_comp, g.ev_scratch, 0));
        CK(cudaStreamWaitEvent(g.s_comp2, g.ev_scratch, 0));
    }
    CK(cudaEventRecord(g.ev_t0, g.s_h2d));
    CK(cudaMemcpyAsync(g.off.p, h.off, S * 8, cudaMemcpyHostToDevice, g.s_h2d));
    CK(cudaMemcpyAsync(g.dep.p, h.dep, S * 8, cudaMemcpyHostToDevice, g.s_h2d));
    if (h.tobs) CK(cudaMemcpyAsync(g.tobs.p, h.tobs, S * 8, cudaMemcpyHostToDevice, g.s_h2d));

    // Chunk boundaries are multiples of the tile size.  The default chunk is a whole number of
    // waves of the persistent grid (every CTA gets the same number of tiles), and consecutive
    // chunks alternate between two compute streams so the first CTAs of chunk j+1 take the SM
    // slots the last CTAs of chunk j leave instead of waiting for the whole grid to drain.
    const size_t wave = (size_t)g.sms * g.last_ctas * cfg.M;
    size_t chunk = g.opt_chunk_models > 0 ? (size_t)g.opt_chunk_models
                                          : std::max<size_t>(1, (65536 + wave / 2) / wave) * wave;
    const int ncomp = g.opt_comp_streams == 1 ? 1 : 2;
    chunk = std::max(chunk, (B + kMaxChunks - 1) / kMaxChunks);
    chunk = (chunk + cfg.M - 1) / cfg.M * cfg.M;
    // The first chunk is short (one wave when the default chunking is in force) so that the GPU
    // starts after a quarter of the copy time a full chunk would take; `lead` is its size.
    size_t lead = chunk;
    if (g.opt_chunk_models <= 0 && wave >= (size_t)cfg.M && wave < chunk && B > 2 * chunk &&
        (B - wave + chunk - 1) / chunk + 1 <= (size_t)kMaxChunks)
        lead = wave;
    const int nchunks = (int)(1 + (B > lead ? (B - lead + chunk - 1) / chunk : 0));

    const double logc = h.logL ? log_norm_const(h.nsrc) : 0.0;
    // A cudaMemcpyAsync from pageable memory is staged by the driver on the calling thread and
    // blocks it, so copy and compute no longer overlap.  Pageable inputs (what R vectors, Fortran
    // arrays and numpy arrays are) go through a pinned ring instead: a few host threads copy chunk
    // j+1 into its slot while the GPU works on chunk j, and the H2D from the slot is asynchronous.
    const size_t row_bytes = (size_t)h.ldv * 8 + (size_t)ldz * 8 + 4 + (h.sigma ? 8 : 0) + (h.idxar ? 12 : 0);
    const bool stage = g.opt_stage == 1 || (g.opt_stage < 0 && is_pageable(h.vels) && B * row_bytes > (8u << 20));
    constexpr int kSlots = 4;
    const size_t slot_models = std::max(chunk, lead);
    auto up64 = [](size_t x) { return (x + 63) & ~(size_t)63; };
    const size_t so_v = 0, so_z = so_v + up64(slot_models * h.ldv * 8), so_n = so_z + up64(slot_models * ldz * 8),
                 so_s = so_n + up64(slot_models * 4), so_i = so_s + up64(slot_models * 8),
                 so_a = so_i + up64(slot_models * 4), slot_bytes = so_a + up64(slot_models * 8);
    if (stage) {
        if (g.stage_cap < kSlots * slot_bytes) {
            if (g.lat) cudaFreeHost(g.lat);
    g.lat = nullptr;
    g.lat_cap = 0;
    if (g.stage) cudaFreeHost(g.stage);
            g.stage = nullptr; g.stage_cap = 0;
            CK(cudaMallocHost(&g.stage, kSlots * slot_bytes));
            g.stage_cap = kSlots * slot_bytes;
        }
        for (int i = 0; i < kSlots; ++i)
            if (!g.ev_slot[i]) CK(cudaEventCreateWithFlags(&g.ev_slot[i], cudaEventDisableTiming));
    }
    // logL comes back through a pinned bounce buffer when the caller's array is pageable
    double *logL_host = h.logL;
    if (h.logL && (g.opt_stage == 1 || (g.opt_stage < 0 && is_pageable(h.logL)))) {
        if (g.stage_out_cap < B * 8) {
            if (g.stage_out) cudaFreeHost(g.stage_out);
            g.stage_out = nullptr; g.stage_out_cap = 0;
            CK(cudaMallocHost(&g.stage_out, B * 8 + 4096));
            g.stage_out_cap = B * 8 + 4096;
        }
        logL_host = static_cast<double *>(g.stage_out);
    }
    for (int j = 0; j < nchunks; ++j) {
        const size_t j0 = j == 0 ? 0 : lead + (size_t)(j - 1) * chunk;
        const size_t j1 = std::min(B, j == 0 ? lead : j0 + chunk), nb = j1 - j0;
        const double *sv = h.vels + j0 * h.ldv, *sz = ldz > 0 ? h.depths + j0 * ldz : nullptr;
        const int    *sn = h.nlayers + j0, *si = h.idxar ? h.idxar + j0 : nullptr;
        const double *ss = h.sigma ? h.sigma + j0 : nullptr, *sa = h.idxar ? h.arpar + j0 : nullptr;
        if (stage) {
            const int slot = j % kSlots;
            char *base = static_cast<char *>(g.stage) + (size_t)slot * slot_bytes;
            if (j >= kSlots) CK(cudaEventSynchronize(g.ev_slot[slot]));     // the slot's last H2D is done
            parallel_memcpy(base + so_v, sv, nb * h.ldv * 8);
            if (sz) parallel_memcpy(base + so_z, sz, nb * ldz * 8);
            memcpy(base + so_n, sn, nb * 4);
            if (ss) memcpy(base + so_s, ss, nb * 8);
            if (si) { memcpy(base + so_i, si, nb * 4); memcpy(base + so_a, sa, nb * 8); }
            sv = reinterpret_cast<double *>(base + so_v);
            sz = sz ? reinterpret_cast<double *>(base + so_z) : nullptr;
            sn = reinterpret_cast<int *>(base + so_n);
            ss = ss ? reinterpret_cast<double *>(base + so_s) : nullptr;
            si = si ? reinterpret_cast<int *>(base + so_i) : nullptr;
            sa = sa ? reinterpret_cast<double *>(base + so_a) : nullptr;
        }
        CK(cudaMemcpyAsync(g.vels.as<double>() + j0 * h.ldv, sv, nb * h.ldv * 8,
                           cudaMemcpyHostToDevice, g.s_h2d));
        if (sz)
            CK(cudaMemcpyAsync(g.depths.as<double>() + j0 * ldz, sz, nb * ldz * 8, cudaMemcpyHostToDevice,
                               g.s_h2d));
        CK(cudaMemcpyAsync(g.nl.as<int>() + j0, sn, nb * 4, cudaMemcpyHostToDevice, g.s_h2d));
        if (ss) CK(cudaMemcpyAsync(g.sigma.as<double>() + j0, ss, nb * 8, cudaMemcpyHostToDevice, g.s_h2d));
        if (si) {
            CK(cudaMemcpyAsync(g.idxar.as<int>() + j0, si, nb * 4, cudaMemcpyHostToDevice, g.s_h2d));
            CK(cudaMemcpyAsync(g.arparb.as<double>() + j0, sa, nb * 8, cudaMemcpyHostToDevice, g.s_h2d));
        }
        if (stage) CK(cudaEventRecord(g.ev_slot[j % kSlots], g.s_h2d));
        CK(cudaEventRecord(g.ev_h2d[j], g.s_h2d));

        BatchArgs a{};
        a.vels = g.vels.as<double>() + j0 * h.ldv;
        a.depths = g.depths.as<double>() + j0 * ldz;
        a.nlayers = g.nl.as<int>() + j0;
        a.B = (int)nb; a.ldv = h.ldv; a.ldz = ldz; a.kmode = h.kmode;
        a.src_offset = g.off.as<double>(); a.src_depth = g.dep.as<double>();
        a.tobs = h.tobs ? g.tobs.as<double>() : nullptr;
        a.nsrc = h.nsrc;
        a.sigma = h.sigma ? g.sigma.as<double>() + j0 : nullptr;
        a.timeP = h.timeP ? g.timeP.as<double>() + j0 * S : nullptr;
        a.p_out = h.p_out ? g.pout.as<double>() + j0 * S : nullptr;
        a.logL = h.logL ? g.logL.as<double>() + j0 : nullptr;
        a.logc = logc;
        a.padded = 1;
        a.idxar = h.idxar ? g.idxar.as<int>() + j0 : nullptr;
        a.arpar = h.idxar ? g.arparb.as<double>() + j0 : nullptr;
        a.armx = h.armx;
        TileCfg cj = cfg;
        const int ntiles = (int)((nb + cfg.M - 1) / cfg.M);
        cj.grid = std::max(1, std::min(ntiles, g.sms * g.last_ctas));
        cudaStream_t sc = (j % ncomp) ? g.s_comp2 : g.s_comp;
        CK(cudaStreamWaitEvent(sc, g.ev_h2d[j], 0));
        CK(cudaEventRecord(g.ev_k0[j], sc));
        a.sched = next_sched();
        CK(rtb::launch_batch(a, cj, sc));
        CK(cudaEventRecord(g.ev_k1[j], sc));
        g.launches++;
        g.last = cj;

        CK(cudaStreamWaitEvent(g.s_d2h, g.ev_k1[j], 0));
        if (h.timeP)
            CK(cudaMemcpyAsync(h.timeP + j0 * S, a.timeP, nb * S * 8, cudaMemcpyDeviceToHost,
                               g.s_d2h));
        if (h.p_out)
            CK(cudaMemcpyAsync(h.p_out + j0 * S, a.p_out, nb * S * 8, cudaMemcpyDeviceToHost,
                               g.s_d2h));
        if (h.logL) {
            CK(cudaMemcpyAsync(logL_host + j0, a.logL, nb * 8, cudaMemcpyDeviceToHost, g.s_d2h));
            if (logL_host != h.logL) CK(cudaEventRecord(g.ev_d2h[j], g.s_d2h));
        }
    }
    CK(cudaEventRecord(g.ev_t1, g.s_d2h));
    if (h.logL && logL_host != h.logL) {
        // hand the chunks' logL to the caller's array as they arrive, under the later chunks' work
        for (int j = 0; j < nchunks; ++j) {
            const size_t j0 = j == 0 ? 0 : lead + (size_t)(j - 1) * chunk;
            const size_t j1 = std::min(B, j == 0 ? lead : j0 + chunk);
            CK(cudaEventSynchronize(g.ev_d2h[j]));
            memcpy(h.logL + j0, logL_host + j0, (j1 - j0) * 8);
        }
    }
    CK(cudaStreamSynchronize(g.s_d2h));
    CK(cudaStreamSynchronize(g.s_comp));
    CK(cudaStreamSynchronize(g.s_comp2));
    for (int j = 0; j < nchunks; ++j) {
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, g.ev_k0[j], g.ev_k1[j]));
        g.kernel_ms += ms;
    }
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, g.ev_t0, g.ev_t1) == cudaSuccess) g.total_ms = ms;
    return 0;
}

void nan_fill(double *p, size_t n) {
    if (!p) return;
    for (size_t i = 0; i < n; ++i) p[i] = std::numeric_limits<double>::quiet_NaN();
}

void complain() {
    if (!g.warned) {
        fprintf(stderr, "libraytrace_b200: %s\n", g.err.c_str());
        g.warned = true;
    }
}

// gfortran list-directed REAL(8): 17 significant digits (the look of the reference's rays.dat)
void put_ld(FILE *fh, double x) {
    char buf[64];
    const double ax = std::fabs(x);
    if (x == 0.0) {
        snprintf(buf, sizeof buf, "0.0000000000000000");
    } else if (ax >= 0.1 && ax < 1e17) {
        const int e10 = (int)std::floor(std::log10(ax));
        int dec = e10 < 0 ? 17 : 16 - e10;
        if (dec < 0) dec = 0;
        snprintf(buf, sizeof buf, "%.*f", dec, x);
    } else if (std::isfinite(x)) {
        const int e10 = (int)std::floor(std::log10(ax));
        snprintf(buf, sizeof buf, "%.16fE%+04d", x / std::pow(10.0, e10), e10);
        fprintf(fh, "%26s", buf);
        return;
    } else {
        snprintf(buf, sizeof buf, "%s", std::isnan(x) ? "NaN" : (x > 0 ? "Infinity" : "-Infinity"));
    }
    fprintf(fh, "%21s     ", buf);
}

// keep_delta > 0: rewrite ./rays.dat from the converged ray parameters
// (subroutineR-quiet.f90:98-105,157-164,432-433).  Formatting of results, host side.
void write_rays_dat(const double *vels, const double *depths, int NL, const double *off,
                    const double *dep, int nsrc, const double *p) {
    FILE *fh = fopen("rays.dat", "w");
    if (!fh) return;
    std::vector<double> H((size_t)NL + 2);
    for (int k = 0; k < nsrc; ++k) {
        int    inN = 0;
        double diff = 0.0;
        for (int i = 1; i <= NL; ++i) { inN = i; diff = depths[i - 1] - dep[k]; if (diff > 0.0) break; }
        const int nl = NL <= 0 ? 1 : (diff < 0.0 ? NL + 1 : inN);
        if (nl == 1) {
            put_ld(fh, off[k]); fputc('\n', fh);
            put_ld(fh, dep[k]); fputc('\n', fh);
            continue;
        }
        H[0] = depths[0];
        for (int i = 1; i < nl - 1; ++i) H[i] = depths[i] - depths[i - 1];
        H[nl - 1] = dep[k] - depths[nl - 2];
        for (int i = 0; i < nl; ++i) {
            volatile double pv = (p[k] * p[k]) * (vels[i] * vels[i]);
            volatile double cosv = std::sqrt(1.0 - pv);
            volatile double q = H[i] / cosv;
            volatile double q2 = q * q, h2 = H[i] * H[i];
            put_ld(fh, std::sqrt(q2 - h2));
        }
        fputc('\n', fh);
        for (int i = 0; i < nl; ++i) put_ld(fh, H[i]);
        fputc('\n', fh);
    }
    fclose(fh);
}

// The reference opens rays.dat with status='REPLACE' on every call (subroutineR-quiet.f90:432-433,
// :481-482), so after a call with keep_delta <= 0 the file is empty.  Doing that on every call
// would put a file open/close on the latency path; it is done when it is observable: on the first
// call of the process if the file exists, and after a call that wrote ray geometry.
bool g_rays_dirty = true;

void dff_impl(const double *vels, const double *depths, int NL, const double *off,
              const double *dep, int nsrc, double *timeP, int keep_delta) {
    if (keep_delta <= 0 && g_rays_dirty) {
        if (FILE *fh = fopen("rays.dat", "r")) {
            fclose(fh);
            if ((fh = fopen("rays.dat", "w"))) fclose(fh);
        }
        g_rays_dirty = false;
    }
    if (keep_delta > 0) g_rays_dirty = true;
    if (nsrc <= 0) return;
    std::vector<double> p;
    if (keep_delta > 0) p.resize((size_t)nsrc);
    HostCall h{};
    h.vels = vels; h.depths = depths; h.nlayers = &NL;
    h.B = 1; h.ldv = std::max(NL, 0) + 1; h.ldz = std::max(NL, 0); h.kmode = 0;
    h.off = off; h.dep = dep; h.nsrc = nsrc;
    h.timeP = timeP; h.p_out = keep_delta > 0 ? p.data() : nullptr;
    if (run_host(h) != 0) {
        nan_fill(timeP, (size_t)nsrc);
        complain();
        return;
    }
    if (keep_delta > 0) write_rays_dat(vels, depths, NL, off, dep, nsrc, p.data());
}

}  // namespace

// Every public entry takes this lock: calls from several host threads are serialised (the context
// below them -- cached buffers, options, the scratch of the chain moves -- is one per process).
static std::recursive_mutex g_api_mu;
struct ApiLock {
    std::lock_guard<std::recursive_mutex> l{g_api_mu};
};

extern "C" {

#ifdef RTB200_DFF_IS_7ARG
#define RTB200_DFF8 dff8_
#define RTB200_DFF7 dff_
#else
#define RTB200_DFF8 dff_
#define RTB200_DFF7 dff7_
#endif

void RTB200_DFF8(const double *vels, const double *depths, const int *NLayers,
                 const double *src_offset, const double *src_depth, const int *NSrc,
                 double *timeP, const int *keep_delta) {
    ApiLock api_lock_;
    dff_impl(vels, depths, *NLayers, src_offset, src_depth, *NSrc, timeP,
             keep_delta ? *keep_delta : -1);
}

void RTB200_DFF7(const double *vels, const double *depths, const int *NLayers,
                 const double *src_offset, const double *src_depth, const int *NSrc,
                 double *timeP) {
    ApiLock api_lock_;
    dff_impl(vels, depths, *NLayers, src_offset, src_depth, *NSrc, timeP, -1);
}

void tracerays_(const double *vels, const double *depths, const int *NLayers,
                const double *src_offset, const double *src_depth, const int *NSrc,
                double *timeP, const int *keep_delta) {
    ApiLock api_lock_;
    dff_impl(vels, depths, *NLayers, src_offset, src_depth, *NSrc, timeP,
             keep_delta ? *keep_delta : -1);
}

// module raymod's TraceRays under the names Fortran compilers give a module procedure, so objects
// compiled against the reference's raymod.mod (loglhood.o) link without the shim: explicit-shape
// arrays are plain pointers and scalars go by reference, the same ABI as tracerays_.
#define RTB200_TRACERAYS_ALIAS(name)                                                        \
    void name(const double *vels, const double *depths, const int *NLayers,                 \
              const double *src_offset, const double *src_depth, const int *NSrc,           \
              double *timeP, const int *keep_delta) {                                       \
        tracerays_(vels, depths, NLayers, src_offset, src_depth, NSrc, timeP, keep_delta);  \
    }
RTB200_TRACERAYS_ALIAS(__raymod_MOD_tracerays)   // gfortran
RTB200_TRACERAYS_ALIAS(raymod_mp_tracerays_)     // ifort / ifx
RTB200_TRACERAYS_ALIAS(raymod_tracerays_)        // nvfortran / PGI (the compiler of the shipped binary)
#undef RTB200_TRACERAYS_ALIAS

int dff_batch(const double *vels, const double *depths, const int *nlayers, const int *B,
              const int *ldv, const int *ldz, const double *src_offset, const double *src_depth,
              const int *NSrc, double *timeP, const double *tobs, const double *sigma,
              double *logL, double *p_out) {
    ApiLock api_lock_;
    HostCall h{};
    h.vels = vels; h.depths = depths; h.nlayers = nlayers;
    h.B = *B; h.ldv = *ldv; h.ldz = *ldz; h.kmode = 0;
    h.off = src_offset; h.dep = src_depth; h.nsrc = *NSrc;
    h.timeP = timeP; h.tobs = tobs; h.sigma = sigma; h.logL = logL; h.p_out = p_out;
    return run_host(h);
}

void dff_batch_status(const double *vels, const double *depths, const int *nlayers, const int *B,
                      const int *ldv, const int *ldz, const double *src_offset,
                      const double *src_depth, const int *NSrc, double *timeP, const double *tobs,
                      const double *sigma, double *logL, double *p_out, const int *want,
                      int *status) {
    ApiLock api_lock_;
    const bool wt = want && want[0], wl = want && want[1], wp = want && want[2];
    const int rc = dff_batch(vels, depths, nlayers, B, ldv, ldz, src_offset, src_depth, NSrc,
                             wt ? timeP : nullptr, wl ? tobs : nullptr, wl ? sigma : nullptr,
                             wl ? logL : nullptr, wp ? p_out : nullptr);
    if (status) *status = rc;
    if (rc != 0) complain();
}

void dff_batch_status_(const double *vels, const double *depths, const int *nlayers, const int *B,
                       const int *ldv, const int *ldz, const double *src_offset,
                       const double *src_depth, const int *NSrc, double *timeP, const double *tobs,
                       const double *sigma, double *logL, double *p_out, const int *want,
                       int *status) {
    ApiLock api_lock_;
    dff_batch_status(vels, depths, nlayers, B, ldv, ldz, src_offset, src_depth, NSrc, timeP, tobs,
                     sigma, logL, p_out, want, status);
}

int loglhood_batch(const int *k, const double *vp, const double *ziface, const int *B,
                   const int *ldv, const int *ldz, const double *src_offset,
                   const double *src_depth, const int *NSrc, const double *tobs,
                   const double *sigma, double *logL, double *tpred) {
    ApiLock api_lock_;
    HostCall h{};
    h.vels = vp; h.depths = ziface; h.nlayers = k;
    h.B = *B; h.ldv = *ldv; h.ldz = *ldz; h.kmode = 1;
    h.off = src_offset; h.dep = src_depth; h.nsrc = *NSrc;
    h.timeP = tpred; h.tobs = tobs; h.sigma = sigma; h.logL = logL; h.p_out = nullptr;
    return run_host(h);
}

int loglhood_batch_ar(const int *k, const double *vp, const double *ziface, const int *B,
                      const int *ldv, const int *ldz, const double *src_offset,
                      const double *src_depth, const int *NSrc, const double *tobs,
                      const double *sigma, const int *idxar, const double *arpar,
                      const double *armx, double *logL, double *tpred) {
    ApiLock api_lock_;
    HostCall h{};
    h.vels = vp; h.depths = ziface; h.nlayers = k;
    h.B = *B; h.ldv = *ldv; h.ldz = *ldz; h.kmode = 1;
    h.off = src_offset; h.dep = src_depth; h.nsrc = *NSrc;
    h.timeP = tpred; h.tobs = tobs; h.sigma = sigma; h.logL = logL; h.p_out = nullptr;
    h.idxar = idxar; h.arpar = arpar; h.armx = armx ? *armx : 0.5;
    if (idxar && !arpar) return fail("loglhood_batch_ar needs arpar with idxar");
    return run_host(h);
}

int loglhood_batch_voro(const int *k, const double *voro, const int *B, const int *ldk,
                        const double *src_offset, const double *src_depth, const int *NSrc,
                        const double *tobs, const double *sigma, double *logL, double *tpred,
                        double *voro_sorted) {
    ApiLock api_lock_;
    if (int rc = ensure_init()) return rc;
    g.err.clear();
    g.kernel_ms = g.total_ms = 0.0;
    const int nb = *B, ld = *ldk, ns = *NSrc;
    if (nb <= 0 || ns <= 0) return 0;
    if (ld < 1 || ld > 64) return fail("loglhood_batch_voro supports 1..64 nodes per state");
    if (!logL || !tobs || !sigma) return fail("loglhood_batch_voro needs tobs, sigma and logL");
    const size_t Bz = (size_t)nb, S = (size_t)ns;
    TileCfg cfg;
    if (int rc = choose_cfg(nb, ld, ld, ns, true, cfg)) return rc;
    const size_t Bpad = (Bz + cfg.M - 1) / cfg.M * cfg.M + cfg.M;
    CK(g.voro.reserve(Bz * 2 * ld * 8));
    if (voro_sorted) CK(g.vsorted.reserve(Bz * 2 * ld * 8));
    CK(g.vels.reserve(Bpad * ld * 8));
    CK(g.depths.reserve(Bpad * ld * 8));
    CK(g.nl.reserve(Bpad * 4));
    CK(g.off.reserve(S * 8)); CK(g.dep.reserve(S * 8)); CK(g.tobs.reserve(S * 8));
    CK(g.sigma.reserve(Bz * 8)); CK(g.logL.reserve(Bz * 8));
    if (tpred) CK(g.timeP.reserve(Bz * S * 8));
    cudaStream_t st = g.s_comp;
    if (int rc = scratch_acquire(st)) return rc;
    CK(cudaMemcpyAsync(g.voro.p, voro, Bz * 2 * ld * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(g.nl.p, k, Bz * 4, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(g.off.p, src_offset, S * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(g.dep.p, src_depth, S * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(g.tobs.p, tobs, S * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(g.sigma.p, sigma, Bz * 8, cudaMemcpyHostToDevice, st));
    CK(rtb::launch_prep_voro(g.nl.as<int>(), g.voro.as<double>(), nb, ld, g.vels.as<double>(),
                             g.depths.as<double>(), voro_sorted ? g.vsorted.as<double>() : nullptr, st));
    BatchArgs a{};
    a.vels = g.vels.as<double>(); a.depths = g.depths.as<double>(); a.nlayers = g.nl.as<int>();
    a.B = nb; a.ldv = ld; a.ldz = ld; a.kmode = 1;
    a.src_offset = g.off.as<double>(); a.src_depth = g.dep.as<double>();
    a.tobs = g.tobs.as<double>(); a.nsrc = ns; a.sigma = g.sigma.as<double>();
    a.timeP = tpred ? g.timeP.as<double>() : nullptr; a.p_out = nullptr; a.logL = g.logL.as<double>();
    a.logc = log_norm_const(ns);
    a.padded = 1;
    CK(cudaEventRecord(g.ev_k0[0], st));
    a.sched = next_sched();
    CK(rtb::launch_batch(a, cfg, st));
    CK(cudaEventRecord(g.ev_k1[0], st));
    g.launches += 2;
    g.last = cfg;
    CK(cudaMemcpyAsync(logL, g.logL.p, Bz * 8, cudaMemcpyDeviceToHost, st));
    if (tpred) CK(cudaMemcpyAsync(tpred, g.timeP.p, Bz * S * 8, cudaMemcpyDeviceToHost, st));
    if (voro_sorted) CK(cudaMemcpyAsync(voro_sorted, g.vsorted.p, Bz * 2 * ld * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, g.ev_k0[0], g.ev_k1[0]) == cudaSuccess) g.kernel_ms = g.total_ms = ms;
    return 0;
}

int rtb200_dff_batch_device(const double *d_vels, const double *d_depths, const int *d_nlayers,
                            int B, int ldv, int ldz, const double *d_src_offset,
                            const double *d_src_depth, int NSrc, double *d_timeP,
                            const double *d_tobs, const double *d_sigma, double *d_logL,
                            double *d_p_out, int kmode, void *stream) {
    ApiLock api_lock_;
    if (int rc = ensure_init()) return rc;
    g.err.clear();
    if (B <= 0 || NSrc <= 0) return 0;
    if (d_logL && (!d_tobs || !d_sigma)) return fail("logL needs tobs and sigma");
    cudaStream_t st = stream ? (cudaStream_t)stream : g.s_comp;
    TileCfg cfg;
    const bool al = aligned16(d_vels) && aligned16(d_depths);
    if (int rc = choose_cfg(B, ldv, std::max(ldz, 0), NSrc, al, cfg)) return rc;
    BatchArgs a{};
    a.vels = d_vels; a.depths = d_depths; a.nlayers = d_nlayers;
    a.B = B; a.ldv = ldv; a.ldz = std::max(ldz, 0); a.kmode = kmode;
    a.src_offset = d_src_offset; a.src_depth = d_src_depth;
    a.tobs = d_tobs; a.nsrc = NSrc; a.sigma = d_sigma;
    a.timeP = d_timeP; a.p_out = d_p_out; a.logL = d_logL;
    a.logc = d_logL ? log_norm_const(NSrc) : 0.0;
    CK(cudaEventRecord(g.ev_k0[0], st));
    a.sched = next_sched();
    CK(rtb::launch_batch(a, cfg, st));
    CK(cudaEventRecord(g.ev_k1[0], st));
    g.launches++;
    g.last = cfg;
    if (!stream) {
        CK(cudaStreamSynchronize(st));
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, g.ev_k0[0], g.ev_k1[0]));
        g.kernel_ms = g.total_ms = ms;
    }
    return 0;
}

extern "C++" {   // device_launch is a template
namespace {

// The row-length rule of dff_batch, which every derivative entry checks first.
int check_ldv(int ldv) {
    if (ldv < 1) return fail("ldv must be >= 1");
    if (ldv > 255) return fail("more than 254 interfaces per model are not supported");
    return 0;
}

// A device entry's inputs from the forward; `who_needs` names the derivative in the message
// ("the gradient needs").
int check_forward(const char *who_needs, int nsrc, const void *timeP, const void *p) {
    if (nsrc > 0 && (!timeP || !p)) return fail(std::string(who_needs) + " the forward's timeP and p");
    return 0;
}

// The inputs every derivative kernel reads, from the arguments of the entries (whose order puts
// kmode last).
rtb::DerivArgs deriv_args(const double *vels, const double *depths, const int *nlayers, int B, int ldv,
                          int ldz, const double *off, const double *dep, int nsrc, const double *timeP,
                          const double *p, int kmode) {
    return {vels, depths, nlayers, B, ldv, ldz, kmode, off, dep, nsrc, timeP, p};
}

// The host derivative entries' copy-in and forward on g.s_comp, after each has reserved its own
// buffers: models and sources into the scratch (padded to whole tiles as in run_host), `in`
// (in_bytes: the entry's one further input, or null) to `in_dev`, ev_k0, then the batch kernel
// for timeP and p.  With no source there is nothing to copy of them and no forward.  `d` is set to
// the inputs of the derivative kernel over the scratch.
int host_forward(const double *vels, const double *depths, const int *nlayers, int nb, int lv, int lz,
                 const double *off, const double *dep, int ns, void *in_dev, const double *in,
                 size_t in_bytes, rtb::DerivArgs &d) {
    const size_t Bz = (size_t)nb, S = (size_t)ns;
    TileCfg cfg{};
    if (ns > 0)
        if (int rc = choose_cfg(nb, lv, lz, ns, true, cfg)) return rc;
    const size_t M = ns > 0 ? (size_t)cfg.M : 1, Bpad = (Bz + M - 1) / M * M + M;
    CK(g.vels.reserve(Bpad * lv * 8));
    CK(g.depths.reserve(Bpad * std::max(lz, 1) * 8));
    CK(g.nl.reserve(Bpad * 4));
    CK(g.off.reserve(std::max<size_t>(S, 1) * 8));
    CK(g.dep.reserve(std::max<size_t>(S, 1) * 8));
    CK(g.timeP.reserve(std::max<size_t>(Bz * S, 1) * 8));
    CK(g.pout.reserve(std::max<size_t>(Bz * S, 1) * 8));
    cudaStream_t st = g.s_comp;
    if (int rc = scratch_acquire(st)) return rc;
    CK(cudaMemcpyAsync(g.vels.p, vels, Bz * lv * 8, cudaMemcpyHostToDevice, st));
    if (lz > 0) CK(cudaMemcpyAsync(g.depths.p, depths, Bz * lz * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(g.nl.p, nlayers, Bz * 4, cudaMemcpyHostToDevice, st));
    if (ns > 0) {
        CK(cudaMemcpyAsync(g.off.p, off, S * 8, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(g.dep.p, dep, S * 8, cudaMemcpyHostToDevice, st));
        if (in) CK(cudaMemcpyAsync(in_dev, in, in_bytes, cudaMemcpyHostToDevice, st));
    }
    CK(cudaEventRecord(g.ev_k0[0], st));
    d = deriv_args(g.vels.as<double>(), g.depths.as<double>(), g.nl.as<int>(), nb, lv, lz, g.off.as<double>(),
                   g.dep.as<double>(), ns, g.timeP.as<double>(), g.pout.as<double>(), 0);
    if (ns > 0) {
        BatchArgs a{};
        a.vels = g.vels.as<double>(); a.depths = g.depths.as<double>(); a.nlayers = g.nl.as<int>();
        a.B = nb; a.ldv = lv; a.ldz = lz; a.kmode = 0;
        a.src_offset = g.off.as<double>(); a.src_depth = g.dep.as<double>(); a.nsrc = ns;
        a.timeP = g.timeP.as<double>(); a.p_out = g.pout.as<double>();
        a.padded = 1;
        a.sched = next_sched();
        CK(rtb::launch_batch(a, cfg, st));
        g.launches++;
        g.last = cfg;
    }
    return 0;
}

// The host derivative entries' tail, after each has recorded ev_k1 and queued its own outputs: the
// forward's timeP and p out where asked for, the wait, and the kernel time.
int host_finish(const rtb::DerivArgs &d, double *timeP, double *p_out) {
    cudaStream_t st = g.s_comp;
    const size_t bytes = (size_t)d.B * (size_t)d.nsrc * 8;
    if (d.nsrc > 0) {
        if (timeP) CK(cudaMemcpyAsync(timeP, g.timeP.p, bytes, cudaMemcpyDeviceToHost, st));
        if (p_out) CK(cudaMemcpyAsync(p_out, g.pout.p, bytes, cudaMemcpyDeviceToHost, st));
    }
    CK(cudaStreamSynchronize(st));
    if (int rc = scratch_release(st, true)) return rc;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, g.ev_k0[0], g.ev_k1[0]) == cudaSuccess) g.kernel_ms = g.total_ms = ms;
    return 0;
}

// A device entry's work, enqueue(st), between the kernel-time events on the caller's stream (or
// the library's); without a caller stream it is waited for and timed.
template <class Enqueue>
int device_launch(void *stream, Enqueue enqueue) {
    cudaStream_t st = stream ? (cudaStream_t)stream : g.s_comp;
    CK(cudaEventRecord(g.ev_k0[0], st));
    if (int rc = enqueue(st)) return rc;
    CK(cudaEventRecord(g.ev_k1[0], st));
    if (!stream) {
        CK(cudaStreamSynchronize(st));
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, g.ev_k0[0], g.ev_k1[0]));
        g.kernel_ms = g.total_ms = ms;
    }
    return 0;
}

// The argument checks both gradient entries share (the shape rules of dff_batch).
int check_grad_args(int ldv, int ldz, const void *vels, const void *nlayers, const void *off,
                    const void *dep, int nsrc, const void *w, const void *gvels, const void *gdepths) {
    if (int rc = check_ldv(ldv)) return rc;
    if (!vels || !nlayers || !gvels || (ldz > 0 && !gdepths))
        return fail("the gradient needs vels, nlayers, gvels and (ldz > 0) gdepths");
    if (nsrc > 0 && (!off || !dep || !w)) return fail("the gradient needs src_offset, src_depth and w");
    return 0;
}

// The argument checks both Jacobian entries share; timeP and p are checked by the device entry,
// whose inputs they are.
int check_jac_args(int ldv, int ldz, const void *vels, const void *nlayers, const void *off,
                   const void *dep, const void *jvels, const void *jdepths) {
    if (int rc = check_ldv(ldv)) return rc;
    if (!vels || !nlayers || !jvels) return fail("the Jacobian needs vels, nlayers and jvels");
    if (ldz > 0 && !jdepths) return fail("the Jacobian needs jdepths when ldz > 0");
    if (!off || !dep) return fail("the Jacobian needs src_offset and src_depth");
    return 0;
}

// The argument checks both normal-equations entries share; timeP and p are checked by the device
// entry, whose inputs they are.
int check_normal_args(int ldv, int ldz, int nsrc, const void *vels, const void *nlayers,
                      const void *off, const void *dep, const void *JtJ, const void *tobs,
                      const void *Jtr) {
    if (int rc = check_ldv(ldv)) return rc;
    if (!vels || !nlayers || !JtJ) return fail("the normal equations need vels, nlayers and JtJ");
    // empty source arrays may arrive as NULL: with no source there is nothing to read
    if ((tobs && !Jtr) || (!tobs && Jtr && nsrc > 0)) return fail("tobs and Jtr must be given together");
    if (nsrc > 0 && (!off || !dep)) return fail("the normal equations need src_offset and src_depth");
    return 0;
}

// The argument checks both second-derivative entries share; timeP and p are checked by the
// device entry, whose inputs they are.
int check_hess_args(int ldv, int nsrc, const void *vels, const void *nlayers, const void *off,
                    const void *dep, const void *w, const void *H) {
    if (int rc = check_ldv(ldv)) return rc;
    if (!vels || !nlayers || !H) return fail("the second derivatives need vels, nlayers and H");
    // empty source arrays may arrive as NULL: with no source there is nothing to read
    if (nsrc > 0 && (!off || !dep || !w)) return fail("the second derivatives need src_offset, src_depth and w");
    return 0;
}

}  // namespace
}  // extern "C++"

int rtb200_dff_grad_device(const double *d_vels, const double *d_depths, const int *d_nlayers,
                           int B, int ldv, int ldz, const double *d_src_offset,
                           const double *d_src_depth, int NSrc, const double *d_timeP,
                           const double *d_p, const double *d_w, double *d_gvels,
                           double *d_gdepths, double *d_dtdr, double *d_dtdd, int kmode,
                           void *stream) {
    ApiLock api_lock_;
    if (int rc = ensure_init()) return rc;
    g.err.clear();
    if (B <= 0) return 0;
    ldz = std::max(ldz, 0);
    NSrc = std::max(NSrc, 0);
    if (int rc = check_grad_args(ldv, ldz, d_vels, d_nlayers, d_src_offset, d_src_depth, NSrc, d_w,
                                 d_gvels, d_gdepths))
        return rc;
    if (int rc = check_forward("the gradient needs", NSrc, d_timeP, d_p)) return rc;
    const rtb::GradArgs a{deriv_args(d_vels, d_depths, d_nlayers, B, ldv, ldz, d_src_offset, d_src_depth,
                                     NSrc, d_timeP, d_p, kmode),
                          d_w, d_gvels, d_gdepths, d_dtdr, d_dtdd};
    return device_launch(stream, [&](cudaStream_t st) {
        CK(rtb::launch_grad(a, st));
        g.launches++;
        return 0;
    });
}

int dff_batch_grad(const double *vels, const double *depths, const int *nlayers, const int *B,
                   const int *ldv, const int *ldz, const double *src_offset,
                   const double *src_depth, const int *NSrc, const double *w, double *timeP,
                   double *p_out, double *gvels, double *gdepths, double *dtdr, double *dtdd) {
    ApiLock api_lock_;
    if (int rc = ensure_init()) return rc;
    g.err.clear();
    g.kernel_ms = g.total_ms = 0.0;
    const int nb = *B, lv = *ldv, lz = std::max(*ldz, 0), ns = std::max(*NSrc, 0);
    if (nb <= 0) return 0;
    if (int rc = check_grad_args(lv, lz, vels, nlayers, src_offset, src_depth, ns, w, gvels, gdepths))
        return rc;
    // copy in, forward, gradient, copy out; with no source the gradient kernel alone writes zeros
    const size_t Bz = (size_t)nb, S = (size_t)ns;
    CK(g.w.reserve(std::max<size_t>(Bz * S, 1) * 8));
    CK(g.dvels.reserve(Bz * lv * 8));
    CK(g.ddepths.reserve(std::max<size_t>(Bz * lz, 1) * 8));
    if (dtdr) CK(g.dtdr.reserve(std::max<size_t>(Bz * S, 1) * 8));
    if (dtdd) CK(g.dtdd.reserve(std::max<size_t>(Bz * S, 1) * 8));
    rtb::DerivArgs d;
    if (int rc = host_forward(vels, depths, nlayers, nb, lv, lz, src_offset, src_depth, ns, g.w.p, w,
                              Bz * S * 8, d))
        return rc;
    cudaStream_t st = g.s_comp;
    const rtb::GradArgs ga{d, g.w.as<double>(), g.dvels.as<double>(), g.ddepths.as<double>(),
                           dtdr ? g.dtdr.as<double>() : nullptr, dtdd ? g.dtdd.as<double>() : nullptr};
    CK(rtb::launch_grad(ga, st));
    CK(cudaEventRecord(g.ev_k1[0], st));
    g.launches++;
    CK(cudaMemcpyAsync(gvels, g.dvels.p, Bz * lv * 8, cudaMemcpyDeviceToHost, st));
    if (lz > 0) CK(cudaMemcpyAsync(gdepths, g.ddepths.p, Bz * lz * 8, cudaMemcpyDeviceToHost, st));
    if (ns > 0) {
        if (dtdr) CK(cudaMemcpyAsync(dtdr, g.dtdr.p, Bz * S * 8, cudaMemcpyDeviceToHost, st));
        if (dtdd) CK(cudaMemcpyAsync(dtdd, g.dtdd.p, Bz * S * 8, cudaMemcpyDeviceToHost, st));
    }
    return host_finish(d, timeP, p_out);
}

int rtb200_dff_jac_device(const double *d_vels, const double *d_depths, const int *d_nlayers,
                          int B, int ldv, int ldz, const double *d_src_offset,
                          const double *d_src_depth, int NSrc, const double *d_timeP,
                          const double *d_p, double *d_jvels, double *d_jdepths, double *d_dtdr,
                          double *d_dtdd, int kmode, void *stream) {
    ApiLock api_lock_;
    if (int rc = ensure_init()) return rc;
    g.err.clear();
    if (B <= 0 || NSrc <= 0) return 0;
    ldz = std::max(ldz, 0);
    if (int rc = check_jac_args(ldv, ldz, d_vels, d_nlayers, d_src_offset, d_src_depth, d_jvels,
                                d_jdepths))
        return rc;
    if (int rc = check_forward("the Jacobian needs", NSrc, d_timeP, d_p)) return rc;
    const rtb::JacArgs a{deriv_args(d_vels, d_depths, d_nlayers, B, ldv, ldz, d_src_offset, d_src_depth,
                                    NSrc, d_timeP, d_p, kmode),
                         d_jvels, d_jdepths, d_dtdr, d_dtdd};
    return device_launch(stream, [&](cudaStream_t st) {
        CK(rtb::launch_jac(a, st));
        g.launches++;
        return 0;
    });
}

int dff_batch_jac(const double *vels, const double *depths, const int *nlayers, const int *B,
                  const int *ldv, const int *ldz, const double *src_offset,
                  const double *src_depth, const int *NSrc, double *timeP, double *p_out,
                  double *jvels, double *jdepths, double *dtdr, double *dtdd) {
    ApiLock api_lock_;
    if (int rc = ensure_init()) return rc;
    g.err.clear();
    g.kernel_ms = g.total_ms = 0.0;
    const int nb = *B, lv = *ldv, lz = std::max(*ldz, 0), ns = *NSrc;
    if (nb <= 0 || ns <= 0) return 0;
    if (int rc = check_jac_args(lv, lz, vels, nlayers, src_offset, src_depth, jvels, jdepths))
        return rc;
    // copy in, forward, Jacobian, copy out
    const size_t Bz = (size_t)nb, S = (size_t)ns;
    CK(g.dvels.reserve(Bz * S * lv * 8));
    if (lz > 0) CK(g.ddepths.reserve(Bz * S * lz * 8));
    if (dtdr) CK(g.dtdr.reserve(Bz * S * 8));
    if (dtdd) CK(g.dtdd.reserve(Bz * S * 8));
    rtb::DerivArgs d;
    if (int rc = host_forward(vels, depths, nlayers, nb, lv, lz, src_offset, src_depth, ns, nullptr, nullptr,
                              0, d))
        return rc;
    cudaStream_t st = g.s_comp;
    const rtb::JacArgs ja{d, g.dvels.as<double>(), lz > 0 ? g.ddepths.as<double>() : nullptr,
                          dtdr ? g.dtdr.as<double>() : nullptr, dtdd ? g.dtdd.as<double>() : nullptr};
    CK(rtb::launch_jac(ja, st));
    CK(cudaEventRecord(g.ev_k1[0], st));
    g.launches++;
    CK(cudaMemcpyAsync(jvels, g.dvels.p, Bz * S * lv * 8, cudaMemcpyDeviceToHost, st));
    if (lz > 0) CK(cudaMemcpyAsync(jdepths, g.ddepths.p, Bz * S * lz * 8, cudaMemcpyDeviceToHost, st));
    if (dtdr) CK(cudaMemcpyAsync(dtdr, g.dtdr.p, Bz * S * 8, cudaMemcpyDeviceToHost, st));
    if (dtdd) CK(cudaMemcpyAsync(dtdd, g.dtdd.p, Bz * S * 8, cudaMemcpyDeviceToHost, st));
    return host_finish(d, timeP, p_out);
}

int rtb200_dff_normal_device(const double *d_vels, const double *d_depths, const int *d_nlayers,
                             int B, int ldv, int ldz, const double *d_src_offset,
                             const double *d_src_depth, int NSrc, const double *d_timeP,
                             const double *d_p, const double *d_tobs, double *d_JtJ,
                             double *d_Jtr, int kmode, void *stream) {
    ApiLock api_lock_;
    if (int rc = ensure_init()) return rc;
    g.err.clear();
    if (B <= 0) return 0;
    ldz = std::max(ldz, 0);
    if (int rc = check_normal_args(ldv, ldz, NSrc, d_vels, d_nlayers, d_src_offset, d_src_depth,
                                   d_JtJ, d_tobs, d_Jtr))
        return rc;
    if (int rc = check_forward("the normal equations need", NSrc, d_timeP, d_p)) return rc;
    const size_t P = (size_t)(ldv + ldz);
    const rtb::NormalArgs a{deriv_args(d_vels, d_depths, d_nlayers, B, ldv, ldz, d_src_offset, d_src_depth,
                                       NSrc, d_timeP, d_p, kmode),
                            d_tobs, d_JtJ, d_Jtr};
    return device_launch(stream, [&](cudaStream_t st) {
        if (NSrc <= 0) {        // sums over no source
            CK(cudaMemsetAsync(d_JtJ, 0, (size_t)B * P * P * 8, st));
            if (d_Jtr) CK(cudaMemsetAsync(d_Jtr, 0, (size_t)B * P * 8, st));
        } else {
            CK(rtb::launch_normal(a, st));
            g.launches++;
        }
        return 0;
    });
}

int dff_batch_normal(const double *vels, const double *depths, const int *nlayers, const int *B,
                     const int *ldv, const int *ldz, const double *src_offset,
                     const double *src_depth, const int *NSrc, const double *tobs, double *timeP,
                     double *p_out, double *JtJ, double *Jtr) {
    ApiLock api_lock_;
    if (int rc = ensure_init()) return rc;
    g.err.clear();
    g.kernel_ms = g.total_ms = 0.0;
    const int nb = *B, lv = *ldv, lz = std::max(*ldz, 0), ns = *NSrc;
    if (nb <= 0) return 0;
    if (int rc = check_normal_args(lv, lz, ns, vels, nlayers, src_offset, src_depth, JtJ, tobs, Jtr))
        return rc;
    const size_t Bz = (size_t)nb, P = (size_t)(lv + lz);
    if (ns <= 0) {              // sums over no source
        std::memset(JtJ, 0, Bz * P * P * 8);
        if (Jtr) std::memset(Jtr, 0, Bz * P * 8);
        return 0;
    }
    // copy in, forward, normal equations, copy out
    const size_t S = (size_t)ns;
    CK(g.JtJ.reserve(Bz * P * P * 8));
    if (tobs) {
        CK(g.tobs.reserve(S * 8));
        CK(g.Jtr.reserve(Bz * P * 8));
    }
    rtb::DerivArgs d;
    if (int rc = host_forward(vels, depths, nlayers, nb, lv, lz, src_offset, src_depth, ns, g.tobs.p, tobs,
                              S * 8, d))
        return rc;
    cudaStream_t st = g.s_comp;
    const rtb::NormalArgs na{d, tobs ? g.tobs.as<double>() : nullptr, g.JtJ.as<double>(),
                             tobs ? g.Jtr.as<double>() : nullptr};
    CK(rtb::launch_normal(na, st));
    CK(cudaEventRecord(g.ev_k1[0], st));
    g.launches++;
    CK(cudaMemcpyAsync(JtJ, g.JtJ.p, Bz * P * P * 8, cudaMemcpyDeviceToHost, st));
    if (tobs) CK(cudaMemcpyAsync(Jtr, g.Jtr.p, Bz * P * 8, cudaMemcpyDeviceToHost, st));
    return host_finish(d, timeP, p_out);
}

int rtb200_dff_hess_device(const double *d_vels, const double *d_depths, const int *d_nlayers,
                           int B, int ldv, int ldz, const double *d_src_offset,
                           const double *d_src_depth, int NSrc, const double *d_timeP,
                           const double *d_p, const double *d_w, double *d_H, int kmode,
                           void *stream) {
    ApiLock api_lock_;
    if (int rc = ensure_init()) return rc;
    g.err.clear();
    if (B <= 0) return 0;
    ldz = std::max(ldz, 0);
    if (int rc = check_hess_args(ldv, NSrc, d_vels, d_nlayers, d_src_offset, d_src_depth, d_w, d_H))
        return rc;
    if (int rc = check_forward("the second derivatives need", NSrc, d_timeP, d_p)) return rc;
    const size_t P = (size_t)(ldv + ldz);
    const rtb::HessArgs a{deriv_args(d_vels, d_depths, d_nlayers, B, ldv, ldz, d_src_offset, d_src_depth,
                                     NSrc, d_timeP, d_p, kmode),
                          d_w, d_H};
    return device_launch(stream, [&](cudaStream_t st) {
        if (NSrc <= 0) {        // sums over no source
            CK(cudaMemsetAsync(d_H, 0, (size_t)B * P * P * 8, st));
        } else {
            CK(rtb::launch_hess(a, st));
            g.launches++;
        }
        return 0;
    });
}

int dff_batch_hess(const double *vels, const double *depths, const int *nlayers, const int *B,
                   const int *ldv, const int *ldz, const double *src_offset,
                   const double *src_depth, const int *NSrc, const double *w, double *timeP,
                   double *p_out, double *H) {
    ApiLock api_lock_;
    if (int rc = ensure_init()) return rc;
    g.err.clear();
    g.kernel_ms = g.total_ms = 0.0;
    const int nb = *B, lv = *ldv, lz = std::max(*ldz, 0), ns = *NSrc;
    if (nb <= 0) return 0;
    if (int rc = check_hess_args(lv, ns, vels, nlayers, src_offset, src_depth, w, H)) return rc;
    const size_t Bz = (size_t)nb, P = (size_t)(lv + lz);
    if (ns <= 0) {              // sums over no source
        std::memset(H, 0, Bz * P * P * 8);
        return 0;
    }
    // copy in, forward, second derivatives, copy out (H in the normal equations' scratch)
    const size_t S = (size_t)ns;
    CK(g.JtJ.reserve(Bz * P * P * 8));
    CK(g.w.reserve(Bz * S * 8));
    rtb::DerivArgs d;
    if (int rc = host_forward(vels, depths, nlayers, nb, lv, lz, src_offset, src_depth, ns, g.w.p, w,
                              Bz * S * 8, d))
        return rc;
    cudaStream_t st = g.s_comp;
    const rtb::HessArgs ha{d, g.w.as<double>(), g.JtJ.as<double>()};
    CK(rtb::launch_hess(ha, st));
    CK(cudaEventRecord(g.ev_k1[0], st));
    g.launches++;
    CK(cudaMemcpyAsync(H, g.JtJ.p, Bz * P * P * 8, cudaMemcpyDeviceToHost, st));
    return host_finish(d, timeP, p_out);
}

extern "C++" {   // the helpers below include templates
namespace {

rtb::MhPrior make_prior(const double *prior, int enos = 0) {
    rtb::MhPrior pr;
    pr.enos = enos ? 1 : 0;
    pr.scale[0] = prior[0]; pr.scale[1] = prior[1];
    pr.minlim[0] = prior[2]; pr.minlim[1] = prior[3];
    pr.maxlim[0] = prior[4]; pr.maxlim[1] = prior[5];
    pr.hmin = prior[6];
    return pr;
}

rtb::BdPrior make_bd_prior(const double *pk, int kmin, int kmax) {
    rtb::BdPrior bd{};
    bd.kmin = kmin; bd.kmax = kmax; bd.use_pk = pk ? 1 : 0;
    for (int i = kmin; pk && i <= kmax; ++i) bd.logpk[i - 1] = std::log(pk[i - 1]);   // LOG(pk(i)), libm
    return bd;
}

// What every chain move reads: the chains' state (k [B], voro [B][2][ldk], logL, sigma, beta [B]),
// the data and the likelihood's tile geometry.  The entries' const qualifiers say which state they
// leave alone; one struct serves every move.
struct MoveCtx {
    int          *k;
    double       *voro, *logL, *sigma;
    const double *beta;
    int           B, ldk;
    const double *src_offset, *src_depth, *tobs;
    int           NSrc;
    TileCfg       cfg;
};

MoveCtx move_ctx(const int *k, const double *voro, double *logL, const double *sigma, const double *beta,
                 int B, int ldk, const double *src_offset, const double *src_depth, const double *tobs,
                 int NSrc) {
    return {const_cast<int *>(k), const_cast<double *>(voro), logL, const_cast<double *>(sigma), beta, B,
            ldk, src_offset, src_depth, tobs, NSrc, TileCfg{}};
}

// The argument checks every chain-move entry makes; `name` starts the refusal.
int check_move_args(const char *name, int NSrc, int ldk) {
    if (NSrc <= 0) return fail(std::string(name) + " needs at least one source");
    if (ldk < 1 || ldk > 64) return fail(std::string(name) + " supports 1..64 nodes per state");
    return 0;
}

// The start every chain-move entry shares after its checks: the stream (the caller's or the
// library's own), the likelihood's tile geometry and the scratch of a move -- the proposal as
// (vp, ziface) rows for the batch kernel, its node count, its sorted nodes, its logL and the
// outside / no-move code; with `ar` also the AR move's proposal (a graph's key holds its address,
// so it is reserved before any capture) -- with the stream ordered behind the scratch's last user.
int begin_move(MoveCtx &m, void *stream, bool ar, cudaStream_t &st) {
    st = stream ? (cudaStream_t)stream : g.s_comp;
    if (int rc = choose_cfg(m.B, m.ldk, m.ldk, m.NSrc, true, m.cfg)) return rc;
    const size_t Bz = (size_t)m.B, Bpad = (Bz + m.cfg.M - 1) / m.cfg.M * m.cfg.M + m.cfg.M;
    CK(g.vels.reserve(Bpad * m.ldk * 8));
    CK(g.depths.reserve(Bpad * m.ldk * 8));
    CK(g.nl.reserve(Bpad * 4));
    CK(g.vsorted.reserve(Bz * 2 * m.ldk * 8));
    CK(g.mh_ll.reserve(Bz * 8));
    CK(g.mh_out.reserve(Bz * 4));
    CK(g.mh_kp.reserve(Bz * 4));
    CK(g.mh_lpr.reserve(Bz * 8));
    if (ar) {
        CK(g.idxar.reserve(Bz * 4));
        CK(g.arparb.reserve(Bz * 8));
    }
    return scratch_acquire(st);
}

// The end every chain-move entry shares: `launches` kernels counted; without a caller stream the
// work is waited for (`timed`: the likelihood's time goes to kernel_ms), then the scratch released.
int end_move(const MoveCtx &m, long long launches, bool timed, void *stream, cudaStream_t st) {
    g.launches += launches;
    g.last = m.cfg;
    if (!stream) {
        CK(cudaStreamSynchronize(st));
        if (timed) {
            float ms = 0.f;
            CK(cudaEventElapsedTime(&ms, g.ev_k0[0], g.ev_k1[0]));
            g.kernel_ms = g.total_ms = ms;
        }
    }
    return scratch_release(st, stream == nullptr);
}

// The batch kernel's arguments for evaluating the scratch rows in k-mode; logL goes to g.mh_ll.
BatchArgs move_eval_args(const MoveCtx &m, const double *sigma, int *sched) {
    BatchArgs a{};
    a.vels = g.vels.as<double>(); a.depths = g.depths.as<double>(); a.nlayers = g.nl.as<int>();
    a.B = m.B; a.ldv = m.ldk; a.ldz = m.ldk; a.kmode = 1;
    a.src_offset = m.src_offset; a.src_depth = m.src_depth;
    a.tobs = m.tobs; a.nsrc = m.NSrc; a.sigma = sigma;
    a.logL = g.mh_ll.as<double>();
    a.logc = log_norm_const(m.NSrc);
    a.padded = 1;
    a.sched = sched;
    a.idxar = g.chain_idxar;         // IAR = 1 (rtb200_set_chain_ar); null otherwise
    a.arpar = g.chain_arpar;
    a.armx  = g.chain_armx;
    return a;
}

// The likelihood of a move's proposals: the batch kernel, or LOGLHOOD2's constant when the
// sampler draws from the prior (ISMPPRIOR = 1, prjmh_temper_rf.f90:693-694, :739-740, ...).
// `timed`: between ev_k0 and ev_k1 (events are not recorded inside a graph capture).
cudaError_t launch_move_eval(const MoveCtx &m, const BatchArgs &a, bool timed, cudaStream_t st) {
    cudaError_t e = timed ? cudaEventRecord(g.ev_k0[0], st) : cudaSuccess;
    if (e == cudaSuccess)
        e = g.opt_ismpprior ? rtb::launch_fill_f64(a.logL, a.B, 1.0, st) : rtb::launch_batch(a, m.cfg, st);
    if (e == cudaSuccess && timed) e = cudaEventRecord(g.ev_k1[0], st);
    return e;
}

// The enqueue_* functions issue one move of every chain on `st`: propose -> launch_move_eval ->
// accept, the likelihood on tile-scheduler slot `sched`.
// The fixed-dimension MH move.  The proposal and its likelihood do not read beta; only the accept
// test does, and it waits for `beta_ready` when one is given.
cudaError_t enqueue_mh(const MoveCtx &m, const rtb::MhPrior &pr, const int *ivo, const int *iwhich,
                       const double *dev, const double *u_acc, int *accept, cudaEvent_t beta_ready,
                       int *sched, bool timed, cudaStream_t st) {
    cudaError_t e = rtb::launch_propose_voro(m.k, m.voro, m.B, m.ldk, ivo, iwhich, dev, pr, g.vels.as<double>(),
                                             g.depths.as<double>(), g.nl.as<int>(), g.vsorted.as<double>(),
                                             g.mh_lpr.as<double>(), g.mh_out.as<int>(), st);
    if (e == cudaSuccess) e = launch_move_eval(m, move_eval_args(m, m.sigma, sched), timed, st);
    if (e == cudaSuccess && beta_ready) e = cudaStreamWaitEvent(st, beta_ready, 0);
    if (e == cudaSuccess)
        e = rtb::launch_mh_accept(m.k, m.voro, g.vsorted.as<double>(), m.logL, g.mh_ll.as<double>(),
                                  g.mh_lpr.as<double>(), g.mh_out.as<int>(), u_acc, m.beta, m.B, m.ldk, accept, st);
    return e;
}

// The birth/death move.
cudaError_t enqueue_bd(const MoveCtx &m, const rtb::MhPrior &pr, const rtb::BdPrior &bd, const double *u_k,
                       const int *idel, const double *u_z, const double *u_v, const double *u_acc, int *accept,
                       int *sched, bool timed, cudaStream_t st) {
    cudaError_t e = rtb::launch_propose_bd(m.k, m.voro, m.B, m.ldk, u_k, idel, u_z, u_v, pr, bd,
                                           g.vels.as<double>(), g.depths.as<double>(), g.nl.as<int>(),
                                           g.mh_kp.as<int>(), g.vsorted.as<double>(), g.mh_lpr.as<double>(),
                                           g.mh_out.as<int>(), st);
    if (e == cudaSuccess) e = launch_move_eval(m, move_eval_args(m, m.sigma, sched), timed, st);
    if (e == cudaSuccess)
        e = rtb::launch_bd_accept(m.k, m.voro, g.vsorted.as<double>(), g.mh_kp.as<int>(), g.mh_lpr.as<double>(),
                                  m.logL, g.mh_ll.as<double>(), g.mh_out.as<int>(), u_acc, m.beta, m.B, m.ldk,
                                  accept, st);
    return e;
}

// The data-error move; its likelihood uses the proposed sigma.
cudaError_t enqueue_sd(const MoveCtx &m, const double *sd_prior, const double *u_gate, const double *gauss,
                       const double *u_acc, int *accept, int *sched, bool timed, cudaStream_t st) {
    cudaError_t e = rtb::launch_propose_sd(m.k, m.voro, m.B, m.ldk, m.sigma, u_gate, gauss, sd_prior[0],
                                           sd_prior[1], sd_prior[2], g.vels.as<double>(), g.depths.as<double>(),
                                           g.nl.as<int>(), g.mh_lpr.as<double>(), g.mh_out.as<int>(), st);
    if (e == cudaSuccess) e = launch_move_eval(m, move_eval_args(m, g.mh_lpr.as<double>(), sched), timed, st);
    if (e == cudaSuccess)
        e = rtb::launch_sd_accept(m.sigma, g.mh_lpr.as<double>(), m.logL, g.mh_ll.as<double>(),
                                  g.mh_out.as<int>(), u_acc, m.beta, m.B, accept, st);
    return e;
}

// The AR(1) move; its likelihood uses the proposed (idxar, arpar) and armx = ar_prior[3].
cudaError_t enqueue_ar(const MoveCtx &m, int *idxar, double *arpar, const double *ar_prior,
                       const double *u_choice, const double *u_prop, const double *gauss, const double *u_acc,
                       int *accept, int *sched, bool timed, cudaStream_t st) {
    cudaError_t e = rtb::launch_propose_ar(m.k, m.voro, m.B, m.ldk, idxar, arpar, u_choice, u_prop, gauss,
                                           ar_prior[0], ar_prior[1], ar_prior[2], std::log(0.5), std::log(2.0),
                                           g.vels.as<double>(), g.depths.as<double>(), g.nl.as<int>(),
                                           g.idxar.as<int>(), g.arparb.as<double>(), g.mh_lpr.as<double>(),
                                           g.mh_out.as<int>(), st);
    BatchArgs a = move_eval_args(m, m.sigma, sched);
    a.idxar = g.idxar.as<int>();
    a.arpar = g.arparb.as<double>();
    a.armx  = ar_prior[3];
    if (e == cudaSuccess) e = launch_move_eval(m, a, timed, st);
    if (e == cudaSuccess)
        e = rtb::launch_ar_accept(idxar, arpar, g.idxar.as<int>(), g.arparb.as<double>(), g.mh_lpr.as<double>(),
                                  m.logL, g.mh_ll.as<double>(), g.mh_out.as<int>(), u_acc, m.beta, m.B, accept, st);
    return e;
}

// The tile-scheduler slot kernel node `i` of a captured graph owns (past the round-robin slots).
int *graph_slot(int i) { return g.opt_static_tiles ? nullptr : g.sched.as<int>() + 2 * (kSchedSlots + i); }

// Appends integers and pointers to a graph's key as they are, doubles by their bits.
template <class... T> void key_add(std::vector<size_t> &key, T... xs) {
    auto add = [&key](auto x) {
        if constexpr (std::is_floating_point_v<decltype(x)>) {
            size_t bits;
            memcpy(&bits, &x, sizeof bits);
            key.push_back(bits);
        } else {
            key.push_back((size_t)x);
        }
    };
    (add(xs), ...);
}

// The part of a move graph's key every such graph shares: the chain state and data, every field
// of the tile geometry (by name: TileCfg has padding and an unused member), the likelihood
// constant, the scratch, the options and the registered AR state.
std::vector<size_t> move_key(const MoveCtx &m) {
    std::vector<size_t> key;
    const TileCfg &c = m.cfg;
    key_add(key, m.k, m.voro, m.logL, m.sigma, m.beta, m.B, m.ldk, m.src_offset, m.src_depth, m.tobs, m.NSrc);
    key_add(key, c.M, c.SC, c.LP, c.TS, c.threads, c.grid, c.variant, c.use_tma, c.logl_shuffle, c.smem,
            log_norm_const(m.NSrc));
    key_add(key, g.vels.p, g.depths.p, g.nl.p, g.vsorted.p, g.mh_ll.p, g.mh_out.p, g.mh_kp.p, g.mh_lpr.p,
            g.idxar.p, g.arparb.p, g.opt_static_tiles, g.opt_ismpprior, g.chain_idxar, g.chain_arpar,
            g.chain_armx);
    return key;
}

// Replays the graph cached in `c` n times on `st`.  When `key` differs from the cached graph's,
// the graph is first captured anew from `enqueue(stream)` on the capture stream; `what` names the
// capture in a failure.
template <class Enqueue>
int run_graph(GraphCache &c, std::vector<size_t> &key, const TileCfg &cfg, const char *what, Enqueue enqueue,
              int n, cudaStream_t st) {
    if (!c.exec || key != c.key) {
        c.reset();
        if (!g.s_cap) CK(cudaStreamCreateWithFlags(&g.s_cap, cudaStreamNonBlocking));
        if (rtb::max_ctas_per_sm(cfg) < 1) return fail("batch kernel cannot be resident");   // sets the smem attribute
        CK(cudaStreamBeginCapture(g.s_cap, cudaStreamCaptureModeThreadLocal));
        cudaError_t e = enqueue(g.s_cap);
        cudaGraph_t graph = nullptr;
        const cudaError_t e2 = cudaStreamEndCapture(g.s_cap, &graph);
        if (e != cudaSuccess) { if (graph) cudaGraphDestroy(graph); return fail(what, e); }
        if (e2 != cudaSuccess) return fail("cudaStreamEndCapture", e2);
        e = cudaGraphInstantiate(&c.exec, graph, 0);
        cudaGraphDestroy(graph);
        if (e != cudaSuccess) { c.exec = nullptr; return fail("cudaGraphInstantiate", e); }
        c.key.swap(key);
    }
    for (int i = 0; i < n; ++i) CK(cudaGraphLaunch(c.exec, st));
    return 0;
}

}  // namespace
}  // extern "C++"

int rtb200_mh_step_device(const int *d_k, double *d_voro, double *d_logL, int B, int ldk,
                          const int *d_ivo, const int *d_iwhich, const double *d_cauchy,
                          const double *d_uacc, const double *d_beta, const double *d_sigma,
                          const double *prior, const double *d_src_offset,
                          const double *d_src_depth, const double *d_tobs, int NSrc,
                          int *d_accept, void *stream) {
    ApiLock api_lock_;
    return rtb200_mh_step_device_ev(d_k, d_voro, d_logL, B, ldk, d_ivo, d_iwhich, d_cauchy, d_uacc,
                                    d_beta, d_sigma, prior, d_src_offset, d_src_depth, d_tobs, NSrc,
                                    d_accept, stream, nullptr, 0);
}

int rtb200_mh_step_device_ev(const int *d_k, double *d_voro, double *d_logL, int B, int ldk,
                             const int *d_ivo, const int *d_iwhich, const double *d_cauchy,
                             const double *d_uacc, const double *d_beta, const double *d_sigma,
                             const double *prior, const double *d_src_offset,
                             const double *d_src_depth, const double *d_tobs, int NSrc,
                             int *d_accept, void *stream, void *beta_ready_event, int enos) {
    ApiLock api_lock_;
    if (int rc = ensure_init()) return rc;
    g.err.clear();
    if (B <= 0) return 0;
    if (int rc = check_move_args("rtb200_mh_step_device", NSrc, ldk)) return rc;
    if (!prior) return fail("rtb200_mh_step_device needs the prior array");
    MoveCtx m = move_ctx(d_k, d_voro, d_logL, d_sigma, d_beta, B, ldk, d_src_offset, d_src_depth, d_tobs, NSrc);
    cudaStream_t st;
    if (int rc = begin_move(m, stream, false, st)) return rc;
    CK(enqueue_mh(m, make_prior(prior, enos), d_ivo, d_iwhich, d_cauchy, d_uacc, d_accept,
                  (cudaEvent_t)beta_ready_event, next_sched(), true, st));
    return end_move(m, 3, true, stream, st);
}

// n_moves fixed-dimension moves back to back.  A move is three dependent launches (propose,
// evaluate, accept) of a few hundred microseconds at most, so a run of moves is launch-bound; the
// run is captured once into a CUDA graph and replayed while the caller keeps passing the same
// buffers and options (the key is everything the capture bakes in).  Each kernel node owns its
// tile-scheduler slot.
int rtb200_mh_moves_device(const int *d_k, double *d_voro, double *d_logL, int B, int ldk,
                           int n_moves, const int *d_ivo, const int *d_iwhich,
                           const double *d_cauchy, const double *d_uacc, const double *d_beta,
                           const double *d_sigma, const double *prior, const double *d_src_offset,
                           const double *d_src_depth, const double *d_tobs, int NSrc,
                           int *d_accept, void *stream) {
    ApiLock api_lock_;
    return rtb200_mh_moves_device_ex(d_k, d_voro, d_logL, B, ldk, n_moves, d_ivo, d_iwhich, d_cauchy, d_uacc,
                                     d_beta, d_sigma, prior, d_src_offset, d_src_depth, d_tobs, NSrc,
                                     d_accept, stream, 0);
}

int rtb200_mh_moves_device_ex(const int *d_k, double *d_voro, double *d_logL, int B, int ldk,
                              int n_moves, const int *d_ivo, const int *d_iwhich,
                              const double *d_cauchy, const double *d_uacc, const double *d_beta,
                              const double *d_sigma, const double *prior, const double *d_src_offset,
                              const double *d_src_depth, const double *d_tobs, int NSrc,
                              int *d_accept, void *stream, int enos) {
    ApiLock api_lock_;
    if (int rc = ensure_init()) return rc;
    g.err.clear();
    if (B <= 0 || n_moves <= 0) return 0;
    if (int rc = check_move_args("rtb200_mh_moves_device", NSrc, ldk)) return rc;
    if (!prior) return fail("rtb200_mh_moves_device needs the prior array");
    if (n_moves > kGraphSlots) return fail("rtb200_mh_moves_device: at most 512 moves per call");
    MoveCtx m = move_ctx(d_k, d_voro, d_logL, d_sigma, d_beta, B, ldk, d_src_offset, d_src_depth, d_tobs, NSrc);
    cudaStream_t st;
    if (int rc = begin_move(m, stream, false, st)) return rc;
    std::vector<size_t> key = move_key(m);
    key_add(key, n_moves, d_ivo, d_iwhich, d_cauchy, d_uacc, d_accept, enos ? 1 : 0);
    for (int i = 0; i < 7; ++i) key_add(key, prior[i]);
    auto capture = [&](cudaStream_t sc) {
        const rtb::MhPrior pr = make_prior(prior, enos);
        cudaError_t e = cudaSuccess;
        for (int i = 0; i < n_moves && e == cudaSuccess; ++i) {
            const size_t o = (size_t)i * (size_t)B;
            e = enqueue_mh(m, pr, d_ivo + o, d_iwhich + o, d_cauchy + o, d_uacc + o, d_accept + o, nullptr,
                           graph_slot(i), false, sc);
        }
        return e;
    };
    if (int rc = run_graph(g.mv, key, m.cfg, "capturing the MH moves", capture, 1, st)) return rc;
    return end_move(m, 3LL * n_moves, false, stream, st);
}

int rtb200_bd_step_device(int *d_k, double *d_voro, double *d_logL, int B, int ldk,
                          const double *d_uk, const int *d_idel, const double *d_uz,
                          const double *d_uv, const double *d_uacc, const double *d_beta,
                          const double *d_sigma, const double *prior, const double *pk, int kmin,
                          int kmax, const double *d_src_offset, const double *d_src_depth,
                          const double *d_tobs, int NSrc, int *d_accept, void *stream) {
    ApiLock api_lock_;
    return rtb200_bd_step_device_ex(d_k, d_voro, d_logL, B, ldk, d_uk, d_idel, d_uz, d_uv, d_uacc, d_beta,
                                    d_sigma, prior, pk, kmin, kmax, d_src_offset, d_src_depth, d_tobs, NSrc,
                                    d_accept, stream, 0);
}

int rtb200_bd_step_device_ex(int *d_k, double *d_voro, double *d_logL, int B, int ldk,
                             const double *d_uk, const int *d_idel, const double *d_uz,
                             const double *d_uv, const double *d_uacc, const double *d_beta,
                             const double *d_sigma, const double *prior, const double *pk, int kmin,
                             int kmax, const double *d_src_offset, const double *d_src_depth,
                             const double *d_tobs, int NSrc, int *d_accept, void *stream, int enos) {
    ApiLock api_lock_;
    if (int rc = ensure_init()) return rc;
    g.err.clear();
    if (B <= 0) return 0;
    if (int rc = check_move_args("rtb200_bd_step_device", NSrc, ldk)) return rc;
    if (!prior) return fail("rtb200_bd_step_device needs the prior array");
    if (kmin < 1 || kmax < kmin || kmax > ldk) return fail("rtb200_bd_step_device needs 1 <= kmin <= kmax <= ldk");
    MoveCtx m = move_ctx(d_k, d_voro, d_logL, d_sigma, d_beta, B, ldk, d_src_offset, d_src_depth, d_tobs, NSrc);
    cudaStream_t st;
    if (int rc = begin_move(m, stream, false, st)) return rc;
    CK(enqueue_bd(m, make_prior(prior, enos), make_bd_prior(pk, kmin, kmax), d_uk, d_idel, d_uz, d_uv, d_uacc,
                  d_accept, next_sched(), true, st));
    return end_move(m, 3, true, stream, st);
}

int rtb200_sd_step_device(const int *d_k, const double *d_voro, double *d_logL, double *d_sigma,
                          int B, int ldk, const double *d_ugate, const double *d_gauss,
                          const double *d_uacc, const double *d_beta, const double *sd_prior,
                          const double *d_src_offset, const double *d_src_depth,
                          const double *d_tobs, int NSrc, int *d_accept, void *stream) {
    ApiLock api_lock_;
    if (int rc = ensure_init()) return rc;
    g.err.clear();
    if (B <= 0) return 0;
    if (int rc = check_move_args("rtb200_sd_step_device", NSrc, ldk)) return rc;
    if (!sd_prior) return fail("rtb200_sd_step_device needs the sd_prior array");
    MoveCtx m = move_ctx(d_k, d_voro, d_logL, d_sigma, d_beta, B, ldk, d_src_offset, d_src_depth, d_tobs, NSrc);
    cudaStream_t st;
    if (int rc = begin_move(m, stream, false, st)) return rc;
    CK(enqueue_sd(m, sd_prior, d_ugate, d_gauss, d_uacc, d_accept, next_sched(), true, st));
    return end_move(m, 3, true, stream, st);
}

int rtb200_set_chain_ar(const int *d_idxar, const double *d_arpar, double armx) {
    ApiLock api_lock_;
    g.err.clear();
    if ((d_idxar == nullptr) != (d_arpar == nullptr)) return fail("rtb200_set_chain_ar needs both arrays or neither");
    g.chain_idxar = d_idxar;
    g.chain_arpar = d_arpar;
    g.chain_armx  = armx;
    return 0;
}

int rtb200_ar_step_device(const int *d_k, const double *d_voro, double *d_logL,
                          const double *d_sigma, int *d_idxar, double *d_arpar, int B, int ldk,
                          const double *d_uchoice, const double *d_uprop, const double *d_gauss,
                          const double *d_uacc, const double *d_beta, const double *ar_prior,
                          const double *d_src_offset, const double *d_src_depth,
                          const double *d_tobs, int NSrc, int *d_accept, void *stream) {
    ApiLock api_lock_;
    if (int rc = ensure_init()) return rc;
    g.err.clear();
    if (B <= 0) return 0;
    if (int rc = check_move_args("rtb200_ar_step_device", NSrc, ldk)) return rc;
    if (!ar_prior) return fail("rtb200_ar_step_device needs the ar_prior array");
    MoveCtx m = move_ctx(d_k, d_voro, d_logL, d_sigma, d_beta, B, ldk, d_src_offset, d_src_depth, d_tobs, NSrc);
    cudaStream_t st;
    if (int rc = begin_move(m, stream, true, st)) return rc;
    CK(enqueue_ar(m, d_idxar, d_arpar, ar_prior, d_uchoice, d_uprop, d_gauss, d_uacc, d_accept, next_sched(),
                  true, st));
    return end_move(m, 3, true, stream, st);
}

size_t rtb200_mcmc_workspace_bytes(int B, int n_moves) {
    ApiLock api_lock_;
    return (B > 0 && n_moves >= 0) ? rtb::mcmc_ws_bytes((size_t)B, (size_t)n_moves) : 0;
}

// One whole iteration of the sampler's worker loop (prjmh_temper_rf.f90:420-458) for B chains --
// birth/death move, n_moves fixed-dimension moves of every chain's own sweep, data-error move --
// with every random deviate drawn on the device, captured once as a CUDA graph and replayed
// n_iterations times: no host synchronisation, no per-move host work.
int rtb200_mcmc_iterations_device(int *d_k, double *d_voro, double *d_logL, double *d_sigma,
                                  const double *d_beta, int *d_pos, int B, int ldk, int n_moves,
                                  const double *prior, const double *sd_prior, const double *pk,
                                  int kmin, int kmax, int enos, const double *d_src_offset,
                                  const double *d_src_depth, const double *d_tobs, int NSrc,
                                  unsigned long long seed, unsigned long long *d_counter,
                                  void *d_workspace, long long *d_tally, int n_iterations,
                                  int *d_idxar, double *d_arpar, const double *ar_prior,
                                  void *stream) {
    ApiLock api_lock_;
    if (int rc = ensure_init()) return rc;
    g.err.clear();
    if (B <= 0 || n_iterations <= 0) return 0;
    if ((d_idxar == nullptr) != (d_arpar == nullptr) || (d_idxar && !ar_prior))
        return fail("rtb200_mcmc_iterations_device: the AR move needs idxar, arpar and ar_prior together");
    if (int rc = check_move_args("rtb200_mcmc_iterations_device", NSrc, ldk)) return rc;
    if (!prior || !sd_prior) return fail("rtb200_mcmc_iterations_device needs the prior and sd_prior arrays");
    if (kmin < 1 || kmax < kmin || kmax > ldk) return fail("rtb200_mcmc_iterations_device needs 1 <= kmin <= kmax <= ldk");
    if (n_moves < 0 || n_moves + 3 > kGraphSlots) return fail("rtb200_mcmc_iterations_device: at most 509 moves per iteration");
    if (!d_counter || !d_workspace || !d_pos) return fail("rtb200_mcmc_iterations_device needs counter, workspace and pos");
    MoveCtx m = move_ctx(d_k, d_voro, d_logL, d_sigma, d_beta, B, ldk, d_src_offset, d_src_depth, d_tobs, NSrc);
    cudaStream_t st;
    if (int rc = begin_move(m, stream, d_idxar != nullptr, st)) return rc;
    const rtb::McmcWs w = rtb::mcmc_ws_layout(d_workspace, (size_t)B, (size_t)n_moves);
    // IAR = 1: with the AR move in the iteration, every likelihood of the iteration uses the chains'
    // AR state (as if registered with rtb200_set_chain_ar); the registration is restored on return
    struct ArScope {
        const int *i; const double *a; double m; bool on;
        ~ArScope() { if (on) { g.chain_idxar = i; g.chain_arpar = a; g.chain_armx = m; } }
    } ar_scope{g.chain_idxar, g.chain_arpar, g.chain_armx, d_idxar != nullptr};
    if (d_idxar) {
        g.chain_idxar = d_idxar;
        g.chain_arpar = d_arpar;
        g.chain_armx  = ar_prior[3];
    }
    std::vector<size_t> key = move_key(m);
    key_add(key, d_pos, n_moves, kmin, kmax, enos ? 1 : 0, seed, d_counter, d_workspace, d_tally, pk ? 1 : 0,
            d_idxar, d_arpar);
    for (int i = 0; i < 7; ++i) key_add(key, prior[i]);
    for (int i = 0; i < 3; ++i) key_add(key, sd_prior[i]);
    for (int i = kmin; pk && i <= kmax; ++i) key_add(key, pk[i - 1]);
    for (int i = 0; d_idxar && i < 4; ++i) key_add(key, ar_prior[i]);
    // kernel nodes take the graph slots past the MH-moves graph's
    auto capture = [&](cudaStream_t sc) {
        const rtb::MhPrior pr = make_prior(prior, enos);
        // ---- deviates of the birth/death and data-error moves, then the birth/death move
        cudaError_t e = rtb::launch_mcmc_draw(d_counter, seed, d_k, B, w, sc);
        if (e == cudaSuccess && kmin != kmax)
            e = enqueue_bd(m, pr, make_bd_prior(pk, kmin, kmax), w.u_k, w.idel, w.u_z, w.u_v, w.u_acc_bd,
                           w.acc_bd, graph_slot(kGraphSlots), false, sc);
        // ---- every chain's next n_moves fixed-dimension moves (schedule from the node counts now)
        if (e == cudaSuccess && n_moves > 0)
            e = rtb::launch_mcmc_sweep_draw(d_counter, seed, d_k, d_pos, B, n_moves, enos, w, sc);
        for (int i = 0; i < n_moves && e == cudaSuccess; ++i) {
            const size_t o = (size_t)i * (size_t)B;
            e = enqueue_mh(m, pr, w.ivo + o, w.iwhich + o, w.dev + o, w.u_acc + o, w.acc_mh + o, nullptr,
                           graph_slot(kGraphSlots + 1 + i), false, sc);
        }
        // ---- the data-error move, then the AR(1) move (IAR = 1)
        if (e == cudaSuccess)
            e = enqueue_sd(m, sd_prior, w.u_gate, w.gauss, w.u_acc_sd, w.acc_sd, graph_slot(kGraphSlots + 1 + n_moves),
                           false, sc);
        if (e == cudaSuccess && d_idxar)
            e = enqueue_ar(m, d_idxar, d_arpar, ar_prior, w.u_choice, w.u_prop_ar, w.gauss_ar, w.u_acc_ar, w.acc_ar,
                           graph_slot(kGraphSlots + 2 + n_moves), false, sc);
        if (e == cudaSuccess) e = rtb::launch_mcmc_finish(d_counter, d_k, d_pos, B, n_moves, w, d_tally, sc);
        return e;
    };
    if (int rc = run_graph(g.mc, key, m.cfg, "capturing the MCMC iteration", capture, n_iterations, st)) return rc;
    const long long per_iteration =
        3LL * n_moves + (kmin != kmax ? 3 : 0) + 3 + (d_idxar ? 3 : 0) + 2 + (n_moves > 0 ? 1 : 0);
    return end_move(m, (long long)n_iterations * per_iteration, false, stream, st);
}

int rtb200_swap_pack_device(const double *d_logL, const double *d_beta, int n, double *d_out,
                            void *stream) {
    ApiLock api_lock_;
    if (int rc = ensure_init()) return rc;
    g.err.clear();
    if (n <= 0) return 0;
    if (!d_logL || !d_beta || !d_out) return fail("rtb200_swap_pack_device needs logL, beta and out");
    cudaStream_t st = stream ? (cudaStream_t)stream : g.s_comp;
    CK(rtb::launch_swap_pack(d_logL, d_beta, n, d_out, st));
    g.launches++;
    if (!stream) CK(cudaStreamSynchronize(st));
    return 0;
}

int rtb200_swap_round_device(const double *d_all, int n, int lo, int n_local,
                             unsigned long long seed, unsigned long long round,
                             double *d_beta_local, int *d_accept, int *d_partner, void *stream) {
    ApiLock api_lock_;
    if (int rc = ensure_init()) return rc;
    g.err.clear();
    if (n <= 0 || n_local <= 0) return 0;
    if (!d_all || !d_beta_local) return fail("rtb200_swap_round_device needs the gathered pairs and beta_local");
    if (lo < 0 || lo + n_local > n) return fail("rtb200_swap_round_device: [lo, lo + n_local) must lie inside [0, n)");
    if (n > (1 << 30)) return fail("rtb200_swap_round_device: at most 2^30 chains");
    cudaStream_t st = stream ? (cudaStream_t)stream : g.s_comp;
    CK(rtb::launch_swap_round(d_all, n, lo, n_local, seed, round, d_beta_local, d_accept, d_partner, st));
    g.launches++;
    if (!stream) CK(cudaStreamSynchronize(st));
    return 0;
}

int rtb200_init(int device) {
    ApiLock api_lock_;
    const int rc = ensure_init(device);
    if (rc == 0) g.err.clear();
    return rc;
}

void rtb200_shutdown(void) {
    ApiLock api_lock_;
    if (!g.inited || !g.ok) { g.inited = false; return; }
    cudaSetDevice(g.device);
    cudaDeviceSynchronize();
    if (g.pin) cudaFreeHost(g.pin);
    g.pin = nullptr;
    g.pin_cap = 0;
    if (g.stage) cudaFreeHost(g.stage);
    if (g.stage_out) cudaFreeHost(g.stage_out);
    g.stage = g.stage_out = nullptr;
    g.stage_cap = g.stage_out_cap = 0;
    for (auto &e : g.ev_slot) { if (e) cudaEventDestroy(e); e = nullptr; }
    for (DevBuf *b : {&g.vels, &g.depths, &g.nl, &g.off, &g.dep, &g.tobs, &g.sigma,
                      &g.timeP, &g.pout, &g.logL, &g.arena, &g.voro, &g.vsorted, &g.idxar, &g.arparb,
                      &g.sched, &g.mh_ll, &g.mh_out, &g.mh_kp, &g.mh_lpr, &g.w, &g.dvels, &g.ddepths,
                      &g.dtdr, &g.dtdd, &g.JtJ, &g.Jtr})
        b->release();
    for (int i = 0; i < kMaxChunks; ++i) {
        cudaEventDestroy(g.ev_h2d[i]);
        cudaEventDestroy(g.ev_d2h[i]);
        cudaEventDestroy(g.ev_k0[i]);
        cudaEventDestroy(g.ev_k1[i]);
    }
    cudaEventDestroy(g.ev_t0);
    cudaEventDestroy(g.ev_t1);
    if (g.ev_scratch) cudaEventDestroy(g.ev_scratch);
    g.ev_scratch = nullptr;
    g.scratch_pending = false;
    cudaStreamDestroy(g.s_comp);
    cudaStreamDestroy(g.s_comp2);
    g.mv.reset();
    g.mc.reset();
    g.chain_idxar = nullptr;
    g.chain_arpar = nullptr;
    if (g.s_cap) cudaStreamDestroy(g.s_cap);
    g.s_cap = nullptr;
    cudaStreamDestroy(g.s_h2d);
    cudaStreamDestroy(g.s_d2h);
    g.inited = g.ok = false;
}

const char *rtb200_last_error(void) {
    // a copy per calling thread: the pointer stays valid while other threads go on calling
    ApiLock api_lock_;
    static thread_local std::string copy;
    copy = g.err;
    return copy.c_str();
}

int rtb200_device_count(void) {
    ApiLock api_lock_;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int rtb200_set_option(const char *name, double value) {
    ApiLock api_lock_;
    const int v = (int)value;
    if (!strcmp(name, "variant")) g.opt_variant = v < 0 ? -1 : v;
    else if (!strcmp(name, "threads")) g.opt_threads = v;
    else if (!strcmp(name, "tile_models")) g.opt_tile_models = v > 0 ? v : 0;
    else if (!strcmp(name, "tile_sources")) g.opt_tile_sources = v;
    else if (!strcmp(name, "chunk_models")) g.opt_chunk_models = v;
    else if (!strcmp(name, "ctas_per_sm")) g.opt_ctas = v;
    else if (!strcmp(name, "comp_streams")) g.opt_comp_streams = v;
    else if (!strcmp(name, "static_tiles")) g.opt_static_tiles = v > 0 ? 1 : 0;
    else if (!strcmp(name, "logl_shuffle")) g.opt_logl_shuffle = v > 0 ? 1 : 0;
    else if (!strcmp(name, "stage_pageable")) g.opt_stage = v < 0 ? -1 : (v > 0 ? 1 : 0);
    else if (!strcmp(name, "latency_path")) g.opt_latency = v == 0 ? 0 : 1;
    else if (!strcmp(name, "stable_lognorm")) g.opt_stable_lognorm = v > 0 ? 1 : 0;
    else if (!strcmp(name, "ismpprior")) g.opt_ismpprior = v > 0 ? 1 : 0;
    else return -1;
    return 0;
}

double rtb200_get_stat(const char *name) {
    ApiLock api_lock_;
    if (!strcmp(name, "kernel_ms")) return g.kernel_ms;
    if (!strcmp(name, "total_ms")) return g.total_ms;
    if (!strcmp(name, "launches")) return (double)g.launches;
    if (!strcmp(name, "tile_models")) return g.last.M;
    if (!strcmp(name, "tile_sources")) return g.last.SC;
    if (!strcmp(name, "smem_bytes")) return (double)g.last.smem;
    if (!strcmp(name, "grid")) return g.last.grid;
    if (!strcmp(name, "threads")) return g.last.threads;
    if (!strcmp(name, "ctas_per_sm")) return g.last_ctas;
    if (!strcmp(name, "variant")) return g.last.variant;
    if (!strcmp(name, "sms")) return g.sms;
    return std::numeric_limits<double>::quiet_NaN();
}

double rtb200_fp64_peak_tflops(int repeats) {
    ApiLock api_lock_;
    if (ensure_init()) return std::numeric_limits<double>::quiet_NaN();
    g.err.clear();
    double tf = 0.0;
    if (rtb::fp64_peak(&tf, repeats, g.s_comp) != cudaSuccess)
        return std::numeric_limits<double>::quiet_NaN();
    g.launches += 1 + (repeats > 0 ? repeats : 3);
    return tf;
}

double rtb200_selftest_fast_division(double samples, unsigned long long seed) {
    ApiLock api_lock_;
    if (ensure_init()) return -1.0;
    g.err.clear();
    double bad = -1.0;
    if (rtb::fastpath_selftest(samples, seed, &bad, g.s_comp) != cudaSuccess) return -1.0;
    g.launches += 1;
    return bad;
}

void rtb200_shard_range(long long B, int rank, int world, long long *lo, long long *hi) {
    if (world < 1) world = 1;
    const long long q = B / world, r = B % world;
    *lo = rank * q + std::min<long long>(rank, r);
    *hi = *lo + q + (rank < r ? 1 : 0);
}

}  // extern "C"
