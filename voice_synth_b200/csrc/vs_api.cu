/* vs_api.cu -- host side of libvoicesynth_cuda: context, parameter validation, cosine tables,
 * time-chunk planning, kernel launches and (for host buffers) slab-pipelined PCIe copies.
 *
 * What stays on the host, and why it is still bit-exact with the reference:
 *   - nSamples / P / T2 per stream: three scalar expressions (flowgen_shimmer.c:242,244,317) evaluated
 *     here with the same C types; x86-64 has no FMA contraction by default and the file is built
 *     with -ffp-contract=off.
 *   - cos(PI*i/T2) tables, one per distinct T2 of the batch, computed with the system libm exactly
 *     as the reference evaluates them (PI = 4.0*atan(1.0), flowgen_shimmer.c:39,319,328).  The
 *     kernels only ever multiply/add/ceil these doubles, so the int16 pulse cannot differ by an ulp
 *     of a device cosine.
 */
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <map>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/voicesynth.h"
#include "vs_internal.h"
#include "vs_presets.h"

enum { VS_MODE_FLOW = 0, VS_MODE_SYNTH = 1, VS_MODE_FILTER = 2 };
enum { VS_GEN_FAST = 0, VS_GEN_SIMPLE = 1 };
enum { VS_FILT_INT = 0, VS_FILT_FMA = 1, VS_FILT_EXACT = 2 };
cudaError_t vs_launch_plan(const VsPlanArgs &a, bool want_log, bool need_pulse, bool warp_per_stream, cudaStream_t s);
cudaError_t vs_launch_render(const VsRenderArgs &a, const VsTractBlock *tb, int mode, int gen, bool noise, int filt, cudaStream_t s);
static_assert(VS_MAX_TRACTS == VS_MAX_TRACTS_I, "tract count");
static_assert(VS_MAX_TRACTS <= 256, "a stream's tract index is a uint8_t");
cudaError_t vs_render_init_device();
int vs_render_window(int mode);
int vs_render_tiles(int mode);
cudaError_t vs_launch_flow_rows(const VsRenderArgs &a, cudaStream_t s);
int vs_flow_rows_warps(void);
cudaError_t vs_launch_fp64_peak(double *scratch, int blocks, int iters, cudaStream_t s);
cudaError_t vs_launch_vnoise(int16_t *pcm, const VsNoiseRow *rows, uint32_t n_rows, cudaStream_t s);
cudaError_t vs_launch_analyze(const int16_t *flow, const VsAnalyzeRow *rows, uint32_t n_rows, uint32_t *onsets, uint32_t *counts,
                              vs_flow_stats *out, cudaStream_t s);

namespace {

/* calls in flight per device slot: while call k renders, the plan kernels of calls k+1 and k+2 run side by side
 * (the period walk is latency bound: two of them on neighbouring SMs finish in the time of one) and the host
 * prepares call k+3 */
#define VS_DEPTH 4

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
};
struct PinBuf {
    void *p = nullptr;
    size_t cap = 0;
};

struct Slot {
    int dev = 0;
    int sm_count = 148;
    cudaStream_t compute = nullptr;
    bool own_compute = true;
    cudaStream_t copy = nullptr, copy2 = nullptr;    /* device->host: large runs go home in pieces alternating between the two */
    cudaEvent_t copy2_done = nullptr;
    cudaStream_t plans[2] = {nullptr, nullptr};      /* descriptor upload + plan kernel; calls alternate between the two */
    cudaEvent_t call_done[VS_DEPTH] = {};            /* everything of the call that used ring slot p has finished (compute) */
    cudaEvent_t plan_done[VS_DEPTH] = {};
    cudaEvent_t render_done[VS_DEPTH] = {};
    unsigned call_parity = 0;
    cudaEvent_t slab_done[2] = {nullptr, nullptr};   /* D2H of the slab using pcm[k] finished */
    cudaEvent_t slab_ready = nullptr;                /* render of the current slab finished   */
    DevBuf streams[VS_DEPTH], chunks[VS_DEPTH], order[VS_DEPTH], table[VS_DEPTH], snap[VS_DEPTH], nper[VS_DEPTH], status[VS_DEPTH];
    DevBuf costab, pcm[2], raw[2], flowin[2], log, ticket, analyze;
    unsigned burst = 0;                              /* calls since one found the device idle */
    uint32_t ticket_base = 0;                        /* value of the row counter of vs_flow_rows_kernel before the next launch */
    PinBuf h_streams[VS_DEPTH], h_chunks[VS_DEPTH], h_order[VS_DEPTH], h_nper[VS_DEPTH], h_status[VS_DEPTH];
    size_t costab_uploaded = 0;
    std::vector<cudaEvent_t> tev;                    /* timing events (slot 0 only) */
    size_t tev_used = 0;
    unsigned scratch_parity = 0;                     /* which pcm[]/raw[]/flowin[] the next slab uses */
    bool slab_done_valid[2] = {false, false};
    /* chunk plan of the previous call, reused when the batch has the same shape */
    std::vector<uint64_t> plan_sig;
    std::vector<VsChunk> plan_chunks;
    std::vector<uint32_t> plan_order, plan_nch;
    struct PlanGeom {                                /* per slab: what the render launch needs besides the rows */
        uint32_t cta_end[VS_MAX_TRACTS_I];           /* group ends: presets in blocks of 32 rows, tracts in CTAs  */
        uint32_t cache_doubles;                      /* pulse-table cache a warp needs (fast generator)        */
    };
    std::vector<PlanGeom> plan_geom;
    std::vector<size_t> plan_slab_c0, plan_slab_r0;
    uint64_t plan_tab_total = 0, plan_warm_total = 0;
    uint64_t plan_version = 1, uploaded_version[VS_DEPTH] = {};        /* which plan the device copies of chunks/order hold (0 = none) */
    std::chrono::steady_clock::time_point last_enqueue{};
    uint64_t plan_for_version = 0;                   /* vs_ctx::in_version of the inputs the plan was made (or confirmed) for */
    uint64_t streams_version[VS_DEPTH] = {};         /* which inputs the device copies of the stream descriptors hold          */
};

} // namespace

struct vs_ctx {
    std::vector<Slot> slots;
    double opt_chunk = 0;        /* 0 auto, <0 never, >0 fixed */
    double opt_tol = 1e-12;      /* x |state| <= ~2e5 at the default gain: 2e-7 before quantisation, 50 x under the 1e-5 bar */
    int opt_plan_warps = -1;     /* -1 auto, 0 one thread per stream, 1 one warp per stream */
    int opt_exact = 0;
    int opt_slab = 0;
    double opt_warps = 2.0;
    int opt_async_host = 0;
    int opt_debug = 0;
    int opt_simple_gen = 0;      /* 1: never use the branch-free generator (debug / A-B) */
    std::vector<double> cos_host;
    std::map<int, uint32_t> cos_index;
    std::vector<uint32_t> cos_fast;      /* T2 -> table offset, direct index in front of the map */
    std::map<uint64_t, uint32_t> pulse_index;   /* (T2, bits of K) -> offset of the h / K*c-K+1 table */
    uint64_t pulse_last_key = ~0ull;
    uint32_t pulse_last_off = 0;
    int warm[VS_NUM_PRESETS];    /* warm-up samples per preset at opt_tol (gain-independent part) */
    double l1gain[VS_NUM_PRESETS]; /* sum |h[n]| of each preset: |y| <= l1gain * gain * max|x| */
    std::unordered_map<std::string, int> tract_warm;   /* warm-up at opt_tol of every tract seen, keyed by its 23 coefficients' bytes */
    std::string err;
    vs_timing timing;
    bool timing_pending = false;
    /* the previous call's inputs, byte for byte, and everything derived from them on the host: a call with the same
     * parameters (a corpus generator re-running a shape, the benchmark loop) skips validation, descriptor
     * building, chunk planning and the descriptor upload */
    std::vector<unsigned char> in_blob;
    std::vector<VsStream> in_hs;
    struct Facts {
        uint64_t max_n = 0;
        bool any_noise = false, any_kvar = false, int_filter = true, amp_fits = true, noise_simple = true;
        int t_min = 0x7fffffff, t_max = 0, t2_min = 0x7fffffff;
    } in_facts;
    std::vector<int> in_warm;      /* warm-up per filter group of the inputs: per preset, or per tract of a _tract call */
    std::vector<double> in_ncoef;  /* [n_tracts][VS_ORDER] = -A[1..22] of the inputs' tracts (tract calls) */
    uint64_t in_version = 0;     /* bumped whenever in_hs changes */
    bool env_profile_host = false, env_sync_plan = false;
};

namespace {

/* the ABI has no globals: a call leaves the caller's current device as it found it */
struct DeviceGuard {
    int prev = -1;
    DeviceGuard() { if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; cudaGetLastError(); } }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

int fail(vs_ctx *c, int code, const char *fmt, ...)
{
    if (c) {
        char buf[512];
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(buf, sizeof buf, fmt, ap);
        va_end(ap);
        c->err = buf;
    }
    return code;
}

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(ctx, VS_ECUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

int dev_reserve(vs_ctx *ctx, Slot &s, DevBuf &b, size_t bytes)
{
    if (bytes <= b.cap) return VS_OK;
    if (b.p) {
        CU(cudaStreamSynchronize(s.plans[0]));
        CU(cudaStreamSynchronize(s.plans[1]));
        CU(cudaStreamSynchronize(s.compute));
        CU(cudaStreamSynchronize(s.copy2));
        CU(cudaStreamSynchronize(s.copy));
        CU(cudaFree(b.p));
        b.p = nullptr; b.cap = 0;
    }
    size_t cap = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&b.p, cap);
    if (e != cudaSuccess) { b.p = nullptr; return fail(ctx, VS_ENOMEM, "cudaMalloc(%zu) failed: %s", cap, cudaGetErrorString(e)); }
    b.cap = cap;
    return VS_OK;
}

int pin_reserve(vs_ctx *ctx, PinBuf &b, size_t bytes)
{
    if (bytes <= b.cap) return VS_OK;
    if (b.p) { cudaFreeHost(b.p); b.p = nullptr; b.cap = 0; }
    size_t cap = bytes + bytes / 8 + 256;
    cudaError_t e = cudaHostAlloc(&b.p, cap, cudaHostAllocDefault);
    if (e != cudaSuccess) { b.p = nullptr; return fail(ctx, VS_ENOMEM, "cudaHostAlloc(%zu) failed: %s", cap, cudaGetErrorString(e)); }
    b.cap = cap;
    return VS_OK;
}

/* ---- parameter access with the reference defaults (flowgen_shimmer.c:87, vowel_new.c:76-77) ---- */
struct FlowRow {
    float dur, jitter, shimmer, cq, K, Kvar, F0, DC, noise;
    int32_t amp, fs;
    uint8_t flags;
    uint32_t seed;
};

FlowRow flow_row(const vs_flow_params *p, size_t i)
{
    FlowRow r;
    r.dur = p && p->dur ? p->dur[i] : 1.0f;
    r.jitter = p && p->jitter ? p->jitter[i] : 0.0f;
    r.shimmer = p && p->shimmer ? p->shimmer[i] : 0.0f;
    r.cq = p && p->cq ? p->cq[i] : 0.55f;
    r.K = p && p->K ? p->K[i] : 0.65f;
    r.Kvar = p && p->Kvar ? p->Kvar[i] : 0.0f;
    r.F0 = p && p->F0 ? p->F0[i] : 120.0f;
    r.DC = p && p->DC ? p->DC[i] : 0.0f;
    r.noise = p && p->noise ? p->noise[i] : 0.0f;
    r.amp = p && p->amp ? p->amp[i] : 12000;
    r.fs = p && p->fs ? p->fs[i] : 22050;
    r.flags = p && p->flags ? p->flags[i] : 0;
    r.seed = p && p->seed ? p->seed[i] : 1u;
    return r;
}

uint64_t row_nsamples(const FlowRow &r)
{
    /* `(unsigned long) par.fs*par.dur`: unsigned long * float is a float product (:242) */
    volatile float prod = (float)(uint64_t)(int64_t)r.fs * r.dur;
    if (!(prod >= 0.0f) || prod >= 1.8e19f) return 0;
    return (uint64_t)prod;
}

int row_P(const FlowRow &r)
{
    volatile float q = (float)(int64_t)r.fs / r.F0;                   /* :244 */
    if (!(q > -2147483648.0f && q < 2147483648.0f)) return 0;
    return (int)q;
}

int row_T2(const FlowRow &r, int P)
{
    volatile double h = 0.5 * (double)r.cq;                           /* :317 */
    volatile double v = h * P;
    return (int)std::ceil(v);
}

int row_validate(const FlowRow &r, int *P_out = nullptr, uint64_t *n_out = nullptr)
{
    if (!(r.fs > 0) || !std::isfinite(r.dur) || !(r.dur > 0.0f)) return VS_ERANGE;
    if (!std::isfinite(r.F0) || !(r.F0 > 0.0f)) return VS_ERANGE;
    const int P = row_P(r);
    if (P < 1 || P > 27000) return VS_ERANGE;                        /* T <= 1.2*P is stored in a short (:289) */
    const uint64_t n = row_nsamples(r);
    if (n < 1 || n > 0x7fffffffull) return VS_ERANGE;
    if (P_out) *P_out = P;
    if (n_out) *n_out = n;
    if (!(r.jitter >= 0.0f && r.jitter <= 10.0f)) return VS_ERANGE;   /* :478 */
    if (!(r.shimmer >= 0.0f && r.shimmer <= 1.0f)) return VS_ERANGE;  /* :544 */
    if (!(r.cq >= 0.0f && r.cq <= 1.0f)) return VS_ERANGE;            /* :490 */
    if (!std::isfinite(r.K) || !(r.K >= 0.0f)) return VS_ERANGE;
    if (!(r.Kvar >= 0.0f && r.Kvar <= 1.0f)) return VS_ERANGE;        /* :530 */
    if (!(r.amp >= 0 && r.amp < 32767)) return VS_ERANGE;             /* :518 */
    if (!std::isfinite(r.DC) || !(r.DC >= 0.0f) || r.DC > 32767.0f) return VS_ERANGE;
    /* the tool accepts 0..50 dB, i.e. noise = 10^(dB/10) >= 1 (:505-511).  Below 0.1 (-10 dB) NoiseDistWidth could pass
     * 2^19, the range the render kernel's two-operation noise sample is proven for (tests/tools/noisecheck.c) */
    if ((r.flags & VS_F_NOISE) && (!std::isfinite(r.noise) || !(r.noise >= 0.1f))) return VS_ERANGE;
    if (r.flags & ~(VS_F_JITTER | VS_F_SHIMMER | VS_F_NOISE)) return VS_EINVAL;
    /* Falling branch (:327-332): x = (short)ceil(A*(K*c - K + 1)), left at the first x < DC.  Between two samples
     * the argument drops by at most A*K*2*sin(pi/(2*T2)); while that step stays below 2^15 the first value under DC
     * still fits the short and the reference stops there.  Beyond it the cast wraps before the DC test and what
     * the reference emits is an accident of 16-bit wrap-around: refused (SURVEY.md 8a, hazards).  (A above 32767
     * needs no bound: x[T2] = (short)ceil(A) is negative and the branch is left at once.) */
    const int T2 = row_T2(r, P);
    if (T2 >= 2) {
        const double amax = std::min(32767.0, ((r.flags & VS_F_SHIMMER) && r.shimmer != 0.0f ? 1.8 : 1.0) * (double)r.amp);
        const double kmax = (double)r.K * (1.0 + (double)r.Kvar);
        if (amax * kmax * 2.0 * std::sin(3.141592653589793 / (2.0 * (double)T2)) > 32768.0) return VS_ERANGE;
    }
    return VS_OK;
}

uint32_t row_max_periods(const FlowRow &r, uint64_t n, int P)
{
    const bool jit = (r.flags & VS_F_JITTER) && r.jitter != 0.0f;
    int tmin = P;
    if (jit) {
        tmin = (int)std::floor(0.8f * (float)P);                      /* accepted T satisfy (float)T >= (float)0.8*P */
        if (tmin < 1) tmin = 1;
    }
    return (uint32_t)(n / (uint64_t)tmin + 2);
}

int preset_index(int key)
{
    const char *q = key ? strchr(vs_preset_keys, key) : nullptr;
    return q ? (int)(q - vs_preset_keys) : -1;
}

/* Samples after which the free response of an arbitrary unit-bounded initial state has decayed below
 * tol: W = 1 + last n with sum_j |(Phi^n)[0][j]| >= tol, Phi the companion matrix of the preset. */
int warmup_for(const double *A, double tol, int limit = 60000)
{
    const int N = VS_ORDER;
    /* column j holds the free response state started from unit vector e_j */
    std::vector<double> st(N * N, 0.0);
    for (int j = 0; j < N; j++) st[j * N + j] = 1.0;       /* st[j*N + k] = y[n-1-k] of response j */
    int last = 0;
    const int horizon = 60000;
    int quiet = 0;
    for (int n = 0; n < horizon; n++) {
        double g = 0.0;
        for (int j = 0; j < N; j++) {
            double *s = &st[j * N];
            double y0 = 0.0;
            for (int k = 0; k < N; k++) y0 -= A[k + 1] * s[k];
            for (int k = N - 1; k > 0; k--) s[k] = s[k - 1];
            s[0] = y0;
            g += std::fabs(y0);
        }
        if (!(g < tol)) { last = n + 1; quiet = 0; if (last >= limit) break; }    /* (a response that overflowed: not decayed) */
        else if (++quiet > 4096) break;
    }
    return last + 1;
}

double l1_gain_for(const double *A)
{
    double s[VS_ORDER] = {0.0};
    double sum = 0.0;
    for (int n = 0; n < 60000; n++) {
        double y0 = n == 0 ? 1.0 : 0.0;
        for (int k = 0; k < VS_ORDER; k++) y0 -= A[k + 1] * s[k];
        for (int k = VS_ORDER - 1; k > 0; k--) s[k] = s[k - 1];
        s[0] = y0;
        sum += std::fabs(y0);
    }
    return sum;
}

void compute_warmups(vs_ctx *ctx)
{
    for (int k = 0; k < VS_NUM_PRESETS; k++) {
        ctx->warm[k] = warmup_for(vs_preset_den[k], ctx->opt_tol);
        ctx->l1gain[k] = l1_gain_for(vs_preset_den[k]);
    }
}

uint32_t cos_table_for(vs_ctx *ctx, int T2)
{
    if (T2 >= 0 && (size_t)T2 < ctx->cos_fast.size() && ctx->cos_fast[T2] != 0xffffffffu) return ctx->cos_fast[T2];
    auto it = ctx->cos_index.find(T2);
    if (it != ctx->cos_index.end()) return it->second;
    const uint32_t off = (uint32_t)ctx->cos_host.size();
    volatile double one = 1.0;
    const double pi = 4.0 * std::atan(one);                           /* #define PI 4.0*atan(1.0) (:39) */
    /* layout per T2: h[0..T2) then c[0..T2), so that the open-phase index i in [0,2*T2) addresses it
     * directly.  h[i] = 0.5*(1-c[i]): (A*0.5)*(1.0-c) == A*h bit for bit, scaling by 0.5 being exact (:319) */
    std::vector<double> c((size_t)T2);
    for (int i = 0; i < T2; i++) {
        volatile double num = pi * i;                                 /* PI*i/T2 == ((4.0*atan(1.0))*i)/T2 */
        volatile double arg = num / T2;
        c[i] = std::cos(arg);
    }
    for (int i = 0; i < T2; i++) {
        volatile double om = 1.0 - c[i];
        volatile double h = 0.5 * om;
        const double hv = h;
        ctx->cos_host.push_back(hv);
    }
    for (int i = 0; i < T2; i++) ctx->cos_host.push_back(c[i]);
    ctx->cos_index[T2] = off;
    if (T2 >= 0 && T2 < 65536) {
        if ((size_t)T2 >= ctx->cos_fast.size()) ctx->cos_fast.resize((size_t)T2 + 64, 0xffffffffu);
        ctx->cos_fast[T2] = off;
    }
    return off;
}

/* Open-phase table of a stream whose closure speed never varies (-z absent: Knew == K in every period):
 * h[0..T2) as above, then f[i] = (K*c[i] - K) + 1.0 with the reference's three roundings (:328), so that a
 * falling-branch sample is ceil(A * f[i]) like a rising one is ceil(A * h[i]).  Saves the render kernel three of
 * its five FP64 operations per open-phase sample. */
uint32_t pulse_table_for(vs_ctx *ctx, int T2, float K)
{
    uint32_t kb;
    memcpy(&kb, &K, 4);
    const uint64_t key = ((uint64_t)(uint32_t)T2 << 32) | kb;
    if (key == ctx->pulse_last_key) return ctx->pulse_last_off;
    auto it = ctx->pulse_index.find(key);
    uint32_t off;
    if (it != ctx->pulse_index.end()) off = it->second;
    else {
        const uint32_t src = cos_table_for(ctx, T2);                  /* h then c; may grow cos_host */
        if (ctx->cos_host.size() & 1) ctx->cos_host.push_back(0.0);   /* 16-byte aligned */
        off = (uint32_t)ctx->cos_host.size();
        for (int i = 0; i < T2; i++) { const double h = ctx->cos_host[src + i]; ctx->cos_host.push_back(h); }
        const double Kd = (double)K;
        for (int i = 0; i < T2; i++) {
            volatile double kc = Kd * ctx->cos_host[src + T2 + i];
            volatile double d = kc - Kd;
            volatile double f = d + 1.0;
            const double fv = f;
            ctx->cos_host.push_back(fv);
        }
        /* for vs_flow_rows_kernel, which reads two neighbouring entries with one 16-byte load: two zeros (the closed
         * phase), then the same table again moved up by one entry, so that a pair is 16-byte aligned in one of the two
         * copies whatever its parity */
        const size_t n2 = 2 * (size_t)T2;
        ctx->cos_host.push_back(0.0);
        ctx->cos_host.push_back(0.0);
        for (size_t k = 0; k < n2 + 2; k++) { const double v = k + 1 < n2 + 2 ? ctx->cos_host[off + k + 1] : 0.0; ctx->cos_host.push_back(v); }
        ctx->pulse_index[key] = off;
    }
    ctx->pulse_last_key = key;
    ctx->pulse_last_off = off;
    return off;
}

enum PtrKind { PK_HOST_PAGEABLE, PK_HOST_PINNED, PK_DEVICE };

PtrKind classify(const void *p, int *dev_out)
{
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return PK_HOST_PAGEABLE; }
    if (at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged) { if (dev_out) *dev_out = at.device; return PK_DEVICE; }
    if (at.type == cudaMemoryTypeHost) return PK_HOST_PINNED;
    return PK_HOST_PAGEABLE;
}

cudaEvent_t timing_event(Slot &s)
{
    if (s.tev_used == s.tev.size()) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        s.tev.push_back(e);
    }
    return s.tev[s.tev_used++];
}

struct Batch {
    int mode;
    size_t n;
    const vs_flow_params *fp;
    const vs_filter_params *ff;
    const vs_tract_params *ft;     /* _tract calls: caller-defined tracts instead of ff */
    const int16_t *flow_in;
    const uint64_t *in_offsets;
    const uint64_t *nsamp;
    int16_t *pcm_out;
    const uint64_t *offsets;
    double *raw_out;
    vs_period_log *log;
};

/* SMs the render kernel leaves to the plan kernels of the next calls.  A plan CTA keeps an SM for one plan time; the
 * plan of a step takes a little longer than its render (measured: 1.2x on the bench workload and on the noise
 * grid), so 1.5 SMs per plan CTA -- two plans partly side by side -- keep the plans ahead of the renders.  Large
 * batches get none: their plan needs every SM anyway and simply alternates with the render. */
int vs_plan_reserve(int plan_ctas)
{
    return 2 * plan_ctas <= VS_PLAN_SMS ? (3 * plan_ctas + 1) / 2 : 0;
}

/* Choose the time-chunk length for a group of streams (SURVEY.md 7 "Occupancy").
 * Filtering modes: the FP64 pipe of an SM sub-partition is saturated by ONE consumer warp, so the
 * kernel time is  waves * (L + warm-up)  sample-steps with  waves = ceil(warps / (SMs*4));  every
 * chunk but the first pays the warm-up again.  Pick the chunk count per stream that minimises it.
 * Flow mode has no carry, chunks are free: aim at `8*opt_warps` warps per sub-partition. */
uint32_t choose_chunk(vs_ctx *ctx, const Slot &slot, int mode, size_t n_streams, uint64_t total, double avg_warm, bool flow_rows)
{
    if (ctx->opt_chunk < 0) return 0;
    if (mode != VS_MODE_FLOW && ctx->opt_exact) return 0;
    if (flow_rows) {
        /* lanes along the row (vs_flow_rows_kernel): a warp takes a row at a time, 256 samples per step, rows handed out
         * by a ticket -- about four rows per warp balance the SMs and keep the cost of opening a row (its descriptors,
         * the first batch of periods: five dependent memory round trips) small.  Measured on the bench batch: 2.6 / 3.5 /
         * 5.2 / 7.8 rows per warp = 0.078 / 0.076 / 0.078 / 0.080 ms */
        double L = ctx->opt_chunk > 0 ? ctx->opt_chunk : std::ceil((double)total / ((double)slot.sm_count * 4.0 * vs_flow_rows_warps() * 4.0));
        if (L < 512.0) L = 512.0;
        if (L > 1048576.0) L = 1048576.0;
        return ((uint32_t)L + 255u) & ~255u;
    }
    if (ctx->opt_chunk > 0) {
        uint32_t L = (uint32_t)ctx->opt_chunk;
        L = (L + 7u) & ~7u;
        return L < 64 ? 64 : L;
    }
    const double smsp = (double)slot.sm_count * 4.0;
    const double avg_n = (double)total / (double)n_streams;
    if (mode == VS_MODE_FLOW) {
        /* the flow has no carry, chunks are free: one full wave of rows (4 CTAs of VS_NT rows per SM), or whole
         * waves of >= 512-sample chunks when the batch is small */
        (void)smsp; (void)avg_n;
        const double lanes = (double)slot.sm_count * 4.0 * VS_NT * 0.97;
        if ((double)n_streams >= lanes) return 0;
        double L = std::ceil((double)total / lanes);
        if (L < 512.0) L = 512.0;
        return ((uint32_t)L + 7u) & ~7u;
    }
    double best_cost = 1e300;
    uint32_t best_L = 0;
    for (int C = 1; C <= 256; C++) {
        const double L = std::ceil(avg_n / C / 8.0) * 8.0;
        if (C > 1 && L < 512.0) break;
        const double warps = std::ceil((double)n_streams * C / 32.0);
        const double waves = std::ceil(warps / smsp);
        const double cost = waves * (L + (C > 1 ? avg_warm : 0.0));
        if (cost < best_cost * 0.999) { best_cost = cost; best_L = C == 1 ? 0u : (uint32_t)L; }
    }
    return best_L;
}

/* Per-stream chunk counts for the filtering modes.  A chunk of stream s costs  W_s + L_s  sample
 * steps (W_s = carry warm-up of its preset); the kernel time is that of the most expensive chunk
 * times the number of waves, one wave = one CTA of VS_NT rows per SM.  So: give every stream the
 * chunk length  L_s = budget - W_s  and pick the smallest budget whose rows fit in `waves` waves;
 * take the wave count with the smallest  waves * budget. */
void plan_filter_chunks(vs_ctx *ctx, const Slot &slot, const std::vector<VsStream> &hs, size_t a0, size_t a1,
                        std::vector<uint32_t> &nchunks, int plan_nt, const int *warm, bool tracts)
{
    const size_t ns = a1 - a0;
    nchunks.assign(ns, 1u);
    if (ctx->opt_chunk < 0 || ctx->opt_exact) return;
    if (ctx->opt_chunk > 0) {
        uint32_t L = ((uint32_t)ctx->opt_chunk + 7u) & ~7u;
        if (L < 64) L = 64;
        for (size_t i = 0; i < ns; i++) nchunks[i] = hs[a0 + i].n <= L ? 1u : (uint32_t)((hs[a0 + i].n + L - 1) / L);
        return;
    }
    /* rows per wave; a few SMs stay free for the plan kernels of the next two calls (one CTA of VS_PLAN_NT streams per
     * SM each, see VS_PLAN_SMEM) */
    const int plan_ctas = (int)((ns + (size_t)plan_nt - 1) / (size_t)plan_nt);
    const int reserve = vs_plan_reserve(plan_ctas);
    const int render_sms = slot.sm_count > 4 * VS_PLAN_SMS ? slot.sm_count - reserve : slot.sm_count;
    const double cap = (double)render_sms * VS_NT;
    /* streams of equal (length, preset) get equal chunk counts: plan over the distinct classes */
    std::map<std::pair<uint32_t, uint8_t>, uint32_t> classes;
    uint32_t nmax = 0;
    for (size_t i = 0; i < ns; i++) {
        classes[{hs[a0 + i].n, hs[a0 + i].preset}]++;
        nmax = std::max(nmax, hs[a0 + i].n);
    }
    /* the first chunk of a stream needs no warm-up, so it emits `budget` samples, the others budget - W */
    auto chunks_of = [&](uint32_t n, uint8_t preset, double budget) -> uint32_t {
        if ((double)n <= budget) return 1u;
        const double L = std::max(512.0, budget - (double)warm[preset]);
        return 1u + (uint32_t)std::ceil(((double)n - budget) / L);
    };
    /* presets: groups padded to blocks of 32 rows, a 3 % allowance covers that; tracts: groups padded to whole CTAs,
     * counted exactly */
    const double fill = tracts ? 1.0 : 0.97;
    auto rows_for = [&](double budget) -> double {
        if (!tracts) {
            double rows = 0;
            for (const auto &kv : classes) rows += (double)kv.second * chunks_of(kv.first.first, kv.first.second, budget);
            return rows;
        }
        double per[VS_MAX_TRACTS_I] = {0.0};
        for (const auto &kv : classes) per[kv.first.second] += (double)kv.second * chunks_of(kv.first.first, kv.first.second, budget);
        double rows = 0;
        for (int t = 0; t < VS_MAX_TRACTS_I; t++) rows += std::ceil(per[t] / VS_NT) * VS_NT;
        return rows;
    };
    double best_cost = 1e300, best_budget = (double)nmax;
    for (int waves = 1; waves <= 8; waves++) {
        if (rows_for((double)nmax) > waves * cap) continue;                    /* even unchunked does not fit */
        double lo = 512.0, hi = (double)nmax;                                  /* smallest budget that fits */
        for (int it = 0; it < 30; it++) {
            const double mid = 0.5 * (lo + hi);
            if (rows_for(mid) <= waves * cap * fill) hi = mid; else lo = mid;
        }
        const double cost = waves * hi;
        if (cost < best_cost * 0.98) { best_cost = cost; best_budget = hi; }
    }
    for (size_t i = 0; i < ns; i++) nchunks[i] = chunks_of(hs[a0 + i].n, hs[a0 + i].preset, best_budget);
}

/* a tract's warm-up at the ctx's tolerance, computed once per context; -1 if it is not acceptable */
#define VS_TRACT_MAX_WARMUP 16384
int tract_warmup(vs_ctx *ctx, const double *A)
{
    const std::string key(reinterpret_cast<const char *>(A), (VS_ORDER + 1) * sizeof(double));
    auto it = ctx->tract_warm.find(key);
    if (it != ctx->tract_warm.end()) return it->second;
    const int w = warmup_for(A, ctx->opt_tol, VS_TRACT_MAX_WARMUP + 1);
    if (ctx->tract_warm.size() >= (1u << 16)) ctx->tract_warm.clear();   /* a bound on what a stream of one-off tracts leaves behind */
    ctx->tract_warm.emplace(key, w);
    return w;
}

struct HostProf {
    bool on;
    std::chrono::steady_clock::time_point t0;
    explicit HostProf(bool enabled) : on(enabled), t0(std::chrono::steady_clock::now()) {}
    void mark(const char *what)
    {
        if (!on) return;
        auto t = std::chrono::steady_clock::now();
        fprintf(stderr, "[vs host] %-28s %8.1f us\n", what, std::chrono::duration<double, std::micro>(t - t0).count());
        t0 = t;
    }
};

/* the inputs of a batch call as one byte string: scalars, which arrays are present, and the arrays' contents */
void snapshot_inputs(const Batch &b, bool want_log, const void *extra, size_t extra_bytes, std::vector<unsigned char> &blob)
{
    blob.clear();
    auto put = [&](const void *p, size_t bytes) {
        const unsigned char *c = static_cast<const unsigned char *>(p);
        blob.insert(blob.end(), c, c + bytes);
    };
    auto arr = [&](const void *p, size_t elem) {
        const unsigned char have = p != nullptr;
        put(&have, 1);
        if (p) put(p, elem * b.n);
    };
    const uint64_t head[4] = {(uint64_t)b.mode, (uint64_t)b.n, (uint64_t)want_log, (uint64_t)(b.raw_out != nullptr)};
    put(head, sizeof head);
    put(extra, extra_bytes);
    if (b.fp) {
        arr(b.fp->dur, 4); arr(b.fp->jitter, 4); arr(b.fp->shimmer, 4); arr(b.fp->cq, 4); arr(b.fp->K, 4); arr(b.fp->Kvar, 4);
        arr(b.fp->F0, 4); arr(b.fp->DC, 4); arr(b.fp->noise, 4); arr(b.fp->amp, 4); arr(b.fp->fs, 4); arr(b.fp->flags, 1); arr(b.fp->seed, 4);
    }
    if (b.ff) { arr(b.ff->preset, 1); arr(b.ff->gain, 4); arr(b.ff->pre, 4); }
    if (b.ft) {
        const uint64_t nt = b.ft->n_tracts;
        put(&nt, sizeof nt);
        if (b.ft->den && nt <= VS_MAX_TRACTS) put(b.ft->den, nt * (VS_ORDER + 1) * sizeof(double));
        arr(b.ft->tract, 1); arr(b.ft->gain, 4); arr(b.ft->pre, 4);
    }
    arr(b.nsamp, 8); arr(b.in_offsets, 8); arr(b.offsets, 8);
    if (want_log) put(b.log->rec_offsets, 8 * (b.n + 1));
}

/* half-open sample ranges [lo, hi) of the rows: do any two intersect? */
bool rows_overlap(std::vector<std::pair<uint64_t, uint64_t>> &r)
{
    std::sort(r.begin(), r.end());
    for (size_t i = 1; i < r.size(); i++)
        if (r[i].first < r[i - 1].second) return true;
    return false;
}

int run_batch(vs_ctx *ctx, const Batch &b)
{
    if (!ctx) return VS_EINVAL;
    DeviceGuard restore_device;
    HostProf prof(ctx->env_profile_host);
    if (b.n == 0) return VS_OK;
    if (!b.pcm_out) return fail(ctx, VS_EINVAL, "pcm_out is NULL");
    if (b.mode == VS_MODE_FILTER && (!b.flow_in || !b.nsamp)) return fail(ctx, VS_EINVAL, "flow_in/nsamp is NULL");
    if (b.n > 0x7fffffffull) return fail(ctx, VS_EINVAL, "too many streams");
    const size_t n = b.n;
    const bool want_log = b.log && b.log->rec && b.log->rec_offsets && b.mode != VS_MODE_FILTER;

    /* ---- 1. per-stream descriptors (or last call's, when the inputs are the same bytes) -------- */
    static thread_local std::vector<unsigned char> blob;
    int odev = -1;
    const PtrKind out_kind = classify(b.pcm_out, &odev);
    {   /* what the chunk plan depends on besides the parameter arrays */
        const double key[10] = {ctx->opt_chunk, ctx->opt_tol, (double)ctx->opt_exact, (double)ctx->opt_slab, ctx->opt_warps, (double)ctx->opt_simple_gen,
                                (double)(out_kind == PK_DEVICE), (double)(reinterpret_cast<uintptr_t>(b.pcm_out) & 127), (double)ctx->slots.size(),
                                b.ft ? 1.0 : 0.0};
        snapshot_inputs(b, want_log, key, sizeof key, blob);
    }
    const bool same_inputs = blob.size() == ctx->in_blob.size() && memcmp(blob.data(), ctx->in_blob.data(), blob.size()) == 0;
    if (!same_inputs) {
    ctx->in_blob.clear();                                    /* nothing is cached while the tables below may fail half way */
    std::vector<VsStream> &hs = ctx->in_hs;
    hs.assign(n, VsStream());
    uint64_t max_n = 0;
    bool any_noise = false, any_kvar = false;
    bool int_filter = true;          /* every stream: integral gain, pre-emphasis 0 or 1 -> both commute to the integer input */
    int t_min = 0x7fffffff, t_max = 0;   /* bounds on the pitch period lengths of the batch */
    int t2_min = 0x7fffffff;             /* shortest half open phase */
    bool amp_fits = true;            /* no amplitude can pass 32767 (fast generator) */
    bool noise_simple = true;        /* every noisy stream has DC <= 1 (then T4 == 0) and T2 >= 16: 16-byte period entries do */
    /* filter groups: the ten presets, or the caller's tracts (validated, warm-ups from the ctx's cache) */
    ctx->in_warm.assign(ctx->warm, ctx->warm + VS_NUM_PRESETS);
    ctx->in_ncoef.clear();
    if (b.ft) {
        const uint32_t nt = b.ft->n_tracts;
        if (!b.ft->den || nt == 0 || nt > VS_MAX_TRACTS) return fail(ctx, VS_EINVAL, "n_tracts %u outside 1..%d (or den is NULL)", nt, VS_MAX_TRACTS);
        ctx->in_warm.assign(nt, 0);
        ctx->in_ncoef.assign((size_t)nt * VS_ORDER, 0.0);
        for (uint32_t t = 0; t < nt; t++) {
            const double *A = b.ft->den + (size_t)t * (VS_ORDER + 1);
            for (int j = 0; j <= VS_ORDER; j++)
                if (!std::isfinite(A[j])) return fail(ctx, VS_ERANGE, "tract %u: coefficient %d is not finite", t, j);
            if (A[0] != 1.0) return fail(ctx, VS_ERANGE, "tract %u: A[0] = %g, must be 1", t, A[0]);
            const int w = tract_warmup(ctx, A);
            if (w > VS_TRACT_MAX_WARMUP) return fail(ctx, VS_ERANGE, "tract %u: unstable or nearly marginal (carry warm-up above %d samples)", t, VS_TRACT_MAX_WARMUP);
            ctx->in_warm[t] = w;
            for (int j = 1; j <= VS_ORDER; j++) ctx->in_ncoef[(size_t)t * VS_ORDER + j - 1] = -A[j];
        }
    }
    for (size_t i = 0; i < n; i++) {
        VsStream &s = hs[i];
        memset(&s, 0, sizeof s);
        if (b.mode == VS_MODE_FILTER) {
            if (b.nsamp[i] > 0x7fffffffull) return fail(ctx, VS_EOVERLAP, "stream %zu: too many samples", i);
            s.n = (uint32_t)b.nsamp[i];
        } else {
            const FlowRow r = flow_row(b.fp, i);
            int P = 0;
            uint64_t nn = 0;
            const int rc = row_validate(r, &P, &nn);
            if (rc) return fail(ctx, rc, "stream %zu: flow parameter out of range", i);
            s.n = (uint32_t)nn;
            s.P = P;
            s.T2 = row_T2(r, s.P);
            s.cos_off = cos_table_for(ctx, s.T2);
            t2_min = std::min(t2_min, (int)s.T2);
            any_kvar |= r.Kvar != 0.0f;
            s.amp = r.amp; s.DC = r.DC; s.jitter = r.jitter; s.shimmer = r.shimmer; s.K = r.K; s.Kvar = r.Kvar;
            s.noise = r.noise; s.seed = r.seed; s.flags = r.flags;
            s.DCs = (int16_t)(int32_t)r.DC;                            /* x[i] = par.DC (:321,:335) */
            s.tab_cap = row_max_periods(r, s.n, s.P);
            any_noise |= (r.flags & VS_F_NOISE) != 0;
            if ((r.flags & VS_F_NOISE) && !(r.DC <= 1.0f && s.T2 >= 16)) noise_simple = false;
            {   /* accepted periods satisfy 0.8*P <= T <= 1.2*P (flowgen_shimmer.c:290) */
                const bool jit = (r.flags & VS_F_JITTER) && r.jitter != 0.0f;
                t_min = std::min(t_min, jit ? std::max(1, (int)std::floor(0.8f * (float)P)) : P);
                const int tm = jit ? (int)std::ceil(1.2f * (float)P) + 1 : P;
                t_max = std::max(t_max, tm);
                s.tpad = (uint32_t)((tm + 9) & ~1);                     /* refined per table below */
                if ((r.flags & VS_F_SHIMMER) && r.shimmer != 0.0f ? 1.8f * (float)r.amp > 32767.0f : r.amp > 32767) amp_fits = false;
            }
        }
        if (b.mode != VS_MODE_FLOW && b.ft) {
            const uint32_t t = b.ft->tract ? b.ft->tract[i] : 0u;
            if (t >= b.ft->n_tracts) return fail(ctx, VS_EINVAL, "stream %zu: tract index %u >= n_tracts %u", i, t, b.ft->n_tracts);
            s.preset = (uint8_t)t;                                      /* the filter group: here a tract */
            s.gain = b.ft->gain ? b.ft->gain[i] : 10.0f;
            s.pre = b.ft->pre ? b.ft->pre[i] : 1.0f;
        } else if (b.mode != VS_MODE_FLOW) {
            const int key = b.ff && b.ff->preset ? b.ff->preset[i] : 'a';
            const int pi = preset_index(key);
            if (pi < 0) return fail(ctx, VS_EPRESET, "stream %zu: unknown vowel preset 0x%02x", i, key);
            s.preset = (uint8_t)pi;
            s.gain = b.ff && b.ff->gain ? b.ff->gain[i] : 10.0f;
            s.pre = b.ff && b.ff->pre ? b.ff->pre[i] : 1.0f;
        }
        if (b.mode != VS_MODE_FLOW) {
            if (!std::isfinite(s.gain) || !std::isfinite(s.pre)) return fail(ctx, VS_ERANGE, "stream %zu: gain/pre not finite", i);
            if (!(s.gain == std::floor(s.gain) && std::fabs(s.gain) <= 32767.0f && (s.pre == 0.0f || s.pre == 1.0f))) int_filter = false;
        }
        max_n = std::max<uint64_t>(max_n, s.n);
    }
    for (size_t i = 0; i < n; i++) {
        hs[i].out_off = b.offsets ? b.offsets[i] : (uint64_t)i * max_n;
        if (b.mode == VS_MODE_FILTER) hs[i].in_off = b.in_offsets ? b.in_offsets[i] : (uint64_t)i * max_n;
        if (want_log) hs[i].log_off = b.log->rec_offsets[i];
    }
    /* the table the render kernel reads: with no -z anywhere in the batch, the falling branch pre-multiplied by K
     * (one table per distinct (T2, K); a batch with a different K on every stream keeps the general path instead
     * of growing the tables without bound) */
    if (b.mode != VS_MODE_FILTER) {
        for (size_t i = 0; i < n && !any_kvar; i++) {
            const size_t before = ctx->cos_host.size();
            hs[i].pulse_off = pulse_table_for(ctx, hs[i].T2, hs[i].K);
            if (ctx->cos_host.size() > before && ctx->cos_host.size() > VS_PULSE_TABLE_CAP) any_kvar = true;
        }
        if (any_kvar)
            for (size_t i = 0; i < n; i++) hs[i].pulse_off = hs[i].cos_off;
        /* streams that share a table share its padded length */
        std::map<uint32_t, uint32_t> pad;
        for (size_t i = 0; i < n; i++) { uint32_t &v = pad[hs[i].pulse_off]; v = std::max(v, hs[i].tpad); }
        for (size_t i = 0; i < n; i++) hs[i].tpad = pad[hs[i].pulse_off];
    }

    /* output rows must not intersect, nor may a filter's output overlap another row's input except in place */
    {
        std::vector<std::pair<uint64_t, uint64_t>> rows(n);
        for (size_t i = 0; i < n; i++) rows[i] = {hs[i].out_off, hs[i].out_off + hs[i].n};
        if (rows_overlap(rows)) return fail(ctx, VS_EOVERLAP, "output rows overlap");
    }
    vs_ctx::Facts &fc = ctx->in_facts;
    fc.max_n = max_n; fc.any_noise = any_noise; fc.any_kvar = any_kvar; fc.int_filter = int_filter; fc.amp_fits = amp_fits;
    fc.noise_simple = noise_simple; fc.t_min = t_min; fc.t_max = t_max; fc.t2_min = t2_min;
    ctx->in_blob.swap(blob);
    ctx->in_version++;
    }
    std::vector<VsStream> &hs = ctx->in_hs;
    const vs_ctx::Facts &fc = ctx->in_facts;
    const bool any_noise = fc.any_noise, any_kvar = fc.any_kvar, int_filter = fc.int_filter, amp_fits = fc.amp_fits, noise_simple = fc.noise_simple;
    const int t_min = fc.t_min, t_max = fc.t_max;
    const bool tracts = b.ft != nullptr;
    const int *gwarm = ctx->in_warm.data();          /* warm-up per filter group (preset or tract) */
    const int n_groups = tracts ? VS_MAX_TRACTS_I : VS_NUM_PRESETS;
    const size_t group_rows = tracts ? VS_NT : 32;   /* groups are padded to whole CTAs (tracts) or blocks of 32 rows (presets) */

    prof.mark("stream descriptors");
    /* ---- 2. where do the buffers live ------------------------------------------------------- */
    const PtrKind raw_kind = b.raw_out ? classify(b.raw_out, nullptr) : out_kind;
    const PtrKind in_kind = b.flow_in ? classify(b.flow_in, nullptr) : out_kind;
    const bool out_dev = out_kind == PK_DEVICE;
    if ((b.raw_out && (raw_kind == PK_DEVICE) != out_dev) || (b.flow_in && (in_kind == PK_DEVICE) != out_dev))
        return fail(ctx, VS_EINVAL, "pcm/raw/flow buffers must be all host or all device");
    if (out_dev && ctx->slots.size() != 1) return fail(ctx, VS_EINVAL, "device buffers need a single-device ctx");
    if (out_dev && odev != ctx->slots[0].dev) return fail(ctx, VS_EINVAL, "device buffer lives on device %d, ctx on %d", odev, ctx->slots[0].dev);
    if (out_dev && b.mode == VS_MODE_FILTER) {
        /* time-chunks of a row read flow samples that belong to the previous chunk's output range (carry warm-up):
         * the filter cannot run in place on device memory (host buffers are staged apart) */
        uint64_t ilo = ~0ull, ihi = 0, olo = ~0ull, ohi = 0;
        for (size_t i = 0; i < n; i++) {
            ilo = std::min(ilo, hs[i].in_off); ihi = std::max(ihi, hs[i].in_off + hs[i].n);
            olo = std::min(olo, hs[i].out_off); ohi = std::max(ohi, hs[i].out_off + hs[i].n);
        }
        const uintptr_t i0 = reinterpret_cast<uintptr_t>(b.flow_in + ilo), i1 = reinterpret_cast<uintptr_t>(b.flow_in + ihi);
        const uintptr_t o0 = reinterpret_cast<uintptr_t>(b.pcm_out + olo), o1 = reinterpret_cast<uintptr_t>(b.pcm_out + ohi);
        if (i0 < o1 && o0 < i1) return fail(ctx, VS_EOVERLAP, "flow_in and pcm_out overlap in device memory");
    }

    /* ---- 3. contiguous stream ranges per device slot, balanced by samples (SURVEY.md 8e) ------ */
    const size_t nslots = ctx->slots.size();
    std::vector<size_t> cut(nslots + 1, n);
    {
        uint64_t total = 0;
        for (size_t i = 0; i < n; i++) total += hs[i].n;
        cut[0] = 0;
        uint64_t acc = 0;
        size_t g = 1;
        for (size_t i = 0; i < n && g < nslots; i++) {
            acc += hs[i].n;
            while (g < nslots && acc * nslots >= total * g) cut[g++] = i + 1;
        }
    }

    memset(&ctx->timing, 0, sizeof ctx->timing);
    ctx->timing_pending = true;
    const bool exact = ctx->opt_exact != 0;
    /* period table format: 8-byte entries (amplitude, length) where they suffice, 16-byte ones for plain glottal noise */
    const int compact = (any_kvar || want_log) ? VS_TAB_FULL : !any_noise ? VS_TAB_C8 : noise_simple ? VS_TAB_N16 : VS_TAB_FULL;
    /* flow without glottal noise: lanes along the row (vs_flow_rows_kernel).  T2 >= 2: row_validate() bounds A*K then */
    const bool flow_rows = b.mode == VS_MODE_FLOW && compact == VS_TAB_C8 && amp_fits && !ctx->opt_simple_gen && t_min >= 24 && fc.t2_min >= 2;
    const uint64_t ph_mask = flow_rows ? 63u : 7u;
    /* streams per CTA of the thread-form plan kernel: without glottal noise and period log its lean form (vs_plan.cu) */
    const int plan_nt = (any_noise || want_log) ? VS_PLAN_NT : VS_PLAN_NT_LEAN;           /* rows keep their position inside a 128-byte line / a 16-byte piece */

    /* ---- 4. per slot: descriptors up, then slabs of plan -> render -> copy ------------------- */
    for (size_t g = 0; g < nslots; g++) {
        Slot &sl = ctx->slots[g];
        const size_t s0 = cut[g], s1 = cut[g + 1];
        if (s1 <= s0) continue;
        const size_t ns = s1 - s0;
        CU(cudaSetDevice(sl.dev));
        if (g == 0) sl.tev_used = 0;

        uint64_t total = 0;
        double warm_sum = 0.0;
        for (size_t i = s0; i < s1; i++) {
            total += hs[i].n;
            if (b.mode != VS_MODE_FLOW) warm_sum += gwarm[hs[i].preset];
        }
        /* slabs: groups of consecutive streams that are launched and copied together */
        size_t slab_streams = ns;
        if (!out_dev) {
            if (ctx->opt_slab > 0) slab_streams = (size_t)ctx->opt_slab;
            else {
                /* one slab per call unless the device mirror of the output would be huge; PCIe/compute
                 * overlap comes from alternating two scratch buffers ACROSS calls (VS_OPT_ASYNC_HOST) */
                const uint64_t bytes = total * 2;
                size_t want = (size_t)std::max<uint64_t>(1, (bytes + (1ull << 30) - 1) >> 30);
                slab_streams = (ns + want - 1) / want;
            }
            if (slab_streams < 1) slab_streams = 1;
        }
        const size_t n_slabs = (ns + slab_streams - 1) / slab_streams;

        /* chunk plan + row order: a function of the batch SHAPE only (lengths, presets, row phases,
         * options), so a call shaped like the previous one reuses it */
        std::vector<uint64_t> sig;
        const bool known_plan = same_inputs && sl.plan_for_version == ctx->in_version;     /* same bytes as the call that made the plan */
        if (!known_plan) {
        sig.reserve(3 * ns + 8);
        sig.push_back(((uint64_t)b.mode << 48) ^ ((uint64_t)n_slabs << 24) ^ (uint64_t)slab_streams ^ ((uint64_t)plan_nt << 52));
        sig.push_back((uint64_t)(int64_t)ctx->opt_chunk ^ ((uint64_t)ctx->opt_exact << 62) ^ ((uint64_t)sl.sm_count << 40));
        { double t = ctx->opt_tol, w = ctx->opt_warps; uint64_t u; memcpy(&u, &t, 8); sig.push_back(u); memcpy(&u, &w, 8); sig.push_back(u); }
        sig.push_back((uint64_t)tracts);
        if (tracts) for (int w : ctx->in_warm) sig.push_back((uint64_t)w);   /* the chunk plan depends on the tracts' warm-ups */
        for (size_t i = s0; i < s1; i++) {
            const uint64_t base_addr = out_dev ? (reinterpret_cast<uintptr_t>(b.pcm_out) >> 1) + hs[i].out_off : hs[i].out_off;
            sig.push_back((uint64_t)hs[i].n | ((uint64_t)hs[i].preset << 32) | ((base_addr & ph_mask) << 40));
            sig.push_back((uint64_t)hs[i].tab_cap | ((uint64_t)hs[i].pulse_off << 32));          /* row order and table cache depend on these */
            sig.push_back((uint64_t)(uint32_t)hs[i].T2 | ((uint64_t)hs[i].tpad << 32));
        }
        }
        const bool plan_hit = known_plan || sig == sl.plan_sig;
        sl.plan_for_version = ctx->in_version;
        if (!plan_hit) {
        std::vector<VsChunk> &hc = sl.plan_chunks;
        hc.clear();
        sl.plan_nch.assign(ns, 1u);
        std::vector<size_t> &slab_c0 = sl.plan_slab_c0;
        slab_c0.assign(n_slabs + 1, 0);
        uint64_t tab_total = 0, warm_total = 0;
        for (size_t k = 0; k < n_slabs; k++) {
            const size_t a0 = s0 + k * slab_streams, a1 = std::min(s1, a0 + slab_streams);
            uint64_t tot = 0;
            for (size_t i = a0; i < a1; i++) tot += hs[i].n;
            const uint32_t Lflow = b.mode == VS_MODE_FLOW ? choose_chunk(ctx, sl, b.mode, a1 - a0, tot, 0.0, flow_rows) : 0u;
            std::vector<uint32_t> nch;
            if (b.mode != VS_MODE_FLOW) plan_filter_chunks(ctx, sl, hs, a0, a1, nch, plan_nt, gwarm, tracts);
            slab_c0[k] = hc.size();
            for (size_t i = a0; i < a1; i++) {
                VsStream &s = hs[i];
                const uint64_t base_addr = out_dev ? (reinterpret_cast<uintptr_t>(b.pcm_out) >> 1) + s.out_off : s.out_off;
                /* host outputs are mirrored on the device at the same offsets relative to a 16-byte
                 * aligned slab base, so the phase of a row is its sample offset mod 8 either way */
                const uint32_t ph = (uint32_t)(base_addr & ph_mask);
                const uint32_t W = (b.mode == VS_MODE_FLOW) ? 0u : (uint32_t)gwarm[s.preset];
                /* chunk c > 0 emits [L0 + (c-1)*L - ph, L0 + c*L - ph); L0 and L are multiples of 8 (of 256 for the
                 * lanes-along-the-row flow kernel, whose steps then never straddle two chunks) */
                uint32_t C, L, L0;
                if (b.mode == VS_MODE_FLOW) {
                    L = L0 = Lflow;
                    C = (L == 0 || s.n <= L) ? 1u : (uint32_t)((s.n + L - 1) / L);
                } else {
                    C = nch[i - a0];
                    L = L0 = 0u;
                    if (C > 1) {
                        if (ctx->opt_chunk == 0 && (uint64_t)s.n > (uint64_t)W + 64ull * C) {       /* auto planning */
                            /* equal WORK per row: the first chunk has no warm-up and emits W samples more */
                            L = (uint32_t)(((s.n - W + C - 1) / C + 7u) & ~7u);
                            const uint32_t rest = (C - 1) * L;
                            L0 = rest < s.n ? ((s.n - rest + 7u) & ~7u) : 0u;
                        }
                        if (L0 == 0u || L0 < L) {                      /* stream barely longer than the warm-up: equal chunks */
                            L = L0 = (uint32_t)(((s.n + C - 1) / C + 7u) & ~7u);
                        }
                        C = s.n <= L0 ? 1u : 1u + (uint32_t)((s.n - L0 + L - 1) / L);
                    }
                }
                sl.plan_nch[i - s0] = C;
                tab_total += s.tab_cap;
                for (uint32_t c = 0; c < C; c++) {
                    VsChunk ck;
                    memset(&ck, 0, sizeof ck);
                    ck.stream = (uint32_t)(i - s0);
                    ck.emit_lo = c == 0 ? 0u : L0 + (c - 1) * L - ph;
                    ck.emit_hi = c + 1 == C ? s.n : L0 + c * L - ph;
                    ck.gen_target = ck.emit_lo > W ? ck.emit_lo - W : 0u;
                    if (c > 0) warm_total += ck.emit_lo - ck.gen_target;
                    hc.push_back(ck);
                }
            }
        }
        slab_c0[n_slabs] = hc.size();
        sl.plan_tab_total = tab_total;
        sl.plan_warm_total = warm_total;
        prof.mark("chunk plan");
        /* render rows: ONE launch per slab.  Rows are grouped by vowel preset and every preset group is padded to whole
         * CTAs with VS_NO_CHUNK rows, so that a CTA's preset is a function of blockIdx (its coefficients then sit in
         * uniform registers).  Inside a preset: longest first (the 32 lanes of a warp run a similar number of windows),
         * rows of equal work next to each other by pulse table (a warp stages each distinct table of its rows once). */
        std::vector<uint32_t> &order = sl.plan_order;
        order.clear();
        sl.plan_geom.assign(n_slabs, Slot::PlanGeom());
        sl.plan_slab_r0.assign(n_slabs + 1, 0);
        for (size_t k = 0; k < n_slabs; k++) {
            sl.plan_slab_r0[k] = order.size();
            std::vector<uint32_t> ids(slab_c0[k + 1] - slab_c0[k]);
            auto preset_of = [&](uint32_t c) -> int { return b.mode == VS_MODE_FLOW ? 0 : hs[s0 + hc[c].stream].preset; };
            {   /* sort by one 64-bit key per row (preset, work descending, pulse table), then by id: the comparator of a
                 * sort over the descriptors themselves cost 2.6 ms per 16 384 rows */
                std::vector<std::pair<uint64_t, uint32_t>> keyed(ids.size());
                for (size_t c = 0; c < ids.size(); c++) {
                    const uint32_t id = (uint32_t)(slab_c0[k] + c);
                    /* (flow-only chunks are all about one length: keep rows that share a pulse table together instead) */
                    const uint32_t work = b.mode == VS_MODE_FLOW ? 0u : (hc[id].emit_hi - hc[id].gen_target) >> 6;
                    keyed[c] = {((uint64_t)preset_of(id) << 57) | ((uint64_t)(0x01ffffffu - std::min(work, 0x01ffffffu)) << 32) |
                                    (uint64_t)hs[s0 + hc[id].stream].pulse_off, id};
                }
                std::sort(keyed.begin(), keyed.end());
                for (size_t c = 0; c < ids.size(); c++) ids[c] = keyed[c].second;
            }
            Slot::PlanGeom &gm = sl.plan_geom[k];
            const size_t r_first = order.size();
            size_t i0 = 0;
            int pr_done = 0;
            while (i0 < ids.size()) {
                size_t i1 = i0;
                const int pr = preset_of(ids[i0]);
                while (i1 < ids.size() && preset_of(ids[i1]) == pr) i1++;
                for (; pr_done < pr; pr_done++) gm.cta_end[pr_done] = (uint32_t)((order.size() - r_first) / group_rows);
                for (size_t i = i0; i < i1; i++) order.push_back(ids[i]);
                while ((order.size() - r_first) % group_rows) order.push_back(VS_NO_CHUNK);
                i0 = i1;
            }
            for (; pr_done < n_groups; pr_done++) gm.cta_end[pr_done] = (uint32_t)((order.size() - r_first) / group_rows);
            /* pulse-table cache: the largest sum of distinct (padded) tables over the warps of the slab */
            gm.cache_doubles = 0;
            if (b.mode != VS_MODE_FILTER) {
                for (size_t r = r_first; r < order.size(); r += 32) {
                    uint32_t seen[32], nseen = 0, sum = 0;
                    for (size_t j = r; j < r + 32; j++) {
                        if (order[j] == VS_NO_CHUNK) continue;
                        const VsStream &st = hs[s0 + hc[order[j]].stream];
                        bool dup = false;
                        for (uint32_t u = 0; u < nseen; u++) dup |= seen[u] == st.pulse_off;
                        if (!dup) { seen[nseen++] = st.pulse_off; sum += st.tpad; }
                    }
                    gm.cache_doubles = std::max(gm.cache_doubles, sum);
                }
            }
        }
        sl.plan_slab_r0[n_slabs] = order.size();
        sl.plan_sig.swap(sig);
        sl.plan_version++;
        prof.mark("row order");
        }
        const std::vector<VsChunk> &hc = sl.plan_chunks;
        const std::vector<uint32_t> &order = sl.plan_order;
        const std::vector<size_t> &slab_c0 = sl.plan_slab_c0, &slab_r0 = sl.plan_slab_r0;
        const uint64_t tab_total = sl.plan_tab_total, warm_total = sl.plan_warm_total;
        {
            uint32_t c0acc = 0;
            uint64_t tacc = 0;
            for (size_t i = s0; i < s1; i++) {
                hs[i].chunk0 = c0acc; hs[i].n_chunks = sl.plan_nch[i - s0]; hs[i].tab_off = tacc;
                c0acc += hs[i].n_chunks; tacc += hs[i].tab_cap;
            }
        }
        const size_t nc = hc.size(), nrows = order.size();
        ctx->timing.chunks += (uint32_t)nc;
        ctx->timing.samples += total;
        ctx->timing.warmup_samples += warm_total;

        /* device memory: descriptor/table buffers alternate between calls (parity cp), so that the
         * upload + plan kernel of this call can run while the previous call still renders */
        const unsigned cp = sl.call_parity;
        sl.call_parity = (sl.call_parity + 1u) % VS_DEPTH;
        cudaStream_t pstream = sl.plans[cp & 1u];
        CU(cudaEventSynchronize(sl.call_done[cp]));                   /* the call before the previous one is done with them */
        int rc;
        /* The descriptor / table buffers form a ring of VS_DEPTH sets.  When one of them has to grow, the same buffer of
         * every set grows with it: a new batch shape pays for its memory in its FIRST call (growing means a device-wide
         * synchronisation, cudaFree / cudaMalloc / cudaHostAlloc), not in each of its first VS_DEPTH calls. */
        auto drain = [&]() -> int {
            CU(cudaStreamSynchronize(sl.plans[0]));
            CU(cudaStreamSynchronize(sl.plans[1]));
            CU(cudaStreamSynchronize(sl.compute));
            CU(cudaStreamSynchronize(sl.copy2));
            CU(cudaStreamSynchronize(sl.copy));
            return VS_OK;
        };
        auto ring_dev = [&](DevBuf (&ring)[VS_DEPTH], size_t bytes) -> int {
            if (bytes <= ring[cp].cap) return VS_OK;
            for (unsigned d = 0; d < VS_DEPTH; d++) {
                const void *before = ring[d].p;
                const int r = dev_reserve(ctx, sl, ring[d], bytes);
                if (r) return r;
                if (before != ring[d].p) { sl.uploaded_version[d] = 0; sl.streams_version[d] = 0; }   /* its contents are gone */
            }
            return VS_OK;
        };
        auto ring_pin = [&](PinBuf (&ring)[VS_DEPTH], size_t bytes) -> int {
            if (bytes <= ring[cp].cap) return VS_OK;
            const int r0 = drain();                                   /* copies of the calls in flight read from these */
            if (r0) return r0;
            for (unsigned d = 0; d < VS_DEPTH; d++) {
                const int r = pin_reserve(ctx, ring[d], bytes);
                if (r) return r;
            }
            return VS_OK;
        };
        if ((rc = ring_dev(sl.streams, ns * sizeof(VsStream)))) return rc;
        if ((rc = ring_dev(sl.chunks, nc * sizeof(VsChunk)))) return rc;
        if ((rc = ring_dev(sl.order, nrows * sizeof(uint32_t) + 16))) return rc;
        if ((rc = ring_dev(sl.nper, ns * sizeof(uint32_t)))) return rc;
        if ((rc = ring_dev(sl.status, sizeof(int32_t)))) return rc;
        if (b.mode != VS_MODE_FILTER) {
            if ((rc = ring_dev(sl.table, (tab_total + 8) * VS_TAB_ENTRY_BYTES(compact)))) return rc;
            if (any_noise && (rc = ring_dev(sl.snap, nc * 32 * sizeof(uint32_t)))) return rc;
            if ((rc = dev_reserve(ctx, sl, sl.costab, (ctx->cos_host.size() + VS_COS_SLACK) * sizeof(double)))) return rc;
            if (sl.costab_uploaded != ctx->cos_host.size()) {
                /* tables only ever grow; a synchronous copy keeps the host vector free to grow again */
                /* stream-ordered on the plan stream (a plain cudaMemcpy from pageable memory may still be in
                 * flight when it returns, and non-blocking streams do not order after the legacy stream) */
                CU(cudaStreamSynchronize(sl.compute));
                CU(cudaStreamSynchronize(sl.plans[0]));
                CU(cudaStreamSynchronize(sl.plans[1]));
                CU(cudaMemcpyAsync(sl.costab.p, ctx->cos_host.data(), ctx->cos_host.size() * sizeof(double), cudaMemcpyHostToDevice, pstream));
                CU(cudaStreamSynchronize(pstream));
                ctx->timing.h2d_bytes += ctx->cos_host.size() * sizeof(double);
                sl.costab_uploaded = ctx->cos_host.size();
            }
        }
        if ((rc = ring_pin(sl.h_streams, ns * sizeof(VsStream)))) return rc;
        if ((rc = ring_pin(sl.h_chunks, nc * sizeof(VsChunk)))) return rc;
        if ((rc = ring_pin(sl.h_order, nrows * sizeof(uint32_t) + 16))) return rc;
        if ((rc = ring_pin(sl.h_nper, ns * sizeof(uint32_t)))) return rc;
        if ((rc = ring_pin(sl.h_status, sizeof(int32_t)))) return rc;

        /* log span of this slot */
        uint64_t log_lo = 0, log_hi = 0;
        if (want_log) {
            log_lo = b.log->rec_offsets[s0];
            log_hi = b.log->rec_offsets[s1];
            for (size_t i = s0; i < s1; i++) {
                if (b.log->rec_offsets[i + 1] < b.log->rec_offsets[i] || b.log->rec_offsets[i + 1] - b.log->rec_offsets[i] < hs[i].tab_cap)
                    return fail(ctx, VS_EINVAL, "stream %zu: period log too small (need %u records)", i, hs[i].tab_cap);
                hs[i].log_off = b.log->rec_offsets[i] - log_lo;
            }
            if ((rc = dev_reserve(ctx, sl, sl.log, std::max<uint64_t>(1, log_hi - log_lo) * sizeof(vs_period_rec)))) return rc;
            CU(cudaMemsetAsync(sl.log.p, 0, (log_hi - log_lo) * sizeof(vs_period_rec), pstream));
        }

        /* device-side offsets: rows of a slab live at (offset - slab_min) + pad to keep the phase */
        struct SlabGeom { uint64_t out_min, out_max, in_min, in_max; };
        std::vector<SlabGeom> geom(n_slabs);
        uint64_t span_max = 0, in_span_max = 0;
        for (size_t k = 0; k < n_slabs; k++) {
            const size_t a0 = s0 + k * slab_streams, a1 = std::min(s1, a0 + slab_streams);
            SlabGeom gm = {~0ull, 0, ~0ull, 0};
            for (size_t i = a0; i < a1; i++) {
                gm.out_min = std::min(gm.out_min, hs[i].out_off);
                gm.out_max = std::max(gm.out_max, hs[i].out_off + hs[i].n);
                gm.in_min = std::min(gm.in_min, hs[i].in_off);
                gm.in_max = std::max(gm.in_max, hs[i].in_off + hs[i].n);
            }
            gm.out_min &= ~63ull;                                     /* keep (offset mod 64) on the device */
            gm.in_min &= ~7ull;
            geom[k] = gm;
            span_max = std::max(span_max, gm.out_max - gm.out_min);
            in_span_max = std::max(in_span_max, gm.in_max - gm.in_min);
        }
        if (!out_dev) {
            for (int d = 0; d < 2; d++) {
                if ((rc = dev_reserve(ctx, sl, sl.pcm[d], span_max * sizeof(int16_t) + 256))) return rc;
                if (b.raw_out && (rc = dev_reserve(ctx, sl, sl.raw[d], span_max * sizeof(double) + 64))) return rc;
                if (b.mode == VS_MODE_FILTER && (rc = dev_reserve(ctx, sl, sl.flowin[d], in_span_max * sizeof(int16_t) + 64))) return rc;
            }
        }

        /* upload descriptors; the previous call on this slot must be done with the staging buffers
         * (everything above overlapped with it) */
        /* (the device copy of slot `cp` may still hold exactly these descriptors: three calls ago, same inputs) */
        const bool upload_streams = sl.streams_version[cp] != ctx->in_version;     /* (0 after the buffer was reallocated) */
        VsStream *ps = (VsStream *)sl.h_streams[cp].p;
        for (size_t k = 0; upload_streams && k < n_slabs; k++) {
            const size_t a0 = s0 + k * slab_streams, a1 = std::min(s1, a0 + slab_streams);
            for (size_t i = a0; i < a1; i++) {
                ps[i - s0] = hs[i];
                if (!out_dev) {
                    ps[i - s0].out_off = hs[i].out_off - geom[k].out_min;
                    ps[i - s0].in_off = hs[i].in_off - geom[k].in_min;
                }
            }
        }
        /* chunk geometry and row order depend on the batch shape only; the plan kernel rewrites every
         * chunk's first_period each call.  Re-upload them only when the plan changed. */
        const bool upload_plan = sl.uploaded_version[cp] != sl.plan_version;
        if (upload_plan) {
            memcpy(sl.h_chunks[cp].p, hc.data(), nc * sizeof(VsChunk));
            memcpy(sl.h_order[cp].p, order.data(), nrows * sizeof(uint32_t));
        }
        *(int32_t *)sl.h_status[cp].p = 0;
        if (upload_streams) {
            CU(cudaMemcpyAsync(sl.streams[cp].p, sl.h_streams[cp].p, ns * sizeof(VsStream), cudaMemcpyHostToDevice, pstream));
            sl.streams_version[cp] = ctx->in_version;
            ctx->timing.h2d_bytes += ns * sizeof(VsStream);
        }
        if (upload_plan) {
            CU(cudaMemcpyAsync(sl.chunks[cp].p, sl.h_chunks[cp].p, nc * sizeof(VsChunk), cudaMemcpyHostToDevice, pstream));
            CU(cudaMemcpyAsync(sl.order[cp].p, sl.h_order[cp].p, nrows * sizeof(uint32_t), cudaMemcpyHostToDevice, pstream));
            sl.uploaded_version[cp] = sl.plan_version;
            ctx->timing.h2d_bytes += nc * sizeof(VsChunk) + nrows * sizeof(uint32_t);
        }
        CU(cudaMemsetAsync(sl.status[cp].p, 0, sizeof(int32_t), pstream));

        prof.mark("reserve + descriptor upload");
        /* ---- plan stream: descriptors are up (above), now the plan kernel(s) of every slab -------- */
        if (g == 0) { cudaEvent_t t_first = timing_event(sl); CU(cudaEventRecord(t_first, pstream)); }
        if (b.mode != VS_MODE_FILTER) {
            for (size_t k = 0; k < n_slabs; k++) {
                const size_t a0 = s0 + k * slab_streams, a1 = std::min(s1, a0 + slab_streams);
                VsPlanArgs pa;
                memset(&pa, 0, sizeof pa);
                pa.streams = (const VsStream *)sl.streams[cp].p + (a0 - s0);
                pa.n_streams = (uint32_t)(a1 - a0);
                pa.chunks = (VsChunk *)sl.chunks[cp].p;
                pa.table = sl.table[cp].p;
                pa.compact = compact;
                pa.rng_snap = any_noise ? (uint32_t *)sl.snap[cp].p : nullptr;
                pa.n_periods = (uint32_t *)sl.nper[cp].p + (a0 - s0);
                pa.costab = (const double *)sl.costab.p;
                pa.log = want_log ? sl.log.p : nullptr;
                pa.status = (int32_t *)sl.status[cp].p;
                pa.need_pulse = want_log;
                /* One warp per stream while the batch is too small to fill the GPU with one thread per stream
                 * (measured crossover on B200: ~8 k streams, ~14 k with glottal noise, where a thread walks
                 * hundreds of serial pulse samples and draws per period).  The warp form issues ~7x the
                 * instructions, though: when the previous call is still rendering it would take issue slots
                 * from the FP64-bound render warps, while the thread form hides on its own SMs -- so with a
                 * call in flight only really small batches take it. */
                bool plan_warps;
                if (ctx->opt_plan_warps >= 0) plan_warps = ctx->opt_plan_warps != 0;
                else {
                    /* "in flight" = the previous call has not finished, or it was enqueued less than 2 ms ago (a
                     * loop of calls whose host side momentarily fell behind the GPU is still a pipeline) */
                    bool busy = cudaEventQuery(sl.call_done[(cp + VS_DEPTH - 1u) % VS_DEPTH]) == cudaErrorNotReady;
                    (void)cudaGetLastError();
                    const auto now = std::chrono::steady_clock::now();
                    if (std::chrono::duration<double, std::milli>(now - sl.last_enqueue).count() < 2.0) busy = true;
                    sl.last_enqueue = now;
                    /* the second call of a burst that began on an idle device: its plan must be ready when the first
                     * call's render ends, one render time from now -- the thread form (0.39 ms on the bench batch, and it
                     * has to wait for free SMs behind the first call's warp-form plan) would be late by a quarter of a
                     * step, and every call behind it too until the pipeline has settled */
                    sl.burst = busy ? sl.burst + 1u : 0u;
                    const bool early = busy && sl.burst == 1u && !any_noise;     /* (with glottal noise the warp form is too heavy to share the SMs with a render: cfg3 157 -> 150 Gsamples/s) */
                    plan_warps = pa.n_streams <= (busy && !early ? VS_PLAN_WARP_MAX : any_noise ? VS_PLAN_WARP_MAX_NOISE : VS_PLAN_WARP_MAX_IDLE);
                }
                CU(vs_launch_plan(pa, want_log, any_noise || want_log, plan_warps, pstream));
                ctx->timing.launches++;
            }
        }
        if (g == 0) { cudaEvent_t t_plan = timing_event(sl); CU(cudaEventRecord(t_plan, pstream)); }
        CU(cudaEventRecord(sl.plan_done[cp], pstream));
        if (ctx->env_sync_plan) CU(cudaStreamSynchronize(pstream));
        CU(cudaStreamWaitEvent(sl.compute, sl.plan_done[cp], 0));

        /* ---- compute stream: render (and copy) slab by slab ------------------------------------------ */
        for (size_t k = 0; k < n_slabs; k++) {
            const size_t a0 = s0 + k * slab_streams, a1 = std::min(s1, a0 + slab_streams);
            const size_t c0 = slab_c0[k], c1 = slab_c0[k + 1];
            const int d = (int)((sl.scratch_parity + k) & 1);
            int16_t *d_pcm = out_dev ? b.pcm_out : (int16_t *)sl.pcm[d].p;
            double *d_raw = b.raw_out ? (out_dev ? b.raw_out : (double *)sl.raw[d].p) : nullptr;
            const int16_t *d_in = nullptr;

            if (!out_dev && sl.slab_done_valid[d]) CU(cudaStreamWaitEvent(sl.compute, sl.slab_done[d], 0));   /* its last D2H */

            if (b.mode == VS_MODE_FILTER) {
                if (out_dev) d_in = b.flow_in;
                else {
                    d_in = (const int16_t *)sl.flowin[d].p;
                    CU(cudaMemcpyAsync(sl.flowin[d].p, b.flow_in + geom[k].in_min, (geom[k].in_max - geom[k].in_min) * sizeof(int16_t),
                                       cudaMemcpyHostToDevice, sl.compute));
                    ctx->timing.h2d_bytes += (geom[k].in_max - geom[k].in_min) * sizeof(int16_t);
                }
            }
            if (g == 0) { cudaEvent_t e1 = timing_event(sl); CU(cudaEventRecord(e1, sl.compute)); }

            VsRenderArgs ra;
            memset(&ra, 0, sizeof ra);
            ra.streams = (const VsStream *)sl.streams[cp].p;
            ra.chunks = (const VsChunk *)sl.chunks[cp].p;
            ra.order = (const uint32_t *)sl.order[cp].p + slab_r0[k];
            ra.n_rows = (uint32_t)(slab_r0[k + 1] - slab_r0[k]);
            memcpy(ra.cta_end, sl.plan_geom[k].cta_end, sizeof ra.cta_end);
            ra.table = sl.table[cp].p;
            ra.compact = compact;
            ra.n_periods = (const uint32_t *)sl.nper[cp].p;
            ra.rng_snap = any_noise ? (const uint32_t *)sl.snap[cp].p : nullptr;
            ra.costab = (const double *)sl.costab.p;
            ra.flow_in = d_in;
            ra.pcm_out = d_pcm;
            ra.raw_out = d_raw;
            ra.general_pulse = any_kvar ? 1 : 0;
            ra.debug = (uint32_t)ctx->opt_debug;
            ra.status = (int32_t *)sl.status[cp].p;
            /* shared-memory geometry.  The fast generator keeps, per lane, a ring of upcoming period entries (filled
             * one window ahead) and, per warp, the pulse tables of its rows; when the pitch periods of the batch are
             * too short or the tables too many for that, the general generator takes over. */
            const int win = vs_render_window(b.mode);
            const uint32_t tile_bytes = (uint32_t)vs_render_tiles(b.mode) * 32u * (uint32_t)win * 2u;
            int gen = VS_GEN_SIMPLE;
            ra.warp_bytes = tile_bytes;
            if (b.mode != VS_MODE_FILTER && compact != VS_TAB_FULL && amp_fits && !ctx->opt_simple_gen && t_min >= 24 && t_max <= 8192) {
                /* pitch periods a lane can enter in one window (+1: the generator may already have promoted the period
                 * that starts with the next window); the ring holds two windows' worth */
                const uint32_t per_win = (uint32_t)((win + t_min - 1) / t_min) + 1u;
                const uint32_t ahead = 2u * per_win + 2u;
                uint32_t R = 8;
                while (R < ahead) R <<= 1;
                /* the pulse-table cache: what the typical warp of this row order needs, as far as shared memory goes
                 * (a warp that needs more renders its rows with the general generator) */
                const uint32_t budget = (b.mode == VS_MODE_FLOW ? 100u : 200u) * 1024u / 4u;
                const uint32_t fixed = tile_bytes + R * 32u * VS_TAB_ENTRY_BYTES(compact);
                uint32_t cache = std::max(16u, (sl.plan_geom[k].cache_doubles + 1u) & ~1u);
                if (fixed + 4096u <= budget) cache = std::min(cache, ((budget - fixed) / 8u) & ~1u);
                const uint32_t wbytes = fixed + cache * 8u;
                if (R <= 64 && wbytes <= budget) {
                    gen = VS_GEN_FAST;
                    ra.warp_bytes = wbytes; ra.ring_R = R; ra.ring_fetch = per_win + 2u; ra.ring_ahead = ahead; ra.cache_doubles = cache;
                }
            }
            uint32_t render_sms = 1;
            {   /* persistent grid: one CTA per render SM (the plan kernels of the next calls own the others); the
                 * flow-only kernel is small, a few of its CTAs share an SM */
                const uint32_t blocks = (ra.n_rows / 32u + 3u) / 4u;
                const int plan_ctas = (int)((ns + (size_t)plan_nt - 1) / (size_t)plan_nt);
                const int reserve = vs_plan_reserve(plan_ctas);
                const uint32_t sms = (uint32_t)std::max(1, sl.sm_count - reserve);
                uint32_t per_sm = 1;
                if (b.mode == VS_MODE_FLOW) per_sm = std::max(1u, std::min(4u, (220u * 1024u) / (4u * ra.warp_bytes + (any_noise ? 16u * 1024u : 0u) + 1024u)));
                ra.grid = std::min(blocks, sms * per_sm);
                render_sms = sms;
            }
            const int filt = exact ? VS_FILT_EXACT : ((int_filter && !b.raw_out) ? VS_FILT_INT : VS_FILT_FMA);
            if (flow_rows) {
                if (!sl.ticket.p) {
                    if ((rc = dev_reserve(ctx, sl, sl.ticket, 256))) return rc;
                    CU(cudaMemsetAsync(sl.ticket.p, 0, 256, sl.compute));
                    sl.ticket_base = 0;
                }
                ra.ticket = (uint32_t *)sl.ticket.p;
                ra.ticket_base = sl.ticket_base;
                const uint32_t rows_per_cta = (uint32_t)vs_flow_rows_warps();
                ra.grid = std::max(1u, std::min((ra.n_rows + rows_per_cta - 1u) / rows_per_cta, render_sms * 4u));
                CU(vs_launch_flow_rows(ra, sl.compute));
                sl.ticket_base += ra.n_rows + ra.grid * rows_per_cta;       /* wraps like the device counter does */
            } else if (tracts) {
                VsTractBlock tb;                             /* copied into the launch's parameter space */
                memcpy(tb.cta_end, sl.plan_geom[k].cta_end, sizeof tb.cta_end);
                memset(tb.ncoef, 0, sizeof tb.ncoef);
                memcpy(tb.ncoef, ctx->in_ncoef.data(), ctx->in_ncoef.size() * sizeof(double));
                CU(vs_launch_render(ra, &tb, b.mode, gen, any_noise, filt, sl.compute));
            } else
                CU(vs_launch_render(ra, nullptr, b.mode, gen, any_noise, filt, sl.compute));
            ctx->timing.launches++;
            ctx->timing.render_path = (gen == VS_GEN_FAST || flow_rows ? 1u : 0u) | (any_noise ? 2u : 0u) | ((uint32_t)(b.raw_out && filt == VS_FILT_INT ? VS_FILT_FMA : filt) << 2) |
                                      (flow_rows ? 32u : 0u) | (tracts ? 64u : 0u);
            if (g == 0) { cudaEvent_t e2 = timing_event(sl); CU(cudaEventRecord(e2, sl.compute)); }

            if (!out_dev) {
                /* PCM home over PCIe on the copy stream while the next slab renders */
                CU(cudaEventRecord(sl.slab_ready, sl.compute));
                CU(cudaStreamWaitEvent(sl.copy, sl.slab_ready, 0));
                CU(cudaStreamWaitEvent(sl.copy2, sl.slab_ready, 0));
                /* merge rows that touch into runs: a dense batch is one copy per slab -- cut into 16 MB pieces that
                 * alternate between two copy streams, so that a second DMA engine keeps the link busy while the first
                 * one finishes a piece */
                uint64_t run_lo = hs[a0].out_off, run_hi = hs[a0].out_off + hs[a0].n;
                auto flush = [&](uint64_t lo, uint64_t hi) -> cudaError_t {
                    ctx->timing.d2h_bytes += (hi - lo) * (sizeof(int16_t) + (b.raw_out ? sizeof(double) : 0));
                    cudaError_t e = cudaSuccess;
                    const uint64_t piece = 8u << 20;                               /* samples */
                    unsigned which = 0;
                    for (uint64_t p0 = lo; p0 < hi && e == cudaSuccess; p0 += piece, which ^= 1u) {
                        const uint64_t p1 = std::min(hi, p0 + piece);
                        e = cudaMemcpyAsync(b.pcm_out + p0, d_pcm + (p0 - geom[k].out_min), (p1 - p0) * sizeof(int16_t),
                                            cudaMemcpyDeviceToHost, which ? sl.copy2 : sl.copy);
                    }
                    if (e == cudaSuccess && b.raw_out)
                        e = cudaMemcpyAsync(b.raw_out + lo, d_raw + (lo - geom[k].out_min), (hi - lo) * sizeof(double),
                                            cudaMemcpyDeviceToHost, sl.copy);
                    return e;
                };
                for (size_t i = a0 + 1; i < a1; i++) {
                    if (hs[i].out_off == run_hi) run_hi += hs[i].n;
                    else { CU(flush(run_lo, run_hi)); run_lo = hs[i].out_off; run_hi = run_lo + hs[i].n; }
                }
                CU(flush(run_lo, run_hi));
                CU(cudaEventRecord(sl.copy2_done, sl.copy2));
                CU(cudaStreamWaitEvent(sl.copy, sl.copy2_done, 0));
                CU(cudaEventRecord(sl.slab_done[d], sl.copy));
                sl.slab_done_valid[d] = true;
            }
        }
        if (want_log) ctx->timing.d2h_bytes += (log_hi - log_lo) * sizeof(vs_period_rec);
        if (want_log)
            CU(cudaMemcpyAsync(b.log->rec + log_lo, sl.log.p, (log_hi - log_lo) * sizeof(vs_period_rec), cudaMemcpyDeviceToHost, sl.compute));
        if (want_log && b.log->count)
            CU(cudaMemcpyAsync(sl.h_nper[cp].p, sl.nper[cp].p, ns * sizeof(uint32_t), cudaMemcpyDeviceToHost, sl.compute));
        if (!out_dev) sl.scratch_parity = (unsigned)((sl.scratch_parity + n_slabs) & 1);
        if (g == 0) { cudaEvent_t t_last = timing_event(sl); CU(cudaEventRecord(t_last, sl.compute)); }
        /* the device's error flag comes home on the copy stream: nothing sits between this call's render kernel and
         * the next call's on the compute stream */
        CU(cudaEventRecord(sl.render_done[cp], sl.compute));
        CU(cudaStreamWaitEvent(sl.copy, sl.render_done[cp], 0));
        CU(cudaMemcpyAsync(sl.h_status[cp].p, sl.status[cp].p, sizeof(int32_t), cudaMemcpyDeviceToHost, sl.copy));
        CU(cudaEventRecord(sl.call_done[cp], sl.copy));               /* parity-cp buffers are free once this fires */
    }

    prof.mark("launches enqueued");
    /* ---- 5. host buffers: the call returns when the data has landed -------------------------- */
    const bool may_return_early = ctx->opt_async_host && out_kind == PK_HOST_PINNED && !want_log &&
                                  (!b.raw_out || raw_kind == PK_HOST_PINNED) && (!b.flow_in || in_kind == PK_HOST_PINNED);
    if ((!out_dev && !may_return_early) || want_log) {
        const int rc = vs_sync(ctx);
        if (rc) return rc;
        prof.mark("sync (data landed)");
        if (want_log && b.log->count) {
            for (size_t g = 0; g < nslots; g++) {
                const size_t s0 = cut[g], s1 = cut[g + 1];
                if (s1 > s0) memcpy(b.log->count + s0, ctx->slots[g].h_nper[(ctx->slots[g].call_parity + VS_DEPTH - 1u) % VS_DEPTH].p, (s1 - s0) * sizeof(uint32_t));
            }
        }
    }
    return VS_OK;
}

} // namespace

/* ================================================================================================
 * exported C ABI
 * ============================================================================================== */
extern "C" {

int vs_abi_version(void) { return VS_ABI_VERSION; }

int vs_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

const char *vs_strerror(int code)
{
    switch (code) {
    case VS_OK: return "ok";
    case VS_EINVAL: return "invalid argument";
    case VS_ERANGE: return "stream parameter out of range";
    case VS_EPRESET: return "unknown vowel preset";
    case VS_ENOMEM: return "out of memory";
    case VS_ECUDA: return "CUDA error";
    case VS_ENODEV: return "no usable sm_100 device";
    case VS_EOVERLAP: return "bad output layout";
    default: return "unknown error";
    }
}

const char *vs_last_error(vs_ctx *ctx) { return ctx ? ctx->err.c_str() : ""; }

int vs_ctx_create(vs_ctx **out, const int *devices, int n_devices, uint32_t flags)
{
    (void)flags;
    if (!out) return VS_EINVAL;
    *out = nullptr;
    DeviceGuard restore_device;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) { cudaGetLastError(); return VS_ENODEV; }
    std::vector<int> devs;
    if (!devices || n_devices <= 0) devs.push_back(0);
    else devs.assign(devices, devices + n_devices);
    vs_ctx *ctx = new (std::nothrow) vs_ctx();
    if (!ctx) return VS_ENOMEM;
    ctx->env_profile_host = getenv("VS_PROFILE_HOST") != nullptr;     /* debugging aids, read once */
    ctx->env_sync_plan = getenv("VS_DEBUG_SYNCPLAN") != nullptr;
    compute_warmups(ctx);
    for (int d : devs) {
        if (d < 0 || d >= count) { vs_ctx_destroy(ctx); return VS_ENODEV; }
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, d) != cudaSuccess || prop.major != 10) {
            /* the only code in the library is sm_100a SASS: anything else cannot run it */
            cudaGetLastError();
            vs_ctx_destroy(ctx);
            return VS_ENODEV;
        }
        Slot s;
        s.dev = d;
        s.sm_count = prop.multiProcessorCount;
        bool ok = cudaSetDevice(d) == cudaSuccess &&
                  cudaStreamCreateWithFlags(&s.compute, cudaStreamNonBlocking) == cudaSuccess &&
                  cudaStreamCreateWithFlags(&s.copy, cudaStreamNonBlocking) == cudaSuccess &&
                  cudaStreamCreateWithFlags(&s.copy2, cudaStreamNonBlocking) == cudaSuccess &&
                  cudaEventCreateWithFlags(&s.copy2_done, cudaEventDisableTiming) == cudaSuccess &&
                  cudaStreamCreateWithFlags(&s.plans[0], cudaStreamNonBlocking) == cudaSuccess &&
                  cudaStreamCreateWithFlags(&s.plans[1], cudaStreamNonBlocking) == cudaSuccess &&

                  cudaEventCreateWithFlags(&s.slab_done[0], cudaEventDisableTiming) == cudaSuccess &&
                  cudaEventCreateWithFlags(&s.slab_done[1], cudaEventDisableTiming) == cudaSuccess &&
                  cudaEventCreateWithFlags(&s.slab_ready, cudaEventDisableTiming) == cudaSuccess &&
                  vs_render_init_device() == cudaSuccess &&
                  true;
        for (int k = 0; ok && k < VS_DEPTH; k++)
            ok = cudaEventCreateWithFlags(&s.call_done[k], cudaEventDisableTiming) == cudaSuccess &&
                 cudaEventCreateWithFlags(&s.render_done[k], cudaEventDisableTiming) == cudaSuccess &&
                 cudaEventCreateWithFlags(&s.plan_done[k], cudaEventDisableTiming) == cudaSuccess;
        ctx->slots.push_back(s);
        if (!ok) { cudaGetLastError(); vs_ctx_destroy(ctx); return VS_ECUDA; }
    }
    *out = ctx;
    return VS_OK;
}

void vs_ctx_destroy(vs_ctx *ctx)
{
    if (!ctx) return;
    DeviceGuard restore_device;
    for (Slot &s : ctx->slots) {
        cudaSetDevice(s.dev);
        if (s.compute) cudaStreamSynchronize(s.compute);
        if (s.copy2) cudaStreamSynchronize(s.copy2);
        if (s.copy) cudaStreamSynchronize(s.copy);
        for (int k = 0; k < 2; k++) if (s.plans[k]) cudaStreamSynchronize(s.plans[k]);
        std::vector<DevBuf *> bufs = {&s.costab, &s.pcm[0], &s.pcm[1], &s.raw[0], &s.raw[1], &s.flowin[0], &s.flowin[1], &s.log, &s.ticket, &s.analyze};
        std::vector<PinBuf *> pins;
        for (int k = 0; k < VS_DEPTH; k++) {
            for (DevBuf *b : {&s.streams[k], &s.chunks[k], &s.order[k], &s.table[k], &s.snap[k], &s.nper[k], &s.status[k]}) bufs.push_back(b);
            for (PinBuf *b : {&s.h_streams[k], &s.h_chunks[k], &s.h_order[k], &s.h_nper[k], &s.h_status[k]}) pins.push_back(b);
        }
        for (DevBuf *b : bufs) if (b->p) cudaFree(b->p);
        for (PinBuf *b : pins) if (b->p) cudaFreeHost(b->p);
        for (cudaEvent_t e : s.tev) cudaEventDestroy(e);
        for (int k = 0; k < VS_DEPTH; k++) {
            if (s.call_done[k]) cudaEventDestroy(s.call_done[k]);
            if (s.plan_done[k]) cudaEventDestroy(s.plan_done[k]);
            if (s.render_done[k]) cudaEventDestroy(s.render_done[k]);
        }
        for (int k = 0; k < 2; k++) if (s.plans[k]) cudaStreamDestroy(s.plans[k]);
        if (s.slab_done[0]) cudaEventDestroy(s.slab_done[0]);
        if (s.slab_done[1]) cudaEventDestroy(s.slab_done[1]);
        if (s.slab_ready) cudaEventDestroy(s.slab_ready);
        if (s.copy2_done) cudaEventDestroy(s.copy2_done);
        if (s.copy2) cudaStreamDestroy(s.copy2);
        if (s.copy) cudaStreamDestroy(s.copy);
        if (s.compute && s.own_compute) cudaStreamDestroy(s.compute);
    }
    cudaGetLastError();
    delete ctx;
}

int vs_ctx_set_option(vs_ctx *ctx, int option, double value)
{
    if (!ctx) return VS_EINVAL;
    switch (option) {
    case VS_OPT_CHUNK_SAMPLES: ctx->opt_chunk = value; return VS_OK;
    case VS_OPT_CARRY_TOL:
        if (!(value > 0.0 && value < 1.0)) return VS_EINVAL;
        ctx->opt_tol = value; compute_warmups(ctx); ctx->tract_warm.clear(); return VS_OK;
    case VS_OPT_EXACT_FILTER: ctx->opt_exact = value != 0.0; return VS_OK;
    case VS_OPT_SLAB_STREAMS: ctx->opt_slab = value > 0 ? (int)value : 0; return VS_OK;
    case VS_OPT_TARGET_WARPS: if (!(value > 0)) return VS_EINVAL; ctx->opt_warps = value; return VS_OK;
    case VS_OPT_ASYNC_HOST: ctx->opt_async_host = value != 0.0; return VS_OK;
    case VS_OPT_PLAN_WARPS: ctx->opt_plan_warps = value < 0 ? -1 : (value != 0.0); return VS_OK;
    case VS_OPT_SIMPLE_GEN: ctx->opt_simple_gen = value != 0.0; return VS_OK;
    case 100: ctx->opt_debug = (int)value; return VS_OK;             /* undocumented: timing experiments */
    default: return VS_EINVAL;
    }
}

int vs_ctx_set_stream(vs_ctx *ctx, int slot, void *cuda_stream)
{
    if (!ctx || slot < 0 || (size_t)slot >= ctx->slots.size()) return VS_EINVAL;
    Slot &s = ctx->slots[slot];
    DeviceGuard restore_device;
    CU(cudaSetDevice(s.dev));
    CU(cudaStreamSynchronize(s.compute));
    if (s.own_compute) CU(cudaStreamDestroy(s.compute));
    s.compute = (cudaStream_t)cuda_stream;
    s.own_compute = false;
    return VS_OK;
}

int vs_sync(vs_ctx *ctx)
{
    if (!ctx) return VS_EINVAL;
    DeviceGuard restore_device;
    int status = 0;
    for (Slot &s : ctx->slots) {
        CU(cudaSetDevice(s.dev));
        CU(cudaStreamSynchronize(s.plans[0]));
        CU(cudaStreamSynchronize(s.plans[1]));
        CU(cudaStreamSynchronize(s.compute));
        CU(cudaStreamSynchronize(s.copy2));
        CU(cudaStreamSynchronize(s.copy));
        s.last_enqueue = {};                                  /* the device is idle: the next call may take the latency form of the plan kernel */
        for (int k = 0; k < VS_DEPTH; k++)
            if (s.h_status[k].p && *(int32_t *)s.h_status[k].p) { status = *(int32_t *)s.h_status[k].p; *(int32_t *)s.h_status[k].p = 0; }
    }
    if (ctx->timing_pending) {
        Slot &s = ctx->slots[0];
        ctx->timing_pending = false;
        if (s.tev_used >= 3) {
            /* layout: t_first, t_plan (plan stream), then (e1,e2) per slab, then t_last (compute stream) */
            float ms = 0.0f;
            if (cudaEventElapsedTime(&ms, s.tev[0], s.tev[1]) == cudaSuccess) ctx->timing.plan_ms = ms;
            for (size_t k = 2; k + 1 < s.tev_used - 1; k += 2)
                if (cudaEventElapsedTime(&ms, s.tev[k], s.tev[k + 1]) == cudaSuccess) ctx->timing.render_ms += ms;
            if (cudaEventElapsedTime(&ms, s.tev[0], s.tev[s.tev_used - 1]) == cudaSuccess) ctx->timing.total_ms = ms;
            cudaGetLastError();
        }
    }
    if (status) return fail(ctx, status, "a device kernel reported: %s", vs_strerror(status));
    return VS_OK;
}

int vs_get_timing(vs_ctx *ctx, vs_timing *out)
{
    if (!ctx || !out) return VS_EINVAL;
    const int rc = vs_sync(ctx);
    *out = ctx->timing;
    return rc;
}

void *vs_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void vs_host_free(void *p) { if (p) cudaFreeHost(p); }

int vs_measure_fp64_peak(vs_ctx *ctx, double *tflops_out, double *sm_mhz_out)
{
    if (!ctx || !tflops_out) return VS_EINVAL;
    DeviceGuard restore_device;
    Slot &s = ctx->slots[0];
    CU(cudaSetDevice(s.dev));
    const int blocks = s.sm_count * 8, iters = 1 << 16;
    double *scratch = nullptr;
    CU(cudaMalloc(&scratch, (size_t)blocks * 256 * sizeof(double)));
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0));
    CU(cudaEventCreate(&e1));
    float best = 1e30f;
    for (int rep = 0; rep < 4; rep++) {
        CU(cudaEventRecord(e0, s.compute));
        CU(vs_launch_fp64_peak(scratch, blocks, iters, s.compute));
        CU(cudaEventRecord(e1, s.compute));
        CU(cudaEventSynchronize(e1));
        float ms = 0.0f;
        CU(cudaEventElapsedTime(&ms, e0, e1));
        if (rep > 0 && ms < best) best = ms;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(scratch);
    const double fma = (double)blocks * 256.0 * 8.0 * (double)iters;
    *tflops_out = 2.0 * fma / ((double)best * 1e-3) / 1e12;
    if (sm_mhz_out) *sm_mhz_out = fma / ((double)best * 1e-3) / ((double)s.sm_count * 64.0) / 1e6;  /* if 64 DFMA/clk/SM */
    return VS_OK;
}

int vs_flow_nsamples(const vs_flow_params *p, size_t n, uint64_t *out)
{
    if (!out) return VS_EINVAL;
    for (size_t i = 0; i < n; i++) out[i] = row_nsamples(flow_row(p, i));
    return VS_OK;
}

int vs_flow_max_periods(const vs_flow_params *p, size_t n, uint64_t *out)
{
    if (!out) return VS_EINVAL;
    for (size_t i = 0; i < n; i++) {
        const FlowRow r = flow_row(p, i);
        if (row_validate(r)) { out[i] = 0; continue; }
        out[i] = row_max_periods(r, row_nsamples(r), row_P(r));
    }
    return VS_OK;
}

int vs_flow_validate(const vs_flow_params *p, size_t n, size_t *bad)
{
    for (size_t i = 0; i < n; i++) {
        const int rc = row_validate(flow_row(p, i));
        if (rc) { if (bad) *bad = i; return rc; }
    }
    return VS_OK;
}

int vs_filter_warmup(vs_ctx *ctx, int preset_key, float gain)
{
    (void)gain;
    if (!ctx) return VS_EINVAL;
    const int k = preset_index(preset_key);
    return k < 0 ? VS_EPRESET : ctx->warm[k];
}

int vs_flowgen_batch(vs_ctx *ctx, const vs_flow_params *p, size_t n, int16_t *pcm_out, const uint64_t *offsets, vs_period_log *log)
{
    Batch b = {VS_MODE_FLOW, n, p, nullptr, nullptr, nullptr, nullptr, nullptr, pcm_out, offsets, nullptr, log};
    return run_batch(ctx, b);
}

int vs_vowel_filter_batch(vs_ctx *ctx, const int16_t *flow_in, const uint64_t *in_offsets, const uint64_t *nsamp,
                          const vs_filter_params *f, size_t n, int16_t *pcm_out, const uint64_t *out_offsets, double *raw_out)
{
    Batch b = {VS_MODE_FILTER, n, nullptr, f, nullptr, flow_in, in_offsets, nsamp, pcm_out, out_offsets, raw_out, nullptr};
    return run_batch(ctx, b);
}

int vs_vowel_filter_batch_tract(vs_ctx *ctx, const int16_t *flow_in, const uint64_t *in_offsets, const uint64_t *nsamp,
                                const vs_tract_params *t, size_t n, int16_t *pcm_out, const uint64_t *out_offsets, double *raw_out)
{
    if (!t) return fail(ctx, VS_EINVAL, "tract params are NULL");
    Batch b = {VS_MODE_FILTER, n, nullptr, nullptr, t, flow_in, in_offsets, nsamp, pcm_out, out_offsets, raw_out, nullptr};
    return run_batch(ctx, b);
}

int vs_vowel_noise_batch(vs_ctx *ctx, int16_t *pcm, const uint64_t *offsets, const uint64_t *nsamp, const float *snr,
                         const int32_t *fs, const uint32_t *seed, size_t n)
{
    if (!ctx || !pcm || !nsamp || !snr) return VS_EINVAL;
    if (n == 0) return VS_OK;
    if (n > 0x7fffffffull) return fail(ctx, VS_EINVAL, "too many streams");
    int rc = vs_sync(ctx);                                    /* in-place: earlier work on this PCM must have landed */
    if (rc) return rc;
    DeviceGuard restore_device;
    Slot &sl = ctx->slots[0];                                 /* one warp per stream and 0.75 ms for 4096 x 1 s: one device is plenty */
    CU(cudaSetDevice(sl.dev));
    std::vector<VsNoiseRow> rows(n);
    uint64_t max_n = 0, lo = ~0ull, hi = 0;
    for (size_t i = 0; i < n; i++) max_n = std::max(max_n, nsamp[i]);
    for (size_t i = 0; i < n; i++) {
        if (nsamp[i] > 0x7fffffffull) return fail(ctx, VS_EOVERLAP, "stream %zu: too many samples", i);
        const int32_t rate = fs ? fs[i] : 22050;
        if (rate <= 0) return fail(ctx, VS_ERANGE, "stream %zu: sampling rate", i);
        const int ms1 = (int)((uint32_t)rate * 0.001 / 2.0) * 2;       /* vowel_new.c:361 */
        const long frame = 50L * ms1;                                  /* :363 */
        if (snr[i] > 0.0f && (frame <= 0 || frame > 32767)) return fail(ctx, VS_ERANGE, "stream %zu: frame length %ld", i, frame);
        rows[i].off = offsets ? offsets[i] : (uint64_t)i * max_n;
        rows[i].n = (uint32_t)nsamp[i];
        rows[i].frame = (uint32_t)frame;
        rows[i].snr = snr[i];
        rows[i].seed = seed ? seed[i] : 1u;
        lo = std::min(lo, rows[i].off);
        hi = std::max(hi, rows[i].off + rows[i].n);
    }
    int dev = -1;
    const bool on_dev = classify(pcm, &dev) == PK_DEVICE;
    if (on_dev && dev != sl.dev) return fail(ctx, VS_EINVAL, "device buffer lives on device %d, ctx on %d", dev, sl.dev);
    if ((rc = dev_reserve(ctx, sl, sl.log, n * sizeof(VsNoiseRow)))) return rc;          /* the log scratch doubles as row storage */
    CU(cudaMemcpyAsync(sl.log.p, rows.data(), n * sizeof(VsNoiseRow), cudaMemcpyHostToDevice, sl.compute));
    int16_t *d_pcm = pcm;
    if (!on_dev) {
        if ((rc = dev_reserve(ctx, sl, sl.pcm[0], (hi - lo) * sizeof(int16_t) + 64))) return rc;
        d_pcm = (int16_t *)sl.pcm[0].p - lo;
        CU(cudaMemcpyAsync(sl.pcm[0].p, pcm + lo, (hi - lo) * sizeof(int16_t), cudaMemcpyHostToDevice, sl.compute));
    }
    CU(vs_launch_vnoise(d_pcm, (const VsNoiseRow *)sl.log.p, (uint32_t)n, sl.compute));
    if (!on_dev) {
        /* only the rows come back (gaps between them are not ours); rows that touch travel as one copy */
        uint64_t run_lo = 0, run_hi = 0;
        for (size_t i = 0; i <= n; i++) {
            const bool take = i < n && rows[i].n && rows[i].snr > 0.0f;
            if (take && run_hi > run_lo && rows[i].off == run_hi) { run_hi += rows[i].n; continue; }
            if (run_hi > run_lo)
                CU(cudaMemcpyAsync(pcm + run_lo, d_pcm + run_lo, (run_hi - run_lo) * sizeof(int16_t), cudaMemcpyDeviceToHost, sl.compute));
            run_lo = take ? rows[i].off : 0;
            run_hi = take ? rows[i].off + rows[i].n : 0;
        }
    }
    CU(cudaStreamSynchronize(sl.compute));                    /* `rows` is pageable host memory */
    return VS_OK;
}

int vs_flow_analyze_batch(vs_ctx *ctx, const int16_t *flow, const uint64_t *offsets, const uint64_t *nsamp, const int32_t *fs,
                          const int16_t *lo, const int16_t *hi, size_t n, vs_flow_stats *stats)
{
    if (!ctx || !flow || !nsamp || !stats) return VS_EINVAL;
    if (n == 0) return VS_OK;
    if (n > 0x7fffffffull) return fail(ctx, VS_EINVAL, "too many streams");
    int rc = vs_sync(ctx);                                    /* the flow may be the output of a call still in flight */
    if (rc) return rc;
    DeviceGuard restore_device;
    Slot &sl = ctx->slots[0];
    CU(cudaSetDevice(sl.dev));
    std::vector<VsAnalyzeRow> rows(n);
    uint64_t max_n = 0, first = ~0ull, last = 0, slots = 0;
    for (size_t i = 0; i < n; i++) max_n = std::max(max_n, nsamp[i]);
    for (size_t i = 0; i < n; i++) {
        if (nsamp[i] > 0x7fffffffull) return fail(ctx, VS_EOVERLAP, "stream %zu: too many samples", i);
        const int32_t rate = fs ? fs[i] : 22050;
        if (rate <= 0) return fail(ctx, VS_ERANGE, "stream %zu: sampling rate", i);
        const int16_t tl = lo ? lo[i] : (int16_t)0, th = hi ? hi[i] : (int16_t)0;
        if (tl > th) return fail(ctx, VS_ERANGE, "stream %zu: thresholds lo > hi", i);
        VsAnalyzeRow &r = rows[i];
        r.off = offsets ? offsets[i] : (uint64_t)i * max_n;
        r.n = (uint32_t)nsamp[i];
        r.cap = r.n / 16u + 4u;
        r.ons_off = slots;
        r.fs = rate; r.lo = tl; r.hi = th;
        slots += r.cap;
        first = std::min(first, r.off);
        last = std::max(last, r.off + r.n);
    }
    int dev = -1;
    const bool on_dev = classify(flow, &dev) == PK_DEVICE;
    if (on_dev && dev != sl.dev) return fail(ctx, VS_EINVAL, "device buffer lives on device %d, ctx on %d", dev, sl.dev);
    /* scratch: rows | per-stream onset counts | stats | onset lists */
    const size_t rows_b = (n * sizeof(VsAnalyzeRow) + 255) & ~(size_t)255, cnt_b = (n * sizeof(uint32_t) + 255) & ~(size_t)255;
    const size_t st_b = (n * sizeof(vs_flow_stats) + 255) & ~(size_t)255;
    if ((rc = dev_reserve(ctx, sl, sl.analyze, rows_b + cnt_b + st_b + slots * sizeof(uint32_t)))) return rc;
    unsigned char *base = (unsigned char *)sl.analyze.p;
    CU(cudaMemcpyAsync(base, rows.data(), n * sizeof(VsAnalyzeRow), cudaMemcpyHostToDevice, sl.compute));
    const int16_t *d_flow = flow;
    if (!on_dev) {
        if ((rc = dev_reserve(ctx, sl, sl.pcm[0], (last - first) * sizeof(int16_t) + 256))) return rc;
        d_flow = (const int16_t *)sl.pcm[0].p - first;
        CU(cudaMemcpyAsync(sl.pcm[0].p, flow + first, (last - first) * sizeof(int16_t), cudaMemcpyHostToDevice, sl.compute));
    }
    CU(vs_launch_analyze(d_flow, (const VsAnalyzeRow *)base, (uint32_t)n, (uint32_t *)(base + rows_b + cnt_b + st_b),
                         (uint32_t *)(base + rows_b), (vs_flow_stats *)(base + rows_b + cnt_b), sl.compute));
    CU(cudaMemcpyAsync(stats, base + rows_b + cnt_b, n * sizeof(vs_flow_stats), cudaMemcpyDeviceToHost, sl.compute));
    CU(cudaStreamSynchronize(sl.compute));                    /* `rows` and `stats` are the caller's / pageable memory */
    return VS_OK;
}

int vs_synth_batch(vs_ctx *ctx, const vs_flow_params *p, const vs_filter_params *f, size_t n, int16_t *pcm_out,
                   const uint64_t *offsets, double *raw_out)
{
    Batch b = {VS_MODE_SYNTH, n, p, f, nullptr, nullptr, nullptr, nullptr, pcm_out, offsets, raw_out, nullptr};
    return run_batch(ctx, b);
}

int vs_synth_batch_tract(vs_ctx *ctx, const vs_flow_params *p, const vs_tract_params *t, size_t n, int16_t *pcm_out,
                         const uint64_t *offsets, double *raw_out)
{
    if (!t) return fail(ctx, VS_EINVAL, "tract params are NULL");
    Batch b = {VS_MODE_SYNTH, n, p, nullptr, t, nullptr, nullptr, nullptr, pcm_out, offsets, raw_out, nullptr};
    return run_batch(ctx, b);
}

int vs_tract_from_formants(const float *freq_hz, const float *bw_hz, int n_formants, int32_t fs, double den[23])
{
    if (!freq_hz || !bw_hz || !den || n_formants < 1 || 2 * n_formants > VS_ORDER) return VS_EINVAL;
    if (fs <= 0) return VS_ERANGE;
    const double pi = 3.14159265358979323846, rate = (double)fs;
    for (int k = 0; k < n_formants; k++) {
        const double F = freq_hz[k], B = bw_hz[k];
        if (!(F > 0.0 && F < 0.5 * rate) || !(B > 0.0) || !std::isfinite(B)) return VS_ERANGE;
    }
    double d[VS_ORDER + 1] = {1.0};
    for (int k = 0; k < n_formants; k++) {
        const double r = std::exp(-pi * (double)bw_hz[k] / rate), th = 2.0 * pi * (double)freq_hz[k] / rate;
        const double b1 = -2.0 * r * std::cos(th), b2 = r * r;
        for (int j = 2 * k + 2; j >= 1; j--) {         /* d <- d * (1 + b1 z^-1 + b2 z^-2), in place from the top */
            double v = d[j] + b1 * d[j - 1];
            if (j >= 2) v += b2 * d[j - 2];
            d[j] = v;
        }
    }
    memcpy(den, d, sizeof d);
    return VS_OK;
}

int vs_tract_from_preset(int preset_key, double den[23])
{
    const int k = preset_index(preset_key);
    if (k < 0) return VS_EPRESET;
    if (!den) return VS_EINVAL;
    memcpy(den, vs_preset_den[k], (VS_ORDER + 1) * sizeof(double));
    return VS_OK;
}

} /* extern "C" */
