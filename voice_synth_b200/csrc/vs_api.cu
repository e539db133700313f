/* vs_api.cu -- host side of libvoicesynth_cuda: contexts, device slots and their buffers, the caches that let a repeated
 * call skip work, uploads, launches and PCIe copies.  What a batch call computes is the planner's (vs_batch_plan.cpp). */
#include <cuda_runtime.h>

#include <algorithm>
#include <array>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <string>
#include <vector>

#include "vs_batch_plan.h"

cudaError_t vs_launch_plan(const VsPlanArgs &a, const VsShape &sh, bool warps, cudaStream_t s);
cudaError_t vs_launch_render(const VsRenderArgs &a, const VsTractBlock *tb, const VsShape &sh, int gen, cudaStream_t s);
static_assert(VS_MAX_TRACTS == VS_MAX_TRACTS_I, "tract count");
static_assert(VS_MAX_TRACTS <= 256, "a stream's tract index is a uint8_t");
cudaError_t vs_render_init_device();
cudaError_t vs_launch_flow_rows(const VsRenderArgs &a, cudaStream_t s);
cudaError_t vs_launch_fp64_peak(double *scratch, int blocks, int iters, cudaStream_t s);
cudaError_t vs_launch_vnoise(int16_t *pcm, const VsNoiseRow *rows, uint32_t n_rows, cudaStream_t s);
cudaError_t vs_launch_analyze(const int16_t *flow, const VsAnalyzeRow *rows, uint32_t n_rows, uint32_t *onsets, uint32_t *counts,
                              vs_flow_stats *out, cudaStream_t s);
cudaError_t vs_launch_report(const int16_t *flow, const VsAnalyzeRow *rows, uint32_t n_rows, uint32_t *onsets, uint32_t *counts,
                             vs_flow_stats *stats, int32_t *peaks, vs_flow_report *out, cudaStream_t s);
cudaError_t vs_launch_formants(const VsFormantArgs &a, vs_formant_stats *stats, vs_formant_frame *frames, cudaStream_t s);

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
    VsPlan plan;
    uint64_t plan_version = 1, uploaded_version[VS_DEPTH] = {};        /* which plan the device copies of chunks/order hold (0 = none) */
    std::chrono::steady_clock::time_point last_enqueue{};
    uint64_t plan_for_version = 0;                   /* vs_ctx::in_version of the inputs the plan was made (or confirmed) for */
    uint64_t streams_version[VS_DEPTH] = {};         /* which inputs the device copies of the stream descriptors hold          */
    std::array<cudaStream_t, 5> all_streams() const { return {plans[0], plans[1], compute, copy2, copy}; }
    std::vector<cudaEvent_t *> events()              /* the events the slot owns (not the timing events) */
    {
        std::vector<cudaEvent_t *> e = {&copy2_done, &slab_done[0], &slab_done[1], &slab_ready};
        for (int k = 0; k < VS_DEPTH; k++) e.insert(e.end(), {&call_done[k], &plan_done[k], &render_done[k]});
        return e;
    }
};

} // namespace

struct vs_ctx {
    std::vector<Slot> slots;
    VsPlanOptions opt;           /* opt.tol = 1e-12: x |state| <= ~2e5 at the default gain: 2e-7 before quantisation, 50 x under the 1e-5 bar */
    int opt_plan_warps = -1;     /* -1 auto, 0 one thread per stream, 1 one warp per stream */
    int opt_async_host = 0;
    int opt_debug = 0;
    VsTables tables;
    std::string err;
    vs_timing timing;
    bool timing_pending = false;
    /* the previous call's inputs, byte for byte, and everything derived from them on the host: a call with the same
     * parameters (a corpus generator re-running a shape, the benchmark loop) skips validation, descriptor
     * building, chunk planning and the descriptor upload */
    std::vector<unsigned char> in_blob;
    VsDescriptors in;
    uint64_t in_version = 0;     /* bumped whenever in.hs changes */
    bool env_profile_host = false, env_sync_plan = false;
};

namespace {

/* the ABI has no globals: a call leaves the caller's current device as it found it */
struct DeviceGuard {
    int prev = -1;
    DeviceGuard() { if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; cudaGetLastError(); } }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

#define fail(c, ...) vs_error((c) ? &(c)->err : nullptr, __VA_ARGS__)

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(ctx, VS_ECUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

/* wait until all five streams of the slot are idle (a null compute stream is the caller's legacy default stream) */
int drain(vs_ctx *ctx, Slot &s)
{
    for (cudaStream_t st : s.all_streams()) CU(cudaStreamSynchronize(st));
    return VS_OK;
}

int dev_reserve(vs_ctx *ctx, Slot &s, DevBuf &b, size_t bytes)
{
    if (bytes <= b.cap) return VS_OK;
    if (b.p) {
        const int rc = drain(ctx, s);
        if (rc) return rc;
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
void snapshot_inputs(const VsBatch &b, bool want_log, const void *extra, size_t extra_bytes, std::vector<unsigned char> &blob)
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

/* one batch call, as the launch code of a slot sees it */
struct Call {
    const VsBatch &b;
    bool want_log, same_inputs, out_dev;
    VsShape sh;
    uint64_t out_base;           /* the sample address of out_off 0: device output; 0 for host output (mirrored 64-aligned) */
    HostProf &prof;
};

/* host address range of a slab's rows, and of its input rows (filter mode) */
struct SlabSpan { uint64_t out_min, out_max, in_min, in_max; };

/* Stage 4 of a slot: chunk plan + row order.  A function of the batch SHAPE only (lengths, groups, row phases, tables,
 * options), so a call shaped like the previous one reuses it. */
void slot_plan(vs_ctx *ctx, Slot &sl, const Call &c, size_t s0, size_t s1, const std::vector<VsRange> &slabs, size_t slab_streams)
{
    const std::vector<VsStream> &hs = ctx->in.hs;
    std::vector<uint64_t> sig;
    const bool known_plan = c.same_inputs && sl.plan_for_version == ctx->in_version;     /* same bytes as the call that made the plan */
    if (!known_plan) {
        const VsPlanOptions &o = ctx->opt;
        sig.reserve(3 * (s1 - s0) + 8);
        sig.push_back(((uint64_t)c.b.mode << 48) ^ ((uint64_t)slabs.size() << 24) ^ (uint64_t)slab_streams ^ ((uint64_t)c.sh.plan_nt << 52));
        sig.push_back((uint64_t)(int64_t)o.chunk ^ ((uint64_t)o.exact << 62) ^ ((uint64_t)sl.sm_count << 40));
        { uint64_t u; memcpy(&u, &o.tol, 8); sig.push_back(u); }
        sig.push_back((uint64_t)c.sh.tracts);
        if (c.sh.tracts) for (int w : ctx->in.warm) sig.push_back((uint64_t)w);   /* the chunk plan depends on the tracts' warm-ups */
        for (size_t i = s0; i < s1; i++) {
            sig.push_back((uint64_t)hs[i].n | ((uint64_t)hs[i].preset << 32) | (((c.out_base + hs[i].out_off) & c.sh.ph_mask) << 40));
            sig.push_back((uint64_t)hs[i].tab_cap | ((uint64_t)hs[i].pulse_off << 32));          /* row order and table cache depend on these */
            sig.push_back((uint64_t)(uint32_t)hs[i].T2 | ((uint64_t)hs[i].tpad << 32));
        }
    }
    const bool plan_hit = known_plan || sig == sl.plan_sig;
    sl.plan_for_version = ctx->in_version;
    if (plan_hit) return;
    vs_plan_chunks(ctx->opt, c.sh, sl.sm_count, hs, s0, s1, slabs, ctx->in.warm.data(), c.out_base, sl.plan);
    c.prof.mark("chunk plan");
    vs_plan_rows(c.sh, hs, s0, sl.plan);
    sl.plan_sig.swap(sig);
    sl.plan_version++;
    c.prof.mark("row order");
}

/* Device and staging memory of a call on ring slot cp, and the cosine tables.  The descriptor / table buffers form a
 * ring of VS_DEPTH sets.  When one of them has to grow, the same buffer of every set grows with it: a new batch shape
 * pays for its memory in its FIRST call (growing means a device-wide synchronisation, cudaFree / cudaMalloc /
 * cudaHostAlloc), not in each of its first VS_DEPTH calls. */
int slot_reserve(vs_ctx *ctx, Slot &sl, const Call &c, unsigned cp, size_t ns, cudaStream_t pstream)
{
    const size_t nc = sl.plan.chunks.size(), nrows = sl.plan.order.size();
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
        const int r0 = drain(ctx, sl);                            /* copies of the calls in flight read from these */
        if (r0) return r0;
        for (unsigned d = 0; d < VS_DEPTH; d++) {
            const int r = pin_reserve(ctx, ring[d], bytes);
            if (r) return r;
        }
        return VS_OK;
    };
    int rc;
    if ((rc = ring_dev(sl.streams, ns * sizeof(VsStream)))) return rc;
    if ((rc = ring_dev(sl.chunks, nc * sizeof(VsChunk)))) return rc;
    if ((rc = ring_dev(sl.order, nrows * sizeof(uint32_t) + 16))) return rc;
    if ((rc = ring_dev(sl.nper, ns * sizeof(uint32_t)))) return rc;
    if ((rc = ring_dev(sl.status, sizeof(int32_t)))) return rc;
    if (c.b.mode != VS_MODE_FILTER) {
        const std::vector<double> &cos_host = ctx->tables.cos_host;
        if ((rc = ring_dev(sl.table, (sl.plan.tab_total + 8) * VS_TAB_ENTRY_BYTES(c.sh.compact)))) return rc;
        if (c.sh.noise && (rc = ring_dev(sl.snap, nc * 32 * sizeof(uint32_t)))) return rc;
        if ((rc = dev_reserve(ctx, sl, sl.costab, (cos_host.size() + VS_COS_SLACK) * sizeof(double)))) return rc;
        if (sl.costab_uploaded != cos_host.size()) {
            /* tables only ever grow; a synchronous copy keeps the host vector free to grow again */
            /* stream-ordered on the plan stream (a plain cudaMemcpy from pageable memory may still be in
             * flight when it returns, and non-blocking streams do not order after the legacy stream).  The copies
             * of the calls in flight need not finish: they do not read the tables. */
            CU(cudaStreamSynchronize(sl.compute));
            CU(cudaStreamSynchronize(sl.plans[0]));
            CU(cudaStreamSynchronize(sl.plans[1]));
            CU(cudaMemcpyAsync(sl.costab.p, cos_host.data(), cos_host.size() * sizeof(double), cudaMemcpyHostToDevice, pstream));
            CU(cudaStreamSynchronize(pstream));
            ctx->timing.h2d_bytes += cos_host.size() * sizeof(double);
            sl.costab_uploaded = cos_host.size();
        }
    }
    if ((rc = ring_pin(sl.h_streams, ns * sizeof(VsStream)))) return rc;
    if ((rc = ring_pin(sl.h_chunks, nc * sizeof(VsChunk)))) return rc;
    if ((rc = ring_pin(sl.h_order, nrows * sizeof(uint32_t) + 16))) return rc;
    if ((rc = ring_pin(sl.h_nper, ns * sizeof(uint32_t)))) return rc;
    if ((rc = ring_pin(sl.h_status, sizeof(int32_t)))) return rc;
    return VS_OK;
}

/* the plan kernel of every slab, on the plan stream (flow and synth modes) */
int launch_plans(vs_ctx *ctx, Slot &sl, const Call &c, unsigned cp, size_t s0, const std::vector<VsRange> &slabs, cudaStream_t pstream)
{
    for (const VsRange &slab : slabs) {
        VsPlanArgs pa;
        memset(&pa, 0, sizeof pa);
        pa.streams = (const VsStream *)sl.streams[cp].p + (slab.first - s0);
        pa.n_streams = (uint32_t)(slab.second - slab.first);
        pa.chunks = (VsChunk *)sl.chunks[cp].p;
        pa.table = sl.table[cp].p;
        pa.compact = c.sh.compact;
        pa.rng_snap = c.sh.noise ? (uint32_t *)sl.snap[cp].p : nullptr;
        pa.n_periods = (uint32_t *)sl.nper[cp].p + (slab.first - s0);
        pa.costab = (const double *)sl.costab.p;
        pa.log = c.want_log ? sl.log.p : nullptr;
        pa.status = (int32_t *)sl.status[cp].p;
        bool busy = false;
        if (ctx->opt_plan_warps < 0) {
            /* "in flight" = the previous call has not finished, or it was enqueued less than 2 ms ago (a
             * loop of calls whose host side momentarily fell behind the GPU is still a pipeline) */
            busy = cudaEventQuery(sl.call_done[(cp + VS_DEPTH - 1u) % VS_DEPTH]) == cudaErrorNotReady;
            (void)cudaGetLastError();
            const auto now = std::chrono::steady_clock::now();
            if (std::chrono::duration<double, std::milli>(now - sl.last_enqueue).count() < 2.0) busy = true;
            sl.last_enqueue = now;
            sl.burst = busy ? sl.burst + 1u : 0u;
        }
        const bool warps = vs_plan_warps(ctx->opt_plan_warps, pa.n_streams, c.sh.noise, c.want_log, busy, sl.burst);
        CU(vs_launch_plan(pa, c.sh, warps, pstream));
        ctx->timing.launches++;
    }
    return VS_OK;
}

/* slab k: its input up (filter mode, host buffers), its render launch, its PCM home (host buffers) */
int render_slab(vs_ctx *ctx, Slot &sl, const Call &c, unsigned cp, size_t ns, size_t k, const VsRange &slab, const SlabSpan &sp,
                bool timed)
{
    const VsBatch &b = c.b;
    const std::vector<VsStream> &hs = ctx->in.hs;
    const int d = (int)((sl.scratch_parity + k) & 1);
    int16_t *d_pcm = c.out_dev ? b.pcm_out : (int16_t *)sl.pcm[d].p;
    double *d_raw = b.raw_out ? (c.out_dev ? b.raw_out : (double *)sl.raw[d].p) : nullptr;
    const int16_t *d_in = nullptr;

    if (!c.out_dev && sl.slab_done_valid[d]) CU(cudaStreamWaitEvent(sl.compute, sl.slab_done[d], 0));   /* its last D2H */

    if (b.mode == VS_MODE_FILTER) {
        if (c.out_dev) d_in = b.flow_in;
        else {
            d_in = (const int16_t *)sl.flowin[d].p;
            CU(cudaMemcpyAsync(sl.flowin[d].p, b.flow_in + sp.in_min, (sp.in_max - sp.in_min) * sizeof(int16_t), cudaMemcpyHostToDevice, sl.compute));
            ctx->timing.h2d_bytes += (sp.in_max - sp.in_min) * sizeof(int16_t);
        }
    }
    if (timed) { cudaEvent_t e1 = timing_event(sl); CU(cudaEventRecord(e1, sl.compute)); }

    const VsPlan &pl = sl.plan;
    VsRenderArgs ra;
    memset(&ra, 0, sizeof ra);
    const int gen = vs_render_geometry(ctx->opt, c.sh, ctx->in.facts, sl.sm_count, ns, pl, k, ra);
    ra.streams = (const VsStream *)sl.streams[cp].p;
    ra.chunks = (const VsChunk *)sl.chunks[cp].p;
    ra.order = (const uint32_t *)sl.order[cp].p + pl.slab_r0[k];
    ra.table = sl.table[cp].p;
    ra.n_periods = (const uint32_t *)sl.nper[cp].p;
    ra.rng_snap = c.sh.noise ? (const uint32_t *)sl.snap[cp].p : nullptr;
    ra.costab = (const double *)sl.costab.p;
    ra.flow_in = d_in;
    ra.pcm_out = d_pcm;
    ra.raw_out = d_raw;
    ra.debug = (uint32_t)ctx->opt_debug;
    ra.status = (int32_t *)sl.status[cp].p;
    if (c.sh.flow_rows) {
        if (!sl.ticket.p) {
            const int rc = dev_reserve(ctx, sl, sl.ticket, 256);
            if (rc) return rc;
            CU(cudaMemsetAsync(sl.ticket.p, 0, 256, sl.compute));
            sl.ticket_base = 0;
        }
        ra.ticket = (uint32_t *)sl.ticket.p;
        ra.ticket_base = sl.ticket_base;
        CU(vs_launch_flow_rows(ra, sl.compute));
        sl.ticket_base += ra.n_rows + ra.grid * VS_FLOWROWS_WARPS;     /* wraps like the device counter does */
    } else if (c.sh.tracts) {
        VsTractBlock tb;                             /* copied into the launch's parameter space */
        memcpy(tb.cta_end, pl.geom[k].cta_end, sizeof tb.cta_end);
        memset(tb.ncoef, 0, sizeof tb.ncoef);
        memcpy(tb.ncoef, ctx->in.ncoef.data(), ctx->in.ncoef.size() * sizeof(double));
        CU(vs_launch_render(ra, &tb, c.sh, gen, sl.compute));
    } else
        CU(vs_launch_render(ra, nullptr, c.sh, gen, sl.compute));
    ctx->timing.launches++;
    ctx->timing.render_path = vs_render_path(c.sh, gen);
    if (timed) { cudaEvent_t e2 = timing_event(sl); CU(cudaEventRecord(e2, sl.compute)); }
    if (c.out_dev) return VS_OK;

    /* PCM home over PCIe on the copy stream while the next slab renders */
    CU(cudaEventRecord(sl.slab_ready, sl.compute));
    CU(cudaStreamWaitEvent(sl.copy, sl.slab_ready, 0));
    CU(cudaStreamWaitEvent(sl.copy2, sl.slab_ready, 0));
    /* merge rows that touch into runs: a dense batch is one copy per slab -- cut into 16 MB pieces that
     * alternate between two copy streams, so that a second DMA engine keeps the link busy while the first
     * one finishes a piece */
    uint64_t run_lo = hs[slab.first].out_off, run_hi = hs[slab.first].out_off + hs[slab.first].n;
    auto flush = [&](uint64_t lo, uint64_t hi) -> cudaError_t {
        ctx->timing.d2h_bytes += (hi - lo) * (sizeof(int16_t) + (b.raw_out ? sizeof(double) : 0));
        cudaError_t e = cudaSuccess;
        const uint64_t piece = 8u << 20;                               /* samples */
        unsigned which = 0;
        for (uint64_t p0 = lo; p0 < hi && e == cudaSuccess; p0 += piece, which ^= 1u) {
            const uint64_t p1 = std::min(hi, p0 + piece);
            e = cudaMemcpyAsync(b.pcm_out + p0, d_pcm + (p0 - sp.out_min), (p1 - p0) * sizeof(int16_t),
                                cudaMemcpyDeviceToHost, which ? sl.copy2 : sl.copy);
        }
        if (e == cudaSuccess && b.raw_out)
            e = cudaMemcpyAsync(b.raw_out + lo, d_raw + (lo - sp.out_min), (hi - lo) * sizeof(double), cudaMemcpyDeviceToHost, sl.copy);
        return e;
    };
    for (size_t i = slab.first + 1; i < slab.second; i++) {
        if (hs[i].out_off == run_hi) run_hi += hs[i].n;
        else { CU(flush(run_lo, run_hi)); run_lo = hs[i].out_off; run_hi = run_lo + hs[i].n; }
    }
    CU(flush(run_lo, run_hi));
    CU(cudaEventRecord(sl.copy2_done, sl.copy2));
    CU(cudaStreamWaitEvent(sl.copy, sl.copy2_done, 0));
    CU(cudaEventRecord(sl.slab_done[d], sl.copy));
    sl.slab_done_valid[d] = true;
    return VS_OK;
}

/* the streams [s0, s1) on device slot g: plan, buffers, uploads, then slabs of plan -> render -> copy */
int run_slot(vs_ctx *ctx, Slot &sl, const Call &c, size_t g, size_t s0, size_t s1)
{
    const VsBatch &b = c.b;
    std::vector<VsStream> &hs = ctx->in.hs;
    const size_t ns = s1 - s0;
    CU(cudaSetDevice(sl.dev));
    if (g == 0) sl.tev_used = 0;

    size_t slab_streams = 0;
    const std::vector<VsRange> slabs = vs_slabs(hs, s0, s1, c.out_dev, ctx->opt.slab, &slab_streams);
    const size_t n_slabs = slabs.size();
    slot_plan(ctx, sl, c, s0, s1, slabs, slab_streams);
    const VsPlan &pl = sl.plan;
    vs_plan_assign(pl, hs, s0, s1);
    const size_t nc = pl.chunks.size(), nrows = pl.order.size();
    ctx->timing.chunks += (uint32_t)nc;
    for (size_t i = s0; i < s1; i++) ctx->timing.samples += hs[i].n;
    ctx->timing.warmup_samples += pl.warm_total;

    /* device memory: descriptor/table buffers alternate between calls (parity cp), so that the
     * upload + plan kernel of this call can run while the previous call still renders */
    const unsigned cp = sl.call_parity;
    sl.call_parity = (sl.call_parity + 1u) % VS_DEPTH;
    cudaStream_t pstream = sl.plans[cp & 1u];
    CU(cudaEventSynchronize(sl.call_done[cp]));                   /* the call before the previous one is done with them */
    int rc;
    if ((rc = slot_reserve(ctx, sl, c, cp, ns, pstream))) return rc;

    /* log span of this slot */
    uint64_t log_lo = 0, log_hi = 0;
    if (c.want_log) {
        const uint64_t *ro = b.log->rec_offsets;
        log_lo = ro[s0];
        log_hi = ro[s1];
        for (size_t i = s0; i < s1; i++) {
            if (ro[i + 1] < ro[i] || ro[i + 1] - ro[i] < hs[i].tab_cap)
                return fail(ctx, VS_EINVAL, "stream %zu: period log too small (need %u records)", i, hs[i].tab_cap);
            hs[i].log_off = ro[i] - log_lo;
        }
        if ((rc = dev_reserve(ctx, sl, sl.log, std::max<uint64_t>(1, log_hi - log_lo) * sizeof(vs_period_rec)))) return rc;
        CU(cudaMemsetAsync(sl.log.p, 0, (log_hi - log_lo) * sizeof(vs_period_rec), pstream));
    }

    /* device-side offsets: rows of a slab live at (offset - slab_min) + pad to keep the phase */
    std::vector<SlabSpan> span(n_slabs);
    uint64_t span_max = 0, in_span_max = 0;
    for (size_t k = 0; k < n_slabs; k++) {
        SlabSpan sp = {~0ull, 0, ~0ull, 0};
        for (size_t i = slabs[k].first; i < slabs[k].second; i++) {
            sp.out_min = std::min(sp.out_min, hs[i].out_off);
            sp.out_max = std::max(sp.out_max, hs[i].out_off + hs[i].n);
            sp.in_min = std::min(sp.in_min, hs[i].in_off);
            sp.in_max = std::max(sp.in_max, hs[i].in_off + hs[i].n);
        }
        sp.out_min &= ~63ull;                                     /* keep (offset mod 64) on the device */
        sp.in_min &= ~7ull;
        span[k] = sp;
        span_max = std::max(span_max, sp.out_max - sp.out_min);
        in_span_max = std::max(in_span_max, sp.in_max - sp.in_min);
    }
    if (!c.out_dev) {
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
        for (size_t i = slabs[k].first; i < slabs[k].second; i++) {
            ps[i - s0] = hs[i];
            if (!c.out_dev) {
                ps[i - s0].out_off = hs[i].out_off - span[k].out_min;
                ps[i - s0].in_off = hs[i].in_off - span[k].in_min;
            }
        }
    }
    /* chunk geometry and row order depend on the batch shape only; the plan kernel rewrites every
     * chunk's first_period each call.  Re-upload them only when the plan changed. */
    const bool upload_plan = sl.uploaded_version[cp] != sl.plan_version;
    if (upload_plan) {
        memcpy(sl.h_chunks[cp].p, pl.chunks.data(), nc * sizeof(VsChunk));
        memcpy(sl.h_order[cp].p, pl.order.data(), nrows * sizeof(uint32_t));
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
    c.prof.mark("reserve + descriptor upload");

    /* ---- plan stream: descriptors are up (above), now the plan kernel(s) of every slab -------- */
    if (g == 0) { cudaEvent_t t_first = timing_event(sl); CU(cudaEventRecord(t_first, pstream)); }
    if (b.mode != VS_MODE_FILTER && (rc = launch_plans(ctx, sl, c, cp, s0, slabs, pstream))) return rc;
    if (g == 0) { cudaEvent_t t_plan = timing_event(sl); CU(cudaEventRecord(t_plan, pstream)); }
    CU(cudaEventRecord(sl.plan_done[cp], pstream));
    if (ctx->env_sync_plan) CU(cudaStreamSynchronize(pstream));
    CU(cudaStreamWaitEvent(sl.compute, sl.plan_done[cp], 0));

    /* ---- compute stream: render (and copy) slab by slab ------------------------------------------ */
    for (size_t k = 0; k < n_slabs; k++)
        if ((rc = render_slab(ctx, sl, c, cp, ns, k, slabs[k], span[k], g == 0))) return rc;
    if (c.want_log) ctx->timing.d2h_bytes += (log_hi - log_lo) * sizeof(vs_period_rec);
    if (c.want_log)
        CU(cudaMemcpyAsync(b.log->rec + log_lo, sl.log.p, (log_hi - log_lo) * sizeof(vs_period_rec), cudaMemcpyDeviceToHost, sl.compute));
    if (c.want_log && b.log->count)
        CU(cudaMemcpyAsync(sl.h_nper[cp].p, sl.nper[cp].p, ns * sizeof(uint32_t), cudaMemcpyDeviceToHost, sl.compute));
    if (!c.out_dev) sl.scratch_parity = (unsigned)((sl.scratch_parity + n_slabs) & 1);
    if (g == 0) { cudaEvent_t t_last = timing_event(sl); CU(cudaEventRecord(t_last, sl.compute)); }
    /* the device's error flag comes home on the copy stream: nothing sits between this call's render kernel and
     * the next call's on the compute stream */
    CU(cudaEventRecord(sl.render_done[cp], sl.compute));
    CU(cudaStreamWaitEvent(sl.copy, sl.render_done[cp], 0));
    CU(cudaMemcpyAsync(sl.h_status[cp].p, sl.status[cp].p, sizeof(int32_t), cudaMemcpyDeviceToHost, sl.copy));
    CU(cudaEventRecord(sl.call_done[cp], sl.copy));               /* parity-cp buffers are free once this fires */
    return VS_OK;
}

int run_batch(vs_ctx *ctx, const VsBatch &b)
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
    const VsPlanOptions &o = ctx->opt;
    {   /* what the chunk plan depends on besides the parameter arrays */
        const double key[9] = {o.chunk, o.tol, (double)o.exact, (double)o.slab, (double)o.simple_gen, (double)(out_kind == PK_DEVICE),
                               (double)(reinterpret_cast<uintptr_t>(b.pcm_out) & 127), (double)ctx->slots.size(), b.ft ? 1.0 : 0.0};
        snapshot_inputs(b, want_log, key, sizeof key, blob);
    }
    const bool same_inputs = blob.size() == ctx->in_blob.size() && memcmp(blob.data(), ctx->in_blob.data(), blob.size()) == 0;
    if (!same_inputs) {
        ctx->in_blob.clear();                                    /* nothing is cached while the tables below may fail half way */
        std::string err;
        const int rc = vs_build_descriptors(b, want_log, ctx->tables, ctx->in, err);
        if (rc) return fail(ctx, rc, "%s", err.c_str());
        ctx->in_blob.swap(blob);
        ctx->in_version++;
    }
    const std::vector<VsStream> &hs = ctx->in.hs;
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
    const std::vector<size_t> cut = vs_split_slots(hs, nslots);
    memset(&ctx->timing, 0, sizeof ctx->timing);
    ctx->timing_pending = true;

    /* ---- 4. per slot: plan, descriptors up, then slabs of plan -> render -> copy -------------- */
    const Call call = {b, want_log, same_inputs, out_dev,
                       vs_shape(b.mode, b.ft != nullptr, want_log, ctx->in.facts, o),
                       out_dev ? (uint64_t)(reinterpret_cast<uintptr_t>(b.pcm_out) >> 1) : 0u, prof};
    for (size_t g = 0; g < nslots; g++) {
        if (cut[g + 1] <= cut[g]) continue;
        const int rc = run_slot(ctx, ctx->slots[g], call, g, cut[g], cut[g + 1]);
        if (rc) return rc;
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

/* ---- calls on PCM the caller owns: output noise, flow analysis and report, formants ---------------------------------- */
/* the checks of these calls, in index order so that the first offender decides: the stream count, then per stream its
 * length, its sampling rate (fs NULL: 22050 Hz) and the call's own checks, stream(i, rate) */
template <class Stream>
int check_streams(std::string *err, const uint64_t *nsamp, const int32_t *fs, size_t n, Stream stream)
{
    if (n > 0x7fffffffull) return vs_error(err, VS_EINVAL, "too many streams");
    for (size_t i = 0; i < n; i++) {
        if (nsamp[i] > 0x7fffffffull) return vs_error(err, VS_EOVERLAP, "stream %zu: too many samples", i);
        const int32_t rate = fs ? fs[i] : 22050;
        if (rate <= 0) return vs_error(err, VS_ERANGE, "stream %zu: sampling rate", i);
        if (const int rc = stream(i, rate)) return rc;
    }
    return VS_OK;
}

/* sets rows[i].off, where stream i starts in the caller's PCM (offsets NULL: dense rows at a stride of the longest
 * one), and returns the samples [first, last) the rows cover */
struct Span { uint64_t first, last; };
template <class Row>
Span place_rows(const uint64_t *offsets, const uint64_t *nsamp, std::vector<Row> &rows)
{
    uint64_t stride = 0;
    for (size_t i = 0; i < rows.size(); i++) stride = std::max(stride, nsamp[i]);
    Span s = {~0ull, 0};
    for (size_t i = 0; i < rows.size(); i++) {
        rows[i].off = offsets ? offsets[i] : (uint64_t)i * stride;
        s.first = std::min(s.first, rows[i].off);
        s.last = std::max(s.last, rows[i].off + nsamp[i]);
    }
    return s;
}

/* a call's device scratch: pieces at 256-byte aligned offsets, in the order they are taken */
struct Scratch {
    size_t bytes = 0;
    size_t take(size_t b) { const size_t at = bytes; bytes = (bytes + b + 255) & ~(size_t)255; return at; }
};

/* the device side of a call whose arguments have passed: earlier work must have landed (the PCM may be the output of
 * a call still in flight, and the noise call writes it in place); slot 0 runs it (one device is plenty: 0.75 ms for
 * the noise of 4096 x 1 s); the scratch and the staged PCM.  The caller holds a DeviceGuard. */
template <class T> struct PcmDev {
    cudaStream_t st;
    T *pcm;                      /* the PCM as the kernels address it: row offsets are relative to this */
    bool staged;                 /* the caller's PCM is host memory, staged into pcm[0] */
    unsigned char *scratch;
};
template <class T>
int pcm_call_begin(vs_ctx *ctx, T *pcm, const Span &span, size_t scratch_bytes, PcmDev<T> &d)
{
    int rc, dev = -1;
    if ((rc = vs_sync(ctx))) return rc;
    Slot &sl = ctx->slots[0];
    CU(cudaSetDevice(sl.dev));
    d = {sl.compute, pcm, classify(pcm, &dev) != PK_DEVICE, nullptr};
    if (!d.staged && dev != sl.dev) return fail(ctx, VS_EINVAL, "device buffer lives on device %d, ctx on %d", dev, sl.dev);
    if ((rc = dev_reserve(ctx, sl, sl.analyze, scratch_bytes))) return rc;
    d.scratch = (unsigned char *)sl.analyze.p;
    if (d.staged) {
        const size_t bytes = (span.last - span.first) * sizeof(int16_t);
        if ((rc = dev_reserve(ctx, sl, sl.pcm[0], bytes + 256))) return rc;
        d.pcm = (T *)sl.pcm[0].p - span.first;
        CU(cudaMemcpyAsync(sl.pcm[0].p, pcm + span.first, bytes, cudaMemcpyHostToDevice, d.st));
    }
    return VS_OK;
}

/* device-to-host copy of n rows, row(i) = {offset in src, offset in dst, elements}; a row that continues the previous
 * non-empty one on both sides travels with it as one copy */
struct RowCopy { uint64_t s, d, n; };
template <class T, class Row>
int copy_rows_home(vs_ctx *ctx, T *dst, const T *src, size_t n, Row row, cudaStream_t st)
{
    RowCopy run = {0, 0, 0};
    for (size_t i = 0; i <= n; i++) {
        const RowCopy r = i < n ? row(i) : RowCopy{0, 0, 0};
        if (i < n && !r.n) continue;
        if (r.n && run.n && r.s == run.s + run.n && r.d == run.d + run.n) { run.n += r.n; continue; }
        if (run.n) CU(cudaMemcpyAsync(dst + run.d, src + run.s, run.n * sizeof(T), cudaMemcpyDeviceToHost, st));
        run = r;
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
    ctx->tables.set_tol(ctx->opt.tol);
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
        bool ok = cudaSetDevice(d) == cudaSuccess;
        for (cudaStream_t *st : {&s.compute, &s.copy, &s.copy2, &s.plans[0], &s.plans[1]})
            ok = ok && cudaStreamCreateWithFlags(st, cudaStreamNonBlocking) == cudaSuccess;
        for (cudaEvent_t *e : s.events()) ok = ok && cudaEventCreateWithFlags(e, cudaEventDisableTiming) == cudaSuccess;
        ok = ok && vs_render_init_device() == cudaSuccess;
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
        for (cudaStream_t st : s.all_streams()) if (st) cudaStreamSynchronize(st);    /* a half-built slot lacks some */
        std::vector<DevBuf *> bufs = {&s.costab, &s.pcm[0], &s.pcm[1], &s.raw[0], &s.raw[1], &s.flowin[0], &s.flowin[1], &s.log, &s.ticket, &s.analyze};
        std::vector<PinBuf *> pins;
        for (int k = 0; k < VS_DEPTH; k++) {
            for (DevBuf *b : {&s.streams[k], &s.chunks[k], &s.order[k], &s.table[k], &s.snap[k], &s.nper[k], &s.status[k]}) bufs.push_back(b);
            for (PinBuf *b : {&s.h_streams[k], &s.h_chunks[k], &s.h_order[k], &s.h_nper[k], &s.h_status[k]}) pins.push_back(b);
        }
        for (DevBuf *b : bufs) if (b->p) cudaFree(b->p);
        for (PinBuf *b : pins) if (b->p) cudaFreeHost(b->p);
        for (cudaEvent_t e : s.tev) cudaEventDestroy(e);
        for (cudaEvent_t *e : s.events()) if (*e) cudaEventDestroy(*e);
        for (cudaStream_t st : {s.plans[0], s.plans[1], s.copy2, s.copy}) if (st) cudaStreamDestroy(st);
        if (s.compute && s.own_compute) cudaStreamDestroy(s.compute);
    }
    cudaGetLastError();
    delete ctx;
}

int vs_ctx_set_option(vs_ctx *ctx, int option, double value)
{
    if (!ctx) return VS_EINVAL;
    switch (option) {
    case VS_OPT_CHUNK_SAMPLES: ctx->opt.chunk = value; return VS_OK;
    case VS_OPT_CARRY_TOL:
        if (!(value > 0.0 && value < 1.0)) return VS_EINVAL;
        ctx->opt.tol = value; ctx->tables.set_tol(value); return VS_OK;
    case VS_OPT_EXACT_FILTER: ctx->opt.exact = value != 0.0; return VS_OK;
    case VS_OPT_SLAB_STREAMS: ctx->opt.slab = value > 0 ? (int)value : 0; return VS_OK;
    case VS_OPT_TARGET_WARPS: return value > 0 ? VS_OK : VS_EINVAL;       /* accepted, no effect */
    case VS_OPT_ASYNC_HOST: ctx->opt_async_host = value != 0.0; return VS_OK;
    case VS_OPT_PLAN_WARPS: ctx->opt_plan_warps = value < 0 ? -1 : (value != 0.0); return VS_OK;
    case VS_OPT_SIMPLE_GEN: ctx->opt.simple_gen = value != 0.0; return VS_OK;
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
        const int rc = drain(ctx, s);
        if (rc) return rc;
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

int vs_filter_warmup(vs_ctx *ctx, int preset_key, float gain)
{
    (void)gain;
    if (!ctx) return VS_EINVAL;
    const int k = preset_index(preset_key);
    return k < 0 ? VS_EPRESET : ctx->tables.warm[k];
}

int vs_flowgen_batch(vs_ctx *ctx, const vs_flow_params *p, size_t n, int16_t *pcm_out, const uint64_t *offsets, vs_period_log *log)
{
    VsBatch b = {VS_MODE_FLOW, n, p, nullptr, nullptr, nullptr, nullptr, nullptr, pcm_out, offsets, nullptr, log};
    return run_batch(ctx, b);
}

int vs_vowel_filter_batch(vs_ctx *ctx, const int16_t *flow_in, const uint64_t *in_offsets, const uint64_t *nsamp,
                          const vs_filter_params *f, size_t n, int16_t *pcm_out, const uint64_t *out_offsets, double *raw_out)
{
    VsBatch b = {VS_MODE_FILTER, n, nullptr, f, nullptr, flow_in, in_offsets, nsamp, pcm_out, out_offsets, raw_out, nullptr};
    return run_batch(ctx, b);
}

int vs_vowel_filter_batch_tract(vs_ctx *ctx, const int16_t *flow_in, const uint64_t *in_offsets, const uint64_t *nsamp,
                                const vs_tract_params *t, size_t n, int16_t *pcm_out, const uint64_t *out_offsets, double *raw_out)
{
    if (!t) return fail(ctx, VS_EINVAL, "tract params are NULL");
    VsBatch b = {VS_MODE_FILTER, n, nullptr, nullptr, t, flow_in, in_offsets, nsamp, pcm_out, out_offsets, raw_out, nullptr};
    return run_batch(ctx, b);
}

int vs_vowel_noise_batch(vs_ctx *ctx, int16_t *pcm, const uint64_t *offsets, const uint64_t *nsamp, const float *snr,
                         const int32_t *fs, const uint32_t *seed, size_t n)
{
    if (!ctx || !pcm || !nsamp || !snr) return VS_EINVAL;
    if (n == 0) return VS_OK;
    std::vector<VsNoiseRow> rows;
    int rc = check_streams(&ctx->err, nsamp, fs, n, [&](size_t i, int32_t rate) {
        const int ms1 = (int)((uint32_t)rate * 0.001 / 2.0) * 2;       /* vowel_new.c:361 */
        const long frame = 50L * ms1;                                  /* :363 */
        if (snr[i] > 0.0f && (frame <= 0 || frame > 32767)) return fail(ctx, VS_ERANGE, "stream %zu: frame length %ld", i, frame);
        if (i == 0) rows.resize(n);                                    /* n has passed the stream-count check */
        rows[i] = {0, (uint32_t)nsamp[i], (uint32_t)frame, snr[i], seed ? seed[i] : 1u};
        return VS_OK;
    });
    if (rc) return rc;
    const Span span = place_rows(offsets, nsamp, rows);
    DeviceGuard restore_device;
    PcmDev<int16_t> d;
    if ((rc = pcm_call_begin(ctx, pcm, span, n * sizeof(VsNoiseRow), d))) return rc;
    CU(cudaMemcpyAsync(d.scratch, rows.data(), n * sizeof(VsNoiseRow), cudaMemcpyHostToDevice, d.st));
    CU(vs_launch_vnoise(d.pcm, (const VsNoiseRow *)d.scratch, (uint32_t)n, d.st));
    /* host memory: only the noised rows come back, the bytes between and around them are the caller's */
    auto noised = [&](size_t i) { return RowCopy{rows[i].off, rows[i].off, rows[i].snr > 0.0f ? rows[i].n : 0u}; };
    if (d.staged && (rc = copy_rows_home(ctx, pcm, d.pcm, n, noised, d.st))) return rc;
    CU(cudaStreamSynchronize(d.st));                          /* `rows` is pageable host memory */
    return VS_OK;
}

/* vs_flow_analyze_batch (report NULL: stats is the caller's) and vs_flow_report_batch (stats NULL: the statistics
 * stay on the device, the report kernel copies them into report[i].base) */
static int flow_analysis(vs_ctx *ctx, const int16_t *flow, const uint64_t *offsets, const uint64_t *nsamp, const int32_t *fs,
                         const int16_t *lo, const int16_t *hi, size_t n, vs_flow_stats *stats, vs_flow_report *report)
{
    if (n == 0) return VS_OK;
    std::vector<VsAnalyzeRow> rows;
    uint64_t slots = 0;
    int rc = check_streams(&ctx->err, nsamp, fs, n, [&](size_t i, int32_t rate) {
        const int16_t tl = lo ? lo[i] : (int16_t)0, th = hi ? hi[i] : (int16_t)0;
        if (tl > th) return fail(ctx, VS_ERANGE, "stream %zu: thresholds lo > hi", i);
        const uint32_t len = (uint32_t)nsamp[i], cap = len / 16u + 4u;
        if (i == 0) rows.resize(n);                                    /* n has passed the stream-count check */
        rows[i] = {0, slots, len, cap, rate, tl, th};
        slots += cap;
        return VS_OK;
    });
    if (rc) return rc;
    const Span span = place_rows(offsets, nsamp, rows);
    /* scratch: rows | per-stream onset counts | stats | onset lists, and for the report: | peak lists | reports */
    Scratch sc;
    const size_t o_rows = sc.take(n * sizeof(VsAnalyzeRow)), o_cnt = sc.take(n * sizeof(uint32_t));
    const size_t o_st = sc.take(n * sizeof(vs_flow_stats)), o_ons = sc.take(slots * sizeof(uint32_t));
    const size_t o_peaks = report ? sc.take(slots * sizeof(uint32_t)) : 0, o_rep = report ? sc.take(n * sizeof(vs_flow_report)) : 0;
    DeviceGuard restore_device;
    PcmDev<const int16_t> d;
    if ((rc = pcm_call_begin(ctx, flow, span, sc.bytes, d))) return rc;
    const VsAnalyzeRow *d_rows = (const VsAnalyzeRow *)(d.scratch + o_rows);
    uint32_t *d_cnt = (uint32_t *)(d.scratch + o_cnt), *d_ons = (uint32_t *)(d.scratch + o_ons);
    vs_flow_stats *d_st = (vs_flow_stats *)(d.scratch + o_st);
    CU(cudaMemcpyAsync(d.scratch + o_rows, rows.data(), n * sizeof(VsAnalyzeRow), cudaMemcpyHostToDevice, d.st));
    if (!report) {
        CU(vs_launch_analyze(d.pcm, d_rows, (uint32_t)n, d_ons, d_cnt, d_st, d.st));
        CU(cudaMemcpyAsync(stats, d_st, n * sizeof(vs_flow_stats), cudaMemcpyDeviceToHost, d.st));
    } else {
        vs_flow_report *d_rep = (vs_flow_report *)(d.scratch + o_rep);
        CU(vs_launch_report(d.pcm, d_rows, (uint32_t)n, d_ons, d_cnt, d_st, (int32_t *)(d.scratch + o_peaks), d_rep, d.st));
        CU(cudaMemcpyAsync(report, d_rep, n * sizeof(vs_flow_report), cudaMemcpyDeviceToHost, d.st));
    }
    CU(cudaStreamSynchronize(d.st));                          /* `rows` and the results are the caller's / pageable memory */
    return VS_OK;
}

int vs_flow_analyze_batch(vs_ctx *ctx, const int16_t *flow, const uint64_t *offsets, const uint64_t *nsamp, const int32_t *fs,
                          const int16_t *lo, const int16_t *hi, size_t n, vs_flow_stats *stats)
{
    if (!ctx || !flow || !nsamp || !stats) return VS_EINVAL;
    return flow_analysis(ctx, flow, offsets, nsamp, fs, lo, hi, n, stats, nullptr);
}

int vs_flow_report_batch(vs_ctx *ctx, const int16_t *flow, const uint64_t *offsets, const uint64_t *nsamp, const int32_t *fs,
                         const int16_t *lo, const int16_t *hi, size_t n, vs_flow_report *out)
{
    if (!ctx || !flow || !nsamp || !out) return VS_EINVAL;
    return flow_analysis(ctx, flow, offsets, nsamp, fs, lo, hi, n, nullptr, out);
}

/* the option and per-stream checks of vs_formant_frames and vs_formant_batch, in the header's order; fills o (the
 * defaults for in == NULL), each stream's frame count and, unless rows is NULL, its row but for off, win_off and mu */
static int formant_geometry(const vs_formant_opts *in, const uint64_t *nsamp, const int32_t *fs, size_t n, vs_formant_opts &o,
                            VsFormantRow *rows, uint64_t *frames, std::string *err)
{
    o = in ? *in : vs_formant_opts{25.0f, 10.0f, 50.0f, 700.0f, 14u, 5u};
    if (o.order < 2 || o.order > VS_FMT_MAX_ORDER || (o.order & 1u)) return vs_error(err, VS_EINVAL, "order %u: even, 2..%d", o.order, VS_FMT_MAX_ORDER);
    if (o.n_formants < 1 || o.n_formants > VS_MAX_FORMANTS || o.n_formants > o.order / 2)
        return vs_error(err, VS_EINVAL, "n_formants %u: 1..%d and at most order / 2", o.n_formants, VS_MAX_FORMANTS);
    if (!(o.preemph_hz >= 0.0f) || !(o.bmax_hz >= 0.0f)) return vs_error(err, VS_ERANGE, "preemph_hz and bmax_hz must be >= 0");
    return check_streams(err, nsamp, fs, n, [&](size_t i, int32_t rate) {
        const double wl = (double)o.win_ms * rate / 1000.0, hl = (double)o.hop_ms * rate / 1000.0;
        const long nw = wl > -1e9 && wl < 1e9 ? lround(wl) : -1;
        if (nw < (long)o.order + 1 || nw > VS_FORMANT_MAX_WIN)
            return vs_error(err, VS_ERANGE, "stream %zu: window of %ld samples, needs %u..%d", i, nw, o.order + 1, VS_FORMANT_MAX_WIN);
        if (!(hl >= 0.5 && hl < 2147483647.5)) return vs_error(err, VS_ERANGE, "stream %zu: frame step below 1 sample or above 2^31-1", i);
        const uint64_t h = (uint64_t)lround(hl);
        if (rows) rows[i] = {0, (uint32_t)nsamp[i], (uint32_t)nw, (uint32_t)h, 0, 0.0, (double)rate};
        frames[i] = nsamp[i] >= (uint64_t)nw ? (nsamp[i] - (uint64_t)nw) / h + 1 : 0;
        return VS_OK;
    });
}

int vs_formant_frames(const vs_formant_opts *o, const uint64_t *nsamp, const int32_t *fs, size_t n, uint64_t *frames_out)
{
    if (!nsamp || !frames_out) return VS_EINVAL;
    vs_formant_opts oo;
    return formant_geometry(o, nsamp, fs, n, oo, nullptr, frames_out, nullptr);
}

int vs_formant_batch(vs_ctx *ctx, const int16_t *pcm, const uint64_t *offsets, const uint64_t *nsamp, const int32_t *fs,
                     size_t n, const vs_formant_opts *o, vs_formant_stats *stats, vs_formant_frame *frames,
                     const uint64_t *frame_offsets)
{
    if (!ctx || !pcm || !nsamp || !stats) return VS_EINVAL;
    vs_formant_opts op;
    std::vector<VsFormantRow> rows(n);
    std::vector<uint64_t> nfr(n);
    int rc = formant_geometry(o, nsamp, fs, n, op, rows.data(), nfr.data(), &ctx->err);
    if (rc) return rc;
    if (n == 0) return VS_OK;

    /* pre-emphasis, the frame prefix and one window table per distinct window length; host libm in double */
    const double pi = 3.14159265358979323846;
    std::vector<uint64_t> frame0(n + 1, 0);
    std::vector<double> win;
    std::vector<std::pair<uint32_t, uint32_t>> win_at;        /* (Nw, offset) */
    uint32_t max_nw = 0;
    for (size_t i = 0; i < n; i++) {
        VsFormantRow &r = rows[i];
        r.mu = op.preemph_hz > 0.0f ? std::exp(-2.0 * pi * (double)op.preemph_hz / r.fs) : 0.0;
        auto it = std::find_if(win_at.begin(), win_at.end(), [&](const std::pair<uint32_t, uint32_t> &e) { return e.first == r.Nw; });
        if (it == win_at.end()) {
            win_at.push_back({r.Nw, (uint32_t)win.size()});
            for (uint32_t m = 0; m < r.Nw; m++) win.push_back(0.54 - 0.46 * std::cos(2.0 * pi * (double)m / (double)(r.Nw - 1)));
            it = win_at.end() - 1;
        }
        r.win_off = it->second;
        max_nw = std::max(max_nw, r.Nw);
        frame0[i + 1] = frame0[i] + nfr[i];
    }
    const Span span = place_rows(offsets, nsamp, rows);
    const uint64_t F = frame0[n];
    VsFormantArgs a = {};
    a.n_rows = (uint32_t)n; a.order = op.order; a.nf = op.n_formants; a.max_nw = max_nw; a.n_frames = F; a.bmax = op.bmax_hz;
    for (uint32_t j = 0; j < op.order; j++) {
        const double t = 2.0 * pi * (double)j / (double)op.order + 0.4;
        a.seed_re[j] = 0.9 * std::cos(t);
        a.seed_im[j] = 0.9 * std::sin(t);
    }

    /* scratch: rows | frame prefix | windows | per-frame found/flags | per-frame F, B | stats | frame records */
    Scratch sc;
    const size_t o_rows = sc.take(n * sizeof(VsFormantRow)), o_pre = sc.take((n + 1) * sizeof(uint64_t));
    const size_t o_win = sc.take(win.size() * sizeof(double)), o_ff = sc.take(F * sizeof(uint32_t));
    const size_t o_fb = sc.take(F * 2 * op.n_formants * sizeof(double)), o_st = sc.take(n * sizeof(vs_formant_stats));
    const size_t o_fr = sc.take(frames ? F * sizeof(vs_formant_frame) : 0);
    DeviceGuard restore_device;
    PcmDev<const int16_t> d;
    if ((rc = pcm_call_begin(ctx, pcm, span, sc.bytes, d))) return rc;
    a.pcm = d.pcm;
    a.rows = (const VsFormantRow *)(d.scratch + o_rows);
    a.frame0 = (const uint64_t *)(d.scratch + o_pre);
    a.win = (const double *)(d.scratch + o_win);
    a.ff = (uint32_t *)(d.scratch + o_ff);
    a.fb = (double *)(d.scratch + o_fb);
    vs_formant_stats *d_stats = (vs_formant_stats *)(d.scratch + o_st);
    vs_formant_frame *d_frames = frames ? (vs_formant_frame *)(d.scratch + o_fr) : nullptr;
    CU(cudaMemcpyAsync((void *)a.rows, rows.data(), n * sizeof(VsFormantRow), cudaMemcpyHostToDevice, d.st));
    CU(cudaMemcpyAsync((void *)a.frame0, frame0.data(), (n + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, d.st));
    CU(cudaMemcpyAsync((void *)a.win, win.data(), win.size() * sizeof(double), cudaMemcpyHostToDevice, d.st));
    CU(vs_launch_formants(a, d_stats, d_frames, d.st));
    CU(cudaMemcpyAsync(stats, d_stats, n * sizeof(vs_formant_stats), cudaMemcpyDeviceToHost, d.st));
    /* stream i's records: frame0[i] on the device, frame_offsets[i] (NULL: the same dense prefix) on the host */
    auto records = [&](size_t i) { return RowCopy{frame0[i], frame_offsets ? frame_offsets[i] : frame0[i], nfr[i]}; };
    if (frames && (rc = copy_rows_home(ctx, frames, d_frames, n, records, d.st))) return rc;
    CU(cudaStreamSynchronize(d.st));                          /* `rows` and the results are pageable host memory */
    return VS_OK;
}

int vs_synth_batch(vs_ctx *ctx, const vs_flow_params *p, const vs_filter_params *f, size_t n, int16_t *pcm_out,
                   const uint64_t *offsets, double *raw_out)
{
    VsBatch b = {VS_MODE_SYNTH, n, p, f, nullptr, nullptr, nullptr, nullptr, pcm_out, offsets, raw_out, nullptr};
    return run_batch(ctx, b);
}

int vs_synth_batch_tract(vs_ctx *ctx, const vs_flow_params *p, const vs_tract_params *t, size_t n, int16_t *pcm_out,
                         const uint64_t *offsets, double *raw_out)
{
    if (!t) return fail(ctx, VS_EINVAL, "tract params are NULL");
    VsBatch b = {VS_MODE_SYNTH, n, p, nullptr, t, nullptr, nullptr, nullptr, pcm_out, offsets, raw_out, nullptr};
    return run_batch(ctx, b);
}

} /* extern "C" */
