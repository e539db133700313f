/* vs_render.cu -- the sm_100a render kernel of libvoicesynth_cuda: ONE THREAD PER STREAM-CHUNK.
 *
 * A CTA is 4 warps (one per SM sub-partition); lane l of a warp owns one row = one time-chunk of one voice
 * and walks down it sample by sample, all 32 lanes in lock step (SIMT across voices):
 *
 *   G  generate   the glottal flow sample (flowgen_shimmer.c:316-336, noise :385-406) from the period table the
 *                 plan kernel wrote: x = ceil(A * table[i]) inside the open phase, DC outside.  Branch free:
 *                 8 samples at a time, the lane's current and next pitch period both in registers, a sample
 *                 picks its period by a bit of a per-group mask (GEN_FAST).  Period entries reach the lane
 *                 through a small per-lane ring in shared memory that cp.async refills one window ahead;
 *                 pulse tables are staged in shared memory once per warp.
 *   F  filter     the order-22 all-pole recurrence (vowel_new.c:266-289) in FP64 registers: a 24-entry ring,
 *                 fully unrolled, coefficients in UNIFORM registers (the vowel preset is a function of
 *                 blockIdx and kernel parameters).  23 FP64-pipe instructions per sample when gain is integral and
 *                 pre-emphasis 0 or 1 (both commute to the integer input: x' = gain*(x[n] - pre*x[n-1])),
 *                 25 otherwise; the FP64 pipe is the bound.  Quantiser: one F2I + clamp.
 *   W  write      every lane packs 8 results into one 16-byte shared-memory store down its own tile row
 *                 (row stride 16 x odd bytes: conflict free); once per window every lane hands its row
 *                 to the TMA engine as one bulk shared->global copy (cp.async.bulk, SASS UBLKCP) -- whole
 *                 16-byte pieces, 16-byte aligned in HBM -- and carries on with the other tile.
 *
 * The flow never exists in memory: in the fused mode only int16 PCM leaves the SM.
 * GEN_SIMPLE is the general generator (per-sample, branching): glottal noise, -z, very short pitch periods.
 * Exact mode (VS_OPT_EXACT_FILTER) keeps the reference's unfused multiply/subtract order and its floor-based
 * round2int() bit for bit.
 */
#include "vs_device.cuh"
#include "vs_presets.h"

#include <type_traits>

static_assert(VS_NUM_PRESETS == VS_NUM_PRESETS_I, "preset count");

__constant__ double c_ncoef[VS_NUM_PRESETS][VS_RING];      /* c_ncoef[p][j] = -A_p[j], j = 1..22 (vowel_new.c:450-544) */

#define VS_BIG_T 0x3fffffff
#define VS_GROUP 8

/* ---- PTX: async copies -------------------------------------------------------------------------------- */
__device__ __forceinline__ void vs_cp_async8(uint32_t dst_smem, const void *src)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst_smem), "l"(src) : "memory");
}
template <uint32_t BYTES>
__device__ __forceinline__ void vs_cp_async(uint32_t dst_smem, const void *src)
{
    if (BYTES == 16) asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst_smem), "l"(src) : "memory");
    else asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst_smem), "l"(src) : "memory");
}
__device__ __forceinline__ void vs_cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
/* this thread's shared-memory writes become visible to the async proxy (the TMA engine) */
__device__ __forceinline__ void vs_fence_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void vs_bulk_s2g(void *gdst, uint32_t src_smem, uint32_t bytes)
{
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(src_smem), "r"(bytes) : "memory");
}
__device__ __forceinline__ void vs_bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void vs_bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }

/* shared-memory accesses by 32-bit shared-window address: no generic-to-shared conversion in the sample loop, the
 * constant part of the address folds into the instruction */
__device__ __forceinline__ double vs_lds_f64(uint32_t addr)
{
    double v;
    asm("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t vs_lds_u32(uint32_t addr)
{
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void vs_sts_u32(uint32_t addr, uint32_t v)
{
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

/* the glottal-noise sample (flowgen_shimmer.c:387,394) in two FP64 operations: t = r/M - 1/2, w = ceil(t*NDW).
 * Equal to the reference's divide / multiply / subtract / ceil for every r and NDW < 2^19 (proof and exhaustive
 * check around every breakpoint: tests/tools/noisecheck.c). */
__device__ __forceinline__ int vs_noise_w2(int32_t r, double ndwd)
{
    /* r == M would have to give t = 1/2 exactly; r = M-1 gives 1/2 - 5e-10, the same ceiling for NDW < 2^19 */
    const double t = __fma_rn((double)min(r, 2147483646), VS_INV_RM, -0.5);
    return vs_ceil_s16(__dmul_rn(t, ndwd));
}

__device__ __forceinline__ void vs_pair_barrier(int pair)
{
    asm volatile("bar.sync %0, 64;" ::"r"(1 + pair) : "memory");
}

/* ---- F: one lane, one row: the order-22 recurrence (vowel_new.c:266-289) window after window, in place ------- *
 * Coefficients: PRESET >= 0 reads c_ncoef[PRESET] at literal constant-bank addresses; PRESET < 0 reads tcoef[0..21]
 * (= -A[1..22]) inside the kernel's parameter block (the tract kernels).  The operations and their order are the
 * same either way. */
template <int WIN, int NT, int FILT, bool RAW, int PRESET>
__device__ __forceinline__ void vs_filter_rows(unsigned char *tiles /* the lane's row in tile 0 */, const int pair, const int nwin,
                                               const double gaind, const double pred, double *rrow, const int blk0, const int lo, const int hi,
                                               const double *tcoef)
{
#define VS_NC(j) (PRESET >= 0 ? c_ncoef[PRESET < 0 ? 0 : PRESET][j] : tcoef[(j) - 1])
    constexpr int TILE = 32 * WIN * 2;
    double y[VS_RING];
#pragma unroll
    for (int j = 0; j < VS_RING; j++) y[j] = 0.0;
    const int gain_i = (int)gaind;
    /* FILT_INT: the bytes {-pre, 1} of a two-way 16x8 dot product (pre is 0 or 1) */
    const int pre_b = (int)(((uint32_t)-(int)pred & 0xffu) | 0x100u);
    uint32_t w_prev = 0;                                    /* the last input word read: its high half is x[n-1] */
    int mbase = blk0, ti = 0;

    vs_pair_barrier(pair);                                  /* window 0 generated */
    for (int w = 0; w < nwin; w++) {
        unsigned char *trow = tiles + (uint32_t)ti * TILE;
        ti = ti == NT - 1 ? 0 : ti + 1;
#pragma unroll 1
        for (int b = 0; b < WIN / VS_RING; b++) {
#pragma unroll
            for (int g = 0; g < VS_RING / VS_GROUP; g++) {
                uint4 *piece = reinterpret_cast<uint4 *>(trow + (b * VS_RING + g * VS_GROUP) * 2);
                const uint4 xv = *piece;
                const uint32_t xw[4] = {xv.x, xv.y, xv.z, xv.w};
                uint32_t ow[VS_GROUP / 2];
                int qv[VS_GROUP];
#pragma unroll
                for (int u = 0; u < VS_GROUP; u++) {
                    const int k = g * VS_GROUP + u;
                    const int xi = (u & 1) ? (int)xw[u >> 1] >> 16 : (int)(int16_t)(xw[u >> 1] & 0xffffu);
                    double acc, v;
                    if (FILT == VS_FILT_INT) {
                        /* gain and pre-emphasis on the integer input; the recurrence then yields the
                         * pre-emphasised waveform directly (the filter is LTI).  x[n] - pre*x[n-1] is one
                         * dp2a on a word whose halves are (x[n-1], x[n]): an input word itself for odd u, the
                         * high half of the previous word and the low half of this one for even u. */
                        const uint32_t xx = (u & 1) ? xw[u >> 1] : __byte_perm(u == 0 ? w_prev : xw[(u >> 1) - 1], xw[u >> 1], 0x5432);
                        acc = (double)(__dp2a_lo((int)xx, pre_b, 0) * gain_i);
#pragma unroll
                        for (int j = VS_ORDER; j >= 1; j--) acc = __fma_rn(y[(k + VS_RING - j) % VS_RING], VS_NC(j), acc);
                        v = acc;
                    } else if (FILT == VS_FILT_FMA) {
                        acc = __dmul_rn((double)xi, gaind);                                          /* vowel_new.c:266-269 */
#pragma unroll
                        for (int j = VS_ORDER; j >= 1; j--) acc = __fma_rn(y[(k + VS_RING - j) % VS_RING], VS_NC(j), acc);
                        v = __fma_rn(-pred, y[(k + VS_RING - 1) % VS_RING], acc);                    /* :284 */
                    } else {
                        acc = __dmul_rn((double)xi, gaind);
#pragma unroll
                        for (int j = 1; j <= VS_ORDER; j++)                                          /* :279-281, same order, unfused */
                            acc = __dsub_rn(acc, __dmul_rn(-VS_NC(j), y[(k + VS_RING - j) % VS_RING]));
                        v = __dsub_rn(acc, __dmul_rn(pred, y[(k + VS_RING - 1) % VS_RING]));
                    }
                    y[k] = acc;                                                                      /* :287-289 (ring) */
                    /* quantiser: round2int() of vowel_new.c:413-427, literally, in exact mode; otherwise one F2I
                     * (saturating; ties -- never hit -- go to even), clipped to +-32767 two samples at a time by the
                     * saturating pack and a 16x2 maximum below */
                    qv[u] = FILT == VS_FILT_EXACT ? vs_round2int(v) : __double2int_rn(v);
                    if (RAW) {
                        const int m = mbase + u;
                        if (rrow && m >= lo && m < hi) rrow[m] = v;
                    }
                }
#pragma unroll
                for (int u = 0; u < VS_GROUP; u += 2) {
                    uint32_t pk;
                    asm("cvt.pack.sat.s16.s32 %0, %1, %2;" : "=r"(pk) : "r"(qv[u + 1]), "r"(qv[u]));
                    ow[u >> 1] = FILT == VS_FILT_EXACT ? pk : __vmaxs2(pk, 0x80018001u);             /* -32768 -> -32767 */
                }
                *piece = make_uint4(ow[0], ow[1], ow[2], ow[3]);
                w_prev = xw[3];
                mbase += VS_GROUP;
            }
        }
        vs_fence_async();                                   /* the TMA engine will read what this lane wrote */
        vs_pair_barrier(pair);                              /* window w filtered; window w+1 generated */
    }
#undef VS_NC
}

#define VS_RENDER_THREADS(MODE) ((MODE) == VS_MODE_FLOW ? VS_NT : 2 * VS_NT)

/* the second parameter block: the caller's vocal tracts (vs_*_batch_tract), nothing for the preset kernels */
struct VsNoTracts {};
template <bool TRACT> using VsTractParam = typename std::conditional<TRACT, VsTractBlock, VsNoTracts>::type;

template <int MODE, int GEN, bool NOISE, int FILT, bool RAW, bool TRACT>
__global__ void __launch_bounds__(VS_RENDER_THREADS(MODE), MODE == VS_MODE_FLOW ? 4 : 1)
vs_render_kernel(const VsRenderArgs a, const __grid_constant__ VsTractParam<TRACT> tr)
{
    constexpr int WIN = VS_WIN(MODE), TSB = WIN * 2, TILE = 32 * TSB, NGRP = WIN / VS_GROUP;
    constexpr int NT = VS_RENDER_TILES(MODE);
    constexpr bool HASGEN = MODE != VS_MODE_FILTER, HASFILT = MODE != VS_MODE_FLOW;
    constexpr bool FAST = HASGEN && GEN == VS_GEN_FAST;
    static_assert((WIN % VS_RING) == 0 && ((WIN / VS_RING) & 1) == 1, "window = odd number of ring blocks");
    extern __shared__ __align__(128) unsigned char smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    /* Roles.  Rows come in groups of 32 ("pairs"); pair p of a CTA is served by warp p+4, the FILTER warp (F), and
     * warp p, the GENERATOR warp (G): both sit on SM sub-partition p, where F keeps the FP64 pipe busy and G's
     * integer work fills the issue slots in between.  Flow-only mode has G warps alone. */
    const int pair = warp & 3;
    const bool is_f = HASFILT && warp >= 4;                 /* the higher warp id wins the issue slot when both are ready */

    /* shared memory: per pair [NT tiles | period ring | pulse-table cache | row descriptors], then the CTA's RNG states */
    const uint32_t tile_off = (uint32_t)pair * a.warp_bytes;
    const uint32_t ring_off = tile_off + (uint32_t)NT * TILE;
    const uint32_t cache_off = ring_off + a.ring_R * (32u * ((GEN == VS_GEN_FAST && NOISE && MODE != VS_MODE_FILTER) ? 16u : 8u));
    const uint32_t smem_base = (uint32_t)__cvta_generic_to_shared(smem);
    uint32_t *s_rng = reinterpret_cast<uint32_t *>(smem + 4u * a.warp_bytes);      /* [31][VS_NT], NOISE only */

    /* PERSISTENT: the grid has one CTA per render SM (the host keeps the other SMs free for the plan kernels of the
     * next calls); a pair of warps takes blocks of 32 rows round robin until the batch is done.  Rows are sorted
     * longest first inside a preset, so every pair gets a similar mix. */
    const uint32_t n_blocks = a.n_rows / 32u;
    for (uint32_t pb = blockIdx.x * 4u + (uint32_t)pair, cb = blockIdx.x; pb < n_blocks; pb += gridDim.x * 4u, cb += gridDim.x) {
    /* vowel preset of this block of rows: a function of its index and kernel parameters (rows are grouped by preset
     * and padded to whole blocks) */
    int preset = 0;
    if (HASFILT && !TRACT) {
#pragma unroll
        for (int p = 0; p < VS_NUM_PRESETS - 1; p++) preset += pb >= a.cta_end[p] ? 1 : 0;
    }
    /* vocal tract of this CTA's rows (tract kernels): a binary search over the group ends, which are counted in CTAs
     * (tract groups are padded to whole CTAs, so the 4 pairs of a CTA share a tract).  The tract is CTA-uniform, but
     * the compiler does not prove it inside this loop, whose body branches on the warp role: it loads the 22
     * coefficients into registers once per block of rows and the F loop runs three-register DFMAs (DESIGN.md 4.6). */
    const double *tcoef = nullptr;
    if constexpr (TRACT) {
        int t = 0;
#pragma unroll
        for (int s = VS_MAX_TRACTS_I / 2; s > 0; s >>= 1) t += cb >= tr.cta_end[t + s - 1] ? s : 0;
        tcoef = tr.ncoef[t];
    }

    /* ---- the lane's row (lane l of F and lane l of G serve the same row) -------------------------------- */
    const uint32_t t = pb * 32u + (uint32_t)lane;
    const uint32_t chunk_id = t < a.n_rows ? __ldg(a.order + t) : VS_NO_CHUNK;
    bool active = chunk_id != VS_NO_CHUNK;
    int lo = 0, hi = 0, nstart = 0;
    uint32_t stream_id = 0, q0u = 0;
    int16_t *orow = nullptr;
    if (active) {
        const VsChunk ck = a.chunks[chunk_id];
        stream_id = ck.stream;
        orow = a.pcm_out + a.streams[stream_id].out_off;
        lo = (int)ck.emit_lo; hi = (int)ck.emit_hi;
        q0u = ck.first_period;
        nstart = MODE == VS_MODE_FILTER ? (int)ck.gen_target : (int)ck.first_start;
        if (HASGEN) {
            const uint32_t np = __ldg(a.n_periods + stream_id);
            if (q0u >= np || q0u >= a.streams[stream_id].tab_cap) {   /* the plan kernel did not reach this chunk: refuse to walk garbage */
                if (!is_f) atomicExch(a.status, VS_ECUDA);
                active = false; hi = 0; lo = 0; nstart = 0; orow = nullptr;
            }
        }
    }
    const VsStream *st = a.streams + stream_id;
    /* windows are anchored on the 16-byte grid of the row's own address in HBM */
    const int phase = (int)((reinterpret_cast<uintptr_t>(orow) >> 1) & 7);
    const int blk0 = nstart - ((phase + nstart) & 7);
    int nwin = active ? (hi - blk0 + WIN - 1) / WIN : 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) nwin = max(nwin, __shfl_xor_sync(VS_FULL, nwin, o));

    /* =====================================================================================================
     * F: the order-22 recurrence down the lane's own tile row, in place.  One copy of the loop per vowel preset:
     * the coefficients are then constant-bank operands of the DFMAs at literal addresses (a DFMA with two
     * register operands and one constant operand issues every ~2.2 cycles per sub-partition, the three-register
     * form only every ~3.1: tests/tools/dfma_ops.cu).  A CTA runs one preset, so one copy is hot per SM.
     * =================================================================================================== */
    if (is_f) {
        const double gaind = active ? (double)st->gain : 0.0, pred = active ? (double)st->pre : 0.0;
        double *rrow = (RAW && active && a.raw_out) ? a.raw_out + st->out_off : nullptr;
        unsigned char *tiles = smem + tile_off + (uint32_t)lane * TSB;
        if constexpr (TRACT) vs_filter_rows<WIN, NT, FILT, RAW, -1>(tiles, pair, nwin, gaind, pred, rrow, blk0, lo, hi, tcoef);
        else switch (preset) {
#define VS_F_CASE(P) case P: vs_filter_rows<WIN, NT, FILT, RAW, P>(tiles, pair, nwin, gaind, pred, rrow, blk0, lo, hi, nullptr); break;
            VS_F_CASE(0) VS_F_CASE(1) VS_F_CASE(2) VS_F_CASE(3) VS_F_CASE(4) VS_F_CASE(5) VS_F_CASE(6) VS_F_CASE(7) VS_F_CASE(8)
            default: vs_filter_rows<WIN, NT, FILT, RAW, 9>(tiles, pair, nwin, gaind, pred, rrow, blk0, lo, hi, nullptr); break;
#undef VS_F_CASE
        }
        continue;
    }

    /* =====================================================================================================
     * G: generate (or load) window after window, hand finished windows to the TMA engine
     * =================================================================================================== */
    int T2 = 0, DCi = 0, DCs = 0, nper = 0;
    uint32_t pulse_off = 0xffffffffu;
    bool nz = false;
    const unsigned char *ptab = nullptr;                    /* the row's period table */
    if (HASGEN && active) {
        ptab = reinterpret_cast<const unsigned char *>(a.table) + st->tab_off * VS_TAB_ENTRY_BYTES(a.compact);
        T2 = st->T2;
        DCi = (int)ceilf(st->DC);                           /* (float)x < DC  <=>  x < ceil(DC) for integer x */
        DCs = st->DCs;
        nz = (st->flags & VS_F_NOISE) != 0;
        pulse_off = st->pulse_off;
        nper = (int)__ldg(a.n_periods + stream_id);
    }
    const int q0 = (int)q0u;
    const int qlast = nper - 1;
    int q = q0 - 1;                                         /* index of the current period                         */
    /* fast generator: cur = (Adc, Tc), next = (An, Tn); ic = in-period index of the group's first sample.  Past the
     * row's last period it keeps running on periods of amplitude 0 and length tpad (never stored) */
    const int tpad = (HASGEN && active) ? (int)st->tpad : VS_GROUP;
    int ic = 0, Tc = nstart - blk0, Tn = tpad;
    /* ... with glottal noise (VsPeriodN entries): closure instants, noise widths, draws to skip; the generator
     * state as the slot it will overwrite next (byte offset into the lane's column) and its last three values */
    constexpr uint32_t EB = (FAST && NOISE) ? 16u : 8u;     /* ring entry bytes */
    int T3c = VS_BIG_T, T3n = VS_BIG_T, npn = 0, skip = 0;
    double ndwc = 0.0;
    int ndwn = 0;
    uint32_t rf = 3u * VS_NT * 4u, r1 = 0, r2 = 0, r3 = 0;
    double Adc = 0.0;
    float An = 0.0f;
    uint32_t tb = cache_off;                                /* the row's pulse table in shared memory (byte offset) */
    uint32_t qf = (uint32_t)q0;                             /* first period entry not yet requested                */
    const uint32_t Rm = a.ring_R - 1u;
    /* simple generator */
    int si = 0, sT = nstart - blk0, snopen = 0, sT3 = VS_BIG_T, sT4 = 0, snpert = 0, dcs_cur = 0;   /* no noise in the slots before the first period */
    double sAd = 0.0, sKd = 0.0, sndwd = 0.0;
    const double *gtab = a.costab + (pulse_off == 0xffffffffu ? 0u : pulse_off);
    VsRng rng;
    rng.r = s_rng + (uint32_t)pair * 32u + (uint32_t)lane;
    rng.f = 3;

    /* A above 32767: x[T2] = (short)ceil(A) < 0, the falling branch is left at once (flowgen_shimmer.c:329) */
    auto nopen_of = [&](float A, int T) -> int { return min(T, A > 32767.0f ? T2 : 2 * T2); };

    /* Do the pulse tables of this warp's rows fit the pair's cache?  Nearly always (the host sorts rows by table and
     * sizes the cache for the typical warp); a warp with too many distinct tables -- the odd one that collects the
     * first or last chunks of many voices -- falls back to the general generator for its 32 rows. */
    bool wfast = FAST;
    if (FAST) {
        vs_cp_async_wait_all();                             /* ring entries still in flight from the previous block of rows */
        /* pulse tables into the pair's cache: one copy per distinct table of the warp's rows */
        const uint32_t key = active ? pulse_off : 0xffffffffu;
        const uint32_t grp = __match_any_sync(VS_FULL, key);
        const int leader = __ffs((int)grp) - 1;
        /* a table is h[0..T2), f[0..T2) and then zeros up to tpad entries: a sample is ceil(A * table[i]) for EVERY
         * in-period index i, open phase or not (tpad is the same for all rows that share a table) */
        const uint32_t len = active ? 2u * (uint32_t)T2 : 0u;
        const uint32_t mine = (active && lane == leader) ? (uint32_t)tpad : 0u;
        uint32_t incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t up = __shfl_up_sync(VS_FULL, incl, o);
            if (lane >= o) incl += up;
        }
        const uint32_t base = incl - mine;
        const uint32_t lbase = __shfl_sync(VS_FULL, base, leader);
        wfast = __shfl_sync(VS_FULL, incl, 31) <= a.cache_doubles;
#ifdef VS_DEBUG_BOUNDS
        if (active && 2u * (uint32_t)T2 > (uint32_t)tpad) atomicExch(a.status, -110);
        if (cache_off + a.cache_doubles * 8u > 4u * a.warp_bytes) atomicExch(a.status, -111);
#endif
        uint32_t leaders = wfast ? __ballot_sync(VS_FULL, mine > 0u) : 0u;
        double *cache = reinterpret_cast<double *>(smem + cache_off);
        while (leaders) {
            const int L = __ffs((int)leaders) - 1;
            leaders &= leaders - 1u;
            const uint32_t src = __shfl_sync(VS_FULL, pulse_off, L), n = __shfl_sync(VS_FULL, len, L), dst = __shfl_sync(VS_FULL, base, L);
            const uint32_t np = __shfl_sync(VS_FULL, mine, L);
            for (uint32_t k = lane; k < np; k += 32) cache[dst + k] = k < n ? __ldg(a.costab + src + k) : 0.0;
        }
        tb = active ? cache_off + lbase * 8u : cache_off;  /* rows of padding read (and discard) the cache's first entries */
        /* first entries of the period ring, then the first period as `next` of an empty current period that
         * covers the slots before the row's first sample */
        if (active && wfast) {
            const uint32_t want = min((uint32_t)q0 + a.ring_ahead, (uint32_t)nper);
            for (; qf < want; qf++)
                vs_cp_async<EB>(smem_base + ring_off + ((qf & Rm) * 32u + lane) * EB, ptab + (size_t)qf * EB);
        }
        vs_cp_async_wait_all();
        __syncwarp();
        if (active && wfast && q0 <= qlast) {
            if (NOISE) {
                const uint4 e = *reinterpret_cast<const uint4 *>(smem + ring_off + (((uint32_t)q0 & Rm) * 32u + lane) * EB);
                An = __uint_as_float(e.x); Tn = (int)(e.y & 0xffffu); T3n = (int)e.z; ndwn = (int)e.w;
                npn = 0;                                    /* the chunk's first period: its perturbation draws are behind the snapshot */
            } else {
                const uint2 e = *reinterpret_cast<const uint2 *>(smem + ring_off + (((uint32_t)q0 & Rm) * 32u + lane) * EB);
                An = __uint_as_float(e.x); Tn = (int)e.y;
            }
        }
    }
    if (NOISE && HASGEN && active && nz) {
        /* the plan kernel's snapshot is taken after the first period's K draw; it is stored with f = 3:
         * word 3 is the oldest value r[n-31], words 0..2 are r[n-3], r[n-2], r[n-1] */
        for (int k = 0; k < VS_RNG_DEG; k++) rng.r[k * VS_NT] = __ldg(a.rng_snap + (size_t)chunk_id * 32 + k);
        r3 = rng.r[0]; r2 = rng.r[VS_NT]; r1 = rng.r[2 * VS_NT];
    }
    const int16_t *fin = (MODE == VS_MODE_FILTER && active) ? a.flow_in + st->in_off : nullptr;

    /* ---- G, fast: 8 samples of the lane's row, branch free -------------------------------------------- *
     * At most one pitch period ends inside a group (T >= 24).  A sample's in-period index is ic+u in the current
     * period or ic+u-Tc in the next: the unsigned minimum of the two.  Both periods read the same table (T2 and K
     * belong to the stream); the amplitude is picked by the sign of ic+u-Tc.  With the table zero beyond the open
     * phase and A <= 32767, flowgen_shimmer.c:319-335 is  x = max(ceil(A * table[i]), (short)DC):  values below DC
     * become DC (the rising branch's test :320; on the falling branch the first such value ends it, :329, and the
     * factor only decreases from there), the closed phase is ceil(0) = 0 <= DC.
     * Output: the group's 8 samples as 4 words of int16 pairs.  Without noise the maximum is taken two samples at a
     * time after a saturating pack: ceil(A * table[i]) <= 32767 (A <= 32767, table <= 1), and a value below -32768
     * saturates to -32768 <= (short)DC, so max16(sat16(v), DC) == max(v, DC). */
    const uint32_t dcs2 = (uint32_t)(uint16_t)DCs * 0x10001u;
    auto gen_fast = [&](uint32_t (&ow)[VS_GROUP / 2], const bool first) {
        int x[VS_GROUP];
        const int icT = ic - Tc;
        const double Adn = (double)An;
        uint32_t bc = smem_base + tb + (uint32_t)ic * 8u, bn = smem_base + tb + (uint32_t)(icT * 8);   /* table entry of sample 0 in the current / next period */
        asm("" : "+r"(bc), "+r"(bn));                       /* keep them as two addresses: one select per sample, not select + scale + add */
        /* glottal noise (flowgen_shimmer.c:385-399 with T4 == 0): the samples from the closure instant T3 to the
         * period's end each take one random() value.  Bit u of nm: sample u is one of them. */
        uint32_t nm = 0;
        double ndwn_d = 0.0;
        if (NOISE) {
            auto low = [](int k) -> uint32_t { return (1u << min(max(k, 0), VS_GROUP)) - 1u; };     /* bits [0, k) */
            const uint32_t lk = low(-icT);                                                           /* samples of the current period */
            nm = nz ? ((~low(T3c - ic) & lk) | (~low(T3n - icT) & ~lk)) & 0xffu : 0u;
            ndwn_d = (double)ndwn;
        }
        const uint32_t rcol = (uint32_t)__cvta_generic_to_shared(rng.r);
#pragma unroll
        for (int u = 0; u < VS_GROUP; u++) {
            const bool nx = icT + u >= 0;                   /* the sample belongs to the next period */
            const double fac = vs_lds_f64((nx ? bn : bc) + (uint32_t)(u * 8));
            const double A = nx ? Adn : Adc;
            const int v = __double2int_ru(__dmul_rn(A, fac));
            if (!NOISE && !first) { x[u] = v; continue; }   /* the maximum with DC comes after the pack */
            int xv = max(v, first ? (nx ? DCs : 0) : DCs);
            if (NOISE) {
                /* glibc random(): r[n] = r[n-31] + r[n-3]; the slot of r[n-31] takes r[n].  Branch free: every lane
                 * computes the value, a lane that does not draw writes its slot's old content back.  A draw is
                 * a noise sample (bit u of nm) or one of the period's perturbation draws still to be stepped over
                 * (`skip`; they are used up before the period's first noise sample at T3 >= 16) */
                const bool ns = ((nm >> u) & 1u) != 0u;
                const bool dr = ns || skip > 0;
                skip = max(skip - 1, 0);
                const uint32_t old = vs_lds_u32(rcol + rf);
                const uint32_t val = old + r3;
                vs_sts_u32(rcol + rf, dr ? val : old);
                const uint32_t rfn = rf + VS_NT * 4u == VS_RNG_DEG * VS_NT * 4u ? 0u : rf + VS_NT * 4u;
                rf = dr ? rfn : rf;
                r3 = dr ? r2 : r3; r2 = dr ? r1 : r2; r1 = dr ? val : r1;
                const int w = vs_noise_w2((int32_t)(val >> 1), nx ? ndwn_d : ndwc);
                xv = ns ? vs_add_clip(xv, w) : xv;
            }
            x[u] = xv;
        }
#pragma unroll
        for (int u = 0; u < VS_GROUP; u += 2) {
            if (!NOISE && !first) {
                uint32_t pk;
                asm("cvt.pack.sat.s16.s32 %0, %1, %2;" : "=r"(pk) : "r"(x[u + 1]), "r"(x[u]));
                ow[u >> 1] = __vmaxs2(pk, dcs2);
            } else {
                ow[u >> 1] = __byte_perm((uint32_t)x[u], (uint32_t)x[u + 1], 0x5410);
            }
        }
        /* the group's last sample may have been the period's last: promote `next`, read the entry after it */
        const bool pr = icT + VS_GROUP >= 0;
        ic += VS_GROUP;
        if (pr) { ic -= Tc; Adc = Adn; Tc = Tn; q++; }
#ifdef VS_DEBUG_BOUNDS
        if (active && (Tc < VS_GROUP || Tc > tpad || ic < 0 || ic >= Tc)) { atomicExch(a.status, -100 - (Tc > tpad ? 1 : Tc < VS_GROUP ? 2 : 3)); Tc = tpad; ic = 0; }
#endif
        const bool valid = q < qlast;
        if (NOISE) {
            /* the promoted period's jitter / shimmer / K draws come before its noise draws (:283,:298,:325); none of
             * its noise samples lie in this group or in the first half of the next (T3 >= T2 >= 16) */
            if (pr) { T3c = T3n; ndwc = ndwn_d; skip = nz ? npn : 0; }
            while (__any_sync(VS_FULL, skip > 4)) {         /* rejection-heavy streams only: the next group's first samples take four */
                const uint32_t val = vs_lds_u32(rcol + rf) + r3;
                if (skip > 4) {
                    vs_sts_u32(rcol + rf, val);
                    rf = rf + VS_NT * 4u == VS_RNG_DEG * VS_NT * 4u ? 0u : rf + VS_NT * 4u;
                    r3 = r2; r2 = r1; r1 = val;
                    skip--;
                }
            }
            const uint4 e = *reinterpret_cast<const uint4 *>(smem + ring_off + ((((uint32_t)(q + 1)) & Rm) * 32u + lane) * EB);
            An = valid ? __uint_as_float(e.x) : 0.0f;
            Tn = valid ? (int)(e.y & 0xffffu) : tpad;
            npn = valid ? (int)(e.y >> 16) : 0;
            T3n = valid ? (int)e.z : VS_BIG_T;
            ndwn = valid ? (int)e.w : 0;
        } else {
            const uint2 e = *reinterpret_cast<const uint2 *>(smem + ring_off + ((((uint32_t)(q + 1)) & Rm) * 32u + lane) * EB);
            An = valid ? __uint_as_float(e.x) : 0.0f;
            Tn = valid ? (int)e.y : tpad;
        }
    };

    /* keep the ring `ring_ahead` periods ahead of the current one (called once per window) */
    auto ring_refill = [&]() {
        vs_cp_async_wait_all();                             /* what the previous window requested has long landed */
        const uint32_t want = min((uint32_t)(q + 1) + a.ring_ahead, (uint32_t)max(nper, 0));
        for (uint32_t k = 0; k < a.ring_fetch; k++) {
            const uint32_t idx = qf + k;
            if (idx < want) vs_cp_async<EB>(smem_base + ring_off + ((idx & Rm) * 32u + lane) * EB, ptab + (size_t)idx * EB);
        }
        qf = max(qf, min(want, qf + a.ring_fetch));
    };

    /* ---- G, simple: one sample (any parameters: glottal noise, -z, short periods) ---------------------- */
    auto gen_simple = [&]() -> int {
        while (si >= sT) {                                  /* next pitch period */
            q++;
            si = 0;
            if (q > qlast) { sT = VS_BIG_T; snopen = 0; sAd = 0.0; break; }
            dcs_cur = DCs;
            float A;
            if (a.compact == VS_TAB_C8) {
                const uint2 e = __ldg(reinterpret_cast<const uint2 *>(ptab) + q);           /* VsPeriodC */
                A = __uint_as_float(e.x); sT = (int)e.y;
            } else if (a.compact == VS_TAB_N16) {
                const uint4 e = __ldg(reinterpret_cast<const uint4 *>(ptab) + q);           /* VsPeriodN: T4 == 0 */
                A = __uint_as_float(e.x); sT = (int)(e.y & 0xffffu); snpert = (int)(e.y >> 16);
                sT3 = (int)e.z; sT4 = 0; sndwd = (double)(int)e.w;
                if (NOISE && nz && q != q0)
                    for (int k = 0; k < snpert; k++) (void)vs_rng_next<VS_NT>(rng);
            } else {
                const VsPeriod *e = reinterpret_cast<const VsPeriod *>(ptab) + q;
                const double2 ak = __ldg(reinterpret_cast<const double2 *>(e));
                const int4 b = __ldg(reinterpret_cast<const int4 *>(e) + 1);
                A = (float)ak.x; sKd = ak.y;
                sT = b.y & 0xffff; snpert = (int)((uint32_t)b.y >> 16);
                sT3 = b.z & 0xffff; sT4 = (int)((uint32_t)b.z >> 16);
                sndwd = (double)b.w;
                if (NOISE && nz && q != q0)                 /* the period's jitter / shimmer / K draws (:283,:298,:325) */
                    for (int k = 0; k < snpert; k++) (void)vs_rng_next<VS_NT>(rng);
            }
            sAd = (double)A;
            snopen = nopen_of(A, sT);                       /* A above 32767: x[T2] = (short)ceil(A) < 0, the falling branch is left at once */
        }
        int x = dcs_cur;
        if (si < snopen) {
            double fac = __ldg(gtab + si);
            if (a.general_pulse && si >= T2) fac = __dadd_rn(__dsub_rn(__dmul_rn(sKd, fac), sKd), 1.0);      /* :328 */
            const int v = __double2int_ru(__dmul_rn(sAd, fac));
            if (v >= DCi && v <= 32767) x = v;
        }
        if (NOISE && nz && sT != VS_BIG_T && (si < sT4 || si >= sT3)) {                                      /* :385-399 */
            const int32_t r = vs_rng_next<VS_NT>(rng);
            x = vs_add_clip(x, vs_noise_w2(r, sndwd));
        }
        si++;
        return x;
    };

    /* one window of the pair's 32 rows into tile `ti`: generated lane = row, or (filter-only mode) loaded row by
     * row with the lanes along the row, i.e. coalesced */
    auto fill_window = [&](const int w, const int ti) {
        unsigned char *tbase = smem + tile_off + (uint32_t)ti * TILE;
        if (MODE == VS_MODE_FILTER) {
            /* lane = row.  Where the input row has the 16-byte phase of the output row (dense layouts) the lane
             * fetches its window as whole 16-byte pieces, all requested before the first is used: one memory
             * latency per window.  Any other layout, and the pieces that straddle the row's ends, go sample by
             * sample. */
            unsigned char *trow = tbase + (uint32_t)lane * TSB;
            const int wb = blk0 + w * WIN;
            const bool aligned = ((reinterpret_cast<uintptr_t>(fin + blk0)) & 15) == 0;
            uint4 pc[NGRP];
#pragma unroll
            for (int g = 0; g < NGRP; g++) {
                const int m0 = wb + g * VS_GROUP;
                if (aligned && m0 >= nstart && m0 + VS_GROUP <= hi) pc[g] = __ldg(reinterpret_cast<const uint4 *>(fin + m0));
                else {
                    uint32_t h[VS_GROUP];
#pragma unroll
                    for (int u = 0; u < VS_GROUP; u++) {
                        const int m = m0 + u;
                        h[u] = (m >= nstart && m < hi) ? (uint32_t)(uint16_t)__ldg(fin + m) : 0u;
                    }
                    pc[g] = make_uint4(h[0] | (h[1] << 16), h[2] | (h[3] << 16), h[4] | (h[5] << 16), h[6] | (h[7] << 16));
                }
            }
#pragma unroll
            for (int g = 0; g < NGRP; g++) *reinterpret_cast<uint4 *>(trow + g * VS_GROUP * 2) = pc[g];
            return;
        }
        unsigned char *trow = tbase + (uint32_t)lane * TSB;
        auto put = [&](const int g, const uint32_t (&ow)[VS_GROUP / 2]) {
            *reinterpret_cast<uint4 *>(trow + g * VS_GROUP * 2) = make_uint4(ow[0], ow[1], ow[2], ow[3]);
        };
        uint32_t ow[VS_GROUP / 2];
        if (FAST && wfast) {                                /* (the choice of generator is made once per window, not per group) */
            ring_refill();
            if (w == 0) gen_fast(ow, true);
            else gen_fast(ow, false);
            put(0, ow);
#pragma unroll 1
            for (int g = 1; g < NGRP; g++) {
                gen_fast(ow, false);
                put(g, ow);
            }
        } else {
#pragma unroll 1
            for (int g = 0; g < NGRP; g++) {
                int x[VS_GROUP];
#pragma unroll
                for (int u = 0; u < VS_GROUP; u++) x[u] = gen_simple();
#pragma unroll
                for (int u = 0; u < VS_GROUP; u += 2) ow[u >> 1] = __byte_perm((uint32_t)x[u], (uint32_t)x[u + 1], 0x5410);
                put(g, ow);
            }
        }
    };

    /* ---- W: a finished window leaves through the TMA engine: per lane one bulk copy of its row's whole 16-byte
     * pieces inside [lo, hi); the few samples of a stream's unaligned first / last piece go as 2-byte stores ---- */
    auto store_window = [&](const int w, const int ti) {
        const int wb = blk0 + w * WIN;
        const int a0 = max(wb, lo), b0 = min(wb + WIN, hi);
#ifdef VS_DEBUG_BOUNDS
        if (b0 > a0 && (orow == nullptr || a0 < 0 || b0 - wb > WIN || a0 < wb)) { atomicExch(a.status, -120); return; }
#endif
        if (b0 > a0) {
            const uint32_t trow = tile_off + (uint32_t)ti * TILE + (uint32_t)lane * TSB;
            const int a8 = wb + ((a0 - wb + 7) & ~7), b8 = wb + ((b0 - wb) & ~7);
            if (b8 > a8 && !(a.debug & 1)) vs_bulk_s2g(orow + a8, smem_base + trow + (uint32_t)(a8 - wb) * 2u, (uint32_t)(b8 - a8) * 2u);
            const int16_t *tr = reinterpret_cast<const int16_t *>(smem + trow);
            const int hend = min(a8, b0);
            for (int m = a0; m < hend; m++) orow[m] = tr[m - wb];
            for (int m = max(b8, hend); m < b0; m++) orow[m] = tr[m - wb];
        }
        vs_bulk_commit();
    };

    if (!HASFILT) {
        /* ======== flow only: generate, store, next window.  (Storing straight from registers, one 16-byte store per
         * lane and group, was measured slower: 0.166 ms against 0.144 ms on the bench batch -- the L2 sees half
         * sectors -- so the flow leaves through a tile and the TMA engine like everything else.) ======== */
        for (int w = 0; w < nwin; w++) {
            vs_bulk_wait_read<0>();                         /* the copy that last read the tile has finished */
            fill_window(w, 0);
            vs_fence_async();
            store_window(w, 0);
        }
    } else {
        /* ======== G runs one window ahead of F; three tiles: F's, G's, and the one the TMA engine reads ======== */
        int ti = 0;                                         /* tile of window w */
        if (nwin > 0) fill_window(0, 0);
        vs_pair_barrier(pair);                              /* window 0 generated */
        for (int w = 0; w < nwin; w++) {
            const int tn1 = ti == NT - 1 ? 0 : ti + 1;
            if (w + 1 < nwin) {
                vs_bulk_wait_read<1>();                     /* the copy of window w-2 has finished reading tile tn1 */
                fill_window(w + 1, tn1);
            }
            vs_pair_barrier(pair);                          /* window w filtered (and fenced) by F */
            store_window(w, ti);
            ti = tn1;
        }
    }
    vs_bulk_wait_read<0>();                                 /* shared memory must outlive the copies that read it */
    }   /* next block of 32 rows */
}

/* ------------------------------------------------------------------------------------------------
 * host side of the kernel: coefficient upload, shared-memory size, launch
 * ---------------------------------------------------------------------------------------------- */
cudaError_t vs_render_init_device()
{
    static double h[VS_NUM_PRESETS][VS_RING];
    for (int p = 0; p < VS_NUM_PRESETS; p++)
        for (int j = 0; j < VS_RING; j++) h[p][j] = j <= VS_ORDER ? -vs_preset_den[p][j] : 0.0;
    return cudaMemcpyToSymbol(c_ncoef, h, sizeof h);
}

template <int MODE, int GEN, bool NOISE, int FILT, bool RAW, bool TRACT = false>
static cudaError_t vs_go(const VsRenderArgs &a, const VsTractBlock *tb, cudaStream_t s)
{
    const unsigned grid = a.grid;
    const int dyn = 4 * (int)a.warp_bytes + (NOISE ? VS_RNG_DEG * VS_NT * 4 : 0);      /* warp_bytes: per pair of warps */
    /* the attribute is per device and per kernel: set it whenever a launch needs more than the last one did */
    static int granted[16] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 16 && granted[dev] < dyn) {
        const cudaError_t e = cudaFuncSetAttribute(vs_render_kernel<MODE, GEN, NOISE, FILT, RAW, TRACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn);
        if (e != cudaSuccess) return e;
        granted[dev] = dyn;
    } else if (dev >= 16) {
        cudaFuncSetAttribute(vs_render_kernel<MODE, GEN, NOISE, FILT, RAW, TRACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn);
    }
    if constexpr (TRACT) vs_render_kernel<MODE, GEN, NOISE, FILT, RAW, true><<<grid, VS_RENDER_THREADS(MODE), dyn, s>>>(a, *tb);
    else vs_render_kernel<MODE, GEN, NOISE, FILT, RAW, false><<<grid, VS_RENDER_THREADS(MODE), dyn, s>>>(a, VsNoTracts());
    return cudaGetLastError();
}

template <int MODE, int GEN, bool NOISE, bool TRACT>
static cudaError_t vs_go_filt(const VsRenderArgs &a, const VsTractBlock *tb, int filt, cudaStream_t s)
{
    const bool raw = a.raw_out != nullptr;
    if (filt == VS_FILT_EXACT) return raw ? vs_go<MODE, GEN, NOISE, VS_FILT_EXACT, true, TRACT>(a, tb, s) : vs_go<MODE, GEN, NOISE, VS_FILT_EXACT, false, TRACT>(a, tb, s);
    if (raw) return vs_go<MODE, GEN, NOISE, VS_FILT_FMA, true, TRACT>(a, tb, s);
    if (filt == VS_FILT_INT) return vs_go<MODE, GEN, NOISE, VS_FILT_INT, false, TRACT>(a, tb, s);
    return vs_go<MODE, GEN, NOISE, VS_FILT_FMA, false, TRACT>(a, tb, s);
}

template <bool TRACT>
static cudaError_t vs_go_filter_modes(const VsRenderArgs &a, const VsTractBlock *tb, int mode, int gen, bool noise, int filt, cudaStream_t s)
{
    if (mode == VS_MODE_FILTER) return vs_go_filt<VS_MODE_FILTER, VS_GEN_SIMPLE, false, TRACT>(a, tb, filt, s);
    if (gen == VS_GEN_FAST) return noise ? vs_go_filt<VS_MODE_SYNTH, VS_GEN_FAST, true, TRACT>(a, tb, filt, s) : vs_go_filt<VS_MODE_SYNTH, VS_GEN_FAST, false, TRACT>(a, tb, filt, s);
    return noise ? vs_go_filt<VS_MODE_SYNTH, VS_GEN_SIMPLE, true, TRACT>(a, tb, filt, s) : vs_go_filt<VS_MODE_SYNTH, VS_GEN_SIMPLE, false, TRACT>(a, tb, filt, s);
}

/* gen: VS_GEN_FAST / VS_GEN_SIMPLE; filt: VS_FILT_INT / _FMA / _EXACT (raw output forces _FMA or _EXACT);
 * tb: the caller's vocal tracts (synth and filter modes), nullptr for the presets */
cudaError_t vs_launch_render(const VsRenderArgs &a, const VsTractBlock *tb, int mode, int gen, bool noise, int filt, cudaStream_t s)
{
    if (mode == VS_MODE_FLOW) {
        if (gen == VS_GEN_FAST) return noise ? vs_go<VS_MODE_FLOW, VS_GEN_FAST, true, VS_FILT_FMA, false>(a, nullptr, s) : vs_go<VS_MODE_FLOW, VS_GEN_FAST, false, VS_FILT_FMA, false>(a, nullptr, s);
        return noise ? vs_go<VS_MODE_FLOW, VS_GEN_SIMPLE, true, VS_FILT_FMA, false>(a, nullptr, s) : vs_go<VS_MODE_FLOW, VS_GEN_SIMPLE, false, VS_FILT_FMA, false>(a, nullptr, s);
    }
    return tb ? vs_go_filter_modes<true>(a, tb, mode, gen, noise, filt, s) : vs_go_filter_modes<false>(a, nullptr, mode, gen, noise, filt, s);
}
