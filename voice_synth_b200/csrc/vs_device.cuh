/* vs_device.cuh -- device helpers shared by the plan kernels (vs_plan.cu) and the render kernel (vs_render.cu):
 * x86-64 conversion semantics, the constant-divisor division, glibc random() in its per-thread and
 * warp-cooperative forms, pulse / noise sample arithmetic and the reference quantiser; and by the analysis
 * kernels: warp reductions, the stream of a frame and the quiet NaNs. */
#ifndef VS_DEVICE_CUH
#define VS_DEVICE_CUH
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/voicesynth.h"
#include "vs_internal.h"

#define VS_RAND_MAX_D 2147483647.0

#define VS_FULL 0xffffffffu

/* ------------------------------------------------------------------------------------------------
 * conversions with x86-64 semantics (cvttsd2si: out-of-range -> 0x80000000, then keep low 16 bits)
 * ---------------------------------------------------------------------------------------------- */
__device__ __forceinline__ int32_t vs_d2i(double v)
{
    if (!(v > -2147483649.0 && v < 2147483648.0)) return (int32_t)0x80000000u;
    return __double2int_rz(v);
}
__device__ __forceinline__ int16_t vs_d2s(double v)
{
    return (int16_t)(uint16_t)(uint32_t)vs_d2i(v);
}
/* (short)ceil(v) for |v| < 2^31 (every pulse/noise value: |v| <= 1.8*32767 resp. NDW): one F2I */
__device__ __forceinline__ int vs_ceil_s16(double v)
{
    return (int)(int16_t)(uint16_t)(uint32_t)__double2int_ru(v);
}

/* r / d for a CONSTANT d with the reciprocal-multiply + FMA-residual sequence.  Exact (== IEEE
 * division) for every r in [0, 2^31) and both constants used here: checked exhaustively by
 * tests/tools/divcheck.c. */
__device__ __forceinline__ double vs_div_const(double r, double d, double inv)
{
    const double q0 = __dmul_rn(r, inv);
    const double rem = __fma_rn(-q0, d, r);
    return __fma_rn(rem, inv, q0);
}
#define VS_INV_RM  (1.0 / 2147483647.0)
#define VS_RM4     (2147483647.0 * 10000.0)
#define VS_INV_RM4 (1.0 / (2147483647.0 * 10000.0))

/* ------------------------------------------------------------------------------------------------
 * glibc random() TYPE_3 (r[i] = r[i-3] + r[i-31], output >> 1).  State lives in shared memory,
 * word-major ([31][VS_NT]) so that lanes never collide on a bank whatever their private index is.
 * ---------------------------------------------------------------------------------------------- */
struct VsRng {
    uint32_t *r;   /* shared memory base + threadIdx.x */
    int f;         /* front index; back index is f-3 (mod 31) */
};

template <int STRIDE = VS_NT>
__device__ __forceinline__ int32_t vs_rng_next(VsRng &g)
{
    const int b = g.f >= 3 ? g.f - 3 : g.f + 28;
    const uint32_t v = g.r[g.f * STRIDE] + g.r[b * STRIDE];
    g.r[g.f * STRIDE] = v;
    g.f = (g.f == VS_RNG_DEG - 1) ? 0 : g.f + 1;
    return (int32_t)(v >> 1);
}

template <int STRIDE = VS_NT>
__device__ void vs_rng_seed(VsRng &g, uint32_t seed)
{
    int32_t w = (int32_t)(seed ? seed : 1u);
    g.r[0] = (uint32_t)w;
    for (int i = 1; i < VS_RNG_DEG; i++) {          /* 16807*w mod (2^31-1), Schrage, signed */
        const int32_t hi = w / 127773, lo = w % 127773;
        w = 16807 * lo - 2836 * hi;
        if (w < 0) w += 2147483647;
        g.r[i * STRIDE] = (uint32_t)w;
    }
    g.f = 3;
    for (int i = 0; i < 310; i++) (void)vs_rng_next<STRIDE>(g);
}

/* store the state rotated so that a reader may assume f = 3: words 0..2 are the newest, word 3 the oldest */
template <int STRIDE = VS_NT>
__device__ void vs_rng_save(const VsRng &g, uint32_t *dst)
{
    int j = g.f >= 3 ? g.f - 3 : g.f + 28;
    for (int k = 0; k < VS_RNG_DEG; k++) {
        dst[k] = g.r[j * STRIDE];
        j = (j == VS_RNG_DEG - 1) ? 0 : j + 1;
    }
}
/* ------------------------------------------------------------------------------------------------
 * pulse samples (flowgen_shimmer.c:319, :328) and the noise sample (:387, :394, :591-600)
 *   rising : ceil((A*0.5)*(1-c)) == ceil(A*h) with h = 0.5*(1-c) tabulated (scaling by 0.5 is exact)
 *   falling: ceil(A*((K*c - K) + 1.0))
 * ---------------------------------------------------------------------------------------------- */
__device__ __forceinline__ int vs_rising(double Ad, double h)
{
    return vs_ceil_s16(__dmul_rn(Ad, h));
}
__device__ __forceinline__ int vs_falling(double Ad, double Kd, double c)
{
    return vs_ceil_s16(__dmul_rn(Ad, __dadd_rn(__dsub_rn(__dmul_rn(Kd, c), Kd), 1.0)));
}
__device__ __forceinline__ int vs_noise_w(int32_t r, int32_t ndw)
{
    const double u = vs_div_const((double)r, VS_RAND_MAX_D, VS_INV_RM);
    const double nd = (double)ndw;
    return vs_ceil_s16(__dsub_rn(__dmul_rn(u, nd), __dmul_rn(nd, 0.5)));
}
/* truncate((float)x + w): both are 16-bit integers, so the float sum is exact and ceil is a no-op */
__device__ __forceinline__ int vs_add_clip(int x, int w)
{
    const int s = x + w;
    return s > 32767 ? 32767 : (s < -32767 ? -32767 : s);
}


/* ---- noise: the warp steps ONE row's random() 31 values at a time ------------------------------------
 * glibc TYPE_3 is r[n] = r[n-31] + r[n-3] (mod 2^32), output r[n] >> 1.  With lane l < 31 holding
 * st[l] = r[n-31+l], the next 31 words are prefix sums along the three stride-3 chains:
 *     new[l] = st[l] + (l < 3 ? st[28+l] : new[l-3])
 * i.e. an inclusive scan with shuffle distances 3, 6, 12, 24 (chains are at most 11 long). */
__device__ __forceinline__ uint32_t vs_rng_round(uint32_t st, int lane)
{
    const uint32_t wrap = __shfl_sync(VS_FULL, st, (lane + 28) & 31);
    uint32_t v = st + (lane < 3 ? wrap : 0u), u;
    u = __shfl_up_sync(VS_FULL, v, 3);  if (lane >= 3)  v += u;
    u = __shfl_up_sync(VS_FULL, v, 6);  if (lane >= 6)  v += u;
    u = __shfl_up_sync(VS_FULL, v, 12); if (lane >= 12) v += u;
    u = __shfl_up_sync(VS_FULL, v, 24); if (lane >= 24) v += u;
    return v;
}

/* srandom() for the warp-cooperative generator: every lane runs the 30 Schrage steps and keeps the word that
 * is (lane)-th oldest once f = 3, i.e. word (lane+3) mod 31; the 310 discarded values are 10 rounds. */
__device__ __forceinline__ uint32_t vs_rng_seed_warp(uint32_t seed, int lane)
{
    int32_t w = (int32_t)(seed ? seed : 1u);
    const int want = (lane + 3) % VS_RNG_DEG;
    uint32_t rs = (uint32_t)w;
    for (int i = 1; i < VS_RNG_DEG; i++) {
        const int32_t hi = w / 127773, lo = w % 127773;
        w = 16807 * lo - 2836 * hi;
        if (w < 0) w += 2147483647;
        if (i == want) rs = (uint32_t)w;
    }
    for (int k = 0; k < 10; k++) rs = vs_rng_round(rs, lane);
    return rs;
}

/* advance the row's generator by m values; they go to out[0..m) when out is not NULL.  Returns the new
 * state (lanes 0..30).  m is warp-uniform. */
__device__ __forceinline__ uint32_t vs_rng_gen(uint32_t st, int m, int lane, int32_t *out)
{
    int done = 0;
    for (; m - done >= VS_RNG_DEG; done += VS_RNG_DEG) {
        st = vs_rng_round(st, lane);
        if (out && lane < VS_RNG_DEG) out[done + lane] = (int32_t)(st >> 1);
    }
    const int u = m - done;
    if (u > 0) {                                     /* part of a round: the state window slides by u words */
        const uint32_t nx = vs_rng_round(st, lane);
        if (out && lane < u) out[done + lane] = (int32_t)(nx >> 1);
        const int src = lane + u;
        const uint32_t keep = __shfl_sync(VS_FULL, st, src & 31);
        const uint32_t fresh = __shfl_sync(VS_FULL, nx, (src - VS_RNG_DEG) & 31);
        st = src < VS_RNG_DEG ? keep : fresh;
    }
    return st;
}


/* vowel_new.c:413-427, literally: round half DOWN, clip to +-32767 */
__device__ __forceinline__ int vs_round2int(double v)
{
    const double dec = __dsub_rn(v, floor(v));
    if (dec > 0.5) v = __dadd_rn(v, 1.0);
    if (v > 32767.0) v = 32767.0;
    else if (v < -32767.0) v = -32767.0;
    return (int)vs_d2s(floor(v));
}

/* ------------------------------------------------------------------------------------------------
 * analysis kernels (vs_analyze.cu, vs_formants.cu, vs_pitch.cu, vs_marks.cu): warp reductions whose butterfly gives
 * every lane the result, the stream of a frame, and the quiet NaN their records hold where a value is undefined
 * ---------------------------------------------------------------------------------------------- */
#define VS_QNAN_F __int_as_float(0x7fc00000)
#define VS_QNAN_D __longlong_as_double(0x7ff8000000000000ll)

template <class T>
__device__ __forceinline__ T vs_warp_sum(T v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(VS_FULL, v, o);
    return v;
}
template <class T>
__device__ __forceinline__ T vs_warp_max(T v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(VS_FULL, v, o));
    return v;
}
template <class T>
__device__ __forceinline__ T vs_warp_min(T v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(VS_FULL, v, o));
    return v;
}

/* the stream of frame g: the last s with frame0[s] <= g (streams without frames have frame0[s] == frame0[s+1]) */
__device__ __forceinline__ uint32_t vs_frame_stream(const uint64_t *frame0, uint32_t n_rows, uint64_t g)
{
    uint32_t lo = 0, hi = n_rows;
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (frame0[mid] <= g) lo = mid; else hi = mid;
    }
    return lo;
}

/* the launches of a frame-wise call (formants, pitch): the frame kernel, one warp per frame and `warps` of them per CTA
 * with `smem` bytes of dynamic shared memory, when there are frames; then the stats kernel, one warp per stream in CTAs
 * of stats_nt threads */
template <class Args, class Stats, class Frame>
cudaError_t vs_launch_frame_kernels(void (*frame_kernel)(Args), void (*stats_kernel)(Args, Stats *, Frame *), const Args &a,
                                    uint32_t warps, size_t smem, uint32_t stats_nt, Stats *stats, Frame *frames, cudaStream_t s)
{
    if (a.n_frames) {
        cudaError_t e = cudaFuncSetAttribute(frame_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        const uint64_t grid = (a.n_frames + warps - 1) / warps;
        if (grid > 0x7fffffffull) return cudaErrorInvalidConfiguration;
        frame_kernel<<<(unsigned)grid, 32 * warps, smem, s>>>(a);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    stats_kernel<<<(a.n_rows + stats_nt / 32 - 1) / (stats_nt / 32), stats_nt, 0, s>>>(a, stats, frames);
    return cudaGetLastError();
}

#endif