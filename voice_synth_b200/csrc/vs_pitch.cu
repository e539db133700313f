/* vs_pitch.cu -- pitch and harmonicity of PCM (vs_pitch_batch; definitions in include/voicesynth.h, restated in numpy
 * by tests/pitch_ref.py).
 *
 *   vs_pitch_frame_kernel  one warp per FRAME, so that one long stream spreads over the GPU: the warp finds its stream
 *                          by a binary search of the frame prefix, stages the mean-free, windowed frame in shared
 *                          memory in FP64, forms r_a(0) with lanes along m and r_a(tau_lo-1 .. tau_hi+1) with lanes
 *                          along tau (each lane a run of K consecutive lags, register-blocked), normalises by r_a(0)
 *                          and the host's window correction, and picks the strongest candidate with lanes along tau
 *                          and a warp argmax.  Writes tau*, r*, the local peak and the flags in FP64.
 *   vs_pitch_stats_kernel  one warp per stream, lanes along its frames: the stream's peak G, the QUIET and VOICED
 *                          rules, FP64 sums in two passes (the means, then the squared deviations), the statistics,
 *                          and the caller's float frame records when asked for.
 */
#include "vs_device.cuh"

#define VS_PITCH_NT   128        /* threads per CTA of the stats kernel, and most of the frame kernel's    */
#define VS_PITCH_KMAX 13         /* most lags per lane and pass (odd: see vs_pitch_lags)                   */

/* r_a(tau) for tau = t_first .. t_end-1 into rr[tau - t_first].  Lane l of a pass owns the K lags tl = t0 + l K ..
 * tl + K - 1 and walks m: per step one broadcast load of y[m] and one load of y[m + tl + K - 1] into a ring of K
 * registers feed K FMAs.  The ring index is a compile-time constant because the loop over m is unrolled K times.
 * K is odd, so the lanes' ring loads (K doubles apart) fall on distinct bank pairs.  y is zero past Nw (32 doubles
 * are enough for 2K - 1 < 32), so the terms past a lag's range add exact zeros. */
template <int K>
__device__ __forceinline__ void vs_pitch_lags(const double *y, double *rr, uint32_t Nw, uint32_t t_first, uint32_t t_end, int lane)
{
    for (uint32_t t0 = t_first; t0 < t_end; t0 += 32u * K) {
        const uint32_t tl = t0 + (uint32_t)lane * K;
        if (tl >= t_end) continue;
        double acc[K], ring[K];
#pragma unroll
        for (int k = 0; k < K; k++) { acc[k] = 0.0; ring[k] = y[tl + k]; }
        const uint32_t mlen = Nw - tl;                        /* tl < t_end <= Nw - 1 */
        for (uint32_t m = 0; m < mlen; m += K) {
#pragma unroll
            for (int j = 0; j < K; j++) {
                const double ym = y[m + j];
#pragma unroll
                for (int k = 0; k < K; k++) acc[k] = __fma_rn(ym, ring[(j + k) % K], acc[k]);
                ring[j] = y[m + j + tl + K];
            }
        }
#pragma unroll
        for (int k = 0; k < K; k++)
            if (tl + k < t_end) rr[tl + k - t_first] = acc[k];
    }
}

__global__ void __launch_bounds__(VS_PITCH_NT) vs_pitch_frame_kernel(const __grid_constant__ VsPitchArgs a)
{
    extern __shared__ double vs_pitch_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t g = (uint64_t)blockIdx.x * a.warps + (uint64_t)warp;
    if (g >= a.n_frames) return;

    const uint32_t sid = vs_frame_stream(a.frame0, a.n_rows, g);
    const VsPitchRow r = a.rows[sid];
    const int16_t *x = a.pcm + r.off + (g - a.frame0[sid]) * (uint64_t)r.H;
    const uint32_t Nw = r.Nw, L = r.tau_hi - r.tau_lo + 3;
    const double *w = a.tab + r.tab, *cw = w + Nw;
    double *y = vs_pitch_smem + (size_t)warp * a.warp_doubles;
    double *rr = y + Nw + 32;                                 /* r(tau) at rr[tau - (tau_lo - 1)] */

    /* mean (an exact integer sum), y = (x - mean) w with zeros past Nw, the local peak and r_a(0) */
    int sum = 0;
    for (uint32_t m = (uint32_t)lane; m < Nw; m += 32) sum += x[m];
    const double mu = (double)__reduce_add_sync(VS_FULL, sum) / (double)Nw;
    double peak = 0.0, e = 0.0;
    for (uint32_t m = (uint32_t)lane; m < Nw + 32; m += 32) {
        double v = 0.0;
        if (m < Nw) {
            const double am = (double)x[m] - mu;
            peak = fmax(peak, fabs(am));
            v = am * w[m];
            e = __fma_rn(v, v, e);
        }
        y[m] = v;
    }
    peak = vs_warp_max(peak);
    e = vs_warp_sum(e);                                       /* the butterfly gives every lane the same sum */
    if (e == 0.0) {
        if (lane == 0) a.cand[g] = VsPitchCand{VS_QNAN_D, VS_QNAN_D, peak, VS_PITCH_SILENT, 0u};
        return;
    }
    __syncwarp();

    /* lags tau_lo-1 .. tau_hi+1: as few passes as K <= VS_PITCH_KMAX allows, K odd */
    const uint32_t passes = (L + 32 * VS_PITCH_KMAX - 1) / (32 * VS_PITCH_KMAX);
    const uint32_t K = ((L + 32 * passes - 1) / (32 * passes)) | 1u;
    const uint32_t t_first = r.tau_lo - 1, t_end = r.tau_hi + 2;
    switch (K) {
    case 1:  vs_pitch_lags<1>(y, rr, Nw, t_first, t_end, lane); break;
    case 3:  vs_pitch_lags<3>(y, rr, Nw, t_first, t_end, lane); break;
    case 5:  vs_pitch_lags<5>(y, rr, Nw, t_first, t_end, lane); break;
    case 7:  vs_pitch_lags<7>(y, rr, Nw, t_first, t_end, lane); break;
    case 9:  vs_pitch_lags<9>(y, rr, Nw, t_first, t_end, lane); break;
    case 11: vs_pitch_lags<11>(y, rr, Nw, t_first, t_end, lane); break;
    default: vs_pitch_lags<13>(y, rr, Nw, t_first, t_end, lane); break;
    }
    __syncwarp();
    for (uint32_t i = (uint32_t)lane; i < L; i += 32) rr[i] = rr[i] / e * cw[i];
    __syncwarp();

    /* candidates, lanes along tau in ascending order (a strict > keeps the smaller tau of a tie), then a warp argmax */
    double bS = -__longlong_as_double(0x7ff0000000000000ll), bt = VS_QNAN_D, br = VS_QNAN_D;
    uint32_t bi = 0xffffffffu;
    for (uint32_t t = r.tau_lo + (uint32_t)lane; t <= r.tau_hi; t += 32) {
        const uint32_t i = t - r.tau_lo + 1;
        const double pa = rr[i - 1], pb = rr[i], pc = rr[i + 1];
        if (pb > pa && pb >= pc && pb > 0.0) {
            const double d = 0.5 * (pa - pc) / (pa - 2.0 * pb + pc);
            const double ts = (double)t + d;
            double rs = pb - 0.25 * (pa - pc) * d;
            if (rs > 1.0) rs = 1.0 / rs;
            const double S = rs - a.octave_cost * log2(a.f_min * ts / r.fs);
            if (S > bS) { bS = S; bt = ts; br = rs; bi = t; }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double oS = __shfl_xor_sync(VS_FULL, bS, o), ot = __shfl_xor_sync(VS_FULL, bt, o);
        const double orr = __shfl_xor_sync(VS_FULL, br, o);
        const uint32_t oi = __shfl_xor_sync(VS_FULL, bi, o);
        if (oS > bS || (oS == bS && oi < bi)) { bS = oS; bt = ot; br = orr; bi = oi; }
    }
    if (lane == 0) a.cand[g] = VsPitchCand{bt, br, peak, bi == 0xffffffffu ? VS_PITCH_NOPEAK : 0u, 0u};
}

/* a frame's flags after the stream rules, and its F0 (voiced) and HNR (periodic) */
__device__ __forceinline__ uint32_t vs_pitch_classify(const VsPitchCand &c, double quiet, double voicing, double fs,
                                                      double &f0, double &hnr)
{
    uint32_t fl = c.flags;
    if (!fl && c.peak < quiet) fl = VS_PITCH_QUIET;
    if (fl) return fl;
    hnr = 10.0 * log10(c.r / (1.0 - c.r));
    if (!(c.r >= voicing)) return 0u;
    f0 = fs / c.tau;
    return VS_PITCH_VOICED;
}

__global__ void __launch_bounds__(VS_PITCH_NT) vs_pitch_stats_kernel(const __grid_constant__ VsPitchArgs a, vs_pitch_stats *stats,
                                                                    vs_pitch_frame *frames)
{
    const int lane = threadIdx.x & 31;
    const uint32_t s = blockIdx.x * (VS_PITCH_NT / 32) + (threadIdx.x >> 5);
    if (s >= a.n_rows) return;
    const uint64_t g0 = a.frame0[s], g1 = a.frame0[s + 1];
    const double fs = a.rows[s].fs;
    const float qnan = VS_QNAN_F;
    double G = 0.0;
    for (uint64_t g = g0 + (uint64_t)lane; g < g1; g += 32) G = fmax(G, a.cand[g].peak);
    const double quiet = a.silence * vs_warp_max(G);

    uint32_t periodic = 0, voiced = 0;
    double sf = 0.0, sh = 0.0, sr = 0.0, lo = __longlong_as_double(0x7ff0000000000000ll), hi = -lo;
    for (uint64_t g = g0 + (uint64_t)lane; g < g1; g += 32) {
        const VsPitchCand c = a.cand[g];
        double f0 = 0.0, hnr = 0.0;
        const uint32_t fl = vs_pitch_classify(c, quiet, a.voicing, fs, f0, hnr);
        if (!fl || fl == VS_PITCH_VOICED) { periodic++; sh += hnr; sr += c.r; }
        if (fl == VS_PITCH_VOICED) { voiced++; sf += f0; lo = fmin(lo, f0); hi = fmax(hi, f0); }
        if (frames) {
            vs_pitch_frame o;
            o.f0_hz = fl == VS_PITCH_VOICED ? (float)f0 : qnan;
            o.strength = fl & (VS_PITCH_SILENT | VS_PITCH_NOPEAK) ? qnan : (float)c.r;
            o.hnr_db = !fl || fl == VS_PITCH_VOICED ? (float)hnr : qnan;
            o.flags = fl;
            frames[g] = o;
        }
    }
    periodic = __reduce_add_sync(VS_FULL, periodic);
    voiced = __reduce_add_sync(VS_FULL, voiced);
    sf = vs_warp_sum(sf);
    sh = vs_warp_sum(sh);
    sr = vs_warp_sum(sr);
    lo = vs_warp_min(lo);
    hi = vs_warp_max(hi);
    const double mf = voiced ? sf / (double)voiced : 0.0, mh = periodic ? sh / (double)periodic : 0.0;
    double qf = 0.0, qh = 0.0;
    for (uint64_t g = g0 + (uint64_t)lane; g < g1; g += 32) {
        const VsPitchCand c = a.cand[g];
        double f0 = 0.0, hnr = 0.0;
        const uint32_t fl = vs_pitch_classify(c, quiet, a.voicing, fs, f0, hnr);
        if (!fl || fl == VS_PITCH_VOICED) { const double d = hnr - mh; qh += d * d; }
        if (fl == VS_PITCH_VOICED) { const double d = f0 - mf; qf += d * d; }
    }
    qf = vs_warp_sum(qf);
    qh = vs_warp_sum(qh);
    if (lane == 0) {
        vs_pitch_stats st;
        st.frames = (uint32_t)(g1 - g0);
        st.periodic = periodic;
        st.voiced = voiced;
        st.f0_mean_hz = voiced ? (float)mf : qnan;
        st.f0_sd_hz = voiced >= 2 ? (float)sqrt(qf / (double)(voiced - 1)) : qnan;
        st.f0_min_hz = voiced ? (float)lo : qnan;
        st.f0_max_hz = voiced ? (float)hi : qnan;
        st.hnr_mean_db = periodic ? (float)mh : qnan;
        st.hnr_sd_db = periodic >= 2 ? (float)sqrt(qh / (double)(periodic - 1)) : qnan;
        st.strength_mean = periodic ? (float)(sr / (double)periodic) : qnan;
        st.reserved[0] = st.reserved[1] = 0u;
        stats[s] = st;
    }
}

cudaError_t vs_launch_pitch(const VsPitchArgs &a, vs_pitch_stats *stats, vs_pitch_frame *frames, cudaStream_t s)
{
    const size_t smem = (size_t)a.warps * a.warp_doubles * sizeof(double);
    return vs_launch_frame_kernels(vs_pitch_frame_kernel, vs_pitch_stats_kernel, a, a.warps, smem, VS_PITCH_NT, stats, frames, s);
}
