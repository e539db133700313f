/* vs_formants.cu -- formant analysis of PCM (vs_formant_batch; definitions in include/voicesynth.h, restated in numpy by
 * tests/formant_ref.py).
 *
 *   vs_formant_frame_kernel  one warp per FRAME, so that one long stream spreads over the GPU: the warp finds its stream
 *                            by a binary search of the frame prefix, stages the pre-emphasised, windowed frame in shared
 *                            memory in FP64, forms r[0..p] with lanes along m (p+1 partial sums per lane, then a
 *                            butterfly reduction), runs Levinson-Durbin with lanes along the coefficients, finds the p
 *                            roots with Aberth-Ehrlich (lane j = root j) plus one Newton step, and ranks the kept roots
 *                            by F with a count of the candidates below each lane.  Writes the frame's F and B in FP64.
 *   vs_formant_stats_kernel  one warp per stream, lanes along its frames: FP64 sums (two passes: the means, then the
 *                            squared deviations), the statistics, and the caller's float frame records when asked for.
 */
#include "vs_device.cuh"

#define VS_FMT_NT    128         /* threads per CTA of both kernels                               */
#define VS_FMT_ITERS 64          /* Aberth iteration cap                                          */
#define VS_FMT_TOL   1e-13       /* relative correction at which a root counts as converged       */

/* per-warp shared memory: the frame y[0..max_nw + 32) (zeros past Nw, for the lags), r[0..32], the coefficients
 * c[0..32] and the roots */
__host__ __device__ inline size_t vs_fmt_warp_doubles(uint32_t max_nw) { return (size_t)max_nw + 32 + 33 + 33 + 64; }

/* (a + ib) / (c + id) */
__device__ __forceinline__ void vs_cdiv(double a, double b, double c, double d, double &re, double &im)
{
    const double inv = 1.0 / (c * c + d * d);
    re = (a * c + b * d) * inv;
    im = (b * c - a * d) * inv;
}

/* P(z) and P'(z) of the monic polynomial c[0] = 1, c[1..p] by Horner */
__device__ __forceinline__ void vs_horner(const double *c, uint32_t p, double zr, double zi, double &pr, double &pi, double &dr, double &di)
{
    pr = 1.0; pi = 0.0; dr = 0.0; di = 0.0;
    for (uint32_t j = 1; j <= p; j++) {
        const double ndr = dr * zr - di * zi + pr, ndi = dr * zi + di * zr + pi;
        const double npr = pr * zr - pi * zi + c[j], npi = pr * zi + pi * zr;
        dr = ndr; di = ndi; pr = npr; pi = npi;
    }
}

__global__ void __launch_bounds__(VS_FMT_NT) vs_formant_frame_kernel(const __grid_constant__ VsFormantArgs a)
{
    extern __shared__ double vs_fmt_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t g = (uint64_t)blockIdx.x * (VS_FMT_NT / 32) + (uint64_t)warp;
    if (g >= a.n_frames) return;
    double *y = vs_fmt_smem + (size_t)warp * vs_fmt_warp_doubles(a.max_nw);
    double *rr = y + a.max_nw + 32, *c = rr + 33, *zs = c + 33;

    /* the stream: the last s with frame0[s] <= g (streams without frames have frame0[s] == frame0[s+1]) */
    uint32_t lo = 0, hi = a.n_rows;
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (a.frame0[mid] <= g) lo = mid; else hi = mid;
    }
    const VsFormantRow r = a.rows[lo];
    const uint64_t start = (g - a.frame0[lo]) * (uint64_t)r.H;
    const int16_t *x = a.pcm + r.off + start;
    const double *w = a.win + r.win_off;
    const uint32_t p = a.order, Nw = r.Nw;
    for (uint32_t m = (uint32_t)lane; m < Nw + 32; m += 32) {
        double v = 0.0;
        if (m < Nw) {
            const double prev = (start + m > 0) ? (double)x[(int64_t)m - 1] : 0.0;
            v = ((double)x[m] - r.mu * prev) * w[m];
        }
        y[m] = v;
    }
    __syncwarp();

    /* r[k], k = 0..p: lanes along m */
    double acc[VS_FMT_MAX_ORDER + 1];
#pragma unroll
    for (int k = 0; k <= VS_FMT_MAX_ORDER; k++) acc[k] = 0.0;
    for (uint32_t m = (uint32_t)lane; m < Nw; m += 32) {
        const double ym = y[m];
#pragma unroll
        for (int k = 0; k <= VS_FMT_MAX_ORDER; k++)
            if ((uint32_t)k <= p) acc[k] = __fma_rn(ym, y[m + k], acc[k]);
    }
#pragma unroll
    for (int k = 0; k <= VS_FMT_MAX_ORDER; k++)
        if ((uint32_t)k <= p) {
            const double s = vs_warp_sum(acc[k]);
            if (lane == 0) rr[k] = s;
        }
    __syncwarp();

    uint32_t flags = 0;
    if (rr[0] == 0.0) flags = VS_FRAME_SILENT;

    /* Levinson-Durbin, lane j holds a_{j+1}.  The butterfly gives every lane the same sums, so every lane takes the
     * same branches. */
    double av = 0.0;
    if (!flags) {
        double E = rr[0];
        const uint32_t j1 = (uint32_t)lane + 1;
        for (uint32_t i = 1; i <= p; i++) {
            const double t = vs_warp_sum(j1 < i ? av * rr[i - j1] : 0.0);
            const double k = -(rr[i] + t) / E;
            if (!(fabs(k) < 1.0)) { flags = VS_FRAME_SINGULAR; break; }
            const double partner = __shfl_sync(VS_FULL, av, (int)((i - j1 - 1) & 31));
            if (j1 < i) av = av + k * partner;
            else if (j1 == i) av = k;
            E = E * (1.0 - k * k);
            if (!(E > 0.0)) { flags = VS_FRAME_SINGULAR; break; }
        }
    }

    double zr = 0.0, zi = 0.0;
    bool keep = false;
    double F = 0.0, B = 0.0;
    if (!flags) {
        if (lane == 0) c[0] = 1.0;
        if ((uint32_t)lane < p) c[lane + 1] = av;
        const bool mine = (uint32_t)lane < p;
        if (mine) { zr = a.seed_re[lane]; zi = a.seed_im[lane]; }
        double *zsr = zs, *zsi = zs + 32;
        bool done = false;
        for (int it = 0; it < VS_FMT_ITERS && !done; it++) {
            __syncwarp();
            if (mine) { zsr[lane] = zr; zsi[lane] = zi; }
            __syncwarp();
            bool conv = true;
            if (mine) {
                double pr, pi, dr, di, wr, wi;
                vs_horner(c, p, zr, zi, pr, pi, dr, di);
                vs_cdiv(pr, pi, dr, di, wr, wi);                        /* Newton correction P / P' */
                double sr = 0.0, si = 0.0;                              /* sum_{j != i} 1 / (z_i - z_j) */
                for (uint32_t j = 0; j < p; j++) {
                    if (j == (uint32_t)lane) continue;
                    const double er = zr - zsr[j], ei = zi - zsi[j], inv = 1.0 / (er * er + ei * ei);
                    sr += er * inv;
                    si -= ei * inv;
                }
                const double qr = 1.0 - (wr * sr - wi * si), qi = -(wr * si + wi * sr);
                double d_r, d_i;
                vs_cdiv(wr, wi, qr, qi, d_r, d_i);
                zr -= d_r; zi -= d_i;
                conv = d_r * d_r + d_i * d_i <= VS_FMT_TOL * VS_FMT_TOL * (zr * zr + zi * zi);   /* false for NaN */
            }
            done = __all_sync(VS_FULL, conv);
        }
        if (!done) {
            flags = VS_FRAME_NOCONV;
        } else if (mine) {
            double pr, pi, dr, di, wr, wi;
            vs_horner(c, p, zr, zi, pr, pi, dr, di);
            vs_cdiv(pr, pi, dr, di, wr, wi);
            if (isfinite(wr) && isfinite(wi)) { zr -= wr; zi -= wi; }
            if (zi > 0.0) {
                F = atan2(zi, zr) * r.fs / (2.0 * 3.141592653589793);
                B = -log(hypot(zr, zi)) * r.fs / 3.141592653589793;
                keep = F > 50.0 && F < r.fs / 2.0 - 50.0 && (a.bmax <= 0.0 || B < a.bmax);
            }
        }
    }

    /* rank = kept roots with a smaller F (ties: the lower lane first) */
    const uint32_t kmask = __ballot_sync(VS_FULL, keep);
    uint32_t rank = 0;
    for (int j = 0; j < 32; j++) {
        const double Fj = __shfl_sync(VS_FULL, F, j);
        if (((kmask >> j) & 1u) && (Fj < F || (Fj == F && j < lane))) rank++;
    }
    const uint32_t nf = a.nf;
    const uint32_t found = min((uint32_t)__popc(kmask), nf);
    double *fb = a.fb + g * (2 * (uint64_t)nf);
    if (keep && rank < nf) { fb[rank] = F; fb[nf + rank] = B; }
    if (lane == 0) a.ff[g] = found | (flags << 16);
}

__global__ void __launch_bounds__(VS_FMT_NT) vs_formant_stats_kernel(const __grid_constant__ VsFormantArgs a, vs_formant_stats *stats,
                                                                    vs_formant_frame *frames)
{
    const int lane = threadIdx.x & 31;
    const uint32_t s = blockIdx.x * (VS_FMT_NT / 32) + (threadIdx.x >> 5);
    if (s >= a.n_rows) return;
    const uint64_t g0 = a.frame0[s], g1 = a.frame0[s + 1];
    const uint32_t nf = a.nf;
    const float qnan = VS_QNAN_F;
    uint32_t cnt[VS_MAX_FORMANTS], analysed = 0, unconv = 0;
    double sF[VS_MAX_FORMANTS], sB[VS_MAX_FORMANTS], sQ[VS_MAX_FORMANTS];
#pragma unroll
    for (int k = 0; k < VS_MAX_FORMANTS; k++) { cnt[k] = 0; sF[k] = 0.0; sB[k] = 0.0; sQ[k] = 0.0; }
    for (uint64_t g = g0 + (uint64_t)lane; g < g1; g += 32) {
        const uint32_t v = a.ff[g], found = v & 0xffffu, fl = v >> 16;
        const double *fb = a.fb + g * (2 * (uint64_t)nf);
        if (fl & VS_FRAME_NOCONV) unconv++;
        if (!fl) analysed++;
#pragma unroll
        for (int k = 0; k < VS_MAX_FORMANTS; k++)
            if (!fl && (uint32_t)k < found) { cnt[k]++; sF[k] += fb[k]; sB[k] += fb[nf + k]; }
        if (frames) {
            vs_formant_frame o;
#pragma unroll
            for (int k = 0; k < VS_MAX_FORMANTS; k++) {
                const bool has = !fl && (uint32_t)k < found;
                o.f_hz[k] = has ? (float)fb[k] : qnan;
                o.bw_hz[k] = has ? (float)fb[nf + k] : qnan;
            }
            o.found = fl ? 0u : found;
            o.flags = fl;
            frames[g] = o;
        }
    }
    double mF[VS_MAX_FORMANTS];
#pragma unroll
    for (int k = 0; k < VS_MAX_FORMANTS; k++) {
        cnt[k] = __reduce_add_sync(VS_FULL, cnt[k]);
        sF[k] = vs_warp_sum(sF[k]);
        sB[k] = vs_warp_sum(sB[k]);
        mF[k] = cnt[k] ? sF[k] / (double)cnt[k] : 0.0;
    }
    analysed = __reduce_add_sync(VS_FULL, analysed);
    unconv = __reduce_add_sync(VS_FULL, unconv);
    for (uint64_t g = g0 + (uint64_t)lane; g < g1; g += 32) {
        const uint32_t v = a.ff[g], found = v & 0xffffu, fl = v >> 16;
        const double *fb = a.fb + g * (2 * (uint64_t)nf);
#pragma unroll
        for (int k = 0; k < VS_MAX_FORMANTS; k++)
            if (!fl && (uint32_t)k < found) { const double d = fb[k] - mF[k]; sQ[k] += d * d; }
    }
#pragma unroll
    for (int k = 0; k < VS_MAX_FORMANTS; k++) sQ[k] = vs_warp_sum(sQ[k]);
    if (lane == 0) {
        vs_formant_stats st;
        st.frames = (uint32_t)(g1 - g0);
        st.analysed = analysed;
        st.unconverged = unconv;
        st.reserved = 0;
#pragma unroll
        for (int k = 0; k < VS_MAX_FORMANTS; k++) {
            st.count[k] = cnt[k];
            st.f_mean_hz[k] = cnt[k] ? (float)mF[k] : qnan;
            st.bw_mean_hz[k] = cnt[k] ? (float)(sB[k] / (double)cnt[k]) : qnan;
            st.f_sd_hz[k] = cnt[k] >= 2 ? (float)sqrt(sQ[k] / (double)(cnt[k] - 1)) : qnan;
        }
        stats[s] = st;
    }
}

cudaError_t vs_launch_formants(const VsFormantArgs &a, vs_formant_stats *stats, vs_formant_frame *frames, cudaStream_t s)
{
    const size_t smem = (VS_FMT_NT / 32) * vs_fmt_warp_doubles(a.max_nw) * sizeof(double);
    return vs_launch_frame_kernels(vs_formant_frame_kernel, vs_formant_stats_kernel, a, VS_FMT_NT / 32, smem, VS_FMT_NT, stats, frames, s);
}
