/* vs_analyze.cu -- SURVEY.md 8f row N4: cycle-to-cycle analysis of generated glottal flow on the GPU (F0, local
 * jitter, local shimmer), the measurements the reference's missing `acoustic` tools are described to make
 * (/root/reference README:14-16; no code in the tree, so the definitions are this library's own and are stated in
 * include/voicesynth.h; tests/analysis_ref.py restates them in numpy).
 *
 *   vs_onsets_kernel   one warp per stream, lanes along the stream, 32 samples per step.  A two-threshold trigger
 *                      (armed by x <= lo, fired by x > hi) is a scan over the composition of per-sample state maps
 *                      {arm, disarm, keep}: the state in front of a sample is that of the LAST arm/disarm before it
 *                      -- two ballots and one unsigned compare of the masked masks.  Onsets are written compactly.
 *   vs_cycles_kernel   one warp per stream, lanes along the cycles: length and peak of each cycle, exact integer
 *                      sums of lengths, peaks and absolute first differences, statistics in FP64 by lane 0.
 *   vs_report_kernel   the voice report on top of them (vs_flow_report_batch; vs_vowel_report_batch runs the cycles
 *                      and report kernels on the period marks of vs_marks.cu), below.
 */
#include "vs_device.cuh"

#define VS_AN_NT 128

__global__ void __launch_bounds__(VS_AN_NT) vs_onsets_kernel(const int16_t *flow, const VsAnalyzeRow *rows, uint32_t n_rows,
                                                             uint32_t *onsets, uint32_t *counts)
{
    const int lane = threadIdx.x & 31;
    const uint32_t s = blockIdx.x * (VS_AN_NT / 32) + (threadIdx.x >> 5);
    if (s >= n_rows) return;
    const VsAnalyzeRow r = rows[s];
    const int16_t *x = flow + r.off;
    uint32_t *ons = onsets + r.ons_off;
    const uint32_t below = (1u << lane) - 1u;
    bool armed = true;                                      /* a stream begins in its closed phase */
    uint32_t count = 0;
    for (uint32_t base = 0; base < r.n; base += 32) {
        const uint32_t m = base + (uint32_t)lane;
        const bool valid = m < r.n;
        const int v = valid ? (int)x[m] : 0;
        const uint32_t A = __ballot_sync(VS_FULL, valid && v <= (int)r.lo);     /* arms */
        const uint32_t D = __ballot_sync(VS_FULL, valid && v > (int)r.hi);      /* fires if armed, disarms */
        const uint32_t la = A & below, ld = D & below;
        /* the masks are disjoint: the one with the higher top bit is the larger number */
        const bool armed_here = (la | ld) ? la > ld : armed;
        const bool fire = ((D >> lane) & 1u) && armed_here;
        const uint32_t F = __ballot_sync(VS_FULL, fire);
        if (fire) {
            const uint32_t k = count + (uint32_t)__popc(F & below);
            if (k < r.cap) ons[k] = m;
        }
        count += (uint32_t)__popc(F);
        if (A | D) armed = A > D;
    }
    if (lane == 0) counts[s] = count;
}

__global__ void __launch_bounds__(VS_AN_NT) vs_cycles_kernel(const int16_t *flow, const VsAnalyzeRow *rows, uint32_t n_rows,
                                                             const uint32_t *onsets, const uint32_t *counts, vs_flow_stats *out)
{
    const int lane = threadIdx.x & 31;
    const uint32_t s = blockIdx.x * (VS_AN_NT / 32) + (threadIdx.x >> 5);
    if (s >= n_rows) return;
    const VsAnalyzeRow r = rows[s];
    const int16_t *x = flow + r.off;
    const uint32_t *ons = onsets + r.ons_off;
    const uint32_t K = counts[s];
    vs_flow_stats st;
    st.cycles = 0; st.flags = 0; st.f0_hz = 0.0f; st.jitter_pct = 0.0f; st.shimmer_pct = 0.0f; st.mean_period = 0.0f; st.mean_peak = 0.0f;
    st.onsets = K;
    if (K > r.cap) {                                        /* more onsets than the scratch holds: thresholds inside the noise? */
        st.flags = VS_STATS_OVERFLOW;
        if (lane == 0) out[s] = st;
        return;
    }
    const uint32_t nc = K >= 2 ? K - 1 : 0;                 /* complete cycles */
    long long sT = 0, sP = 0, sdT = 0, sdP = 0;
    int carry_peak = 0;                                     /* peak of the cycle before this step's first */
    for (uint32_t k0 = 0; k0 < nc; k0 += 32) {
        const uint32_t k = k0 + (uint32_t)lane;
        const bool valid = k < nc;
        int T = 0, peak = -32768, Tprev = 0;
        if (valid) {
            const uint32_t o0 = ons[k], o1 = ons[k + 1];
            T = (int)(o1 - o0);
            if (k > 0) Tprev = (int)(o0 - ons[k - 1]);
            for (uint32_t m = o0; m < o1; m++) peak = max(peak, (int)x[m]);
        }
        int pprev = __shfl_up_sync(VS_FULL, peak, 1);
        if (lane == 0) pprev = carry_peak;
        carry_peak = __shfl_sync(VS_FULL, peak, 31);
        if (valid) {
            sT += T; sP += peak;
            if (k > 0) { sdT += abs(T - Tprev); sdP += abs(peak - pprev); }
        }
    }
    sT = vs_warp_sum(sT); sP = vs_warp_sum(sP); sdT = vs_warp_sum(sdT); sdP = vs_warp_sum(sdP);
    if (lane == 0) {
        st.cycles = nc;
        if (nc >= 1) {
            const double mT = (double)sT / (double)nc, mP = (double)sP / (double)nc;
            st.mean_period = (float)mT;
            st.mean_peak = (float)mP;
            st.f0_hz = (float)((double)r.fs / mT);
            if (nc >= 2) {
                st.jitter_pct = (float)(100.0 * ((double)sdT / (double)(nc - 1)) / mT);
                st.shimmer_pct = mP != 0.0 ? (float)(100.0 * ((double)sdP / (double)(nc - 1)) / mP) : 0.0f;
            }
        }
        out[s] = st;
    }
}

/* ---- voice report (vs_flow_report_batch): Praat's jitter and shimmer quotients and a cycle-averaged HNR ----------
 *   vs_report_kernel   one warp per stream, after the two kernels above, whose onset lists and statistics it reads.
 *                      HNR pass: lanes along j, 32*VS_RPT_R values of j per tile held as int64 S_j in registers
 *                      while the loop runs over the cycles; the same reads give each cycle's peak P_k (a warp max,
 *                      written to a list parallel to the onset list), so every sample of a cycle is read once.
 *                      Quotients: lanes along the cycles, exact int64 windowed sums over T_k and over P_k. */
#define VS_RPT_R 16

struct VsWinSums {
    long long s0;          /* sum v_k */
    long long d1;          /* sum_{k>=1} |v_k - v_k-1|, for the periods (the peaks' is the base's shimmer_pct) */
    long long n3;          /* sum_{k=1..K-2} |3 v_k - (v_k-1 + v_k + v_k+1)|  (= sum |v_k+1 - 2 v_k + v_k-1|) */
    long long n5;          /* sum_{k=2..K-3} |5 v_k - (v_k-2 + ... + v_k+2)| */
    long long n11;         /* sum_{k=5..K-6} |11 v_k - (v_k-5 + ... + v_k+5)|, when asked for */
    double    db;          /* sum_{k>=1} |20 log10(v_k / v_k-1)|, when asked for */
    bool      nonpos;      /* some v_k <= 0 */
};

template <bool PEAKS, typename V>
__device__ __forceinline__ VsWinSums vs_window_sums(uint32_t K, int lane, V v)
{
    VsWinSums w = {0, 0, 0, 0, 0, 0.0, false};
    for (uint32_t k = (uint32_t)lane; k < K; k += 32) {
        const long long c = v(k);
        w.s0 += c;
        if (PEAKS) w.nonpos |= c <= 0;
        if (k >= 1) {
            const long long p = v(k - 1);
            if (!PEAKS) w.d1 += llabs(c - p);
            if (PEAKS && c > 0 && p > 0) w.db += fabs(20.0 * log10((double)c / (double)p));
        }
        if (k >= 1 && k + 1 < K) w.n3 += llabs(3 * c - (v(k - 1) + c + v(k + 1)));
        if (k >= 2 && k + 2 < K) w.n5 += llabs(5 * c - (v(k - 2) + v(k - 1) + c + v(k + 1) + v(k + 2)));
        if (PEAKS && k >= 5 && k + 5 < K) {
            long long t = 0;
#pragma unroll
            for (int i = -5; i <= 5; i++) t += v(k + i);
            w.n11 += llabs(11 * c - t);
        }
    }
    w.s0 = vs_warp_sum(w.s0); w.n3 = vs_warp_sum(w.n3); w.n5 = vs_warp_sum(w.n5);
    if (!PEAKS) w.d1 = vs_warp_sum(w.d1);
    if (PEAKS) {
        w.n11 = vs_warp_sum(w.n11);
        w.db = vs_warp_sum(w.db);
        w.nonpos = __any_sync(VS_FULL, w.nonpos);
    }
    return w;
}

__device__ __forceinline__ unsigned __int128 vs_warp_sum_u128(unsigned __int128 v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long lo = __shfl_xor_sync(VS_FULL, (unsigned long long)v, o);
        const unsigned long long hi = __shfl_xor_sync(VS_FULL, (unsigned long long)(v >> 64), o);
        v += ((unsigned __int128)hi << 64) | lo;
    }
    return v;
}

__device__ __forceinline__ double vs_u128_to_double(unsigned __int128 v)
{
    return (double)(unsigned long long)(v >> 64) * 0x1p64 + (double)(unsigned long long)v;
}

__global__ void __launch_bounds__(VS_AN_NT) vs_report_kernel(const int16_t *__restrict__ flow, const VsAnalyzeRow *rows, uint32_t n_rows,
                                                             const uint32_t *__restrict__ onsets, const vs_flow_stats *stats,
                                                             int32_t *__restrict__ peaks, vs_flow_report *out)
{
    const int lane = threadIdx.x & 31;
    const uint32_t s = blockIdx.x * (VS_AN_NT / 32) + (threadIdx.x >> 5);
    if (s >= n_rows) return;
    const VsAnalyzeRow r = rows[s];
    vs_flow_report rep;
    rep.base = stats[s];
    rep.jitter_abs_us = rep.jitter_rap_pct = rep.jitter_ppq5_pct = rep.jitter_ddp_pct = VS_QNAN_F;
    rep.shimmer_db = rep.shimmer_apq3_pct = rep.shimmer_apq5_pct = rep.shimmer_apq11_pct = rep.shimmer_dda_pct = VS_QNAN_F;
    rep.hnr_db = VS_QNAN_F;
    rep.hnr_len = 0; rep.reserved = 0;
    const uint32_t K = rep.base.cycles;                     /* 0 when the onset list overflowed */
    if ((rep.base.flags & VS_STATS_OVERFLOW) || K == 0) {
        if (lane == 0) out[s] = rep;
        return;
    }
    const int16_t *__restrict__ x = flow + r.off;
    const uint32_t *__restrict__ ons = onsets + r.ons_off;
    int32_t *__restrict__ pk = peaks + r.ons_off;

    /* jitter sums and L = min T_k */
    const VsWinSums wt = vs_window_sums<false>(K, lane, [&](uint32_t k) { return (long long)ons[k + 1] - (long long)ons[k]; });
    uint32_t L = 0xffffffffu;
    for (uint32_t k = (uint32_t)lane; k < K; k += 32) L = min(L, ons[k + 1] - ons[k]);
    L = __reduce_min_sync(VS_FULL, L);

    /* HNR sums and peaks: tile t covers j in [j0, j0 + W) of every cycle; the last tile also takes [j0 + W, T_k) for
     * the peaks, so each sample of [o_0, o_K) is read once */
    const uint32_t W = 32u * VS_RPT_R;
    long long E = 0;
    unsigned __int128 H = 0;
    for (uint32_t j0 = 0; j0 < L; j0 += W) {
        const bool last = L - j0 <= W;
        long long S[VS_RPT_R];
#pragma unroll
        for (int q = 0; q < VS_RPT_R; q++) S[q] = 0;
        for (uint32_t kb = 0; kb < K; kb += 32) {
            /* onsets kb .. kb+32 travel in registers: lane i holds o_{kb+i} */
            const uint32_t o_lane = kb + (uint32_t)lane <= K ? ons[kb + lane] : 0u;
            const uint32_t o_next = kb + 32u <= K ? ons[kb + 32u] : 0u;
            const uint32_t nk = min(32u, K - kb);
            for (uint32_t i = 0; i < nk; i++) {
                const uint32_t o0 = __shfl_sync(VS_FULL, o_lane, i);
                uint32_t o1 = __shfl_sync(VS_FULL, o_lane, (i + 1) & 31);
                if (i == 31) o1 = o_next;
                const uint32_t Tk = o1 - o0;
                const int16_t *__restrict__ xc = x + o0;
                int pmax = -32768;
#pragma unroll
                for (int q = 0; q < VS_RPT_R; q++) {
                    const uint32_t j = j0 + (uint32_t)q * 32u + (uint32_t)lane;
                    if (j < L) {
                        const int v = xc[j];
                        S[q] += v;
                        E += v * v;
                        pmax = max(pmax, v);
                    } else if (last && j < Tk) {
                        pmax = max(pmax, (int)xc[j]);
                    }
                }
                if (last)
                    for (uint32_t j = j0 + W + (uint32_t)lane; j < Tk; j += 32) pmax = max(pmax, (int)xc[j]);
                pmax = __reduce_max_sync(VS_FULL, pmax);
                if (lane == 0) pk[kb + i] = j0 == 0 ? pmax : max(pk[kb + i], pmax);
            }
        }
#pragma unroll
        for (int q = 0; q < VS_RPT_R; q++) {
            const unsigned long long a = (unsigned long long)llabs(S[q]);
            H += (unsigned __int128)a * a;
        }
    }
    __syncwarp();                                           /* lane 0's peaks, for every lane */
    const VsWinSums wp = vs_window_sums<true>(K, lane, [&](uint32_t k) { return (long long)pk[k]; });
    E = vs_warp_sum(E);
    H = vs_warp_sum_u128(H);

    if (lane == 0) {
        const double mT = (double)(ons[K] - ons[0]) / (double)K, mP = (double)wp.s0 / (double)K;
        if (K >= 2) {
            rep.jitter_abs_us = (float)(1e6 * ((double)wt.d1 / (double)(K - 1)) / (double)r.fs);
            if (!wp.nonpos) rep.shimmer_db = (float)(wp.db / (double)(K - 1));
            const unsigned __int128 KE = (unsigned __int128)K * (unsigned long long)E;
            const unsigned __int128 D = KE - H;             /* >= 0: (sum_k x_k)^2 <= K sum_k x_k^2 */
            rep.hnr_db = D == 0 ? __int_as_float(0x7f800000) : (float)(10.0 * log10(vs_u128_to_double(H) / vs_u128_to_double(D)));
            rep.hnr_len = L;
        }
        if (K >= 3) {
            rep.jitter_rap_pct = (float)(100.0 * ((double)wt.n3 / 3.0 / (double)(K - 2)) / mT);
            rep.jitter_ddp_pct = (float)(100.0 * ((double)wt.n3 / (double)(K - 2)) / mT);
            if (mP > 0.0) {
                rep.shimmer_apq3_pct = (float)(100.0 * ((double)wp.n3 / 3.0 / (double)(K - 2)) / mP);
                rep.shimmer_dda_pct = (float)(100.0 * ((double)wp.n3 / (double)(K - 2)) / mP);
            }
        }
        if (K >= 5) {
            rep.jitter_ppq5_pct = (float)(100.0 * ((double)wt.n5 / 5.0 / (double)(K - 4)) / mT);
            if (mP > 0.0) rep.shimmer_apq5_pct = (float)(100.0 * ((double)wp.n5 / 5.0 / (double)(K - 4)) / mP);
        }
        if (K >= 11 && mP > 0.0) rep.shimmer_apq11_pct = (float)(100.0 * ((double)wp.n11 / 11.0 / (double)(K - 10)) / mP);
        out[s] = rep;
    }
}

/* the onset kernel when find_onsets (otherwise the onset lists are in place already: the period marks of
 * vs_vowel_report_batch), then the cycles kernel and, when peaks and out are given, the report kernel (peaks: one slot
 * per onset slot) */
cudaError_t vs_launch_analyze(const int16_t *x, const VsAnalyzeRow *rows, uint32_t n_rows, bool find_onsets, uint32_t *onsets,
                              uint32_t *counts, vs_flow_stats *stats, int32_t *peaks, vs_flow_report *out, cudaStream_t s)
{
    const unsigned grid = (n_rows + VS_AN_NT / 32 - 1) / (VS_AN_NT / 32);
    cudaError_t e;
    if (find_onsets) {
        vs_onsets_kernel<<<grid, VS_AN_NT, 0, s>>>(x, rows, n_rows, onsets, counts);
        if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    vs_cycles_kernel<<<grid, VS_AN_NT, 0, s>>>(x, rows, n_rows, onsets, counts, stats);
    if ((e = cudaGetLastError()) != cudaSuccess || !peaks || !out) return e;
    vs_report_kernel<<<grid, VS_AN_NT, 0, s>>>(x, rows, n_rows, onsets, stats, peaks, out);
    return cudaGetLastError();
}
