/* vs_marks.cu -- period marks of vowel PCM for its voice report (vs_vowel_report_batch; definitions in
 * include/voicesynth.h, restated in numpy by tests/vowel_report_ref.py).
 *
 *   vs_marks_kernel  one warp per stream, after the pitch kernels, whose frame records it reads.  The voiced run: lanes
 *                    along the frames, a ballot per 32 frames gives each voiced frame the length of the run ending
 *                    there, and a warp max of (length, ~end) picks the longest, first run.  The marks: a walk that is
 *                    sequential over periods.  Per step the warp stages the reference period and the span of its
 *                    candidates in shared memory, forms E(m_k) with lanes along j, then spreads the candidates over
 *                    the lanes: each forms C(m) and E(m) in exact integers (one broadcast and one conflict-free load
 *                    per term) and keeps its best r; a shuffle argmax with ties to the smaller m picks the next mark.
 *                    Marks go to the onset lists of the report kernels (VsAnalyzeRow::ons_off, at most cap of them),
 *                    the count to counts[], so that vs_cycles_kernel and vs_report_kernel run on them unchanged.
 * Positions are 64-bit where they are formed from a frame index or a period, so rows of 2^31-1 samples stay exact.
 */
#include "vs_device.cuh"

#define VS_MARK_NT 128           /* threads per CTA: four streams */

__device__ __forceinline__ uint64_t vs_mark_lround(double v)   /* lround of a positive value, as C's */
{
    return (uint64_t)llround(v);
}

__global__ void __launch_bounds__(VS_MARK_NT) vs_marks_kernel(const __grid_constant__ VsMarkArgs a)
{
    extern __shared__ int16_t vs_mark_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t s = blockIdx.x * (VS_MARK_NT / 32) + (uint32_t)warp;
    if (s >= a.n_rows) return;
    const VsPitchRow pr = a.prows[s];
    const VsAnalyzeRow ar = a.arows[s];
    const vs_pitch_frame *fr = (const vs_pitch_frame *)a.frames + a.frame0[s];
    const uint32_t nf = (uint32_t)(a.frame0[s + 1] - a.frame0[s]);

    /* the run: key = length << 32 | ~end of the voiced run ending at each frame; the largest is the longest, first run */
    uint64_t best = 0;
    uint32_t cur = 0;                                         /* length of the run reaching the previous step's end */
    for (uint32_t f0 = 0; f0 < nf; f0 += 32) {
        const uint32_t f = f0 + (uint32_t)lane;
        const bool v = f < nf && fr[f].flags == VS_PITCH_VOICED;
        const uint32_t B = __ballot_sync(VS_FULL, v);
        const uint32_t zeros = ~B & (0xffffffffu >> (31 - lane));          /* unvoiced at or below this lane */
        const uint32_t len = !v ? 0u : zeros ? (uint32_t)lane - (31u - (uint32_t)__clz(zeros)) : cur + (uint32_t)lane + 1u;
        if (v) best = max(best, ((uint64_t)len << 32) | (uint32_t)~f);
        cur = __shfl_sync(VS_FULL, len, 31);
    }
    best = vs_warp_max(best);
    if (best == 0) {
        if (lane == 0) { a.counts[s] = 0; a.run[s] = VsMarkRun{0, 0, 0, 0}; }
        return;
    }
    const uint32_t run_frames = (uint32_t)(best >> 32), fb = ~(uint32_t)best, fa = fb - run_frames + 1;
    const uint64_t H = pr.H, rs = (uint64_t)fa * H, re = (uint64_t)fb * H + pr.Nw;

    /* T(t) from the record of the run frame nearest to t */
    const uint64_t half_h = H / 2, half_w = pr.Nw / 2;
    auto period = [&](uint64_t t) {
        uint64_t f = t + half_h >= half_w ? (t + half_h - half_w) / H : 0;
        f = min(max(f, (uint64_t)fa), (uint64_t)fb);
        return pr.fs / (double)fr[f].f0_hz;
    };
    const int16_t *x = a.pcm + ar.off;
    uint32_t *marks = a.marks + ar.ons_off;
    int16_t *xs = vs_mark_smem + (size_t)warp * a.stage;

    /* anchor: the first index of max |x| in the period around the centre of the run's first frame */
    uint64_t m;
    {
        const uint64_t c = rs + half_w;
        const uint32_t L = (uint32_t)vs_mark_lround(period(c));
        const uint64_t a0 = c - L / 2;
        uint64_t key = 0;                                     /* |x| << 32 | ~j: the largest, then the first */
        for (uint32_t j = (uint32_t)lane; j < L; j += 32) key = max(key, ((uint64_t)abs((int)x[a0 + j]) << 32) | (uint32_t)~j);
        key = vs_warp_max(key);
        m = a0 + ~(uint32_t)key;
    }

    uint32_t K = 0;
    for (;;) {
        if (lane == 0 && K < ar.cap) marks[K] = (uint32_t)m;
        K++;
        const double T = period(m);
        const uint64_t L = vs_mark_lround(T);
        const uint64_t lo = m + vs_mark_lround(VS_MARK_STEP_MIN * T), hi = m + vs_mark_lround(VS_MARK_STEP_MAX * T);
        if (hi + L > re) break;                               /* a search cut short by the run's end would pick a wrong period */
        const uint32_t span = (uint32_t)(hi + L - m);
        if (span > a.stage) break;                            /* a guard: the host sizes the stage above any frame's period */
        __syncwarp();
        for (uint32_t j = (uint32_t)lane; j < span; j += 32) xs[j] = x[m + j];
        __syncwarp();

        long long e0 = 0;
        for (uint32_t j = (uint32_t)lane; j < (uint32_t)L; j += 32) { const int v = xs[j]; e0 += v * v; }
        const double de0 = (double)vs_warp_sum(e0);

        /* candidates d = m' - m_k, ascending per lane: a strict > keeps the smaller d of a tie */
        double br = -__longlong_as_double(0x7ff0000000000000ll);
        uint32_t bd = 0xffffffffu;
        const uint32_t d_hi = (uint32_t)(hi - m);
        for (uint32_t d = (uint32_t)(lo - m) + (uint32_t)lane; d <= d_hi; d += 32) {
            long long c = 0, e = 0;
            const int16_t *xd = xs + d;
            for (uint32_t j = 0; j < (uint32_t)L; j++) {
                const int u = xs[j], w = xd[j];
                c += (long long)u * w;
                e += (long long)w * w;
            }
            const double den = de0 * (double)e;
            const double r = den == 0.0 ? 0.0 : (double)c / sqrt(den);
            if (r > br) { br = r; bd = d; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double orr = __shfl_xor_sync(VS_FULL, br, o);
            const uint32_t od = __shfl_xor_sync(VS_FULL, bd, o);
            if (orr > br || (orr == br && od < bd)) { br = orr; bd = od; }
        }
        if (!(br > 0.0)) break;
        m += bd;
    }
    if (lane == 0) {
        a.counts[s] = K;
        a.run[s] = VsMarkRun{fa, run_frames, (uint32_t)rs, (uint32_t)(re - rs)};
    }
}

cudaError_t vs_launch_marks(const VsMarkArgs &a, cudaStream_t s)
{
    const size_t smem = (size_t)(VS_MARK_NT / 32) * a.stage * sizeof(int16_t);
    cudaError_t e = cudaFuncSetAttribute(vs_marks_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    vs_marks_kernel<<<(a.n_rows + VS_MARK_NT / 32 - 1) / (VS_MARK_NT / 32), VS_MARK_NT, smem, s>>>(a);
    return cudaGetLastError();
}
