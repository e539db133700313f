/* vs_plan.cu -- the sequential half of flowgen_shimmer.c:246-423 on sm_100a, plus vowel -n.
 *
 *   vs_plan_kernel       one THREAD per stream: glibc random() state, jitter and shimmer random walks with
 *                        their rejection loops, the closure-speed draw, and (with -n) the pulse power and the
 *                        number of noise draws.  Emits a period table and, per time-chunk, the period the chunk
 *                        starts in plus the RNG state there.  The throughput form (many streams).
 *   vs_plan_warp_kernel  the same table from one WARP per stream: random() 31 values per step by
 *                        shuffles, the values' meanings worked out lane-parallel, the walk warp-uniform.
 *                        The latency form (few or long streams, glottal noise).
 *   vs_vnoise_kernel     vowel -n (vowel_new.c:302-324), one warp per stream.
 *
 * The render kernel (vs_render.cu) turns the period table into samples.
 * Every operation that decides an integer (period length, amplitude, sample value, draw count) is
 * written with explicit round-to-nearest intrinsics in the reference's evaluation order, so those
 * results are bit-exact.
 */
#include "vs_batch_plan.h"
#include "vs_device.cuh"

/* ================================================================================================
 * PLAN: one thread per stream
 * ============================================================================================== */
/* step over n random() values (the period's noise draws are the render kernel's business).  Three at a time: value k
 * needs r[k-31] from the state array and r[k-3], which for the next three values are the three just made -- they stay
 * in registers, so consecutive trios depend on each other through one integer add only, the loads of the old
 * values run ahead and the stores trail behind. */
template <int STRIDE>
__device__ __forceinline__ void vs_rng_skip(VsRng &g, uint32_t n)
{
    if (n >= 3) {
        int f = g.f;
        int b = f >= 3 ? f - 3 : f + 28;
        uint32_t p0 = g.r[b * STRIDE];
        b = b == VS_RNG_DEG - 1 ? 0 : b + 1;
        uint32_t p1 = g.r[b * STRIDE];
        b = b == VS_RNG_DEG - 1 ? 0 : b + 1;
        uint32_t p2 = g.r[b * STRIDE];
        do {
            const int f0 = f, f1 = f0 == VS_RNG_DEG - 1 ? 0 : f0 + 1, f2 = f1 == VS_RNG_DEG - 1 ? 0 : f1 + 1;
            p0 += g.r[f0 * STRIDE];
            p1 += g.r[f1 * STRIDE];
            p2 += g.r[f2 * STRIDE];
            g.r[f0 * STRIDE] = p0;
            g.r[f1 * STRIDE] = p1;
            g.r[f2 * STRIDE] = p2;
            f = f2 == VS_RNG_DEG - 1 ? 0 : f2 + 1;
            n -= 3;
        } while (n >= 3);
        g.f = f;
    }
    for (; n > 0; n--) (void)vs_rng_next<STRIDE>(g);
}

/* one period into the table, in the format the render kernel asked for */
__device__ __forceinline__ void vs_store_period(void *table, int fmt, uint64_t idx, float A, float Knew, uint32_t start, int T,
                                                uint32_t nd, int T3, int T4, int ndw)
{
    if (fmt == VS_TAB_C8) {
        VsPeriodC e;
        e.A = A; e.T = (uint32_t)T;
        reinterpret_cast<VsPeriodC *>(table)[idx] = e;
    } else if (fmt == VS_TAB_N16) {
        reinterpret_cast<uint4 *>(table)[idx] = make_uint4(__float_as_uint(A), (uint32_t)T | (nd << 16), (uint32_t)T3, (uint32_t)ndw);
    } else {
        VsPeriod e;
        e.Ad = (double)A; e.Kd = (double)Knew; e.start = start;
        e.T_np = (uint32_t)T | (nd << 16);
        e.T34 = (uint32_t)T3 | ((uint32_t)T4 << 16);
        e.ndw = ndw;
        reinterpret_cast<VsPeriod *>(table)[idx] = e;
    }
}

/* PULSE: some stream of the batch needs the open phase evaluated in the plan (glottal noise, period log).  Without it
 * the kernel is the two random walks alone and fits 64 registers: NT = 1024 streams per CTA, half the SMs kept off
 * the render kernel */
template <bool LOG, bool PULSE, int NT>
__global__ void __launch_bounds__(NT, 1) vs_plan_kernel(const VsPlanArgs a)
{
    extern __shared__ __align__(16) uint32_t s_rng[];                  /* [31][NT] RNG states (+ padding up to VS_PLAN_SMEM) */
    const uint32_t s = blockIdx.x * NT + threadIdx.x;
    if (s >= a.n_streams) return;
    const VsStream st = a.streams[s];
    VsRng g;
    g.r = s_rng + threadIdx.x;
    vs_rng_seed<NT>(g, st.seed);                                             /* flowgen_shimmer.c:241 */

    const bool do_jit = (st.flags & VS_F_JITTER) && st.jitter != 0.0f;    /* :248 */
    const bool do_shm = (st.flags & VS_F_SHIMMER) && st.shimmer != 0.0f;  /* :295 */
    const bool noise = PULSE && (st.flags & VS_F_NOISE) != 0;             /* :373 */
    const bool pulse = PULSE && (LOG || noise);
    const int P = st.P, T2 = st.T2;
    const float Pf = (float)P, ampf = (float)st.amp;
    const float t_hi = __fmul_rn(1.2f, Pf), t_lo = __fmul_rn(0.8f, Pf);
    const float a_hi = __fmul_rn(1.8f, ampf), a_lo = __fmul_rn(0.2f, ampf);
    const double jit = (double)st.jitter, shm = (double)st.shimmer;
    const double jit2 = __dmul_rn(2.0, jit), shm2 = __dmul_rn(2.0, shm);
    const double P2 = __dmul_rn(2.0, (double)P), amp2 = __dmul_rn(2.0, (double)st.amp);
    const double Kbase = (double)st.K, kv2 = (double)__fmul_rn(2.0f, st.Kvar);
    const double *ht = a.costab + st.cos_off;      /* h[0..T2) = 0.5*(1-c), then c[0..T2) */
    const double *ct = ht + T2;
    const int DCi = (int)ceilf(st.DC);             /* (float)x < DC  <=>  x < ceil(DC) for integer x */
    const int DCs = st.DCs;

    int T = P, T4 = 0, ndw = 0;
    float dper = 0.0f, dsh = 0.0f;
    uint32_t count = 0, np = 0, next_c = 0;
    VsChunk *chunks = a.chunks + st.chunk0;
    uint32_t next_target = st.n_chunks ? chunks[0].gen_target : 0xffffffffu;
    vs_period_rec *log = LOG ? (vs_period_rec *)a.log + st.log_off : nullptr;
    int guard = 0;

    do {
        uint32_t nd = 0;
        if (do_jit) {                                                     /* :276-290 */
            const double prev = (double)dper;
            float cur;
            do {
                const int32_t r = vs_rng_next<NT>(g); nd++;
                double t = vs_div_const((double)r, VS_RM4, VS_INV_RM4);
                t = __dmul_rn(__dmul_rn(t, 40000.0), jit);
                const double J = (double)__double2float_rn(__dsub_rn(t, jit2));
                const double den = __dsub_rn(2.0, J);
                const double q1 = __ddiv_rn(__dmul_rn(prev, __dadd_rn(2.0, J)), den);
                const double q2 = __ddiv_rn(__dmul_rn(P2, J), den);
                cur = __double2float_rn(__dadd_rn(q1, q2));
                T = (int)vs_d2s(ceil((double)__fadd_rn(Pf, cur)));
                if (++guard > (1 << 22)) { atomicExch(a.status, VS_ERANGE); return; }
            } while ((float)T > t_hi || (float)T < t_lo);
            dper = cur;
        }
        float A = ampf, S = 0.0f;
        if (do_shm) {                                                     /* :296-306 */
            const double prev = (double)dsh;
            float cur;
            do {
                const int32_t r = vs_rng_next<NT>(g); nd++;
                const float eps = __fmul_rn((float)r, 4.656612873077393e-10f);   /* / (float)RAND_MAX == * 2^-31, exact */
                S = __double2float_rn(__dsub_rn(__dmul_rn(__dmul_rn((double)eps, 4.0), shm), shm2));
                const double den = __dsub_rn(2.0, (double)S);
                const double q1 = __ddiv_rn(__dmul_rn(prev, __dadd_rn(2.0, (double)S)), den);
                const double q2 = __ddiv_rn(__dmul_rn(amp2, (double)S), den);
                cur = __double2float_rn(__dadd_rn(q1, q2));
                A = __fadd_rn(ampf, cur);
                if (++guard > (1 << 22)) { atomicExch(a.status, VS_ERANGE); return; }
            } while (A > a_hi || A < a_lo);
            dsh = cur;
        }
        if (T < 1 || T > 32767) { atomicExch(a.status, VS_ERANGE); return; }

        /* closure-speed draw, always consumed (:325) */
        const int32_t rk = vs_rng_next<NT>(g); nd++;
        const double kq = __dsub_rn(vs_div_const((double)rk, VS_RAND_MAX_D, VS_INV_RM), 0.5);
        const float Knew = __double2float_rn(__dmul_rn(Kbase, __dadd_rn(1.0, __dmul_rn(kv2, kq))));

        /* chunks whose generation starts inside this period: remember where we are */
        while (next_target < count + (uint32_t)T) {
            chunks[next_c].first_period = np;
            chunks[next_c].first_start = count;
            if (noise && a.rng_snap) vs_rng_save<NT>(g, a.rng_snap + (size_t)(st.chunk0 + next_c) * 32);
            next_c++;
            next_target = next_c < st.n_chunks ? chunks[next_c].gen_target : 0xffffffffu;
        }

        int T3 = 2 * T2;
        float x_pow = 0.0f, w_pow = 0.0f;
        uint32_t n_noise = 0;
        if (pulse) {
            /* one pass over the open phase: T4 = last rising index below DC (:320-323), T3 = first
             * falling index below DC (:329), and the float power sum over [T4,T3) in index order
             * (:374-378).  The sum restarts whenever T4 moves; if T4 never moves in this period the
             * sum that started at the stale T4 is the one the reference computes. */
            const double Ad = (double)A, Kd = (double)Knew;
            float aux_new = 0.0f, aux_old = 0.0f;
            bool moved = false;
            const int T4_old = T4;
#pragma unroll 4
            for (int i = 0; i < T2; i++) {
                int x = vs_rising(Ad, __ldg(ht + i));
                if (x < DCi) { x = DCs; T4 = i; moved = true; aux_new = 0.0f; }
                const float sq = __fmul_rn((float)x, (float)x);
                if (moved) aux_new = __fadd_rn(aux_new, sq);
                else if (i >= T4_old) aux_old = __fadd_rn(aux_old, sq);
            }
            float aux = moved ? aux_new : aux_old;
            int i;
#pragma unroll 4
            for (i = T2; i < 2 * T2; i++) {
                const int x = vs_falling(Ad, Kd, __ldg(ct + i - T2));
                if (x < DCi) break;
                aux = __fadd_rn(aux, __fmul_rn((float)x, (float)x));
            }
            T3 = i;
            if (noise) {                                                  /* :378-382 */
                const float span = __fsub_rn((float)T3, (float)T4);
                x_pow = __fdiv_rn(aux, span);
                const float ax = __double2float_rn(__dadd_rn(1.0, (double)__fdiv_rn(span, (float)T)));
                ndw = vs_d2i(sqrt((double)__fdiv_rn(__fmul_rn(__fmul_rn(12.0f, ax), x_pow), st.noise)));
                n_noise = (uint32_t)(T4 + (T > T3 ? T - T3 : 0));
                if (LOG) {
                    float wa = 0.0f;
                    for (uint32_t k = 0; k < n_noise; k++) {
                        const int w = vs_noise_w(vs_rng_next<NT>(g), ndw);
                        wa = __fadd_rn(wa, __fmul_rn((float)w, (float)w));
                    }
                    w_pow = __fdiv_rn(wa, (float)T);
                } else {
                    vs_rng_skip<NT>(g, n_noise);
                }
            }
        }

        if (np >= st.tab_cap || nd > 65535u || T3 > 65535 || T4 > 65535) {
            atomicExch(a.status, np >= st.tab_cap ? VS_ENOMEM : VS_ERANGE);
            return;
        }
        vs_store_period(a.table, a.compact, st.tab_off + np, A, Knew, count, T, nd, T3, T4, ndw);
        if (LOG) {
            vs_period_rec r;
            r.T = T; r.T2 = T2; r.T3 = T3; r.T4 = T4; r.A = A; r.Knew = Knew; r.S = S;
            r.ndraws = (int32_t)(nd + n_noise); r.ndw = ndw; r.x_pow = x_pow; r.w_pow = w_pow; r.reserved = 0;
            r.start = count;
            log[np] = r;
        }
        count += (uint32_t)T;                                             /* :413 */
        np++;
    } while (count < st.n);                                               /* :423 */
    a.n_periods[s] = np;
}

/* ================================================================================================
 * PLAN, one WARP per stream: for small batches (a single ten-minute stream is 71 k sequential periods)
 * and for streams with glottal noise, where one thread per stream leaves the GPU idle or crawls through
 * hundreds of serial pulse samples and noise draws per period.
 *   - random(): 31 values per round by the whole warp (vs_rng_round);
 *   - every value's three possible meanings (jitter draw, shimmer draw, closure-speed draw; they do not
 *     depend on the walk's state) are worked out lane-parallel, one value per lane, incl. the two
 *     divisions whose numerator is state-free and a refined reciprocal for the one that is not;
 *   - the walk itself (flowgen_shimmer.c:276-325) runs warp-uniform, reading those values back by
 *     broadcast; its remaining division is the reciprocal-multiply sequence with an exactness check and
 *     an IEEE division when the check is inconclusive;
 *   - with noise: the open phase is evaluated 32 samples per step, the float power sum then runs in
 *     index order over the 32 squares (the sum is not associative), and the period's noise draws are
 *     stepped over with vs_rng_gen.
 * Same tables, chunk marks and RNG snapshots as vs_plan_kernel<false>.
 * ============================================================================================== */
#define VS_PLANW_NT 128

/* n/d given y ~ 1/d; sets doubt unless the result is provably the correctly rounded quotient */
__device__ __forceinline__ double vs_div_checked_y(double n, double d, double y, bool &doubt)
{
    const double q0 = __dmul_rn(n, y);
    const double q = __fma_rn(__fma_rn(-q0, d, n), y, q0);
    const double rem = __fma_rn(-q, d, n);
    const int e = (__double2hiint(q) >> 20) & 0x7ff;                /* ulp(q)/2 = 2^(e-53-1023) */
    const double half_ulp = __hiloint2double((e - 53) << 20, 0);
    const bool sure = (e > 60 && e < 0x7fe) && (fabs(rem) < __dmul_rn(half_ulp, fabs(d)));
    doubt = !sure && !(q == 0.0 && rem == 0.0);
    return q;
}
__device__ __forceinline__ double vs_recip_refined(double d)
{
    double y = (double)__frcp_rn((float)d);
    y = __fma_rn(y, __fma_rn(-d, y, 1.0), y);
    y = __fma_rn(y, __fma_rn(-d, y, 1.0), y);
    y = __fma_rn(y, __fma_rn(-d, y, 1.0), y);
    return y;
}

__global__ void __launch_bounds__(VS_PLANW_NT) vs_plan_warp_kernel(const VsPlanArgs a)
{
    /* per random() value, in a ring of 64 slots (two rounds of 31 are outstanding at most):
     * 2+J, 2-J, 1/(2-J), 2P*J/(2-J); the same four for S; Knew */
    __shared__ double s_itp[VS_PLANW_NT / 32][12][64];
    __shared__ float s_kn[VS_PLANW_NT / 32][64];
    __shared__ __align__(16) float s_sq[VS_PLANW_NT / 32][32];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const uint32_t s = blockIdx.x * (VS_PLANW_NT / 32) + wib;
    if (s >= a.n_streams) return;
    const VsStream st = a.streams[s];
    double (*itp)[64] = s_itp[wib];
    float *kn = s_kn[wib];
    float *sqb = s_sq[wib];

    const bool do_jit = (st.flags & VS_F_JITTER) && st.jitter != 0.0f;    /* :248 */
    const bool do_shm = (st.flags & VS_F_SHIMMER) && st.shimmer != 0.0f;  /* :295 */
    const bool noise = (st.flags & VS_F_NOISE) != 0;                      /* :373 */
    const int P = st.P, T2 = st.T2;
    const float Pf = (float)P, ampf = (float)st.amp;
    const float t_hi = __fmul_rn(1.2f, Pf), t_lo = __fmul_rn(0.8f, Pf);
    const float a_hi = __fmul_rn(1.8f, ampf), a_lo = __fmul_rn(0.2f, ampf);
    const double jit = (double)st.jitter, shm = (double)st.shimmer;
    const double jit2 = __dmul_rn(2.0, jit), shm2 = __dmul_rn(2.0, shm);
    const double P2 = __dmul_rn(2.0, (double)P), amp2 = __dmul_rn(2.0, (double)st.amp);
    const double Kbase = (double)st.K, kv2 = (double)__fmul_rn(2.0f, st.Kvar);
    const double *ht = a.costab + st.cos_off;
    const double *ct = ht + T2;
    const int DCi = (int)ceilf(st.DC);
    const int DCs = st.DCs;

    uint32_t rs = vs_rng_seed_warp(st.seed, lane);                       /* flowgen_shimmer.c:241 */

    /* Value source.  Values are numbered from the last reset; value i lives in ring slot i & 63.
     * rs = generator state before round A; nxa = round A = values [base, base+31); nxb = round B =
     * values [base+31, base+62) once have_b; pos = next value to use. */
    uint32_t nxa = 0, nxb = 0;
    int base = 0, pos = 0;
    bool have_b = false;
    auto interpret = [&](uint32_t words, int first) {     /* lane-parallel: what each value means as J, S, K draw */
        __syncwarp();
        if (lane < VS_RNG_DEG) {
            const int32_t r = (int32_t)(words >> 1);
            const int slot = (first + lane) & 63;
            if (do_jit) {                                                  /* :277-281 */
                double t = vs_div_const((double)r, VS_RM4, VS_INV_RM4);
                t = __dmul_rn(__dmul_rn(t, 40000.0), jit);
                const double J = (double)__double2float_rn(__dsub_rn(t, jit2));
                const double den = __dsub_rn(2.0, J), y = vs_recip_refined(den), num = __dmul_rn(P2, J);
                bool doubt;
                double q = vs_div_checked_y(num, den, y, doubt);
                if (doubt) q = __ddiv_rn(num, den);
                itp[0][slot] = __dadd_rn(2.0, J);
                itp[1][slot] = den;
                itp[2][slot] = y;
                itp[3][slot] = q;
                /* the same step as one FMA, dPer' ~ dPer*a + q (tight loop below), and the part of its error bound
                 * that does not depend on dPer */
                itp[8][slot] = __ddiv_rn(__dadd_rn(2.0, J), den);
                itp[9][slot] = __dmul_rn(fabs(q), 1.7763568394002505e-15);
            }
            if (do_shm) {                                                  /* :297-301 */
                const float eps = __fmul_rn((float)r, 4.656612873077393e-10f);
                const double S = (double)__double2float_rn(__dsub_rn(__dmul_rn(__dmul_rn((double)eps, 4.0), shm), shm2));
                const double den = __dsub_rn(2.0, S), y = vs_recip_refined(den), num = __dmul_rn(amp2, S);
                bool doubt;
                double q = vs_div_checked_y(num, den, y, doubt);
                if (doubt) q = __ddiv_rn(num, den);
                itp[4][slot] = __dadd_rn(2.0, S);
                itp[5][slot] = den;
                itp[6][slot] = y;
                itp[7][slot] = q;
                itp[10][slot] = __ddiv_rn(__dadd_rn(2.0, S), den);
                itp[11][slot] = __dmul_rn(fabs(q), 1.7763568394002505e-15);
            }
            const double kq = __dsub_rn(vs_div_const((double)r, VS_RAND_MAX_D, VS_INV_RM), 0.5);   /* :325 */
            kn[slot] = __double2float_rn(__dmul_rn(Kbase, __dadd_rn(1.0, __dmul_rn(kv2, kq))));
        }
        __syncwarp();
    };
    auto restart = [&](uint32_t state) {                  /* value numbering starts again at this generator state */
        rs = state;
        nxa = vs_rng_round(rs, lane);
        base = 0; pos = 0; have_b = false;
        interpret(nxa, 0);
    };
    auto make_b = [&]() {
        nxb = vs_rng_round(nxa, lane);
        interpret(nxb, base + VS_RNG_DEG);
        have_b = true;
    };
    auto refill = [&](bool ahead) {                       /* afterwards pos < base+31, and round B exists if `ahead` */
        while (pos >= base + VS_RNG_DEG) {
            if (!have_b) make_b();
            rs = nxa; nxa = nxb; base += VS_RNG_DEG; have_b = false;
        }
        if (ahead && !have_b) make_b();
    };
    auto slide = [&](uint32_t before, uint32_t words, int u) -> uint32_t {   /* state after u (0..31) values of a round */
        const int src = lane + u;
        const uint32_t keep = __shfl_sync(VS_FULL, before, src & 31);
        const uint32_t fr = __shfl_sync(VS_FULL, words, (src - VS_RNG_DEG) & 31);
        return src < VS_RNG_DEG ? keep : fr;
    };
    auto state_now = [&]() -> uint32_t {                  /* lanes 0..30, oldest word first */
        const int off = pos - base;                       /* 0..62 */
        return off <= VS_RNG_DEG ? slide(rs, nxa, off) : slide(nxa, nxb, off - VS_RNG_DEG);
    };
    restart(rs);

    int T = P, T4 = 0, ndw = 0;
    float dper = 0.0f, dsh = 0.0f;
    uint32_t count = 0, np = 0, next_c = 0;
    VsChunk *chunks = a.chunks + st.chunk0;
    uint32_t next_target = st.n_chunks ? chunks[0].gen_target : 0xffffffffu;
    /* the target after that is fetched one mark ahead: a single long stream crosses a chunk start every few
     * periods and would otherwise wait for a dependent global load each time */
    uint32_t after_target = st.n_chunks > 1 ? chunks[1].gen_target : 0xffffffffu;
    int guard = 0;
    const bool both = do_jit && do_shm;

    do {
        /* Tight loop for the common stream (jitter and shimmer on, no noise) while everything goes the common
         * way: three values per period straight off the ring, both draws accepted, divisions conclusive.  It
         * leaves to the general period below for anything else -- values running out (refill), a rejected
         * draw, an inconclusive division -- and comes back afterwards. */
        if (both && !noise) {
            const int lim = base + (have_b ? 2 * VS_RNG_DEG : VS_RNG_DEG);
            while (pos + 3 <= lim && count < st.n && np < st.tab_cap) {
                const int pj = pos & 63, ps = (pos + 1) & 63, pk = (pos + 2) & 63;
                /* The reference rounds  fl(fl(dPer*(2+J))/(2-J)) + q  to FLOAT (:286-287).  One FMA with a = fl((2+J)/(2-J))
                 * is within  e = 2^-49 (|dPer*a| + |q|)  of that double; if s-e and s+e round to the same float, so
                 * does the reference's value (rounding is monotone) and the serial chain of a period is
                 * float->double, FMA, double->float.  Otherwise (about once in 10^7 periods): the general period below. */
                const double dJ = (double)dper, dS = (double)dsh;
                const double aJ = itp[8][pj], aS = itp[10][ps];
                const double sJ = __fma_rn(dJ, aJ, itp[3][pj]), sS = __fma_rn(dS, aS, itp[7][ps]);
                const double eJ = __fma_rn(fabs(__dmul_rn(dJ, aJ)), 1.7763568394002505e-15, itp[9][pj]);
                const double eS = __fma_rn(fabs(__dmul_rn(dS, aS)), 1.7763568394002505e-15, itp[11][ps]);
                const float curJ = __double2float_rn(sJ), curS = __double2float_rn(sS);
                const bool dj = !(__double2float_rn(__dsub_rn(sJ, eJ)) == __double2float_rn(__dadd_rn(sJ, eJ)));
                const bool ds = !(__double2float_rn(__dsub_rn(sS, eS)) == __double2float_rn(__dadd_rn(sS, eS)));
                const float Tf = ceilf(__fadd_rn(Pf, curJ));
                const float An = __fadd_rn(ampf, curS);
                if (dj || ds || Tf > t_hi || Tf < t_lo || !(Tf >= 1.0f && Tf <= 32767.0f) || An > a_hi || An < a_lo) break;
                dper = curJ; dsh = curS; T = (int)Tf;
                pos += 3;
                while (next_target < count + (uint32_t)T) {
                    if (lane == 0) { chunks[next_c].first_period = np; chunks[next_c].first_start = count; }
                    next_c++;
                    next_target = after_target;
                    after_target = next_c + 1 < st.n_chunks ? chunks[next_c + 1].gen_target : 0xffffffffu;
                }
                if (lane == 0) vs_store_period(a.table, a.compact, st.tab_off + np, An, kn[pk], count, T, 3u, 2 * T2, 0, 0);
                count += (uint32_t)T;
                np++;
            }
            if (count >= st.n) break;
        }
        uint32_t nd = 0;
        float A = ampf, Knew = 0.0f;
        bool committed = false;
        /* without noise the values of consecutive periods are consecutive: keep a round in reserve so that
         * the common case never meets a round boundary */
        if (pos >= base + VS_RNG_DEG || !(noise || have_b)) refill(!noise);
        /* Common case first: jitter and shimmer both on, every draw accepted at once.  The two random walks
         * are independent recurrences, so their division chains run side by side; acceptance is tested on
         * ceilf(P + dPer), the same integer as (short)ceil((double)..) when it is in range.  Anything else
         * -- a rejected draw, an inconclusive division check -- takes the literal loops below from pos. */
        if (both && (have_b || pos + 3 <= base + VS_RNG_DEG)) {
            const int pj = pos & 63, ps = (pos + 1) & 63, pk = (pos + 2) & 63;
            const double numj = __dmul_rn((double)dper, itp[0][pj]);
            const double nums = __dmul_rn((double)dsh, itp[4][ps]);
            bool dj, ds;
            const double qj = vs_div_checked_y(numj, itp[1][pj], itp[2][pj], dj);
            const double qs = vs_div_checked_y(nums, itp[5][ps], itp[6][ps], ds);
            const float curJ = __double2float_rn(__dadd_rn(qj, itp[3][pj]));
            const float curS = __double2float_rn(__dadd_rn(qs, itp[7][ps]));
            const float Tf = ceilf(__fadd_rn(Pf, curJ));
            const float An = __fadd_rn(ampf, curS);
            const bool ok = !dj && !ds && !(Tf > t_hi || Tf < t_lo) && Tf >= 1.0f && Tf <= 32767.0f && !(An > a_hi || An < a_lo);
            if (ok) {
                dper = curJ; dsh = curS; T = (int)Tf; A = An;
                Knew = kn[pk];
                nd = 3u;
                pos += 3;
                committed = true;
            }
        }
        if (!committed) {
            if (do_jit) {                                                     /* :276-290 */
                const double prev = (double)dper;
                float cur;
                for (;;) {
                    refill(false);
                    const int p = pos++ & 63; nd++;
                    const double num = __dmul_rn(prev, itp[0][p]), den = itp[1][p];
                    bool doubt;
                    double q1 = vs_div_checked_y(num, den, itp[2][p], doubt);
                    if (doubt) q1 = __ddiv_rn(num, den);
                    cur = __double2float_rn(__dadd_rn(q1, itp[3][p]));
                    T = (int)vs_d2s(ceil((double)__fadd_rn(Pf, cur)));
                    if (++guard > (1 << 22)) { atomicExch(a.status, VS_ERANGE); return; }
                    if (!((float)T > t_hi || (float)T < t_lo)) break;
                }
                dper = cur;
            }
            if (do_shm) {                                                     /* :296-306 */
                const double prev = (double)dsh;
                float cur;
                for (;;) {
                    refill(false);
                    const int p = pos++ & 63; nd++;
                    const double num = __dmul_rn(prev, itp[4][p]), den = itp[5][p];
                    bool doubt;
                    double q1 = vs_div_checked_y(num, den, itp[6][p], doubt);
                    if (doubt) q1 = __ddiv_rn(num, den);
                    cur = __double2float_rn(__dadd_rn(q1, itp[7][p]));
                    A = __fadd_rn(ampf, cur);
                    if (++guard > (1 << 22)) { atomicExch(a.status, VS_ERANGE); return; }
                    if (!(A > a_hi || A < a_lo)) break;
                }
                dsh = cur;
            }
            if (T < 1 || T > 32767) { atomicExch(a.status, VS_ERANGE); return; }
            refill(false);                                                    /* closure-speed draw (:325) */
            Knew = kn[pos++ & 63]; nd++;
        }

        while (next_target < count + (uint32_t)T) {
            if (lane == 0) { chunks[next_c].first_period = np; chunks[next_c].first_start = count; }
            if (noise && a.rng_snap) {
                const uint32_t now = state_now();
                if (lane < VS_RNG_DEG) a.rng_snap[(size_t)(st.chunk0 + next_c) * 32 + (lane + 3) % VS_RNG_DEG] = now;
            }
            next_c++;
            next_target = after_target;
            after_target = next_c + 1 < st.n_chunks ? chunks[next_c + 1].gen_target : 0xffffffffu;
        }

        int T3 = 2 * T2;
        if (noise) {
            const double Ad = (double)A, Kd = (double)Knew;
            float aux = 0.0f;
            /* rising branch (:318-323): T4 = last index below DC; the power sum covers [T4, T2) whether T4
             * moved in this period or is the stale one */
            for (int b0 = 0; b0 < T2; b0 += 32) {
                const int i = b0 + lane;
                const bool valid = i < T2;
                int x = valid ? vs_rising(Ad, __ldg(ht + i)) : 0;
                const bool below = valid && x < DCi;
                const uint32_t m = __ballot_sync(VS_FULL, below);
                if (m) { T4 = b0 + 31 - __clz((int)m); aux = 0.0f; }
                if (below) x = DCs;
                sqb[lane] = (valid && i >= T4) ? __fmul_rn((float)x, (float)x) : 0.0f;
                __syncwarp();
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    const float4 v = reinterpret_cast<const float4 *>(sqb)[k];
                    aux = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(aux, v.x), v.y), v.z), v.w);
                }
                __syncwarp();
            }
            /* falling branch (:327-332): stops at the first index below DC = T3 */
            for (int b0 = T2; b0 < 2 * T2; b0 += 32) {
                const int i = b0 + lane;
                const bool valid = i < 2 * T2;
                const int x = valid ? vs_falling(Ad, Kd, __ldg(ct + i - T2)) : 0;
                const uint32_t m = __ballot_sync(VS_FULL, valid && x < DCi);
                const int first = m ? __ffs((int)m) - 1 : 32;
                sqb[lane] = (valid && lane < first) ? __fmul_rn((float)x, (float)x) : 0.0f;
                __syncwarp();
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    const float4 v = reinterpret_cast<const float4 *>(sqb)[k];
                    aux = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(aux, v.x), v.y), v.z), v.w);
                }
                __syncwarp();
                if (m) { T3 = b0 + first; break; }
            }
            /* :378-382 */
            const float span = __fsub_rn((float)T3, (float)T4);
            const float x_pow = __fdiv_rn(aux, span);
            const float ax = __double2float_rn(__dadd_rn(1.0, (double)__fdiv_rn(span, (float)T)));
            ndw = vs_d2i(sqrt((double)__fdiv_rn(__fmul_rn(__fmul_rn(12.0f, ax), x_pow), st.noise)));
            const uint32_t n_noise = (uint32_t)(T4 + (T > T3 ? T - T3 : 0));
            /* the period's noise values are the render kernel's business: step over them */
            restart(vs_rng_gen(state_now(), (int)n_noise, lane, nullptr));
        }

        if (np >= st.tab_cap || (!committed && nd > 65535u) || (noise && (T3 > 65535 || T4 > 65535))) {
            atomicExch(a.status, np >= st.tab_cap ? VS_ENOMEM : VS_ERANGE);
            return;
        }
        if (lane == 0) vs_store_period(a.table, a.compact, st.tab_off + np, A, Knew, count, T, nd, T3, T4, ndw);
        count += (uint32_t)T;                                             /* :413 */
        np++;
    } while (count < st.n);                                               /* :423 */
    if (lane == 0) a.n_periods[s] = np;
}

/* ================================================================================================
 * vowel -n (SURVEY 8f N1): output noise in place (vowel_new.c:302-324), one WARP per stream.
 * Per frame of `frame` samples: the float power sum runs in sample order (not associative: every lane
 * adds the same 32 squares, staged through shared memory); the frame's random() values come 31 at a time
 * (vs_rng_gen) into a per-warp scratch and the noise is added lane-parallel.
 * ============================================================================================== */
#define VS_VN_NT      128
#define VS_VN_SCRATCH 1024            /* random() values per piece of a frame */

__global__ void __launch_bounds__(VS_VN_NT) vs_vnoise_kernel(int16_t *pcm, const VsNoiseRow *rows, uint32_t n_rows)
{
    __shared__ int32_t s_draws[VS_VN_NT / 32][VS_VN_SCRATCH];
    __shared__ __align__(16) float s_sq[VS_VN_NT / 32][32];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const uint32_t s = blockIdx.x * (VS_VN_NT / 32) + wib;
    if (s >= n_rows) return;
    const VsNoiseRow r = rows[s];
    if (!(r.snr > 0.0f) || r.frame == 0) return;
    int32_t *draws = s_draws[wib];
    float *sqb = s_sq[wib];
    uint32_t st = vs_rng_seed_warp(r.seed, lane);                        /* :234 */
    int16_t *y = pcm + r.off;
    for (uint32_t base = 0; base < r.n; base += r.frame) {
        const uint32_t ni = min(r.frame, r.n - base);
        float aux = 0.0f;
        for (uint32_t b0 = 0; b0 < ni; b0 += 32) {                       /* :304-306, float, in order */
            const uint32_t i = b0 + lane;
            const float v = i < ni ? (float)y[base + i] : 0.0f;
            sqb[lane] = __fmul_rn(v, v);                                 /* +0.0f beyond the frame: adds nothing */
            __syncwarp();
#pragma unroll
            for (int k = 0; k < 8; k++) {
                const float4 q = reinterpret_cast<const float4 *>(sqb)[k];
                aux = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(aux, q.x), q.y), q.z), q.w);
            }
            __syncwarp();
        }
        const float sig_power = __fdiv_rn(aux, (float)(int16_t)ni);      /* `ni` is a signed short (:65) */
        const float width = __double2float_rn(sqrt((double)__fdiv_rn(__fmul_rn(12.0f, sig_power), r.snr)));   /* :309 */
        for (uint32_t p0 = 0; p0 < ni; p0 += VS_VN_SCRATCH) {            /* :314-319 */
            const uint32_t m = min((uint32_t)VS_VN_SCRATCH, ni - p0);
            st = vs_rng_gen(st, (int)m, lane, draws);
            __syncwarp();
            for (uint32_t k = lane; k < m; k += 32) {
                const float nv = __double2float_rn(vs_div_const((double)draws[k], VS_RAND_MAX_D, VS_INV_RM));
                const float a = __double2float_rn(__dmul_rn((double)width, __dsub_rn((double)nv, 0.5)));
                int16_t *dst = y + base + p0 + k;
                *dst = (int16_t)vs_round2int(__dadd_rn((double)*dst, (double)a));
            }
            __syncwarp();
        }
    }
}

cudaError_t vs_launch_vnoise(int16_t *pcm, const VsNoiseRow *rows, uint32_t n_rows, cudaStream_t s)
{
    vs_vnoise_kernel<<<(n_rows + VS_VN_NT / 32 - 1) / (VS_VN_NT / 32), VS_VN_NT, 0, s>>>(pcm, rows, n_rows);
    return cudaGetLastError();
}

/* ------------------------------------------------------------------------------------------------
 * FP64 pipe peak: 8 independent DFMA chains per thread, every SM full.  Used by bench.py to put a
 * measured denominator next to the HBM-write roofline (SURVEY.md 8d).
 * ---------------------------------------------------------------------------------------------- */
__global__ void __launch_bounds__(256) vs_fp64_peak_kernel(double *out, int iters, double a, double b)
{
    double x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
    for (int i = 0; i < iters; i++) {
        x0 = __fma_rn(x0, a, b); x1 = __fma_rn(x1, a, b); x2 = __fma_rn(x2, a, b); x3 = __fma_rn(x3, a, b);
        x4 = __fma_rn(x4, a, b); x5 = __fma_rn(x5, a, b); x6 = __fma_rn(x6, a, b); x7 = __fma_rn(x7, a, b);
    }
    const double s = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
    if (s == 123.456) out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

cudaError_t vs_launch_fp64_peak(double *scratch, int blocks, int iters, cudaStream_t s)
{
    vs_fp64_peak_kernel<<<blocks, 256, 0, s>>>(scratch, iters, 0.999999, 1e-9);
    return cudaGetLastError();
}

/* ------------------------------------------------------------------------------------------------
 * launch wrappers (called from vs_api.cu)
 * ---------------------------------------------------------------------------------------------- */
/* warps: the warp form (vs_plan_warps); otherwise the record's thread form, sh.plan_nt streams per CTA */
cudaError_t vs_launch_plan(const VsPlanArgs &a, const VsShape &sh, bool warps, cudaStream_t s)
{
    if (warps) {
        vs_plan_warp_kernel<<<(a.n_streams + VS_PLANW_NT / 32 - 1) / (VS_PLANW_NT / 32), VS_PLANW_NT, 0, s>>>(a);
        return cudaGetLastError();
    }
    const unsigned grid = (a.n_streams + sh.plan_nt - 1) / sh.plan_nt;
    static_assert(VS_PLAN_SMEM >= VS_RNG_DEG * VS_PLAN_NT * 4, "plan kernel shared memory");
    if (sh.plan == VS_PLAN_LOG) {
        cudaFuncSetAttribute(vs_plan_kernel<true, true, VS_PLAN_NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, VS_PLAN_SMEM);
        vs_plan_kernel<true, true, VS_PLAN_NT><<<grid, VS_PLAN_NT, VS_PLAN_SMEM, s>>>(a);
    } else if (sh.plan == VS_PLAN_PULSE) {
        cudaFuncSetAttribute(vs_plan_kernel<false, true, VS_PLAN_NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, VS_PLAN_SMEM);
        vs_plan_kernel<false, true, VS_PLAN_NT><<<grid, VS_PLAN_NT, VS_PLAN_SMEM, s>>>(a);
    } else {
        constexpr int smem = VS_RNG_DEG * VS_PLAN_NT_LEAN * 4;
        static_assert(smem >= VS_PLAN_SMEM, "the lean plan CTA must not share an SM with a render CTA either");
        cudaFuncSetAttribute(vs_plan_kernel<false, false, VS_PLAN_NT_LEAN>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        vs_plan_kernel<false, false, VS_PLAN_NT_LEAN><<<grid, VS_PLAN_NT_LEAN, smem, s>>>(a);
    }
    return cudaGetLastError();
}
