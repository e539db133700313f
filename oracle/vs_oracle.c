/* vs_oracle.c -- TEST INFRASTRUCTURE ONLY (see vs_oracle.h).
 *
 * A from-scratch CPU restatement of the reference arithmetic, written as small pure functions with
 * every float/double rounding point spelled out.  Compile with -ffp-contract=off (oracle/Makefile):
 * the reference is built for baseline x86-64 (SSE2, FLT_EVAL_METHOD 0, no FMA).
 *
 * Third-party arithmetic the reference pulls in and that is NOT in its tree:
 *   glibc 2.39 (Ubuntu 2.39-0ubuntu8.5) random()/srandom()  -> restated below (TYPE_3, x^31+x^3+1)
 *   glibc 2.39 libm cos/ceil/floor/sqrt/pow                 -> called from the system libm
 */
#include "vs_oracle.h"
#include "vs_oracle_presets.h"
#include <ctype.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

/* ------------------------------------------------------------------ RNG (glibc random_r.c) ---- */
void vso_srandom(vso_rng *g, uint32_t seed)
{
    int32_t w = (int32_t)(seed ? seed : 1u);
    g->r[0] = (uint32_t)w;
    for (int i = 1; i < 31; i++) {              /* Park-Miller via Schrage, signed 32-bit */
        int32_t hi = w / 127773, lo = w % 127773;
        w = 16807 * lo - 2836 * hi;
        if (w < 0) w += 2147483647;
        g->r[i] = (uint32_t)w;
    }
    g->f = 3; g->b = 0;
    for (int i = 0; i < 310; i++) (void)vso_random(g);
}

int32_t vso_random(vso_rng *g)
{
    g->r[g->f] += g->r[g->b];
    int32_t out = (int32_t)(g->r[g->f] >> 1);
    if (++g->f == 31) g->f = 0;
    if (++g->b == 31) g->b = 0;
    return out;
}

#define VSO_RAND_MAX 2147483647

/* what `short = <double expr>` does on x86-64: cvttsd2si to 32 bits, keep the low 16 */
static int16_t d2s(double v)
{
    if (!(v > -2147483649.0 && v < 2147483648.0)) return 0;   /* "integer indefinite" 0x80000000 */
    return (int16_t)(uint16_t)(uint32_t)(int32_t)v;
}
static int32_t d2i(double v)
{
    if (!(v > -2147483649.0 && v < 2147483648.0)) return (int32_t)0x80000000u;
    return (int32_t)v;
}

/* ------------------------------------------------------------------ flowgen parameters -------- */
void vso_flow_par_default(vso_flow_par *p)
{
    memset(p, 0, sizeof *p);
    p->dur = 1.0f; p->jitter = 0.0f; p->cq = 0.55f; p->K = 0.65f; p->Fg = 125.0f; p->F0 = 120.0f;
    p->DC = 0.0f;  p->noise = 0.0f;  p->fs = 22050; p->amp = 12000; p->Kvar = 0.0f; p->shimmer = 0.0f;
    p->seed = 1;
}

int vso_flow_par_from_cli(int argc, const char *const *argv, vso_flow_par *p)
{
    /* indices of the value strings, -1 = flag absent (struct ARG, flowgen_shimmer.c:90-102) */
    int a_wav = -1, a_dur = -1, a_jit = -1, a_cq = -1, a_K = -1, a_Fg = -1, a_F0 = -1, a_DC = -1,
        a_noise = -1, a_fs = -1, a_amp = -1, a_Kvar = -1, a_sh = -1;
    uint32_t seed = p->seed;
    vso_flow_par_default(p);
    p->seed = seed;
    if (argc < 2) return -1;
    int i;
    for (i = 1; i < argc && argv[i][0] == '-'; i++) {
        if (argc <= i + 1) return -1;                       /* every flag takes a value (:135) */
        int c = tolower((unsigned char)argv[i][1]);
        i++;
        switch (c) {
        case 'o': a_wav = i; break;   case 'g': a_Fg = i; break;   case 'f': a_F0 = i; break;
        case 'd': a_dur = i; break;   case 'c': a_cq = i; break;   case 'j': a_jit = i; break;
        case 'k': a_K = i; break;     case 'r': a_fs = i; break;   case 'a': a_amp = i; break;
        case 'l': a_DC = i; break;    case 'z': a_Kvar = i; break; case 's': a_sh = i; break;
        case 'n': p->DC = 0.25f; a_noise = i; break;        /* side effect at parse time (:182) */
        default: return -1;
        }
    }
    if ((i != argc && argv[i][0] != 'i') || a_wav == -1) return -1;          /* :219 */

    float f;                                                /* initialization(), :463-547, in its order */
    if (a_dur != -1)  { f = (float)atof(argv[a_dur]);          if (f >= 0.5) p->dur = f; else return -1; }
    if (a_jit != -1)  { f = (float)(atof(argv[a_jit]) / 100.0); if (f >= 0.0 && f <= 10.0) p->jitter = f; else return -1; }
    if (a_K != -1)    { f = (float)atof(argv[a_K]);            if (f >= 0.50) p->K = f; else return -1; }
    if (a_cq != -1)   { f = (float)atof(argv[a_cq]);           if (f >= 0.0 && f <= 1.0) p->cq = f; else return -1; }
    if (a_Fg != -1)   { f = (float)atof(argv[a_Fg]);           if (f >= 50) p->Fg = f; else return -1; }
    if (a_F0 != -1)   { f = (float)atof(argv[a_F0]);           if (f >= 50 && f < p->Fg) p->F0 = f; else return -1; }
    if (a_noise != -1){ f = (float)atof(argv[a_noise]);
                        if (f >= 0.0 && f <= 50) p->noise = (float)pow(10, (double)(f / 10)); else return -1; }
    if (a_amp != -1)  { int v = atoi(argv[a_amp]);             if (v >= 0 && v < 32767) p->amp = v; else return -1; }
    if (a_DC != -1)   { f = (float)atof(argv[a_DC]);           if (f >= 0 && f <= 0.3) p->DC = f * (float)p->amp; else return -1; }
    if (a_Kvar != -1) { f = (float)atof(argv[a_Kvar]);         if (f >= 0 && f <= 1) p->Kvar = f; else return -1; }
    if (a_fs != -1)   { long l = atol(argv[a_fs]);             /* the reference's test accepts everything but 22050 (:537) */
                        if (l == 44100L || l != 22050L || l == 11025L) p->fs = l; else return -1; }
    if (a_sh != -1)   { f = (float)atof(argv[a_sh]);           if (f >= 0 && f <= 100) p->shimmer = f / 100; else return -1; }
    p->has_jitter = a_jit != -1; p->has_shimmer = a_sh != -1; p->has_noise = a_noise != -1;
    return 0;
}

uint64_t vso_flow_nsamples(const vso_flow_par *p)
{
    /* `(unsigned long) par.fs*par.dur`: the cast binds to fs; ulong*float is a FLOAT product (:242) */
    float prod = (float)(uint64_t)p->fs * p->dur;
    return (uint64_t)prod;
}

/* ------------------------------------------------------------------ flowgen hot loop ---------- */
static inline double vso_pi(void) { return 4.0 * atan(1.0); }          /* #define PI, :39 */

/* flowgen_shimmer.c:276-290 -- one accepted jitter step; returns the new period length */
static int jitter_step(vso_rng *g, const vso_flow_par *p, int P, float *dper, int *ndraws)
{
    const float prev = *dper;
    const double jit = (double)p->jitter;
    float cur; int T;
    do {
        int32_t r = vso_random(g); (*ndraws)++;
        float J = (float)((((double)r / (VSO_RAND_MAX * 10000.0)) * 40000.0) * jit - 2.0 * jit);
        double den = 2.0 - (double)J;
        cur = (float)(((double)prev * (2.0 + (double)J)) / den + ((2.0 * P) * (double)J) / den);
        T = (int)d2s(ceil((double)((float)P + cur)));
    } while ((float)T > (float)1.2 * (float)P || (float)T < (float)0.8 * (float)P);
    *dper = cur;
    return T;
}

/* flowgen_shimmer.c:295-306 -- one accepted shimmer step; returns the period amplitude */
static float shimmer_step(vso_rng *g, const vso_flow_par *p, float *dsh, float *S_out, int *ndraws)
{
    const float prev = *dsh;
    const double sh = (double)p->shimmer;
    float cur, A, S;
    do {
        int32_t r = vso_random(g); (*ndraws)++;
        float eps = (float)r / (float)VSO_RAND_MAX;
        S = (float)(((double)eps * 4.0) * sh - 2.0 * sh);
        double den = 2.0 - (double)S;
        cur = (float)(((double)prev * (2.0 + (double)S)) / den + ((2.0 * p->amp) * (double)S) / den);
        A = (float)p->amp + cur;
    } while (A > (float)1.8 * (float)p->amp || A < (float)0.2 * (float)p->amp);
    *dsh = cur; *S_out = S;
    return A;
}

/* flowgen_shimmer.c:591-600 */
static int16_t clip_ceil(float v)
{
    if (v > 32767) return 32767;
    if (v < -32767) return -32767;
    return d2s(ceil((double)v));
}

int vso_flowgen(const vso_flow_par *p, int16_t *out, vso_period *log, size_t log_cap, size_t *n_periods)
{
    vso_rng g;
    vso_srandom(&g, p->seed);                                               /* :241 */
    const uint64_t n_total = vso_flow_nsamples(p);
    const int P = (int)((float)p->fs / p->F0);                              /* :244 */
    if (P < 1) return -1;
    int T = P, T4 = 0;   /* T4 is uninitialised in the reference (UB when never assigned); we define 0 */
    const int T2 = (int)ceil((0.5 * (double)p->cq) * P);                    /* :317 */
    const size_t cap = (size_t)(2 * T2 + (int)(1.2 * P) + 64);
    int16_t *x = (int16_t *)calloc(cap, sizeof *x);
    if (!x) return -2;
    const double pi = vso_pi();
    const float DC = p->DC;
    float dper = 0.0f, dsh = 0.0f;
    uint64_t count = 0; size_t np = 0;
    int ndw = 0;

    do {
        vso_period rec; memset(&rec, 0, sizeof rec);
        int nd = 0;
        rec.start = count;
        if (p->has_jitter && p->jitter != 0.0) T = jitter_step(&g, p, P, &dper, &nd);       /* :248 */
        float A, S = 0.0f;
        if (p->has_shimmer && p->shimmer != 0.0) A = shimmer_step(&g, p, &dsh, &S, &nd);    /* :295 */
        else A = (float)p->amp;

        /* rising branch :318-324 */
        for (int i = 0; i < T2; i++) {
            double c = cos((pi * i) / T2);
            x[i] = d2s(ceil(((double)A * 0.5) * (1.0 - c)));
            if ((float)x[i] < DC) { x[i] = d2s((double)DC); T4 = i; }
        }
        /* closure-speed draw: always consumed :325 */
        int32_t rk = vso_random(&g); nd++;
        float Knew = (float)((double)p->K * (1 + (double)(2 * p->Kvar) * (((1.0 * rk) / VSO_RAND_MAX) - 0.5)));
        /* falling branch :327-332 */
        int i;
        for (i = T2; i < 2 * T2; i++) {
            double c = cos((pi * (i - T2)) / T2);
            x[i] = d2s(ceil((double)A * (((double)Knew * c - (double)Knew) + 1.0)));
            if ((float)x[i] < DC) break;
        }
        const int T3 = i;
        for (i = T3; i < T; i++) x[i] = d2s((double)DC);                    /* :334-336 */

        if (p->has_noise) {                                                 /* :373-411 */
            float aux = 0.0f;
            for (i = T4; i < T3; i++) aux += (float)x[i] * (float)x[i];
            float span = (float)T3 - (float)T4;
            float x_pow = aux / span;
            aux = (float)(1.0 + (double)(span / (float)T));
            ndw = d2i(sqrt((double)(((12 * aux) * x_pow) / p->noise)));
            aux = 0.0f;
            for (int pass = 0; pass < 2; pass++) {
                int lo = pass ? T3 : 0, hi = pass ? T : T4;
                for (i = lo; i < hi; i++) {
                    int32_t r = vso_random(&g); nd++;
                    int w = d2s(ceil(((1.0 * r) / VSO_RAND_MAX) * ndw - ndw / 2.0));
                    aux += (float)w * (float)w;
                    x[i] = clip_ceil((float)x[i] + (float)w);
                }
            }
            rec.x_pow = x_pow; rec.w_pow = aux / (float)T;
        }

        count += (uint64_t)T;                                               /* :413-421 */
        uint64_t k = (count > n_total) ? (uint64_t)T - (count - n_total) : (uint64_t)T;
        memcpy(out + (count - (uint64_t)T), x, (size_t)k * sizeof *x);

        rec.T = T; rec.T2 = T2; rec.T3 = T3; rec.T4 = T4; rec.A = A; rec.Knew = Knew; rec.S = S;
        rec.ndraws = nd; rec.ndw = ndw;
        if (log && np < log_cap) log[np] = rec;
        np++;
    } while (count < n_total);

    free(x);
    if (n_periods) *n_periods = np;
    return 0;
}

/* ------------------------------------------------------------------ vowel filter -------------- */
const double *vso_preset(int key)
{
    const char *q = strchr(vso_preset_keys, key);
    if (!q || !key) return NULL;
    return vso_preset_den[q - vso_preset_keys];
}

int16_t vso_round2int(double x)
{
    double dec = x - floor(x);
    if (dec > 0.5) x = x + 1;
    if (x > 32767) x = 32767; else if (x < -32767) x = -32767;
    return d2s(floor(x));
}

int vso_vowel(const int16_t *in, size_t n, int preset_key, float gain, float pre, int16_t *out, double *raw)
{
    const double *A = vso_preset(preset_key);
    if (!A) return -1;
    double yd[VS_FILTER_ORDER + 1];
    for (int j = 0; j <= VS_FILTER_ORDER; j++) yd[j] = 0.0;
    for (size_t i = 0; i < n; i++) {
        /* zeros (:266-269): B == [1,0,...]; the 22 zero products add +-0.0 and change nothing */
        yd[0] = 0.0 + (1.0 * (double)in[i]) * (double)gain;
        for (int j = 1; j <= VS_FILTER_ORDER; j++) yd[0] = yd[0] - A[j] * yd[j];     /* :279-281 */
        double v = yd[0] - (double)pre * yd[1];                                        /* :284 */
        if (raw) raw[i] = v;
        out[i] = vso_round2int(v);
        for (int j = VS_FILTER_ORDER; j > 0; j--) yd[j] = yd[j - 1];                  /* :287-289 */
    }
    return 0;
}

int vso_vowel_noise(const int16_t *in, size_t n, int preset_key, float gain, float pre,
                    float snr_db_arg, int64_t fs, uint32_t seed, int16_t *out)
{
    if (vso_vowel(in, n, preset_key, gain, pre, out, NULL)) return -1;
    return vso_noise(out, n, snr_db_arg, fs, seed);
}

int vso_noise(int16_t *out, size_t n, float snr_db_arg, int64_t fs, uint32_t seed)
{
    if (!(snr_db_arg > 0)) return -1;                                                  /* :141-143 */
    float snr = (float)pow(10, (double)(snr_db_arg / 10));
    int ms1 = (int)((uint64_t)fs * 0.001 / 2.0) * 2;                                   /* :361 */
    size_t frame = (size_t)(50 * ms1);                                                 /* :363 */
    if (frame == 0) return -1;
    vso_rng g; vso_srandom(&g, seed);                                                  /* :234 */
    for (size_t base = 0; base < n; base += frame) {
        size_t ni = (n - base < frame) ? n - base : frame;
        int16_t *y = out + base;
        float aux = 0.0f;
        for (size_t i = 0; i < ni; i++) aux += (float)y[i] * (float)y[i];
        float sig_power = aux / (float)(int16_t)ni;
        float width = (float)sqrt((double)((12 * sig_power) / snr));
        for (size_t i = 0; i < ni; i++) {
            float nv = (float)((1.0 * vso_random(&g)) / VSO_RAND_MAX);
            float a = (float)((double)width * ((double)nv - 0.5));
            y[i] = vso_round2int(1.0 * y[i] + 1.0 * (double)a);
        }
    }
    return 0;
}
