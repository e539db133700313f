/* vs_oracle.h -- TEST INFRASTRUCTURE ONLY.
 *
 * CPU restatement of the reference's source-filter synthesis path (flowgen_shimmer.c, vowel_new.c
 * and the glibc-2.39 random()/srandom() generator they call).  It exists to CHECK the CUDA path.
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load
 * it; nothing in voice_synth_b200/ or host/ may include, link or dlopen anything under oracle/.
 *
 * Parity pin: this restatement is checked byte-for-byte against the UNMODIFIED reference binaries
 * (oracle/_ref, built by oracle/Makefile from /root/reference) in tests/test_oracle_vs_ref.py and
 * against the committed fixtures in tests/golden/ (made from those binaries by
 * tests/golden/make_golden.py).  The reference itself ships no tests or vectors (SURVEY.md 4).
 */
#ifndef VS_ORACLE_H
#define VS_ORACLE_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* glibc TYPE_3 additive-feedback generator (random_r.c; call sites flowgen_shimmer.c:241,283,298,
 * 325,387,398 and vowel_new.c:234,315). */
typedef struct { uint32_t r[31]; int f, b; } vso_rng;
void    vso_srandom(vso_rng *g, uint32_t seed);
int32_t vso_random(vso_rng *g);

/* struct PAR of flowgen_shimmer.c:73-87 plus the "argument was given" bits of struct ARG (:90-102)
 * that the main loop tests (:248, :295, :373). */
typedef struct {
    float   dur, jitter, cq, K, Fg, F0, DC, noise;
    int64_t fs;
    int32_t amp;
    float   Kvar, shimmer;
    int32_t has_jitter, has_shimmer, has_noise;
    uint32_t seed;
} vso_flow_par;

/* one record per pitch period -- everything the reference computes per period */
typedef struct {
    int32_t T, T2, T3, T4;
    float   A, Knew, S;
    int32_t ndraws;     /* random() calls consumed by this period (perturbation + K + noise) */
    int32_t ndw;        /* par.NoiseDistWidth after this period (0 without -n) */
    float   x_pow, w_pow;
    uint64_t start;     /* index of the period's first sample in the stream */
} vso_period;

void   vso_flow_par_default(vso_flow_par *p);                       /* flowgen_shimmer.c:87 */
/* argv-style parse + initialization() (flowgen_shimmer.c:128-219, 463-547).
 * returns 0, or -1 where the reference would print usage() and exit. */
int    vso_flow_par_from_cli(int argc, const char *const *argv, vso_flow_par *p);
uint64_t vso_flow_nsamples(const vso_flow_par *p);                  /* flowgen_shimmer.c:242 */
/* Hot loop flowgen_shimmer.c:246-423.  Writes exactly vso_flow_nsamples() samples to out.
 * log (nullable) receives up to log_cap period records; *n_periods (nullable) the period count. */
int    vso_flowgen(const vso_flow_par *p, int16_t *out, vso_period *log, size_t log_cap,
                   size_t *n_periods);

/* preset key 'a','i','u','1'..'7' -> 23 denominator coefficients, NULL if unknown */
const double *vso_preset(int key);
/* vowel_new.c:252-296 + round2int :413-427.  raw (nullable) receives the FP64 value handed to
 * round2int (the "pre-quantisation waveform"). */
int    vso_vowel(const int16_t *in, size_t n, int preset_key, float gain, float pre,
                 int16_t *out, double *raw);
/* vowel -n (vowel_new.c:302-324): per-frame output noise, frame = 50*((int)(fs*0.001/2.0)*2). */
int    vso_vowel_noise(const int16_t *in, size_t n, int preset_key, float gain, float pre,
                       float snr_db_arg, int64_t fs, uint32_t seed, int16_t *out);
/* vso_vowel_noise's second half: the output noise of `vowel -n`, in place on already filtered PCM */
int    vso_noise(int16_t *out, size_t n, float snr_db, int64_t fs, uint32_t seed);
int16_t vso_round2int(double x);                                     /* vowel_new.c:413-427 */

#ifdef __cplusplus
}
#endif
#endif
