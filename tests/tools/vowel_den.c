/* vowel_den.c -- TEST ONLY: the reference's vocal-tract filter (vowel_new.c:252-296, round2int :413-427) with the
 * denominator A[0..22] as an argument instead of one of its ten tables.  The same loop, in the same order and with the
 * same conversions, as the oracle's vso_vowel (oracle/vs_oracle.c); tests/test_tracts_host.py checks that the two
 * agree sample for sample on every preset table.  Build with -ffp-contract=off (tests/vowel_den_ref.py). */
#include <math.h>
#include <stddef.h>
#include <stdint.h>

#define ORDER 22

/* what `short = <double expr>` does on x86-64: cvttsd2si to 32 bits, keep the low 16 */
static int16_t d2s(double v)
{
    if (!(v > -2147483649.0 && v < 2147483648.0)) return 0;
    return (int16_t)(uint16_t)(uint32_t)(int32_t)v;
}

static int16_t round2int(double x)                                                 /* vowel_new.c:413-427 */
{
    double dec = x - floor(x);
    if (dec > 0.5) x = x + 1;
    if (x > 32767) x = 32767; else if (x < -32767) x = -32767;
    return d2s(floor(x));
}

int vowel_den(const int16_t *in, size_t n, const double *A, float gain, float pre, int16_t *out, double *raw)
{
    if (!A) return -1;
    double yd[ORDER + 1];
    for (int j = 0; j <= ORDER; j++) yd[j] = 0.0;
    for (size_t i = 0; i < n; i++) {
        yd[0] = 0.0 + (1.0 * (double)in[i]) * (double)gain;                          /* :266-269 */
        for (int j = 1; j <= ORDER; j++) yd[0] = yd[0] - A[j] * yd[j];                /* :279-281 */
        double v = yd[0] - (double)pre * yd[1];                                        /* :284 */
        if (raw) raw[i] = v;
        out[i] = round2int(v);
        for (int j = ORDER; j > 0; j--) yd[j] = yd[j - 1];                             /* :287-289 */
    }
    return 0;
}
