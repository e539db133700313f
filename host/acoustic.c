/* acoustic -- cycle-to-cycle measurements of a glottal-flow WAV on the GPU: F0, local jitter, local shimmer
 * (SURVEY.md 8f N4).  The reference's README (:14-16) describes `acoustic` analysis tools that are not in its tree;
 * this one makes the measurements vs_flow_analyze_batch() defines (include/voicesynth.h).
 *
 *   acoustic [-l lo] [-h hi] [-x] file.wav [file.wav ...]  thresholds of the onset trigger (default 0 0; with glottal
 *                                                          noise: above the noise, below the weakest pulse)
 * One line per file:  name  fs  samples  cycles  F0[Hz]  jitter[%]  shimmer[%]  mean_period  mean_peak
 * -x (voice report, vs_flow_report_batch) appends ten columns:  jitter_abs[us]  RAP[%]  PPQ5[%]  DDP[%]  shimmer[dB]
 *    APQ3[%]  APQ5[%]  APQ11[%]  DDA[%]  HNR[dB]   (nan where a measure needs more cycles, see include/voicesynth.h)
 *
 *   acoustic -F [-p order] file.wav [file.wav ...]         formant analysis of vowel PCM (vs_formant_batch, default
 *                                                          options; -p sets the LPC order, 2..32, even)
 * One line per file:  name  fs  samples  frames  analysed  F1..Fn[Hz]  B1..Bn[Hz]   (the means over the analysed frames,
 *    n = min(5, order/2); nan where no frame has that many formants) */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "voicesynth.h"
#include "vs_wav.h"

int main(int argc, char **argv)
{
    int lo = 0, hi = 0, a = 1, report = 0, formants = 0, order = 14;
    for (;;) {
        if (a < argc && strcmp(argv[a], "-x") == 0) {
            report = 1;
            a += 1;
        } else if (a < argc && strcmp(argv[a], "-F") == 0) {
            formants = 1;
            a += 1;
        } else if (a + 1 < argc && strcmp(argv[a], "-p") == 0) {
            order = atoi(argv[a + 1]);
            a += 2;
        } else if (a + 1 < argc && argv[a][0] == '-' && (argv[a][1] == 'l' || argv[a][1] == 'h') && argv[a][2] == 0) {
            if (argv[a][1] == 'l') lo = atoi(argv[a + 1]); else hi = atoi(argv[a + 1]);
            a += 2;
        } else {
            break;
        }
    }
    if (a >= argc || lo > hi || lo < -32768 || hi > 32767 || order < 2 || order > 32 || order % 2) {
        printf("usage: acoustic [-l lo] [-h hi] [-x] file.wav [file.wav ...]   (lo <= hi: thresholds of the onset trigger;"
               " -x: voice report columns)\n"
               "       acoustic -F [-p order] file.wav [file.wav ...]          (formants of vowel PCM; order even, 2..32)\n");
        return 0;
    }
    const size_t n = (size_t)(argc - a);
    int16_t **rows = (int16_t **)calloc(n, sizeof *rows);
    uint64_t *ns = (uint64_t *)calloc(n, sizeof *ns), *offs = (uint64_t *)calloc(n, sizeof *offs);
    int32_t *fs = (int32_t *)calloc(n, sizeof *fs);
    int16_t *tl = (int16_t *)calloc(n, sizeof *tl), *th = (int16_t *)calloc(n, sizeof *th);
    uint64_t total = 0;
    for (size_t i = 0; i < n; i++) {
        FILE *in = fopen(argv[a + i], "rb");
        if (!in) { printf(".wav file not found (%s)\n", argv[a + i]); return 1; }
        vs_wav_info wi;
        if (vs_wav_read_header(in, &wi) || wi.format_tag != 1 || wi.bits_per_sample != 16) { printf("%s: not a 16-bit PCM WAV file\n", argv[a + i]); return 1; }
        size_t k = 0;
        rows[i] = vs_wav_read_samples(in, &wi, &k);
        fclose(in);
        if (!rows[i]) { printf("Error while reading %s\n", argv[a + i]); return 1; }
        ns[i] = k; offs[i] = total; fs[i] = (int32_t)wi.sample_rate; tl[i] = (int16_t)lo; th[i] = (int16_t)hi;
        total += k;
    }
    int16_t *flow = (int16_t *)malloc((total ? total : 1) * sizeof *flow);
    for (size_t i = 0; i < n; i++) memcpy(flow + offs[i], rows[i], ns[i] * sizeof *flow);

    int dev = getenv("VS_DEVICE") ? atoi(getenv("VS_DEVICE")) : 0;
    vs_ctx *ctx = NULL;
    int rc = vs_ctx_create(&ctx, &dev, 1, 0);
    if (rc) { fprintf(stderr, "acoustic: no CUDA device: %s\n", vs_strerror(rc)); return 1; }
    if (formants) {
        vs_formant_opts fo = {25.0f, 10.0f, 50.0f, 700.0f, (uint32_t)order, (uint32_t)(order / 2 < 5 ? order / 2 : 5)};
        vs_formant_stats *fs_out = (vs_formant_stats *)calloc(n, sizeof *fs_out);
        rc = vs_formant_batch(ctx, flow, offs, ns, fs, n, &fo, fs_out, NULL, NULL);
        if (rc) { fprintf(stderr, "acoustic: %s (%s)\n", vs_strerror(rc), vs_last_error(ctx)); return 1; }
        for (size_t i = 0; i < n; i++) {
            printf("%s %d %llu %u %u", argv[a + i], fs[i], (unsigned long long)ns[i], fs_out[i].frames, fs_out[i].analysed);
            for (uint32_t k = 0; k < fo.n_formants; k++) printf(" %.1f", fs_out[i].f_mean_hz[k]);
            for (uint32_t k = 0; k < fo.n_formants; k++) printf(" %.1f", fs_out[i].bw_mean_hz[k]);
            printf("\n");
        }
        vs_ctx_destroy(ctx);
        return 0;
    }
    vs_flow_stats *st = (vs_flow_stats *)calloc(n, sizeof *st);
    vs_flow_report *rp = report ? (vs_flow_report *)calloc(n, sizeof *rp) : NULL;
    rc = report ? vs_flow_report_batch(ctx, flow, offs, ns, fs, tl, th, n, rp) : vs_flow_analyze_batch(ctx, flow, offs, ns, fs, tl, th, n, st);
    if (rc) { fprintf(stderr, "acoustic: %s (%s)\n", vs_strerror(rc), vs_last_error(ctx)); return 1; }
    for (size_t i = 0; i < n; i++) {
        if (report) st[i] = rp[i].base;
        if (st[i].flags & VS_STATS_OVERFLOW) {
            printf("%s %d %llu: %u onsets -- the thresholds lie inside an oscillation, raise them\n", argv[a + i], fs[i], (unsigned long long)ns[i], st[i].onsets);
            continue;
        }
        printf("%s %d %llu %u %.3f %.4f %.4f %.3f %.2f", argv[a + i], fs[i], (unsigned long long)ns[i], st[i].cycles,
               st[i].f0_hz, st[i].jitter_pct, st[i].shimmer_pct, st[i].mean_period, st[i].mean_peak);
        if (report)
            printf(" %.3f %.4f %.4f %.4f %.4f %.4f %.4f %.4f %.4f %.3f", rp[i].jitter_abs_us, rp[i].jitter_rap_pct, rp[i].jitter_ppq5_pct,
                   rp[i].jitter_ddp_pct, rp[i].shimmer_db, rp[i].shimmer_apq3_pct, rp[i].shimmer_apq5_pct, rp[i].shimmer_apq11_pct,
                   rp[i].shimmer_dda_pct, rp[i].hnr_db);
        printf("\n");
    }
    vs_ctx_destroy(ctx);
    return 0;
}
