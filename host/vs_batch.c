/* vs_batch -- batch driver: many voices in one vs_synth_batch() call over all visible GPUs.
 *
 *   vs_batch -m manifest.txt [-G ngpus] [-S voices_per_slab] [-W writer_threads]
 *
 * Each manifest line describes one voice with the reference tools' own flags:
 *   <out.wav> <vowel> <seed> [flowgen_shimmer flags, e.g. -d 1 -f 120 -j 1 -s 3] [-V gain] [-P pre]
 * which is what   VS_SEED=<seed> flowgen_shimmer -o tmp.wav <flags>; vowel -i tmp.wav -o <out.wav> -v <vowel>
 * would produce, without the intermediate file.
 *
 * <vowel> is a preset key ('a','i','u','1'..'7') or a formant tract  f:F1/B1,F2/B2,...  (Hz, 1 to 11 formants),
 * built at the voice's own sampling rate (-r) by vs_tract_from_formants.  A slab with formant voices renders through
 * vs_synth_batch_tract (presets become tracts, identical (spec, rate) pairs share one entry, at most VS_MAX_TRACTS
 * distinct tracts per slab); a slab without any takes vs_synth_batch. */
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include "voicesynth.h"
#include "vs_cli.h"
#include "vs_wav.h"

#define MAXTOK 64
#define MAXFORMANTS 11

/* "f:F1/B1,F2/B2,..." -> den; 0, or -1 for a malformed spec, or the VS_E* code of vs_tract_from_formants */
static int formant_tract(const char *spec, int32_t fs, double den[23])
{
    float F[MAXFORMANTS + 1], B[MAXFORMANTS + 1];
    int k = 0;
    const char *c = spec + 2;
    while (*c) {
        char *e;
        if (k > MAXFORMANTS) return -1;
        F[k] = strtof(c, &e);
        if (e == c || *e != '/') return -1;
        c = e + 1;
        B[k] = strtof(c, &e);
        if (e == c || (*e != ',' && *e != 0)) return -1;
        k++;
        c = *e ? e + 1 : e;
    }
    if (k == 0) return -1;
    return vs_tract_from_formants(F, B, k, fs, den) ? -2 : 0;
}

/* ---- writer pool: a slab of voices is handed over as one job; the threads pull voices off it ---------- */
typedef struct {
    const int16_t *pcm;
    char **outs;
    const uint64_t *offs, *ns;
    const int32_t *fs;
    size_t n, next, done;
    int active;
} write_job;

typedef struct {
    pthread_t th[64];
    int nth, quit, errors;
    write_job job[2];                /* one per pinned buffer */
    pthread_mutex_t mu;
    pthread_cond_t work, idle;
} writer_pool;

static void *writer_main(void *arg)
{
    writer_pool *wp = arg;
    pthread_mutex_lock(&wp->mu);
    for (;;) {
        write_job *j = NULL;
        for (int k = 0; k < 2; k++)
            if (wp->job[k].active && wp->job[k].next < wp->job[k].n) { j = &wp->job[k]; break; }
        if (!j) {
            if (wp->quit) break;
            pthread_cond_wait(&wp->work, &wp->mu);
            continue;
        }
        const size_t i = j->next++;
        pthread_mutex_unlock(&wp->mu);
        int bad = 0;
        FILE *o = fopen(j->outs[i], "wb");
        if (!o) { perror(j->outs[i]); bad = 1; }
        else {
            if (vs_wav_write_header(o, (uint32_t)j->fs[i], (uint32_t)(j->ns[i] * 2))) bad = 1;
            if (fwrite(j->pcm + j->offs[i], 2, j->ns[i], o) != j->ns[i]) bad = 1;
            if (fclose(o)) bad = 1;
        }
        pthread_mutex_lock(&wp->mu);
        wp->errors += bad;
        if (++j->done == j->n) { j->active = 0; pthread_cond_broadcast(&wp->idle); }
    }
    pthread_mutex_unlock(&wp->mu);
    return NULL;
}

static void pool_start(writer_pool *wp, int nth)
{
    memset(wp, 0, sizeof *wp);
    pthread_mutex_init(&wp->mu, NULL);
    pthread_cond_init(&wp->work, NULL);
    pthread_cond_init(&wp->idle, NULL);
    wp->nth = nth;
    for (int i = 0; i < nth; i++) pthread_create(&wp->th[i], NULL, writer_main, wp);
}

static void pool_submit(writer_pool *wp, int slot, const int16_t *pcm, char **outs, const uint64_t *offs, const uint64_t *ns,
                        const int32_t *fs, size_t n)
{
    pthread_mutex_lock(&wp->mu);
    write_job *j = &wp->job[slot];
    j->pcm = pcm; j->outs = outs; j->offs = offs; j->ns = ns; j->fs = fs;
    j->n = n; j->next = 0; j->done = 0; j->active = n > 0;
    pthread_cond_broadcast(&wp->work);
    pthread_mutex_unlock(&wp->mu);
}

static void pool_wait(writer_pool *wp, int slot)       /* until the job that uses pinned buffer `slot` is on disk */
{
    pthread_mutex_lock(&wp->mu);
    while (wp->job[slot].active) pthread_cond_wait(&wp->idle, &wp->mu);
    pthread_mutex_unlock(&wp->mu);
}

static int pool_stop(writer_pool *wp)
{
    pthread_mutex_lock(&wp->mu);
    wp->quit = 1;
    pthread_cond_broadcast(&wp->work);
    pthread_mutex_unlock(&wp->mu);
    for (int i = 0; i < wp->nth; i++) pthread_join(wp->th[i], NULL);
    return wp->errors;
}

int main(int argc, char **argv)
{
    const char *manifest = NULL;
    int ngpu = 0, nwriters = 8;
    size_t slab = 0;
    for (int i = 1; i + 1 < argc; i += 2) {
        if (!strcmp(argv[i], "-m")) manifest = argv[i + 1];
        else if (!strcmp(argv[i], "-G")) ngpu = atoi(argv[i + 1]);
        else if (!strcmp(argv[i], "-S")) slab = (size_t)strtoull(argv[i + 1], NULL, 10);
        else if (!strcmp(argv[i], "-W")) nwriters = atoi(argv[i + 1]);
    }
    if (nwriters < 1) nwriters = 1;
    if (nwriters > 64) nwriters = 64;
    if (!manifest) { puts("usage: vs_batch -m manifest.txt [-G ngpus] [-S voices_per_slab] [-W writer_threads]\nline: <out.wav> <vowel> <seed> [flowgen_shimmer flags] [-V gain] [-P pre]"); return 0; }
    FILE *mf = fopen(manifest, "r");
    if (!mf) { perror(manifest); return 1; }

    size_t n = 0, cap = 0;
    vs_cli_flow *rows = NULL;
    char **outs = NULL;
    uint8_t *preset = NULL;
    char **spec = NULL;              /* formant spec of a voice, NULL for a preset voice */
    size_t *lineno = NULL, nline = 0, nformant = 0;
    uint32_t *seed = NULL;
    float *gain = NULL, *pre = NULL;
    char line[4096];
    while (fgets(line, sizeof line, mf)) {
        nline++;
        char *tok[MAXTOK];
        int nt = 0;
        for (char *t = strtok(line, " \t\r\n"); t && nt < MAXTOK; t = strtok(NULL, " \t\r\n")) tok[nt++] = t;
        if (nt == 0 || tok[0][0] == '#') continue;
        if (nt < 3) { fprintf(stderr, "vs_batch: line %zu: need <out> <vowel> <seed>\n", n + 1); return 1; }
        if (n == cap) {
            cap = cap ? cap * 2 : 1024;
            rows = realloc(rows, cap * sizeof *rows); outs = realloc(outs, cap * sizeof *outs);
            preset = realloc(preset, cap); seed = realloc(seed, cap * sizeof *seed);
            spec = realloc(spec, cap * sizeof *spec); lineno = realloc(lineno, cap * sizeof *lineno);
            gain = realloc(gain, cap * sizeof *gain); pre = realloc(pre, cap * sizeof *pre);
        }
        outs[n] = strdup(tok[0]);
        const int is_formant = !strncmp(tok[1], "f:", 2);
        preset[n] = is_formant ? (uint8_t)'a' : (uint8_t)tok[1][0];
        spec[n] = is_formant ? strdup(tok[1]) : NULL;
        lineno[n] = nline;
        nformant += is_formant;
        seed[n] = (uint32_t)strtoul(tok[2], NULL, 10);
        gain[n] = 10.0f; pre[n] = 1.0f;
        /* split our two extra flags from the flowgen flags */
        char *fargv[MAXTOK + 1];
        int fargc = 1;
        fargv[0] = "vs_batch";
        for (int i = 3; i < nt; i++) {
            if (!strcmp(tok[i], "-V") && i + 1 < nt) gain[n] = (float)atof(tok[++i]);
            else if (!strcmp(tok[i], "-P") && i + 1 < nt) pre[n] = (float)atof(tok[++i]);
            else fargv[fargc++] = tok[i];
        }
        if (fargc == 1) { fargv[fargc++] = "-d"; fargv[fargc++] = "1"; }
        if (vs_cli_parse_flow(fargc, fargv, 0, &rows[n])) { fprintf(stderr, "vs_batch: line %zu: bad flowgen flags\n", n + 1); return 1; }
        if (is_formant) {
            double den[23];
            const int frc = formant_tract(spec[n], rows[n].fs, den);
            if (frc) {
                fprintf(stderr, "vs_batch: line %zu: %s formant tract '%s' (want f:F1/B1,F2/B2,... with 1 to %d formants, 0 < F < fs/2 = %d/2, B > 0)\n",
                        nline, frc == -1 ? "malformed" : "out-of-range", spec[n], MAXFORMANTS, (int)rows[n].fs);
                return 1;
            }
        }
        n++;
    }
    fclose(mf);
    if (!n) return 0;

    /* AoS rows -> the SoA the ABI takes */
    float *dur = malloc(n * 4), *jit = malloc(n * 4), *shm = malloc(n * 4), *cq = malloc(n * 4), *K = malloc(n * 4),
          *Kv = malloc(n * 4), *F0 = malloc(n * 4), *DC = malloc(n * 4), *noise = malloc(n * 4);
    int32_t *amp = malloc(n * 4), *fs = malloc(n * 4);
    uint8_t *flags = malloc(n);
    for (size_t i = 0; i < n; i++) {
        dur[i] = rows[i].dur; jit[i] = rows[i].jitter; shm[i] = rows[i].shimmer; cq[i] = rows[i].cq; K[i] = rows[i].K;
        Kv[i] = rows[i].Kvar; F0[i] = rows[i].F0; DC[i] = rows[i].DC; noise[i] = rows[i].noise; amp[i] = rows[i].amp;
        fs[i] = rows[i].fs; flags[i] = rows[i].flags;
    }
    const vs_flow_params p = {dur, jit, shm, cq, K, Kv, F0, DC, noise, amp, fs, flags, seed};

    int count = vs_device_count();
    if (ngpu <= 0 || ngpu > count) ngpu = count;
    int devs[16];
    for (int d = 0; d < ngpu && d < 16; d++) devs[d] = d;
    vs_ctx *ctx = NULL;
    int rc = vs_ctx_create(&ctx, devs, ngpu, 0);
    if (rc) { fprintf(stderr, "vs_batch: %s\n", vs_strerror(rc)); return 1; }

    uint64_t *ns = malloc(n * sizeof *ns), *offs = malloc(n * sizeof *offs);
    vs_flow_nsamples(&p, n, ns);

    /* Slabs of consecutive voices, two pinned buffers: while the writer threads put slab k on disk the
     * GPUs render slab k+1 into the other buffer (SURVEY.md 8f N2: the file system is the bottleneck once
     * the kernels are fast). */
    if (slab == 0) slab = 16384;
    uint64_t buf_samples = 0;
    for (size_t a0 = 0; a0 < n; a0 += slab) {
        uint64_t tot = 0;
        for (size_t i = a0; i < n && i < a0 + slab; i++) { offs[i] = tot; tot += (ns[i] + 7) & ~7ull; }   /* 16-byte aligned rows */
        if (tot > buf_samples) buf_samples = tot;
    }
    /* the tract table of a slab with formant voices: presets and (spec, rate) pairs, each once */
    double *tden = NULL;
    uint8_t *tidx = NULL;
    if (nformant) {
        tden = malloc(sizeof(double) * 23 * VS_MAX_TRACTS);
        tidx = malloc(slab);
    }
    int16_t *buf[2];
    for (int k = 0; k < 2; k++) {
        buf[k] = vs_host_alloc(buf_samples * sizeof(int16_t));
        if (!buf[k]) { fprintf(stderr, "vs_batch: out of pinned memory\n"); return 1; }
    }
    writer_pool pool;
    pool_start(&pool, nwriters);
    double plan_ms = 0, render_ms = 0;
    unsigned long long samples = 0, launches = 0;
    struct timespec t0, t1;
    clock_gettime(CLOCK_MONOTONIC, &t0);
    size_t k = 0;
    for (size_t a0 = 0; a0 < n; a0 += slab, k++) {
        const size_t cnt = n - a0 < slab ? n - a0 : slab;
        int16_t *pcm = buf[k & 1];
        pool_wait(&pool, k & 1);                                   /* slab k-2 is on disk */
        vs_flow_params ps = {dur + a0, jit + a0, shm + a0, cq + a0, K + a0, Kv + a0, F0 + a0, DC + a0, noise + a0,
                             amp + a0, fs + a0, flags + a0, seed + a0};
        int any_formant = 0;
        for (size_t i = a0; i < a0 + cnt && !any_formant; i++) any_formant = spec[i] != NULL;
        if (!any_formant) {
            vs_filter_params fs_ = {preset + a0, gain + a0, pre + a0};
            rc = vs_synth_batch(ctx, &ps, &fs_, cnt, pcm, offs + a0, NULL);
        } else {
            /* entry t: a preset (key_spec[t] NULL, key_p[t] its key) or a formant spec at rate key_fs[t] */
            const char *key_spec[VS_MAX_TRACTS];
            int key_p[VS_MAX_TRACTS];
            int32_t key_fs[VS_MAX_TRACTS];
            uint32_t nt = 0;
            for (size_t i = a0; i < a0 + cnt; i++) {
                uint32_t t = 0;
                for (; t < nt; t++) {
                    if (spec[i] ? (key_spec[t] && key_fs[t] == fs[i] && !strcmp(key_spec[t], spec[i])) : (!key_spec[t] && key_p[t] == preset[i])) break;
                }
                if (t == nt) {
                    if (nt == VS_MAX_TRACTS) {
                        fprintf(stderr, "vs_batch: line %zu: more than %d distinct vocal tracts in one slab of %zu voices (lower -S)\n",
                                lineno[i], VS_MAX_TRACTS, slab);
                        return 1;
                    }
                    key_spec[nt] = spec[i]; key_p[nt] = preset[i]; key_fs[nt] = fs[i];
                    const int trc = spec[i] ? formant_tract(spec[i], fs[i], tden + 23 * nt) : vs_tract_from_preset(preset[i], tden + 23 * nt);
                    if (trc) { fprintf(stderr, "vs_batch: line %zu: bad vowel '%s'\n", lineno[i], spec[i] ? spec[i] : "?"); return 1; }
                    nt++;
                }
                tidx[i - a0] = (uint8_t)t;
            }
            vs_tract_params tp = {tden, nt, tidx, gain + a0, pre + a0};
            rc = vs_synth_batch_tract(ctx, &ps, &tp, cnt, pcm, offs + a0, NULL);
        }
        if (!rc) rc = vs_sync(ctx);
        if (rc) { fprintf(stderr, "vs_batch: %s (%s)\n", vs_strerror(rc), vs_last_error(ctx)); return 1; }
        vs_timing t;
        vs_get_timing(ctx, &t);
        plan_ms += t.plan_ms; render_ms += t.render_ms; samples += t.samples; launches += t.launches;
        pool_submit(&pool, k & 1, pcm, outs + a0, offs + a0, ns + a0, fs + a0, cnt);
    }
    pool_wait(&pool, 0);
    pool_wait(&pool, 1);
    const int werr = pool_stop(&pool);
    clock_gettime(CLOCK_MONOTONIC, &t1);
    const double wall = (double)(t1.tv_sec - t0.tv_sec) + 1e-9 * (double)(t1.tv_nsec - t0.tv_nsec);
    if (werr) { fprintf(stderr, "vs_batch: %d file(s) could not be written\n", werr); return 1; }
    printf("vs_batch: %zu voices, %llu samples on %d GPU(s) in %zu slab(s): plan %.3f ms, render %.3f ms, %llu launches; "
           "%.3f s with files (%d writer threads)\n", n, samples, ngpu, k, plan_ms, render_ms, launches, wall, nwriters);
    vs_host_free(buf[0]);
    vs_host_free(buf[1]);
    vs_ctx_destroy(ctx);
    return 0;
}
