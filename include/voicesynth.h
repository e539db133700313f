/* voicesynth.h -- C ABI of libvoicesynth_cuda (sm_100a).
 *
 * The reference (jsansao/voice_synth) has no in-process API: its only boundary is argv + WAV files
 * (SURVEY.md 8b).  This ABI is what a maintainer would bind in place of the two hot loops:
 *
 *   vs_flowgen_batch       replaces the per-period do{}while loop   flowgen_shimmer.c:246-423
 *   vs_vowel_filter_batch  replaces the framed IIR loop             vowel_new.c:237-331
 *   vs_synth_batch         replaces the pipeline  flowgen_shimmer | vowel  (README:31-33) for a
 *                          whole batch of independent voices; the int16 flow never reaches HBM
 *
 * Conventions
 *   - plain C, pointers + sizes, no CUDA or torch types in any signature;
 *   - return VS_OK (0) or a negative VS_E* code; the library never exits, prints or writes files;
 *   - no globals: vs_ctx owns devices, streams, constant tables, scratch and pinned staging;
 *   - the caller owns every I/O buffer.  pcm/flow/raw pointers may be HOST (pageable or pinned) or
 *     DEVICE memory of the ctx's device (detected with cudaPointerGetAttributes; device pointers
 *     need a single-device ctx).  Parameter arrays are always host memory;
 *   - all stream positions ("offsets") are in SAMPLES relative to the buffer pointer;
 *   - work is enqueued on the ctx's CUDA streams.  Calls whose I/O buffers are DEVICE memory return
 *     after enqueueing; call vs_sync() before touching the results (and to learn about device-side
 *     errors).  Calls with HOST buffers return when the data has landed (PCM travels over PCIe on
 *     a side stream, slab by slab, while the next slab renders; pinned buffers avoid staging);
 *   - there is NO CPU fallback: without a usable sm_100 device vs_ctx_create() fails.
 *
 * Arithmetic contract (tests/): pitch periods, amplitudes, pulse boundaries, random() draws and
 * the int16 flow are bit-exact with the reference; filtered waveforms are within 1e-5 max-abs
 * before quantisation and +-1 LSB after it (FP64 recurrence with FMA contraction).
 */
#ifndef VOICESYNTH_H
#define VOICESYNTH_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VS_ABI_VERSION 1

/* ---- error codes ---------------------------------------------------------------------------- */
#define VS_OK        0
#define VS_EINVAL   -1   /* NULL/ill-formed argument                                            */
#define VS_ERANGE   -2   /* a stream parameter is outside what the reference accepts or defines  */
#define VS_EPRESET  -3   /* vowel key not in "aiu1234567" (vowel_new.c:153-156,548-632)          */
#define VS_ENOMEM   -4   /* host or device allocation failed                                    */
#define VS_ECUDA    -5   /* CUDA runtime error; see vs_last_error()                             */
#define VS_ENODEV   -6   /* no usable sm_100 device / bad device index                          */
#define VS_EOVERLAP -7   /* output rows overlap each other (or, for device buffers, the filter's input), or a stream
                            exceeds the 2^31-1 samples limit                                    */

/* ---- stream flags: "the argument was given" bits the reference main loop tests -------------- */
#define VS_F_JITTER  0x01u   /* -j given  (flowgen_shimmer.c:248: arg.jitter != -1)             */
#define VS_F_SHIMMER 0x02u   /* -s given  (flowgen_shimmer.c:295)                               */
#define VS_F_NOISE   0x04u   /* -n given  (flowgen_shimmer.c:373)                               */

typedef struct vs_ctx vs_ctx;

/* Flow (glottal source) parameters, SoA: one entry per stream, same meaning, units and C type as
 * `struct PAR` after initialization() (flowgen_shimmer.c:73-87, 463-547).  A NULL array means the
 * reference default for every stream (flowgen_shimmer.c:87).  */
typedef struct vs_flow_params {
    const float    *dur;      /* seconds (default 1.0); samples = (uint64)((float)fs * dur) (:242)  */
    const float    *jitter;   /* fraction = CLI % / 100.0 (default 0)                              */
    const float    *shimmer;  /* fraction = CLI % / 100   (default 0)                              */
    const float    *cq;       /* closed quotient (0.55)                                            */
    const float    *K;        /* speed of closure (0.65)                                           */
    const float    *Kvar;     /* closure-speed variation (0)                                       */
    const float    *F0;       /* Hz (120)                                                          */
    const float    *DC;       /* DC flow in SAMPLE units: CLI fraction * amp, or .25 with -n (:182,:524) */
    const float    *noise;    /* linear cycle SNR = (float)pow(10, dB/10) (:511); used with VS_F_NOISE */
    const int32_t  *amp;      /* peak amplitude (12000)                                            */
    const int32_t  *fs;       /* sampling rate (22050)                                             */
    const uint8_t  *flags;    /* VS_F_* (default 0)                                                */
    const uint32_t *seed;     /* srandom() seed per stream (default 1); the reference uses time(NULL) (:241) */
} vs_flow_params;

/* Vocal-tract filter parameters, SoA (vowel_new.c:76-77, 116-192). NULL = reference default. */
typedef struct vs_filter_params {
    const uint8_t *preset;    /* 'a','i','u','1'..'7' (default 'a')                                */
    const float   *gain;      /* default 10.0f                                                     */
    const float   *pre;       /* pre-emphasis, default 1.0f                                        */
} vs_filter_params;

/* One record per pitch period: everything the reference computes (and prints) per period. */
typedef struct vs_period_rec {
    int32_t  T, T2, T3, T4;   /* period length, rise time, closure instant, DC-crossing instant    */
    float    A, Knew, S;      /* amplitude, closure speed, shimmer draw (printed "%5.2f \n", :307) */
    int32_t  ndraws;          /* random() calls consumed by this period                            */
    int32_t  ndw;             /* par.NoiseDistWidth (:382), 0 without VS_F_NOISE                   */
    float    x_pow, w_pow;    /* signal / noise power of the period; SNRdb = 10*log10(x_pow/w_pow) (:409) */
    uint32_t reserved;
    uint64_t start;           /* index of the period's first sample                                */
} vs_period_rec;

/* Optional per-period log.  rec has room for rec_offsets[n] records; stream i owns
 * rec[rec_offsets[i] .. rec_offsets[i+1]) and needs at least vs_flow_max_periods() of them. */
typedef struct vs_period_log {
    vs_period_rec  *rec;          /* host memory */
    const uint64_t *rec_offsets;  /* [n+1], host */
    uint32_t       *count;        /* [n], host: periods written per stream */
} vs_period_log;

/* Timing of the most recent batch call, measured with CUDA events on the ctx's compute stream of
 * device slot 0 (valid after vs_sync). */
typedef struct vs_timing {
    float    plan_ms;         /* period-plan kernel(s)                                   */
    float    render_ms;       /* flow / filter / fused render kernel(s)                  */
    float    total_ms;        /* first launch .. last launch or copy on slot 0           */
    uint32_t launches;        /* kernels launched by the call (all device slots)         */
    uint32_t chunks;          /* time-chunks the streams were split into                 */
    uint64_t samples;         /* output samples produced                                 */
    uint64_t warmup_samples;  /* extra samples filtered only to settle chunk carries     */
    uint64_t h2d_bytes;       /* host->device bytes the call copied (descriptors, tables, flow_in) */
    uint64_t d2h_bytes;       /* device->host bytes the call copied (PCM, raw, period log)         */
    uint32_t render_path;     /* which render kernel ran (last launch): bit 0 = branch-free generator, bit 1 = glottal-noise
                                 variant, bits 2-3 = filter arithmetic (0 integer pre-emphasis, 1 FMA, 2 exact),
                                 bit 5 = flow only on the warp-per-row kernel (lanes along the row),
                                 bit 6 = caller-defined tract coefficients (vs_*_batch_tract)                          */
    uint32_t reserved;
} vs_timing;

/* ---- options (vs_ctx_set_option) ------------------------------------------------------------ */
#define VS_OPT_CHUNK_SAMPLES   1  /* time-chunk length; 0 = auto (fill the SMs), <0 = never chunk      */
#define VS_OPT_CARRY_TOL       2  /* relative size the free response must decay to during warm-up (1e-12) */
#define VS_OPT_EXACT_FILTER    3  /* 1: unfused mul+sub in the reference's order (bit-exact, 2x FP64 work, no chunking) */
#define VS_OPT_SLAB_STREAMS    4  /* streams per launch/copy slab for host outputs; 0 = auto            */
#define VS_OPT_TARGET_WARPS    5  /* no effect; a value > 0 is accepted for compatibility                */
#define VS_OPT_ASYNC_HOST      7  /* 1: calls with PINNED host buffers also return after enqueueing; the
                                     PCM of call k crosses PCIe while call k+1 renders (two device
                                     scratch buffers alternate).  vs_sync() before reading.  (0)          */
#define VS_OPT_PLAN_WARPS      8  /* period-table kernel: 1 = one warp per stream, 0 = one thread per
                                     stream, -1 = auto: warps for small batches and glottal noise (-1)    */

#define VS_OPT_SIMPLE_GEN      9  /* 1: render with the general (per-sample, branching) generator even where
                                     the branch-free one applies -- for A/B checks (0)                    */

/* ---- context -------------------------------------------------------------------------------- */
int         vs_ctx_create(vs_ctx **out, const int *devices, int n_devices, uint32_t flags);
void        vs_ctx_destroy(vs_ctx *ctx);
int         vs_ctx_set_option(vs_ctx *ctx, int option, double value);
/* use an existing cudaStream_t (passed as void*) as the compute stream of device slot `slot` */
int         vs_ctx_set_stream(vs_ctx *ctx, int slot, void *cuda_stream);
int         vs_sync(vs_ctx *ctx);
int         vs_get_timing(vs_ctx *ctx, vs_timing *out);
const char *vs_strerror(int code);
const char *vs_last_error(vs_ctx *ctx);
int         vs_abi_version(void);
int         vs_device_count(void);

/* DFMA throughput of device slot 0 (8 independent chains/thread, all SMs): the FP64-pipe roofline
 * denominator.  *sm_mhz_out (nullable) = the SM clock this rate implies at 64 DFMA/clk/SM. */
int         vs_measure_fp64_peak(vs_ctx *ctx, double *tflops_out, double *sm_mhz_out);

/* pinned host memory for zero-staging transfers */
void       *vs_host_alloc(size_t bytes);
void        vs_host_free(void *p);

/* ---- host-side helpers (no GPU work) -------------------------------------------------------- */
/* samples per stream, (uint64)((float)fs*dur) as in flowgen_shimmer.c:242 */
int vs_flow_nsamples(const vs_flow_params *p, size_t n, uint64_t *nsamples_out);
/* upper bound on the number of pitch periods per stream (for vs_period_log sizing) */
int vs_flow_max_periods(const vs_flow_params *p, size_t n, uint64_t *max_periods_out);
/* validate parameters exactly as the batch calls do; *bad_index (nullable) = first offender */
int vs_flow_validate(const vs_flow_params *p, size_t n, size_t *bad_index);
/* warm-up samples the chunked filter uses for a preset at the ctx's carry tolerance */
int vs_filter_warmup(vs_ctx *ctx, int preset_key, float gain);

/* ---- the three batch entry points ----------------------------------------------------------- */

/* n glottal-flow streams.  Stream i writes vs_flow_nsamples()[i] int16 samples at
 * pcm_out + offsets[i]  (offsets NULL: dense rows of stride max_i nsamples). */
int vs_flowgen_batch(vs_ctx *ctx, const vs_flow_params *p, size_t n,
                     int16_t *pcm_out, const uint64_t *offsets, vs_period_log *log);

/* n independent filters.  Stream i reads nsamp[i] int16 samples at flow_in + in_offsets[i] and
 * writes as many at pcm_out + out_offsets[i] (NULL offsets: dense rows of stride max nsamp).
 * raw_out (nullable, same offsets as pcm_out) receives the FP64 pre-quantisation waveform. */
int vs_vowel_filter_batch(vs_ctx *ctx, const int16_t *flow_in, const uint64_t *in_offsets,
                          const uint64_t *nsamp, const vs_filter_params *f, size_t n,
                          int16_t *pcm_out, const uint64_t *out_offsets, double *raw_out);

/* SURVEY 8f N4 -- cycle-to-cycle analysis of glottal flow (the measurements of the reference's `acoustic` tools,
 * README:14-16; their code is not in the reference tree, so the definitions below are this library's own).
 * Per stream, with thresholds lo[i] <= hi[i] (NULL: 0, the closed-phase level of a flow generated without -l):
 *   a trigger, armed at the start and by every sample x <= lo, fires at the first sample x > hi while armed: an ONSET
 *   (for noise-free flow with lo = hi = (short)DC: the second sample of every pitch period);
 *   cycle k = [onset k, onset k+1), length T_k, peak P_k = its largest sample;
 *   mean_period = mean T_k, mean_peak = mean P_k, f0_hz = fs / mean_period,
 *   jitter_pct  = 100 * mean |T_k - T_k-1| / mean_period   (local jitter),
 *   shimmer_pct = 100 * mean |P_k - P_k-1| / mean_peak     (local shimmer);
 * sums are exact integers, the quotients FP64 rounded to float.  With glottal noise put the thresholds above the
 * noise (e.g. 25 % and 50 % of the amplitude).  flow may be host or device memory; stats is host memory. */
typedef struct vs_flow_stats {
    uint32_t onsets;       /* trigger events found                                       */
    uint32_t cycles;       /* complete cycles = onsets - 1 (0 if flags != 0)             */
    uint32_t flags;        /* VS_STATS_OVERFLOW: more than nsamp/16 + 4 onsets           */
    float    f0_hz, jitter_pct, shimmer_pct, mean_period, mean_peak;
} vs_flow_stats;
#define VS_STATS_OVERFLOW 1u
int vs_flow_analyze_batch(vs_ctx *ctx, const int16_t *flow, const uint64_t *offsets, const uint64_t *nsamp,
                          const int32_t *fs, const int16_t *lo, const int16_t *hi, size_t n, vs_flow_stats *stats);

/* Voice report: vs_flow_stats plus the perturbation quotients of Praat's voice report and a cycle-synchronous
 * harmonics-to-noise ratio.  Same arguments, checks and error codes as vs_flow_analyze_batch; `base` is byte for
 * byte what that call returns for the same stream and thresholds.  With K = base.cycles complete cycles k = 0..K-1
 * of the trigger above, their lengths T_k, peaks P_k and means mean T, mean P (Praat's formulas, without its
 * period-exclusion rules):
 *   jitter_abs_us   = 1e6 * (sum_{k>=1} |T_k - T_k-1| / (K-1)) / fs                              K >= 2
 *   jitter_rap_pct  = 100 * (sum_{k=1..K-2} |3 T_k - (T_k-1 + T_k + T_k+1)| / 3 / (K-2)) / mean T   K >= 3
 *   jitter_ppq5_pct = the same with the 5-point window: k = 2..K-3, / 5 / (K-4)                 K >= 5
 *   jitter_ddp_pct  = 100 * (sum_{k=1..K-2} |T_k+1 - 2 T_k + T_k-1| / (K-2)) / mean T  (= 3 * RAP)  K >= 3
 *   shimmer_apq3_pct, shimmer_apq5_pct, shimmer_dda_pct: RAP, PPQ5 and DDP applied to P_k over mean P;
 *   shimmer_apq11_pct: the 11-point window, k = 5..K-6, / 11 / (K-10), K >= 11; all four need mean P > 0
 *   shimmer_db      = sum_{k>=1} |20 log10(P_k / P_k-1)| / (K-1)                      K >= 2 and every P_k > 0
 *   hnr_db, by cycle-synchronous averaging (Yumoto, Gould and Baer 1982): L = hnr_len = min T_k; the cycles are
 *   aligned at their onsets o_k, S_j = sum_k x[o_k + j] and E = sum_k sum_{j<L} x[o_k + j]^2 for j < L;
 *     hnr_db = 10 log10( sum_j S_j^2 / (K E - sum_j S_j^2) ),  +inf when the denominator is 0;   K >= 2
 *   The average of the aligned cycles is the harmonic part, the rest is noise.  Amplitude perturbation counts as
 *   noise: 3 % shimmer alone brings a noise-free voice down to about 10 dB.  This generator's jitter only changes
 *   the closed phase, after the first L samples of a cycle, so a jitter-only noise-free voice gives +inf.  For
 *   noise-only voices hnr_db is the SNR of the period log, sum x_pow (T3 - T4) / sum w_pow T, within 0.1 dB
 *   (about 2.2 dB below the -n value, which relates the open phase's power to the noise).
 * Sums are exact integers (S_j and E in int64, K E and sum S_j^2 in 128 bits) up to the final FP64 quotient,
 * except the logarithms of shimmer_db; each field is rounded to float.  A field whose condition fails is NaN;
 * hnr_len is L when hnr_db is defined (K >= 2), else 0.  With VS_STATS_OVERFLOW in base.flags every new field is
 * NaN and hnr_len is 0. */
typedef struct vs_flow_report {
    vs_flow_stats base;        /* what vs_flow_analyze_batch returns                          */
    float    jitter_abs_us;    /* local absolute jitter                                       */
    float    jitter_rap_pct, jitter_ppq5_pct, jitter_ddp_pct;
    float    shimmer_db, shimmer_apq3_pct, shimmer_apq5_pct, shimmer_apq11_pct, shimmer_dda_pct;
    float    hnr_db;           /* cycle-synchronous average, above                            */
    uint32_t hnr_len;          /* L: samples per cycle the HNR compares                       */
    uint32_t reserved;
} vs_flow_report;              /* 80 bytes */
int vs_flow_report_batch(vs_ctx *ctx, const int16_t *flow, const uint64_t *offsets, const uint64_t *nsamp,
                         const int32_t *fs, const int16_t *lo, const int16_t *hi, size_t n, vs_flow_report *out);

/* Formant analysis of PCM (vowels rendered by vs_synth_batch, vs_vowel_filter_batch and their tract forms): frame-wise
 * LPC, its poles, and per-stream formant statistics.  The definitions are this library's own (the reference has no
 * formant tool); tests/formant_ref.py restates them in numpy.  With fs the stream's rate (fs NULL: 22050 for every
 * stream) and p = order:
 *   frames     Nw = lround(win_ms fs / 1000), H = lround(hop_ms fs / 1000), in double; a stream of n samples has
 *              n >= Nw ? (n - Nw) / H + 1 : 0 frames, frame f covers samples [f H, f H + Nw);
 *   signal     y[m] = (x[fH+m] - mu x[fH+m-1]) w[m], m = 0..Nw-1, in FP64, mu = exp(-2 pi preemph_hz / fs) (0 when
 *              preemph_hz is 0), w[m] = 0.54 - 0.46 cos(2 pi m / (Nw - 1)); x[-1] = 0 only at the stream's first
 *              sample.  w and mu are computed on the host with libm in double;
 *   LPC        r[k] = sum_m y[m] y[m+k], k = 0..p, FP64 in any order; r[0] == 0: the frame is VS_FRAME_SILENT.
 *              Levinson-Durbin gives A(z) = 1 + a1 z^-1 + ... + ap z^-p; a reflection coefficient with |k_i| >= 1 or a
 *              prediction error <= 0: VS_FRAME_SINGULAR (a numerical guard: for a frame that is not all zero the
 *              autocorrelation matrix is positive definite, and no input is known to reach it);
 *   poles      all p roots of z^p + a1 z^(p-1) + ... + ap in FP64 (Aberth-Ehrlich from 0.9 exp(i (2 pi j / p + 0.4)),
 *              until every root's correction is at most 1e-13 of its modulus, at most 64 iterations, then one Newton
 *              step; more iterations needed: VS_FRAME_NOCONV).  Each root with Im z > 0 gives
 *              F = atan2(Im z, Re z) fs / (2 pi) and B = -ln|z| fs / pi; kept when 50 < F < fs/2 - 50 and, when
 *              bmax_hz > 0, B < bmax_hz; sorted by ascending F, the first n_formants are the frame's formants;
 *   frames[]   f_hz[k], bw_hz[k] for k < found (float), NaN past it; a flagged frame has found = 0;
 *   stats      over the frames without a flag ("analysed"): count[k] = frames with found > k, the mean of F_k, its
 *              sample SD (NaN for count[k] < 2) and the mean of B_k, in FP64 from the unrounded values, each rounded
 *              to float; NaN where count[k] == 0.  frames = the stream's frames, unconverged = its VS_FRAME_NOCONV
 *              frames.
 * Errors (vs_formant_frames returns the same ones, in the same order): NULL ctx / pcm / nsamp / stats, an odd order or
 * one outside 2..32, n_formants outside 1..VS_MAX_FORMANTS or above p/2 -> VS_EINVAL; a negative (or NaN) preemph_hz
 * or bmax_hz, then per stream in index order: a row above 2^31-1 samples -> VS_EOVERLAP; fs <= 0, Nw < p+1,
 * Nw > VS_FORMANT_MAX_WIN (the kernel stages a frame in shared memory), H < 1 or H > 2^31-1 -> VS_ERANGE.
 * pcm may be host or device memory (as for vs_flow_analyze_batch); offsets NULL: dense rows of stride max nsamp.
 * stats [n] and frames are host memory; stream i's frames go to frames + frame_offsets[i] (frame_offsets NULL: the
 * prefix sum of the frame counts, densely packed); frames NULL: no per-frame output, the statistics are the same. */
#define VS_MAX_FORMANTS     8
#define VS_FORMANT_MAX_WIN  4096
#define VS_FRAME_SILENT     1u
#define VS_FRAME_SINGULAR   2u
#define VS_FRAME_NOCONV     4u
typedef struct vs_formant_opts {      /* NULL = all defaults; a non-NULL struct is taken literally    */
    float    win_ms;                  /* Hamming window length (25)                                   */
    float    hop_ms;                  /* frame step (10)                                              */
    float    preemph_hz;              /* pre-emphasis corner, 0 = none (50)                           */
    float    bmax_hz;                 /* drop poles with bandwidth >= bmax; 0 = no limit (700)        */
    uint32_t order;                   /* LPC order p, even, 2..32 (14)                                */
    uint32_t n_formants;              /* 1..VS_MAX_FORMANTS and <= p/2 (5)                            */
} vs_formant_opts;

typedef struct vs_formant_frame {     /* 72 bytes */
    float    f_hz[VS_MAX_FORMANTS], bw_hz[VS_MAX_FORMANTS];   /* ascending F; NaN past `found`                */
    uint32_t found;                   /* formants found in the frame                                  */
    uint32_t flags;                   /* VS_FRAME_SILENT | VS_FRAME_SINGULAR | VS_FRAME_NOCONV        */
} vs_formant_frame;

typedef struct vs_formant_stats {     /* 144 bytes */
    uint32_t frames, analysed, unconverged, reserved;
    uint32_t count[VS_MAX_FORMANTS];  /* analysed frames with found > k                               */
    float    f_mean_hz[VS_MAX_FORMANTS], f_sd_hz[VS_MAX_FORMANTS], bw_mean_hz[VS_MAX_FORMANTS];
} vs_formant_stats;

/* host only: validates exactly as vs_formant_batch does (first offender -> its error) and returns frames per stream */
int vs_formant_frames(const vs_formant_opts *o, const uint64_t *nsamp, const int32_t *fs, size_t n, uint64_t *frames_out);
int vs_formant_batch(vs_ctx *ctx, const int16_t *pcm, const uint64_t *offsets, const uint64_t *nsamp, const int32_t *fs,
                     size_t n, const vs_formant_opts *o, vs_formant_stats *stats,
                     vs_formant_frame *frames, const uint64_t *frame_offsets);

/* Pitch and harmonicity of PCM (the F0 and noise axes of rendered vowels): Boersma's (1993) autocorrelation corrected
 * for the window, frame by frame, without Praat's path finder; the options and their defaults are those of Praat's
 * "To Pitch (ac)" (periods = 4.5 gives the window of "To Harmonicity (ac)").  The definitions are the library's own;
 * tests/pitch_ref.py restates them in numpy.  With fs the stream's rate (fs NULL: 22050 for every stream):
 *   geometry   Nw = lround(periods fs / f_min), H = lround(hop_ms fs / 1000), tau_lo = max(2, ceil(fs / f_max)),
 *              tau_hi = floor(fs / f_min), all in double; a stream of n samples has n >= Nw ? (n - Nw) / H + 1 : 0
 *              frames, frame f covers samples [f H, f H + Nw);
 *   signal     mu_f = the frame's mean (an exact integer sum over Nw), a[m] = x[fH+m] - mu_f, the local peak
 *              P_f = max |a[m]|; w[m] = 0.5 - 0.5 cos(2 pi (m + 1/2) / Nw), y[m] = a[m] w[m], in FP64.  w and r_w are
 *              computed on the host with libm in double, r_w in index order;
 *   lags       r_a(tau) = sum_{m < Nw - tau} y[m] y[m+tau] in FP64 in any order, for tau = 0 and tau_lo-1 .. tau_hi+1;
 *              r_w(tau) the same sum over w; r(tau) = (r_a(tau) / r_a(0)) (r_w(0) / r_w(tau)).  r_a(0) == 0 (a constant
 *              frame): VS_PITCH_SILENT;
 *   candidate  a tau in [tau_lo, tau_hi] with r(tau) > r(tau-1), r(tau) >= r(tau+1) and r(tau) > 0.  With a, b, c =
 *              r(tau-1), r(tau), r(tau+1): d = 0.5 (a - c) / (a - 2b + c), tau* = tau + d, r* = b - 0.25 (a - c) d, and
 *              r* > 1 (the parabola overshoots) becomes 1 / r*.  Strength S = r* - octave_cost log2(f_min tau* / fs);
 *              the largest S wins, a tie goes to the smaller tau.  No candidate: VS_PITCH_NOPEAK;
 *   per stream G = max_f P_f.  A frame without a flag is VS_PITCH_QUIET when P_f < silence_threshold G; a frame with
 *              none of these three flags is "periodic", and VS_PITCH_VOICED as well when r* >= voicing_threshold.
 *              F0 = fs / tau* (voiced frames), hnr_db = 10 log10(r* / (1 - r*)) (periodic frames; +inf for r* = 1);
 *   frames[]   f0_hz (NaN unless voiced), strength = r* (NaN for SILENT and NOPEAK), hnr_db (NaN unless periodic), flags;
 *   stats      the stream's frames, periodic and voiced frames; over the voiced frames the mean, sample SD, min and max
 *              of F0; over the periodic frames the mean and sample SD of hnr_db and the mean r*.  FP64 from the unrounded
 *              values in two passes (the means, then the squared deviations), each rounded to float; NaN where a
 *              statistic has no frame (an SD: fewer than two); an hnr_db of +inf makes the mean +inf and the SD NaN.
 * Errors (vs_pitch_frames returns the same ones, in the same order): NULL ctx / pcm / nsamp / stats -> VS_EINVAL; an
 * option that is not finite, f_min_hz <= 0, f_max_hz <= f_min_hz, periods < 2, a threshold outside [0, 1] or
 * octave_cost < 0 -> VS_ERANGE; then per stream in index order: a row above 2^31-1 samples -> VS_EOVERLAP; fs <= 0,
 * tau_lo >= tau_hi, tau_hi + 1 >= Nw, Nw > VS_PITCH_MAX_WIN (the kernel stages a frame in shared memory), H < 1 or
 * H > 2^31-1 -> VS_ERANGE.  Input, offsets, staging, stats and frame placement (frame_offsets) are as for
 * vs_formant_batch; frames NULL: no per-frame output, the statistics are the same. */
#define VS_PITCH_MAX_WIN    4096
#define VS_PITCH_SILENT     1u
#define VS_PITCH_NOPEAK     2u
#define VS_PITCH_QUIET      4u
#define VS_PITCH_VOICED     8u
typedef struct vs_pitch_opts {        /* NULL = all defaults; a non-NULL struct is taken literally    */
    float    f_min_hz;                /* pitch floor: the longest lag and, with periods, the window (75) */
    float    f_max_hz;                /* pitch ceiling: the shortest lag (600)                        */
    float    periods;                 /* window length in periods of f_min, >= 2 (3)                  */
    float    hop_ms;                  /* frame step (10)                                              */
    float    voicing_threshold;       /* r* at which a periodic frame is voiced, 0..1 (0.45)          */
    float    silence_threshold;       /* local peak below this share of the stream's peak: QUIET (0.03) */
    float    octave_cost;             /* favours the shorter of two similar lags, >= 0 (0.01)         */
} vs_pitch_opts;

typedef struct vs_pitch_frame {       /* 16 bytes */
    float    f0_hz, strength, hnr_db;
    uint32_t flags;                   /* VS_PITCH_*                                                   */
} vs_pitch_frame;

typedef struct vs_pitch_stats {       /* 48 bytes */
    uint32_t frames, periodic, voiced;
    float    f0_mean_hz, f0_sd_hz, f0_min_hz, f0_max_hz;   /* voiced frames                             */
    float    hnr_mean_db, hnr_sd_db, strength_mean;         /* periodic frames                           */
    uint32_t reserved[2];
} vs_pitch_stats;

/* host only: validates exactly as vs_pitch_batch does (first offender -> its error) and returns frames per stream */
int vs_pitch_frames(const vs_pitch_opts *o, const uint64_t *nsamp, const int32_t *fs, size_t n, uint64_t *frames_out);
int vs_pitch_batch(vs_ctx *ctx, const int16_t *pcm, const uint64_t *offsets, const uint64_t *nsamp, const int32_t *fs,
                   size_t n, const vs_pitch_opts *o, vs_pitch_stats *stats, vs_pitch_frame *frames,
                   const uint64_t *frame_offsets);

/* Voice report of vowel PCM (the jitter and shimmer axes of rendered vowels, which vs_flow_report_batch measures only on
 * glottal flow): period marks by cross-correlation guided by the pitch track, in the spirit of Praat's "To PointProcess
 * (periodic, cc)", then the voice report above on those marks.  The definitions are the library's own; they make every
 * mark an exact integer decided by exact integer sums.  tests/vowel_report_ref.py restates them in numpy.  Per stream,
 * with x the PCM, fs its rate and the options o (NULL: the defaults of vs_pitch_opts):
 *   track      the frames of vs_pitch_batch with the same options, and its Nw and H;
 *   run        the longest sequence of consecutive VS_PITCH_VOICED frames f_a .. f_b (the first of equal ones); its
 *              samples are [s, e) = [f_a H, f_b H + Nw).  No voiced frame: run_frames = 0, no mark, and rep is the report
 *              of an empty onset list (onsets = cycles = 0, every quotient NaN);
 *   period     T(t) = fs / (double)f0_hz with f0_hz the float frame record of frame f = clamp(floor((t - floor(Nw/2) +
 *              floor(H/2)) / H), f_a, f_b) (integer arithmetic), and L(t) = lround(T(t));
 *   anchor     m_0 = the first index of max |x| in [c - floor(L(c)/2), c - floor(L(c)/2) + L(c)), the period around the
 *              centre c = s + floor(Nw/2) of the run's first frame (a voiced frame's window may begin in silence);
 *   step       from m_k, with T = T(m_k) and L = lround(T), and only while every candidate's period lies in the run
 *              (m_k + lround(VS_MARK_STEP_MAX T) + L <= e): the candidates are the m in
 *              [m_k + lround(VS_MARK_STEP_MIN T), m_k + lround(VS_MARK_STEP_MAX T)];
 *              C(m) = sum_{j<L} x[m_k+j] x[m+j] and E(p) = sum_{j<L} x[p+j]^2, exact integers;
 *              r(m) = C(m) / sqrt((double)E(m_k) (double)E(m)) (IEEE multiply, square root and divide; 0 when the
 *              product is 0).  The largest r wins, a tie goes to the smaller m; m_k+1 is the winner unless there is no
 *              candidate or the best r <= 0, which ends the marks;
 *   report     the marks m_0 < ... < m_K-1 (stream coordinates) are the onsets of the vs_flow_report definitions, with
 *              x the PCM: base.onsets = K, base.cycles = K - 1, the peaks P_k the largest sample of each period, the
 *              quotients and the cycle-synchronous HNR.
 * vs_vowel_mark_slots bounds the marks of a stream (base.flags is never VS_STATS_OVERFLOW): with tau_lo of the pitch
 * geometry every step is at least lround(VS_MARK_STEP_MIN T_lo) >= 1 samples, T_lo = (tau_lo - 1/2) (1 - 2^-20) below
 * any period a frame record can publish; a stream of n >= Nw samples has at most (n - 1) / step + 1 marks, 0 below Nw.
 * Errors (vs_vowel_mark_slots returns the same ones, in the same order): NULL ctx / pcm / nsamp / out -> VS_EINVAL, then
 * those of vs_pitch_batch.  Input, offsets and staging are as for vs_pitch_batch.  marks (nullable) and mark_offsets are
 * host memory: stream i's base.onsets marks go to marks + mark_offsets[i] (mark_offsets NULL: the prefix sum of the
 * slots, densely packed); marks NULL: no marks are written, out is the same. */
#define VS_MARK_STEP_MIN 0.8
#define VS_MARK_STEP_MAX 1.25
typedef struct vs_vowel_report {      /* 96 bytes */
    vs_flow_report rep;               /* the voice report over the marks: rep.base.onsets = marks, .cycles = periods */
    uint32_t run_frame, run_frames;   /* the analysed voiced run, in pitch frames; run_frames 0: no voiced frame     */
    uint32_t run_start, run_len;      /* the same run in samples                                                    */
} vs_vowel_report;

/* host only: validates exactly as vs_vowel_report_batch does; per stream the number of mark slots it may fill */
int vs_vowel_mark_slots(const vs_pitch_opts *o, const uint64_t *nsamp, const int32_t *fs, size_t n, uint64_t *slots_out);
int vs_vowel_report_batch(vs_ctx *ctx, const int16_t *pcm, const uint64_t *offsets, const uint64_t *nsamp,
                          const int32_t *fs, size_t n, const vs_pitch_opts *o, vs_vowel_report *out,
                          uint32_t *marks, const uint64_t *mark_offsets);

/* SURVEY 8f N1 -- `vowel -n`: white noise added to already filtered PCM, IN PLACE (vowel_new.c:302-324).
 * Per stream and per frame of 50*((int)(fs*0.001/2.0)*2) samples: float power of the frame, uniform
 * noise of width sqrt(12*power/snr) drawn with random() seeded by srandom(seed[i]) (vowel_new.c:234),
 * round2int() again.  snr = (float)pow(10, dB/10) as the tool computes it (:143); streams with
 * snr[i] <= 0 are left untouched.  pcm may be host or device memory. */
int vs_vowel_noise_batch(vs_ctx *ctx, int16_t *pcm, const uint64_t *offsets, const uint64_t *nsamp,
                         const float *snr, const int32_t *fs, const uint32_t *seed, size_t n);

/* n voices, flow generation fused with the filter: only the final PCM is written. */
int vs_synth_batch(vs_ctx *ctx, const vs_flow_params *p, const vs_filter_params *f, size_t n,
                   int16_t *pcm_out, const uint64_t *offsets, double *raw_out);

/* ---- caller-defined vocal tracts ------------------------------------------------------------ */
/* The same filter as the presets (vowel_new.c:266-289: gain, the all-pole recurrence 1/A(z) of order <= 22,
 * pre-emphasis), with the denominator supplied by the caller instead of one of the ten tables.  A tract holding a
 * preset's table (vs_tract_from_preset) computes exactly what the preset does.
 *
 * Validation, per call:
 *   n_tracts 0 or above VS_MAX_TRACTS, a stream's tract index >= n_tracts             -> VS_EINVAL
 *   a coefficient not finite, A[0] != 1, or a carry warm-up (vs_filter_warmup at the ctx's VS_OPT_CARRY_TOL) above
 *   16384 samples: unstable filters and nearly marginal ones (pole radius above ~0.998)  -> VS_ERANGE
 * The warm-up of a tract is computed once per context (a few ms) and remembered, keyed by its coefficients. */
#define VS_MAX_TRACTS 128
typedef struct vs_tract_params {
    const double  *den;       /* [n_tracts][23]: A[0..22] of 1/A(z); A[0] must be 1.0; lower orders end in zeros */
    uint32_t       n_tracts;  /* 1..VS_MAX_TRACTS                                                                 */
    const uint8_t *tract;     /* [n] index into den per stream (NULL: 0 for every stream)                        */
    const float   *gain;      /* NULL: 10.0f  (same meaning as vs_filter_params)                                 */
    const float   *pre;       /* NULL: 1.0f                                                                       */
} vs_tract_params;

/* vs_synth_batch / vs_vowel_filter_batch with caller-defined tracts: same buffers, offsets, raw output, options
 * and arithmetic contract. */
int vs_synth_batch_tract(vs_ctx *ctx, const vs_flow_params *p, const vs_tract_params *t, size_t n,
                         int16_t *pcm_out, const uint64_t *offsets, double *raw_out);
int vs_vowel_filter_batch_tract(vs_ctx *ctx, const int16_t *flow_in, const uint64_t *in_offsets, const uint64_t *nsamp,
                                const vs_tract_params *t, size_t n, int16_t *pcm_out, const uint64_t *out_offsets,
                                double *raw_out);

/* host-only helpers, no GPU needed.
 * vs_tract_from_formants: den = the product, in the order given, of  1 - 2 r_k cos(th_k) z^-1 + r_k^2 z^-2  with
 * r_k = exp(-pi B_k / fs), th_k = 2 pi F_k / fs, in double; orders above 2*n_formants are zero.  n_formants is
 * 1..11 (else VS_EINVAL); a formant is refused (VS_ERANGE) unless 0 < F_k < fs/2 and B_k > 0 (fs > 0).
 * vs_tract_from_preset: the preset's table ('a','i','u','1'..'7'), for mixing presets and custom tracts in one
 * call; an unknown key gives VS_EPRESET. */
int vs_tract_from_formants(const float *freq_hz, const float *bw_hz, int n_formants, int32_t fs, double den[23]);
int vs_tract_from_preset(int preset_key, double den[23]);

#ifdef __cplusplus
}
#endif
#endif /* VOICESYNTH_H */
