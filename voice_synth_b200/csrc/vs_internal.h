/* vs_internal.h -- structures shared by the host side (vs_api.cu, vs_batch_plan.cpp) and the kernels.
 * Not part of the ABI. */
#ifndef VS_INTERNAL_H
#define VS_INTERNAL_H
#include <stdint.h>

#define VS_NUM_PRESETS_I 10   /* == VS_NUM_PRESETS (vs_presets.h) */
#define VS_ORDER   22          /* vowel_new.c:172 */
#define VS_RING    24          /* state ring / samples per unrolled filter block (>= VS_ORDER, 3 x 16 B of PCM) */
#define VS_NT      128         /* rows per CTA of the render kernel (and its RNG stride)           */
#define VS_PLAN_NT 512         /* threads per CTA of the plan kernel.  With VS_PLAN_SMEM of shared memory a plan
                                  CTA cannot share an SM with a render CTA: the plan kernel of call k+1 runs on
                                  the VS_PLAN_SMS SMs the chunk planner keeps free, instead of being starved of
                                  issue slots by the render warps of call k (measured: 0.35 -> 0.7 ms)        */
#define VS_PLAN_NT_LEAN 1024   /* ... of its form without the open phase (no glottal noise, no period log): 64 registers */
#define VS_PLAN_SMEM (96 * 1024)
#define VS_PLAN_SMS  32         /* most SMs the chunk planner leaves to the plan kernels of the next two calls */
/* batches up to this many streams get one WARP per stream in the plan kernel (vs_batch_plan.cpp, vs_plan_warps) */
#define VS_PLAN_WARP_MAX       1024    /* while the previous call is still on the GPU */
#define VS_PLAN_WARP_MAX_IDLE  6144    /* GPU idle: the plan kernel is the call's critical path */
#define VS_PLAN_WARP_MAX_NOISE 12288   /* some streams carry glottal noise */
#define VS_RNG_DEG 31          /* glibc TYPE_3 */
#define VS_NO_CHUNK 0xffffffffu
#define VS_PULSE_TABLE_CAP (16u << 20)   /* doubles of cosine / pulse tables a context may accumulate (128 MB) */
#define VS_COS_SLACK 64         /* doubles allocated past the last cosine table */
/* samples per row and render window (vs_render.cu): multiples of the 24-sample filter ring with an ODD number of
 * ring blocks, so that the tile row stride (2*WIN bytes) is 16 x odd -- every lane's 16-byte stores down its own
 * row are bank-conflict free and every row is a legal source of a bulk (TMA) store */
#define VS_WIN_SYNTH  168
#define VS_WIN_FLOW   120
#define VS_WIN_FILTER 120

/* what a batch call computes, which generator the render kernel uses for the flow, and how it filters */
enum { VS_MODE_FLOW = 0, VS_MODE_SYNTH = 1, VS_MODE_FILTER = 2 };
enum { VS_GEN_FAST = 0, VS_GEN_SIMPLE = 1 };
enum { VS_FILT_INT = 0, VS_FILT_FMA = 1, VS_FILT_EXACT = 2 };
enum { VS_PLAN_LEAN = 0, VS_PLAN_PULSE = 1, VS_PLAN_LOG = 2 };   /* thread-form plan kernel: no pulse, pulse, pulse + log */
#define VS_WIN(MODE) ((MODE) == VS_MODE_SYNTH ? VS_WIN_SYNTH : (MODE) == VS_MODE_FLOW ? VS_WIN_FLOW : VS_WIN_FILTER)
/* tiles per 32 rows of the render kernel.  Fused / filter-only: F's, G's and the one the TMA engine reads.  Flow
 * only: one -- four CTAs share an SM and the other warps run while a warp waits for its tile to be read out */
#define VS_RENDER_TILES(MODE) ((MODE) == VS_MODE_FLOW ? 1 : 3)
#define VS_FLOWROWS_WARPS 8     /* warps per CTA of vs_flow_rows_kernel, one row each at a time */

/* per-stream descriptor, prepared on the host, read once per thread */
struct VsStream {
    uint32_t n;            /* samples in the stream, flowgen_shimmer.c:242                        */
    int32_t  P;            /* nominal period (int)((float)fs/F0), :244                            */
    int32_t  T2;           /* ceil(0.5*cq*P), :317                                                */
    uint32_t cos_off;      /* first entry of this T2's cosine table                               */
    int32_t  amp;
    float    DC;
    float    jitter, shimmer, K, Kvar, noise;
    uint32_t seed;
    float    gain, pre;
    int16_t  DCs;          /* (short)DC                                                           */
    uint8_t  flags;        /* VS_F_*                                                              */
    uint8_t  preset;       /* index into "aiu1234567"                                             */
    uint32_t chunk0;       /* id of the stream's first chunk                                      */
    uint32_t n_chunks;
    uint32_t tab_cap;      /* period-table capacity                                               */
    uint32_t pulse_off;    /* first entry of the table the render kernel evaluates the open phase from: h[0..T2) then either
                              c[0..T2) (== cos_off) or, for a stream whose closure speed never varies, K*c - K + 1           */
    uint32_t tpad;         /* entries of that table's zero-padded copy in shared memory (fast generator): above the longest
                              pitch period of any stream that uses the table                                                 */
    uint64_t out_off;      /* samples, relative to pcm_out (and raw_out)                          */
    uint64_t in_off;       /* samples, relative to flow_in (filter-only mode)                     */
    uint64_t tab_off;      /* first entry of the stream's period table                            */
    uint64_t log_off;      /* first record of the stream's user-facing period log                 */
};

/* one time-chunk of one stream = one render thread */
struct VsChunk {
    uint32_t stream;
    uint32_t emit_lo, emit_hi;   /* samples [emit_lo, emit_hi) are written by this chunk           */
    uint32_t gen_target;         /* generation starts at the period containing this sample         */
    uint32_t first_period;       /* filled by the plan kernel: the period containing gen_target    */
    uint32_t first_start;        /* filled by the plan kernel: first sample of that period         */
    uint32_t pad[2];
};

/* period table entry (32 B) written by the plan kernel, read by the render kernel */
struct VsPeriod {
    double   Ad;           /* (double)Amplitude                                                   */
    double   Kd;           /* (double)Knew                                                        */
    uint32_t start;        /* first sample of the period                                          */
    uint32_t T_np;         /* period length T (low 16 bits) | random() draws of the period before
                              its first noise draw (high 16 bits)                                 */
    uint32_t T34;          /* T3 (low 16) | T4 (high 16): closure / DC-crossing instants (noise)  */
    int32_t  ndw;          /* NoiseDistWidth                                                      */
};

/* Period table formats (VsPlanArgs / VsRenderArgs ::compact) */
#define VS_TAB_FULL 0      /* VsPeriod, 32 B: anything (-z, noise with large DC, period log)                        */
#define VS_TAB_C8   1      /* VsPeriodC, 8 B: a batch without glottal noise and without -z                           */
#define VS_TAB_N16  2      /* VsPeriodN, 16 B: glottal noise with DC <= 1 (then T4 == 0: noise on [T3, T)), no -z    */
#define VS_TAB_ENTRY_BYTES(fmt) ((fmt) == VS_TAB_C8 ? 8u : (fmt) == VS_TAB_N16 ? 16u : 32u)

struct VsPeriodC {
    float    A;            /* Amplitude                                                           */
    uint32_t T;            /* period length                                                       */
};
struct VsPeriodN {
    float    A;
    uint32_t T_np;         /* T (low 16) | random() draws of the period before its first noise draw (high 16) */
    uint32_t T3;           /* closure instant: the period's noise samples are [T3, T)             */
    int32_t  ndw;          /* NoiseDistWidth                                                      */
};

/* kernel launch argument blocks */
struct VsPlanArgs {
    const VsStream *streams;
    uint32_t        n_streams;
    VsChunk        *chunks;
    void           *table;          /* VsPeriod[], VsPeriodC[] or VsPeriodN[]                     */
    int             compact;        /* VS_TAB_*                                                   */
    uint32_t       *rng_snap;       /* [n_chunks][32] or NULL                                     */
    uint32_t       *n_periods;      /* [n_streams]                                                */
    const double   *costab;
    void           *log;            /* vs_period_rec* or NULL                                     */
    int32_t        *status;         /* device error flag                                          */
};

struct VsRenderArgs {
    const VsStream *streams;
    const VsChunk  *chunks;
    const uint32_t *order;          /* render row t works on chunk order[t]; VS_NO_CHUNK = padding   */
    uint32_t        cta_end[VS_NUM_PRESETS_I];   /* blocks of 32 rows [cta_end[p-1], cta_end[p]) belong to vowel preset p      */
    uint32_t        n_rows;         /* rows incl. padding, multiple of 32                            */
    uint32_t        grid;           /* CTAs to launch: one per render SM (flow only: a few per SM); they take the blocks
                                       of 32 rows round robin                                        */
    const void     *table;          /* VsPeriod[], VsPeriodC[] or VsPeriodN[]                        */
    int             compact;        /* VS_TAB_*                                                      */
    const uint32_t *n_periods;      /* [n_streams] periods the plan kernel wrote                     */
    const uint32_t *rng_snap;
    const double   *costab;
    const int16_t  *flow_in;        /* filter-only mode                                           */
    int16_t        *pcm_out;
    double         *raw_out;        /* nullable                                                   */
    int             general_pulse;  /* 1: some stream has -z Kvar > 0, its falling branch needs Knew of each period; 0: every
                                       pulse_off table already holds K*c - K + 1, a sample is ceil(A * table[i])              */
    int32_t        *status;         /* device error flag (shared with the plan kernel)              */
    /* shared-memory geometry chosen by the host (vs_batch_plan.cpp, vs_render_geometry) */
    uint32_t        warp_bytes;     /* per-warp region: 2 tiles | period ring | pulse-table cache    */
    uint32_t        ring_R;         /* period-ring entries per lane (power of two)                   */
    uint32_t        ring_fetch;     /* entries a lane may fetch per window                           */
    uint32_t        ring_ahead;     /* how far beyond the current period the ring is kept filled     */
    uint32_t        cache_doubles;  /* pulse-table cache per warp                                    */
    uint32_t        debug;          /* timing experiments (VS_OPT_DEBUG): bit 0 = skip the bulk stores */
    uint32_t       *ticket;         /* vs_flow_rows_kernel: the counter rows are handed out by ...   */
    uint32_t        ticket_base;    /* ... and its value when the launch starts                      */
};

/* the caller's vocal tracts (vs_synth_batch_tract, vs_vowel_filter_batch_tract): the render kernel's second,
 * __grid_constant__ parameter block, one per launch.  Rows are grouped by tract and every group is padded to whole
 * CTAs of VS_NT rows, so that a CTA's tract -- and the address of its coefficients -- is uniform. */
#define VS_MAX_TRACTS_I 128   /* == VS_MAX_TRACTS (voicesynth.h) */
struct VsTractBlock {
    uint32_t cta_end[VS_MAX_TRACTS_I];          /* CTAs [cta_end[t-1], cta_end[t]) of the launch belong to tract t */
    double   ncoef[VS_MAX_TRACTS_I][VS_ORDER];  /* ncoef[t][j-1] = -A_t[j], j = 1..22                              */
};

/* vowel -n (N1): one entry per stream */
struct VsNoiseRow {
    uint64_t off;          /* samples, relative to the pcm pointer */
    uint32_t n;
    uint32_t frame;        /* 50 * ((int)(fs*0.001/2.0)*2), vowel_new.c:361-363 */
    float    snr;
    uint32_t seed;
};

/* flow analysis (N4): one entry per stream */
struct VsAnalyzeRow {
    uint64_t off;          /* samples, relative to the flow pointer */
    uint64_t ons_off;      /* first slot of the stream's onset list */
    uint32_t n;
    uint32_t cap;          /* slots in the onset list */
    int32_t  fs;
    int16_t  lo, hi;       /* trigger thresholds */
};

/* formant analysis (vs_formant_batch): one entry per stream */
struct VsFormantRow {
    uint64_t off;          /* samples, relative to the pcm pointer                  */
    uint32_t n;            /* samples                                               */
    uint32_t Nw, H;        /* window length and frame step                          */
    uint32_t win_off;      /* first entry of the stream's window in the table       */
    double   mu;           /* pre-emphasis factor                                   */
    double   fs;
};

/* the launch arguments of the two formant kernels */
#define VS_FMT_MAX_ORDER 32
struct VsFormantArgs {
    const int16_t      *pcm;
    const VsFormantRow *rows;
    const uint64_t     *frame0;     /* [n_rows + 1]: global index of each stream's first frame (prefix sum)   */
    const double       *win;        /* window tables, one per distinct Nw                                   */
    double             *fb;         /* [frame][2 * nf]: F_0..F_nf-1, B_0..B_nf-1 of each frame, unrounded      */
    uint32_t           *ff;         /* [frame]: found | flags << 16                                         */
    uint32_t            n_rows;
    uint32_t            order, nf;
    uint32_t            max_nw;     /* longest window of the call: the shared-memory stride of a warp        */
    uint64_t            n_frames;
    double              bmax;
    double              seed_re[VS_FMT_MAX_ORDER], seed_im[VS_FMT_MAX_ORDER];   /* root-finder start points */
};

/* pitch analysis (vs_pitch_batch): one entry per stream */
struct VsPitchRow {
    uint64_t off;          /* samples, relative to the pcm pointer                                      */
    uint32_t Nw, H;        /* window length and frame step                                              */
    uint32_t tau_lo, tau_hi;
    uint32_t tab;          /* offset of the stream's table: w[0..Nw), then r_w(0) / r_w(tau) for
                              tau = tau_lo-1 .. tau_hi+1                                                */
    uint32_t reserved;
    double   fs;
};

/* what the frame kernel leaves for the stats kernel, per frame */
struct VsPitchCand {
    double   tau, r;       /* tau* and r* of the winning candidate (NaN for SILENT and NOPEAK)          */
    double   peak;         /* P_f                                                                       */
    uint32_t flags;        /* VS_PITCH_SILENT | VS_PITCH_NOPEAK                                         */
    uint32_t reserved;
};

/* the launch arguments of the two pitch kernels */
struct VsPitchArgs {
    const int16_t    *pcm;
    const VsPitchRow *rows;
    const uint64_t   *frame0;       /* [n_rows + 1]: global index of each stream's first frame (prefix sum)     */
    const double     *tab;          /* windows and lag corrections, one table per distinct (Nw, tau_lo, tau_hi) */
    VsPitchCand      *cand;         /* [n_frames]                                                               */
    uint32_t          n_rows;
    uint32_t          warps;        /* warps per CTA of the frame kernel (1..4: the shared memory must fit)     */
    uint32_t          warp_doubles; /* shared-memory stride of a warp, in doubles                               */
    uint64_t          n_frames;
    double            f_min, voicing, silence, octave_cost;
};

/* period marks (vs_vowel_report_batch): the voiced run a stream's marks lie in, as vs_vowel_report holds it */
struct VsMarkRun {
    uint32_t frame, frames;   /* first pitch frame and frame count of the run                             */
    uint32_t start, len;      /* its samples                                                              */
};

/* the launch arguments of the marks kernel: the pitch call's geometry and frame records in, onset lists out */
struct VsMarkArgs {
    const int16_t      *pcm;
    const VsPitchRow   *prows;      /* Nw, H and fs of each stream                                              */
    const uint64_t     *frame0;     /* [n_rows + 1]: each stream's first frame record (prefix sum)              */
    const void         *frames;     /* vs_pitch_frame[n_frames], as vs_pitch_batch returns them                 */
    const VsAnalyzeRow *arows;      /* row offset, onset-list slot and capacity of each stream                  */
    uint32_t           *marks;      /* the onset lists of the report kernels                                   */
    uint32_t           *counts;     /* [n_rows] marks per stream                                                */
    VsMarkRun          *run;        /* [n_rows]                                                                  */
    uint32_t            n_rows;
    uint32_t            stage;      /* int16 samples of shared memory per warp: the longest reference period plus
                                       the span of its candidates                                              */
};

#endif
