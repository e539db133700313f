/* vs_batch_plan.h -- the batch planner: what the host decides about a batch call as a pure function of its inputs, the
 * context's options and the SM count.  No CUDA here: vs_api.cu owns buffers, uploads and launches, and
 * tests/test_batch_plan_host.py runs the planner on the CPU. */
#ifndef VS_BATCH_PLAN_H
#define VS_BATCH_PLAN_H
#include <map>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>

#include "../../include/voicesynth.h"
#include "vs_internal.h"
#include "vs_presets.h"

/* internal to the library: none of this is exported from libvoicesynth_cuda.so */
#pragma GCC visibility push(hidden)

#define VS_TRACT_MAX_WARMUP 16384   /* a tract whose carry warm-up is longer is refused */

int preset_index(int key);          /* index of a vowel preset key in "aiu1234567", -1 if none */
int vs_error(std::string *err, int code, const char *fmt, ...);   /* printf into *err (if err), return code */

struct VsPlanOptions {              /* the options of a context that change a plan (VS_OPT_*) */
    double chunk = 0;               /* 0 auto, <0 never, >0 fixed */
    double tol = 1e-12;             /* x |state| <= ~2e5 at the default gain: 2e-7 before quantisation, 50 x under the 1e-5 bar */
    int exact = 0, slab = 0, simple_gen = 0;
};

/* what a context keeps from call to call: the cosine and pulse tables (one array, uploaded whole: offsets never change)
 * and the carry warm-ups at its tolerance */
struct VsTables {
    std::vector<double> cos_host;
    std::map<int, uint32_t> cos_index;
    std::vector<uint32_t> cos_fast;                    /* T2 -> table offset, direct index in front of the map */
    std::map<uint64_t, uint32_t> pulse_index;          /* (T2, bits of K) -> offset of the h / K*c-K+1 table */
    uint64_t pulse_last_key = ~0ull;
    uint32_t pulse_last_off = 0;
    double tol = 0;
    int warm[VS_NUM_PRESETS];                          /* warm-up samples per preset at tol (gain-independent part) */
    std::unordered_map<std::string, int> tract_warm;   /* warm-up at tol of every tract seen, keyed by its coefficients' bytes */
    void set_tol(double t);                            /* the presets' warm-ups at t; forgets the tracts' */
    uint32_t cos_table(int T2);
    uint32_t pulse_table(int T2, float K);
    int tract_warmup(const double *A);
};

struct VsBatch {                    /* the arguments of a batch call */
    int mode;                       /* VS_MODE_* */
    size_t n;
    const vs_flow_params *fp;
    const vs_filter_params *ff;
    const vs_tract_params *ft;      /* _tract calls: caller-defined tracts instead of ff */
    const int16_t *flow_in;
    const uint64_t *in_offsets, *nsamp;
    int16_t *pcm_out;
    const uint64_t *offsets;
    double *raw_out;
    vs_period_log *log;
};

/* stage 1: validated stream descriptors and what the kernel choice needs to know about the whole batch */
struct VsFacts {
    uint64_t max_n = 0;
    bool any_noise = false, any_kvar = false;
    bool int_filter = true;         /* every stream: integral gain, pre-emphasis 0 or 1 -> both commute to the integer input */
    bool amp_fits = true;           /* no amplitude can pass 32767 (fast generator) */
    bool noise_simple = true;       /* every noisy stream has DC <= 1 (then T4 == 0) and T2 >= 16: 16-byte period entries do */
    int t_min = 0x7fffffff, t_max = 0, t2_min = 0x7fffffff;   /* bounds on the pitch periods; shortest half open phase */
};
struct VsDescriptors {
    std::vector<VsStream> hs;
    VsFacts facts;
    std::vector<int> warm;          /* warm-up per filter group: per preset, or per tract of a _tract call */
    std::vector<double> ncoef;      /* [n_tracts][VS_ORDER] = -A[1..22] of the tracts (tract calls) */
};
/* VS_OK, or an error code and its message in err; the tables may have grown either way */
int vs_build_descriptors(const VsBatch &b, bool want_log, VsTables &tab, VsDescriptors &d, std::string &err);

struct VsShape {                    /* the kernel forms of a batch */
    int mode;
    bool tracts, flow_rows;         /* flow_rows: flow on vs_flow_rows_kernel, a warp per row */
    int compact;                    /* period table format, VS_TAB_* */
    uint64_t ph_mask;               /* a row's phase is its output address (in samples) & ph_mask */
    int plan_nt;                    /* streams per CTA of the thread-form plan kernel */
    int n_groups;                   /* filter groups: presets or tracts ... */
    size_t group_rows;              /* ... each padded to this many rows */
};
VsShape vs_shape(int mode, bool tracts, bool want_log, const VsFacts &fc, const VsPlanOptions &o);

/* stage 3: streams [cut[g], cut[g+1]) go to device slot g; a slot's streams go in slabs, launched and copied together */
typedef std::pair<size_t, size_t> VsRange;
std::vector<size_t> vs_split_slots(const std::vector<VsStream> &hs, size_t nslots);
std::vector<VsRange> vs_slabs(const std::vector<VsStream> &hs, size_t s0, size_t s1, bool out_dev, int opt_slab, size_t *slab_streams);

/* stage 4: the chunks and render rows of one slot */
struct VsPlan {
    std::vector<VsChunk> chunks;
    std::vector<uint32_t> nch;                   /* chunks per stream */
    std::vector<size_t> slab_c0, slab_r0;        /* first chunk / row of each slab, then the totals */
    uint64_t tab_total = 0, warm_total = 0;      /* period-table entries; warm-up samples of all chunks */
    std::vector<uint32_t> order;                 /* render rows: chunk ids, VS_NO_CHUNK = padding */
    struct Geom {                                /* per slab: what the render launch needs besides the rows */
        uint32_t cta_end[VS_MAX_TRACTS_I];       /* group ends: presets in blocks of 32 rows, tracts in CTAs */
        uint32_t cache_doubles;                  /* pulse-table cache a warp needs (fast generator) */
    };
    std::vector<Geom> geom;
};
/* 4a, chunks; out_base: the sample address of out_off 0 for device output, 0 for host output */
void vs_plan_chunks(const VsPlanOptions &o, const VsShape &sh, int sm_count, const std::vector<VsStream> &hs, size_t s0,
                    size_t s1, const std::vector<VsRange> &slabs, const int *warm, uint64_t out_base, VsPlan &p);
void vs_plan_rows(const VsShape &sh, const std::vector<VsStream> &hs, size_t s0, VsPlan &p);   /* 4b, row order */
void vs_plan_assign(const VsPlan &p, std::vector<VsStream> &hs, size_t s0, size_t s1);         /* chunk0, n_chunks, tab_off */

/* the generator (VS_GEN_*), shared-memory geometry and grid of a slab's render launch, into ra (n_rows set); ns: the
 * slot's streams */
int vs_render_geometry(const VsPlanOptions &o, const VsShape &sh, const VsFacts &fc, int sm_count, size_t ns,
                       uint32_t cache_doubles, VsRenderArgs &ra);

#pragma GCC visibility pop
#endif
