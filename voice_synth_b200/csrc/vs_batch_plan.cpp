/* vs_batch_plan.cpp -- the batch planner (vs_batch_plan.h).
 *
 * What stays on the host, and why it is still bit-exact with the reference:
 *   - nSamples / P / T2 per stream: three scalar expressions (flowgen_shimmer.c:242,244,317) evaluated
 *     here with the same C types; x86-64 has no FMA contraction by default and the file is built
 *     with -ffp-contract=off.
 *   - cos(PI*i/T2) tables, one per distinct T2 of the batch, computed with the system libm exactly
 *     as the reference evaluates them (PI = 4.0*atan(1.0), flowgen_shimmer.c:39,319,328).  The
 *     kernels only ever multiply/add/ceil these doubles, so the int16 pulse cannot differ by an ulp
 *     of a device cosine.
 */
#include "vs_batch_plan.h"

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>

/* parameter access with the reference defaults (flowgen_shimmer.c:87, vowel_new.c:76-77) */
struct FlowRow {
    float dur, jitter, shimmer, cq, K, Kvar, F0, DC, noise;
    int32_t amp, fs;
    uint8_t flags;
    uint32_t seed;
};

static FlowRow flow_row(const vs_flow_params *p, size_t i)
{
    FlowRow r;
    r.dur = p && p->dur ? p->dur[i] : 1.0f;
    r.jitter = p && p->jitter ? p->jitter[i] : 0.0f;
    r.shimmer = p && p->shimmer ? p->shimmer[i] : 0.0f;
    r.cq = p && p->cq ? p->cq[i] : 0.55f;
    r.K = p && p->K ? p->K[i] : 0.65f;
    r.Kvar = p && p->Kvar ? p->Kvar[i] : 0.0f;
    r.F0 = p && p->F0 ? p->F0[i] : 120.0f;
    r.DC = p && p->DC ? p->DC[i] : 0.0f;
    r.noise = p && p->noise ? p->noise[i] : 0.0f;
    r.amp = p && p->amp ? p->amp[i] : 12000;
    r.fs = p && p->fs ? p->fs[i] : 22050;
    r.flags = p && p->flags ? p->flags[i] : 0;
    r.seed = p && p->seed ? p->seed[i] : 1u;
    return r;
}

static uint64_t row_nsamples(const FlowRow &r)
{
    /* `(unsigned long) par.fs*par.dur`: unsigned long * float is a float product (:242) */
    volatile float prod = (float)(uint64_t)(int64_t)r.fs * r.dur;
    if (!(prod >= 0.0f) || prod >= 1.8e19f) return 0;
    return (uint64_t)prod;
}

static int row_P(const FlowRow &r)
{
    volatile float q = (float)(int64_t)r.fs / r.F0;                   /* :244 */
    if (!(q > -2147483648.0f && q < 2147483648.0f)) return 0;
    return (int)q;
}

static int row_T2(const FlowRow &r, int P)
{
    volatile double h = 0.5 * (double)r.cq;                           /* :317 */
    volatile double v = h * P;
    return (int)std::ceil(v);
}

static int row_validate(const FlowRow &r, int *P_out = nullptr, uint64_t *n_out = nullptr)
{
    if (!(r.fs > 0) || !std::isfinite(r.dur) || !(r.dur > 0.0f)) return VS_ERANGE;
    if (!std::isfinite(r.F0) || !(r.F0 > 0.0f)) return VS_ERANGE;
    const int P = row_P(r);
    if (P < 1 || P > 27000) return VS_ERANGE;                        /* T <= 1.2*P is stored in a short (:289) */
    const uint64_t n = row_nsamples(r);
    if (n < 1 || n > 0x7fffffffull) return VS_ERANGE;
    if (P_out) *P_out = P;
    if (n_out) *n_out = n;
    if (!(r.jitter >= 0.0f && r.jitter <= 10.0f)) return VS_ERANGE;   /* :478 */
    if (!(r.shimmer >= 0.0f && r.shimmer <= 1.0f)) return VS_ERANGE;  /* :544 */
    if (!(r.cq >= 0.0f && r.cq <= 1.0f)) return VS_ERANGE;            /* :490 */
    if (!std::isfinite(r.K) || !(r.K >= 0.0f)) return VS_ERANGE;
    if (!(r.Kvar >= 0.0f && r.Kvar <= 1.0f)) return VS_ERANGE;        /* :530 */
    if (!(r.amp >= 0 && r.amp < 32767)) return VS_ERANGE;             /* :518 */
    if (!std::isfinite(r.DC) || !(r.DC >= 0.0f) || r.DC > 32767.0f) return VS_ERANGE;
    /* the tool accepts 0..50 dB, i.e. noise = 10^(dB/10) >= 1 (:505-511).  Below 0.1 (-10 dB) NoiseDistWidth could pass
     * 2^19, the range the render kernel's two-operation noise sample is proven for (tests/tools/noisecheck.c) */
    if ((r.flags & VS_F_NOISE) && (!std::isfinite(r.noise) || !(r.noise >= 0.1f))) return VS_ERANGE;
    if (r.flags & ~(VS_F_JITTER | VS_F_SHIMMER | VS_F_NOISE)) return VS_EINVAL;
    /* Falling branch (:327-332): x = (short)ceil(A*(K*c - K + 1)), left at the first x < DC.  Between two samples
     * the argument drops by at most A*K*2*sin(pi/(2*T2)); while that step stays below 2^15 the first value under DC
     * still fits the short and the reference stops there.  Beyond it the cast wraps before the DC test and what
     * the reference emits is an accident of 16-bit wrap-around: refused (SURVEY.md 8a, hazards).  (A above 32767
     * needs no bound: x[T2] = (short)ceil(A) is negative and the branch is left at once.) */
    const int T2 = row_T2(r, P);
    if (T2 >= 2) {
        const double amax = std::min(32767.0, ((r.flags & VS_F_SHIMMER) && r.shimmer != 0.0f ? 1.8 : 1.0) * (double)r.amp);
        const double kmax = (double)r.K * (1.0 + (double)r.Kvar);
        if (amax * kmax * 2.0 * std::sin(3.141592653589793 / (2.0 * (double)T2)) > 32768.0) return VS_ERANGE;
    }
    return VS_OK;
}

static uint32_t row_max_periods(const FlowRow &r, uint64_t n, int P)
{
    const bool jit = (r.flags & VS_F_JITTER) && r.jitter != 0.0f;
    int tmin = P;
    if (jit) {
        tmin = (int)std::floor(0.8f * (float)P);                      /* accepted T satisfy (float)T >= (float)0.8*P */
        if (tmin < 1) tmin = 1;
    }
    return (uint32_t)(n / (uint64_t)tmin + 2);
}

int preset_index(int key)
{
    const char *q = key ? strchr(vs_preset_keys, key) : nullptr;
    return q ? (int)(q - vs_preset_keys) : -1;
}

/* Samples after which the free response of an arbitrary unit-bounded initial state has decayed below
 * tol: W = 1 + last n with sum_j |(Phi^n)[0][j]| >= tol, Phi the companion matrix of the preset. */
static int warmup_for(const double *A, double tol, int limit = 60000)
{
    const int N = VS_ORDER;
    /* column j holds the free response state started from unit vector e_j */
    std::vector<double> st(N * N, 0.0);
    for (int j = 0; j < N; j++) st[j * N + j] = 1.0;       /* st[j*N + k] = y[n-1-k] of response j */
    int last = 0;
    const int horizon = 60000;
    int quiet = 0;
    for (int n = 0; n < horizon; n++) {
        double g = 0.0;
        for (int j = 0; j < N; j++) {
            double *s = &st[j * N];
            double y0 = 0.0;
            for (int k = 0; k < N; k++) y0 -= A[k + 1] * s[k];
            for (int k = N - 1; k > 0; k--) s[k] = s[k - 1];
            s[0] = y0;
            g += std::fabs(y0);
        }
        if (!(g < tol)) { last = n + 1; quiet = 0; if (last >= limit) break; }    /* (a response that overflowed: not decayed) */
        else if (++quiet > 4096) break;
    }
    return last + 1;
}

void VsTables::set_tol(double t)
{
    tol = t;
    for (int k = 0; k < VS_NUM_PRESETS; k++) warm[k] = warmup_for(vs_preset_den[k], tol);
    tract_warm.clear();
}

/* a tract's warm-up at the tolerance, computed once per context */
int VsTables::tract_warmup(const double *A)
{
    const std::string key(reinterpret_cast<const char *>(A), (VS_ORDER + 1) * sizeof(double));
    auto it = tract_warm.find(key);
    if (it != tract_warm.end()) return it->second;
    const int w = warmup_for(A, tol, VS_TRACT_MAX_WARMUP + 1);
    if (tract_warm.size() >= (1u << 16)) tract_warm.clear();   /* a bound on what a stream of one-off tracts leaves behind */
    tract_warm.emplace(key, w);
    return w;
}

uint32_t VsTables::cos_table(int T2)
{
    if (T2 >= 0 && (size_t)T2 < cos_fast.size() && cos_fast[T2] != 0xffffffffu) return cos_fast[T2];
    auto it = cos_index.find(T2);
    if (it != cos_index.end()) return it->second;
    const uint32_t off = (uint32_t)cos_host.size();
    volatile double one = 1.0;
    const double pi = 4.0 * std::atan(one);                           /* #define PI 4.0*atan(1.0) (:39) */
    /* layout per T2: h[0..T2) then c[0..T2), so that the open-phase index i in [0,2*T2) addresses it
     * directly.  h[i] = 0.5*(1-c[i]): (A*0.5)*(1.0-c) == A*h bit for bit, scaling by 0.5 being exact (:319) */
    std::vector<double> c((size_t)T2);
    for (int i = 0; i < T2; i++) {
        volatile double num = pi * i;                                 /* PI*i/T2 == ((4.0*atan(1.0))*i)/T2 */
        volatile double arg = num / T2;
        c[i] = std::cos(arg);
    }
    for (int i = 0; i < T2; i++) {
        volatile double om = 1.0 - c[i];
        volatile double h = 0.5 * om;
        const double hv = h;
        cos_host.push_back(hv);
    }
    for (int i = 0; i < T2; i++) cos_host.push_back(c[i]);
    cos_index[T2] = off;
    if (T2 >= 0 && T2 < 65536) {
        if ((size_t)T2 >= cos_fast.size()) cos_fast.resize((size_t)T2 + 64, 0xffffffffu);
        cos_fast[T2] = off;
    }
    return off;
}

/* Open-phase table of a stream whose closure speed never varies (-z absent: Knew == K in every period):
 * h[0..T2) as above, then f[i] = (K*c[i] - K) + 1.0 with the reference's three roundings (:328), so that a
 * falling-branch sample is ceil(A * f[i]) like a rising one is ceil(A * h[i]).  Saves the render kernel three of
 * its five FP64 operations per open-phase sample. */
uint32_t VsTables::pulse_table(int T2, float K)
{
    uint32_t kb;
    memcpy(&kb, &K, 4);
    const uint64_t key = ((uint64_t)(uint32_t)T2 << 32) | kb;
    if (key == pulse_last_key) return pulse_last_off;
    auto it = pulse_index.find(key);
    uint32_t off;
    if (it != pulse_index.end()) off = it->second;
    else {
        const uint32_t src = cos_table(T2);                           /* h then c; may grow cos_host */
        if (cos_host.size() & 1) cos_host.push_back(0.0);             /* 16-byte aligned */
        off = (uint32_t)cos_host.size();
        for (int i = 0; i < T2; i++) { const double h = cos_host[src + i]; cos_host.push_back(h); }
        const double Kd = (double)K;
        for (int i = 0; i < T2; i++) {
            volatile double kc = Kd * cos_host[src + T2 + i];
            volatile double d = kc - Kd;
            volatile double f = d + 1.0;
            const double fv = f;
            cos_host.push_back(fv);
        }
        /* for vs_flow_rows_kernel, which reads two neighbouring entries with one 16-byte load: two zeros (the closed
         * phase), then the same table again moved up by one entry, so that a pair is 16-byte aligned in one of the two
         * copies whatever its parity */
        const size_t n2 = 2 * (size_t)T2;
        cos_host.push_back(0.0);
        cos_host.push_back(0.0);
        for (size_t k = 0; k < n2 + 2; k++) { const double v = k + 1 < n2 + 2 ? cos_host[off + k + 1] : 0.0; cos_host.push_back(v); }
        pulse_index[key] = off;
    }
    pulse_last_key = key;
    pulse_last_off = off;
    return off;
}

int vs_error(std::string *err, int code, const char *fmt, ...)
{
    if (err) {
        char buf[512];
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(buf, sizeof buf, fmt, ap);
        va_end(ap);
        *err = buf;
    }
    return code;
}

int vs_build_descriptors(const VsBatch &b, bool want_log, VsTables &tab, VsDescriptors &d, std::string &err)
{
    const size_t n = b.n;
    std::vector<VsStream> &hs = d.hs;
    hs.assign(n, VsStream());
    VsFacts fc;
    fc.raw = b.raw_out != nullptr;
    /* filter groups: the ten presets, or the caller's tracts (validated, warm-ups from the context's cache) */
    d.warm.assign(tab.warm, tab.warm + VS_NUM_PRESETS);
    d.ncoef.clear();
    if (b.ft) {
        const uint32_t nt = b.ft->n_tracts;
        if (!b.ft->den || nt == 0 || nt > VS_MAX_TRACTS) return vs_error(&err, VS_EINVAL, "n_tracts %u outside 1..%d (or den is NULL)", nt, VS_MAX_TRACTS);
        d.warm.assign(nt, 0);
        d.ncoef.assign((size_t)nt * VS_ORDER, 0.0);
        for (uint32_t t = 0; t < nt; t++) {
            const double *A = b.ft->den + (size_t)t * (VS_ORDER + 1);
            for (int j = 0; j <= VS_ORDER; j++)
                if (!std::isfinite(A[j])) return vs_error(&err, VS_ERANGE, "tract %u: coefficient %d is not finite", t, j);
            if (A[0] != 1.0) return vs_error(&err, VS_ERANGE, "tract %u: A[0] = %g, must be 1", t, A[0]);
            const int w = tab.tract_warmup(A);
            if (w > VS_TRACT_MAX_WARMUP) return vs_error(&err, VS_ERANGE, "tract %u: unstable or nearly marginal (carry warm-up above %d samples)", t, VS_TRACT_MAX_WARMUP);
            d.warm[t] = w;
            for (int j = 1; j <= VS_ORDER; j++) d.ncoef[(size_t)t * VS_ORDER + j - 1] = -A[j];
        }
    }
    for (size_t i = 0; i < n; i++) {
        VsStream &s = hs[i];
        memset(&s, 0, sizeof s);
        if (b.mode == VS_MODE_FILTER) {
            if (b.nsamp[i] > 0x7fffffffull) return vs_error(&err, VS_EOVERLAP, "stream %zu: too many samples", i);
            s.n = (uint32_t)b.nsamp[i];
        } else {
            const FlowRow r = flow_row(b.fp, i);
            int P = 0;
            uint64_t nn = 0;
            const int rc = row_validate(r, &P, &nn);
            if (rc) return vs_error(&err, rc, "stream %zu: flow parameter out of range", i);
            s.n = (uint32_t)nn;
            s.P = P;
            s.T2 = row_T2(r, s.P);
            s.cos_off = tab.cos_table(s.T2);
            fc.t2_min = std::min(fc.t2_min, (int)s.T2);
            fc.any_kvar |= r.Kvar != 0.0f;
            s.amp = r.amp; s.DC = r.DC; s.jitter = r.jitter; s.shimmer = r.shimmer; s.K = r.K; s.Kvar = r.Kvar;
            s.noise = r.noise; s.seed = r.seed; s.flags = r.flags;
            s.DCs = (int16_t)(int32_t)r.DC;                            /* x[i] = par.DC (:321,:335) */
            s.tab_cap = row_max_periods(r, s.n, s.P);
            fc.any_noise |= (r.flags & VS_F_NOISE) != 0;
            if ((r.flags & VS_F_NOISE) && !(r.DC <= 1.0f && s.T2 >= 16)) fc.noise_simple = false;
            /* accepted periods satisfy 0.8*P <= T <= 1.2*P (flowgen_shimmer.c:290) */
            const bool jit = (r.flags & VS_F_JITTER) && r.jitter != 0.0f;
            fc.t_min = std::min(fc.t_min, jit ? std::max(1, (int)std::floor(0.8f * (float)P)) : P);
            const int tm = jit ? (int)std::ceil(1.2f * (float)P) + 1 : P;
            fc.t_max = std::max(fc.t_max, tm);
            s.tpad = (uint32_t)((tm + 9) & ~1);                         /* refined per table below */
            if ((r.flags & VS_F_SHIMMER) && r.shimmer != 0.0f ? 1.8f * (float)r.amp > 32767.0f : r.amp > 32767) fc.amp_fits = false;
        }
        if (b.mode != VS_MODE_FLOW && b.ft) {
            const uint32_t t = b.ft->tract ? b.ft->tract[i] : 0u;
            if (t >= b.ft->n_tracts) return vs_error(&err, VS_EINVAL, "stream %zu: tract index %u >= n_tracts %u", i, t, b.ft->n_tracts);
            s.preset = (uint8_t)t;                                      /* the filter group: here a tract */
            s.gain = b.ft->gain ? b.ft->gain[i] : 10.0f;
            s.pre = b.ft->pre ? b.ft->pre[i] : 1.0f;
        } else if (b.mode != VS_MODE_FLOW) {
            const int key = b.ff && b.ff->preset ? b.ff->preset[i] : 'a';
            const int pi = preset_index(key);
            if (pi < 0) return vs_error(&err, VS_EPRESET, "stream %zu: unknown vowel preset 0x%02x", i, key);
            s.preset = (uint8_t)pi;
            s.gain = b.ff && b.ff->gain ? b.ff->gain[i] : 10.0f;
            s.pre = b.ff && b.ff->pre ? b.ff->pre[i] : 1.0f;
        }
        if (b.mode != VS_MODE_FLOW) {
            if (!std::isfinite(s.gain) || !std::isfinite(s.pre)) return vs_error(&err, VS_ERANGE, "stream %zu: gain/pre not finite", i);
            if (!(s.gain == std::floor(s.gain) && std::fabs(s.gain) <= 32767.0f && (s.pre == 0.0f || s.pre == 1.0f))) fc.int_filter = false;
        }
        fc.max_n = std::max<uint64_t>(fc.max_n, s.n);
    }
    for (size_t i = 0; i < n; i++) {
        hs[i].out_off = b.offsets ? b.offsets[i] : (uint64_t)i * fc.max_n;
        if (b.mode == VS_MODE_FILTER) hs[i].in_off = b.in_offsets ? b.in_offsets[i] : (uint64_t)i * fc.max_n;
        if (want_log) hs[i].log_off = b.log->rec_offsets[i];
    }
    /* the table the render kernel reads: with no -z anywhere in the batch, the falling branch pre-multiplied by K
     * (one table per distinct (T2, K); a batch with a different K on every stream keeps the general path instead
     * of growing the tables without bound) */
    if (b.mode != VS_MODE_FILTER) {
        for (size_t i = 0; i < n && !fc.any_kvar; i++) {
            const size_t before = tab.cos_host.size();
            hs[i].pulse_off = tab.pulse_table(hs[i].T2, hs[i].K);
            if (tab.cos_host.size() > before && tab.cos_host.size() > VS_PULSE_TABLE_CAP) fc.any_kvar = true;
        }
        if (fc.any_kvar)
            for (size_t i = 0; i < n; i++) hs[i].pulse_off = hs[i].cos_off;
        /* streams that share a table share its padded length */
        std::map<uint32_t, uint32_t> pad;
        for (size_t i = 0; i < n; i++) { uint32_t &v = pad[hs[i].pulse_off]; v = std::max(v, hs[i].tpad); }
        for (size_t i = 0; i < n; i++) hs[i].tpad = pad[hs[i].pulse_off];
    }

    /* output rows, half-open sample ranges, must not intersect */
    std::vector<std::pair<uint64_t, uint64_t>> rows(n);
    for (size_t i = 0; i < n; i++) rows[i] = {hs[i].out_off, hs[i].out_off + hs[i].n};
    std::sort(rows.begin(), rows.end());
    for (size_t i = 1; i < n; i++)
        if (rows[i].first < rows[i - 1].second) return vs_error(&err, VS_EOVERLAP, "output rows overlap");
    d.facts = fc;
    return VS_OK;
}

/* what both branch-free generators (VS_GEN_FAST, vs_flow_rows_kernel) need: amplitudes within a short, periods >= 24 */
static bool branch_free(const VsFacts &fc, const VsPlanOptions &o) { return fc.amp_fits && !o.simple_gen && fc.t_min >= 24; }

VsShape vs_shape(int mode, bool tracts, bool want_log, const VsFacts &fc, const VsPlanOptions &o)
{
    VsShape sh;
    sh.mode = mode;
    sh.tracts = tracts;
    /* period table format: 8-byte entries (amplitude, length) where they suffice, 16-byte ones for plain glottal noise */
    sh.compact = (fc.any_kvar || want_log) ? VS_TAB_FULL : !fc.any_noise ? VS_TAB_C8 : fc.noise_simple ? VS_TAB_N16 : VS_TAB_FULL;
    /* flow without glottal noise: lanes along the row (vs_flow_rows_kernel).  T2 >= 2: row_validate() bounds A*K then */
    sh.flow_rows = mode == VS_MODE_FLOW && sh.compact == VS_TAB_C8 && branch_free(fc, o) && fc.t2_min >= 2;
    sh.ph_mask = sh.flow_rows ? 63u : 7u;
    /* the plan kernel evaluates the open phase only for glottal noise and the period log; without either its lean form */
    sh.plan = want_log ? VS_PLAN_LOG : fc.any_noise ? VS_PLAN_PULSE : VS_PLAN_LEAN;
    sh.plan_nt = sh.plan == VS_PLAN_LEAN ? VS_PLAN_NT_LEAN : VS_PLAN_NT;
    /* no integer-filter kernel writes raw output.  (Flow-only calls run no filter; render_path reports this value anyway) */
    sh.filt = o.exact ? VS_FILT_EXACT : fc.int_filter && !fc.raw ? VS_FILT_INT : VS_FILT_FMA;
    sh.raw = fc.raw;
    sh.noise = fc.any_noise;
    sh.general_pulse = fc.any_kvar;
    sh.n_groups = tracts ? VS_MAX_TRACTS_I : VS_NUM_PRESETS;
    sh.group_rows = tracts ? VS_NT : 32;   /* groups are padded to whole CTAs (tracts) or blocks of 32 rows (presets) */
    return sh;
}

std::vector<size_t> vs_split_slots(const std::vector<VsStream> &hs, size_t nslots)
{
    const size_t n = hs.size();
    std::vector<size_t> cut(nslots + 1, n);
    uint64_t total = 0;
    for (size_t i = 0; i < n; i++) total += hs[i].n;
    cut[0] = 0;
    uint64_t acc = 0;
    size_t g = 1;
    for (size_t i = 0; i < n && g < nslots; i++) {
        acc += hs[i].n;
        while (g < nslots && acc * nslots >= total * g) cut[g++] = i + 1;
    }
    return cut;
}

std::vector<VsRange> vs_slabs(const std::vector<VsStream> &hs, size_t s0, size_t s1, bool out_dev, int opt_slab,
                              size_t *slab_streams)
{
    const size_t ns = s1 - s0;
    size_t per = ns;
    if (!out_dev) {
        if (opt_slab > 0) per = (size_t)opt_slab;
        else {
            /* one slab per call unless the device mirror of the output would be huge; PCIe/compute
             * overlap comes from alternating two scratch buffers ACROSS calls (VS_OPT_ASYNC_HOST) */
            uint64_t total = 0;
            for (size_t i = s0; i < s1; i++) total += hs[i].n;
            const uint64_t bytes = total * 2;
            size_t want = (size_t)std::max<uint64_t>(1, (bytes + (1ull << 30) - 1) >> 30);
            per = (ns + want - 1) / want;
        }
        if (per < 1) per = 1;
    }
    std::vector<VsRange> slabs;
    for (size_t a0 = s0; a0 < s1; a0 += per) slabs.push_back({a0, std::min(s1, a0 + per)});
    *slab_streams = per;
    return slabs;
}

/* SMs the render kernel leaves to the plan kernels of the next calls.  A plan CTA keeps an SM for one plan time; the
 * plan of a step takes a little longer than its render (measured: 1.2x on the bench workload and on the noise
 * grid), so 1.5 SMs per plan CTA -- two plans partly side by side -- keep the plans ahead of the renders.  Large
 * batches get none: their plan needs every SM anyway and simply alternates with the render. */
static int vs_plan_reserve(int plan_ctas)
{
    return 2 * plan_ctas <= VS_PLAN_SMS ? (3 * plan_ctas + 1) / 2 : 0;
}

/* a fixed chunk length (VS_OPT_CHUNK_SAMPLES > 0) for the lane-per-row kernels: on the 8-sample grid, at least 64 */
static uint32_t fixed_chunk(const VsPlanOptions &o)
{
    const uint32_t L = ((uint32_t)o.chunk + 7u) & ~7u;
    return L < 64 ? 64 : L;
}

/* The time-chunk length of a flow-only slab (SURVEY.md 7 "Occupancy"); 0: no chunking.  The flow has no carry, so
 * chunks cost nothing but their rows: fill the GPU once. */
static uint32_t choose_chunk(const VsPlanOptions &o, int sm_count, size_t n_streams, uint64_t total, bool flow_rows)
{
    if (o.chunk < 0) return 0;
    if (flow_rows) {
        /* lanes along the row (vs_flow_rows_kernel): a warp takes a row at a time, 256 samples per step, rows handed out
         * by a ticket -- about four rows per warp balance the SMs and keep the cost of opening a row (its descriptors,
         * the first batch of periods: five dependent memory round trips) small.  Measured on the bench batch: 2.6 / 3.5 /
         * 5.2 / 7.8 rows per warp = 0.078 / 0.076 / 0.078 / 0.080 ms */
        double L = o.chunk > 0 ? o.chunk : std::ceil((double)total / ((double)sm_count * 4.0 * VS_FLOWROWS_WARPS * 4.0));
        if (L < 512.0) L = 512.0;
        if (L > 1048576.0) L = 1048576.0;
        return ((uint32_t)L + 255u) & ~255u;
    }
    if (o.chunk > 0) return fixed_chunk(o);
    /* lane per row: one full wave of rows (4 CTAs of VS_NT rows per SM), or whole waves of >= 512-sample chunks when
     * the batch is small */
    const double lanes = (double)sm_count * 4.0 * VS_NT * 0.97;
    if ((double)n_streams >= lanes) return 0;
    double L = std::ceil((double)total / lanes);
    if (L < 512.0) L = 512.0;
    return ((uint32_t)L + 7u) & ~7u;
}

/* Per-stream chunk counts for the filtering modes.  A chunk of stream s costs  W_s + L_s  sample
 * steps (W_s = carry warm-up of its preset); the kernel time is that of the most expensive chunk
 * times the number of waves, one wave = one CTA of VS_NT rows per SM.  So: give every stream the
 * chunk length  L_s = budget - W_s  and pick the smallest budget whose rows fit in `waves` waves;
 * take the wave count with the smallest  waves * budget. */
static void plan_filter_chunks(const VsPlanOptions &o, int sm_count, const std::vector<VsStream> &hs, size_t a0, size_t a1,
                               std::vector<uint32_t> &nchunks, int plan_nt, const int *warm, bool tracts)
{
    const size_t ns = a1 - a0;
    nchunks.assign(ns, 1u);
    if (o.chunk < 0 || o.exact) return;
    if (o.chunk > 0) {
        const uint32_t L = fixed_chunk(o);
        for (size_t i = 0; i < ns; i++) nchunks[i] = hs[a0 + i].n <= L ? 1u : (uint32_t)((hs[a0 + i].n + L - 1) / L);
        return;
    }
    /* rows per wave; a few SMs stay free for the plan kernels of the next two calls (one CTA of VS_PLAN_NT streams per
     * SM each, see VS_PLAN_SMEM) */
    const int plan_ctas = (int)((ns + (size_t)plan_nt - 1) / (size_t)plan_nt);
    const int reserve = vs_plan_reserve(plan_ctas);
    const int render_sms = sm_count > 4 * VS_PLAN_SMS ? sm_count - reserve : sm_count;
    const double cap = (double)render_sms * VS_NT;
    /* streams of equal (length, preset) get equal chunk counts: plan over the distinct classes */
    std::map<std::pair<uint32_t, uint8_t>, uint32_t> classes;
    uint32_t nmax = 0;
    for (size_t i = 0; i < ns; i++) {
        classes[{hs[a0 + i].n, hs[a0 + i].preset}]++;
        nmax = std::max(nmax, hs[a0 + i].n);
    }
    /* the first chunk of a stream needs no warm-up, so it emits `budget` samples, the others budget - W */
    auto chunks_of = [&](uint32_t n, uint8_t preset, double budget) -> uint32_t {
        if ((double)n <= budget) return 1u;
        const double L = std::max(512.0, budget - (double)warm[preset]);
        return 1u + (uint32_t)std::ceil(((double)n - budget) / L);
    };
    /* presets: groups padded to blocks of 32 rows, a 3 % allowance covers that; tracts: groups padded to whole CTAs,
     * counted exactly */
    const double fill = tracts ? 1.0 : 0.97;
    auto rows_for = [&](double budget) -> double {
        if (!tracts) {
            double rows = 0;
            for (const auto &kv : classes) rows += (double)kv.second * chunks_of(kv.first.first, kv.first.second, budget);
            return rows;
        }
        double per[VS_MAX_TRACTS_I] = {0.0};
        for (const auto &kv : classes) per[kv.first.second] += (double)kv.second * chunks_of(kv.first.first, kv.first.second, budget);
        double rows = 0;
        for (int t = 0; t < VS_MAX_TRACTS_I; t++) rows += std::ceil(per[t] / VS_NT) * VS_NT;
        return rows;
    };
    double best_cost = 1e300, best_budget = (double)nmax;
    for (int waves = 1; waves <= 8; waves++) {
        if (rows_for((double)nmax) > waves * cap) continue;                    /* even unchunked does not fit */
        double lo = 512.0, hi = (double)nmax;                                  /* smallest budget that fits */
        for (int it = 0; it < 30; it++) {
            const double mid = 0.5 * (lo + hi);
            if (rows_for(mid) <= waves * cap * fill) hi = mid; else lo = mid;
        }
        const double cost = waves * hi;
        if (cost < best_cost * 0.98) { best_cost = cost; best_budget = hi; }
    }
    for (size_t i = 0; i < ns; i++) nchunks[i] = chunks_of(hs[a0 + i].n, hs[a0 + i].preset, best_budget);
}

void vs_plan_chunks(const VsPlanOptions &o, const VsShape &sh, int sm_count, const std::vector<VsStream> &hs, size_t s0,
                    size_t s1, const std::vector<VsRange> &slabs, const int *warm, uint64_t out_base, VsPlan &p)
{
    const bool flow = sh.mode == VS_MODE_FLOW;
    std::vector<VsChunk> &hc = p.chunks;
    hc.clear();
    p.nch.assign(s1 - s0, 1u);
    p.slab_c0.assign(slabs.size() + 1, 0);
    p.tab_total = p.warm_total = 0;
    for (size_t k = 0; k < slabs.size(); k++) {
        const size_t a0 = slabs[k].first, a1 = slabs[k].second;
        uint32_t Lflow = 0;
        std::vector<uint32_t> nch;
        if (flow) {
            uint64_t tot = 0;
            for (size_t i = a0; i < a1; i++) tot += hs[i].n;
            Lflow = choose_chunk(o, sm_count, a1 - a0, tot, sh.flow_rows);
        } else
            plan_filter_chunks(o, sm_count, hs, a0, a1, nch, sh.plan_nt, warm, sh.tracts);
        p.slab_c0[k] = hc.size();
        for (size_t i = a0; i < a1; i++) {
            const VsStream &s = hs[i];
            /* host outputs are mirrored on the device at the same offsets relative to a 16-byte
             * aligned slab base, so the phase of a row is its sample offset mod 8 either way */
            const uint32_t ph = (uint32_t)((out_base + s.out_off) & sh.ph_mask);
            const uint32_t W = flow ? 0u : (uint32_t)warm[s.preset];
            /* chunk c > 0 emits [L0 + (c-1)*L - ph, L0 + c*L - ph); L0 and L are multiples of 8 (of 256 for the
             * lanes-along-the-row flow kernel, whose steps then never straddle two chunks) */
            uint32_t C, L, L0;
            if (flow) {
                L = L0 = Lflow;
                C = (L == 0 || s.n <= L) ? 1u : (uint32_t)((s.n + L - 1) / L);
            } else {
                C = nch[i - a0];
                L = L0 = 0u;
                if (C > 1) {
                    if (o.chunk == 0 && (uint64_t)s.n > (uint64_t)W + 64ull * C) {       /* auto planning */
                        /* equal WORK per row: the first chunk has no warm-up and emits W samples more */
                        L = (uint32_t)(((s.n - W + C - 1) / C + 7u) & ~7u);
                        const uint32_t rest = (C - 1) * L;
                        L0 = rest < s.n ? ((s.n - rest + 7u) & ~7u) : 0u;
                    }
                    if (L0 == 0u || L0 < L) {                      /* stream barely longer than the warm-up: equal chunks */
                        L = L0 = (uint32_t)(((s.n + C - 1) / C + 7u) & ~7u);
                    }
                    C = s.n <= L0 ? 1u : 1u + (uint32_t)((s.n - L0 + L - 1) / L);
                }
            }
            p.nch[i - s0] = C;
            p.tab_total += s.tab_cap;
            for (uint32_t c = 0; c < C; c++) {
                VsChunk ck;
                memset(&ck, 0, sizeof ck);
                ck.stream = (uint32_t)(i - s0);
                ck.emit_lo = c == 0 ? 0u : L0 + (c - 1) * L - ph;
                ck.emit_hi = c + 1 == C ? s.n : L0 + c * L - ph;
                ck.gen_target = ck.emit_lo > W ? ck.emit_lo - W : 0u;
                if (c > 0) p.warm_total += ck.emit_lo - ck.gen_target;
                hc.push_back(ck);
            }
        }
    }
    p.slab_c0[slabs.size()] = hc.size();
}

/* Render rows: ONE launch per slab.  Rows are grouped by filter group (vowel preset or tract) and every group is padded
 * to whole blocks of rows with VS_NO_CHUNK rows, so that a block's group is a function of blockIdx (its coefficients
 * then sit in uniform registers).  Inside a group: longest first (the 32 lanes of a warp run a similar number of
 * windows), rows of equal work next to each other by pulse table (a warp stages each distinct table of its rows once). */
void vs_plan_rows(const VsShape &sh, const std::vector<VsStream> &hs, size_t s0, VsPlan &p)
{
    const bool flow = sh.mode == VS_MODE_FLOW;
    const std::vector<VsChunk> &hc = p.chunks;
    const size_t n_slabs = p.slab_c0.size() - 1;
    std::vector<uint32_t> &order = p.order;
    order.clear();
    p.geom.assign(n_slabs, VsPlan::Geom());
    p.slab_r0.assign(n_slabs + 1, 0);
    auto group_of = [&](uint32_t c) -> int { return flow ? 0 : hs[s0 + hc[c].stream].preset; };
    for (size_t k = 0; k < n_slabs; k++) {
        p.slab_r0[k] = order.size();
        std::vector<uint32_t> ids(p.slab_c0[k + 1] - p.slab_c0[k]);
        {   /* sort by one 64-bit key per row (group, work descending, pulse table), then by id: the comparator of a
             * sort over the descriptors themselves cost 2.6 ms per 16 384 rows */
            std::vector<std::pair<uint64_t, uint32_t>> keyed(ids.size());
            for (size_t c = 0; c < ids.size(); c++) {
                const uint32_t id = (uint32_t)(p.slab_c0[k] + c);
                /* (flow-only chunks are all about one length: keep rows that share a pulse table together instead) */
                const uint32_t work = flow ? 0u : (hc[id].emit_hi - hc[id].gen_target) >> 6;
                keyed[c] = {((uint64_t)group_of(id) << 57) | ((uint64_t)(0x01ffffffu - std::min(work, 0x01ffffffu)) << 32) |
                                (uint64_t)hs[s0 + hc[id].stream].pulse_off, id};
            }
            std::sort(keyed.begin(), keyed.end());
            for (size_t c = 0; c < ids.size(); c++) ids[c] = keyed[c].second;
        }
        VsPlan::Geom &gm = p.geom[k];
        const size_t r_first = order.size();
        size_t i0 = 0;
        int done = 0;
        while (i0 < ids.size()) {
            size_t i1 = i0;
            const int gr = group_of(ids[i0]);
            while (i1 < ids.size() && group_of(ids[i1]) == gr) i1++;
            for (; done < gr; done++) gm.cta_end[done] = (uint32_t)((order.size() - r_first) / sh.group_rows);
            for (size_t i = i0; i < i1; i++) order.push_back(ids[i]);
            while ((order.size() - r_first) % sh.group_rows) order.push_back(VS_NO_CHUNK);
            i0 = i1;
        }
        for (; done < sh.n_groups; done++) gm.cta_end[done] = (uint32_t)((order.size() - r_first) / sh.group_rows);
        /* pulse-table cache: the largest sum of distinct (padded) tables over the warps of the slab */
        gm.cache_doubles = 0;
        if (sh.mode != VS_MODE_FILTER) {
            for (size_t r = r_first; r < order.size(); r += 32) {
                uint32_t seen[32], nseen = 0, sum = 0;
                for (size_t j = r; j < r + 32; j++) {
                    if (order[j] == VS_NO_CHUNK) continue;
                    const VsStream &st = hs[s0 + hc[order[j]].stream];
                    bool dup = false;
                    for (uint32_t u = 0; u < nseen; u++) dup |= seen[u] == st.pulse_off;
                    if (!dup) { seen[nseen++] = st.pulse_off; sum += st.tpad; }
                }
                gm.cache_doubles = std::max(gm.cache_doubles, sum);
            }
        }
    }
    p.slab_r0[n_slabs] = order.size();
}

void vs_plan_assign(const VsPlan &p, std::vector<VsStream> &hs, size_t s0, size_t s1)
{
    uint32_t c0acc = 0;
    uint64_t tacc = 0;
    for (size_t i = s0; i < s1; i++) {
        hs[i].chunk0 = c0acc; hs[i].n_chunks = p.nch[i - s0]; hs[i].tab_off = tacc;
        c0acc += hs[i].n_chunks; tacc += hs[i].tab_cap;
    }
}

int vs_render_geometry(const VsPlanOptions &o, const VsShape &sh, const VsFacts &fc, int sm_count, size_t ns, const VsPlan &p,
                       size_t k, VsRenderArgs &ra)
{
    ra.n_rows = (uint32_t)(p.slab_r0[k + 1] - p.slab_r0[k]);
    memcpy(ra.cta_end, p.geom[k].cta_end, sizeof ra.cta_end);
    ra.compact = sh.compact;
    ra.general_pulse = sh.general_pulse ? 1 : 0;
    /* shared-memory geometry.  The fast generator keeps, per lane, a ring of upcoming period entries (filled
     * one window ahead) and, per warp, the pulse tables of its rows; when the pitch periods of the batch are
     * too short or the tables too many for that, the general generator takes over. */
    const int win = VS_WIN(sh.mode);
    const uint32_t tile_bytes = (uint32_t)VS_RENDER_TILES(sh.mode) * 32u * (uint32_t)win * 2u;
    int gen = VS_GEN_SIMPLE;
    ra.warp_bytes = tile_bytes;
    if (sh.mode != VS_MODE_FILTER && sh.compact != VS_TAB_FULL && branch_free(fc, o) && fc.t_max <= 8192) {
        /* pitch periods a lane can enter in one window (+1: the generator may already have promoted the period
         * that starts with the next window); the ring holds two windows' worth */
        const uint32_t per_win = (uint32_t)((win + fc.t_min - 1) / fc.t_min) + 1u;
        const uint32_t ahead = 2u * per_win + 2u;
        uint32_t R = 8;
        while (R < ahead) R <<= 1;
        /* the pulse-table cache: what the typical warp of this row order needs, as far as shared memory goes
         * (a warp that needs more renders its rows with the general generator) */
        const uint32_t budget = (sh.mode == VS_MODE_FLOW ? 100u : 200u) * 1024u / 4u;
        const uint32_t fixed = tile_bytes + R * 32u * VS_TAB_ENTRY_BYTES(sh.compact);
        uint32_t cache = std::max(16u, (p.geom[k].cache_doubles + 1u) & ~1u);
        if (fixed + 4096u <= budget) cache = std::min(cache, ((budget - fixed) / 8u) & ~1u);
        const uint32_t wbytes = fixed + cache * 8u;
        if (R <= 64 && wbytes <= budget) {
            gen = VS_GEN_FAST;
            ra.warp_bytes = wbytes; ra.ring_R = R; ra.ring_fetch = per_win + 2u; ra.ring_ahead = ahead; ra.cache_doubles = cache;
        }
    }
    /* persistent grid: one CTA per render SM (the plan kernels of the next calls own the others); the flow-only kernel
     * is small, a few of its CTAs share an SM */
    const uint32_t blocks = (ra.n_rows / 32u + 3u) / 4u;
    const int plan_ctas = (int)((ns + (size_t)sh.plan_nt - 1) / (size_t)sh.plan_nt);
    const uint32_t sms = (uint32_t)std::max(1, sm_count - vs_plan_reserve(plan_ctas));
    uint32_t per_sm = 1;
    if (sh.mode == VS_MODE_FLOW) per_sm = std::max(1u, std::min(4u, (220u * 1024u) / (4u * ra.warp_bytes + (sh.noise ? 16u * 1024u : 0u) + 1024u)));
    ra.grid = std::min(blocks, sms * per_sm);
    if (sh.flow_rows) {
        const uint32_t rows_per_cta = VS_FLOWROWS_WARPS;
        ra.grid = std::max(1u, std::min((ra.n_rows + rows_per_cta - 1u) / rows_per_cta, sms * 4u));
    }
    return gen;
}

uint32_t vs_render_path(const VsShape &sh, int gen)
{
    return (gen == VS_GEN_FAST || sh.flow_rows ? 1u : 0u) | (sh.noise ? 2u : 0u) | ((uint32_t)sh.filt << 2) | (sh.flow_rows ? 32u : 0u) |
           (sh.tracts ? 64u : 0u);
}

/* One warp per stream while the batch is too small to fill the GPU with one thread per stream (measured crossover on
 * B200: ~8 k streams, ~14 k with glottal noise).  The warp form issues ~7x the instructions, though: next to a render
 * still running it would take issue slots from the FP64-bound render warps, while the thread form hides on its own SMs
 * -- so with a call in flight only really small batches take it. */
bool vs_plan_warps(int opt_plan_warps, size_t n_streams, bool any_noise, bool want_log, bool busy, unsigned burst)
{
    if (want_log) return false;                     /* the warp form writes no period log */
    if (opt_plan_warps >= 0) return opt_plan_warps != 0;
    /* the second call of a burst that began on an idle device: its plan must be ready when the first call's render ends;
     * the thread form (0.39 ms on the bench batch, behind the first call's warp-form plan) would be late by a quarter of a
     * step, and every call behind it too.  (With glottal noise the warp form is too heavy to share the SMs with a render:
     * cfg3 157 -> 150 Gsamples/s) */
    const bool early = busy && burst == 1u && !any_noise;
    return n_streams <= (busy && !early ? VS_PLAN_WARP_MAX : any_noise ? VS_PLAN_WARP_MAX_NOISE : VS_PLAN_WARP_MAX_IDLE);
}

/* ---- the C ABI's helpers that do no GPU work ------------------------------------------------------------------- */
extern "C" {

int vs_flow_nsamples(const vs_flow_params *p, size_t n, uint64_t *out)
{
    if (!out) return VS_EINVAL;
    for (size_t i = 0; i < n; i++) out[i] = row_nsamples(flow_row(p, i));
    return VS_OK;
}

int vs_flow_max_periods(const vs_flow_params *p, size_t n, uint64_t *out)
{
    if (!out) return VS_EINVAL;
    for (size_t i = 0; i < n; i++) {
        const FlowRow r = flow_row(p, i);
        if (row_validate(r)) { out[i] = 0; continue; }
        out[i] = row_max_periods(r, row_nsamples(r), row_P(r));
    }
    return VS_OK;
}

int vs_flow_validate(const vs_flow_params *p, size_t n, size_t *bad)
{
    for (size_t i = 0; i < n; i++) {
        const int rc = row_validate(flow_row(p, i));
        if (rc) { if (bad) *bad = i; return rc; }
    }
    return VS_OK;
}

int vs_tract_from_formants(const float *freq_hz, const float *bw_hz, int n_formants, int32_t fs, double den[23])
{
    if (!freq_hz || !bw_hz || !den || n_formants < 1 || 2 * n_formants > VS_ORDER) return VS_EINVAL;
    if (fs <= 0) return VS_ERANGE;
    const double pi = 3.14159265358979323846, rate = (double)fs;
    for (int k = 0; k < n_formants; k++) {
        const double F = freq_hz[k], B = bw_hz[k];
        if (!(F > 0.0 && F < 0.5 * rate) || !(B > 0.0) || !std::isfinite(B)) return VS_ERANGE;
    }
    double d[VS_ORDER + 1] = {1.0};
    for (int k = 0; k < n_formants; k++) {
        const double r = std::exp(-pi * (double)bw_hz[k] / rate), th = 2.0 * pi * (double)freq_hz[k] / rate;
        const double b1 = -2.0 * r * std::cos(th), b2 = r * r;
        for (int j = 2 * k + 2; j >= 1; j--) {         /* d <- d * (1 + b1 z^-1 + b2 z^-2), in place from the top */
            double v = d[j] + b1 * d[j - 1];
            if (j >= 2) v += b2 * d[j - 2];
            d[j] = v;
        }
    }
    memcpy(den, d, sizeof d);
    return VS_OK;
}

int vs_tract_from_preset(int preset_key, double den[23])
{
    const int k = preset_index(preset_key);
    if (k < 0) return VS_EPRESET;
    if (!den) return VS_EINVAL;
    memcpy(den, vs_preset_den[k], (VS_ORDER + 1) * sizeof(double));
    return VS_OK;
}

} /* extern "C" */
