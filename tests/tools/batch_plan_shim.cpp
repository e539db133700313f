/* batch_plan_shim.cpp -- drives the batch planner (voice_synth_b200/csrc/vs_batch_plan.cpp) without a GPU, for
 * tests/test_batch_plan_host.py: one call plans a batch on one device slot, the other copies the plan out. */
#include <cstring>

#include "../../voice_synth_b200/csrc/vs_batch_plan.h"

static VsDescriptors g_d;
static VsShape g_sh;
static std::vector<VsRange> g_slabs;
static VsPlan g_plan;
static std::vector<int> g_gen;
static std::string g_err;

/* info[]: chunks, rows, slabs, warm-up samples, flow_rows, group_rows, n_groups, filter groups with a warm-up, then the
 * rest of the record: compact, tracts, plan, plan_nt, filt, raw, noise, general_pulse */
extern "C" int shim_plan(int mode, size_t n, const vs_flow_params *fp, const vs_filter_params *ff, const vs_tract_params *ft,
                         const uint64_t *nsamp, const uint64_t *offsets, const uint64_t *rec_offsets, double chunk, int exact,
                         int slab, int simple_gen, int raw, int sm_count, int out_dev, uint64_t out_base, uint64_t *info)
{
    VsPlanOptions o;
    o.chunk = chunk;
    o.exact = exact;
    o.slab = slab;
    o.simple_gen = simple_gen;
    VsTables tab;
    tab.set_tol(o.tol);
    vs_period_log log = {nullptr, const_cast<uint64_t *>(rec_offsets), nullptr};
    double raw_out = 0.0;            /* the planner only asks whether there is one */
    const VsBatch b = {mode, n, fp, ff, ft, nullptr, nullptr, nsamp, nullptr, offsets, raw ? &raw_out : nullptr, &log};
    const bool want_log = rec_offsets != nullptr;
    const int rc = vs_build_descriptors(b, want_log, tab, g_d, g_err);
    if (rc) return rc;
    g_sh = vs_shape(mode, ft != nullptr, want_log, g_d.facts, o);
    const std::vector<size_t> cut = vs_split_slots(g_d.hs, 1);
    size_t per = 0;
    g_slabs = vs_slabs(g_d.hs, cut[0], cut[1], out_dev != 0, o.slab, &per);
    vs_plan_chunks(o, g_sh, sm_count, g_d.hs, cut[0], cut[1], g_slabs, g_d.warm.data(), out_base, g_plan);
    vs_plan_rows(g_sh, g_d.hs, cut[0], g_plan);
    vs_plan_assign(g_plan, g_d.hs, cut[0], cut[1]);
    g_gen.resize(g_slabs.size());
    for (size_t k = 0; k < g_slabs.size(); k++) {
        VsRenderArgs ra;
        memset(&ra, 0, sizeof ra);
        g_gen[k] = vs_render_geometry(o, g_sh, g_d.facts, sm_count, cut[1] - cut[0], g_plan, k, ra);
    }
    const uint64_t v[16] = {g_plan.chunks.size(), g_plan.order.size(), g_slabs.size(), g_plan.warm_total, g_sh.flow_rows,
                            g_sh.group_rows, (uint64_t)g_sh.n_groups, g_d.warm.size(), (uint64_t)g_sh.compact, g_sh.tracts,
                            (uint64_t)g_sh.plan, (uint64_t)g_sh.plan_nt, (uint64_t)g_sh.filt, g_sh.raw, g_sh.noise,
                            g_sh.general_pulse};
    memcpy(info, v, sizeof v);
    return VS_OK;
}

extern "C" int shim_plan_warps(int opt_plan_warps, size_t n_streams, int any_noise, int want_log, int busy, unsigned burst)
{
    return vs_plan_warps(opt_plan_warps, n_streams, any_noise != 0, want_log != 0, busy != 0, burst);
}

/* streams[n][7]: n, group, pulse_off, tpad, chunk0, n_chunks, out_off; chunks[c][4]: stream, emit_lo, emit_hi,
 * gen_target; slabs[k][4]: first stream, end, first chunk, first row (k = n_slabs: the totals); cta_end[k][n_groups];
 * per slab its pulse-table cache, generator and render_path */
extern "C" void shim_fetch(uint64_t *streams, uint32_t *chunks, uint32_t *order, uint64_t *slabs, uint32_t *cta_end,
                           uint32_t *cache_doubles, int32_t *warm, int32_t *gen, uint32_t *render_path)
{
    for (size_t i = 0; i < g_d.hs.size(); i++) {
        const VsStream &s = g_d.hs[i];
        const uint64_t v[7] = {s.n, s.preset, s.pulse_off, s.tpad, s.chunk0, s.n_chunks, s.out_off};
        memcpy(streams + 7 * i, v, sizeof v);
    }
    for (size_t c = 0; c < g_plan.chunks.size(); c++) {
        const VsChunk &ck = g_plan.chunks[c];
        const uint32_t v[4] = {ck.stream, ck.emit_lo, ck.emit_hi, ck.gen_target};
        memcpy(chunks + 4 * c, v, sizeof v);
    }
    memcpy(order, g_plan.order.data(), g_plan.order.size() * sizeof(uint32_t));
    for (size_t k = 0; k <= g_slabs.size(); k++) {
        const bool end = k == g_slabs.size();
        const uint64_t v[4] = {end ? g_slabs.back().second : g_slabs[k].first, end ? 0 : g_slabs[k].second, g_plan.slab_c0[k],
                               g_plan.slab_r0[k]};
        memcpy(slabs + 4 * k, v, sizeof v);
    }
    for (size_t k = 0; k < g_slabs.size(); k++) {
        memcpy(cta_end + k * g_sh.n_groups, g_plan.geom[k].cta_end, g_sh.n_groups * sizeof(uint32_t));
        cache_doubles[k] = g_plan.geom[k].cache_doubles;
        gen[k] = g_gen[k];
        render_path[k] = vs_render_path(g_sh, g_gen[k]);
    }
    memcpy(warm, g_d.warm.data(), g_d.warm.size() * sizeof(int32_t));
}
