"""The batch planner (voice_synth_b200/csrc/vs_batch_plan.cpp) on the CPU: the invariants the render and plan kernels rely
on, checked on the plans of the bench shapes and of every option that changes a plan.  The planner is compiled with a
small shim (tests/tools/batch_plan_shim.cpp) and the host flags of the library."""
import ctypes as C
import pathlib
import subprocess

import numpy as np
import pytest

from voice_synth_b200 import api, workloads

ROOT = pathlib.Path(__file__).resolve().parents[1]

SM_COUNT = 148                     # B200
OUT_BASE = (0x7F12_3400_0000 >> 1)  # a 256-byte aligned device output, in samples
FLOW, SYNTH, FILTER = 0, 1, 2
NO_CHUNK = 0xFFFFFFFF


def _nsamples(L, p):
    out = np.zeros(p.n, dtype=np.uint64)
    assert L.vs_flow_nsamples(C.byref(p._c()), C.c_size_t(p.n), C.c_void_p(out.ctypes.data)) == 0
    return out


def _den(L, call, *args):
    den = np.zeros(23, dtype=np.float64)
    assert call(*args, C.c_void_p(den.ctypes.data)) == 0
    return den


def _preset_tracts(L):
    return np.stack([_den(L, L.vs_tract_from_preset, C.c_int(ord(k))) for k in workloads.PRESETS])


def _formant_tracts(L, nt):
    bw = np.array([60.0, 90.0, 120.0, 150.0], dtype=np.float32)
    fr = [np.array([300.0 + 9.0 * t, 1200.0 + 11.0 * t, 2500.0, 3400.0], dtype=np.float32) for t in range(nt)]
    return np.stack([_den(L, L.vs_tract_from_formants, C.c_void_p(f.ctypes.data), C.c_void_p(bw.ctypes.data), C.c_int(4),
                          C.c_int32(22050)) for f in fr])


SHAPES = ["cfg2", "cfg3_shard", "cfg5_slice", "flow_cfg2", "flow_cfg3_shard", "filter_only", "tracts_10", "tracts_128",
          "no_chunks", "fixed_chunks", "flow_fixed_chunks", "exact", "slab_97", "ragged", "period_log",
          "simple_gen", "flow_simple_gen", "raw", "gain_10_5", "flow_exact", "kvar",
          "limit_filter", "limit_filter_chunk_2e27", "limit_filter_no_chunks", "limit_flow", "limit_flow_no_chunks",
          "limit_flow_simple_gen", "limit_flow_noise", "limit_synth", "limit_synth_no_chunks", "limit_tracts_10",
          "limit_tracts_10_no_chunks"]

# The longest rows the ABI accepts: 2^31 - 1 samples of caller PCM, and the longest flow (float)fs * dur can give,
# 2^31 - 128 samples (16 kHz for 134217.71875 s)
LIMIT_NSAMP = 2**31 - 1
LIMIT_FLOW_NSAMP = 2**31 - 128


def limit_flow_params(noise=0.0):
    """one voice of LIMIT_FLOW_NSAMP samples: strictly periodic (160 samples a period), with glottal noise if noise > 0"""
    return api.FlowParams(1, fs=16000, dur=134217.71875, F0=100.0, noise=noise, seed=7, flags=4 if noise > 0 else 0)


def shapes(L):
    """name -> the arguments of one batch call: mode, flow params, filter or tract params, nsamp (filter mode), offsets,
    period log, options and where the output lives.  L: a library with the C ABI's host helpers (vs_flow_nsamples,
    vs_tract_from_*), the planner shim or libvoicesynth_cuda.so"""
    p2, f2 = workloads.cfg2()
    p3, f3 = workloads.cfg3(n=8192, first=20480)
    p5, f5 = workloads.cfg5(n=6144, first=300000)
    rng = np.random.default_rng(5)
    ns_filter = rng.integers(500, 90000, 3000).astype(np.uint64)
    f_filter = api.FilterParams(3000)
    f_filter.preset[...] = [ord(workloads.PRESETS[(i * 7) % 10]) for i in range(3000)]
    f_gain = f2.select(np.arange(f2.n))
    f_gain.gain[0] = 10.5
    p_kvar = p2.select(np.arange(p2.n))
    p_kvar.Kvar[::7] = 0.3
    sub = np.arange(1024)
    p_lim = limit_flow_params()
    f_lim = api.FilterParams(1, preset="u")
    t_lim = api.TractParams(1, _preset_tracts(L), tract=[workloads.PRESETS.index("u")])     # the preset 'u' as a tract
    p_lim_noise = limit_flow_params(noise=10.0)
    p_sub, f_sub = p2.select(sub), f2.select(sub)
    ns_sub = _nsamples(L, p_sub)
    ragged = np.concatenate([[0], np.cumsum(ns_sub[:-1] + rng.integers(0, 300, 1023).astype(np.uint64))]).astype(np.uint64) + 3
    t10 = api.TractParams(4096, _preset_tracts(L), tract=np.arange(4096) % 10)
    t128 = api.TractParams(4096, _formant_tracts(L, 128), tract=(np.arange(4096) * 37) % 128)
    d = dict(mode=SYNTH, f=None, nsamp=None, offsets=None, log=False, chunk=0, exact=0, slab=0, simple_gen=0, raw=False,
             out_dev=True)
    return {
        "cfg2": dict(d, p=p2, f=f2),
        "cfg3_shard": dict(d, p=p3, f=f3),
        "cfg5_slice": dict(d, p=p5, f=f5),
        "flow_cfg2": dict(d, mode=FLOW, p=p2),
        "flow_cfg3_shard": dict(d, mode=FLOW, p=p3),
        "filter_only": dict(d, mode=FILTER, p=None, f=f_filter, nsamp=ns_filter),
        "tracts_10": dict(d, p=p2, f=t10),
        "tracts_128": dict(d, p=p2, f=t128),
        "no_chunks": dict(d, p=p2, f=f2, chunk=-1),
        "fixed_chunks": dict(d, p=p2, f=f2, chunk=3000),
        "flow_fixed_chunks": dict(d, mode=FLOW, p=p2, chunk=3000),
        "exact": dict(d, p=p2, f=f2, exact=1),
        "slab_97": dict(d, p=p2, f=f2, slab=97, out_dev=False),
        "ragged": dict(d, p=p_sub, f=f_sub, offsets=ragged),
        "period_log": dict(d, mode=FLOW, p=p3.select(np.arange(512)), log=True),
        "simple_gen": dict(d, p=p2, f=f2, simple_gen=1),
        "flow_simple_gen": dict(d, mode=FLOW, p=p2, simple_gen=1),
        "raw": dict(d, p=p2, f=f2, raw=True),
        "gain_10_5": dict(d, p=p2, f=f_gain),
        "flow_exact": dict(d, mode=FLOW, p=p2, exact=1),
        "kvar": dict(d, p=p_kvar, f=f2),
        "limit_filter": dict(d, mode=FILTER, p=None, f=f_lim, nsamp=[LIMIT_NSAMP]),
        "limit_filter_chunk_2e27": dict(d, mode=FILTER, p=None, f=f_lim, nsamp=[LIMIT_NSAMP], chunk=2**27),
        "limit_filter_no_chunks": dict(d, mode=FILTER, p=None, f=f_lim, nsamp=[LIMIT_NSAMP], chunk=-1),
        "limit_flow": dict(d, mode=FLOW, p=p_lim),
        "limit_flow_no_chunks": dict(d, mode=FLOW, p=p_lim, chunk=-1),
        "limit_flow_simple_gen": dict(d, mode=FLOW, p=p_lim, simple_gen=1),
        "limit_flow_noise": dict(d, mode=FLOW, p=p_lim_noise),
        "limit_synth": dict(d, p=p_lim, f=f_lim),
        "limit_synth_no_chunks": dict(d, p=p_lim, f=f_lim, chunk=-1),
        "limit_tracts_10": dict(d, p=p_lim, f=t_lim),
        "limit_tracts_10_no_chunks": dict(d, p=p_lim, f=t_lim, chunk=-1),
    }


# total chunks and warm-up samples that vs_get_timing reports for these calls on a B200 (148 SMs), device output
PINNED = {"cfg2": (17614, 32765084), "cfg3_shard": (30310, 53758613), "cfg5_slice": (15967, 24523171)}


# The kernels of each shape: the record vs_shape makes (table format, warp-per-row flow, tracts, filter groups and their
# padding, the thread-form plan kernel and its streams per CTA, filter arithmetic, raw output, glottal noise, -z), then
# the generator and the vs_timing::render_path of every slab.  (Flow-only calls report the filter bits although they
# run no filter.)
TAB_FULL, TAB_C8, TAB_N16 = 0, 1, 2
LEAN, PULSE, LOG = 0, 1, 2
F_INT, F_FMA, F_EXACT = 0, 1, 2
FAST, SIMPLE = 0, 1
KERNELS = {
    "cfg2":               (TAB_C8, 0, 0, 10, 32, LEAN, 1024, F_INT, 0, 0, 0, FAST, 1),
    "cfg3_shard":         (TAB_N16, 0, 0, 10, 32, PULSE, 512, F_INT, 0, 1, 0, FAST, 3),
    "cfg5_slice":         (TAB_N16, 0, 0, 10, 32, PULSE, 512, F_INT, 0, 1, 0, FAST, 3),
    "flow_cfg2":          (TAB_C8, 1, 0, 10, 32, LEAN, 1024, F_INT, 0, 0, 0, FAST, 33),
    "flow_cfg3_shard":    (TAB_N16, 0, 0, 10, 32, PULSE, 512, F_INT, 0, 1, 0, FAST, 3),
    "filter_only":        (TAB_C8, 0, 0, 10, 32, LEAN, 1024, F_INT, 0, 0, 0, SIMPLE, 0),
    "tracts_10":          (TAB_C8, 0, 1, 128, 128, LEAN, 1024, F_INT, 0, 0, 0, FAST, 65),
    "tracts_128":         (TAB_C8, 0, 1, 128, 128, LEAN, 1024, F_INT, 0, 0, 0, FAST, 65),
    "no_chunks":          (TAB_C8, 0, 0, 10, 32, LEAN, 1024, F_INT, 0, 0, 0, FAST, 1),
    "fixed_chunks":       (TAB_C8, 0, 0, 10, 32, LEAN, 1024, F_INT, 0, 0, 0, FAST, 1),
    "flow_fixed_chunks":  (TAB_C8, 1, 0, 10, 32, LEAN, 1024, F_INT, 0, 0, 0, FAST, 33),
    "exact":              (TAB_C8, 0, 0, 10, 32, LEAN, 1024, F_EXACT, 0, 0, 0, FAST, 9),
    "slab_97":            (TAB_C8, 0, 0, 10, 32, LEAN, 1024, F_INT, 0, 0, 0, FAST, 1),
    "ragged":             (TAB_C8, 0, 0, 10, 32, LEAN, 1024, F_INT, 0, 0, 0, FAST, 1),
    "period_log":         (TAB_FULL, 0, 0, 10, 32, LOG, 512, F_INT, 0, 1, 0, SIMPLE, 2),
    "simple_gen":         (TAB_C8, 0, 0, 10, 32, LEAN, 1024, F_INT, 0, 0, 0, SIMPLE, 0),
    "flow_simple_gen":    (TAB_C8, 0, 0, 10, 32, LEAN, 1024, F_INT, 0, 0, 0, SIMPLE, 0),
    "raw":                (TAB_C8, 0, 0, 10, 32, LEAN, 1024, F_FMA, 1, 0, 0, FAST, 5),
    "gain_10_5":          (TAB_C8, 0, 0, 10, 32, LEAN, 1024, F_FMA, 0, 0, 0, FAST, 5),
    "flow_exact":         (TAB_C8, 1, 0, 10, 32, LEAN, 1024, F_EXACT, 0, 0, 0, FAST, 41),
    "kvar":               (TAB_FULL, 0, 0, 10, 32, LEAN, 1024, F_INT, 0, 0, 1, SIMPLE, 0),
    "limit_filter":       (TAB_C8, 0, 0, 10, 32, LEAN, 1024, F_INT, 0, 0, 0, SIMPLE, 0),
    "limit_filter_chunk_2e27": (TAB_C8, 0, 0, 10, 32, LEAN, 1024, F_INT, 0, 0, 0, SIMPLE, 0),
    "limit_filter_no_chunks": (TAB_C8, 0, 0, 10, 32, LEAN, 1024, F_INT, 0, 0, 0, SIMPLE, 0),
    "limit_flow":         (TAB_C8, 1, 0, 10, 32, LEAN, 1024, F_INT, 0, 0, 0, FAST, 33),
    "limit_flow_no_chunks": (TAB_C8, 1, 0, 10, 32, LEAN, 1024, F_INT, 0, 0, 0, FAST, 33),
    "limit_flow_simple_gen": (TAB_C8, 0, 0, 10, 32, LEAN, 1024, F_INT, 0, 0, 0, SIMPLE, 0),
    "limit_flow_noise":   (TAB_N16, 0, 0, 10, 32, PULSE, 512, F_INT, 0, 1, 0, FAST, 3),
    "limit_synth":        (TAB_C8, 0, 0, 10, 32, LEAN, 1024, F_INT, 0, 0, 0, FAST, 1),
    "limit_synth_no_chunks": (TAB_C8, 0, 0, 10, 32, LEAN, 1024, F_INT, 0, 0, 0, FAST, 1),
    "limit_tracts_10":    (TAB_C8, 0, 1, 128, 128, LEAN, 1024, F_INT, 0, 0, 0, FAST, 65),
    "limit_tracts_10_no_chunks": (TAB_C8, 0, 1, 128, 128, LEAN, 1024, F_INT, 0, 0, 0, FAST, 65),
}

# VS_OPT_PLAN_WARPS, streams, glottal noise, period log, busy, burst -> the plan kernel's warp form
PLAN_WARPS = [
    (-1, 1024, 0, 0, 1, 2, 1), (-1, 1025, 0, 0, 1, 2, 0),        # a call in flight
    (-1, 6144, 0, 0, 0, 0, 1), (-1, 6145, 0, 0, 0, 0, 0),        # an idle device
    (-1, 12288, 1, 0, 0, 0, 1), (-1, 12289, 1, 0, 0, 0, 0),      # an idle device, glottal noise
    (-1, 1024, 1, 0, 1, 2, 1), (-1, 1025, 1, 0, 1, 2, 0),        # a call in flight, glottal noise
    (-1, 6144, 0, 0, 1, 1, 1), (-1, 6145, 0, 0, 1, 1, 0),        # the second call of a burst: the idle limit ...
    (-1, 1024, 1, 0, 1, 1, 1), (-1, 1025, 1, 0, 1, 1, 0),        # ... but not with glottal noise
    (0, 16, 0, 0, 0, 0, 0), (0, 16, 1, 0, 1, 1, 0),              # option 0: the thread form
    (1, 50000, 0, 0, 1, 5, 1), (1, 50000, 1, 0, 0, 0, 1),        # option 1: the warp form
    (-1, 16, 0, 1, 0, 0, 0), (1, 16, 1, 1, 1, 1, 0),             # a period log: the thread form whatever else
]


def build_shim(out_dir):
    """the planner and the shim as a shared library in out_dir"""
    out = pathlib.Path(out_dir) / "libbatch_plan_shim.so"
    subprocess.run(["g++", "-O3", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-o", str(out),
                    str(ROOT / "tests" / "tools" / "batch_plan_shim.cpp"), str(ROOT / "voice_synth_b200" / "csrc" / "vs_batch_plan.cpp")],
                   check=True)
    L = C.CDLL(str(out))
    L.shim_plan.restype = C.c_int
    L.shim_plan.argtypes = [C.c_int, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                            C.c_double, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_void_p]
    L.shim_fetch.restype = None
    L.shim_plan_warps.restype = C.c_int
    L.shim_plan_warps.argtypes = [C.c_int, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_uint]
    L.vs_flow_max_periods.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p]
    return L


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    return build_shim(tmp_path_factory.mktemp("batch_plan"))


@pytest.fixture(scope="module")
def all_shapes(shim):
    return shapes(shim)


def plan(L, s):
    """run the planner on shape s; the plan as numpy arrays"""
    keep = []

    def ref(x):
        if x is None:
            return None
        keep.append(x)
        return C.addressof(x)

    mode, p, f = s["mode"], s["p"], s["f"]
    n = p.n if p is not None else len(s["nsamp"])
    fp = ref(p._c()) if p is not None else None
    ff = ref(f._c()) if isinstance(f, api.FilterParams) else None
    ft = ref(f._c()) if isinstance(f, api.TractParams) else None
    rec = None
    if s["log"]:
        mp = np.zeros(n, dtype=np.uint64)
        L.vs_flow_max_periods(fp, n, mp.ctypes.data)
        rec = np.concatenate([[0], np.cumsum(mp)]).astype(np.uint64)
    nsamp = None if s["nsamp"] is None else np.ascontiguousarray(s["nsamp"], dtype=np.uint64)
    offs = None if s["offsets"] is None else np.ascontiguousarray(s["offsets"], dtype=np.uint64)
    ptr = lambda a: None if a is None else a.ctypes.data  # noqa: E731
    info = np.zeros(16, dtype=np.uint64)
    rc = L.shim_plan(mode, n, fp, ff, ft, ptr(nsamp), ptr(offs), ptr(rec), float(s["chunk"]), s["exact"], s["slab"],
                     s["simple_gen"], int(s["raw"]), SM_COUNT, int(s["out_dev"]), OUT_BASE if s["out_dev"] else 0, info.ctypes.data)
    assert rc == 0, rc
    nc, nr, nsl, warm_total, flow_rows, group_rows, n_groups, n_warm = (int(v) for v in info[:8])
    r = dict(warm_total=warm_total, flow_rows=bool(flow_rows), group_rows=group_rows, n_groups=n_groups,
             record=tuple(int(v) for v in info[8:]),
             streams=np.zeros((n, 7), dtype=np.uint64), chunks=np.zeros((nc, 4), dtype=np.uint32),
             order=np.zeros(nr, dtype=np.uint32), slabs=np.zeros((nsl + 1, 4), dtype=np.uint64),
             cta_end=np.zeros((nsl, n_groups), dtype=np.uint32), cache=np.zeros(nsl, dtype=np.uint32),
             warm=np.zeros(n_warm, dtype=np.int32), gen=np.zeros(nsl, dtype=np.int32), render_path=np.zeros(nsl, dtype=np.uint32))
    L.shim_fetch(*(r[k].ctypes.data_as(C.c_void_p)
                   for k in ("streams", "chunks", "order", "slabs", "cta_end", "cache", "warm", "gen", "render_path")))
    return r


@pytest.mark.parametrize("name", SHAPES)
def test_batch_plan_invariants(shim, all_shapes, name):
    s = all_shapes[name]
    r = plan(shim, s)
    st, ck, order = r["streams"], r["chunks"].astype(np.int64), r["order"]
    n = len(st)
    flow = s["mode"] == FLOW
    W = np.zeros(1, dtype=np.int64) if flow else r["warm"].astype(np.int64)
    grp = np.zeros(n, dtype=np.int64) if flow else st[:, 1].astype(np.int64)
    ph_mask, grid = (63, 256) if r["flow_rows"] else (7, 8)
    phase = ((OUT_BASE if s["out_dev"] else 0) + st[:, 6]) & np.uint64(ph_mask)
    if s["slab"]:
        assert len(r["slabs"]) - 1 == -(-n // s["slab"])

    # 1. the chunks of each stream are consecutive, tile [0, n) and start on the phase grid
    assert st[0, 4] == 0 and np.array_equal(st[1:, 4], np.cumsum(st[:-1, 5])) and st[:, 5].sum() == len(ck)
    sid = np.repeat(np.arange(n), st[:, 5].astype(np.int64))
    assert np.array_equal(ck[:, 0], sid)
    first = st[:, 4].astype(np.int64)
    last = first + st[:, 5].astype(np.int64) - 1
    assert np.all(ck[first, 1] == 0) and np.array_equal(ck[last, 2], st[:, 0].astype(np.int64))
    inner = np.ones(len(ck), dtype=bool)
    inner[first] = False
    assert np.all(ck[:, 1] < ck[:, 2])
    assert np.array_equal(ck[np.flatnonzero(inner), 1], ck[np.flatnonzero(inner) - 1, 2])
    assert np.all((ck[inner, 1] + phase[sid[inner]].astype(np.int64)) % grid == 0)
    if s["chunk"] < 0 or s["exact"]:
        assert flow or len(ck) == n

    # 2. generation starts W samples before a chunk's output; the warm-ups add up to the reported total
    w = W[grp[sid]] if not flow else 0
    assert np.array_equal(ck[:, 3], np.maximum(0, ck[:, 1] - w))
    assert (ck[:, 1] - ck[:, 3]).sum() == r["warm_total"]

    # 3. + 4. per slab: rows, groups, group ends and the pulse-table cache
    gr = r["group_rows"]
    for k in range(len(r["slabs"]) - 1):
        a0, a1, c0, r0 = (int(v) for v in r["slabs"][k])
        c1, r1 = int(r["slabs"][k + 1][2]), int(r["slabs"][k + 1][3])
        assert np.array_equal(np.unique(sid[c0:c1]), np.arange(a0, a1))
        rows = order[r0:r1]
        real = rows[rows != NO_CHUNK].astype(np.int64)
        assert len(real) == c1 - c0 and np.array_equal(np.sort(real), np.arange(c0, c1))
        assert len(rows) % gr == 0 and len(rows) % 32 == 0
        blocks = rows.reshape(-1, gr)
        bgroup = []
        for b in blocks:
            m = b != NO_CHUNK
            assert m[0] and np.all(m[:m.sum()]), "padding only at the end of a group's last block"
            g = np.unique(grp[sid[b[m]]])
            assert len(g) == 1
            bgroup.append(int(g[0]))
        bgroup = np.array(bgroup)
        assert np.all(np.diff(bgroup) >= 0)
        for b in range(len(blocks) - 1):
            if bgroup[b] == bgroup[b + 1]:
                assert np.all(blocks[b] != NO_CHUNK), "only a group's last block is padded"
        cta = r["cta_end"][k]
        assert np.all(np.diff(cta.astype(np.int64)) >= 0)
        assert np.array_equal(cta, [(bgroup <= g).sum() for g in range(r["n_groups"])])
        if not flow:
            work = (ck[real, 2] - ck[real, 3]) >> 6
            g_real = grp[sid[real]]
            same = g_real[1:] == g_real[:-1]
            assert np.all(work[1:][same] <= work[:-1][same]), "within a group, work does not increase"
        if s["mode"] != FILTER:
            for wr in rows.reshape(-1, 32):
                ids = wr[wr != NO_CHUNK].astype(np.int64)
                tabs = {int(st[i, 2]): int(st[i, 3]) for i in sid[ids]}
                assert r["cache"][k] >= sum(tabs.values())
    if name in PINNED:
        assert (len(ck), r["warm_total"]) == PINNED[name]


@pytest.mark.parametrize("name", SHAPES)
def test_batch_plan_kernels(shim, all_shapes, name):
    r = plan(shim, all_shapes[name])
    compact, tracts, plan_form, plan_nt, filt, raw, noise, general_pulse = r["record"]
    record = (compact, int(r["flow_rows"]), tracts, r["n_groups"], r["group_rows"], plan_form, plan_nt, filt, raw, noise, general_pulse)
    assert record == KERNELS[name][:11]
    assert set(r["gen"].tolist()) == {KERNELS[name][11]} and set(r["render_path"].tolist()) == {KERNELS[name][12]}


def test_plan_warps(shim):
    for *args, warps in PLAN_WARPS:
        assert shim.shim_plan_warps(*args) == warps, args


def test_batch_plan_shapes_listed(all_shapes):
    assert list(all_shapes) == SHAPES


def test_batch_plan_paths(shim, all_shapes):
    """the kernel forms the shapes are meant to reach"""
    sh = all_shapes
    assert plan(shim, sh["flow_cfg2"])["flow_rows"]
    assert not plan(shim, sh["flow_cfg3_shard"])["flow_rows"]          # glottal noise
    assert plan(shim, sh["tracts_128"])["group_rows"] == 128 and plan(shim, sh["cfg2"])["group_rows"] == 32
