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
          "no_chunks", "fixed_chunks", "flow_fixed_chunks", "exact", "slab_97", "ragged", "period_log"]


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
    sub = np.arange(1024)
    p_sub, f_sub = p2.select(sub), f2.select(sub)
    ns_sub = _nsamples(L, p_sub)
    ragged = np.concatenate([[0], np.cumsum(ns_sub[:-1] + rng.integers(0, 300, 1023).astype(np.uint64))]).astype(np.uint64) + 3
    t10 = api.TractParams(4096, _preset_tracts(L), tract=np.arange(4096) % 10)
    t128 = api.TractParams(4096, _formant_tracts(L, 128), tract=(np.arange(4096) * 37) % 128)
    d = dict(mode=SYNTH, f=None, nsamp=None, offsets=None, log=False, chunk=0, exact=0, slab=0, out_dev=True)
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
    }


# total chunks and warm-up samples that vs_get_timing reports for these calls on a B200 (148 SMs), device output
PINNED = {"cfg2": (17614, 32765084), "cfg3_shard": (30310, 53758613), "cfg5_slice": (15967, 24523171)}


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    out = tmp_path_factory.mktemp("batch_plan") / "libbatch_plan_shim.so"
    subprocess.run(["g++", "-O3", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-o", str(out),
                    str(ROOT / "tests" / "tools" / "batch_plan_shim.cpp"), str(ROOT / "voice_synth_b200" / "csrc" / "vs_batch_plan.cpp")],
                   check=True)
    L = C.CDLL(str(out))
    L.shim_plan.restype = C.c_int
    L.shim_plan.argtypes = [C.c_int, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                            C.c_double, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_void_p]
    L.shim_fetch.restype = None
    L.vs_flow_max_periods.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p]
    return L


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
    info = np.zeros(8, dtype=np.uint64)
    rc = L.shim_plan(mode, n, fp, ff, ft, ptr(nsamp), ptr(offs), ptr(rec), float(s["chunk"]), s["exact"], s["slab"], SM_COUNT,
                     int(s["out_dev"]), OUT_BASE if s["out_dev"] else 0, info.ctypes.data)
    assert rc == 0, rc
    nc, nr, nsl, warm_total, flow_rows, group_rows, n_groups, n_warm = (int(v) for v in info)
    r = dict(warm_total=warm_total, flow_rows=bool(flow_rows), group_rows=group_rows, n_groups=n_groups,
             streams=np.zeros((n, 7), dtype=np.uint64), chunks=np.zeros((nc, 4), dtype=np.uint32),
             order=np.zeros(nr, dtype=np.uint32), slabs=np.zeros((nsl + 1, 4), dtype=np.uint64),
             cta_end=np.zeros((nsl, n_groups), dtype=np.uint32), cache=np.zeros(nsl, dtype=np.uint32),
             warm=np.zeros(n_warm, dtype=np.int32))
    L.shim_fetch(*(r[k].ctypes.data_as(C.c_void_p) for k in ("streams", "chunks", "order", "slabs", "cta_end", "cache", "warm")))
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


def test_batch_plan_shapes_listed(all_shapes):
    assert list(all_shapes) == SHAPES


def test_batch_plan_paths(shim, all_shapes):
    """the kernel forms the shapes are meant to reach"""
    sh = all_shapes
    assert plan(shim, sh["flow_cfg2"])["flow_rows"]
    assert not plan(shim, sh["flow_cfg3_shard"])["flow_rows"]          # glottal noise
    assert plan(shim, sh["tracts_128"])["group_rows"] == 128 and plan(shim, sh["cfg2"])["group_rows"] == 32
