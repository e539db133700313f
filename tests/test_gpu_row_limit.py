"""Rows at the longest length the ABI accepts: 2^31 - 1 samples of caller PCM for the vowel filter, and 2^31 - 128 samples of
flow (the most (float)fs * dur gives) for flowgen and synth.  Near the end of such a row a sample position plus a window
(render kernel, 120 or 168 samples) or a step (flow-rows kernel, 256 samples) passes 2^31; the kernels count those
bounds so that nothing wraps.

walk() restates, in exact integers, the windows and steps the kernels take down each chunk of a plan (the batch
planner through tests/tools/batch_plan_shim.cpp) and the samples each one stores.  It runs without a GPU, and picks the
row placements of the GPU tests: a placement whose last window or step crosses 2^31 for every kernel where one exists,
and one whose does not.  The render kernel's flow mode has none: a flow row ends at 2^31 - 128 at the latest and its
windows are 120 samples, so a window that holds a row sample ends at 2^31 - 8 at the latest.

The GPU tests compare against the oracle: the flow bit for bit over the whole row, filtered PCM on windows (the
reference filter from zero state, started 40 000 samples before each checked window: the first and last 2^20 samples,
+-4096 around chunk boundaries, seeded random windows), and guard bands around every output row."""
import numpy as np
import pytest

import test_batch_plan_host as BP

INT_MAX = 2**31 - 1
N_PCM, N_FLOW = BP.LIMIT_NSAMP, BP.LIMIT_FLOW_NSAMP
PERIOD = 160                        # BP.limit_flow_params(): 16 kHz, F0 = 100 Hz, no jitter
WIN = {BP.FLOW: 120, BP.SYNTH: 168, BP.FILTER: 120}
LEAD = 40000                        # reference filter start before a checked window
GUARD = 256                         # sentinel samples before and after an output row
SENTINEL = -32768                   # no filtered or flow sample takes this value (outputs are clipped to +-32767, flow >= DC)


def walk(chunks, mode, phase, flow_rows=False):
    """The windows (render kernel) or steps (flow-rows kernel) of every chunk (stream, emit_lo, emit_hi, gen_target) of
    a one-stream plan whose output row starts `phase` samples past a 16-byte (render) or 128-byte (flow rows) boundary.
    Asserts that the samples they store tile each chunk's [emit_lo, emit_hi) exactly once; returns the chunks whose
    last window or step ends at or past 2^31 (its end does not fit an int) as (chunk index, its start, its end)."""
    cross = []
    for c, (_, lo, hi, gt) in enumerate(np.asarray(chunks, dtype=np.int64).tolist()):
        if flow_rows:
            span, first = 256, lo - ((phase + lo) % 64)
            assert (phase + first) % 64 == 0
        else:
            # synth and flow start generating at the first sample of the period that holds gen_target
            nstart = gt if mode == BP.FILTER else gt - gt % PERIOD
            span, first = WIN[mode], nstart - ((phase + nstart) % 8)
            assert (phase + first) % 8 == 0 and first <= nstart <= lo
        assert first <= lo
        n = -(-(hi - first) // span)                              # windows / steps: the kernels' count
        starts = first + span * np.arange(n, dtype=np.int64)
        a = np.maximum(starts, lo)
        b = np.minimum(starts + span, hi)
        keep = b > a                                              # windows of the warm-up store nothing
        assert np.all(keep[np.argmax(keep):]), "no empty window after the first that stores"
        a, b = a[keep], b[keep]
        assert a[0] == lo and b[-1] == hi and np.all(b[:-1] == a[1:])
        if starts[-1] + span > INT_MAX:                           # the end of the last one does not fit an int
            cross.append((c, int(starts[-1]), int(starts[-1] + span)))
    return cross


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    return BP.build_shim(tmp_path_factory.mktemp("row_limit"))


@pytest.fixture(scope="module")
def limit_shapes(shim):
    return BP.shapes(shim)


# shape -> [(phase of the output row in samples, whether the last window or step of its last chunk ends past 2^31 - 1)]:
# the placements the GPU tests run.  A filter row of 2^31 - 1 samples crosses at every phase, a chunked synth row of
# 2^31 - 128 samples at none, an unchunked one at every phase but 0.  Rows in host memory are rendered into a 16-byte
# aligned device slab, so their kernel phase is 0 whatever the host address.
PLACEMENTS = {
    "limit_filter": [(0, True)],
    "limit_filter_chunk_2e27": [(0, True)],
    "limit_filter_no_chunks": [(0, True)],
    "limit_flow": [(0, True), (5, False)],
    "limit_flow_simple_gen": [(0, False)],
    "limit_flow_noise": [(0, False)],
    "limit_synth": [(0, False)],
    "limit_tracts_10_no_chunks": [(1, True)],
}


def test_walk_covers_every_limit_chunk_and_finds_the_crossings(shim, limit_shapes):
    for name in BP.SHAPES:
        if not name.startswith("limit"):
            continue
        s = limit_shapes[name]
        r = BP.plan(shim, s)
        ck = r["chunks"].astype(np.int64)
        found = {}
        for ph in range(64 if r["flow_rows"] else 8):
            cross = walk(ck, s["mode"], ph, r["flow_rows"])
            assert all(c == len(ck) - 1 for c, _, _ in cross), "only a row's last chunk reaches 2^31"
            found[ph] = bool(cross)
        for ph, crosses in PLACEMENTS.get(name, []):
            assert found[ph] == crosses, (name, ph)
        if name.startswith("limit_flow"):
            # the render kernel's flow windows on the same plan: none can cross (see above)
            assert not any(walk(ck, s["mode"], ph) for ph in range(8)), name


# ---------------------------------------------------------------------------------------------------------------------
# On the GPU.  Host memory at peak: one 4 GiB input row, one 4 GiB oracle flow and one 4 GiB copy of an output row.

SEG = 1000003                       # the filter input: a jittery voice of this many samples, repeated along the row


@pytest.fixture(scope="module")
def vs():
    from voice_synth_b200 import api
    return api


@pytest.fixture(scope="module")
def ctx(vs):
    c = vs.Context()
    yield c
    c.close()


@pytest.fixture(scope="module")
def pcm_in(oracle):
    par = oracle.flow_par_from_cli(["-o", "x", "-d", "70", "-f", "117", "-j", "2", "-s", "3", "-r", "16000"], 5)
    seg = oracle.flowgen(par)[:SEG]
    assert seg.size == SEG
    return np.resize(seg, N_PCM)


def _oracle_par(oracle, p):
    q = oracle.FlowPar()
    for k in ("dur", "jitter", "cq", "K", "F0", "DC", "noise", "Kvar", "shimmer"):
        setattr(q, k, float(getattr(p, k)[0]))
    q.fs, q.amp, q.seed = int(p.fs[0]), int(p.amp[0]), int(p.seed[0])
    q.has_jitter, q.has_shimmer, q.has_noise = [int(bool(p.flags[0] & b)) for b in (1, 2, 4)]
    return q


@pytest.fixture(scope="module")
def limit_flow(oracle):
    p = BP.limit_flow_params()
    f = oracle.flowgen(_oracle_par(oracle, p))
    assert f.size == N_FLOW
    return p, f


@pytest.fixture(scope="module")
def vowel_den(tmp_path_factory):
    from vowel_den_ref import VowelDen
    return VowelDen(tmp_path_factory.mktemp("vowel_den_limit"))


def _row_buffer(n, phase, dtype, fill):
    """a device buffer with the row at GUARD + phase, everything set to fill; (buffer, pointer to the row)"""
    import torch
    buf = torch.full((n + 2 * GUARD + 8,), fill, dtype=dtype, device="cuda")
    return buf, buf.data_ptr() + (GUARD + phase) * buf.element_size()


def _take_row(buf, n, phase, fill):
    """the row (a device view); asserts that both guard bands still hold fill and that every row sample was written"""
    import torch
    torch.cuda.synchronize()
    a, b = GUARD + phase, GUARD + phase + n
    assert bool((buf[:a] == fill).all()) and bool((buf[b:] == fill).all()), "a guard band was written"
    row = buf[a:b]
    assert int((row == fill).sum()) == 0, "samples of the row were never written"
    return row


def _windows(n, plan_chunks, seed, tail_boundaries=2**24):
    """the first and last 2^20 samples, +-4096 around the chunk boundaries (all of them in the row's last
    tail_boundaries samples, 64 seeded others), 64 seeded random windows of 4096: sorted, merged [a, b).  An auto plan
    has about 18 000 boundaries; with the reference started LEAD samples early, all of them would be about 870 M
    reference samples, some 50 s of one CPU core per call.  The boundaries near 2^31, where the positions wrapped,
    are all checked."""
    rng = np.random.default_rng(seed)
    w = [(0, 2**20), (n - 2**20, n)]
    bnd = np.asarray(plan_chunks, dtype=np.int64)[1:, 1]
    late = bnd[bnd >= n - tail_boundaries]
    early = bnd[bnd < n - tail_boundaries]
    if early.size:
        late = np.concatenate([late, rng.choice(early, min(64, early.size), replace=False)])
    w += [(max(0, int(x) - 4096), min(n, int(x) + 4096)) for x in late]
    w += [(int(a), int(a) + 4096) for a in rng.integers(0, n - 4096, 64)]
    w.sort()
    out = [list(w[0])]
    for a, b in w[1:]:
        if a <= out[-1][1]:
            out[-1][1] = max(out[-1][1], b)
        else:
            out.append([a, b])
    return out


def _check_windows(x, got, wins, ref, raw=None, exact=False, what=""):
    """got (int16 row) and raw (its pre-quantisation values) against ref(segment) -> (pcm, raw) on each window, the
    reference started LEAD samples before it from zero state"""
    for a, b in wins:
        s = max(0, a - LEAD)
        opcm, oraw = ref(x[s:b])
        opcm, oraw = opcm[a - s:], oraw[a - s:]
        d = np.abs(got[a:b].astype(np.int32) - opcm.astype(np.int32)).max()
        assert d <= (0 if exact else 1), f"{what}: PCM off by {d} in [{a}, {b})"
        if raw is not None:
            e = np.abs(raw[a:b].cpu().numpy() - oraw).max()
            assert e <= 1e-5, f"{what}: raw error {e} in [{a}, {b})"


def _filters(vs, oracle, vowel_den, kind):
    """(filter params, reference) of one voice: preset 'u', or the same vowel as a caller-defined tract"""
    if kind == "preset":
        return vs.FilterParams(1, preset="u"), lambda seg: oracle.vowel(seg, "u", want_raw=True)
    from voice_synth_b200 import workloads
    den = np.stack([vs.tract_from_preset(k) for k in workloads.PRESETS])
    t = workloads.PRESETS.index("u")
    return vs.TractParams(1, den, tract=[t]), lambda seg: vowel_den(seg, den[t], want_raw=True)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["preset", "tract"])
def test_filter_at_the_limit(ctx, vs, oracle, vowel_den, shim, limit_shapes, pcm_in, kind):
    """vs_vowel_filter_batch on one row of 2^31 - 1 samples: device buffers with raw output (auto chunks, the last window
    crosses 2^31), then pageable host buffers (2^27-sample chunks)"""
    import torch
    f, ref = _filters(vs, oracle, vowel_den, kind)
    ns = np.array([N_PCM], dtype=np.uint64)
    zero = np.zeros(1, dtype=np.uint64)
    (ph, crosses), = PLACEMENTS["limit_filter"]
    wins = _windows(N_PCM, BP.plan(shim, limit_shapes["limit_filter"])["chunks"], 11)
    ctx.set_option(vs.OPT_CHUNK_SAMPLES, 0)
    inb, inp = _row_buffer(N_PCM, ph, torch.int16, 0)
    inb[GUARD + ph: GUARD + ph + N_PCM].copy_(torch.from_numpy(pcm_in))
    outb, outp = _row_buffer(N_PCM, ph, torch.int16, SENTINEL)
    rawb, rawp = _row_buffer(N_PCM, ph, torch.float64, 1e300)
    ctx.vowel_filter_batch(inp, ns, f, in_offsets=zero, out=outp, out_offsets=zero, want_raw=rawp)
    raw = _take_row(rawb, N_PCM, ph, 1e300)
    got = _take_row(outb, N_PCM, ph, SENTINEL).cpu().numpy()
    del inb, outb
    _check_windows(pcm_in, got, wins, ref, raw=raw, what=f"{kind}, device, phase {ph}")
    del raw, rawb, got
    torch.cuda.empty_cache()

    # pageable host memory, 2^27-sample chunks
    wins = _windows(N_PCM, BP.plan(shim, limit_shapes["limit_filter_chunk_2e27"])["chunks"], 12)
    out = np.full(N_PCM + 2 * GUARD, SENTINEL, dtype=np.int16)
    ctx.set_option(vs.OPT_CHUNK_SAMPLES, 2**27)
    try:
        ctx.vowel_filter_batch(pcm_in, ns, f, out=out[GUARD:], out_offsets=zero)
    finally:
        ctx.set_option(vs.OPT_CHUNK_SAMPLES, 0)
    assert np.all(out[:GUARD] == SENTINEL) and np.all(out[GUARD + N_PCM:] == SENTINEL)
    got = out[GUARD: GUARD + N_PCM]
    assert not np.any(got == SENTINEL)
    _check_windows(pcm_in, got, wins, ref, what=f"{kind}, host, chunks of 2^27")


@pytest.mark.gpu
def test_filter_exact_unchunked_at_the_limit(ctx, vs, oracle, pcm_in):
    """exact mode never chunks: one lane walks all 2^31 - 1 samples, [blk0, hi) is longer than 2^31 - 8; bit for bit"""
    import torch
    f = vs.FilterParams(1, preset="u")
    ns = np.array([N_PCM], dtype=np.uint64)
    zero = np.zeros(1, dtype=np.uint64)
    (ph, _), = PLACEMENTS["limit_filter_no_chunks"]
    inb, inp = _row_buffer(N_PCM, ph, torch.int16, 0)
    inb[GUARD + ph: GUARD + ph + N_PCM].copy_(torch.from_numpy(pcm_in))
    outb, outp = _row_buffer(N_PCM, ph, torch.int16, SENTINEL)
    ctx.set_option(vs.OPT_EXACT_FILTER, 1)
    try:
        ctx.vowel_filter_batch(inp, ns, f, in_offsets=zero, out=outp, out_offsets=zero)
        got = _take_row(outb, N_PCM, ph, SENTINEL).cpu().numpy()
    finally:
        ctx.set_option(vs.OPT_EXACT_FILTER, 0)
    del inb, outb
    torch.cuda.empty_cache()
    wins = _windows(N_PCM, np.zeros((1, 4)), 13)
    _check_windows(pcm_in, got, wins, lambda seg: oracle.vowel(seg, "u", want_raw=True), exact=True, what="exact")


@pytest.mark.gpu
def test_flowgen_at_the_limit(ctx, vs, oracle, limit_flow):
    """vs_flowgen_batch on one voice of 2^31 - 128 samples, bit for bit with the oracle: the flow-rows kernel at a
    placement whose last step ends at 2^31 and at one whose does not, then the render kernel (VS_OPT_SIMPLE_GEN)"""
    import torch
    p, want = limit_flow
    zero = np.zeros(1, dtype=np.uint64)
    runs = [(ph, 0) for ph, _ in PLACEMENTS["limit_flow"]] + [(0, 1)]
    for ph, simple in runs:
        buf, ptr = _row_buffer(N_FLOW, ph, torch.int16, SENTINEL)
        ctx.set_option(vs.OPT_SIMPLE_GEN, simple)
        try:
            ctx.flowgen_batch(p, out=ptr, offsets=zero)
            got = _take_row(buf, N_FLOW, ph, SENTINEL).cpu().numpy()
            path = ctx.timing()["render_path"]
        finally:
            ctx.set_option(vs.OPT_SIMPLE_GEN, 0)
        del buf
        torch.cuda.empty_cache()
        assert bool(path & 32) == (not simple), path
        bad = np.flatnonzero(got != want)
        assert bad.size == 0, f"phase {ph}, simple {simple}: {bad.size} samples differ, first at {bad[0]}"
        del got


@pytest.mark.gpu
def test_flowgen_with_glottal_noise_at_the_limit(ctx, vs, oracle):
    """the lane-per-row generator with glottal noise on one voice of 2^31 - 128 samples, bit for bit"""
    import torch
    p = BP.limit_flow_params(noise=10.0)
    want = oracle.flowgen(_oracle_par(oracle, p))
    assert want.size == N_FLOW
    ph = 0
    buf, ptr = _row_buffer(N_FLOW, ph, torch.int16, SENTINEL)
    ctx.flowgen_batch(p, out=ptr, offsets=np.zeros(1, dtype=np.uint64))
    got = _take_row(buf, N_FLOW, ph, SENTINEL).cpu().numpy()
    del buf
    torch.cuda.empty_cache()
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, f"{bad.size} samples differ, first at {bad[0]}"


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["preset", "tract"])
def test_synth_at_the_limit(ctx, vs, oracle, vowel_den, shim, limit_shapes, limit_flow, kind):
    """vs_synth_batch on one voice of 2^31 - 128 samples against the reference filter of the oracle's flow: the preset
    in auto chunks, the tract unchunked at a phase where the last window crosses 2^31 (one lane walks the whole row)"""
    import torch
    p, flow = limit_flow
    f, ref = _filters(vs, oracle, vowel_den, kind)
    shape, chunk = ("limit_synth", 0) if kind == "preset" else ("limit_tracts_10_no_chunks", -1)
    (ph, _), = PLACEMENTS[shape]
    wins = _windows(N_FLOW, BP.plan(shim, limit_shapes[shape])["chunks"], 14)
    buf, ptr = _row_buffer(N_FLOW, ph, torch.int16, SENTINEL)
    ctx.set_option(vs.OPT_CHUNK_SAMPLES, chunk)
    try:
        ctx.synth_batch(p, f, out=ptr, offsets=np.zeros(1, dtype=np.uint64))
        got = _take_row(buf, N_FLOW, ph, SENTINEL).cpu().numpy()
    finally:
        ctx.set_option(vs.OPT_CHUNK_SAMPLES, 0)
    del buf
    torch.cuda.empty_cache()
    _check_windows(flow, got, wins, ref, what=f"synth {kind}, chunk option {chunk}, phase {ph}")


# ---- the calls on caller PCM: a strictly periodic row of 2^31 - 1 samples --------------------------------------------
# One period is PCM_T = 221 samples at 22050 Hz, the hop of the pitch and formant frames (lround(10 ms * 22050)), so
# every frame sees the same samples: the per-stream statistics are those of any one frame, the counts follow from the
# row length, and the flow analysis finds one cycle per period with no jitter and no shimmer.

PCM_FS, PCM_T, PCM_PEAK = 22050, 221, 12000


@pytest.fixture(scope="module")
def periodic(oracle):
    """(flow period, PCM period): a pulse that the trigger lo = hi = 0 finds once per period, and the preset 'a' on it
    in its steady state (the filter's response to the first periods has died out to below half a step)"""
    import report_ref
    cyc = report_ref.pulse_train([PCM_T], [PCM_PEAK])[:PCM_T]
    pcm = oracle.vowel(np.tile(cyc // 10, 400), "a")           # a tenth of the amplitude: no sample clips
    assert np.array_equal(pcm[-PCM_T:], pcm[-2 * PCM_T:-PCM_T])
    return cyc, pcm[-PCM_T:].copy()


def _periodic_row(period, n):
    """period repeated over n samples, on the device"""
    import torch
    return torch.from_numpy(np.resize(period, n)).cuda()


@pytest.mark.gpu
def test_flow_analysis_and_report_at_the_limit(ctx, vs, periodic):
    """vs_flow_analyze_batch and vs_flow_report_batch on a periodic flow row of 2^31 - 1 samples"""
    import report_ref
    cyc, _ = periodic
    row = _periodic_row(cyc, N_PCM)
    ns = [N_PCM]
    st = ctx.flow_analyze_batch(row, ns, fs=PCM_FS, lo=0, hi=0)[0]
    rep = ctx.flow_report_batch(row, ns, fs=PCM_FS, lo=0, hi=0)[0]
    del row
    onsets = -(-N_PCM // PCM_T)                              # one at the first sample of every period
    assert (int(st["onsets"]), int(st["cycles"]), int(st["flags"])) == (onsets, onsets - 1, 0)
    assert float(st["f0_hz"]) == np.float32(PCM_FS / PCM_T)
    assert (float(st["jitter_pct"]), float(st["shimmer_pct"])) == (0.0, 0.0)
    assert (float(st["mean_period"]), float(st["mean_peak"])) == (PCM_T, PCM_PEAK)
    assert rep["base"].tobytes() == st.tobytes()
    # the report's quotients of a periodic voice do not depend on its length: those of 64 periods
    short = report_ref.report(np.resize(cyc, 64 * PCM_T + 1), fs=PCM_FS)
    for k in report_ref.FIELDS:
        if k in ("base", "hnr_len"):
            continue
        w, g = short[k], float(rep[k])
        assert (np.isnan(g) and np.isnan(w)) or g == np.float32(w), (k, g, w)


def _tail(period, n, first, count):
    """samples [first, first + count) of period repeated over n samples"""
    return np.resize(np.roll(period, -(first % len(period))), min(count, n - first))


@pytest.mark.gpu
def test_pitch_at_the_limit(ctx, vs, periodic):
    """vs_pitch_batch on a periodic PCM row of 2^31 - 1 samples: the last 256 frame records against the restatement on
    the row's tail, the statistics against those of one frame"""
    import math
    import pitch_ref as pr
    _, per = periodic
    o = pr.opts_with()
    Nw, H, _, _ = pr.geometry(PCM_FS, o)
    assert H == PCM_T
    nf = pr.n_frames(N_PCM, Nw, H)
    st, frames = ctx.pitch_batch(_periodic_row(per, N_PCM), [N_PCM], fs=PCM_FS, want_frames=True)
    st, frames = st[0], frames[0]
    assert len(frames) == nf == int(st["frames"])
    f0 = nf - 256
    want, _ = pr.analyse(_tail(per, N_PCM, f0 * H, N_PCM), PCM_FS, o)
    assert len(want) == 256
    for j, (g, w) in enumerate(zip(frames[f0:], want)):
        assert w["margin"] > pr.MARGIN and w["flags"] == pr.VOICED, (j, w)
        assert int(g["flags"]) == w["flags"], (j, g, w)
        assert math.isclose(float(g["f0_hz"]), w["f0"], rel_tol=1e-6), (j, g["f0_hz"], w["f0"])
        assert math.isclose(float(g["strength"]), w["r"], rel_tol=1e-6), (j, g["strength"], w["r"])
        assert math.isclose(float(g["hnr_db"]), w["hnr"], rel_tol=1e-5, abs_tol=1e-3), (j, g["hnr_db"], w["hnr"])
    w = want[-1]
    assert (int(st["periodic"]), int(st["voiced"])) == (nf, nf)
    for k, v in (("f0_mean_hz", w["f0"]), ("f0_min_hz", w["f0"]), ("f0_max_hz", w["f0"]), ("strength_mean", w["r"])):
        assert math.isclose(float(st[k]), v, rel_tol=1e-6), (k, st[k], v)
    assert math.isclose(float(st["hnr_mean_db"]), w["hnr"], rel_tol=1e-5, abs_tol=1e-3)
    assert abs(float(st["f0_sd_hz"])) <= 1e-3 and abs(float(st["hnr_sd_db"])) <= 1e-3


@pytest.mark.gpu
def test_formants_at_the_limit(ctx, vs, periodic):
    """vs_formant_batch on a periodic PCM row of 2^31 - 1 samples: the last 256 frame records against the restatement
    on the row's tail (one frame more in front: a frame's pre-emphasis reads the sample before it), the statistics
    against those of one frame"""
    import math
    import formant_ref as fr
    _, per = periodic
    o = fr.opts_with()
    Nw, H = fr.geometry(PCM_FS, o)
    assert H == PCM_T
    nf = fr.n_frames(N_PCM, Nw, H)
    st, frames = ctx.formant_batch(_periodic_row(per, N_PCM), [N_PCM], fs=PCM_FS, want_frames=True)
    st, frames = st[0], frames[0]
    assert len(frames) == nf == int(st["frames"])
    f0 = nf - 256
    want, _ = fr.analyse(_tail(per, N_PCM, (f0 - 1) * H, N_PCM), PCM_FS, o)
    want = want[1:]
    assert len(want) == 256
    for j, (g, w) in enumerate(zip(frames[f0:], want)):
        assert not w["ambiguous"] and w["flags"] == 0, (j, w)
        assert int(g["flags"]) == 0 and int(g["found"]) == len(w["F"]), (j, g, w)
        for k in range(len(w["F"])):
            assert math.isclose(float(g["f_hz"][k]), w["F"][k], rel_tol=1e-6), (j, k, g["f_hz"][k], w["F"][k])
            assert math.isclose(float(g["bw_hz"][k]), w["B"][k], rel_tol=1e-5, abs_tol=1e-3), (j, k)
    w = want[-1]
    nk = min(len(w["F"]), int(o["n_formants"]))
    assert (int(st["analysed"]), int(st["unconverged"])) == (nf, 0)
    assert list(st["count"][:nk]) == [nf] * nk
    for k in range(nk):
        assert math.isclose(float(st["f_mean_hz"][k]), w["F"][k], rel_tol=1e-6), k
        assert math.isclose(float(st["bw_mean_hz"][k]), w["B"][k], rel_tol=1e-5, abs_tol=1e-3), k
        assert abs(float(st["f_sd_hz"][k])) <= 1e-2, k


@pytest.mark.gpu
def test_output_noise_at_the_limit(ctx, vs, oracle, periodic):
    """vs_vowel_noise_batch on a periodic PCM row of 2^31 - 1 samples, in place on the device: bit for bit the
    oracle's `vowel -n` noise over the whole row"""
    import torch
    _, per = periodic
    x = np.resize(per, N_PCM)
    buf, ptr = _row_buffer(N_PCM, 0, torch.int16, SENTINEL)
    buf[GUARD: GUARD + N_PCM].copy_(torch.from_numpy(x))
    ctx.vowel_noise_batch(ptr, [N_PCM], 20.0, [4000000007 % 2**32], fs=PCM_FS)
    torch.cuda.synchronize()
    assert bool((buf[:GUARD] == SENTINEL).all()) and bool((buf[GUARD + N_PCM:] == SENTINEL).all())
    got = buf[GUARD: GUARD + N_PCM].cpu().numpy()
    del buf
    torch.cuda.empty_cache()
    want = oracle.noise(x, 20.0, 4000000007 % 2**32, PCM_FS)
    del x
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, f"{bad.size} samples differ, first at {bad[0]}"
