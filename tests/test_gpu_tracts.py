"""Caller-defined vocal tracts on the GPU (vs_synth_batch_tract, vs_vowel_filter_batch_tract) against the preset calls
and the reference filter with the same denominator on the CPU (tests/tools/vowel_den.c).  Run on the B200 box: pytest -m gpu."""
import pathlib
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = pathlib.Path(__file__).resolve().parents[1]
PRESETS = "aiu1234567"


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
def vowel_den(tmp_path_factory):
    """the reference filter with any denominator (tests/tools/vowel_den.c)"""
    from vowel_den_ref import VowelDen
    return VowelDen(tmp_path_factory.mktemp("vowel_den"))


@pytest.fixture(autouse=True)
def _defaults(ctx, vs):
    yield
    ctx.set_option(vs.OPT_CHUNK_SAMPLES, 0)
    ctx.set_option(vs.OPT_EXACT_FILTER, 0)
    ctx.set_option(vs.OPT_SLAB_STREAMS, 0)
    ctx.set_option(vs.OPT_ASYNC_HOST, 0)


def _as_tracts(vs, f):
    """FilterParams -> TractParams holding the ten preset tables as tracts 0..9"""
    den = np.stack([vs.tract_from_preset(k) for k in PRESETS])
    idx = np.array([PRESETS.index(chr(c)) for c in f.preset], dtype=np.uint8)
    t = vs.TractParams(f.n, den, tract=idx)
    t.gain[...] = f.gain
    t.pre[...] = f.pre
    return t


def _rows(buf, offs, ns, i):
    return buf[int(offs[i]): int(offs[i]) + int(ns[i])]


def _check_ref(vowel_den, flow, foffs, ns, t, pcm, offs, raw=None, exact=False, streams=None):
    for i in (range(len(ns)) if streams is None else streams):
        x = _rows(flow, foffs, ns, i)
        want, wraw = vowel_den(x, t.den[t.tract[i]], float(t.gain[i]), float(t.pre[i]), want_raw=True)
        got = _rows(pcm, offs, ns, i)
        if exact:
            assert np.array_equal(got, want), i
        else:
            assert np.abs(got.astype(np.int32) - want.astype(np.int32)).max() <= 1, i
        if raw is not None:
            assert np.abs(_rows(raw, offs, ns, i) - wraw).max() <= 1e-5, i


def _batches(vs):
    from voice_synth_b200 import workloads as W
    p2, f2 = W.cfg2(n=1024, dur=0.5)
    p3, f3 = W.cfg3(n=160, dur=0.4)
    return [("cfg2", p2, f2), ("cfg3", p3, f3)]


def test_presets_as_tracts_are_the_preset_path(ctx, vs, vowel_den):
    for name, p, f in _batches(vs):
        t = _as_tracts(vs, f)
        flow, foffs, ns = ctx.flowgen_batch(p)
        for chunk in (-1, 4096):
            ctx.set_option(vs.OPT_CHUNK_SAMPLES, chunk)
            for raw in (False, True):
                a = ctx.synth_batch(p, f, want_raw=raw)
                b = ctx.synth_batch(p, t, want_raw=raw)
                assert ctx.timing()["render_path"] & 64
                assert np.array_equal(a[0], b[0]), (name, chunk, raw)
                if raw:
                    assert np.array_equal(a[3], b[3]), (name, chunk)
                a = ctx.vowel_filter_batch(flow, ns, f, in_offsets=foffs, want_raw=raw)
                b = ctx.vowel_filter_batch(flow, ns, t, in_offsets=foffs, want_raw=raw)
                assert np.array_equal(a[0], b[0]), (name, "filter", chunk, raw)
                if raw:
                    assert np.array_equal(a[2], b[2]), (name, "filter", chunk)
        ctx.set_option(vs.OPT_CHUNK_SAMPLES, 0)
        ctx.set_option(vs.OPT_EXACT_FILTER, 1)
        a = ctx.synth_batch(p, f, want_raw=True)
        b = ctx.synth_batch(p, t, want_raw=True)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[3], b[3]), (name, "exact")
        ctx.set_option(vs.OPT_EXACT_FILTER, 0)
        # auto chunking: tract groups are padded to whole CTAs, so the plan may differ from the preset call's
        a = ctx.synth_batch(p, f)
        b, offs, _, raw = ctx.synth_batch(p, t, want_raw=True)
        assert np.abs(a[0].astype(np.int32) - b.astype(np.int32)).max() <= 1, name
        _check_ref(vowel_den, flow, foffs, ns, t, b, offs, raw)


def _random_pole_tract(rng, rmax):
    den = np.array([1.0])
    for _ in range(11):
        r = rng.uniform(0.3, rmax)
        th = rng.uniform(0.05, np.pi - 0.05)
        den = np.convolve(den, [1.0, -2.0 * r * np.cos(th), r * r])
    return den


def _l1(den, n=30000):
    from scipy.signal import lfilter
    x = np.zeros(n)
    x[0] = 1.0
    return np.abs(lfilter([1.0], den, x)).sum()


def _custom_batch(vs, rng, n_tracts, per_tract, dur=0.3):
    """random formant tracts at three rates plus random-pole order-22 tracts; each voice at its tract's rate, gain
    chosen so that |raw| stays below 2.5e5"""
    dens, rates = [], []
    for k in range(n_tracts):
        if k % 4 == 3:
            dens.append(_random_pole_tract(rng, 0.995))
            rates.append(22050)
        else:
            fs = (11025, 22050, 44100)[k % 3]
            nf = int(rng.integers(2, 12))
            freqs = np.sort(rng.uniform(200.0, 0.45 * fs, nf))
            # 30-400 Hz at 22 050 Hz, the same pole radii at the other rates (30 Hz at 44 100 Hz is a radius of
            # 0.9979: a warm-up above the library's bound)
            dens.append(vs.tract_from_formants(freqs, rng.uniform(30.0, 400.0, nf) * (fs / 22050.0), fs))
            rates.append(fs)
    den = np.stack(dens)
    counts = per_tract if np.ndim(per_tract) else [per_tract] * n_tracts
    idx = np.concatenate([np.full(c, k, dtype=np.uint8) for k, c in enumerate(counts)])
    rng.shuffle(idx)
    n = idx.size
    p = vs.FlowParams(n, dur=dur)
    p.fs[...] = np.array(rates)[idx]
    p.F0[...] = rng.uniform(90.0, 220.0, n).astype(np.float32)
    p.jitter[...] = 0.01
    p.shimmer[...] = 0.03
    p.flags[...] = vs.VS_F_JITTER | vs.VS_F_SHIMMER
    p.seed[...] = np.arange(n) + 7
    l1 = np.array([_l1(d) for d in den])
    gain = np.minimum(10.0, 2.5e5 / (l1[idx] * 1.8 * 12000.0)).astype(np.float32)
    t = vs.TractParams(n, den, tract=idx, pre=1.0)
    t.gain[...] = gain
    return p, t


def test_custom_tracts_against_the_reference_filter(ctx, vs, vowel_den):
    rng = np.random.default_rng(2024)
    p, t = _custom_batch(vs, rng, 16, 6)
    flow, foffs, ns = ctx.flowgen_batch(p)
    n_max = int(ns.max())
    for chunks in (1, 2, 5):
        ctx.set_option(vs.OPT_CHUNK_SAMPLES, -1 if chunks == 1 else (n_max + chunks - 1) // chunks)
        pcm, offs, _, raw = ctx.synth_batch(p, t, want_raw=True)
        _check_ref(vowel_den, flow, foffs, ns, t, pcm, offs, raw)
        pcm2, offs2 = ctx.synth_batch(p, t)[:2]
        _check_ref(vowel_den, flow, foffs, ns, t, pcm2, offs2)
        fpcm, fo, fraw = ctx.vowel_filter_batch(flow, ns, t, in_offsets=foffs, want_raw=True)
        _check_ref(vowel_den, flow, foffs, ns, t, fpcm, fo, fraw)
    ctx.set_option(vs.OPT_CHUNK_SAMPLES, 0)
    ctx.set_option(vs.OPT_EXACT_FILTER, 1)
    pcm, offs, _ = ctx.synth_batch(p, t)
    _check_ref(vowel_den, flow, foffs, ns, t, pcm, offs, exact=True)
    fpcm, fo = ctx.vowel_filter_batch(flow, ns, t, in_offsets=foffs)
    _check_ref(vowel_den, flow, foffs, ns, t, fpcm, fo, exact=True)


def test_128_tracts_in_one_call(ctx, vs, vowel_den):
    rng = np.random.default_rng(128)
    counts = rng.integers(1, 61, 128)
    p, t = _custom_batch(vs, rng, 128, counts, dur=0.15)
    flow, foffs, ns = ctx.flowgen_batch(p)
    # exact mode: every stream must equal the reference filter bit for bit, so a stream filtered with another group's tract
    # cannot pass.  (In the FMA mode some of these random order-22 direct-form tracts amplify the rounding
    # difference between fused and unfused products past 1e-5 within a few thousand samples -- DESIGN.md 4.6.)
    ctx.set_option(vs.OPT_EXACT_FILTER, 1)
    pcm, offs, _ = ctx.synth_batch(p, t)
    _check_ref(vowel_den, flow, foffs, ns, t, pcm, offs, exact=True)
    ctx.set_option(vs.OPT_EXACT_FILTER, 0)
    too_many = vs.TractParams(p.n, np.concatenate([t.den, t.den[:1]]), tract=t.tract)
    with pytest.raises(vs.VsError) as e:
        ctx.synth_batch(p, too_many)
    assert e.value.code == vs.VS_EINVAL
    few = vs.TractParams(p.n, t.den[:100], tract=t.tract)          # indices up to 127 >= n_tracts
    with pytest.raises(vs.VsError) as e:
        ctx.synth_batch(p, few)
    assert e.value.code == vs.VS_EINVAL


def test_refusals(ctx, vs):
    p = vs.FlowParams(2, dur=0.1)
    good = vs.tract_from_preset("a")

    def pole_tract(r):
        den = np.zeros(23)
        den[:3] = [1.0, -2.0 * r * np.cos(0.3), r * r]
        return den

    bad_a0 = good.copy()
    bad_a0[0] = 2.0
    nan = good.copy()
    nan[5] = np.nan
    for den in (bad_a0, nan, pole_tract(1.01), pole_tract(0.9995)):
        with pytest.raises(vs.VsError) as e:
            ctx.synth_batch(p, vs.TractParams(2, np.stack([good, den]), tract=[0, 0]))
        assert e.value.code == vs.VS_ERANGE
    ctx.synth_batch(p, vs.TractParams(2, np.stack([good, pole_tract(0.99)]), tract=[0, 1]))
    with pytest.raises(vs.VsError) as e:
        ctx.synth_batch(p, vs.FilterParams(2, "x"))
    assert e.value.code == vs.VS_EPRESET


def test_same_flow_different_coefficients(ctx, vs, vowel_den):
    """the same-inputs fast path must notice a change of den alone"""
    rng = np.random.default_rng(5)
    p, t = _custom_batch(vs, rng, 4, 8)
    flow, foffs, ns = ctx.flowgen_batch(p)
    t2 = vs.TractParams(p.n, t.den[::-1].copy(), tract=t.tract)
    t2.gain[...] = np.minimum(t.gain, 0.05)
    for tt in (t, t2, t):
        pcm, offs, _ = ctx.synth_batch(p, tt)
        _check_ref(vowel_den, flow, foffs, ns, tt, pcm, offs)


def test_pipeline_device_buffers_pinned_and_two_devices(ctx, vs):
    import torch
    from voice_synth_b200 import workloads as W
    p, f = W.cfg2(n=512, dur=0.4)
    rng = np.random.default_rng(9)
    pc, tc = _custom_batch(vs, rng, 24, 20, dur=0.4)
    calls = [(p, f), (pc, tc), (p, _as_tracts(vs, f)), (pc, tc), (p, f), (pc, tc)]
    alone = [ctx.synth_batch(pp, ff)[:3] for pp, ff in calls]
    outs = []
    for (pp, ff), (ref, offs, ns) in zip(calls, alone):
        d = torch.zeros(ref.size, dtype=torch.int16, device="cuda")
        ctx.synth_batch(pp, ff, out=d)
        outs.append(d)
    ctx.sync()
    for d, (ref, _, _) in zip(outs, alone):
        assert np.array_equal(d.cpu().numpy(), ref)
    # pinned host output, small slabs, asynchronous return
    ctx.set_option(vs.OPT_SLAB_STREAMS, 97)
    ctx.set_option(vs.OPT_ASYNC_HOST, 1)
    pins = []
    for (pp, ff), (ref, _, _) in zip(calls, alone):
        buf = torch.zeros(ref.size, dtype=torch.int16).pin_memory()
        ctx.synth_batch(pp, ff, out=buf.numpy())
        pins.append(buf)
    ctx.sync()
    for buf, (ref, _, _) in zip(pins, alone):
        assert np.array_equal(buf.numpy(), ref)
    if torch.cuda.device_count() >= 2:
        c2 = vs.Context(devices=[0, 1])
        try:
            for (pp, ff), (ref, _, _) in zip(calls, alone):
                assert np.array_equal(c2.synth_batch(pp, ff)[0], ref)
        finally:
            c2.close()


def test_batch_driver_with_formant_voices(ctx, vs, tmp_path):
    tools = ROOT / "host" / "bin"
    specs = [("a", 22050), ("f:700/80,1220/90,2600/120", 22050), ("i", 44100), ("f:700/80,1220/90,2600/120", 44100),
             ("f:300/60,2300/100,3000/150,3500/200", 44100), ("u", 22050), ("f:700/80,1220/90,2600/120", 22050)]
    lines = []
    for i, (v, fs) in enumerate(specs):
        rate = f" -r {fs}" if fs != 22050 else ""
        lines.append(f"{tmp_path}/v{i}.wav {v} {100 + i} -d 0.5 -f {110 + 7 * i} -g 200 -j 1 -s 2{rate}")
    m = tmp_path / "manifest.txt"
    m.write_text("\n".join(lines) + "\n")
    r = subprocess.run([str(tools / "vs_batch"), "-m", str(m)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr + r.stdout
    # the same voices through the Python tract call
    p = vs.FlowParams.from_cli([ln.split(maxsplit=3)[3] for ln in lines], [100 + i for i in range(len(specs))])
    keys = sorted(set(specs), key=specs.index)
    dens = []
    for v, fs in keys:
        if v.startswith("f:"):
            fb = [tuple(map(float, x.split("/"))) for x in v[2:].split(",")]
            dens.append(vs.tract_from_formants([a for a, _ in fb], [b for _, b in fb], fs))
        else:
            dens.append(vs.tract_from_preset(v))
    t = vs.TractParams(len(specs), np.stack(dens), tract=[keys.index(s) for s in specs])
    pcm, offs, ns = ctx.synth_batch(p, t)
    for i in range(len(specs)):
        data = (tmp_path / f"v{i}.wav").read_bytes()
        payload = np.frombuffer(data[data.index(b"data") + 8:], dtype="<i2")
        assert np.array_equal(payload, _rows(pcm, offs, ns, i)), i
    # more than 128 distinct tracts in a slab: refused, naming the line
    many = [f"{tmp_path}/w{i}.wav f:{300 + i}/80,{1500 + i}/100 {i} -d 0.5" for i in range(130)]
    m.write_text("\n".join(many) + "\n")
    r = subprocess.run([str(tools / "vs_batch"), "-m", str(m)], capture_output=True, text=True)
    assert r.returncode != 0 and "line 129" in r.stderr, r.stderr
