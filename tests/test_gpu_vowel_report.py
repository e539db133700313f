"""vs_vowel_report_batch on the GPU against the numpy restatement (tests/vowel_report_ref.py) fed the GPU's own pitch frame
records (vs_pitch_batch with the same options): the voiced run and every mark exactly, the report fields with the
tolerances of test_gpu_report.py.  Presets with glottal and output noise, tract voices at 22 050 and 44 100 Hz, the pitch
option extremes, the synthetic rows of the host test, ragged, empty, short and odd-offset rows, host and device input,
marks NULL and mark_offsets, the error codes, the slot bound at the extreme f_max, a periodic row of 2^31 - 1 samples and
`acoustic -V`."""
import ctypes as C
import math
import pathlib
import subprocess
import wave

import numpy as np
import pytest

import report_ref as rr
import vowel_report_ref as vr
from test_gpu_pitch import OPTS, PRESETS, TRACTS, _flow_params, _ragged, _rows
from test_vowel_report_host import synthetic_rows

pytestmark = pytest.mark.gpu
ROOT = pathlib.Path(__file__).resolve().parents[1]


@pytest.fixture(scope="module")
def vs():
    from voice_synth_b200 import api
    return api


@pytest.fixture(scope="module")
def ctx(vs):
    c = vs.Context()
    yield c
    c.close()


def _close(g, w, rel):
    if math.isnan(w):
        return math.isnan(g)
    if math.isinf(w):
        return g == w
    return math.isclose(g, float(np.float32(w)), rel_tol=rel, abs_tol=1e-30)


def _check_report(got, want, what):
    """the report_ref fields of one stream, as test_gpu_report.py compares them"""
    b = got["rep"]["base"]
    assert (int(b["onsets"]), int(b["cycles"]), int(b["flags"])) == (want["base"]["onsets"], want["base"]["cycles"], 0), what
    for k in ("f0_hz", "jitter_pct", "shimmer_pct", "mean_period", "mean_peak"):
        assert math.isclose(float(b[k]), float(np.float32(want["base"][k])), rel_tol=2e-6, abs_tol=1e-30), (what, k, b[k], want["base"][k])
    assert int(got["rep"]["hnr_len"]) == want["hnr_len"] and int(got["rep"]["reserved"]) == 0, what
    for k in rr.FIELDS:
        g, w = float(got["rep"][k]), want[k]
        rel = 1e-5 if k == "shimmer_db" else 2e-6
        ok = _close(g, w, rel) or (k == "hnr_db" and abs(g - w) <= 1e-6)
        assert ok, (what, k, g, w)


def _analyse(ctx, pcm, ns, offsets=None, fs=None, opts=None, what=""):
    """the call from host and device input (byte-identical), with and without marks (the same records); every stream
    against the restatement on the frames of vs_pitch_batch.  Returns the records, the marks and the frame records."""
    import torch
    out, marks = ctx.vowel_report_batch(pcm, ns, offsets=offsets, fs=fs, opts=opts, want_marks=True)
    dev, dev_marks = ctx.vowel_report_batch(torch.from_numpy(pcm).cuda(), ns, offsets=offsets, fs=fs, opts=opts, want_marks=True)
    assert out.tobytes() == dev.tobytes() and all(np.array_equal(a, b) for a, b in zip(marks, dev_marks)), what
    assert ctx.vowel_report_batch(pcm, ns, offsets=offsets, fs=fs, opts=opts).tobytes() == out.tobytes(), what
    _, frames = ctx.pitch_batch(pcm, ns, offsets=offsets, fs=fs, opts=opts, want_frames=True)
    slots = vs_slots(ns, fs, opts)
    o = vr.pr.opts_with(**(opts or {}))
    offs = offsets if offsets is not None else np.arange(len(ns), dtype=np.uint64) * (int(max(ns)) if len(ns) else 0)
    for i in range(len(ns)):
        rate = int(np.broadcast_to(fs, (len(ns),))[i]) if fs is not None else 22050
        x = pcm[int(offs[i]): int(offs[i]) + int(ns[i])]
        mk, rn = vr.marks(x, frames[i]["flags"], frames[i]["f0_hz"], rate, o)
        assert (int(out[i]["run_frame"]), int(out[i]["run_frames"]), int(out[i]["run_start"]), int(out[i]["run_len"])) == rn, (what, i)
        assert list(map(int, marks[i])) == mk, (what, i)
        assert len(mk) <= slots[i], (what, i)
        _check_report(out[i], vr.report_on_marks(x, mk, rate), (what, i))
    return out, marks, frames


def vs_slots(ns, fs, opts):
    from voice_synth_b200 import api
    return api.vowel_mark_slots(ns, fs, opts)


@pytest.mark.parametrize("noise", ["glottal", "output"])
def test_presets_match_restatement(ctx, vs, noise):
    n = 20
    p = _flow_params(vs, n, 31, noise=noise == "glottal")
    pcm, offs, ns = ctx.synth_batch(p, vs.FilterParams(n, "".join(PRESETS[i % 10] for i in range(n))))
    if noise == "output":
        snr = np.array([(10.0, 20.0, 0.0)[i % 3] for i in range(n)], dtype=np.float32)
        ctx.vowel_noise_batch(pcm, ns, snr, np.arange(n) + 5, offsets=offs)
    out, _, _ = _analyse(ctx, pcm, ns, offsets=offs, what=noise)
    assert (out["rep"]["base"]["cycles"] > 50).sum() >= n - 2        # a noisy voice may keep only a short voiced run


@pytest.mark.parametrize("fs", [22050, 44100])
def test_tract_voices_match_restatement(ctx, vs, fs):
    n = 9
    p = _flow_params(vs, n, fs + 5, noise=True, fs=fs)
    den = np.stack([vs.tract_from_formants(*TRACTS[v], fs) for v in "aiu"])
    pcm, offs, ns = ctx.synth_batch(p, vs.TractParams(n, den, tract=np.arange(n) % 3, gain=1.5))
    _analyse(ctx, pcm, ns, offsets=offs, fs=p.fs, what=fs)


@pytest.mark.parametrize("opts", OPTS, ids=["50-1000Hz", "periods2", "periods6", "octave0", "voicing0", "voicing0.9", "harmonicity"])
def test_option_extremes_match_restatement(ctx, vs, opts):
    n = 6
    p = _flow_params(vs, n, 23, noise=True)
    p.fs[3:] = 44100
    pcm, offs, ns = ctx.synth_batch(p, vs.FilterParams(n, PRESETS[:n]))
    ctx.vowel_noise_batch(pcm, ns, np.where(np.arange(n) % 2 == 1, 15.0, 0.0), np.arange(n), offsets=offs, fs=p.fs)
    _analyse(ctx, pcm, ns, offsets=offs, fs=p.fs, opts=opts, what=opts)


def test_synthetic_rows(ctx, vs):
    """the host test's rows: a repeated waveform (equal spacing), a known period sequence, silence, two voiced stretches"""
    rows, _ = synthetic_rows()
    pcm, offs, ns = _ragged(rows, np.random.default_rng(4))
    out, marks, _ = _analyse(ctx, pcm, ns, offsets=offs, what="synthetic")
    assert set(np.diff(marks[0]).tolist()) == {147}
    assert out[2]["run_frames"] == 0 and out[2]["rep"]["base"]["onsets"] == 0


def test_ragged_empty_short_odd_offsets_and_mark_offsets(ctx, vs):
    """rows of 0, 1, Nw - 1, Nw and Nw + 1 samples among voices, at odd offsets with non-silent gaps; marks NULL gives the
    same records, and mark_offsets places each stream's marks where the caller asks"""
    p = _flow_params(vs, 4, 41)
    voice, voffs, vns = ctx.synth_batch(p, vs.FilterParams(4, "a3iu"))
    v = _rows(voice, voffs, vns)
    rows = [v[0], np.zeros(0, np.int16), v[1][:1], v[2][:881], v[3][:882], v[1][:883], v[2], v[3][:5000]]
    pcm, offs, ns = _ragged(rows, np.random.default_rng(9))
    out, marks, _ = _analyse(ctx, pcm, ns, offsets=offs, what="ragged")
    assert [int(out[i]["rep"]["base"]["onsets"]) for i in (1, 2, 3)] == [0, 0, 0]
    # mark_offsets: stream i at a place of the caller's choosing, a guard value everywhere else
    slots = vs.vowel_mark_slots(ns)
    mo = np.concatenate([[5], 5 + np.cumsum(slots[:-1] + 3)]).astype(np.uint64)
    buf = np.full(int(mo[-1] + slots[-1] + 7), 0xdeadbeef, dtype=np.uint32)
    rec = np.zeros(len(ns), dtype=vs.VOWEL_REPORT_DTYPE)
    ns64 = np.ascontiguousarray(ns, dtype=np.uint64)
    rc = ctx.L.vs_vowel_report_batch(ctx.h, pcm.ctypes.data, offs.ctypes.data, ns64.ctypes.data, None, len(ns), None,
                                     rec.ctypes.data, buf.ctypes.data, mo.ctypes.data)
    assert rc == 0 and rec.tobytes() == out.tobytes()
    used = np.zeros(len(buf), bool)
    for i in range(len(ns)):
        k = len(marks[i])
        assert np.array_equal(buf[int(mo[i]): int(mo[i]) + k], marks[i])
        used[int(mo[i]): int(mo[i]) + k] = True
    assert (buf[~used] == 0xdeadbeef).all()


def test_vowel_report_errors(ctx, vs):
    """NULL arguments, then the errors of vs_pitch_batch in the header's order; n = 0 is a no-op"""
    L, h = ctx.L, ctx.h
    pcm = np.zeros(5000, np.int16)
    ns = np.array([5000], np.uint64)
    rec = np.zeros(1, vs.VOWEL_REPORT_DTYPE)
    call = lambda c=h, x=pcm.ctypes.data, n=ns.ctypes.data, o=rec.ctypes.data, fs=None, opts=None, cnt=1: \
        L.vs_vowel_report_batch(c, x, None, n, fs, cnt, opts, o, None, None)
    assert call(c=None) == vs.VS_EINVAL
    assert call(x=None) == vs.VS_EINVAL
    assert call(n=None) == vs.VS_EINVAL
    assert call(o=None) == vs.VS_EINVAL
    bad = vs.pitch_opts(dict(f_min_hz=0.0))
    assert call(opts=C.byref(bad)) == vs.VS_ERANGE
    fs0 = np.array([0], np.int32)
    assert call(fs=fs0.ctypes.data) == vs.VS_ERANGE
    big = np.array([2 ** 31], np.uint64)
    assert call(n=big.ctypes.data) == vs.VS_EOVERLAP
    assert call(cnt=0) == vs.VS_OK
    for o in (dict(f_min_hz=0.0), dict(periods=1.0), dict(voicing_threshold=2.0)):
        with pytest.raises(vs.VsError) as e:
            ctx.vowel_report_batch(pcm, ns, opts=o)
        with pytest.raises(vs.VsError) as e2:
            ctx.pitch_batch(pcm, ns, opts=o)
        assert e.value.args == e2.value.args


@pytest.mark.parametrize("fs", [8000, 22050, 44100])
def test_slot_bound_at_the_extreme_f_max(ctx, vs, fs):
    """f_max at and above fs / 2 (tau_lo = 2: one slot per sample) and just below it, on voices, noise and a row whose
    pitch sits at the shortest lag: the marks stay within their slots, so VS_STATS_OVERFLOW never appears"""
    rng = np.random.default_rng(fs)
    t = np.arange(fs)
    rows = [np.round(9000 * np.sin(2 * np.pi * t / 2.5) + 3000 * np.sin(2 * np.pi * t / 7.0)).astype(np.int16),
            rng.integers(-8000, 8000, fs).astype(np.int16),
            np.round(12000 * np.sin(2 * np.pi * t * 0.37)).astype(np.int16)]
    p = _flow_params(vs, 2, fs, fs=fs)
    voice, voffs, vns = ctx.synth_batch(p, vs.FilterParams(2, "i5"))
    rows += _rows(voice, voffs, vns)
    pcm, offs, ns = _ragged(rows, rng)
    rate = np.full(len(ns), fs, np.int32)
    for o in (dict(f_max_hz=fs / 2.0, voicing_threshold=0.0), dict(f_max_hz=float(fs), voicing_threshold=0.0),
              dict(f_max_hz=fs / 3.0)):
        slots = vs.vowel_mark_slots(ns, rate, o)
        out, marks, _ = _analyse(ctx, pcm, ns, offsets=offs, fs=rate, opts=o, what=(fs, o))
        assert (out["rep"]["base"]["flags"] == 0).all()
        assert all(len(m) <= s for m, s in zip(marks, slots))


# ---- a periodic row of 2^31 - 1 samples -------------------------------------------------------------------------------
N_LIMIT = 2 ** 31 - 1
P_LIMIT = 147


@pytest.fixture(scope="module")
def limit_period():
    """one period of a vowel-like waveform with a single largest sample"""
    t = np.arange(P_LIMIT)
    w = 9000 * np.sin(2 * np.pi * t / P_LIMIT) + 5000 * np.sin(6 * np.pi * t / P_LIMIT + 1.0) + 2500 * np.sin(10 * np.pi * t / P_LIMIT)
    w = np.round(w).astype(np.int16)
    assert (np.abs(w.astype(int)) == np.abs(w.astype(int)).max()).sum() == 1
    return w


def test_periodic_row_at_the_limit(ctx, vs, limit_period):
    """marks over the whole row in closed form (m_k = m_0 + k P), the last ones against the restatement's walk on the
    row's tail with the GPU's frame records, the run over every frame, and the report of equal periods"""
    import torch
    blk = P_LIMIT * ((1 << 22) // P_LIMIT)
    row = torch.from_numpy(np.resize(limit_period, blk)).cuda().repeat(N_LIMIT // blk + 1)[:N_LIMIT].contiguous()
    ns = [N_LIMIT]
    out, marks = ctx.vowel_report_batch(row, ns, want_marks=True)
    _, frames = ctx.pitch_batch(row, ns, want_frames=True)
    del row
    out, mk, frames = out[0], marks[0].astype(np.int64), frames[0]
    Nw, H, _, _ = vr.pr.geometry(22050, vr.pr.DEFAULTS)
    nf = len(frames)
    assert (frames["flags"] == vr.pr.VOICED).all()
    assert (int(out["run_frame"]), int(out["run_frames"]), int(out["run_start"]), int(out["run_len"])) == (0, nf, 0, (nf - 1) * H + Nw)
    e = (nf - 1) * H + Nw
    a0 = Nw // 2 - P_LIMIT // 2                              # the anchor's period, around the first frame's centre
    m0 = a0 + (int(np.argmax(np.abs(limit_period.astype(int)))) - a0) % P_LIMIT
    K = len(mk)
    assert K == int(out["rep"]["base"]["onsets"]) and K <= vs.vowel_mark_slots(ns)[0]
    assert int(out["rep"]["base"]["flags"]) == 0
    # every mark one period after the last, up to the last whose candidates all fit in the run
    assert mk[0] == m0 and (np.diff(mk) == P_LIMIT).all()
    assert mk[-1] + vr.lround(1.25 * 22050.0 / float(frames["f0_hz"][-1])) + P_LIMIT > e - 2 * P_LIMIT
    # the tail: the restatement's walk from mark K-4 over the samples that follow
    base = int(mk[-4]) - 16
    tail = np.resize(np.roll(limit_period, -(base % P_LIMIT)), e - base).astype(np.int64)
    f0 = frames["f0_hz"]

    def period(t):
        f = (t + base - Nw // 2 + H // 2) // H
        return 22050.0 / float(f0[min(max(f, 0), nf - 1)])

    want = vr.walk(tail, int(mk[-4]) - base, e - base, period)
    assert [int(m) + base for m in want] == list(map(int, mk[-4:]))
    # equal periods but perhaps the last: mean period and peak from the marks
    T = np.diff(mk)
    assert float(out["rep"]["base"]["mean_period"]) == np.float32(T.sum() / (K - 1))
    assert float(out["rep"]["base"]["mean_peak"]) == np.float32(limit_period.max())


def _write_wav(path, x, fs):
    with wave.open(str(path), "wb") as w:
        w.setnchannels(1)
        w.setsampwidth(2)
        w.setframerate(fs)
        w.writeframes(np.ascontiguousarray(x, dtype="<i2").tobytes())


def test_acoustic_vowel_report_lines(ctx, vs, tmp_path):
    """host/bin/acoustic -V: one line per file, the columns of -x and the run, from vs_vowel_report_batch"""
    bins = ROOT / "host" / "bin"
    if not (bins / "acoustic").exists():
        subprocess.run(["make", "-s", "-C", str(ROOT), "host"], check=True)
    p = vs.FlowParams.from_cli([f"-d 1 -f {f0} -g {f0 + 30} -j 1 -s 3 -a 6000" for f0 in (100, 150, 200)], [7, 8, 9])
    p.fs[2] = 44100
    pcm, offs, ns = ctx.synth_batch(p, vs.FilterParams(3, "ai3"))
    rows = _rows(pcm, offs, ns)
    files = []
    for i, x in enumerate(rows):
        files.append(tmp_path / f"v{i}.wav")
        _write_wav(files[-1], x, int(p.fs[i]))
    r = subprocess.run([str(bins / "acoustic"), "-V"] + [str(f) for f in files], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lines = r.stdout.strip().splitlines()
    assert len(lines) == 3
    for i, line in enumerate(lines):
        dense = np.zeros(1, np.uint64)
        rec = ctx.vowel_report_batch(rows[i].copy(), [ns[i]], offsets=dense, fs=[int(p.fs[i])])[0]
        rep = rec["rep"]
        want = [str(files[i]), str(int(p.fs[i])), str(int(ns[i])), str(int(rep["base"]["cycles"])), f"{rep['base']['f0_hz']:.3f}",
                f"{rep['base']['jitter_pct']:.4f}", f"{rep['base']['shimmer_pct']:.4f}"]
        assert line.split()[:7] == want, (i, line)
        assert line.split()[-2:] == [str(int(rec["run_start"])), str(int(rec["run_len"]))], (i, line)
