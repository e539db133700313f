"""vs_pitch_batch on the GPU against the numpy restatement (tests/pitch_ref.py): every frame record and every statistic of
the ten presets with glottal and with output noise, tract voices at 22 050 and 44 100 Hz, the option extremes, closed-form
rows, ragged, empty and short rows and a 60-second stream among short ones; host and device input, frames = NULL,
frame_offsets, the error codes, the closed loop on rendered voices and `acoustic -P`."""
import math
import pathlib
import subprocess
import wave

import numpy as np
import pytest

import pitch_ref as pr
from test_pitch_host import F0_BOUND, F0S, HNR_BAND

pytestmark = pytest.mark.gpu
ROOT = pathlib.Path(__file__).resolve().parents[1]
PRESETS = "aiu1234567"
TRACTS = {"a": ([730, 1090, 2440, 3400, 4500], [90, 110, 160, 250, 300]),
          "i": ([270, 2290, 3010, 3600, 4500], [60, 100, 170, 250, 300]),
          "u": ([300, 870, 2240, 3400, 4500], [70, 100, 140, 250, 300])}
F32_REL = 2.5e-7          # two float ulps: the records hold float roundings of FP64 values that agree to ~1e-12


@pytest.fixture(scope="module")
def vs():
    from voice_synth_b200 import api
    return api


@pytest.fixture(scope="module")
def ctx(vs):
    c = vs.Context()
    yield c
    c.close()


def _flow_params(vs, n, seed, noise=False, fs=22050, dur=1.0):
    rng = np.random.default_rng(seed)
    args, seeds = [], []
    for i in range(n):
        f0 = float(rng.uniform(85, 230))
        a = ["-d", f"{dur:.3f}", "-f", f"{f0:.2f}", "-g", f"{f0 + 30:.2f}", "-j", f"{rng.uniform(0, 2):.2f}",
             "-s", f"{rng.uniform(0, 6):.2f}"]
        if noise and i % 2 == 0:
            a += ["-n", f"{rng.uniform(15, 35):.1f}"]
        if fs != 22050:
            a += ["-r", str(fs)]
        args.append(a)
        seeds.append(int(rng.integers(0, 2 ** 31)))
    return vs.FlowParams.from_cli(args, seeds)


def _rows(pcm, offs, ns):
    return [pcm[int(offs[i]): int(offs[i]) + int(ns[i])] for i in range(len(ns))]


def _analyse(ctx, pcm, ns, **kw):
    """the call from host and from device input (byte-identical), with and without frame records (same stats)"""
    import torch
    st, frames = ctx.pitch_batch(pcm, ns, want_frames=True, **kw)
    st_dev, frames_dev = ctx.pitch_batch(torch.from_numpy(pcm).cuda(), ns, want_frames=True, **kw)
    assert st.tobytes() == st_dev.tobytes()
    assert all(a.tobytes() == b.tobytes() for a, b in zip(frames, frames_dev))
    assert ctx.pitch_batch(pcm, ns, **kw).tobytes() == st.tobytes()
    assert (st["reserved"] == 0).all()
    return st, frames


def _close(g, w, rel=F32_REL, abs_=0.0):
    if math.isnan(w):
        return math.isnan(g)
    if math.isinf(w):
        return g == w
    return math.isclose(g, float(np.float32(w)), rel_tol=rel, abs_tol=abs_)


def _check(st, frames, rows, fs, opts, what):
    """every frame and every stats field against the restatement.  Frames within pr.MARGIN of a decision are skipped
    (with the statistics of their stream) and must be under 0.1 % of all frames."""
    o = pr.opts_with(**(opts or {}))
    total = low = 0
    for i, x in enumerate(rows):
        rate = int(fs[i]) if fs is not None else 22050
        want_frames, want = pr.analyse(x, rate, o)
        got = frames[i]
        assert len(got) == len(want_frames) == st[i]["frames"], (what, i)
        near = [w["margin"] <= pr.MARGIN for w in want_frames]
        total += len(want_frames)
        low += sum(near)
        for j, (g, w) in enumerate(zip(got, want_frames)):
            if near[j]:
                continue
            assert int(g["flags"]) == w["flags"], (what, i, j, g, w)
            assert _close(float(g["f0_hz"]), w["f0"]), (what, i, j, g["f0_hz"], w["f0"])
            assert _close(float(g["strength"]), w["r"]), (what, i, j, g["strength"], w["r"])
            hnr_abs = 4e-6 if abs(w["hnr"]) < 60 else 1e-2
            assert _close(float(g["hnr_db"]), w["hnr"], F32_REL, hnr_abs), (what, i, j, g["hnr_db"], w["hnr"])
        if any(near):
            continue
        s = st[i]
        assert (s["periodic"], s["voiced"]) == (want["periodic"], want["voiced"]), (what, i)
        for k in ("f0_mean_hz", "f0_min_hz", "f0_max_hz", "strength_mean"):
            assert _close(float(s[k]), want[k], 1e-6), (what, i, k, s[k], want[k])
        assert _close(float(s["hnr_mean_db"]), want["hnr_mean_db"], 1e-6, 1e-5), (what, i, s["hnr_mean_db"], want["hnr_mean_db"])
        for k in ("f0_sd_hz", "hnr_sd_db"):
            assert _close(float(s[k]), want[k], 1e-5, 1e-4), (what, i, k, s[k], want[k])
    assert low <= 0.001 * max(total, 1), (what, low, total)
    return total


@pytest.mark.parametrize("noise", ["glottal", "output"])
def test_presets_match_restatement(ctx, vs, noise):
    """the ten presets at several F0, with glottal noise on half the voices or output noise (`vowel -n`) on two thirds"""
    n = 30
    p = _flow_params(vs, n, 11, noise=noise == "glottal")
    f = vs.FilterParams(n, "".join(PRESETS[i % 10] for i in range(n)))
    pcm, offs, ns = ctx.synth_batch(p, f)
    if noise == "output":
        snr = np.array([(10.0, 20.0, 0.0)[i % 3] for i in range(n)], dtype=np.float32)
        ctx.vowel_noise_batch(pcm, ns, snr, np.arange(n) + 5, offsets=offs)
    st, frames = _analyse(ctx, pcm, ns, offsets=offs)
    assert _check(st, frames, _rows(pcm, offs, ns), None, None, noise) > 2500
    assert st["voiced"].sum() > 0.9 * st["frames"].sum()


@pytest.mark.parametrize("fs", [22050, 44100])
def test_tract_voices_match_restatement(ctx, vs, fs):
    n = 12
    p = _flow_params(vs, n, fs + 3, noise=True, fs=fs)
    den = np.stack([vs.tract_from_formants(*TRACTS[v], fs) for v in "aiu"])
    t = vs.TractParams(n, den, tract=np.arange(n) % 3, gain=1.5)
    pcm, offs, ns = ctx.synth_batch(p, t)
    st, frames = _analyse(ctx, pcm, ns, offsets=offs, fs=p.fs)
    _check(st, frames, _rows(pcm, offs, ns), p.fs, None, fs)


OPTS = [dict(f_min_hz=50.0, f_max_hz=1000.0), dict(periods=2.0), dict(periods=6.0, hop_ms=7.0), dict(octave_cost=0.0),
        dict(voicing_threshold=0.0), dict(voicing_threshold=0.9, silence_threshold=0.3), dict(periods=4.5)]


@pytest.mark.parametrize("opts", OPTS, ids=["50-1000Hz", "periods2", "periods6", "octave0", "voicing0", "voicing0.9", "harmonicity"])
def test_option_extremes_match_restatement(ctx, vs, opts):
    n = 10
    p = _flow_params(vs, n, 21, noise=True)
    p.fs[5:] = 44100
    pcm, offs, ns = ctx.synth_batch(p, vs.FilterParams(n, PRESETS))
    ctx.vowel_noise_batch(pcm, ns, np.where(np.arange(n) % 2 == 1, 15.0, 0.0), np.arange(n), offsets=offs, fs=p.fs)
    st, frames = _analyse(ctx, pcm, ns, offsets=offs, fs=p.fs, opts=opts)
    _check(st, frames, _rows(pcm, offs, ns), p.fs, opts, opts)


def _synthetic_rows():
    fs = 22050
    t = np.arange(fs)
    rng = np.random.default_rng(2)
    impulses = np.zeros(fs, np.int16)
    impulses[3::147] = 10000
    return [np.round(10000 * np.sin(2 * np.pi * 200 * t / fs)).astype(np.int16), impulses,
            rng.integers(-5000, 5000, fs).astype(np.int16), np.zeros(5000, np.int16), np.full(5000, 1234, np.int16),
            np.round(10000 * np.sin(2 * np.pi * 150 * np.arange(2 * fs) / fs) * np.where(np.arange(2 * fs) < fs, 1, 0.01)).astype(np.int16)]


def _ragged(rows, rng):
    ns = np.array([len(r) for r in rows], dtype=np.uint64)
    offs = np.zeros(len(rows), dtype=np.uint64)
    pos = 3
    for i, r in enumerate(rows):
        offs[i] = pos
        pos += len(r) + 2 * int(rng.integers(0, 40)) + 1
    pcm = np.full(pos + 5, 777, dtype=np.int16)                    # the gaps are not silent: nothing may read them
    for i, r in enumerate(rows):
        pcm[int(offs[i]): int(offs[i]) + len(r)] = r
    return pcm, offs, ns


def test_synthetic_rows(ctx, vs):
    """sine, impulse train of integer period, white noise, silence, DC and a voice fading to 1 %"""
    rows = _synthetic_rows()
    pcm, offs, ns = _ragged(rows, np.random.default_rng(3))
    st, frames = _analyse(ctx, pcm, ns, offsets=offs)
    _check(st, frames, rows, None, None, "synthetic")
    assert st[0]["voiced"] == st[0]["frames"] and abs(st[0]["f0_mean_hz"] - 200) < 0.1
    assert st[1]["voiced"] == st[1]["frames"] and abs(st[1]["f0_mean_hz"] - 150) < 1e-3
    assert st[2]["voiced"] == 0
    assert all((fr["flags"] == vs.PITCH_SILENT).all() for fr in frames[3:5])
    assert 0 < (frames[5]["flags"] == vs.PITCH_QUIET).sum() < len(frames[5])


def test_ragged_empty_short_and_long_rows(ctx, vs):
    """rows at odd offsets with gaps: zero-length, shorter than a window, exactly one window, one 60-second voice among
    short ones in one call; and frame_offsets placing each stream's records"""
    rng = np.random.default_rng(4)
    p = _flow_params(vs, 6, 8, noise=True)
    voices, voffs, vns = ctx.synth_batch(p, vs.FilterParams(6, "ai3u6a"))
    vrows = _rows(voices, voffs, vns)
    long_pcm, _, _ = ctx.synth_batch(_flow_params(vs, 1, 9, dur=60.0), vs.FilterParams(1, "i"))
    Nw, H, _, _ = pr.geometry(22050, pr.DEFAULTS)
    rows = [vrows[0], np.zeros(0, np.int16), vrows[1][:Nw - 1], vrows[2][:Nw], long_pcm, vrows[3], vrows[4][:Nw + H - 1],
            vrows[5][:Nw + H]]
    pcm, offs, ns = _ragged(rows, rng)
    st, frames = _analyse(ctx, pcm, ns, offsets=offs)
    _check(st, frames, rows, None, None, "ragged")
    assert list(st["frames"][[1, 2, 3, 6, 7]]) == [0, 0, 1, 1, 2]
    assert st[1]["periodic"] == 0 and math.isnan(st[1]["f0_mean_hz"]) and math.isnan(st[1]["hnr_mean_db"])
    assert st[4]["frames"] == pr.n_frames(60 * 22050, Nw, H) and st[4]["voiced"] > 0.95 * st[4]["frames"]
    want = np.concatenate(frames)
    fo = np.concatenate([[0], np.cumsum(st["frames"])])[:-1].astype(np.uint64)
    perm = np.arange(len(rows))[::-1]
    place = np.zeros(len(rows), dtype=np.uint64)
    place[perm] = np.concatenate([[0], np.cumsum(st["frames"][perm])])[:-1] + 5
    out = np.zeros(int(st["frames"].sum()) + 10, dtype=vs.PITCH_FRAME_DTYPE)
    st2 = np.zeros(len(rows), dtype=vs.PITCH_STATS_DTYPE)
    ctx._check(ctx.L.vs_pitch_batch(ctx.h, pcm.ctypes.data, offs.ctypes.data, ns.ctypes.data, None, len(rows), None,
                                    st2.ctypes.data, out.ctypes.data, place.ctypes.data))
    assert st2.tobytes() == st.tobytes()
    for i in range(len(rows)):
        k = int(st["frames"][i])
        assert out[int(place[i]): int(place[i]) + k].tobytes() == want[int(fo[i]): int(fo[i]) + k].tobytes(), i


def test_pitch_errors(ctx, vs):
    import torch
    L, h = ctx.L, ctx.h
    x = (np.sin(np.arange(4000) / 10.0) * 5000).astype(np.int16)
    ns = np.array([4000], dtype=np.uint64)
    st = np.zeros(1, dtype=vs.PITCH_STATS_DTYPE)
    bad_fs = np.array([0], dtype=np.int32)
    works = lambda: ctx.pitch_batch(x, [4000])["voiced"][0] > 0
    call = lambda pcm, n_, fs, stats: L.vs_pitch_batch(h, pcm, None, n_, fs, 1, None, stats, None, None)
    assert call(None, ns.ctypes.data, None, st.ctypes.data) == vs.VS_EINVAL and works()
    assert call(x.ctypes.data, None, None, st.ctypes.data) == vs.VS_EINVAL and works()
    assert call(x.ctypes.data, ns.ctypes.data, None, None) == vs.VS_EINVAL and works()
    assert L.vs_pitch_batch(None, x.ctypes.data, None, ns.ctypes.data, None, 1, None, st.ctypes.data, None, None) == vs.VS_EINVAL
    assert call(x.ctypes.data, ns.ctypes.data, bad_fs.ctypes.data, st.ctypes.data) == vs.VS_ERANGE and works()
    big = np.array([2 ** 31], dtype=np.uint64)
    assert call(x.ctypes.data, big.ctypes.data, None, st.ctypes.data) == vs.VS_EOVERLAP and works()
    for o in [dict(f_min_hz=0.0), dict(f_max_hz=70.0), dict(periods=1.5), dict(voicing_threshold=2.0), dict(octave_cost=-1.0),
              dict(hop_ms=math.nan), dict(f_min_hz=10.0), dict(hop_ms=0.0), dict(f_min_hz=500.0, f_max_hz=505.0)]:
        with pytest.raises(vs.VsError) as e:
            ctx.pitch_batch(x, [4000], opts=o)
        assert e.value.code == vs.VS_ERANGE, o
        with pytest.raises(vs.VsError) as e:
            vs.pitch_frames([4000], None, o)
        assert e.value.code == vs.VS_ERANGE, o
        assert works()
    assert L.vs_pitch_batch(h, x.ctypes.data, None, ns.ctypes.data, None, 0, None, st.ctypes.data, None, None) == vs.VS_OK
    if torch.cuda.device_count() > 1:
        other = torch.zeros(4000, dtype=torch.int16, device="cuda:1")
        assert L.vs_pitch_batch(h, other.data_ptr(), None, ns.ctypes.data, None, 1, None, st.ctypes.data, None, None) == vs.VS_EINVAL
    assert works()


def test_closed_loop_on_rendered_voices(ctx, vs):
    """the host's closed loop (test_pitch_host) on voices the library renders: F0 against the period log of the same
    flow, and the HNR of `vowel -n` output noise from vs_vowel_noise_batch, inside the bands measured on the oracle"""
    args, keys = [], []
    for key in PRESETS:
        for f0 in F0S:
            args.append(f"-d 1 -f {f0} -g {f0 + 30} -j 1 -s 3")
            keys.append(key)
    p = vs.FlowParams.from_cli(args, [7] * len(args))
    _, _, _, logs = ctx.flowgen_batch(p, want_log=True)
    pcm, offs, ns = ctx.synth_batch(p, vs.FilterParams(len(args), "".join(keys)))
    st = ctx.pitch_batch(pcm, ns, offsets=offs)
    for i, key in enumerate(keys):
        assert st[i]["voiced"] == st[i]["frames"] == 96, i
        assert abs(st[i]["f0_mean_hz"] / (22050 / np.mean(logs[i]["T"])) - 1) <= F0_BOUND[key], (i, key, st[i]["f0_mean_hz"])
    q = vs.FlowParams.from_cli([f"-d 1 -f {f0} -g {f0 + 30}" for _ in PRESETS for f0 in F0S], [7] * len(args))
    for snr, (lo, hi) in HNR_BAND.items():
        pcm, offs, ns = ctx.synth_batch(q, vs.FilterParams(len(args), "".join(keys)))
        ctx.vowel_noise_batch(pcm, ns, snr, 3, offsets=offs)
        st = ctx.pitch_batch(pcm, ns, offsets=offs)
        assert ((st["hnr_mean_db"] >= lo) & (st["hnr_mean_db"] <= hi)).all(), (snr, st["hnr_mean_db"])


def _write_wav(path, x, fs):
    with wave.open(str(path), "wb") as w:
        w.setnchannels(1)
        w.setsampwidth(2)
        w.setframerate(fs)
        w.writeframes(np.ascontiguousarray(x, dtype="<i2").tobytes())


def test_acoustic_pitch_lines(ctx, vs, tmp_path):
    """host/bin/acoustic -P: one line per file with the statistics of vs_pitch_batch; a `vowel -n 20` voice lands in the
    closed loop's 20 dB band"""
    bins = ROOT / "host" / "bin"
    if not (bins / "acoustic").exists():
        subprocess.run(["make", "-s", "-C", str(ROOT), "host"], check=True)
    p = vs.FlowParams.from_cli([f"-d 1 -f {f0} -g {f0 + 30}" for f0 in (100, 120, 150, 200)], [7, 8, 9, 10])
    p.fs[2:] = 44100
    pcm, offs, ns = ctx.synth_batch(p, vs.FilterParams(4, "aiu3"))
    ctx.vowel_noise_batch(pcm, ns, [20.0, 0.0, 0.0, 0.0], 3, offsets=offs, fs=p.fs)
    rows = _rows(pcm, offs, ns)
    files = []
    for i, x in enumerate(rows):
        files.append(tmp_path / f"v{i}.wav")
        _write_wav(files[-1], x, int(p.fs[i]))
    r = subprocess.run([str(bins / "acoustic"), "-P"] + [str(f) for f in files], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lines = r.stdout.strip().splitlines()
    dense = np.concatenate([[0], np.cumsum(ns)[:-1]]).astype(np.uint64)
    st = ctx.pitch_batch(np.concatenate(rows), ns, offsets=dense, fs=p.fs)
    assert len(lines) == 4
    for i, line in enumerate(lines):
        t = line.split()
        assert t == [str(files[i]), str(int(p.fs[i])), str(int(ns[i])), str(int(st[i]["frames"])), str(int(st[i]["voiced"])),
                     f"{st[i]['f0_mean_hz']:.3f}", f"{st[i]['f0_sd_hz']:.3f}", f"{st[i]['hnr_mean_db']:.2f}"], i
    lo, hi = HNR_BAND[20.0]
    assert lo <= st[0]["hnr_mean_db"] <= hi
