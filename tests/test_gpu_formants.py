"""vs_formant_batch on the GPU against the numpy restatement (tests/formant_ref.py): every frame record and every
statistic of the ten presets, tract voices at 22 050 and 44 100 Hz, voices with glottal and with output noise, the
extreme orders and formant counts, ragged, empty, silent and short rows, and a 60-second stream among short ones; host
and device input, frames = NULL, the error codes and `acoustic -F`."""
import math
import pathlib
import subprocess
import wave

import numpy as np
import pytest

import formant_ref as fr

pytestmark = pytest.mark.gpu
ROOT = pathlib.Path(__file__).resolve().parents[1]
PRESETS = "aiu1234567"
TRACTS = {"a": ([730, 1090, 2440, 3400, 4500], [90, 110, 160, 250, 300]),
          "i": ([270, 2290, 3010, 3600, 4500], [60, 100, 170, 250, 300]),
          "u": ([300, 870, 2240, 3400, 4500], [70, 100, 140, 250, 300])}


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
    st, frames = ctx.formant_batch(pcm, ns, want_frames=True, **kw)
    st_dev, frames_dev = ctx.formant_batch(torch.from_numpy(pcm).cuda(), ns, want_frames=True, **kw)
    assert st.tobytes() == st_dev.tobytes()
    assert all(a.tobytes() == b.tobytes() for a, b in zip(frames, frames_dev))
    assert ctx.formant_batch(pcm, ns, **kw).tobytes() == st.tobytes()
    assert (st["reserved"] == 0).all()
    return st, frames


def _close(g, w, rel, abs_=0.0):
    if math.isnan(w):
        return math.isnan(g)
    return math.isclose(g, float(np.float32(w)), rel_tol=rel, abs_tol=abs_)


def _check(st, frames, rows, fs, opts, what):
    """every frame and every stats field against the restatement; frames the restatement marks ambiguous are skipped
    (with the statistics of their stream) and must be under 0.1 % of all frames"""
    o = fr.opts_with(**(opts or {}))
    nf = int(o["n_formants"])
    total = ambiguous = 0
    for i, x in enumerate(rows):
        rate = int(fs[i]) if fs is not None else 22050
        want_frames, want = fr.analyse(x, rate, o)
        got = frames[i]
        assert len(got) == len(want_frames) == st[i]["frames"], (what, i)
        amb = sum(f["ambiguous"] for f in want_frames)
        total += len(want_frames)
        ambiguous += amb
        for j, (g, w) in enumerate(zip(got, want_frames)):
            if w["ambiguous"]:
                continue
            assert int(g["flags"]) == w["flags"] and int(g["found"]) == len(w["F"]), (what, i, j, g, w)
            for k in range(8):
                if k < len(w["F"]):
                    assert _close(float(g["f_hz"][k]), w["F"][k], 1e-6), (what, i, j, k, g["f_hz"][k], w["F"][k])
                    assert _close(float(g["bw_hz"][k]), w["B"][k], 1e-5, 1e-3), (what, i, j, k, g["bw_hz"][k], w["B"][k])
                else:
                    assert math.isnan(g["f_hz"][k]) and math.isnan(g["bw_hz"][k]), (what, i, j, k)
        assert st[i]["unconverged"] == 0, (what, i)
        if amb:
            continue
        s = st[i]
        assert (s["frames"], s["analysed"]) == (want["frames"], want["analysed"]), (what, i)
        assert list(s["count"]) == want["count"], (what, i, s["count"], want["count"])
        for k in range(8):
            assert _close(float(s["f_mean_hz"][k]), want["f_mean_hz"][k], 1e-6), (what, i, k)
            assert _close(float(s["bw_mean_hz"][k]), want["bw_mean_hz"][k], 1e-5, 1e-3), (what, i, k)
            assert _close(float(s["f_sd_hz"][k]), want["f_sd_hz"][k], 1e-5, 1e-3), (what, i, k)
        assert all(math.isnan(s[f][k]) for f in ("f_mean_hz", "f_sd_hz", "bw_mean_hz") for k in range(nf, 8))
    assert ambiguous <= 0.001 * max(total, 1), (what, ambiguous, total)
    return total


OPTS = [None, dict(order=2, n_formants=1), dict(order=32, n_formants=8), dict(order=16, n_formants=8, bmax_hz=0.0, preemph_hz=0.0)]


@pytest.mark.parametrize("opts", OPTS, ids=["defaults", "p2_n1", "p32_n8", "p16_n8_nolimit"])
def test_presets_match_restatement(ctx, vs, opts):
    """the ten presets at several F0, half the voices with glottal noise and then output noise (`vowel -n`)"""
    n = 30
    p = _flow_params(vs, n, 11, noise=True)
    f = vs.FilterParams(n, "".join(PRESETS[i % 10] for i in range(n)))
    pcm, offs, ns = ctx.synth_batch(p, f)
    noisy = np.array([20.0 if i % 3 == 1 else 0.0 for i in range(n)], dtype=np.float32)
    ctx.vowel_noise_batch(pcm, ns, noisy, np.arange(n) + 5, offsets=offs)
    st, frames = _analyse(ctx, pcm, ns, offsets=offs, opts=opts)
    assert _check(st, frames, _rows(pcm, offs, ns), None, opts, opts) > 2500


@pytest.mark.parametrize("fs,opts", [(22050, None), (44100, dict(order=24)), (44100, dict(order=32, n_formants=8))])
def test_tract_voices_match_restatement(ctx, vs, fs, opts):
    n = 12
    p = _flow_params(vs, n, fs + 3, noise=True, fs=fs)
    den = np.stack([vs.tract_from_formants(*TRACTS[v], fs) for v in "aiu"])
    t = vs.TractParams(n, den, tract=np.arange(n) % 3, gain=1.5)
    pcm, offs, ns = ctx.synth_batch(p, t)
    st, frames = _analyse(ctx, pcm, ns, offsets=offs, fs=p.fs, opts=opts)
    _check(st, frames, _rows(pcm, offs, ns), p.fs, opts, (fs, opts))


def test_ragged_empty_silent_short_and_long_rows(ctx, vs):
    """rows at odd offsets with gaps: zero-length, shorter than a window, exactly one window, silent, silent but for the
    last frame, and one 60-second voice among short ones in one call"""
    rng = np.random.default_rng(4)
    p = _flow_params(vs, 6, 8, noise=True)
    f = vs.FilterParams(6, "ai3u6a")
    voices, voffs, vns = ctx.synth_batch(p, f)
    vrows = _rows(voices, voffs, vns)
    long_p = _flow_params(vs, 1, 9, dur=60.0)
    long_pcm, _, _ = ctx.synth_batch(long_p, vs.FilterParams(1, "i"))
    Nw, H = fr.geometry(22050, fr.DEFAULTS)
    last_only = np.zeros(5000, dtype=np.int16)
    F = fr.n_frames(5000, Nw, H)
    last_only[(F - 2) * H + Nw:] = rng.integers(-3000, 3000, 5000 - ((F - 2) * H + Nw))
    rows = [vrows[0], np.zeros(0, np.int16), vrows[1][:Nw - 1], vrows[2][:Nw], np.zeros(3000, np.int16), last_only,
            long_pcm, vrows[3], vrows[4][:Nw + H - 1], vrows[5][:Nw + H]]
    ns = np.array([len(r) for r in rows], dtype=np.uint64)
    offs = np.zeros(len(rows), dtype=np.uint64)
    pos = 3
    for i, r in enumerate(rows):
        offs[i] = pos
        pos += len(r) + 2 * int(rng.integers(0, 40)) + 1
    pcm = np.full(pos + 5, 777, dtype=np.int16)                    # the gaps are not silent: nothing may read them
    for i, r in enumerate(rows):
        pcm[int(offs[i]): int(offs[i]) + len(r)] = r
    st, frames = _analyse(ctx, pcm, ns, offsets=offs)
    _check(st, frames, rows, None, None, "ragged")
    assert list(st["frames"][[1, 2, 3, 8, 9]]) == [0, 0, 1, 1, 2]
    assert st[4]["analysed"] == 0 and all(fm["flags"] == vs.FRAME_SILENT for fm in frames[4])
    assert st[5]["analysed"] == 1 and frames[5][-1]["flags"] == 0
    assert st[6]["frames"] == fr.n_frames(60 * 22050, Nw, H) and st[6]["analysed"] == st[6]["frames"]
    # frame_offsets: the records of each stream wherever the caller wants them
    want = np.concatenate(frames)
    fo = np.concatenate([[0], np.cumsum(st["frames"])])[:-1].astype(np.uint64)
    perm = np.arange(len(rows))[::-1]
    place = np.zeros(len(rows), dtype=np.uint64)
    place[perm] = np.concatenate([[0], np.cumsum(st["frames"][perm])])[:-1] + 5
    out = np.zeros(int(st["frames"].sum()) + 10, dtype=vs.FORMANT_FRAME_DTYPE)
    st2 = np.zeros(len(rows), dtype=vs.FORMANT_STATS_DTYPE)
    ctx._check(ctx.L.vs_formant_batch(ctx.h, pcm.ctypes.data, offs.ctypes.data, ns.ctypes.data, None, len(rows), None,
                                      st2.ctypes.data, out.ctypes.data, place.ctypes.data))
    assert st2.tobytes() == st.tobytes()
    for i in range(len(rows)):
        k = int(st["frames"][i])
        assert out[int(place[i]): int(place[i]) + k].tobytes() == want[int(fo[i]): int(fo[i]) + k].tobytes(), i


def test_formant_errors(ctx, vs):
    import torch
    L, h = ctx.L, ctx.h
    x = np.zeros(2000, dtype=np.int16)
    ns = np.array([2000], dtype=np.uint64)
    st = np.zeros(1, dtype=vs.FORMANT_STATS_DTYPE)
    bad_fs = np.array([0], dtype=np.int32)
    call = lambda pcm, n_, fs, o, stats: L.vs_formant_batch(h, pcm, None, n_, fs, 1, o, stats, None, None)
    assert call(None, ns.ctypes.data, None, None, st.ctypes.data) == vs.VS_EINVAL
    assert call(x.ctypes.data, None, None, None, st.ctypes.data) == vs.VS_EINVAL
    assert call(x.ctypes.data, ns.ctypes.data, None, None, None) == vs.VS_EINVAL
    assert L.vs_formant_batch(None, x.ctypes.data, None, ns.ctypes.data, None, 1, None, st.ctypes.data, None, None) == vs.VS_EINVAL
    assert call(x.ctypes.data, ns.ctypes.data, bad_fs.ctypes.data, None, st.ctypes.data) == vs.VS_ERANGE
    for o, code in [(dict(order=13), vs.VS_EINVAL), (dict(n_formants=9), vs.VS_EINVAL), (dict(bmax_hz=-1.0), vs.VS_ERANGE),
                    (dict(win_ms=0.2), vs.VS_ERANGE), (dict(win_ms=500.0), vs.VS_ERANGE), (dict(hop_ms=0.0), vs.VS_ERANGE)]:
        with pytest.raises(vs.VsError) as e:
            ctx.formant_batch(x, [2000], opts=o)
        assert e.value.code == code, o
        with pytest.raises(vs.VsError) as e:
            vs.formant_frames([2000], None, o)
        assert e.value.code == code, o
    assert L.vs_formant_batch(h, x.ctypes.data, None, ns.ctypes.data, None, 0, None, st.ctypes.data, None, None) == vs.VS_OK
    if torch.cuda.device_count() > 1:
        other = torch.zeros(2000, dtype=torch.int16, device="cuda:1")
        assert L.vs_formant_batch(h, other.data_ptr(), None, ns.ctypes.data, None, 1, None, st.ctypes.data, None, None) == vs.VS_EINVAL
    assert ctx.formant_batch(x, [2000])["analysed"][0] == 0        # the context still works


def _write_wav(path, x, fs):
    with wave.open(str(path), "wb") as w:
        w.setnchannels(1)
        w.setsampwidth(2)
        w.setframerate(fs)
        w.writeframes(np.ascontiguousarray(x, dtype="<i2").tobytes())


def test_acoustic_formant_lines(ctx, vs, tmp_path):
    """host/bin/acoustic -F [-p order]: one line per file with the means of vs_formant_batch"""
    bins = ROOT / "host" / "bin"
    if not (bins / "acoustic").exists():
        subprocess.run(["make", "-s", "-C", str(ROOT), "host"], check=True)
    p = _flow_params(vs, 4, 31)
    p.fs[2:] = 44100
    pcm, offs, ns = ctx.synth_batch(p, vs.FilterParams(4, "aiu3"))
    rows = _rows(pcm, offs, ns)
    files = []
    for i, x in enumerate(rows):
        files.append(tmp_path / f"v{i}.wav")
        _write_wav(files[-1], x, int(p.fs[i]))
    for order in (None, 24, 6):
        args = [str(bins / "acoustic"), "-F"] + (["-p", str(order)] if order else []) + [str(f) for f in files]
        r = subprocess.run(args, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        lines = r.stdout.strip().splitlines()
        nf = min(5, (order or 14) // 2)
        opts = None if order is None else dict(order=order, n_formants=nf)
        dense = np.concatenate([[0], np.cumsum(ns)[:-1]]).astype(np.uint64)
        st = ctx.formant_batch(np.concatenate(rows), ns, offsets=dense, fs=p.fs, opts=opts)
        assert len(lines) == 4
        for i, line in enumerate(lines):
            t = line.split()
            assert t[:5] == [str(files[i]), str(int(p.fs[i])), str(int(ns[i])), str(int(st[i]["frames"])), str(int(st[i]["analysed"]))]
            assert len(t) == 5 + 2 * nf
            want = [f"{v:.1f}" for v in list(st[i]["f_mean_hz"][:nf]) + list(st[i]["bw_mean_hz"][:nf])]
            assert t[5:] == want, (order, i)
