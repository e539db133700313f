"""Formant analysis without a GPU: vs_formant_frames through the library (frame counts and every refusal), and the numpy
restatement of the definitions (tests/formant_ref.py) in a closed loop: oracle flow through formant tracts
(vs_tract_from_formants, the reference filter of tests/tools/vowel_den.c), analysed, against the formants the tracts
were built from."""
import math

import numpy as np
import pytest
import scipy.linalg

import formant_ref as fr
from voice_synth_b200 import api

# tract vowels: F1..F5 and their bandwidths (Peterson & Barney's men's averages for F1-F3)
VOWELS = {"a": ([730, 1090, 2440, 3400, 4500], [90, 110, 160, 250, 300]),
          "i": ([270, 2290, 3010, 3600, 4500], [60, 100, 170, 250, 300]),
          "u": ([300, 870, 2240, 3400, 4500], [70, 100, 140, 250, 300]),
          "e": ([530, 1840, 2480, 3500, 4500], [80, 100, 150, 250, 300]),
          "o": ([570, 840, 2410, 3400, 4500], [80, 100, 150, 250, 300])}


@pytest.mark.parametrize("fs", [8000, 22050, 44100, 48000])
def test_formant_frames_counts(fs):
    o = fr.DEFAULTS
    Nw, H = fr.geometry(fs, o)
    ns = [0, 1, Nw - 1, Nw, Nw + 1, Nw + H - 1, Nw + H, Nw + 7 * H + 3, fs, 60 * fs]
    got = api.formant_frames(ns, fs)
    assert list(got) == [fr.n_frames(n, Nw, H) for n in ns]
    assert list(got[:7]) == [0, 0, 0, 1, 1, 1, 2]


def test_formant_frames_options_and_rounding():
    # 25 ms at 22050 Hz is 551.25 samples, 10 ms 220.5: lround gives 551 and 221 (halves away from zero)
    assert fr.geometry(22050, fr.DEFAULTS) == (551, 221)
    assert list(api.formant_frames([551, 771, 772], 22050)) == [1, 1, 2]
    o = dict(win_ms=5.0, hop_ms=1.0, order=32, n_formants=8)
    Nw, H = fr.geometry(16000, fr.opts_with(**o))
    assert (Nw, H) == (80, 16)
    assert list(api.formant_frames([79, 80, 96, 1000], 16000, o)) == [0, 1, 2, (1000 - 80) // 16 + 1]
    # fs NULL is 22050 for every stream
    assert list(api.formant_frames([10000, 20000])) == list(api.formant_frames([10000, 20000], [22050, 22050]))


def _code(ns, fs=None, **o):
    with pytest.raises(api.VsError) as e:
        api.formant_frames(ns, fs, o)
    return e.value.code


def test_formant_frames_refusals():
    assert _code([1000], order=0) == api.VS_EINVAL
    assert _code([1000], order=15) == api.VS_EINVAL
    assert _code([1000], order=34, n_formants=5) == api.VS_EINVAL
    assert _code([1000], n_formants=0) == api.VS_EINVAL
    assert _code([1000], n_formants=9, order=32) == api.VS_EINVAL
    assert _code([1000], order=8, n_formants=5) == api.VS_EINVAL          # more than p/2
    assert _code([1000], preemph_hz=-1.0) == api.VS_ERANGE
    assert _code([1000], bmax_hz=-1.0) == api.VS_ERANGE
    assert _code([1000], bmax_hz=math.nan) == api.VS_ERANGE
    assert _code([1000], [0]) == api.VS_ERANGE
    assert _code([1000], [-22050]) == api.VS_ERANGE
    assert _code([1000], [22050], win_ms=0.5) == api.VS_ERANGE              # Nw = 11 < p + 1
    assert _code([1000], [22050], win_ms=200.0) == api.VS_ERANGE            # Nw = 4410 > 4096
    assert _code([1000], [22050], hop_ms=0.02) == api.VS_ERANGE             # H = 0
    assert _code([1000], [22050], win_ms=math.inf) == api.VS_ERANGE
    assert _code([2 ** 31], [22050]) == api.VS_EOVERLAP
    # the first offender decides: stream 0's bad rate before stream 1's length
    assert _code([1000, 2 ** 31], [0, 22050]) == api.VS_ERANGE
    assert _code([2 ** 31, 1000], [22050, 0]) == api.VS_EOVERLAP
    # the limits themselves pass
    assert api.formant_frames([5000], [22050], dict(order=2, n_formants=1, win_ms=3 / 22.05, hop_ms=0.05)).size == 1
    assert api.formant_frames([5000], [4096 * 40], dict(win_ms=25.0)).size == 1
    L = api._lib.load()
    out = np.zeros(1, dtype=np.uint64)
    ns = np.array([100], dtype=np.uint64)
    assert L.vs_formant_frames(None, None, None, 1, out.ctypes.data) == api.VS_EINVAL
    assert L.vs_formant_frames(None, ns.ctypes.data, None, 1, None) == api.VS_EINVAL
    assert L.vs_formant_frames(None, ns.ctypes.data, None, 0, out.ctypes.data) == api.VS_OK


def test_restatement_levinson_solves_the_normal_equations():
    rng = np.random.default_rng(5)
    y = rng.normal(size=551) * fr.window(551)
    for p in (2, 14, 32):
        r = fr.autocorr(y, p)
        a = fr.levinson(r, p)
        want = scipy.linalg.solve_toeplitz(r[:p], -np.array(r[1: p + 1]))
        assert np.allclose(a, want, rtol=1e-9, atol=1e-12), p


@pytest.fixture(scope="module")
def vowel_den(tmp_path_factory):
    from vowel_den_ref import VowelDen
    return VowelDen(tmp_path_factory.mktemp("vowel_den"))


def tract_voice(oracle, vowel_den, fs, f0, vowel, seed=7):
    """1 s of oracle flow (jitter 1 %, shimmer 3 %) through the tract of `vowel` built at fs, pre-emphasis 1, scaled to
    0.7 of full scale"""
    a = ["-o", "x", "-d", "1", "-f", str(f0), "-g", str(f0 + 30), "-j", "1", "-s", "3"] + (["-r", str(fs)] if fs != 22050 else [])
    flow = oracle.flowgen(oracle.flow_par_from_cli(a, seed))
    den = api.tract_from_formants(*VOWELS[vowel], fs)
    _, raw = vowel_den(flow, den, gain=1.0, pre=1.0, want_raw=True)
    return vowel_den(flow, den, gain=0.7 * 32767 / np.abs(raw).max(), pre=1.0)


# largest relative error of the F1, F2, F3 means over F0 = 100, 120, 150 Hz (measured with this restatement; DESIGN 4.2d)
CLOSED_LOOP = [(22050, 14, "aiueo", (0.13, 0.08, 0.10)), (44100, 24, "aie", (0.12, 0.07, 0.09))]


@pytest.mark.parametrize("fs,order,vowels,bound", CLOSED_LOOP, ids=["22050-p14", "44100-p24"])
def test_closed_loop_tract_vowels(oracle, vowel_den, fs, order, vowels, bound):
    o = fr.opts_with(order=order)
    for v in vowels:
        for f0 in (100, 120, 150):
            frames, st = fr.analyse(tract_voice(oracle, vowel_den, fs, f0, v), fs, o)
            assert st["frames"] == st["analysed"] == 98 and st["unconverged"] == 0
            for k in range(3):
                assert st["count"][k] > 0, (fs, v, f0, k)
                err = abs(st["f_mean_hz"][k] / VOWELS[v][0][k] - 1.0)
                assert err <= bound[k], (fs, v, f0, k, st["f_mean_hz"][k], VOWELS[v][0][k])


def test_silent_frames():
    o = fr.DEFAULTS
    Nw, H = fr.geometry(22050, o)
    frames, st = fr.analyse(np.zeros(5000, dtype=np.int16), 22050, o)
    assert st["frames"] == fr.n_frames(5000, Nw, H) and st["analysed"] == 0
    assert all(f["flags"] == fr.SILENT for f in frames)
    assert st["count"] == [0] * 8 and all(math.isnan(v) for v in st["f_mean_hz"] + st["f_sd_hz"] + st["bw_mean_hz"])
    # sound only where the last frame alone reaches
    n = 5000
    F = fr.n_frames(n, Nw, H)
    x = np.zeros(n, dtype=np.int16)
    tail = (F - 2) * H + Nw
    x[tail:] = (np.random.default_rng(1).normal(size=n - tail) * 3000).astype(np.int16)
    frames, st = fr.analyse(x, 22050, o)
    assert [f["flags"] for f in frames] == [fr.SILENT] * (F - 1) + [0]
    assert st["analysed"] == 1 and all(math.isnan(v) for v in st["f_sd_hz"])


def test_preemphasis_uses_the_real_previous_sample():
    x = np.arange(1, 2000, dtype=np.int16)
    Nw, H, mu = 551, 221, 0.9
    w = np.ones(Nw)
    y0 = fr.frame_signal(x, 0, Nw, H, mu, w)
    y1 = fr.frame_signal(x, 1, Nw, H, mu, w)
    assert y0[0] == 1.0 and y1[0] == x[H] - mu * x[H - 1]
