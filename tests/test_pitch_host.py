"""Pitch analysis without a GPU: vs_pitch_frames through the library (frame counts and every refusal), the numpy
restatement of the definitions (tests/pitch_ref.py) against closed forms, and the closed loop on oracle voices: the mean
voiced F0 against the period log, and the mean HNR against the SNR handed to `vowel -n`."""
import math

import numpy as np
import pytest

import pitch_ref as pr
from voice_synth_b200 import api


@pytest.mark.parametrize("fs", [8000, 22050, 44100, 48000])
def test_pitch_frames_counts(fs):
    Nw, H, tau_lo, tau_hi = pr.geometry(fs, pr.DEFAULTS)
    assert 2 <= tau_lo < tau_hi < Nw - 1 and Nw <= pr.MAX_WIN
    ns = [0, 1, Nw - 1, Nw, Nw + 1, Nw + H - 1, Nw + H, Nw + 7 * H + 3, fs, 60 * fs]
    got = api.pitch_frames(ns, fs)
    assert list(got) == [pr.n_frames(n, Nw, H) for n in ns]
    assert list(got[:7]) == [0, 0, 0, 1, 1, 1, 2]


def test_pitch_frames_geometry_and_rounding():
    # 3 periods of 75 Hz at 22050 Hz: 882 samples; 10 ms: 220.5 -> 221 (halves away from zero); lags ceil(36.75) = 37
    # to floor(294) = 294
    assert pr.geometry(22050, pr.DEFAULTS) == (882, 221, 37, 294)
    assert list(api.pitch_frames([882, 1102, 1103], 22050)) == [1, 1, 2]
    o = dict(f_min_hz=100.0, f_max_hz=1000.0, periods=2.0, hop_ms=1.0)
    assert pr.geometry(16000, pr.opts_with(**o)) == (320, 16, 16, 160)
    assert list(api.pitch_frames([319, 320, 336, 1000], 16000, o)) == [0, 1, 2, (1000 - 320) // 16 + 1]
    # fs NULL is 22050 for every stream
    assert list(api.pitch_frames([10000, 20000])) == list(api.pitch_frames([10000, 20000], [22050, 22050]))


def _code(ns, fs=None, **o):
    with pytest.raises(api.VsError) as e:
        api.pitch_frames(ns, fs, o)
    return e.value.code


def test_pitch_frames_refusals():
    for k in pr.DEFAULTS:
        assert _code([5000], **{k: math.nan}) == api.VS_ERANGE, k
        assert _code([5000], **{k: math.inf}) == api.VS_ERANGE, k
    assert _code([5000], f_min_hz=0.0) == api.VS_ERANGE
    assert _code([5000], f_min_hz=-75.0) == api.VS_ERANGE
    assert _code([5000], f_max_hz=75.0) == api.VS_ERANGE                    # f_max == f_min
    assert _code([5000], periods=1.99) == api.VS_ERANGE
    for k in ("voicing_threshold", "silence_threshold"):
        assert _code([5000], **{k: -0.01}) == api.VS_ERANGE, k
        assert _code([5000], **{k: 1.01}) == api.VS_ERANGE, k
    assert _code([5000], octave_cost=-0.01) == api.VS_ERANGE
    assert _code([5000], [0]) == api.VS_ERANGE
    assert _code([5000], [-22050]) == api.VS_ERANGE
    assert _code([5000], [22050], f_min_hz=500.0, f_max_hz=510.0) == api.VS_ERANGE   # lags 44..44
    assert _code([5000], [100]) == api.VS_ERANGE                                     # lags 2..1
    assert _code([5000], [22050], f_min_hz=16.0) == api.VS_ERANGE                    # Nw = 4134 > 4096
    assert _code([5000], [22050], hop_ms=0.02) == api.VS_ERANGE                      # H = 0
    assert _code([5000], [22050], hop_ms=-10.0) == api.VS_ERANGE
    assert _code([5000], [48000], hop_ms=1e8) == api.VS_ERANGE                       # H above 2^31-1
    assert _code([2 ** 31], [22050]) == api.VS_EOVERLAP
    # the first offender decides: stream 0's bad rate before stream 1's length, and the other way round
    assert _code([1000, 2 ** 31], [0, 22050]) == api.VS_ERANGE
    assert _code([2 ** 31, 1000], [22050, 0]) == api.VS_EOVERLAP
    # option checks come before the streams
    assert _code([2 ** 31], [22050], periods=1.0) == api.VS_ERANGE
    # the limits themselves pass: Nw = 4096, the narrowest lag range, periods 2, thresholds 0 and 1, H = 1
    assert api.pitch_frames([5000], [4096 * 25], dict(periods=3.0)).size == 1
    assert api.pitch_frames([5000], [22050], dict(f_min_hz=500.0, f_max_hz=515.0)).size == 1       # lags 43..44
    assert api.pitch_frames([5000], [22050], dict(periods=2.0, voicing_threshold=0.0, silence_threshold=1.0,
                                                  octave_cost=0.0, hop_ms=1 / 22.05)).size == 1
    L = api._lib.load()
    out = np.zeros(1, dtype=np.uint64)
    ns = np.array([100], dtype=np.uint64)
    assert L.vs_pitch_frames(None, None, None, 1, out.ctypes.data) == api.VS_EINVAL
    assert L.vs_pitch_frames(None, ns.ctypes.data, None, 1, None) == api.VS_EINVAL
    assert L.vs_pitch_frames(None, ns.ctypes.data, None, 2 ** 31, out.ctypes.data) == api.VS_EINVAL
    assert L.vs_pitch_frames(None, ns.ctypes.data, None, 0, out.ctypes.data) == api.VS_OK


FS = 22050


def test_restatement_sinusoid():
    t = np.arange(FS)
    for f in (80.0, 200.0, 440.0):
        x = np.round(10000 * np.sin(2 * np.pi * f * t / FS)).astype(np.int16)
        frames, st = pr.analyse(x, FS)
        assert st["voiced"] == st["frames"] == 96, f
        assert abs(st["f0_mean_hz"] / f - 1) < 5e-4 and st["f0_sd_hz"] < 0.01 * f, (f, st)
        assert st["strength_mean"] > 0.998 and st["hnr_mean_db"] > 25, (f, st)


def test_restatement_impulse_train_integer_period():
    for T in (60, 150, 257):
        x = np.zeros(FS, dtype=np.int16)
        x[7::T] = 10000
        frames, st = pr.analyse(x, FS)
        assert st["voiced"] == st["frames"], T
        assert all(abs(f["tau"] - T) < 1e-6 and f["tau_int"] == T for f in frames), T
        assert abs(st["f0_mean_hz"] - FS / T) < 1e-6 * FS / T


def test_restatement_white_noise_is_unvoiced():
    x = np.random.default_rng(1).integers(-5000, 5000, FS).astype(np.int16)
    frames, st = pr.analyse(x, FS)
    assert st["voiced"] == 0 and st["periodic"] > 0
    assert st["strength_mean"] < 0.3 and st["hnr_mean_db"] < -3


def test_restatement_silence_and_dc_are_silent():
    for v in (0, 1234, -32768):
        frames, st = pr.analyse(np.full(5000, v, dtype=np.int16), FS)
        assert st["frames"] == 19 and st["periodic"] == st["voiced"] == 0
        assert all(f["flags"] == pr.SILENT for f in frames)
        assert all(math.isnan(st[k]) for k in ("f0_mean_hz", "f0_sd_hz", "f0_min_hz", "f0_max_hz", "hnr_mean_db",
                                                "hnr_sd_db", "strength_mean"))


def test_restatement_quiet_frames():
    """a voice that fades to a whisper: the frames whose local peak falls below 3 % of the stream's peak are QUIET"""
    t = np.arange(2 * FS)
    x = np.round(10000 * np.sin(2 * np.pi * 150 * t / FS) * np.where(t < FS, 1.0, 0.01)).astype(np.int16)
    frames, st = pr.analyse(x, FS)
    G = max(f["peak"] for f in frames)
    assert [f["flags"] == pr.QUIET for f in frames] == [f["peak"] < 0.03 * G for f in frames]
    assert 0 < sum(f["flags"] == pr.QUIET for f in frames) < st["frames"]


def test_window_correction():
    """for a periodic frame r(T) is 1 up to the signal's own rounding: the window's autocorrelation is divided out.
    Without the correction the normalised autocorrelation at one period is r_w(T) / r_w(0), 0.83 here."""
    T = 147
    x = np.round(8000 * np.sin(2 * np.pi * np.arange(FS) / T) + 4000 * np.sin(6 * np.pi * np.arange(FS) / T)).astype(np.int16)
    Nw, _, tau_lo, tau_hi = pr.geometry(FS, pr.DEFAULTS)
    r, _, _ = pr.lag_curve(x[:Nw], Nw, tau_lo, tau_hi)
    corrected = r[T - (tau_lo - 1)]
    raw = corrected / pr.correction(Nw, tau_lo, tau_hi)[T - (tau_lo - 1)]
    assert abs(corrected - 1) < 1e-4 and raw < 0.85
    w = pr.window(Nw)
    assert abs(pr.r_w(w, T) / pr.r_w(w, 0) - raw) < 1e-3


# closed loop, measured with scripts/pitch_accuracy.py (DESIGN 4.2e): per preset, the largest |mean voiced F0 / (fs / mean
# T) - 1| over F0 = 100, 120, 150, 200 Hz with jitter 1 % and shimmer 3 %; per `vowel -n` SNR, the band of the mean HNR
F0_BOUND = {"a": 0.025, "i": 0.04, "u": 0.011, "1": 0.022, "2": 0.007, "3": 0.012, "4": 0.022, "5": 0.14, "6": 0.022,
            "7": 0.016}
HNR_BAND = {10.0: (9.5, 13.7), 20.0: (19.5, 24.5), 30.0: (25.0, 34.6)}
F0S = (100, 120, 150, 200)


def _flow(oracle, f0, jitter):
    a = ["-o", "x", "-d", "1", "-f", str(f0), "-g", str(f0 + 30)] + (["-j", "1", "-s", "3"] if jitter else [])
    return oracle.flowgen(oracle.flow_par_from_cli(a, 7), want_log=True)


@pytest.mark.parametrize("preset", list(F0_BOUND))
def test_closed_loop_f0(oracle, preset):
    for f0 in F0S:
        x, log = _flow(oracle, f0, True)
        _, st = pr.analyse(oracle.vowel(x, preset), FS)
        assert st["voiced"] == st["frames"] == 96, (preset, f0)
        assert abs(st["f0_mean_hz"] / (FS / np.mean(log["T"])) - 1) <= F0_BOUND[preset], (preset, f0, st["f0_mean_hz"])


@pytest.mark.parametrize("snr", list(HNR_BAND))
def test_closed_loop_hnr(oracle, snr):
    lo, hi = HNR_BAND[snr]
    for preset in "aiu1234567":
        for f0 in F0S:
            x, _ = _flow(oracle, f0, False)
            _, st = pr.analyse(oracle.vowel_noise(x, preset, snr, 3), FS)
            assert lo <= st["hnr_mean_db"] <= hi, (snr, preset, f0, st["hnr_mean_db"])
