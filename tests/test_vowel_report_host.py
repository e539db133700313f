"""Voice report of vowel PCM without a GPU: vs_vowel_mark_slots through the library (the slot bound and every refusal),
the numpy restatement of the marks (tests/vowel_report_ref.py) on synthetic rows whose periods are known, and the closed
loop on oracle voices without jitter: the marks' periods against the period log."""
import math

import numpy as np
import pytest

import pitch_ref as pr
import report_ref as rr
import vowel_report_ref as vr
from voice_synth_b200 import api

FS = 22050


def synthetic_rows():
    """(rows, the periods each row's marks must have or None): a repeated int16 waveform with a constant period, pulses of
    a known period sequence through a short fixed FIR, silence, and two voiced stretches around silence (the longer
    second one is analysed)"""
    t = np.arange(FS)
    wave_ = np.round(9000 * np.sin(2 * np.pi * t[:147] / 147) + 4000 * np.sin(6 * np.pi * t[:147] / 147 + 0.5)).astype(np.int16)
    periodic = np.resize(wave_, FS)
    T = 140 + np.round(3 * np.sin(np.arange(160) / 4.0)).astype(np.int64)     # slow enough for the pitch track's window
    onsets = np.concatenate([[0], np.cumsum(T)])
    onsets = onsets[onsets < FS - 200]
    pulses = np.zeros(FS)
    pulses[onsets] = 7000
    fir = np.array([1.0, 0.6, -0.5, -0.7, 0.2, 0.4, -0.1, -0.2])
    train = np.round(np.convolve(pulses, fir)[:FS]).astype(np.int16)
    stretches = np.zeros(2 * FS, np.int16)
    stretches[2000:8000] = periodic[:6000]
    stretches[12000:30000] = periodic[:18000]
    return [periodic, train, np.zeros(5000, np.int16), stretches], [147, np.diff(onsets), None, 147]


def test_mark_slots_bound_and_refusals():
    for fs in (8000, 22050, 44100):
        Nw, H, tau_lo, _ = pr.geometry(fs, pr.DEFAULTS)
        ns = [0, Nw - 1, Nw, fs, 2 ** 31 - 1]
        got = api.vowel_mark_slots(ns, fs)
        assert list(got) == [vr.mark_slots(n, fs) for n in ns]
        assert list(got[:3]) == [0, 0, (Nw - 1) // vr.lround(0.8 * (tau_lo - 0.5) * (1 - 2.0 ** -20)) + 1]
    # the extreme f_max: tau_lo = 2, a step of 1, a slot per sample
    for f_max in (11025.0, 22050.0, 1e9):
        assert list(api.vowel_mark_slots([5000, 22050], FS, dict(f_max_hz=f_max))) == [5000, 22050]
    # the refusals of vs_pitch_frames, in the same order
    for o in (dict(f_min_hz=0.0), dict(f_max_hz=75.0), dict(periods=1.5), dict(silence_threshold=1.5), dict(octave_cost=-1.0),
              dict(f_min_hz=5.0), dict(hop_ms=0.01)):
        with pytest.raises(api.VsError) as a:
            api.vowel_mark_slots([5000], FS, o)
        with pytest.raises(api.VsError) as b:
            api.pitch_frames([5000], FS, o)
        assert a.value.args == b.value.args, o
    for ns, fs in (([2 ** 31], None), ([5000, 5000], [22050, 0])):
        with pytest.raises(api.VsError) as a:
            api.vowel_mark_slots(ns, fs)
        with pytest.raises(api.VsError) as b:
            api.pitch_frames(ns, fs)
        assert a.value.args == b.value.args


def test_run_rule():
    V, Q = pr.VOICED, pr.QUIET
    assert vr.run([]) == (0, 0) and vr.run([Q, 0, Q]) == (0, 0)
    assert vr.run([V, V, Q, V, V, V, 0, V, V, V]) == (3, 3)          # the first of two equal longest runs
    assert vr.run([Q, V, V, V, V]) == (1, 4)


def test_restatement_periodic_waveform():
    """a fixed waveform repeated every 147 samples: equal spacing, no jitter or shimmer, an HNR of +inf"""
    rows, want = synthetic_rows()
    mk, rn, rep = vr.analyse(rows[0], FS)
    assert rn[:2] == (0, pr.n_frames(FS, *pr.geometry(FS, pr.DEFAULTS)[:2]))
    assert set(np.diff(mk).tolist()) == {want[0]} and len(mk) >= 140
    b = rep["base"]
    assert (b["jitter_pct"], b["shimmer_pct"], rep["jitter_abs_us"], rep["shimmer_apq3_pct"]) == (0.0, 0.0, 0.0, 0.0)
    assert rep["hnr_db"] == math.inf and rep["hnr_len"] == 147


def test_restatement_known_period_sequence():
    """pulses of periods 137..143 through a fixed FIR: the marks are one per pulse, at a fixed offset from it"""
    rows, want = synthetic_rows()
    mk, rn, rep = vr.analyse(rows[1], FS)
    d = np.diff(mk)
    T = want[1]
    # the run begins inside the train: find the pulse the first mark follows, then every period after it
    k0 = int(np.searchsorted(np.concatenate([[0], np.cumsum(T)]), mk[0], side="right")) - 1
    assert np.array_equal(d, T[k0: k0 + len(d)]), (d[:20], T[k0: k0 + 20])
    assert len(d) >= 120
    assert rep["base"]["cycles"] == len(d) and rep["base"]["jitter_pct"] > 0.3


def test_restatement_silence_and_stretches():
    rows, _ = synthetic_rows()
    mk, rn, rep = vr.analyse(rows[2], FS)
    assert mk == [] and rn == (0, 0, 0, 0)
    assert rep["base"]["onsets"] == rep["base"]["cycles"] == 0 and math.isnan(rep["hnr_db"])
    Nw, H, _, _ = pr.geometry(FS, pr.DEFAULTS)
    flags, f0 = vr.frame_records(rows[3], FS)
    fa, nrun = vr.run(flags)
    assert fa * H >= 12000 - Nw and (fa + nrun - 1) * H + Nw <= 30000 + Nw      # the second, longer stretch
    mk, rn, _ = vr.analyse(rows[3], FS, records=(flags, f0))
    d = np.diff(mk)            # the last period may reach into the silence that the last frame's window covers
    assert rn[:2] == (fa, nrun) and mk[0] >= rn[2] and set(d[:-1].tolist()) == {147} and len(d) >= 100


# closed loop, measured with scripts/vowel_report_accuracy.py (DESIGN 4.2f): voices without jitter, shimmer or noise give
# marks whose periods equal the period log's in at least 98 % of the periods (the rest: octave errors of the pitch track at
# the run's start) and a PCM jitter of at most 0.2 %
@pytest.mark.parametrize("preset", ["a", "i", "u", "3", "7"])
def test_closed_loop_constant_period(oracle, preset):
    for f0 in (100, 150, 200):
        flow, log = oracle.flowgen(oracle.flow_par_from_cli(["-o", "x", "-d", "1", "-f", str(f0), "-g", str(f0 + 30), "-a", "6000"], 7),
                                   want_log=True)
        assert len(set(np.asarray(log["T"]).tolist())) == 1
        pcm = oracle.vowel(flow, preset)
        mk, rn, rep = vr.analyse(pcm, FS)
        d = np.diff(mk)
        share = float(np.mean(d == int(log["T"][0])))
        assert share >= 0.98, (preset, f0, share)
        assert rep["base"]["jitter_pct"] <= 0.2, (preset, f0, rep["base"]["jitter_pct"])
        assert rr.report(flow, FS)["base"]["jitter_pct"] == 0.0
