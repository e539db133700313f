"""The voice report's definitions (include/voicesynth.h, vs_flow_report_batch) as tests/report_ref.py states them, on
the CPU: closed forms on hand-built pulse trains, where each measure starts to exist, a stream whose sum of S_j^2
needs more than 64 bits, and the HNR of the oracle's noise-only voices against the SNR of the generator's period log."""
import math

import numpy as np
import pytest

import analysis_ref as ar
import report_ref as rr


def _alternating(a, b, K):
    return np.array([a if k % 2 == 0 else b for k in range(K)], dtype=np.int64)


def test_pulse_train_has_the_cycles_it_was_built_from():
    rng = np.random.default_rng(3)
    T, P = rng.integers(3, 300, 40), rng.integers(1, 32000, 40)
    x = rr.pulse_train(T, P)
    o, T2, P2 = rr.cycles(x)
    assert np.array_equal(T2, T) and np.array_equal(P2, P) and o[0] == 0
    st = ar.stats(x)
    assert st["cycles"] == 40 and st["flags"] == 0


@pytest.mark.parametrize("a,b,p,q", [(100, 110, 9000, 8000), (183, 147, 3000, 3600), (50, 51, 20000, 19999)])
def test_alternating_cycles_closed_forms(a, b, p, q):
    """periods a, b, a, b, ... and peaks p, q, p, q, ... over an even number of cycles"""
    K, fs = 24, 22050
    rep = rr.report(rr.pulse_train(_alternating(a, b, K), _alternating(p, q, K)), fs=fs)
    mT, mP = (a + b) / 2, (p + q) / 2
    want = {
        "jitter_abs_us": 1e6 * abs(a - b) / fs,
        "jitter_rap_pct": 100 * (2 * abs(a - b) / 3) / mT,
        "jitter_ppq5_pct": 100 * (2 * abs(a - b) / 5) / mT,
        "jitter_ddp_pct": 100 * (2 * abs(a - b)) / mT,
        "shimmer_db": abs(20 * math.log10(p / q)),
        "shimmer_apq3_pct": 100 * (2 * abs(p - q) / 3) / mP,
        "shimmer_apq5_pct": 100 * (2 * abs(p - q) / 5) / mP,
        "shimmer_apq11_pct": 100 * (6 * abs(p - q) / 11) / mP,      # a window holds 5 of its centre's peak, 6 of the other
        "shimmer_dda_pct": 100 * (2 * abs(p - q)) / mP,
    }
    for k, v in want.items():
        assert math.isclose(rep[k], v, rel_tol=1e-9), (k, rep[k], v)
    assert rep["jitter_ddp_pct"] == pytest.approx(3 * rep["jitter_rap_pct"], rel=1e-15)
    assert rep["shimmer_dda_pct"] == pytest.approx(3 * rep["shimmer_apq3_pct"], rel=1e-15)
    assert rep["hnr_len"] == min(a, b) and math.isfinite(rep["hnr_db"])
    assert rep["base"]["jitter_pct"] == pytest.approx(100 * abs(a - b) / mT)


def test_constant_cycles_give_zero_quotients_and_infinite_hnr():
    rep = rr.report(rr.pulse_train([137] * 30, [12000] * 30))
    for k in rr.FIELDS[:-1]:
        assert rep[k] == 0.0, k
    assert rep["hnr_db"] == math.inf and rep["hnr_len"] == 137


@pytest.mark.parametrize("K", [0, 1, 2, 3, 4, 5, 10, 11])
def test_where_each_measure_starts_to_exist(K):
    rng = np.random.default_rng(K)
    x = rr.pulse_train(rng.integers(20, 200, K), rng.integers(100, 30000, K))
    rep = rr.report(x)
    assert rep["base"]["cycles"] == K
    need = {"jitter_abs_us": 2, "shimmer_db": 2, "hnr_db": 2, "jitter_rap_pct": 3, "jitter_ddp_pct": 3, "shimmer_apq3_pct": 3,
            "shimmer_dda_pct": 3, "jitter_ppq5_pct": 5, "shimmer_apq5_pct": 5, "shimmer_apq11_pct": 11}
    for k in rr.FIELDS:
        assert math.isnan(rep[k]) == (K < need[k]), (K, k, rep[k])
    assert (rep["hnr_len"] > 0) == (K >= 2)


def test_nonpositive_peak_leaves_shimmer_db_undefined():
    """thresholds below zero: a cycle whose peak is 0 has no level in dB"""
    x = np.array([0, -5, 3, 1, -5, 0, -1, -5, 4, -5, 0] + [-5] * 60, dtype=np.int16)
    rep = rr.report(x, lo=-5, hi=-2)
    _, T, P = rr.cycles(x, -5, -2)
    assert len(T) == 4 and (P <= 0).any() and P.sum() > 0
    assert math.isnan(rep["shimmer_db"]) and math.isfinite(rep["shimmer_apq3_pct"])


def test_overflow_leaves_every_new_field_undefined():
    x = np.zeros(4096, dtype=np.int16)
    x[::2] = 5
    rep = rr.report(x)
    assert rep["base"]["flags"] == 1 and rep["hnr_len"] == 0 and all(math.isnan(rep[k]) for k in rr.FIELDS)


def test_hnr_sums_beyond_64_bits():
    """40 000 cycles of peaks near full scale: sum_j S_j^2 exceeds 2^64, K*E exceeds it as well; the integers stay exact"""
    K = 40000
    x = rr.pulse_train([100] * K, _alternating(30000, 29990, K))
    o, T, P = rr.cycles(x)
    L, H, E = rr.hnr_sums(x, o)
    assert L == 100 and H > 2 ** 64 and K * E > 2 ** 64
    assert K * E - H > 0
    # the same number in floating point (loses the low bits, not the ratio)
    M = np.stack([x[o[k]: o[k] + L].astype(np.float64) for k in range(K)])
    S = M.sum(0)
    approx = 10 * math.log10((S * S).sum() / (K * (M * M).sum() - (S * S).sum()))
    assert rr.report(x)["hnr_db"] == pytest.approx(approx, rel=1e-6)


NOISE_ONLY = [["-n", "20"], ["-n", "30"], ["-n", "40"], ["-n", "25", "-f", "200", "-g", "230", "-r", "44100"],
              ["-n", "35", "-f", "90", "-g", "120", "-a", "5000"], ["-n", "30", "-r", "44100", "-a", "20000"]]


def period_log_snr(log, K):
    """SNR the generator logged over the first K pitch periods: open-phase power x span over noise power x period"""
    lg = log[:K]
    return 10 * math.log10(float((lg["x_pow"].astype(np.float64) * (lg["T3"] - lg["T4"])).sum()) /
                           float((lg["w_pow"].astype(np.float64) * lg["T"]).sum()))


def noise_only_voice(oracle, args, seed):
    par = oracle.flow_par_from_cli(["-o", "x.wav", "-d", "2"] + args, seed=seed)
    flow, log = oracle.flowgen(par, want_log=True)
    amp = int(par.amp)
    return flow, log, int(par.fs), int(amp * 0.08), int(amp * 0.15)


@pytest.mark.parametrize("args", NOISE_ONLY, ids=lambda a: "_".join(a).replace("-", ""))
def test_hnr_of_noise_only_voices_is_the_logged_snr(oracle, args):
    flow, log, fs, lo, hi = noise_only_voice(oracle, args, 7)
    rep = rr.report(flow, fs=fs, lo=lo, hi=hi)
    K = rep["base"]["cycles"]
    assert K > 100 and abs(K - len(log)) <= 2
    assert abs(rep["hnr_db"] - period_log_snr(log, K)) < 0.1, (args, rep["hnr_db"], period_log_snr(log, K))
