"""TEST ONLY: numpy restatement of vs_vowel_report_batch's definitions (include/voicesynth.h), written from the header.

It takes a stream's pitch frame records (flags and float f0_hz, as vs_pitch_batch returns them, or as pitch_ref computes
them) and the PCM, finds the longest voiced run, walks the period marks by cross-correlation with exact Python-integer
sums and the same IEEE double operations as the device, and computes the voice report on the marks with report_ref's
formulas.  So the marks of the GPU can be compared mark for mark with the restatement fed the GPU's own frame records."""
import math

import numpy as np

import pitch_ref as pr
import report_ref as rr

STEP_MIN, STEP_MAX = 0.8, 1.25


def lround(v):
    """C's lround of a positive double (halves away from zero), exactly"""
    f = math.floor(v)
    return int(f) + (1 if v - f >= 0.5 else 0)


def run(flags):
    """(f_a, frames) of the longest run of VOICED frames, the first of equal ones; (0, 0) without a voiced frame"""
    best, start, cur = (0, 0), 0, 0
    for f, fl in enumerate(flags):
        if int(fl) == pr.VOICED:
            if cur == 0:
                start = f
            cur += 1
            if cur > best[1]:
                best = (start, cur)
        else:
            cur = 0
    return best


def mark_slots(n, fs=22050, o=None):
    """vs_vowel_mark_slots of one stream"""
    Nw, _, tau_lo, _ = pr.geometry(fs, o or pr.DEFAULTS)
    if n < Nw:
        return 0
    step = lround(STEP_MIN * ((tau_lo - 0.5) * (1.0 - 2.0 ** -20)))
    return (n - 1) // step + 1


def marks(x, flags, f0_hz, fs=22050, o=None):
    """(marks, (run_frame, run_frames, run_start, run_len)) of one stream from its frame records"""
    Nw, H, _, _ = pr.geometry(fs, o or pr.DEFAULTS)
    fa, nrun = run(flags)
    if nrun == 0:
        return [], (0, 0, 0, 0)
    fb = fa + nrun - 1
    s, e = fa * H, fb * H + Nw
    xi = np.asarray(x, dtype=np.int64)
    f0 = np.asarray(f0_hz, dtype=np.float32)

    def period(t):
        f = (t - Nw // 2 + H // 2) // H                        # Python's // floors, as the definition asks
        return float(fs) / float(f0[min(max(f, fa), fb)])

    c = s + Nw // 2
    L = lround(period(c))
    a0 = c - L // 2
    m = a0 + int(np.argmax(np.abs(xi[a0: a0 + L])))            # argmax: the first of equal values
    return walk(xi, m, e, period), (fa, nrun, s, e - s)


def walk(xi, m, e, period):
    """the marks from m_0 = m on: the step rule up to the run's end e; period(t) is T(t); xi int64 samples whose index
    0 is the stream's (or any) origin of m, e and t"""
    out = [m]
    while True:
        T = period(m)
        L = lround(T)
        lo, hi = m + lround(STEP_MIN * T), m + lround(STEP_MAX * T)
        if hi + L > e:
            break
        ref = xi[m: m + L]
        e0 = int(ref @ ref)
        best_r, best_m = -math.inf, None
        for c in range(lo, hi + 1):
            seg = xi[c: c + L]
            C, E = int(ref @ seg), int(seg @ seg)            # < 2^42: exact in int64
            den = float(e0) * float(E)
            r = 0.0 if den == 0.0 else float(C) / math.sqrt(den)
            if r > best_r:
                best_r, best_m = r, c
        if not best_r > 0.0:
            break
        m = best_m
        out.append(m)
    return out


def report_on_marks(x, o, fs=22050):
    """the vs_flow_report fields (report_ref.report's dict) of the cycles between consecutive marks o"""
    o = np.asarray(o, dtype=np.int64)
    xi = np.asarray(x, dtype=np.int64)
    K = max(len(o) - 1, 0)
    base = {"onsets": len(o), "cycles": K, "flags": 0, "f0_hz": 0.0, "jitter_pct": 0.0, "shimmer_pct": 0.0,
            "mean_period": 0.0, "mean_peak": 0.0}
    out = dict.fromkeys(rr.FIELDS, rr.NAN)
    out["base"], out["hnr_len"] = base, 0
    if K == 0:
        return out
    T = np.diff(o)
    P = np.array([xi[o[k]: o[k + 1]].max() for k in range(K)], dtype=np.int64)
    mT, mP = int(T.sum()) / K, int(P.sum()) / K
    base.update(mean_period=mT, mean_peak=mP, f0_hz=fs / mT)
    if K >= 2:
        base["jitter_pct"] = 100.0 * (int(np.abs(np.diff(T)).sum()) / (K - 1)) / mT
        base["shimmer_pct"] = 100.0 * (int(np.abs(np.diff(P)).sum()) / (K - 1)) / mP if mP != 0 else 0.0
        out["jitter_abs_us"] = 1e6 * (int(np.abs(np.diff(T)).sum()) / (K - 1)) / fs
        if (P > 0).all():
            out["shimmer_db"] = float(np.abs(20.0 * np.log10(P[1:] / P[:-1])).sum()) / (K - 1)
        L, Hs, E = rr.hnr_sums(x, o)
        out["hnr_db"], out["hnr_len"] = rr.hnr_db(K, Hs, E), L
    if K >= 3:
        out["jitter_rap_pct"] = 100.0 * (rr._ppq(T, 3) / 3 / (K - 2)) / mT
        out["jitter_ddp_pct"] = 100.0 * (rr._ddp(T) / (K - 2)) / mT
        if mP > 0:
            out["shimmer_apq3_pct"] = 100.0 * (rr._ppq(P, 3) / 3 / (K - 2)) / mP
            out["shimmer_dda_pct"] = 100.0 * (rr._ddp(P) / (K - 2)) / mP
    if K >= 5:
        out["jitter_ppq5_pct"] = 100.0 * (rr._ppq(T, 5) / 5 / (K - 4)) / mT
        if mP > 0:
            out["shimmer_apq5_pct"] = 100.0 * (rr._ppq(P, 5) / 5 / (K - 4)) / mP
    if K >= 11 and mP > 0:
        out["shimmer_apq11_pct"] = 100.0 * (rr._ppq(P, 11) / 11 / (K - 10)) / mP
    return out


def frame_records(x, fs=22050, o=None):
    """(flags, f0_hz float32) of pitch_ref's frames of one stream, as vs_pitch_batch publishes them"""
    frames, _ = pr.analyse(x, fs, o)
    flags = np.array([f["flags"] for f in frames], dtype=np.uint32)
    f0 = np.array([f["f0"] for f in frames], dtype=np.float64).astype(np.float32)
    return flags, f0


def analyse(x, fs=22050, o=None, records=None):
    """(marks, run, report dict) of one stream; records: its (flags, f0_hz) frame records, else pitch_ref's"""
    flags, f0 = records if records is not None else frame_records(x, fs, o)
    mk, rn = marks(x, flags, f0, fs, o)
    return mk, rn, report_on_marks(x, mk, fs)
