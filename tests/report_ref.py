"""numpy restatement of vs_flow_report_batch (include/voicesynth.h): Praat's jitter and shimmer quotients over the cycles
of analysis_ref's trigger, and the cycle-synchronous HNR with exact Python-integer sums.  Written from the header's
definitions, independently of the CUDA kernel, for the tests."""
import math

import numpy as np

import analysis_ref as ar

NAN = float("nan")
FIELDS = ("jitter_abs_us", "jitter_rap_pct", "jitter_ppq5_pct", "jitter_ddp_pct", "shimmer_db", "shimmer_apq3_pct",
          "shimmer_apq5_pct", "shimmer_apq11_pct", "shimmer_dda_pct", "hnr_db")


def _ppq(v, w):
    """sum over k = h..K-1-h of |w v_k - (v_k-h + ... + v_k+h)|, h = w // 2, as a Python integer"""
    h = w // 2
    return sum(abs(w * int(v[k]) - int(v[k - h: k + h + 1].sum())) for k in range(h, len(v) - h))


def _ddp(v):
    return sum(abs(int(v[k + 1]) - 2 * int(v[k]) + int(v[k - 1])) for k in range(1, len(v) - 1))


def hnr_sums(x, o):
    """(L, sum_j S_j^2, E) over the cycles starting at o[0..K-1] (o[K] ends the last one), exact Python integers"""
    T = np.diff(o)
    L = int(T.min())
    xi = np.asarray(x, dtype=np.int64)
    M = np.stack([xi[int(o[k]): int(o[k]) + L] for k in range(len(T))])
    S = M.sum(0)                                             # |S_j| <= K * 32768: exact in int64
    H = sum(int(s) * int(s) for s in S)
    E = int((M * M).sum())
    return L, H, E


def hnr_db(K, H, E):
    D = K * E - H
    return math.inf if D == 0 else 10.0 * math.log10(H / D)


def cycles(x, lo=0, hi=0):
    """onsets, cycle lengths T_k and peaks P_k (int64) of the complete cycles"""
    o = ar.onsets(x, lo, hi)
    xi = np.asarray(x, dtype=np.int64)
    T = np.diff(o).astype(np.int64)
    P = np.array([xi[o[k]: o[k + 1]].max() for k in range(len(T))], dtype=np.int64)
    return o, T, P


def report(x, fs=22050, lo=0, hi=0):
    base = ar.stats(x, fs=fs, lo=lo, hi=hi)
    out = dict.fromkeys(FIELDS, NAN)
    out["base"] = base
    out["hnr_len"] = 0
    if base["flags"]:
        return out
    o, T, P = cycles(x, lo, hi)
    K = len(T)
    if K == 0:
        return out
    mT, mP = int(T.sum()) / K, int(P.sum()) / K
    if K >= 2:
        out["jitter_abs_us"] = 1e6 * (int(np.abs(np.diff(T)).sum()) / (K - 1)) / fs
        if (P > 0).all():
            out["shimmer_db"] = float(np.abs(20.0 * np.log10(P[1:] / P[:-1])).sum()) / (K - 1)
        L, H, E = hnr_sums(x, o)
        out["hnr_db"], out["hnr_len"] = hnr_db(K, H, E), L
    if K >= 3:
        out["jitter_rap_pct"] = 100.0 * (_ppq(T, 3) / 3 / (K - 2)) / mT
        out["jitter_ddp_pct"] = 100.0 * (_ddp(T) / (K - 2)) / mT
        if mP > 0:
            out["shimmer_apq3_pct"] = 100.0 * (_ppq(P, 3) / 3 / (K - 2)) / mP
            out["shimmer_dda_pct"] = 100.0 * (_ddp(P) / (K - 2)) / mP
    if K >= 5:
        out["jitter_ppq5_pct"] = 100.0 * (_ppq(T, 5) / 5 / (K - 4)) / mT
        if mP > 0:
            out["shimmer_apq5_pct"] = 100.0 * (_ppq(P, 5) / 5 / (K - 4)) / mP
    if K >= 11 and mP > 0:
        out["shimmer_apq11_pct"] = 100.0 * (_ppq(P, 11) / 11 / (K - 10)) / mP
    return out


def pulse_train(T, P, closed=0):
    """int16 flow whose trigger (lo = hi = closed) finds cycles of lengths T[k] and peaks P[k]: each cycle is a ramp
    from above `closed` up to P[k], then closed + 1 until its last sample, which is `closed` (that re-arms the
    trigger); one extra onset ends the last cycle"""
    x = []
    for t, p in zip(T, P):
        t, p = int(t), int(p)
        assert t >= 3 and p > closed
        up = (t - 1) // 2
        c = [closed + 1 + (p - closed - 1) * (i + 1) // up for i in range(up)]
        c = c + [closed + 1] * (t - 1 - len(c)) + [closed]
        x += c
    x += [closed + 1, closed]
    return np.asarray(x, dtype=np.int16)
