"""TEST ONLY: numpy restatement of vs_formant_batch's definitions (include/voicesynth.h), written from the header.

Per stream: frames of Nw = lround(win_ms fs / 1000) samples every H = lround(hop_ms fs / 1000); pre-emphasis with the
real previous sample (x[-1] = 0 only at the stream's first sample), a Hamming window, the FP64 autocorrelation, the
Levinson-Durbin recursion in Python floats, np.roots for the poles, then selection and per-stream statistics.

SINGULAR is only a numerical guard: for a frame that is not all zero the autocorrelation-method Toeplitz matrix is
positive definite, so every reflection coefficient has |k_i| < 1 and the prediction error stays positive.  No input is
known to reach it; the restatement flags it the way the header says and no test builds one.

A frame is AMBIGUOUS when a root with Im z > 0 lies within 1e-6 relative of a selection boundary (50 Hz, fs/2 - 50 Hz
or bmax): there the library's root finder and np.roots may legitimately choose differently.  The GPU comparison skips
such frames."""
import math

import numpy as np

MAX_FORMANTS = 8
SILENT, SINGULAR, NOCONV = 1, 2, 4
DEFAULTS = dict(win_ms=25.0, hop_ms=10.0, preemph_hz=50.0, bmax_hz=700.0, order=14, n_formants=5)
AMBIG_REL = 1e-6


def opts_with(**kw):
    o = dict(DEFAULTS)
    o.update(kw)
    return o


def lround(x):
    return int(math.floor(x + 0.5)) if x >= 0 else -int(math.floor(-x + 0.5))


def geometry(fs, o):
    """(Nw, H) of a stream at rate fs; the option floats are float32 in the C struct"""
    Nw = lround(float(np.float32(o["win_ms"])) * fs / 1000.0)
    H = lround(float(np.float32(o["hop_ms"])) * fs / 1000.0)
    return Nw, H


def n_frames(n, Nw, H):
    return (n - Nw) // H + 1 if n >= Nw else 0


def window(Nw):
    return np.array([0.54 - 0.46 * math.cos(2.0 * math.pi * m / (Nw - 1)) for m in range(Nw)])


def preemph_mu(fs, o):
    ph = float(np.float32(o["preemph_hz"]))
    return math.exp(-2.0 * math.pi * ph / fs) if ph > 0 else 0.0


def frame_signal(x, f, Nw, H, mu, w):
    """the windowed, pre-emphasised frame f of stream x"""
    s = f * H
    cur = x[s: s + Nw].astype(np.float64)
    prev = np.empty(Nw)
    prev[1:] = x[s: s + Nw - 1]
    prev[0] = float(x[s - 1]) if s > 0 else 0.0
    return (cur - mu * prev) * w


def autocorr(y, p):
    return [float(np.dot(y[: len(y) - k], y[k:])) for k in range(p + 1)]


def levinson(r, p):
    """a[1..p] of A(z) = 1 + a1 z^-1 + ... + ap z^-p, or None when the recursion is singular"""
    a = [0.0] * (p + 1)
    E = r[0]
    for i in range(1, p + 1):
        acc = r[i]
        for j in range(1, i):
            acc += a[j] * r[i - j]
        k = -acc / E
        if not abs(k) < 1.0:
            return None
        prev = a[:]
        for j in range(1, i):
            a[j] = prev[j] + k * prev[i - j]
        a[i] = k
        E *= 1.0 - k * k
        if not E > 0.0:
            return None
    return a[1:]


def select(roots, fs, o):
    """(F, B) of the kept roots in ascending F, the first n_formants of them, and whether the frame is ambiguous"""
    bmax = float(np.float32(o["bmax_hz"]))
    lo, hi = 50.0, fs / 2.0 - 50.0
    kept, ambiguous = [], False
    for z in roots:
        if not z.imag > 0:
            continue
        F = math.atan2(z.imag, z.real) * fs / (2.0 * math.pi)
        B = -math.log(abs(z)) * fs / math.pi
        near = lambda v, edge: abs(v - edge) <= AMBIG_REL * abs(edge)
        if near(F, lo) or near(F, hi) or (bmax > 0 and near(B, bmax)):
            ambiguous = True
        if lo < F < hi and (bmax <= 0 or B < bmax):
            kept.append((F, B))
    kept.sort()
    return kept[: int(o["n_formants"])], ambiguous


def analyse_frame(y, fs, o):
    """{'F', 'B' (lists, unrounded), 'flags', 'ambiguous'} of one windowed frame"""
    p = int(o["order"])
    r = autocorr(y, p)
    if r[0] == 0.0:
        return dict(F=[], B=[], flags=SILENT, ambiguous=False)
    a = levinson(r, p)
    if a is None:
        return dict(F=[], B=[], flags=SINGULAR, ambiguous=False)
    kept, amb = select(np.roots([1.0] + a), fs, o)
    return dict(F=[k[0] for k in kept], B=[k[1] for k in kept], flags=0, ambiguous=amb)


def analyse(x, fs=22050, o=None):
    """(list of per-frame dicts, stats dict) of one stream"""
    o = o or DEFAULTS
    x = np.asarray(x, dtype=np.int16)
    Nw, H = geometry(fs, o)
    w, mu = window(Nw), preemph_mu(fs, o)
    frames = [analyse_frame(frame_signal(x, f, Nw, H, mu, w), fs, o) for f in range(n_frames(len(x), Nw, H))]
    return frames, stats(frames, o)


def stats(frames, o):
    nf = int(o["n_formants"])
    good = [fr for fr in frames if fr["flags"] == 0]
    st = dict(frames=len(frames), analysed=len(good), unconverged=sum(1 for fr in frames if fr["flags"] & NOCONV),
              count=[0] * MAX_FORMANTS, f_mean_hz=[math.nan] * MAX_FORMANTS, f_sd_hz=[math.nan] * MAX_FORMANTS,
              bw_mean_hz=[math.nan] * MAX_FORMANTS)
    for k in range(nf):
        F = [fr["F"][k] for fr in good if len(fr["F"]) > k]
        B = [fr["B"][k] for fr in good if len(fr["B"]) > k]
        st["count"][k] = len(F)
        if F:
            m = math.fsum(F) / len(F)
            st["f_mean_hz"][k] = m
            st["bw_mean_hz"][k] = math.fsum(B) / len(B)
            if len(F) >= 2:
                st["f_sd_hz"][k] = math.sqrt(math.fsum((v - m) ** 2 for v in F) / (len(F) - 1))
    return st
