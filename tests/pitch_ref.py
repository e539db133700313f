"""TEST ONLY: numpy restatement of vs_pitch_batch's definitions (include/voicesynth.h), written from the header.

Per stream: frames of Nw = lround(periods fs / f_min) samples every H = lround(hop_ms fs / 1000); the frame's mean
removed (an exact integer sum), the Hann-like window w[m] = 0.5 - 0.5 cos(2 pi (m + 1/2) / Nw), the FP64
autocorrelation divided by r_a(0) and corrected by r_w(0) / r_w(tau) (w and r_w from libm through Python's math module,
r_w summed in index order by np.cumsum, as the library's host does), the candidates with parabolic refinement and
octave cost, then the per-stream QUIET / VOICED rules and statistics.

The device sums r_a in its own order, so r(tau) differs from this restatement in the last bits.  `margin` is how far a
frame is from a decision that such a difference could flip: the smallest gap of a candidate test (r(tau) against its
neighbours and against 0, where the candidate it makes or unmakes could reach the winner's strength: the refined r* of
a peak is at most 1.25 times the largest of its three values), the gap between the two strongest candidates, and r*
against the voicing threshold.  The GPU
comparison requires identical decisions wherever the margin exceeds MARGIN."""
import functools
import math

import numpy as np

SILENT, NOPEAK, QUIET, VOICED = 1, 2, 4, 8
DEFAULTS = dict(f_min_hz=75.0, f_max_hz=600.0, periods=3.0, hop_ms=10.0, voicing_threshold=0.45, silence_threshold=0.03,
                octave_cost=0.01)
MAX_WIN = 4096
MARGIN = 1e-9


def opts_with(**kw):
    o = dict(DEFAULTS)
    o.update(kw)
    return o


def f32(v):
    """an option as the C struct holds it"""
    return float(np.float32(v))


def lround(x):
    return int(math.floor(x + 0.5)) if x >= 0 else -int(math.floor(-x + 0.5))


def geometry(fs, o):
    """(Nw, H, tau_lo, tau_hi) of a stream at rate fs"""
    Nw = lround(f32(o["periods"]) * fs / f32(o["f_min_hz"]))
    H = lround(f32(o["hop_ms"]) * fs / 1000.0)
    tau_lo = max(2, math.ceil(fs / f32(o["f_max_hz"])))
    tau_hi = math.floor(fs / f32(o["f_min_hz"]))
    return Nw, H, tau_lo, tau_hi


def n_frames(n, Nw, H):
    return (n - Nw) // H + 1 if n >= Nw else 0


@functools.lru_cache(maxsize=None)
def window(Nw):
    return np.array([0.5 - 0.5 * math.cos(2.0 * math.pi * (m + 0.5) / Nw) for m in range(Nw)])


def r_w(w, tau):
    return float(np.cumsum(w[: len(w) - tau] * w[tau:])[-1])


@functools.lru_cache(maxsize=None)
def correction(Nw, tau_lo, tau_hi):
    """r_w(0) / r_w(tau) for tau = tau_lo-1 .. tau_hi+1"""
    w = window(Nw)
    rw0 = r_w(w, 0)
    return np.array([rw0 / r_w(w, t) for t in range(tau_lo - 1, tau_hi + 2)])


def lag_curve(seg, Nw, tau_lo, tau_hi):
    """(r(tau) for tau = tau_lo-1 .. tau_hi+1, P_f, r_a(0)) of one frame of int16 samples"""
    mu = int(np.asarray(seg, dtype=np.int64).sum()) / Nw
    a = np.asarray(seg, dtype=np.float64) - mu
    y = a * window(Nw)
    ra = np.correlate(y, y, "full")[Nw - 1:]
    peak = float(np.abs(a).max())
    if ra[0] == 0.0:
        return None, peak, 0.0
    return (ra[tau_lo - 1: tau_hi + 2] / ra[0]) * correction(Nw, tau_lo, tau_hi), peak, float(ra[0])


def candidates(r, tau_lo, fs, o):
    """[(S, tau, tau*, r*)] in ascending tau; per tau the smallest gap of its candidate tests, and a bound above the
    strength it could have if a test flipped"""
    a, b, c = r[:-2], r[1:-1], r[2:]
    gap = np.minimum(np.minimum(np.abs(b - a), np.abs(b - c)), np.abs(b))
    out = []
    fmin, oc = f32(o["f_min_hz"]), f32(o["octave_cost"])
    taus = tau_lo + np.arange(len(b))
    reach = np.maximum(np.maximum(a, b), c) * 1.25 - oc * np.log2(fmin * (taus - 0.5) / fs)
    for i in np.nonzero((b > a) & (b >= c) & (b > 0.0))[0]:
        pa, pb, pc = float(a[i]), float(b[i]), float(c[i])
        d = 0.5 * (pa - pc) / (pa - 2.0 * pb + pc)
        t = tau_lo + int(i)
        ts = t + d
        rs = pb - 0.25 * (pa - pc) * d
        if rs > 1.0:
            rs = 1.0 / rs
        out.append((rs - oc * math.log2(fmin * ts / fs), t, ts, rs))
    return out, gap, reach


def analyse_frame(seg, fs, o):
    """{'tau', 'r', 'peak', 'flags' (SILENT / NOPEAK / 0), 'margin', 'tau_int'} of one frame"""
    Nw, _, tau_lo, tau_hi = geometry(fs, o)
    r, peak, _ = lag_curve(seg, Nw, tau_lo, tau_hi)
    if r is None:
        return dict(tau=math.nan, r=math.nan, peak=peak, flags=SILENT, margin=math.inf, tau_int=0)
    cands, gap, reach = candidates(r, tau_lo, fs, o)
    if not cands:
        return dict(tau=math.nan, r=math.nan, peak=peak, flags=NOPEAK, margin=float(gap.min()), tau_int=0)
    best = cands[0]
    for cd in cands[1:]:
        if cd[0] > best[0]:
            best = cd
    others = [cd[0] for cd in cands if cd is not best]
    # a flipped test matters where the candidate it makes or unmakes could reach the winner's strength
    near = gap[reach >= best[0]]
    margin = min([abs(best[3] - f32(o["voicing_threshold"]))] + ([float(near.min())] if near.size else []) +
                 ([best[0] - max(others)] if others else []))
    return dict(tau=best[2], r=best[3], peak=peak, flags=0, margin=margin, tau_int=best[1])


def hnr_db(r):
    return math.inf if r == 1.0 else 10.0 * math.log10(r / (1.0 - r))


def analyse(x, fs=22050, o=None):
    """(list of per-frame dicts with the stream rules applied: 'flags', 'f0', 'hnr' added, stats dict) of one stream"""
    o = o or DEFAULTS
    x = np.asarray(x, dtype=np.int16)
    Nw, H, _, _ = geometry(fs, o)
    frames = [analyse_frame(x[f * H: f * H + Nw], fs, o) for f in range(n_frames(len(x), Nw, H))]
    G = max((fr["peak"] for fr in frames), default=0.0)
    quiet = f32(o["silence_threshold"]) * G
    for fr in frames:
        fr["f0"] = fr["hnr"] = math.nan
        if not fr["flags"] and fr["peak"] < quiet:
            fr["flags"] = QUIET
        if not fr["flags"]:
            fr["hnr"] = hnr_db(fr["r"])
            if fr["r"] >= f32(o["voicing_threshold"]):
                fr["flags"] = VOICED
                fr["f0"] = fs / fr["tau"]
    return frames, stats(frames)


def _mean_sd(v):
    if not v:
        return math.nan, math.nan
    m = math.fsum(v) / len(v)
    if len(v) < 2:
        return m, math.nan
    return m, math.sqrt(math.fsum((u - m) ** 2 for u in v) / (len(v) - 1))      # an hnr of +inf: m = inf, the SD NaN


def stats(frames):
    voiced = [fr for fr in frames if fr["flags"] == VOICED]
    periodic = [fr for fr in frames if fr["flags"] in (0, VOICED)]
    f0 = [fr["f0"] for fr in voiced]
    f0_mean, f0_sd = _mean_sd(f0)
    hnr_mean, hnr_sd = _mean_sd([fr["hnr"] for fr in periodic])
    return dict(frames=len(frames), periodic=len(periodic), voiced=len(voiced), f0_mean_hz=f0_mean, f0_sd_hz=f0_sd,
                f0_min_hz=min(f0) if f0 else math.nan, f0_max_hz=max(f0) if f0 else math.nan, hnr_mean_db=hnr_mean,
                hnr_sd_db=hnr_sd, strength_mean=math.fsum(fr["r"] for fr in periodic) / len(periodic) if periodic else math.nan)
