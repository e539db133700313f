"""Closed-loop accuracy of the voice report of vowel PCM (DESIGN 4.2f), on the CPU: python scripts/vowel_report_accuracy.py

1-second oracle voices (seed 7, amplitude 6000) go through the reference vowel filter, or through caller-defined formant tracts, and are
analysed with tests/vowel_report_ref.py (the restatement the GPU is pinned to) on pitch_ref's frame records, at the
default options.  The flow of the same voice goes through report_ref.report, whose periods are those of the period log.
Printed per filter and per (jitter, shimmer) level, the largest over F0 = 100, 150 and 200 Hz of:
  the PCM jitter_pct and shimmer_pct next to the flow's, and the smallest share of PCM periods that equal the logged
  period they start in.
Then the same with `vowel -n` output noise at 20 dB (seed 3)."""
import pathlib
import sys

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT), str(ROOT / "tests")]
import numpy as np

import report_ref as rr
import vowel_report_ref as vr
from oracle import pyoracle as O

FS = 22050
AMP = 6000          # at the default 12000 the filters clip shimmered voices at 32767, and clipped peaks read as no shimmer
F0S = (100, 150, 200)
LEVELS = ((0.0, 0.0), (1.0, 0.0), (3.0, 0.0), (0.0, 3.0), (0.0, 7.5), (1.0, 3.0), (3.0, 7.5))
TRACTS = {"Ta": ([730, 1090, 2440, 3400, 4500], [90, 110, 160, 250, 300]),
          "Ti": ([270, 2290, 3010, 3600, 4500], [60, 100, 170, 250, 300])}
FILTERS = list("aiu1234567") + list(TRACTS)


def voice(f0, jitter, shimmer, filt, snr=None):
    """(pcm, flow, period log) of one oracle voice"""
    a = ["-o", "x", "-d", "1", "-f", str(f0), "-g", str(f0 + 30), "-a", str(AMP)]
    if jitter:
        a += ["-j", str(jitter)]
    if shimmer:
        a += ["-s", str(shimmer)]
    flow, log = O.flowgen(O.flow_par_from_cli(a, 7), want_log=True)
    if filt in TRACTS:
        pcm = tract_filter(flow, *TRACTS[filt])
        if snr is not None:
            pcm = O.noise(pcm, snr, 3)
    else:
        pcm = O.vowel(flow, filt) if snr is None else O.vowel_noise(flow, filt, snr, 3)
    return pcm, flow, log


def tract_filter(flow, F, B):
    """a formant tract as the library applies it (gain 10, pre-emphasis 1: 10 (x[n] - x[n-1]) through 1/A(z)), rounded"""
    from scipy.signal import lfilter
    from voice_synth_b200 import api
    y = lfilter([10.0, -10.0], api.tract_from_formants(F, B, FS), np.asarray(flow, dtype=np.float64))
    return np.clip(np.round(y), -32768, 32767).astype(np.int16)


def measure(pcm, flow, log):
    mk, rn, rep = vr.analyse(pcm, FS)
    fl = rr.report(flow, FS)
    starts = np.asarray(log["start"], dtype=np.int64)
    T = np.asarray(log["T"], dtype=np.int64)
    d = np.diff(mk)
    p = np.searchsorted(starts, np.asarray(mk[:-1]), side="right") - 1
    share = float(np.mean(d == T[p])) if len(d) else 0.0
    return rep, fl, share, rn


def main(filters=FILTERS, levels=LEVELS, snr=None):
    """per filter and level over F0S: the PCM and flow jitter_pct and shimmer_pct where they differ most, the share"""
    print(f"| filter | jitter, shimmer (%) | PCM jitter % (flow) | PCM shimmer % (flow) | PCM periods = logged |"
          f"{'' if snr is None else f' output noise {snr:.0f} dB'}")
    print("|---|---|---|---|---|")
    out = {}
    for filt in filters:
        for j, s in levels:
            rows = []
            for f0 in F0S:
                rep, fl, share, _ = measure(*voice(f0, j, s, filt, snr))
                rows.append((rep["base"]["jitter_pct"], fl["base"]["jitter_pct"], rep["base"]["shimmer_pct"],
                             fl["base"]["shimmer_pct"], share))
            wj = max(rows, key=lambda r: abs(r[0] - r[1]))
            ws = max(rows, key=lambda r: abs(r[2] - r[3]))
            share = min(r[4] for r in rows)
            out[(filt, j, s)] = (wj, ws, share)
            print(f"| {filt} | {j:g}, {s:g} | {wj[0]:.3f} ({wj[1]:.3f}) | {ws[2]:.3f} ({ws[3]:.3f}) | {100 * share:.1f} % |",
                  flush=True)
    return out


if __name__ == "__main__":
    main()
    main(levels=((1.0, 3.0),), snr=20.0)
