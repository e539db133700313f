"""Closed-loop accuracy of the formant analysis (DESIGN 4.2d), on the CPU: python scripts/formant_accuracy.py

1-second oracle flows (jitter 1 %, shimmer 3 %, seed 7) at F0 = 100, 120 and 150 Hz go through a tract with the
reference filter of tests/tools/vowel_den.c (pre-emphasis 1, gain scaled to 0.7 of full scale) and are analysed with
tests/formant_ref.py, the numpy restatement the GPU is pinned to.  The specified formants are, for the tract vowels,
those vs_tract_from_formants was given and, for the ten presets, the poles of the preset's own table (the same
selection: 50 Hz < F < fs/2 - 50 Hz, B < 700 Hz).  Printed: the largest |mean F_k / specified F_k - 1| over the three F0
and the smallest share of frames that found F_k."""
import pathlib
import sys
import tempfile

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT), str(ROOT / "tests")]
import numpy as np

import formant_ref as fr
from oracle import pyoracle as O
from test_formants_host import VOWELS
from voice_synth_b200 import api
from vowel_den_ref import VowelDen

vd = VowelDen(tempfile.mkdtemp())


def table_formants(den, fs):
    kept, _ = fr.select(np.roots(den[: 1 + np.max(np.nonzero(den))]), fs, fr.DEFAULTS)
    return [k[0] for k in kept]


def row(name, den, spec, fs, order):
    errs, share = [0.0] * 3, [1.0] * 3
    for f0 in (100, 120, 150):
        a = ["-o", "x", "-d", "1", "-f", str(f0), "-g", str(f0 + 30), "-j", "1", "-s", "3"] + (["-r", str(fs)] if fs != 22050 else [])
        flow = O.flowgen(O.flow_par_from_cli(a, 7))
        _, raw = vd(flow, den, gain=1.0, pre=1.0, want_raw=True)
        pcm = vd(flow, den, gain=0.7 * 32767 / np.abs(raw).max(), pre=1.0)
        _, st = fr.analyse(pcm, fs, fr.opts_with(order=order))
        for k in range(3):
            errs[k] = max(errs[k], abs(st["f_mean_hz"][k] / spec[k] - 1) if st["count"][k] else np.inf)
            share[k] = min(share[k], st["count"][k] / st["frames"])
    print(f"| {name} | {fs} | {order} | " + " | ".join(f"{s:.0f}" for s in spec[:3]) + " | " +
          " | ".join(f"{100 * e:.1f} %" for e in errs) + " | " + " / ".join(f"{100 * s:.0f}" for s in share) + " |", flush=True)


print("| vowel | fs | order | F1 | F2 | F3 | F1 err | F2 err | F3 err | frames with F1 / F2 / F3 (%) |")
print("|---|---|---|---|---|---|---|---|---|---|")
for order in (14, 24):
    for key in "aiu1234567":
        den = O.preset(key)
        row(f"preset {key}", den, table_formants(den, 22050), 22050, order)
for fs, order in ((22050, 14), (44100, 24)):
    for v, (F, B) in VOWELS.items():
        row(f"tract {v}", api.tract_from_formants(F, B, fs), F, fs, order)
