"""Closed-loop accuracy of the pitch analysis (DESIGN 4.2e), on the CPU: python scripts/pitch_accuracy.py

1-second oracle voices go through the reference vowel filter and are analysed with tests/pitch_ref.py, the numpy
restatement the GPU is pinned to, at the default options.
- F0 axis: flow with jitter 1 % and shimmer 3 % (seed 7) at F0 = 100, 120, 150 and 200 Hz through each of the ten
  presets, noise-free.  The truth is fs / mean T of the period log.  Printed per preset: the largest
  |mean voiced F0 / truth - 1| over the four F0, and the smallest share of voiced frames.
- Noise axis: flow without jitter or shimmer at the same F0 through `vowel -n` (output noise at 10, 20 and 30 dB, seed
  3).  Printed per SNR: the range over presets and F0 of mean HNR - SNR, and the noise-free voices' mean HNR."""
import pathlib
import sys

ROOT = pathlib.Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT), str(ROOT / "tests")]
import numpy as np

import pitch_ref as pr
from oracle import pyoracle as O

PRESETS = "aiu1234567"
F0S = (100, 120, 150, 200)


def flow(f0, jitter):
    a = ["-o", "x", "-d", "1", "-f", str(f0), "-g", str(f0 + 30)] + (["-j", "1", "-s", "3"] if jitter else [])
    return O.flowgen(O.flow_par_from_cli(a, 7), want_log=True)


print("| preset | F0 err (largest over 100-200 Hz) | voiced frames (smallest share) |")
print("|---|---|---|")
for key in PRESETS:
    err, share = 0.0, 1.0
    for f0 in F0S:
        x, log = flow(f0, True)
        _, st = pr.analyse(O.vowel(x, key), 22050)
        err = max(err, abs(st["f0_mean_hz"] / (22050 / np.mean(log["T"])) - 1.0))
        share = min(share, st["voiced"] / st["frames"])
    print(f"| {key} | {100 * err:.3f} % | {100 * share:.0f} % |", flush=True)

print()
print("| `vowel -n` SNR | mean HNR - SNR, min .. max over presets and F0 | mean HNR, min .. max |")
print("|---|---|---|")
for snr in (10.0, 20.0, 30.0, None):
    h = []
    for key in PRESETS:
        for f0 in F0S:
            x, _ = flow(f0, False)
            pcm = O.vowel(x, key) if snr is None else O.vowel_noise(x, key, snr, 3)
            h.append(pr.analyse(pcm, 22050)[1]["hnr_mean_db"])
    h = np.array(h)
    d = h - (snr or 0.0)
    print(f"| {'none' if snr is None else f'{snr:.0f} dB'} | {'' if snr is None else f'{d.min():+.2f} .. {d.max():+.2f} dB'} | "
          f"{h.min():.2f} .. {h.max():.2f} dB |", flush=True)
