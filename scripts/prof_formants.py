"""Formant analysis of device-resident vowels: python scripts/prof_formants.py [n_streams]

A cfg5-shaped slice (workloads.cfg5: 1 s utterances, F0 80-250 Hz, jitter, shimmer, glottal noise off/10-40 dB, the ten
presets) is rendered into a device buffer once; vs_formant_batch then analyses it with the default options (order 14,
Hamming 25 ms / 10 ms, pre-emphasis from 50 Hz, bandwidths below 700 Hz, 5 formants).  The context runs on torch's
current stream, so CUDA events recorded there bracket each whole call (row and window upload, both kernels, copy of the
statistics).  Median of 10 timed calls after 3 warm-ups.  A torch.profiler pass then gives the device time of each
kernel.  The DFMA count is the autocorrelation's alone, from shapes: Nw (p + 1) per frame."""
import pathlib
import subprocess
import sys

sys.path.insert(0, str(pathlib.Path(__file__).resolve().parents[1]))
import numpy as np
import torch
from voice_synth_b200 import api, workloads

WARM, REPS = 3, 10
N = int(sys.argv[1]) if len(sys.argv) > 1 else 16384

card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip().splitlines()[0]
print("card:", card, flush=True)

ctx = api.Context(stream=torch.cuda.current_stream().cuda_stream)
p, f = workloads.cfg5(n=N)
ns = api.flow_nsamples(p)
stride = int(ns.max())
pcm = torch.zeros(N * stride, dtype=torch.int16, device="cuda")
ctx.synth_batch(p, f, out=pcm)
offs = np.arange(N, dtype=np.uint64) * np.uint64(stride)
frames = api.formant_frames(ns, p.fs)
F = int(frames.sum())
dfma = F * 551 * 15
print(f"slice: {N} streams, {int(ns.sum())} samples, {2 * int(ns.sum()) / 1e6:.1f} MB of PCM on the device, {F} frames, "
      f"{dfma / 1e9:.2f} G DFMA of autocorrelation", flush=True)

st = ctx.formant_batch(pcm, ns, offsets=offs, fs=p.fs)
print(f"analysed {int(st['analysed'].sum())} of {int(st['frames'].sum())} frames, unconverged {int(st['unconverged'].sum())}, "
      f"mean F1..F3 {[round(float(np.nanmean(st['f_mean_hz'][:, k])), 1) for k in range(3)]}", flush=True)

ms = []
for it in range(WARM + REPS):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    ctx.formant_batch(pcm, ns, offsets=offs, fs=p.fs)
    b.record()
    b.synchronize()
    if it >= WARM:
        ms.append(a.elapsed_time(b))
v = np.array(ms)
print(f"formant_batch call ms median {np.median(v):.3f} min {v.min():.3f} max {v.max():.3f}  "
      f"{F / (np.median(v) * 1e-3) / 1e6:.1f} M frames/s", flush=True)

from torch.profiler import ProfilerActivity, profile
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(3):
        ctx.formant_batch(pcm, ns, offsets=offs, fs=p.fs)
    torch.cuda.synchronize()
for e in prof.key_averages():
    if e.key.startswith("vs_") or "_kernel" in e.key:
        t = e.device_time_total / max(e.count, 1) / 1e3
        print(f"kernel {e.key[:40]:40s} calls {e.count:3d}  mean {t:.3f} ms", flush=True)
ctx.close()
