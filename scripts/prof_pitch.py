"""Pitch analysis of device-resident vowels: python scripts/prof_pitch.py [n_streams]

A cfg5-shaped slice (workloads.cfg5: 1 s utterances, F0 80-250 Hz, jitter, shimmer, glottal noise off/10-40 dB, the ten
presets) is rendered into a device buffer once; vs_pitch_batch then analyses it with the default options (75-600 Hz,
3 periods per window, 10 ms hop).  The context runs on torch's current stream, so CUDA events recorded there bracket
each whole call (row and table upload, both kernels, copy of the statistics).  Median of 10 timed calls after 3
warm-ups.  A torch.profiler pass then gives the device time of each kernel.  The DFMA counts come from shapes: the lag
sums the definitions need, sum over tau in {0, tau_lo-1 .. tau_hi+1} of (Nw - tau) per frame, and the ones the frame
kernel issues (32 lanes x K lags per lane x the steps of the lane with the shortest lag, per pass)."""
import math
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
frames = api.pitch_frames(ns, p.fs)
F = int(frames.sum())
need = issued = 0
for rate in np.unique(p.fs):
    k = int(frames[p.fs == rate].sum())
    Nw = int(round(3.0 * rate / 75.0))
    lo, hi = max(2, math.ceil(rate / 600.0)), math.floor(rate / 75.0)
    L = hi - lo + 3
    need += k * (Nw + sum(Nw - t for t in range(lo - 1, hi + 2)))
    passes = -(-L // (32 * 13))
    K = -(-L // (32 * passes)) | 1
    issued += k * 32 * K * sum(-(-(Nw - t0) // K) * K for t0 in range(lo - 1, hi + 2, 32 * K))
print(f"slice: {N} streams, {int(ns.sum())} samples, {2 * int(ns.sum()) / 1e6:.1f} MB of PCM on the device, {F} frames, "
      f"{need / 1e9:.1f} G DFMA needed, {issued / 1e9:.1f} G issued by the lag sums", flush=True)

st = ctx.pitch_batch(pcm, ns, offsets=offs, fs=p.fs)
print(f"voiced {int(st['voiced'].sum())} of {int(st['frames'].sum())} frames, mean F0 {float(np.nanmean(st['f0_mean_hz'])):.1f} Hz, "
      f"mean HNR {float(np.nanmean(st['hnr_mean_db'])):.2f} dB", flush=True)

ms = []
for it in range(WARM + REPS):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    ctx.pitch_batch(pcm, ns, offsets=offs, fs=p.fs)
    b.record()
    b.synchronize()
    if it >= WARM:
        ms.append(a.elapsed_time(b))
v = np.array(ms)
print(f"pitch_batch call ms median {np.median(v):.3f} min {v.min():.3f} max {v.max():.3f}  "
      f"{F / (np.median(v) * 1e-3) / 1e6:.1f} M frames/s", flush=True)

from torch.profiler import ProfilerActivity, profile
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(3):
        ctx.pitch_batch(pcm, ns, offsets=offs, fs=p.fs)
    torch.cuda.synchronize()
for e in prof.key_averages():
    if e.key.startswith("vs_") or "_kernel" in e.key:
        t = e.device_time_total / max(e.count, 1) / 1e3
        extra = ""
        if "pitch_frame" in e.key:
            extra = f"  {need / (t * 1e-3) / 1e12:.2f} T DFMA/s needed, {issued / (t * 1e-3) / 1e12:.2f} T issued"
        print(f"kernel {e.key[:40]:40s} calls {e.count:3d}  mean {t:.3f} ms{extra}", flush=True)
ctx.close()
