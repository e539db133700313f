"""Voice report of device-resident vowels: python scripts/prof_vowel_report.py [n_streams]

The cfg5 slice of scripts/prof_pitch.py (1 s utterances, F0 80-250 Hz, jitter, shimmer, glottal noise off/10-40 dB, the
ten presets) is rendered into a device buffer once; vs_vowel_report_batch then analyses it with the default pitch
options, and vs_pitch_batch on the same input for comparison.  The context runs on torch's current stream, so CUDA events
recorded there bracket each whole call.  Median of 10 timed calls after 3 warm-ups, the two calls alternating.  A
torch.profiler pass then gives the device time of each kernel of the report call.  The marks kernel's integer work comes
from the marks: per step, (candidates + 1) x L multiply-adds for C and E."""
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

out = ctx.vowel_report_batch(pcm, ns, offsets=offs, fs=p.fs)
rep = out["rep"]
K = rep["base"]["onsets"].astype(np.int64)
mp = rep["base"]["mean_period"].astype(np.float64)
macs = float(np.sum(np.maximum(K - 1, 0) * (0.45 * mp + 2) * mp))        # candidates ~ 0.45 T + 1, L ~ T, plus E(m_k)
print(f"slice: {N} streams, {int(ns.sum())} samples, {int(K.sum())} marks, runs cover "
      f"{out['run_len'].sum() / ns.sum() * 100:.1f} % of the samples, ~{macs / 1e9:.1f} G int MACs for C and E", flush=True)
print(f"mean PCM jitter {float(np.mean(rep['base']['jitter_pct'])):.3f} %, shimmer {float(np.mean(rep['base']['shimmer_pct'])):.3f} %, "
      f"HNR {float(np.nanmean(np.where(np.isinf(rep['hnr_db']), np.nan, rep['hnr_db']))):.2f} dB", flush=True)


def timed(call):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    call()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


calls = {"vowel_report_batch": lambda: ctx.vowel_report_batch(pcm, ns, offsets=offs, fs=p.fs),
         "pitch_batch": lambda: ctx.pitch_batch(pcm, ns, offsets=offs, fs=p.fs)}
ms = {k: [] for k in calls}
for it in range(WARM + REPS):
    for k, c in calls.items():
        t = timed(c)
        if it >= WARM:
            ms[k].append(t)
for k, v in ms.items():
    v = np.array(v)
    print(f"{k} call ms median {np.median(v):.3f} min {v.min():.3f} max {v.max():.3f}", flush=True)

from torch.profiler import ProfilerActivity, profile
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(3):
        calls["vowel_report_batch"]()
    torch.cuda.synchronize()
for e in prof.key_averages():
    if e.key.startswith("vs_") or "_kernel" in e.key:
        t = e.device_time_total / max(e.count, 1) / 1e3
        extra = f"  {macs / (t * 1e-3) / 1e12:.2f} T int MAC/s" if "marks" in e.key else ""
        print(f"kernel {e.key[:40]:40s} calls {e.count:3d}  mean {t:.3f} ms{extra}", flush=True)
ctx.close()
