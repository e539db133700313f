"""Voice report against the plain analysis on device-resident flow: python scripts/prof_report.py [n_streams]

A cfg5-shaped slice (workloads.cfg5: 1 s utterances, F0 80-250 Hz, jitter, shimmer, glottal noise off/10-40 dB) is
generated into a device buffer once; vs_flow_analyze_batch and vs_flow_report_batch then read it with the trigger at
8 % / 15 % of the amplitude.  The context runs on torch's current stream, so CUDA events recorded there bracket each
whole call (row upload, kernels, copy of the results).  3 warm-up and 10 timed calls per arm, arms alternating.  GB/s
is flow bytes (2 B per sample) over call time.  A torch.profiler pass then gives the device time of each kernel."""
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
p, _ = workloads.cfg5(n=N)
ns = api.flow_nsamples(p)
stride = int(ns.max())
flow = torch.zeros(N * stride, dtype=torch.int16, device="cuda")
ctx.flowgen_batch(p, out=flow)
offs = np.arange(N, dtype=np.uint64) * np.uint64(stride)
lo, hi = (p.amp * 0.08).astype(np.int16), (p.amp * 0.15).astype(np.int16)
kw = dict(offsets=offs, fs=p.fs, lo=lo, hi=hi)
flow_bytes = 2 * int(ns.sum())
print(f"slice: {N} streams, {int(ns.sum())} samples, {flow_bytes / 1e6:.1f} MB of flow on the device", flush=True)

st = ctx.flow_analyze_batch(flow, ns, **kw)
rep = ctx.flow_report_batch(flow, ns, **kw)
assert rep["base"].tobytes() == st.tobytes(), "report base differs from the analysis"
ok = rep["base"]["flags"] == 0
print(f"streams without overflow {int(ok.sum())}, mean cycles {rep['base']['cycles'][ok].mean():.1f}, "
      f"mean hnr_len {rep['hnr_len'][ok].mean():.1f}, finite HNR {int(np.isfinite(rep['hnr_db']).sum())}", flush=True)

arms = {"analyze": ctx.flow_analyze_batch, "report": ctx.flow_report_batch}
ms = {k: [] for k in arms}
for it in range(WARM + REPS):
    for k, call in arms.items():
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        call(flow, ns, **kw)
        b.record()
        b.synchronize()
        if it >= WARM:
            ms[k].append(a.elapsed_time(b))
for k, v in ms.items():
    v = np.array(v)
    print(f"{k:8s} call ms median {np.median(v):.3f} min {v.min():.3f} max {v.max():.3f}  "
          f"{flow_bytes / (np.median(v) * 1e-3) / 1e9:.1f} GB/s of flow", flush=True)
print(f"report / analyze = {np.median(ms['report']) / np.median(ms['analyze']):.3f}", flush=True)

from torch.profiler import ProfilerActivity, profile
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(3):
        ctx.flow_report_batch(flow, ns, **kw)
    torch.cuda.synchronize()
for e in prof.key_averages():
    if e.key.startswith("vs_") or "_kernel" in e.key:
        t = e.device_time_total / max(e.count, 1) / 1e3
        print(f"kernel {e.key[:40]:40s} calls {e.count:3d}  mean {t:.3f} ms  {flow_bytes / (t * 1e-3) / 1e9:.1f} GB/s of flow", flush=True)
ctx.close()
