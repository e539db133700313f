"""Caller-defined tracts against the preset path on the bench batch (cfg2): python scripts/prof_tracts.py

(a) cfg2 through vs_synth_batch and through vs_synth_batch_tract with the ten presets as tracts 0..9 (outputs must be
    byte-identical), (b) cfg2 with 10, 32 and 128 distinct formant tracts, (c) host time of the first call that brings
    128 new tracts and of the call after it.  One process, 5 warm-up and 20 timed steps per arm, arms alternating,
    render_ms from vs_get_timing."""
import pathlib
import subprocess
import sys
import time

sys.path.insert(0, str(pathlib.Path(__file__).resolve().parents[1]))
import numpy as np
import torch
from voice_synth_b200 import api, workloads

WARM, STEPS = 5, 20
PRESETS = "aiu1234567"

card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip().splitlines()[0]
print("card:", card, flush=True)

ctx = api.Context()
p, f = workloads.cfg2()
ns = api.flow_nsamples(p)
dev = torch.zeros(int(ns.sum()), dtype=torch.int16, device="cuda")


def presets_as_tracts(f):
    den = np.stack([api.tract_from_preset(k) for k in PRESETS])
    t = api.TractParams(f.n, den, tract=[PRESETS.index(chr(c)) for c in f.preset])
    t.gain[...] = f.gain
    t.pre[...] = f.pre
    return t


def formant_tracts(n_tracts, seed):
    rng = np.random.default_rng(seed)
    dens = []
    for _ in range(n_tracts):
        nf = 5
        freqs = np.sort(rng.uniform(250.0, 4500.0, nf))
        dens.append(api.tract_from_formants(freqs, rng.uniform(60.0, 250.0, nf), 22050))
    t = api.TractParams(p.n, np.stack(dens), tract=np.arange(p.n) % n_tracts)
    t.gain[...] = 0.5
    return t


def timed(arms):
    """arms: name -> filter params; alternate the arms step by step"""
    res = {k: [] for k in arms}
    info = {}
    for step in range(WARM + STEPS):
        for k, ff in arms.items():
            ctx.synth_batch(p, ff, out=dev)
            t = ctx.timing()
            if step >= WARM:
                res[k].append(t["render_ms"])
            info[k] = t
    return res, info


# (a)
t10 = presets_as_tracts(f)
a, _ = ctx.synth_batch(p, f)[:2]
b, _ = ctx.synth_batch(p, t10)[:2]
assert np.array_equal(a, b), "presets as tracts differ from the preset path"
print("(a) outputs byte-identical:", a.size, "samples", flush=True)
res, info = timed({"preset": f, "tract": t10})
for k in res:
    v = np.array(res[k])
    print(f"(a) {k:7s} render_ms median {np.median(v):.4f} min {v.min():.4f} max {v.max():.4f}  chunks {info[k]['chunks']} "
          f"path {info[k]['render_path']}", flush=True)
print(f"(a) tract / preset = {np.median(res['tract']) / np.median(res['preset']):.4f}", flush=True)

# (b)
arms = {f"{n}": formant_tracts(n, n) for n in (10, 32, 128)}
res, info = timed(arms)
for k in res:
    v = np.array(res[k])
    print(f"(b) {k:>3s} tracts: render_ms median {np.median(v):.4f} min {v.min():.4f}  chunks {info[k]['chunks']} "
          f"warmup_samples {info[k]['warmup_samples']}", flush=True)

# (c)
fresh = formant_tracts(128, 999)
fresh.den[:, 22] += 1e-9                  # coefficients the context has never seen
for label in ("first call with 128 new tracts", "the call after it"):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ctx.synth_batch(p, fresh, out=dev)
    t1 = time.perf_counter()
    ctx.sync()
    print(f"(c) {label}: host {1e3 * (t1 - t0):.2f} ms (enqueue, device buffers)", flush=True)
    fresh = api.TractParams(p.n, fresh.den, tract=(np.asarray(fresh.tract) + 1) % 128)   # same tracts, new inputs
ctx.close()
