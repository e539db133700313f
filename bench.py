#!/usr/bin/env python3
"""bench.py -- BASELINE.json's metric on BASELINE.json's config, on 1..8 B200 of one node.

  python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run)
  python bench.py --impl reference ...                      (the reference's own CPU tools, all host cores)

metric   synthesized samples/sec (Msamples/s); % of HBM-write roofline   (BASELINE.json:metric)
workload configs[1]: batch of 4096 streams x 1 s covering every vowel preset, fused flowgen+vowel
         kernel (vs_synth_batch).  With N GPUs every rank synthesises its own 4096 streams (weak
         scaling: streams are independent, no collective on the data path -- SURVEY.md 8e).
step     one vs_synth_batch call over the rank's whole batch.
value    kernel path, PCM left resident in HBM (device output buffer, 180 MB per step > 126 MB L2).
e2e      the same call with a pinned HOST output buffer: parameter/descriptor H2D and the PCM D2H
         over PCIe are inside the timed region.
The line also carries the dominant kernel's roofline (HBM-write as BASELINE asks, plus the FP64 pipe
that actually binds it) and the reference CPU tools timed on this box's cores (cpu_baseline).
"""
import argparse
import atexit
import json
import os
import pathlib
import subprocess
import sys
import tempfile
import threading
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = pathlib.Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "synthesized samples/sec (Msamples/s); % of HBM-write roofline"
N_STREAMS = 4096
FP64_INSTR_PER_SAMPLE = 25          # 1 mul + 22 FMA + pre-emphasis FMA + quantiser add (DESIGN.md)


# ------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the unmodified reference tools (oracle/_ref), one process per core
# ------------------------------------------------------------------------------------------------
def _ref_tools():
    ref = ROOT / "oracle" / "_ref"
    if all((ref / f).exists() for f in ("flowgen_shimmer", "vowel", "timeshim.so")):
        return ref
    return None


def _run_ref_stream(job):
    ref, tmpdir, idx, fargs, preset, seed, suffix = job
    env = dict(os.environ, VS_SEED=str(seed), LD_PRELOAD=str(ref / "timeshim.so"))
    # file names relative to the scratch directory: the tools strcpy() them into char[30] (flowgen_shimmer.c:143-146)
    f, o = f"f{idx}.wav", f"o{idx}.wav"
    subprocess.run([str(ref / ("flowgen_shimmer" + suffix)), "-o", f] + fargs, env=env, cwd=tmpdir, stdout=subprocess.DEVNULL, check=True)
    subprocess.run([str(ref / ("vowel" + suffix)), "-i", f, "-o", o, "-v", preset], env=env, cwd=tmpdir, stdout=subprocess.DEVNULL, check=True)
    n = (os.path.getsize(os.path.join(tmpdir, o)) - 72) // 2
    os.unlink(os.path.join(tmpdir, f))
    os.unlink(os.path.join(tmpdir, o))
    return n


def _run_port_stream(job):
    from oracle import pyoracle as O
    _, _, idx, fargs, preset, seed, _ = job
    par = O.flow_par_from_cli(["-o", "x"] + fargs, seed)
    return int(O.vowel(O.flowgen(par), preset).size)


def cpu_reference_throughput(n_streams, first=0, o2=False):
    """Msamples/s of the reference CPU pipeline over `n_streams` streams of the bench workload: the unmodified tools,
    one process per core (flowgen_shimmer -> WAV on tmpfs -> vowel), built with the Makefile's flags (-O0) or -O2."""
    from voice_synth_b200 import workloads
    p, f = workloads.cfg2(n=N_STREAMS)
    ref = _ref_tools()
    suffix = "_O2" if (o2 and ref and (ref / "vowel_O2").exists()) else ""
    cores = os.cpu_count() or 1
    tmpdir = tempfile.mkdtemp(dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    jobs = [(ref, tmpdir, i, workloads.cli_args(p, i % N_STREAMS), chr(f.preset[i % N_STREAMS]), int(p.seed[i % N_STREAMS]), suffix)
            for i in range(first, first + n_streams)]
    fn = _run_ref_stream if ref else _run_port_stream
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=cores) as ex:
        total = sum(ex.map(fn, jobs, chunksize=4))
    dt = time.perf_counter() - t0
    try:
        os.rmdir(tmpdir)
    except OSError:
        pass
    return total / dt / 1e6, cores, ("reference" if ref else "port"), dt, total


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    per_step = args.ref_streams
    vals = []
    for it in range(args.warmup + args.steps):
        v, cores, kind, dt, total = cpu_reference_throughput(per_step, first=(it * per_step) % N_STREAMS)
        if it >= args.warmup:
            vals.append((v, dt))
    value = sum(v for v, _ in vals) / len(vals)
    ms = 1e3 * sum(d for _, d in vals) / len(vals)
    sample = (f"{per_step} of the workload's {N_STREAMS} streams per step (a rate on the same stream distribution, not the whole batch): "
              f"flowgen_shimmer -> tmpfs WAV -> vowel, "
              f"{'unmodified reference tools built with the Makefile flags (-O0)' if kind == 'reference' else 'oracle port'}, "
              f"one process per core")
    line = {"impl": "reference", "metric": METRIC, "value": round(value, 3), "unit": "Msamples/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "cfg2: 4096 streams x 1 s x 10 vowel presets (bounded sample per step)",
                       "streams_per_step": per_step},
            "cpu_baseline": {"value": round(value, 3), "unit": "Msamples/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": round(value, 3), "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# clocks during the timed region
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_indices):
        """ONE nvidia-smi for all the GPUs of the job, started by rank 0 (a sampler per rank means N processes taking
        the driver's locks twenty times a second next to N ranks launching kernels)"""
        self.rows = []
        self.proc = None
        self.gpus = list(gpu_indices)

    def start(self):
        if not self.gpus:
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50",
                                          "-i", ",".join(str(g) for g in self.gpus)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
            atexit.register(self.proc.terminate)          # the sampler loops until stopped: not past an early exit
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        mx = [int(r[2]) for r in self.rows if len(r) >= 8 and r[2].isdigit()]
        per_gpu = {}
        for r in self.rows:
            if len(r) >= 8 and r[1].isdigit():
                per_gpu.setdefault(r[0], []).append(int(r[1]))
        # per GPU the median of its busy samples; the job's figure is the slowest GPU's
        meds = []
        for v in per_gpu.values():
            v.sort()
            b = v[len(v) // 2:]
            meds.append(b[len(b) // 2])
        sm = sorted(x for v in per_gpu.values() for x in v)
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        # the busy samples are the upper half (the sampler also sees idle gaps between steps)
        return {"sm_mhz": min(meds) if meds else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "gpus": len(per_gpu)}


# ------------------------------------------------------------------------------------------------
def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    """DRAM bytes (read + write) of ONE launch of the fused render kernel, from the committed ncu capture."""
    p = ROOT / "profiles" / "ncu_summary.json"
    if p.exists():
        try:
            return json.loads(p.read_text()).get("render_dram_bytes_per_launch")
        except Exception:
            return None
    return None


def _cpus_of(spec):
    cpus = set()
    for part in spec.strip().split(","):
        lo, _, hi = part.partition("-")
        cpus.update(range(int(lo), int(hi or lo) + 1))
    return cpus


def _topo_affinity(index):
    """CPU affinity of GPU `index` as `nvidia-smi topo -m` reports it (used when sysfs has no NUMA node for the device)."""
    out = subprocess.run(["nvidia-smi", "topo", "-m"], capture_output=True, text=True, timeout=20).stdout
    header = None
    for line in out.splitlines():
        cols = [c for c in line.replace("\x1b[4m", "").replace("\x1b[0m", "").split("\t") if c.strip() != ""]
        if header is None and "CPU Affinity" in line:
            header = [c.strip() for c in cols]
            continue
        if header and cols and cols[0].strip() == f"GPU{index}":
            pos = header.index("CPU Affinity") + 1          # the row has the GPU name in front
            if pos < len(cols):
                return cols[pos].strip()
    return None


def bind_near_gpu(index):
    """Run this rank on the CPUs of its GPU's NUMA node, so that the pinned host buffers it allocates are
    node-local (first touch) and the PCM does not cross the socket interconnect after crossing PCIe.
    Returns what was done, for the JSON line."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(index)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int((pathlib.Path("/sys/bus/pci/devices") / bdf / "numa_node").read_text())
        how = "sysfs"
        if node >= 0:
            cpus = _cpus_of(pathlib.Path(f"/sys/devices/system/node/node{node}/cpulist").read_text())
        else:
            spec = _topo_affinity(index)
            if not spec:
                return {"gpu": bdf, "node": node, "bound": False}
            cpus, how = _cpus_of(spec), "nvidia-smi topo -m"
        use = cpus & os.sched_getaffinity(0)
        if not use:
            return {"gpu": bdf, "node": node, "bound": False, "why": "no allowed CPU near the GPU"}
        os.sched_setaffinity(0, use)
        return {"gpu": bdf, "node": node, "bound": True, "cpus": len(use), "from": how}
    except Exception as e:                                  # no sysfs, no such property: run unbound
        return {"bound": False, "why": type(e).__name__}


def sample_streams(buf, ns, k, seed):
    """A fixed, seeded choice of k streams of a dense batch (stream i at i * max(ns), as vs_synth_batch lays it out without
    offsets): {"pcm": their samples one after the other as float32, "streams": their indices, "nsamples": their lengths}."""
    import numpy as np
    import torch
    idx = np.sort(np.random.default_rng(seed).choice(len(ns), size=min(k, len(ns)), replace=False))
    stride = int(ns.max())
    t = torch.as_tensor(buf)
    pcm = torch.cat([t[int(i) * stride: int(i) * stride + int(ns[i])] for i in idx]).float().cpu().numpy()
    return {"pcm": pcm, "streams": idx.astype(np.float64), "nsamples": ns[idx].astype(np.float64)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--ref-streams", type=int, default=1024, help="streams per step of the reference arm")
    ap.add_argument("--cpu-sample", type=int, default=2048, help="streams of the cpu_baseline sample (0 = skip)")
    ap.add_argument("--no-other", action="store_true", help="skip the cfg3 / cfg5 workloads")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the PCM of the last timed step of each workload (a seeded sample of its streams, float32) "
                         "to DIR/<workload>_{pcm,streams,nsamples}.npy; rank 0 only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from voice_synth_b200 import api, sharding, workloads

    if args.warmup < 3:
        args.warmup = 3
    torch.cuda.set_device(local_rank)
    numa = bind_near_gpu(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(vals):
        t = torch.tensor(vals, dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t]

    # the rank's share of the job: its own 4096 streams (distinct seeds), nothing is exchanged
    p, f = workloads.cfg2(n=N_STREAMS)
    p.seed[...] = sharding.rank_seeds(N_STREAMS, rank)
    ns = api.flow_nsamples(p)
    samples_per_step = int(ns.sum())

    stream = torch.cuda.current_stream()
    ctx = api.Context(devices=[local_rank], stream=stream.cuda_stream)
    dev_out = torch.empty(samples_per_step, dtype=torch.int16, device="cuda")
    host_out_t = torch.empty(samples_per_step, dtype=torch.int16).pin_memory()
    host_out = host_out_t.numpy()

    def step_device():
        ctx.synth_batch(p, f, out=dev_out)

    def step_host():
        ctx.synth_batch(p, f, out=host_out)

    # ---- value: device-resident ----------------------------------------------------------------
    def gpu_ids():                      # nvidia-smi does not honour CUDA_VISIBLE_DEVICES: name the job's GPUs by UUID
        ids = []
        for i in range(min(world, torch.cuda.device_count())):
            try:
                ids.append("GPU-" + str(torch.cuda.get_device_properties(i).uuid))
            except Exception:
                ids.append(str(i))
        return ids
    sampler = ClockSampler(gpu_ids() if rank == 0 else [])
    sampler.start()                      # runs across warm-up and both timed regions (nvidia-smi needs ~0.1 s to start)
    for _ in range(args.warmup):
        step_device()
    ctx.sync()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = 0
    e0.record(stream)
    for _ in range(args.steps):
        step_device()                    # asynchronous: the host prepares step k+1 while step k runs
    e1.record(stream)
    barrier()
    dev_ms = e0.elapsed_time(e1) / args.steps
    # taken before any later leg reuses the output buffers; 56 MB in all with the cfg3 and cfg5 samples below
    dumps = {}
    if args.dump_outputs:
        dumps["cfg2"] = sample_streams(dev_out, ns, 256, seed=0)
    t = ctx.timing()
    launches += t["launches"] * args.steps
    warm = t["warmup_samples"]
    path = t["render_path"]
    n_chunks = t["chunks"]

    # per-kernel durations (CUDA events on the launching stream, recorded by the library around the
    # plan and render launches of a call), averaged over a few more steps of the same loop
    render_ms, plan_ms = [], []
    for _ in range(min(args.steps, 10)):
        step_device()
        t = ctx.timing()
        render_ms.append(t["render_ms"])
        plan_ms.append(t["plan_ms"])

    # ---- e2e: pinned host output, PCIe inside the timed region -------------------------------------
    # VS_OPT_ASYNC_HOST: the PCM of step k crosses PCIe while step k+1 renders; everything has landed
    # in host memory when the closing sync returns, which is inside the timed region.
    ctx.set_option(api.OPT_ASYNC_HOST, 1)
    for _ in range(3):
        step_host()
    ctx.sync()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_host()
    ctx.sync()
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    barrier()
    t = ctx.timing()
    h2d, d2h = t["h2d_bytes"], t["d2h_bytes"]
    launches += t["launches"] * args.steps
    ctx.set_option(api.OPT_ASYNC_HOST, 0)

    # the ceiling of that number: the same bytes as plain device-to-host copies into the same pinned buffer, all ranks at
    # once (on an 8-GPU box the GPUs share PCIe switches: the per-rank rate is a property of the box, not of the library)
    cs = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(cs):
        host_out_t.copy_(dev_out, non_blocking=True)
    cs.synchronize()
    barrier()
    t0 = time.perf_counter()
    with torch.cuda.stream(cs):
        for _ in range(5):
            host_out_t.copy_(dev_out, non_blocking=True)
    cs.synchronize()
    copy_ms = (time.perf_counter() - t0) * 1e3 / 5
    barrier()

    # ---- the two stand-alone kernels on the same batch (device-resident): vs_flowgen_batch, vs_vowel_filter_batch ----
    def best_render(fn, reps=6):
        best = None
        for _ in range(reps):
            fn()
            tt = ctx.timing()
            if best is None or tt["render_ms"] < best["render_ms"]:
                best = tt
        return best

    flow_dev = torch.empty(samples_per_step, dtype=torch.int16, device="cuda")
    t_flow = best_render(lambda: ctx.flowgen_batch(p, out=flow_dev))
    t_filt = best_render(lambda: ctx.vowel_filter_batch(flow_dev, ns, f, out=dev_out))
    launches += (t_flow["launches"] + t_filt["launches"]) * 6
    del flow_dev

    # ---- BASELINE.json's multi-GPU configurations, this rank's share of each -------------------------
    other = {}
    if not args.no_other:
        # configs[2]: 65 536 streams x 2 s, glottal noise, 8 192-stream shard per GPU; device-resident like `value`
        p3, f3 = workloads.cfg3(n=8192, first=rank * 8192)
        n3 = int(api.flow_nsamples(p3).sum())
        out3 = torch.empty(n3, dtype=torch.int16, device="cuda")
        for _ in range(5):                  # (the first call of a new shape sizes the library's buffers)
            ctx.synth_batch(p3, f3, out=out3)
        ctx.sync()
        barrier()
        k3 = 10
        e0.record(stream)
        for _ in range(k3):
            ctx.synth_batch(p3, f3, out=out3)
        e1.record(stream)
        barrier()
        ms3 = e0.elapsed_time(e1) / k3
        t3 = ctx.timing()
        launches += t3["launches"] * (k3 + 5)
        if args.dump_outputs:
            dumps["cfg3"] = sample_streams(out3, api.flow_nsamples(p3), 128, seed=0)
        del out3
        # configs[4]: 1 M utterances x 1 s, 131 072 per GPU, PCM streamed to pinned host memory: eight calls of
        # 16 384 utterances alternate between two pinned buffers, PCIe inside the timed region
        sub, nsub = 16384, 8
        parts = [workloads.cfg5(n=sub, first=(rank * nsub + k) * sub) for k in range(nsub)]
        n5 = [int(api.flow_nsamples(pp).sum()) for pp, _ in parts]
        ring = [torch.empty(max(n5), dtype=torch.int16).pin_memory().numpy() for _ in range(2)]
        ctx.set_option(api.OPT_ASYNC_HOST, 1)

        def sweep():
            for k, (pp, ff) in enumerate(parts):
                ctx.synth_batch(pp, ff, out=ring[k & 1])
            ctx.sync()

        sweep()
        barrier()
        t0 = time.perf_counter()
        sweep()
        ms5 = (time.perf_counter() - t0) * 1e3
        barrier()
        if args.dump_outputs:                # the sweep's last call: parts[-1] into ring[(nsub - 1) & 1]
            dumps["cfg5"] = sample_streams(ring[(nsub - 1) & 1], api.flow_nsamples(parts[-1][0]), 128, seed=0)
        t5 = ctx.timing()
        launches += t5["launches"] * nsub * 2
        ctx.set_option(api.OPT_ASYNC_HOST, 0)
        # the same bytes as bare device-to-host copies into the same pinned buffers, all ranks at once
        dev5 = torch.empty(max(n5), dtype=torch.int16, device="cuda")
        hosts5 = [torch.from_numpy(r) for r in ring]
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        with torch.cuda.stream(cs):
            for k in range(nsub):
                hosts5[k & 1][: n5[k]].copy_(dev5[: n5[k]], non_blocking=True)
        cs.synchronize()
        copy5 = (time.perf_counter() - t0) * 1e3
        barrier()
        del ring, hosts5, dev5
        ms3, ms5, copy5 = max_over_ranks([ms3, ms5, copy5])
        other = {
            "cfg3": {"workload": "65 536 streams x 2 s, jitter x shimmer x F0 grid, glottal noise 20 dB: 8 192-stream shard per GPU, "
                                 "fused vs_synth_batch, PCM resident in HBM",
                     "value": round(n3 * world / (ms3 * 1e-3) / 1e6, 1), "unit": "Msamples/s", "ms_per_step": round(ms3, 4),
                     "plan_ms": round(t3["plan_ms"], 4), "render_ms": round(t3["render_ms"], 4), "render_path": t3["render_path"]},
            "cfg5": {"workload": "1 M utterances x 1 s (hashed F0 / jitter / shimmer / SNR / vowel): 131 072 per GPU as 8 calls of 16 384 "
                                 "into two alternating pinned host buffers, PCIe inside the timed region",
                     "value": round(sum(n5) * world / (ms5 * 1e-3) / 1e6, 1), "unit": "Msamples/s", "ms_per_sweep": round(ms5, 2),
                     "d2h_bytes_per_sweep": int(2 * sum(n5)), "render_path": t5["render_path"],
                     "plain_copy_ms_per_sweep": round(copy5, 2), "sweep_over_plain_copy": round(copy5 / ms5, 4)},
        }
    clocks = sampler.stop()

    fp64_tflops, fp64_mhz = ctx.fp64_peak()

    # max over ranks; every rank's own e2e as well
    e2e_all, dev_all, copy_all = [e2e_ms], [dev_ms], [copy_ms]
    if world > 1:
        gathered = [torch.zeros(3, dtype=torch.float64, device="cuda") for _ in range(world)]
        dist.all_gather(gathered, torch.tensor([e2e_ms, dev_ms, copy_ms], dtype=torch.float64, device="cuda"))
        e2e_all = [float(g[0]) for g in gathered]
        dev_all = [float(g[1]) for g in gathered]
        copy_all = [float(g[2]) for g in gathered]
    dev_ms, e2e_ms = max_over_ranks([dev_ms, e2e_ms])
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        out_dir = pathlib.Path(args.dump_outputs)
        out_dir.mkdir(parents=True, exist_ok=True)
        for w, arrays in dumps.items():
            for name, a in arrays.items():
                np.save(out_dir / f"{w}_{name}.npy", a)

    total_samples = samples_per_step * world
    value = total_samples / (dev_ms * 1e-3) / 1e6
    e2e = total_samples / (e2e_ms * 1e-3) / 1e6
    peak, peak_src = measured_peaks()
    r_ms = float(np.mean(render_ms))
    achieved = 2.0 * samples_per_step / (r_ms * 1e-3) / 1e9            # algorithmic bytes: 2 B per output sample
    # FP64-pipe instructions per sample of the kernel that ran: the recurrence's 22 FMAs (+ gain multiply and
    # pre-emphasis FMA unless both were moved to the integer input) + the generator's one multiply
    filt = (path >> 2) & 3
    per_sample = {0: 22, 1: 24, 2: 46}[filt] + 1
    peak_dfma = fp64_tflops / 2
    issued = per_sample * (samples_per_step + warm) / (r_ms * 1e-3) / 1e12
    useful = per_sample * samples_per_step / (r_ms * 1e-3) / 1e12
    sm_mhz = clocks.get("sm_mhz") or 0
    peak_at_clock = 64 * 148 * sm_mhz * 1e6 / 1e12 if sm_mhz else None   # 64 DFMA / clk / SM at the clock sampled under load
    gen_name = "branch-free" if path & 1 else "general"
    line = {
        "metric": METRIC, "value": round(value, 1), "unit": "Msamples/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(dev_ms, 4), "ms_per_step_per_rank": [round(m, 4) for m in dev_all],
        "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "cfg2: 4096 streams x 1 s (22050 samples) per GPU, presets a,i,u,1..7 round-robin, F0 80-237.5 Hz, "
                               "jitter 0-3.5 %, shimmer 0-7.5 %, fused vs_synth_batch",
                   "streams_per_gpu": N_STREAMS, "samples_per_step_per_gpu": samples_per_step,
                   "l2": "output 180.6 MB per step > 126 MB L2, rewritten every step",
                   "plan_ms": round(float(np.mean(plan_ms)), 4), "render_ms": round(r_ms, 4),
                   "chunks": int(n_chunks), "warmup_samples_per_step": int(warm),
                   "other_workloads": other},
        "e2e": {"value": round(e2e, 1), "unit": "Msamples/s", "ms_per_step": round(e2e_ms, 3),
                "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "per_rank_Msamples_s": [round(samples_per_step / (m * 1e-3) / 1e6, 1) for m in e2e_all],
                "plain_copy": {"what": "the same 180.6 MB per rank as bare cudaMemcpyAsync device-to-host into the same pinned buffer, all ranks at once",
                               "per_rank_GBs": [round(2.0 * samples_per_step / (m * 1e-3) / 1e9, 2) for m in copy_all],
                               "Msamples_s": round(total_samples / (max(copy_all) * 1e-3) / 1e6, 1),
                               "e2e_over_plain_copy": round(max(copy_all) / e2e_ms, 4)}},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "kernel": f"vs_render_kernel<SYNTH> ({gen_name} generator, one launch per step)",
                     "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                     "traffic": ncu_traffic(), "peak_source": peak_src,
                     "note": "the FP64 recurrence, not HBM, binds this kernel (SURVEY.md 8d): see fp64",
                     "fp64": {"dfma_per_sample": per_sample, "peak_tdfma_s": round(peak_dfma, 3),
                              "peak_source": "vs_measure_fp64_peak on this GPU (64 DFMA/clk/SM at the clock it implies)",
                              "implied_sm_mhz": round(fp64_mhz),
                              "achieved_tdfma_s": round(issued, 3), "frac": round(issued / peak_dfma, 4),
                              "counts": "frac / achieved: useful + carry warm-up samples; frac_useful / useful_tdfma_s: output samples only",
                              "useful_tdfma_s": round(useful, 3), "frac_useful": round(useful / peak_dfma, 4),
                              "peak_at_sampled_clock_tdfma_s": round(peak_at_clock, 3) if peak_at_clock else None,
                              "frac_useful_at_sampled_clock": round(useful / peak_at_clock, 4) if peak_at_clock else None}},
        "roofline_flow": {"bound": "hbm", "kernel": "vs_flow_rows_kernel (a warp per row, lanes along the row) via vs_flowgen_batch, same batch, PCM resident in HBM",
                          "bytes_per_sample": 2, "render_ms": round(t_flow["render_ms"], 4), "plan_ms": round(t_flow["plan_ms"], 4),
                          "achieved": round(2.0 * samples_per_step / (t_flow["render_ms"] * 1e-3) / 1e9, 1), "peak": peak, "unit": "GB/s",
                          "frac": round(2.0 * samples_per_step / (t_flow["render_ms"] * 1e-3) / 1e9 / peak, 4)},
        "roofline_filter": {"bound": "hbm", "kernel": "vs_render_kernel<FILTER> via vs_vowel_filter_batch, same batch, flow and PCM resident in HBM",
                            "bytes_per_sample": 4, "render_ms": round(t_filt["render_ms"], 4),
                            "achieved": round(4.0 * samples_per_step / (t_filt["render_ms"] * 1e-3) / 1e9, 1), "peak": peak, "unit": "GB/s",
                            "frac": round(4.0 * samples_per_step / (t_filt["render_ms"] * 1e-3) / 1e9 / peak, 4),
                            "note": "FP64 bound like the fused kernel; warm-up samples are read again per chunk"},
        "clocks": clocks,
        "numa": numa,
    }
    if world == 1 and args.cpu_sample > 0:
        try:
            v, cores, kind, dt, total = cpu_reference_throughput(args.cpu_sample)
            line["cpu_baseline"] = {"value": round(v, 3), "unit": "Msamples/s", "cores": cores, "kind": kind,
                                    "sample": f"{args.cpu_sample} of the {N_STREAMS} streams ({total} samples, {dt:.1f} s wall): "
                                              "flowgen_shimmer -> tmpfs WAV -> vowel, one process per core, Makefile flags (-O0)"}
            v2, _, kind2, dt2, total2 = cpu_reference_throughput(args.cpu_sample, o2=True)
            if kind2 == "reference":
                line["cpu_baseline"]["o2"] = {"value": round(v2, 3), "unit": "Msamples/s",
                                              "sample": f"the same {args.cpu_sample} streams with the tools built at -O2 (bit-identical PCM), {dt2:.1f} s wall"}
        except Exception as ex:  # the baseline is a report, never a reason to lose the GPU numbers
            line["cpu_baseline"] = {"value": None, "unit": "Msamples/s", "cores": os.cpu_count(), "kind": "reference", "sample": f"failed: {ex}"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
