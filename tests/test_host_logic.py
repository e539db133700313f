"""CPU-only checks of the host side: the C ABI surface, the Python mirror of the reference's argv
handling, the workload generators, the product/oracle separation and the rank sharding (gloo)."""
import os
import pathlib
import re
import subprocess
import sys

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parents[1]


def test_abi_library_exports_every_declared_symbol():
    from voice_synth_b200 import _lib
    hdr = (ROOT / "include" / "voicesynth.h").read_text()
    declared = set(re.findall(r"\b(vs_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"vs_ctx"}
    assert {"vs_flowgen_batch", "vs_vowel_filter_batch", "vs_synth_batch", "vs_ctx_create", "vs_sync"} <= declared
    out = subprocess.run(["nm", "-D", "--defined-only", str(_lib.LIB_PATH)], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r" T (vs_[a-z0-9_]+)", out))
    assert declared <= exported, declared - exported
    assert set(_lib.EXPORTS) <= exported
    L = _lib.load()                      # loads without a GPU; only ctx creation needs one
    assert L.vs_abi_version() == 1
    assert L.vs_strerror(-6).decode().startswith("no usable")


def test_no_gpu_means_loud_failure_not_fallback():
    # in a child that sees no CUDA device, so that the check runs on machines with a GPU as well
    code = ("from voice_synth_b200 import api\n"
            "try:\n    api.Context()\nexcept api.VsError as e:\n    print(e.code)\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert r.stdout.strip() == "-6", r.stdout


def test_product_never_touches_the_oracle():
    bad = []
    for path in list((ROOT / "voice_synth_b200").rglob("*")) + list((ROOT / "host").rglob("*")) + list((ROOT / "include").rglob("*")):
        if path.is_file() and path.suffix in {".py", ".c", ".h", ".cu", ".cuh", ""} and "lib" not in path.parts and "bin" not in path.parts:
            text = path.read_text(errors="ignore")
            if re.search(r"oracle|vso_|vs_oracle", text):
                bad.append(str(path))
    assert not bad, bad


def test_python_cli_mirror_matches_oracle_parser(golden, oracle):
    from voice_synth_b200 import api
    lines = [c["args"] for c in golden["cases"]] + ["-d 3.7 -f 97.3 -g 99 -j 0.73 -s 11.1 -n 17.5 -l 0.07 -a 9999 -z 0.33 -k 0.77 -c 0.61 -r 16000"]
    for line in lines:
        row = api.FlowParams.cli_row(line.split())
        par = oracle.flow_par_from_cli(["-o", "x"] + line.split(), 1)
        assert row is not None and par is not None
        for k, ok in (("dur", "dur"), ("jitter", "jitter"), ("shimmer", "shimmer"), ("cq", "cq"), ("K", "K"), ("Kvar", "Kvar"),
                      ("F0", "F0"), ("DC", "DC"), ("noise", "noise")):
            assert np.float32(row[k]) == np.float32(getattr(par, ok)), (line, k)
        assert int(row["amp"]) == par.amp and int(row["fs"]) == par.fs
        assert bool(row["flags"] & 1) == bool(par.has_jitter) and bool(row["flags"] & 2) == bool(par.has_shimmer)
        assert bool(row["flags"] & 4) == bool(par.has_noise)
    for bad in ["-d 0.4", "-j 1001", "-f 130", "-r 22050", "-a 32767", "-l 0.31", "-q 1", "-n 51", "-s 101", "-z 1.5", "-k 0.4", "-g 40"]:
        assert api.FlowParams.cli_row(bad.split()) is None, bad
        assert oracle.flow_par_from_cli(["-o", "x"] + bad.split(), 1) is None, bad


def test_workloads_are_valid_reference_command_lines():
    """every synthetic stream is also a command line of the unmodified reference tools"""
    from voice_synth_b200 import api, workloads
    for p, f in (workloads.cfg1(), workloads.cfg2(n=200), workloads.cfg3(n=300, first=65000), workloads.cfg5(n=300, first=123456)):
        for i in range(0, p.n, 7):
            row = api.FlowParams.cli_row(workloads.cli_args(p, i))
            assert row is not None, workloads.cli_args(p, i)
            for k in ("dur", "jitter", "shimmer", "F0", "DC", "noise"):
                assert np.float32(row[k]) == getattr(p, k)[i], (i, k, workloads.cli_args(p, i))
            assert int(row["fs"]) == int(p.fs[i]) and int(row["flags"]) == int(p.flags[i])
        assert set(chr(c) for c in f.preset) <= set("aiu1234567")
        ns = api.flow_nsamples(p)
        assert np.all(ns == (np.float32(p.fs.astype(np.float32)) * p.dur).astype(np.uint64))
    p, f = workloads.cfg2()
    assert p.n == 4096 and int(api.flow_nsamples(p).sum()) == 4096 * 22050
    assert len(set(p.seed.tolist())) == 4096


def test_flow_validate_and_helpers():
    import ctypes as C
    from voice_synth_b200 import api, _lib
    L = _lib.load()
    p = api.FlowParams(3)
    bad = C.c_size_t(99)
    assert L.vs_flow_validate(C.byref(p._c()), 3, C.byref(bad)) == 0
    p.amp[1] = 40000
    assert L.vs_flow_validate(C.byref(p._c()), 3, C.byref(bad)) == -2 and bad.value == 1
    p.amp[1] = 12000
    p.F0[2] = 0.0
    assert L.vs_flow_validate(C.byref(p._c()), 3, C.byref(bad)) == -2 and bad.value == 2
    p.F0[2] = 120.0
    mp = np.zeros(3, dtype=np.uint64)
    L.vs_flow_max_periods(C.byref(p._c()), 3, mp.ctypes.data)
    assert np.all(mp == 22050 // 183 + 2)                   # no jitter: T == P == 183


def test_const_division_trick_is_exact(tmp_path):
    """r/RAND_MAX and r/(RAND_MAX*10000) by reciprocal multiply + FMA residual == IEEE division for every r (exhaustive)"""
    exe = tmp_path / "vs_divcheck"
    subprocess.run(["gcc", "-O2", "-mfma", "-fopenmp", "-ffp-contract=off", str(ROOT / "tests" / "tools" / "divcheck.c"), "-o", str(exe), "-lm"], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout
    assert out.count("mismatches with correction: 0,") == 2, out


def test_sharding_rules():
    from voice_synth_b200 import sharding
    for n in (1, 7, 8, 4096, 65536, 1000003):
        for world in (1, 2, 4, 8):
            r = [sharding.shard_range(n, k, world) for k in range(world)]
            assert r[0][0] == 0 and r[-1][1] == n and all(r[k][1] == r[k + 1][0] for k in range(world - 1))
            sizes = [b - a for a, b in r]
            assert max(sizes) - min(sizes) <= 1
    cuts = sharding.shard_by_samples([10, 10, 10, 10, 40, 10, 10], 2)
    assert cuts[0] == 0 and cuts[-1] == 7 and 0 < cuts[1] < 7


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    import torch
    from voice_synth_b200 import sharding
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    n = 65536
    lo, hi = sharding.shard_range(n, rank, world)
    seeds = sharding.rank_seeds(4096, rank)
    mine = torch.tensor([lo, hi, int(seeds.min()), int(seeds.max())], dtype=torch.int64)
    allr = [torch.zeros(4, dtype=torch.int64) for _ in range(world)]
    dist.all_gather(allr, mine)
    t = torch.tensor([1.0 + rank], dtype=torch.float64)          # bench.py: time = max over ranks
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dist.barrier()
    if rank == 0:
        q.put(([x.tolist() for x in allr], float(t)))
    dist.destroy_process_group()


def test_two_rank_partition_over_gloo():
    """world_size 2 on CPU: ranks own disjoint contiguous stream ranges and disjoint seeds; timing reduces with MAX"""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    import socket
    with socket.socket() as s:                                  # a port no other job on the machine holds
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    rows, tmax = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert rows[0][0] == 0 and rows[0][1] == rows[1][0] and rows[1][1] == 65536
    assert rows[0][3] < rows[1][2]                              # seed ranges do not overlap
    assert tmax == 2.0


def test_analysis_restatement_trigger_is_the_sequential_one():
    """tests/analysis_ref.py states vs_flow_analyze_batch's two-threshold trigger with array operations: it must be the
    sequential state machine of include/voicesynth.h"""
    import analysis_ref as ar
    rng = np.random.default_rng(1)
    for _ in range(300):
        x = rng.integers(-5, 6, 257)
        lo = int(rng.integers(-3, 2))
        hi = lo + int(rng.integers(0, 3))
        armed, want = True, []
        for m, v in enumerate(x):
            if v > hi:
                if armed:
                    want.append(m)
                armed = False
            elif v <= lo:
                armed = True
        assert list(ar.onsets(x, lo, hi)) == want
    cycle = np.array([0] * 20 + [3, 9, 3] + [0] * 17, dtype=np.int16)
    s = ar.stats(np.tile(cycle, 50), fs=8000)
    assert s["cycles"] == 49 and s["mean_period"] == 40.0 and s["f0_hz"] == 200.0 and s["jitter_pct"] == 0.0 and s["mean_peak"] == 9.0
    assert ar.stats(np.tile(np.array([0, 5], dtype=np.int16), 100))["flags"] == 1     # a cycle every 2 samples: flagged
