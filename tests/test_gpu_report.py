"""vs_flow_report_batch (the voice report: Praat's jitter and shimmer quotients and a cycle-averaged HNR) on the GPU:
`base` byte for byte what vs_flow_analyze_batch returns, every new field against the numpy restatement
(tests/report_ref.py), the HNR of noise-only voices against the SNR of the generator's own period log, the error
codes, and `acoustic -x`."""
import math
import os
import pathlib
import subprocess

import numpy as np
import pytest

import report_ref as rr

pytestmark = pytest.mark.gpu
ROOT = pathlib.Path(__file__).resolve().parents[1]


@pytest.fixture(scope="module")
def vs():
    from voice_synth_b200 import api
    return api


@pytest.fixture(scope="module")
def ctx(vs):
    c = vs.Context()
    yield c
    c.close()


def _voices(vs, n, seed, noise=False):
    rng = np.random.default_rng(seed)
    args, seeds = [], []
    for i in range(n):
        f0 = float(rng.uniform(70, 320))
        a = ["-d", f"{rng.uniform(0.5, 1.5):.3f}", "-f", f"{f0:.2f}", "-g", f"{f0 + 30:.2f}"]
        if i % 4 != 0:
            a += ["-j", f"{rng.uniform(0.2, 4):.2f}"]
        if i % 4 != 1:
            a += ["-s", f"{rng.uniform(0.5, 12):.2f}"]
        if noise:
            a += ["-n", f"{rng.uniform(30, 45):.1f}"]
        if rng.random() < 0.5:
            a += ["-a", str(int(rng.integers(3000, 18000)))]
        if rng.random() < 0.25:
            a += ["-r", "44100"]
        args.append(a)
        seeds.append(int(rng.integers(0, 2**32)))
    return vs.FlowParams.from_cli(args, seeds)


def _check_fields(got, want, what):
    assert int(got["hnr_len"]) == want["hnr_len"], (what, got["hnr_len"], want["hnr_len"])
    for k in rr.FIELDS:
        g, w = float(got[k]), want[k]
        if math.isnan(w) or math.isinf(w):
            assert (math.isnan(g) and math.isnan(w)) or g == w, (what, k, g, w)
            continue
        rel = 1e-5 if k == "shimmer_db" else 2e-6
        assert math.isclose(g, float(np.float32(w)), rel_tol=rel, abs_tol=1e-6 if k == "hnr_db" else 1e-30), (what, k, g, w)


def _check_base(got, want, what):
    assert int(got["onsets"]) == want["onsets"] and int(got["cycles"]) == want["cycles"] and int(got["flags"]) == want["flags"], (what, got, want)
    for k in ("f0_hz", "jitter_pct", "shimmer_pct", "mean_period", "mean_peak"):
        assert math.isclose(float(got[k]), float(np.float32(want[k])), rel_tol=2e-6, abs_tol=1e-30), (what, k, got[k], want[k])


def _report_everywhere(ctx, flow, ns, **kw):
    """the report from host and from device input, which agree byte for byte, and the analysis of the same streams"""
    import torch
    rep = ctx.flow_report_batch(flow, ns, **kw)
    rep_dev = ctx.flow_report_batch(torch.from_numpy(flow).cuda(), ns, **kw)
    assert rep.tobytes() == rep_dev.tobytes()
    st = ctx.flow_analyze_batch(flow, ns, **kw)
    assert rep["base"].tobytes() == st.tobytes()
    assert (rep["reserved"] == 0).all()
    return rep


def test_report_noise_free_voices(ctx, vs):
    n = 64
    p = _voices(vs, n, 21)
    flow, offs, ns = ctx.flowgen_batch(p)
    rep = _report_everywhere(ctx, flow, ns, offsets=offs, fs=p.fs)
    for i in range(n):
        x = flow[int(offs[i]): int(offs[i]) + int(ns[i])]
        want = rr.report(x, fs=int(p.fs[i]))
        _check_base(rep[i]["base"], want["base"], i)
        _check_fields(rep[i], want, i)
        # a voice without shimmer has no amplitude perturbation: every cycle starts alike, HNR is +inf
        if not (p.flags[i] & vs.VS_F_SHIMMER and p.shimmer[i] > 0):
            assert rep[i]["hnr_db"] == np.inf and rep[i]["shimmer_apq3_pct"] == 0.0, i


def test_report_noisy_voices_ragged_rows(ctx, vs):
    """glottal noise, thresholds at 8 % / 15 % of the amplitude, rows at odd offsets with gaps"""
    n = 48
    p = _voices(vs, n, 22, noise=True)
    ns = vs.flow_nsamples(p)
    rng = np.random.default_rng(6)
    gaps = rng.integers(0, 50, n).astype(np.uint64) * 2 + 1
    offs = (np.concatenate([[0], np.cumsum(ns + gaps)[:-1]]) + gaps).astype(np.uint64)
    flow = np.zeros(int(offs[-1] + ns[-1]), dtype=np.int16)
    ctx.flowgen_batch(p, out=flow, offsets=offs)
    lo, hi = (p.amp * 0.08).astype(np.int16), (p.amp * 0.15).astype(np.int16)
    rep = _report_everywhere(ctx, flow, ns, offsets=offs, fs=p.fs, lo=lo, hi=hi)
    for i in range(n):
        x = flow[int(offs[i]): int(offs[i]) + int(ns[i])]
        want = rr.report(x, fs=int(p.fs[i]), lo=int(lo[i]), hi=int(hi[i]))
        _check_base(rep[i]["base"], want["base"], i)
        _check_fields(rep[i], want, i)
        assert np.isfinite(rep[i]["hnr_db"]), i


def _alternating(a, b, K):
    return np.array([a if k % 2 == 0 else b for k in range(K)], dtype=np.int64)


def test_report_edge_cases(ctx, vs):
    """K = 0..11 cycles, a cycle of 100 000+ samples (L > one tile of j), 40 000 full-scale cycles (sum S_j^2 > 2^64),
    a zero peak (no shimmer in dB), an overflowed onset list, silence; one call, odd offsets"""
    rng = np.random.default_rng(9)
    rows, names = [], []
    for K in range(12):
        rows.append(rr.pulse_train(rng.integers(20, 400, K), rng.integers(100, 32000, K)))
        names.append(f"K={K}")
    long = rr.pulse_train([100000, 120000, 100500, 100001], [20000, 19000, 20001, 25000])
    long[5000:220000:7] += rng.integers(0, 50, len(long[5000:220000:7])).astype(np.int16)    # stays above the threshold
    rows.append(long); names.append("L>=100000")
    big = rr.pulse_train([100] * 40000, _alternating(30000, 29990, 40000))
    rows.append(big); names.append("sum S^2 > 2^64")
    rows.append(np.array([0, -5, 3, 1, -5, 0, -1, -5, 4, -5, 0] + [-5] * 60, dtype=np.int16)); names.append("zero peak")
    over = np.zeros(4096, dtype=np.int16)
    over[::2] = 5
    rows.append(over); names.append("overflow")
    rows.append(np.zeros(1000, dtype=np.int16)); names.append("silence")
    n = len(rows)
    ns = np.array([len(r) for r in rows], dtype=np.uint64)
    offs = np.zeros(n, dtype=np.uint64)
    pos = 3
    for i, r in enumerate(rows):
        offs[i] = pos
        pos += len(r) + 5
    flow = np.zeros(pos, dtype=np.int16)
    for i, r in enumerate(rows):
        flow[int(offs[i]): int(offs[i]) + len(r)] = r
    lo = np.array([-5 if nm == "zero peak" else 0 for nm in names], dtype=np.int16)
    hi = np.array([-2 if nm == "zero peak" else 0 for nm in names], dtype=np.int16)
    fs = np.array([44100 if i % 3 == 0 else 22050 for i in range(n)], dtype=np.int32)
    rep = _report_everywhere(ctx, flow, ns, offsets=offs, fs=fs, lo=lo, hi=hi)
    for i, nm in enumerate(names):
        want = rr.report(rows[i], fs=int(fs[i]), lo=int(lo[i]), hi=int(hi[i]))
        _check_base(rep[i]["base"], want["base"], nm)
        _check_fields(rep[i], want, nm)
    r = {nm: rep[i] for i, nm in enumerate(names)}
    assert r["L>=100000"]["hnr_len"] == 100000 and np.isfinite(r["L>=100000"]["hnr_db"])
    assert r["sum S^2 > 2^64"]["hnr_len"] == 100 and np.isfinite(r["sum S^2 > 2^64"]["hnr_db"])
    assert np.isnan(r["zero peak"]["shimmer_db"]) and np.isfinite(r["zero peak"]["shimmer_apq3_pct"])
    assert r["overflow"]["base"]["flags"] == 1 and r["overflow"]["hnr_len"] == 0
    for nm in ("overflow", "silence", "K=0", "K=1"):
        assert all(np.isnan(r[nm][k]) for k in rr.FIELDS), nm
    assert np.isnan(r["K=10"]["shimmer_apq11_pct"]) and np.isfinite(r["K=11"]["shimmer_apq11_pct"])


NOISE_ONLY = ["-n 20", "-n 30", "-n 40", "-n 25 -f 200 -g 230 -r 44100", "-n 35 -f 90 -g 120 -a 5000",
              "-n 30 -r 44100 -a 20000", "-n 20 -r 44100 -a 5000"]


def test_hnr_of_gpu_generated_noise_only_voices(ctx, vs):
    """noise only (no jitter, no shimmer): the cycle-averaged HNR is the SNR the generator logged"""
    args = [("-d 2 " + a).split() for a in NOISE_ONLY]
    p = vs.FlowParams.from_cli(args, list(range(40, 40 + len(args))))
    flow, offs, ns, log = ctx.flowgen_batch(p, want_log=True)
    lo, hi = (p.amp * 0.08).astype(np.int16), (p.amp * 0.15).astype(np.int16)
    rep = ctx.flow_report_batch(flow, ns, offsets=offs, fs=p.fs, lo=lo, hi=hi)
    for i in range(p.n):
        K = int(rep[i]["base"]["cycles"])
        lg = log[i][:K]
        snr = 10 * math.log10(float((lg["x_pow"].astype(np.float64) * (lg["T3"] - lg["T4"])).sum()) /
                              float((lg["w_pow"].astype(np.float64) * lg["T"]).sum()))
        assert K > 100 and abs(K - len(log[i])) <= 2, NOISE_ONLY[i]
        assert abs(float(rep[i]["hnr_db"]) - snr) < 0.1, (NOISE_ONLY[i], rep[i]["hnr_db"], snr)


def test_report_errors_match_analysis(ctx, vs):
    L, h = ctx.L, ctx.h
    x = np.zeros(64, dtype=np.int16)
    ns = np.array([64], dtype=np.uint64)
    lo, hi = np.array([3], dtype=np.int16), np.array([2], dtype=np.int16)
    bad_fs = np.array([0], dtype=np.int32)
    st = np.zeros(1, dtype=vs.FLOW_STATS_DTYPE)
    rep = np.zeros(1, dtype=vs.FLOW_REPORT_DTYPE)
    p = lambda a: None if a is None else a.ctypes.data
    cases = [(x, ns, None, lo, hi, vs.VS_ERANGE), (x, ns, bad_fs, None, None, vs.VS_ERANGE),
             (None, ns, None, None, None, vs.VS_EINVAL), (x, None, None, None, None, vs.VS_EINVAL)]
    for flow, n_, fs, tl, th, code in cases:
        a = L.vs_flow_analyze_batch(h, p(flow), None, p(n_), p(fs), p(tl), p(th), 1, st.ctypes.data)
        b = L.vs_flow_report_batch(h, p(flow), None, p(n_), p(fs), p(tl), p(th), 1, rep.ctypes.data)
        assert a == b == code
    assert L.vs_flow_report_batch(h, x.ctypes.data, None, ns.ctypes.data, None, None, None, 1, None) == vs.VS_EINVAL
    assert L.vs_flow_report_batch(None, x.ctypes.data, None, ns.ctypes.data, None, None, None, 1, rep.ctypes.data) == vs.VS_EINVAL
    assert L.vs_flow_report_batch(h, x.ctypes.data, None, ns.ctypes.data, None, None, None, 0, rep.ctypes.data) == vs.VS_OK
    with pytest.raises(vs.VsError):
        ctx.flow_report_batch(x, [64], lo=3, hi=2)
    ctx.flow_report_batch(x, [64])                    # the context still works


def _payload(path):
    data = pathlib.Path(path).read_bytes()
    return np.frombuffer(data[44:], dtype="<i2")


def test_acoustic_tool_report_columns(tmp_path):
    """host/bin/acoustic -x on WAV files written by host/bin/flowgen_shimmer: the first nine columns are the line
    without -x, the ten after them the report of tests/report_ref.py"""
    bins = ROOT / "host" / "bin"
    if not (bins / "acoustic").exists():
        subprocess.run(["make", "-s", "-C", str(ROOT), "host"], check=True)
    files = []
    for k, args in enumerate(["-d 1 -f 110 -g 140 -j 2 -s 6", "-d 0.8 -f 201 -g 260", "-d 1.2 -f 87 -g 120 -j 0.5 -a 9000",
                              "-d 1 -f 130 -g 160 -s 3 -n 30"]):
        f = tmp_path / f"v{k}.wav"
        r = subprocess.run([str(bins / "flowgen_shimmer"), "-o", str(f)] + args.split(), env=dict(os.environ, VS_SEED=str(200 + k)),
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        files.append(f)
    lo, hi = "960", "1800"                               # 8 % and 15 % of the amplitude: above the noise, below every pulse
    plain = subprocess.run([str(bins / "acoustic"), "-l", lo, "-h", hi] + [str(f) for f in files], capture_output=True, text=True)
    ext = subprocess.run([str(bins / "acoustic"), "-l", lo, "-x", "-h", hi] + [str(f) for f in files], capture_output=True, text=True)
    assert plain.returncode == 0 and ext.returncode == 0, plain.stderr + ext.stderr
    plain_lines, ext_lines = plain.stdout.strip().splitlines(), ext.stdout.strip().splitlines()
    assert len(plain_lines) == len(ext_lines) == len(files)
    for f, pl, el in zip(files, plain_lines, ext_lines):
        t = el.split()
        assert len(t) == 19 and t[:9] == pl.split()
        want = rr.report(_payload(f), fs=22050, lo=int(lo), hi=int(hi))
        for got, key, nd in zip(t[9:], rr.FIELDS, (3, 4, 4, 4, 4, 4, 4, 4, 4, 3)):
            w = want[key]
            if math.isnan(w) or math.isinf(w):
                assert got == str(w).lower(), (f.name, key, got, w)
            else:
                assert abs(float(got) - w) <= 0.6 * 10 ** -nd + 1e-5 * abs(w), (f.name, key, got, w)
    # the second voice has neither jitter nor shimmer: every quotient is 0, the HNR +inf
    t = ext_lines[1].split()
    assert all(float(v) == 0.0 for v in t[9:18]) and t[18] == "inf"
