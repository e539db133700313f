"""numpy-level wrappers of the three batch entry points (include/voicesynth.h).

`FlowParams.from_cli()` mirrors the reference's argv handling and initialization()
(flowgen_shimmer.c:128-219, 463-547) value for value, so the parity tests read like invocations of
the reference tools.
"""
import ctypes as C
import math
import re

import numpy as np

from . import _lib
from ._lib import FilterParamsC, FlowParamsC, FormantOptsC, PeriodLogC, TimingC, TractParamsC

VS_F_JITTER, VS_F_SHIMMER, VS_F_NOISE = 1, 2, 4
VS_OK, VS_EINVAL, VS_ERANGE, VS_EPRESET, VS_ENOMEM, VS_ECUDA, VS_ENODEV, VS_EOVERLAP = 0, -1, -2, -3, -4, -5, -6, -7
OPT_CHUNK_SAMPLES, OPT_CARRY_TOL, OPT_EXACT_FILTER, OPT_SLAB_STREAMS, OPT_TARGET_WARPS, OPT_ASYNC_HOST, OPT_PLAN_WARPS, OPT_SIMPLE_GEN = 1, 2, 3, 4, 5, 7, 8, 9

PERIOD_DTYPE = np.dtype([("T", "<i4"), ("T2", "<i4"), ("T3", "<i4"), ("T4", "<i4"), ("A", "<f4"), ("Knew", "<f4"),
                         ("S", "<f4"), ("ndraws", "<i4"), ("ndw", "<i4"), ("x_pow", "<f4"), ("w_pow", "<f4"),
                         ("reserved", "<u4"), ("start", "<u8")])
assert PERIOD_DTYPE.itemsize == 56
FLOW_STATS_DTYPE = np.dtype([("onsets", "<u4"), ("cycles", "<u4"), ("flags", "<u4"), ("f0_hz", "<f4"), ("jitter_pct", "<f4"),
                             ("shimmer_pct", "<f4"), ("mean_period", "<f4"), ("mean_peak", "<f4")])
assert FLOW_STATS_DTYPE.itemsize == 32
FLOW_REPORT_DTYPE = np.dtype([("base", FLOW_STATS_DTYPE), ("jitter_abs_us", "<f4"), ("jitter_rap_pct", "<f4"),
                              ("jitter_ppq5_pct", "<f4"), ("jitter_ddp_pct", "<f4"), ("shimmer_db", "<f4"),
                              ("shimmer_apq3_pct", "<f4"), ("shimmer_apq5_pct", "<f4"), ("shimmer_apq11_pct", "<f4"),
                              ("shimmer_dda_pct", "<f4"), ("hnr_db", "<f4"), ("hnr_len", "<u4"), ("reserved", "<u4")])
assert FLOW_REPORT_DTYPE.itemsize == 80
MAX_FORMANTS = 8
FRAME_SILENT, FRAME_SINGULAR, FRAME_NOCONV = 1, 2, 4
FORMANT_FRAME_DTYPE = np.dtype([("f_hz", "<f4", (MAX_FORMANTS,)), ("bw_hz", "<f4", (MAX_FORMANTS,)), ("found", "<u4"),
                                ("flags", "<u4")])
assert FORMANT_FRAME_DTYPE.itemsize == 72
FORMANT_STATS_DTYPE = np.dtype([("frames", "<u4"), ("analysed", "<u4"), ("unconverged", "<u4"), ("reserved", "<u4"),
                                ("count", "<u4", (MAX_FORMANTS,)), ("f_mean_hz", "<f4", (MAX_FORMANTS,)),
                                ("f_sd_hz", "<f4", (MAX_FORMANTS,)), ("bw_mean_hz", "<f4", (MAX_FORMANTS,))])
assert FORMANT_STATS_DTYPE.itemsize == 144
FORMANT_DEFAULTS = dict(win_ms=25.0, hop_ms=10.0, preemph_hz=50.0, bmax_hz=700.0, order=14, n_formants=5)

_FLOW_FIELDS = [("dur", np.float32, 1.0), ("jitter", np.float32, 0.0), ("shimmer", np.float32, 0.0),
                ("cq", np.float32, 0.55), ("K", np.float32, 0.65), ("Kvar", np.float32, 0.0), ("F0", np.float32, 120.0),
                ("DC", np.float32, 0.0), ("noise", np.float32, 0.0), ("amp", np.int32, 12000), ("fs", np.int32, 22050),
                ("flags", np.uint8, 0), ("seed", np.uint32, 1)]


class VsError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libvoicesynth_cuda error {code}: {msg}")
        self.code = code


def lib_path():
    return _lib.LIB_PATH


def _atof(s):
    m = re.match(r"\s*[-+]?(\d+\.?\d*([eE][-+]?\d+)?|\.\d+([eE][-+]?\d+)?|inf|nan)", s, flags=re.I)
    return float(m.group(0)) if m else 0.0


def _atoi(s):
    m = re.match(r"\s*[-+]?\d+", s)
    return int(m.group(0)) if m else 0


class FlowParams:
    """SoA flow parameters (struct PAR after initialization(), flowgen_shimmer.c:73-87)."""

    def __init__(self, n, **kw):
        self.n = n
        for name, dt, default in _FLOW_FIELDS:
            setattr(self, name, np.full(n, default, dtype=dt))
        for k, v in kw.items():
            arr = getattr(self, k)
            arr[...] = v

    @staticmethod
    def cli_row(args):
        """One stream from reference-style CLI args (without -o). Returns a dict, or None where the
        reference would print usage() and exit (flowgen_shimmer.c:463-547)."""
        f32 = np.float32
        row = {name: dt(default) for name, dt, default in _FLOW_FIELDS}
        given = {}
        args = list(args)
        i = 0
        while i < len(args) and args[i].startswith("-"):
            if i + 1 >= len(args):
                return None
            c = args[i][1:2].lower()
            if c not in "ogfdcjknralzs" or c == "":
                return None
            if c == "n":
                row["DC"] = f32(0.25)
            given[c] = args[i + 1]
            i += 2
        if i != len(args) and not args[i].startswith("i"):
            return None
        Fg = f32(125.0)
        if "d" in given:
            f = f32(_atof(given["d"]))
            if not f >= 0.5:
                return None
            row["dur"] = f
        if "j" in given:
            f = f32(_atof(given["j"]) / 100.0)
            if not (f >= 0.0 and f <= 10.0):
                return None
            row["jitter"] = f
        if "k" in given:
            f = f32(_atof(given["k"]))
            if not f >= 0.5:
                return None
            row["K"] = f
        if "c" in given:
            f = f32(_atof(given["c"]))
            if not (f >= 0.0 and f <= 1.0):
                return None
            row["cq"] = f
        if "g" in given:
            f = f32(_atof(given["g"]))
            if not f >= 50:
                return None
            Fg = f
        if "f" in given:
            f = f32(_atof(given["f"]))
            if not (f >= 50 and f < Fg):
                return None
            row["F0"] = f
        if "n" in given:
            f = f32(_atof(given["n"]))
            if not (f >= 0.0 and f <= 50):
                return None
            row["noise"] = f32(math.pow(10.0, float(f / f32(10))))
        if "a" in given:
            v = _atoi(given["a"])
            if not (0 <= v < 32767):
                return None
            row["amp"] = np.int32(v)
        if "l" in given:
            f = f32(_atof(given["l"]))
            if not (f >= 0 and f <= f32(0.3) + 0 and float(f) <= 0.3):
                return None
            row["DC"] = f * f32(row["amp"])
        if "z" in given:
            f = f32(_atof(given["z"]))
            if not (f >= 0 and f <= 1):
                return None
            row["Kvar"] = f
        if "r" in given:
            v = _atoi(given["r"])
            if v == 22050:          # the reference's range test rejects exactly this value (:537)
                return None
            row["fs"] = np.int32(v)
        if "s" in given:
            f = f32(_atof(given["s"]))
            if not (f >= 0 and f <= 100):
                return None
            row["shimmer"] = f / f32(100)
        row["flags"] = np.uint8((VS_F_JITTER if "j" in given else 0) | (VS_F_SHIMMER if "s" in given else 0) |
                                (VS_F_NOISE if "n" in given else 0))
        return row

    @classmethod
    def from_cli(cls, arg_lists, seeds):
        """arg_lists: list of CLI strings/lists (no -o needed); seeds: per-stream srandom() seeds."""
        p = cls(len(arg_lists))
        for i, a in enumerate(arg_lists):
            row = cls.cli_row(a.split() if isinstance(a, str) else a)
            if row is None:
                raise ValueError(f"stream {i}: the reference rejects {a!r} (usage)")
            for name, _, _ in _FLOW_FIELDS:
                if name != "seed":
                    getattr(p, name)[i] = row[name]
        p.seed[...] = np.asarray(seeds, dtype=np.uint32)
        return p

    def select(self, idx):
        q = FlowParams(len(idx))
        for name, _, _ in _FLOW_FIELDS:
            getattr(q, name)[...] = getattr(self, name)[idx]
        if getattr(self, "meta", None):
            q.meta = {k: (None if v is None else v[idx]) for k, v in self.meta.items()}
        return q

    def _c(self):
        c = FlowParamsC()
        for name, dt, _ in _FLOW_FIELDS:
            arr = np.ascontiguousarray(getattr(self, name), dtype=dt)
            setattr(self, name, arr)
            setattr(c, name, arr.ctypes.data)
        return c


class FilterParams:
    """SoA vowel filter parameters (vowel_new.c:76-77,116-192)."""

    def __init__(self, n, preset="a", gain=10.0, pre=1.0):
        self.n = n
        if isinstance(preset, str) and len(preset) == n and n > 1:
            preset = [ord(ch) for ch in preset]
        elif isinstance(preset, str):
            preset = ord(preset)
        self.preset = np.full(n, 0, dtype=np.uint8)
        self.preset[...] = preset
        self.gain = np.full(n, gain, dtype=np.float32)
        self.pre = np.full(n, pre, dtype=np.float32)

    def select(self, idx):
        q = FilterParams(len(idx))
        q.preset[...] = self.preset[idx]
        q.gain[...] = self.gain[idx]
        q.pre[...] = self.pre[idx]
        return q

    def _c(self):
        c = FilterParamsC()
        c.preset, c.gain, c.pre = self.preset.ctypes.data, self.gain.ctypes.data, self.pre.ctypes.data
        return c


class TractParams:
    """Caller-defined vocal tracts (vs_tract_params): den is [n_tracts][23] (A[0..22] of 1/A(z), A[0] = 1), tract the
    per-stream index into it (None: 0 for every stream); gain and pre as in FilterParams."""

    def __init__(self, n, den, tract=None, gain=10.0, pre=1.0):
        self.n = n
        self.den = np.ascontiguousarray(np.atleast_2d(np.asarray(den, dtype=np.float64)))
        if self.den.shape[1] != 23:
            raise ValueError(f"den must be [n_tracts][23], got {self.den.shape}")
        self.tract = np.zeros(n, dtype=np.uint8)
        if tract is not None:
            self.tract[...] = tract
        self.gain = np.full(n, gain, dtype=np.float32)
        self.pre = np.full(n, pre, dtype=np.float32)

    def select(self, idx):
        q = TractParams(len(idx), self.den)
        q.tract[...] = self.tract[idx]
        q.gain[...] = self.gain[idx]
        q.pre[...] = self.pre[idx]
        return q

    def _c(self):
        return TractParamsC(self.den.ctypes.data, self.den.shape[0], self.tract.ctypes.data, self.gain.ctypes.data,
                            self.pre.ctypes.data)


def _den_or_raise(rc, den):
    if rc:
        raise VsError(rc, _lib.load().vs_strerror(rc).decode())
    return den


def tract_from_formants(freqs, bws, fs):
    """den[23] of the cascade of formant resonators (F_k, B_k in Hz) at sampling rate fs (vs_tract_from_formants)."""
    f = np.ascontiguousarray(freqs, dtype=np.float32)
    b = np.ascontiguousarray(bws, dtype=np.float32)
    if f.shape != b.shape:
        raise ValueError("freqs and bws differ in length")
    den = np.zeros(23, dtype=np.float64)
    return _den_or_raise(_lib.load().vs_tract_from_formants(f.ctypes.data, b.ctypes.data, f.size, int(fs), den.ctypes.data), den)


def tract_from_preset(key):
    """den[23] of a vowel preset ('a','i','u','1'..'7'), for mixing presets and custom tracts in one call."""
    den = np.zeros(23, dtype=np.float64)
    return _den_or_raise(_lib.load().vs_tract_from_preset(ord(key), den.ctypes.data), den)


def flow_validate(p):
    """(VS_OK, None) or (error code, index of the first offending stream): the checks vs_*_batch apply up front."""
    bad = C.c_size_t(0)
    rc = _lib.load().vs_flow_validate(C.byref(p._c()), p.n, C.byref(bad))
    return (rc, None) if rc == 0 else (rc, int(bad.value))


def flow_nsamples(p):
    out = np.zeros(p.n, dtype=np.uint64)
    _lib.load().vs_flow_nsamples(C.byref(p._c()), p.n, out.ctypes.data)
    return out


def formant_opts(opts=None):
    """vs_formant_opts from a dict of the fields to change (the rest keep FORMANT_DEFAULTS); None stays None (NULL)"""
    if opts is None or isinstance(opts, FormantOptsC):
        return opts
    unknown = set(opts) - set(FORMANT_DEFAULTS)
    if unknown:
        raise ValueError(f"unknown formant options {sorted(unknown)}")
    return FormantOptsC(**{**FORMANT_DEFAULTS, **opts})


def formant_frames(nsamp, fs=None, opts=None):
    """frames per stream of vs_formant_batch (host only, validates like the batch call; raises VsError)"""
    ns = np.ascontiguousarray(nsamp, dtype=np.uint64)
    rate = _per_stream(fs, np.int32, len(ns))
    o = formant_opts(opts)
    out = np.zeros(len(ns), dtype=np.uint64)
    rc = _lib.load().vs_formant_frames(None if o is None else C.byref(o), ns.ctypes.data, _ptr(rate), len(ns), out.ctypes.data)
    if rc:
        raise VsError(rc, _lib.load().vs_strerror(rc).decode())
    return out


def _per_stream(x, dtype, n):
    """a per-stream argument as n contiguous values of dtype (a scalar stands for every stream); None stays None (NULL)"""
    return None if x is None else np.ascontiguousarray(np.broadcast_to(np.asarray(x, dtype=dtype), (n,)))


def _ptr(x):
    """numpy array -> host pointer; int -> raw (device) pointer; object with data_ptr() -> torch tensor."""
    if x is None:
        return None
    if isinstance(x, np.ndarray):
        assert x.flags["C_CONTIGUOUS"]
        return x.ctypes.data
    if hasattr(x, "data_ptr"):
        return x.data_ptr()
    return int(x)


class Context:
    """vs_ctx wrapper. devices: list of CUDA device indices (default [0])."""

    def __init__(self, devices=None, stream=None):
        self.L = _lib.load()
        self.h = C.c_void_p()
        devs = list(devices) if devices else [0]
        arr = (C.c_int * len(devs))(*devs)
        rc = self.L.vs_ctx_create(C.byref(self.h), arr, len(devs), 0)
        if rc:
            raise VsError(rc, self.L.vs_strerror(rc).decode())
        if stream is not None:
            self._check(self.L.vs_ctx_set_stream(self.h, 0, C.c_void_p(stream)))

    def close(self):
        if self.h:
            self.L.vs_ctx_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc:
            raise VsError(rc, f"{self.L.vs_strerror(rc).decode()}: {self.L.vs_last_error(self.h).decode()}")

    def set_option(self, opt, value):
        self._check(self.L.vs_ctx_set_option(self.h, opt, float(value)))

    def sync(self):
        self._check(self.L.vs_sync(self.h))

    def timing(self):
        t = TimingC()
        self._check(self.L.vs_get_timing(self.h, C.byref(t)))
        return {k: getattr(t, k) for k, _ in TimingC._fields_}

    def fp64_peak(self):
        t, mhz = C.c_double(), C.c_double()
        self._check(self.L.vs_measure_fp64_peak(self.h, C.byref(t), C.byref(mhz)))
        return t.value, mhz.value

    def filter_warmup(self, preset, gain=10.0):
        return self.L.vs_filter_warmup(self.h, ord(preset), gain)

    # ---- batch calls -------------------------------------------------------------------------
    def _layout(self, ns, offsets):
        if offsets is None:
            stride = int(ns.max())
            offs = np.arange(len(ns), dtype=np.uint64) * np.uint64(stride)
            total = stride * len(ns)
            return None, offs, total
        offs = np.ascontiguousarray(offsets, dtype=np.uint64)
        return offs, offs, int((offs + ns).max())

    def flowgen_batch(self, p, out=None, offsets=None, want_log=False):
        ns = flow_nsamples(p)
        offs_arg, offs, total = self._layout(ns, offsets)
        if out is None:
            out = np.zeros(total, dtype=np.int16)
        logc, log = None, None
        if want_log:
            mp = np.zeros(p.n, dtype=np.uint64)
            self.L.vs_flow_max_periods(C.byref(p._c()), p.n, mp.ctypes.data)
            ro = np.concatenate([[0], np.cumsum(mp)]).astype(np.uint64)
            rec = np.zeros(int(ro[-1]), dtype=PERIOD_DTYPE)
            cnt = np.zeros(p.n, dtype=np.uint32)
            logc = PeriodLogC(rec.ctypes.data, ro.ctypes.data, cnt.ctypes.data)
            log = (rec, ro, cnt)
        self._check(self.L.vs_flowgen_batch(self.h, C.byref(p._c()), p.n, _ptr(out), _ptr(offs_arg),
                                            C.byref(logc) if logc else None))
        if want_log:
            rec, ro, cnt = log
            return out, offs, ns, [rec[int(ro[i]): int(ro[i]) + int(cnt[i])] for i in range(p.n)]
        return out, offs, ns

    def vowel_filter_batch(self, flow, nsamp, f, in_offsets=None, out=None, out_offsets=None, want_raw=False):
        ns = np.ascontiguousarray(nsamp, dtype=np.uint64)
        in_arg, _, _ = self._layout(ns, in_offsets)
        out_arg, offs, total = self._layout(ns, out_offsets)
        if out is None:
            out = np.zeros(total, dtype=np.int16)
        raw = np.zeros(total, dtype=np.float64) if want_raw is True else (want_raw if want_raw is not False else None)
        call = self.L.vs_vowel_filter_batch_tract if isinstance(f, TractParams) else self.L.vs_vowel_filter_batch
        self._check(call(self.h, _ptr(flow), _ptr(in_arg), ns.ctypes.data, C.byref(f._c()), len(ns), _ptr(out), _ptr(out_arg),
                         _ptr(raw)))
        return (out, offs, raw) if want_raw is not False else (out, offs)

    def vowel_noise_batch(self, pcm, nsamp, snr_db, seeds, offsets=None, fs=None):
        """`vowel -n`: in-place output noise on filtered PCM (vowel_new.c:302-324). snr_db <= 0 leaves a stream alone."""
        ns = np.ascontiguousarray(nsamp, dtype=np.uint64)
        n = len(ns)
        db = np.broadcast_to(np.asarray(snr_db, dtype=np.float32), (n,))
        snr = np.array([np.float32(math.pow(10.0, float(d / np.float32(10)))) if d > 0 else np.float32(0) for d in db], dtype=np.float32)
        offs, rate, sd = (_per_stream(x, dt, n) for x, dt in ((offsets, np.uint64), (fs, np.int32), (seeds, np.uint32)))
        self._check(self.L.vs_vowel_noise_batch(self.h, _ptr(pcm), _ptr(offs), ns.ctypes.data, snr.ctypes.data,
                                                _ptr(rate), sd.ctypes.data, n))
        return pcm

    def flow_analyze_batch(self, flow, nsamp, offsets=None, fs=None, lo=None, hi=None):
        """cycle-to-cycle analysis of glottal flow (SURVEY 8f N4, include/voicesynth.h): F0, local jitter and shimmer
        per stream as a structured array (FLOW_STATS_DTYPE). flow: numpy array or device tensor."""
        return self._analysis(self.L.vs_flow_analyze_batch, FLOW_STATS_DTYPE, flow, nsamp, offsets, fs, lo, hi)

    def flow_report_batch(self, flow, nsamp, offsets=None, fs=None, lo=None, hi=None):
        """voice report of glottal flow (include/voicesynth.h): flow_analyze_batch's statistics in `base`, Praat's jitter
        and shimmer quotients and a cycle-averaged HNR, per stream as a structured array (FLOW_REPORT_DTYPE)."""
        return self._analysis(self.L.vs_flow_report_batch, FLOW_REPORT_DTYPE, flow, nsamp, offsets, fs, lo, hi)

    def _analysis(self, call, dtype, flow, nsamp, offsets, fs, lo, hi):
        ns = np.ascontiguousarray(nsamp, dtype=np.uint64)
        n = len(ns)
        offs, rate, tl, th = (_per_stream(x, dt, n) for x, dt in ((offsets, np.uint64), (fs, np.int32), (lo, np.int16), (hi, np.int16)))
        res = np.zeros(n, dtype=dtype)
        self._check(call(self.h, _ptr(flow), _ptr(offs), ns.ctypes.data, _ptr(rate), _ptr(tl), _ptr(th), n, res.ctypes.data))
        return res

    def formant_batch(self, pcm, nsamp, offsets=None, fs=None, opts=None, want_frames=False):
        """formant analysis (vs_formant_batch): per-stream statistics (FORMANT_STATS_DTYPE) and, with want_frames, the
        list of each stream's frame records (FORMANT_FRAME_DTYPE).  pcm: numpy array or device tensor; opts: None (the
        defaults) or a dict of the vs_formant_opts fields to change."""
        ns = np.ascontiguousarray(nsamp, dtype=np.uint64)
        n = len(ns)
        offs, rate = (_per_stream(x, dt, n) for x, dt in ((offsets, np.uint64), (fs, np.int32)))
        o = formant_opts(opts)
        st = np.zeros(n, dtype=FORMANT_STATS_DTYPE)
        fr, fo = None, None
        if want_frames:
            fo = np.concatenate([[0], np.cumsum(formant_frames(ns, fs, opts))]).astype(np.uint64)
            fr = np.zeros(int(fo[-1]), dtype=FORMANT_FRAME_DTYPE)
        self._check(self.L.vs_formant_batch(self.h, _ptr(pcm), _ptr(offs), ns.ctypes.data, _ptr(rate), n,
                                            None if o is None else C.byref(o), st.ctypes.data, _ptr(fr), None))
        if want_frames:
            return st, [fr[int(fo[i]): int(fo[i + 1])] for i in range(n)]
        return st

    def synth_batch(self, p, f, out=None, offsets=None, want_raw=False):
        """f: FilterParams (the presets) or TractParams (caller-defined tracts, vs_synth_batch_tract)."""
        call = self.L.vs_synth_batch_tract if isinstance(f, TractParams) else self.L.vs_synth_batch
        if out is not None and offsets is None and want_raw is False:
            # fast path for repeated calls into a caller-owned dense buffer: nothing to size or return
            self._check(call(self.h, C.byref(p._c()), C.byref(f._c()), p.n, _ptr(out), None, None))
            return out, None, None
        ns = flow_nsamples(p)
        offs_arg, offs, total = self._layout(ns, offsets)
        if out is None:
            out = np.zeros(total, dtype=np.int16)
        raw = np.zeros(total, dtype=np.float64) if want_raw is True else (want_raw if want_raw is not False else None)
        self._check(call(self.h, C.byref(p._c()), C.byref(f._c()), p.n, _ptr(out), _ptr(offs_arg), _ptr(raw)))
        return (out, offs, ns, raw) if want_raw is not False else (out, offs, ns)
