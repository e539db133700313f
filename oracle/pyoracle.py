"""ctypes front-end of the CPU oracle (oracle/vs_oracle.c).  TEST INFRASTRUCTURE ONLY.

May be imported by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs -- never by voice_synth_b200/ (tests/test_no_oracle_in_product.py enforces that).
"""
import ctypes as C
import os
import pathlib
import subprocess

import numpy as np

HERE = pathlib.Path(__file__).resolve().parent
LIB = HERE / "_build" / "libvs_oracle.so"
REF_DIR = HERE / "_ref"


class FlowPar(C.Structure):
    _fields_ = [("dur", C.c_float), ("jitter", C.c_float), ("cq", C.c_float), ("K", C.c_float),
                ("Fg", C.c_float), ("F0", C.c_float), ("DC", C.c_float), ("noise", C.c_float),
                ("fs", C.c_int64), ("amp", C.c_int32), ("Kvar", C.c_float), ("shimmer", C.c_float),
                ("has_jitter", C.c_int32), ("has_shimmer", C.c_int32), ("has_noise", C.c_int32),
                ("seed", C.c_uint32)]


class Period(C.Structure):
    _fields_ = [("T", C.c_int32), ("T2", C.c_int32), ("T3", C.c_int32), ("T4", C.c_int32),
                ("A", C.c_float), ("Knew", C.c_float), ("S", C.c_float), ("ndraws", C.c_int32),
                ("ndw", C.c_int32), ("x_pow", C.c_float), ("w_pow", C.c_float), ("start", C.c_uint64)]


PERIOD_DTYPE = np.dtype([("T", "<i4"), ("T2", "<i4"), ("T3", "<i4"), ("T4", "<i4"), ("A", "<f4"),
                         ("Knew", "<f4"), ("S", "<f4"), ("ndraws", "<i4"), ("ndw", "<i4"),
                         ("x_pow", "<f4"), ("w_pow", "<f4"), ("_pad", "<i4"), ("start", "<u8")])
assert PERIOD_DTYPE.itemsize == C.sizeof(Period)


class Rng(C.Structure):
    _fields_ = [("r", C.c_uint32 * 31), ("f", C.c_int), ("b", C.c_int)]


_lib = None


def build():
    subprocess.run(["make", "-s", "-C", str(HERE), "oracle"], check=True)


def lib():
    global _lib
    if _lib is None:
        if not LIB.exists() or LIB.stat().st_mtime < (HERE / "vs_oracle.c").stat().st_mtime:
            build()
        L = C.CDLL(str(LIB))
        L.vso_random.restype = C.c_int32
        L.vso_flow_nsamples.restype = C.c_uint64
        L.vso_preset.restype = C.POINTER(C.c_double)
        L.vso_round2int.restype = C.c_int16
        L.vso_round2int.argtypes = [C.c_double]
        L.vso_flow_par_from_cli.argtypes = [C.c_int, C.POINTER(C.c_char_p), C.POINTER(FlowPar)]
        L.vso_flowgen.argtypes = [C.POINTER(FlowPar), C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]
        L.vso_vowel.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_float, C.c_float, C.c_void_p, C.c_void_p]
        L.vso_vowel_noise.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_float, C.c_float, C.c_float,
                                      C.c_int64, C.c_uint32, C.c_void_p]
        L.vso_noise.argtypes = [C.c_void_p, C.c_size_t, C.c_float, C.c_int64, C.c_uint32]
        _lib = L
    return _lib


def random_sequence(seed, n):
    g = Rng()
    lib().vso_srandom(C.byref(g), C.c_uint32(seed))
    return [lib().vso_random(C.byref(g)) for _ in range(n)]


def flow_par_from_cli(args, seed=1):
    """args: list like ['-o','x.wav','-d','1', ...] -> FlowPar, or None where the reference prints usage."""
    argv = [b"flowgen_shimmer"] + [a.encode() for a in args]
    arr = (C.c_char_p * len(argv))(*argv)
    p = FlowPar()
    p.seed = seed
    rc = lib().vso_flow_par_from_cli(len(argv), arr, C.byref(p))
    return p if rc == 0 else None


def flowgen(par, want_log=False):
    n = lib().vso_flow_nsamples(C.byref(par))
    out = np.zeros(n, dtype=np.int16)
    npd = C.c_size_t(0)
    cap = int(n // max(1, int(0.8 * int(par.fs / par.F0)) - 1) + 8) if want_log else 0
    log = np.zeros(cap, dtype=PERIOD_DTYPE)
    rc = lib().vso_flowgen(C.byref(par), out.ctypes.data, log.ctypes.data if want_log else None, cap, C.byref(npd))
    if rc:
        raise RuntimeError(f"vso_flowgen rc={rc}")
    if want_log:
        assert npd.value <= cap
        return out, log[: npd.value]
    return out


def vowel(flow, preset, gain=10.0, pre=1.0, want_raw=False):
    flow = np.ascontiguousarray(flow, dtype=np.int16)
    out = np.zeros_like(flow)
    raw = np.zeros(flow.size, dtype=np.float64) if want_raw else None
    rc = lib().vso_vowel(flow.ctypes.data, flow.size, ord(preset), gain, pre, out.ctypes.data,
                         raw.ctypes.data if want_raw else None)
    if rc:
        raise RuntimeError(f"vso_vowel rc={rc}")
    return (out, raw) if want_raw else out


def vowel_noise(flow, preset, snr_db, seed, gain=10.0, pre=1.0, fs=22050):
    flow = np.ascontiguousarray(flow, dtype=np.int16)
    out = np.zeros_like(flow)
    rc = lib().vso_vowel_noise(flow.ctypes.data, flow.size, ord(preset), gain, pre, snr_db, fs, seed, out.ctypes.data)
    if rc:
        raise RuntimeError(f"vso_vowel_noise rc={rc}")
    return out


def noise(pcm, snr_db, seed, fs=22050):
    """`vowel -n`'s output noise on already filtered PCM (the second half of vowel_noise): a new array"""
    out = np.array(pcm, dtype=np.int16, copy=True, order="C")
    rc = lib().vso_noise(out.ctypes.data, out.size, snr_db, fs, seed)
    if rc:
        raise RuntimeError(f"vso_noise rc={rc}")
    return out


def preset(key):
    p = lib().vso_preset(ord(key))
    return np.array([p[i] for i in range(23)])


# ---------------------------------------------------------------- unmodified reference binaries
def ref_available():
    return all((REF_DIR / f).exists() for f in ("flowgen_shimmer", "vowel", "timeshim.so"))


WAV_HDR_LP64 = 72   # sizeof(header) of the 64-bit build (SURVEY.md discrepancy 4)


def ref_flowgen(args, seed, workdir, opt="", name="f.wav"):
    """Run the unmodified reference flowgen_shimmer; returns (pcm int16 array, stdout text)."""
    path = pathlib.Path(workdir) / name
    env = dict(os.environ, VS_SEED=str(seed), LD_PRELOAD=str(REF_DIR / "timeshim.so"))
    r = subprocess.run([str(REF_DIR / ("flowgen_shimmer" + opt)), "-o", str(path)] + list(args),
                       env=env, capture_output=True, check=True)
    data = path.read_bytes()[WAV_HDR_LP64:]
    return np.frombuffer(data, dtype="<i2").copy(), r.stdout.decode(errors="replace")


def ref_vowel(in_wav, preset, seed, workdir, extra=(), opt="", name="v.wav"):
    path = pathlib.Path(workdir) / name
    env = dict(os.environ, VS_SEED=str(seed), LD_PRELOAD=str(REF_DIR / "timeshim.so"))
    subprocess.run([str(REF_DIR / ("vowel" + opt)), "-i", str(in_wav), "-o", str(path), "-v", preset] + list(extra),
                   env=env, capture_output=True, check=True)
    return np.frombuffer(path.read_bytes()[WAV_HDR_LP64:], dtype="<i2").copy()
