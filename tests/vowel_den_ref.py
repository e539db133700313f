"""TEST ONLY: ctypes front-end of tests/tools/vowel_den.c, the reference's vocal-tract filter with a caller-given
denominator -- the yardstick of the tract calls (vs_synth_batch_tract, vs_vowel_filter_batch_tract)."""
import ctypes as C
import pathlib
import subprocess

import numpy as np

SRC = pathlib.Path(__file__).resolve().parent / "tools" / "vowel_den.c"


class VowelDen:
    def __init__(self, build_dir):
        so = pathlib.Path(build_dir) / "libvowel_den.so"
        subprocess.run(["gcc", "-O2", "-fPIC", "-shared", "-ffp-contract=off", str(SRC), "-o", str(so), "-lm"], check=True)
        self.L = C.CDLL(str(so))
        self.L.vowel_den.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_float, C.c_float, C.c_void_p, C.c_void_p]

    def __call__(self, flow, den, gain=10.0, pre=1.0, want_raw=False):
        flow = np.ascontiguousarray(flow, dtype=np.int16)
        A = np.ascontiguousarray(den, dtype=np.float64)
        assert A.shape == (23,)
        out = np.zeros_like(flow)
        raw = np.zeros(flow.size, dtype=np.float64) if want_raw else None
        rc = self.L.vowel_den(flow.ctypes.data, flow.size, A.ctypes.data, gain, pre, out.ctypes.data,
                              raw.ctypes.data if want_raw else None)
        assert rc == 0
        return (out, raw) if want_raw else out
