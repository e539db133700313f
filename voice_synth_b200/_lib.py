"""ctypes declarations for include/voicesynth.h.  Loading fails loudly if the .so is missing."""
import ctypes as C
import pathlib

LIB_PATH = pathlib.Path(__file__).resolve().parent / "lib" / "libvoicesynth_cuda.so"

EXPORTS = ["vs_abi_version", "vs_device_count", "vs_strerror", "vs_last_error", "vs_ctx_create", "vs_ctx_destroy",
           "vs_ctx_set_option", "vs_ctx_set_stream", "vs_sync", "vs_get_timing", "vs_measure_fp64_peak", "vs_host_alloc", "vs_host_free",
           "vs_flow_nsamples", "vs_flow_max_periods", "vs_flow_validate", "vs_filter_warmup",
           "vs_flowgen_batch", "vs_vowel_filter_batch", "vs_synth_batch", "vs_vowel_noise_batch", "vs_flow_analyze_batch",
           "vs_flow_report_batch", "vs_synth_batch_tract", "vs_vowel_filter_batch_tract", "vs_tract_from_formants", "vs_tract_from_preset",
           "vs_formant_frames", "vs_formant_batch", "vs_pitch_frames", "vs_pitch_batch",
           "vs_vowel_mark_slots", "vs_vowel_report_batch"]


class FlowParamsC(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("dur", "jitter", "shimmer", "cq", "K", "Kvar", "F0", "DC", "noise",
                                          "amp", "fs", "flags", "seed")]


class FilterParamsC(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("preset", "gain", "pre")]


class TractParamsC(C.Structure):
    _fields_ = [("den", C.c_void_p), ("n_tracts", C.c_uint32), ("tract", C.c_void_p), ("gain", C.c_void_p), ("pre", C.c_void_p)]


class FormantOptsC(C.Structure):
    _fields_ = [("win_ms", C.c_float), ("hop_ms", C.c_float), ("preemph_hz", C.c_float), ("bmax_hz", C.c_float),
                ("order", C.c_uint32), ("n_formants", C.c_uint32)]


class PitchOptsC(C.Structure):
    _fields_ = [(k, C.c_float) for k in ("f_min_hz", "f_max_hz", "periods", "hop_ms", "voicing_threshold", "silence_threshold",
                                         "octave_cost")]


class PeriodLogC(C.Structure):
    _fields_ = [("rec", C.c_void_p), ("rec_offsets", C.c_void_p), ("count", C.c_void_p)]


class TimingC(C.Structure):
    _fields_ = [("plan_ms", C.c_float), ("render_ms", C.c_float), ("total_ms", C.c_float), ("launches", C.c_uint32),
                ("chunks", C.c_uint32), ("samples", C.c_uint64), ("warmup_samples", C.c_uint64),
                ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
                ("render_path", C.c_uint32), ("reserved", C.c_uint32)]


_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise ImportError(f"{LIB_PATH} is missing: build it with `make lib` (nvcc, sm_100a). "
                          "voice_synth_b200 has no CPU fallback.")
    L = C.CDLL(str(LIB_PATH))
    L.vs_strerror.restype = C.c_char_p
    L.vs_strerror.argtypes = [C.c_int]
    L.vs_last_error.restype = C.c_char_p
    L.vs_last_error.argtypes = [C.c_void_p]
    L.vs_ctx_create.argtypes = [C.POINTER(C.c_void_p), C.POINTER(C.c_int), C.c_int, C.c_uint32]
    L.vs_ctx_destroy.argtypes = [C.c_void_p]
    L.vs_ctx_destroy.restype = None
    L.vs_ctx_set_option.argtypes = [C.c_void_p, C.c_int, C.c_double]
    L.vs_ctx_set_stream.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    L.vs_sync.argtypes = [C.c_void_p]
    L.vs_get_timing.argtypes = [C.c_void_p, C.POINTER(TimingC)]
    L.vs_measure_fp64_peak.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.vs_host_alloc.restype = C.c_void_p
    L.vs_host_alloc.argtypes = [C.c_size_t]
    L.vs_host_free.argtypes = [C.c_void_p]
    L.vs_host_free.restype = None
    L.vs_flow_nsamples.argtypes = [C.POINTER(FlowParamsC), C.c_size_t, C.c_void_p]
    L.vs_flow_max_periods.argtypes = [C.POINTER(FlowParamsC), C.c_size_t, C.c_void_p]
    L.vs_flow_validate.argtypes = [C.POINTER(FlowParamsC), C.c_size_t, C.POINTER(C.c_size_t)]
    L.vs_filter_warmup.argtypes = [C.c_void_p, C.c_int, C.c_float]
    L.vs_flowgen_batch.argtypes = [C.c_void_p, C.POINTER(FlowParamsC), C.c_size_t, C.c_void_p, C.c_void_p,
                                   C.POINTER(PeriodLogC)]
    L.vs_vowel_filter_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(FilterParamsC),
                                        C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]
    L.vs_vowel_noise_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_size_t]
    L.vs_synth_batch.argtypes = [C.c_void_p, C.POINTER(FlowParamsC), C.POINTER(FilterParamsC), C.c_size_t,
                                 C.c_void_p, C.c_void_p, C.c_void_p]
    L.vs_flow_analyze_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_size_t, C.c_void_p]
    L.vs_flow_report_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_size_t, C.c_void_p]
    L.vs_synth_batch_tract.argtypes = [C.c_void_p, C.POINTER(FlowParamsC), C.POINTER(TractParamsC), C.c_size_t,
                                       C.c_void_p, C.c_void_p, C.c_void_p]
    L.vs_vowel_filter_batch_tract.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(TractParamsC),
                                              C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]
    L.vs_tract_from_formants.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int32, C.c_void_p]
    L.vs_tract_from_preset.argtypes = [C.c_int, C.c_void_p]
    L.vs_formant_frames.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    L.vs_formant_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p]
    L.vs_pitch_frames.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    L.vs_pitch_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_void_p]
    L.vs_vowel_mark_slots.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    L.vs_vowel_report_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p]
    _lib = L
    return L
