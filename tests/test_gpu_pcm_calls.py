"""The calls on PCM the caller owns: output noise (vs_vowel_noise_batch) on ragged rows in pageable, pinned and device
memory, and the refusals of the noise, flow analysis and voice report calls, each followed by a call that works."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
BIG = 2 ** 31                  # one sample above the 2^31-1 limit of a row


@pytest.fixture(scope="module")
def vs():
    from voice_synth_b200 import api
    return api


@pytest.fixture(scope="module")
def ctx(vs):
    c = vs.Context()
    yield c
    c.close()


def _arr(dtype, *v):
    return np.array(v, dtype=dtype)


def _p(a):
    return None if a is None else a.ctypes.data


@pytest.mark.parametrize("gap", [3, 0])
def test_noise_host_memory_ragged_rows(ctx, vs, gap):
    """the device batch of test_gpu_parity's output-noise test (a stream left alone by snr 0, a 1-sample stream) plus a
    zero-length stream, with `gap` samples between rows (0: touching rows come home as one copy): pageable, pinned and
    device memory give the same PCM, and every sample outside the noised rows is the input's"""
    import torch
    ns = _arr(np.uint64, 22050, 5000, 0, 1100, 1, 30000, 22050)
    offs = np.concatenate([[0], np.cumsum(ns + gap)[:-1]]).astype(np.uint64)
    snr = [30.0, 12.5, 25.0, 5.0, 20.0, 0.0, 40.0]
    fs = [22050, 44100, 22050, 11025, 22050, 22050, 16000]
    seeds = [1, 2, 9, 3, 4, 5, 4000000000]
    base = np.random.default_rng(4).integers(-20000, 20000, int(offs[-1] + ns[-1]) + 8).astype(np.int16)

    pageable = base.copy()
    ctx.vowel_noise_batch(pageable, ns, snr, seeds, offsets=offs, fs=fs)
    ptr = ctx.L.vs_host_alloc(base.nbytes)
    assert ptr
    try:
        view = np.ctypeslib.as_array((C.c_int16 * base.size).from_address(ptr))
        view[:] = base
        ctx.vowel_noise_batch(view, ns, snr, seeds, offsets=offs, fs=fs)
        pinned = view.copy()
    finally:
        ctx.L.vs_host_free(ptr)
    dev = torch.from_numpy(base.copy()).cuda()
    ctx.vowel_noise_batch(dev, ns, snr, seeds, offsets=offs, fs=fs)
    device = dev.cpu().numpy()

    assert np.array_equal(pageable, device) and np.array_equal(pinned, device)
    noised = np.zeros(base.size, dtype=bool)
    for i in range(len(ns)):
        if snr[i] > 0:
            noised[int(offs[i]): int(offs[i] + ns[i])] = True
    assert np.array_equal(device[~noised], base[~noised])
    assert np.array_equal(device[int(offs[5]): int(offs[5] + ns[5])], base[int(offs[5]): int(offs[5] + ns[5])])
    for i in (0, 1, 3, 6):
        row = slice(int(offs[i]), int(offs[i] + ns[i]))
        assert not np.array_equal(device[row], base[row]), i


def test_noise_refusals(ctx, vs):
    L, h = ctx.L, ctx.h
    x = np.random.default_rng(5).integers(-20000, 20000, 4000).astype(np.int16)
    ns, snr, seed = _arr(np.uint64, 4000), _arr(np.float32, 100.0), _arr(np.uint32, 7)

    def call(pcm, nsamp, snr_, fs=None):
        seeds = np.arange(7, 7 + len(nsamp), dtype=np.uint32)
        return L.vs_vowel_noise_batch(h, pcm.ctypes.data, None, nsamp.ctypes.data, snr_.ctypes.data, _p(fs), seeds.ctypes.data,
                                      len(nsamp))

    want = x.copy()
    assert call(want, ns, snr) == vs.VS_OK
    assert not np.array_equal(want, x)

    def still_works():
        y = x.copy()
        assert call(y, ns, snr) == vs.VS_OK
        assert np.array_equal(y, want)

    p = (x.ctypes.data, None, ns.ctypes.data, snr.ctypes.data, None, seed.ctypes.data, 1)
    for null in range(4):                      # ctx, pcm, nsamp, snr
        args = [h, *p]
        args[[0, 1, 3, 4][null]] = None
        assert L.vs_vowel_noise_batch(*args) == vs.VS_EINVAL, null
        still_works()
    cases = [(_arr(np.uint64, BIG), None, vs.VS_EOVERLAP, "stream 0: too many samples"),
             (ns, _arr(np.int32, 0), vs.VS_ERANGE, "stream 0: sampling rate"),
             (ns, _arr(np.int32, 40), vs.VS_ERANGE, "stream 0: frame length 0"),
             (ns, _arr(np.int32, 700000), vs.VS_ERANGE, "stream 0: frame length 35000")]
    for nsamp, fs, code, msg in cases:
        assert call(x, nsamp, snr, fs) == code, msg
        assert L.vs_last_error(h).decode() == msg
        still_works()
    y = x.copy()
    assert call(y, ns, _arr(np.float32, 0.0), _arr(np.int32, 40)) == vs.VS_OK    # no noise: the frame length is not used
    assert np.array_equal(y, x)
    still_works()
    # two bad streams: the first one decides
    two = _arr(np.float32, 100.0, 100.0)
    for nsamp, fs, code, msg in [(_arr(np.uint64, BIG, 100), _arr(np.int32, 22050, 0), vs.VS_EOVERLAP, "stream 0: too many samples"),
                                 (_arr(np.uint64, 100, BIG), _arr(np.int32, 0, 22050), vs.VS_ERANGE, "stream 0: sampling rate")]:
        assert call(x, nsamp, two, fs) == code, msg
        assert L.vs_last_error(h).decode() == msg
        still_works()


@pytest.mark.parametrize("report", [False, True])
def test_analysis_refusals(ctx, vs, report):
    """the refusals of vs_flow_analyze_batch and vs_flow_report_batch that test_report_errors_match_analysis leaves out: a
    row above 2^31-1 samples, and the first of two bad streams decides"""
    L, h = ctx.L, ctx.h
    call = L.vs_flow_report_batch if report else L.vs_flow_analyze_batch
    wrapper = ctx.flow_report_batch if report else ctx.flow_analyze_batch
    out = np.zeros(2, dtype=vs.FLOW_REPORT_DTYPE if report else vs.FLOW_STATS_DTYPE)
    t = np.arange(11025)
    flow = np.maximum(0, 12000 * np.sin(2 * np.pi * 120 * t / 22050)).astype(np.int16)
    want = wrapper(flow, [flow.size])
    cases = [(_arr(np.uint64, BIG), None, None, None, vs.VS_EOVERLAP, "stream 0: too many samples"),
             (_arr(np.uint64, BIG, 64), _arr(np.int32, 22050, 0), None, None, vs.VS_EOVERLAP, "stream 0: too many samples"),
             (_arr(np.uint64, 64, BIG), None, _arr(np.int16, 3, 0), _arr(np.int16, 2, 0), vs.VS_ERANGE,
              "stream 0: thresholds lo > hi")]
    for nsamp, fs, lo, hi, code, msg in cases:
        assert call(h, flow.ctypes.data, None, nsamp.ctypes.data, _p(fs), _p(lo), _p(hi), len(nsamp), out.ctypes.data) == code, msg
        assert L.vs_last_error(h).decode() == msg
        assert wrapper(flow, [flow.size]).tobytes() == want.tobytes()
