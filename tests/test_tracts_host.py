"""Caller-defined vocal tracts, host side (no GPU): the formant and preset helpers of the C ABI, and the reference
filter with an arbitrary denominator that the GPU tests measure the tract calls against (tests/tools/vowel_den.c)."""
import numpy as np
import pytest

from voice_synth_b200 import api

PRESETS = "aiu1234567"


@pytest.fixture(scope="module")
def vowel_den(tmp_path_factory):
    """the reference filter with any denominator (tests/tools/vowel_den.c)"""
    from vowel_den_ref import VowelDen
    return VowelDen(tmp_path_factory.mktemp("vowel_den"))


def _np_formants(freqs, bws, fs):
    """numpy restatement of vs_tract_from_formants: the product of the resonators' quadratics, in the order given."""
    den = np.array([1.0])
    for F, B in zip(np.float32(freqs), np.float32(bws)):
        r = np.exp(-np.pi * float(B) / fs)
        th = 2.0 * np.pi * float(F) / fs
        den = np.convolve(den, [1.0, -2.0 * r * np.cos(th), r * r])
    return np.concatenate([den, np.zeros(23 - den.size)])


@pytest.mark.parametrize("fs", [11025, 22050, 44100])
@pytest.mark.parametrize("nf", [1, 5, 11])
def test_tract_from_formants_is_the_product_of_resonators(fs, nf):
    rng = np.random.default_rng(fs + nf)
    freqs = np.sort(rng.uniform(150.0, 0.45 * fs, nf))
    bws = rng.uniform(30.0, 400.0, nf)
    den = api.tract_from_formants(freqs, bws, fs)
    ref = _np_formants(freqs, bws, fs)
    assert den.shape == (23,) and den[0] == 1.0
    assert np.all(den[2 * nf + 1:] == 0.0)
    scale = np.abs(ref).max()
    assert np.abs(den - ref).max() <= 1e-12 * scale, np.abs(den - ref).max() / scale


def test_tract_from_formants_refusals():
    ok = api.tract_from_formants([500.0], [60.0], 22050)
    assert ok[0] == 1.0
    for freqs, bws, fs, code in [([11025.0], [60.0], 22050, api.VS_ERANGE),      # F >= fs/2
                                 ([12000.0], [60.0], 22050, api.VS_ERANGE),
                                 ([0.0], [60.0], 22050, api.VS_ERANGE),          # F <= 0
                                 ([500.0], [0.0], 22050, api.VS_ERANGE),         # B <= 0
                                 ([500.0], [-5.0], 22050, api.VS_ERANGE),
                                 ([500.0], [60.0], 0, api.VS_ERANGE),            # no sampling rate
                                 ([], [], 22050, api.VS_EINVAL),                 # 0 formants
                                 ([500.0] * 12, [60.0] * 12, 22050, api.VS_EINVAL)]:  # 12 formants: order 24 > 22
        with pytest.raises(api.VsError) as e:
            api.tract_from_formants(freqs, bws, fs)
        assert e.value.code == code, (freqs[:1], bws[:1], fs)


def test_tract_from_preset_is_the_preset_table(oracle):
    for key in PRESETS:
        assert np.array_equal(api.tract_from_preset(key), oracle.preset(key)), key
    with pytest.raises(api.VsError) as e:
        api.tract_from_preset("x")
    assert e.value.code == api.VS_EPRESET


def test_filter_with_preset_tables_is_the_oracle_preset_filter(oracle, vowel_den):
    rng = np.random.default_rng(7)
    flow = rng.integers(-12000, 12000, 3000).astype(np.int16)
    for key, gain, pre in zip(PRESETS, [10.0, 3.5, 10.0, 1.0, 7.0, 10.0, 2.0, 10.0, 0.5, 10.0],
                              [1.0, 0.0, 0.9, 1.0, 1.0, 0.3, 1.0, 1.0, 0.0, 1.0]):
        pcm, raw = oracle.vowel(flow, key, gain, pre, want_raw=True)
        pcm2, raw2 = vowel_den(flow, oracle.preset(key), gain, pre, want_raw=True)
        assert np.array_equal(pcm, pcm2) and np.array_equal(raw, raw2), key


def test_tract_params_select():
    den = np.stack([api.tract_from_preset(k) for k in "ai"])
    t = api.TractParams(4, den, tract=[0, 1, 1, 0], gain=[1, 2, 3, 4], pre=0.5)
    q = t.select([3, 1])
    assert q.n == 2 and np.array_equal(q.den, den)
    assert list(q.tract) == [0, 1] and list(q.gain) == [4.0, 2.0] and list(q.pre) == [0.5, 0.5]
    with pytest.raises(ValueError):
        api.TractParams(1, np.zeros((2, 22)))
