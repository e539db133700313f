"""A fresh context reports no device error that no kernel raised.

vs_sync reads the error flag of each of the ring slots a batch call may use.  A slot no call has used yet must read 0
whatever the pinned memory behind it held before: here the process first fills and frees pinned blocks with a nonzero
pattern, so that a new context's allocations are likely to land on such memory, and then every first call of a new
context must succeed."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _dirty_pinned(L, blocks=256, size=4096):
    """pinned blocks filled with the int32 value 12000 (a flow amplitude), then freed"""
    ptrs = []
    for _ in range(blocks):
        p = L.vs_host_alloc(size)
        assert p
        np.ctypeslib.as_array((C.c_int32 * (size // 4)).from_address(p))[:] = 12000
        ptrs.append(p)
    for p in ptrs:
        L.vs_host_free(C.c_void_p(p))


def test_first_calls_of_fresh_contexts_report_no_error():
    from voice_synth_b200 import _lib, api
    L = _lib.load()
    args = [f"-d 0.5 -f {90 + 7 * k} -g {130 + 7 * k} -j 1 -s 3" + (" -n 20" if k % 2 == 0 else "") for k in range(20)]
    p = api.FlowParams.from_cli(args, list(range(31, 51)))
    for round_ in range(3):
        _dirty_pinned(L)
        ctx = api.Context()
        try:
            pcm, offs, ns = ctx.synth_batch(p, api.FilterParams(20, "aiu1234567" * 2))
            ctx.sync()
            assert len(ns) == 20 and (ns > 0).all(), round_
            ctx.pitch_batch(pcm, ns, offsets=offs)          # a call on caller PCM after it: the flags stay clear
            ctx.sync()
        finally:
            ctx.close()
