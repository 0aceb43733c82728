"""CPU tests of progressive rendering (rh_render_accumulate / Accumulator / progressiveRayTrace): the new entry points
are bound, they fail loudly without a device, and progressiveRayTrace's batch split (with the library stubbed)."""
import ctypes as C

import numpy as np
import pytest

import rayhs_b200 as rh
from rayhs_b200 import capi, host

NEW_SYMBOLS = ("rh_accum_create", "rh_accum_reset", "rh_accum_destroy", "rh_render_accumulate")


def test_new_symbols_are_exported_and_bound():
    L = capi.lib()
    for name in NEW_SYMBOLS:
        assert name in capi.SIGNATURES, name
        fn = getattr(L, name)
        assert fn.argtypes == capi.SIGNATURES[name][1], name
    assert len(capi.SIGNATURES["rh_render_accumulate"][1]) == 8
    assert capi.SIGNATURES["rh_accum_create"][1][5] is C.c_uint32


def test_without_a_device_the_calls_fail_loudly():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    L = capi.lib()
    acc = C.c_void_p()
    assert L.rh_accum_create(64, 48, 0, 1, 0, 8, C.byref(acc)) == capi.RH_ERR_STATE
    assert b"rh_init" in L.rh_last_error()
    assert not acc.value
    o = capi.rh_render_opts()
    o.width, o.height, o.spp = 4, 4, 1
    rgb = np.empty((4, 4, 3), dtype=np.uint8)
    assert L.rh_render_accumulate(None, None, C.byref(o), None, rgb.ctypes.data, None, None, None) == capi.RH_ERR_STATE
    assert b"rh_init" in L.rh_last_error()
    assert L.rh_accum_reset(None) == capi.RH_ERR_ARG
    L.rh_accum_destroy(None)  # a no-op


class _FakeAccumulator:
    """Stands in for the library: records the calls progressiveRayTrace makes."""
    made = []

    def __init__(self, job, stream_spp=0, **kw):
        self.job, self.stream_spp, self.calls, self.closed, self.n = job, stream_spp, [], False, 0
        _FakeAccumulator.made.append(self)

    def add(self, spp, seed=None, **kw):
        assert not self.closed
        self.calls.append((spp, seed, kw))
        self.n += spp
        assert self.n <= self.stream_spp
        return host.Image(4, 3, np.full((3, 4, 3), self.n, dtype=np.uint8), {"n": self.n})

    def close(self):
        self.closed = True


@pytest.mark.parametrize("spp,batch,want", [(64, 8, [8] * 8), (64, 16, [16] * 4), (10, 4, [4, 4, 2]), (5, 8, [5]),
                                            (7, 1, [1] * 7), (1, 1, [1])])
def test_progressive_ray_trace_splits_the_batches(monkeypatch, spp, batch, want):
    monkeypatch.setattr(host, "Accumulator", _FakeAccumulator)
    _FakeAccumulator.made.clear()
    job = object()
    images = list(rh.progressiveRayTrace(job, spp=spp, batch=batch, seed=99))
    (acc,) = _FakeAccumulator.made
    assert acc.job is job and acc.stream_spp == spp
    assert [c[0] for c in acc.calls] == want
    assert all(c[1] == 99 for c in acc.calls)  # every batch continues the same stream
    assert [img.stats["n"] for img in images] == list(np.cumsum(want))
    assert acc.closed


def test_progressive_ray_trace_closes_when_abandoned(monkeypatch):
    monkeypatch.setattr(host, "Accumulator", _FakeAccumulator)
    _FakeAccumulator.made.clear()
    gen = rh.progressiveRayTrace(object(), spp=64, batch=8)
    next(gen)
    gen.close()
    assert _FakeAccumulator.made[0].closed and len(_FakeAccumulator.made[0].calls) == 1


@pytest.mark.parametrize("spp,batch", [(0, 8), (8, 0), (-1, 1)])
def test_progressive_ray_trace_rejects_empty_batches(spp, batch):
    with pytest.raises(ValueError):
        next(rh.progressiveRayTrace(object(), spp=spp, batch=batch))


def test_image_linear_defaults_to_none():
    img = rh.Image(1, 1, np.zeros((1, 1, 3), dtype=np.uint8))
    assert img.linear is None and img.hit_ids is None
