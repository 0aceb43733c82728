"""CPU tests of adaptive sampling (rh_render_adaptive / AdaptiveAccumulator / adaptiveRayTrace): the new entry points are
bound, rh_adaptive_opts has the header's layout, the calls fail loudly without a device, the numpy restatement of the
selection rule on hand-made states, and adaptiveRayTrace's loop with the library stubbed."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import rayhs_b200 as rh
from rayhs_b200 import capi, host
from tests.adaptive_rule import active_pixels, fold

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW_SYMBOLS = ("rh_adaptive_create", "rh_adaptive_reset", "rh_adaptive_destroy", "rh_render_adaptive", "rh_adaptive_state")


def test_new_symbols_are_exported_and_bound():
    L = capi.lib()
    for name in NEW_SYMBOLS:
        assert name in capi.SIGNATURES, name
        fn = getattr(L, name)
        assert fn.argtypes == capi.SIGNATURES[name][1], name
    assert len(capi.SIGNATURES["rh_render_adaptive"][1]) == 9
    assert capi.SIGNATURES["rh_adaptive_create"][1][5] is C.c_uint32
    assert capi.SIGNATURES["rh_adaptive_destroy"][0] is None


def test_adaptive_opts_layout_matches_the_header():
    fields = ("threshold", "min_spp", "reserved_")
    src = ('#include <stdio.h>\n#include <stddef.h>\n#include "rayhs_b200.h"\nint main(void){printf("%zu", sizeof(rh_adaptive_opts));'
           + "".join(f'printf(" %zu", offsetof(rh_adaptive_opts, {f}));' for f in fields) + "return 0;}")
    exe = os.path.join(ROOT, "build", "adaptive_opts_layout")
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    with open(exe + ".c", "w") as f:
        f.write(src)
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), exe + ".c", "-o", exe])
    size, *offs = (int(v) for v in subprocess.check_output([exe], text=True).split())
    assert size == C.sizeof(capi.rh_adaptive_opts) == 16
    assert offs == [getattr(capi.rh_adaptive_opts, f).offset for f in fields] == [0, 8, 12]


def test_without_a_device_the_calls_fail_loudly():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    L = capi.lib()
    ad = C.c_void_p()
    assert L.rh_adaptive_create(64, 48, 0, 1, 0, 16, C.byref(ad)) == capi.RH_ERR_STATE
    assert b"rh_init" in L.rh_last_error()
    assert not ad.value
    o = capi.rh_render_opts()
    o.width, o.height, o.spp = 4, 4, 1
    ao = capi.rh_adaptive_opts()
    ao.min_spp = 2
    n = C.c_uint64(7)
    assert L.rh_render_adaptive(None, None, C.byref(o), C.byref(ao), None, None, None, C.byref(n), None) == capi.RH_ERR_STATE
    assert b"rh_init" in L.rh_last_error() and n.value == 7
    assert L.rh_adaptive_state(None, None, None, None, 0) == capi.RH_ERR_STATE
    assert L.rh_adaptive_reset(None) == capi.RH_ERR_ARG
    L.rh_adaptive_destroy(None)  # a no-op


def _state(rows):
    """(counts, S, Q) of a row of hand-made pixels: each entry (n, [(S, Q)] * 3)."""
    counts = np.array([r[0] for r in rows], dtype=np.uint32)
    S = np.array([[c[0] for c in r[1]] for r in rows], dtype=np.float64)
    Q = np.array([[c[1] for c in r[1]] for r in rows], dtype=np.float64)
    return counts, S, Q


def test_rule_min_spp_and_stream_end():
    flat = [(0.0, 0.0)] * 3  # zero variance
    counts, S, Q = _state([(0, flat), (7, flat), (8, flat), (60, flat), (62, flat)])
    # fewer than min_spp samples: active whatever the variance, unless the stream has no spp more samples
    assert active_pixels(counts, S, Q, spp=4, stream_spp=64, min_spp=8, threshold=1.0).tolist() == [True, True, False, False, False]
    assert active_pixels(counts, S, Q, spp=4, stream_spp=10, min_spp=8, threshold=1.0).tolist() == [True, False, False, False, False]
    assert active_pixels(counts, S, Q, spp=2, stream_spp=64, min_spp=61, threshold=1.0).tolist() == [True, True, True, True, False]
    # spp larger than the stream: nothing is ever active
    assert not active_pixels(counts, S, Q, spp=65, stream_spp=64, min_spp=8, threshold=0.0).any()


def test_rule_variance_threshold_and_operation_order():
    # samples 0 and 1 (n = 2): S = 1, Q = 1, d = 1 - 1 * (1 / 2) = 0.5; n (n - 1) = 2; active iff 0.5 > tt * 2
    x = np.array([[[0.0, 0.0, 0.0]], [[1.0, 0.0, 0.0]]])
    S, Q = fold(x)
    counts = np.array([2], dtype=np.uint32)
    assert active_pixels(counts, S, Q, 1, 64, 2, threshold=0.49)[0]
    assert not active_pixels(counts, S, Q, 1, 64, 2, threshold=0.5)[0]  # 0.5 > 0.25 * 2 is false
    # threshold 0: any positive d keeps the pixel; d == 0 does not
    assert active_pixels(counts, S, Q, 1, 64, 2, threshold=0.0)[0]
    flat = np.ones((4, 1, 3)) * 0.3
    S2, Q2 = fold(flat)
    d = Q2 - S2 * (S2 / 4.0)
    assert active_pixels(np.array([4], dtype=np.uint32), S2, Q2, 1, 64, 2, 0.0)[0] == bool((d > 0).any())


def test_rule_negative_d_and_nan_count_as_converged():
    n = 16
    # Q a little below S * (S / n): cancellation leaves d < 0
    S = np.array([[1.6, 0.0, 0.0]])
    Q = np.array([[1.6 * (1.6 / n) - 1e-12, 0.0, 0.0]])
    counts = np.array([n], dtype=np.uint32)
    assert (Q - S * (S / n))[0, 0] < 0
    assert not active_pixels(counts, S, Q, 1, 64, 2, threshold=0.0)[0]
    # a NaN channel does not keep a pixel active; another channel above the threshold does
    S = np.array([[np.nan, 0.0, 0.0], [np.nan, 0.0, 1.0]])
    Q = np.array([[np.nan, 0.0, 0.0], [np.nan, 0.0, 1.0]])
    counts = np.array([n, n], dtype=np.uint32)
    assert active_pixels(counts, S, Q, 1, 64, 2, threshold=0.0).tolist() == [False, True]
    # and an infinite threshold stops every pixel at min_spp
    assert not active_pixels(counts, S, Q, 1, 64, 2, threshold=np.inf).any()
    # padding rows are never active
    assert active_pixels(np.array([0, 0], dtype=np.uint32), np.zeros((2, 3)), np.zeros((2, 3)), 1, 64, 2, 0.0,
                         valid=np.array([True, False])).tolist() == [True, False]


def test_fold_rounds_each_square():
    x = np.array([[[0.1, 0.2, 0.3]], [[0.7, 1e-9, 3.0]], [[0.4, 0.5, 0.6]]])
    S, Q = fold(x)
    assert S.tolist() == [[(0.1 + 0.7) + 0.4, (0.2 + 1e-9) + 0.5, (0.3 + 3.0) + 0.6]]
    assert Q[0, 0] == (0.1 * 0.1 + 0.7 * 0.7) + 0.4 * 0.4


class _FakeAdaptive:
    """Stands in for the library: each add() reports the next active count of a script."""
    made = []
    script = []

    def __init__(self, job, stream_spp=0, **kw):
        self.job, self.stream_spp, self.calls, self.closed = job, stream_spp, [], False
        self.left = list(_FakeAdaptive.script)
        _FakeAdaptive.made.append(self)

    def add(self, spp, seed, threshold, min_spp=8, **kw):
        assert not self.closed
        self.calls.append((spp, seed, threshold, min_spp, kw))
        n = self.left.pop(0)
        return host.Image(4, 3, np.zeros((3, 4, 3), dtype=np.uint8), {"n_active": n})

    def close(self):
        self.closed = True


@pytest.mark.parametrize("script", [[12, 12, 5, 1, 0], [12, 0], [3, 3, 3, 3, 0]])
def test_adaptive_ray_trace_runs_until_nothing_is_active(monkeypatch, script):
    monkeypatch.setattr(host, "AdaptiveAccumulator", _FakeAdaptive)
    _FakeAdaptive.made.clear()
    _FakeAdaptive.script = script
    job = object()
    images = list(rh.adaptiveRayTrace(job, max_spp=32, batch=4, min_spp=8, threshold=0.01, seed=99))
    (ad,) = _FakeAdaptive.made
    assert ad.job is job and ad.stream_spp == 32
    assert [img.stats["n_active"] for img in images] == script[:-1]  # the round that traced nothing is not yielded
    assert len(ad.calls) == len(script)
    assert all(c[:4] == (4, 99, 0.01, 8) for c in ad.calls)  # every round continues the same stream with the same rule
    assert ad.closed


def test_adaptive_ray_trace_default_threshold_is_half_an_rgb8_step(monkeypatch):
    monkeypatch.setattr(host, "AdaptiveAccumulator", _FakeAdaptive)
    _FakeAdaptive.made.clear()
    _FakeAdaptive.script = [1, 0]
    list(rh.adaptiveRayTrace(object()))
    (ad,) = _FakeAdaptive.made
    assert ad.stream_spp == 64 and ad.calls[0][:4] == (4, 24, 0.5 / 255, 8)


def test_adaptive_ray_trace_closes_when_abandoned(monkeypatch):
    monkeypatch.setattr(host, "AdaptiveAccumulator", _FakeAdaptive)
    _FakeAdaptive.made.clear()
    _FakeAdaptive.script = [5, 5, 5, 0]
    gen = rh.adaptiveRayTrace(object())
    next(gen)
    gen.close()
    assert _FakeAdaptive.made[0].closed and len(_FakeAdaptive.made[0].calls) == 1


@pytest.mark.parametrize("kw", [dict(max_spp=0), dict(batch=0), dict(max_spp=4, batch=8), dict(min_spp=1)])
def test_adaptive_ray_trace_rejects_bad_arguments(kw):
    with pytest.raises(ValueError):
        next(rh.adaptiveRayTrace(object(), **kw))
