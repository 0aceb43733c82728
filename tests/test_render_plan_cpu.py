"""The chunk planner of the wavefront (rayhs_b200/csrc/render_plan.h), compiled alone through
tests/render_plan_driver.cpp: exact plans and processing orders for every branch, and the invariants every plan keeps.
Needs no GPU and no librayhs_b200.so."""
import ctypes as C
import os

import numpy as np
import pytest

from tests.util import temp_library

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SOURCES = [os.path.join(ROOT, "tests", "render_plan_driver.cpp"), os.path.join(ROOT, "rayhs_b200", "csrc", "render_plan.h")]
FLAGS = ["-std=c++17", "-O2", "-Wall", "-Werror", "-fPIC", "-shared"]

MI = 1 << 20
B200_MEM = 180 << 30   # device memory of a B200
SMALL_MEM = 16 << 30   # a device on which the bench frame needs several chunks
BENCH_ROWS, BENCH_ROW = 2160, 3840 * 16  # bench.py's frame: 3840 x 2160 at 16 spp
TRACE_ROW = 4096                          # rh_trace_rays: rays per row


def row_costs(rows):
    """Kernel ms per row as a streamed frame measures them: an expensive band (an object) over a ripple."""
    r = np.arange(rows)
    return (1.0 + 3.0 * (np.abs(r - 0.55 * rows) < 0.15 * rows) + 0.01 * ((r * 37) % 17)).astype(np.float32)


# name: (local rows, samples per row, chunk_samples, device memory, pass-0 items stream from the host,
#        row costs of the last streamed frame or None, that frame was compute-bound)
CASES = {
    "device_offsets_bench": (BENCH_ROWS, BENCH_ROW, 0, B200_MEM, False, None, False),
    "device_offsets_small_memory": (BENCH_ROWS, BENCH_ROW, 0, SMALL_MEM, False, None, False),
    "explicit_chunk_device": (BENCH_ROWS, BENCH_ROW, 5_000_000, B200_MEM, False, None, False),
    "explicit_chunk_streamed": (BENCH_ROWS, BENCH_ROW, 16 * MI, B200_MEM, True, row_costs(BENCH_ROWS), True),
    "first_streamed_bench": (BENCH_ROWS, BENCH_ROW, 0, B200_MEM, True, None, False),
    "first_streamed_short_tail": (654, BENCH_ROW, 0, B200_MEM, True, None, False),
    "first_streamed_tail_cap": (114, 600_000, 0, B200_MEM, True, None, False),
    "known_cost_upload_bound": (BENCH_ROWS, BENCH_ROW, 0, B200_MEM, True, row_costs(BENCH_ROWS), False),
    "known_cost_compute_bound": (BENCH_ROWS, BENCH_ROW, 0, B200_MEM, True, row_costs(BENCH_ROWS), True),
    "known_cost_compute_bound_merge": (1961, BENCH_ROW, 0, B200_MEM, True, row_costs(1961), True),
    "known_cost_compute_bound_narrow": (100, 1536 * 1024, 0, B200_MEM, True, row_costs(100), True),
    "known_cost_compute_bound_small_frame": (500, BENCH_ROW, 0, B200_MEM, True, row_costs(500), True),
    "row_wider_than_budget_streamed": (8, 20 * MI, 0, B200_MEM, True, None, False),
    "row_wider_than_chunk": (5, 4096, 1000, B200_MEM, False, None, False),
    "trace_16mi_host": (4096, TRACE_ROW, 0, B200_MEM, True, None, False),
    "trace_16mi_device": (4096, TRACE_ROW, 0, B200_MEM, False, None, False),
    "trace_16mi_chunk_rays": (4096, TRACE_ROW, MI, B200_MEM, True, None, False),
    "trace_64mi_host": (16384, TRACE_ROW, 0, B200_MEM, True, None, False),
    "trace_small_host": (25, TRACE_ROW, 0, B200_MEM, True, None, False),
}

# name: (rows per chunk, processing order, n_tail, ramped), from the chunk plan and processing order of the library
# before the planner was split out of the render loop
EXPECTED = {
    "device_offsets_bench": ([2160], [0], 0, False),
    "device_offsets_small_memory": ([114, 114, 114, 114, 114, 114, 114, 114, 114, 114, 114, 114, 114, 114, 114, 114, 114, 114, 108], [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18], 0, False),
    "explicit_chunk_device": ([81, 81, 81, 81, 81, 81, 81, 81, 81, 81, 81, 81, 81, 81, 81, 81, 81, 81, 81, 81, 81, 81, 81, 81, 81, 81, 54], [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 24, 25, 26], 0, False),
    "explicit_chunk_streamed": ([273, 273, 273, 273, 273, 273, 273, 249], [0, 1, 2, 3, 4, 5, 6, 7], 0, False),
    "first_streamed_bench": ([68, 273, 273, 273, 273, 273, 273, 273, 91, 45, 23, 22], [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11], 4, False),
    "first_streamed_short_tail": ([68, 273, 273, 20, 20], [0, 1, 2, 3, 4], 2, False),
    "first_streamed_tail_cap": ([6, 27, 27, 27, 14, 7, 3, 2, 1], [0, 1, 2, 3, 4, 5, 6, 7, 8], 5, False),
    "known_cost_upload_bound": ([68, 273, 273, 273, 273, 273, 273, 273, 91, 45, 23, 22], [0, 5, 4, 6, 3, 2, 7, 1, 8, 9, 10, 11], 4, False),
    "known_cost_compute_bound": ([273, 273, 273, 273, 34, 34, 68, 137, 273, 273, 249], [4, 5, 6, 7, 3, 8, 10, 2, 1, 9, 0], 0, True),
    "known_cost_compute_bound_merge": ([273, 273, 273, 273, 34, 34, 68, 137, 273, 323], [4, 5, 6, 7, 3, 2, 8, 9, 1, 0], 0, True),
    "known_cost_compute_bound_narrow": ([10, 10, 10, 10, 10, 10, 10, 10, 10, 10], [6, 5, 4, 7, 2, 3, 9, 1, 8, 0], 0, True),
    "known_cost_compute_bound_small_frame": ([68, 273, 159], [0, 1, 2], 0, False),
    "row_wider_than_budget_streamed": ([1, 1, 1, 1, 1, 1, 1, 1], [0, 1, 2, 3, 4, 5, 6, 7], 1, False),
    "row_wider_than_chunk": ([1, 1, 1, 1, 1], [0, 1, 2, 3, 4], 0, False),
    "trace_16mi_host": ([1024, 3072], [0, 1], 0, False),
    "trace_16mi_device": ([4096], [0], 0, False),
    "trace_16mi_chunk_rays": ([256, 256, 256, 256, 256, 256, 256, 256, 256, 256, 256, 256, 256, 256, 256, 256], [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15], 0, False),
    "trace_64mi_host": ([1024, 4096, 4096, 4096, 1536, 768, 384, 384], [0, 1, 2, 3, 4, 5, 6, 7], 4, False),
    "trace_small_host": ([25], [0], 0, False),
}

_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = temp_library("render_plan", SOURCES, FLAGS)
        ip = C.POINTER(C.c_int)
        _lib.rp_plan.restype = C.c_int
        _lib.rp_plan.argtypes = [C.c_int, C.c_ulonglong, C.c_int, C.c_ulonglong, C.c_int, C.POINTER(C.c_float), C.c_int,
                                 C.c_int, ip, ip, ip, ip]
    return _lib


def plan(rows_local, row_samples, chunk_samples, mem, host_offsets, costs, compute_bound):
    """(rows per chunk, first row per chunk, processing order, n_tail, ramped)"""
    cap = 4096
    rows, first, order = (np.zeros(cap, np.int32) for _ in range(3))
    info = np.zeros(2, np.int32)
    if costs is not None:
        costs = np.ascontiguousarray(costs, np.float32)
        assert len(costs) == rows_local
    cost_p = None if costs is None else costs.ctypes.data_as(C.POINTER(C.c_float))
    n = lib().rp_plan(rows_local, row_samples, chunk_samples, mem, int(host_offsets), cost_p, int(compute_bound), cap,
                      *(a.ctypes.data_as(C.POINTER(C.c_int)) for a in (rows, first, order, info)))
    assert 0 < n <= cap
    return rows[:n].tolist(), first[:n].tolist(), order[:n].tolist(), int(info[0]), bool(info[1])


@pytest.mark.parametrize("name", sorted(CASES))
def test_plan_matches(name):
    rows, _, order, n_tail, ramped = plan(*CASES[name])
    assert (rows, order, n_tail, ramped) == EXPECTED[name]


@pytest.mark.parametrize("name", sorted(CASES))
def test_plan_invariants(name):
    rows_local, row_samples = CASES[name][:2]
    rows, first, order, n_tail, _ = plan(*CASES[name])
    assert min(rows) >= 1 and sum(rows) == rows_local
    assert first == np.concatenate([[0], np.cumsum(rows)[:-1]]).tolist()
    assert sorted(order) == list(range(len(rows)))
    assert max(rows) * row_samples <= 0x7FFFFFFF  # the render's "chunk too large" guard
    if n_tail:  # tail pieces stay last, in row order
        assert order[-n_tail:] == list(range(len(rows) - n_tail, len(rows)))


def test_cases_cover_every_branch():
    """Each branch of the planner is taken by some case."""
    got = {name: plan(*c) for name, c in CASES.items()}
    assert len(got["device_offsets_bench"][0]) == 1
    assert len(got["device_offsets_small_memory"][0]) > 2                       # two lanes: half the budget each
    assert got["first_streamed_bench"][0][0] * BENCH_ROW <= 4 * MI              # small first chunk
    assert got["first_streamed_tail_cap"][3] == 5                               # four halvings, then the rest
    assert 0 < got["first_streamed_short_tail"][3] < 5                          # halving stopped at ~1 Mi samples
    assert got["known_cost_compute_bound"][4] and got["known_cost_compute_bound_merge"][4]
    assert not got["known_cost_compute_bound_small_frame"][4]                   # too small to ramp
    assert not got["known_cost_upload_bound"][4] and got["known_cost_upload_bound"][3] > 0
    assert got["explicit_chunk_streamed"][2] == list(range(len(got["explicit_chunk_streamed"][0])))  # costs unused
