"""The bodies of the motion-search `-m gpu` tests, run on the CPU against the host build of the device code through a
stand-in module (tests/_fake_kb.py): a typo, a wrong view or a swapped argument in a GPU-only test would otherwise surface
only on the B200 box.  Validates the test code and tools/bench_me.py's bookkeeping, not the device."""
import pytest
import torch

import test_me_search as A
import test_zz_me_frac as B
from _fake_kb import FakeKB
from _me_cases import MC_CASES, BIPRED_CASES, CAND_CASES, CASES, FRAC_CASES, GPU_FIRST_RUN_DONE, MERGE_CASES


@pytest.fixture()
def kb(monkeypatch):
    A._hostsim()                                              # builds the host library if it is missing
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    return FakeKB()


def test_search_and_candidate_test_bodies(kb, ref, ref10):
    for name in sorted(CASES):
        A.check_cuda_case(kb, name, ref, ref10)
    A.test_cuda_full_picture_matches_reference(kb, ref, ref10, 416, 240, 8, 16)
    A.test_cuda_full_picture_matches_reference(kb, ref, ref10, 208, 136, 10, 32)
    for name in sorted(CAND_CASES):
        A.test_cuda_candidates_match_golden_and_reference(kb, ref, name)
    A.test_cuda_candidates_feed_the_search(kb, ref)
    assert set(GPU_FIRST_RUN_DONE) <= set(CASES)


def test_fractional_test_bodies(kb, ref, ref10):
    for name in sorted(FRAC_CASES):
        B.test_cuda_matches_golden_and_reference(kb, name, ref, ref10)
    B.test_cuda_integer_then_fractional_full_picture(kb, ref, ref10, 416, 240, 8, 16)
    B.test_cuda_integer_then_fractional_full_picture(kb, ref, ref10, 208, 136, 10, 32)
    for name in sorted(MERGE_CASES):
        B.test_cuda_merge_analysis_matches_golden_and_reference(kb, name, ref, ref10)
    for name in sorted(BIPRED_CASES):
        B.test_cuda_bipred_matches_golden_and_reference(kb, name, ref, ref10)
    for name in sorted(MC_CASES):
        B.test_cuda_motion_compensation_matches_golden_and_reference(kb, name, ref, ref10)


def test_bench_me_bookkeeping(kb, monkeypatch):
    """tools/bench_me.py's measure() with the stand-in: every stage reports `identical` against the reference's outputs for
    the same run, committed as tests/golden/bench_me_416x240.npz (tools/make_golden_me.py)"""
    import os
    import time
    import numpy as np
    import kvazaar_b200
    import bench_me
    import me_cases
    for name in ("init", "to_dev", "me_search_batch", "me_frac_search_batch", "me_candidates_batch", "me_merge_cost_batch"):
        monkeypatch.setattr(kvazaar_b200, name, getattr(kb, name), raising=False)
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "bench_me_416x240.npz"))
    monkeypatch.setattr(me_cases, "RefShim", lambda bitdepth=8: None)
    monkeypatch.setattr(me_cases, "run_reference", lambda *a: g["integer"].view(me_cases.RESULT))
    monkeypatch.setattr(me_cases, "run_frac_reference", lambda *a: g["fractional"].view(me_cases.RESULT))
    monkeypatch.setattr(me_cases, "run_cand_reference", lambda *a: g["candidates"].view(me_cases.CAND_OUT))
    monkeypatch.setattr(me_cases, "run_merge_reference", lambda *a: (g["merge"].view(me_cases.MERGE_COST), tuple(g["merge_bits"])))

    def timed(fn, iters):
        t = time.perf_counter()
        fn()
        return (time.perf_counter() - t) * 1e3
    monkeypatch.setattr(bench_me, "timed", timed)
    line = bench_me.measure("416x240", 16, "hexbs", 8, 1, 4, True)
    assert line["integer"]["identical"] and line["fractional"]["identical"] and line["candidates"]["identical"] and line["merge_analysis"]["identical"]
    assert line["pus"] == (416 // 16) * (240 // 16) and line["fractional"]["positions_per_pu"] > 8
