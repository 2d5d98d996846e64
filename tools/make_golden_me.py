#!/usr/bin/env python
"""Writes tests/golden/me_search.npz: what the UNMODIFIED reference's integer motion search (oracle/ref_me.c: the reference's
own search_inter.c compiled in place) returns for the cases of tools/me_cases.py.  Run in the container that has
/root/reference (make -C oracle ref); the tests that read the file need neither the reference nor its build."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from _me_cases import (MC_CASES, make_mc_case, run_mc_reference, BIPRED_CASES, CAND_CASES, CASES, FRAC_CASES, MERGE_CASES, make_bipred_case, run_bipred_reference, make_cand_case, make_case, make_frac_case, make_merge_case,  # noqa: E402
                       run_cand_reference, run_frac_reference, run_merge_reference, run_reference)
from _oracle import Ref  # noqa: E402

refs = {}
out = {}
for name in sorted(CASES):
    p, cur, ref, pus = make_case(name)
    shim = refs.setdefault(p.bitdepth, Ref(p.bitdepth))
    r = run_reference(shim, p, cur, ref, pus)
    out[name + "/mv"] = r["mv"].copy()
    out[name + "/bits"] = r["bits"].copy()
    out[name + "/cost"] = r["cost"].copy()
    print(name, len(pus), "PUs")
for name in sorted(CAND_CASES):
    f, crp, clx, cus, col, pus = make_cand_case(name)
    r = run_cand_reference(refs.setdefault(8, Ref(8)), f, crp, clx, cus, col, pus)
    out["cand/" + name] = np.frombuffer(r.tobytes(), np.uint8).copy()
    print("cand", name, len(pus), "PUs")
for name in sorted(FRAC_CASES):
    p, level, cur, ref, pus = make_frac_case(name)
    r = run_frac_reference(refs.setdefault(p.bitdepth, Ref(p.bitdepth)), p, level, cur, ref, pus)
    out["frac/" + name + "/mv"] = r["mv"].copy()
    out["frac/" + name + "/bits"] = r["bits"].copy()
    out["frac/" + name + "/cost"] = r["cost"].copy()
    print("frac", name, len(pus), "PUs")
for name in sorted(MERGE_CASES):
    p, c, cur, planes, pus, cu = make_merge_case(name)
    r, bits = run_merge_reference(refs.setdefault(p.bitdepth, Ref(p.bitdepth)), p, c, cur, planes, pus, cu)
    out["merge/" + name] = np.frombuffer(r.tobytes(), np.uint8).copy()
    out["merge/" + name + "/bits"] = np.array(bits, np.float64)
    print("merge", name, len(pus), "PUs")
for name in sorted(BIPRED_CASES):
    p, c, cur, planes, pus = make_bipred_case(name)
    r = run_bipred_reference(refs.setdefault(p.bitdepth, Ref(p.bitdepth)), p, c, cur, planes, pus)
    out["bipred/" + name] = np.frombuffer(r.tobytes(), np.uint8).copy()
    print("bipred", name, len(pus), "PUs")
import hashlib
for name in sorted(MC_CASES):
    p, c, planes, us, vs, pus, cu = make_mc_case(name)
    oy, ou, ov = run_mc_reference(refs.setdefault(p.bitdepth, Ref(p.bitdepth)), p, c, planes, us, vs, pus, cu)
    out["mc/" + name] = np.frombuffer(b"".join(hashlib.sha256(a.tobytes()).digest() for a in (oy, ou, ov)), np.uint8).copy()      # sha256 of Y, U, V
    print("mc", name, len(pus), "PUs")
np.savez_compressed(os.path.join(ROOT, "tests", "golden", "me_search.npz"), **out)

# tests/golden/bench_me_416x240.npz: what the reference returns in tools/bench_me.py's measure("416x240", 16, "hexbs", 8, 1, 4),
# the run tests/test_gpu_test_bodies_on_cpu.py checks with the host build of the device code standing in for the device
import bench_me  # noqa: E402
import kvazaar_b200  # noqa: E402
import me_cases  # noqa: E402
from _fake_kb import FakeKB  # noqa: E402

fake = FakeKB()
for n in ("init", "to_dev", "me_search_batch", "me_frac_search_batch", "me_candidates_batch", "me_merge_cost_batch"):
    setattr(kvazaar_b200, n, getattr(fake, n))
bench_me.timed = lambda fn, iters: (fn(), 1.0)[1]
recorded = {}
for key, name in (("integer", "run_reference"), ("fractional", "run_frac_reference"), ("candidates", "run_cand_reference"), ("merge", "run_merge_reference")):
    def recording(*a, _key=key, _fn=getattr(me_cases, name)):
        recorded[_key] = _fn(*a)
        return recorded[_key]
    setattr(me_cases, name, recording)
line = bench_me.measure("416x240", 16, "hexbs", 8, 1, 4, True)
assert all(line[k]["identical"] for k in ("integer", "fractional", "candidates", "merge_analysis")), line
merge, merge_bits = recorded.pop("merge")
bench = {k: np.frombuffer(v.tobytes(), np.uint8).copy() for k, v in recorded.items()}
bench["merge"] = np.frombuffer(merge.tobytes(), np.uint8).copy()
bench["merge_bits"] = np.array(merge_bits, np.float64)
np.savez_compressed(os.path.join(ROOT, "tests", "golden", "bench_me_416x240.npz"), **bench)
print("bench_me 416x240:", {k: v.size for k, v in bench.items()})
