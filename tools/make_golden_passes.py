#!/usr/bin/env python
"""Writes tests/golden/pass_digests.json: the sha256 of every section of the result blob the reference's own frame-level
passes (oracle/ref_framepass.c, oracle/ref_interpass.c in the 8- and 10-bit reference builds) produce for the cases of the
GPU parity tests in tests/test_framepass.py, tests/test_10bit.py and tests/test_interpass.py.  Needs the reference build
under oracle/_ref (__graft_entry__.build() with the reference sources present); the tests that read the file do not."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from kvazaar_b200 import api  # noqa: E402
import test_10bit as T  # noqa: E402
import test_framepass as F  # noqa: E402
import test_interpass as I  # noqa: E402
from _golden import PATH, fp_case, ip_case, section_digests  # noqa: E402
from _oracle import Ref, ref_frame_pass, ref_inter_pass  # noqa: E402

threads = os.cpu_count() or 8
refs = {8: Ref(8), 10: Ref(10)}
out = {}


def frame_pass(src, W, H, qp, signhide, rdoq, trskip, bitdepth=8):
    lay = api.fp_layout_for(W, H, qp, signhide, bitdepth)
    blob = ref_frame_pass(refs[bitdepth], src, W, H, qp, lay, nthreads=threads, signhide=signhide, rdoq=rdoq, trskip=trskip)
    case = fp_case(W, H, qp, signhide, rdoq, trskip, bitdepth)
    out[case] = section_digests(blob, api.fp_sections(lay, W, H, bitdepth))
    print(case, flush=True)


for (W, H), qp, signhide, r in F.PARITY_CASES:
    frame_pass(F.parity_frame(W, H, qp, r >> 1), W, H, qp, signhide, r & 1, r >> 1)
for (W, H), qp, signhide, rdoq, trskip, idx in F.FULL_SIZE_CASES.values():
    frame_pass(F.synth_frame(W, H, frame_idx=idx), W, H, qp, signhide, rdoq, trskip)
for (W, H), qp, signhide, rdoq, trskip in T.PARITY10_CASES:
    frame_pass(T.synth_frame10(W, H, W + qp), W, H, qp, signhide, rdoq, trskip, 10)
(W, H), qp, signhide, rdoq, trskip, idx = T.FULL_SIZE10_CASE
frame_pass(T.synth_frame10(W, H, idx), W, H, qp, signhide, rdoq, trskip, 10)
for (W, H), qp, rng in I.PARITY_CASES:
    cur, rf = I.moving_pair(W, H, seed=W)
    lay = api.ip_layout_for(W, H, qp, rng)
    out[ip_case(W, H, qp, rng)] = section_digests(ref_inter_pass(refs[8], cur, rf, W, H, qp, rng, lay, nthreads=threads), api.ip_sections(lay, W, H))
    print(ip_case(W, H, qp, rng), flush=True)
with open(PATH, "w") as f:
    json.dump(out, f, indent=1, sort_keys=True)
    f.write("\n")
