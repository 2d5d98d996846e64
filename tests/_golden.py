"""What the reference computes for the frame-level passes, stored as one sha256 per section of the result blob
(tests/golden/pass_digests.json, written by tools/make_golden_passes.py from the reference build).  The GPU tests compare
the device's blob with these digests, so they need no reference build; the CPU tests named *_matches_golden pin the
digests to the reference wherever it is built."""
import hashlib
import json
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pass_digests.json")


def fp_case(w, h, qp, signhide, rdoq, trskip, bitdepth=8):
    return f"fp{bitdepth}_{w}x{h}_q{qp}_s{signhide}_r{rdoq}_t{trskip}"


def ip_case(w, h, qp, search_range):
    return f"ip8_{w}x{h}_q{qp}_r{search_range}"


def section_digests(blob, sections):
    from kvazaar_b200.api import fp_section
    return {name: hashlib.sha256(np.ascontiguousarray(fp_section(blob, sections, name)).tobytes()).hexdigest() for name in sections}


def assert_matches_reference(blob, sections, case):
    with open(PATH) as f:
        want = json.load(f)[case]
    got = section_digests(blob, sections)
    assert sorted(got) == sorted(want), case
    bad = [name for name in sorted(want) if got[name] != want[name]]
    assert not bad, f"{case}: sections that differ from the reference's: {bad}"
