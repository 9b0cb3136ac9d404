#!/usr/bin/env python
"""Reference fixtures for SURVEY.md 8(f1): runs the reference's OWN host code of ORBmatcher::SearchByProjection (oracle/_ref/libsbpref.so,
built by `make -C oracle/ref_build sbp` from the reference checkout) on seeded synthetic frame pairs and stores what it returns in
tests/golden/sbpref_<case>.npz.  The inputs are regenerated from the seed by tests/sbp_cases.py; the fixture holds only the
reference's outputs (nmatches, cur_match, the level mode it chose) and a checksum of the inputs.
usage: python tools/make_golden_sbp.py        (needs /root/reference at build time; run in this container, commit the .npz)"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import sbp_cases  # noqa: E402
from oracle import ref_sbp  # noqa: E402


def main():
    if not ref_sbp.available():
        raise SystemExit("oracle/_ref/libsbpref.so is missing: make -C oracle/ref_build sbp")
    for name in [*sbp_cases.CASES, *sbp_cases.MORE_CASES]:
        c = sbp_cases.build(name)
        r = ref_sbp.search_by_projection(c["frame_last"], c["frame_cur"], c["pose_last"], c["pose_cur"], **c["camera"], th=c["th"],
                                         scale_factors=sbp_cases.SF, mono=c["mono"], check_orientation=c["check_orientation"])
        path = os.path.join(ROOT, "tests", "golden", f"sbpref_{name}.npz")
        np.savez_compressed(path, nmatches=np.array(r["nmatches"]), cur_match=r["cur_match"], level_mode=np.array(r["level_mode"]),
                            input_checksum=np.array(sbp_cases.checksum(c), np.uint64))
        print(f"{name:28s} nmatches {r['nmatches']:5d}  level_mode {r['level_mode']}  -> {os.path.relpath(path, ROOT)}")


if __name__ == "__main__":
    main()
