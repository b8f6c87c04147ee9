"""Generate tests/golden/reference_pins.json: what the reference computes and prints on the cases the tests compare
with it, so that those comparisons also run where the reference is not at hand.  TEST INFRASTRUCTURE ONLY.

    python oracle/gen_reference_pins.py --reference DIR   # DIR = the reference's checkout, oracle/_ref built from it
    python oracle/gen_reference_pins.py --from-project    # lbm_oracle.c and this repo's headers instead

Recorded:
  cases        tests/test_oracle_pins.py LIVE_CASES: SHA-256 of f_current, f_next, rho, ux, uy and the solid mask after
               the run, and forces.csv, of the strict build (oracle/_ref/lbm_ref_strict, one thread)
  instability  the timestep at which that build reports the tau = 0.52, u = 0.1 case of test_oracle_pins unstable
  utils_dump   what tests/cpp/utils_dump.cpp prints built against the reference's include/LBMUtils.h
  params_dump  what tests/cpp/params_dump.cpp prints built against the reference's include/LBMConfig.h

--from-project records the same quantities from lbm_oracle.c and include/ of this repository: the same values as
long as those files are unchanged since the tests last compared them with the reference live (the tests do so, bit
for bit and text for text, wherever the reference is present).  The file's `source` says which side it came from.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import re
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import oracle as O  # noqa: E402
from test_oracle_pins import INSTABILITY_CASE, INSTABILITY_STEPS, LIVE_CASES  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "reference_pins.json")
FIELDS = ("f_current", "f_next", "rho", "ux", "uy", "solid")


def sha256(a) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def dump_text(src: str, inc: str, std: str, flags) -> str:
    with tempfile.TemporaryDirectory() as d:
        exe = os.path.join(d, "dump")
        subprocess.run(["g++", "-std=" + std, "-O1"] + list(flags) + ["-ffp-contract=off", "-I" + inc, src, "-o", exe], check=True)
        return subprocess.run([exe], capture_output=True, text=True, check=True).stdout


def main():
    ap = argparse.ArgumentParser()
    g = ap.add_mutually_exclusive_group(required=True)
    g.add_argument("--reference", metavar="DIR", help="the reference's checkout (oracle/_ref built from it: make -C oracle REF=DIR)")
    g.add_argument("--from-project", action="store_true", help="lbm_oracle.c and include/ of this repository")
    a = ap.parse_args()
    if a.reference:
        if not O.have_ref():
            raise SystemExit("oracle/_ref is not built: make -C oracle REF=%s" % a.reference)
        inc, std = os.path.join(a.reference, "include"), "c++20"
        source = "the reference: oracle/_ref/lbm_ref_strict (one thread) and the headers under its include/"
    else:
        inc, std = os.path.join(ROOT, "include"), "c++17"
        source = ("this repository: oracle/lbm_oracle.c, include/LBMUtils.h and include/LBMConfig.h, unchanged since these "
                  "tests last ran live against the reference's strict build and headers and found them equal bit for bit "
                  "and text for text (the instability timestep is also the one SURVEY.md section 8c records for the "
                  "reference)")
    cases = {}
    for case, steps in LIVE_CASES:
        if a.reference:
            ref = O.run_ref(case, steps, strict=True)
            assert ref["returncode"] == 0, ref["stderr"][-2000:]
            got, csv = {k: ref[k] for k in FIELDS}, ref["forces_csv"]
        else:
            o = O.Oracle(case)
            rows, bad = o.run(steps)
            assert bad == -1
            got, csv = {k: getattr(o, k) for k in FIELDS}, O.format_forces_csv(rows)
        cases[" ".join(case.ref_args(steps))] = {"sha256": {k: sha256(v) for k, v in got.items()}, "forces_csv": csv}
    if a.reference:
        ref = O.run_ref(INSTABILITY_CASE, INSTABILITY_STEPS, strict=True)
        unstable_at = int(re.search(r"Simulation unstable at timestep (\d+)", ref["stderr"]).group(1))
    else:
        unstable_at = O.Oracle(INSTABILITY_CASE).run(INSTABILITY_STEPS)[1]
    out = {
        "source": source,
        "cases": cases,
        "instability": {"case": " ".join(INSTABILITY_CASE.ref_args(INSTABILITY_STEPS)), "unstable_at": unstable_at},
        "utils_dump": dump_text(os.path.join(ROOT, "tests", "cpp", "utils_dump.cpp"), inc, std, ["-mavx2", "-mfma"]),
        "params_dump": dump_text(os.path.join(ROOT, "tests", "cpp", "params_dump.cpp"), inc, std, []),
    }
    with open(OUT, "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
