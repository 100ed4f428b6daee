#!/usr/bin/env python
"""Generate tests/golden/oracle_golden.json, ref_log_golden.json and ref_rules_golden.json from the COMPILED REFERENCE HEADER
(oracle/_ref/libapus_ref.so = /root/reference/src/include/dare/dare_log.h built
by oracle/Makefile).  Run in the build container, where /root/reference exists:

    python tests/golden/gen_golden.py

The fixture pins the restated oracle on machines that have no reference tree
(the GPU box): tests/test_golden.py replays the same scenarios through
oracle/liboracle_port.so and compares offsets, return values, apply traces and
SHA-256 of every log image; test_oracle_vs_ref.py and test_oracle_engine_rules.py compare the oracle with
ref_log_golden.json and ref_rules_golden.json the same way.
"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

import orc as O                          # noqa: E402
import refgold                           # noqa: E402
import scenarios                         # noqa: E402
import test_oracle_engine_rules as TER   # noqa: E402
import test_oracle_vs_ref as TVR         # noqa: E402

if __name__ == "__main__":
    O.build_oracle()
    assert O.have_ref(), "needs /root/reference to build oracle/_ref"
    ref = O.Oracle("ref")
    out = dict(source="oracle/_ref/libapus_ref.so (reference dare_log.h, unmodified)",
               reference_commit="896959f", scenarios=scenarios.all_scenarios(ref))
    path = os.path.join(HERE, "oracle_golden.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
    print("wrote", path, len(out["scenarios"]), "scenarios")
    src = "oracle/_ref/libapus_ref.so (reference dare_log.h, unmodified, commit 896959f)"
    refgold.write("ref_log_golden.json", src, TVR.record(ref))
    refgold.write("ref_rules_golden.json", src, refgold.digest(TER.record(ref, O.Oracle("orc"))))
    print("wrote ref_log_golden.json, ref_rules_golden.json")
