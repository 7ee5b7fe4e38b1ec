#!/usr/bin/env python3
"""Generate tests/golden/ref_pins.json from THE REFERENCE'S OWN SOURCES (oracle/_ref, built by `make -C oracle ref refprog`
where the reference tree is present).  Runs every scenario of tests/test_ref_pin.py and tests/test_ref_prog_pin.py through the
reference and records what those tests compare; the tests then require the restatement to reproduce it.

--leaves writes tests/golden/ref_pins_leaves.json instead: the scenarios of tests/test_leaves_ref_pin.py (getVoxelCenters,
getOccupiedVoxelIndices, isEmpty)."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import leaves_py, oracle_py  # noqa: E402
from tests import test_leaves_ref_pin, test_ref_pin, test_ref_prog_pin  # noqa: E402


def main():
    leaves = "--leaves" in sys.argv[1:]
    for lib in (leaves_py.REF_LEAVES_LIB,) if leaves else (oracle_py.REF_LIB, oracle_py.REFPROG_LIB):
        if not os.path.exists(lib):
            raise SystemExit(f"{lib} is not built: run `make -C oracle ref refprog REF=<reference tree>` and "
                             "`make -f oracle/leaves.mk REF=<reference tree>`")
    if leaves:
        out, path = test_leaves_ref_pin.observe_all("reference"), test_leaves_ref_pin.GOLDEN
        out["source"] = "oracle/_ref: the reference's src/lib/*.cpp compiled verbatim (sdmiller/cpu_tsdf @ 9b973cb)"
    else:
        out, path = {**test_ref_pin.observe_all("reference"), **test_ref_prog_pin.observe_all("reference")}, test_ref_pin.GOLDEN
        out["source"] = "oracle/_ref: the reference's src/lib/*.cpp and src/prog/integrate.cpp compiled verbatim (sdmiller/cpu_tsdf @ 9b973cb)"
    with open(path, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote", path, f"({len(out) - 1} cases)")


if __name__ == "__main__":
    main()
