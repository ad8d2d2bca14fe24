#!/usr/bin/env python
"""Writes tests/golden/reference_function_level.json: the reference side of every comparison in
tests/test_oracle_vs_reference.py, as fingerprints (length + sha256) of the outputs and of the inputs.

With the reference's sources readable (oracle/Makefile's REFERENCE, or SCCG_REFERENCE_SRC), the values come from the compiled
reference itself.  Without them, --from-oracle takes them from the C oracle instead; the file records which side made it.

    SCCG_REFERENCE_SRC=<checkout of the reference> python tests/golden/make_function_goldens.py
"""
from __future__ import annotations

import json
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
sys.path[:0] = [str(HERE.parent), str(HERE.parent.parent)]

import oracle_lib as ol  # noqa: E402
import test_oracle_vs_reference as T  # noqa: E402


def main() -> None:
    if ol.build_reference():
        side, source = T.Reference, "the compiled reference (Jan-Celin/SCCG-genome-compression, unmodified, g++ -O3 -std=c++17)"
    elif "--from-oracle" in sys.argv:
        side, source = T.Oracle, ("the C oracle (oracle/sccg_oracle.c), the reference's sources being unavailable; the oracle is unchanged since "
                                  "it was last compared with the compiled reference on these inputs")
    else:
        sys.exit("reference not available: set SCCG_REFERENCE_SRC to a checkout of its sources (or pass --from-oracle)")
    out = {"generator": "tests/golden/make_function_goldens.py", "source": source, "sections": {}}
    for section, (run, keys) in T.SECTIONS.items():
        out["sections"][section] = {str(k): run(side, k) for k in keys}
        print(f"{section}: {len(keys)} cases")
    T.GOLDEN_FILE.write_text(json.dumps(out, indent=1, sort_keys=True) + "\n")
    print("wrote", T.GOLDEN_FILE)


if __name__ == "__main__":
    main()
