#!/usr/bin/env python
"""Regenerates tests/golden/reference_outputs.json by running the UNMODIFIED reference
(compiled by oracle/Makefile into oracle/_ref/, 7z replaced by oracle/7z_shim.sh) on every case
of tests/cases.py.  The reference ships no golden vectors of its own (SURVEY.md section 4), so
these are the pin: outputs of the reference itself, produced from a checkout of its sources.
Never edit the JSON by hand.

    SCCG_REFERENCE_SRC=<checkout of the reference> python tests/golden/make_golden.py
"""
from __future__ import annotations

import base64
import hashlib
import json
import sys
import tempfile
import zlib
from pathlib import Path

HERE = Path(__file__).resolve().parent
sys.path[:0] = [str(HERE.parent), str(HERE.parent.parent)]

import oracle_lib as ol  # noqa: E402
from cases import cases, fasta_cases  # noqa: E402


def sha(b: bytes) -> str:
    return hashlib.sha256(b).hexdigest()


def pack(b: bytes) -> str:
    return base64.b64encode(zlib.compress(b, 9)).decode()


def run_files(ref_file: bytes, tgt_file: bytes) -> dict:
    with tempfile.TemporaryDirectory() as d:
        d = Path(d)
        (d / "ref.fa").write_bytes(ref_file)
        (d / "tgt.fa").write_bytes(tgt_file)
        rc_c, inter = ol.ref_compress_cli(d / "ref.fa", d / "tgt.fa", d / "out")
        rc_d, recon, err = ol.ref_decompress_cli(d / "out" / "compressed_genome.txt.7z", d / "ref.fa", d / "dec")
    return {
        "rc_compress": rc_c, "rc_decompress": rc_d,
        "intermediate_z": pack(inter), "intermediate_sha256": sha(inter),
        "reconstructed_z": pack(recon), "reconstructed_sha256": sha(recon),
        "roundtrip": recon == tgt_file,
    }


def main() -> None:
    assert ol.build_reference(), "reference not available: set SCCG_REFERENCE_SRC to a checkout of its sources"
    out = {"generator": "tests/golden/make_golden.py", "reference": "Jan-Celin/SCCG-genome-compression (unmodified, g++ -O3 -std=c++17)",
           "cases": {}, "fasta_cases": {}}
    for c in cases():
        with tempfile.TemporaryDirectory() as d:
            d = Path(d)
            ol.write_fasta(d / "r.fa", c.ref, b">ref")
            ol.write_fasta(d / "t.fa", c.tgt, c.header if c.header else None)
            g = run_files((d / "r.fa").read_bytes(), (d / "t.fa").read_bytes())
        g["ref_sha256"] = sha(c.ref); g["tgt_sha256"] = sha(c.tgt)
        lines = ol.split_intermediate(zlib.decompress(base64.b64decode(g["intermediate_z"])))
        g["mode"] = 0 if lines[2] == b"," else 1
        out["cases"][c.name] = g
        print(f"{c.name:42s} mode={g['mode']} rc={g['rc_compress']},{g['rc_decompress']} roundtrip={g['roundtrip']}")
    for fc in fasta_cases():
        g = run_files(fc.ref_file, fc.tgt_file)
        g["ref_file_sha256"] = sha(fc.ref_file); g["tgt_file_sha256"] = sha(fc.tgt_file)
        out["fasta_cases"][fc.name] = g
        print(f"fasta:{fc.name:36s} rc={g['rc_compress']},{g['rc_decompress']} roundtrip={g['roundtrip']}")
    (HERE / "reference_outputs.json").write_text(json.dumps(out, indent=1, sort_keys=True) + "\n")
    print("wrote", HERE / "reference_outputs.json")


if __name__ == "__main__":
    main()
