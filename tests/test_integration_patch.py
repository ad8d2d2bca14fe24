"""INTEGRATION.md section 2, compiled and run: the reference's OWN programs (its main, argv handling, FASTA readers, 7z calls)
with only compress_genome's middle and reconstruct_genome's body replaced by the C-ABI calls (integration/patch_reference.py).
  * CPU: the patched sources are linked against the SIMT-emulator build of the library (needs the reference's sources);
  * GPU (`-m gpu`): the binaries that build() leaves in oracle/_ref/patched, linked against libsccg_b200.so.
Both run the FASTA-level goldens -- files produced by the unmodified reference -- through the patched executables."""
import base64
import os
import subprocess
import zlib
from pathlib import Path

import pytest

import __graft_entry__ as g
import oracle_lib as ol
from cases import fasta_cases

ROOT = Path(__file__).resolve().parent.parent
REF_SRC = g.reference_sources()


def unpack(s):
    return zlib.decompress(base64.b64decode(s))


def run_goldens(bindir: Path, golden, tmp_path, extra_env=None):
    env = ol.shim_env()                                      # PATH with the `7z` copy shim (oracle/_ref/bin)
    env.update(extra_env or {})
    for fc in fasta_cases():
        g = golden["fasta_cases"][fc.name]
        d = tmp_path / fc.name; d.mkdir()
        (d / "ref.fa").write_bytes(fc.ref_file); (d / "tgt.fa").write_bytes(fc.tgt_file)
        r = subprocess.run([str(bindir / "compress"), str(d / "ref.fa"), str(d / "tgt.fa"), str(d / "out")], env=env, capture_output=True)
        assert r.returncode == g["rc_compress"], (fc.name, r.stderr[-300:])
        assert (d / "out" / "compressed_genome.txt").read_bytes() == unpack(g["intermediate_z"]), fc.name
        assert b"Time taken to compress" in r.stdout or g["rc_compress"] != 0       # the reference's own main printed it
        if g["rc_compress"] != 0:
            continue
        r = subprocess.run([str(bindir / "decompress"), str(d / "out" / "compressed_genome.txt.7z"), str(d / "ref.fa"), str(d / "dec")], env=env, capture_output=True)
        assert r.returncode == g["rc_decompress"], (fc.name, r.stderr[-300:])
        if g["rc_decompress"] == 0:
            assert (d / "dec" / "reconstructed_genome.fa").read_bytes() == unpack(g["reconstructed_z"]), fc.name
    # the bounds error of the decoder keeps the reference's message and exit code (decompression.cpp:223-229)
    (tmp_path / "ref.fa").write_bytes(b">r\nACGTACGTACGTACGTACGT\n")
    (tmp_path / "bad.txt.7z").write_bytes(b">h\n\n,\n(5,100)")
    r = subprocess.run([str(bindir / "decompress"), str(tmp_path / "bad.txt.7z"), str(tmp_path / "ref.fa"), str(tmp_path / "d")], env=env, capture_output=True)
    assert r.returncode == 1 and b"exceeds reference genome size" in r.stderr


@pytest.mark.skipif(not (REF_SRC and ol.have_reference()), reason="needs the reference's sources (not part of this repository; SCCG_REFERENCE_SRC) and oracle/_ref")
def test_patched_reference_on_the_emulator(golden, tmp_path):
    from emu_lib import EMU_DIR, emu_context
    emu_context().close()
    bindir = g.build_patched_reference(REF_SRC, lib_dir=EMU_DIR, lib_name="sccg_b200_emu", out_dir=tmp_path / "patched_bin")
    run_goldens(bindir, golden, tmp_path, {"SCCG_EMU_THREADS": "2"})


@pytest.mark.gpu
def test_patched_reference_on_the_gpu(golden, tmp_path):
    bindir = ROOT / "oracle" / "_ref" / "patched"
    if not (bindir / "compress").exists() or not ol.have_reference():
        pytest.skip("oracle/_ref/patched not built (build() creates it where the reference's sources are readable)")
    run_goldens(bindir, golden, tmp_path)
