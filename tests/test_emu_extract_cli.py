"""`decompress --regions <regions.bed> <compressed_file> <reference_file> <output_folder>` on the CPU (the program linked against
the SIMT-emulator build, as in test_emu_cli.py): regions.fa holds one ">name:start-end" record per BED line, 50 columns per
line; malformed BED and regions past the end exit 1 and leave no regions.fa."""
import subprocess

import oracle_lib as ol
from test_emu_cli import BIN, env  # noqa: F401  (env: the module fixture that builds the programs)


def render(D: bytes, bed):
    """the contract: ">name:start-end\\n" and D[start:end] in lines of 50, every line newline-terminated"""
    out = bytearray()
    for name, a, b in bed:
        out += b">%s:%d-%d\n" % (name.encode(), a, b)
        for p in range(a, b, 50):
            out += D[p:min(b, p + 50)] + b"\n"
    return bytes(out)


def make_archive(tmp_path, shape="local"):
    from sccg_genome_compression_b200 import synth
    if shape == "local":
        ref, tgt = synth.local_pair(60_000, synth.seed_for(2, 64))
    else:
        ref, tgt = synth.global_gap_pair(50_000, 45_000, synth.seed_for(1, 64))
    ref, tgt = ref.tobytes(), tgt.tobytes()
    tgt = tgt[:1000] + tgt[1000:1200].lower() + b"N" * 77 + tgt[1277:]
    ol.write_fasta(tmp_path / "ref.fa", ref, b">ref")
    ol.write_fasta(tmp_path / "tgt.fa", tgt, b">chrT")
    return ref, tgt


def run(env, *args):  # noqa: F811
    return subprocess.run([str(a) for a in args], env=env, capture_output=True)


def test_regions_fa(env, tmp_path):  # noqa: F811
    for shape in ("local", "gap"):
        d = tmp_path / shape; d.mkdir()
        make_archive(d, shape)
        r = run(env, BIN / "compress", d / "ref.fa", d / "tgt.fa", d / "out")
        assert r.returncode == 0, r.stderr
        arc = d / "out" / "compressed_genome.txt.7z"
        r = run(env, BIN / "decompress", arc, d / "ref.fa", d / "full")
        assert r.returncode == 0, r.stderr
        image = (d / "full" / "reconstructed_genome.fa").read_bytes()
        rc, exp = ol.orc_decompress(ol.orc_parse_reference_fasta((d / "ref.fa").read_bytes()), (d / "out" / "compressed_genome.txt").read_bytes())
        assert rc == 0 and image == exp                                   # the 3-argument form is unchanged
        D = image.split(b"\n", 1)[1].replace(b"\n", b"")
        Lm = len(D)
        bed = [("chrT", 990, 1300), ("g2", 0, 1), ("empty", 500, 500), ("chrT", 1000, 1101), ("tail", Lm - 120, Lm), ("chrT", 990, 1300)]
        text = "# a comment\ntrack name=test\nbrowser position chrT:1-100\n\n"
        text += "".join(f"{n}\t{a}\t{b}" + ("\tfeature\t0\t+" if i % 2 else "") + "\n" for i, (n, a, b) in enumerate(bed))
        text = text.replace("g2\t0\t1", "g2 0  1")                    # spaces separate columns as well
        (d / "r.bed").write_text(text)
        r = run(env, BIN / "decompress", "--regions", d / "r.bed", arc, d / "ref.fa", d / "reg")
        assert r.returncode == 0, r.stderr
        assert (d / "reg" / "regions.fa").read_bytes() == render(D, bed)
        # errors: exit 1, message, no regions.fa
        for i, bad in enumerate(["chrT\t10\n", "chrT\tx\t20\n", "chrT\t30\t20\n", "chrT\t-1\t5\n", f"chrT\t0\t{Lm + 1}\n"]):
            (d / "bad.bed").write_text("# ok\n" + bad)
            out = d / f"bad{i}"
            r = run(env, BIN / "decompress", "--regions", d / "bad.bed", arc, d / "ref.fa", out)
            assert r.returncode == 1 and r.stderr, bad
            assert not (out / "regions.fa").exists() and not (out / "regions.fa.part").exists()
        assert b"past the end" in r.stderr
