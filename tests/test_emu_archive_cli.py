"""`decompress --regions <regions.bed> --archives <list> <reference_file> <output_folder>` on the CPU (the program linked against
the SIMT-emulator build, as in test_emu_cli.py): every BED region from every archive of the list, records
">archive_stem::name:start-end" (+ "(-)" on the minus strand, from BED column 6) in lines of 50; a malformed list or BED file,
an out-of-range region or a bad archive exits 1 and leaves no regions.fa."""
import subprocess

import oracle_lib as ol
from test_emu_archive import revcomp
from test_emu_cli import BIN, env  # noqa: F401  (env: the module fixture that builds the programs)


def render(stems, Ds, bed):
    out = bytearray()
    for stem, D in zip(stems, Ds):
        for name, a, b, strand in bed:
            piece = revcomp(D[a:b]) if strand == "-" else D[a:b]
            out += b">%s::%s:%d-%d%s\n" % (stem.encode(), name.encode(), a, b, b"(-)" if strand == "-" else b"")
            for p in range(0, len(piece), 50):
                out += piece[p:p + 50] + b"\n"
    return bytes(out)


def run(env, *args):  # noqa: F811
    return subprocess.run([str(a) for a in args], env=env, capture_output=True)


def test_regions_from_archives(env, tmp_path):  # noqa: F811
    from sccg_genome_compression_b200 import synth
    ref, tgt = synth.local_pair(60_000, synth.seed_for(2, 65))
    ref, tgt = ref.tobytes(), tgt.tobytes()
    ol.write_fasta(tmp_path / "ref.fa", ref, b">ref")
    targets = [tgt[:1000] + tgt[1000:1200].lower() + b"N" * 77 + tgt[1277:], ref[:500] + ref[4000:], tgt[:30_000]]
    arcs, stems, Ds = [], [], []
    for i, t in enumerate(targets):
        d = tmp_path / f"ind{i}"; d.mkdir()
        ol.write_fasta(d / "tgt.fa", t, b">chrT")
        r = run(env, BIN / "compress", tmp_path / "ref.fa", d / "tgt.fa", d / "out")
        assert r.returncode == 0, r.stderr
        arc = d / "out" / "compressed_genome.txt.7z"
        renamed = d / f"ind{i}.txt.7z"
        arc.rename(renamed)
        arcs.append(renamed); stems.append(f"ind{i}.txt")
        rc, image = ol.orc_decompress(ref, (d / "out" / "compressed_genome.txt").read_bytes())
        assert rc == 0
        Ds.append(image.split(b"\n", 1)[1].replace(b"\n", b""))
    Lmin = min(len(D) for D in Ds)
    bed = [("g1", 990, 1300, "+"), ("g2", 0, 1, "-"), ("empty", 500, 500, "-"), ("g3", 1000, 1101, None), ("tail", Lmin - 120, Lmin, "-"),
           ("g1", 990, 1300, ".")]
    text = "# a comment\ntrack name=test\n\n"
    text += "".join(f"{n}\t{a}\t{b}" + (f"\tfeature\t0\t{s}" if s else "") + "\n" for n, a, b, s in bed)
    (tmp_path / "r.bed").write_text(text)
    (tmp_path / "list.txt").write_text("\n".join(str(a) for a in arcs) + "\n\n")
    r = run(env, BIN / "decompress", "--regions", tmp_path / "r.bed", "--archives", tmp_path / "list.txt", tmp_path / "ref.fa", tmp_path / "reg")
    assert r.returncode == 0, r.stderr
    assert (tmp_path / "reg" / "regions.fa").read_bytes() == render(stems, Ds, bed)
    # errors: exit 1, a message, no regions.fa
    (tmp_path / "good.bed").write_text("g\t0\t10\t.\t0\t-\n")
    (tmp_path / "missing.txt").write_text(str(arcs[0]) + "\n" + str(tmp_path / "nope.7z") + "\n")
    (tmp_path / "empty.txt").write_text("\n  \n")
    (tmp_path / "bad_arc").mkdir()
    (tmp_path / "bad.txt").write_bytes(b">h\n\n,\n(400,2000000)")                # a record that reaches past the reference
    subprocess.run(["7z", "a", "-mx=9", tmp_path / "bad_arc" / "bad.txt.7z", tmp_path / "bad.txt"], env=env, check=True, capture_output=True)
    (tmp_path / "badarc.txt").write_text(str(tmp_path / "bad_arc" / "bad.txt.7z") + "\n")
    cases = [("good.bed", "empty.txt"), ("good.bed", "missing.txt"), ("good.bed", "nolist.txt"), ("good.bed", "badarc.txt")]
    for i, bad in enumerate(["g\t10\n", "g\tx\t20\n", "g\t30\t20\n", "g\t0\t5\t.\t0\t*\n", f"g\t0\t{Lmin + 1}\n"]):
        (tmp_path / f"bad{i}.bed").write_text("# ok\n" + bad)
        cases.append((f"bad{i}.bed", "list.txt"))
    for i, (b, lst) in enumerate(cases):
        out = tmp_path / f"err{i}"
        r = run(env, BIN / "decompress", "--regions", tmp_path / b, "--archives", tmp_path / lst, tmp_path / "ref.fa", out)
        assert r.returncode == 1 and r.stderr, (b, lst)
        assert not (out / "regions.fa").exists() and not (out / "regions.fa.part").exists(), (b, lst)
    assert b"past the end" in r.stderr
