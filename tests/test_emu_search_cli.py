"""`decompress --search <patterns.fa> --archives <list> [--regions <bed>] [--mismatches K] [--strand both|+|-] <reference_file>
<output_folder>` on the CPU (the program linked against the SIMT-emulator build, as in test_emu_cli.py): hits.bed must hold
the NumPy brute force's hits, archive by archive; every error exits 1 and leaves neither hits.bed nor hits.bed.part."""
import subprocess

import oracle_lib as ol
from test_emu_cli import BIN, env  # noqa: F401  (env: the module fixture that builds the programs)
from test_emu_search import brute


def run(env, *args):  # noqa: F811
    return subprocess.run([str(a) for a in args], env=env, capture_output=True)


def render(stems, names, pats, hits, win_arc):
    return "".join(f"{stems[win_arc[w]]}\t{p}\t{p + len(pats[i])}\t{names[i]}\t{m}\t{'-' if s else '+'}\n" for w, p, i, s, m in hits.tolist()).encode()


def test_search_archives(env, tmp_path):  # noqa: F811
    from sccg_genome_compression_b200 import synth
    ref, tgt = synth.local_pair(60_000, synth.seed_for(2, 66))
    ref, tgt = ref.tobytes(), tgt.tobytes()
    ol.write_fasta(tmp_path / "ref.fa", ref, b">ref")
    targets = [tgt[:1000] + tgt[1000:1200].lower() + b"N" * 77 + tgt[1277:], ref[:500] + ref[4000:], tgt[:30_000]]
    arcs, stems, Ds = [], [], []
    for i, t in enumerate(targets):
        d = tmp_path / f"ind{i}"; d.mkdir()
        ol.write_fasta(d / "tgt.fa", t, b">chrT")
        r = run(env, BIN / "compress", tmp_path / "ref.fa", d / "tgt.fa", d / "out")
        assert r.returncode == 0, r.stderr
        renamed = d / f"ind{i}.txt.7z"
        (d / "out" / "compressed_genome.txt.7z").rename(renamed)
        arcs.append(renamed); stems.append(f"ind{i}.txt")
        rc, image = ol.orc_decompress(ref, (d / "out" / "compressed_genome.txt").read_bytes())
        assert rc == 0
        Ds.append(image.split(b"\n", 1)[1].replace(b"\n", b""))
    names = ["guide1", "nrun", "site", "g2"]
    pats = [Ds[0][5000:5023], b"NNNNNN", b"GAATTC", Ds[2][20_000:20_012].lower()]
    fa = f">{names[0]} first guide\n{pats[0][:10].decode()}\n{pats[0][10:].decode()}\r\n\n>{names[1]}\n{pats[1].decode()}\n" \
         f">{names[2]}\tsite\n{pats[2].decode()}\n>{names[3]}\n{pats[3].decode()}\n"
    (tmp_path / "p.fa").write_text(fa)
    (tmp_path / "list.txt").write_text("\n".join(str(a) for a in arcs) + "\n")
    Lmin = min(len(D) for D in Ds)
    bed = [("r1", 900, 1400), ("r2", 4990, 5030), ("r3", 0, Lmin), ("r1", 900, 1400)]
    (tmp_path / "r.bed").write_text("# regions\n" + "".join(f"{n}\t{a}\t{b}\n" for n, a, b in bed))
    forms = [((), [(a, 0, len(D)) for a, D in enumerate(Ds)], 0, 3),
             (("--regions", tmp_path / "r.bed", "--mismatches", "2", "--strand", "+"), [(a, s, e) for a in range(3) for _, s, e in bed], 2, 1),
             (("--strand", "-", "--mismatches", "1"), [(a, 0, len(D)) for a, D in enumerate(Ds)], 1, 2)]
    for j, (opts, wins, k, strands) in enumerate(forms):
        out = tmp_path / f"out{j}"
        r = run(env, BIN / "decompress", "--search", tmp_path / "p.fa", "--archives", tmp_path / "list.txt", *opts, tmp_path / "ref.fa", out)
        assert r.returncode == 0, r.stderr
        hits = brute(Ds, wins, pats, k, strands)
        assert len(hits) > 0
        assert (out / "hits.bed").read_bytes() == render(stems, names, pats, hits, [a for a, _, _ in wins]), opts
    # errors: exit 1, a message, no hits.bed and no hits.bed.part
    bad_pats = {"empty.fa": "", "noseq.fa": ">a\nACGT\n>b\n", "before.fa": "ACGT\n>a\nACGT\n", "long.fa": ">a\n" + "A" * 65 + "\n",
                "noseq2.fa": ">a\n\n"}
    for name, text in bad_pats.items():
        (tmp_path / name).write_text(text)
    (tmp_path / "bad.bed").write_text("g\t30\t20\n")
    (tmp_path / "far.bed").write_text(f"g\t0\t{Lmin + 1}\n")
    (tmp_path / "empty.txt").write_text("\n")
    (tmp_path / "missing.txt").write_text(str(arcs[0]) + "\n" + str(tmp_path / "nope.7z") + "\n")
    good = ("--archives", tmp_path / "list.txt")
    cases = [(tmp_path / n, good) for n in bad_pats]
    cases += [(tmp_path / "p.fa", good + o) for o in (("--mismatches", "x"), ("--mismatches", "-1"), ("--mismatches", "6"), ("--strand", "up"),
                                                      ("--regions", tmp_path / "bad.bed"), ("--regions", tmp_path / "far.bed"),
                                                      ("--regions", tmp_path / "nope.bed"), ("--bogus", "1"))]
    cases += [(tmp_path / "p.fa", ("--archives", tmp_path / lst)) for lst in ("empty.txt", "missing.txt", "nolist.txt")]
    cases += [(tmp_path / "nope.fa", good), (tmp_path / "p.fa", ())]
    for i, (p, opts) in enumerate(cases):
        out = tmp_path / f"err{i}"
        r = run(env, BIN / "decompress", "--search", p, *opts, tmp_path / "ref.fa", out)
        assert r.returncode == 1 and r.stderr, (p, opts)
        assert not (out / "hits.bed").exists() and not (out / "hits.bed.part").exists(), (p, opts)
