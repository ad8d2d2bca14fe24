"""`decompress --search <patterns.fa> --archives <list> [--regions <bed>] --edits K [--strand both|+|-] <reference_file>
<output_folder>` on the CPU (the program linked against the SIMT-emulator build, as in test_emu_cli.py): hits.bed must hold the
edit-distance hits of tests/edit_probe.cpp, archive by archive; a bad --edits value, and --edits with --mismatches, exit 1 and
leave neither hits.bed nor hits.bed.part."""
import subprocess

import oracle_lib as ol
from test_emu_cli import BIN, env  # noqa: F401  (env: the module fixture that builds the programs)
from test_emu_search_edits import expect, probe  # noqa: F401  (probe: the module fixture that builds the reference)


def run(env, *args):  # noqa: F811
    return subprocess.run([str(a) for a in args], env=env, capture_output=True)


def render(stems, names, hits, win_arc):
    return "".join(f"{stems[win_arc[w]]}\t{s}\t{e}\t{names[i]}\t{d}\t{'-' if st else '+'}\n" for w, s, e, i, st, d in hits.tolist()).encode()


def test_search_edits(env, probe, tmp_path):  # noqa: F811
    from sccg_genome_compression_b200 import synth
    ref, tgt = synth.local_pair(40_000, synth.seed_for(2, 67))
    ref, tgt = ref.tobytes(), tgt.tobytes()
    ol.write_fasta(tmp_path / "ref.fa", ref, b">ref")
    targets = [tgt[:1000] + tgt[1000:1200].lower() + b"N" * 77 + tgt[1277:], tgt[:5010] + tgt[5011:20_000]]
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
    names = ["guide1", "site", "g2"]
    pats = [Ds[0][5000:5023], b"GAATTC", Ds[1][12_000:12_012].lower()]
    (tmp_path / "p.fa").write_text("".join(f">{n} x\n{p.decode()}\n" for n, p in zip(names, pats)))
    (tmp_path / "list.txt").write_text("\n".join(str(a) for a in arcs) + "\n")
    bed = [("r1", 900, 1400), ("r2", 4990, 5030), ("r3", 0, 19_000)]
    (tmp_path / "r.bed").write_text("".join(f"{n}\t{a}\t{b}\n" for n, a, b in bed))
    forms = [(("--edits", "1"), [(a, 0, len(D)) for a, D in enumerate(Ds)], 1, 3),
             (("--regions", tmp_path / "r.bed", "--edits", "2", "--strand", "+"), [(a, s, e) for a in range(2) for _, s, e in bed], 2, 1),
             (("--strand", "-", "--edits", "0"), [(a, 0, len(D)) for a, D in enumerate(Ds)], 0, 2)]
    for j, (opts, wins, k, strands) in enumerate(forms):
        out = tmp_path / f"out{j}"
        r = run(env, BIN / "decompress", "--search", tmp_path / "p.fa", "--archives", tmp_path / "list.txt", *opts, tmp_path / "ref.fa", out)
        assert r.returncode == 0, r.stderr
        hits = expect(probe, Ds, wins, pats, k, strands)
        assert len(hits) > 0
        assert (out / "hits.bed").read_bytes() == render(stems, names, hits, [a for a, _, _ in wins]), opts
    # errors: exit 1, a message, no hits.bed and no hits.bed.part
    good = ("--archives", tmp_path / "list.txt")
    cases = [good + o for o in (("--edits", "x"), ("--edits", "-1"), ("--edits", "6"), ("--edits", ""), ("--edits", "123"),
                                ("--edits", "1", "--mismatches", "1"), ("--mismatches", "0", "--edits", "0"))]
    for i, opts in enumerate(cases):
        out = tmp_path / f"err{i}"
        r = run(env, BIN / "decompress", "--search", tmp_path / "p.fa", *opts, tmp_path / "ref.fa", out)
        assert r.returncode == 1 and r.stderr, opts
        assert not (out / "hits.bed").exists() and not (out / "hits.bed.part").exists(), opts
