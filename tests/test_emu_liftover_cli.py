"""`decompress --liftover <bed> --archives <list> [--from reference|archive] <reference_file> <output_folder>` and
`decompress --regions <bed> --archives <list> --reference-coords <reference_file> <output_folder>` on the CPU (the programs
linked against the SIMT-emulator build, as in test_emu_cli.py): lifted.bed must be byte-equal to the lines rendered from the
closed form of tests/liftover_lib.py in both directions, a hits.bed written by --search must feed back directly, and
regions.fa must hold the lifted slices of each D under the labels of `--regions --archives`; errors exit 1 and leave no
output file."""
import subprocess

import numpy as np

import liftover_lib as ll
import oracle_lib as ol
import variants_lib as vl
from test_emu_archive import revcomp
from test_emu_cli import BIN, env  # noqa: F401  (env: the module fixture that builds the programs)


def run(env, *args):  # noqa: F811
    return subprocess.run([str(a) for a in args], env=env, capture_output=True)


def bed_lines(text: str) -> list:
    """(chrom, start, end, column 4, column 6) of each region line ("." for an absent column)"""
    out = []
    for line in text.splitlines():
        f = line.split()
        if not f or f[0].startswith("#") or f[0] in ("track", "browser"):
            continue
        out.append((f[0], int(f[1]), int(f[2]), f[3] if len(f) > 3 else ".", f[5] if len(f) > 5 else "."))
    return out


def render(rows, lines, targets, sources) -> bytes:
    return "".join(f"{t}\t{r[0]}\t{r[1]}\t{ln[3]}\t{r[2]}\t{ln[4]}\t{r[3]}\t{r[4]}\t{r[5]}\t{s}:{ln[1]}-{ln[2]}\n"
                   for r, ln, t, s in zip(rows.tolist(), lines, targets, sources)).encode()


def test_liftover_archives(env, tmp_path):  # noqa: F811
    from sccg_genome_compression_b200 import synth
    ref, tgt = synth.local_pair(60_000, synth.seed_for(2, 68), snp=0.003, indels_per_mbp=300)
    ref, tgt = ref.tobytes(), tgt.tobytes()
    ol.write_fasta(tmp_path / "ref.fa", ref, b">chr7 test reference")
    targets = [tgt, ref[:500] + b"GATTACA" + ref[500:9000] + ref[9003:40_000] + ref[40_050:], b"GG" + ref[:30_000]]
    arcs, stems, Ds, wholes = [], [], [], []
    for i, t in enumerate(targets):
        d = tmp_path / f"ind{i}"; d.mkdir()
        ol.write_fasta(d / "tgt.fa", t, b">chrT")
        r = run(env, BIN / "compress", tmp_path / "ref.fa", d / "tgt.fa", d / "out")
        assert r.returncode == 0, r.stderr
        renamed = d / f"ind{i}.txt.7z"
        (d / "out" / "compressed_genome.txt.7z").rename(renamed)
        arcs.append(renamed); stems.append(f"ind{i}.txt")
        inter = (d / "out" / "compressed_genome.txt").read_bytes()
        Ds.append(vl.decoded(ref, inter))
        wholes.append(vl.variants_whole(ref, inter, Ds[-1]))
    assert Ds[0] == tgt
    L = len(ref)
    dlens = [len(D) for D in Ds]
    (tmp_path / "list.txt").write_text("\n".join(str(a) for a in arcs) + "\n")
    # ---- --from reference: every region into every archive, archive by archive
    text = "# genes\ntrack name=t\n" + "chr7\t490\t9010\tgeneA\t0\t+\nchr7\t0\t0\nchr7\t8990\t9005\tx\t5\t-\n" \
           f"chr7\t39990\t40100\tgap\nchr7\t0\t{L}\tall\t0\t.\nchr7\t{L}\t{L}\tend\n"
    (tmp_path / "genes.bed").write_text(text)
    lines = bed_lines(text)
    q = [(k, s, e, 0) for k in range(len(arcs)) for _, s, e, _, _ in lines]
    rows = ll.lift_queries(wholes, L, dlens, q)
    exp = render(rows, lines * len(arcs), [stems[k] for k, _, _, _ in q], ["chr7"] * len(q))
    for opts in ((), ("--from", "reference")):
        r = run(env, BIN / "decompress", "--liftover", tmp_path / "genes.bed", "--archives", tmp_path / "list.txt", *opts, tmp_path / "ref.fa", tmp_path / "lo")
        assert r.returncode == 0, r.stderr
        assert (tmp_path / "lo" / "lifted.bed").read_bytes() == exp
    assert (rows[:, 5] & ll.LENGTH_CHANGE).any() and (rows[:, 0] != np.array([s for _, s, _, _ in q])).any()
    # ---- --from archive, fed with the hits.bed of --search
    (tmp_path / "p.fa").write_text(f">p1\n{Ds[1][9100:9123].decode()}\n>p2\n{Ds[0][20_000:20_015].decode()}\n>site\nGAATTC\n")
    r = run(env, BIN / "decompress", "--search", tmp_path / "p.fa", "--archives", tmp_path / "list.txt", "--mismatches", "1", tmp_path / "ref.fa", tmp_path / "hits")
    assert r.returncode == 0, r.stderr
    hits_text = (tmp_path / "hits" / "hits.bed").read_text()
    lines = bed_lines(hits_text)
    assert len(lines) > 10 and {ln[0] for ln in lines} == set(stems)
    q = [(stems.index(c), s, e, 1) for c, s, e, _, _ in lines]
    rows = ll.lift_queries(wholes, L, dlens, q)
    r = run(env, BIN / "decompress", "--liftover", tmp_path / "hits" / "hits.bed", "--archives", tmp_path / "list.txt", "--from", "archive",
            tmp_path / "ref.fa", tmp_path / "back")
    assert r.returncode == 0, r.stderr
    assert (tmp_path / "back" / "lifted.bed").read_bytes() == render(rows, lines, ["chr7"] * len(q), [c for c, *_ in lines])
    # ---- --reference-coords: the lifted slices of each D, labelled with the reference coordinates
    reg = [("chr7", 490, 9010, "+"), ("chr7", 8990, 9005, "-"), ("chr7", 100, 100, "+"), ("chr7", 29_950, 30_000, "-"), ("chr7", 0, 60, "-")]
    (tmp_path / "reg.bed").write_text("".join(f"{c}\t{a}\t{b}\tn\t0\t{s}\n" for c, a, b, s in reg))
    r = run(env, BIN / "decompress", "--regions", tmp_path / "reg.bed", "--archives", tmp_path / "list.txt", "--reference-coords",
            tmp_path / "ref.fa", tmp_path / "rc")
    assert r.returncode == 0, r.stderr
    out = bytearray()
    for k, D in enumerate(Ds):
        lifted = ll.lift_queries(wholes, L, dlens, [(k, a, b, 0) for _, a, b, _ in reg])
        for (c, a, b, s), (x, y) in zip(reg, lifted[:, :2].tolist()):
            piece = revcomp(D[x:y]) if s == "-" else D[x:y]
            out += b">%s::%s:%d-%d%s\n" % (stems[k].encode(), c.encode(), a, b, b"(-)" if s == "-" else b"")
            for p in range(0, len(piece), 50):
                out += piece[p:p + 50] + b"\n"
    assert (tmp_path / "rc" / "regions.fa").read_bytes() == bytes(out)
    # ---- errors: exit 1, a message, no lifted.bed and no lifted.bed.part
    (tmp_path / "unknown.bed").write_text(f"{stems[0]}\t0\t10\n# skipped\nind9.txt\t0\t10\n")
    (tmp_path / "past.bed").write_text(f"chr7\t0\t{L + 1}\n")
    (tmp_path / "pastd.bed").write_text(f"{stems[2]}\t0\t{dlens[2] + 1}\n")
    for j, (bed, opts, msg) in enumerate([("unknown.bed", ("--from", "archive"), b"BED line 3 names no listed archive: ind9.txt"),
                                          ("past.bed", (), b"ends past the end of the reference"),
                                          ("pastd.bed", ("--from", "archive"), b"ends past the end of"),
                                          ("genes.bed", ("--from", "both"), b"--from takes reference or archive")]):
        o = tmp_path / f"err{j}"
        r = run(env, BIN / "decompress", "--liftover", tmp_path / bed, "--archives", tmp_path / "list.txt", *opts, tmp_path / "ref.fa", o)
        assert r.returncode == 1 and msg in r.stderr, (bed, r.stderr)
        assert not (o / "lifted.bed").exists() and not (o / "lifted.bed.part").exists()
