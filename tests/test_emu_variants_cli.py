"""`decompress --variants --archives <list> [--regions <bed>] <reference_file> <output_folder>` on the CPU (the program linked
against the SIMT-emulator build, as in test_emu_cli.py): variants.vcf must be byte-equal to the VCF rendered from the
reference implementation of tests/variants_lib.py; every error exits 1 and leaves neither variants.vcf nor variants.vcf.part."""
import subprocess

import oracle_lib as ol
import variants_lib as vl
from test_emu_cli import BIN, env  # noqa: F401  (env: the module fixture that builds the programs)


def run(env, *args):  # noqa: F811
    return subprocess.run([str(a) for a in args], env=env, capture_output=True)


def render_vcf(chrom: str, R: bytes, stems, Ds, wholes, regions) -> bytes:
    """the VCF of the decompress header comment, from whole-archive records of the reference implementation"""
    UR = vl.up(R)
    rows = {}
    for k, W in enumerate(wholes):
        keep = set()
        for s, e in regions:
            e = e + 1 if e == len(R) else e
            keep |= {tuple(r) for r in W[(W[:, 0] >= s) & (W[:, 0] < e)].tolist()}
        for pos, end, ds, de in keep:
            ref, alt, p = UR[pos:end], vl.up(Ds[k][ds:de]), pos + 1
            if not ref or not alt:
                if pos > 0:
                    b = UR[pos - 1:pos]; ref, alt, p = b + ref, b + alt, pos
                else:
                    b = UR[end:end + 1] or b"N"; ref, alt = ref + b, alt + b
            rows.setdefault((p, ref, alt), set()).add(k)
    out = [b"##fileformat=VCFv4.2", b"##contig=<ID=%s,length=%d>" % (chrom.encode(), len(R)),
           b'##FORMAT=<ID=GT,Number=1,Type=String,Description="Genotype">',
           b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + "\t".join(stems).encode()]
    for (p, ref, alt), carriers in sorted(rows.items()):
        out.append(b"%s\t%d\t.\t%s\t%s\t.\t.\t.\tGT\t" % (chrom.encode(), p, ref, alt) +
                   b"\t".join(b"1" if k in carriers else b"0" for k in range(len(wholes))))
    return b"\n".join(out) + b"\n"


def test_variants_archives(env, tmp_path):  # noqa: F811
    from sccg_genome_compression_b200 import synth
    ref, tgt = synth.local_pair(60_000, synth.seed_for(2, 67), snp=0.003, indels_per_mbp=300)
    ref, tgt = ref.tobytes(), tgt.tobytes()
    ol.write_fasta(tmp_path / "ref.fa", ref, b">chr7 test reference")
    ol.write_fasta(tmp_path / "nohead.fa", ref, None)
    targets = [tgt, ref[:500] + b"GATTACA" + ref[500:9000] + ref[9003:], tgt[:30_000] + ref[30_000:], b"GG" + ref]
    arcs, stems, Ds = [], [], []
    for i, t in enumerate(targets):
        d = tmp_path / f"ind{i}"; d.mkdir()
        ol.write_fasta(d / "tgt.fa", t, b">chrT")
        r = run(env, BIN / "compress", tmp_path / "ref.fa", d / "tgt.fa", d / "out")
        assert r.returncode == 0, r.stderr
        renamed = d / f"ind{i}.txt.7z"
        (d / "out" / "compressed_genome.txt.7z").rename(renamed)
        arcs.append(renamed); stems.append(f"ind{i}.txt")
        Ds.append(vl.decoded(ref, (d / "out" / "compressed_genome.txt").read_bytes()))
    wholes = [vl.variants_whole(ref, (tmp_path / f"ind{i}" / "out" / "compressed_genome.txt").read_bytes(), D) for i, D in enumerate(Ds)]
    (tmp_path / "list.txt").write_text("\n".join(str(a) for a in arcs) + "\n")
    bed = [("chr7", 0, 700), ("chr7", 400, 9500), ("chr7", 20_000, 40_000), ("chr7", 20_000, 40_000), ("chr7", 59_000, len(ref))]
    (tmp_path / "r.bed").write_text("# regions\n" + "".join(f"{n}\t{a}\t{b}\n" for n, a, b in bed))
    forms = [((), "ref.fa", "chr7", [(0, len(ref))]),
             (("--regions", tmp_path / "r.bed"), "ref.fa", "chr7", [(a, b) for _, a, b in bed]),
             ((), "nohead.fa", "nohead", [(0, len(ref))])]
    for j, (opts, rf, chrom, regions) in enumerate(forms):
        out = tmp_path / f"out{j}"
        r = run(env, BIN / "decompress", "--variants", "--archives", tmp_path / "list.txt", *opts, tmp_path / rf, out)
        assert r.returncode == 0, r.stderr
        got = (out / "variants.vcf").read_bytes()
        assert got == render_vcf(chrom, ref, stems, Ds, wholes, regions), opts
        assert got.count(b"\n") > 10
        assert not (out / "variants.vcf.part").exists()
    # errors: exit 1, a message, no variants.vcf and no variants.vcf.part
    (tmp_path / "bad.bed").write_text("g\t30\t20\n")
    (tmp_path / "far.bed").write_text(f"g\t0\t{len(ref) + 1}\n")
    (tmp_path / "empty.txt").write_text("\n")
    (tmp_path / "missing.txt").write_text(str(arcs[0]) + "\n" + str(tmp_path / "nope.7z") + "\n")
    good = ("--archives", tmp_path / "list.txt")
    cases = [good + o for o in (("--regions", tmp_path / "bad.bed"), ("--regions", tmp_path / "far.bed"), ("--regions", tmp_path / "nope.bed"),
                                ("--bogus", "1"))]
    cases += [("--archives", tmp_path / lst) for lst in ("empty.txt", "missing.txt", "nolist.txt")]
    cases += [("--regions", tmp_path / "r.bed")]
    for i, opts in enumerate(cases):
        out = tmp_path / f"err{i}"
        r = run(env, BIN / "decompress", "--variants", *opts, tmp_path / "ref.fa", out)
        assert r.returncode == 1 and r.stderr, opts
        assert not (out / "variants.vcf").exists() and not (out / "variants.vcf.part").exists(), opts
    out = tmp_path / "errref"
    r = run(env, BIN / "decompress", "--variants", *good, tmp_path / "nope.fa", out)
    assert r.returncode == 1 and not (out / "variants.vcf").exists()


def hand_archive(env, d, name: str, inter: bytes):  # noqa: F811
    """a record file written by hand, packed as <name>.txt.7z"""
    d.mkdir(exist_ok=True)
    (d / f"{name}.txt").write_bytes(inter)
    r = run(env, "7z", "a", "-mx=9", d / f"{name}.txt.7z", d / f"{name}.txt")
    assert r.returncode == 0, r.stderr
    return d / f"{name}.txt.7z"


def test_variants_edges(env, tmp_path):  # noqa: F811
    """records at pos 0 (deletion, insertion, complex), an insertion at len(R), an empty target (all of R deleted), two
    archives sharing a row, overlapping BED regions, an identical target alone (a header-only VCF); then a target whose
    ALT bytes are not letters: exit 1 naming the position, no variants.vcf and no variants.vcf.part"""
    from test_emu_search_space import odd_target_archive
    from test_emu_variants import hand_file, tokens
    from test_emu_variants_space import bases
    R = bases(3000, 31)
    L = len(R)
    ol.write_fasta(tmp_path / "ref.fa", R, b">chr2 edges")
    snp = b"T" if R[1200:1201] != b"T" else b"G"
    files = {"del0": tokens((5, L - 5)), "ins0": b"GG" + tokens((0, L)), "cx0": b"TTTT" + tokens((2, L - 2)),
             "insL": tokens((0, L)) + b"CC", "empty": b"", "snpA": tokens((0, 1200), snp, (1201, L - 1201)),
             "snpB": tokens((0, 1200), snp, (1201, 1000), (2300, L - 2300))}
    arcs, Ds, wholes = [], [], []
    for name, body in files.items():
        inter = hand_file(body)
        arcs.append(hand_archive(env, tmp_path / "a", name, inter))
        Ds.append(vl.decoded(R, inter))
        wholes.append(vl.variants_whole(R, inter, Ds[-1]))
    stems = [a.stem for a in arcs]
    (tmp_path / "list.txt").write_text("".join(f"{a}\n" for a in arcs))
    bed = [(0, 1500), (1000, L), (1100, 1300), (L - 10, L)]
    (tmp_path / "r.bed").write_text("".join(f"chr2\t{a}\t{b}\n" for a, b in bed))
    for j, (opts, regions) in enumerate((((), [(0, L)]), (("--regions", tmp_path / "r.bed"), bed))):
        out = tmp_path / f"out{j}"
        r = run(env, BIN / "decompress", "--variants", "--archives", tmp_path / "list.txt", *opts, tmp_path / "ref.fa", out)
        assert r.returncode == 0, r.stderr
        got = (out / "variants.vcf").read_bytes()
        assert got == render_vcf("chr2", R, stems, Ds, wholes, regions), opts
        rows = [l.split(b"\t") for l in got.splitlines() if not l.startswith(b"#")]
        assert sum(1 for f in rows if f[1] == b"1") >= 3                   # three records at pos 0 (POS 1)
        assert any(f[-2:] == [b"1", b"1"] for f in rows)                  # the SNP both snpA and snpB carry: one row
        assert any(f[3] == vl.up(R[:L]) + b"N" for f in rows)             # the empty target: all of R deleted
    # an identical target alone: a header-only VCF
    (tmp_path / "same.txt").write_text(f"{hand_archive(env, tmp_path / 's', 'same', hand_file(tokens((0, L))))}\n")
    r = run(env, BIN / "decompress", "--variants", "--archives", tmp_path / "same.txt", tmp_path / "ref.fa", tmp_path / "outs")
    assert r.returncode == 0, r.stderr
    got = (tmp_path / "outs" / "variants.vcf").read_bytes()
    assert got == render_vcf("chr2", R, ["same.txt"], [R], [vl.variants_whole(R, hand_file(tokens((0, L))))], [(0, L)]) and got.count(b"\n") == 4
    # ALT bytes that are not letters (tab, ',', control bytes, bytes >= 0x80): refused, nothing written
    ref2, inter2, _, _, D2 = odd_target_archive()
    ol.write_fasta(tmp_path / "ref2.fa", ref2, b">chrO")
    (tmp_path / "odd.txt").write_text(f"{hand_archive(env, tmp_path / 'o', 'odd', inter2)}\n")
    out = tmp_path / "outo"
    r = run(env, BIN / "decompress", "--variants", "--archives", tmp_path / "odd.txt", tmp_path / "ref2.fa", out)
    assert r.returncode == 1 and b"position" in r.stderr and b"letters" in r.stderr, r.stderr
    assert not (out / "variants.vcf").exists() and not (out / "variants.vcf.part").exists()
    # the same archive in a region of letter records only is written
    W = vl.variants_whole(ref2, inter2, D2)
    bad = [int(p) for p, e, s, t in W.tolist() if not all(65 <= c <= 90 for c in vl.up(D2[s:t]) + vl.up(ref2[p:e]))]
    assert bad and bad[0] > 0
    (tmp_path / "first.bed").write_text(f"chrO\t0\t{bad[0]}\n")
    r = run(env, BIN / "decompress", "--variants", "--archives", tmp_path / "odd.txt", "--regions", tmp_path / "first.bed", tmp_path / "ref2.fa", out)
    assert r.returncode == 0, r.stderr
    assert (out / "variants.vcf").read_bytes() == render_vcf("chrO", ref2, ["odd.txt"], [D2], [W], [(0, bad[0])])
