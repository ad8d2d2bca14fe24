"""Region extraction on the B200 (`-m gpu`): the parity battery of test_emu_extract.py through the product library, full-size
pairs (BASELINE cfg 2: chr1-sized, local mode; cfg 1: chr19-shaped gap pair, global mode) and the product CLI."""
import random
import subprocess
from pathlib import Path

import numpy as np
import pytest

import oracle_lib as ol
import sccg_b200
from test_emu_extract import (boundary_pairs, check_argument_errors, check_boundaries, check_chunk_selection, check_golden_cases,
                              check_interleaving, check_random_streams, check_resident, check_unsorted_run_lists, expect)
from test_emu_extract_cli import render

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent


@pytest.fixture(scope="module")
def ctx():
    c = sccg_b200.Context(0)
    yield c
    c.close()


def test_golden_cases(ctx, golden):
    check_golden_cases(ctx, golden)


def test_random_record_streams(ctx):
    check_random_streams(ctx, range(40))


def test_region_edges(ctx):
    check_boundaries(ctx, boundary_pairs(400_000))


def test_reference_chunk_selection(ctx):
    check_chunk_selection(ctx)


def test_unsorted_run_lists(ctx):
    check_unsorted_run_lists(ctx)


def test_resident(ctx):
    check_resident(ctx)


def test_argument_errors(ctx):
    check_argument_errors(ctx)


def test_decompress_extract_decompress(ctx):
    check_interleaving(ctx)


@pytest.mark.parametrize("cfg", [2, 1])
def test_full_size(ctx, cfg):
    """lossless synthetic pairs: D is the target's symbols"""
    from sccg_genome_compression_b200 import synth
    if cfg == 2:
        ref, tgt = synth.local_pair(synth.CHR1_LEN, synth.seed_for(2, 0))
    else:
        ref, tgt = synth.global_gap_pair(63_811_651, 59_128_983, synth.seed_for(1, 0))
    ref, tgt = ref.tobytes(), tgt.tobytes()
    inter, mode = ctx.compress(ref, tgt, b">full")
    assert mode == (0 if cfg == 2 else 1)
    Lm = len(tgt)
    assert ctx.extract(ref, inter, [(0, Lm)]) == tgt
    h2d_whole = ctx.profile()["h2d_ms"]
    r = np.random.default_rng(cfg)
    starts = r.integers(0, Lm - 10_000, 10_000)
    regs = np.stack([starts, starts + r.integers(1, 10_001, 10_000)], axis=1).astype(np.int64)
    assert ctx.extract(ref, inter, regs) == expect(tgt, regs.tolist())
    w0 = int(r.integers(0, Lm - 2_000_000))
    starts = w0 + r.integers(0, 2_000_000 - 1000, 1000)
    regs = np.stack([starts, starts + 1000], axis=1).astype(np.int64)
    assert ctx.extract(ref, inter, regs) == expect(tgt, regs.tolist())
    if cfg == 2:
        assert ctx.profile()["h2d_ms"] < h2d_whole / 3                      # one or two 16 MiB chunks, not the whole reference
    ctx.set_reference(ref)
    assert ctx.extract_resident(inter, regs) == expect(tgt, regs.tolist())
    ctx.clear_reference()


def test_cli_regions(tmp_path):
    """the product program: `decompress --regions` on a mid-size pair"""
    import os
    import shutil
    from sccg_genome_compression_b200 import synth
    ref, tgt = synth.local_pair(3_000_000, synth.seed_for(2, 65))
    ref, tgt = ref.tobytes(), tgt.tobytes()
    ol.write_fasta(tmp_path / "ref.fa", ref, b">ref")
    rc, inter, mode = ol.orc_compress(ref, tgt, b">chrM")
    assert rc == 0
    d = tmp_path / "shim"; d.mkdir()
    shutil.copy(ROOT / "oracle" / "7z_shim.sh", d / "7z"); os.chmod(d / "7z", 0o755)
    arc = tmp_path / "compressed_genome.txt.7z"
    arc.write_bytes(inter)                                                  # the shim "extracts" by copying
    r = random.Random(65)
    bed = [(f"r{i}", a, min(len(tgt), a + r.randint(0, 3000))) for i, a in enumerate(r.randrange(len(tgt)) for _ in range(300))]
    (tmp_path / "r.bed").write_text("".join(f"{n}\t{a}\t{b}\n" for n, a, b in bed))
    e = dict(os.environ); e["PATH"] = str(d) + os.pathsep + e.get("PATH", "")
    p = subprocess.run([str(ROOT / "sccg-genome-compression_b200" / "bin" / "decompress"), "--regions", str(tmp_path / "r.bed"), str(arc),
                        str(tmp_path / "ref.fa"), str(tmp_path / "out")], env=e, capture_output=True)
    assert p.returncode == 0, p.stderr
    assert (tmp_path / "out" / "regions.fa").read_bytes() == render(tgt, bed)
