"""Record-body tokens outside the canonical "(d,l)" text on the CPU (SIMT emulator build) against the oracle, and the oracle's
token loop against libstdc++'s own find / substr / stoi (tests/stoi_probe.cpp).  The check_* functions live in
token_grammar_cases.py and are shared with test_gpu_token_grammar.py."""
import random
import subprocess
from pathlib import Path

import pytest

import oracle_lib as ol
import token_grammar_cases as tg
from emu_lib import emu_context
from test_emu_cli import BIN, env  # noqa: F401  (env: the emulator CLIs and the 7z shim)

HERE = Path(__file__).resolve().parent


@pytest.fixture(scope="module")
def ctx():
    c = emu_context()
    yield c
    c.close()


def test_body_table(ctx):
    tg.check_table(ctx)


def test_phase_and_length_sweep(ctx):
    tg.check_sweep(ctx)


@pytest.mark.parametrize("seeds", [range(0, 4), range(4, 8), range(8, 12)], ids=["0-3", "4-7", "8-11"])
def test_fuzzed_bodies(ctx, seeds):
    tg.check_fuzz(ctx, seeds)


def test_every_entry_point(ctx):
    tg.check_entry_corpus(ctx)


def test_own_round_trip(ctx):
    tg.check_roundtrips(ctx)


@pytest.mark.parametrize("piece", [b"(5,+3)", b"(1,2,3)", b"(5,3x)"], ids=["plus", "second_comma", "trailing_x"])
def test_cli_round_trip(env, tmp_path, piece):  # noqa: F811
    """compress then decompress through the command-line programs (emulator build): the exit code and
    reconstructed_genome.fa are the oracle's.  (The FASTA reader drops isspace, so "(5, 3)" reaches the body as "(5,3)".)"""
    ref, tgt = tg.piece_pair(piece, False)
    ol.write_fasta(tmp_path / "ref.fa", ref, b">ref")
    ol.write_fasta(tmp_path / "tgt.fa", tgt, b">tgt")
    ref_seq = ol.orc_parse_reference_fasta((tmp_path / "ref.fa").read_bytes())
    tgt_seq, header = ol.orc_parse_target_fasta((tmp_path / "tgt.fa").read_bytes())
    rc_c, inter, mode = ol.orc_compress(ref_seq, tgt_seq, header)
    assert rc_c == 0 and piece in tgt_seq
    rc_o, image = ol.orc_decompress(ref_seq, inter)
    r = subprocess.run([str(BIN / "compress"), str(tmp_path / "ref.fa"), str(tmp_path / "tgt.fa"), str(tmp_path / "out")], env=env, capture_output=True)
    assert r.returncode == 0, r.stderr
    assert (tmp_path / "out" / "compressed_genome.txt").read_bytes() == inter
    r = subprocess.run([str(BIN / "decompress"), str(tmp_path / "out" / "compressed_genome.txt.7z"), str(tmp_path / "ref.fa"), str(tmp_path / "dec")],
                       env=env, capture_output=True)
    assert rc_o == 0 and tg.pinned_class(ol.split_intermediate(inter)[3]) is None
    assert r.returncode == 0, r.stderr
    assert (tmp_path / "dec" / "reconstructed_genome.fa").read_bytes() == image


# ------------------------------------------------------------------------------------------------ the oracle's witness
@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    exe = tmp_path_factory.mktemp("stoi_probe") / "stoi_probe"
    subprocess.check_call(["/usr/bin/g++" if Path("/usr/bin/g++").exists() else "g++", "-O1", "-std=c++17", "-fwrapv",
                           str(HERE / "stoi_probe.cpp"), "-o", str(exe)])
    return exe


def wrap50(rec: bytes) -> bytes:
    """decompression.cpp:266-274 on a record without run lists"""
    return b"".join(rec[p:p + 50] + (b"\n" if p + 50 < len(rec) else b"") for p in range(0, len(rec), 50)) + b"\n"


def probe_corpus():
    rows = [(tg.TABLE_REF, b) for b in tg.token_table() + tg.sweep_bodies()]
    rows += [(ref, body) for ref, body, _, _ in tg.fuzz_corpus(range(12))]
    r = random.Random("probe")                              # and bodies that are mostly grammar bytes
    for _ in range(3000):
        rows.append((tg.TABLE_REF, bytes(r.choice(b"(),,+-  \t0123456789AC") for _ in range(r.randint(1, 30)))))
    return rows


def test_stoi_probe_agrees_with_oracle(probe, tmp_path):
    """the oracle's token loop (orc_reconstruct, empty run lists) against the reference's loop run on libstdc++'s find /
    substr / stoi, over the table, the sweep, the fuzz corpus and random grammar soup"""
    rows = [(ref, body) for ref, body in probe_corpus() if b"\n" not in body]
    (tmp_path / "cases").write_bytes(b"".join(ref.hex().encode() + b" " + body.hex().encode() + b"\n" for ref, body in rows))
    out = subprocess.run([str(probe), str(tmp_path / "cases")], capture_output=True, check=True).stdout.split(b"\n")
    assert len(out) == len(rows) + 1
    verdicts = {"ok": 0, "fail": 0}
    for (ref, body), line in zip(rows, out):
        rc, exp = ol.orc_reconstruct(ref, body, b"", b"")
        status, _, rest = line.partition(b" ")
        if status == b"ok":
            assert rc == 0 and exp == wrap50(bytes.fromhex(rest.decode())), body
            verdicts["ok"] += 1
        else:
            assert rc == (3 if rest == b"bounds" else 1), (body, line, rc)
            verdicts["fail"] += 1
    assert verdicts["ok"] > 1000 and verdicts["fail"] > 1000
