"""Pins the C oracle against the UNMODIFIED reference at function level and at CLI level on seeded random inputs.

Every case runs the same steps on two sides -- the C oracle and the reference -- and compares what the original comparison
looked at.  The reference side is tests/golden/reference_function_level.json (made by tests/golden/make_function_goldens.py:
a fingerprint, length + sha256, of every output, next to fingerprints of the inputs), so the comparison runs everywhere.  Where
oracle/_ref has been built from the reference's sources (not part of this repository), the compiled reference is run as well."""
import hashlib
import json
import random
import tempfile
from pathlib import Path

import pytest

import oracle_lib as ol
from cases import rnd

GOLDEN_FILE = Path(__file__).resolve().parent / "golden" / "reference_function_level.json"


def fp(data: bytes) -> str:
    """fingerprint of an output: its length and sha256"""
    return f"{len(data)}:{hashlib.sha256(data).hexdigest()}"


def fp_records(recs) -> str:
    return fp(json.dumps([[r.p, r.l, r.lit.hex()] for r in recs]).encode())


# ----------------------------------------------------------------------------------------- inputs
def _pair(seed, n, alphabet=b"ACGT", snp=0.01, indel=0.0):
    r = random.Random(repr(seed))
    ref = bytes(r.choice(alphabet) for _ in range(n))
    t = bytearray()
    for c in ref:
        x = r.random()
        if x < snp:
            t.append(r.choice(alphabet))
        elif x < snp + indel / 2:
            continue
        elif x < snp + indel:
            t.append(c); t.append(r.choice(alphabet))
        else:
            t.append(c)
    return ref, bytes(t)


def local_inputs(seed):
    alphabet = [b"ACGT", b"AC", b"ACGTN", b"A"][seed % 4]
    return _pair(("loc", seed), random.Random(seed).randint(5, 1000), alphabet, snp=0.02, indel=0.004)


def global_inputs(seed):
    alphabet = [b"ACGT", b"ACGT", b"AC"][seed % 3]
    n = 20000 if alphabet == b"ACGT" else 3000
    ref, tgt = _pair(("glob", seed), n, alphabet, snp=0.01, indel=0.002)
    r = random.Random(seed)
    if seed % 2:                       # rearrange blocks so the parse gets lost and re-syncs by chance
        cut = sorted(r.sample(range(len(tgt)), 4))
        parts = [tgt[:cut[0]], tgt[cut[0]:cut[1]], tgt[cut[1]:cut[2]], tgt[cut[2]:cut[3]], tgt[cut[3]:]]
        r.shuffle(parts)
        tgt = b"".join(parts)
    return ref, tgt


def e2e_inputs(seed):
    r = random.Random(repr(("e2e", seed)))
    n = r.randint(3000, 40000)
    ref, tgt = _pair(("e2e", seed), n, b"ACGT", snp=0.003, indel=0.0005 if seed % 2 else 0.0)
    t = bytearray(tgt)
    for _ in range(8):                 # lowercase + N runs
        a = r.randrange(len(t)); b = min(len(t), a + r.choice([1, 2, 30, 700]))
        t[a:b] = bytes(t[a:b]).lower()
        a = r.randrange(len(t)); b = min(len(t), a + r.choice([1, 5, 120]))
        t[a:b] = b"N" * (b - a)
    return ref, bytes(t), b">e2e %d" % seed


DELTA_TEXTS = [
    b">h\n\n,\n(0,500)(7,(503,497)(1000,1000)",
    b"\n,\n(10,5)AC(4,6)(100,1)",
    b">chr1 (x,1)\n(5,2)\n,\n(7,7)(9,9)",
    b">h\n(3,4)9,\n(1,2)\n(100,5)(90,5)ACGT(2000000000,7)(-5,3)",
    b">h\n\n,\nACGT",
    b">h\n\n,\n(12)(3,4)(5",
]

MALFORMED = [
    (b"(0,100)ACGT(50,20)", b"", b"(3,4)10,200"),
    (b"(0,100)ACGT(50,20)", b"2,(5,3)(100,2)", b""),
    (b"AC(10,-3)GT", b"", b""),                      # negative length: substr count wraps -> rest of reference
    (b"(0,10)x5y", b"", b"0,1,1,"),
    (b"(5,5)", b"", b"(0,2),(4,2)7"),
]
STOI_THROWS = [b"(a,5)", b"(5,)", b"(99999999999,5)"]


def grammar_inputs(seed):
    from test_emu_compress import grammar_pair
    ref, tgt = grammar_pair(seed, make_global=(seed % 4 >= 2))
    return ref, tgt, b">gram (alt) 1,2"


SHAPES = ["shifted_tail", "leftover_only", "reference_insertion", "small_shift"]


def mismatch_inputs(shape):
    n = 200_000
    ref = rnd(n, "probe")
    r = random.Random("probe" + shape)
    t = bytearray(ref)
    for p in r.sample(range(n), 150):
        t[p] = r.choice(b"ACGT")
    if shape == "shifted_tail":
        tgt = bytes(t[:60_000]) + bytes(t[63_000:])
    elif shape == "leftover_only":
        tgt = bytes(t) + rnd(5_000, "extra")
    elif shape == "reference_insertion":
        tgt = bytes(t); ref = ref[:20_000] + rnd(2_500, "ins") + ref[20_000:]
    else:
        tgt = bytes(t[:90_000]) + b"ACGTTGCAAC" * 3 + bytes(t[90_000:]) + rnd(1_200, "tail")
    return ref, tgt


# -------------------------------------------------------------------- the two sides of a comparison
class Oracle:
    name = "oracle"
    match = staticmethod(ol.orc_match_sequences)
    reconstruct = staticmethod(ol.orc_reconstruct)
    delta_encode = staticmethod(ol.orc_delta_encode)

    @staticmethod
    def compress_cli(ref, tgt, header):
        """-> (the program failed, the compressed_genome.txt it left)"""
        rc, text, _ = ol.orc_compress(ref, tgt, header)
        return rc != 0, text

    @staticmethod
    def roundtrip(ref, tgt, header):
        rc_c, inter, _ = ol.orc_compress(ref, tgt, header)
        rc_d, recon = ol.orc_decompress(ref, inter)
        return rc_c == 0, inter, rc_d == 0, recon


class Reference:
    """the compiled reference (oracle/_ref): its functions through the harness library, its programs with 7z as a copy"""
    name = "reference"
    match = staticmethod(ol.ref_match_sequences)

    @staticmethod
    def reconstruct(ref, enc, n_idx, low_idx):
        return ol.ref_reconstruct(ref, enc, n_idx, low_idx)[:2]

    @staticmethod
    def delta_encode(text):
        with tempfile.TemporaryDirectory() as d:
            p = Path(d) / "f.txt"
            p.write_bytes(text)
            rc = ol.ref().sccg_ref_delta_encode(str(p).encode())
            return rc, p.read_bytes()

    @staticmethod
    def compress_cli(ref, tgt, header):
        with tempfile.TemporaryDirectory() as d:
            d = Path(d)
            ol.write_fasta(d / "r.fa", ref, b">ref")
            ol.write_fasta(d / "t.fa", tgt, header)
            rc, inter = ol.ref_compress_cli(d / "r.fa", d / "t.fa", d / "out")
        return rc != 0, inter

    @staticmethod
    def roundtrip(ref, tgt, header):
        res = ol.ref_roundtrip(ref, tgt, header)
        return res["rc_compress"] == 0, res["intermediate"], res["rc_decompress"] == 0, res["reconstructed"]


# ------------------------------------------------------------- what each comparison looks at, per side
def run_local(side, seed):
    ref, tgt = local_inputs(seed)
    return {"inputs": fp(ref + b"\0" + tgt), **{f"k{k}": fp_records(side.match(ref, tgt, k, 0, False, 7000)) for k in (14, 10)}}


def run_global(side, seed):
    ref, tgt = global_inputs(seed)
    return {"inputs": fp(ref + b"\0" + tgt), "records": fp_records(side.match(ref, tgt, 14, 100, True, 0))}


def run_e2e(side, seed):
    ref, tgt, header = e2e_inputs(seed)
    c_ok, inter, d_ok, recon = side.roundtrip(ref, tgt, header)
    _, low, nline, body = ol.split_intermediate(inter)            # function-level reconstruct_genome as well
    rc, out = side.reconstruct(ol.prepare_reference(ref, nline), body, b"" if nline == b"," else nline, low)
    return {"inputs": fp(ref + b"\0" + tgt), "compress_ok": c_ok, "intermediate": fp(inter), "decompress_ok": d_ok,
            "reconstructed": fp(recon), "reconstruct_rc": rc, "reconstruct_out": fp(out)}


def run_delta(side, i):
    rc, out = side.delta_encode(DELTA_TEXTS[i])
    return {"inputs": fp(DELTA_TEXTS[i]), "rc": rc, "out": fp(out)}


def run_malformed(side, _=None):
    ref = rnd(500, "mal")
    out = {"inputs": fp(ref + b"\0" + repr(MALFORMED).encode() + repr(STOI_THROWS).encode())}
    for i, (enc, nidx, low) in enumerate(MALFORMED):
        rc, text = side.reconstruct(ref, enc, nidx, low)
        out[f"case{i}"] = [rc, fp(text)]
    out["stoi_rc"] = [side.reconstruct(ref, enc, b"", b"")[0] for enc in STOI_THROWS]
    return out


def run_grammar(side, seed):
    ref, tgt, header = grammar_inputs(seed)
    failed, inter = side.compress_cli(ref, tgt, header)
    return {"inputs": fp(ref + b"\0" + tgt), "failed": failed, "intermediate": fp(inter)}


def run_mismatch(side, shape):
    ref, tgt = mismatch_inputs(shape)
    c_ok, inter, d_ok, recon = side.roundtrip(ref, tgt, b">probe")
    return {"inputs": fp(ref + b"\0" + tgt), "compress_ok": c_ok, "intermediate": fp(inter), "decompress_ok": d_ok,
            "reconstructed": fp(recon)}


SECTIONS = {"match_local": (run_local, range(12)), "match_global": (run_global, range(10)), "end_to_end": (run_e2e, range(6)),
            "delta_encode": (run_delta, range(len(DELTA_TEXTS))), "reconstruct_malformed": (run_malformed, [0]),
            "grammar_cli": (run_grammar, range(24)), "length_mismatch": (run_mismatch, SHAPES)}


@pytest.fixture(scope="module")
def reference_side():
    return json.loads(GOLDEN_FILE.read_text())["sections"]


def compare(reference_side, section, key):
    """the oracle's view of one case == the stored reference's view (inputs first), and == the compiled reference's view
    where it is built"""
    run = SECTIONS[section][0]
    got = run(Oracle, key)
    want = reference_side[section][str(key)]
    assert got["inputs"] == want["inputs"], "input generator drifted from the stored reference outputs"
    assert got == want
    if ol.have_reference():
        assert got == run(Reference, key)
    return got


@pytest.mark.parametrize("seed", range(12))
def test_match_sequences_local(seed, reference_side):
    compare(reference_side, "match_local", seed)


@pytest.mark.parametrize("seed", range(10))
def test_match_sequences_global(seed, reference_side):
    compare(reference_side, "match_global", seed)


@pytest.mark.parametrize("seed", range(6))
def test_compress_and_reconstruct_end_to_end(seed, reference_side):
    got = compare(reference_side, "end_to_end", seed)
    assert got["compress_ok"] and got["decompress_ok"] and got["reconstruct_rc"] == 0


@pytest.mark.parametrize("i", range(len(DELTA_TEXTS)))
def test_delta_encode_text(i, reference_side):
    got = compare(reference_side, "delta_encode", i)
    assert got["rc"] == 0


def test_reconstruct_malformed_inputs_agree(reference_side):
    got = compare(reference_side, "reconstruct_malformed", 0)
    assert got["stoi_rc"] == [1, 1, 1]                  # stoi throws


@pytest.mark.parametrize("seed", range(24))
def test_grammar_symbols_in_target_cli_level(seed, reference_side):
    """literal '(' ')' ',' digits in the target (SURVEY N2 / experiment J): the oracle's text-level delta_encode against
    the reference program itself, incl. the stoi failure (exit 1, compressed_genome.txt left un-rewritten)"""
    compare(reference_side, "grammar_cli", seed)


@pytest.mark.parametrize("shape", SHAPES)
def test_length_mismatch_shapes_end_to_end(shape, reference_side):
    """pairs of different length, > 160 segment pairs: the shapes for which the GPU path probes the last segments for a T2
    abort before the bulk launch (DESIGN 4.7c).  The oracle's verdict (local vs global) and bytes are the reference's."""
    got = compare(reference_side, "length_mismatch", shape)
    assert got["compress_ok"] and got["decompress_ok"]
    ref, tgt = mismatch_inputs(shape)
    assert ol.orc_compress(ref, tgt, b">probe")[2] == (1 if shape in ("shifted_tail", "reference_insertion") else 0)
