"""Archives (sccg_archive_open / sccg_archive_extract, include/sccg.h) on the CPU (SIMT emulator build): every query must give
the bytes of D, the decoded sequence of the whole-image decoder, or the reverse complement of a slice of it, and every error
must be the one the contract names.  The check_* functions are shared with test_gpu_archive.py."""
import ctypes as C
import random

import numpy as np
import pytest

import oracle_lib as ol
import sccg_b200
from cases import cases, rnd
from emu_lib import emu_context
from test_emu_extract import CASES, PATHS, env, mixed_regions, seq_of, tolerance_cases, unpack

ARG = sccg_b200.SCCG_E_ARG


@pytest.fixture(scope="module")
def ctx():
    c = emu_context()
    yield c
    c.close()


def _comp_table() -> bytes:
    t = bytearray(range(256))
    for a, b in (b"AT", b"CG", b"RY", b"KM", b"BV", b"DH"):
        for x, y in ((a, b), (a | 0x20, b | 0x20)):
            t[x], t[y] = y, x
    return bytes(t)


COMP = _comp_table()


def revcomp(s: bytes) -> bytes:
    return s.translate(COMP)[::-1]


def expect(Ds, queries) -> bytes:
    """Ds: D of every archive; queries: rows [archive, start, end, strand]"""
    out = []
    for a, s, e, st in queries:
        piece = Ds[a][s:e]
        out.append(revcomp(piece) if st else piece)
    return b"".join(out)


def check_query(ctx, archives, Ds, queries, path="auto"):
    with env(SCCG_EXT_LANE_MIN=PATHS[path]):
        got = ctx.query(archives, queries)
    exp = expect(Ds, queries)
    assert len(got) == len(exp)
    if got != exp:
        bad = next(i for i in range(len(exp)) if got[i] != exp[i])
        raise AssertionError(f"first difference at output byte {bad} ({path}): got {got[bad:bad + 16]!r}, expected {exp[bad:bad + 16]!r}")


def both_strands(a: int, regions, seed):
    r = random.Random(repr(seed))
    return [(a, s, e, r.randrange(2)) for s, e in regions] + [(a, s, e, 1) for s, e in regions[:8]]


def check_golden_archives(ctx, golden):
    """every golden case as an archive: the opens that must fail fail with decompress_resident's code, the others answer
    mixed_regions queries on both strands"""
    for case in CASES:
        g = golden["cases"][case.name]
        inter = unpack(g["intermediate_z"])
        ctx.set_reference(case.ref)
        try:
            image = ctx.decompress_resident(inter)
        except sccg_b200.SccgError as e1:
            with pytest.raises(sccg_b200.SccgError) as e2:
                ctx.open_archive(inter)
            assert e2.value.code == e1.code, case.name
            continue
        D = seq_of(image)
        with ctx.open_archive(inter) as a:
            assert a.seq_len == len(D), case.name
            assert a.mode == (0 if inter.split(b"\n")[(2 if inter.startswith(b">") else 1)] == b"," else 1), case.name
            assert a.device_bytes > 0
            check_query(ctx, [a], [D], both_strands(0, mixed_regions(len(D), case.name), case.name))
    ctx.clear_reference()


def archive_set(n: int = 120_000, seed: int = 71):
    """one reference and the record files of several targets against it: a local-mode target with N runs and lowercase runs,
    a global-mode target (an uncompensated deletion near the start), a hand-written file with out-of-order run lists, and a
    second local-mode target -> (ref, [(intermediate, D, mode)])"""
    from sccg_genome_compression_b200 import synth
    ref_np, tgt_np = synth.local_pair(n, synth.seed_for(2, seed))
    ref = ref_np.tobytes()
    t = bytearray(tgt_np.tobytes())
    for a, b in ((4090, 4100), (8191, 8193), (20_000, 24_500), (50_001, 50_002)):
        t[a:b] = b"N" * (b - a)
    for a, b in ((3000, 3001), (4095, 4200), (12_288, 16_400), (60_000, 60_999)):
        t[a:b] = bytes(t[a:b]).lower()
    rng = np.random.default_rng(seed)
    g = ref_np.copy()
    synth.substitute(rng, g, 0.001)
    gtgt = np.concatenate([g[:1000], g[6000:]]).tobytes()                  # 5 kb deleted near the start, not compensated
    l2 = ref_np.copy()
    synth.substitute(rng, l2, 0.002)
    synth.lowercase_runs(rng, l2, 0.3, 10, 2000)
    out = []
    for tgt in (bytes(t), gtgt, l2.tobytes()):
        rc, inter, mode = ol.orc_compress(ref, tgt, b">arch")
        assert rc == 0
        rc, image = ol.orc_decompress(ref, inter)
        assert rc == 0
        out.append((inter, seq_of(image), mode))
    assert [m for _, _, m in out] == [0, 1, 0]
    enc, nidx, low = tolerance_cases()[2]                                  # N and lowercase run lists out of order
    inter = b">tolerant\n" + low + b"\n" + nidx + b"\n" + enc
    rc, image = ol.orc_decompress(ref, inter)
    assert rc == 0
    out.insert(2, (inter, seq_of(image), 1))
    return ref, out


def query_sets(Ds, seed):
    """interleaved across archives and strands (tiles that mix archives), and grouped by archive (tiles of one archive)"""
    r = random.Random(seed)
    n = len(Ds)
    mixed = []
    for k in range(3000):
        a = k % n
        L = len(Ds[a])
        s = r.randrange(L + 1)
        mixed.append((a, s, min(L, s + r.choice([0, 1, 1, 2, 7, 40, 150, 999, 5000])), r.randrange(2)))
    grouped = []
    for a in range(n):
        L = len(Ds[a])
        grouped += [(a, s, s + 1, r.randrange(2)) for s in (r.randrange(L) for _ in range(1500))]
        grouped += [(a, s, min(L, s + 150), r.randrange(2)) for s in (r.randrange(L) for _ in range(40))]
    long_ = [(a, 0, len(Ds[a]), st) for a in range(n) for st in (0, 1)]
    edges = [(a, s, e, st) for a in range(n) for s, e in mixed_regions(len(Ds[a]), (seed, a), 30) for st in (0, 1)]
    r.shuffle(edges)
    return [mixed, grouped, long_, edges]


def check_many_archives(ctx, paths=tuple(PATHS)):
    ref, files = archive_set()
    ctx.set_reference(ref)
    archives = [ctx.open_archive(inter) for inter, _, _ in files]
    Ds = [D for _, D, _ in files]
    assert [a.mode for a in archives] == [m for _, _, m in files]
    assert [a.seq_len for a in archives] == [len(D) for D in Ds]
    for qs in query_sets(Ds, 5):
        for path in paths:
            check_query(ctx, archives, Ds, qs, path)
    q = np.array(query_sets(Ds, 6)[0], dtype=np.int64)                    # an (n, 4) int64 array goes straight through
    assert ctx.query(archives, q) == expect(Ds, q.tolist())
    for a in archives:
        a.close()


def check_lifetime(ctx):
    """the tables of an archive survive every other call on the context; closing one archive leaves the others"""
    ref, files = archive_set(60_000, 72)
    ctx.set_reference(ref)
    A = ctx.open_archive(files[0][0])
    DA = files[0][1]
    qs = [(0, 5, 4000, 0), (0, 100, 250, 1), (0, len(DA) - 7, len(DA), 1)]
    other = rnd(20_000, "life")
    img, _ = ctx.compress(ref, other, b">x")
    ctx.decompress(ref, img)
    ctx.extract(ref, files[1][0], [(0, 100)])
    ctx.decompress_resident(files[2][0])
    ctx.compress_resident(other)
    B = ctx.open_archive(files[1][0])
    C_ = ctx.open_archive(files[2][0])
    check_query(ctx, [A], [DA], qs)
    check_query(ctx, [B, A, C_], [files[1][1], DA, files[2][1]], [(1, 3, 900, 1), (0, 10, 20, 0), (2, 0, 64, 1), (1, 0, 5, 0)])
    B.close()
    check_query(ctx, [A, C_], [DA, files[2][1]], [(1, 0, len(files[2][1]), 1), (0, 0, 5000, 0)])
    with pytest.raises(sccg_b200.SccgError) as e:                          # a closed archive is a NULL entry
        ctx.query([B], [(0, 0, 1, 0)])
    assert e.value.code == ARG
    A.close(); C_.close()


def check_reference_generation(ctx):
    ref, files = archive_set(60_000, 73)
    ctx.set_reference(ref)
    A = ctx.open_archive(files[0][0])
    G = ctx.open_archive(files[1][0])
    q = [(0, 0, 300, 1), (1, 10, 80, 0)]
    Ds = [files[0][1], files[1][1]]
    check_query(ctx, [A, G], Ds, q)
    for change in (lambda: ctx.set_reference(rnd(len(ref), "other")), ctx.clear_reference, lambda: ctx.set_reference(ref)):
        change()
        with pytest.raises(sccg_b200.SccgError) as e:
            ctx.query([A, G], q)
        assert e.value.code == ARG and "resident reference" in str(e.value)
        assert ctx.query([A, G], []) == b""                                # a stale archive that no query names is fine
    A.close(); G.close()                                                   # stale archives can still be closed
    ctx.set_reference(ref)
    A = ctx.open_archive(files[0][0])
    G = ctx.open_archive(files[1][0])
    check_query(ctx, [A, G], Ds, q)
    A.close(); G.close()
    ctx.clear_reference()
    with pytest.raises(sccg_b200.SccgError) as e:
        ctx.open_archive(files[0][0])
    assert e.value.code == ARG


def check_argument_errors(ctx, ctx2):
    ref, files = archive_set(30_000, 74)
    ctx.set_reference(ref)
    A = ctx.open_archive(files[0][0])
    D = files[0][1]
    L = len(D)
    good = [(0, 3, 40, 1), (0, 0, L, 0)]

    def fails(msg, archives, queries, *out):
        with pytest.raises(sccg_b200.SccgError) as e:
            ctx.query(archives, queries, *out)
        assert e.value.code == ARG and msg in str(e.value), str(e.value)
        check_query(ctx, [A], [D], good)                                   # the context survived
        return e.value
    lib = ctx.lib
    n = C.c_int64()
    arr = (C.c_void_p * 1)(A.handle)
    qa = np.array([[0, 0, 1, 0]], dtype=np.int64)
    buf = C.create_string_buffer(64)
    assert lib.sccg_archive_extract(ctx.handle, None, 1, qa.ctypes.data, 1, buf, 64, C.byref(n)) == ARG          # NULL with a count
    assert lib.sccg_archive_extract(ctx.handle, arr, 1, None, 1, buf, 64, C.byref(n)) == ARG
    assert lib.sccg_archive_extract(ctx.handle, arr, -1, qa.ctypes.data, 1, buf, 64, C.byref(n)) == ARG
    assert lib.sccg_archive_extract(ctx.handle, arr, 1, qa.ctypes.data, 1, buf, 64, None) == ARG
    assert lib.sccg_archive_extract(ctx.handle, None, 0, None, 0, None, 0, C.byref(n)) == 0 and n.value == 0
    fails("out of range", [A], [(1, 0, 1, 0)])
    fails("out of range", [A], [(-1, 0, 1, 0)])
    fails("null argument", [A, type("Closed", (), {"handle": None})()], [(1, 0, 1, 0)])
    ctx2.set_reference(ref)
    X = ctx2.open_archive(files[0][0])
    fails("another context", [A, X], [(1, 0, 1, 0)])
    assert ctx2.query([X], good) == expect([D], good)
    X.close()
    fails("start <= end", [A], [(0, -1, 3, 0)])
    fails("start <= end", [A], [(0, 5, 4, 1)])
    fails("past the end", [A], [(0, 0, L + 1, 0)])
    fails("past the end", [A], [(0, L + 5, L + 5, 0)])
    fails("strand", [A], [(0, 0, 1, 2)])
    fails("strand", [A], [(0, 0, 1, -1)])
    k = (1 << 31) // L + 1
    fails("2^31 bytes", [A], np.tile(np.array([[0, 0, L, 0]], dtype=np.int64), (k, 1)))
    e = fails("too small", [A], [(0, 0, 100, 1)], C.cast(buf, C.c_void_p).value, 99)
    assert e.out_len == 100
    # the order of the list in include/sccg.h, whichever queries commit the errors; totals and the buffer last
    ctx2.set_reference(ref)
    X = ctx2.open_archive(files[0][0])
    fails("out of range", [A, X], [(0, 0, 1, 7), (1, 0, 1, 0), (0, L + 1, L + 1, 0), (2, 0, 1, 0)])
    fails("another context", [A, X], [(0, 9, 1, 7), (0, 0, L + 1, 0), (1, 0, 1, 0)])
    X.close()
    fails("start <= end", [A], [(0, 0, 1, 7), (0, 0, L + 1, 0), (0, 9, 1, 0)])
    fails("past the end", [A], [(0, 0, 1, 7), (0, 0, L + 1, 0)])
    fails("strand", [A], [(0, 0, 1, 7)] + [(0, 0, L, 0)] * k, C.cast(buf, C.c_void_p).value, 1)
    assert ctx.query([A], [(0, 7, 60, 1)], C.cast(buf, C.c_void_p).value, 64) == 53 and buf.raw[:53] == revcomp(D[7:60])
    assert ctx.query([A], []) == b""
    A.close()
    ctx.clear_reference()


def every_byte_archive():
    """the reference holds every byte but '\n' (which D cannot hold; tokens copy them, upper-cased), literals add IUPAC
    codes and other bytes in both cases, a lowercase run lowers a stretch -> (ref, intermediate, D)"""
    ref = bytes(b for b in range(256) if b != 10) * 8
    lits = bytes(b for b in range(256) if b not in b"()\n,-0123456789")
    body = b"(0,2040)" + lits + b"(500,300)acgtrykmbvdhswnACGTRYKMBVDHSWN"
    inter = b">comp\n(2100,120)\n,\n" + body
    rc, image = ol.orc_decompress(ref, inter)
    assert rc == 0
    D = seq_of(image)
    assert set(D) == set(range(256)) - {10}
    return ref, inter, D


def check_complement_table(ctx):
    """every byte value D can hold through the minus strand (every_byte_archive)"""
    ref, inter, D = every_byte_archive()
    ctx.set_reference(ref)
    with ctx.open_archive(inter) as a:
        assert a.seq_len == len(D)
        for path in PATHS:
            check_query(ctx, [a], [D], [(0, 0, len(D), 1), (0, 0, len(D), 0)] + [(0, i, i + 1, 1) for i in range(len(D))], path)
    ctx.clear_reference()


def check_no_body_line(ctx):
    """a file whose last line is the N line (the compressor writes one when the record body is empty; the last '\n' ends a
    line and starts none) has no body line for getline: the oracle, decompress, decompress_resident and open_archive all
    refuse it with the same code"""
    ref = b"GGGACGTACGTACGTTT"
    files = [b">x\n(3,12)\n,\n", b"(3,12)\n,\n", b">x\n\n,"]
    rc, inter, mode = ol.orc_compress(ref, b"ACGTNNNNACGTACG", b">x")
    assert rc == 0 and ol.split_intermediate(inter) is None
    assert ctx.compress(ref, b"ACGTNNNNACGTACG", b">x") == (inter, mode)
    files.append(inter)
    ctx.set_reference(ref)
    for f in files:
        assert ol.split_intermediate(f) is None and ol.orc_decompress(ref, f)[0] != 0, f
        for call in (lambda: ctx.decompress(ref, f), lambda: ctx.decompress_resident(f), lambda: ctx.open_archive(f)):
            with pytest.raises(sccg_b200.SccgError) as e:
                call()
            assert e.value.code == sccg_b200.SCCG_E_FORMAT, (f, str(e.value))
    # one more '\n' gives an empty body line: an empty D
    rc, image = ol.orc_decompress(ref, b">x\n\n,\n\n")
    assert rc == 0 and seq_of(image) == b"" and ctx.decompress(ref, b">x\n\n,\n\n") == image
    ctx.clear_reference()


def test_comp_table():
    assert revcomp(b"ACGTacgtRYKMBVDHSWNrykmbvdhswn!\x00\xff") == b"\xff\x00!nwsdhbvkmryNWSDHBVKMRYacgtACGT"
    assert all(COMP[COMP[b]] == b for b in range(256))


def test_golden_cases(ctx, golden):
    check_golden_archives(ctx, golden)


def test_many_archives(ctx):
    check_many_archives(ctx)


def test_lifetime(ctx):
    check_lifetime(ctx)


def test_reference_generation(ctx):
    check_reference_generation(ctx)


def test_argument_errors(ctx):
    ctx2 = emu_context()
    try:
        check_argument_errors(ctx, ctx2)
    finally:
        ctx2.close()


def test_complement_table(ctx):
    check_complement_table(ctx)


def test_no_body_line(ctx):
    check_no_body_line(ctx)
