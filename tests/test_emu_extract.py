"""Region extraction (sccg_extract*, include/sccg.h) on the CPU (SIMT emulator build): every output must equal the
concatenated slices of D, the decoded sequence of sccg_decompress's image (first line and newlines removed), and every
error must be the one the contract names.  The check_* functions are shared with test_gpu_extract.py."""
import base64
import os
import random
import zlib
from contextlib import contextmanager

import numpy as np
import pytest

import oracle_lib as ol
import sccg_b200
from cases import cases, fasta_cases, rnd
from emu_lib import emu_context
from test_emu_decode import make_record_stream

CASES = cases()


@pytest.fixture(scope="module")
def ctx():
    c = emu_context()
    yield c
    c.close()


def unpack(s):
    return zlib.decompress(base64.b64decode(s))


def seq_of(image: bytes) -> bytes:
    """D: the reconstructed image without its first line and without newlines"""
    return image.split(b"\n", 1)[1].replace(b"\n", b"") if b"\n" in image else b""


def expect(D: bytes, regions) -> bytes:
    return b"".join(D[a:b] for a, b in regions)


@contextmanager
def env(**kv):
    old = {k: os.environ.get(k) for k in kv}
    os.environ.update({k: str(v) for k, v in kv.items() if v is not None})
    for k, v in kv.items():
        if v is None:
            os.environ.pop(k, None)
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


PATHS = {"auto": None, "lanes": 0, "warps": 1 << 30}         # SCCG_EXT_LANE_MIN: default threshold, every tile per lane, every tile per warp


def mixed_regions(Lm: int, seed, n: int = 50):
    """unsorted, overlapping, touching 0 and Lm, some empty"""
    r = random.Random(repr(seed))
    regs = [(0, min(Lm, 7)), (max(0, Lm - 5), Lm), (0, Lm), (Lm // 2, Lm // 2)]
    while len(regs) < n:
        a = r.randrange(Lm + 1)
        b = min(Lm, a + r.choice([0, 1, 2, 17, 150, 999, 5000, Lm]))
        regs.append((a, b))
    r.shuffle(regs)
    return regs


def check_extract(ctx, ref, inter, D, regions, path="auto"):
    with env(SCCG_EXT_LANE_MIN=PATHS[path]):
        got = ctx.extract(ref, inter, regions)
    assert ctx.last_seq_len == len(D)
    exp = expect(D, regions)
    assert len(got) == len(exp)
    if got != exp:
        bad = next(i for i in range(len(exp)) if got[i] != exp[i])
        raise AssertionError(f"first difference at output byte {bad} ({path}): got {got[bad:bad + 16]!r}, expected {exp[bad:bad + 16]!r}")


def check_golden_cases(ctx, golden):
    for case in CASES:
        g = golden["cases"][case.name]
        inter = unpack(g["intermediate_z"])
        if g["rc_decompress"] != 0:
            with pytest.raises(sccg_b200.SccgError) as e1:
                ctx.decompress(case.ref, inter)
            with pytest.raises(sccg_b200.SccgError) as e2:
                ctx.extract(case.ref, inter, [(0, 0)])
            assert e2.value.code == e1.value.code, case.name
            continue
        D = seq_of(unpack(g["reconstructed_z"]))
        Lm = len(D)
        for regs in ([(0, Lm)], [(0, 0), (Lm, Lm)], mixed_regions(Lm, case.name)):
            check_extract(ctx, case.ref, inter, D, regs)
    for fc in fasta_cases():
        g = golden["fasta_cases"][fc.name]
        inter = unpack(g["intermediate_z"])
        D = seq_of(unpack(g["reconstructed_z"]))
        regs = mixed_regions(len(D), fc.name)
        assert ctx.extract_fasta(fc.ref_file, inter, regs) == expect(D, regs), fc.name


def check_random_streams(ctx, seeds):
    for seed in seeds:
        ref, body, nlist, low = make_record_stream(seed)
        inter = b">r\n" + low + b"\n" + nlist + b"\n" + body
        rc, image = ol.orc_decompress(ref, inter)
        if rc != 0:
            with pytest.raises(sccg_b200.SccgError) as e1:
                ctx.decompress(ref, inter)
            with pytest.raises(sccg_b200.SccgError) as e2:
                ctx.extract(ref, inter, [(0, 0)])
            assert e2.value.code == e1.value.code, seed
            continue
        D = seq_of(image)
        for path in PATHS:
            check_extract(ctx, ref, inter, D, mixed_regions(len(D), ("rs", seed)), path)


def boundary_pairs(n=120_000):
    """a local-mode pair with N runs and lowercase runs in the target, and a global-mode gap pair"""
    from sccg_genome_compression_b200 import synth
    ref, tgt = synth.local_pair(n, synth.seed_for(2, 61))
    t = bytearray(tgt.tobytes())
    for a, b in ((4090, 4100), (8191, 8193), (20_000, 24_500), (50_001, 50_002)):
        t[a:b] = b"N" * (b - a)
    for a, b in ((3000, 3001), (4095, 4200), (12_288, 16_400), (60_000, 60_999), (20_100, 20_200)):
        t[a:b] = bytes(t[a:b]).lower()
    out = [(ref.tobytes(), bytes(t))]
    gref, gtgt = synth.global_gap_pair(90_000, 80_000, synth.seed_for(1, 61))
    out.append((gref.tobytes(), gtgt.tobytes()))
    return out


def boundary_region_sets(D: bytes, seed):
    Lm = len(D)
    r = random.Random(seed)
    edges = set()
    for pat in (b"N", b"acgtn"):                                       # N-run edges, lowercase-run edges
        inside = [(c in pat) for c in D]
        for i in range(1, Lm):
            if inside[i] != inside[i - 1]:
                edges.add(i)
    for i in range(1, Lm // 1000 + 1):                                  # segment edges
        edges.update((1000 * i - 1, 1000 * i, 1000 * i + 1))
    edges = sorted(e for e in edges if 0 < e < Lm)
    sets = []
    sets.append([(max(0, e - d), min(Lm, e + d2)) for e in edges for d, d2 in ((1, 0), (0, 1), (3, 5))])
    # joins exactly on 4 KiB output-tile borders: region lengths that add up to multiples of 4096
    joins = []
    for k in range(12):
        a = r.randrange(Lm - 5000)
        joins.append((a, a + (4096 if k % 3 == 0 else r.choice([1, 4095, 2048, 3000]))))
    pos = sum(b - a for a, b in joins)
    joins.append((0, 4096 - pos % 4096))
    joins += [(a, a + 4096) for a in range(0, Lm - 4096, 9001)]
    sets.append(joins)
    sets.append([(a, min(Lm, a + r.randint(4097, 30_000))) for a in sorted(r.randrange(Lm) for _ in range(8))])     # longer than a tile
    sets.append([(a, a + 1) for a in (r.randrange(Lm) for _ in range(5000))])                                    # single bases
    sets.append([(a, min(Lm, a + r.randint(0, 40))) for a in (r.randrange(Lm) for _ in range(20_000))])           # many short regions
    return sets


def check_boundaries(ctx, pairs, paths=tuple(PATHS)):
    for ref, tgt in pairs:
        rc, inter, mode = ol.orc_compress(ref, tgt, b">edges")
        assert rc == 0
        D = seq_of(ctx.decompress(ref, inter))
        for regs in boundary_region_sets(D, len(D)):
            for path in paths:
                check_extract(ctx, ref, inter, D, regs, path)
        arr = np.array(boundary_region_sets(D, 7)[-1], dtype=np.int64)         # an (n, 2) int64 array goes straight through
        assert ctx.extract(ref, inter, arr) == expect(D, arr.tolist())


def check_chunk_selection(ctx, n=260_000):
    """local-mode files upload / upper-case only the reference chunks the regions copy from: every other chunk is poisoned"""
    from sccg_genome_compression_b200 import synth
    ref, tgt = synth.local_pair(n, synth.seed_for(2, 31))
    ref, tgt = ref.tobytes(), tgt.tobytes()
    tgt = tgt[:100_000] + tgt[100_000:100_900][::-1] + tgt[100_900:150_000] + b"N" * 300 + tgt[150_300:]     # literal segments
    rc, inter, mode = ol.orc_compress(ref, tgt, b">chunks")
    assert rc == 0 and mode == 0
    far_ref = rnd(120_000, "pipe")
    far = b">x\n\n,\n(110000,5000)(-110000,30000)ACGT(60000,100)(-50000,20000)"
    with env(SCCG_PIPE_CHUNK=4096, SCCG_PIPE_POISON=1):
        for rf, it in ((ref, inter), (far_ref, far)):
            D = seq_of(ctx.decompress(rf, it))
            Lm = len(D)
            r = random.Random(Lm)
            sets = [
                [(a, a + 700) for a in range(Lm // 3, Lm // 3 + 6000, 900)],                # clustered
                [(a, min(Lm, a + 50)) for a in (r.randrange(Lm) for _ in range(40))],       # scattered
                [(35_000, 35_004)] if it is far else [(100_100, 100_800), (150_010, 150_290)],       # literal bytes / N only
                [(Lm - 1, Lm)],
            ]
            for regs in sets:
                check_extract(ctx, rf, it, D, regs)
                ctx.set_reference(rf)
                assert ctx.extract_resident(it, regs) == expect(D, regs)


def tolerance_cases():
    """the (body, N list, lowercase list) streams of robustness_cases.check_decoder_tolerance: run lists out of order, overlapping,
    past the end, and two shuffled 3,000-run lists"""
    body = b"(0,1000)ACGT(1000,2000)TT(2100,1500)"
    out = [
        (body, b"", b"(50,10)(-45,3),(12,20)(30,100)"),
        (body, b"", b"(4400,50)(-4400,10)4600,"),
        (body, b"(100,2)(-95,3),50", b"(60,10)(-58,3)"),
        (body, b"(4000,3)(-3990,2)", b"(10,4000)"),
        (b"(0,100)ACGT(50,20)", b"2,(5,3)(100,2)", b"(3,4)10,200"),
        (body, b"(10,5)(2,5)", b""),
        (body, b"", b"(50,10)(-60,3)"),
        (body, b"(5000,10)", b""),
    ]
    r = random.Random("tolerance")
    runs, pos = [], 0
    for _ in range(3000):
        pos += r.randint(1, 3); ln = r.randint(1, 2); runs.append((pos, ln)); pos += ln
    big_body = b"(0,6000)" + b"(-100,6000)" * 2
    for which in ("low", "n"):
        rr = runs[:]; r.shuffle(rr)
        if which == "low":
            rr += [(x + 1, 3) for x, _ in rr[:200]]
        text = bytearray(); prev = 0
        for st, ln in rr:
            text += (b"%d," % (st - prev)) if ln == 1 and r.random() < 0.7 else b"(%d,%d)" % (st - prev, ln)
            prev = st
        out.append((big_body, bytes(text) if which == "n" else b"", bytes(text) if which == "low" else b""))
    return out


def check_unsorted_run_lists(ctx):
    ref = rnd(6000, "tol")
    for enc, nidx, low in tolerance_cases():
        inter = b">tolerant\n" + low + b"\n" + nidx + b"\n" + enc
        try:
            image = ctx.decompress(ref, inter)
        except sccg_b200.SccgError as e1:
            with pytest.raises(sccg_b200.SccgError) as e2:
                ctx.extract(ref, inter, [(0, 0)])
            assert e2.value.code == e1.code
            continue
        D = seq_of(image)
        for path in PATHS:
            check_extract(ctx, ref, inter, D, mixed_regions(len(D), (enc, nidx, low)) if len(D) else [(0, 0)], path)


def check_resident(ctx):
    from sccg_genome_compression_b200 import synth
    ref, tgt = synth.global_gap_pair(60_000, 55_000, synth.seed_for(1, 62))
    ref, tgt = ref.tobytes(), tgt.tobytes()
    lref, ltgt = synth.local_pair(50_000, synth.seed_for(2, 62))
    for rf, tg in ((ref, tgt), (lref.tobytes(), ltgt.tobytes())):
        rc, inter, mode = ol.orc_compress(rf, tg, b">res")
        D = seq_of(ctx.decompress(rf, inter))
        regs = mixed_regions(len(D), "res")
        ctx.set_reference(rf)
        assert ctx.extract_resident(inter, regs) == ctx.extract(rf, inter, regs) == expect(D, regs)
    ctx.clear_reference()
    with pytest.raises(sccg_b200.SccgError) as e:
        ctx.extract_resident(inter, [(0, 1)])
    assert e.value.code == sccg_b200.SCCG_E_ARG


def check_argument_errors(ctx):
    import ctypes as C
    ref = rnd(3000, "args")
    inter = b">a\n\n,\n(0,1000)ACGT(1000,500)"
    D = seq_of(ctx.decompress(ref, inter))
    Lm = len(D)
    good = [(3, 40), (0, Lm)]

    def fails(code, fn):
        with pytest.raises(sccg_b200.SccgError) as e:
            fn()
        assert e.value.code == code, str(e.value)
        assert ctx.extract(ref, inter, good) == expect(D, good)          # the context survived
        return e.value
    fails(sccg_b200.SCCG_E_ARG, lambda: ctx.extract(ref, inter, [(-1, 3)]))
    fails(sccg_b200.SCCG_E_ARG, lambda: ctx.extract(ref, inter, [(5, 4)]))
    fails(sccg_b200.SCCG_E_ARG, lambda: ctx.extract(ref, inter, [(0, 1 << 31)]))
    fails(sccg_b200.SCCG_E_ARG, lambda: ctx.extract(ref, inter, [(0, 1 << 30), (0, 1 << 30)]))
    e = fails(sccg_b200.SCCG_E_ARG, lambda: ctx.extract(ref, inter, [(0, 3), (10, Lm + 1)]))
    assert e.seq_len == Lm
    e = fails(sccg_b200.SCCG_E_ARG, lambda: ctx.extract(ref, inter, [(Lm + 5, Lm + 5)]))          # an empty region past the end
    assert e.seq_len == Lm
    buf = C.create_string_buffer(64)
    e = fails(sccg_b200.SCCG_E_ARG, lambda: ctx.extract(ref, inter, [(0, 100)], C.cast(buf, C.c_void_p).value, 99))
    assert e.out_len == 100
    assert ctx.extract(ref, inter, [(7, 60)], C.cast(buf, C.c_void_p).value, 64) == 53 and buf.raw[:53] == D[7:60]
    # argument errors come before the record stream is looked at; a malformed stream fails like decompress whatever the regions
    fails(sccg_b200.SCCG_E_ARG, lambda: ctx.extract(ref, b">h\n\n,\n(a,5)", [(4, 3)]))
    fails(sccg_b200.SCCG_E_FORMAT, lambda: ctx.extract(ref, b">h\n\n,\n(a,5)", [(0, 1 << 20)]))
    fails(sccg_b200.SCCG_E_BOUNDS, lambda: ctx.extract(ref, b">h\n\n,\n(400,20000)", [(0, 0)]))
    fails(sccg_b200.SCCG_E_FORMAT, lambda: ctx.extract(ref, b"", [(0, 0)]))
    assert ctx.extract(ref, inter, []) == b"" and ctx.last_seq_len == Lm


def check_interleaving(ctx):
    from sccg_genome_compression_b200 import synth
    ref, tgt = synth.local_pair(70_000, synth.seed_for(2, 63))
    ref, tgt = ref.tobytes(), tgt.tobytes()
    rc, inter, mode = ol.orc_compress(ref, tgt, b">inter")
    rc, image = ol.orc_decompress(ref, inter)
    assert ctx.decompress(ref, inter) == image
    D = seq_of(image)
    regs = [(5, 5000), (100, 101)]
    assert ctx.extract(ref, inter, regs) == expect(D, regs)
    assert ctx.decompress(ref, inter) == image


def test_golden_cases(ctx, golden):
    check_golden_cases(ctx, golden)


def test_random_record_streams(ctx):
    check_random_streams(ctx, range(24))


@pytest.mark.parametrize("path", list(PATHS))
def test_region_edges(ctx, path):
    check_boundaries(ctx, boundary_pairs(), (path,))


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
