"""Both archive search engines (sccg_archive_search and sccg_archive_search_edits, include/sccg.h) over the whole of their
contract on the CPU (SIMT emulator build): D holding every byte value, every width of the Hamming engine's mismatch counter
(k up to 63), the edit engine's widest look-behind (m = 64, k = 63), 1,024 patterns in one call, windows and launch cuts at
their edges, and three properties that need no reference: strand symmetry, case invariance and monotone k.  Every hit list
is compared in full with brute() (test_emu_search.py) or the probe (tests/edit_probe.cpp), count-only totals included.  The
check_* functions are shared with test_gpu_search_space.py."""
import random

import numpy as np
import pytest

import oracle_lib as ol
from emu_lib import emu_context
from test_emu_archive import archive_set, every_byte_archive, revcomp
from test_emu_extract import seq_of
from test_emu_search import check_search, whole
from test_emu_search_edits import check_edits, probe  # noqa: F401

IUPAC = b"RYSWKMBDHVNryswkmbdhvn"
PUNCT = b"!#$%&'*+./:;<=>?@[\\]^_`{|}~\""


@pytest.fixture(scope="module")
def ctx():
    c = emu_context()
    yield c
    c.close()


def check_both(ctx, probe, archives, Ds, patterns, windows, k, strands=3, path="auto", split=None):
    """one hit list of each engine, each against its reference -> (Hamming hits, edit hits)"""
    return (check_search(ctx, archives, Ds, patterns, windows, k, strands, path, split),
            check_edits(ctx, probe, archives, Ds, patterns, windows, k, strands, path, split))


def odd_target_archive():
    """a target compressed by the oracle whose literals hold IUPAC codes in both cases, punctuation, control bytes and bytes
    >= 0x80, with lowercase runs over IUPAC letters and N runs -> (ref, intermediate, mode, tgt, D)"""
    from sccg_genome_compression_b200 import synth
    ref_np, tgt_np = synth.local_pair(12_000, synth.seed_for(2, 77))
    ref = ref_np.tobytes()
    t = bytearray(tgt_np.tobytes())
    r = random.Random(77)
    odd = IUPAC + PUNCT + b"\x00\x01\x1f\x7f" + bytes(range(0x80, 0x100))
    for i in range(50, len(t), 61):                                     # single odd bytes: literals between matches
        t[i] = r.choice(odd)
    for a in (2000, 5000, 9000):                                        # stretches of odd bytes
        t[a:a + 40] = bytes(r.choice(odd) for _ in range(40))
    t[3000:3100] = bytes(r.choice(b"RYSWKMBDHVN") for _ in range(100))
    for a, b in ((3050, 3150), (5010, 5030), (7000, 7400)):             # lowercase runs, over IUPAC letters too
        t[a:b] = bytes(t[a:b]).lower()
    for a, b in ((4000, 4100), (6000, 6001), (7300, 7350)):             # N runs, one inside a lowercase run
        t[a:b] = b"N" * (b - a)
    tgt = bytes(t)
    rc, inter, mode = ol.orc_compress(ref, tgt, b">odd")
    assert rc == 0
    rc, image = ol.orc_decompress(ref, inter)
    assert rc == 0
    D = seq_of(image)
    assert max(D) >= 0x80 and b"n" in D and b"N" in D and set(b"rykm") <= set(D) and set(b"RYKM") <= set(D)
    return ref, inter, mode, tgt, D


def substituted_pieces(D, seed, lens, n_each=3):
    """pieces of D with up to two bytes replaced by random ones (any value), some swap-cased"""
    r = random.Random(seed)
    out = []
    for L in lens:
        for t in range(n_each):
            s = r.randrange(len(D) - L + 1)
            p = bytearray(D[s:s + L])
            for _ in range(r.randrange(3)):
                p[r.randrange(L)] = r.randrange(256)
            out.append(bytes(p).swapcase() if t == 2 else bytes(p))
    return out


def check_every_byte(ctx, probe, paths=("lanes", "warps")):
    """archives whose D holds every byte value: all 256 single bytes in one call, IUPAC codes in both cases, 0x00, 0xff
    and punctuation, and pieces of D with random bytes substituted; both engines, every strand setting, both build paths"""
    ref, inter, D = every_byte_archive()
    ref2, inter2, mode2, tgt2, D2 = odd_target_archive()
    assert ctx.compress(ref2, tgt2, b">odd") == (inter2, mode2)
    singles = [bytes([b]) for b in range(256)]
    odd = [b"RYSWKMBDHVN", b"ryswkmbdhvn", b"Ry", b"sW", b"Kmb", b"DhV", b"NnNn", b"\x00\xff", b"\xff\x80\xfe", b"!#$%",
           b"@[`{", b"NGG", b"rYkM", b"\x00\x00", b"~\x7f", b"Nn!"]
    for r, a_inter, X in ((ref, inter, D), (ref2, inter2, D2)):
        ctx.set_reference(r)
        with ctx.open_archive(a_inter) as a:
            L = len(X)
            wins = [(0, 0, L), (0, L // 3, L), (0, 17, 97)]
            pieces = substituted_pieces(X, L, [2, 5, 17, 31, 32, 33, 63, 64])
            for strands in (1, 2, 3):
                got, _ = check_both(ctx, probe, [a], [X], singles, wins, 0, strands)
                assert X is not D or len(np.unique(got[:, 2])) == 255                   # every byte but '\n' hits
                check_both(ctx, probe, [a], [X], odd + pieces, wins, 1, strands)
            for path in paths:
                check_both(ctx, probe, [a], [X], singles, wins[:1], 0, 3, path)
                check_both(ctx, probe, [a], [X], odd + pieces, wins[:1], 1, 3, path)
            long_ = [p for p in pieces if len(p) >= 17]
            for k in (8, 16):
                check_both(ctx, probe, [a], [X], long_, wins[:1], k)
            check_properties(ctx, [a], odd + pieces, wins, 1)
        ctx.clear_reference()


def planted(Ds, windows, L, seed, subs=(0, 1)):
    """L-mers taken from inside the windows, one for each count in subs of bytes replaced by other bases: each has a hit
    with exactly that many mismatches where it was taken"""
    r = random.Random(seed)
    out = []
    for t, n in enumerate(subs):
        a, s, e = windows[r.randrange(len(windows))]
        x = r.randrange(s, e - L + 1)
        p = bytearray(Ds[a][x:x + L])
        for j in r.sample(range(L), n):
            p[j] = r.choice([c for c in b"ACGT" if c != p[j] & 0xdf])
        out.append(bytes(p).lower() if t % 2 else bytes(p))
    return out


WIDTHS = ((8, (4, 7)), (16, (7, 8, 15)), (33, (15, 16, 31, 32)), (64, (31, 32, 63)))


def check_counter_widths(ctx, probe):
    """every width of the Hamming engine's bit-sliced counter (bits(k + 1) = 3 to 6 here; 1 to 3 run elsewhere) and the edit
    engine on the same lengths, up to m = 64 with k = 63 (126 bytes of look-behind) at tile starts and launch cuts; mixed
    lengths where the shortest pattern bounds k and a 64-byte one sets the look-ahead or look-behind"""
    ref, files = archive_set()
    ctx.set_reference(ref)
    archives = [ctx.open_archive(inter) for inter, _, _ in files]
    Ds = [D for _, D, _ in files]
    part = [(a, 0, min(6000, len(D))) for a, D in enumerate(Ds)]
    short = [(0, 0, 3000), (1, 1000, 4000)]                              # tile 1 starts 1,096 bytes into window 1
    for L, ks in WIDTHS:
        pats = planted(Ds, short, L, L, (0,) + ks)
        for k in ks:
            got = check_search(ctx, archives, Ds, pats, part, k)
            assert (got[:, 4] == k).any() and (got[:, 4] < k // 2).any(), (L, k)
            check_edits(ctx, probe, archives, Ds, pats, short, k)
        check_edits(ctx, probe, archives, Ds, pats, short, ks[-1], split=1000)
        check_search(ctx, archives, Ds, pats, part, ks[-1], split=1000)
    mixed = planted(Ds, short, 8, 1) + planted(Ds, short, 64, 2) + planted(Ds, short, 33, 3)
    for k in (3, 7):
        check_both(ctx, probe, archives, Ds, mixed, short, k)
        check_both(ctx, probe, archives, Ds, mixed, short, k, split=700)
    mixed = planted(Ds, short, 16, 4) + planted(Ds, short, 64, 5)
    check_both(ctx, probe, archives, Ds, mixed, short, 15, 2)
    for a in archives:
        a.close()
    ctx.clear_reference()


def offset_calls(ctx, archives, patterns, windows, k, edits, per=256):
    """the hits of len(patterns) / per calls of per patterns each, with their pattern indices offset, in call order"""
    col = 3 if edits else 2
    parts = []
    for b in range(0, len(patterns), per):
        h = (ctx.search_edits(archives, patterns[b:b + per], windows, max_edits=k) if edits
             else ctx.search(archives, patterns[b:b + per], windows, max_mismatches=k))
        h[:, col] += b
        parts.append(h)
    h = np.concatenate(parts)
    key = (h[:, 4], h[:, 3], h[:, 2], h[:, 0]) if edits else (h[:, 3], h[:, 2], h[:, 1], h[:, 0])
    return h[np.lexsort(key)]


def check_many_patterns(ctx, probe):
    """1,024 patterns in one call: hits for pattern indices >= 256 and >= 1,000, a pattern listed twice gives the same rows
    under both indices, and the call equals four calls of 256 patterns"""
    ref, files = archive_set()
    ctx.set_reference(ref)
    archives = [ctx.open_archive(inter) for inter, _, _ in files]
    Ds = [D for _, D, _ in files]
    wins = [(a, 1000 * a, 1000 * a + 400) for a in range(len(Ds))] + [(0, 4000, 4300)]
    r = random.Random(9)
    pats = []
    for i in range(1024):
        a, s, e = wins[i % len(wins)]
        L = r.randrange(6, 13)
        x = r.randrange(s, e - L + 1)
        p = Ds[a][x:x + L]
        pats.append(p.swapcase() if i % 3 == 0 else p)
    pats[1000] = pats[3]
    pats[700] = pats[1023]
    got_h, got_e = check_both(ctx, probe, archives, Ds, pats, wins, 1)
    for got, col in ((got_h, 2), (got_e, 3)):
        idx = set(got[:, col].tolist())
        assert any(i >= 256 for i in idx) and len({i for i in idx if i >= 1000}) >= 10
        for i, j in ((3, 1000), (700, 1023)):
            gi, gj = got[got[:, col] == i], got[got[:, col] == j]
            gj[:, col] = i
            assert len(gi) > 0 and np.array_equal(gi, gj), (i, j)
    assert np.array_equal(offset_calls(ctx, archives, pats, wins, 1, False), got_h)
    assert np.array_equal(offset_calls(ctx, archives, pats, wins, 1, True), got_e)
    for a in archives:
        a.close()
    ctx.clear_reference()


SPLITS = (1, 31, 32, 33, 4095, 4096, 4097)


def check_window_shapes(ctx, probe):
    """duplicate and overlapping windows, archives named out of order, windows of exactly minlen and minlen - 1 bytes
    (edits: minlen - k and minlen - k - 1), windows ending at len(D), windows across N runs and lowercase runs; then
    SCCG_SEARCH_SPLIT at 1, 31, 32, 33, 4095, 4096, 4097 and 4096 + maxlen, each giving the unsplit hits"""
    ref, files = archive_set()
    ctx.set_reference(ref)
    archives = [ctx.open_archive(inter) for inter, _, _ in files]
    Ds = [D for _, D, _ in files]
    k = 2
    pats = [Ds[0][4080:4087], Ds[1][500:507].lower(), Ds[2][900:907], Ds[0][4093:4100], Ds[2][900:923], Ds[0][12_250:12_314],
            b"NNNNNNN", b"acgtnnn"]
    minlen, maxlen = 7, 64
    wins = [(0, 4000, 4300), (0, 4000, 4300), (0, 4200, 4500), (2, 850, 1000), (0, 50, 350), (1, 450, 560), (3, 0, 200)]
    wins += [(0, 8150, 8250), (0, 19_950, 20_100), (0, 24_450, 24_600), (0, 2990, 3010), (0, 12_200, 12_400), (0, 16_350, 16_450)]
    for a, x in ((0, 4080), (1, 500), (2, 900), (0, 4093)):             # a hit's start; the last is inside an N run
        for n in (minlen, minlen - 1, minlen - k, minlen - k - 1):
            wins += [(a, x, x + n), (a, x + 1, x + 1 + n)]
    for a, D in enumerate(Ds):
        wins += [(a, len(D) - 100, len(D)), (a, len(D) - minlen, len(D)), (a, len(D) - minlen + k, len(D)), (a, len(D), len(D))]
    for strands in (1, 2, 3):
        got_h, got_e = check_both(ctx, probe, archives, Ds, pats, wins, k, strands)
        assert len(got_h) and len(got_e)
    small = wins[3:6] + wins[-4 * len(Ds):]
    big = wins + [(1, 0, 3000), (3, 1000, 4000)]
    assert sum(e - s for _, s, e in small) < 1100 and sum(e - s for _, s, e in big) > 2 * 4096 + maxlen
    for split in SPLITS + (4096 + maxlen,):
        check_both(ctx, probe, archives, Ds, pats, small if split < 4000 else big, k, split=split)
    for a in archives:
        a.close()
    ctx.clear_reference()


def check_properties(ctx, archives, patterns, windows, k):
    """strand symmetry (strand-2 hits of P are the strand-1 hits of revcomp(P)), case invariance (swap-cased patterns give
    the same hits) and monotone k (the hits at k are the rows of k + 1 within k; an edit hit keeps its start, since d(e) does
    not depend on k), for both engines -> (Hamming hits at k, edit hits at k)"""
    out = []
    for edits in (False, True):
        def run(pats, kk, strands="both"):
            return (ctx.search_edits(archives, pats, windows, max_edits=kk, strands=strands) if edits
                    else ctx.search(archives, pats, windows, max_mismatches=kk, strands=strands))
        sc, dc = (4, 5) if edits else (3, 4)
        got = run(patterns, k)
        minus = run(patterns, k, "-")
        plus_rc = run([revcomp(p) for p in patterns], k, "+")
        plus_rc[:, sc] = 1
        assert len(got) and np.array_equal(minus, plus_rc), edits
        assert np.array_equal(minus, got[got[:, sc] == 1]), edits
        assert np.array_equal(run([p.swapcase() for p in patterns], k), got), edits
        if k + 1 < min(len(p) for p in patterns):
            up = run(patterns, k + 1)
            assert np.array_equal(up[up[:, dc] <= k], got), edits
        if k > 0:
            down = run(patterns, k - 1)
            assert np.array_equal(got[got[:, dc] <= k - 1], down), edits
        out.append(got)
    return out


def check_properties_archive_set(ctx):
    """the three properties on whole archives, with A/C/G/T, IUPAC and other patterns"""
    ref, files = archive_set()
    ctx.set_reference(ref)
    archives = [ctx.open_archive(inter) for inter, _, _ in files]
    Ds = [D for _, D, _ in files]
    pats = [Ds[0][700:723], Ds[3][5000:5012].lower(), b"RGAATTCY", b"AC!GTN", b"WSKMBDHVNNACGTAC"]
    check_properties(ctx, archives, pats, whole(Ds), 2)
    for a in archives:
        a.close()
    ctx.clear_reference()


def test_every_byte(ctx, probe):  # noqa: F811
    check_every_byte(ctx, probe)


def test_counter_widths(ctx, probe):  # noqa: F811
    check_counter_widths(ctx, probe)


def test_many_patterns(ctx, probe):  # noqa: F811
    check_many_patterns(ctx, probe)


def test_window_shapes(ctx, probe):  # noqa: F811
    check_window_shapes(ctx, probe)


def test_properties(ctx):
    check_properties_archive_set(ctx)

