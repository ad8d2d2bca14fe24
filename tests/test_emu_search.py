"""Pattern search in open archives (sccg_archive_search, include/sccg.h) on the CPU (SIMT emulator build): every hit list must
equal a NumPy brute force over D (the oracle's decoded sequence) with a 256 x 256 match table built from the rule of the
header, and equal a brute force over the bytes sccg_archive_extract returns for each window; every error must be the one the
contract names.  The check_* functions are shared with test_gpu_search.py."""
import ctypes as C
import random

import numpy as np
import pytest

import sccg_b200
from emu_lib import emu_context
from test_emu_archive import COMP, archive_set, revcomp
from test_emu_extract import CASES, PATHS, env, seq_of, unpack

ARG = sccg_b200.SCCG_E_ARG
IUPAC = {b"R": b"AG", b"Y": b"CT", b"S": b"CG", b"W": b"AT", b"K": b"GT", b"M": b"AC", b"B": b"CGT", b"D": b"AGT", b"H": b"ACT",
         b"V": b"ACG", b"N": b"ACGT"}


@pytest.fixture(scope="module")
def ctx():
    c = emu_context()
    yield c
    c.close()


def _up(b: int) -> int:
    return b - 32 if 97 <= b <= 122 else b


def _match_table() -> np.ndarray:
    """M[p, d]: pattern byte p matches D byte d"""
    M = np.zeros((256, 256), dtype=bool)
    for p in range(256):
        P = _up(p)
        allowed = IUPAC.get(bytes([P]), b"")
        for d in range(256):
            M[p, d] = _up(d) == P or _up(d) in allowed
    return M


MISS = ~_match_table()


def brute(Ds, windows, patterns, k, strands=3) -> np.ndarray:
    """every hit [window, pos, pattern, strand, mismatches], in (window, pos, pattern, strand) order"""
    rows = []
    for w, (a, s, e) in enumerate(windows):
        seg = np.frombuffer(Ds[a][s:e], dtype=np.uint8)
        for i, p in enumerate(patterns):
            L = len(p)
            if len(seg) < L:
                continue
            n = len(seg) - L + 1
            for st in (0, 1):
                if not (strands >> st) & 1:
                    continue
                pp = revcomp(p) if st else p
                mm = np.zeros(n, dtype=np.int16)
                for j in range(L):
                    mm += MISS[pp[j]][seg[j:j + n]]
                pos = np.flatnonzero(mm <= k)
                rows.append(np.stack([np.full(len(pos), w), s + pos, np.full(len(pos), i), np.full(len(pos), st), mm[pos]], axis=1))
    if not rows:
        return np.zeros((0, 5), dtype=np.int64)
    h = np.concatenate(rows).astype(np.int64)
    return h[np.lexsort((h[:, 3], h[:, 2], h[:, 1], h[:, 0]))]


def check_search(ctx, archives, Ds, patterns, windows, k, strands=3, path="auto", split=None, via_query=False):
    with env(SCCG_EXT_LANE_MIN=PATHS[path], SCCG_SEARCH_SPLIT=split):
        got = ctx.search(archives, patterns, windows, max_mismatches=k, strands={1: "+", 2: "-", 3: "both"}[strands])
        n = ctx.search(archives, patterns, windows, max_mismatches=k, strands=strands, count_only=True)
    exp = brute(Ds, windows, patterns, k, strands)
    assert got.shape == exp.shape and n == len(exp), (got.shape, exp.shape, n, path, split)
    if not np.array_equal(got, exp):
        bad = next(i for i in range(len(exp)) if not np.array_equal(got[i], exp[i]))
        raise AssertionError(f"hit {bad} ({path}, split {split}): got {got[bad].tolist()}, expected {exp[bad].tolist()}")
    if via_query:                                                          # the bytes sccg_archive_extract gives for each window
        pieces = [ctx.query(archives, [(a, s, e, 0)]) for a, s, e in windows]
        exp2 = brute(pieces, [(w, 0, e - s) for w, (_, s, e) in enumerate(windows)], patterns, k, strands)
        exp2[:, 1] += np.array([windows[w][1] for w in exp2[:, 0]], dtype=np.int64).reshape(-1)
        assert np.array_equal(got, exp2)
    return got


def sampled(Ds, seed, lens, n_each=2):
    """k-mers of D (so hits exist), upper- and lower-cased"""
    r = random.Random(seed)
    out = []
    for L in lens:
        for t in range(n_each):
            D = Ds[r.randrange(len(Ds))]
            s = r.randrange(len(D) - L + 1)
            p = D[s:s + L]
            out.append(p.lower() if t % 2 else p.upper())
    return out


SPECIAL = [b"NGG", b"RGAATTCY", b"NNNNN", b"GAATTC", b"AC!G", b"acgtn", b"WSKMBDHV", b"nnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnnn"]


def whole(Ds):
    return [(a, 0, len(D)) for a, D in enumerate(Ds)]


def edge_windows(Ds, hits, patterns, seed):
    """windows ending exactly on a hit's end or one byte short of it, around multiples of 4096, overlapping, shorter than a
    pattern, empty"""
    r = random.Random(seed)
    out = []
    for w, pos, i, st, mm in hits[:: max(1, len(hits) // 20)].tolist():
        e = pos + len(patterns[i])
        out += [(w, max(0, pos - r.randrange(50)), e), (w, max(0, pos - 3), e - 1), (w, pos, e)]
    for a, D in enumerate(Ds):
        for m in range(4096, len(D) - 9000, 4096 * 7):
            out += [(a, m - 1, m + 4097), (a, m, m + 4096), (a, m + 1, m + 8191), (a, m - 30, m + 30)]
        out += [(a, 0, 1), (a, 5, 5), (a, len(D) - 2, len(D)), (a, 100, 5000), (a, 2000, 7000)]
    return [(a, min(s, len(Ds[a])), min(e, len(Ds[a]))) for a, s, e in out]


def check_archive_set(ctx, paths=tuple(PATHS)):
    ref, files = archive_set()
    ctx.set_reference(ref)
    archives = [ctx.open_archive(inter) for inter, _, _ in files]
    Ds = [D for _, D, _ in files]
    # short and special patterns find hits nearly everywhere: a part of each archive, with archive 0's 4.5 kb N run
    part = [(a, 0, min(20_000, len(D))) for a, D in enumerate(Ds)] + [(0, 19_000, 26_000)]
    mixed = sampled([D[:20_000] for D in Ds], 1, [1, 2, 23, 63, 64]) + SPECIAL
    check_search(ctx, archives, Ds, mixed, part, 0, via_query=True)
    long_ = sampled(Ds, 2, [12, 23, 40]) + [b"WSKMBDHVNNACGTAC"]
    got = check_search(ctx, archives, Ds, long_, whole(Ds), 3, via_query=True)
    edges = edge_windows(Ds, got, long_, 3)
    for path in paths:
        check_search(ctx, archives, Ds, long_, edges, 2, 3, path)
    for k, strands in ((1, 1), (2, 2), (3, 3)):
        check_search(ctx, archives, Ds, long_, edges, k, strands)
    r = random.Random(4)
    tiny = []
    for t in range(3000):
        a = t % len(Ds)
        s = r.randrange(len(Ds[a]) - 30)
        tiny.append((a, s, s + r.choice([1, 3, 4, 9, 25])))
    for path in paths:
        check_search(ctx, archives, Ds, [b"NGG", b"acg", b"T", b"GANNT"] + sampled(Ds, 5, [3, 9]), tiny, 0, path=path)
    # many launches: a limit far below one window, and one that cuts windows at odd places
    for split in (4096, 9001):
        check_search(ctx, archives, Ds, long_, whole(Ds) + edges[:40], 1, split=split)
    for a in archives:
        a.close()
    ctx.clear_reference()


def check_golden_search(ctx, golden):
    """every golden case that opens as an archive, searched whole with k-mers of its own D"""
    for case in CASES:
        g = golden["cases"][case.name]
        inter = unpack(g["intermediate_z"])
        ctx.set_reference(case.ref)
        try:
            D = seq_of(ctx.decompress_resident(inter))
        except sccg_b200.SccgError:
            continue
        if not D:
            continue
        with ctx.open_archive(inter) as a:
            pats = sampled([D], case.name, [min(len(D), L) for L in (1, 5, 23)]) + [b"NGG", b"NNN"]
            pats = [p for p in pats if p]
            check_search(ctx, [a], [D], pats, [(0, 0, len(D)), (0, len(D) // 3, len(D))], 0)
    ctx.clear_reference()


def check_contract(ctx, ctx2):
    """count-only, a buffer one hit too small, every argument error in the documented order, other contexts, stale archives,
    zero windows"""
    ref, files = archive_set(30_000, 74)
    ctx.set_reference(ref)
    A = ctx.open_archive(files[0][0])
    D = files[0][1]
    L = len(D)
    lib = ctx.lib
    pats = [b"NGG", D[100:110]]
    exp = brute([D], [(0, 0, L)], pats, 1)
    assert ctx.search([A], pats, max_mismatches=1, count_only=True) == len(exp) > 3
    assert ctx.search([A], pats, [], max_mismatches=1).shape == (0, 5)
    assert ctx.search([A], pats, [], count_only=True) == 0

    arr = (C.c_void_p * 1)(A.handle)
    win = np.array([[0, 0, L]], dtype=np.int64)
    blob = b"".join(pats)
    off = np.array([0, 3, 13], dtype=np.int64)
    n = C.c_int64()
    hits = np.zeros(len(exp), dtype=ctx._HIT)

    def raw(archives=arr, na=1, w=win.ctypes.data, nw=1, p=blob, o=off.ctypes.data, npat=2, k=1, strands=3, h=hits.ctypes.data, cap=len(exp), nh=None):
        return lib.sccg_archive_search(ctx.handle, archives, na, w, nw, p, o, npat, k, strands, h, cap, C.byref(n) if nh is None else nh)
    assert raw() == 0 and n.value == len(exp)
    assert raw(cap=len(exp) - 1) == ARG and n.value == len(exp)            # one too small: the required count
    assert raw(h=None, cap=0) == 0 and n.value == len(exp)
    got = np.stack([hits["window"], hits["pos"], hits["pattern"], hits["strand"], hits["mismatches"]], axis=1)
    assert np.array_equal(got, exp)

    def fails(msg, **kw):
        rc = raw(**kw)
        assert rc == ARG and msg in lib.sccg_last_error().decode(), (rc, lib.sccg_last_error().decode(), kw)
    # 1. pointers and counts
    fails("null argument", archives=None)
    fails("null argument", w=None)
    fails("null argument", p=None)
    fails("null argument", o=None)
    fails("null argument", nh=C.cast(None, C.POINTER(C.c_int64)))
    fails("null argument", na=-1)
    fails("null argument", nw=-1, o=None, k=99)                            # before any pattern check
    fails("2^31", nw=1 << 31, npat=0)
    # 2. patterns, in order
    fails("1 to 1024 patterns", npat=0, k=-1)
    big = np.arange(1026, dtype=np.int64)
    fails("1 to 1024 patterns", o=big.ctypes.data, npat=1025, p=b"A" * 1025)
    bad_off = np.array([1, 3, 13], dtype=np.int64)
    fails("pattern_off", o=bad_off.ctypes.data, k=-1)
    dec = np.array([0, 3, 2], dtype=np.int64)
    fails("1 to 64 bytes", o=dec.ctypes.data, k=-1, strands=0)
    long_off = np.array([0, 3, 68], dtype=np.int64)
    fails("1 to 64 bytes", o=long_off.ctypes.data, p=b"A" * 68, k=-1)
    fails("max_mismatches", k=-1, strands=0)
    fails("max_mismatches", k=3, strands=0)                                # the shortest pattern has 3 bytes
    fails("strands", strands=0, w=np.array([[5, 0, 1]], dtype=np.int64).ctypes.data)
    fails("strands", strands=4)
    # 3. windows: the order of sccg_archive_extract's checks, whichever window commits them
    ctx2.set_reference(ref)
    X = ctx2.open_archive(files[0][0])
    arr2 = (C.c_void_p * 3)(A.handle, X.handle, None)

    def wins(*rows):
        w = np.array(rows, dtype=np.int64)
        wins.keep = w
        return w.ctypes.data
    fails("out of range", archives=arr2, na=3, w=wins((0, -1, 3), (1, 0, 1), (2, 0, 1), (3, 0, 1)), nw=4)
    fails("out of range", w=wins((-1, 0, 1)))
    fails("null argument", archives=arr2, na=3, w=wins((0, 0, L + 1), (1, 0, 1), (2, 0, 1)), nw=3)
    fails("another context", archives=arr2, na=3, w=wins((0, 9, 1), (1, 0, 1)), nw=2)
    fails("start <= end", w=wins((0, 0, L + 1), (0, 9, 1)), nw=2)
    fails("start <= end", w=wins((0, -1, 3)))
    fails("past the end", w=wins((0, 0, L + 1)))
    X.close()
    with env(SCCG_SEARCH_SPLIT=4096):
        assert np.array_equal(ctx.search([A], pats, max_mismatches=1), exp)
    # an archive of another context, a stale reference generation
    X = ctx2.open_archive(files[0][0])
    with pytest.raises(sccg_b200.SccgError) as e:
        ctx.search([X], pats)
    assert e.value.code == ARG and "another context" in str(e.value)
    X.close()
    ctx.set_reference(ref)
    with pytest.raises(sccg_b200.SccgError) as e:
        ctx.search([A], pats)
    assert e.value.code == ARG and "resident reference" in str(e.value)
    assert ctx.search([A], pats, []).shape == (0, 5)                       # a stale archive no window names is fine
    A.close()
    ctx.clear_reference()
    ctx2.clear_reference()


def test_match_table():
    M = ~MISS
    for p in b"ACGTacgt":
        assert M[p].sum() == 2
    assert M[ord("N"), ord("n")] and M[ord("n"), ord("A")] and not M[ord("N"), ord("R")]
    assert M[ord("R"), ord("g")] and M[ord("r"), ord("R")] and not M[ord("R"), ord("C")] and not M[ord("A"), ord("N")]
    assert M[ord("!"), ord("!")] and M[ord("!")].sum() == 1 and not M[1, 0x21]
    assert revcomp(b"NGG") == b"CCN" and COMP[ord("R")] == ord("Y")


def test_archive_set(ctx):
    check_archive_set(ctx)


def test_golden_cases(ctx, golden):
    check_golden_search(ctx, golden)


def test_contract(ctx):
    ctx2 = emu_context()
    try:
        check_contract(ctx, ctx2)
    finally:
        ctx2.close()
