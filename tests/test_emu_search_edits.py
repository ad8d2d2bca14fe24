"""Edit-distance pattern search in open archives (sccg_archive_search_edits, include/sccg.h) on the CPU (SIMT emulator build):
every hit list must equal the one of tests/edit_probe.cpp, a plain Sellers DP over D (the oracle's decoded sequence) with the
match rule of the header; the two properties the header states must hold against sccg_archive_search; every error must be the
one the contract names.  The check_* functions are shared with test_gpu_search_edits.py."""
import ctypes as C
import random
import subprocess
from pathlib import Path

import numpy as np
import pytest

import sccg_b200
from emu_lib import emu_context
from test_emu_archive import archive_set, revcomp
from test_emu_extract import CASES, PATHS, env, seq_of, unpack
from test_emu_search import SPECIAL, edge_windows, sampled, whole

ARG = sccg_b200.SCCG_E_ARG
HERE = Path(__file__).resolve().parent


@pytest.fixture(scope="module")
def ctx():
    c = emu_context()
    yield c
    c.close()


def build_probe(directory: Path) -> Path:
    exe = directory / "edit_probe"
    subprocess.check_call(["/usr/bin/g++" if Path("/usr/bin/g++").exists() else "g++", "-O2", "-std=c++17", str(HERE / "edit_probe.cpp"), "-o", str(exe)])
    return exe


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    return build_probe(tmp_path_factory.mktemp("edit_probe"))


def expect(probe, Ds, windows, patterns, k, strands=3) -> np.ndarray:
    """the probe's hits [window, start, end, pattern, strand, edits] in (window, end, pattern, strand) order"""
    lines = [f"{k} {strands}", str(len(patterns))] + [p.hex() for p in patterns] + [str(len(Ds))] + [D.hex() or "-" for D in Ds]
    lines += [str(len(windows))] + [f"{a} {s} {e}" for a, s, e in windows]
    inp = probe.parent / "input.txt"
    inp.write_text("\n".join(lines) + "\n")
    out = subprocess.run([str(probe), str(inp)], capture_output=True, check=True).stdout
    h = np.array([[int(x) for x in ln.split()] for ln in out.decode().splitlines()], dtype=np.int64).reshape(-1, 6)
    return h[np.lexsort((h[:, 4], h[:, 3], h[:, 2], h[:, 0]))]


def expect_acgt(probe, D: bytes, patterns, k: int) -> np.ndarray:
    """every hit of A/C/G/T patterns on both strands over the whole of D.  An alignment with at most k edits leaves one of
    k + 1 disjoint parts of the pattern unedited, and that part occurs exactly (A/C/G/T match only themselves, in either case)
    within k bytes of its offset from the alignment's start.  So each exact occurrence at t of the part at offset a gives the
    region [t - a - k, t - a + m + 2k), which holds the whole alignment; overlapping regions are merged, so every region that
    holds an end also holds its best alignment, and the probe scores the merged regions."""
    U = D.upper()
    rows = []
    for i, p in enumerate(patterns):
        m = len(p)
        cut = [m * j // (k + 1) for j in range(k + 2)]
        for st in (0, 1):
            pp = revcomp(p) if st else p
            reg = []
            for a, b in zip(cut, cut[1:]):
                part = pp[a:b].upper()
                at = U.find(part)
                while at >= 0:
                    reg.append((max(0, at - a - k), min(len(D), at - a + m + 2 * k)))
                    at = U.find(part, at + 1)
            reg.sort()
            merged = []
            for s, e in reg:
                if merged and s <= merged[-1][1]:
                    merged[-1][1] = max(merged[-1][1], e)
                else:
                    merged.append([s, e])
            pieces = [D[s:e] for s, e in merged]
            h = expect(probe, pieces, [(j, 0, len(x)) for j, x in enumerate(pieces)], [pp], k, 1)
            base = np.array([s for s, _ in merged], dtype=np.int64)
            h[:, 1] += base[h[:, 0]]
            h[:, 2] += base[h[:, 0]]
            h[:, 0] = 0
            h[:, 3] = i
            h[:, 4] = st
            rows.append(h)
    h = np.concatenate(rows)
    return h[np.lexsort((h[:, 4], h[:, 3], h[:, 2], h[:, 0]))]


def check_edits(ctx, probe, archives, Ds, patterns, windows, k, strands=3, path="auto", split=None):
    with env(SCCG_EXT_LANE_MIN=PATHS[path], SCCG_SEARCH_SPLIT=split):
        got = ctx.search_edits(archives, patterns, windows, max_edits=k, strands={1: "+", 2: "-", 3: "both"}[strands])
        n = ctx.search_edits(archives, patterns, windows, max_edits=k, strands=strands, count_only=True)
    exp = expect(probe, Ds, windows, patterns, k, strands)
    assert got.shape == exp.shape and n == len(exp), (got.shape, exp.shape, n, path, split)
    if not np.array_equal(got, exp):
        bad = next(i for i in range(len(exp)) if not np.array_equal(got[i], exp[i]))
        raise AssertionError(f"hit {bad} (k {k}, {path}, split {split}): got {got[bad].tolist()}, expected {exp[bad].tolist()}")
    return got


def check_properties(ctx, archives, patterns, windows, k, got_k=None):
    """max_edits = 0 gives exactly the Hamming k = 0 hits; every Hamming hit with m <= k mismatches has an edit hit at its end
    with at most m edits (got_k: the edit hits at k, when already computed)"""
    lens = np.array([len(p) for p in patterns], dtype=np.int64)
    e0 = ctx.search_edits(archives, patterns, windows, max_edits=0)
    h0 = ctx.search(archives, patterns, windows, max_mismatches=0)
    x0 = np.stack([h0[:, 0], h0[:, 1], h0[:, 1] + lens[h0[:, 2]], h0[:, 2], h0[:, 3], h0[:, 4]], axis=1).reshape(-1, 6)
    assert np.array_equal(e0, x0[np.lexsort((x0[:, 4], x0[:, 3], x0[:, 2], x0[:, 0]))])    # (window, end, pattern, strand) order
    ek = ctx.search_edits(archives, patterns, windows, max_edits=k) if got_k is None else got_k
    hk = ctx.search(archives, patterns, windows, max_mismatches=k)
    best = {(w, e, i, s): d for w, _, e, i, s, d in ek.tolist()}
    for w, pos, i, s, m in hk.tolist():
        assert best.get((w, pos + len(patterns[i]), i, s), m + 1) <= m, (w, pos, i, s, m)
    return ek, hk


def indel_patterns(Ds, seed, lens, n_each=2):
    """L-mers of D with one or two bases deleted from the middle or inserted into it, upper- and lower-cased"""
    r = random.Random(seed)
    out = []
    for L in lens:
        for t in range(n_each):
            D = Ds[r.randrange(len(Ds))]
            while True:
                s = r.randrange(len(D) - L - 3)
                if set(D[s:s + L + 2].upper()) <= set(b"ACGT"):
                    break
            nd = 1 + t % 2
            c = r.randrange(L // 3, 2 * L // 3)
            if (t // 2) % 2 == 0:
                p = D[s:s + c] + D[s + c + nd:s + L + nd]                           # a deletion from the pattern's view of D
            else:
                p = D[s:s + c] + bytes(r.choice(b"ACGT") for _ in range(nd)) + D[s + c:s + L - nd]
            out.append(p.lower() if t % 2 else p.upper())
    return out


def near_windows(Ds, hits, seed):
    """windows starting or ending on a hit's start or end, or one byte inside or outside it"""
    r = random.Random(seed)
    out = []
    for w, s, e, i, st, d in hits[:: max(1, len(hits) // 20)].tolist():
        out += [(w, s, e), (w, s + 1, e), (w, max(0, s - 1), e - 1), (w, max(0, s - r.randrange(60)), e + 1), (w, s, e + r.randrange(9))]
    return [(a, min(s, len(Ds[a])), min(e, len(Ds[a]))) for a, s, e in out]


def check_archive_set(ctx, probe, paths=tuple(PATHS)):
    ref, files = archive_set()
    ctx.set_reference(ref)
    archives = [ctx.open_archive(inter) for inter, _, _ in files]
    Ds = [D for _, D, _ in files]
    # short and special patterns, k = 0 (a 1-byte pattern allows no edit): a part of each archive with archive 0's N run
    part = [(a, 0, min(20_000, len(D))) for a, D in enumerate(Ds)] + [(0, 19_000, 26_000)]
    mixed = sampled([D[:20_000] for D in Ds], 1, [1, 2, 23, 63, 64]) + SPECIAL
    check_edits(ctx, probe, archives, Ds, mixed, part, 0)
    check_properties(ctx, archives, mixed, part, 0)
    # planted indels: the Hamming search misses an occurrence that the edit search finds
    indel = indel_patterns(Ds, 2, [12, 23, 40])
    long_ = sampled(Ds, 3, [12, 23, 40]) + [b"WSKMBDHVNNACGTAC", b"AC!GT"] + indel
    got = check_edits(ctx, probe, archives, Ds, long_, whole(Ds), 3)
    _, hk = check_properties(ctx, archives, long_, whole(Ds), 3, got)
    lens = np.array([len(p) for p in long_], dtype=np.int64)
    ham_ends = {(w, pos + lens[i], i, s) for w, pos, i, s, _ in hk.tolist()}
    missed = [h for h in got.tolist() if h[3] >= len(long_) - len(indel) and (h[0], h[2], h[3], h[4]) not in ham_ends]
    assert len(missed) >= 1
    edges = edge_windows(Ds, np.stack([got[:, 0], got[:, 1], got[:, 3], got[:, 4], got[:, 5]], axis=1), long_, 3)
    edges += near_windows(Ds, got, 4)
    for path in paths:
        check_edits(ctx, probe, archives, Ds, long_, edges, 2, 3, path)
    for k, strands in ((0, 3), (1, 1), (2, 2), (3, 3)):
        check_edits(ctx, probe, archives, Ds, long_, edges, k, strands)
    # k = 10 on 40-mers
    check_edits(ctx, probe, archives, Ds, indel_patterns(Ds, 5, [40]) + sampled(Ds, 6, [40]), part, 10)
    # tiny windows, down to minlen - k bytes, in tiles made of many pieces or of few
    r = random.Random(7)
    tiny = []
    for t in range(3000):
        a = t % len(Ds)
        s = r.randrange(len(Ds[a]) - 30)
        tiny.append((a, s, s + r.choice([1, 2, 3, 4, 5, 9, 25])))
    short = [b"NGG", b"acgta", b"GANNT"] + sampled(Ds, 8, [5, 9])
    for path in paths:
        check_edits(ctx, probe, archives, Ds, short, tiny, 2, path=path)
    check_edits(ctx, probe, archives, Ds, [b"ACG", b"ttg", b"NGG"], tiny[:800], 1)
    # many launches: a limit far below one window, and one that cuts windows at odd places
    for split in (4096, 9001):
        check_edits(ctx, probe, archives, Ds, long_, whole(Ds) + edges[:40], 2, split=split)
    for a in archives:
        a.close()
    ctx.clear_reference()


def check_golden_search(ctx, probe, golden):
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
            pats = sampled([D], case.name, [min(len(D), L) for L in (5, 23)]) + [b"NGG", b"NNN"]
            pats = [p for p in pats if len(p) >= 2]
            check_edits(ctx, probe, [a], [D], pats, [(0, 0, len(D)), (0, len(D) // 3, len(D))], 1)
    ctx.clear_reference()


def check_contract(ctx, ctx2, probe):
    """count-only, a buffer one hit too small, every argument error in the documented order, other contexts, stale archives,
    zero windows"""
    ref, files = archive_set(30_000, 74)
    ctx.set_reference(ref)
    A = ctx.open_archive(files[0][0])
    D = files[0][1]
    L = len(D)
    lib = ctx.lib
    pats = [b"NGG", D[100:110]]
    exp = expect(probe, [D], [(0, 0, L)], pats, 1)
    assert ctx.search_edits([A], pats, max_edits=1, count_only=True) == len(exp) > 3
    assert ctx.search_edits([A], pats, [], max_edits=1).shape == (0, 6)
    assert ctx.search_edits([A], pats, [], count_only=True) == 0

    arr = (C.c_void_p * 1)(A.handle)
    win = np.array([[0, 0, L]], dtype=np.int64)
    blob = b"".join(pats)
    off = np.array([0, 3, 13], dtype=np.int64)
    n = C.c_int64()
    hits = np.zeros(len(exp), dtype=ctx._EDIT_HIT)

    def raw(archives=arr, na=1, w=win.ctypes.data, nw=1, p=blob, o=off.ctypes.data, npat=2, k=1, strands=3, h=hits.ctypes.data, cap=len(exp), nh=None):
        return lib.sccg_archive_search_edits(ctx.handle, archives, na, w, nw, p, o, npat, k, strands, h, cap, C.byref(n) if nh is None else nh)
    assert raw() == 0 and n.value == len(exp)
    got = np.stack([hits["window"], hits["start"], hits["end"], hits["pattern"], hits["strand"], hits["edits"]], axis=1)
    assert np.array_equal(got, exp)
    assert raw(cap=len(exp) - 1) == ARG and n.value == len(exp)            # one too small: the required count
    assert raw(h=None, cap=0) == 0 and n.value == len(exp)

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
    fails("null argument", cap=-1)
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
    fails("max_edits", k=-1, strands=0)
    fails("max_edits", k=3, strands=0)                                     # the shortest pattern has 3 bytes
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
        assert np.array_equal(ctx.search_edits([A], pats, max_edits=1), exp)
    # an archive of another context, a stale reference generation
    X = ctx2.open_archive(files[0][0])
    with pytest.raises(sccg_b200.SccgError) as e:
        ctx.search_edits([X], pats)
    assert e.value.code == ARG and "another context" in str(e.value)
    X.close()
    ctx.set_reference(ref)
    with pytest.raises(sccg_b200.SccgError) as e:
        ctx.search_edits([A], pats)
    assert e.value.code == ARG and "resident reference" in str(e.value)
    assert ctx.search_edits([A], pats, []).shape == (0, 6)                 # a stale archive no window names is fine
    A.close()
    ctx.clear_reference()
    ctx2.clear_reference()


def test_probe(probe):
    """the probe on hand-checked cases: the shortest text for an insertion, an exact occurrence and its neighbours at one edit,
    the reverse complement"""
    D = b"TTTTACGTACGGTTTT"
    assert [0, 4, 12, 0, 0, 1] in expect(probe, [D], [(0, 0, len(D))], [b"ACGTAGG"], 1, 1).tolist()     # ACGTACGG: one C inserted
    h = expect(probe, [b"GGACGTGG"], [(0, 0, 8)], [b"ACGT"], 1, 1).tolist()
    assert h == [[0, 2, 5, 0, 0, 1], [0, 2, 6, 0, 0, 0], [0, 2, 7, 0, 0, 1]]
    assert expect(probe, [b"ACGNT"], [(0, 0, 5)], [b"G"], 0, 3).tolist() == [[0, 1, 2, 0, 1, 0], [0, 2, 3, 0, 0, 0]]


def test_archive_set(ctx, probe):
    check_archive_set(ctx, probe)


def test_golden_cases(ctx, probe, golden):
    check_golden_search(ctx, probe, golden)


def test_contract(ctx, probe):
    ctx2 = emu_context()
    try:
        check_contract(ctx, ctx2, probe)
    finally:
        ctx2.close()
